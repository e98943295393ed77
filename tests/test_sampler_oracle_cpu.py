"""The sampler replay oracle (oracle/sampler_oracle.py) on the CPU: Philox known answers, replay frequencies against exact
probabilities, tie and -inf rules, and the reference's own golden draws against the bf16 candidate sets."""
import os

import pytest
import torch
from scipy import stats

from oracle.sampler_oracle import (M32, Policy, candidate_set_bf16, philox4x32_10, predictor_draw, replay, replayer,
                                   stream_key, talker_draw, uniform)

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "sampling_golden.pt")


def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32_10."""
    assert philox4x32_10((0, 0, 0, 0), (0, 0)) == (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)
    assert philox4x32_10((M32,) * 4, (M32, M32)) == (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)


def test_uniform_key_and_schedule():
    u = uniform(0, 0)
    assert u == (0x6627E8D5 >> 8) / 2.0**24
    # the 64-bit key and draw index split into (lo, hi) words
    assert uniform(2**32 + 7, 2**33 + 5) == (philox4x32_10((5, 2, 0, 0), (7, 1))[0] >> 8) / 2.0**24
    assert stream_key(5, 0, False) == stream_key(5, 3, True) == 5 ^ 0x9E3779B97F4A7C15
    assert stream_key(5, 1, False) == (5 ^ (2 * 0x9E3779B97F4A7C15)) % 2**64
    assert stream_key(2**64 - 1, 0, True) == (2**64 - 1) ^ 0x9E3779B97F4A7C15
    # prefill draws 0; frame f: codebooks 33f+2 .. 33f+16, then the talker 33(f+1); every index used once
    used = [0] + [d for f in range(4) for d in [predictor_draw(f, i) for i in range(15)] + [talker_draw(f)]]
    assert len(set(used)) == len(used)
    assert (predictor_draw(0, 0), predictor_draw(0, 14), talker_draw(0), predictor_draw(1, 0)) == (2, 16, 33, 35)


def test_replay_frequencies_match_exact_probabilities():
    """2^16 draws of one key against the float64 softmax, chi-square, including a token of probability 1e-3."""
    p = torch.tensor([0.4, 0.25, 0.15, 0.1, 0.05, 0.03, 0.019, 0.001], dtype=torch.float64)
    logits = torch.log(p).float()
    p = torch.softmax(logits.double(), 0)
    pol = Policy(top_k=0, top_p=1.0, temperature=1.0)
    r = replayer(logits, pol)
    n = 2**16
    key = stream_key(1234, 0, True)
    counts = torch.zeros(8, dtype=torch.float64)
    n_amb = 0
    for d in range(n):
        t, amb = r.draw(key, d)
        counts[t] += 1
        n_amb += amb
    assert n_amb < 10
    res = stats.chisquare(counts.numpy(), (p * n).numpy())
    print(f"counts {counts.tolist()} expected {(p * n).tolist()} chi2 p={res.pvalue:.3f}")
    assert res.pvalue > 1e-3
    assert counts[7] > 0


def test_replay_ties_neg_inf_and_greedy():
    # ties at the k-th value all survive top-k; -inf is never drawn
    logits = torch.tensor([1.0, 3.0, 2.0, 2.0, float("-inf"), 2.0, 0.5, float("-inf")])
    pol = Policy(top_k=2, top_p=1.0, temperature=1.0)
    assert candidate_set_bf16(logits, pol).tolist() == [False, True, True, True, False, True, False, False]
    drawn = {replay(logits, pol, None, 99, d)[0] for d in range(400)}
    assert drawn == {1, 2, 3, 5}
    pol0 = Policy(top_k=0, top_p=1.0, temperature=1.0)
    drawn = {replayer(logits, pol0).draw(7, d)[0] for d in range(2000)}
    assert 4 not in drawn and 7 not in drawn and drawn == {0, 1, 2, 3, 5, 6}
    # greedy: lowest index of the maximum, after penalty and suppression
    x = torch.tensor([0.0, 2.0, 1.0, 2.0, 2.0])
    assert replay(x, Policy(do_sample=False), None, 0, 0) == (1, False)
    assert replay(x, Policy(do_sample=False, repetition_penalty=1.5), [1, 1, -3, 9], 0, 0) == (3, False)
    assert replay(x, Policy(do_sample=False, suppress_tail=2, eos=4), None, 0, 0) == (1, False)
    # top_p tiny keeps the argmax only, ties at the top included by neither side beyond rank 0
    assert {replay(x, Policy(top_k=0, top_p=1e-3, temperature=1.0), None, 3, d)[0] for d in range(100)} == {1}


def test_top_p_bf16_threshold():
    """bf16 logits: probabilities and the cumulative sum are bf16, and `cum > top_p` compares with bf16(top_p) =
    0.80078125 — a prefix of 0.8005 is kept in bf16 and dropped in fp32."""
    p = torch.tensor([0.5, 0.3005, 0.1995, 0.0], dtype=torch.float64)
    logits = torch.log(p[:3]).float()
    pol = Policy(top_k=0, top_p=0.8, temperature=1.0)
    k32 = candidate_set_bf16(logits, pol)
    assert k32.tolist() == [True, False, False]
    xb = logits.to(torch.bfloat16)
    pb = torch.softmax(xb.float(), 0).to(torch.bfloat16)
    cum = torch.cumsum(pb, 0)
    want = (~(cum > 0.8)).tolist()
    want[0] = True
    assert candidate_set_bf16(xb, pol).tolist() == [w or i == 0 for i, w in enumerate(want)] == [True, True, False]
    r = replayer(xb, pol)
    assert set(r.sets[0][0].tolist()) == set(torch.nonzero(candidate_set_bf16(xb, pol)).reshape(-1).tolist())


def test_top_p_bf16_prefix_on_the_midpoint_rounds_to_even():
    """bf16 probabilities 0.5, 0.302734375, ...: the prefix 0.802734375 lies exactly on the midpoint between
    bf16(0.8) = 0.80078125 (odd mantissa) and 0.8046875, rounds to the even one, so `cum > 0.8` drops rank 1."""
    xb = torch.tensor([0.0, -0.5, -1.40625, -1.90625], dtype=torch.bfloat16)
    pb = torch.softmax(xb.float(), 0).to(torch.bfloat16)
    assert float(pb[0]) + float(pb[1]) == 0.802734375
    pol = Policy(top_k=0, top_p=0.8, temperature=1.0)
    assert candidate_set_bf16(xb, pol).tolist() == [True, False, False, False]
    r = replayer(xb, pol)
    assert r.sets[0][0].tolist() == [0]
    assert {r.draw(5, d) for d in range(64)} == {(0, False)}
    # under top_p = 0.9 the same prefix is kept
    assert candidate_set_bf16(xb, Policy(top_k=0, top_p=0.9, temperature=1.0)).tolist() == [True, True, False, False]


@pytest.mark.parametrize("top_p", [0.8, 0.95, 0.9, 0.5])
def test_replay_top_p_set_equals_candidate_set(top_p):
    """On 400 random rows (bf16 and fp32, top_k 0 and 50) the replay's nominal kept set is candidate_set_bf16."""
    g = torch.Generator().manual_seed(int(top_p * 100))
    for row in range(400):
        V = (3072, 2048, 257)[row % 3]
        dtype = torch.bfloat16 if row % 2 else torch.float32
        x = (3.0 * torch.randn(V, generator=g)).to(dtype)
        pol = Policy(top_k=50 if row % 4 < 2 else 0, top_p=top_p, temperature=0.9)
        cand = torch.nonzero(candidate_set_bf16(x, pol)).reshape(-1).tolist()
        assert replayer(x, pol).sets[0][0].tolist() == cand, (row, V, dtype)


@pytest.mark.parametrize("ci", range(12))
def test_golden_draws_lie_in_bf16_candidate_set(ci):
    """Every token the reference's sampling.py drew (tests/golden/sampling_golden.pt, bf16 cases included) lies in
    candidate_set_bf16, and the replay's kept set is that candidate set."""
    g = torch.load(GOLDEN, weights_only=False)
    case = g["cases"][ci]
    lg = case["logits"][0]
    V = lg.numel()
    for (k, p), drawn in case["drawn"].items():
        pol = Policy(top_k=k, top_p=p, temperature=0.9, suppress_tail=1024, eos=case["eos"])
        cand = candidate_set_bf16(lg, pol)
        assert cand.shape == (V,)
        assert bool(cand[drawn].all()), (ci, k, p)
        assert not bool(cand[case["smask"]].any())
        nominal = replayer(lg, pol).sets[0][0]
        assert set(nominal.tolist()) == set(torch.nonzero(cand).reshape(-1).tolist()), (ci, k, p)
    assert replay(lg, Policy(do_sample=False, suppress_tail=1024, eos=case["eos"], suppress_eos=True), None, 0, 0)[0] == \
        int(case["greedy"])
