"""Every draw of the engine's three samplers replayed against oracle/sampler_oracle.py (Philox + float64 restatement of
sampling.py): the stand-alone fq3_sample (`sample_row` on fp32 / bf16 logits), and the in-kernel `sample_fast` and
`sample_row` on LL words through the prefill, predictor and frame-loop entry points.

Pass rule of every configuration: each draw the oracle does not call ambiguous equals the replay and lies in the
reference's candidate set (`candidate_set_bf16` in the logits' dtype, on the CPU: see the oracle's docstring for why not on
CUDA); at most 10 % of the draws are ambiguous."""
import pytest
import torch

from helpers import make_cfg, make_engine, make_weights, synth_prompt
from oracle.sampler_oracle import Policy, candidate_set_bf16, replayer, stream_key, talker_draw

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

N_DRAWS = 256


def _sp(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    return SamplingPolicy(**kw)


def _sub(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SubPolicy
    return SubPolicy(**kw)


class Tally:
    """Draws, mismatches (non-ambiguous draws that differ from the replay), draws outside the candidate set, ambiguous."""

    def __init__(self, name):
        self.name, self.n, self.bad, self.out, self.amb, self.first = name, 0, 0, 0, 0, None

    def add(self, tok, rep, cand, where=None):
        t, amb = rep
        self.n += 1
        self.amb += amb
        if not amb and tok != t:
            self.bad += 1
            self.first = self.first or (where, tok, t)
        if not amb and not bool(cand[tok]):  # an ambiguous draw may sit on a boundary token either side keeps
            self.out += 1
            self.first = self.first or (where, tok, "outside the candidate set")

    def check(self):
        print(f"{self.name}: draws {self.n} mismatches {self.bad} outside {self.out} ambiguous {self.amb}")
        assert self.n >= N_DRAWS, self.name
        assert self.bad == 0 and self.out == 0, (self.name, self.bad, self.out, self.first)
        assert self.amb <= 0.1 * self.n, (self.name, self.amb, self.n)


def _policy(sp, V, eos=-1, suppress_eos=False):
    return Policy(do_sample=sp.do_sample, top_k=sp.top_k, top_p=sp.top_p, temperature=sp.temperature,
                  repetition_penalty=sp.repetition_penalty, suppress_tail=sp.suppress_tail, eos=eos, suppress_eos=suppress_eos)


# ------------------------------------------------------------------------------------------------
# a. stand-alone fq3_sample
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng1():
    cfg = make_cfg("tiny")
    eng = make_engine(cfg, make_weights(cfg, seed=0))
    yield eng
    eng.close()


def _designed(kind, V, g):
    if kind == "randn":
        return 3.0 * torch.randn(V, generator=g)
    if kind == "ties":  # bf16-exact values in a few large tie groups
        return torch.randint(-12, 5, (V,), generator=g).float() * 0.5
    if kind == "dominant":  # p(top) ~ 1 - 1e-7 after / T = 0.9
        x = torch.full((V,), -4.0)
        x[V // 3] = -4.0 + 0.9 * float(torch.log(torch.tensor(V / 1e-7)))
        return x
    if kind == "zeros":  # +0.0 and -0.0 in one tie group straddling the k-th value and the top-p boundary
        x = torch.full((V,), -10.0)
        x[:V // 2] = torch.randn(V // 2, generator=g) - 12.0
        zi = torch.randperm(V, generator=g)[:40]
        x[zi] = torch.where(torch.arange(40) % 2 == 0, torch.tensor(0.0), torch.tensor(-0.0))
        x[zi[0]] = 1.0
        return x
    if kind == "two":
        x = torch.full((V,), float("-inf"))
        x[V // 5], x[V - 2] = 1.0, 0.25
        return x
    raise ValueError(kind)


def _sweep(eng, name, logits, sp, history=None, eos=-1, suppress_eos=False, seed=0):
    """N_DRAWS draws of fq3_sample over draw indices seed*1000 + d, replayed."""
    V = logits.numel()
    lg = logits.cuda()
    hist = None if history is None else torch.tensor(history, dtype=torch.long)
    outs = [eng.sample(lg, hist, sp, eos_id=eos, suppress_eos=suppress_eos, draw_index=seed * 1000 + d) for d in range(N_DRAWS)]
    toks = torch.cat(outs).cpu().tolist()
    pol = _policy(sp, V, eos, suppress_eos)
    seen = None if history is None else history
    r = replayer(logits, pol, seen)
    cand = candidate_set_bf16(logits, pol, seen) if sp.do_sample else torch.nn.functional.one_hot(
        torch.tensor(r.greedy), V).bool()
    t = Tally(name)
    for d, tok in enumerate(toks):
        t.add(tok, r.draw(sp.seed, seed * 1000 + d), cand, d)
    t.check()
    return toks


TOPK_TOPP_T = [(0, 1.0, 0.9), (1, 1.0, 0.9), (5, 0.95, 3.0), (50, 1.0, 0.05), (50, 0.8, 0.9), ("V", 0.5, 0.9),
               ("V+", 0.95, 3.0), (0, 1e-3, 0.9), (0, 0.8, 0.05), (50, 0.95, 0.9)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("V", [3072, 2048, 257, 5120])
def test_fq3_sample_replay_matrix(eng1, V, dtype):
    g = torch.Generator().manual_seed(V)
    x = _designed("randn", V, g).to(dtype)
    for i, (k, p, T) in enumerate(TOPK_TOPP_T):
        k = V if k == "V" else V + 7 if k == "V+" else k
        sp = _sp(do_sample=True, top_k=k, top_p=p, temperature=T, repetition_penalty=1.0, suppress_tail=0, seed=1 + i)
        _sweep(eng1, f"V={V} {dtype} k={k} p={p} T={T}", x, sp, seed=i)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fq3_sample_replay_suppression_and_penalty(eng1, dtype):
    V, eos = 3072, 2172
    g = torch.Generator().manual_seed(5)
    x = _designed("randn", V, g).to(dtype)
    x[eos] = x.max()  # EOS would win when it is allowed
    hist = [7, 7, 19, 19, 19, eos, 3000, V + 5, 10**9, -1, -40, int(torch.argmax(x[:2000]))]
    for i, (pen, sup_eos, k, p) in enumerate([(1.05, False, 50, 1.0), (1.05, True, 0, 0.9), (0.9, False, 50, 0.8),
                                             (0.9, True, 5, 1.0), (1.0, False, 0, 0.95)]):
        sp = _sp(do_sample=True, top_k=k, top_p=p, temperature=0.9, repetition_penalty=pen, suppress_tail=1024, seed=40 + i)
        toks = _sweep(eng1, f"{dtype} suppress_tail 1024 eos={sup_eos} penalty {pen} k={k} p={p}", x, sp, hist, eos, sup_eos, seed=i)
        assert all(t < V - 1024 or (t == eos and not sup_eos) for t in toks)
    sp = _sp(do_sample=False, repetition_penalty=1.3, suppress_tail=1024)
    _sweep(eng1, f"{dtype} greedy penalty 1.3", x, sp, hist, eos, True)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kind", ["ties", "dominant", "zeros", "two"])
def test_fq3_sample_replay_designed_logits(eng1, kind, dtype):
    V = 3072
    g = torch.Generator().manual_seed(11)
    x = _designed(kind, V, g).to(dtype)
    xs = (x.float() / 0.9).to(dtype).float()
    srt = torch.sort(xs[torch.isfinite(xs)], descending=True).values
    ks = [0, 1, 50]
    if kind in ("ties", "zeros"):
        kth_in_group = int((srt > srt[20]).sum()) + 3  # k-th value inside the tie group of rank 20
        assert srt[kth_in_group - 1] == srt[kth_in_group], kind
        ks.append(kth_in_group)
    for i, k in enumerate(ks):
        for j, p in enumerate([1.0, 0.95, 0.8, 0.5]):
            sp = _sp(do_sample=True, top_k=k, top_p=p, temperature=0.9, repetition_penalty=1.0, suppress_tail=0, seed=100 + i)
            _sweep(eng1, f"{kind} {dtype} k={k} p={p}", x, sp, seed=10 * i + j)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fq3_sample_top_p_prefix_on_the_midpoint(eng1, dtype):
    """bf16 probabilities 0.5 + 0.302734375 = 0.802734375, exactly the midpoint above bf16(0.8) = 0.80078125, which rounds
    to the even 0.8046875 > bf16(0.8): sampling.py keeps rank 0 alone (fp32 logits: 0.8027 > 0.8 as well)."""
    V = 3072
    x = torch.full((V,), float("-inf"))
    x[[700, 11, 2900, 5]] = torch.tensor([0.0, -0.5, -1.40625, -1.90625])
    sp = _sp(do_sample=True, top_k=0, top_p=0.8, temperature=1.0, repetition_penalty=1.0, suppress_tail=0, seed=9)
    assert set(_sweep(eng1, f"midpoint {dtype}", x.to(dtype), sp)) == {700}


def test_fq3_sample_refuses_vocab_above_scratch(eng1):
    from qwen3_tts_cuda_graphs_b200._lib import Fq3Error
    with pytest.raises(Fq3Error, match="fq3 error 5"):
        eng1.sample(torch.randn(5121, device="cuda"), None, _sp(), eos_id=-1, suppress_eos=False)


# ------------------------------------------------------------------------------------------------
# b. in-kernel samplers through the prefill and predictor entry points, on weights with exact logit ties
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tied():
    """tiny preset; 200 rows of the codec head and of lm_head.3 zeroed (logits exactly 0) and a few rows duplicated."""
    cfg = make_cfg("tiny")
    w = make_weights(cfg, seed=0)
    g = torch.Generator().manual_seed(2)
    Vt, Vp = cfg.talker.vocab_size, cfg.predictor.vocab_size
    head = w["talker.codec_head.weight"]
    head[torch.randperm(Vt - 1024, generator=g)[:200]] = 0
    for a, b in [(10, 11), (500, 1500), (600, 601), (1700, 20)]:
        head[b] = head[a]
    lm = w["talker.code_predictor.lm_head.3.weight"]
    lm[torch.randperm(Vp, generator=g)[:200]] = 0
    for a, b in [(5, 6), (700, 1400)]:
        lm[b] = lm[a]
    eng = make_engine(cfg, w, max_streams=2)
    yield cfg, eng
    eng.close()


def _has_ties(lg):
    return int((lg == 0).sum()) >= 190 and int(torch.unique(lg).numel()) < lg.numel() - 190


@pytest.mark.parametrize("top_p", [1.0, 0.95, 0.8])
def test_prefill_first_token_replay(tied, top_p):
    """SMP_PREFILL draws index 0 with key seed ^ K (slot + 1), or seed ^ K with a policy record: dense and chunked paths,
    slot 0, slot 1 without a record, slot 1 with one; EOS suppressed (min_new_tokens > 0) or not; tail suppression; top_k
    50 and a top_k whose k-th value lies in the group of 200 exact zeros."""
    cfg, eng = tied
    V, eos = cfg.talker.vocab_size, cfg.talker.codec_eos_token_id
    tie, _, _, _ = synth_prompt(cfg, T=40)
    lg0 = eng.prefill(0, tie[0].cuda(), 0, _sp(do_sample=False), want_logits=True).cpu().to(torch.bfloat16)
    assert _has_ties(lg0[:V - 1024])
    xs = (lg0.float()[:V - 1024] / 0.9).to(torch.bfloat16).float()
    k_tie = int((xs > 0).sum()) + 50
    variants = [("dense slot0", 0, False, True), ("chunked slot0", 0, False, False), ("chunked slot1", 1, False, False),
                ("dense slot1 record", 1, True, True)]
    for name, slot, own, dense in variants:
        for mnt in (2, 0):
            t = Tally(f"prefill {name} top_p={top_p} min_new_tokens={mnt}")
            for s in range(N_DRAWS):
                sp = _sp(do_sample=True, top_k=50 if s % 2 else k_tie, top_p=top_p, temperature=0.9, repetition_penalty=1.3,
                         min_new_tokens=mnt, suppress_tail=1024, seed=1000 * slot + 7 * s + 3)
                if own:
                    eng.set_stream_policy(slot, sp)
                lg = eng.prefill(slot, tie[0].cuda(), 0, sp, want_logits=True, dense=dense).cpu().to(torch.bfloat16)
                tok = eng.status(slot).token
                pol = _policy(sp, V, eos, mnt > 0)
                rep = replayer(lg, pol).draw(stream_key(sp.seed, slot, own), 0)
                t.add(tok, rep, candidate_set_bf16(lg, pol), s)
            if own:
                eng.set_stream_policy(slot, None)
            t.check()


@pytest.mark.parametrize("top_p", [1.0, 0.9])
@pytest.mark.parametrize("top_k", [0, 1, 50])
def test_predictor_replay(tied, top_k, top_p):
    """fq3_predictor_run on a reset stream: codebook i draws index i + 1 with key seed ^ K, from the bf16 logits returned."""
    cfg, eng = tied
    Vp = cfg.predictor.vocab_size
    g = torch.Generator().manual_seed(3)
    x = (0.5 * torch.randn(1, 2, cfg.talker.hidden_size, generator=g)).to(torch.bfloat16).cuda()
    t = Tally(f"predictor top_k={top_k} top_p={top_p}")
    sub = _sub(do_sample=True, top_k=top_k, top_p=top_p, temperature=0.9)
    pol = Policy(top_k=top_k, top_p=top_p, temperature=0.9)
    for seed in range(N_DRAWS // 15 + 1):
        eng.reset_stream(0)
        codes, logits = eng.predictor_run(0, x, sub, seed=seed * 7919, want_logits=True)
        codes, logits = codes.cpu().tolist(), logits.cpu().to(torch.bfloat16)
        if seed == 0:
            assert _has_ties(logits[3])
        key = stream_key(seed * 7919, 0, False)
        for i in range(eng.ncb):
            t.add(codes[i], replayer(logits[i], pol).draw(key, i + 1), candidate_set_bf16(logits[i], pol), (seed, i))
    t.check()


# ------------------------------------------------------------------------------------------------
# c. the frame loop's talker sampler (repetition penalty bitmap, min_new_tokens by frame count, draw schedule)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("top_p", [1.0, 0.9])
def test_frame_loop_talker_replay(tied, top_p):
    cfg, eng = tied
    V, eos = cfg.talker.vocab_size, cfg.talker.codec_eos_token_id
    tie, _, tth, tpe = synth_prompt(cfg, T=20)
    t = Tally(f"frame loop talker top_p={top_p}")
    for seed in range(7):
        sp = _sp(do_sample=True, top_k=50, top_p=top_p, temperature=0.9, repetition_penalty=1.3, min_new_tokens=4,
                 suppress_tail=1024, seed=31 * seed + 5)
        sub = _sub(do_sample=True, top_k=50, temperature=0.9)
        key = stream_key(sp.seed, 0, False)
        eng.reset_stream(0)
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, sp)
        for f in range(40):
            eng.decode_frames(1, 1, sp, sub)
            lg = eng.debug_talker_logits(0).cpu().to(torch.bfloat16)
            st = eng.status(0)
            assert st.error == 0 and st.n_frames == f + 1
            codes = eng.read_codes(0, 0, f + 1)
            seen = codes[:f + 1, 0].tolist()
            pol = _policy(sp, V, eos, f + 1 < sp.min_new_tokens)
            t.add(st.token, replayer(lg, pol, seen).draw(key, talker_draw(f)),
                  candidate_set_bf16(lg, pol, seen), (seed, f))
            if st.done:
                break
    t.check()
    eng.prefill(0, tie[0].cuda(), 0, _sp(do_sample=False))
    with pytest.raises(Exception, match="fq3 error 1"):  # the hook refuses once another launch has used the logits rows
        eng.debug_talker_logits(0)
