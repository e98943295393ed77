"""GPU parity tests of the persistent weight-streaming engine against the CPU oracle (through the C ABI).

Tolerances (stated per BASELINE.json north_star):
  * bf16 activations / logits: max |a-b| <= 3e-2 * max|b|  (about 4 bf16 ulps at the top magnitude; the two
    sides round at the same points but accumulate in different orders);
  * greedy ids: identical to the oracle's argmax wherever the oracle's top-2 margin exceeds the logit
    tolerance (teacher-forced), identical run-to-run and chunking-to-chunking unconditionally.
"""
import pytest
import torch

from helpers import make_cfg, make_engine, make_oracle, make_weights, margin_argmax_agree, rel_err, synth_prompt

pytestmark = pytest.mark.gpu

TOL = 3e-2


def _sp(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    return SamplingPolicy(**kw)


def _sub(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SubPolicy
    return SubPolicy(**kw)


# ------------------------------------------------------------------------------------------------
# GEMV phase
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny():
    cfg = make_cfg("tiny")
    w = make_weights(cfg, seed=0)
    eng = make_engine(cfg, w)
    yield cfg, w, eng
    eng.close()


def _ref_linear(W, x, gamma, eps, bias, residual, swiglu):
    from oracle.qwen3_tts_oracle import rms_norm
    h = rms_norm(x, gamma, eps) if gamma is not None else x
    y = torch.nn.functional.linear(h.float(), W.float())
    if bias is not None:
        y = y + bias.float()
    y = y.to(torch.bfloat16)
    if swiglu:
        g, u = y[:, 0::2], y[:, 1::2]
        y = torch.nn.functional.silu(g) * u
    if residual is not None:
        y = residual + y
    return y


@pytest.mark.parametrize(
    "N,K,M,norm,bias,resid,swiglu",
    [
        (4096, 1024, 1, True, False, False, False),   # 0.6B talker fused qkv
        (1024, 2048, 1, False, False, True, False),   # o_proj + residual
        (6144, 1024, 1, True, False, False, True),    # gate/up + SiLU*mul
        (6144, 1024, 2, True, False, False, True),    # predictor pass 0 (two rows)
        (1024, 3072, 1, False, False, True, False),   # down + residual
        (3072, 1024, 1, True, False, False, False),   # codec_head
        (1024, 2048, 2, False, True, False, False),   # small_to_mtp (1.7B) with bias
        (2048, 6144, 4, False, False, True, False),   # 1.7B down, one row per tile, 8-way k split
        (8192, 2048, 3, True, False, False, False),   # 1.7B qkv, prefill rows
        (100, 128, 8, False, False, False, False),    # ragged: N not a multiple of anything, 16 chunks per row
        (6, 256, 5, True, True, True, False),         # fewer rows than CTAs
    ],
)
def test_linear_matches_torch(tiny, N, K, M, norm, bias, resid, swiglu):
    _, _, eng = tiny
    g = torch.Generator().manual_seed(N * 7 + K + M)
    W = (0.05 * torch.randn(N, K, generator=g)).to(torch.bfloat16).cuda()
    x = torch.randn(M, K, generator=g).to(torch.bfloat16).cuda()
    gamma = (1 + 0.1 * torch.randn(K, generator=g)).to(torch.bfloat16).cuda() if norm else None
    b = (0.1 * torch.randn(N, generator=g)).to(torch.bfloat16).cuda() if bias else None
    No = N // 2 if swiglu else N
    r = torch.randn(M, No, generator=g).to(torch.bfloat16).cuda() if resid else None
    y = eng.linear(W, x, gamma=gamma, eps=1e-6, bias=b, residual=r, swiglu=swiglu)
    torch.cuda.synchronize()
    ref = _ref_linear(W, x, gamma, 1e-6, b, r, swiglu)
    assert y.shape == ref.shape
    assert rel_err(y, ref) <= 1.0 / 64, rel_err(y, ref)
    # the bulk must be bit-identical bf16 (same rounding points); allow isolated 1-ulp flips
    frac_exact = (y == ref).float().mean().item()
    assert frac_exact > 0.9, frac_exact


def test_linear_f32_logits_are_bf16_rounded(tiny):
    _, _, eng = tiny
    g = torch.Generator().manual_seed(5)
    W = (0.05 * torch.randn(2048, 1024, generator=g)).to(torch.bfloat16).cuda()
    x = torch.randn(1, 1024, generator=g).to(torch.bfloat16).cuda()
    y = eng.linear(W, x, out_f32=True)
    torch.cuda.synchronize()
    assert y.dtype == torch.float32
    assert torch.equal(y, y.to(torch.bfloat16).float())
    ref = torch.nn.functional.linear(x.float(), W.float())
    assert rel_err(y, ref) <= 1.0 / 64


# ------------------------------------------------------------------------------------------------
# talker step / prefill / predictor against the oracle
# ------------------------------------------------------------------------------------------------
CONFIGS = [("tiny", None, None), ("0.6B-Base", 2, 2), ("1.7B-Base", 1, 1)]


@pytest.fixture(scope="module", params=CONFIGS, ids=[c[0] for c in CONFIGS])
def pair(request):
    name, tl, pl = request.param
    cfg = make_cfg(name, tl, pl)
    w = make_weights(cfg, seed=11)
    eng = make_engine(cfg, w, max_seq_len=272)
    orc = make_oracle(cfg, w)
    yield cfg, w, eng, orc
    eng.close()


def test_talker_step_matches_oracle(pair):
    cfg, w, eng, orc = pair
    tie, tam, tth, tpe = synth_prompt(cfg, T=14)
    logits0, past_hidden, T = orc.talker_prefill(tie, tam)
    eng.reset_stream(0)
    for l, (k, v) in enumerate(orc.talker.cache):
        eng.import_kv(0, l, k[0].cuda(), v[0].cuda())
    g = torch.Generator().manual_seed(3)
    for step in range(3):
        x = (0.05 * torch.randn(1, 1, cfg.talker.hidden_size, generator=g)).to(torch.bfloat16)
        ref_h = orc.talker_step(x, T + step)
        ref_l = orc.codec_head(ref_h[:, -1, :])[0]
        h, lg = eng.talker_step(0, x.cuda(), T + step)
        torch.cuda.synchronize()
        assert rel_err(h, ref_h) <= TOL, (step, rel_err(h, ref_h))
        assert rel_err(lg, ref_l) <= TOL, (step, rel_err(lg, ref_l))
        assert margin_argmax_agree(lg, ref_l, TOL * float(ref_l.float().abs().max()))


@pytest.mark.parametrize("T", [1, 14, 37])
def test_prefill_matches_oracle(pair, T):
    cfg, w, eng, orc = pair
    tie, tam, tth, tpe = synth_prompt(cfg, T=T, seed=T)
    ref_logits, ref_hidden, _ = orc.talker_prefill(tie, tam)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    lg = eng.prefill(0, tie[0].cuda(), 0, _sp(do_sample=False, repetition_penalty=1.0), want_logits=True)
    st = eng.status(0)
    assert st.position == T and st.n_frames == 0 and st.error == 0
    assert rel_err(lg, ref_logits[0]) <= TOL, rel_err(lg, ref_logits[0])
    # first token = argmax with the tail and EOS suppressed (generate.py:124-134)
    x = ref_logits[0].float().clone()
    x[cfg.talker.vocab_size - 1024:] = float("-inf")
    assert margin_argmax_agree(lg.masked_fill(torch.arange(lg.numel(), device=lg.device) >= cfg.talker.vocab_size - 1024, float("-inf")),
                               x, TOL * float(ref_logits.float().abs().max()))
    # the KV written in place must serve the next decode step
    xg = (0.05 * torch.randn(1, 1, cfg.talker.hidden_size, generator=torch.Generator().manual_seed(9))).to(torch.bfloat16)
    ref_h = orc.talker_step(xg, T)
    h, _ = eng.talker_step(0, xg.cuda(), T)
    torch.cuda.synchronize()
    assert rel_err(h, ref_h) <= TOL, rel_err(h, ref_h)


def test_prefill_with_left_padding_matches_unpadded(pair):
    cfg, w, eng, orc = pair
    tie, tam, tth, tpe = synth_prompt(cfg, T=11, seed=4)
    pol = _sp(do_sample=False, repetition_penalty=1.0)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    a = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True).clone()
    pad = torch.zeros(5, cfg.talker.hidden_size, dtype=torch.bfloat16)
    b = eng.prefill(0, torch.cat([pad, tie[0]]).cuda(), 5, pol, want_logits=True).clone()
    torch.cuda.synchronize()
    # left pads are masked and rope positions shifted by -n_pad (talker_graph.py:172-196): same logits
    assert rel_err(b, a) <= 1e-2, rel_err(b, a)


def test_predictor_matches_oracle_teacher_forced(pair):
    cfg, w, eng, orc = pair
    g = torch.Generator().manual_seed(21)
    x = (0.5 * torch.randn(1, 2, cfg.talker.hidden_size, generator=g)).to(torch.bfloat16)
    codes, logits = eng.predictor_run(0, x.cuda(), _sub(do_sample=False), want_logits=True)
    torch.cuda.synchronize()
    orc.sub.do_sample = False
    ref_codes, ref_logits = orc.predictor_loop(x, forced=codes.cpu())
    scale = max(float(r.abs().max()) for r in ref_logits)
    for i in range(orc.ncb):
        assert rel_err(logits[i], ref_logits[i]) <= TOL, (i, rel_err(logits[i], ref_logits[i]))
        assert margin_argmax_agree(logits[i], ref_logits[i], TOL * scale), i
        assert int(codes[i]) == int(logits[i].argmax()), i  # greedy = lowest-index argmax of its own logits
    assert codes.min() >= 0 and codes.max() < cfg.predictor.vocab_size


def test_frame_loop_teacher_forced_against_oracle(pair):
    """Every id the device loop emits must be the oracle's greedy choice at that step, up to bf16 near-ties."""
    cfg, w, eng, orc = pair
    _frame_loop_teacher_forced(cfg, eng, orc, T=14, n=10)


def _frame_loop_teacher_forced(cfg, eng, orc, T, n):
    tie, tam, tth, tpe = synth_prompt(cfg, T=T, R=3)
    pol = _sp(do_sample=False, repetition_penalty=1.05, min_new_tokens=2)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    eng.prefill(0, tie[0].cuda(), 0, pol)
    tok0 = eng.status(0).token
    eng.decode_frames(1, n, pol, _sub(do_sample=False))
    st = eng.status(0)
    assert st.error == 0 and st.n_frames == n and st.position == T + n and st.gen_step == n
    codes = eng.read_codes(0, 0, n)
    assert codes[0, 0] == tok0
    orc.sub.do_sample = False
    trace = {}
    frames = list(orc.generate_frames(tie, tam, tth, tpe, max_new_tokens=n, min_new_tokens=2, do_sample=False,
                                      repetition_penalty=1.05, max_seq_len=eng.max_seq_len, trace=trace, forced=codes))
    assert len(frames) == n
    bad = []
    tscale = float(trace["prefill_logits"].abs().max())
    for i in range(n):
        nxt = int(codes[i + 1, 0]) if i + 1 < n else st.token
        fin = trace["talker_final"][i]
        if float(fin.max() - fin[nxt]) > TOL * tscale:
            bad.append(("talker", i, nxt, int(fin.argmax())))
        pl = trace["pred_logits"][i]
        pscale = float(pl.abs().max())
        for c in range(orc.ncb):
            if float(pl[c].max() - pl[c][int(codes[i, c + 1])]) > TOL * pscale:
                bad.append(("pred", i, c))
    assert not bad, bad
    # structural invariants the reference asserts on real checkpoints (tests/test_e2e_parity.py:40-101)
    assert codes.shape == (n, 16) and codes.min() >= 0
    assert (codes[:, 0] < cfg.talker.vocab_size - 1024).all()
    assert (codes[:, 0] != cfg.talker.codec_eos_token_id).all()
    assert (codes[:, 1:] < cfg.predictor.vocab_size).all()


def test_left_padded_prompt_and_frames_against_oracle(pair):
    """Left-padded prompt (the batched layout of model.py:519-551: zero rows in front, attention mask 0 there, rope positions
    shifted by -n_pad: talker_graph.py:172-196) through prefill AND the frame loop, against the oracle run on the same padded
    input with the same mask — the padding path checked against the reference's semantics, not only against the unpadded run."""
    cfg, w, eng, orc = pair
    tie, tam, tth, tpe = synth_prompt(cfg, T=12, R=2, seed=6)
    n_pad, n = 4, 6
    H = cfg.talker.hidden_size
    tie_p = torch.cat([torch.zeros(1, n_pad, H, dtype=torch.bfloat16), tie], dim=1)
    tam_p = torch.cat([torch.zeros(1, n_pad, dtype=torch.long), tam], dim=1)
    pol = _sp(do_sample=False, repetition_penalty=1.05, min_new_tokens=2)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    logits = eng.prefill(0, tie_p[0].cuda(), n_pad, pol, want_logits=True).clone()
    ref_logits, _, plen = orc.talker_prefill(tie_p, tam_p)
    assert plen == 12 + n_pad
    assert rel_err(logits, ref_logits[0]) <= TOL, rel_err(logits, ref_logits[0])
    eng.decode_frames(1, n, pol, _sub(do_sample=False))
    st = eng.status(0)
    assert st.error == 0 and st.n_frames == n and st.position == 12 + n_pad + n
    codes = eng.read_codes(0, 0, n)
    orc.sub.do_sample = False
    trace = {}
    frames = list(orc.generate_frames(tie_p, tam_p, tth, tpe, max_new_tokens=n, min_new_tokens=2, do_sample=False,
                                      repetition_penalty=1.05, max_seq_len=272, trace=trace, forced=codes))
    assert len(frames) == n
    tscale = float(trace["prefill_logits"].abs().max())
    bad = []
    for i in range(n):
        nxt = int(codes[i + 1, 0]) if i + 1 < n else st.token
        fin = trace["talker_final"][i]
        if float(fin.max() - fin[nxt]) > TOL * tscale:
            bad.append(("talker", i, nxt, int(fin.argmax())))
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# loop control: determinism, chunking, EOS / min_new_tokens, cache bound
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sample", [False, True])
def test_streaming_chunks_equal_one_launch(tiny, sample):
    """tests/test_e2e_parity.py:726-780 — streaming == non-streaming token for token (chunk_size=8)."""
    cfg, w, eng = tiny
    tie, tam, tth, tpe = synth_prompt(cfg, T=14, R=2)
    pol = _sp(do_sample=sample, seed=1234)
    sub = _sub(do_sample=sample)

    def run(chunks):
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, pol)
        for c in chunks:
            eng.decode_frames(1, c, pol, sub)
            assert eng.status(0).error == 0
        n = eng.status(0).n_frames
        return eng.read_codes(0, 0, n)

    a = run([24])
    b = run([8, 8, 8])
    c = run([5, 7, 12])
    assert a.shape[0] == 24
    assert torch.equal(a, b) and torch.equal(a, c)
    assert torch.equal(a, run([24]))  # run-to-run deterministic


def test_min_new_tokens_suppresses_early_eos():
    """tests/test_sampling.py:24-118 restated on the device loop: EOS is the greedy choice from the start, but
    it may only be taken once min_new_tokens frames exist; it never appears in the output."""
    from dataclasses import replace
    cfg = make_cfg("tiny")
    cfg = replace(cfg, talker=replace(cfg.talker, codec_eos_token_id=0))
    w = make_weights(cfg, seed=2)
    w["talker.codec_head.weight"].zero_()  # all logits tie at 0 -> lowest index (= EOS) wins unless suppressed
    eng = make_engine(cfg, w)
    tie, tam, tth, tpe = synth_prompt(cfg, T=3)
    for mn, expect in [(2, 2), (5, 5), (0, 0)]:
        pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=mn)
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, pol)
        eng.decode_frames(1, 16, pol, _sub(do_sample=False))
        st = eng.status(0)
        assert st.error == 0
        assert st.n_frames == expect, (mn, st.n_frames)
        codes = eng.read_codes(0, 0, st.n_frames)
        assert (codes[:, 0] != 0).all()
        assert st.done == 1
    eng.close()


def test_static_cache_bound_stops_silently():
    """generate.py:174-177 — the frame that hits max_seq_len-1 is kept, then decoding stops without error."""
    cfg = make_cfg("tiny")
    w = make_weights(cfg, seed=6)
    eng = make_engine(cfg, w, max_seq_len=24)
    orc = make_oracle(cfg, w)
    tie, tam, tth, tpe = synth_prompt(cfg, T=14)
    pol = _sp(do_sample=False, repetition_penalty=1.0)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    eng.prefill(0, tie[0].cuda(), 0, pol)
    eng.decode_frames(1, 64, pol, _sub(do_sample=False))
    st = eng.status(0)
    orc.sub.do_sample = False
    ref, _ = orc.fast_generate(tie, tam, tth, tpe, max_new_tokens=64, do_sample=False, repetition_penalty=1.0, max_seq_len=24)
    assert st.error == 0 and st.done == 2
    assert st.n_frames == ref.shape[0] == 24 - 14
    with pytest.raises(RuntimeError, match="Input is too long"):
        eng.prefill(0, torch.zeros(25, cfg.talker.hidden_size, dtype=torch.bfloat16).cuda(), 0, pol)
    eng.close()


def test_two_streams_match_single_stream(tiny):
    """Request-parallel lock-step decode: each stream's ids equal its single-stream run."""
    cfg, w, _ = tiny
    eng = make_engine(cfg, w, max_streams=2)
    pol = _sp(do_sample=False, repetition_penalty=1.05)
    sub = _sub(do_sample=False)
    prompts = [synth_prompt(cfg, T=14, seed=1), synth_prompt(cfg, T=9, seed=2)]
    singles = []
    for tie, tam, tth, tpe in prompts:
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, pol)
        eng.decode_frames(1, 12, pol, sub)
        singles.append(eng.read_codes(0, 0, eng.status(0).n_frames))
    for i, (tie, tam, tth, tpe) in enumerate(prompts):
        eng.set_text_conditioning(i, tth[0].cuda(), tpe.cuda())
        eng.prefill(i, tie[0].cuda(), 0, pol)
    eng.decode_frames(2, 12, pol, sub)
    for i in range(2):
        st = eng.status(i)
        assert st.error == 0 and st.n_frames == 12
        assert torch.equal(eng.read_codes(i, 0, 12), singles[i]), i
    eng.close()


def _batch_vs_single(cfg, w, n_streams, n_frames, lens, max_seq_len=256):
    """Every stream of a lock-step batch must produce exactly the ids of its own single-stream run (greedy + repetition
    penalty): the wide frame program splits predictor pass 0 in two and stages up to 16 rows, none of which may change a
    stream's arithmetic."""
    eng = make_engine(cfg, w, max_streams=n_streams, max_seq_len=max_seq_len)
    pol = _sp(do_sample=False, repetition_penalty=1.05)
    sub = _sub(do_sample=False)
    prompts = [synth_prompt(cfg, T=lens[i % len(lens)], seed=10 + i) for i in range(n_streams)]
    singles = []
    for tie, tam, tth, tpe in prompts:
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, pol)
        eng.decode_frames(1, n_frames, pol, sub)
        singles.append(eng.read_codes(0, 0, eng.status(0).n_frames))
    for i, (tie, tam, tth, tpe) in enumerate(prompts):
        eng.set_text_conditioning(i, tth[0].cuda(), tpe.cuda())
        eng.prefill(i, tie[0].cuda(), 0, pol)
    # two launches: the second one starts from the state the first one left on the device
    eng.decode_frames(n_streams, n_frames // 2, pol, sub)
    eng.decode_frames(n_streams, n_frames - n_frames // 2, pol, sub)
    bad = []
    for i in range(n_streams):
        st = eng.status(i)
        assert st.error == 0
        got = eng.read_codes(i, 0, st.n_frames)
        if st.n_frames != singles[i].shape[0] or not torch.equal(got, singles[i]):
            bad.append(i)
    group = eng.lockstep_group
    eng.close()
    assert not bad, (bad, group)


@pytest.mark.parametrize("n_streams", [3, 4, 5, 8, 16])
def test_wide_streams_match_single_stream_tiny(tiny, n_streams):
    cfg, w, _ = tiny
    _batch_vs_single(cfg, w, n_streams, 10, lens=[14, 9, 21, 5])


def test_wide_groups_match_single_stream_tiny(tiny):
    """More streams than one lock-step group holds: groups of 16 follow each other (40 streams -> 14 + 13 + 13)."""
    cfg, w, _ = tiny
    _batch_vs_single(cfg, w, 40, 6, lens=[14, 9, 21, 5, 30])


def test_wide_streams_match_single_stream_real_dims():
    """0.6B dims (k-parts in shared memory, 3072-column rows, split attention off), two layers each, 16 streams, contexts on both
    sides of the 48-position short-range attention path."""
    cfg = make_cfg("0.6B-Base", 2, 2)
    w = make_weights(cfg, seed=0)
    _batch_vs_single(cfg, w, 16, 8, lens=[14, 60, 37, 101])


def test_wide_streams_match_single_stream_past_768():
    """0.6B dims, two layers, 16 streams with contexts on both sides of 768 positions: past 768 a split holds more than 48
    positions (the long-range path) and the wide program's attention leaves its one-item-per-stream path for the generic walk,
    which mixes the short streams' items with the long streams' split items in one launch."""
    cfg = make_cfg("0.6B-Base", 2, 2)
    w = make_weights(cfg, seed=0)
    _batch_vs_single(cfg, w, 16, 4, lens=[700, 768, 769, 1500], max_seq_len=2048)


def test_wide_streams_match_single_stream_full_depth():
    """The real 0.6B stack at full depth (28 + 5 layers), 16 streams with contexts from 14 to 201 positions (one to five KV
    splits): 8 frames of every stream equal its single-stream run."""
    cfg = make_cfg("0.6B-Base")
    w = make_weights(cfg, seed=0)
    _batch_vs_single(cfg, w, 16, 8, lens=[14, 60, 137, 201])


def test_normal_program_after_wide_program(tiny):
    """The two frame programs keep the predictor's cross-launch rows in different layouts; the host converts between them."""
    cfg, w, _ = tiny
    eng = make_engine(cfg, w, max_streams=6)
    pol = _sp(do_sample=False, repetition_penalty=1.05)
    sub = _sub(do_sample=False)
    prompts = [synth_prompt(cfg, T=8 + i, seed=30 + i) for i in range(6)]
    ref = []
    for tie, tam, tth, tpe in prompts[:2]:
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        eng.prefill(0, tie[0].cuda(), 0, pol)
        eng.decode_frames(1, 9, pol, sub)
        ref.append(eng.read_codes(0, 0, 9))
    for i, (tie, tam, tth, tpe) in enumerate(prompts):
        eng.set_text_conditioning(i, tth[0].cuda(), tpe.cuda())
        eng.prefill(i, tie[0].cuda(), 0, pol)
    eng.decode_frames(6, 3, pol, sub)   # wide
    eng.decode_frames(2, 3, pol, sub)   # reference-shaped program on streams 0, 1
    eng.decode_frames(6, 3, pol, sub)   # wide again (streams 2-5 are three frames behind)
    for i in range(2):
        assert eng.status(i).n_frames == 9
        assert torch.equal(eng.read_codes(i, 0, 9), ref[i]), i
    eng.close()


# ------------------------------------------------------------------------------------------------
# in-kernel samplers (sampling.py:32-66 semantics inside the persistent kernel)
# ------------------------------------------------------------------------------------------------
def _bf16_div(x, t):
    return (x.to(torch.bfloat16) / t).float()  # the reference divides a bf16 tensor: the quotient is rounded to bf16


def test_predictor_sampler_draws_from_reference_candidate_set(tiny):
    """Every code the in-kernel predictor sampler draws must be one sample_logits could draw from the same logits
    (top-k support with ties, sampling.py:54-56), for several seeds; greedy must be the lowest-index argmax."""
    from oracle.qwen3_tts_oracle import candidate_set
    cfg, w, eng = tiny
    g = torch.Generator().manual_seed(3)
    x = (0.5 * torch.randn(1, 2, cfg.talker.hidden_size, generator=g)).to(torch.bfloat16).cuda()
    seen_codes = set()
    for seed in range(6):
        for k in (50, 5, 1):
            codes, logits = eng.predictor_run(0, x, _sub(do_sample=True, top_k=k, temperature=0.9), seed=seed, want_logits=True)
            torch.cuda.synchronize()
            for i in range(eng.ncb):
                lg = logits[i].cpu().to(torch.bfloat16)
                cand = candidate_set(_bf16_div(lg, 0.9).unsqueeze(0), temperature=1.0, top_k=k, top_p=1.0)[0]
                assert bool(cand[int(codes[i])]), (seed, k, i, int(codes[i]))
                if k == 1:  # only the maximum survives (bf16 ties at the maximum all do, sampling.py:54-56)
                    scaled = _bf16_div(lg, 0.9)
                    assert float(scaled[int(codes[i])]) == float(scaled.max()), (seed, i)
            seen_codes.add(tuple(int(c) for c in codes))
    assert len(seen_codes) > 3  # different seeds / k really draw different codes


def test_first_token_sampler_respects_suppression_and_top_k(tiny):
    """SMP_PREFILL: suppress tail (except EOS), EOS while min_new_tokens > 0, temperature, top-k (generate.py:124-134)."""
    from oracle.qwen3_tts_oracle import candidate_set
    cfg, w, eng = tiny
    tie, tam, tth, tpe = synth_prompt(cfg, T=9)
    V = cfg.talker.vocab_size
    eos = cfg.talker.codec_eos_token_id
    smask = torch.zeros(V, dtype=torch.bool)
    smask[V - 1024:] = True
    smask[eos] = False
    drawn = set()
    for seed in range(8):
        pol = _sp(do_sample=True, top_k=20, temperature=0.8, repetition_penalty=1.0, min_new_tokens=2, seed=seed)
        lg = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True)
        torch.cuda.synchronize()
        tok = eng.status(0).token
        cand = candidate_set(_bf16_div(lg.cpu(), 0.8).unsqueeze(0), temperature=1.0, top_k=20, top_p=1.0, suppress_mask=smask,
                             suppress_tokens=[eos])[0]
        assert bool(cand[tok]), (seed, tok)
        assert tok < V - 1024 and tok != eos
        drawn.add(tok)
    assert len(drawn) > 1
    pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=2)
    lg = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True)
    torch.cuda.synchronize()
    ref = lg.cpu().clone()
    ref[smask] = float("-inf")
    ref[eos] = float("-inf")
    assert eng.status(0).token == int(ref.argmax())


# ------------------------------------------------------------------------------------------------
# dense (tcgen05) prefill against the chunked decode-kernel prefill
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [17, 40, 130, 240, 2047])
def test_dense_prefill_matches_chunked_prefill(pair, T, monkeypatch, request):
    """The tensor-core prefill must give the logits and the first token of the all-decode-kernel prefill, and the K/V it wrote
    must serve the next decode step (hidden state vs the oracle) — in both of its forms: all T rows through all layers +
    fq3_prefill_head (default), and rows [0, T-1) + the last row through the decode kernel (fq3_prefill_tail, FQ3_DENSE_FULL=0).
    T = 2047 (fq3c_attn_prefill_kernel takes M <= 2048) runs on the tiny preset's 2048-position engine."""
    cfg, w, eng, orc = pair
    if T >= eng.max_seq_len:
        if cfg.talker.num_key_value_heads != 2:
            pytest.skip("prompt longer than this fixture's cache")
        cfg, w, eng, orc = request.getfixturevalue("long_pair")
    tie, tam, tth, tpe = synth_prompt(cfg, T=T, seed=5)
    pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=2)
    xg = (0.05 * torch.randn(1, 1, cfg.talker.hidden_size, generator=torch.Generator().manual_seed(9))).to(torch.bfloat16)
    out = {}
    for mode in ("chunked", "full", "tail"):
        if mode != "chunked":
            monkeypatch.setenv("FQ3_DENSE_FULL", "1" if mode == "full" else "0")
            if eng._dense is not None:
                eng._dense.close()
            eng._dense, eng._dense_tried = None, False  # rebuilt under the new setting
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        lg = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True, dense=(mode != "chunked"))
        st = eng.status(0)
        assert st.position == T and st.error == 0
        if mode != "chunked":
            assert eng._dense is not None and eng._dense.full == (mode == "full")
        h, _ = eng.talker_step(0, xg.cuda(), T)
        torch.cuda.synchronize()
        out[mode] = (lg.cpu(), st.token, h.cpu())
    ref_logits, _, _ = orc.talker_prefill(tie, tam)
    ref_h = orc.talker_step(xg, T)
    scale = float(ref_logits.float().abs().max())
    for mode in ("full", "tail"):
        assert rel_err(out[mode][0], out["chunked"][0]) <= TOL, mode
        assert rel_err(out[mode][0], ref_logits[0]) <= TOL, mode
        assert margin_argmax_agree(out[mode][0], out["chunked"][0], TOL * scale), mode
        assert rel_err(out[mode][2], ref_h) <= TOL, (mode, rel_err(out[mode][2], ref_h))
        assert rel_err(out[mode][2], out["chunked"][2]) <= TOL, mode
    monkeypatch.delenv("FQ3_DENSE_FULL")
    eng._dense.close()
    eng._dense, eng._dense_tried = None, False


@pytest.mark.parametrize("T", [40, 240])
def test_dense_prefill_fused_row_norm_is_bit_identical(pair, T, monkeypatch):
    """fq3c_op.norm_out: the RMSNorm behind an o / down projection runs inside the split-K reduction (or as one small launch)
    with the arithmetic of the stand-alone op — logits, first token and the next step's hidden state do not change by a bit,
    the op list loses two launches per layer."""
    cfg, w, eng, orc = pair
    if T >= eng.max_seq_len:
        pytest.skip("prompt longer than this fixture's cache")
    tie, tam, tth, tpe = synth_prompt(cfg, T=T, seed=6)
    pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=2)
    xg = (0.05 * torch.randn(1, 1, cfg.talker.hidden_size, generator=torch.Generator().manual_seed(10))).to(torch.bfloat16)
    out, n_ops = {}, {}
    for fuse in ("1", "0"):
        monkeypatch.setenv("FQ3C_FUSE_NORM", fuse)
        if eng._dense is not None:
            eng._dense.close()
        eng._dense, eng._dense_tried = None, False
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        lg = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True, dense=True)
        tok = eng.status(0).token
        h, _ = eng.talker_step(0, xg.cuda(), T)
        torch.cuda.synchronize()
        out[fuse], n_ops[fuse] = (lg.cpu(), tok, h.cpu()), len(eng._dense.ops)
    assert n_ops["0"] - n_ops["1"] == 2 * cfg.talker.num_hidden_layers - 1  # every norm but the first rides on a GEMM
    assert torch.equal(out["1"][0], out["0"][0]) and out["1"][1] == out["0"][1] and torch.equal(out["1"][2], out["0"][2])
    monkeypatch.delenv("FQ3C_FUSE_NORM")
    eng._dense.close()
    eng._dense, eng._dense_tried = None, False


# ------------------------------------------------------------------------------------------------
# long contexts: split-KV attention (48 positions per CTA) with the combine step, up to 16 splits; beyond 768 positions a
# split holds more than 48 (the half-warp online-softmax path)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def long_pair():
    name, tl, pl = CONFIGS[0]
    cfg = make_cfg(name, tl, pl)
    w = make_weights(cfg, seed=13)
    eng = make_engine(cfg, w, max_seq_len=2048)
    orc = make_oracle(cfg, w)
    yield cfg, w, eng, orc
    eng.close()


@pytest.mark.parametrize("T", [49, 97, 150, 192, 193, 300, 470, 760, 767, 768, 1200, 2046])
def test_talker_step_long_context_matches_oracle(long_pair, T):
    """A decode step at position T attends to T+1 positions: one CTA per (kv head, split) and the combine step of split 0, for
    2 to 16 splits (four combine rounds), splits of more than 48 positions from T = 768 on.  Hidden state and the prefill logits
    against the oracle."""
    cfg, w, eng, orc = long_pair
    tie, tam, tth, tpe = synth_prompt(cfg, T=T, seed=100 + T)
    pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=2)
    ref_logits, _, _ = orc.talker_prefill(tie, tam)
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
    lg = eng.prefill(0, tie[0].cuda(), 0, pol, want_logits=True, dense=False)
    assert eng.status(0).error == 0
    assert rel_err(lg, ref_logits[0]) <= TOL, rel_err(lg, ref_logits[0])
    g = torch.Generator().manual_seed(T)
    for step in range(2):
        xg = (0.05 * torch.randn(1, 1, cfg.talker.hidden_size, generator=g)).to(torch.bfloat16)
        ref_h = orc.talker_step(xg, T + step)
        h, _ = eng.talker_step(0, xg.cuda(), T + step)
        torch.cuda.synchronize()
        assert eng.status(0).error == 0
        assert rel_err(h, ref_h) <= TOL, (step, rel_err(h, ref_h))


def test_frame_loop_teacher_forced_across_768(long_pair):
    """A 760-row prompt and 16 greedy frames: the talker's context runs from 761 to 776 positions, so the frame loop moves from
    the two-pass split path to the long-range path mid-stream."""
    cfg, w, eng, orc = long_pair
    _frame_loop_teacher_forced(cfg, eng, orc, T=760, n=16)
