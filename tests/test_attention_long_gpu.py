"""The talker's decode attention alone, against float64, across the whole 2048-position cache.

The attention phase of the persistent kernel picks its code path from the context length L = pos + 1 - n_pad (positions
attended) and the grid: nsplit = min(ceil(L / 48), cap) splits with cap = min(G // n_kv_heads, 16).  Up to 48 * cap
positions (768 for every shipped shape at the default grid) every split takes the two-pass short path; beyond that a split
holds more than 48 positions and takes the half-warp online-softmax path with its per-warp merge.  Each way the kernel groups
the work is driven here: one talker step (cross-CTA splits + combine), the reference-shaped frame program with 1, 2 and 4
streams (generic two-pass walk), the wide frame program with 16 streams (one item per stream and kv head, or the generic walk
mixing those items with long split items), and chunked prefill rows on top of an imported cache.

Reference: the device's own raw q|k|v projection row of the last talker layer (fq3_debug_read_talker_attn) and its cache rows
[n_pad, pos] read after the launch.  q is restated with the kernel's rounding points (oracle rms_norm, bf16 rope at
pos + rope_delta), then softmax(q K^T / sqrt(128)) V per q head in float64.

Bound, per element: |attn - ref| <= ulp_bf16(|ref|) + 2^-12 * sum_i p_i |v_i|.  The device keeps scores, softmax and the
weighted sum in fp32 and rounds once to bf16 (half an ulp); the floor covers fp32 accumulation against cancellation and the
rare 1-ulp flip of a restated q element.

Inputs are built so that a position dropped, counted twice or given to the wrong split moves the output by many ulps: K is
scaled so the scores spread over several units, V is 16x larger at the marker positions (n_pad, pos - 1 and the first and
last position of every split), and the left-pad positions hold V = +-1000.
"""
import ctypes as C
import math

import pytest
import torch

from helpers import make_cfg, make_engine, make_weights, synth_prompt

pytestmark = pytest.mark.gpu

D = 128
SPLIT = 48       # positions per split of the two-pass path (kAttnShort)
MAX_SPLITS = 16  # kMaxSplits
MAX_SEQ = 2048
K_SCALE = 1.5    # score spread: q is RMS-normalised, so a score is ~ N(0, K_SCALE^2)
MARK = 16.0

LENGTHS = [1, 2, 47, 48, 49, 97, 480, 481, 720, 721, 767, 768, 769, 770, 1023, 1024, 1537, 2047, 2048]
PADDED = [(49, 5), (769, 5), (1024, 300), (1537, 300), (2, 300)]  # (L, n_pad)


def _sp(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    return SamplingPolicy(**kw)


def _sub(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SubPolicy
    return SubPolicy(**kw)


class _DeviceArray:
    """Zero-copy view of device memory for torch.as_tensor (int16 storage, reinterpreted as bf16 by the caller)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i2", "data": (int(ptr), False), "version": 3}


def cache(eng, idx, layer):
    """(K, V) bf16 [n_kv_heads, max_seq_len, 128] of one layer of one stream, aliasing the engine's static cache."""
    t = eng.cfg.talker
    out = []
    for which in (0, 1):
        ptr = eng.lib.fq3_kv_cache_ptr(eng.h, idx, layer, which)
        assert ptr
        out.append(torch.as_tensor(_DeviceArray(ptr, (t.num_key_value_heads, eng.max_seq_len, D))).view(torch.bfloat16))
    return out


def cap_of(eng):
    G = eng.reduced_grid() or eng.num_sms
    return max(1, min(G // eng.cfg.talker.num_key_value_heads, MAX_SPLITS))


def splits(L, n_pad, cap):
    """[a, b) of every split of a row at position n_pad + L - 1 (kernel: num_splits, attn_row)."""
    nsplit = max(1, min(-(-L // SPLIT), cap))
    per = -(-L // nsplit)
    pos = n_pad + L - 1
    return [(n_pad + s * per, min(n_pad + (s + 1) * per, pos + 1)) for s in range(nsplit)]


def markers(L, n_pad, cap):
    m = {n_pad, n_pad + L - 2}
    for a, b in splits(L, n_pad, cap):
        m |= {a, b - 1}
    return sorted(i for i in m if n_pad <= i < n_pad + L - 1)  # cached positions only: the row at pos is the device's


def import_state(eng, idx, L, n_pad, seed, cap):
    """Cache rows [0, pos) of every layer with the sensitivity pattern above; the stream's n_pad / rope_delta."""
    t = eng.cfg.talker
    pos = n_pad + L - 1
    g = torch.Generator(device=eng.device).manual_seed(seed)
    mk = markers(L, n_pad, cap)
    for layer in range(t.num_hidden_layers):
        k = K_SCALE * torch.randn(t.num_key_value_heads, pos, D, generator=g, device=eng.device)
        v = torch.randn(t.num_key_value_heads, pos, D, generator=g, device=eng.device)
        if mk:
            v[:, mk] *= MARK
        if n_pad:
            v[:, :n_pad] = 1000.0 * torch.sign(torch.randn(t.num_key_value_heads, n_pad, D, generator=g, device=eng.device))
        eng.import_kv(idx, layer, k.to(torch.bfloat16), v.to(torch.bfloat16))
    eng.set_generation_state(idx, n_pad, -n_pad)
    return pos


def norm_rope(x, gamma, pos, t):
    """head_norm_rope with the kernel's rounding points (fq3_kernel.cuh head_norm_rope): bf16 [n, 128] -> bf16 [n, 128]."""
    from oracle.qwen3_tts_oracle import rms_norm, rope_cos_sin, rotate_half
    y = rms_norm(x.cpu(), gamma, t.rms_norm_eps)
    cos, sin = rope_cos_sin(torch.tensor([pos]), D, t.rope_theta, torch.bfloat16)
    return (y * cos) + (rotate_half(y) * sin)


def reference(w, t, qkv, K, V, pos, n_pad, rope_delta):
    """float64 attention of one row: (out [nq, 128], floor [nq, 128], expected K row [nkv, 128] bf16, raw V row)."""
    nq, nkv = t.num_attention_heads, t.num_key_value_heads
    last = t.num_hidden_layers - 1
    pre = f"talker.model.layers.{last}.self_attn"
    qkv = qkv.cpu()
    q = norm_rope(qkv[: nq * D].view(nq, D), w[f"{pre}.q_norm.weight"], pos + rope_delta, t)
    k = norm_rope(qkv[nq * D:(nq + nkv) * D].view(nkv, D), w[f"{pre}.k_norm.weight"], pos + rope_delta, t)
    v = qkv[(nq + nkv) * D:].view(nkv, D)
    qd = q.double().to(K.device) / math.sqrt(D)
    Kd, Vd = K[:, n_pad:pos + 1].double(), V[:, n_pad:pos + 1].double()
    out = torch.empty(nq, D, dtype=torch.float64, device=K.device)
    floor = torch.empty_like(out)
    for h in range(nq):
        kvh = h // (nq // nkv)
        p = torch.softmax(Kd[kvh] @ qd[h], dim=0)
        out[h] = p @ Vd[kvh]
        floor[h] = 2.0 ** -12 * (p @ Vd[kvh].abs())
    return out, floor, k, v


def ulp_bf16(x):
    a = x.abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


STATS = {"worst": 0.0, "k_flips": 0, "k_elems": 0}


def check_row(eng, w, row, idx, pos, n_pad, tag=""):
    """The attention row of activation row `row` (stream slot idx, query position pos, rope position pos - n_pad) against
    float64; returns the row."""
    t = eng.cfg.talker
    qkv, attn = eng.debug_talker_attn(row)
    K, V = cache(eng, idx, t.num_hidden_layers - 1)
    torch.cuda.synchronize()
    ref, floor, k_exp, v_raw = reference(w, t, qkv, K, V, pos, n_pad, -n_pad)
    # the appended row at pos: V is the raw projection, K its norm + rope (equal up to rare 1-ulp flips)
    assert torch.equal(V[:, pos].cpu(), v_raw), (tag, "V row at pos")
    k_dev = K[:, pos].cpu().float()
    diff = (k_dev - k_exp.float()).abs()
    flips = int((diff > 0).sum())
    assert bool((diff <= ulp_bf16(k_exp.float()) + 1e-30).all()), (tag, "K row at pos differs by more than one ulp")
    STATS["k_flips"] += flips
    STATS["k_elems"] += diff.numel()
    err = (attn.view(t.num_attention_heads, D).double() - ref).abs()
    bound = ulp_bf16(ref) + floor
    worst = float((err / bound).max())
    STATS["worst"] = max(STATS["worst"], worst)
    bad = err > bound
    if bool(bad.any()):
        h, d = [int(x) for x in torch.nonzero(bad)[0]]
        raise AssertionError(f"{tag}: pos={pos} n_pad={n_pad}: {int(bad.sum())} elements out of bound, worst err/bound {worst:.2f}; "
                             f"first head {h} dim {d}: dev {float(attn.view(-1, D)[h, d])} ref {float(ref[h, d])}")
    return attn.clone()


@pytest.fixture(scope="module", autouse=True)
def report():
    """Printed once the module is done (visible with -s): the margin the bound left and the 1-ulp flips of appended K rows."""
    yield
    print(f"\nattention rows: largest err/bound {STATS['worst']:.3f}; appended K rows: {STATS['k_flips']} 1-ulp flips in "
          f"{STATS['k_elems']} elements")


# ------------------------------------------------------------------------------------------------
# engines
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny2k():
    cfg = make_cfg("tiny")
    w = make_weights(cfg, seed=21)
    eng = make_engine(cfg, w, max_seq_len=MAX_SEQ, max_streams=2, max_frames=16)
    yield cfg, w, eng
    eng.close()


@pytest.fixture(scope="module")
def dims06():
    cfg = make_cfg("0.6B-Base", 2, 2)
    w = make_weights(cfg, seed=22)
    eng = make_engine(cfg, w, max_seq_len=MAX_SEQ, max_streams=16, max_frames=16)
    yield cfg, w, eng
    eng.close()


def _cases():
    return [(L, 0) for L in LENGTHS] + PADDED


# ------------------------------------------------------------------------------------------------
# A: fq3_talker_step, one stream (cross-CTA splits + combine)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L,n_pad", _cases())
def test_talker_step_attention(tiny2k, L, n_pad):
    cfg, w, eng = tiny2k
    eng.reset_stream(0)
    pos = import_state(eng, 0, L, n_pad, seed=L * 7 + n_pad, cap=cap_of(eng))
    x = 0.05 * torch.randn(cfg.talker.hidden_size, generator=torch.Generator().manual_seed(L))
    eng.talker_step(0, x.to(torch.bfloat16).cuda(), pos, want_logits=False)
    check_row(eng, w, 0, 0, pos, n_pad, tag=f"talker_step L={L}")
    with pytest.raises(Exception, match="did not run this row"):
        eng.debug_talker_attn(1)


@pytest.mark.parametrize("L", [47, 575, 576, 577, 768, 769, 2048])
def test_talker_step_attention_real_dims(dims06, L):
    """0.6B dims: 8 kv heads x 16 splits = 128 items on the grid."""
    cfg, w, eng = dims06
    eng.reset_stream(0)
    pos = import_state(eng, 0, L, 0, seed=L, cap=cap_of(eng))
    x = 0.05 * torch.randn(cfg.talker.hidden_size, generator=torch.Generator().manual_seed(L))
    eng.talker_step(0, x.to(torch.bfloat16).cuda(), pos, want_logits=False)
    check_row(eng, w, 0, 0, pos, 0, tag=f"0.6B talker_step L={L}")


@pytest.mark.parametrize("L", [575, 576, 577, 769])
def test_talker_step_attention_grid96(L, monkeypatch):
    """FQ3_GRID=96 at 0.6B dims: cap = 96 // 8 = 12, so the long-range path starts above 576 positions."""
    monkeypatch.setenv("FQ3_GRID", "96")
    cfg = make_cfg("0.6B-Base", 1, 1)
    w = make_weights(cfg, seed=23)
    eng = make_engine(cfg, w, max_seq_len=1024, max_frames=16)
    try:
        assert eng.num_sms == 96 and cap_of(eng) == 12
        pos = import_state(eng, 0, L, 0, seed=L + 1, cap=12)
        x = 0.05 * torch.randn(cfg.talker.hidden_size, generator=torch.Generator().manual_seed(L))
        eng.talker_step(0, x.to(torch.bfloat16).cuda(), pos, want_logits=False)
        check_row(eng, w, 0, 0, pos, 0, tag=f"grid96 L={L}")
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------
# B / C / E: fq3_decode_frames, one frame, every row live
# ------------------------------------------------------------------------------------------------
def frame_states(eng, cfg, specs, seed):
    """Stream i at (L, n_pad) = specs[i], ready for one frame; returns the query positions."""
    H = cfg.talker.hidden_size
    cap = cap_of(eng)
    poss = []
    for i, (L, n_pad) in enumerate(specs):
        _, _, tth, tpe = synth_prompt(cfg, T=2, R=4, seed=seed + i)
        eng.reset_stream(i)
        eng.set_text_conditioning(i, tth[0].cuda(), tpe.cuda())
        pos = import_state(eng, i, L, n_pad, seed=seed * 100 + i, cap=cap)
        ph = 0.5 * torch.randn(H, generator=torch.Generator().manual_seed(seed + 50 + i))
        eng.set_loop_state(i, (37 * i + 5) % 1000, ph.to(torch.bfloat16).cuda(), pos, 0)
        poss.append(pos)
    return poss


def run_frame(eng, n):
    eng.decode_frames(n, 1, _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=8), _sub(do_sample=False))


def check_frame(eng, w, specs, poss, tag):
    rows = []
    for i, ((L, n_pad), pos) in enumerate(zip(specs, poss)):
        st = eng.status(i)
        assert st.error == 0 and st.n_frames == 1, (tag, i, st.error, st.n_frames)
        assert st.position == pos + 1 or pos == eng.max_seq_len - 1, (tag, i, st.position)
        rows.append(check_row(eng, w, i, i, pos, n_pad, tag=f"{tag} stream {i} L={L}"))
    with pytest.raises(Exception, match="did not run this row"):
        eng.debug_talker_attn(len(specs))
    return rows


@pytest.mark.parametrize("specs", [
    [(1, 0)], [(481, 0)], [(769, 0)], [(1537, 300)], [(2048, 0)],
    [(768, 0), (769, 0)], [(47, 5), (2047, 0)], [(2, 300), (1024, 0)],
], ids=lambda s: "-".join(f"{L}p{p}" if p else str(L) for L, p in s))
def test_frame_attention_reference_program(tiny2k, specs):
    cfg, w, eng = tiny2k
    poss = frame_states(eng, cfg, specs, seed=len(specs) * 10 + specs[0][0])
    run_frame(eng, len(specs))
    check_frame(eng, w, specs, poss, "frames")


WIDE_SHORT = [(L, 0) for L in (1, 2, 47, 48, 49, 97, 480, 481, 720, 721, 767, 768)] + [(300, 5), (600, 0), (700, 300), (10, 0)]
WIDE_MIXED = [(47, 0), (700, 0), (768, 0), (769, 0), (770, 0), (1023, 0), (1024, 0), (1500, 0), (1537, 0), (2047, 0),
              (2048, 0), (1, 0), (481, 0), (721, 5), (49, 0), (1200, 300)]


@pytest.mark.parametrize("specs", [WIDE_SHORT, WIDE_MIXED], ids=["all-short", "straddling-768"])
def test_frame_attention_wide_program(dims06, specs):
    """16 streams in one wide launch: every row against float64, and bit for bit the row of a single-stream launch of the
    same state (the split structure depends on L alone, fq3_kernel.cuh attn_phase)."""
    cfg, w, eng = dims06
    assert eng.lockstep_group >= 16
    poss = frame_states(eng, cfg, specs, seed=7)
    run_frame(eng, len(specs))
    wide = check_frame(eng, w, specs, poss, "wide")
    for i, (L, n_pad) in enumerate(specs):
        _, _, tth, tpe = synth_prompt(cfg, T=2, R=4, seed=7 + i)
        eng.reset_stream(0)
        eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())
        pos = import_state(eng, 0, L, n_pad, seed=7 * 100 + i, cap=cap_of(eng))
        ph = 0.5 * torch.randn(cfg.talker.hidden_size, generator=torch.Generator().manual_seed(7 + 50 + i))
        eng.set_loop_state(0, (37 * i + 5) % 1000, ph.to(torch.bfloat16).cuda(), pos, 0)
        run_frame(eng, 1)
        _, single = eng.debug_talker_attn(0)
        assert torch.equal(single, wide[i]), (i, L, n_pad)


def test_frame_attention_four_streams_1p7b():
    """1.7B dims have no wide program (lock-step group of 4): the reference-shaped program's generic walk with 4 rows."""
    cfg = make_cfg("1.7B-Base", 1, 1)
    w = make_weights(cfg, seed=24)
    eng = make_engine(cfg, w, max_seq_len=MAX_SEQ, max_streams=4, max_frames=16)
    try:
        assert eng.lockstep_group == 4
        specs = [(767, 0), (769, 0), (1537, 5), (2048, 0)]
        poss = frame_states(eng, cfg, specs, seed=3)
        run_frame(eng, 4)
        check_frame(eng, w, specs, poss, "1.7B")
    finally:
        eng.close()


def test_cache_bound_at_full_size(tiny2k):
    """A stream at position 2046 of a 2048-position cache keeps the frames at 2046 and 2047 (the frame that reaches
    max_seq_len - 1 is kept, then decoding stops: generate.py:174-177) and ends with done = 2; the attention row of the talker
    pass at 2047 matches float64."""
    cfg, w, eng = tiny2k
    specs = [(2047, 0)]
    poss = frame_states(eng, cfg, specs, seed=99)
    assert poss == [2046]
    eng.decode_frames(1, 4, _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=8), _sub(do_sample=False))
    st = eng.status(0)
    assert st.error == 0 and st.done == 2 and st.n_frames == MAX_SEQ - 2046, (st.error, st.done, st.n_frames)
    check_row(eng, w, 0, 0, MAX_SEQ - 1, 0, tag="cache bound")


# ------------------------------------------------------------------------------------------------
# D: fq3_prefill_tail on top of imported cache rows (chunk rows on the long path with fresh rows of the same chunk)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,n_tail", [(769, 8), (1030, 8), (2048, 8), (2048, 3), (800, 1)])
def test_prefill_tail_attention(tiny2k, T, n_tail):
    """fq3_prefill_tail keeps the cache rows before T - n_tail (prefill_impl only writes the rows it computes), so every row of
    its last chunk attends to the imported rows plus the chunk's own fresh rows."""
    cfg, w, eng = tiny2k
    t = cfg.talker
    start = T - n_tail
    eng.reset_stream(0)
    import_state(eng, 0, start + 1, 0, seed=T + n_tail, cap=cap_of(eng))  # rows [0, start)
    K0, _ = cache(eng, 0, t.num_hidden_layers - 1)
    before = K0[:, :start].clone()
    tail = 0.05 * torch.randn(n_tail, t.hidden_size, generator=torch.Generator().manual_seed(T))
    from qwen3_tts_cuda_graphs_b200 import _lib
    pol = _sp(do_sample=False, repetition_penalty=1.0, min_new_tokens=2).c()
    e = tail.to(torch.bfloat16).cuda()
    _lib.check(eng.lib.fq3_prefill_tail(eng.h, 0, e.data_ptr(), T, n_tail, C.byref(pol), None, torch.cuda.current_stream().cuda_stream))
    st = eng.status(0)
    assert st.error == 0 and st.position == T
    n_last = 0
    while n_last < 8:
        try:
            eng.debug_talker_attn(n_last)
        except Exception:
            break
        n_last += 1
    assert 1 <= n_last <= n_tail
    for r in range(n_last):
        check_row(eng, w, r, 0, T - n_last + r, 0, tag=f"prefill_tail T={T} row {r}")
    assert torch.equal(K0[:, :start], before)
