"""Draw-for-draw specification of the engine's samplers — TEST INFRASTRUCTURE ONLY.

`qwen3_tts_oracle.sample_logits` restates the reference's sampling.py with torch.multinomial, so it can only say which
tokens a draw may land on.  The engine draws with a counter-based Philox stream instead, so every draw is a function of
(logits, policy, key, draw index) and can be replayed exactly.  This module is that function:

  * `philox4x32_10`, `uniform`: the generator of csrc/fq3_kernel.cuh (`philox4x32_10`, and `(x >> 8) / 2**24` of its
    first output word in `sample_row` / `sample_fast`).
  * `stream_key`: the Philox key of a stream: `seed ^ K * (slot + 1)`, or `seed ^ K` when the stream has its own policy
    record (fq3_set_stream_policy), K = 0x9E3779B97F4A7C15.
  * The draw schedule (the counter is 0 after fq3_reset_stream, and every prefill resets the stream): the prefill's
    first-codebook token draws index 0; in frame f the predictor's codebook i (0..14) draws 33 f + i + 2 and the talker
    then draws 33 (f + 1); `fq3_predictor_run` on a freshly reset stream draws i + 1.  See `predictor_draw`,
    `talker_draw`.
  * `candidate_set_bf16`: sampling.py restated op by op on tensors of the logits' dtype, on whatever device they are on
    (the engine's set is the CPU one, see below): penalty -> suppression -> / T -> keep x >= k-th largest -> top-p on the stable
    descending sort (softmax, cumsum, `cum > top_p`, rank 0 kept).
  * `replay`: the token the engine must draw.  Greedy is the lowest-index maximum.  Otherwise the weights of the kept set
    are float64 `exp(x - max)` and the token is the first one, in index order, whose cumulative weight exceeds
    `u * total` (the device walks the same CDF; when fp32 rounding makes it fall off the end it takes the maximum).

Intended deviations of the engine from sampling.py, which this oracle encodes:
  * The multinomial: the reference draws from bf16-rounded softmax probabilities with torch.multinomial, the engine from
    fp32 `exp(x - max)` by inverse CDF on one Philox uniform.  Per-token probabilities therefore differ by at most 2^-8
    relative; no test can resolve that at a sane number of draws, and the replay follows the engine.
  * Rounding of the reference's bf16 ops, measured with torch 2.11 on a B200 (profiles/r03b_torch_bf16_rounding.log):
    - `bf16 / float` on CUDA is `x * (1 / T)` in fp32, rounded to bf16.  Over all finite bf16 values that equals the
      correctly rounded quotient (what the engine and torch on the CPU compute) at T = 0.05, 0.7, 0.8, 0.9, 1.1, 1.3, 1.5
      and 3.0, and differs in 1012 of 65 280 values by one bf16 ulp at T = 0.6.  The engine keeps the quotient.
    - softmax of a bf16 row on CUDA is the fp32 softmax rounded to bf16, as here.
    - cumsum of a bf16 row on CUDA rounds the partial sums of its parallel scan to bf16: 69 % of the prefixes of 200
      sampled rows differ from the correctly rounded prefix, and the top-p kept count differs in 57 / 154 of them at
      top_p = 0.8 / 0.95.  The set then depends on the scan's association order, which is no specification, so the engine
      and `candidate_set_bf16` (run on the CPU, where torch accumulates the prefix in fp32 and rounds it) keep a prefix
      while its correctly rounded value is at most bf16(top_p) (an exact tie rounds to even: for 0.8 and 0.95, whose
      bf16 mantissas are odd, a prefix exactly on the midpoint is dropped).

Everything a draw depends on but float64 cannot pin (fp32 `expf`, summation order) is bounded by `AMBIG`: a draw is
ambiguous when `u * total` lies within AMBIG * total of a CDF boundary, or when the top-p set read with that much slack
(fp32: the cumulative against the threshold; bf16: each probability against its bf16 rounding midpoints) draws a
different token than the nominal set.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

M32 = 0xFFFFFFFF
M64 = 0xFFFFFFFFFFFFFFFF
KEY_MUL = 0x9E3779B97F4A7C15
AMBIG = 4e-6  # fp32 prefix sums of <= 5120 terms in the device's scan order stay well inside it


# ------------------------------------------------------------------------------------------------
# Philox stream and draw schedule
# ------------------------------------------------------------------------------------------------
def philox4x32_10(ctr: Sequence[int], key: Sequence[int]) -> Tuple[int, int, int, int]:
    """Random123 Philox4x32-10: counter (4 words) and key (2 words) as Python ints."""
    c0, c1, c2, c3 = (int(v) & M32 for v in ctr)
    k0, k1 = (int(v) & M32 for v in key)
    for _ in range(10):
        p0 = 0xD2511F53 * c0
        p1 = 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> 32) ^ c3 ^ k1) & M32, p0 & M32
        k0 = (k0 + 0x9E3779B9) & M32
        k1 = (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


def uniform(key64: int, draw64: int) -> float:
    """The sampler's uniform in [0, 1): 24 bits of the first Philox word (exact in fp32 and float64)."""
    key64, draw64 = int(key64) & M64, int(draw64) & M64
    x = philox4x32_10((draw64 & M32, draw64 >> 32, 0, 0), (key64 & M32, key64 >> 32))[0]
    return (x >> 8) / 2.0**24


def stream_key(seed: int, slot: int, own: bool) -> int:
    """Philox key of a stream's draws: the stream's policy record makes it independent of the slot."""
    return (int(seed) ^ (KEY_MUL * (1 if own else slot + 1))) & M64


def predictor_draw(frame: int, i: int) -> int:
    """Draw index of predictor codebook i (0..14) in frame `frame` of the frame loop."""
    return 33 * frame + i + 2


def talker_draw(frame: int) -> int:
    """Draw index of the first-codebook token sampled at the end of frame `frame` (the prefill's token draws 0)."""
    return 33 * (frame + 1)


# ------------------------------------------------------------------------------------------------
# sampling.py in the logits' dtype
# ------------------------------------------------------------------------------------------------
@dataclass
class Policy:
    do_sample: bool = True
    top_k: int = 50
    top_p: float = 1.0
    temperature: float = 0.9
    repetition_penalty: float = 1.0
    suppress_tail: int = 0       # ids >= V - suppress_tail are masked, except eos
    eos: int = -1
    suppress_eos: bool = False


def _mask(V: int, pol: Policy) -> torch.Tensor:
    m = torch.zeros(V, dtype=torch.bool)
    if pol.suppress_tail > 0:
        m[max(0, V - pol.suppress_tail):] = True
        if 0 <= pol.eos < V:
            m[pol.eos] = False
    if pol.suppress_eos and 0 <= pol.eos < V:
        m[pol.eos] = True
    return m


def penalised(logits: torch.Tensor, pol: Policy, seen: Optional[Iterable[int]]) -> torch.Tensor:
    """Repetition penalty (sampling.py:10-29) over the unique in-range history, then suppression; 1-D, logits' dtype."""
    x = logits.reshape(-1).clone()
    V = x.numel()
    if seen is not None and pol.repetition_penalty != 1.0:
        ids = sorted({int(t) for t in seen if 0 <= int(t) < V})
        if ids:
            ids_t = torch.tensor(ids, dtype=torch.long, device=x.device)
            picked = x[ids_t]
            x[ids_t] = torch.where(picked > 0, picked / pol.repetition_penalty, picked * pol.repetition_penalty)
    x[_mask(V, pol).to(x.device)] = float("-inf")
    return x


def scale(x: torch.Tensor, temperature: float) -> torch.Tensor:
    """x / T as the engine computes it: the correctly rounded fp32 quotient, rounded to the logits' dtype."""
    q = x.float().cpu() / torch.tensor(float(temperature), dtype=torch.float32)
    return q.to(x.dtype).to(x.device)


def candidate_set_bf16(logits: torch.Tensor, pol: Policy, seen: Optional[Iterable[int]] = None) -> torch.Tensor:
    """Boolean [V] mask of the tokens sampling.py can draw, every intermediate a tensor of the logits' dtype on the
    logits' device: softmax and cumsum of a bf16 row give bf16 results, and `cum > top_p` compares against top_p
    rounded to that dtype.  On CUDA the bf16 cumsum is not correctly rounded (module docstring): pass CPU tensors for the
    set the engine implements."""
    x = penalised(logits, pol, seen) / pol.temperature
    neg = float("-inf")
    V = x.numel()
    if pol.top_k > 0:
        kth = torch.topk(x, min(pol.top_k, V)).values[-1]
        x = torch.where(x < kth, torch.full_like(x, neg), x)
    if pol.top_p < 1.0:
        srt, idx = torch.sort(x, descending=True, stable=True)
        cum = torch.cumsum(F.softmax(srt, dim=-1), dim=-1)
        drop = cum > pol.top_p
        drop[0] = False
        srt = srt.masked_fill(drop, neg)
        x = torch.full_like(x, neg).scatter_(-1, idx, srt)
    return torch.isfinite(x)


# ------------------------------------------------------------------------------------------------
# replay
# ------------------------------------------------------------------------------------------------
def _top_p_keep(x64: torch.Tensor, finite: torch.Tensor, top_p: float, bf16: bool, reading: int) -> torch.Tensor:
    """Top-p kept mask of the engine's arithmetic in float64: rank j (stable descending order) survives iff its
    cumulative probability, through j, is at most the threshold; rank 0 always.  fp32 mode: the threshold is
    fp32(top_p), moved by reading * AMBIG.  bf16 mode: every probability is rounded to bf16 (after scaling it by
    1 + reading * AMBIG, so that a probability within fp32 noise of a bf16 rounding midpoint rounds both ways across the
    readings) and the prefix — a sum of bf16 values, exact here and on the device — is kept while it rounds to at most
    bf16(top_p): below the midpoint above bf16(top_p), or on it when bf16(top_p) is even (round to nearest even).  That
    means the same as the reference's bf16 `cum > top_p` with a correctly rounded cumsum."""
    V = x64.numel()
    order = torch.sort(x64, descending=True, stable=True).indices
    xs = x64[order]
    p = torch.where(torch.isfinite(xs), torch.exp(xs - xs[0]), torch.zeros_like(xs))
    p = p / p.sum()
    if bf16:
        p = (p * (1.0 + reading * AMBIG)).float().to(torch.bfloat16).double()
        thr, strict = bf16_top_p_threshold(top_p)
        cum = torch.cumsum(p, 0)
        keep_s = (cum < thr) | ((cum == thr) & (not strict))
    else:
        thr = float(torch.tensor(top_p, dtype=torch.float32))
        keep_s = torch.cumsum(p, 0) <= thr + reading * AMBIG
    keep_s[0] = True
    keep = torch.zeros(V, dtype=torch.bool)
    keep[order] = keep_s
    return keep & finite


def bf16_top_p_threshold(v: float) -> Tuple[float, bool]:
    """(midpoint between bf16(v) and the next bf16 value, whether a sum exactly on it rounds up): a prefix rounds to at
    most bf16(v) iff it lies below the midpoint, or on it when bf16(v) has an even mantissa."""
    b = torch.tensor(v, dtype=torch.float32).to(torch.bfloat16)
    bits = int(b.view(torch.int16)) & 0xFFFF
    nxt = torch.tensor(bits + 1, dtype=torch.int32).to(torch.int16).view(torch.bfloat16)
    return (float(b) + float(nxt)) / 2.0, bool(bits & 1)


@dataclass
class Replay:
    """The engine's sampler on one (logits, policy, seen): `draw(key, index) -> (token, ambiguous)`."""
    greedy: int
    do_sample: bool
    sets: List[Tuple[torch.Tensor, torch.Tensor]]   # (kept index list, float64 cumulative weights): nominal reading first
    amax: int

    def draw(self, key: int, index: int) -> Tuple[int, bool]:
        if not self.do_sample:
            return self.greedy, False
        u = uniform(key, index)
        toks, amb = [], False
        for idx, cum in self.sets:
            total = float(cum[-1])
            target = u * total
            j = int(torch.searchsorted(cum, torch.tensor([target], dtype=torch.float64), right=True)[0])
            toks.append(int(idx[j]) if j < idx.numel() else self.amax)
            amb |= bool((cum - target).abs().min() <= AMBIG * total)
        return toks[0], amb or len(set(toks)) > 1


def replayer(logits: torch.Tensor, pol: Policy, seen: Optional[Iterable[int]] = None) -> Replay:
    """Set up the replay of every draw on these logits: bf16 logits are sampled with every intermediate rounded to bf16
    (the in-kernel samplers, and fq3_sample with flag 1), fp32 logits in fp32."""
    bf16 = logits.dtype == torch.bfloat16
    seen = None if seen is None else list(seen)
    x = penalised(logits.cpu(), pol, seen)
    greedy = int(torch.argmax(x.float()))  # first maximum
    if not pol.do_sample:
        return Replay(greedy, False, [], greedy)
    xs = scale(x, pol.temperature).double()
    V = xs.numel()
    finite = torch.isfinite(xs)
    if pol.top_k > 0 and pol.top_k < V:
        kth = torch.topk(xs, pol.top_k).values[-1]
        finite &= xs >= kth
    xs = torch.where(finite, xs, torch.full_like(xs, float("-inf")))
    amax = int(torch.argmax(xs))
    readings = [finite]
    if pol.top_p < 1.0:
        readings = [_top_p_keep(xs, finite, pol.top_p, bf16, r) for r in (0, -1, 1)]
    sets = []
    vmax = float(xs.max())
    for keep in readings:
        idx = torch.nonzero(keep).reshape(-1)
        w = torch.exp(xs[idx] - vmax)
        sets.append((idx, torch.cumsum(w, 0)))
    return Replay(greedy, True, sets, amax)


def replay(logits: torch.Tensor, pol: Policy, seen: Optional[Iterable[int]], key: int, draw: int) -> Tuple[int, bool]:
    """(token, ambiguous) of the engine's draw `draw` under Philox key `key`."""
    return replayer(logits, pol, seen).draw(key, draw)
