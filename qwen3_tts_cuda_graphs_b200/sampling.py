"""Fused CUDA sampling: suppress -> temperature -> top-k -> top-p -> draw, and HF repetition penalty.

Same call signatures as the reference's `faster_qwen3_tts/sampling.py:10-66`; the arithmetic runs in one
block-wide kernel of libfq3.so (`fq3_sample`, csrc/fq3_kernel.cuh `sample_row`) instead of ~15 ATen launches
with two host synchronisations (SURVEY.md §2c).  The draw uses a counter-based Philox stream, so the draws are not
torch.multinomial's, while greedy / top-k and top-p sets / penalties are exact; oracle/sampler_oracle.py replays every draw.
"""
from __future__ import annotations

from typing import Iterable, Optional

import torch

from .engine import Engine, SamplingPolicy

_default_engine: Optional[Engine] = None
_draw_counter = 0


def set_default_engine(engine: Optional[Engine]) -> None:
    global _default_engine
    _default_engine = engine


def _engine(engine: Optional[Engine]) -> Engine:
    e = engine or _default_engine
    if e is None:
        raise RuntimeError("no fq3 engine is loaded: sampling runs on the CUDA engine only (no CPU fallback)")
    return e


def apply_repetition_penalty(logits: torch.Tensor, token_history: torch.Tensor, repetition_penalty: float) -> torch.Tensor:
    """In-place HF-style penalty over the unique history (sampling.py:10-29).

    Kept for API parity with the reference's host loop; the device frame loop applies the penalty inside
    the sampling phase from a per-stream bitmap and never materialises the history.
    """
    if repetition_penalty == 1.0 or token_history.numel() == 0:
        return logits
    return _engine(None).apply_repetition_penalty(logits, token_history, repetition_penalty)


def sample_logits(
    logits: torch.Tensor,
    *,
    temperature: float,
    top_k: int,
    top_p: float,
    do_sample: bool,
    suppress_mask: Optional[torch.Tensor] = None,
    suppress_tokens: Optional[Iterable[int]] = None,
    engine: Optional[Engine] = None,
    seed: int = 0,
    draw_index: Optional[int] = None,
) -> torch.Tensor:
    """sampling.py:32-66 on the GPU.  logits [1, V] (or [V]) -> int64 [1]."""
    global _draw_counter
    e = _engine(engine)
    x = logits.reshape(-1)
    if suppress_mask is not None or suppress_tokens:
        x = x.clone()
        if suppress_mask is not None:
            x[suppress_mask.reshape(-1).to(x.device)] = float("-inf")
        if suppress_tokens:
            x[list(suppress_tokens)] = float("-inf")
    if draw_index is None:
        draw_index = _draw_counter
        _draw_counter += 1
    pol = SamplingPolicy(do_sample=do_sample, top_k=top_k, top_p=top_p, temperature=temperature,
                         repetition_penalty=1.0, min_new_tokens=0, suppress_tail=0, seed=seed)
    return e.sample(x, None, pol, eos_id=-1, suppress_eos=False, draw_index=draw_index)
