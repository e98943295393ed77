"""Thin Python wrapper over the C ABI: turns torch tensors into device pointers on the current stream.

PyTorch is plumbing here (device memory + stream handle); all arithmetic happens in libfq3.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from .config import TTSConfig
from .weights import LAYER_FIELDS, Arena


@dataclass
class SamplingPolicy:
    """First-codebook sampler arguments of generate.py:16-37."""

    do_sample: bool = True
    top_k: int = 50
    top_p: float = 1.0
    temperature: float = 0.9
    repetition_penalty: float = 1.05
    min_new_tokens: int = 2
    suppress_tail: int = 1024
    seed: int = 0

    def validate(self, vocab: Optional[int] = None) -> "SamplingPolicy":
        """ValueError for out-of-range sampling values: what fq3_set_stream_policy refuses (fq3.h: top_k < 0, top_p outside
        (0, 1], temperature <= 0 with do_sample, repetition_penalty <= 0, suppress_tail outside [0, vocab]), a negative
        min_new_tokens and a seed that does not fit 64 bits."""
        if int(self.top_k) < 0:
            raise ValueError(f"top_k must be >= 0, got {self.top_k}")
        if not 0.0 < float(self.top_p) <= 1.0:
            raise ValueError(f"top_p must be in (0, 1], got {self.top_p}")
        if self.do_sample and not float(self.temperature) > 0.0:
            raise ValueError(f"temperature must be > 0 when sampling, got {self.temperature}")
        if not float(self.repetition_penalty) > 0.0:
            raise ValueError(f"repetition_penalty must be > 0, got {self.repetition_penalty}")
        if int(self.min_new_tokens) < 0:
            raise ValueError(f"min_new_tokens must be >= 0, got {self.min_new_tokens}")
        if int(self.suppress_tail) < 0 or (vocab is not None and int(self.suppress_tail) > vocab):
            raise ValueError(f"suppress_tail must be in [0, {vocab}], got {self.suppress_tail}")
        if not 0 <= int(self.seed) < 2**64:
            raise ValueError(f"seed must be in [0, 2**64), got {self.seed}")
        return self

    def c(self) -> _lib.Policy:
        return _lib.Policy(
            int(self.do_sample), int(self.top_k), float(self.top_p), float(self.temperature),
            float(self.repetition_penalty), int(self.min_new_tokens), int(self.suppress_tail), int(self.seed) & (2**64 - 1),
        )


@dataclass
class SubPolicy:
    """Predictor sampler attributes frozen at capture time in the reference (predictor_graph.py:34-50)."""

    do_sample: bool = True
    top_k: int = 50
    top_p: float = 1.0
    temperature: float = 0.9

    def c(self) -> _lib.SubPolicy:
        return _lib.SubPolicy(int(self.do_sample), int(self.top_k), float(self.top_p), float(self.temperature))


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class Engine:
    def __init__(self, cfg: TTSConfig, arena: Arena, max_seq_len: int, max_streams: int = 1, max_frames: int = 4096):
        if not arena.buf.is_cuda:
            raise ValueError("the fq3 engine needs its weight arena on a CUDA device")
        self.lib = _lib.load()
        self.cfg, self.arena = cfg, arena
        self.max_seq_len, self.max_streams, self.max_frames = max_seq_len, max_streams, max_frames
        self.device = arena.buf.device
        t, p = cfg.talker, cfg.predictor
        self.ncb = p.num_codebooks
        self._keep = []

        def stack(prefix, sc, rope, max_pos, rope_len):
            offs = (C.c_uint64 * (sc.num_hidden_layers * 8))()
            for l in range(sc.num_hidden_layers):
                for j, f in enumerate(LAYER_FIELDS):
                    offs[l * 8 + j] = arena.offsets[f"{prefix}.layers.{l}.{f}"]
            self._keep.append(offs)
            return _lib.StackDesc(
                sc.hidden_size, sc.intermediate_size, sc.num_hidden_layers, sc.num_attention_heads,
                sc.num_key_value_heads, sc.head_dim, sc.vocab_size, sc.rms_norm_eps,
                C.cast(offs, C.POINTER(C.c_uint64)), arena.offsets[f"{prefix}.norm"],
                arena.offsets[f"rope.{rope}.cos"], arena.offsets[f"rope.{rope}.sin"], rope_len, max_pos,
            )

        lm = (C.c_uint64 * self.ncb)(*[arena.offsets[f"talker.code_predictor.lm_head.{i}"] for i in range(self.ncb)])
        pe = (C.c_uint64 * self.ncb)(*[arena.offsets[f"talker.code_predictor.codec_embedding.{i}"] for i in range(self.ncb)])
        self._keep += [lm, pe]
        has_s2m = t.hidden_size != p.hidden_size
        desc = _lib.ModelDesc(
            _lib.ABI_VERSION, arena.buf.data_ptr(), arena.buf.numel(),
            stack("talker.model", t, "talker", max_seq_len, arena.shapes["rope.talker.cos"][0]),
            stack("talker.code_predictor.model", p, "pred", p.num_code_groups + 1, arena.shapes["rope.pred.cos"][0]),
            arena.offsets["talker.codec_head"], arena.offsets["talker.codec_embedding"], p.num_code_groups,
            C.cast(lm, C.POINTER(C.c_uint64)), C.cast(pe, C.POINTER(C.c_uint64)),
            int(has_s2m),
            arena.offsets.get("talker.code_predictor.s2m.weight", 0), arena.offsets.get("talker.code_predictor.s2m.bias", 0),
            t.codec_eos_token_id, max_streams, max_frames,
        )
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.fq3_create(C.byref(desc), C.byref(h)))
        self.h = h
        self._dense = None        # dense tensor-core prefill plan (prefill_dense.py), built on first use
        self._dense_tried = False

    def close(self):
        if getattr(self, "_dense", None) is not None:
            self._dense.close()
            self._dense = None
        if getattr(self, "h", None):
            self.lib.fq3_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reduced_grid(self) -> int:
        """CTAs of the engine's reduced frame-loop grid (0 = none): see include/fq3.h, fq3_set_decode_grid."""
        return int(self.lib.fq3_reduced_grid(self.h))

    def set_decode_grid(self, n_ctas: int = 0) -> None:
        """Grid of the following decode_frames launches: 0 / num_sms = full, reduced_grid() = leave SMs free for the codec."""
        _lib.check(self.lib.fq3_set_decode_grid(self.h, int(n_ctas)))

    # ---- helpers ----
    def _bf16(self, x: torch.Tensor) -> torch.Tensor:
        x = x.to(device=self.device, dtype=torch.bfloat16).contiguous()
        self._scratch_ref = x
        return x

    @property
    def num_sms(self) -> int:
        return self.lib.fq3_num_sms(self.h)

    @property
    def launch_count(self) -> int:
        return int(self.lib.fq3_launch_count(self.h))

    # ---- per-utterance set-up ----
    def reset_stream(self, idx: int = 0):
        _lib.check(self.lib.fq3_reset_stream(self.h, idx, _stream()))

    def retire_stream(self, idx: int):
        """Take a slot out of the lock-step frame loop until its next reset + prefill (fq3.h: fq3_retire_stream)."""
        _lib.check(self.lib.fq3_retire_stream(self.h, idx, _stream()))

    def set_stream_policy(self, idx: int, policy: Optional[SamplingPolicy]):
        """A stream's own sampling policy, seed included, used by its prefill and every frame-loop launch instead of the launch's
        policy (fq3.h: fq3_set_stream_policy); None clears it.  Survives prefill; reset_stream clears it."""
        pol = None if policy is None else C.byref(policy.c())
        _lib.check(self.lib.fq3_set_stream_policy(self.h, int(idx), pol, _stream()))

    def set_generation_state(self, idx: int, n_left_pad: int, rope_delta: int):
        _lib.check(self.lib.fq3_set_generation_state(self.h, idx, int(n_left_pad), int(rope_delta), _stream()))

    def set_text_conditioning(self, idx: int, trailing: torch.Tensor, pad_embed: torch.Tensor):
        H = self.cfg.talker.hidden_size
        tr = self._bf16(trailing.reshape(-1, H))
        pe = self._bf16(pad_embed.reshape(H))
        _lib.check(self.lib.fq3_set_text_conditioning(self.h, idx, tr.data_ptr(), tr.shape[0], pe.data_ptr(), _stream()))
        self._cond_ref = (tr, pe)

    def open_text(self, idx: int, pad_embed: torch.Tensor):
        """Empty the stream's trailing text and leave it open: its rows arrive through append_text while it decodes, and a frame
        whose text row has not arrived waits (status.done = 4) instead of running (fq3.h: fq3_open_text)."""
        pe = self._bf16(pad_embed.reshape(self.cfg.talker.hidden_size))
        _lib.check(self.lib.fq3_open_text(self.h, int(idx), pe.data_ptr(), _stream()))
        self._open_ref = pe

    def append_text(self, idx: int, rows: torch.Tensor, close: bool = False):
        """Append bf16 text rows [n, H_t] to an open stream's trailing text; close=True ends the text (fq3.h: fq3_append_text).
        Fq3Error when the stream's text is not open, RuntimeError past max_seq_len rows."""
        r = self._bf16(rows.reshape(-1, self.cfg.talker.hidden_size))
        ptr = r.data_ptr() if r.shape[0] > 0 else None
        _lib.check(self.lib.fq3_append_text(self.h, int(idx), ptr, int(r.shape[0]), int(bool(close)), _stream()))
        self._append_ref = r

    def import_kv(self, idx: int, layer: int, k: torch.Tensor, v: torch.Tensor):
        k, v = self._bf16(k), self._bf16(v)  # [nkv, T, d]
        self._kv_ref = (k, v)
        _lib.check(self.lib.fq3_import_kv(self.h, idx, layer, k.data_ptr(), v.data_ptr(), k.shape[-2], _stream()))

    def set_loop_state(self, idx: int, token: int, past_hidden: torch.Tensor, position: int, gen_step: int):
        ph = self._bf16(past_hidden.reshape(-1))
        _lib.check(self.lib.fq3_set_loop_state(self.h, idx, int(token), ph.data_ptr(), int(position), int(gen_step), _stream()))

    # ---- hot path ----
    def prefill(self, idx: int, embeds: torch.Tensor, n_left_pad: int, policy: SamplingPolicy, want_logits: bool = False,
                dense: Optional[bool] = None):
        """Prompt prefill (generate.py:107-134).  Prompts of more than a few rows take the dense tensor-core path for rows
        [0, T-1) (prefill_dense.py) and the decode kernel for the last row; `dense=False` forces the chunked path."""
        H = self.cfg.talker.hidden_size
        e = self._bf16(embeds.reshape(-1, H))
        T = e.shape[0]
        logits = torch.empty(self.cfg.talker.vocab_size, dtype=torch.float32, device=self.device) if want_logits else None
        pol = policy.c()
        if dense is None:
            dense = True
        if dense and int(n_left_pad) == 0 and T <= self.max_seq_len:
            if self._dense is None and not self._dense_tried:
                self._dense_tried = True
                from . import prefill_dense
                self._dense = prefill_dense.make(self)
            if self._dense is not None and T - 1 >= self._dense.MIN_ROWS:
                if self._dense.full:
                    self._dense.run(idx, e, T)
                    last = self._dense.x_last[T - 1]
                    _lib.check(self.lib.fq3_prefill_head(self.h, idx, last.data_ptr(), T, C.byref(pol), _ptr(logits), _stream()))
                else:
                    self._dense.run(idx, e, T - 1)
                    _lib.check(self.lib.fq3_prefill_tail(self.h, idx, e[T - 1:].data_ptr(), T, 1, C.byref(pol), _ptr(logits), _stream()))
                return logits
        _lib.check(self.lib.fq3_prefill(self.h, idx, e.data_ptr(), T, int(n_left_pad), C.byref(pol), _ptr(logits), _stream()))
        return logits

    def talker_step(self, idx: int, embeds: torch.Tensor, position: int, want_logits: bool = True):
        H = self.cfg.talker.hidden_size
        e = self._bf16(embeds.reshape(H))
        hidden = torch.empty(H, dtype=torch.bfloat16, device=self.device)
        logits = torch.empty(self.cfg.talker.vocab_size, dtype=torch.float32, device=self.device) if want_logits else None
        _lib.check(self.lib.fq3_talker_step(self.h, idx, e.data_ptr(), int(position), hidden.data_ptr(), _ptr(logits), _stream()))
        return hidden, logits

    def predictor_run(self, idx: int, pred_input: torch.Tensor, sub: SubPolicy, seed: int = 0, want_logits: bool = False):
        H = self.cfg.talker.hidden_size
        x = self._bf16(pred_input.reshape(2, H))
        codes = torch.empty(self.ncb, dtype=torch.int64, device=self.device)
        logits = (
            torch.empty(self.ncb, self.cfg.predictor.vocab_size, dtype=torch.float32, device=self.device) if want_logits else None
        )
        s = sub.c()
        _lib.check(self.lib.fq3_predictor_run(self.h, idx, x.data_ptr(), C.byref(s), int(seed) & (2**64 - 1), codes.data_ptr(), _ptr(logits), _stream()))
        return codes, logits

    def sample(self, logits: torch.Tensor, history: Optional[torch.Tensor], policy: SamplingPolicy, eos_id: int,
               suppress_eos: bool, draw_index: int = 0) -> torch.Tensor:
        flags = 1 if logits.dtype == torch.bfloat16 else 0
        lg = logits.reshape(-1).to(device=self.device, dtype=torch.float32).contiguous()
        hist = None
        if history is not None and history.numel() > 0:
            hist = history.reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
        out = torch.empty(1, dtype=torch.int64, device=self.device)
        pol = policy.c()
        _lib.check(self.lib.fq3_sample(
            self.h, lg.data_ptr(), lg.numel(), _ptr(hist), 0 if hist is None else hist.numel(), C.byref(pol),
            int(eos_id), int(bool(suppress_eos)), flags, int(draw_index), out.data_ptr(), _stream()))
        self._sample_ref = (lg, hist)
        return out

    def apply_repetition_penalty(self, logits: torch.Tensor, history: torch.Tensor, penalty: float) -> torch.Tensor:
        """In place on a CUDA tensor (sampling.py:10-29)."""
        if not logits.is_cuda:
            raise RuntimeError("fq3 repetition penalty runs on CUDA tensors only (no CPU fallback)")
        V = logits.shape[-1]
        flags = 1 if logits.dtype == torch.bfloat16 else 0
        work = logits.reshape(-1, V)[0].to(torch.float32).contiguous()
        hist = history.reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
        _lib.check(self.lib.fq3_apply_repetition_penalty(
            self.h, work.data_ptr(), V, hist.data_ptr(), hist.numel(), float(penalty), flags, _stream()))
        logits.reshape(-1, V)[0].copy_(work)
        return logits

    def assemble_prompt(self, tp_rows: torch.Tensor, desc: torch.Tensor, spk_rows: Optional[torch.Tensor], ref_codes: Optional[torch.Tensor],
                        out: torch.Tensor) -> None:
        """fq3.h: fq3_assemble_prompt.  desc int32 [n, 4] on the device; out bf16 [n, H_t]."""
        assert desc.dtype == torch.int32 and desc.is_cuda and desc.is_contiguous() and out.is_contiguous() and tp_rows.is_contiguous()
        _lib.check(self.lib.fq3_assemble_prompt(self.h, tp_rows.data_ptr(), desc.data_ptr(), int(desc.shape[0]), _ptr(spk_rows),
                                                _ptr(ref_codes), out.data_ptr(), _stream()))

    @property
    def lockstep_group(self) -> int:
        """Streams that share one weight sweep of the frame loop (fq3.h: fq3_lockstep_group); more streams run in groups."""
        return int(self.lib.fq3_lockstep_group(self.h))

    def decode_frames(self, n_streams: int, n_frames: int, policy: SamplingPolicy, sub: SubPolicy):
        pol, s = policy.c(), sub.c()
        _lib.check(self.lib.fq3_decode_frames(self.h, int(n_streams), int(n_frames), C.byref(pol), C.byref(s), _stream()))

    def debug_talker_logits(self, idx: int = 0) -> torch.Tensor:
        """fp32 [V_t]: the logits stream idx's last talker sampler consumed, right after decode_frames (fq3.h test hook)."""
        out = torch.empty(self.cfg.talker.vocab_size, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.fq3_debug_read_talker_logits(self.h, int(idx), out.data_ptr(), _stream()))
        return out

    def last_hidden(self, row: int = 0) -> torch.Tensor:
        out = torch.empty(self.cfg.talker.hidden_size, dtype=torch.bfloat16, device=self.device)
        _lib.check(self.lib.fq3_last_hidden(self.h, int(row), out.data_ptr(), _stream()))
        return out

    def status(self, idx: int = 0) -> _lib.Status:
        st = _lib.Status()
        _lib.check(self.lib.fq3_get_status(self.h, idx, C.byref(st), _stream()))
        return st

    def read_codes(self, idx: int, first: int, n: int) -> torch.Tensor:
        """int64 [n, num_code_groups] on the host (one D2H copy of n*16 int32)."""
        g = self.cfg.talker.num_code_groups
        buf = np.empty((max(n, 0), g), dtype=np.int32)
        if n > 0:
            _lib.check(self.lib.fq3_read_codes(self.h, idx, int(first), int(n), buf.ctypes.data_as(C.POINTER(C.c_int32)), _stream()))
        return torch.from_numpy(buf.astype(np.int64))

    def linear(self, W: torch.Tensor, x: torch.Tensor, *, gamma=None, eps: float = 1e-6, bias=None, residual=None,
               swiglu: bool = False, out_f32: bool = False, silu: bool = False) -> torch.Tensor:
        """Parity-test hook: y = epilogue(W @ prologue(x)) through the streaming kernel."""
        M, K = x.shape
        N = W.shape[0]
        flags = (1 if gamma is not None else 0) | (2 if bias is not None else 0) | (4 if residual is not None else 0) | \
                (8 if swiglu else 0) | (16 if out_f32 else 0) | (32 if silu else 0)
        y = torch.empty(M, N // 2 if swiglu else N, dtype=torch.float32 if out_f32 else torch.bfloat16, device=self.device)
        _lib.check(self.lib.fq3_linear(
            self.h, W.data_ptr(), x.data_ptr(), y.data_ptr(), M, N, K, flags, _ptr(gamma), float(eps), _ptr(bias),
            _ptr(residual), _stream()))
        return y
