"""ctypes binding of libfq3.so (C ABI in include/fq3.h).  Loading fails loudly: there is no fallback."""
from __future__ import annotations

import ctypes as C
import os
import shutil

from . import build as _build


class StackDesc(C.Structure):
    _fields_ = [
        ("hidden", C.c_int32), ("inter", C.c_int32), ("n_layers", C.c_int32), ("n_q_heads", C.c_int32),
        ("n_kv_heads", C.c_int32), ("head_dim", C.c_int32), ("vocab", C.c_int32), ("rms_eps", C.c_float),
        ("layer_offs", C.POINTER(C.c_uint64)), ("final_norm_off", C.c_uint64),
        ("rope_cos_off", C.c_uint64), ("rope_sin_off", C.c_uint64), ("rope_len", C.c_int32), ("max_pos", C.c_int32),
    ]


class ModelDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("arena", C.c_void_p), ("arena_bytes", C.c_uint64),
        ("talker", StackDesc), ("predictor", StackDesc),
        ("codec_head_off", C.c_uint64), ("codec_embed_off", C.c_uint64), ("n_code_groups", C.c_int32),
        ("lm_head_offs", C.POINTER(C.c_uint64)), ("pred_embed_offs", C.POINTER(C.c_uint64)),
        ("has_s2m", C.c_int32), ("s2m_w_off", C.c_uint64), ("s2m_b_off", C.c_uint64),
        ("eos_id", C.c_int32), ("max_streams", C.c_int32), ("max_frames", C.c_int32),
    ]


class Policy(C.Structure):
    _fields_ = [
        ("do_sample", C.c_int32), ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float),
        ("repetition_penalty", C.c_float), ("min_new_tokens", C.c_int32), ("suppress_tail", C.c_int32),
        ("seed", C.c_uint64),
    ]


class SubPolicy(C.Structure):
    _fields_ = [("do_sample", C.c_int32), ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float)]


class Status(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("done", C.c_int32), ("position", C.c_int32), ("gen_step", C.c_int32),
        ("token", C.c_int32), ("error", C.c_int32),
    ]


ABI_VERSION = 2  # FQ3_ABI_VERSION of include/fq3.h

# every symbol include/fq3.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "fq3_abi_version": (C.c_int, []),
    "fq3_last_error": (C.c_char_p, []),
    "fq3_create": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(_P)]),
    "fq3_destroy": (C.c_int, [_P]),
    "fq3_num_sms": (C.c_int, [_P]),
    "fq3_launch_count": (C.c_int64, [_P]),
    "fq3_reset_stream": (C.c_int, [_P, C.c_int, _P]),
    "fq3_retire_stream": (C.c_int, [_P, C.c_int, _P]),
    "fq3_set_stream_policy": (C.c_int, [_P, C.c_int, C.POINTER(Policy), _P]),
    "fq3_set_generation_state": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P]),
    "fq3_set_text_conditioning": (C.c_int, [_P, C.c_int, _P, C.c_int, _P, _P]),
    "fq3_open_text": (C.c_int, [_P, C.c_int, _P, _P]),
    "fq3_append_text": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, _P]),
    "fq3_import_kv": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_int, _P]),
    "fq3_set_loop_state": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P]),
    "fq3_prefill": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, C.POINTER(Policy), _P, _P]),
    "fq3_prefill_tail": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, C.POINTER(Policy), _P, _P]),
    "fq3_prefill_head": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(Policy), _P, _P]),
    "fq3_kv_cache_ptr": (_P, [_P, C.c_int, C.c_int, C.c_int]),
    "fq3_talker_step": (C.c_int, [_P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "fq3_predictor_run": (C.c_int, [_P, C.c_int, _P, C.POINTER(SubPolicy), C.c_uint64, _P, _P, _P]),
    "fq3_sample": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.POINTER(Policy), C.c_int, C.c_int, C.c_int, C.c_uint64, _P, _P]),
    "fq3_apply_repetition_penalty": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, C.c_int, _P]),
    "fq3_decode_frames": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(Policy), C.POINTER(SubPolicy), _P]),
    "fq3_reduced_grid": (C.c_int, [_P]),
    "fq3_lockstep_group": (C.c_int, [_P]),
    "fq3_assemble_prompt": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, _P]),
    "fq3_set_decode_grid": (C.c_int, [_P, C.c_int]),
    "fq3_clear_fault": (C.c_int, [_P, _P]),
    "fq3_debug_set_epoch": (C.c_int, [_P, C.c_uint32]),
    "fq3_debug_read_talker_logits": (C.c_int, [_P, C.c_int, _P, _P]),
    "fq3_debug_read_talker_attn": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "fq3_get_status": (C.c_int, [_P, C.c_int, C.POINTER(Status), _P]),
    "fq3_read_codes": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), _P]),
    "fq3_last_hidden": (C.c_int, [_P, C.c_int, _P, _P]),
    "fq3_codes_device_ptr": (_P, [_P, C.c_int]),
    "fq3_debug_read_prof": (C.c_int, [_P, C.POINTER(C.c_longlong), C.c_int]),
    "fq3_linear": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_float, _P, _P, _P]),
}

_lib = None


class Fq3Error(RuntimeError):
    pass


def load():
    """dlopen the in-tree library (building it first when nvcc is present and sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.lib_path("libfq3.so")
    if (not os.path.exists(path) or _build.is_stale("libfq3.so")) and (shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc")):
        _build.build_lib("libfq3.so")
    if not os.path.exists(path):
        raise Fq3Error(
            f"{path} is missing: build it with `python -m qwen3_tts_cuda_graphs_b200.build`. "
            "This engine has no CPU or PyTorch fallback."
        )
    if os.environ.get("FQ3_LIB_PATH"):  # development: A/B a differently compiled build of the same sources
        path = os.environ["FQ3_LIB_PATH"]
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the ABI lost a symbol
        fn.restype = res
        fn.argtypes = args
    if lib.fq3_abi_version() != ABI_VERSION:
        raise Fq3Error("libfq3.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().fq3_last_error().decode("utf-8", "replace")
        if -rc == 3:
            raise RuntimeError(msg)  # talker_graph.py:163-167 raises RuntimeError for over-long input
        raise Fq3Error(f"fq3 error {-rc}: {msg}")
