"""ctypes binding of ``libneutts_b200.so`` (the C-ABI declared in ``include/neutts_b200.h``).

There is no CPU fallback: if the shared object is missing or a call fails, the error is
raised to the caller (``NT_ERR_INVALID`` -> ValueError, everything else -> RuntimeError).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libneutts_b200.so"

NT_BF16, NT_TF32 = 0, 1
NT_ACT_NONE, NT_ACT_SILU, NT_ACT_SWIGLU = 0, 1, 2


class GemmArgs(C.Structure):
    _fields_ = [
        ("dtype", C.c_int), ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("A", C.c_void_p), ("lda", C.c_int64), ("W", C.c_void_p), ("ldw", C.c_int64),
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("ldr", C.c_int64), ("act", C.c_int),
        ("out_f32", C.c_void_p), ("out_bf16", C.c_void_p), ("ldc", C.c_int64),
        ("valid_period", C.c_int), ("valid_len", C.c_int),
    ]


class LMConfig(C.Structure):
    _fields_ = [
        ("vocab_size", C.c_int), ("hidden", C.c_int), ("inter", C.c_int), ("n_layers", C.c_int),
        ("n_heads", C.c_int), ("n_kv_heads", C.c_int), ("head_dim", C.c_int),
        ("rms_eps", C.c_float), ("rope_theta", C.c_float),
        ("max_batch", C.c_int), ("max_ctx", C.c_int), ("page_size", C.c_int), ("num_pages", C.c_int),
        ("max_prefill_tokens", C.c_int),
    ]


class LMWeights(C.Structure):
    _fields_ = [
        ("embed", C.c_void_p), ("lm_head", C.c_void_p), ("final_norm", C.c_void_p),
        ("ln1", C.POINTER(C.c_void_p)), ("wqkv", C.POINTER(C.c_void_p)), ("bqkv", C.POINTER(C.c_void_p)),
        ("wo", C.POINTER(C.c_void_p)), ("ln2", C.POINTER(C.c_void_p)), ("wgu", C.POINTER(C.c_void_p)),
        ("wd", C.POINTER(C.c_void_p)),
    ]


class LMState(C.Structure):
    _fields_ = [
        ("kv_pages", C.c_void_p), ("page_table", C.c_void_p), ("seq_lens", C.c_void_p),
        ("cur_token", C.c_void_p), ("out_tokens", C.c_void_p), ("n_generated", C.c_void_p),
        ("done", C.c_void_p), ("max_new", C.c_int32),
    ]


class Sampling(C.Structure):
    _fields_ = [
        ("eos_id", C.c_int32), ("min_new_tokens", C.c_int32), ("max_new_tokens", C.c_int32),
        ("top_k", C.c_int32), ("temperature", C.c_float), ("seed", C.c_uint64), ("greedy", C.c_int32),
        ("forced", C.c_void_p), ("limits", C.c_void_p), ("slot_base", C.c_int32),
    ]


class CodecConfig(C.Structure):
    _fields_ = [
        ("hidden", C.c_int), ("depth", C.c_int), ("heads", C.c_int), ("head_dim", C.c_int),
        ("mlp_hidden", C.c_int), ("groups", C.c_int), ("embed_kernel", C.c_int),
        ("n_fft", C.c_int), ("hop", C.c_int), ("fsq_levels", C.c_int), ("fsq_dims", C.c_int),
        ("norm_eps", C.c_float), ("rope_base", C.c_float), ("mag_clip", C.c_float),
        ("rope_time_axis", C.c_int), ("max_batch", C.c_int), ("max_frames", C.c_int), ("precision", C.c_int),
    ]


_PP = C.POINTER(C.c_void_p)


class CodecWeights(C.Structure):
    _fields_ = [
        ("fsq_w", C.c_void_p), ("fsq_b", C.c_void_p), ("embed_w", C.c_void_p), ("embed_b", C.c_void_p),
        ("rn_n1w", _PP), ("rn_n1b", _PP), ("rn_c1w", _PP), ("rn_c1b", _PP),
        ("rn_n2w", _PP), ("rn_n2b", _PP), ("rn_c2w", _PP), ("rn_c2b", _PP),
        ("att_norm", _PP), ("wqkv", _PP), ("wproj", _PP), ("ffn_norm", _PP), ("fc1", _PP), ("fc2", _PP),
        ("final_ln_w", C.c_void_p), ("final_ln_b", C.c_void_p), ("head_w", C.c_void_p), ("head_b", C.c_void_p),
        ("idft_basis", C.c_void_p),
    ]


# every symbol include/neutts_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "nt_last_error", "nt_abi_version", "nt_launch_count", "nt_gemm",
    "nt_lm_workspace_bytes", "nt_lm_create", "nt_lm_destroy", "nt_lm_prefill", "nt_lm_decode", "nt_lm_head_gemv",
    "nt_lm_debug_set_layers", "nt_lm_debug_ptr", "nt_lm_debug_set_profile", "nt_debug_launch_chain",
    "nt_codec_workspace_bytes", "nt_codec_create", "nt_codec_destroy", "nt_codec_decode",
    "nt_codec_decode_ragged",
    "nt_op_rmsnorm", "nt_op_topk_sample",
]

_lib = None


def lib() -> C.CDLL:
    """Load the shared object (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = LIB_PATH
    if os.environ.get("NT_LIB_PATH"):      # A/B measurements against an older build of the library (profiles/ab/)
        path = Path(os.environ["NT_LIB_PATH"])
    if not path.exists():
        raise RuntimeError(
            f"{path} is missing: build it with `python -m neutts_air_b200.build` "
            "(nvcc, sm_100a). neutts_air_b200 has no CPU or PyTorch fallback.")
    L = C.CDLL(str(path))
    L.nt_last_error.restype = C.c_char_p
    L.nt_abi_version.restype = C.c_int
    L.nt_launch_count.restype = C.c_uint64
    L.nt_gemm.argtypes = [C.POINTER(GemmArgs), C.c_void_p]
    L.nt_lm_workspace_bytes.restype = C.c_size_t
    L.nt_lm_workspace_bytes.argtypes = [C.POINTER(LMConfig)]
    L.nt_lm_create.argtypes = [C.POINTER(LMConfig), C.POINTER(LMWeights), C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.nt_lm_destroy.argtypes = [C.c_void_p]
    L.nt_lm_prefill.argtypes = [C.c_void_p, C.POINTER(LMState), C.c_void_p, C.POINTER(C.c_int32), C.c_int,
                                C.POINTER(Sampling), C.c_void_p, C.c_void_p]
    L.nt_lm_decode.argtypes = [C.c_void_p, C.POINTER(LMState), C.c_int, C.c_int, C.POINTER(Sampling), C.c_void_p, C.c_void_p]
    L.nt_lm_head_gemv.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.nt_lm_debug_set_layers.argtypes = [C.c_void_p, C.c_int]
    L.nt_lm_debug_ptr.restype = C.c_void_p
    L.nt_lm_debug_ptr.argtypes = [C.c_void_p, C.c_char_p]
    L.nt_lm_debug_set_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.nt_debug_launch_chain.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.nt_codec_workspace_bytes.restype = C.c_size_t
    L.nt_codec_workspace_bytes.argtypes = [C.POINTER(CodecConfig)]
    L.nt_codec_create.argtypes = [C.POINTER(CodecConfig), C.POINTER(CodecWeights), C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.nt_codec_destroy.argtypes = [C.c_void_p]
    L.nt_codec_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.nt_codec_decode_ragged.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_int, C.c_void_p, C.c_void_p]
    L.nt_op_rmsnorm.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nt_op_topk_sample.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(Sampling), C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    _lib = L
    return L


def check(rc: int) -> None:
    """Map a C-ABI status to the reference's error convention (Python exceptions,
    neutts/neutts.py:196,210,295)."""
    if rc == 0:
        return
    msg = lib().nt_last_error().decode(errors="replace")
    if rc == -1:
        raise ValueError(f"neutts_b200: {msg}")
    raise RuntimeError(f"neutts_b200 (status {rc}): {msg}")


def ptr_array(tensors) -> "C.Array":
    """Host array of device pointers (keeps no reference: callers hold the tensors)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def current_stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
