"""ctypes binding of libits_b200.so (include/its_b200.h).

The library is the product: if it is missing or a symbol is absent this module
raises — there is no fallback implementation anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ITS_LIB: another build of the same ABI (A/B measurements of a kernel change on one box)
LIB_PATH = os.environ.get("ITS_LIB") or os.path.join(_HERE, "libits_b200.so")

MAX_SRC, MAX_TAPS, MAX_PHASES = 3, 36, 4

SYMBOLS = [
    "its_version", "its_last_error_string", "its_device_sm_count", "its_abi_sizeof", "its_ddpm_step",
    "its_philox_normal", "its_step_advance", "its_time_embed", "its_embed_rows", "its_linear",
    "its_group_norm", "its_conv_head", "its_conv_tail", "its_conv_igemm", "its_softmax_rows",
    "its_attention_small", "its_image_stats", "its_candidate_scores", "its_argmax_first",
    "its_group_norm_apply", "its_conv_stats_parts", "its_set_pdl", "its_attention_fused", "its_head_patches",
    "its_attention_flash", "its_attention_group", "its_conv_gn_sync_words",
    "its_f32_nchw_to_nhwc", "its_f32_conv2d", "its_f32_group_norm", "its_f32_attention",
    "its_topk_first", "its_ddpm_step_x0", "its_path_expand", "its_topk_first_segmented",
    "its_level_inputs", "its_denoise_scores", "its_resample_systematic",
]


class Src(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("c_pitch", C.c_int32), ("c_off", C.c_int32), ("C", C.c_int32),
                ("H", C.c_int32), ("W", C.c_int32), ("stride", C.c_int32), ("bcast", C.c_int32),
                ("fp16", C.c_int32)]


class Phase(C.Structure):
    _fields_ = [("ntaps", C.c_int32), ("w_k0", C.c_int32), ("py", C.c_int32), ("px", C.c_int32),
                ("src", C.c_int8 * MAX_TAPS), ("dy", C.c_int8 * MAX_TAPS), ("dx", C.c_int8 * MAX_TAPS)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("src", Src * MAX_SRC), ("nsrc", C.c_int32),
        ("phase", Phase * MAX_PHASES), ("nphases", C.c_int32),
        ("B", C.c_int32), ("Hm", C.c_int32), ("Wm", C.c_int32),
        ("w", C.c_void_p), ("w_pitch", C.c_int32), ("w_batch_stride", C.c_int64), ("Cout", C.c_int32),
        ("out", C.c_void_p), ("out_fp32", C.c_int32),
        ("Hout", C.c_int32), ("Wout", C.c_int32), ("out_scale", C.c_int32),
        ("out_c_pitch", C.c_int32), ("out_c_off", C.c_int32),
        ("bias", C.c_void_p),
        ("vec", C.c_void_p), ("vec_stride", C.c_int32), ("vec_off", C.c_int32),
        ("vec2", C.c_void_p), ("vec2_stride", C.c_int32), ("vec2_off", C.c_int32),
        ("res", C.c_void_p), ("res_c_pitch", C.c_int32), ("res_c_off", C.c_int32),
        ("alpha", C.c_float), ("bn", C.c_int32),
        ("out_nchw", C.c_int32), ("splits", C.c_int32), ("ws", C.c_void_p), ("ws_elems", C.c_int64),
        ("cluster", C.c_int32), ("dbg", C.c_void_p),
        ("stats", C.c_void_p), ("stats_parts", C.c_int32), ("schedule", C.c_int32),
        ("out_fp16", C.c_int32),
        ("gn_out", C.c_void_p), ("gn_c_pitch", C.c_int32), ("gn_gamma", C.c_void_p), ("gn_beta", C.c_void_p),
        ("gn_groups", C.c_int32), ("gn_eps", C.c_float), ("gn_silu", C.c_int32), ("gn_only", C.c_int32),
        ("gn_sync", C.c_void_p),
    ]


_lib = None


def lib() -> C.CDLL:
    """dlopen the extension (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first; "
            "its_b200 has no CPU or torch fallback")
    L = C.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(L, s)]
    if missing:
        raise RuntimeError(f"libits_b200.so lacks symbols {missing}; rebuild it")
    vp, i32, i64, u64, f32, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double
    L.its_version.restype = i32
    L.its_last_error_string.restype = C.c_char_p
    L.its_device_sm_count.argtypes = [C.POINTER(C.c_int)]
    L.its_abi_sizeof.argtypes = [i32]
    L.its_set_pdl.argtypes = [i32]
    L.its_ddpm_step.argtypes = [vp, vp, vp, vp, i64, i64, i64, vp, vp, f64, u64, i64, vp, i32, vp]
    L.its_ddpm_step_x0.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, vp, vp, vp, f64, u64, vp, vp, i32, vp]
    L.its_path_expand.argtypes = [vp, vp, vp, i32, i32, i64, i64, i64, i64, f32, f32, vp, u64, i64, i32, vp]
    L.its_philox_normal.argtypes = [vp, vp, i32, f32, i64, i64, u64, i64, i32, vp]
    L.its_step_advance.argtypes = [vp, i32, vp]
    L.its_time_embed.argtypes = [vp, vp, vp, vp, i32, i32, vp]
    L.its_embed_rows.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
    L.its_linear.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    L.its_group_norm.argtypes = [vp, vp, i32, vp, i32, vp, vp, i32, i32, i32, f32, i32, vp, i32, i32, vp]
    L.its_group_norm_apply.argtypes = [vp, vp, i32, vp, i32, vp, i32, vp, i32, vp, vp, i32, i32, i32, f32, i32, i32, vp]
    L.its_conv_stats_parts.argtypes = [C.POINTER(ConvDesc)]
    L.its_conv_gn_sync_words.argtypes = [C.POINTER(ConvDesc)]
    L.its_conv_head.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    L.its_head_patches.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp]
    L.its_conv_tail.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    L.its_conv_igemm.argtypes = [C.POINTER(ConvDesc), i32, vp]
    L.its_softmax_rows.argtypes = [vp, vp, i64, i32, vp]
    L.its_attention_small.argtypes = [vp, vp, i32, i32, i32, f32, vp]
    L.its_attention_fused.argtypes = [vp, vp, vp, vp, i32, i32, i32, f32, vp]
    L.its_attention_flash.argtypes = [vp, vp, vp, vp, i32, i32, i32, f32, vp]
    L.its_attention_group.argtypes = [vp, vp, vp, i32, i32, i32, f32, vp]
    L.its_f32_nchw_to_nhwc.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp]
    L.its_f32_conv2d.argtypes = [vp, vp, i32, vp, i32, vp, vp, vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]
    L.its_f32_group_norm.argtypes = [vp, vp, i32, vp, i32, vp, vp, i32, i32, i32, f32, i32, vp]
    L.its_f32_attention.argtypes = [vp, vp, i32, i32, i32, f32, vp]
    L.its_image_stats.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    L.its_candidate_scores.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    L.its_argmax_first.argtypes = [vp, vp, vp, i32, vp]
    L.its_topk_first.argtypes = [vp, vp, vp, i32, i32, vp]
    L.its_topk_first_segmented.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    L.its_level_inputs.argtypes = [vp, vp, vp, vp, i32, i32, i64, vp]
    L.its_denoise_scores.argtypes = [vp, vp, vp, vp, i32, i32, i32, i64, vp]
    L.its_resample_systematic.argtypes = [vp, vp, vp, vp, vp, f32, i32, i32, u64, i64, i32, vp]
    for s in SYMBOLS:
        if s not in ("its_version", "its_last_error_string"):
            getattr(L, s).restype = i32
    for which, struct in ((0, ConvDesc), (1, Src), (2, Phase)):
        if L.its_abi_sizeof(which) != C.sizeof(struct):
            raise RuntimeError(f"ctypes layout of {struct.__name__} ({C.sizeof(struct)} B) does not match "
                               f"the library ({L.its_abi_sizeof(which)} B)")
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    """Raise RuntimeError with the library's message on a non-zero return code."""
    if rc != 0:
        msg = lib().its_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"libits_b200 {what} failed (code {rc}): {msg}")


def require_cuda():
    """The product path runs on a CUDA device only."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("its_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    lib()


def stream_ptr(device=None) -> int:
    """The caller's current stream.  With `device` (a tensor's device) the stream of THAT device; the library
    launches into the current CUDA context, so a tensor on another device than the current one is refused."""
    import torch
    if device is not None and device.type == "cuda":
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if idx != torch.cuda.current_device():
            raise RuntimeError(f"its_b200: tensor on cuda:{idx} but the current device is cuda:"
                               f"{torch.cuda.current_device()} (wrap the call in torch.cuda.device(...))")
    return torch.cuda.current_stream().cuda_stream
