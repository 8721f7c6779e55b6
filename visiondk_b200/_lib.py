"""ctypes binding of libvdk_b200.so — the only way Python reaches the CUDA kernels.

There is no CPU fallback anywhere in this package: if the library is missing it must be built
(`python -m visiondk_b200.build`), and every compute entry point raises RuntimeError when the C ABI
returns a non-zero status (e.g. no sm_100 device).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libvdk_b200.so"

VDK_OK = 0
VDK_ERR_INVALID, VDK_ERR_CUDA, VDK_ERR_WORKSPACE, VDK_ERR_OVERFLOW = -1, -2, -3, -4
DTYPE_BF16, DTYPE_FP16, DTYPE_FP32 = 0, 1, 2
EPI_NONE, EPI_GELU, EPI_SCALE_RESIDUAL, EPI_LAYERNORM, EPI_MUL_GELU_GRAD = 0, 1, 2, 3, 4


class HeadDesc(C.Structure):
    _fields_ = [("kind", C.c_int), ("batch", C.c_int), ("feat_dim", C.c_int), ("num_class", C.c_int),
                ("margin_arc", C.c_float), ("margin_am", C.c_float), ("scale", C.c_float),
                ("margin", C.c_float), ("gamma", C.c_float), ("label_smooth", C.c_float),
                ("mv_weight", C.c_float), ("is_am", C.c_int)]


class TopkPlan(C.Structure):
    _fields_ = [
        ("n_query", C.c_int64),
        ("n_gallery", C.c_int64),
        ("dim", C.c_int),
        ("k", C.c_int),
        ("cand_capacity", C.c_int),
        ("carry_capacity", C.c_int),
        ("n_stages", C.c_int),
        ("dense_mask", C.c_int),
        ("stage_end", C.c_int64 * 8),
    ]


_p, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t


class ImageDesc(C.Structure):
    _fields_ = [("offset", C.c_int64), ("width", C.c_int), ("height", C.c_int)]


class ProfTotal(C.Structure):
    _fields_ = [("launches", C.c_longlong), ("ms", C.c_double), ("flops", C.c_double), ("bytes", C.c_double)]


PROF_CATEGORIES = ("gemm", "depthwise", "attention", "score_filter", "other")


class GemmDesc(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("D", C.c_void_p),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("lda", C.c_int), ("ldb", C.c_int), ("ldd", C.c_int),
        ("in_dtype", C.c_int), ("out_dtype", C.c_int), ("epilogue", C.c_int),
        ("bias", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p), ("residual", C.c_void_p),
        ("ldr", C.c_int), ("ln_eps", C.c_float), ("split_k", C.c_int), ("split_stride", C.c_longlong), ("aux_out", C.c_void_p), ("trans_a", C.c_int),
        ("trans_b", C.c_int),
    ]


# name -> (restype, argtypes); must list every symbol include/vdk_b200.h declares (tests check this).
SIGNATURES = {
    "vdk_version": (_i, []),
    "vdk_struct_sizes": (_i, [_p, _i]),
    "vdk_last_error_string": (C.c_char_p, []),
    "vdk_device_check": (_i, []),
    "vdk_preprocess_workspace_bytes": (_sz, [C.POINTER(ImageDesc), _i, _i]),
    "vdk_preprocess_resize_pad_normalize": (_i, [_p, C.POINTER(ImageDesc), _i, _i, C.POINTER(C.c_float), C.POINTER(C.c_float), _p, _p,
                                                 _sz, _p]),
    "vdk_prof_begin": (_i, []),
    "vdk_prof_end": (_i, [C.POINTER(ProfTotal), _i]),
    "vdk_gemm": (_i, [_p, _p]),
    "vdk_gemm_effective_splits": (_i, [_i, _i]),
    "vdk_dwconv7_ln": (_i, [_p, _i, _i, _i, _i, _p, _p, _p, _p, C.c_float, _p, _p]),
    "vdk_layernorm_patchify": (_i, [_p, _i, _i, _i, _i, _p, _p, C.c_float, _i, _p, _p]),
    "vdk_dwconv7": (_i, [_i, _p, _i, _i, _i, _i, _p, _p, _p, _p, C.c_float, _p, _p, _p, _p]),
    "vdk_dwconv7_wgrad": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "vdk_layernorm_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _p, _i, _p, _p, _p, _p, _p]),
    "vdk_batchnorm_train_fwd": (_i, [_p, _i, _i, _i, _p, _p, C.c_float, C.c_float, _p, _p, _p, _p, _p, _p]),
    "vdk_batchnorm_train_bwd": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
    "vdk_convnext_pack": (_i, [_p, _p, _p]),
    "vdk_convnext_pack_flip": (_i, [_p, _p]),
    "vdk_convnext_train_workspace_bytes": (_sz, [_p, _i]),
    "vdk_convnext_train_forward": (_i, [_p, _p, _p, _i, C.c_float, _p, _p, _sz, _p]),
    "vdk_convnext_train_backward": (_i, [_p, _p, _p, _p, _i, _p, _sz, _p]),
    "vdk_convnext_train_backward_units": (_i, [_p]),
    "vdk_convnext_train_backward_range": (_i, [_p, _p, _p, _p, _i, _p, _sz, _p, _i, _i]),
    "vdk_vit_workspace_bytes": (_sz, [_p, _i]),
    "vdk_vit_pack": (_i, [_p, _p, _p]),
    "vdk_vit_train_workspace_bytes": (_sz, [_p, _i]),
    "vdk_vit_train_forward": (_i, [_p, _p, _p, _i, C.c_float, _p, _p, _sz, _p]),
    "vdk_vit_train_backward": (_i, [_p, _p, _p, _p, _i, _p, _sz, _p]),
    "vdk_vit_train_backward_units": (_i, [_p]),
    "vdk_vit_train_backward_range": (_i, [_p, _p, _p, _p, _i, _p, _sz, _p, _i, _i]),
    "vdk_attention_fwd_lse": (_i, [_p, _i, _i, _i, _i, _p, _p, _p]),
    "vdk_attention_bwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "vdk_attention_bwd_tc_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "vdk_attention_bwd_tc": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _sz, _p]),
    "vdk_vit_forward": (_i, [_p, _p, _i, _i, _p, _p, _sz, _p]),
    "vdk_attention_fwd": (_i, [_p, _i, _i, _i, _i, _p, _p]),
    "vdk_convnext_workspace_bytes": (_sz, [_p, _i]),
    "vdk_convnext_forward": (_i, [_p, _p, _i, _i, _p, _p, _sz, _p]),
    "vdk_head_workspace_bytes": (_sz, [_p]),
    "vdk_head_forward": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "vdk_head_backward": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "vdk_grad_sumsq_workspace_bytes": (_sz, []),
    "vdk_grad_sumsq": (_i, [_p, _i64, _p, _i, _p, _sz, _p]),
    "vdk_sgd_clip_ema_step": (_i, [_p, _p, _p, _p, _i64, _p, C.c_float, C.c_float, C.c_float, C.c_float, _i, C.c_float,
                                   C.c_float, _i, _p]),
    "vdk_ema_update": (_i, [_p, _p, _i64, C.c_float, C.c_float, _p]),
    "vdk_gemm_tn": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _i, _p]),
    "vdk_rows_prepare": (_i, [_p, _i64, _i, _i, _p, _p, _p, _p, _p]),
    "vdk_topk_plan_default": (_i, [C.POINTER(TopkPlan), _i64, _i64, _i, _i]),
    "vdk_topk_workspace_bytes": (_sz, [C.POINTER(TopkPlan)]),
    "vdk_ip_topk": (_i, [C.POINTER(TopkPlan), _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "vdk_ip_topk_filter": (_i, [C.POINTER(TopkPlan), _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "vdk_ip_topk_filter_stages": (_i, [C.POINTER(TopkPlan), _p, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "vdk_ip_topk_rerank": (_i, [C.POINTER(TopkPlan), _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "vdk_ip_topk_rank_sketch": (_i, [C.POINTER(TopkPlan), _i, C.POINTER(C.c_int32), _i, _p, _p, _sz, _p]),
    "vdk_topk_bound_from_sketches": (_i, [_p, _i, _i64, C.POINTER(C.c_int32), _i, _i, _p, _p]),
    "vdk_topk_row_flags": (_i, [C.POINTER(TopkPlan), _p, _sz, C.POINTER(C.c_void_p)]),
    "vdk_score_range": (_i, [C.POINTER(TopkPlan), _p, _p, _i64, _i64, _i, _p, _sz, _p]),
    "vdk_reduce_max": (_i, [_p, _i64, _p, _p]),
    "vdk_topk_merge": (_i, [_p, _p, _i, _i64, _i, _p, _p, _p]),
    "vdk_topk_pack": (_i, [_p, _p, _i64, _p, _p]),
    "vdk_topk_merge_packed": (_i, [_p, _i, _i64, _i, _p, _p, _p]),
    "vdk_ip_exact_pairs": (_i, [_p, _p, _i, _p, _p, _i64, _p, _p]),
    "vdk_ip_topk_exhaustive_workspace_bytes": (_sz, [_i64]),
    "vdk_ip_topk_exhaustive": (_i, [_p, _i64, _p, _i64, _i, _i, _i64, _p, _p, _p, _sz, _p]),
}

_lib = None


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Loads libvdk_b200.so and types its symbols.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -m visiondk_b200.build` "
            "(there is no CPU fallback for the hot path)")
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().vdk_last_error_string().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != VDK_OK:
        raise RuntimeError(f"{what} failed (status {rc}): {last_error()}")


def require_device() -> None:
    check(load().vdk_device_check(), "vdk_device_check")


class profile:
    """`with _lib.profile() as p: step()` -> p.totals = {category: {launches, ms, flops, bytes}} (vdk_prof_begin / vdk_prof_end)."""

    def __enter__(self):
        check(load().vdk_prof_begin(), "vdk_prof_begin")
        self.totals = None
        return self

    def __exit__(self, *exc):
        arr = (ProfTotal * len(PROF_CATEGORIES))()
        rc = load().vdk_prof_end(arr, len(PROF_CATEGORIES))
        self.totals = {name: {"launches": int(arr[i].launches), "ms": float(arr[i].ms), "flops": float(arr[i].flops),
                              "bytes": float(arr[i].bytes)} for i, name in enumerate(PROF_CATEGORIES)}
        if exc[0] is None:
            check(rc, "vdk_prof_end")
        return False


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
