"""ctypes binding of libinfltm.so (include/infltm.h).  No CPU fallback: if the library is missing or
a call fails, this raises."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libinfltm.so")
_lib = None

c_f32p = C.c_void_p
c_i32p = C.c_void_p
c_f64p = C.c_void_p
c_u8p = C.c_void_p


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("lda", C.c_int64), ("strideA", C.c_int64), ("a_kmajor", C.c_int),
        ("B", C.c_void_p), ("ldb", C.c_int64), ("strideB", C.c_int64), ("b_kmajor", C.c_int),
        ("B2", C.c_void_p), ("ldb2", C.c_int64), ("strideB2", C.c_int64), ("K1", C.c_int),
        ("bias", C.c_void_p),
        ("C", C.c_void_p), ("ldc", C.c_int64), ("strideC", C.c_int64),
        ("M", C.c_int), ("Nc", C.c_int), ("K", C.c_int), ("batch", C.c_int),
        ("precision", C.c_int), ("impl", C.c_int),
        ("CT", C.c_void_p), ("ct_cols", C.c_int), ("ct_group", C.c_int),
        ("c_group", C.c_int), ("c_group_stride", C.c_int64), ("bias_stride", C.c_int64),
        ("round_tf32", C.c_int), ("ab_fp16", C.c_int),
        ("a_group", C.c_int), ("a_group_stride", C.c_int64), ("c_fp16", C.c_int),
        ("C_lo", C.c_void_p), ("max_ctas", C.c_int),
    ]


class RectStepArgs(C.Structure):
    _fields_ = [
        ("Bv", C.c_int), ("L", C.c_int), ("T", C.c_int), ("e", C.c_int), ("N", C.c_int), ("Q", C.c_int),
        ("H", C.c_int), ("d", C.c_int), ("S", C.c_int), ("splits", C.c_int), ("sticky", C.c_int),
        ("precision", C.c_int), ("gemm_impl", C.c_int),
        ("seg_ptr0", C.c_void_p), ("seg_mem0", C.c_void_p), ("g0", C.c_void_p),
        ("seg_ptr1", C.c_void_p), ("seg_mem1", C.c_void_p), ("g1", C.c_void_p),
        ("jb", C.c_void_p), ("tb", C.c_void_p), ("bins", C.c_void_p), ("bin2basis", C.c_void_p),
        ("idx_uniform", C.c_void_p),
        ("W", C.c_void_p), ("W_out", C.c_float),
        ("Wkv", C.c_void_p), ("bkv", C.c_void_p),
        ("B_past", C.c_void_p), ("B_new", C.c_void_p),
        ("hist_part", C.c_void_p),
        ("xpart", C.c_void_p), ("KV", C.c_void_p), ("Kt", C.c_void_p), ("V", C.c_void_p),
        ("b_draw", C.c_void_p), ("idx", C.c_void_p), ("ts", C.c_void_p),
        ("p", C.c_void_p), ("scores", C.c_void_p),
        ("k_dev", C.c_void_p), ("q_dev", C.c_void_p), ("u_dev", C.c_void_p), ("new_doc_dev", C.c_void_p),
        ("ctx_dev", C.c_void_p),
        ("prof_events", C.c_void_p * 10),
        ("X", C.c_void_p), ("c_none", C.c_float),
        ("B_half", C.c_void_p), ("Wkv_half", C.c_void_p),
        ("KV_past", C.c_void_p), ("jf", C.c_int), ("proj_precision", C.c_int),
        ("attn_part", C.c_void_p),
        ("kv_half", C.c_int), ("X16", C.c_void_p),
        ("binned", C.c_int), ("xb_rows", C.c_int),
        ("fbin_ptr", C.c_void_p), ("seg_ptr1b", C.c_void_p), ("seg_mem1b", C.c_void_p),
        ("gemm_ctas", C.c_int),
        ("lengths", C.c_void_p), ("frame_offs", C.c_void_p), ("frames", C.c_int), ("n_idle", C.c_int),
        ("bank_seg_ptr0", C.c_void_p), ("bank_seg_mem0", C.c_void_p), ("bank_g0", C.c_void_p),
        ("bank_seg_ptr1", C.c_void_p), ("bank_seg_mem1", C.c_void_p), ("bank_g1", C.c_void_p),
        ("hist_keep", C.c_void_p),
        ("k_dtype", C.c_int),
        ("k_ptrs", C.c_void_p),
    ]


class Overlap(C.Structure):
    _fields_ = [
        ("main_stream", C.c_void_p), ("side_stream", C.c_void_p), ("compute_stream", C.c_void_p),
        ("ev_fork_pool", C.c_void_p), ("ev_pooled_cur", C.c_void_p), ("ev_pooled_next", C.c_void_p),
        ("ev_fork", C.c_void_p), ("ev_join", C.c_void_p),
        ("k_next", C.c_void_p), ("xpart_next", C.c_void_p), ("pool_ctas", C.c_int),
        ("next_binned", C.c_int),
        ("next_lengths", C.c_void_p), ("next_offs", C.c_void_p), ("next_frames", C.c_int), ("next_splits", C.c_int),
        ("next_dtype", C.c_int),
        ("next_ptrs", C.c_void_p),
    ]


_I, _F, _P, _L = C.c_int, C.c_float, C.c_void_p, C.c_int64
_SIGS = {
    "ltm_version": (C.c_int, []),
    "ltm_last_error": (C.c_char_p, []),
    "ltm_device_check": (C.c_int, []),
    "ltm_pool_mean": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_convert": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_fold_sample_columns": (C.c_int, [_P, _L, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_cont_attn_gauss_tc16": (C.c_int, [_P, _P, _P, _L, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_split_half3": (C.c_int, [_P, _P, _L, _I, _I, _P]),
    "ltm_pool_bins": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_16": (C.c_int, [_P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_16_grid": (C.c_int, [_P, _I, _P, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_grid": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_ragged": (C.c_int, [_P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_ptrs": (C.c_int, [_P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_pool_mean_convert_ragged": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_sticky_hist_rect": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "ltm_sticky_hist_rect_tiles": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "ltm_density_rect": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "ltm_sticky_hist_gauss": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "ltm_resample": (C.c_int, [_P, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _P]),
    "ltm_consolidate_rect": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_consolidate_rect_h": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_consolidate_rect_kv": (C.c_int, [_P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I,
                                          _I, _I, _I, _I, _I, _I, _P]),
    "ltm_gemm": (C.c_int, [C.POINTER(GemmArgs), _P]),
    "ltm_gemm_extents": (C.c_int, [C.POINTER(GemmArgs), _P, _P, _P]),
    "ltm_project_kv": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_project_kv_t": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "ltm_project_kv_r": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_attn_fast_supported": (C.c_int, [_I, _I]),
    "ltm_attn_tc_supported": (C.c_int, [_I, _I]),
    "ltm_cont_attn_rect_tc": (C.c_int, [_P, _P, _P, _L, _P, _P, _F, _F, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_attn_tc_split_supported": (C.c_int, [_I, _I]),
    "ltm_attn_tc_split_workspace_floats": (C.c_int64, [_I, _I, _I]),
    "ltm_cont_attn_rect_tc_split": (C.c_int, [_P, _P, _P, _L, _P, _P, _F, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I,
                                              _P]),
    "ltm_cont_attn_rect_tc16": (C.c_int, [_P, _P, _P, _L, _P, _P, _F, _F, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_cont_attn_rect_tc16_split": (C.c_int, [_P, _P, _P, _L, _P, _P, _F, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I,
                                                _I, _P]),
    "ltm_cont_attn_rect_t": (C.c_int, [_P, _P, _P, _L, _P, _F, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_cont_attn_gauss_t": (C.c_int, [_P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_cont_attn_rect": (C.c_int, [_P, _P, _P, _F, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_cont_attn_gauss": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ltm_kl_gauss": (C.c_int, [_P, _P, _F, _F, _P, _L, _P]),
    "ltm_rbf_eval": (C.c_int, [_P, _P, _P, _P, _P, _L, _I, _I, _P]),
    "ltm_ridge_workspace_doubles": (C.c_int64, [_I, _I]),
    "ltm_ridge_solve": (C.c_int, [_P, _I, _I, _I, _P, _P, _I, C.c_double, _P, _P, _L, _P, _P]),
    "ltm_gather_rows": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "ltm_softmax_rows": (C.c_int, [_P, _P, _I, _I, _I, _F, _P]),
    "ltm_softmax_rows_h": (C.c_int, [_P, _P, _P, _I, _I, _I, _F, _P]),
    "ltm_softmax_rows_h_len": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _F, _P]),
    "ltm_to_half": (C.c_int, [_P, _P, _L, _P]),
    "ltm_blend": (C.c_int, [_P, _P, _F, _P, _L, _P]),
    "ltm_event_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "ltm_event_create_sync": (C.c_int, [C.POINTER(C.c_void_p)]),
    "ltm_event_record": (C.c_int, [_P, _P]),
    "ltm_stream_wait_event": (C.c_int, [_P, _P]),
    "ltm_event_elapsed_ms": (C.c_int, [_P, _P, C.POINTER(C.c_float)]),
    "ltm_event_destroy": (C.c_int, [_P]),
    "ltm_rect_step": (C.c_int, [C.POINTER(RectStepArgs), _P, _P, _P, _P, _P, _P]),
    "ltm_rect_step_overlap": (C.c_int, [C.POINTER(RectStepArgs), C.POINTER(Overlap), _P, _P, _P, _P]),
    "ltm_rect_step_host": (C.c_int, [C.POINTER(RectStepArgs), _P, _P, _P, _P, _P, _P]),
}
EXPORTED = tuple(_SIGS)


def lib():
    """The loaded library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m infinite_video_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback for the LTM consolidation path.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().ltm_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libinfltm {what} failed (rc={rc}): {msg}")


def ptr(t):
    """Device (or pinned host) pointer of a contiguous tensor; None -> NULL."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("libinfltm needs contiguous tensors")
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ValueError("libinfltm operates on CUDA tensors only (no CPU fallback)")
