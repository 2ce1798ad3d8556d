"""ctypes binding of include/rgbmp.h.  Fails loudly when the CUDA library is absent."""
from __future__ import annotations

import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RGBMP_LIB") or os.path.join(HERE, "librgbmp.so")   # RGBMP_LIB: A/B builds (tools/)

F32, BF16 = 0, 1
EINVAL, EALIGN, ERANGE, EWORKSPACE = -1, -2, -3, -4

c_i32, c_i64, c_f32, c_vp, c_sz = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t


class GraphStruct(C.Structure):
    """rgbmp_graph_t"""
    _fields_ = [("n_rows", c_i64), ("n_cols", c_i64), ("nnz", c_i64), ("rowptr", c_vp), ("col", c_vp),
                ("chunk", c_i32), ("long_chunk", c_i32), ("n_long", c_i64), ("n_items", c_i64),
                ("long_rows", c_vp), ("long_item_ptr", c_vp), ("item_long", c_vp), ("item_start", c_vp),
                ("row_order", c_vp), ("col_tagged", c_i32)]


class Epilogue(C.Structure):
    """rgbmp_epilogue_t"""
    _fields_ = [("row_scale", c_vp), ("row_div", c_i32), ("reset_mask", c_vp), ("reset_val", c_vp),
                ("ld_reset", c_i64), ("reset_when", c_i32), ("a", c_f32), ("b", c_f32), ("T", c_vp),
                ("ldt", c_i64), ("clamp", c_i32), ("lo", c_f32), ("hi", c_f32), ("out2_scale", c_vp),
                ("Y2", c_vp), ("ldy2", c_i64), ("acc_in", c_vp), ("ld_acc", c_i64), ("skip_empty", c_i32),
                ("peer_out", c_vp * 8), ("n_peers", c_i32), ("peer_row0", c_i64), ("ld_peer", c_i64),
                ("row_map", c_vp)]


class DropoutStruct(C.Structure):
    """rgbmp_dropout_t"""
    _fields_ = [("seed", c_vp), ("eid", c_vp), ("eid_t", c_vp), ("thresh", C.c_uint32), ("scale", c_f32)]


class SgatSampleStruct(C.Structure):
    """rgbmp_sgat_sample_t"""
    _fields_ = [("seed", c_vp), ("eid", c_vp), ("eid_t", c_vp), ("keep_thresh", C.c_uint64)]


_lib = None


def lib():
    """Load librgbmp.so once; raise (never fall back) when it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"rgb-experiment_b200: {LIB_PATH} is missing -- build it with "
            "`python rgb-experiment_b200/build.py` (nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    GP, EP, DP = C.POINTER(GraphStruct), C.POINTER(Epilogue), C.POINTER(DropoutStruct)
    SP = C.POINTER(SgatSampleStruct)
    sig = {
        "rgbmp_version": (C.c_int, []),
        "rgbmp_last_error": (C.c_char_p, []),
        "rgbmp_edge_edit_workspace_bytes": (c_sz, [c_i64, c_i64]),
        "rgbmp_edge_edit": (C.c_int, [c_vp, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_csr_build_workspace_bytes": (c_sz, [c_i64, c_i64]),
        "rgbmp_csr_build": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_degree_norm": (C.c_int, [c_vp, c_i64, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_gcn_edge_weight": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, C.c_int, c_vp]),
        "rgbmp_edge_permute": (C.c_int, [c_vp, c_vp, c_i64, C.c_int, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_longrow_count": (C.c_int, [c_vp, c_i64, c_i32, c_i32, c_vp, C.c_int, c_vp]),
        "rgbmp_longrow_fill_workspace_bytes": (c_sz, [c_i64]),
        "rgbmp_longrow_fill": (C.c_int, [c_vp, c_i64, c_i32, c_i32, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                         C.c_int, c_vp]),
        "rgbmp_longrow_fill_ordered": (C.c_int, [c_vp, c_i64, c_i32, c_i32, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                                 C.c_int, c_vp]),
        "rgbmp_row_order_grouped": (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_i32, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_set_khop_cta": (C.c_int, [C.c_int]),
        "rgbmp_set_push_bulk": (C.c_int, [C.c_int]),
        "rgbmp_khop_cta_calls": (C.c_longlong, []),
        "rgbmp_cluster_workspace_bytes": (c_sz, [c_i64]),
        "rgbmp_cluster_lpa": (C.c_int, [GP, c_vp, c_i32, C.c_int, C.POINTER(c_f32), c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_cluster_connectivity": (C.c_int, [GP, c_vp, c_i32, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_row_order_workspace_bytes": (c_sz, [c_i64]),
        "rgbmp_row_order": (C.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_spmm_workspace_bytes": (c_sz, [GP, C.c_int]),
        "rgbmp_spmm": (C.c_int, [GP, c_vp, c_vp, c_i64, c_vp, c_i64, C.c_int, C.c_int, EP, C.c_int, c_vp, c_sz,
                                 C.c_int, c_vp]),
        "rgbmp_khop": (C.c_int, [GP, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, C.c_int,
                                 C.c_int, C.c_int, EP, C.c_int, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_row_scale": (C.c_int, [c_vp, c_i64, c_vp, C.c_int, c_vp, c_i64, c_i64, C.c_int, C.c_int, C.c_int, c_vp]),
        "rgbmp_stage_rows": (C.c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, C.c_int, C.c_int, c_vp]),
        "rgbmp_appnp_host": (C.c_int, [GP, c_vp, c_vp, c_vp, C.c_int, C.c_int, c_f32, c_vp, c_vp, c_vp, c_vp, c_i64,
                                       c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_appnp_host_mapped": (C.c_int, [GP, c_vp, c_vp, c_vp, c_vp, C.c_int, C.c_int, c_f32, c_vp, c_vp, c_vp, c_vp,
                                              c_i64, c_vp, c_sz, C.c_int, c_vp]),
    }
    optional = {
        "rgbmp_att_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
        "rgbmp_att_forward_workspace_bytes": (c_sz, [GP, C.c_int, C.c_int]),
        "rgbmp_att_forward": (C.c_int, [GP, C.c_int, c_vp, c_i64, c_vp, c_vp, c_vp, C.c_int, C.c_int, c_f32, c_f32, c_vp, DP,
                                        c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_att_backward_workspace_bytes": (c_sz, [GP, GP, C.c_int, C.c_int]),
        "rgbmp_att_backward": (C.c_int, [GP, GP, C.c_int, c_vp, c_i64, c_vp, c_vp, c_vp, C.c_int, C.c_int, c_f32, c_f32, c_vp,
                                         c_vp, DP, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp,
                                         c_i64, c_vp, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_dropout_mask": (C.c_int, [DP, c_i64, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_sgat_negative_sampling_workspace_bytes": (c_sz, [c_i64]),
        "rgbmp_sgat_negative_sampling": (C.c_int, [c_vp, c_vp, c_i64, SP, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, C.c_int,
                                                   c_vp]),
        "rgbmp_sgat_keep_mask": (C.c_int, [SP, c_i64, c_vp, C.c_int, c_vp]),
        "rgbmp_sgat_loss_workspace_bytes": (c_sz, [c_i64]),
        "rgbmp_sgat_loss_forward": (C.c_int, [GP, GP, SP, c_vp, c_i64, C.c_int, c_f32, c_vp, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_sgat_loss_backward": (C.c_int, [GP, GP, GP, GP, SP, c_vp, c_i64, C.c_int, c_f32, c_vp, c_vp, c_vp, c_i64,
                                               C.c_int, c_vp]),
        "rgbmp_coalesce_workspace_bytes": (c_sz, [c_i64, c_i64, C.c_int]),
        "rgbmp_coalesce": (C.c_int, [c_vp, c_vp, c_i64, c_i64, C.c_int, c_vp, c_vp, c_vp, c_vp, c_sz, C.c_int, c_vp]),
        "rgbmp_peer_alloc": (C.c_int, [c_sz, c_vp, c_vp, C.c_int]),
        "rgbmp_peer_free": (C.c_int, [c_vp, C.c_int]),
        "rgbmp_peer_open": (C.c_int, [c_vp, c_vp, C.c_int]),
        "rgbmp_peer_close": (C.c_int, [c_vp, C.c_int]),
        "rgbmp_l2_persist": (C.c_int, [C.c_int, c_sz, c_vp]),
        "rgbmp_col_freq": (C.c_int, [c_vp, c_i64, c_i64, c_vp, C.c_int, c_vp]),
        "rgbmp_col_tag": (C.c_int, [c_vp, c_i64, c_vp, c_i32, c_vp, C.c_int, c_vp]),
        "rgbmp_microbench_gather": (C.c_int, [c_vp, c_i64, C.c_int, c_i64, C.c_uint32, c_vp, c_i64, C.c_int, c_vp]),
        "rgbmp_rowdot": (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, C.c_int, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_sddmm": (C.c_int, [GP, c_vp, c_i64, c_vp, c_i64, C.c_int, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_u_add_v": (C.c_int, [GP, c_vp, c_vp, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_seg_softmax": (C.c_int, [GP, c_vp, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_seg_softmax_backward": (C.c_int, [GP, c_vp, c_vp, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_seg_sum": (C.c_int, [GP, c_vp, C.c_int, c_vp, C.c_int, c_vp]),
        "rgbmp_spmm_heads": (C.c_int, [GP, c_vp, c_vp, c_i64, C.c_int, C.c_int, c_vp, c_i64, C.c_int, c_vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)          # AttributeError here = library/header mismatch: fail loudly
        fn.restype, fn.argtypes = res, args
    for name, (res, args) in optional.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    if L.rgbmp_version() != 101:
        raise RuntimeError("librgbmp.so version mismatch")
    _lib = L
    return L


EXPORTS = None  # filled by tests from include/rgbmp.h


def check(rc: int, what: str = ""):
    """0 ok; anything else -> RuntimeError (the reference's callers treat RuntimeError as OOM/failure,
    examples/all_dataset_baseline.py:65-66)."""
    if rc != 0:
        msg = lib().rgbmp_last_error()
        msg = msg.decode() if msg else ""
        kind = "CUDA error" if rc > 0 else "argument error"
        raise RuntimeError(f"librgbmp {what}: {kind} {rc}: {msg}")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_of(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"rgb-experiment_b200: `{name}` must be a CUDA tensor (got {t.device}); "
                           "this package has no CPU path")


def require_f32(t: torch.Tensor, name: str):
    """The attention / edge-score kernels read every operand as float32: refuse any other dtype before a launch
    instead of reinterpreting its bytes."""
    if t.dtype != torch.float32:
        raise RuntimeError(f"rgb-experiment_b200: {name} takes float32 only (got {t.dtype})")


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise RuntimeError(f"rgb-experiment_b200: unsupported feature dtype {t.dtype} (float32 / bfloat16 only)")
