"""ctypes binding of ``libgte_b200.so`` (C ABI declared in ``include/gte.h``).

The shared library is built in-tree by ``csrc/build.sh`` (``__graft_entry__.build()``)
and loaded from the package directory.  There is no CPU fallback: if the library
is missing, ``lib()`` raises -- the product path never computes on the host.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# GTE_LIB: load another build of the same ABI; never a fallback
LIB_PATH = os.environ.get("GTE_LIB") or os.path.join(_HERE, "libgte_b200.so")
ABI_VERSION = 3
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "gte.h")

_lib: Optional[C.CDLL] = None

i32, i64, f32, vp, sz, ci = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t, C.c_int

# name -> (restype, argtypes); mirrors include/gte.h one to one
SIGNATURES = {
    "gte_abi_version": (ci, []),
    "gte_last_error_string": (C.c_char_p, []),
    "gte_launch_count": (i64, []),
    "gte_set_tuning": (ci, [ci, ci]),
    "gte_get_tuning": (ci, [ci]),
    "gte_device_info": (ci, [C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]),
    "gte_csx_from_coo_workspace_bytes": (sz, [i32, i64]),
    "gte_csx_from_coo": (ci, [vp, vp, i32, i64, vp, vp, vp, vp, sz, vp]),
    "gte_csx_from_coo_checked": (ci, [vp, vp, i32, i32, i64, vp, vp, vp, vp, vp, sz, vp]),
    "gte_batch_concat_csx": (ci, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]),
    "gte_gather_f32": (ci, [vp, vp, vp, i64, vp]),
    "gte_degree_norm": (ci, [vp, i32, ci, vp, vp]),
    "gte_spmm": (ci, [vp, vp, vp, vp, vp, ci, vp, i64, vp, i64, vp, i64, i32, i32, vp]),
    "gte_spmm_paged": (ci, [vp, vp, vp, vp, vp, ci, vp, i64, vp, i64, vp, i64, vp, i32, i32, i32, i32, i32, vp]),
    "gte_paged_pack_edges": (ci, [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
    "gte_spmm_paged_packed_smem_bytes": (sz, [i32, i32, i32]),
    "gte_spmm_paged_packed": (ci, [vp, vp, vp, vp, vp, vp, vp, vp, ci, vp, i64, vp, i64, vp, i64, vp, i32, i32, i32, i32, i32, vp]),
    "gte_gram_stream_workspace_bytes": (sz, [i32, i32]),
    "gte_gram_stream": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, i32, i32, vp, i64, i64, vp, i64, i64, vp, ci, vp, sz, vp]),
    "gte_wide_out": (ci, [vp, i64, i32, vp, i64, i32, vp, vp, i64, i64, vp, vp, vp, f32, ci, ci, vp, vp, i64, vp, i64, vp, vp,
                          i32, i32, vp]),
    "gte_linear_fwd": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, vp, vp, i64, i32, i32, vp]),
    "gte_linear_bwd_data": (ci, [vp, i64, i32, vp, i64, i32, i32, vp, vp, i64, i32, ci, vp]),
    "gte_linear_bwd_data2": (ci, [vp, i64, i32, vp, i64, i32, i32, vp, i64, i32, vp, vp, i64, i32, ci, vp]),
    "gte_linear_bwd_weight_workspace_bytes": (sz, [i32, i32, i32, i32]),
    "gte_linear_bwd_weight": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, i32, vp, i64, vp, ci, i32, vp, sz, vp]),
    "gte_linear_bwd_weight2": (ci, [vp, i64, vp, i64, i32, vp, i64, i32, vp, i64, i32, i32, vp, ci, i32, vp, sz, vp]),
    "gte_umma_supported": (ci, [i32, i32]),
    "gte_umma_pack_bytes": (sz, [i32, i32, i32]),
    "gte_umma_pack_weights": (ci, [vp, i64, i32, i32, i32, vp, vp]),
    "gte_umma_linear_fwd": (ci, [vp, i64, vp, i64, i32, vp, vp, vp, vp, f32, ci, ci, vp, i64, vp, i64, vp, vp, i32, i32, vp]),
    "gte_umma_linear_bwd_data": (ci, [vp, i64, i32, vp, i32, vp, i64, vp, i64, i32, i32, vp]),
    "gte_umma_linear_fwd_stacked": (ci, [vp, i64, i32, vp, vp, i32, vp, i64, i32, vp]),
    "gte_umma_linear_bwd_data2": (ci, [vp, i64, vp, i64, i32, vp, vp, i64, i32, i32, vp]),
    "gte_umma_bwd_weight_supported": (ci, [i32, i32, i32]),
    "gte_umma_bwd_weight_workspace_bytes": (sz, [i32, i32, i32, i32]),
    "gte_umma_linear_bwd_weight": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, i32, vp, i64, vp, ci, i32, vp, sz, vp]),
    "gte_umma_bwd_weight2_workspace_bytes": (sz, [i32, i32, i32]),
    "gte_umma_linear_bwd_weight2": (ci, [vp, i64, vp, i64, i32, vp, i64, i32, vp, i64, i32, i32, vp, ci, i32, vp, sz, vp]),
    "gte_umma_pack_weights_batch": (ci, [vp, i32, vp]),
    "gte_umma_linear_fwd_comb": (ci, [vp, i64, i32, vp, vp, vp, vp, f32, ci, ci, vp, i64, vp, i64, vp, vp, i32, i32, vp]),
    "gte_umma_linear_bwd_data_comb": (ci, [vp, i64, i32, vp, vp, i64, i32, i32, vp]),
    "gte_umma_linear_bwd_weight_comb": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, vp, ci, i32, vp, sz, vp]),
    "gte_umma_linear_bwd_weight2_comb": (ci, [vp, i64, i32, vp, i64, i32, vp, i64, i32, i32, vp, ci, i32, vp, sz, vp]),
    "gte_layernorm_act_fwd": (ci, [vp, i64, vp, vp, f32, ci, vp, i64, vp, vp, i32, i32, vp]),
    "gte_layernorm_act_bwd_workspace_bytes": (sz, [i32, i32]),
    "gte_layernorm_act_bwd": (ci, [vp, i64, vp, i64, vp, vp, vp, vp, ci, vp, i64, vp, vp, vp, ci, i32, i32, vp, sz, vp]),
    "gte_relu_l2norm_fwd": (ci, [vp, i64, f32, vp, i64, i32, i32, vp]),
    "gte_relu_l2norm_bwd": (ci, [vp, i64, vp, i64, f32, vp, i64, i32, i32, vp]),
    "gte_relu_l2norm_bwd_colsum_workspace_bytes": (sz, [i32, i32]),
    "gte_relu_l2norm_bwd_colsum": (ci, [vp, i64, vp, i64, f32, vp, i64, vp, ci, i32, i32, vp, sz, vp]),
    "gte_relu_fwd": (ci, [vp, i64, vp, i64, i32, i32, vp]),
    "gte_dropout_concat": (ci, [vp, i64, i32, vp, i64, i32, i32, f32, C.c_uint64, C.c_uint64, vp, vp, i64, vp, i64, vp]),
    "gte_rng_advance": (ci, [vp, i64, vp]),
    "gte_relu_bwd": (ci, [vp, i64, vp, i64, vp, i64, i32, i32, vp]),
    "gte_cross_entropy_workspace_bytes": (sz, [i32]),
    "gte_cross_entropy_fwd": (ci, [vp, i64, vp, ci, vp, i32, i32, vp, vp, sz, vp]),
    "gte_cross_entropy_bwd": (ci, [vp, i64, vp, ci, vp, i32, i32, vp, vp, i64, vp]),
    "gte_cross_entropy_bwd_padded": (ci, [vp, i64, vp, ci, vp, i32, i32, vp, vp, i64, i32, vp]),
    "gte_eval_workspace_bytes": (sz, [i32]),
    "gte_eval_accumulate": (ci, [vp, i64, vp, ci, vp, i32, i32, vp, vp, sz, vp]),
    "gte_comb_fill": (ci, [vp, i64, i32, vp, i64, i64, vp]),
    "gte_page_predictions": (ci, [vp, i64, i32, i32, vp, ci, vp, i32, vp, vp, vp]),
    "gte_build_page_formats_smem_bytes": (sz, [i32, i32]),
    "gte_build_page_formats": (ci, [vp, vp, vp, vp, vp, i32, i32, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gte_pad_batch": (ci, [vp, i32, i64, i32, vp, vp, vp, vp, vp, vp, i64, i32, vp, vp, vp]),
    "gte_gather_plan": (ci, [vp, vp, vp, i32, i32, i64, i32, i32, i32, i32, i64, i32, vp, vp]),
    "gte_gather_pages": (ci, [vp, vp, i32, i64, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]),
    "gte_bbox_features": (ci, [vp, vp, i32, vp, i64, vp]),
    "gte_adam_step": (ci, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, vp, f32, vp, vp]),
    "gte_dp_allreduce_adam": (ci, [vp, vp, i32, i32, i64, i64, vp, vp, vp, vp, f32, f32, f32, f32, f32, vp, vp, vp]),
    "gte_adam_step_dev": (ci, [vp, vp, vp, vp, i64, vp, i64, vp, f32, vp, vp]),
    "gte_dp_allreduce_adam_dev": (ci, [vp, vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp]),
}

PACK_BATCH_MAX = 8


class PackDesc(C.Structure):
    """gte_pack_desc_t (gte.h)"""
    _fields_ = [("W", C.c_void_p), ("ldw", C.c_int64), ("fo", C.c_int32), ("fin", C.c_int32), ("nseg", C.c_int32),
                ("pack", C.c_void_p)]


GTE_TUNE_UMMA_PAIR = 0
GTE_AGG_SUM, GTE_AGG_SUM_NORM, GTE_AGG_MEAN = 0, 1, 2
GTE_NORM_INV_DEG_ZERO, GTE_NORM_INV_DEG_CLAMP = 0, 1
GTE_LABEL_I64, GTE_LABEL_I32, GTE_LABEL_F32 = 0, 1, 2
GTE_EPI_NONE, GTE_EPI_LN, GTE_EPI_L2 = 0, 1, 2  # the fuse_ln selector of gte_umma_linear_fwd(_comb)


class GteError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the native library; raise loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GteError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or gnn_tableextraction_b200/csrc/build.sh). There is no CPU fallback for the graph-convolution path."
        )
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(l, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if l.gte_abi_version() != ABI_VERSION:
        raise GteError(f"libgte_b200 ABI version {l.gte_abi_version()} != {ABI_VERSION}: rebuild with csrc/build.sh")
    _lib = l
    return l


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().gte_last_error_string()
        raise GteError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")
