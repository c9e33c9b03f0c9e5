"""Tensor-level wrappers over the C ABI (``include/gte.h``).

PyTorch is plumbing here: it owns device memory and the current stream; every
function below validates its tensors, then passes raw device pointers, sizes and
``torch.cuda.current_stream()`` to ``libgte_b200.so``.  CPU tensors are rejected
(no CPU fallback).  Matrices are 2-D fp32 with unit column stride; the row stride
is passed as the leading dimension, so padded / sliced views work unchanged.
"""
from __future__ import annotations

from typing import Optional, Tuple

import ctypes as C

import torch

from . import _lib
from ._lib import GteError, check, lib

_WS = {}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise GteError("gnn_tableextraction_b200: CPU tensor passed to the CUDA hot path (no CPU fallback exists)")


def _mat(t: torch.Tensor, name: str) -> Tuple[int, int, int]:
    """(ptr, ld, cols) of a 2-D fp32 CUDA matrix with unit column stride."""
    if t.dtype != torch.float32 or t.dim() != 2:
        raise GteError(f"{name}: expected a 2-D float32 tensor, got {t.dtype} {tuple(t.shape)}")
    _req_cuda(t)
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise GteError(f"{name}: column stride must be 1 (got strides {t.stride()})")
    ld = t.stride(0) if t.shape[0] > 1 else max(int(t.shape[1]), 1)
    if ld < t.shape[1]:
        raise GteError(f"{name}: row stride {ld} < columns {t.shape[1]}")
    return t.data_ptr(), int(ld), int(t.shape[1])


def _vec(t: Optional[torch.Tensor], name: str, dtype=torch.float32, n: Optional[int] = None) -> Optional[int]:
    if t is None:
        return None
    _req_cuda(t)
    if t.dtype != dtype or not t.is_contiguous():
        raise GteError(f"{name}: expected contiguous {dtype}, got {t.dtype} contiguous={t.is_contiguous()}")
    if n is not None and t.numel() < n:
        raise GteError(f"{name}: {t.numel()} elements < required {n}")
    return t.data_ptr()


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    """Scratch buffer for one kernel call.

    Eager calls share a per-(device, stream) buffer that only ever grows (kernels on one stream serialise, so sharing
    it across calls is safe).  While the stream is being CAPTURED into a CUDA graph the cache is bypassed: a captured
    kernel keeps the pointer it was recorded with, so the buffer must belong to the graph's own memory pool (torch
    keeps that pool alive as long as the graph, and re-uses the block for later kernels of the same capture in stream
    order) -- a cached buffer could be re-allocated by a later, larger eager call and leave the graph with a dangling
    pointer."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream())
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def padded_cols(f: int) -> int:
    """Leading dimension used for internally allocated feature matrices: rows 16-byte aligned (128-bit
    accesses, TMA); wide rows start on 128-byte lines (32 floats) so that a warp's row segments never straddle
    cache lines -- 218 columns live in 224."""
    a = 32 if f > 32 else 4
    return (f + a - 1) // a * a


def empty_padded(n: int, f: int, device) -> torch.Tensor:
    """[n, f] view of an [n, round_up(f, 4)] buffer so that rows are 128-bit aligned."""
    return torch.empty((n, padded_cols(f)), dtype=torch.float32, device=device)[:, :f]


# ------------------------------------------------------------------ graph ---
def csx_from_coo(key: torch.Tensor, other: torch.Tensor, n: int, n_other: Optional[int] = None,
                 bad: Optional[torch.Tensor] = None):
    """Stable compressed rows over ``key``: (indptr[n+1], indices[E], eid[E]) int32.  ``bad`` (device int32[1],
    caller-cleared) is raised when an id lies outside [0, n) / [0, n_other) -- see gte_csx_from_coo_checked."""
    _req_cuda(key, other)
    if key.dtype != torch.int32 or other.dtype != torch.int32:
        raise GteError("csx_from_coo: ids must be int32 (builder.py:425)")
    key, other = key.contiguous(), other.contiguous()
    e = key.numel()
    dev = key.device
    indptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
    indices = torch.empty(e, dtype=torch.int32, device=dev)
    eid = torch.empty(e, dtype=torch.int32, device=dev)
    l = lib()
    need = l.gte_csx_from_coo_workspace_bytes(n, e)
    ws = workspace(need, dev)
    check(
        l.gte_csx_from_coo_checked(key.data_ptr(), other.data_ptr(), n, n if n_other is None else int(n_other), e,
                                   indptr.data_ptr(), indices.data_ptr(), eid.data_ptr(),
                                   _vec(bad, "bad", torch.int32, 1), ws.data_ptr(), ws.numel(), _stream()),
        "gte_csx_from_coo_checked",
    )
    return indptr, indices, eid


def batch_concat_csx(pool_indptr, pool_indices, pool_eid, pool_w, pool_node_off, pool_edge_off, page_ids,
                     batch_node_off, batch_edge_off, n_total: int, e_total: int):
    dev = pool_indptr.device
    _req_cuda(pool_indptr, pool_indices, pool_eid, pool_w, pool_node_off, pool_edge_off, page_ids, batch_node_off,
              batch_edge_off)
    p = int(page_ids.numel())
    indptr = torch.empty(n_total + 1, dtype=torch.int32, device=dev)
    indices = torch.empty(e_total, dtype=torch.int32, device=dev)
    eid = torch.empty(e_total, dtype=torch.int32, device=dev) if pool_eid is not None else None
    w = torch.empty(e_total, dtype=torch.float32, device=dev) if pool_w is not None else None
    if p == 0:
        indptr.zero_()
    check(
        lib().gte_batch_concat_csx(_ptr(pool_indptr), _ptr(pool_indices), _ptr(pool_eid), _ptr(pool_w),
                                   _ptr(pool_node_off), _ptr(pool_edge_off), _ptr(page_ids), _ptr(batch_node_off),
                                   _ptr(batch_edge_off), p, _ptr(indptr), _ptr(indices), _ptr(eid), _ptr(w),
                                   _stream()),
        "gte_batch_concat_csx",
    )
    return indptr, indices, eid, w


def gather_f32(src: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _req_cuda(src, idx)
    out = torch.empty(idx.numel(), dtype=torch.float32, device=src.device)
    check(lib().gte_gather_f32(_vec(src, "gather.in"), _vec(idx, "gather.idx", torch.int32), out.data_ptr(),
                               idx.numel(), _stream()), "gte_gather_f32")
    return out


def degree_norm(indptr: torch.Tensor, mode: int = _lib.GTE_NORM_INV_DEG_ZERO) -> torch.Tensor:
    n = indptr.numel() - 1
    out = torch.empty(n, dtype=torch.float32, device=indptr.device)
    check(lib().gte_degree_norm(_vec(indptr, "indptr", torch.int32), n, mode, out.data_ptr(), _stream()),
          "gte_degree_norm")
    return out


# ------------------------------------------------------------ aggregation ---
def spmm(indptr, indices, w, x, *, mode=_lib.GTE_AGG_SUM, row_norm=None, pre_scale=None, addend=None, out=None,
         pages=None):
    """y[r] = post(r) * sum_j w[j] * pre[c_j] * x[c_j] (+ addend[r]); see gte.h.
    ``pages`` = (page_off int32 [P+1] device tensor, P, max_page_nodes, max_page_edges) selects the
    shared-memory staged kernel for block-diagonal page batches."""
    xp, ldx, f = _mat(x, "spmm.x")
    n_rows = indptr.numel() - 1
    if out is None:
        out = empty_padded(n_rows, f, x.device)
    yp, ldy, fy = _mat(out, "spmm.y")
    if fy != f or out.shape[0] != n_rows:
        raise GteError("spmm: output shape mismatch")
    ap, lda = None, 0
    if addend is not None:
        ap, lda, fa = _mat(addend, "spmm.addend")
        if fa != f or addend.shape[0] != n_rows:
            raise GteError("spmm: addend shape mismatch")
    if pages is not None and pages[1] > 0:
        page_off, num_pages, max_nodes, max_edges = pages[:4]
        check(
            lib().gte_spmm_paged(_vec(indptr, "indptr", torch.int32), _vec(indices, "indices", torch.int32),
                                 _vec(w, "w", n=indices.numel()), _vec(pre_scale, "pre_scale"),
                                 _vec(row_norm, "row_norm", n=n_rows), mode, xp, ldx, ap, lda, yp, ldy,
                                 _vec(page_off, "page_off", torch.int32, num_pages + 1), num_pages, max_nodes, max_edges, n_rows, f,
                                 _stream()),
            "gte_spmm_paged",
        )
        return out
    check(
        lib().gte_spmm(_vec(indptr, "indptr", torch.int32), _vec(indices, "indices", torch.int32),
                       _vec(w, "w", n=indices.numel()), _vec(pre_scale, "pre_scale"), _vec(row_norm, "row_norm", n=n_rows),
                       mode, xp, ldx, ap, lda, yp, ldy, n_rows, f, _stream()),
        "gte_spmm",
    )
    return out


class PackedEdges:
    """Edges of one direction of a page batch in the layout ``gte_spmm_paged_packed`` stages:
    ``packed`` [E] int64 = (page-local source row | weight * source scale), ``page_flag`` [P] int32.
    Holds the raw arrays the kernel's slow path (edges leaving a page) falls back to."""

    __slots__ = ("packed", "page_flag", "indices", "eid", "w", "pre_scale")

    def __init__(self, packed, page_flag, indices, eid, w, pre_scale):
        self.packed, self.page_flag, self.indices, self.eid, self.w, self.pre_scale = packed, page_flag, indices, eid, w, pre_scale


def paged_packed_supported(pages, f: int) -> bool:
    """Do two shared-memory stages of the largest page fit (``gte_spmm_paged_packed_smem_bytes`` > 0)?"""
    if pages is None or pages[1] <= 0 or f <= 0:
        return False
    return lib().gte_spmm_paged_packed_smem_bytes(int(pages[2]), int(pages[3]), int(f)) > 0


def paged_pack_edges(indptr, indices, w, pages, *, eid=None, pre_scale=None) -> PackedEdges:
    """Pack one direction's edges once per batch: ``w`` is in row order, or in edge order with ``eid``
    (then ``edata['feat'][eid]`` is folded into the packing); ``pre_scale`` is the source-side scale."""
    page_off, num_pages = pages[0], pages[1]
    _req_cuda(indptr, indices, w, eid, pre_scale, page_off)
    e = indices.numel()
    packed = torch.empty(e + 2, dtype=torch.int64, device=indices.device)  # 16-byte bulk copies may over-read one entry
    flag = torch.empty(max(num_pages, 1), dtype=torch.int32, device=indices.device)
    check(
        lib().gte_paged_pack_edges(_vec(indptr, "indptr", torch.int32), _vec(indices, "indices", torch.int32),
                                   _vec(eid, "eid", torch.int32, e), _vec(w, "w", n=e), _vec(pre_scale, "pre_scale"),
                                   _vec(page_off, "page_off", torch.int32, num_pages + 1), num_pages, packed.data_ptr(),
                                   flag.data_ptr(), _stream()),
        "gte_paged_pack_edges",
    )
    return PackedEdges(packed, flag, indices, eid, w, pre_scale)


def spmm_packed(indptr, pk: PackedEdges, x, pages, *, mode=_lib.GTE_AGG_SUM, row_norm=None, addend=None, out=None):
    """``spmm`` on pre-packed page edges (the persistent, double-buffered kernel); same result."""
    xp, ldx, f = _mat(x, "spmm.x")
    n_rows = indptr.numel() - 1
    if out is None:
        out = empty_padded(n_rows, f, x.device)
    yp, ldy, fy = _mat(out, "spmm.y")
    if fy != f or out.shape[0] != n_rows:
        raise GteError("spmm: output shape mismatch")
    ap, lda = None, 0
    if addend is not None:
        ap, lda, fa = _mat(addend, "spmm.addend")
        if fa != f or addend.shape[0] != n_rows:
            raise GteError("spmm: addend shape mismatch")
    page_off, num_pages, max_nodes, max_edges = pages[:4]
    check(
        lib().gte_spmm_paged_packed(_vec(indptr, "indptr", torch.int32), pk.packed.data_ptr(), pk.page_flag.data_ptr(),
                                    _vec(pk.indices, "indices", torch.int32), _vec(pk.eid, "eid", torch.int32),
                                    _vec(pk.w, "w"), _vec(pk.pre_scale, "pre_scale"), _vec(row_norm, "row_norm", n=n_rows),
                                    mode, xp, ldx, ap, lda, yp, ldy, _vec(page_off, "page_off", torch.int32, num_pages + 1),
                                    num_pages, max_nodes, max_edges, n_rows, f, _stream()),
        "gte_spmm_paged_packed",
    )
    return out


# ------------------------------------------------- narrow dense streams ---
def gram_stream_supported(wide: int, nq: int, *mats) -> bool:
    return 0 < wide <= 256 and 0 < nq <= 32 and _aligned_mat(mats[0]) and all(m is None or m.is_cuda for m in mats)


def gram_stream(P, Q1, Q2, out1, sa1: int, sb1: int, out2=None, sa2: int = 0, sb2: int = 0, qsum=None, accumulate=False):
    """C[a][b] = sum_r P[r,a] * [Q1|Q2][r,b] scattered to ``out1`` / ``out2`` with element strides
    (``sa``, ``sb``); ``qsum`` = column sums of Q1.  See gte.h (gte_gram_stream)."""
    pp, ldp, wide = _mat(P, "gram.P")
    n = P.shape[0]
    q1p, ldq1, nq1 = _mat(Q1, "gram.Q1")
    q2p, ldq2, nq2 = (None, 0, 0)
    if Q2 is not None:
        q2p, ldq2, nq2 = _mat(Q2, "gram.Q2")
    if Q1.shape[0] != n or (Q2 is not None and Q2.shape[0] != n):
        raise GteError("gram_stream: row mismatch")
    _req_cuda(out1, out2, qsum)
    l = lib()
    need = l.gte_gram_stream_workspace_bytes(n, wide)
    ws = workspace(need, P.device)
    check(l.gte_gram_stream(pp, ldp, wide, q1p, ldq1, nq1, q2p, ldq2, nq2, n, out1.data_ptr(), sa1, sb1, _ptr(out2), sa2, sb2,
                            _ptr(qsum), 1 if accumulate else 0, ws.data_ptr(), ws.numel(), _stream()), "gte_gram_stream")


def wide_out_supported(k1: int, k2: int, c: int, *mats) -> bool:
    return 0 < k1 <= 16 and 0 <= k2 <= 16 and 0 < c <= 256 and all(m is None or _aligned_mat(m) for m in mats)


def wide_out(A1, A2, B1_ptr: int, B2_ptr: Optional[int], sj: int, sc: int, c: int, bias=None, *, gamma=None, beta=None,
             eps: float = 1e-5, relu: bool = False, fuse_ln: bool = False, row_scale=None):
    """z = [A1|A2] B (+ bias) (* row_scale) with the narrow operand on the contraction side; with
    ``fuse_ln`` returns (z, y, mean, rstd), else (z, None, None, None).  See gte.h (gte_wide_out)."""
    a1p, lda1, k1 = _mat(A1, "wide_out.A1")
    n = A1.shape[0]
    a2p, lda2, k2 = (None, 0, 0)
    if A2 is not None:
        a2p, lda2, k2 = _mat(A2, "wide_out.A2")
    dev = A1.device
    z = empty_padded(n, c, dev)
    zp, ldz, _ = _mat(z, "wide_out.z")
    y = mean = rstd = None
    yp, ldy = None, 0
    if fuse_ln:
        y = empty_padded(n, c, dev)
        yp, ldy, _ = _mat(y, "wide_out.y")
        mean = torch.empty(n, dtype=torch.float32, device=dev)
        rstd = torch.empty(n, dtype=torch.float32, device=dev)
    check(lib().gte_wide_out(a1p, lda1, k1, a2p, lda2, k2, B1_ptr, B2_ptr, sj, sc, _vec(bias, "bias", n=c),
                             _vec(gamma, "gamma", n=c), _vec(beta, "beta", n=c), eps, 1 if relu else 0, 1 if fuse_ln else 0,
                             _vec(row_scale, "row_scale", n=n), zp, ldz, yp, ldy, _ptr(mean), _ptr(rstd), n, c, _stream()),
          "gte_wide_out")
    return z, y, mean, rstd


# ------------------------------------------------------------------ dense ---
def linear_fwd(x1, x2, W, bias, out=None, w_col0: int = 0):
    """z = x1 W[:, c0:c0+k1]^T + x2 W[:, c0+k1:c0+k1+k2]^T + bias (x2 may be None)."""
    x1p, ld1, k1 = _mat(x1, "linear.x1")
    n = x1.shape[0]
    x2p, ld2, k2 = (None, 0, 0)
    if x2 is not None:
        x2p, ld2, k2 = _mat(x2, "linear.x2")
        if x2.shape[0] != n:
            raise GteError("linear_fwd: x1/x2 row mismatch")
    Wp, ldw, kw = _mat(W, "linear.W")
    fo = W.shape[0]
    if w_col0 + k1 + k2 > kw:
        raise GteError(f"linear_fwd: W has {kw} columns < {w_col0 + k1 + k2}")
    if out is None:
        out = empty_padded(n, fo, x1.device)
    zp, ldz, fz = _mat(out, "linear.z")
    if fz != fo or out.shape[0] != n:
        raise GteError("linear_fwd: output shape mismatch")
    check(
        lib().gte_linear_fwd(x1p, ld1, k1, x2p, ld2, k2, Wp + 4 * w_col0, ldw, _vec(bias, "bias", n=fo), zp, ldz, n, fo,
                             _stream()),
        "gte_linear_fwd",
    )
    return out


def linear_bwd_data(dz, W, col0: int, k: int, row_scale=None, out=None, accumulate=False):
    dzp, lddz, fo = _mat(dz, "bwd_data.dz")
    Wp, ldw, kw = _mat(W, "bwd_data.W")
    if W.shape[0] != fo or col0 + k > kw:
        raise GteError("linear_bwd_data: W shape mismatch")
    n = dz.shape[0]
    if out is None:
        if accumulate:
            raise GteError("linear_bwd_data: accumulate needs an output")
        out = empty_padded(n, k, dz.device)
    dxp, lddx, kx = _mat(out, "bwd_data.dx")
    if kx != k or out.shape[0] != n:
        raise GteError("linear_bwd_data: output shape mismatch")
    check(
        lib().gte_linear_bwd_data(dzp, lddz, fo, Wp, ldw, col0, k, _vec(row_scale, "row_scale", n=n), dxp, lddx, n,
                                  1 if accumulate else 0, _stream()),
        "gte_linear_bwd_data",
    )
    return out


def linear_bwd_data2(dz1, col1: int, dz2, col2: int, W, k: int, row_scale=None, out=None, accumulate=False):
    """dx (+)= (dz1 W[:, col1:col1+k] + dz2 W[:, col2:col2+k]) * row_scale -- one launch."""
    d1p, ld1, fo = _mat(dz1, "bwd_data2.dz1")
    d2p, ld2, fo2 = _mat(dz2, "bwd_data2.dz2")
    Wp, ldw, kw = _mat(W, "bwd_data2.W")
    if fo2 != fo or W.shape[0] != fo or max(col1, col2) + k > kw or dz2.shape[0] != dz1.shape[0]:
        raise GteError("linear_bwd_data2: shape mismatch")
    n = dz1.shape[0]
    if out is None:
        if accumulate:
            raise GteError("linear_bwd_data2: accumulate needs an output")
        out = empty_padded(n, k, dz1.device)
    dxp, lddx, kx = _mat(out, "bwd_data2.dx")
    if kx != k or out.shape[0] != n:
        raise GteError("linear_bwd_data2: output shape mismatch")
    check(
        lib().gte_linear_bwd_data2(d1p, ld1, col1, d2p, ld2, col2, fo, Wp, ldw, k, _vec(row_scale, "row_scale", n=n), dxp,
                                   lddx, n, 1 if accumulate else 0, _stream()),
        "gte_linear_bwd_data2",
    )
    return out


def linear_bwd_weight(dz, x1, x2, dW, db, accumulate=False, w_col0: int = 0):
    """dW[:, c0:c0+k1+k2] (+)= dz^T [x1 | x2]; db (+)= colsum(dz) (db may be None)."""
    dzp, lddz, fo = _mat(dz, "bwd_weight.dz")
    n = dz.shape[0]
    x1p, ld1, k1 = _mat(x1, "bwd_weight.x1")
    x2p, ld2, k2 = (None, 0, 0)
    if x2 is not None:
        x2p, ld2, k2 = _mat(x2, "bwd_weight.x2")
    dWp, lddw, kw = _mat(dW, "bwd_weight.dW")
    if dW.shape[0] != fo or w_col0 + k1 + k2 > kw:
        raise GteError("linear_bwd_weight: dW shape mismatch")
    l = lib()
    need = l.gte_linear_bwd_weight_workspace_bytes(n, fo, k1, k2)
    ws = workspace(need, dz.device)
    check(
        l.gte_linear_bwd_weight(dzp, lddz, fo, x1p, ld1, k1, x2p, ld2, k2, dWp + 4 * w_col0, lddw,
                                _vec(db, "db", n=fo), 1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_linear_bwd_weight",
    )


def linear_bwd_weight2(dz1, dz2, x, dW, col1: int, col2: int, db, accumulate=False):
    """dW[:, col1:col1+k] (+)= dz1^T x ; dW[:, col2:col2+k] (+)= dz2^T x ; db (+)= colsum(dz1) -- x is read once."""
    d1p, ld1, fo = _mat(dz1, "bwd_weight2.dz1")
    d2p, ld2, fo2 = _mat(dz2, "bwd_weight2.dz2")
    xp, ldx, k = _mat(x, "bwd_weight2.x")
    dWp, lddw, kw = _mat(dW, "bwd_weight2.dW")
    n = dz1.shape[0]
    if fo2 != fo or dW.shape[0] != fo or max(col1, col2) + k > kw or dz2.shape[0] != n or x.shape[0] != n:
        raise GteError("linear_bwd_weight2: shape mismatch")
    l = lib()
    ws = workspace(l.gte_linear_bwd_weight_workspace_bytes(n, fo, k, k), dz1.device)
    check(
        l.gte_linear_bwd_weight2(d1p, ld1, d2p, ld2, fo, xp, ldx, k, dWp, lddw, col1, col2, _vec(db, "db", n=fo),
                                 1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_linear_bwd_weight2",
    )


# ------------------------------------------------ tensor-core route --------
def umma_supported(fo: int, fin: int) -> bool:
    return bool(lib().gte_umma_supported(fo, fin))


def _aligned_mat(t: torch.Tensor) -> bool:
    return t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.data_ptr() % 16 == 0 and (
        t.shape[0] <= 1 or t.stride(0) % 4 == 0) and (t.shape[1] <= 1 or t.stride(1) == 1)


def umma_pack_weights(W: torch.Tensor, fin: int, nseg: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Split W [fo, nseg*fin] into tf32 hi/lo tiles (forward + transposed backward layouts)."""
    Wp, ldw, kw = _mat(W, "umma_pack.W")
    fo = W.shape[0]
    l = lib()
    nbytes = l.gte_umma_pack_bytes(fo, fin, nseg)
    if nbytes == 0 or kw < nseg * fin:
        raise GteError(f"umma_pack_weights: unsupported shape fo={fo} fin={fin} nseg={nseg}")
    if out is None:
        out = torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
    check(l.gte_umma_pack_weights(Wp, ldw, fo, fin, nseg, _vec(out, "pack", n=nbytes // 4), _stream()),
          "gte_umma_pack_weights")
    return out


def umma_pack_weights_batch(items, outs=None):
    """``umma_pack_weights`` for several ``(W, fin, nseg)`` in ONE launch; returns the list of pack buffers
    (``outs``: reuse these buffers)."""
    l = lib()
    res = []
    for lo in range(0, len(items), _lib.PACK_BATCH_MAX):
        chunk = items[lo:lo + _lib.PACK_BATCH_MAX]
        arr = (_lib.PackDesc * len(chunk))()
        for i, (W, fin, nseg) in enumerate(chunk):
            Wp, ldw, kw = _mat(W, "umma_pack.W")
            fo = W.shape[0]
            nbytes = l.gte_umma_pack_bytes(fo, fin, nseg)
            if nbytes == 0 or kw < nseg * fin:
                raise GteError(f"umma_pack_weights_batch: unsupported shape fo={fo} fin={fin} nseg={nseg}")
            out = outs[lo + i] if outs is not None else torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
            arr[i].W, arr[i].ldw, arr[i].fo, arr[i].fin, arr[i].nseg = Wp, ldw, fo, fin, nseg
            arr[i].pack = _vec(out, "pack", n=nbytes // 4)
            res.append(out)
        check(l.gte_umma_pack_weights_batch(C.cast(arr, C.c_void_p), len(chunk), _stream()), "gte_umma_pack_weights_batch")
    return res


def set_tuning(key: int, value: int) -> None:
    """Process-wide A/B switch of the native library (tests / measurements; see gte.h gte_set_tuning)."""
    check(lib().gte_set_tuning(int(key), int(value)), "gte_set_tuning")


def get_tuning(key: int) -> int:
    return int(lib().gte_get_tuning(int(key)))


def _epilogue(fuse_ln: bool, l2: bool) -> int:
    if fuse_ln and l2:
        raise GteError("umma_linear_fwd: fuse_ln and l2 are two different epilogues")
    return _lib.GTE_EPI_L2 if l2 else (_lib.GTE_EPI_LN if fuse_ln else _lib.GTE_EPI_NONE)


def umma_linear_fwd(x1, x2, fin: int, pack, bias, fo: int, *, gamma=None, beta=None, eps: float = 1e-5,
                    relu: bool = False, fuse_ln: bool = False, want_y: bool = False, want_z: bool = True,
                    l2: bool = False):
    """(z, y, mean, rstd): z = [x1 | x2] W^T + b ; y = act(LN(z)) / act(z) (None unless requested).
    ``l2``: y = relu(z) / max(||relu(z)||_2, eps) per row (F.relu + F.normalize; ``eps`` is the normalise eps, mean
    and rstd are None).  ``want_z=False`` (inference: nothing is saved for a backward pass) skips the z stores when y
    exists."""
    x1p, ld1, k1 = _mat(x1, "umma.x1")
    n = x1.shape[0]
    x2p, ld2 = None, 0
    if x2 is not None:
        x2p, ld2, k2 = _mat(x2, "umma.x2")
        if k2 != fin or x2.shape[0] != n:
            raise GteError("umma_linear_fwd: x2 shape mismatch")
    if k1 != fin:
        raise GteError("umma_linear_fwd: x1 shape mismatch")
    dev = x1.device
    mode = _epilogue(fuse_ln, l2)
    need_y = fuse_ln or want_y or relu or l2
    z = empty_padded(n, fo, dev) if (want_z or not need_y) else None
    zp, ldz = (None, 0) if z is None else _mat(z, "umma.z")[:2]
    y = empty_padded(n, fo, dev) if need_y else None
    yp, ldy = (None, 0) if y is None else _mat(y, "umma.y")[:2]
    mean = torch.empty(n, dtype=torch.float32, device=dev) if fuse_ln else None
    rstd = torch.empty(n, dtype=torch.float32, device=dev) if fuse_ln else None
    check(
        lib().gte_umma_linear_fwd(x1p, ld1, x2p, ld2, fin, _vec(pack, "pack"), _vec(bias, "bias", n=fo),
                                  _vec(gamma, "gamma", n=fo), _vec(beta, "beta", n=fo), float(eps), 1 if relu else 0,
                                  mode, zp, ldz, yp, ldy, _ptr(mean), _ptr(rstd), n, fo, _stream()),
        "gte_umma_linear_fwd",
    )
    return z, y, mean, rstd


def umma_linear_bwd_data(dz, pack, fin: int, nseg: int):
    """(dx1, dx2) = dz W[:, :fin], dz W[:, fin:2 fin]."""
    dzp, lddz, fo = _mat(dz, "umma_bwd.dz")
    n = dz.shape[0]
    dx1 = empty_padded(n, fin, dz.device)
    dx2 = empty_padded(n, fin, dz.device) if nseg == 2 else None
    d1p, ld1, _ = _mat(dx1, "umma_bwd.dx1")
    d2p, ld2 = (None, 0) if dx2 is None else _mat(dx2, "umma_bwd.dx2")[:2]
    check(lib().gte_umma_linear_bwd_data(dzp, lddz, fo, _vec(pack, "pack"), nseg, d1p, ld1, d2p, ld2, n, fin, _stream()),
          "gte_umma_linear_bwd_data")
    return dx1, dx2


def umma_linear_fwd_stacked(x, fin: int, pack, bias, fo: int):
    """[n, 32] buffer: cols [0, fo) = x Ws^T + b, cols [16, 16+fo) = x Wn^T (class layer, one pass over x)."""
    xp, ldx, k = _mat(x, "umma_stacked.x")
    if k != fin:
        raise GteError("umma_linear_fwd_stacked: x shape mismatch")
    n = x.shape[0]
    out = torch.empty((n, 32), dtype=torch.float32, device=x.device)
    check(lib().gte_umma_linear_fwd_stacked(xp, ldx, fin, _vec(pack, "pack"), _vec(bias, "bias", n=fo), fo, out.data_ptr(),
                                            32, n, _stream()), "gte_umma_linear_fwd_stacked")
    return out


def umma_linear_bwd_data2(dz1, dz2, pack, fin: int):
    """dx = dz1 W[:, :fin] + dz2 W[:, fin:2 fin] on tensor cores."""
    d1p, ld1, fo = _mat(dz1, "umma_bwd2.dz1")
    d2p, ld2, fo2 = _mat(dz2, "umma_bwd2.dz2")
    if fo2 != fo or dz2.shape[0] != dz1.shape[0]:
        raise GteError("umma_linear_bwd_data2: shape mismatch")
    n = dz1.shape[0]
    dx = empty_padded(n, fin, dz1.device)
    dxp, lddx, _ = _mat(dx, "umma_bwd2.dx")
    check(lib().gte_umma_linear_bwd_data2(d1p, ld1, d2p, ld2, fo, _vec(pack, "pack"), dxp, lddx, n, fin, _stream()),
          "gte_umma_linear_bwd_data2")
    return dx


def umma_bwd_weight_supported(fo: int, k1: int, k2: int) -> bool:
    return bool(lib().gte_umma_bwd_weight_supported(fo, k1, k2))


def umma_linear_bwd_weight(dz, x1, x2, dW, db, accumulate=False, w_col0: int = 0):
    """Tensor-core dW[:, c0:c0+k1+k2] (+)= dz^T [x1 | x2]; db (+)= colsum(dz) (needs k1 % 32 != 0)."""
    dzp, lddz, fo = _mat(dz, "umma_dw.dz")
    n = dz.shape[0]
    x1p, ld1, k1 = _mat(x1, "umma_dw.x1")
    x2p, ld2, k2 = (None, 0, 0)
    if x2 is not None:
        x2p, ld2, k2 = _mat(x2, "umma_dw.x2")
    dWp, lddw, kw = _mat(dW, "umma_dw.dW")
    if dW.shape[0] != fo or w_col0 + k1 + k2 > kw:
        raise GteError("umma_linear_bwd_weight: dW shape mismatch")
    l = lib()
    ws = workspace(l.gte_umma_bwd_weight_workspace_bytes(n, fo, k1, k2), dz.device)
    check(
        l.gte_umma_linear_bwd_weight(dzp, lddz, fo, x1p, ld1, k1, x2p, ld2, k2, dWp + 4 * w_col0, lddw, _vec(db, "db", n=fo),
                                     1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_umma_linear_bwd_weight",
    )


def umma_linear_bwd_weight2(dz1, dz2, x, dW, col1: int, col2: int, db, accumulate=False):
    """Tensor-core narrow-dz form: dW[:, col1:+k] (+)= dz1^T x ; dW[:, col2:+k] (+)= dz2^T x ; db (+)= colsum(dz1)."""
    d1p, ld1, fo = _mat(dz1, "umma_dw2.dz1")
    d2p, ld2, fo2 = _mat(dz2, "umma_dw2.dz2")
    xp, ldx, k = _mat(x, "umma_dw2.x")
    dWp, lddw, kw = _mat(dW, "umma_dw2.dW")
    n = dz1.shape[0]
    if fo2 != fo or dW.shape[0] != fo or max(col1, col2) + k > kw or dz2.shape[0] != n or x.shape[0] != n:
        raise GteError("umma_linear_bwd_weight2: shape mismatch")
    l = lib()
    ws = workspace(l.gte_umma_bwd_weight2_workspace_bytes(n, fo, k), dz1.device)
    check(
        l.gte_umma_linear_bwd_weight2(d1p, ld1, d2p, ld2, fo, xp, ldx, k, dWp, lddw, col1, col2, _vec(db, "db", n=fo),
                                      1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_umma_linear_bwd_weight2",
    )


# -- combined [n, 32] operands (columns [0, w) = self block, [16, 16+w) = neighbour block, the rest zero) --------
COMB_W = 16   # widest block a combined operand can hold
COMB_LD = 32


def comb_buffer(n: int, device) -> torch.Tensor:
    """Zeroed [n, 32] combined operand (the padding columns meet zero weights, so they must be finite)."""
    return torch.zeros((n, COMB_LD), dtype=torch.float32, device=device)


def comb_from(x: torch.Tensor) -> torch.Tensor:
    """[n, 32] combined operand with ``x`` [n, w <= 16] as its self block and zeros elsewhere, in one native kernel
    (x may have unaligned rows, e.g. the raw [N, 13] BBOX features); the neighbour block is written afterwards."""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.shape[1] <= COMB_W
            and (x.shape[1] <= 1 or x.stride(1) == 1)):
        raise GteError("comb_from: float32 CUDA matrix [n, w <= 16] with unit column stride expected")
    n, w = x.shape
    out = torch.empty((n, COMB_LD), dtype=torch.float32, device=x.device)
    check(lib().gte_comb_fill(x.data_ptr(), x.stride(0) if n > 1 else max(w, 1), w, out.data_ptr(), COMB_LD, n, _stream()),
          "gte_comb_fill")
    return out


def comb_views(buf: torch.Tensor, w: int):
    """(self block, neighbour block) column views of a combined operand."""
    return buf[:, :w], buf[:, COMB_W:COMB_W + w]


def _comb(buf, what):
    if not (buf.is_cuda and buf.dtype == torch.float32 and buf.dim() == 2 and buf.shape[1] == COMB_LD
            and buf.stride(1) == 1 and buf.stride(0) % 4 == 0 and buf.data_ptr() % 16 == 0):
        raise GteError(f"{what}: a combined operand is a float32 [n, {COMB_LD}] CUDA matrix, 16-byte aligned")
    return buf.data_ptr(), buf.stride(0)


def umma_linear_fwd_comb(xc, fin: int, pack, bias, fo: int, *, gamma=None, beta=None, eps: float = 1e-5,
                         relu: bool = False, fuse_ln: bool = False, want_y: bool = False, want_z: bool = True,
                         l2: bool = False):
    """umma_linear_fwd for a narrow input (fin <= 16) held as one combined operand xc = [h | A_hat h]."""
    xp, ldx = _comb(xc, "umma_linear_fwd_comb.xc")
    n = xc.shape[0]
    dev = xc.device
    mode = _epilogue(fuse_ln, l2)
    need_y = fuse_ln or want_y or relu or l2
    z = empty_padded(n, fo, dev) if (want_z or not need_y) else None
    zp, ldz = (None, 0) if z is None else _mat(z, "umma.z")[:2]
    y = empty_padded(n, fo, dev) if need_y else None
    yp, ldy = (None, 0) if y is None else _mat(y, "umma.y")[:2]
    mean = torch.empty(n, dtype=torch.float32, device=dev) if fuse_ln else None
    rstd = torch.empty(n, dtype=torch.float32, device=dev) if fuse_ln else None
    check(
        lib().gte_umma_linear_fwd_comb(xp, ldx, fin, _vec(pack, "pack"), _vec(bias, "bias", n=fo),
                                       _vec(gamma, "gamma", n=fo), _vec(beta, "beta", n=fo), float(eps),
                                       1 if relu else 0, mode, zp, ldz, yp, ldy, _ptr(mean), _ptr(rstd),
                                       n, fo, _stream()),
        "gte_umma_linear_fwd_comb",
    )
    return z, y, mean, rstd


def umma_linear_bwd_data_comb(dc, fo: int, pack, fin: int):
    """dx = dc[:, :fo] W[:, :fin] + dc[:, 16:16+fo] W[:, fin:2 fin] (class layer; dc = [dz | A_hat^T dz])."""
    dp, ldd = _comb(dc, "umma_linear_bwd_data_comb.dc")
    n = dc.shape[0]
    dx = empty_padded(n, fin, dc.device)
    dxp, lddx, _ = _mat(dx, "umma_bwd_comb.dx")
    check(lib().gte_umma_linear_bwd_data_comb(dp, ldd, fo, _vec(pack, "pack"), dxp, lddx, n, fin, _stream()),
          "gte_umma_linear_bwd_data_comb")
    return dx


def umma_linear_bwd_weight_comb(dz, xc, w: int, dW, db, accumulate=False):
    """dW[:, :w] (+)= dz^T xc[:, :w] ; dW[:, w:2w] (+)= dz^T xc[:, 16:16+w] ; db (+)= colsum(dz) (w < 16)."""
    dzp, lddz, fo = _mat(dz, "umma_dw_comb.dz")
    xp, ldx = _comb(xc, "umma_linear_bwd_weight_comb.xc")
    dWp, lddw, kw = _mat(dW, "umma_dw_comb.dW")
    n = dz.shape[0]
    if dW.shape[0] != fo or 2 * w > kw or xc.shape[0] != n:
        raise GteError("umma_linear_bwd_weight_comb: shape mismatch")
    l = lib()
    ws = workspace(l.gte_umma_bwd_weight_workspace_bytes(n, fo, 256, 0), dz.device)
    check(
        l.gte_umma_linear_bwd_weight_comb(dzp, lddz, fo, xp, ldx, w, dWp, lddw, _vec(db, "db", n=fo),
                                          1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_umma_linear_bwd_weight_comb",
    )


def umma_linear_bwd_weight2_comb(dc, fo: int, x, dW, col1: int, col2: int, db, accumulate=False):
    """dW[:, col1:+k] (+)= dc[:, :fo]^T x ; dW[:, col2:+k] (+)= dc[:, 16:16+fo]^T x ; db (+)= colsum(dc[:, :fo])."""
    dp, ldd = _comb(dc, "umma_linear_bwd_weight2_comb.dc")
    xp, ldx, k = _mat(x, "umma_dw2_comb.x")
    dWp, lddw, kw = _mat(dW, "umma_dw2_comb.dW")
    n = dc.shape[0]
    if dW.shape[0] != fo or max(col1, col2) + k > kw or x.shape[0] != n:
        raise GteError("umma_linear_bwd_weight2_comb: shape mismatch")
    l = lib()
    ws = workspace(l.gte_umma_bwd_weight_workspace_bytes(n, fo, 256, 0), dc.device)
    check(
        l.gte_umma_linear_bwd_weight2_comb(dp, ldd, fo, xp, ldx, k, dWp, lddw, col1, col2, _vec(db, "db", n=fo),
                                           1 if accumulate else 0, n, ws.data_ptr(), ws.numel(), _stream()),
        "gte_umma_linear_bwd_weight2_comb",
    )


# ---------------------------------------------------------------- row ops ---
def layernorm_act_fwd(z, gamma, beta, eps: float, relu: bool, out=None):
    zp, ldz, f = _mat(z, "ln.z")
    n = z.shape[0]
    if out is None:
        out = empty_padded(n, f, z.device)
    yp, ldy, _ = _mat(out, "ln.y")
    mean = torch.empty(n, dtype=torch.float32, device=z.device)
    rstd = torch.empty(n, dtype=torch.float32, device=z.device)
    check(
        lib().gte_layernorm_act_fwd(zp, ldz, _vec(gamma, "gamma", n=f), _vec(beta, "beta", n=f), float(eps),
                                    1 if relu else 0, yp, ldy, mean.data_ptr(), rstd.data_ptr(), n, f, _stream()),
        "gte_layernorm_act_fwd",
    )
    return out, mean, rstd


def layernorm_act_bwd(dy, z, mean, rstd, gamma, beta, relu: bool, dgamma, dbeta, accumulate=False, out=None,
                      dz_colsum=None):
    dyp, lddy, f = _mat(dy, "ln_bwd.dy")
    zp, ldz, _ = _mat(z, "ln_bwd.z")
    n = dy.shape[0]
    if out is None:
        out = empty_padded(n, f, dy.device)
    dzp, lddz, _ = _mat(out, "ln_bwd.dz")
    l = lib()
    need = l.gte_layernorm_act_bwd_workspace_bytes(n, f)
    ws = workspace(need, dy.device)
    check(
        l.gte_layernorm_act_bwd(dyp, lddy, zp, ldz, _vec(mean, "mean", n=n), _vec(rstd, "rstd", n=n),
                                _vec(gamma, "gamma", n=f), _vec(beta, "beta", n=f), 1 if relu else 0, dzp, lddz,
                                _vec(dgamma, "dgamma", n=f), _vec(dbeta, "dbeta", n=f), _vec(dz_colsum, "dz_colsum", n=f),
                                1 if accumulate else 0, n, f,
                                ws.data_ptr(), ws.numel(), _stream()),
        "gte_layernorm_act_bwd",
    )
    return out


def relu_l2norm_fwd(z, eps: float = 1e-12, out=None):
    zp, ldz, f = _mat(z, "l2.z")
    n = z.shape[0]
    if out is None:
        out = empty_padded(n, f, z.device)
    yp, ldy, _ = _mat(out, "l2.y")
    check(lib().gte_relu_l2norm_fwd(zp, ldz, float(eps), yp, ldy, n, f, _stream()), "gte_relu_l2norm_fwd")
    return out


def relu_l2norm_bwd(dy, z, eps: float = 1e-12, out=None):
    dyp, lddy, f = _mat(dy, "l2_bwd.dy")
    zp, ldz, _ = _mat(z, "l2_bwd.z")
    n = dy.shape[0]
    if out is None:
        out = empty_padded(n, f, dy.device)
    dzp, lddz, _ = _mat(out, "l2_bwd.dz")
    check(lib().gte_relu_l2norm_bwd(dyp, lddy, zp, ldz, float(eps), dzp, lddz, n, f, _stream()), "gte_relu_l2norm_bwd")
    return out


def relu_l2norm_bwd_colsum(dy, z, eps: float = 1e-12, dz_colsum=None, accumulate=False, out=None):
    """``relu_l2norm_bwd`` (the same dz bits) that also writes ``dz_colsum`` [f] (+)= the column sums of dz: the bias
    gradient of the linear before the normalisation, in a fixed-order two-stage reduction."""
    dyp, lddy, f = _mat(dy, "l2_bwd.dy")
    zp, ldz, _ = _mat(z, "l2_bwd.z")
    n = dy.shape[0]
    if out is None:
        out = empty_padded(n, f, dy.device)
    dzp, lddz, _ = _mat(out, "l2_bwd.dz")
    l = lib()
    ws = workspace(l.gte_relu_l2norm_bwd_colsum_workspace_bytes(n, f), dy.device)
    check(l.gte_relu_l2norm_bwd_colsum(dyp, lddy, zp, ldz, float(eps), dzp, lddz, _vec(dz_colsum, "dz_colsum", n=f),
                                       1 if accumulate else 0, n, f, ws.data_ptr(), ws.numel(), _stream()),
          "gte_relu_l2norm_bwd_colsum")
    return out


def dropout_concat(x1, x2, p: float, seed: int = 0, offset: int = 0, rng_dev: Optional[torch.Tensor] = None,
                   inplace: bool = False, out=None):
    """Training-mode ``nn.Dropout(p)`` on the concatenation ``[x1 | x2]`` without materialising it (models.py:60-61);
    ``x2`` may be None (input features, models.py:113).  Returns (y1, y2).  The mask depends only on
    (seed, offset, element index): call it again on the gradients with the same arguments for the backward pass."""
    x1p, ld1, f1 = _mat(x1, "dropout.x1")
    n = x1.shape[0]
    x2p, ld2, f2 = (None, 0, 0)
    if x2 is not None:
        x2p, ld2, f2 = _mat(x2, "dropout.x2")
        if x2.shape[0] != n:
            raise GteError("dropout_concat: row mismatch")
    if out is not None:
        y1, y2 = out
    else:
        y1 = x1 if inplace else empty_padded(n, f1, x1.device)
        y2 = None if x2 is None else (x2 if inplace else empty_padded(n, f2, x1.device))
    y1p, ldy1, _ = _mat(y1, "dropout.y1")
    y2p, ldy2 = (None, 0) if y2 is None else _mat(y2, "dropout.y2")[:2]
    check(lib().gte_dropout_concat(x1p, ld1, f1, x2p, ld2, f2, n, float(p), int(seed) & (2 ** 64 - 1), int(offset),
                                   _vec(rng_dev, "rng_dev", torch.int64, 2), y1p, ldy1, y2p, ldy2, _stream()),
          "gte_dropout_concat")
    return y1, y2


def dropout_counters(n: int, f: int) -> int:
    """Philox counters one dropout_concat launch over n x f elements consumes."""
    return (int(n) * int(f) + 3) // 4


def rng_advance(rng_dev: torch.Tensor, by: int) -> None:
    check(lib().gte_rng_advance(_vec(rng_dev, "rng_dev", torch.int64, 2), int(by), _stream()), "gte_rng_advance")


def relu_fwd(z, out=None):
    zp, ldz, f = _mat(z, "relu.z")
    n = z.shape[0]
    if out is None:
        out = empty_padded(n, f, z.device)
    yp, ldy, _ = _mat(out, "relu.y")
    check(lib().gte_relu_fwd(zp, ldz, yp, ldy, n, f, _stream()), "gte_relu_fwd")
    return out


def relu_bwd(dy, z, out=None):
    dyp, lddy, f = _mat(dy, "relu_bwd.dy")
    zp, ldz, _ = _mat(z, "relu_bwd.z")
    n = dy.shape[0]
    if out is None:
        out = empty_padded(n, f, dy.device)
    dzp, lddz, _ = _mat(out, "relu_bwd.dz")
    check(lib().gte_relu_bwd(dyp, lddy, zp, ldz, dzp, lddz, n, f, _stream()), "gte_relu_bwd")
    return out


# ------------------------------------------------------- loss / optimiser ---
_LABEL_DT = {torch.int64: _lib.GTE_LABEL_I64, torch.int32: _lib.GTE_LABEL_I32, torch.float32: _lib.GTE_LABEL_F32}


def _labels(labels: torch.Tensor):
    _req_cuda(labels)
    if labels.dtype not in _LABEL_DT or not labels.is_contiguous():
        raise GteError(f"labels: expected contiguous int64/int32/float32, got {labels.dtype}")
    return labels.data_ptr(), _LABEL_DT[labels.dtype]


def cross_entropy_fwd(logits, labels, class_w=None, stats=None):
    """stats = [sum w*nll, sum w, #correct] (float32[3], device)."""
    lp, ld, c = _mat(logits, "ce.logits")
    n = logits.shape[0]
    yp, ydt = _labels(labels)
    if labels.numel() != n:
        raise GteError("cross_entropy: labels/logits row mismatch")
    if stats is None:
        stats = torch.empty(3, dtype=torch.float32, device=logits.device)
    l = lib()
    ws = workspace(l.gte_cross_entropy_workspace_bytes(n), logits.device)
    check(
        l.gte_cross_entropy_fwd(lp, ld, yp, ydt, _vec(class_w, "class_w", n=c), n, c, _vec(stats, "stats", n=3),
                                ws.data_ptr(), ws.numel(), _stream()),
        "gte_cross_entropy_fwd",
    )
    return stats


def eval_accumulate(logits, labels, class_w, totals):
    """Add one batch's validation statistics to ``totals`` (float64 [2 + C*C], device; gte_eval_accumulate):
    [0] += sum w[y]*nll, [1] += sum w[y], [2 + y*C + argmax] += 1 over the rows with a label in [0, C)."""
    lp, ld, c = _mat(logits, "eval.logits")
    n = logits.shape[0]
    yp, ydt = _labels(labels)
    if labels.numel() != n:
        raise GteError("eval_accumulate: labels/logits row mismatch")
    tp = _vec(totals, "eval.totals", torch.float64)
    if totals.numel() != 2 + c * c:
        raise GteError(f"eval_accumulate: totals has {totals.numel()} elements, expected 2 + {c}*{c}")
    l = lib()
    ws = workspace(l.gte_eval_workspace_bytes(n), logits.device)
    check(l.gte_eval_accumulate(lp, ld, yp, ydt, _vec(class_w, "class_w", n=c), n, c, tp, ws.data_ptr(), ws.numel(),
                                _stream()), "gte_eval_accumulate")
    return totals


def cross_entropy_bwd_comb(logits, labels, class_w, denominator, width: int = COMB_LD):
    """d logits written in place as the self block of a fresh combined [n, 32] operand (other columns zero).
    ``width`` (tests): any multiple of 4 >= c gives an [n, width] matrix with columns [c, width) zeroed."""
    lp, ld, c = _mat(logits, "ce.logits")
    n = logits.shape[0]
    if width == COMB_LD and c > COMB_W:
        raise GteError("cross_entropy_bwd_comb: more than 16 classes")
    yp, ydt = _labels(labels)
    _req_cuda(denominator)
    out = torch.empty((n, width), dtype=torch.float32, device=logits.device)
    check(
        lib().gte_cross_entropy_bwd_padded(lp, ld, yp, ydt, _vec(class_w, "class_w", n=c), n, c, denominator.data_ptr(),
                                           out.data_ptr(), width, width, _stream()),
        "gte_cross_entropy_bwd_padded",
    )
    return out


def cross_entropy_bwd(logits, labels, class_w, denominator, out=None):
    lp, ld, c = _mat(logits, "ce.logits")
    n = logits.shape[0]
    yp, ydt = _labels(labels)
    if out is None:
        out = empty_padded(n, c, logits.device)
    dp, ldd, _ = _mat(out, "ce.dlogits")
    _req_cuda(denominator)
    check(
        lib().gte_cross_entropy_bwd(lp, ld, yp, ydt, _vec(class_w, "class_w", n=c), n, c, denominator.data_ptr(), dp,
                                    ldd, _stream()),
        "gte_cross_entropy_bwd",
    )
    return out


def _hparams_or_values(where: str, hparams, values):
    """``hparams`` (device float32 [5]: lr, beta1, beta2, eps, weight_decay) or the five values, not both"""
    given = [v is not None for v in values]
    if hparams is not None:
        if any(given):
            raise GteError(f"{where}: pass the hyper-parameters either as values or as an hparams tensor, not both")
        return _vec(hparams, "hparams", n=5)
    if not all(given):
        raise GteError(f"{where}: the hyper-parameters are required, as values or as an hparams tensor")
    return None


def adam_step(param, grad, exp_avg, exp_avg_sq, *, lr=None, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
              step: int = 0, step_dev: Optional[torch.Tensor] = None, grad_scale: float = 1.0,
              grad_den: Optional[torch.Tensor] = None, count: Optional[int] = None,
              hparams: Optional[torch.Tensor] = None):
    """Adam over flat buffers (gte.h).  ``hparams`` (device float32 [5] = [lr, beta1, beta2, eps, weight_decay]) takes
    the place of the five values: the kernel reads them when it runs, so a captured step follows later writes."""
    count = param.numel() if count is None else int(count)
    for t, nm in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _vec(t, nm, n=count)
    if step_dev is not None:
        _vec(step_dev, "step_dev", torch.int64, 1)
    hp = _hparams_or_values("adam_step", hparams, (lr,))
    if hp is not None:
        check(lib().gte_adam_step_dev(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                      count, hp, int(step), _ptr(step_dev), float(grad_scale),
                                      _vec(grad_den, "grad_den", n=1), _stream()),
              "gte_adam_step_dev")
        return
    check(
        lib().gte_adam_step(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), count,
                            float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
                            _ptr(step_dev), float(grad_scale), _vec(grad_den, "grad_den", n=1), _stream()),
        "gte_adam_step",
    )


def dp_allreduce_adam(peer_grad_ptrs_dev: int, peer_signal_ptrs_dev: int, rank: int, world: int, count: int, stats_off: int,
                      param, exp_avg, exp_avg_sq, stats_out, *, lr=None, beta1=None, beta2=None, eps=None,
                      weight_decay=None, step_dev, local_words, hparams: Optional[torch.Tensor] = None):
    """One-shot all-reduce of the ranks' flat gradient buffers over NVLink peer memory fused with Adam (gte.h); the
    hyper-parameters as five values or as a device ``hparams`` tensor (see ``adam_step``)."""
    for t, nm in ((param, "param"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _vec(t, nm, n=count)
    hp = _hparams_or_values("dp_allreduce_adam", hparams, (lr, beta1, beta2, eps, weight_decay))
    head = (int(peer_grad_ptrs_dev), int(peer_signal_ptrs_dev), int(rank), int(world), int(count), int(stats_off),
            param.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), _vec(stats_out, "stats_out", n=3))
    tail = (_vec(step_dev, "step_dev", torch.int64, 1), _vec(local_words, "local_words", torch.int32, 4), _stream())
    if hp is not None:
        check(lib().gte_dp_allreduce_adam_dev(*head, hp, *tail), "gte_dp_allreduce_adam_dev")
    else:
        check(lib().gte_dp_allreduce_adam(*head, float(lr), float(beta1), float(beta2), float(eps), float(weight_decay),
                                          *tail), "gte_dp_allreduce_adam")


# ------------------------------------------- either side of the layers ----
def page_predictions(logits, page_off, num_pages: int, labels=None):
    """``logits.argmax(1)`` for a batch of pages + per-page number of correct predictions
    (model_predict.py:144-148).  Returns (preds int32 [N], page_correct int32 [P] or None)."""
    lp, ld, c = _mat(logits, "page_predictions.logits")
    n = logits.shape[0]
    preds = torch.empty(n, dtype=torch.int32, device=logits.device)
    correct = None
    labp, ldt = None, _lib.GTE_LABEL_I64
    if labels is not None:
        if labels.numel() != n:
            raise GteError("page_predictions: one label per node expected")
        labp, ldt = _labels(labels)
        correct = torch.empty(max(num_pages, 1), dtype=torch.int32, device=logits.device)
    check(lib().gte_page_predictions(lp, ld, n, c, labp, ldt, _vec(page_off, "page_off", torch.int32, num_pages + 1), num_pages,
                                     preds.data_ptr(), _ptr(correct), _stream()), "gte_page_predictions")
    return preds, (correct[:num_pages] if correct is not None else None)


def page_formats_supported(pages) -> bool:
    return pages is not None and pages[1] > 0 and lib().gte_build_page_formats_smem_bytes(int(pages[2]), int(pages[3])) > 0


def build_page_formats(src, dst, w, page_off, edge_off, num_pages: int, n: int, max_nodes: int, max_edges: int):
    """One-kernel batch assembly (gte_build_page_formats): returns
    (csc, csr, norm, pk_csc, pk_csr, bad) with csc/csr = (indptr, indices, eid), pk_* = PackedEdges, bad = device int32
    flag (1 when an edge leaves its page: the dgl.batch contract is broken and the results are undefined)."""
    _req_cuda(src, dst, w, page_off, edge_off)
    e = src.numel()
    dev = src.device
    i32 = torch.int32
    csc = (torch.empty(n + 1, dtype=i32, device=dev), torch.empty(e, dtype=i32, device=dev), torch.empty(e, dtype=i32, device=dev))
    csr = (torch.empty(n + 1, dtype=i32, device=dev), torch.empty(e, dtype=i32, device=dev), torch.empty(e, dtype=i32, device=dev))
    pk_in = torch.empty(e + 2, dtype=torch.int64, device=dev)
    pk_out = torch.empty(e + 2, dtype=torch.int64, device=dev)
    norm = torch.empty(n, dtype=torch.float32, device=dev)
    flag = torch.empty(max(num_pages, 1), dtype=i32, device=dev)
    bad = torch.empty(1, dtype=i32, device=dev)
    check(lib().gte_build_page_formats(_vec(src, "src", i32), _vec(dst, "dst", i32), _vec(w, "w", n=e),
                                       _vec(page_off, "page_off", i32, num_pages + 1), _vec(edge_off, "edge_off", i32, num_pages + 1),
                                       num_pages, n, e, max_nodes, max_edges, csc[0].data_ptr(), csc[1].data_ptr(), csc[2].data_ptr(),
                                       pk_in.data_ptr(), csr[0].data_ptr(), csr[1].data_ptr(), csr[2].data_ptr(), pk_out.data_ptr(),
                                       norm.data_ptr(), flag.data_ptr(), bad.data_ptr(), _stream()), "gte_build_page_formats")
    pk_csc = PackedEdges(pk_in, flag, csc[1], csc[2], w, None)
    pk_csr = PackedEdges(pk_out, flag, csr[1], csr[2], w, norm)
    return csc, csr, norm, pk_csc, pk_csr, bad


def pad_batch(word, page_off, edge_off, src, dst, weight, feat, label, bad: Optional[torch.Tensor] = None):
    """Pad a page batch in place to the capacity shape its buffers have (gte_pad_batch): ``word`` = device int32
    (n, e, P) of the real prefix, ``page_off`` / ``edge_off`` the full int32 page table [p_cap + 1] (real pages,
    padding pages, empty pages), ``src`` / ``dst`` int32 and ``weight`` fp32 [e_cap], ``feat`` [n_cap, f],
    ``label`` fp32 [n_cap].  Returns the device int32 flag (bit 0: word outside the capacity, bit 1: page table
    inconsistent)."""
    i32 = torch.int32
    _req_cuda(word, page_off, edge_off, src, dst, weight, feat, label, bad)
    fp, ldf, f = _mat(feat, "pad_batch.feat")
    n_cap, e_cap, p_cap = int(feat.shape[0]), int(src.numel()), int(page_off.numel()) - 1
    if dst.numel() != e_cap or weight.numel() != e_cap or label.numel() != n_cap or edge_off.numel() != p_cap + 1:
        raise GteError("pad_batch: src / dst / weight need e_cap, label n_cap, edge_off p_cap + 1 entries")
    if bad is None:
        bad = torch.empty(1, dtype=i32, device=feat.device)
    check(lib().gte_pad_batch(_vec(word, "word", i32, 3), n_cap, e_cap, p_cap, _vec(page_off, "page_off", i32),
                              _vec(edge_off, "edge_off", i32), _vec(src, "src", i32), _vec(dst, "dst", i32),
                              _vec(weight, "weight"), fp, ldf, f, _vec(label, "label"), _vec(bad, "bad", i32, 1),
                              _stream()), "gte_pad_batch")
    return bad


PLAN_HEADER = 8  # [cursor, flag, nfit, B, L, 0, 0, 0] ahead of the ids and slice starts of an epoch plan


def gather_plan(plan, pool_num_nodes, pool_num_edges, capacity, meta):
    """Plan the next batch of an epoch plan on the device (gte_gather_plan): ``plan`` int32 [8 + 2 * pool pages]
    (layout in gte.h), ``pool_num_nodes`` / ``pool_num_edges`` int32 per pool page, ``capacity`` a BatchCapacity,
    ``meta`` the static set's int32 [4 + 2 * (P_cap + 1)] = (n, e, P, start | padded page table), written when the
    batch fits.  Raises plan[1] bits on the device: 1 = cursor past the plan, 2 = batch refused."""
    i32 = torch.int32
    pages = int(pool_num_nodes.numel())
    n_cap, e_cap, p_cap = capacity.shape
    if pool_num_edges.numel() != pages or pages < 1:
        raise GteError("gather_plan: need one node and one edge count per pool page")
    check(lib().gte_gather_plan(_vec(plan, "plan", i32, PLAN_HEADER + 2 * pages), _vec(pool_num_nodes, "pool_num_nodes", i32),
                                _vec(pool_num_edges, "pool_num_edges", i32), pages, capacity.nodes, capacity.edges,
                                capacity.pages, capacity.page_nodes, capacity.page_edges, n_cap, e_cap, p_cap,
                                _vec(meta, "meta", i32, 4 + 2 * (p_cap + 1)), _stream()), "gte_gather_plan")


def gather_pages(plan, meta, capacity, pool_node_off, pool_edge_off, pool_src, pool_dst, pool_weight, pool_feat,
                 pool_label, src, dst, weight, feat, label):
    """Copy the batch ``meta`` describes (gather_plan) from the pool into the real prefix of a capacity static set
    (gte_gather_pages): ``pool_*`` = page-local COO, weights, features [N_pool, f], labels and int64 node / edge
    offsets [pool pages + 1]; ``src`` / ``dst`` / ``weight`` [E_cap], ``feat`` [N_cap, f] contiguous, ``label``
    [N_cap].  Copies nothing while plan[1] is non-zero (the plan kernel refused the batch); a page the page table
    does not describe raises plan[1] bit 4 and is skipped."""
    i32, i64 = torch.int32, torch.int64
    n_cap, e_cap, p_cap = capacity.shape
    pages = int(pool_node_off.numel()) - 1
    f = int(feat.shape[1]) if feat.dim() == 2 else -1
    if pool_feat.dim() != 2 or int(pool_feat.shape[1]) != f or not feat.is_contiguous() or not pool_feat.is_contiguous():
        raise GteError(f"gather_pages: pool features {tuple(pool_feat.shape)} and batch features {tuple(feat.shape)} "
                       "must be contiguous with the same width")
    if feat.shape[0] != n_cap or label.numel() != n_cap or src.numel() != e_cap or dst.numel() != e_cap \
            or weight.numel() != e_cap or pool_edge_off.numel() != pages + 1:
        raise GteError("gather_pages: static set or pool offsets of the wrong size")
    check(lib().gte_gather_pages(_vec(plan, "plan", i32, PLAN_HEADER + 2 * pages), _vec(meta, "meta", i32, 4 + 2 * (p_cap + 1)),
                                 n_cap, e_cap, p_cap, capacity.pages, _vec(pool_node_off, "pool_node_off", i64),
                                 _vec(pool_edge_off, "pool_edge_off", i64), pages, _vec(pool_src, "pool_src", i32),
                                 _vec(pool_dst, "pool_dst", i32), _vec(pool_weight, "pool_weight"),
                                 _vec(pool_feat, "pool_feat"), _vec(pool_label, "pool_label"), f, _vec(src, "src", i32),
                                 _vec(dst, "dst", i32), _vec(weight, "weight"), _vec(feat, "feat"),
                                 _vec(label, "label"), _stream()), "gte_gather_pages")


def bbox_features(boxes: torch.Tensor, counts: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """13 BBOX features per text box (bbox.py:49-111) from int32 boxes [n,4] and character-class counts [n,3]."""
    _req_cuda(boxes, counts)
    if boxes.dtype != torch.int32 or counts.dtype != torch.int32 or boxes.dim() != 2 or boxes.shape[1] != 4 \
            or counts.shape != (boxes.shape[0], 3):
        raise GteError("bbox_features: boxes int32 [n,4] and counts int32 [n,3] expected")
    n = boxes.shape[0]
    if out is None:
        out = empty_padded(n, 13, boxes.device)
    op, ldo, f = _mat(out, "bbox_features.out")
    if f != 13 or out.shape[0] != n:
        raise GteError("bbox_features: output must be [n, 13]")
    check(lib().gte_bbox_features(boxes.contiguous().data_ptr(), counts.contiguous().data_ptr(), n, op, ldo, _stream()),
          "gte_bbox_features")
    return out
