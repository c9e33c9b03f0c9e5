"""Forward / backward of one GraphSAGE layer on the CUDA kernels.

Restates ``GcnSAGELayer.forward`` (/root/reference/src/components/graphs/models.py:46-78)
and ``WeightedMeanSAGELayer.forward`` (models.py:133-152) plus what torch/DGL
autograd derives from them, as explicit kernel sequences:

    ah  = post(v) * sum_{u->v} w_e h[u]           gte_spmm on the CSC
    z   = [h | ah] W^T + b                        gte_linear_fwd (no concat buffer)
    out = relu(LayerNorm(z))                      gte_layernorm_act_fwd
    out = relu(z) / max(||relu(z)||, eps)         gte_relu_l2norm_fwd (``l2``: MeanSAGE's F.relu + F.normalize)

The tensor-core projection fuses either epilogue (gte_umma_linear_fwd's fuse_ln selector).

Two algebraically equal orders are used (A.(H W2^T) = (A.H) W2^T):
  * ``agg``  aggregate-then-project  (Fin <= Fout: aggregate the narrow input)
  * ``proj`` project-then-aggregate  (Fout <  Fin: e.g. 218 -> 9 aggregates 9 columns)

Backward (dz -> dW, db, dh) is the transposed pipeline with the reversed-graph
SpMM on the CSR (deterministic, no atomics).  Nothing here runs on the CPU.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import torch

from . import _lib, ops
from .graph import PageGraphBatch

# Dense-contraction route: wide hidden layers (a real dense contraction, SURVEY 8a) of batches of at least
# UMMA_MIN_ROWS nodes go to the tcgen05 3xTF32 kernels and everything else to the exact-fp32 FFMA kernels.
UMMA_MIN_ROWS = 1024
UMMA_MIN_WIDTH = 64
SKINNY_MIN_ROWS = 256  # below this the generic kernels are launch-latency bound anyway

GCN = "gcn"    # sum, then * 1/in_deg (0 for isolated nodes)  -- GcnSAGELayer
MEAN = "mean"  # sum / max(in_deg, 1)                          -- WeightedMeanSAGELayer (DGL fn.mean)


@dataclass
class DropoutSpec:
    """Training-mode dropout of one call site: probability + where its mask lives in the Philox stream (ops.dropout_concat)."""

    p: float
    seed: int = 0
    offset: int = 0
    rng_dev: Optional[torch.Tensor] = None  # device int64[2] (seed, base offset): captured steps draw fresh masks per replay

    def active(self) -> bool:
        return self.p > 0.0


@dataclass
class LayerCtx:
    strategy: str = "agg"
    agg: str = GCN
    h: Optional[torch.Tensor] = None
    ah: Optional[torch.Tensor] = None
    z: Optional[torch.Tensor] = None
    mean: Optional[torch.Tensor] = None
    rstd: Optional[torch.Tensor] = None
    w_edge: Optional[torch.Tensor] = None
    pack: Optional[torch.Tensor] = None  # tf32 hi/lo weight tiles when the layer ran on tensor cores
    ln: bool = False
    relu: bool = False
    fin: int = 0
    fout: int = 0
    drop: Optional[DropoutSpec] = None  # the mask of [h | ah] is recomputed from this in the backward pass
    comb: Optional[torch.Tensor] = None  # narrow input (fin <= 16): [h | ah] side by side in one [n, 32] operand
    l2: bool = False  # out = relu(z) / max(||relu(z)||, l2_eps): the backward recomputes the norm from z
    l2_eps: float = 1e-12


def pick_strategy(fin: int, fout: int, use_pp: bool) -> str:
    if use_pp:
        return "pp"
    return "proj" if fout < fin else "agg"


def use_umma(n: int, fin: int, fout: int, *mats) -> bool:
    """Tensor-core projection.  Also used for narrow K (input layer, K = 2*13): the kernel then is an
    output-bandwidth-bound fused bias+LayerNorm+ReLU epilogue, still far ahead of GEMM + separate LayerNorm."""
    if not ops.umma_supported(fout, fin):
        return False
    if not all(ops._aligned_mat(m) for m in mats if m is not None):
        return False
    return n >= UMMA_MIN_ROWS and max(fin, fout) >= UMMA_MIN_WIDTH


def use_umma_dw(n: int, fo: int, k1: int, k2: int, db_needed: bool, *mats) -> bool:
    """Tensor-core weight gradient: any width up to 256 (the reduction over all nodes is the long axis)."""
    if not ops.umma_bwd_weight_supported(fo, k1, k2):
        return False
    if not all(ops._aligned_mat(m) for m in mats if m is not None):
        return False
    if db_needed and k1 % 32 == 0:
        return False
    return n >= UMMA_MIN_ROWS


def _use_packed(g: PageGraphBatch, x: torch.Tensor, addend: Optional[torch.Tensor]) -> bool:
    """The persistent page kernel needs a page table, 16-byte aligned rows and two stages of the
    largest page in shared memory; everything else goes to gte_spmm_paged / gte_spmm."""
    if 16 < x.shape[1] <= 32:
        return False  # 5..8 chunks per row: the one-CTA-per-(page, slice) kernel measures faster (conv sweep, F = 32)
    return (ops.paged_packed_supported(g.pages(), x.shape[1]) and ops._aligned_mat(x)
            and (addend is None or ops._aligned_mat(addend)))


def _agg_mode(agg: str) -> int:
    return _lib.GTE_AGG_SUM_NORM if agg == GCN else _lib.GTE_AGG_MEAN


def aggregate_forward(g: PageGraphBatch, h: torch.Tensor, w_edge: torch.Tensor, agg: str = GCN,
                      addend: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``update_all(u_mul_e, sum|mean)`` (+ ``* norm``): models.py:53-54,69-71,149."""
    g.prepare(w_edge)  # first call per batch: CSC + CSR + norm + packed edges in one kernel
    indptr, indices, _ = g.csc()
    if _use_packed(g, h, addend):
        return ops.spmm_packed(indptr, g.packed_edges("csc", w_edge), h, g.pages(), mode=_agg_mode(agg),
                               row_norm=g.norm() if agg == GCN else None, addend=addend, out=out)
    return ops.spmm(indptr, indices, g.weights_csc(w_edge), h, mode=_agg_mode(agg),
                    row_norm=g.norm() if agg == GCN else None, addend=addend, pages=g.pages(), out=out)


def aggregate_backward(g: PageGraphBatch, d_out: torch.Tensor, w_edge: torch.Tensor,
                       addend: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d h[u] = sum_{u->v} w_e * norm[v] * d_out[v] (+ addend[u]) on the CSR (reverse graph)."""
    g.prepare(w_edge)
    indptr, indices, _ = g.csr()
    if _use_packed(g, d_out, addend):
        return ops.spmm_packed(indptr, g.packed_edges("csr", w_edge), d_out, g.pages(), mode=_lib.GTE_AGG_SUM,
                               addend=addend, out=out)
    return ops.spmm(indptr, indices, g.weights_csr(w_edge), d_out, mode=_lib.GTE_AGG_SUM, pre_scale=g.norm(),
                    addend=addend, pages=g.pages(), out=out)


def relu_l2norm_forward(z: torch.Tensor, eps: float) -> torch.Tensor:
    """``F.normalize(F.relu(z))`` of a layer whose projection did not fuse it (models.py:167-169)."""
    return ops.relu_l2norm_fwd(z, eps)


def relu_l2norm_backward(dy: torch.Tensor, z: torch.Tensor, eps: float, db: Optional[torch.Tensor],
                         accumulate: bool) -> torch.Tensor:
    """dz of ``F.normalize(F.relu(z))`` (the norm recomputed from z); ``db`` (may be None) receives (accumulate: gains)
    the column sums of dz, the linear-bias gradient, from the same pass."""
    if db is None:
        return ops.relu_l2norm_bwd(dy, z, eps)
    return ops.relu_l2norm_bwd_colsum(dy, z, eps, dz_colsum=db, accumulate=accumulate)


def _comb_rows(n: int) -> bool:
    """Combined [n, 32] operands for the narrow layers: a tensor-core batch."""
    return n >= UMMA_MIN_ROWS


def wants_pack(n: int, fin: int, fout: int, use_pp: bool) -> bool:
    """Could sage_layer_forward take a tensor-core branch for this layer (so a caller may pre-pack W for it)?"""
    return (not use_pp) and n >= UMMA_MIN_ROWS and ops.umma_supported(fout, fin)


def wants_class_grad_comb(ctx: "LayerCtx", n: int) -> bool:
    """The class layer's backward wants its incoming gradient as the self block of a combined [n, 32] operand
    (d logits | A_hat^T d logits): a caller that PRODUCES that gradient (the trainer's loss backward) builds it with
    ``ops.cross_entropy_bwd_comb`` (or ``ops.comb_from``) and passes the buffer as ``dy_comb``."""
    return (ctx.strategy == "proj" and not ctx.ln and not ctx.relu and not ctx.l2 and ctx.fout <= ops.COMB_W and ctx.pack is not None
            and _comb_rows(n) and ctx.fin <= 256 and ctx.fin % 32 != 0 and ops._aligned_mat(ctx.h))
    # fin % 32 != 0: the bias gradient rides on a free padding column of the input operand


def sage_layer_forward(g: Optional[PageGraphBatch], h: torch.Tensor, w_edge: Optional[torch.Tensor],
                       W: torch.Tensor, b: Optional[torch.Tensor], gamma: Optional[torch.Tensor],
                       beta: Optional[torch.Tensor], *, ln: bool, relu: bool, eps: float = 1e-5, agg: str = GCN,
                       use_pp: bool = False, strategy: Optional[str] = None, save_for_backward: bool = True,
                       dropout: Optional[DropoutSpec] = None, pack: Optional[torch.Tensor] = None,
                       l2: bool = False):
    """Returns (out [N, Fout], LayerCtx).  ``l2`` (MeanSAGE's hidden layers, models.py:167-169): out =
    relu(z) / max(||relu(z)||_2, eps) with ``eps`` the normalise eps (ln and relu off); the narrow input layer's
    tensor-core projection fuses it into its epilogue, the other routes run ``ops.relu_l2norm_fwd`` after the layer.  ``save_for_backward=False`` (inference): the fused tensor-core epilogue does not
    write the pre-activation z (it only exists for the backward pass).  ``dropout`` (training): nn.Dropout on the
    concatenation [h | ah * norm] before the linear (models.py:60-61), in-kernel Philox, never materialising the concat.
    ``pack``: ``ops.umma_pack_weights(W, fin, 2)`` of the CURRENT W when the caller already made it (the trainer packs all
    layers in one launch); otherwise the tensor-core branches pack W themselves."""
    fout = W.shape[0]
    fin = W.shape[1] if use_pp else W.shape[1] // 2
    if l2 and (ln or relu):
        raise _lib.GteError("sage_layer_forward: l2 is its own epilogue (ReLU included); pass ln=False, relu=False")
    if h.shape[1] != (W.shape[1] if use_pp else fin):
        raise _lib.GteError(f"layer expects {W.shape[1] if use_pp else fin} input features, got {h.shape[1]}")
    st = strategy or pick_strategy(fin, fout, use_pp)
    drop = dropout if (dropout is not None and dropout.active()) else None
    if drop is not None and st == "proj":
        st = "agg"  # the mask acts on [h | ah]: aggregate first
    xc = ahs = None
    if st == "agg" and fin <= ops.COMB_W and _comb_rows(h.shape[0]) and ops.umma_supported(fout, fin):
        # narrow input (the [N, 13] BBOX features): h and A_hat h side by side in one zero-padded [n, 32] operand --
        # aligned rows for the gather, ONE k-block for the projection, one full-row TMA box for the weight gradient
        xc = ops.comb_from(h)
        hs, ahs = ops.comb_views(xc, fin)
        h = hs
    elif h.shape[0] >= UMMA_MIN_ROWS and not ops._aligned_mat(h):
        # unaligned rows: one padded copy gives 16-byte aligned rows for TMA / 128-bit loads
        hp = ops.empty_padded(h.shape[0], h.shape[1], h.device)
        hp.copy_(h)
        h = hp
    ctx = LayerCtx(strategy=st, agg=agg, h=h, ln=ln, relu=relu, fin=fin, fout=fout, w_edge=w_edge, drop=drop, l2=l2,
                   l2_eps=eps if l2 else 1e-12)
    if st == "pp":  # pre-propagated input: plain linear (models.py:49)
        if drop is not None:
            h, _ = ops.dropout_concat(h, None, drop.p, drop.seed, drop.offset, drop.rng_dev)
            ctx.h = h
        z = ops.linear_fwd(h, None, W, b)
    elif st == "agg":
        ah = aggregate_forward(g, h, w_edge, agg, out=ahs)
        if drop is not None:
            # the dropped operands are what the linear (and, in backward, dW) sees; d[h | ah] gets the same mask back
            outs = None
            if xc is not None:
                xc = ops.comb_buffer(h.shape[0], h.device)
                outs = ops.comb_views(xc, fin)
            h, ah = ops.dropout_concat(h, ah, drop.p, drop.seed, drop.offset, drop.rng_dev, out=outs)
            ctx.h = h
        ctx.ah = ah
        if xc is not None:
            ctx.comb = xc
            ctx.pack = pack if pack is not None else ops.umma_pack_weights(W, fin, 2)
            z, y, ctx.mean, ctx.rstd = ops.umma_linear_fwd_comb(xc, fin, ctx.pack, b, fout, gamma=gamma, beta=beta,
                                                                eps=eps, relu=relu, fuse_ln=ln, want_z=save_for_backward,
                                                                l2=l2)
            ctx.z = z
            return (y if y is not None else z), ctx
        if use_umma(h.shape[0], fin, fout, h, ah):
            # tensor cores: projection + bias + LayerNorm + ReLU in one kernel.  ReLU + L2-normalise is not fused here:
            # these k loops (more than two k-blocks) keep one TMEM accumulator stage, whose second epilogue pass holds
            # up the next tile's MMAs -- at 218 -> 218 the projection followed by gte_relu_l2norm_fwd measured faster
            # (profiles/meansage_bench.json)
            ctx.pack = pack if pack is not None else ops.umma_pack_weights(W, fin, 2)
            z, y, ctx.mean, ctx.rstd = ops.umma_linear_fwd(h, ah, fin, ctx.pack, b, fout, gamma=gamma, beta=beta,
                                                           eps=eps, relu=relu, fuse_ln=ln,
                                                           want_z=save_for_backward or l2)
            if not l2:
                ctx.z = z
                return (y if y is not None else z), ctx
        elif (ln or not relu) and ops.wide_out_supported(fin, fin, fout, h, ah) and h.shape[0] >= SKINNY_MIN_ROWS:
            # exact-fp32 route for a narrow input (K = 2 * fin <= 32): one streaming pass, bias + LayerNorm + ReLU fused
            z, y, ctx.mean, ctx.rstd = ops.wide_out(h, ah, W.data_ptr(), W.data_ptr() + 4 * fin, 1, W.stride(0), fout, b,
                                                    gamma=gamma, beta=beta, eps=eps, relu=relu, fuse_ln=ln)
            if not l2:
                ctx.z = z
                return (y if y is not None else z), ctx
        else:
            z = ops.linear_fwd(h, ah, W, b)
    elif st == "proj":
        if fout <= 16 and use_umma(h.shape[0], fin, fout, h):
            # one tensor-core pass over h: [h Ws^T + b | h Wn^T] side by side, aggregated through column views
            ctx.pack = pack if pack is not None else ops.umma_pack_weights(W, fin, 2)
            sp = ops.umma_linear_fwd_stacked(h, fin, ctx.pack, b, fout)
            s, p = sp[:, :fout], sp[:, 16:16 + fout]
        else:
            s = ops.linear_fwd(h, None, W, b, w_col0=0)
            p = ops.linear_fwd(h, None, W, None, w_col0=fin)
        z = aggregate_forward(g, p, w_edge, agg, addend=s)
    else:
        raise _lib.GteError(f"unknown strategy {st}")
    ctx.z = z
    if ln:
        out, ctx.mean, ctx.rstd = ops.layernorm_act_fwd(z, gamma, beta, eps, relu)
    elif l2:
        out = relu_l2norm_forward(z, eps)
    elif relu:
        out = ops.relu_fwd(z)
    else:
        out = z
    return out, ctx


def sage_layer_backward(g: Optional[PageGraphBatch], ctx: LayerCtx, dy: torch.Tensor, W: torch.Tensor,
                        gamma: Optional[torch.Tensor], beta: Optional[torch.Tensor], dW: torch.Tensor,
                        db: Optional[torch.Tensor], dgamma: Optional[torch.Tensor], dbeta: Optional[torch.Tensor],
                        *, need_dh: bool, accumulate: bool = False,
                        dy_comb: Optional[torch.Tensor] = None, dh_agg_first: bool = False) -> Optional[torch.Tensor]:
    """Writes dW/db/dgamma/dbeta (overwrite or accumulate) and returns dh (or None).  ``dy_comb``: the buffer from
    class_grad_buffer() whose self block IS ``dy`` (saves one copy of the class-layer gradient).  ``dh_agg_first``: an
    aggregate-first tensor-core layer with fout <= fin and no dropout may build dh as [dz | A_hat^T dz] W (one SpMM of
    the narrower dz without an addend, one two-segment projection) instead of A_hat^T (dz Wn) + dz Ws; the sums then run
    in a different order, so callers that compare against the per-layer order leave it off."""
    fin, fout = ctx.fin, ctx.fout
    if ctx.ln:
        # the linear-bias gradient (column sums of dz) falls out of the same pass
        dz = ops.layernorm_act_bwd(dy, ctx.z, ctx.mean, ctx.rstd, gamma, beta, ctx.relu, dgamma, dbeta, accumulate,
                                   dz_colsum=db)
        db = None
    elif ctx.l2:
        # the same pass yields the linear-bias gradient, so the weight gradient below needs no bias column: every width
        # <= 256 keeps the tensor-core dW (its bias column needs fin % 32 != 0)
        dz = relu_l2norm_backward(dy, ctx.z, ctx.l2_eps, db, accumulate)
        db = None
    elif ctx.relu:
        dz = ops.relu_bwd(dy, ctx.z)
    else:
        dz = dy
    drop = ctx.drop
    if ctx.strategy == "pp":
        ops.linear_bwd_weight(dz, ctx.h, None, dW, db, accumulate)
        if not need_dh:
            return None
        dh = ops.linear_bwd_data(dz, W, 0, W.shape[1])
        if drop is not None:
            ops.dropout_concat(dh, None, drop.p, drop.seed, drop.offset, drop.rng_dev, inplace=True)
        return dh
    if ctx.strategy == "agg":
        if ctx.comb is not None and ops._aligned_mat(dz) and fout <= 256 and (db is None or fin < ops.COMB_W):
            ops.umma_linear_bwd_weight_comb(dz, ctx.comb, fin, dW, db, accumulate)
        elif use_umma_dw(dz.shape[0], fout, fin, fin, db is not None, dz, ctx.h, ctx.ah):
            ops.umma_linear_bwd_weight(dz, ctx.h, ctx.ah, dW, db, accumulate)
        elif (db is None and 2 * fin <= 32 and dz.shape[0] >= SKINNY_MIN_ROWS and dW.stride(1) == 1
              and ops.gram_stream_supported(fout, 2 * fin, dz, ctx.h, ctx.ah)):
            # narrow input: stream dz once against [h | ah] (exact fp32, fixed-order reduction)
            ops.gram_stream(dz, ctx.h, ctx.ah, dW, dW.stride(0), 1, dW[:, fin:], dW.stride(0), 1, accumulate=accumulate)
        else:
            ops.linear_bwd_weight(dz, ctx.h, ctx.ah, dW, db, accumulate)
        if not need_dh:
            return None
        if dh_agg_first and drop is None and fout <= fin and ctx.pack is not None and ops._aligned_mat(dz):
            # dh = dz Ws + A_hat^T (dz Wn) = [dz | A_hat^T dz] W: 5 instead of 6 passes over an [n, fin] matrix
            # (the mask of [h | ah] sits between the projection and A_hat^T, hence no dropout)
            return ops.umma_linear_bwd_data2(dz, aggregate_backward(g, dz, ctx.w_edge), ctx.pack, fin)
        if ctx.pack is not None and ops._aligned_mat(dz):
            d_self, d_ah = ops.umma_linear_bwd_data(dz, ctx.pack, fin, 2)
        else:
            d_self = ops.linear_bwd_data(dz, W, 0, fin)
            d_ah = ops.linear_bwd_data(dz, W, fin, fin)
        if drop is not None:  # same mask as in the forward pass, recomputed
            ops.dropout_concat(d_self, d_ah, drop.p, drop.seed, drop.offset, drop.rng_dev, inplace=True)
        return aggregate_backward(g, d_ah, ctx.w_edge, addend=d_self)
    # proj: z = h Ws^T + b + A_hat (h Wn^T)  =>  with G = A_hat^T dz:
    #   dWs = dz^T h, dWn = G^T h, dh = dz Ws + G Wn
    dc = dy_comb
    if dc is None and wants_class_grad_comb(ctx, dz.shape[0]):
        dc = ops.comb_from(dz)
    if dc is not None:
        # [dz | A_hat^T dz] side by side: one full-row TMA box for the weight gradient, one k-block for dh
        dzv, gqv = ops.comb_views(dc, fout)
        aggregate_backward(g, dzv, ctx.w_edge, out=gqv)
        ops.umma_linear_bwd_weight2_comb(dc, fout, ctx.h, dW, 0, fin, db, accumulate)
        return ops.umma_linear_bwd_data_comb(dc, fout, ctx.pack, fin) if need_dh else None
    gq = aggregate_backward(g, dz, ctx.w_edge)
    if (2 * fout <= 32 and dz.shape[0] >= SKINNY_MIN_ROWS and dW.stride(1) == 1
            and ops.gram_stream_supported(fin, 2 * fout, ctx.h, dz, gq)):
        # class layer: stream the wide input once against [dz | A^T dz]; the column sums of dz are the bias gradient
        ops.gram_stream(ctx.h, dz, gq, dW, 1, dW.stride(0), dW[:, fin:], 1, dW.stride(0), qsum=db, accumulate=accumulate)
    elif (fout <= 32 and fin <= 256 and (db is None or fin % 128 != 0) and dz.shape[0] >= UMMA_MIN_ROWS and
            all(ops._aligned_mat(m) for m in (dz, gq, ctx.h))):
        ops.umma_linear_bwd_weight2(dz, gq, ctx.h, dW, 0, fin, db, accumulate)
    else:
        ops.linear_bwd_weight2(dz, gq, ctx.h, dW, 0, fin, db, accumulate)
    if not need_dh:
        return None
    if ctx.pack is not None and ops._aligned_mat(dz) and ops._aligned_mat(gq):
        return ops.umma_linear_bwd_data2(dz, gq, ctx.pack, fin)
    if ops.wide_out_supported(fout, fout, fin, dz, gq) and dz.shape[0] >= SKINNY_MIN_ROWS and W.stride(1) == 1:
        return ops.wide_out(dz, gq, W.data_ptr(), W.data_ptr() + 4 * fin, W.stride(0), 1, fin)[0]  # exact fp32
    return ops.linear_bwd_data2(dz, 0, gq, fin, W, fin)


# ------------------------------------------------------------- autograd ----
def _as_mat(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() != 2:
        raise _lib.GteError(f"expected a 2-D feature matrix, got {tuple(t.shape)}")
    if t.shape[1] > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if t.shape[0] > 1 and t.stride(0) < t.shape[1]:
        t = t.contiguous()
    return t


def _no_edge_grad(w_edge):
    """The reference's edge weights are data (loader.py:332-344): DGL would compute d(edata) through gsddmm only if
    they required grad.  That kernel is not part of this path, so refuse instead of silently returning None."""
    if w_edge is not None and w_edge.requires_grad:
        raise _lib.GteError("edge weights that require grad are not supported (no edge-weight gradient kernel); "
                            "detach edata['feat'] -- the reference never trains them")


class SageLayerFunction(torch.autograd.Function):
    """One fused autograd node per layer (replaces ~10 ATen/DGL nodes of the reference)."""

    @staticmethod
    def forward(ctx, h, W, b, gamma, beta, w_edge, g, ln, relu, eps, agg, use_pp, drop=None):
        _no_edge_grad(w_edge)
        ctx.in_dtype = h.dtype
        h = _as_mat(h.detach())
        with torch.cuda.device(h.device):  # launch on the tensors' device, whatever the caller's current device is
            out, lctx = sage_layer_forward(g, h, None if w_edge is None else w_edge.detach(), W.detach(),
                                           None if b is None else b.detach(),
                                           None if gamma is None else gamma.detach(),
                                           None if beta is None else beta.detach(),
                                           ln=ln, relu=relu, eps=eps, agg=agg, use_pp=use_pp, dropout=drop)
        ctx.lctx = lctx  # kept until the node is freed, so backward(retain_graph=True) can run again
        ctx.g = g
        ctx.save_for_backward(W, gamma, beta)
        ctx.has_b = b is not None
        return out

    @staticmethod
    def backward(ctx, dy):
        W, gamma, beta = ctx.saved_tensors
        lctx = ctx.lctx
        dy = _as_mat(dy)
        dev = dy.device
        dW = torch.empty_like(W)
        db = torch.empty(W.shape[0], dtype=torch.float32, device=dev) if ctx.has_b else None
        dgamma = torch.empty_like(gamma) if lctx.ln else None
        dbeta = torch.empty_like(beta) if lctx.ln else None
        with torch.cuda.device(dev):
            dh = sage_layer_backward(ctx.g, lctx, dy, W.detach(), None if gamma is None else gamma.detach(),
                                     None if beta is None else beta.detach(), dW, db, dgamma, dbeta,
                                     need_dh=ctx.needs_input_grad[0])
        if dh is not None and dh.dtype != ctx.in_dtype:
            dh = dh.to(ctx.in_dtype)
        return dh, dW, db, dgamma, dbeta, None, None, None, None, None, None, None, None


class DropoutFunction(torch.autograd.Function):
    """``nn.Dropout(p)`` in training mode on one feature matrix (models.py:113), native kernel, mask recomputed in backward."""

    @staticmethod
    def forward(ctx, x, drop):
        ctx.drop, ctx.in_dtype = drop, x.dtype
        x = _as_mat(x.detach())
        with torch.cuda.device(x.device):
            return ops.dropout_concat(x, None, drop.p, drop.seed, drop.offset, drop.rng_dev)[0]

    @staticmethod
    def backward(ctx, dy):
        dy = _as_mat(dy)
        d = ctx.drop
        with torch.cuda.device(dy.device):
            dx = ops.dropout_concat(dy, None, d.p, d.seed, d.offset, d.rng_dev)[0]
        return (dx if dx.dtype == ctx.in_dtype else dx.to(ctx.in_dtype)), None


def torch_generator_dropout_spec(p: float, device: torch.device, n: int, f: int) -> DropoutSpec:
    """A DropoutSpec keyed from torch's CUDA generator of `device` (the seed torch.manual_seed set), advancing that
    generator's Philox offset past the counters this call site will consume -- reproducible under the same seed."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    gen = torch.cuda.default_generators[idx]
    seed, off = int(gen.initial_seed()), int(gen.get_offset())
    need = ops.dropout_counters(n, f)
    gen.set_offset(off + 4 * need)  # torch keeps the offset a multiple of 4; the next call site starts past this one
    return DropoutSpec(float(p), seed, off)


class AggregateFunction(torch.autograd.Function):
    """``update_all(u_mul_e, sum|mean)`` (+ norm) as a stand-alone differentiable op."""

    @staticmethod
    def forward(ctx, h, w_edge, g, agg):
        _no_edge_grad(w_edge)
        ctx.in_dtype = h.dtype
        h = _as_mat(h.detach())
        ctx.g, ctx.w_edge = g, w_edge.detach()
        with torch.cuda.device(h.device):
            return aggregate_forward(g, h, ctx.w_edge, agg)

    @staticmethod
    def backward(ctx, dy):
        dy = _as_mat(dy)
        with torch.cuda.device(dy.device):
            dh = aggregate_backward(ctx.g, dy, ctx.w_edge)
        return (dh if dh.dtype == ctx.in_dtype else dh.to(ctx.in_dtype)), None, None, None


class ReluL2NormFunction(torch.autograd.Function):
    """``F.normalize(F.relu(z))`` (models.py:167-169)."""

    @staticmethod
    def forward(ctx, z, eps):
        z = _as_mat(z.detach())
        ctx.z, ctx.eps = z, eps
        with torch.cuda.device(z.device):
            return ops.relu_l2norm_fwd(z, eps)

    @staticmethod
    def backward(ctx, dy):
        dy = _as_mat(dy)
        with torch.cuda.device(dy.device):
            return ops.relu_l2norm_bwd(dy, ctx.z, ctx.eps), None


class CrossEntropyFunction(torch.autograd.Function):
    """``nn.CrossEntropyLoss(weight)(logits, labels)`` (model_train.py:171,327)."""

    @staticmethod
    def forward(ctx, logits, labels, class_w):
        logits = _as_mat(logits.detach())
        with torch.cuda.device(logits.device):
            stats = ops.cross_entropy_fwd(logits, labels, class_w)
        ctx.logits, ctx.labels, ctx.class_w, ctx.stats = logits, labels, class_w, stats
        return stats[0] / stats[1]

    @staticmethod
    def backward(ctx, dloss):
        with torch.cuda.device(ctx.logits.device):
            dl = ops.cross_entropy_bwd(ctx.logits, ctx.labels, ctx.class_w, ctx.stats[1:2])
        return dl * dloss, None, None


def cross_entropy(logits: torch.Tensor, labels: torch.Tensor, weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    if labels.dtype not in (torch.int64, torch.int32, torch.float32):
        labels = labels.long()
    return CrossEntropyFunction.apply(logits, labels.contiguous(), weight)
