"""torch.autograd.Function drop-ins over the C ABI (include/rgbmp.h).

Every function here enqueues hand-written sm_100a kernels from librgbmp.so on the current
CUDA stream.  Nothing falls back to PyTorch arithmetic for the aggregation itself; PyTorch only
provides the tensors (device memory), the stream and the autograd graph.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple, Optional, Tuple

import torch

from . import _lib, memo
from ._lib import Epilogue, check, dtype_code, lib, ptr, stream_of
from .graph import CSR, Graph, NORM_COUNT, NORM_INV_SQRT, oom_retry

RESET_NONE, RESET_BEFORE_TELEPORT, RESET_AFTER_CLAMP = 0, 1, 2
TUNE_OVERRIDE = 0      # experiments (tools/): launch-shape word applied to every SpMM / K-hop call that passes tune=0


# ------------------------------------------------------------------------------------------
# buffer helpers: the vector path wants 16-byte aligned rows (ld % 4 == 0 fp32, % 8 bf16)
# ------------------------------------------------------------------------------------------
def _vec(dtype) -> int:
    return 8 if dtype == torch.bfloat16 else 4


def padded_width(F: int, dtype=torch.float32) -> int:
    v = _vec(dtype)
    return (F + v - 1) // v * v


def as_rows(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Return (tensor usable by the kernels, leading dimension).  No copy when `x` is already
    row-major with an aligned row stride; otherwise one copy into a zero-padded buffer."""
    _lib.require_cuda(x, "x")
    if x.dim() != 2:
        raise RuntimeError("feature matrix must be 2-D [rows, F]")
    N, F = x.shape
    v = _vec(x.dtype)
    if (x.stride(1) == 1 or F == 1) and x.stride(0) % v == 0 and x.stride(0) >= padded_width(F, x.dtype) \
            and x.data_ptr() % 16 == 0:
        return x, x.stride(0)
    Fp = padded_width(F, x.dtype)
    if Fp == F:
        buf = x.contiguous()
        if buf.data_ptr() % 16 == 0:
            return buf, F
    buf = torch.zeros((N, Fp), dtype=x.dtype, device=x.device)
    buf[:, :F].copy_(x)
    return buf[:, :F], Fp


def alloc_rows(N: int, F: int, dtype, device) -> Tuple[torch.Tensor, int]:
    """Fresh [N, F] tensor whose rows are padded(F) elements apart (16-byte aligned rows for the vector kernels).
    NOT a view: the result of an autograd.Function must tolerate the caller's in-place update (`out += x_r`,
    graphsage.py:60, SURVEY B8), which autograd forbids on a view created inside a custom Function -- so the
    strided tensor is bound to the padded storage directly instead of slicing a [N, padded(F)] tensor."""
    Fp = padded_width(F, dtype)
    buf = torch.empty((N, Fp), dtype=dtype, device=device)
    if Fp == F:
        return buf, Fp
    out = torch.empty(0, dtype=dtype, device=device).set_(buf.untyped_storage(), buf.storage_offset(), (N, F), (Fp, 1))
    return out, Fp


def make_epilogue(*, row_scale=None, row_div=False, a=1.0, b=0.0, T=None, ldt=0, clamp=None,
                  reset_mask=None, reset_val=None, ld_reset=0, reset_when=RESET_NONE,
                  out2_scale=None, acc_in=None, ld_acc=0, skip_empty=False, peers=(), peer_row0=0,
                  ld_peer=0, row_map=None) -> Epilogue:
    e = Epilogue()
    e.row_scale, e.row_div = ptr(row_scale), int(bool(row_div))
    e.reset_mask, e.reset_val, e.ld_reset, e.reset_when = ptr(reset_mask), ptr(reset_val), ld_reset, reset_when
    e.a, e.b, e.T, e.ldt = float(a), float(b), ptr(T), ldt
    if clamp is not None:
        e.clamp, e.lo, e.hi = 1, float(clamp[0]), float(clamp[1])
    e.out2_scale = ptr(out2_scale)
    e.acc_in, e.ld_acc, e.skip_empty = ptr(acc_in), ld_acc, int(bool(skip_empty))
    if len(peers) > 8:
        raise RuntimeError("at most 8 peer buffers (one NVSwitch box)")
    for q, pp in enumerate(peers):          # raw device pointers (ints) of peer-mapped buffers
        e.peer_out[q] = int(pp)
    e.n_peers, e.peer_row0, e.ld_peer = len(peers), int(peer_row0), int(ld_peer)
    e.row_map = ptr(row_map)
    return e


def reset_rows(mask: torch.Tensor, vals: torch.Tensor, F: int) -> dict:
    """make_epilogue keywords of label propagation's fixed-scale post-step: after the clamp, the rows where `mask` is set
    take the first F columns of their `vals` (RESET_AFTER_CLAMP).  The epilogue reads a byte per row and the values as
    float32 rows whatever the feature dtype; tensors already in that form are used without a copy."""
    _lib.require_cuda(mask, "reset mask")
    rv, ldr = as_rows(vals[:, :F].float())
    return dict(reset_mask=mask.to(torch.uint8).contiguous(), reset_val=rv, ld_reset=ldr, reset_when=RESET_AFTER_CLAMP)


def _graph_ref(csr, row_bytes: int, hot: bool = True):
    if hot and hasattr(csr, "hot_ref"):
        return csr.hot_ref(row_bytes)
    return csr.ref


def spmm_raw(csr: CSR, x: torch.Tensor, val: Optional[torch.Tensor] = None, **kw) -> Optional[torch.Tensor]:
    """y[i] = epilogue(sum_k val[k] * x[col[k]]); see _spmm_raw.  A CUDA OOM empties the graph / memo caches and
    retries once (graph.oom_retry)."""
    return oom_retry(lambda: _spmm_raw(csr, x, val, **kw))


def _spmm_raw(csr: CSR, x: torch.Tensor, val: Optional[torch.Tensor] = None, *, ep: Optional[Epilogue] = None,
              keep=(), tune: int = 0, out: Optional[torch.Tensor] = None, hot: bool = True,
              store_local: bool = True) -> Optional[torch.Tensor]:
    """`keep` holds tensors referenced by `ep`.
    hot=True lets feature matrices beyond the L2 budget use the hot-tagged column ids (graph.CSR.hot_ref)."""
    tune = tune or TUNE_OVERRIDE
    xb, ldx = as_rows(x)
    F = x.size(1)
    if x.size(0) < csr.n_cols:
        raise RuntimeError(f"x has {x.size(0)} rows but the graph addresses {csr.n_cols}")
    if not store_local:                       # every store goes through ep.peer_out / ep.Y2
        y, ldy = None, 0
    elif out is None:
        y, ldy = alloc_rows(csr.n_rows, F, x.dtype, x.device)
    else:
        y, ldy = out, out.stride(0)
    ws = csr.spmm_workspace(F)
    dev = x.device
    check(lib().rgbmp_spmm(_graph_ref(csr, ldx * xb.element_size(), hot), ptr(val), ptr(xb), ldx, ptr(y), ldy, F, dtype_code(x),
                           C.byref(ep) if ep is not None else None, tune, ptr(ws),
                           0 if ws is None else ws.numel(), dev.index, stream_of(dev)), "spmm")
    return y


def row_scale(x: torch.Tensor, scale: torch.Tensor, divide: bool = False) -> torch.Tensor:
    xb, ldx = as_rows(x)
    y, ldy = alloc_rows(x.size(0), x.size(1), x.dtype, x.device)
    dev = x.device
    check(lib().rgbmp_row_scale(ptr(xb), ldx, ptr(scale), int(divide), ptr(y), ldy, x.size(0), x.size(1),
                                dtype_code(x), dev.index, stream_of(dev)), "row_scale")
    return y


def khop_raw(csr: CSR, x0: torch.Tensor, K: int, **kw):
    """K fused hops.  Returns the final iterate, or (final, [K, N, F] hop outputs) when hops=True."""
    return oom_retry(lambda: _khop_raw(csr, x0, K, **kw))


def _khop_raw(csr: CSR, x0: torch.Tensor, K: int, *, val=None, ep: Optional[Epilogue] = None, keep=(),
              hops: bool = False, tune: int = 0, hot: bool = True):
    tune = tune or TUNE_OVERRIDE
    xb, ldx = as_rows(x0)
    N, F = x0.shape
    dev, dt = x0.device, x0.dtype
    Fp = padded_width(F, dt)
    out, ldo = alloc_rows(N, F, dt, dev)
    ping = pong = None
    if K > 1:
        ping = torch.empty((N, Fp), dtype=dt, device=dev)
        pong = torch.empty((N, Fp), dtype=dt, device=dev)
    hop_buf = torch.empty((K, N, Fp), dtype=dt, device=dev) if hops else None
    ws = csr.spmm_workspace(F)
    check(lib().rgbmp_khop(_graph_ref(csr, Fp * xb.element_size(), hot), ptr(val), ptr(xb), ldx, ptr(ping), ptr(pong), Fp, ptr(out), ldo,
                           ptr(hop_buf), Fp, N * Fp, F, dtype_code(x0), K,
                           C.byref(ep) if ep is not None else None, tune, ptr(ws),
                           0 if ws is None else ws.numel(), dev.index, stream_of(dev)), "khop")
    if hops:
        return out, hop_buf[:, :, :F]
    return out


# ------------------------------------------------------------------------------------------
# single-hop propagate  (MessagePassing.propagate / GCNConv / SAGEConv / GINConv ...)
# ------------------------------------------------------------------------------------------
class _Propagate(torch.autograd.Function):
    """kind: 'sum' (aggr='add', message=x_j), 'mean' (aggr='mean'), 'gcn' (symmetric norm weights).
    Backward = the same kernel on the transpose CSR (linear operator, nothing but the graph saved)."""

    @staticmethod
    def forward(ctx, x, graph: Graph, kind: str):
        ctx.graph, ctx.kind = graph, kind
        csr = graph.fwd
        if kind == "sum":
            return spmm_raw(csr, x)
        if kind == "mean":
            cnt = csr.norm(NORM_COUNT)
            return spmm_raw(csr, x, ep=make_epilogue(row_scale=cnt, row_div=True), keep=(cnt,))
        if kind == "gcn":
            return spmm_raw(csr, x, graph.gcn_val(False))
        raise ValueError(kind)

    @staticmethod
    def backward(ctx, dy):
        g, kind = ctx.graph, ctx.kind
        if kind == "sum":
            return spmm_raw(g.bwd, dy), None, None
        if kind == "mean":
            return spmm_raw(g.bwd, row_scale(dy, g.fwd.norm(NORM_COUNT), divide=True)), None, None
        return spmm_raw(g.bwd, dy, g.gcn_val(True)), None, None


def _work(graph: Graph, x: torch.Tensor) -> float:
    return float(graph.nnz) * float(x.size(-1) if x.dim() > 1 else 1)


def propagate(x: torch.Tensor, graph: Graph, kind: str = "sum") -> torch.Tensor:
    # memo.cached: the second of the caller's two identical eval forwards reuses the first (SURVEY 8f f2)
    return memo.cached(graph, ("propagate", kind), (x,), _work(graph, x), lambda: _Propagate.apply(x, graph, kind))


class _PropagateWeighted(torch.autograd.Function):
    """y[i] = sum_{e: dst=i} w[e] * x[src[e]] with per-edge weights given in EDGE order [nnz]
    (Prop.message, dagnn.py:57-59; generic edge_weight).  dw[e] = <dy[dst], x[src]> (SDDMM)."""

    @staticmethod
    def forward(ctx, x, w, graph: Graph):
        ctx.graph = graph
        val = graph.to_csr_order(w, transpose=False)
        ctx.save_for_backward(x if ctx.needs_input_grad[1] else None, w)
        return spmm_raw(graph.fwd, x, val)

    @staticmethod
    def backward(ctx, dy):
        g = ctx.graph
        x, w = ctx.saved_tensors
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = spmm_raw(g.bwd, dy, g.to_csr_order(w, transpose=True))
        if ctx.needs_input_grad[1]:       # the SDDMM kernel is fp32-only: a bf16 dy / x widens exactly
            dw = g.to_edge_order(sddmm(g.fwd, dy.float(), x.float(), 1, dy.size(1))).view_as(w).to(w.dtype)
        return dx, dw, None


def propagate_weighted(x, w, graph: Graph):
    return memo.cached(graph, ("propagate_weighted",), (x, w), _work(graph, x),
                       lambda: _PropagateWeighted.apply(x, w, graph))


# ------------------------------------------------------------------------------------------
# K-hop families
# ------------------------------------------------------------------------------------------
FOLD_KHOP = True     # K-hop families apply D^-1/2 (A+I) D^-1/2 as row scalings around an unweighted sum (no per-edge
                     # weight stream, 4 B/edge less and adds instead of FMAs); False: per-edge gcn_norm weights as PyG multiplies them
NAMED_KHOP = True    # folded fp32 K-hop forwards (APPNP, SGC, K >= 2) on a locality-grouped graph run on Graph.named_fwd, the
                     # nodes renamed in schedule order: the iterate, teleport and output rows are read and written in order
                     # and each group's feature rows are contiguous (bit-identical results); False: on fwd, ids as given
FUSED_DROPOUT = False  # GATConv / SuperGATConv / FAConv in training mode: True = attention dropout generated inside the
                       # attention kernels (counter-based, keyed by edge id, nothing edge-sized allocated); False = a torch
                       # F.dropout mask per call, so the same torch.manual_seed draws the same masks as it always has
FUSED_SUPERGAT_LOSS = False  # SuperGATConv in training mode: True = its attention loss on the device (seeded edge and
                             # negative sampling, fused pair-logit BCE, nothing edge-sized); False = torch sampling and
                             # [pairs, H, C] gathers, so the same torch.manual_seed draws the same samples as it always has


def _khop_gcn(csr: CSR, graph: Graph, x0b: torch.Tensor, K: int, transpose: bool, fold: bool, **epkw):
    """K hops of z <- epilogue(A_hat z) on the chosen orientation.  fold: the iterate travels pre-scaled
    (u = D^-1/2 z, what the next hop gathers) and the epilogue scales the row sum by D^-1/2 again; the
    in-degree vector serves both orientations (A_hat^T = D^-1/2 A^T D^-1/2 with the same D)."""
    if fold:
        d = graph.dinv()
        return khop_raw(csr, row_scale(x0b, d), K, ep=make_epilogue(row_scale=d, out2_scale=d, **epkw))
    return khop_raw(csr, x0b, K, val=graph.gcn_val(transpose), ep=make_epilogue(**epkw))


def _staged(x: torch.Tensor, d: torch.Tensor, src_map: Optional[torch.Tensor] = None, teleport: bool = True):
    """(z0 padded to an aligned row stride, u0 = D^-1/2 z0) from an UNALIGNED fp32 input in ONE kernel (instead of a zero
    fill, a copy and a row scale): the case of every class count that is not a multiple of four (47, 10, ...).
    src_map: row i is input row src_map[i] (a renamed graph's node order); teleport=False: no z0 (None)."""
    N, F = x.shape
    Fp = padded_width(F, x.dtype)
    z0 = torch.empty((N, Fp), dtype=x.dtype, device=x.device) if teleport else None
    u0 = torch.empty((N, Fp), dtype=x.dtype, device=x.device)
    xc = x if x.stride(1) == 1 else x.contiguous()
    dev = x.device
    check(lib().rgbmp_stage_rows(ptr(xc), xc.stride(0), ptr(src_map), ptr(d), ptr(z0), ptr(u0), Fp, N, F, dev.index,
                                 stream_of(dev)), "stage_rows")
    return (None if z0 is None else z0[:, :F]), u0[:, :F], Fp


def _named_csr(graph: Graph, x: torch.Tensor, K: int, transpose: bool, fold: bool) -> Optional[CSR]:
    """graph.named_fwd when this K-hop call runs on the renamed graph (NAMED_KHOP), else None."""
    if not (NAMED_KHOP and fold and not transpose and K >= 2 and x.dim() == 2 and x.dtype == torch.float32
            and x.size(0) > 0 and x.size(0) == getattr(graph, "N", -1)):
        return None
    return getattr(graph, "named_fwd", None)


def _khop_named(nf: CSR, graph: Graph, x: torch.Tensor, K: int, a: float = 1.0, b: Optional[float] = None):
    """Folded K hops of z <- a * A_hat z (+ b * x) on the renamed graph nf: the staging pass reads x in nf's node order,
    the last hop stores under the original ids.  Same operator, same per-row sums and roundings as on graph.fwd."""
    d = nf.norm(NORM_INV_SQRT)              # dinv in the renamed order
    order = graph.fwd.row_order             # row i of nf is node order[i]
    z0, u0, ld = _staged(x, d, order, teleport=b is not None)
    ep = make_epilogue(row_scale=d, out2_scale=d, a=a, b=0.0 if b is None else b, T=z0, ldt=ld if z0 is not None else 0,
                       row_map=order)
    return khop_raw(nf, u0, K, ep=ep, keep=(z0, d, order))


def _appnp_khop(csr: CSR, graph: Graph, x: torch.Tensor, K: int, alpha: float, transpose: bool, fold: bool):
    _lib.require_cuda(x, "x")
    nf = _named_csr(graph, x, K, transpose, fold)
    if nf is not None:
        return _khop_named(nf, graph, x, K, a=1.0 - alpha, b=alpha)
    if fold and x.dim() == 2 and x.dtype == torch.float32 and x.size(1) % 4 != 0 and x.size(0) > 0:
        d = graph.dinv()
        z0, u0, ld = _staged(x, d)
        ep = make_epilogue(row_scale=d, out2_scale=d, a=1.0 - alpha, b=alpha, T=z0, ldt=ld)
        return khop_raw(csr, u0, K, ep=ep, keep=(z0, d))
    xb, ldx = as_rows(x)
    return _khop_gcn(csr, graph, xb, K, transpose, fold, a=1.0 - alpha, b=alpha, T=xb, ldt=ldx)


class _APPNP(torch.autograd.Function):
    """z = x; K x { z = (1-alpha) * A_hat z + alpha * x }  (A8; appnp_stack.py:22).
    The map is linear, z_K = M x with M = alpha*sum_{k<K} B^k + B^K, B=(1-alpha)A_hat, so the
    backward is the same recursion on the transpose graph -- no hop activations are kept."""

    @staticmethod
    def forward(ctx, x, graph: Graph, K: int, alpha: float, fold: bool):
        ctx.graph, ctx.K, ctx.alpha, ctx.fold = graph, K, alpha, fold
        return _appnp_khop(graph.fwd, graph, x, K, alpha, False, fold)

    @staticmethod
    def backward(ctx, dz):
        g = ctx.graph
        return _appnp_khop(g.bwd, g, dz, ctx.K, ctx.alpha, True, ctx.fold), None, None, None, None


def appnp(x, graph: Graph, K: int, alpha: float, fold: Optional[bool] = None):
    if K == 0:
        return x
    K, alpha, fold = int(K), float(alpha), bool(FOLD_KHOP if fold is None else fold)
    return memo.cached(graph, ("appnp", K, alpha, fold), (x,), K * _work(graph, x),
                       lambda: _APPNP.apply(x, graph, K, alpha, fold))


class _PowerHops(torch.autograd.Function):
    """x <- A_hat^K x (A9 SGConv, sgc.py:9-10)."""

    @staticmethod
    def forward(ctx, x, graph: Graph, K: int, fold: bool):
        ctx.graph, ctx.K, ctx.fold = graph, K, fold
        _lib.require_cuda(x, "x")
        nf = _named_csr(graph, x, K, False, fold)
        if nf is not None:
            return _khop_named(nf, graph, x, K)
        return _khop_gcn(graph.fwd, graph, as_rows(x)[0], K, False, fold)

    @staticmethod
    def backward(ctx, dy):
        g = ctx.graph
        return _khop_gcn(g.bwd, g, as_rows(dy)[0], ctx.K, True, ctx.fold), None, None, None


def gcn_power(x, graph: Graph, K: int, fold: Optional[bool] = None):
    if K == 0:
        return x
    fold = bool(FOLD_KHOP if fold is None else fold)
    return memo.cached(graph, ("gcn_power", int(K), fold), (x,), K * _work(graph, x),
                       lambda: _PowerHops.apply(x, graph, int(K), fold))


class _DagnnHops(torch.autograd.Function):
    """[N, K+1, C] stack (x, A_hat x, ..., A_hat^K x) in one K-hop call that keeps every hop (dagnn.py:43-49).
    Backward: g_K = dS_K; g_k = dS_k + A_hat^T g_{k+1} -- K transposed SpMMs with the add in the epilogue."""

    @staticmethod
    def forward(ctx, x, graph: Graph, K: int):
        ctx.graph, ctx.K = graph, K
        _, hops = khop_raw(graph.fwd, x, K, val=graph.gcn_val(False), hops=True)
        return torch.cat([x.detach().unsqueeze(0), hops], dim=0).permute(1, 0, 2)

    @staticmethod
    def backward(ctx, dS):
        g, K = ctx.graph, ctx.K
        val = g.gcn_val(True)
        acc = dS[:, K, :].contiguous()
        for k in range(K - 1, -1, -1):
            t, ldt = as_rows(dS[:, k, :])
            acc = spmm_raw(g.bwd, acc, val, ep=make_epilogue(a=1.0, b=1.0, T=t, ldt=ldt), keep=(t,))
        return acc, None, None


def dagnn_hops(x: torch.Tensor, graph: Graph, K: int) -> torch.Tensor:
    """[N, K+1, C] stack of x and its K propagated versions (dagnn.py:43-49), differentiable."""
    return _DagnnHops.apply(x, graph, int(K))


def label_propagation(graph: Graph, out0: torch.Tensor, num_layers: int, alpha: float, *,
                      clamp=(0.0, 1.0), reset_mask=None, reset_val=None, fold: Optional[bool] = None) -> torch.Tensor:
    """A15 LP core: res=(1-a)*out0; L x { out = a * A_hat out + res; post_step }.
    post_step = clamp(lo,hi) (default / autoscale) or `out[mask] = reset_val[mask]` (fixed scale).
    `graph` must be built with LOOP_NONE (gcn_norm(add_self_loops=False))."""
    if num_layers == 0:
        return out0
    xb, ldx = as_rows(out0)
    kw = {}
    if reset_mask is not None:
        kw = reset_rows(reset_mask, reset_val, out0.size(1))
        clamp = None
    return _khop_gcn(graph.fwd, graph, xb, num_layers, False, bool(FOLD_KHOP if fold is None else fold),
                     a=alpha, b=1.0 - alpha, T=xb, ldt=ldx, clamp=clamp, **kw)


# ------------------------------------------------------------------------------------------
# PTA graph ops (itexperiments.py:671-719, pta.py:79-84).  The PTA adjacency aggregates at
# row = edge_index[0], i.e. it is the gcn propagation of the REVERSED graph, with A+I doubling
# an existing self loop (SURVEY.md Appendix B7) -> build the graph with LOOP_ADD on the flipped
# edge_index: duplicates and pre-existing loops then count exactly like the scipy COO sum.
# ------------------------------------------------------------------------------------------
def pta_graph(edge_index: torch.Tensor, num_nodes: int) -> Graph:
    from .graph import LOOP_ADD, get_graph
    return get_graph(edge_index, num_nodes, LOOP_ADD, reverse=True)


def pta_inference(h: torch.Tensor, graph: Graph, K: int, alpha: float) -> torch.Tensor:
    y0 = torch.softmax(h, dim=-1)
    xb, ldx = as_rows(y0)
    return _khop_gcn(graph.fwd, graph, xb, K, False, FOLD_KHOP, a=1.0 - alpha, b=alpha, T=xb, ldt=ldx)


def pta_label_propagation(graph: Graph, labels: torch.Tensor, idx: torch.Tensor, K: int, alpha: float):
    N = labels.size(0)
    Cn = int(labels.max().item()) + 1
    y0 = torch.zeros((N, Cn), dtype=torch.float32, device=labels.device)
    y0[idx, labels[idx]] = 1.0
    mask = torch.zeros(N, dtype=torch.uint8, device=labels.device)
    mask[idx] = 1
    xb, ldx = as_rows(y0)
    # y <- A y ; y[idx] <- onehot[idx] (= y0[idx]) ; y <- (1-a) y + a y0
    return _khop_gcn(graph.fwd, graph, xb, K, False, FOLD_KHOP, a=1.0 - alpha, b=alpha, T=xb, ldt=ldx, reset_mask=mask,
                     reset_val=xb, ld_reset=ldx, reset_when=RESET_BEFORE_TELEPORT)


# ------------------------------------------------------------------------------------------
# attention / edge-score kernels
# ------------------------------------------------------------------------------------------
def sddmm(csr: CSR, A: torch.Tensor, B: torch.Tensor, H: int, Cc: int) -> torch.Tensor:
    """out[k,h] = <A[row_i,h,:], B[col[k],h,:]> in CSR order."""
    _lib.require_f32(A, "sddmm A")
    _lib.require_f32(B, "sddmm B")
    Ab, lda = as_rows(A)
    Bb, ldb = as_rows(B)
    out = torch.empty((csr.nnz, H), dtype=torch.float32, device=A.device)
    dev = A.device
    check(lib().rgbmp_sddmm(csr.ref, ptr(Ab), lda, ptr(Bb), ldb, H, Cc, ptr(out), dev.index, stream_of(dev)), "sddmm")
    return out


def _edge_call(fn_name, csr: CSR, *args):
    dev = csr.device
    check(getattr(lib(), fn_name)(csr.ref, *args, dev.index, stream_of(dev)), fn_name)


def spmm_heads_raw(csr: CSR, w: torch.Tensor, X: torch.Tensor, H: int, Cc: int) -> torch.Tensor:
    _lib.require_f32(w, "spmm_heads w")
    _lib.require_f32(X, "spmm_heads X")
    Xb, ldx = as_rows(X)
    out, ldo = alloc_rows(csr.n_rows, H * Cc, torch.float32, X.device)
    _edge_call("rgbmp_spmm_heads", csr, ptr(w.contiguous()), ptr(Xb), ldx, H, Cc, ptr(out), ldo)
    return out


def seg_sum_raw(csr: CSR, vals: torch.Tensor, H: int) -> torch.Tensor:
    _lib.require_f32(vals, "seg_sum")
    out = torch.empty((csr.n_rows, H), dtype=torch.float32, device=vals.device)
    _edge_call("rgbmp_seg_sum", csr, ptr(vals.contiguous()), H, ptr(out))
    return out


class _SDDMM(torch.autograd.Function):
    """out[k,h] = <A[i,h,:], B[j,h,:]> for every edge j->i, forward-CSR order (SuperGAT MX logits)."""

    @staticmethod
    def forward(ctx, A, B, graph: Graph, H: int, Cc: int):
        ctx.graph, ctx.H, ctx.Cc = graph, H, Cc
        ctx.save_for_backward(A, B)
        return sddmm(graph.fwd, A, B, H, Cc)

    @staticmethod
    def backward(ctx, g):
        A, B = ctx.saved_tensors
        gr, H, Cc = ctx.graph, ctx.H, ctx.Cc
        g = g.contiguous()
        dA = spmm_heads_raw(gr.fwd, g, B, H, Cc) if ctx.needs_input_grad[0] else None
        dB = spmm_heads_raw(gr.bwd, gr.fwd_to_bwd(g), A, H, Cc) if ctx.needs_input_grad[1] else None
        return dA, dB, None, None, None


class _UAddV(torch.autograd.Function):
    """out[k,h] = u[j,h] + v[i,h] for every edge j->i (forward-CSR order)."""

    @staticmethod
    def forward(ctx, u, v, graph: Graph):
        _lib.require_f32(u, "u_add_v u")
        _lib.require_f32(v, "u_add_v v")
        ctx.graph = graph
        H = u.size(1)
        out = torch.empty((graph.nnz, H), dtype=torch.float32, device=u.device)
        _edge_call("rgbmp_u_add_v", graph.fwd, ptr(u.contiguous()), ptr(v.contiguous()), H, ptr(out))
        return out

    @staticmethod
    def backward(ctx, g):
        gr = ctx.graph
        g = g.contiguous()
        H = g.size(1)
        du = seg_sum_raw(gr.bwd, gr.fwd_to_bwd(g), H) if ctx.needs_input_grad[0] else None
        dv = seg_sum_raw(gr.fwd, g, H) if ctx.needs_input_grad[1] else None
        return du, dv, None


class _SegSoftmax(torch.autograd.Function):
    """Edge softmax over the in-edges of each target (A11), forward-CSR order."""

    @staticmethod
    def forward(ctx, e, graph: Graph):
        _lib.require_f32(e, "edge_softmax")
        ctx.graph = graph
        e = e.contiguous()
        out = torch.empty_like(e)
        _edge_call("rgbmp_seg_softmax", graph.fwd, ptr(e), e.size(1), ptr(out))
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, g):
        (alpha,) = ctx.saved_tensors
        g = g.contiguous()
        out = torch.empty_like(g)
        _edge_call("rgbmp_seg_softmax_backward", ctx.graph.fwd, ptr(alpha), ptr(g), g.size(1), ptr(out))
        return out, None


class _SpmmHeads(torch.autograd.Function):
    """out[i,h,:] = sum_{j->i} w[k,h] * X[j,h,:], w in forward-CSR order."""

    @staticmethod
    def forward(ctx, w, X, graph: Graph, H: int, Cc: int):
        ctx.graph, ctx.H, ctx.Cc = graph, H, Cc
        ctx.save_for_backward(w, X)
        return spmm_heads_raw(graph.fwd, w, X, H, Cc)

    @staticmethod
    def backward(ctx, dout):
        w, X = ctx.saved_tensors
        gr, H, Cc = ctx.graph, ctx.H, ctx.Cc
        dw = sddmm(gr.fwd, dout, X, H, Cc) if ctx.needs_input_grad[0] else None
        dX = spmm_heads_raw(gr.bwd, gr.fwd_to_bwd(w), dout, H, Cc) if ctx.needs_input_grad[1] else None
        return dw, dX, None, None, None


def edge_sddmm(A, B, graph, H, Cc):
    return _SDDMM.apply(A, B, graph, H, Cc)


def edge_u_add_v(u, v, graph):
    return _UAddV.apply(u, v, graph)


def edge_softmax(e, graph):
    return _SegSoftmax.apply(e, graph)


def spmm_heads(w, X, graph, H, Cc):
    return _SpmmHeads.apply(w, X, graph, H, Cc)


ATT_GAT, ATT_MX, ATT_FA, ATT_SD = 0, 1, 2, 3


def _head_pad(H: int, Cc: int) -> int:
    """Channels per head the fused kernels run with: C itself for a single head, else the next power of two >= 8
    (a lane's 8 channels must stay inside one head; zero channels change neither dot products nor sums)."""
    if H == 1:
        return Cc
    c = 8
    while c < Cc:
        c <<= 1
    return c


def att_fusable(score: int, H: int, Cc: int) -> bool:
    return bool(lib().rgbmp_att_supported(score, H, _head_pad(H, Cc)))


def gat_fusable(H: int, Cc: int) -> bool:
    return att_fusable(ATT_GAT, H, Cc)


def _rows_zero_padded(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """as_rows, but the padding columns up to roundup(F,4) are guaranteed ZERO (the H == 1 kernels take dot
    products over whole float4 vectors)."""
    F = x.size(1)
    if F % 4 == 0:
        return as_rows(x)
    Fp = padded_width(F, x.dtype)
    buf = torch.zeros((x.size(0), Fp), dtype=x.dtype, device=x.device)
    buf[:, :F].copy_(x)
    return buf[:, :F], Fp


class _Att(torch.autograd.Function):
    """Fused edge-score attention + aggregate (csrc/att.cu): GATConv (A10/A11; gat.py:18-21), SuperGATConv-MX
    (A12; supergat.py:15-21), SuperGATConv-SD (A12; no score scalars: a_nbr = a_own = None, the logit <x_i, x_j>
    scaled by logit_scale) and FAConv (A13; fagcn.py:15,31).  Nothing edge-sized is allocated: the forward saves
    per-node statistics (max, sum and -- in training mode -- the second aggregate that yields the gradient of the
    target-side score term), the backward recomputes the edge weights.  Deterministic (no atomics).
    Attention dropout: either an explicit mask in forward-CSR order (drop_csr) or a device seed tensor (seed, rate p)
    from which forward and backward regenerate the same multipliers inside the kernels -- still nothing edge-sized."""

    @staticmethod
    def forward(ctx, x, a_nbr, a_own, graph: Graph, score: int, H: int, Cc: int, slope: float, drop_csr, seed, p,
                logit_scale: float):
        _lib.require_cuda(x, "x")
        for t, nm in ((x, "x"), (a_nbr, "a_nbr"), (a_own, "a_own")):
            if t is not None:
                _lib.require_f32(t, f"fused attention {nm}")
        xb, ldx = _rows_zero_padded(x)
        a_n = a_o = None
        if score != ATT_SD:
            a_n, a_o = a_nbr.contiguous().view(-1, H), a_own.contiguous().view(-1, H)
        N, dev = graph.N, x.device
        train = any(ctx.needs_input_grad[:3])
        out, ldo = alloc_rows(N, H * Cc, torch.float32, dev)
        rmax = rsum = rowq = out2 = dinv = None
        ldo2 = 0
        if score != ATT_FA:
            rmax = torch.empty((N, H), dtype=torch.float32, device=dev)
            rsum = torch.empty((N, H), dtype=torch.float32, device=dev)
        else:
            dinv = graph.dinv()
        if train and score in (ATT_GAT, ATT_FA):
            out2, ldo2 = alloc_rows(N, H * Cc, torch.float32, dev)
            if score == ATT_GAT:
                rowq = torch.empty((N, H), dtype=torch.float32, device=dev)
        L = lib()
        wsb = L.rgbmp_att_forward_workspace_bytes(graph.fwd.ref, H, Cc)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        d = None if seed is None else C.byref(_dropout_struct(p, seed, graph))
        check(L.rgbmp_att_forward(graph.fwd.ref, score, ptr(xb), ldx, ptr(a_n), ptr(a_o), ptr(dinv), H, Cc, slope,
                                  logit_scale, ptr(drop_csr), d, ptr(out), ldo, ptr(rmax), ptr(rsum), ptr(out2), ldo2,
                                  ptr(rowq), ptr(ws), wsb, dev.index, stream_of(dev)), "att_forward")
        ctx.graph, ctx.score, ctx.H, ctx.Cc, ctx.slope, ctx.p, ctx.logit_scale = graph, score, H, Cc, slope, p, logit_scale
        ctx.save_for_backward(xb, a_n, a_o, rmax, rsum, rowq, out, out2, drop_csr, seed)
        return out

    @staticmethod
    def backward(ctx, dout):
        xb, a_n, a_o, rmax, rsum, rowq, out, out2, drop, seed = ctx.saved_tensors
        g, score, H, Cc = ctx.graph, ctx.score, ctx.H, ctx.Cc
        dev, N = dout.device, g.N
        db, ldd = _rows_zero_padded(dout)
        dx, lddx = alloc_rows(N, H * Cc, torch.float32, dev)
        dxf, lddxf = (alloc_rows(N, H * Cc, torch.float32, dev) if score in (ATT_MX, ATT_SD) else (None, 0))
        tpos = g.tpos() if drop is not None else None
        dinv = g.dinv() if score == ATT_FA else None
        L = lib()
        wsb = L.rgbmp_att_backward_workspace_bytes(g.fwd.ref, g.bwd.ref, H, Cc)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        da_n = da_o = None                                   # SD has no score scalars
        if score != ATT_SD:
            da_n = torch.empty((N, H), dtype=torch.float32, device=dev)
            da_o = torch.empty((N, H), dtype=torch.float32, device=dev)
        ld2 = 0 if out2 is None else out2.stride(0)
        d = None if seed is None else C.byref(_dropout_struct(ctx.p, seed, g, backward=True))
        check(L.rgbmp_att_backward(g.fwd.ref, g.bwd.ref, score, ptr(xb), xb.stride(0), ptr(a_n), ptr(a_o), ptr(dinv), H, Cc,
                                   ctx.slope, ctx.logit_scale, ptr(drop), ptr(tpos), d, ptr(rmax), ptr(rsum), ptr(rowq),
                                   ptr(out), out.stride(0), ptr(out2), ld2, ptr(db), ldd, ptr(dx), lddx, ptr(dxf), lddxf,
                                   ptr(da_n), ptr(da_o), ptr(ws), wsb, dev.index, stream_of(dev)), "att_backward")
        return dx, da_n, da_o, None, None, None, None, None, None, None, None, None


def _att(score: int, name: str, x, a_nbr, a_own, graph: Graph, H: int, Cc: int, slope: float, drop_edge,
         dropout_p: float = 0.0, seed: Optional[torch.Tensor] = None):
    """Pads heads to the kernel's channel count (torch ops on node-sized tensors, autograd-transparent), memoises
    the no-grad call, applies the fused op.  seed: fused dropout at rate dropout_p (see dropout_mask).  SD scales
    its logit by 1/sqrt(Cc) of the unpadded head width."""
    Cp = _head_pad(H, Cc)
    N = x.size(0)
    xk = x if Cp == Cc else torch.nn.functional.pad(x.view(N, H, Cc), (0, Cp - Cc)).reshape(N, H * Cp)
    drop_csr = None if drop_edge is None else graph.to_csr_order(drop_edge)
    ls = 1.0 / math.sqrt(Cc) if score == ATT_SD else 0.0
    if drop_csr is None and seed is None:
        ins = tuple(t for t in (xk, a_nbr, a_own) if t is not None)
        out = memo.cached(graph, (name, H, Cc, float(slope)), ins, _work(graph, xk),
                          lambda: _Att.apply(xk, a_nbr, a_own, graph, score, H, Cp, float(slope), None, None, 0.0, ls))
    else:
        out = _Att.apply(xk, a_nbr, a_own, graph, score, H, Cp, float(slope), drop_csr, seed, float(dropout_p), ls)
    return out if Cp == Cc else out.view(N, H, Cp)[:, :, :Cc].reshape(N, H * Cc)


# ------------------------------------------------------------------------------------------
# attention dropout generated from a seed (csrc/philox.cuh): multiplier of edge e, head h =
#   Philox4x32-10(counter (e, h, 0, 0), key (seed lo, seed hi)).word0 < floor(p 2^32) ? 0 : float32(1/(1-p))
# ------------------------------------------------------------------------------------------
def dropout_seed(device, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """One int64 drawn on the device from its CUDA generator (or `generator`): no host synchronisation,
    governed by torch.manual_seed / fork_rng, safe under graph capture."""
    return torch.empty(1, dtype=torch.int64, device=device).random_(generator=generator)


def _dropout_struct(p: float, seed: torch.Tensor, graph: Optional[Graph] = None, backward: bool = False):
    """rgbmp_dropout_t for rate p (thresh = floor(p 2^32) exactly; p == 1 -> every multiplier 0)."""
    if p >= 1.0:
        thresh, scale = 0xFFFFFFFF, 0.0
    else:
        thresh, scale = int(math.floor(p * 4294967296.0)), 1.0 / (1.0 - p)    # c_float rounds scale to float32
    eid = eid_t = None
    if graph is not None:
        if graph.fwd.eid is None:
            raise RuntimeError("fused attention dropout needs the edge ids of the graph")
        eid = graph.fwd.eid
        eid_t = graph.bwd.eid if backward else None
    return _lib.DropoutStruct(ptr(seed), ptr(eid), ptr(eid_t), thresh, scale)


def dropout_mask(graph: Graph, H: int, p: float, seed: torch.Tensor) -> torch.Tensor:
    """[nnz, H] float32 multipliers in EDGE order: the mask the fused kernels apply for `seed` (unfused paths, tests)."""
    out = torch.empty((graph.nnz, H), dtype=torch.float32, device=graph.device)
    d = _dropout_struct(float(p), seed)
    check(lib().rgbmp_dropout_mask(C.byref(d), graph.nnz, H, ptr(out), graph.device.index, stream_of(graph.device)),
          "dropout_mask")
    return out


def _draw_dropout(graph: Graph, drop_edge, dropout_p: float, generator) -> Optional[torch.Tensor]:
    """Validate the dropout arguments; the seed tensor when dropout_p > 0, else None."""
    p = float(dropout_p)
    if not 0.0 <= p <= 1.0:
        raise ValueError(f"dropout_p must lie in [0, 1] (got {dropout_p})")
    if p > 0.0 and drop_edge is not None:
        raise ValueError("drop_edge and dropout_p are mutually exclusive")
    return dropout_seed(graph.device, generator) if p > 0.0 else None


def gat(xp, a_src, a_dst, graph: Graph, H: int, Cc: int, slope: float = 0.2, drop_edge: Optional[torch.Tensor] = None,
        dropout_p: float = 0.0, generator: Optional[torch.Generator] = None):
    """xp [N,H*C], a_src/a_dst [N,H] -> [N,H*C].  drop_edge: optional [nnz,H] keep-mask/(1-p) in EDGE order.
    dropout_p: attention dropout drawn from a seed (`generator` or the device's default CUDA generator) and
    generated inside the kernels; exclusive with drop_edge."""
    seed = _draw_dropout(graph, drop_edge, dropout_p, generator)
    if att_fusable(ATT_GAT, H, Cc):
        return _att(ATT_GAT, "gat", xp, a_src, a_dst, graph, H, Cc, slope, drop_edge, dropout_p, seed)
    if seed is not None:
        drop_edge = dropout_mask(graph, H, dropout_p, seed)
    e = torch.nn.functional.leaky_relu(edge_u_add_v(a_src, a_dst, graph), slope)
    alpha = edge_softmax(e, graph)
    if drop_edge is not None:
        alpha = alpha * graph.to_csr_order(drop_edge)
    return spmm_heads(alpha, xp, graph, H, Cc)


def supergat_mx(xp, a_l, a_r, graph: Graph, H: int, Cc: int, slope: float = 0.2,
                drop_edge: Optional[torch.Tensor] = None, dropout_p: float = 0.0,
                generator: Optional[torch.Generator] = None):
    """SuperGATConv MX attention + aggregate (A12): alpha = softmax(leaky_relu((a_l[j] + a_r[i]) * sigmoid(<x_i, x_j>))).
    drop_edge / dropout_p / generator as in gat."""
    seed = _draw_dropout(graph, drop_edge, dropout_p, generator)
    if att_fusable(ATT_MX, H, Cc):
        return _att(ATT_MX, "supergat_mx", xp, a_l, a_r, graph, H, Cc, slope, drop_edge, dropout_p, seed)
    if seed is not None:
        drop_edge = dropout_mask(graph, H, dropout_p, seed)
    logits = edge_sddmm(xp, xp, graph, H, Cc)
    alpha = torch.nn.functional.leaky_relu(edge_u_add_v(a_l, a_r, graph) * logits.sigmoid(), slope)
    alpha = edge_softmax(alpha, graph)
    if drop_edge is not None:
        alpha = alpha * graph.to_csr_order(drop_edge)
    return spmm_heads(alpha, xp, graph, H, Cc)


def supergat_sd(xp, graph: Graph, H: int, Cc: int, slope: float = 0.2, drop_edge: Optional[torch.Tensor] = None,
                dropout_p: float = 0.0, generator: Optional[torch.Generator] = None):
    """SuperGATConv SD attention + aggregate (A12): alpha = softmax(leaky_relu(<x_i, x_j> / sqrt(Cc))) per head.
    xp [N,H*C] float32 -> [N,H*C].  drop_edge / dropout_p / generator as in gat."""
    _lib.require_f32(xp, "supergat_sd xp")
    seed = _draw_dropout(graph, drop_edge, dropout_p, generator)
    if att_fusable(ATT_SD, H, Cc):
        return _att(ATT_SD, "supergat_sd", xp, None, None, graph, H, Cc, slope, drop_edge, dropout_p, seed)
    if seed is not None:
        drop_edge = dropout_mask(graph, H, dropout_p, seed)
    alpha = torch.nn.functional.leaky_relu(edge_sddmm(xp, xp, graph, H, Cc) / math.sqrt(Cc), slope)
    alpha = edge_softmax(alpha, graph)
    if drop_edge is not None:
        alpha = alpha * graph.to_csr_order(drop_edge)
    return spmm_heads(alpha, xp, graph, H, Cc)


def faconv(x, a_l, a_r, graph: Graph, drop_edge: Optional[torch.Tensor] = None, dropout_p: float = 0.0,
           generator: Optional[torch.Generator] = None):
    """FAConv aggregate (A13): out[i] = sum_j tanh(a_l[j] + a_r[i]) * gcn_norm_ij * mask_ij * x[j]; a_l, a_r [N,1].
    drop_edge / dropout_p / generator as in gat (head 0)."""
    Cc = x.size(1)
    seed = _draw_dropout(graph, drop_edge, dropout_p, generator)
    if att_fusable(ATT_FA, 1, Cc):
        return _att(ATT_FA, "faconv", x, a_l, a_r, graph, 1, Cc, 0.0, None if drop_edge is None else drop_edge.view(-1, 1),
                    dropout_p, seed)
    if seed is not None:
        drop_edge = dropout_mask(graph, 1, dropout_p, seed)
    c = edge_u_add_v(a_l.view(-1, 1), a_r.view(-1, 1), graph).tanh()
    if drop_edge is not None:
        c = c * graph.to_csr_order(drop_edge).view(-1, 1)
    return spmm_heads(c * graph.gcn_val(False).view(-1, 1), x, graph, 1, Cc)


# ------------------------------------------------------------------------------------------
# SuperGAT's self-supervised attention loss (supergat.py:26,29) on the device (csrc/supergat_loss.cu):
#   positive edge e kept iff Philox(counter (e, 0, 1, 0)).word0 >= floor((1 - edge_sample_ratio) 2^32)
#   negative candidate k of round r: Philox(counter (k, r, 2, 0)) -> (umulhi64(w1:w0, N), umulhi64(w3:w2, N)),
#   rejected when it is a pair of U (Graph.undirected_csr), survivors compacted stably and cut to num_neg
#   loss = BCE-with-logits(att_x.mean(-1), y) = (sum_pos softplus(-s) + sum_neg softplus(s)) / P, s = scale <x'_i, x'_j>
# ------------------------------------------------------------------------------------------
class SupergatSamples(NamedTuple):
    seed: torch.Tensor                     # int64 [1] on the device
    keep_thresh: int                       # positive edge e dropped iff its draw < keep_thresh (0: all kept)
    keep_mask: Optional[torch.Tensor]      # bool [nnz] in edge order, when asked for
    neg_edge_index: torch.Tensor           # int64 [2, n]: (src, dst) of the negatives


def supergat_keep_thresh(edge_sample_ratio: float) -> int:
    """floor(p 2^32) for the dropout_adj rate p = 1 - edge_sample_ratio (2^32 at ratio 0: every edge dropped)."""
    p = 1.0 - float(edge_sample_ratio)
    if not 0.0 <= p <= 1.0:
        raise ValueError(f"edge_sample_ratio must lie in [0, 1] (got {edge_sample_ratio})")
    return int(math.floor(p * 4294967296.0))


def supergat_neg_counts(N: int, E_u: int, num_neg_samples: int) -> Tuple[int, int]:
    """(num_neg, sample_size) with negative_sampling's own formulas; E_u = the size of the edge set it is given."""
    size = N * N
    num_neg = min(int(num_neg_samples), size - E_u)
    if num_neg <= 0:
        return num_neg, 0
    alpha = abs(1 / (1 - 1.1 * (E_u / size)))
    return num_neg, int(alpha * num_neg)


def _sgat_struct(seed: torch.Tensor, keep_thresh: int, graph: Optional[Graph] = None, backward: bool = False):
    eid = eid_t = None
    if graph is not None and keep_thresh != 0:
        eid = graph.fwd.eid
        eid_t = graph.bwd.eid if backward else None
    return _lib.SgatSampleStruct(ptr(seed), ptr(eid), ptr(eid_t), keep_thresh)


def _sgat_negatives(graph: Graph, seed: torch.Tensor, num_neg_samples: int, is_undirected: bool):
    """(src, dst) int32 of the device negative sampler; sizing the result is the call's one host synchronisation."""
    dev = graph.device
    rowptr, col = graph.undirected_csr(symmetrize=not is_undirected)
    E_u = graph.nnz if is_undirected else col.numel()        # the torch path counts duplicates when is_undirected
    num_neg, S = supergat_neg_counts(graph.N, E_u, num_neg_samples)
    if num_neg <= 0:
        empty = torch.empty(0, dtype=torch.int32, device=dev)
        return empty, empty
    if S >= 1 << 31:
        raise RuntimeError(f"negative sampling: sample_size {S} >= 2^31 candidates per round")
    L = lib()
    src = torch.empty(num_neg, dtype=torch.int32, device=dev)
    dst = torch.empty(num_neg, dtype=torch.int32, device=dev)
    count = torch.empty(1, dtype=torch.int64, device=dev)
    wsb = L.rgbmp_sgat_negative_sampling_workspace_bytes(S)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    s = _sgat_struct(seed, 0)
    check(L.rgbmp_sgat_negative_sampling(ptr(rowptr), ptr(col), graph.N, C.byref(s), num_neg, S, ptr(src), ptr(dst),
                                         ptr(count), ptr(ws), wsb, dev.index, stream_of(dev)), "sgat_negative_sampling")
    n = int(count.item())
    return src[:n], dst[:n]


def supergat_samples(graph: Graph, edge_sample_ratio: float = 1.0, neg_sample_ratio: float = 0.5,
                     is_undirected: bool = False, seed: Optional[torch.Tensor] = None, mask: bool = False,
                     generator: Optional[torch.Generator] = None) -> SupergatSamples:
    """The samples supergat_att_loss draws for `seed` (default: one drawn like dropout_seed): the positive keep rule
    (and, with mask=True, its bool [nnz] mask in edge order) and the negatives as int64 [2, n]."""
    seed = dropout_seed(graph.device, generator) if seed is None else seed
    thresh = supergat_keep_thresh(edge_sample_ratio)
    keep = None
    if mask:
        out = torch.empty(graph.nnz, dtype=torch.uint8, device=graph.device)
        s = _sgat_struct(seed, thresh)
        check(lib().rgbmp_sgat_keep_mask(C.byref(s), graph.nnz, ptr(out), graph.device.index, stream_of(graph.device)),
              "sgat_keep_mask")
        keep = out.bool()
    num = int(neg_sample_ratio * edge_sample_ratio * graph.nnz)
    src, dst = _sgat_negatives(graph, seed, num, is_undirected)
    return SupergatSamples(seed, thresh, keep, torch.stack([src, dst]).to(torch.int64))


def _pair_csrs(graph: Graph, src: torch.Tensor, dst: torch.Tensor):
    """The negatives as two CSRs over the N nodes: keyed by dst (columns src) and its transpose."""
    from ._lib import GraphStruct
    out = []
    for key, other in ((dst, src), (src, dst)):
        csr = CSR(key, other, graph.N, graph.N, finish=False)
        st = GraphStruct(graph.N, graph.N, csr.nnz, ptr(csr.rowptr), ptr(csr.col), 0, 0, 0, 0, None, None, None, None,
                         None, 0)
        out.append((csr, st))
    return out


class _SupergatLoss(torch.autograd.Function):
    """Pair-logit BCE over the kept positives and the negatives; saves only node-sized rows, the seed, the pair count
    and the negatives' CSRs.  The backward recomputes every logit."""

    @staticmethod
    def forward(ctx, xp, graph: Graph, scale: float, seed, keep_thresh: int, neg):
        xb, ldx = _rows_zero_padded(xp)
        dev, F = xp.device, xp.size(1)
        L = lib()
        loss = torch.empty((), dtype=torch.float32, device=dev)
        npairs = torch.empty(1, dtype=torch.int64, device=dev)
        wsb = L.rgbmp_sgat_loss_workspace_bytes(graph.N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        s = _sgat_struct(seed, keep_thresh, graph)
        check(L.rgbmp_sgat_loss_forward(graph.fwd.ref, C.byref(neg[0][1]), C.byref(s), ptr(xb), ldx, F, scale, ptr(loss),
                                        ptr(npairs), ptr(ws), wsb, dev.index, stream_of(dev)), "sgat_loss_forward")
        ctx.graph, ctx.scale, ctx.keep_thresh, ctx.neg = graph, scale, keep_thresh, neg
        ctx.save_for_backward(xb, seed, npairs)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        xb, seed, npairs = ctx.saved_tensors
        g, neg = ctx.graph, ctx.neg
        dev, N, F = xb.device, g.N, xb.size(1)
        dl = dloss.detach().to(torch.float32).reshape(1).contiguous()
        dx, lddx = alloc_rows(N, F, torch.float32, dev)
        s = _sgat_struct(seed, ctx.keep_thresh, g, backward=True)
        check(lib().rgbmp_sgat_loss_backward(g.fwd.ref, g.bwd.ref, C.byref(neg[0][1]), C.byref(neg[1][1]), C.byref(s),
                                             ptr(xb), xb.stride(0), F, ctx.scale, ptr(npairs), ptr(dl), ptr(dx), lddx,
                                             dev.index, stream_of(dev)), "sgat_loss_backward")
        return dx, None, None, None, None, None


def supergat_att_loss(xp: torch.Tensor, graph: Graph, H: int, Cc: int, scale: float, edge_sample_ratio: float = 1.0,
                      neg_sample_ratio: float = 0.5, is_undirected: bool = False,
                      neg_edge_index: Optional[torch.Tensor] = None,
                      generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """SuperGATConv's get_attention_loss() as one fused op: BCE-with-logits of s = scale * <x'_i, x'_j> (MX: 1/H,
    SD: 1/(H sqrt(C)) -- att_x.mean(-1) of the per-head dots) over the kept positive edges of `graph` (y = 1) and the
    negatives (y = 0).  The negatives are `neg_edge_index` (int64 [2, n], ids in [0, N)) or drawn on the device; the
    seed of the positive sampling and of the sampler is drawn like dropout_seed (`generator` or the device's CUDA
    generator).  One host synchronisation: the negative count (or, for a given neg_edge_index, its range check)."""
    _lib.require_cuda(xp, "xp")
    _lib.require_f32(xp, "supergat_att_loss xp")
    if xp.dim() != 2 or xp.size(1) != H * Cc or xp.size(0) != graph.N:
        raise RuntimeError(f"supergat_att_loss: xp must be [N, H*C] = [{graph.N}, {H * Cc}] (got {tuple(xp.shape)})")
    if graph.fwd.eid is None:
        raise RuntimeError("supergat_att_loss needs the edge ids of the graph")
    seed = dropout_seed(graph.device, generator)
    thresh = supergat_keep_thresh(edge_sample_ratio)
    if neg_edge_index is None:
        num = int(neg_sample_ratio * edge_sample_ratio * graph.nnz)
        src, dst = _sgat_negatives(graph, seed, num, is_undirected)
    else:
        _lib.require_cuda(neg_edge_index, "neg_edge_index")
        if neg_edge_index.dim() != 2 or neg_edge_index.size(0) != 2:
            raise RuntimeError("neg_edge_index must have shape [2, n]")
        if neg_edge_index.numel() and bool(((neg_edge_index < 0) | (neg_edge_index >= graph.N)).any()):
            raise RuntimeError(f"neg_edge_index contains node ids outside [0, {graph.N})")
        src, dst = (neg_edge_index[i].to(torch.int32).contiguous() for i in (0, 1))
    return _SupergatLoss.apply(xp, graph, float(scale), seed, thresh, _pair_csrs(graph, src, dst))


class _EidView:
    """The forward CSR re-read with col = eid: row i then lists the EDGE ids of its in-edges, so an
    SpMM over a per-edge message matrix [nnz, F] is the segmented reduction of scatter(msg, dst)."""

    def __init__(self, csr: CSR):
        from ._lib import GraphStruct
        self.n_rows, self.n_cols, self.nnz, self.device = csr.n_rows, csr.nnz, csr.nnz, csr.device
        self._csr = csr
        self.struct = GraphStruct(csr.n_rows, csr.nnz, csr.nnz, ptr(csr.rowptr), ptr(csr.eid), csr.chunk,
                                  csr.long_chunk, csr.n_long, csr.n_items, ptr(csr.long_rows),
                                  ptr(csr.long_item_ptr), ptr(csr.item_long), ptr(csr.item_start),
                                  ptr(csr.row_order))
        self.ref = C.byref(self.struct)

    def spmm_workspace(self, F):
        return self._csr.spmm_workspace(F)

    def norm(self, mode):
        return self._csr.norm(mode)


class _SegmentReduce(torch.autograd.Function):
    """out[i] = sum (or mean) of msg[e] over edges e with dst[e] == i  -- the aggregate step of a
    MessagePassing layer whose user-defined `message` produced msg in edge order (A6)."""

    @staticmethod
    def forward(ctx, msg, graph: Graph, mean: bool):
        view = graph._vals.get("eid_view")
        if view is None:
            view = _EidView(graph.fwd)
            graph._vals["eid_view"] = view
        ctx.graph, ctx.mean = graph, mean
        if mean:
            cnt = graph.fwd.norm(NORM_COUNT)
            return spmm_raw(view, msg, ep=make_epilogue(row_scale=cnt, row_div=True), keep=(cnt,))
        return spmm_raw(view, msg)

    @staticmethod
    def backward(ctx, dy):
        g = ctx.graph
        if ctx.mean:
            dy = row_scale(dy, g.fwd.norm(NORM_COUNT), divide=True)
        return dy.index_select(0, g.e_dst.long()), None, None


def segment_reduce(msg: torch.Tensor, graph: Graph, mean: bool = False) -> torch.Tensor:
    return _SegmentReduce.apply(msg, graph, bool(mean))


class HostAppnpPlan:
    """Device scratch for the host-buffer entry point, allocated once and reused across calls."""

    def __init__(self, graph: Graph, F: int):
        N, dev = graph.N, graph.device
        self.graph, self.F, self.ld = graph, F, padded_width(F)
        self.bufs = [torch.empty((N, self.ld), dtype=torch.float32, device=dev) for _ in range(4)]
        nf = graph.named_fwd if NAMED_KHOP else None      # the renamed graph, as in _appnp_khop
        self.csr = graph.fwd if nf is None else nf
        self.row_map = None if nf is None else graph.fwd.row_order
        self.ws = self.csr.spmm_workspace(F)
        self.dinv = self.csr.norm(NORM_INV_SQRT)


def appnp_host(graph: Graph, z0_host: torch.Tensor, out_host: torch.Tensor, K: int, alpha: float,
               plan: Optional[HostAppnpPlan] = None) -> torch.Tensor:
    """End-to-end APPNP propagation with HOST buffers (pinned for full PCIe speed): one C-ABI call
    does H2D, the D^-1/2 pre-scale, K fused hops and D2H, and returns when `out_host` is valid."""
    if z0_host.is_cuda or out_host.is_cuda:
        raise RuntimeError("appnp_host takes host tensors")
    if z0_host.dtype != torch.float32 or not z0_host.is_contiguous() or not out_host.is_contiguous():
        raise RuntimeError("appnp_host needs contiguous float32 host tensors")
    N, F = z0_host.shape
    if plan is None:
        plan = HostAppnpPlan(graph, F)
    dev = graph.device
    z0d, ping, pong, outd = plan.bufs
    check(lib().rgbmp_appnp_host_mapped(plan.csr.hot_ref(plan.ld * 4), ptr(plan.row_map), ptr(plan.dinv), z0_host.data_ptr(),
                                        out_host.data_ptr(), F, K, float(alpha), ptr(z0d), ptr(ping), ptr(pong), ptr(outd),
                                        plan.ld, ptr(plan.ws), 0 if plan.ws is None else plan.ws.numel(), dev.index,
                                        stream_of(dev)), "appnp_host")
    return out_host
