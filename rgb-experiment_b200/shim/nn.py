"""PyG layer classes the reference imports, as nn.Modules over the CUDA ops (SURVEY.md 8b).

Import sites: models/gcn.py:3, graphsage.py:3, graphsage2.py:5, gat.py:3, supergat.py:6,
appnp_stack.py:3, sgc.py:4, dagnn.py:8, fagcn.py:4, ggnn.py:3, gin.py:6, itexperiments.py:21.
Constructor signatures, parameter creation order and initialisers follow SURVEY.md Appendix A
(and are kept identical to oracle/layers.py so that a fixed seed gives identical weights).
Dense pieces (Linear, BatchNorm, GRUCell, bias add) stay PyTorch; every aggregation is a call
into librgbmp.so.
"""
from __future__ import annotations

import inspect
import math
from typing import Optional

import torch
import torch.nn.functional as F
from torch import Tensor, nn

from .. import ops
from ..graph import LOOP_ADD_REMAINING, LOOP_NONE, LOOP_REMOVE_THEN_ADD, get_graph
from . import utils as U


def glorot_(t: Tensor) -> Tensor:
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        return t.uniform_(-a, a)


def _is_weighted_message(cls, extra: str) -> bool:
    """True when cls.message(x_j, <extra>) computes extra.view(-1,1) * x_j (probed once per class
    on a tiny tensor, e.g. Prop.message at dagnn.py:57-59)."""
    cache = cls.__dict__.get("_rgbmp_weighted_probe")
    if cache is not None and extra in cache:
        return cache[extra]
    ok = False
    try:
        g = torch.Generator().manual_seed(7)
        xj = torch.rand(5, 3, generator=g) + 0.5
        w = torch.rand(5, generator=g) + 0.5
        dummy = object.__new__(cls)
        out = cls.message(dummy, **{"x_j": xj, extra: w})
        ok = torch.is_tensor(out) and out.shape == xj.shape and torch.equal(out, w.view(-1, 1) * xj)
    except Exception:
        ok = False
    if cache is None:
        cache = {}
        setattr(cls, "_rgbmp_weighted_probe", cache)
    cache[extra] = ok
    return ok


class MessagePassing(nn.Module):
    """A6.  ``propagate`` fast paths (both hand-written CUDA, autograd-aware):
      * default message (x_j) with aggr add / mean            -> unweighted CSR SpMM
      * message(x_j, w) == w.view(-1,1) * x_j with aggr add   -> weighted CSR SpMM
    Anything else: gather (torch index_select) -> the user's message -> segmented reduce kernel."""

    def __init__(self, aggr: Optional[str] = "add", flow: str = "source_to_target", node_dim: int = -2):
        super().__init__()
        if flow != "source_to_target":
            raise NotImplementedError("flow='target_to_source' is not used by the reference")
        self.aggr, self.flow, self.node_dim = aggr, flow, node_dim

    def propagate(self, edge_index: Tensor, size=None, **kwargs):
        x = kwargs.get("x")
        params = [p for p in inspect.signature(self.message).parameters]
        msg_is_default = type(self).message is MessagePassing.message
        if x is not None and x.dim() == 2 and size is None:
            N = x.size(0)
            if msg_is_default and self.aggr in ("add", "sum", "mean"):
                g = get_graph(edge_index, N, LOOP_NONE)
                return self.update(ops.propagate(x, g, "mean" if self.aggr == "mean" else "sum"))
            if (len(params) == 2 and params[0] == "x_j" and self.aggr in ("add", "sum")
                    and torch.is_tensor(kwargs.get(params[1])) and kwargs[params[1]].dim() == 1
                    and kwargs[params[1]].numel() == edge_index.size(1)
                    and _is_weighted_message(type(self), params[1])):
                g = get_graph(edge_index, N, LOOP_NONE)
                return self.update(ops.propagate_weighted(x, kwargs[params[1]], g))
        return self.update(self._generic(edge_index, size, params, kwargs))

    def _generic(self, edge_index, size, params, kwargs):
        row, col = edge_index[0], edge_index[1]
        N = None
        for v in kwargs.values():
            if torch.is_tensor(v) and v.dim() >= 2:
                N = v.size(0)
                break
        if size is not None:
            N = size[1] if isinstance(size, (tuple, list)) else size
        args = {}
        for name in params:
            if name.endswith("_j"):
                args[name] = kwargs[name[:-2]].index_select(0, row)
            elif name.endswith("_i"):
                args[name] = kwargs[name[:-2]].index_select(0, col)
            elif name in ("index", "edge_index_i"):
                args[name] = col
            elif name == "edge_index_j":
                args[name] = row
            elif name == "ptr":
                args[name] = None
            elif name == "size_i":
                args[name] = N
            elif name in kwargs:
                args[name] = kwargs[name]
        msg = self.message(**args)
        if self.aggr not in ("add", "sum", "mean"):
            raise NotImplementedError(f"aggr={self.aggr!r} has no CUDA path (the reference uses add / mean)")
        g = get_graph(edge_index, N, LOOP_NONE)
        shape = msg.shape
        out = ops.segment_reduce(msg.reshape(shape[0], -1), g, self.aggr == "mean")
        return out.view(N, *shape[1:])

    def message(self, x_j):
        return x_j

    def update(self, inputs):
        return inputs


class GCNConv(MessagePassing):
    """A7 (models/gcn.py:18-21): gcn_norm + X.W + SpMM + bias; the built graph is cached."""

    def __init__(self, in_channels, out_channels, improved=False, cached=False, add_self_loops=True,
                 normalize=True, bias=True, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        if improved:
            raise NotImplementedError("GCNConv(improved=True) is not used by the reference")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.improved, self.cached = improved, cached
        self.add_self_loops, self.normalize = add_self_loops, normalize
        self.lin = nn.Linear(in_channels, out_channels, bias=False)
        self.bias = nn.Parameter(torch.empty(out_channels)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x, edge_index, edge_weight=None):
        if edge_weight is not None:
            raise NotImplementedError("GCNConv with explicit edge_weight is not used by the reference")
        x = self.lin(x)
        if self.normalize:
            g = get_graph(edge_index, x.size(0), LOOP_ADD_REMAINING if self.add_self_loops else LOOP_NONE)
            out = ops.propagate(x, g, "gcn")
        else:
            out = ops.propagate(x, get_graph(edge_index, x.size(0), LOOP_NONE), "sum")
        if self.bias is not None:
            out = out + self.bias
        return out


class SAGEConv(MessagePassing):
    """A14 (models/graphsage2.py:20-23)."""

    def __init__(self, in_channels, out_channels, normalize=False, root_weight=True, bias=True, **kwargs):
        kwargs.setdefault("aggr", "mean")
        super().__init__(**kwargs)
        self.normalize, self.root_weight = normalize, root_weight
        self.lin_l = nn.Linear(in_channels, out_channels, bias=bias)
        if root_weight:
            self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, edge_index):
        out = ops.propagate(x, get_graph(edge_index, x.size(0), LOOP_NONE), "mean")
        out = self.lin_l(out)
        if self.root_weight:
            out = out + self.lin_r(x)
        if self.normalize:
            out = F.normalize(out, p=2.0, dim=-1)
        return out


class GATConv(MessagePassing):
    """A10 (models/gat.py:18-21): fused edge-softmax + aggregate."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, dropout=0.0,
                 add_self_loops=True, bias=True, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.negative_slope, self.dropout = concat, negative_slope, dropout
        self.add_self_loops = add_self_loops
        self.lin = nn.Linear(in_channels, heads * out_channels, bias=False)
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        if bias:
            self.bias = nn.Parameter(torch.empty(heads * out_channels if concat else out_channels))
        else:
            self.bias = None
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        glorot_(self.att_src)
        glorot_(self.att_dst)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x, edge_index):
        H, C = self.heads, self.out_channels
        xp = self.lin(x)
        x3 = xp.view(-1, H, C)
        a_s = (x3 * self.att_src).sum(-1)
        a_d = (x3 * self.att_dst).sum(-1)
        N = xp.size(0)
        g = get_graph(edge_index, N, LOOP_REMOVE_THEN_ADD if self.add_self_loops else LOOP_NONE)
        drop, p = None, 0.0
        if self.training and self.dropout > 0:
            if ops.FUSED_DROPOUT:                                     # generated inside the kernels from a seed
                p = self.dropout
            else:
                drop = F.dropout(torch.ones((g.nnz, H), device=x.device), p=self.dropout, training=True)
        out = ops.gat(xp, a_s, a_d, g, H, C, self.negative_slope, drop, dropout_p=p)
        out = out if self.concat else out.view(-1, H, C).mean(dim=1)
        if self.bias is not None:
            out = out + self.bias
        return out


class SuperGATConv(MessagePassing):
    """A12, MX and SD attention (models/supergat.py:15-21,26,29): scores, edge softmax and aggregate in ONE fused
    kernel pass (ops.supergat_mx / ops.supergat_sd, csrc/att.cu; backward = one pass per orientation, nothing
    edge-sized is allocated).  Edge sampling and the BCE loss on the sampled pairs stay PyTorch (node-pair sized) unless
    ops.FUSED_SUPERGAT_LOSS: then both run on the device (ops.supergat_att_loss) and nothing edge-sized is allocated."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True, negative_slope=0.2, dropout=0.0,
                 add_self_loops=True, bias=True, attention_type="MX", neg_sample_ratio=0.5,
                 edge_sample_ratio=1.0, is_undirected=False, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        assert attention_type in ("MX", "SD")
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.negative_slope, self.dropout = concat, negative_slope, dropout
        self.add_self_loops, self.attention_type = add_self_loops, attention_type
        self.neg_sample_ratio, self.edge_sample_ratio = neg_sample_ratio, edge_sample_ratio
        self.is_undirected = is_undirected
        self.lin = nn.Linear(in_channels, heads * out_channels, bias=False)
        if attention_type == "MX":
            self.att_l = nn.Parameter(torch.empty(1, heads, out_channels))
            self.att_r = nn.Parameter(torch.empty(1, heads, out_channels))
        else:
            self.register_parameter("att_l", None)
            self.register_parameter("att_r", None)
        self.att_x = self.att_y = None
        self._att_loss = None
        if bias:
            self.bias = nn.Parameter(torch.empty(heads * out_channels if concat else out_channels))
        else:
            self.bias = None
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        if self.att_l is not None:
            glorot_(self.att_l)
            glorot_(self.att_r)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def get_attention(self, x_i, x_j, return_logits=False):
        """Dense (sampled-edge) form used for the self-supervised loss only."""
        if self.attention_type == "MX":
            logits = (x_i * x_j).sum(dim=-1)
            if return_logits:
                return logits
            alpha = (x_j * self.att_l).sum(-1) + (x_i * self.att_r).sum(-1)
            alpha = alpha * logits.sigmoid()
        else:
            alpha = (x_i * x_j).sum(dim=-1) / math.sqrt(self.out_channels)
            if return_logits:
                return alpha
        return F.leaky_relu(alpha, self.negative_slope)

    def forward(self, x, edge_index, neg_edge_index=None):
        N, H, C = x.size(0), self.heads, self.out_channels
        g = get_graph(edge_index, N, LOOP_REMOVE_THEN_ADD if self.add_self_loops else LOOP_NONE)
        xp = self.lin(x)
        x3 = xp.view(-1, H, C)
        keep, p = None, 0.0
        if self.training and self.dropout > 0:
            if ops.FUSED_DROPOUT:                                     # generated from a seed (like GATConv)
                p = self.dropout
            else:                                                     # PyTorch RNG mask, edge order (like GATConv)
                keep = F.dropout(torch.ones((g.nnz, H), device=x.device), p=self.dropout, training=True)
        if self.attention_type == "MX":
            a_l = (x3 * self.att_l).sum(-1)
            a_r = (x3 * self.att_r).sum(-1)
            out = ops.supergat_mx(xp, a_l, a_r, g, H, C, self.negative_slope, keep, dropout_p=p)      # one fused pass
        else:                                                         # SD attention (the reference's models use MX)
            out = ops.supergat_sd(xp, g, H, C, self.negative_slope, keep, dropout_p=p)                # one fused pass
        if self.training and ops.FUSED_SUPERGAT_LOSS:                # sampling and BCE on the device
            scale = 1.0 / H if self.attention_type == "MX" else 1.0 / (H * math.sqrt(C))     # att_x.mean(-1)
            self._att_loss = ops.supergat_att_loss(xp, g, H, C, scale, self.edge_sample_ratio, self.neg_sample_ratio,
                                                   self.is_undirected, neg_edge_index)
            self.att_x = self.att_y = None
        elif self.training:
            ei = g.edge_index()
            pos_ei, _ = U.dropout_adj(ei, p=1.0 - self.edge_sample_ratio, training=True)
            ei_for_neg = U.to_undirected(ei, N) if not self.is_undirected else ei
            if neg_edge_index is None:
                num_neg = int(self.neg_sample_ratio * self.edge_sample_ratio * ei.size(1))
                neg_edge_index = U.negative_sampling(ei_for_neg, N, num_neg)
            pos_att = self.get_attention(x3[pos_ei[1]], x3[pos_ei[0]], return_logits=True)
            neg_att = self.get_attention(x3[neg_edge_index[1]], x3[neg_edge_index[0]], return_logits=True)
            self.att_x = torch.cat([pos_att, neg_att], dim=0)
            self.att_y = self.att_x.new_zeros(self.att_x.size(0))
            self.att_y[:pos_ei.size(1)] = 1.0
        out = out if self.concat else out.view(-1, H, C).mean(dim=1)
        if self.bias is not None:
            out = out + self.bias
        return out

    def get_attention_loss(self):
        if not self.training:
            return torch.tensor([0], device=self.lin.weight.device)
        if self.att_x is None and self._att_loss is not None:
            return self._att_loss
        return F.binary_cross_entropy_with_logits(self.att_x.mean(dim=-1), self.att_y)


class APPNP(MessagePassing):
    """A8 (models/appnp_stack.py:22): fused K-hop propagation with the teleport term in the
    SpMM epilogue; backward = the same recursion on the transpose graph."""

    fold_norm = None       # None: ops.FOLD_KHOP (folded D^-1/2 row scalings, the measured path of bench.py);
                           # False: per-edge gcn_norm weights exactly as PyG multiplies them

    def __init__(self, K, alpha, dropout=0.0, cached=False, add_self_loops=True, normalize=True, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        self.K, self.alpha, self.dropout = K, alpha, dropout
        self.add_self_loops, self.normalize = add_self_loops, normalize

    def forward(self, x, edge_index, edge_weight=None):
        if edge_weight is not None or not self.normalize:
            raise NotImplementedError("APPNP with explicit edge_weight / normalize=False is not used by the reference")
        g = get_graph(edge_index, x.size(0), LOOP_ADD_REMAINING if self.add_self_loops else LOOP_NONE)
        if self.dropout > 0 and self.training:
            h = x
            for _ in range(self.K):                                 # edge-weight dropout: per-hop weighted SpMM
                w = F.dropout(g.to_edge_order(g.gcn_val(False)), p=self.dropout)
                x = ops.propagate_weighted(x, w, g)
                x = x * (1 - self.alpha)
                x = x + self.alpha * h
            return x
        return ops.appnp(x, g, self.K, self.alpha, self.fold_norm)


class SGConv(MessagePassing):
    """A9 (models/sgc.py:9-10): K fused hops on the raw features, cached outside state_dict."""

    def __init__(self, in_channels, out_channels, K=1, cached=False, add_self_loops=True, bias=True, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        self.K, self.cached, self.add_self_loops = K, cached, add_self_loops
        self._cached_x = None
        self.lin = nn.Linear(in_channels, out_channels, bias=bias)

    def forward(self, x, edge_index, edge_weight=None):
        cache = self._cached_x
        if cache is None:
            g = get_graph(edge_index, x.size(0), LOOP_ADD_REMAINING if self.add_self_loops else LOOP_NONE)
            x = ops.gcn_power(x, g, self.K)
            if self.cached:
                self._cached_x = x
        else:
            x = cache
        return self.lin(x)


class FAConv(MessagePassing):
    """A13 (models/fagcn.py:15,31): out[i] = sum_j tanh(a_l[j]+a_r[i]) * gcn_norm_ij * x[j], fused (ops.faconv)."""

    def __init__(self, channels, eps=0.1, dropout=0.0, cached=False, add_self_loops=True, normalize=True, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        self.channels, self.eps, self.dropout = channels, eps, dropout
        self.add_self_loops, self.normalize = add_self_loops, normalize
        self.att_l = nn.Linear(channels, 1, bias=False)
        self.att_r = nn.Linear(channels, 1, bias=False)

    def forward(self, x, x_0, edge_index, edge_weight=None):
        if not self.normalize:
            raise NotImplementedError("FAConv(normalize=False) is not used by the reference")
        N = x.size(0)
        g = get_graph(edge_index, N, LOOP_ADD_REMAINING if self.add_self_loops else LOOP_NONE)
        keep, p = None, 0.0
        if self.training and self.dropout > 0:
            if ops.FUSED_DROPOUT:                                     # generated inside the kernel from a seed
                p = self.dropout
            else:
                keep = F.dropout(torch.ones(g.nnz, device=x.device), p=self.dropout, training=True)
        out = ops.faconv(x, self.att_l(x), self.att_r(x), g, keep, dropout_p=p)   # tanh score * gcn weight, fused
        if self.eps != 0.0:
            out = out + self.eps * x_0
        return out


class GINConv(MessagePassing):
    """A14 (models/gin.py:14-32)."""

    def __init__(self, nn_module, eps=0.0, train_eps=False, **kwargs):
        kwargs.setdefault("aggr", "add")
        super().__init__(**kwargs)
        self.nn = nn_module
        self.initial_eps = eps
        if train_eps:
            self.eps = nn.Parameter(torch.tensor([float(eps)]))
        else:
            self.register_buffer("eps", torch.tensor([float(eps)]))

    def reset_parameters(self):
        for m in self.nn.modules():
            if m is not self.nn and hasattr(m, "reset_parameters"):
                m.reset_parameters()
        self.eps.data.fill_(self.initial_eps)

    def forward(self, x, edge_index):
        out = ops.propagate(x, get_graph(edge_index, x.size(0), LOOP_NONE), "sum")
        out = out + (1 + self.eps) * x
        return self.nn(out)


class GatedGraphConv(MessagePassing):
    """A14 (models/ggnn.py:20)."""

    def __init__(self, out_channels, num_layers, aggr="add", bias=True, **kwargs):
        super().__init__(aggr=aggr, **kwargs)
        self.out_channels, self.num_layers = out_channels, num_layers
        self.weight = nn.Parameter(torch.empty(num_layers, out_channels, out_channels))
        self.rnn = nn.GRUCell(out_channels, out_channels, bias=bias)
        bound = 1.0 / math.sqrt(out_channels)
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)

    def forward(self, x, edge_index):
        if x.size(-1) > self.out_channels:
            raise ValueError("input width larger than out_channels")
        if x.size(-1) < self.out_channels:
            x = torch.cat([x, x.new_zeros(x.size(0), self.out_channels - x.size(-1))], dim=1)
        g = get_graph(edge_index, x.size(0), LOOP_NONE)
        for i in range(self.num_layers):
            m = torch.matmul(x, self.weight[i])
            m = ops.propagate(m, g, "mean" if self.aggr == "mean" else "sum")
            x = self.rnn(m, x)
        return x


class LabelPropagation(nn.Module):
    """A15."""

    def __init__(self, num_layers, alpha):
        super().__init__()
        self.num_layers, self.alpha = num_layers, alpha

    @torch.no_grad()
    def forward(self, y, edge_index, mask=None, edge_weight=None, post_step=None):
        if edge_weight is not None or post_step is not None:
            raise NotImplementedError("LabelPropagation with edge_weight / custom post_step has no CUDA path")
        if y.dtype == torch.long:
            y = F.one_hot(y.view(-1)).to(torch.float)
        out = y
        if mask is not None:
            out = torch.zeros_like(y)
            out[mask] = y[mask]
        g = get_graph(edge_index, y.size(0), LOOP_NONE)
        return ops.label_propagation(g, out, self.num_layers, self.alpha)


class CorrectAndSmooth(nn.Module):
    """A15 (itexperiments.py:520-526): both 50-hop label propagations run as fused K-hop kernels
    (teleport + clamp / row reset in the SpMM epilogue)."""

    def __init__(self, num_correction_layers, correction_alpha, num_smoothing_layers, smoothing_alpha,
                 autoscale=True, scale=1.0):
        super().__init__()
        self.autoscale, self.scale = autoscale, scale
        self.prop1 = LabelPropagation(num_correction_layers, correction_alpha)
        self.prop2 = LabelPropagation(num_smoothing_layers, smoothing_alpha)

    @torch.no_grad()
    def correct(self, y_soft, y_true, mask, edge_index, edge_weight=None):
        assert abs(float(y_soft.sum()) / y_soft.size(0) - 1.0) < 1e-2
        numel = int(mask.sum()) if mask.dtype == torch.bool else mask.size(0)
        if y_true.dtype == torch.long:
            y_true = F.one_hot(y_true.view(-1), y_soft.size(-1)).to(y_soft.dtype)
        error = torch.zeros_like(y_soft)
        error[mask] = y_true - y_soft[mask]
        g = get_graph(edge_index, y_soft.size(0), LOOP_NONE)
        if self.autoscale:
            smoothed = ops.label_propagation(g, error, self.prop1.num_layers, self.prop1.alpha, clamp=(-1.0, 1.0))
            sigma = error[mask].abs().sum() / numel
            scale = sigma / smoothed.abs().sum(dim=1, keepdim=True)
            scale[scale.isinf() | (scale > 1000)] = 1.0
            return y_soft + scale * smoothed
        rmask = mask if mask.dtype == torch.bool else torch.zeros(
            y_soft.size(0), dtype=torch.bool, device=y_soft.device).index_fill_(0, mask, True)
        smoothed = ops.label_propagation(g, error, self.prop1.num_layers, self.prop1.alpha,
                                         reset_mask=rmask, reset_val=error)
        return y_soft + self.scale * smoothed

    @torch.no_grad()
    def smooth(self, y_soft, y_true, mask, edge_index, edge_weight=None):
        if y_true.dtype == torch.long:
            y_true = F.one_hot(y_true.view(-1), y_soft.size(-1)).to(y_soft.dtype)
        y_soft = y_soft.clone()
        y_soft[mask] = y_true
        g = get_graph(edge_index, y_soft.size(0), LOOP_NONE)
        return ops.label_propagation(g, y_soft, self.prop2.num_layers, self.prop2.alpha)
