"""SuperGATConv's SD attention fused into the attention kernel family (csrc/att.cu, RGBMP_ATT_SD; ops.supergat_sd):
forward and backward against an fp64 statement of SD over every head shape class, long rows in both orientations,
with and without a mask; fused dropout bit-identical to the explicit mask; repeatability; nothing edge-sized
allocated; the shim layer against the oracle layer and its dropout switch; memo and argument checks; guard bands."""
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import CASES, relerr
from oracle import layers as OL
from oracle import pyg_restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5
CASE_NAMES = ["tiny", "loops_dups", "isolated", "hub", "medium"]
# (1, 130) is wider than the kernels take: the unfused chain; (8, 10), (2, 47), (8, 47) run with padded heads and
# only agree with the oracle when the logit is scaled by the UNPADDED width
SHAPES = [(8, 8), (8, 10), (3, 4), (2, 47), (8, 47), (1, 16), (1, 41), (1, 7), (5, 32), (1, 130)]


def P():
    import rgb_experiment_b200 as P_
    return P_


def _gen(s):
    return torch.Generator(device=DEV).manual_seed(s)


def sd_oracle(x64, ei, n, H, Cc, slope=0.2, keep=None):
    """SD attention + aggregate in fp64 from the edge list: x64 [n, H, C], keep [E, H] in edge order."""
    ed = R.edit_loops(ei, n, R.LOOP_REMOVE_THEN_ADD)
    e = F.leaky_relu((x64[ed[1]] * x64[ed[0]]).sum(-1) / math.sqrt(Cc), slope)
    alpha = R.softmax(e, ed[1], num_nodes=n)
    if keep is not None:
        alpha = alpha * keep
    return R.scatter_add(x64[ed[0]] * alpha.unsqueeze(-1), ed[1], dim=0, dim_size=n).reshape(n, H * Cc)


# ------------------------------------------------------------------------------------------
# 1. forward and backward vs fp64
# ------------------------------------------------------------------------------------------
KINK = 1e-6


def _away_from_kink(ei, n, H, C, seed):
    """The first generator from `seed` on whose x keeps every fp64 logit <x_i, x_j>/sqrt(C) at least KINK from 0.
    leaky_relu has no derivative at 0; a logit within fp32 rounding of it (about 4e-8 here) takes either slope
    depending on the summation order, so the gradient is only compared where both sides see the same branch."""
    ed = R.edit_loops(ei, n, R.LOOP_REMOVE_THEN_ADD)
    for s in range(seed, seed + 50):
        gen = torch.Generator().manual_seed(s)
        xp = torch.randn(n, H, C, generator=gen) * 0.7
        x64 = xp.double()
        if bool(((x64[ed[1]] * x64[ed[0]]).sum(-1).abs() / math.sqrt(C) >= KINK).all()):
            return gen, xp, ed
    raise AssertionError("no seed keeps the logits away from the kink")


@pytest.mark.parametrize("case", CASE_NAMES)
@pytest.mark.parametrize("H,C", SHAPES)
@pytest.mark.parametrize("masked", [False, True])
def test_supergat_sd_forward_backward(case, H, C, masked):
    p = P()
    ei, n = CASES[case]()
    gen, xp, ed = _away_from_kink(ei, n, H, C, H * 100 + C)
    dout = torch.randn(n, H * C, generator=gen)
    keep = (torch.rand(ed.size(1), H, generator=gen) > 0.3).float() / 0.7 if masked else None
    xo = xp.double().requires_grad_(True)
    out_o = sd_oracle(xo, ei, n, H, C, keep=None if keep is None else keep.double())
    out_o.backward(dout.double())
    g = p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD)
    xg = xp.view(n, H * C).to(DEV).requires_grad_(True)
    out = p.ops.supergat_sd(xg, g, H, C, 0.2, None if keep is None else keep.to(DEV))
    out.backward(dout.to(DEV))
    assert relerr(out.detach(), out_o.detach()) <= TOL
    assert relerr(xg.grad, xo.grad.reshape(n, H * C)) <= 2e-5


def test_fusable_shapes_and_split_rows():
    """The shapes above run fused except (1, 130); hub and medium have long rows in both orientations."""
    p = P()
    ops = p.ops
    assert [ops.att_fusable(ops.ATT_SD, H, C) for H, C in SHAPES] == [True] * 9 + [False]
    for case in ("hub", "medium"):
        ei, n = CASES[case]()
        g = p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD)
        assert g.fwd.n_long > 0 and g.bwd.n_long > 0, case


# ------------------------------------------------------------------------------------------
# 2. fused dropout == explicit mask, bit for bit
# ------------------------------------------------------------------------------------------
def _run(fn, x, dout):
    x = x.clone().requires_grad_(True)
    out = fn(x)
    out.backward(dout)
    return out.detach(), x.grad


@pytest.mark.parametrize("case", CASE_NAMES)
@pytest.mark.parametrize("H,C", SHAPES)
@pytest.mark.parametrize("p", [0.3, 0.5])
def test_fused_dropout_equals_explicit_mask(case, H, C, p):
    p_ = P()
    ops = p_.ops
    ei, n = CASES[case]()
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_REMOVE_THEN_ADD)
    gen = torch.Generator(device=DEV).manual_seed(H * 100 + C)
    x = torch.randn(n, H * C, device=DEV, generator=gen) * 0.7
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    s = 9 + H * C
    fused = _run(lambda t: ops.supergat_sd(t, g, H, C, 0.2, dropout_p=p, generator=_gen(s)), x, dout)
    mask = ops.dropout_mask(g, H, p, ops.dropout_seed(DEV, _gen(s)))
    explicit = _run(lambda t: ops.supergat_sd(t, g, H, C, 0.2, mask), x, dout)
    for i, (a, b) in enumerate(zip(fused, explicit)):
        assert torch.equal(a, b), (i, (a - b).abs().max().item())


# ------------------------------------------------------------------------------------------
# 3. repeatability
# ------------------------------------------------------------------------------------------
def test_same_seed_reproduces_and_backward_is_deterministic():
    p = P()
    ops = p.ops
    ei, n = CASES["hub"]()
    H, C = 8, 8
    g = p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD)
    gen = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn(n, H * C, device=DEV, generator=gen)
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    runs = []
    for _ in range(2):
        xs = x.clone().requires_grad_(True)
        out = ops.supergat_sd(xs, g, H, C, 0.2, dropout_p=0.5, generator=_gen(42))
        out.backward(dout, retain_graph=True)
        first = xs.grad.clone()
        xs.grad = None
        out.backward(dout)                                   # the saved seed regenerates the forward's mask
        assert torch.equal(first, xs.grad)
        runs.append((out.detach(), first))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert not torch.equal(ops.supergat_sd(x, g, H, C, 0.2, dropout_p=0.5, generator=_gen(43)), runs[0][0])
    grads = []                                               # no dropout, no atomics: identical bits
    for _ in range(2):
        xs = x.clone().requires_grad_(True)
        ops.supergat_sd(xs, g, H, C, 0.2).backward(dout)
        grads.append(xs.grad)
    assert torch.equal(grads[0], grads[1])


# ------------------------------------------------------------------------------------------
# 4. memory
# ------------------------------------------------------------------------------------------
def test_sd_allocates_nothing_edge_sized():
    """8x8 heads on the 4 M-edge graph: the eval forward's peak stays below a quarter of one [nnz, H] fp32 tensor.
    The training step (fused dropout, forward + backward) must hold node-sized buffers -- its input, out, dX, the
    dXf scratch, rowmax / rowsum and a workspace -- that at 80 edges per node already add up to more than that
    quarter, so its peak minus those buffers (sized from the shapes and the workspace queries) must stay below it;
    the chain of edge-sized tensors the layer ran before exceeds a whole [nnz, H] tensor on the same step."""
    p = P()
    ops = p.ops
    import rgb_experiment_b200.synth as S
    sg = S.make_graph(50_000, 4_000_000, 8, 4, features=False, device=DEV)
    n, H, C = sg.num_nodes, 8, 8
    g = p.Graph(sg.edge_index, n, p.LOOP_REMOVE_THEN_ADD)
    g.bwd, g.tpos()                                          # graph-side caches built outside the measured steps
    gen = torch.Generator(device=DEV).manual_seed(0)
    xp = torch.randn(n, H * C, device=DEV, generator=gen)
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    edge_bytes = g.nnz * H * 4

    def peak_of(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    def train(fused):
        def run():
            x = xp.clone().requires_grad_(True)
            if fused:
                out = ops.supergat_sd(x, g, H, C, 0.2, dropout_p=0.5)
            else:                                            # the layer's former chain
                keep = F.dropout(torch.ones((g.nnz, H), device=DEV), p=0.5, training=True)
                a = F.leaky_relu(ops.edge_sddmm(x, x, g, H, C) / math.sqrt(C), 0.2)
                out = ops.spmm_heads(ops.edge_softmax(a, g) * g.to_csr_order(keep), x, g, H, C)
            out.backward(dout)
        return run

    with torch.no_grad():
        ops.supergat_sd(xp, g, H, C, 0.2)
        p.memo.clear()
        x2 = xp * 1.0001
        eval_peak = peak_of(lambda: ops.supergat_sd(x2, g, H, C, 0.2))
    assert eval_peak < edge_bytes / 4, (eval_peak, edge_bytes)
    for fused in (True, False):                              # warm-up
        train(fused)()
    L = p._lib.lib()
    node = (4 * n * H * C * 4 + 2 * n * H * 4 + 8
            + max(L.rgbmp_att_forward_workspace_bytes(g.fwd.ref, H, C),
                  L.rgbmp_att_backward_workspace_bytes(g.fwd.ref, g.bwd.ref, H, C)))
    fused_peak = peak_of(train(True))
    assert fused_peak - node < edge_bytes / 4, (fused_peak, node, edge_bytes)
    assert peak_of(train(False)) > edge_bytes, edge_bytes


# ------------------------------------------------------------------------------------------
# 5. the shim layer
# ------------------------------------------------------------------------------------------
def _layers(kw, seed=0):
    import importlib
    PL = importlib.import_module("rgb_experiment_b200.shim.nn")
    torch.manual_seed(seed)
    o = OL.SuperGATConv(12, kw.pop("out"), attention_type="SD", **kw).double()
    torch.manual_seed(seed)
    g = PL.SuperGATConv(12, o.out_channels, attention_type="SD", **kw)
    g.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    with torch.no_grad():
        o.bias.normal_()
        g.bias.copy_(o.bias.float())
    return o, g.to(DEV)


@pytest.mark.parametrize("heads,out,concat", [(4, 8, True), (3, 10, False), (8, 7, False)])
@pytest.mark.parametrize("training", [False, True])
def test_layer_matches_oracle(heads, out, concat, training):
    ei, n = CASES["hub"]()
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(n, 12, generator=gen)
    neg = torch.randint(n, (2, 150), generator=gen)
    o, g = _layers({"heads": heads, "out": out, "concat": concat, "dropout": 0.0, "edge_sample_ratio": 1.0})
    o.train(training)
    g.train(training)
    xo, xg = x.double().requires_grad_(True), x.to(DEV).requires_grad_(True)
    args_o, args_g = ((ei, neg), (ei.to(DEV), neg.to(DEV))) if training else ((ei,), (ei.to(DEV),))
    yo, yg = o(xo, *args_o), g(xg, *args_g)
    lo_, lg_ = yo.pow(2).sum(), yg.pow(2).sum()
    if training:
        lo_, lg_ = lo_ + 4.0 * o.get_attention_loss(), lg_ + 4.0 * g.get_attention_loss()
    lo_.backward()
    lg_.backward()
    assert relerr(yg.detach(), yo.detach()) <= TOL
    assert relerr(xg.grad, xo.grad) <= 3e-5
    po, pg = dict(o.named_parameters()), dict(g.named_parameters())
    for k in po:
        assert relerr(pg[k].grad, po[k].grad) <= 5e-5, k


def _explicit(layer, x, ei, keep_of):
    """the layer's arithmetic through ops with the explicit mask keep_of(g)"""
    p = P()
    g = p.get_graph(ei, x.size(0), p.LOOP_REMOVE_THEN_ADD)
    H, C = layer.heads, layer.out_channels
    return p.ops.supergat_sd(layer.lin(x), g, H, C, layer.negative_slope, keep_of(g)) + layer.bias, g


def test_layer_dropout_switch(monkeypatch):
    p = P()
    ops = p.ops
    from rgb_experiment_b200.shim import nn as SN
    assert ops.FUSED_DROPOUT is False
    torch.manual_seed(0)
    layer = SN.SuperGATConv(16, 8, heads=8, dropout=0.5, attention_type="SD").to(DEV).train()
    ei, n = CASES["medium"]()
    ei = ei.to(DEV)
    x = torch.randn(n, 16, device=DEV)
    H = 8
    nnz = p.get_graph(ei, n, p.LOOP_REMOVE_THEN_ADD).nnz
    calls = []
    real_dropout = F.dropout

    def counting_dropout(t, *a, **kw):
        calls.append(tuple(t.shape))
        return real_dropout(t, *a, **kw)

    # off: the mask of the same F.dropout call as before, drawn at the same point of the torch RNG stream
    monkeypatch.setattr(SN.F, "dropout", counting_dropout)
    with torch.no_grad():
        torch.manual_seed(5)
        out = layer(x, ei)
        torch.manual_seed(5)
        ref, g = _explicit(layer, x, ei, lambda g: real_dropout(torch.ones((g.nnz, H), device=DEV), p=0.5, training=True))
    assert (nnz, H) in calls
    assert torch.equal(out, ref)
    with torch.no_grad():                                    # and that mask means what the oracle says
        torch.manual_seed(5)
        keep = real_dropout(torch.ones((nnz, H), device=DEV), p=0.5, training=True)
        x3 = layer.lin(x).view(n, H, 8).double().cpu()
        want = sd_oracle(x3, ei.cpu(), n, H, 8, keep=keep.double().cpu()) + layer.bias.double().cpu()
    assert relerr(out, want) <= TOL
    # on: one seed drawn where the shim drew it before, the kernels generate the mask; nothing edge-sized in torch
    calls.clear()
    monkeypatch.setattr(ops, "FUSED_DROPOUT", True)
    xs = [x.clone().requires_grad_(True) for _ in range(2)]
    dout = torch.randn(n, 64, device=DEV)
    torch.manual_seed(77)
    out = layer(xs[0], ei)
    out.backward(dout)
    w_grad = layer.lin.weight.grad.clone()
    layer.zero_grad()
    assert not any(s and s[0] == nnz for s in calls)
    torch.manual_seed(77)
    seed = ops.dropout_seed(DEV)
    ref, _ = _explicit(layer, xs[1], ei, lambda g: ops.dropout_mask(g, H, 0.5, seed))
    ref.backward(dout)
    assert torch.equal(out.detach(), ref.detach())
    assert torch.equal(xs[0].grad, xs[1].grad) and torch.equal(w_grad, layer.lin.weight.grad)
    layer.eval()
    with torch.no_grad():
        assert torch.equal(layer(x, ei), _explicit(layer, x, ei, lambda g: None)[0])


# ------------------------------------------------------------------------------------------
# 6. memo, dtypes, argument checks
# ------------------------------------------------------------------------------------------
def test_eval_memo_returns_the_stored_result():
    p = P()
    M = p.memo
    import rgb_experiment_b200.synth as S
    sg = S.make_graph(50_000, 4_000_000, 8, 4, features=False, device=DEV)
    g = p.Graph(sg.edge_index, sg.num_nodes, p.LOOP_REMOVE_THEN_ADD)
    x = torch.randn(sg.num_nodes, 64, device=DEV)
    M.clear()
    with torch.no_grad():
        h0, m0 = M.stats["hits"], M.stats["misses"]
        a = p.ops.supergat_sd(x, g, 8, 8, 0.2)
        b = p.ops.supergat_sd(x.clone(), g, 8, 8, 0.2)
        assert M.stats["misses"] == m0 + 1 and M.stats["hits"] == h0 + 1
        assert torch.equal(a, b)
        p.ops.supergat_sd(x * 1.5, g, 8, 8, 0.2)
        assert M.stats["misses"] == m0 + 2
        a = torch.randn(sg.num_nodes, 8, device=DEV)
        p.ops.supergat_mx(x, a, a, g, 8, 8, 0.2)            # another op on the same graph: its own entry
        assert M.stats["misses"] == m0 + 3
    M.clear()


def test_dtypes_and_argument_checks():
    p = P()
    ops = p.ops
    ei, n = CASES["tiny"]()
    g = p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD)
    x = torch.randn(n, 64, device=DEV)
    for dt in (torch.bfloat16, torch.float64):
        for H, C in ((8, 8), (1, 130)):
            with pytest.raises(RuntimeError, match="float32"):
                ops.supergat_sd(torch.randn(n, H * C, device=DEV).to(dt), g, H, C)
    with pytest.raises(ValueError):
        ops.supergat_sd(x, g, 8, 8, 0.2, torch.ones(g.nnz, 8, device=DEV), dropout_p=0.5)
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError):
            ops.supergat_sd(x, g, 8, 8, 0.2, dropout_p=bad)
    out = ops.supergat_sd(x, g, 8, 8, 0.2, dropout_p=1.0)    # p == 1 drops everything, like F.dropout
    assert torch.equal(out, torch.zeros_like(out))


# ------------------------------------------------------------------------------------------
# 7. guard bands
# ------------------------------------------------------------------------------------------
def test_sd_entry_points_under_guard_bands():
    from test_gpu_guard_bands import GuardedAllocator
    p = P()
    ops = p.ops
    p.graph.clear_cache()
    p.memo.clear()
    ga = GuardedAllocator()
    ga.install()
    results = []
    try:
        for case in ("loops_dups", "hub", "isolated"):
            ei, n = CASES[case]()
            g = p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD)
            for H, C in ((8, 8), (3, 16), (1, 41), (2, 47)):
                for kw in ({"dropout_p": 0.4}, {"drop_edge": ops.dropout_mask(g, H, 0.4, ops.dropout_seed(DEV))}, {}):
                    x = torch.randn(n, H * C, device=DEV).requires_grad_(True)
                    out = ops.supergat_sd(x, g, H, C, 0.2, **kw)
                    out.backward(torch.randn_like(out))
                    results += [out.detach(), x.grad]
        torch.cuda.synchronize()
    finally:
        ga.uninstall()
    assert len(ga.records) > 50
    assert ga.violations() == 0
    assert all(bool(torch.isfinite(r).all()) for r in results)
