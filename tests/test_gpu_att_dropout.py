"""Attention dropout generated inside the fused GAT / SuperGAT-MX / FAConv kernels from a device seed
(csrc/philox.cuh): the device mask equals the numpy restatement (philox_ref); a fused call is bit-identical to the
explicit-mask call fed the mask rgbmp_dropout_mask writes for the same seed (output and every gradient); the same
seed reproduces; nothing edge-sized is allocated; the shim's switch; guard bands."""
import pytest
import torch
import torch.nn.functional as F

import philox_ref as PR
from helpers import CASES

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CASE_NAMES = ["tiny", "loops_dups", "isolated", "hub", "medium"]


def P():
    import rgb_experiment_b200 as P_
    return P_


def _gen(s):
    return torch.Generator(device=DEV).manual_seed(s)


def _seed_of(s):
    """the seed tensor a call given generator _gen(s) draws"""
    return P().ops.dropout_seed(DEV, _gen(s))


# ------------------------------------------------------------------------------------------
# 1. the device mask
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", [1, 3, 8])
@pytest.mark.parametrize("p", [0.2, 0.5])
def test_dropout_mask_equals_numpy_restatement(H, p):
    ops = P().ops
    ei, n = CASES["medium"]()
    g = P().Graph(ei.to(DEV), n, P().LOOP_REMOVE_THEN_ADD)
    seed = _seed_of(11 + H)
    m = ops.dropout_mask(g, H, p, seed)
    want = PR.mask(int(seed.item()), g.nnz, H, p)
    assert m.shape == (g.nnz, H)
    assert torch.equal(m.cpu(), torch.from_numpy(want))


def test_dropout_mask_keep_fraction_and_seeding():
    p_ = P()
    import rgb_experiment_b200.synth as S
    sg = S.make_graph(50_000, 4_000_000, 8, 4, features=False, device=DEV)
    g = p_.Graph(sg.edge_index, sg.num_nodes, p_.LOOP_REMOVE_THEN_ADD)
    H, p = 8, 0.5
    torch.manual_seed(123)
    m1 = p_.ops.dropout_mask(g, H, p, p_.ops.dropout_seed(DEV))
    m2 = p_.ops.dropout_mask(g, H, p, p_.ops.dropout_seed(DEV))          # the next draw of the same generator
    torch.manual_seed(123)
    m3 = p_.ops.dropout_mask(g, H, p, p_.ops.dropout_seed(DEV))
    assert torch.equal(m1, m3)
    assert not torch.equal(m1, m2)
    n = g.nnz
    sigma = (p * (1 - p) / n) ** 0.5
    frac = (m1 != 0).double().mean(0)
    assert ((frac - (1 - p)).abs() < 5 * sigma).all(), frac
    assert set(torch.unique(m1).tolist()) == {0.0, float(torch.tensor(1 / (1 - p), dtype=torch.float32))}
    assert torch.equal(p_.ops.dropout_mask(g, 2, 1.0, p_.ops.dropout_seed(DEV)), torch.zeros(n, 2, device=DEV))


# ------------------------------------------------------------------------------------------
# 2. fused == explicit mask, bit for bit
# ------------------------------------------------------------------------------------------
def _run(fn, ins, dout):
    ins = [t.clone().requires_grad_(True) for t in ins]
    out = fn(*ins)
    out.backward(dout)
    return [out.detach()] + [t.grad for t in ins]


def _assert_equal(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), (i, (x - y).abs().max().item())


@pytest.mark.parametrize("case", CASE_NAMES)
@pytest.mark.parametrize("H,C", [(8, 8), (1, 41), (1, 7), (2, 16), (4, 4), (3, 5), (1, 130), (5, 32), (8, 47)])
@pytest.mark.parametrize("p", [0.3, 0.5])
def test_gat_fused_dropout_equals_explicit_mask(case, H, C, p):
    p_ = P()
    ops = p_.ops
    ei, n = CASES[case]()
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_REMOVE_THEN_ADD)
    gen = torch.Generator(device=DEV).manual_seed(H * 1000 + C)
    ins = [torch.randn(n, H * C, device=DEV, generator=gen), torch.randn(n, H, device=DEV, generator=gen),
           torch.randn(n, H, device=DEV, generator=gen)]
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    s = 7 + H + C
    fused = _run(lambda x, a, b: ops.gat(x, a, b, g, H, C, 0.2, dropout_p=p, generator=_gen(s)), ins, dout)
    mask = ops.dropout_mask(g, H, p, _seed_of(s))
    explicit = _run(lambda x, a, b: ops.gat(x, a, b, g, H, C, 0.2, mask), ins, dout)
    _assert_equal(fused, explicit)


@pytest.mark.parametrize("case", CASE_NAMES)
@pytest.mark.parametrize("H,C", [(8, 8), (8, 10), (3, 4), (2, 47), (1, 16), (1, 41), (5, 32), (1, 130)])
@pytest.mark.parametrize("p", [0.3, 0.5])
def test_supergat_mx_fused_dropout_equals_explicit_mask(case, H, C, p):
    p_ = P()
    ops = p_.ops
    ei, n = CASES[case]()
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_REMOVE_THEN_ADD)
    gen = torch.Generator(device=DEV).manual_seed(H * 100 + C)
    ins = [torch.randn(n, H * C, device=DEV, generator=gen) * 0.7, torch.randn(n, H, device=DEV, generator=gen),
           torch.randn(n, H, device=DEV, generator=gen)]
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    s = 5 + H * C
    fused = _run(lambda x, a, b: ops.supergat_mx(x, a, b, g, H, C, 0.2, dropout_p=p, generator=_gen(s)), ins, dout)
    mask = ops.dropout_mask(g, H, p, _seed_of(s))
    explicit = _run(lambda x, a, b: ops.supergat_mx(x, a, b, g, H, C, 0.2, mask), ins, dout)
    _assert_equal(fused, explicit)


@pytest.mark.parametrize("case", CASE_NAMES)
@pytest.mark.parametrize("C", [64, 16, 7, 100, 130])
@pytest.mark.parametrize("p", [0.3, 0.5])
def test_faconv_fused_dropout_equals_explicit_mask(case, C, p):
    p_ = P()
    ops = p_.ops
    ei, n = CASES[case]()
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_ADD_REMAINING)
    gen = torch.Generator(device=DEV).manual_seed(C)
    ins = [torch.randn(n, C, device=DEV, generator=gen), torch.randn(n, 1, device=DEV, generator=gen),
           torch.randn(n, 1, device=DEV, generator=gen)]
    dout = torch.randn(n, C, device=DEV, generator=gen)
    s = 3 + C
    fused = _run(lambda x, a, b: ops.faconv(x, a, b, g, dropout_p=p, generator=_gen(s)), ins, dout)
    mask = ops.dropout_mask(g, 1, p, _seed_of(s)).view(-1)
    explicit = _run(lambda x, a, b: ops.faconv(x, a, b, g, mask), ins, dout)
    _assert_equal(fused, explicit)


def test_dropout_argument_checks():
    p_ = P()
    ops = p_.ops
    ei, n = CASES["tiny"]()
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_REMOVE_THEN_ADD)
    x, a = torch.randn(n, 8, device=DEV), torch.randn(n, 1, device=DEV)
    with pytest.raises(ValueError):
        ops.gat(x, a, a, g, 1, 8, 0.2, torch.ones(g.nnz, 1, device=DEV), dropout_p=0.5)
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError):
            ops.faconv(x, a, a, g, dropout_p=bad)
        with pytest.raises(ValueError):
            ops.supergat_mx(x, a, a, g, 1, 8, 0.2, dropout_p=bad)
    out = ops.gat(x, a, a, g, 1, 8, 0.2, dropout_p=1.0)                # p == 1 drops everything, like F.dropout
    assert torch.equal(out, torch.zeros_like(out))


# ------------------------------------------------------------------------------------------
# 3. reproducibility
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["gat", "supergat_mx", "faconv"])
def test_same_seed_reproduces_and_backward_regenerates(name):
    p_ = P()
    ops = p_.ops
    ei, n = CASES["hub"]()
    H, C = (1, 64) if name == "faconv" else (8, 8)
    g = p_.Graph(ei.to(DEV), n, p_.LOOP_ADD_REMAINING if name == "faconv" else p_.LOOP_REMOVE_THEN_ADD)
    gen = torch.Generator(device=DEV).manual_seed(1)
    ins = [torch.randn(n, H * C, device=DEV, generator=gen), torch.randn(n, H, device=DEV, generator=gen),
           torch.randn(n, H, device=DEV, generator=gen)]
    dout = torch.randn(n, H * C, device=DEV, generator=gen)

    def call(x, a, b, s):
        if name == "faconv":
            return ops.faconv(x, a, b, g, dropout_p=0.5, generator=_gen(s))
        return getattr(ops, name)(x, a, b, g, H, C, 0.2, dropout_p=0.5, generator=_gen(s))

    runs = []
    for _ in range(2):
        xs = [t.clone().requires_grad_(True) for t in ins]
        out = call(*xs, 42)
        out.backward(dout, retain_graph=True)
        first = [t.grad.clone() for t in xs]
        for t in xs:
            t.grad = None
        out.backward(dout)                                   # the saved seed regenerates the forward's mask
        _assert_equal(first, [t.grad for t in xs])
        runs.append([out.detach()] + first)
    _assert_equal(runs[0], runs[1])
    other = call(*ins, 43)
    assert not torch.equal(other, runs[0][0])


# ------------------------------------------------------------------------------------------
# 4. memory
# ------------------------------------------------------------------------------------------
def _peak_of_step(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


@pytest.mark.parametrize("name", ["supergat_mx", "faconv"])
def test_fused_dropout_allocates_nothing_edge_sized(name):
    """Training forward + backward at p = 0.5 on a 4 M-edge graph: the fused step's peak exceeds the no-dropout
    step's by less than a quarter of one [nnz, H] fp32 tensor; the torch-mask step's by more than a whole one."""
    p_ = P()
    ops = p_.ops
    import rgb_experiment_b200.synth as S
    sg = S.make_graph(50_000, 4_000_000, 8, 4, features=False, device=DEV)
    n = sg.num_nodes
    if name == "faconv":
        H, C = 1, 64
        g = p_.Graph(sg.edge_index, n, p_.LOOP_ADD_REMAINING)
    else:
        H, C = 8, 8
        g = p_.Graph(sg.edge_index, n, p_.LOOP_REMOVE_THEN_ADD)
    g.bwd, g.dinv(), g.tpos()                                  # graph-side caches built outside the measured steps
    gen = torch.Generator(device=DEV).manual_seed(0)
    x = torch.randn(n, H * C, device=DEV, generator=gen)
    a_l, a_r = torch.randn(n, H, device=DEV, generator=gen), torch.randn(n, H, device=DEV, generator=gen)
    dout = torch.randn(n, H * C, device=DEV, generator=gen)

    def step(mode):
        def run():
            xs = [t.clone().requires_grad_(True) for t in (x, a_l, a_r)]
            kw = {}
            if mode == "fused":
                kw = dict(dropout_p=0.5)
            elif mode == "torch":
                shape = (g.nnz,) if name == "faconv" else (g.nnz, H)
                kw = dict(drop_edge=F.dropout(torch.ones(shape, device=DEV), p=0.5, training=True))
            if name == "faconv":
                out = ops.faconv(*xs, g, **kw)
            else:
                out = ops.supergat_mx(*xs, g, H, C, 0.2, **kw)
            out.backward(dout)
        return run

    for m in ("none", "fused", "torch"):                       # warm-up: workspaces, kernels, allocator pools
        step(m)()
    base = _peak_of_step(step("none"))
    fused = _peak_of_step(step("fused"))
    torch_mask = _peak_of_step(step("torch"))
    edge_bytes = g.nnz * H * 4
    assert fused - base < edge_bytes / 4, (fused, base, edge_bytes)
    assert torch_mask - base > edge_bytes, (torch_mask, base, edge_bytes)


# ------------------------------------------------------------------------------------------
# 5. the shim's switch
# ------------------------------------------------------------------------------------------
def _layers():
    from rgb_experiment_b200.shim import nn as SN
    torch.manual_seed(0)
    return {
        "gat": (SN.GATConv(16, 8, heads=8, dropout=0.5), 8, 8),
        "supergat": (SN.SuperGATConv(16, 8, heads=8, dropout=0.5, attention_type="MX"), 8, 8),
        "faconv": (SN.FAConv(16, 0.3, 0.5), 1, 16),
    }


def _layer_call(layer, name, x, ei):
    return layer(x, x, ei) if name == "faconv" else layer(x, ei)


def _reference(layer, name, x, ei, H, C, p_mask):
    """the layer's arithmetic through ops, with the explicit mask `p_mask(g)` (None: no dropout)"""
    p_ = P()
    ops = p_.ops
    if name == "faconv":
        g = p_.get_graph(ei, x.size(0), p_.LOOP_ADD_REMAINING)
        m = p_mask(g, 1)
        return ops.faconv(x, layer.att_l(x), layer.att_r(x), g, None if m is None else m.view(-1)) + layer.eps * x
    g = p_.get_graph(ei, x.size(0), p_.LOOP_REMOVE_THEN_ADD)
    xp = layer.lin(x)
    x3 = xp.view(-1, H, C)
    m = p_mask(g, H)
    if name == "gat":
        out = ops.gat(xp, (x3 * layer.att_src).sum(-1), (x3 * layer.att_dst).sum(-1), g, H, C, layer.negative_slope, m)
    else:
        out = ops.supergat_mx(xp, (x3 * layer.att_l).sum(-1), (x3 * layer.att_r).sum(-1), g, H, C,
                              layer.negative_slope, m)
    return out + layer.bias


@pytest.mark.parametrize("name", ["gat", "supergat", "faconv"])
def test_shim_switch(name, monkeypatch):
    p_ = P()
    ops = p_.ops
    from rgb_experiment_b200.shim import nn as SN
    assert ops.FUSED_DROPOUT is False
    layer, H, C = _layers()[name]
    layer = layer.to(DEV)
    ei, n = CASES["medium"]()
    ei = ei.to(DEV)
    x = torch.randn(n, 16, device=DEV)
    calls = []
    real_dropout = F.dropout

    def counting_dropout(t, *a, **kw):
        calls.append(tuple(t.shape))
        return real_dropout(t, *a, **kw)

    monkeypatch.setattr(SN.F, "dropout", counting_dropout)
    layer.train()
    with torch.no_grad():
        _layer_call(layer, name, x, ei)
    nnz = p_.get_graph(ei, n, p_.LOOP_ADD_REMAINING if name == "faconv" else p_.LOOP_REMOVE_THEN_ADD).nnz
    assert any(s[0] == nnz for s in calls)                     # switch off: the torch mask, as before
    calls.clear()
    monkeypatch.setattr(ops, "FUSED_DROPOUT", True)
    with torch.no_grad():
        torch.manual_seed(77)
        out = _layer_call(layer, name, x, ei)
        torch.manual_seed(77)
        seed = ops.dropout_seed(DEV)
        ref = _reference(layer, name, x, ei, H, C, lambda g, h: ops.dropout_mask(g, h, 0.5, seed))
    assert not any(s and s[0] == nnz for s in calls)           # no edge-sized torch mask
    assert torch.equal(out, ref)
    layer.eval()
    with torch.no_grad():
        out = _layer_call(layer, name, x, ei)
        ref = _reference(layer, name, x, ei, H, C, lambda g, h: None)
    assert torch.equal(out, ref)


# ------------------------------------------------------------------------------------------
# 6. guard bands
# ------------------------------------------------------------------------------------------
def test_fused_dropout_entry_points_under_guard_bands():
    from test_gpu_guard_bands import GuardedAllocator
    p_ = P()
    ops = p_.ops
    p_.graph.clear_cache()
    p_.memo.clear()
    ga = GuardedAllocator()
    ga.install()
    results = []
    try:
        for case in ("loops_dups", "hub", "isolated"):
            ei, n = CASES[case]()
            for name, H, C in (("gat", 8, 8), ("supergat_mx", 3, 16), ("faconv", 1, 41), ("gat", 1, 130)):
                loop = p_.LOOP_ADD_REMAINING if name == "faconv" else p_.LOOP_REMOVE_THEN_ADD
                g = p_.Graph(ei.to(DEV), n, loop)
                xs = [torch.randn(n, H * C, device=DEV).requires_grad_(True),
                      torch.randn(n, H, device=DEV).requires_grad_(True),
                      torch.randn(n, H, device=DEV).requires_grad_(True)]
                if name == "faconv":
                    out = ops.faconv(*xs, g, dropout_p=0.4)
                else:
                    out = getattr(ops, name)(*xs, g, H, C, 0.2, dropout_p=0.4)
                out.backward(torch.randn_like(out))
                results += [out.detach()] + [t.grad for t in xs]
                results.append(ops.dropout_mask(g, H, 0.4, ops.dropout_seed(DEV)))
        torch.cuda.synchronize()
    finally:
        ga.uninstall()
    assert len(ga.records) > 50
    assert ga.violations() == 0
    assert all(bool(torch.isfinite(r).all()) for r in results)
