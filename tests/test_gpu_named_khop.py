"""K-hop forwards on the renamed graph (Graph.named_fwd, ops.NAMED_KHOP): the nodes of a locality-grouped graph renamed
in schedule order give the same operator with the same per-row summation order, so every result must be bit-identical
to the K-hop on the graph as built -- on the products-shaped graph, on a graph whose long rows go through the combine
kernel, for aligned and unaligned widths, and through the host-buffer entry point."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAPH_SEED = 20261018         # bench.py's products-shaped graph


def P():
    import rgb_experiment_b200 as P_
    return P_


@pytest.fixture(scope="module")
def products():
    p = P()
    import rgb_experiment_b200.synth as S_
    sg = S_.make_named("products", seed=GRAPH_SEED, device=DEV, features=False)
    g = p.Graph(sg.edge_index, sg.num_nodes, p.LOOP_ADD_REMAINING)
    assert g.groups is not None and g.fwd.clustered
    yield g
    del g
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def split_rows():
    """Grouped graph with small chunk / long_chunk: hundreds of long rows, stored by the combine kernel."""
    p = P()
    from rgb_experiment_b200 import graph as G
    import rgb_experiment_b200.synth as S_
    mp = pytest.MonkeyPatch()
    mp.setattr(G, "CLUSTER", "1")
    mp.setattr(G, "CLUSTER_SEEDS", 64)
    sg = S_.make_graph(60_000, 3_000_000, 8, 12, seed=9, features=False, device=DEV)
    g = p.Graph(sg.edge_index, sg.num_nodes, p.LOOP_ADD_REMAINING, chunk=64, long_chunk=256)
    mp.undo()
    assert g.groups is not None
    return g


def _both(monkeypatch, fn):
    p = P()
    monkeypatch.setattr(p.ops, "NAMED_KHOP", False)
    old = fn()
    monkeypatch.setattr(p.ops, "NAMED_KHOP", True)
    new = fn()
    return old, new


def _check_named(g):
    nf = g.named_fwd
    assert nf is not None and nf.row_order is None and nf.clustered and nf.eid is None
    assert (nf.n_long, nf.n_items) == (g.fwd.n_long, g.fwd.n_items)
    order = g.fwd.row_order.long()
    assert torch.equal(nf.degree(), g.fwd.degree()[order])
    assert torch.equal(nf.norm(P().graph.NORM_INV_SQRT), g.dinv()[order])
    if nf.n_long:                                   # long rows listed in id order = schedule order
        assert bool((nf.long_rows[1:] > nf.long_rows[:-1]).all())


@pytest.mark.parametrize("F", [47, 64])
def test_products_appnp_k10_and_sgc_k2_bit_identical(monkeypatch, products, F):
    p, g = P(), products
    x = torch.randn(g.N, F, device=DEV, generator=torch.Generator(device=DEV).manual_seed(F))
    old, new = _both(monkeypatch, lambda: p.ops._appnp_khop(g.fwd, g, x, 10, 0.1, False, True))
    _check_named(g)
    assert old.shape == new.shape and torch.equal(old, new)
    old, new = _both(monkeypatch, lambda: p.ops._PowerHops.apply(x, g, 2, True))
    assert torch.equal(old, new)


@pytest.mark.parametrize("F", [47, 64])
def test_long_rows_through_the_combine_kernel_bit_identical(monkeypatch, split_rows, F):
    p, g = P(), split_rows
    assert g.fwd.n_long > 100
    x = torch.randn(g.N, F, device=DEV, generator=torch.Generator(device=DEV).manual_seed(F + 1))
    old, new = _both(monkeypatch, lambda: p.ops._appnp_khop(g.fwd, g, x, 3, 0.1, False, True))
    _check_named(g)
    assert torch.equal(old, new)
    old, new = _both(monkeypatch, lambda: p.ops._PowerHops.apply(x, g, 2, True))
    assert torch.equal(old, new)
    old, new = _both(monkeypatch, lambda: p.ops._appnp_khop(g.fwd, g, x[:, :F - 3], 2, 0.2, False, True))   # non-contiguous
    assert torch.equal(old, new)


def test_appnp_host_bit_identical(monkeypatch, products):
    p, g = P(), products
    F = 47
    z0 = torch.randn(g.N, F, generator=torch.Generator().manual_seed(3)).pin_memory()
    outs = []
    for named in (False, True):
        monkeypatch.setattr(p.ops, "NAMED_KHOP", named)
        plan = p.ops.HostAppnpPlan(g, F)
        assert (plan.row_map is not None) == named
        out = torch.empty(g.N, F).pin_memory()
        p.ops.appnp_host(g, z0, out, 10, 0.1, plan)
        outs.append(out)
        del plan
    assert torch.equal(outs[0], outs[1])


def test_backward_and_unfolded_calls_keep_the_built_graph(monkeypatch, split_rows):
    """Gradients run on the transpose CSR, unfolded and bf16 calls on fwd: the same results with the flag on or off."""
    p, g = P(), split_rows
    x = torch.randn(g.N, 16, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
    dz = torch.randn_like(x)

    def fwd_bwd():
        xg = x.clone().requires_grad_(True)
        z = p.ops._APPNP.apply(xg, g, 3, 0.1, True)
        z.backward(dz)
        return torch.cat([z.detach(), xg.grad])

    old, new = _both(monkeypatch, fwd_bwd)
    assert torch.equal(old, new)
    old, new = _both(monkeypatch, lambda: p.ops._appnp_khop(g.fwd, g, x, 3, 0.1, False, False))
    assert torch.equal(old, new)


def test_graph_without_groups_never_builds_the_renamed_graph(monkeypatch):
    p = P()
    from rgb_experiment_b200 import graph as G
    import rgb_experiment_b200.synth as S_
    monkeypatch.setattr(G, "CLUSTER_MIN_NODES", 1000)
    sg = S_.make_graph(50_000, 1_000_000, 8, 4, seed=3, features=False, device=DEV, power_law=False, homophily=0.0)
    g = p.Graph(sg.edge_index, sg.num_nodes, p.LOOP_ADD_REMAINING)
    assert g.groups is None
    x = torch.randn(g.N, 47, device=DEV)
    p.ops._appnp_khop(g.fwd, g, x, 4, 0.1, False, True)
    p.ops.HostAppnpPlan(g, 47)
    assert g._named is None and g.named_fwd is None


def test_row_map_is_refused_where_it_does_not_apply(split_rows):
    """The map redirects the Y store only: not with a partial-sum input, reset rows or peers (rgbmp_spmm), nor with
    every hop's output kept (rgbmp_khop)."""
    p, g = P(), split_rows
    L = p._lib.lib()
    csr = g.named_fwd
    x = torch.zeros(g.N, 16, device=DEV)
    y = torch.empty_like(x)
    order = g.fwd.row_order
    st = p._lib.stream_of(x.device)
    for kw in (dict(acc_in=x, ld_acc=16), dict(reset_mask=torch.zeros(g.N, dtype=torch.uint8, device=DEV), reset_val=x,
                                                  ld_reset=16, reset_when=1)):
        ep = p.ops.make_epilogue(row_map=order, **kw)
        rc = L.rgbmp_spmm(csr.ref, None, x.data_ptr(), 16, y.data_ptr(), 16, 16, 0, C.byref(ep), 0, None, 0, 0, st)
        assert rc == p._lib.EINVAL and b"row_map" in L.rgbmp_last_error()
    ep = p.ops.make_epilogue(row_map=order)
    hops = torch.empty(2, g.N, 16, device=DEV)
    rc = L.rgbmp_khop(csr.ref, None, x.data_ptr(), 16, y.data_ptr(), y.data_ptr(), 16, y.data_ptr(), 16, hops.data_ptr(),
                      16, g.N * 16, 16, 0, 2, C.byref(ep), 0, None, 0, 0, st)
    assert rc == p._lib.EINVAL and b"row_map" in L.rgbmp_last_error()
