"""The PRODUCT shim against what the reference package asks of it, in the build container (no GPU).

The reference's ``models/__init__.py:1-13`` imports all 13 model files eagerly, so every name of the
import surface (SURVEY.md 8b, exact list with call sites) must resolve through the installed shim, and every
layer must accept the constructor calls the model files make (8b, "constructor / call signatures").  A CPU
run must fail LOUDLY (the product has no CPU path) instead of silently falling back, and the opt-in PTA
rebinding must bind and restore the five names of the reference's PTA prelude (itexperiments.py:671-719,
models/pta.py:79-84), here on stand-in modules that carry those names."""
import types

import pytest
import scipy.sparse as sp
import torch


@pytest.fixture()
def shim():
    from oracle import shim as oshim
    import rgb_experiment_b200 as R
    oshim.uninstall()
    R.install_shim()
    yield R
    R.uninstall_shim()


def test_reference_imports_and_builds_every_model_on_the_product_shim(shim):
    import torch.nn as nn
    import torch_geometric
    from torch_geometric.nn.conv import GCNConv, MessagePassing, GATConv, APPNP, SAGEConv, FAConv
    from torch_geometric.nn import SGConv, SuperGATConv, GINConv, GatedGraphConv, CorrectAndSmooth
    from torch_geometric.utils import (remove_self_loops, add_self_loops, add_remaining_self_loops,  # noqa: F401
                                       to_networkx, to_undirected)
    from torch_geometric.data import Data
    from torch_scatter import scatter_add  # noqa: F401
    from torch_sparse import coalesce  # noqa: F401
    import matplotlib  # noqa: F401
    import matplotlib.pyplot  # noqa: F401
    from matplotlib.font_manager import FontProperties  # noqa: F401
    assert getattr(torch_geometric, "__rgbmp_shim__", False)

    class MeanConv(MessagePassing):                          # graphsage.py:39-40, dagnn.py:36
        def __init__(self):
            super().__init__(aggr="mean")

    built = {
        "GCN": GCNConv(12, 8),
        "GAT": GATConv(12, 2, 4),
        "GAT out": GATConv(8, 3, 1, concat=False),
        "APPNPStack": APPNP(5, 0.1),
        "GraphSAGE2": SAGEConv(12, 8),
        "SGC": SGConv(12, 3, K=2, cached=True, add_self_loops=True),
        "FAGCN": FAConv(8, 0.3, 0.5),
        "SuperGAT": SuperGATConv(12, 2, heads=4, dropout=0.6, edge_sample_ratio=0.8, neg_sample_ratio=0.5),
        "SuperGAT out": SuperGATConv(8, 3, heads=4, concat=False, dropout=0.6, edge_sample_ratio=0.8,
                                     neg_sample_ratio=0.5),
        "GIN": GINConv(nn.Sequential(nn.Linear(12, 8), nn.ReLU(), nn.Linear(8, 8))),
        "GGNN": GatedGraphConv(16, 2),
        "GraphSAGE / DAGNN base": MeanConv(),
        "add base": MessagePassing(aggr="add"),
    }
    import rgb_experiment_b200.shim.nn as PL
    for name, layer in built.items():
        assert isinstance(layer, PL.MessagePassing), name
    for cs in (CorrectAndSmooth(50, 0.8, 50, 0.8, True), CorrectAndSmooth(50, 0.8, 50, 0.8, False, 1.0)):
        assert isinstance(cs, PL.CorrectAndSmooth)
    d = Data(x=torch.randn(5, 3), y=torch.zeros(5, dtype=torch.long), edge_index=torch.tensor([[0, 1], [1, 0]]))
    d2 = d.clone()
    assert type(d2) == Data and d2.num_nodes == 5 and d2.num_node_features == 3      # noqa: E721


def test_cpu_run_fails_loudly_not_silently(shim):
    """The first aggregation of a CPU run (the GCN model's GCNConv) raises instead of computing on the host."""
    from torch_geometric.nn.conv import GCNConv
    import rgb_experiment_b200.synth as S
    g = S.make_graph(120, 600, 8, 3, seed=1)
    conv = GCNConv(8, 4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        conv(g.x, g.edge_index)


def test_patch_pta_binds_and_restores_the_reference_names():
    from rgb_experiment_b200.shim.pta import PtaAdjacency, patch

    def fell_through(*a, **k):
        raise AssertionError("the reference's original was called for a handle")

    class PTA:
        inference = fell_through

    it = types.ModuleType("rgb_experiment.itexperiments")
    it.edge_index2sparse_matrix = it.normalize_adj = it.sparse_mx_to_torch_sparse_tensor = fell_through
    it.label_propagation = fell_through
    pm = types.ModuleType("rgb_experiment.models.pta")
    pm.PTA = PTA
    orig = (it.edge_index2sparse_matrix, it.normalize_adj, it.label_propagation, pm.PTA.inference)
    restore = patch(it, pm)
    try:
        assert patch(it, pm) is restore                       # idempotent
        h = it.edge_index2sparse_matrix(torch.tensor([[0, 1], [1, 0]]), 2)
        assert isinstance(h, PtaAdjacency)
        h = it.sparse_mx_to_torch_sparse_tensor(it.normalize_adj(h + sp.eye(2)))
        with pytest.raises(RuntimeError, match="CUDA"):       # product backend: no CPU path
            h.to("cpu")
    finally:
        restore()
    assert (it.edge_index2sparse_matrix, it.normalize_adj, it.label_propagation, pm.PTA.inference) == orig
