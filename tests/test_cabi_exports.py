"""CPU-side checks of the drop-in boundary: librgbmp.so loads and exports every symbol that
include/rgbmp.h declares; argument errors are reported through the return code / last_error
without touching a GPU; the product package refuses CPU tensors."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rgbmp.h")
LIB = os.path.join(ROOT, "rgb-experiment_b200", "librgbmp.so")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rgbmp_[a-z0-9_]+)\s*\(", src)))


def test_library_is_built():
    assert os.path.exists(LIB), "run `python rgb-experiment_b200/build.py` (or __graft_entry__.build())"


def test_every_declared_symbol_is_exported():
    lib = ctypes.CDLL(LIB)
    names = declared_symbols()
    assert len(names) >= 25
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_binding_loads_and_version_is_101():
    import rgb_experiment_b200 as R
    L = R._lib.lib()
    assert L.rgbmp_version() == 101
    for n in declared_symbols():
        assert getattr(L, n).argtypes is not None or n in ("rgbmp_version", "rgbmp_last_error"), n


def test_argument_errors_do_not_need_a_gpu():
    import rgb_experiment_b200 as R
    L = R._lib.lib()
    rc = L.rgbmp_edge_edit(None, None, 5, 3, 0, None, None, None, None, 0, 0, None)
    assert rc == R._lib.EINVAL
    assert b"rgbmp_edge_edit" in L.rgbmp_last_error()
    rc = L.rgbmp_spmm(None, None, None, 0, None, 0, 4, 0, None, 0, None, 0, 0, None)
    assert rc == R._lib.EINVAL
    with pytest.raises(RuntimeError):
        R._lib.check(rc, "spmm")
    assert L.rgbmp_csr_build_workspace_bytes(1000, 10) > 0


def test_product_path_has_no_cpu_fallback():
    import rgb_experiment_b200 as R
    ei = torch.tensor([[0, 1], [1, 0]])
    with pytest.raises(RuntimeError, match="CUDA"):
        R.get_graph(ei, 2, R.LOOP_NONE)
    with pytest.raises(RuntimeError, match="CUDA"):
        R.ops.as_rows(torch.zeros(3, 4))
    src = open(os.path.join(ROOT, "rgb-experiment_b200", "ops.py")).read() + \
        open(os.path.join(ROOT, "rgb-experiment_b200", "graph.py")).read()
    assert "oracle" not in src                      # the product never imports the checker
    pkg = os.path.join(ROOT, "rgb-experiment_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", text, flags=re.M), os.path.join(dirpath, f)


def test_shim_exposes_every_name_the_reference_imports():
    """SURVEY.md 8b import list."""
    import sys
    import rgb_experiment_b200 as R
    mods = R.install_shim()
    try:
        need = {
            "torch_geometric.nn.conv": ["GCNConv", "MessagePassing", "GATConv", "APPNP", "SAGEConv", "FAConv"],
            "torch_geometric.nn": ["SGConv", "SuperGATConv", "GINConv", "GatedGraphConv", "CorrectAndSmooth"],
            "torch_geometric.utils": ["remove_self_loops", "add_self_loops", "add_remaining_self_loops",
                                      "to_networkx", "to_undirected"],
            "torch_geometric.data": ["Data"],
            "torch_scatter": ["scatter_add"],
            "torch_sparse": ["coalesce"],
        }
        for m, names in need.items():
            for n in names:
                assert hasattr(sys.modules[m], n), (m, n)
    finally:
        R.uninstall_shim()
    assert "torch_geometric" not in sys.modules or not getattr(sys.modules["torch_geometric"], "__rgbmp_shim__", False)


def test_oracle_and_product_layers_create_identical_parameters():
    """Same seed -> same state_dict, so accuracy parity runs start from identical weights."""
    from oracle import layers as OL
    import importlib
    PL = importlib.import_module("rgb_experiment_b200.shim.nn")
    specs = [("GCNConv", (12, 5), {}), ("SAGEConv", (12, 5), {}), ("GATConv", (12, 4), {"heads": 3}),
             ("GATConv", (12, 4), {"heads": 1, "concat": False}),
             ("SuperGATConv", (12, 4), {"heads": 2, "dropout": 0.1, "edge_sample_ratio": 0.8, "neg_sample_ratio": 0.5}),
             ("SGConv", (12, 5), {"K": 2, "cached": True}), ("FAConv", (8, 0.3, 0.5), {}),
             ("GatedGraphConv", (8, 2), {}), ("APPNP", (10, 0.1), {})]
    for name, args, kw in specs:
        torch.manual_seed(5)
        a = getattr(OL, name)(*args, **kw)
        torch.manual_seed(5)
        b = getattr(PL, name)(*args, **kw)
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa.keys()) == list(sb.keys()), name
        for k in sa:
            assert torch.equal(sa[k], sb[k]), (name, k)
