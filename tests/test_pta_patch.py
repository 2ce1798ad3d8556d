"""SURVEY.md 8f f4: the PTA prelude rebinding (rgb-experiment_b200/shim/pta.py).

CPU part: the handle's own rules, with the CPU oracle standing in for the kernels.
GPU part: the same call sequence on the CUDA backend against the golden vectors produced by the
reference's verbatim code (tests/golden/make_golden.py)."""
import pytest
import scipy.sparse as sp
import torch

from helpers import GOLDEN, load_golden, relerr

import rgb_experiment_b200.shim.pta as PT


class OracleBackend:
    """Test stand-in for the kernels: oracle.pyg_restated's PTA functions (itexperiments.py:671-719)."""

    @staticmethod
    def graph(edge_index, num_nodes, add_identity):
        assert add_identity
        return edge_index, num_nodes

    @staticmethod
    def label_propagation(graph, labels, idx, K, alpha):
        from oracle import pyg_restated as R
        return R.pta_label_propagation(graph[0], graph[1], labels, idx, K, alpha)

    @staticmethod
    def inference(h, graph, K, alpha):
        from oracle import pyg_restated as R
        return R.pta_inference(h, graph[0], graph[1], K, alpha)


def _identity_fns(backend):
    boom = lambda *a, **k: "original"            # noqa: E731
    return PT.make_functions(boom, boom, boom, boom, boom, backend=backend)


def test_handle_accepts_exactly_the_drivers_sequence():
    e2s, norm, conv, lp, inf = _identity_fns(OracleBackend)
    ei = torch.tensor([[0, 1, 2], [1, 2, 0]])
    adj = e2s(ei, 3)
    assert isinstance(adj, PT.PtaAdjacency) and adj.shape == (3, 3)
    with pytest.raises(RuntimeError):
        adj.to("cpu")                             # not normalised yet
    with pytest.raises(RuntimeError):
        adj + sp.eye(4)                           # wrong size
    with pytest.raises(RuntimeError):
        adj + 2 * sp.eye(3)                       # not the identity
    a1 = adj + sp.eye(adj.shape[0])
    with pytest.raises(RuntimeError):
        a1 + sp.eye(3)                            # twice
    a2 = conv(norm(a1))
    with pytest.raises(RuntimeError):
        norm(a2)
    with pytest.raises(RuntimeError):
        lp(a2, torch.tensor([0, 1, 0]), torch.tensor([0]), 2, 0.1, "cpu")   # not on its device yet
    a3 = a2.to("cpu")
    y = lp(a3, torch.tensor([0, 1, 0]), torch.tensor([0, 1]), 2, 0.1, "cpu")
    assert y.shape == (3, 2) and not adj.identity_added and a3.identity_added and a3.normalized


def test_non_handle_arguments_fall_through_to_the_reference():
    e2s, norm, conv, lp, inf = _identity_fns(OracleBackend)
    m = sp.eye(3).tocoo()
    assert norm(m) == "original" and conv(m) == "original"
    assert lp(torch.eye(3).to_sparse(), None, None, 1, 0.1, "cpu") == "original"
    assert inf(object(), torch.zeros(3, 2), torch.eye(3).to_sparse()) == "original"
    assert e2s([[0], [1]], 2) == "original"       # not a tensor


def test_default_backend_refuses_cpu_tensors():
    """The product backend has no CPU path: moving the handle to the CPU raises."""
    e2s, norm, conv, lp, inf = _identity_fns(PT._CudaBackend)
    adj = norm(e2s(torch.tensor([[0, 1], [1, 0]]), 2) + sp.eye(2))
    with pytest.raises(RuntimeError):
        adj.to("cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=lambda p: p.split("/")[-1])
def test_patched_sequence_on_cuda_matches_reference_golden(path):
    gold = load_golden(path)
    if "pta_lp" not in gold:
        pytest.skip("no PTA vectors in this fixture")
    dev = "cuda:0"
    boom = lambda *a, **k: (_ for _ in ()).throw(AssertionError("fell through"))   # noqa: E731
    e2s, norm, conv, lp, inf = PT.make_functions(boom, boom, boom, boom, boom)
    ei, n = gold["edge_index"], int(gold["num_nodes"])
    adj = e2s(ei.cpu(), n)                                   # the driver hands over a CPU edge_index (:352)
    adj = conv(norm(adj + sp.eye(adj.shape[0]))).to(dev)
    y = lp(adj, gold["pta_labels"].to(dev), gold["pta_idx"].to(dev), gold["pta_K"], gold["pta_alpha"], dev)
    assert y.is_cuda and relerr(y, gold["pta_lp"]) <= 1e-5

    class M:                                                 # PTA.inference reads only K and alpha (pta.py:79-84)
        K, alpha = gold["pta_K"], gold["pta_alpha"]

    out = inf(M(), gold["pta_h"].to(dev).requires_grad_(True), adj)
    assert not out.requires_grad and relerr(out, gold["pta_inference"]) <= 1e-5
