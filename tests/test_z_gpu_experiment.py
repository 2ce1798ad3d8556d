"""Two behaviours of the product layers that the reference's models rely on (SURVEY.md 8c K5): the SGConv
feature cache across ``load_state_dict`` and an in-place add on a ``propagate`` result.  The file is named
test_z_* so that it runs after the kernel-level parity tests.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import experiment_cases as EC  # noqa: E402

pytestmark = pytest.mark.gpu


def test_sgconv_cache_survives_load_state_dict_and_stays_out_of_it():
    """itexperiments.py:507 reloads the best weights into the SAME module; SGConv(cached=True) keeps its
    propagated features across that (sgc.py:7) and must not leak them into state_dict.  Checked on the
    product's SGConv itself, the layer the reference's SGC model wraps."""
    import rgb_experiment_b200.shim.nn as SN
    x, y, ei = EC.make_data("mid")
    dev = "cuda:0"
    torch.manual_seed(0)
    m = SN.SGConv(x.size(1), int(y.max()) + 1, K=2, cached=True).to(dev)
    m.eval()
    xd, eid = x.to(dev), ei.to(dev)
    with torch.no_grad():
        o1 = m(xd, eid)
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        assert all("cached" not in k for k in sd)
        m.load_state_dict(sd)
        o2 = m(xd, eid)
    assert torch.equal(o1, o2)


def test_in_place_add_on_propagate_output_is_legal():
    """models/graphsage.py:60 does ``out += x_r`` on the tensor an autograd.Function returned (SURVEY B8).
    The layer below has that shape: the self-loop edit, mean aggregation of lin_l(x) through the product's
    MessagePassing, then the root term added in place."""
    import torch.nn as nn
    import rgb_experiment_b200.shim.nn as SN
    import rgb_experiment_b200.shim.utils as SU

    class SageLike(SN.MessagePassing):
        def __init__(self, fin, fout):
            super().__init__(aggr="mean")
            self.lin_l, self.lin_r = nn.Linear(fin, fout), nn.Linear(fin, fout)

        def forward(self, x, edge_index):
            edge_index, _ = SU.remove_self_loops(edge_index)
            edge_index, _ = SU.add_self_loops(edge_index, num_nodes=x.size(0))
            out = self.propagate(edge_index, x=self.lin_l(x))
            x_r = self.lin_r(x)
            out += x_r
            return out

    x, y, ei = EC.make_data("mid")
    dev = "cuda:0"
    for width in (16, 10):                 # 10: rows padded to 12 floats -- the propagate result must still not be a view
        conv = SageLike(x.size(1), width).to(dev)
        xd = x.to(dev).requires_grad_(True)
        out = conv(xd, ei.to(dev))
        out.sum().backward()
        assert torch.isfinite(xd.grad).all() and xd.grad.abs().sum() > 0
