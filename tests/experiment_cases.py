"""Shared definition of the end-to-end ``experiment()`` parity cases (SURVEY.md 8c K5).

Used by ``tests/golden/make_experiment_golden.py``, which runs the UNMODIFIED reference driver on the CPU
oracle shim and records the accuracies as ``tests/golden/experiment_acc.json`` (it needs the original
package, which this repository does not contain); ``tests/test_z_gpu_experiment.py`` takes its graphs
from ``make_data``.

The stochastic forwards of the reference (dropout inside DAGNN / FAGCN / GIN / SuperGAT, SuperGAT's
edge sampling; SURVEY Appendix B5) draw from different RNG streams on CPU and CUDA, so those cases
run with the dropout probabilities at 0 and the SuperGAT attention loss weighted by 0 -- every case
is then a deterministic function of the seeded initial weights and accuracies are comparable to
0.5 pt.  ``need_to_reappear=True`` seeds the model init (itexperiments.py:305-310).
"""
import os

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_JSON = os.path.join(ROOT, "tests", "golden", "experiment_acc.json")


def make_data(shape: str):
    """(x, y, edge_index) on the CPU.  Features carry a WEAK class signal (x = 0.25*M[y] + N(0,1)) so that
    a model without aggregation stays far from 100 % and the neighbourhood aggregation decides the score."""
    import rgb_experiment_b200.synth as S
    if shape == "mid":
        n, e, f, c, seed = 20_000, 300_000, 64, 10, 5
    elif shape == "arxiv":
        n, e, f, c = S.SHAPES["arxiv"]
        seed = 20261018
    else:
        raise KeyError(shape)
    sg = S.make_graph(n, e, f, c, seed=seed, features=False)
    g = torch.Generator().manual_seed(1234 + n)
    M = torch.randn(c, f, generator=g)
    x = torch.randn(n, f, generator=g) + 0.25 * M[sg.y]
    return x, sg.y, sg.edge_index


COMMON = dict(specify_data=True, need_to_reappear=True, print_print=False, learning_rate=0.01, epoch=40)

# name -> (shape, model_name, model_init_param, extra experiment() kwargs)
CASES = {
    "mlp": ("mid", "mlp", {"num_layers": 3, "hidden_unit": 64, "dropout_rate": 0.5}, {}),
    "gcn": ("mid", "gcn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5}, {}),
    "graphsage": ("mid", "graphsage", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5}, {}),
    "graphsage2": ("mid", "graphsage2", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5}, {}),
    "gat": ("mid", "gat", {"num_layers": 2, "hidden_unit": 8, "dropout_rate": 0.5, "heads": 8}, {}),
    "ggnn": ("mid", "ggnn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5}, {}),
    "appnpstack": ("mid", "appnpstack", {"hidden_unit": 64, "dropout_rate": 0.5, "alpha": 0.1, "K": 10}, {}),
    "sgc": ("mid", "sgc", {"K": 2}, {}),
    "dagnn": ("mid", "dagnn", {"hidden_dim": 64, "K": 10, "dropout_rate": 0.0}, {}),
    "gin": ("mid", "gin", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.0}, {}),
    "fagcn": ("mid", "fagcn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.0, "epsilon": 0.3}, {}),
    "supergat": ("mid", "supergat", {"hidden_dim": 8, "heads": 8, "dropout_rate": 0.0, "edge_sample_ratio": 1.0,
                                     "neg_sample_ratio": 0.5}, {"supergat_graph_lambda": 0.0}),
    "gcn_cs": ("mid", "gcn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5},
               {"post_cs": True, "cs_param": {"num_correction_layers": 50, "correction_alpha": 0.8,
                                              "num_smoothing_layers": 50, "smoothing_alpha": 0.8, "autoscale": True}}),
    "mlp_cs_fixed_scale": ("mid", "mlp", {"num_layers": 3, "hidden_unit": 64, "dropout_rate": 0.0},
                           {"post_cs": True, "cs_param": {"num_correction_layers": 50, "correction_alpha": 0.8,
                                                          "num_smoothing_layers": 50, "smoothing_alpha": 0.8,
                                                          "autoscale": False, "scale": 1.0}}),
    "pta": ("mid", "pta", {"nhid": 64, "dropout": 0, "epsilon": 100, "mode": 2, "K": 10, "alpha": 0.1}, {}),
    "gcn_undirected": ("mid", "gcn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5},
                       {"to_undirected_graph": True}),
    # BASELINE.json configs[1]: GraphSAGE (MessagePassing mean aggregation, 3 layers, hidden 256), arxiv-shaped
    "arxiv_graphsage": ("arxiv", "graphsage", {"num_layers": 3, "hidden_unit": 256, "dropout_rate": 0.5}, {"epoch": 15}),
    "arxiv_gcn": ("arxiv", "gcn", {"num_layers": 2, "hidden_unit": 64, "dropout_rate": 0.5}, {"epoch": 20}),
    "arxiv_appnpstack": ("arxiv", "appnpstack", {"hidden_unit": 64, "dropout_rate": 0.5, "alpha": 0.1, "K": 10},
                         {"epoch": 20}),
}


def run_case(rgb, Data, name: str, device_kwargs: dict, data_cache: dict):
    """Call the reference's experiment() for one case; returns its result dict."""
    shape, model_name, params, extra = CASES[name]
    if shape not in data_cache:
        data_cache[shape] = make_data(shape)
    x, y, ei = data_cache[shape]
    kw = dict(COMMON)
    kw.update(extra)
    kw.update(device_kwargs)
    return rgb.experiment(dict(params), model_name=model_name, data=Data(x=x, y=y, edge_index=ei), **kw)
