"""SuperGAT's self-supervised attention loss on the device (csrc/supergat_loss.cu, ops.supergat_att_loss):
the device keep mask and negatives equal the numpy restatement (supergat_sampling_ref) bit for bit; negatives avoid
U and follow the seed; the fused loss and dx' match an fp64 restatement of BCE(att_x.mean(-1)); the shim layer with
ops.FUSED_SUPERGAT_LOSS matches the oracle layer; repeat calls are bit-identical; nothing edge-sized is allocated;
guard bands."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import supergat_sampling_ref as SR
from helpers import CASES, random_graph, relerr
from oracle import layers as OL

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def P():
    import rgb_experiment_b200 as P_
    return P_


def _graph(case, loop=None):
    p = P()
    if case == "dense":                          # density 0.75, alpha ~ 6
        ei, n = random_graph(12, 90, 5), 12
    elif case == "saturated":                    # K20 minus one pair: three rounds return fewer than num_neg
        n = 20
        pairs = [(i, j) for i in range(n) for j in range(n) if (i, j) not in ((3, 7), (7, 3))]
        ei = torch.tensor(pairs).t().contiguous()
    elif case == "near_complete":                # K36 minus 18 pairs, density 0.97: alpha ~ 14, a round keeps ~ 2/5 num_neg
        n = 36
        pairs = [(i, j) for i in range(n) for j in range(n) if i // 2 != j // 2 or i == j]
        ei = torch.tensor(pairs).t().contiguous()
    elif case == "selfloops":
        ei, n = random_graph(40, 100, 6, self_loops=80), 40
    else:
        ei, n = CASES[case]()
    return p.Graph(ei.to(DEV), n, p.LOOP_REMOVE_THEN_ADD if loop is None else loop), ei, n


def _seed(v):
    return torch.tensor([v], dtype=torch.int64, device=DEV)


def _u_keys(g, undirected_input):
    src, dst = g.e_src.long().cpu().numpy(), g.e_dst.long().cpu().numpy()
    return SR.undirected_keys(src, dst, g.N, symmetrize=not undirected_input)


def _ref_negatives(g, seed, ratio_e, ratio_n, is_undirected):
    keys = _u_keys(g, is_undirected)
    E_u = g.nnz if is_undirected else keys.size
    num_neg, S = SR.neg_counts(g.N, E_u, int(ratio_n * ratio_e * g.nnz))
    return SR.negatives(seed, g.N, keys, num_neg, S), num_neg


# ------------------------------------------------------------------------------------------
# 1. sampler and keep mask vs numpy
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["dense", "near_complete", "loops_dups", "hub", "medium", "saturated"])
@pytest.mark.parametrize("is_undirected", [False, True])
@pytest.mark.parametrize("ratio_e,ratio_n", [(1.0, 0.5), (0.6, 1.5)])
def test_samples_equal_numpy_restatement(case, is_undirected, ratio_e, ratio_n):
    g, _, _ = _graph(case)
    seed = 0x1234567 + g.N
    if case == "saturated":                      # a seed whose three rounds find fewer than num_neg survivors
        seed = next(v for v in range(seed, seed + 200)
                    if _ref_negatives(g, v, ratio_e, ratio_n, is_undirected)[0][0].size
                    < _ref_negatives(g, v, ratio_e, ratio_n, is_undirected)[1])
    s = P().ops.supergat_samples(g, ratio_e, ratio_n, is_undirected, seed=_seed(seed), mask=True)
    (row, col, rounds), num_neg = _ref_negatives(g, seed, ratio_e, ratio_n, is_undirected)
    assert s.neg_edge_index.dtype == torch.int64
    assert np.array_equal(s.neg_edge_index[0].cpu().numpy(), row)
    assert np.array_equal(s.neg_edge_index[1].cpu().numpy(), col)
    assert np.array_equal(s.keep_mask.cpu().numpy(), SR.keep_mask(seed, g.nnz, ratio_e))
    assert s.keep_thresh == SR.keep_thresh(ratio_e)
    if case == "saturated":
        assert rounds == 3 and row.size < num_neg


def test_sampler_fills_num_neg_in_the_third_round():
    """A round's expected survivors are num_neg (1 - d) / |1 - 1.1 d| for density d = E_u / N^2: above num_neg below
    d = 1/1.1, so there the first round nearly always fills.  On a near-complete graph a round keeps ~2/5 of num_neg and
    the third round completes it; most seeds show it (checked in numpy first, then on the device)."""
    g, _, _ = _graph("near_complete")
    keys = _u_keys(g, False)
    num_neg, S = SR.neg_counts(g.N, keys.size, int(1.0 * g.nnz))
    assert 10.0 < S / num_neg < 20.0                    # alpha of the near-complete graph
    seed = next(v for v in range(100) if SR.negatives(v, g.N, keys, num_neg, S)[2] == 3
                and SR.negatives(v, g.N, keys, num_neg, S)[0].size == num_neg)
    row, col, _ = SR.negatives(seed, g.N, keys, num_neg, S)
    s = P().ops.supergat_samples(g, 1.0, 1.0, False, seed=_seed(seed))
    assert torch.equal(s.neg_edge_index.cpu(), torch.from_numpy(np.stack([row, col])))


def test_no_negatives_when_num_neg_is_not_positive():
    g, _, _ = _graph("saturated")
    s = P().ops.supergat_samples(g, 1.0, 0.0, False, seed=_seed(3))
    assert s.neg_edge_index.shape == (2, 0)
    full = P().Graph(torch.tensor([[i for i in range(4) for _ in range(4)], list(range(4)) * 4]).to(DEV), 4,
                     P().LOOP_NONE)                   # every pair: size - E_u = 0
    assert P().ops.supergat_samples(full, 1.0, 0.5, False, seed=_seed(3)).neg_edge_index.shape == (2, 0)


# ------------------------------------------------------------------------------------------
# 2. negatives avoid U; seeding
# ------------------------------------------------------------------------------------------
def test_negatives_avoid_u_and_follow_the_seed():
    ops = P().ops
    g, _, _ = _graph("medium")
    keys = torch.from_numpy(_u_keys(g, False)).to(DEV)
    torch.manual_seed(77)
    a = ops.supergat_samples(g, 0.8, 0.5, False)
    b = ops.supergat_samples(g, 0.8, 0.5, False)
    torch.manual_seed(77)
    c = ops.supergat_samples(g, 0.8, 0.5, False)
    neg = a.neg_edge_index
    assert neg.size(1) == int(0.5 * 0.8 * g.nnz)
    assert not torch.isin(neg[0] * g.N + neg[1], keys).any()
    assert torch.equal(a.seed, c.seed) and torch.equal(a.neg_edge_index, c.neg_edge_index)
    assert not torch.equal(a.neg_edge_index, b.neg_edge_index)
    d = ops.supergat_samples(g, 0.8, 0.5, False, generator=torch.Generator(device=DEV).manual_seed(5))
    e = ops.supergat_samples(g, 0.8, 0.5, False, generator=torch.Generator(device=DEV).manual_seed(5))
    assert torch.equal(d.neg_edge_index, e.neg_edge_index)


# ------------------------------------------------------------------------------------------
# 3. loss and dx' vs fp64 with the samples fixed
# ------------------------------------------------------------------------------------------
def _ref_loss(x64, pos, neg, scale):
    xi = torch.cat([x64[pos[1]], x64[neg[1]]])
    xj = torch.cat([x64[pos[0]], x64[neg[0]]])
    s = scale * (xi * xj).sum(-1)
    y = torch.zeros_like(s)
    y[:pos.size(1)] = 1.0
    return F.binary_cross_entropy_with_logits(s, y)


@pytest.mark.parametrize("case", ["loops_dups", "hub", "selfloops"])
@pytest.mark.parametrize("H,C", [(8, 8), (8, 41), (1, 7), (4, 4), (3, 5), (2, 16)])
@pytest.mark.parametrize("mode", ["MX", "SD"])
def test_loss_and_grad_match_fp64(case, H, C, mode):
    ops = P().ops
    g, _, n = _graph(case)
    gen = torch.Generator().manual_seed(H * 100 + C)
    x = torch.randn(n, H * C, generator=gen) * 0.4
    neg = torch.randint(n, (2, 3 * n), generator=gen)
    neg[:, :5] = torch.arange(5).repeat(2, 1)             # self pairs among the negatives too
    scale = 1.0 / H if mode == "MX" else 1.0 / (H * math.sqrt(C))
    xg = x.to(DEV).requires_grad_(True)
    loss = ops.supergat_att_loss(xg, g, H, C, scale, 0.7, 0.5, False, neg.to(DEV),
                                 generator=torch.Generator(device=DEV).manual_seed(9))
    loss.backward()
    seed = ops.dropout_seed(DEV, torch.Generator(device=DEV).manual_seed(9))
    keep = ops.supergat_samples(g, 0.7, 0.0, False, seed=seed, mask=True).keep_mask.cpu()
    pos = g.edge_index().cpu()[:, keep]
    x64 = x.double().requires_grad_(True)
    ref = _ref_loss(x64, pos, neg, scale)
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert relerr(xg.grad, x64.grad) <= 2e-5


def test_unsupported_inputs_raise():
    ops = P().ops
    g, _, n = _graph("loops_dups")
    x = torch.randn(n, 64, device=DEV)
    with pytest.raises(RuntimeError, match="outside"):
        ops.supergat_att_loss(x, g, 8, 8, 0.125, 1.0, 0.5, False, torch.tensor([[0, n], [1, 2]], device=DEV))
    with pytest.raises(RuntimeError, match="outside"):
        ops.supergat_att_loss(x, g, 8, 8, 0.125, 1.0, 0.5, False, torch.tensor([[0, -1], [1, 2]], device=DEV))
    with pytest.raises(RuntimeError, match="float32"):
        ops.supergat_att_loss(x.double(), g, 8, 8, 0.125)
    with pytest.raises(RuntimeError, match="argument error"):
        ops.supergat_att_loss(torch.randn(n, 520, device=DEV), g, 8, 65, 0.125)
    with pytest.raises(ValueError):
        ops.supergat_att_loss(x, g, 8, 8, 0.125, 1.5)


# ------------------------------------------------------------------------------------------
# 4. the shim layer
# ------------------------------------------------------------------------------------------
def _layers(kw, seed=0):
    import importlib
    PL = importlib.import_module("rgb_experiment_b200.shim.nn")
    torch.manual_seed(seed)
    o = OL.SuperGATConv(12, 8, **kw).double()
    torch.manual_seed(seed)
    g = PL.SuperGATConv(12, 8, **kw)
    g.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    return o.train(), g.to(DEV).train()


@pytest.fixture
def fused_switch():
    ops = P().ops
    old = ops.FUSED_SUPERGAT_LOSS
    ops.FUSED_SUPERGAT_LOSS = True
    yield
    ops.FUSED_SUPERGAT_LOSS = old


@pytest.mark.parametrize("att", ["MX", "SD"])
def test_layer_matches_oracle_with_fixed_samples(fused_switch, att):
    ei, n = CASES["loops_dups"]()
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(n, 12, generator=gen)
    neg = torch.randint(n, (2, 150), generator=gen)
    o, g = _layers({"heads": 4, "dropout": 0.0, "edge_sample_ratio": 1.0, "neg_sample_ratio": 0.5,
                    "attention_type": att})
    xo, xg = x.double().requires_grad_(True), x.to(DEV).requires_grad_(True)
    yo, yg = o(xo, ei, neg), g(xg, ei.to(DEV), neg.to(DEV))
    assert g.att_x is None and g.att_y is None
    lo_, lg_ = yo.pow(2).sum() + 4.0 * o.get_attention_loss(), yg.pow(2).sum() + 4.0 * g.get_attention_loss()
    lo_.backward()
    lg_.backward()
    assert relerr(yg.detach(), yo.detach()) <= 1e-5
    assert abs(float(lg_) - float(lo_)) <= 1e-4 * abs(float(lo_))
    assert relerr(xg.grad, xo.grad) <= 3e-5
    po, pg = dict(o.named_parameters()), dict(g.named_parameters())
    for k in po:
        assert relerr(pg[k].grad, po[k].grad) <= 5e-5, k


def test_layer_with_sampling_equals_torch_formula_on_the_same_samples(fused_switch):
    p = P()
    ei, n = CASES["medium"]()
    x = torch.randn(n, 12, generator=torch.Generator().manual_seed(3)).to(DEV)
    _, layer = _layers({"heads": 4, "edge_sample_ratio": 0.8, "neg_sample_ratio": 0.5})
    eid = ei.to(DEV)
    torch.manual_seed(21)
    layer(x, eid)
    fused = layer.get_attention_loss()
    torch.manual_seed(21)
    seed = p.ops.dropout_seed(DEV)                     # the layer's first draw: dropout is 0
    g = p.get_graph(eid, n, p.LOOP_REMOVE_THEN_ADD)
    s = p.ops.supergat_samples(g, 0.8, 0.5, False, seed=seed, mask=True)
    with torch.no_grad():
        x3 = layer.lin(x).view(n, 4, 8).double()
        pos = g.edge_index()[:, s.keep_mask]
        neg = s.neg_edge_index
        att = torch.cat([(x3[pos[1]] * x3[pos[0]]).sum(-1), (x3[neg[1]] * x3[neg[0]]).sum(-1)])
        y = torch.zeros(att.size(0), dtype=torch.float64, device=DEV)
        y[:pos.size(1)] = 1.0
        want = F.binary_cross_entropy_with_logits(att.mean(-1), y)
    assert abs(float(fused) - float(want)) <= 1e-4 * abs(float(want))


def test_switch_off_and_eval_keep_the_torch_path():
    ei, n = CASES["loops_dups"]()
    _, layer = _layers({"heads": 2})
    assert P().ops.FUSED_SUPERGAT_LOSS is False
    layer(torch.randn(n, 12, device=DEV), ei.to(DEV))
    assert layer.att_x is not None and layer._att_loss is None
    layer.eval()
    assert float(layer.get_attention_loss()) == 0.0


# ------------------------------------------------------------------------------------------
# 5. bit-reproducible
# ------------------------------------------------------------------------------------------
def test_repeat_calls_are_bit_identical():
    ops = P().ops
    g, _, n = _graph("hub")
    x = torch.randn(n, 8 * 41, device=DEV)
    outs = []
    for _ in range(2):
        xg = x.clone().requires_grad_(True)
        loss = ops.supergat_att_loss(xg, g, 8, 41, 1 / 8, 0.7, 0.5, False,
                                     generator=torch.Generator(device=DEV).manual_seed(4))
        loss.backward()
        outs.append((loss.detach(), xg.grad))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# ------------------------------------------------------------------------------------------
# 6. memory: nothing edge-sized
# ------------------------------------------------------------------------------------------
def test_training_step_allocates_nothing_edge_sized():
    p = P()
    import rgb_experiment_b200.synth as S
    sg = S.make_graph(20_000, 4_000_000, 8, 4, features=False, device=DEV)
    N, H, C = sg.num_nodes, 8, 8
    Fw = H * C
    g = p.Graph(sg.edge_index, N, p.LOOP_REMOVE_THEN_ADD)
    _ = g.bwd, g.undirected_csr(True)                  # built once per graph and held on it, like the transpose CSR
    x = torch.randn(N, Fw, device=DEV).requires_grad_(True)
    num_neg = int(0.5 * g.nnz)
    _, Ssz = p.ops.supergat_neg_counts(N, g.undirected_csr(True)[1].numel(), num_neg)
    torch.cuda.synchronize()
    start = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    loss = p.ops.supergat_att_loss(x, g, H, C, 1 / H)
    loss.backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - start
    mib = 1 << 20
    # node-sized: dX and the loss workspace; the negatives: int32 (src, dst) plus two CSRs (rowptr, col, eid) and
    # the CSR build's workspace; the sampler's workspace: one flag byte and 4/256 bytes of block counts per candidate;
    # 16 MiB for allocator rounding
    csr_ws = p._lib.lib().rgbmp_csr_build_workspace_bytes(num_neg, N)
    bound = (4 * N * Fw + 8 * N + 2 * 4 * num_neg + 2 * (8 * (N + 1) + 8 * num_neg) + csr_ws + Ssz + Ssz // 64
             + 16 * mib)
    edge_tensor = g.nnz * H * C * 4                      # one [nnz, H, C] gather
    assert peak <= bound, (peak, bound)
    assert bound < edge_tensor / 4
    # the torch formula on the same graph keeps [pairs, H, C] gathers alive
    del loss
    x.grad = None
    torch.cuda.synchronize()
    start = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    from rgb_experiment_b200.shim import utils as U
    ei = g.edge_index()
    neg = U.negative_sampling(U.to_undirected(ei, N), N, num_neg)
    x3 = x.view(N, H, C)
    att = torch.cat([(x3[ei[1]] * x3[ei[0]]).sum(-1), (x3[neg[1]] * x3[neg[0]]).sum(-1)])
    y = torch.zeros(att.size(0), device=DEV)
    y[:ei.size(1)] = 1.0
    F.binary_cross_entropy_with_logits(att.mean(-1), y).backward()
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - start > bound


# ------------------------------------------------------------------------------------------
# 7. guard bands
# ------------------------------------------------------------------------------------------
def test_supergat_loss_entry_points_under_guard_bands():
    from test_gpu_guard_bands import GuardedAllocator
    p = P()
    p.graph.clear_cache()
    p.memo.clear()
    ga = GuardedAllocator()
    ga.install()
    try:
        for case, H, C in (("loops_dups", 3, 5), ("hub", 8, 41), ("dense", 2, 16), ("saturated", 1, 7)):
            g, _, n = _graph(case)
            s = p.ops.supergat_samples(g, 0.6, 1.5, False, seed=_seed(n), mask=True)
            assert s.keep_mask.numel() == g.nnz
            neg = s.neg_edge_index
            assert neg.numel() == 0 or (int(neg.min()) >= 0 and int(neg.max()) < n)
            x = torch.randn(n, H * C, device=DEV).requires_grad_(True)
            loss = p.ops.supergat_att_loss(x, g, H, C, 1.0 / H, 0.6, 1.5, False)
            loss.backward()
            assert torch.isfinite(loss) and torch.isfinite(x.grad).all(), case
        torch.cuda.synchronize()
    finally:
        ga.uninstall()
    assert len(ga.records) > 20
    assert ga.violations() == 0
