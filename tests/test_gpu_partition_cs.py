"""Label propagation and Correct & Smooth through the partitioned K-hop (partition.PartitionedAPPNP with the
label-propagation post-step, partition.DistCorrectAndSmooth) on one GPU, against the single-GPU ops / shim paths.

The graph is LOOP_NONE (gcn_norm(add_self_loops=False)) with nodes that receive no edge (D^-1/2 = 0), some of which
send edges, and a hub row of 3,000 edges, so that the long-row and combine kernels run.  F = 47 > 16 keeps
ops.label_propagation off the one-cluster small-graph K-hop, which orders a row's sums differently: both sides then
launch the same SpMM kernels on the same rows, and the results are compared bit for bit."""
import pytest
import torch

from helpers import CASES, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F = 47
K = 12


def P():
    import rgb_experiment_b200 as P_
    return P_


def _graph():
    """CASES['medium'] (5,000 nodes, a 3,000-edge hub row) plus 300 nodes without in-edges, 150 of which send edges."""
    ei, n = CASES["medium"]()
    g = torch.Generator().manual_seed(9)
    extra_src = torch.randint(n, n + 150, (600,), generator=g)
    extra_dst = torch.randint(n, (600,), generator=g)
    ei = torch.cat([ei, torch.stack([extra_src, extra_dst])], dim=1)
    return ei, n + 300


def _problem(n, dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    y_soft = torch.softmax(torch.randn(n, F, generator=g) * 2.0, dim=1)
    labels = torch.randint(F, (n,), generator=g)
    train = torch.rand(n, generator=g) < 0.3
    train[n - 300:] = False                                # rows without in-edges and without error: L1 = 0
    return y_soft.to(dtype).to(DEV), labels.to(DEV), train.to(DEV)


def _block(ei, n):
    import rgb_experiment_b200.partition as PT
    p = P()
    return PT.LocalBlock(ei.to(DEV), n, p.LOOP_NONE, 0, 1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("post", ["clamp", "reset"])
def test_one_block_label_propagation_is_bit_equal_to_ops(dtype, post):
    """World 1 runs the per-edge-weight form (PartitionedAPPNP's all-gather mode): ops.label_propagation(fold=False)
    launches the same SpMM per hop with the same epilogue, so the iterates agree bit for bit."""
    import rgb_experiment_b200.partition as PT
    p = P()
    ei, n = _graph()
    y_soft, labels, train = _problem(n, dtype)
    error = torch.zeros_like(y_soft)
    error[train] = torch.nn.functional.one_hot(labels[train], F).to(dtype) - y_soft[train]
    g = p.Graph(ei.to(DEV), n, p.LOOP_NONE)
    blk = _block(ei, n)
    assert blk.csr.n_items > 0                             # the long-row and combine kernels run
    alpha = 0.8
    if post == "clamp":
        want = p.ops.label_propagation(g, error, K, alpha, clamp=(-1.0, 1.0), fold=False)
        kw = dict(clamp=(-1.0, 1.0))
    else:
        want = p.ops.label_propagation(g, error, K, alpha, reset_mask=train, reset_val=error, fold=False)
        kw = dict(reset=(train, error))
    prop = PT.PartitionedAPPNP(blk, F, dtype=dtype)
    z0 = torch.zeros((blk.R, prop.ld), dtype=dtype, device=DEV)
    z0[:, :F] = error
    got = prop.run(z0, K, teleport=(alpha, 1.0 - alpha), **kw)[:n, :F]
    assert torch.equal(got, want)
    if post == "reset":
        assert torch.equal(got[train].float(), error[train].float())


@pytest.mark.parametrize("F_,dtype", [(47, torch.float32), (100, torch.float32), (128, torch.bfloat16)])
@pytest.mark.parametrize("post", ["clamp", "reset"])
def test_push_epilogue_with_clamp_and_reset_fills_every_copy_in_both_forms(F_, dtype, post):
    """The multi-GPU hop's kernel on one GPU: with the label-propagation post-step in the epilogue, every `peer_out`
    buffer (three local ones) receives rows [peer_row0, peer_row0 + n) = dinv * (the clamped or reset row), the
    16-byte and the bulk (TMA) push forms write the same bytes, and nothing outside those rows is touched."""
    p = P()
    L = p._lib.lib()
    ei, n = _graph()
    g = p.Graph(ei.to(DEV), n, p.LOOP_NONE)
    assert g.fwd.n_items > 0
    d = g.dinv()
    x = torch.randn(n, F_, generator=torch.Generator().manual_seed(F_)).to(DEV).to(dtype)
    xb, ldx = p.ops.as_rows(x)
    ld = p.ops.padded_width(F_, dtype)
    row0, tail = 3, 2
    lo, hi = -0.25, 0.25
    mask = (torch.rand(n, generator=torch.Generator().manual_seed(1)) < 0.3).to(DEV)
    rv, ldr = p.ops.as_rows(torch.randn(n, F_, generator=torch.Generator().manual_seed(2)).to(DEV))
    m8 = mask.to(torch.uint8)
    post_kw = (dict(clamp=(lo, hi)) if post == "clamp"
               else dict(clamp=(lo, hi), reset_mask=m8, reset_val=rv, ld_reset=ldr, reset_when=p.ops.RESET_AFTER_CLAMP))
    tele = dict(a=0.8, b=0.2, T=xb, ldt=ldx, **post_kw)
    y = p.ops.spmm_raw(g.fwd, x, None, ep=p.ops.make_epilogue(row_scale=d, **tele), keep=(xb, d, m8, rv))
    # the local result holds the post-step: clamped rows, and the reset rows' values (after the clamp)
    yf = y.float()
    if post == "clamp":
        assert float(yf.min()) >= lo and float(yf.max()) <= hi and float(yf.max()) == hi
    else:
        assert torch.equal(yf[mask], rv[mask].to(dtype).float())
        assert float(yf[~mask].min()) >= lo and float(yf[~mask].max()) <= hi
    want = (yf * d.view(-1, 1)).to(dtype)                 # what the next hop gathers
    got = {}
    old = L.rgbmp_set_push_bulk(1)
    try:
        for bulk in (1, 0):
            L.rgbmp_set_push_bulk(bulk)
            bufs = [torch.full((row0 + n + tail, ld), float("nan"), dtype=dtype, device=DEV) for _ in range(3)]
            ep = p.ops.make_epilogue(row_scale=d, out2_scale=d, peers=[b.data_ptr() for b in bufs], peer_row0=row0,
                                     ld_peer=ld, **tele)
            assert p.ops.spmm_raw(g.fwd, x, None, ep=ep, keep=(xb, d, m8, rv, bufs), store_local=False) is None
            torch.cuda.synchronize()
            for b in bufs:
                if dtype == torch.float32:
                    assert torch.equal(b[row0:row0 + n, :F_], want)
                else:                                     # `want` was rounded to bf16 before the scale, the kernel rounds after
                    assert relerr(b[row0:row0 + n, :F_].float(), want.float()) <= 2 ** -7
                assert torch.isnan(b[:row0].float()).all() and torch.isnan(b[row0 + n:].float()).all()
            got[bulk] = bufs
    finally:
        L.rgbmp_set_push_bulk(old)
    for a, b in zip(got[0], got[1]):
        assert torch.equal(torch.nan_to_num(a[row0:row0 + n].float(), nan=7.0), torch.nan_to_num(b[row0:row0 + n].float(), nan=7.0))


@pytest.mark.parametrize("mask_form", ["bool", "index"])
def test_dist_correct_and_smooth_on_one_gpu_matches_the_shim(mask_form, monkeypatch):
    """World 1: DistCorrectAndSmooth over PartitionedAPPNP against shim.nn.CorrectAndSmooth, both in the per-edge-weight
    form (ops.FOLD_KHOP off for the shim), so only the sums of sigma and of the row L1 norms are ordered differently."""
    import rgb_experiment_b200.partition as PT
    from rgb_experiment_b200.shim import nn as PL
    p = P()
    monkeypatch.setattr(p.ops, "FOLD_KHOP", False)
    ei, n = _graph()
    y_soft, labels, train = _problem(n, torch.float32, seed=3)
    mask = train if mask_form == "bool" else torch.nonzero(train).view(-1)
    y_true = labels[mask]
    blk = _block(ei, n)
    prop = PT.PartitionedAPPNP(blk, F)
    assert prop.ld == PT.DistCorrectAndSmooth.slice_ld(PT.Grid(0, 1), F)
    for autoscale in (True, False):
        kw = dict(num_correction_layers=50, correction_alpha=0.8, num_smoothing_layers=50, smoothing_alpha=0.8,
                  autoscale=autoscale, scale=0.7)
        ref = PL.CorrectAndSmooth(**kw)
        cs = PT.DistCorrectAndSmooth(**kw, grid=PT.Grid(0, 1), N=n, runner=prop.run)
        want = ref.correct(y_soft, y_true, mask, ei.to(DEV))
        got = cs.correct(y_soft, y_true, mask)
        assert got.shape == (n, F)
        assert relerr(got, want) <= 1e-6, (autoscale, relerr(got, want))
        want_s = ref.smooth(want, y_true, mask, ei.to(DEV))
        got_s = cs.smooth(want, torch.nn.functional.one_hot(y_true, F).float(), mask)
        assert relerr(got_s, want_s) <= 1e-6
        assert float(got_s.min()) >= 0.0 and float(got_s.max()) <= 1.0


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64])
def test_other_dtypes_raise_before_a_launch(dtype):
    import rgb_experiment_b200.partition as PT
    ei, n = _graph()
    blk = _block(ei, n)
    with pytest.raises(RuntimeError):
        PT.PartitionedAPPNP(blk, F, dtype=dtype)
    prop = PT.PartitionedAPPNP(blk, F)
    z0 = torch.zeros((blk.R, prop.ld), dtype=dtype, device=DEV)
    with pytest.raises(RuntimeError):
        prop.run(z0, 3, teleport=(0.8, 0.2), clamp=(0.0, 1.0))
    cs = PT.DistCorrectAndSmooth(3, 0.8, 3, 0.8, grid=PT.Grid(0, 1), N=n, runner=prop.run)
    y = torch.full((n, F), 1.0 / F, dtype=dtype, device=DEV)
    idx = torch.arange(4, device=DEV)
    with pytest.raises(RuntimeError):
        cs.correct(y, torch.zeros(4, dtype=torch.long, device=DEV), idx)
    with pytest.raises(RuntimeError):
        cs.smooth(y, torch.zeros(4, dtype=torch.long, device=DEV), idx)
