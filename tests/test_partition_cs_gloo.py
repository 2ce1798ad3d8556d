"""Correct & Smooth on a row partition, on CPU under gloo: the partitioned label-propagation driver and
partition.DistCorrectAndSmooth, with the CPU oracle standing in for the SpMM kernel (as in test_partition_gloo.py).

The graph has N not divisible by the world size, nodes without in-edges (D^-1/2 = 0 on the LOOP_NONE graph, and
rows whose smoothed error is exactly zero: the autoscale rule's inf -> 1 case) and a training mask that lies in the
first row block only, so the ranks of the second block have none.  On a pure row partition every label-propagation
iterate equals the single-process oracle bit for bit; correct / smooth agree with the oracle's cs_correct / cs_smooth
to 1e-6 norm-wise -- sigma and the row L1 norms are summed in another order."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N, F, K, ALPHA = 103, 10, 6, 0.8
N_SINKLESS = 9                 # nodes N-9 .. N-1 receive no edge


def _problem():
    g = torch.Generator().manual_seed(0)
    src = torch.randint(N, (1100,), generator=g)
    dst = torch.randint(N - N_SINKLESS, (1100,), generator=g)
    ei = torch.stack([src, dst])
    y_soft = torch.softmax(torch.randn(N, F, generator=g) * 2.0, dim=1)
    labels = torch.randint(F, (N,), generator=g)
    train = torch.zeros(N, dtype=torch.bool)
    train[torch.randperm(40, generator=g)[:15]] = True   # inside the first row block at 2 and 4 ranks
    return ei, y_soft, labels, train


def _setup(rank, world, port):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _stand_in(grid, ed, w):
    """The oracle's gather -> scale -> scatter over my row block, then the hop's teleport and post-step."""
    import rgb_experiment_b200.partition as PT
    Rr = PT.rows_per_rank(N, grid.Pr)
    lo, hi = PT.row_range(N, grid.rp, grid.Pr)
    key, src = PT.local_edges(ed[0], ed[1], lo, hi)
    wl = w[(ed[1] >= lo) & (ed[1] < hi)]

    def spmm(x_full, z0_local, a, b, clamp=None, reset=None):
        out = torch.zeros(Rr, x_full.size(1)).index_add_(0, key.long(), wl.view(-1, 1) * x_full[src.long()])
        out = out * a + b * z0_local
        if clamp is not None:
            out.clamp_(*clamp)
        if reset is not None:
            m = reset[0].bool()
            out[m] = reset[1][m, : out.size(1)].float()
        return out

    drv = PT.PartitionedPropagator(N, grid.rp, grid.Pr, spmm, group=grid.row_group)

    def runner(z0, K_, alpha=0.0, *, teleport=None, clamp=None, reset=None):
        a, b = (1.0 - alpha, alpha) if teleport is None else teleport
        return drv.run(z0, K_, a, b, clamp=clamp, reset=reset)

    return drv, runner, Rr, lo, hi


def _local(t, lo, hi, Rr):
    out = torch.zeros((Rr,) + tuple(t.shape[1:]), dtype=t.dtype)
    out[: hi - lo] = t[lo:hi]
    return out


def _relerr(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


def _worker(rank, world, Pf, port, ret):
    _setup(rank, world, port)
    try:
        import rgb_experiment_b200.partition as PT
        from oracle import pyg_restated as R
        ei, y_soft, labels, train = _problem()
        ed, w = R.gcn_norm(ei, None, N, add_self_loops=False, dtype=torch.float32)
        grid = PT.Grid(rank, world, Pf)
        drv, runner, Rr, lo, hi = _stand_in(grid, ed, w)
        checks = {}
        error = torch.zeros(N, F)
        error[train] = torch.nn.functional.one_hot(labels[train], F).float() - y_soft[train]
        # the autoscale rule's inf -> 1 case is exercised: some real rows' smoothed error is exactly zero
        smoothed = R.lp_propagate(error, ei, K, ALPHA, post_step=lambda x: x.clamp_(-1.0, 1.0))
        checks["zero_error_rows"] = bool((smoothed.abs().sum(1) == 0).any())

        # label-propagation iterates on a pure row partition: bit-equal to the oracle, for clamp and for reset
        if Pf == 1:
            e_loc, m_loc = _local(error, lo, hi, Rr), _local(train, lo, hi, Rr)
            for name, kw, post in (
                    ("lp_clamp", dict(clamp=(-1.0, 1.0)), lambda x: x.clamp_(-1.0, 1.0)),
                    ("lp_reset", dict(reset=(m_loc, e_loc)), None)):
                if post is None:
                    def post(x):
                        x[train] = error[train]
                        return x
                got = drv.run(e_loc, K, ALPHA, 1.0 - ALPHA, **kw)
                full = torch.empty(Rr * world, F)
                dist.all_gather_into_tensor(full, got.contiguous())
                want = R.lp_propagate(error, ei, K, ALPHA, post_step=post)
                checks[name] = torch.equal(full[:N], want)

        # DistCorrectAndSmooth: world 2 takes a bool mask and long labels, the 2x2 grid a local index mask and one-hot rows
        y_loc = _local(y_soft, lo, hi, Rr)
        if Pf == 1:
            mask_loc = _local(train, lo, hi, Rr)
            yt_loc = labels[lo:hi][train[lo:hi]]
        else:
            idx = torch.nonzero(train[lo:hi]).view(-1)
            mask_loc = idx
            yt_loc = torch.nn.functional.one_hot(labels[lo + idx], F).float()
        if rank >= Pf:
            checks["empty_mask_here"] = int(mask_loc.sum() if mask_loc.dtype == torch.bool else mask_loc.numel()) == 0
        yt_glob = labels[train]
        for autoscale, scale in ((True, 1.0), (False, 0.7)):
            cs = PT.DistCorrectAndSmooth(K, ALPHA, K + 2, 0.6, autoscale, scale, grid=grid, N=N, runner=runner)
            got = cs.correct(y_loc, yt_loc, mask_loc)
            want = R.cs_correct(y_soft, yt_glob, train, ei, K, ALPHA, autoscale, scale)
            checks[f"correct_{autoscale}"] = _relerr(got[: hi - lo], want[lo:hi]) <= 1e-6
            checks[f"correct_{autoscale}_pad_finite"] = bool(torch.isfinite(got).all())
        got = cs.smooth(y_loc, yt_loc, mask_loc)
        want = R.cs_smooth(y_soft, yt_glob, train, ei, K + 2, 0.6)
        checks["smooth"] = _relerr(got[: hi - lo], want[lo:hi]) <= 1e-6
        checks["smooth_pad_finite"] = bool(torch.isfinite(got).all())
        ret[rank] = checks
    finally:
        dist.destroy_process_group()


def _spawn(world, Pf, port):
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, world, Pf, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=240)
        assert p.exitcode == 0
    return dict(ret)


def test_cs_on_a_row_partition_matches_the_oracle():
    ret = _spawn(2, 1, 35500 + (os.getpid() % 2000))
    for r in range(2):
        assert ret[r] and all(ret[r].values()), (r, ret[r])
        assert ret[r]["lp_clamp"] and ret[r]["lp_reset"]


def test_cs_on_a_row_by_feature_grid_matches_the_oracle():
    ret = _spawn(4, 2, 37500 + (os.getpid() % 2000))
    for r in range(4):
        assert ret[r] and all(ret[r].values()), (r, ret[r])


def test_dist_cs_rejects_other_dtypes_before_propagating():
    import rgb_experiment_b200.partition as PT

    def runner(*a, **k):
        raise AssertionError("no propagation may start")

    cs = PT.DistCorrectAndSmooth(2, 0.8, 2, 0.8, grid=PT.Grid(0, 1), N=5, runner=runner)
    for dt in (torch.float16, torch.float64):
        y = torch.full((5, 3), 1 / 3, dtype=dt)
        with pytest.raises(RuntimeError):
            cs.correct(y, torch.zeros(1, dtype=torch.long), torch.tensor([0]))
        with pytest.raises(RuntimeError):
            cs.smooth(y, torch.zeros(1, dtype=torch.long), torch.tensor([0]))
