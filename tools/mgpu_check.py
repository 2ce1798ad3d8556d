#!/usr/bin/env python
"""Multi-GPU parity + timing of the row-partitioned K-hop propagation (run under torchrun, one rank
per GPU):  push mode (SpMM epilogue stores into every peer over NVLink) and all-gather mode (NCCL)
must both equal the single-GPU result -- bit for bit on a pure row partition, within the fp32 bar
(1e-5 norm-wise) with feature slices.  Push is compared with the single-GPU folded-D^-1/2 path,
all-gather with the per-edge-weight path (the arithmetic each mode runs).
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29511 tools/mgpu_check.py [--family appnp|sgc|cs] [--workload products] [--steps 5]

--family appnp  APPNP K=10, alpha=0.1, F=47 (the default)
--family sgc    SGC's propagation: K=2, alpha=0, F=100, against ops.gcn_power
--family cs     Correct & Smooth, F=47, 50 + 50 hops, alpha 0.8, on the LOOP_NONE graph: a planted y_soft (softmax
                of a seeded matrix) with a seeded training mask through partition.DistCorrectAndSmooth -- correct
                with autoscale, correct with a fixed scale, smooth -- against shim.nn.CorrectAndSmooth (1e-6), and
                the three label propagations' final iterates against ops.label_propagation.
                A step is the reference's C&S post-process, correct (autoscale) + smooth: 100 hops."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DEFAULTS = {"appnp": (47, 10), "sgc": (100, 2), "cs": (47, 50)}      # F, K
CS_ALPHA, CS_SCALE, CS_TRAIN = 0.8, 1.0, 0.08


def device_info(dev):
    """Card name and power limit of this rank's GPU, read in the run that measures."""
    power = None
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(dev.index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(q)
    except (OSError, subprocess.SubprocessError, ValueError):
        pass
    return {"gpu": torch.cuda.get_device_name(dev), "power_limit_w": power}


def timed(fn, steps, dev):
    """ms per call: CUDA events over `steps` calls after two warm-up calls, max over ranks."""
    for _ in range(2):
        fn()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def assemble(out, grid, R, F, world, dev):
    """Every rank's [R, ld] result (row block rp, feature slice fp) -> the [R * Pr, F] matrix, on every rank."""
    ldmax = torch.tensor([out.size(1)], device=dev)
    dist.all_reduce(ldmax, op=dist.ReduceOp.MAX)
    ldm = int(ldmax.item())
    mine = torch.zeros((R, ldm), dtype=out.dtype, device=dev)
    mine[:, :out.size(1)] = out
    allb = torch.empty((world * R, ldm), dtype=out.dtype, device=dev)
    dist.all_gather_into_tensor(allb, mine)
    allb = allb.view(world, R, ldm)
    y = torch.empty((R * grid.Pr, F), dtype=out.dtype, device=dev)
    for r in range(world):                           # rank r = rp * Pf + fp holds rows block rp, feature slice fp
        a, b = grid.feature_slice(F, fp=r % grid.Pf)
        rp = r // grid.Pf
        y[rp * R:(rp + 1) * R, a:b] = allb[r, :, :b - a]
    return y


def full_rows(out, grid, R, F, world, dev):
    """[R, F] full-width rows of every rank -> [R * Pr, F] (the ranks of a row block hold the same rows)."""
    allb = torch.empty((world * R, F), dtype=out.dtype, device=dev)
    dist.all_gather_into_tensor(allb, out.contiguous())
    allb = allb.view(world, R, F)
    return torch.cat([allb[rp * grid.Pf] for rp in range(grid.Pr)])


def compare(y, ref, Pf, bit_equal):
    """(matches, relerr).  Propagations (bit_equal): bit-equal on a pure row partition.  C&S outputs: 1e-6 there (sigma
    and the row L1 norms are summed in another order).  With feature slices everything is held to the fp32 bar (1e-5
    norm-wise): a feature-sliced grid reorders the partial sums of split long rows."""
    err = float((y - ref).abs().max() / ref.abs().max())
    if Pf > 1:
        return err <= 1e-5, err
    return (bool(torch.equal(y, ref)) if bit_equal else err <= 1e-6), err


def run_khop(args, family, F, K, alpha, sg, grid, blk, dev, P, PT):
    """APPNP / SGC: the existing parity + timing of PartitionedAPPNP.run(z0, K, alpha)."""
    rank, world, N, R = grid.rank, grid.world, sg.num_nodes, blk.R
    flo, fhi = grid.feature_slice(F)
    Fl = fhi - flo
    z0 = torch.randn(N, F, device=dev, generator=torch.Generator(device=dev).manual_seed(1))   # same on every rank
    res = {}
    for mode in ("allgather", "push"):
        prop = PT.PartitionedAPPNP(blk, Fl, group=grid.row_group, mode=mode)
        z0l = torch.zeros((R, prop.ld), device=dev)
        z0l[: blk.hi - blk.lo, :Fl] = z0[blk.lo:blk.hi, flo:fhi]
        out = prop.run(z0l, K, alpha).clone()
        ms = timed(lambda: prop.run(z0l, K, alpha), args.steps, dev)
        res[mode] = (assemble(out, grid, R, F, world, dev)[:N].clone(), ms, prop.mode)
        prop.close()
        del prop
    ok, err = {}, {}
    if rank == 0:
        g = P.Graph(sg.edge_index, N, P.LOOP_ADD_REMAINING)
        for mode, (y, _, ran) in res.items():
            fold = ran == "push"                       # one rank runs the all-gather form whatever was asked
            ref = P.ops.appnp(z0, g, K, alpha, fold) if family == "appnp" else P.ops.gcn_power(z0, g, K, fold)
            ok[mode], err[mode] = compare(y, ref, grid.Pf, True)
    line = {"matches_single_gpu": ok, "relerr": err,
            "ms_per_step": {m: round(v[1], 3) for m, v in res.items()},
            "ms_per_hop": {m: round(v[1] / K, 4) for m, v in res.items()},
            "gteps": {m: round(blk.nnz_global * K / v[1] / 1e6, 2) for m, v in res.items()}}
    return line, ok


def run_cs(args, F, K, sg, grid, blk, dev, P, PT):
    """Correct & Smooth through DistCorrectAndSmooth over PartitionedAPPNP, both modes."""
    from rgb_experiment_b200.shim import nn as SN
    rank, world, N, R = grid.rank, grid.world, sg.num_nodes, blk.R
    gen = torch.Generator(device=dev).manual_seed(2)
    y_soft = torch.softmax(torch.randn(N, F, device=dev, generator=gen), dim=1)       # same on every rank
    labels = torch.randint(F, (N,), device=dev, generator=gen)
    train = torch.rand(N, device=dev, generator=gen) < CS_TRAIN
    n = blk.hi - blk.lo
    y_loc = torch.zeros((R, F), device=dev)
    y_loc[:n] = y_soft[blk.lo:blk.hi]
    m_loc = torch.zeros(R, dtype=torch.bool, device=dev)
    m_loc[:n] = train[blk.lo:blk.hi]
    yt_loc = labels[blk.lo:blk.hi][train[blk.lo:blk.hi]]
    # the three label propagations' start matrices, for the iterate check
    error = torch.zeros_like(y_soft)
    error[train] = torch.nn.functional.one_hot(labels[train], F).float() - y_soft[train]
    smooth0 = y_soft.clone()
    smooth0[train] = torch.nn.functional.one_hot(labels[train], F).float()
    flo, fhi = grid.feature_slice(F)
    Fl = fhi - flo
    ld = PT.DistCorrectAndSmooth.slice_ld(grid, F)
    tele = (CS_ALPHA, 1.0 - CS_ALPHA)
    lp_kw = {"lp_clamp": lambda z: dict(clamp=(-1.0, 1.0)), "lp_reset": lambda z: dict(reset=(m_loc, z)),
             "lp_smooth": lambda z: dict(clamp=(0.0, 1.0))}
    res = {}
    for mode in ("allgather", "push"):
        prop = PT.PartitionedAPPNP(blk, Fl, group=grid.row_group, mode=mode, ld=ld)
        lps = {}
        for name, start in (("lp_clamp", error), ("lp_reset", error), ("lp_smooth", smooth0)):
            z0 = torch.zeros((R, ld), device=dev)
            z0[:n, :Fl] = start[blk.lo:blk.hi, flo:fhi]
            out = prop.run(z0, K, teleport=tele, **lp_kw[name](z0)).clone()
            lps[name] = assemble(out, grid, R, F, world, dev)[:N].clone()
        auto = PT.DistCorrectAndSmooth(K, CS_ALPHA, K, CS_ALPHA, True, grid=grid, N=N, runner=prop.run)
        fixed = PT.DistCorrectAndSmooth(K, CS_ALPHA, K, CS_ALPHA, False, CS_SCALE, grid=grid, N=N, runner=prop.run)
        outs = {"correct_autoscale": auto.correct(y_loc, yt_loc, m_loc),
                "correct_fixed": fixed.correct(y_loc, yt_loc, m_loc)}
        outs["smooth"] = auto.smooth(outs["correct_autoscale"], yt_loc, m_loc)
        outs = {k: full_rows(v, grid, R, F, world, dev)[:N].clone() for k, v in outs.items()}
        ms = {"correct_autoscale": timed(lambda: auto.correct(y_loc, yt_loc, m_loc), args.steps, dev),
              "correct_fixed": timed(lambda: fixed.correct(y_loc, yt_loc, m_loc), args.steps, dev),
              "smooth": timed(lambda: auto.smooth(y_loc, yt_loc, m_loc), args.steps, dev),
              "lp": timed(lambda: prop.run(z0, K, teleport=tele, clamp=(0.0, 1.0)), args.steps, dev)}
        res[mode] = (lps, outs, ms, prop.mode)
        prop.close()
        del prop
    ok, err = {}, {}
    if rank == 0:
        import rgb_experiment_b200.ops as ops
        g = P.Graph(sg.edge_index, N, P.LOOP_NONE)
        for mode, (lps, outs, _, ran) in res.items():
            fold = ran == "push"                       # one rank runs the all-gather form whatever was asked
            want = {"lp_clamp": ops.label_propagation(g, error, K, CS_ALPHA, clamp=(-1.0, 1.0), fold=fold),
                    "lp_reset": ops.label_propagation(g, error, K, CS_ALPHA, reset_mask=train, reset_val=error, fold=fold),
                    "lp_smooth": ops.label_propagation(g, smooth0, K, CS_ALPHA, clamp=(0.0, 1.0), fold=fold)}
            checks = {k: compare(lps[k], want[k], grid.Pf, True) for k in want}
            old = ops.FOLD_KHOP
            ops.FOLD_KHOP = fold                       # the shim takes the same normalisation form as the mode
            try:
                ref_a = SN.CorrectAndSmooth(K, CS_ALPHA, K, CS_ALPHA, True)
                ref_f = SN.CorrectAndSmooth(K, CS_ALPHA, K, CS_ALPHA, False, CS_SCALE)
                ei = sg.edge_index
                c_a = ref_a.correct(y_soft, labels[train], train, ei)
                ref = {"correct_autoscale": c_a, "correct_fixed": ref_f.correct(y_soft, labels[train], train, ei),
                       "smooth": ref_a.smooth(c_a, labels[train], train, ei)}
            finally:
                ops.FOLD_KHOP = old
            checks.update({k: compare(outs[k], ref[k], grid.Pf, False) for k in ref})
            ok[mode] = all(v[0] for v in checks.values())
            err[mode] = {k: v[1] for k, v in checks.items()}
    hops = 2 * K
    line = {"matches_single_gpu": ok, "relerr": err,
            "ms_per_step": {m: round(v[2]["correct_autoscale"] + v[2]["smooth"], 3) for m, v in res.items()},
            "ms_per_hop": {m: round(v[2]["lp"] / K, 4) for m, v in res.items()},
            "gteps": {m: round(blk.nnz_global * hops / (v[2]["correct_autoscale"] + v[2]["smooth"]) / 1e6, 2)
                      for m, v in res.items()},
            "ms": {m: {k: round(t, 3) for k, t in v[2].items()} for m, v in res.items()}}
    return line, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--family", choices=sorted(DEFAULTS), default="appnp")
    ap.add_argument("--workload", default="medium")
    ap.add_argument("--F", type=int, default=None)
    ap.add_argument("--K", type=int, default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--feature-groups", type=int, default=1)
    args = ap.parse_args()
    F = DEFAULTS[args.family][0] if args.F is None else args.F
    K = DEFAULTS[args.family][1] if args.K is None else args.K
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    import rgb_experiment_b200 as P
    import rgb_experiment_b200.graph as G_
    import rgb_experiment_b200.partition as PT
    import rgb_experiment_b200.synth as S
    if args.workload == "medium":
        sg = S.make_graph(300_001, 6_000_000, 8, 4, device=dev, features=False)
    else:
        sg = S.make_named(args.workload, device=dev, features=False)
    N = sg.num_nodes
    grid = PT.Grid(rank, world, args.feature_groups)
    loop = P.LOOP_NONE if args.family == "cs" else P.LOOP_ADD_REMAINING
    blk = PT.LocalBlock(sg.edge_index, N, loop, grid.rp, grid.Pr, group=grid.row_group)
    # the single-GPU reference splits long rows where the blocks do (blocks of a million rows and more split them at
    # 256 edges, the whole graph at 1,024): the split orders a long row's partial sums
    G_.DEFAULT_CHUNK, G_.DEFAULT_LONG_CHUNK = blk.csr.chunk, blk.csr.long_chunk
    if args.family == "cs":
        line, ok = run_cs(args, F, K, sg, grid, blk, dev, P, PT)
    else:
        line, ok = run_khop(args, args.family, F, K, 0.1 if args.family == "appnp" else 0.0, sg, grid, blk, dev, P, PT)
    if rank == 0:
        head = {"family": args.family, "workload": args.workload, "N": N, "nnz": blk.nnz_global, "F": F, "K": K,
                "world": world, "grid": f"{grid.Pr}x{grid.Pf}", **device_info(dev)}
        print(json.dumps({**head, **line}), flush=True)
    flag = torch.tensor([1 if (rank != 0 or all(ok.values())) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
