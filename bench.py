#!/usr/bin/env python
"""bench.py -- the message-passing hot path on the BASELINE.json shapes, one JSON line per run.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]

Workloads (BASELINE.json `configs`; the default is the one the headline metric is quoted on):
  products     configs[3]: APPNP K=10 propagation on the ogbn-products-shaped graph (N 2.45 M / 126.2 M edges with
               loops / F=47 fp32), 1/2/4/8 GPUs.  step = the 10 fused hops of one APPNP forward, called through the
               shim layer the reference's APPNPStack constructs (appnp_stack.py:22,30).           [default]
  arxiv_sage   configs[1]: GraphSAGE (3 layers, hidden 256) on the ogbn-arxiv-shaped graph, 1 GPU.  step = the three
               mean aggregations of one forward (F = 256, 256, 40; graphsage.py:58) through MessagePassing.propagate.
  reddit_gat   configs[2]: GAT 8 heads x 8 on the Reddit-shaped graph (114.8 M edges with loops), 1 GPU.  step = the
               edge-softmax + aggregate of the first layer (gat.py:18), forward.
  papers100m   configs[4]: GCN propagation, bf16 features, papers100M-shaped row-generated graph (111 M nodes / 3.3 B
               edges / F=128), row-partitioned over 2/4/8 GPUs (--scale shrinks it for fewer GPUs).  step = 2 hops.
value = aggregated edges / s (GTEPS) over all ranks, inputs resident in HBM, CUDA events, max over ranks.
e2e   = the same metric through the public call with HOST buffers: H2D of the step's input from pinned memory and D2H
        of its result inside the timed region.
roofline = algorithmic bytes (SURVEY.md 8d gather model, no cache credit) per hop / measured hop time against the
        measured HBM copy peak; for L2-resident feature matrices also against the device's random row-gather peak
        measured live (csrc/microbench.cu) -- the HBM fraction of such a kernel is meaningless.
--impl reference times the reference's CPU path (the oracle's restated PyG gather -> scale -> scatter_add_, this
tier's definition) on the host cores, rank 0 only.  Prints ONE JSON line on rank 0.
--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (see dump_outputs), so that two builds
run with the same arguments -- hence on the same seeded inputs -- can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K_HOPS, ALPHA, F_CLASSES = 10, 0.1, 47
GRAPH_SEED = 20261018
CPU_SAMPLE_FRACTION = 0.10          # share of the target rows used by the bounded CPU sample (products)
DUMP_BYTES = 60 << 20               # --dump-outputs: payload of all .npy files of a run together, all ranks (< 64 MB)
DUMP_SEED = 20261019
METRIC = {"products": "appnp_propagate_gteps", "arxiv_sage": "sage_mean_aggregate_gteps",
          "reddit_gat": "gat_layer_forward_gteps", "papers100m": "gcn_propagate_bf16_gteps"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def algorithmic_bytes_per_hop(nnz: int, n: int, F: int, weighted: bool, esz: int = 4, teleport: bool = True) -> int:
    """SURVEY.md 8d gather model, no cache credit: nnz*(F*s + 4 [col] + s_w) + N*F*s [store] + (N+1)*8 [rowptr]
    (+ N*F*s [teleport read] for K-hop families)."""
    return nnz * (F * esz + 4 + (4 if weighted else 0)) + n * F * esz + (n + 1) * 8 + (n * F * esz if teleport else 0)


def workload_name(wl: str, N: int, nnz: int) -> str:
    """config.workload, shared by both arms (the reference arm runs a bounded sample of the same workload)."""
    if wl == "products":
        return (f"APPNP K={K_HOPS} alpha={ALPHA} propagate, ogbn-products-shaped R-MAT graph "
                f"(N={N}, E={nnz - N} directed + {N} self loops, F={F_CLASSES} fp32)")
    if wl == "arxiv_sage":
        return (f"GraphSAGE 3x256 mean aggregations (F=256,256,40 fp32) of one forward, ogbn-arxiv-shaped R-MAT graph "
                f"(N={N}, nnz={nnz} with self loops)")
    if wl == "reddit_gat":
        return f"GATConv 8 heads x 8 edge-softmax + aggregate forward, Reddit-shaped R-MAT graph (N={N}, nnz={nnz} with self loops)"
    return f"GCN propagation 2 hops, bf16 F=128, papers100M-shaped row-generated graph (N={N}, nnz={nnz} with self loops)"


def dump_outputs(out_dir: str, arrays: dict, budget: int = DUMP_BYTES, seed: int = DUMP_SEED) -> None:
    """Write every tensor of `arrays` (name -> tensor, rows first) as out_dir/<name>.npy: float64 stays float64, every
    other dtype becomes float32.  When the arrays hold more than `budget` bytes together, each keeps the same share of
    its rows: a sorted sample drawn from a generator seeded with `seed`, so the same shapes always give the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(v.numel() * (8 if v.dtype == torch.float64 else 4) for v in arrays.values())      # bytes as written
    keep = budget / total if total > budget else 1.0
    for name, v in arrays.items():
        v = v.detach()
        if keep < 1.0:                   # sample first: a bf16 output is never widened at full size
            n = v.size(0)
            rows = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[: max(1, int(n * keep))].sort().values
            v = v.index_select(0, rows.to(v.device))
        if v.dtype != torch.float64:
            v = v.float()
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy())


def make_products(device):
    import rgb_experiment_b200.synth as S
    return S.make_named("products", seed=GRAPH_SEED, device=device, features=False)


# ------------------------------------------------------------------------------------------------------------
# CPU side (reference arm and cpu_baseline): the literal PyG-on-CPU form from the oracle, bounded samples
# ------------------------------------------------------------------------------------------------------------
def cpu_sample_products(sg):
    """Bounded CPU sample: the edges (after add_remaining_self_loops) whose target is one of the first 10% of the
    nodes, with their gcn_norm weights, and z [N, 47]."""
    N = sg.num_nodes
    ei = sg.edge_index
    loop = torch.arange(N, device=ei.device)
    src = torch.cat([ei[0], loop])
    dst = torch.cat([ei[1], loop])
    dinv = torch.bincount(dst, minlength=N).float().pow(-0.5)
    n_sub = int(N * CPU_SAMPLE_FRACTION)
    m = dst < n_sub
    s, d = src[m], dst[m]
    w = dinv[s] * dinv[d]
    z = torch.randn(N, F_CLASSES, generator=torch.Generator().manual_seed(1))
    return s.cpu(), d.cpu(), w.cpu(), z, n_sub


def cpu_hop_products(s, d, w, z, n_sub, alpha=ALPHA):
    """The literal PyG-on-CPU form (oracle.pyg_restated.propagate): index_select -> mul -> scatter_add_."""
    from oracle import pyg_restated as R
    out = R.scatter_add(w.view(-1, 1) * z.index_select(0, s), d, dim=0, dim_size=n_sub)
    return out * (1 - alpha) + alpha * z[:n_sub]


def cpu_strong_baseline(s, d, w, z, n_sub, budget_s=10.0, alpha=ALPHA):
    """SURVEY.md 8d (ii): the same hop as one torch.sparse CSR product A @ z on the host cores -- no [nnz, F] message
    tensor, the strongest CPU form available in this image.  Reported beside the literal PyG form, never instead of it."""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        perm = torch.argsort(d, stable=True)
        crow = torch.zeros(n_sub + 1, dtype=torch.int64)
        crow[1:] = torch.cumsum(torch.bincount(d, minlength=n_sub), 0)
        A = torch.sparse_csr_tensor(crow, s[perm], w[perm], size=(n_sub, z.size(0)))
        best, hops, t_all = None, 0, time.perf_counter()
        while hops < 6 and (hops < 2 or time.perf_counter() - t_all < budget_s):
            t0 = time.perf_counter()
            out = (A @ z) * (1 - alpha) + alpha * z[:n_sub]
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
            hops += 1
    del out
    return {"value": s.numel() / best / 1e9, "unit": "GTEPS", "kind": "torch.sparse CSR A @ z on the same sample and weights",
            "best_of": hops}


def cpu_case(wl: str, dev):
    """(fn, edges_per_call, sample description, extra) for the bounded CPU run of workload `wl`."""
    import rgb_experiment_b200.synth as S
    from oracle import pyg_restated as R
    if wl == "products":
        sg = make_products(dev)
        s, d, w, z, n_sub = cpu_sample_products(sg)
        del sg
        desc = (f"1 hop over the {s.numel()} edges whose target is in the first {int(CPU_SAMPLE_FRACTION * 100)}% of nodes; "
                "literal index_select->mul->scatter_add_ fp32")
        return (lambda: cpu_hop_products(s, d, w, z, n_sub)), s.numel(), desc, (s, d, w, z, n_sub)
    if wl == "arxiv_sage":
        sg = S.make_named("arxiv", seed=GRAPH_SEED, device="cpu", features=False)
        N = sg.num_nodes
        ei = R.edit_loops(sg.edge_index, N, R.LOOP_REMOVE_THEN_ADD)
        x = torch.randn(N, 256, generator=torch.Generator().manual_seed(1))
        desc = f"1 mean aggregation at F=256 over all {ei.size(1)} edges; literal index_select->scatter(mean) fp32 (graphsage.py:58)"
        return (lambda: R.scatter(x.index_select(0, ei[0]), ei[1], 0, N, "mean")), ei.size(1), desc, None
    if wl == "reddit_gat":
        sg = S.make_named("reddit", seed=GRAPH_SEED, device=dev, features=False)
        N, H, C = sg.num_nodes, 8, 8
        n_sub = N // 50
        ei = sg.edge_index
        m = (ei[1] < n_sub) & (ei[0] != ei[1])
        loop = torch.arange(n_sub, device=ei.device)
        row = torch.cat([ei[0][m], loop]).cpu()
        col = torch.cat([ei[1][m], loop]).cpu()
        del sg, ei, m
        g = torch.Generator().manual_seed(1)
        xp = torch.randn(N, H, C, generator=g)
        a_s, a_d = torch.randn(N, H, generator=g), torch.randn(N, H, generator=g)

        def fn():
            e = torch.nn.functional.leaky_relu(a_s[row] + a_d[col], 0.2)
            alpha = R.softmax(e, col, num_nodes=n_sub)
            return R.scatter_add(xp[row] * alpha.unsqueeze(-1), col, dim=0, dim_size=n_sub)

        desc = (f"GATConv attention + aggregate over the {row.numel()} edges whose target is in the first 2% of nodes; literal "
                "PyG form (gathers, scatter-max/sum softmax, [nnz,8,8] message) fp32")
        return fn, row.numel(), desc, None
    raise RuntimeError(f"no CPU case for workload {wl}")


def run_reference(args, rank):
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the other ranks have already left, so rank 0 takes every
    # host core it is allowed to run on (the same thread count a plain `python bench.py --impl reference` gets)
    try:
        torch.set_num_threads(len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        torch.set_num_threads(os.cpu_count() or 1)
    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    wl = args.workload
    if wl == "papers100m":
        print(json.dumps({"impl": "reference", "metric": METRIC[wl],
                          "unavailable": "papers100M-shaped graph (3.3 B edges) has no bounded CPU form here; see --workload products"}))
        return
    import rgb_experiment_b200.synth as S
    fn, edges, sample, extra = cpu_case(wl, dev)
    shape = {"products": "products", "arxiv_sage": "arxiv", "reddit_gat": "reddit"}[wl]
    N_full = S.SHAPES[shape][0]
    nnz_full = N_full + S.SHAPES[shape][1]
    cores = torch.get_num_threads()
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps - 1):
        fn()
    last = fn()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": last})
    del last
    val = edges * args.steps / dt / 1e9
    sample = "per step: " + sample
    cpu = {"value": val, "unit": "GTEPS", "cores": cores, "kind": "port", "sample": sample}
    if wl == "products":
        cpu["strong"] = cpu_strong_baseline(*extra)
    line = {"impl": "reference", "metric": METRIC[wl], "value": val, "unit": "GTEPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(wl, N_full, nnz_full), "hops_per_step": 1, "nnz": nnz_full,
                       "parallelism": f"{cores} host threads", "sample": sample},
            "cpu_baseline": cpu,
            "e2e": {"value": val, "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------
def gather_peak(dev, table_bytes: int, row_bytes: int):
    """GB/s of random row gathers from a table of `table_bytes` (csrc/microbench.cu), best of 3."""
    import rgb_experiment_b200 as P
    L = P._lib.lib()
    n_rows = max(1, table_bytes // row_bytes)
    table = torch.randn(n_rows * row_bytes // 4, device=dev)
    G = row_bytes // 16
    n_groups = 148 * 4 * 256 // G * 4
    per = 1024
    out = torch.empty(n_groups * 4, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    best = None
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        P._lib.check(L.rgbmp_microbench_gather(table.data_ptr(), n_rows, row_bytes, per, 1234 + it, out.data_ptr(), n_groups,
                                               dev.index, st), "microbench_gather")
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if it > 0:
            best = ms if best is None else min(best, ms)
    return n_groups * per * row_bytes / best / 1e6


def run_epoch_guarded(rank, world, dev, line, limit_s=300):
    """The second half of the BASELINE metric ("full-batch epoch ms at 1/2/4/8 GPU"): the reference's APPNPStack
    epoch (1 train forward + backward + Adam, 2 eval forwards; itexperiments.py:417-473) on the same products-shaped
    graph, measured by tools/bench_epoch.py AFTER the timed region and reported under "epoch" (single GPU: also AS
    CALLED, through the reference's own model class and test()/compare_pred_label from baseline/_ref).  It never
    costs the headline line: an exception becomes {"error": ...}, and if nothing comes back within `limit_s` seconds
    (a rank stuck in a collective) a watchdog prints the line without it and ends the process with status 0."""
    import importlib.util
    done = threading.Event()

    def watchdog():
        if done.wait(limit_s):
            return
        if line is not None:
            line["epoch"] = {"error": f"no result within {limit_s} s"}
            print(json.dumps(line), flush=True)
        os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    try:
        spec = importlib.util.spec_from_file_location("_bench_epoch", os.path.join(ROOT, "tools", "bench_epoch.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        res = mod.run(mod.default_args(), rank, world, dev)
        res.pop("check_vs_single_gpu", None)
        if world == 1:
            torch.cuda.empty_cache()
            try:
                res["as_called"] = mod.run_as_called(mod.default_args(epochs=3, warmup=1), dev)
            except Exception as e:                                    # noqa: BLE001
                res["as_called"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    except Exception as e:                                        # noqa: BLE001 -- reported, never fatal for the line
        res = {"error": f"{type(e).__name__}: {e}"[:300]}
        if line is None:                                          # a peer may now be waiting for me: leave quietly
            done.set()
            os._exit(0)
    done.set()
    return res


class Case:
    """What a workload hands to the timing harness."""
    step = None                  # () -> tensor: one pass of the hot path, inputs resident in HBM
    e2e_step = None              # () -> None: the same from pinned host buffers, result back on the host
    edges_per_step = 0           # aggregated edges (all ranks) per step
    hops_per_step = 1
    launches_per_step = 0
    h2d = d2h = 0
    hop_bytes = 0                # algorithmic bytes of the dominant kernel's launch (per GPU)
    kernel = ""
    dtype = "f32"
    config = None
    l2_table = None              # (table bytes, row bytes): feature matrix is L2-resident -> also report the gather roofline
    gathered_bytes_per_step = 0
    check = None                 # () -> dict, run after the timed region
    outputs = None               # (what step returned) -> {name: tensor} a caller receives; None: {"out": it}
    close = None
    scaling = "strong"
    keep = None


def case_products(args, dev, rank, world):
    import rgb_experiment_b200 as P
    import rgb_experiment_b200.partition as PT
    c = Case()
    sg = make_products(dev)
    N, F = sg.num_nodes, F_CLASSES
    t0 = time.perf_counter()
    if world == 1:
        g = P.get_graph(sg.edge_index, N, P.LOOP_ADD_REMAINING)      # what the layer's first forward does
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        nnz = g.nnz
        z0 = torch.randn(N, F, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
        # the call the reference's APPNPStack makes (appnp_stack.py:22,30): the shim layer, its graph-cache lookup
        # and the autograd.Function are inside the timed region; --fold 1 is the layer's default form
        import rgb_experiment_b200.shim.nn as SN
        layer = SN.APPNP(K_HOPS, ALPHA)
        layer.fold_norm = bool(args.fold)
        ei = sg.edge_index                              # stays alive: the cached graph lives as long as this tensor
        c.step = lambda: layer(z0, ei)
        c.launches_per_step = K_HOPS * (1 + (2 if g.fwd.n_items > 0 else 0)) + (1 if args.fold else 0)
        z0h = z0.cpu().pin_memory()
        outh = torch.empty_like(z0h).pin_memory()
        plan = P.ops.HostAppnpPlan(g, F)
        c.e2e_step = lambda: P.ops.appnp_host(g, z0h, outh, K_HOPS, ALPHA, plan)      # returns after the D2H completed
        c.h2d = c.d2h = N * F * 4
        weighted = not args.fold
        c.hop_bytes = algorithmic_bytes_per_hop(nnz, N, F, weighted)
        par = "single"
        c.keep = (g, ei, plan, z0, z0h, outh)
        sched = dict(P.graph.cluster_stats["last"] or {}, used=g.fwd.clustered)
    else:
        Pf = args.feature_groups if args.feature_groups > 0 else PT.auto_feature_groups(world, F)
        grid = PT.Grid(rank, world, Pf)
        grid.warm_up(dev)                               # sub-communicator set-up (seconds) is not graph-build time
        t0 = time.perf_counter()
        flo, fhi = grid.feature_slice(F)
        F_local = fhi - flo
        # row blocks are runs of whole communities (nodes renamed by locality group; same operator on the renamed graph,
        # z0 is synthetic either way): --relabel 0 keeps the id-range blocks
        blk = PT.LocalBlock(sg.edge_index, N, P.LOOP_ADD_REMAINING, grid.rp, grid.Pr, group=grid.row_group,
                            relabel=bool(args.relabel), row_bytes=F_local * 4)
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        nnz = blk.nnz_global
        prop = PT.PartitionedAPPNP(blk, F_local, group=grid.row_group, mode=args.exchange)
        z0l = torch.zeros((blk.R, prop.ld), device=dev)
        z0l[: blk.hi - blk.lo, :F_local] = torch.randn(blk.hi - blk.lo, F, device=dev,
                                                       generator=torch.Generator(device=dev).manual_seed(1 + grid.rp))[:, flo:fhi]
        c.step = lambda: prop.run(z0l, K_HOPS, ALPHA)
        c.launches_per_step = K_HOPS * prop.launches_per_hop
        z0h = z0l.cpu().pin_memory()
        outh = torch.empty_like(z0h).pin_memory()

        def e2e():
            z0l.copy_(z0h, non_blocking=True)
            outh.copy_(c.step(), non_blocking=True)
            torch.cuda.synchronize()

        c.e2e_step = e2e
        c.h2d = c.d2h = z0l.numel() * 4 * world
        weighted = args.exchange == "allgather"          # the push path folds D^-1/2 too
        c.hop_bytes = algorithmic_bytes_per_hop(nnz // grid.Pr, N // grid.Pr, F_local, weighted)
        par = f"{grid.Pr} row blocks x {grid.Pf} feature slices, exchange={args.exchange}"
        sched = {"used": bool(getattr(blk.csr, "clustered", False)), "community_row_blocks": blk.inv is not None}

        def check():
            """Rank 0 (row block 0, feature slice 0) recomputes ITS rows on its own GPU from the whole graph and the
            whole z0 (every row block's rows regenerated from their seeds) and compares with the partitioned result."""
            out = prop.run(z0l, K_HOPS, ALPHA).clone()
            res = None
            if rank == 0:
                ei_chk = sg.edge_index if blk.inv is None else blk.inv[sg.edge_index]     # the renamed graph
                g1 = P.Graph(ei_chk, N, P.LOOP_ADD_REMAINING)
                R_ = blk.R
                z_full = torch.cat([torch.randn(min(N, (q + 1) * R_) - q * R_, F, device=dev,
                                                generator=torch.Generator(device=dev).manual_seed(1 + q))
                                    for q in range(grid.Pr)])
                ref = P.ops._appnp_khop(g1.fwd, g1, z_full, K_HOPS, ALPHA, False, True)[blk.lo:blk.hi, flo:fhi]
                got = out[: blk.hi - blk.lo, :F_local]
                err = float((got - ref).abs().max() / ref.abs().max())
                res = {"rank0_rows_vs_single_gpu_relerr": err, "bit_equal": bool(torch.equal(got, ref)), "rows": blk.hi - blk.lo}
                del g1
            return res

        c.check = check
        c.outputs = lambda z: {"out": z[: blk.hi - blk.lo, :F_local]}      # this rank's rows (renamed ids) and slice
        c.close = prop.close
        c.keep = (blk, prop, z0l, z0h, outh, sg)
    c.edges_per_step, c.hops_per_step = nnz * K_HOPS, K_HOPS
    c.kernel = "spmm_rows_kernel<float,4,...> (+long/combine)"
    c.config = {"workload": workload_name("products", N, nnz), "hops_per_step": K_HOPS, "nnz": nnz, "parallelism": par,
                "l2": "inputs larger than L2 (features 470 MB, col 505 MB vs 126 MB L2)",
                "norm": "per-edge weights" if weighted else "folded row scaling (same operator, no per-edge weight stream)",
                "graph_build_ms": build_ms, "row_schedule": sched}
    return c


def case_arxiv_sage(args, dev, rank, world):
    import rgb_experiment_b200 as P
    import rgb_experiment_b200.shim.nn as SN
    import rgb_experiment_b200.shim.utils as SU
    import rgb_experiment_b200.synth as S
    if world != 1:
        raise RuntimeError("--workload arxiv_sage is a single-GPU configuration (BASELINE.json configs[1])")
    c = Case()
    sg = S.make_named("arxiv", seed=GRAPH_SEED, device=dev, features=False)
    N, ei = sg.num_nodes, sg.edge_index
    widths = (256, 256, 40)
    xs = [torch.randn(N, F, device=dev, generator=torch.Generator(device=dev).manual_seed(1 + i)) for i, F in enumerate(widths)]
    mp = SN.MessagePassing(aggr="mean")                  # my_SAGEConv's base class and call (graphsage.py:39,53-58)

    def edited():
        e2, _ = SU.remove_self_loops(ei)
        return SU.add_self_loops(e2, num_nodes=N)[0]

    def step():
        return [mp.propagate(edited(), x=x) for x in xs]

    c.step = step
    c.outputs = lambda outs: {f"aggr{i}": o for i, o in enumerate(outs)}
    g = P.get_graph(edited(), N, P.LOOP_NONE)
    nnz = g.nnz
    xh = [x.cpu().pin_memory() for x in xs]
    outh = [torch.empty_like(x).pin_memory() for x in xh]

    def e2e():
        for x, xhost, oh in zip(xs, xh, outh):
            x.copy_(xhost, non_blocking=True)
            oh.copy_(mp.propagate(edited(), x=x), non_blocking=True)
        torch.cuda.synchronize()

    c.e2e_step = e2e
    c.h2d = c.d2h = sum(N * F * 4 for F in widths)
    c.edges_per_step, c.hops_per_step = nnz * len(widths), len(widths)
    c.launches_per_step = len(widths) * (1 + (2 if g.fwd.n_items > 0 else 0))
    c.hop_bytes = sum(algorithmic_bytes_per_hop(nnz, N, F, False, teleport=False) for F in widths) // len(widths)
    c.kernel = "spmm_rows_kernel<float,4,G32/G16,...> mean epilogue (+long/combine)"
    c.l2_table = (N * 256 * 4, 512)                      # gathered in 512-byte units (32 lanes x 16 B), the widest the LSU sees
    c.gathered_bytes_per_step = sum(nnz * F * 4 for F in widths)
    c.config = {"workload": workload_name("arxiv_sage", N, nnz), "hops_per_step": len(widths), "nnz": nnz, "parallelism": "single",
                "l2": "feature matrices 173 / 173 / 27 MB vs 126 MB L2: mostly L2-resident; between timed steps the three "
                      "matrices (373 MB) evict one another"}
    c.keep = (sg, g, xs, xh, outh)
    return c


def case_reddit_gat(args, dev, rank, world):
    import rgb_experiment_b200 as P
    import rgb_experiment_b200.synth as S
    if world != 1:
        raise RuntimeError("--workload reddit_gat is a single-GPU configuration (BASELINE.json configs[2])")
    c = Case()
    sg = S.make_named("reddit", seed=GRAPH_SEED, device=dev, features=False)
    N, ei, H, C = sg.num_nodes, sg.edge_index, 8, 8
    g = P.get_graph(ei, N, P.LOOP_REMOVE_THEN_ADD)
    nnz = g.nnz
    gen = torch.Generator(device=dev).manual_seed(1)
    # two input sets used alternately (2 x 67 MB)
    sets = [(torch.randn(N, H * C, device=dev, generator=gen), torch.randn(N, H, device=dev, generator=gen),
             torch.randn(N, H, device=dev, generator=gen)) for _ in range(2)]
    state = {"i": 0}

    def step():
        xp, a_s, a_d = sets[state["i"] & 1]
        state["i"] += 1
        return P.ops.gat(xp, a_s, a_d, g, H, C, 0.2)       # grad mode on, no input requires grad: eval-form kernels, no memo

    c.step = step
    hs = tuple(t.cpu().pin_memory() for t in sets[0])
    outh = torch.empty(N, H * C).pin_memory()

    def e2e():
        for t, th in zip(sets[0], hs):
            t.copy_(th, non_blocking=True)
        outh.copy_(P.ops.gat(*sets[0], g, H, C, 0.2), non_blocking=True)
        torch.cuda.synchronize()

    c.e2e_step = e2e
    c.h2d, c.d2h = N * (H * C + 2 * H) * 4, N * H * C * 4
    c.edges_per_step, c.hops_per_step = nnz, 1
    c.launches_per_step = 2 + 1 + (2 if g.fwd.n_items > 0 else 0)
    c.hop_bytes = nnz * (H * C * 4 + H * 4 + 4) + N * H * C * 4 + 2 * N * H * 4
    c.kernel = "att_fwd_rows_kernel<GAT,eval,G8> (+att_fwd_long/combine)"
    c.l2_table = (N * H * C * 4, H * C * 4)
    c.gathered_bytes_per_step = nnz * (H * C * 4 + H * 4)
    c.config = {"workload": workload_name("reddit_gat", N, nnz), "hops_per_step": 1, "nnz": nnz, "parallelism": "single",
                "l2": "X' 59.6 MB + a_src 7.5 MB are L2-resident (126 MB L2); two input sets alternate between steps"}
    c.keep = (sg, g, sets, hs, outh)
    return c


def case_papers100m(args, dev, rank, world):
    import rgb_experiment_b200.partition as PT
    import rgb_experiment_b200.synth as S
    c = Case()
    N0, E0, F = S.PAPERS100M
    scale = args.scale if args.scale > 0 else (1.0 if world >= 2 else 0.25)
    N, E = int(N0 * scale), int(E0 * scale)
    dt, esz, hops = torch.bfloat16, 2, 2
    Pf = args.feature_groups if args.feature_groups > 0 else (2 if world >= 4 else 1)
    grid = PT.Grid(rank, world, Pf)
    grid.warm_up(dev)
    t0 = time.perf_counter()
    blk = PT.LocalBlock.from_rowgen(N, E, grid.rp, grid.Pr, group=grid.row_group, device=dev, locality=args.locality)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3
    flo, fhi = grid.feature_slice(F, align=16 // esz)
    Fl = fhi - flo
    prop = PT.PartitionedAPPNP(blk, Fl, group=grid.row_group, mode=args.exchange, dtype=dt)
    z0l = torch.zeros((blk.R, prop.ld), dtype=dt, device=dev)
    z0l[: blk.hi - blk.lo, :Fl] = torch.randn(blk.hi - blk.lo, Fl, device=dev,
                                              generator=torch.Generator(device=dev).manual_seed(1 + rank)).to(dt)
    c.step = lambda: prop.run(z0l, hops, 0.0)
    c.outputs = lambda z: {"out": z[: blk.hi - blk.lo, :Fl]}
    z0h = z0l.cpu().pin_memory()
    outh = torch.empty_like(z0h).pin_memory()

    def e2e():
        z0l.copy_(z0h, non_blocking=True)
        outh.copy_(c.step(), non_blocking=True)
        torch.cuda.synchronize()

    c.e2e_step = e2e
    c.h2d = c.d2h = z0l.numel() * esz * world
    c.edges_per_step, c.hops_per_step = blk.nnz_global * hops, hops
    c.launches_per_step = hops * prop.launches_per_hop + 1
    c.hop_bytes = blk.nnz_local * (Fl * esz + 4) + blk.R * Fl * esz + (blk.R + 1) * 8
    c.kernel = "spmm_rows_kernel<bf16,8,...> with the fused peer-store epilogue (+long/combine)"
    c.dtype = "bf16 storage, fp32 accumulate"
    c.config = {"workload": workload_name("papers100m", N, blk.nnz_global), "hops_per_step": hops, "nnz": blk.nnz_global,
                "scale": scale, "parallelism": f"{grid.Pr} row blocks x {grid.Pf} feature slices, exchange={args.exchange}",
                "l2": "inputs larger than L2 (per-GPU iterate copy 28 GB at scale 1)", "graph_build_ms": build_ms,
                "locality": args.locality, "norm": "folded row scaling"}
    c.close = prop.close
    c.keep = (blk, prop, z0l, z0h, outh)
    return c


CASES = {"products": case_products, "arxiv_sage": case_arxiv_sage, "reddit_gat": case_reddit_gat, "papers100m": case_papers100m}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="products", choices=sorted(CASES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-epoch", action="store_true",
                    help="skip the full-batch epoch measurement (the second half of the BASELINE metric) after the timed region")
    ap.add_argument("--fold", type=int, default=1,
                    help="products: 1 (the shim layer's default): D^-1/2 (A+I) D^-1/2 applied as row scalings around an unweighted "
                         "sum (no per-edge weight stream); 0: per-edge gcn_norm weights exactly as PyG multiplies them")
    ap.add_argument("--relabel", type=int, default=1,
                    help="N > 1: 1 = row blocks are runs of whole locality groups (nodes renamed), 0 = id ranges")
    ap.add_argument("--feature-groups", type=int, default=0,
                    help="N>1: Pf of the Pr x Pf process grid (features split Pf ways, rows N/Pf ways); 0 = auto")
    ap.add_argument("--exchange", default="push", choices=["push", "allgather"],
                    help="N>1: fused push of finished rows into every peer over NVLink (default) or NCCL all-gather")
    ap.add_argument("--scale", type=float, default=0.0, help="papers100m: shrink nodes and edges together (0 = full size)")
    ap.add_argument("--locality", type=float, default=0.0, help="papers100m: share of neighbours within +-N/64 of the row")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32, a seeded "
                         "sample of rows where the whole would exceed 60 MiB; with N GPUs, <name>_rank<r>.npy per rank)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    import rgb_experiment_b200 as P

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    nccl_init_ms = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        t0 = time.perf_counter()
        dist.init_process_group("nccl", device_id=dev)
        dist.all_reduce(torch.zeros(1, device=dev))                # communicator set-up is NOT part of the graph build
        torch.cuda.synchronize()
        nccl_init_ms = (time.perf_counter() - t0) * 1e3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    _warm = P.Graph(torch.tensor([[0, 1, 2], [1, 2, 0]], device=dev), 3, P.LOOP_ADD_REMAINING)   # loads the build kernels
    _ = _warm.bwd
    del _warm
    torch.cuda.synchronize()
    wl = args.workload
    c = CASES[wl](args, dev, rank, world)
    if nccl_init_ms is not None:
        c.config["nccl_init_ms"] = nccl_init_ms

    for _ in range(args.warmup):
        c.step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps - 1):
        c.step()
    last = c.step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs:
        outs = c.outputs(last) if c.outputs is not None else {"out": last}
        suffix = f"_rank{rank}" if world > 1 else ""
        dump_outputs(args.dump_outputs, {k + suffix: v for k, v in outs.items()}, budget=DUMP_BYTES // world)
        del outs
    del last
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    gteps = c.edges_per_step * args.steps / (ms * 1e-3) / 1e9

    # ---- e2e: host buffers through the public call, copies inside the timed region ----
    for _ in range(2):
        c.e2e_step()
    n_e2e = max(3, args.steps // 2)
    barrier()
    w0 = time.perf_counter()
    for _ in range(n_e2e):
        c.e2e_step()
    barrier()
    wall = torch.tensor([time.perf_counter() - w0], device=dev)
    if world > 1:
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    wall = float(wall.item())
    e2e = {"value": c.edges_per_step * n_e2e / wall / 1e9, "unit": "GTEPS", "h2d_bytes_per_step": c.h2d,
           "d2h_bytes_per_step": c.d2h, "ms_per_step": wall / n_e2e * 1e3}

    check = c.check() if c.check is not None else None
    l2 = None
    if c.l2_table is not None and rank == 0:
        pk = gather_peak(dev, *c.l2_table)
        ach = c.gathered_bytes_per_step / (ms_per_step * 1e-3) / 1e9
        l2 = {"what": "gathered feature bytes per second vs the device's random row-gather peak for a table of the same size and "
                      "row width (csrc/microbench.cu, measured in this run)", "achieved": ach, "peak": pk, "unit": "GB/s",
              "frac": ach / pk, "table_bytes": c.l2_table[0], "row_bytes": c.l2_table[1]}
    if c.close is not None:
        torch.cuda.synchronize()
        c.close()
    c.keep = None
    c.step = c.e2e_step = c.check = None
    P.graph.clear_cache()
    torch.cuda.empty_cache()
    do_epoch = wl == "products" and not args.no_epoch
    if rank != 0:
        if do_epoch:
            run_epoch_guarded(rank, world, dev, None)
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = peaks()
    hop_ms = ms_per_step / c.hops_per_step
    achieved = c.hop_bytes / (hop_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_kind": peak_kind, "kernel": c.kernel, "bytes_per_launch": c.hop_bytes, "launch_ms": hop_ms,
                "note": "algorithmic bytes = SURVEY 8d gather model, no cache credit: frac > 1 means L2 served part of the gathers; "
                        "`traffic` = DRAM bytes ncu counted for one hop of this workload at this GPU count (null: not captured)"}
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            roofline["traffic"] = (json.load(open(tr)).get(f"{wl}@{world}") or {}).get("hop_bytes_total")
        except Exception:
            pass
    if l2 is not None:
        roofline["l2_gather"] = l2

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline and wl != "papers100m":
        fn, edges, sample, extra = cpu_case(wl, dev)
        fn()
        best, tot0, hops = None, time.perf_counter(), 0
        while hops < 10 and time.perf_counter() - tot0 < 25:
            c0 = time.perf_counter()
            fn()
            dtc = time.perf_counter() - c0
            best = dtc if best is None else min(best, dtc)
            hops += 1
        cpu_baseline = {"value": edges / best / 1e9, "unit": "GTEPS", "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"best of {hops}: " + sample}
        if wl == "products":
            cpu_baseline["strong"] = cpu_strong_baseline(*extra)

    line = {"metric": METRIC[wl], "value": gteps, "unit": "GTEPS", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": c.scaling,
            "vs_baseline": None, "dtype": c.dtype, "data": "synthetic", "config": c.config,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": c.launches_per_step * args.steps, "clocks": sampler.result()}
    if check is not None:
        line["check"] = check
    if do_epoch:
        line["epoch"] = run_epoch_guarded(rank, world, dev, line)
    print(json.dumps(line), flush=True)
    if "error" in (line.get("epoch") or {}):
        os._exit(0)                    # a failed epoch measurement may have left a collective half-entered
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
