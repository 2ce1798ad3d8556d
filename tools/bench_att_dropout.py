"""One training step (forward + backward) of a fused attention layer in three attention-dropout modes, alternated
in one process:

    none    no dropout
    torch   F.dropout on an edge-sized ones tensor, passed as drop_edge (what the shim layers do by default)
    fused   dropout_p: the mask is generated inside the kernels from a device seed (ops.FUSED_DROPOUT = True)

Workloads: SuperGAT-MX 8x8 and GAT 8x8 on the Reddit-shaped synthetic graph, FAConv F = 64 on the products-shaped
one.  Prints per workload and mode: ms per step (CUDA events, median over --steps after --warmup), ms of the fused
forward kernels alone (torch.profiler, a separate pass), and the peak allocated bytes above the allocation before
the step.  Needs a CUDA device.

    python tools/bench_att_dropout.py [--steps 30] [--warmup 5] [--p 0.5] [--workloads mx,fa,gat]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys
import warnings

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rgb_experiment_b200 as P  # noqa: E402
import rgb_experiment_b200.synth as S  # noqa: E402

DEV = "cuda:0"
MODES = ("none", "torch", "fused")
WORKLOADS = {                      # name: (graph, op, H, C)
    "mx": ("reddit", "supergat_mx", 8, 8),
    "fa": ("products", "faconv", 1, 64),
    "gat": ("reddit", "gat", 8, 8),
}


def make_workload(key):
    gname, op, H, C = WORKLOADS[key]
    sg = S.make_named(gname, features=False, device=DEV)
    n = sg.num_nodes
    loop = P.LOOP_ADD_REMAINING if op == "faconv" else P.LOOP_REMOVE_THEN_ADD
    g = P.Graph(sg.edge_index, n, loop)
    del sg
    g.bwd, g.dinv(), g.tpos()                                # graph-side caches built once, outside the steps
    gen = torch.Generator(device=DEV).manual_seed(0)
    ins = [torch.randn(n, H * C, device=DEV, generator=gen), torch.randn(n, H, device=DEV, generator=gen),
           torch.randn(n, H, device=DEV, generator=gen)]
    dout = torch.randn(n, H * C, device=DEV, generator=gen)
    return gname, op, H, C, g, ins, dout


def step_fn(op, H, C, g, ins, dout, mode, p):
    def forward(xs):
        kw = {}
        if mode == "fused":
            kw = dict(dropout_p=p)
        elif mode == "torch":
            shape = (g.nnz,) if op == "faconv" else (g.nnz, H)
            kw = dict(drop_edge=F.dropout(torch.ones(shape, device=DEV), p=p, training=True))
        if op == "faconv":
            return P.ops.faconv(*xs, g, **kw)
        return getattr(P.ops, op)(*xs, g, H, C, 0.2, **kw)

    def run():
        xs = [t.requires_grad_(True) for t in ins]
        out = forward(xs)
        out.backward(dout)
        for t in xs:
            t.grad = None
    return run


def time_steps(fns, steps, warmup):
    for _ in range(warmup):
        for f in fns.values():
            f()
    times = {m: [] for m in fns}
    peaks = {m: 0 for m in fns}
    for _ in range(steps):
        for m, f in fns.items():                            # modes alternated within every repetition
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1))
            peaks[m] = max(peaks[m], torch.cuda.max_memory_allocated() - base)
    return times, peaks


def forward_kernel_ms(fns, reps=5):
    """device time of the att_fwd_* kernels per step, from a profiler pass of its own"""
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", message=".*Profiler clears events")
    res = {}
    for m, f in fns.items():
        f()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                f()
            torch.cuda.synchronize()
        us = sum(e.device_time_total for e in prof.key_averages() if "att_fwd" in e.key)
        res[m] = us / 1000.0 / reps
    return res


def device_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"device: {name} ({q})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--p", type=float, default=0.5)
    ap.add_argument("--workloads", default="mx,fa,gat")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_att_dropout: needs a CUDA device")
    if a.steps < 20:
        raise SystemExit("bench_att_dropout: --steps must be at least 20")
    print(device_line())
    print(f"p = {a.p}, {a.steps} timed steps after {a.warmup} warm-up steps, modes alternated; step = forward + backward")
    for key in a.workloads.split(","):
        gname, op, H, C, g, ins, dout = make_workload(key)
        fns = {m: step_fn(op, H, C, g, ins, dout, m, a.p) for m in MODES}
        times, peaks = time_steps(fns, a.steps, a.warmup)
        fwd = forward_kernel_ms(fns)
        edge_bytes = g.nnz * H * 4
        print(f"\n{op} H={H} C={C} on {gname}-shaped graph: N={g.N:,} nnz={g.nnz:,} ([nnz,H] fp32 = {edge_bytes / 1e9:.2f} GB)")
        print(f"  {'mode':6s} {'ms/step (median)':>17s} {'min':>8s} {'fwd kernels ms':>15s} {'peak above base GB':>19s}")
        for m in MODES:
            t = times[m]
            print(f"  {m:6s} {statistics.median(t):17.3f} {min(t):8.3f} {fwd[m]:15.3f} {peaks[m] / 1e9:19.3f}")
        del g, ins, dout, fns
        P.graph.clear_cache()
        P.memo.clear()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
