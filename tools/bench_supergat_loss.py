"""One training step (forward, loss, backward) of the reference's two-layer SuperGAT model (in -> 8 heads x 8 -> 8
heads x classes with concat=False, MX attention, edge_sample_ratio 1.0, neg_sample_ratio 0.5, attention dropout 0)
with its self-supervised attention loss computed two ways, alternated in one process:

    torch   the shim's default: to_undirected + torch negative sampling + [pairs, H, C] gathers and autograd
    fused   ops.FUSED_SUPERGAT_LOSS: cached U, device sampler, fused pair-logit BCE (csrc/supergat_loss.cu)

Graphs: arxiv-, Reddit- and products-shaped synthetic graphs (rgb_experiment_b200.synth).  Per graph and mode: ms per
step (CUDA events, median over --steps after --warmup), the peak allocated bytes above the allocation before the step,
and, from separate passes, the ms of the new kernels alone (torch.profiler, every sgat_* kernel) and of the sampler
alone (CUDA events around ops.supergat_samples' negatives).  The torch mode only runs where its bytes, computed from
the shapes, fit the free device memory; otherwise the line says how much it would need.  Needs a CUDA device.

    python tools/bench_supergat_loss.py [--steps 20] [--warmup 3] [--graphs arxiv,reddit,products] [--out FILE]
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
from rgb_experiment_b200.shim import nn as PL  # noqa: E402

DEV = "cuda:0"
H, HID = 8, 8
LAMBDA = 4.0
MODES = ("torch", "fused")


class Net(torch.nn.Module):
    def __init__(self, fin, classes):
        super().__init__()
        self.c1 = PL.SuperGATConv(fin, HID, heads=H, dropout=0.0, attention_type="MX")
        self.c2 = PL.SuperGATConv(H * HID, classes, heads=H, concat=False, dropout=0.0, attention_type="MX")

    def forward(self, x, ei):
        h = F.elu(self.c1(x, ei))
        return F.log_softmax(self.c2(h, ei), dim=-1)


def step_fn(model, x, y, ei, mode):
    def run():
        P.ops.FUSED_SUPERGAT_LOSS = mode == "fused"
        try:
            out = model(x, ei)
            loss = F.nll_loss(out, y) + LAMBDA * (model.c1.get_attention_loss() + model.c2.get_attention_loss())
            loss.backward()
            model.zero_grad(set_to_none=True)
            model.c1.att_x = model.c1.att_y = model.c2.att_x = model.c2.att_y = None
            model.c1._att_loss = model.c2._att_loss = None
            return float(loss)
        finally:
            P.ops.FUSED_SUPERGAT_LOSS = False
    return run


def torch_bytes(nnz, n, fin, classes):
    """What the torch loss keeps alive or builds per step, from the shapes: per layer two [pairs, F] gathers and
    their product for the positives and the negatives, plus the 2 nnz coalesce of to_undirected (int64 pairs,
    sort keys and permutations)."""
    pairs = nnz + nnz // 2
    per_layer = [3 * pairs * H * HID * 4, 3 * pairs * H * classes * 4]
    return sum(per_layer) + 2 * nnz * 8 * 6


def device_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"device: {name} ({q})"


def time_steps(fns, steps, warmup, emit):
    for _ in range(warmup):
        for f in fns.values():
            f()
    times = {m: [] for m in fns}
    peaks = {m: 0 for m in fns}
    losses = {m: None for m in fns}
    emit(device_line())
    for _ in range(steps):
        for m, f in fns.items():                            # modes alternated within every repetition
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            losses[m] = f()
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1))
            peaks[m] = max(peaks[m], torch.cuda.max_memory_allocated() - base)
    return times, peaks, losses


def kernel_ms(f, reps=3):
    """device time of the sgat_* kernels per step, from a profiler pass of its own"""
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", message=".*Profiler clears events")
    f()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            f()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if "sgat_" in e.key) / 1000.0 / reps


def sampler_ms(g, reps=10):
    """one layer's negatives (0.5 nnz of them) from the cached U, CUDA events, median"""
    g.undirected_csr(True)
    num = int(0.5 * 1.0 * g.nnz)
    out = []
    for r in range(reps + 2):
        seed = P.ops.dropout_seed(DEV)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        P.ops._sgat_negatives(g, seed, num, False)
        e1.record()
        torch.cuda.synchronize()
        if r >= 2:
            out.append(e0.elapsed_time(e1))
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--graphs", default="arxiv,reddit,products")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_supergat_loss: needs a CUDA device")
    fout = open(a.out, "w") if a.out else None

    def emit(s=""):
        print(s, flush=True)
        if fout:
            fout.write(s + "\n")
            fout.flush()

    emit(device_line())
    emit(f"two-layer SuperGAT (MX, {H} heads x {HID} -> {H} heads x classes, concat=False), loss = NLL + {LAMBDA} x "
         f"attention losses; {a.steps} timed steps after {a.warmup} warm-up steps, modes alternated")
    for gname in a.graphs.split(","):
        n, _, fin, classes = S.SHAPES[gname]
        sg = S.make_named(gname, device=DEV)
        ei, x, y = sg.edge_index, sg.x, sg.y
        del sg
        torch.manual_seed(0)
        model = Net(fin, classes).to(DEV).train()
        g = P.get_graph(ei, n, P.LOOP_REMOVE_THEN_ADD)
        g.bwd, g.undirected_csr(True)                      # graph-side caches built once, outside the steps
        need = torch_bytes(g.nnz, n, fin, classes)
        free = torch.cuda.mem_get_info()[0]
        modes = [m for m in MODES if m == "fused" or need < 0.8 * free]
        emit(f"\n{gname}-shaped graph: N={n:,} nnz={g.nnz:,} F_in={fin} classes={classes}")
        if "torch" not in modes:
            emit(f"  torch  not run: needs {need / 1e9:.1f} GB ({free / 1e9:.1f} GB free)")
        fns = {m: step_fn(model, x, y, ei, m) for m in modes}
        times, peaks, losses = time_steps(fns, a.steps, a.warmup, emit)
        emit(f"  {'mode':6s} {'ms/step (median)':>17s} {'min':>8s} {'sgat kernels ms':>16s} {'share':>6s} "
             f"{'peak above base GB':>19s} {'loss':>10s}")
        for m in modes:
            t = times[m]
            kms = kernel_ms(fns[m]) if m == "fused" else float("nan")
            share = kms / statistics.median(t) if m == "fused" else float("nan")
            emit(f"  {m:6s} {statistics.median(t):17.3f} {min(t):8.3f} {kms:16.3f} {share:6.1%} "
                 f"{peaks[m] / 1e9:19.3f} {losses[m]:10.5f}")
        emit(f"  sampler alone (one layer's {int(0.5 * g.nnz):,} negatives): {sampler_ms(g):.3f} ms")
        del model, g, fns, ei, x, y
        P.graph.clear_cache()
        P.memo.clear()
        torch.cuda.empty_cache()
    if fout:
        fout.close()


if __name__ == "__main__":
    main()
