"""SuperGATConv's SD attention (ops.supergat_sd) two ways, alternated in one process:

    fused   the RGBMP_ATT_SD kernels of csrc/att.cu: one forward pass, one backward pass per orientation, dropout
            generated inside the kernels -- nothing edge-sized
    chain   what the layer ran before: edge_sddmm / sqrt(C), leaky_relu, edge_softmax, the [nnz, H] dropout mask
            (rgbmp_dropout_mask of the same seed) and spmm_heads, each an [nnz, H] tensor

Shapes: the first layer's 8 heads x 8 and the second layer's 8 heads x classes with concat=False (head mean);
graphs: the arxiv-, Reddit- and products-shaped synthetic graphs (rgb_experiment_b200.synth).  Per shape, graph and
mode (eval forward; forward + backward at dropout 0 and 0.5): ms per call (CUDA events, median over --steps after
--warmup) and the peak allocated bytes above the allocation before the call.  Before a time is reported, the fused
output is checked against the chain's on the timed inputs (norm-wise relative error <= 1e-5).  With backward the
x-gradient difference is reported beside the number of logits within 1e-6 of leaky_relu's kink: there the two
fp32 summation orders can land on opposite sides of 0 and take different slopes, so that difference is not gated.
The chain only runs where its bytes, computed from the shapes, fit the free device memory;
otherwise the line says how much it would need.  The fused MX layer on the same inputs (a_l, a_r drawn at random)
is timed alongside as the comparison.  The eval memo is off, so every eval call computes.  Needs a CUDA device.

    python tools/bench_supergat_sd.py [--steps 20] [--warmup 3] [--graphs arxiv,reddit,products] [--out FILE]
"""
from __future__ import annotations

import argparse
import math
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rgb_experiment_b200 as P  # noqa: E402
import rgb_experiment_b200.synth as S  # noqa: E402

DEV = "cuda:0"
H = 8
SLOPE = 0.2
MODES = (("eval", 0.0), ("train", 0.0), ("train", 0.5))
TOL = 1e-5


def device_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"device: {name} ({q})"


def chain_bytes(nnz, train):
    """[nnz, H] fp32 tensors the chain holds at its peak, from the shapes: logits, scaled logits, leaky_relu,
    softmax (+ mask and masked weights); the backward adds their gradients while the saved ones live."""
    return (8 if train else 4) * nnz * H * 4


def relerr(a, b):
    a, b = a.double(), b.double()
    den = b.abs().max().item()
    return (a - b).abs().max().item() / (den if den > 0 else 1.0)


def sd_chain(xp, g, C, p, seed):
    a = F.leaky_relu(P.ops.edge_sddmm(xp, xp, g, H, C) / math.sqrt(C), SLOPE)
    alpha = P.ops.edge_softmax(a, g)
    if p > 0:
        alpha = alpha * g.to_csr_order(P.ops.dropout_mask(g, H, p, P.ops.dropout_seed(DEV, seed())))
    return P.ops.spmm_heads(alpha, xp, g, H, C)


def call_fn(impl, mode, p, g, C, concat, x, a_l, a_r, dout):
    """one call: returns (out, x.grad or None)"""
    def seed():
        return torch.Generator(device=DEV).manual_seed(1234)        # the same multipliers for fused and chain

    def op(xp):
        if impl == "fused":
            out = P.ops.supergat_sd(xp, g, H, C, SLOPE, dropout_p=p, generator=seed() if p > 0 else None)
        elif impl == "mx":
            out = P.ops.supergat_mx(xp, a_l, a_r, g, H, C, SLOPE)
        else:
            out = sd_chain(xp, g, C, p, seed)
        return out if concat else out.view(-1, H, C).mean(dim=1)

    def run():
        if mode == "eval":
            with torch.no_grad():
                return op(x), None
        xs = x.detach().requires_grad_(True)
        out = op(xs)
        out.backward(dout)
        return out.detach(), xs.grad
    return run


def time_calls(fns, steps, warmup):
    for _ in range(warmup):
        for f in fns.values():
            f()
    times = {k: [] for k in fns}
    peaks = {k: 0 for k in fns}
    for _ in range(steps):
        for k, f in fns.items():                               # implementations alternated within every repetition
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = f()
            e1.record()
            torch.cuda.synchronize()
            del r
            times[k].append(e0.elapsed_time(e1))
            peaks[k] = max(peaks[k], torch.cuda.max_memory_allocated() - base)
    return times, peaks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--graphs", default="arxiv,reddit,products")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_supergat_sd: needs a CUDA device")
    fout = open(a.out, "w") if a.out else None

    def emit(s=""):
        print(s, flush=True)
        if fout:
            fout.write(s + "\n")
            fout.flush()

    P.memo.set_budget_mb(0)
    emit(device_line())
    emit(f"SuperGATConv SD attention + aggregate, fused vs chain (and fused MX on the same inputs); {a.steps} timed "
         f"calls after {a.warmup} warm-up calls, implementations alternated; out err: fused vs chain, norm-wise, "
         f"must be <= {TOL:g}; grad err: x-gradient, fused vs chain; kink: logits with |<x_i,x_j>/sqrt(C)| < 1e-6")
    for gname in a.graphs.split(","):
        n, _, _, classes = S.SHAPES[gname]
        sg = S.make_named(gname, features=False, device=DEV)
        g = P.Graph(sg.edge_index, n, P.LOOP_REMOVE_THEN_ADD)
        del sg
        g.bwd, g.tpos()                                        # graph-side caches built once, outside the calls
        emit(f"\n{gname}-shaped graph: N={n:,} nnz={g.nnz:,} ([nnz, H] fp32 = {g.nnz * H * 4 / 1e9:.2f} GB)")
        emit(f"  {'shape':13s} {'mode':12s} {'impl':6s} {'ms (median)':>12s} {'min':>8s} {'peak above start GB':>20s} "
             f"{'out err':>9s} {'grad err':>9s} {'kink':>6s}")
        for C, concat in ((8, True), (classes, False)):
            gen = torch.Generator(device=DEV).manual_seed(C)
            x = torch.randn(n, H * C, device=DEV, generator=gen) * 0.5
            a_l, a_r = torch.randn(n, H, device=DEV, generator=gen), torch.randn(n, H, device=DEV, generator=gen)
            dout = torch.randn(n, H * C if concat else C, device=DEV, generator=gen)
            shape = f"{H}x{C}" + ("" if concat else " mean")
            for mode, p in MODES:
                train = mode == "train"
                free = torch.cuda.mem_get_info()[0]
                need = chain_bytes(g.nnz, train)
                impls = ["fused"] + (["chain"] if need < 0.8 * free else []) + (["mx"] if p == 0 else [])
                fns = {k: call_fn(k, mode, p, g, C, concat, x, a_l, a_r, dout) for k in impls}
                check = ""
                if "chain" in fns:                              # on the timed inputs, before any time is reported
                    fo, fg = fns["fused"]()
                    co, cg = fns["chain"]()
                    err = relerr(fo, co)
                    if not err <= TOL:
                        raise SystemExit(f"{gname} {shape} {mode} p={p}: fused vs chain relative error {err:.3g} > {TOL:g}")
                    check = f"{err:9.1e}"
                    if fg is not None:
                        with torch.no_grad():
                            kink = int((P.ops.sddmm(g.fwd, x, x, H, C).abs() < 1e-6 * math.sqrt(C)).sum())
                        check += f" {relerr(fg, cg):9.1e} {kink:6d}"
                    del fo, fg, co, cg
                times, peaks = time_calls(fns, a.steps, a.warmup)
                label = "eval fwd" if not train else f"fwd+bwd p{p:g}"
                for k in impls:
                    t = times[k]
                    emit(f"  {shape:13s} {label:12s} {k:6s} {statistics.median(t):12.3f} {min(t):8.3f} "
                         f"{peaks[k] / 1e9:20.3f} {check if k == 'chain' else ''}")
                if "chain" not in fns:
                    emit(f"  {shape:13s} {label:12s} chain  not run: needs {need / 1e9:.1f} GB ({free / 1e9:.1f} GB free)")
                del fns
            del x, a_l, a_r, dout
        del g
        P.graph.clear_cache()
        torch.cuda.empty_cache()
    emit()
    emit(device_line())
    if fout:
        fout.close()


if __name__ == "__main__":
    main()
