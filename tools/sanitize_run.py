#!/usr/bin/env python
"""The small-graph workout for memory-safety checking (SURVEY.md section 5 "race detection"; VERDICT r1 item 7):
every kernel family of librgbmp.so on the edge-case graphs of tests/helpers.CASES -- graph build (all three radix
variants), loop edits, coalesce, locality groups, SpMM (vector, scalar / unaligned, bf16, long rows, every epilogue),
K-hop (fp32 and bf16), fused attention forward + backward for GAT / SuperGAT-MX / FAConv (all head shape classes, long rows), the
generic edge-score kernels.  Every result and gradient is checked to be finite.

Meant for   compute-sanitizer --tool memcheck|racecheck|initcheck python tools/sanitize_run.py   (one tool per call).
On this pool compute-sanitizer is CLOSED (gpurun answers "closed ... stays closed: runs under it have left GPUs
needing a reset", profiles/r02_sanitizer.txt), so tests/test_gpu_guard_bands.py runs the same workout with every
device allocation wrapped in canary guard bands and NaN-poisoned payloads instead.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def fin(t):
    """Results and gradients must be finite: a read of poisoned (uninitialised / out-of-bounds) memory is not."""
    if isinstance(t, tuple):
        for v in t:
            fin(v)
        return t
    assert torch.isfinite(t.float()).all(), "non-finite value"
    return t


def back(y, *leaves):
    fin(y).sum().backward()
    for v in leaves:
        fin(v.grad)
        v.grad = None


def main():
    import rgb_experiment_b200 as P
    from rgb_experiment_b200 import graph as G
    import rgb_experiment_b200.shim.utils as U
    from helpers import CASES
    dev = torch.device("cuda:0")
    G.CLUSTER_SEEDS = 16
    n_calls = 0
    for variant in ("3", "1", "2"):
        os.environ["RGBMP_BUILD_VARIANT"] = variant
        for name in ("tiny", "loops_dups", "isolated", "hub", "empty", "single_node"):
            ei, n = CASES[name]()
            for mode in (P.LOOP_NONE, P.LOOP_ADD, P.LOOP_ADD_REMAINING, P.LOOP_REMOVE_THEN_ADD):
                g = P.Graph(ei.to(dev), n, mode)
                _ = g.bwd
                n_calls += 1
    os.environ["RGBMP_BUILD_VARIANT"] = "3"
    for name in ("loops_dups", "isolated", "hub"):
        ei, n = CASES[name]()
        eid = ei.to(dev)
        U.to_undirected(eid, n)
        U.coalesce(eid, None, n, n)
        G.CLUSTER = "1"
        g = P.Graph(eid, n, P.LOOP_ADD_REMAINING)              # locality groups forced on: LPA + connectivity + grouped order
        G.CLUSTER = "auto"
        gn = P.Graph(eid, n, P.LOOP_NONE)
        gr = P.Graph(eid, n, P.LOOP_REMOVE_THEN_ADD)
        gen = torch.Generator(device=dev).manual_seed(0)
        for F, dt in ((48, torch.float32), (23, torch.float32), (7, torch.float32), (100, torch.float32), (260, torch.float32),
                      (64, torch.bfloat16)):
            x = torch.randn(n, F, device=dev, generator=gen).to(dt)
            if dt == torch.float32:
                x.requires_grad_(True)
                for kind in ("sum", "mean", "gcn"):
                    back(P.ops.propagate(x, g, kind), x)
                back(P.ops.appnp(x, g, 3, 0.1, False), x)
                back(P.ops.appnp(x, g, 3, 0.1, True), x)
                fin(P.ops.gcn_power(x.detach(), g, 2))
                m = torch.zeros(n, dtype=torch.bool, device=dev)
                m[::3] = True
                fin(P.ops.label_propagation(gn, x.detach(), 3, 0.8, clamp=(-1.0, 1.0)))
                fin(P.ops.label_propagation(gn, x.detach(), 3, 0.8, reset_mask=m, reset_val=x.detach()))
                w = torch.rand(g.nnz, device=dev, generator=gen, requires_grad=True)
                back(P.ops.propagate_weighted(x, w, g), x, w)
                if F <= 16:                                    # the same K-hop families on the K-launch path (cluster path off)
                    L_ = P._lib.lib()
                    old = L_.rgbmp_set_khop_cta(0)
                    try:
                        fin(P.ops.appnp(x.detach(), g, 3, 0.1))
                        fin(P.ops.label_propagation(gn, x.detach(), 3, 0.8, clamp=(-1.0, 1.0)))
                    finally:
                        L_.rgbmp_set_khop_cta(old)
                # fused all-gather epilogue into two local "peer" copies, as stores and as bulk (TMA) copies
                d = g.dinv()
                xb, ldx = P.ops.as_rows(x.detach())
                ldp = P.ops.padded_width(F, dt)
                for bulk in (0, 1):
                    oldb = P._lib.lib().rgbmp_set_push_bulk(bulk)
                    try:
                        bufs = [torch.zeros((n + 4, ldp), dtype=dt, device=dev) for _ in range(2)]
                        ep = P.ops.make_epilogue(row_scale=d, out2_scale=d, a=0.9, b=0.1, T=xb, ldt=ldx,
                                                 peers=[b_.data_ptr() for b_ in bufs], peer_row0=2, ld_peer=ldp)
                        P.ops.spmm_raw(g.fwd, x.detach(), None, ep=ep, keep=(xb, d, bufs), store_local=False)
                        for b_ in bufs:
                            fin(b_)
                    finally:
                        P._lib.lib().rgbmp_set_push_bulk(oldb)
            else:
                fin(P.ops.spmm_raw(g.fwd, x, None))
                # bf16 K-hop (always the K-launch driver), every epilogue form, reset rows (read as fp32)
                d = g.dinv()
                xb, ldx = P.ops.as_rows(x)
                m = torch.zeros(n, dtype=torch.bool, device=dev)
                m[::3] = True
                m8, rv = m.to(torch.uint8), x.float()
                fin(P.ops.spmm_raw(g.fwd, x, g.gcn_val(False), ep=P.ops.make_epilogue(
                    row_scale=d, a=0.9, b=0.1, T=xb, ldt=ldx, clamp=(-1.0, 1.0), acc_in=xb, ld_acc=ldx,
                    reset_mask=m8, reset_val=rv, ld_reset=F, reset_when=2), keep=(xb, d, m8, rv)))
                for fold in (False, True):
                    fin(P.ops.appnp(x, g, 3, 0.1, fold))
                    fin(P.ops.gcn_power(x, g, 2, fold))
                    fin(P.ops.label_propagation(gn, x, 3, 0.8, clamp=(-1.0, 1.0), fold=fold))
                    fin(P.ops.label_propagation(gn, x, 3, 0.8, reset_mask=m, reset_val=x, fold=fold))
                fin(P.ops.dagnn_hops(x, g, 3))
            n_calls += 8
        for H, C in ((8, 8), (1, 41), (3, 5), (5, 32), (2, 47)):
            xp = (torch.randn(n, H * C, device=dev, generator=gen) * 0.5).requires_grad_(True)
            a = torch.randn(n, H, device=dev, generator=gen, requires_grad=True)
            b = torch.randn(n, H, device=dev, generator=gen, requires_grad=True)
            keep = (torch.rand(gr.nnz, H, device=dev, generator=gen) > 0.3).float() / 0.7
            for drop in (None, keep):
                back(P.ops.gat(xp, a, b, gr, H, C, 0.2, drop), xp, a, b)
                back(P.ops.supergat_mx(xp, a, b, gr, H, C, 0.2, drop), xp, a, b)
            with torch.no_grad():
                fin(P.ops.gat(xp, a, b, gr, H, C, 0.2))
                fin(P.ops.supergat_mx(xp, a, b, gr, H, C, 0.2))
            n_calls += 6
        for C in (64, 7):
            x = torch.randn(n, C, device=dev, generator=gen, requires_grad=True)
            al = torch.randn(n, 1, device=dev, generator=gen, requires_grad=True)
            ar = torch.randn(n, 1, device=dev, generator=gen, requires_grad=True)
            back(P.ops.faconv(x, al, ar, g), x, al, ar)
            back(P.ops.faconv(x, al, ar, g, (torch.rand(g.nnz, device=dev, generator=gen) > 0.5).float() * 2), x, al, ar)
        A = torch.randn(n, 18, device=dev, generator=gen, requires_grad=True)
        s = P.ops.edge_sddmm(A, A, gn, 3, 6)
        back(P.ops.spmm_heads(P.ops.edge_softmax(s, gn), A, gn, 3, 6), A)
        u = torch.randn(n, 3, device=dev, generator=gen, requires_grad=True)
        back(P.ops.edge_u_add_v(u, u, gn), u)
    torch.cuda.synchronize()
    print(f"sanitize_run ok: {n_calls} op groups")
    return n_calls


if __name__ == "__main__":
    main()
