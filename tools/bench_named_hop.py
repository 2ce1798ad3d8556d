#!/usr/bin/env python
"""Does naming the nodes in schedule order make the one-GPU K-hop faster?  Times ops._appnp_khop (APPNP K=10,
folded) on the products-shaped graph with ops.NAMED_KHOP off (the graph as built: locality-grouped schedule, nodes
keep their ids) and on (Graph.named_fwd: nodes renamed pos = inverse(row_order), identity schedule; the input is
renamed by the staging pass and the result by the last hop's store, both inside the timed call).  Repetitions
alternate between the two; the outputs must be bit-identical.
    python tools/bench_named_hop.py [--reps 5] [--calls 10] [--F 47]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # noqa: BLE001 -- the card's name still comes from torch
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10, help="K-hop calls per timed repetition")
    ap.add_argument("--F", type=int, default=47)
    ap.add_argument("--K", type=int, default=10)
    args = ap.parse_args()
    import rgb_experiment_b200 as P
    import rgb_experiment_b200.synth as S
    dev = torch.device("cuda:0")
    sg = S.make_named("products", seed=20261018, device=dev, features=False)     # bench.py's GRAPH_SEED
    N = sg.num_nodes
    g = P.Graph(sg.edge_index, N, P.LOOP_ADD_REMAINING)
    if not g.fwd.clustered:
        raise SystemExit("the graph has no locality-grouped schedule: nothing to rename")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nf = g.named_fwd
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3

    x = torch.randn(N, args.F, device=dev, generator=torch.Generator(device=dev).manual_seed(1))

    def run(named):
        P.ops.NAMED_KHOP = named
        return P.ops._appnp_khop(g.fwd, g, x, args.K, 0.1, False, True)

    y_old, y_new = run(False), run(True)
    torch.cuda.synchronize()
    equal = bool(torch.equal(y_new, y_old))
    for _ in range(3):
        run(False)
        run(True)
    torch.cuda.synchronize()

    def timed(named):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.calls):
            run(named)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.calls

    old, new = [], []
    for _ in range(args.reps):
        old.append(timed(False))
        new.append(timed(True))
    res = {"card": card(), "N": N, "nnz": g.nnz, "F": args.F, "K": args.K, "calls_per_rep": args.calls,
           "n_long_rows": g.fwd.n_long, "n_items": g.fwd.n_items, "named_fwd_build_ms": round(build_ms, 1),
           "old_ms_per_call": [round(v, 3) for v in old], "named_ms_per_call": [round(v, 3) for v in new],
           "old_ms_per_hop_mean": round(sum(old) / len(old) / args.K, 4),
           "named_ms_per_hop_mean": round(sum(new) / len(new) / args.K, 4),
           "gain_mean": round(1 - sum(new) / sum(old), 4),
           "gain_worst_case": round(1 - max(new) / min(old), 4),
           "outputs_bit_equal": equal}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
