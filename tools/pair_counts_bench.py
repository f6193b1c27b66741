"""Per-pair posterior counts on one GPU (mb_pair_counts) against the summed E-step (mb_counts) on the same batch, and against
the route that had to serve per-pair counts before: one mb_counts call per pair, each on a batch of its own.

    python tools/pair_counts_bench.py OUT_DIR [--quick] [--reps N]

Workloads: 4 096 dnapsw pairs of 1 kb (bench.py's E-step shape), 10 000 protpsw pairs of 300 aa, 1 000 PF00516 reads of
50 - 500.  mb_counts and mb_pair_counts alternate, reps times each, after a warm-up call of each on the whole batch (module
loading, the per-pair count module's compilation, scratch allocation).  Device time is mb_last_kernel_ms (CUDA events around
the call's kernels); wall clock is the whole call, the copy of the rows to the host included.  The loop times the first 200
pairs, one batch and one mb_counts call per pair.  Writes OUT_DIR/pair_counts_bench.json with the card's name and power limit
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench  # noqa: E402  (the benchmark's machines and synthetic data)

SEED = 20261022
LOOP_PAIRS = 200


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(call, b):
    t0 = time.perf_counter()
    out = call()
    wall = time.perf_counter() - t0
    ms, launches = b.last_kernel_ms()
    return out, {"kernel_ms": ms, "launches": launches, "wall_s": wall, "redo": b.last_redo()}


def run_workload(capi, name, mj, x, x_off, y, y_off, reps):
    m = bench.make_machine(capi, mj)
    n_pairs = len(x_off) - 1
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    capi.counts(m, b)
    rows = capi.pair_counts(m, b)
    summed, per_pair = [], []
    for _ in range(reps):
        (c, ll), r = timed(lambda: capi.counts(m, b), b)
        summed.append(r)
        (rows, rll), r = timed(lambda: capi.pair_counts(m, b, loglike=True), b)
        per_pair.append(r)
    scale = max(1.0, float(np.abs(c).max()))
    check = {"max_abs_diff_sum_of_rows_vs_counts_over_max_count": float(np.abs(rows.sum(axis=0) - c).max() / scale),
             "loglike_bit_identical": bool(np.array_equal(ll, rll))}
    # the route before: a batch and an mb_counts call per pair
    n_loop = min(LOOP_PAIRS, n_pairs)
    one = lambda k: capi.Batch(x=x[x_off[k]:x_off[k + 1]], x_off=np.array([0, x_off[k + 1] - x_off[k]], np.int64),
                               y=y[y_off[k]:y_off[k + 1]], y_off=np.array([0, y_off[k + 1] - y_off[k]], np.int64))
    capi.counts(m, one(0))
    loop_ms, t0 = 0.0, time.perf_counter()
    for k in range(n_loop):
        bk = one(k)
        capi.counts(m, bk)
        loop_ms += bk.last_kernel_ms()[0]
        bk.close()
    loop_wall = time.perf_counter() - t0
    best = lambda runs: min(runs, key=lambda r: r["kernel_ms"])
    out = {"workload": name, "pairs": n_pairs, "transitions": int(len(mj["lw"])), "states": mj["n_states"], "engine": m.engine,
           "mb_counts_runs": summed, "mb_pair_counts_runs": per_pair,
           "mb_counts_kernel_ms": best(summed)["kernel_ms"], "mb_pair_counts_kernel_ms": best(per_pair)["kernel_ms"],
           "mb_counts_wall_s": min(r["wall_s"] for r in summed), "mb_pair_counts_wall_s": min(r["wall_s"] for r in per_pair),
           "loop": {"pairs": n_loop, "wall_s": loop_wall, "wall_s_per_pair": loop_wall / n_loop, "kernel_ms_per_pair": loop_ms / n_loop},
           "check": check}
    out["pair_counts_over_counts_kernel"] = out["mb_pair_counts_kernel_ms"] / out["mb_counts_kernel_ms"]
    out["batched_wall_s_per_pair"] = out["mb_pair_counts_wall_s"] / n_pairs
    b.close()
    m.close()
    print(json.dumps({k: v for k, v in out.items() if not k.endswith("_runs")}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--quick", action="store_true", help="a tenth of each workload")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    from machineboss_b200 import capi
    scale = 10 if args.quick else 1
    result = {"card": card(), "workloads": []}
    print(json.dumps(result["card"]), flush=True)

    # dnapsw: 1 kb pairs, each output its input with 10 % substitutions and 2 % indels
    mj = bench.eval_machine("dnapsw")
    n = 4096 // scale
    x, x_off, _, _ = bench.synth_batch(SEED, 0, n, 1000, 1000, 4)
    y, y_off = bench.mutate_batch(SEED, x, x_off, 4)
    result["workloads"].append(run_workload(capi, "dnapsw, %d pairs of 1 kb" % n, mj, x, x_off, y, y_off, args.reps))

    # protpsw: 300 aa pairs
    mj = bench.eval_machine("protpsw")
    n = 10000 // scale
    x, x_off, _, _ = bench.synth_batch(SEED + 1, 0, n, 300, 300, 20)
    y, y_off = bench.mutate_batch(SEED + 1, x, x_off, 20)
    result["workloads"].append(run_workload(capi, "protpsw, %d pairs of 300 aa" % n, mj, x, x_off, y, y_off, args.reps))

    # PF00516 profile: reads of 50 - 500 residues, no input sequence
    mj = bench.eval_machine("PF00516")
    n = 1000 // scale
    lens = 50 + (np.arange(n, dtype=np.int64) * 7919) % 451
    y, y_off = bench.synth_ragged(SEED + 2, lens, mj["n_out"])
    result["workloads"].append(run_workload(capi, "PF00516, %d reads of 50 - 500" % n, mj, np.zeros(0, np.uint8), np.zeros(n + 1, np.int64),
                                            y, y_off, args.reps))

    result["card_after"] = card()
    with open(os.path.join(args.out_dir, "pair_counts_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
