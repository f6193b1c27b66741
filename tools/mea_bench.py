"""Posterior decoding on one GPU: device time of mb_mea (the Forward and Backward fills, the MEA fill and both traceback passes)
and of mb_path_posteriors on each pair's Viterbi path (the two fills and the path walk), on three workloads.

    python tools/mea_bench.py OUT_DIR [--quick] [--reps N]

Writes OUT_DIR/mea_bench.json with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))

import bench  # noqa: E402  (the benchmark's machines and synthetic data)
from sample_paths_bench import card, chunk_plan, free_bytes  # noqa: E402

SEED = 20261022


def timed(b, reps, call):
    """Runs call() reps times; per run the device time of its kernels (mb_last_kernel_ms) and the wall clock."""
    runs, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = call()
        wall = time.perf_counter() - t0
        ms, launches = b.last_kernel_ms()
        runs.append({"kernel_ms": ms, "launches": launches, "wall_s": wall})
    return out, runs, min(runs, key=lambda r: r["kernel_ms"])


def run_workload(capi, name, mj, x, x_off, y, y_off, reps):
    m = bench.make_machine(capi, mj)
    n_pairs = len(x_off) - 1
    warm = capi.Batch(x=x, x_off=x_off[:9] - x_off[0], y=y, y_off=y_off[:9] - y_off[0])      # first launches: module loading
    capi.mea(m, warm)
    warm.close()
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    free = free_bytes()
    (gain, ll, lengths, off, ids, post), mea_runs, mea_best = timed(b, reps, lambda: capi.mea(m, b))
    score, vpaths = capi.viterbi(m, b)
    keep = np.nonzero(np.isfinite(score))[0]
    voff = np.concatenate([[0], np.cumsum([len(vpaths[k]) for k in keep])]).astype(np.int64)
    vids = np.concatenate([vpaths[k] for k in keep] + [np.zeros(0, np.int32)])
    vpost, pp_runs, pp_best = timed(b, reps, lambda: capi.path_posteriors(m, b, keep, voff, vids))
    c = (np.asarray(mj["tin"])[vids] > 0).astype(np.float64) + (np.asarray(mj["tout"])[vids] > 0)
    vgain = np.bincount(np.repeat(np.arange(len(keep)), np.diff(voff)), weights=c * vpost, minlength=len(keep))
    fin = np.isfinite(gain)
    tokens = (np.diff(x_off) + np.diff(y_off)).astype(np.float64)
    out = {"workload": name, "pairs": n_pairs, "states": mj["n_states"], "cell_states": float(b.cell_states(mj["n_states"])),
           "finite_pairs": int(fin.sum()), "mean_mea_path_length": float(lengths.mean()),
           "mean_expected_accuracy": float((gain[fin] / np.maximum(tokens[fin], 1)).mean()) if fin.any() else None,
           "mean_viterbi_expected_accuracy": float((vgain / np.maximum(tokens[keep], 1)).mean()) if len(keep) else None,
           "mea_gain_minus_viterbi_gain_min": float((gain[keep] - vgain).min()) if len(keep) else None,
           "mea": {"runs": mea_runs, "kernel_ms": mea_best["kernel_ms"], "launches": mea_best["launches"],
                   "pairs_per_s_kernel": n_pairs / (mea_best["kernel_ms"] / 1e3), "chunks": len(chunk_plan(x_off, y_off, 3 * mj["n_states"], free))},
           "path_posteriors_viterbi": {"runs": pp_runs, "kernel_ms": pp_best["kernel_ms"], "launches": pp_best["launches"],
                                       "paths_per_s_kernel": len(keep) / (pp_best["kernel_ms"] / 1e3), "steps": int(voff[-1]),
                                       "chunks": len(chunk_plan(x_off, y_off, 2 * mj["n_states"], free))}}
    b.close()
    m.close()
    print(json.dumps({k: (v if k not in ("mea", "path_posteriors_viterbi") else {q: w for q, w in v.items() if q != "runs"}) for k, v in out.items()}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--quick", action="store_true", help="a tenth of each workload")
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    from machineboss_b200 import capi
    scale = 10 if args.quick else 1
    result = {"card": card(), "seed": SEED, "workloads": []}
    print(json.dumps(result["card"]), flush=True)

    # dnapsw: 1 kb pairs, each output its input with 10 % substitutions and 2 % indels
    mj = bench.eval_machine("dnapsw")
    n = 2000 // scale
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
    result["workloads"].append(run_workload(capi, "PF00516, %d reads of 50 - 500" % n, mj, np.zeros(0, np.uint8), np.zeros(n + 1, np.int64), y, y_off, args.reps))

    result["card_after"] = card()
    with open(os.path.join(args.out_dir, "mea_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
