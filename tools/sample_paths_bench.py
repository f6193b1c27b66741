"""Posterior path sampling on one GPU (mb_sample_paths): device time of the full-storage Forward fill and the two walk passes,
paths per second and the stored matrix per chunk, on three workloads; and, as the comparison, the route that draws one path per
pair on the host (boss_b200 --sample-paths: a single-CTA fill per pair, the whole matrix copied to the host, a host traceback).

    python tools/sample_paths_bench.py OUT_DIR [--quick]

Writes OUT_DIR/sample_paths_bench.json with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench  # noqa: E402  (the benchmark's machines and synthetic data)

SAMPLES = 8
SEED = 20261022


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def free_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


def chunk_plan(x_off, y_off, n_states, free):
    """The chunks plan_chunks (csrc/mb_generic.cu) makes for full storage: 80 % of free memory per chunk, in pair order."""
    need = (np.diff(x_off) + 1).astype(np.float64) * (np.diff(y_off) + 1) * n_states
    budget = 0.80 * free / 8.0
    chunks, cur, n = [], 0.0, 0
    for v in need:
        if n and (cur + v > budget or n >= 65535 * 16):
            chunks.append(cur)
            cur, n = 0.0, 0
        cur += v
        n += 1
    if n:
        chunks.append(cur)
    return [int(c) * 8 for c in chunks]


def run_workload(capi, name, mj, x, x_off, y, y_off, reps):
    m = bench.make_machine(capi, mj)
    n_pairs = len(x_off) - 1
    warm = capi.Batch(x=x, x_off=x_off[:9] - x_off[0], y=y, y_off=y_off[:9] - y_off[0])      # first launches: module loading
    capi.sample_paths(m, warm, SAMPLES, SEED)
    warm.close()
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    plan = chunk_plan(x_off, y_off, mj["n_states"], free_bytes())
    runs = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ll, lengths, off, ids = capi.sample_paths(m, b, SAMPLES, SEED)
        wall = time.perf_counter() - t0
        ms, launches = b.last_kernel_ms()
        runs.append({"kernel_ms": ms, "launches": launches, "wall_s": wall})
    best = min(runs, key=lambda r: r["kernel_ms"])
    paths = n_pairs * SAMPLES
    out = {"workload": name, "pairs": n_pairs, "samples_per_pair": SAMPLES, "states": mj["n_states"],
           "cell_states": float(b.cell_states(mj["n_states"])), "finite_pairs": int(np.isfinite(ll).sum()),
           "mean_path_length": float(lengths.mean()), "runs": runs,
           "kernel_ms": best["kernel_ms"], "launches": best["launches"],
           "paths_per_s_kernel": paths / (best["kernel_ms"] / 1e3), "paths_per_s_wall": paths / best["wall_s"],
           "chunks": len(plan), "stored_matrix_bytes_per_chunk": plan}
    b.close()
    m.close()
    print(json.dumps({k: v for k, v in out.items() if k != "runs"}), flush=True)
    return out


def host_route(pairs):
    """boss_b200 --sample-paths (one path per pair through the host) against --posterior-paths 1 on the same pairs, wall clock
    of the whole process with the machine's compiled kernels already in a cache directory.  pairs: {label: (x, x_off, y, y_off)}.
    The host route follows the reference's random_index, whose unshifted weights exp(v) are all 0 once the Forward values fall
    below about -745: it then stops with "Zero weights", which is recorded."""
    from machineboss_b200 import build
    cli = build.build_host()
    with open(os.path.join(REPO, "machineboss_b200", "presets", "dnapsw.eval.json")) as f:
        pj = json.load(f)
    ia, oa = [""] + pj["inAlphabet"], [""] + pj["outAlphabet"]
    tmp = tempfile.mkdtemp(prefix="sample_paths_bench_")
    out = {}
    for label, (x, x_off, y, y_off) in pairs.items():
        n_pairs = len(x_off) - 1
        data = os.path.join(tmp, "pairs.json")
        with open(data, "w") as f:
            json.dump([{"input": {"name": "x%d" % k, "sequence": [ia[t] for t in x[x_off[k]:x_off[k + 1]]]},
                        "output": {"name": "y%d" % k, "sequence": [oa[t] for t in y[y_off[k]:y_off[k + 1]]]}} for k in range(n_pairs)], f)
        base = [cli, "--preset", "dnapsw", "-D", data, "--kernel-cache", os.path.join(tmp, "kernels"), "--gpus", "1"]
        subprocess.run(base + ["-L"], check=True, capture_output=True)      # compiles the machine's kernels into the cache
        res = {"pairs": n_pairs}
        for key, extra in (("sample_paths_host", ["--sample-paths", "1"]), ("posterior_paths_device", ["--posterior-paths", "1"])):
            t0 = time.perf_counter()
            r = subprocess.run(base + extra, capture_output=True, text=True)
            wall = time.perf_counter() - t0
            if r.returncode:
                res[key] = {"failed": r.stderr.strip()[-200:], "wall_s": wall}
                continue
            assert len(json.loads(r.stdout)) == n_pairs
            res[key] = {"wall_s": wall, "s_per_path": wall / n_pairs}
        out[label] = res
        print(json.dumps({label: res}), flush=True)
    shutil.rmtree(tmp, ignore_errors=True)
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
    result = {"card": card(), "samples_per_pair": SAMPLES, "seed": SEED, "workloads": []}
    print(json.dumps(result["card"]), flush=True)

    # dnapsw: 1 kb pairs, each output its input with 10 % substitutions and 2 % indels
    mj = bench.eval_machine("dnapsw")
    n = 2000 // scale
    x, x_off, _, _ = bench.synth_batch(SEED, 0, n, 1000, 1000, 4)
    y, y_off = bench.mutate_batch(SEED, x, x_off, 4)
    result["workloads"].append(run_workload(capi, "dnapsw, %d pairs of 1 kb x %d samples" % (n, SAMPLES), mj, x, x_off, y, y_off, args.reps))
    nh = 50 // (5 if args.quick else 1)
    xs, xs_off, _, _ = bench.synth_batch(SEED + 3, 0, nh, 300, 300, 4)
    ys, ys_off = bench.mutate_batch(SEED + 3, xs, xs_off, 4)
    result["host_route_dnapsw"] = host_route({"%d pairs of 1 kb" % nh: (x, x_off[:nh + 1], y, y_off[:nh + 1]),
                                              "%d pairs of 300 nt" % nh: (xs, xs_off, ys, ys_off)})

    # protpsw: 300 aa pairs
    mj = bench.eval_machine("protpsw")
    n = 10000 // scale
    x, x_off, _, _ = bench.synth_batch(SEED + 1, 0, n, 300, 300, 20)
    y, y_off = bench.mutate_batch(SEED + 1, x, x_off, 20)
    result["workloads"].append(run_workload(capi, "protpsw, %d pairs of 300 aa x %d samples" % (n, SAMPLES), mj, x, x_off, y, y_off, args.reps))

    # PF00516 profile: reads of 50 - 500 residues, no input sequence
    mj = bench.eval_machine("PF00516")
    n = 1000 // scale
    lens = 50 + (np.arange(n, dtype=np.int64) * 7919) % 451
    y, y_off = bench.synth_ragged(SEED + 2, lens, mj["n_out"])
    result["workloads"].append(run_workload(capi, "PF00516, %d reads of 50 - 500 x %d samples" % (n, SAMPLES), mj, np.zeros(0, np.uint8),
                                            np.zeros(n + 1, np.int64), y, y_off, args.reps))

    result["card_after"] = card()
    with open(os.path.join(args.out_dir, "sample_paths_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
