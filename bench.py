#!/usr/bin/env python3
"""bench.py -- batched Forward + Viterbi throughput of preset dnapsw on synthetic 1 kb DNA pairs.

One "step" = one pass of the hot path over one batch: Forward log-likelihood (boss -L) and Viterbi
score + traceback (boss -V/-A) for every pair of the batch.  Metric (BASELINE.json): DP cell-state
updates per second, in GCUPS, summed over both sweeps and over all ranks; pairs/s beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--len L] [--impl reference] [--no-configs]
                  [--dump-outputs DIR]

N > 1: launched by torchrun, one rank per GPU; every rank processes its own P pairs (weak scaling,
no data-path collective; the E-step's count all-reduce is timed separately as "em").  Times are
taken per step between device synchronisations, L2 is flushed between steps, the maximum over
ranks is used, and SM clocks / throttle reasons are sampled with nvidia-smi during the timed region.

Beside the headline line's own keys the JSON carries
  "set_b"    the same step on HARD data: peaked parameters (SURVEY 8d set B), every output the input with 10 %
             substitutions and 2 % indels, with the number of pairs the linear sweeps handed to the log domain;
  "strong"   strong scaling: 10 000 pairs IN TOTAL dealt over the ranks by the library's sharder (mb_shard_pairs);
  "configs"  (one GPU only) BASELINE configs 2 - 5 at their stated sizes or a stated sub-sample, each with GCUPS,
             pairs/s, the pairs re-run in the log domain, and its own roofline fraction.

--impl reference times the reference's own CPU implementation (oracle/_ref/refdrv, the unmodified
reference sources; falls back to the C restatement if that binary is absent) on the host cores.

--dump-outputs DIR writes what the last timed step computed on rank 0 as float64 .npy files (see dump_outputs), so
that two builds can be compared output for output: the inputs depend on the arguments only.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "forward_viterbi_gcups"
UNIT = "GCUPS"
SEED = 12345


# ---------------------------------------------------------------------------------------------
# workload: preset dnapsw, `boss -U` default parameters (src/constraints.cpp:65-75)
# ---------------------------------------------------------------------------------------------
def dnapsw_machine():
    """The flat evaluated dnapsw machine from the committed fixture (generated from the reference)."""
    with open(os.path.join(REPO, "tests", "golden", "dnapsw_synth64.json")) as f:
        j = json.load(f)["machine"]
    t = j["trans"]

    def num(v):
        return float("-inf") if v == "-Infinity" else float(v)
    return dict(n_states=j["nStates"], n_in=len(j["inAlphabet"]), n_out=len(j["outAlphabet"]),
                src=np.array([r[0] for r in t], np.int32), dst=np.array([r[1] for r in t], np.int32),
                tin=np.array([r[2] for r in t], np.int32), tout=np.array([r[3] for r in t], np.int32),
                lw=np.array([num(r[4]) for r in t], np.float64))


def eval_machine(preset: str):
    """A shipped pre-evaluated machine (machineboss_b200/presets/NAME.eval.json[.gz], boss -U default parameters)."""
    import gzip
    base = os.path.join(REPO, "machineboss_b200", "presets", preset + ".eval.json")
    if os.path.exists(base):
        with open(base) as f:
            j = json.load(f)
    else:
        with gzip.open(base + ".gz", "rt") as f:
            j = json.load(f)
    return _flat(j)


def fixture_machine(name: str):
    """The evaluated machine of a committed fixture (tests/golden), e.g. dnapsw with the peaked parameter set B."""
    import gzip
    base = os.path.join(REPO, "tests", "golden", name + ".json")
    if os.path.exists(base):
        with open(base) as f:
            j = json.load(f)
    else:
        with gzip.open(base + ".gz", "rt") as f:
            j = json.load(f)
    return _flat(j["machine"])


def _flat(j):
    t = j["trans"]

    def num(v):
        return float("-inf") if v == "-Infinity" else float(v)
    return dict(n_states=j["nStates"], n_in=len(j["inAlphabet"]), n_out=len(j["outAlphabet"]),
                src=np.array([r[0] for r in t], np.int32), dst=np.array([r[1] for r in t], np.int32),
                tin=np.array([r[2] for r in t], np.int32), tout=np.array([r[3] for r in t], np.int32),
                lw=np.array([num(r[4]) for r in t], np.float64))


def make_machine(capi, mj):
    return capi.Machine(mj["n_states"], mj["n_in"], mj["n_out"], mj["src"], mj["dst"], mj["tin"], mj["tout"], mj["lw"])


def _splitmix64(x):
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))


def synth_batch(seed: int, first_pair: int, n_pairs: int, li: int, lo: int, n_sym: int):
    """iid uniform tokens; same stream as oracle/synth.h (pair k, stream which, position p)."""
    out = []
    for which, length in ((0, li), (1, lo)):
        with np.errstate(over="ignore"):
            k = (np.arange(first_pair, first_pair + n_pairs, dtype=np.uint64) * np.uint64(2) + np.uint64(which))
            base = np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + k * np.uint64(0xD1B54A32D192ED03)
            p = base[:, None] + np.arange(length, dtype=np.uint64)[None, :]
        out.append((1 + (_splitmix64(p) % np.uint64(n_sym))).astype(np.uint8).reshape(-1))
    x_off = np.arange(n_pairs + 1, dtype=np.int64) * li
    y_off = np.arange(n_pairs + 1, dtype=np.int64) * lo
    return out[0], x_off, out[1], y_off


def synth_ragged(seed: int, lengths, n_sym: int, which: int = 1):
    """iid uniform tokens for sequences of the given lengths (the stream of synth_batch, pair k = index k)."""
    lengths = np.asarray(lengths, dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    total = int(off[-1])
    pair = np.repeat(np.arange(len(lengths), dtype=np.uint64), lengths)
    pos = (np.arange(total, dtype=np.int64) - np.repeat(off[:-1], lengths)).astype(np.uint64)
    with np.errstate(over="ignore"):
        base = np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + (pair * np.uint64(2) + np.uint64(which)) * np.uint64(0xD1B54A32D192ED03)
        tok = (1 + (_splitmix64(base + pos) % np.uint64(n_sym))).astype(np.uint8)
    return tok, off


def mutate_batch(seed: int, x: np.ndarray, x_off: np.ndarray, n_sym: int, sub: float = 0.10, indel: float = 0.02):
    """SURVEY 8(d) set B data: every output = its input with `sub` substitutions and `indel` indels per position
    (half deletions, half insertions), vectorised over the whole batch."""
    n = int(x.shape[0])
    with np.errstate(over="ignore"):
        r = _splitmix64(np.arange(3 * n, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x5851F42D4C957F2D))
    u = (r[:n] >> np.uint64(11)).astype(np.float64) / float(1 << 53)
    alt = (r[n:2 * n] % np.uint64(n_sym - 1)).astype(np.int64)
    ins = (1 + r[2 * n:] % np.uint64(n_sym)).astype(np.uint8)
    base = np.where(u < indel / 2 + sub, (1 + (x.astype(np.int64) + alt) % n_sym).astype(np.uint8), x)
    count = np.where(u < indel / 2, 0, np.where(u > 1.0 - indel / 2, 2, 1)).astype(np.int64)      # deleted / kept / kept + insertion
    start = np.concatenate([[0], np.cumsum(count)]).astype(np.int64)
    y = np.empty(int(start[-1]), dtype=np.uint8)
    kept = count >= 1
    y[start[:-1][kept]] = base[kept]
    two = count == 2
    y[start[:-1][two] + 1] = ins[two]
    y_off = start[x_off]
    return y, y_off.astype(np.int64)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            f = [c.strip() for c in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU reference arm
# ---------------------------------------------------------------------------------------------
def cpu_reference(li: int, lo: int, n_pairs: int, threads: int, seed: int = SEED):
    """Forward (rolling, as boss -L) + Viterbi with traceback on `n_pairs` synthetic pairs.

    Returns (gcups, pairs_per_s, kind, seconds)."""
    refdrv = os.path.join(REPO, "oracle", "_ref", "refdrv")
    cells = float(li + 1) * float(lo + 1) * 8 * n_pairs
    if os.path.exists(refdrv):
        r = subprocess.run([refdrv, "--machine", "preset:dnapsw", "--synth", "%d,%d,%d,%d" % (n_pairs, li, lo, seed),
                            "--do", "rolling,viterbi,path", "--threads", str(threads), "--quiet-results"],
                           check=True, capture_output=True, text=True)
        secs = float(json.loads(r.stdout)["seconds"])
        return 2 * cells / secs / 1e9, n_pairs / secs, "reference", secs
    # the C restatement (single-threaded per call; run `threads` processes' worth sequentially is
    # pointless, so time one thread and say so)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import FlatMachine, Oracle, load_golden, synth_tokens
    orc = Oracle(FlatMachine.from_json(load_golden("dnapsw_synth64")["machine"]))
    t0 = time.perf_counter()
    for k in range(n_pairs):
        x, y = synth_tokens(seed, k, 0, li, 4), synth_tokens(seed, k, 1, lo, 4)
        orc.forward(x, y)
        orc.viterbi(x, y)
    secs = time.perf_counter() - t0
    return 2 * cells / secs / 1e9, n_pairs / secs, "port", secs


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = max(threads, 8)
    for _ in range(args.warmup if args.warmup < 1 else 1):     # one bounded warm-up pass is enough on a CPU
        cpu_reference(args.len, args.len, min(n, threads), threads)
    vals, secs = [], []
    kind = "reference"
    for _ in range(args.steps):
        g, pps, kind, s = cpu_reference(args.len, args.len, n, threads)
        vals.append(g); secs.append(s)
    value = statistics.mean(vals)
    sample = "%d synthetic %dx%d dnapsw pairs per step (Forward rolling + Viterbi with traceback), %d threads" % (n, args.len, args.len, threads)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(secs), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args, n), pairs_per_gpu=None, pairs_total=n, parallelism="host threads on rank 0 only (%d); the other ranks exit" % threads),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "pairs_per_s": n / statistics.mean(secs)}))


def workload_config(args, pairs_per_rank):
    return {"workload": "preset dnapsw (S=8, 34 transitions, boss -U default parameters), %d synthetic iid-uniform pairs of "
                        "%d x %d nt per GPU: Forward log-likelihood + Viterbi score and traceback for every pair"
                        % (pairs_per_rank, args.len, args.len),
            "pairs_per_gpu": pairs_per_rank, "len_in": args.len, "len_out": args.len, "seed": SEED,
            "l2": "256 MiB buffer written between timed steps (L2 flush)", "parallelism": "pairs sharded, %d rank(s)" % args.gpus}


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=int(os.environ.get("MB_BENCH_PAIRS", "10000")), help="pairs per GPU")
    ap.add_argument("--len", type=int, default=1000)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--engine", type=int, default=-1)
    ap.add_argument("--em-pairs", type=int, default=4096, help="pairs per GPU in the E-step (counts) leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the set-B, strong-scaling and configs 2-5 legs")
    ap.add_argument("--strong-pairs", type=int, default=10000, help="pairs IN TOTAL of the strong-scaling leg")
    ap.add_argument("--cfg3-pairs", type=int, default=100000)
    ap.add_argument("--cfg4-pairs", type=int, default=1000)
    ap.add_argument("--cfg5-reads", type=int, default=131072)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results here as .npy files")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no results")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from machineboss_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    capi.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    mj = dnapsw_machine()
    capi.set_engine(args.engine)
    mach = capi.Machine(mj["n_states"], mj["n_in"], mj["n_out"], mj["src"], mj["dst"], mj["tin"], mj["tout"], mj["lw"])
    capi.set_engine(-1)
    S = mj["n_states"]
    P = args.pairs
    x, x_off, y, y_off = synth_batch(SEED, rank * P, P, args.len, args.len, 4)
    # pinned host staging for the end-to-end leg
    px = torch.from_numpy(x).pin_memory()
    py = torch.from_numpy(y).pin_memory()
    cells = float(args.len + 1) * float(args.len + 1) * S * P      # cell-states per sweep per rank
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    batch = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    kernel_ms = {"forward": [], "viterbi": []}
    launches = 0

    def step_resident():
        nonlocal launches
        ll = capi.forward(mach, batch)
        ms, n = batch.last_kernel_ms(); kernel_ms["forward"].append(ms); launches += n
        sc, plen = capi.viterbi_lengths(mach, batch)
        ms, n = batch.last_kernel_ms(); kernel_ms["viterbi"].append(ms); launches += n
        return ll, sc, plen

    # end-to-end leg: host buffers in, host buffers out, through the C ABI.  Inputs are copied from
    # pinned host memory, results land in pinned host memory the caller owns (allocated once, as a
    # service would): per-pair log-likelihoods, Viterbi scores, path lengths and the packed paths
    # (global transition ids, one byte each for a machine this small).
    path_cap = P * (2 * args.len + 2) * 2
    h_ll = torch.empty(P, dtype=torch.float64).pin_memory().numpy()
    h_sc = torch.empty(P, dtype=torch.float64).pin_memory().numpy()
    h_len = torch.empty(P, dtype=torch.int64).pin_memory().numpy()
    h_off = torch.empty(P + 1, dtype=torch.int64).pin_memory().numpy()
    # transition ids as bytes when the machine has at most 256 transitions (dnapsw: 34), mb_viterbi_paths_narrow
    id_dtype = torch.uint8 if len(mj["lw"]) <= 256 else torch.int32
    h_paths = torch.empty(path_cap, dtype=id_dtype).pin_memory().numpy()

    def step_e2e():
        b = capi.Batch(x=px.numpy(), x_off=x_off, y=py.numpy(), y_off=y_off)      # H2D from pinned memory
        total = capi.viterbi_start(mach, b, h_sc, h_len, h_off, h_paths)          # D2H of scores and lengths; the packed paths leave through the copy engine ...
        capi.forward_into(mach, b, h_ll)                                          # ... while the Forward sweep of the same pairs runs
        b.wait()                                                                  # paths have arrived
        b.close()
        return h_ll, h_sc, (h_paths[:total], h_off)

    for _ in range(args.warmup):
        step_resident()
    kernel_ms = {"forward": [], "viterbi": []}
    launches = 0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    times = []
    for _ in range(args.steps):
        flush.fill_(1)
        barrier()
        t0 = time.perf_counter()
        ll, sc, plen = step_resident()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    e2e_times = []
    d2h = 0
    for n in range(args.warmup + args.steps):      # W untimed steps first: a fresh batch's scratch comes from the allocator until the pool is warm
        flush.fill_(1)
        barrier()
        t0 = time.perf_counter()
        ll2, sc2, paths = step_e2e()
        torch.cuda.synchronize()
        if n >= args.warmup:
            e2e_times.append(time.perf_counter() - t0)
        d2h = ll2.nbytes + sc2.nbytes + paths[0].nbytes + paths[1].nbytes
    e2e_total = sum(e2e_times)
    clocks = sampler.stop() if rank == 0 else None
    assert np.array_equal(ll, ll2) and np.array_equal(sc, sc2)

    # E-step of Baum-Welch on a bounded slice of the same batch: Forward (stored) + Backward fused with
    # the posterior counts, then the path's one exchange step, the all-reduce of nTrans+1 doubles.
    from machineboss_b200 import shard
    n_em = min(P, args.em_pairs)
    em_batch = capi.Batch(x=x[: n_em * args.len], x_off=x_off[: n_em + 1], y=y[: n_em * args.len], y_off=y_off[: n_em + 1])
    capi.counts(mach, em_batch)
    barrier()
    t0 = time.perf_counter()
    cnt, cll = capi.counts(mach, em_batch)
    em_kernel_ms, em_launches = em_batch.last_kernel_ms()
    cnt, tot_ll = shard.allreduce_counts(cnt, float(cll.sum()), device="cuda")
    torch.cuda.synchronize()
    em_secs = time.perf_counter() - t0
    em_batch.close()

    # strong scaling: a fixed list of pairs dealt over the ranks by the library's sharder (longest-processing-time first by
    # cell count; mb_shard_pairs is also what mb_group_batch_create applies inside one process), resident, same step
    sp = args.strong_pairs
    sx, sx_off, sy, sy_off = synth_batch(SEED + 2, 0, sp, args.len, args.len, 4)
    mine = np.flatnonzero(capi.shard_pairs(sx_off, sy_off, world) == rank)
    sel = (mine[:, None] * args.len + np.arange(args.len)[None, :]).reshape(-1)
    s_off = np.arange(len(mine) + 1, dtype=np.int64) * args.len
    s_batch = capi.Batch(x=sx[sel], x_off=s_off, y=sy[sel], y_off=s_off)
    for _ in range(2):
        capi.forward(mach, s_batch); capi.viterbi_lengths(mach, s_batch)
    strong_times = []
    for _ in range(max(3, args.steps)):
        barrier()
        t0 = time.perf_counter()
        capi.forward(mach, s_batch); capi.viterbi_lengths(mach, s_batch)
        torch.cuda.synchronize()
        strong_times.append(time.perf_counter() - t0)
    strong_secs = sum(strong_times) / len(strong_times)
    s_batch.close()

    if world > 1:
        t = torch.tensor([total, e2e_total, em_secs, strong_secs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total, e2e_total, em_secs, strong_secs = float(t[0]), float(t[1]), float(t[2]), float(t[3])

    if rank == 0:
        K = args.steps
        value = 2 * cells * world * K / total / 1e9
        e2e = 2 * cells * world * K / e2e_total / 1e9
        fwd_ms = statistics.mean(kernel_ms["forward"])
        vit_ms = statistics.mean(kernel_ms["viterbi"])
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, P),
            "pairs_per_s": P * world * K / total,
            "forward_gcups": cells / fwd_ms / 1e6, "viterbi_gcups": cells / vit_ms / 1e6,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(x.nbytes + y.nbytes + x_off.nbytes + y_off.nbytes),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_total / K},
            "gpu_launches": launches, "clocks": clocks, "engine": mach.engine,
            "check": {"forward_ll_pair0": float(ll[0]), "viterbi_pair0": float(sc[0]), "path_len_pair0": int(plen[0])},
        }
        em_cells = float(args.len + 1) * float(args.len + 1) * S * n_em
        out["em"] = {"what": "E-step (MachineCounts over the list): stored Forward + fused Backward/posterior counts on %d pairs per GPU, then all-reduce of %d doubles" % (n_em, len(cnt) + 1),
                     "pairs_per_s": n_em * world / em_secs, "gcups_2_sweeps": 2 * em_cells * world / em_secs / 1e9,
                     "kernel_ms": em_kernel_ms, "launches": em_launches, "sum_counts": float(cnt.sum()), "loglike": tot_ll}
        out["roofline"] = roofline(mj, cells, fwd_ms, vit_ms)
        out["strong"] = {"what": "strong scaling: %d pairs of %d x %d IN TOTAL, dealt over %d rank(s) by mb_shard_pairs; Forward + Viterbi with traceback, resident" % (sp, args.len, args.len, world),
                         "value": 2 * float(args.len + 1) ** 2 * S * sp / strong_secs / 1e9, "unit": UNIT, "ms_per_step": 1e3 * strong_secs,
                         "pairs_total": sp, "pairs_this_rank": int(len(mine)), "scaling": "strong"}
        if not args.no_configs:
            out["set_b"] = run_set_b(capi, P, args.len)
            if world == 1:
                out["configs"] = run_configs(capi, args)
                out["ingest"] = run_ingest()
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            n = max(8, threads)
            g, pps, kind, secs = cpu_reference(args.len, args.len, n, threads)
            out["cpu_baseline"] = {"value": g, "unit": UNIT, "cores": threads, "kind": kind, "seconds": secs,
                                   "sample": "%d of the same synthetic %dx%d pairs, Forward (rolling) + Viterbi with traceback, %d threads"
                                             % (n, args.len, args.len, threads)}
        if args.dump_outputs:      # the paths of the last timed step are still held by its batch
            dump_outputs(args.dump_outputs, ll, sc, plen, *capi.viterbi_paths(batch, plen))
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT = 60 << 20      # bytes of array data: with the .npy headers the files stay under 64 MB
DUMP_PATHS = 256           # pairs whose Viterbi paths are written


def dump_outputs(out_dir: str, ll, sc, plen, trans, off):
    """Write the headline step's results to out_dir as float64 .npy files:
      pairs, forward_loglike, viterbi_score, viterbi_path_length   per pair (every pair, or a seeded sample of them when
                                                                   the batch is too large for DUMP_LIMIT; `pairs` names them)
      viterbi_path_pairs, viterbi_path_offsets, viterbi_paths      the paths (global transition ids) of a seeded sample of
                                                                   DUMP_PATHS pairs, concatenated, within what is left"""
    n = len(ll)
    rng = np.random.default_rng(SEED)
    cap = DUMP_LIMIT // 2 // (4 * 8)
    pairs = np.arange(n) if n <= cap else np.sort(rng.choice(n, cap, replace=False))
    arrays = {"pairs": pairs, "forward_loglike": ll[pairs], "viterbi_score": sc[pairs], "viterbi_path_length": plen[pairs]}
    budget = DUMP_LIMIT - 8 * 4 * len(pairs)
    path_pairs, paths = [], []
    for k in np.sort(rng.choice(n, min(n, DUMP_PATHS), replace=False)):
        budget -= 8 * (int(off[k + 1] - off[k]) + 2)
        if budget < 0:
            break
        path_pairs.append(k)
        paths.append(trans[off[k]:off[k + 1]])
    arrays["viterbi_path_pairs"] = np.array(path_pairs)
    arrays["viterbi_path_offsets"] = np.concatenate([[0], np.cumsum([len(p) for p in paths])])
    arrays["viterbi_paths"] = np.concatenate(paths) if paths else np.zeros(0)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def machine_groups(mj: dict):
    """Transition groups of a machine: (groups per cell = T_c of SURVEY 8, second-and-later groups of a state,
    states whose first silent group the normalised linear sweep turns into a plain copy)."""
    groups, seen = set(), {}
    for t in range(len(mj["src"])):
        a, b = int(mj["tin"][t]), int(mj["tout"][t])
        if a == 0 and b == 0 and mj["dst"][t] <= mj["src"][t]:
            continue
        kind = 0 if (a and b) else 1 if a else 2 if b else 3
        key = (int(mj["dst"][t]), kind, int(mj["src"][t]), (a, b))
        rank = seen.get(key, 0)
        seen[key] = rank + 1
        groups.add((int(mj["dst"][t]), kind, int(mj["src"][t]), rank))
    t_c = len(groups)
    n_2nd = t_c - len({g[0] for g in groups})
    n_unit = len({g[0] for g in groups if g[1] == 3})
    return t_c, n_2nd, n_unit


def pipe_peaks():
    """FP64 pipe rates measured on this pool's B200 by tools/pipe_peaks.cu (Gop/s, chip-wide, from CUDA events)."""
    pipe, src = {}, None
    for name in ("r02_pipe_peaks.json", "r01_pipe_peaks.json"):
        pp = os.path.join(REPO, "profiles", name)
        if os.path.exists(pp):
            with open(pp) as f:
                pipe = {r["op"]: r["gops_per_s"] for r in json.load(f)["results"]}
            src = "profiles/" + name
            break
    return {"dfma": pipe.get("dfma", 17895.0), "dadd": pipe.get("dadd", 17775.0), "dsetp_sel": pipe.get("dsetp_sel", 8475.0), "source": src or "fallback constants"}


def hbm_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def issue_roofline(mj: dict, what: str, cells: float, ms: float, groups_per_cell=None) -> dict:
    """Issue roofline of one sweep over the per-cell transition fan-in (BASELINE.json; DESIGN.md section 6).

      sums (scaled linear domain): one FP64 multiply-add per transition group      peak = S * DFMA / T_c
      Viterbi (exact FP64 add + compare): one add per group, one compare + select
        per second-and-later group of a state                                      peak = S / (T_c / DADD + n_2nd / DSETP_SEL)
    T_c counts EVERY group of a cell (dnapsw: 13, 5 of them second groups).  What the kernels execute is less: the
    end state is only formed in a pair's last cell (Viterbi: 11 adds + 4 compares), and the normalised sums turn each
    state's first silent group into a copy (7 multiply-adds) -- `executed` gives the fraction against that count too."""
    S = mj["n_states"]
    t_c, n_2nd, n_unit = machine_groups(mj)
    if groups_per_cell:
        t_c = groups_per_cell
    pk = pipe_peaks()
    ach = cells / ms / 1e6
    if what == "viterbi":
        peak = S / (t_c / pk["dadd"] + n_2nd / pk["dsetp_sel"])
        bound = "issue (FP64 add + compare/select)"
        ex_adds, ex_cmp = t_c - 2, n_2nd - 1      # the end state's two groups are only formed in the last cell
        executed = {"adds": ex_adds, "compares": ex_cmp, "peak": S / (ex_adds / pk["dadd"] + ex_cmp / pk["dsetp_sel"])}
    else:
        peak = S * pk["dfma"] / t_c
        bound = "issue (FP64 FMA pipe)"
        ex = max(t_c - n_unit - 2, 1)               # (the end state's groups likewise)
        executed = {"multiply_adds": ex, "peak": S * pk["dfma"] / ex}
    executed["frac"] = ach / executed["peak"]
    return {"bound": bound, "achieved": ach, "peak": peak, "unit": "GCUPS", "frac": ach / peak, "ms_per_launch": ms,
            "per_cell": {"transition_groups": t_c, "second_groups": n_2nd, "states": S}, "executed": executed}


def roofline(mj: dict, cells: float, fwd_ms: float, vit_ms: float) -> dict:
    """Roofline block of the headline step: the dominant kernel (longest) at top level, both sweeps inside."""
    pk = pipe_peaks()
    hbm, hbm_src = hbm_peak()
    S = mj["n_states"]
    fwd = dict(issue_roofline(mj, "forward", cells, fwd_ms), kernel="mb_k_forward_lin")
    vit = dict(issue_roofline(mj, "viterbi", cells, vit_ms), kernel="mb_k_viterbi (+ traceback kernels: the whole mb_viterbi call)")
    vit["hbm"] = {"algorithmic_bytes_per_launch": cells / S * 1.0, "achieved_gbs": cells / S / vit_ms / 1e6, "peak_gbs": hbm,
                  "frac": cells / S / vit_ms / 1e6 / hbm, "peak_source": hbm_src}
    top = dict(vit if vit_ms >= fwd_ms else fwd)
    # DRAM bytes (read + write) of one launch of that kernel from the committed `ncu --set full` capture, taken at
    # this bench's default size (10 000 pairs of 1000 x 1000)
    top["traffic"] = None
    for name in ("r02_ncu_summary.json", "r01_ncu_summary.json"):
        sp = os.path.join(REPO, "profiles", name)
        if os.path.exists(sp) and abs(cells - 1001.0 * 1001.0 * 8 * 10000) < 1:
            with open(sp) as f:
                kk = json.load(f).get("kernels", {})
            k = kk.get("mb_k_viterbi_i") or kk.get("mb_k_viterbi_i2") or kk.get("mb_k_viterbi") or {}
            if vit_ms < fwd_ms:
                k = kk.get("mb_k_forward_lin", {})
            if k.get("dram_traffic_bytes") and k.get("pairs", 10000) == 10000:
                top["traffic"] = k["dram_traffic_bytes"]
                top["traffic_source"] = "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum (profiles/%s)" % name
                break
    top["peak_source"] = "measured DFMA %.0f, DADD %.0f, DSETP+SEL %.0f Gop/s (%s)" % (pk["dfma"], pk["dadd"], pk["dsetp_sel"], pk["source"])
    top["forward"] = fwd
    top["viterbi"] = vit
    return top


# ---------------------------------------------------------------------------------------------
# the other legs: hard data, strong scaling, BASELINE configs 2 - 5
# ---------------------------------------------------------------------------------------------
def timed_passes(capi, mach, batch, passes, reps=2):
    """Kernel milliseconds (device events inside the library) and wall seconds per pass, best of `reps` after a warm-up."""
    out = {}
    for name in passes:
        fn = {"forward": lambda: capi.forward(mach, batch), "viterbi": lambda: capi.viterbi_lengths(mach, batch),
              "viterbi_score": lambda: capi.viterbi(mach, batch, paths=False), "counts": lambda: capi.counts(mach, batch)}[name]
        fn()
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            res = fn()
            wall = time.perf_counter() - t0
            ms, nl = batch.last_kernel_ms()
            if best is None or ms < best["kernel_ms"]:
                best = {"kernel_ms": ms, "wall_ms": 1e3 * wall, "launches": nl}
        best["redo"] = batch.last_redo() if name in ("forward", "counts") else 0
        out[name] = (best, res)
    return out


def run_set_b(capi, P, L):
    """The headline step on hard data: peaked dnapsw parameters, mutated copies (SURVEY 8d set B)."""
    mj = fixture_machine("dnapsw_peaked")
    mach = make_machine(capi, mj)
    x, x_off, _, _ = synth_batch(SEED + 1, 0, P, L, L, 4)
    y, y_off = mutate_batch(SEED + 1, x, x_off, 4)
    batch = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    cells = batch.cell_states(mj["n_states"])
    r = timed_passes(capi, mach, batch, ["forward", "viterbi"])
    f, v = r["forward"][0], r["viterbi"][0]
    ms = f["kernel_ms"] + v["kernel_ms"]
    out = {"what": "set B: peaked dnapsw parameters (sub 0.91 / 0.03, gapOpen 0.05, gapExtend 0.5), %d pairs, input %d nt iid, output = input with 10 %% substitutions + 2 %% indels" % (P, L),
           "value": 2 * cells / ms / 1e6, "unit": UNIT, "forward_gcups": cells / f["kernel_ms"] / 1e6, "viterbi_gcups": cells / v["kernel_ms"] / 1e6,
           "pairs_per_s": P / (ms / 1e3), "redo_pairs": f["redo"], "redo_frac": f["redo"] / P,
           "loglike_pair0": float(r["forward"][1][0]), "viterbi_pair0": float(r["viterbi"][1][0][0])}
    batch.close(); mach.close()
    return out


def run_ingest(n_pairs=100000, length=300):
    """SURVEY 8(f) rank 2: sequence files -> packed tokens on the host (boss_b200_ingest.h), timed by the host mirror's own
    CLI on config 3's data (protein pairs as two FASTA files), to be read next to the GPU time of the same pairs."""
    import tempfile
    from machineboss_b200 import build
    try:
        cli = build.build_host()
    except Exception as e:      # no host compiler on this box
        return {"unavailable": str(e)[:200]}
    aa = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)
    x, _, y, _ = synth_batch(SEED + 3, 0, n_pairs, length, length, 20)
    out = {"what": "%d protein pairs of %d aa: two FASTA files -> packed tokens, host only, one thread" % (n_pairs, length)}
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for toks, prefix in ((x, b"x"), (y, b"y")):
            seqs = aa[toks - 1].reshape(n_pairs, length)
            path = os.path.join(tmp, prefix.decode() + ".fa")
            with open(path, "wb") as f:
                for k in range(n_pairs):
                    f.write(b">" + prefix + str(k).encode() + b"\n" + seqs[k].tobytes() + b"\n")
            paths.append(path)
        r = subprocess.run([cli, "--preset", "protpsw", "--paired-fasta", paths[0], paths[1], "--ingest-only"], capture_output=True, text=True)
        if r.returncode != 0:
            return {"unavailable": r.stderr[-200:]}
        out.update(json.loads(r.stdout))
    return out


def run_configs(capi, args):
    """BASELINE configs 2 - 5 on one GPU, each at its stated size or a stated sub-sample of it."""
    out = []
    hbm, _ = hbm_peak()

    def entry(name, workload, sample, mj, batch, n_pairs, r, extra=None, groups=None):
        cells = batch.cell_states(mj["n_states"])
        e = {"config": name, "workload": workload, "sample": sample, "pairs": n_pairs, "cell_states_per_pass": cells, "states": mj["n_states"], "transitions": int(len(mj["lw"]))}
        for k, (t, _) in r.items():
            e[k] = {"gcups": cells / t["kernel_ms"] / 1e6, "pairs_per_s": n_pairs / (t["wall_ms"] / 1e3), "kernel_ms": t["kernel_ms"], "launches": t["launches"], "redo_pairs": t["redo"]}
            if k in ("forward", "viterbi", "viterbi_score"):
                rf = issue_roofline(mj, "viterbi" if k.startswith("viterbi") else "forward", cells, t["kernel_ms"], groups)
                e[k]["roofline"] = {kk: rf[kk] for kk in ("bound", "peak", "frac", "unit")}
        if extra:
            e.update(extra)
        out.append(e)

    # config 2: E-step (stored Forward + fused Backward / posterior counts) on dnapsw 1 kb pairs, one GPU's share
    mj = eval_machine("dnapsw")
    mach = make_machine(capi, mj)
    n = args.em_pairs
    x, x_off, y, y_off = synth_batch(SEED, 0, n, 1000, 1000, 4)
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    r = timed_passes(capi, mach, b, ["counts"])
    t = r["counts"][0]
    algo_bytes = 2.0 * 16.0 * 1001 * 1001 * n * 1.03      # 16-byte stored Forward cells written once and read once (+3 % ramps)
    entry("cfg2", "preset dnapsw Baum-Welch E-step (Forward stored + Backward fused with posterior counts), 10 000 pairs of 1 kb over 8 GPUs",
          "%d pairs of 1000 x 1000 on one GPU (the config's share per GPU is 1250)" % n, mj, b, n, r,
          {"counts_sum_per_pair": float(r["counts"][1][0].sum()) / n,
           "roofline": {"bound": "hbm", "achieved": algo_bytes / t["kernel_ms"] / 1e6, "peak": hbm, "unit": "GB/s", "frac": algo_bytes / t["kernel_ms"] / 1e6 / hbm}})
    b.close(); mach.close()

    # config 3: protpsw Viterbi alignment, 300 aa pairs
    mj = eval_machine("protpsw")
    mach = make_machine(capi, mj)
    n = args.cfg3_pairs
    x, x_off, y, y_off = synth_batch(SEED + 3, 0, n, 300, 300, 20)
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    entry("cfg3", "preset protpsw Viterbi alignment (score + traceback), 100 000 pairs of 300 aa", "%d pairs of 300 x 300" % n, mj, b, n,
          timed_passes(capi, mach, b, ["viterbi", "forward"]))
    b.close(); mach.close()

    # config 4: the GeneWise-style composite, protein against 10 kb of DNA
    mj = eval_machine("prot2dna_dnapsw")
    mach = make_machine(capi, mj)
    n = args.cfg4_pairs
    x, x_off, _, _ = synth_batch(SEED + 4, 0, n, 300, 300, mj["n_in"])
    _, _, y, y_off = synth_batch(SEED + 4, 0, n, 10000, 10000, mj["n_out"])
    b = capi.Batch(x=x, x_off=x_off, y=y, y_off=y_off)
    entry("cfg4", "prot2dna => dnapsw (308 states), Forward + Viterbi, 1000 pairs of 300 aa x 10 kb", "%d pairs of 300 aa x 10 000 nt" % n, mj, b, n,
          timed_passes(capi, mach, b, ["forward", "viterbi_score", "viterbi"], reps=1))
    b.close(); mach.close()

    # config 5: a profile HMM composed with an error model scoring reads of 50 - 500 residues (length-bucketed inside the engine)
    for preset, n in (("PF00516", args.cfg5_reads), ("PF00516_protpsw", args.cfg5_reads // 4)):
        mj = eval_machine(preset)
        mach = make_machine(capi, mj)
        lens = 50 + (np.arange(n, dtype=np.int64) * 7919) % 451
        y, y_off = synth_ragged(SEED + 5, lens, mj["n_out"])
        b = capi.Batch(x=np.zeros(0, np.uint8), x_off=np.zeros(n + 1, np.int64), y=y, y_off=y_off)
        entry("cfg5" if preset == "PF00516_protpsw" else "cfg5-core",
              "HMMER profile %s (%d states), Forward + Viterbi on 1 000 000 reads of 50 - 500 residues" % (preset.replace("_", " => "), mj["n_states"]),
              "%d reads, lengths 50 - 500 (uniform, ragged)" % n, mj, b, n, timed_passes(capi, mach, b, ["forward", "viterbi_score", "viterbi"], reps=3))
        b.close(); mach.close()
    return out


if __name__ == "__main__":
    main()
