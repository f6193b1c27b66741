"""CPU test of bench.py's reference arm (`--impl reference`): the reference's own CPU implementation of the path (oracle/_ref/refdrv,
the reference compiled unmodified; where that is not built, the C restatement oracle/mb_oracle.c) timed on this box's host cores,
printing ONE JSON line with the contract's keys -- and that the product arm refuses to run without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    # the reference's sources are not part of this repository: without its binary the arm times the C restatement
    kind = "reference" if os.path.exists(os.path.join(REPO, "oracle", "_ref", "refdrv")) else "port"
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, cwd=REPO, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "GCUPS" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_product_arm_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "1", "--warmup", "0", "--no-configs", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=REPO, timeout=600)
    assert r.returncode != 0      # no CPU fallback: the product path fails loudly without CUDA


def test_dump_outputs_writes_float64_arrays_within_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: every array float64, the paths of a seeded sample of pairs cut from the packed list, the same sample
    on every run, and a batch too large for the limit sampled instead of cut off."""
    sys.path.insert(0, REPO)
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    n = 1000
    plen = rng.integers(1, 50, n)
    off = np.concatenate([[0], np.cumsum(plen)])
    trans = rng.integers(0, 34, int(off[-1])).astype(np.int32)
    ll, sc = rng.normal(size=n), rng.normal(size=n)

    def dump(d):
        bench.dump_outputs(str(d), ll, sc, plen, trans, off)
        return {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}

    a, b = dump(tmp_path / "a"), dump(tmp_path / "b")
    assert sorted(a) == ["forward_loglike", "pairs", "viterbi_path_length", "viterbi_path_offsets", "viterbi_path_pairs",
                         "viterbi_paths", "viterbi_score"]
    assert all(v.dtype == np.float64 and np.array_equal(v, b[k]) for k, v in a.items())
    assert np.array_equal(a["pairs"], np.arange(n)) and np.array_equal(a["forward_loglike"], ll)
    assert np.array_equal(a["viterbi_score"], sc) and np.array_equal(a["viterbi_path_length"], plen)
    kept = a["viterbi_path_pairs"].astype(np.int64)
    assert len(kept) == bench.DUMP_PATHS and np.all(np.diff(kept) > 0)
    po = a["viterbi_path_offsets"].astype(np.int64)
    for j, k in enumerate(kept):
        assert np.array_equal(a["viterbi_paths"][po[j]:po[j + 1]], trans[off[k]:off[k + 1]])

    monkeypatch.setattr(bench, "DUMP_LIMIT", 16 * 1024)
    c = dump(tmp_path / "c")
    assert sum(v.nbytes for v in c.values()) <= 16 * 1024
    pairs = c["pairs"].astype(np.int64)
    assert 0 < len(pairs) < n and np.all(np.diff(pairs) > 0)
    assert np.array_equal(c["forward_loglike"], ll[pairs]) and np.array_equal(c["viterbi_path_length"], plen[pairs])


@pytest.mark.gpu
def test_dumped_outputs_are_the_oracles(tmp_path):
    """bench.py --dump-outputs on a small batch: the Forward log-likelihoods, Viterbi scores and paths it writes are the C
    oracle's for the same synthetic pairs, and the JSON line counts the timed steps asked for."""
    import numpy as np
    from helpers import FlatMachine, Oracle, load_golden, synth_tokens
    sys.path.insert(0, REPO)
    import bench
    n, length = 300, 200
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--pairs", str(n), "--len", str(length), "--steps", "2",
                        "--warmup", "1", "--no-configs", "--no-cpu-baseline", "--strong-pairs", str(n), "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=REPO, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.splitlines()[-1])["steps"] == 2
    a = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert np.array_equal(a["pairs"], np.arange(n))
    orc = Oracle(FlatMachine.from_json(load_golden("dnapsw_synth64")["machine"]))
    kept = a["viterbi_path_pairs"].astype(np.int64)
    po = a["viterbi_path_offsets"].astype(np.int64)
    assert len(kept) == bench.DUMP_PATHS
    for j in range(0, len(kept), 8):
        k = int(kept[j])
        x, y = synth_tokens(bench.SEED, k, 0, length, 4), synth_tokens(bench.SEED, k, 1, length, 4)
        f = orc.forward(x, y)
        v, p = orc.viterbi(x, y)
        assert abs(a["forward_loglike"][k] - f) <= 1e-4 * abs(f), (k, a["forward_loglike"][k], f)
        assert a["viterbi_score"][k] == v and a["viterbi_path_length"][k] == len(p), k
        assert a["viterbi_paths"][po[j]:po[j + 1]].astype(np.int64).tolist() == p.tolist(), k
