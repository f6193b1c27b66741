"""Posterior paths drawn on the device for a whole batch (mb_sample_paths, -m gpu).

Each path is replayed on the host over the pair's stored Forward matrix (mb_matrix, the same fill with the same bits) with the
host Philox4x32-10 and the sampler's selection rule, and must match id for id.  The mean use of each transition over many
draws must match the pair's expected counts (mb_counts), and every path must be a valid alignment of its pair."""
import json
import math
import subprocess
import tempfile

import numpy as np
import pytest

from helpers import FlatMachine, load_golden, pairs_from_golden
from sample_replay import Incoming, replay

pytestmark = pytest.mark.gpu


def _capi():
    from machineboss_b200 import capi
    return capi


def golden_machine(name):
    return FlatMachine.from_json(load_golden(name)["machine"])


def make(capi, fm, engine=-1):
    capi.set_engine(engine)
    try:
        return capi.Machine(fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    finally:
        capi.set_engine(-1)


def reads(name, lens):
    return [(x, y[:lo]) for (x, y), lo in zip(pairs_from_golden(load_golden(name)), lens)]


def split(lengths, off, ids):
    """[[path j of pair k]] from sample_paths' packed result."""
    n = lengths.shape[1]
    return [[ids[off[k * n + j]:off[k * n + j + 1]].tolist() for j in range(n)] for k in range(lengths.shape[0])]


def banded(li, lo, w):
    """Rows |i - o Li / Lo| <= w, widened where the band is steeper than one column per row so that it stays connected."""
    if lo == 0:
        return [(0, li + 1)]
    c = [(o * li) // lo for o in range(lo + 1)] + [li]
    return [(max(0, c[o] - w), min(li, max(c[o] + w, c[o + 1] - w - 1)) + 1) for o in range(lo + 1)]


def check_valid(fm, x, y, path, env=None):
    """The path chains from state 0 to the end state, spells out x and y, has a finite weight and stays in the envelope."""
    s, i, o, w = 0, 0, 0, 0.0
    inside = (lambda i, o: env[o][0] <= i < env[o][1]) if env is not None else (lambda i, o: True)
    assert inside(0, 0)
    for t in path:
        assert fm.src[t] == s
        if fm.tin[t]:
            assert i < len(x) and fm.tin[t] == x[i]
            i += 1
        if fm.tout[t]:
            assert o < len(y) and fm.tout[t] == y[o]
            o += 1
        s = int(fm.dst[t])
        w += float(fm.lw[t])
        assert inside(i, o), (i, o)
    assert s == fm.n_states - 1 and i == len(x) and o == len(y) and math.isfinite(w)


# ---------------------------------------------------------------------------------------------
# 1. exact replay
# ---------------------------------------------------------------------------------------------
REPLAY_CASES = ["dnapsw_small", "unitindel", "stutter_noise_difflen", "hmmer_pf00516_reads"]


@pytest.mark.parametrize("name", REPLAY_CASES)
def test_paths_replay_on_the_host(name):
    capi = _capi()
    fm = golden_machine(name)
    pairs = reads(name, (12, 30)) if name == "hmmer_pf00516_reads" else pairs_from_golden(load_golden(name))
    m = make(capi, fm)
    b = capi.Batch(pairs)
    inc = Incoming(fm)
    mats = [capi.matrix(m, b, k, 0) for k in range(len(pairs))]
    n_checked = 0
    for seed, n in ((1, 5), (2 ** 40 + 77, 3), (123456789, 4)):
        ll, lengths, off, ids = capi.sample_paths(m, b, n, seed)
        got = split(lengths, off, ids)
        for k, (x, y) in enumerate(pairs):
            for j in range(n):
                want = replay(inc, mats[k], x, y, seed, k, j)
                assert got[k][j] == want, (name, seed, k, j)
                n_checked += len(want) > 0
    assert n_checked >= 6


# ---------------------------------------------------------------------------------------------
# 2. posterior statistics
# ---------------------------------------------------------------------------------------------
def usage_stats(lengths, off, ids, n_trans, expected):
    """Per transition: mean use per path and its standard error, over the paths of one pair.  The variance is at least that of
    a use with probability min(E, 1): a rare transition that no draw took has a sample variance of 0, not its true one."""
    n = lengths.size
    path_of = np.repeat(np.arange(n), lengths.ravel())
    keys, c = np.unique(path_of.astype(np.int64) * n_trans + ids.astype(np.int64), return_counts=True)
    t = keys % n_trans
    s1 = np.bincount(t, weights=c, minlength=n_trans)
    s2 = np.bincount(t, weights=c.astype(np.float64) ** 2, minlength=n_trans)
    mean = s1 / n
    p = np.minimum(expected, 1.0)
    var = np.maximum(np.maximum(s2 / n - mean ** 2, 0.0) * n / (n - 1), p * (1 - p))
    return mean, np.sqrt(var / n)


def check_posterior(capi, fm, pairs, envs=None, n=4000, seed=2024):
    m = make(capi, fm)
    for k, pair in enumerate(pairs):
        b = capi.Batch([pair])
        if envs is not None:
            b.set_envelopes([envs[k]])
        expected, ll = capi.counts(m, b)
        assert math.isfinite(ll[0])
        _, lengths, off, ids = capi.sample_paths(m, b, n, seed + k)
        mean, se = usage_stats(lengths, off, ids, fm.n_trans, expected)
        bound = 6 * se + 1e-3 * (1 + expected)
        bad = np.nonzero(np.abs(mean - expected) > bound)[0]
        assert bad.size == 0, [(int(t), mean[t], expected[t], se[t]) for t in bad[:5]]
        assert expected.sum() > 0


def test_posterior_usage_dnapsw():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = [p for p in pairs_from_golden(load_golden("dnapsw_small")) if len(p[0]) + len(p[1]) >= 6]
    assert len(pairs) >= 2
    check_posterior(capi, fm, pairs)


def test_posterior_usage_prot2dna_dnapsw():
    capi = _capi()
    check_posterior(capi, golden_machine("prot2dna_dnapsw"), pairs_from_golden(load_golden("prot2dna_dnapsw"))[:1])


def test_posterior_usage_profile_reads():
    capi = _capi()
    check_posterior(capi, golden_machine("hmmer_pf00516_reads"), reads("hmmer_pf00516_reads", (20, 35)))


def test_posterior_usage_banded_envelope():
    capi = _capi()
    case = load_golden("dnapsw_small")
    pairs = [p for p in pairs_from_golden(case) if len(p[0]) >= 4 and len(p[1]) >= 3][:2]
    envs = [banded(len(x), len(y), 1) for x, y in pairs]
    check_posterior(capi, golden_machine("dnapsw_small"), pairs, envs)


# ---------------------------------------------------------------------------------------------
# 3. validity, 4. log-likelihoods
# ---------------------------------------------------------------------------------------------
def trap_without_b():
    """State 1 emits a's and never leaves; state 2 emits a's and reaches the end; nothing emits b: a read with b has no path."""
    trans = [(0, 1, 0, 0, 0.0), (0, 2, 0, 0, 0.0), (1, 1, 0, 1, 0.0), (2, 2, 0, 1, math.log(0.125)), (2, 2, 0, 2, -math.inf), (2, 3, 0, 0, 0.0)]
    a = np.array(trans)
    return FlatMachine(4, 0, 2, a[:, 0].astype(np.int32), a[:, 1].astype(np.int32), a[:, 2].astype(np.int32),
                       a[:, 3].astype(np.int32), a[:, 4].astype(np.float64), [], ["a", "b"])


def test_paths_are_valid_and_impossible_pairs_get_none():
    capi = _capi()
    fm = trap_without_b()
    pairs = [(np.zeros(0, np.uint8), np.array(y, np.uint8)) for y in ([1] * 40, [1, 1, 2], [1] * 400, [])]      # 400 a's: every path's weight is below exp(-745)
    m = make(capi, fm)
    b = capi.Batch(pairs)
    ll, lengths, off, ids = capi.sample_paths(m, b, 6, 99)
    got = split(lengths, off, ids)
    assert math.isinf(ll[1]) and (lengths[1] == 0).all()
    for k in (0, 2, 3):
        assert math.isfinite(ll[k])
        for p in got[k]:
            check_valid(fm, *pairs[k], p)


def test_paths_stay_in_their_envelopes():
    capi = _capi()
    full = golden_machine("dnapsw_small")
    keep = ~((full.tin > 0) & (full.tout > 0))
    no_match = FlatMachine(full.n_states, full.n_in, full.n_out, full.src[keep], full.dst[keep], full.tin[keep], full.tout[keep],
                           full.lw[keep], full.in_alphabet, full.out_alphabet)
    rng = np.random.default_rng(5)
    pairs = [(rng.integers(1, 5, li).astype(np.uint8), rng.integers(1, 5, lo).astype(np.uint8)) for li, lo in ((20, 24), (15, 15), (30, 26), (9, 9))]
    envs = [banded(20, 24, 1), [(o, o + 1) for o in range(16)], banded(30, 26, 0), None]
    # without match transitions no path follows the diagonal (nor, here, the narrow bands); the envelope-free pair keeps one
    for fm, impossible, possible in ((full, (), (0, 1, 2, 3)), (no_match, (1,), (3,))):
        m = make(capi, fm)
        b = capi.Batch(pairs)
        b.set_envelopes(envs)
        ll, lengths, off, ids = capi.sample_paths(m, b, 8, 31)
        got = split(lengths, off, ids)
        assert all(math.isinf(ll[k]) for k in impossible) and all(math.isfinite(ll[k]) for k in possible), ll
        for k, (x, y) in enumerate(pairs):
            if math.isinf(ll[k]):
                assert (lengths[k] == 0).all()
                continue
            for p in got[k]:
                check_valid(fm, x, y, p, envs[k])


@pytest.mark.parametrize("name", ["dnapsw_small", "prot2dna_dnapsw", "hmmer_pf00516_reads"])
def test_loglike_is_the_generic_forward(name):
    capi = _capi()
    fm = golden_machine(name)
    pairs = reads(name, (15, 40, 60)) if name == "hmmer_pf00516_reads" else pairs_from_golden(load_golden(name))
    m = make(capi, fm, capi.ENGINE_GENERIC)
    b = capi.Batch(pairs)
    want = capi.forward(m, b)
    ll, lengths, _, _ = capi.sample_paths(m, b, 2, 5)
    assert ll.tobytes() == want.tobytes()
    m2 = make(capi, fm)      # the machine's own engine does not matter: sampling runs on the generic engine
    ll2, _, _, _ = capi.sample_paths(m2, b, 2, 5)
    assert ll2.tobytes() == want.tobytes()


# ---------------------------------------------------------------------------------------------
# 5. determinism and independence, 6. the two path stores
# ---------------------------------------------------------------------------------------------
def test_paths_depend_only_on_seed_pair_and_sample():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    case = load_golden("dnapsw_small")
    pairs = [p for p in pairs_from_golden(case) if len(p[0]) + len(p[1]) >= 6][:3]
    m = make(capi, fm)
    b3 = capi.Batch(pairs)
    first = capi.sample_paths(m, b3, 4, 77)
    again = capi.sample_paths(m, b3, 4, 77)
    assert all(np.array_equal(u, v) for u, v in zip(first, again))
    b2 = capi.Batch(pairs[:2])
    two = capi.sample_paths(m, b2, 4, 77)
    assert split(*two[1:])[:2] == split(*first[1:])[:2]
    other = capi.sample_paths(m, b3, 4, 78)
    assert split(*other[1:]) != split(*first[1:])
    for width in (1, 2):
        narrow = capi.sample_paths(m, b3, 4, 77, bytes_per_id=width)
        assert narrow[3].dtype.itemsize == width and np.array_equal(narrow[3].astype(np.int32), first[3])
    big = make(capi, golden_machine("hmmer_pf00516_reads"))
    rb = capi.Batch(reads("hmmer_pf00516_reads", (10,)))
    with pytest.raises(capi.MachineBossError, match="do not fit in 1 byte"):
        capi.sample_paths(big, rb, 2, 1, bytes_per_id=1)


def fetch_fails(capi, b):
    """mb_sampled_paths refuses (nothing stored): returns the message."""
    assert capi.lib().mb_sampled_paths(b.h, None, 4, None) != 0
    return capi.lib().mb_last_error().decode()


def test_viterbi_and_sampled_paths_are_stored_apart():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = pairs_from_golden(load_golden("dnapsw_small"))
    m = make(capi, fm)
    b = capi.Batch(pairs)
    assert "no samples stored" in fetch_fails(capi, b)
    score, plen = capi.viterbi_lengths(m, b)
    vit = capi.viterbi_paths(b, plen)
    ll, lengths, off, ids = capi.sample_paths(m, b, 3, 11)
    assert off[-1] > 0
    assert all(np.array_equal(u, v) for u, v in zip(capi.viterbi_paths(b, plen), vit))      # Viterbi paths survive sampling
    capi.viterbi_lengths(m, b)
    again = np.empty_like(ids)
    capi._check(capi.lib().mb_sampled_paths(b.h, again.ctypes.data, 4, off.ctypes.data))
    assert np.array_equal(again, ids)      # samples survive a Viterbi call
    with pytest.raises(capi.MachineBossError, match="nSamples must be at least 1"):
        capi.sample_paths(m, b, 0, 1)
    assert "no samples stored" in fetch_fails(capi, b)      # a failed call leaves no samples stored
    assert all(np.array_equal(u, v) for u, v in zip(capi.viterbi_paths(b, plen), vit))


# ---------------------------------------------------------------------------------------------
# 7. the CLI
# ---------------------------------------------------------------------------------------------
def test_cli_posterior_paths_match_the_library():
    from machineboss_b200 import build
    capi = _capi()
    case = load_golden("dnapsw_small")
    m = case["machine"]
    ia, oa = [""] + m["inAlphabet"], [""] + m["outAlphabet"]
    mf = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
    json.dump(m, mf)
    mf.close()
    pf = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
    json.dump([{"input": {"name": "x%d" % k, "sequence": [ia[t] for t in p["x"]]},
                "output": {"name": "y%d" % k, "sequence": [oa[t] for t in p["y"]]}} for k, p in enumerate(case["pairs"])], pf)
    pf.close()
    r = subprocess.run([build.build_host(), "--evaluated-machine", mf.name, "-D", pf.name, "--posterior-paths", "3", "--posterior-seed", "7"],
                       capture_output=True, text=True, check=True)
    got = json.loads(r.stdout)
    fm = FlatMachine.from_json(m)
    pairs = pairs_from_golden(case)
    ll, lengths, off, ids = capi.sample_paths(make(capi, fm), capi.Batch(pairs), 3, 7)
    want = [paths if math.isfinite(ll[k]) else [] for k, paths in enumerate(split(lengths, off, ids))]
    assert got == want
