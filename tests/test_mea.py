"""Posterior decoding for a whole batch on the device (mb_mea, mb_mea_paths, mb_path_posteriors; -m gpu).

Every result is recomputed on the host by tests/mea_reference.py over the same pair's stored Forward and Backward matrices
(mb_matrix: the same fills with the same bits), and the MEA gain is checked to be at least that of the Viterbi path and of
paths drawn from the posterior."""
import json
import math
import subprocess
import tempfile

import numpy as np
import pytest

from helpers import FlatMachine, load_golden, pairs_from_golden, synth_tokens
from mea_reference import gain_of, mea_path, path_gammas
from sample_replay import Incoming

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


def split(off, ids):
    return [ids[off[k]:off[k + 1]].astype(np.int64).tolist() for k in range(len(off) - 1)]


def check_against_reference(capi, fm, pairs, envs=None):
    """mb_mea against the host DP over the pair's own mb_matrix values."""
    m = make(capi, fm)
    b = capi.Batch(pairs)
    if envs is not None:
        b.set_envelopes(envs)
    gain, ll, lengths, off, ids, post = capi.mea(m, b)
    inc = Incoming(fm)
    n_compared = 0
    for k, (x, y) in enumerate(pairs):
        env = envs[k] if envs is not None else None
        F, B = capi.matrix(m, b, k, 0), capi.matrix(m, b, k, 1)
        want, ref_ids, _, ties = mea_path(inc, F, B, x, y, env)
        got = ids[off[k]:off[k + 1]].astype(np.int64).tolist()
        if want == -math.inf:
            assert gain[k] == -math.inf and lengths[k] == 0
            continue
        assert abs(gain[k] - want) <= 1e-9 * max(1.0, abs(want)), (k, gain[k], want)
        check_valid(fm, x, y, got, env)
        g = post[off[k]:off[k + 1]]
        np.testing.assert_allclose(g, path_gammas(fm, F, B, x, y, got), rtol=0, atol=1e-12)
        assert abs(gain_of(fm, got, g) - gain[k]) <= 1e-9 * max(1.0, abs(gain[k]))
        assert ((g >= 0) & (g <= 1 + 1e-4)).all()
        # the traceback walks from the end: the paths agree step for step until the host meets a near tie
        for j in range(1, len(ref_ids) + 1):
            if ties[-j]:
                break
            assert j <= len(got) and got[-j] == ref_ids[-j], (k, j)
        else:
            assert len(got) == len(ref_ids)
        n_compared += 1
    return n_compared


# ---------------------------------------------------------------------------------------------
# 1. against the host restatement
# ---------------------------------------------------------------------------------------------
REFERENCE_CASES = ["dnapsw_small", "unitindel", "stutter_noise_difflen", "bitnoise_p09", "prot2dna_dnapsw", "hmmer_pf00516_reads"]


@pytest.mark.parametrize("name", REFERENCE_CASES)
def test_mea_matches_the_reference(name):
    capi = _capi()
    fm = golden_machine(name)
    pairs = pairs_from_golden(load_golden(name))
    if name == "prot2dna_dnapsw":
        pairs = [(x[:3], y[:9]) for x, y in pairs] + [(x[:2], y[:7]) for x, y in pairs]
    if name == "hmmer_pf00516_reads":
        pairs = [(x, y[:lo]) for (x, y), lo in zip(pairs, (12, 20, 16))]
    assert check_against_reference(capi, fm, pairs) >= 1


def test_loglike_is_the_generic_forward():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = pairs_from_golden(load_golden("dnapsw_small"))
    b = capi.Batch(pairs)
    want = capi.forward(make(capi, fm, capi.ENGINE_GENERIC), b)
    _, ll, _, _, _, _ = capi.mea(make(capi, fm), b)
    assert ll.tobytes() == want.tobytes()


# ---------------------------------------------------------------------------------------------
# 2. optimality, 3. validity
# ---------------------------------------------------------------------------------------------
def path_gains(fm, off, ids, post):
    """Gain of each packed path, summed start -> end."""
    n = len(off) - 1
    c = ((fm.tin[ids] > 0).astype(np.float64) + (fm.tout[ids] > 0).astype(np.float64))
    return np.bincount(np.repeat(np.arange(n), np.diff(off)), weights=c * post, minlength=n)


def check_optimal(capi, fm, pairs, n_samples=64):
    m = make(capi, fm)
    b = capi.Batch(pairs)
    gain, ll, lengths, off, ids, post = capi.mea(m, b)
    n = len(pairs)
    assert ((post >= 0) & (post <= 1 + 1e-4)).all()
    for k, p in enumerate(split(off, ids)):
        if math.isfinite(gain[k]):
            check_valid(fm, *pairs[k], p)
    tol = 1e-12 * (1 + np.abs(np.where(np.isfinite(gain), gain, 0)))      # gains are sums of up to Li + Lo + silent terms
    score, vpaths = capi.viterbi(m, b)
    ok = np.isfinite(score)
    keep = np.nonzero(ok)[0]
    voff = np.concatenate([[0], np.cumsum([len(vpaths[k]) for k in keep])]).astype(np.int64)
    vids = np.concatenate([vpaths[k] for k in keep] + [np.zeros(0, np.int32)])
    vg = path_gains(fm, voff, vids.astype(np.int64), capi.path_posteriors(m, b, keep, voff, vids))
    assert (gain[ok] >= vg - tol[ok]).all(), np.min(gain[ok] - vg)
    _, slen, soff, sids = capi.sample_paths(m, b, n_samples, 4242)
    spair = np.repeat(np.arange(n), n_samples)
    spost = capi.path_posteriors(m, b, spair, soff, sids)
    sg = path_gains(fm, soff, sids.astype(np.int64), spost)
    has = slen.ravel() > 0
    assert (gain[spair[has]] >= sg[has] - tol[spair[has]]).all(), np.min(gain[spair[has]] - sg[has])
    assert ((spost >= 0) & (spost <= 1 + 1e-4)).all()
    assert (gain[ok] <= np.array([len(x) + len(y) for x, y in pairs])[ok] + 1e-9).all()
    return int(ok.sum())


def test_mea_gain_beats_viterbi_and_samples_dnapsw_small():
    capi = _capi()
    assert check_optimal(capi, golden_machine("dnapsw_small"), pairs_from_golden(load_golden("dnapsw_small"))) >= 5


def test_mea_gain_beats_viterbi_and_samples_synthetic_300():
    capi = _capi()
    fm = golden_machine("dnapsw_synth300")
    pairs = [(synth_tokens(102, k, 0, 300 - k % 7, 4), synth_tokens(102, k, 1, 257 + k % 5, 4)) for k in range(300)]
    assert check_optimal(capi, fm, pairs) == 300


# ---------------------------------------------------------------------------------------------
# 4. envelopes
# ---------------------------------------------------------------------------------------------
def test_envelopes():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    rng = np.random.default_rng(8)
    pairs = [(rng.integers(1, 5, li).astype(np.uint8), rng.integers(1, 5, lo).astype(np.uint8)) for li, lo in ((20, 24), (15, 15), (30, 26), (9, 9))]
    envs = [banded(20, 24, 1), [(o, o + 1) for o in range(16)], banded(30, 26, 0), None]
    assert check_against_reference(capi, fm, pairs, envs) == 4


# ---------------------------------------------------------------------------------------------
# 5. edge cases
# ---------------------------------------------------------------------------------------------
def trap_without_b():
    """State 1 emits a's and never leaves; state 2 emits a's and reaches the end; nothing emits b: a read with b has no path."""
    trans = [(0, 1, 0, 0, 0.0), (0, 2, 0, 0, 0.0), (1, 1, 0, 1, 0.0), (2, 2, 0, 1, math.log(0.125)), (2, 2, 0, 2, -math.inf), (2, 3, 0, 0, 0.0)]
    a = np.array(trans)
    return FlatMachine(4, 0, 2, a[:, 0].astype(np.int32), a[:, 1].astype(np.int32), a[:, 2].astype(np.int32),
                       a[:, 3].astype(np.int32), a[:, 4].astype(np.float64), [], ["a", "b"])


def test_impossible_and_empty_pairs():
    capi = _capi()
    fm = trap_without_b()
    pairs = [(np.zeros(0, np.uint8), np.array(y, np.uint8)) for y in ([1] * 40, [1, 1, 2], [])]
    gain, ll, lengths, off, ids, post = capi.mea(make(capi, fm), capi.Batch(pairs))
    assert gain[1] == -math.inf and lengths[1] == 0 and ll[1] == -math.inf
    assert abs(gain[0] - 40) <= 1e-9 and gain[2] == 0
    paths = split(off, ids)
    check_valid(fm, *pairs[0], paths[0])
    # the empty read's only path is silent and forced: each step has posterior 1
    check_valid(fm, *pairs[2], paths[2])
    assert paths[2] == [1, 5] and np.allclose(post[off[2]:off[3]], 1, rtol=0, atol=1e-12)
    # unitindel's empty pair: one silent step, forced
    ufm = golden_machine("unitindel")
    g, _, ul, uoff, uids, upost = capi.mea(make(capi, ufm), capi.Batch([(np.zeros(0, np.uint8), np.zeros(0, np.uint8))]))
    assert g[0] == 0 and uids.tolist() == [3] and abs(upost[0] - 1) <= 1e-12


def test_one_state_machine():
    capi = _capi()
    fm = golden_machine("bitnoise_tiny")
    assert fm.n_states == 1
    x, y = pairs_from_golden(load_golden("bitnoise_tiny"))[0]
    pairs = [(np.zeros(0, np.uint8), np.zeros(0, np.uint8)), (x, y)]
    gain, ll, lengths, off, ids, post = capi.mea(make(capi, fm), capi.Batch(pairs))
    assert gain[0] == 0 and lengths[0] == 0
    assert lengths[1] == 3 and abs(gain[1] - 6) <= 1e-9 and np.allclose(post, 1, atol=1e-12)


# ---------------------------------------------------------------------------------------------
# 6. determinism, independence, engines, narrowing, the three path stores
# ---------------------------------------------------------------------------------------------
def test_determinism_and_independence():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = [p for p in pairs_from_golden(load_golden("dnapsw_small")) if len(p[0]) + len(p[1]) >= 6][:3]
    m = make(capi, fm)
    b3 = capi.Batch(pairs)
    first = capi.mea(m, b3)
    again = capi.mea(m, b3)
    assert all(np.array_equal(u, v) for u, v in zip(first, again))
    two = capi.mea(m, capi.Batch(pairs[:2]))
    assert np.array_equal(two[0], first[0][:2]) and split(two[3], two[4]) == split(first[3], first[4])[:2]
    assert np.array_equal(two[5], first[5][: two[3][-1]])
    gen = capi.mea(make(capi, fm, capi.ENGINE_GENERIC), b3)
    jit = capi.mea(make(capi, fm, capi.ENGINE_JIT), b3)
    assert all(np.array_equal(u, v) for u, v in zip(gen, jit)) and all(np.array_equal(u, v) for u, v in zip(gen, first))
    for width in (1, 2):
        narrow = capi.mea(m, b3, bytes_per_id=width)
        assert narrow[4].dtype.itemsize == width and np.array_equal(narrow[4].astype(np.int32), first[4])
        assert np.array_equal(narrow[5], first[5])
    big = make(capi, golden_machine("hmmer_pf00516_reads"))
    x, y = pairs_from_golden(load_golden("hmmer_pf00516_reads"))[0]
    with pytest.raises(capi.MachineBossError, match="do not fit in 1 byte"):
        capi.mea(big, capi.Batch([(x, y[:10])]), bytes_per_id=1)


def mea_fetch_fails(capi, b):
    assert capi.lib().mb_mea_paths(b.h, None, 4, None, None) != 0
    return capi.lib().mb_last_error().decode()


def test_three_path_stores_are_kept_apart():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = pairs_from_golden(load_golden("dnapsw_small"))
    m = make(capi, fm)
    b = capi.Batch(pairs)
    assert "no MEA paths stored" in mea_fetch_fails(capi, b)
    score, plen = capi.viterbi_lengths(m, b)
    vit = capi.viterbi_paths(b, plen)
    _, slen, soff, sids = capi.sample_paths(m, b, 3, 11)
    gain, _, lengths, off, ids, post = capi.mea(m, b)
    assert off[-1] > 0
    assert all(np.array_equal(u, v) for u, v in zip(capi.viterbi_paths(b, plen), vit))      # Viterbi paths survive mb_mea
    again = np.empty_like(sids)
    capi._check(capi.lib().mb_sampled_paths(b.h, again.ctypes.data, 4, soff.ctypes.data))
    assert np.array_equal(again, sids)      # and so do the samples
    capi.viterbi_lengths(m, b)
    capi.sample_paths(m, b, 2, 5)
    ids2, post2 = np.empty_like(ids), np.empty_like(post)
    capi._check(capi.lib().mb_mea_paths(b.h, ids2.ctypes.data, 4, off.ctypes.data, post2.ctypes.data))
    assert np.array_equal(ids2, ids) and np.array_equal(post2, post)      # MEA paths survive both
    assert capi.lib().mb_mea(m.h, b.h, None, None, None) != 0      # a failed call (null gain) ...
    assert "null gain" in capi.lib().mb_last_error().decode()
    assert "no MEA paths stored" in mea_fetch_fails(capi, b)      # ... leaves no MEA paths stored
    assert all(np.array_equal(u, v) for u, v in zip(capi.viterbi_paths(b, plen), vit))


# ---------------------------------------------------------------------------------------------
# 7. rejections
# ---------------------------------------------------------------------------------------------
def test_path_posteriors_rejects_paths_that_are_not_paths_of_their_pair():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = pairs_from_golden(load_golden("dnapsw_small"))
    m = make(capi, fm)
    b = capi.Batch(pairs)
    _, vpaths = capi.viterbi(m, b)
    has_match = [k for k in range(len(pairs)) if any(fm.tin[t] and fm.tout[t] for t in vpaths[k])]
    k = max(has_match, key=lambda k: len(vpaths[k]))      # the longest Viterbi path with a match step
    good = vpaths[k].astype(np.int64).tolist()
    other = max(range(len(pairs)), key=lambda j: len(vpaths[j]) if j != k else -1)

    def run(paths):      # a valid path of pair `other`, then `paths` (one path of pair k)
        pair_of = [other, k]
        off = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.int64)
        return capi.path_posteriors(m, b, pair_of, off, np.concatenate([np.array(p, np.int32) for p in paths]))

    post = run([vpaths[other].tolist(), good])
    assert post.shape[0] == len(good) + len(vpaths[other])
    # step n of the path: a match whose input token is replaced by another from the same state
    n = next(n for n, t in enumerate(good) if fm.tin[t] and fm.tout[t])
    t = good[n]
    swap = next(u for u in range(fm.n_trans) if fm.src[u] == fm.src[t] and fm.dst[u] == fm.dst[t] and fm.tout[u] == fm.tout[t] and fm.tin[u] not in (0, fm.tin[t]))
    cases = [
        (good[:n] + [swap] + good[n + 1:], "path 1 \\(pair %d\\), step %d: transition %d does not read the pair's next input token" % (k, n, swap)),
        ([next(u for u in range(fm.n_trans) if fm.src[u] != 0)] + good, "path 1 \\(pair %d\\), step 0: .* does not leave the state the path is in" % k),
        (good[:-1], "path 1 \\(pair %d\\), step %d: the path ends before" % (k, len(good) - 1)),
    ]
    for path, msg in cases:
        with pytest.raises(capi.MachineBossError, match=msg):
            run([vpaths[other].tolist(), path])
    with pytest.raises(capi.MachineBossError, match="path 0 belongs to pair %d" % len(pairs)):
        capi.path_posteriors(m, b, [len(pairs)], [0, len(good)], np.array(good, np.int32))
    with pytest.raises(capi.MachineBossError, match="path 0, step 2: transition %d is not one of the machine's" % fm.n_trans):
        capi.path_posteriors(m, b, [k], [0, 3], np.array(good[:2] + [fm.n_trans], np.int32))
    # outside the envelope: a path drawn over the full matrix that leaves a one-cell-wide band
    xs, ys = (np.array([1, 2, 3, 4] * 3, np.uint8), np.array([1, 2, 3, 4] * 2, np.uint8))
    full = capi.Batch([(xs, ys)])
    _, slen, soff, sids = capi.sample_paths(m, full, 64, 3)
    env = banded(len(xs), len(ys), 0)
    band = capi.Batch([(xs, ys)])
    band.set_envelopes([env])

    def leaves(p):
        i = o = 0
        for t in p:
            i, o = i + (fm.tin[t] > 0), o + (fm.tout[t] > 0)
            if not env[o][0] <= i < env[o][1]:
                return True
        return False

    out = next(p for p in split(soff, sids) if leaves(p))
    with pytest.raises(capi.MachineBossError, match="path 0 \\(pair 0\\), step .*leaves the pair's envelope"):
        capi.path_posteriors(m, band, [0], [0, len(out)], np.array(out, np.int32))


# ---------------------------------------------------------------------------------------------
# 8. the CLI
# ---------------------------------------------------------------------------------------------
def test_cli_mea_and_viterbi_post_prob_match_the_library():
    from machineboss_b200 import build
    capi = _capi()
    case = load_golden("dnapsw_small")
    mj = case["machine"]
    ia, oa = [""] + mj["inAlphabet"], [""] + mj["outAlphabet"]
    mf = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
    json.dump(mj, mf)
    mf.close()
    pf = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
    json.dump([{"input": {"name": "x%d" % k, "sequence": [ia[t] for t in p["x"]]},
                "output": {"name": "y%d" % k, "sequence": [oa[t] for t in p["y"]]}} for k, p in enumerate(case["pairs"])]
              + [{"input": {"name": "bad", "sequence": ["Z"]}, "output": {"name": "bad", "sequence": [oa[1]]}}], pf)      # not tokenisable
    pf.close()
    cli = build.build_host()
    mea_out = json.loads(subprocess.run([cli, "--evaluated-machine", mf.name, "-D", pf.name, "--mea"], capture_output=True, text=True, check=True).stdout)
    vpp = json.loads(subprocess.run([cli, "--evaluated-machine", mf.name, "-D", pf.name, "--viterbi-post-prob"], capture_output=True, text=True, check=True).stdout)
    fm = FlatMachine.from_json(mj)
    pairs = pairs_from_golden(case)
    m = make(capi, fm)
    b = capi.Batch(pairs)
    gain, _, _, off, ids, post = capi.mea(m, b)
    score, vpaths = capi.viterbi(m, b)
    assert len(mea_out) == len(vpp) == len(pairs) + 1
    assert mea_out[-1] == {"input": "bad", "output": "bad", "gain": "-Infinity", "path": [], "postProb": []} and vpp[-1] == []
    for k in range(len(pairs)):
        e = mea_out[k]
        assert (e["input"], e["output"]) == ("x%d" % k, "y%d" % k)
        if math.isfinite(gain[k]):
            assert e["gain"] == pytest.approx(gain[k], rel=1e-15, abs=1e-15)
            assert e["path"] == ids[off[k]:off[k + 1]].tolist()
            assert e["postProb"] == pytest.approx(post[off[k]:off[k + 1]].tolist(), rel=1e-15, abs=1e-300)
        else:
            assert e["gain"] == "-Infinity" and e["path"] == [] and e["postProb"] == []
        want = capi.path_posteriors(m, b, [k], [0, len(vpaths[k])], vpaths[k]) if math.isfinite(score[k]) else []
        assert vpp[k] == pytest.approx(list(want), rel=1e-15, abs=1e-300)
