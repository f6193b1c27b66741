"""Viterbi tie-breaking, the wide engine's launch shapes and envelope-restricted DP, every engine against the C oracle.

Under fitted or random weights two candidates of a cell almost never have the same FP64 score, so an engine's rule for
picking the FIRST maximum (dpmatrix.defs.h:171-174) is never consulted.  Here every finite log-weight is replaced by a small
integer (tied()): every path score is an exact integer sum, ties are real and frequent, and the tie-break decides the path
in most cells.  Viterbi scores must still equal the oracle's bit for bit and the paths must be the oracle's, and Forward
must equal the exact-sum oracle to 1e-9 relative (the weights lie well inside the linear sweeps' window).

The GPU tests are marked gpu; the host emulations of the column and lane programs at the end run without a device.
"""
import math
import re

import numpy as np
import pytest

from helpers import LSE_EXACT, FlatMachine, Oracle, load_golden, synth_tokens, synthetic_profile
from test_gpu_parity import forward_agrees
from test_lane_program_host import _walk as lane_walk

ROUTE = re.compile(r"^(mb_forward|mb_viterbi|mb_viterbi \(scores\)|mb_backward|mb_counts): (\S+) engine$", re.M)
NONE = np.zeros(0, np.uint8)


def tied(fm: FlatMachine, seed: int, values=(-1.0, -2.0)) -> FlatMachine:
    """The machine with every finite log-weight replaced by one of `values` (drawn with a fixed seed); -inf stays -inf."""
    rng = np.random.default_rng(seed)
    draw = rng.choice(np.asarray(values, dtype=np.float64), size=fm.n_trans)
    return fm.with_weights(np.where(np.isfinite(fm.lw), draw, fm.lw))


def golden_machine(name: str) -> FlatMachine:
    return FlatMachine.from_json(load_golden(name)["machine"])


def with_emitting_accumulator(fm: FlatMachine, n_nodes: int) -> FlatMachine:
    """synthetic_profile with a token-consuming M(k) -> E transition for every node and token: the column engine then
    sums into an emitting accumulator for the suffix (col_emulate info[7] == 2)."""
    E = 3 + 3 * n_nodes
    rows = list(zip(fm.src, fm.dst, fm.tin, fm.tout, fm.lw))
    for k in range(1, n_nodes + 1):
        for c in range(1, fm.n_out + 1):
            rows.append((3 + 3 * (k - 1), E, 0, c, -1.0))
    rows.sort(key=lambda r: r[0])      # the reference enumerates transitions state by state
    a = np.array(rows, dtype=np.float64)
    return FlatMachine(fm.n_states, 0, fm.n_out, a[:, 0].astype(np.int32), a[:, 1].astype(np.int32), a[:, 2].astype(np.int32),
                       a[:, 3].astype(np.int32), a[:, 4], [], fm.out_alphabet)


def without_matches(fm: FlatMachine) -> FlatMachine:
    """The machine without its match transitions (those consuming an input and an output token)."""
    keep = ~((fm.tin > 0) & (fm.tout > 0))
    return FlatMachine(fm.n_states, fm.n_in, fm.n_out, fm.src[keep], fm.dst[keep], fm.tin[keep], fm.tout[keep], fm.lw[keep],
                       fm.in_alphabet, fm.out_alphabet)


def machine(capi, fm: FlatMachine, engine: int = -1, **options):
    """A device machine created under a forced engine and options (None: the built-in choice)."""
    capi.set_engine(engine)
    for k, v in options.items():
        capi.set_option(k, v)
    try:
        return capi.Machine(fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    finally:
        capi.set_engine(-1)
        for k in options:
            capi.set_option(k, None)


def pairs_of(fm, seed, shapes):
    return [(synth_tokens(seed, k, 0, li, max(fm.n_in, 1)) if li else NONE, synth_tokens(seed, k, 1, lo, fm.n_out))
            for k, (li, lo) in enumerate(shapes)]


def reads_of(fm, seed, lens):
    return [(NONE, synth_tokens(seed, k, 1, lo, fm.n_out)) for k, lo in enumerate(lens)]


def full_envelopes(pairs):
    return [[(0, len(x) + 1)] * (len(y) + 1) for x, y in pairs]


def oracle_results(fm, pairs, envs=None):
    """[(Viterbi score, path, exact Forward)] per pair, each under its envelope (None: the full matrix)."""
    orc = Oracle(fm)
    out = []
    try:
        for k, (x, y) in enumerate(pairs):
            orc.set_envelope(envs[k] if envs is not None else None)
            v, p = orc.viterbi(x, y)
            out.append((v, p.tolist(), orc.forward(x, y, mode=LSE_EXACT)))
    finally:
        orc.set_envelope(None)
    return out


_CACHE = {}


def oracle_cached(key, fm, pairs):
    if key not in _CACHE:
        _CACHE[key] = oracle_results(fm, pairs)
    return _CACHE[key]


def exact(got, want, rel=1e-9):
    if math.isinf(want):
        return got == want
    return abs(got - want) <= rel * max(1.0, abs(want))


def check_sweeps(capi, m, b, want, forward=True, what=""):
    """Forward (if the engine serves it), Viterbi with and without paths, against the oracle's results `want`.  Forward to
    1e-9 relative from the linear sweeps; when the call re-ran pairs in the log domain, whose softplus is FP32 (<= 1.2e-7
    absolute per operation), to 1e-6."""
    ll = capi.forward(m, b) if forward else None
    rel = 1e-9 if not forward or b.last_redo() == 0 else 1e-6
    sc, paths = capi.viterbi(m, b)
    sc2 = capi.viterbi(m, b, paths=False)
    for k, (v, p, f) in enumerate(want):
        assert sc[k] == v and sc2[k] == v, (what, k, sc[k], sc2[k], v)      # bit for bit
        assert paths[k].tolist() == p, (what, k, len(paths[k]), len(p))
        if forward:
            assert exact(ll[k], f, rel), (what, k, ll[k], f, b.last_redo())
    return sc, paths


def routes(capfd):
    return dict(ROUTE.findall(capfd.readouterr().err))


def _capi():
    from machineboss_b200 import capi
    return capi


# ---------------------------------------------------------------------------------------------
# 1. exact ties in every engine
# ---------------------------------------------------------------------------------------------
RAGGED = [(0, 0), (1, 0), (0, 1), (1, 1), (5, 40), (40, 5), (33, 33), (64, 64), (127, 129), (200, 150), (31, 32), (257, 3),
          (128, 100), (256, 316), (129, 77), (131, 40), (255, 64), (127, 33), (384, 20), (130, 0)]


def fitted_shapes(c):
    top = 32 * c - 1      # every pair in one strip of 32 * c columns
    return [(top, 120), (top - 1, 33), (0, 7), (1, 0), (top // 2, 200), (31, 64), (32, 31), (33, 400)]


LONG = [(1025, 900), (600, 700), (257, 300), (0, 7), (255, 1000), (511, 40)]
CHUNKED = [(300 - 11 * k, 280 + 9 * k) for k in range(12)]

JIT_VARIANTS = {
    "narrow0": (dict(jit_narrow=0), RAGGED, None),
    "narrow1": (dict(jit_narrow=1), RAGGED, None),
    "fit10": (dict(jit_fit_c=10), fitted_shapes(10), "fitted to the batch compiled: 10 columns per lane"),
    "fit5": (dict(jit_fit_c=5), fitted_shapes(5), "fitted to the batch compiled: 5 columns per lane"),
    "split": (dict(jit_split=1), LONG, "split-mode module compiled"),
    "tb_chunks": (dict(jit_tb_budget_mb=1), CHUNKED, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(JIT_VARIANTS))
@pytest.mark.parametrize("name", ["dnapsw_small", "protpsw_synth"])
def test_jit_engine_on_ties(capfd, name, variant):
    capi = _capi()
    options, shapes, note = JIT_VARIANTS[variant]
    fm = tied(golden_machine(name), 1)
    pairs = pairs_of(fm, 61, shapes)
    want = oracle_cached((name, variant), fm, pairs)
    m = machine(capi, fm, 1, verbose=1, **options)
    assert m.engine == capi.ENGINE_JIT
    b = capi.Batch(pairs)
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=(name, variant))
    bl = capi.backward(m, b)
    for k, (_, _, f) in enumerate(want):
        assert exact(bl[k], f, 1e-9 if b.last_redo() == 0 else 1e-6), (name, variant, k, bl[k], f, b.last_redo())
    err = capfd.readouterr().err
    assert "mb_viterbi: jit engine" in err
    if note:
        assert note in err, (variant, err[-2000:])
    if variant == "tb_chunks":      # the back-pointers went out in several chunks: the same paths through the packed entry point
        sc, paths = capi.viterbi(m, b)
        score, plen, off = np.empty(len(pairs)), np.zeros(len(pairs), np.int64), np.zeros(len(pairs) + 1, np.int64)
        trans = np.zeros(sum(len(p) for p in paths), dtype=np.uint16)
        capi.viterbi_into(m, b, score, plen, off, trans)
        for k, (_, p, _) in enumerate(want):
            assert trans[off[k]:off[k + 1]].tolist() == p, k


BIG_SHAPES = [(120, 700), (70, 150), (33, 400), (3, 10), (0, 4), (64, 64), (1, 0), (0, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("options", [dict(big_early_store=0), dict(big_early_store=1), dict(big_warps=1), dict(big_warps=4), dict(big_warps=8)],
                         ids=lambda o: "-".join("%s=%s" % kv for kv in o.items()))
def test_big_engine_on_ties(capfd, options):
    capi = _capi()
    fm = tied(golden_machine("prot2dna_dnapsw"), 2)
    pairs = pairs_of(fm, 31, BIG_SHAPES)
    want = oracle_cached("big", fm, pairs)
    m = machine(capi, fm, 2, verbose=1, **options)
    b = capi.Batch(pairs)
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=options)
    r = routes(capfd)
    assert r.get("mb_forward") == "big" and r.get("mb_viterbi") == "big" and r.get("mb_viterbi (scores)") == "big", r
    capi.forward(m, b)
    assert b.last_redo() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dnapsw_small", "prot2dna_dnapsw"])
def test_generic_engine_on_ties(name):
    capi = _capi()
    fm = tied(golden_machine(name), 1 if name == "dnapsw_small" else 2)
    pairs = pairs_of(fm, 61, RAGGED) if name == "dnapsw_small" else pairs_of(fm, 31, BIG_SHAPES)
    want = oracle_cached((name, "narrow0") if name == "dnapsw_small" else "big", fm, pairs)
    m = machine(capi, fm, 0)
    assert m.engine == capi.ENGINE_GENERIC
    b = capi.Batch(pairs)
    check_sweeps(capi, m, b, want, forward=False, what=name)
    # the generic engine's softplus stops at the reference's table cut-off (logsumexp.h:52): Forward by test_gpu_parity's rule
    ll, orc = capi.forward(m, b), Oracle(fm)
    for k, (x, y) in enumerate(pairs):
        assert forward_agrees(fm, x, y, ll[k], orc.forward(x, y)), (name, k, ll[k])


WIDE_2D_SHAPES = [(40, 130), (17, 60), (16, 33), (0, 5), (3, 0), (35, 90), (70, 150), (1, 1)]
WIDE_2D_DNA_SHAPES = [(70, 66), (33, 40), (0, 5), (6, 0), (129, 120), (1, 1)]
SHAPES_RUN = {}      # (machine, G) -> {W: "ran" / "no fit"}, for the report at the end of the session


@pytest.mark.gpu
@pytest.mark.parametrize("g", [32, 16, 8])
@pytest.mark.parametrize("name", ["prot2dna_dnapsw", "dnapsw_small"])
def test_wide_2d_launch_shapes_on_ties(capfd, name, g):
    """Every lane-group width G and W in {1, 2, 4, the default} column warps.  prot2dna => dnapsw has no match transitions
    (a ring of 2 cells); dnapsw has them (3 cells).  A combination is skipped only when no launch shape fits."""
    capi = _capi()
    base = golden_machine(name)
    fm = tied(base, 3)
    shapes = WIDE_2D_SHAPES if name == "prot2dna_dnapsw" else WIDE_2D_DNA_SHAPES
    pairs = pairs_of(fm, 11, shapes)
    want = oracle_cached(("wide2d", name), fm, pairs)
    has_match = bool(((fm.tin > 0) & (fm.tout > 0)).any())
    assert has_match == (name == "dnapsw_small")
    ran = {}
    for w in (1, 2, 4, None):
        m = machine(capi, fm, 2, no_big=1, verbose=1, wide_g=g, wide_w=w)
        assert "G=%d " % g in capfd.readouterr().err
        b = capi.Batch(pairs)
        try:
            capi.viterbi(m, b, paths=False)
        except capi.MachineBossError as e:
            if "no launch shape fits" not in str(e):
                raise
            ran[w] = "no fit"
            continue
        check_sweeps(capi, m, b, want, what=(name, g, w))
        r = routes(capfd)
        assert r.get("mb_forward") == "wide" and r.get("mb_viterbi") == "wide", r
        ran[w] = "ran"
    SHAPES_RUN[(name, g)] = ran
    print("wide 2-D %s G=%d: %s" % (name, g, ", ".join("W=%s %s" % (w or "default", s) for w, s in ran.items())))
    assert sum(s == "ran" for s in ran.values()) >= 2, ran


def _pf00516_lens():
    return [0, 1, 2, 15, 16, 17, 31, 32, 33, 50, 150, 275] + [5 + (k * 37) % 200 for k in range(20)]


@pytest.mark.gpu
@pytest.mark.parametrize("g", [32, 16, 8, None], ids=lambda g: "G=%s" % (g or "default"))
def test_wide_1d_sweep_on_ties(capfd, g):
    """Generator reads with envelopes go to the wide engine's 1-D sweep.  PF00516's end state has a list of 975 sources: 2-byte
    back-pointers, and lists cut into pieces whose best candidates meet in the shuffle tree."""
    capi = _capi()
    fm = tied(golden_machine("hmmer_pf00516"), 4)
    _, counts = np.unique(np.stack([fm.dst, fm.tin, fm.tout], 1), axis=0, return_counts=True)
    assert counts.max() > 63
    pairs = reads_of(fm, 27, _pf00516_lens())
    want = oracle_cached("pf00516", fm, pairs)
    m = machine(capi, fm, 2, verbose=1, wide_g=g)
    err = capfd.readouterr().err
    assert "bp 2 bytes" in err and (g is None or "G=%d " % g in err), err[-2000:]
    b = capi.Batch(pairs)
    b.set_envelopes(full_envelopes(pairs))
    check_sweeps(capi, m, b, want, what=g)
    r = routes(capfd)
    assert r.get("mb_forward") == "wide" and r.get("mb_viterbi") == "wide", r


SYNTH_LENS = [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, 64, 150, 301] + [5 + (k * 13) % 120 for k in range(60)]


def profile(name):
    if name == "synthetic":
        return tied(synthetic_profile(n_nodes=90), 5)
    if name == "synthetic_emit_acc":
        return tied(with_emitting_accumulator(synthetic_profile(n_nodes=90), 90), 6)
    return tied(golden_machine("hmmer_pf00516"), 4)


PROFILES = ["synthetic", "synthetic_emit_acc", "hmmer_pf00516"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synthetic", "synthetic_emit_acc"])
def test_wide_1d_sweep_on_tied_synthetic_profiles(capfd, name):
    capi = _capi()
    fm = profile(name)
    pairs = reads_of(fm, 39, SYNTH_LENS)
    want = oracle_cached(("profile", name), fm, pairs)
    m = machine(capi, fm, 2, verbose=1)
    b = capi.Batch(pairs)
    b.set_envelopes(full_envelopes(pairs))
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=name)
    r = routes(capfd)
    assert r.get("mb_forward") == "wide" and r.get("mb_viterbi") == "wide", r


def _profile_pairs(name, fm):
    lens = SYNTH_LENS if name != "hmmer_pf00516" else _pf00516_lens()
    return reads_of(fm, 39 if name != "hmmer_pf00516" else 27, lens)


def _profile_want(name, fm, pairs):
    return oracle_cached(("profile", name) if name != "hmmer_pf00516" else "pf00516", fm, pairs)


@pytest.mark.gpu
@pytest.mark.parametrize("options", [dict(col_c=1), dict(col_c=2), dict(col_c=3), dict(col_r=2)], ids=lambda o: "-".join("%s=%s" % kv for kv in o.items()))
@pytest.mark.parametrize("name", PROFILES)
def test_column_engine_on_ties(capfd, name, options):
    capi = _capi()
    fm = profile(name)
    pairs = _profile_pairs(name, fm)
    want = _profile_want(name, fm, pairs)
    m = machine(capi, fm, 2, verbose=1, **options)
    b = capi.Batch(pairs)
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=(name, options))
    r = routes(capfd)
    assert r.get("mb_forward") == "column" and r.get("mb_viterbi") == "column" and r.get("mb_viterbi (scores)") == "column", r


@pytest.mark.gpu
@pytest.mark.parametrize("reads_per_lane", [1, 2, 4])
@pytest.mark.parametrize("name", PROFILES)
def test_lane_engine_on_ties(capfd, name, reads_per_lane):
    capi = _capi()
    fm = profile(name)
    pairs = _profile_pairs(name, fm)
    want = _profile_want(name, fm, pairs)
    m = machine(capi, fm, 2, verbose=1, no_col=1, lane_r=reads_per_lane)
    b = capi.Batch(pairs)
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=(name, reads_per_lane))
    r = routes(capfd)
    assert r.get("mb_forward") == "lane" and r.get("mb_viterbi") == "lane" and r.get("mb_viterbi (scores)") == "lane", r


# ---------------------------------------------------------------------------------------------
# 2. envelope-restricted DP
# ---------------------------------------------------------------------------------------------
def banded(li, lo, w):
    """Rows |i - o Li / Lo| <= w, widened where the band is steeper than one column per row so that it stays connected."""
    if lo == 0:
        return [(0, li + 1)]
    c = [(o * li) // lo for o in range(lo + 1)] + [li]
    return [(max(0, c[o] - w), min(li, max(c[o] + w, c[o + 1] - w - 1)) + 1) for o in range(lo + 1)]


def ragged(li, lo, seed):
    """Rows around a random monotone path from (0, 0) to (Li, Lo), each widened by 0 - 2 cells on either side at random."""
    rng = np.random.default_rng(seed)
    ends = sorted(rng.integers(0, li + 1, lo).tolist()) + [li]
    rows, start = [], 0
    for o in range(lo + 1):
        a, e = start, ends[o]
        rows.append((max(0, a - int(rng.integers(0, 3))), min(li, e + int(rng.integers(0, 3))) + 1))
        start = e
    return rows


def diagonal(li, lo):
    """One cell per row on the diagonal (Li == Lo): connected, but only match transitions can follow it."""
    assert li == lo
    return [(o, o + 1) for o in range(lo + 1)]


ENV_CASES = [((30, 34), ("band", 0)), ((30, 34), ("band", 1)), ((40, 33), ("band", 3)), ((25, 29), ("ragged", 1)),
             ((50, 47), ("ragged", 2)), ((12, 12), ("diagonal",)), ((20, 25), None), ((0, 6), ("band", 1)), ((7, 0), ("band", 1)),
             ((45, 45), ("diagonal",)), ((9, 11), None), ((60, 52), ("band", 3))]


def envelope_of(shape, kind):
    li, lo = shape
    if kind is None:
        return None
    if kind[0] == "band":
        return banded(li, lo, kind[1])
    if kind[0] == "ragged":
        return ragged(li, lo, kind[1])
    return diagonal(li, lo)


def counts_agree_with_envelopes(fm, pairs, envs, got):
    """The rule of test_gpu_parity.counts_agree, each pair's oracle counts under its envelope: within 1e-4 relative of the
    table-based counts, or within 1e-5 of the exact sums while the table's own values sit within 5e-4 of those."""
    orc = Oracle(fm)
    table, ex = np.zeros(fm.n_trans), np.zeros(fm.n_trans)
    try:
        for k, (x, y) in enumerate(pairs):
            orc.set_envelope(envs[k])
            if math.isinf(orc.forward(x, y, mode=LSE_EXACT)):
                continue      # an impossible pair contributes nothing
            orc.counts(x, y, counts=table)
            orc.counts(x, y, mode=LSE_EXACT, counts=ex)
    finally:
        orc.set_envelope(None)
    if np.allclose(got, table, rtol=1e-4, atol=1e-7):
        return True
    return np.allclose(got, ex, rtol=1e-5, atol=1e-7) and np.allclose(table, ex, rtol=5e-4, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["random", "tied"])
@pytest.mark.parametrize("name", ["dnapsw", "dnapsw_without_matches"])
def test_envelopes_on_a_jit_machine(capfd, name, weights):
    """Banded (w = 0, 1, 3), ragged and diagonal envelopes next to envelope-less pairs: Forward and Viterbi on the wide engine,
    Backward, counts and whole matrices on the generic engine.  Without match transitions the diagonal envelope is connected
    but no path follows it: -inf, and an empty path."""
    capi = _capi()
    fm = golden_machine("dnapsw_synth64")
    if name == "dnapsw_without_matches":
        fm = without_matches(fm)
    fm = tied(fm, 7) if weights == "tied" else fm
    pairs = pairs_of(fm, 71, [s for s, _ in ENV_CASES])
    envs = [envelope_of(s, kind) for s, kind in ENV_CASES]
    want = oracle_results(fm, pairs, envs)
    if name == "dnapsw_without_matches":      # (most envelopes leave such a machine no path; the envelope-less pairs have one)
        assert all(math.isinf(want[k][0]) for k, (_, kind) in enumerate(ENV_CASES) if kind == ("diagonal",))
        assert sum(math.isfinite(v) for v, _, _ in want) >= 3
    else:
        assert all(math.isfinite(v) for v, _, _ in want)
    m = machine(capi, fm, -1, verbose=1)
    assert m.engine == capi.ENGINE_JIT
    b = capi.Batch(pairs)
    b.set_envelopes(envs)
    capfd.readouterr()
    check_sweeps(capi, m, b, want, what=(name, weights))
    bl = capi.backward(m, b)
    cnt, cll = capi.counts(m, b)
    r = routes(capfd)
    assert r == {"mb_forward": "wide", "mb_viterbi": "wide", "mb_viterbi (scores)": "wide", "mb_backward": "generic", "mb_counts": "generic"}, r
    orc = Oracle(fm)
    try:
        for k, (x, y) in enumerate(pairs):
            orc.set_envelope(envs[k])
            f = want[k][2]
            # the generic engine's softplus stops at the reference's table cut-off (logsumexp.h:52): test_gpu_parity's rule
            table = orc.forward(x, y)
            assert forward_agrees(fm, x, y, bl[k], table) and forward_agrees(fm, x, y, cll[k], table), (k, bl[k], cll[k], table)
            if k in (0, 3, 5, 6):      # band, ragged, diagonal, none: whole Forward / Backward / Viterbi matrices
                for kind, ref in ((0, orc.forward(x, y, matrix=True)[1]), (1, orc.backward(x, y, matrix=True)[1]),
                                  (2, orc.viterbi(x, y, path=False, matrix=True)[1])):
                    got = capi.matrix(m, b, k, kind)
                    fin = np.isfinite(ref)
                    assert np.array_equal(np.isfinite(got), fin), (k, kind)
                    if kind == 2:
                        assert np.array_equal(got[fin], ref[fin]), k
                    else:
                        np.testing.assert_allclose(got[fin], ref[fin], rtol=1e-4, atol=1e-5)      # the table interpolates
    finally:
        orc.set_envelope(None)
    # counts over the pairs that have a path (the reference's counts are NaN-poisoned by impossible pairs)
    live = [k for k, (v, _, _) in enumerate(want) if math.isfinite(v)]
    if len(live) < len(pairs):
        b = capi.Batch([pairs[k] for k in live])
        b.set_envelopes([envs[k] for k in live])
        cnt, _ = capi.counts(m, b)
    assert counts_agree_with_envelopes(fm, [pairs[k] for k in live], [envs[k] for k in live], cnt)


ENV_WIDE_CASES = [((40, 130), ("band", 3)), ((70, 150), ("band", 1)), ((35, 90), ("ragged", 3)), ((17, 60), None), ((66, 200), ("band", 0)),
                  ((50, 140), ("ragged", 4)), ((0, 5), ("band", 1))]


@pytest.mark.gpu
@pytest.mark.parametrize("g", [32, 16, 8])
@pytest.mark.parametrize("weights", ["random", "tied"])
def test_envelopes_on_multi_strip_pairs(capfd, weights, g):
    capi = _capi()
    fm = golden_machine("prot2dna_dnapsw")
    fm = tied(fm, 8) if weights == "tied" else fm
    pairs = pairs_of(fm, 13, [s for s, _ in ENV_WIDE_CASES])
    envs = [envelope_of(s, kind) for s, kind in ENV_WIDE_CASES]
    want = _CACHE.get(("env_wide", weights)) or _CACHE.setdefault(("env_wide", weights), oracle_results(fm, pairs, envs))
    assert sum(math.isfinite(v) for v, _, _ in want) >= 5
    m = machine(capi, fm, -1, verbose=1, wide_g=g)
    assert "G=%d " % g in capfd.readouterr().err
    b = capi.Batch(pairs)
    b.set_envelopes(envs)
    check_sweeps(capi, m, b, want, what=(weights, g))
    r = routes(capfd)
    assert r.get("mb_forward") == "wide" and r.get("mb_viterbi") == "wide", r


# ---------------------------------------------------------------------------------------------
# 3. the big engine hands pairs without a path to the wide engine's log-domain sweep
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_big_engine_hands_impossible_pairs_to_the_log_domain(capfd):
    """prot2dna => dnapsw that cannot emit nucleotide 1: pairs whose output holds it have no path.  The big engine's Forward
    re-runs exactly those through the wide engine's log-domain sweep; they come back -inf with empty paths, the rest match
    the oracle."""
    capi = _capi()
    base = tied(golden_machine("prot2dna_dnapsw"), 9)
    fm = base.with_weights(np.where(base.tout == 1, -np.inf, base.lw))
    pairs = []
    for k, (li, lo) in enumerate([(40, 130), (17, 60), (33, 100), (5, 14), (70, 150), (12, 40), (0, 3), (25, 80)]):
        x, y = synth_tokens(17, k, 0, li, fm.n_in), synth_tokens(17, k, 1, lo, fm.n_out)
        if k % 2:
            y = np.where(y == 1, 3, y).astype(np.uint8)
        pairs.append((x, y))
    want = oracle_results(fm, pairs)
    impossible = [k for k, (v, _, _) in enumerate(want) if math.isinf(v)]
    assert len(impossible) >= 3 and len(impossible) < len(pairs) - 2
    m = machine(capi, fm, -1, verbose=1)
    b = capi.Batch(pairs)
    capfd.readouterr()
    ll = capi.forward(m, b)
    assert b.last_redo() == len(impossible)
    sc, paths = check_sweeps(capi, m, b, want, forward=False)
    r = routes(capfd)
    assert r.get("mb_forward") == "big" and r.get("mb_viterbi") == "big", r
    for k, (v, p, f) in enumerate(want):
        if k in impossible:
            assert ll[k] == -np.inf and sc[k] == -np.inf and len(paths[k]) == 0, k
        else:
            assert exact(ll[k], f), (k, ll[k], f)


# ---------------------------------------------------------------------------------------------
# host emulation of the column and lane programs (no device)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", PROFILES)
def test_column_program_on_ties_on_the_host(name):
    from machineboss_b200 import capi
    fm = profile(name)
    args = (fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    orc = Oracle(fm)
    for k, lo in enumerate([0, 1, 2, 3, 5, 9, 17, 40, 95]):
        y = synth_tokens(41, k, 1, lo, fm.n_out)
        v, info, walked = capi.col_emulate(*args, y, 1, path=True)
        assert info[0] == 1
        want_v, want_p = orc.viterbi(NONE, y)
        assert v == want_v, (name, lo, v, want_v)
        assert walked.tolist() == want_p.tolist(), (name, lo)
    if name == "synthetic_emit_acc":
        assert info[7] == 2, info      # the suffix sums into an emitting accumulator


@pytest.mark.parametrize("name", ["hmmer_pf00516", "unitindel"])
def test_lane_program_on_ties_on_the_host(name):
    from machineboss_b200 import capi
    fm = tied(golden_machine(name), 10)
    args = (fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    orc = Oracle(fm)
    for k, lo in enumerate([0, 1, 3, 9, 30]):
        y = synth_tokens(43, k, 1, lo, fm.n_out)
        v, info, bp = capi.lane_emulate(*args, y, 1, back_pointers=True)
        assert info[0] == 1
        want_v, want_p = orc.viterbi(NONE, y)
        assert v == want_v, (name, lo, v, want_v)
        if math.isfinite(want_v):
            assert lane_walk(fm, y, bp, int(info[7])) == want_p.tolist(), (name, lo)
