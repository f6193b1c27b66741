"""Posterior counts of each pair of a batch on its own (mb_pair_counts, -m gpu).

Row k must be what mb_counts gives for a batch holding only pair k: the C oracle's counts for that pair, the same row whatever
the batch around it and however it is chunked, and summing to mb_counts over the batch.  Impossible pairs get a zero row."""
import json
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from helpers import GOLDEN, LSE_EXACT, FlatMachine, Oracle, load_golden, mutate_tokens, pairs_from_golden, synth_tokens

pytestmark = pytest.mark.gpu

REL = 1e-4
SAME = 1e-12      # the same pair's row computed twice: atomics add in another order, nothing else differs


def _capi():
    from machineboss_b200 import capi
    return capi


def make(capi, fm, engine=-1, **options):
    capi.set_engine(engine)
    for k, v in options.items():
        capi.set_option(k, v)
    try:
        return capi.Machine(fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    finally:
        capi.set_engine(-1)
        for k in options:
            capi.set_option(k, None)


def golden_machine(name):
    return FlatMachine.from_json(load_golden(name)["machine"])


def counts_agree(fm, pairs, got, want):
    """test_gpu_parity's rule: within 1e-4 relative of the reference's table-based counts, or, where the table's own error
    is larger, within 1e-5 of the exact sums while the table's values sit within 5e-4 of those."""
    got, want = np.asarray(got), np.asarray(want)
    if np.allclose(got, want, rtol=REL, atol=1e-7):
        return True
    orc = Oracle(fm)
    exact = np.zeros(fm.n_trans)
    for x, y in pairs:
        orc.counts(x, y, mode=LSE_EXACT, counts=exact)
    return np.allclose(got, exact, rtol=1e-5, atol=1e-7) and np.allclose(want, exact, rtol=5e-4, atol=1e-7)


def counts_agree_with_envelopes(fm, pairs, envs, got):
    """counts_agree, each pair's oracle counts under its envelope."""
    orc = Oracle(fm)
    table, ex = np.zeros(fm.n_trans), np.zeros(fm.n_trans)
    try:
        for k, (x, y) in enumerate(pairs):
            orc.set_envelope(envs[k])
            if math.isinf(orc.forward(x, y, mode=LSE_EXACT)):
                continue
            orc.counts(x, y, counts=table)
            orc.counts(x, y, mode=LSE_EXACT, counts=ex)
    finally:
        orc.set_envelope(None)
    if np.allclose(got, table, rtol=1e-4, atol=1e-7):
        return True
    return np.allclose(got, ex, rtol=1e-5, atol=1e-7) and np.allclose(table, ex, rtol=5e-4, atol=1e-7)


def same_rows(a, b, rel=SAME):
    """Equal to `rel` relative per transition, with an absolute floor of rel times the row's largest count."""
    a, b = np.asarray(a), np.asarray(b)
    floor = rel * max(1.0, float(np.abs(b).max(initial=0.0)))
    return np.allclose(a, b, rtol=rel, atol=floor)


def check_rows_against_oracle(fm, pairs, rows, ll):
    orc = Oracle(fm)
    assert rows.shape == (len(pairs), fm.n_trans)
    for k, (x, y) in enumerate(pairs):
        f, _, want = orc.counts(x, y)
        if math.isinf(f):
            assert ll[k] == -math.inf and not rows[k].any(), k
            continue
        fe = orc.forward(x, y, mode=LSE_EXACT)
        assert abs(ll[k] - f) <= REL * max(1.0, abs(f)) or abs(ll[k] - fe) <= 1e-6 * max(1.0, abs(fe)), (k, ll[k], f, fe)
        assert counts_agree(fm, [(x, y)], rows[k], want), (k, np.abs(rows[k] - want).max())


def synth_pairs(n, lengths, seed=11, n_sym=4):
    out = []
    for k in range(n):
        x = synth_tokens(seed, k, 0, int(lengths[k % len(lengths)]), n_sym)
        out.append((x, mutate_tokens(seed, k, x, n_sym)))
    return out


# ---------------------------------------------------------------------------------------------
# 1. row by row against the oracle, on the default engine and on the generic engine
# ---------------------------------------------------------------------------------------------
ORACLE_CASES = ["dnapsw_small", "dnapsw_1k", "dnapsw_peaked_1k", "protpsw_300_batch", "prot2dna_dnapsw", "hmmer_pf00516_reads"]


@pytest.mark.parametrize("engine", ["default", "generic"])
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_rows_match_the_oracle(name, engine):
    capi = _capi()
    fm = golden_machine(name)
    pairs = pairs_from_golden(load_golden(name))
    m = make(capi, fm, -1 if engine == "default" else capi.ENGINE_GENERIC)
    rows, ll = capi.pair_counts(m, capi.Batch(pairs), loglike=True)
    check_rows_against_oracle(fm, pairs, rows, ll)


# ---------------------------------------------------------------------------------------------
# 2. the rows add up to mb_counts; the log-likelihoods are mb_counts' bit for bit
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["dnapsw", "protpsw_300_batch", "hmmer_pf00516_reads"])
def test_rows_sum_to_the_batch_counts(name):
    capi = _capi()
    if name == "dnapsw":
        fm = golden_machine("dnapsw_small")
        pairs = synth_pairs(48, (40, 300, 700, 120))
    else:
        fm = golden_machine(name)
        pairs = pairs_from_golden(load_golden(name))
    m = make(capi, fm)
    b = capi.Batch(pairs)
    rows, ll = capi.pair_counts(m, b, loglike=True)
    if m.engine == capi.ENGINE_JIT:
        assert b.last_redo() == 0
    c, cll = capi.counts(m, b)
    assert np.array_equal(ll, cll)
    assert same_rows(rows.sum(axis=0), c)


# ---------------------------------------------------------------------------------------------
# 3. a pair's row does not depend on the batch around it or on the chunking
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ["default", "generic"])
def test_rows_do_not_depend_on_batch_or_chunking(engine):
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    eng = -1 if engine == "default" else capi.ENGINE_GENERIC
    pairs = synth_pairs(64, (150, 60, 140, 90))
    m = make(capi, fm, eng)
    rows = capi.pair_counts(m, capi.Batch(pairs))
    rev = capi.pair_counts(m, capi.Batch(pairs[::-1]))[::-1]
    for k in (0, 5, 33, 63):
        alone = capi.pair_counts(m, capi.Batch([pairs[k]]))[0]
        single, _ = capi.counts(m, capi.Batch([pairs[k]]))
        assert same_rows(rows[k], alone) and same_rows(rev[k], alone) and same_rows(alone, single), k
    if engine == "generic":
        return
    # pairs of one input length: the smallest Forward budget (whole MB) that holds one of them holds no two, so every pair
    # sits in a chunk of its own
    pairs = synth_pairs(32, (150,), seed=12)
    rows = capi.pair_counts(m, capi.Batch(pairs))
    for mb in range(1, 9):
        mc = make(capi, fm, eng, jit_f_budget_mb=mb)
        b = capi.Batch(pairs)
        try:
            tiny = capi.pair_counts(mc, b)
        except capi.MachineBossError as e:
            assert "does not fit" in str(e)
            continue
        break
    else:
        pytest.fail("no budget of up to 8 MB holds one pair")
    assert b.last_redo() == 0 and b.last_kernel_ms()[1] == 2 * len(pairs)      # a Forward and a count launch per chunk
    for k in range(len(pairs)):
        assert same_rows(tiny[k], rows[k]), k


# ---------------------------------------------------------------------------------------------
# 4. a few long pairs: fewer pairs than resident warps
# ---------------------------------------------------------------------------------------------
def test_few_long_pairs():
    capi = _capi()
    fm = golden_machine("dnapsw_3k")
    x, y = pairs_from_golden(load_golden("dnapsw_3k"))[0]
    pairs = [(x[: 3000 - 150 * k], y[: 2900 - 120 * k]) for k in range(4)]
    m = make(capi, fm)
    assert m.engine == capi.ENGINE_JIT
    rows, ll = capi.pair_counts(m, capi.Batch(pairs), loglike=True)
    for k, p in enumerate(pairs):
        single, sll = capi.counts(m, capi.Batch([p]))
        assert math.isfinite(ll[k]) and same_rows(rows[k], single), k
    check_rows_against_oracle(fm, pairs[:1], rows[:1], ll[:1])


# ---------------------------------------------------------------------------------------------
# 5. pairs the scaled linear sweep flags are re-run in the log domain; their batch-mates keep their rows
# ---------------------------------------------------------------------------------------------
def _trap_machine():
    """test_gpu_parity's machine: a 'fast but doomed' branch next to a slow real one.  After n a's the live path is 8^-n
    below the trap in the same cell, which the scaled linear sweep must hand over."""
    w8 = math.log(0.125)
    trans = [(0, 1, 0, 0, 0.0), (0, 2, 0, 0, 0.0), (1, 1, 0, 1, 0.0), (2, 2, 0, 1, w8), (2, 2, 0, 2, w8), (2, 3, 0, 0, 0.0)]
    a = np.array(trans)
    return FlatMachine(4, 0, 2, a[:, 0].astype(np.int32), a[:, 1].astype(np.int32), a[:, 2].astype(np.int32),
                       a[:, 3].astype(np.int32), a[:, 4].astype(np.float64), [], ["a", "b"])


def test_flagged_pairs_are_rerun_alone():
    capi = _capi()
    fm = _trap_machine()
    read = lambda n, tail: np.array([1] * n + tail, dtype=np.uint8)
    short = [read(n, [2, 1, 2][: 1 + n % 3]) for n in (1, 3, 5, 10, 20, 7, 2)]
    long_ = [read(n, [2]) for n in (250, 400, 900)]
    ys = [read(10, [2])] + long_[:1] + short[:3] + long_[1:] + short[3:]
    pairs = [(np.zeros(0, np.uint8), y) for y in ys]
    m = make(capi, fm, capi.ENGINE_JIT)
    b = capi.Batch(pairs)
    rows, ll = capi.pair_counts(m, b, loglike=True)
    assert b.last_redo() == len(long_)
    check_rows_against_oracle(fm, pairs, rows, ll)
    is_long = [len(y) > 200 for y in ys]
    kept = [p for p, lg in zip(pairs, is_long) if not lg]
    ref = capi.pair_counts(m, capi.Batch(kept))
    for r, k in zip(ref, [k for k, lg in enumerate(is_long) if not lg]):
        assert same_rows(rows[k], r), k


# ---------------------------------------------------------------------------------------------
# 6. impossible and empty pairs
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ["default", "generic"])
def test_impossible_and_empty_pairs(engine):
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    fm = fm.with_weights(np.where(fm.tout == 1, -np.inf, fm.lw))      # no path emits output token 1
    x = np.array([2, 3, 4, 2], np.uint8)
    pairs = [(x, np.array([2, 4, 3], np.uint8)), (x, np.array([2, 1, 3], np.uint8)), (np.zeros(0, np.uint8), np.zeros(0, np.uint8)),
             (np.array([3, 3], np.uint8), np.array([4], np.uint8))]
    m = make(capi, fm, -1 if engine == "default" else capi.ENGINE_GENERIC)
    rows, ll = capi.pair_counts(m, capi.Batch(pairs), loglike=True)
    assert ll[1] == -math.inf and not rows[1].any()
    assert all(math.isfinite(ll[k]) for k in (0, 2, 3))
    check_rows_against_oracle(fm, pairs, rows, ll)
    empty, ell = capi.pair_counts(m, capi.Batch([]), loglike=True)
    assert empty.shape == (0, fm.n_trans) and ell.shape == (0,)


# ---------------------------------------------------------------------------------------------
# 7. envelopes (generic engine)
# ---------------------------------------------------------------------------------------------
def banded(li, lo, w):
    """Rows |i - o Li / Lo| <= w, widened where the band is steeper than one column per row so that it stays connected."""
    if lo == 0:
        return [(0, li + 1)]
    c = [(o * li) // lo for o in range(lo + 1)] + [li]
    return [(max(0, c[o] - w), min(li, max(c[o] + w, c[o + 1] - w - 1)) + 1) for o in range(lo + 1)]


def ragged(li, lo, seed):
    """A connected envelope whose rows start and end at random places around the diagonal."""
    rng = np.random.default_rng(seed)
    rows, prev_end = [], 1
    for o in range(lo + 1):
        c = (o * li) // max(lo, 1)
        s = max(0, min(c - int(rng.integers(0, 4)), prev_end - 1))
        e = min(li + 1, max(c + 1 + int(rng.integers(0, 4)), s + 1))
        if o == lo:
            e = li + 1
        rows.append((s, e))
        prev_end = e
    return rows


def test_envelopes_row_by_row(capfd):
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = synth_pairs(6, (30, 45, 20))
    shapes = [lambda li, lo: banded(li, lo, 1), lambda li, lo: None, lambda li, lo: banded(li, lo, 3), lambda li, lo: ragged(li, lo, 5),
              lambda li, lo: banded(li, lo, 0), lambda li, lo: ragged(li, lo, 9)]
    envs = [shape(len(x), len(y)) for shape, (x, y) in zip(shapes, pairs)]
    m = make(capi, fm, verbose=1)
    b = capi.Batch(pairs)
    b.set_envelopes(envs)
    capfd.readouterr()
    rows, ll = capi.pair_counts(m, b, loglike=True)
    assert "mb_pair_counts: generic engine" in capfd.readouterr().err
    for k, (x, y) in enumerate(pairs):
        assert counts_agree_with_envelopes(fm, [(x, y)], [envs[k]], rows[k]), k
        if not math.isfinite(ll[k]):
            assert not rows[k].any()


# ---------------------------------------------------------------------------------------------
# 8. errors and the route line
# ---------------------------------------------------------------------------------------------
def test_errors_and_route(capfd):
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = pairs_from_golden(load_golden("dnapsw_small"))
    for eng, line in ((-1, "mb_pair_counts: jit engine"), (capi.ENGINE_GENERIC, "mb_pair_counts: generic engine")):
        m = make(capi, fm, eng, verbose=1)
        b = capi.Batch(pairs)
        capfd.readouterr()
        capi.pair_counts(m, b)
        assert line in capfd.readouterr().err
        assert capi.lib().mb_pair_counts(m.h, b.h, None, None) != 0
        assert "mb_pair_counts" in capi.lib().mb_last_error().decode()


# ---------------------------------------------------------------------------------------------
# 9. groups
# ---------------------------------------------------------------------------------------------
def _group_rows(capi, fm, pairs, devices):
    g = capi.Group(devices)
    gm = capi.GroupMachine(g, fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    gb = capi.GroupBatch(g, pairs)
    out = capi.group_pair_counts(gm, gb, loglike=True)
    gb.close(), gm.close(), g.close()
    return out


def test_group_of_one_device():
    capi = _capi()
    fm = golden_machine("dnapsw_small")
    pairs = synth_pairs(24, (80, 200, 30))
    rows, ll = capi.pair_counts(make(capi, fm), capi.Batch(pairs), loglike=True)
    grows, gll = _group_rows(capi, fm, pairs, [0])
    assert np.array_equal(ll, gll)
    for k in range(len(pairs)):
        assert same_rows(grows[k], rows[k]), k


def test_group_of_every_device():
    capi = _capi()
    if capi.device_count() < 2:
        pytest.skip("needs at least 2 GPUs (%d visible)" % capi.device_count())
    fm = golden_machine("dnapsw_small")
    pairs = synth_pairs(40, (80, 200, 30, 500))
    rows, ll = capi.pair_counts(make(capi, fm), capi.Batch(pairs), loglike=True)
    grows, gll = _group_rows(capi, fm, pairs, None)
    assert np.array_equal(ll, gll)
    for k in range(len(pairs)):
        assert same_rows(grows[k], rows[k]), k


# ---------------------------------------------------------------------------------------------
# 10. the CLI
# ---------------------------------------------------------------------------------------------
def _write(obj):
    f = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
    f.write(obj if isinstance(obj, str) else json.dumps(obj))
    f.close()
    return f.name


def test_cli_per_pair_counts():
    from machineboss_b200 import build
    cli = build.build_host()
    case = load_golden("dnapsw_small")
    m = case["machine"]
    ia, oa = [""] + m["inAlphabet"], [""] + m["outAlphabet"]
    spl = [{"input": {"name": "x%d" % k, "sequence": [ia[t] for t in p["x"]]},
            "output": {"name": "y%d" % k, "sequence": [oa[t] for t in p["y"]]}} for k, p in enumerate(case["pairs"])]
    mf = _write(m)
    got = json.loads(subprocess.run([cli, "--evaluated-machine", mf, "-D", _write(spl), "-C", "--per-pair"], capture_output=True, text=True, check=True).stdout)
    assert len(got) == len(spl)
    for k, sp in enumerate(spl):
        alone = json.loads(subprocess.run([cli, "--evaluated-machine", mf, "-D", _write([sp]), "-C"], capture_output=True, text=True, check=True).stdout)
        assert np.allclose(np.array([v for r in got[k] for v in r]), np.array([v for r in alone for v in r]), rtol=2e-5, atol=1e-9), k
    # a symbolic machine gives parameter counts
    with open(os.path.join(GOLDEN, "aux_fit_inputs.json")) as f:
        fi = json.load(f)
    mf, pf = _write(fi["bitnoise_machine"]), _write(fi["params"])
    data = json.loads(fi["seqpairlist"])
    got = json.loads(subprocess.run([cli, "--machine", mf, "-P", pf, "-D", _write(data), "-C", "--per-pair"], capture_output=True, text=True, check=True).stdout)
    assert len(got) == len(data)
    for k, sp in enumerate(data):
        alone = json.loads(subprocess.run([cli, "--machine", mf, "-P", pf, "-D", _write([sp]), "-C"], capture_output=True, text=True, check=True).stdout)
        assert isinstance(alone, dict) and alone and set(got[k]) == set(alone)
        for name, v in alone.items():
            assert math.isclose(got[k][name], v, rel_tol=2e-5, abs_tol=1e-9), (k, name)
