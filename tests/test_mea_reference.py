"""The posterior-decoding definitions (tests/mea_reference.py) against brute force, without a device: on small pairs every
complete path is enumerated.  A step's gamma must be the total posterior probability of the paths that take that transition from
that cell, and the MEA gain must be the largest gain of any complete path."""
import math

import numpy as np
import pytest

from helpers import LSE_EXACT, FlatMachine, Oracle, load_golden, pairs_from_golden
from mea_reference import gain_of, mea_path, path_gammas, tokens_of
from sample_replay import Incoming


def complete_paths(fm, x, y):
    """Every path from (0, 0, state 0) to (len x, len y, end state) of finite weight: (ids, weight, steps), a step being
    (inPos, outPos, transition) at the cell it leaves.  Non-advancing silent transitions (only possible on state 0) are left out, as
    in the DP."""
    li, lo, end = len(x), len(y), fm.n_states - 1
    out_of = {}
    for t in range(fm.n_trans):
        if fm.tin[t] == 0 and fm.tout[t] == 0 and fm.dst[t] <= fm.src[t]:
            continue
        if math.isfinite(fm.lw[t]):
            out_of.setdefault(int(fm.src[t]), []).append(t)
    found = []

    def walk(i, o, s, ids, w, steps):
        if (i, o, s) == (li, lo, end):
            found.append((list(ids), w, list(steps)))
        for t in out_of.get(s, []):
            a, c = int(fm.tin[t]), int(fm.tout[t])
            if a and (i >= li or x[i] != a):
                continue
            if c and (o >= lo or y[o] != c):
                continue
            ids.append(t)
            steps.append((i, o, t))
            walk(i + (1 if a else 0), o + (1 if c else 0), int(fm.dst[t]), ids, w + float(fm.lw[t]), steps)
            ids.pop()
            steps.pop()

    walk(0, 0, 0, [], 0.0, [])
    return found


def case_pairs():
    out = []
    for name in ("bitnoise_tiny", "unitindel", "stutter_noise_difflen"):
        case = load_golden(name)
        fm = FlatMachine.from_json(case["machine"])
        out += [(name, k, fm, x, y) for k, (x, y) in enumerate(pairs_from_golden(case))]
    case = load_golden("dnapsw_small")
    x, y = pairs_from_golden(case)[0]
    out.append(("dnapsw_small", 0, FlatMachine.from_json(case["machine"]), x[:3], y[:3]))
    return out


@pytest.mark.parametrize("name,k,fm,x,y", case_pairs(), ids=lambda v: v if isinstance(v, (str, int)) else "")
def test_gamma_and_mea_gain_against_enumeration(name, k, fm, x, y):
    paths = complete_paths(fm, x, y)
    orc = Oracle(fm)
    _, F = orc.forward(x, y, mode=LSE_EXACT, matrix=True)
    _, B = orc.backward(x, y, mode=LSE_EXACT, matrix=True)
    inc = Incoming(fm)
    gain, ids, gs, _ = mea_path(inc, F, B, x, y)
    if not paths:
        assert gain == -math.inf and ids == []
        return
    ws = np.array([w for _, w, _ in paths])
    ll = float(np.logaddexp.reduce(ws))
    exact = {}
    for (_, w, steps) in paths:
        for st in steps:
            exact[st] = exact.get(st, 0.0) + math.exp(w - ll)
    # gamma of every step of every path equals the summed posterior of the paths that take it
    best = -math.inf
    for (p, _, steps) in paths:
        g = path_gammas(fm, F, B, x, y, p)
        for st, v in zip(steps, g):
            assert abs(v - exact[st]) <= 1e-9, (name, k, st, v, exact[st])
        best = max(best, gain_of(fm, p, g))
    # the MEA path is a complete path, its gain the enumerated maximum, and the sum of c(t) * gamma over its own steps
    assert tuple(ids) in {tuple(p) for p, _, _ in paths}
    assert abs(gain - best) <= 1e-12, (name, k, gain, best)
    assert abs(gain_of(fm, ids, gs) - gain) <= 1e-12
    assert gs == path_gammas(fm, F, B, x, y, ids)
    assert 0 <= gain <= len(x) + len(y) + 1e-9
    assert sum(tokens_of(fm, t) for t in ids) == len(x) + len(y)
