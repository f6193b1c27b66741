"""Posterior decoding restated in numpy over given Forward / Backward matrices F[o, i, s], B[o, i, s] (definitions: mb_mea in
include/machineboss_b200.h): the posterior gamma of a step, the maximum expected accuracy (MEA) DP with its candidate order and
first-maximum rule, its traceback, and the gammas of a given path.  Test helper, not a test file."""
from __future__ import annotations

import math

import numpy as np

from sample_replay import Incoming

NEG_INF = -math.inf


def tokens_of(fm, t) -> int:
    """c(t): the number of tokens transition t consumes."""
    return (1 if fm.tin[t] else 0) + (1 if fm.tout[t] else 0)


def gamma(f, ll, b, w):
    """(gamma, admissible) of a step from f = F(source cell)[src] to b = B(destination cell)[dst] with log-weight w."""
    if not ll > NEG_INF:
        return 0.0, False
    e = (f - ll) + (b + w)
    return (math.exp(e), True) if e > NEG_INF else (0.0, False)


def candidates(inc: Incoming, x, y, i, o, s):
    """(transition id, source inPos, source outPos) into state s at cell (i, o), in the reference's order: match, delete,
    insert, silent; each by source state then transition index."""
    fm = inc.fm
    a = int(x[i - 1]) if i else 0
    c = int(y[o - 1]) if o else 0
    out = []
    if i and o:
        out += [(p, i - 1, o - 1) for p in inc.get(s, a, c)]
    if i:
        out += [(p, i - 1, o) for p in inc.get(s, a, 0)]
    if o:
        out += [(p, i, o - 1) for p in inc.get(s, 0, c)]
    out += [(p, i, o) for p in inc.get(s, 0, 0)]
    return out


def _scored(inc, A, F, B, ll, x, y, i, o, s):
    """[(value, gamma, id, si, so)] of the admissible candidates into (i, o, s)."""
    fm = inc.fm
    out = []
    bs = float(B[o, i, s])
    if not (ll > NEG_INF and bs > NEG_INF):
        return out
    for p, si, so in candidates(inc, x, y, i, o, s):
        src = int(fm.src[p])
        g, ok = gamma(float(F[so, si, src]), ll, bs, float(fm.lw[p]))
        if ok:
            out.append((float(A[so, si, src]) + tokens_of(fm, p) * g, g, p, si, so))
    return out


def inside(env, i, o):
    return env is None or env[o][0] <= i < env[o][1]


def mea_fill(inc: Incoming, F, B, x, y, env=None):
    """The MEA matrix A[o, i, s]; ll = B[0, 0, 0] (the Backward log-likelihood)."""
    S = inc.fm.n_states
    li, lo = len(x), len(y)
    ll = float(B[0, 0, 0])
    A = np.full((lo + 1, li + 1, S), NEG_INF)
    for o in range(lo + 1):      # sources precede: lower cells, and lower states of the same cell (silent transitions ascend)
        for i in range(li + 1):
            if not inside(env, i, o):
                continue
            for s in range(S):
                acc = 0.0 if (i, o, s) == (0, 0, 0) else NEG_INF
                for v, _, _, _, _ in _scored(inc, A, F, B, ll, x, y, i, o, s):
                    if acc < v:
                        acc = v
                A[o, i, s] = acc
    return A


def mea_path(inc: Incoming, F, B, x, y, env=None, tie=1e-12):
    """(gain, ids, gammas, near_tie): the MEA path start -> end, the gamma of each step, and per step whether another admissible
    candidate came within `tie` of the chosen one (where a device path may legitimately part from this one)."""
    fm = inc.fm
    S = fm.n_states
    li, lo = len(x), len(y)
    ll = float(B[0, 0, 0])
    A = mea_fill(inc, F, B, x, y, env)
    gain = float(A[lo, li, S - 1]) if inside(env, li, lo) else NEG_INF
    ids, gs, ties = [], [], []
    if gain > NEG_INF:
        i, o, s = li, lo, S - 1
        while i > 0 or o > 0 or s != 0:
            cand = _scored(inc, A, F, B, ll, x, y, i, o, s)
            best = None
            for c in cand:
                if best is None or best[0] < c[0]:
                    best = c
            assert best is not None
            v, g, p, si, so = best
            ties.append(sum(1 for c in cand if abs(c[0] - v) <= tie) > 1)
            ids.append(p)
            gs.append(g)
            i, o, s = si, so, int(fm.src[p])
    return gain, ids[::-1], gs[::-1], ties[::-1]


def path_gammas(fm, F, B, x, y, path):
    """The gamma of each step of a valid path of the pair (a non-advancing silent step, left out of the DP, gets 0)."""
    ll = float(B[0, 0, 0])
    i, o, s, out = 0, 0, 0, []
    for t in path:
        a, c, d = int(fm.tin[t]), int(fm.tout[t]), int(fm.dst[t])
        assert int(fm.src[t]) == s
        ni, no = i + (1 if a else 0), o + (1 if c else 0)
        g = 0.0
        if a or c or d > s:
            g, _ = gamma(float(F[o, i, s]), ll, float(B[no, ni, d]), float(fm.lw[t]))
        out.append(g)
        i, o, s = ni, no, d
    return out


def gain_of(fm, path, gammas) -> float:
    g = 0.0
    for t, v in zip(path, gammas):
        g += tokens_of(fm, t) * v
    return g
