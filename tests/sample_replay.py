"""Host replay of mb_sample_paths: Philox4x32-10 and the sampler's walk over a stored Forward matrix, written out step by step
so that a device path can be checked id for id.

Philox4x32-10 is Random123's philox4x32 with 10 rounds (Salmon, Moraes, Dror and Shaw, SC'11).  The walk follows
sample_kernel (csrc/mb_generic.cu): candidates in traceback order (match, delete, insert, silent; each by source state then
transition index), weights exp(v - max v), the first candidate with a positive weight whose running sum exceeds u * norm.
"""
from __future__ import annotations

import math

import numpy as np

M32 = 0xFFFFFFFF
_MUL = (0xD2511F53, 0xCD9E8D57)
_WEYL = (0x9E3779B9, 0xBB67AE85)


def philox4x32_10(ctr, key):
    """The four output words for counter ctr (4 words) and key (2 words)."""
    c0, c1, c2, c3 = (int(v) & M32 for v in ctr)
    k0, k1 = (int(v) & M32 for v in key)
    for r in range(10):
        if r:
            k0, k1 = (k0 + _WEYL[0]) & M32, (k1 + _WEYL[1]) & M32
        p0, p1 = _MUL[0] * c0, _MUL[1] * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & M32, (p0 >> 32) ^ c3 ^ k1, p0 & M32
    return c0, c1, c2, c3


def uniform(seed: int, k: int, j: int, t: int) -> float:
    """The sampler's u in [0, 1) for step t of sample j of pair k."""
    r = philox4x32_10((t, j, k & M32, k >> 32), (seed & M32, (seed >> 32) & M32))
    return float(((r[0] << 21) | (r[1] >> 11))) * 2.0 ** -53


class Incoming:
    """The token-indexed incoming lists of a flat machine (DevCsr): transitions into a state with given tokens, by source
    state then id.  A silent transition that does not advance (only possible on state 0) is left out, as on the device."""

    def __init__(self, fm):
        self.fm = fm
        self.lists = {}
        for t in range(fm.n_trans):
            if fm.tin[t] == 0 and fm.tout[t] == 0 and fm.dst[t] <= fm.src[t]:
                continue
            self.lists.setdefault((int(fm.dst[t]), int(fm.tin[t]), int(fm.tout[t])), []).append(t)
        for v in self.lists.values():
            v.sort(key=lambda t: (int(fm.src[t]), t))

    def get(self, s, a, c):
        return self.lists.get((s, a, c), [])


def replay(inc: Incoming, F: np.ndarray, x, y, seed: int, k: int, j: int) -> list:
    """Path j of pair k (global transition ids, start -> end) drawn over the Forward matrix F[o, i, s]."""
    fm = inc.fm
    li, lo = len(x), len(y)
    s = fm.n_states - 1
    if not F[lo, li, s] > -math.inf:
        return []
    i, o, t, rev = li, lo, 0, []
    while i > 0 or o > 0 or s != 0:
        a = int(x[i - 1]) if i else 0
        c = int(y[o - 1]) if o else 0
        cand = []      # (id, value, di, do)
        if i and o:
            cand += [(p, float(F[o - 1, i - 1, fm.src[p]]) + float(fm.lw[p]), 1, 1) for p in inc.get(s, a, c)]
        if i:
            cand += [(p, float(F[o, i - 1, fm.src[p]]) + float(fm.lw[p]), 1, 0) for p in inc.get(s, a, 0)]
        if o:
            cand += [(p, float(F[o - 1, i, fm.src[p]]) + float(fm.lw[p]), 0, 1) for p in inc.get(s, 0, c)]
        cand += [(p, float(F[o, i, fm.src[p]]) + float(fm.lw[p]), 0, 0) for p in inc.get(s, 0, 0)]
        mx = max(v for _, v, _, _ in cand)
        assert mx > -math.inf
        w = [math.exp(v - mx) for _, v, _, _ in cand]
        norm = 0.0
        for wn in w:
            norm += wn
        thr = uniform(seed, k, j, t) * norm
        run, pick, last = 0.0, None, None
        for n, wn in enumerate(w):
            if not wn > 0:
                continue
            run += wn
            last = n
            if run > thr:
                pick = n
                break
        p, _, di, do = cand[pick if pick is not None else last]
        rev.append(p)
        i, o, s, t = i - di, o - do, int(fm.src[p]), t + 1
    return rev[::-1]
