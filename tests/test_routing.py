"""Which engine serves a call (-m gpu).  Every engine gives the same results, so a call routed to the wrong one only
shows as lost speed: with the verbose option mb_forward, mb_viterbi, mb_backward and mb_counts each name on stderr
the engine that ran, and these tests pin that routing."""
import re

import numpy as np
import pytest

from helpers import FlatMachine, load_golden, pairs_from_golden, synth_tokens

pytestmark = pytest.mark.gpu

ROUTE = re.compile(r"^(mb_forward|mb_viterbi|mb_viterbi \(scores\)|mb_backward|mb_counts): (\S+) engine$", re.M)
PASSES = ("forward", "viterbi", "scores", "backward", "counts")


def _machine(capi, fm, engine=-1, **options):
    capi.set_engine(engine)
    for k, v in dict(options, verbose=1).items():
        capi.set_option(k, v)
    try:
        return capi.Machine(fm.n_states, fm.n_in, fm.n_out, fm.src, fm.dst, fm.tin, fm.tout, fm.lw)
    finally:
        capi.set_engine(-1)
        for k in dict(options, verbose=1):
            capi.set_option(k, None)


def _full_envelopes(pairs):
    return [[(0, len(x) + 1)] * (len(y) + 1) for x, y in pairs]


def _golden_pairs(name):
    return pairs_from_golden(load_golden(name))


def _reads(name, lens):
    return [(x, y[:lo]) for (x, y), lo in zip(_golden_pairs(name), lens)]


# machine, batch, engine, options, the engine named for Forward, Viterbi with paths, Viterbi scores, Backward, counts (None: not run)
CASES = [
    ("dnapsw_small", "auto", -1, {}, ("jit", "jit", "jit", "jit", "jit")),
    ("dnapsw_small", "envelopes", -1, {}, ("wide", "wide", "wide", "generic", "generic")),
    ("dnapsw_small", "auto", 0, {}, ("generic",) * 5),
    ("prot2dna_dnapsw", "auto", -1, {}, ("big", "big", "big", "generic", "generic")),
    ("prot2dna_dnapsw", "auto", -1, {"no_big": 1}, ("wide", "wide", "wide", "generic", "generic")),
    ("prot2dna_dnapsw", "envelopes", -1, {}, ("wide", "wide", "wide", "generic", "generic")),
    ("hmmer_pf00516_reads", "auto", -1, {}, ("column", "column", "column", "generic", "generic")),
    ("hmmer_pf00516_reads", "auto", -1, {"no_col": 1}, ("lane", "lane", "lane", "generic", "generic")),
    ("hmmer_pf00516_reads", "auto", -1, {"col_no_traceback": 1}, ("column", "lane", "column", None, None)),
    ("unitindel", "empty inputs", 2, {}, ("lane", "lane", "lane", "generic", "generic")),
]


def _case_id(c):
    name, batch, engine, options, _ = c
    forced = {-1: [], 0: ["set_engine(0)"], 2: ["set_engine(2)"]}[engine]
    return "-".join([name, batch.replace(" ", "_")] + forced + ["%s=%s" % kv for kv in options.items()])


@pytest.mark.parametrize("name,batch,engine,options,want", CASES, ids=[_case_id(c) for c in CASES])
def test_routing_table(capfd, name, batch, engine, options, want):
    from machineboss_b200 import capi
    fm = FlatMachine.from_json(load_golden(name)["machine"])
    if name == "hmmer_pf00516_reads":
        pairs = _reads(name, (10, 7, 12))      # short reads keep the generic Backward and counts cheap
    elif batch == "empty inputs":
        pairs = [(np.zeros(0, np.uint8), synth_tokens(5, k, 1, lo, fm.n_out)) for k, lo in enumerate((6, 0, 9))]
    else:
        pairs = _golden_pairs(name)[:4]
    m = _machine(capi, fm, engine, **options)
    b = capi.Batch(pairs)
    if batch == "envelopes":
        b.set_envelopes(_full_envelopes(pairs))
    calls = {"forward": lambda: capi.forward(m, b), "viterbi": lambda: capi.viterbi(m, b), "scores": lambda: capi.viterbi(m, b, paths=False),
             "backward": lambda: capi.backward(m, b), "counts": lambda: capi.counts(m, b)}
    capfd.readouterr()
    for p, engine_name in zip(PASSES, want):
        if engine_name is None:
            continue
        calls[p]()
        routes = ROUTE.findall(capfd.readouterr().err)
        assert len(routes) == 1 and routes[0][1] == engine_name, (p, routes)


def test_failed_lane_preparation_is_not_left_half_built():
    """A generator whose output list into one state holds 16383 entries, more than the lane engine's back-pointers can
    index: its machine is WIDE (no input alphabet), and preparing the lane engine fails.  The failure leaves no
    half-built lane engine behind, so a second call fails in the same way instead of sweeping with empty tables."""
    from machineboss_b200 import capi
    n = 16383
    src = np.concatenate([np.arange(1, n + 1), [n + 1]]).astype(np.int32)
    dst = np.concatenate([np.full(n, n + 1), [n + 2]]).astype(np.int32)
    tin = np.zeros(n + 1, np.int32)
    tout = np.concatenate([np.ones(n), [0]]).astype(np.int32)
    lw = np.full(n + 1, -1.0)
    m = capi.Machine(n + 3, 0, 1, src, dst, tin, tout, lw)
    assert m.engine == capi.ENGINE_WIDE
    b = capi.Batch([(np.zeros(0, np.uint8), np.ones(3, np.uint8))])
    with pytest.raises(capi.MachineBossError, match="lane engine: a transition list has more than 16382 entries") as first:
        capi.forward(m, b)
    with pytest.raises(capi.MachineBossError) as second:
        capi.forward(m, b)
    assert str(second.value) == str(first.value)
