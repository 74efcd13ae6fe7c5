"""GPU suite (-m gpu): the device state a step starts from.  One launch at the start of classify restores the pile table
and clears the counters, the earliest events, the look-back pool and the build / transitive counters; the first
containment pass clears what the final pass counts into.  Every entry point must see the same state as a fresh session:
repeated runs (eager, captured, replayed), the stage calls one by one, stages called again, and all of these after a
larger batch left its counters, pool words and earliest events behind in the same session."""
import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth
from tests.replay import assert_same

pytestmark = pytest.mark.gpu

KEYS = ("n_overlaps", "n_internals", "n_candidates", "n_rounds", "n_final_candidates", "n_alive_piles", "n_nodes", "n_edges",
        "n_two_hop", "n_transitive_pairs")


def _inputs(seed, genome_len):
    ds = synth.generate(genome_len, 40, 9000, len_sd=2500, seed=seed, noise=60, dual=True, chimera_frac=0.03)
    piles = ds.flat_piles()
    rng = np.random.Generator(np.random.PCG64(seed))
    flags = (rng.random(ds.n_reads) < 0.04).astype(np.uint8) * 2
    return ds.records, piles, flags


def _check(G, P, what):
    assert_same(G.edges(), P.edges, f"edges, {what}")
    assert_same(G.marked(), P.marked, f"marks, {what}")
    assert_same(G.piles(), P.piles, f"piles, {what}")
    c = G.counts()
    assert c["n_nodes"] == P.n_nodes and c["n_transitive_pairs"] == P.n_pairs, (what, c)
    return {k: c[k] for k in KEYS}


def test_run_and_stage_calls_start_from_the_same_state_after_a_dirty_batch(ctx):
    big = _inputs(91, 1_600_000)
    small = _inputs(92, 900_000)
    P_big = O.Pipeline(*big).run()
    P = O.Pipeline(*small).run()
    G = api.Graph(ctx)

    def load(inp):
        rec, piles, flags = inp
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec)

    load(big)
    G.run()
    _check(G, P_big, "larger batch")
    load(small)
    want = None
    for i in range(4):   # eager (new shape), captured, replayed twice: the larger batch's words are still in the buffers
        G.run()
        got = _check(G, P, f"run {i}")
        want = want or got
        assert got == want, (i, got, want)
        ovl, inl = G.lists()
        assert_same(ovl, P.ovl, f"final overlaps, run {i}")
        assert_same(inl, P.int, f"final internals, run {i}")

    # the stage calls one by one on the state the runs left behind
    fresh = api.Graph(ctx)
    rec, piles, flags = small
    fresh.set_piles(piles, flags).set_hills(None).set_overlaps(rec)
    fresh.classify()
    want_classified = fresh.counts()
    fresh.close()
    load(small)
    G.classify()
    c = G.counts()
    assert c == want_classified, (c, want_classified)
    assert (c["n_candidates"], c["n_rounds"]) == (want["n_candidates"], want["n_rounds"]), c
    G.retrim()
    G.retrim_promote()
    G.finalize()
    G.build()
    G.transitive()
    assert _check(G, P, "stage calls") == want
    G.transitive()   # again, on the same CSR: its counters are cleared by the call itself
    assert _check(G, P, "transitive twice") == want

    # the larger batch through the stage calls, then the smaller one through a replayed run again
    load(big)
    G.classify()
    G.finalize()
    G.build()
    G.transitive()
    _check(G, P_big, "larger batch, stage calls")
    load(small)
    for i in range(2):
        G.run()
        assert _check(G, P, f"run after the stage calls {i}") == want
    G.close()


def test_retrim_rounds_beyond_one_step_of_look_back_words(ctx):
    """Every retrim pass takes look-back words; rounds beyond what a step holds clear the pool again and stay exact:
    six rounds leave what one round leaves."""
    rec, piles, flags = _inputs(93, 800_000)

    def session(rounds):
        G = api.Graph(ctx)
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec)
        G.classify()
        counts = []
        for _ in range(rounds):
            G.set_piles(piles, flags)   # a changed table: neither pass is skipped
            G.retrim()
            G.retrim_promote()
            c = G.counts()
            counts.append((c["n_overlaps"], c["n_internals"]))
        lists = [x.copy() for x in G.lists()]
        G.finalize()
        G.build()
        G.transitive()
        out = (G.edges().copy(), G.marked().copy(), {k: G.counts()[k] for k in KEYS})
        G.close()
        return counts, lists, out

    c1, l1, o1 = session(1)
    c6, l6, o6 = session(6)
    assert c6 == c1 * 6, (c1, c6)
    assert_same(l6[0], l1[0], "overlaps after the retrim rounds")
    assert_same(l6[1], l1[1], "internals after the retrim rounds")
    assert_same(o6[0], o1[0], "edges")
    assert_same(o6[1], o1[1], "marks")
    assert o6[2] == o1[2]
