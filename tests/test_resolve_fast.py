"""The earliest-event test of the containment resolution (k_resolve_fast in containment.cu) and the hard path behind it,
against the oracle.

A victim v whose earliest event is (t1, c1) dies at t1 when c1 == v, when c1 has no event, or when c1's own earliest
event is later than t1.  Every other victim is "hard": only its events are grouped and resolved by k_resolve, and an event
whose container is already settled to die before it is dropped on the way.  The record sets below are built so that
each branch is taken many times; a CPU test checks that they are, the GPU tests compare the whole pipeline with the
oracle through the first pass, the final pass (containers with a chimeric region) and the first pass with hill counters.
"""
import functools
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth

INF = np.iinfo(np.int64).max
MARGIN = 15          # flat piles: [15, L - 15)
DOVE = 800


# ---------------------------------------------------------------------------------------------------------------------
# record sets
# ---------------------------------------------------------------------------------------------------------------------
class Design:
    """Designed reads (ids after the background's) and their records in file order."""

    def __init__(self, rng, n_bg, bg_len):
        self.rng, self.n_bg, self.bg_len = rng, n_bg, bg_len
        self.len, self.rec = [], []

    def read(self, length=None):
        self.len.append(int(length if length is not None else self.rng.integers(2000, 4000)))
        return len(self.len) - 1

    def contain(self, v, c):
        """an event with victim v and container c (KB written as (v, c), KA as (c, v) when c is longer)"""
        lv, lc = self.len[v], self.len[c]
        assert lc >= lv
        ori = int(self.rng.integers(0, 2))
        off = MARGIN + int(self.rng.integers(0, lc - lv + 1))
        if v == c:
            ori = 0
        if v == c or lc == lv or self.rng.random() < 0.5:
            self.rec.append((v, c, MARGIN, lv - MARGIN, off, off + lv - 2 * MARGIN, ori))
        else:
            self.rec.append((c, v, off, off + lv - 2 * MARGIN, MARGIN, lv - MARGIN, ori))

    def dovetail(self, x):
        """x's suffix on the prefix of a background read (of another designed read without background): an edge iff
        both survive"""
        if self.n_bg:
            g = -1 - int(self.rng.integers(0, self.n_bg))
        else:
            g = int(self.rng.integers(0, len(self.len) - 1))
            g += g >= x
        self.rec.append((x, g, self.len[x] - DOVE, self.len[x] - MARGIN, MARGIN, DOVE, 0))


def _mixed(d):
    """Random containments among designed reads (a container is never shorter than its victim), self-containments and
    hand-made cases: a container without events, one whose first event is later, an easy container (the victim's first
    event is void), and hard containers that die before, after or never relative to their victim's event."""
    rng = d.rng
    xs = sorted((d.read() for _ in range(3000)), key=lambda x: d.len[x])
    for _ in range(6000):
        i, j = sorted(rng.integers(0, len(xs), 2))
        if rng.random() < 0.06:
            d.contain(xs[i], xs[i])
        else:
            d.contain(xs[i], xs[j])
    rng.shuffle(d.rec)
    for _ in range(200):
        v, c, x, y, z = (d.read(2000 + 300 * k) for k in range(5))
        d.contain(c, x)          # c dies at once: x has no events
        d.contain(v, c)          # v's first event: c is easy and dead -> void
        d.contain(v, y)          # fires
        u, w = d.read(2000), d.read(2100)
        d.contain(u, w)          # w has no events: u easy
        d.contain(w, z)          # w's first event is later than u's
        # hard containers: h's first event is void (its container died first), then h dies at its second or never
        for fate in ("before", "after", "never"):
            p, q, h, r, s, vv = d.read(3900), d.read(3800), d.read(3000), d.read(3950), d.read(3990), d.read(2500)
            d.contain(q, p)      # q dies
            d.contain(h, q)      # void: h is hard
            if fate == "before":
                d.contain(h, r)  # h dies here
                d.contain(vv, h)   # vv hard, its event void
                d.contain(vv, s)   # fires
            elif fate == "after":
                d.contain(vv, h)   # h alive: fires
                d.contain(h, r)
            else:
                d.contain(vv, h)   # h never dies: fires


def _all_easy(d):
    """One event per victim, containers without events: every victim settles from its earliest event (no background
    reads, whose containments would leave some victims hard)"""
    cs = [d.read(3900) for _ in range(300)]
    for _ in range(3000):
        d.contain(d.read(int(d.rng.integers(2000, 3800))), cs[int(d.rng.integers(0, len(cs)))])


def _all_hard(d):
    """Reverse-time chains: x_{k} in x_{k+1} at decreasing times, so every victim but the first of each chain has a
    container whose earliest event is earlier.  (The victim with the globally earliest event is always easy.)"""
    chains = [[d.read(2000 + k) for k in range(40)] for _ in range(100)]
    links = []
    for xs in chains:
        links.append([(xs[k], xs[k + 1]) for k in range(len(xs) - 2, -1, -1)])
    for step in range(39):
        for lk in links:
            d.contain(*lk[step])


def _deep(d):
    """A reverse-time chain 20 000 links deep (far past the chase stack of 24) and 600 chains of 60 links (more open
    victims than the single-block tail takes after the first sweep): the hard path must go round its worklist."""
    chains = [[d.read(2000 + k) for k in range(20_001)]] + [[d.read(2000 + k) for k in range(61)] for _ in range(600)]
    links = [[(xs[k], xs[k + 1]) for k in range(len(xs) - 2, -1, -1)] for xs in chains]
    for step in range(max(len(lk) for lk in links)):
        for lk in links:
            if step < len(lk):
                d.contain(*lk[step])


FAMILIES = {"mixed": _mixed, "all_easy": _all_easy, "all_hard": _all_hard, "deep": _deep}


@functools.lru_cache(maxsize=None)
def build(name, flagged=False, hills=False):
    """Background synth read set, the designed reads after it and the designed records at random places in the file.
    flagged: every designed container has a chimeric region (the final pass resolves their events).  hills: hill
    counters on a tenth of the designed reads."""
    rng = np.random.Generator(np.random.PCG64(7000 + list(FAMILIES).index(name)))
    bg = synth.generate(120_000, 6, 5000, seed=31) if name != "all_easy" else \
        SimpleNamespace(n_reads=0, read_len=np.zeros(0, np.int64), n_overlaps=0, records=np.zeros((0, 7), np.int64))
    n_bg = bg.n_reads
    d = Design(rng, n_bg, bg.read_len)
    FAMILIES[name](d)
    n_des = len(d.len)
    for x in rng.choice(n_des, size=n_des // 6, replace=False).tolist():
        d.dovetail(x)
    drec = np.array(d.rec, dtype=np.int64)
    dove = drec[:, 1] < 0
    drec[~dove, 1] += n_bg
    drec[dove, 1] = -1 - drec[dove, 1]
    drec[:, 0] += n_bg
    n_piles = n_bg + n_des
    records = np.empty((bg.n_overlaps + drec.shape[0], 7), dtype=np.int64)
    is_des = np.zeros(records.shape[0], bool)
    is_des[np.sort(rng.choice(records.shape[0], size=drec.shape[0], replace=False))] = True
    records[is_des] = drec
    records[~is_des] = bg.records
    lens = np.concatenate([bg.read_len, d.len]).astype(np.int64)
    piles = np.stack([np.full(n_piles, MARGIN), lens - MARGIN], 1).astype(np.uint32)
    flags = np.zeros(n_piles, dtype=np.uint8)
    rec = records.astype(np.uint32)
    if flagged:
        _, types = O.trim_type_batch(rec, piles)
        cont = np.where(types == O.KB, rec[:, 1], rec[:, 0])
        is_ev = np.isin(types, (O.KA, O.KB)) & is_des
        flags[np.unique(cont[is_ev])] = 2
    hill_rows = None
    if hills:
        hp = n_bg + np.sort(rng.choice(n_des, size=n_des // 10, replace=False))
        flags[hp] = 3
        mid = (piles[hp, 0].astype(np.int64) + piles[hp, 1]) // 2
        hill_rows = np.stack([hp, mid - 100, mid + 100], 1).astype(np.uint32)
    return SimpleNamespace(records=rec, piles=piles, flags=flags, hills=hill_rows, n_piles=n_piles, n_bg=n_bg)


# ---------------------------------------------------------------------------------------------------------------------
# which branch each victim takes
# ---------------------------------------------------------------------------------------------------------------------
def first_pass_events(ds):
    rec, types = O.trim_type_batch(ds.records, ds.piles)
    a, b = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
    kb = (types == O.KB) & ((ds.flags[b] & 2) == 0)
    ka = (types == O.KA) & ((ds.flags[a] & 2) == 0)
    t = np.nonzero(kb | ka)[0]
    return np.where(kb[t], a[t], b[t]), np.where(kb[t], b[t], a[t]), t.astype(np.int64)


def sequential(v, c, t, n):
    alive = np.ones(n, bool)
    D = np.full(n, INF)
    for i in np.argsort(t, kind="stable"):
        if alive[v[i]] and alive[c[i]]:
            alive[v[i]] = False
            D[v[i]] = t[i]
    return D


def branches(v, c, t, n):
    """Per victim: the branch of k_resolve_fast, and for hard victims what their earliest container does."""
    D = sequential(v, c, t, n)
    tmin = np.full(n, INF)
    np.minimum.at(tmin, v, t)
    o = np.lexsort((t, v))
    first = np.r_[0, np.flatnonzero(np.diff(v[o])) + 1]
    fv, fc, ft = v[o][first], c[o][first], t[o][first]
    self_ = fc == fv
    no_ev = ~self_ & (tmin[fc] == INF)
    later = ~self_ & ~no_ev & (tmin[fc] > ft)
    easy = self_ | no_ev | later
    assert np.array_equal(D[fv[easy]], ft[easy]), "an easy victim dies at its earliest event"
    hard = ~easy
    c_easy = np.zeros(n, bool)
    c_easy[fv[easy]] = True
    hv, hc, ht = fv[hard], fc[hard], ft[hard]
    return {"self": int(self_.sum()), "no_events": int(no_ev.sum()), "later": int(later.sum()),
            "hard": int(hard.sum()), "hard_easy_container": int(c_easy[hc].sum()),
            "hard_container_dies_before": int(((~c_easy[hc]) & (D[hc] < ht)).sum()),
            "hard_container_dies_after": int(((~c_easy[hc]) & (D[hc] > ht) & (D[hc] != INF)).sum()),
            "hard_container_never": int(((~c_easy[hc]) & (D[hc] == INF)).sum())}


def test_record_sets_take_every_branch():
    ds = build("mixed")
    b = branches(*first_pass_events(ds), ds.n_piles)
    assert all(x >= 100 for x in b.values()), b
    ds = build("all_easy")
    b = branches(*first_pass_events(ds), ds.n_piles)
    assert b["hard"] == 0 and b["no_events"] >= 3000, b
    ds = build("all_hard")
    b = branches(*first_pass_events(ds), ds.n_piles)
    assert b["hard"] >= 3800, b
    for name in ("mixed", "all_hard"):    # flagged: the designed containments wait for the final pass
        ds = build(name, flagged=True)
        v, c, t = first_pass_events(ds)
        assert not np.any(c >= ds.n_bg)
    ds = build("mixed", hills=True)
    assert ds.hills.shape[0] >= 100
    ds = build("deep")
    b = branches(*first_pass_events(ds), ds.n_piles)
    assert b["hard"] >= 20_000 + 600 * 59 - 601, b


# ---------------------------------------------------------------------------------------------------------------------
# GPU against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _same(G, P, label):
    c = G.counts()
    assert np.array_equal(G.piles(), P.piles), f"{label}: piles"
    ovl, inl = G.lists()
    assert np.array_equal(ovl, P.ovl), f"{label}: final overlaps"
    assert np.array_equal(inl, P.int), f"{label}: final internals (filtered by the death times)"
    assert np.array_equal(G.edges(), P.edges), f"{label}: edges"
    assert np.array_equal(G.marked(), P.marked), f"{label}: marks"
    assert np.array_equal(G.seq_to_node(), P.seq_to_node), f"{label}: node ids"
    assert c["n_nodes"] == P.n_nodes and c["n_transitive_pairs"] == P.n_pairs, label
    return c


CASES = [("mixed", False, False), ("all_easy", False, False), ("all_hard", False, False),
         ("mixed", True, False), ("all_hard", True, False), ("mixed", False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,flagged,hills", CASES)
def test_resolution_matches_the_oracle(ctx, name, flagged, hills):
    ds = build(name, flagged, hills)
    first = O.Pipeline(ds.records, ds.piles, ds.flags, ds.hills).classify()
    P = O.Pipeline(ds.records, ds.piles, ds.flags, ds.hills).run()
    G = api.Graph(ctx)
    try:
        G.use_cuda_graph(False)
        G.set_piles(ds.piles, ds.flags).set_hills(ds.hills).set_overlaps(ds.records)
        G.classify()
        assert np.array_equal(G.piles(), first.piles), "piles after the first pass"
        if hills:
            assert np.array_equal(G.hill_coverage(), first.hill_cov), "hill counters"
            assert first.hill_cov.sum() > 0
        G.run()
        c = _same(G, P, "eager")
        G.use_cuda_graph(True)
        for i in range(2):
            G.run()
            _same(G, P, f"graph run {i}")
    finally:
        G.close()
    if name == "all_easy":
        assert c["n_rounds"] == 0, "nothing hard: the worklist is empty"
    if flagged:
        assert c["n_final_rounds"] >= 1, "the final pass has hard victims"


@pytest.mark.gpu
def test_deep_chains_still_reach_the_chase_and_the_worklist(ctx):
    """Chains far deeper than the chase stack are hard but for their first link: the resolution must still go round the
    worklist, and end in the oracle's answer."""
    ds = build("deep")
    P = O.Pipeline(ds.records, ds.piles, ds.flags).run()
    G = api.Graph(ctx)
    try:
        G.set_piles(ds.piles, ds.flags).set_hills(None).set_overlaps(ds.records)
        G.run()
        c = _same(G, P, "deep")
    finally:
        G.close()
    assert c["n_rounds"] > 1, c["n_rounds"]
