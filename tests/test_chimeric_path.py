"""The chimeric-pile path of Graph::construct: piles with chimeric hills or regions, hill counters bumped in the first pass
(Pile::check_chimeric_hills, SURVEY.md A.6), and a pile table the host changes between the passes (hill breaking, then
the pit loop).  The CUDA session against the oracle, bit for bit, stage by stage; the oracle against hand-derived
answers and against a numpy restatement of the first pass (A.3 + A.6).

The host's Pile calls are replaced by `PileDriver`, a deterministic stand-in that changes the table the way pile
breaking does (cuts, kills, rounds that change nothing) without reproducing pile.cpp's rules.
"""
import functools
from types import SimpleNamespace

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from oracle import oracle as O
from rala_b200 import api, synth
from tests.replay import assert_same

INF = np.iinfo(np.int64).max
K_HILL_THREADS = 2 * 148 * 256    # k_hill_coverage's grid (two blocks of 256 per SM): more records go round its loop
K_TILE = 1024                     # entries per look-back tile of the ordered list passes


# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement of the first pass: death times (A.3) and hill counters (A.6)
# ---------------------------------------------------------------------------------------------------------------------
def first_pass(records, piles, flags):
    """Trimmed records, types, death times and the record sides that land on a pile, computed without the oracle's
    sequential loop: D[x] = min{t : record t kills x and its container is alive at t}, iterated to its fixed point."""
    rec, types = O.trim_type_batch(records, piles)        # static gates: valid, ids known, piles alive, trim accepts
    n, n_piles = rec.shape[0], piles.shape[0]
    ok = types != O.REJECT
    a = np.where(ok, rec[:, 0], 0).astype(np.int64)
    b = np.where(ok, rec[:, 1], 0).astype(np.int64)
    kill_a = ok & (types == O.KB) & ((flags[b] & 2) == 0)   # a contained in b, which has no chimeric region
    kill_b = ok & (types == O.KA) & ((flags[a] & 2) == 0)
    ev = np.nonzero(kill_a | kill_b)[0]
    v = np.where(kill_a[ev], a[ev], b[ev])
    c = np.where(kill_a[ev], b[ev], a[ev])
    D = np.full(n_piles, INF, dtype=np.int64)
    for _ in range(10000):
        fire = (D[c] > ev) | (c == v)                        # a self overlap kills its pile whatever its fate
        nxt = np.full(n_piles, INF, dtype=np.int64)
        np.minimum.at(nxt, v[fire], ev[fire])
        if np.array_equal(nxt, D):
            break
        D = nxt
    else:
        raise AssertionError("death times did not converge")
    t = np.arange(n)
    processed = ok & (D[a] >= t) & (D[b] >= t)
    # the two sides of every accepted record: pile, lo = begin_ + start, hi = begin_ + end (A.6)
    begin = piles[:, 0].astype(np.int64)
    b_lo = np.where(a == b, rec[:, 2], rec[:, 4]).astype(np.int64)
    b_hi = np.where(a == b, rec[:, 3], rec[:, 5]).astype(np.int64)
    side = SimpleNamespace(
        pile=np.concatenate([a[ok], b[ok]]),
        lo=np.concatenate([begin[a[ok]] + rec[ok, 2], begin[b[ok]] + b_lo[ok]]),
        hi=np.concatenate([begin[a[ok]] + rec[ok, 3], begin[b[ok]] + b_hi[ok]]),
        t=np.concatenate([t[ok], t[ok]]),
        processed=np.concatenate([processed[ok], processed[ok]]))
    return SimpleNamespace(rec=rec, types=types, ok=ok, a=a, b=b, D=D, processed=processed, side=side)


def hill_pairs(hills, side, flags):
    """(side index, hill row) of every side on a pile with hills, against every hill of that pile."""
    hp = hills[:, 0].astype(np.int64)
    on = np.nonzero((flags[side.pile] & 1) != 0)[0]
    start = np.searchsorted(hp, side.pile[on], "left")
    stop = np.searchsorted(hp, side.pile[on], "right")
    si, hi = [], []
    for k in range(int((stop - start).max(initial=0))):
        m = start + k < stop
        si.append(on[m])
        hi.append(start[m] + k)
    if not si:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(si), np.concatenate(hi)


def model_coverage(hills, fp, flags):
    si, hi = hill_pairs(hills, fp.side, flags)
    s = fp.side
    hit = s.processed[si] & (s.lo[si] < hills[hi, 1]) & (s.hi[si] > hills[hi, 2])
    return np.bincount(hi[hit], minlength=hills.shape[0]).astype(np.uint32)


# ---------------------------------------------------------------------------------------------------------------------
# input builder
# ---------------------------------------------------------------------------------------------------------------------
def chimeric_input(ds, seed, hill_frac=0.08, region_frac=0.04, dead_frac=0.01):
    """A synth dataset as the chimeric path sees it: a realistic pile table (begins 0 .. 3 000, shortened ends, a few dead
    piles), flags as the reference sets them (3 = hills, which imply a chimeric region; 2 = region only) and 1 .. 6 hills
    per hill pile, mostly placed on the bounds of the trimmed spans of records that land on the pile."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = ds.n_reads
    end = ds.read_len.astype(np.int64) - rng.integers(0, 1500, n)
    begin = np.minimum(rng.integers(0, 3001, n), np.maximum(end - 1500, 0))
    piles = np.stack([begin, end], 1).astype(np.uint32)
    dead = rng.random(n) < dead_frac
    dead[[0, n - 1]] = False
    piles[dead] = 0
    has_hill = (rng.random(n) < hill_frac) & ~dead
    has_hill[[0, n - 1]] = True                              # the first and the last row of the hill table
    region = (rng.random(n) < region_frac) & ~dead & ~has_hill
    flags = np.where(has_hill, 3, np.where(region, 2, 0)).astype(np.uint8)

    fp = first_pass(ds.records, piles, flags)
    s = fp.side
    order = np.argsort(s.pile, kind="stable")
    sp, slo, shi, st = s.pile[order], s.lo[order], s.hi[order], s.t[order]
    rows = []
    for x in np.nonzero(has_hill)[0].tolist():
        i0, i1 = np.searchsorted(sp, [x, x + 1])
        lo, hi, t = slo[i0:i1], shi[i0:i1], st[i0:i1]
        mine = []
        if fp.D[x] != INF:            # dies in the first pass: a hill just inside the span of the record that kills it
            j = int(np.nonzero(t == fp.D[x])[0][0])
            mine.append((int(lo[j]) + 1, int(hi[j]) - 1))
        for _ in range(int(rng.integers(1, 7)) - len(mine)):
            u = rng.random()
            if lo.size == 0:
                f = int(piles[x, 0]) + int(rng.integers(0, 3000))
                mine.append((f, f + 500))
            elif u < 0.12:            # no record spans it
                top = int(hi.max())
                mine.append((top, top + 50))
            elif u < 0.3:             # deep inside the pile: more than 3 hits
                m = int(np.median((lo + hi) // 2))
                mine.append((m, m + int(rng.integers(1, 300))))
            else:                     # on a record's bounds: exactly at, one below, one above
                j = int(rng.integers(lo.size))
                f = max(int(lo[j]) + int(rng.integers(-1, 2)), 0)
                later = np.nonzero(hi > f + 1)[0]
                k = j if rng.random() < 0.5 or later.size == 0 else int(later[rng.integers(later.size)])
                mine.append((f, max(f, int(hi[k]) + int(rng.integers(-1, 2)))))
        rows += [(x, f, s_) for f, s_ in sorted(mine)]
    hills = np.asarray(rows, dtype=np.uint32).reshape(-1, 3)
    return SimpleNamespace(records=ds.records, piles=piles, flags=flags, hills=hills, fp=fp, seed=seed)


DATASETS = {
    # noisy, both directions of every overlap listed: the big one (> 75 776 records on hill piles, lists of many tiles)
    "noisy_dual": (dict(genome_len=3_000_000, coverage=40, read_len=9000, len_sd=2500, seed=101, noise=80, dual=True), 0.13),
    "chimeras_repeats": (dict(genome_len=1_500_000, coverage=45, read_len=10000, len_sd=3000, seed=102, noise=30,
                              chimera_frac=0.05, repeats=(2, 10, 3000)), 0.08),
    "jittered": (dict(genome_len=1_500_000, coverage=35, read_len=10000, len_sd=3000, seed=103, noise=400), 0.08),
}


@functools.lru_cache(maxsize=None)
def dataset(name):
    kw, frac = DATASETS[name]
    return chimeric_input(synth.generate(**kw), kw["seed"], hill_frac=frac)


# ---------------------------------------------------------------------------------------------------------------------
# test-only pile breaking
# ---------------------------------------------------------------------------------------------------------------------
def _mix(*xs):
    h = np.full(np.broadcast(*[np.asarray(x) for x in xs]).shape, 0x9E3779B97F4A7C15, dtype=np.uint64)
    for x in xs:
        h = (h ^ np.asarray(x, dtype=np.uint64)) * np.uint64(0xBF58476D1CE4E5B9)
        h ^= h >> np.uint64(29)
    return h


class PileDriver:
    """Deterministic stand-in for the host's Pile calls between the passes.

    Hill step: every hill with coverage <= 3 cuts its pile to the longer side of the hill (hill coordinates carry the
    pile's begin once more, A.6, and the cut takes it off again); a pile with fewer than 1 000 bases left dies.  Bit 0
    of the flags is cleared afterwards.  Pit rounds: rounds 0 .. change_rounds - 1 shrink or kill a hash-chosen subset
    of the piles of every component of the connections (at least one per component); later rounds change nothing."""

    def __init__(self, hills, flags, seed):
        self.hills = np.asarray(hills, dtype=np.int64).reshape(-1, 3)
        self.flags = np.asarray(flags, dtype=np.uint8).copy()
        self.seed = seed
        self.change_rounds = 2 + seed % 2

    def hill_step(self, cov, piles):
        p = piles.astype(np.int64)
        for (x, first, second), c in zip(self.hills.tolist(), np.asarray(cov).tolist()):
            b, e = p[x]
            if e == 0 or c > 3:       # dead, or a hill with more than 3 hits is ignored (pile.cpp:479)
                continue
            f, s = min(max(first - b, b), e), min(max(second - b, b), e)
            b, e = (b, f) if f - b >= e - s else (s, e)
            p[x] = (b, e) if e - b >= 1000 else (0, 0)
        self.flags &= np.uint8(0xFE)
        return p.astype(np.uint32), self.flags.copy()

    def pit_round(self, connections, piles, r):
        if r >= self.change_rounds:
            return None
        n = piles.shape[0]
        conn = np.asarray(connections, dtype=np.int64).reshape(-1, 2)
        g = coo_matrix((np.ones(conn.shape[0]), (conn[:, 0], conn[:, 1])), shape=(n, n))
        _, label = connected_components(g, directed=False)
        touched = np.unique(conn)
        h = _mix(touched, self.seed, r)
        pick = h % np.uint64(4) == 0
        by_comp = np.lexsort((h, label[touched]))          # the smallest hash of every component is picked too
        comp = label[touched][by_comp]
        pick[by_comp[np.r_[0, np.nonzero(comp[1:] != comp[:-1])[0] + 1]]] = True
        p = piles.astype(np.int64)
        for x, hx in zip(touched[pick].tolist(), h[pick].tolist()):
            b, e = p[x]
            if e == 0:
                continue
            cut = 500 + (hx >> 8) % 3500                     # off one end: what is left is often inside an overlap
            b, e = (b + cut, e) if hx & 16 else (b, e - cut)
            p[x] = (b, e) if (hx >> 20) % 9 and e - b >= 1000 else (0, 0)
        return p.astype(np.uint32), self.flags.copy()


class PileOps:
    """The pile_ops interface of api.Graph.construct around a PileDriver.  `table` returns the session's pile table.
    With `want` (the calls an oracle-driven construct made), every input is compared with the oracle's before the
    driver runs, so a divergence is reported at the stage where it starts."""

    def __init__(self, driver, table, want=None):
        self.driver, self.table, self.want, self.calls = driver, table, want, []

    def _inputs(self, what, x):
        piles = self.table()
        k = len(self.calls)
        if self.want is not None:
            assert k < len(self.want), f"{what}: call {k}, the oracle made {len(self.want)}"
            w = self.want[k]
            assert w[0] == what, (k, what, w[0])
            assert_same(x, w[1], f"{what} call {k}: input")
            assert_same(piles, w[2], f"{what} call {k}: pile table")
        self.calls.append((what, np.array(x, copy=True), piles.copy()))
        return piles

    def break_over_chimeric_hills(self, cov):
        return self.driver.hill_step(cov, self._inputs("hills", cov))

    def break_over_chimeric_pits(self, connections):
        return self.driver.pit_round(connections, self._inputs("pits", connections), len(self.calls) - 2)


def oracle_construct(inp, ops):
    """api.Graph.construct's flow on the oracle pipeline; returns (pipeline, is_changed of every pit round)."""
    P = O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills).classify()
    ops.table = lambda: P.piles
    upd = ops.break_over_chimeric_hills(P.hill_cov.copy())
    if upd is not None:
        P.set_piles(upd[0])
    P.retrim()
    changed = []
    while True:
        upd = ops.break_over_chimeric_pits(np.ascontiguousarray(P.ovl[:, :2]))
        if upd is not None:
            P.set_piles(upd[0])
        changed.append(P.retrim_promote())
        if not changed[-1]:
            break
    return P, changed


def final_events(P):
    """kA / kB entries the final containment pass sees (both lists, typed against the final table)."""
    lst = np.concatenate([P.ovl, P.int])
    _, t = O.trim_type_batch(lst, P.piles)
    return int(((t == O.KA) | (t == O.KB)).sum())


@functools.lru_cache(maxsize=None)
def constructed(name):
    inp = dataset(name)
    ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), None)
    P, changed = oracle_construct(inp, ops)
    n_final = final_events(P)
    P.final_containment().build_edges().transitive()
    return P, changed, ops.calls, n_final


# ---------------------------------------------------------------------------------------------------------------------
# hand-derived known answers
# ---------------------------------------------------------------------------------------------------------------------
S = (100, 9900)      # a pile with valid region [100, 9900): lo = 100 + start, hi = 100 + end
KAB, KBA, KA, KB, KX, REJ = O.KAB, O.KBA, O.KA, O.KB, O.KX, O.REJECT


def _case(piles, flags, hills, records, types, want):
    return dict(piles=np.asarray(piles, np.uint32).reshape(-1, 2), flags=np.asarray(flags, np.uint8),
                hills=np.asarray(hills, np.uint32).reshape(-1, 3), records=np.asarray(records, np.uint32).reshape(-1, 7),
                types=types, want=want)


# Every expected count follows A.6: lo = begin_ + start', hi = begin_ + end' of the trimmed record on the hill's pile,
# a hit iff lo < first && hi > second, for records that pass the static gates while both their piles are alive.
KNOWN = {
    # a side: lo = 100 + 1000 = 1100, hi = 100 + 9000 = 9100
    "first_bound": _case([S, S], [3, 0], [(0, 1099, 5000), (0, 1100, 5000), (0, 1101, 5000)],
                         [(0, 1, 1000, 9000, 100, 8100, 0)], [KAB], [0, 0, 1]),
    "second_bound": _case([S, S], [3, 0], [(0, 2000, 9099), (0, 2000, 9100), (0, 2000, 9101)],
                          [(0, 1, 1000, 9000, 100, 8100, 0)], [KAB], [1, 0, 0]),
    # b side: lo = 100 + 100 = 200, hi = 100 + 8100 = 8200
    "b_side_bounds": _case([S, S], [0, 3], [(1, 199, 4000), (1, 200, 4000), (1, 201, 4000), (1, 300, 8199), (1, 300, 8200),
                                            (1, 300, 8201)],
                           [(0, 1, 1000, 9000, 100, 8100, 0)], [KAB], [0, 0, 1, 1, 0, 0]),
    # begin_ = 2000: [2500, 11500) spans [3000, 11000] in read coordinates, but lo = 4500, hi = 13500
    "begin_quirk": _case([(2000, 12000), S], [3, 0], [(0, 3000, 11000), (0, 4600, 13000)],
                         [(0, 1, 2500, 11500, 100, 8100, 0)], [KAB], [0, 1]),
    # a begins before the pile: trim moves it to 100, so lo = 200 (the raw start would give 150)
    "trimmed_coordinates": _case([S, S], [3, 0], [(0, 180, 5000), (0, 201, 5000)],
                                 [(0, 1, 50, 9000, 100, 9050, 0)], [KA], [0, 1]),
    # lo = 3100, hi = 6100: an internal counts, the bump comes before type()
    "internal_counts": _case([S, S], [3, 0], [(0, 3200, 6000), (0, 3100, 6000)],
                             [(0, 1, 3000, 6000, 3000, 6000, 0)], [KX], [1, 0]),
    # 50 bases left after the cut at 9900: rejected by trim (its raw span [9950, 10090] would span the hill)
    "trim_rejects": _case([S, S], [3, 0], [(0, 9960, 9990)], [(0, 1, 9850, 9990, 100, 240, 0)], [REJ], [0]),
    "invalid_record": _case([S, S], [3, 0], [(0, 1101, 5000)], [(0, 1, 1000, 9000, 100, 8100, 2)], [REJ], [0]),
    "dead_on_input": _case([S, (0, 0)], [3, 0], [(0, 1101, 5000)], [(0, 1, 1000, 9000, 100, 8100, 0)], [REJ], [0]),
    # t=0 dovetail (lo 1100, hi 5200); t=1 kills pile 0 (lo 200, hi 5200) and still counts; t=2 finds pile 0 dead
    "killed_at_its_own_time": _case([(100, 5100), S, S], [3, 0, 0], [(0, 300, 5000), (0, 1200, 5000)],
                                    [(0, 2, 1000, 5100, 100, 4200, 0), (0, 1, 100, 5100, 2000, 7000, 0),
                                     (0, 2, 100, 5100, 2000, 7000, 0)], [KAB, KB, KB], [1, 2]),
    # t=0 kills pile 1; t=1 would span the hill of pile 0 but its other pile is dead; t=2 counts
    "partner_dead": _case([S, (100, 5100), S], [3, 0, 0], [(0, 1101, 5000)],
                          [(1, 2, 100, 5100, 2000, 7000, 0), (0, 1, 1000, 5000, 100, 4100, 0), (0, 2, 1000, 9000, 100, 8100, 0)],
                          [KB, KX, KAB], [1]),
    # the container of t=0 has a chimeric region: no kill, t=1 counts and kills, t=2 does not count
    "region_blocks_the_kill": _case([(100, 5100), S, S], [3, 2, 0], [(0, 300, 5000)],
                                    [(0, 1, 100, 5100, 2000, 7000, 0), (0, 2, 100, 5100, 2000, 7000, 0),
                                     (0, 1, 100, 5100, 2000, 7000, 0)], [KB, KB, KB], [2]),
    # the hill pile contains its partner twice over; its region keeps the partner alive, both records count
    "hill_pile_as_container": _case([S, (100, 5100)], [3, 0], [(0, 2101, 7099)],
                                    [(0, 1, 2000, 7000, 100, 5100, 0), (1, 0, 100, 5100, 2000, 7000, 0)], [KA, KB], [2]),
    # reverse complement: the 50 bases cut off a's end move b's start to 4900, so b's lo = 5000, hi = 10000
    "reverse_complement": _case([S, S], [0, 3], [(1, 4990, 9000), (1, 5001, 9999), (1, 5001, 10000)],
                                [(0, 1, 5000, 9950, 4850, 9900, 1)], [KAB], [0, 1, 0]),
    # both piles have hills: a (1100, 9100) and b (200, 8200) each bump their own pile only
    "both_piles_have_hills": _case([S, S], [3, 3], [(0, 1101, 9099), (0, 201, 8199), (1, 201, 8199), (1, 1101, 9099)],
                                   [(0, 1, 1000, 9000, 100, 8100, 0)], [KAB], [1, 0, 1, 0]),
    # hills of several piles: the search finds each pile's rows, the last pile's included
    "several_piles": _case([S] * 6, [3, 0, 3, 0, 0, 3],
                           [(0, 1101, 5000), (2, 1099, 5000), (2, 1101, 5000), (2, 2000, 9099), (5, 199, 8199), (5, 201, 8199)],
                           [(2, 1, 1000, 9000, 100, 8100, 0), (1, 5, 1000, 9000, 100, 8100, 0)], [KAB, KAB],
                           [0, 0, 1, 1, 0, 1]),
    "more_than_three_hits": _case([S] * 6, [3, 0, 0, 0, 0, 0], [(0, 1101, 9099), (0, 1100, 9099)],
                                  [(0, k, 1000, 9000, 100, 8100, 0) for k in range(1, 6)], [KAB] * 5, [5, 0]),
    # a self overlap (a == b) bumps its pile twice, both times with the a-side span lo = 1100, hi = 3100
    "self_overlap": _case([S], [3], [(0, 1200, 3000), (0, 6200, 8000)], [(0, 0, 1000, 3000, 6000, 8000, 0)], [KX], [2, 0]),
}


def test_known_answers_are_what_the_oracle_counts():
    """The hand-derived counts above, and the record types their derivations assume, against the oracle."""
    for name, k in KNOWN.items():
        _, types = O.trim_type_batch(k["records"], k["piles"])
        assert types.tolist() == k["types"], (name, types.tolist())
        P = O.Pipeline(k["records"], k["piles"], k["flags"], k["hills"]).classify()
        assert P.hill_cov.tolist() == k["want"], (name, P.hill_cov.tolist())
        fp = first_pass(k["records"], k["piles"], k["flags"])
        assert model_coverage(k["hills"], fp, k["flags"]).tolist() == k["want"], name


def test_self_overlap_counts_the_a_side_twice():
    """A self overlap (a == b) on a pile with hills.  The reference's Pile::check_chimeric_hills picks the side by comparing
    the overlap's a id with the pile's own id (SURVEY.md A.6: `x == a ? ab' : bb'`), so both of its calls for a self
    overlap take the a-side span.  The reference's duplicate filter never lets a self overlap through, but the session
    API accepts one, and the oracle and the kernel follow A.6.  test_reference_hill_coverage_matches_the_oracle pins
    this against the compiled reference where that build is present."""
    k = KNOWN["self_overlap"]
    rec = k["records"].copy()
    P = O.Pipeline(rec, k["piles"], k["flags"], k["hills"]).classify()
    assert P.hill_cov.tolist() == [2, 0]
    rec[0, 2:6] = (6000, 8000, 1000, 3000)            # the mirrored record: now the other span is the a side
    P = O.Pipeline(rec, k["piles"], k["flags"], k["hills"]).classify()
    assert P.hill_cov.tolist() == [0, 2]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the builder and the driver give the GPU tests what they rely on
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(DATASETS))
def test_builder_inputs_cover_the_hard_cases(name):
    inp = dataset(name)
    n_piles = inp.piles.shape[0]
    hp = inp.hills[:, 0]
    assert (np.diff(hp.astype(np.int64)) >= 0).all(), "hills grouped by ascending pile id"
    assert hp[0] == 0 and hp[-1] == n_piles - 1
    counts = np.bincount(hp, minlength=n_piles)
    has = (inp.flags & 1) != 0
    assert (counts[has] >= 1).all() and counts.max() <= 6 and not counts[~has].any()
    assert ((inp.flags == 0) | (inp.flags == 2) | (inp.flags == 3)).all(), "flag 1 alone is off-contract"
    assert (inp.piles[:, 1] == 0).sum() > 0 and inp.piles[:, 0].max() > 2500

    P = O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills).classify()
    fp = inp.fp
    assert_same(model_coverage(inp.hills, fp, inp.flags), P.hill_cov, "hill coverage: numpy model vs oracle")
    cov = P.hill_cov
    assert (cov == 0).any() and ((cov >= 1) & (cov <= 3)).any() and (cov > 3).sum() > 10

    # records on both sides of both strict inequalities, at the bound itself
    si, hi = hill_pairs(inp.hills, fp.side, inp.flags)
    s = fp.side
    pr = s.processed[si]
    lo, up = s.lo[si], s.hi[si]
    first, second = inp.hills[hi, 1].astype(np.int64), inp.hills[hi, 2].astype(np.int64)
    assert (pr & (lo == first) & (up > second)).sum() > 20, "lo == first (not a hit; one with <=)"
    assert (pr & (lo + 1 == first) & (up > second)).sum() > 20, "lo one below first (a hit)"
    assert (pr & (up == second) & (lo < first)).sum() > 20, "hi == second (not a hit; one with >=)"
    assert (pr & (up == second + 1) & (lo < first)).sum() > 20, "hi one above second (a hit)"
    # a hill pile that dies in the first pass, bumped by the record that kills it (D[x] == t is still alive)
    dies = has & (fp.D != INF)
    killer = pr & (s.t[si] == fp.D[s.pile[si]]) & (lo < first) & (up > second)
    assert dies.sum() > 20 and killer.sum() > 20
    # ... and records on it after its death that would have counted
    assert (~pr & (s.t[si] > fp.D[s.pile[si]]) & (lo < first) & (up > second)).sum() > 0
    # kA / kB whose container is a hill pile (it has a chimeric region): kept in `overlaps`
    _, t1 = O.trim_type_batch(P.ovl, P.piles)
    kept = ((t1 == O.KA) & ((inp.flags[P.ovl[:, 0]] & 1) != 0)) | ((t1 == O.KB) & ((inp.flags[P.ovl[:, 1]] & 1) != 0))
    assert kept.sum() > 20
    if name == "noisy_dual":
        on_hill_piles = fp.ok & (((inp.flags[fp.a] | inp.flags[fp.b]) & 1) != 0)
        assert on_hill_piles.sum() > K_HILL_THREADS, "k_hill_coverage goes around its grid-stride loop"
        assert P.ovl.shape[0] > 10 * K_TILE, "the list passes span many look-back tiles"
    if name == "chimeras_repeats":
        assert P.int.shape[0] > 100, "internals (repeat-induced overlaps) for the pit loop to promote"


@pytest.mark.parametrize("name", list(DATASETS))
def test_driver_changes_the_pile_table_between_the_passes(name):
    inp = dataset(name)
    P, changed, calls, n_final = constructed(name)
    assert calls[0][0] == "hills" and all(c[0] == "pits" for c in calls[1:])
    after_hills = PileDriver(inp.hills, inp.flags, inp.seed).hill_step(calls[0][1], calls[0][2])[0]
    assert (after_hills != calls[0][2]).any(axis=1).sum() > 50, "the hill step cuts piles"
    assert len(changed) >= 2 and any(changed), changed
    assert n_final >= (1000 if name == "noisy_dual" else 200), f"{n_final} containment events in the final pass"
    assert P.edges.shape[0] > 1000 and P.n_pairs > 0


# ---------------------------------------------------------------------------------------------------------------------
# reference (skips where oracle/_ref is not built)
# ---------------------------------------------------------------------------------------------------------------------
def _ref_hills(tmp_path, tag, records, piles, flags, hills):
    prefix = str(tmp_path / tag)
    O.write_hotpath_inputs(prefix, records, piles, flags, hills)
    O.ref_run(["hotpath", prefix, prefix])
    return O.load_u32(prefix + ".stage.s1.hills.u32", 4)


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (needs /root/reference)")
def test_reference_hill_coverage_matches_the_oracle(tmp_path):
    """The compiled reference's hill counters (rala_ref hotpath, stage s1: hills of the piles still alive) against the
    oracle, on the known answers (the self overlap included) and on the builder's inputs."""
    inputs = [(name, k["records"], k["piles"], k["flags"], k["hills"]) for name, k in KNOWN.items()]
    inputs.append(("jittered",) + tuple(getattr(dataset("jittered"), f) for f in ("records", "piles", "flags", "hills")))
    for name, records, piles, flags, hills in inputs:
        P = O.Pipeline(records, piles, flags, hills).classify()
        alive = P.piles[hills[:, 0], 1] != 0
        want = np.concatenate([hills[alive], P.hill_cov[alive, None]], 1)
        assert_same(_ref_hills(tmp_path, name, records, piles, flags, hills), want, f"{name}: hills after classify")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _same_lists(G, P, what):
    ovl, inl = G.lists()
    assert_same(ovl, P.ovl, f"{what} overlaps")
    assert_same(inl, P.int, f"{what} internals")


@pytest.mark.gpu
def test_known_answers_on_the_gpu(ctx):
    G = api.Graph(ctx)
    for name, k in KNOWN.items():
        G.set_piles(k["piles"], k["flags"]).set_hills(k["hills"]).set_overlaps(k["records"])
        G.classify()
        assert G.hill_coverage().tolist() == k["want"], name
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DATASETS))
def test_stage_by_stage_with_changing_pile_tables(ctx, name):
    inp = dataset(name)
    P = O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills)
    G = api.Graph(ctx)
    G.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_overlaps(inp.records)
    P.classify()
    G.classify()
    _same_lists(G, P, "s1")
    cov = G.hill_coverage()
    assert_same(cov, P.hill_cov, "hill coverage")
    assert_same(G.piles(), P.piles, "s1 piles")
    assert_same(G.connections(), P.ovl[:, :2], "s1 connections")

    drv = PileDriver(inp.hills, inp.flags, inp.seed)
    piles, flags = drv.hill_step(cov, P.piles)
    P.set_piles(piles).retrim()
    G.set_piles(piles, flags).retrim()
    _same_lists(G, P, "after the hill step")
    r = 0
    while True:
        conn = G.connections()
        assert_same(conn, P.ovl[:, :2], f"connections before pit round {r}")
        assert_same(G.piles(), P.piles, f"piles before pit round {r}")
        upd = drv.pit_round(conn, P.piles, r)
        if upd is not None:
            P.set_piles(upd[0])
            G.set_piles(*upd)
        want_changed = P.retrim_promote()
        assert G.retrim_promote() == want_changed, f"is_changed of pit round {r}"
        _same_lists(G, P, f"pit round {r}")
        r += 1
        if not want_changed:
            break
    assert r >= 2
    assert_same(G.hill_coverage(), cov, "hill coverage after the pile table changed")

    P.final_containment()
    G.finalize()
    _same_lists(G, P, "final")
    assert_same(G.piles(), P.piles, "final piles")
    P.build_edges()
    G.build()
    c = G.counts()
    assert c["n_nodes"] == P.n_nodes and c["n_edges"] == P.edges.shape[0]
    assert_same(G.edges(), P.edges, "edges")
    assert_same(G.seq_to_node(), P.seq_to_node, "seq_to_node")
    P.transitive()
    G.transitive()
    assert G.counts()["n_transitive_pairs"] == P.n_pairs
    assert_same(G.marked(), P.marked, "marks")
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DATASETS))
def test_construct_with_pile_breaking_matches_the_oracle(ctx, name):
    """api.Graph.construct with the driver, every input of the driver compared with what the oracle-driven construct
    handed it, then the final lists, piles, edges, node ids and the transitive pass."""
    inp = dataset(name)
    P, changed, calls, _ = constructed(name)
    G = api.Graph(ctx)
    ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), G.piles, want=calls)
    G.construct(inp.records, inp.piles, inp.flags, inp.hills, pile_ops=ops)
    assert len(ops.calls) == len(calls)
    _same_lists(G, P, "final")
    assert_same(G.piles(), P.piles, "final piles")
    assert G.n_nodes == P.n_nodes
    assert_same(G.edges(), P.edges, "edges")
    assert_same(G.seq_to_node(), P.seq_to_node, "seq_to_node")
    assert G.remove_transitive_edges() == P.n_pairs
    assert_same(G.removed, P.marked, "marks")
    G.close()


@pytest.mark.gpu
def test_run_with_hills_eager_captured_and_replayed(ctx):
    """rala_b200_graph_run with hills and a frozen pile table: the first pass decodes the death times separately so the
    hill counters can read them, and the counters are zeroed inside every run, replays of the captured graph included."""
    inp = dataset("jittered")
    rng = np.random.Generator(np.random.PCG64(7))
    h2 = inp.hills.copy()                                  # same count, new contents
    h2[:, 1:] += rng.integers(-40, 41, (h2.shape[0], 1)).astype(np.uint32)
    h3 = inp.hills[rng.random(inp.hills.shape[0]) < 0.7]   # another count
    plain = O.Pipeline(inp.records, inp.piles, inp.flags).run()
    G0 = api.Graph(ctx)
    G0.set_piles(inp.piles, inp.flags).set_hills(None).set_overlaps(inp.records).run()
    want_edges, want_marks = G0.edges(), G0.marked()
    G0.close()
    assert_same(want_edges, plain.edges, "edges without hills")
    assert_same(want_marks, plain.marked, "marks without hills")

    G = api.Graph(ctx)
    G.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_overlaps(inp.records)
    for label, hills, runs in (("hills", inp.hills, 5), ("same count, new contents", h2, 3), ("another count", h3, 3),
                               ("no hills", None, 3), ("hills again", inp.hills, 3)):
        if label != "hills":
            G.set_hills(hills)
        P = O.Pipeline(inp.records, inp.piles, inp.flags, hills).run()
        for i in range(runs):
            G.run()
            cov = G.hill_coverage()
            if hills is None:
                assert cov.shape == (0,)
            else:
                assert_same(cov, P.hill_cov, f"{label}, run {i}: hill coverage")
                assert (P.hill_cov > 0).sum() > 100
            assert_same(G.edges(), P.edges, f"{label}, run {i}: edges")
            assert_same(G.marked(), P.marked, f"{label}, run {i}: marks")
            assert_same(G.edges(), want_edges, f"{label}, run {i}: edges as without hills")
            assert_same(G.marked(), want_marks, f"{label}, run {i}: marks as without hills")
    G.close()


@pytest.mark.gpu
def test_hill_api_edges(ctx):
    inp = dataset("jittered")
    G = api.Graph(ctx)
    j = int(np.nonzero(inp.hills[:, 0] > inp.hills[0, 0])[0][0])   # the first row of the second pile with hills
    bad = inp.hills.copy()
    bad[[0, j]] = bad[[j, 0]]
    assert bad[0, 0] > bad[1, 0]
    with pytest.raises(api.RalaB200Error, match="ascending pile id"):
        G.set_hills(bad)
    G.set_piles(inp.piles, inp.flags).set_hills(None).set_overlaps(inp.records)
    G.classify()
    assert G.hill_coverage().shape == (0,)
    # the flags of the first pass passed again with a later table (or left out): the same result as the oracle's
    P = O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills).classify()
    piles, _ = PileDriver(inp.hills, inp.flags, inp.seed).hill_step(P.hill_cov, P.piles)
    P.set_piles(piles).retrim()
    while P.retrim_promote():
        pass
    P.final_containment().build_edges()
    for flags in (inp.flags, None):
        G.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_overlaps(inp.records)
        G.classify()
        assert_same(G.hill_coverage(), O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills).classify().hill_cov, "coverage")
        G.set_piles(piles, flags).retrim()
        while G.retrim_promote():
            pass
        G.finalize()
        _same_lists(G, P, f"final, flags {'again' if flags is not None else 'left out'}")
        G.build()
        assert_same(G.edges(), P.edges, "edges")
    G.close()
