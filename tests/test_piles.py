"""The pile table from the overlap records (Graph::initialize's coverage half, SURVEY.md 8(f) row 1 second half): the plain-C
restatement (tests/piles_oracle.c) pinned to the begin, end and median of every golden pile the reference's own initialize()
left in tests/golden, its unpinned boundary choices fixed by hand-built cases; on the GPU (-m gpu) the device build
(rala_b200_build_piles, rala_b200_graph_build_piles) against it, and PAF text -> device piles -> transitive marks."""
import numpy as np
import pytest

from rala_b200 import api, synth
from tests import datasets
from tests import piles_oracle as PO
from tests.test_paf_reader import golden_anchor

TOP = np.uint32(0x80000000)


def golden_columns(name):
    st = datasets.Stages(datasets.load_golden(name))
    return st, PO.columns(st.records)


def rule(cols, read_len):
    """The rule of include/rala_b200.h in numpy, read by read: (piles, medians)."""
    piles = np.zeros((len(read_len), 2), np.uint32)
    med = np.zeros(len(read_len), np.uint16)
    for r in range(len(read_len)):
        cov = PO.coverage(cols, read_len, r)
        hi = np.concatenate([[False], cov >= 4, [False]]).astype(np.int8)
        d = np.diff(hi)
        starts, ends = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
        if starts.size:
            k = int(np.argmax(ends - starts))          # the first longest
            if ends[k] - starts[k] >= 1260:
                piles[r] = starts[k], ends[k]
                med[r] = np.sort(cov[starts[k]:ends[k]])[(ends[k] - starts[k]) // 2]
    return piles, med


class Hand:
    """Hand-built records: coverage on read 0 from intervals, partners are reads 1.. (each far too thin to live)."""

    def __init__(self, len0=10000, n_partners=64, partner_len=60000):
        self.read_len = np.array([len0] + [partner_len] * n_partners, np.uint32)
        self.rows = []
        self.next = 1

    def cover(self, lo, hi, times=1):
        """`times` records that add [lo, hi) to read 0."""
        for _ in range(times):
            p = self.next
            self.next = self.next % (len(self.read_len) - 1) + 1
            self.rows.append([0, p, lo - 15, hi + 15, 100 * (p % 100), 100 * (p % 100) + hi - lo + 30])
        return self

    def cols(self):
        return np.asarray(self.rows, np.uint32).reshape(-1, 6).T.copy()


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_oracle_reproduces_the_reference_piles(name):
    st, cols = golden_columns(name)
    o = PO.build_piles(cols, st.read_len)
    assert np.array_equal(o["piles"], st.piles), "begin / end"
    assert np.array_equal(o["medians"], st.medians), "median"
    assert o["stats"]["n_counted"] == int((st.records[:, 0] != 0xFFFFFFFF).sum())
    for r in (0, 7, len(st.read_len) - 1):
        assert np.array_equal(PO.expand_runs(*o["runs"], st.read_len, r), PO.coverage(cols, st.read_len, r))


def test_coverage_counts_the_records_the_duplicate_filter_drops():
    st, cols = golden_columns("g_noisy")
    filtered = cols.copy()
    filtered[0] |= np.where((st.records[:, 6] & 2) != 0, TOP, np.uint32(0))
    o = PO.build_piles(filtered, st.read_len, runs=False)
    assert np.array_equal(o["piles"], st.piles)                  # begin and end do not tell the two rules apart ...
    assert int((o["medians"] != st.medians).sum()) > 50          # ... the medians do


def test_hand_built_boundaries():
    # two regions of 1 500 with coverage 4: the first one wins, and the stats say a tie decided it
    h = Hand().cover(100, 1600, 4).cover(3000, 4500, 4)
    o = PO.build_piles(h.cols(), h.read_len)
    assert tuple(o["piles"][0]) == (100, 1600) and o["medians"][0] == 4 and o["stats"]["n_tied"] == 1
    # 1 259 dies, 1 260 lives
    for length, alive in ((1259, False), (1260, True)):
        h = Hand().cover(500, 500 + length, 5)
        o = PO.build_piles(h.cols(), h.read_len)
        assert tuple(o["piles"][0]) == ((500, 500 + length) if alive else (0, 0)) and o["medians"][0] == (5 if alive else 0)
        assert o["stats"]["n_exact_min"] == int(alive) and o["stats"]["n_live"] == int(alive)
    # a dip below 4 for one base splits the region; the longer half wins
    h = Hand().cover(100, 3000, 3).cover(100, 1000).cover(1001, 3000).cover(2000, 2500, 2)
    o = PO.build_piles(h.cols(), h.read_len)
    assert tuple(o["piles"][0]) == (1001, 3000) and o["medians"][0] == 4
    off, rb, rc = o["runs"]
    assert list(rb[off[0]:off[1]]) == [0, 100, 1000, 1001, 2000, 2500, 3000]
    assert list(rc[off[0]:off[1]]) == [0, 4, 3, 4, 6, 4, 0]
    # a read no record touches: dead, one run of coverage 0
    h = Hand(n_partners=2).cover(100, 2000, 4)
    h.read_len = np.append(h.read_len, 5000).astype(np.uint32)
    o = PO.build_piles(h.cols(), h.read_len)
    off, rb, rc = o["runs"]
    assert tuple(o["piles"][-1]) == (0, 0) and o["medians"][-1] == 0
    assert list(rb[off[-2]:off[-1]]) == [0] and list(rc[off[-2]:off[-1]]) == [0]
    for h in (Hand().cover(100, 1600, 4).cover(3000, 4500, 4), Hand().cover(100, 3000, 3).cover(100, 1000).cover(1001, 3000)):
        p, m = rule(h.cols(), h.read_len)
        o = PO.build_piles(h.cols(), h.read_len)
        assert np.array_equal(o["piles"], p) and np.array_equal(o["medians"], m)


def refusal_cases():
    """(cols, read_len, record, kind): one refusal each, the offending record at index 5 behind a second one at 9."""
    out = []
    base = Hand().cover(100, 3000, 12)
    for kind, col, value in (("self", 1, 0), ("a_empty", 3, 100 - 15 + 30), ("a_empty", 3, 10), ("a_beyond", 3, 10001),
                             ("b_empty", 5, 600 - 15 + 15), ("b_beyond", 5, 60001), ("id", 1, 65)):
        cols = base.cols()
        for k in (9, 5):
            cols[col, k] = value
            if kind == "b_empty":
                cols[4, k] = 600 - 15
        out.append((cols, base.read_len, 5, kind))
    return out


def test_oracle_refusals():
    for cols, rl, rec, kind in refusal_cases():
        with pytest.raises(PO.Refused) as e:
            PO.build_piles(cols, rl)
        assert (e.value.record, e.value.kind) == (rec, kind), kind
    h = Hand(n_partners=60000, partner_len=20000).cover(100, 2000, 65536)
    with pytest.raises(PO.CoverageLimit):
        PO.build_piles(h.cols(), h.read_len)
    cols = Hand().cover(100, 2000, 4).cols()
    cols[0, 2] |= TOP   # an unresolved record is skipped, whatever it holds
    cols[3, 2] = 0
    PO.build_piles(cols, Hand().read_len)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def check_device(ctx, cols, read_len):
    o = PO.build_piles(cols, read_len, runs=False)
    piles, med, stats = ctx.build_piles(cols, read_len)
    assert np.array_equal(piles, o["piles"]) and np.array_equal(med, o["medians"]) and stats == o["stats"], stats
    return stats


@pytest.mark.gpu
def test_device_equals_the_oracle_on_goldens_synthetic_and_hand_built_sets(ctx):
    for name in datasets.GOLDEN:
        st, cols = golden_columns(name)
        check_device(ctx, cols, st.read_len)
        piles, med, _ = ctx.build_piles(cols, st.read_len)
        assert np.array_equal(piles, st.piles) and np.array_equal(med, st.medians), name
    sets = [synth.generate(genome_len=600_000, coverage=40, read_len=8000, len_sd=2500, seed=21, min_ovl=1000, noise=30),
            synth.generate(genome_len=300_000, coverage=30, read_len=10000, seed=22, min_ovl=1000, dual=True),
            synth.generate(genome_len=600_000, coverage=45, read_len=10000, len_sd=3000, seed=23, min_ovl=1000, noise=30,
                           chimera_frac=0.05, adapter_frac=0.08, repeats=(1, 8, 4000))]
    for d in sets:
        cols = PO.columns(d.records)
        cols[0, ::97] |= TOP                                        # a sprinkle of unresolved records
        check_device(ctx, cols, d.read_len)
    for h in (Hand().cover(100, 1600, 4).cover(3000, 4500, 4), Hand().cover(500, 1759, 5), Hand().cover(500, 1760, 5),
              Hand().cover(100, 3000, 3).cover(100, 1000).cover(1001, 3000).cover(2000, 2500, 2)):
        check_device(ctx, h.cols(), h.read_len)
    piles, med, stats = ctx.build_piles([np.zeros(0, np.uint32)] * 6, np.array([0, 7, 5000], np.uint32))
    assert not piles.any() and not med.any() and stats["n_runs"] == 2


@pytest.mark.gpu
def test_device_on_repeat_hubs_and_a_large_set(ctx):
    hubs = synth.generate_repeat_hubs(genome_len=2_000_000, n_hubs=4, spokes=2601)
    s = check_device(ctx, PO.columns(hubs.records), hubs.read_len)
    assert s["max_coverage"] >= 1000, s
    big = synth.generate(genome_len=12_000_000, coverage=40, read_len=10000, len_sd=3000, seed=24, min_ovl=1000)
    cols = PO.columns(big.records)
    s = check_device(ctx, cols, big.read_len)
    assert cols.shape[1] * 4 > 100 * 2048, "events span many sort tiles"


@pytest.mark.gpu
def test_device_refusals_name_the_first_record(ctx):
    for cols, rl, rec, kind in refusal_cases():
        with pytest.raises(api.RalaB200Error) as e:
            ctx.build_piles(cols, rl)
        assert f"record {rec} " in str(e.value) and "status -2" in str(e.value), (kind, e.value)
    h = Hand(n_partners=60000, partner_len=20000).cover(100, 2000, 65536)
    with pytest.raises(api.RalaB200Error, match="65536") as e:
        ctx.build_piles(h.cols(), h.read_len)
    assert "status -5" in str(e.value)


def session(ctx, name):
    text, names, rl, st = golden_anchor(name)
    G = api.Graph(ctx)
    G.set_reads(names, rl).set_overlaps_paf(text)
    return G, text, names, rl, st


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_paf_text_to_device_piles_to_transitive_marks(ctx, name):
    G, text, names, rl, st = session(ctx, name)
    stats = G.build_piles()                                         # no pile table from the host
    assert stats["n_live"] == len(rl)
    assert np.array_equal(G.piles(), st.piles) and np.array_equal(G.medians(), st.medians)
    G.set_hills(None).run()
    c = G.counts()
    assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes
    assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed)
    G.close()


@pytest.mark.gpu
def test_coverage_runs_expand_to_the_oracle_coverage(ctx):
    G, text, names, rl, st = session(ctx, "g_noisy")
    stats = G.build_piles()
    off, rb, rc = G.coverage_runs()
    o = PO.build_piles(PO.columns(st.records), rl)
    assert stats["n_runs"] == int(off[-1]) == o["stats"]["n_runs"]
    for got, want in zip((off, rb, rc), o["runs"]):
        assert np.array_equal(got, want)
    cols = PO.columns(st.records)
    for r in (0, 1, 999, len(rl) - 1):
        assert np.array_equal(PO.expand_runs(off, rb, rc, rl, r), PO.coverage(cols, rl, r))
    G.close()


@pytest.mark.gpu
def test_noisy_golden_with_device_piles_and_golden_flags_and_hills(ctx):
    G, text, names, rl, st = session(ctx, "g_noisy")
    G.build_piles()
    ref = api.Graph(ctx)
    ref.set_piles(st.piles, st.pflags).set_hills(st.hills).set_overlaps(st.records).classify()
    G.set_piles(G.piles(), st.pflags).set_hills(st.hills).classify()
    for got, want in zip(G.lists(), ref.lists()):
        assert np.array_equal(got, want)
    assert np.array_equal(G.hill_coverage(), st.hill_cov)
    G.close()
    ref.close()


@pytest.mark.gpu
def test_refused_build_leaves_the_session_usable_and_order_is_checked(ctx):
    G, text, names, rl, st = session(ctx, "g_clean")
    lines = text.split(b"\n")
    f = lines[40].split(b"\t")
    f[5] = f[0]                                                     # a self overlap on line 41
    f[6] = f[1]
    lines[40] = b"\t".join(f)
    G.set_overlaps_paf(b"\n".join(lines))
    G.set_piles(st.piles)
    with pytest.raises(api.RalaB200Error, match="PAF line 41 ") as e:
        G.build_piles()
    assert "self overlap" in str(e.value)
    assert np.array_equal(G.piles(), st.piles)                      # the table set before is still there
    G.set_overlaps_paf(text)
    G.build_piles()
    G.run()
    assert G.counts()["n_transitive_pairs"] == st.n_pairs
    G.set_overlaps_columns(api.records_to_columns(st.records))
    with pytest.raises(api.RalaB200Error, match="status -3"):
        G.build_piles()
    G.set_overlaps_paf(text)
    G.set_reads(names, rl)
    with pytest.raises(api.RalaB200Error, match="status -3"):
        G.build_piles()
    G.close()
    H = api.Graph(ctx)
    with pytest.raises(api.RalaB200Error, match="status -3"):
        H.medians()
    H.close()
