"""MHAP text -> records (SURVEY.md 8(f) row 2, record mapping of 8(a) row a1): the plain-C reader (tests/mhap_oracle.c)
plus the oracle's duplicate filter against the reference's records in tests/golden, and against a Python restatement of
the contract on an adversarial corpus; on the GPU (-m gpu) the device reader (rala_b200_parse_mhap,
rala_b200_graph_set_overlaps_mhap) against both, down to the reference's piles and transitive marks."""
import os
import re
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth
from tests import datasets
from tests import mhap_oracle as M

TOP = np.uint32(0x80000000)


def text_of(d, fmt: str) -> bytes:
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "o." + fmt)
        getattr(d, "write_" + fmt)(path)
        with open(path, "rb") as f:
            return f.read()


def read_names(n: int):
    return [b"r%d" % i for i in range(n)]


def golden_anchor(name: str):
    g = datasets.load_golden(name)
    return text_of(datasets.make(name), "mhap"), g["in.read_len"], datasets.Stages(g)


def records_from(cols):
    """Parsed columns + the oracle's duplicate filter -> rala_ovl_t rows as the reference's front end dumps them."""
    valid = O.filter_duplicates(cols[0], cols[1], cols[6]).astype(bool)
    rec = np.zeros((cols.shape[1], 7), np.uint32)
    rec[:, 0] = cols[0]
    rec[:, 1] = cols[1] & ~TOP
    rec[:, 2:6] = cols[2:6].T
    rec[:, 6] = (cols[1] >> 31) | np.where(valid, 0, 2).astype(np.uint32)
    return rec


def query_rc(text: bytes) -> int:
    """a_rc = 1 records, counted with numpy on the raw fields."""
    lines = [ln for ln in text.split(b"\n") if ln]
    return int(np.count_nonzero(np.array([ln.split(b" ")[4] for ln in lines]) == b"1"))


# ---- adversarial corpus ---------------------------------------------------------------------------------------------
def corpus(seed: int, n_lines: int = 300):
    rng = np.random.Generator(np.random.PCG64(seed))
    n_reads = 120
    read_len = rng.integers(1000, 60000, n_reads).astype(np.uint32)
    big = int(rng.integers(0, n_lines))
    lines = []
    for i in range(n_lines):
        ia, ib = (int(x) for x in rng.integers(0, n_reads, 2))
        ia = 0 if i % 40 == 3 else ia                               # id 1
        ib = n_reads - 1 if i % 40 == 4 else ib                     # id n_reads
        la, lb = int(read_len[ia]), int(read_len[ib])
        if rng.random() < 0.03:
            lb += 1                                                 # a read length the reads contradict
        num = lambda v: (b"0" * int(rng.integers(1, 4)) if rng.random() < 0.1 else b"") + b"%d" % v   # noqa: E731
        a_rc, b_rc = (int(x) for x in rng.integers(0, 2, 2))
        ab, ae = (int(x) for x in rng.integers(0, la, 2))           # about half inverted: the span wraps mod 2^32
        bb, be = (int(x) for x in rng.integers(0, lb, 2))
        err = b"" if rng.random() < 0.1 else b"0.%d" % int(rng.integers(0, 999))
        mm = b"" if rng.random() < 0.1 else b"%d" % int(rng.integers(0, 9999))
        f = [num(ia + 1), num(ib + 1), err, mm, b"%d" % a_rc, num(ab), num(ae), num(la), b"%d" % b_rc, num(bb), num(be), num(lb)]
        if rng.random() > 0.3:
            f += [b"x%d" % k for k in range(int(rng.integers(1, 21)))]
        if i == big:
            f.append(b"y" * 100_000)                                # a 100 KB trailing field
        line = b" ".join(f)
        if rng.random() < 0.2:
            line += b"\r"                                           # CRLF
        lines.append(line)
    text = b"\n".join(lines) + (b"\n" if seed % 2 == 0 else b"")
    return text, read_len


def refusals(text: bytes, n_reads: int):
    """(text, line, kind, field) for every refusal of the contract, each placed on a different line."""
    lines = text.rstrip(b"\n").split(b"\n")
    out = []

    def with_field(k, f, value):
        g = lines[k - 1].split(b" ")
        g[f - 1] = value
        return b"\n".join(lines[:k - 1] + [b" ".join(g)] + lines[k:]) + b"\n"

    cut = lines[:]
    cut[6] = b" ".join(cut[6].split(b" ")[:11])
    out.append((b"\n".join(cut) + b"\n", 7, "fields", 11))
    out.append((b"\n".join(lines[:30] + [b""] + lines[30:]) + b"\n", 31, "empty", 1))
    out.append((with_field(55, 7, b"4294967296"), 55, "overflow", 7))
    out.append((with_field(120, 8, lines[119].split(b" ")[7] + b"x"), 120, "digit", 8))
    out.append((with_field(60, 1, b"0"), 60, "read id", 1))
    out.append((with_field(70, 2, b"%d" % (n_reads + 1)), 70, "read id", 2))
    out.append((with_field(80, 9, b"2"), 80, "strand", 9))
    out.append((with_field(90, 6, b" " + lines[89].split(b" ")[5]), 90, "digit", 6))   # a double space before field 6
    # within a line the smallest field wins; of two lines, the smaller one
    g = lines[99].split(b" ")
    g[8], g[1] = b"2", b"0"
    out.append((b"\n".join(lines[:99] + [b" ".join(g)] + lines[100:]) + b"\n", 100, "read id", 2))
    two = lines[:]
    g = two[199].split(b" ")
    g[4] = b"-"
    two[199] = b" ".join(g)
    two[249] = b"x y"
    out.append((b"\n".join(two), 200, "strand", 5))
    return out


@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_c_reader_plus_filter_give_the_reference_records(name):
    text, rl, st = golden_anchor(name)
    cols, stats = M.parse(text, rl)
    assert stats["n_records"] == st.records.shape[0] and stats["n_length_mismatch"] == 0 and stats["n_query_rc"] == 0
    assert np.array_equal(records_from(cols), st.records)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_c_reader_matches_the_restated_contract(seed):
    text, rl = corpus(seed)
    cols, stats = M.parse(text, rl)
    want, wstats = M.restate(text, rl)
    assert np.array_equal(cols, want) and stats == wstats
    assert stats["n_length_mismatch"] > 0 and 0 < stats["n_query_rc"] == query_rc(text) < stats["n_records"]
    assert {0, len(rl) - 1} <= set((cols[0]).tolist()) | set((cols[1] & ~TOP).tolist())
    assert (cols[3] < cols[2]).any() and (cols[6] > 2**31).any(), "inverted spans"
    lines = text.split(b"\n")
    assert any(ln.endswith(b"\r") and ln.count(b" ") == 11 for ln in lines), "CRLF on a 12-field line"
    assert len(set((cols[1] >> 31).tolist())) == 2


def test_c_reader_refuses_like_the_restated_contract():
    text, rl = corpus(4)
    for bad, line, kind, field in refusals(text, len(rl)):
        for fn in (M.parse, M.restate):
            with pytest.raises(M.MhapRefused) as e:
                fn(bad, rl)
            assert (e.value.line, e.value.kind, e.value.field) == (line, kind, field), fn


# ---- GPU ------------------------------------------------------------------------------------------------------------
def refused_line(err) -> int:
    return int(re.search(r"MHAP line (\d+)", str(err)).group(1))


def names_field(kind, field) -> str:
    return f"has {field} space-separated fields" if kind == "fields" else f"field {field}:"


@pytest.mark.gpu
def test_device_parse_matches_the_c_reader(ctx):
    for name in datasets.GOLDEN:
        text, rl, st = golden_anchor(name)
        want, wstats = M.parse(text, rl)
        got, stats, ms = ctx.parse_mhap(text, rl, with_time=True)
        assert np.array_equal(got, want) and {k: stats[k] for k in wstats} == wstats, name
        assert ms > 0 and stats["n_bytes"] == len(text) and stats["n_chunks"] == 1
    for seed in (1, 2, 3):
        text, rl = corpus(seed)
        want, wstats = M.parse(text, rl)
        got, stats = ctx.parse_mhap(np.frombuffer(text, np.uint8), rl)
        assert np.array_equal(got, want) and {k: stats[k] for k in wstats} == wstats, seed
        assert stats["n_query_rc"] == query_rc(text)
    empty, stats = ctx.parse_mhap(b"", rl)
    assert empty.shape == (7, 0) and stats["n_records"] == 0
    # nothing but the shortest valid lines (22 bytes): the record buffers are exactly full
    tight = b"\n".join([b"1 2   0 0 5 5 1 0 5 5"] * 100_000)
    got, stats = ctx.parse_mhap(tight, [5, 5])
    want, _ = M.parse(tight, [5, 5])
    assert stats["n_records"] == 100_000 and np.array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_session_from_mhap_classifies_like_the_reference_records(ctx, name):
    text, rl, st = golden_anchor(name)
    ref = api.Graph(ctx)
    ref.set_piles(st.piles, st.pflags).set_hills(st.hills).set_overlaps(st.records).classify()
    G = api.Graph(ctx)
    G.set_reads(read_names(len(rl)), rl)
    stats = G.set_overlaps_mhap(text)
    assert stats["n_records"] == st.records.shape[0] and stats["n_length_mismatch"] == 0
    G.set_piles(st.piles, st.pflags).set_hills(st.hills).classify()
    for got, want in zip(G.lists(), ref.lists()):
        assert np.array_equal(got, want)
    assert np.array_equal(G.hill_coverage(), ref.hill_coverage()) and np.array_equal(G.piles(), ref.piles())
    G.close()
    ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_mhap_text_to_device_piles_to_transitive_marks(ctx, name):
    text, rl, st = golden_anchor(name)
    G = api.Graph(ctx)
    G.set_reads(read_names(len(rl)), rl).set_overlaps_mhap(text)
    G.build_piles()                                                 # no pile table from the host
    assert np.array_equal(G.piles(), st.piles) and np.array_equal(G.medians(), st.medians)
    G.set_hills(None).run()
    c = G.counts()
    assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes
    assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed)
    G.close()


@pytest.mark.gpu
def test_coverage_runs_equal_those_of_the_paf_session(ctx):
    d = datasets.make("g_noisy")
    names = read_names(d.read_len.shape[0])
    runs = []
    for fmt in ("paf", "mhap"):
        G = api.Graph(ctx)
        G.set_reads(names, d.read_len)
        getattr(G, "set_overlaps_" + fmt)(text_of(d, fmt))
        G.build_piles()
        runs.append(G.coverage_runs())
        G.close()
    for got, want in zip(*runs):
        assert np.array_equal(got, want)


@pytest.mark.gpu
def test_text_of_several_chunks_with_lines_across_every_cut(ctx):
    import torch
    block, rl, _ = golden_anchor("g_clean")
    assert api.PAF_CHUNK_BYTES % len(block)
    text = block * (2 * api.PAF_CHUNK_BYTES // len(block) + 3)
    want, wstats = M.parse(text, rl)
    got, stats = ctx.parse_mhap(text, rl)
    assert stats["n_chunks"] >= 3 and np.array_equal(got, want) and stats["n_records"] == wstats["n_records"]
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()   # uploaded in place
    got2, stats2 = ctx.parse_mhap(pinned, rl)
    assert np.array_equal(got2, want) and stats2 == stats
    # the session: a fixed number of kernels per call and per chunk
    G = api.Graph(ctx)
    G.set_reads(read_names(len(rl)), rl)
    per_call = []
    for t in (block, text):
        before = ctx.launch_count
        s = G.set_overlaps_mhap(t)
        per_call.append((ctx.launch_count - before, s["n_chunks"]))
    (l1, c1), (l2, c2) = per_call
    assert c1 == 1 and c2 == stats["n_chunks"] and l1 == 2 + 2 * c1 and l2 == 2 + 2 * c2, per_call
    G.close()


@pytest.mark.gpu
def test_refusals_name_the_line_and_field_and_leave_the_session_usable(ctx):
    text, rl, st = golden_anchor("g_clean")
    names = read_names(len(rl))
    G = api.Graph(ctx)
    with pytest.raises(api.RalaB200Error, match="set_reads") as e:
        G.set_overlaps_mhap(text)
    assert "status -3" in str(e.value)
    G.set_reads(names, rl)
    for bad, line, kind, field in refusals(text, len(rl)):
        with pytest.raises(api.RalaB200Error) as e:
            ctx.parse_mhap(bad, rl)
        assert refused_line(e.value) == line and names_field(kind, field) in str(e.value), (kind, e.value)
        with pytest.raises(api.RalaB200Error) as e:
            G.set_overlaps_mhap(bad)
        assert refused_line(e.value) == line and names_field(kind, field) in str(e.value), (kind, e.value)
        with pytest.raises(api.RalaB200Error, match="set_overlaps"):
            G.set_piles(st.piles, st.pflags).classify()                 # the session holds no records
        assert G.set_overlaps_mhap(text)["n_records"] == st.records.shape[0]   # a good call works
    # a record that stays valid after the duplicate filter with a b_length the reads contradict
    lines = text.split(b"\n")
    k = int(np.nonzero((st.records[:, 6] & 2) == 0)[0][100])
    f = lines[k].split(b" ")
    f[11] = b"%d" % (int(f[11]) + 1)
    lines[k] = b" ".join(f)
    wrong = b"\n".join(lines)
    _, stats = ctx.parse_mhap(wrong, rl)
    assert stats["n_length_mismatch"] == 1 and stats["first_length_mismatch"] == k
    with pytest.raises(api.RalaB200Error, match="read length") as e:
        G.set_overlaps_mhap(wrong)
    assert refused_line(e.value) == k + 1
    with pytest.raises(api.RalaB200Error, match="set_overlaps"):
        G.set_piles(st.piles, st.pflags).classify()
    # a self overlap: build_piles names its MHAP line
    lines = text.split(b"\n")
    f = lines[40].split(b" ")
    f[1], f[11] = f[0], f[7]
    lines[40] = b" ".join(f)
    G.set_overlaps_mhap(b"\n".join(lines))
    with pytest.raises(api.RalaB200Error, match="MHAP line 41 ") as e:
        G.build_piles()
    assert "self overlap" in str(e.value)
    G.set_overlaps_mhap(text)
    G.build_piles()
    G.set_hills(None).run()
    assert G.counts()["n_transitive_pairs"] == st.n_pairs
    G.close()


@pytest.mark.gpu
def test_one_session_alternating_paf_and_mhap_text(ctx):
    d = datasets.make("g_clean")
    texts = {fmt: text_of(d, fmt) for fmt in ("paf", "mhap")}
    G = api.Graph(ctx)
    G.set_reads(read_names(d.read_len.shape[0]), d.read_len)
    results = []
    for fmt in ("paf", "mhap", "paf"):
        getattr(G, "set_overlaps_" + fmt)(texts[fmt])
        G.build_piles()
        G.set_hills(None).run()
        results.append((G.edges(), G.marked(), G.piles(), G.medians()))
    for other in results[1:]:
        for got, want in zip(other, results[0]):
            assert np.array_equal(got, want)
    assert results[0][0].shape[0] > 0
    G.close()
