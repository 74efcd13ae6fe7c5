"""PAF text -> records (SURVEY.md 8(f) row 2): the plain-C reader (tests/paf_oracle.c) pinned to what the reference's own
PafParser + name_to_id_ + duplicate filter left in tests/golden, checked against a Python restatement of the contract on
an adversarial corpus; on the GPU (-m gpu) the device reader (rala_b200_parse_paf, rala_b200_graph_set_overlaps_paf)
against both, down to the reference's transitive marks."""
import os
import re
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth
from tests import datasets
from tests import paf_oracle as P

TOP = np.uint32(0x80000000)


def paf_text(d) -> bytes:
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "o.paf")
        d.write_paf(path)
        with open(path, "rb") as f:
            return f.read()


def read_names(n: int):
    return [b"r%d" % i for i in range(n)]


def dups_anchor():
    d = synth.generate_duplicate_groups(big_groups=1, big_size=1500)   # the seed tests/golden/make_golden.py used
    return paf_text(d), read_names(d.read_len.shape[0]), d.read_len, np.load(os.path.join(datasets.GOLDEN_DIR, "dups.npz"))


def golden_anchor(name: str):
    g = datasets.load_golden(name)
    return paf_text(datasets.make(name)), read_names(g["in.read_len"].shape[0]), g["in.read_len"], datasets.Stages(g)


def records_from(cols):
    """Parsed columns + the oracle's duplicate filter -> rala_ovl_t rows as the reference's front end dumps them."""
    valid = O.filter_duplicates(cols[0], cols[1], cols[6]).astype(bool)
    known = (cols[0] & TOP) == 0
    rec = np.zeros((cols.shape[1], 7), np.uint32)
    rec[:, 0] = np.where(known, cols[0], 0xFFFFFFFF)
    rec[:, 1] = np.where(known, cols[1] & ~TOP, 0xFFFFFFFF)
    rec[:, 2:6] = cols[2:6].T
    rec[:, 6] = (cols[1] >> 31) | np.where(valid, 0, 2).astype(np.uint32)
    return rec


def check_dups(cols, stats, z):
    known = (z["a"] & TOP) == 0
    assert np.array_equal((cols[0] & TOP) == 0, known), "unresolved set"
    assert np.array_equal(cols[0][known], z["a"][known]) and np.array_equal((cols[1] & ~TOP)[known], z["b"][known])
    assert np.array_equal(cols[6], z["length"])
    assert stats["n_unresolved"] == int((~known).sum()) and stats["n_length_mismatch"] == 0
    assert np.array_equal(O.filter_duplicates(cols[0], cols[1], cols[6]), z["valid"])


def check_golden(cols, stats, st):
    assert stats["n_records"] == st.records.shape[0] and stats["n_length_mismatch"] == 0
    got, want = records_from(cols), st.records
    assert np.array_equal(got[:, 2:7], want[:, 2:7]), "coordinates / orientation / invalid bit"
    known = want[:, 0] != 0xFFFFFFFF
    assert np.array_equal(got[known, :2], want[known, :2]), "ids"


# ---- adversarial corpus ---------------------------------------------------------------------------------------------
def corpus(seed: int, n_lines: int = 300):
    rng = np.random.Generator(np.random.PCG64(seed))
    names = read_names(40)                                     # r1 is a prefix of r10 .. r19
    while len(names) < 120:
        nm = bytes(rng.integers(33, 127, int(rng.integers(1, 301)), dtype=np.uint8))
        if nm not in names:
            names.append(nm)
    read_len = rng.integers(1000, 60000, len(names)).astype(np.uint32)
    unknown = [b"r40", b"r1x", b"ghost", names[50][:-1] or b"?", names[60] + b"z"]
    big = int(rng.integers(0, n_lines))
    lines = []
    for i in range(n_lines):
        ia, ib = rng.integers(0, len(names), 2)
        a = names[ia] if rng.random() > 0.05 else unknown[int(rng.integers(0, len(unknown)))]
        b = names[ib] if rng.random() > 0.05 else unknown[int(rng.integers(0, len(unknown)))]
        la, lb = int(read_len[ia]), int(read_len[ib])
        if rng.random() < 0.03:
            la += 1                                            # a read length the reads contradict
        num = lambda v: (b"0" * int(rng.integers(1, 4)) if rng.random() < 0.1 else b"") + b"%d" % v   # noqa: E731
        length = 4294967295 if rng.random() < 0.05 else int(rng.integers(0, 2**32))
        f = [a, num(la), num(int(rng.integers(0, la))), num(int(rng.integers(0, la))),
             [b"+", b"-", b"*", b"", b"+-", b"-+"][int(rng.integers(0, 6))], b, num(lb), num(int(rng.integers(0, lb))),
             num(int(rng.integers(0, lb))), b"%d" % int(rng.integers(0, 99999)), num(length), b"255"]
        f += [b"tg:i:%d" % k for k in range(int(rng.integers(0, 21)))]
        if i == big:
            f.append(b"cg:Z:" + b"10M" * 34000)             # a 100 KB tag
        line = b"\t".join(f)
        if rng.random() < 0.2:
            line += b"\r"                                      # CRLF
        lines.append(line)
    text = b"\n".join(lines) + (b"\n" if seed % 2 == 0 else b"")
    return text, names, read_len


def refusals(text: bytes):
    """(text, line, kind, column) for every refusal of the contract, each placed on a different line."""
    lines = text.rstrip(b"\n").split(b"\n")
    out = []
    k = 7
    cut = lines[:]
    cut[k - 1] = b"\t".join(cut[k - 1].split(b"\t")[:11])
    out.append((b"\n".join(cut) + b"\n", k, "fields", 11))
    k = 31
    out.append((b"\n".join(lines[:k - 1] + [b""] + lines[k - 1:]) + b"\n", k, "empty", 1))
    k = 55
    f = lines[k - 1].split(b"\t")
    f[10] = b"4294967296"
    out.append((b"\n".join(lines[:k - 1] + [b"\t".join(f)] + lines[k:]) + b"\n", k, "overflow", 11))
    k = 120
    f = lines[k - 1].split(b"\t")
    f[7] = f[7] + b"x"
    out.append((b"\n".join(lines[:k - 1] + [b"\t".join(f)] + lines[k:]) + b"\n", k, "digit", 8))
    # the smallest offending line wins
    f = lines[199].split(b"\t")
    f[1] = b"abc"
    two = lines[:]
    two[199] = b"\t".join(f)
    two[249] = b"x\ty"
    out.append((b"\n".join(two), 200, "digit", 2))
    return out


def test_c_reader_matches_the_reference_dups_golden():
    text, names, rl, z = dups_anchor()
    cols, stats = P.parse(text, names, rl)
    check_dups(cols, stats, z)


@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_c_reader_plus_filter_give_the_reference_records(name):
    text, names, rl, st = golden_anchor(name)
    cols, stats = P.parse(text, names, rl)
    check_golden(cols, stats, st)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_c_reader_matches_the_restated_contract(seed):
    text, names, rl = corpus(seed)
    cols, stats = P.parse(text, names, rl)
    want, wstats = P.restate(text, names, rl)
    assert np.array_equal(cols, want) and stats == wstats
    assert 0 < stats["n_unresolved"] < stats["n_records"] and stats["n_length_mismatch"] > 0
    assert (cols[6] == 0xFFFFFFFF).any() and len(set((cols[1] >> 31).tolist())) == 2


def test_c_reader_refuses_like_the_restated_contract():
    text, names, rl = corpus(4)
    for bad, line, kind, col in refusals(text):
        for fn in (P.parse, P.restate):
            with pytest.raises(P.PafRefused) as e:
                fn(bad, names, rl)
            assert (e.value.line, e.value.kind, e.value.column) == (line, kind, col), fn
    with pytest.raises(P.DuplicateName):
        P.parse(text, names + [names[3]], np.append(rl, 5))


# ---- GPU ------------------------------------------------------------------------------------------------------------
def refused_line(err) -> int:
    return int(re.search(r"line (\d+)", str(err)).group(1))


@pytest.mark.gpu
def test_device_parse_matches_the_c_reader(ctx):
    text, names, rl, z = dups_anchor()
    cols, stats, ms = ctx.parse_paf(text, names, rl, with_time=True)
    check_dups(cols, stats, z)
    assert ms > 0 and stats["n_bytes"] == len(text) and stats["n_chunks"] == 1
    text, names, rl, st = golden_anchor("g_noisy")
    cols, stats = ctx.parse_paf(np.frombuffer(text, np.uint8), names, rl)
    check_golden(cols, stats, st)
    for seed in (1, 2, 3):
        text, names, rl = corpus(seed)
        want, wstats = P.parse(text, names, rl)
        blob = b"".join(names)
        ends = np.cumsum([len(n) for n in names]).astype(np.uint64)
        got, stats = ctx.parse_paf(text, (blob, ends), rl)
        assert np.array_equal(got, want) and {k: stats[k] for k in wstats} == wstats, seed
    empty, stats = ctx.parse_paf(b"", names, rl)
    assert empty.shape == (7, 0) and stats["n_records"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_session_from_paf_classifies_like_the_reference_records(ctx, name):
    text, names, rl, st = golden_anchor(name)
    ref = api.Graph(ctx)
    ref.set_piles(st.piles, st.pflags).set_hills(st.hills).set_overlaps(st.records).classify()
    G = api.Graph(ctx)
    G.set_reads(names, rl)
    stats = G.set_overlaps_paf(text)
    assert stats["n_records"] == st.records.shape[0] and stats["n_unresolved"] == 0
    G.set_piles(st.piles, st.pflags).set_hills(st.hills).classify()
    for got, want in zip(G.lists(), ref.lists()):
        assert np.array_equal(got, want)
    assert np.array_equal(G.hill_coverage(), ref.hill_coverage()) and np.array_equal(G.piles(), ref.piles())
    G.close()
    ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_paf_text_to_transitive_marks_matches_the_reference(ctx, name):
    text, names, rl, st = golden_anchor(name)
    G = api.Graph(ctx)
    G.set_reads(names, rl).set_overlaps_paf(text)
    G.set_piles(st.piles, st.pflags).set_hills(st.hills).run()
    c = G.counts()
    assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes
    assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed)
    G.close()


@pytest.mark.gpu
def test_text_of_several_chunks_with_lines_across_every_cut(ctx):
    import torch
    block, names, rl, _ = golden_anchor("g_clean")
    assert api.PAF_CHUNK_BYTES % len(block)
    text = block * (2 * api.PAF_CHUNK_BYTES // len(block) + 3)
    want, wstats = P.parse(text, names, rl)
    got, stats = ctx.parse_paf(text, names, rl)
    assert stats["n_chunks"] >= 3 and np.array_equal(got, want) and stats["n_records"] == wstats["n_records"]
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()   # uploaded in place
    got2, stats2 = ctx.parse_paf(pinned, names, rl)
    assert np.array_equal(got2, want) and stats2 == stats
    # the session: a fixed number of kernels per call and per chunk
    G = api.Graph(ctx)
    G.set_reads(names, rl)
    per_call = []
    for t in (block, text):
        before = ctx.launch_count
        s = G.set_overlaps_paf(t)
        per_call.append((ctx.launch_count - before, s["n_chunks"]))
    (l1, c1), (l2, c2) = per_call
    assert c1 == 1 and (l2 - l1) == 2 * (c2 - c1) and l1 == 2 + 2 * c1, per_call
    G.close()


@pytest.mark.gpu
def test_refusals_name_the_line_and_leave_the_session_usable(ctx):
    text, names, rl, st = golden_anchor("g_clean")
    G = api.Graph(ctx)
    G.set_reads(names, rl)
    for bad, line, kind, col in refusals(text):
        with pytest.raises(api.RalaB200Error) as e:
            ctx.parse_paf(bad, names, rl)
        assert refused_line(e.value) == line and (kind == "fields" or f"column {col}" in str(e.value)), e.value
        with pytest.raises(api.RalaB200Error) as e:
            G.set_overlaps_paf(bad)
        assert refused_line(e.value) == line, e.value
        with pytest.raises(api.RalaB200Error, match="set_overlaps"):
            G.set_piles(st.piles, st.pflags).classify()                 # the session holds no records
    # a record that stays valid after the duplicate filter with a read length the reads contradict
    lines = text.split(b"\n")
    k = int(np.nonzero((st.records[:, 6] & 2) == 0)[0][100])
    f = lines[k].split(b"\t")
    f[1] = b"%d" % (int(f[1]) + 1)
    lines[k] = b"\t".join(f)
    wrong = b"\n".join(lines)
    _, stats = ctx.parse_paf(wrong, names, rl)
    assert stats["n_length_mismatch"] >= 1 and stats["first_length_mismatch"] <= k
    with pytest.raises(api.RalaB200Error, match="read length") as e:
        G.set_overlaps_paf(wrong)
    assert refused_line(e.value) == k + 1
    # after every refusal a good call on the same session works
    assert G.set_overlaps_paf(text)["n_records"] == st.records.shape[0]
    G.set_piles(st.piles, st.pflags).set_hills(st.hills).run()
    assert G.counts()["n_transitive_pairs"] == st.n_pairs
    with pytest.raises(api.RalaB200Error, match="same name"):
        G.set_reads(names + [names[7]], np.append(rl, 10))
    with pytest.raises(api.RalaB200Error, match="set_reads"):
        G.set_overlaps_paf(text)
    with pytest.raises(api.RalaB200Error, match="same name"):
        ctx.parse_paf(text, [b"r0", b"r1", b"r0"], [1, 2, 3])
    G.close()
