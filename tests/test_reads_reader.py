"""FASTA / FASTQ text -> the session's read names and lengths (rala_b200_graph_set_reads_text): the plain-C reader
(tests/reads_oracle.c) checked against a Python restatement of the contract on an adversarial corpus and against the
lengths of the reference's goldens; on the GPU (-m gpu) the device reader against the C reader, and sequence text plus
overlap text down to the reference's transitive marks with the pile table built on the device."""
import functools
import os
import re
import tempfile

import numpy as np
import pytest

from rala_b200 import api
from tests import datasets
from tests import reads_oracle as R

ACGT = np.frombuffer(b"ACGT", np.uint8)


# ---- text builders --------------------------------------------------------------------------------------------------
def wrap(seq: bytes, width) -> bytes:
    """seq as lines of `width` bytes (None: one line), each ending in '\\n'."""
    if not width or width >= len(seq):
        return seq + b"\n"
    a = np.frombuffer(seq, np.uint8)
    full = len(a) // width * width
    rows = np.concatenate([a[:full].reshape(-1, width), np.full((full // width, 1), 10, np.uint8)], axis=1).tobytes()
    return rows + (a[full:].tobytes() + b"\n" if full < len(a) else b"")


def fastq(names, seqs, quals=None) -> bytes:
    quals = quals or [b"I" * len(s) for s in seqs]
    return b"".join(b"@%s\n%s\n+\n%s\n" % (n, s, q) for n, s, q in zip(names, seqs, quals))


def random_seq(rng, n: int) -> bytes:
    return ACGT[rng.integers(0, 4, n)].tobytes()


def corpus(seed: int, fmt: str) -> bytes:
    """Adversarial but valid text: wrapping widths 1 / 60 / 80 / unwrapped, names of 1 and 300 bytes and names that are
    prefixes of others, descriptions after a space and after a tab, '>' and '@' inside sequence lines, quality lines
    starting with '@' or '+', and (odd seeds) a last line without '\\n'."""
    rng = np.random.Generator(np.random.PCG64(seed))
    names = [b"r%d" % i for i in range(25)] + [b"x", b"N" * 300]         # r1 is a prefix of r10 .. r19
    while len(names) < 60:
        nm = bytes(rng.choice(np.r_[33:127, 128:256], int(rng.integers(1, 40))).astype(np.uint8))
        if nm not in names:
            names.append(nm)
    order = rng.permutation(len(names))
    out = []
    for k, i in enumerate(order):
        n = int(rng.integers(1, 400)) if k % 7 else int(rng.integers(3000, 9000))
        seq = bytearray(rng.integers(0x21, 0x7F, n).astype(np.uint8).tobytes())   # any base byte, '>' '@' '+' included
        head = names[i]
        if k % 3 == 1:
            head += b" " + bytes(rng.integers(0x20, 0x7F, int(rng.integers(0, 30))).astype(np.uint8))
        elif k % 3 == 2:
            head += b"\t" + b"len=%d\tx y" % n
        if fmt == "fasta":
            width = [1, 60, 80, None][k % 4] if n < 400 or k % 4 else 80
            if k % 5 == 0:
                seq[len(seq) // 2] = ord(">")
            for p in range(0, n, width or n):
                if seq[p] == ord(">"):
                    seq[p] = ord("A")                                        # a line starting with '>' is a header
            out.append(b">" + head + b"\n" + wrap(bytes(seq), width))
        else:
            if k % 5 == 0:
                seq[0] = ord("@")
            qual = bytearray(rng.integers(0x21, 0x7F, n).astype(np.uint8).tobytes())
            qual[0] = [ord("@"), ord("+"), qual[0]][k % 3]
            plus = b"+" + (names[i] if k % 2 else b"")
            out.append(b"@" + head + b"\n" + bytes(seq) + b"\n" + plus + b"\n" + bytes(qual) + b"\n")
    text = b"".join(out)
    return text[:-1] if seed % 2 else text


def lines_of(text: bytes):
    return text[:-1].split(b"\n") if text.endswith(b"\n") else text.split(b"\n")


def join(lines) -> bytes:
    return b"\n".join(lines) + b"\n"


def refusals(fmt: str):
    """(text, line, kind, column) for every refusal kind the corpus can carry, each on a line of its own.  (A read of 2^32
    bases and the 2^31st read need gigabytes of text and are left out.)"""
    text = corpus(6, fmt)
    ls = lines_of(text)
    hdr = [i for i, x in enumerate(ls) if (x[:1] == b">" if fmt == "fasta" else i % 4 == 0)]
    out = [(b"x" + text[1:], 1, "format", 1)]
    out.append((join(ls[:hdr[3]] + [b""] + ls[hdr[3]:]), hdr[3] + 1, "empty", 1))   # before a header
    k = hdr[3] + 1                                                   # a sequence line
    t = ls[:]
    t[k] = t[k][:2] + b"\r" + t[k][2:]
    out.append((join(t), k + 1, "cr", 3))
    t = ls[:]
    t[k] = t[k][:4] + b" " + t[k][5:]
    out.append((join(t), k + 1, "seq_byte", 5))
    h = hdr[5]
    t = ls[:]
    t[h] = t[h][:1] + b" description"
    out.append((join(t), h + 1, "name_empty", 2))
    t = ls[:]
    t[h] = t[h][:1] + b"ab\x01c d\x02"
    out.append((join(t), h + 1, "name_byte", 4))
    t = ls[:]
    t[h] = t[h][:1] + b"ab\x7f"
    out.append((join(t), h + 1, "name_byte", 4))
    t = ls[:]
    t[h] = t[h] + b" desc\r"
    out.append((join(t), h + 1, "cr", len(t[h])))
    if fmt == "fasta":
        h = hdr[8]
        out.append((join(ls[:h + 1] + ls[hdr[9]:]), h + 1, "no_seq", 1))   # a header followed by a header
        out.append((text.rstrip(b"\n") + b"\n>last\n", len(ls) + 1, "no_seq", 1))   # the last line is a header
    else:
        h = hdr[8]
        t = ls[:]
        t[h] = b"x" + t[h][1:]
        out.append((join(t), h + 1, "header", 1))
        t = ls[:]
        t[h + 2] = b"-"
        out.append((join(t), h + 3, "plus", 1))
        t = ls[:]
        t[h + 3] = t[h + 3][:-1]
        out.append((join(t), h + 4, "qual_len", len(t[h + 3]) + 1))
        t = ls[:]
        t[h + 3] = t[h + 3] + b"II"
        out.append((join(t), h + 4, "qual_len", len(ls[h + 1]) + 1))
        out.append((join(ls[:hdr[-1] + 2]), hdr[-1] + 1, "truncated", 1))   # ends behind the last sequence line
        t = ls[:]
        t[h + 1] = b""
        out.append((join(t), h + 1, "no_seq", 1))                   # empty sequence: the read has none
    # the smallest offending line wins, and within it the smallest column
    t = ls[:]
    t[hdr[2] + 1] = t[hdr[2] + 1][:6] + b" \r" + t[hdr[2] + 1][8:]
    t[hdr[4]] = t[hdr[4]][:1]
    out.append((join(t), hdr[2] + 2, "seq_byte", 7))
    return out


def duplicated(fmt: str) -> bytes:
    """The corpus with read 7 named as read 0."""
    ls = lines_of(corpus(6, fmt))
    hdr = [i for i, x in enumerate(ls) if (x[:1] == b">" if fmt == "fasta" else i % 4 == 0)]
    first = re.split(rb"[ \t]", ls[hdr[0]][1:])[0]
    ls[hdr[7]] = ls[hdr[7]][:1] + first + b" copy"
    return join(ls)


@functools.lru_cache(maxsize=None)
def golden_texts(name: str):
    """The golden's reads as FASTA (what the reference read) and FASTQ, and its overlaps as PAF and MHAP text."""
    d = datasets.make(name)
    with tempfile.TemporaryDirectory() as tmp:
        out = {}
        for ext, write in (("fasta", d.write_fasta), ("paf", d.write_paf), ("mhap", d.write_mhap)):
            path = os.path.join(tmp, "o." + ext)
            write(path)
            with open(path, "rb") as f:
                out[ext] = f.read()
    ls = out["fasta"].split(b"\n")
    out["fastq"] = b"".join(b"@%s\n%s\n+\n%s\n" % (h[1:], s, b"5" * len(s)) for h, s in zip(ls[0::2], ls[1::2]))
    return out


def same(got, want):
    (gb, ge, gl), (wb, we, wl) = got[:3], want[:3]
    return bytes(gb) == bytes(wb) and np.array_equal(ge, we) and np.array_equal(gl, wl)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["fasta", "fastq"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_c_reader_matches_the_restated_contract(fmt, seed):
    text = corpus(seed, fmt)
    got, want = R.read(text), R.restate(text)
    assert same(got, want) and got[3] == want[3]
    st = got[3]
    assert st["n_reads"] == 60 and st["n_described"] == 40 and st["format"] == (1 if fmt == "fasta" else 2)
    assert st["max_len"] >= 3000 and st["n_bases"] == int(got[2].sum())
    empty = R.read(b"")
    assert same(empty, R.restate(b"")) and empty[3] == R.restate(b"")[3] and empty[3]["n_reads"] == 0


@pytest.mark.parametrize("fmt", ["fasta", "fastq"])
def test_c_reader_refuses_like_the_restated_contract(fmt):
    for bad, line, kind, col in refusals(fmt):
        for fn in (R.read, R.restate):
            with pytest.raises(R.ReadsRefused) as e:
                fn(bad)
            assert (e.value.line, e.value.kind, e.value.column) == (line, kind, col), (fn, kind)
    good = corpus(6, fmt)
    for fn in (R.read, R.restate):
        with pytest.raises(R.DuplicateName) as e:
            fn(duplicated(fmt))
        assert (e.value.earlier, e.value.later) == (0, 7)


@pytest.mark.parametrize("name", list(datasets.GOLDEN))
def test_c_reader_gives_the_golden_read_names_and_lengths(name):
    rl = datasets.load_golden(name)["in.read_len"]
    blob, ends, lens, st = R.read(golden_texts(name)["fasta"])
    assert np.array_equal(lens, rl) and st["n_reads"] == rl.shape[0] and st["n_described"] == 0
    names = [b"r%d" % i for i in range(rl.shape[0])]
    assert blob == b"".join(names) and np.array_equal(ends, np.cumsum([len(n) for n in names]))
    assert same(R.read(golden_texts(name)["fastq"]), (blob, ends, lens))


# ---- GPU ------------------------------------------------------------------------------------------------------------
def refused_at(err):
    m = re.search(r"line (\d+), column (\d+)", str(err))
    return int(m.group(1)), int(m.group(2))


@pytest.mark.gpu
def test_device_equals_the_c_reader_on_the_corpus(ctx):
    G = api.Graph(ctx)
    for fmt in ("fasta", "fastq"):
        for seed in (1, 2, 3):
            text = corpus(seed, fmt)
            want = R.read(text)
            st = G.set_reads_text(text)
            assert same(G.reads(), want), (fmt, seed)
            assert {k: st[k] for k in want[3]} == want[3] and st["n_bytes"] == len(text) and st["n_chunks"] == 1
            assert st["device_ms"] > 0
    st = G.set_reads_text(b"")
    assert st["n_reads"] == 0 and st["format"] == 0 and G.reads()[1].shape == (0,)
    G.close()


@pytest.mark.gpu
def test_reads_round_trip_what_set_reads_was_given(ctx):
    G = api.Graph(ctx)
    names = [b"r%d" % i for i in range(30)] + [b"\xff\x80 is not cut here", b"z" * 300]
    rl = np.arange(1, len(names) + 1, dtype=np.uint32) * 997
    G.set_reads(names, rl)
    blob, ends, lens = G.reads()
    assert bytes(blob) == b"".join(names) and np.array_equal(ends, np.cumsum([len(n) for n in names])) and np.array_equal(lens, rl)
    G.close()


@pytest.mark.gpu
def test_refusals_name_line_and_column_and_leave_the_session_without_reads(ctx):
    t = golden_texts("g_clean")
    G = api.Graph(ctx)
    for fmt in ("fasta", "fastq"):
        for bad, line, kind, col in refusals(fmt):
            with pytest.raises(api.RalaB200Error) as e:
                G.set_reads_text(bad)
            assert refused_at(e.value) == (line, col), (fmt, kind, str(e.value))
            with pytest.raises(api.RalaB200Error, match="set_reads"):
                G.set_overlaps_paf(t["paf"])                           # the session holds no reads
            with pytest.raises(api.RalaB200Error, match="set_reads"):
                G.reads()
        with pytest.raises(api.RalaB200Error, match="same name"):
            G.set_reads_text(duplicated(fmt))
        with pytest.raises(api.RalaB200Error, match="set_reads"):
            G.set_overlaps_mhap(t["mhap"])
    # a good call on the same session works again
    st = G.set_reads_text(t["fasta"])
    assert G.set_overlaps_paf(t["paf"])["n_unresolved"] == 0 and st["n_reads"] == G.reads()[2].shape[0]
    G.close()


def big_text(fmt: str, rng):
    """More than 2 x PAF_CHUNK_BYTES with reads across every cut: FASTA has one wrapped read longer than a chunk (so one
    chunk holds no header at all) between reads of many lengths and widths; FASTQ records of many lengths straddle the cuts."""
    names, seqs = [], []
    total = 0
    while total < 2 * api.PAF_CHUNK_BYTES + (5 << 20):
        n = int(rng.integers(1, 60000))
        if fmt == "fasta" and len(names) == 40:
            n = api.PAF_CHUNK_BYTES + 12345
        names.append(b"read_%d" % len(names))
        seqs.append(random_seq(rng, n))
        total += n * (1 if fmt == "fasta" else 2)
    if fmt == "fastq":
        return fastq(names, seqs)
    return b"".join(b">" + nm + b" d\n" + wrap(s, [60, 80, None][i % 3] if len(s) < 1e6 else 80)
                    for i, (nm, s) in enumerate(zip(names, seqs)))


@pytest.mark.gpu
def test_text_of_several_chunks_with_reads_across_every_cut(ctx):
    import torch
    rng = np.random.Generator(np.random.PCG64(9))
    G = api.Graph(ctx)
    for fmt in ("fasta", "fastq"):
        text = big_text(fmt, rng)
        want = R.read(text)
        st = G.set_reads_text(text)
        assert st["n_chunks"] >= 3 and same(G.reads(), want) and {k: st[k] for k in want[3]} == want[3], fmt
        pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()   # uploaded in place
        st2 = G.set_reads_text(pinned)
        assert same(G.reads(), want) and {k: st2[k] for k in want[3]} == want[3]
        # a fixed number of kernels per call and per chunk
        small = corpus(1, fmt)
        per_call = []
        for t in (small, text):
            before = ctx.launch_count
            s = G.set_reads_text(t)
            per_call.append((ctx.launch_count - before, s["n_chunks"]))
        (l1, c1), (l2, c2) = per_call
        assert c1 == 1 and l2 - l1 == 3 * (c2 - c1) and l1 == 2 + 3 * c1, per_call
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_sequence_and_overlap_text_to_transitive_marks_match_the_reference(ctx, name):
    st = datasets.Stages(datasets.load_golden(name))
    t = golden_texts(name)
    for reads in ("fasta", "fastq"):
        for ovl in ("paf", "mhap"):
            G = api.Graph(ctx)
            rs = G.set_reads_text(t[reads])
            assert rs["n_reads"] == st.read_len.shape[0] and np.array_equal(G.reads()[2], st.read_len)
            (G.set_overlaps_paf if ovl == "paf" else G.set_overlaps_mhap)(t[ovl])
            G.build_piles()                                             # no pile table from the host
            G.set_hills(None).run()
            c = G.counts()
            assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes, (reads, ovl)
            assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed), (reads, ovl)
            G.close()
