"""Plain gzip input (rala_b200_inflate_gzip and the readers' _gzip calls): synth.write_gzip against gzip; the chunked
inflate of rala_b200/csrc/gzip.cu run sequentially on the CPU (tests/host_gzip.cu, the same decoder, finder, verification
walk, symbol pass, window chain and resolve) against zlib, with the finder's entries and with hostile ones; on the GPU
(-m gpu) the device inflate against zlib, its refusals, BGZF through the gzip call, and every reader's _gzip call against
the plain call on the same text, down to the reference's transitive marks."""
import functools
import gzip
import os
import re
import shutil
import struct
import subprocess
import tempfile
import zlib

import numpy as np
import pytest

from rala_b200 import api, synth
from tests import datasets
from tests import test_bgzf_reader as TB
from tests import test_mhap_reader as TM
from tests import test_paf_reader as TP
from tests import test_reads_reader as TR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = TB.LEVELS
STRATEGIES = TB.STRATEGIES


def oracle(z: bytes) -> bytes:
    """zlib, one decompressobj(wbits=31) per member; zero bytes between and after members are skipped."""
    out, p = [], 0
    while p < len(z):
        d = zlib.decompressobj(wbits=31)
        out.append(d.decompress(z[p:]))
        if not d.eof:
            raise ValueError("truncated member")
        rest = d.unused_data
        p = len(z) - len(rest)
        while p < len(z) and z[p] == 0:
            p += 1
    return b"".join(out)


def sample_text(rng, n: int) -> bytes:
    return TB.sample_text(rng, n)


def decoys(rng, n: int) -> bytes:
    """Text full of valid dynamic-block headers (non-final DEFLATE blocks), so that the finder proposes false entries
    inside the stored blocks that carry it."""
    units = []
    while sum(map(len, units)) < n:
        piece = TR.random_seq(rng, int(rng.integers(200, 3000))) + sample_text(rng, 400)[:int(rng.integers(0, 300))]
        units.append(synth.gzip_deflate(piece, 6, final=False))
    return b"".join(units)[:n]


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_write_gzip_round_trips(level, strategy):
    rng = np.random.Generator(np.random.PCG64(level * 10 + strategy))
    text = sample_text(rng, 150_000)
    for kw in ({}, {"members": 3}, {"members": [0, 10, 10, 70_000]}, {"sync_every": 40_000},
               {"fname": b"reads.fa", "comment": b"c", "extra": b"XY\x02\x00ab", "hcrc": True}):
        z = synth.write_gzip(text, level, strategy, **kw)
        assert gzip.decompress(z) == text and oracle(z) == text, kw
    assert synth.write_gzip(b"")[:3] == b"\x1f\x8b\x08" and gzip.decompress(synth.write_gzip(b"")) == b""


@functools.lru_cache(maxsize=None)
def host_harness() -> str:
    nvcc = "/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else shutil.which("nvcc")
    assert nvcc, "nvcc is needed to compile the host harness"
    exe = os.path.join(tempfile.mkdtemp(prefix="host_gzip_"), "host_gzip")
    # AddressSanitizer: a read or write outside the input, the symbols or the text aborts the harness
    subprocess.run([nvcc, "-O1", "-g", "-std=c++17", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fsanitize=address",
                    "-o", exe, os.path.join(ROOT, "tests", "host_gzip.cu")], check=True)
    return exe


def host_inflate(z: bytes, chunk: int, entries=None) -> dict:
    head = struct.pack("<QQQ", len(z), chunk, 2**64 - 1 if entries is None else len(entries))
    if entries is not None:
        head += b"".join(struct.pack("<Q", int(e)) for e in entries)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    out = subprocess.run([host_harness()], input=head + z, capture_output=True, check=True, env=env).stdout
    status, _, member, at, corrected, rounds, chunks, n = struct.unpack_from("<IIQQQQQQ", out)
    return {"status": status, "member": member, "at": at, "corrected": corrected, "rounds": rounds, "chunks": chunks,
            "text": out[56:] if status == 0 else None, "n": n}


def corpus():
    """(name, gzip bytes): every level and strategy, members shorter than a chunk and longer than many, pigz-style
    members, every header field, 32 768-back references across cuts, zero padding, the empty input."""
    rng = np.random.Generator(np.random.PCG64(21))
    text = sample_text(rng, 300_000)
    out = [(f"level{lv}_s{st}", synth.write_gzip(text, lv, st)) for lv in LEVELS for st in STRATEGIES]
    out.append(("many_members", synth.write_gzip(text, 6, members=[1, 2, 3, 500, 40_000, 40_001, 299_999])))
    out.append(("pigz", synth.write_gzip(text, 6, sync_every=50_000)))
    out.append(("pigz_members", synth.write_gzip(text, 1, members=2, sync_every=20_000)))
    out.append(("headers", synth.write_gzip(text[:50_000], 9, fname=b"x.paf", comment=b"made by hand", extra=b"AB\x01\x00z",
                                            hcrc=True, members=2)))
    block = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    out.append(("distance_32768", synth.write_gzip(block * 6, 9)))
    out.append(("zero_padding", synth.write_gzip(text[:20_000]) + b"\x00" * 7 + synth.write_gzip(text[20_000:60_000]) + b"\x00" * 3))
    out.append(("one_byte", synth.write_gzip(b"A")))
    out.append(("empty_member", synth.write_gzip(b"") + synth.write_gzip(b"abc")))
    out.append(("decoys", synth.write_gzip(decoys(rng, 200_000), 0)))
    out.append(("empty", b""))
    return out


@pytest.mark.parametrize("chunk", [5, 64, 997, 8192, 65536])
def test_host_harness_equals_zlib(chunk):
    for name, z in corpus():
        want = oracle(z)
        got = host_inflate(z, chunk)
        assert got["status"] == 0 and got["text"] == want, (name, chunk, got["status"], got["member"], got["at"])


def test_hostile_entries_still_give_zlibs_bytes():
    rng = np.random.Generator(np.random.PCG64(22))
    text = sample_text(rng, 200_000)
    cases = [synth.write_gzip(text, 6), synth.write_gzip(text, 0), synth.write_gzip(text, 1, sync_every=30_000),
             synth.write_gzip(text, 6, members=4)]
    for z in cases:
        want = oracle(z)
        end = len(z) * 8
        rand = sorted(set(int(x) for x in rng.integers(1, end, 60)))
        stored = [8 * int(p) for p in rng.integers(20, len(z) - 20, 30)]        # byte offsets, often inside stored data
        near = []
        for b in rand[:20]:
            near += [b - 1, b, b + 1]
        total = 0
        for entries in (rand, sorted(set(stored)), sorted(set(near)), [end - 1]):
            got = host_inflate(z, 4096, entries)
            assert got["status"] == 0 and got["text"] == want
            total += got["corrected"]
        assert total > 0


def test_decoys_make_the_finder_wrong_and_the_walk_corrects_it():
    rng = np.random.Generator(np.random.PCG64(23))
    z = synth.write_gzip(decoys(rng, 400_000), 0)
    got = host_inflate(z, 8192)
    assert got["status"] == 0 and got["text"] == oracle(z) and got["corrected"] > 0


def test_corrupted_streams_are_refused_or_equal_zlib():
    rng = np.random.Generator(np.random.PCG64(24))
    text = sample_text(rng, 40_000)
    base = [synth.write_gzip(text, lv, st, members=m) for lv in (0, 6) for st in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED)
            for m in (1, 3)]
    kinds = set()
    for i in range(300):
        zb = bytearray(base[i % len(base)])
        what = i % 4
        if what == 0:
            for _ in range(int(rng.integers(1, 4))):
                zb[int(rng.integers(0, len(zb)))] ^= 1 << int(rng.integers(0, 8))
        elif what == 1:
            zb = zb[:int(rng.integers(0, len(zb)))]
        elif what == 2:
            zb[int(rng.integers(len(zb) - 8, len(zb)))] ^= 0x40          # trailer
        else:
            zb[int(rng.integers(0, 10))] ^= 1 << int(rng.integers(0, 8))   # header
        z = bytes(zb)
        try:
            want = oracle(z)
        except (zlib.error, ValueError, EOFError):
            want = None
        got = host_inflate(z, int(rng.choice([64, 1024, 8192])))
        kinds.add(got["status"])
        if want is None:
            assert got["status"] != 0, i
        elif got["status"] == 0:
            assert got["text"] == want, i
    assert len(kinds) >= 6, kinds


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_inflate_gzip_equals_zlib(ctx):
    for name, z in corpus():
        got, st = ctx.inflate_gzip(z)
        want = oracle(z)
        assert bytes(got) == want, name
        assert st["n_bytes"] == len(want) and st["n_compressed"] == len(z) and st["bgzf"] == 0, name
        assert st["inflate_ms"] >= 0


@pytest.mark.gpu
@pytest.mark.parametrize("pigz", [False, True])
def test_inflate_gzip_of_more_than_100_mib(ctx, pigz):
    rng = np.random.Generator(np.random.PCG64(25))
    seq = TR.random_seq(rng, 100 << 20)
    text = b"".join(b">r%d\n" % i + TR.wrap(seq[i << 20:(i + 1) << 20], 80) for i in range(100))
    z = synth.write_gzip(text, 1, sync_every=(4 << 20) if pigz else None)
    assert len(z) > api.PAF_CHUNK_BYTES   # more than one upload piece
    got, st = ctx.inflate_gzip(z)
    assert st["n_bytes"] == len(text) and np.array_equal(got, np.frombuffer(text, np.uint8))
    assert st["n_chunks"] > 100 and st["n_members"] == 1
    G = api.Graph(ctx)
    plain = G.set_reads_text(text)
    want = G.reads()
    rs, zs = G.set_reads_gzip(z)
    assert TR.same(G.reads(), want) and TB.strip(rs) == TB.strip(plain) and zs["inflate_ms"] > 0
    G.close()


@pytest.mark.gpu
def test_decoy_inputs_are_corrected(ctx):
    rng = np.random.Generator(np.random.PCG64(26))
    d = decoys(rng, 3 << 20)
    z = synth.write_gzip(d, 0)
    got, st = ctx.inflate_gzip(z)
    assert bytes(got) == d and st["n_corrected"] > 0
    z = synth.write_gzip(d, 6, members=3)
    got, st = ctx.inflate_gzip(z)
    assert bytes(got) == d


def refusal_cases():
    """(name, gzip bytes, member, byte offset, message part)."""
    good = synth.write_gzip(b"ACGT" * 40000 + bytes(range(256)) * 50, 6)
    two = synth.write_gzip(b"hello " * 1000) + good
    m1 = len(synth.write_gzip(b"hello " * 1000))
    out = [("magic", b"\x1f\x8c" + good[2:], 0, 0, "not a gzip member"),
           ("method", good[:2] + b"\x07" + good[3:], 0, 0, "compression method"),
           ("reserved flags", good[:3] + b"\x20" + good[4:], 0, 0, "reserved header flag"),
           ("header end", good[:6], 0, 0, "inside the member header"),
           ("second header end", two[:m1 + 5], 1, m1, "inside the member header"),
           ("trailer end", good[:-3], 0, len(good) - 8, "inside the member trailer"),
           ("stream end", good[:len(good) // 2], 0, None, "inside a DEFLATE stream"),
           ("after last", good + b"\x00\x00junk", 1, len(good) + 2, "after the last member")]
    b = bytearray(good)
    b[-8] ^= 1
    out.append(("crc", bytes(b), 0, len(good) - 8, "CRC32"))
    b = bytearray(two)
    b[-1] ^= 1
    out.append(("isize", bytes(b), 1, len(two) - 8, "ISIZE"))
    h = synth.write_gzip(b"abc", hcrc=True)
    b = bytearray(h)
    b[10] ^= 1
    out.append(("header crc", bytes(b), 0, 0, "FHCRC"))
    w = TB.BitWriter()   # a fixed block: literal 'a', then length 3 at distance 2, before the member's start
    w.put(1, 1), w.put(1, 2), w.code(0x30 + ord("a"), 8), w.code(1, 7), w.code(1, 5), w.code(0, 7)
    head = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"
    far = head + w.bytes() + struct.pack("<II", 0, 4)
    out.append(("distance before the member", synth.write_gzip(b"xyz") + far, 1, len(synth.write_gzip(b"xyz")) + 10,
                "before the start of the member"))
    w = TB.BitWriter()
    w.put(1, 1), w.put(3, 2)
    out.append(("btype 3", head + w.bytes() + b"\x00" * 8, 0, 10, "type 3"))
    b = bytearray(synth.write_gzip(b"hello world " * 1000, 0))
    b[10 + 2] ^= 0x20   # LEN of the first stored block
    out.append(("stored nlen", bytes(b), 0, 10, "complement of NLEN"))
    # a later member's CRC is reported before an error further on
    bad = bytearray(synth.write_gzip(b"first " * 100))
    bad[-5] ^= 1
    out.append(("earliest error first", bytes(bad) + good[:-20], 0, len(bad) - 8, "CRC32"))
    return out


@pytest.mark.gpu
def test_malformed_inputs_are_refused_naming_member_and_offset(ctx):
    for name, z, member, off, why in refusal_cases():
        with pytest.raises(api.RalaB200Error) as e:
            ctx.inflate_gzip(z)
        msg = str(e.value)
        m = re.search(r"status (-?\d+): gzip member (\d+) \(byte offset (\d+)\): (.*)", msg)
        assert m and int(m.group(1)) == -2 and int(m.group(2)) == member and why in m.group(4), (name, msg)
        if off is not None:
            assert int(m.group(3)) == off, (name, msg)
        got = host_inflate(z, 4096)
        assert got["status"] != 0 and got["member"] == member and (off is None or got["at"] == off), (name, got["status"])


@pytest.mark.gpu
def test_bgzf_through_the_gzip_call_equals_inflate_bgzf(ctx):
    rng = np.random.Generator(np.random.PCG64(27))
    text = sample_text(rng, 500_000)
    z = synth.write_bgzf(text, 6)
    want, bs = ctx.inflate_bgzf(z)
    got, st = ctx.inflate_gzip(z)
    assert np.array_equal(got, want) and st["bgzf"] == 1 and st["n_chunks"] == 0 and st["n_members"] == bs["n_blocks"]
    G = api.Graph(ctx)
    fa = b"".join(b">r%d\n" % i + TR.random_seq(rng, 500) + b"\n" for i in range(200))
    rs, zs = G.set_reads_gzip(synth.write_bgzf(fa))
    assert zs["bgzf"] == 1 and TB.strip(rs) == TB.strip(G.set_reads_text(fa))
    G.close()


# ---- the readers through gzip -------------------------------------------------------------------------------------------
def members_in(text: bytes, rng):
    """Member cuts inside names, numbers, newlines and records (the BGZF test's block cuts)."""
    return TB.cuts_in(text, rng)


@pytest.mark.gpu
def test_reads_through_gzip_equal_the_plain_call(ctx):
    rng = np.random.Generator(np.random.PCG64(31))
    G = api.Graph(ctx)
    for fmt in ("fasta", "fastq"):
        texts = [TR.corpus(seed, fmt) for seed in (1, 2, 3)] + [TR.duplicated(fmt)] + [t for t, *_ in TR.refusals(fmt)]
        for i, text in enumerate(texts):
            kw = {"members": members_in(text, rng)} if i % 2 else {"sync_every": 3000}
            z = synth.write_gzip(text, int(rng.choice(LEVELS)), **kw)
            if TB.same_call(G.set_reads_text, G.set_reads_gzip, text, z) is not None:
                want = G.reads()
                G.set_reads_text(text)
                assert TR.same(want, G.reads())
    G.close()


@pytest.mark.gpu
def test_overlaps_through_gzip_equal_the_plain_call(ctx):
    rng = np.random.Generator(np.random.PCG64(32))
    G = api.Graph(ctx)
    for seed in (1, 2):
        text, names, rl = TP.corpus(seed)
        G.set_reads(names, rl)
        for t in [text] + [b for b, *_ in TP.refusals(text)]:
            TB.same_call(G.set_overlaps_paf, G.set_overlaps_paf_gzip, t, synth.write_gzip(t, 6, members=members_in(t, rng)))
        mtext, mrl = TM.corpus(seed)
        G.set_reads(TM.read_names(len(mrl)), mrl)
        for t in [mtext] + [b for b, *_ in TM.refusals(mtext, len(mrl))]:
            TB.same_call(G.set_overlaps_mhap, G.set_overlaps_mhap_gzip, t, synth.write_gzip(t, 1, sync_every=5000))
    good = TP.golden_anchor("g_clean")
    G.set_reads(good[1], good[2])
    with pytest.raises(api.RalaB200Error, match="gzip member"):
        G.set_overlaps_paf_gzip(synth.write_gzip(good[0])[:-40])
    with pytest.raises(api.RalaB200Error, match="set_overlaps"):
        G.build_piles()
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_gzip_sequence_and_overlap_files_to_transitive_marks_match_the_reference(ctx, name):
    st = datasets.Stages(datasets.load_golden(name))
    t = TR.golden_texts(name)
    for reads in ("fasta", "fastq"):
        for ovl in ("paf", "mhap"):
            G = api.Graph(ctx)
            rs, _ = G.set_reads_gzip(synth.write_gzip(t[reads], 6))
            assert rs["n_reads"] == st.read_len.shape[0] and np.array_equal(G.reads()[2], st.read_len)
            (G.set_overlaps_paf_gzip if ovl == "paf" else G.set_overlaps_mhap_gzip)(synth.write_gzip(t[ovl], 6, sync_every=20_000))
            G.build_piles()
            G.set_hills(None).run()
            c = G.counts()
            assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes, (reads, ovl)
            assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed), (reads, ovl)
            G.close()
