"""BGZF input (rala_b200_inflate_bgzf and the readers' _bgzf calls): synth.write_bgzf against gzip and the BGZF header
contract; the block decoder of rala_b200/csrc/bgzf.cuh compiled for the CPU (tests/host_bgzf.cu) against zlib on random
blocks of every kind and on corrupted ones; on the GPU (-m gpu) the device inflate against gzip, its refusals, and every
reader's _bgzf call against the plain call on the same text, down to the reference's transitive marks."""
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
from tests import test_mhap_reader as TM
from tests import test_paf_reader as TP
from tests import test_reads_reader as TR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = (0, 1, 6, 9)
STRATEGIES = (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)


def members(data: bytes):
    """(offset, BSIZE, header length, CRC32, ISIZE) of every BGZF member, read the way the format defines them."""
    out, off = [], 0
    while off < len(data):
        assert data[off:off + 4] == b"\x1f\x8b\x08\x04"
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        p, bsize = off + 12, None
        while p < off + 12 + xlen:
            si, slen = data[p:p + 2], struct.unpack_from("<H", data, p + 2)[0]
            if si == b"BC" and slen == 2:
                bsize = struct.unpack_from("<H", data, p + 4)[0] + 1
            p += 4 + slen
        crc, isize = struct.unpack_from("<II", data, off + bsize - 8)
        out.append((off, bsize, 12 + xlen, crc, isize))
        off += bsize
    assert off == len(data)
    return out


def sample_text(rng, n: int) -> bytes:
    """A mix that makes zlib use stored, fixed and dynamic blocks: random bytes, DNA, runs and repeats."""
    parts = [rng.integers(0, 256, n // 4, dtype=np.uint8).tobytes(), TR.random_seq(rng, n // 4), b"\x00" * (n // 8),
             (b"read_%d\t" % n) * (n // 64), bytes(range(256)) * (n // 1024 + 1)]
    return b"".join(parts)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_write_bgzf_round_trips_and_keeps_the_bgzf_contract(level, strategy):
    rng = np.random.Generator(np.random.PCG64(level * 10 + strategy))
    text = sample_text(rng, 200_000)
    z = synth.write_bgzf(text, level, strategy)
    assert gzip.decompress(z) == text
    ms = members(z)
    assert z[ms[-1][0]:] == synth.BGZF_EOF and ms[-1][4] == 0
    pos = 0
    for off, bsize, hl, crc, isize in ms:
        assert isize <= synth.BGZF_BLOCK and bsize <= 65536
        chunk = text[pos:pos + isize]
        assert zlib.decompress(z[off + hl:off + bsize - 8], -15) == chunk and zlib.crc32(chunk) == crc
        pos += isize
    assert pos == len(text)
    cut = synth.write_bgzf(b"abcdef", level, strategy, cuts=[0, 1, 1, 4])   # an empty first and an empty middle block
    assert gzip.decompress(cut) == b"abcdef" and [m[4] for m in members(cut)] == [0, 1, 0, 3, 2, 0]


@functools.lru_cache(maxsize=None)
def host_decoder() -> str:
    nvcc = "/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else shutil.which("nvcc")
    assert nvcc, "nvcc is needed to compile the host harness"
    out_dir = tempfile.mkdtemp(prefix="host_bgzf_")
    exe = os.path.join(out_dir, "host_bgzf")
    # AddressSanitizer: a read or write outside a block's own input or output buffer aborts the harness
    subprocess.run([nvcc, "-O1", "-g", "-std=c++17", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fsanitize=address",
                    "-o", exe, os.path.join(ROOT, "tests", "host_bgzf.cu")], check=True)
    return exe


def host_inflate(items):
    """(raw DEFLATE, isize, crc) per block -> (status, output or None) per block from the host build of the decoder."""
    buf = b"".join(struct.pack("<III", len(z), isize, crc) + z for z, isize, crc in items)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    out = subprocess.run([host_decoder()], input=buf, capture_output=True, check=True, env=env).stdout
    res, p = [], 0
    for _, isize, _ in items:
        rc = struct.unpack_from("<I", out, p)[0]
        p += 4
        res.append((rc, out[p:p + isize] if rc == 0 else None))
        if rc == 0:
            p += isize
    assert p == len(out)
    return res


def random_blocks(seed: int, n: int):
    """n random blocks of every kind: sizes from 0 to 65536, bytes from random to constant, every level and strategy."""
    rng = np.random.Generator(np.random.PCG64(seed))
    sizes = np.where(rng.random(n) < 0.9, rng.integers(0, 600, n), rng.integers(0, 65537, n))
    out = []
    for i, size in enumerate(sizes.tolist()):
        kind = i % 6
        if kind == 0:
            d = rng.integers(0, 256, size, dtype=np.uint8).tobytes()
        elif kind == 1:
            d = TR.random_seq(rng, size)
        elif kind == 2:
            d = bytes([i & 255]) * size
        elif kind == 3:
            d = rng.integers(0, 3, size, dtype=np.uint8).tobytes()
        elif kind == 4:
            unit = rng.integers(0, 256, int(rng.integers(1, 40)), dtype=np.uint8).tobytes()
            d = (unit * (size // len(unit) + 1))[:size]
        else:
            d = (b"r%d\t%d\t" % (i, size)) * (size // 8)
        level = LEVELS[int(rng.integers(0, 4))]
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, STRATEGIES[int(rng.integers(0, 5))])
        out.append((c.compress(d) + c.flush(), d))
    return out


def test_host_decoder_equals_zlib_on_random_blocks():
    blocks = random_blocks(1, 100_000)
    res = host_inflate([(z, len(d), zlib.crc32(d)) for z, d in blocks])
    bad = [i for i, ((rc, got), (_, d)) in enumerate(zip(res, blocks)) if rc != 0 or got != d]
    assert not bad, bad[:10]


def test_host_decoder_refuses_corrupted_blocks_or_equals_zlib():
    rng = np.random.Generator(np.random.PCG64(2))
    items, want = [], []
    for z, d in random_blocks(3, 30_000):
        zb = bytearray(z)
        for _ in range(int(rng.integers(1, 4))):
            if zb:
                zb[int(rng.integers(0, len(zb)))] ^= 1 << int(rng.integers(0, 8))
        if rng.random() < 0.2:
            zb = zb[:int(rng.integers(0, len(zb) + 1))]
        if rng.random() < 0.1:
            zb += bytes(rng.integers(0, 256, int(rng.integers(1, 5)), dtype=np.uint8))
        isize = len(d) + (int(rng.integers(-2, 3)) if rng.random() < 0.1 else 0)
        items.append((bytes(zb), max(isize, 0), zlib.crc32(d)))
        want.append(d)
    res = host_inflate(items)
    kinds = set()
    for (rc, got), d in zip(res, want):
        kinds.add(rc)
        assert rc != 0 or got == d   # accepted only when the CRC matched, and then it is the original block
    assert len(kinds) >= 10, kinds  # the corruptions reach most of the refusals


# ---- GPU ------------------------------------------------------------------------------------------------------------
def member(deflate: bytes, crc: int, isize: int, extra: bytes = b"") -> bytes:
    """One BGZF member around a raw DEFLATE stream, with optional extra subfields before the BC one."""
    xlen = len(extra) + 6
    head = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", xlen) + extra + b"BC\x02\x00"
    return head + struct.pack("<H", len(head) + 2 + len(deflate) + 8 - 1) + deflate + struct.pack("<II", crc, isize)


class BitWriter:
    def __init__(self):
        self.bits = []

    def put(self, v: int, n: int):           # LSB first (header fields)
        self.bits += [(v >> i) & 1 for i in range(n)]

    def code(self, v: int, n: int):          # MSB first (Huffman codes)
        self.bits += [(v >> (n - 1 - i)) & 1 for i in range(n)]

    def bytes(self) -> bytes:
        b = self.bits + [0] * (-len(self.bits) % 8)
        return bytes(sum(b[i + k] << k for k in range(8)) for i in range(0, len(b), 8))


def inflate_cases():
    rng = np.random.Generator(np.random.PCG64(5))
    text = sample_text(rng, 400_000)
    cases = {f"level{lv}_s{st}": synth.write_bgzf(text, lv, st) for lv in LEVELS for st in STRATEGIES}
    cases["empty_and_one_byte_blocks"] = synth.write_bgzf(b"ab" + text[:1000], 6, cuts=[0, 0, 1, 1, 2, 3, 500])
    noise = rng.integers(0, 256, 65280 * 3, dtype=np.uint8).tobytes()
    cases["incompressible_65280"] = synth.write_bgzf(noise, 6)
    runs = b"A" * 65536 + TR.random_seq(rng, 65536) + b"\n" * 65536
    cases["isize_65536"] = synth.write_bgzf(runs, 9, cuts=[65536, 131072])
    cases["all_byte_values"] = synth.write_bgzf(bytes(range(256)) * 300 + bytes(range(255, -1, -1)) * 300, 6)
    cases["eof_in_the_middle"] = synth.write_bgzf(text[:70000], 6) + synth.write_bgzf(text[70000:140000], 1)
    d = text[:5000]
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    z = c.compress(d) + c.flush()
    cases["extra_subfields"] = (member(z, zlib.crc32(d), len(d), extra=b"XY\x03\x00abc")
                                + member(z, zlib.crc32(d), len(d), extra=b"AB\x00\x00") + synth.BGZF_EOF)
    cases["empty_file"] = b""
    cases["only_eof"] = synth.BGZF_EOF
    return cases


@pytest.mark.gpu
def test_inflate_equals_gzip(ctx):
    for name, z in inflate_cases().items():
        got, st = ctx.inflate_bgzf(z)
        want = gzip.decompress(z) if z else b""
        assert bytes(got) == want, name
        assert st["n_bytes"] == len(want) and st["n_compressed"] == len(z) and st["n_blocks"] == (len(members(z)) if z else 0), name
        assert st["inflate_ms"] >= 0


@pytest.mark.gpu
def test_inflate_of_more_than_100_mib_over_several_chunks(ctx):
    rng = np.random.Generator(np.random.PCG64(6))
    seq = TR.random_seq(rng, 100 << 20)
    text = b"".join(b">r%d\n" % i + TR.wrap(seq[i << 20:(i + 1) << 20], 80) for i in range(100))
    z = synth.write_bgzf(text, 1)
    got, st = ctx.inflate_bgzf(z)
    assert st["n_bytes"] == len(text) and np.array_equal(got, np.frombuffer(text, np.uint8))
    G = api.Graph(ctx)
    plain = G.set_reads_text(text)
    want = G.reads()
    rs, zs = G.set_reads_bgzf(z)
    assert TR.same(G.reads(), want) and strip(rs) == strip(plain) and rs["n_chunks"] > 3 and zs["inflate_ms"] > 0
    G.close()


def refusal_cases():
    """(name, BGZF bytes, block, byte offset, message part): each malformed input and where it is refused."""
    good = synth.write_bgzf(b"ACGT" * 40000, 6)
    ms = members(good)
    out = [("magic", b"\x1f\x8c" + good[2:], 0, 0, "not a gzip member"),
           ("plain gzip", gzip.compress(b"ACGT" * 1000), 0, 0, "not BGZF"),
           ("truncated", good[:-40], len(ms) - 2, ms[-2][0], "past the end of the input")]
    big = bytearray(good)
    struct.pack_into("<H", big, ms[1][0] + 16, 0xFFFF)
    out.append(("bsize past the end", bytes(synth.write_bgzf(b"x" * 100) + bytes(big[ms[1][0]:ms[1][0] + 200])), 2, None,
                "past the end"))
    one = synth.write_bgzf(b"abc")[:-28]
    out.append(("btype 3", one + member(b"\x07", 0, 0), 1, len(one), "type 3"))
    stored = bytearray(member(b"\x01\x03\x00\xfc\xff" + b"xyz", zlib.crc32(b"xyz"), 3))
    stored[18 + 3] ^= 1
    out.append(("stored nlen", one + bytes(stored), 1, len(one), "complement of NLEN"))
    w = BitWriter()
    w.put(1, 1), w.put(2, 2), w.put(0, 5), w.put(0, 5), w.put(15, 4)
    for _ in range(19):
        w.put(1, 3)
    out.append(("over-subscribed", one + member(w.bytes(), 0, 0), 1, len(one), "over-subscribed"))
    w = BitWriter()
    w.put(1, 1), w.put(1, 2), w.code(1, 7), w.put(0, 0), w.code(0, 5), w.code(0, 7)   # length 3, distance 1, at offset 0
    out.append(("distance before the start", one + member(w.bytes(), 0, 3), 1, len(one), "before the start"))
    for delta, what in ((-1, "more than ISIZE"), (1, "fewer than ISIZE")):
        b = bytearray(good)
        struct.pack_into("<I", b, ms[2][0] + ms[2][1] - 4, ms[2][4] + delta)
        out.append((f"isize {delta:+d}", bytes(b), 2, ms[2][0], what))
    b = bytearray(good)
    struct.pack_into("<I", b, ms[1][0] + ms[1][1] - 4, 65537)
    out.append(("isize above 65536", bytes(b), 1, ms[1][0], "above 65536"))
    b = bytearray(good)
    b[ms[3][0] + ms[3][1] - 8] ^= 0x10
    out.append(("crc field", bytes(b), 3, ms[3][0], "CRC32"))
    st = synth.write_bgzf(b"hello world " * 1000, 0)
    b = bytearray(st)
    b[100] ^= 0x20
    out.append(("byte in a stored block", bytes(b), 0, 0, "CRC32"))
    return out


@pytest.mark.gpu
def test_malformed_inputs_are_refused_naming_block_and_offset(ctx):
    for name, z, block, off, why in refusal_cases():
        with pytest.raises(api.RalaB200Error) as e:
            ctx.inflate_bgzf(z)
        msg = str(e.value)
        m = re.search(r"status (-?\d+): BGZF block (\d+) \(byte offset (\d+)\): (.*)", msg)
        assert m and int(m.group(1)) == -2 and int(m.group(2)) == block and why in m.group(4), (name, msg)
        if off is not None:
            assert int(m.group(3)) == off, (name, msg)
    with pytest.raises(api.RalaB200Error, match="bgzip"):
        ctx.inflate_bgzf(gzip.compress(b"ACGT"))


# ---- the readers through BGZF -----------------------------------------------------------------------------------------
def strip(st: dict) -> dict:
    return {k: v for k, v in st.items() if k != "device_ms"}


def cuts_in(text: bytes, rng, marks=(b"\t", b"\n", b" ", b"@", b"+", b">")):
    """Block cuts at random offsets and right before and after bytes of each kind (separators, record starts), at most
    65536 bytes apart."""
    n = len(text)
    pts = set(int(x) for x in rng.integers(0, n + 1, max(4, n // 3000)))
    for m in marks:
        at = [i for i in range(min(n, 200_000)) if text[i] == m[0]]
        for i in at[:: max(1, len(at) // 20)][:20]:
            pts.update((i, i + 1))
    pts = sorted(p for p in pts if 0 < p < n)
    out, last = [], 0
    for p in pts + [n]:
        while p - last > 65536:
            last += 65536
            out.append(last)
        if p > last:
            out.append(p)
            last = p
    return out[:-1] if out and out[-1] == n else out


def same_call(plain, bgzf, text: bytes, z: bytes):
    """plain(text) and bgzf(z) both succeed with the same stats, or both fail with the same status and message."""
    try:
        want = plain(text)
    except api.RalaB200Error as e:
        with pytest.raises(api.RalaB200Error) as got:
            bgzf(z)
        tail = lambda err: str(err).split(": ", 1)[1]   # noqa: E731  (past the name of the call)
        assert tail(got.value) == tail(e), (str(got.value), str(e))
        return None
    got, zs = bgzf(z)
    assert strip(got) == strip(want) and zs["n_bytes"] == len(text)
    return got


@pytest.mark.gpu
def test_reads_through_bgzf_equal_the_plain_call(ctx):
    rng = np.random.Generator(np.random.PCG64(11))
    G = api.Graph(ctx)
    for fmt in ("fasta", "fastq"):
        texts = [TR.corpus(seed, fmt) for seed in (1, 2, 3)] + [TR.duplicated(fmt)] + [t for t, *_ in TR.refusals(fmt)]
        for text in texts:
            z = synth.write_bgzf(text, int(rng.choice(LEVELS)), cuts=cuts_in(text, rng))
            if same_call(G.set_reads_text, G.set_reads_bgzf, text, z) is not None:
                want = G.reads()
                G.set_reads_text(text)
                assert TR.same(want, G.reads())
    G.close()


@pytest.mark.gpu
def test_overlaps_through_bgzf_equal_the_plain_call(ctx):
    rng = np.random.Generator(np.random.PCG64(12))
    G = api.Graph(ctx)
    for seed in (1, 2):
        text, names, rl = TP.corpus(seed)
        G.set_reads(names, rl)
        for t in [text] + [b for b, *_ in TP.refusals(text)]:
            same_call(G.set_overlaps_paf, G.set_overlaps_paf_bgzf, t, synth.write_bgzf(t, 6, cuts=cuts_in(t, rng)))
        mtext, mrl = TM.corpus(seed)
        G.set_reads(TM.read_names(len(mrl)), mrl)
        for t in [mtext] + [b for b, *_ in TM.refusals(mtext, len(mrl))]:
            same_call(G.set_overlaps_mhap, G.set_overlaps_mhap_bgzf, t, synth.write_bgzf(t, 1, cuts=cuts_in(t, rng)))
    # a refused BGZF call leaves the session without records, as the plain refusal does
    good = TP.golden_anchor("g_clean")
    G.set_reads(good[1], good[2])
    with pytest.raises(api.RalaB200Error, match="BGZF block"):
        G.set_overlaps_paf_bgzf(synth.write_bgzf(good[0])[:-40])
    with pytest.raises(api.RalaB200Error, match="set_overlaps"):
        G.build_piles()
    G.close()


@pytest.mark.gpu
def test_a_line_as_long_as_the_chunk_is_read_by_both_paths(ctx):
    import torch
    rng = np.random.Generator(np.random.PCG64(13))
    G = api.Graph(ctx)
    for extra in (0, 1):
        seq = TR.random_seq(rng, api.PAF_CHUNK_BYTES - 1 + extra)      # the line with its '\n': the chunk, or one more
        text = b">r0\n" + seq + b"\n>r1\nACGT\n"
        z = synth.write_bgzf(text, 1)
        for pinned in (False, True):
            src_t, src_z = text, z
            if pinned:
                src_t = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
                src_z = torch.frombuffer(bytearray(z), dtype=torch.uint8).pin_memory()
            got = same_call(G.set_reads_text, G.set_reads_bgzf, src_t, src_z)
            assert (got is None) == bool(extra), (extra, pinned)
            if got is not None:
                assert list(G.reads()[2]) == [len(seq), 4]
    with pytest.raises(api.RalaB200Error, match="longer than the upload chunk"):
        G.set_reads_bgzf(z)
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", datasets.FROZEN_GOLDEN)
def test_bgzf_sequence_and_overlap_files_to_transitive_marks_match_the_reference(ctx, name):
    st = datasets.Stages(datasets.load_golden(name))
    t = TR.golden_texts(name)
    rng = np.random.Generator(np.random.PCG64(14))
    for reads in ("fasta", "fastq"):
        for ovl in ("paf", "mhap"):
            plain = api.Graph(ctx)
            plain.set_reads_text(t[reads])
            (plain.set_overlaps_paf if ovl == "paf" else plain.set_overlaps_mhap)(t[ovl])
            plain.build_piles()
            G = api.Graph(ctx)
            rs, _ = G.set_reads_bgzf(synth.write_bgzf(t[reads], 6, cuts=cuts_in(t[reads], rng)))
            assert rs["n_reads"] == st.read_len.shape[0] and np.array_equal(G.reads()[2], st.read_len)
            (G.set_overlaps_paf_bgzf if ovl == "paf" else G.set_overlaps_mhap_bgzf)(synth.write_bgzf(t[ovl], 6, cuts=cuts_in(t[ovl], rng)))
            G.build_piles()
            assert np.array_equal(G.medians(), plain.medians()), (reads, ovl)
            G.set_hills(None).run()
            c = G.counts()
            assert c["n_transitive_pairs"] == st.n_pairs and c["n_nodes"] == st.n_nodes, (reads, ovl)
            assert np.array_equal(G.edges(), st.edges) and np.array_equal(G.marked(), st.removed), (reads, ovl)
            G.close()
            plain.close()
