"""BGZF input on one B200: the configs[2] PAF text (bench_paf.py's) and the configs[2] FASTA wrapped at 80 (bench_reads.py's),
both written as BGZF at zlib level 6 (blocks of 65 280 bytes, as bgzip cuts them).

    python bench_bgzf.py [--out FILE] [--repeats 3] [--level 6]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_bgzf.json (or --out).  Per file:
  - blocks, compressed bytes and the ratio; the time to compress (a process pool, outside every timed window);
  - the inflate kernels' device time (inflate_ms of the call) and GB/s of inflated text;
  - the _bgzf call from pinned memory against the plain call from pinned text on the same text, timed alternately, and
    the reader's own kernel time of each (PAF: rala_b200_parse_paf's device_ms on the text; FASTA: device_ms);
  - a pinned host-to-device copy of the compressed bytes (the upload floor of the _bgzf call);
  - host zlib inflate of the same file (zlib.decompressobj(-15) per block) on one core and on every core;
  - parity: the _bgzf call's stats, reads (FASTA) and pile medians (PAF, after build_piles) equal the plain call's.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import struct
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from bench_paf import card, format_paf, next_tag  # noqa: E402
from bench_reads import format_reads, reads_layout  # noqa: E402

_TEXT = None   # the text being compressed or the file being inflated, shared with the forked workers


def _compress(args):
    from rala_b200 import synth
    lo, hi, level = args
    return b"".join(synth.bgzf_block(_TEXT[p:min(p + synth.BGZF_BLOCK, hi)], level) for p in range(lo, hi, synth.BGZF_BLOCK))


def _inflate_range(r):
    return _inflate(_TEXT[r[0]:r[1]])


def _inflate(z):
    out, off = 0, 0
    while off < len(z):
        xlen = struct.unpack_from("<H", z, off + 10)[0]
        bsize = struct.unpack_from("<H", z, off + 16)[0] + 1   # the BC subfield is the only one synth writes
        out += len(zlib.decompressobj(-15).decompress(z[off + 12 + xlen:off + bsize - 8]))
        off += bsize
    return out


def to_bgzf(text, level: int, workers: int) -> bytes:
    """BGZF of text on every core, one range of whole blocks per task."""
    global _TEXT
    from rala_b200 import synth
    _TEXT = text
    step = synth.BGZF_BLOCK * max(1, len(text) // synth.BGZF_BLOCK // (8 * workers) + 1)
    with mp.get_context("fork").Pool(workers) as pool:
        parts = pool.map(_compress, [(p, min(p + step, len(text)), level) for p in range(0, len(text), step)])
    return b"".join(parts) + synth.BGZF_EOF


def inflate_all_cores(z: bytes, workers: int) -> tuple:
    """Host zlib inflate of z on every core -> (inflated bytes, seconds; the pool's start is not timed)."""
    global _TEXT
    _TEXT = z
    with mp.get_context("fork").Pool(workers) as pool:
        pool.map(int, range(workers))
        t0 = time.perf_counter()
        n = sum(pool.map(_inflate_range, ranges_of(z, 4 * workers)))
        return n, time.perf_counter() - t0


def ranges_of(z: bytes, parts: int):
    """z cut at block boundaries into about `parts` (start, end) ranges."""
    cuts, off, want = [0], 0, len(z) / parts
    while off < len(z):
        off += struct.unpack_from("<H", z, off + 16)[0] + 1
        if off - cuts[-1] >= want:
            cuts.append(off)
    if cuts[-1] != len(z):
        cuts.append(len(z))
    return list(zip(cuts[:-1], cuts[1:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--level", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from rala_b200 import api, synth

    workers = os.cpu_count() or 1
    t0 = time.perf_counter()
    ds = bench.make_dataset("c3", 1)
    paf = format_paf(ds.read_len, ds.records)
    rs = synth.generate(100_000_000, 40, 10000, seed=3)
    fasta = np.zeros(reads_layout(rs.read_len, "fasta", 80)[2], np.uint8)
    format_reads(rs.read_len, "fasta", fasta, 80)
    fasta = fasta.tobytes()
    names = [b"r%d" % i for i in range(ds.n_reads)]
    gen_s = time.perf_counter() - t0

    ctx = api.Context(0)
    res = {"metric": "bgzf_inflate_bytes_per_sec", "unit": "B/s", "higher_is_better": True, "card": card(),
           "workload": "configs[2]: bench_paf.py's PAF text and bench_reads.py's FASTA (width 80), BGZF at zlib level %d" % args.level,
           "host_cores": workers, "gen_s": gen_s}
    for name, text in (("paf", paf), ("fasta", fasta)):
        t0 = time.perf_counter()
        z = to_bgzf(text, args.level, workers)
        prep_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        n_one = _inflate(z)
        zlib_one_s = time.perf_counter() - t0
        n_all, zlib_all_s = inflate_all_cores(z, workers)
        assert n_one == n_all == len(text)
        ptext = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
        pz = torch.frombuffer(bytearray(z), dtype=torch.uint8).pin_memory()
        dev = torch.empty(len(z), dtype=torch.uint8, device="cuda")
        G, H = api.Graph(ctx), api.Graph(ctx)
        if name == "paf":
            G.set_reads(names, ds.read_len)
            H.set_reads(names, ds.read_len)
            plain, via = H.set_overlaps_paf, G.set_overlaps_paf_bgzf
        else:
            plain, via = H.set_reads_text, G.set_reads_bgzf
        t_plain, t_bgzf, t_copy, inflate, reader_ms = [], [], [], [], []
        for _ in range(args.repeats + 1):
            ctx.synchronize()
            t0 = time.perf_counter()
            want = plain(ptext)
            t_plain.append(time.perf_counter() - t0)
            ctx.synchronize()
            t0 = time.perf_counter()
            got, zs = via(pz)
            t_bgzf.append(time.perf_counter() - t0)
            inflate.append(zs["inflate_ms"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev.copy_(pz, non_blocking=True)
            torch.cuda.synchronize()
            t_copy.append(time.perf_counter() - t0)
            if name == "paf":
                reader_ms.append(ctx.parse_paf(ptext, names, ds.read_len, with_time=True)[2])
            else:
                reader_ms.append(got["device_ms"])
        t_plain, t_bgzf, t_copy, inflate, reader_ms = (x[1:] for x in (t_plain, t_bgzf, t_copy, inflate, reader_ms))
        strip = lambda s: {k: v for k, v in s.items() if k != "device_ms"}   # noqa: E731
        parity = strip(got) == strip(want) and zs["n_bytes"] == len(text)
        if name == "paf":
            G.build_piles()
            H.build_piles()
            parity = parity and bool(np.array_equal(G.medians(), H.medians()))
        else:
            parity = parity and all(np.array_equal(a, b) for a, b in zip(G.reads(), H.reads()))
        G.close()
        H.close()
        del dev
        med = lambda v: float(np.median(v))   # noqa: E731
        res[name] = {"text_bytes": len(text), "compressed_bytes": len(z), "ratio": len(z) / len(text),
                     "blocks": zs["n_blocks"], "compress_s_pool": prep_s,
                     "inflate_ms": med(inflate), "inflate_runs_ms": inflate, "inflate_gbs": len(text) / med(inflate) / 1e6,
                     "bgzf_call_ms": 1e3 * med(t_bgzf), "bgzf_call_runs_ms": [1e3 * x for x in t_bgzf],
                     "plain_call_ms": 1e3 * med(t_plain), "plain_call_runs_ms": [1e3 * x for x in t_plain],
                     "reader_kernel_ms": med(reader_ms), "compressed_copy_ms": 1e3 * med(t_copy),
                     "zlib_one_core_s": zlib_one_s, "zlib_all_cores_s": zlib_all_s, "parity": bool(parity)}
        del ptext, pz
    res["value"] = res["fasta"]["text_bytes"] / (res["fasta"]["inflate_ms"] * 1e-3)
    res["parity"] = res["paf"]["parity"] and res["fasta"]["parity"]
    res["note"] = ("calls: host wall clock from pinned memory (every call synchronises), _bgzf and plain alternating; "
                   "compressed_copy_ms: pinned host-to-device copy of the BGZF bytes to a device synchronise; reader_kernel_ms: "
                   "the reader's kernels on the same text (PAF: parse_paf device_ms; FASTA: set_reads_bgzf device_ms)")
    line = json.dumps(res)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_bgzf.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")
    ctx.close()
    if not res["parity"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
