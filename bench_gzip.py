"""Plain gzip input on one B200: the configs[2] PAF text (bench_paf.py's) as one zlib level-6 stream (`minimap2 | gzip`),
and the configs[2] FASTA wrapped at 80 (bench_reads.py's) pigz-style (128 KiB pieces, each with the 32 KiB before it as
dictionary, joined by Z_SYNC_FLUSH, compressed by a process pool), plus a prefix of that FASTA as one zlib stream.

    python bench_gzip.py [--out FILE] [--repeats 3] [--fasta-stream-mib 512]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_gzip.json (or --out).  Per file:
  - compressed bytes, chunks, the chunk size C, corrected chunk decodes, counting rounds;
  - the inflate kernels' device time per stage (finder, counting, symbols, window chain, resolve + CRC32);
  - the _gzip call from pinned memory against the plain call on the inflated text and the _bgzf call on the same text
    (BGZF at level 6), timed alternately;
  - host zlib inflate of the same file on one core (zlib.decompressobj(wbits=31));
  - parity: the _gzip call's stats, reads (FASTA) and pile medians (PAF, after build_piles) equal the plain call's.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from bench_bgzf import to_bgzf  # noqa: E402
from bench_paf import card, format_paf, next_tag  # noqa: E402
from bench_reads import format_reads, reads_layout  # noqa: E402

PIGZ_PIECE = 128 << 10


def host_inflate(z: bytes) -> tuple:
    t0 = time.perf_counter()
    d = zlib.decompressobj(wbits=31)
    n = len(d.decompress(z))
    return n, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--fasta-stream-mib", type=int, default=512)
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
    prefix = fasta[:args.fasta_stream_mib << 20]
    prefix = prefix[:prefix.rindex(b"\n>") + 1]   # whole records
    gen_s = time.perf_counter() - t0

    ctx = api.Context(0)
    res = {"metric": "gzip_call_speedup_over_one_core_zlib", "unit": "x", "higher_is_better": True, "card": card(),
           "workload": ("configs[2]: bench_paf.py's PAF text as one zlib level-6 stream; bench_reads.py's FASTA (width 80) "
                        "pigz-style at level 6 (128 KiB pieces); a %d MiB record-aligned prefix of that FASTA as one level-6 "
                        "stream" % args.fasta_stream_mib),
           "host_cores": workers, "gen_s": gen_s}
    with mp.get_context("fork").Pool(workers) as pool:
        inputs = [("paf", paf, lambda t: synth.write_gzip(t, 6)),
                  ("fasta_pigz", fasta, lambda t: synth.write_gzip(t, 6, sync_every=PIGZ_PIECE, pool=pool)),
                  ("fasta_stream_prefix", prefix, lambda t: synth.write_gzip(t, 6))]
        for name, text, compress in inputs:
            t0 = time.perf_counter()
            z = compress(text)
            prep_s = time.perf_counter() - t0
            bz = to_bgzf(text, 6, workers)
            n_one, zlib_one_s = host_inflate(z)
            assert n_one == len(text)
            ptext = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
            pz = torch.frombuffer(bytearray(z), dtype=torch.uint8).pin_memory()
            pb = torch.frombuffer(bytearray(bz), dtype=torch.uint8).pin_memory()
            G, H, B = api.Graph(ctx), api.Graph(ctx), api.Graph(ctx)
            if name == "paf":
                for X in (G, H, B):
                    X.set_reads(names, ds.read_len)
                plain, via, via_bgzf = H.set_overlaps_paf, G.set_overlaps_paf_gzip, B.set_overlaps_paf_bgzf
            else:
                plain, via, via_bgzf = H.set_reads_text, G.set_reads_gzip, B.set_reads_bgzf
            t_plain, t_gzip, t_bgzf, stats = [], [], [], []
            for _ in range(args.repeats + 1):
                ctx.synchronize()
                t0 = time.perf_counter()
                want = plain(ptext)
                t_plain.append(time.perf_counter() - t0)
                ctx.synchronize()
                t0 = time.perf_counter()
                got, zs = via(pz)
                t_gzip.append(time.perf_counter() - t0)
                stats.append(zs)
                ctx.synchronize()
                t0 = time.perf_counter()
                via_bgzf(pb)
                t_bgzf.append(time.perf_counter() - t0)
            t_plain, t_gzip, t_bgzf, stats = (x[1:] for x in (t_plain, t_gzip, t_bgzf, stats))
            strip = lambda s: {k: v for k, v in s.items() if k != "device_ms"}   # noqa: E731
            parity = strip(got) == strip(want) and zs["n_bytes"] == len(text)
            if name == "paf":
                G.build_piles()
                H.build_piles()
                parity = parity and bool(np.array_equal(G.medians(), H.medians()))
            else:
                parity = parity and all(np.array_equal(a, b) for a, b in zip(G.reads(), H.reads()))
            for X in (G, H, B):
                X.close()
            med = lambda v: float(np.median(v))   # noqa: E731
            gz_ms = 1e3 * med(t_gzip)
            res[name] = {"text_bytes": len(text), "compressed_bytes": len(z), "ratio": len(z) / len(text), "compress_s": prep_s,
                         "chunk_bytes": zs["chunk_bytes"], "chunks": zs["n_chunks"], "corrected": zs["n_corrected"],
                         "rounds": zs["rounds"], "members": zs["n_members"],
                         "inflate_ms": med([s["inflate_ms"] for s in stats]),
                         "stage_ms": {k: med([s["stage_ms"][k] for s in stats]) for k in api.GZIP_STAGES},
                         "gzip_call_ms": gz_ms, "gzip_call_runs_ms": [1e3 * x for x in t_gzip],
                         "plain_call_ms": 1e3 * med(t_plain), "plain_call_runs_ms": [1e3 * x for x in t_plain],
                         "bgzf_call_ms": 1e3 * med(t_bgzf), "bgzf_call_runs_ms": [1e3 * x for x in t_bgzf],
                         "zlib_one_core_s": zlib_one_s, "speedup_over_zlib_one_core": zlib_one_s * 1e3 / gz_ms,
                         "gzip_over_bgzf_call": gz_ms / (1e3 * med(t_bgzf)), "parity": bool(parity)}
            del ptext, pz, pb
    res["value"] = min(res[k]["speedup_over_zlib_one_core"] for k in ("paf", "fasta_pigz", "fasta_stream_prefix"))
    res["parity"] = all(res[k]["parity"] for k in ("paf", "fasta_pigz", "fasta_stream_prefix"))
    res["note"] = ("calls: host wall clock from pinned memory (every call synchronises), plain, _gzip and _bgzf alternating; "
                   "zlib_one_core_s: zlib.decompressobj(wbits=31) of the same gzip file on one core")
    line = json.dumps(res)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_gzip.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")
    ctx.close()
    if not res["parity"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
