"""FASTA / FASTQ text -> the session's read names, lengths and name table on one B200, on the configs[2] read set
(synth.generate(100_000_000, 40, 10000, seed=3): ~400k reads of 10 kbp).

    python bench_reads.py [--out FILE] [--repeats 3] [--width 80]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_reads.json (or --out):
  - kernel time of rala_b200_graph_set_reads_text (line scan, roles, byte rules, lengths, name table: its device_ms), text
    bytes per second and the share of the HBM bound on the bytes the kernels have to move, for FASTA (wrapped at --width,
    about 4 GB) and FASTQ (about 8 GB);
  - the call from pinned host text next to a plain host-to-device copy of the same bytes, timed in the same run;
  - the plain-C reader (tests/reads_oracle.c) on one core of this host;
  - a full step: FASTA text + PAF text -> build_piles -> run, parity-gated against the session fed by
    set_reads(synth names, lengths) with the same PAF text.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload generator and HBM peak of the main benchmark)
from bench_paf import _digits, card, format_paf, next_tag  # noqa: E402


def reads_layout(read_len: np.ndarray, fmt: str, width: int | None):
    """Record starts, header lengths and the total size of ">r<i>\\n" + sequence (wrapped at width) or
    "@r<i>\\n" + sequence + "\\n+\\n" + quality + "\\n" for every read."""
    L = read_len.astype(np.int64)
    _, nd = _digits(np.arange(L.shape[0], dtype=np.uint32))
    hdr = nd + 3
    if fmt == "fasta":
        body = L + (-(-L // width) if width else 1)
    else:
        body = 2 * L + 4
    size = hdr + body
    start = np.concatenate([[0], np.cumsum(size)[:-1]])
    return start, hdr, int(size.sum())


def format_reads(read_len: np.ndarray, fmt: str, out: np.ndarray, width: int | None = 80, seed: int = 7):
    """The reads as FASTA or FASTQ text into out (reads_layout's size), vectorised: the bases (and the FASTQ qualities) are a
    seeded random ACGT block of prime length repeated over the text, the headers, line ends and '+' lines go on top."""
    n = read_len.shape[0]
    L = read_len.astype(np.int64)
    start, hdr, total = reads_layout(read_len, fmt, width)
    assert out.shape[0] == total
    rng = np.random.Generator(np.random.PCG64(seed))
    block = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 1_048_573)]
    for p in range(0, total, block.shape[0]):
        q = min(total, p + block.shape[0])
        out[p:q] = block[:q - p]
    d, nd = _digits(np.arange(n, dtype=np.uint32))
    out[start] = ord(">") if fmt == "fasta" else ord("@")
    out[start + 1] = ord("r")
    cols = np.arange(d.shape[1])
    mask = cols[None, :] < nd[:, None]
    out[(start[:, None] + 2 + cols[None, :])[mask]] = d[mask]
    out[start + 2 + nd] = 10
    seq = start + hdr
    if fmt == "fasta":
        k = -(-L // width) if width else np.ones(n, np.int64)
        w = width or int(L.max())
        read = np.repeat(np.arange(n), k)
        line = np.arange(int(k.sum())) - np.repeat(np.cumsum(k) - k, k)
        out[seq[read] + line * (w + 1) + np.minimum(w, L[read] - line * w)] = 10
    else:
        out[seq + L] = 10
        out[seq + L + 1] = ord("+")
        out[seq + L + 2] = 10
        out[seq + 2 * L + 3] = 10


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--width", type=int, default=80, help="FASTA line width (0: unwrapped)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from rala_b200 import api, synth
    from tests import reads_oracle as R

    t0 = time.perf_counter()
    ds = synth.generate(100_000_000, 40, 10000, seed=3)
    names = [b"r%d" % i for i in range(ds.n_reads)]
    small = ds.read_len[:50]
    for fmt in ("fasta", "fastq"):   # the formatter gives what the contract reads back
        buf = np.zeros(reads_layout(small, fmt, args.width or None)[2], np.uint8)
        format_reads(small, fmt, buf, args.width or None)
        blob, _, lens, _ = R.read(buf.tobytes())
        assert blob == b"".join(names[:50]) and np.array_equal(lens, small), fmt
    paf = format_paf(ds.read_len, ds.records)
    prep_s = time.perf_counter() - t0
    peak, peak_src = bench.measured_peaks()

    ctx = api.Context(0)
    G = api.Graph(ctx)
    res = {"metric": "fasta_text_bytes_per_sec", "unit": "B/s", "higher_is_better": True, "card": card(),
           "workload": "configs[2] read set: synth.generate(100_000_000, 40, 10000, seed=3)",
           "counts": {"n_reads": ds.n_reads, "n_bases": int(ds.read_len.astype(np.int64).sum()), "paf_bytes": len(paf),
                      "fasta_width": args.width or None, "prep_s": prep_s}}
    for fmt in ("fasta", "fastq"):
        t0 = time.perf_counter()
        total = reads_layout(ds.read_len, fmt, args.width or None)[2]
        pinned = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        text = pinned.numpy()
        format_reads(ds.read_len, fmt, text, args.width or None)
        gen_s = time.perf_counter() - t0
        # CPU: the plain-C reader on one core
        t0 = time.perf_counter()
        wblob, wends, wlens, wst = R.read(text, cap=ds.n_reads + 1)
        cpu_s = time.perf_counter() - t0
        assert np.array_equal(wlens, ds.read_len) and wblob == b"".join(names)
        # the call from pinned host text (it synchronises) next to a plain copy of the same bytes
        dev = torch.empty(total, dtype=torch.uint8, device="cuda")
        call, copy, kern = [], [], []
        for _ in range(args.repeats + 1):
            ctx.synchronize()
            t0 = time.perf_counter()
            st = G.set_reads_text(pinned)
            call.append(time.perf_counter() - t0)
            kern.append(st["device_ms"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev.copy_(pinned, non_blocking=True)
            torch.cuda.synchronize()
            copy.append(time.perf_counter() - t0)
        call, copy, kern = call[1:], copy[1:], kern[1:]
        del dev
        gblob, gends, glens = G.reads()
        parity = bool(bytes(gblob) == wblob and np.array_equal(gends, wends) and np.array_equal(glens, wlens)
                      and all(st[k] == v for k, v in wst.items()))
        k_ms, c_ms, u_ms = float(np.median(kern)), 1e3 * float(np.median(call)), 1e3 * float(np.median(copy))
        # bytes the kernels have to move at least: the text once, the line ends written and read (8 B per line)
        algo = total + 8 * st["n_lines"]
        res[fmt] = {"text_bytes": total, "n_lines": st["n_lines"], "n_chunks": st["n_chunks"], "parity_with_c_reader": parity,
                    "kernel_ms": k_ms, "kernel_repeats_ms": kern, "text_gbs": total / (k_ms * 1e-3) / 1e9,
                    "algorithmic_bytes": algo, "frac_of_hbm_bound": algo / (k_ms * 1e-3) / 1e9 / peak,
                    "call_ms": c_ms, "call_runs_ms": [1e3 * x for x in call], "copy_ms": u_ms,
                    "copy_runs_ms": [1e3 * x for x in copy], "call_over_copy": c_ms / u_ms,
                    "c_reader_one_core_s": cpu_s, "gen_s": gen_s}
        if fmt == "fasta":
            res["value"] = total / (k_ms * 1e-3)
            fasta_pinned = pinned
        else:
            del pinned, text
    res["hbm_peak_gbs"], res["peak_source"] = peak, peak_src
    res["call_note"] = ("host wall clock around set_reads_text from pinned host memory (the call synchronises); the copy is a "
                        "host-to-device copy of the same pinned bytes into device memory, timed to a device synchronise")

    # a full step from text, parity-gated against the session fed the synth names and lengths with the same PAF text
    ppaf = torch.frombuffer(bytearray(paf), dtype=torch.uint8).pin_memory()
    del paf
    H = api.Graph(ctx)
    H.set_reads(names, ds.read_len).set_overlaps_paf(ppaf)
    H.build_piles()
    H.set_hills(None).run()
    want_edges, want_marked, want_med = H.edges(), H.marked(), H.medians()
    steps = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        G.set_reads_text(fasta_pinned)
        G.set_overlaps_paf(ppaf)
        G.build_piles()
        G.set_hills(None).run()
        c = G.counts()
        steps.append(time.perf_counter() - t0)
    steps = steps[1:]
    parity = bool(np.array_equal(G.edges(), want_edges) and np.array_equal(G.marked(), want_marked)
                  and np.array_equal(G.medians(), want_med))
    res["parity"] = parity and res["fasta"]["parity_with_c_reader"] and res["fastq"]["parity_with_c_reader"]
    res["step"] = {"fasta_plus_paf_to_marks_ms": 1e3 * float(np.median(steps)), "runs_ms": [1e3 * x for x in steps],
                   "edges": c["n_edges"], "transitive_pairs": c["n_transitive_pairs"], "parity_with_set_reads_session": parity}
    line = json.dumps(res)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_reads.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")
    G.close()
    H.close()
    ctx.close()
    if not res["parity"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
