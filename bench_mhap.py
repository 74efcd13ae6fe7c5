"""MHAP text -> session records on one B200 (SURVEY.md 8(f) row 2), on bench.py's default workload (c3 = configs[2]).

    python bench_mhap.py [--out FILE] [--repeats 3]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_mhap.json (or --out):
  - kernel time of the parse stage (line scan + parse: rala_b200_parse_mhap's device time; duplicate filter:
    rala_b200_filter_duplicates' device time), text bytes per second and the share of the HBM bound on the bytes the
    stage has to move (the accounting of bench_paf.py);
  - the call from pinned host text to the session's records (PCIe included) next to the 24-byte column upload of the
    same records;
  - a full set_overlaps_mhap + build_piles + run step, parity-gated against set_overlaps_paf + build_piles + run on the
    PAF text of the same records (edges, marks, piles, medians), and the parsed columns against the plain-C reader
    (tests/mhap_oracle.c);
  - that C reader on one core of this host.
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


def format_mhap(read_len: np.ndarray, records: np.ndarray, block: int = 1 << 20) -> bytes:
    """synth.Dataset.write_mhap's text, vectorised: "<a+1> <b+1> 0.0 <span> 0 <ab> <ae> <la> <ori> <bb> <be> <lb>\\n"."""
    parts = []
    for s in range(0, records.shape[0], block):
        q = records[s:s + block]
        n = q.shape[0]
        span = np.maximum(q[:, 3] - q[:, 2], q[:, 5] - q[:, 4])
        fields = []
        for v in (q[:, 0] + 1, q[:, 1] + 1, b"0.0", span, b"0", q[:, 2], q[:, 3], read_len[q[:, 0]], q[:, 6] & 1, q[:, 4], q[:, 5],
                  read_len[q[:, 1]]):
            if isinstance(v, bytes):
                fields.append((np.tile(np.frombuffer(v, np.uint8), (n, 1)), np.full(n, len(v), np.int64)))
            else:
                fields.append(_digits(v))
        line_len = sum(nd + 1 for _, nd in fields)
        start = np.concatenate([[0], np.cumsum(line_len)[:-1]])
        out = np.empty(int(line_len.sum()), np.uint8)
        off = start.copy()
        for k, (d, nd) in enumerate(fields):
            cols = np.arange(d.shape[1])
            mask = cols[None, :] < nd[:, None]
            out[(off[:, None] + cols[None, :])[mask]] = d[mask]
            out[off + nd] = 10 if k == len(fields) - 1 else 32
            off = off + nd + 1
        parts.append(out.tobytes())
    return b"".join(parts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=list(bench.WORKLOADS))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import tempfile

    import torch
    from rala_b200 import api, synth
    from tests import mhap_oracle as M

    t0 = time.perf_counter()
    ds = bench.make_dataset(args.workload, 1)
    small = synth.Dataset(ds.read_len, ds.records[:2000], 0)
    with tempfile.TemporaryDirectory() as tmp:
        small.write_mhap(os.path.join(tmp, "s.mhap"))
        with open(os.path.join(tmp, "s.mhap"), "rb") as f:
            assert f.read() == format_mhap(ds.read_len, small.records), "vectorised formatter differs from synth.Dataset.write_mhap"
    text = format_mhap(ds.read_len, ds.records)
    names = [b"r%d" % i for i in range(ds.n_reads)]
    prep_s = time.perf_counter() - t0
    n_rec, n_bytes = ds.n_overlaps, len(text)

    # CPU: the plain-C reader on one core
    t0 = time.perf_counter()
    ocols, ostats = M.parse(text, ds.read_len)
    cpu_parse_s = time.perf_counter() - t0
    assert ostats["n_records"] == n_rec and ostats["n_length_mismatch"] == 0

    ctx = api.Context(0)
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
    del text
    paf_pinned = torch.frombuffer(bytearray(format_paf(ds.read_len, ds.records)), dtype=torch.uint8).pin_memory()

    # kernel time of the parse stage
    kern, filt = [], []
    for _ in range(args.repeats + 1):
        cols, stats, ms = ctx.parse_mhap(pinned, ds.read_len, with_time=True)
        _, fms = ctx.filter_duplicates(cols[0], cols[1], cols[6], with_time=True)
        kern.append(ms)
        filt.append(fms)
    columns_parity = bool(np.array_equal(cols, ocols))
    del ocols
    kern, filt = kern[1:], filt[1:]
    k_ms, f_ms = float(np.median(kern)), float(np.median(filt))
    peak, peak_src = bench.measured_peaks()
    # bytes the stage has to move at least: the text once, the line ends written and read, 29 B of columns per record;
    # the filter reads three columns and writes one byte
    parse_bytes = n_bytes + n_rec * (4 + 4 + 29)
    filter_bytes = n_rec * 13
    stage_ms = k_ms + f_ms

    # the call from pinned host text to the session's records, next to the column upload
    G = api.Graph(ctx)
    G.set_reads(names, ds.read_len)
    call = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        G.set_overlaps_mhap(pinned)
        call.append(time.perf_counter() - t0)
    call = call[1:]
    pcols = torch.from_numpy(np.ascontiguousarray(cols[:6])).pin_memory()
    H = api.Graph(ctx)
    up = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        H.set_overlaps_columns([pcols[k] for k in range(6)])
        ctx.synchronize()
        up.append(time.perf_counter() - t0)
    up = up[1:]
    H.close()

    # full steps from text, MHAP and PAF alternating on one session each, parity-gated against each other
    P = api.Graph(ctx)
    P.set_reads(names, ds.read_len)
    steps = {"mhap": [], "paf": []}
    out = {}
    for _ in range(args.repeats + 1):
        for fmt, S, src in (("mhap", G, pinned), ("paf", P, paf_pinned)):
            ctx.synchronize()
            t0 = time.perf_counter()
            getattr(S, "set_overlaps_" + fmt)(src)
            S.build_piles()
            S.set_hills(None).run()
            c = S.counts()
            steps[fmt].append(time.perf_counter() - t0)
            out[fmt] = (S.edges(), S.marked(), S.piles(), S.medians())
    steps = {k: v[1:] for k, v in steps.items()}
    step_parity = all(np.array_equal(x, y) for x, y in zip(out["mhap"], out["paf"]))
    parity = columns_parity and step_parity

    res = {
        "metric": "mhap_text_bytes_per_sec", "value": n_bytes / (k_ms * 1e-3), "unit": "B/s", "higher_is_better": True,
        "parity": parity, "parity_detail": {"columns_vs_c_reader": columns_parity, "step_vs_paf_text": step_parity},
        "card": card(), "workload": bench.WORKLOADS[args.workload][3],
        "counts": {"n_records": n_rec, "n_reads": ds.n_reads, "text_bytes": n_bytes, "bytes_per_line": n_bytes / n_rec,
                   "n_chunks": stats["n_chunks"], "n_query_rc": stats["n_query_rc"], "edges": c["n_edges"], "prep_s": prep_s},
        "kernels": {"scan_parse_ms": k_ms, "filter_ms": f_ms, "stage_ms": stage_ms, "repeats_ms": kern,
                    "text_gbs": n_bytes / (k_ms * 1e-3) / 1e9,
                    "algorithmic_bytes": {"scan_parse": parse_bytes, "filter": filter_bytes},
                    "frac_of_hbm_bound": {"scan_parse": parse_bytes / (k_ms * 1e-3) / 1e9 / peak,
                                          "stage": (parse_bytes + filter_bytes) / (stage_ms * 1e-3) / 1e9 / peak},
                    "hbm_peak_gbs": peak, "peak_source": peak_src},
        "call": {"set_overlaps_mhap_ms": 1e3 * float(np.median(call)), "runs_ms": [1e3 * x for x in call],
                 "set_overlaps_columns_ms": 1e3 * float(np.median(up)), "columns_bytes": 24 * n_rec,
                 "note": "host wall clock around the call from pinned host memory (it synchronises); the column upload is "
                         "timed to a stream synchronise"},
        "step": {"set_overlaps_mhap_build_piles_run_ms": 1e3 * float(np.median(steps["mhap"])),
                 "set_overlaps_paf_build_piles_run_ms": 1e3 * float(np.median(steps["paf"])),
                 "runs_ms": {k: [1e3 * x for x in v] for k, v in steps.items()},
                 "note": "the two steps alternate in one loop; PAF text of the same records is the parity reference"},
        "cpu": {"c_reader_one_core_s": cpu_parse_s, "c_reader_ns_per_overlap": 1e9 * cpu_parse_s / n_rec,
                "host_cores_available": os.cpu_count()},
    }
    line = json.dumps(res)
    print(line)
    path = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_mhap.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        f.write(line + "\n")
    G.close()
    P.close()
    ctx.close()
    if not parity:
        sys.exit(1)


if __name__ == "__main__":
    main()
