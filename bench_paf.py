"""PAF text -> session records on one B200 (SURVEY.md 8(f) row 2), on bench.py's default workload (c3 = configs[2]).

    python bench_paf.py [--out FILE] [--repeats 3]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_paf.json (or --out):
  - kernel time of the parse stage (line scan + parse + name lookup: rala_b200_parse_paf's device time; duplicate filter:
    rala_b200_filter_duplicates' device time), text bytes per second and the share of the HBM bound on the bytes the
    stage has to move;
  - the call from pinned host text to the session's records (PCIe included) next to the 24-byte column upload of the
    same records;
  - a full set_overlaps_paf + run step, parity-gated against the session fed by set_overlaps_columns with the columns
    of the plain-C reader (tests/paf_oracle.c) and the oracle's duplicate filter;
  - that C reader on one core of this host.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import glob
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload generator and HBM peak of the main benchmark)

# BASELINE.md, measured by the survey on another host (one core): bioparser's PAF parse and transmute's name lookup
BASELINE_NS_PER_OVERLAP = {"parse": [490, 565], "transmute_lookup": [105, 127]}


def _digits(v: np.ndarray):
    """u32 -> (n, 10) ASCII digit matrix, left aligned, and the digit counts."""
    v = v.astype(np.int64)
    nd = np.ones(v.shape[0], np.int64)
    for p in range(1, 10):
        nd += v >= 10 ** p
    out = np.zeros((v.shape[0], 10), np.uint8)
    for j in range(10):
        p = np.maximum(nd - 1 - j, 0)
        out[:, j] = 48 + (v // 10 ** p) % 10
    return out, nd


def format_paf(read_len: np.ndarray, records: np.ndarray, block: int = 1 << 20) -> bytes:
    """synth.Dataset.write_paf's text, vectorised: "r<a>\\t<la>\\t<ab>\\t<ae>\\t<+|->\\tr<b>\\t<lb>\\t<bb>\\t<be>\\t<span>\\t<span>\\t255\\n"."""
    parts = []
    for s in range(0, records.shape[0], block):
        q = records[s:s + block]
        n = q.shape[0]
        span = np.maximum(q[:, 3] - q[:, 2], q[:, 5] - q[:, 4])
        fields = []
        for kind, v in (("r", q[:, 0]), ("n", read_len[q[:, 0]]), ("n", q[:, 2]), ("n", q[:, 3]), ("s", q[:, 6]), ("r", q[:, 1]),
                        ("n", read_len[q[:, 1]]), ("n", q[:, 4]), ("n", q[:, 5]), ("n", span), ("n", span), ("c", None)):
            if kind == "s":
                fields.append((np.where((v & 1) != 0, 45, 43).astype(np.uint8)[:, None], np.ones(n, np.int64)))
            elif kind == "c":
                fields.append((np.tile(np.frombuffer(b"255", np.uint8), (n, 1)), np.full(n, 3, np.int64)))
            else:
                d, nd = _digits(v)
                if kind == "r":
                    d, nd = np.concatenate([np.full((n, 1), 114, np.uint8), d], 1), nd + 1
                fields.append((d, nd))
        line_len = sum(nd + 1 for _, nd in fields)
        start = np.concatenate([[0], np.cumsum(line_len)[:-1]])
        out = np.empty(int(line_len.sum()), np.uint8)
        off = start.copy()
        for k, (d, nd) in enumerate(fields):
            cols = np.arange(d.shape[1])
            mask = cols[None, :] < nd[:, None]
            out[(off[:, None] + cols[None, :])[mask]] = d[mask]
            out[off + nd] = 10 if k == len(fields) - 1 else 9
            off = off + nd + 1
        parts.append(out.tobytes())
    return b"".join(parts)


def next_tag() -> str:
    tags = [m.group(1) for p in glob.glob(os.path.join(ROOT, "profiles", "r02*")) if (m := re.match(r"r02([a-z]{1,2})_", os.path.basename(p)))]
    last = max(tags, key=lambda t: (len(t), t)) if tags else "a"
    chars = list(last)
    i = len(chars) - 1
    while i >= 0 and chars[i] == "z":
        chars[i] = "a"
        i -= 1
    if i < 0:
        chars.insert(0, "a")
    else:
        chars[i] = chr(ord(chars[i]) + 1)
    return "r02" + "".join(chars)


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # the numbers below still stand; say what is missing
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=list(bench.WORKLOADS))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from oracle import oracle as O
    from rala_b200 import api, synth
    from tests import paf_oracle as P

    t0 = time.perf_counter()
    ds = bench.make_dataset(args.workload, 1)
    small = synth.Dataset(ds.read_len, ds.records[:2000], 0)
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        small.write_paf(os.path.join(tmp, "s.paf"))
        with open(os.path.join(tmp, "s.paf"), "rb") as f:
            assert f.read() == format_paf(ds.read_len, small.records), "vectorised formatter differs from synth.Dataset.write_paf"
    text = format_paf(ds.read_len, ds.records)
    names = [b"r%d" % i for i in range(ds.n_reads)]
    prep_s = time.perf_counter() - t0
    n_rec, n_bytes = ds.n_overlaps, len(text)

    # CPU: the plain-C reader on one core, then the oracle's filter for the parity gate
    t0 = time.perf_counter()
    ocols, ostats = P.parse(text, names, ds.read_len)
    cpu_parse_s = time.perf_counter() - t0
    assert ostats["n_records"] == n_rec and ostats["n_unresolved"] == 0
    valid = O.filter_duplicates(ocols[0], ocols[1], ocols[6]).astype(bool)
    oracle_columns = np.ascontiguousarray(ocols[:6].copy())
    oracle_columns[0] |= np.where(valid, 0, 0x80000000).astype(np.uint32)

    ctx = api.Context(0)
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
    del text

    # kernel time of the parse stage
    kern, filt = [], []
    for _ in range(args.repeats + 1):
        cols, stats, ms = ctx.parse_paf(pinned, names, ds.read_len, with_time=True)
        _, fms = ctx.filter_duplicates(cols[0], cols[1], cols[6], with_time=True)
        kern.append(ms)
        filt.append(fms)
    assert np.array_equal(cols, ocols), "device parse differs from the C reader"
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
        st = G.set_overlaps_paf(pinned)
        call.append(time.perf_counter() - t0)
    call = call[1:]
    pcols = torch.from_numpy(oracle_columns).pin_memory()
    H = api.Graph(ctx)
    up = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        H.set_overlaps_columns([pcols[k] for k in range(6)])
        ctx.synchronize()
        up.append(time.perf_counter() - t0)
    up = up[1:]

    # a full step from text, parity-gated against the session fed the oracle's columns
    piles = ds.flat_piles()
    H.set_piles(piles).set_hills(None).run()
    want_edges, want_marked = H.edges(), H.marked()
    steps = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        G.set_overlaps_paf(pinned)
        G.set_piles(piles).set_hills(None).run()
        c = G.counts()
        steps.append(time.perf_counter() - t0)
    steps = steps[1:]
    parity = bool(np.array_equal(G.edges(), want_edges) and np.array_equal(G.marked(), want_marked))

    res = {
        "metric": "paf_text_bytes_per_sec", "value": n_bytes / (k_ms * 1e-3), "unit": "B/s", "higher_is_better": True,
        "parity": parity, "card": card(), "workload": bench.WORKLOADS[args.workload][3],
        "counts": {"n_records": n_rec, "n_reads": ds.n_reads, "text_bytes": n_bytes, "bytes_per_line": n_bytes / n_rec,
                   "n_chunks": stats["n_chunks"], "edges": c["n_edges"], "prep_s": prep_s},
        "kernels": {"scan_parse_lookup_ms": k_ms, "filter_ms": f_ms, "stage_ms": stage_ms, "repeats_ms": kern,
                    "text_gbs": n_bytes / (k_ms * 1e-3) / 1e9,
                    "algorithmic_bytes": {"scan_parse_lookup": parse_bytes, "filter": filter_bytes},
                    "frac_of_hbm_bound": {"scan_parse_lookup": parse_bytes / (k_ms * 1e-3) / 1e9 / peak,
                                          "stage": (parse_bytes + filter_bytes) / (stage_ms * 1e-3) / 1e9 / peak},
                    "hbm_peak_gbs": peak, "peak_source": peak_src},
        "call": {"set_overlaps_paf_ms": 1e3 * float(np.median(call)), "runs_ms": [1e3 * x for x in call],
                 "set_overlaps_columns_ms": 1e3 * float(np.median(up)), "columns_bytes": 24 * n_rec,
                 "note": "host wall clock around the call from pinned host memory (it synchronises); the column upload is "
                         "timed to a stream synchronise"},
        "step": {"set_overlaps_paf_plus_run_ms": 1e3 * float(np.median(steps)), "runs_ms": [1e3 * x for x in steps]},
        "cpu": {"c_reader_one_core_s": cpu_parse_s, "c_reader_ns_per_overlap": 1e9 * cpu_parse_s / n_rec,
                "host_cores_available": os.cpu_count(),
                "survey_baseline_ns_per_overlap": BASELINE_NS_PER_OVERLAP,
                "survey_baseline_s_at_this_size": {k: [v[0] * n_rec * 1e-9, v[1] * n_rec * 1e-9] for k, v in BASELINE_NS_PER_OVERLAP.items()},
                "note": "the survey figures are bioparser + transmute as BASELINE.md measured them on another host, not re-measured here"},
    }
    line = json.dumps(res)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_paf.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(line + "\n")
    G.close()
    H.close()
    ctx.close()
    if not parity:
        sys.exit(1)


if __name__ == "__main__":
    main()
