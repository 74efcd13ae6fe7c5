"""The pile table from the overlap records on one B200 (Graph::initialize's coverage half), on bench.py's default workload
(c3 = configs[2]) built as bench_paf.py builds it.

    python bench_piles.py [--out FILE] [--repeats 3]

Prints one JSON line and writes it to profiles/<next free r02 tag>_bench_piles.json (or --out):
  - kernel time of rala_b200_build_piles (events, radix sort, walk; uploads excluded) and the bytes the algorithm moves
    (events written, sorted and scanned) as a share of the HBM bound;
  - the call from host columns (PCIe and the download of piles and medians included);
  - a text -> set_overlaps_paf -> build_piles -> run step, parity-gated: the device piles and medians equal the plain-C
    restatement (tests/piles_oracle.c), and the run's edges and marks equal a session fed the oracle's piles;
  - that restatement on one core of this host.
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

import bench  # noqa: E402
from bench_paf import card, format_paf, next_tag  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=list(bench.WORKLOADS))
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from rala_b200 import api
    from tests import piles_oracle as PO

    ds = bench.make_dataset(args.workload, 1)
    text = format_paf(ds.read_len, ds.records)
    names = [b"r%d" % i for i in range(ds.n_reads)]
    n_rec = ds.n_overlaps
    cols = PO.columns(ds.records)

    # CPU: the restatement on one core (the parity reference)
    t0 = time.perf_counter()
    o = PO.build_piles(cols, ds.read_len, runs=False)
    cpu_s = time.perf_counter() - t0

    ctx = api.Context(0)
    kern, call = [], []
    for _ in range(args.repeats + 1):
        t0 = time.perf_counter()
        piles, med, stats, ms = ctx.build_piles(cols, ds.read_len, with_time=True)
        call.append(time.perf_counter() - t0)
        kern.append(ms)
    kern, call = kern[1:], call[1:]
    parity_piles = bool(np.array_equal(piles, o["piles"]) and np.array_equal(med, o["medians"]) and stats == o["stats"])
    k_ms = float(np.median(kern))
    peak, peak_src = bench.measured_peaks()
    # bytes the algorithm moves: 4 events of 8 B per record written, then per radix pass every key read twice (histogram,
    # scatter) and written once, then read once by the walk, which writes 6 B per run and 10 B per read
    n_keys = 4 * n_rec
    pbits = int(2 * int(ds.read_len.max()) + 1).bit_length()
    passes = (int(ds.n_reads).bit_length() + pbits + 7) // 8
    model = {"events_written": 8 * n_keys, "sorted": passes * 24 * n_keys, "walk": 8 * n_keys + 6 * stats["n_runs"] + 10 * ds.n_reads}
    total = sum(model.values())

    # text -> records -> device piles -> run, gated against a session fed the oracle's piles and the same records
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()
    G = api.Graph(ctx)
    G.set_reads(names, ds.read_len)
    H = api.Graph(ctx)
    H.set_reads(names, ds.read_len).set_overlaps_paf(pinned)
    H.set_piles(o["piles"]).set_hills(None).run()
    want_edges, want_marked = H.edges(), H.marked()
    G.set_overlaps_paf(pinned)
    G.build_piles()
    parity_table = bool(np.array_equal(G.piles(), o["piles"]))   # before the run: containment kills piles in the table
    steps = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        G.set_overlaps_paf(pinned)
        G.build_piles()
        G.set_hills(None).run()
        c = G.counts()
        steps.append(time.perf_counter() - t0)
    steps = steps[1:]
    parity_run = bool(parity_table and np.array_equal(G.edges(), want_edges) and np.array_equal(G.marked(), want_marked)
                      and np.array_equal(G.medians(), o["medians"]))
    # the same step with the table from the host (what a caller without build_piles runs after its host initialize())
    host = []
    for _ in range(args.repeats + 1):
        ctx.synchronize()
        t0 = time.perf_counter()
        H.set_overlaps_paf(pinned)
        H.set_piles(o["piles"]).set_hills(None).run()
        H.counts()
        host.append(time.perf_counter() - t0)
    host = host[1:]
    parity = parity_piles and parity_run

    res = {
        "metric": "build_piles_kernel_ms", "value": k_ms, "unit": "ms", "higher_is_better": False,
        "parity": parity, "parity_piles": parity_piles, "parity_run": parity_run, "card": card(),
        "workload": bench.WORKLOADS[args.workload][3],
        "counts": {"n_records": n_rec, "n_reads": ds.n_reads, "events": n_keys, "radix_passes": passes, "edges": c["n_edges"], **stats},
        "kernels": {"build_piles_ms": k_ms, "repeats_ms": kern, "algorithmic_bytes": model,
                    "achieved_gbs": total / (k_ms * 1e-3) / 1e9, "frac_of_hbm_bound": total / (k_ms * 1e-3) / 1e9 / peak,
                    "hbm_peak_gbs": peak, "peak_source": peak_src},
        "call": {"build_piles_from_host_columns_ms": 1e3 * float(np.median(call)), "runs_ms": [1e3 * x for x in call],
                 "note": "host wall clock around rala_b200_build_piles from pageable numpy columns: 24 B per record up, piles "
                         "and medians down"},
        "step": {"set_overlaps_paf_build_piles_run_ms": 1e3 * float(np.median(steps)), "runs_ms": [1e3 * x for x in steps],
                 "set_overlaps_paf_host_piles_run_ms": 1e3 * float(np.median(host)), "host_runs_ms": [1e3 * x for x in host]},
        "cpu": {"oracle_one_core_s": cpu_s, "host_cores_available": os.cpu_count(),
                "note": "tests/piles_oracle.c: per read, sorted bounds + the add_layers walk + region scan + counted median"},
    }
    line = json.dumps(res)
    print(line)
    out = args.out or os.path.join(ROOT, "profiles", next_tag() + "_bench_piles.json")
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
