#!/usr/bin/env python
"""tests/quick_check.py — TEST INFRASTRUCTURE (uses the oracle as the checker): a GPU check that fits in seconds (no torch import): parity of the product library
against the oracle on a small noisy batch, then device-resident step times on a 20 Mbp batch.
Prints one JSON line."""
import json
import os
import sys
import time

T0 = time.time()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
from oracle import oracle as O  # noqa: E402
from rala_b200 import api, synth  # noqa: E402

out = {"libs": {}}
small = synth.generate(2_000_000, 30, 9000, len_sd=2500, seed=5, noise=40, dual=True)
sp = small.flat_piles()
P = O.Pipeline(small.records, sp).run()
big = synth.generate(int(sys.argv[1]) if len(sys.argv) > 1 else 20_000_000, 40, 10000, seed=3)
bp = big.flat_piles()
out["t_setup_s"] = round(time.time() - T0, 2)
r = {}
try:
    ctx = api.Context(0)
    G = api.Graph(ctx)
    for _ in range(3):   # eager, capture, replay
        G.set_piles(sp).set_hills(None).set_overlaps(small.records)
        G.run()
    ovl, inl = G.lists()
    r["parity"] = bool(np.array_equal(G.edges(), P.edges) and np.array_equal(G.marked(), P.marked)
                       and G.counts()["n_transitive_pairs"] == P.n_pairs and np.array_equal(ovl, P.ovl)
                       and np.array_equal(inl, P.int) and np.array_equal(G.piles(), P.piles))
    G.set_piles(bp).set_hills(None).set_overlaps(big.records)
    for _ in range(4):
        G.run()
    ctx.synchronize()
    ctx.event_record(0)
    for _ in range(50):
        G.run()
    ctx.event_record(1)
    r["ms_per_step"] = ctx.event_elapsed_ms() / 50
    r["edges"] = G.counts()["n_edges"]
    G.close()
    ctx.close()
except Exception as exc:   # noqa: BLE001
    r["error"] = f"{type(exc).__name__}: {exc}"
out["libs"]["product"] = r
out["t_s"] = round(time.time() - T0, 2)
print(json.dumps(out), flush=True)
