"""Staged construct (pile tables that change between the passes) on one GPU and on several ranks.

    python bench_staged.py [--scale 2] [--world N] [--repeats 3]

Builds a chimeric dataset (tests/test_chimeric_path.py's builder on a synth genome `scale` times the size of its
`chimeras_repeats` set), then drives Graph::construct's flow with the deterministic PileDriver stand-in for the host's
Pile calls: once through the single-GPU session (api.Graph.construct + remove_transitive_edges) and once through the
multi-GPU session (api.Multi.construct) with `world` ranks, one per GPU when there are that many, otherwise sharing
device 0.  Prints one JSON line with what it measures, named for what it is:
  host_ms          per staged call, a host clock around the call and a device synchronise (so it includes the launch and
                   copy overhead of the call: device kernel time alone is not measured here)
  round_trips      staged calls and pile-op calls per construct (each one waits for the device)
  device_used_mb   device memory in use per GPU after the construct (cudaMemGetInfo: every process and every rank sharing
                   the GPU together; the library allocates with cudaMalloc, outside torch's allocator statistics)
  parity           edges, marks and final lists of the multi-GPU construct against the single session
The frozen one-step chain (bench_multi.py) is reported as "not measured" on a machine with one GPU.  Nothing is written
to the working tree.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # ranks sharing a GPU wait for each other inside kernels
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from rala_b200 import api, synth  # noqa: E402
from tests.test_chimeric_path import DATASETS, PileDriver, PileOps, chimeric_input  # noqa: E402


class Timed:
    """Wraps the staged calls of a session: wall time of each call up to a device synchronise."""

    CALLS = ("classify", "retrim", "retrim_promote", "finish", "finalize", "build", "transitive", "hill_coverage",
             "connections", "set_piles")

    def __init__(self, obj, sync):
        self.obj, self.sync, self.ms = obj, sync, {}
        for name in self.CALLS:
            if hasattr(obj, name):
                setattr(obj, name, self._wrap(name, getattr(obj, name)))

    def _wrap(self, name, fn):
        def call(*a, **k):
            self.sync()
            t = time.perf_counter()
            r = fn(*a, **k)
            self.sync()
            self.ms.setdefault(name, []).append((time.perf_counter() - t) * 1e3)
            return r
        return call

    def summary(self):
        return {k: {"calls": len(v), "host_ms_total": round(sum(v), 3), "host_ms_max": round(max(v), 3)} for k, v in self.ms.items()}


def mem_used_mb(devices):
    out = {}
    for d in sorted(set(devices)):
        free, total = torch.cuda.mem_get_info(d)
        out[str(d)] = round((total - free) / 2**20, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=2.0, help="genome size relative to the test set chimeras_repeats")
    ap.add_argument("--world", type=int, default=0, help="ranks of the multi-GPU run (default: the GPUs present, at least 2)")
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_staged.py measures on a B200: no CUDA device")
    n_gpus = torch.cuda.device_count()
    world = a.world or max(2, n_gpus)
    devices = list(range(world)) if n_gpus >= world else [0] * world
    kw, frac = DATASETS["chimeras_repeats"]
    kw = dict(kw, genome_len=int(kw["genome_len"] * a.scale))
    inp = chimeric_input(synth.generate(**kw), kw["seed"], hill_frac=frac)

    result = {"gpu": torch.cuda.get_device_name(0), "n_gpus": n_gpus, "world": world, "devices": devices,
              "n_records": int(inp.records.shape[0]), "n_piles": int(inp.piles.shape[0]), "n_hills": int(inp.hills.shape[0])}
    ctx = api.Context(0)
    single, multi = [], []
    for rep in range(a.repeats):
        G = api.Graph(ctx)
        tg = Timed(G, ctx.synchronize)
        ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), G.piles)
        t = time.perf_counter()
        G.construct(inp.records, inp.piles, inp.flags, inp.hills, pile_ops=ops)
        pairs = G.remove_transitive_edges()
        ctx.synchronize()
        single.append({"host_ms": round((time.perf_counter() - t) * 1e3, 3), "calls": tg.summary(),
                       "pile_op_calls": len(ops.calls), "device_used_mb": mem_used_mb([0])})
        want = dict(edges=G.edges(), marked=G.removed, lists=G.lists(), pairs=pairs)
        G.close()

        M = api.Multi(devices)
        tm = Timed(M, M.synchronize)
        ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), M.piles)
        t = time.perf_counter()
        M.construct(inp.records, inp.piles, inp.flags, inp.hills, pile_ops=ops)
        M.synchronize()
        wall = (time.perf_counter() - t) * 1e3
        edges, marked = M.all_edges()
        ovl, inl = M.lists()
        c = M.counts()
        runs = [int(M.edge_runs(k).shape[0]) for k in range(M.n_local)]
        multi.append({"host_ms_with_plan": round(wall, 3), "calls": tm.summary(), "pile_op_calls": len(ops.calls),
                      "round_trips": sum(v["calls"] for k, v in tm.summary().items()
                                                if k in ("classify", "retrim", "retrim_promote", "finish")),
                      "edge_runs_per_rank": runs, "device_used_mb": mem_used_mb(devices)})
        parity = {"edges": bool(np.array_equal(edges, want["edges"])), "marks": bool(np.array_equal(marked, want["marked"])),
                  "overlaps": bool(np.array_equal(ovl, want["lists"][0])), "internals": bool(np.array_equal(inl, want["lists"][1])),
                  "transitive_pairs": c["n_transitive_pairs"] == want["pairs"], "n_edges": int(edges.shape[0])}
        result.setdefault("parity", []).append(parity)
        M.close()
    result["single_gpu"] = single
    result["multi"] = multi
    result["frozen_bench_multi_step"] = "not measured (one GPU)" if n_gpus < 2 else "run bench_multi.py"
    result["note"] = ("host_ms: host clock around staged calls that end in a device synchronise, not device kernel time; "
                      "device_used_mb: device-wide, after the construct, not a per-rank peak")
    print(json.dumps(result))
    if not all(all(v for k, v in p.items() if k != "n_edges") for p in result["parity"]):
        raise SystemExit("parity failed")


if __name__ == "__main__":
    main()
