#!/usr/bin/env python
"""profiles/same_kernels.py [out.json] — the kernels one eager step of every driver launches, with this tree's library
and the parent commit's (rala_b200/variants/librala_b200_prev.so, built by profiles/build_prev.sh), on the same seeded
inputs, in one process.  For each driver and library: kernel names in launch order (CUDA correlation id, from a
torch.profiler trace) and the library's launch-count delta.  A refactor of the drivers must leave both equal; kernels
without a data dependence between them may change places, so the multiset of names is compared as well.

Drivers: Graph.run eager on configs[2]; Context.transitive_reduce on the 60 000-spoke star of test_transitive_paths;
Multi world 2 on one device (run, and the staged construct); the NCCL fallback's phase calls at world 1, where an
all-gather of one block is the block and the all-reduce of the marks is the identity."""
import ctypes as C
import json
import os
import sys
import tempfile
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # two ranks of the multi-GPU session share one device
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from rala_b200 import api  # noqa: E402
from rala_b200 import build as B  # noqa: E402
from tests.test_transitive_paths import star_graph  # noqa: E402


def kernels_of(step, counter):
    """Run step() once under the profiler: (kernel names in launch order, launch-count delta)."""
    torch.cuda.synchronize()
    n0 = counter()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    delta = counter() - n0
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    ks = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["args"]["correlation"])
    return [e["name"].split("(")[0].replace("void ", "") for e in ks], delta


def single(lib, ds):
    ctx = api.Context(0, lib=lib)
    G = api.Graph(ctx)
    G.set_piles(ds.flat_piles()).set_hills(None).set_overlaps(ds.records)
    G.use_cuda_graph(False)
    G.run()
    out = kernels_of(G.run, lambda: ctx.launch_count)
    G.close()
    ctx.close()
    return out


def reduce(lib, n, e):
    ctx = api.Context(0, lib=lib)
    ctx.transitive_reduce(n, e)
    out = kernels_of(lambda: ctx.transitive_reduce(n, e), lambda: ctx.launch_count)
    ctx.close()
    return out


def multi(lib, ds, staged):
    M = api.Multi([0, 0], lib=lib)
    M.set_barrier_timeout_ms(20000)
    M.use_cuda_graph(False)
    M.set_piles(ds.flat_piles()).set_shards(ds.records).plan()

    def step():
        if staged:   # the staged construct with a frozen pile table (the list passes skip themselves)
            M.classify().retrim().retrim_promote()
            M.finish()
        else:
            M.run()

    step()
    out = kernels_of(step, lambda: M.launch_count)
    M.close()
    return out


def nccl_world1(lib, ds):
    ctx = api.Context(0, lib=lib)
    G = api.Graph(ctx)
    G.set_piles(ds.flat_piles()).set_hills(None).set_overlaps(ds.records)
    G._call("rala_b200_graph_set_shard", C.c_uint32(0), C.c_int(0), C.c_int(1))
    cap = len(ds.records) + 4096
    blk = [torch.zeros(int(lib.rala_b200_exchange_block_words(C.c_int(k), C.c_uint32(c))), dtype=torch.int32, device="cuda")
           for k, c in ((0, cap), (0, cap), (1, 2 * cap))]
    pair = torch.zeros(2, dtype=torch.int32, device="cuda")
    marks = torch.zeros(2 * cap, dtype=torch.uint8, device="cuda")
    dp = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731

    def step():
        torch.cuda.synchronize()   # the library enqueues on its own stream
        G._call("rala_b200_graph_phase_events")
        G._call("rala_b200_graph_export_padded", C.c_int(0), dp(blk[0]), C.c_uint32(cap))
        G._call("rala_b200_graph_import_gathered", C.c_int(0), dp(blk[0]), C.c_uint32(cap), C.c_int(1))
        G._call("rala_b200_graph_phase_resolve", C.c_int(1))
        G._call("rala_b200_graph_phase_survivors")
        G._call("rala_b200_graph_export_list_counts", dp(pair))
        G._call("rala_b200_graph_phase_final_events_gathered", dp(pair), C.c_int(1))
        G._call("rala_b200_graph_export_padded", C.c_int(0), dp(blk[1]), C.c_uint32(cap))
        G._call("rala_b200_graph_import_gathered", C.c_int(0), dp(blk[1]), C.c_uint32(cap), C.c_int(1))
        G._call("rala_b200_graph_phase_resolve", C.c_int(0))
        G._call("rala_b200_graph_phase_emit_edges")
        G._call("rala_b200_graph_export_padded", C.c_int(1), dp(blk[2]), C.c_uint32(2 * cap))
        G._call("rala_b200_graph_import_gathered", C.c_int(1), dp(blk[2]), C.c_uint32(2 * cap), C.c_int(1))
        G._call("rala_b200_graph_phase_csr")
        G._call("rala_b200_graph_phase_transitive")
        G._call("rala_b200_graph_export_marks", dp(marks), C.c_uint32(marks.shape[0]))
        G._call("rala_b200_graph_phase_marks", dp(marks), C.c_uint32(marks.shape[0]))
        ctx.synchronize()

    step()
    out = kernels_of(step, lambda: ctx.launch_count)
    e, m = G.edges(), G.marked()
    G.close()
    ctx.close()
    return out, e, m


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    libs = {"product": api.load_path(api.LIB_PATH), "prev": api.load_path(B.variant_path("prev"))}
    c3 = bench.make_dataset("c3", 1)
    small = bench.make_dataset("c1", 1)
    n, e, _ = star_graph(1, 60_000, 1000, seed=1)
    res = {"gpu": torch.cuda.get_device_name(0), "drivers": {}}
    nccl_out = {}
    for name, lib in libs.items():
        runs = {
            "graph_run_eager_c3": single(lib, c3),
            "transitive_reduce_star60000": reduce(lib, n, e),
            "multi_world2_run": multi(lib, small, False),
            "multi_world2_construct": multi(lib, small, True),
        }
        (k, d), edges, marked = nccl_world1(lib, c3)
        runs["nccl_phases_world1_c3"] = (k, d)
        nccl_out[name] = (edges, marked)
        for drv, (k, d) in runs.items():
            res["drivers"].setdefault(drv, {})[name] = {"launch_count_delta": d, "kernels": k}
    for drv, v in res["drivers"].items():
        a, b = v["product"], v["prev"]
        v["same_order"] = a["kernels"] == b["kernels"]
        v["same_multiset"] = Counter(a["kernels"]) == Counter(b["kernels"])
        v["same_launch_count"] = a["launch_count_delta"] == b["launch_count_delta"]
        v["n_kernels"] = len(a["kernels"])
        if not v["same_order"]:
            v["moved"] = [(i, x, y) for i, (x, y) in enumerate(zip(a["kernels"], b["kernels"])) if x != y]
    res["nccl_world1_same_edges_and_marks"] = bool(np.array_equal(nccl_out["product"][0], nccl_out["prev"][0]) and
                                                   np.array_equal(nccl_out["product"][1], nccl_out["prev"][1]))
    text = json.dumps(res, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text)
    summary = {d: {k: v[k] for k in ("n_kernels", "same_order", "same_multiset", "same_launch_count", "moved") if k in v}
               for d, v in res["drivers"].items()}
    print(json.dumps({"summary": summary, "nccl_same_results": res["nccl_world1_same_edges_and_marks"]}, indent=1))


if __name__ == "__main__":
    main()
