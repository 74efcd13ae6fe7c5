"""Per-kernel device times of the flagship step (bench.py's workload), from torch.profiler's CUDA activity records.

    python profiles/kernel_times.py [--steps 20] [--libs product,prev] [--out FILE]

Each library (the product, and rala_b200/variants/librala_b200_<name>.so for the others) runs the eager chain (no CUDA
graph) `--steps` times under the profiler after a warm-up; the JSON gives the mean microseconds per step of every kernel
and memset.  Tracing slows the host, not the kernels: these are shares, the step time comes from bench.py.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--libs", default="product,prev")
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from rala_b200 import api, build as B
    ds = bench.make_dataset(args.workload, 1)
    piles = ds.flat_piles()
    result = {}
    for name in args.libs.split(","):
        path = api.LIB_PATH if name == "product" else B.variant_path(name)
        if not os.path.exists(path):
            continue
        ctx = api.Context(0, lib=api.load_path(path))
        G = api.Graph(ctx)
        G.set_piles(piles).set_hills(None).set_overlaps(ds.records)
        G.use_cuda_graph(False)
        for _ in range(3):
            G.run()
        ctx.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                G.run()
            ctx.synchronize()
        acc = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                acc.setdefault(ev.name, [0.0, 0])
                acc[ev.name][0] += ev.device_time
                acc[ev.name][1] += 1
        result[name] = {k: {"us_per_step": round(v[0] / args.steps, 2), "launches_per_step": v[1] / args.steps}
                        for k, v in sorted(acc.items(), key=lambda kv: -kv[1][0])}
        G.close()
        ctx.close()
    text = json.dumps({"steps": args.steps, "workload": bench.WORKLOADS[args.workload][3], "kernels": result}, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
