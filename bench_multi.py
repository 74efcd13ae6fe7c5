"""bench_multi.py — the N > 1 leg of bench.py: one process per GPU (launched by torch.distributed.run), the
library's multi-GPU session through rala_b200.multi.FabricGraph, and the parity gate that checks the assembled
result of all ranks on rank 0 before a line is printed.  Bench infrastructure, not product code: the checker
imports the oracle here (the product package rala_b200/ never does)."""
from __future__ import annotations

import os
import time

import numpy as np
import torch
import torch.distributed as dist

from rala_b200 import api
from rala_b200.multi import CudaShardSession, DistributedGraph, FabricGraph, make_graph  # noqa: F401


# -------------------------------------------------------------------------------------------------------------
# bench entry (python -m torch.distributed.run ... bench.py --gpus N)
# -------------------------------------------------------------------------------------------------------------
def _global_dataset(args, rank, world, device):
    """Weak scaling: `world` chromosomes of the single-GPU workload; read ids are shuffled GLOBALLY, so every
    shard's records reference piles (and later CSR rows) owned by all the other shards.  Each rank generates
    one chromosome, then the records are redistributed by query-id range with an all-to-all (setup, untimed)."""
    import bench
    from rala_b200 import synth
    genome, cov, rl, _ = bench.WORKLOADS[args.workload]
    ds = synth.generate(genome, cov, rl, seed=3 + rank)
    n_chr = ds.n_reads
    n_total = n_chr * world
    perm = np.random.Generator(np.random.PCG64(12345)).permutation(n_total).astype(np.uint32)   # same on all ranks
    gid = perm[rank * n_chr:(rank + 1) * n_chr]
    rec = ds.records.copy()
    a, b = gid[rec[:, 0]], gid[rec[:, 1]]
    swap = a > b                                     # keep "listed once under the lower id as query"
    rec[:, 0], rec[:, 1] = np.where(swap, b, a), np.where(swap, a, b)
    ab, ae, bb, be = rec[:, 2].copy(), rec[:, 3].copy(), rec[:, 4].copy(), rec[:, 5].copy()
    rec[:, 2], rec[:, 3] = np.where(swap, bb, ab), np.where(swap, be, ae)
    rec[:, 4], rec[:, 5] = np.where(swap, ab, bb), np.where(swap, ae, be)
    # destination rank = owner of the query-id range; the ranges are cut so that every rank holds the same
    # number of RECORDS (pairs are listed under the lower id, so low ids own more records): contiguous
    # file ranges of equal length, the partition rala_b200.multi.shard_bounds describes
    hist = torch.from_numpy(np.bincount(rec[:, 0], minlength=n_total).astype(np.int64)).to(device)
    dist.all_reduce(hist, op=dist.ReduceOp.SUM)
    cum = torch.cumsum(hist, 0).cpu().numpy()
    cuts = np.searchsorted(cum, cum[-1] * np.arange(1, world) / world, side="left")   # last query id of ranks 0 .. world-2
    dest = np.searchsorted(cuts, rec[:, 0], side="left").astype(np.int64)
    order = np.argsort(dest, kind="stable")
    rec = rec[order]
    send_counts = np.bincount(dest, minlength=world).astype(np.int64)
    sc = torch.tensor(send_counts, device=device)
    rc = torch.empty_like(sc)
    dist.all_to_all_single(rc, sc)
    send = torch.from_numpy(rec.view(np.int32)).to(device)
    recv = torch.empty((int(rc.sum().item()), 7), dtype=torch.int32, device=device)
    dist.all_to_all_single(recv, send, output_split_sizes=rc.tolist(), input_split_sizes=sc.tolist())
    local = recv.cpu().numpy().view(np.uint32)
    local = local[np.lexsort((local[:, 2], local[:, 1], local[:, 0]))]     # grouped by query, ascending
    # replicated pile table: read lengths of every chromosome (fixed-length reads here) at their global ids
    lens = torch.zeros(n_total, dtype=torch.int32, device=device)
    lens[torch.from_numpy(gid.astype(np.int64)).to(device)] = torch.from_numpy(ds.read_len.astype(np.int32)).to(device)
    dist.all_reduce(lens, op=dist.ReduceOp.SUM)
    read_len = lens.cpu().numpy().astype(np.uint32)
    piles = np.empty((n_total, 2), dtype=np.uint32)
    piles[:, 0] = 15
    piles[:, 1] = read_len - 15
    counts = torch.tensor([local.shape[0]], dtype=torch.int64, device=device)
    allc = [torch.empty_like(counts) for _ in range(world)]
    dist.all_gather(allc, counts)
    allc = [int(c.item()) for c in allc]
    t0 = sum(allc[:rank])
    return np.ascontiguousarray(local), piles, t0, sum(allc)


def verify_against_single_gpu_and_oracle(records, piles, flags, edges, marked, device_index: int, oracle_max_records: int):
    """Rank 0, outside every timed region: the edge list + removed-edge set assembled from all ranks must be
    bit-identical to (a) the single-GPU session of this library on the whole batch, which the GPU suite pins against
    the oracle at this size, and (b) the plain-C oracle itself when the batch is small enough to finish in about a
    minute.  Returns the `parity` object of the bench line; raises on a mismatch."""
    import zlib
    out = {"edges": int(edges.shape[0]), "marks_crc32": zlib.crc32(marked.tobytes(), zlib.crc32(edges.tobytes()))}
    ctx = api.Context(device_index)
    G = api.Graph(ctx)
    G.set_piles(piles, flags).set_hills(None).set_overlaps(records)
    G.run()
    e1, m1 = G.edges(), G.marked()
    G.close()
    ctx.close()
    if not (np.array_equal(e1, edges) and np.array_equal(m1, marked)):
        raise api.RalaB200Error(f"multi-GPU result differs from the single-GPU session on the same batch "
                                f"({edges.shape[0]} vs {e1.shape[0]} edges)")
    out["vs_single_gpu_same_batch"] = True
    if records.shape[0] <= oracle_max_records:
        from oracle import oracle as O   # bench.py's checker leg: the oracle is never on the measured path
        t0 = time.perf_counter()
        P = O.Pipeline(records, piles, flags).run()
        if not (np.array_equal(P.edges, edges) and np.array_equal(P.marked, marked)):
            raise api.RalaB200Error("multi-GPU result differs from the oracle")
        out["vs_oracle"] = True
        out["oracle_seconds"] = round(time.perf_counter() - t0, 2)
    else:
        out["vs_oracle"] = f"skipped: {records.shape[0]} records > {oracle_max_records} (the single-GPU session is pinned against the oracle)"
    return out


def _share_through_files(rank, world, arrays: dict):
    """Single node: every rank leaves its arrays in a directory rank 0 names; rank 0 reads them all back."""
    import shutil
    import tempfile
    plumbing = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    need = torch.tensor([sum(int(v.nbytes) for v in arrays.values())], dtype=torch.int64, device=plumbing)
    dist.all_reduce(need)
    where = None
    if rank == 0:   # the RAM disk when it has room for everything (it is often only 64 MB inside a container), else the default temp dir
        for cand in ("/dev/shm", tempfile.gettempdir()):
            if os.path.isdir(cand) and shutil.disk_usage(cand).free > 1.2 * int(need.item()) + (64 << 20):
                where = cand
                break
    box = [tempfile.mkdtemp(prefix="rala_b200_", dir=where) if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    for k, v in arrays.items():
        np.save(os.path.join(box[0], f"{k}_{rank}.npy"), v)
    dist.barrier()
    got = None
    if rank == 0:
        got = {k: [np.load(os.path.join(box[0], f"{k}_{r}.npy")) for r in range(world)] for k in arrays}
        shutil.rmtree(box[0], ignore_errors=True)
    dist.barrier()
    return got


def bench_main(args):
    import json
    import bench

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    # a rank stuck in a collective (a peer died) must not hold N GPUs until somebody else's time limit
    import threading
    watchdog = threading.Timer(1500.0, lambda: os._exit(3))
    watchdog.daemon = True
    watchdog.start()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)
    records, piles, t0, n_total_records = _global_dataset(args, rank, world, device)
    steps, warmup = args.steps, max(args.warmup, 3)

    kind, dg = make_graph(local_rank, rank, world, records, piles, None, t0)
    if kind == "fabric":
        dg.plan()
        run, sync, launches_now = dg.run, dg.M.synchronize, (lambda: dg.M.launch_count)
    else:
        sess = dg.s
        run, sync, launches_now = dg.run, (lambda: torch.cuda.synchronize()), (lambda: sess.ctx.launch_count)
    for _ in range(warmup + 2):   # eager, capture, replays
        run()
    sync()
    sampler = bench.ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = launches_now()
    dist.barrier()
    torch.cuda.synchronize()
    t_wall = time.perf_counter()
    if kind == "fabric":
        dg.M.event_record(0)
        for _ in range(steps):
            run()
        dg.M.event_record(1)
        dev_ms = dg.M.event_elapsed_ms()
    else:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            run()
        ev1.record()
        torch.cuda.synchronize()
        dev_ms = ev0.elapsed_time(ev1)
    sync()
    dist.barrier()
    wall_ms = 1e3 * (time.perf_counter() - t_wall)
    launches = launches_now() - launches0
    t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)           # max over ranks
    ms_per_step = float(t[0].item()) / steps
    clocks = sampler.stop() if sampler else None

    # ---- results of the timed steps: validity, then parity (outside the timed region) -----------------------------
    if kind == "fabric":
        c = dg.check()                                  # raises if a step did not fit its buffers / rounds
        (first, n_mine), e_mine, m_mine = dg.edges()
        E = c["n_edges"]
        sums = torch.tensor([c["n_two_hop"], c["n_transitive_pairs"], c["n_candidates"], c["n_final_candidates"]],
                            dtype=torch.int64, device=device)
        dist.all_reduce(sums)
        n_two_hop, n_pairs, n_events, n_final_events = [int(x) for x in sums.tolist()]
        n_nodes, rounds = c["n_nodes"], [c["n_rounds"], c["n_final_rounds"]]
    else:
        if not dg.check():
            raise api.RalaB200Error("a capacity-bounded exchange overflowed during the timed region")
        c = sess.counts()
        E, n_nodes, n_pairs, n_two_hop = c["n_edges"], c["n_nodes"], c["n_transitive_pairs"], c["n_two_hop"]
        # the imported event lists are every rank's: these counts are totals over the ranks
        n_events, n_final_events, rounds = c["n_candidates"], c["n_final_candidates"], [c["n_rounds"], c["n_final_rounds"]]
        first = 0
        e_mine, m_mine = (sess.edges(), sess.marked()) if rank == 0 else (np.zeros((0, 3), np.uint32), np.zeros(0, np.uint8))
    parity = None
    if not args.skip_parity:
        got = _share_through_files(rank, world, {"rec": records, "edges": e_mine, "marked": m_mine,
                                                 "first": np.array([first], np.int64)})
        if rank == 0:
            order = np.argsort([int(f[0]) for f in got["first"]], kind="stable") if kind == "fabric" else [0]
            edges = np.concatenate([got["edges"][r] for r in order])
            marked = np.concatenate([got["marked"][r] for r in order])
            assert edges.shape[0] == E, (edges.shape, E)
            parity = verify_against_single_gpu_and_oracle(np.concatenate(got["rec"]), piles, None, edges, marked, local_rank,
                                                          args.parity_oracle_max)
            del got
        dist.barrier()

    # ---- stage times of one eager step (CUDA events between the kernels do not exist inside a graph) ---------------
    if kind == "fabric":
        dg.M.use_cuda_graph(False)
        for _ in range(2):
            run()
        sync()
        stage = dg.M.stage_ms(0)
        dg.M.use_cuda_graph(True)
    else:
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        stage = sess.G.stage_ms()

    # ---- end to end: pinned host shard -> device, one step, the edges this rank emitted + their marks back ---------
    cols_pin = torch.from_numpy(api.records_to_columns(records)).pin_memory()   # 24 B / record, the device layout
    packed = api.records_to_packed(records) if kind == "fabric" else None       # 12 B / record when coordinates fit 16 bits
    ok = torch.tensor([0 if packed is None else 1], dtype=torch.int32, device=device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    packed_pin = packed.pin() if int(ok.item()) else None
    piles_pin = torch.from_numpy(piles).pin_memory()
    e2e_steps = max(3, min(steps, 10))
    n_out = max(int(e_mine.shape[0]), 1) if kind == "fabric" else max(E, 1)
    edges_pin = torch.empty((n_out, 3), dtype=torch.int32).pin_memory()
    marked_pin = torch.empty(n_out, dtype=torch.uint8).pin_memory()
    if kind == "fabric":
        dg.M.set_outputs(0, edges_pin, marked_pin)

        def e2e_step():
            dg.M.set_piles(piles_pin)
            if packed_pin is not None:
                dg.M.set_overlaps_packed(0, packed_pin, t0)
            else:
                dg.M.set_overlaps_columns(0, cols_pin, t0)
            dg.M.run()
            dg.M.synchronize()           # edges_pin / marked_pin are complete
    else:
        def e2e_step():
            sess.G.set_piles(piles_pin).set_overlaps_columns(cols_pin)
            dg.run()
            if rank == 0:                # the result is replicated: one download
                sess.G.edges(out=edges_pin)
                sess.G.marked(out=marked_pin)
            torch.cuda.synchronize()
    for _ in range(4):                   # new shape: eager, capture, replay
        e2e_step()
    dist.barrier()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    dist.barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t1) / e2e_steps], dtype=torch.float64, device=device)
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    if kind == "fabric":
        dg.check()
        assert np.array_equal(edges_pin.numpy().view(np.uint32)[:e_mine.shape[0]], e_mine) and \
            np.array_equal(marked_pin.numpy()[:m_mine.shape[0]], m_mine), "e2e outputs differ from the resident run"
        dg.M.set_outputs(0, None, None)

    if rank == 0:
        peak, peak_src = bench.measured_peaks()
        k1_ms = stage["k1_classify_kernel"] + stage["k1_survivors_kernel"]   # both passes over the shard, as at N = 1
        k1_gbs = bench.K1_BYTES_PER_OVERLAP * records.shape[0] / (k1_ms * 1e-3) / 1e9 if k1_ms > 0 else 0.0
        step_bytes = (bench.K1_BYTES_PER_OVERLAP * n_total_records + bench.K3_BYTES_PER_VISIT * n_two_hop + 9 * E + 8 * n_nodes
                      + 20 * (n_events + n_final_events) + 4 * int(piles.shape[0]) * world + 73 * E)
        agg_gbs = step_bytes / (ms_per_step * 1e-3) / 1e9
        parallelism = (f"{world} GPUs: records by file range; containment events to the victim's owner, edges to the source node's "
                       "owner, CSR slices pushed to every replica, marks back to the emitting rank: all as kernels storing into "
                       "peer memory (NVLink, CUDA IPC) between device-side barriers" if kind == "fabric" else
                       f"{world} GPUs, NCCL fallback: records by file range, CSR replicated (all-gather), marks all-reduce(max)")
        print(json.dumps({
            "metric": "graph_edges_per_sec", "value": E / (ms_per_step * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": bench.workload_config(args.workload, world),
            "counts": {"n_overlaps": n_total_records, "n_overlaps_per_gpu": int(records.shape[0]), "n_reads": int(piles.shape[0]),
                       "edges": E, "nodes": n_nodes, "two_hop_visits": n_two_hop, "transitive_pairs": n_pairs,
                       "containment_events": n_events, "final_containment_events": n_final_events, "resolution_rounds": rounds,
                       "parallelism": parallelism, "transport": kind,
                       "record_bytes_streamed_per_rank_per_step": int(records.nbytes * 6 // 7),
                       "step_graph": "one CUDA graph per rank and step (kernels only: the exchanges are kernels)" if kind == "fabric"
                                     else "eager (NCCL collectives between the phases)",
                       "exchange_capacities": dict(zip(api.CAP_NAMES, [int(x) for x in dg.caps])) if kind == "fabric" else dg.caps},
            "parity": parity,
            "wall_ms_per_step": float(t[1].item()) / steps,
            "e2e": {"value": E / e2e_s, "unit": "edges/s", "h2d_bytes_per_step": int(((packed_pin.nbytes if packed_pin is not None else cols_pin.numel() * 4) + piles.nbytes) * world),
                    "d2h_bytes_per_step": int(13 * E) if kind == "fabric" else int(13 * E), "ms_per_step": 1e3 * e2e_s,
                    "path": "per rank: set_piles + " + ("set_overlaps_packed (pinned, 12 B/record)" if packed_pin is not None else "set_overlaps_columns (pinned, 24 B/record)") + " + run + the rows / marks of the edges the rank emitted "
                            "written to pinned host memory by the GPU + synchronize"},
            "gpu_launches": int(launches) * (world if kind == "fabric" else 1),
            "roofline": {"bound": "hbm", "kernel": "k_classify_first", "achieved": k1_gbs, "peak": peak, "unit": "GB/s",
                         "frac": k1_gbs / peak, "traffic": None, "peak_source": peak_src,
                         "note": "rank 0's two passes over its record shard (events + survivors kernels); stage_ms are rank 0's eager step",
                         "aggregate_whole_step": {"algorithmic_bytes": int(step_bytes), "gbs": agg_gbs, "peak_gbs": peak * world,
                                                  "frac": agg_gbs / (peak * world)},
                         "stage_ms": stage},
            "cpu_baseline": None, "clocks": clocks,
        }))
    dist.barrier()
    dg.close() if kind == "fabric" else sess.close()
    dist.destroy_process_group()
