"""GPU suite: one PROCESS per rank, against the single-process oracle.

  fabric  the product path (rala_b200.multi.FabricGraph): the library's multi-GPU session, arenas mapped between the
          processes with CUDA IPC, exchanges as kernels over peer memory.  world = 1, 2, 4, 8 with one GPU per rank
          (skipped when the box has fewer), plus world = 2 with BOTH processes on device 0 (CUDA IPC works between
          processes on one device too; the kernels of the two processes are time-sliced, so this is slow but it
          exercises the IPC mapping on a one-GPU box).
  nccl    the fallback transport (DistributedGraph over CudaShardSession, NCCL collectives between the phases).
tests/test_multi_fabric.py covers world 1 .. 8 of the product path inside one process on any GPU box."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402
from rala_b200 import api, multi, synth  # noqa: E402

pytestmark = pytest.mark.gpu

KW = dict(genome_len=3_000_000, coverage=30, read_len=9000, len_sd=2500, seed=71, noise=50, dual=True, min_ovl=900)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _flags(ds):
    return (np.random.Generator(np.random.PCG64(1)).random(ds.n_reads) < 0.05).astype(np.uint8) * 2


def _worker(rank, world, port, out_dir, transport, same_device):
    import signal
    signal.alarm(420)    # a rank stuck waiting for a peer must not hold the GPU suite (and the box) for its whole time limit
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = 0 if same_device else rank
    torch.cuda.set_device(dev)
    if same_device:
        dist.init_process_group("gloo", rank=rank, world_size=world)      # NCCL refuses two ranks on one GPU
    else:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    try:
        ds = synth.generate(**KW)
        piles, flags = ds.flat_piles(), _flags(ds)
        lo, hi = multi.shard_bounds(ds.n_overlaps, world)[rank]
        shard = np.ascontiguousarray(ds.records[lo:hi])
        if transport == "fabric":
            fg = multi.FabricGraph(dev, rank, world)
            fg.M.set_barrier_timeout_ms(60000 if same_device else 10000)
            fg.set_inputs(shard, piles, flags, lo)
            fg.plan()
            for _ in range(2 if same_device else 4):     # eager, captured, replayed
                fg.run()
            c = fg.check()
            (first, n), edges, marked = fg.edges()
            np.savez(os.path.join(out_dir, f"r{rank}.npz"), edges=edges, marked=marked, first=first, piles=fg.M.piles(),
                     n_edges=c["n_edges"], n_pairs=c["n_transitive_pairs"], n_nodes=c["n_nodes"])
            dist.barrier()
            fg.close()
        else:
            torch.cuda.set_stream(torch.cuda.Stream(torch.device("cuda", dev)))
            sess = multi.CudaShardSession(dev)
            sess.set_inputs(shard, piles, flags, lo, rank, world)
            dg = multi.DistributedGraph(sess, rank, world)
            for _ in range(3):   # planned, then capacity-bounded passes
                dg.run()
            assert dg.check()
            c = sess.counts()
            np.savez(os.path.join(out_dir, f"r{rank}.npz"), edges=sess.edges() if rank == 0 else np.zeros((0, 3), np.uint32),
                     marked=sess.marked() if rank == 0 else np.zeros(0, np.uint8), first=0 if rank == 0 else c["n_edges"],
                     piles=sess.G.piles(), n_edges=c["n_edges"], n_pairs=c["n_transitive_pairs"] if rank == 0 else 0, n_nodes=c["n_nodes"],
                     n_candidates=c["n_candidates"], n_final_candidates=c["n_final_candidates"])
            dist.barrier()
            sess.close()
    finally:
        dist.destroy_process_group()


def _run_and_compare(world, transport, same_device, tmp_path):
    ds = synth.generate(**KW)
    want = O.Pipeline(ds.records, ds.flat_piles(), _flags(ds)).run()
    assert want.edges.shape[0] > 5000
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), transport, same_device), nprocs=world, join=True)
    parts = sorted((np.load(tmp_path / f"r{r}.npz") for r in range(world)), key=lambda z: int(z["first"]))
    assert np.array_equal(np.concatenate([z["edges"] for z in parts]), want.edges), "edge list"
    assert np.array_equal(np.concatenate([z["marked"] for z in parts]), want.marked), "removed-edge set"
    assert sum(int(z["n_pairs"]) for z in parts) == want.n_pairs
    for z in parts:
        assert np.array_equal(z["piles"], want.piles), "pile liveness"
        assert int(z["n_nodes"]) == want.n_nodes and int(z["n_edges"]) == want.edges.shape[0]
    return parts


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_fabric_one_process_per_gpu(world, tmp_path):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    _run_and_compare(world, "fabric", False, tmp_path)


def test_fabric_two_processes_on_one_device(tmp_path):
    _run_and_compare(2, "fabric", True, tmp_path)


@pytest.mark.parametrize("world", [1, 2])
def test_nccl_fallback_transport(world, tmp_path):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    parts = _run_and_compare(world, "nccl", False, tmp_path)
    # every rank imports all ranks' events: its containment-event counts are those of one GPU on the whole batch
    ds = synth.generate(**KW)
    ctx = api.Context(0)
    G = api.Graph(ctx)
    G.set_piles(ds.flat_piles(), _flags(ds)).set_hills(None).set_overlaps(ds.records)
    G.run()
    want = G.counts()
    G.close()
    ctx.close()
    assert want["n_candidates"] > 0
    for z in parts:
        assert int(z["n_candidates"]) == want["n_candidates"], "containment events of the first pass"
        assert int(z["n_final_candidates"]) == want["n_final_candidates"], "containment events of the final pass"
