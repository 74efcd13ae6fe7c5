"""Multi-GPU hot path, one process per GPU.

PRODUCT PATH — `FabricGraph`: the multi-GPU session of the C ABI (rala_b200_multi_*, include/rala_b200.h).  The
whole orchestration and every exchange live inside the library as CUDA kernels that write straight into the peer
GPUs' memory over NVLink (CUDA IPC between the processes) with device-side barriers in between; torch.distributed is
only the plumbing around it: it carries the 64-byte IPC handles and the capacity agreement at set-up time, and the
timing reductions of the bench.  A step enqueues kernels only and is replayed as one CUDA graph per rank.

FALLBACK TRANSPORT — `DistributedGraph` over `CudaShardSession`: the round-1 path, NCCL collectives issued through
torch.distributed between the library's phases, with the CSR built on every rank.  Used only when the GPUs cannot map
each other's memory (no peer access / no CUDA IPC); both are checked against the oracle by the same tests.  Every
exchange all-gathers fixed-capacity blocks that carry their own element counts, so a pass never waits for the host;
like the product path, `DistributedGraph.plan` sizes the capacities from real passes.

Partition of the fallback transport (BASELINE.json north_star; SURVEY.md 8e):
  * overlap records are sharded by contiguous FILE RANGE (rank r holds records [t0_r, t0_r + n_r)); the
    pile table is replicated;
  * the containment events of all shards are all-gathered and the ordered-containment resolution runs
    replicated (its result, the set of dead piles, is needed by every rank);
  * every rank emits the edges of its own surviving overlaps; the edge lists are all-gathered in rank
    order (= global edge-id order) and the CSR of the whole graph is built on every rank, because the
    two-hop lookups of the transitive pass cross shards;
  * the transitive pass is split by source-node range (equal edge share per rank); the per-edge marks are
    merged with an all-reduce(max), which is OR on 0/1 bytes.

`DistributedGraph` is written against the small `ShardSession` interface so that the orchestration
(sharding arithmetic, padding, offsets, collectives) is testable on CPU with the gloo backend and a
stand-in session (tests/test_multi_gloo.py); the product session is `CudaShardSession`.
"""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from . import api


class CudaShardSession:
    """The CUDA phases of one rank (include/rala_b200.h, "Multi-GPU phases").  Enqueues on torch's current
    stream, so NCCL collectives issued through torch.distributed are ordered with the kernels."""

    def __init__(self, device_index: int):
        self.device = torch.device("cuda", device_index)
        torch.cuda.set_device(self.device)
        lib = api.load()
        self.ctx = api.Context.__new__(api.Context)
        self.ctx.lib = lib
        self.ctx.handle = C.c_void_p()
        self.ctx.device = device_index
        self.ctx._graphs = []
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = lib.rala_b200_create_on_stream(C.byref(self.ctx.handle), C.c_int(device_index), C.c_void_p(stream))
        if rc != 0:
            raise api.RalaB200Error(f"rala_b200_create_on_stream failed with status {rc} (no CPU fallback)")
        self.G = api.Graph(self.ctx)

    # ---- inputs -------------------------------------------------------------------------------------------
    def set_inputs(self, records, piles, flags, t0: int, rank: int, world: int):
        self.n_records = len(records)
        self.G.set_piles(piles, flags).set_hills(None).set_overlaps(records)
        self.G._call("rala_b200_graph_set_shard", C.c_uint32(t0), C.c_int(rank), C.c_int(world))

    @staticmethod
    def _dp(t: torch.Tensor):
        return C.c_void_p(t.data_ptr())

    # ---- phases: none reads a count back to the host (counts travel inside the exchange blocks) -------------------
    def phase_events(self):
        self.G._call("rala_b200_graph_phase_events")

    def phase_resolve(self, first: bool):
        self.G._call("rala_b200_graph_phase_resolve", C.c_int(1 if first else 0))

    def phase_survivors(self):
        self.G._call("rala_b200_graph_phase_survivors")

    def phase_emit_edges(self):
        self.G._call("rala_b200_graph_phase_emit_edges")

    def phase_csr(self):
        self.G._call("rala_b200_graph_phase_csr")

    def phase_transitive(self):
        self.G._call("rala_b200_graph_phase_transitive")

    def export_marks(self, t: torch.Tensor):
        self.G._call("rala_b200_graph_export_marks", self._dp(t), C.c_uint32(t.shape[0]))

    def phase_marks(self, t: torch.Tensor):
        self.G._call("rala_b200_graph_phase_marks", self._dp(t), C.c_uint32(t.shape[0]))

    def block_words(self, kind: int, cap: int) -> int:
        """32-bit words of one exchange block: a 4-word header and three columns of `cap` words."""
        return int(self.ctx.lib.rala_b200_exchange_block_words(C.c_int(kind), C.c_uint32(cap)))

    def export_padded(self, kind: int, block: torch.Tensor, cap: int):
        self.G._call("rala_b200_graph_export_padded", C.c_int(kind), self._dp(block), C.c_uint32(cap))

    def import_gathered(self, kind: int, gathered: torch.Tensor, cap: int, world: int):
        self.G._call("rala_b200_graph_import_gathered", C.c_int(kind), self._dp(gathered), C.c_uint32(cap), C.c_int(world))

    def export_list_counts(self, pair: torch.Tensor):
        self.G._call("rala_b200_graph_export_list_counts", self._dp(pair))

    def phase_final_events_gathered(self, counts: torch.Tensor, world: int):
        self.G._call("rala_b200_graph_phase_final_events_gathered", self._dp(counts), C.c_int(world))

    def overflowed(self) -> bool:
        """Synchronises; True when an exchange block (or any device list) was too small in the last run."""
        try:
            self.G.counts()
            return False
        except api.RalaB200Error:
            return True

    # ---- results (replicated on every rank) ------------------------------------------------------------------
    def counts(self):
        return self.G.counts()

    def edges(self):
        return self.G.edges()

    def marked(self):
        return self.G.marked()

    def close(self):
        self.G.close()
        self.ctx.close()


def default_caps(n_records: int, world: int) -> dict:
    """Exchange capacities of a first planning pass over a shard of n_records, in the proportions of
    rala_b200_multi_default_caps (the events of both containment passes share its event capacity)."""
    align = lambda n: (n + 255) // 256 * 256   # noqa: E731
    events = align(n_records // (4 if world > 1 else 1) + 4096)
    edges = align(n_records // (2 if world > 1 else 1) * (1 if world > 1 else 2) + 4096)
    return {"events": events, "final_events": events, "edges": edges}


def _slack(n: int) -> int:
    return int(n * 1.25) + 4096


class DistributedGraph:
    """Drives one ShardSession per rank through the phases, with the collectives in between.
    It runs the frozen-pile chain only (no hills, no host pile breaking between the passes): the staged construct for
    pile tables that change between the passes needs the peer-memory fabric (rala_b200_multi_classify .. finish).
    A pass never reads a count back to the host, so its results are valid only if check() says so."""

    def __init__(self, session, rank: int, world: int, group=None):
        self.s, self.rank, self.world, self.group = session, rank, world, group
        self.device = session.device
        self.comm_bytes = 0   # bytes this rank received through collectives in the last run
        self.caps = None      # per-rank exchange capacities, set by plan()
        self._bufs = {}
        self._graph = None    # one bounded pass (kernels + NCCL collectives) captured in a CUDA graph
        self.graph_launches = 0
        self.graph_error = None

    def run(self):
        """One pass of the hot path.  Without capacities (the first pass, and the first after check() found an
        overflow) it plans them, which leaves the results of the pass that fitted."""
        if self.caps is None:
            self.plan()
        else:
            self.run_bounded()

    def plan(self, max_attempts: int = 4):
        """Size the exchange blocks from real passes (collective): run, read from the gathered blocks what every rank
        needed, set each capacity to slack(need), until a pass fits.  The first events exchange depends on no capacity,
        the final events only on it and the edges on both, so the fourth pass fits at the latest.  The capacities
        that stay are slack(largest per-rank count) of the pass that fitted, whatever the capacities it ran with."""
        caps = default_caps(self.s.n_records, self.world)
        t = torch.tensor(list(caps.values()), dtype=torch.int64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        caps = dict(zip(caps, (int(v) for v in t.tolist())))
        for _ in range(max_attempts):
            self.caps = caps
            self.run_bounded()
            # word 2 of a block = its rank's count; the gathered blocks are the same on every rank, so all ranks read
            # the same needs without another collective (the read-back synchronises)
            need = dict(zip(caps, torch.stack([self._bufs[(name, cap)][1][:, 2].max() for name, cap in caps.items()]).tolist()))
            fits = all(need[name] <= cap for name, cap in caps.items())
            caps = {"events": _slack(need["events"]), "final_events": _slack(need["final_events"]),
                    "edges": (_slack(need["edges"]) + 1) // 2 * 2}
            if fits:
                self.caps = caps
                keep = set(caps.items()) | {("marks", caps["edges"] * self.world), "pair"}
                self._bufs = {k: v for k, v in self._bufs.items() if k in keep}
                return self
        self.caps = None
        raise api.RalaB200Error("plan: the exchange blocks still did not fit")

    def check(self) -> bool:
        """After bounded passes: did every block fit?  (synchronises)  On overflow the next run() plans again."""
        if self.caps is not None and self.s.overflowed():
            self.caps = None
            self._bufs = {}
            self._graph = None
            return False
        return True

    def capture(self) -> bool:
        """Capture one capacity-bounded pass, NCCL collectives included, in a CUDA graph: `replay()` then costs one
        launch per step instead of ~50 kernel launches, ~20 library calls and 5 collectives issued from Python.
        Requires planned capacities (it plans when there are none) and a session created on a non-default stream that
        is torch's current stream.  Returns False (and keeps the eager path) when the capture fails."""
        if self.caps is None:
            self.plan()
        self.run_bounded()          # every exchange buffer exists before the capture starts
        torch.cuda.synchronize(self.device)
        stream = torch.cuda.current_stream(self.device)
        launches0 = self.s.ctx.launch_count
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream, capture_error_mode="thread_local"):
                self.run_bounded()
            self._graph = graph
            self.graph_launches = self.s.ctx.launch_count - launches0
            self.graph_error = None
        except Exception as exc:   # noqa: BLE001 — the eager bounded path stays available
            self._graph = None
            self.graph_error = f"{type(exc).__name__}: {exc}"
        return self._graph is not None

    def replay(self):
        """One pass: the captured graph when there is one, else run().  The counts of the pass stay on the device:
        session.counts() after check() reads them."""
        if self._graph is not None:
            self._graph.replay()
        else:
            self.run()

    def _buffers(self, name: str, cap: int, kind: int = 0):
        key = (name, cap)
        if key not in self._bufs:
            words = self.s.block_words(kind, cap) if hasattr(self.s, "block_words") else 3 * cap + 4
            self._bufs[key] = (torch.zeros(words, dtype=torch.int32, device=self.device),
                               torch.zeros((self.world, words), dtype=torch.int32, device=self.device))
        return self._bufs[key]

    def _exchange(self, name: str, kind: int, cap: int):
        block, gathered = self._buffers(name, cap, kind)
        self.s.export_padded(kind, block, cap)
        dist.all_gather_into_tensor(gathered.view(-1), block, group=self.group)
        self.comm_bytes += block.numel() * 4 * (self.world - 1)
        self.s.import_gathered(kind, gathered, cap, self.world)

    def run_bounded(self):
        """One pass with the current capacities; enqueues only (no count is read back)."""
        s, caps = self.s, self.caps
        self.comm_bytes = 0
        # graph.cpp:443-518
        s.phase_events()
        self._exchange("events", 0, caps["events"])
        s.phase_resolve(True)
        s.phase_survivors()
        # graph.cpp:831-877 — time of a list entry = its position in the GLOBAL overlaps ++ internals order
        if "pair" not in self._bufs:
            self._bufs["pair"] = (torch.zeros(2, dtype=torch.int32, device=self.device),
                                  torch.zeros((self.world, 2), dtype=torch.int32, device=self.device))
        pair, pairs = self._bufs["pair"]
        s.export_list_counts(pair)
        dist.all_gather_into_tensor(pairs.view(-1), pair, group=self.group)
        s.phase_final_events_gathered(pairs, self.world)
        self._exchange("final_events", 0, caps["final_events"])
        s.phase_resolve(False)
        # graph.cpp:552-632 — edge ids follow the global list order = rank order of the shards
        s.phase_emit_edges()
        self._exchange("edges", 1, caps["edges"])
        s.phase_csr()
        # graph.cpp:1281-1318 — split by source node; marks merged with all-reduce(max)
        s.phase_transitive()
        n_marks = caps["edges"] * self.world
        if ("marks", n_marks) not in self._bufs:
            self._bufs[("marks", n_marks)] = torch.zeros(n_marks, dtype=torch.uint8, device=self.device)
        marks = self._bufs[("marks", n_marks)]
        s.export_marks(marks)
        dist.all_reduce(marks, op=dist.ReduceOp.MAX, group=self.group)
        self.comm_bytes += marks.numel() * 2 * (self.world - 1) // self.world
        s.phase_marks(marks)


def shard_bounds(n_records: int, world: int):
    """Contiguous, 4-record aligned shards of a file of n_records (the reference's own chunking is by
    bytes, graph.cpp:24; alignment keeps every shard start 16-byte aligned for the TMA tile loads)."""
    per = (n_records + world - 1) // world
    per = (per + 3) // 4 * 4
    return [(min(n_records, r * per), min(n_records, (r + 1) * per)) for r in range(world)]


# -------------------------------------------------------------------------------------------------------------
# product path: the library's own multi-GPU session, one rank per process
# -------------------------------------------------------------------------------------------------------------
class FabricGraph:
    """One rank of rala_b200_multi.  Collective calls (every rank must make them): connect(), plan()."""

    def __init__(self, local_rank: int, rank: int, world: int, group=None, session=None):
        self.rank, self.world, self.group = rank, world, group
        self.device = torch.device("cuda", local_rank) if session is None else torch.device("cpu")
        # session: anything with the interface of api.Multi (tests/test_multi_gloo.py drives the set-up logic on CPU with a stand-in)
        self.M = api.Multi([local_rank], first_rank=rank, world=world) if session is None else session
        self.caps = None

    # ---- inputs (local) ---------------------------------------------------------------------------------------
    def set_inputs(self, records, piles, flags, t0: int, hills=None):
        self.M.set_piles(piles, flags)
        if hills is not None:   # only the staged construct counts them
            self.M.set_hills(hills)
        self.M.set_overlaps(0, records, t0)
        return self

    # ---- set-up (collective) ----------------------------------------------------------------------------------
    def _plumbing_device(self):
        """NCCL moves CUDA tensors, gloo (tests with several ranks on one GPU: NCCL refuses those) CPU tensors."""
        return self.device if dist.get_backend(self.group) == "nccl" else torch.device("cpu")

    def _max_over_ranks(self, values):
        t = torch.tensor([int(v) for v in values], dtype=torch.int64, device=self._plumbing_device())
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return [int(v) for v in t.cpu().tolist()]

    def connect(self, caps=None):
        """Agree on the exchange capacities, allocate the arenas and map every peer's arena (CUDA IPC)."""
        if caps is None:
            caps = self.M.default_caps()
        self.caps = np.array(self._max_over_ranks(caps), dtype=np.uint64)
        self.M.reserve(self.caps)
        mine = torch.frombuffer(bytearray(self.M.export_handle(0)), dtype=torch.uint8).to(self._plumbing_device())
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(parts, mine, group=self.group)
        self.M.import_handles(b"".join(bytes(p.cpu().numpy().tobytes()) for p in parts))
        dist.barrier(group=self.group)   # nobody starts a step before every rank has mapped every arena
        return self

    def plan(self, max_attempts: int = 6):
        """Size the exchange buffers from real steps: run, read what the step needed, grow what did not fit (all ranks
        together), until a step fits."""
        if self.caps is None:
            self.connect()
        for _ in range(max_attempts):
            self.M.use_cuda_graph(False)
            self.M.run().synchronize()
            need, fits = self.M.demand()
            agreed = self._max_over_ranks(list(need) + [0 if fits else 1])
            need, misfit = np.array(agreed[:-1], dtype=np.uint64), agreed[-1]
            if not misfit:
                self.M.use_cuda_graph(True)
                return self
            caps = self.caps.copy()
            for i in range(3):
                if need[i] > caps[i]:
                    caps[i] = (int(need[i]) * 5 // 4 + 1024 + 255) // 256 * 256
            caps[3], caps[4], caps[5] = max(int(caps[3]), int(need[3])), max(int(caps[4]), int(need[4])), max(int(caps[5]), int(need[5]))
            self.connect(caps)
        raise api.RalaB200Error("plan: the exchange buffers still did not fit")

    # ---- step / results ----------------------------------------------------------------------------------------
    def run(self):
        self.M.run()
        return self

    def check(self) -> dict:
        """Synchronises; raises when the last step did not fit its buffers or rounds, or a peer went missing."""
        return self.M.counts()

    # ---- staged construct (collective: every rank makes the same calls) ----------------------------------------
    def connections(self):
        """(a_id, b_id) of the whole `overlaps` list in the reference's order: every rank's entries with their global
        positions, all-gathered (the host's pit loop needs the whole list, graph.cpp:740-744)."""
        ovl, pos, _, _ = self.M.local_lists(0)
        mine = np.concatenate([pos.astype(np.int64)[:, None], ovl[:, :2].astype(np.int64)], 1)
        parts = [None] * self.world
        dist.all_gather_object(parts, mine, group=self.group)
        rows = np.concatenate(parts)
        return np.ascontiguousarray(rows[np.argsort(rows[:, 0], kind="stable"), 1:].astype(np.uint32))

    def construct(self, pile_ops=None):
        """Graph::construct's hot half and remove_transitive_edges with the same `pile_ops` contract as
        api.Graph.construct; every rank passes pile ops that compute the same answers from the same inputs.  Hill
        counters and is_changed come replicated from the library; the only host exchange added is the all-gather of
        the connection list.  Raises when the staged passes outgrew the exchange buffers plan() sized from a frozen step
        (the results are then incomplete): connect() again with the capacities demand() reports."""
        if self.caps is None:
            self.plan()
        M = self.M
        M.classify()
        if pile_ops is not None:
            upd = pile_ops.break_over_chimeric_hills(M.hill_coverage(0))
            if upd is not None:
                M.set_piles(*upd)
        M.retrim()
        while True:
            if pile_ops is not None:
                upd = pile_ops.break_over_chimeric_pits(self.connections())
                if upd is not None:
                    M.set_piles(*upd)
            if not M.retrim_promote():
                break
        M.finish().synchronize()
        need, fits = M.demand()
        if self._max_over_ranks([0 if fits else 1])[0]:
            raise api.RalaB200Error(f"construct: the staged passes did not fit the exchange buffers (rank {self.rank} needs "
                                    f"{need.tolist()}, has {self.caps.tolist()}): connect() with larger capacities")
        return self

    def edges(self):
        return self.M.edge_range(0), self.M.edges(0), self.M.marked(0)

    def close(self):
        self.M.close()


def make_graph(local_rank: int, rank: int, world: int, records, piles, flags, t0: int):
    """The product path when the GPUs can map each other's memory, else the NCCL fallback transport.
    Returns (kind, object); collective."""
    ok, fg, err = 1, None, ""
    try:
        fg = FabricGraph(local_rank, rank, world)
        fg.set_inputs(records, piles, flags, t0)
        fg.connect()
    except api.RalaB200Error as exc:   # e.g. cudaIpcOpenMemHandle refused: the other ranks must take the same branch
        ok, err = 0, str(exc)
    t = torch.tensor([ok], dtype=torch.int32, device=torch.device("cuda", local_rank))
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if int(t.item()):
        return "fabric", fg
    if fg is not None:
        fg.close()
    if rank == 0:
        print(f"[rala_b200.multi] peer memory unavailable ({err or 'on another rank'}): falling back to NCCL collectives",
              file=__import__("sys").stderr)
    torch.cuda.set_stream(torch.cuda.Stream(torch.device("cuda", local_rank)))
    sess = CudaShardSession(local_rank)
    sess.set_inputs(records, piles, flags, t0, rank, world)
    return "nccl", DistributedGraph(sess, rank, world)
