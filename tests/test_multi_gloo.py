"""CPU suite, world_size 2 and 3 over gloo: the multi-GPU ORCHESTRATION (rala_b200/multi.py: sharding,
padding, offsets, time bases, exchange order) driven with a stand-in session whose phases are computed
with the oracle.  The product session (CudaShardSession) has the same interface; its kernels are covered
by tests/test_gpu_parity.py and tests/test_multi_gpu.py."""
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
from rala_b200 import multi, synth  # noqa: E402

INF = 0xFFFFFFFF


class OracleShardSession:
    """ShardSession stand-in: every phase computed on the host with the oracle's trim / type."""

    def __init__(self, records, piles, flags, t0, rank, world):
        self.device = torch.device("cpu")
        self.rec = np.ascontiguousarray(records, dtype=np.uint32).reshape(-1, 7)
        self.piles0 = np.ascontiguousarray(piles, dtype=np.uint32).copy()
        self.piles = self.piles0.copy()
        self._overflow = False
        self.flags = np.zeros(len(piles), np.uint8) if flags is None else np.asarray(flags, np.uint8)
        self.t0, self.rank, self.world = t0, rank, world
        self.n_records = len(self.rec)
        self.events = np.zeros((0, 3), np.uint32)
        self.edges_all = np.zeros((0, 3), np.uint32)

    def _trim_type(self, r):
        a, b = int(r[0]), int(r[1])
        if r[6] & 2 or a >= len(self.piles) or b >= len(self.piles) or self.piles[a, 1] == 0 or self.piles[b, 1] == 0:
            return False, r, O.REJECT
        return O.trim_type(r, self.piles[a], self.piles[b])

    def phase_events(self):
        self.piles = self.piles0.copy()   # re-runnable, like the CUDA session
        self._overflow = False
        ev = []
        for i, r in enumerate(self.rec):
            ok, tr, t = self._trim_type(r)
            if not ok:
                continue
            a, b = int(r[0]), int(r[1])
            if t == O.KB and not (self.flags[b] & 2):
                ev.append((a, b, self.t0 + i))
            elif t == O.KA and not (self.flags[a] & 2):
                ev.append((b, a, self.t0 + i))
        self.events = np.asarray(ev, np.uint32).reshape(-1, 3)
        self.n_first_events = len(ev)

    def phase_resolve(self, first):
        # the reference's sequential semantics: in time order, an event fires iff both piles are still alive
        ev = self.events_all[np.argsort(self.events_all[:, 2], kind="stable")] if len(self.events_all) else self.events_all
        alive = self.piles[:, 1] != 0
        self.death = np.full(len(self.piles), INF, np.uint64)
        for v, c, t in ev.tolist():
            if alive[v] and alive[c]:
                alive[v] = False
                self.death[v] = t
        self.pre_final_alive = self.piles[:, 1] != 0
        self.piles[~alive] = 0

    def phase_survivors(self):
        ovl, inl = [], []
        for r in self.rec:
            ok, tr, t = self._trim_type(r)
            if ok:
                tr[0], tr[1] = r[0], r[1]   # O.trim_type works on a two-pile table and renumbers the ids
                (inl if t == O.KX else ovl).append(tr)
        self.ovl = np.asarray(ovl, np.uint32).reshape(-1, 7)
        self.inl = np.asarray(inl, np.uint32).reshape(-1, 7)

    def export_list_counts(self, pair):
        pair[0], pair[1] = len(self.ovl), len(self.inl)

    def phase_final_events_gathered(self, counts, world):
        c = counts.numpy().astype(np.int64)
        ovl_base, int_base = int(c[:self.rank, 0].sum()), int(c[:, 0].sum() + c[:self.rank, 1].sum())
        ev = []
        for base, lst in ((ovl_base, self.ovl), (int_base, self.inl)):
            for i, r in enumerate(lst):
                piles2 = np.ascontiguousarray(self.piles[[r[0], r[1]]])
                rr = r.copy(); rr[0], rr[1] = 0, 1
                t = O.lib().ora_type(O._p(rr), O._p(piles2))
                if t == O.KA:
                    ev.append((int(r[1]), int(r[0]), base + i))
                elif t == O.KB:
                    ev.append((int(r[0]), int(r[1]), base + i))
        self.events = np.asarray(ev, np.uint32).reshape(-1, 3)

    def phase_emit_edges(self):
        alive = self.piles[:, 1] != 0
        s2n = np.full(len(self.piles), INF, np.uint64)
        s2n[alive] = 2 * np.arange(int(alive.sum()))
        self.n_nodes = 2 * int(alive.sum())
        keep = [r for r in self.ovl if alive[r[0]] and alive[r[1]]]
        P = O.Pipeline(np.zeros((0, 7), np.uint32), self.piles)
        P.ovl = np.asarray(keep, np.uint32).reshape(-1, 7)
        P.build_edges()      # local node numbering == global: the pile table is replicated
        self.edges = P.edges

    def phase_csr(self):
        pass

    def phase_transitive(self):
        e = self.edges_all
        E = len(e)
        row_start = np.searchsorted(np.sort(e[:, 0]), np.arange(self.n_nodes + 1)) if E else np.zeros(self.n_nodes + 1, int)

        def begin(r):
            if r == 0:
                return 0
            if r >= self.world:
                return self.n_nodes
            return int(np.searchsorted(row_start[:self.n_nodes], E * r // self.world, side="left"))

        lo, hi = begin(self.rank), begin(self.rank + 1)
        out = {}
        for i, (s, d, l) in enumerate(e.tolist()):
            out.setdefault(s, []).append((d, l, i))
        T = np.zeros(E, np.uint8)
        for a in range(lo, hi):
            cand = {}
            for d, l, i in out.get(a, []):
                if d not in cand or cand[d][1] < i:
                    cand[d] = (l, i)
            for b, lab, _ in out.get(a, []):
                for c, lbc, _ in out.get(b, []):
                    if c in cand and O.comparable((lab + lbc) & 0xFFFFFFFF, cand[c][0]):
                        T[cand[c][1]] = 1
        self.T = T

    def export_marks(self, t):
        t.zero_()
        t[:len(self.T)] = torch.from_numpy(self.T)

    def phase_marks(self, t):
        T = t.numpy()[:len(self.edges_all)]
        m = (T[0::2] | T[1::2])
        self.marked = np.repeat(m, 2).astype(np.uint8)

    # ---- exchange blocks: [n clamped to cap | overflow flag | n | 0 | three columns of cap] ----------------------
    def export_padded(self, kind, block, cap):
        arr = self.events if kind == 0 else self.edges
        n = len(arr)
        m = min(n, cap)
        b = block.numpy().view(np.uint32)
        b[:4] = (m, int(n > cap), n, 0)
        for k in range(3):
            b[4 + k * cap: 4 + k * cap + m] = arr[:m, k]

    def import_gathered(self, kind, gathered, cap, world):
        g = gathered.numpy().view(np.uint32)
        parts = []
        for r in range(world):
            n = int(g[r, 0])
            self._overflow |= bool(g[r, 1])
            parts.append(np.stack([g[r, 4 + k * cap: 4 + k * cap + n] for k in range(3)], 1))
        merged = np.concatenate(parts).astype(np.uint32)
        if kind == 0:
            self.events_all = merged
        else:
            self.edges_all = merged

    def overflowed(self):
        return self._overflow


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, kw, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ds = synth.generate(**kw)
        piles = ds.flat_piles()
        flags = (np.random.Generator(np.random.PCG64(1)).random(ds.n_reads) < 0.05).astype(np.uint8) * 2
        lo, hi = multi.shard_bounds(ds.n_overlaps, world)[rank]
        sess = OracleShardSession(ds.records[lo:hi], piles, flags, lo, rank, world)
        dg = multi.DistributedGraph(sess, rank, world)
        passes = []
        bounded = dg.run_bounded
        dg.run_bounded = lambda: (passes.append(dict(dg.caps)), bounded())[1]

        dg.run()                                          # plans: the default capacities fit this data
        assert dg.check() and len(passes) == 1
        # this rank's element count of every exchange, from the pass that fitted
        counts = [sess.n_first_events, len(sess.events), len(sess.edges)]
        caps = dict(dg.caps)
        first = (sess.edges_all.copy(), sess.marked.copy(), sess.piles.copy())

        def same_results():
            return all(np.array_equal(x, y) for x, y in zip(first, (sess.edges_all, sess.marked, sess.piles)))

        dg.run()                                          # one pass with the planned capacities
        assert len(passes) == 2 and passes[-1] == caps and dg.check() and same_results()

        dg.caps = {k: 8 for k in dg.caps}                 # far too small: must be detected, and the next run plans again
        dg._bufs = {}
        dg.run()
        assert not dg.check() and dg.caps is None
        dg.run()
        assert dg.check() and dg.caps == caps and same_results()

        # defaults too small for the data: plan() grows until a pass fits and ends where it would have started
        multi.default_caps = lambda n_records, world: {"events": 8, "final_events": 8, "edges": 8}
        del passes[:]
        dg.caps = None
        dg.run()
        grown = len(passes)
        assert dg.check() and dg.caps == caps and same_results()
        # buffers of the sizes it grew through are dropped
        assert set(k for k in dg._bufs if k != "pair") <= set(caps.items()) | {("marks", caps["edges"] * world)}

        np.savez(os.path.join(out_dir, f"r{rank}.npz"), edges=sess.edges_all, marked=sess.marked, piles=sess.piles,
                 counts=counts, caps=[caps["events"], caps["final_events"], caps["edges"]], grown=grown)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_orchestration_plans_capacities_and_matches_single_process_oracle(world, tmp_path):
    kw = dict(genome_len=150_000, coverage=30, read_len=6000, len_sd=1500, seed=61, noise=60, dual=True, min_ovl=800)
    ds = synth.generate(**kw)
    flags = (np.random.Generator(np.random.PCG64(1)).random(ds.n_reads) < 0.05).astype(np.uint8) * 2
    want = O.Pipeline(ds.records, ds.flat_piles(), flags).run()
    assert want.edges.shape[0] > 200 and want.n_pairs > 20
    mp.spawn(_worker, args=(world, _free_port(), kw, str(tmp_path)), nprocs=world, join=True)
    got = [np.load(tmp_path / f"r{r}.npz") for r in range(world)]
    # the capacities a pass sized on the host would choose: slack(largest per-rank count), edges rounded to even
    most = np.max([z["counts"] for z in got], axis=0)
    assert (most > 0).all()
    slack = [int(n * 1.25) + 4096 for n in most.tolist()]
    slack[2] = (slack[2] + 1) // 2 * 2
    for r, z in enumerate(got):
        assert np.array_equal(z["edges"], want.edges), f"rank {r}: edge list"
        assert np.array_equal(z["marked"], want.marked), f"rank {r}: removed-edge set"
        assert np.array_equal(z["piles"], want.piles), f"rank {r}: pile liveness"
        assert z["caps"].tolist() == slack, f"rank {r}: planned capacities"
        assert 2 <= int(z["grown"]) <= 4, f"rank {r}: passes of the growing plan"


def test_shard_bounds():
    for n, w in ((0, 2), (5, 2), (1000, 3), (1001, 8), (14403721, 8)):
        b = multi.shard_bounds(n, w)
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
        assert all(lo % 4 == 0 for lo, hi in b if lo < n)


# ---------------------------------------------------------------------------------------------------------------
# The product path's host side (multi.FabricGraph): capacity agreement, handle exchange in rank order, the
# grow-until-it-fits loop.  The session is a stand-in with the interface of api.Multi; the kernels behind the real one
# are covered on the GPU (tests/test_multi_fabric.py, tests/test_multi_gpu.py).
# ---------------------------------------------------------------------------------------------------------------
class StubMulti:
    """Needs `need` per capacity (different on every rank); a step fits when every capacity is at least the GLOBAL need."""

    def __init__(self, rank, world, need, default):
        self.rank, self.world, self.need, self.default = rank, world, np.array(need, np.uint64), np.array(default, np.uint64)
        self.caps = None
        self.handles = None
        self.log = []

    def default_caps(self):
        return self.default.copy()

    def reserve(self, caps):
        self.caps = np.array(caps, np.uint64)
        self.handles = None
        self.log.append(("reserve", self.caps.tolist()))
        return self

    def export_handle(self, k):
        assert self.caps is not None
        return bytes([self.rank]) * 32 + int(self.caps[0]).to_bytes(32, "little")

    def import_handles(self, blob):
        assert len(blob) == 64 * self.world
        self.handles = [blob[64 * q:64 * q + 64] for q in range(self.world)]
        return self

    def use_cuda_graph(self, on):
        self.log.append(("graph", bool(on)))
        return self

    def run(self):
        assert self.handles is not None, "a step before the arenas were connected"
        self.log.append(("run",))
        return self

    def synchronize(self):
        return self

    def demand(self):
        fits = bool((self.need[:3] <= self.caps[:3]).all())
        return self.need.copy(), fits


def _fabric_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        # rank r needs more events the higher r is; rank 0 alone needs a large slice; defaults differ per rank
        need = [1000 * (rank + 1), 500, 9000 if rank == 0 else 100, 3 + rank, 1, 4000 + rank]
        default = [1500, 600 + rank, 800, 4096, 4096, 4000 + rank]
        stub = StubMulti(rank, world, need, default)
        fg = multi.FabricGraph(0, rank, world, session=stub)
        fg.plan()
        np.savez(os.path.join(out_dir, f"f{rank}.npz"), caps=fg.caps, handles=np.frombuffer(b"".join(stub.handles), np.uint8),
                 reserves=np.array([e[1] for e in stub.log if e[0] == "reserve"], np.uint64),
                 runs=sum(1 for e in stub.log if e[0] == "run"), graph=[e[1] for e in stub.log if e[0] == "graph"][-1])
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_fabric_graph_agrees_on_capacities_and_regrows(world, tmp_path):
    mp.spawn(_fabric_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    got = [np.load(tmp_path / f"f{r}.npz") for r in range(world)]
    for r, z in enumerate(got):
        # every rank ends with the SAME capacities, large enough for the neediest rank
        assert np.array_equal(z["caps"], got[0]["caps"])
        assert z["caps"][0] >= 1000 * world and z["caps"][2] >= 9000 and z["caps"][1] >= 600 + world - 1
        # first reservation = element-wise maximum of the ranks' defaults; then it grew (events at world 3, the slice always)
        assert z["reserves"][0].tolist() == [1500, 600 + world - 1, 800, 4096, 4096, 4000 + world - 1]
        assert len(z["reserves"]) == 2 and int(z["runs"]) == 2 and bool(z["graph"]) is True
        # handles arrive in rank order and were exchanged AFTER the last reservation (they carry the capacity)
        h = z["handles"].reshape(world, 64)
        assert [int(h[q, 0]) for q in range(world)] == list(range(world))
        assert all(int.from_bytes(bytes(h[q, 32:64]), "little") == int(z["caps"][0]) for q in range(world))


def _share_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import bench_multi
        got = bench_multi._share_through_files(rank, world, {"edges": np.full((rank + 1, 3), rank, np.uint32),
                                                             "first": np.array([10 * rank], np.int64)})
        if rank == 0:
            assert [g.shape[0] for g in got["edges"]] == list(range(1, world + 1))
            assert all(int(got["edges"][r][0, 0]) == r and int(got["first"][r][0]) == 10 * r for r in range(world))
            open(os.path.join(out_dir, "ok"), "w").write("1")
        else:
            assert got is None
    finally:
        dist.destroy_process_group()


def test_bench_parity_gate_collects_every_ranks_arrays_in_rank_order(tmp_path):
    """bench_multi._share_through_files: how rank 0 gets the other ranks' edge rows and marks for the parity gate."""
    mp.spawn(_share_worker, args=(3, _free_port(), str(tmp_path)), nprocs=3, join=True)
    assert (tmp_path / "ok").exists()


def test_shard_bounds_are_contiguous_aligned_and_cover_everything():
    for n in (0, 1, 5, 1023, 1024, 100_003):
        for world in (1, 2, 3, 8):
            b = multi.shard_bounds(n, world)
            assert len(b) == world and b[0][0] == 0 and b[-1][1] == n
            assert all(lo <= hi and (lo % 4 == 0 or lo == hi) for lo, hi in b) and all(b[i][1] == b[i + 1][0] for i in range(world - 1))
