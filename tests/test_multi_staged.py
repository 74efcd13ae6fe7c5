"""GPU suite: the staged construct of the multi-GPU session (rala_b200_multi_classify .. finish) with pile tables that
change between the passes (hill counters summed over the ranks, hill breaking, the pit loop and its promotions) against
the oracle, stage by stage.  Several ranks share device 0, as in tests/test_multi_fabric.py.  The host's Pile calls are
tests/test_chimeric_path.py's deterministic PileDriver."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402
from rala_b200 import api  # noqa: E402
from tests.replay import assert_same  # noqa: E402
from tests.test_chimeric_path import DATASETS, PileDriver, PileOps, constructed, dataset  # noqa: E402

pytestmark = pytest.mark.gpu


def _same_lists(M, P, what):
    ovl, inl = M.lists()
    assert_same(ovl, P.ovl, f"{what} overlaps")
    assert_same(inl, P.int, f"{what} internals")


def _multi(inp, world, bounds=None):
    M = api.Multi([0] * world)
    M.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_shards(inp.records, bounds).plan()
    return M


def _check_final(M, P, what):
    _same_lists(M, P, f"{what}: final")
    assert_same(M.piles(), P.piles, f"{what}: final piles")
    edges, marked = M.all_edges()
    assert_same(edges, P.edges, f"{what}: edges")
    assert_same(M.seq_to_node(), P.seq_to_node, f"{what}: seq_to_node")
    c = M.counts()
    assert c["n_nodes"] == P.n_nodes and c["n_edges"] == P.edges.shape[0], what
    assert c["n_transitive_pairs"] == P.n_pairs, what
    assert_same(marked, P.marked, f"{what}: marks")


def _runs(M):
    return [M.edge_runs(k) for k in range(M.n_local)]


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("name", list(DATASETS))
def test_stage_by_stage_with_changing_pile_tables(name, world):
    inp = dataset(name)
    P = O.Pipeline(inp.records, inp.piles, inp.flags, inp.hills)
    M = _multi(inp, world)
    P.classify()
    M.classify()
    _same_lists(M, P, "s1")
    cov = M.hill_coverage(0)
    assert_same(cov, P.hill_cov, "hill coverage")
    for k in range(1, world):
        assert_same(M.hill_coverage(k), cov, f"hill coverage of local rank {k}")
    assert_same(M.piles(), P.piles, "s1 piles")
    assert_same(M.connections(), P.ovl[:, :2], "s1 connections")

    drv = PileDriver(inp.hills, inp.flags, inp.seed)
    piles, flags = drv.hill_step(cov, P.piles)
    P.set_piles(piles).retrim()
    M.set_piles(piles, flags).retrim()
    _same_lists(M, P, "after the hill step")
    r = 0
    while True:
        conn = M.connections()
        assert_same(conn, P.ovl[:, :2], f"connections before pit round {r}")
        assert_same(M.piles(), P.piles, f"piles before pit round {r}")
        upd = drv.pit_round(conn, P.piles, r)
        if upd is not None:
            P.set_piles(upd[0])
            M.set_piles(*upd)
        want_changed = P.retrim_promote()
        assert M.retrim_promote() == want_changed, f"is_changed of pit round {r}"
        _same_lists(M, P, f"pit round {r}")
        r += 1
        if not want_changed:
            break
    assert r >= 2

    P.final_containment().build_edges().transitive()
    M.finish()
    _check_final(M, P, f"{name}, world {world}")
    runs = _runs(M)
    if name == "chimeras_repeats":   # the pit loop promotes repeat-induced internals that end up as edges
        assert max(len(x) for x in runs) > 1, "a rank with edges in more than one segment"
    for k, x in enumerate(runs):
        if len(x) > 1:
            with pytest.raises(api.RalaB200Error, match="edge_runs"):
                M.edge_range(k)
        else:
            assert M.edge_range(k) == ((int(x[0, 0]), int(x[0, 1])) if len(x) else (0, 0))
    M.close()


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("name", ["chimeras_repeats", "jittered"])
def test_construct_matches_the_oracle(name, world):
    """Multi.construct with the driver: every input the pile ops receive equals the oracle-driven construct's."""
    inp = dataset(name)
    P, changed, calls, _ = constructed(name)
    M = api.Multi([0] * world)
    ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), M.piles, want=calls)
    M.construct(inp.records, inp.piles, inp.flags, inp.hills, pile_ops=ops)
    assert len(ops.calls) == len(calls)
    assert M.n_nodes == P.n_nodes
    _check_final(M, P, f"{name}, world {world}")
    M.close()


def test_empty_shard():
    """Rank 1 of 3 has no records at all (no entries, no internals, no edges); rank 2 holds only the last 8 records."""
    name = "chimeras_repeats"
    inp = dataset(name)
    P, _, calls, _ = constructed(name)
    n = inp.records.shape[0]
    bounds = [(0, n - 8), (n - 8, n - 8), (n - 8, n)]
    M = api.Multi([0] * 3)
    M.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_shards(inp.records, bounds).plan()
    ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), M.piles, want=calls)
    M.classify()
    assert M.local_lists(1)[0].shape[0] == 0
    upd = ops.break_over_chimeric_hills(M.hill_coverage(1))
    M.set_piles(*upd).retrim()
    while True:
        upd = ops.break_over_chimeric_pits(M.connections())
        if upd is not None:
            M.set_piles(*upd)
        if not M.retrim_promote():
            break
        assert [x.shape[0] for x in M.local_lists(1)] == [0, 0, 0, 0]
    M.finish()
    _check_final(M, P, "empty shard")
    assert M.edge_runs(1).shape[0] == 0 and M.edges(1).shape[0] == 0
    M.close()


def test_staged_calls_out_of_order_then_a_frozen_run_on_the_same_session():
    inp = dataset("jittered")
    M = api.Multi([0] * 2)
    M.set_piles(inp.piles, inp.flags).set_hills(inp.hills).set_shards(inp.records)
    with pytest.raises(api.RalaB200Error, match="status -3"):
        M.classify()                     # nothing reserved yet
    M.plan()
    for call in (M.retrim, M.retrim_promote, M.finish):
        with pytest.raises(api.RalaB200Error, match="status -3"):
            call()
    with pytest.raises(api.RalaB200Error, match="status -3"):
        M.lists()
    M.classify()
    M.finish()
    with pytest.raises(api.RalaB200Error, match="status -3"):
        M.retrim()                       # finished: classify again first
    # the same session, a frozen table and the library's one-step chain: eager, captured, replayed
    flags = (inp.flags & 2).astype(np.uint8)
    want = O.Pipeline(inp.records, inp.piles, flags).run()
    M.set_piles(inp.piles, flags)
    for i in range(4):
        M.run()
        edges, marked = M.all_edges()
        assert_same(edges, want.edges, f"frozen run {i}: edges")
        assert_same(marked, want.marked, f"frozen run {i}: marks")
        assert_same(M.piles(), want.piles, f"frozen run {i}: piles")
        assert M.counts()["n_transitive_pairs"] == want.n_pairs
        for k in range(2):
            assert M.edge_runs(k).shape[0] <= 1
    M.close()


# ---------------------------------------------------------------------------------------------------------------------
# parallel edges across segments: the tie-break of graph.cpp:1291-1293 (the highest edge id among parallel edges is the
# candidate) decides which of two A -> B edges the triangle A -> C -> B removes
# ---------------------------------------------------------------------------------------------------------------------
_L = 10000
_INVALID = (0, 1, 0, 0, 0, 0, 2)
TIE_PILES = np.array([[0, _L]] * 3, np.uint32)                      # reads A = 0, B = 1, C = 2
TIE_RECORDS = np.array([(0, 1, 6000, 9000, 0, 3000, 0),             # rank 0: A-B internal, a dovetail once A ends at 9000
                        _INVALID, _INVALID, _INVALID,
                        (0, 1, 6000, _L, 0, 4000, 0),                # rank 1: A -> B dovetail (segment 0)
                        (0, 2, 3000, _L, 0, 7000, 0),                #         A -> C
                        (2, 1, 3000, _L, 0, 7000, 0)], np.uint32)    #         C -> B: the triangle
TIE_BOUNDS = [(0, 4), (4, 7)]
TIE_CUT = TIE_PILES.copy()
TIE_CUT[0] = (0, 9000)


def _tie_stages(G):
    """classify, retrim, a pit round that promotes rank 0's internal, a round that changes nothing; is_changed of both"""
    G.classify()
    G.retrim()
    changed = []
    for _ in range(2):
        G.set_piles(TIE_CUT)
        changed.append(G.retrim_promote())
    return changed


def test_parallel_edges_across_segments_take_the_segment_major_tie_break(ctx):
    P = O.Pipeline(TIE_RECORDS, TIE_PILES)
    want_changed = _tie_stages(P)
    assert P.ovl.shape[0] == 4 and P.int.shape[0] == 0, "the internal was promoted to the end of `overlaps`"
    P.final_containment().build_edges().transitive()
    marked_entries = P.marked[0::2].copy()
    assert marked_entries.tolist() == [0, 0, 0, 1], "the promoted A -> B (highest ids) is the one removed"

    # rank-major ids (rank 0's promoted entry first) would remove the other A -> B edge
    Q = O.Pipeline(TIE_RECORDS, TIE_CUT)
    Q.ovl, Q.int = P.ovl[[3, 0, 1, 2]].copy(), P.int.copy()
    Q.build_edges().transitive()
    assert not np.array_equal(Q.marked[0::2][[1, 2, 3, 0]], marked_entries)

    M = api.Multi([0, 0])
    M.set_piles(TIE_PILES).set_hills(None).set_shards(TIE_RECORDS, TIE_BOUNDS).plan()
    M.classify()
    M.retrim()
    M.set_piles(TIE_CUT)
    assert M.retrim_promote() == want_changed[0]
    assert M.local_lists(0)[2].shape[0] == 0, "rank 0's only internal was promoted"
    ovl_before = [M.local_lists(k) for k in range(2)]
    M.set_piles(TIE_CUT)
    assert M.retrim_promote() == want_changed[1]      # nobody promotes: no segment opens, nothing moves
    for k in range(2):
        after = M.local_lists(k)
        assert_same(after[0], ovl_before[k][0], f"rank {k}: overlaps after a round without promotions")
        assert_same(after[1], ovl_before[k][1], f"rank {k}: global positions after a round without promotions")
    M.finish()
    _check_final(M, P, "parallel edges across segments")
    assert M.edge_runs(0).tolist() == [[6, 2]] and M.edge_runs(1).tolist() == [[0, 6]]

    G = api.Graph(ctx)
    G.set_piles(TIE_PILES).set_hills(None).set_overlaps(TIE_RECORDS)
    assert _tie_stages(G) == want_changed
    G.finalize().build()
    assert G.remove_transitive_edges() == P.n_pairs
    assert_same(G.edges(), M.all_edges()[0], "single GPU vs multi-GPU: edges")
    assert_same(G.removed, M.all_edges()[1], "single GPU vs multi-GPU: marks")
    G.close()
    M.close()


# ---------------------------------------------------------------------------------------------------------------------
# one process per rank: every process reads hill totals, list counts and is_changed from its own arena
# ---------------------------------------------------------------------------------------------------------------------
def _process_worker(rank, world, port, out_dir, name):
    import signal
    import socket  # noqa: F401
    import torch
    import torch.distributed as dist
    from rala_b200 import multi
    signal.alarm(420)    # a rank stuck waiting for a peer must not hold the GPU suite for its whole time limit
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # NCCL refuses two ranks on one GPU
    try:
        inp = dataset(name)
        _, _, calls, _ = constructed(name)
        lo, hi = multi.shard_bounds(inp.records.shape[0], world)[rank]
        fg = multi.FabricGraph(0, rank, world)
        fg.M.set_barrier_timeout_ms(60000)
        fg.set_inputs(np.ascontiguousarray(inp.records[lo:hi]), inp.piles, inp.flags, lo, hills=inp.hills)
        fg.plan()
        ops = PileOps(PileDriver(inp.hills, inp.flags, inp.seed), fg.M.piles, want=calls)   # asserts every input
        fg.construct(ops)
        c = fg.check()
        ovl, opos, inl, ipos = fg.M.local_lists(0)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), ids=fg.M.edge_ids(0), edges=fg.M.edges(0), marked=fg.M.marked(0),
                 ovl=ovl, opos=opos, inl=inl, ipos=ipos, cov=fg.M.hill_coverage(0), piles=fg.M.piles(),
                 s2n=fg.M.seq_to_node(), n_calls=len(ops.calls), n_pairs=c["n_transitive_pairs"], n_nodes=c["n_nodes"],
                 n_edges=c["n_edges"])
        dist.barrier()
        fg.close()
    finally:
        dist.destroy_process_group()


def test_fabric_construct_two_processes_on_one_device(tmp_path):
    import socket
    import torch.multiprocessing as mp
    name = "chimeras_repeats"
    P, _, calls, _ = constructed(name)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_process_worker, args=(2, port, str(tmp_path), name), nprocs=2, join=True)
    parts = [np.load(tmp_path / f"r{r}.npz") for r in range(2)]
    ids = np.concatenate([z["ids"] for z in parts])
    order = np.argsort(ids, kind="stable")
    assert np.array_equal(ids[order], np.arange(P.edges.shape[0])), "every edge id exactly once"
    assert_same(np.concatenate([z["edges"] for z in parts])[order], P.edges, "edges")
    assert_same(np.concatenate([z["marked"] for z in parts])[order], P.marked, "marks")
    for which, want in (("ovl", P.ovl), ("inl", P.int)):
        pos = np.concatenate([z["opos" if which == "ovl" else "ipos"] for z in parts])
        rows = np.concatenate([z[which] for z in parts])
        assert_same(rows[np.argsort(pos, kind="stable")], want, f"final {which}")
    assert sum(int(z["n_pairs"]) for z in parts) == P.n_pairs
    for z in parts:
        assert int(z["n_calls"]) == len(calls)
        assert_same(z["cov"], calls[0][1], "hill coverage, as each process read it")
        assert_same(z["piles"], P.piles, "final piles")
        assert_same(z["s2n"], P.seq_to_node, "seq_to_node")
        assert int(z["n_nodes"]) == P.n_nodes and int(z["n_edges"]) == P.edges.shape[0]
