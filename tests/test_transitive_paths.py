"""K3, the transitive-edge reduction (rala_b200/csrc/transitive.cu), at every hand-off between its three kernels, against
the oracle's literal restatement of graph.cpp:1281-1318 (O.transitive).

The kernel picks a path per node from its out-degree d and its two-hop visits W(a) = sum of deg(b) over the edges a -> b:
  k_transitive_group   2 <= d <= 16,  W <= 4096           (W > 4096: handed to the heavy kernel as one item)
  k_transitive_light   17 <= d <= 64, W <= 32768          (W > 32768: one heavy item)
  k_transitive_heavy   d > 64: num_hash_chunks(d) x ceil(d / 256) items (hash chunk of the destinations x stream chunk)
Every graph here is built so that it sits on one of these boundaries, and an unmarked test asserts that it does, with
the selection restated below in numpy: a graph that drifts off its boundary fails without a GPU.

Graphs follow the pair(e) = e ^ 1 convention of synth.hub_graph.  Forward edges join even nodes; every twin edge
b^1 -> a^1 has the length TWIN, so a triangle among twins compares 2 TWIN with TWIN and never passes: the marks come
from the forward triangles, whose lengths the tests choose (the twins still run through the kernels, as negatives)."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api, synth
from tests.replay import assert_same

# ---- the kernel's selection, restated (transitive.cu) ------------------------------------------------------------------
GROUP_MAX_DEG, GROUP_MAX_VISITS = 16, 4096
LIGHT_MAX_DEG, LIGHT_MAX_VISITS = 64, 32768
HEAVY_HASH_CHUNK, HEAVY_CHUNK_FILL, HEAVY_CAP, HEAVY_NBR_CHUNK = 1024, 768, 2048, 256
TWIN = 10**6
# comparable(l_ab + l_bc = 200, l_ac, 0.12) holds for l_ac in [176, 227] (test_gpu_parity.test_transitive_edge_cases)
BOUNDS = ((176, 1), (175, 0), (227, 1), (228, 0))


def num_hash_chunks(d):
    d = np.asarray(d, np.int64)
    return np.where(d <= HEAVY_HASH_CHUNK, 1, (d + HEAVY_CHUNK_FILL - 1) // HEAVY_CHUNK_FILL)


def hash_chunk_of(key, n):
    key = np.asarray(key, np.uint64)
    return np.where(n == 1, 0, (((key * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)) >> np.uint64(12)) % np.uint64(n))


class Model:
    """Which kernel takes each node, and the counters the pass reports."""

    def __init__(self, n_nodes, edges):
        e = np.asarray(edges, np.int64).reshape(-1, 3)
        self.src, self.dst = e[:, 0], e[:, 1]
        self.deg = np.bincount(self.src, minlength=n_nodes)
        self.W = np.bincount(self.src, weights=self.deg[self.dst], minlength=n_nodes).astype(np.int64)
        d, W = self.deg, self.W
        small, mid = (d >= 2) & (d <= GROUP_MAX_DEG), (d > GROUP_MAX_DEG) & (d <= LIGHT_MAX_DEG)
        self.group, self.group_to_heavy = small & (W <= GROUP_MAX_VISITS), small & (W > GROUP_MAX_VISITS)
        self.light, self.light_to_heavy = mid & (W <= LIGHT_MAX_VISITS), mid & (W > LIGHT_MAX_VISITS)
        self.heavy = d > LIGHT_MAX_DEG
        self.chunked = d > HEAVY_HASH_CHUNK

    def items_of(self, a):
        d = int(self.deg[a])
        if d > LIGHT_MAX_DEG:
            return int(num_hash_chunks(d)) * ((d + HEAVY_NBR_CHUNK - 1) // HEAVY_NBR_CHUNK)
        return int(self.group_to_heavy[a] or self.light_to_heavy[a])

    def heavy_items(self):
        d = self.deg[self.heavy]
        return int((num_hash_chunks(d) * ((d + HEAVY_NBR_CHUNK - 1) // HEAVY_NBR_CHUNK)).sum()
                   + self.group_to_heavy.sum() + self.light_to_heavy.sum())

    def two_hop(self):
        return int(self.W[self.deg >= 2].sum())

    def chunk_load(self, a):
        """distinct destinations of node a per hash chunk"""
        keys = np.unique(self.dst[self.src == a])
        n = int(num_hash_chunks(self.deg[a]))
        return np.bincount(hash_chunk_of(keys, n).astype(np.int64), minlength=n)


class Builder:
    """Forward edges a -> b (even nodes) with their twins b^1 -> a^1 of length TWIN; pairs sorted by a key, so that
    edge ids can be placed (random by default)."""

    def __init__(self, seed, base=0):
        self.rng = np.random.Generator(np.random.PCG64(seed))
        self.base = base
        self.n_fresh = 0
        self.rows = []   # (a, b, len, key)
        self.expect = []   # (row, marked)

    def fresh(self, n):
        ids = self.base + 2 * (self.n_fresh + np.arange(n))
        self.n_fresh += n
        return [int(x) for x in ids]

    def add(self, a, b, ln, key=None):
        self.rows.append((a, b, ln, self.rng.random() if key is None else key))
        return len(self.rows) - 1

    def test(self, a, b, ln, want, key=None):
        self.expect.append((self.add(a, b, ln, key), want))

    def graph(self, n_nodes=None):
        r = np.asarray(self.rows, np.float64)
        order = np.argsort(r[:, 3], kind="stable")
        self.pos = np.empty(len(order), np.int64)
        self.pos[order] = np.arange(len(order))
        f = r[order, :3].astype(np.int64)
        e = np.empty((2 * f.shape[0], 3), np.uint32)
        e[0::2] = f
        e[1::2, 0], e[1::2, 1], e[1::2, 2] = f[:, 1] ^ 1, f[:, 0] ^ 1, TWIN
        n = self.base + 2 * self.n_fresh if n_nodes is None else n_nodes
        return n, e

    def expected(self):
        """(forward edge ids, whether each is marked) of the edges added with test()"""
        rows = np.array([r for r, _ in self.expect], np.int64)
        return 2 * self.pos[rows], np.array([w for _, w in self.expect], np.uint8)


def degree_fan(B, d):
    """A node of out-degree d: every third neighbour t_i (i = 0, 3, ...) has the edge t_i -> t_{i+1}, which witnesses
    a -> t_{i+1} (sum 200) with l_ac cycling through BOUNDS; the remaining neighbours have no witness."""
    a = B.fresh(1)[0]
    t = B.fresh(d)
    k = 0
    for i in range(d):
        if i % 3 == 0 and i + 1 < d:
            B.add(a, t[i], 100)
            B.add(t[i], t[i + 1], 100)
        elif i % 3 == 1:
            ln, want = BOUNDS[k % len(BOUNDS)]
            k += 1
            B.test(a, t[i], ln, want)
        else:
            B.add(a, t[i], 1000)
    return a


DEGREES = (0, 1, 2, 16, 17, 64, 65, 256, 257, 512, 513, 1024, 1025, 1536, 1537)


def degree_graph(base=0, n_nodes=None, seed=3):
    B = Builder(seed, base)
    subjects = {d: degree_fan(B, d) for d in DEGREES}
    n, e = B.graph(n_nodes)
    return B, subjects, n, e


def visits_graph():
    """Group nodes (d = 16) with W = 4096 and 4097, light nodes (d = 32) with W = 32768 and 32769: half of the
    neighbours (b) carry the long rows, the other half (c) sit in those rows and are tested against them."""
    B = Builder(5)
    subjects = {}
    for name, d, w in (("group_4096", 16, 4096), ("group_4097", 16, 4097), ("light_32768", 32, 32768), ("light_32769", 32, 32769)):
        a = B.fresh(1)[0]
        nb = d // 2
        row = w // nb
        rows = [row] * nb
        rows[0] += w - row * nb
        pool = B.fresh(max(rows))
        for j in range(nb):
            b = B.fresh(1)[0]
            B.add(a, b, 100)
            for c in pool[:rows[j]]:
                B.add(b, c, 100)
        for j in range(d - nb):
            ln, want = BOUNDS[j % len(BOUNDS)]
            B.test(a, pool[j], ln, want)
        subjects[name] = a
    n, e = B.graph()
    return B, subjects, n, e


# (copies, the highest id passes?) of one destination; the copies spread over the whole edge-id range
PARALLEL = ((2, True), (2, False), (3, True), (3, False), (4, True), (4, False))


def parallel_graph():
    """Parallel edges a -> c (2-4 copies) in every class: either the highest id is comparable and the lower ones are
    not (the pair of the highest copy is marked), or the reverse (nothing is marked: graph.cpp:1291-1293 keeps the
    highest id as the candidate)."""
    B = Builder(7)
    subjects = {}
    classes = (("group_a", 12, PARALLEL[:3]), ("group_b", 16, PARALLEL[3:]), ("light", 40, PARALLEL),
               ("heavy", 300, PARALLEL), ("heavy_chunked", 1500, PARALLEL))
    for name, d, groups in classes:
        a = B.fresh(1)[0]
        used = 0
        for copies, high_passes in groups:
            b, c = B.fresh(2)
            B.add(a, b, 100)
            B.add(b, c, 100)
            keys = (np.arange(copies) + B.rng.uniform(0.1, 0.9, copies)) / copies   # ascending: copy k has the k-th id
            for k in range(copies):
                last = k == copies - 1
                passes = last if high_passes else k == 0
                B.test(a, c, 200 if passes else 1000, int(high_passes and last), key=float(keys[k]))
            used += 1 + copies
        for t in B.fresh(d - used):
            B.add(a, t, 1000)
        subjects[name] = a
    n, e = B.graph()
    return B, subjects, n, e


def star_graph(hubs, spokes, links, seed):
    """`hubs` stars of `spokes` spokes, `links` spoke -> next spoke edges each (their witnesses for hub -> next spoke)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    e = []
    for h in range(hubs):
        hub = 2 * h * (spokes + 1)
        s = hub + 2 * (1 + np.arange(spokes))
        ln = rng.integers(1000, 5000, spokes)
        e.append(np.stack([np.full(spokes, hub), s, ln], 1))
        k = np.sort(rng.choice(spokes - 1, links, replace=False))
        e.append(np.stack([s[k], s[k + 1], rng.integers(1, 1000, links)], 1))
    f = np.concatenate(e)
    out = np.empty((2 * f.shape[0], 3), np.uint32)
    out[0::2] = f
    out[1::2, 0], out[1::2, 1], out[1::2, 2] = f[:, 1] ^ 1, f[:, 0] ^ 1, TWIN
    return 2 * hubs * (spokes + 1), out, [2 * h * (spokes + 1) for h in range(hubs)]


def full_chunk_graph(keys_in_chunk):
    """One node whose destinations all hash into chunk 0 of its 3 hash chunks (2048 <= d < 2304), so that the table of
    that chunk holds `keys_in_chunk` keys.  Some destinations b lead to destinations c (tested, BOUNDS) and to nodes x
    outside the node's row, half of them in chunk 0 too: absent keys whose probe crosses the whole full table."""
    ids = 2 + 2 * np.arange(20 * keys_in_chunk)
    in0 = ids[hash_chunk_of(ids, 3) == 0]
    dests, absent0 = in0[:keys_in_chunk], in0[keys_in_chunk:keys_in_chunk + 64]
    absent1 = ids[hash_chunk_of(ids, 3) == 1][:64]
    B = Builder(11)
    a = 0
    for j in range(keys_in_chunk):
        if j % 16 == 0 and j + 1 < keys_in_chunk:
            b, c = int(dests[j]), int(dests[j + 1])
            B.add(b, c, 100)
            B.add(b, int(absent0[(j // 16) % 64]), 100)
            B.add(b, int(absent1[(j // 16) % 64]), 100)
            B.add(a, b, 100)
        elif j % 16 == 1:
            ln, want = BOUNDS[(j // 16) % len(BOUNDS)]
            B.test(a, int(dests[j]), ln, want)
        else:
            B.add(a, int(dests[j]), 1000)
    n_nodes = int(max(in0.max(), absent1.max())) + 2
    n, e = B.graph(n_nodes)
    return B, a, n, e


def star_records(spokes, seed=13):
    """Overlap records with one read that `spokes` others begin on (the hub - spoke geometry of
    synth.generate_repeat_hubs), the spokes tiled onto each other in pairs, on a small uniform background."""
    base = synth.generate(200_000, 30, 10000, seed=seed)
    rng = np.random.Generator(np.random.PCG64(seed))
    L, hub = 10000, base.n_reads
    ids = hub + 1 + np.arange(spokes)
    o = np.empty(spokes, np.int64)            # repeat bases at the start of each spoke: hub[L - o, L) ~ spoke[0, o)
    o[0::2] = 2900 - rng.integers(0, 200, (spokes + 1) // 2)
    o[1::2] = o[0::2][:spokes // 2] - rng.integers(600, 901, spokes // 2)
    z = np.zeros(spokes, np.int64)
    hub_rows = np.stack([np.full(spokes, hub), ids, L - o, np.full(spokes, L), z, o, z], 1)
    i, j = ids[0::2][:spokes // 2], ids[1::2]   # spoke j starts o_i - o_j bases after spoke i
    d = o[0::2][:spokes // 2] - o[1::2]
    z = np.zeros(j.shape[0], np.int64)
    tile_rows = np.stack([i, j, d, np.full(j.shape[0], L), z, L - d, z], 1)
    rec = np.concatenate([base.records, hub_rows.astype(np.uint32), tile_rows.astype(np.uint32)])
    rec = np.ascontiguousarray(rec[np.lexsort((rec[:, 2], rec[:, 1], rec[:, 0]))])
    read_len = np.concatenate([base.read_len, np.full(spokes + 1, L, np.uint32)])
    return synth.Dataset(read_len=read_len, records=rec, genome_len=base.genome_len, meta=dict(base.meta, hub=hub))


def oracle_expectations(B, n, e):
    """the oracle marks exactly the tested edges meant to pass"""
    m, _ = O.transitive(n, e)
    ids, want = B.expected()
    assert_same(m[ids], want, "oracle marks of the tested edges")
    assert_same(m[ids + 1], want, "... and of their twins")
    assert 0 < int(want.sum()) < want.shape[0]


# ---- CPU: the graphs contain what they claim ---------------------------------------------------------------------------
def test_degree_graph_covers_every_class():
    B, subj, n, e = degree_graph()
    M = Model(n, e)
    for d, a in subj.items():
        assert M.deg[a] == d
    g = lambda d: subj[d]
    assert not M.group[g(0)] and not M.group[g(1)] and not M.light[g(1)]
    assert M.group[g(2)] and M.group[g(16)] and M.light[g(17)] and M.light[g(64)]
    for d in (65, 256, 257, 512, 513, 1024):
        assert M.heavy[g(d)] and not M.chunked[g(d)] and M.items_of(g(d)) == (d + 255) // 256
    for d, nca in ((1025, 2), (1536, 2), (1537, 3)):
        assert M.chunked[g(d)] and M.items_of(g(d)) == nca * ((d + 255) // 256)
        assert M.chunk_load(g(d)).max() <= HEAVY_CAP
    # stream chunks end at 256 and 512 entries: one node on each side
    assert [(M.deg[g(d)] + 255) // 256 for d in (256, 257, 512, 513)] == [1, 2, 2, 3]
    # witnesses for some edges of every node of degree >= 2, on both sides of the 12 % bounds
    ids, want = B.expected()
    src = e[ids, 0]
    for d in DEGREES[2:]:
        w = want[src == g(d)]
        assert w.any() and (d < 5 or not w.all()), d
    oracle_expectations(B, n, e)


def test_visits_graph_sits_on_the_hand_offs():
    B, subj, n, e = visits_graph()
    M = Model(n, e)
    for name, (d, w, cls, to_heavy) in {"group_4096": (16, 4096, M.group, False), "group_4097": (16, 4097, M.group_to_heavy, True),
                                         "light_32768": (32, 32768, M.light, False),
                                         "light_32769": (32, 32769, M.light_to_heavy, True)}.items():
        a = subj[name]
        assert (M.deg[a], M.W[a]) == (d, w) and cls[a], name
        assert M.items_of(a) == int(to_heavy)
    oracle_expectations(B, n, e)


def test_parallel_graph_has_copies_in_every_class():
    B, subj, n, e = parallel_graph()
    M = Model(n, e)
    a = subj
    assert M.group[a["group_a"]] and M.group[a["group_b"]] and M.light[a["light"]]
    assert M.heavy[a["heavy"]] and not M.chunked[a["heavy"]] and M.chunked[a["heavy_chunked"]]
    for name, node in subj.items():
        fwd = e[0::2]
        mine = fwd[fwd[:, 0] == node]
        dst, cnt = np.unique(mine[:, 1], return_counts=True)
        assert sorted(cnt[cnt > 1].tolist()) == sorted(c for c, _ in (PARALLEL[:3] if name == "group_a" else
                                                                      PARALLEL[3:] if name == "group_b" else PARALLEL))
        # the copies span the edge-id range: the first and the last copy of each destination are far apart
        ids = np.flatnonzero((e[:, 0] == node) & np.isin(e[:, 1], dst[cnt > 1]))
        for c in dst[cnt > 1]:
            cid = ids[e[ids, 1] == c]
            assert cid.max() - cid.min() > e.shape[0] // 20
    oracle_expectations(B, n, e)


def test_sparse_graph_keeps_its_edges_at_the_top_ids():
    n_nodes = 6_000_000
    B, subj, n, e = degree_graph(base=n_nodes - 60_000, n_nodes=n_nodes, seed=4)
    assert n == n_nodes and e[:, :2].min() >= n_nodes - 60_000 and e[:, :2].max() < n_nodes - 1000
    M = Model(n, e)
    assert M.group.any() and M.light.any() and M.heavy.any() and M.chunked.any()
    oracle_expectations(B, n, e)


def test_star_demand_exceeds_a_list_sized_from_the_edge_count():
    """Heavy items grow with d^2, edges with d: a list of E / 16 + 4096 items cannot hold one large hub."""
    n, e, hubs = star_graph(1, 60_000, 1000, seed=1)
    M = Model(n, e)
    assert e.shape[0] == 122_000 and M.items_of(hubs[0]) == 79 * 235 > e.shape[0] // 16 + 4096
    n, e, hubs = star_graph(3, 40_000, 500, seed=2)
    M = Model(n, e)
    assert sum(M.items_of(h) for h in hubs) == 3 * 53 * 157 > e.shape[0] // 16 + 4096
    _, pairs = O.transitive(n, e)
    assert 0 < pairs < 1500


@pytest.mark.parametrize("keys", [HEAVY_CAP, HEAVY_CAP + 1])
def test_full_chunk_graph_fills_one_chunk(keys):
    B, a, n, e = full_chunk_graph(keys)
    M = Model(n, e)
    assert M.chunked[a] and num_hash_chunks(M.deg[a]) == 3
    assert M.chunk_load(a).tolist() == [keys, 0, 0]
    # lookups of destinations outside the row, hashed into the full chunk and into an empty one
    two_hop = np.unique(e[np.isin(e[:, 0], e[e[:, 0] == a, 1]), 1])
    absent = np.setdiff1d(two_hop, e[e[:, 0] == a, 1])
    assert (hash_chunk_of(absent, 3) == 0).sum() >= 32 and (hash_chunk_of(absent, 3) == 1).sum() >= 32
    if keys == HEAVY_CAP:
        oracle_expectations(B, n, e)


def test_session_graph_counters_model():
    ds = synth.generate_repeat_hubs(genome_len=2_000_000, n_hubs=2)
    P = O.Pipeline(ds.records, ds.flat_piles()).run()
    M = Model(P.n_nodes, P.edges)
    assert M.chunked.sum() >= 2 and M.heavy_items() > 0 and M.two_hop() > 0


def test_star_records_give_one_large_hub():
    ds = star_records(70_000)
    P = O.Pipeline(ds.records, ds.flat_piles()).run()
    M = Model(P.n_nodes, P.edges)
    hub = int(np.argmax(M.deg))
    assert M.deg[hub] == 70_000 and P.n_pairs > 1000
    # more items than a list sized from the session's edge capacity (2 x the records, / 16 + 4096) would hold
    assert M.items_of(hub) > 2 * ds.records.shape[0] // 16 + 4096


# ---- GPU: every path against the oracle --------------------------------------------------------------------------------
def _same_as_oracle(ctx, n, e, what):
    want, want_pairs = O.transitive(n, e)
    got, got_pairs = ctx.transitive_reduce(n, e)
    assert got_pairs == want_pairs, what
    assert_same(got, want, what)


@pytest.mark.gpu
def test_degree_boundaries_match_oracle(ctx):
    _, _, n, e = degree_graph()
    _same_as_oracle(ctx, n, e, "degree boundaries")


@pytest.mark.gpu
def test_visit_hand_offs_match_oracle(ctx):
    _, _, n, e = visits_graph()
    _same_as_oracle(ctx, n, e, "visit hand-offs")


@pytest.mark.gpu
def test_parallel_edges_match_oracle(ctx):
    _, _, n, e = parallel_graph()
    _same_as_oracle(ctx, n, e, "parallel edges")


@pytest.mark.gpu
def test_sparse_ids_match_oracle(ctx):
    n_nodes = 6_000_000
    _, _, n, e = degree_graph(base=n_nodes - 60_000, n_nodes=n_nodes, seed=4)
    _same_as_oracle(ctx, n, e, "sparse ids")


@pytest.mark.gpu
@pytest.mark.parametrize("hubs,spokes,links", [(1, 60_000, 1000), (3, 40_000, 500)])
def test_heavy_work_list_demand_matches_oracle(ctx, hubs, spokes, links):
    n, e, _ = star_graph(hubs, spokes, links, seed=hubs)
    _same_as_oracle(ctx, n, e, f"{hubs} x {spokes}-spoke star")


@pytest.mark.gpu
def test_full_hash_chunk_matches_oracle(ctx):
    _, _, n, e = full_chunk_graph(HEAVY_CAP)
    _same_as_oracle(ctx, n, e, "a hash chunk of exactly 2048 destinations")


@pytest.mark.gpu
def test_overfull_hash_chunk_is_refused(ctx):
    _, _, n, e = full_chunk_graph(HEAVY_CAP + 1)
    with pytest.raises(api.RalaB200Error, match="hash chunk"):
        ctx.transitive_reduce(n, e)


@pytest.mark.gpu
def test_session_counters_match_the_model(ctx):
    ds = synth.generate_repeat_hubs(genome_len=2_000_000, n_hubs=2)
    piles = ds.flat_piles()
    P = O.Pipeline(ds.records, piles).run()
    M = Model(P.n_nodes, P.edges)
    G = api.Graph(ctx)
    G.set_piles(piles).set_hills(None).set_overlaps(ds.records)
    for _ in range(3):   # eager, captured, replayed
        G.run()
        c = G.counts()
        assert c["n_heavy_items"] == M.heavy_items()
        assert c["n_two_hop"] == M.two_hop()
    assert_same(G.marked(), P.marked, "marks")
    G.close()


@pytest.mark.gpu
def test_large_hub_through_the_session_and_two_ranks(ctx):
    ds = star_records(70_000)
    piles = ds.flat_piles()
    P = O.Pipeline(ds.records, piles).run()
    G = api.Graph(ctx)
    G.set_piles(piles).set_hills(None).set_overlaps(ds.records)
    G.run()
    c = G.counts()
    assert c["n_heavy_items"] == Model(P.n_nodes, P.edges).heavy_items()
    assert_same(G.edges(), P.edges, "edges")
    assert_same(G.marked(), P.marked, "marks")
    G.close()
    M = api.Multi([0, 0])
    M.set_barrier_timeout_ms(20000)
    M.set_piles(piles).set_shards(ds.records).plan().run()
    e, m = M.all_edges()
    assert_same(e, P.edges, "edges (2 ranks)")
    assert_same(m, P.marked, "marks (2 ranks)")
    assert M.counts()["n_transitive_pairs"] == P.n_pairs
    M.close()


@pytest.mark.gpu
def test_a_shard_refuses_the_whole_session_stages(ctx):
    """After set_shard(world > 1) the session holds one rank's records: build, transitive and run refuse (status -3,
    RALA_B200_ERR_STATE) instead of giving a partial CSR or no marks; back at world 1 the same session runs."""
    ds = star_records(2_000)
    piles = ds.flat_piles()
    P = O.Pipeline(ds.records, piles).run()
    G = api.Graph(ctx)
    G.set_piles(piles).set_hills(None).set_overlaps(ds.records)
    G._call("rala_b200_graph_set_shard", C.c_uint32(0), C.c_int(1), C.c_int(2))
    G.classify()
    G.finalize()
    for stage in (G.build, G.transitive, G.run):
        with pytest.raises(api.RalaB200Error, match=r"status -3: .*rank 1 of 2.*phase calls"):
            stage()
    G._call("rala_b200_graph_set_shard", C.c_uint32(0), C.c_int(0), C.c_int(1))
    G.run()
    assert_same(G.edges(), P.edges, "edges")
    assert_same(G.marked(), P.marked, "marks")
    G.close()
