"""K2, the graph build (rala_b200/csrc/graph_build.cu), at its tile, scan and hand-off boundaries, against the oracle's
restatement of graph.cpp:552-632 (O.Pipeline.build_edges) and the transitive pass that reads its CSR rows.

The build runs three kernels over the final `overlaps` list and the pile table:
  k_count_edges  per 512-entry list tile (kEmitTile = 256 threads x 2 items, item r of thread t = entry r * 256 + t): the
                 dovetails (tag kAB / kBA, both piles alive) of the tile, and the out-degree of their two source slots
  k_scan_piles   block 0 first turns the tile counts into edge-id bases, 1 024 tiles per chunk with a carry between
                 chunks; then one look-back over the piles, 1 024 piles per tile (4 per thread: a 16-byte path and a
                 scalar path for the last, ragged group), two packed counts (alive piles, edges): seq_to_node, row_ptr
                 and the fill cursor of both nodes of a pile; the last tile writes row_ptr[n_nodes] = E
  k_emit_edges   edge pair 2j, 2j + 1 of the j-th dovetail, ranked inside its tile in (item, warp, lane) order, straight
                 into its CSR rows (col = {dst, len}, col_eid), clearing its bytes of T; k_scan_piles clears T[E, E
                 rounded up to 16), which k_finalize_marks reads
The count and emit grids are sized from the session's list capacity (the largest record count seen, rounded up to 128,
at least 1 024), capped at 148 x 8 = 1 184 and 148 x 5 = 740 blocks: above those tile counts a block loops over tiles.

Every input here sits on one of these boundaries, and an unmarked test asserts that it does (list lengths, per-tile
dovetail counts, dead-pile positions, final-pass kills, the stale T window): an input that drifts off its boundary fails
without a GPU.  The GPU tests compare edges, node ids, counts, marks and the CSR rows themselves with the oracle."""
import contextlib
import functools

import numpy as np
import pytest

from oracle import oracle as O
from rala_b200 import api
from tests.replay import assert_same

# ---- the kernels' boundaries, restated (graph_build.cu, lists.cuh, common.cuh) -----------------------------------------
EMIT_TILE = 512
SCAN_CHUNK = 1024            # list tiles per block-0 chunk of k_scan_piles
PILE_TILE = 1024             # piles per look-back tile
COUNT_BLOCKS, EMIT_BLOCKS = 148 * 8, 148 * 5
HAS_HILL, HAS_REGION = 1, 2
INF = 0xFFFFFFFF

L = 10_000                   # every read and every alive pile: [0, L)


def list_cap(n):
    """the session's list capacity after set_overlaps of n records (never shrinks)"""
    return max(1024, (n + 127) // 128 * 128)


def tiles(n):
    return (n + EMIT_TILE - 1) // EMIT_TILE


# ---- builders ----------------------------------------------------------------------------------------------------------
def layout(ids, seed, gap=(600, 1400), chain=(1, 12)):
    """Pure dovetail records among the piles `ids`: the piles, in random order, are cut into chains of reads laid along a
    genome (gaps drawn from `gap`), each read on a random strand.  Two reads of a chain whose starts are 1 000 .. 8 000
    bases apart overlap by 2 000 .. 9 000 (at most 0.9 L: the near-containment rule never applies) and give one record,
    with a random one of the two as a: kAB and kBA, orientation 0 and 1, all occur.  Chains of one read leave a pile
    without edges, chains of two give out-degree 1, longer chains use both slots; shared geometry gives transitive
    triangles."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ids = rng.permutation(np.asarray(ids, np.int64))
    n = ids.shape[0]
    if n == 0:
        return np.zeros((0, 7), np.uint32)
    chain_of = np.repeat(np.arange(n), rng.integers(chain[0], chain[1] + 1, n))[:n]
    pos = np.cumsum(rng.integers(gap[0], gap[1] + 1, n)) + chain_of * 100_000
    strand = rng.integers(0, 2, n)
    rows, keys = [], []
    for j in range(1, 16):
        i = np.arange(n - j)
        k = i + j
        d = pos[k] - pos[i]
        ok = (chain_of[i] == chain_of[k]) & (d >= 1000) & (d <= 8000)
        i, k, d = i[ok], k[ok], d[ok]
        if not i.shape[0]:
            continue
        # the overlap in each read's own coordinates (forward strand of the read)
        ci = np.where(strand[i] == 0, np.stack([d, np.full_like(d, L)]), np.stack([np.zeros_like(d), L - d])).T
        ck = np.where(strand[k] == 0, np.stack([np.zeros_like(d), L - d]), np.stack([d, np.full_like(d, L)])).T
        ori = strand[i] ^ strand[k]
        first = rng.integers(0, 2, i.shape[0]).astype(bool)   # which read is a
        a = np.where(first, ids[i], ids[k])
        b = np.where(first, ids[k], ids[i])
        ca = np.where(first[:, None], ci, ck)
        cb = np.where(first[:, None], ck, ci)
        rows.append(np.column_stack([a, b, ca, cb, ori]))
        keys.append(np.minimum(i, k) * 16 + j)
    if not rows:
        return np.zeros((0, 7), np.uint32)
    r = np.concatenate(rows)
    return np.ascontiguousarray(r[np.argsort(np.concatenate(keys), kind="stable")].astype(np.uint32))


def filler(ids, n, seed):
    """n non-dovetail entries between the piles `ids`: internals (kX) and containments (kA, kB), both orientations.  Kept
    lists are not resolved again, so the containments kill nothing."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ids = np.asarray(ids, np.int64)
    a = ids[rng.integers(0, ids.shape[0], n)]
    b = ids[(np.searchsorted(ids, a) + 1 + rng.integers(0, ids.shape[0] - 1, n)) % ids.shape[0]]
    kind = rng.integers(0, 3, n)
    coords = np.array([[1000, 3000, 1000, 3000],          # kX: large overhangs on both sides
                       [100, L - 100, 0, L],              # kA: b inside a
                       [0, L, 100, L - 100]])             # kB: a inside b
    return np.ascontiguousarray(np.column_stack([a, b, coords[kind], rng.integers(0, 2, n)]).astype(np.uint32))


def hub(x, partners, seed):
    """one record x -> y per partner, every one a kAB from slot 2x (orientation 0 or 1): one row of len(partners) edges"""
    rng = np.random.Generator(np.random.PCG64(seed))
    y = np.asarray(partners, np.int64)
    d = rng.integers(1000, 8001, y.shape[0])
    ori = rng.integers(0, 2, y.shape[0])
    bb = np.where(ori == 0, 0, d)
    be = np.where(ori == 0, L - d, L)
    return np.ascontiguousarray(np.column_stack([np.full_like(y, x), y, d, np.full_like(d, L), bb, be, ori]).astype(np.uint32))


def invalid(n):
    """n records the duplicate filter dropped: they size the session's lists and reach no list"""
    r = np.zeros((n, 7), np.uint32)
    r[:, 6] = 2
    return r


def pile_table(n, dead=(), seed=0):
    """n piles [0, L), the `dead` ones 0 0; random HAS_HILL / HAS_REGION flags on the alive ones (pile.y carries them in
    its top bits)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    piles = np.zeros((n, 2), np.uint32)
    piles[:, 1] = L
    flags = rng.integers(0, 4, n).astype(np.uint8)
    dead = np.asarray(list(dead), np.int64)
    piles[dead] = 0
    flags[dead] = 0
    return piles, flags


def alive_ids(piles):
    return np.flatnonzero(piles[:, 1] != 0)


# ---- case 1: list lengths through run() --------------------------------------------------------------------------------
LENGTHS = [0, 1, 511, 512, 513,
           EMIT_BLOCKS * EMIT_TILE - 1, EMIT_BLOCKS * EMIT_TILE, EMIT_BLOCKS * EMIT_TILE + 1,
           SCAN_CHUNK * EMIT_TILE - 1, SCAN_CHUNK * EMIT_TILE, SCAN_CHUNK * EMIT_TILE + 1,
           COUNT_BLOCKS * EMIT_TILE - 1, COUNT_BLOCKS * EMIT_TILE, COUNT_BLOCKS * EMIT_TILE + 1,
           2 * SCAN_CHUNK * EMIT_TILE + 513]
LENGTH_PILES = 400_000


@functools.lru_cache(maxsize=1)
def length_inputs():
    piles, flags = pile_table(LENGTH_PILES, seed=1)
    rec = layout(np.arange(LENGTH_PILES), seed=2)
    assert rec.shape[0] >= max(LENGTHS)
    return piles, flags, rec


@functools.lru_cache(maxsize=None)
def length_oracle(n):
    piles, flags, rec = length_inputs()
    return O.Pipeline(rec[:n], piles, flags).run()


# ---- case 2: per-tile patterns through set_kept_overlaps ---------------------------------------------------------------
def _pattern(name, rng):
    m = np.zeros(EMIT_TILE, bool)
    if name == "one":
        m[rng.integers(0, EMIT_TILE)] = True
    elif name == "first":
        m[0] = True
    elif name == "last":
        m[-1] = True
    elif name == "all_but_one":
        m[:] = True
        m[rng.integers(0, EMIT_TILE)] = False
    elif name == "all":
        m[:] = True
    elif name == "item0":
        m[:256] = True
    elif name == "item1":
        m[256:] = True
    elif name == "item0_odd_lanes":
        m[1:256:2] = True
    elif name == "item1_one_warp":
        w = int(rng.integers(0, 8))
        m[256 + 32 * w:256 + 32 * (w + 1)] = True
    elif name == "random":
        m[:] = rng.random(EMIT_TILE) < 0.5
    return m


PATTERNS = ["none", "one", "first", "last", "all_but_one", "all", "item0", "item1", "item0_odd_lanes", "item1_one_warp", "random"]
KEPT_TILES = (12, COUNT_BLOCKS + 16)   # a few tiles; more than both grids have blocks
KEPT_TAIL = 300                        # a last, ragged tile
KEPT_PILES = 90_000


@functools.lru_cache(maxsize=None)
def kept_inputs(n_tiles):
    """(piles, flags, kept list, dovetail mask, pattern of every tile): tile t follows PATTERNS[t % len], dovetails in
    file order from a layout, filler elsewhere"""
    rng = np.random.Generator(np.random.PCG64(n_tiles))
    piles, flags = pile_table(KEPT_PILES, seed=3)
    names = [PATTERNS[t % len(PATTERNS)] for t in range(n_tiles)]
    mask = np.concatenate([_pattern(nm, rng) for nm in names] + [rng.random(KEPT_TAIL) < 0.5])
    dov = layout(np.arange(KEPT_PILES), seed=4)
    k = int(mask.sum())
    assert dov.shape[0] >= k
    kept = np.empty((mask.shape[0], 7), np.uint32)
    kept[mask] = dov[:k]
    kept[~mask] = filler(np.arange(KEPT_PILES), int((~mask).sum()), seed=5)
    return piles, flags, kept, mask, names


@functools.lru_cache(maxsize=None)
def kept_oracle(n_tiles):
    piles, flags, kept, _, _ = kept_inputs(n_tiles)
    P = O.Pipeline(np.zeros((0, 7), np.uint32), piles, flags)
    P.ovl = kept.copy()
    return P.build_edges().transitive()


# ---- case 3: pile tables -----------------------------------------------------------------------------------------------
def _dead_mod(n, m):
    """piles at positions = m mod 4 in every third group of four"""
    i = np.arange(n)
    return i[(i % 4 == m) & ((i // 4) % 3 == 0)]


def _random_dead(n, frac, seed):
    """random dead piles, and one in the ragged last group of four"""
    rng = np.random.Generator(np.random.PCG64(seed))
    dead = rng.random(n) < frac
    if n % 4:
        dead[n - n % 4 + (n % 4) // 2] = True
    return np.flatnonzero(dead)


BIG_PILES = 300_001
HUB_EDGES = 70_000
TABLES = {
    "n1": (1, []), "n2": (2, []), "n3": (3, []), "n4": (4, []), "n5": (5, []),
    "n5_dead1": (5, [1]),
    "n1024_dead_mod0": (1024, _dead_mod(1024, 0)), "n1024_dead_mod1": (1024, _dead_mod(1024, 1)),
    "n1024_dead_mod2": (1024, _dead_mod(1024, 2)), "n1024_dead_mod3": (1024, _dead_mod(1024, 3)),
    "n1023_random": (1023, _random_dead(1023, 0.3, 6)), "n1025_random": (1025, _random_dead(1025, 0.3, 7)),
    "n2049_random": (2049, _random_dead(2049, 0.3, 8)),
    "dead_tile": (3 * PILE_TILE + 7, np.arange(PILE_TILE, 2 * PILE_TILE)),
    "last_alive": (2049, np.arange(2048)),
    "all_dead": (1025, np.arange(1025)),
    "big_hub": (BIG_PILES, _random_dead(BIG_PILES, 0.1, 9)),
}


@functools.lru_cache(maxsize=None)
def table_inputs(name):
    n, dead = TABLES[name]
    piles, flags = pile_table(n, dead, seed=10)
    ids = alive_ids(piles)
    big = name == "big_hub"
    rec = layout(ids, seed=11, gap=(2000, 3000) if big else (600, 1400), chain=(1, 6) if big else (1, 12))
    if big:
        x = int(ids[0])
        rng = np.random.Generator(np.random.PCG64(12))
        rec = np.concatenate([rec, hub(x, rng.choice(ids[1:], HUB_EDGES, replace=False), seed=13)])
    return piles, flags, rec


@functools.lru_cache(maxsize=None)
def table_oracle(name):
    piles, flags, rec = table_inputs(name)
    return O.Pipeline(rec, piles, flags).run()


# ---- case 5: final-pass kills ------------------------------------------------------------------------------------------
KILL_GROUPS = 64


@functools.lru_cache(maxsize=1)
def kill_inputs():
    """Groups of three reads c, a, b (starts 0, 2 000, 4 000 on one strand) behind a layout background, in file order
    (c, b), (c, a), (a, b): all dovetails on the first table.  The second table cuts b's pile to [0, 8 000), where a's
    overlap ends: in the final pass (c, b) still types kAB, then (a, b) types kA and kills b, so (c, b), tagged as a
    dovetail, is dropped (graph.cpp:869-876) and b gets no node id."""
    n_bg = 5000
    n = n_bg + 3 * KILL_GROUPS
    piles, flags = pile_table(n, seed=14)
    bg = layout(np.arange(n_bg), seed=15)
    g = n_bg + 3 * np.arange(KILL_GROUPS)
    c, a, b = g, g + 1, g + 2
    z, full = np.zeros_like(g), np.full_like(g, L)
    rows = np.stack([np.stack([c, b, z + 4000, full, z, z + 6000, z], 1),
                     np.stack([c, a, z + 2000, full, z, z + 8000, z], 1),
                     np.stack([a, b, z + 2000, full, z, z + 8000, z], 1)], 1).reshape(-1, 7)
    rec = np.ascontiguousarray(np.concatenate([bg[:len(bg) // 2], rows, bg[len(bg) // 2:]]).astype(np.uint32))
    cut = piles.copy()
    cut[b, 1] = 8000
    return piles, cut, flags, rec, b


def kill_oracle_stages():
    piles, cut, flags, rec, _ = kill_inputs()
    P = O.Pipeline(rec, piles, flags).classify()
    P.set_piles(cut).retrim()
    while P.retrim_promote():
        pass
    before = P.ovl.copy()
    P.final_containment().build_edges().transitive()
    return before, P


# ---- case 6: one session, a large graph, then smaller ones -------------------------------------------------------------
REUSE_PILES = 60_000


@functools.lru_cache(maxsize=1)
def reuse_inputs():
    """The large record list and, for E % 16 = 2 and 14, the shortest prefix whose edges end inside a 16-edge group that
    the large graph marked behind them: a T byte left over from the large graph changes n_transitive_pairs."""
    piles, flags = pile_table(REUSE_PILES, seed=16)
    rec = layout(np.arange(REUSE_PILES), seed=17)
    big = O.Pipeline(rec, piles, flags).run()
    sizes = {}
    for r in (2, 14):
        n = 2000 + (r // 2 - 2000) % 8
        while True:
            e = 2 * n
            if big.marked[e:(e + 15) // 16 * 16].any():
                break
            n += 8
        sizes[r] = n
    return piles, flags, rec, big, sizes


@functools.lru_cache(maxsize=None)
def reuse_oracle(n):
    piles, flags, rec, big, _ = reuse_inputs()
    return big if n == rec.shape[0] else O.Pipeline(rec[:n], piles, flags).run()


# ---- case 7: the multi-GPU edge phase ----------------------------------------------------------------------------------
SHARDS = {2: [(0, 0), (0, 513)], 3: [(0, 511), (511, 1023), (1023, 1536)]}


@functools.lru_cache(maxsize=1)
def multi_inputs():
    piles, flags = pile_table(3000, seed=18)
    return piles, flags, layout(np.arange(3000), seed=19)[:1536]


def lone_pile_inputs():
    """one alive pile of 9: two nodes, fewer than the ranks of the 3-rank session"""
    piles, flags = pile_table(9, [0, 1, 2, 3, 5, 6, 7, 8], seed=20)
    return piles, flags, invalid(7)


# ---- CPU: the inputs are what they claim -------------------------------------------------------------------------------
def test_designed_records_type_as_intended():
    piles, _, rec = length_inputs()
    _, t = O.trim_type_batch(rec[:200_000], piles)
    assert np.isin(t, (O.KAB, O.KBA)).all()
    combos = {(int(x), int(o)) for x, o in zip(t, rec[:200_000, 6] & 1)}
    assert combos == {(O.KAB, 0), (O.KAB, 1), (O.KBA, 0), (O.KBA, 1)}
    f = filler(np.arange(1000), 3000, seed=0)
    _, t = O.trim_type_batch(f, pile_table(1000)[0])
    want = np.select([f[:, 2] == 1000, f[:, 2] == 100, f[:, 2] == 0], [O.KX, O.KA, O.KB], 255)
    assert_same(t, want.astype(np.uint8), "filler types")
    for o in (0, 1):
        assert set(t[(f[:, 6] & 1) == o].tolist()) == {O.KX, O.KA, O.KB}
    h = hub(0, np.arange(1, 101), seed=0)
    _, t = O.trim_type_batch(h, pile_table(101)[0])
    assert (t == O.KAB).all() and set((h[:, 6] & 1).tolist()) == {0, 1}


@pytest.mark.parametrize("n", [513, 20_000])
def test_run_keeps_the_dovetails_in_file_order(n):
    piles, flags, rec = length_inputs()
    P = length_oracle(n)
    assert_same(P.ovl, rec[:n], "final overlaps")
    assert P.int.shape[0] == 0 and P.edges.shape[0] == 2 * n
    assert P.n_pairs > 0 and (P.seq_to_node != INF).all()


def test_list_lengths_sit_on_the_grid_and_chunk_boundaries():
    t = [tiles(n) for n in LENGTHS]
    assert t[:5] == [0, 1, 1, 1, 2]
    count_grid = [min(tiles(list_cap(n)), COUNT_BLOCKS) for n in LENGTHS]
    emit_grid = [min(tiles(list_cap(n)), EMIT_BLOCKS) for n in LENGTHS]
    # one length on each side of the point where the emit grid (740 blocks) and the count grid (1 184) start to loop
    assert [tiles(list_cap(n)) > EMIT_BLOCKS for n in LENGTHS[5:8]] == [False, False, True]
    assert [tiles(list_cap(n)) > COUNT_BLOCKS for n in LENGTHS[11:14]] == [False, False, True]
    assert emit_grid[7] == EMIT_BLOCKS and count_grid[13] == COUNT_BLOCKS
    # block 0's chunks of 1 024 tiles: exactly one chunk, one chunk, a second chunk of one tile; past two full chunks
    assert [tiles(n) for n in LENGTHS[8:11]] == [SCAN_CHUNK, SCAN_CHUNK, SCAN_CHUNK + 1]
    assert tiles(LENGTHS[-1]) > 2 * SCAN_CHUNK
    # the records themselves are the list: pure dovetails
    piles, _, rec = length_inputs()
    _, ty = O.trim_type_batch(rec[:max(LENGTHS)], piles)
    assert np.isin(ty, (O.KAB, O.KBA)).all()
    # the reused session runs from large to small: its grids stay those of the largest list
    assert tiles(list_cap(max(LENGTHS))) > COUNT_BLOCKS


@pytest.mark.parametrize("n_tiles", KEPT_TILES)
def test_kept_lists_have_the_claimed_tile_patterns(n_tiles):
    piles, _, kept, mask, names = kept_inputs(n_tiles)
    _, ty = O.trim_type_batch(kept, piles)
    dov = np.isin(ty, (O.KAB, O.KBA))
    assert_same(dov, mask, "dovetails where the pattern puts them")
    assert set(ty[~mask].tolist()) == {O.KX, O.KA, O.KB}
    per_tile = [int(dov[t * EMIT_TILE:(t + 1) * EMIT_TILE].sum()) for t in range(tiles(kept.shape[0]))]
    assert {0, 1, 511, 512} <= set(per_tile)
    assert kept.shape[0] % EMIT_TILE == KEPT_TAIL
    items = dov[:n_tiles * EMIT_TILE].reshape(n_tiles, 2, 256)   # [tile, item, thread]
    only0 = [t for t in range(n_tiles) if items[t, 0].any() and not items[t, 1].any()]
    only1 = [t for t in range(n_tiles) if items[t, 1].any() and not items[t, 0].any()]
    assert only0 and only1
    if n_tiles > COUNT_BLOCKS:
        assert tiles(list_cap(kept.shape[0])) > COUNT_BLOCKS
    P = kept_oracle(n_tiles)
    assert P.edges.shape[0] == 2 * int(mask.sum()) and P.n_pairs > 0


@pytest.mark.parametrize("name", list(TABLES))
def test_pile_tables_have_the_claimed_shapes(name):
    n, dead = TABLES[name]
    piles, flags, rec = table_inputs(name)
    alive = piles[:, 1] != 0
    assert piles.shape[0] == n and not alive[np.asarray(dead, np.int64)].any()
    assert alive.sum() == n - len(dead)
    # list entries only touch alive piles
    assert alive[rec[:, 0]].all() and alive[rec[:, 1]].all()
    P = table_oracle(name)
    assert_same(P.ovl, rec, "final overlaps")
    if name.startswith("n1024_dead_mod"):
        m = int(name[-1])
        assert set((np.flatnonzero(~alive) % 4).tolist()) == {m}
    if name in ("n1023_random", "n1025_random", "n2049_random"):
        assert set((np.flatnonzero(~alive) % 4).tolist()) == {0, 1, 2, 3} and n % 4 != 0
        assert not alive[n - n % 4:].all()   # a dead pile in the ragged last group
    if name == "dead_tile":
        assert not alive[PILE_TILE:2 * PILE_TILE].any() and alive[:PILE_TILE].all() and alive[2 * PILE_TILE:].all()
    if name == "last_alive":
        assert np.flatnonzero(alive).tolist() == [n - 1]
    if name == "all_dead":
        assert not alive.any() and P.n_nodes == 0
    if alive.sum() >= 20:
        # flags in the top bits of alive piles, and every out-degree class: none, one, both slots used
        assert set(flags[alive].tolist()) == {0, HAS_HILL, HAS_REGION, HAS_HILL | HAS_REGION}
        deg = np.bincount(P.edges[:, 0].astype(np.int64), minlength=P.n_nodes).reshape(-1, 2)
        assert (deg.sum(1) == 0).any() and (deg.sum(1) == 1).any() and (deg > 0).all(1).any()
    if name == "big_hub":
        deg = np.bincount(P.edges[:, 0].astype(np.int64), minlength=P.n_nodes)
        assert deg.max() >= HUB_EDGES and deg.max() < HUB_EDGES + 100


def test_final_pass_kills_a_tagged_dovetail():
    piles, cut, flags, rec, victims = kill_inputs()
    before, P = kill_oracle_stages()
    # on the table of the final pass, (c, b) types as a dovetail and a later entry (a, b) as kA
    _, ty = O.trim_type_batch(before, cut)
    cb = np.flatnonzero(np.isin(before[:, 1], victims) & (before[:, 2] == 4000))
    ab = np.flatnonzero(np.isin(before[:, 1], victims) & (before[:, 2] == 2000))
    assert cb.shape[0] == ab.shape[0] == KILL_GROUPS
    assert (ty[cb] == O.KAB).all() and (ty[ab] == O.KA).all() and (cb < ab).all()
    # both piles alive when (c, b) comes up; b is dead at the end: (c, b) is dropped and b has no node
    assert (P.piles[victims, 1] == 0).all() and (P.seq_to_node[victims] == INF).all()
    assert not np.isin(P.ovl[:, 1], victims).any() and not np.isin(P.ovl[:, 0], victims).any()
    assert P.ovl.shape[0] == before.shape[0] - 2 * KILL_GROUPS
    assert P.n_pairs > 0


def test_session_reuse_leaves_a_marked_window_behind_the_small_graphs():
    _, _, rec, big, sizes = reuse_inputs()
    assert big.edges.shape[0] == 2 * rec.shape[0] and big.n_pairs > 1000
    for r, n in sizes.items():
        P = reuse_oracle(n)
        e = P.edges.shape[0]
        assert e == 2 * n and e % 16 == r
        assert big.marked[e:(e + 15) // 16 * 16].any()


def test_multi_shards_sit_on_tile_boundaries():
    piles, flags, rec = multi_inputs()
    assert [e - b for b, e in SHARDS[2]] == [0, 513]
    assert [e - b for b, e in SHARDS[3]] == [511, 512, 513]
    P = O.Pipeline(rec, piles, flags).run()
    assert_same(P.ovl, rec, "final overlaps")
    piles, flags, rec = lone_pile_inputs()
    P = O.Pipeline(rec, piles, flags).run()
    assert P.n_nodes == 2 < 3 and P.edges.shape[0] == 0


# ---- GPU: against the oracle -------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _closing(session):
    try:
        yield session
    finally:
        session.close()


def check_csr(G, n_nodes, edges, what):
    """row_ptr = exclusive scan of the out-degrees, each row (sorted by edge id) = the oracle's edges of that source,
    col_eid a permutation of the edge ids"""
    row_ptr, col, eid = G.csr()
    e = edges.shape[0]
    deg = np.bincount(edges[:, 0].astype(np.int64), minlength=n_nodes)
    assert_same(row_ptr, np.concatenate([[0], np.cumsum(deg)]).astype(np.uint32), f"{what}: row_ptr")
    assert_same(np.sort(eid), np.arange(e, dtype=np.uint32), f"{what}: col_eid is a permutation")
    src = np.repeat(np.arange(n_nodes), deg)
    order = np.lexsort((eid, src))
    got = np.column_stack([src[order], col[order, 0], col[order, 1], eid[order]]).astype(np.int64)
    ids = np.lexsort((np.arange(e), edges[:, 0]))
    want = np.column_stack([edges[ids, 0], edges[ids, 1], edges[ids, 2], ids]).astype(np.int64)
    assert_same(got, want, f"{what}: CSR rows (source, dst, len, edge id)")


def check_build(G, P, what):
    c = G.counts()
    assert (c["n_nodes"], c["n_edges"], c["n_alive_piles"]) == (P.n_nodes, P.edges.shape[0], int((P.seq_to_node != INF).sum())), what
    assert_same(G.edges(), P.edges, f"{what}: edges")
    assert_same(G.seq_to_node(), P.seq_to_node, f"{what}: seq_to_node")
    check_csr(G, P.n_nodes, P.edges, what)


def check_all(G, P, what):
    check_build(G, P, what)
    assert_same(G.marked(), P.marked, f"{what}: marks")
    assert G.counts()["n_transitive_pairs"] == P.n_pairs, what


def eager_captured_replayed(G, P, what):
    G.use_cuda_graph(False)
    G.run()
    check_all(G, P, f"{what} eager")
    G.use_cuda_graph(True)
    for i in range(3):   # eager (new shape), captured + launched, replayed
        G.run()
        check_all(G, P, f"{what} graph run {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", LENGTHS)
def test_list_length_matches_oracle(ctx, n):
    piles, flags, rec = length_inputs()
    with _closing(api.Graph(ctx)) as G:
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec[:n])
        eager_captured_replayed(G, length_oracle(n), f"{n} entries")


@pytest.mark.gpu
def test_list_lengths_large_to_small_on_one_session(ctx):
    piles, flags, rec = length_inputs()
    with _closing(api.Graph(ctx)) as G:
        G.set_piles(piles, flags).set_hills(None)
        for n in sorted(LENGTHS, reverse=True):
            G.set_overlaps(rec[:n])
            G.use_cuda_graph(False)
            G.run()
            check_all(G, length_oracle(n), f"{n} entries after larger lists")
            G.use_cuda_graph(True)
            G.run()
            G.run()
            check_all(G, length_oracle(n), f"{n} entries after larger lists, captured")


def _kept_session(G, piles, flags, kept):
    G.set_piles(piles, flags).set_hills(None).set_overlaps(invalid(kept.shape[0]))
    G.classify().finalize()
    G.set_kept_overlaps(kept)


@pytest.mark.gpu
@pytest.mark.parametrize("n_tiles", KEPT_TILES)
def test_tile_patterns_match_oracle(ctx, n_tiles):
    piles, flags, kept, _, _ = kept_inputs(n_tiles)
    P = kept_oracle(n_tiles)
    with _closing(api.Graph(ctx)) as G:
        _kept_session(G, piles, flags, kept)
        G.build()
        check_build(G, P, f"{n_tiles} tiles: build")
        G.transitive()
        check_all(G, P, f"{n_tiles} tiles")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TABLES))
def test_pile_table_matches_oracle(ctx, name):
    piles, flags, rec = table_inputs(name)
    with _closing(api.Graph(ctx)) as G:
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec)
        eager_captured_replayed(G, table_oracle(name), name)


@pytest.mark.gpu
def test_final_pass_kills_match_oracle(ctx):
    piles, cut, flags, rec, victims = kill_inputs()
    _, P = kill_oracle_stages()
    with _closing(api.Graph(ctx)) as G:
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec)
        G.classify()
        G.set_piles(cut, flags).retrim()
        while G.retrim_promote():
            pass
        G.finalize().build()
        check_build(G, P, "final-pass kills: build")
        assert (G.seq_to_node()[victims] == INF).all()
        G.transitive()
        check_all(G, P, "final-pass kills")


@pytest.mark.gpu
def test_session_reuse_eager(ctx):
    piles, flags, rec, _, sizes = reuse_inputs()
    with _closing(api.Graph(ctx)) as G:
        G.use_cuda_graph(False)
        G.set_piles(piles, flags).set_hills(None)
        for n in (rec.shape[0], sizes[2], sizes[14], 0, sizes[14]):
            G.set_overlaps(rec[:n]).run()
            check_all(G, reuse_oracle(n), f"{n} records after a larger graph")


@pytest.mark.gpu
def test_session_reuse_replayed(ctx):
    """One record count throughout (the rest flagged invalid): after the large graph, every smaller one replays the
    captured run."""
    piles, flags, rec, big, sizes = reuse_inputs()
    with _closing(api.Graph(ctx)) as G:
        G.use_cuda_graph(True)
        G.set_piles(piles, flags).set_hills(None).set_overlaps(rec)
        for i in range(3):   # eager (fresh piles), eager (new shape), captured + launched
            G.run()
            check_all(G, big, f"large graph run {i}")
        launches = ctx.launch_count
        for n in (sizes[2], sizes[14], 0):
            masked = rec.copy()
            masked[n:, 6] |= 2
            P = O.Pipeline(masked, piles, flags).run()
            assert P.edges.shape[0] == 2 * n
            G.set_overlaps(masked).run()
            check_all(G, P, f"{n} valid records, replayed")
        assert ctx.launch_count > launches


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("inputs", ["shards", "lone_pile"])
def test_multi_edge_phase_matches_oracle(world, inputs):
    piles, flags, rec = multi_inputs() if inputs == "shards" else lone_pile_inputs()
    bounds = SHARDS[world] if inputs == "shards" else None
    if bounds:
        rec = rec[:bounds[-1][1]]
    P = O.Pipeline(rec, piles, flags).run()
    with _closing(api.Multi([0] * world)) as M:
        M.set_barrier_timeout_ms(20000)
        M.set_piles(piles, flags).set_hills(None).set_shards(rec, bounds).plan()
        M.use_cuda_graph(False)
        for i in range(3):
            M.run()
            edges, marked = M.all_edges()
            what = f"{world} ranks, {inputs}, run {i}"
            assert_same(edges, P.edges, f"{what}: edges")
            assert_same(marked, P.marked, f"{what}: marks")
            assert_same(M.seq_to_node(), P.seq_to_node, f"{what}: seq_to_node")
            c = M.counts()
            assert (c["n_nodes"], c["n_edges"], c["n_transitive_pairs"]) == (P.n_nodes, P.edges.shape[0], P.n_pairs), what
            M.use_cuda_graph(True)
