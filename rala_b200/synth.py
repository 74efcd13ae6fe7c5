"""Deterministic synthetic reads + overlaps of the shapes BASELINE.json names.

Used by the tests (to feed the reference front end through FASTA + PAF text) and by
``bench.py`` (to build the binary ``rala_ovl_t`` / ``rala_pile_t`` arrays directly, as
SURVEY.md section 8(d) allows for the large configurations).  Everything is a pure function
of the arguments and ``seed`` (numpy ``PCG64``).

Coordinate conventions follow PAF as the reference consumes it
(/root/reference/src/overlap.cpp:22-31): begin/end of an overlap are given on each
read's own forward strand ("as sequenced"), ``flags bit0`` (orientation) is 1 when the two
reads come from opposite genome strands.

Records are listed grouped by query in ascending query id, which is the grouping
the reference's duplicate filter assumes (/root/reference/src/graph.cpp:343-350).
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass, field

import numpy as np

OVL_WORDS = 7  # a_id b_id a_begin a_end b_begin b_end flags  (include/rala_b200.h: rala_ovl_t)


@dataclass
class Dataset:
    read_len: np.ndarray          # (n_reads,) uint32
    records: np.ndarray           # (n_ovl, 7) uint32, file order
    genome_len: int
    meta: dict = field(default_factory=dict)

    @property
    def n_reads(self) -> int:
        return int(self.read_len.shape[0])

    @property
    def n_overlaps(self) -> int:
        return int(self.records.shape[0])

    def flat_piles(self, margin: int = 15) -> np.ndarray:
        """Pile table the reference front end produces on clean, well-covered data:
        valid region [margin, len - margin) (graph.cpp:317-324 shrinks every overlap by 15 bp
        before it is layered, pile.cpp:329 keeps coverage >= 4).  (n_reads, 2) uint32."""
        p = np.empty((self.n_reads, 2), dtype=np.uint32)
        p[:, 0] = margin
        p[:, 1] = self.read_len - margin
        return p

    def write_fasta(self, path: str, seed: int = 7) -> None:
        rng = np.random.Generator(np.random.PCG64(seed))
        alphabet = np.frombuffer(b"ACGT", dtype=np.uint8)
        with open(path, "wb") as f:
            for i, n in enumerate(self.read_len.tolist()):
                f.write(b">r%d\n" % i)
                f.write(alphabet[rng.integers(0, 4, size=n, dtype=np.uint8)].tobytes())
                f.write(b"\n")

    def write_paf(self, path: str) -> None:
        r = self.records
        ln = self.read_len
        with open(path, "w") as f:
            chunk = 1 << 18
            for s in range(0, r.shape[0], chunk):
                q = r[s:s + chunk]
                a, b = q[:, 0], q[:, 1]
                span = np.maximum(q[:, 3] - q[:, 2], q[:, 5] - q[:, 4])
                lines = [
                    "r%d\t%d\t%d\t%d\t%s\tr%d\t%d\t%d\t%d\t%d\t%d\t255\n" % (
                        a_, la, ab, ae, "-" if fl & 1 else "+", b_, lb, bb, be, sp, sp)
                    for a_, la, ab, ae, fl, b_, lb, bb, be, sp in zip(
                        a.tolist(), ln[a].tolist(), q[:, 2].tolist(), q[:, 3].tolist(), q[:, 6].tolist(),
                        b.tolist(), ln[b].tolist(), q[:, 4].tolist(), q[:, 5].tolist(), span.tolist())
                ]
                f.write("".join(lines))

    def write_mhap(self, path: str) -> None:
        """The same records as MHAP: "a+1 b+1 0.0 <span> 0 ab ae la ori bb be lb" (1-based ids, a_rc = 0, b_rc = orientation;
        the shared-minmers field carries the span, which no reader uses)."""
        r = self.records
        ln = self.read_len
        with open(path, "w") as f:
            chunk = 1 << 18
            for s in range(0, r.shape[0], chunk):
                q = r[s:s + chunk]
                a, b = q[:, 0], q[:, 1]
                span = np.maximum(q[:, 3] - q[:, 2], q[:, 5] - q[:, 4])
                lines = [
                    "%d %d 0.0 %d 0 %d %d %d %d %d %d %d\n" % (a_ + 1, b_ + 1, sp, ab, ae, la, fl & 1, bb, be, lb)
                    for a_, b_, sp, ab, ae, la, fl, bb, be, lb in zip(
                        a.tolist(), b.tolist(), span.tolist(), q[:, 2].tolist(), q[:, 3].tolist(), ln[a].tolist(),
                        q[:, 6].tolist(), q[:, 4].tolist(), q[:, 5].tolist(), ln[b].tolist())
                ]
                f.write("".join(lines))


def _pairs_sorted(g0: np.ndarray, g1: np.ndarray, min_ovl: int):
    """All (i, j), i < j in g0-sorted order, whose genome intervals share >= min_ovl bases."""
    n = g0.shape[0]
    hi = np.searchsorted(g0, g1 - min_ovl, side="right")  # j with g0[j] <= g1[i] - min_ovl
    idx = np.arange(n, dtype=np.int64)
    cnt = np.maximum(hi - idx - 1, 0)
    total = int(cnt.sum())
    if total == 0:
        z = np.zeros(0, dtype=np.int64)
        return z, z
    i = np.repeat(idx, cnt)
    start = np.cumsum(cnt) - cnt
    j = np.arange(total, dtype=np.int64) - np.repeat(start, cnt) + i + 1
    ov = np.minimum(g1[i], g1[j]) - np.maximum(g0[i], g0[j])
    keep = ov >= min_ovl
    return i[keep], j[keep]


def _to_read_coords(x0, x1, g0, g1, off, rc):
    """Genome interval [x0, x1) inside segment [g0, g1) -> coordinates on the read as sequenced."""
    b = np.where(rc, off + (g1 - x1), off + (x0 - g0))
    e = np.where(rc, off + (g1 - x0), off + (x1 - g0))
    return b, e


def generate(genome_len: int, coverage: float, read_len: int = 10000, len_sd: int = 0, min_len: int = 1500,
             seed: int = 1, min_ovl: int = 1000, shuffle: bool = True, dual: bool = False, noise: int = 0,
             chimera_frac: float = 0.0, adapter_frac: float = 0.0, repeats: tuple | None = None,
             n_reads: int | None = None) -> Dataset:
    """Uniform random genome sampling.

    repeats = (n_families, n_copies, repeat_len): every family places ``n_copies`` copies of a
    ``repeat_len`` segment in the genome; reads covering different copies get an extra,
    repeat-induced overlap restricted to the repeat (the way an overlapper would report it).
    """
    rng = np.random.Generator(np.random.PCG64(seed))
    n = int(n_reads if n_reads is not None else genome_len * coverage / read_len)
    if len_sd > 0:
        length = np.clip(np.rint(rng.normal(read_len, len_sd, n)), min_len, genome_len // 4).astype(np.int64)
    else:
        length = np.full(n, read_len, dtype=np.int64)

    # --- segments -----------------------------------------------------------------------------
    is_chim = rng.random(n) < chimera_frac
    adapter = np.where(rng.random(n) < adapter_frac, rng.integers(40, 121, n), 0).astype(np.int64)
    split = np.where(is_chim, (length * rng.uniform(0.3, 0.7, n)).astype(np.int64), length)
    seg_read = np.concatenate([np.arange(n), np.nonzero(is_chim)[0]]).astype(np.int64)
    seg_len = np.concatenate([split, (length - split)[is_chim]])
    seg_off = np.concatenate([adapter, (adapter + split)[is_chim]])
    n_seg = seg_read.shape[0]
    seg_g0 = (rng.random(n_seg) * (genome_len - seg_len)).astype(np.int64)
    seg_g1 = seg_g0 + seg_len
    seg_rc = rng.random(n_seg) < 0.5
    total_len = length + adapter

    # read ids: position order -> shuffled ids (real data has no id/position correlation)
    order = np.argsort(seg_g0[:n], kind="stable")
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    rid = rng.permutation(n)[rank] if shuffle else rank
    read_len_out = np.empty(n, dtype=np.uint32)
    read_len_out[rid] = total_len.astype(np.uint32)

    def emit(sr, g0, g1, off, rc, tag, min_o):
        o = np.argsort(g0, kind="stable")
        sr, g0, g1, off, rc = sr[o], g0[o], g1[o], off[o], rc[o]
        tag_s = tag[o] if tag is not None else None
        i, j = _pairs_sorted(g0, g1, min_o)
        ok = sr[i] != sr[j]
        if tag_s is not None:
            ok &= tag_s[i] != tag_s[j]
        i, j = i[ok], j[ok]
        x0 = np.maximum(g0[i], g0[j])
        x1 = np.minimum(g1[i], g1[j])
        ib, ie = _to_read_coords(x0, x1, g0[i], g1[i], off[i], rc[i])
        jb, je = _to_read_coords(x0, x1, g0[j], g1[j], off[j], rc[j])
        return rid[sr[i]], rid[sr[j]], ib, ie, jb, je, (rc[i] != rc[j])

    parts = [emit(seg_read, seg_g0, seg_g1, seg_off, seg_rc, None, min_ovl)]

    if repeats is not None:
        n_fam, n_copies, rep_len = repeats
        for f in range(n_fam):
            copies = np.sort((rng.random(n_copies) * (genome_len - rep_len)).astype(np.int64))
            a_sr, a_g0, a_g1, a_off, a_rc, a_tag = [], [], [], [], [], []
            for m, c in enumerate(copies.tolist()):
                lo = np.maximum(seg_g0, c)
                hi = np.minimum(seg_g1, c + rep_len)
                hit = np.nonzero(hi - lo >= min_ovl)[0]
                if hit.size == 0:
                    continue
                # the part of the segment inside the copy, re-expressed in the family's own coordinates
                rb, re_ = _to_read_coords(lo[hit], hi[hit], seg_g0[hit], seg_g1[hit], seg_off[hit], seg_rc[hit])
                a_sr.append(seg_read[hit])
                a_g0.append(lo[hit] - c)
                a_g1.append(hi[hit] - c)
                # offset such that _to_read_coords on the alias interval reproduces rb/re_
                a_off.append(rb)
                a_rc.append(seg_rc[hit])
                a_tag.append(np.full(hit.size, m, dtype=np.int64))
            if not a_sr:
                continue
            parts.append(emit(np.concatenate(a_sr), np.concatenate(a_g0), np.concatenate(a_g1),
                              np.concatenate(a_off), np.concatenate(a_rc), np.concatenate(a_tag), min_ovl))

    qa = np.concatenate([p[0] for p in parts])
    qb = np.concatenate([p[1] for p in parts])
    ab = np.concatenate([p[2] for p in parts])
    ae = np.concatenate([p[3] for p in parts])
    bb = np.concatenate([p[4] for p in parts])
    be = np.concatenate([p[5] for p in parts])
    ori = np.concatenate([p[6] for p in parts])

    if noise > 0:
        la, lb = read_len_out[qa].astype(np.int64), read_len_out[qb].astype(np.int64)
        ab = np.clip(ab + rng.integers(-noise, noise + 1, ab.shape[0]), 0, la)
        ae = np.clip(ae + rng.integers(-noise, noise + 1, ab.shape[0]), 0, la)
        bb = np.clip(bb + rng.integers(-noise, noise + 1, ab.shape[0]), 0, lb)
        be = np.clip(be + rng.integers(-noise, noise + 1, ab.shape[0]), 0, lb)
        ok = (ae - ab >= 100) & (be - bb >= 100)
        qa, qb, ab, ae, bb, be, ori = qa[ok], qb[ok], ab[ok], ae[ok], bb[ok], be[ok], ori[ok]

    # list every pair once under the lower read id as query (optionally also the mirrored record)
    swap = qa > qb
    qa2 = np.where(swap, qb, qa)
    qb2 = np.where(swap, qa, qb)
    ab2, ae2 = np.where(swap, bb, ab), np.where(swap, be, ae)
    bb2, be2 = np.where(swap, ab, bb), np.where(swap, ae, be)
    if dual:
        qa2, qb2 = np.concatenate([qa2, qb2]), np.concatenate([qb2, qa2])
        ab2, bb2 = np.concatenate([ab2, bb2]), np.concatenate([bb2, ab2])
        ae2, be2 = np.concatenate([ae2, be2]), np.concatenate([be2, ae2])
        ori = np.concatenate([ori, ori])
    o = np.lexsort((ab2, qb2, qa2))
    rec = np.empty((qa2.shape[0], OVL_WORDS), dtype=np.uint32)
    rec[:, 0] = qa2[o]
    rec[:, 1] = qb2[o]
    rec[:, 2] = ab2[o]
    rec[:, 3] = ae2[o]
    rec[:, 4] = bb2[o]
    rec[:, 5] = be2[o]
    rec[:, 6] = ori[o].astype(np.uint32)
    return Dataset(read_len=read_len_out, records=rec, genome_len=genome_len,
                   meta=dict(seed=seed, coverage=coverage, read_len=read_len, len_sd=len_sd, min_ovl=min_ovl,
                             shuffle=shuffle, dual=dual, noise=noise, chimera_frac=chimera_frac,
                             adapter_frac=adapter_frac, repeats=repeats))


def hub_graph(n_hubs: int = 4, spokes: int = 2500, links_per_spoke: int = 6, seed: int = 5):
    """Config-5 style injected graph at the K3 boundary (SURVEY.md 8(d) item 5 fallback): hub nodes
    with out-degree ``spokes`` whose spokes are chained so that hub->spoke edges have two-hop witnesses.
    Returns (n_nodes, edges (E,3) uint32 [src dst len]) with pair(e) = e ^ 1 and pair(node) = node ^ 1."""
    rng = np.random.Generator(np.random.PCG64(seed))
    reads_per_hub = spokes + 1
    n_reads = n_hubs * reads_per_hub
    edges = []

    def add(a, b, ln_ab, ln_ba):
        edges.append((a, b, ln_ab))
        edges.append((b ^ 1, a ^ 1, ln_ba))

    for h in range(n_hubs):
        base = 2 * h * reads_per_hub
        hub = base
        # spoke k starts 100 + 3k bases after the hub's start (so hub->spoke length = 100 + 3k)
        pos = 100 + 3 * np.arange(spokes)
        for k in range(spokes):
            s = base + 2 * (k + 1)
            add(hub, s, int(pos[k]), int(pos[k]) + 50)
            for d in rng.choice(np.arange(1, 40), size=links_per_spoke, replace=False).tolist():
                if k + d < spokes:
                    t = base + 2 * (k + d + 1)
                    jitter = int(rng.integers(-4, 5))
                    add(s, t, max(1, int(pos[k + d] - pos[k]) + jitter), int(pos[k + d] - pos[k]) + 7)
    e = np.asarray(edges, dtype=np.uint32)
    return 2 * n_reads, e


def generate_repeat_hubs(genome_len: int = 20_000_000, coverage: float = 30, read_len: int = 10000, n_hubs: int = 8,
                         spokes: int = 2601, chain: int = 3, internals_per_spoke: int = 3, seed: int = 5) -> Dataset:
    """BASELINE.json configs[4]: a genome with segmental repeats that give node degrees > 2 000 THROUGH the whole hot path
    (classification, containment, edges, transitive reduction), not only at the graph boundary (SURVEY.md 8(d) item 5).

    On top of a uniform ``generate()`` background, every hub read ends in a 3 kbp repeat unit that ``spokes`` other reads
    (from as many other copies of the repeat) begin with.  Geometry, in read coordinates:
      hub - spoke      hub[L - o, L) ~ spoke[0, o), 1000 <= o <= 2900: begin offsets differ by L - o >= 7100 > 5 % of L, so the
                       type is a dovetail (overlap.cpp:236-258), never a near-containment, and the hub keeps every spoke;
      spoke chains     the spokes of one repeat copy are `chain` reads tiled 600 - 900 bp apart (again > 5 % of L), all
                       pairwise overlaps listed: hub -> 2nd / 3rd spoke and 1st -> 3rd spoke are transitive
                       (graph.cpp:1301-1306), hub -> 1st is not;
      spoke - spoke    a few overlaps per spoke between DIFFERENT copies, confined to the repeat: they diverge behind it,
                       so they type as internal (kX, overlap.cpp:221-224), the way an overlapper reports repeats.
    The new reads overlap nothing else, so none of them is contained: the hub's out-degree is exactly `spokes`."""
    base = generate(genome_len, coverage, read_len, seed=seed)
    rng = np.random.Generator(np.random.PCG64(seed + 1000))
    L = read_len
    n0 = base.n_reads
    loci = (spokes + chain - 1) // chain
    rows = []
    next_id = n0
    for _h in range(n_hubs):
        hub = next_id
        next_id += 1
        fam = []   # (read id, repeat bases at its start)
        for _l in range(loci):
            o = 2900 - int(rng.integers(0, 200))
            ids, offs = [], []
            for k in range(chain):
                if len(fam) + len(ids) >= spokes or o < 1000:
                    break
                ids.append(next_id)
                offs.append(o)
                next_id += 1
                o -= int(rng.integers(600, 901))
            # hub - spoke, listed under the lower id (the hub was created first)
            for r, ov in zip(ids, offs):
                rows.append((hub, r, L - ov, L, 0, ov, 0))
            # the chain's own tiling overlaps: read j starts offs[i] - offs[j] bases after read i
            for i in range(len(ids)):
                for j in range(i + 1, len(ids)):
                    d = offs[i] - offs[j]
                    rows.append((ids[i], ids[j], d, L, 0, L - d, 0))
            fam += list(zip(ids, offs))
        # repeat-induced overlaps between different copies: the common part of the two repeat prefixes
        fam_ids = np.array([f[0] for f in fam])
        fam_o = np.array([f[1] for f in fam])
        for k in range(len(fam)):
            for p in rng.choice(len(fam), size=internals_per_spoke, replace=False).tolist():
                if abs(int(fam_ids[p]) - int(fam_ids[k])) < chain:   # same copy (or itself): already listed above
                    continue
                a, b = (k, p) if fam_ids[k] < fam_ids[p] else (p, k)
                m = int(min(fam_o[a], fam_o[b]))
                rows.append((int(fam_ids[a]), int(fam_ids[b]), int(fam_o[a]) - m, int(fam_o[a]), int(fam_o[b]) - m, int(fam_o[b]), 0))
    extra = np.unique(np.asarray(rows, dtype=np.uint32), axis=0)
    rec = np.concatenate([base.records, extra])
    rec = rec[np.lexsort((rec[:, 2], rec[:, 1], rec[:, 0]))]
    read_len_out = np.concatenate([base.read_len, np.full(next_id - n0, L, dtype=np.uint32)])
    return Dataset(read_len=read_len_out, records=np.ascontiguousarray(rec), genome_len=genome_len,
                   meta=dict(base.meta, n_hubs=n_hubs, spokes=spokes, chain=chain, first_hub=n0))


# ---------------------------------------------------------------------------------------------
# Input of the front end's duplicate filter (Graph::initialize, graph.cpp:273-303): query groups in which the same
# target shows up several times (repeats), with ties in the alignment length, self overlaps, records whose names are
# not in the read set (they are skipped INSIDE a group) and queries that come back in a later group.
# ---------------------------------------------------------------------------------------------
@dataclass
class DuplicateGroups:
    read_len: np.ndarray      # (n_reads,) uint32
    a: np.ndarray             # (n,) int64, -1 = name not in the read set
    b: np.ndarray             # (n,) int64, -1 likewise
    coords: np.ndarray        # (n, 4) uint32: a_begin a_end b_begin b_end
    ori: np.ndarray           # (n,) uint8
    length: np.ndarray        # (n,) uint32: PAF column 11, what Overlap::length() returns before any trimming

    @property
    def n(self) -> int:
        return int(self.a.shape[0])

    def columns(self):
        """(a_id with RALA_INVALID_BIT for unknown records, b_id, length) as the device filter takes them."""
        known = (self.a >= 0) & (self.b >= 0)
        a = np.where(known, self.a, 0x80000000).astype(np.uint32)
        b = np.where(known, self.b, 0).astype(np.uint32)
        return a, b, self.length.astype(np.uint32)

    def write_fasta(self, path: str, seed: int = 7) -> None:
        Dataset(self.read_len, np.zeros((0, 7), np.uint32), 0).write_fasta(path, seed)

    def write_paf(self, path: str) -> None:
        ln = self.read_len
        with open(path, "w") as f:
            for i in range(self.n):
                a, b = int(self.a[i]), int(self.b[i])
                an, la = ("r%d" % a, int(ln[a])) if a >= 0 else ("ghost%d" % i, 9000)
                bn, lb = ("r%d" % b, int(ln[b])) if b >= 0 else ("ghost%d" % i, 9000)
                c = self.coords[i]
                f.write("%s\t%d\t%d\t%d\t%s\t%s\t%d\t%d\t%d\t%d\t%d\t255\n" % (
                    an, la, c[0], c[1], "-" if self.ori[i] else "+", bn, lb, c[2], c[3], int(self.length[i]) // 2, int(self.length[i])))


def generate_duplicate_groups(n_reads: int = 300, n_groups: int = 500, max_group: int = 40, pool: int = 6, big_groups: int = 0,
                              big_size: int = 3000, ghost_frac: float = 0.03, self_frac: float = 0.03, seed: int = 11) -> DuplicateGroups:
    rng = np.random.Generator(np.random.PCG64(seed))
    read_len = rng.integers(4000, 12000, n_reads).astype(np.uint32)
    A, B, C, O, L = [], [], [], [], []
    sizes = rng.integers(1, max_group + 1, n_groups).tolist()
    for k in rng.choice(n_groups, size=min(big_groups, n_groups), replace=False).tolist():
        sizes[k] = big_size
    prev_a = -1
    for g in sizes:
        a = int(rng.integers(0, n_reads))
        while a == prev_a:           # two groups in a row with the same query would be ONE group for the reference
            a = int(rng.integers(0, n_reads))
        prev_a = a
        targets = rng.choice(n_reads, size=min(pool, n_reads), replace=False)
        base = int(rng.integers(300, 3000))
        for _ in range(g):
            b = int(targets[rng.integers(0, len(targets))])
            if rng.random() < self_frac:
                b = a
            ghost = rng.random() < ghost_frac
            la, lb = int(read_len[a]), int(read_len[b])
            span = int(rng.integers(200, min(la, lb) - 100))
            ab = int(rng.integers(0, la - span)); bb = int(rng.integers(0, lb - span))
            A.append(-1 if ghost and rng.random() < 0.5 else a)
            B.append(-1 if ghost and A[-1] >= 0 else b)
            C.append((ab, ab + span, bb, bb + span))
            O.append(int(rng.integers(0, 2)))
            L.append(base + int(rng.integers(0, 4)))   # few distinct lengths: ties are common
    return DuplicateGroups(read_len, np.asarray(A, np.int64), np.asarray(B, np.int64), np.asarray(C, np.uint32),
                           np.asarray(O, np.uint8), np.asarray(L, np.uint32))


BGZF_BLOCK = 65280   # input bytes per block, as htslib's bgzip cuts them (the compressed block then fits the 16-bit BSIZE)
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_block(data: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY) -> bytes:
    """One BGZF member: raw DEFLATE of `data` (<= 65536 bytes) with the BC subfield, CRC32 and ISIZE."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    z = c.compress(data) + c.flush()
    if len(z) + 26 > 65536:
        raise ValueError(f"a block of {len(data)} bytes compresses to {len(z)}: BSIZE would not fit 16 bits")
    head = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(z) + 25)
    return head + z + struct.pack("<II", zlib.crc32(data), len(data))


def write_bgzf(text, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, cuts=None) -> bytes:
    """`text` as BGZF (what `bgzip` writes): blocks of at most BGZF_BLOCK input bytes, or cut at the offsets `cuts`
    (ascending, each block <= 65536 bytes), raw DEFLATE from zlib.compressobj(level, DEFLATED, -15, 8, strategy), the
    28-byte end-of-file marker at the end.  Blocks are independent, so a caller may compress them in a process pool."""
    text = bytes(text)
    bounds = list(range(0, len(text), BGZF_BLOCK)) if cuts is None else [0] + [int(c) for c in cuts]
    bounds.append(len(text))
    out = [bgzf_block(text[a:b], level, strategy) for a, b in zip(bounds[:-1], bounds[1:]) if b > a or cuts is not None]
    return b"".join(out) + BGZF_EOF


def gzip_deflate(text, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, dictionary: bytes = b"", final: bool = True) -> bytes:
    """Raw DEFLATE of `text`, primed with `dictionary` (at most the last 32 KiB count); not final: ends with Z_SYNC_FLUSH
    (an empty stored block, byte-aligned), so that the next piece's stream can follow it, as pigz joins its pieces."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy, **({"zdict": dictionary[-32768:]} if dictionary else {}))
    return c.compress(bytes(text)) + c.flush(zlib.Z_FINISH if final else zlib.Z_SYNC_FLUSH)


def write_gzip(text, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, members=1, sync_every=None, fname=None,
               comment=None, extra=None, hcrc: bool = False, pool=None) -> bytes:
    """`text` as plain gzip: `members` members (a count of equal parts, or a list of cut offsets), each one raw DEFLATE
    stream, or with sync_every=N pigz-style pieces of N bytes, each compressed with the 32 KiB before it as dictionary and
    joined by Z_SYNC_FLUSH (pool: an executor with .map to compress the pieces in parallel).  fname / comment (bytes
    without NUL), extra (the FEXTRA payload) and hcrc (FHCRC) go into every member header."""
    text = bytes(text)
    if isinstance(members, int):
        step = -(-len(text) // max(members, 1)) if text else 0
        cuts = [min(i * step, len(text)) for i in range(1, max(members, 1))]
    else:
        cuts = [int(c) for c in members]
    bounds = [0] + cuts + [len(text)]
    flg = (4 if extra is not None else 0) | (8 if fname is not None else 0) | (16 if comment is not None else 0) | (2 if hcrc else 0)
    head = b"\x1f\x8b\x08" + bytes([flg]) + b"\x00\x00\x00\x00\x00\xff"
    if extra is not None:
        head += struct.pack("<H", len(extra)) + bytes(extra)
    if fname is not None:
        head += bytes(fname) + b"\x00"
    if comment is not None:
        head += bytes(comment) + b"\x00"
    if hcrc:
        head += struct.pack("<H", zlib.crc32(head) & 0xFFFF)
    out = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        part = text[a:b]
        if sync_every:
            starts = list(range(0, len(part), sync_every)) or [0]
            args = [(part[s:s + sync_every], level, strategy, part[max(0, s - 32768):s], s + sync_every >= len(part)) for s in starts]
            pieces = list((pool.map if pool else map)(_gzip_piece, args))
            body = b"".join(pieces)
        else:
            body = gzip_deflate(part, level, strategy)
        out.append(head + body + struct.pack("<II", zlib.crc32(part), len(part) & 0xFFFFFFFF))
    return b"".join(out)


def _gzip_piece(a):
    return gzip_deflate(*a)
