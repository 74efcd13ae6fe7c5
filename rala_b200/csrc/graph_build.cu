// graph_build.cu — K2: node ids, edge list with reverse-complement twins, CSR adjacency.
//
// Replaces graph.cpp:552-632 (reference): sequence_id_to_node_id (:553-574), the two Edge objects per
// dovetail overlap with their lengths (:576-632) and the implicit adjacency (suffix_edges_ vectors).
#include <cstdlib>

#include "kernels.h"
#include "lists.cuh"

namespace rb {

// The build runs over the final `overlaps` in three kernels, without a fill pass over the finished edges:
//   k_count_edges  every dovetail (tag kAB / kBA, both piles alive) adds one to the degree of its two source SLOTS, and
//                  every tile of the list records how many dovetails it holds
//   k_scan_piles   one look-back over the piles: node ids, the rows of the alive piles' slots, and the edge-id base of
//                  every list tile
//   k_emit_edges   the edge pair of every dovetail, in list order, straight into its CSR rows
// A slot 2x + s is the node 2 rank(x) + s of pile x (rank among the alive piles, graph.cpp:553-561): node ids are monotone
// in pile order, so the slots of the alive piles are the nodes in order, and a dead pile's slots count nothing.
// The tags are the final containment pass's types (k_classify_final), taken against the pile table before that pass's
// deaths: an entry whose pile the pass killed still carries kAB / kBA, so liveness is checked here.  Alive piles keep
// their coordinates through the deaths, so the tag of an entry with two alive piles is its type on the final table.
constexpr int kEmitTile = kTileThreads * kEmitItems;   // list entries per tile: item r of thread t is entry r * 256 + t
constexpr int kEmitMinBlocks = 5;                      // k_emit_edges: resident blocks per SM (48 registers, no spills)

__device__ __forceinline__ bool is_dovetail(uint8_t tag) { return tag == kAB || tag == kBA; }

// source slots of the two edges of a dovetail (node ids of graph.cpp:578-580 / 594-629 by pile): kAB 2a -> 2b + ori,
// its twin 2b + !ori -> 2a + 1; kBA 2b + ori -> 2a, its twin 2a + 1 -> 2b + !ori
__global__ void __launch_bounds__(kTileThreads) k_count_edges(List ovl, const uint32_t* __restrict__ n_ptr, uint32_t cap,
                                                             const uint2* __restrict__ piles, uint32_t* __restrict__ slot_degree,
                                                             uint32_t* __restrict__ tile_dov) {
    __shared__ uint32_t s_cnt;
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*n_ptr, cap);
    const uint32_t num_tiles = (n + kEmitTile - 1) / kEmitTile;
    const uint32_t* pile_y = reinterpret_cast<const uint32_t*>(piles) + 1;   // end | flags << 30 (end == 0: dead)
    for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        if (tid == 0) s_cnt = 0;
        uint32_t a[kEmitItems], b[kEmitItems];
        uint8_t tag[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            const uint32_t idx = tile * kEmitTile + r * kTileThreads + tid;
            tag[r] = kRejected;
            if (idx < n) {
                a[r] = ovl.a[idx];
                b[r] = ovl.b[idx];
                tag[r] = ovl.tag[idx];
            }
        }
        uint32_t ya[kEmitItems], yb[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            ya[r] = yb[r] = 0u;
            if (is_dovetail(tag[r])) {
                ya[r] = __ldg(pile_y + 2 * (size_t) a[r]);
                yb[r] = __ldg(pile_y + 2 * (size_t) (b[r] & 0x7FFFFFFFu));
            }
        }
        uint32_t c = 0;
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            if ((ya[r] & kEndMask) && (yb[r] & kEndMask)) {
                ++c;
                if (slot_degree) {
                    const uint32_t ori = b[r] >> 31, bb = b[r] & 0x7FFFFFFFu;
                    const bool ab = tag[r] == kAB;
                    atomicAdd(&slot_degree[ab ? 2 * a[r] : 2 * bb + ori], 1u);
                    atomicAdd(&slot_degree[ab ? 2 * bb + (ori ^ 1u) : 2 * a[r] + 1], 1u);
                }
            }
        }
        c = __reduce_add_sync(0xFFFFFFFFu, c);
        __syncthreads();
        if (lane_id() == 0 && c) atomicAdd(&s_cnt, c);
        __syncthreads();
        if (tid == 0) tile_dov[tile] = s_cnt;
    }
}

// One decoupled look-back over the piles with two counts per tile (alive piles | edges of their slots).  Writes
// seq_to_node (2 rank, kInf when dead), C_ALIVE / C_NODES, and with the CSR outputs on (cursor != nullptr) the row offsets of
// nodes 2r / 2r+1 from the degrees of slots 2x / 2x+1, the same values into the fill cursor, and row_ptr[n_nodes] = E.
// Each thread owns 4 consecutive piles (16-byte loads and stores).  Before it takes a tile, block 0 turns the per-tile
// dovetail counts of the list into exclusive bases in place (C_DOVETAILS, C_EDGES, C_OVERFLOW), and clears the bytes of T
// between E and E rounded up to 16, which k_emit_edges does not write and k_finalize_marks reads.
__global__ void __launch_bounds__(kTileThreads) k_scan_piles(const uint2* __restrict__ piles, uint32_t n_piles,
                                                            const uint32_t* __restrict__ slot_degree, uint32_t* __restrict__ seq_to_node,
                                                            uint32_t* __restrict__ row_ptr, uint32_t* __restrict__ cursor,
                                                            uint32_t* __restrict__ tile_dov, const uint32_t* __restrict__ n_ptr,
                                                            uint32_t cap, uint32_t edge_cap, uint8_t* __restrict__ T,
                                                            uint32_t* __restrict__ counters, unsigned long long* __restrict__ status,
                                                            uint32_t* __restrict__ ticket) {
    __shared__ uint32_t s_a[kTileWarps], s_e[kTileWarps];
    __shared__ uint32_t s_tile, s_base_a, s_base_e;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    if (blockIdx.x == 0) {
        const uint32_t n_tiles = (min(*n_ptr, cap) + kEmitTile - 1) / kEmitTile;
        uint32_t carry = 0;
        for (uint32_t t0 = 0; t0 < n_tiles; t0 += kTile) {
            const uint32_t i0 = t0 + tid * 4;
            uint32_t v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = i0 + k < n_tiles ? tile_dov[i0 + k] : 0u;
            const uint32_t tsum = v[0] + v[1] + v[2] + v[3];
            const uint32_t inc = warp_inclusive_scan(tsum);
            if (lane == 31) s_a[warp] = inc;
            __syncthreads();
            if (warp == 0) {
                const uint32_t w = lane < kTileWarps ? s_a[lane] : 0u, winc = warp_inclusive_scan(w);
                if (lane < kTileWarps) s_e[lane] = winc - w;
                if (lane == kTileWarps - 1) s_base_a = winc;
            }
            __syncthreads();
            uint32_t run = carry + s_e[warp] + inc - tsum;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (i0 + k < n_tiles) tile_dov[i0 + k] = run;
                run += v[k];
            }
            carry += s_base_a;
            __syncthreads();
        }
        const uint32_t edges = 2u * carry;
        if (tid == 0) {
            counters[C_DOVETAILS] = carry;
            counters[C_EDGES] = edges;
            if (2ull * carry > edge_cap) counters[C_OVERFLOW] = 1u;
            if (cursor && n_piles == 0) row_ptr[0] = 0u;
        }
        if (cursor && edges <= edge_cap && tid < 16 && edges + tid < ((edges + 15u) & ~15u)) T[edges + tid] = 0;
    }
    const uint32_t num_tiles = (n_piles + kTile - 1) / kTile;
    while (true) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= num_tiles) break;
        const uint32_t i0 = tile * kTile + tid * 4;
        uint32_t y[4] = {0u, 0u, 0u, 0u}, d[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        if (i0 + 3 < n_piles) {
            const uint4 p01 = *reinterpret_cast<const uint4*>(piles + i0), p23 = *reinterpret_cast<const uint4*>(piles + i0 + 2);
            y[0] = p01.y; y[1] = p01.w; y[2] = p23.y; y[3] = p23.w;
            if (cursor) {
                const uint4 d0 = *reinterpret_cast<const uint4*>(slot_degree + 2 * i0);
                const uint4 d1 = *reinterpret_cast<const uint4*>(slot_degree + 2 * i0 + 4);
                d[0] = d0.x; d[1] = d0.y; d[2] = d0.z; d[3] = d0.w; d[4] = d1.x; d[5] = d1.y; d[6] = d1.z; d[7] = d1.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (i0 + k < n_piles) {
                    y[k] = piles[i0 + k].y;
                    if (cursor) { d[2 * k] = slot_degree[2 * (i0 + k)]; d[2 * k + 1] = slot_degree[2 * (i0 + k) + 1]; }
                }
        }
        uint32_t ca = 0, ce = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ca += (y[k] & kEndMask) ? 1u : 0u;
            ce += d[2 * k] + d[2 * k + 1];   // a dead pile's slots have no edges
        }
        const uint32_t inc_a = warp_inclusive_scan(ca), inc_e = warp_inclusive_scan(ce);
        if (lane == 31) {
            s_a[warp] = inc_a;
            s_e[warp] = inc_e;
        }
        __syncthreads();
        if (warp == 0) {
            const uint32_t wa = lane < kTileWarps ? s_a[lane] : 0u, we = lane < kTileWarps ? s_e[lane] : 0u;
            const uint32_t ia = warp_inclusive_scan(wa), ie = warp_inclusive_scan(we);
            const uint32_t ta = __shfl_sync(0xFFFFFFFFu, ia, kTileWarps - 1), te = __shfl_sync(0xFFFFFFFFu, ie, kTileWarps - 1);
            const unsigned long long agg = pack_counts(ta, te);
            const unsigned long long excl = lookback_exclusive(status, tile, agg);
            if (lane < kTileWarps) {
                s_a[lane] = ia - wa;
                s_e[lane] = ie - we;
            }
            if (lane == 0) {
                s_base_a = count_a(excl);
                s_base_e = count_b(excl);
                if (tile == num_tiles - 1) {
                    const uint32_t alive = count_a(excl + agg);
                    counters[C_ALIVE] = alive;
                    counters[C_NODES] = 2u * alive;
                    if (cursor) row_ptr[2u * alive] = count_b(excl + agg);
                }
            }
        }
        __syncthreads();
        uint32_t node = 2u * (s_base_a + s_a[warp] + inc_a - ca), row = s_base_e + s_e[warp] + inc_e - ce;
        uint32_t ids[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ids[k] = kInf;
            if (y[k] & kEndMask) {
                ids[k] = node;
                if (cursor) {
                    const uint2 rows = make_uint2(row, row + d[2 * k]);
                    *reinterpret_cast<uint2*>(row_ptr + node) = rows;
                    *reinterpret_cast<uint2*>(cursor + node) = rows;
                }
                node += 2u;
                row += d[2 * k] + d[2 * k + 1];
            }
        }
        if (i0 + 3 < n_piles) *reinterpret_cast<uint4*>(seq_to_node + i0) = make_uint4(ids[0], ids[1], ids[2], ids[3]);
        else
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (i0 + k < n_piles) seq_to_node[i0 + k] = ids[k];
        __syncthreads();
    }
}

// Two edges per dovetail overlap, ids 2j / 2j+1 in list order (graph.cpp:576-632): j = the tile's base from k_scan_piles
// + the dovetail's rank inside its tile.  With the CSR outputs on (cursor != nullptr) each edge also takes a slot of its
// source row (slot order inside a row is arbitrary: the transitive pass orders a row by (dst, edge id)) and clears its
// byte of T for the transitive pass.
__global__ void __launch_bounds__(kTileThreads, kEmitMinBlocks) k_emit_edges(
    List ovl, const uint32_t* __restrict__ n_ptr, uint32_t cap, const uint2* __restrict__ piles,
    const uint32_t* __restrict__ seq_to_node, const uint32_t* __restrict__ tile_base, uint32_t* __restrict__ src,
    uint32_t* __restrict__ dst, uint32_t* __restrict__ len, uint32_t edge_cap, uint32_t* __restrict__ cursor,
    uint2* __restrict__ col, uint32_t* __restrict__ col_eid, uint8_t* __restrict__ T) {
    __shared__ uint32_t s_cnt[kEmitItems * kTileWarps];
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t n = min(*n_ptr, cap);
    const uint32_t num_tiles = (n + kEmitTile - 1) / kEmitTile;
    for (uint32_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        // every gather is issued before the first one is used: the entry (7 columns), then both piles and both node ids
        Entry e[kEmitItems];
        uint8_t tag[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            const uint32_t idx = tile * kEmitTile + r * kTileThreads + tid;
            tag[r] = kRejected;
            if (idx < n) {
                e[r] = load_entry(ovl, idx);
                tag[r] = ovl.tag[idx];
            }
        }
        uint2 pa[kEmitItems], pb[kEmitItems];
        uint32_t na[kEmitItems], nb[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            na[r] = nb[r] = kInf;
            pa[r] = pb[r] = make_uint2(0u, 0u);
            if (is_dovetail(tag[r])) {
                pa[r] = __ldg(piles + e[r].a);
                pb[r] = __ldg(piles + e[r].b);
                na[r] = __ldg(seq_to_node + e[r].a);
                nb[r] = __ldg(seq_to_node + e[r].b);
            }
        }
        bool dov[kEmitItems];
        uint32_t e_len[kEmitItems], c_len[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            dov[r] = na[r] != kInf && nb[r] != kInf;   // a dovetail with both piles alive
            Pile A, B;
            A.begin = pa[r].x; A.end = pa[r].y & kEndMask;
            B.begin = pb[r].x; B.end = pb[r].y & kEndMask;
            const Rel q = relative(e[r].c, e[r].ori, A, B);
            e_len[r] = q.a0 - q.b0;                     // kAB, :594-610 (kBA, :612-629, negates both)
            c_len[r] = (q.bl - q.b1) - (q.al - q.a1);
        }
        uint32_t lane_rank[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, dov[r]);
            lane_rank[r] = __popc(m & ((1u << lane) - 1u));
            if (lane == 0) s_cnt[r * kTileWarps + warp] = __popc(m);
        }
        __syncthreads();
        if (warp == 0) {
            const uint32_t c = lane < kEmitItems * kTileWarps ? s_cnt[lane] : 0u;
            const uint32_t inc = warp_inclusive_scan(c);
            if (lane < kEmitItems * kTileWarps) s_cnt[lane] = inc - c;
        }
        __syncthreads();
        const uint32_t base = tile_base[tile];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            const uint32_t j = base + s_cnt[r * kTileWarps + warp] + lane_rank[r];
            if (dov[r] && 2ull * j + 1 < edge_cap) {
                uint32_t from = na[r], to = nb[r] + e[r].ori, l = e_len[r], cl = c_len[r];
                if (tag[r] == kBA) {
                    const uint32_t t = from; from = to; to = t;
                    l = 0u - l; cl = 0u - cl;
                }
                // edge 2j = (from -> to), edge 2j+1 = (to^1 -> from^1): one 8-byte store per column
                reinterpret_cast<uint2*>(src)[j] = make_uint2(from, to ^ 1u);
                reinterpret_cast<uint2*>(dst)[j] = make_uint2(to, from ^ 1u);
                reinterpret_cast<uint2*>(len)[j] = make_uint2(l, cl);
                if (cursor) {
                    const uint32_t p0 = atomicAdd(&cursor[from], 1u), p1 = atomicAdd(&cursor[to ^ 1u], 1u);
                    if (p0 < edge_cap) { col[p0] = make_uint2(to, l); col_eid[p0] = 2u * j; }
                    if (p1 < edge_cap) { col[p1] = make_uint2(from ^ 1u, cl); col_eid[p1] = 2u * j + 1u; }
                    reinterpret_cast<uint16_t*>(T)[j] = 0;
                }
            }
        }
        __syncthreads();
    }
}

__global__ void k_degree_hist(const uint32_t* __restrict__ src, const uint32_t* __restrict__ n_edges_ptr, uint32_t edge_cap,
                              uint32_t* __restrict__ degree) {
    const uint32_t n = min(*n_edges_ptr, edge_cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        atomicAdd(&degree[src[i]], 1u);
    }
}

// Exclusive scan of the degree histogram into row_ptr (and a copy into the fill cursor), single pass.
// Each thread owns 4 consecutive values (one 16-byte load).
__global__ void __launch_bounds__(kTileThreads) k_scan_degrees(uint32_t* __restrict__ cursor, uint32_t* __restrict__ row_ptr,
                                                              uint32_t n, unsigned long long* __restrict__ status,
                                                              uint32_t* __restrict__ ticket, const uint32_t* __restrict__ skip,
                                                              const uint32_t* __restrict__ run_if, const uint32_t* __restrict__ live) {
    if ((skip && *skip) || (run_if && *run_if == 0u)) return;
    if (live) n = min(n, *live + 1u);   // values behind the live count are zero and nobody reads their prefix
    __shared__ uint32_t s_warp[kTileWarps];
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_base;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t num_tiles = (n + kTile - 1) / kTile;
    while (true) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= num_tiles) break;
        const uint32_t i0 = tile * kTile + tid * 4;
        uint32_t v[4] = {0u, 0u, 0u, 0u};
        if (i0 + 3 < n) {
            uint4 q = *reinterpret_cast<const uint4*>(cursor + i0);
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (i0 + k < n) v[k] = cursor[i0 + k];
        }
        const uint32_t tsum = v[0] + v[1] + v[2] + v[3];
        const uint32_t inc = warp_inclusive_scan(tsum);
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = lane < kTileWarps ? s_warp[lane] : 0u;
            uint32_t winc = warp_inclusive_scan(w);
            uint32_t total = __shfl_sync(0xFFFFFFFFu, winc, kTileWarps - 1);
            unsigned long long excl = lookback_exclusive(status, tile, (unsigned long long) total);
            if (lane < kTileWarps) s_warp[lane] = winc - w;
            if (lane == 0) s_base = excl;
        }
        __syncthreads();
        uint32_t run = (uint32_t) s_base + s_warp[warp] + inc - tsum;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (i0 + k < n) {
                row_ptr[i0 + k] = run;
                cursor[i0 + k] = run;
            }
            run += v[k];
        }
        __syncthreads();
    }
}

// Scatter every edge of a list that did not come from k_emit_edges (edges received from other ranks, the stateless
// transitive stage) into its source row.  Slot order inside a row is arbitrary (atomic cursor); nothing downstream depends
// on it: the transitive pass resolves parallel edges by edge id.
// Also clears the per-edge "transitive test passed" bytes T[0 .. n rounded up to 16) for the pass that follows
// (k_finalize_marks reads whole 16-byte groups): a memset of the buffer's CAPACITY (2 x the record count) would
// write ~15 x more bytes than there are edges.
// eight edges in flight per thread, or twice the blocks, changed nothing (profiles/r02ab_ab.json)
constexpr int kFillInflight = 4;
constexpr int kFillBlocks = 8;   // per SM
__global__ void k_fill_csr(const uint32_t* __restrict__ src, const uint32_t* __restrict__ dst,
                           const uint32_t* __restrict__ len, const uint32_t* __restrict__ n_edges_ptr, uint32_t edge_cap,
                           uint32_t* __restrict__ cursor, uint2* __restrict__ col, uint32_t* __restrict__ col_eid,
                           uint8_t* __restrict__ T) {
    const uint32_t n = min(*n_edges_ptr, edge_cap);
    {
        const uint32_t n16 = (n + 15u) / 16u;   // T is padded to a multiple of 256 bytes
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x)
            reinterpret_cast<uint4*>(T)[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    // load -> returning atomic -> store is a chain of three dependent round trips: keep four edges of it in flight
    const uint32_t stride = gridDim.x * blockDim.x;
    constexpr int F = kFillInflight;
    for (uint32_t e0 = blockIdx.x * blockDim.x + threadIdx.x; e0 < n; e0 += F * stride) {
        uint32_t s[F], d[F], l[F], p[F];
#pragma unroll
        for (int k = 0; k < F; ++k) {
            const uint32_t e = e0 + k * stride;
            if (e < n) { s[k] = src[e]; d[k] = dst[e]; l[k] = len[e]; }
        }
#pragma unroll
        for (int k = 0; k < F; ++k)
            if (e0 + k * stride < n) p[k] = atomicAdd(&cursor[s[k]], 1u);
#pragma unroll
        for (int k = 0; k < F; ++k) {
            const uint32_t e = e0 + k * stride;
            if (e < n) {
                col[p[k]] = make_uint2(d[k], l[k]);
                col_eid[p[k]] = e;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Adjacency VIEW for the host (rala_b200_graph_get_adjacency): per node the ids of its out- (key = src) or in-edges
// (key = dst) in ASCENDING EDGE ID, marked edges left out on request: what suffix_edges_ / prefix_edges_ hold after
// Graph::remove_marked_objects (graph.cpp:2118-2151, shrinkToFit :31-54).  Off the hot step (a download path): counting
// sort by node with atomic slots, then every row is ordered by a rank sort (edge ids are distinct).
// ---------------------------------------------------------------------------------------------
__global__ void k_adj_hist(const uint32_t* __restrict__ key, const uint8_t* __restrict__ marked, const uint32_t* __restrict__ n_edges_ptr,
                           uint32_t edge_cap, uint32_t n_nodes, uint32_t* __restrict__ degree) {
    const uint32_t n = min(*n_edges_ptr, edge_cap);
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x)
        if (!(marked && marked[e]) && key[e] < n_nodes) atomicAdd(&degree[key[e]], 1u);
}

__global__ void k_adj_fill(const uint32_t* __restrict__ key, const uint8_t* __restrict__ marked, const uint32_t* __restrict__ n_edges_ptr,
                           uint32_t edge_cap, uint32_t n_nodes, uint32_t* __restrict__ cursor, uint32_t* __restrict__ ids) {
    const uint32_t n = min(*n_edges_ptr, edge_cap);
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x)
        if (!(marked && marked[e]) && key[e] < n_nodes) ids[atomicAdd(&cursor[key[e]], 1u)] = e;
}

// one warp per row: out[row start + #(ids of the row below mine)] = mine
__global__ void __launch_bounds__(256) k_adj_sort_rows(const uint32_t* __restrict__ row_ptr, uint32_t n_nodes, const uint32_t* __restrict__ ids,
                                                      uint32_t* __restrict__ sorted) {
    const uint32_t lane = lane_id(), warps = gridDim.x * (blockDim.x / 32);
    for (uint32_t row = blockIdx.x * (blockDim.x / 32) + warp_id(); row < n_nodes; row += warps) {
        const uint32_t r0 = row_ptr[row], d = row_ptr[row + 1] - r0;
        for (uint32_t i = lane; i < d; i += 32) {
            const uint32_t mine = ids[r0 + i];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < d; ++j) rank += ids[r0 + j] < mine ? 1u : 0u;
            sorted[r0 + rank] = mine;
        }
    }
}

// edge columns -> rala_edge_t rows (download path).  Rows are staged in shared memory and leave as 16-byte stores
// of consecutive threads: `out` may be pinned HOST memory the GPU writes over PCIe (rala_b200_graph_set_outputs),
// where three strided 4-byte stores per row would triple the number of write transactions.
__global__ void __launch_bounds__(256) k_pack_edges(const uint32_t* __restrict__ src, const uint32_t* __restrict__ dst,
                                                   const uint32_t* __restrict__ len, const uint32_t* __restrict__ n_edges_ptr,
                                                   uint32_t edge_cap, uint32_t* __restrict__ out, int vec16) {
    __shared__ __align__(16) uint32_t rows[256 * 3];
    const uint32_t n = min(*n_edges_ptr, edge_cap), tid = threadIdx.x;
    for (uint32_t base = blockIdx.x * 256u; base < n; base += gridDim.x * 256u) {
        const uint32_t e = base + tid;
        if (e < n) {
            rows[3 * tid] = src[e];
            rows[3 * tid + 1] = dst[e];
            rows[3 * tid + 2] = len[e];
        }
        __syncthreads();
        const uint32_t words = 3u * min(256u, n - base);
        uint32_t* o = out + 3 * (size_t) base;   // 3072 bytes per full block iteration: 16-byte aligned when `out` is
        if (vec16) {
            const uint32_t w = 4u * tid;
            if (w + 3u < words) *reinterpret_cast<uint4*>(o + w) = *reinterpret_cast<const uint4*>(rows + w);
            else for (uint32_t k = w; k < words; ++k) o[k] = rows[k];
        } else {
            for (uint32_t k = tid; k < words; k += 256u) o[k] = rows[k];
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Capacity-bounded exchange blocks of the multi-GPU path: the element count travels INSIDE the block, so the
// host never has to read it (no synchronisation around the collectives).  Word 2 is the rank's whole count, so after an
// overflow the caller learns from the gathered blocks how large `cap` has to be.
//   block = [n clamped to cap | overflow flag | n | 0 | column 0 [cap] | column 1 [cap] | column 2 [cap]]
// ---------------------------------------------------------------------------------------------
__global__ void k_export_padded(const uint32_t* __restrict__ c0, const uint32_t* __restrict__ c1, const uint32_t* __restrict__ c2,
                                const uint32_t* __restrict__ n_ptr, uint32_t src_cap, uint32_t cap, uint32_t* __restrict__ block) {
    const uint32_t n = min(*n_ptr, src_cap), m = min(n, cap);
    if (blockIdx.x == 0 && threadIdx.x < 4) block[threadIdx.x] = threadIdx.x == 0 ? m : (threadIdx.x == 1 ? (n > cap ? 1u : 0u) : (threadIdx.x == 2 ? n : 0u));
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        block[4 + i] = c0[i];
        block[4 + (size_t) cap + i] = c1[i];
        block[4 + 2 * (size_t) cap + i] = c2[i];
    }
}

// gathered = `world` blocks back to back; rank r's elements land behind those of ranks < r (blockIdx.y = r)
__global__ void k_import_gathered(const uint32_t* __restrict__ gathered, uint32_t cap, uint32_t world, uint32_t* __restrict__ d0,
                                  uint32_t* __restrict__ d1, uint32_t* __restrict__ d2, uint32_t dst_cap, uint32_t* __restrict__ n_out,
                                  uint32_t* __restrict__ overflow) {
    const size_t stride = 3 * (size_t) cap + 4;
    const uint32_t r = blockIdx.y;
    uint32_t offset = 0;
    for (uint32_t q = 0; q < r; ++q) offset += gathered[q * stride];
    const uint32_t* blk = gathered + r * stride;
    const uint32_t n = blk[0];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (blk[1] || offset + n > dst_cap) *overflow = 1u;
        if (r == world - 1) *n_out = min(offset + n, dst_cap);
    }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (offset + i < dst_cap) {
            d0[offset + i] = blk[4 + i];
            d1[offset + i] = blk[4 + (size_t) cap + i];
            d2[offset + i] = blk[4 + 2 * (size_t) cap + i];
        }
    }
}

// time bases of the local lists in the final containment pass (graph.cpp:831-866): position in the GLOBAL
// overlaps ++ internals order.  counts = (n_overlaps, n_internals) of every rank.
__global__ void k_time_bases(const uint32_t* __restrict__ counts, uint32_t rank, uint32_t world, uint32_t* __restrict__ bases) {
    if (blockIdx.x || threadIdx.x) return;
    uint32_t total_ovl = 0, ovl_before = 0, int_before = 0;
    for (uint32_t q = 0; q < world; ++q) {
        if (q < rank) {
            ovl_before += counts[2 * q];
            int_before += counts[2 * q + 1];
        }
        total_ovl += counts[2 * q];
    }
    bases[0] = ovl_before;
    bases[1] = total_ovl + int_before;
}

void launch_adjacency_view(Launch& L, const uint32_t* key, const uint8_t* marked, const uint32_t* n_edges_ptr, uint32_t edge_cap,
                           uint32_t n_nodes, uint32_t* degree_cursor, uint32_t* row_ptr, uint32_t* ids_tmp, uint32_t* ids_sorted,
                           unsigned long long* status, uint32_t* ticket) {
    cudaMemsetAsync(degree_cursor, 0, ((size_t) n_nodes + 8) * 4, L.stream);
    k_adj_hist<<<grid_for(edge_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(key, marked, n_edges_ptr, edge_cap, n_nodes, degree_cursor);
    L.count++;
    k_scan_degrees<<<grid_for(n_nodes + 1, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(degree_cursor, row_ptr, n_nodes + 1, status, ticket,
                                                                                          nullptr, nullptr, nullptr);
    L.count++;
    k_adj_fill<<<grid_for(edge_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(key, marked, n_edges_ptr, edge_cap, n_nodes, degree_cursor, ids_tmp);
    L.count++;
    k_adj_sort_rows<<<grid_for(n_nodes, 8, kNumSMs * 8), 256, 0, L.stream>>>(row_ptr, n_nodes, ids_tmp, ids_sorted);
    L.count++;
}

void launch_count_scan(Launch& L, List ovl, const uint32_t* n_ptr, uint32_t cap, const uint2* piles, uint32_t n_piles, GraphArrays g,
                       uint32_t edge_cap, uint32_t* tile_dov, uint32_t* counters, unsigned long long* status, uint32_t* ticket) {
    k_count_edges<<<grid_for(cap, kEmitTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(ovl, n_ptr, cap, piles,
                                                                                       g.cursor ? g.slot_degree : nullptr, tile_dov);
    L.count++;
    k_scan_piles<<<grid_for(n_piles, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(
        piles, n_piles, g.slot_degree, g.seq_to_node, g.row_ptr, g.cursor, tile_dov, n_ptr, cap, edge_cap, g.T, counters, status, ticket);
    L.count++;
}

void launch_emit_edges(Launch& L, List ovl, const uint32_t* n_ptr, uint32_t cap, const uint2* piles, GraphArrays g, uint32_t edge_cap,
                       const uint32_t* tile_base) {
    k_emit_edges<<<grid_for(cap, kEmitTile, kNumSMs * kEmitMinBlocks), kTileThreads, 0, L.stream>>>(
        ovl, n_ptr, cap, piles, g.seq_to_node, tile_base, g.src, g.dst, g.len, edge_cap, g.cursor, g.col, g.col_eid, g.T);
    L.count++;
}

void launch_pack_edges(Launch& L, cudaStream_t stream, GraphArrays g, uint32_t edge_cap, const uint32_t* n_edges_ptr, uint32_t* out) {
    k_pack_edges<<<grid_for(edge_cap, 256, kNumSMs * 8), 256, 0, stream>>>(g.src, g.dst, g.len, n_edges_ptr, edge_cap, out,
                                                                           (reinterpret_cast<uintptr_t>(out) & 15u) == 0 ? 1 : 0);
    L.count++;
}

void launch_degree_hist(Launch& L, const uint32_t* src, const uint32_t* n_edges_ptr, uint32_t edge_cap, uint32_t* cursor) {
    k_degree_hist<<<grid_for(edge_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(src, n_edges_ptr, edge_cap, cursor);
    L.count++;
}

void launch_export_padded(Launch& L, const uint32_t* c0, const uint32_t* c1, const uint32_t* c2, const uint32_t* n_ptr,
                          uint32_t src_cap, uint32_t cap, uint32_t* block) {
    k_export_padded<<<grid_for(cap, 256, kNumSMs * 4), 256, 0, L.stream>>>(c0, c1, c2, n_ptr, src_cap, cap, block);
    L.count++;
}

void launch_import_gathered(Launch& L, const uint32_t* gathered, uint32_t cap, uint32_t world, uint32_t* d0, uint32_t* d1,
                            uint32_t* d2, uint32_t dst_cap, uint32_t* n_out, uint32_t* overflow) {
    dim3 grid(grid_for(cap, 256, kNumSMs * 2), world);
    k_import_gathered<<<grid, 256, 0, L.stream>>>(gathered, cap, world, d0, d1, d2, dst_cap, n_out, overflow);
    L.count++;
}

void launch_time_bases(Launch& L, const uint32_t* counts, uint32_t rank, uint32_t world, uint32_t* bases) {
    k_time_bases<<<1, 32, 0, L.stream>>>(counts, rank, world, bases);
    L.count++;
}

// exclusive scan of n values: exclusive_out[i] and values_inout[i] both receive the prefix
void launch_scan_u32(Launch& L, uint32_t* values_inout, uint32_t* exclusive_out, uint32_t n, unsigned long long* status,
                     uint32_t* ticket, const uint32_t* skip, const uint32_t* run_if, const uint32_t* live) {
    k_scan_degrees<<<grid_for(n, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(values_inout, exclusive_out, n, status, ticket, skip, run_if, live);
    L.count++;
}

void launch_build_csr(Launch& L, GraphArrays g, uint32_t n_nodes_max, uint32_t edge_cap, uint32_t* counters,
                      unsigned long long* status, uint32_t* ticket) {
    // row_ptr has n_nodes_max + 1 entries; degrees beyond the live node count are zero
    k_scan_degrees<<<grid_for(n_nodes_max + 1, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(
        g.cursor, g.row_ptr, n_nodes_max + 1, status, ticket, nullptr, nullptr, counters + C_NODES);
    L.count++;
    k_fill_csr<<<grid_for(edge_cap, 256, kNumSMs * kFillBlocks), 256, 0, L.stream>>>(g.src, g.dst, g.len, counters + C_EDGES,
                                                                            edge_cap, g.cursor, g.col, g.col_eid, g.T);
    L.count++;
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_graph_build() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_count_edges);
    cudaFuncGetAttributes(&a, k_scan_piles);
    cudaFuncGetAttributes(&a, k_adj_hist);
    cudaFuncGetAttributes(&a, k_adj_fill);
    cudaFuncGetAttributes(&a, k_adj_sort_rows);
    cudaFuncGetAttributes(&a, k_emit_edges);
    cudaFuncGetAttributes(&a, k_degree_hist);
    cudaFuncGetAttributes(&a, k_scan_degrees);
    cudaFuncGetAttributes(&a, k_fill_csr);
    cudaFuncGetAttributes(&a, k_pack_edges);
    cudaFuncGetAttributes(&a, k_export_padded);
    cudaFuncGetAttributes(&a, k_import_gathered);
    cudaFuncGetAttributes(&a, k_time_bases);
}

}  // namespace rb
