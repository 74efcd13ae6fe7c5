// graph_build.cu — K2: node ids, edge list with reverse-complement twins, CSR adjacency.
//
// Replaces graph.cpp:552-632 (reference): sequence_id_to_node_id (:553-574), the two Edge objects per
// dovetail overlap with their lengths (:576-632) and the implicit adjacency (suffix_edges_ vectors).
#include <cstdlib>

#include "kernels.h"
#include "lists.cuh"

namespace rb {

// sequence_id_to_node_id[i] = 2 * rank(i among alive piles)  (graph.cpp:553-561)
__global__ void __launch_bounds__(kTileThreads) k_node_ids(const uint2* __restrict__ piles, uint32_t n_piles,
                                                          uint32_t* __restrict__ seq_to_node,
                                                          uint32_t* __restrict__ counters,
                                                          unsigned long long* __restrict__ status,
                                                          uint32_t* __restrict__ ticket) {
    __shared__ TileShared sh;
    const uint32_t tid = threadIdx.x;
    const uint32_t num_tiles = (n_piles + kTile - 1) / kTile;
    while (true) {
        if (tid == 0) sh.tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = sh.tile;
        if (tile >= num_tiles) break;
        int dest[kTileItems];
#pragma unroll
        for (int r = 0; r < kTileItems; ++r) {
            const uint32_t idx = tile * kTile + r * kTileThreads + tid;
            dest[r] = (idx < n_piles && (__ldg(piles + idx).y & kEndMask) != 0u) ? 1 : 0;
        }
        uint32_t pos[kTileItems];
        unsigned long long inclusive = 0;
        tile_rank<kTileItems>(sh, status, tile, dest, pos, &inclusive);
        if (tid == 0 && tile == num_tiles - 1) {
            counters[C_ALIVE] = count_a(inclusive);
            counters[C_NODES] = 2u * count_a(inclusive);
        }
#pragma unroll
        for (int r = 0; r < kTileItems; ++r) {
            const uint32_t idx = tile * kTile + r * kTileThreads + tid;
            if (idx < n_piles) seq_to_node[idx] = dest[r] ? 2u * pos[r] : kInf;
        }
        __syncthreads();
    }
}

// Two edges per dovetail overlap, ids 2j / 2j+1 in list order (graph.cpp:576-632), plus the
// out-degree histogram the CSR build needs.
constexpr int kEmitTile = kTileThreads * kEmitItems;
__global__ void __launch_bounds__(kTileThreads) k_emit_edges(List ovl, const uint32_t* __restrict__ n_ptr, uint32_t cap,
                                                            const uint2* __restrict__ piles,
                                                            const uint32_t* __restrict__ seq_to_node,
                                                            uint32_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                            uint32_t* __restrict__ len, uint32_t edge_cap,
                                                            uint32_t* __restrict__ degree, uint32_t* __restrict__ rank,
                                                            uint32_t* __restrict__ counters,
                                                            unsigned long long* __restrict__ status,
                                                            uint32_t* __restrict__ ticket) {
    __shared__ TileShared sh;
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*n_ptr, cap);
    const uint32_t num_tiles = (n + kEmitTile - 1) / kEmitTile;
    while (true) {
        if (tid == 0) sh.tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = sh.tile;
        if (tile >= num_tiles) break;
        int dest[kEmitItems];
        uint32_t e_src[kEmitItems], e_dst[kEmitItems], e_len[kEmitItems], c_len[kEmitItems];
        // all gathers of the thread's four entries are issued before the first one is used: the entry (7 columns), then
        // both piles and both node ids (they only depend on the ids), 16 independent gathers in flight per thread
        // (issuing them entry by entry, behind the liveness test of the entry before, left the kernel at 15 % issue activity)
        Entry e[kEmitItems];
        bool have[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            const uint32_t idx = tile * kEmitTile + r * kTileThreads + tid;
            have[r] = idx < n;
            e[r] = load_entry(ovl, have[r] ? idx : 0u);
        }
        uint2 pa[kEmitItems], pb[kEmitItems];
        uint32_t na[kEmitItems], nb[kEmitItems];
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            pa[r] = __ldg(piles + e[r].a);
            pb[r] = __ldg(piles + e[r].b);
            na[r] = __ldg(seq_to_node + e[r].a);
            nb[r] = __ldg(seq_to_node + e[r].b);
        }
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            dest[r] = 0;
            Pile A, B;
            A.begin = pa[r].x; A.end = pa[r].y & kEndMask; A.flags = pa[r].y >> 30;
            B.begin = pb[r].x; B.end = pb[r].y & kEndMask; B.flags = pb[r].y >> 30;
            if (have[r] && A.alive() && B.alive()) {
                const Rel q = relative(e[r].c, e[r].ori, A, B);
                const uint8_t t = classify(e[r].c, q);                       // it->type(piles_) at :594 / :612
                const uint32_t node_a = na[r], node_b = nb[r] + e[r].ori;    // :578-580
                if (t == kAB) {                                              // :594-610
                    dest[r] = 1;
                    e_src[r] = node_a; e_dst[r] = node_b;
                    e_len[r] = q.a0 - q.b0;
                    c_len[r] = (q.bl - q.b1) - (q.al - q.a1);
                } else if (t == kBA) {                                       // :612-629
                    dest[r] = 1;
                    e_src[r] = node_b; e_dst[r] = node_a;
                    e_len[r] = q.b0 - q.a0;
                    c_len[r] = (q.al - q.a1) - (q.bl - q.b1);
                }
            }
        }
        uint32_t pos[kEmitItems];
        unsigned long long inclusive = 0;
        tile_rank<kEmitItems>(sh, status, tile, dest, pos, &inclusive);
        if (tid == 0 && tile == num_tiles - 1) {
            counters[C_DOVETAILS] = count_a(inclusive);
            counters[C_EDGES] = 2u * count_a(inclusive);
            if (2ull * count_a(inclusive) > edge_cap) counters[C_OVERFLOW] = 1u;
        }
#pragma unroll
        for (int r = 0; r < kEmitItems; ++r) {
            if (dest[r] && 2ull * pos[r] + 1 < edge_cap) {
                const uint32_t j = pos[r];
                // edge 2j = (from -> to), edge 2j+1 = (to^1 -> from^1): one 8-byte store per column
                reinterpret_cast<uint2*>(src)[j] = make_uint2(e_src[r], e_dst[r] ^ 1u);
                reinterpret_cast<uint2*>(dst)[j] = make_uint2(e_dst[r], e_src[r] ^ 1u);
                reinterpret_cast<uint2*>(len)[j] = make_uint2(e_len[r], c_len[r]);
                if (degree) {   // nullptr: the edges are routed to the owners of their source nodes, who count them
                    const uint32_t r0 = atomicAdd(&degree[e_src[r]], 1u);
                    const uint32_t r1 = atomicAdd(&degree[e_dst[r] ^ 1u], 1u);
                    // the count an edge found is its slot inside its row (any order of a row is as good as another)
                    if (rank) reinterpret_cast<uint2*>(rank)[j] = make_uint2(r0, r1);
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

// Scatter every edge into its source row.  Slot order inside a row is arbitrary (atomic cursor);
// nothing downstream depends on it: the transitive pass resolves parallel edges by edge id.
// Also clears the per-edge "transitive test passed" bytes T[0 .. n rounded up to 16) for the pass that follows
// (k_finalize_marks reads whole 16-byte groups): a memset of the buffer's CAPACITY (2 x the record count) would
// write ~15 x more bytes than there are edges.
// eight edges in flight per thread, or twice the blocks, changed nothing (profiles/r02ab_ab.json)
constexpr int kFillInflight = 4;
constexpr int kFillBlocks = 8;   // per SM
__global__ void k_fill_csr(const uint32_t* __restrict__ src, const uint32_t* __restrict__ dst,
                           const uint32_t* __restrict__ len, const uint32_t* __restrict__ n_edges_ptr, uint32_t edge_cap,
                           uint32_t* __restrict__ cursor, uint2* __restrict__ col, uint32_t* __restrict__ col_eid,
                           uint8_t* __restrict__ T, const uint32_t* __restrict__ rank, const uint32_t* __restrict__ row_ptr) {
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
        if (rank) {   // slots were handed out while the degrees were counted: a gather instead of a returning atomic
#pragma unroll
            for (int k = 0; k < F; ++k)
                if (e0 + k * stride < n) p[k] = rank[e0 + k * stride];
#pragma unroll
            for (int k = 0; k < F; ++k)
                if (e0 + k * stride < n) p[k] += row_ptr[s[k]];
        } else {
#pragma unroll
            for (int k = 0; k < F; ++k)
                if (e0 + k * stride < n) p[k] = atomicAdd(&cursor[s[k]], 1u);
        }
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

void launch_node_ids(Launch& L, const uint2* piles, uint32_t n_piles, uint32_t* seq_to_node, uint32_t* counters,
                     unsigned long long* status, uint32_t* ticket) {
    if (n_piles == 0) return;
    k_node_ids<<<grid_for(n_piles, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(piles, n_piles, seq_to_node, counters,
                                                                                      status, ticket);
    L.count++;
}

void launch_emit_edges(Launch& L, List ovl, const uint32_t* n_ptr, uint32_t cap, const uint2* piles, GraphArrays g,
                       uint32_t edge_cap, uint32_t* counters, unsigned long long* status, uint32_t* ticket) {
    k_emit_edges<<<grid_for(cap, kEmitTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(
        ovl, n_ptr, cap, piles, g.seq_to_node, g.src, g.dst, g.len, edge_cap, g.cursor, g.rank, counters, status, ticket);
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
                     uint32_t* ticket, const uint32_t* skip, const uint32_t* run_if) {
    k_scan_degrees<<<grid_for(n, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(values_inout, exclusive_out, n, status, ticket, skip, run_if, nullptr);
    L.count++;
}

void launch_build_csr(Launch& L, GraphArrays g, uint32_t n_nodes_max, uint32_t edge_cap, uint32_t* counters,
                      unsigned long long* status, uint32_t* ticket, bool ranked) {
    // row_ptr has n_nodes_max + 1 entries; degrees beyond the live node count are zero
    k_scan_degrees<<<grid_for(n_nodes_max + 1, kTile, kNumSMs * 8), kTileThreads, 0, L.stream>>>(
        g.cursor, g.row_ptr, n_nodes_max + 1, status, ticket, nullptr, nullptr, counters + C_NODES);
    L.count++;
    k_fill_csr<<<grid_for(edge_cap, 256, kNumSMs * kFillBlocks), 256, 0, L.stream>>>(g.src, g.dst, g.len, counters + C_EDGES,
                                                                            edge_cap, g.cursor, g.col, g.col_eid, g.T,
                                                                            ranked ? g.rank : nullptr, g.row_ptr);
    L.count++;
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_graph_build() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_node_ids);
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
