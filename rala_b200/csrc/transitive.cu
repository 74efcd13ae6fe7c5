// transitive.cu — K3: transitive-edge reduction on the CSR adjacency.
//
// Replaces Graph::remove_transitive_edges, graph.cpp:1281-1318 (reference), in its order-free form
// (SURVEY.md A.4):  cand(a,c) = highest-id edge a->c;  T(e = cand(a,c)) = exists a->b, b->c with
// comparable(len_ab + len_bc, len_e, 0.12);  marked(e) = T(e) | T(e^1);  return = #{j : marked(2j)}.
//
// Per node a the neighbour set N+(a) is staged in shared memory: rank-sorted by (destination, edge id) and searched with
// a branch-free binary search on the group path (the last key <= x is the highest edge id: "highest id wins" for
// parallel edges, graph.cpp:1291-1293), an open-addressing hash table keyed by destination (value = edge id << 32 |
// length, merged with max) on the light and heavy paths.  The two-hop stream  { (b, j) : b in N+(a), j < deg(b) }  is
// FLATTENED: lanes take consecutive flat indices, so several short rows N+(b) are in flight per
// iteration and every load is an 8-byte (dst, len) element of a contiguous CSR row.
//   group path : 8 lanes per node, 4 nodes per warp   (2 <= deg <= 16 and <= 4096 two-hop visits: almost every
//                node of an overlap graph, mean out-degree ~9; a full warp per such node leaves 3/4 of
//                the lanes idle during set-up and pays the per-node overhead four times as often)
//   light path : one warp per node      (16 < deg <= 64 and <= 32768 two-hop visits)
//   heavy path : one block per (node, hash chunk of 1024 neighbours, stream chunk of 256 neighbours); the two kernels
//                above hand it NODES, and its blocks map onto the work items of each node through a prefix
// Measured alternatives that lost (profiles/README.md): one thread per edge with a linear or (rows sorted)
// binary-search membership test, and the group path streaming one row N+(b) at a time: both expose the
// latency of dependent L2 gathers; the flattened stream keeps 4 independent gathers in flight per lane.
#include "kernels.h"
#include "common.cuh"

namespace rb {

constexpr uint32_t kEmpty = 0xFFFFFFFFu;
constexpr int kGroupLanes = 8;
constexpr int kGroupsPerWarp = 32 / kGroupLanes;
constexpr int kGroupMaxDeg = 16;
constexpr uint32_t kGroupMaxVisits = 4096;
constexpr int kLightMaxDeg = 64;
constexpr int kLightCap = 128;
constexpr uint32_t kLightMaxVisits = 32768;
constexpr int kLightWarps = 8;
constexpr int kHeavyHashChunk = 1024;   // a node with more neighbours than this is split into hash chunks ...
constexpr int kHeavyChunkFill = 768;    // ... of this expected size, assigned BY DESTINATION (see hash_chunk_of)
constexpr int kHeavyCap = 2048;
constexpr int kHeavyNbrChunk = 256;
constexpr int kHeavyThreads = 256;

__device__ __forceinline__ uint32_t hash_slot(uint32_t key, uint32_t log2cap) {
    return (key * 0x9E3779B1u) >> (32u - log2cap);
}

// Number of hash chunks of a node with d neighbours, and the chunk a destination belongs to.  Chunks
// partition N+(a) by destination, not by position, so that parallel edges a->c always meet in the same
// table and "highest id wins" stays a per-table decision.
__host__ __device__ __forceinline__ uint32_t num_hash_chunks(uint32_t d) {
    return d <= (uint32_t) kHeavyHashChunk ? 1u : (d + kHeavyChunkFill - 1) / kHeavyChunkFill;
}
__device__ __forceinline__ uint32_t hash_chunk_of(uint32_t key, uint32_t n_chunks) {
    return n_chunks == 1 ? 0u : ((key * 0x85EBCA6Bu) >> 12) % n_chunks;
}

__device__ __forceinline__ void table_insert(uint32_t* keys, unsigned long long* vals, uint32_t mask, uint32_t log2cap,
                                             uint32_t key, unsigned long long val) {
    uint32_t s = hash_slot(key, log2cap);
    while (true) {
        uint32_t prev = atomicCAS(&keys[s], kEmpty, key);
        if (prev == kEmpty || prev == key) {
            atomicMax(&vals[s], val);
            return;
        }
        s = (s + 1u) & mask;
    }
}

// same, but gives up (returns false) after probing the whole table
__device__ __forceinline__ bool table_insert_bounded(uint32_t* keys, unsigned long long* vals, uint32_t mask, uint32_t log2cap,
                                                     uint32_t key, unsigned long long val) {
    uint32_t s = hash_slot(key, log2cap);
    for (uint32_t probes = 0; probes <= mask; ++probes) {
        uint32_t prev = atomicCAS(&keys[s], kEmpty, key);
        if (prev == kEmpty || prev == key) {
            atomicMax(&vals[s], val);
            return true;
        }
        s = (s + 1u) & mask;
    }
    return false;
}

// returns the slot of key or kEmpty.  The light path's table has at least 2d slots for its d keys: it is at most half
// full, so the probe always meets an empty slot.
__device__ __forceinline__ uint32_t table_find(const uint32_t* keys, uint32_t mask, uint32_t log2cap, uint32_t key) {
    uint32_t s = hash_slot(key, log2cap);
    while (true) {
        uint32_t k = keys[s];
        if (k == key) return s;
        if (k == kEmpty) return kEmpty;
        s = (s + 1u) & mask;
    }
}

// same, but gives up (returns kEmpty: the key is absent) after probing the whole table.  A hash chunk of the heavy path
// can hold exactly kHeavyCap keys, which leaves no empty slot to stop at.
__device__ __forceinline__ uint32_t table_find_bounded(const uint32_t* keys, uint32_t mask, uint32_t log2cap, uint32_t key) {
    uint32_t s = hash_slot(key, log2cap);
    for (uint32_t probes = 0; probes <= mask; ++probes) {
        const uint32_t k = keys[s];
        if (k == key) return s;
        if (k == kEmpty) return kEmpty;
        s = (s + 1u) & mask;
    }
    return kEmpty;
}

// Hands node a to k_transitive_heavy as `units` work items.  The node count (low word) and the item count (high word)
// move in ONE 64-bit atomic, so entry i's unit base is the sum of the items of entries 0 .. i-1: the bases ascend with
// the entry index, and k_transitive_heavy finds the entry of an item by search.  A node is handed over at most once,
// so the node count stays below heavy.cap (= n_nodes_max); more than 2^32 items in all is an overflow.
__device__ __forceinline__ void heavy_append(HeavyItems heavy, uint32_t* counters, uint32_t a, unsigned long long units) {
    const unsigned long long old =
        atomicAdd(reinterpret_cast<unsigned long long*>(counters + C_HEAVY_NODES), (units << 32) | 1ull);
    const uint32_t i = (uint32_t) old;
    if (i < heavy.cap && (old >> 32) + units <= 0xFFFFFFFFull) {
        heavy.node[i] = a;
        heavy.unit_base[i] = (uint32_t) (old >> 32);
    } else {
        counters[C_OVERFLOW] = 1u;
    }
}

// largest i < n with base[i] <= u (base[0] == 0 <= u, base ascending): a 32-ary search, one probe per lane and
// ceil(log32 n) dependent loads; every lane of the warp returns the same i
__device__ __forceinline__ uint32_t heavy_entry(const uint32_t* __restrict__ base, uint32_t n, uint32_t u, uint32_t lane) {
    uint32_t lo = 0, hi = n;   // base[lo] <= u, and hi == n or base[hi] > u
    while (hi - lo > 1) {
        const uint32_t step = (hi - lo + 31) / 32;
        const uint32_t p = lo + lane * step;
        const uint32_t le = __ballot_sync(0xFFFFFFFFu, p < hi && base[p] <= u);   // lanes 0 .. k, lane 0 always
        lo += (31 - __clz(le)) * step;
        hi = min(hi, lo + step);
    }
    return lo;
}


// ---------------------------------------------------------------------------------------------
// group path: 8 lanes per node
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t group_inclusive_scan(uint32_t v, uint32_t gl) {
#pragma unroll
    for (int d = 1; d < kGroupLanes; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d, kGroupLanes);
        if ((int) gl >= d) v += t;
    }
    return v;
}

// Membership of a two-hop destination in N+(a) is a BRANCH-FREE binary search over the (at most 16) neighbours,
// sorted by (destination, edge id) with a rank sort during set-up: four dependent shared-memory loads, the same
// for every lane.  The open-addressing table this replaces cost 48 % of the kernel's instructions at 7 of 32
// lanes active: every lane left its probe loop after a different number of steps (profiles/r01i, source view).
// Parallel edges a->c sit next to each other in edge-id order and the search returns the LAST key <= x, i.e. the
// highest id: the candidate of graph.cpp:1291-1293; earlier duplicates can never be hit.
struct GroupSmem {
    unsigned long long ukey[kGroupMaxDeg];   // as loaded: destination << 32 | edge id, padded with ~0
    uint32_t keys[kGroupMaxDeg];             // destinations, sorted; kEmpty behind the last one
    uint32_t eid[kGroupMaxDeg];              // edge id at that position
    uint2 iv[kGroupMaxDeg];                  // comparable(sum, len of that edge)  <=>  sum - iv.x <= iv.y
    uint2 prow[kGroupMaxDeg];                // per neighbour b: (start of row b in col - its offset in the flat stream, len of a->b)
    uint32_t noff[kGroupMaxDeg + 1];
    uint32_t hit;                            // bit j: the edge at sorted position j passed the test
};

// resident blocks per SM: 6 (40 registers) is a sharp optimum: 115 us, against 134 us at 4 or 5 and 148 us at 7 or 8
// (profiles/r02ab_ab.json, r02ad_ab.json): the kernel lives on its shared-memory / L1 data path (69 % of peak)
constexpr int kGroupMinBlocks = 6;
__global__ void __launch_bounds__(kLightWarps * 32, kGroupMinBlocks) k_transitive_group(
    const uint32_t* __restrict__ row_ptr, const uint2* __restrict__ col, const uint32_t* __restrict__ col_eid,
    uint8_t* __restrict__ T, const uint32_t* __restrict__ node_range, const uint32_t* __restrict__ n_nodes_ptr,
    uint32_t* __restrict__ work_counter, HeavyItems heavy, uint32_t* __restrict__ counters) {
    static_assert(kGroupMaxDeg == 16 && kGroupLanes == 8, "the search below is written for 16 keys, two per lane");
    __shared__ GroupSmem smem[kLightWarps][kGroupsPerWarp];
    const uint32_t lane = lane_id(), gl = lane & (kGroupLanes - 1), grp = lane / kGroupLanes;
    GroupSmem& S = smem[warp_id()][grp];
    const uint32_t node_begin = node_range ? node_range[0] : 0u;
    const uint32_t n_end = node_range ? min(node_range[1], *n_nodes_ptr) : *n_nodes_ptr;
    unsigned long long visits = 0;

    while (true) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(work_counter, 32u);
        base = node_begin + __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= n_end) break;
        uint32_t r0 = 0, deg = 0;
        if (base + lane < n_end) {
            r0 = row_ptr[base + lane];
            deg = row_ptr[base + lane + 1] - r0;
        }
#pragma unroll 1
        for (uint32_t round = 0; round < 32 / kGroupsPerWarp; ++round) {
            const uint32_t from = round * kGroupsPerWarp + grp;
            const uint32_t a = base + from;
            const uint32_t ra0 = __shfl_sync(0xFFFFFFFFu, r0, from);
            const uint32_t d = __shfl_sync(0xFFFFFFFFu, deg, from);
            bool act = d >= 2u && d <= (uint32_t) kGroupMaxDeg;   // < 2 neighbours: no two-hop witness can exist
            if (!__any_sync(0xFFFFFFFFu, act)) continue;
            // ---- this lane's (at most two) neighbours ----
            unsigned long long mine[2] = {~0ull, ~0ull};
            uint32_t dg[2] = {0u, 0u}, my_len[2] = {0u, 0u};
            uint32_t rs2[2] = {0u, 0u};
            if (act) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t i = gl + h * kGroupLanes;
                    if (i < d) {
                        const uint2 e = col[ra0 + i];
                        mine[h] = ((unsigned long long) e.x << 32) | col_eid[ra0 + i];
                        my_len[h] = e.y;
                        const uint32_t rs = row_ptr[e.x];
                        dg[h] = row_ptr[e.x + 1] - rs;
                        rs2[h] = rs;
                    }
                    S.ukey[i] = mine[h];
                }
                if (gl == 0) S.hit = 0u;
            }
            const uint32_t inc0 = group_inclusive_scan(dg[0], gl), inc1 = group_inclusive_scan(dg[1], gl);
            const uint32_t tot0 = __shfl_sync(0xFFFFFFFFu, inc0, kGroupLanes - 1, kGroupLanes);
            const uint32_t W = tot0 + __shfl_sync(0xFFFFFFFFu, inc1, kGroupLanes - 1, kGroupLanes);
            if (act) {
                if (gl < d) S.noff[gl] = inc0 - dg[0];
                if (gl + kGroupLanes < d) S.noff[gl + kGroupLanes] = tot0 + inc1 - dg[1];
                if (gl == 0) S.noff[d] = W;
                // element f of the flat stream that falls into row i is col[prow[i].x + f]
                if (gl < d) S.prow[gl] = make_uint2(rs2[0] - (inc0 - dg[0]), my_len[0]);
                if (gl + kGroupLanes < d) S.prow[gl + kGroupLanes] = make_uint2(rs2[1] - (tot0 + inc1 - dg[1]), my_len[1]);
            }
            __syncwarp();
            if (act && W > kGroupMaxVisits) {   // short row, very long rows behind it: give the node to a block
                if (gl == 0) heavy_append(heavy, counters, a, 1ull);
                act = false;
            }
            // ---- rank sort by (destination, edge id): composites are distinct, pads (~0) sort behind every edge ----
            if (act) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t i = gl + h * kGroupLanes;
                    if (i < d) {
                        uint32_t rank = 0;
#pragma unroll
                        for (int j = 0; j < kGroupMaxDeg; ++j) rank += S.ukey[j] < mine[h] ? 1u : 0u;
                        S.keys[rank] = (uint32_t) (mine[h] >> 32);
                        S.eid[rank] = (uint32_t) mine[h];
                        S.iv[rank] = comparable_interval(my_len[h]);
                    } else {
                        S.keys[i] = kEmpty;   // positions d .. 15
                    }
                }
            }
            __syncwarp();
            if (act) {
                if (gl == 0) visits += W;
                uint32_t i = 0;
                for (uint32_t f0 = 0; f0 < W; f0 += 4 * kGroupLanes) {
                    uint2 e[4];
                    uint32_t lab[4];
                    bool ok[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const uint32_t f = f0 + u * kGroupLanes + gl;
                        ok[u] = f < W;
                        e[u] = make_uint2(kEmpty, 0u);
                        lab[u] = 0u;
                        if (ok[u]) {
                            while (f >= S.noff[i + 1]) ++i;
                            const uint2 row = S.prow[i];
                            e[u] = col[row.x + f];
                            lab[u] = row.y;
                        }
                    }
                    uint32_t pass = 0;   // bit j: a witness for the edge at sorted position j
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const uint32_t x = e[u].x;   // kEmpty for idle lanes: matches no key below position d
                        uint32_t j = S.keys[8] <= x ? 8u : 0u;
                        j += S.keys[j + 4] <= x ? 4u : 0u;
                        j += S.keys[j + 2] <= x ? 2u : 0u;
                        j += S.keys[j + 1] <= x ? 1u : 0u;
                        const uint2 iv = S.iv[j];
                        if (ok[u] && S.keys[j] == x && lab[u] + e[u].y - iv.x <= iv.y) pass |= 1u << j;   // graph.cpp:1301-1306
                    }
                    if (pass & ~S.hit) atomicOr(&S.hit, pass);
                }
            }
            __syncwarp();
            if (act) {
                const uint32_t h = S.hit;
#pragma unroll
                for (uint32_t j = gl; j < (uint32_t) kGroupMaxDeg; j += kGroupLanes) {
                    if ((h >> j) & 1u) T[S.eid[j]] = 1;
                }
            }
            __syncwarp();
        }
    }
    visits = warp_sum64(visits);
    if (lane == 0 && visits) atomicAdd(reinterpret_cast<unsigned long long*>(counters + C_HOP_LO), visits);
}

struct LightSmem {
    unsigned long long vals[kLightCap];
    uint32_t keys[kLightCap];
    uint32_t nrow[kLightMaxDeg];
    uint32_t nlen[kLightMaxDeg];
    uint32_t noff[kLightMaxDeg + 1];
    uint8_t hit[kLightCap];
};

__global__ void __launch_bounds__(kLightWarps * 32) k_transitive_light(
    const uint32_t* __restrict__ row_ptr, const uint2* __restrict__ col, const uint32_t* __restrict__ col_eid,
    uint8_t* __restrict__ T, const uint32_t* __restrict__ node_range, const uint32_t* __restrict__ n_nodes_ptr,
    uint32_t* __restrict__ work_counter, HeavyItems heavy, uint32_t* __restrict__ counters) {
    __shared__ LightSmem smem[kLightWarps];
    LightSmem& S = smem[warp_id()];
    const uint32_t lane = lane_id();
    // multi-GPU: this rank's share of the source nodes, computed on the device
    const uint32_t node_begin = node_range ? node_range[0] : 0u;
    const uint32_t n_end = node_range ? min(node_range[1], *n_nodes_ptr) : *n_nodes_ptr;
    unsigned long long visits = 0;

    while (true) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(work_counter, 32u);
        base = node_begin + __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= n_end) break;
        const uint32_t node = base + lane;
        uint32_t r0 = 0, deg = 0;
        if (node < n_end) {
            r0 = row_ptr[node];
            deg = row_ptr[node + 1] - r0;
        }
        uint32_t todo = __ballot_sync(0xFFFFFFFFu, deg > (uint32_t) kGroupMaxDeg);   // smaller nodes: k_transitive_group
        while (todo) {
            const uint32_t l = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t a = base + l;
            const uint32_t ra0 = __shfl_sync(0xFFFFFFFFu, r0, l);
            const uint32_t d = __shfl_sync(0xFFFFFFFFu, deg, l);
            if (d > (uint32_t) kLightMaxDeg) {   // one work item per (hash chunk, stream chunk)
                if (lane == 0)
                    heavy_append(heavy, counters, a, (unsigned long long) num_hash_chunks(d) * ((d + kHeavyNbrChunk - 1) / kHeavyNbrChunk));
                continue;
            }
            // table capacity: power of two >= 2d, at least 16
            uint32_t log2cap = 4;
            while ((1u << log2cap) < 2u * d) ++log2cap;
            const uint32_t cap = 1u << log2cap, mask = cap - 1u;
            for (uint32_t s = lane; s < cap; s += 32) {
                S.keys[s] = kEmpty;
                S.vals[s] = 0ull;
                S.hit[s] = 0;
            }
            __syncwarp();
            uint32_t carry = 0;
            for (uint32_t i0 = 0; i0 < d; i0 += 32) {
                const uint32_t i = i0 + lane;
                uint32_t dg = 0;
                if (i < d) {
                    const uint2 e = col[ra0 + i];
                    const uint32_t eid = col_eid[ra0 + i];
                    table_insert(S.keys, S.vals, mask, log2cap, e.x, ((unsigned long long) eid << 32) | e.y);
                    const uint32_t rs = row_ptr[e.x];
                    dg = row_ptr[e.x + 1] - rs;
                    S.nrow[i] = rs;
                    S.nlen[i] = e.y;
                }
                const uint32_t inc = warp_inclusive_scan(dg);
                if (i < d) S.noff[i] = carry + inc - dg;
                carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
            }
            const uint32_t W = carry;
            if (lane == 0) S.noff[d] = W;
            __syncwarp();
            if (W > kLightMaxVisits) {   // few neighbours but very long rows behind them: give it to a block (one item)
                if (lane == 0) heavy_append(heavy, counters, a, 1ull);
                __syncwarp();
                continue;
            }
            if (lane == 0) visits += W;

            // flattened two-hop stream, 4 independent loads in flight per lane
            uint32_t i = 0;
            for (uint32_t f0 = 0; f0 < W; f0 += 128) {
                uint2 e[4];
                uint32_t lab[4];
                bool ok[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t f = f0 + u * 32 + lane;
                    ok[u] = f < W;
                    if (ok[u]) {
                        while (f >= S.noff[i + 1]) ++i;
                        e[u] = col[S.nrow[i] + (f - S.noff[i])];
                        lab[u] = S.nlen[i];
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (ok[u]) {
                        const uint32_t s = table_find(S.keys, mask, log2cap, e[u].x);
                        if (s != kEmpty && !S.hit[s]) {
                            if (comparable(lab[u] + e[u].y, (uint32_t) S.vals[s])) S.hit[s] = 1;   // graph.cpp:1301-1306
                        }
                    }
                }
            }
            __syncwarp();
            for (uint32_t s = lane; s < cap; s += 32) {
                if (S.hit[s]) T[(uint32_t) (S.vals[s] >> 32)] = 1;
            }
            __syncwarp();
        }
    }
    visits = warp_sum64(visits);
    if (lane == 0 && visits) atomicAdd(reinterpret_cast<unsigned long long*>(counters + C_HOP_LO), visits);
}

struct HeavySmem {
    unsigned long long vals[kHeavyCap];
    uint32_t keys[kHeavyCap];
    uint32_t nrow[kHeavyNbrChunk];
    uint32_t nlen[kHeavyNbrChunk];
    uint32_t noff[kHeavyNbrChunk + 1];
    uint32_t warp_sums[kHeavyThreads / 32];
    uint8_t hit[kHeavyCap];
};

__global__ void __launch_bounds__(kHeavyThreads) k_transitive_heavy(
    const uint32_t* __restrict__ row_ptr, const uint2* __restrict__ col, const uint32_t* __restrict__ col_eid,
    uint8_t* __restrict__ T, HeavyItems heavy, uint32_t* __restrict__ counters) {
    __shared__ HeavySmem S;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t n_nodes = min(counters[C_HEAVY_NODES], heavy.cap);
    const uint32_t n_items = n_nodes ? counters[C_HEAVY] : 0u;
    unsigned long long visits = 0;
    for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
        // node a's items: hash chunk ca (slow) x stream chunk cb (fast)
        const uint32_t k = heavy_entry(heavy.unit_base, n_nodes, item, lane);
        const uint32_t a = heavy.node[k], local = item - heavy.unit_base[k];
        const uint32_t ra0 = row_ptr[a], d = row_ptr[a + 1] - ra0;
        const uint32_t nca = num_hash_chunks(d), ncb = (d + kHeavyNbrChunk - 1) / kHeavyNbrChunk;
        const uint32_t ca = local / ncb, cb = local % ncb;
        if (ca >= nca) continue;   // only behind an overflow (the result is refused): the block agrees, no barrier is skipped
        const uint32_t k0 = cb * kHeavyNbrChunk, k1 = min(d, k0 + kHeavyNbrChunk), nb = k1 - k0;
        uint32_t log2cap = 4;
        while ((1u << log2cap) < 2u * min(d, (uint32_t) kHeavyHashChunk)) ++log2cap;
        const uint32_t cap = 1u << log2cap, mask = cap - 1u;
        for (uint32_t s = tid; s < cap; s += kHeavyThreads) {
            S.keys[s] = kEmpty;
            S.vals[s] = 0ull;
            S.hit[s] = 0;
        }
        __syncthreads();
        for (uint32_t i = tid; i < d; i += kHeavyThreads) {
            const uint2 e = col[ra0 + i];
            if (hash_chunk_of(e.x, nca) != ca) continue;
            if (!table_insert_bounded(S.keys, S.vals, mask, log2cap, e.x, ((unsigned long long) col_eid[ra0 + i] << 32) | e.y))
                counters[C_OVERFLOW] = 1u;   // > kHeavyCap distinct destinations hashed into one chunk: reported as an error
        }
        uint32_t dg = 0;
        if (tid < nb) {
            const uint2 e = col[ra0 + k0 + tid];
            const uint32_t rs = row_ptr[e.x];
            dg = row_ptr[e.x + 1] - rs;
            S.nrow[tid] = rs;
            S.nlen[tid] = e.y;
        }
        const uint32_t inc = warp_inclusive_scan(dg);
        if (lane == 31) S.warp_sums[warp] = inc;
        __syncthreads();
        uint32_t woff = 0;
        for (uint32_t w = 0; w < warp; ++w) woff += S.warp_sums[w];
        if (tid < nb) S.noff[tid] = woff + inc - dg;
        if (tid == kHeavyThreads - 1) S.noff[nb] = woff + inc;   // dg == 0 beyond nb, so this is the total
        __syncthreads();
        const uint32_t W = S.noff[nb];
        if (ca == 0 && tid == 0) visits += W;

        for (uint32_t f0 = 0; f0 < W; f0 += kHeavyThreads * 4) {
            uint2 e[4];
            uint32_t lab[4];
            bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t f = f0 + u * kHeavyThreads + tid;
                ok[u] = f < W;
                if (ok[u]) {
                    uint32_t lo = 0, hi = nb;   // largest i with noff[i] <= f
                    while (hi - lo > 1) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (S.noff[mid] <= f) lo = mid; else hi = mid;
                    }
                    e[u] = col[S.nrow[lo] + (f - S.noff[lo])];
                    lab[u] = S.nlen[lo];
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (ok[u]) {
                    const uint32_t s = table_find_bounded(S.keys, mask, log2cap, e[u].x);
                    if (s != kEmpty && !S.hit[s]) {
                        if (comparable(lab[u] + e[u].y, (uint32_t) S.vals[s])) S.hit[s] = 1;
                    }
                }
            }
        }
        __syncthreads();
        for (uint32_t s = tid; s < cap; s += kHeavyThreads) {
            if (S.hit[s]) T[(uint32_t) (S.vals[s] >> 32)] = 1;
        }
        __syncthreads();
    }
    if (tid == 0 && visits) atomicAdd(reinterpret_cast<unsigned long long*>(counters + C_HOP_LO), visits);
}

// marked(e) = T(e) | T(e^1); count of marked pairs = the reference's return value (graph.cpp:1305-1309, 1334).
// 16 edges (one 16-byte load / store) per thread: T and marked are padded to a multiple of 256 bytes and T is zero
// behind the last edge.  marked_copy, when given, is the caller's buffer (rala_b200_graph_set_outputs: pinned host
// memory the GPU addresses directly, so the marks cross PCIe as 16-byte stores while they are produced).
__global__ void k_finalize_marks(const uint8_t* __restrict__ T, uint8_t* __restrict__ marked,
                                 const uint32_t* __restrict__ n_edges_ptr, uint32_t edge_cap, uint32_t* __restrict__ counters,
                                 uint8_t* __restrict__ marked_copy, uint32_t copy_cap) {
    const uint32_t n = min(*n_edges_ptr, edge_cap);
    const uint32_t n16 = (n + 15u) / 16u;
    const bool copy_vec = marked_copy && (reinterpret_cast<uintptr_t>(marked_copy) & 15u) == 0;
    uint32_t local = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) {
        const uint4 t = reinterpret_cast<const uint4*>(T)[i];
        uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // bytes are 0 / 1: each 16-bit half holds one pair (e, e ^ 1)
            const uint32_t any = (w[k] | (w[k] >> 8)) & 0x00010001u;
            local += __popc(any);
            w[k] = any | (any << 8);
        }
        const uint4 m = make_uint4(w[0], w[1], w[2], w[3]);
        reinterpret_cast<uint4*>(marked)[i] = m;
        if (marked_copy) {   // exactly min(n, copy_cap) bytes of the caller's buffer are written
            const uint32_t lim = min(n, copy_cap);
            if (copy_vec && 16u * i + 15u < lim) {
                reinterpret_cast<uint4*>(marked_copy)[i] = m;
            } else {
                for (uint32_t k = 0; k < 16u && 16u * i + k < lim; ++k)
                    marked_copy[16u * i + k] = (uint8_t) (w[k >> 2] >> (8u * (k & 3u)));
            }
        }
    }
#pragma unroll
    for (int dlt = 16; dlt > 0; dlt >>= 1) local += __shfl_xor_sync(0xFFFFFFFFu, local, dlt);
    if (lane_id() == 0 && local) atomicAdd(&counters[C_PAIRS], local);
}

// Source-node range of `rank`: nodes are split so that every rank owns about the same number of edges
// (begin(r) = first node whose row starts at or after E * r / world).
__global__ void k_node_range(const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ n_nodes_ptr,
                             const uint32_t* __restrict__ n_edges_ptr, uint32_t rank, uint32_t world, uint32_t* __restrict__ out) {
    if (threadIdx.x >= 2) return;
    const uint32_t n_nodes = *n_nodes_ptr;
    const unsigned long long E = *n_edges_ptr;
    const uint32_t r = rank + threadIdx.x;   // thread 0: begin(rank), thread 1: begin(rank + 1)
    uint32_t result = n_nodes;
    if (r == 0) result = 0;
    else if (r < world) {
        const uint32_t target = (uint32_t) (E * r / world);
        uint32_t lo = 0, hi = n_nodes;   // first node with row_ptr[node] >= target
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (row_ptr[mid] < target) lo = mid + 1; else hi = mid;
        }
        result = lo;
    }
    out[threadIdx.x] = result;
}

void launch_node_range(Launch& L, GraphArrays g, const uint32_t* counters, uint32_t rank, uint32_t world, uint32_t* out) {
    k_node_range<<<1, 32, 0, L.stream>>>(g.row_ptr, counters + C_NODES, counters + C_EDGES, rank, world, out);
    L.count++;
}

void launch_transitive(Launch& L, GraphArrays g, uint32_t n_nodes_max, HeavyItems heavy, uint32_t* work_counter, uint32_t* counters,
                       const uint32_t* node_range) {
    const int blocks = grid_for(n_nodes_max, 32 * kLightWarps, kNumSMs * 8);
    // the group and the light kernel take disjoint sets of nodes (by out-degree) and only meet in atomics (heavy work
    // list, visit counter): the light one (14 us, mostly idle SMs) runs beside the group one on a forked stream
    const bool forked = fork_side(L, 1);
    k_transitive_group<<<blocks, kLightWarps * 32, 0, L.stream>>>(g.row_ptr, g.col, g.col_eid, g.T, node_range, counters + C_NODES,
                                                                 work_counter + 1, heavy, counters);
    L.count++;
    k_transitive_light<<<blocks, kLightWarps * 32, 0, forked ? L.side[1] : L.stream>>>(
        g.row_ptr, g.col, g.col_eid, g.T, node_range, counters + C_NODES, work_counter, heavy, counters);
    L.count++;
    if (forked) join_side(L, 1);
    k_transitive_heavy<<<kNumSMs * 4, kHeavyThreads, 0, L.stream>>>(g.row_ptr, g.col, g.col_eid, g.T, heavy, counters);
    L.count++;
}

void launch_finalize_marks(Launch& L, GraphArrays g, uint32_t edge_cap, uint32_t* counters, uint8_t* marked_copy, uint32_t copy_cap) {
    uint64_t blocks = (edge_cap / 16 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > (uint64_t) kNumSMs * 8) blocks = kNumSMs * 8;
    k_finalize_marks<<<(int) blocks, 256, 0, L.stream>>>(g.T, g.marked, counters + C_EDGES, edge_cap, counters, marked_copy, copy_cap);
    L.count++;
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_transitive() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_transitive_group);
    cudaFuncGetAttributes(&a, k_transitive_light);
    cudaFuncGetAttributes(&a, k_transitive_heavy);
    cudaFuncGetAttributes(&a, k_finalize_marks);
    cudaFuncGetAttributes(&a, k_node_range);
}

}  // namespace rb
