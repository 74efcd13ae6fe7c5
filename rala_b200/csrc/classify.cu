// classify.cu — K1 / K1b / K1c: overlap trimming + classification, ordered containment as a
// death-time fixed point, chimeric-hill counters, and the ordered list compactions between them.
//
// Replaces (reference file:line): Overlap::trim / Overlap::type overlap.cpp:117-259 as driven by
// graph.cpp:443-518 (classify loop), 722-736 and 801-824 (re-trim, promotion of internals),
// 831-877 (final containment), and Pile::check_chimeric_hills pile.cpp:457-469.
#include <cstdlib>

#include "kernels.h"
#include "lists.cuh"

namespace rb {

// =============================================================================================
// K1 (graph.cpp:443-518) runs as two streaming kernels over the device-resident records, with the
// containment resolution between them:
//   k_classify_events    every record: static gates, trim, type; emits only what the ORDER-DEPENDENT
//                        part needs: the containment events (victim, container, time) of kA/kB records
//                        and the indices of records touching a pile with chimeric hills.
//   k_classify_survivors every record again, once the final pile liveness is known: records whose two
//                        piles are still alive are trimmed, typed and written, in FILE ORDER, to
//                        `overlaps` (kA/kB with a chimeric container, kAB, kBA) or `internals` (kX).
// No intermediate list: on clean data ~95 % of the records are dovetails at classification time but
// only ~7 % survive the dead-pile filter, so materialising the "potential survivors" costs more than
// re-reading the records.
//
// Layout in HBM: the 28-byte rala_ovl_t rows the host marshals are transposed ONCE, at upload
// (k_records_to_soa), into six 4-byte columns (a | invalid << 31, b | orientation << 31, a_begin, a_end,
// b_begin, b_end: 24 B / record).  Each thread owns 4 consecutive records and reads every column with
// one 16-byte load, so a warp touches 512 contiguous bytes per column: fully coalesced, no staging, no
// barriers in the first pass.  The second pass reads only the two id columns (8 B / record) plus one
// bit per pile of an L1-resident liveness bitmap, and gathers the coordinates of the few survivors.
// =============================================================================================
constexpr int kEventsItems = 4;                           // consecutive records per thread in k_classify_events (one 16-byte load per column)
constexpr int kEventsMinBlocks = 3;                       // its resident blocks per SM
constexpr int kRecItems = 4;                              // consecutive records per thread (one uint4 per column)
constexpr int kRecTile = kTileThreads * kRecItems;        // records per block iteration
constexpr uint32_t kRunRecords = 512;                     // survivors pass: records per warp iteration = one run
constexpr int kRunGroups = kRunRecords / 128;             // 128-record groups per run (one 16-byte load per column, lane and group)

__global__ void k_records_to_soa(const uint32_t* __restrict__ aos, uint32_t n, List recs) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t* q = aos + (size_t) i * 7;
        const uint32_t flags = q[6];
        // ids beyond 2^31 cannot name a pile (rala_b200.h limits): such a record is invalid
        const bool bad = (flags & 2u) || (q[0] & kInvalidBit) || (q[1] & kInvalidBit);
        recs.a[i] = (q[0] & ~kInvalidBit) | (bad ? kInvalidBit : 0u);
        recs.b[i] = (q[1] & ~kInvalidBit) | ((flags & 1u) << 31);
        recs.ab[i] = q[2];
        recs.ae[i] = q[3];
        recs.bb[i] = q[4];
        recs.be[i] = q[5];
    }
}

// compact upload -> columns (rala_b200_graph_set_overlaps_packed): four records per thread; the query id comes from the
// group table (one binary search per thread, then a short walk), the coordinates from two 16 + 16 bit words
__global__ void __launch_bounds__(256) k_unpack_records(const uint32_t* __restrict__ query_id, const uint32_t* __restrict__ group_end,
                                                       uint32_t n_groups, const uint32_t* __restrict__ a_span,
                                                       const uint32_t* __restrict__ b_span, uint32_t n, List recs) {
    const uint32_t n4 = (n + 3u) / 4u;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += gridDim.x * blockDim.x) {
        const uint32_t i0 = 4u * q;
        uint32_t lo = 0, hi = n_groups;   // first group whose end lies behind record i0
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(group_end + mid) <= i0) lo = mid + 1; else hi = mid;
        }
        uint32_t k = lo, end = k < n_groups ? __ldg(group_end + k) : 0xFFFFFFFFu;
        const uint4 sa = reinterpret_cast<const uint4*>(a_span)[q], sb = reinterpret_cast<const uint4*>(b_span)[q];
        const uint32_t wa[4] = {sa.x, sa.y, sa.z, sa.w}, wb[4] = {sb.x, sb.y, sb.z, sb.w};
        uint32_t a[4], ab[4], ae[4], bb[4], be[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            while (i0 + r >= end && k + 1 < n_groups) {
                ++k;
                end = __ldg(group_end + k);
            }
            const bool have = i0 + r < n && k < n_groups && i0 + r < end;
            a[r] = have ? (__ldg(query_id + k) & ~kInvalidBit) : kInvalidBit;   // records behind the last group do not exist
            ab[r] = wa[r] & 0xFFFFu; ae[r] = wa[r] >> 16;
            bb[r] = wb[r] & 0xFFFFu; be[r] = wb[r] >> 16;
        }
        reinterpret_cast<uint4*>(recs.a)[q] = make_uint4(a[0], a[1], a[2], a[3]);
        reinterpret_cast<uint4*>(recs.ab)[q] = make_uint4(ab[0], ab[1], ab[2], ab[3]);
        reinterpret_cast<uint4*>(recs.ae)[q] = make_uint4(ae[0], ae[1], ae[2], ae[3]);
        reinterpret_cast<uint4*>(recs.bb)[q] = make_uint4(bb[0], bb[1], bb[2], bb[3]);
        reinterpret_cast<uint4*>(recs.be)[q] = make_uint4(be[0], be[1], be[2], be[3]);
    }
}

__device__ __forceinline__ void unpack4(const uint4 v, uint32_t (&out)[4]) {
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
}

// R consecutive values of a column, one 16- or 8-byte load (q counts groups of R values)
__device__ __forceinline__ void load_group(const uint32_t* __restrict__ col, uint32_t q, uint32_t (&out)[4]) {
    unpack4(reinterpret_cast<const uint4*>(col)[q], out);
}
__device__ __forceinline__ void load_group(const uint32_t* __restrict__ col, uint32_t q, uint32_t (&out)[2]) {
    const uint2 v = reinterpret_cast<const uint2*>(col)[q];
    out[0] = v.x; out[1] = v.y;
}

constexpr int kEvStage = 96;   // per-warp staging of events before one aggregated global append

// Tried and measured (profiles/r02ac_ab.json): staging the record tiles in shared memory with bulk copies (cp.async.bulk +
// mbarrier, 2 .. 4 tiles deep) made this kernel SLOWER, 126 .. 172 us against 109 us: it is bound by the integer ALU pipe
// (65 % of its peak at 57 % issue activity, profiles/r02v), not by load latency, and the block-wide hand-over of a stage
// keeps the eight warps of a block in step.  A software prefetch of the next trip's lines into L2 changed nothing; two
// records per thread at 4 .. 6 blocks per SM lost 6 .. 15 us (profiles/r02aa_ab.json).
template <int MINB, int R>
__global__ void __launch_bounds__(kTileThreads, MINB) k_classify_events(
    List recs, uint32_t n, uint32_t t0, const uint2* __restrict__ piles, uint32_t n_piles,
    Events ev, uint32_t ev_cap, unsigned long long* __restrict__ first, uint32_t* __restrict__ hill_rec, uint32_t hill_cap,
    uint32_t* __restrict__ counters) {
    __shared__ uint32_t s_ev[kTileWarps][3][kEvStage];
    const uint32_t lane = lane_id(), warp = warp_id();
    const uint32_t n4 = (n + R - 1u) / R;   // groups of R records
    uint32_t staged = 0;   // warp-uniform

    auto flush = [&]() {
        uint32_t gbase = 0;
        if (lane == 0) gbase = atomicAdd(&counters[C_EV], staged);
        gbase = __shfl_sync(0xFFFFFFFFu, gbase, 0);
        for (uint32_t i = lane; i < staged; i += 32) {
            if (gbase + i < ev_cap) {
                ev.v[gbase + i] = s_ev[warp][0][i];
                ev.c[gbase + i] = s_ev[warp][1][i];
                ev.t[gbase + i] = s_ev[warp][2][i];
            }
        }
        __syncwarp();
        staged = 0;
    };

    for (uint32_t qbase = blockIdx.x * kTileThreads; qbase < n4; qbase += gridDim.x * kTileThreads) {
        const uint32_t q = qbase + threadIdx.x;
        uint32_t a[R], b[R], ab[R], ae[R], bb[R], be[R];
        uint2 pa[R], pb[R];
        bool live[R];
        if (q < n4) {
            load_group(recs.a, q, a);
            load_group(recs.b, q, b);
            load_group(recs.ab, q, ab);
            load_group(recs.ae, q, ae);
            load_group(recs.bb, q, bb);
            load_group(recs.be, q, be);
        }
        // all eight pile gathers of the thread's records are in flight before the first one is used
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t idb = b[r] & 0x7FFFFFFFu;
            live[r] = q < n4 && (uint32_t) R * q + r < n && !(a[r] & kInvalidBit) && a[r] < n_piles && idb < n_piles;   // graph.cpp:450-451
            pa[r] = pb[r] = make_uint2(0u, 0u);   // a dead pile: rejects itself
            if (live[r]) {
                pa[r] = __ldg(piles + a[r]);
                pb[r] = __ldg(piles + idb);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            // straight-line trim + type (common.cuh event_code): a dead pile (end == 0) rejects itself
            const uint32_t idb = b[r] & 0x7FFFFFFFu;
            const uint32_t code = event_code(ab[r], ae[r], bb[r], be[r], b[r] >> 31, pa[r].x, pa[r].y & kEndMask,
                                             pb[r].x, pb[r].y & kEndMask);                              // :451-452
            const uint32_t fa = pa[r].y >> 30, fb = pb[r].y >> 30;
            if ((code & 1u) && ((fa | fb) & 1u)) {                                                      // :457-462, resolved by k_hill_coverage
                uint32_t slot = atomicAdd(&counters[C_HILL], 1u);
                if (slot < hill_cap) hill_rec[slot] = (uint32_t) R * q + r;
            }
            const bool ev_b = (code & 2u) && !(fb & 2u);                                                // :469-474
            const bool ev_a = (code & 4u) && !(fa & 2u);                                                // :475-480
            const bool is_ev = ev_a | ev_b;
            const uint32_t evv = ev_b ? a[r] : idb, evc = ev_b ? idb : a[r];
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, is_ev);
            if (m) {
                if (is_ev) {
                    const uint32_t t = t0 + (uint32_t) R * q + r;
                    atomicMin(&first[evv], ((unsigned long long) t << 32) | evc);   // the victim's earliest event (containment.cu)
                    const uint32_t p = staged + __popc(m & ((1u << lane) - 1u));
                    s_ev[warp][0][p] = evv;
                    s_ev[warp][1][p] = evc;
                    s_ev[warp][2][p] = t;
                }
                staged += __popc(m);
                __syncwarp();
                if (staged > kEvStage - 32) flush();
            }
        }
    }
    if (staged) flush();
}

// Survivors pass.  Every warp takes RUNS of 512 consecutive records (4 x 4 per lane) from an atomic ticket, so a run only
// ever waits on runs whose warps are resident or finished.  The survivors of a run go straight to their file-order
// places in `overlaps` and `internals`: the run publishes its two counts as its aggregate and takes its exclusive prefix
// with the decoupled look-back (one status word per run); the last run writes both list lengths.
//
// Only ~7 % of the records have two live piles, so the pass is split in phases per run:
//   1. liveness: 16 records per lane, both id columns as 16-byte loads, 32 bitmap gathers in flight per lane;
//      the candidates' positions inside the run are COMPACTED into a per-warp queue in shared memory (one packed
//      warp scan ranks all four 128-record groups at once: one byte per group, each <= 128);
//   2. trim + type run over the queue with (almost) every lane busy, instead of sixteen times over mostly idle
//      warps (the first version of this kernel executed 12 of 32 lanes per instruction, profiles/r01f); the type goes
//      back into the queue entry beside the position, and the run's counts are published;
//   3. the run's prefix is awaited only after phases 1 and 2 of the warp's NEXT run (two queues per warp), when the
//      runs before it have long published theirs; then the survivors' coordinates are gathered again (L2 hits), trimmed
//      again and written.
// This replaced scratch slots per run plus a scan and a relocation kernel (one 32-byte write and read per survivor, two
// launches).  Waiting for the prefix right after phase 2 instead keeps thousands of resident warps spinning on a
// straggler: that fusion once cost +39 us (profiles/r02w_ab.json); see profiles/r02ap_* for this one.
// 5 resident blocks per SM and a grid of two waves: survivors stage 83 us against 91 us at 4 resident blocks (64 registers);
// one persistent wave loses 15 us, 6 resident blocks spill 104 bytes and win nothing (profiles/r02ae_ab.json, r02af_ab.json)
constexpr int kSurvMinBlocks = 5;
constexpr int kSurvBlocks = 10;   // grid = this many blocks per SM at most
constexpr uint32_t kQueueTagShift = 9;   // queue entry: position in the run (9 bits) | type << 9 (kQueueRejected: no survivor)
constexpr uint32_t kQueueRejected = 7;
static_assert(kRunRecords <= (1u << kQueueTagShift) && kBA < kQueueRejected, "a queue entry holds a run position and a type");

// phases 1 and 2 of `run`: the queue holds the candidates' positions and types; returns their number and the run's counts
__device__ __forceinline__ uint32_t survivors_queue(const List& recs, uint32_t n, const uint2* __restrict__ piles,
                                                    const uint32_t* __restrict__ alive_bits, uint32_t n_piles, uint32_t run,
                                                    uint16_t* queue, uint32_t& n_a, uint32_t& n_b) {
    const uint32_t lane = lane_id();
    uint32_t a[kRunGroups][4], b[kRunGroups][4];
#pragma unroll
    for (int j = 0; j < kRunGroups; ++j) {
        const uint32_t q = run * (kRunRecords / 4) + j * 32u + lane;     // this lane's j-th group of 4 records
#pragma unroll
        for (int r = 0; r < 4; ++r) { a[j][r] = kInvalidBit; b[j][r] = 0u; }
        if (4u * q < n) {
            unpack4(reinterpret_cast<const uint4*>(recs.a)[q], a[j]);
            unpack4(reinterpret_cast<const uint4*>(recs.b)[q], b[j]);
        }
    }
    uint32_t cand = 0;   // bit j * 4 + r
#pragma unroll
    for (int j = 0; j < kRunGroups; ++j) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {   // both piles alive at the end (graph.cpp:493-515)?  one L1-resident bit each
            const uint32_t i = run * kRunRecords + j * 128u + 4u * lane + r, ida = a[j][r], idb = b[j][r] & 0x7FFFFFFFu;
            const bool ok = i < n && !(ida & kInvalidBit) && ida < n_piles && idb < n_piles &&
                            ((__ldg(alive_bits + (ida >> 5)) >> (ida & 31u)) & 1u) && ((__ldg(alive_bits + (idb >> 5)) >> (idb & 31u)) & 1u);
            cand |= ok ? 1u << (j * 4 + r) : 0u;
        }
    }
    // rank of every candidate in record order (group-major, then lane, then r)
    uint32_t packed = 0;
#pragma unroll
    for (int j = 0; j < kRunGroups; ++j) packed |= (uint32_t) __popc((cand >> (4 * j)) & 0xFu) << (8 * j);
    const uint32_t inc = warp_inclusive_scan(packed);
    const uint32_t tot = __shfl_sync(0xFFFFFFFFu, inc, 31);
    uint32_t group_base = 0;
#pragma unroll
    for (int j = 0; j < kRunGroups; ++j) {
        uint32_t p = group_base + (((inc - packed) >> (8 * j)) & 0xFFu);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if ((cand >> (j * 4 + r)) & 1u) queue[p++] = (uint16_t) (j * 128u + 4u * lane + r);
        }
        group_base += (tot >> (8 * j)) & 0xFFu;
    }
    const uint32_t total = group_base;
    __syncwarp();
    n_a = 0;
    n_b = 0;
    for (uint32_t k0 = 0; k0 < total; k0 += 32) {
        const uint32_t k = k0 + lane;
        uint8_t tag = kRejected;
        if (k < total) {   // only now fetch the coordinates and the two piles
            Entry e = load_entry(recs, run * kRunRecords + queue[k]);
            const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
            if (trim(e.c, e.ori, pa, pb)) tag = classify(e.c, relative(e.c, e.ori, pa, pb));   // a surviving kA/kB has a chimeric container (:470, :476)
            queue[k] |= (uint16_t) ((tag == kRejected ? kQueueRejected : (uint32_t) tag) << kQueueTagShift);
        }
        n_a += __popc(__ballot_sync(0xFFFFFFFFu, tag != kRejected && tag != kX));
        n_b += __popc(__ballot_sync(0xFFFFFFFFu, tag == kX));
    }
    __syncwarp();   // the types in the queue are visible to every lane
    return total;
}

// phase 3 of `run`: its survivors to their places behind the exclusive prefix `excl`
__device__ __forceinline__ void survivors_write(const List& recs, const uint2* __restrict__ piles, uint32_t run, const uint16_t* queue,
                                                uint32_t total, unsigned long long excl, const List& ovl, const List& inl, uint32_t cap) {
    const uint32_t lane = lane_id();
    uint32_t pos_a = count_a(excl), pos_b = count_b(excl);
    for (uint32_t k0 = 0; k0 < total; k0 += 32) {
        const uint32_t k = k0 + lane;
        const uint32_t qe = k < total ? queue[k] : kQueueRejected << kQueueTagShift;
        const uint8_t tag = (uint8_t) (qe >> kQueueTagShift);
        const int dest = tag == kQueueRejected ? 0 : tag == kX ? 2 : 1;
        const uint32_t ma = __ballot_sync(0xFFFFFFFFu, dest == 1), mb = __ballot_sync(0xFFFFFFFFu, dest == 2);
        const uint32_t below = (1u << lane) - 1u;
        const uint32_t p = dest == 1 ? pos_a + __popc(ma & below) : pos_b + __popc(mb & below);
        if (dest && p < cap) {
            Entry e = load_entry(recs, run * kRunRecords + (qe & ((1u << kQueueTagShift) - 1u)));
            const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
            trim(e.c, e.ori, pa, pb);
            store_entry(dest == 1 ? ovl : inl, p, e, tag);
        }
        pos_a += __popc(ma);
        pos_b += __popc(mb);
    }
}

__global__ void __launch_bounds__(kTileThreads, kSurvMinBlocks) k_classify_survivors(
    List recs, uint32_t n, const uint2* __restrict__ piles, const uint32_t* __restrict__ alive_bits, uint32_t n_piles,
    List ovl, uint32_t* __restrict__ n_ovl, List inl, uint32_t* __restrict__ n_inl, uint32_t cap,
    unsigned long long* __restrict__ status, uint32_t* __restrict__ ticket) {
    __shared__ uint16_t s_queue[kTileWarps][2][kRunRecords];
    const uint32_t lane = lane_id(), warp = warp_id();
    const uint32_t num_runs = (n + kRunRecords - 1) / kRunRecords;
    uint32_t cur = 0, prev_run = 0xFFFFFFFFu, prev_total = 0;   // warp-uniform; prev_run: the run awaiting its prefix
    unsigned long long prev_agg = 0;
    while (true) {
        uint32_t run = 0;
        if (lane == 0) run = atomicAdd(ticket, 1u);
        run = __shfl_sync(0xFFFFFFFFu, run, 0);
        uint32_t total = 0;
        unsigned long long agg = 0;
        if (run < num_runs) {
            uint32_t n_a, n_b;
            total = survivors_queue(recs, n, piles, alive_bits, n_piles, run, s_queue[warp][cur], n_a, n_b);
            agg = pack_counts(n_a, n_b);
            lookback_publish(status, run, agg);
        }
        if (prev_run != 0xFFFFFFFFu) {
            const unsigned long long excl = lookback_wait(status, prev_run, prev_agg);
            if (prev_run == num_runs - 1 && lane == 0) {
                *n_ovl = count_a(excl + prev_agg);
                *n_inl = count_b(excl + prev_agg);
            }
            survivors_write(recs, piles, prev_run, s_queue[warp][cur ^ 1], prev_total, excl, ovl, inl, cap);
            __syncwarp();   // that queue is refilled by the next run
        }
        if (run >= num_runs) break;
        prev_run = run;
        prev_total = total;
        prev_agg = agg;
        cur ^= 1;
    }
}

// K1c: Pile::check_chimeric_hills (pile.cpp:457-469) for every PROCESSED record that touches a pile
// with hills.  Processed = passed the static gates and both piles were still alive at its time.
__global__ void k_hill_coverage(List recs, uint32_t t0, const uint2* __restrict__ piles,
                                const uint32_t* __restrict__ hill_rec, uint32_t hill_cap,
                                const uint32_t* __restrict__ hill_pile, const uint32_t* __restrict__ hill_begin,
                                const uint32_t* __restrict__ hill_end, uint32_t n_hills, uint32_t* __restrict__ hill_cov,
                                const uint32_t* __restrict__ D, const uint32_t* __restrict__ counters) {
    const uint32_t n = min(counters[C_HILL], hill_cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t idx = hill_rec[i];
        Entry e = load_entry(recs, idx);   // the record passed the static gates: the invalid bit of column a is clear
        const uint32_t t = t0 + idx;
        if (D[e.a] < t || D[e.b] < t) continue;   // a pile was already dead: transmute() rejected it (overlap.cpp:51,70)
        const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
        trim(e.c, e.ori, pa, pb);
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const Pile& p = side ? pb : pa;
            if (!(p.flags & 1u)) continue;
            const uint32_t id = side ? e.b : e.a;
            // begin_ added to absolute coordinates, as in :459-462; the pile takes the b side only when it is not also the
            // a pile (it compares the overlap's a id with its own), so a self overlap counts its a-side span twice
            const bool b_side = side && e.a != e.b;
            const uint32_t lo = p.begin + (b_side ? e.c.bb : e.c.ab);
            const uint32_t hi = p.begin + (b_side ? e.c.be : e.c.ae);
            uint32_t l = 0, h = n_hills;
            while (l < h) {
                uint32_t m = (l + h) >> 1;
                if (hill_pile[m] < id) l = m + 1; else h = m;
            }
            for (uint32_t k = l; k < n_hills && hill_pile[k] == id; ++k) {
                if (lo < hill_begin[k] && hi > hill_end[k]) atomicAdd(&hill_cov[k], 1u);
            }
        }
    }
}

// Piles with a finite death time die (piles_[x].reset(), graph.cpp:471,477,838,842).
// Also refreshes the one-bit-per-pile liveness bitmap the survivors pass tests first.
// DECODE: dbuf still holds the resolution's state words (containment.cu: settled bit | death time, 0x7FFFFFFF = never);
// they are turned into death times (kInf = never) on the way, which saves the separate k_decode_state launch.
// reset (first pass only, also when the pass is skipped): nothing reads the first pass's earliest events or event count
// any more, so this sweep clears them for the final pass and keeps the first pass's event and round counts.
template <bool DECODE>
__global__ void k_apply_deaths(uint2* __restrict__ piles, uint32_t* __restrict__ D, uint32_t n_piles, uint32_t* __restrict__ alive_bits,
                               const uint32_t* __restrict__ skip, const uint32_t* __restrict__ run_if, FinalPassReset reset) {
    if (reset.counters) {
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < reset.n_first; i += gridDim.x * blockDim.x) reset.first[i] = ~0ull;
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            uint32_t* c = reset.counters;
            c[C_EV_FIRST] = c[C_EV];
            c[C_ROUNDS_FIRST] = c[C_ROUNDS];
            c[C_EV] = 0u;
        }
    }
    if ((skip && *skip) || (run_if && *run_if == 0u)) return;
    for (uint32_t base = blockIdx.x * blockDim.x; base < n_piles; base += gridDim.x * blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        bool alive = false;
        if (i < n_piles) {
            uint32_t d = D[i];
            if (DECODE) {
                d &= 0x7FFFFFFFu;
                d = d == 0x7FFFFFFFu ? kInf : d;
                D[i] = d;
            }
            if (d != kInf) piles[i] = make_uint2(0u, 0u);
            else alive = (piles[i].y & kEndMask) != 0u;
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, alive);
        if (lane_id() == 0 && i < n_piles) alive_bits[i >> 5] = m;
    }
}

// n words of p set to v by the whole grid, 16 bytes per store where p allows
__device__ __forceinline__ void fill_words(uint32_t* p, size_t n, uint32_t v, size_t tid, size_t threads) {
    size_t head = ((16u - ((uintptr_t) p & 15u)) & 15u) / 4u;
    head = head < n ? head : n;
    const size_t n4 = (n - head) / 4;
    uint4* q = reinterpret_cast<uint4*>(p + head);
    for (size_t i = tid; i < head; i += threads) p[i] = v;
    for (size_t i = tid; i < n4; i += threads) q[i] = make_uint4(v, v, v, v);
    for (size_t i = head + 4 * n4 + tid; i < n; i += threads) p[i] = v;
}

// The clears and the copy a step starts from, in one launch (StepPrologue).
__global__ void __launch_bounds__(256) k_step_prologue(StepPrologue p) {
    const size_t tid = (size_t) blockIdx.x * blockDim.x + threadIdx.x, threads = (size_t) gridDim.x * blockDim.x;
    const uint4* src = reinterpret_cast<const uint4*>(p.snapshot ? p.piles : p.piles_initial);   // 256-byte aligned tables
    uint4* dst = reinterpret_cast<uint4*>(p.snapshot ? p.piles_initial : p.piles);
    for (size_t i = tid; i < p.n_piles / 2; i += threads) dst[i] = src[i];
    if (tid == 0 && (p.n_piles & 1u)) {
        const uint2* s2 = reinterpret_cast<const uint2*>(src);
        reinterpret_cast<uint2*>(dst)[p.n_piles - 1] = s2[p.n_piles - 1];
    }
    fill_words(reinterpret_cast<uint32_t*>(p.first), 2 * (size_t) p.n_first, ~0u, tid, threads);
    for (int k = 0; k < StepPrologue::kZero; ++k)
        if (p.zero[k]) fill_words(p.zero[k], p.zero_words[k], 0u, tid, threads);
}

// =============================================================================================
// Ordered list passes.  MODE selects what happens to an entry:
//   kRetrim       list -> list, dropping entries trim() rejects                          :722-736, 801-807
//   kPromote      internals -> internals / appended to overlaps when now a dovetail      :809-824
//   kFinalOvl     overlaps -> overlaps, keeping entries with both piles alive and not kA/kB  :831-848, 869-877
//   kFinalInt     internals -> internals (alive at their own time, not kA/kB)            :849-867
// =============================================================================================
enum ListMode { kRetrim = 1, kPromote = 2, kFinalOvl = 3, kFinalInt = 4 };

// 4 blocks per SM (64 registers): unbounded, ptxas gives kFinalInt 79 registers and kRetrim / kFinalOvl a small spill
template <int MODE>
__global__ void __launch_bounds__(kTileThreads, 4) k_list_pass(
    List in, const uint32_t* __restrict__ n_in_ptr, uint32_t in_cap, const uint2* __restrict__ piles,
    List out_a, uint32_t* __restrict__ n_out_a, List out_b, uint32_t* __restrict__ n_out_b,
    const uint32_t* __restrict__ b_base_ptr, uint32_t cap, const uint32_t* __restrict__ D, const uint32_t* __restrict__ time_base_ptr,
    unsigned long long* __restrict__ status, uint32_t* __restrict__ ticket) {
    __shared__ TileShared sh;
    const uint32_t tid = threadIdx.x;
    const uint32_t n = min(*n_in_ptr, in_cap);
    const uint32_t num_tiles = (n + kTile - 1) / kTile;
    // kPromote appends behind the current end of `overlaps` (count in a slot this kernel never writes)
    const uint32_t b_off = b_base_ptr ? *b_base_ptr : 0u;
    const uint32_t time_base = time_base_ptr ? *time_base_ptr : 0u;
    __syncthreads();

    while (true) {
        if (tid == 0) sh.tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = sh.tile;
        if (tile >= num_tiles) break;
        const uint32_t base = tile * kTile;

        Entry e[kTileItems];
        uint8_t tag[kTileItems];
        int dest[kTileItems];
#pragma unroll
        for (int r = 0; r < kTileItems; ++r) {
            const uint32_t idx = base + r * kTileThreads + tid;
            dest[r] = 0;
            tag[r] = kRejected;
            if (idx < n) {
                e[r] = load_entry(in, idx);
                tag[r] = in.tag[idx];
                const Pile pa = load_pile(piles, e[r].a), pb = load_pile(piles, e[r].b);
                if (MODE == kRetrim) {
                    if (pa.alive() && pb.alive() && trim(e[r].c, e[r].ori, pa, pb)) dest[r] = 1;
                } else if (MODE == kPromote) {
                    if (pa.alive() && pb.alive() && trim(e[r].c, e[r].ori, pa, pb)) {
                        tag[r] = classify(e[r].c, relative(e[r].c, e[r].ori, pa, pb));
                        dest[r] = (tag[r] == kAB || tag[r] == kBA) ? 2 : 1;
                    }
                } else if (MODE == kFinalOvl) {
                    if (pa.alive() && pb.alive() && tag[r] != kA && tag[r] != kB) dest[r] = 1;
                } else {   // kFinalInt: alive before the pass (alive now, or killed by it) and still alive at its own time
                    const uint32_t t = time_base + idx;
                    const uint32_t da = D[e[r].a], db = D[e[r].b];
                    if ((pa.alive() || da != kInf) && (pb.alive() || db != kInf) && da > t && db > t && tag[r] != kA &&
                        tag[r] != kB)
                        dest[r] = 1;
                }
            }
        }
        uint32_t pos[kTileItems];
        unsigned long long inclusive = 0;
        tile_rank<kTileItems>(sh, status, tile, dest, pos, &inclusive);
        if (tid == 0 && tile == num_tiles - 1) {
            *n_out_a = count_a(inclusive);
            if (n_out_b) *n_out_b = b_off + count_b(inclusive);
        }
#pragma unroll
        for (int r = 0; r < kTileItems; ++r) {
            if (dest[r] == 1 && pos[r] < cap) store_entry(out_a, pos[r], e[r], tag[r]);
            if (dest[r] == 2 && b_off + pos[r] < cap) store_entry(out_b, b_off + pos[r], e[r], tag[r]);
        }
        __syncthreads();
    }
}

// Final containment, classification half (graph.cpp:831-866): type of every entry of `overlaps`
// then `internals` against the final pile table; kA/kB become events with time = position in the
// concatenation.  No chimeric gating in this pass.
// blockIdx.y selects the list: 0 = `overlaps`, 1 = `internals` (one launch for both: the second list is tiny on clean data).
__global__ void k_classify_final(List lst0, const uint32_t* __restrict__ n_ptr0, const uint32_t* __restrict__ time_base_ptr0,
                                 List lst1, const uint32_t* __restrict__ n_ptr1, const uint32_t* __restrict__ time_base_ptr1,
                                 uint32_t cap, const uint2* __restrict__ piles, Events ev,
                                 uint32_t ev_cap, unsigned long long* __restrict__ first, uint32_t* __restrict__ counters) {
    const List lst = blockIdx.y ? lst1 : lst0;
    const uint32_t* n_ptr = blockIdx.y ? n_ptr1 : n_ptr0;
    const uint32_t* time_base_ptr = blockIdx.y ? time_base_ptr1 : time_base_ptr0;
    const uint32_t n = min(*n_ptr, cap);
    const uint32_t time_base = time_base_ptr ? *time_base_ptr : 0u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Entry e = load_entry(lst, i);
        const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
        uint8_t t = kRejected;
        if (pa.alive() && pb.alive()) {
            t = classify(e.c, relative(e.c, e.ori, pa, pb));
            if (t == kA || t == kB) {
                // warp-aggregated append
                uint32_t m = __activemask();
                m = __match_any_sync(m, 1);
                uint32_t leader = __ffs(m) - 1, rank = __popc(m & ((1u << lane_id()) - 1u));
                uint32_t gbase = 0;
                if (lane_id() == leader) gbase = atomicAdd(&counters[C_EV], (uint32_t) __popc(m));
                gbase = __shfl_sync(m, gbase, leader);
                uint32_t p = gbase + rank;
                const uint32_t v = t == kA ? e.b : e.a, c = t == kA ? e.a : e.b;
                if (p < ev_cap) {
                    ev.v[p] = v;
                    ev.c[p] = c;
                    ev.t[p] = time_base + i;
                }
                atomicMin(&first[v], ((unsigned long long) (time_base + i) << 32) | c);
            }
        }
        lst.tag[i] = t;
    }
}

// Stateless unit stage: trim + type for n independent records (C ABI rala_b200_trim_classify).
__global__ void k_trim_classify_aos(uint32_t* __restrict__ rec, uint32_t n, const uint2* __restrict__ piles,
                                    uint32_t n_piles, uint8_t* __restrict__ type_out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t* q = rec + (size_t) i * 7;
        Entry e;
        e.a = q[0]; e.b = q[1]; e.c.ab = q[2]; e.c.ae = q[3]; e.c.bb = q[4]; e.c.be = q[5]; e.ori = q[6] & 1u;
        uint8_t t = kRejected;
        if (!(q[6] & 2u) && e.a < n_piles && e.b < n_piles) {
            const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
            if (pa.alive() && pb.alive() && trim(e.c, e.ori, pa, pb)) {
                t = classify(e.c, relative(e.c, e.ori, pa, pb));
                q[2] = e.c.ab; q[3] = e.c.ae; q[4] = e.c.bb; q[5] = e.c.be;
            }
        }
        type_out[i] = t;
    }
}

// host table {begin,end} + flag bytes -> packed device table
__global__ void k_pack_piles(const uint2* __restrict__ in, const uint8_t* __restrict__ flags, uint2* __restrict__ out,
                             uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 v = in[i];
        uint32_t f = flags ? (flags[i] & 3u) : 0u;
        out[i] = v.y == 0u ? make_uint2(0u, 0u) : make_uint2(v.x, (v.y & kEndMask) | (f << 30));
    }
}

__global__ void k_unpack_piles(const uint2* __restrict__ in, uint2* __restrict__ out, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint2 v = in[i];
        out[i] = make_uint2(v.x, v.y & kEndMask);
    }
}

// SoA list -> rala_ovl_t rows (download path)
__global__ void k_list_to_aos(List l, const uint32_t* __restrict__ n_ptr, uint32_t cap, uint32_t* __restrict__ out) {
    const uint32_t n = min(*n_ptr, cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Entry e = load_entry(l, i);
        uint32_t* q = out + (size_t) i * 7;
        q[0] = e.a; q[1] = e.b; q[2] = e.c.ab; q[3] = e.c.ae; q[4] = e.c.bb; q[5] = e.c.be; q[6] = e.ori;
    }
}

// rala_ovl_t rows -> SoA list (upload of a host-filtered `overlaps`, C ABI rala_b200_graph_set_kept_overlaps).  Each entry
// is typed against the pile table as it stands, as edge creation does (graph.cpp:594, no trim): the build trusts the tag.
__global__ void k_aos_to_list(const uint32_t* __restrict__ aos, uint32_t n, const uint2* __restrict__ piles, uint32_t n_piles, List l) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t* q = aos + (size_t) i * 7;
        Entry e;
        e.a = q[0]; e.b = q[1] & 0x7FFFFFFFu; e.c.ab = q[2]; e.c.ae = q[3]; e.c.bb = q[4]; e.c.be = q[5]; e.ori = q[6] & 1u;
        uint8_t t = kRejected;
        if (e.a < n_piles && e.b < n_piles) {
            const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
            if (pa.alive() && pb.alive()) t = classify(e.c, relative(e.c, e.ori, pa, pb));
        }
        store_entry(l, i, e, t);
    }
}

__global__ void k_list_connections(List l, const uint32_t* __restrict__ n_ptr, uint32_t cap, uint32_t* __restrict__ out) {
    const uint32_t n = min(*n_ptr, cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        out[2 * (size_t) i] = l.a[i];
        out[2 * (size_t) i + 1] = l.b[i] & 0x7FFFFFFFu;
    }
}

// ---------------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------------
void launch_records_to_soa(Launch& L, const uint32_t* aos, uint32_t n, List recs) {
    if (n == 0) return;
    k_records_to_soa<<<grid_for(n, 256, kNumSMs * 8), 256, 0, L.stream>>>(aos, n, recs);
    L.count++;
}

void launch_unpack_records(Launch& L, const uint32_t* query_id, const uint32_t* group_end, uint32_t n_groups, const uint32_t* a_span,
                           const uint32_t* b_span, uint32_t n, List recs) {
    if (n == 0) return;
    k_unpack_records<<<grid_for((n + 3) / 4, 256, kNumSMs * 8), 256, 0, L.stream>>>(query_id, group_end, n_groups, a_span, b_span, n, recs);
    L.count++;
}

void launch_classify_events(Launch& L, List recs, uint32_t n, uint32_t t0, const uint2* piles, uint32_t n_piles,
                            Events ev, uint32_t ev_cap, unsigned long long* first, uint32_t* hill_rec, uint32_t hill_cap, uint32_t* counters) {
    if (n == 0) return;
    // 3 blocks / SM at 80 registers: 4 and 5 blocks (64 / 48 registers) lost 15 and 25 us per step (profiles/r02a_ab.json)
    k_classify_events<kEventsMinBlocks, kEventsItems><<<grid_for(n, kTileThreads * kEventsItems, kNumSMs * kEventsMinBlocks), kTileThreads, 0, L.stream>>>(recs, n, t0, piles, n_piles, ev, ev_cap, first,
                                                                                        hill_rec, hill_cap, counters);
    L.count++;
}

uint32_t classify_num_runs(uint32_t n) { return (n + kRunRecords - 1) / kRunRecords; }

void launch_classify_survivors(Launch& L, List recs, uint32_t n, const uint2* piles, const uint32_t* alive_bits, uint32_t n_piles,
                               List ovl, uint32_t* n_ovl, List inl, uint32_t* n_inl, uint32_t cap, unsigned long long* status,
                               uint32_t* ticket) {
    if (n == 0) return;   // n_ovl / n_inl were zeroed by the caller
    const uint32_t num_runs = classify_num_runs(n);
    k_classify_survivors<<<grid_for(num_runs, kTileWarps, kNumSMs * kSurvBlocks), kTileThreads, 0, L.stream>>>(
        recs, n, piles, alive_bits, n_piles, ovl, n_ovl, inl, n_inl, cap, status, ticket);
    L.count++;
}


void launch_hill_coverage(Launch& L, List recs, uint32_t t0, const uint2* piles, const uint32_t* hill_rec,
                          uint32_t hill_cap, const uint32_t* hill_pile, const uint32_t* hill_begin,
                          const uint32_t* hill_end, uint32_t n_hills, uint32_t* hill_cov, const uint32_t* dbuf,
                          const uint32_t* counters) {
    k_hill_coverage<<<kNumSMs * 2, 256, 0, L.stream>>>(recs, t0, piles, hill_rec, hill_cap, hill_pile, hill_begin, hill_end,
                                                       n_hills, hill_cov, dbuf, counters);
    L.count++;
}

void launch_apply_deaths(Launch& L, uint2* piles, uint32_t* dbuf, uint32_t n_piles, uint32_t* alive_bits, bool decode,
                         const uint32_t* skip, const uint32_t* run_if, FinalPassReset reset) {
    if (n_piles == 0 && !reset.counters) return;
    const int grid = grid_for(n_piles > reset.n_first ? n_piles : reset.n_first, 256, kNumSMs * 8);
    if (decode) k_apply_deaths<true><<<grid, 256, 0, L.stream>>>(piles, dbuf, n_piles, alive_bits, skip, run_if, reset);
    else k_apply_deaths<false><<<grid, 256, 0, L.stream>>>(piles, dbuf, n_piles, alive_bits, skip, run_if, reset);
    L.count++;
}

void launch_step_prologue(Launch& L, const StepPrologue& p) {
    k_step_prologue<<<kNumSMs * 4, 256, 0, L.stream>>>(p);
    L.count++;
}

void launch_list_pass(Launch& L, int mode, List in, const uint32_t* n_in, uint32_t in_cap, const uint2* piles, List out_a,
                      uint32_t* n_out_a, List out_b, uint32_t* n_out_b, const uint32_t* b_base, uint32_t cap, const uint32_t* dbuf,
                      const uint32_t* time_base, unsigned long long* status, uint32_t* ticket) {
    int grid = grid_for(in_cap, kTile, kNumSMs * 8);
#define RB_LP(M) k_list_pass<M><<<grid, kTileThreads, 0, L.stream>>>(in, n_in, in_cap, piles, out_a, n_out_a, out_b, \
        n_out_b, b_base, cap, dbuf, time_base, status, ticket)
    switch (mode) {
        case kRetrim: RB_LP(kRetrim); break;
        case kPromote: RB_LP(kPromote); break;
        case kFinalOvl: RB_LP(kFinalOvl); break;
        default: RB_LP(kFinalInt); break;
    }
#undef RB_LP
    L.count++;
}

void launch_classify_final(Launch& L, List ovl, const uint32_t* n_ovl, const uint32_t* ovl_time_base, List inl,
                           const uint32_t* n_inl, const uint32_t* inl_time_base, uint32_t cap, const uint2* piles, Events ev,
                           uint32_t ev_cap, unsigned long long* first, uint32_t* counters) {
    k_classify_final<<<dim3(grid_for(cap, 256, kNumSMs * 4), 2), 256, 0, L.stream>>>(ovl, n_ovl, ovl_time_base, inl, n_inl, inl_time_base,
                                                                                     cap, piles, ev, ev_cap, first, counters);
    L.count++;
}

void launch_trim_classify_aos(Launch& L, uint32_t* rec, uint32_t n, const uint2* piles, uint32_t n_piles, uint8_t* type_out) {
    if (n == 0) return;
    k_trim_classify_aos<<<grid_for(n, 256, kNumSMs * 8), 256, 0, L.stream>>>(rec, n, piles, n_piles, type_out);
    L.count++;
}

void launch_pack_piles(Launch& L, const uint2* in, const uint8_t* flags, uint2* out, uint32_t n) {
    if (n == 0) return;
    k_pack_piles<<<grid_for(n, 256, kNumSMs * 8), 256, 0, L.stream>>>(in, flags, out, n);
    L.count++;
}

void launch_unpack_piles(Launch& L, const uint2* in, uint2* out, uint32_t n) {
    if (n == 0) return;
    k_unpack_piles<<<grid_for(n, 256, kNumSMs * 8), 256, 0, L.stream>>>(in, out, n);
    L.count++;
}

void launch_list_to_aos(Launch& L, List l, const uint32_t* n_ptr, uint32_t cap, uint32_t* out) {
    k_list_to_aos<<<grid_for(cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(l, n_ptr, cap, out);
    L.count++;
}

void launch_aos_to_list(Launch& L, const uint32_t* aos, uint32_t n, const uint2* piles, uint32_t n_piles, List l) {
    if (n == 0) return;
    k_aos_to_list<<<grid_for(n, 256, kNumSMs * 8), 256, 0, L.stream>>>(aos, n, piles, n_piles, l);
    L.count++;
}

void launch_list_connections(Launch& L, List l, const uint32_t* n_ptr, uint32_t cap, uint32_t* out) {
    k_list_connections<<<grid_for(cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(l, n_ptr, cap, out);
    L.count++;
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_classify() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_records_to_soa);
    cudaFuncGetAttributes(&a, k_unpack_records);
    cudaFuncGetAttributes(&a, k_classify_events<kEventsMinBlocks, kEventsItems>);
    cudaFuncGetAttributes(&a, k_classify_survivors);
    cudaFuncGetAttributes(&a, k_hill_coverage);
    cudaFuncGetAttributes(&a, k_apply_deaths<true>);
    cudaFuncGetAttributes(&a, k_apply_deaths<false>);
    cudaFuncGetAttributes(&a, k_step_prologue);
    cudaFuncGetAttributes(&a, k_list_pass<kRetrim>);
    cudaFuncGetAttributes(&a, k_list_pass<kPromote>);
    cudaFuncGetAttributes(&a, k_list_pass<kFinalOvl>);
    cudaFuncGetAttributes(&a, k_list_pass<kFinalInt>);
    cudaFuncGetAttributes(&a, k_classify_final);
    cudaFuncGetAttributes(&a, k_trim_classify_aos);
    cudaFuncGetAttributes(&a, k_pack_piles);
    cudaFuncGetAttributes(&a, k_unpack_piles);
    cudaFuncGetAttributes(&a, k_list_to_aos);
    cudaFuncGetAttributes(&a, k_aos_to_list);
    cudaFuncGetAttributes(&a, k_list_connections);
}

}  // namespace rb
