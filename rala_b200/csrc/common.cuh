// common.cuh — device-side building blocks shared by the hot-path kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace rb {

constexpr uint32_t kInf = 0xFFFFFFFFu;         // "never dies" death time
constexpr uint32_t kEndMask = 0x3FFFFFFFu;     // pile.y = end | flags << 30
constexpr uint32_t kInvalidBit = 0x80000000u;  // in the a_id column of the device records: is_valid_overlap_ false / transmute failed
constexpr int kNumSMs = 148;

enum : uint8_t { kX = 0, kA = 1, kB = 2, kAB = 3, kBA = 4, kRejected = 255 };

// ---------------------------------------------------------------------------------------------
// Pile table entry as stored on the device: x = begin, y = end | flags << 30 (end == 0: dead pile).
// ---------------------------------------------------------------------------------------------
struct Pile {
    uint32_t begin, end, flags;
    __host__ __device__ __forceinline__ bool alive() const { return end != 0; }
};

__device__ __forceinline__ Pile load_pile(const uint2* __restrict__ piles, uint32_t id) {
    uint2 v = __ldg(piles + id);
    Pile p;
    p.begin = v.x;
    p.end = v.y & kEndMask;
    p.flags = v.y >> 30;
    return p;
}

struct Coords {
    uint32_t ab, ae, bb, be;
};

// Overlap::trim, /root/reference/src/overlap.cpp:117-192 (SURVEY.md A.1).  u32 wrap-around is part
// of the contract.  Both piles are alive.
__host__ __device__ __forceinline__ bool trim(Coords& c, uint32_t ori, const Pile& pa, const Pile& pb) {
    if (c.ab >= pa.end || c.ae <= pa.begin || c.bb >= pb.end || c.be <= pb.begin) return false;   // :139-142
    uint32_t cut_lb = c.bb < pb.begin ? pb.begin - c.bb : 0u, cut_rb = c.be > pb.end ? c.be - pb.end : 0u;
    uint32_t cut_la = c.ab < pa.begin ? pa.begin - c.ab : 0u, cut_ra = c.ae > pa.end ? c.ae - pa.end : 0u;
    uint32_t nab = c.ab + (ori ? cut_rb : cut_lb);                                                // :146-164
    uint32_t nae = c.ae - (ori ? cut_lb : cut_rb);
    uint32_t nbb = c.bb + (ori ? cut_ra : cut_la);
    uint32_t nbe = c.be - (ori ? cut_la : cut_ra);
    if (nab >= pa.end || nae <= pa.begin || nbb >= pb.end || nbe <= pb.begin) return false;       // :166-169
    nab = max(nab, pa.begin); nae = min(nae, pa.end);                                             // :171-174
    nbb = max(nbb, pb.begin); nbe = min(nbe, pb.end);
    if (nab >= nae || nae - nab < 84u || nbb >= nbe || nbe - nbb < 84u) return false;             // :176-179
    c.ab = nab; c.ae = nae; c.bb = nbb; c.be = nbe;
    return true;
}

// Trimmed-read coordinates used by type() and by edge creation (overlap.cpp:206-216, graph.cpp:582-592).
struct Rel {
    uint32_t a0, a1, b0, b1, al, bl;
};

__host__ __device__ __forceinline__ Rel relative(const Coords& c, uint32_t ori, const Pile& pa, const Pile& pb) {
    Rel r;
    r.al = pa.end - pa.begin;
    r.a0 = c.ab - pa.begin;
    r.a1 = c.ae - pa.begin;
    r.bl = pb.end - pb.begin;
    r.b0 = ori ? r.bl - c.be + pb.begin : c.bb - pb.begin;
    r.b1 = ori ? r.bl - c.bb + pb.begin : c.be - pb.begin;
    return r;
}

__host__ __device__ __forceinline__ uint32_t absdiff(uint32_t a, uint32_t b) { return a > b ? a - b : b - a; }

// ---------------------------------------------------------------------------------------------
// The reference's floating point on this path is three IEEE double products compared with integers
// (overlap.cpp:221-222, 236-237; graph.cpp:26-29).  u32 -> f64 conversions run on the XU pipe
// (16 lanes / clk / SM) and made K1 and K3 XU-bound (profiles/r01a_pipes_stalls.txt), so each
// comparison is evaluated in EXACT integer arithmetic instead.  Bit-identical for every u32 input
// (proofs in DESIGN.md "Exact integer forms"; tests/test_exact_arith.py checks every boundary case
// of the u32 range against IEEE doubles):
//   (double)s <  (double)t * 0.875        <=>  8 s < 7 t            (0.875 = 7/8, product exact)
//   (double)d <  (double)L * 0.01         <=>  100 d < L            (RN(L * 0.01) == L / 100 when 100 | L)
//   (u32)(0.05 * (double)M)                ==  M / 20               (RN(M * 0.05) == M / 20 when 20 | M)
//   a >= b * (1 - 0.12), a <= b * (1 + 0.12)  <=>  25 a >= 22 b,  25 a <= 28 b
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ bool lt_7_8(uint32_t s, uint32_t t) {   // (double)s < (double)t * 0.875
    return (unsigned long long) s * 8ull < (unsigned long long) t * 7ull;
}

// Overlap::type, overlap.cpp:194-259 (SURVEY.md A.2).
__host__ __device__ __forceinline__ uint8_t classify(const Coords& c, const Rel& r) {
    uint32_t overhang = min(r.a0, r.b0) + min(r.al - r.a1, r.bl - r.b1);                          // :218-219
    uint32_t sa = r.a1 - r.a0, sb = r.b1 - r.b0;
    if (lt_7_8(sa, sa + overhang) || lt_7_8(sb, sb + overhang)) return kX;                        // :221-224
    uint32_t ta = r.al - r.a1, tb = r.bl - r.b1;
    if (r.a0 <= r.b0 && ta <= tb) return kB;                                                      // :225-227
    if (r.a0 >= r.b0 && ta >= tb) return kA;                                                      // :228-230
    uint32_t span_a = c.ae - c.ab, span_b = c.be - c.bb;
    uint32_t length = max(span_a, span_b);                                                        // length_ (:189)
    if ((unsigned long long) absdiff(span_a, span_b) * 100ull < (unsigned long long) length) {    // :236
        uint32_t min_ext = max(r.al, r.bl) / 20u;                                                 // :237
        if (absdiff(r.a0, r.b0) < min_ext) return ta >= tb ? kA : kB;                             // :239-245
        if (absdiff(ta, tb) < min_ext) return r.a0 >= r.b0 ? kA : kB;                             // :246-252
    }
    return r.a0 > r.b0 ? kAB : kBA;                                                               // :255-258
}

// Event detection of the first pass over the records (k_classify_events): trim() followed by classify(), reduced to
// what the ORDER-DEPENDENT part needs, as straight-line predicate arithmetic (no early returns: the compiler's branchy
// translation of the two functions above executed ~220 warp instructions per record with divergent lanes waiting at
// every reconvergence point, profiles/r01h).  Returns
//     bit 0   trim() accepts the record (both piles alive)
//     bit 1   type is kB (a contained in b)        bit 2   type is kA (b contained in a)
// p = a's pile [p0, p1), q = b's pile [q0, q1); a dead pile has end == 0 and fails the first test below by itself.
// Exactness (tests/test_exact_arith.py compares with trim() + classify() on boundary and random inputs): pile
// ends are < 2^30 (rala_b200.h limits), so once the two range tests have passed every trimmed coordinate lies in
// [0, 2^30]: differences fit a signed compare, span + overhang cannot wrap, and  8 s < 7 (s + oh)  <=>  s < 7 oh.
__host__ __device__ __forceinline__ uint32_t event_code(uint32_t ab, uint32_t ae, uint32_t bb, uint32_t be, uint32_t ori,
                                                        uint32_t p0, uint32_t p1, uint32_t q0, uint32_t q1) {
    const bool r1 = (ab >= p1) | (ae <= p0) | (bb >= q1) | (be <= q0);                            // overlap.cpp:139-142
    const uint32_t cut_lb = max(q0, bb) - bb, cut_rb = be - min(be, q1);                          // :146-164
    const uint32_t cut_la = max(p0, ab) - ab, cut_ra = ae - min(ae, p1);
    uint32_t nab = ab + (ori ? cut_rb : cut_lb);
    uint32_t nae = ae - (ori ? cut_lb : cut_rb);
    uint32_t nbb = bb + (ori ? cut_ra : cut_la);
    uint32_t nbe = be - (ori ? cut_la : cut_ra);
    const bool r2 = (nab >= p1) | (nae <= p0) | (nbb >= q1) | (nbe <= q0);                        // :166-169
    nab = max(nab, p0); nae = min(nae, p1); nbb = max(nbb, q0); nbe = min(nbe, q1);               // :171-174
    const uint32_t sa = nae - nab, sb = nbe - nbb;
    const bool r3 = ((int32_t) sa < 84) | ((int32_t) sb < 84);                                    // :176-179
    // Overlap::type on the trimmed coordinates (overlap.cpp:206-258)
    const uint32_t a0 = nab - p0, ta = p1 - nae, x = nbb - q0, y = q1 - nbe;
    const uint32_t b0 = ori ? y : x, tb = ori ? x : y;                                            // b flipped if RC (:211-216)
    const unsigned long long oh7 = (unsigned long long) (min(a0, b0) + min(ta, tb)) * 7ull;       // :218-219
    const bool kx = ((unsigned long long) sa < oh7) | ((unsigned long long) sb < oh7);            // :221-224
    const bool a_ge = a0 >= b0, t_ge = ta >= tb;
    const bool cont_b = (a0 <= b0) & (ta <= tb), cont_a = a_ge & t_ge;                            // :225-230
    const uint32_t len = max(sa, sb);
    const bool nearly = (unsigned long long) (len - min(sa, sb)) * 100ull < (unsigned long long) len;   // :236
    const uint32_t me = max(p1 - p0, q1 - q0) / 20u;                                              // :237
    const bool n1 = absdiff(a0, b0) < me, n2 = absdiff(ta, tb) < me;
    const bool near_a = nearly & ((n1 & t_ge) | (!n1 & n2 & a_ge));                               // :239-252
    const bool near_b = nearly & ((n1 & !t_ge) | (!n1 & n2 & !a_ge));
    const bool is_b = cont_b | (!cont_a & near_b);
    const bool is_a = !cont_b & (cont_a | near_a);
    const bool ok = !(r1 | r2 | r3);
    return (ok ? 1u : 0u) | ((ok & !kx & is_b) ? 2u : 0u) | ((ok & !kx & is_a) ? 4u : 0u);
}

// comparable(a, b, 0.12), graph.cpp:26-29; a = (double)(u32)(len_ab + len_bc), b = (double)len_ac:
//   (a >= 0.88 b && a <= 1.12 b) || (b >= 0.88 a && b <= 1.12 a)
// In exact arithmetic the two clauses are the intervals [22b/25, 28b/25] and [25b/28, 25b/22] for a; they
// overlap (25/28 < 28/25), so their union is the hull:  25 a >= 22 b  &&  22 a <= 25 b.
__host__ __device__ __forceinline__ bool comparable(uint32_t a, uint32_t b) {
    return (unsigned long long) a * 25ull >= (unsigned long long) b * 22ull &&
           (unsigned long long) a * 22ull <= (unsigned long long) b * 25ull;
}

// The same test as an interval of a for a fixed b: comparable(a, b) <=> a - lo <= range (unsigned),
// lo = ceil(22 b / 25), range = min(floor(25 b / 22), 2^32 - 1) - lo.
__host__ __device__ __forceinline__ uint2 comparable_interval(uint32_t b) {
    const unsigned long long lo = ((unsigned long long) b * 22ull + 24ull) / 25ull;
    unsigned long long hi = (unsigned long long) b * 25ull / 22ull;
    if (hi > 0xFFFFFFFFull) hi = 0xFFFFFFFFull;
    return make_uint2((uint32_t) lo, (uint32_t) (hi - lo));   // lo <= b <= hi always
}

// ---------------------------------------------------------------------------------------------
// Front end: the duplicate filter of Graph::initialize (graph.cpp:273-303, grouping loop :340-361).
// A query group = a maximal run of records with the same a_id among the records whose names resolved (bit 31 of a[i]
// set = the reference holds nullptr there: such records are skipped wherever they stand, also inside a group).  The
// reference's nested loop (every record of a group, valid or not, knocks out the later records with the same b_id that
// are shorter, and stops - knocked out itself - at the first one that is not) leaves exactly ONE record per (group,
// b_id): the LAST one of maximal length().  Hence record k survives iff no later record of its group with the same b_id
// is at least as long and no earlier one is longer.  (Why the earlier clause needs no "reaches k" condition: take the last
// earlier record that is longer than k; everything between it and k is no longer than k, so nothing stopped it.)
// Self overlaps (a_id == b_id) are dropped and knock out nobody (:278-288).  tests/host_dupfilter.cu checks this function
// against the oracle's literal restatement of the loops on the CPU; tests/golden/dups.npz pins both to the reference.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ bool duplicate_filter_keeps(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                                                const uint32_t* __restrict__ len, uint64_t n, uint64_t k) {
    const uint32_t ak = a[k];
    if (ak & kInvalidBit) return false;
    const uint32_t bk = b[k] & 0x7FFFFFFFu;
    if (ak == bk) return false;
    const uint32_t lk = len[k];
    for (uint64_t j = k + 1; j < n; ++j) {
        const uint32_t aj = a[j];
        if (aj & kInvalidBit) continue;
        if (aj != ak) break;
        if ((b[j] & 0x7FFFFFFFu) == bk && len[j] >= lk) return false;
    }
    for (uint64_t j = k; j-- > 0;) {
        const uint32_t aj = a[j];
        if (aj & kInvalidBit) continue;
        if (aj != ak) break;
        if ((b[j] & 0x7FFFFFFFu) == bk && len[j] > lk) return false;
    }
    return true;
}

// ---------------------------------------------------------------------------------------------
// Warp / block helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint32_t warp_id() { return threadIdx.x >> 5; }

__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if ((int) lane_id() >= d) v += t;
    }
    return v;
}

__device__ __forceinline__ unsigned long long warp_sum64(unsigned long long v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
    return v;
}

// ---------------------------------------------------------------------------------------------
// Single-pass ordered compaction: decoupled look-back over tile aggregates.
// One 64-bit status word per tile: [63:62] state (0 empty, 1 aggregate, 2 inclusive prefix),
// [61:31] count B, [30:0] count A.  Two independent 31-bit counters ride in one word so a kernel
// can split its input into two ordered output lists in one pass.
// Tiles are handed out through an atomic ticket, so a tile only ever waits on tiles that are
// already resident or finished (forward progress without co-residency assumptions).
// ---------------------------------------------------------------------------------------------
constexpr unsigned long long kStateAgg = 1ull << 62, kStateInc = 2ull << 62, kStateMask = 3ull << 62;
constexpr unsigned long long kCountMask = (1ull << 62) - 1;

__device__ __forceinline__ unsigned long long pack_counts(uint32_t a, uint32_t b) {
    return (unsigned long long) a | ((unsigned long long) b << 31);
}
__device__ __forceinline__ uint32_t count_a(unsigned long long v) { return (uint32_t) (v & 0x7FFFFFFFull); }
__device__ __forceinline__ uint32_t count_b(unsigned long long v) { return (uint32_t) ((v >> 31) & 0x7FFFFFFFull); }

__device__ __forceinline__ unsigned long long ld_status(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_status(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// The two halves of lookback_exclusive, for a warp that has other work between them: publish `tile`'s aggregate (lane 0
// stores), then later wait for its exclusive prefix (ONE full warp) and publish the inclusive one.
__device__ __forceinline__ void lookback_publish(unsigned long long* status, uint32_t tile, unsigned long long aggregate) {
    if (lane_id() == 0) st_status(status + tile, (tile == 0 ? kStateInc : kStateAgg) | aggregate);
}

__device__ __forceinline__ unsigned long long lookback_wait(unsigned long long* status, uint32_t tile, unsigned long long aggregate) {
    const uint32_t lane = lane_id();
    if (tile == 0) return 0ull;
    unsigned long long exclusive = 0ull;
    int64_t look = (int64_t) tile - 1;
    while (true) {
        int64_t idx = look - (int64_t) lane;
        unsigned long long s = kStateInc;  // virtual tile before tile 0: inclusive prefix 0
        if (idx >= 0) {
            s = ld_status(status + idx);
            while ((s & kStateMask) == 0ull) s = ld_status(status + idx);
        }
        uint32_t inc_mask = __ballot_sync(0xFFFFFFFFu, (s & kStateMask) == kStateInc);
        uint32_t first = inc_mask ? (uint32_t) (__ffs(inc_mask) - 1) : 32u;   // nearest tile holding an inclusive prefix
        unsigned long long contrib = lane <= first ? (s & kCountMask) : 0ull;
        exclusive += warp_sum64(contrib);
        if (inc_mask) break;
        look -= 32;
    }
    if (lane == 0) st_status(status + tile, kStateInc | ((exclusive + aggregate) & kCountMask));
    return exclusive;
}

// Called by ONE full warp of the block.  Returns the exclusive prefix (packed counts) of `tile`.
__device__ __forceinline__ unsigned long long lookback_exclusive(unsigned long long* status, uint32_t tile,
                                                                  unsigned long long aggregate) {
    lookback_publish(status, tile, aggregate);
    return lookback_wait(status, tile, aggregate);
}

}  // namespace rb
