// containment.cu — K1b: the reference's ORDER-DEPENDENT containment removal, resolved in parallel.
//
// Reference semantics (graph.cpp:469-480 and 831-866, with the "pile is already dead" gate of
// Overlap::transmute, overlap.cpp:51,70): records are processed in order; a kA/kB record at time t
// kills its victim iff victim AND container are both still alive at t.  Hence, for every pile x,
//     D[x] = time of the first event (x, c, t) whose container c is alive at t      (+inf if none)
// which is well-founded on t.  The classify kernels keep every victim's earliest event; about half of the victims are
// settled by it alone (k_resolve_fast, DESIGN.md section 2).  Instead of iterating whole-array Jacobi rounds over the
// others ("hard" victims), their events are grouped by victim (counting sort over dense indices: count, scan, scatter)
// and every unsettled victim walks its own events in time order, reading only MONOTONE state of other piles:
//     S[x] = h          (bit 31 clear)  unsettled, x cannot die before time h
//     S[x] = 0x80000000 | t             settled: x dies at t     (t = 0x7FFFFFFF: never; non-victims start there)
// Every update is an atomicMax, so the state of a pile only ever grows (bounds rise, settled beats unsettled):
// concurrent, redundant resolution of the same pile by several threads is harmless, and in-place asynchronous
// reads always see valid information.  A thread that finds its victim blocked on a container whose fate is
// open CHASES the dependency (explicit stack; event times strictly decrease along a chain, so it terminates)
// instead of waiting for another round, so almost every victim settles in the first sweep; the few that
// exceed the chase budget go to a worklist that a cooperative loop (then a single block) drains.
#include <cooperative_groups.h>

#include "kernels.h"
#include "lists.cuh"

namespace cg = cooperative_groups;

namespace rb {

constexpr uint32_t kSettled = 0x80000000u;
constexpr uint32_t kNever = 0x7FFFFFFFu;
constexpr uint32_t kDeadEvent = 0xFFFFFFFFu;
constexpr uint32_t kTailMax = 512;
constexpr int kChaseDepth = 24;
constexpr int kChaseBudget = 96;
constexpr unsigned long long kNoEvent = ~0ull;   // first[] of a pile without events; a segment entry known not to fire

// an event as one word: the earliest event is the smallest word
__device__ __forceinline__ unsigned long long pack_event(uint32_t t, uint32_t c) { return ((unsigned long long) t << 32) | c; }

__device__ __forceinline__ uint32_t ld_state(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// earliest event per victim of an imported event list (the classify kernels build it on the fly otherwise)
__global__ void k_events_first(Events ev, const uint32_t* __restrict__ n_events, uint32_t ev_cap, unsigned long long* __restrict__ first) {
    const uint32_t n = min(*n_events, ev_cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        atomicMin(&first[ev.v[i]], pack_event(ev.t[i], ev.c[i]));
}

// Slots in a list counted by *total for every thread's n entries, one atomic per block (a warp-level atomic on the one
// counter serialises at L2).  Block-uniform call: every thread of the block, 256 threads.
__device__ __forceinline__ uint32_t block_reserve(uint32_t n, uint32_t* total, uint32_t* s_warp /* kTileWarps words */) {
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t inc = warp_inclusive_scan(n);
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < kTileWarps ? s_warp[lane] : 0u;
        const uint32_t winc = warp_inclusive_scan(w);
        uint32_t base = 0;
        if (lane == kTileWarps - 1 && winc) base = atomicAdd(total, winc);
        base = __shfl_sync(0xFFFFFFFFu, base, kTileWarps - 1);
        if (lane < kTileWarps) s_warp[lane] = base + winc - w;
    }
    __syncthreads();
    const uint32_t first_slot = s_warp[warp] + inc - n;
    __syncthreads();   // s_warp is reused by the next call
    return first_slot;
}

// One thread per pile: settle every victim that its earliest event (t1, c1) settles on its own, D = t1 when
//     c1 == v,  or c1 has no event,  or c1's earliest event is later than t1 (then D[c1] >= tmin[c1] > t1),
// (times are unique record positions) and hand every other victim ("hard") a dense index, a zeroed event count and its
// worklist slot.  A hard victim starts from the lower bound t1: nothing can kill it earlier.
__global__ void __launch_bounds__(256) k_resolve_fast(const unsigned long long* __restrict__ first, uint32_t n_piles,
                                                     uint32_t* __restrict__ S, uint32_t* __restrict__ hidx,
                                                     uint32_t* __restrict__ hcount, uint32_t* __restrict__ work,
                                                     uint32_t* __restrict__ n_work, const uint32_t* __restrict__ n_events,
                                                     int skip_if_empty) {
    if (skip_if_empty && *n_events == 0u) return;
    __shared__ uint32_t s_warp[kTileWarps];
    for (uint32_t base = blockIdx.x * blockDim.x; base < n_piles; base += gridDim.x * blockDim.x) {   // block-uniform trips
        const uint32_t x = base + threadIdx.x;
        bool hard = false;
        if (x < n_piles) {
            const unsigned long long f = first[x];
            uint32_t s = kSettled | kNever;
            if (f != kNoEvent) {
                const uint32_t t1 = (uint32_t) (f >> 32), c1 = (uint32_t) f;
                s = kSettled | t1;
                if (c1 != x && (first[c1] >> 32) <= t1) {   // c1 may die before t1: left to the full resolution
                    hard = true;
                    s = t1;
                }
            }
            S[x] = s;
        }
        const uint32_t d = block_reserve(hard ? 1u : 0u, &n_work[0], s_warp);
        if (hard) {
            work[d] = x;
            hidx[x] = d;
            hcount[d] = 0u;
        }
    }
}

// Events of hard victims only, each with its rank inside its victim's segment, into a compact list {dense index, rank, t, c}
// (n_work[3] entries).  An event whose container is already settled to die before it never fires and is dropped: this
// removes the earliest event of every hard victim whose earliest container k_resolve_fast settled.
__global__ void __launch_bounds__(256) k_resolve_filter(Events ev, const uint32_t* __restrict__ n_events, uint32_t ev_cap,
                                                       const uint32_t* __restrict__ S, const uint32_t* __restrict__ hidx,
                                                       uint32_t* __restrict__ hcount, uint4* __restrict__ hev,
                                                       uint32_t* __restrict__ n_work) {
    if (n_work[0] == 0u) return;   // nothing is hard (or the pass has no events)
    const uint32_t n = min(*n_events, ev_cap);
    __shared__ uint32_t s_warp[kTileWarps];
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < n; i0 += 4u * stride) {   // block-uniform trips
        uint32_t c[4], t[4], d[4], r[4];
        bool keep[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // four independent chains: event -> states + dense index -> count
            const uint32_t i = i0 + k * stride + threadIdx.x;
            keep[k] = false;
            if (i < n) {
                const uint32_t v = ev.v[i];
                c[k] = ev.c[i];
                t[k] = ev.t[i];
                const uint32_t sv = S[v], sc = S[c[k]];
                d[k] = hidx[v];
                keep[k] = !(sv & kSettled) && !((sc & kSettled) && (sc & kNever) < t[k]);
            }
        }
        uint32_t kept = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (keep[k]) r[k] = atomicAdd(&hcount[d[k]], 1u);
            kept += keep[k] ? 1u : 0u;
        }
        uint32_t slot = block_reserve(kept, &n_work[3], s_warp);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (keep[k]) hev[slot++] = make_uint4(d[k], r[k], t[k], c[k]);
    }
}

// compact list -> the hard victims' segments (offsets from the scan of the counts), one packed word per event; and each
// hard victim's segment bounds by pile, so that k_resolve finds a pile's events with one load beside its state
__global__ void __launch_bounds__(256) k_resolve_scatter(const uint4* __restrict__ hev, const uint32_t* __restrict__ n_work,
                                                        const uint32_t* __restrict__ hstart, const uint32_t* __restrict__ work,
                                                        unsigned long long* __restrict__ seg, uint2* __restrict__ seg_range) {
    const uint32_t n_ev = n_work[3], n_hard = n_work[0];
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < max(n_ev, n_hard); j += gridDim.x * blockDim.x) {
        if (j < n_ev) {
            const uint4 e = hev[j];
            seg[hstart[e.x] + e.y] = pack_event(e.z, e.w);
        }
        if (j < n_hard) seg_range[work[j]] = make_uint2(hstart[j], hstart[j + 1]);
    }
}

// Settle hard victim v0 (returns false only when the chase budget ran out; v0 then stays on the worklist).  Every pile the
// chase reaches is hard: it is only pushed while its state is open.
__device__ __forceinline__ bool resolve_victim(uint32_t v0, const uint2* __restrict__ seg_range, unsigned long long* __restrict__ seg,
                                               uint32_t* __restrict__ S) {
    uint32_t stack_v[kChaseDepth], stack_need[kChaseDepth];   // need: the time up to which the pile's fate matters
    int sp = 0, budget = kChaseBudget;
    stack_v[0] = v0;
    stack_need[0] = kNever;
    while (sp >= 0) {
        const uint32_t v = stack_v[sp];
        const uint2 r = __ldg(&seg_range[v]);     // in flight together with the state
        if (ld_state(&S[v]) & kSettled) { --sp; continue; }
        const uint32_t s0 = r.x, s1 = r.y;
        unsigned long long best = kNoEvent;
        uint32_t best_p = 0;
        for (uint32_t p = s0; p < s1; ++p) {
            const unsigned long long e = seg[p];
            if (e < best) { best = e; best_p = p; }
        }
        const uint32_t best_t = (uint32_t) (best >> 32);
        if (best_t == kDeadEvent) {               // every event found its container dead: v is never killed
            atomicMax(&S[v], kSettled | kNever);
            --sp;
            continue;
        }
        atomicMax(&S[v], best_t);                 // v cannot die before its earliest open event
        if (best_t > stack_need[sp]) { --sp; continue; }   // whoever asked only cares about earlier times
        const uint32_t c = (uint32_t) best;
        // a record with a_id == b_id makes the pile its own container: both "are alive" at that time and the pile dies
        // (graph.cpp:469-480 reset piles_[a] either way); without this the pile would wait for its own fate for ever
        const uint32_t q = c == v ? (kSettled | kNever) : ld_state(&S[c]);
        if (q & kSettled) {
            if ((q & kNever) > best_t) {          // container still alive at best_t: the event fires
                atomicMax(&S[v], kSettled | best_t);
                --sp;
            } else {
                seg[best_p] = kNoEvent;           // container died before this event: it never fires; look again
            }
            continue;
        }
        if (q > best_t) {                         // open, but certainly alive at best_t
            atomicMax(&S[v], kSettled | best_t);
            --sp;
            continue;
        }
        if (sp + 1 >= kChaseDepth || --budget <= 0) return false;
        ++sp;                                     // the container may die before best_t: find out
        stack_v[sp] = c;
        stack_need[sp] = best_t;
    }
    return true;
}

// death times for the consumers: kInf = never
__global__ void k_decode_state(uint32_t* __restrict__ S, uint32_t n_piles) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_piles; i += gridDim.x * blockDim.x) {
        const uint32_t d = S[i] & kNever;
        S[i] = d == kNever ? kInf : d;
    }
}

// the hard worklist (k_resolve_fast) in rounds; an empty list only writes the counters
__global__ void __launch_bounds__(256) k_resolve(const uint2* __restrict__ seg_range, unsigned long long* __restrict__ seg,
                                                uint32_t* __restrict__ S,
                                                uint32_t* __restrict__ work0, uint32_t* __restrict__ work1,
                                                uint32_t* __restrict__ n_work /* 3 rotating counters */,
                                                uint32_t* __restrict__ counters) {
    cg::grid_group grid = cg::this_grid();
    const uint32_t stride = gridDim.x * blockDim.x, gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = lane_id();
    uint32_t round = 0;
    uint32_t n = n_work[0];
    while (n > kTailMax) {
        const uint32_t* in = (round & 1) ? work1 : work0;
        uint32_t* out = (round & 1) ? work0 : work1;
        uint32_t* n_out = &n_work[(round + 1) % 3];
        if (gtid == 0) n_work[(round + 2) % 3] = 0u;   // last read in round-1, first written in round+1
        for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride) {
            const uint32_t i = base + threadIdx.x;
            uint32_t v = 0;
            bool keep = false;
            if (i < n) {
                v = in[i];
                keep = !resolve_victim(v, seg_range, seg, S);
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, keep);
            if (m) {
                uint32_t gb = 0;
                if (lane == 0) gb = atomicAdd(n_out, (uint32_t) __popc(m));
                gb = __shfl_sync(0xFFFFFFFFu, gb, 0);
                if (keep) out[gb + __popc(m & ((1u << lane) - 1u))] = v;
            }
        }
        grid.sync();
        ++round;
        n = ld_state(&n_work[round % 3]);
    }
    if (blockIdx.x != 0) return;
    // tail: one block, block barriers only
    __shared__ uint32_t s_n[2];
    const uint32_t* in = (round & 1) ? work1 : work0;
    uint32_t* out = (round & 1) ? work0 : work1;
    int k = 0;
    if (threadIdx.x == 0) { s_n[0] = n; s_n[1] = 0u; }
    __syncthreads();
    uint32_t stalled = 0, prev_n = 0xFFFFFFFFu;
    while (true) {
        const uint32_t m_n = s_n[k];
        if (m_n == 0) break;
        // every sweep settles at least the victim with the globally earliest open event, so the list shrinks; a list
        // that stops shrinking means the events are not well-founded (corrupt input): give up instead of spinning
        stalled = m_n >= prev_n ? stalled + 1u : 0u;
        prev_n = m_n;
        if (stalled > 64u) {
            if (threadIdx.x == 0) counters[C_OVERFLOW] = 1u;
            break;
        }
        for (uint32_t i = threadIdx.x; i < m_n; i += blockDim.x) {
            const uint32_t v = in[i];
            if (!resolve_victim(v, seg_range, seg, S)) out[atomicAdd(&s_n[k ^ 1], 1u)] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) s_n[k] = 0u;
        __syncthreads();
        k ^= 1;
        const uint32_t* tmp = in;
        in = out;
        out = const_cast<uint32_t*>(tmp);
        ++round;
    }
    if (threadIdx.x == 0) counters[C_ROUNDS] = round;
}

void launch_events_first(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, unsigned long long* first) {
    k_events_first<<<grid_for(ev_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(ev, n_events, ev_cap, first);
    L.count++;
}

int resolve_max_blocks() {
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_resolve, 256, 0);
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int dev = 0, sms = kNumSMs;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return per_sm * sms;
}

// rb.first holds every pile's earliest event on entry (filled by the classify kernels)
void launch_resolve(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, ResolveBufs rb, uint32_t n_piles,
                    uint32_t* counters, unsigned long long* status, uint32_t* ticket, int coop_blocks, bool decode, bool skip_if_empty) {
    int skip = skip_if_empty ? 1 : 0;
    cudaMemsetAsync(rb.n_work, 0, 16, L.stream);
    k_resolve_fast<<<grid_for(n_piles, 256, kNumSMs * 8), 256, 0, L.stream>>>(rb.first, n_piles, rb.S, rb.hidx, rb.vcursor, rb.work0,
                                                                           rb.n_work, n_events, skip);
    L.count++;
    // the hard path: every launch returns at once when nothing is hard
    k_resolve_filter<<<grid_for(ev_cap, 1024, kNumSMs * 8), 256, 0, L.stream>>>(ev, n_events, ev_cap, rb.S, rb.hidx, rb.vcursor,
                                                                             rb.hev, rb.n_work);
    L.count++;
    launch_scan_u32(L, rb.vcursor, rb.vstart, n_piles + 1, status, ticket, nullptr, rb.n_work, rb.n_work);
    uint2* seg_range = reinterpret_cast<uint2*>(rb.first);   // first[] is not read after k_resolve_fast
    k_resolve_scatter<<<grid_for(ev_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(rb.hev, rb.n_work, rb.vstart, rb.work0, rb.seg,
                                                                            seg_range);
    L.count++;
    void* args[] = {&seg_range, &rb.seg, &rb.S, &rb.work0, &rb.work1, &rb.n_work, &counters};
    cudaLaunchCooperativeKernel((void*) k_resolve, dim3(coop_blocks), dim3(256), args, 0, L.stream);
    L.count++;
    if (decode) {   // otherwise k_apply_deaths decodes while it applies (no consumer in between)
        k_decode_state<<<grid_for(n_piles, 256, kNumSMs * 8), 256, 0, L.stream>>>(rb.S, n_piles);
        L.count++;
    }
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_containment() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_events_first);
    cudaFuncGetAttributes(&a, k_resolve_fast);
    cudaFuncGetAttributes(&a, k_resolve_filter);
    cudaFuncGetAttributes(&a, k_resolve_scatter);
    cudaFuncGetAttributes(&a, k_decode_state);
    cudaFuncGetAttributes(&a, k_resolve);
}

}  // namespace rb
