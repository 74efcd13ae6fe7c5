// containment.cu — K1b: the reference's ORDER-DEPENDENT containment removal, resolved in parallel.
//
// Reference semantics (graph.cpp:469-480 and 831-866, with the "pile is already dead" gate of
// Overlap::transmute, overlap.cpp:51,70): records are processed in order; a kA/kB record at time t
// kills its victim iff victim AND container are both still alive at t.  Hence, for every pile x,
//     D[x] = time of the first event (x, c, t) whose container c is alive at t      (+inf if none)
// which is well-founded on t.  Instead of iterating whole-array Jacobi rounds, events are grouped by
// victim (counting sort: histogram in the classify kernel, scan, scatter) and every unsettled victim
// walks its own events in time order, reading only MONOTONE state of other piles:
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

__device__ __forceinline__ uint32_t ld_state(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void k_events_hist(Events ev, const uint32_t* __restrict__ n_events, uint32_t ev_cap, uint32_t* __restrict__ vcount) {
    const uint32_t n = min(*n_events, ev_cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&vcount[ev.v[i]], 1u);
}

// Two independent jobs that both follow the scan of the victim histogram, in one launch: the first `fill_blocks` blocks
// scatter the events into their victim's segment (order inside a segment is irrelevant), the others initialise the
// states and the worklist.
__global__ void __launch_bounds__(256) k_resolve_prepare(Events ev, const uint32_t* __restrict__ n_events, uint32_t ev_cap,
                                                        uint32_t* __restrict__ vcursor, uint32_t* __restrict__ seg_c,
                                                        uint32_t* __restrict__ seg_t, const uint32_t* __restrict__ vstart,
                                                        uint32_t n_piles, uint32_t* __restrict__ S, uint32_t* __restrict__ work,
                                                        uint32_t* __restrict__ n_work, uint32_t fill_blocks, int skip_if_empty) {
    if (skip_if_empty && *n_events == 0u) return;
    if (blockIdx.x < fill_blocks) {
        const uint32_t n = min(*n_events, ev_cap);
        const uint32_t stride = fill_blocks * blockDim.x;   // four independent load -> atomic -> store chains per thread
        for (uint32_t i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += 4u * stride) {
            uint32_t v[4], c[4], t[4], p[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t i = i0 + k * stride;
                if (i < n) { v[k] = ev.v[i]; c[k] = ev.c[i]; t[k] = ev.t[i]; }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (i0 + k * stride < n) p[k] = atomicAdd(&vcursor[v[k]], 1u);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (i0 + k * stride < n) {
                    seg_c[p[k]] = c[k];
                    seg_t[p[k]] = t[k];
                }
            }
        }
        return;
    }
    const uint32_t init_blocks = gridDim.x - fill_blocks, b = blockIdx.x - fill_blocks;
    for (uint32_t base = b * blockDim.x; base < n_piles; base += init_blocks * blockDim.x) {
        const uint32_t x = base + threadIdx.x;
        bool victim = false;
        if (x < n_piles) {
            victim = vstart[x + 1] != vstart[x];
            S[x] = victim ? 0u : (kSettled | kNever);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, victim);
        if (m) {
            uint32_t gb = 0;
            if (lane_id() == 0) gb = atomicAdd(n_work, (uint32_t) __popc(m));
            gb = __shfl_sync(0xFFFFFFFFu, gb, 0);
            if (victim) work[gb + __popc(m & ((1u << lane_id()) - 1u))] = x;
        }
    }
}

// Settle victim v0 (returns false only when the chase budget ran out; v0 then stays on the worklist).
__device__ __forceinline__ bool resolve_victim(uint32_t v0, const uint32_t* __restrict__ vstart,
                                               const uint32_t* __restrict__ seg_c, uint32_t* __restrict__ seg_t,
                                               uint32_t* __restrict__ S) {
    uint32_t stack_v[kChaseDepth], stack_need[kChaseDepth];   // need: the time up to which the pile's fate matters
    int sp = 0, budget = kChaseBudget;
    stack_v[0] = v0;
    stack_need[0] = kNever;
    while (sp >= 0) {
        const uint32_t v = stack_v[sp];
        if (ld_state(&S[v]) & kSettled) { --sp; continue; }
        const uint32_t s0 = vstart[v], s1 = vstart[v + 1];
        uint32_t best_t = kDeadEvent, best_p = 0;
        for (uint32_t p = s0; p < s1; ++p) {
            const uint32_t t = seg_t[p];
            if (t < best_t) { best_t = t; best_p = p; }
        }
        if (best_t == kDeadEvent) {               // every event found its container dead: v is never killed
            atomicMax(&S[v], kSettled | kNever);
            --sp;
            continue;
        }
        atomicMax(&S[v], best_t);                 // v cannot die before its earliest open event
        if (best_t > stack_need[sp]) { --sp; continue; }   // whoever asked only cares about earlier times
        const uint32_t c = seg_c[best_p];
        // a record with a_id == b_id makes the pile its own container: both "are alive" at that time and the pile dies
        // (graph.cpp:469-480 reset piles_[a] either way); without this the pile would wait for its own fate for ever
        const uint32_t q = c == v ? (kSettled | kNever) : ld_state(&S[c]);
        if (q & kSettled) {
            if ((q & kNever) > best_t) {          // container still alive at best_t: the event fires
                atomicMax(&S[v], kSettled | best_t);
                --sp;
            } else {
                seg_t[best_p] = kDeadEvent;       // container died before this event: it never fires; look again
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

__global__ void __launch_bounds__(256) k_resolve(const uint32_t* __restrict__ vstart, const uint32_t* __restrict__ seg_c,
                                                uint32_t* __restrict__ seg_t, uint32_t* __restrict__ S,
                                                uint32_t* __restrict__ work0, uint32_t* __restrict__ work1,
                                                uint32_t* __restrict__ n_work /* 3 rotating counters */,
                                                uint32_t* __restrict__ counters, const uint32_t* __restrict__ n_events, int skip_if_empty) {
    if (skip_if_empty && *n_events == 0u) {   // every block takes this branch: no grid barrier is left waiting
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            counters[C_ROUNDS] = 0u;
            counters[C_DSEL] = 0u;
        }
        return;
    }
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
                keep = !resolve_victim(v, vstart, seg_c, seg_t, S);
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
            if (!resolve_victim(v, vstart, seg_c, seg_t, S)) out[atomicAdd(&s_n[k ^ 1], 1u)] = v;
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
    if (threadIdx.x == 0) {
        counters[C_ROUNDS] = round;
        counters[C_DSEL] = 0u;
    }
}

void launch_events_hist(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, uint32_t* vcount) {
    k_events_hist<<<grid_for(ev_cap, 256, kNumSMs * 8), 256, 0, L.stream>>>(ev, n_events, ev_cap, vcount);
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

// vcursor holds the per-victim event histogram on entry (filled by the classify kernels)
void launch_resolve(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, ResolveBufs rb, uint32_t n_piles,
                    uint32_t* counters, unsigned long long* status, uint32_t* ticket, int coop_blocks, bool decode, bool skip_if_empty) {
    int skip = skip_if_empty ? 1 : 0;
    launch_scan_u32(L, rb.vcursor, rb.vstart, n_piles + 1, status, ticket, nullptr, skip_if_empty ? n_events : nullptr);
    cudaMemsetAsync(rb.n_work, 0, 16, L.stream);
    const int fill_blocks = grid_for(ev_cap, 1024, kNumSMs * 4), init_blocks = grid_for(n_piles, 256, kNumSMs * 4);
    k_resolve_prepare<<<fill_blocks + init_blocks, 256, 0, L.stream>>>(ev, n_events, ev_cap, rb.vcursor, rb.seg_c, rb.seg_t, rb.vstart,
                                                                     n_piles, rb.S, rb.work0, rb.n_work, (uint32_t) fill_blocks, skip);
    L.count++;
    void* args[] = {&rb.vstart, &rb.seg_c, &rb.seg_t, &rb.S, &rb.work0, &rb.work1, &rb.n_work, &counters, &n_events, &skip};
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
    cudaFuncGetAttributes(&a, k_events_hist);
    cudaFuncGetAttributes(&a, k_resolve_prepare);
    cudaFuncGetAttributes(&a, k_decode_state);
    cudaFuncGetAttributes(&a, k_resolve);
}

}  // namespace rb
