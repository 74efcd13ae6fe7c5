// fabric.cu — kernels of the multi-rank exchange layer (fabric.cuh): flag barrier over peer memory, routing of
// containment events / edges / transitive marks to their owners, the distributed containment resolution, and the
// replication of the owner-built CSR slices.  Every remote access is a store or a reduction INTO the consumer's
// arena; consumers only ever read their own memory.
#include "fabric.cuh"
#include "kernels.h"

namespace rb {

// ---------------------------------------------------------------------------------------------
// system-scope accesses (peer memory over NVLink)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_max_sys(uint32_t* p, uint32_t v) {
    asm volatile("red.relaxed.sys.global.max.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ FabricHdr* hdr_of(const Peers& P, int q) { return reinterpret_cast<FabricHdr*>(P.base[q]); }
template <class T>
__device__ __forceinline__ T* section(const Peers& P, int q, size_t off) { return reinterpret_cast<T*>(P.base[q] + off); }

// x-dimension of a grid whose y-dimension is the source rank: about 8 blocks per SM over the whole grid, at least one per SM
// (with kNumSMs blocks per source the inbox kernels ran on 148 blocks at world = 1 and took 2 - 3 x their time, profiles/r02v)
static inline int blocks_per_source(int world) {
    const int b = kNumSMs * 8 / (world < 1 ? 1 : world);
    return b < kNumSMs ? kNumSMs : b;
}

// ---------------------------------------------------------------------------------------------
// Barrier.  Lane q publishes this rank's mail to peer q, makes everything this rank pushed before visible
// (the pushes were issued by EARLIER kernels of the same stream, so they are complete; the fence orders the mail),
// raises its flag in q's header and waits for q's flag in its own header.  Epochs count up for ever, so flags never
// have to be reset; mail is double-buffered by epoch parity because a peer may enter the next barrier (and publish
// again) while this rank still reads the mail of the current one.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_fabric_barrier(Peers P, Publish pub) {
    const int q = threadIdx.x, me = P.rank, W = P.world;
    FabricHdr* mine = hdr_of(P, me);
    const uint32_t e = mine->epoch + 1u, par = e & 1u;
    if (pub.skippable && mine->skip_pass) {   // every rank took the same decision from the same mail: nobody signals, nobody waits
        __syncwarp();
        if (q == 0) {
            if (pub.bookkeeping == 1 && pub.round == 0) mine->rounds_needed[pub.pass] = 1u;
            mine->tlog[e % kBarrierLog][0] = mine->tlog[e % kBarrierLog][1] = global_timer_ns();
            mine->epoch = e;
        }
        return;
    }
    if (q == 0) mine->tlog[e % kBarrierLog][0] = global_timer_ns();
    if (q < W) {
        FabricHdr* peer = hdr_of(P, q);
#pragma unroll
        for (int k = 0; k < kMailSlots; ++k)
            if (pub.scalar[k]) st_sys(&peer->mail[par][me][k], *pub.scalar[k]);
        if (pub.per_dst) st_sys(&peer->mail[par][me][M_SENT_TO_YOU], pub.per_dst[q]);
        if (pub.bcast)
            for (int d = 0; d < W; ++d) st_sys(&peer->sent[par][me][d], pub.bcast[d]);
        __threadfence_system();
        st_release_sys(&peer->flag[me], e);
        // a peer that never arrives must not hang the GPU: after the timeout the fabric is dead, and no later barrier waits
        const unsigned long long t0 = global_timer_ns();
        while ((int32_t) (ld_acquire_sys(&mine->flag[q]) - e) < 0) {
            if (ld_relaxed_sys(&mine->dead) || global_timer_ns() - t0 > pub.timeout_ns) {
                atomicOr(&mine->error, (uint32_t) FE_TIMEOUT);
                if (atomicExch(&mine->dead, 1u) == 0u) {
                    mine->dead_epoch = e;
                    mine->dead_peer = (uint32_t) q;
                }
                break;
            }
            __nanosleep(64);
        }
    }
    __syncwarp();
    if (q == 0) {
        if (pub.bookkeeping == 2) {   // events of a pass routed: a pass without a single event anywhere is skipped by every rank
            uint32_t emitted = 0;
            for (int p = 0; p < W; ++p) emitted += mine->mail[par][p][M_EMITTED];
            mine->skip_pass = (pub.pass == 1 && emitted == 0u) ? 1u : 0u;
        }
        if (pub.bookkeeping == 1) {   // after a resolution round: is any victim still open anywhere?
            uint32_t open = 0;
            for (int p = 0; p < W; ++p) open += mine->mail[par][p][M_UNSETTLED];
            if (open == 0u && mine->rounds_needed[pub.pass] == 0u) mine->rounds_needed[pub.pass] = (uint32_t) pub.round + 1u;
            if (open != 0u && pub.round == pub.last_round) atomicOr(&mine->error, (uint32_t) FE_ROUNDS);
        }
        mine->tlog[e % kBarrierLog][1] = global_timer_ns();
        __threadfence();
        mine->epoch = e;
    }
}

const uint32_t* skip_flag(const Peers& P) { return &reinterpret_cast<const FabricHdr*>(P.base[P.rank])->skip_pass; }

void launch_fabric_barrier(Launch& L, Peers P, Publish pub) {
    k_fabric_barrier<<<1, 32, 0, L.stream>>>(P, pub);
    L.count++;
}

// ---------------------------------------------------------------------------------------------
// Routing: items (containment events, edges) -> the arena of the rank that owns them, a fused all-to-all.  A block
// takes 1024 items, sorts them by destination in shared memory (counting sort over <= 16 bins), reserves one run of
// slots per destination with ONE global atomic each, and writes every run with consecutive threads on consecutive
// addresses: 512 contiguous bytes per column and destination on average at world = 8.  (Letting each warp store its own
// items wrote 16-byte pieces at world = 8, one NVLink write each: profiles/r02n, 60 - 90 us slower per routing.)
// The per-destination counters keep counting beyond the capacity, so they are also the observed demand.
// ---------------------------------------------------------------------------------------------
constexpr int kRouteTile = 1024;

template <int COLS>
struct RouteSmem {
    uint32_t cnt[kMaxRanks], base[kMaxRanks], off[kMaxRanks + 1];
    uint32_t buf[COLS][kRouteTile];
    uint8_t dst[kRouteTile];
};

// dest[r] / val[r][c]: this thread's items r = 0..3 of the tile (dest = 0xFF: no item).  block_cols: start of this rank's
// block in the destination's inbox, as a word offset from the destination's arena section; cap = capacity of a column.
template <int COLS>
__device__ __forceinline__ void route_tile(RouteSmem<COLS>& sh, const Peers& P, size_t section_off, size_t block_words, uint32_t cap,
                                           const uint32_t (&dest)[4], const uint32_t (&val)[4][COLS], uint32_t* __restrict__ out_cnt) {
    const uint32_t tid = threadIdx.x, W = (uint32_t) P.world;
    if (tid < (uint32_t) kMaxRanks) sh.cnt[tid] = 0u;
    __syncthreads();
    uint32_t rank[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) rank[r] = dest[r] != 0xFFu ? atomicAdd(&sh.cnt[dest[r]], 1u) : 0u;
    __syncthreads();
    if (tid < W) sh.base[tid] = sh.cnt[tid] ? atomicAdd(&out_cnt[tid], sh.cnt[tid]) : 0u;
    if (tid == 0) {
        uint32_t run = 0;
        for (uint32_t q = 0; q < W; ++q) {
            sh.off[q] = run;
            run += sh.cnt[q];
        }
        sh.off[W] = run;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (dest[r] == 0xFFu) continue;
        const uint32_t pos = sh.off[dest[r]] + rank[r];
#pragma unroll
        for (int c = 0; c < COLS; ++c) sh.buf[c][pos] = val[r][c];
        sh.dst[pos] = (uint8_t) dest[r];
    }
    __syncthreads();
    const uint32_t total = sh.off[W];
    for (uint32_t pos = tid; pos < total; pos += blockDim.x) {
        const uint32_t q = sh.dst[pos], slot = sh.base[q] + (pos - sh.off[q]);
        if (slot < cap) {
            uint32_t* blk = reinterpret_cast<uint32_t*>(P.base[q] + section_off) + block_words;
#pragma unroll
            for (int c = 0; c < COLS; ++c) blk[(size_t) c * cap + slot] = sh.buf[c][pos];
        }
    }
    __syncthreads();
}

// containment events -> the rank that owns the victim pile (inbox block = this rank)
__global__ void __launch_bounds__(256) k_route_events(Peers P, ArenaLayout A, Events ev, const uint32_t* __restrict__ n_events,
                                                     uint32_t ev_cap, uint32_t* __restrict__ out_cnt) {
    __shared__ RouteSmem<3> sh;
    const uint32_t n = min(*n_events, ev_cap);
    for (uint32_t base = blockIdx.x * kRouteTile; base < n; base += gridDim.x * kRouteTile) {
        uint32_t dest[4], val[4][3];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint32_t i = base + r * 256u + threadIdx.x;
            dest[r] = 0xFFu;
            if (i < n) {
                val[r][0] = ev.v[i]; val[r][1] = ev.c[i]; val[r][2] = ev.t[i];
                dest[r] = pile_owner(val[r][0], (uint32_t) P.world);
            }
        }
        route_tile<3>(sh, P, A.ev_inbox, (size_t) P.rank * 3u * A.cap_ev, A.cap_ev, dest, val, out_cnt);
    }
}

void launch_route_events(Launch& L, Peers P, ArenaLayout A, Events ev, const uint32_t* n_events, uint32_t ev_cap, uint32_t* out_cnt) {
    k_route_events<<<grid_for(ev_cap, kRouteTile, kNumSMs * 4), 256, 0, L.stream>>>(P, A, ev, n_events, ev_cap, out_cnt);
    L.count++;
}

// inbox blocks (counts in the mail of the barrier just passed) -> one local event list, per-victim histogram for the
// counting sort, earliest event time per victim (initial lower bound of its death time).  blockIdx.y = source rank.
__global__ void __launch_bounds__(256) k_gather_events(Peers P, ArenaLayout A, Events ev, uint32_t ev_cap, uint32_t* __restrict__ n_events_out,
                                                      uint32_t* __restrict__ vcount, uint32_t* __restrict__ tmin) {
    FabricHdr* mine = hdr_of(P, P.rank);
    if (mine->skip_pass) {
        if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *n_events_out = 0u;
        return;
    }
    const uint32_t par = mine->epoch & 1u, src = blockIdx.y;
    uint32_t offset = 0;
    for (uint32_t p = 0; p < src; ++p) offset += min(mine->mail[par][p][M_SENT_TO_YOU], A.cap_ev);
    const uint32_t sent = mine->mail[par][src][M_SENT_TO_YOU], n = min(sent, A.cap_ev);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (sent > A.cap_ev || offset + n > ev_cap) atomicOr(&mine->error, (uint32_t) FE_INBOX);
        if (src == (uint32_t) P.world - 1u) *n_events_out = min(offset + n, ev_cap);
    }
    const uint32_t* blk = section<uint32_t>(P, P.rank, A.ev_inbox) + (size_t) src * 3u * A.cap_ev;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (offset + i >= ev_cap) break;
        const uint32_t v = blk[i], c = blk[(size_t) A.cap_ev + i], t = blk[2 * (size_t) A.cap_ev + i];
        ev.v[offset + i] = v;
        ev.c[offset + i] = c;
        ev.t[offset + i] = t;
        if (v < A.n_piles) {
            atomicAdd(&vcount[v], 1u);
            atomicMin(&tmin[v], t);
        }
    }
}

void launch_gather_events(Launch& L, Peers P, ArenaLayout A, Events ev, uint32_t ev_cap, uint32_t* n_events_out, uint32_t* vcount,
                          uint32_t* tmin) {
    dim3 grid(grid_for(A.cap_ev, 256, blocks_per_source(P.world)), P.world);
    k_gather_events<<<grid, 256, 0, L.stream>>>(P, A, ev, ev_cap, n_events_out, vcount, tmin);
    L.count++;
}

// ---------------------------------------------------------------------------------------------
// Distributed ordered containment.  Same monotone state word per pile as containment.cu
//     S[x] = h (bit 31 clear)   open: x cannot die before time h        S[x] = 0x80000000 | t   settled (t = 0x7FFFFFFF: never)
// replicated on every rank.  A rank resolves the piles it OWNS (it holds all their events) and pushes every change
// of their state to all replicas with a remote max-reduction; states of foreign piles are only read.  A victim whose
// earliest open event hangs on a foreign container that is still open stays on the worklist for the next round.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kSettled = 0x80000000u;
constexpr uint32_t kNever = 0x7FFFFFFFu;
constexpr uint32_t kDeadEvent = 0xFFFFFFFFu;
constexpr int kChaseDepth = 24;
constexpr int kChaseBudget = 96;

// scatter the gathered events into their victim's segment; initialise the states of the OWNED piles and the worklist
__global__ void __launch_bounds__(256) k_fabric_prepare(Peers P, ArenaLayout A, Events ev, const uint32_t* __restrict__ n_events, uint32_t ev_cap,
                                                       uint32_t* __restrict__ vcursor, uint32_t* __restrict__ seg_c, uint32_t* __restrict__ seg_t,
                                                       const uint32_t* __restrict__ vstart, const uint32_t* __restrict__ tmin,
                                                       uint32_t* __restrict__ work, uint32_t* __restrict__ n_work, uint32_t fill_blocks) {
    if (hdr_of(P, P.rank)->skip_pass) return;
    if (blockIdx.x < fill_blocks) {
        const uint32_t n = min(*n_events, ev_cap);
        const uint32_t stride = fill_blocks * blockDim.x;
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
    uint32_t* S = section<uint32_t>(P, P.rank, A.S);
    const uint32_t init_blocks = gridDim.x - fill_blocks, b = blockIdx.x - fill_blocks;
    for (uint32_t base = b * blockDim.x; base < A.ppr; base += init_blocks * blockDim.x) {
        const uint32_t x = owned_pile(base + threadIdx.x, (uint32_t) P.rank, (uint32_t) P.world);
        bool victim = false;
        if (base + threadIdx.x < A.ppr && x < A.n_piles) {
            victim = vstart[x + 1] != vstart[x];
            S[x] = victim ? min(tmin[x], kNever - 1u) : (kSettled | kNever);
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

void launch_fabric_prepare(Launch& L, Peers P, ArenaLayout A, Events ev, const uint32_t* n_events, uint32_t ev_cap, ResolveBufs rb,
                           const uint32_t* tmin) {
    const int fill_blocks = grid_for(ev_cap, 1024, kNumSMs * 2), init_blocks = grid_for(A.ppr, 256, kNumSMs * 2);
    k_fabric_prepare<<<fill_blocks + init_blocks, 256, 0, L.stream>>>(P, A, ev, n_events, ev_cap, rb.vcursor, rb.seg_c, rb.seg_t, rb.vstart,
                                                                    tmin, rb.work0, rb.n_work, (uint32_t) fill_blocks);
    L.count++;
}

// everything a containment pass starts from, in one launch (six memset nodes otherwise): pile states of the replica and
// the per-victim histogram to 0, earliest-event times and the "waiting for" notes to ~0, worklist counters and the control
// block of the resolution kernel to 0.  The arrays are padded to a multiple of 64 words.
__global__ void __launch_bounds__(256) k_pass_reset(uint4* __restrict__ S, uint4* __restrict__ hist, uint4* __restrict__ tmin,
                                                   uint4* __restrict__ wait_pile, uint32_t n4, uint32_t* __restrict__ n_work,
                                                   uint32_t* __restrict__ ctl, uint32_t ctl_words) {
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u), ones = make_uint4(~0u, ~0u, ~0u, ~0u);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        S[i] = zero;
        hist[i] = zero;
        tmin[i] = ones;
        wait_pile[i] = ones;
    }
    if (blockIdx.x == 0) {
        if (threadIdx.x < 4) n_work[threadIdx.x] = 0u;
        for (uint32_t i = threadIdx.x; i < ctl_words; i += blockDim.x) ctl[i] = 0u;
    }
}

void launch_pass_reset(Launch& L, Peers P, ArenaLayout A, ResolveBufs rb, uint32_t* tmin, uint32_t* wait, uint32_t* ctl) {
    const uint32_t n4 = (A.n_piles + 64u) / 4u;   // every array holds n_piles + 64 words
    k_pass_reset<<<grid_for(n4, 256, kNumSMs * 4), 256, 0, L.stream>>>(
        reinterpret_cast<uint4*>(P.base[P.rank] + A.S), reinterpret_cast<uint4*>(rb.vcursor), reinterpret_cast<uint4*>(tmin),
        reinterpret_cast<uint4*>(wait), n4, rb.n_work, ctl, (uint32_t) (kResolveCtlBytes / 4));
    L.count++;
}

// the initial states of the owned piles -> every replica: one warp per owned block of 32 piles (128 contiguous bytes)
__global__ void __launch_bounds__(256) k_push_slice(Peers P, ArenaLayout A) {
    if (hdr_of(P, P.rank)->skip_pass) return;
    const uint32_t* S = section<uint32_t>(P, P.rank, A.S);
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < A.ppr; j += gridDim.x * blockDim.x) {
        const uint32_t x = owned_pile(j, (uint32_t) P.rank, (uint32_t) P.world);
        if (x >= A.n_piles) continue;
        const uint32_t v = S[x];
        for (int q = 0; q < P.world; ++q)
            if (q != P.rank) section<uint32_t>(P, q, A.S)[x] = v;
    }
}

void launch_push_slice(Launch& L, Peers P, ArenaLayout A) {
    if (P.world == 1) return;
    k_push_slice<<<grid_for(A.ppr, 256, kNumSMs * 2), 256, 0, L.stream>>>(P, A);
    L.count++;
}

// tell every replica the state of an OWNED pile (max-reduction: replicas only ever move forward)
__device__ __forceinline__ void push_state(const Peers& P, const ArenaLayout& A, uint32_t x, uint32_t val, bool& pushed) {
    if (P.world == 1) return;
    pushed = true;
    for (int q = 0; q < P.world; ++q)
        if (q != P.rank) red_max_sys(section<uint32_t>(P, q, A.S) + x, val);
}

constexpr uint32_t kNoWait = 0xFFFFFFFFu;

// Settle victim v0 (owned).  Returns false when it has to wait: for a foreign container whose fate is open, or
// because the chase budget ran out.  In the first case every pile on the chase stack is frozen until that foreign
// pile's state moves past the time in question; (pile, time) is noted for each of them (wait_pile / wait_time), so
// the next sweeps test one state word instead of walking the whole chain again only to stop at the same place.
// Replicas hear about a pile ONCE per visit: when it settles, or, if it stays open, its new lower bound when the chase
// leaves it (a bound that is overtaken by the settled state within the same visit is never sent).
__device__ __forceinline__ bool resolve_owned(const Peers& P, const ArenaLayout& A, uint32_t v0,
                                              const uint32_t* __restrict__ vstart, const uint32_t* __restrict__ seg_c,
                                              uint32_t* __restrict__ seg_t, uint32_t* __restrict__ S, uint32_t* __restrict__ wait_pile,
                                              uint32_t* __restrict__ wait_time, bool& pushed) {
    uint32_t stack_v[kChaseDepth], stack_need[kChaseDepth], stack_bound[kChaseDepth];   // bound: raised locally, not pushed yet (0: nothing)
    int sp = 0, budget = kChaseBudget;
    stack_v[0] = v0;
    stack_need[0] = kNever;
    stack_bound[0] = 0u;
    auto settle = [&](uint32_t v, uint32_t val) {
        atomicMax(&S[v], val);
        push_state(P, A, v, val, pushed);
    };
    auto leave_open = [&](int from) {   // the piles stack[from .. sp] stay open: send the bounds that were raised on the way
        for (int i = from; i <= sp; ++i)
            if (stack_bound[i]) push_state(P, A, stack_v[i], stack_bound[i], pushed);
    };
    while (sp >= 0) {
        const uint32_t v = stack_v[sp];
        const uint32_t cur = ld_relaxed_sys(&S[v]);
        if (cur & kSettled) { --sp; continue; }
        const uint32_t s0 = vstart[v], s1 = vstart[v + 1];
        uint32_t best_t = kDeadEvent, best_p = 0;
        for (uint32_t p = s0; p < s1; ++p) {
            const uint32_t t = seg_t[p];
            if (t < best_t) { best_t = t; best_p = p; }
        }
        if (best_t == kDeadEvent) {               // every event found its container dead: v is never killed
            settle(v, kSettled | kNever);
            --sp;
            continue;
        }
        if (best_t > cur) {                       // v cannot die before its earliest open event
            atomicMax(&S[v], best_t);
            stack_bound[sp] = best_t;
        }
        if (best_t > stack_need[sp]) {            // whoever asked only cares about earlier times: v stays open
            leave_open(sp);
            --sp;
            continue;
        }
        const uint32_t c = seg_c[best_p];
        const uint32_t q = c == v ? kSettled | kNever : ld_relaxed_sys(&S[c]);   // a == b record: the pile is its own (alive) container
        if (q & kSettled) {
            if ((q & kNever) > best_t) {          // container alive at best_t: the event fires
                settle(v, kSettled | best_t);
                --sp;
            } else {
                seg_t[best_p] = kDeadEvent;       // container died first: the event never fires; look again
            }
            continue;
        }
        if (q > best_t) {                         // open, but certainly alive at best_t
            settle(v, kSettled | best_t);
            --sp;
            continue;
        }
        if (pile_owner(c, (uint32_t) P.world) != (uint32_t) P.rank) {   // foreign and open: its owner will tell
            for (int i = 0; i <= sp; ++i) {
                wait_pile[stack_v[i]] = c;
                wait_time[stack_v[i]] = best_t;
            }
            leave_open(0);
            return false;
        }
        if (sp + 1 >= kChaseDepth || --budget <= 0) {
            leave_open(0);
            return false;
        }
        ++sp;
        stack_v[sp] = c;
        stack_need[sp] = best_t;
        stack_bound[sp] = 0u;
    }
    return true;
}

// ---------------------------------------------------------------------------------------------
// The resolution itself: ONE persistent kernel per rank and pass, no barrier with the peers inside.  The grid sweeps
// the worklist of open owned victims again and again; every state change is pushed to the replicas as it happens, so
// news from the peers arrives while a sweep runs, and a rank never waits for a slower peer to finish its own sweep.
// After every sweep block 0 tells the peers how many victims are still open here (tagged with the barrier epoch of the
// pass, so a value of the previous pass is never mistaken for a current one); the pass ends on a rank when every
// rank has reported zero.  A rank that has used up its sweeps with victims still open reports kGaveUp instead; a peer
// that sees it gives up too (after its current sweep, or its watching threads stop), and the pass ends on a rank when
// every rank has reported zero or kGaveUp, with FE_ROUNDS set if any gave up.  So even a pass that runs out of sweeps
// ends in step on every rank, after every push has landed: the replicas agree, the step is void but consistent, and no
// rank waits out the barrier timeout for a peer that stopped (a dead fabric lets the ranks run out of step).
// Ordering: each thread fences (system scope) after its pushes and before the grid barrier, so a peer that reads
// "0 open" (or kGaveUp) from this rank already holds every state this rank owns.
// The grid is sized to be co-resident (launch_fabric_resolve), which the software grid barrier needs.
// ---------------------------------------------------------------------------------------------
struct ResolveCtl {
    uint32_t arrived;   // grid barrier: blocks that have arrived, counts up for ever
    uint32_t released;  // grid barrier: phases released so far
    uint32_t go;        // decision of block 0 after a sweep: 1 = sweep again, 0 = the pass is over
    uint32_t sweeps;
    uint32_t settled;   // poll phase: victims whose watching thread is done with them
    uint32_t stopped;   // poll phase: a watching thread stopped because a peer gave up, its victim still open
    uint32_t pad[2];
    unsigned long long log[kSweepLog][2];   // diagnostics: (open victims at the start of the sweep, ns since the kernel started) per sweep
};
static_assert(sizeof(ResolveCtl) == kResolveCtlBytes, "fabric.cuh sizes the control block");

// `deadline` (ns, %globaltimer): a grid that is not resident as a whole, or a peer that never answers block 0, must not hang
// the GPU: after the deadline the waiting blocks mark the fabric dead and go on (the step's results are void then)
__device__ __forceinline__ void grid_barrier(ResolveCtl* ctl, uint32_t& phase, uint32_t* dead, unsigned long long deadline) {
    __syncthreads();
    if (threadIdx.x == 0) {
        phase += 1u;
        __threadfence();
        if (atomicAdd(&ctl->arrived, 1u) + 1u == phase * gridDim.x) {
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&ctl->released), "r"(phase) : "memory");
        } else {
            uint32_t seen, spins = 0;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(&ctl->released) : "memory");
                if ((++spins & 4095u) == 0u && global_timer_ns() > deadline) {
                    atomicExch(dead, 1u);
                    break;
                }
            } while ((int32_t) (seen - phase) < 0);
        }
    }
    __syncthreads();
}

constexpr uint32_t kGaveUp = 0xFFFFFFFFu;   // progress word of a rank that ran out of sweeps with victims still open

__device__ __forceinline__ void st_release_sys64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// one sweep over work list `in` (n entries) by the threads first, first + stride, ...: victims that stay open go to `out`
__device__ __forceinline__ void sweep_worklist(const Peers& P, const ArenaLayout& A, const uint32_t* __restrict__ vstart,
                                               const uint32_t* __restrict__ seg_c, uint32_t* __restrict__ seg_t, uint32_t* __restrict__ S,
                                               uint32_t* __restrict__ wait_pile, uint32_t* __restrict__ wait_time,
                                               const uint32_t* __restrict__ in, uint32_t n, uint32_t* __restrict__ out,
                                               uint32_t* __restrict__ n_out, uint32_t first_block, uint32_t n_blocks) {
    const uint32_t lane = lane_id();
    bool pushed = false;
    for (uint32_t base = first_block * blockDim.x; base < n; base += n_blocks * blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        uint32_t v = 0;
        bool keep = false;
        if (i < n) {
            v = in[i];
            const uint32_t f = wait_pile[v];
            bool frozen = false;
            if (f != kNoWait) {   // still waiting for foreign pile f to move past wait_time[v]?
                const uint32_t q = ld_relaxed_sys(&S[f]);
                frozen = !(q & kSettled) && q <= wait_time[v];
            }
            keep = frozen || !resolve_owned(P, A, v, vstart, seg_c, seg_t, S, wait_pile, wait_time, pushed);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, keep);
        if (m) {
            uint32_t gb = 0;
            if (lane == 0) gb = atomicAdd(n_out, (uint32_t) __popc(m));
            gb = __shfl_sync(0xFFFFFFFFu, gb, 0);
            if (keep) out[gb + __popc(m & ((1u << lane) - 1u))] = v;
        }
    }
    // this thread's pushes have reached the replicas before anybody hears that the sweep is over (a system-scope fence is
    // expensive: only threads that pushed something pay for it)
    if (pushed) __threadfence_system();
}

__global__ void __launch_bounds__(256) k_fabric_resolve(Peers P, ArenaLayout A, const uint32_t* __restrict__ vstart,
                                                       const uint32_t* __restrict__ seg_c, uint32_t* __restrict__ seg_t,
                                                       uint32_t* __restrict__ work0, uint32_t* __restrict__ work1,
                                                       uint32_t* __restrict__ n_work, uint32_t* __restrict__ wait_pile,
                                                       uint32_t* __restrict__ wait_time, ResolveCtl* __restrict__ ctl, int pass,
                                                       uint32_t max_sweeps, unsigned long long timeout_ns) {
    __shared__ uint32_t s_word;   // block 0: what this rank reports after a sweep (open victims, or kGaveUp)
    FabricHdr* mine = hdr_of(P, P.rank);
    if (mine->skip_pass) {
        if (blockIdx.x == 0 && threadIdx.x == 0) mine->rounds_needed[pass] = 1u;
        return;
    }
    uint32_t* S = section<uint32_t>(P, P.rank, A.S);
    const unsigned long long tag = (unsigned long long) mine->epoch << 32;   // no barrier runs on this rank while the kernel does
    const uint32_t me = (uint32_t) P.rank, W = (uint32_t) P.world;
    const unsigned long long t_start = global_timer_ns();
    uint32_t phase = 0;

    auto peer_gave_up = [&]() -> bool {
        for (uint32_t q = 0; q < W; ++q)
            if (ld_acquire_sys64(&mine->progress[q]) == (tag | kGaveUp)) return true;
        return false;
    };

    // block 0, thread 0, after a sweep that left `word` (open victims, or kGaveUp): decide.  Returns 0 = the pass is over,
    // 1 = sweep again.  (`word` was published to the peers by the lanes of warp 0, see publish_open)
    auto after_sweep = [&](uint32_t sweep, uint32_t n_before, uint32_t word) -> uint32_t {
        uint32_t go = 1u;
        bool dead = ld_relaxed_sys(&mine->dead) != 0u || global_timer_ns() - t_start > timeout_ns;
        bool gave_up = word == kGaveUp;
        if (word == 0u || gave_up) {   // everything here is settled (or given up) and pushed: wait until that is true everywhere
            while (!dead) {
                bool all = true;
                for (uint32_t q = 0; q < W; ++q) {
                    const unsigned long long p = ld_acquire_sys64(&mine->progress[q]);
                    gave_up = gave_up || p == (tag | kGaveUp);
                    all = all && (p == tag || p == (tag | kGaveUp));
                }
                if (all) break;
                __nanosleep(100);
                dead = ld_relaxed_sys(&mine->dead) != 0u || global_timer_ns() - t_start > timeout_ns;
            }
            if (gave_up) atomicOr(&mine->error, (uint32_t) FE_ROUNDS);
            go = 0u;
        }
        if (dead) {
            atomicOr(&mine->error, (uint32_t) FE_TIMEOUT);
            if (atomicExch(&mine->dead, 1u) == 0u) {
                mine->dead_epoch = mine->epoch;
                mine->dead_peer = 0xFFFFu;
            }
            go = 0u;
        }
        ctl->sweeps = sweep + 1u;
        if (sweep < (uint32_t) kSweepLog) {
            ctl->log[sweep][0] = n_before;
            ctl->log[sweep][1] = global_timer_ns() - t_start;
        }
        if (!go) mine->rounds_needed[pass] = (!gave_up && !dead) ? sweep + 1u : 0u;
        return go;
    };

    // block 0, warp 0: lane q tells rank q how many victims are still open here.  One release store per lane, all at once:
    // eight of them issued by one thread one after the other cost ~25 us per sweep on 8 GPUs (profiles/r02n)
    auto publish_open = [&](uint32_t open) {
        if (threadIdx.x < W) st_release_sys64(&hdr_of(P, (int) threadIdx.x)->progress[me], tag | open);
        __syncwarp();
    };

    const uint32_t n_threads = gridDim.x * blockDim.x, gtid = blockIdx.x * blockDim.x + threadIdx.x;
    for (uint32_t sweep = 0;; ++sweep) {
        const uint32_t n = n_work[sweep % 3u];
        if (blockIdx.x == 0 && threadIdx.x == 0) n_work[(sweep + 2u) % 3u] = 0u;   // read last in sweep - 1, written next in sweep + 1
        const uint32_t* out = (sweep & 1u) ? work0 : work1;
        sweep_worklist(P, A, vstart, seg_c, seg_t, S, wait_pile, wait_time, (sweep & 1u) ? work1 : work0, n, (sweep & 1u) ? work0 : work1,
                       &n_work[(sweep + 1u) % 3u], blockIdx.x, gridDim.x);
        grid_barrier(ctl, phase, &mine->dead, t_start + 2ull * timeout_ns);
        uint32_t open;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(open) : "l"(&n_work[(sweep + 1u) % 3u]) : "memory");
        const bool poll = open != 0u && open <= n_threads;

        if (poll) {
            // Every open victim gets a thread of its own, which watches the one foreign state its chain is frozen on and
            // goes on the moment it moves: the rest of the pass costs the longest cross-rank dependency chain (a push over
            // NVLink + a few local hops per link) instead of one whole-grid sweep, two grid barriers and the longest local
            // chase of the sweep per link (8 - 12 sweeps of 30 - 80 us on 8 GPUs, profiles/r02n).
            bool gave_up = false, stopped = false;
            if (gtid < open) {
                const uint32_t v = out[gtid];
                for (uint32_t it = 1;; ++it) {
                    if ((it & 255u) == 0u && (ld_relaxed_sys(&mine->dead) != 0u || global_timer_ns() - t_start > timeout_ns)) {
                        gave_up = true;
                        break;
                    }
                    if ((it & 255u) == 128u && peer_gave_up()) {   // the foreign state this victim waits for may never move
                        stopped = true;
                        break;
                    }
                    const uint32_t f = wait_pile[v];
                    if (f != kNoWait) {
                        const uint32_t q = ld_relaxed_sys(&S[f]);
                        if (!(q & kSettled) && q <= wait_time[v]) {
                            __nanosleep(64);
                            continue;
                        }
                    }
                    bool pushed = false;
                    const bool done = resolve_owned(P, A, v, vstart, seg_c, seg_t, S, wait_pile, wait_time, pushed);
                    if (pushed) __threadfence_system();   // before this victim counts as settled
                    if (done) break;
                }
                if (gave_up) atomicExch(&mine->dead, 1u);
                if (stopped) {
                    atomicExch(&ctl->stopped, 1u);
                    __threadfence();   // before block 0 counts this victim as done
                }
                atomicAdd(&ctl->settled, 1u);
            }
        }
        if (blockIdx.x == 0) {
            const uint32_t done_sweeps = poll ? sweep + 1u : sweep;
            if (threadIdx.x == 0) {
                if (poll) {   // all victims of this rank settled (or somebody gave up)?
                    uint32_t got;
                    do {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(got) : "l"(&ctl->settled) : "memory");
                        if (got < open) __nanosleep(100);
                    } while (got < open);
                }
                uint32_t word = poll ? (*(volatile uint32_t*) &ctl->stopped ? kGaveUp : 0u) : open;
                // victims still open after the last sweep allowed, or a peer has given up: give up too (FE_ROUNDS)
                if (word != 0u && word != kGaveUp && (done_sweeps + 1u >= max_sweeps || peer_gave_up())) word = kGaveUp;
                s_word = word;
            }
            __syncthreads();
            if (threadIdx.x < 32) publish_open(s_word);
            if (threadIdx.x == 0) {
                ctl->go = after_sweep(done_sweeps, poll ? open : n, s_word);
                __threadfence();
            }
        }
        grid_barrier(ctl, phase, &mine->dead, t_start + 2ull * timeout_ns);
        uint32_t go;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(go) : "l"(&ctl->go) : "memory");
        if (!go) break;
    }
}

int fabric_resolve_max_blocks() {
    int per_sm = 0, dev = 0, sms = kNumSMs;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fabric_resolve, 256, 0);
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (per_sm < 1) per_sm = 1;
    return per_sm * sms;
}

void launch_fabric_resolve(Launch& L, Peers P, ArenaLayout A, ResolveBufs rb, uint32_t* wait /* 2 x (n_piles + 64) words */, uint32_t* ctl,
                           int pass, uint32_t max_sweeps, unsigned long long timeout_ns, int blocks) {
    const size_t stride = (size_t) A.n_piles + 64;   // wait_pile | wait_time; launch_pass_reset cleared wait_pile and the control block
    k_fabric_resolve<<<blocks, 256, 0, L.stream>>>(P, A, rb.vstart, rb.seg_c, rb.seg_t, rb.work0, rb.work1, rb.n_work, wait, wait + stride,
                                                  reinterpret_cast<ResolveCtl*>(ctl), pass, max_sweeps, timeout_ns);
    L.count++;
}

// time bases of the local lists in the final containment pass (graph.cpp:831-866): position in the GLOBAL
// overlaps ++ internals order, from the list counts every rank published in the barrier just passed
__global__ void k_time_bases_mail(Peers P, uint32_t* __restrict__ bases) {
    if (blockIdx.x || threadIdx.x) return;
    const FabricHdr* mine = hdr_of(P, P.rank);
    const uint32_t par = mine->epoch & 1u;
    uint32_t total_ovl = 0, ovl_before = 0, int_before = 0;
    for (int q = 0; q < P.world; ++q) {
        if (q < P.rank) {
            ovl_before += mine->mail[par][q][M_NOVL];
            int_before += mine->mail[par][q][M_NINL];
        }
        total_ovl += mine->mail[par][q][M_NOVL];
    }
    bases[0] = ovl_before;
    bases[1] = total_ovl + int_before;
}

void launch_time_bases_mail(Launch& L, Peers P, uint32_t* bases) {
    k_time_bases_mail<<<1, 32, 0, L.stream>>>(P, bases);
    L.count++;
}

// ---------------------------------------------------------------------------------------------
// Build stage.  Node ids are split EVENLY over the ranks (whole reverse-complement pairs): node_begin[q] =
// min(n_nodes, q * 2 * ceil(n_nodes / 2 / world)).  The surviving piles are not spread evenly over the pile ids
// (the ordered containment favours late ids), so following the pile ownership would give the last rank several
// times the rows of the first.
// ---------------------------------------------------------------------------------------------
__global__ void k_node_bounds(Peers P, ArenaLayout A, const uint32_t* __restrict__ n_nodes_ptr, BuildMeta* __restrict__ meta) {
    const uint32_t q = threadIdx.x;
    if (q > (uint32_t) P.world) return;
    const uint32_t n_nodes = min(*n_nodes_ptr, A.n_nodes_max);
    const uint32_t per = 2u * ((n_nodes / 2u + (uint32_t) P.world - 1u) / (uint32_t) P.world);
    meta->node_begin[q] = (unsigned long long) q * per < n_nodes ? q * per : n_nodes;
}

void launch_node_bounds(Launch& L, Peers P, ArenaLayout A, const uint32_t* n_nodes_ptr, BuildMeta* meta) {
    k_node_bounds<<<1, 32, 0, L.stream>>>(P, A, n_nodes_ptr, meta);
    L.count++;
}

// zero bytes [0, *n_ptr rounded up to 16) of a 256-byte padded buffer
__global__ void k_clear_bytes16(uint8_t* __restrict__ p, const uint32_t* __restrict__ n_ptr, uint32_t cap) {
    const uint32_t n16 = (min(*n_ptr, cap) + 15u) / 16u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x)
        reinterpret_cast<uint4*>(p)[i] = make_uint4(0u, 0u, 0u, 0u);
}

void launch_clear_bytes16(Launch& L, uint8_t* p, const uint32_t* n_ptr, uint32_t cap) {
    k_clear_bytes16<<<grid_for(cap / 16 + 1, 256, kNumSMs * 2), 256, 0, L.stream>>>(p, n_ptr, cap);
    L.count++;
}

__device__ __forceinline__ uint32_t owner_of(const uint32_t* bounds, uint32_t world, uint32_t x) {   // bounds[q] <= x < bounds[q + 1]
    uint32_t q = 0;
    while (q + 1u < world && x >= bounds[q + 1u]) ++q;
    return q;
}

// Edges -> the rank that owns their source node (src | dst | len | LOCAL edge id; the receiver adds the emitting
// rank's id base, which it learns from the edge counts published in the same barrier).
__global__ void __launch_bounds__(256) k_route_edges(Peers P, ArenaLayout A, const uint32_t* __restrict__ src, const uint32_t* __restrict__ dst,
                                                    const uint32_t* __restrict__ len, const uint32_t* __restrict__ n_edges, uint32_t edge_cap,
                                                    const BuildMeta* __restrict__ meta, uint32_t* __restrict__ out_cnt) {
    __shared__ RouteSmem<4> sh;
    __shared__ uint32_t s_bounds[kMaxRanks + 1];
    if (threadIdx.x <= (uint32_t) P.world) s_bounds[threadIdx.x] = meta->node_begin[threadIdx.x];
    __syncthreads();
    const uint32_t n = min(*n_edges, edge_cap);
    for (uint32_t base = blockIdx.x * kRouteTile; base < n; base += gridDim.x * kRouteTile) {
        uint32_t dest[4], val[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint32_t e = base + r * 256u + threadIdx.x;
            dest[r] = 0xFFu;
            if (e < n) {
                val[r][0] = src[e]; val[r][1] = dst[e]; val[r][2] = len[e]; val[r][3] = e;
                dest[r] = owner_of(s_bounds, (uint32_t) P.world, val[r][0]);
            }
        }
        route_tile<4>(sh, P, A.edge_inbox, (size_t) P.rank * 4u * A.cap_edge, A.cap_edge, dest, val, out_cnt);
    }
}

void launch_route_edges(Launch& L, Peers P, ArenaLayout A, const uint32_t* src, const uint32_t* dst, const uint32_t* len,
                        const uint32_t* n_edges, uint32_t edge_cap, const BuildMeta* meta, uint32_t* out_cnt) {
    k_route_edges<<<grid_for(edge_cap, kRouteTile, kNumSMs * 4), 256, 0, L.stream>>>(P, A, src, dst, len, n_edges, edge_cap, meta, out_cnt);
    L.count++;
}

// after the edge barrier: global edge-id bases (edge counts of the emitting ranks), slice sizes (column sums of the
// send-count matrix) and slice offsets of the replicated CSR
__global__ void k_edge_meta(Peers P, ArenaLayout A, BuildMeta* __restrict__ meta, uint32_t* __restrict__ counters) {
    if (blockIdx.x || threadIdx.x) return;
    FabricHdr* mine = hdr_of(P, P.rank);
    const uint32_t par = mine->epoch & 1u;
    uint32_t base = 0, off = 0, widest = 0;
    bool overflow = false;
    for (int q = 0; q < P.world; ++q) {
        meta->eid_base[q] = base;
        base += mine->mail[par][q][M_NEDGES];
        uint32_t slice = 0, wanted = 0;
        for (int p = 0; p < P.world; ++p) {
            const uint32_t s = mine->sent[par][p][q];
            if (s > A.cap_edge) overflow = true;
            slice += min(s, A.cap_edge);
            wanted += s;
        }
        widest = max(widest, wanted);
        if (slice > A.cap_slice) { overflow = true; slice = A.cap_slice; }
        meta->off[q] = off;
        off += slice;
    }
    mine->demand[2] = widest;
    meta->eid_base[P.world] = base;
    meta->off[P.world] = off;
    if (overflow) atomicOr(&mine->error, (uint32_t) FE_INBOX);
    (void) counters;
}

void launch_edge_meta(Launch& L, Peers P, ArenaLayout A, BuildMeta* meta, uint32_t* counters) {
    k_edge_meta<<<1, 32, 0, L.stream>>>(P, A, meta, counters);
    L.count++;
}

// out-degree histogram of the owned rows over the received edges (blockIdx.y = emitting rank)
__global__ void __launch_bounds__(256) k_inbox_degree(Peers P, ArenaLayout A, const BuildMeta* __restrict__ meta, uint32_t* __restrict__ degree) {
    const FabricHdr* mine = hdr_of(P, P.rank);
    const uint32_t par = mine->epoch & 1u, from = blockIdx.y;
    const uint32_t n = min(mine->sent[par][from][P.rank], A.cap_edge);
    const uint32_t nb = meta->node_begin[P.rank], owned = meta->node_begin[P.rank + 1] - nb;
    const uint32_t* blk = section<uint32_t>(P, P.rank, A.edge_inbox) + (size_t) from * 4u * A.cap_edge;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t row = blk[i] - nb;
        if (row < owned) atomicAdd(&degree[row], 1u);
    }
}

void launch_inbox_degree(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, uint32_t* degree) {
    dim3 grid(grid_for(A.cap_edge, 256, blocks_per_source(P.world)), P.world);
    k_inbox_degree<<<grid, 256, 0, L.stream>>>(P, A, meta, degree);
    L.count++;
}

// scatter the received edges into the rows of this rank's slice of the replicated CSR (slot order inside a row is
// arbitrary, as in k_fill_csr).  col_eid[pos] = GLOBAL edge id (the transitive kernels break ties between parallel
// edges by it, graph.cpp:1291-1293, and address their result bytes with it); T[that id] is cleared on the way.
// RUNS: the emitting rank's local ids fall into several runs of global ids (EdgeRuns, staged construct)
template <bool RUNS>
__global__ void __launch_bounds__(256) k_inbox_fill(Peers P, ArenaLayout A, const BuildMeta* __restrict__ meta, uint32_t* __restrict__ cursor,
                                                   uint32_t* __restrict__ col_eid, uint8_t* __restrict__ T, const EdgeRuns* __restrict__ runs) {
    const FabricHdr* mine = hdr_of(P, P.rank);
    const uint32_t par = mine->epoch & 1u, from = blockIdx.y;
    const uint32_t n = min(mine->sent[par][from][P.rank], A.cap_edge);
    const uint32_t nb = meta->node_begin[P.rank], owned = meta->node_begin[P.rank + 1] - nb;
    const uint32_t off = meta->off[P.rank], slice = meta->off[P.rank + 1] - off, id_base = meta->eid_base[from];
    const uint32_t* blk = section<uint32_t>(P, P.rank, A.edge_inbox) + (size_t) from * 4u * A.cap_edge;
    uint2* col = section<uint2>(P, P.rank, A.col);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t row = blk[i] - nb;
        if (row >= owned) continue;
        const uint32_t p = atomicAdd(&cursor[row], 1u);
        if (p >= slice) continue;
        uint32_t e = id_base + blk[3 * (size_t) A.cap_edge + i];
        if (RUNS) {   // the last segment whose local run starts at or before the id holds it
            const uint32_t x = blk[3 * (size_t) A.cap_edge + i], W = runs->world;
            uint32_t lo = 0, hi = runs->n_seg;
            while (hi - lo > 1u) {
                const uint32_t mid = (lo + hi) >> 1;
                if (runs->lb[mid * W + from] <= x) lo = mid; else hi = mid;
            }
            e = runs->gb[lo * W + from] + (x - runs->lb[lo * W + from]);
        }
        col[off + p] = make_uint2(blk[(size_t) A.cap_edge + i], blk[2 * (size_t) A.cap_edge + i]);
        col_eid[off + p] = e;
        T[e] = 0;
    }
}

void launch_inbox_fill(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, uint32_t* cursor, uint32_t* col_eid, uint8_t* T,
                       const EdgeRuns* runs) {
    dim3 grid(grid_for(A.cap_edge, 256, blocks_per_source(P.world)), P.world);
    if (runs) k_inbox_fill<true><<<grid, 256, 0, L.stream>>>(P, A, meta, cursor, col_eid, T, runs);
    else k_inbox_fill<false><<<grid, 256, 0, L.stream>>>(P, A, meta, cursor, col_eid, T, nullptr);
    L.count++;
}

// this rank's slice -> every replica: row offsets (rebased to the slice's position) and (dst, len) entries, as
// coalesced stores; blockIdx.y = destination rank (the own replica only needs the row offsets)
__global__ void __launch_bounds__(256) k_push_csr(Peers P, ArenaLayout A, const BuildMeta* __restrict__ meta, const uint32_t* __restrict__ row_ptr_local) {
    const int q = blockIdx.y;
    const uint32_t nb = meta->node_begin[P.rank], owned = meta->node_begin[P.rank + 1] - nb;
    const uint32_t off = meta->off[P.rank], slice = meta->off[P.rank + 1] - off;
    uint32_t* rp = section<uint32_t>(P, q, A.row_ptr);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= owned; i += gridDim.x * blockDim.x)
        if (nb + i <= A.n_nodes_max) rp[nb + i] = off + min(row_ptr_local[i], slice);
    if (q == P.rank) return;
    const uint2* mine = section<uint2>(P, P.rank, A.col) + off;
    uint2* theirs = section<uint2>(P, q, A.col) + off;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < slice; i += gridDim.x * blockDim.x) theirs[i] = mine[i];
}

void launch_push_csr(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, const uint32_t* row_ptr_local) {
    dim3 grid(grid_for(A.cap_slice, 1024, blocks_per_source(P.world)), P.world);
    k_push_csr<<<grid, 256, 0, L.stream>>>(P, A, meta, row_ptr_local);
    L.count++;
}

// T(e) = 1 results of the owned candidate edges -> the rank that emitted e (its T_in byte array, indexed by local edge id)
template <bool RUNS>
__global__ void __launch_bounds__(256) k_route_marks(Peers P, ArenaLayout A, const BuildMeta* __restrict__ meta, const uint8_t* __restrict__ T,
                                                    const uint32_t* __restrict__ col_eid, const EdgeRuns* __restrict__ runs) {
    __shared__ uint32_t s_base[kMaxRanks + 1];
    if (threadIdx.x <= (uint32_t) P.world) s_base[threadIdx.x] = meta->eid_base[threadIdx.x];
    __syncthreads();
    const uint32_t off = meta->off[P.rank], slice = meta->off[P.rank + 1] - off;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < slice; p += gridDim.x * blockDim.x) {
        const uint32_t e = col_eid[off + p];
        if (!T[e]) continue;
        uint32_t r, local;
        if (RUNS) {   // the last run starting at or before e holds it (empty runs start where the next one does)
            const uint32_t W = runs->world;
            uint32_t lo = 0, hi = runs->n_seg * W;
            while (hi - lo > 1u) {
                const uint32_t mid = (lo + hi) >> 1;
                if (runs->gb[mid] <= e) lo = mid; else hi = mid;
            }
            r = lo % W;
            local = runs->lb[lo] + (e - runs->gb[lo]);
        } else {
            r = owner_of(s_base, (uint32_t) P.world, e);
            local = e - s_base[r];
        }
        if (local < A.t_cap) section<uint8_t>(P, (int) r, A.T_in)[local] = 1;
    }
}

void launch_route_marks(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, const uint8_t* T, const uint32_t* col_eid,
                        const EdgeRuns* runs) {
    if (runs) k_route_marks<true><<<grid_for(A.cap_slice, 256, kNumSMs * 4), 256, 0, L.stream>>>(P, A, meta, T, col_eid, runs);
    else k_route_marks<false><<<grid_for(A.cap_slice, 256, kNumSMs * 4), 256, 0, L.stream>>>(P, A, meta, T, col_eid, nullptr);
    L.count++;
}

// observed demands of this step, for the capacity planning of the host (max over the destinations)
__global__ void k_fabric_demand(Peers P, const uint32_t* __restrict__ ev_cnt0, const uint32_t* __restrict__ ev_cnt1,
                                const uint32_t* __restrict__ edge_cnt, const BuildMeta* __restrict__ meta) {
    if (blockIdx.x || threadIdx.x) return;
    FabricHdr* mine = hdr_of(P, P.rank);
    uint32_t ev = 0, ed = 0;
    for (int q = 0; q < P.world; ++q) {
        ev = max(ev, max(ev_cnt0[q], ev_cnt1[q]));
        ed = max(ed, edge_cnt[q]);
    }
    mine->demand[0] = ev;
    mine->demand[1] = ed;
    (void) meta;
}

void launch_demand(Launch& L, Peers P, const uint32_t* ev_cnt0, const uint32_t* ev_cnt1, const uint32_t* edge_cnt, const BuildMeta* meta) {
    k_fabric_demand<<<1, 32, 0, L.stream>>>(P, ev_cnt0, ev_cnt1, edge_cnt, meta);
    L.count++;
}

// ---------------------------------------------------------------------------------------------
// Staged construct: the host changes the pile table between the passes (hill breaking, the pit loop of graph.cpp:704-829).
// Every list pass leaves per-segment counts that all ranks need (global positions, is_changed, edge ids): each rank counts
// its own, pushes them into every peer's seg_mail section and a barrier publishes them.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_seg_count(List l, const uint32_t* __restrict__ lo, uint32_t n_seg, const uint2* __restrict__ piles,
                                                  int mode, uint32_t* __restrict__ out) {
    __shared__ uint32_t s_lo[kMaxSegs + 1], s_cnt[2 * kMaxSegs];
    for (uint32_t s = threadIdx.x; s <= n_seg; s += blockDim.x) s_lo[s] = lo[s];
    for (uint32_t s = threadIdx.x; s < 2 * n_seg; s += blockDim.x) s_cnt[s] = 0u;
    __syncthreads();
    const uint32_t n = s_lo[n_seg];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t a = 0, b = n_seg;   // segment of entry i: the last one starting at or before it
        while (b - a > 1u) {
            const uint32_t mid = (a + b) >> 1;
            if (s_lo[mid] <= i) a = mid; else b = mid;
        }
        Entry e = load_entry(l, i);
        const Pile pa = load_pile(piles, e.a), pb = load_pile(piles, e.b);
        if (!pa.alive() || !pb.alive()) continue;
        if (mode == kSegRetrim) {   // k_list_pass<kRetrim>: trim() accepts
            if (trim(e.c, e.ori, pa, pb)) atomicAdd(&s_cnt[a], 1u);
        } else {                    // k_list_pass<kFinalOvl> keeps it; k_emit_edges makes two edges of it
            const uint8_t tag = l.tag[i];
            if (tag != kA && tag != kB) atomicAdd(&s_cnt[a], 1u);
            const uint8_t t = classify(e.c, relative(e.c, e.ori, pa, pb));
            if (t == kAB || t == kBA) atomicAdd(&s_cnt[n_seg + a], 1u);
        }
    }
    __syncthreads();
    for (uint32_t s = threadIdx.x; s < 2 * n_seg; s += blockDim.x)
        if (s_cnt[s]) atomicAdd(&out[s], s_cnt[s]);
}

void launch_seg_count(Launch& L, List l, const uint32_t* lo, uint32_t n_seg, const uint2* piles, int mode, uint32_t* out) {
    k_seg_count<<<kNumSMs * 4, 256, 0, L.stream>>>(l, lo, n_seg, piles, mode, out);
    L.count++;
}

__global__ void __launch_bounds__(32) k_seg_push(Peers P, ArenaLayout A, const uint32_t* __restrict__ box, uint32_t n) {
    const int q = threadIdx.x;
    if (q >= P.world) return;
    const uint32_t par = (hdr_of(P, P.rank)->epoch + 1u) & 1u;   // the barrier that follows on this stream
    uint32_t* dst = section<uint32_t>(P, q, A.seg_mail) + ((size_t) par * kMaxRanks + (size_t) P.rank) * kSegMail;
    for (uint32_t k = 0; k < n; ++k) st_sys(dst + k, box[k]);
}

void launch_seg_push(Launch& L, Peers P, ArenaLayout A, const uint32_t* box, uint32_t n) {
    k_seg_push<<<1, 32, 0, L.stream>>>(P, A, box, n);
    L.count++;
}

__global__ void k_decode_states(Peers P, ArenaLayout A) {
    uint32_t* S = section<uint32_t>(P, P.rank, A.S);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_piles; i += gridDim.x * blockDim.x) {
        const uint32_t d = S[i] & kNever;
        S[i] = d == kNever ? kInf : d;
    }
}

void launch_decode_states(Launch& L, Peers P, ArenaLayout A) {
    k_decode_states<<<grid_for(A.n_piles, 256, kNumSMs * 4), 256, 0, L.stream>>>(P, A);
    L.count++;
}

__device__ __forceinline__ void red_add_sys(uint32_t* p, uint32_t v) {
    asm volatile("red.relaxed.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__global__ void k_push_hills(Peers P, ArenaLayout A, const uint32_t* __restrict__ cov, uint32_t n_hills) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_hills; k += gridDim.x * blockDim.x) {
        const uint32_t c = cov[k];
        if (!c) continue;
        for (int q = 0; q < P.world; ++q) red_add_sys(section<uint32_t>(P, q, A.hills) + k, c);
    }
}

void launch_push_hills(Launch& L, Peers P, ArenaLayout A, const uint32_t* cov, uint32_t n_hills) {
    if (!n_hills) return;
    k_push_hills<<<grid_for(n_hills, 256, kNumSMs), 256, 0, L.stream>>>(P, A, cov, n_hills);
    L.count++;
}

__global__ void k_final_deaths(Peers P, ArenaLayout A, uint32_t* __restrict__ dst) {
    const uint32_t* S = section<uint32_t>(P, P.rank, A.S);
    const bool skipped = hdr_of(P, P.rank)->skip_pass != 0u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_piles; i += gridDim.x * blockDim.x) dst[i] = skipped ? kInf : S[i];
}

void launch_final_deaths(Launch& L, Peers P, ArenaLayout A, uint32_t* dst) {
    k_final_deaths<<<grid_for(A.n_piles, 256, kNumSMs * 4), 256, 0, L.stream>>>(P, A, dst);
    L.count++;
}

// CUDA loads kernels lazily, at their first launch, and that load waits for the device to drain: fatal when the
// first launch of a kernel happens while another rank's barrier kernel is spinning on the same device (ranks sharing
// a GPU) — the barrier waits for this rank, this rank's kernel waits for the barrier.  rala_b200_create loads them all.
void preload_fabric() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_fabric_barrier);
    cudaFuncGetAttributes(&a, k_route_events);
    cudaFuncGetAttributes(&a, k_gather_events);
    cudaFuncGetAttributes(&a, k_fabric_prepare);
    cudaFuncGetAttributes(&a, k_push_slice);
    cudaFuncGetAttributes(&a, k_fabric_resolve);
    cudaFuncGetAttributes(&a, k_pass_reset);
    cudaFuncGetAttributes(&a, k_time_bases_mail);
    cudaFuncGetAttributes(&a, k_node_bounds);
    cudaFuncGetAttributes(&a, k_clear_bytes16);
    cudaFuncGetAttributes(&a, k_route_edges);
    cudaFuncGetAttributes(&a, k_edge_meta);
    cudaFuncGetAttributes(&a, k_inbox_degree);
    cudaFuncGetAttributes(&a, k_inbox_fill<false>);
    cudaFuncGetAttributes(&a, k_inbox_fill<true>);
    cudaFuncGetAttributes(&a, k_push_csr);
    cudaFuncGetAttributes(&a, k_route_marks<false>);
    cudaFuncGetAttributes(&a, k_route_marks<true>);
    cudaFuncGetAttributes(&a, k_fabric_demand);
    cudaFuncGetAttributes(&a, k_seg_count);
    cudaFuncGetAttributes(&a, k_seg_push);
    cudaFuncGetAttributes(&a, k_decode_states);
    cudaFuncGetAttributes(&a, k_push_hills);
    cudaFuncGetAttributes(&a, k_final_deaths);
}

}  // namespace rb
