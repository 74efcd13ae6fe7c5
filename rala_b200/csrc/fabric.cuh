// fabric.cuh — the multi-rank exchange layer: every rank owns one ARENA of device memory whose layout is identical on
// all ranks, and holds a device pointer to the arena of every peer (NVLink peer memory: cudaDeviceEnablePeerAccess in
// one process, cudaIpcOpenMemHandle between processes; plain pointers when several ranks share a device in the tests).
// All data-path exchanges are PUSHES by the producing kernel straight into the consumer's arena (remote stores /
// remote atomics over NVLink), separated by a flag barrier (k_fabric_barrier): no staging copy, no host
// synchronisation, no library collective inside a step.
//
// What is exchanged (reference: none — rvaser/rala is single-process; partition per BASELINE.json north_star):
//   containment events -> owner of the victim pile     (ordered containment, graph.cpp:469-480 / 831-866)
//   pile states        -> every rank                    (death times: every rank filters its own records with them)
//   edges              -> owner of the source node      (adjacency rows, graph.cpp:576-632)
//   built CSR slices   -> every rank                    (two-hop lookups of graph.cpp:1281-1318 cross shards)
//   transitive marks   -> the rank that emitted the edge (marked(e) = T(e) | T(e ^ 1), graph.cpp:1305-1309)
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"
#include "lists.cuh"

namespace rb {

constexpr int kMaxRanks = 16;
constexpr int kMailSlots = 8;
constexpr int kBarrierLog = 128;
constexpr int kSweepLog = 48;
constexpr int kResolveCtlBytes = 32 + kSweepLog * 16;
// Staged construct (pile table changed by the host between the passes): the promotions of a pit round are appended to the
// end of the GLOBAL `overlaps`, so a rank's local list is a run of SEGMENTS (segment 0: its entries of the first pass,
// segment k: what it promoted in the k-th round that promoted anything), at most kMaxSegs of them.
constexpr int kMaxSegs = 64;
constexpr int kSegMail = 2 * kMaxSegs + 4;   // words one rank sends every peer after a staged list pass

// mail slots: small scalars a rank publishes to every peer inside a barrier
enum Mail { M_UNSETTLED = 0, M_NOVL, M_NINL, M_NEDGES, M_SENT_TO_YOU, M_EMITTED, M_SPARE1, M_SPARE2 };

enum FabricError : uint32_t {
    FE_TIMEOUT = 1u,     // a peer did not reach a barrier in time
    FE_ROUNDS = 2u,      // the containment resolution needed more rounds than the step was built with
    FE_INBOX = 4u,       // an inbox / slice capacity was exceeded
};

// At offset 0 of every arena; zeroed when the arena is allocated.
struct FabricHdr {
    uint32_t flag[kMaxRanks];                       // flag[q]: last barrier epoch peer q has entered (written by q)
    uint32_t epoch;                                 // barriers this rank has passed
    uint32_t error;                                 // FabricError bits
    uint32_t rounds_needed[2];                      // per resolution pass: rounds until no rank had an open victim
    uint32_t demand[4];                             // observed: events sent to one peer, edges sent to one peer, slice size, (spare)
    uint32_t dead;                                  // sticky: a barrier timed out; later barriers do not wait any more (cleared by a new reservation)
    uint32_t dead_epoch, dead_peer;                 // which barrier / which peer timed out first (diagnostics)
    uint32_t skip_pass;                             // no rank has a containment event in the current pass: its kernels and barriers return at once
    uint32_t pad[4];
    uint32_t mail[2][kMaxRanks][kMailSlots];        // [epoch parity][source rank][slot]
    uint32_t sent[2][kMaxRanks][kMaxRanks];         // [epoch parity][source rank][destination]: edges routed src -> dst
    unsigned long long progress[kMaxRanks];         // progress[q]: (epoch of the pass << 32 | victims still open on rank q), written by q after every sweep
    unsigned long long tlog[kBarrierLog][2];        // ring by epoch: %globaltimer when the barrier kernel started / when every peer had arrived
};

struct Peers {
    uint8_t* base[kMaxRanks];
    int rank, world;
};

// Byte offsets of the arena sections (same on every rank).
struct ArenaLayout {
    size_t ev_inbox;      // world blocks of 3 * cap_ev words: victim | container | time, block index = source rank
    size_t edge_inbox;    // world blocks of 4 * cap_edge words: src | dst | len | local edge id
    size_t S;             // n_piles words: pile states (containment.cu encoding), replicated
    size_t T_in;          // t_cap bytes: transitive test results for the edges THIS rank emitted, written by their evaluators
    size_t row_ptr;       // n_nodes_max + 2 words: CSR row offsets of the whole graph
    size_t col;           // world * cap_slice x (dst, len): CSR of the whole graph, slices in rank order
    size_t seg_mail;      // [2 epoch parities][kMaxRanks source ranks][kSegMail] words: per-segment list counts of a staged pass
    size_t hills;         // n_hills words: hill counters summed over the ranks (remote reductions of the first pass)
    size_t total;
    uint32_t cap_ev, cap_edge, cap_slice, t_cap;
    uint32_t n_piles, n_nodes_max, n_hills;
    uint32_t ppr;         // piles per rank, rounded up to whole blocks of 32 (sizes the per-rank loops)
    uint32_t npr_max;     // upper bound of the nodes one rank owns (sizes the row scan)
};

// Piles are owned BLOCK-CYCLICALLY, 32 piles per block: owner(x) = (x / 32) % world.  Ranges of ids would be simpler,
// but ids correlate with file order (a pair is listed under its lower id), so the low range would resolve almost
// everything locally while the high range waits for it, and the surviving piles pile up in the high range
// (profiles/r02g: 2.5 x the work on the last rank).  One block = 128 contiguous bytes of every per-pile array.
__host__ __device__ __forceinline__ uint32_t pile_owner(uint32_t x, uint32_t world) { return (x >> 5) % world; }
// j-th pile slot owned by `rank` (j = 0 .. ppr): may be >= n_piles in the last block
__host__ __device__ __forceinline__ uint32_t owned_pile(uint32_t j, uint32_t rank, uint32_t world) {
    return ((j >> 5) * world + rank) * 32u + (j & 31u);
}

// values published by a rank when it enters a barrier
struct Publish {
    const uint32_t* scalar[kMailSlots];   // device scalars -> mail[parity][me][k] on every peer (nullptr: skip)
    const uint32_t* per_dst;              // world entries: element q -> mail[parity][me][M_SENT_TO_YOU] on peer q
    const uint32_t* bcast;                // world entries: the whole vector -> sent[parity][me][*] on every peer
    int bookkeeping;                      // 0 none; 1 after a resolution round: record rounds_needed[pass], flag FE_ROUNDS on the last round;
                                          // 2 after the events of a pass were routed: set skip_pass when no rank emitted any
    int pass, round, last_round;
    int skippable;                        // belongs to a pass that is skipped when it has no events (skip_pass)
    unsigned long long timeout_ns;        // how long to wait for a peer before the fabric is declared dead
};

// device-side meta data of the build stage, computed by k_edge_meta after the edge barrier
struct BuildMeta {
    uint32_t eid_base[kMaxRanks + 1];   // global id of the first edge emitted by rank p
    uint32_t off[kMaxRanks + 1];        // start of rank p's slice in the replicated CSR
    uint32_t node_begin[kMaxRanks + 1]; // first node owned by rank p
};

// Global edge ids of a staged construct: the dovetails of run (segment s, rank r) are edges [gb[i], gb[i] + 2 x count) with
// i = s * world + r, and rank r emitted them as its local edges [lb[i], ...).  Runs are in global id order (segment-major).
struct EdgeRuns {
    uint32_t n_seg, world;
    uint32_t gb[kMaxSegs * kMaxRanks];
    uint32_t lb[kMaxSegs * kMaxRanks];
};

// launchers (fabric.cu)
void launch_fabric_barrier(Launch& L, Peers P, Publish pub);
void launch_route_events(Launch& L, Peers P, ArenaLayout A, Events ev, const uint32_t* n_events, uint32_t ev_cap, uint32_t* out_cnt);
void launch_gather_events(Launch& L, Peers P, ArenaLayout A, Events ev, uint32_t ev_cap, uint32_t* n_events_out, uint32_t* vcount,
                          uint32_t* tmin);
const uint32_t* skip_flag(const Peers& P);   // device address of this rank's skip_pass word
void launch_fabric_prepare(Launch& L, Peers P, ArenaLayout A, Events ev, const uint32_t* n_events, uint32_t ev_cap, ResolveBufs rb,
                           const uint32_t* tmin);
void launch_push_slice(Launch& L, Peers P, ArenaLayout A);
// before the events of a pass are routed: clears the replica's pile states, the victim histogram, tmin, the wait notes,
// the worklist counters and the resolution kernel's control block (ctl: kResolveCtlBytes)
void launch_pass_reset(Launch& L, Peers P, ArenaLayout A, ResolveBufs rb, uint32_t* tmin, uint32_t* wait, uint32_t* ctl);
// ctl: kResolveCtlBytes zeroable bytes of device memory per rank and pass; blocks: co-resident grid size (fabric_resolve_max_blocks() shared
// between the ranks that live on one device)
void launch_fabric_resolve(Launch& L, Peers P, ArenaLayout A, ResolveBufs rb, uint32_t* wait /* 2 x (n_piles + 64) words */, uint32_t* ctl,
                           int pass, uint32_t max_sweeps, unsigned long long timeout_ns, int blocks);
int fabric_resolve_max_blocks();
void launch_time_bases_mail(Launch& L, Peers P, uint32_t* bases);
void launch_node_bounds(Launch& L, Peers P, ArenaLayout A, const uint32_t* n_nodes_ptr, BuildMeta* meta);
void launch_clear_bytes16(Launch& L, uint8_t* p, const uint32_t* n_ptr, uint32_t cap);
void launch_route_edges(Launch& L, Peers P, ArenaLayout A, const uint32_t* src, const uint32_t* dst, const uint32_t* len,
                        const uint32_t* n_edges, uint32_t edge_cap, const BuildMeta* meta, uint32_t* out_cnt);
void launch_edge_meta(Launch& L, Peers P, ArenaLayout A, BuildMeta* meta, uint32_t* counters);
void launch_inbox_degree(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, uint32_t* degree);
// runs: nullptr = one contiguous id range per emitting rank (meta->eid_base); otherwise the runs of a staged construct
void launch_inbox_fill(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, uint32_t* cursor, uint32_t* col_eid, uint8_t* T,
                       const EdgeRuns* runs);
void launch_push_csr(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, const uint32_t* row_ptr_local);
void launch_route_marks(Launch& L, Peers P, ArenaLayout A, const BuildMeta* meta, const uint8_t* T, const uint32_t* col_eid,
                        const EdgeRuns* runs);
void launch_demand(Launch& L, Peers P, const uint32_t* ev_cnt0, const uint32_t* ev_cnt1, const uint32_t* edge_cnt, const BuildMeta* meta);

// staged construct
enum SegCountMode { kSegRetrim = 0, kSegFinal = 1 };
// per-segment counts of a local list whose segment s is entries [lo[s], lo[s + 1]): kSegRetrim -> out[s] = entries a retrim keeps;
// kSegFinal -> out[s] = entries the final filter keeps, out[n_seg + s] = dovetails that become edges.  out must be zeroed.
void launch_seg_count(Launch& L, List l, const uint32_t* lo, uint32_t n_seg, const uint2* piles, int mode, uint32_t* out);
// box[0 .. n) -> seg_mail[parity of the next barrier][this rank] of every rank (the barrier that follows publishes it)
void launch_seg_push(Launch& L, Peers P, ArenaLayout A, const uint32_t* box, uint32_t n);
// the replica's settled pile states -> death times (kInf = never) in place, before the deaths are applied
void launch_decode_states(Launch& L, Peers P, ArenaLayout A);
// this rank's hill counters added into every rank's hills section (zeroed before the events barrier of the same pass)
void launch_push_hills(Launch& L, Peers P, ArenaLayout A, const uint32_t* cov, uint32_t n_hills);
// death times of the final pass -> dst (kInf everywhere when the pass was skipped for want of events)
void launch_final_deaths(Launch& L, Peers P, ArenaLayout A, uint32_t* dst);

}  // namespace rb
