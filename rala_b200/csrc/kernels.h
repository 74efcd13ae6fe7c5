// kernels.h — host-callable launchers of the hot-path kernels (internal to librala_b200.so).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "lists.cuh"

namespace rb {


// slots of the device-side counter block (uint32 each)
enum Counter {
    C_EV = 0,       // containment events of the current resolution
    C_HILL,         // records touching a pile with hills
    C_ROUNDS,       // fixed-point rounds
    C_NODES,        // nodes_.size()
    C_ALIVE,        // alive piles
    C_DOVETAILS,    // dovetail overlaps = edges / 2
    C_EDGES,        // edges_.size()
    C_PAIRS,        // marked pairs
    C_HEAVY_NODES, C_HEAVY,   // nodes handed to k_transitive_heavy and their work items (one 64-bit word, see heavy_append)
    C_HOP_LO, C_HOP_HI,   // two-hop visits (64-bit)
    C_TBASE_OVL, C_TBASE_INL,     // multi-GPU: global time bases of the local lists in the final pass
    C_EV_FIRST, C_ROUNDS_FIRST,   // events / rounds of the first-pass resolution (C_EV / C_ROUNDS are reused by the final pass)
    C_OVERFLOW,     // some list hit its capacity
    C_LIST0,        // 16 rotating list-count slots follow
    C_COUNT = C_LIST0 + 16
};
static_assert(C_HEAVY_NODES % 2 == 0 && C_HOP_LO % 2 == 0, "64-bit counters sit on 8-byte boundaries");

struct Launch {
    cudaStream_t stream;
    uint64_t count;   // kernels launched so far
    // forked work inside one step (also inside a stream capture: the side streams join the capture through the
    // fork event and are joined back before it ends): [0] results written to the caller's memory while the
    // transitive pass runs, [1] kernels that do not depend on each other
    cudaStream_t side[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork[2] = {nullptr, nullptr}, ev_join[2] = {nullptr, nullptr};
};

// grid of a grid-stride kernel: one block per per_block items, at least 1, at most max_blocks
inline int grid_for(uint64_t n, int per_block, int max_blocks) {
    uint64_t b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return (int) (b < (uint64_t) max_blocks ? b : (uint64_t) max_blocks);
}

// side[k] continues from the current end of the main stream; false when the context has no side streams
inline bool fork_side(Launch& L, int k) {
    if (!L.side[k]) return false;
    if (cudaEventRecord(L.ev_fork[k], L.stream) != cudaSuccess) return false;
    return cudaStreamWaitEvent(L.side[k], L.ev_fork[k], 0) == cudaSuccess;
}
// the main stream waits for everything enqueued on side[k]
inline void join_side(Launch& L, int k) {
    cudaEventRecord(L.ev_join[k], L.side[k]);
    cudaStreamWaitEvent(L.stream, L.ev_join[k], 0);
}

// classify.cu
void launch_records_to_soa(Launch& L, const uint32_t* aos, uint32_t n, List recs);
void launch_unpack_records(Launch& L, const uint32_t* query_id, const uint32_t* group_end, uint32_t n_groups, const uint32_t* a_span,
                           const uint32_t* b_span, uint32_t n, List recs);
void launch_classify_events(Launch& L, List recs, uint32_t n, uint32_t t0, const uint2* piles, uint32_t n_piles,
                            Events ev, uint32_t ev_cap, unsigned long long* first, uint32_t* hill_rec, uint32_t hill_cap, uint32_t* counters);
// the survivors in file order straight into `overlaps` / `internals` with their counts; the look-back takes one status word
// per run of classify_num_runs(n)
void launch_classify_survivors(Launch& L, List recs, uint32_t n, const uint2* piles, const uint32_t* alive_bits, uint32_t n_piles,
                               List ovl, uint32_t* n_ovl, List inl, uint32_t* n_inl, uint32_t cap, unsigned long long* status,
                               uint32_t* ticket);
uint32_t classify_num_runs(uint32_t n);
void launch_hill_coverage(Launch& L, List recs, uint32_t t0, const uint2* piles, const uint32_t* hill_rec,
                          uint32_t hill_cap, const uint32_t* hill_pile, const uint32_t* hill_begin,
                          const uint32_t* hill_end, uint32_t n_hills, uint32_t* hill_cov, const uint32_t* dbuf,
                          const uint32_t* counters);
// what the first pass's k_apply_deaths clears for the final pass: `first` (n_first words) to all ones, counters[C_EV] to
// zero after C_EV / C_ROUNDS went to C_EV_FIRST / C_ROUNDS_FIRST.  counters == nullptr: nothing.
struct FinalPassReset {
    unsigned long long* first = nullptr;
    uint32_t n_first = 0;
    uint32_t* counters = nullptr;
};
// skip: optional device flag, non-zero = do nothing (multi-GPU: a containment pass without events); run_if: optional device
// count, zero = do nothing (single GPU: the final containment pass when it has no events).  reset is done in either case.
void launch_apply_deaths(Launch& L, uint2* piles, uint32_t* dbuf, uint32_t n_piles, uint32_t* alive_bits, bool decode,
                         const uint32_t* skip = nullptr, const uint32_t* run_if = nullptr, FinalPassReset reset = {});
// the device state a step starts from, in one launch: the pile table restored from piles_initial (snapshot: the other
// way), the earliest events (n_first words) all ones, and the zero[k] regions (counters, hill coverage, look-back pool,
// slot degrees, transitive work counters) cleared; a null region is left alone
struct StepPrologue {
    static constexpr int kZero = 5;
    uint2 *piles, *piles_initial;
    uint32_t n_piles;
    bool snapshot;
    unsigned long long* first;
    uint32_t n_first;
    uint32_t* zero[kZero];
    size_t zero_words[kZero];
};
void launch_step_prologue(Launch& L, const StepPrologue& p);
void launch_list_pass(Launch& L, int mode, List in, const uint32_t* n_in, uint32_t in_cap, const uint2* piles, List out_a,
                      uint32_t* n_out_a, List out_b, uint32_t* n_out_b, const uint32_t* b_base, uint32_t cap,
                      const uint32_t* dbuf, const uint32_t* time_base, unsigned long long* status, uint32_t* ticket);
void launch_classify_final(Launch& L, List ovl, const uint32_t* n_ovl, const uint32_t* ovl_time_base, List inl,
                           const uint32_t* n_inl, const uint32_t* inl_time_base, uint32_t cap, const uint2* piles, Events ev,
                           uint32_t ev_cap, unsigned long long* first, uint32_t* counters);
void launch_trim_classify_aos(Launch& L, uint32_t* rec, uint32_t n, const uint2* piles, uint32_t n_piles, uint8_t* type_out);
void launch_pack_piles(Launch& L, const uint2* in, const uint8_t* flags, uint2* out, uint32_t n);
void launch_unpack_piles(Launch& L, const uint2* in, uint2* out, uint32_t n);
void launch_list_to_aos(Launch& L, List l, const uint32_t* n_ptr, uint32_t cap, uint32_t* out);
void launch_aos_to_list(Launch& L, const uint32_t* aos, uint32_t n, const uint2* piles, uint32_t n_piles, List l);
void launch_list_connections(Launch& L, List l, const uint32_t* n_ptr, uint32_t cap, uint32_t* out);

// containment.cu
// The classify kernels (and launch_events_first) keep every victim's earliest event in `first` (an atomicMin of
// t << 32 | container; all ones = no event: clear to all ones before).  launch_resolve settles the victims that event
// settles alone and groups the events of the others ("hard" victims, dense indices 0 .. n_work[0] - 1) by victim.
struct ResolveBufs {
    uint32_t* S;         // n_piles: state during the resolution, death times (kInf = never) afterwards
    unsigned long long* first;   // n_piles: earliest event per pile; after k_resolve_fast, the hard victims' segment bounds
                                 // by pile (uint2 {begin, end}) for k_resolve
    uint32_t* hidx;      // n_piles: dense index of a hard victim (the event filter's segment)
    uint32_t* vcursor;   // n_piles + 1: events per segment (hard victim; multi-GPU fabric: pile), then a copy of vstart
    uint32_t* vstart;    // n_piles + 1: segment offsets
    uint32_t *work0, *work1;   // n_piles each
    uint32_t* n_work;    // 4 words: [0..2] rotating worklist counters (the first = hard victims), [3] events of hard victims
    unsigned long long* seg;   // event capacity: events of the hard victims by segment, t << 32 | container
    uint4* hev;          // event capacity: events of the hard victims before the scatter {dense index, rank in segment, t, c}
    uint32_t *seg_c, *seg_t;   // multi-GPU fabric: per-pile segments, container and time columns (in seg's memory)
};
int resolve_max_blocks();
void launch_events_first(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, unsigned long long* first);
// decode = false leaves the resolution's state encoding in rb.S: the following launch_apply_deaths(decode = true) turns
// it into death times while it applies them (one launch less when nothing reads the death times in between)
// skip_if_empty: with no events at all every kernel returns at once (nobody dies; rb.S is left as it is)
void launch_resolve(Launch& L, Events ev, const uint32_t* n_events, uint32_t ev_cap, ResolveBufs rb, uint32_t n_piles,
                    uint32_t* counters, unsigned long long* status, uint32_t* ticket, int coop_blocks, bool decode,
                    bool skip_if_empty = false);

// graph_build.cu
// live: optional device count, only the first *live + 1 values are scanned
void launch_scan_u32(Launch& L, uint32_t* values_inout, uint32_t* exclusive_out, uint32_t n, unsigned long long* status,
                     uint32_t* ticket, const uint32_t* skip = nullptr, const uint32_t* run_if = nullptr, const uint32_t* live = nullptr);
struct GraphArrays {
    uint32_t* seq_to_node;   // n_piles
    uint32_t *src, *dst, *len;   // edge id order
    uint32_t* row_ptr;       // n_nodes_max + 1
    uint32_t* cursor;        // n_nodes_max + 1: fill cursor (the degree histogram first, on the paths that fill with k_fill_csr)
    uint32_t* slot_degree;   // 2 per pile: out-degree of slot 2x + s = node 2 rank(x) + s (k_count_edges -> k_scan_piles)
    uint2* col;              // CSR (dst, len)
    uint32_t* col_eid;       // CSR edge id
    uint8_t* T;              // per edge: transitive test passed
    uint8_t* marked;         // per edge: removed
};
// Edges of the final `overlaps` (graph.cpp:552-632) in two launches, with node ids and, when g.cursor is set, the CSR rows:
//   launch_count_scan  slot degrees and per-tile dovetail counts (k_count_edges), then one look-back over the piles for
//                      seq_to_node, C_NODES / C_ALIVE, row_ptr + cursor, and the edge-id bases of the list tiles with
//                      C_DOVETAILS / C_EDGES / C_OVERFLOW (k_scan_piles).  slot_degree must be zero on entry.
//   launch_emit_edges  the edge columns, and with g.cursor set the CSR slots and T cleared (k_emit_edges)
// g.cursor == nullptr switches the CSR outputs off (multi-GPU: the edges are routed to the owners of their source nodes).
// tile_dov holds emit_tiles(cap) words.  The look-back needs the scan state of n_piles.
// list entries per thread of k_count_edges / k_emit_edges (their tiles are 256 x this).  4 entries (64 registers, 4 blocks per
// SM, a small spill) measured +17 us per step and 1 entry (8 blocks per SM) +11 us against 2 at 5 blocks (profiles/r02am_*)
constexpr int kEmitItems = 2;
inline uint64_t emit_tiles(uint64_t cap) { return (cap + 256 * kEmitItems - 1) / (256 * kEmitItems); }
void launch_count_scan(Launch& L, List ovl, const uint32_t* n_ptr, uint32_t cap, const uint2* piles, uint32_t n_piles, GraphArrays g,
                       uint32_t edge_cap, uint32_t* tile_dov, uint32_t* counters, unsigned long long* status, uint32_t* ticket);
void launch_emit_edges(Launch& L, List ovl, const uint32_t* n_ptr, uint32_t cap, const uint2* piles, GraphArrays g, uint32_t edge_cap,
                       const uint32_t* tile_base);
void launch_pack_edges(Launch& L, cudaStream_t stream, GraphArrays g, uint32_t edge_cap, const uint32_t* n_edges_ptr, uint32_t* out);
// degree histogram for an edge list that did not come from emit_edges (stateless transitive stage)
void launch_degree_hist(Launch& L, const uint32_t* src, const uint32_t* n_edges_ptr, uint32_t edge_cap, uint32_t* cursor);
void launch_export_padded(Launch& L, const uint32_t* c0, const uint32_t* c1, const uint32_t* c2, const uint32_t* n_ptr,
                          uint32_t src_cap, uint32_t cap, uint32_t* block);
void launch_import_gathered(Launch& L, const uint32_t* gathered, uint32_t cap, uint32_t world, uint32_t* d0, uint32_t* d1,
                            uint32_t* d2, uint32_t dst_cap, uint32_t* n_out, uint32_t* overflow);
void launch_time_bases(Launch& L, const uint32_t* counts, uint32_t rank, uint32_t world, uint32_t* bases);
// host-facing adjacency view: ids of the (unmarked) edges per node, ascending edge id; key = src (suffix) or dst (prefix) column
void launch_adjacency_view(Launch& L, const uint32_t* key, const uint8_t* marked, const uint32_t* n_edges_ptr, uint32_t edge_cap,
                           uint32_t n_nodes, uint32_t* degree_cursor, uint32_t* row_ptr, uint32_t* ids_tmp, uint32_t* ids_sorted,
                           unsigned long long* status, uint32_t* ticket);
// CSR of an edge list that did not come from emit_edges: g.cursor holds its degree histogram (launch_degree_hist)
void launch_build_csr(Launch& L, GraphArrays g, uint32_t n_nodes_max, uint32_t edge_cap, uint32_t* counters,
                      unsigned long long* status, uint32_t* ticket);

// transitive.cu
// nodes of the transitive pass that one block per work item takes (k_transitive_heavy): one entry per node, so a list
// of n_nodes_max entries never overflows; unit_base[i] = work items of the entries before i (ascending in i)
struct HeavyItems {
    uint32_t *node, *unit_base;
    uint32_t cap;
};
// node_range: device {begin, end} of the source nodes to evaluate; nullptr = all of them
void launch_transitive(Launch& L, GraphArrays g, uint32_t n_nodes_max, HeavyItems heavy, uint32_t* work_counter, uint32_t* counters,
                       const uint32_t* node_range);
void launch_node_range(Launch& L, GraphArrays g, const uint32_t* counters, uint32_t rank, uint32_t world, uint32_t* out);
void launch_finalize_marks(Launch& L, GraphArrays g, uint32_t edge_cap, uint32_t* counters, uint8_t* marked_copy /* nullable */,
                           uint32_t copy_cap);

// force-load every kernel of a translation unit (CUDA's lazy loading otherwise loads at the first launch, which waits
// for the device to drain: a deadlock next to a spinning barrier kernel, see fabric.cu)
void preload_classify();
void preload_containment();
void preload_graph_build();
void preload_transitive();
void preload_fabric();
void preload_frontend();
void preload_paf();
void preload_piles();
void preload_reads();
void preload_bgzf();
void preload_gzip();

// frontend.cu
void launch_filter_duplicates(Launch& L, const uint32_t* a, const uint32_t* b, const uint32_t* len, uint32_t n, uint8_t* valid);

}  // namespace rb
