// session.h — internal state of librala_b200.so shared by api.cu (single-GPU session, C ABI) and multi_api.cu
// (multi-rank orchestration over peer memory).  Not part of the public interface (include/rala_b200.h).
#pragma once

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/rala_b200.h"
#include "kernels.h"
#include "lists.cuh"

using namespace rb;

struct rala_b200_ctx {
    bool owns_stream = true;
    cudaEvent_t ev[2]{};
    int device = 0;
    Launch L{nullptr, 0};
    std::string error;
    int coop_blocks = 0;
};

inline int fail(rala_b200_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->error = buf;
    return code;
}

#define CU(ctx, call)                                                                                   \
    do {                                                                                                \
        cudaError_t err__ = (call);                                                                     \
        if (err__ != cudaSuccess)                                                                       \
            return fail((ctx), RALA_B200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), \
                        __FILE__, __LINE__);                                                            \
    } while (0)

// ---------------------------------------------------------------------------------------------
// device buffer helper
// ---------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    cudaError_t reserve(size_t want) {
        if (want <= bytes) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct ListBuf {
    DevBuf buf;
    List view{};
    cudaError_t reserve(uint32_t cap) {
        size_t col = align_up((size_t) cap * 4, 256);
        cudaError_t e = buf.reserve(col * 6 + align_up(cap, 256));
        if (e != cudaSuccess) return e;
        char* b = buf.as<char>();
        view.a = (uint32_t*) b;
        view.b = (uint32_t*) (b + col);
        view.ab = (uint32_t*) (b + 2 * col);
        view.ae = (uint32_t*) (b + 3 * col);
        view.bb = (uint32_t*) (b + 4 * col);
        view.be = (uint32_t*) (b + 5 * col);
        view.tag = (uint8_t*) (b + 6 * col);
        return cudaSuccess;
    }
};

// the overlap text a session's records were parsed from (paf.cu); build_piles names refused records by its lines
enum TextFormat : uint8_t { kTextNone = 0, kTextPaf, kTextMhap };

// how far the session's stages got on the current inputs
enum SessionState { SS_EMPTY = 0, SS_INPUTS, SS_CLASSIFIED, SS_FINALIZED, SS_BUILT, SS_REDUCED };

enum StepCleared : uint32_t { kStepBuild = 1, kStepTransitive = 2 };

enum Stage { ST_CLASSIFY = 0, ST_RETRIM, ST_FINALIZE, ST_BUILD, ST_TRANSITIVE, ST_K1_KERNEL, ST_K1B_KERNEL, ST_K3_KERNELS, ST_K1S_KERNEL };

struct rala_b200_graph {
    rala_b200_ctx* ctx = nullptr;
    // inputs
    DevBuf rec;        // the host's rala_ovl_t rows as uploaded (staging of the transpose)
    ListBuf recs;      // device-resident records: six columns, 24 B / record (classify.cu)
    DevBuf alive_bits; // one bit per pile: alive after the last containment resolution
    uint32_t n_rec = 0;
    DevBuf piles, piles_raw, pile_flags_raw, piles_initial;
    bool piles_fresh = false;       // set_piles since the last classify
    uint32_t n_piles = 0;
    DevBuf hills;   // 4 columns of n_hills: pile begin end cov
    uint32_t n_hills = 0;
    // lists
    uint32_t cap = 0;      // capacity of every overlap list
    uint32_t ev_cap = 0;   // capacity of the event arrays and victim segments (multi-GPU: events of ALL ranks)
    int rank = 0, world = 1;   // multi-GPU: which share of the source nodes the transitive phase takes
    uint32_t t0 = 0;       // global time (file position) of the first local record (multi-GPU shards)
    ListBuf ovl[2], inl[2];
    int ovl_cur = 0, inl_cur = 0;
    int slot_ovl = C_LIST0, slot_inl = C_LIST0 + 1, next_slot = C_LIST0 + 2;
    DevBuf events, hill_rec;
    DevBuf dbuf, flags, segs;   // dbuf: S | vcursor | vstart | work0 | work1 | hidx | first (2 strides) ; segs: seg | hev
    DevBuf counters;
    // look-back status words: one region per step, zeroed by the step prologue (phase_events) and handed out in order by
    // scan_state; words [scan_used, scan_pool_words) are zero while scan_zeroed holds
    DevBuf scan_pool;
    size_t scan_pool_words = 0, scan_used = 0;
    bool scan_zeroed = false;
    // counters and buffers of a later stage the step prologue cleared and no stage has used since (kStep*): that stage
    // skips its own clears
    uint32_t step_cleared = 0;
    // graph
    DevBuf edges_aos;
    DevBuf seq_to_node, edges, row_ptr, cursor, col, col_eid, T, marked, heavy, work_counter;
    DevBuf slot_degree;   // 2 per pile: out-degrees of the node slots (k_count_edges -> k_scan_piles)
    DevBuf tile_dov;      // per tile of the list: dovetails, then the tile's edge-id base (k_count_edges -> k_scan_piles -> k_emit_edges)
    uint32_t edge_cap = 0, heavy_cap = 0, n_nodes_max = 0;
    // results written straight into the caller's memory by the run (rala_b200_graph_set_outputs)
    uint32_t* out_edges = nullptr;   // device-visible address of the caller's rala_edge_t rows
    uint8_t* out_marked = nullptr;
    uint32_t out_edges_cap = 0, out_marked_cap = 0;
    bool in_run = false;             // build is part of a whole run: the edge download may overlap the transitive pass
    bool download_pending = false;   // side stream 0 is still writing edges: joined at the end of the transitive stage
    // bookkeeping
    int final_time_base_slot = C_LIST0;   // counter slot holding the time base of `internals` in the final pass
    bool final_lists_ready = true;  // after finalize: have the filtered lists of graph.cpp:867-877 been written out?
    bool piles_dirty = true;        // pile table changed since the lists were last trimmed against it
    bool skip_clean_retrim = true;  // re-trimming against an unchanged table is the identity: skip the pass
    bool promote_pending = true;    // the table changed since the internals were last TYPED against it (retrim() trims but does not
                                    // re-type them): the next retrim_promote must run even if retrim() already cleared piles_dirty
    bool scan_pool_exhausted = false;   // a look-back kernel asked for more status words than the pool holds: the run is void
    SessionState state = SS_EMPTY;
    uint32_t retrim_passes = 0;
    cudaEvent_t ev_start[RALA_B200_N_STAGES]{}, ev_stop[RALA_B200_N_STAGES]{};
    bool ev_valid[RALA_B200_N_STAGES]{};
    // rala_b200_graph_run as a replayed CUDA graph (see run_key / RunGraph below)
    bool use_cuda_graph = true, capturing = false;
    struct RunGraph* run_graphs = nullptr;   // two cached instances: first run after set_piles / repeated run
    struct PafReader* paf = nullptr;         // read-name table and text upload buffers (paf.cu), from the first set_reads*
    TextFormat text_records = kTextNone;     // the records came from set_overlaps_paf / _mhap: its parsed columns are still there
    struct PileBuilder* pile_builder = nullptr;   // event, sort and run buffers of build_piles (piles.cu)

    uint32_t* cnt() const { return counters.as<uint32_t>(); }
    Events events_view() const {
        Events e;
        size_t col = align_up((size_t) ev_cap * 4, 256);
        char* b = events.as<char>();
        e.v = (uint32_t*) b;
        e.c = (uint32_t*) (b + col);
        e.t = (uint32_t*) (b + 2 * col);
        return e;
    }
    GraphArrays graph_view() const {
        GraphArrays g;
        size_t col_b = align_up((size_t) edge_cap * 4, 256);
        g.seq_to_node = seq_to_node.as<uint32_t>();
        g.src = (uint32_t*) edges.as<char>();
        g.dst = (uint32_t*) (edges.as<char>() + col_b);
        g.len = (uint32_t*) (edges.as<char>() + 2 * col_b);
        g.row_ptr = row_ptr.as<uint32_t>();
        g.cursor = cursor.as<uint32_t>();
        g.col = col.as<uint2>();
        g.col_eid = col_eid.as<uint32_t>();
        g.slot_degree = slot_degree.as<uint32_t>();
        g.T = T.as<uint8_t>();
        g.marked = marked.as<uint8_t>();
        return g;
    }
    HeavyItems heavy_view() const {
        HeavyItems h;
        size_t colb = align_up((size_t) heavy_cap * 4, 256);
        h.node = (uint32_t*) heavy.as<char>();
        h.unit_base = (uint32_t*) (heavy.as<char>() + colb);
        h.cap = heavy_cap;
        return h;
    }
    int new_slot() {
        int s = next_slot;
        next_slot = next_slot + 1 >= C_COUNT ? C_LIST0 : next_slot + 1;
        if (s == slot_ovl || s == slot_inl) return new_slot();
        return s;
    }
};


// ---- internals of api.cu used by the multi-rank orchestration (multi_api.cu) --------------------------------
size_t tiles_of(uint64_t n);
bool scan_state(rala_b200_graph* g, uint64_t n_max, unsigned long long** status, uint32_t** ticket);
bool stream_capturing(const rala_b200_graph* g);
cudaError_t stage_event(rala_b200_graph* g, cudaEvent_t ev);
cudaError_t begin_stage(rala_b200_graph* g, int stage);
cudaError_t end_stage(rala_b200_graph* g, int stage);
cudaError_t zero_counter(rala_b200_graph* g, int slot, int n = 1);
ResolveBufs resolve_bufs(const rala_b200_graph* g);
cudaError_t clear_earliest_events(rala_b200_graph* g);
// handed to the first containment pass's launch_apply_deaths: it prepares the final pass (kernels.h)
FinalPassReset final_pass_reset(const rala_b200_graph* g);
int reserve_events(rala_b200_graph* g, uint32_t ev_cap);
int reserve_edges(rala_b200_graph* g, uint32_t edge_cap);
int read_counters(rala_b200_graph* g, uint32_t* h);
int materialize_final_lists(rala_b200_graph* g);
int reserve_for_records(rala_b200_graph* g, uint64_t n);

// ---- the per-rank stages every driver runs (single session, NCCL phase calls, fabric ranks, stateless reduce) -----------
int phase_events(rala_b200_graph* g);
int phase_survivors(rala_b200_graph* g);
// final containment pass (graph.cpp:831-877): begin keeps the first pass's event / round counts and clears the events;
// `internals` are timed from counter slot time_base_slot.  end closes the stage: the session is finalized.
int begin_final_pass(rala_b200_graph* g, int time_base_slot);
int end_final_pass(rala_b200_graph* g);
int phase_final_events(rala_b200_graph* g, const uint32_t* ovl_base /* device, nullable */, int inl_base_slot);
// node ids and the edges of the final `overlaps`, with csr their CSR rows (opens ST_BUILD); then, when the caller gave an
// edge buffer (rala_b200_graph_set_outputs), their rows into it on side stream 0, joined by marks_stage
int emit_edges(rala_b200_graph* g, bool csr);
void fork_edge_download(rala_b200_graph* g);
// CSR rows of an edge list that did not come from emit_edges (C_NODES / C_EDGES set, n_nodes_max rows)
int csr_from_edge_list(rala_b200_graph* g);
int end_build(rala_b200_graph* g);
// K3 on the CSR in `ga` for the source nodes in node_range (device {begin, end}; nullptr = all), then marked(e) from ga.T
int transitive_stage(rala_b200_graph* g, const GraphArrays& ga, const uint32_t* node_range);
int marks_stage(rala_b200_graph* g, const GraphArrays& ga, uint8_t* copy /* nullable */, uint32_t copy_cap);

// ---- paf.cu: the read names and the chunked text upload, shared by the overlap readers and reads.cu --------------
// device name table: name i = blob[end[i-1], end[i]), slots = open addressing by name hash (k_paf_names)
struct NameTable {
    const uint8_t* blob;
    const unsigned long long* end;   // name i = blob[end[i-1], end[i])
    const uint32_t* read_len;
    unsigned long long* slots;       // hash >> 32 << 32 | id, ~0 = empty
    uint32_t mask;
};

struct PafCols {
    uint32_t *a, *b, *ab, *ae, *bb, *be, *len;
    uint8_t* mismatch;
};

// device words of one text call: the first four start at ~0 (minima), the rest at 0; line bases of the chunks follow
enum { W_ERR = 0, W_DUP, W_FIRST_MISMATCH, W_FIRST_BAD, W_UNRESOLVED, W_MISMATCH, W_QUERY_RC, W_BASES = 8 };

struct PafReader {
    DevBuf names;                 // blob | ends | read lengths | table slots (NamesLayout)
    NameTable table{};
    uint32_t n_reads = 0, max_len = 0;
    uint64_t name_bytes = 0;
    bool have_names = false;
    DevBuf text[2];               // device side of the staging pair
    DevBuf line_end, status, words, cols, valid;
    char* pinned[2] = {nullptr, nullptr};
    cudaStream_t copy = nullptr;  // uploads: chunk k + 1 crosses PCIe while chunk k is parsed
    cudaEvent_t copied[2]{}, parsed[2]{};
    std::vector<cudaEvent_t> timing;   // (start, stop) around the kernels of every chunk
    unsigned long long rec_cap = 0;
    std::vector<unsigned long long> w;   // the words of the last call, read back
    // compressed input (bgzf.cu, gzip.cu): the compressed bytes, the BGZF block table + error word, the inflated text,
    // the chunk cut and its read-back; gzip's chunk table, decoded symbols, member trailers and CRC32 segments
    DevBuf packed, bgzf_meta, inflated, bgzf_cut, gz_meta, gz_sym, gz_trailers, gz_seg;
    unsigned long long* cut_host = nullptr;

    PafCols view() const {
        const size_t col = align_up((size_t) rec_cap * 4, 256);
        char* b = cols.as<char>();
        return PafCols{(uint32_t*) b, (uint32_t*) (b + col), (uint32_t*) (b + 2 * col), (uint32_t*) (b + 3 * col),
                       (uint32_t*) (b + 4 * col), (uint32_t*) (b + 5 * col), (uint32_t*) (b + 6 * col), (uint8_t*) (b + 7 * col)};
    }
    ~PafReader() {
        if (copy) cudaStreamSynchronize(copy);
        DevBuf* bufs[] = {&names, &text[0], &text[1], &line_end, &status, &words, &cols, &valid, &packed, &bgzf_meta, &inflated, &bgzf_cut,
                          &gz_meta, &gz_sym, &gz_trailers, &gz_seg};
        for (DevBuf* b : bufs) b->release();
        for (int k = 0; k < 2; ++k) {
            if (pinned[k]) cudaFreeHost(pinned[k]);
            if (copied[k]) cudaEventDestroy(copied[k]);
            if (parsed[k]) cudaEventDestroy(parsed[k]);
        }
        if (cut_host) cudaFreeHost(cut_host);
        for (cudaEvent_t e : timing) cudaEventDestroy(e);
        if (copy) cudaStreamDestroy(copy);
    }
};

// byte offsets of the read names in PafReader::names for n reads with `blob` name bytes
struct NamesLayout {
    size_t o_end, o_len, o_slots, bytes;
    uint32_t slots;
};
NamesLayout names_layout(uint32_t n_reads, uint64_t blob);
// R.names holds the names, ends and lengths of n_reads reads in names_layout(n_reads, blob) and R.max_len is set: builds
// the name table (k_paf_names; ev0 / ev1 nullable, recorded around it) and refuses a name listed twice
int names_table(rala_b200_ctx* ctx, PafReader& R, uint32_t n_reads, uint64_t blob, cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr);
// the launches of one upload chunk k after its line scan: text (scan_len bytes, ends in '\n') at dtext, its line ends in
// R.line_end, the lines before it at words[W_BASES + k] and behind it at words[W_BASES + k + 1]
typedef int (*ChunkKernels)(void* self, rala_b200_ctx* ctx, uint32_t k, const uint8_t* dtext, uint32_t scan_len);
uint64_t text_max_chunks(uint64_t n_bytes);
size_t text_status_words();
// The whole text through the pinned staging pair (page-locked caller memory in place) in chunks of
// RALA_B200_PAF_CHUNK_BYTES cut behind their last '\n', each one line-scanned and handed to `kernels`; R.w holds the
// call's words afterwards (W_BASES + *n_chunks = lines).  W_ERR .. W_FIRST_BAD start at ~0, the rest at 0.
// kernel_ms (nullable) = device time of the chunks' kernels.  A refused call returns with no upload in flight.
// on_device: text is device memory (an inflated BGZF or gzip file); the cuts are found on the device and the chunks copied
// device to device into the same buffers, so chunks, line numbers and refusals are those of the host text.
int text_chunks(rala_b200_ctx* ctx, PafReader& R, const char* label, const char* text, uint64_t n_bytes, bool on_device,
                ChunkKernels kernels, void* self, float* kernel_ms, uint32_t* n_chunks);
void destroy_paf_reader(PafReader* r);
// ---- bgzf.cu: BGZF input --------------------------------------------------------------------------------------
// The BGZF file data[0, n) inflated into R.inflated (stats: blocks, bytes, inflate_ms); host_out (nullable, cap bytes)
// also receives the text.  A refused call returns with no upload in flight.
int bgzf_inflate(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_bgzf_stats_t* st,
                 uint8_t* host_out = nullptr, uint64_t cap = 0);
// position + 1 of the last '\n' in device text[lo, hi), 0 when there is none (on R.copy, synchronised)
int inflated_cut(rala_b200_ctx* ctx, PafReader& R, const uint8_t* text, uint64_t lo, uint64_t hi, uint64_t* found);
// whether the BGZF header walk accepts data[0, n) (sets no error text)
bool is_bgzf(const uint8_t* data, uint64_t n);
// ---- gzip.cu: plain gzip input -----------------------------------------------------------------------------------
// The gzip file data[0, n) inflated into R.inflated (BGZF input through bgzf_inflate); host_out as for bgzf_inflate;
// size_only: the finder and the counting pass only, R.inflated untouched.  A refused call returns with no upload in flight.
int gzip_inflate(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_gzip_stats_t* st,
                 uint8_t* host_out = nullptr, uint64_t cap = 0, bool size_only = false);
// A compressed input of the readers' _bgzf / _gzip calls (exactly one of the two set): inflated into R.inflated, whose
// length goes to *n_bytes, before the reader parses it.
struct Packed {
    rala_b200_bgzf_stats_t* bgzf;
    rala_b200_gzip_stats_t* gzip;
};
int inflate_packed(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, const Packed& z, uint64_t* n_bytes);
// the overlap columns build_piles counts: the parsed records of the last successful set_overlaps_paf / _mhap, before the
// duplicate filter was folded in (bit 31 of a = unresolved name), and the reads' lengths (device); returns the text format
// they came from, kTextNone when there are none
struct PileCols {
    const uint32_t *a, *b, *ab, *ae, *bb, *be;
};
TextFormat text_records_view(const rala_b200_graph* g, PileCols* cols, const uint32_t** read_len, uint32_t* n_reads, uint32_t* max_len);

// ---- piles.cu --------------------------------------------------------------------------------------------------
void destroy_pile_builder(PileBuilder* p);
