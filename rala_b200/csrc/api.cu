// api.cu — the C ABI (include/rala_b200.h): context, stateless stages, and the graph session that
// chains the kernels of classify.cu / graph_build.cu / transitive.cu with no host synchronisation
// between stages (every data-dependent size stays on the device).
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/rala_b200.h"
#include "session.h"

using namespace rb;

extern "C" int rala_b200_abi_version(void) { return RALA_B200_ABI_VERSION; }

extern "C" int rala_b200_create(rala_b200_ctx** out, int device) {
    if (!out) return RALA_B200_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device < 0 || device >= n) return RALA_B200_ERR_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return RALA_B200_ERR_NO_DEVICE;
    if (prop.major != 10) return RALA_B200_ERR_NO_DEVICE;   // sm_100a SASS only: no other target, no fallback
    rala_b200_ctx* ctx = new rala_b200_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->L.stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return RALA_B200_ERR_CUDA;
    }
    ctx->coop_blocks = resolve_max_blocks();
    preload_classify();
    preload_containment();
    preload_graph_build();
    preload_transitive();
    preload_fabric();
    preload_frontend();
    preload_paf();
    preload_reads();
    preload_bgzf();
    preload_gzip();
    preload_piles();
    cudaGetLastError();
    cudaEventCreate(&ctx->ev[0]);
    cudaEventCreate(&ctx->ev[1]);
    for (int k = 0; k < 2; ++k) {   // forked work inside a step (kernels.h Launch); without them everything stays on the main stream
        if (cudaStreamCreateWithFlags(&ctx->L.side[k], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->L.ev_fork[k], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->L.ev_join[k], cudaEventDisableTiming) != cudaSuccess) {
            ctx->L.side[k] = nullptr;
            cudaGetLastError();
        }
    }
    *out = ctx;
    return RALA_B200_OK;
}

extern "C" int rala_b200_create_on_stream(rala_b200_ctx** out, int device, void* cuda_stream) {
    int rc = rala_b200_create(out, device);
    if (rc) return rc;
    cudaStreamDestroy((*out)->L.stream);
    (*out)->L.stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    (*out)->owns_stream = false;
    return RALA_B200_OK;
}

extern "C" void rala_b200_destroy(rala_b200_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->L.stream && ctx->owns_stream) cudaStreamDestroy(ctx->L.stream);
    for (int k = 0; k < 2; ++k) {
        if (ctx->L.side[k]) cudaStreamDestroy(ctx->L.side[k]);
        if (ctx->L.ev_fork[k]) cudaEventDestroy(ctx->L.ev_fork[k]);
        if (ctx->L.ev_join[k]) cudaEventDestroy(ctx->L.ev_join[k]);
    }
    delete ctx;
}

extern "C" int rala_b200_event_record(rala_b200_ctx* ctx, int which) {
    if (!ctx || which < 0 || which > 1) return RALA_B200_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaEventRecord(ctx->ev[which], ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_event_elapsed_ms(rala_b200_ctx* ctx, float* ms) {
    if (!ctx || !ms) return RALA_B200_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaEventSynchronize(ctx->ev[1]));
    CU(ctx, cudaEventElapsedTime(ms, ctx->ev[0], ctx->ev[1]));
    return RALA_B200_OK;
}

extern "C" int rala_b200_synchronize(rala_b200_ctx* ctx) {
    if (!ctx) return RALA_B200_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" const char* rala_b200_last_error(const rala_b200_ctx* ctx) { return ctx ? ctx->error.c_str() : "no context"; }
extern "C" uint64_t rala_b200_launch_count(const rala_b200_ctx* ctx) { return ctx ? ctx->L.count : 0; }

size_t tiles_of(uint64_t n) { return (size_t) ((n + kTile - 1) / kTile) + 1; }

// a fresh, zeroed (status words, ticket) pair from the pool for one look-back kernel with `tiles` tiles
static bool scan_words(rala_b200_graph* g, uint64_t tiles, unsigned long long** status, uint32_t** ticket) {
    const size_t words = (size_t) tiles + 1;
    if (!g->scan_zeroed || g->scan_used + words > g->scan_pool_words) {
        // The step prologue zeroes the pool, which is sized for a step (reserve_scan_pool).  Calls outside a step, and
        // steps with more list passes (retrim rounds), clear it again: the clear is ordered behind every look-back kernel
        // already enqueued.  Handing out words a look-back kernel already wrote would give wrong prefixes (or spin): a
        // single kernel that asks for more than the whole pool declares the run void (read_counters reports it), and the
        // words are recycled only so that the kernel arguments stay valid.
        if (words > g->scan_pool_words || cudaMemsetAsync(g->scan_pool.p, 0, g->scan_pool_words * 8, g->ctx->L.stream) != cudaSuccess)
            g->scan_pool_exhausted = true;
        g->scan_used = 0;
        g->scan_zeroed = true;
    }
    unsigned long long* base = g->scan_pool.as<unsigned long long>() + g->scan_used;
    *ticket = reinterpret_cast<uint32_t*>(base);
    *status = base + 1;
    g->scan_used = words > g->scan_pool_words ? 0 : g->scan_used + words;
    return !g->scan_pool_exhausted;
}

bool scan_state(rala_b200_graph* g, uint64_t n_max, unsigned long long** status, uint32_t** ticket) {
    return scan_words(g, tiles_of(n_max), status, ticket);
}

// stage timers: plain event records, left out of a stream capture (an event recorded inside a capture cannot be timed)
// `capturing` covers the library's own capture (rala_b200_graph_run); a caller may also capture the phase calls
// into a graph of its own (rala_b200/multi.py: kernels + NCCL collectives of one multi-GPU step), so ask the stream.
bool stream_capturing(const rala_b200_graph* g) {
    if (g->capturing) return true;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(g->ctx->L.stream, &st) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return st != cudaStreamCaptureStatusNone;
}

cudaError_t stage_event(rala_b200_graph* g, cudaEvent_t ev) {
    return stream_capturing(g) ? cudaSuccess : cudaEventRecord(ev, g->ctx->L.stream);
}

cudaError_t begin_stage(rala_b200_graph* g, int stage) { return stage_event(g, g->ev_start[stage]); }

cudaError_t end_stage(rala_b200_graph* g, int stage) {
    g->ev_valid[stage] = !stream_capturing(g);
    return stage_event(g, g->ev_stop[stage]);
}

cudaError_t zero_counter(rala_b200_graph* g, int slot, int n) {
    return cudaMemsetAsync(g->cnt() + slot, 0, 4 * (size_t) n, g->ctx->L.stream);
}

extern "C" int rala_b200_graph_create(rala_b200_ctx* ctx, rala_b200_graph** out) {
    if (!ctx || !out) return RALA_B200_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    rala_b200_graph* g = new rala_b200_graph();
    g->ctx = ctx;
    for (int i = 0; i < RALA_B200_N_STAGES; ++i) {
        cudaEventCreate(&g->ev_start[i]);
        cudaEventCreate(&g->ev_stop[i]);
    }
    cudaError_t e = g->counters.reserve(C_COUNT * 4);
    if (e == cudaSuccess) e = g->flags.reserve(64);
    if (e == cudaSuccess) e = g->work_counter.reserve(64);
    if (e == cudaSuccess) e = cudaMemset(g->counters.p, 0, C_COUNT * 4);
    if (e != cudaSuccess) {
        delete g;
        return fail(ctx, RALA_B200_ERR_CUDA, "graph_create: %s", cudaGetErrorString(e));
    }
    *out = g;
    return RALA_B200_OK;
}

static void drop_run_graphs(rala_b200_graph* g);

extern "C" void rala_b200_graph_destroy(rala_b200_graph* g) {
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->ctx->L.stream);
    drop_run_graphs(g);
    destroy_paf_reader(g->paf);
    destroy_pile_builder(g->pile_builder);
    DevBuf* bufs[] = {&g->rec, &g->recs.buf, &g->alive_bits, &g->piles, &g->piles_raw, &g->pile_flags_raw, &g->piles_initial, &g->hills, &g->ovl[0].buf,
                      &g->ovl[1].buf, &g->inl[0].buf, &g->inl[1].buf, &g->events, &g->hill_rec, &g->dbuf, &g->flags, &g->segs,
                      &g->counters, &g->scan_pool, &g->seq_to_node, &g->edges, &g->row_ptr, &g->cursor, &g->col,
                      &g->col_eid, &g->T, &g->marked, &g->heavy, &g->work_counter, &g->edges_aos, &g->slot_degree, &g->tile_dov};
    for (DevBuf* b : bufs) b->release();
    for (int i = 0; i < RALA_B200_N_STAGES; ++i) {
        cudaEventDestroy(g->ev_start[i]);
        cudaEventDestroy(g->ev_stop[i]);
    }
    delete g;
}

int reserve_events(rala_b200_graph* g, uint32_t ev_cap) {
    if (ev_cap <= g->ev_cap) return RALA_B200_OK;
    rala_b200_ctx* ctx = g->ctx;
    // growing re-allocates: contents are not preserved (callers grow before they fill)
    g->ev_cap = ev_cap;
    CU(ctx, g->events.reserve(align_up((size_t) ev_cap * 4, 256) * 3));
    CU(ctx, g->segs.reserve(align_up((size_t) ev_cap * 8, 256) + (size_t) ev_cap * 16));
    return RALA_B200_OK;
}

int reserve_edges(rala_b200_graph* g, uint32_t edge_cap) {
    if (edge_cap <= g->edge_cap) return RALA_B200_OK;
    rala_b200_ctx* ctx = g->ctx;
    g->edge_cap = edge_cap;
    CU(ctx, g->edges.reserve(align_up((size_t) edge_cap * 4, 256) * 3));
    CU(ctx, g->col.reserve((size_t) edge_cap * 8));
    CU(ctx, g->col_eid.reserve((size_t) edge_cap * 4));
    CU(ctx, g->T.reserve(align_up(edge_cap, 256)));
    CU(ctx, g->marked.reserve(align_up(edge_cap, 256)));
    return RALA_B200_OK;
}

static int reserve_scan_pool(rala_b200_graph* g) {
    // one step: the survivors pass (a word per run), two containment resolutions over the piles and their scans (the
    // fabric ranks), the pile scan of build or the CSR scan over the nodes of the multi-GPU paths, one retrim + promote
    // round (three list passes) and, after the step, the two final list passes of get_lists / counts
    const size_t piles = tiles_of((uint64_t) g->n_piles + 1) + 1, nodes = tiles_of((uint64_t) g->n_nodes_max + 8) + 1,
                 lists = tiles_of(g->cap) + 1;
    const size_t words = classify_num_runs(g->n_rec) + 1 + 4 * piles + 2 * nodes + 5 * lists + 64;
    if (words > g->scan_pool_words) {
        CU(g->ctx, g->scan_pool.reserve(words * 8));
        g->scan_pool_words = words;
        g->scan_zeroed = false;
    }
    return RALA_B200_OK;
}

// node arrays of the graph: CSR rows, fill cursor, slot degrees and the heavy work list
static int reserve_nodes(rala_b200_graph* g, uint32_t n_nodes) {
    rala_b200_ctx* ctx = g->ctx;
    g->n_nodes_max = n_nodes;
    CU(ctx, g->row_ptr.reserve(((size_t) n_nodes + 8) * 4));
    CU(ctx, g->cursor.reserve(((size_t) n_nodes + 8) * 4));
    CU(ctx, g->slot_degree.reserve(((size_t) n_nodes + 8) * 4));
    g->heavy_cap = n_nodes;   // one entry per node (HeavyItems)
    CU(ctx, g->heavy.reserve(align_up((size_t) g->heavy_cap * 4, 256) * 2));
    return reserve_scan_pool(g);
}

// device lists sized for n records (worst case every record survives)
int reserve_for_records(rala_b200_graph* g, uint64_t n) {
    rala_b200_ctx* ctx = g->ctx;
    g->n_rec = (uint32_t) n;
    g->text_records = kTextNone;   // set_overlaps_paf / _mhap set it again once their records are in place
    CU(ctx, g->recs.reserve((uint32_t) ((n + 3) / 4 * 4 + 4)));
    uint32_t cap = (uint32_t) align_up((size_t) n, 128);
    if (cap < 1024) cap = 1024;
    if (cap > g->cap) {
        for (int i = 0; i < 2; ++i) {
            CU(ctx, g->ovl[i].reserve(cap));
            CU(ctx, g->inl[i].reserve(cap));
        }
        CU(ctx, g->hill_rec.reserve((size_t) cap * 4));
        CU(ctx, g->tile_dov.reserve((emit_tiles(cap) + 8) * 4));
        g->cap = cap;
        int rc2 = reserve_events(g, cap);
        if (!rc2) rc2 = reserve_edges(g, 2 * cap);
        if (rc2) return rc2;
    }
    int rc = reserve_scan_pool(g);
    if (rc) return rc;
    if (g->state == SS_EMPTY && g->n_piles) g->state = SS_INPUTS;
    if (g->state > SS_INPUTS) g->state = SS_INPUTS;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_set_overlaps(rala_b200_graph* g, const rala_ovl_t* ovl, uint64_t n) {
    if (!g || (n && !ovl)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (n >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many overlap records (%llu >= 2^31)", (unsigned long long) n);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, g->rec.reserve(align_up((size_t) n * sizeof(rala_ovl_t) + 16, 256)));
    if (n) CU(ctx, cudaMemcpyAsync(g->rec.p, ovl, (size_t) n * sizeof(rala_ovl_t), cudaMemcpyHostToDevice, ctx->L.stream));
    int rc = reserve_for_records(g, n);
    if (rc) return rc;
    // layout in HBM: rows -> six columns, once per upload (the kernels read 16 bytes per column and thread)
    launch_records_to_soa(ctx->L, g->rec.as<uint32_t>(), (uint32_t) n, g->recs.view);
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

// The same records as six host columns in the device layout: 24 bytes per record cross PCIe instead of 28 and
// land where the kernels read them (no staging buffer, no transpose kernel).
extern "C" int rala_b200_graph_set_overlaps_columns(rala_b200_graph* g, const uint32_t* a_id, const uint32_t* b_id,
                                                    const uint32_t* a_begin, const uint32_t* a_end, const uint32_t* b_begin,
                                                    const uint32_t* b_end, uint64_t n) {
    if (!g || (n && (!a_id || !b_id || !a_begin || !a_end || !b_begin || !b_end))) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (n >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many overlap records (%llu >= 2^31)", (unsigned long long) n);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = reserve_for_records(g, n);
    if (rc) return rc;
    if (n) {
        const List& r = g->recs.view;
        const uint32_t* src[6] = {a_id, b_id, a_begin, a_end, b_begin, b_end};
        uint32_t* dst[6] = {r.a, r.b, r.ab, r.ae, r.bb, r.be};
        for (int k = 0; k < 6; ++k)
            CU(ctx, cudaMemcpyAsync(dst[k], src[k], (size_t) n * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    }
    return RALA_B200_OK;
}

// Compact upload (12 B / record): b_id lands in place, the two span columns and the group table go through the staging
// buffer and are expanded by one kernel.
extern "C" int rala_b200_graph_set_overlaps_packed(rala_b200_graph* g, const uint32_t* query_id, const uint32_t* group_end, uint32_t n_groups,
                                                   const uint32_t* b_id, const uint32_t* a_span, const uint32_t* b_span, uint64_t n) {
    if (!g || (n && (!query_id || !group_end || !b_id || !a_span || !b_span || !n_groups))) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (n >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many overlap records (%llu >= 2^31)", (unsigned long long) n);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = reserve_for_records(g, n);
    if (rc) return rc;
    if (!n) return RALA_B200_OK;
    const size_t col = align_up(((size_t) n + 4) * 4, 256), grp = align_up((size_t) n_groups * 4, 256);
    CU(ctx, g->rec.reserve(2 * col + 2 * grp));
    char* st = g->rec.as<char>();
    uint32_t *d_a = (uint32_t*) st, *d_b = (uint32_t*) (st + col), *d_q = (uint32_t*) (st + 2 * col), *d_e = (uint32_t*) (st + 2 * col + grp);
    CU(ctx, cudaMemcpyAsync(g->recs.view.b, b_id, (size_t) n * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(d_a, a_span, (size_t) n * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(d_b, b_span, (size_t) n * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(d_q, query_id, (size_t) n_groups * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(d_e, group_end, (size_t) n_groups * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    launch_unpack_records(ctx->L, d_q, d_e, n_groups, d_a, d_b, (uint32_t) n, g->recs.view);
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

// Results straight into the caller's memory (pinned host memory or device memory the GPU can address).
extern "C" int rala_b200_graph_set_outputs(rala_b200_graph* g, rala_edge_t* edges_out, uint64_t edges_cap, uint8_t* marked_out,
                                           uint64_t marked_cap) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    void* dev[2] = {nullptr, nullptr};
    const void* host[2] = {edges_out, marked_out};
    for (int k = 0; k < 2; ++k) {
        if (!host[k]) continue;
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, host[k]) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered || !attr.devicePointer) {
            cudaGetLastError();
            return fail(ctx, RALA_B200_ERR_ARG, "set_outputs: the %s buffer is not addressable by the GPU (use cudaHostAlloc / cudaHostRegister "
                        "memory, or get_edges / get_marked for pageable memory)", k ? "marks" : "edge");
        }
        dev[k] = attr.devicePointer;
    }
    if (edges_cap >= (1ull << 31)) edges_cap = (1ull << 31) - 1;
    if (marked_cap >= (1ull << 31)) marked_cap = (1ull << 31) - 1;
    g->out_edges = reinterpret_cast<uint32_t*>(dev[0]);
    g->out_edges_cap = edges_out ? (uint32_t) edges_cap : 0u;
    g->out_marked = reinterpret_cast<uint8_t*>(dev[1]);
    g->out_marked_cap = marked_out ? (uint32_t) marked_cap : 0u;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_set_piles(rala_b200_graph* g, const rala_pile_t* piles, const uint8_t* flags,
                                         uint32_t n_piles) {
    if (!g || (n_piles && !piles)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (n_piles >= (1u << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many piles");
    // event_code (common.cuh) and the packed table (end | flags << 30) rely on the documented limit: valid regions end below 2^30
    // (two branch-free passes over the table as 64-bit words, begin in the low half: it is re-uploaded for every batch; the
    // offender is only looked for when there is one)
    {
        static_assert(sizeof(rala_pile_t) == 8, "a pile is one 64-bit word: begin | end << 32");
        unsigned long long any = 0, inverted = 0;
        for (uint32_t i = 0; i < n_piles; ++i) {
            unsigned long long w;
            memcpy(&w, &piles[i], 8);
            any |= w;
            inverted += (unsigned long long) (((uint32_t) w > (uint32_t) (w >> 32)) & ((w >> 32) != 0));
        }
        if ((any >> 62) || inverted) {
            for (uint32_t i = 0; i < n_piles; ++i) {
                if (piles[i].end >= (1u << 30)) return fail(ctx, RALA_B200_ERR_LIMIT, "pile %u ends at %u: read lengths must be < 2^30", i, piles[i].end);
                if (piles[i].end && piles[i].begin > piles[i].end) return fail(ctx, RALA_B200_ERR_ARG, "pile %u: begin %u > end %u", i, piles[i].begin, piles[i].end);
            }
        }
    }
    CU(ctx, g->piles.reserve((size_t) n_piles * 8 + 16));
    CU(ctx, g->piles_raw.reserve((size_t) n_piles * 8 + 16));
    CU(ctx, g->piles_initial.reserve((size_t) n_piles * 8 + 16));
    CU(ctx, g->pile_flags_raw.reserve((size_t) n_piles + 16));
    CU(ctx, cudaMemcpyAsync(g->piles_raw.p, piles, (size_t) n_piles * 8, cudaMemcpyHostToDevice, ctx->L.stream));
    if (flags) CU(ctx, cudaMemcpyAsync(g->pile_flags_raw.p, flags, n_piles, cudaMemcpyHostToDevice, ctx->L.stream));
    launch_pack_piles(ctx->L, g->piles_raw.as<uint2>(), flags ? g->pile_flags_raw.as<uint8_t>() : nullptr,
                      g->piles.as<uint2>(), n_piles);
    if (n_piles != g->n_piles) {
        g->n_piles = n_piles;
        CU(ctx, g->dbuf.reserve(align_up((size_t) n_piles + 64, 64) * 4 * 8));
        CU(ctx, g->alive_bits.reserve(((size_t) n_piles / 32 + 2) * 4));
        CU(ctx, g->seq_to_node.reserve((size_t) n_piles * 4 + 16));
        int rc = reserve_nodes(g, 2 * n_piles);
        if (rc) return rc;
    }
    g->piles_dirty = true;
    g->promote_pending = true;
    g->piles_fresh = true;
    if (g->state == SS_EMPTY && g->n_rec) g->state = SS_INPUTS;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_set_hills(rala_b200_graph* g, const rala_hill_t* hills, uint32_t n_hills) {
    if (!g || (n_hills && !hills)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    g->n_hills = n_hills;
    if (!n_hills) return RALA_B200_OK;
    std::vector<uint32_t> cols((size_t) n_hills * 4, 0u);
    for (uint32_t i = 0; i < n_hills; ++i) {
        if (i && hills[i].pile < hills[i - 1].pile) return fail(ctx, RALA_B200_ERR_ARG, "hills must be grouped by ascending pile id");
        cols[i] = hills[i].pile;
        cols[n_hills + i] = hills[i].begin;
        cols[2 * (size_t) n_hills + i] = hills[i].end;
    }
    CU(ctx, g->hills.reserve(cols.size() * 4));
    CU(ctx, cudaMemcpyAsync(g->hills.p, cols.data(), cols.size() * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));   // cols is a stack-owned staging vector
    return RALA_B200_OK;
}

ResolveBufs resolve_bufs(const rala_b200_graph* g) {
    ResolveBufs r;
    const size_t stride = align_up((size_t) g->n_piles + 64, 64);   // 256-byte aligned sub-arrays (16-byte vector loads)
    uint32_t* b = g->dbuf.as<uint32_t>();
    r.S = b;
    r.vcursor = b + stride;
    r.vstart = b + 2 * stride;
    r.work0 = b + 3 * stride;
    r.work1 = b + 4 * stride;
    r.hidx = b + 5 * stride;
    r.first = reinterpret_cast<unsigned long long*>(b + 6 * stride);   // two strides
    r.n_work = g->flags.as<uint32_t>();
    r.seg = g->segs.as<unsigned long long>();
    r.hev = reinterpret_cast<uint4*>(g->segs.as<char>() + align_up((size_t) g->ev_cap * 8, 256));
    r.seg_c = g->segs.as<uint32_t>();
    r.seg_t = (uint32_t*) (g->segs.as<char>() + align_up((size_t) g->ev_cap * 4, 256));
    return r;
}

// the classify kernels keep every victim's earliest event while they emit events: clear it to "none" (all ones) first
cudaError_t clear_earliest_events(rala_b200_graph* g) {
    return cudaMemsetAsync(resolve_bufs(g).first, 0xFF, ((size_t) g->n_piles + 64) * 8, g->ctx->L.stream);
}

FinalPassReset final_pass_reset(const rala_b200_graph* g) {
    FinalPassReset r;
    r.first = resolve_bufs(g).first;
    r.n_first = r.first ? g->n_piles + 64 : 0u;
    r.counters = g->cnt();
    return r;
}

static int resolve_containment(rala_b200_graph* g, bool decode, bool skip_if_empty) {
    rala_b200_ctx* ctx = g->ctx;
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, (uint64_t) g->n_piles + 1, &status, &ticket);
    launch_resolve(ctx->L, g->events_view(), g->cnt() + C_EV, g->ev_cap, resolve_bufs(g), g->n_piles, g->cnt(), status, ticket,
                   ctx->coop_blocks, decode, skip_if_empty);
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

// ---- graph.cpp:443-518 in three phases (the multi-GPU path exchanges events between them) ----------------
int phase_events(rala_b200_graph* g) {
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_INPUTS) return fail(ctx, RALA_B200_ERR_STATE, "classify: set_overlaps and set_piles first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_CLASSIFY));
    // classify kills piles in the working table: keep the table it started from, so that calling classify
    // again without a new set_piles re-runs on the same input (bench loops, retries).  One launch also clears what the
    // step's stages count into: the counters, the hill coverage, the look-back pool, the earliest events of the first
    // pass, the slot degrees of build and the node counters of the transitive pass.
    StepPrologue pro{};
    pro.piles = g->piles.as<uint2>();
    pro.piles_initial = g->piles_initial.as<uint2>();
    pro.n_piles = g->n_piles;
    pro.snapshot = g->piles_fresh;
    pro.first = resolve_bufs(g).first;
    pro.n_first = pro.first ? g->n_piles + 64 : 0u;
    uint32_t* zero[StepPrologue::kZero] = {g->cnt(), g->n_hills ? g->hills.as<uint32_t>() + 3 * (size_t) g->n_hills : nullptr,
                                           g->scan_pool.as<uint32_t>(), g->slot_degree.as<uint32_t>(), g->work_counter.as<uint32_t>()};
    const size_t words[StepPrologue::kZero] = {C_COUNT, g->n_hills, 2 * g->scan_pool_words, (size_t) g->n_nodes_max + 8, 2};
    for (int k = 0; k < StepPrologue::kZero; ++k) {
        pro.zero[k] = zero[k];
        pro.zero_words[k] = words[k];
    }
    launch_step_prologue(ctx->L, pro);
    g->piles_fresh = false;
    g->scan_used = 0;
    g->scan_zeroed = true;
    g->step_cleared = kStepBuild | kStepTransitive;
    CU(ctx, stage_event(g, g->ev_start[ST_K1_KERNEL]));
    launch_classify_events(ctx->L, g->recs.view, g->n_rec, g->t0, g->piles.as<uint2>(), g->n_piles, g->events_view(),
                           g->ev_cap, resolve_bufs(g).first, g->hill_rec.as<uint32_t>(), g->cap, g->cnt());
    CU(ctx, end_stage(g, ST_K1_KERNEL));
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

static int phase_resolve(rala_b200_graph* g, bool first_pass) {
    rala_b200_ctx* ctx = g->ctx;
    // the hill counters read the death times BEFORE the deaths are applied to the pile table; without hills nothing
    // sits between the resolution and k_apply_deaths, which then decodes the states itself
    const bool fused_decode = !(first_pass && g->n_hills);
    CU(ctx, stage_event(g, g->ev_start[ST_K1B_KERNEL]));
    // The final pass (graph.cpp:831-866) has no events at all on clean data: scan, scatter, resolution and the sweep over the
    // pile table then return at once (nobody dies; the death times of the first pass, all "never" for the piles still
    // in the lists, stay in place).  The first pass always runs: it also builds the liveness bitmap.
    const bool skip_if_empty = !first_pass && fused_decode;
    int rc = resolve_containment(g, !fused_decode, skip_if_empty);
    if (rc) return rc;
    CU(ctx, end_stage(g, ST_K1B_KERNEL));
    if (first_pass && g->n_hills) {
        const uint32_t* h = g->hills.as<uint32_t>();
        launch_hill_coverage(ctx->L, g->recs.view, g->t0, g->piles.as<uint2>(), g->hill_rec.as<uint32_t>(), g->cap, h,
                             h + g->n_hills, h + 2 * (size_t) g->n_hills, g->n_hills,
                             g->hills.as<uint32_t>() + 3 * (size_t) g->n_hills, g->dbuf.as<uint32_t>(), g->cnt());
    }
    FinalPassReset reset;
    if (first_pass) reset = final_pass_reset(g);
    launch_apply_deaths(ctx->L, g->piles.as<uint2>(), g->dbuf.as<uint32_t>(), g->n_piles, g->alive_bits.as<uint32_t>(), fused_decode,
                        nullptr, skip_if_empty ? g->cnt() + C_EV : nullptr, reset);
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

int phase_survivors(rala_b200_graph* g) {
    rala_b200_ctx* ctx = g->ctx;
    g->ovl_cur = 0;
    g->inl_cur = 0;
    g->slot_ovl = C_LIST0;
    g->slot_inl = C_LIST0 + 1;
    g->next_slot = C_LIST0 + 2;
    if (!g->n_rec) CU(ctx, zero_counter(g, C_LIST0, 2));   // otherwise the last run writes both counts
    CU(ctx, stage_event(g, g->ev_start[ST_K1S_KERNEL]));
    unsigned long long* status;
    uint32_t* ticket;
    scan_words(g, classify_num_runs(g->n_rec), &status, &ticket);
    launch_classify_survivors(ctx->L, g->recs.view, g->n_rec, g->piles.as<uint2>(), g->alive_bits.as<uint32_t>(), g->n_piles,
                              g->ovl[0].view, g->cnt() + g->slot_ovl, g->inl[0].view, g->cnt() + g->slot_inl, g->cap, status, ticket);
    CU(ctx, end_stage(g, ST_K1S_KERNEL));
    CU(ctx, cudaGetLastError());
    CU(ctx, end_stage(g, ST_CLASSIFY));
    g->piles_dirty = false;   // lists are trimmed against the table as it stands (only liveness changed, and the split filtered on it)
    g->promote_pending = false;   // and every internal was typed against it
    g->state = SS_CLASSIFIED;
    g->final_lists_ready = true;
    g->retrim_passes = 0;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_classify(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    int rc = phase_events(g);
    if (!rc) rc = phase_resolve(g, true);
    if (!rc) rc = phase_survivors(g);
    return rc;
}

static int retrim_list(rala_b200_graph* g, ListBuf* bufs, int* cur, int* slot) {
    rala_b200_ctx* ctx = g->ctx;
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, g->cap, &status, &ticket);
    int out_slot = g->new_slot();
    CU(ctx, zero_counter(g, out_slot));
    List none{};
    launch_list_pass(ctx->L, 1 /*kRetrim*/, bufs[*cur].view, g->cnt() + *slot, g->cap, g->piles.as<uint2>(), bufs[*cur ^ 1].view,
                     g->cnt() + out_slot, none, nullptr, nullptr, g->cap, nullptr, nullptr, status, ticket);
    *cur ^= 1;
    *slot = out_slot;
    return RALA_B200_OK;
}

// graph.cpp:722-736
extern "C" int rala_b200_graph_retrim(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state != SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "retrim: classify first");
    if (!g->piles_dirty && g->skip_clean_retrim) return RALA_B200_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_RETRIM));
    int rc = retrim_list(g, g->ovl, &g->ovl_cur, &g->slot_ovl);
    if (!rc) rc = retrim_list(g, g->inl, &g->inl_cur, &g->slot_inl);
    if (rc) return rc;
    CU(ctx, cudaGetLastError());
    CU(ctx, end_stage(g, ST_RETRIM));
    g->piles_dirty = false;
    g->retrim_passes += 1;
    return RALA_B200_OK;
}

// graph.cpp:801-824
extern "C" int rala_b200_graph_retrim_promote(rala_b200_graph* g, int* is_changed) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state != SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "retrim_promote: classify first");
    if (is_changed) *is_changed = 0;
    // Against a pile table the internals were already trimmed AND typed with, trim() is the identity and they keep their
    // (non-dovetail) type.  retrim() trims them but does not re-type them: after set_piles -> retrim the promotion of
    // graph.cpp:809-823 still has to run (promote_pending), although piles_dirty is clear.
    if (!g->piles_dirty && !g->promote_pending && g->skip_clean_retrim) return RALA_B200_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_RETRIM));
    int before_slot = g->slot_ovl;
    int rc = retrim_list(g, g->ovl, &g->ovl_cur, &g->slot_ovl);
    if (rc) return rc;
    int after_slot = g->slot_ovl;
    // internals: survivors stay (stream A), new dovetails are appended to `overlaps` (stream B)
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, g->cap, &status, &ticket);
    int inl_out = g->new_slot(), ovl_out = g->new_slot();
    CU(ctx, zero_counter(g, inl_out));
    CU(ctx, cudaMemcpyAsync(g->cnt() + ovl_out, g->cnt() + after_slot, 4, cudaMemcpyDeviceToDevice, ctx->L.stream));
    launch_list_pass(ctx->L, 2 /*kPromote*/, g->inl[g->inl_cur].view, g->cnt() + g->slot_inl, g->cap, g->piles.as<uint2>(),
                     g->inl[g->inl_cur ^ 1].view, g->cnt() + inl_out, g->ovl[g->ovl_cur].view, g->cnt() + ovl_out,
                     g->cnt() + after_slot, g->cap, nullptr, nullptr, status, ticket);
    g->inl_cur ^= 1;
    g->slot_inl = inl_out;
    g->slot_ovl = ovl_out;
    CU(ctx, cudaGetLastError());
    CU(ctx, end_stage(g, ST_RETRIM));
    g->piles_dirty = false;
    g->promote_pending = false;
    g->retrim_passes += 1;
    if (is_changed) {
        uint32_t h[C_COUNT];
        CU(ctx, cudaMemcpyAsync(h, g->counters.p, C_COUNT * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
        CU(ctx, cudaStreamSynchronize(ctx->L.stream));
        *is_changed = h[after_slot] != h[before_slot];
    }
    return RALA_B200_OK;
}

// graph.cpp:849-877 on demand: the final `internals` (alive at their own time, not kA/kB) and `overlaps`
// (both piles alive at the end, not kA/kB)
int materialize_final_lists(rala_b200_graph* g) {
    if (g->final_lists_ready || g->state < SS_FINALIZED) return RALA_B200_OK;
    rala_b200_ctx* ctx = g->ctx;
    unsigned long long* status;
    uint32_t* ticket;
    List none{};
    scan_state(g, g->cap, &status, &ticket);
    int inl_out = g->new_slot();
    CU(ctx, zero_counter(g, inl_out));
    launch_list_pass(ctx->L, 4 /*kFinalInt*/, g->inl[g->inl_cur].view, g->cnt() + g->slot_inl, g->cap, g->piles.as<uint2>(),
                     g->inl[g->inl_cur ^ 1].view, g->cnt() + inl_out, none, nullptr, nullptr, g->cap, g->dbuf.as<uint32_t>(),
                     g->cnt() + g->final_time_base_slot, status, ticket);
    g->inl_cur ^= 1;
    g->slot_inl = inl_out;
    scan_state(g, g->cap, &status, &ticket);
    int ovl_out = g->new_slot();
    CU(ctx, zero_counter(g, ovl_out));
    launch_list_pass(ctx->L, 3 /*kFinalOvl*/, g->ovl[g->ovl_cur].view, g->cnt() + g->slot_ovl, g->cap, g->piles.as<uint2>(),
                     g->ovl[g->ovl_cur ^ 1].view, g->cnt() + ovl_out, none, nullptr, nullptr, g->cap, nullptr, nullptr, status, ticket);
    g->ovl_cur ^= 1;
    g->slot_ovl = ovl_out;
    CU(ctx, cudaGetLastError());
    g->final_lists_ready = true;
    return RALA_B200_OK;
}

// ---- graph.cpp:831-877 in two phases ---------------------------------------------------------------------
int begin_final_pass(rala_b200_graph* g, int time_base_slot) {
    rala_b200_ctx* ctx = g->ctx;
    if (g->state != SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "finalize: classify first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_FINALIZE));   // the first pass's k_apply_deaths kept its counts and cleared the events (FinalPassReset)
    g->final_time_base_slot = time_base_slot;
    return RALA_B200_OK;
}

int end_final_pass(rala_b200_graph* g) {
    // The filtered `overlaps` / `internals` vectors of graph.cpp:867-877 are NOT materialised here: edge creation
    // (build) applies the same filter on the fly (both piles alive, type kAB/kBA), and nothing else on the path
    // reads them.  get_lists / counts materialise them on demand (materialize_final_lists).
    g->final_lists_ready = false;
    CU(g->ctx, end_stage(g, ST_FINALIZE));
    g->state = SS_FINALIZED;
    return RALA_B200_OK;
}

int phase_final_events(rala_b200_graph* g, const uint32_t* ovl_base, int inl_base_slot) {
    rala_b200_ctx* ctx = g->ctx;
    int rc = begin_final_pass(g, inl_base_slot);
    if (rc) return rc;
    launch_classify_final(ctx->L, g->ovl[g->ovl_cur].view, g->cnt() + g->slot_ovl, ovl_base, g->inl[g->inl_cur].view,
                          g->cnt() + g->slot_inl, g->cnt() + inl_base_slot, g->cap, g->piles.as<uint2>(), g->events_view(), g->ev_cap,
                          resolve_bufs(g).first, g->cnt());
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

static int phase_final_resolve(rala_b200_graph* g) {
    int rc = phase_resolve(g, false);
    return rc ? rc : end_final_pass(g);
}

extern "C" int rala_b200_graph_finalize(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    int rc = phase_final_events(g, nullptr, g->slot_ovl);   // internals are timed after every entry of `overlaps`
    if (!rc) rc = phase_final_resolve(g);
    return rc;
}

// node ids + the edges of the overlaps in list order (graph.cpp:552-632), and with `csr` their CSR rows.  In a multi-GPU
// phase the list is the local shard's and the node ids are global: the pile table is replicated.
int emit_edges(rala_b200_graph* g, bool csr) {
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_BUILD));
    GraphArrays ga = g->graph_view();
    if (!(g->step_cleared & kStepBuild)) {   // not already cleared by the step prologue
        CU(ctx, zero_counter(g, C_NODES, 4));   // C_NODES, C_ALIVE, C_DOVETAILS, C_EDGES
        if (csr) CU(ctx, cudaMemsetAsync(ga.slot_degree, 0, ((size_t) g->n_nodes_max + 8) * 4, ctx->L.stream));
    }
    g->step_cleared &= ~kStepBuild;
    if (!csr) ga.cursor = nullptr;
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, g->n_piles, &status, &ticket);
    const List ovl = g->ovl[g->ovl_cur].view;
    const uint32_t* n_ovl = g->cnt() + g->slot_ovl;
    launch_count_scan(ctx->L, ovl, n_ovl, g->cap, g->piles.as<uint2>(), g->n_piles, ga, g->edge_cap, g->tile_dov.as<uint32_t>(), g->cnt(),
                      status, ticket);
    launch_emit_edges(ctx->L, ovl, n_ovl, g->cap, g->piles.as<uint2>(), ga, g->edge_cap, g->tile_dov.as<uint32_t>());
    return RALA_B200_OK;
}

// the edge list is final: rows into the caller's buffer on a forked stream, beside (inside a whole run) the transitive
// pass; edges beyond the caller's capacity are not written (n_edges tells)
void fork_edge_download(rala_b200_graph* g) {
    Launch& L = g->ctx->L;
    if (!g->out_edges || !g->out_edges_cap || !fork_side(L, 0)) return;
    launch_pack_edges(L, L.side[0], g->graph_view(), g->edge_cap < g->out_edges_cap ? g->edge_cap : g->out_edges_cap, g->cnt() + C_EDGES,
                      g->out_edges);
    g->download_pending = true;
}

// CSR over an edge list whose columns and counts are in place (the NCCL phases' gathered edges, transitive_reduce)
int csr_from_edge_list(rala_b200_graph* g) {
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaMemsetAsync(g->cursor.p, 0, ((size_t) g->n_nodes_max + 8) * 4, ctx->L.stream));
    GraphArrays ga = g->graph_view();
    launch_degree_hist(ctx->L, ga.src, g->cnt() + C_EDGES, g->edge_cap, ga.cursor);
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, (uint64_t) g->n_nodes_max + 1, &status, &ticket);
    launch_build_csr(ctx->L, ga, g->n_nodes_max, g->edge_cap, g->cnt(), status, ticket);
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

int end_build(rala_b200_graph* g) {
    CU(g->ctx, cudaGetLastError());
    CU(g->ctx, end_stage(g, ST_BUILD));
    g->state = SS_BUILT;
    return RALA_B200_OK;
}

// build, transitive and run take every source node; a shard of a multi-GPU step takes part only through the phase calls
static int refuse_shard(rala_b200_graph* g, const char* what) {
    return fail(g->ctx, RALA_B200_ERR_STATE, "%s: the session is rank %d of %d (rala_b200_graph_set_shard): use the phase calls "
                "(rala_b200_graph_phase_*) or the multi-GPU session", what, g->rank, g->world);
}

// graph.cpp:552-632
extern "C" int rala_b200_graph_build(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->world > 1) return refuse_shard(g, "build");
    if (g->state != SS_FINALIZED) return fail(ctx, RALA_B200_ERR_STATE, "build: finalize first");
    int rc = emit_edges(g, true);
    if (rc) return rc;
    fork_edge_download(g);
    if (g->download_pending && !g->in_run) {
        join_side(ctx->L, 0);
        g->download_pending = false;
    }
    return end_build(g);
}

int transitive_stage(rala_b200_graph* g, const GraphArrays& ga, const uint32_t* node_range) {
    rala_b200_ctx* ctx = g->ctx;
    if (!(g->step_cleared & kStepTransitive)) {   // not already cleared by the step prologue
        CU(ctx, zero_counter(g, C_PAIRS, 5));   // C_PAIRS, C_HEAVY_NODES, C_HEAVY, C_HOP_LO, C_HOP_HI
        // the two node counters of K3 (a node range of the NCCL phase sits behind them, in words 4 and 5)
        CU(ctx, cudaMemsetAsync(g->work_counter.p, 0, 8, ctx->L.stream));
    }
    g->step_cleared &= ~kStepTransitive;
    CU(ctx, stage_event(g, g->ev_start[ST_K3_KERNELS]));
    launch_transitive(ctx->L, ga, g->n_nodes_max, g->heavy_view(), g->work_counter.as<uint32_t>(), g->cnt(), node_range);
    CU(ctx, end_stage(g, ST_K3_KERNELS));
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

// marked(e) = T(e) | T(e ^ 1) (copied into `copy` too when given); closes ST_TRANSITIVE
int marks_stage(rala_b200_graph* g, const GraphArrays& ga, uint8_t* copy, uint32_t copy_cap) {
    rala_b200_ctx* ctx = g->ctx;
    launch_finalize_marks(ctx->L, ga, g->edge_cap, g->cnt(), copy, copy_cap);
    if (g->download_pending) {
        join_side(ctx->L, 0);
        g->download_pending = false;
    }
    CU(ctx, cudaGetLastError());
    CU(ctx, end_stage(g, ST_TRANSITIVE));
    g->state = SS_REDUCED;
    return RALA_B200_OK;
}

// graph.cpp:1281-1318
extern "C" int rala_b200_graph_transitive(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->world > 1) return refuse_shard(g, "transitive");
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "transitive: build first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_TRANSITIVE));
    const GraphArrays ga = g->graph_view();
    int rc = transitive_stage(g, ga, nullptr);
    return rc ? rc : marks_stage(g, ga, g->out_marked, g->out_marked_cap);
}

static int run_eager(rala_b200_graph* g) {
    int rc = rala_b200_graph_classify(g);
    if (!rc) rc = rala_b200_graph_retrim(g);
    if (!rc) rc = rala_b200_graph_retrim_promote(g, nullptr);
    if (!rc) rc = rala_b200_graph_finalize(g);
    g->in_run = true;    // the transitive stage follows: it joins the forked edge download
    if (!rc) rc = rala_b200_graph_build(g);
    g->in_run = false;
    if (!rc) rc = rala_b200_graph_transitive(g);
    if (g->download_pending) {   // build forked, transitive failed before joining
        join_side(g->ctx->L, 0);
        g->download_pending = false;
    }
    return rc;
}

// Everything the sequence of stream operations of one run depends on.  The chain itself has no host
// synchronisation and every data-dependent size stays on the device, so for a fixed key the ~45 stream
// operations (27 kernels, memsets, small copies) are identical from run to run: the second run with a key is
// captured into a CUDA graph and later runs replay it with one launch.
struct RunKey {
    const void *rec, *recs, *piles, *piles_initial, *events, *segs, *dbuf, *edges, *col, *scan_pool, *ovl0, *inl0, *hills, *heavy;
    const void *out_edges, *out_marked;
    uint32_t n_rec, n_piles, n_hills, cap, ev_cap, edge_cap, heavy_cap, t0, out_edges_cap, out_marked_cap;
    int world, rank, coop_blocks;
    bool piles_fresh, skip_clean_retrim;
};

// host-side bookkeeping a run leaves behind (restored after a replay)
struct RunHostState {
    int ovl_cur, inl_cur, slot_ovl, slot_inl, next_slot, final_time_base_slot;
    SessionState state;
    bool final_lists_ready, piles_dirty, piles_fresh, promote_pending;
    uint32_t retrim_passes;
    size_t scan_used;
    bool scan_zeroed;
    uint32_t step_cleared;
};

struct RunGraph {
    RunKey key{};
    bool seen = false;          // the key was run once (eagerly): capture on the next occurrence
    cudaGraphExec_t exec = nullptr;
    RunHostState after{};
    uint64_t launches = 0;      // kernels inside the graph
};

static RunKey run_key(const rala_b200_graph* g) {
    RunKey k;
    memset(&k, 0, sizeof(k));   // padding included: keys are compared with memcmp
    k.rec = g->rec.p; k.recs = g->recs.buf.p; k.piles = g->piles.p; k.piles_initial = g->piles_initial.p;
    k.events = g->events.p; k.segs = g->segs.p; k.dbuf = g->dbuf.p; k.edges = g->edges.p; k.col = g->col.p;
    k.scan_pool = g->scan_pool.p; k.ovl0 = g->ovl[0].buf.p; k.inl0 = g->inl[0].buf.p; k.hills = g->hills.p;
    k.heavy = g->heavy.p;   // sized from n_piles, which can shrink and grow back without a new allocation
    k.n_rec = g->n_rec; k.n_piles = g->n_piles; k.n_hills = g->n_hills; k.cap = g->cap; k.ev_cap = g->ev_cap;
    k.edge_cap = g->edge_cap; k.heavy_cap = g->heavy_cap; k.t0 = g->t0;
    k.out_edges = g->out_edges; k.out_marked = g->out_marked; k.out_edges_cap = g->out_edges_cap; k.out_marked_cap = g->out_marked_cap;
    k.world = g->world; k.rank = g->rank; k.coop_blocks = g->ctx->coop_blocks;
    k.piles_fresh = g->piles_fresh; k.skip_clean_retrim = g->skip_clean_retrim;
    return k;
}

static RunHostState host_state(const rala_b200_graph* g) {
    return RunHostState{g->ovl_cur, g->inl_cur, g->slot_ovl, g->slot_inl, g->next_slot, g->final_time_base_slot, g->state,
                        g->final_lists_ready, g->piles_dirty, g->piles_fresh, g->promote_pending, g->retrim_passes, g->scan_used,
                        g->scan_zeroed, g->step_cleared};
}

static void drop_run_graphs(rala_b200_graph* g) {
    if (!g->run_graphs) return;
    for (int i = 0; i < 2; ++i)
        if (g->run_graphs[i].exec) cudaGraphExecDestroy(g->run_graphs[i].exec);
    delete[] g->run_graphs;
    g->run_graphs = nullptr;
}

extern "C" int rala_b200_graph_use_cuda_graph(rala_b200_graph* g, int enabled) {
    if (!g) return RALA_B200_ERR_ARG;
    g->use_cuda_graph = enabled != 0;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_run(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->world > 1) return refuse_shard(g, "run");
    if (!g->use_cuda_graph) return run_eager(g);
    if (g->state < SS_INPUTS) return fail(ctx, RALA_B200_ERR_STATE, "run: set_overlaps and set_piles first");
    CU(ctx, cudaSetDevice(ctx->device));
    if (!g->run_graphs) g->run_graphs = new RunGraph[2];
    const RunKey key = run_key(g);
    RunGraph& R = g->run_graphs[key.piles_fresh ? 1 : 0];
    if (!R.seen || memcmp(&R.key, &key, sizeof(key)) != 0) {   // new shape: run it eagerly once (this also sizes every buffer)
        if (R.exec) cudaGraphExecDestroy(R.exec);
        R.exec = nullptr;
        R.key = key;
        R.seen = true;
        return run_eager(g);
    }
    if (!R.exec) {
        const uint64_t launches0 = ctx->L.count;
        cudaGraph_t graph = nullptr;
        CU(ctx, cudaStreamBeginCapture(ctx->L.stream, cudaStreamCaptureModeThreadLocal));
        g->capturing = true;
        const int rc = run_eager(g);
        g->capturing = false;
        const cudaError_t e = cudaStreamEndCapture(ctx->L.stream, &graph);
        if (rc || e != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            R.seen = false;
            ctx->L.count = launches0;
            if (rc) return rc;
            return fail(ctx, RALA_B200_ERR_CUDA, "run: stream capture failed: %s", cudaGetErrorString(e));
        }
        const cudaError_t ei = cudaGraphInstantiate(&R.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) {
            R.exec = nullptr;
            R.seen = false;
            return fail(ctx, RALA_B200_ERR_CUDA, "run: cudaGraphInstantiate failed: %s", cudaGetErrorString(ei));
        }
        R.launches = ctx->L.count - launches0;
        R.after = host_state(g);
        ctx->L.count = launches0;   // counted per replay below
    }
    CU(ctx, cudaGraphLaunch(R.exec, ctx->L.stream));
    ctx->L.count += R.launches;
    const RunHostState& a = R.after;
    g->ovl_cur = a.ovl_cur; g->inl_cur = a.inl_cur; g->slot_ovl = a.slot_ovl; g->slot_inl = a.slot_inl; g->next_slot = a.next_slot;
    g->final_time_base_slot = a.final_time_base_slot; g->state = a.state; g->final_lists_ready = a.final_lists_ready;
    g->piles_dirty = a.piles_dirty; g->piles_fresh = a.piles_fresh; g->promote_pending = a.promote_pending; g->retrim_passes = a.retrim_passes; g->scan_used = a.scan_used;
    g->scan_zeroed = a.scan_zeroed; g->step_cleared = a.step_cleared;
    for (int i = 0; i < RALA_B200_N_STAGES; ++i) g->ev_valid[i] = false;   // no stage timers inside a graph
    return RALA_B200_OK;
}

int read_counters(rala_b200_graph* g, uint32_t* h) {
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(h, g->counters.p, C_COUNT * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    if (g->scan_pool_exhausted)
        return fail(ctx, RALA_B200_ERR_LIMIT, "the look-back status pool was exhausted inside a stage (%zu words): the results are void", g->scan_pool_words);
    if (h[C_OVERFLOW] || (g->state >= SS_CLASSIFIED && (h[g->slot_ovl] > g->cap || h[g->slot_inl] > g->cap)) || h[C_EV] > g->ev_cap ||
        h[C_EV_FIRST] > g->ev_cap || h[C_HILL] > g->cap)
        return fail(ctx, RALA_B200_ERR_LIMIT, "a device list overflowed its capacity (cap=%u events=%u hills=%u heavy items=%u)",
                    g->cap, h[C_EV], h[C_HILL], h[C_HEAVY]);
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_counts(rala_b200_graph* g, rala_b200_counts_t* out) {
    if (!g || !out) return RALA_B200_ERR_ARG;
    uint32_t h[C_COUNT];
    int rc = materialize_final_lists(g);
    if (!rc) rc = read_counters(g, h);
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    out->n_records = g->n_rec;
    out->n_overlaps = g->state >= SS_CLASSIFIED ? h[g->slot_ovl] : 0;
    out->n_internals = g->state >= SS_CLASSIFIED ? h[g->slot_inl] : 0;
    // the first pass's k_apply_deaths moved its counts to *_FIRST (FinalPassReset)
    out->n_candidates = g->state >= SS_CLASSIFIED ? h[C_EV_FIRST] : h[C_EV];
    out->n_rounds = g->state >= SS_CLASSIFIED ? h[C_ROUNDS_FIRST] : h[C_ROUNDS];
    out->n_final_candidates = g->state >= SS_FINALIZED ? h[C_EV] : 0;
    out->n_final_rounds = g->state >= SS_FINALIZED ? h[C_ROUNDS] : 0;
    out->n_piles = g->n_piles;
    out->n_alive_piles = h[C_ALIVE];
    out->n_nodes = h[C_NODES];
    out->n_edges = h[C_EDGES];
    out->n_two_hop = (uint64_t) h[C_HOP_LO] | ((uint64_t) h[C_HOP_HI] << 32);
    out->n_transitive_pairs = h[C_PAIRS];
    out->n_heavy_items = h[C_HEAVY];
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_hill_coverage(rala_b200_graph* g, uint32_t* cov_out) {
    if (!g || (g->n_hills && !cov_out)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (g->n_hills)
        CU(ctx, cudaMemcpyAsync(cov_out, g->hills.as<uint32_t>() + 3 * (size_t) g->n_hills, (size_t) g->n_hills * 4,
                                cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_piles(rala_b200_graph* g, rala_pile_t* piles_out) {
    if (!g || !piles_out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    launch_unpack_piles(ctx->L, g->piles.as<uint2>(), g->piles_raw.as<uint2>(), g->n_piles);
    CU(ctx, cudaMemcpyAsync(piles_out, g->piles_raw.p, (size_t) g->n_piles * 8, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_connections(rala_b200_graph* g, uint32_t* ab_out) {
    if (!g || !ab_out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "get_connections: classify first");
    uint32_t h[C_COUNT];
    int rc = read_counters(g, h);
    if (rc) return rc;
    uint32_t n = h[g->slot_ovl];
    if (!n) return RALA_B200_OK;
    DevBuf tmp;
    CU(ctx, tmp.reserve((size_t) n * 8));
    launch_list_connections(ctx->L, g->ovl[g->ovl_cur].view, g->cnt() + g->slot_ovl, g->cap, tmp.as<uint32_t>());
    CU(ctx, cudaMemcpyAsync(ab_out, tmp.p, (size_t) n * 8, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    tmp.release();
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_lists(rala_b200_graph* g, rala_ovl_t* overlaps_out, rala_ovl_t* internals_out) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "get_lists: classify first");
    uint32_t h[C_COUNT];
    int rc = materialize_final_lists(g);
    if (!rc) rc = read_counters(g, h);
    if (rc) return rc;
    DevBuf tmp;
    for (int which = 0; which < 2; ++which) {
        rala_ovl_t* out = which ? internals_out : overlaps_out;
        uint32_t n = which ? h[g->slot_inl] : h[g->slot_ovl];
        if (!out || !n) continue;
        CU(ctx, tmp.reserve((size_t) n * 28));
        launch_list_to_aos(ctx->L, which ? g->inl[g->inl_cur].view : g->ovl[g->ovl_cur].view,
                           g->cnt() + (which ? g->slot_inl : g->slot_ovl), g->cap, tmp.as<uint32_t>());
        CU(ctx, cudaMemcpyAsync(out, tmp.p, (size_t) n * 28, cudaMemcpyDeviceToHost, ctx->L.stream));
        CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    }
    tmp.release();
    return RALA_B200_OK;
}

// graph.cpp:523 / 882-1054: the host filtered `overlaps` (Graph::preprocess(overlaps, sensitive_path) only ever drops
// entries); the device list is replaced by what is left, in the same order.
extern "C" int rala_b200_graph_set_kept_overlaps(rala_b200_graph* g, const rala_ovl_t* kept, uint64_t n) {
    if (!g || (n && !kept)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state != SS_FINALIZED) return fail(ctx, RALA_B200_ERR_STATE, "set_kept_overlaps: finalize first");
    if (n > g->cap) return fail(ctx, RALA_B200_ERR_LIMIT, "set_kept_overlaps: %llu entries exceed the list capacity %u", (unsigned long long) n, g->cap);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = materialize_final_lists(g);   // `internals` keeps its final form
    if (rc) return rc;
    DevBuf tmp;
    CU(ctx, tmp.reserve((size_t) n * 28 + 16));
    if (n) CU(ctx, cudaMemcpyAsync(tmp.p, kept, (size_t) n * 28, cudaMemcpyHostToDevice, ctx->L.stream));
    launch_aos_to_list(ctx->L, tmp.as<uint32_t>(), (uint32_t) n, g->piles.as<uint2>(), g->n_piles, g->ovl[g->ovl_cur].view);
    const uint32_t n32 = (uint32_t) n;
    CU(ctx, cudaMemcpyAsync(g->cnt() + g->slot_ovl, &n32, 4, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    tmp.release();
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_seq_to_node(rala_b200_graph* g, uint32_t* out) {
    if (!g || !out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "get_seq_to_node: build first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(out, g->seq_to_node.p, (size_t) g->n_piles * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

// the CSR adjacency build wrote for the transitive pass (k_scan_piles / k_emit_edges); the transitive pass only reads it
extern "C" int rala_b200_graph_get_csr(rala_b200_graph* g, uint32_t* row_ptr_out, uint32_t* col_out, uint32_t* col_eid_out) {
    if (!g || !row_ptr_out || !col_out || !col_eid_out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "get_csr: build first");
    uint32_t h[C_COUNT];
    int rc = read_counters(g, h);
    if (rc) return rc;
    const uint32_t n_nodes = h[C_NODES], n_edges = h[C_EDGES];
    CU(ctx, cudaMemcpyAsync(row_ptr_out, g->row_ptr.p, ((size_t) n_nodes + 1) * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    if (n_edges) {
        CU(ctx, cudaMemcpyAsync(col_out, g->col.p, (size_t) n_edges * 8, cudaMemcpyDeviceToHost, ctx->L.stream));
        CU(ctx, cudaMemcpyAsync(col_eid_out, g->col_eid.p, (size_t) n_edges * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    }
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_edges(rala_b200_graph* g, rala_edge_t* out) {
    if (!g || !out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "get_edges: build first");
    uint32_t h[C_COUNT];
    int rc = read_counters(g, h);
    if (rc) return rc;
    uint32_t n = h[C_EDGES];
    if (!n) return RALA_B200_OK;
    // columns -> rows on the device, then one contiguous copy
    CU(ctx, g->edges_aos.reserve((size_t) g->edge_cap * 12));
    launch_pack_edges(ctx->L, ctx->L.stream, g->graph_view(), g->edge_cap, g->cnt() + C_EDGES, g->edges_aos.as<uint32_t>());
    CU(ctx, cudaMemcpyAsync(out, g->edges_aos.p, (size_t) n * 12, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_marked(rala_b200_graph* g, uint8_t* out) {
    if (!g || !out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_REDUCED) return fail(ctx, RALA_B200_ERR_STATE, "get_marked: transitive first");
    uint32_t h[C_COUNT];
    int rc = read_counters(g, h);
    if (rc) return rc;
    if (h[C_EDGES]) CU(ctx, cudaMemcpyAsync(out, g->marked.p, h[C_EDGES], cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

// suffix_edges_ / prefix_edges_ of every node as the reference keeps them (ascending edge id), optionally after the removal of
// the marked edges: graph.cpp:603-606 / 622-625 and 2118-2151
extern "C" int rala_b200_graph_get_adjacency(rala_b200_graph* g, int which, int skip_marked, uint32_t* off_out, uint32_t* ids_out,
                                             uint64_t* n_ids_out) {
    if (!g || !off_out || !ids_out || !n_ids_out || which < 0 || which > 1) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "get_adjacency: build first");
    if (skip_marked && g->state < SS_REDUCED) return fail(ctx, RALA_B200_ERR_STATE, "get_adjacency: transitive first (or pass skip_marked = 0)");
    uint32_t h[C_COUNT];
    int rc = read_counters(g, h);
    if (rc) return rc;
    const uint32_t n_nodes = h[C_NODES], n_edges = h[C_EDGES];
    *n_ids_out = 0;
    CU(ctx, cudaSetDevice(ctx->device));
    DevBuf deg, rp, tmp, sorted;
    CU(ctx, deg.reserve(((size_t) n_nodes + 8) * 4));
    CU(ctx, rp.reserve(((size_t) n_nodes + 8) * 4));
    CU(ctx, tmp.reserve(((size_t) n_edges + 8) * 4));
    CU(ctx, sorted.reserve(((size_t) n_edges + 8) * 4));
    GraphArrays ga = g->graph_view();
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, (uint64_t) n_nodes + 1, &status, &ticket);
    launch_adjacency_view(ctx->L, which ? ga.dst : ga.src, skip_marked ? ga.marked : nullptr, g->cnt() + C_EDGES, g->edge_cap, n_nodes,
                          deg.as<uint32_t>(), rp.as<uint32_t>(), tmp.as<uint32_t>(), sorted.as<uint32_t>(), status, ticket);
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(off_out, rp.p, ((size_t) n_nodes + 1) * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    const uint32_t total = off_out[n_nodes];
    if (total) CU(ctx, cudaMemcpyAsync(ids_out, sorted.p, (size_t) total * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    *n_ids_out = total;
    deg.release(); rp.release(); tmp.release(); sorted.release();
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_stage_ms(rala_b200_graph* g, float* ms_out) {
    if (!g || !ms_out) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    for (int i = 0; i < RALA_B200_N_STAGES; ++i) {
        ms_out[i] = 0.f;
        if (g->ev_valid[i]) CU(ctx, cudaEventElapsedTime(&ms_out[i], g->ev_start[i], g->ev_stop[i]));
    }
    return RALA_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// stateless stages
// ---------------------------------------------------------------------------------------------
extern "C" int rala_b200_trim_classify(rala_b200_ctx* ctx, rala_ovl_t* ovl, uint64_t n, const rala_pile_t* piles,
                                       uint32_t n_piles, uint8_t* type_out) {
    if (!ctx || (n && (!ovl || !type_out)) || (n_piles && !piles)) return RALA_B200_ERR_ARG;
    if (n >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many records");
    if (n == 0) return RALA_B200_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    DevBuf rec, praw, ppacked, types;
    CU(ctx, rec.reserve((size_t) n * 28));
    CU(ctx, praw.reserve((size_t) n_piles * 8 + 16));
    CU(ctx, ppacked.reserve((size_t) n_piles * 8 + 16));
    CU(ctx, types.reserve(n));
    CU(ctx, cudaMemcpyAsync(rec.p, ovl, (size_t) n * 28, cudaMemcpyHostToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(praw.p, piles, (size_t) n_piles * 8, cudaMemcpyHostToDevice, ctx->L.stream));
    launch_pack_piles(ctx->L, praw.as<uint2>(), nullptr, ppacked.as<uint2>(), n_piles);
    launch_trim_classify_aos(ctx->L, rec.as<uint32_t>(), (uint32_t) n, ppacked.as<uint2>(), n_piles, types.as<uint8_t>());
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(ovl, rec.p, (size_t) n * 28, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(type_out, types.p, n, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    rec.release(); praw.release(); ppacked.release(); types.release();
    return RALA_B200_OK;
}

// the stateless reduction on a throw-away session: its node and edge arrays hold the caller's graph
static int transitive_reduce_on(rala_b200_graph* g, uint32_t n_nodes, uint32_t n_edges, const rala_edge_t* edges, uint8_t* marked_out,
                                uint64_t* n_pairs) {
    rala_b200_ctx* ctx = g->ctx;
    cudaStream_t s = ctx->L.stream;
    int rc = reserve_nodes(g, n_nodes);
    if (!rc) rc = reserve_edges(g, n_edges);
    if (rc) return rc;
    CU(ctx, g->edges_aos.reserve((size_t) n_edges * 12));
    const GraphArrays ga = g->graph_view();
    CU(ctx, cudaMemcpyAsync(g->edges_aos.p, edges, (size_t) n_edges * 12, cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemcpy2DAsync(ga.src, 4, g->edges_aos.as<char>(), 12, 4, n_edges, cudaMemcpyDeviceToDevice, s));
    CU(ctx, cudaMemcpy2DAsync(ga.dst, 4, g->edges_aos.as<char>() + 4, 12, 4, n_edges, cudaMemcpyDeviceToDevice, s));
    CU(ctx, cudaMemcpy2DAsync(ga.len, 4, g->edges_aos.as<char>() + 8, 12, 4, n_edges, cudaMemcpyDeviceToDevice, s));
    uint32_t h[C_COUNT];
    memset(h, 0, sizeof(h));
    h[C_NODES] = n_nodes;
    h[C_EDGES] = n_edges;
    CU(ctx, cudaMemcpyAsync(g->counters.p, h, sizeof(h), cudaMemcpyHostToDevice, s));
    CU(ctx, begin_stage(g, ST_TRANSITIVE));
    rc = csr_from_edge_list(g);
    if (!rc) rc = transitive_stage(g, ga, nullptr);
    if (!rc) rc = marks_stage(g, ga, nullptr, 0u);
    if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(marked_out, g->marked.p, n_edges, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(h, g->counters.p, sizeof(h), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    if (h[C_OVERFLOW])
        return fail(ctx, RALA_B200_ERR_LIMIT, "transitive_reduce: more than 2048 destinations of one node in one hash chunk, "
                                              "or more than 2^32 heavy work items");
    if (n_pairs) *n_pairs = h[C_PAIRS];
    return RALA_B200_OK;
}

extern "C" int rala_b200_transitive_reduce(rala_b200_ctx* ctx, uint32_t n_nodes, uint64_t n_edges, const rala_edge_t* edges,
                                           uint8_t* marked_out, uint64_t* n_pairs) {
    if (!ctx || (n_edges && (!edges || !marked_out))) return RALA_B200_ERR_ARG;
    if (n_edges >= (1ull << 31) || (n_edges & 1)) return fail(ctx, RALA_B200_ERR_ARG, "edge count must be even and < 2^31 (pair(e) = e ^ 1)");
    if (n_pairs) *n_pairs = 0;
    if (n_edges == 0) return RALA_B200_OK;
    for (uint64_t i = 0; i < n_edges; ++i) {
        if (edges[i].src >= n_nodes || edges[i].dst >= n_nodes) return fail(ctx, RALA_B200_ERR_ARG, "edge %llu references a node >= n_nodes", (unsigned long long) i);
    }
    CU(ctx, cudaSetDevice(ctx->device));
    rala_b200_graph* g = nullptr;
    int rc = rala_b200_graph_create(ctx, &g);
    if (rc) return rc;
    rc = transitive_reduce_on(g, n_nodes, (uint32_t) n_edges, edges, marked_out, n_pairs);
    rala_b200_graph_destroy(g);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// Multi-GPU phases (one process per GPU).  The records are sharded by contiguous file range, the pile
// table is replicated; the collectives between the phases belong to the caller (NCCL through
// torch.distributed in rala_b200/multi.py), which passes DEVICE pointers of its exchange buffers:
//   phase_events -> export_padded -> [all-gather] -> import_gathered -> phase_resolve(1) -> phase_survivors
//   -> export_list_counts -> [all-gather] -> phase_final_events_gathered -> export_padded -> [all-gather]
//   -> import_gathered -> phase_resolve(0) -> phase_emit_edges -> export_padded -> [all-gather] -> import_gathered
//   -> phase_csr -> phase_transitive -> export_marks -> [all-reduce(max)] -> phase_marks
// No call reads a count back to the host: counts travel inside the exchange blocks (k_export_padded has the layout),
// the time bases of the final pass are computed on the device, and a block too small for its rank's elements raises
// the session's overflow flag.
// ---------------------------------------------------------------------------------------------
extern "C" int rala_b200_graph_set_shard(rala_b200_graph* g, uint32_t t0, int rank, int world) {
    if (!g || world < 1 || rank < 0 || rank >= world) return RALA_B200_ERR_ARG;
    g->t0 = t0;
    g->rank = rank;
    g->world = world;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_phase_events(rala_b200_graph* g) { return g ? phase_events(g) : RALA_B200_ERR_ARG; }

extern "C" int rala_b200_graph_phase_resolve(rala_b200_graph* g, int first_pass) {
    if (!g) return RALA_B200_ERR_ARG;
    return first_pass ? phase_resolve(g, true) : phase_final_resolve(g);
}

extern "C" int rala_b200_graph_phase_survivors(rala_b200_graph* g) { return g ? phase_survivors(g) : RALA_B200_ERR_ARG; }

// node ids (replicated) + the edges of the LOCAL overlaps, in local list order, with global node ids
extern "C" int rala_b200_graph_phase_emit_edges(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state != SS_FINALIZED) return fail(ctx, RALA_B200_ERR_STATE, "emit_edges: finalize first");
    int rc = emit_edges(g, false);   // the CSR is built over the edges of all ranks (phase_csr)
    if (rc) return rc;
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_export_padded(rala_b200_graph* g, int kind, uint32_t* d_block, uint32_t cap) {
    if (!g || !d_block || cap == 0 || (kind != 0 && kind != 1)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (kind == 0) {
        Events ev = g->events_view();
        launch_export_padded(ctx->L, ev.v, ev.c, ev.t, g->cnt() + C_EV, g->ev_cap, cap, d_block);
    } else {
        GraphArrays ga = g->graph_view();
        launch_export_padded(ctx->L, ga.src, ga.dst, ga.len, g->cnt() + C_EDGES, g->edge_cap, cap, d_block);
    }
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_import_gathered(rala_b200_graph* g, int kind, const uint32_t* d_gathered, uint32_t cap, int world) {
    if (!g || !d_gathered || cap == 0 || world < 1 || (kind != 0 && kind != 1)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    const uint64_t total_cap = (uint64_t) cap * world;
    if (total_cap >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "exchange capacity too large");
    if (kind == 0) {
        int rc = reserve_events(g, (uint32_t) total_cap);   // the local events were exported before
        if (rc) return rc;
        Events ev = g->events_view();
        launch_import_gathered(ctx->L, d_gathered, cap, (uint32_t) world, ev.v, ev.c, ev.t, g->ev_cap, g->cnt() + C_EV, g->cnt() + C_OVERFLOW);
        CU(ctx, clear_earliest_events(g));
        launch_events_first(ctx->L, g->events_view(), g->cnt() + C_EV, g->ev_cap, resolve_bufs(g).first);
    } else {
        int rc = reserve_edges(g, (uint32_t) total_cap);     // the local edges were exported before
        if (rc) return rc;
        GraphArrays ga = g->graph_view();
        launch_import_gathered(ctx->L, d_gathered, cap, (uint32_t) world, ga.src, ga.dst, ga.len, g->edge_cap, g->cnt() + C_EDGES, g->cnt() + C_OVERFLOW);
    }
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

extern "C" uint64_t rala_b200_exchange_block_words(int kind, uint32_t cap) {
    (void) kind;
    return 3ull * cap + 4ull;
}

extern "C" int rala_b200_graph_export_list_counts(rala_b200_graph* g, uint32_t* d_pair) {
    if (!g || !d_pair) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_CLASSIFIED) return fail(ctx, RALA_B200_ERR_STATE, "export_list_counts: classify first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(d_pair, g->cnt() + g->slot_ovl, 4, cudaMemcpyDeviceToDevice, ctx->L.stream));
    CU(ctx, cudaMemcpyAsync(d_pair + 1, g->cnt() + g->slot_inl, 4, cudaMemcpyDeviceToDevice, ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_phase_final_events_gathered(rala_b200_graph* g, const uint32_t* d_counts, int world) {
    if (!g || !d_counts || world < 1) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    launch_time_bases(ctx->L, d_counts, (uint32_t) g->rank, (uint32_t) world, g->cnt() + C_TBASE_OVL);
    return phase_final_events(g, g->cnt() + C_TBASE_OVL, C_TBASE_INL);
}

// CSR over ALL edges (replicated on every rank)
extern "C" int rala_b200_graph_phase_csr(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = csr_from_edge_list(g);
    return rc ? rc : end_build(g);
}

// T(e) for the candidate edges whose source node this rank owns
extern "C" int rala_b200_graph_phase_transitive(rala_b200_graph* g) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (g->state < SS_BUILT) return fail(ctx, RALA_B200_ERR_STATE, "transitive: build first");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, begin_stage(g, ST_TRANSITIVE));
    const GraphArrays ga = g->graph_view();
    uint32_t* node_range = g->work_counter.as<uint32_t>() + 4;
    launch_node_range(ctx->L, ga, g->cnt(), (uint32_t) g->rank, (uint32_t) g->world, node_range);
    return transitive_stage(g, ga, node_range);
}

extern "C" int rala_b200_graph_export_marks(rala_b200_graph* g, uint8_t* d_T, uint32_t n) {
    if (!g || (n && !d_T)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (n) CU(ctx, cudaMemcpyAsync(d_T, g->T.p, n, cudaMemcpyDeviceToDevice, ctx->L.stream));
    return RALA_B200_OK;
}

// merged T in, marked(e) = T(e) | T(e^1) out
extern "C" int rala_b200_graph_phase_marks(rala_b200_graph* g, const uint8_t* d_T, uint32_t n) {
    if (!g || (n && !d_T)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (n) CU(ctx, cudaMemcpyAsync(g->T.p, d_T, n, cudaMemcpyDeviceToDevice, ctx->L.stream));
    return marks_stage(g, g->graph_view(), nullptr, 0u);
}
