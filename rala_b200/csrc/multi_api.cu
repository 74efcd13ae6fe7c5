// multi_api.cu — the multi-GPU session of the C ABI (include/rala_b200.h, "Multi-GPU session"): `world` ranks, one
// per GPU, each with its own single-GPU session (session.h) for the local stages and one arena of the exchange
// fabric (fabric.cuh).  A step is a fixed sequence of kernels per rank; ranks only meet in device-side barriers, so
// the host enqueues and never waits, and every rank's step is captured once and replayed as one CUDA graph.
//
// Reference stages (rvaser/rala, single process) and who runs them here:
//   graph.cpp:443-518  classify loop            every rank on its own file range; containment events go to the
//                                               owner of the victim pile, which resolves them (fabric.cu)
//   graph.cpp:831-877  final containment        the same with list positions as times
//   graph.cpp:552-632  nodes, edges, adjacency  node ids replicated (a scan of the replicated pile table), edges to
//                                               the owner of their source node, which builds its CSR rows
//   graph.cpp:1281-1318 transitive marks        owner of the source node, on the replicated CSR; results go back to
//                                               the rank that emitted the edge, which forms marked(e) = T(e) | T(e^1)
#include <cstddef>

#include "fabric.cuh"
#include "session.h"

using namespace rb;

namespace {

// word offsets in FabricRank::stage (staged construct)
enum StageWords : size_t {
    SW_LO = 0,                      // kMaxSegs + 1: local start of every segment of `overlaps`, then its end
    SW_BOX = 128,                   // kSegMail: this rank's counts of a staged pass, pushed to every peer
    SW_FIN_N = 384,                 // kMaxSegs: local entries of every segment (final containment events)
    SW_FIN_BASE = 448,              // kMaxSegs: global time of the first of them
    SW_ZERO = 512,                  // a word that stays 0
    SW_WORDS = 520
};
constexpr size_t kStageRunsByte = 4096;   // EdgeRuns

struct FabricRank {
    rala_b200_ctx* ctx = nullptr;
    rala_b200_graph* g = nullptr;
    int device = 0, rank = 0;
    DevBuf arena;
    Peers P{};
    ArenaLayout A{};
    DevBuf meta, out_cnt, tmin, wait, col_eid, T;
    DevBuf stage;                  // staged construct: segment bounds, outgoing counts, time bases, edge runs (StageWords)
    std::vector<uint32_t> stage_host;   // host copy of the words uploaded to `stage` (kept alive for the async copies)
    void* ipc_mapped[kMaxRanks]{};
    cudaGraphExec_t exec[2] = {nullptr, nullptr};   // [0] repeated run, [1] first run after set_piles (phase_events copies the table the other way)
    uint64_t graph_launches[2] = {0, 0};
    cudaEvent_t ev[2]{};
    uint64_t n_rec = 0;
    int resolve_blocks = 1;   // co-resident grid of the resolution kernel (shared with the other ranks on the same device)

    BuildMeta* meta_dev() const { return meta.as<BuildMeta>(); }
    uint32_t* cnt_ev(int pass) const { return out_cnt.as<uint32_t>() + pass * kMaxRanks; }
    uint32_t* cnt_edges() const { return out_cnt.as<uint32_t>() + 2 * kMaxRanks; }
    uint32_t* ctl(int pass) const { return out_cnt.as<uint32_t>() + 3 * kMaxRanks + pass * (kResolveCtlBytes / 4); }
    FabricHdr* hdr() const { return arena.as<FabricHdr>(); }
    uint32_t* stage_w(size_t word) const { return stage.as<uint32_t>() + word; }
    EdgeRuns* runs_dev() const { return reinterpret_cast<EdgeRuns*>(stage.as<uint8_t>() + kStageRunsByte); }
    template <class T> T* sec(size_t off) const { return reinterpret_cast<T*>(arena.as<uint8_t>() + off); }
};

}  // namespace

struct rala_b200_multi {
    int world = 1, first_rank = 0, n_local = 1;
    std::vector<FabricRank> ranks;
    std::string error;
    uint64_t caps[RALA_B200_N_CAPS]{};
    uint32_t n_piles = 0;
    bool reserved = false, connected = false;
    bool use_graph = true;
    uint32_t barrier_timeout_ms = 10000;
    int runs_seen[2] = {0, 0};   // per graph variant: 0 next run is eager, 1 next run is captured, 2 replay
    uint32_t n_hills = 0;
    // staged construct (rala_b200_multi_classify .. finish): what every rank's lists hold, replicated through seg_mail
    int staged = 0;                  // 0 none, 2 classified (list passes may follow), 3 finished
    bool staged_edges = false;       // the last edge list came from finish: ids in runs (EdgeRuns), not one range per rank
    uint32_t n_seg = 0;
    std::vector<uint32_t> seg;       // [kMaxSegs][world]: entries of segment s of `overlaps` on rank r
    std::vector<uint32_t> inl;       // [world]: entries of `internals` on rank r (one rank-major segment: it only shrinks)
    std::vector<uint32_t> dov;       // [kMaxSegs][world]: dovetails of the final `overlaps` (edges / 2)
    EdgeRuns runs{};
};

static int mfail(rala_b200_multi* m, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (m) m->error = buf;
    return code;
}

#define MCU(m, call)                                                                                     \
    do {                                                                                                 \
        cudaError_t err__ = (call);                                                                      \
        if (err__ != cudaSuccess)                                                                        \
            return mfail((m), RALA_B200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), \
                         __FILE__, __LINE__);                                                            \
    } while (0)

// a failing call of the single-GPU layer: carry its message over
#define MRC(m, fr, call)                                                                 \
    do {                                                                                 \
        int rc__ = (call);                                                               \
        if (rc__) return mfail((m), rc__, "rank %d: %s", (fr).rank, (fr).ctx->error.c_str()); \
    } while (0)

static void drop_graphs(rala_b200_multi* m) {
    for (FabricRank& fr : m->ranks) {
        for (int v = 0; v < 2; ++v) {
            if (fr.exec[v]) {
                cudaSetDevice(fr.device);
                cudaGraphExecDestroy(fr.exec[v]);
                fr.exec[v] = nullptr;
            }
        }
    }
    m->runs_seen[0] = m->runs_seen[1] = 0;
}

static void disconnect(rala_b200_multi* m) {
    for (FabricRank& fr : m->ranks) {
        cudaSetDevice(fr.device);
        for (int q = 0; q < kMaxRanks; ++q) {
            if (fr.ipc_mapped[q]) {
                cudaIpcCloseMemHandle(fr.ipc_mapped[q]);
                fr.ipc_mapped[q] = nullptr;
            }
            fr.P.base[q] = nullptr;
        }
    }
    m->connected = false;
}

extern "C" int rala_b200_multi_create(rala_b200_multi** out, const int* devices, int n_local, int first_rank, int world) {
    if (!out || !devices || n_local < 1 || world < 1 || world > kMaxRanks || first_rank < 0 || first_rank + n_local > world)
        return RALA_B200_ERR_ARG;
    *out = nullptr;
    rala_b200_multi* m = new rala_b200_multi();
    m->world = world;
    m->first_rank = first_rank;
    m->n_local = n_local;
    m->ranks.resize(n_local);
    for (int k = 0; k < n_local; ++k) {
        FabricRank& fr = m->ranks[k];
        fr.device = devices[k];
        fr.rank = first_rank + k;
        int rc = rala_b200_create(&fr.ctx, devices[k]);
        if (!rc) rc = rala_b200_graph_create(fr.ctx, &fr.g);
        if (!rc) rc = rala_b200_graph_set_shard(fr.g, 0, fr.rank, world);
        if (rc) {
            rala_b200_multi_destroy(m);
            return rc;
        }
        cudaEventCreate(&fr.ev[0]);
        cudaEventCreate(&fr.ev[1]);
        {   // the driver's own memset / copy kernels load lazily too: use them once before any barrier can be waiting
            DevBuf warm;
            if (warm.reserve(8192) == cudaSuccess) {
                cudaMemsetAsync(warm.p, 0, 4096, fr.ctx->L.stream);
                cudaMemsetAsync(warm.p, 0xFF, 28, fr.ctx->L.stream);
                cudaMemcpyAsync(warm.as<char>() + 4096, warm.p, 4096, cudaMemcpyDeviceToDevice, fr.ctx->L.stream);
                cudaMemcpyAsync(warm.as<char>() + 4096, warm.p, 4, cudaMemcpyDeviceToDevice, fr.ctx->L.stream);
                cudaStreamSynchronize(fr.ctx->L.stream);
                warm.release();
            }
            cudaGetLastError();
        }
        fr.P.rank = fr.rank;
        fr.P.world = world;
    }
    for (FabricRank& fr : m->ranks) {   // the resolution kernels of all ranks on one device must be resident together
        int sharing = 0;
        for (const FabricRank& other : m->ranks) sharing += other.device == fr.device ? 1 : 0;
        cudaSetDevice(fr.device);
        // A rank that has its GPU to itself takes what fits minus one block per SM (nothing else of this rank runs beside
        // the resolution); ranks that share a GPU take half of their share, so that everybody's grid is resident at once.
        const int all = fabric_resolve_max_blocks();
        const int fit = sharing == 1 ? all - kNumSMs : all / (2 * sharing);
        fr.resolve_blocks = fit < 1 ? 1 : fit;
    }
    *out = m;
    return RALA_B200_OK;
}

extern "C" void rala_b200_multi_destroy(rala_b200_multi* m) {
    if (!m) return;
    for (FabricRank& fr : m->ranks) {
        if (fr.ctx) {
            cudaSetDevice(fr.device);
            cudaStreamSynchronize(fr.ctx->L.stream);
        }
    }
    drop_graphs(m);
    disconnect(m);
    for (FabricRank& fr : m->ranks) {
        if (!fr.ctx) continue;
        cudaSetDevice(fr.device);
        if (fr.ev[0]) cudaEventDestroy(fr.ev[0]);
        if (fr.ev[1]) cudaEventDestroy(fr.ev[1]);
        DevBuf* bufs[] = {&fr.arena, &fr.meta, &fr.out_cnt, &fr.tmin, &fr.wait, &fr.col_eid, &fr.T, &fr.stage};
        for (DevBuf* b : bufs) b->release();
        if (fr.g) rala_b200_graph_destroy(fr.g);
        rala_b200_destroy(fr.ctx);
    }
    delete m;
}

extern "C" const char* rala_b200_multi_last_error(const rala_b200_multi* m) { return m ? m->error.c_str() : "no session"; }

extern "C" int rala_b200_multi_set_piles(rala_b200_multi* m, const rala_pile_t* piles, const uint8_t* flags, uint32_t n_piles) {
    if (!m) return RALA_B200_ERR_ARG;
    for (FabricRank& fr : m->ranks) {
        MRC(m, fr, rala_b200_graph_set_piles(fr.g, piles, flags, n_piles));
    }
    if (n_piles != m->n_piles) {
        m->n_piles = n_piles;
        m->reserved = false;
    }
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_hills(rala_b200_multi* m, const rala_hill_t* hills, uint32_t n_hills) {
    if (!m || (n_hills && !hills)) return RALA_B200_ERR_ARG;
    for (FabricRank& fr : m->ranks) MRC(m, fr, rala_b200_graph_set_hills(fr.g, hills, n_hills));
    if (n_hills > (m->reserved ? m->ranks[0].A.n_hills : 0u)) m->reserved = false;   // the arena's hills section grows
    m->n_hills = n_hills;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_overlaps(rala_b200_multi* m, int k, const rala_ovl_t* ovl, uint64_t n, uint64_t t0) {
    if (!m || k < 0 || k >= m->n_local) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    if (t0 + n >= (1ull << 31)) return mfail(m, RALA_B200_ERR_LIMIT, "file positions must stay below 2^31 (t0 = %llu, n = %llu)",
                                             (unsigned long long) t0, (unsigned long long) n);
    MRC(m, fr, rala_b200_graph_set_overlaps(fr.g, ovl, n));
    MRC(m, fr, rala_b200_graph_set_shard(fr.g, (uint32_t) t0, fr.rank, m->world));
    m->staged = 0;
    m->staged_edges = false;
    if (n != fr.n_rec) m->reserved = false;
    fr.n_rec = n;
    drop_graphs(m);
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_overlaps_columns(rala_b200_multi* m, int k, const uint32_t* a_id, const uint32_t* b_id,
                                                    const uint32_t* a_begin, const uint32_t* a_end, const uint32_t* b_begin,
                                                    const uint32_t* b_end, uint64_t n, uint64_t t0) {
    if (!m || k < 0 || k >= m->n_local) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    if (t0 + n >= (1ull << 31)) return mfail(m, RALA_B200_ERR_LIMIT, "file positions must stay below 2^31");
    const bool same_shape = n == fr.n_rec && m->reserved;
    MRC(m, fr, rala_b200_graph_set_overlaps_columns(fr.g, a_id, b_id, a_begin, a_end, b_begin, b_end, n));
    MRC(m, fr, rala_b200_graph_set_shard(fr.g, (uint32_t) t0, fr.rank, m->world));
    m->staged = 0;
    m->staged_edges = false;
    if (!same_shape) {
        m->reserved = false;
        drop_graphs(m);
    }
    fr.n_rec = n;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_overlaps_packed(rala_b200_multi* m, int k, const uint32_t* query_id, const uint32_t* group_end,
                                                   uint32_t n_groups, const uint32_t* b_id, const uint32_t* a_span, const uint32_t* b_span,
                                                   uint64_t n, uint64_t t0) {
    if (!m || k < 0 || k >= m->n_local) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    if (t0 + n >= (1ull << 31)) return mfail(m, RALA_B200_ERR_LIMIT, "file positions must stay below 2^31");
    const bool same_shape = n == fr.n_rec && m->reserved;
    MRC(m, fr, rala_b200_graph_set_overlaps_packed(fr.g, query_id, group_end, n_groups, b_id, a_span, b_span, n));
    MRC(m, fr, rala_b200_graph_set_shard(fr.g, (uint32_t) t0, fr.rank, m->world));
    m->staged = 0;
    m->staged_edges = false;
    if (!same_shape) {
        m->reserved = false;
        drop_graphs(m);
    }
    fr.n_rec = n;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_outputs(rala_b200_multi* m, int k, rala_edge_t* edges_out, uint64_t edges_cap, uint8_t* marked_out,
                                           uint64_t marked_cap) {
    if (!m || k < 0 || k >= m->n_local) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    MRC(m, fr, rala_b200_graph_set_outputs(fr.g, edges_out, edges_cap, marked_out, marked_cap));
    drop_graphs(m);   // the output addresses are part of the captured step
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_default_caps(rala_b200_multi* m, uint64_t* caps) {
    if (!m || !caps) return RALA_B200_ERR_ARG;
    uint64_t n_max = 0;
    for (const FabricRank& fr : m->ranks) n_max = fr.n_rec > n_max ? fr.n_rec : n_max;
    // clean long-read data: ~5.5 % of the records are containment events, ~14 % become edges; the defaults leave
    // a wide margin and rala_b200_multi_demand tells when a step did not fit
    const uint64_t W = (uint64_t) m->world;
    caps[RALA_B200_CAP_EVENTS] = align_up(n_max / (W > 1 ? 4 : 1) + 4096, 256);
    caps[RALA_B200_CAP_EDGES] = align_up(n_max / (W > 1 ? 2 : 1) * (W > 1 ? 1 : 2) + 4096, 256);
    caps[RALA_B200_CAP_SLICE] = align_up(n_max + 4096, 256);
    caps[RALA_B200_CAP_ROUNDS] = 4096;         // sweeps after which the resolution gives up: it ends by itself long before
    caps[RALA_B200_CAP_FINAL_ROUNDS] = 4096;
    caps[RALA_B200_CAP_LOCAL_EDGES] = 0;
    for (const FabricRank& fr : m->ranks)
        caps[RALA_B200_CAP_LOCAL_EDGES] = fr.g->edge_cap > caps[RALA_B200_CAP_LOCAL_EDGES] ? fr.g->edge_cap : caps[RALA_B200_CAP_LOCAL_EDGES];
    return RALA_B200_OK;
}

static ArenaLayout make_layout(const rala_b200_multi* m, const uint64_t* caps) {
    ArenaLayout A{};
    const size_t W = (size_t) m->world;
    A.cap_ev = (uint32_t) caps[RALA_B200_CAP_EVENTS];
    A.cap_edge = (uint32_t) caps[RALA_B200_CAP_EDGES];
    A.cap_slice = (uint32_t) caps[RALA_B200_CAP_SLICE];
    A.t_cap = (uint32_t) align_up(caps[RALA_B200_CAP_LOCAL_EDGES] + 16, 256);
    A.n_piles = m->n_piles;
    A.n_nodes_max = 2 * m->n_piles;
    const size_t blocks = ((size_t) m->n_piles + 31) / 32;
    A.ppr = (uint32_t) (((blocks + W - 1) / W) * 32);   // block-cyclic ownership: whole blocks of 32 piles
    if (A.ppr == 0) A.ppr = 32;
    A.npr_max = (uint32_t) (2 * (((size_t) m->n_piles + W - 1) / W) + 2);   // nodes <= 2 * piles, split evenly in pairs
    size_t off = align_up(sizeof(FabricHdr), 4096);
    A.ev_inbox = off;   off += align_up(W * 3 * (size_t) A.cap_ev * 4, 256);
    A.edge_inbox = off; off += align_up(W * 4 * (size_t) A.cap_edge * 4, 256);
    A.S = off;          off += align_up(((size_t) A.n_piles + 64) * 4, 256);
    A.T_in = off;       off += align_up((size_t) A.t_cap, 256);
    A.row_ptr = off;    off += align_up(((size_t) A.n_nodes_max + 8) * 4, 256);
    A.col = off;        off += align_up(W * (size_t) A.cap_slice * 8, 256);
    A.seg_mail = off;   off += align_up((size_t) 2 * kMaxRanks * kSegMail * 4, 256);
    A.n_hills = m->n_hills;
    A.hills = off;      off += align_up((size_t) A.n_hills * 4 + 4, 256);
    A.total = off;
    return A;
}

extern "C" int rala_b200_multi_reserve(rala_b200_multi* m, const uint64_t* caps) {
    if (!m || !caps) return RALA_B200_ERR_ARG;
    if (!m->n_piles) return mfail(m, RALA_B200_ERR_STATE, "reserve: set_piles first");
    const uint64_t W = (uint64_t) m->world;
    if (caps[RALA_B200_CAP_EVENTS] * W >= (1ull << 31) || caps[RALA_B200_CAP_EDGES] * W >= (1ull << 31) ||
        caps[RALA_B200_CAP_SLICE] * W >= (1ull << 31))
        return mfail(m, RALA_B200_ERR_LIMIT, "exchange capacities too large for 32-bit positions");
    if (caps[RALA_B200_CAP_ROUNDS] < 1 || caps[RALA_B200_CAP_FINAL_ROUNDS] < 1 || caps[RALA_B200_CAP_ROUNDS] > 4096 ||
        caps[RALA_B200_CAP_FINAL_ROUNDS] > 4096)
        return mfail(m, RALA_B200_ERR_ARG, "reserve: round counts must be in [1, 4096]");
    for (FabricRank& fr : m->ranks) {   // nothing may still run on an arena that is about to go away
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    }
    drop_graphs(m);
    disconnect(m);
    memcpy(m->caps, caps, sizeof(m->caps));
    const ArenaLayout A = make_layout(m, caps);
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        fr.A = A;
        fr.arena.release();   // a fresh allocation: the IPC handle of the old one must not be reused
        MCU(m, fr.arena.reserve(A.total));
        MCU(m, cudaMemset(fr.arena.p, 0, align_up(sizeof(FabricHdr), 4096)));
        MCU(m, fr.meta.reserve(align_up(sizeof(BuildMeta), 256)));
        MCU(m, fr.out_cnt.reserve(3 * kMaxRanks * 4 + 2 * kResolveCtlBytes));   // + the control block of the resolution kernel, per pass
        MCU(m, fr.tmin.reserve(((size_t) m->n_piles + 64) * 4));
        MCU(m, fr.wait.reserve(((size_t) m->n_piles + 64) * 8));
        MCU(m, fr.col_eid.reserve(W * (size_t) A.cap_slice * 4 + 256));
        // result bytes of the transitive pass, indexed by GLOBAL edge id: an id is < world x the edges one rank can emit,
        // whatever happened to the exchange buffers (nothing clears the array: the row fill clears the bytes it needs)
        MCU(m, fr.T.reserve(align_up(W * (size_t) A.t_cap + 16, 256)));
        MCU(m, fr.stage.reserve(kStageRunsByte + sizeof(EdgeRuns)));
        MRC(m, fr, reserve_events(fr.g, (uint32_t) (W * A.cap_ev)));
        // the owned rows are scanned over npr_max + 1 entries
        const size_t rows = (size_t) A.npr_max + 16;
        if (rows > (size_t) fr.g->n_nodes_max + 8) {
            MCU(m, fr.g->row_ptr.reserve(rows * 4));
            MCU(m, fr.g->cursor.reserve(rows * 4));
        }
    }
    m->reserved = true;
    if (m->n_local == m->world) {   // all ranks here: plain pointers, plus peer access between different devices
        for (FabricRank& fr : m->ranks) {
            MCU(m, cudaSetDevice(fr.device));
            for (FabricRank& other : m->ranks) {
                fr.P.base[other.rank] = other.arena.as<uint8_t>();
                if (other.device != fr.device) {
                    int can = 0;
                    MCU(m, cudaDeviceCanAccessPeer(&can, fr.device, other.device));
                    if (!can) return mfail(m, RALA_B200_ERR_NO_DEVICE, "device %d cannot access device %d's memory", fr.device, other.device);
                    const cudaError_t e = cudaDeviceEnablePeerAccess(other.device, 0);
                    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                        return mfail(m, RALA_B200_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", fr.device, other.device, cudaGetErrorString(e));
                    cudaGetLastError();
                }
            }
        }
        m->connected = true;
    }
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_rounds(rala_b200_multi* m, uint32_t rounds, uint32_t final_rounds) {
    if (!m || rounds < 1 || final_rounds < 1 || rounds > 4096 || final_rounds > 4096) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "set_rounds: reserve first");
    m->caps[RALA_B200_CAP_ROUNDS] = rounds;
    m->caps[RALA_B200_CAP_FINAL_ROUNDS] = final_rounds;
    drop_graphs(m);   // the rounds are part of the captured step
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_export_handle(rala_b200_multi* m, int k, void* handle64) {
    if (!m || k < 0 || k >= m->n_local || !handle64) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "export_handle: reserve first");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI promises 64-byte handles");
    FabricRank& fr = m->ranks[k];
    MCU(m, cudaSetDevice(fr.device));
    cudaIpcMemHandle_t h;
    MCU(m, cudaIpcGetMemHandle(&h, fr.arena.p));
    memcpy(handle64, &h, 64);
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_import_handles(rala_b200_multi* m, const void* handles) {
    if (!m || !handles) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "import_handles: reserve first");
    disconnect(m);
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        for (int q = 0; q < m->world; ++q) {
            const int local = q - m->first_rank;
            if (local >= 0 && local < m->n_local) {
                fr.P.base[q] = m->ranks[local].arena.as<uint8_t>();
                continue;
            }
            cudaIpcMemHandle_t h;
            memcpy(&h, static_cast<const uint8_t*>(handles) + 64 * (size_t) q, 64);
            void* p = nullptr;
            const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                cudaGetLastError();
                return mfail(m, RALA_B200_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d): %s", q, cudaGetErrorString(e));
            }
            fr.ipc_mapped[q] = p;
            fr.P.base[q] = static_cast<uint8_t*>(p);
        }
    }
    m->connected = true;
    return RALA_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// one step, phase by phase (every phase only enqueues on the rank's stream)
// ---------------------------------------------------------------------------------------------
static Publish no_mail(const rala_b200_multi* m) {
    Publish p;
    memset(&p, 0, sizeof(p));
    p.timeout_ns = 1000000ull * m->barrier_timeout_ms;
    return p;
}

// events of the local records / lists -> owners of the victims; then the barrier that publishes how many went where
static int route_and_meet(rala_b200_multi* m, FabricRank& fr, int pass) {
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    // States of FOREIGN piles are only ever written by their owners' pushes, which start after the barrier below: the
    // replica is cleared here, together with everything else the resolution of this pass starts from.
    launch_pass_reset(L, fr.P, fr.A, resolve_bufs(g), fr.tmin.as<uint32_t>(), fr.wait.as<uint32_t>(), fr.ctl(pass));
    launch_route_events(L, fr.P, fr.A, g->events_view(), g->cnt() + C_EV, g->ev_cap, fr.cnt_ev(pass));
    Publish pub = no_mail(m);
    pub.per_dst = fr.cnt_ev(pass);
    pub.scalar[M_EMITTED] = g->cnt() + C_EV;   // still the number of events this rank emitted (the gather overwrites it)
    pub.bookkeeping = 2;                       // a pass in which no rank has an event is skipped by all of them
    pub.pass = pass;
    launch_fabric_barrier(L, fr.P, pub);
    MCU(m, cudaGetLastError());
    return RALA_B200_OK;
}

// graph.cpp:469-480 / 831-866 on the piles this rank owns
static int resolve_owned_piles(rala_b200_multi* m, FabricRank& fr, int pass, bool hills = false) {
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    const ResolveBufs rb = resolve_bufs(g);
    const uint32_t rounds = (uint32_t) m->caps[pass ? RALA_B200_CAP_FINAL_ROUNDS : RALA_B200_CAP_ROUNDS];
    MCU(m, stage_event(g, g->ev_start[ST_K1B_KERNEL]));
    launch_gather_events(L, fr.P, fr.A, g->events_view(), g->ev_cap, g->cnt() + C_EV, rb.vcursor, fr.tmin.as<uint32_t>());
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, (uint64_t) g->n_piles + 1, &status, &ticket);
    launch_scan_u32(L, rb.vcursor, rb.vstart, g->n_piles + 1, status, ticket, skip_flag(fr.P));
    launch_fabric_prepare(L, fr.P, fr.A, g->events_view(), g->cnt() + C_EV, g->ev_cap, rb, fr.tmin.as<uint32_t>());
    launch_push_slice(L, fr.P, fr.A);
    // no barrier: a state that has not arrived yet reads as "open, cannot die before time 0", which only makes its
    // dependants wait for the next sweep
    launch_fabric_resolve(L, fr.P, fr.A, rb, fr.wait.as<uint32_t>(), fr.ctl(pass), pass, rounds, 1000000ull * m->barrier_timeout_ms,
                          fr.resolve_blocks);
    MCU(m, end_stage(g, ST_K1B_KERNEL));
    // staged construct: the hill counters of the local records (pile.cpp:457-469) read the death times BEFORE the deaths are
    // applied, then go into the replicated total (every rank's hills section, published by the survivors barrier)
    if (hills) {
        const uint32_t* h = g->hills.as<uint32_t>();
        const uint32_t n = g->n_hills;
        launch_decode_states(L, fr.P, fr.A);
        launch_hill_coverage(L, g->recs.view, g->t0, g->piles.as<uint2>(), g->hill_rec.as<uint32_t>(), g->cap, h, h + n, h + 2 * (size_t) n,
                             n, g->hills.as<uint32_t>() + 3 * (size_t) n, fr.sec<uint32_t>(fr.A.S), g->cnt());
        launch_push_hills(L, fr.P, fr.A, h + 3 * (size_t) n, n);
    }
    // every replica now holds every pile's final state: piles with a finite death time die (graph.cpp:471,477,838,842)
    // (a skipped pass killed nobody: the table and the liveness bitmap stay as they are)
    launch_apply_deaths(L, g->piles.as<uint2>(), fr.sec<uint32_t>(fr.A.S), g->n_piles, g->alive_bits.as<uint32_t>(), !hills, skip_flag(fr.P),
                        nullptr, pass == 0 ? final_pass_reset(g) : FinalPassReset{});
    MCU(m, cudaGetLastError());
    return RALA_B200_OK;
}

static int phase_a_events(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    MRC(m, fr, phase_events(fr.g));   // graph.cpp:443-480 on the local records (also resets the counters and the pile table)
    Launch& L = fr.ctx->L;
    MCU(m, cudaMemsetAsync(&fr.hdr()->error, 0, 4 * (1 + 2 + 4), L.stream));   // error, rounds_needed, demand
    MCU(m, cudaMemsetAsync(fr.out_cnt.p, 0, 3 * kMaxRanks * 4, L.stream));
    return route_and_meet(m, fr, 0);
}

static int phase_b_resolve(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    return resolve_owned_piles(m, fr, 0);
}

static int phase_c_survivors(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    MRC(m, fr, phase_survivors(g));   // graph.cpp:493-515 on the local records
    Publish pub = no_mail(m);
    pub.scalar[M_NOVL] = g->cnt() + g->slot_ovl;
    pub.scalar[M_NINL] = g->cnt() + g->slot_inl;
    launch_fabric_barrier(fr.ctx->L, fr.P, pub);
    return RALA_B200_OK;
}

static int phase_d_final_events(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    launch_time_bases_mail(fr.ctx->L, fr.P, g->cnt() + C_TBASE_OVL);
    MRC(m, fr, phase_final_events(g, g->cnt() + C_TBASE_OVL, C_TBASE_INL));   // graph.cpp:831-848 on the local lists
    return route_and_meet(m, fr, 1);
}

static int phase_e_final_resolve(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    int rc = resolve_owned_piles(m, fr, 1);
    if (rc) return rc;
    MRC(m, fr, end_final_pass(fr.g));
    return RALA_B200_OK;
}

// graph.cpp:552-632: node ids (replicated), the edges of the local dovetails, routed to the owners of their sources
static int phase_f_edges(rala_b200_multi* m, FabricRank& fr) {
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    MRC(m, fr, emit_edges(g, false));   // no local CSR: the owners build theirs from what they receive
    fork_edge_download(g);
    launch_node_bounds(L, fr.P, fr.A, g->cnt() + C_NODES, fr.meta_dev());
    const GraphArrays ga = g->graph_view();
    // result bytes of the local edges: cleared now, written by the evaluating ranks after two more barriers
    launch_clear_bytes16(L, fr.sec<uint8_t>(fr.A.T_in), g->cnt() + C_EDGES, fr.A.t_cap);
    launch_route_edges(L, fr.P, fr.A, ga.src, ga.dst, ga.len, g->cnt() + C_EDGES, g->edge_cap, fr.meta_dev(), fr.cnt_edges());
    Publish pub = no_mail(m);
    pub.scalar[M_NEDGES] = g->cnt() + C_EDGES;
    pub.bcast = fr.cnt_edges();
    launch_fabric_barrier(L, fr.P, pub);
    MCU(m, cudaGetLastError());
    return RALA_B200_OK;
}

// the rows this rank owns, then its slice to every replica
static int phase_g_csr(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    launch_edge_meta(L, fr.P, fr.A, fr.meta_dev(), g->cnt());
    const uint32_t rows = fr.A.npr_max + 1u;
    MCU(m, cudaMemsetAsync(g->cursor.p, 0, ((size_t) rows + 7) * 4, L.stream));
    launch_inbox_degree(L, fr.P, fr.A, fr.meta_dev(), g->cursor.as<uint32_t>());
    unsigned long long* status;
    uint32_t* ticket;
    scan_state(g, rows, &status, &ticket);
    launch_scan_u32(L, g->cursor.as<uint32_t>(), g->row_ptr.as<uint32_t>(), rows, status, ticket);
    launch_inbox_fill(L, fr.P, fr.A, fr.meta_dev(), g->cursor.as<uint32_t>(), fr.col_eid.as<uint32_t>(), fr.T.as<uint8_t>(),
                      m->staged_edges ? fr.runs_dev() : nullptr);
    launch_push_csr(L, fr.P, fr.A, fr.meta_dev(), g->row_ptr.as<uint32_t>());
    launch_fabric_barrier(L, fr.P, no_mail(m));
    MRC(m, fr, end_build(g));
    return RALA_B200_OK;
}

// graph.cpp:1281-1318 for the candidate edges whose source node this rank owns
static int phase_h_transitive(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    MCU(m, begin_stage(g, ST_TRANSITIVE));
    GraphArrays ga = g->graph_view();
    ga.row_ptr = fr.sec<uint32_t>(fr.A.row_ptr);
    ga.col = fr.sec<uint2>(fr.A.col);
    ga.col_eid = fr.col_eid.as<uint32_t>();
    ga.T = fr.T.as<uint8_t>();
    MRC(m, fr, transitive_stage(g, ga, fr.meta_dev()->node_begin + fr.rank));
    launch_route_marks(L, fr.P, fr.A, fr.meta_dev(), fr.T.as<uint8_t>(), fr.col_eid.as<uint32_t>(), m->staged_edges ? fr.runs_dev() : nullptr);
    launch_fabric_barrier(L, fr.P, no_mail(m));
    return RALA_B200_OK;
}

// marked(e) = T(e) | T(e ^ 1) for the edges this rank emitted (pairs are emitted together)
static int phase_i_marks(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    GraphArrays ga = g->graph_view();
    ga.T = fr.sec<uint8_t>(fr.A.T_in);
    MRC(m, fr, marks_stage(g, ga, g->out_marked, g->out_marked_cap));
    launch_demand(L, fr.P, fr.cnt_ev(0), fr.cnt_ev(1), fr.cnt_edges(), fr.meta_dev());
    MCU(m, cudaGetLastError());
    return RALA_B200_OK;
}

typedef int (*PhaseFn)(rala_b200_multi*, FabricRank&);
static const PhaseFn kPhases[] = {phase_a_events, phase_b_resolve,  phase_c_survivors,  phase_d_final_events, phase_e_final_resolve,
                                  phase_f_edges,  phase_g_csr,      phase_h_transitive, phase_i_marks};

// Phases outermost, ranks innermost: with several ranks in one process no rank's stream ever holds more than one
// phase that its peers have not been given yet (a barrier kernel waits on the GPU for the peers' kernels).
static int enqueue_step(rala_b200_multi* m) {
    for (PhaseFn phase : kPhases)
        for (FabricRank& fr : m->ranks) {
            int rc = phase(m, fr);
            if (rc) return rc;
        }
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_use_cuda_graph(rala_b200_multi* m, int enabled) {
    if (!m) return RALA_B200_ERR_ARG;
    m->use_graph = enabled != 0;
    if (!m->use_graph) drop_graphs(m);
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_run(rala_b200_multi* m) {
    if (!m) return RALA_B200_ERR_ARG;
    if (!m->reserved || !m->connected) return mfail(m, RALA_B200_ERR_STATE, "run: reserve (and connect) the exchange arenas first");
    for (FabricRank& fr : m->ranks)
        if (fr.g->state < SS_INPUTS) return mfail(m, RALA_B200_ERR_STATE, "run: rank %d has no inputs", fr.rank);
    m->staged = 0;
    m->staged_edges = false;
    const int variant = m->ranks[0].g->piles_fresh ? 1 : 0;
    if (!m->use_graph || m->runs_seen[variant] == 0) {
        const int rc = enqueue_step(m);
        if (!rc && m->use_graph) m->runs_seen[variant] = 1;
        return rc;
    }
    if (m->runs_seen[variant] == 1) {   // same shape as a step before: capture every rank's stream while enqueueing
        std::vector<uint64_t> before;
        for (FabricRank& fr : m->ranks) {
            MCU(m, cudaSetDevice(fr.device));
            before.push_back(fr.ctx->L.count);
            MCU(m, cudaStreamBeginCapture(fr.ctx->L.stream, cudaStreamCaptureModeRelaxed));
            fr.g->capturing = true;
        }
        const int rc = enqueue_step(m);
        bool ok = rc == RALA_B200_OK;
        for (size_t k = 0; k < m->ranks.size(); ++k) {
            FabricRank& fr = m->ranks[k];
            cudaSetDevice(fr.device);
            fr.g->capturing = false;
            cudaGraph_t graph = nullptr;
            const cudaError_t e = cudaStreamEndCapture(fr.ctx->L.stream, &graph);
            if (e != cudaSuccess || !graph) {
                if (ok) mfail(m, RALA_B200_ERR_CUDA, "run: stream capture failed on rank %d: %s", fr.rank, cudaGetErrorString(e));
                ok = false;
            } else if (ok) {
                const cudaError_t ei = cudaGraphInstantiate(&fr.exec[variant], graph, 0);
                if (ei != cudaSuccess) {
                    mfail(m, RALA_B200_ERR_CUDA, "run: cudaGraphInstantiate failed on rank %d: %s", fr.rank, cudaGetErrorString(ei));
                    fr.exec[variant] = nullptr;
                    ok = false;
                }
            }
            if (graph) cudaGraphDestroy(graph);
            fr.graph_launches[variant] = fr.ctx->L.count - before[k];
            fr.ctx->L.count = before[k];
        }
        cudaGetLastError();
        if (!ok) {
            drop_graphs(m);
            return rc ? rc : RALA_B200_ERR_CUDA;
        }
        m->runs_seen[variant] = 2;
        // the capture only recorded the step: the host-side state it left behind is the state after a step, and the
        // step itself still has to run
    }
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaGraphLaunch(fr.exec[variant], fr.ctx->L.stream));
        fr.ctx->L.count += fr.graph_launches[variant];
        fr.g->piles_fresh = false;
        for (int i = 0; i < RALA_B200_N_STAGES; ++i) fr.g->ev_valid[i] = false;
    }
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_set_barrier_timeout_ms(rala_b200_multi* m, uint32_t ms) {
    if (!m || ms == 0) return RALA_B200_ERR_ARG;
    m->barrier_timeout_ms = ms;
    drop_graphs(m);   // the timeout is a kernel argument of the captured barriers
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_synchronize(rala_b200_multi* m) {
    if (!m) return RALA_B200_ERR_ARG;
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    }
    return RALA_B200_OK;
}

static int read_hdr(rala_b200_multi* m, FabricRank& fr, FabricHdr* h) {
    MCU(m, cudaSetDevice(fr.device));
    MCU(m, cudaMemcpyAsync(h, fr.arena.p, offsetof(FabricHdr, mail), cudaMemcpyDeviceToHost, fr.ctx->L.stream));
    MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_demand(rala_b200_multi* m, uint64_t* need, int* fits) {
    if (!m || !need || !fits) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "demand: nothing has run");
    memset(need, 0, sizeof(uint64_t) * RALA_B200_N_CAPS);
    *fits = 1;
    for (FabricRank& fr : m->ranks) {
        FabricHdr h;
        int rc = read_hdr(m, fr, &h);
        if (rc) return rc;
        uint32_t c[C_COUNT];
        MCU(m, cudaMemcpy(c, fr.g->counters.p, sizeof(c), cudaMemcpyDeviceToHost));
        const uint64_t v[RALA_B200_N_CAPS] = {h.demand[0], h.demand[1], h.demand[2], h.rounds_needed[0], h.rounds_needed[1], c[C_EDGES]};
        for (int i = 0; i < RALA_B200_N_CAPS; ++i) need[i] = v[i] > need[i] ? v[i] : need[i];
        if (h.error || c[C_OVERFLOW] || h.rounds_needed[0] == 0 || h.rounds_needed[1] == 0) *fits = 0;
        if (h.error & FE_TIMEOUT)
            return mfail(m, RALA_B200_ERR_CUDA, "rank %d: rank %u did not reach barrier %u within %u ms (epoch now %u; reserve again to reconnect)",
                         fr.rank, h.dead_peer, h.dead_epoch, m->barrier_timeout_ms, h.epoch);
    }
    for (int i = 0; i < 3; ++i)
        if (need[i] > m->caps[i]) *fits = 0;
    if (need[RALA_B200_CAP_LOCAL_EDGES] > m->caps[RALA_B200_CAP_LOCAL_EDGES]) *fits = 0;
    // a round count of 0 = the resolution had not converged when the step's rounds were used up: ask for more
    if (need[RALA_B200_CAP_ROUNDS] == 0) need[RALA_B200_CAP_ROUNDS] = 2 * m->caps[RALA_B200_CAP_ROUNDS];
    if (need[RALA_B200_CAP_FINAL_ROUNDS] == 0) need[RALA_B200_CAP_FINAL_ROUNDS] = 2 * m->caps[RALA_B200_CAP_FINAL_ROUNDS];
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_plan(rala_b200_multi* m) {
    if (!m) return RALA_B200_ERR_ARG;
    if (m->n_local != m->world) return mfail(m, RALA_B200_ERR_STATE, "plan: with one process per GPU the caller agrees on the capacities (see rala_b200.h)");
    uint64_t caps[RALA_B200_N_CAPS];
    int rc = rala_b200_multi_default_caps(m, caps);
    if (rc) return rc;
    for (int attempt = 0; attempt < 6; ++attempt) {
        rc = rala_b200_multi_reserve(m, caps);
        m->staged = 0;
        m->staged_edges = false;
        if (!rc) rc = enqueue_step(m);
        if (!rc) rc = rala_b200_multi_synchronize(m);
        uint64_t need[RALA_B200_N_CAPS];
        int fits = 0;
        if (!rc) rc = rala_b200_multi_demand(m, need, &fits);
        if (rc) return rc;
        if (fits) return RALA_B200_OK;
        for (int i = 0; i < 3; ++i)
            if (need[i] > caps[i]) caps[i] = align_up(need[i] + need[i] / 4 + 1024, 256);
        if (need[RALA_B200_CAP_LOCAL_EDGES] > caps[RALA_B200_CAP_LOCAL_EDGES]) caps[RALA_B200_CAP_LOCAL_EDGES] = need[RALA_B200_CAP_LOCAL_EDGES];
        if (need[RALA_B200_CAP_ROUNDS] > caps[RALA_B200_CAP_ROUNDS]) caps[RALA_B200_CAP_ROUNDS] = need[RALA_B200_CAP_ROUNDS];
        if (need[RALA_B200_CAP_FINAL_ROUNDS] > caps[RALA_B200_CAP_FINAL_ROUNDS]) caps[RALA_B200_CAP_FINAL_ROUNDS] = need[RALA_B200_CAP_FINAL_ROUNDS];
    }
    return mfail(m, RALA_B200_ERR_LIMIT, "plan: the exchange buffers still did not fit after 6 attempts");
}

extern "C" int rala_b200_multi_counts(rala_b200_multi* m, rala_b200_multi_counts_t* out) {
    if (!m || !out) return RALA_B200_ERR_ARG;
    memset(out, 0, sizeof(*out));
    out->world = m->world;
    out->n_local = m->n_local;
    out->n_piles = m->n_piles;
    for (FabricRank& fr : m->ranks) {
        FabricHdr h;
        int rc = read_hdr(m, fr, &h);
        if (rc) return rc;
        uint32_t c[C_COUNT];
        BuildMeta bm;
        MCU(m, cudaMemcpy(c, fr.g->counters.p, sizeof(c), cudaMemcpyDeviceToHost));
        MCU(m, cudaMemcpy(&bm, fr.meta.p, sizeof(bm), cudaMemcpyDeviceToHost));
        out->fabric_error |= h.error | (c[C_OVERFLOW] ? (uint32_t) FE_INBOX : 0u);
        out->n_records += fr.n_rec;
        out->n_alive_piles = c[C_ALIVE];
        out->n_nodes = c[C_NODES];
        out->n_edges = bm.eid_base[m->world];
        out->n_local_edges += c[C_EDGES];
        out->n_rounds = h.rounds_needed[0];
        out->n_final_rounds = h.rounds_needed[1];
        uint32_t sent[3 * kMaxRanks];
        MCU(m, cudaMemcpy(sent, fr.out_cnt.p, sizeof(sent), cudaMemcpyDeviceToHost));
        for (int q = 0; q < m->world; ++q) {
            out->n_candidates += sent[q];
            out->n_final_candidates += sent[kMaxRanks + q];
        }
        out->n_two_hop += (uint64_t) c[C_HOP_LO] | ((uint64_t) c[C_HOP_HI] << 32);
        out->n_transitive_pairs += c[C_PAIRS];
        out->n_heavy_items += c[C_HEAVY];
    }
    if (out->fabric_error)
        return mfail(m, RALA_B200_ERR_LIMIT, "the last step did not fit its exchange buffers or rounds (fabric error bits %u): plan again",
                     out->fabric_error);
    return RALA_B200_OK;
}

// global id runs of local rank k's edges, in local order, adjacent runs merged: out (nullable) holds 2 x RALA_B200_MAX_SEGMENTS
static int edge_runs_of(rala_b200_multi* m, int k, uint64_t* out, uint32_t* n_out) {
    FabricRank& fr = m->ranks[k];
    if (fr.g->state < SS_BUILT) return mfail(m, RALA_B200_ERR_STATE, "edge_runs: run (or finish) first");
    std::vector<uint64_t> r;   // first, count, first, count, ...
    auto add = [&](uint64_t first, uint64_t count) {
        if (!count) return;
        if (!r.empty() && r[r.size() - 2] + r.back() == first) r.back() += count;
        else r.insert(r.end(), {first, count});
    };
    if (m->staged_edges) {
        for (uint32_t s = 0; s < m->runs.n_seg; ++s) {
            const size_t i = (size_t) s * m->world + fr.rank;
            add(m->runs.gb[i], 2ull * m->dov[i]);
        }
    } else {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
        BuildMeta bm;
        MCU(m, cudaMemcpy(&bm, fr.meta.p, sizeof(bm), cudaMemcpyDeviceToHost));
        add(bm.eid_base[fr.rank], bm.eid_base[fr.rank + 1] - bm.eid_base[fr.rank]);
    }
    *n_out = (uint32_t) (r.size() / 2);
    if (out && !r.empty()) memcpy(out, r.data(), r.size() * sizeof(uint64_t));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_edge_runs(rala_b200_multi* m, int k, uint64_t* first_and_count_out, uint32_t* n_runs_out) {
    if (!m || k < 0 || k >= m->n_local || !n_runs_out) return RALA_B200_ERR_ARG;
    return edge_runs_of(m, k, first_and_count_out, n_runs_out);
}

extern "C" int rala_b200_multi_edge_range(rala_b200_multi* m, int k, uint64_t* first_edge, uint64_t* n) {
    if (!m || k < 0 || k >= m->n_local || !first_edge || !n) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    if (fr.g->state < SS_BUILT) return mfail(m, RALA_B200_ERR_STATE, "edge_range: run first");
    if (m->staged_edges) {
        uint64_t r[2 * kMaxSegs];
        uint32_t n_runs = 0;
        int rc = edge_runs_of(m, k, r, &n_runs);
        if (rc) return rc;
        if (n_runs > 1)
            return mfail(m, RALA_B200_ERR_STATE, "edge_range: rank %d's edges are %u runs of global ids (a staged construct promoted "
                         "overlaps): use rala_b200_multi_edge_runs", fr.rank, n_runs);
        *first_edge = n_runs ? r[0] : 0;
        *n = n_runs ? r[1] : 0;
        return RALA_B200_OK;
    }
    MCU(m, cudaSetDevice(fr.device));
    MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    BuildMeta bm;
    MCU(m, cudaMemcpy(&bm, fr.meta.p, sizeof(bm), cudaMemcpyDeviceToHost));
    *first_edge = bm.eid_base[fr.rank];
    *n = bm.eid_base[fr.rank + 1] - bm.eid_base[fr.rank];
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_edges(rala_b200_multi* m, int k, rala_edge_t* out) {
    if (!m || k < 0 || k >= m->n_local || !out) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    MRC(m, fr, rala_b200_graph_get_edges(fr.g, out));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_marked(rala_b200_multi* m, int k, uint8_t* out) {
    if (!m || k < 0 || k >= m->n_local || !out) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    MRC(m, fr, rala_b200_graph_get_marked(fr.g, out));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_seq_to_node(rala_b200_multi* m, uint32_t* out) {
    if (!m || !out) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[0];
    MRC(m, fr, rala_b200_graph_get_seq_to_node(fr.g, out));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_piles(rala_b200_multi* m, rala_pile_t* out) {
    if (!m || !out) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[0];
    MRC(m, fr, rala_b200_graph_get_piles(fr.g, out));
    return RALA_B200_OK;
}

// diagnostics: the last kBarrierLog barriers of local rank k as (start, all peers arrived) device timestamps in ns,
// oldest first; *n_out = how many are valid
extern "C" int rala_b200_multi_barrier_log(rala_b200_multi* m, int k, uint64_t* out, uint32_t* n_out) {
    if (!m || k < 0 || k >= m->n_local || !out || !n_out) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "barrier_log: nothing has run");
    FabricRank& fr = m->ranks[k];
    MCU(m, cudaSetDevice(fr.device));
    MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    std::vector<unsigned char> raw(sizeof(FabricHdr));
    MCU(m, cudaMemcpy(raw.data(), fr.arena.p, sizeof(FabricHdr), cudaMemcpyDeviceToHost));
    const FabricHdr* h = reinterpret_cast<const FabricHdr*>(raw.data());
    const uint32_t n = h->epoch < (uint32_t) kBarrierLog ? h->epoch : (uint32_t) kBarrierLog;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t e = h->epoch - n + 1u + i;
        out[2 * i] = h->tlog[e % kBarrierLog][0];
        out[2 * i + 1] = h->tlog[e % kBarrierLog][1];
    }
    *n_out = n;
    return RALA_B200_OK;
}

// diagnostics: per sweep of the last resolution of `pass` on local rank k: (open victims at its start, ns since the kernel started)
extern "C" int rala_b200_multi_sweep_log(rala_b200_multi* m, int k, int pass, uint64_t* out /* 2 x 48 */, uint32_t* n_out) {
    if (!m || k < 0 || k >= m->n_local || pass < 0 || pass > 1 || !out || !n_out) return RALA_B200_ERR_ARG;
    if (!m->reserved) return mfail(m, RALA_B200_ERR_STATE, "sweep_log: nothing has run");
    FabricRank& fr = m->ranks[k];
    MCU(m, cudaSetDevice(fr.device));
    MCU(m, cudaStreamSynchronize(fr.ctx->L.stream));
    std::vector<uint32_t> raw(kResolveCtlBytes / 4);
    MCU(m, cudaMemcpy(raw.data(), fr.ctl(pass), kResolveCtlBytes, cudaMemcpyDeviceToHost));
    const uint32_t n = raw[3] < (uint32_t) kSweepLog ? raw[3] : (uint32_t) kSweepLog;
    memcpy(out, raw.data() + 8, (size_t) n * 16);
    *n_out = n;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_event_record(rala_b200_multi* m, int which) {
    if (!m || which < 0 || which > 1) return RALA_B200_ERR_ARG;
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaEventRecord(fr.ev[which], fr.ctx->L.stream));
    }
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_event_elapsed_ms(rala_b200_multi* m, float* ms) {
    if (!m || !ms) return RALA_B200_ERR_ARG;
    *ms = 0.f;
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaEventSynchronize(fr.ev[1]));
        float t = 0.f;
        MCU(m, cudaEventElapsedTime(&t, fr.ev[0], fr.ev[1]));
        *ms = t > *ms ? t : *ms;
    }
    return RALA_B200_OK;
}

extern "C" uint64_t rala_b200_multi_launch_count(const rala_b200_multi* m) {
    uint64_t n = 0;
    if (m)
        for (const FabricRank& fr : m->ranks) n += fr.ctx->L.count;
    return n;
}

extern "C" int rala_b200_multi_stage_ms(rala_b200_multi* m, int k, float* ms_out) {
    if (!m || k < 0 || k >= m->n_local || !ms_out) return RALA_B200_ERR_ARG;
    FabricRank& fr = m->ranks[k];
    MRC(m, fr, rala_b200_graph_stage_ms(fr.g, ms_out));
    return RALA_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// Staged construct: Graph::construct with a pile table the host changes between the passes (graph.cpp:443-829), then
// 831-877, 552-632 and 1281-1318.  The reference appends what a pit round promotes to the END of the global `overlaps`
// (:818), so with shards in rank order the global list is segment-major: segment 0 = every rank's entries of the first
// pass in rank order, segment k = what the k-th promoting round promoted, in rank order.  Each rank's local list is its
// part of every segment, in segment order.  Every list pass ends with a barrier that publishes the new per-(segment,
// rank) counts (seg_mail); the host reads them from its own arena, so every process holds the same table and takes the
// same decisions (is_changed, a new segment) without a host collective.
// ---------------------------------------------------------------------------------------------
static List sub_list(const List& l, uint32_t off) {
    List s = l;
    s.a += off; s.b += off; s.ab += off; s.ae += off; s.bb += off; s.be += off; s.tag += off;
    return s;
}

static uint32_t& seg_at(rala_b200_multi* m, std::vector<uint32_t>& v, uint32_t s, int q) { return v[(size_t) s * m->world + q]; }

// local start of every segment of rank `fr`'s `overlaps` (and its end) -> stage words SW_LO ..
static int upload_segment_bounds(rala_b200_multi* m, FabricRank& fr) {
    std::vector<uint32_t>& h = fr.stage_host;
    h.assign(SW_WORDS, 0u);
    uint32_t local = 0;
    for (uint32_t s = 0; s < m->n_seg; ++s) {
        h[SW_LO + s] = local;
        local += seg_at(m, m->seg, s, fr.rank);
    }
    h[SW_LO + m->n_seg] = local;
    MCU(m, cudaMemcpyAsync(fr.stage.p, h.data(), SW_WORDS * 4, cudaMemcpyHostToDevice, fr.ctx->L.stream));
    return RALA_B200_OK;
}

// after a staged barrier: wait for every local rank, then the counts every rank published in it (words per rank)
static int read_seg_mail(rala_b200_multi* m, std::vector<uint32_t>& mail) {
    int rc = rala_b200_multi_synchronize(m);
    if (rc) return rc;
    for (FabricRank& fr : m->ranks) {
        FabricHdr h;
        rc = read_hdr(m, fr, &h);
        if (rc) return rc;
        if (h.error & FE_TIMEOUT)
            return mfail(m, RALA_B200_ERR_CUDA, "rank %d: rank %u did not reach barrier %u within %u ms", fr.rank, h.dead_peer, h.dead_epoch,
                         m->barrier_timeout_ms);
    }
    FabricRank& fr = m->ranks[0];
    uint32_t epoch = 0;
    MCU(m, cudaMemcpy(&epoch, &fr.hdr()->epoch, 4, cudaMemcpyDeviceToHost));
    mail.resize((size_t) m->world * kSegMail);
    const uint32_t* src = fr.sec<uint32_t>(fr.A.seg_mail) + (size_t) (epoch & 1u) * kMaxRanks * kSegMail;
    MCU(m, cudaMemcpy(mail.data(), src, mail.size() * 4, cudaMemcpyDeviceToHost));
    return RALA_B200_OK;
}

static int staged_ready(rala_b200_multi* m, const char* what) {
    if (!m->reserved || !m->connected) return mfail(m, RALA_B200_ERR_STATE, "%s: reserve (and connect) the exchange arenas first", what);
    for (FabricRank& fr : m->ranks)
        if (fr.g->state < SS_INPUTS) return mfail(m, RALA_B200_ERR_STATE, "%s: rank %d has no inputs", what, fr.rank);
    return RALA_B200_OK;
}

// graph.cpp:443-518 (phases a - c of a step) with the hill counters of the first pass summed over the ranks
extern "C" int rala_b200_multi_classify(rala_b200_multi* m) {
    if (!m) return RALA_B200_ERR_ARG;
    int rc = staged_ready(m, "classify");
    if (rc) return rc;
    drop_graphs(m);
    m->staged = 0;
    m->staged_edges = false;
    const bool hills = m->n_hills > 0;
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        if (hills) MCU(m, cudaMemsetAsync(fr.sec<uint32_t>(fr.A.hills), 0, (size_t) m->n_hills * 4, fr.ctx->L.stream));   // before the events barrier
        rc = phase_a_events(m, fr);
        if (rc) return rc;
    }
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        rc = resolve_owned_piles(m, fr, 0, hills);
        if (rc) return rc;
    }
    for (FabricRank& fr : m->ranks) {
        rc = phase_c_survivors(m, fr);
        if (rc) return rc;
        if (hills)
            MCU(m, cudaMemcpyAsync(fr.g->hills.as<uint32_t>() + 3 * (size_t) m->n_hills, fr.sec<uint32_t>(fr.A.hills), (size_t) m->n_hills * 4,
                                   cudaMemcpyDeviceToDevice, fr.ctx->L.stream));
    }
    rc = rala_b200_multi_synchronize(m);
    if (rc) return rc;
    FabricRank& fr = m->ranks[0];
    std::vector<unsigned char> raw(sizeof(FabricHdr));
    MCU(m, cudaMemcpy(raw.data(), fr.arena.p, sizeof(FabricHdr), cudaMemcpyDeviceToHost));
    const FabricHdr* h = reinterpret_cast<const FabricHdr*>(raw.data());
    if (h->error & FE_TIMEOUT) return mfail(m, RALA_B200_ERR_CUDA, "classify: a barrier timed out (rank %u, barrier %u)", h->dead_peer, h->dead_epoch);
    const uint32_t par = h->epoch & 1u;
    m->n_seg = 1;
    m->seg.assign((size_t) kMaxSegs * m->world, 0u);
    m->dov.assign((size_t) kMaxSegs * m->world, 0u);
    m->inl.assign((size_t) m->world, 0u);
    for (int q = 0; q < m->world; ++q) {
        seg_at(m, m->seg, 0, q) = h->mail[par][q][M_NOVL];
        m->inl[q] = h->mail[par][q][M_NINL];
    }
    m->staged = 2;
    return RALA_B200_OK;
}

// one list pass on every local rank (graph.cpp:722-736 / 801-824): count what every segment keeps, run the pass, publish
static int staged_list_pass(rala_b200_multi* m, bool promote, int* is_changed) {
    const char* what = promote ? "retrim_promote" : "retrim";
    if (is_changed) *is_changed = 0;
    if (m->staged != 2) return mfail(m, RALA_B200_ERR_STATE, "%s: classify (rala_b200_multi_classify) first", what);
    // the single session's rule for a pass against an unchanged table (identity: skipped); the flags are the same on every
    // rank and in every process, which all made the same calls
    const rala_b200_graph* g0 = m->ranks[0].g;
    if (!g0->piles_dirty && g0->skip_clean_retrim && (!promote || !g0->promote_pending)) return RALA_B200_OK;
    const uint32_t S = m->n_seg;
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        rala_b200_graph* g = fr.g;
        Launch& L = fr.ctx->L;
        int rc = upload_segment_bounds(m, fr);
        if (rc) return rc;
        MCU(m, cudaMemsetAsync(fr.stage_w(SW_BOX), 0, kSegMail * 4, L.stream));
        launch_seg_count(L, g->ovl[g->ovl_cur].view, fr.stage_w(SW_LO), S, g->piles.as<uint2>(), kSegRetrim, fr.stage_w(SW_BOX));
        MRC(m, fr, promote ? rala_b200_graph_retrim_promote(g, nullptr) : rala_b200_graph_retrim(g));
        MCU(m, cudaMemcpyAsync(fr.stage_w(SW_BOX + S), g->cnt() + g->slot_ovl, 4, cudaMemcpyDeviceToDevice, L.stream));
        MCU(m, cudaMemcpyAsync(fr.stage_w(SW_BOX + S + 1), g->cnt() + g->slot_inl, 4, cudaMemcpyDeviceToDevice, L.stream));
        launch_seg_push(L, fr.P, fr.A, fr.stage_w(SW_BOX), S + 2);
        launch_fabric_barrier(L, fr.P, no_mail(m));
        MCU(m, cudaGetLastError());
    }
    std::vector<uint32_t> mail;
    int rc = read_seg_mail(m, mail);
    if (rc) return rc;
    bool changed = false, promoted = false;
    for (int q = 0; q < m->world; ++q) {
        const uint32_t* box = mail.data() + (size_t) q * kSegMail;
        uint64_t kept = 0, before = 0;
        for (uint32_t s = 0; s < S; ++s) {
            kept += box[s];
            before += seg_at(m, m->seg, s, q);
        }
        changed = changed || kept != before;
        promoted = promoted || box[S] != kept;
    }
    if (promoted && S == (uint32_t) kMaxSegs) {
        m->staged = 0;
        return mfail(m, RALA_B200_ERR_LIMIT, "%s: a pit round promoted overlaps after %d rounds that did: at most %d segments of `overlaps` "
                     "(RALA_B200_MAX_SEGMENTS); the session's lists are void", what, kMaxSegs - 1, kMaxSegs);
    }
    for (int q = 0; q < m->world; ++q) {
        const uint32_t* box = mail.data() + (size_t) q * kSegMail;
        uint32_t kept = 0;
        for (uint32_t s = 0; s < S; ++s) {
            seg_at(m, m->seg, s, q) = box[s];
            kept += box[s];
        }
        if (promoted) seg_at(m, m->seg, S, q) = box[S] - kept;   // a new segment only in a round where some rank promoted
        m->inl[q] = box[S + 1];
    }
    if (promoted) m->n_seg = S + 1;
    if (is_changed) *is_changed = changed ? 1 : 0;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_retrim(rala_b200_multi* m) { return m ? staged_list_pass(m, false, nullptr) : RALA_B200_ERR_ARG; }

extern "C" int rala_b200_multi_retrim_promote(rala_b200_multi* m, int* is_changed) {
    return m ? staged_list_pass(m, true, is_changed) : RALA_B200_ERR_ARG;
}

// graph.cpp:831-848 on the staged lists: the time of an entry is its global position in overlaps ++ internals, one base per
// segment of `overlaps` (classify_final on the segment's part of the local list) and one for `internals`
static int phase_d_staged(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    std::vector<uint32_t>& h = fr.stage_host;
    h.assign(SW_WORDS, 0u);
    uint64_t before = 0;
    uint32_t local = 0;
    for (uint32_t s = 0; s < m->n_seg; ++s) {
        h[SW_LO + s] = local;
        for (int q = 0; q < m->world; ++q) {
            const uint32_t n = seg_at(m, m->seg, s, q);
            if (q == fr.rank) {
                h[SW_FIN_N + s] = n;
                h[SW_FIN_BASE + s] = (uint32_t) before;
                local += n;
            }
            before += n;
        }
    }
    h[SW_LO + m->n_seg] = local;
    for (int q = 0; q < fr.rank; ++q) before += m->inl[q];
    if (before + m->inl[fr.rank] >= (1ull << 31)) return mfail(m, RALA_B200_ERR_LIMIT, "finish: list positions must stay below 2^31");
    h[SW_ZERO + 1] = (uint32_t) before;   // time base of the local `internals`
    MCU(m, cudaMemcpyAsync(fr.stage.p, h.data(), SW_WORDS * 4, cudaMemcpyHostToDevice, L.stream));
    MRC(m, fr, begin_final_pass(g, C_TBASE_INL));
    MCU(m, cudaMemcpyAsync(g->cnt() + C_TBASE_INL, fr.stage_w(SW_ZERO + 1), 4, cudaMemcpyDeviceToDevice, L.stream));
    const List ovl = g->ovl[g->ovl_cur].view;
    for (uint32_t s = 0; s < m->n_seg; ++s) {
        if (s && !h[SW_FIN_N + s]) continue;   // (segment 0's launch also types `internals`)
        launch_classify_final(L, sub_list(ovl, h[SW_LO + s]), fr.stage_w(SW_FIN_N + s), fr.stage_w(SW_FIN_BASE + s), g->inl[g->inl_cur].view,
                              s ? fr.stage_w(SW_ZERO) : g->cnt() + g->slot_inl, g->cnt() + C_TBASE_INL, g->cap, g->piles.as<uint2>(),
                              g->events_view(), g->ev_cap, resolve_bufs(g).first, g->cnt());
    }
    MCU(m, cudaGetLastError());
    return route_and_meet(m, fr, 1);
}

// graph.cpp:867-877: the final lists (what edge creation reads), their per-segment counts and dovetails, published
static int phase_final_lists(rala_b200_multi* m, FabricRank& fr) {
    MCU(m, cudaSetDevice(fr.device));
    rala_b200_graph* g = fr.g;
    Launch& L = fr.ctx->L;
    const uint32_t S = m->n_seg;
    MCU(m, cudaMemsetAsync(fr.stage_w(SW_BOX), 0, kSegMail * 4, L.stream));
    launch_seg_count(L, g->ovl[g->ovl_cur].view, fr.stage_w(SW_LO), S, g->piles.as<uint2>(), kSegFinal, fr.stage_w(SW_BOX));
    launch_final_deaths(L, fr.P, fr.A, g->dbuf.as<uint32_t>());   // the k_list_pass<kFinalInt> filter reads them
    MRC(m, fr, materialize_final_lists(g));
    MCU(m, cudaMemcpyAsync(fr.stage_w(SW_BOX + 2 * S), g->cnt() + g->slot_inl, 4, cudaMemcpyDeviceToDevice, L.stream));
    launch_seg_push(L, fr.P, fr.A, fr.stage_w(SW_BOX), 2 * S + 1);
    launch_fabric_barrier(L, fr.P, no_mail(m));
    MCU(m, cudaGetLastError());
    return RALA_B200_OK;
}

// graph.cpp:831-877, 552-632 and 1281-1318 on the staged lists; edge ids are positions among the final dovetails in
// global list order, so a rank's edges are one run of ids per segment (rala_b200_multi_edge_runs)
extern "C" int rala_b200_multi_finish(rala_b200_multi* m) {
    if (!m) return RALA_B200_ERR_ARG;
    if (m->staged != 2) return mfail(m, RALA_B200_ERR_STATE, "finish: classify (rala_b200_multi_classify) first");
    int rc = staged_ready(m, "finish");
    if (rc) return rc;
    for (FabricRank& fr : m->ranks)
        if ((rc = phase_d_staged(m, fr))) return rc;
    for (FabricRank& fr : m->ranks)
        if ((rc = phase_e_final_resolve(m, fr))) return rc;
    for (FabricRank& fr : m->ranks)
        if ((rc = phase_final_lists(m, fr))) return rc;
    std::vector<uint32_t> mail;
    if ((rc = read_seg_mail(m, mail))) return rc;
    const uint32_t S = m->n_seg;
    const int W = m->world;
    for (int q = 0; q < W; ++q) {
        const uint32_t* box = mail.data() + (size_t) q * kSegMail;
        for (uint32_t s = 0; s < S; ++s) {
            seg_at(m, m->seg, s, q) = box[s];
            seg_at(m, m->dov, s, q) = box[S + s];
        }
        m->inl[q] = box[2 * S];
    }
    EdgeRuns& R = m->runs;
    R.n_seg = S;
    R.world = (uint32_t) W;
    uint64_t g_id = 0;
    std::vector<uint64_t> l_id((size_t) W, 0);
    for (uint32_t s = 0; s < S; ++s)
        for (int q = 0; q < W; ++q) {
            const size_t i = (size_t) s * W + q;
            R.gb[i] = (uint32_t) g_id;
            R.lb[i] = (uint32_t) l_id[q];
            g_id += 2ull * m->dov[i];
            l_id[q] += 2ull * m->dov[i];
        }
    if (g_id >= (1ull << 31)) return mfail(m, RALA_B200_ERR_LIMIT, "finish: %llu edges (ids must stay below 2^31)", (unsigned long long) g_id);
    for (FabricRank& fr : m->ranks) {
        MCU(m, cudaSetDevice(fr.device));
        MCU(m, cudaMemcpyAsync(fr.runs_dev(), &m->runs, sizeof(EdgeRuns), cudaMemcpyHostToDevice, fr.ctx->L.stream));
    }
    m->staged_edges = true;
    static const PhaseFn kBuild[] = {phase_f_edges, phase_g_csr, phase_h_transitive, phase_i_marks};
    for (PhaseFn phase : kBuild)
        for (FabricRank& fr : m->ranks)
            if ((rc = phase(m, fr))) return rc;
    m->staged = 3;
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_hill_coverage(rala_b200_multi* m, int k, uint32_t* cov_out) {
    if (!m || k < 0 || k >= m->n_local) return RALA_B200_ERR_ARG;
    if (m->staged < 2) return mfail(m, RALA_B200_ERR_STATE, "get_hill_coverage: classify (rala_b200_multi_classify) first");
    FabricRank& fr = m->ranks[k];
    MRC(m, fr, rala_b200_graph_get_hill_coverage(fr.g, cov_out));
    return RALA_B200_OK;
}

extern "C" int rala_b200_multi_get_lists(rala_b200_multi* m, int k, rala_ovl_t* ovl_out, uint64_t* ovl_pos_out, rala_ovl_t* int_out,
                                         uint64_t* int_pos_out, uint64_t* counts) {
    if (!m || k < 0 || k >= m->n_local || !counts) return RALA_B200_ERR_ARG;
    if (m->staged < 2) return mfail(m, RALA_B200_ERR_STATE, "get_lists: classify (rala_b200_multi_classify) first");
    FabricRank& fr = m->ranks[k];
    const int me = fr.rank;
    uint64_t n_ovl = 0;
    for (uint32_t s = 0; s < m->n_seg; ++s) n_ovl += seg_at(m, m->seg, s, me);
    counts[0] = n_ovl;
    counts[1] = m->inl[me];
    if (ovl_out || int_out) {
        rala_b200_counts_t c;
        MRC(m, fr, rala_b200_graph_counts(fr.g, &c));
        if (c.n_overlaps != counts[0] || c.n_internals != counts[1])
            return mfail(m, RALA_B200_ERR_STATE, "get_lists: rank %d holds %llu / %llu entries, the segment table says %llu / %llu", me,
                         (unsigned long long) c.n_overlaps, (unsigned long long) c.n_internals, (unsigned long long) counts[0],
                         (unsigned long long) counts[1]);
        MRC(m, fr, rala_b200_graph_get_lists(fr.g, ovl_out, int_out));
    }
    if (ovl_pos_out) {
        uint64_t global = 0, j = 0;
        for (uint32_t s = 0; s < m->n_seg; ++s)
            for (int q = 0; q < m->world; ++q) {
                const uint32_t n = seg_at(m, m->seg, s, q);
                if (q == me)
                    for (uint32_t i = 0; i < n; ++i) ovl_pos_out[j++] = global + i;
                global += n;
            }
    }
    if (int_pos_out) {
        uint64_t base = 0;
        for (int q = 0; q < me; ++q) base += m->inl[q];
        for (uint32_t i = 0; i < m->inl[me]; ++i) int_pos_out[i] = base + i;
    }
    return RALA_B200_OK;
}
