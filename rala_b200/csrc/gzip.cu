// gzip.cu — plain gzip (one DEFLATE stream per member, no block table) in host memory -> its inflated text in device
// memory, for the text readers (paf.cu, reads.cu) and rala_b200_inflate_gzip.
//
// Nothing in a DEFLATE stream says where a block starts or how much it inflates to, so the stream is cut into chunks of
// kChunk compressed bytes and each chunk is decoded from a guessed entry, the guesses verified by the decodes themselves:
//   finder:   one CTA per chunk tests bit offsets from the chunk's start (deflate::entry_at: a dynamic-block header, a
//             byte-aligned stored block, a member header); a chunk without one before its end merges into its predecessor
//   count:    one warp per chunk, lane 0 decodes (deflate::decode_span, counting mode) from the entry to the first
//             boundary at or after the next chunk's entry.  Chunk 0 starts at the stream's start, so a chunk whose
//             predecessor is verified and stopped exactly at its entry is verified too.  The host walks the chunks; where
//             a verified chunk stopped past its successor's entry that entry was false, and the successor is decoded again
//             from the stop in the next round (as is any successor of a chunk whose own entry was matched: a likely true
//             start).  Each round verifies at least one more chunk; decode errors count only in verified chunks.
//   scan:     output offsets of the verified chunks on the host; the text is allocated once.
//   symbols:  per run of chunks with at most kRunBytes of text, lane 0 decodes each chunk again into 16-bit symbols:
//             literal bytes (also written to the text), and markers 256 + (32768 - k) for bytes k places before the chunk,
//             copied like bytes inside it.  A distance before the member's start is refused here.
//   chain:    one CTA walks the run's chunks in order and resolves the markers of each chunk's last 32 KiB against the text
//             before the chunk, which the chain's earlier steps (and the literals) have made final: the window of chunk
//             i + 1 is the text's last 32 KiB before it.  The one sequential stage.
//   resolve:  every chunk resolves the markers of the rest of its text in parallel against the same windows.
//   CRC32:    one warp per 256 KiB segment of a member (warp slices joined by the GF(2) shift); the host joins each
//             member's segments and checks CRC32 and ISIZE against the trailers the symbol pass recorded.
#include <cstring>

#include "deflate.cuh"
#include "kernels.h"
#include "session.h"

namespace rb {

constexpr uint64_t kChunk = 64 << 10;            // compressed bytes per chunk (DESIGN.md §6: the measured trade-off)
constexpr uint64_t kRunBytes = 1ull << 30;        // text per symbol-pass run: the 16-bit scratch holds 2 GiB
constexpr uint32_t kDecodeWarps = 8;              // warps (chunks in flight) per CTA of the decode passes
constexpr uint32_t kSegBytes = 256 << 10;         // CRC32 segment
constexpr uint32_t kFindThreads = 256;
constexpr uint32_t kChainThreads = 1024;
constexpr uint64_t kPiece = RALA_B200_PAF_CHUNK_BYTES;   // compressed bytes per upload piece
constexpr unsigned long long kNone = ~0ull;

struct GzTask {                       // one chunk's decode
    unsigned long long start, stop;   // entry and the boundary it must reach (bits)
    unsigned long long base, cap;     // symbols: output offset in the text, output bytes (from the counting pass)
    long long floor;                  // symbols: the member's start relative to base
    unsigned long long trailers;      // symbols: index of the chunk's first member trailer
};

struct GzSeg {
    unsigned long long at;
    uint32_t len, pad;
};

// chunk c >= 1: the first entry in bits [8 c kChunk, 8 min((c + 1) kChunk, n)), kNone when there is none
__global__ void __launch_bounds__(kFindThreads) k_gzip_find(const uint8_t* __restrict__ in, unsigned long long n,
                                                            unsigned long long* __restrict__ entries) {
    __shared__ unsigned long long s_best;
    const unsigned long long c = blockIdx.x + 1ull, lo = c * kChunk * 8, hi = min((c + 1) * kChunk, n) * 8;
    if (threadIdx.x == 0) s_best = kNone;
    __syncthreads();
    for (unsigned long long b = lo; b < hi; b += kFindThreads) {
        const unsigned long long x = b + threadIdx.x;
        if (x < hi && deflate::entry_at(in, n, x)) atomicMin(&s_best, x);
        __syncthreads();
        if (s_best != kNone) break;
    }
    if (threadIdx.x == 0) entries[c] = s_best;
}

// one warp per task, lane 0 decodes; kWrite: symbols into sym (task.base - sym_base) and literals into text
template <bool kWrite>
__global__ void __launch_bounds__(kDecodeWarps * 32) k_gzip_decode(const uint8_t* __restrict__ in, unsigned long long n,
                                                                   const GzTask* __restrict__ tasks, uint32_t t0, uint32_t t1,
                                                                   uint16_t* sym, unsigned long long sym_base, uint8_t* text,
                                                                   deflate::Trailer* trailers, deflate::Span* __restrict__ spans) {
    __shared__ bgzf::Tables s_tab[kDecodeWarps];
    const uint32_t warp = warp_id();
    if (lane_id() != 0) return;
    for (uint32_t t = t0 + blockIdx.x * kDecodeWarps + warp; t < t1; t += gridDim.x * kDecodeWarps) {
        const GzTask T = tasks[t];
        deflate::Sink sink{nullptr, nullptr, T.cap, T.base, T.floor, nullptr};
        if (kWrite) {
            sink.sym = sym + (T.base - sym_base);
            sink.text = text + T.base;
            sink.trailers = trailers + T.trailers;
        }
        spans[t] = deflate::decode_span<kWrite>(in, n, T.start, T.stop, s_tab[warp], &sink);
    }
}

// The markers of each chunk's last 32 KiB, chunk after chunk: the text before chunk i is final once step i - 1 is done.
// A step is latency-bound, so every thread issues all its loads of a kind before it uses one: the 32 KiB window before
// the chunk into shared memory (coalesced), then the tail's symbols, then the stores (gathers from shared memory).
__global__ void __launch_bounds__(kChainThreads) k_gzip_chain(const uint16_t* __restrict__ sym, unsigned long long sym_base,
                                                              const GzTask* __restrict__ tasks, const deflate::Span* __restrict__ spans,
                                                              uint32_t t0, uint32_t t1, uint8_t* text) {
    constexpr uint32_t kPer = deflate::kWindow / kChainThreads;
    __shared__ uint8_t s_win[deflate::kWindow];
    for (uint32_t t = t0; t < t1; ++t) {
        const unsigned long long base = tasks[t].base, len = spans[t].out, hi = spans[t].last_marker;
        const unsigned long long lo = len > deflate::kWindow ? len - deflate::kWindow : 0;
        if (hi <= lo) continue;   // uniform across the CTA
        const uint16_t* s = sym + (base - sym_base) + lo;
        const uint32_t have = (uint32_t) min(base, (unsigned long long) deflate::kWindow), n = (uint32_t) (hi - lo);
        uint8_t w[kPer];
        uint32_t v[kPer];
#pragma unroll
        for (uint32_t j = 0; j < kPer; ++j) {
            const uint32_t i = threadIdx.x + j * kChainThreads;
            w[j] = i < have ? text[base - have + i] : 0;
            v[j] = i < n ? s[i] : 0u;
        }
#pragma unroll
        for (uint32_t j = 0; j < kPer; ++j) s_win[threadIdx.x + j * kChainThreads] = w[j];
        __syncthreads();
        const uint32_t skip = deflate::kWindow - have;   // marker 256 + skip names s_win[0] (no marker reaches before it)
#pragma unroll
        for (uint32_t j = 0; j < kPer; ++j)
            if (v[j] >= 256) text[base + lo + threadIdx.x + j * kChainThreads] = s_win[v[j] - 256 - skip];
        __syncthreads();
    }
}

// The markers before each chunk's last 32 KiB, all chunks at once (one CTA each).
__global__ void __launch_bounds__(256) k_gzip_resolve(const uint16_t* __restrict__ sym, unsigned long long sym_base,
                                                      const GzTask* __restrict__ tasks, const deflate::Span* __restrict__ spans,
                                                      uint32_t t0, uint8_t* __restrict__ text) {
    const uint32_t t = t0 + blockIdx.x;
    const unsigned long long base = tasks[t].base, len = spans[t].out;
    const unsigned long long head = len > deflate::kWindow ? len - deflate::kWindow : 0;
    const unsigned long long hi = min(head, (unsigned long long) spans[t].last_marker);
    const uint16_t* s = sym + (base - sym_base);
    for (unsigned long long q = threadIdx.x; q < hi; q += blockDim.x) {
        const uint32_t v = s[q];
        if (v >= 256) text[base + q] = text[base - deflate::kWindow + (v - 256)];
    }
}

__global__ void __launch_bounds__(256) k_gzip_crc(const uint8_t* __restrict__ text, const GzSeg* __restrict__ segs, uint32_t n_segs,
                                                  uint32_t* __restrict__ crc) {
    __shared__ uint32_t s_crc[256], s_x2n[32];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_crc[i] = bgzf::crc_table_entry(i);
    if (threadIdx.x == 0) bgzf::x2n_table(s_x2n);
    __syncthreads();
    const uint32_t lane = lane_id();
    for (uint32_t g = blockIdx.x * 8 + warp_id(); g < n_segs; g += gridDim.x * 8) {
        const GzSeg S = segs[g];
        const uint32_t c = bgzf::warp_crc(text + S.at, S.len, lane, s_crc, s_x2n);
        if (lane == 0) crc[g] = c;
    }
}

void preload_gzip() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_gzip_find);
    cudaFuncGetAttributes(&a, k_gzip_decode<false>);
    cudaFuncGetAttributes(&a, k_gzip_decode<true>);
    cudaFuncGetAttributes(&a, k_gzip_chain);
    cudaFuncGetAttributes(&a, k_gzip_resolve);
    cudaFuncGetAttributes(&a, k_gzip_crc);
}

}  // namespace rb

// ---------------------------------------------------------------------------------------------
// host side: the upload, the verification rounds and the launches
// ---------------------------------------------------------------------------------------------
static const char* gzip_error_text(uint32_t e) {
    switch (e) {
        case bgzf::kPastEnd: return "the input ends inside a DEFLATE stream";
        case bgzf::kBtype3: return "a DEFLATE block of type 3 (reserved)";
        case bgzf::kStoredLen: return "a stored block whose LEN is not the complement of NLEN";
        case bgzf::kCounts: return "a dynamic block with more than 286 literal/length or 30 distance codes";
        case bgzf::kOversubscribed: return "an over-subscribed Huffman code";
        case bgzf::kIncomplete: return "an incomplete Huffman code";
        case bgzf::kRepeat: return "a code-length repeat with no previous length or past the lengths it fills";
        case bgzf::kNoEob: return "the literal/length code has no end-of-block code";
        case bgzf::kBadSymbol: return "an invalid literal/length code (not in the code, or 286 / 287)";
        case bgzf::kBadDistSymbol: return "an invalid distance code (not in the code, or 30 / 31)";
        case bgzf::kTooFar: return "a distance that reaches before the start of the member";
        case bgzf::kCrc: return "the CRC32 of the inflated bytes differs from the trailer's";
        case deflate::kMagic: return "not a gzip member (magic 1f 8b expected)";
        case deflate::kMethod: return "compression method other than 8 (deflate)";
        case deflate::kFlags: return "reserved header flag bits set";
        case deflate::kHeaderEnd: return "the input ends inside the member header";
        case deflate::kHeaderCrc: return "the header CRC (FHCRC) differs from the header's CRC32";
        case deflate::kTrailerEnd: return "the input ends inside the member trailer";
        case deflate::kAfterLast: return "non-zero bytes after the last member";
        case deflate::kIsize: return "ISIZE differs from the member's inflated size mod 2^32";
        default: return "an internal decode error";
    }
}

static int gzip_fail(rala_b200_ctx* ctx, uint64_t member, uint64_t at, uint32_t why) {
    return fail(ctx, RALA_B200_ERR_ARG, "gzip member %llu (byte offset %llu): %s", (unsigned long long) member, (unsigned long long) at,
                gzip_error_text(why));
}

namespace {

struct StageTimer {   // (stage, start, stop) events around every launch
    rala_b200_ctx* ctx;
    std::vector<std::pair<int, cudaEvent_t>> ev;
    ~StageTimer() {
        for (auto& e : ev) cudaEventDestroy(e.second);
    }
    cudaError_t mark(int stage) {
        cudaEvent_t e;
        cudaError_t rc = cudaEventCreate(&e);
        if (rc) return rc;
        ev.push_back({stage, e});
        return cudaEventRecord(e, ctx->L.stream);
    }
    // after a synchronise: device time per stage into ms[5]
    void sum(float* ms) {
        for (size_t i = 0; i + 1 < ev.size(); i += 2) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, ev[i].second, ev[i + 1].second) == cudaSuccess) ms[ev[i].first] += t;
        }
    }
};

}  // namespace

// data[0, n) -> R.packed in pieces on the copy stream (pageable memory through the pinned pair); the main stream waits
static int upload(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n) {
    CU(ctx, R.packed.reserve(n + 8));
    if (!R.copy) CU(ctx, cudaStreamCreateWithFlags(&R.copy, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k)
        if (!R.copied[k]) CU(ctx, cudaEventCreateWithFlags(&R.copied[k], cudaEventDisableTiming));
    bool direct = false;   // page-locked caller memory is uploaded in place
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, data) == cudaSuccess) direct = attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    for (int k = 0; !direct && k < 2; ++k)
        if (!R.pinned[k]) CU(ctx, cudaHostAlloc((void**) &R.pinned[k], rb::kPiece + 1, cudaHostAllocDefault));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));   // earlier kernels may still read R.packed
    uint8_t* din = R.packed.as<uint8_t>();
    uint32_t k = 0;
    for (uint64_t lo = 0; lo < n; lo += rb::kPiece, ++k) {
        const uint64_t len = n - lo < rb::kPiece ? n - lo : rb::kPiece;
        const int slot = k & 1;
        const uint8_t* src = data + lo;
        if (!direct) {
            if (k >= 2) CU(ctx, cudaEventSynchronize(R.copied[slot]));   // the upload of piece k - 2 has left the buffer
            memcpy(R.pinned[slot], src, len);
            src = (const uint8_t*) R.pinned[slot];
        }
        CU(ctx, cudaMemcpyAsync(din + lo, src, len, cudaMemcpyHostToDevice, R.copy));
        CU(ctx, cudaEventRecord(R.copied[slot], R.copy));
    }
    if (k) CU(ctx, cudaStreamWaitEvent(ctx->L.stream, R.copied[(k - 1) & 1], 0));
    return RALA_B200_OK;
}

static int gzip_inflate_once(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_gzip_stats_t* st,
                             uint8_t* host_out, uint64_t cap, bool size_only) {
    using namespace rb;
    using deflate::Span;
    using deflate::Trailer;
    CU(ctx, cudaSetDevice(ctx->device));
    *st = rala_b200_gzip_stats_t{};
    st->n_compressed = n;
    st->chunk_bytes = kChunk;
    if (n == 0) return RALA_B200_OK;
    if (is_bgzf(data, n)) {
        rala_b200_bgzf_stats_t z{};
        int rc = RALA_B200_OK;
        if (size_only) {
            rc = rala_b200_inflate_bgzf(ctx, data, n, nullptr, 0, &z);
        } else {
            rc = bgzf_inflate(ctx, R, data, n, &z, host_out, cap);
        }
        st->n_members = z.n_blocks;
        st->n_bytes = z.n_bytes;
        st->bgzf = 1;
        st->chunk_bytes = 0;
        st->inflate_ms = z.inflate_ms;
        return rc;
    }
    cudaStream_t s = ctx->L.stream;
    int rc = upload(ctx, R, data, n);
    if (rc) return rc;
    const uint8_t* din = R.packed.as<uint8_t>();
    StageTimer T{ctx, {}};
    const uint64_t n_cut = (n + kChunk - 1) / kChunk, end = n * 8;
    // chunk table: entries | tasks | spans, sized for every cut
    const size_t o_tasks = align_up(n_cut * 8, 256), o_spans = o_tasks + align_up(n_cut * sizeof(GzTask), 256);
    CU(ctx, R.gz_meta.reserve(o_spans + n_cut * sizeof(Span)));
    unsigned long long* d_entries = R.gz_meta.as<unsigned long long>();
    GzTask* d_tasks = (GzTask*) (R.gz_meta.as<char>() + o_tasks);
    Span* d_spans = (Span*) (R.gz_meta.as<char>() + o_spans);
    std::vector<unsigned long long> cut(n_cut, 0);
    if (n_cut > 1) {
        CU(ctx, T.mark(0));
        k_gzip_find<<<(unsigned) (n_cut - 1), kFindThreads, 0, s>>>(din, n, d_entries);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(0));
        CU(ctx, cudaMemcpyAsync(cut.data() + 1, d_entries + 1, (n_cut - 1) * 8, cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
    }
    std::vector<unsigned long long> E;   // the entries of the chunks (chunks without one merged into their predecessor)
    for (uint64_t c = 0; c < n_cut; ++c)
        if (cut[c] != kNone) E.push_back(cut[c]);

    // ---- counting rounds --------------------------------------------------------------------------------------------
    std::vector<Span> res(E.size());
    std::vector<uint32_t> dirty(E.size());
    for (uint32_t i = 0; i < dirty.size(); ++i) dirty[i] = i;
    std::vector<GzTask> tasks;
    std::vector<Span> got;
    size_t err_chunk = SIZE_MAX;
    while (!dirty.empty()) {
        tasks.clear();
        for (uint32_t i : dirty) tasks.push_back(GzTask{E[i], i + 1 < E.size() ? E[i + 1] : kNone, 0, 0, 0, 0});
        const uint32_t nt = (uint32_t) tasks.size();
        CU(ctx, cudaMemcpyAsync(d_tasks, tasks.data(), nt * sizeof(GzTask), cudaMemcpyHostToDevice, s));
        CU(ctx, T.mark(1));
        k_gzip_decode<false><<<grid_for(nt, kDecodeWarps, kNumSMs * 8), kDecodeWarps * 32, 0, s>>>(din, n, d_tasks, 0, nt, nullptr, 0,
                                                                                                 nullptr, nullptr, d_spans);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(1));
        got.resize(nt);
        CU(ctx, cudaMemcpyAsync(got.data(), d_spans, nt * sizeof(Span), cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
        if (st->rounds) st->n_corrected += nt;
        st->rounds++;
        for (uint32_t j = 0; j < nt; ++j) res[dirty[j]] = got[j];
        const size_t e = deflate::walk(E, res, n * 8, dirty);
        if (e != SIZE_MAX) err_chunk = e;
    }
    const size_t nc = E.size();
    std::vector<unsigned long long> base(nc + 1, 0), mem(nc + 1, 0);
    std::vector<long long> floors(nc, 0);
    unsigned long long member_start = 0;
    for (size_t i = 0; i < nc; ++i) {
        base[i + 1] = base[i] + res[i].out;
        mem[i + 1] = mem[i] + res[i].members;
        floors[i] = (long long) member_start - (long long) base[i];
        if (res[i].last_start) member_start = base[i] + res[i].last_start - 1;
    }
    const uint64_t total = base[nc];
    st->n_chunks = nc;
    if (err_chunk == SIZE_MAX) {
        st->n_members = mem[nc];
        st->n_bytes = total;
    }
    if (total >> 34) return fail(ctx, RALA_B200_ERR_LIMIT, "gzip input inflates to %llu bytes or more: 2^34 or more", (unsigned long long) total);
    if (size_only && err_chunk == SIZE_MAX) {   // a failing stream goes on: an earlier CRC32 or distance error comes first
        T.sum(st->stage_ms);
        for (float ms : st->stage_ms) st->inflate_ms += ms;
        return RALA_B200_OK;
    }
    if (host_out && err_chunk == SIZE_MAX && total > cap)
        return fail(ctx, RALA_B200_ERR_ARG, "inflate_gzip: the input inflates to %llu bytes, the output holds %llu", (unsigned long long) total,
                    (unsigned long long) cap);

    // ---- symbols, chain and resolve per run ----------------------------------------------------------------------------
    tasks.resize(nc);
    uint64_t run_max = 0;
    for (size_t a = 0, b; a < nc; a = b) {
        for (b = a + 1; b < nc && base[b + 1] - base[a] <= kRunBytes;) ++b;
        run_max = std::max<uint64_t>(run_max, base[b] - base[a]);
    }
    for (size_t i = 0; i < nc; ++i)
        tasks[i] = GzTask{E[i], i + 1 < nc ? E[i + 1] : kNone, base[i], res[i].out, floors[i], mem[i]};
    CU(ctx, R.inflated.reserve(total + 1));
    CU(ctx, R.gz_sym.reserve(run_max * 2 + 2));
    CU(ctx, R.gz_trailers.reserve((mem[nc] + 1) * sizeof(Trailer)));
    CU(ctx, cudaMemcpyAsync(d_tasks, tasks.data(), nc * sizeof(GzTask), cudaMemcpyHostToDevice, s));
    uint8_t* text = R.inflated.as<uint8_t>();
    uint16_t* sym = R.gz_sym.as<uint16_t>();
    Trailer* d_trailers = R.gz_trailers.as<Trailer>();
    for (size_t a = 0, b; a < nc; a = b) {
        for (b = a + 1; b < nc && base[b + 1] - base[a] <= kRunBytes;) ++b;
        const uint32_t nr = (uint32_t) (b - a);
        CU(ctx, T.mark(2));
        k_gzip_decode<true><<<grid_for(nr, kDecodeWarps, kNumSMs * 8), kDecodeWarps * 32, 0, s>>>(
            din, n, d_tasks, (uint32_t) a, (uint32_t) b, sym, base[a], text, d_trailers, d_spans);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(2));
        CU(ctx, T.mark(3));
        k_gzip_chain<<<1, kChainThreads, 0, s>>>(sym, base[a], d_tasks, d_spans, (uint32_t) a, (uint32_t) b, text);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(3));
        CU(ctx, T.mark(4));
        k_gzip_resolve<<<nr, 256, 0, s>>>(sym, base[a], d_tasks, d_spans, (uint32_t) a, text);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(4));
    }
    std::vector<Span> sp(nc);
    std::vector<Trailer> tr(mem[nc]);
    CU(ctx, cudaMemcpyAsync(sp.data(), d_spans, nc * sizeof(Span), cudaMemcpyDeviceToHost, s));
    if (mem[nc]) CU(ctx, cudaMemcpyAsync(tr.data(), d_trailers, mem[nc] * sizeof(Trailer), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    // the first decode error in stream order; the members whose trailers come before it are checked below
    uint64_t bad_member = ~0ull, bad_at = ~0ull;
    uint32_t bad_why = 0;
    size_t n_tr = tr.size();
    for (size_t i = 0; i < nc; ++i) {
        if (!sp[i].err) continue;
        bad_member = mem[i] + sp[i].members;
        bad_at = sp[i].err_at;
        bad_why = sp[i].err;
        n_tr = bad_member;
        break;
    }

    // ---- CRC32 and ISIZE -----------------------------------------------------------------------------------------------
    std::vector<GzSeg> segs;
    std::vector<uint32_t> seg_member;
    for (size_t m = 0; m < n_tr; ++m) {
        const unsigned long long lo = m ? tr[m - 1].out_end : 0, hi = tr[m].out_end;
        for (unsigned long long p = lo; p < hi; p += kSegBytes) {
            segs.push_back(GzSeg{p, (uint32_t) std::min<unsigned long long>(kSegBytes, hi - p), 0});
            seg_member.push_back((uint32_t) m);
        }
    }
    std::vector<uint32_t> seg_crc(segs.size());
    if (!segs.empty()) {
        CU(ctx, R.gz_seg.reserve(segs.size() * (sizeof(GzSeg) + 4)));
        GzSeg* d_segs = R.gz_seg.as<GzSeg>();
        uint32_t* d_crc = (uint32_t*) (d_segs + segs.size());
        CU(ctx, cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(GzSeg), cudaMemcpyHostToDevice, s));
        CU(ctx, T.mark(4));
        k_gzip_crc<<<grid_for(segs.size(), 8, kNumSMs * 8), 256, 0, s>>>(text, d_segs, (uint32_t) segs.size(), d_crc);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, T.mark(4));
        CU(ctx, cudaMemcpyAsync(seg_crc.data(), d_crc, segs.size() * 4, cudaMemcpyDeviceToHost, s));
    }
    CU(ctx, cudaStreamSynchronize(s));
    T.sum(st->stage_ms);
    for (float ms : st->stage_ms) st->inflate_ms += ms;
    uint32_t x2n[32];
    bgzf::x2n_table(x2n);
    std::vector<uint32_t> crc(n_tr, 0);
    for (size_t g = 0; g < segs.size(); ++g) crc[seg_member[g]] = bgzf::crc_combine(crc[seg_member[g]], seg_crc[g], segs[g].len, x2n);
    for (size_t m = 0; m < n_tr; ++m) {
        const unsigned long long size = tr[m].out_end - (m ? tr[m - 1].out_end : 0);
        if (crc[m] != tr[m].crc) return gzip_fail(ctx, m, tr[m].at, bgzf::kCrc);
        if ((uint32_t) size != tr[m].isize) return gzip_fail(ctx, m, tr[m].at, deflate::kIsize);
    }
    if (bad_why) return gzip_fail(ctx, bad_member, bad_at, bad_why);
    if (host_out && total) {
        CU(ctx, cudaMemcpyAsync(host_out, text, total, cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
    }
    return RALA_B200_OK;
}

int gzip_inflate(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_gzip_stats_t* st, uint8_t* host_out,
                 uint64_t cap, bool size_only) {
    const int rc = gzip_inflate_once(ctx, R, data, n, st, host_out, cap, size_only);
    if (rc) {
        if (R.copy) cudaStreamSynchronize(R.copy);
        cudaStreamSynchronize(ctx->L.stream);
    }
    return rc;
}

int inflate_packed(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, const Packed& z, uint64_t* n_bytes) {
    const int rc = z.bgzf ? bgzf_inflate(ctx, R, data, n, z.bgzf) : gzip_inflate(ctx, R, data, n, z.gzip);
    *n_bytes = z.bgzf ? z.bgzf->n_bytes : z.gzip->n_bytes;
    return rc;
}

extern "C" int rala_b200_inflate_gzip(rala_b200_ctx* ctx, const uint8_t* data, uint64_t n, uint8_t* out, uint64_t cap,
                                      rala_b200_gzip_stats_t* stats) {
    if (!ctx || (n && !data)) return RALA_B200_ERR_ARG;
    rala_b200_gzip_stats_t st{};
    PafReader R;
    const int rc = gzip_inflate(ctx, R, data, n, &st, out, cap, out == nullptr);
    if (stats && !rc) *stats = st;
    return rc;
}
