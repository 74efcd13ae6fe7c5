// reads.cu — FASTA or FASTQ text in host memory -> the graph session's read names, lengths and name table: the first half
// of Graph::initialize (graph.cpp:249-264, name_to_id_ and one pile per read) without a host parse.  What
// rala_b200_graph_set_reads is given as host arrays is built on the device from the sequence file.
//
//   per upload chunk (the upload and k_paf_line_ends are paf.cu's):
//     k_reads_roles    one thread per line (4 lines per thread, tiles of 1 024 lines): header or not (FASTA: first byte
//                      '>'; FASTQ: the global line index mod 4), one decoupled look-back over (headers, name bytes) whose
//                      running totals are carried from chunk to chunk; the header lines write their names into the blob
//                      with the reads' name ends and header lines, the sequence lines add their lengths to their read
//                      (a read may span any number of chunks), the structure rules (empty line, '@' / '+' lines,
//                      quality length, name bytes) lower the error word
//     k_reads_bytes    one warp per line, 128 bytes per step: the byte rules ('\r' anywhere, sequence bytes 0x21..0x7E)
//   per call:
//     k_reads_finish   per read: the 64-bit sums into the u32 lengths of the set_reads layout, reads without sequence or
//                      of 2^32 bases refused, bases and the longest read counted
//     k_paf_names      the name table and the duplicate check, unchanged (paf.cu)
//
// The text contract is in include/rala_b200.h.  A refusal lowers the call's error word with line << 30 | column << 4 | kind:
// the smallest line wins, then the smallest column, then the smallest kind.
#include <cstring>

#include "kernels.h"
#include "session.h"

namespace rb {

constexpr uint32_t kLineItems = 4;                               // lines per thread of k_reads_roles
constexpr uint32_t kLineTile = kTileThreads * kLineItems;        // lines per tile
constexpr unsigned long long kMaxReads = (1ull << 31) - 1;       // read ids below this: a read count below 2^31
enum : uint32_t { kRdEmpty = 1, kRdCr, kRdHeader, kRdNameEmpty, kRdNameByte, kRdSeqByte, kRdPlus, kRdQualLen, kRdTruncated,
                  kRdNoSeq, kRdTooLong, kRdTooMany, kRdFormat };
// words of one call beside PafReader::words: headers with a description, bases, the longest read; then for chunk k the
// reads and the name bytes before it at RW_RUN + 2k and RW_RUN + 2k + 1
enum { RW_DESCRIBED = 0, RW_BASES, RW_MAX_LEN, RW_RUN = 4 };

struct ReadsOut {
    unsigned long long *len, *name_end, *line;   // per read: bases so far, end of its name in blob, 0-based line of its header
    uint8_t* blob;
    unsigned long long cap;                       // reads the three columns hold
};

__host__ __device__ __forceinline__ unsigned long long reads_err(unsigned long long line, uint32_t column, uint32_t kind) {
    return line << 30 | (unsigned long long) column << 4 | kind;   // line < 2^34, column < 2^26
}

__device__ __forceinline__ unsigned long long warp_inclusive_scan64(unsigned long long v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if ((int) lane_id() >= d) v += t;
    }
    return v;
}

__global__ void __launch_bounds__(kTileThreads) k_reads_roles(const uint8_t* __restrict__ text, const uint32_t* __restrict__ line_end,
                                                             const unsigned long long* __restrict__ lines, unsigned long long* __restrict__ rw,
                                                             uint32_t chunk, uint32_t fastq, ReadsOut out, unsigned long long* __restrict__ status,
                                                             uint32_t* __restrict__ ticket, unsigned long long* __restrict__ words) {
    __shared__ unsigned long long s_warp[kTileWarps];
    __shared__ uint32_t s_tile;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const unsigned long long line0 = lines[chunk];
    const uint32_t n_lines = (uint32_t) (lines[chunk + 1] - line0);
    const unsigned long long rec0 = rw[RW_RUN + 2 * chunk], nb0 = rw[RW_RUN + 2 * chunk + 1];
    const uint32_t num_tiles = (n_lines + kLineTile - 1) / kLineTile;
    unsigned long long err = ~0ull;
    uint32_t described = 0;
    while (true) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= num_tiles) break;
        const uint32_t first = tile * kLineTile + tid * kLineItems;
        uint32_t name_len[kLineItems], hdr_mask = 0, hdrs = 0, bytes = 0;
#pragma unroll
        for (uint32_t r = 0; r < kLineItems; ++r) {
            const uint32_t line = first + r;
            name_len[r] = 0;
            if (line >= n_lines) continue;
            const uint32_t s = line ? line_end[line - 1] + 1u : 0u, e = line_end[line];
            const unsigned long long g = line0 + line;
            if (!(fastq ? (g & 3u) == 0 : e > s && text[s] == '>')) continue;
            hdr_mask |= 1u << r;
            ++hdrs;
            if (e == s) continue;   // an empty FASTQ header line: refused as empty below
            uint32_t p = s + 1, bad = 0;
            for (; p < e; ++p) {   // the name: up to the first space or tab
                const uint32_t c = text[p];
                if (c == ' ' || c == '\t') break;
                if (!bad && ((c < 0x20u && c != '\r') || c == 0x7Fu)) bad = p - s + 1;   // '\r' is k_reads_bytes' refusal
            }
            name_len[r] = p - s - 1;
            bytes += name_len[r];
            described += p < e;
            if (bad) err = min(err, reads_err(g, bad, kRdNameByte));
            if (p == s + 1) err = min(err, reads_err(g, 2, kRdNameEmpty));
        }
        // (headers, name bytes) before this thread's lines: the block's scan, then the tiles' look-back
        const unsigned long long mine = pack_counts(hdrs, bytes), inc = warp_inclusive_scan64(mine);
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long v = lane < kTileWarps ? s_warp[lane] : 0ull, wi = warp_inclusive_scan64(v);
            const unsigned long long total = __shfl_sync(0xFFFFFFFFu, wi, 31);
            const unsigned long long excl = lookback_exclusive(status, tile, total);
            if (lane < kTileWarps) s_warp[lane] = excl + wi - v;
            if (tile == num_tiles - 1 && lane == 0) {
                rw[RW_RUN + 2 * chunk + 2] = rec0 + count_a(excl + total);
                rw[RW_RUN + 2 * chunk + 3] = nb0 + count_b(excl + total);
            }
        }
        __syncthreads();
        const unsigned long long pre = s_warp[warp] + inc - mine;
        unsigned long long rec = rec0 + count_a(pre), nb = nb0 + count_b(pre);
        __syncthreads();   // s_warp is read before the next tile writes it
#pragma unroll
        for (uint32_t r = 0; r < kLineItems; ++r) {
            const uint32_t line = first + r;
            if (line >= n_lines) continue;
            const uint32_t s = line ? line_end[line - 1] + 1u : 0u, e = line_end[line], n = e - s;
            const unsigned long long g = line0 + line;
            if (n == 0) err = min(err, reads_err(g, 1, kRdEmpty));
            if ((hdr_mask >> r) & 1u) {
                if (rec >= kMaxReads) {
                    err = min(err, reads_err(g, 1, kRdTooMany));
                } else if (rec < out.cap) {
                    for (uint32_t i = 0; i < name_len[r]; ++i) out.blob[nb + i] = text[s + 1 + i];
                    out.name_end[rec] = nb + name_len[r];
                    out.line[rec] = g;
                }
                if (fastq && n && text[s] != '@') err = min(err, reads_err(g, 1, kRdHeader));
                ++rec;
                nb += name_len[r];
                continue;
            }
            const unsigned long long cur = rec - 1;   // the read of this line (line 1 is always a header)
            if (n == 0 || rec == 0 || cur >= out.cap) continue;
            const uint32_t role = (uint32_t) (g & 3u);
            if (!fastq) {
                atomicAdd(out.len + cur, (unsigned long long) n);
            } else if (role == 1) {
                out.len[cur] = n;
            } else if (role == 2) {
                if (text[s] != '+') err = min(err, reads_err(g, 1, kRdPlus));
            } else {   // quality: as long as the sequence line two lines up, in this chunk or stored by an earlier one
                const unsigned long long want =
                    line >= 2 ? line_end[line - 2] - (line >= 3 ? line_end[line - 3] + 1u : 0u) : out.len[cur];
                if (n != want) err = min(err, reads_err(g, (uint32_t) min((unsigned long long) n, want) + 1, kRdQualLen));
            }
        }
    }
    if (err != ~0ull) atomicMin(words + W_ERR, err);
    if (described) atomicAdd(rw + RW_DESCRIBED, (unsigned long long) described);
}

// The byte rules, one warp per line: the first byte of the line that is a '\r', or on a sequence line outside 0x21..0x7E.
__global__ void __launch_bounds__(256) k_reads_bytes(const uint8_t* __restrict__ text, const uint32_t* __restrict__ line_end,
                                                     const unsigned long long* __restrict__ lines, uint32_t chunk, uint32_t fastq,
                                                     unsigned long long* __restrict__ words) {
    const unsigned long long line0 = lines[chunk];
    const uint32_t n_lines = (uint32_t) (lines[chunk + 1] - line0);
    const uint32_t lane = lane_id(), warp = warp_id();
    for (uint32_t line = blockIdx.x * kTileWarps + warp; line < n_lines; line += gridDim.x * kTileWarps) {
        const uint32_t s = line ? line_end[line - 1] + 1u : 0u, e = line_end[line];
        const unsigned long long g = line0 + line;
        const bool seq = fastq ? (g & 3u) == 1 : !(e > s && text[s] == '>');
        for (uint32_t w = s & ~3u; w < e; w += 128u) {
            const uint32_t p0 = w + 4u * lane;
            const uint32_t word = *reinterpret_cast<const uint32_t*>(text + p0);
            uint32_t bad = 4, byte = 0;
#pragma unroll
            for (uint32_t k = 0; k < 4; ++k) {
                const uint32_t c = (word >> (8 * k)) & 0xFFu, p = p0 + k;
                if (bad == 4 && p >= s && p < e && (c == '\r' || (seq && (c < 0x21u || c > 0x7Eu)))) {
                    bad = k;
                    byte = c;
                }
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, bad < 4);
            if (m) {
                if (lane == (uint32_t) (__ffs(m) - 1))
                    atomicMin(words + W_ERR, reads_err(g, p0 + bad - s + 1, byte == '\r' ? kRdCr : kRdSeqByte));
                break;
            }
        }
    }
}

// Per read: the 64-bit length into the u32 column of the set_reads layout, the name end next to it; a read without
// sequence or of 2^32 bases is refused at its header line.
__global__ void __launch_bounds__(256) k_reads_finish(ReadsOut in, uint32_t n, unsigned long long* __restrict__ end_out,
                                                      uint32_t* __restrict__ len_out, unsigned long long* __restrict__ rw,
                                                      unsigned long long* __restrict__ words) {
    unsigned long long bases = 0, longest = 0, err = ~0ull;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long len = in.len[i];
        if (len == 0) err = min(err, reads_err(in.line[i], 1, kRdNoSeq));
        if (len >> 32) err = min(err, reads_err(in.line[i], 1, kRdTooLong));
        len_out[i] = (uint32_t) min(len, 0xFFFFFFFFull);
        end_out[i] = in.name_end[i];
        bases += len;
        longest = max(longest, len);
    }
    bases = warp_sum64(bases);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) longest = max(longest, __shfl_xor_sync(0xFFFFFFFFu, longest, d));
    if (lane_id() == 0) {
        if (bases) atomicAdd(rw + RW_BASES, bases);
        if (longest) atomicMax(rw + RW_MAX_LEN, longest);
    }
    if (err != ~0ull) atomicMin(words + W_ERR, err);
}

void preload_reads() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_reads_roles);
    cudaFuncGetAttributes(&a, k_reads_bytes);
    cudaFuncGetAttributes(&a, k_reads_finish);
}

}  // namespace rb

// ---------------------------------------------------------------------------------------------
// host side: the per-read accumulators of one call, grown between chunks, and the hand-over to the name table
// ---------------------------------------------------------------------------------------------
// What one call holds beside the PafReader: the reads' 64-bit sums, name ends, header lines and the name blob, sized
// from the reads seen so far plus what one chunk can add; released when the call returns.
struct ReadsCall {
    PafReader* R = nullptr;
    bool fastq = false;
    DevBuf len, name_end, line, blob, rw;
    unsigned long long cap = 0, blob_cap = 0;
    unsigned long long* host = nullptr;   // pinned: reads and name bytes behind the last chunk launched
    cudaEvent_t counted = nullptr, ev[2] = {nullptr, nullptr};

    ReadsOut view() const {
        return ReadsOut{len.as<unsigned long long>(), name_end.as<unsigned long long>(), line.as<unsigned long long>(),
                        blob.as<uint8_t>(), cap};
    }
    ~ReadsCall() {
        DevBuf* bufs[] = {&len, &name_end, &line, &blob, &rw};
        for (DevBuf* b : bufs) b->release();
        if (host) cudaFreeHost(host);
        if (counted) cudaEventDestroy(counted);
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
    }
};

// b to `want` bytes, its first `used` kept (and the rest zeroed when asked)
static int grow(rala_b200_ctx* ctx, DevBuf& b, size_t used, size_t want, bool zero) {
    DevBuf n;
    cudaStream_t s = ctx->L.stream;
    cudaError_t e = n.reserve(want);
    if (e == cudaSuccess && used) e = cudaMemcpyAsync(n.p, b.p, used, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess && zero) e = cudaMemsetAsync(n.as<char>() + used, 0, want - used, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        n.release();
        return fail(ctx, RALA_B200_ERR_CUDA, "growing the read buffers failed: %s", cudaGetErrorString(e));
    }
    b.release();
    b = n;
    return RALA_B200_OK;
}

// ChunkKernels of set_reads_text
static int reads_chunk(void* self, rala_b200_ctx* ctx, uint32_t k, const uint8_t* dtext, uint32_t scan_len) {
    ReadsCall& c = *static_cast<ReadsCall*>(self);
    PafReader& R = *c.R;
    cudaStream_t s = ctx->L.stream;
    unsigned long long recs = 0, nb = 0;
    if (k) {   // the previous chunk's totals (its roles kernel finished while this chunk was uploaded)
        CU(ctx, cudaEventSynchronize(c.counted));
        recs = c.host[0];
        nb = c.host[1];
    }
    // a header line takes at least 2 bytes, so this chunk adds at most scan_len / 2 + 1 reads and scan_len name bytes
    unsigned long long need = recs + scan_len / 2 + 1;
    if (need > kMaxReads) need = kMaxReads;
    if (need > c.cap) {
        unsigned long long cap = 2 * c.cap > need ? 2 * c.cap : need;
        if (cap > kMaxReads) cap = kMaxReads;
        const size_t used = (size_t) (recs < c.cap ? recs : c.cap) * 8;
        int rc = grow(ctx, c.len, used, (size_t) cap * 8, true);
        if (!rc) rc = grow(ctx, c.name_end, used, (size_t) cap * 8, false);
        if (!rc) rc = grow(ctx, c.line, used, (size_t) cap * 8, false);
        if (rc) return rc;
        c.cap = cap;
    }
    if (nb + scan_len > c.blob_cap) {
        const unsigned long long cap = 2 * c.blob_cap > nb + scan_len ? 2 * c.blob_cap : nb + scan_len;
        const int rc = grow(ctx, c.blob, (size_t) nb, (size_t) cap, false);
        if (rc) return rc;
        c.blob_cap = cap;
    }
    unsigned long long* words = R.words.as<unsigned long long>();
    unsigned long long* rw = c.rw.as<unsigned long long>();
    unsigned long long* st_words = R.status.as<unsigned long long>();
    CU(ctx, cudaMemsetAsync(st_words, 0, text_status_words() * 8, s));
    k_reads_roles<<<grid_for(scan_len, kLineTile * 16, kNumSMs * 8), kTileThreads, 0, s>>>(
        dtext, R.line_end.as<uint32_t>(), words + W_BASES, rw, k, c.fastq, c.view(), st_words + 1, (uint32_t*) st_words, words);
    ctx->L.count++;
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(c.host, rw + RW_RUN + 2 * (k + 1), 16, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaEventRecord(c.counted, s));
    k_reads_bytes<<<grid_for(scan_len, kTileWarps * 64, kNumSMs * 8), 256, 0, s>>>(dtext, R.line_end.as<uint32_t>(), words + W_BASES,
                                                                                  k, c.fastq, words);
    ctx->L.count++;
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

static const char* reads_error_text(uint32_t kind) {
    switch (kind) {
        case kRdEmpty: return "the line is empty";
        case kRdCr: return "a carriage return (CRLF line ends are not read)";
        case kRdHeader: return "the first line of a FASTQ record does not start with '@'";
        case kRdNameEmpty: return "the read name is empty";
        case kRdNameByte: return "a control byte in the read name";
        case kRdSeqByte: return "a sequence byte outside 0x21..0x7E";
        case kRdPlus: return "the third line of a FASTQ record does not start with '+'";
        case kRdQualLen: return "the quality line is not as long as the sequence line";
        case kRdTruncated: return "the text ends inside this FASTQ record";
        case kRdNoSeq: return "the read has no sequence";
        case kRdTooLong: return "the read has 2^32 bases or more";
        case kRdTooMany: return "the 2^31st read (read counts are below 2^31)";
        default: return "the text starts with neither '>' (FASTA) nor '@' (FASTQ)";
    }
}

// z (nullable): text[0, n_bytes) is a BGZF or gzip file, inflated on the device first.
static int reads_text(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_reads_stats_t* st, const Packed* z = nullptr) {
    rala_b200_ctx* ctx = g->ctx;
    if (!g->paf) g->paf = new PafReader();
    PafReader& R = *g->paf;
    R.have_names = false;
    g->text_records = kTextNone;   // the records' ids refer to the reads they were parsed against
    *st = rala_b200_reads_stats_t{};
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->L.stream;
    char first = n_bytes ? text[0] : 0;
    if (z) {
        const int rc = inflate_packed(ctx, R, (const uint8_t*) text, n_bytes, *z, &n_bytes);
        if (rc) return rc;
        text = R.inflated.as<const char>();
        if (n_bytes) {
            CU(ctx, cudaMemcpyAsync(&first, text, 1, cudaMemcpyDeviceToHost, s));
            CU(ctx, cudaStreamSynchronize(s));
        }
    }
    st->n_bytes = n_bytes;
    if (n_bytes == 0) {   // no reads, as set_reads with n_reads = 0
        R.max_len = 0;
        CU(ctx, R.names.reserve(names_layout(0, 0).bytes));
        return names_table(ctx, R, 0, 0);
    }
    if (first != '>' && first != '@')
        return fail(ctx, RALA_B200_ERR_ARG, "FASTA / FASTQ line 1, column 1: %s", reads_error_text(kRdFormat));
    const bool fastq = first == '@';
    const char* label = fastq ? "FASTQ" : "FASTA";
    if (n_bytes >> 34) return fail(ctx, RALA_B200_ERR_LIMIT, "%s text of %llu bytes: 2^34 or more", label, (unsigned long long) n_bytes);
    ReadsCall c;
    c.R = &R;
    c.fastq = fastq;
    const size_t rw_bytes = (RW_RUN + 2 * text_max_chunks(n_bytes) + 4) * 8;
    CU(ctx, c.rw.reserve(rw_bytes));
    CU(ctx, cudaMemsetAsync(c.rw.p, 0, rw_bytes, s));
    CU(ctx, cudaHostAlloc((void**) &c.host, 16, cudaHostAllocDefault));
    CU(ctx, cudaEventCreateWithFlags(&c.counted, cudaEventDisableTiming));
    for (cudaEvent_t& e : c.ev) CU(ctx, cudaEventCreate(&e));
    float ms = 0.f, part = 0.f;
    uint32_t k = 0;
    int rc = text_chunks(ctx, R, label, text, n_bytes, z != nullptr, reads_chunk, &c, &ms, &k);
    if (rc) return rc;
    // text_chunks ended with the stream synchronised: c.host holds the totals behind the last chunk
    const unsigned long long n_lines = R.w[W_BASES + k], n_reads = c.host[0], blob = c.host[1];
    const uint32_t n = (uint32_t) (n_reads < c.cap ? n_reads : c.cap);
    const NamesLayout L = names_layout(n, blob);
    CU(ctx, R.names.reserve(L.bytes));
    char* b = R.names.as<char>();
    if (blob) CU(ctx, cudaMemcpyAsync(b, c.blob.p, blob, cudaMemcpyDeviceToDevice, s));
    unsigned long long* rw = c.rw.as<unsigned long long>();
    CU(ctx, cudaEventRecord(c.ev[0], s));
    if (n) {
        k_reads_finish<<<grid_for(n, 256, kNumSMs * 8), 256, 0, s>>>(c.view(), n, (unsigned long long*) (b + L.o_end),
                                                                     (uint32_t*) (b + L.o_len), rw, R.words.as<unsigned long long>());
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
    }
    CU(ctx, cudaEventRecord(c.ev[1], s));
    unsigned long long err = ~0ull, counts[RW_RUN];
    CU(ctx, cudaMemcpyAsync(&err, R.words.as<unsigned long long>() + W_ERR, 8, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaMemcpyAsync(counts, rw, sizeof counts, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    CU(ctx, cudaEventElapsedTime(&part, c.ev[0], c.ev[1]));
    ms += part;
    if (fastq && n_lines % 4) {
        const unsigned long long t = reads_err(n_lines / 4 * 4, 1, kRdTruncated);
        err = t < err ? t : err;
    }
    if (err != ~0ull)
        return fail(ctx, RALA_B200_ERR_ARG, "%s line %llu, column %u: %s", label, (err >> 30) + 1, (uint32_t) (err >> 4) & 0x3FFFFFFu,
                    reads_error_text((uint32_t) err & 15u));
    R.max_len = (uint32_t) counts[RW_MAX_LEN];
    rc = names_table(ctx, R, n, blob, c.ev[0], c.ev[1]);
    if (rc) return rc;
    CU(ctx, cudaEventElapsedTime(&part, c.ev[0], c.ev[1]));
    ms += part;
    st->format = fastq ? 2 : 1;
    st->n_reads = n;
    st->n_lines = n_lines;
    st->n_bases = counts[RW_BASES];
    st->name_bytes = blob;
    st->max_len = R.max_len;
    st->n_described = (uint32_t) counts[RW_DESCRIBED];
    st->n_chunks = k;
    st->device_ms = ms;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_set_reads_text(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_reads_stats_t* stats) {
    if (!g || (n_bytes && !text)) return RALA_B200_ERR_ARG;
    rala_b200_reads_stats_t st;
    const int rc = reads_text(g, text, n_bytes, &st);
    if (stats && !rc) *stats = st;
    return rc;
}

extern "C" int rala_b200_graph_set_reads_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_reads_stats_t* stats,
                                               rala_b200_bgzf_stats_t* bgzf) {
    if (!g || (n && !data)) return RALA_B200_ERR_ARG;
    rala_b200_reads_stats_t st;
    rala_b200_bgzf_stats_t z{};
    const Packed p{&z, nullptr};
    const int rc = reads_text(g, (const char*) data, n, &st, &p);
    if (stats && !rc) *stats = st;
    if (bgzf && !rc) *bgzf = z;
    return rc;
}

extern "C" int rala_b200_graph_set_reads_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_reads_stats_t* stats,
                                               rala_b200_gzip_stats_t* gzip) {
    if (!g || (n && !data)) return RALA_B200_ERR_ARG;
    rala_b200_reads_stats_t st;
    rala_b200_gzip_stats_t z{};
    const Packed p{nullptr, &z};
    const int rc = reads_text(g, (const char*) data, n, &st, &p);
    if (stats && !rc) *stats = st;
    if (gzip && !rc) *gzip = z;
    return rc;
}

extern "C" int rala_b200_graph_get_reads(rala_b200_graph* g, char* names_out, uint64_t* name_end_out, uint32_t* read_len_out,
                                         uint32_t* n_reads, uint64_t* name_bytes) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (!g->paf || !g->paf->have_names) return fail(ctx, RALA_B200_ERR_STATE, "get_reads: set_reads or set_reads_text first");
    const PafReader& R = *g->paf;
    if (n_reads) *n_reads = R.n_reads;
    if (name_bytes) *name_bytes = R.name_bytes;
    const NamesLayout L = names_layout(R.n_reads, R.name_bytes);
    const char* b = R.names.as<char>();
    cudaStream_t s = ctx->L.stream;
    CU(ctx, cudaSetDevice(ctx->device));
    if (names_out && R.name_bytes) CU(ctx, cudaMemcpyAsync(names_out, b, R.name_bytes, cudaMemcpyDeviceToHost, s));
    if (name_end_out && R.n_reads) CU(ctx, cudaMemcpyAsync(name_end_out, b + L.o_end, (size_t) R.n_reads * 8, cudaMemcpyDeviceToHost, s));
    if (read_len_out && R.n_reads) CU(ctx, cudaMemcpyAsync(read_len_out, b + L.o_len, (size_t) R.n_reads * 4, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return RALA_B200_OK;
}
