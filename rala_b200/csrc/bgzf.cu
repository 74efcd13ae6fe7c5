// bgzf.cu — BGZF (htslib's blocked gzip) in host memory -> its inflated text in device memory, for the text readers
// (paf.cu, reads.cu) and rala_b200_inflate_bgzf.
//
// A BGZF file is a series of gzip members of at most 64 KiB of input each, whose headers carry the member's size (BSIZE,
// the `BC` extra subfield) and whose trailers carry the CRC32 and the inflated size (ISIZE).  So every block's place in
// the compressed and in the inflated text is known from the headers alone:
//   host:    the header walk (bgzf_walk), one hop per block: magic, BC, BSIZE, ISIZE, the blocks tile the input; the
//            output offsets are the exclusive scan of the ISIZEs; the inflated text is allocated once
//   device:  the compressed bytes cross PCIe in pieces of up to RALA_B200_PAF_CHUNK_BYTES on the readers' copy stream
//            (pageable input through the pinned staging pair); every kInflateRun blocks one k_bgzf_inflate launch waits
//            for the pieces it needs.  One warp per block: lane 0 decodes the DEFLATE stream (bgzf.cuh) straight into
//            the block's place in the text, then the 32 lanes take the CRC32 of 32 slices, combined by the GF(2) shift.
//            A failing block lowers the error word with block << 8 | reason: the smallest failing block is reported.
// Launching over many blocks at once matters: one 32 MiB text chunk is only about 512 blocks, 3.5 warps per SM.
#include <cstring>

#include "bgzf.cuh"
#include "kernels.h"
#include "session.h"

namespace rb {

constexpr uint32_t kInflateWarps = 8;            // warps (blocks in flight) per CTA
constexpr uint32_t kInflateRun = 16384;          // BGZF blocks per launch: about two waves of resident warps
constexpr uint32_t kMaxIsize = 65536;

constexpr uint32_t kPiece = RALA_B200_PAF_CHUNK_BYTES;   // compressed bytes per upload piece

struct BgzfBlock {
    unsigned long long at, data, out;   // offset of the block and of its DEFLATE stream in the input, of its output in the text
    uint32_t data_len, isize, crc, pad;
};

__global__ void __launch_bounds__(kInflateWarps * 32) k_bgzf_inflate(const uint8_t* __restrict__ in, const BgzfBlock* __restrict__ blocks,
                                                                     uint32_t b0, uint32_t b1, uint8_t* __restrict__ text,
                                                                     unsigned long long* __restrict__ err) {
    __shared__ uint32_t s_crc[256], s_x2n[32];
    __shared__ bgzf::Tables s_tab[kInflateWarps];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_crc[i] = bgzf::crc_table_entry(i);
    if (threadIdx.x == 0) bgzf::x2n_table(s_x2n);
    __syncthreads();
    const uint32_t lane = lane_id(), warp = warp_id();
    for (uint32_t b = b0 + blockIdx.x * kInflateWarps + warp; b < b1; b += gridDim.x * kInflateWarps) {
        const BgzfBlock B = blocks[b];
        uint8_t* out = text + B.out;
        uint32_t rc = 0;
        if (lane == 0) rc = bgzf::inflate(in + B.data, B.data_len, out, B.isize, s_tab[warp]);
        rc = __shfl_sync(0xFFFFFFFFu, rc, 0);
        __syncwarp();   // lane 0's output is visible to the warp
        if (rc == 0) {
            const uint32_t crc = bgzf::warp_crc(out, B.isize, lane, s_crc, s_x2n);
            if (lane == 0 && crc != B.crc) rc = bgzf::kCrc;
        }
        if (lane == 0 && rc) atomicMin(err, (unsigned long long) b << 8 | rc);
    }
}

// The last '\n' of text[lo, hi) as position + 1 into *found (0: none).  Blocks take 4 KiB tiles from the end and stop
// once a '\n' behind their next tile is known, so a short last line costs one tile.
__global__ void __launch_bounds__(256) k_last_newline(const uint8_t* __restrict__ text, unsigned long long lo, unsigned long long hi,
                                                      unsigned long long* __restrict__ found) {
    __shared__ unsigned long long s_found;
    for (unsigned long long t = blockIdx.x;; t += gridDim.x) {
        if (t * 4096ull >= hi - lo) break;
        const unsigned long long end = hi - t * 4096ull, beg = end - lo > 4096ull ? end - 4096ull : lo;
        if (threadIdx.x == 0) s_found = *(volatile unsigned long long*) found;
        __syncthreads();
        const bool done = s_found > end;
        __syncthreads();
        if (done) break;
        unsigned long long best = 0;
        for (unsigned long long p = beg + threadIdx.x * 16ull, q = p + 16 < end ? p + 16 : end; p < q; ++p)
            if (text[p] == '\n') best = p + 1;
        if (best) atomicMax(found, best);
    }
}

void preload_bgzf() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_bgzf_inflate);
    cudaFuncGetAttributes(&a, k_last_newline);
}

}  // namespace rb

// ---------------------------------------------------------------------------------------------
// host side: the header walk, the upload and the launches
// ---------------------------------------------------------------------------------------------
static uint32_t le16(const uint8_t* p) { return (uint32_t) p[0] | (uint32_t) p[1] << 8; }
static uint32_t le32(const uint8_t* p) { return le16(p) | le16(p + 2) << 16; }

static int walk_fail(rala_b200_ctx* ctx, int code, size_t block, uint64_t off, const char* fmt, ...) {
    char why[384];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(why, sizeof why, fmt, ap);
    va_end(ap);
    return fail(ctx, code, "BGZF block %zu (byte offset %llu): %s", block, (unsigned long long) off, why);
}

// The block table of data[0, n) and the inflated size; refuses (RALA_B200_ERR_ARG) whatever is not BGZF.
static int bgzf_walk(rala_b200_ctx* ctx, const uint8_t* data, uint64_t n, std::vector<BgzfBlock>& blocks, uint64_t* total) {
    blocks.clear();
    uint64_t off = 0, out = 0;
    while (off < n) {
        const size_t k = blocks.size();
        const uint8_t* h = data + off;
        const uint64_t left = n - off;
        if (left < 18) return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "the input ends inside the block header (%llu bytes left)", (unsigned long long) left);
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8)
            return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "not a gzip member (bytes %02x %02x %02x, 1f 8b 08 expected)", h[0], h[1], h[2]);
        const uint32_t xlen = le16(h + 10);
        if ((h[3] & 4) && 12ull + xlen + 8 > left)
            return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "the input ends inside the block header (%llu bytes left)", (unsigned long long) left);
        uint32_t bsize = 0;
        if (h[3] & 4) {
            for (uint32_t p = 12; p + 4 <= 12 + xlen;) {   // subfields SI1 SI2 SLEN data
                const uint32_t slen = le16(h + p + 2);
                if (p + 4 + slen > 12 + xlen) break;
                if (h[p] == 'B' && h[p + 1] == 'C' && slen == 2) bsize = le16(h + p + 4) + 1;
                p += 4 + slen;
            }
        }
        if (!bsize)
            return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "the gzip member has no BC extra subfield: the input is not BGZF (blocked "
                             "gzip); compress it with bgzip");
        if (h[3] != 4) return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "header flags 0x%02x (BGZF sets FEXTRA only)", h[3]);
        if (bsize < 12 + xlen + 8)
            return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "BSIZE %u is smaller than the block's header and trailer", bsize);
        if (bsize > left)
            return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "BSIZE %u reaches past the end of the input (%llu bytes left)", bsize,
                             (unsigned long long) left);
        const uint32_t crc = le32(h + bsize - 8), isize = le32(h + bsize - 4);
        if (isize > kMaxIsize) return walk_fail(ctx, RALA_B200_ERR_ARG, k, off, "ISIZE %u is above 65536", isize);
        blocks.push_back(BgzfBlock{off, off + 12 + xlen, out, bsize - 12 - xlen - 8, isize, crc, 0});
        out += isize;
        off += bsize;
    }
    *total = out;
    return RALA_B200_OK;
}

static const char* inflate_error_text(uint32_t e) {
    switch (e) {
        case bgzf::kPastEnd: return "the DEFLATE stream runs past BSIZE";
        case bgzf::kBtype3: return "a DEFLATE block of type 3 (reserved)";
        case bgzf::kStoredLen: return "a stored block whose LEN is not the complement of NLEN";
        case bgzf::kCounts: return "a dynamic block with more than 286 literal/length or 30 distance codes";
        case bgzf::kOversubscribed: return "an over-subscribed Huffman code";
        case bgzf::kIncomplete: return "an incomplete Huffman code";
        case bgzf::kRepeat: return "a code-length repeat with no previous length or past the lengths it fills";
        case bgzf::kNoEob: return "the literal/length code has no end-of-block code";
        case bgzf::kBadSymbol: return "an invalid literal/length code (not in the code, or 286 / 287)";
        case bgzf::kBadDistSymbol: return "an invalid distance code (not in the code, or 30 / 31)";
        case bgzf::kTooFar: return "a distance that reaches before the start of the block";
        case bgzf::kLong: return "the DEFLATE stream inflates to more than ISIZE bytes";
        case bgzf::kShort: return "the DEFLATE stream inflates to fewer than ISIZE bytes";
        case bgzf::kTrailing: return "bytes between the end of the DEFLATE stream and the trailer";
        default: return "the CRC32 of the inflated bytes differs from the trailer's";
    }
}

struct TimingEvents {
    std::vector<cudaEvent_t> ev;
    ~TimingEvents() {
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
    }
};

static int bgzf_inflate_once(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_bgzf_stats_t* st,
                             uint8_t* host_out, uint64_t cap) {
    CU(ctx, cudaSetDevice(ctx->device));
    std::vector<BgzfBlock> blocks;
    uint64_t total = 0;
    int rc = bgzf_walk(ctx, data, n, blocks, &total);
    if (rc) return rc;
    *st = rala_b200_bgzf_stats_t{blocks.size(), n, total, 0.f};
    if (total >> 34) return fail(ctx, RALA_B200_ERR_LIMIT, "BGZF input inflates to %llu bytes: 2^34 or more", (unsigned long long) total);
    if (host_out && total > cap)
        return fail(ctx, RALA_B200_ERR_ARG, "inflate_bgzf: the input inflates to %llu bytes, the output holds %llu",
                    (unsigned long long) total, (unsigned long long) cap);
    const size_t nb = blocks.size();
    if (total == 0) return RALA_B200_OK;   // only empty blocks: nothing to decode
    cudaStream_t s = ctx->L.stream;
    CU(ctx, R.packed.reserve(n));
    CU(ctx, R.bgzf_meta.reserve(nb * sizeof(BgzfBlock) + 8));
    CU(ctx, R.inflated.reserve(total));
    if (!R.copy) CU(ctx, cudaStreamCreateWithFlags(&R.copy, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k)
        if (!R.copied[k]) CU(ctx, cudaEventCreateWithFlags(&R.copied[k], cudaEventDisableTiming));
    bool direct = false;   // page-locked caller memory is uploaded in place, as the readers do
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, data) == cudaSuccess) direct = attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    for (int k = 0; !direct && k < 2; ++k)
        if (!R.pinned[k]) CU(ctx, cudaHostAlloc((void**) &R.pinned[k], kPiece + 1, cudaHostAllocDefault));
    BgzfBlock* meta = R.bgzf_meta.as<BgzfBlock>();
    unsigned long long* err = (unsigned long long*) (meta + nb);
    CU(ctx, cudaMemcpyAsync(meta, blocks.data(), nb * sizeof(BgzfBlock), cudaMemcpyHostToDevice, s));
    CU(ctx, cudaMemsetAsync(err, 0xFF, 8, s));
    CU(ctx, cudaStreamSynchronize(s));   // the block table has left the host vector; the copy stream starts from settled buffers
    TimingEvents T;
    uint8_t* din = R.packed.as<uint8_t>();
    size_t b = 0, launched = 0;
    for (uint32_t k = 0; b < nb; ++k) {
        const size_t first = b;   // a piece: whole blocks, at most kPiece bytes unless one block is longer
        const uint64_t lo = blocks[first].at;
        while (b < nb && (b == first || (b + 1 < nb ? blocks[b + 1].at : n) - lo <= kPiece)) ++b;
        const uint64_t hi = b < nb ? blocks[b].at : n;
        const int slot = k & 1;
        const uint8_t* src = data + lo;
        if (!direct) {
            if (k >= 2) CU(ctx, cudaEventSynchronize(R.copied[slot]));   // the upload of piece k - 2 has left the buffer
            memcpy(R.pinned[slot], src, hi - lo);
            src = (const uint8_t*) R.pinned[slot];
        }
        CU(ctx, cudaMemcpyAsync(din + lo, src, hi - lo, cudaMemcpyHostToDevice, R.copy));
        CU(ctx, cudaEventRecord(R.copied[slot], R.copy));
        if (b - launched < kInflateRun && b < nb) continue;
        CU(ctx, cudaStreamWaitEvent(s, R.copied[slot], 0));   // pieces are copied in order: this one is the last the launch needs
        cudaEvent_t e[2];
        for (cudaEvent_t& x : e) {
            CU(ctx, cudaEventCreate(&x));
            T.ev.push_back(x);
        }
        CU(ctx, cudaEventRecord(e[0], s));
        const uint32_t n_run = (uint32_t) (b - launched);
        k_bgzf_inflate<<<grid_for(n_run, kInflateWarps, kNumSMs * 8), kInflateWarps * 32, 0, s>>>(
            din, meta, (uint32_t) launched, (uint32_t) b, R.inflated.as<uint8_t>(), err);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaEventRecord(e[1], s));
        launched = b;
    }
    unsigned long long bad = ~0ull;
    CU(ctx, cudaMemcpyAsync(&bad, err, 8, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    for (size_t i = 0; i < T.ev.size(); i += 2) {
        float ms = 0.f;
        CU(ctx, cudaEventElapsedTime(&ms, T.ev[i], T.ev[i + 1]));
        st->inflate_ms += ms;
    }
    if (bad != ~0ull) {
        const size_t k = (size_t) (bad >> 8);
        return walk_fail(ctx, RALA_B200_ERR_ARG, k, blocks[k].at, "%s", inflate_error_text((uint32_t) bad & 0xFFu));
    }
    if (host_out) {
        CU(ctx, cudaMemcpyAsync(host_out, R.inflated.p, total, cudaMemcpyDeviceToHost, s));
        CU(ctx, cudaStreamSynchronize(s));
    }
    return RALA_B200_OK;
}

int bgzf_inflate(rala_b200_ctx* ctx, PafReader& R, const uint8_t* data, uint64_t n, rala_b200_bgzf_stats_t* st, uint8_t* host_out,
                 uint64_t cap) {
    const int rc = bgzf_inflate_once(ctx, R, data, n, st, host_out, cap);
    if (rc) {
        if (R.copy) cudaStreamSynchronize(R.copy);
        cudaStreamSynchronize(ctx->L.stream);
    }
    return rc;
}

int inflated_cut(rala_b200_ctx* ctx, PafReader& R, const uint8_t* text, uint64_t lo, uint64_t hi, uint64_t* found) {
    CU(ctx, R.bgzf_cut.reserve(8));
    if (!R.cut_host) CU(ctx, cudaHostAlloc((void**) &R.cut_host, 8, cudaHostAllocDefault));
    unsigned long long* d = R.bgzf_cut.as<unsigned long long>();
    CU(ctx, cudaMemsetAsync(d, 0, 8, R.copy));
    k_last_newline<<<grid_for(hi - lo, 4096, 64), 256, 0, R.copy>>>(text, lo, hi, d);
    ctx->L.count++;
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(R.cut_host, d, 8, cudaMemcpyDeviceToHost, R.copy));
    CU(ctx, cudaStreamSynchronize(R.copy));
    *found = *R.cut_host;
    return RALA_B200_OK;
}

extern "C" int rala_b200_inflate_bgzf(rala_b200_ctx* ctx, const uint8_t* data, uint64_t n, uint8_t* out, uint64_t cap,
                                      rala_b200_bgzf_stats_t* stats) {
    if (!ctx || (n && !data)) return RALA_B200_ERR_ARG;
    rala_b200_bgzf_stats_t st{};
    PafReader R;
    int rc;
    if (!out) {
        std::vector<BgzfBlock> blocks;
        uint64_t total = 0;
        rc = bgzf_walk(ctx, data, n, blocks, &total);
        st = rala_b200_bgzf_stats_t{blocks.size(), n, total, 0.f};
    } else {
        rc = bgzf_inflate(ctx, R, data, n, &st, out, cap);
    }
    if (stats && !rc) *stats = st;
    return rc;
}

bool is_bgzf(const uint8_t* data, uint64_t n) {
    std::vector<BgzfBlock> blocks;
    uint64_t total = 0;
    return bgzf_walk(nullptr, data, n, blocks, &total) == RALA_B200_OK;
}
