// piles.cu — the coverage half of Graph::initialize on the device (SURVEY.md 8(f) row 1, second half): per-read coverage
// from the overlap records (store_overlap_bounds + Pile::add_layers, graph.cpp:305-321, pile.cpp:274-297), the valid region
// and pile liveness (find_valid_region, pile.cpp:307, 329) and the median (find_median).  No per-base counter is ever
// materialised (one uint16 per base is 8 GB at configs[2]): the kernels work on interval events.
//
//   k_pile_events     4 events per counted record, key = read << pbits | position << 1 | kind (0 begin, 1 end);
//                     per-read event counts; the refusals (smallest offending record wins)
//   k_radix_hist,     LSD radix sort of the keys, 8 bits per pass over the significant bits only; ranks inside a tile
//   k_radix_scatter   come from per-warp digit counters (match.any), tile offsets from a digit-major scan
//   k_pile_walk       one warp per read over its sorted events: constant-coverage runs (maximal: a run starts where the
//                     coverage changes), the longest run of positions with coverage >= 4, then the median by a binary
//                     search on the value over the region's runs
//
// The rule, restated (not pinned where marked): every record whose two names resolved counts, also those the duplicate
// filter drops; it adds [a_begin + 15, a_end - 15) to read a and [b_begin + 15, b_end - 15) to read b, forward-strand
// coordinates as parsed; the valid region is the longest maximal run with coverage >= 4 (ties: the first one wins — not
// pinned), dead if shorter than 1 260 (a run of exactly 1 260 lives — not pinned); the median is element size / 2 of the
// sorted coverage over the region (nth_element).  Refused (not pinned, so not guessed): self overlaps, intervals that are
// empty or inverted after the shrink, coordinates beyond the read length, coverage >= 65 536 (Pile keeps uint16).
#include <algorithm>

#include "kernels.h"
#include "session.h"

namespace rb {

constexpr int kRadixItems = 8;                                  // keys per thread and tile
constexpr uint32_t kRadixTile = kTileThreads * kRadixItems;     // 2048 keys; warp w holds [w * 256, (w + 1) * 256)
constexpr uint32_t kMinRegion = 1260;
constexpr uint32_t kMinCoverage = 4;
constexpr uint32_t kShrink = 15;
enum : uint32_t { kErrId = 1, kErrSelf, kErrAEmpty, kErrABeyond, kErrBEmpty, kErrBBeyond };
// device words of one build: W_ERR starts at ~0 (a minimum), the rest at 0
enum { PW_ERR = 0, PW_COUNTED, PW_RUNS, PW_MAXCOV, PW_LIVE, PW_TIED, PW_EXACT, PW_WORDS };

struct PileOut {
    uint2* piles;
    uint16_t* median;
    uint32_t* n_runs;        // per read (n_reads + 1 words: the last stays 0 for the scan)
    uint32_t* run_begin;     // runs of read r at slots [seg_off[r] + r, ...)
    uint16_t* run_cov;
};

__device__ __forceinline__ uint32_t lanemask_lt() { return (1u << lane_id()) - 1u; }

__global__ void __launch_bounds__(256) k_pile_events(PileCols in, uint32_t n, const uint32_t* __restrict__ read_len, uint32_t n_reads,
                                                     uint32_t pbits, unsigned long long* __restrict__ keys, uint32_t* __restrict__ seg_cnt,
                                                     unsigned long long* __restrict__ words) {
    for (uint32_t k0 = blockIdx.x * blockDim.x; k0 < n; k0 += gridDim.x * blockDim.x) {
        const uint32_t i = k0 + threadIdx.x;
        bool counted = false;
        ulonglong2 lo = make_ulonglong2(~0ull, ~0ull), hi = lo;   // all ones in the read field: behind every read
        if (i < n && !(in.a[i] & kInvalidBit)) {
            const uint32_t a = in.a[i], b = in.b[i] & 0x7FFFFFFFu;
            const unsigned long long ab = in.ab[i], ae = in.ae[i], bb = in.bb[i], be = in.be[i];
            uint32_t err = 0;
            if (a >= n_reads || b >= n_reads) err = kErrId;
            else if (a == b) err = kErrSelf;
            else if (ab + 2 * kShrink >= ae) err = kErrAEmpty;
            else if (ae > __ldg(read_len + a)) err = kErrABeyond;
            else if (bb + 2 * kShrink >= be) err = kErrBEmpty;
            else if (be > __ldg(read_len + b)) err = kErrBBeyond;
            if (err) {
                atomicMin(words + PW_ERR, (unsigned long long) i << 8 | err);
            } else {
                counted = true;
                const unsigned long long ka = (unsigned long long) a << pbits, kb = (unsigned long long) b << pbits;
                lo = make_ulonglong2(ka | (ab + kShrink) << 1, ka | (ae - kShrink) << 1 | 1ull);
                hi = make_ulonglong2(kb | (bb + kShrink) << 1, kb | (be - kShrink) << 1 | 1ull);
                atomicAdd(seg_cnt + a, 2u);
                atomicAdd(seg_cnt + b, 2u);
            }
        }
        if (i < n) {
            reinterpret_cast<ulonglong2*>(keys)[2ull * i] = lo;
            reinterpret_cast<ulonglong2*>(keys)[2ull * i + 1] = hi;
        }
        const uint32_t c = __popc(__ballot_sync(0xFFFFFFFFu, counted));
        if (lane_id() == 0 && c) atomicAdd(words + PW_COUNTED, (unsigned long long) c);
    }
}

// digit histogram of one tile per block, stored digit-major (counts[d * n_tiles + tile]) so that one exclusive scan gives
// every (digit, tile) its output offset
__global__ void __launch_bounds__(kTileThreads) k_radix_hist(const unsigned long long* __restrict__ keys, uint32_t n, uint32_t shift,
                                                            uint32_t* __restrict__ counts, uint32_t n_tiles) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * kRadixTile;
#pragma unroll
    for (int r = 0; r < kRadixItems; ++r) {
        const uint32_t idx = base + r * kTileThreads + threadIdx.x;
        if (idx < n) atomicAdd(&h[(uint32_t) (keys[idx] >> shift) & 255u], 1u);
    }
    __syncthreads();
    counts[(size_t) threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}

// Stable scatter of one tile.  Warp w ranks its 256 keys in 8 rounds of 32 (index order = round, lane): peers with the same
// digit come from match.any, the running per-warp digit counter gives the base.  Then thread d turns the 8 warp counters of
// digit d into offsets behind the tile's scanned offset.
__global__ void __launch_bounds__(kTileThreads) k_radix_scatter(const unsigned long long* __restrict__ in, unsigned long long* __restrict__ out,
                                                               uint32_t n, uint32_t shift, const uint32_t* __restrict__ offs, uint32_t n_tiles) {
    __shared__ uint32_t cnt[kTileWarps][256];
    for (uint32_t j = threadIdx.x; j < kTileWarps * 256; j += kTileThreads) (&cnt[0][0])[j] = 0;
    __syncthreads();
    const uint32_t lane = lane_id(), warp = warp_id();
    const uint32_t base = blockIdx.x * kRadixTile + warp * (32u * kRadixItems);
    unsigned long long k[kRadixItems];
    uint32_t off[kRadixItems];
#pragma unroll
    for (int r = 0; r < kRadixItems; ++r) {
        const uint32_t idx = base + r * 32u + lane;
        const bool valid = idx < n;
        k[r] = valid ? in[idx] : 0ull;
        const uint32_t d = valid ? (uint32_t) (k[r] >> shift) & 255u : 256u + lane;   // a key past the end ranks alone
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
        const uint32_t prev = valid ? cnt[warp][d] : 0u;
        __syncwarp();
        const uint32_t rank = __popc(peers & lanemask_lt());
        if (valid && rank == 0) cnt[warp][d] = prev + __popc(peers);
        __syncwarp();
        off[r] = prev + rank;
    }
    __syncthreads();
    {
        uint32_t run = offs[(size_t) threadIdx.x * n_tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < kTileWarps; ++w) {
            const uint32_t c = cnt[w][threadIdx.x];
            cnt[w][threadIdx.x] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kRadixItems; ++r)
        if (base + r * 32u + lane < n) out[cnt[warp][(uint32_t) (k[r] >> shift) & 255u] + off[r]] = k[r];
}

// One warp per read over its sorted events, 32 at a time.  A boundary is the last event of a position; the coverage after
// it holds from that position on, and a run starts there when it differs from the coverage after the previous boundary.
// Run starts with coverage >= 4 after one below 4 open a region, the reverse closes it (the last run always has coverage 0).
__global__ void __launch_bounds__(256) k_pile_walk(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ seg_off,
                                                   const uint32_t* __restrict__ read_len, uint32_t n_reads, uint32_t pbits, PileOut o,
                                                   unsigned long long* __restrict__ words) {
    const uint32_t lane = lane_id(), lt = lanemask_lt();
    const unsigned long long pmask = (1ull << pbits) - 1ull;
    uint32_t live = 0, tied = 0, exact = 0, maxc_all = 0;
    unsigned long long runs_all = 0;
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_reads; r += (gridDim.x * blockDim.x) >> 5) {
        const uint32_t s = seg_off[r], e = seg_off[r + 1], len = read_len[r];
        uint32_t* rb = o.run_begin + (size_t) s + r;
        uint16_t* rc = o.run_cov + (size_t) s + r;
        uint32_t n_runs = 0;
        if (len) {
            if (lane == 0) { rb[0] = 0; rc[0] = 0; }
            n_runs = 1;
        }
        int cov = 0;               // after the last event seen
        int bcov = 0;              // after the last boundary seen = coverage of the current run
        uint32_t open_pos = 0, open_run = 0;   // start (position, run index) of the region being read
        uint32_t best_len = 0, best_b = 0, best_e = 0, best_rb = 0, best_re = 0, n_best = 0, maxc = 0;
        for (uint32_t c0 = s; c0 < e; c0 += 32) {
            const uint32_t i = c0 + lane;
            const bool valid = i < e;
            const unsigned long long k = valid ? keys[i] : 0ull;
            const uint32_t pos = valid ? (uint32_t) ((k & pmask) >> 1) : 0xFFFFFFFFu;
            uint32_t npos = __shfl_down_sync(0xFFFFFFFFu, pos, 1);
            if (lane == 31) npos = i + 1 < e ? (uint32_t) ((keys[i + 1] & pmask) >> 1) : 0xFFFFFFFFu;
            const uint32_t delta = valid ? ((k & 1ull) ? 0xFFFFFFFFu : 1u) : 0u;
            const int after = cov + (int) warp_inclusive_scan(delta);
            const bool boundary = valid && npos != pos;
            const uint32_t bm = __ballot_sync(0xFFFFFFFFu, boundary);
            const uint32_t lb = bm & lt;
            const int pc = __shfl_sync(0xFFFFFFFFu, after, lb ? 31 - __clz(lb) : lane);
            const int prev = lb ? pc : bcov;
            const bool is_run = boundary && after != prev;
            const uint32_t rm = __ballot_sync(0xFFFFFFFFu, is_run);
            const uint32_t run_idx = n_runs + __popc(rm & lt);
            if (is_run) {
                rb[run_idx] = pos;
                rc[run_idx] = (uint16_t) after;   // >= 65 536 refuses the whole build
            }
            const bool up = is_run && after >= (int) kMinCoverage && prev < (int) kMinCoverage;
            const bool down = is_run && after < (int) kMinCoverage && prev >= (int) kMinCoverage;
            const uint32_t um = __ballot_sync(0xFFFFFFFFu, up), dm = __ballot_sync(0xFFFFFFFFu, down);
            const uint32_t lu = um & lt, src = lu ? 31 - __clz(lu) : lane;
            const uint32_t upos = __shfl_sync(0xFFFFFFFFu, pos, src), urun = __shfl_sync(0xFFFFFFFFu, run_idx, src);
            const uint32_t rstart = lu ? upos : open_pos, rrun = lu ? urun : open_run;
            const uint32_t rlen = down ? pos - rstart : 0u;
            const uint32_t m = __reduce_max_sync(0xFFFFFFFFu, rlen);
            if (m) {
                const uint32_t eq = __ballot_sync(0xFFFFFFFFu, down && rlen == m), f = __ffs(eq) - 1;
                const uint32_t fb = __shfl_sync(0xFFFFFFFFu, rstart, f), fe = __shfl_sync(0xFFFFFFFFu, pos, f);
                const uint32_t frb = __shfl_sync(0xFFFFFFFFu, rrun, f), fre = __shfl_sync(0xFFFFFFFFu, run_idx, f);
                if (m > best_len) {   // strict: the first longest run wins
                    best_len = m; best_b = fb; best_e = fe; best_rb = frb; best_re = fre; n_best = __popc(eq);
                } else if (m == best_len) {
                    n_best += __popc(eq);
                }
            }
            if (um | dm) {
                const uint32_t t = 31 - __clz(um | dm);
                const uint32_t tp = __shfl_sync(0xFFFFFFFFu, pos, t), tr = __shfl_sync(0xFFFFFFFFu, run_idx, t);
                if ((um >> t) & 1u) { open_pos = tp; open_run = tr; }
            }
            if (bm) bcov = __shfl_sync(0xFFFFFFFFu, after, 31 - __clz(bm));
            maxc = max(maxc, __reduce_max_sync(0xFFFFFFFFu, boundary ? (uint32_t) after : 0u));
            n_runs += __popc(rm);
            cov = __shfl_sync(0xFFFFFFFFu, after, 31);
        }
        __syncwarp();   // the runs this warp wrote are read back by every lane below
        const bool alive = best_len >= kMinRegion;
        uint32_t med = 0;
        if (alive) {
            // smallest v with #{x in [b, e) : cov(x) <= v} > size / 2: element size / 2 of the sorted values
            const uint32_t kth = best_len / 2;
            uint32_t lo = kMinCoverage, hi = min(maxc, 65535u);
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                uint32_t w = 0;
                for (uint32_t j = best_rb + lane; j < best_re; j += 32)
                    if (rc[j] <= mid) w += rb[j + 1] - rb[j];
                w = __reduce_add_sync(0xFFFFFFFFu, w);
                if (w > kth) hi = mid; else lo = mid + 1;
            }
            med = lo;
        }
        if (lane == 0) {
            o.piles[r] = alive ? make_uint2(best_b, best_e) : make_uint2(0u, 0u);
            o.median[r] = (uint16_t) med;
            o.n_runs[r] = n_runs;
        }
        live += alive;
        tied += alive && n_best > 1;
        exact += alive && best_len == kMinRegion;
        maxc_all = max(maxc_all, maxc);
        runs_all += n_runs;
    }
    if (lane == 0) {
        if (runs_all) atomicAdd(words + PW_RUNS, runs_all);
        if (maxc_all) atomicMax(words + PW_MAXCOV, (unsigned long long) maxc_all);
        if (live) atomicAdd(words + PW_LIVE, (unsigned long long) live);
        if (tied) atomicAdd(words + PW_TIED, (unsigned long long) tied);
        if (exact) atomicAdd(words + PW_EXACT, (unsigned long long) exact);
    }
}

// the padded runs of every read moved to run_off[r] (one warp per read)
__global__ void __launch_bounds__(256) k_pile_runs_compact(const uint32_t* __restrict__ seg_off, const uint32_t* __restrict__ run_off,
                                                           uint32_t n_reads, const uint32_t* __restrict__ src_begin,
                                                           const uint16_t* __restrict__ src_cov, uint32_t* __restrict__ dst_begin,
                                                           uint16_t* __restrict__ dst_cov) {
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_reads; r += (gridDim.x * blockDim.x) >> 5) {
        const size_t from = (size_t) seg_off[r] + r, to = run_off[r];
        const uint32_t cnt = run_off[r + 1] - run_off[r];
        for (uint32_t j = lane_id(); j < cnt; j += 32) {
            dst_begin[to + j] = src_begin[from + j];
            dst_cov[to + j] = src_cov[from + j];
        }
    }
}

void preload_piles() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_pile_events);
    cudaFuncGetAttributes(&a, k_radix_hist);
    cudaFuncGetAttributes(&a, k_radix_scatter);
    cudaFuncGetAttributes(&a, k_pile_walk);
    cudaFuncGetAttributes(&a, k_pile_runs_compact);
}

}  // namespace rb

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct PileBuilder {
    DevBuf cols, rlen;           // stateless form: the uploaded columns and read lengths
    DevBuf keys[2], counts, scan, seg, words, nruns, run_begin, run_cov, piles, medians;
    uint32_t n_reads = 0;
    uint64_t n_runs = 0;
    const uint32_t* seg_off = nullptr;   // into seg: event offset of every read (its runs sit at seg_off[r] + r)
    bool ready = false;          // the session's runs and medians belong to its current records
    cudaEvent_t ev[2]{};
    ~PileBuilder() {
        DevBuf* bufs[] = {&cols, &rlen, &keys[0], &keys[1], &counts, &scan, &seg, &words, &nruns, &run_begin, &run_cov, &piles, &medians};
        for (DevBuf* b : bufs) b->release();
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
    }
};

void destroy_pile_builder(PileBuilder* p) { delete p; }

static uint32_t bits_for(uint64_t v) {   // smallest b with v < 2^b
    uint32_t b = 0;
    while (b < 64 && (v >> b)) ++b;
    return b;
}

static const char* pile_error_text(uint32_t kind) {
    switch (kind) {
        case kErrId: return "a read id is not below the number of reads";
        case kErrSelf: return "is a self overlap (a_id == b_id)";
        case kErrAEmpty: return "a_begin + 15 >= a_end - 15: the interval on read a is empty or inverted";
        case kErrABeyond: return "a_end is beyond the length of read a";
        case kErrBEmpty: return "b_begin + 15 >= b_end - 15: the interval on read b is empty or inverted";
        default: return "b_end is beyond the length of read b";
    }
}

// in: device columns of n records; read_len: device, n_reads words.  Leaves P.piles / P.medians / the runs filled.
// line_label ("PAF", "MHAP"; nullable): name a refused record by its 1-based line of that text instead of its 0-based index.
static int build_piles_device(rala_b200_ctx* ctx, PileBuilder& P, PileCols in, uint64_t n, const uint32_t* read_len, uint32_t n_reads,
                              uint32_t max_len, const char* line_label, rala_b200_pile_stats_t* st, float* device_ms) {
    P.ready = false;
    if (n >= (1ull << 29)) return fail(ctx, RALA_B200_ERR_LIMIT, "build_piles: too many overlap records (%llu >= 2^29: 4 events each)", (unsigned long long) n);
    if (n_reads >= (1u << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "build_piles: too many reads (%u >= 2^31)", n_reads);
    if (max_len >= (1u << 30)) return fail(ctx, RALA_B200_ERR_LIMIT, "build_piles: a read is %u long: read lengths must be < 2^30", max_len);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->L.stream;
    const uint32_t n_keys = (uint32_t) (4 * n);
    const uint32_t pbits = bits_for(2ull * max_len + 1), kbits = bits_for(n_reads) + pbits;
    const uint32_t passes = (kbits + 7) / 8, n_tiles = (n_keys + kRadixTile - 1) / kRadixTile;
    const uint64_t scan_n = std::max<uint64_t>((uint64_t) 256 * n_tiles, (uint64_t) n_reads + 1);
    const size_t scan_words = tiles_of(scan_n) + 2;
    const size_t seg_words = align_up((size_t) n_reads + 4, 64);
    CU(ctx, P.keys[0].reserve((size_t) n_keys * 8 + 256));
    CU(ctx, P.keys[1].reserve((size_t) n_keys * 8 + 256));
    const size_t cnt_col = align_up((size_t) 256 * n_tiles * 4 + 16, 256);
    CU(ctx, P.counts.reserve(2 * cnt_col));
    CU(ctx, P.scan.reserve(scan_words * 8));
    CU(ctx, P.seg.reserve(2 * seg_words * 4));
    CU(ctx, P.nruns.reserve(seg_words * 4));
    CU(ctx, P.words.reserve(PW_WORDS * 8));
    CU(ctx, P.run_begin.reserve(((size_t) n_keys + n_reads + 1) * 4));
    CU(ctx, P.run_cov.reserve(((size_t) n_keys + n_reads + 1) * 2));
    CU(ctx, P.piles.reserve((size_t) n_reads * 8 + 16));
    CU(ctx, P.medians.reserve((size_t) n_reads * 2 + 16));
    for (cudaEvent_t& e : P.ev)
        if (!e) CU(ctx, cudaEventCreate(&e));
    unsigned long long* words = P.words.as<unsigned long long>();
    unsigned long long* scan = P.scan.as<unsigned long long>();
    uint32_t *seg_cnt = P.seg.as<uint32_t>(), *seg = seg_cnt + seg_words;   // events per read -> their offsets
    uint32_t *cnt = P.counts.as<uint32_t>(), *offs = (uint32_t*) (P.counts.as<char>() + cnt_col);
    CU(ctx, cudaMemsetAsync(words, 0xFF, 8, s));
    CU(ctx, cudaMemsetAsync(words + 1, 0, 8 * (PW_WORDS - 1), s));
    CU(ctx, cudaMemsetAsync(seg_cnt, 0, seg_words * 4, s));
    CU(ctx, cudaMemsetAsync(P.nruns.p, 0, seg_words * 4, s));
    CU(ctx, cudaEventRecord(P.ev[0], s));
    if (n) {
        k_pile_events<<<grid_for(n, 256, kNumSMs * 16), 256, 0, s>>>(in, (uint32_t) n, read_len, n_reads, pbits, P.keys[0].as<unsigned long long>(),
                                                                     seg_cnt, words);
        ctx->L.count++;
    }
    CU(ctx, cudaMemsetAsync(scan, 0, scan_words * 8, s));
    launch_scan_u32(ctx->L, seg_cnt, seg, n_reads + 1, scan + 1, (uint32_t*) scan);
    for (uint32_t p = 0; p < passes && n_keys; ++p) {
        const unsigned long long* src = P.keys[p & 1].as<unsigned long long>();
        unsigned long long* dst = P.keys[(p + 1) & 1].as<unsigned long long>();
        k_radix_hist<<<n_tiles, kTileThreads, 0, s>>>(src, n_keys, 8 * p, cnt, n_tiles);
        ctx->L.count++;
        CU(ctx, cudaMemsetAsync(scan, 0, scan_words * 8, s));
        launch_scan_u32(ctx->L, cnt, offs, 256 * n_tiles, scan + 1, (uint32_t*) scan);
        k_radix_scatter<<<n_tiles, kTileThreads, 0, s>>>(src, dst, n_keys, 8 * p, offs, n_tiles);
        ctx->L.count++;
    }
    const unsigned long long* sorted = P.keys[passes & 1].as<unsigned long long>();
    PileOut o{P.piles.as<uint2>(), P.medians.as<uint16_t>(), P.nruns.as<uint32_t>(), P.run_begin.as<uint32_t>(), P.run_cov.as<uint16_t>()};
    if (n_reads) {
        k_pile_walk<<<grid_for(n_reads, kTileWarps, kNumSMs * 16), 256, 0, s>>>(sorted, seg, read_len, n_reads, pbits, o, words);
        ctx->L.count++;
    }
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaEventRecord(P.ev[1], s));
    unsigned long long w[PW_WORDS];
    CU(ctx, cudaMemcpyAsync(w, words, sizeof(w), cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    if (device_ms) CU(ctx, cudaEventElapsedTime(device_ms, P.ev[0], P.ev[1]));
    if (w[PW_ERR] != ~0ull) {
        const unsigned long long rec = w[PW_ERR] >> 8;
        const uint32_t kind = (uint32_t) (w[PW_ERR] & 0xFF);
        if (line_label) return fail(ctx, RALA_B200_ERR_ARG, "build_piles: %s line %llu %s", line_label, rec + 1, pile_error_text(kind));
        return fail(ctx, RALA_B200_ERR_ARG, "build_piles: record %llu (0-based) %s", rec, pile_error_text(kind));
    }
    if (w[PW_MAXCOV] >= 65536)
        return fail(ctx, RALA_B200_ERR_LIMIT, "build_piles: coverage %llu >= 65536 (the reference's Pile keeps it in 16 bits)", w[PW_MAXCOV]);
    rala_b200_pile_stats_t t{};
    t.n_counted = w[PW_COUNTED];
    t.n_runs = w[PW_RUNS];
    t.max_coverage = (uint32_t) w[PW_MAXCOV];
    t.n_live = (uint32_t) w[PW_LIVE];
    t.n_tied = (uint32_t) w[PW_TIED];
    t.n_exact_min = (uint32_t) w[PW_EXACT];
    if (st) *st = t;
    P.n_reads = n_reads;
    P.n_runs = t.n_runs;
    P.seg_off = seg;
    P.ready = true;
    return RALA_B200_OK;
}

extern "C" int rala_b200_build_piles(rala_b200_ctx* ctx, const uint32_t* a_id, const uint32_t* b_id, const uint32_t* a_begin,
                                     const uint32_t* a_end, const uint32_t* b_begin, const uint32_t* b_end, uint64_t n,
                                     const uint32_t* read_len, uint32_t n_reads, rala_pile_t* piles_out, uint16_t* medians_out,
                                     rala_b200_pile_stats_t* stats, float* device_ms) {
    if (!ctx || (n && (!a_id || !b_id || !a_begin || !a_end || !b_begin || !b_end)) || (n_reads && (!read_len || !piles_out)))
        return RALA_B200_ERR_ARG;
    if (device_ms) *device_ms = 0.f;
    if (n >= (1ull << 29)) return fail(ctx, RALA_B200_ERR_LIMIT, "build_piles: too many overlap records (%llu >= 2^29: 4 events each)", (unsigned long long) n);   // before the upload
    uint32_t max_len = 0;
    for (uint32_t i = 0; i < n_reads; ++i) max_len = std::max(max_len, read_len[i]);
    CU(ctx, cudaSetDevice(ctx->device));
    PileBuilder P;
    const size_t col = align_up((size_t) n * 4 + 4, 256);
    CU(ctx, P.cols.reserve(6 * col));
    CU(ctx, P.rlen.reserve((size_t) n_reads * 4 + 16));
    cudaStream_t s = ctx->L.stream;
    char* b = P.cols.as<char>();
    const uint32_t* src[6] = {a_id, b_id, a_begin, a_end, b_begin, b_end};
    for (int k = 0; k < 6 && n; ++k) CU(ctx, cudaMemcpyAsync(b + k * col, src[k], (size_t) n * 4, cudaMemcpyHostToDevice, s));
    if (n_reads) CU(ctx, cudaMemcpyAsync(P.rlen.p, read_len, (size_t) n_reads * 4, cudaMemcpyHostToDevice, s));
    const PileCols in{(const uint32_t*) b, (const uint32_t*) (b + col), (const uint32_t*) (b + 2 * col), (const uint32_t*) (b + 3 * col),
                      (const uint32_t*) (b + 4 * col), (const uint32_t*) (b + 5 * col)};
    int rc = build_piles_device(ctx, P, in, n, P.rlen.as<uint32_t>(), n_reads, max_len, nullptr, stats, device_ms);
    if (rc) return rc;
    if (n_reads) CU(ctx, cudaMemcpyAsync(piles_out, P.piles.p, (size_t) n_reads * 8, cudaMemcpyDeviceToHost, s));
    if (n_reads && medians_out) CU(ctx, cudaMemcpyAsync(medians_out, P.medians.p, (size_t) n_reads * 2, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_build_piles(rala_b200_graph* g, rala_b200_pile_stats_t* stats) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    PileCols in;
    const uint32_t* read_len = nullptr;
    uint32_t n_reads = 0, max_len = 0;
    const TextFormat fmt = text_records_view(g, &in, &read_len, &n_reads, &max_len);
    if (fmt == kTextNone)
        return fail(ctx, RALA_B200_ERR_STATE, "build_piles: needs the records of a successful set_overlaps_paf or _mhap (records "
                    "given to set_overlaps* have the duplicate filter folded in, and coverage counts the records it drops)");
    if (!g->pile_builder) g->pile_builder = new PileBuilder();
    PileBuilder& P = *g->pile_builder;
    int rc = build_piles_device(ctx, P, in, g->n_rec, read_len, n_reads, max_len, fmt == kTextMhap ? "MHAP" : "PAF", stats, nullptr);
    if (rc) return rc;
    std::vector<rala_pile_t> piles(n_reads);
    if (n_reads) CU(ctx, cudaMemcpyAsync(piles.data(), P.piles.p, (size_t) n_reads * 8, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    rc = rala_b200_graph_set_piles(g, piles.data(), nullptr, n_reads);
    if (rc) {
        P.ready = false;
        return rc;
    }
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_medians(rala_b200_graph* g, uint16_t* out) {
    if (!g) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (!g->pile_builder || !g->pile_builder->ready) return fail(ctx, RALA_B200_ERR_STATE, "get_medians: build_piles first");
    PileBuilder& P = *g->pile_builder;
    if (P.n_reads && !out) return RALA_B200_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    if (P.n_reads) CU(ctx, cudaMemcpyAsync(out, P.medians.p, (size_t) P.n_reads * 2, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_get_coverage_runs(rala_b200_graph* g, uint32_t* run_off, uint32_t* run_begin, uint16_t* run_cov, uint64_t cap) {
    if (!g || !run_off) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    if (!g->pile_builder || !g->pile_builder->ready) return fail(ctx, RALA_B200_ERR_STATE, "get_coverage_runs: build_piles first");
    PileBuilder& P = *g->pile_builder;
    if ((run_begin || run_cov) && (!run_begin || !run_cov || cap < P.n_runs))
        return fail(ctx, RALA_B200_ERR_ARG, "get_coverage_runs: %llu runs, the output holds %llu", (unsigned long long) P.n_runs,
                    (unsigned long long) cap);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->L.stream;
    const uint32_t n_reads = P.n_reads;
    DevBuf off, dst, scan;   // run counts -> offsets, compacted runs, look-back words
    const size_t off_words = align_up((size_t) n_reads + 4, 64), scan_words = tiles_of((uint64_t) n_reads + 1) + 2;
    const size_t col = align_up((size_t) P.n_runs * 4 + 4, 256);
    auto done = [&](int rc) {
        off.release(); dst.release(); scan.release();
        return rc;
    };
#define CUR(call)                                                                                                        \
    do {                                                                                                                 \
        cudaError_t err__ = (call);                                                                                      \
        if (err__ != cudaSuccess)                                                                                        \
            return done(fail(ctx, RALA_B200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__)); \
    } while (0)
    CUR(off.reserve(off_words * 4));
    CUR(scan.reserve(scan_words * 8));
    CUR(cudaMemcpyAsync(off.p, P.nruns.p, off_words * 4, cudaMemcpyDeviceToDevice, s));
    CUR(cudaMemsetAsync(scan.p, 0, scan_words * 8, s));
    launch_scan_u32(ctx->L, off.as<uint32_t>(), off.as<uint32_t>(), n_reads + 1, scan.as<unsigned long long>() + 1, scan.as<uint32_t>());
    if (run_begin && P.n_runs) {
        CUR(dst.reserve(col + (size_t) P.n_runs * 2 + 256));
        k_pile_runs_compact<<<grid_for(n_reads, kTileWarps, kNumSMs * 16), 256, 0, s>>>(P.seg_off, off.as<uint32_t>(), n_reads,
                                                                                       P.run_begin.as<uint32_t>(), P.run_cov.as<uint16_t>(),
                                                                                       dst.as<uint32_t>(), (uint16_t*) (dst.as<char>() + col));
        ctx->L.count++;
        CUR(cudaGetLastError());
        CUR(cudaMemcpyAsync(run_begin, dst.p, (size_t) P.n_runs * 4, cudaMemcpyDeviceToHost, s));
        CUR(cudaMemcpyAsync(run_cov, dst.as<char>() + col, (size_t) P.n_runs * 2, cudaMemcpyDeviceToHost, s));
    }
    CUR(cudaMemcpyAsync(run_off, off.p, ((size_t) n_reads + 1) * 4, cudaMemcpyDeviceToHost, s));
    CUR(cudaStreamSynchronize(s));
#undef CUR
    return done(RALA_B200_OK);
}
