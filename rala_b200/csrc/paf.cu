// paf.cu — PAF or MHAP text in host memory -> the graph session's device-resident records (SURVEY.md 8(f) row 2): the
// parse of bioparser's PafParser / MhapParser (graph.cpp:443-451 runs it once more for every construct pass) and, for PAF,
// the name -> id lookup of Overlap::transmute (overlap.cpp:36-82) on the device, followed by the front end's duplicate
// filter (frontend.cu).
//
//   names once per session:  k_paf_names        open-addressing table of the read names (64-bit hash; a hit is confirmed
//                                                against the name bytes, so a hash collision never resolves to a wrong id)
//   per upload chunk:        k_paf_line_ends    '\n' per tile (16-byte loads), decoupled look-back, one line end per record
//                            k_paf_parse        one warp per line: tab positions by ballot, lane f parses field f
//                         or k_mhap_parse       the same for MHAP: spaces, numeric ids checked against the read count
//   per call (session):      k_filter_duplicates, k_paf_fold   is_valid_overlap_ folded into the INVALID bit
// The upload and line scan (text_chunks) and the name table (names_table) also serve the FASTA / FASTQ reader (reads.cu).
//
// Input contracts (the library refuses what it cannot map onto the reference's reading without guessing; the full text
// is in include/rala_b200.h).  PAF: tab-separated, at least 12 fields; columns 2, 3, 4, 7, 8, 9, 11 plain decimal below
// 2^32; orientation = first byte of column 5 != '+'; names are the exact bytes of columns 1 and 6; columns 10, 12 and
// every extra column are never read.  MHAP: space-separated, at least 12 fields; ids 1..n_reads; strands 0 or 1; fields
// 3, 4 and every extra field are never read.
#include <cstring>

#include "kernels.h"
#include "session.h"

namespace rb {

constexpr uint32_t kPafChunk = RALA_B200_PAF_CHUNK_BYTES;
constexpr int kScanItems = 4;                                          // 16-byte loads per thread and tile
constexpr uint32_t kScanTile = kTileThreads * 16u * kScanItems;        // 16 KiB of text per tile
constexpr uint32_t kPafPad = kScanTile + 256;                          // readable bytes behind a chunk (whole tiles, line words)
constexpr uint32_t kUnknownId = 0x7FFFFFFFu;                           // a name that is not in the table
constexpr uint32_t kMinPafLine = 19;                                   // 11 tabs + 7 digits + '\n': no valid line is shorter
constexpr uint32_t kMinMhapLine = 22;                                  // 11 spaces + 10 digits + '\n' (fields 3, 4 empty)
enum : uint32_t { kErrFields = 1, kErrEmpty = 2, kErrDigit = 3, kErrOverflow = 4, kErrReadId = 5, kErrStrand = 6 };
__device__ __forceinline__ unsigned long long name_hash(const uint8_t* p, uint32_t n) {
    unsigned long long h = 0xcbf29ce484222325ull;   // FNV-1a, then the murmur3 finaliser for the slot bits
    for (uint32_t i = 0; i < n; ++i) h = (h ^ p[i]) * 0x100000001b3ull;
    h ^= h >> 33; h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33; h *= 0xc4ceb9fe1a85ec53ull;
    return h ^ (h >> 33);
}

__device__ __forceinline__ bool same_bytes(const uint8_t* a, const uint8_t* b, uint32_t n) {
    for (uint32_t i = 0; i < n; ++i)
        if (a[i] != b[i]) return false;
    return true;
}

__device__ __forceinline__ uint32_t name_lookup(const NameTable& t, const uint8_t* p, uint32_t n) {
    const unsigned long long h = name_hash(p, n);
    const uint32_t tag = (uint32_t) (h >> 32);
    for (uint32_t s = (uint32_t) h & t.mask;; s = (s + 1) & t.mask) {   // the table is at most half full
        const unsigned long long e = __ldg(t.slots + s);
        if (e == ~0ull) return kUnknownId;
        if ((uint32_t) (e >> 32) == tag) {
            const uint32_t id = (uint32_t) e;
            const unsigned long long b0 = id ? __ldg(t.end + id - 1) : 0ull, b1 = __ldg(t.end + id);
            if (b1 - b0 == n && same_bytes(t.blob + b0, p, n)) return id;
        }
    }
}

// One thread per read name.  Two equal names take the same probe sequence, so whichever claims a slot first is seen by
// the other: every duplicate is found, and the smallest (later id, earlier id) pair is reported.
__global__ void __launch_bounds__(256) k_paf_names(NameTable t, uint32_t n, unsigned long long* __restrict__ dup) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long b0 = i ? t.end[i - 1] : 0ull;
        const uint32_t len = (uint32_t) (t.end[i] - b0);
        const unsigned long long h = name_hash(t.blob + b0, len);
        const unsigned long long mine = (h >> 32 << 32) | i;
        for (uint32_t s = (uint32_t) h & t.mask;; s = (s + 1) & t.mask) {
            const unsigned long long old = atomicCAS(t.slots + s, ~0ull, mine);
            if (old == ~0ull) break;
            if ((old >> 32) != (h >> 32)) continue;
            const uint32_t id = (uint32_t) old;
            const unsigned long long c0 = id ? t.end[id - 1] : 0ull;
            if (t.end[id] - c0 == len && same_bytes(t.blob + c0, t.blob + b0, len)) {
                atomicMin(dup, (unsigned long long) max(i, id) << 32 | min(i, id));
                break;
            }
        }
    }
}

// '\n' positions of one chunk in order.  Item r of thread t covers bytes [r * 4096 + t * 16, +16) of the tile (a warp
// reads 512 contiguous bytes per load); the 32 (item, warp) counts are scanned by one warp, the tile prefix comes from
// the decoupled look-back of common.cuh.  The last tile writes the running line count behind this chunk.
__global__ void __launch_bounds__(kTileThreads) k_paf_line_ends(const uint8_t* __restrict__ text, uint32_t len,
                                                               uint32_t* __restrict__ line_end, unsigned long long* __restrict__ status,
                                                               uint32_t* __restrict__ ticket, unsigned long long* __restrict__ bases,
                                                               uint32_t chunk) {
    static_assert(kScanItems * kTileWarps == 32, "one warp scans the partial counts");
    __shared__ uint32_t s_cnt[kScanItems * kTileWarps];
    __shared__ uint32_t s_tile;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t num_tiles = (len + kScanTile - 1) / kScanTile;
    while (true) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= num_tiles) break;
        uint32_t nl[kScanItems], pre[kScanItems];
#pragma unroll
        for (int r = 0; r < kScanItems; ++r) {
            const uint32_t off = tile * kScanTile + r * (kTileThreads * 16u) + tid * 16u;
            const uint4 q = *reinterpret_cast<const uint4*>(text + off);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
            uint32_t m = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t x = w[j] ^ 0x0A0A0A0Au;   // zero byte <=> '\n' (exact per byte: no borrow between bytes)
                const uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
                m |= (((z >> 7) & 1u) | ((z >> 14) & 2u) | ((z >> 21) & 4u) | ((z >> 28) & 8u)) << (4 * j);
            }
            if (off + 16u > len) m &= off < len ? (1u << (len - off)) - 1u : 0u;
            nl[r] = m;
            const uint32_t c = __popc(m), inc = warp_inclusive_scan(c);
            pre[r] = inc - c;
            if (lane == 31) s_cnt[r * kTileWarps + warp] = inc;
        }
        __syncthreads();
        if (warp == 0) {
            const uint32_t c = s_cnt[lane], inc = warp_inclusive_scan(c);
            const uint32_t total = __shfl_sync(0xFFFFFFFFu, inc, 31);
            const unsigned long long excl = lookback_exclusive(status, tile, total);
            s_cnt[lane] = (uint32_t) excl + inc - c;
            if (tile == num_tiles - 1 && lane == 0) bases[chunk + 1] = bases[chunk] + excl + total;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kScanItems; ++r) {
            const uint32_t off = tile * kScanTile + r * (kTileThreads * 16u) + tid * 16u;
            uint32_t pos = s_cnt[r * kTileWarps + warp] + pre[r], m = nl[r];
            while (m) {
                line_end[pos++] = off + (uint32_t) (__ffs(m) - 1);
                m &= m - 1;
            }
        }
        __syncthreads();
    }
}

// The first `kWant` separators of line [s, e) into pos[] by one warp, 128 bytes per step (a 4-byte word per lane): found
// by ballot, ranked by a warp scan.  Returns how many there are, at most kWant; the walk stops once it has them, so bytes
// behind them (PAF tags, CIGARs of tens of KB; MHAP extra fields) are never read.
template <uint32_t kSep, uint32_t kWant>
__device__ __forceinline__ uint32_t warp_separators(const uint8_t* __restrict__ text, uint32_t s, uint32_t e, uint32_t* pos,
                                                    uint32_t lane) {
    uint32_t n = 0;
    for (uint32_t w = s & ~3u; w < e && n < kWant; w += 128u) {
        const uint32_t p0 = w + 4u * lane;
        const uint32_t word = *reinterpret_cast<const uint32_t*>(text + p0);
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            m |= ((((word >> (8 * k)) & 0xFFu) == kSep) & (p0 + k >= s) & (p0 + k < e) ? 1u : 0u) << k;
        const uint32_t c = __popc(m), inc = warp_inclusive_scan(c);
        for (uint32_t r = n + inc - c; m && r < kWant; ++r, m &= m - 1) pos[r] = p0 + (uint32_t) (__ffs(m) - 1);
        n += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    return n < kWant ? n : kWant;
}

// Plain decimal [fb, fe) below 2^32 (leading zeros allowed).  A refusal sets err = kind << 4 | field: an empty field or a
// non-digit (kErrDigit), or the 33rd bit (kErrOverflow), whichever comes first from the left.
__device__ __forceinline__ uint32_t parse_u32(const uint8_t* __restrict__ text, uint32_t fb, uint32_t fe, uint32_t field, uint32_t& err) {
    unsigned long long v = 0;
    if (fb == fe) err = kErrDigit << 4 | field;
    for (uint32_t p = fb; p < fe; ++p) {
        const uint32_t d = (uint32_t) text[p] - '0';
        if (d > 9u) { err = kErrDigit << 4 | field; break; }
        v = v * 10u + d;
        if (v > 0xFFFFFFFFull) { err = kErrOverflow << 4 | field; break; }
    }
    return (uint32_t) v;
}

// One warp per line: tab positions by warp_separators, stopping at the 11th tab, then lane f parses field f.
// Record index = global line index (file order).  A refused line lowers the error word: (line << 8) | kind << 4 | column.
__global__ void __launch_bounds__(256) k_paf_parse(const uint8_t* __restrict__ text, const uint32_t* __restrict__ line_end,
                                                   const unsigned long long* __restrict__ bases, uint32_t chunk, NameTable t,
                                                   PafCols out, unsigned long long rec_cap, unsigned long long* __restrict__ words) {
    __shared__ uint32_t s_tab[kTileWarps][11];
    const unsigned long long base = bases[chunk];
    const uint32_t n_lines = (uint32_t) (bases[chunk + 1] - base);
    const uint32_t lane = lane_id(), warp = warp_id();
    for (uint32_t line = blockIdx.x * kTileWarps + warp; line < n_lines; line += gridDim.x * kTileWarps) {
        const uint32_t s = line ? line_end[line - 1] + 1u : 0u, e = line_end[line];
        __syncwarp();
        const uint32_t ntab = warp_separators<'\t', 11>(text, s, e, s_tab[warp], lane);
        __syncwarp();
        uint32_t err = 0, val = 0;
        if (e == s) {
            err = kErrEmpty << 4 | 1u;
        } else if (ntab < 11u) {
            err = kErrFields << 4 | (ntab + 1u);   // fields found
        } else if (lane < 11u) {
            const uint32_t fb = lane ? s_tab[warp][lane - 1] + 1u : s, fe = s_tab[warp][lane];
            if (lane == 0 || lane == 5) {
                val = name_lookup(t, text + fb, fe - fb);
            } else if (lane == 4) {
                val = text[fb] != '+';   // fb == fe: the tab itself
            } else if (lane != 9) {
                val = parse_u32(text, fb, fe, lane + 1u, err);
            }
        }
        const unsigned long long gline = base + line;
        const uint32_t bad = __ballot_sync(0xFFFFFFFFu, err != 0u);
        if (bad) {
            const uint32_t code = __shfl_sync(0xFFFFFFFFu, err, __ffs(bad) - 1);
            if (lane == 0) atomicMin(words + W_ERR, gline << 8 | code);
            continue;
        }
        const uint32_t a = __shfl_sync(0xFFFFFFFFu, val, 0), a_len = __shfl_sync(0xFFFFFFFFu, val, 1);
        const uint32_t ab = __shfl_sync(0xFFFFFFFFu, val, 2), ae = __shfl_sync(0xFFFFFFFFu, val, 3);
        const uint32_t ori = __shfl_sync(0xFFFFFFFFu, val, 4), b = __shfl_sync(0xFFFFFFFFu, val, 5);
        const uint32_t b_len = __shfl_sync(0xFFFFFFFFu, val, 6), bb = __shfl_sync(0xFFFFFFFFu, val, 7);
        const uint32_t be = __shfl_sync(0xFFFFFFFFu, val, 8), length = __shfl_sync(0xFFFFFFFFu, val, 10);
        if (lane == 0) {
            const bool ka = a != kUnknownId, kb = b != kUnknownId;
            const bool mism = (ka && a_len != __ldg(t.read_len + a)) || (kb && b_len != __ldg(t.read_len + b));
            if (!(ka && kb)) atomicAdd(words + W_UNRESOLVED, 1ull);
            if (mism) {
                atomicAdd(words + W_MISMATCH, 1ull);
                atomicMin(words + W_FIRST_MISMATCH, gline);
            }
            if (gline < rec_cap) {
                out.a[gline] = a | (ka && kb ? 0u : kInvalidBit);
                out.b[gline] = b | ori << 31;
                out.ab[gline] = ab;
                out.ae[gline] = ae;
                out.bb[gline] = bb;
                out.be[gline] = be;
                out.len[gline] = length;
                out.mismatch[gline] = mism ? 1 : 0;
            }
        }
    }
}

// MHAP: one warp per line, spaces by warp_separators up to the 12th, then lane f parses field f + 1 (lanes 2 and 3, the
// error and the shared minmers, stay idle).  Ids are 1-based, checked against [1, n_reads]; strands are exactly '0' or '1';
// orientation = a_rc != b_rc; Overlap::length() = max(a_end - a_begin, b_end - b_begin) in uint32_t arithmetic, as the
// reference's MHAP constructor computes it.  A '\r' that ends field 12 at the line's end is dropped (CRLF files).
__global__ void __launch_bounds__(256) k_mhap_parse(const uint8_t* __restrict__ text, const uint32_t* __restrict__ line_end,
                                                    const unsigned long long* __restrict__ bases, uint32_t chunk,
                                                    const uint32_t* __restrict__ read_len, uint32_t n_reads, PafCols out,
                                                    unsigned long long rec_cap, unsigned long long* __restrict__ words) {
    __shared__ uint32_t s_sep[kTileWarps][12];
    const unsigned long long base = bases[chunk];
    const uint32_t n_lines = (uint32_t) (bases[chunk + 1] - base);
    const uint32_t lane = lane_id(), warp = warp_id();
    for (uint32_t line = blockIdx.x * kTileWarps + warp; line < n_lines; line += gridDim.x * kTileWarps) {
        const uint32_t s = line ? line_end[line - 1] + 1u : 0u, e = line_end[line];
        __syncwarp();
        const uint32_t nsep = warp_separators<' ', 12>(text, s, e, s_sep[warp], lane);
        __syncwarp();
        uint32_t err = 0, val = 0;
        if (e == s) {
            err = kErrEmpty << 4 | 1u;
        } else if (nsep < 11u) {
            err = kErrFields << 4 | (nsep + 1u);   // fields found
        } else if (lane < 12u && (lane < 2u || lane > 3u)) {
            const uint32_t fb = lane ? s_sep[warp][lane - 1] + 1u : s;
            uint32_t fe = lane < nsep ? s_sep[warp][lane] : e;
            if (lane == 11u && nsep == 11u && fe > fb && text[fe - 1] == '\r') --fe;
            if (lane == 4u || lane == 8u) {
                const uint32_t d = (uint32_t) text[fb] - '0';   // fb == fe: the separator itself
                if (fe - fb != 1u || d > 1u) err = kErrStrand << 4 | (lane + 1u);
                val = d;
            } else {
                val = parse_u32(text, fb, fe, lane + 1u, err);
                if (lane < 2u && !err) {
                    if (val == 0u || val > n_reads) err = kErrReadId << 4 | (lane + 1u);
                    val -= 1u;
                }
            }
        }
        const unsigned long long gline = base + line;
        const uint32_t bad = __ballot_sync(0xFFFFFFFFu, err != 0u);
        if (bad) {
            const uint32_t code = __shfl_sync(0xFFFFFFFFu, err, __ffs(bad) - 1);
            if (lane == 0) atomicMin(words + W_ERR, gline << 8 | code);
            continue;
        }
        const uint32_t a = __shfl_sync(0xFFFFFFFFu, val, 0), b = __shfl_sync(0xFFFFFFFFu, val, 1);
        const uint32_t a_rc = __shfl_sync(0xFFFFFFFFu, val, 4), ab = __shfl_sync(0xFFFFFFFFu, val, 5);
        const uint32_t ae = __shfl_sync(0xFFFFFFFFu, val, 6), a_len = __shfl_sync(0xFFFFFFFFu, val, 7);
        const uint32_t b_rc = __shfl_sync(0xFFFFFFFFu, val, 8), bb = __shfl_sync(0xFFFFFFFFu, val, 9);
        const uint32_t be = __shfl_sync(0xFFFFFFFFu, val, 10), b_len = __shfl_sync(0xFFFFFFFFu, val, 11);
        if (lane == 0) {
            const bool mism = a_len != __ldg(read_len + a) || b_len != __ldg(read_len + b);
            if (a_rc) atomicAdd(words + W_QUERY_RC, 1ull);
            if (mism) {
                atomicAdd(words + W_MISMATCH, 1ull);
                atomicMin(words + W_FIRST_MISMATCH, gline);
            }
            if (gline < rec_cap) {
                out.a[gline] = a;
                out.b[gline] = b | (a_rc ^ b_rc) << 31;
                out.ab[gline] = ab;
                out.ae[gline] = ae;
                out.bb[gline] = bb;
                out.be[gline] = be;
                out.len[gline] = max(ae - ab, be - bb);
                out.mismatch[gline] = mism ? 1 : 0;
            }
        }
    }
}

// is_valid_overlap_ into the INVALID bit while the parsed columns move to the session's records; a record that stays
// valid with a read length the caller's reads contradict lowers W_FIRST_BAD (transmute would exit on it)
__global__ void __launch_bounds__(256) k_paf_fold(PafCols in, const uint8_t* __restrict__ valid, uint32_t n, List recs,
                                                  unsigned long long* __restrict__ words) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const bool v = valid[i] != 0;
        recs.a[i] = in.a[i] | (v ? 0u : kInvalidBit);
        recs.b[i] = in.b[i];
        recs.ab[i] = in.ab[i];
        recs.ae[i] = in.ae[i];
        recs.bb[i] = in.bb[i];
        recs.be[i] = in.be[i];
        if (v && in.mismatch[i]) atomicMin(words + W_FIRST_BAD, (unsigned long long) i);
    }
}

void preload_paf() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_paf_names);
    cudaFuncGetAttributes(&a, k_paf_line_ends);
    cudaFuncGetAttributes(&a, k_paf_parse);
    cudaFuncGetAttributes(&a, k_mhap_parse);
    cudaFuncGetAttributes(&a, k_paf_fold);
}

}  // namespace rb

// ---------------------------------------------------------------------------------------------
// host side: the name table, the chunked upload and the call's bookkeeping
// ---------------------------------------------------------------------------------------------
void destroy_paf_reader(PafReader* r) { delete r; }

NamesLayout names_layout(uint32_t n_reads, uint64_t blob) {
    NamesLayout L;
    L.slots = 1024;
    while (L.slots < 2ull * n_reads) L.slots <<= 1;
    L.o_end = align_up(blob + 1, 256);
    L.o_len = L.o_end + align_up((size_t) n_reads * 8 + 8, 256);
    L.o_slots = L.o_len + align_up((size_t) n_reads * 4 + 4, 256);
    L.bytes = L.o_slots + (size_t) L.slots * 8;
    return L;
}

int names_table(rala_b200_ctx* ctx, PafReader& R, uint32_t n_reads, uint64_t blob, cudaEvent_t ev0, cudaEvent_t ev1) {
    const NamesLayout L = names_layout(n_reads, blob);
    CU(ctx, R.words.reserve(256));
    char* b = R.names.as<char>();
    cudaStream_t s = ctx->L.stream;
    CU(ctx, cudaMemsetAsync(b + L.o_slots, 0xFF, (size_t) L.slots * 8, s));
    CU(ctx, cudaMemsetAsync(R.words.p, 0xFF, 8 * (W_DUP + 1), s));
    R.table = NameTable{(const uint8_t*) b, (const unsigned long long*) (b + L.o_end), (const uint32_t*) (b + L.o_len),
                        (unsigned long long*) (b + L.o_slots), L.slots - 1};
    if (ev0) CU(ctx, cudaEventRecord(ev0, s));
    if (n_reads) {
        k_paf_names<<<grid_for(n_reads, 256, kNumSMs * 8), 256, 0, s>>>(R.table, n_reads, R.words.as<unsigned long long>() + W_DUP);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
    }
    if (ev1) CU(ctx, cudaEventRecord(ev1, s));
    unsigned long long dup = ~0ull;
    CU(ctx, cudaMemcpyAsync(&dup, R.words.as<unsigned long long>() + W_DUP, 8, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    if (dup != ~0ull)
        return fail(ctx, RALA_B200_ERR_ARG, "set_reads: reads %u and %u have the same name (which one name_to_id_ keeps is not pinned)",
                    (unsigned) dup, (unsigned) (dup >> 32));
    R.n_reads = n_reads;
    R.name_bytes = blob;
    R.have_names = true;
    return RALA_B200_OK;
}

static int paf_set_names(rala_b200_ctx* ctx, PafReader& R, const char* names, const uint64_t* name_end, const uint32_t* read_len,
                         uint32_t n_reads) {
    R.have_names = false;
    if (n_reads && (!name_end || !read_len)) return fail(ctx, RALA_B200_ERR_ARG, "set_reads: name ends and read lengths are needed");
    if (n_reads >= (1u << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many reads (%u >= 2^31)", n_reads);
    uint64_t prev = 0;
    for (uint32_t i = 0; i < n_reads; ++i) {
        if (name_end[i] < prev || name_end[i] - prev >= (1ull << 32))
            return fail(ctx, RALA_B200_ERR_ARG, "set_reads: name %u ends at %llu, before its start %llu (or is 4 GiB long)", i,
                        (unsigned long long) name_end[i], (unsigned long long) prev);
        prev = name_end[i];
    }
    const uint64_t blob = n_reads ? name_end[n_reads - 1] : 0;
    if (blob && !names) return fail(ctx, RALA_B200_ERR_ARG, "set_reads: names are missing");
    const NamesLayout L = names_layout(n_reads, blob);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, R.names.reserve(L.bytes));
    char* b = R.names.as<char>();
    cudaStream_t s = ctx->L.stream;
    if (blob) CU(ctx, cudaMemcpyAsync(b, names, blob, cudaMemcpyHostToDevice, s));
    if (n_reads) {
        CU(ctx, cudaMemcpyAsync(b + L.o_end, name_end, (size_t) n_reads * 8, cudaMemcpyHostToDevice, s));
        CU(ctx, cudaMemcpyAsync(b + L.o_len, read_len, (size_t) n_reads * 4, cudaMemcpyHostToDevice, s));
    }
    R.max_len = 0;
    for (uint32_t i = 0; i < n_reads; ++i) R.max_len = read_len[i] > R.max_len ? read_len[i] : R.max_len;
    return names_table(ctx, R, n_reads, blob);
}

static const char* text_error_text(uint32_t kind) {
    switch (kind) {
        case kErrDigit: return "is not a plain decimal number";
        case kErrOverflow: return "does not fit 32 bits";
        case kErrReadId: return "is not a read id (1 to the number of reads given to set_reads)";
        default: return "is not a strand (exactly 0 or 1)";
    }
}

// What one call of either reader counted (the union of the PAF and the MHAP stats).
struct TextStats {
    uint64_t n_records, n_unresolved, n_length_mismatch, first_length_mismatch, n_query_rc, n_bytes, n_chunks;
};

uint64_t text_max_chunks(uint64_t n_bytes) { return n_bytes ? 2 * (n_bytes / kPafChunk) + 2 : 0; }   // two consecutive chunks span >= one chunk size
size_t text_status_words() { return tiles_of((uint64_t) kPafChunk + 1) + 1; }

static int text_chunks_once(rala_b200_ctx* ctx, PafReader& R, const char* label, const char* text, uint64_t n_bytes, bool on_device,
                            ChunkKernels kernels, void* self, float* kernel_ms, uint32_t* n_chunks) {
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->L.stream;
    const uint64_t max_chunks = text_max_chunks(n_bytes);
    CU(ctx, R.words.reserve((W_BASES + max_chunks + 2) * 8));
    CU(ctx, R.line_end.reserve(((size_t) kPafChunk + 2) * 4));
    const size_t status_words = text_status_words();
    CU(ctx, R.status.reserve(status_words * 8));
    for (int k = 0; k < 2; ++k) {
        CU(ctx, R.text[k].reserve((size_t) kPafChunk + 1 + kPafPad));
        if (!R.copied[k]) CU(ctx, cudaEventCreateWithFlags(&R.copied[k], cudaEventDisableTiming));
        if (!R.parsed[k]) CU(ctx, cudaEventCreateWithFlags(&R.parsed[k], cudaEventDisableTiming));
    }
    if (!R.copy) CU(ctx, cudaStreamCreateWithFlags(&R.copy, cudaStreamNonBlocking));
    while (R.timing.size() < 2 * max_chunks) {
        cudaEvent_t e;
        CU(ctx, cudaEventCreate(&e));
        R.timing.push_back(e);
    }
    // caller memory that is page-locked is uploaded in place; anything else goes through the pinned staging pair
    bool direct = false;
    if (n_bytes && !on_device) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, text) == cudaSuccess) direct = attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
    }
    for (int k = 0; !direct && !on_device && n_bytes && k < 2; ++k)
        if (!R.pinned[k]) CU(ctx, cudaHostAlloc((void**) &R.pinned[k], kPafChunk + 1, cudaHostAllocDefault));
    unsigned long long* words = R.words.as<unsigned long long>();
    CU(ctx, cudaMemsetAsync(words, 0xFF, 8 * W_UNRESOLVED, s));
    CU(ctx, cudaMemsetAsync(words + W_UNRESOLVED, 0, 8 * (W_BASES + 1 - W_UNRESOLVED), s));
    char tail = '\n';   // the text's last byte
    if (n_bytes && on_device) CU(ctx, cudaMemcpyAsync(&tail, text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));   // the copy stream starts from settled words and buffers
    if (n_bytes && !on_device) tail = text[n_bytes - 1];
    uint64_t pos = 0;
    uint32_t k = 0;
    for (; pos < n_bytes; ++k) {
        if (k >= max_chunks) return fail(ctx, RALA_B200_ERR_LIMIT, "%s text: more upload chunks than planned", label);
        uint64_t len = n_bytes - pos < kPafChunk ? n_bytes - pos : kPafChunk;
        const bool last = pos + len == n_bytes;
        if (!last) {   // cut behind the last '\n' of the window; the tail goes with the next chunk
            uint64_t cut = 0;   // bytes up to and with the last '\n' of the window, 0 when there is none
            if (on_device) {
                const int rc = inflated_cut(ctx, R, (const uint8_t*) text, pos, pos + len, &cut);
                if (rc) return rc;
                cut = cut ? cut - pos : 0;
            } else {
                const void* nl = memrchr(text + pos, '\n', len);
                cut = nl ? (uint64_t) ((const char*) nl - (text + pos)) + 1 : 0;
            }
            if (!cut) {
                unsigned long long lines = 0;
                CU(ctx, cudaStreamSynchronize(R.copy));
                CU(ctx, cudaMemcpyAsync(&lines, words + W_BASES + k, 8, cudaMemcpyDeviceToHost, s));
                CU(ctx, cudaStreamSynchronize(s));
                return fail(ctx, RALA_B200_ERR_LIMIT, "%s line %llu is longer than the upload chunk (%u bytes)", label, lines + 1, kPafChunk);
            }
            len = cut;
        }
        const int slot = k & 1;
        const char* src = text + pos;
        if (!direct && !on_device) {
            if (k >= 2) CU(ctx, cudaEventSynchronize(R.copied[slot]));   // the upload of chunk k - 2 has left the buffer
            memcpy(R.pinned[slot], src, len);
            src = R.pinned[slot];
        }
        if (k >= 2) CU(ctx, cudaStreamWaitEvent(R.copy, R.parsed[slot], 0));   // chunk k - 2 is parsed: its device buffer is free
        char* dtext = R.text[slot].as<char>();
        CU(ctx, cudaMemcpyAsync(dtext, src, len, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, R.copy));
        uint32_t scan_len = (uint32_t) len;
        if (last && tail != '\n') {   // the final line without its '\n'
            CU(ctx, cudaMemsetAsync(dtext + len, '\n', 1, R.copy));
            ++scan_len;
        }
        CU(ctx, cudaEventRecord(R.copied[slot], R.copy));
        CU(ctx, cudaStreamWaitEvent(s, R.copied[slot], 0));
        CU(ctx, cudaEventRecord(R.timing[2 * k], s));
        CU(ctx, cudaMemsetAsync(R.status.p, 0, status_words * 8, s));
        unsigned long long* st_words = R.status.as<unsigned long long>();
        k_paf_line_ends<<<grid_for(scan_len, kScanTile, kNumSMs * 8), kTileThreads, 0, s>>>(
            (const uint8_t*) dtext, scan_len, R.line_end.as<uint32_t>(), st_words + 1, (uint32_t*) st_words, words + W_BASES, k);
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
        const int rc = kernels(self, ctx, k, (const uint8_t*) dtext, scan_len);
        if (rc) return rc;
        CU(ctx, cudaEventRecord(R.timing[2 * k + 1], s));
        CU(ctx, cudaEventRecord(R.parsed[slot], s));
        pos += len;
    }
    R.w.assign(W_BASES + k + 1, 0ull);
    CU(ctx, cudaMemcpyAsync(R.w.data(), words, R.w.size() * 8, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    if (kernel_ms) {
        *kernel_ms = 0.f;
        for (uint32_t c = 0; c < k; ++c) {
            float ms = 0.f;
            CU(ctx, cudaEventElapsedTime(&ms, R.timing[2 * c], R.timing[2 * c + 1]));
            *kernel_ms += ms;
        }
    }
    *n_chunks = k;
    return RALA_B200_OK;
}

// A refused call returns with no upload in flight: the caller may free its text at once.
int text_chunks(rala_b200_ctx* ctx, PafReader& R, const char* label, const char* text, uint64_t n_bytes, bool on_device,
                ChunkKernels kernels, void* self, float* kernel_ms, uint32_t* n_chunks) {
    const int rc = text_chunks_once(ctx, R, label, text, n_bytes, on_device, kernels, self, kernel_ms, n_chunks);
    if (rc) {
        if (R.copy) cudaStreamSynchronize(R.copy);
        cudaStreamSynchronize(ctx->L.stream);
    }
    return rc;
}

// the parse kernel of one PAF or MHAP chunk (ChunkKernels)
struct OverlapChunk {
    PafReader* R;
    bool mhap;
};

static int overlap_chunk(void* self, rala_b200_ctx* ctx, uint32_t k, const uint8_t* dtext, uint32_t scan_len) {
    const OverlapChunk& c = *static_cast<const OverlapChunk*>(self);
    PafReader& R = *c.R;
    unsigned long long* words = R.words.as<unsigned long long>();
    cudaStream_t s = ctx->L.stream;
    if (c.mhap)
        k_mhap_parse<<<grid_for(scan_len, kTileWarps * 64, kNumSMs * 8), 256, 0, s>>>(
            dtext, R.line_end.as<uint32_t>(), words + W_BASES, k, R.table.read_len, R.n_reads, R.view(), R.rec_cap, words);
    else
        k_paf_parse<<<grid_for(scan_len, kTileWarps * 64, kNumSMs * 8), 256, 0, s>>>(
            dtext, R.line_end.as<uint32_t>(), words + W_BASES, k, R.table, R.view(), R.rec_cap, words);
    ctx->L.count++;
    CU(ctx, cudaGetLastError());
    return RALA_B200_OK;
}

// Parses the whole text into R.cols (record index = line index, file order).  *n_out = records; kernel_ms (nullable) = device
// time of the chunks' kernels (line scan + parse), uploads excluded.  The format decides the parse kernel, the shortest
// valid line and the wording of refusals; upload, line scan and the call's words are the same for both.
static int text_parse(rala_b200_ctx* ctx, PafReader& R, TextFormat fmt, const char* text, uint64_t n_bytes, bool on_device,
                      TextStats* st, float* kernel_ms, uint64_t* n_out) {
    CU(ctx, cudaSetDevice(ctx->device));
    const bool mhap = fmt == kTextMhap;
    const char* label = mhap ? "MHAP" : "PAF";
    const char* field = mhap ? "field" : "column";
    // no valid line is shorter than the format's minimum (the last one may lack its '\n'): more lines than that means a refusal
    R.rec_cap = (n_bytes + 1) / (mhap ? kMinMhapLine : kMinPafLine) + 1;
    if (R.rec_cap > (1ull << 31)) R.rec_cap = 1ull << 31;
    const size_t col = align_up((size_t) R.rec_cap * 4, 256);
    CU(ctx, R.cols.reserve(7 * col + align_up((size_t) R.rec_cap, 256)));
    OverlapChunk chunk{&R, mhap};
    uint32_t k = 0;
    const int rc = text_chunks(ctx, R, label, text, n_bytes, on_device, overlap_chunk, &chunk, kernel_ms, &k);
    if (rc) return rc;
    if (R.w[W_ERR] != ~0ull) {
        const uint32_t code = (uint32_t) (R.w[W_ERR] & 0xFF), kind = code >> 4, column = code & 15;
        const unsigned long long line = (R.w[W_ERR] >> 8) + 1;
        if (kind == kErrFields)
            return fail(ctx, RALA_B200_ERR_ARG, "%s line %llu has %u %s-separated fields, at least 12 are needed", label, line, column,
                        mhap ? "space" : "tab");
        if (kind == kErrEmpty) return fail(ctx, RALA_B200_ERR_ARG, "%s line %llu, %s 1: the line is empty", label, line, field);
        return fail(ctx, RALA_B200_ERR_ARG, "%s line %llu, %s %u: %s", label, line, field, column, text_error_text(kind));
    }
    const unsigned long long n = R.w[W_BASES + k];
    if (n >= (1ull << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many overlap records (%llu >= 2^31)", n);
    st->n_records = n;
    st->n_unresolved = R.w[W_UNRESOLVED];
    st->n_length_mismatch = R.w[W_MISMATCH];
    st->first_length_mismatch = R.w[W_FIRST_MISMATCH];
    st->n_query_rc = R.w[W_QUERY_RC];
    st->n_bytes = n_bytes;
    st->n_chunks = k;
    *n_out = n;
    return RALA_B200_OK;
}

extern "C" int rala_b200_graph_set_reads(rala_b200_graph* g, const char* names, const uint64_t* name_end, const uint32_t* read_len,
                                         uint32_t n_reads) {
    if (!g) return RALA_B200_ERR_ARG;
    if (!g->paf) g->paf = new PafReader();
    g->text_records = kTextNone;   // the records' ids refer to the reads they were parsed against
    return paf_set_names(g->ctx, *g->paf, names, name_end, read_len, n_reads);
}

// Text in file order -> the session's records: parse, duplicate filter, INVALID bit folded in.  *counted = *st holds the
// call's counts (also when a read-length refusal follows).
// z (nullable): text[0, n_bytes) is a BGZF or gzip file, inflated on the device first.
static int set_overlaps_text(rala_b200_graph* g, TextFormat fmt, const char* text, uint64_t n_bytes, TextStats* st, bool* counted,
                             const Packed* z = nullptr) {
    if (!g || (n_bytes && !text)) return RALA_B200_ERR_ARG;
    rala_b200_ctx* ctx = g->ctx;
    const bool mhap = fmt == kTextMhap;
    if (!g->paf || !g->paf->have_names)
        return fail(ctx, RALA_B200_ERR_STATE, "set_overlaps_%s: set_reads first", mhap ? "mhap" : "paf");
    PafReader& R = *g->paf;
    // the session's records are void until this call has succeeded
    g->n_rec = 0;
    g->state = SS_EMPTY;
    g->text_records = kTextNone;
    int rc;
    if (z) {
        rc = inflate_packed(ctx, R, (const uint8_t*) text, n_bytes, *z, &n_bytes);
        if (rc) return rc;
        text = R.inflated.as<const char>();
    }
    uint64_t n = 0;
    rc = text_parse(ctx, R, fmt, text, n_bytes, z != nullptr, st, nullptr, &n);
    if (rc) return rc;
    rc = reserve_for_records(g, n);
    if (rc) return rc;
    if (n) {
        const PafCols c = R.view();
        CU(ctx, R.valid.reserve(align_up((size_t) n, 256)));
        launch_filter_duplicates(ctx->L, c.a, c.b, c.len, (uint32_t) n, R.valid.as<uint8_t>());
        k_paf_fold<<<grid_for(n, 256, kNumSMs * 8), 256, 0, ctx->L.stream>>>(c, R.valid.as<uint8_t>(), (uint32_t) n, g->recs.view,
                                                                             R.words.as<unsigned long long>());
        ctx->L.count++;
        CU(ctx, cudaGetLastError());
    }
    unsigned long long bad = ~0ull;
    CU(ctx, cudaMemcpyAsync(&bad, R.words.as<unsigned long long>() + W_FIRST_BAD, 8, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    *counted = true;
    if (bad != ~0ull) {
        g->n_rec = 0;
        g->state = SS_EMPTY;
        return fail(ctx, RALA_B200_ERR_ARG,
                    "%s line %llu: a read length (%s) differs from the length given to set_reads, and the record is "
                    "valid after the duplicate filter (the reference's transmute exits on it)", mhap ? "MHAP" : "PAF", bad + 1,
                    mhap ? "field 8 or 12" : "column 2 or 7");
    }
    g->text_records = fmt;
    return RALA_B200_OK;
}

static void paf_stats_of(const TextStats& t, rala_b200_paf_stats_t* st) {
    *st = rala_b200_paf_stats_t{t.n_records, t.n_unresolved, t.n_length_mismatch, t.first_length_mismatch, t.n_bytes, t.n_chunks};
}

static void mhap_stats_of(const TextStats& t, rala_b200_mhap_stats_t* st) {
    *st = rala_b200_mhap_stats_t{t.n_records, t.n_length_mismatch, t.first_length_mismatch, t.n_query_rc, t.n_bytes, t.n_chunks};
}

extern "C" int rala_b200_graph_set_overlaps_paf(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_paf_stats_t* stats) {
    TextStats st{};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextPaf, text, n_bytes, &st, &counted);
    if (stats && counted) paf_stats_of(st, stats);
    return rc;
}

extern "C" int rala_b200_graph_set_overlaps_mhap(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_mhap_stats_t* stats) {
    TextStats st{};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextMhap, text, n_bytes, &st, &counted);
    if (stats && counted) mhap_stats_of(st, stats);
    return rc;
}

extern "C" int rala_b200_graph_set_overlaps_paf_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_paf_stats_t* stats,
                                                     rala_b200_bgzf_stats_t* bgzf) {
    TextStats st{};
    rala_b200_bgzf_stats_t z{};
    const Packed p{&z, nullptr};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextPaf, (const char*) data, n, &st, &counted, &p);
    if (stats && counted) paf_stats_of(st, stats);
    if (bgzf && counted) *bgzf = z;
    return rc;
}

extern "C" int rala_b200_graph_set_overlaps_paf_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_paf_stats_t* stats,
                                                     rala_b200_gzip_stats_t* gzip) {
    TextStats st{};
    rala_b200_gzip_stats_t z{};
    const Packed p{nullptr, &z};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextPaf, (const char*) data, n, &st, &counted, &p);
    if (stats && counted) paf_stats_of(st, stats);
    if (gzip && counted) *gzip = z;
    return rc;
}

extern "C" int rala_b200_graph_set_overlaps_mhap_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_mhap_stats_t* stats,
                                                      rala_b200_bgzf_stats_t* bgzf) {
    TextStats st{};
    rala_b200_bgzf_stats_t z{};
    const Packed p{&z, nullptr};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextMhap, (const char*) data, n, &st, &counted, &p);
    if (stats && counted) mhap_stats_of(st, stats);
    if (bgzf && counted) *bgzf = z;
    return rc;
}

extern "C" int rala_b200_graph_set_overlaps_mhap_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_mhap_stats_t* stats,
                                                     rala_b200_gzip_stats_t* gzip) {
    TextStats st{};
    rala_b200_gzip_stats_t z{};
    const Packed p{nullptr, &z};
    bool counted = false;
    const int rc = set_overlaps_text(g, kTextMhap, (const char*) data, n, &st, &counted, &p);
    if (stats && counted) mhap_stats_of(st, stats);
    if (gzip && counted) *gzip = z;
    return rc;
}

TextFormat text_records_view(const rala_b200_graph* g, PileCols* cols, const uint32_t** read_len, uint32_t* n_reads, uint32_t* max_len) {
    if (g->text_records == kTextNone || !g->paf || !g->paf->have_names) return kTextNone;
    const PafCols c = g->paf->view();
    *cols = PileCols{c.a, c.b, c.ab, c.ae, c.bb, c.be};
    *read_len = g->paf->table.read_len;
    *n_reads = g->paf->n_reads;
    *max_len = g->paf->max_len;
    return g->text_records;
}

// The parsed columns of R (n records) into 7 x cap host words.
static int download_columns(rala_b200_ctx* ctx, const PafReader& R, const char* what, uint64_t n, uint32_t* cols_out, uint64_t cap) {
    if (n > cap || (n && !cols_out))
        return fail(ctx, RALA_B200_ERR_ARG, "%s: the text has %llu records, the output holds %llu", what, (unsigned long long) n,
                    (unsigned long long) cap);
    const PafCols c = R.view();
    const uint32_t* src[7] = {c.a, c.b, c.ab, c.ae, c.bb, c.be, c.len};
    for (int k = 0; k < 7 && n; ++k)
        CU(ctx, cudaMemcpyAsync(cols_out + (size_t) k * cap, src[k], (size_t) n * 4, cudaMemcpyDeviceToHost, ctx->L.stream));
    CU(ctx, cudaStreamSynchronize(ctx->L.stream));
    return RALA_B200_OK;
}

extern "C" int rala_b200_parse_paf(rala_b200_ctx* ctx, const char* names, const uint64_t* name_end, const uint32_t* read_len, uint32_t n_reads,
                                   const char* text, uint64_t n_bytes, uint32_t* cols_out, uint64_t cap, rala_b200_paf_stats_t* stats,
                                   float* device_ms) {
    if (!ctx || !stats || (n_bytes && !text)) return RALA_B200_ERR_ARG;
    if (device_ms) *device_ms = 0.f;
    PafReader R;
    int rc = paf_set_names(ctx, R, names, name_end, read_len, n_reads);
    if (rc) return rc;
    uint64_t n = 0;
    TextStats st{};
    rc = text_parse(ctx, R, kTextPaf, text, n_bytes, false, &st, device_ms, &n);
    if (rc) return rc;
    paf_stats_of(st, stats);
    return download_columns(ctx, R, "parse_paf", n, cols_out, cap);
}

extern "C" int rala_b200_parse_mhap(rala_b200_ctx* ctx, const uint32_t* read_len, uint32_t n_reads, const char* text, uint64_t n_bytes,
                                    uint32_t* cols_out, uint64_t cap, rala_b200_mhap_stats_t* stats, float* device_ms) {
    if (!ctx || !stats || (n_bytes && !text) || (n_reads && !read_len)) return RALA_B200_ERR_ARG;
    if (device_ms) *device_ms = 0.f;
    if (n_reads >= (1u << 31)) return fail(ctx, RALA_B200_ERR_LIMIT, "too many reads (%u >= 2^31)", n_reads);
    CU(ctx, cudaSetDevice(ctx->device));
    PafReader R;   // no name table: only the lengths, which the parse checks fields 8 and 12 against
    CU(ctx, R.names.reserve((size_t) n_reads * 4 + 16));
    if (n_reads) CU(ctx, cudaMemcpyAsync(R.names.p, read_len, (size_t) n_reads * 4, cudaMemcpyHostToDevice, ctx->L.stream));
    R.table.read_len = R.names.as<uint32_t>();
    R.n_reads = n_reads;
    uint64_t n = 0;
    TextStats st{};
    int rc = text_parse(ctx, R, kTextMhap, text, n_bytes, false, &st, device_ms, &n);
    if (rc) return rc;
    mhap_stats_of(st, stats);
    return download_columns(ctx, R, "parse_mhap", n, cols_out, cap);
}
