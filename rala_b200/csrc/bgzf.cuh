// bgzf.cuh — the DEFLATE decoder (RFC 1951) of one BGZF block, written for one thread so that the same code runs on lane 0
// of the inflate warp (bgzf.cu) and in the host harness of the test suite (tests/host_bgzf.cu).  Every read of the input
// stays inside [in, in + in_len) and every write inside [out, out + out_len): a malformed stream returns a BgzfError.
//
// Codes are canonical Huffman codes: a symbol whose code is at most kFast bits long is found by one lookup of the next
// kFast stream bits (bit-reversed, every suffix filled); a longer one by the per-length walk of zlib's puff.c.
#pragma once

#include <cstdint>

#if defined(__CUDACC__)
#define BGZF_HD __host__ __device__ __forceinline__
#else
#define BGZF_HD inline
#endif

namespace bgzf {

enum BgzfError : uint32_t {
    kOk = 0,
    kPastEnd,        // the stream reads past the block's compressed bytes
    kBtype3,         // a DEFLATE block of type 3
    kStoredLen,      // a stored block whose LEN is not ~NLEN
    kCounts,         // HLIT > 286 or HDIST > 30
    kOversubscribed, // a code with more codes than its lengths allow
    kIncomplete,     // a code with fewer codes than its lengths allow (one code of length 1 is accepted, as zlib does)
    kRepeat,         // a code-length repeat with no previous length or past the lengths it fills
    kNoEob,          // the literal / length code has no end-of-block symbol
    kBadSymbol,      // a literal / length code that is not in the code, or symbol 286 / 287
    kBadDistSymbol,  // a distance code that is not in the code, or distance code 30 / 31
    kTooFar,         // a distance that reaches before the start of the block
    kLong,           // more output than ISIZE
    kShort,          // less output than ISIZE
    kTrailing,       // bytes left between the end of the DEFLATE stream and the trailer
    kCrc,            // the CRC32 of the output differs from the trailer's
    kNumErrors
};

constexpr int kFastLit = 10;    // lookup bits of the literal / length code
constexpr int kFastDist = 8;    // lookup bits of the distance code

template <int kSymbols, int kFast>
struct Code {
    uint16_t count[16];          // codes of each length
    uint16_t symbol[kSymbols];   // symbols in canonical order
    uint16_t fast[1 << kFast];   // len << 9 | symbol; 0 = longer than kFast bits or not a code
};

// per decoder: two codes and the code lengths of a dynamic header (about 3.6 KB)
struct Tables {
    Code<288, kFastLit> lit;
    Code<32, kFastDist> dist;
    uint8_t lens[320];
};

struct Bits {
    const uint8_t* in;
    uint32_t n, pos, cnt;
    uint64_t buf;

    BGZF_HD void refill() {
        while (cnt <= 56 && pos < n) {
            buf |= (uint64_t) in[pos++] << cnt;
            cnt += 8;
        }
    }
    // the next k <= 32 bits; kPastEnd when the stream has fewer
    BGZF_HD uint32_t take(uint32_t k, uint32_t& err) {
        refill();
        if (cnt < k) {
            err = kPastEnd;
            return 0;
        }
        const uint32_t v = (uint32_t) (buf & ((1ull << k) - 1));
        buf >>= k;
        cnt -= k;
        return v;
    }
};

// canonical code of lens[0, n) into c; kOk, kOversubscribed or kIncomplete
template <int kSymbols, int kFast>
BGZF_HD uint32_t build(Code<kSymbols, kFast>& c, const uint8_t* lens, uint32_t n) {
    for (int l = 0; l < 16; ++l) c.count[l] = 0;
    for (uint32_t s = 0; s < n; ++s) c.count[lens[s]]++;
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left = (left << 1) - c.count[l];
        if (left < 0) return kOversubscribed;
    }
    const uint32_t used = n - c.count[0];
    if (left > 0 && used != 0 && !(used == 1 && c.count[1] == 1)) return kIncomplete;
    uint16_t offs[16], next[16];
    offs[1] = 0;
    next[1] = 0;
    for (int l = 1; l < 15; ++l) {
        offs[l + 1] = offs[l] + c.count[l];
        next[l + 1] = (uint16_t) ((next[l] + c.count[l]) << 1);
    }
    for (int i = 0; i < (1 << kFast); ++i) c.fast[i] = 0;
    for (uint32_t s = 0; s < n; ++s) {
        const uint32_t l = lens[s];
        if (!l) continue;
        c.symbol[offs[l]++] = (uint16_t) s;
        const uint32_t code = next[l]++;
        if (l > (uint32_t) kFast) continue;
        uint32_t rev = 0;
        for (uint32_t b = 0; b < l; ++b) rev |= ((code >> b) & 1u) << (l - 1 - b);
        for (uint32_t i = rev; i < (1u << kFast); i += 1u << l) c.fast[i] = (uint16_t) (l << 9 | s);
    }
    return kOk;
}

// one symbol of c, or -1 (not a code, or the stream ends inside it: err = kPastEnd); B: Bits or another reader with
// the same refill / buf / cnt
template <int kSymbols, int kFast, class B>
BGZF_HD int decode(const Code<kSymbols, kFast>& c, B& b, uint32_t& err) {
    b.refill();
    const uint32_t e = c.fast[b.buf & ((1u << kFast) - 1)];
    uint32_t len = e >> 9;
    int sym = (int) (e & 511u);
    if (!e) {   // puff.c's walk over the lengths
        int code = 0, first = 0, index = 0;
        sym = -1;
        for (len = 1; len < 16; ++len) {
            code |= (int) ((b.buf >> (len - 1)) & 1u);
            const int count = c.count[len];
            if (code - count < first) {
                sym = c.symbol[index + (code - first)];
                break;
            }
            index += count;
            first = (first + count) << 1;
            code <<= 1;
        }
        if (sym < 0) return -1;
    }
    if (len > b.cnt) {
        err = kPastEnd;
        return -1;
    }
    b.buf >>= len;
    b.cnt -= len;
    return sym;
}

BGZF_HD uint32_t cl_order(uint32_t i) {   // the order of the code-length code lengths, 5 bits each
    const uint64_t lo = 0x022CAA324E804A30ull;   // 16 17 18 0 8 7 9 6 10 5 11 4
    const uint64_t hi = 0x00000003C2E1346Cull;   // 12 3 13 2 14 1 15
    return (uint32_t) ((i < 12 ? lo >> (5 * i) : hi >> (5 * (i - 12))) & 31u);
}

// The fixed codes of BTYPE 1 into t.lit / t.dist.
BGZF_HD void fixed_codes(Tables& t) {
    for (uint32_t s = 0; s < 288; ++s) t.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    build(t.lit, t.lens, 288);
    for (uint32_t s = 0; s < 32; ++s) t.lens[s] = 5;
    build(t.dist, t.lens, 32);
}

template <class B>
BGZF_HD uint32_t dynamic_codes(Tables& t, B& b) {
    uint32_t err = kOk;
    const uint32_t nlen = b.take(5, err) + 257, ndist = b.take(5, err) + 1, ncode = b.take(4, err) + 4;
    if (err) return err;
    if (nlen > 286 || ndist > 30) return kCounts;
    for (uint32_t i = 0; i < 19; ++i) t.lens[cl_order(i)] = i < ncode ? (uint8_t) b.take(3, err) : 0;
    if (err) return err;
    uint32_t rc = build(t.lit, t.lens, 19);
    if (rc) return rc;
    for (uint32_t i = 0; i < nlen + ndist;) {
        const int sym = decode(t.lit, b, err);
        if (err) return err;
        if (sym < 0) return kIncomplete;   // a code-length code that is not in the code
        if (sym < 16) {
            t.lens[i++] = (uint8_t) sym;
            continue;
        }
        uint32_t len = 0, rep;
        if (sym == 16) {
            if (i == 0) return kRepeat;
            len = t.lens[i - 1];
            rep = 3 + b.take(2, err);
        } else if (sym == 17) {
            rep = 3 + b.take(3, err);
        } else {
            rep = 11 + b.take(7, err);
        }
        if (err) return err;
        if (i + rep > nlen + ndist) return kRepeat;
        while (rep--) t.lens[i++] = (uint8_t) len;
    }
    if (t.lens[256] == 0) return kNoEob;
    rc = build(t.lit, t.lens, nlen);
    if (rc) return rc;
    return build(t.dist, t.lens + nlen, ndist);
}

// Raw DEFLATE in[0, in_len) -> out[0, out_len) exactly.
BGZF_HD uint32_t inflate(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, Tables& t) {
    Bits b{in, in_len, 0, 0, 0};
    uint32_t err = kOk, o = 0, last = 0;
    while (!last) {
        last = b.take(1, err);
        const uint32_t type = b.take(2, err);
        if (err) return err;
        if (type == 0) {
            const uint32_t drop = b.cnt & 7u;
            b.buf >>= drop;
            b.cnt -= drop;
            const uint32_t len = b.take(16, err), nlen = b.take(16, err);
            if (err) return err;
            if (len != (~nlen & 0xFFFFu)) return kStoredLen;
            if (len > out_len - o) return kLong;
            uint32_t k = 0;
            for (; k < len && b.cnt; ++k) {   // whole bytes still in the bit buffer, then straight from the input
                out[o++] = (uint8_t) b.buf;
                b.buf >>= 8;
                b.cnt -= 8;
            }
            if (len - k > b.n - b.pos) return kPastEnd;
            for (; k < len; ++k) out[o++] = b.in[b.pos++];
            continue;
        }
        if (type == 3) return kBtype3;
        if (type == 1) {
            fixed_codes(t);
        } else {
            const uint32_t rc = dynamic_codes(t, b);
            if (rc) return rc;
        }
        while (true) {
            const int sym = decode(t.lit, b, err);
            if (err) return err;
            if (sym < 0 || sym > 285) return kBadSymbol;
            if (sym < 256) {
                if (o == out_len) return kLong;
                out[o++] = (uint8_t) sym;
                continue;
            }
            if (sym == 256) break;
            const uint32_t s = (uint32_t) sym - 257;
            uint32_t len;
            if (s < 8) {
                len = 3 + s;
            } else if (s == 28) {
                len = 258;
            } else {
                const uint32_t x = (s - 4) >> 2;
                len = ((4u + (s & 3u)) << x) + 3u + b.take(x, err);
            }
            const int d = decode(t.dist, b, err);
            if (err) return err;
            if (d < 0 || d > 29) return kBadDistSymbol;
            uint32_t dist;
            if (d < 4) {
                dist = (uint32_t) d + 1;
            } else {
                const uint32_t x = ((uint32_t) d - 2) >> 1;
                dist = ((2u + ((uint32_t) d & 1u)) << x) + 1u + b.take(x, err);
            }
            if (err) return err;
            if (dist > o) return kTooFar;
            if (len > out_len - o) return kLong;
            const uint8_t* from = out + o - dist;
            for (uint32_t k = 0; k < len; ++k) out[o + k] = from[k];
            o += len;
        }
    }
    if (b.cnt >= 8 || b.pos != b.n) return kTrailing;   // whole bytes behind the final block
    return o == out_len ? kOk : kShort;
}

// ---- CRC32 (reflected, polynomial 0xEDB88320) and its GF(2) shift, as zlib's crc32_combine ---------------------------
constexpr uint32_t kPoly = 0xEDB88320u;

BGZF_HD uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = c & 1u ? (c >> 1) ^ kPoly : c >> 1;
    return c;
}

BGZF_HD uint32_t crc_update(uint32_t crc, const uint8_t* p, uint32_t n, const uint32_t* table) {
    crc = ~crc;
    for (uint32_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xFFu] ^ (crc >> 8);
    return ~crc;
}

// a * b modulo the polynomial (bit-reflected)
BGZF_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    while (true) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1u ? (b >> 1) ^ kPoly : b >> 1;
    }
    return p;
}

// x^(n * 2^k) modulo the polynomial; x2n[j] = x^(2^j)
BGZF_HD uint32_t x2nmodp(uint32_t n, uint32_t k, const uint32_t* x2n) {
    uint32_t p = 1u << 31;
    while (n) {
        if (n & 1u) p = multmodp(x2n[k & 31u], p);
        n >>= 1;
        ++k;
    }
    return p;
}

BGZF_HD void x2n_table(uint32_t* x2n) {
    uint32_t p = 1u << 30;   // x^1
    for (int j = 0; j < 32; ++j) {
        x2n[j] = p;
        p = multmodp(p, p);
    }
}

// CRC32 of A || B from crc(A), crc(B) and |B|
BGZF_HD uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint32_t len_b, const uint32_t* x2n) {
    return multmodp(x2nmodp(len_b, 3, x2n), crc_a) ^ crc_b;
}

#if defined(__CUDACC__)
// CRC32 of p[0, len) by the 32 lanes of a warp, one slice each, joined by the GF(2) shift; lane 0 returns it
__device__ __forceinline__ uint32_t warp_crc(const uint8_t* p, uint32_t len, uint32_t lane, const uint32_t* table, const uint32_t* x2n) {
    const uint32_t slice = (len + 31) / 32, lo = min(lane * slice, len), hi = min(lo + slice, len);
    uint32_t crc = crc_update(0, p + lo, hi - lo, table), n = hi - lo;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {   // lane 2dk absorbs lane 2dk + d: the CRC of the slices behind it
        const uint32_t c2 = __shfl_down_sync(0xFFFFFFFFu, crc, d), l2 = __shfl_down_sync(0xFFFFFFFFu, n, d);
        if ((lane & (2 * d - 1)) == 0) {
            crc = crc_combine(crc, c2, l2, x2n);
            n += l2;
        }
    }
    return crc;
}
#endif

}  // namespace bgzf
