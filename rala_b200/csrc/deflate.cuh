// deflate.cuh — the gzip stream decoder (RFC 1952 members around RFC 1951 DEFLATE) of gzip.cu, written for one thread so
// that the same code runs on lane 0 of the decode warps and in the host harness of the test suite (tests/host_gzip.cu).
//
// decode_span decodes a stretch of a multi-member stream from a boundary to the first boundary at or after a given bit.
// Boundaries are the starts of DEFLATE blocks, the starts of member headers and the end of the input.  Counting mode
// writes nothing; symbol mode writes one 16-bit symbol per output byte: the byte itself, or 256 + (32768 - k) for a byte
// k places before the span's first output byte (a marker, resolved later against the text before the span).  Every read
// stays inside [in, in + n) and every write inside the span's [0, cap): a malformed stream returns an error code.
#pragma once

#include <cstddef>
#include <cstdint>
#include <vector>

#include "bgzf.cuh"

namespace deflate {

// reasons beyond bgzf::BgzfError (whose kPastEnd reads "the input ends inside a DEFLATE stream" here and kTooFar "a
// distance that reaches before the start of the member"; kCrc is the member's CRC32)
enum GzipError : uint32_t {
    kMagic = bgzf::kNumErrors,   // not 1f 8b
    kMethod,                     // compression method other than 8
    kFlags,                      // reserved header flag bits set
    kHeaderEnd,                  // the input ends inside a member header
    kHeaderCrc,                  // FHCRC differs from the header's CRC32
    kTrailerEnd,                 // the input ends inside a member trailer
    kAfterLast,                  // non-zero bytes after the last member that start no member
    kIsize,                      // ISIZE differs from the member's size mod 2^32
    kNumGzipErrors
};

constexpr uint32_t kWindow = 32768;

// bit reader over in[0, n) with 64-bit positions (bgzf::Bits' refill / take / buf / cnt)
struct Stream {
    const uint8_t* in;
    uint64_t n, pos;
    uint32_t cnt;
    uint64_t buf;

    BGZF_HD void refill() {
        while (cnt <= 56 && pos < n) {
            buf |= (uint64_t) in[pos++] << cnt;
            cnt += 8;
        }
    }
    BGZF_HD uint32_t take(uint32_t k, uint32_t& err) {
        refill();
        if (cnt < k) {
            err = bgzf::kPastEnd;
            return 0;
        }
        const uint32_t v = (uint32_t) (buf & ((1ull << k) - 1));
        buf >>= k;
        cnt -= k;
        return v;
    }
    BGZF_HD uint64_t bit() const { return pos * 8 - cnt; }
    BGZF_HD void seek(uint64_t b) {   // b <= 8 n
        pos = b >> 3;
        cnt = 0;
        buf = 0;
        refill();
        buf >>= b & 7;
        cnt -= (uint32_t) (b & 7);
    }
};

BGZF_HD uint32_t crc_bits(uint32_t crc, const uint8_t* p, uint64_t n) {   // CRC32 without a table (member headers)
    crc = ~crc;
    for (uint64_t i = 0; i < n; ++i) {
        crc ^= p[i];
        for (int k = 0; k < 8; ++k) crc = crc & 1u ? (crc >> 1) ^ bgzf::kPoly : crc >> 1;
    }
    return ~crc;
}

// The member header at in[h, n): its length in bytes, or 0 with err set.
BGZF_HD uint64_t member_header(const uint8_t* in, uint64_t n, uint64_t h, uint32_t& err) {
    const uint64_t left = n - h;
    const uint8_t* p = in + h;
    if ((left > 0 && p[0] != 0x1f) || (left > 1 && p[1] != 0x8b)) return err = kMagic, 0;
    if (left > 2 && p[2] != 8) return err = kMethod, 0;
    if (left > 3 && (p[3] & 0xE0)) return err = kFlags, 0;
    if (left < 10) return err = kHeaderEnd, 0;
    const uint32_t flg = p[3];
    uint64_t k = 10;
    if (flg & 4) {   // FEXTRA
        if (left < k + 2) return err = kHeaderEnd, 0;
        k += 2 + ((uint32_t) p[k] | (uint32_t) p[k + 1] << 8);
        if (k > left) return err = kHeaderEnd, 0;
    }
    for (uint32_t f = 8; f <= 16; f <<= 1) {   // FNAME, FCOMMENT: zero-terminated
        if (!(flg & f)) continue;
        while (k < left && p[k]) ++k;
        if (k == left) return err = kHeaderEnd, 0;
        ++k;
    }
    if (flg & 2) {   // FHCRC: the low 16 bits of the CRC32 of the header before it
        if (left < k + 2) return err = kHeaderEnd, 0;
        if ((crc_bits(0, p, k) & 0xFFFFu) != ((uint32_t) p[k] | (uint32_t) p[k + 1] << 8)) return err = kHeaderCrc, 0;
        k += 2;
    }
    return k;
}

// ---- the entry finder's tests ------------------------------------------------------------------------------------------
// The canonical-code rule of bgzf::build on per-length counts: oversubscribed or incomplete (except one code of length 1)
// codes are refused.
BGZF_HD bool code_ok(const uint16_t* count, uint32_t n) {
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left = (left << 1) - count[l];
        if (left < 0) return false;
    }
    const uint32_t used = n - count[0];
    return left == 0 || used == 0 || (used == 1 && count[1] == 1);
}

// A dynamic-block header at bit b that the decoder would accept: BFINAL 0, BTYPE 2, HLIT <= 29, HDIST <= 29, a complete
// code-length code, code lengths that fill exactly HLIT + HDIST + 258 entries and make valid codes, and a code for 256.
BGZF_HD bool dynamic_entry(const uint8_t* in, uint64_t n, uint64_t b) {
    Stream s{in, n, 0, 0, 0};
    s.seek(b);
    uint32_t err = 0;
    if (s.take(3, err) != 4u || err) return false;   // BFINAL 0, BTYPE 2 (bits 0 0 1, read LSB first: 0b100)
    const uint32_t nlen = s.take(5, err) + 257, ndist = s.take(5, err) + 1, ncode = s.take(4, err) + 4;
    if (err || nlen > 286 || ndist > 30) return false;
    uint8_t cl[19];
    uint16_t count[16] = {0};
    for (uint32_t i = 0; i < 19; ++i) {
        cl[bgzf::cl_order(i)] = i < ncode ? (uint8_t) s.take(3, err) : 0;
    }
    if (err) return false;
    for (uint32_t i = 0; i < 19; ++i) count[cl[i]]++;
    int left = 1;
    for (int l = 1; l < 8; ++l) {
        left = (left << 1) - count[l];
        if (left < 0) return false;
    }
    if (left != 0) return false;   // zlib writes complete code-length codes
    uint16_t offs[8], sym[19];
    offs[1] = 0;
    for (int l = 1; l < 7; ++l) offs[l + 1] = offs[l] + count[l];
    for (uint32_t i = 0; i < 19; ++i)
        if (cl[i]) sym[offs[cl[i]]++] = (uint16_t) i;
    uint16_t lc[16] = {0}, dc[16] = {0};
    uint32_t prev = 0;
    bool eob = false;
    for (uint32_t i = 0; i < nlen + ndist;) {
        int code = 0, first = 0, index = 0, v = -1;   // puff.c's walk over the code-length code
        for (int len = 1; len < 8; ++len) {
            code |= (int) s.take(1, err);
            if (err) return false;
            const int c = count[len];
            if (code - c < first) {
                v = sym[index + (code - first)];
                break;
            }
            index += c;
            first = (first + c) << 1;
            code <<= 1;
        }
        if (v < 0) return false;
        uint32_t len = 0, rep = 1;
        if (v < 16) {
            len = (uint32_t) v;
        } else if (v == 16) {
            if (i == 0) return false;
            len = prev;
            rep = 3 + s.take(2, err);
        } else {
            rep = v == 17 ? 3 + s.take(3, err) : 11 + s.take(7, err);
        }
        if (err || i + rep > nlen + ndist) return false;
        for (; rep; --rep, ++i) {
            if (i < nlen) {
                lc[len]++;
                if (i == 256) eob = len != 0;
            } else {
                dc[len]++;
            }
        }
        prev = len;
    }
    return eob && code_ok(lc, nlen) && code_ok(dc, ndist);
}

// A stored block at byte-aligned bit b: the byte holds BFINAL 0, BTYPE 0 and zero padding, then LEN = ~NLEN.
BGZF_HD bool stored_entry(const uint8_t* in, uint64_t n, uint64_t b) {
    const uint64_t p = b >> 3;
    return (b & 7) == 0 && p + 5 <= n && in[p] == 0 && in[p + 1] == (uint8_t) ~in[p + 3] && in[p + 2] == (uint8_t) ~in[p + 4];
}

// A member header at byte-aligned bit b: 1f 8b 08 and no reserved flag.
BGZF_HD bool header_entry(const uint8_t* in, uint64_t n, uint64_t b) {
    const uint64_t p = b >> 3;
    return (b & 7) == 0 && p + 10 <= n && in[p] == 0x1f && in[p + 1] == 0x8b && in[p + 2] == 8 && !(in[p + 3] & 0xE0);
}

BGZF_HD bool entry_at(const uint8_t* in, uint64_t n, uint64_t b) {
    const uint64_t p = b >> 3;
    if (p + 3 > n) return false;
    const uint32_t w = ((uint32_t) in[p] | (uint32_t) in[p + 1] << 8 | (uint32_t) in[p + 2] << 16) >> (b & 7);   // >= 17 bits
    if ((w & 7u) == 4u && ((w >> 3) & 31u) <= 29u && ((w >> 8) & 31u) <= 29u) return dynamic_entry(in, n, b);
    return stored_entry(in, n, b) || header_entry(in, n, b);
}

// ---- the span decoder ----------------------------------------------------------------------------------------------------
struct Trailer {
    unsigned long long at, out_end;   // byte offset of the trailer; output offset of the member's end in the text
    uint32_t crc, isize;
};

struct Span {
    unsigned long long exit;          // the boundary (bit) where the decode stopped
    unsigned long long out;           // output bytes, up to the error when there is one
    unsigned long long last_start;    // output offset + 1 of the last member start inside the span (0: none)
    unsigned long long err_at;        // byte offset of the failing header, trailer or DEFLATE block
    unsigned long long last_marker;   // symbol mode: position + 1 of the last marker written (0: none)
    uint32_t err, members;            // error code (0: none); trailers passed before it
};

struct Sink {                 // symbol mode
    uint16_t* sym;            // the span's symbols [0, cap)
    uint8_t* text;            // the span's place in the text: literal bytes are written there too
    unsigned long long cap, base;   // symbols the span holds; its output offset in the text
    long long floor;          // the earliest position a distance may reach, relative to the span (the member's start)
    Trailer* trailers;        // one per member end in the span
};

// Decodes in[0, n) from boundary `start` (bit; 0 = the first member header) to the first boundary at or after `stop`.
template <bool kWrite>
BGZF_HD Span decode_span(const uint8_t* in, uint64_t n, uint64_t start, uint64_t stop, bgzf::Tables& t, Sink* sink) {
    Span r{start, 0, 0, 0, 0, 0, 0};
    const uint64_t end = n * 8;
    if (start >= end) {
        r.exit = end;
        return r;
    }
    Stream b{in, n, 0, 0, 0};
    b.seek(start);
    // a block never starts with byte 1f (BTYPE 3), so a byte-aligned 1f at a boundary is a member header
    bool header = start == 0 || ((start & 7) == 0 && in[start >> 3] == 0x1f);
    long long floor = kWrite ? sink->floor : 0;
    uint64_t o = 0, marker = 0;
    uint32_t err = 0;
    while (true) {
        const uint64_t at = b.bit();
        if (at >= stop) break;
        r.err_at = at >> 3;
        if (header) {
            const uint64_t h = at >> 3, len = member_header(in, n, h, err);
            if (err) break;
            b.seek((h + len) * 8);
            header = false;
            floor = (long long) o;
            r.last_start = o + 1;
            continue;
        }
        const uint32_t last = b.take(1, err), type = b.take(2, err);
        if (err) break;
        if (type == 0) {
            const uint32_t drop = b.cnt & 7u;
            b.buf >>= drop;
            b.cnt -= drop;
            const uint32_t len = b.take(16, err), nlen = b.take(16, err);
            if (err) break;
            if (len != (~nlen & 0xFFFFu)) {
                err = bgzf::kStoredLen;
                break;
            }
            if (kWrite && len > sink->cap - o) {
                err = bgzf::kLong;
                break;
            }
            uint32_t k = 0;
            for (; k < len && b.cnt; ++k, ++o) {   // whole bytes still in the bit buffer, then straight from the input
                if (kWrite) sink->sym[o] = sink->text[o] = (uint8_t) b.buf;
                b.buf >>= 8;
                b.cnt -= 8;
            }
            if (len - k > b.n - b.pos) {
                err = bgzf::kPastEnd;
                break;
            }
            if (kWrite)
                for (uint32_t j = k; j < len; ++j) sink->sym[o + j - k] = sink->text[o + j - k] = in[b.pos + j - k];
            o += len - k;
            b.pos += len - k;
        } else if (type == 3) {
            err = bgzf::kBtype3;
            break;
        } else {
            if (type == 1) {
                bgzf::fixed_codes(t);
            } else {
                err = bgzf::dynamic_codes(t, b);
                if (err) break;
            }
            while (true) {
                const int sym = bgzf::decode(t.lit, b, err);
                if (err) break;
                if (sym < 0 || sym > 285) {
                    err = bgzf::kBadSymbol;
                    break;
                }
                if (sym < 256) {
                    if (kWrite) {
                        if (o == sink->cap) {
                            err = bgzf::kLong;
                            break;
                        }
                        sink->sym[o] = sink->text[o] = (uint8_t) sym;
                    }
                    ++o;
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
                const int d = bgzf::decode(t.dist, b, err);
                if (err) break;
                if (d < 0 || d > 29) {
                    err = bgzf::kBadDistSymbol;
                    break;
                }
                uint32_t dist;
                if (d < 4) {
                    dist = (uint32_t) d + 1;
                } else {
                    const uint32_t x = ((uint32_t) d - 2) >> 1;
                    dist = ((2u + ((uint32_t) d & 1u)) << x) + 1u + b.take(x, err);
                }
                if (err) break;
                if (kWrite) {
                    if ((long long) o - (long long) dist < floor) {
                        err = bgzf::kTooFar;
                        break;
                    }
                    if (len > sink->cap - o) {
                        err = bgzf::kLong;
                        break;
                    }
                    for (uint32_t k = 0; k < len; ++k) {
                        const long long from = (long long) (o + k) - dist;
                        const uint16_t v = from >= 0 ? sink->sym[from] : (uint16_t) (256 + kWindow + from);
                        sink->sym[o + k] = v;
                        if (v < 256) {
                            sink->text[o + k] = (uint8_t) v;
                        } else {
                            marker = o + k + 1;
                        }
                    }
                }
                o += len;
            }
            if (err) break;
        }
        if (!last) continue;
        // the member's end: trailer, zero padding, then the next member or the end of the input
        const uint32_t drop = b.cnt & 7u;
        b.buf >>= drop;
        b.cnt -= drop;
        const uint64_t tb = b.bit() >> 3;
        r.err_at = tb;
        if (n - tb < 8) {
            err = kTrailerEnd;
            break;
        }
        if (kWrite) {
            const uint8_t* q = in + tb;
            sink->trailers[r.members] = Trailer{tb, sink->base + o, (uint32_t) q[0] | (uint32_t) q[1] << 8 | (uint32_t) q[2] << 16 | (uint32_t) q[3] << 24,
                                                (uint32_t) q[4] | (uint32_t) q[5] << 8 | (uint32_t) q[6] << 16 | (uint32_t) q[7] << 24};
        }
        r.members++;
        uint64_t p = tb + 8;
        while (p < n && in[p] == 0) ++p;
        if (p < n && in[p] != 0x1f) {
            r.err_at = p;
            err = kAfterLast;
            break;
        }
        b.seek(p * 8);
        if (p == n) break;
        header = true;
    }
    r.exit = b.bit();
    r.out = o;
    r.err = err;
    r.last_marker = marker;
    return r;
}

// ---- the verification walk (host) ----------------------------------------------------------------------------------------
// After a counting round: E holds the chunks' entries (E[0] = 0), res their decodes (chunk i stopped at the first boundary
// at or after E[i + 1]).  A chunk is verified when its predecessor is verified and stopped exactly at its entry.  Where a
// verified chunk stopped past its successor's entry, that entry was false: the successor moves to the stop, chunks whose
// entries the decode passed merge into it, and it goes to `dirty` for the next round.  A chunk whose own entry was
// matched hands its stop to its successor the same way (a likely true start, decoded in the same round).  The stream's
// end or a verified decode error cuts the chunk list.  Returns the index of the verified chunk that failed, or SIZE_MAX;
// `dirty` empty means every chunk is verified.
inline size_t walk(std::vector<unsigned long long>& E, std::vector<Span>& res, uint64_t end, std::vector<uint32_t>& dirty) {
    dirty.clear();
    bool verified = true, trusted = true;
    for (size_t i = 0; i < E.size(); ++i) {
        const Span r = res[i];
        if (r.err) {
            if (verified) {
                E.resize(i + 1);
                res.resize(i + 1);
                return i;
            }
            verified = trusted = false;
            continue;
        }
        if (i + 1 == E.size()) break;
        if (r.exit == E[i + 1]) {
            trusted = true;
            continue;
        }
        if (verified) {
            if (r.exit >= end) {   // the stream ends in chunk i
                E.resize(i + 1);
                res.resize(i + 1);
                break;
            }
            size_t j = i + 2;
            while (j < E.size() && E[j] <= r.exit) ++j;
            E.erase(E.begin() + (i + 2), E.begin() + j);
            res.erase(res.begin() + (i + 2), res.begin() + j);
            E[i + 1] = r.exit;
            dirty.push_back((uint32_t) (i + 1));
        } else if (trusted && r.exit < end && (i + 2 >= E.size() || r.exit < E[i + 2])) {
            E[i + 1] = r.exit;
            dirty.push_back((uint32_t) (i + 1));
        }
        verified = trusted = false;
    }
    return SIZE_MAX;
}

}  // namespace deflate
