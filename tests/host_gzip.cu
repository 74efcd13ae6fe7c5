// Host build of the chunked gzip inflate of rala_b200/csrc/gzip.cu, run sequentially with the same pieces (deflate.cuh):
// the finder, the counting rounds and their verification walk, the symbol pass, the window chain, the resolve and the
// CRC32 / ISIZE checks; for the CPU suite (tests/test_gzip_reader.py).
// stdin:  u64 n, u64 chunk bytes, u64 k, then k entry bit offsets (k = ~0: the finder proposes them; otherwise they
//         replace it, chunk 0 still starting at bit 0), then the n input bytes.
// stdout: u32 status (0 or a deflate / bgzf error code), u32 0, u64 member, u64 byte offset, u64 corrected decodes,
//         u64 rounds, u64 chunks, u64 text bytes, then the text when the status is 0.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../rala_b200/csrc/deflate.cuh"

using deflate::Span;
using deflate::Trailer;

static uint64_t get64() {
    uint64_t v = 0;
    if (fread(&v, 8, 1, stdin) != 1) exit(2);
    return v;
}

int main() {
    const uint64_t n = get64(), chunk = get64(), k = get64();
    std::vector<unsigned long long> given;
    if (k != ~0ull)
        for (uint64_t i = 0; i < k; ++i) given.push_back(get64());
    uint8_t* in = (uint8_t*) malloc(n ? n : 1);   // the input ends exactly at the end of its heap block
    if (n && fread(in, 1, n, stdin) != n) return 2;
    const uint64_t end = n * 8;
    uint64_t out[6] = {0, 0, 0, 0, 0, 0};   // member, offset, corrected, rounds, chunks, bytes
    uint32_t status[2] = {0, 0};
    std::vector<uint8_t> text;
    bgzf::Tables* t = new bgzf::Tables;
    if (n) {
        std::vector<unsigned long long> E{0};
        if (k == ~0ull) {
            for (uint64_t c = 1; c * chunk < n; ++c)
                for (uint64_t b = c * chunk * 8, hi = std::min((c + 1) * chunk, n) * 8; b < hi; ++b)
                    if (deflate::entry_at(in, n, b)) {
                        E.push_back(b);
                        break;
                    }
        } else {
            for (unsigned long long b : given)
                if (b > E.back() && b < end) E.push_back(b);
        }
        std::vector<Span> res(E.size());
        std::vector<uint32_t> dirty(E.size());
        for (uint32_t i = 0; i < dirty.size(); ++i) dirty[i] = i;
        while (!dirty.empty()) {   // a verified decode error cuts the chunk list; the symbol pass meets it again
            for (uint32_t i : dirty) res[i] = deflate::decode_span<false>(in, n, E[i], i + 1 < E.size() ? E[i + 1] : ~0ull, *t, nullptr);
            if (out[3]) out[2] += dirty.size();
            out[3]++;
            deflate::walk(E, res, end, dirty);
        }
        const size_t nc = E.size();
        std::vector<unsigned long long> base(nc + 1, 0), mem(nc + 1, 0);
        std::vector<long long> floors(nc);
        unsigned long long member_start = 0;
        for (size_t i = 0; i < nc; ++i) {
            base[i + 1] = base[i] + res[i].out;
            mem[i + 1] = mem[i] + res[i].members;
            floors[i] = (long long) member_start - (long long) base[i];
            if (res[i].last_start) member_start = base[i] + res[i].last_start - 1;
        }
        out[4] = nc;
        const uint64_t total = base[nc];
        text.assign(total, 0xAA);
        std::vector<uint16_t> sym(total + 1);
        std::vector<Trailer> tr(mem[nc] + 1);
        std::vector<Span> sp(nc);
        for (size_t i = 0; i < nc; ++i) {   // symbol pass
            deflate::Sink sink{sym.data() + base[i], text.data() + base[i], res[i].out, base[i], floors[i], tr.data() + mem[i]};
            sp[i] = deflate::decode_span<true>(in, n, E[i], i + 1 < nc ? E[i + 1] : ~0ull, *t, &sink);
        }
        for (int pass = 0; pass < 2; ++pass)   // chain (each chunk's last 32 KiB, in order), then the rest
            for (size_t i = 0; i < nc; ++i) {
                const unsigned long long len = sp[i].out, tail = len > deflate::kWindow ? len - deflate::kWindow : 0;
                const unsigned long long lo = pass ? 0 : tail, hi = pass ? std::min(tail, sp[i].last_marker) : sp[i].last_marker;
                for (unsigned long long q = lo; q < hi; ++q) {
                    const uint32_t v = sym[base[i] + q];
                    if (v >= 256) text[base[i] + q] = text.at(base[i] - deflate::kWindow + (v - 256));
                }
            }
        size_t n_tr = mem[nc];
        uint64_t bad_member = 0, bad_at = 0;
        uint32_t bad = 0;
        for (size_t i = 0; i < nc; ++i)
            if (sp[i].err) {
                bad = sp[i].err;
                bad_member = n_tr = mem[i] + sp[i].members;
                bad_at = sp[i].err_at;
                break;
            }
        uint32_t table[256];
        for (uint32_t i = 0; i < 256; ++i) table[i] = bgzf::crc_table_entry(i);
        for (size_t m = 0; m < n_tr && !status[0]; ++m) {
            const unsigned long long lo = m ? tr[m - 1].out_end : 0, hi = tr[m].out_end;
            if (bgzf::crc_update(0, text.data() + lo, (uint32_t) (hi - lo), table) != tr[m].crc) {
                status[0] = bgzf::kCrc;
            } else if ((uint32_t) (hi - lo) != tr[m].isize) {
                status[0] = deflate::kIsize;
            }
            out[0] = m;
            out[1] = tr[m].at;
        }
        if (!status[0] && bad) {
            status[0] = bad;
            out[0] = bad_member;
            out[1] = bad_at;
        }
        if (!status[0]) out[5] = total;
    }
    fwrite(status, 4, 2, stdout);
    fwrite(out, 8, 6, stdout);
    if (!status[0]) fwrite(text.data(), 1, text.size(), stdout);
    delete t;
    free(in);
    return 0;
}
