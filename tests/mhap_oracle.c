/* tests/mhap_oracle.c — TEST INFRASTRUCTURE: the MHAP reader of include/rala_b200.h (rala_b200_parse_mhap) stated
 * sequentially in plain C, one line after the other, field after field.  The tests pin it to the reference's records in
 * tests/golden (through synth.Dataset.write_mhap and the oracle's duplicate filter), check it against a Python
 * restatement of the contract and compare the device reader with it; bench_mhap.py times it on one core.
 *
 * int ora_parse_mhap(read_len, n_reads, text, n_bytes, cols, cap, stats, err)
 *   cols:  7 x cap words, as rala_b200_parse_mhap writes them
 *   stats: n_records, n_length_mismatch, first_length_mismatch (UINT64_MAX: none), n_query_rc
 *   err:   line (1-based), kind (1 fields, 2 empty, 3 non-digit, 4 >= 2^32, 5 not a read id, 6 not a strand),
 *          field (fields found for kind 1)
 *   returns 0, -1 refused line (err), -3 cap too small */
#include <stdint.h>
#include <string.h>

int ora_parse_mhap(const uint32_t* read_len, uint32_t n_reads, const char* text, uint64_t n_bytes, uint32_t* cols, uint64_t cap,
                   uint64_t* stats, uint64_t* err) {
    stats[0] = stats[1] = stats[3] = 0;
    stats[2] = UINT64_MAX;
    uint64_t pos = 0, line = 0;
    while (pos < n_bytes) {
        const char* nl = (const char*) memchr(text + pos, '\n', n_bytes - pos);
        const uint64_t e = nl ? (uint64_t) (nl - text) : n_bytes;
        ++line;
        uint64_t fb[12], fe[12];
        unsigned nf = 0;
        uint64_t p = pos;
        while (nf < 12) {   /* the first 12 fields; the rest of the line is never looked at */
            fb[nf] = p;
            while (p < e && text[p] != ' ') ++p;
            fe[nf++] = p;
            if (p == e) break;
            ++p;
        }
        if (e == pos) { err[0] = line; err[1] = 2; err[2] = 1; return -1; }
        if (nf < 12) { err[0] = line; err[1] = 1; err[2] = nf; return -1; }
        if (fe[11] == e && fe[11] > fb[11] && text[e - 1] == '\r') --fe[11];   /* CRLF */
        uint32_t v[12] = {0};
        for (int f = 0; f < 12; ++f) {
            if (f == 2 || f == 3) continue;   /* error, shared minmers: never read */
            if (f == 4 || f == 8) {
                if (fe[f] - fb[f] != 1 || (text[fb[f]] != '0' && text[fb[f]] != '1')) { err[0] = line; err[1] = 6; err[2] = f + 1; return -1; }
                v[f] = (uint32_t) (text[fb[f]] - '0');
                continue;
            }
            uint64_t x = 0;
            if (fb[f] == fe[f]) { err[0] = line; err[1] = 3; err[2] = f + 1; return -1; }
            for (uint64_t q = fb[f]; q < fe[f]; ++q) {
                const unsigned d = (unsigned) (uint8_t) text[q] - '0';
                if (d > 9) { err[0] = line; err[1] = 3; err[2] = f + 1; return -1; }
                x = x * 10 + d;
                if (x > 0xFFFFFFFFull) { err[0] = line; err[1] = 4; err[2] = f + 1; return -1; }
            }
            if (f < 2 && (x == 0 || x > n_reads)) { err[0] = line; err[1] = 5; err[2] = f + 1; return -1; }
            v[f] = (uint32_t) x;
        }
        const uint64_t i = line - 1;
        if (i >= cap) return -3;
        const uint32_t a = v[0] - 1, b = v[1] - 1;
        const uint32_t sa = v[6] - v[5], sb = v[10] - v[9];   /* uint32_t: mod 2^32 */
        cols[i] = a;
        cols[cap + i] = b | (v[4] ^ v[8]) << 31;
        cols[2 * cap + i] = v[5];
        cols[3 * cap + i] = v[6];
        cols[4 * cap + i] = v[9];
        cols[5 * cap + i] = v[10];
        cols[6 * cap + i] = sa > sb ? sa : sb;
        if (v[7] != read_len[a] || v[11] != read_len[b]) {
            if (!stats[1]) stats[2] = i;
            ++stats[1];
        }
        stats[3] += v[4];
        stats[0] = line;
        pos = e + 1;
    }
    return 0;
}
