/* Plain-C reader of the FASTA / FASTQ text contract of rala_b200_graph_set_reads_text (include/rala_b200.h), one pass
 * over the text in file order.  Used by tests/reads_oracle.py; never linked into the library.
 *
 * ora_read_seq(text, n, blob, ends, lens, cap, stats, err):
 *   blob (>= n bytes), ends / lens (cap reads) receive the names back to back, their u64 end offsets and u32 lengths;
 *   stats = format, n_reads, n_lines, n_bases, name_bytes, max_len, n_described.
 *   returns 0; -1 refused: err = line (1-based), column, kind; -2 a name listed twice: err = earlier id, later id;
 *   -3 cap too small. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { EMPTY = 1, CR, HEADER, NAME_EMPTY, NAME_BYTE, SEQ_BYTE, PLUS, QUAL_LEN, TRUNCATED, NO_SEQ, TOO_LONG, TOO_MANY, FORMAT };
#define MAX_READS ((1ull << 31) - 1)

static uint64_t best;
static void refuse(uint64_t line, uint64_t column, unsigned kind) {   /* the smallest (line, column, kind) is reported */
    const uint64_t w = line << 30 | column << 4 | kind;
    if (w < best) best = w;
}

static const uint8_t* g_blob;
static const uint64_t* g_ends;
static int by_name(const void* x, const void* y) {
    const uint32_t i = *(const uint32_t*) x, j = *(const uint32_t*) y;
    const uint64_t bi = i ? g_ends[i - 1] : 0, bj = j ? g_ends[j - 1] : 0, li = g_ends[i] - bi, lj = g_ends[j] - bj;
    const int c = memcmp(g_blob + bi, g_blob + bj, li < lj ? li : lj);
    if (c) return c;
    if (li != lj) return li < lj ? -1 : 1;
    return i < j ? -1 : (i > j);
}

int ora_read_seq(const uint8_t* t, uint64_t n, uint8_t* blob, uint64_t* ends, uint32_t* lens, uint64_t cap, uint64_t* stats,
                 uint64_t* err) {
    memset(stats, 0, 7 * sizeof(uint64_t));
    if (n == 0) return 0;
    best = ~0ull;
    if (t[0] != '>' && t[0] != '@') {
        err[0] = 1, err[1] = 1, err[2] = FORMAT;
        return -1;
    }
    const int fastq = t[0] == '@';
    uint64_t* len64 = calloc(cap + 1, 8);
    uint64_t* hdr_line = calloc(cap + 1, 8);
    uint64_t reads = 0, nb = 0, g = 0, s = 0, described = 0;
    for (; s < n; ++g) {
        const uint8_t* nl = memchr(t + s, '\n', n - s);
        const uint64_t e = nl ? (uint64_t) (nl - t) : n, len = e - s;
        if (len == 0) refuse(g, 1, EMPTY);
        const int hdr = fastq ? g % 4 == 0 : len > 0 && t[s] == '>';
        const int seq = fastq ? g % 4 == 1 : !hdr;
        for (uint64_t p = s; p < e; ++p)   /* the byte rules: the line's first offending byte */
            if (t[p] == '\r' || (seq && (t[p] < 0x21 || t[p] > 0x7E))) {
                refuse(g, p - s + 1, t[p] == '\r' ? CR : SEQ_BYTE);
                break;
            }
        if (hdr) {
            uint64_t p = s + 1, name = 0;
            if (len) {
                for (; p < e && t[p] != ' ' && t[p] != '\t'; ++p)
                    if (((t[p] < 0x20 && t[p] != '\r') || t[p] == 0x7F) && !name) name = p - s + 1;
                if (name) refuse(g, name, NAME_BYTE);
                if (p == s + 1) refuse(g, 2, NAME_EMPTY);
                described += p < e;
                if (fastq && t[s] != '@') refuse(g, 1, HEADER);
            }
            const uint64_t nlen = len ? p - s - 1 : 0;
            if (reads >= MAX_READS) {
                refuse(g, 1, TOO_MANY);
            } else {
                if (reads >= cap) {
                    free(len64), free(hdr_line);
                    return -3;
                }
                memcpy(blob + nb, t + s + 1, nlen);
                ends[reads] = nb + nlen;
                hdr_line[reads] = g;
            }
            nb += nlen;
            ++reads;
        } else if (len) {
            const uint64_t cur = reads - 1;   /* line 1 is always a header */
            if (!fastq) {
                len64[cur] += len;
            } else if (g % 4 == 1) {
                len64[cur] = len;
            } else if (g % 4 == 2) {
                if (t[s] != '+') refuse(g, 1, PLUS);
            } else if (len != len64[cur]) {
                refuse(g, (len < len64[cur] ? len : len64[cur]) + 1, QUAL_LEN);
            }
        }
        s = e + 1;
    }
    const uint64_t n_lines = g;
    if (fastq && n_lines % 4) refuse(n_lines / 4 * 4, 1, TRUNCATED);
    const uint64_t kept = reads < MAX_READS ? reads : MAX_READS;
    uint64_t bases = 0, longest = 0;
    for (uint64_t r = 0; r < kept; ++r) {
        if (len64[r] == 0) refuse(hdr_line[r], 1, NO_SEQ);
        if (len64[r] >> 32) refuse(hdr_line[r], 1, TOO_LONG);
        lens[r] = len64[r] >> 32 ? 0xFFFFFFFFu : (uint32_t) len64[r];
        bases += len64[r];
        if (len64[r] > longest) longest = len64[r];
    }
    free(len64), free(hdr_line);
    if (best != ~0ull) {
        err[0] = (best >> 30) + 1, err[1] = (best >> 4) & 0x3FFFFFF, err[2] = best & 15;
        return -1;
    }
    /* a name listed twice: the first read whose name an earlier read has */
    uint32_t* order = malloc((kept + 1) * sizeof(uint32_t));
    for (uint64_t r = 0; r < kept; ++r) order[r] = (uint32_t) r;
    g_blob = blob, g_ends = ends;
    qsort(order, kept, sizeof(uint32_t), by_name);
    uint64_t later = ~0ull, earlier = 0;
    for (uint64_t k = 1; k < kept; ++k) {
        const uint32_t i = order[k - 1], j = order[k];
        const uint64_t bi = i ? ends[i - 1] : 0, bj = j ? ends[j - 1] : 0;
        if (ends[i] - bi == ends[j] - bj && !memcmp(blob + bi, blob + bj, ends[i] - bi) && j < later) {
            uint64_t k0 = k - 1;   /* the earliest read with this name: the first of its run */
            while (k0 > 0) {
                const uint32_t h = order[k0 - 1];
                const uint64_t bh = h ? ends[h - 1] : 0;
                if (ends[h] - bh != ends[i] - bi || memcmp(blob + bh, blob + bi, ends[i] - bi)) break;
                --k0;
            }
            later = j, earlier = order[k0];
        }
    }
    free(order);
    if (later != ~0ull) {
        err[0] = earlier, err[1] = later;
        return -2;
    }
    stats[0] = fastq ? 2 : 1, stats[1] = kept, stats[2] = n_lines, stats[3] = bases, stats[4] = nb, stats[5] = longest;
    stats[6] = described;
    return 0;
}
