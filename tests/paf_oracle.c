/* tests/paf_oracle.c — TEST INFRASTRUCTURE: the PAF reader of include/rala_b200.h (rala_b200_parse_paf) stated
 * sequentially in plain C, one line after the other: digit loops instead of strtoul, a byte-exact name map.  The tests
 * pin it to the reference through tests/golden (ids, lengths, coordinates and the unresolved set that the reference's
 * own PafParser + name_to_id_ produced) and compare the device reader with it; bench_paf.py times it on one core.
 *
 * int ora_parse_paf(names, name_end, read_len, n_reads, text, n_bytes, cols, cap, stats, err)
 *   cols:  7 x cap words, as rala_b200_parse_paf writes them
 *   stats: n_records, n_unresolved, n_length_mismatch, first_length_mismatch (UINT64_MAX: none)
 *   err:   line (1-based), kind (1 fields, 2 empty, 3 non-digit, 4 >= 2^32), column (fields found for kind 1)
 *   returns 0, -1 refused line (err), -2 duplicate read name (err[0] = later id, err[1] = earlier id), -3 cap too small */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define UNKNOWN 0x7FFFFFFFu

typedef struct {
    const char* names;
    const uint64_t* end;
    uint32_t* slot;   /* id + 1, 0 = empty */
    uint64_t mask;
} NameMap;

static uint64_t fnv(const char* p, uint64_t n) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint64_t i = 0; i < n; ++i) h = (h ^ (uint8_t) p[i]) * 0x100000001b3ull;
    return h;
}

static const char* name_of(const NameMap* m, uint32_t id, uint64_t* len) {
    const uint64_t b0 = id ? m->end[id - 1] : 0;
    *len = m->end[id] - b0;
    return m->names + b0;
}

/* returns the id of an equal name already in the map, or inserts id and returns UNKNOWN */
static uint32_t map_find(const NameMap* m, const char* p, uint64_t n, uint32_t insert_id) {
    for (uint64_t s = fnv(p, n) & m->mask;; s = (s + 1) & m->mask) {
        if (!m->slot[s]) {
            if (insert_id != UNKNOWN) m->slot[s] = insert_id + 1;
            return UNKNOWN;
        }
        uint64_t len;
        const char* q = name_of(m, m->slot[s] - 1, &len);
        if (len == n && memcmp(q, p, n) == 0) return m->slot[s] - 1;
    }
}

int ora_parse_paf(const char* names, const uint64_t* name_end, const uint32_t* read_len, uint32_t n_reads, const char* text,
                  uint64_t n_bytes, uint32_t* cols, uint64_t cap, uint64_t* stats, uint64_t* err) {
    NameMap m = {names, name_end, NULL, 0};
    uint64_t slots = 1024;
    while (slots < 2ull * n_reads) slots <<= 1;
    m.mask = slots - 1;
    m.slot = (uint32_t*) calloc(slots, sizeof(uint32_t));
    for (uint32_t i = 0; i < n_reads; ++i) {
        uint64_t len;
        const char* p = name_of(&m, i, &len);
        const uint32_t other = map_find(&m, p, len, i);
        if (other != UNKNOWN) {
            err[0] = i; err[1] = other;
            free(m.slot);
            return -2;
        }
    }
    stats[0] = stats[1] = stats[2] = 0;
    stats[3] = UINT64_MAX;
    uint64_t pos = 0, line = 0;
    int rc = 0;
    while (pos < n_bytes) {
        const char* nl = (const char*) memchr(text + pos, '\n', n_bytes - pos);
        const uint64_t e = nl ? (uint64_t) (nl - text) : n_bytes;
        ++line;
        uint64_t fb[12], fe[12];
        unsigned nf = 0;
        uint64_t p = pos;
        while (nf < 12) {   /* the first 12 fields; the rest of the line is never looked at */
            fb[nf] = p;
            while (p < e && text[p] != '\t') ++p;
            fe[nf++] = p;
            if (p == e) break;
            ++p;
        }
        if (e == pos) { err[0] = line; err[1] = 2; err[2] = 1; rc = -1; break; }
        if (nf < 12) { err[0] = line; err[1] = 1; err[2] = nf; rc = -1; break; }
        static const int numeric[] = {1, 2, 3, 6, 7, 8, 10};
        uint32_t v[12] = {0};
        for (int k = 0; k < 7 && !rc; ++k) {
            const int f = numeric[k];
            uint64_t x = 0;
            if (fb[f] == fe[f]) { err[0] = line; err[1] = 3; err[2] = f + 1; rc = -1; }
            for (uint64_t q = fb[f]; q < fe[f] && !rc; ++q) {
                const unsigned d = (unsigned) (uint8_t) text[q] - '0';
                if (d > 9) { err[0] = line; err[1] = 3; err[2] = f + 1; rc = -1; break; }
                x = x * 10 + d;
                if (x > 0xFFFFFFFFull) { err[0] = line; err[1] = 4; err[2] = f + 1; rc = -1; break; }
            }
            v[f] = (uint32_t) x;
        }
        if (rc) break;
        const uint64_t i = line - 1;
        if (i >= cap) { rc = -3; break; }
        const uint32_t a = map_find(&m, text + fb[0], fe[0] - fb[0], UNKNOWN);
        const uint32_t b = map_find(&m, text + fb[5], fe[5] - fb[5], UNKNOWN);
        const int ka = a != UNKNOWN, kb = b != UNKNOWN;
        const uint32_t ori = text[fb[4]] != '+';
        cols[i] = a | (ka && kb ? 0u : 0x80000000u);
        cols[cap + i] = b | ori << 31;
        cols[2 * cap + i] = v[2];
        cols[3 * cap + i] = v[3];
        cols[4 * cap + i] = v[7];
        cols[5 * cap + i] = v[8];
        cols[6 * cap + i] = v[10];
        stats[1] += !(ka && kb);
        if ((ka && v[1] != read_len[a]) || (kb && v[6] != read_len[b])) {
            if (!stats[2]) stats[3] = i;
            ++stats[2];
        }
        stats[0] = line;
        pos = e + 1;
    }
    free(m.slot);
    return rc;
}
