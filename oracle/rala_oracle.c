/* oracle/rala_oracle.c — TEST INFRASTRUCTURE (see rala_oracle.h): sequential plain-C restatement of
 * rala's hot path in array form.  Parity status: PINNED against the compiled reference
 * (tests/test_oracle_vs_ref.py) and its golden vectors (tests/golden/).
 *
 * It deliberately keeps the reference's SEQUENTIAL formulations (kills applied in processing
 * order, candidate array + is_marked check in the transitive pass) so that it is an independent
 * check of the order-free formulations the CUDA path uses (death-time fixed point, T(e) | T(e^1)).
 */
#include "rala_oracle.h"

#include <stdlib.h>
#include <string.h>

#define REC 7

static inline uint32_t u32min(uint32_t a, uint32_t b) { return a < b ? a : b; }
static inline uint32_t u32max(uint32_t a, uint32_t b) { return a > b ? a : b; }
static inline uint32_t absdiff(uint32_t a, uint32_t b) { return a > b ? a - b : b - a; }
static inline int pile_alive(const uint32_t* piles, uint32_t n_piles, uint32_t id) {
    return id < n_piles && piles[2 * id + 1] != 0;
}

/* graph.cpp:26-29 — (1 - eps), (1 + eps) are formed in double exactly as there */
int ora_comparable(uint32_t a_, uint32_t b_) {
    const double eps = 0.12;
    double a = (double) a_, b = (double) b_;
    return (a >= b * (1 - eps) && a <= b * (1 + eps)) || (b >= a * (1 - eps) && b <= a * (1 + eps));
}

/* overlap.cpp:117-192 (SURVEY.md A.1).  All arithmetic is u32 with wrap-around, as in the reference. */
int ora_trim(uint32_t* r, const uint32_t* piles, uint32_t n_piles) {
    uint32_t a = r[0], b = r[1];
    if (!pile_alive(piles, n_piles, a) || !pile_alive(piles, n_piles, b)) return 0;   /* :123-126 */
    uint32_t pa0 = piles[2 * a], pa1 = piles[2 * a + 1], pb0 = piles[2 * b], pb1 = piles[2 * b + 1];
    uint32_t ab = r[2], ae = r[3], bb = r[4], be = r[5], ori = r[6] & 1u;

    if (ab >= pa1 || ae <= pa0 || bb >= pb1 || be <= pb0) return 0;                     /* :139-142 */

    uint32_t cut_lb = bb < pb0 ? pb0 - bb : 0, cut_rb = be > pb1 ? be - pb1 : 0;
    uint32_t cut_la = ab < pa0 ? pa0 - ab : 0, cut_ra = ae > pa1 ? ae - pa1 : 0;
    uint32_t nab, nae, nbb, nbe;
    if (ori) {                                                                          /* :146-154 */
        nab = ab + cut_rb; nae = ae - cut_lb; nbb = bb + cut_ra; nbe = be - cut_la;
    } else {                                                                            /* :155-164 */
        nab = ab + cut_lb; nae = ae - cut_rb; nbb = bb + cut_la; nbe = be - cut_ra;
    }
    if (nab >= pa1 || nae <= pa0 || nbb >= pb1 || nbe <= pb0) return 0;                 /* :166-169 */
    nab = u32max(nab, pa0); nae = u32min(nae, pa1);                                     /* :171-174 */
    nbb = u32max(nbb, pb0); nbe = u32min(nbe, pb1);
    if (nab >= nae || nae - nab < 84 || nbb >= nbe || nbe - nbb < 84) return 0;         /* :176-179 */
    r[2] = nab; r[3] = nae; r[4] = nbb; r[5] = nbe;                                     /* :181-189 */
    return 1;
}

/* overlap.cpp:194-259 (SURVEY.md A.2).  length_ is max(span_a, span_b) of the stored coordinates:
 * trim() always ran (and set it, :189) before any type() call on the path. */
static int type_with_coords(const uint32_t* r, const uint32_t* piles,
                            uint32_t* A0, uint32_t* A1, uint32_t* B0, uint32_t* B1, uint32_t* AL, uint32_t* BL) {
    uint32_t a = r[0], b = r[1], ori = r[6] & 1u;
    uint32_t pa0 = piles[2 * a], pa1 = piles[2 * a + 1], pb0 = piles[2 * b], pb1 = piles[2 * b + 1];
    uint32_t al = pa1 - pa0, a0 = r[2] - pa0, a1 = r[3] - pa0;                          /* :206-208 */
    uint32_t bl = pb1 - pb0;                                                            /* :210 */
    uint32_t b0 = ori ? bl - r[5] + pb0 : r[4] - pb0;                                   /* :211-213 */
    uint32_t b1 = ori ? bl - r[4] + pb0 : r[5] - pb0;                                   /* :214-216 */
    *A0 = a0; *A1 = a1; *B0 = b0; *B1 = b1; *AL = al; *BL = bl;

    uint32_t overhang = u32min(a0, b0) + u32min(al - a1, bl - b1);                      /* :218-219 */
    if ((double) (uint32_t) (a1 - a0) < (double) (uint32_t) (a1 - a0 + overhang) * 0.875 ||
        (double) (uint32_t) (b1 - b0) < (double) (uint32_t) (b1 - b0 + overhang) * 0.875) {
        return ORA_KX;                                                                  /* :221-224 */
    }
    if (a0 <= b0 && (al - a1) <= (bl - b1)) return ORA_KB;                              /* :225-227 */
    if (a0 >= b0 && (al - a1) >= (bl - b1)) return ORA_KA;                              /* :228-230 */

    uint32_t span_a = r[3] - r[2], span_b = r[5] - r[4];
    uint32_t length = u32max(span_a, span_b);
    if ((double) absdiff(span_a, span_b) < (double) length * 0.01) {                    /* :236 */
        uint32_t min_extension = (uint32_t) (0.05 * (double) u32max(al, bl));           /* :237 */
        if (absdiff(a0, b0) < min_extension) {                                          /* :239-245 */
            return (al - a1) >= (bl - b1) ? ORA_KA : ORA_KB;
        }
        if (absdiff(al - a1, bl - b1) < min_extension) {                                /* :246-252 */
            return a0 >= b0 ? ORA_KA : ORA_KB;
        }
    }
    return a0 > b0 ? ORA_KAB : ORA_KBA;                                                 /* :255-258 */
}

int ora_type(const uint32_t* r, const uint32_t* piles) {
    uint32_t a0, a1, b0, b1, al, bl;
    return type_with_coords(r, piles, &a0, &a1, &b0, &b1, &al, &bl);
}

void ora_trim_type_batch(uint32_t* rec, uint64_t n, const uint32_t* piles, uint32_t n_piles, uint8_t* types) {
    for (uint64_t i = 0; i < n; ++i) {
        uint32_t* r = rec + REC * i;
        types[i] = 255;
        if (!(r[6] & 2u) && ora_trim(r, piles, n_piles)) types[i] = (uint8_t) ora_type(r, piles);
    }
}

/* pile.cpp:457-469 (SURVEY.md A.6): note begin_ is added to coordinates that are already absolute.  The pile picks the
 * side by comparing the overlap's a id with its own id, so a self overlap (a == b) bumps twice with the a-side span. */
static void bump_hills(const uint32_t* hills, uint32_t n_hills, uint32_t* cov,
                       uint32_t pile, uint32_t pile_begin, uint32_t lo, uint32_t hi) {
    uint32_t begin = pile_begin + lo, end = pile_begin + hi;
    /* rows are grouped by ascending pile id: binary search the first row of this pile */
    uint32_t l = 0, h = n_hills;
    while (l < h) {
        uint32_t m = l + (h - l) / 2;
        if (hills[3 * m] < pile) l = m + 1; else h = m;
    }
    for (uint32_t i = l; i < n_hills && hills[3 * i] == pile; ++i) {
        if (begin < hills[3 * i + 1] && end > hills[3 * i + 2]) ++cov[i];
    }
}

/* stable removal of rows whose keep flag is 0 (the reference's shrinkToFit, graph.cpp:31-54, is stable) */
static uint64_t compact(uint32_t* list, uint64_t n, const uint8_t* keep) {
    uint64_t w = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (!keep[i]) continue;
        if (w != i) memcpy(list + REC * w, list + REC * i, REC * sizeof(uint32_t));
        ++w;
    }
    return w;
}

void ora_classify(const uint32_t* rec, uint64_t n, uint32_t* piles, const uint8_t* pflags, uint32_t n_piles,
                  const uint32_t* hills, uint32_t n_hills, uint32_t* hill_cov,
                  uint32_t* ovl_out, uint64_t* n_ovl_out, uint32_t* int_out, uint64_t* n_int_out) {
    uint64_t n_ovl = 0, n_int = 0;
    for (uint64_t i = 0; i < n; ++i) {                                                  /* graph.cpp:448 */
        uint32_t r[REC];
        memcpy(r, rec + REC * i, sizeof(r));
        if (r[6] & 2u) continue;                                                        /* :450 is_valid_overlap_ */
        if (!pile_alive(piles, n_piles, r[0]) || !pile_alive(piles, n_piles, r[1])) continue;  /* :451 transmute */
        if (!ora_trim(r, piles, n_piles)) continue;                                     /* :452 */
        uint32_t a = r[0], b = r[1];
        if (pflags[a] & 1u) bump_hills(hills, n_hills, hill_cov, a, piles[2 * a], r[2], r[3]);   /* :457-459 */
        if (pflags[b] & 1u) bump_hills(hills, n_hills, hill_cov, b, piles[2 * b],
                                       a == b ? r[2] : r[4], a == b ? r[3] : r[5]);              /* :460-462 */
        switch (ora_type(r, piles)) {                                                   /* :464-483 */
            case ORA_KX:
                memcpy(int_out + REC * n_int++, r, sizeof(r));
                break;
            case ORA_KB:
                if (!(pflags[b] & 2u)) { piles[2 * a] = 0; piles[2 * a + 1] = 0; }
                else memcpy(ovl_out + REC * n_ovl++, r, sizeof(r));
                break;
            case ORA_KA:
                if (!(pflags[a] & 2u)) { piles[2 * b] = 0; piles[2 * b + 1] = 0; }
                else memcpy(ovl_out + REC * n_ovl++, r, sizeof(r));
                break;
            default:
                memcpy(ovl_out + REC * n_ovl++, r, sizeof(r));
                break;
        }
    }
    /* :493-515 — at EOF drop whatever touches a dead pile */
    uint64_t w = 0;
    for (uint64_t i = 0; i < n_ovl; ++i) {
        const uint32_t* r = ovl_out + REC * i;
        if (piles[2 * r[0] + 1] == 0 || piles[2 * r[1] + 1] == 0) continue;
        if (w != i) memmove(ovl_out + REC * w, r, REC * sizeof(uint32_t));
        ++w;
    }
    *n_ovl_out = w;
    w = 0;
    for (uint64_t i = 0; i < n_int; ++i) {
        const uint32_t* r = int_out + REC * i;
        if (piles[2 * r[0] + 1] == 0 || piles[2 * r[1] + 1] == 0) continue;
        if (w != i) memmove(int_out + REC * w, r, REC * sizeof(uint32_t));
        ++w;
    }
    *n_int_out = w;
}

uint64_t ora_retrim(uint32_t* list, uint64_t* n, const uint32_t* piles, uint32_t n_piles) {
    uint64_t w = 0, total = *n;
    for (uint64_t i = 0; i < total; ++i) {
        uint32_t* r = list + REC * i;
        if (!ora_trim(r, piles, n_piles)) continue;
        if (w != i) memmove(list + REC * w, r, REC * sizeof(uint32_t));
        ++w;
    }
    *n = w;
    return total - w;
}

void ora_retrim_promote(uint32_t* internals, uint64_t* n_int, uint32_t* ovl, uint64_t* n_ovl,
                        const uint32_t* piles, uint32_t n_piles) {
    uint64_t w = 0, total = *n_int, no = *n_ovl;
    for (uint64_t i = 0; i < total; ++i) {
        uint32_t* r = internals + REC * i;
        if (!ora_trim(r, piles, n_piles)) continue;                                     /* graph.cpp:810-813 */
        int t = ora_type(r, piles);
        if (t == ORA_KAB || t == ORA_KBA) {                                             /* :815-819 */
            memcpy(ovl + REC * no++, r, REC * sizeof(uint32_t));
            continue;
        }
        if (w != i) memmove(internals + REC * w, r, REC * sizeof(uint32_t));
        ++w;
    }
    *n_int = w;
    *n_ovl = no;
}

void ora_final_containment(uint32_t* ovl, uint64_t* n_ovl, uint32_t* internals, uint64_t* n_int,
                           uint32_t* piles, uint32_t n_piles) {
    (void) n_piles;
    uint32_t* lists[2] = {ovl, internals};
    uint64_t* counts[2] = {n_ovl, n_int};
    uint8_t* keep[2];
    for (int l = 0; l < 2; ++l) {                                                       /* graph.cpp:831-866 */
        uint64_t n = *counts[l];
        keep[l] = (uint8_t*) malloc(n ? n : 1);
        for (uint64_t i = 0; i < n; ++i) {
            const uint32_t* r = lists[l] + REC * i;
            uint32_t a = r[0], b = r[1];
            keep[l][i] = 0;
            if (piles[2 * a + 1] == 0 || piles[2 * b + 1] == 0) continue;
            int t = ora_type(r, piles);
            if (t == ORA_KA) { piles[2 * b] = 0; piles[2 * b + 1] = 0; continue; }
            if (t == ORA_KB) { piles[2 * a] = 0; piles[2 * a + 1] = 0; continue; }
            keep[l][i] = 1;
        }
    }
    *n_int = compact(internals, *n_int, keep[1]);                                       /* :867 */
    for (uint64_t i = 0; i < *n_ovl; ++i) {                                             /* :869-876 */
        const uint32_t* r = ovl + REC * i;
        if (keep[0][i] && (piles[2 * r[0] + 1] == 0 || piles[2 * r[1] + 1] == 0)) keep[0][i] = 0;
    }
    *n_ovl = compact(ovl, *n_ovl, keep[0]);
    free(keep[0]);
    free(keep[1]);
}

void ora_build_edges(const uint32_t* ovl, uint64_t n_ovl, const uint32_t* piles, uint32_t n_piles,
                     uint32_t* s2n, uint32_t* n_nodes, uint32_t* edges, uint64_t* n_edges) {
    uint32_t node = 0;
    for (uint32_t i = 0; i < n_piles; ++i) {                                            /* graph.cpp:553-574 */
        if (piles[2 * i + 1] == 0) { s2n[i] = 0xFFFFFFFFu; continue; }
        s2n[i] = node;
        node += 2;
    }
    *n_nodes = node;
    uint64_t e = 0;
    for (uint64_t i = 0; i < n_ovl; ++i) {                                              /* :576-632 */
        const uint32_t* r = ovl + REC * i;
        uint32_t a0, a1, b0, b1, al, bl;
        int t = type_with_coords(r, piles, &a0, &a1, &b0, &b1, &al, &bl);
        uint32_t na = s2n[r[0]], nb = s2n[r[1]] + (r[6] & 1u);
        if (t == ORA_KAB) {                                                             /* :594-610 */
            edges[3 * e] = na; edges[3 * e + 1] = nb; edges[3 * e + 2] = a0 - b0; ++e;
            edges[3 * e] = nb ^ 1u; edges[3 * e + 1] = na ^ 1u; edges[3 * e + 2] = (bl - b1) - (al - a1); ++e;
        } else if (t == ORA_KBA) {                                                      /* :612-629 */
            edges[3 * e] = nb; edges[3 * e + 1] = na; edges[3 * e + 2] = b0 - a0; ++e;
            edges[3 * e] = na ^ 1u; edges[3 * e + 1] = nb ^ 1u; edges[3 * e + 2] = (al - a1) - (bl - b1); ++e;
        }
    }
    *n_edges = e;
}

/* suffix adjacency in ascending edge id (the order emplace_back produced, graph.cpp:604-625) */
static void build_suffix(uint32_t n_nodes, uint64_t n_edges, const uint32_t* edges, int col,
                         const uint8_t* skip, uint32_t* off, uint32_t* ids) {
    memset(off, 0, ((size_t) n_nodes + 1) * sizeof(uint32_t));
    for (uint64_t e = 0; e < n_edges; ++e) {
        if (skip && skip[e]) continue;
        ++off[edges[3 * e + col] + 1];
    }
    for (uint32_t i = 0; i < n_nodes; ++i) off[i + 1] += off[i];
    uint32_t* cur = (uint32_t*) malloc(((size_t) n_nodes + 1) * sizeof(uint32_t));
    memcpy(cur, off, ((size_t) n_nodes + 1) * sizeof(uint32_t));
    for (uint64_t e = 0; e < n_edges; ++e) {
        if (skip && skip[e]) continue;
        ids[cur[edges[3 * e + col]]++] = (uint32_t) e;
    }
    free(cur);
}

uint64_t ora_transitive(uint32_t n_nodes, uint64_t n_edges, const uint32_t* edges, uint8_t* marked) {
    uint32_t* off = (uint32_t*) malloc(((size_t) n_nodes + 1) * sizeof(uint32_t));
    uint32_t* ids = (uint32_t*) malloc((n_edges ? n_edges : 1) * sizeof(uint32_t));
    build_suffix(n_nodes, n_edges, edges, 0, NULL, off, ids);
    int64_t* candidate = (int64_t*) malloc((n_nodes ? n_nodes : 1) * sizeof(int64_t));  /* graph.cpp:1284 */
    for (uint32_t i = 0; i < n_nodes; ++i) candidate[i] = -1;
    memset(marked, 0, n_edges);
    uint64_t count = 0;
    for (uint32_t a = 0; a < n_nodes; ++a) {                                            /* :1286 */
        for (uint32_t p = off[a]; p < off[a + 1]; ++p) candidate[edges[3 * ids[p] + 1]] = ids[p];   /* :1291-1293 */
        for (uint32_t p = off[a]; p < off[a + 1]; ++p) {                                /* :1295 */
            uint32_t ab = ids[p], b = edges[3 * ab + 1];
            for (uint32_t q = off[b]; q < off[b + 1]; ++q) {                            /* :1298 */
                uint32_t bc = ids[q], c = edges[3 * bc + 1];
                int64_t ac = candidate[c];
                if (ac < 0 || marked[ac]) continue;                                     /* :1301 */
                if (ora_comparable(edges[3 * ab + 2] + edges[3 * bc + 2], edges[3 * ac + 2])) {     /* :1302-1303 */
                    marked[ac] = 1;                                                     /* :1305-1309 */
                    marked[ac ^ 1] = 1;
                    ++count;
                }
            }
        }
        for (uint32_t p = off[a]; p < off[a + 1]; ++p) candidate[edges[3 * ids[p] + 1]] = -1;       /* :1315-1317 */
    }
    free(candidate);
    free(ids);
    free(off);
    return count;
}

static int cmp_pair(const void* x, const void* y) {
    const uint32_t* a = (const uint32_t*) x;
    const uint32_t* b = (const uint32_t*) y;
    if (a[0] != b[0]) return a[0] < b[0] ? -1 : 1;
    if (a[1] != b[1]) return a[1] < b[1] ? -1 : 1;
    return 0;
}

uint64_t ora_transitive_pairs(uint64_t n_edges, const uint32_t* edges, const uint8_t* marked, uint32_t* out) {
    uint64_t n = 0;
    for (uint64_t e = 1; e < n_edges; e += 2) {                                         /* graph.cpp:1320-1329 */
        if (!marked[e]) continue;
        uint32_t s = edges[3 * e] & ~1u, d = edges[3 * e + 1] & ~1u;
        out[2 * n] = s; out[2 * n + 1] = d; ++n;
        out[2 * n] = d; out[2 * n + 1] = s; ++n;
    }
    qsort(out, n, 2 * sizeof(uint32_t), cmp_pair);                                      /* :1330 */
    return n;
}

void ora_adjacency(uint32_t n_nodes, uint64_t n_edges, const uint32_t* edges, const uint8_t* marked, int which,
                   uint32_t* off, uint32_t* ids) {
    build_suffix(n_nodes, n_edges, edges, which ? 1 : 0, marked, off, ids);
}

/* ------------------------------------------------------------------------------------------------
 * Front end, duplicate filter (SURVEY.md 8(f) row 1, first half): Graph::initialize, graph.cpp:273-303, driven by the
 * grouping loop :340-361.  Literal restatement: the same loops, the same `break`, records that lost their validity keep
 * acting on later ones (the reference only skips records whose transmute failed, i.e. nullptr).
 * a[i] with bit 31 set = overlaps[i] == nullptr.  Parity pinned: tests/golden/dups.npz holds is_valid_overlap_ of the
 * compiled reference for the same records (rala_ref dupfilter).
 * ---------------------------------------------------------------------------------------------- */
static void remove_duplicate_overlaps(const uint32_t* a, const uint32_t* b, const uint32_t* len, uint64_t begin, uint64_t end,
                                      uint8_t* valid) {
    for (uint64_t i = begin; i < end; ++i) {                                            /* :274 */
        if (a[i] & 0x80000000u) continue;                                               /* :275 nullptr */
        if (a[i] == (b[i] & 0x7FFFFFFFu)) {                                             /* :278 self overlap */
            valid[i] = 0;                                                               /* :286 */
            continue;
        }
        for (uint64_t j = i + 1; j < end; ++j) {                                        /* :290 */
            if (a[j] & 0x80000000u) continue;
            if ((b[i] & 0x7FFFFFFFu) != (b[j] & 0x7FFFFFFFu)) continue;                 /* :294 */
            if (len[i] > len[j]) {                                                      /* :299 */
                valid[j] = 0;
            } else {
                valid[i] = 0;
                break;
            }
        }
    }
}

void ora_filter_duplicates(const uint32_t* a, const uint32_t* b, const uint32_t* len, uint64_t n, uint8_t* valid) {
    uint64_t c = 0;
    for (uint64_t i = 0; i < n; ++i) valid[i] = 1;                                      /* :335 resize(..., true) */
    for (uint64_t i = 0; i < n; ++i) {
        if (a[i] & 0x80000000u) {                                                       /* :339-343 transmute failed */
            valid[i] = 0;
            continue;
        }
        while (a[c] & 0x80000000u) ++c;                                                 /* :345-347 */
        if (a[c] != a[i]) {                                                             /* :348 */
            remove_duplicate_overlaps(a, b, len, c, i, valid);
            c = i;
        }
    }
    remove_duplicate_overlaps(a, b, len, c, n, valid);                                  /* :354-356 */
}
