/* tests/piles_oracle.c — TEST INFRASTRUCTURE: a plain-C, sequential restatement of the coverage half of rala's
 * Graph::initialize, read by read as the reference does it:
 *   store_overlap_bounds (graph.cpp:305-321): per read, the bound list (begin + 15) << 1 and (end - 15) << 1 | 1 of every
 *     record whose two names resolved (also those the duplicate filter drops);
 *   Pile::add_layers (pile.cpp:274-297): the bounds sorted, then the walk that adds the running coverage to every base
 *     between two bounds, into a uint16 buffer of the read's length;
 *   Pile::find_valid_region (pile.cpp:307): the longest run with coverage >= 4, strict > (the first longest wins); a pile
 *     whose region is shorter than 1 260 dies (:329);
 *   Pile::find_median: element size / 2 of the region's sorted values (nth_element), found by counting the values.
 * One read at a time, never a genome-sized array.  Refusals as include/rala_b200.h rala_b200_build_piles; the first
 * offending record in file order is reported.  Runs: the maximal constant-coverage runs of every read's buffer. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { ERR_ID = 1, ERR_SELF, ERR_A_EMPTY, ERR_A_BEYOND, ERR_B_EMPTY, ERR_B_BEYOND };

static int cmp_u32(const void* x, const void* y) {
    const uint32_t a = *(const uint32_t*) x, b = *(const uint32_t*) y;
    return a < b ? -1 : a > b;
}

static uint32_t check(uint32_t a, uint32_t b, uint64_t ab, uint64_t ae, uint64_t bb, uint64_t be, const uint32_t* read_len, uint32_t n_reads) {
    if (a >= n_reads || b >= n_reads) return ERR_ID;
    if (a == b) return ERR_SELF;
    if (ab + 30 >= ae) return ERR_A_EMPTY;
    if (ae > read_len[a]) return ERR_A_BEYOND;
    if (bb + 30 >= be) return ERR_B_EMPTY;
    if (be > read_len[b]) return ERR_B_BEYOND;
    return 0;
}

/* cols: 6 x n words (a_id | unresolved << 31, b_id | orientation << 31, a_begin, a_end, b_begin, b_end).
 * piles: 2 x n_reads, medians: n_reads; stats: counted, runs, max coverage, live, tied, exact 1 260.
 * run_off (n_reads + 1), run_begin / run_cov (run_cap): nullable; the runs are written while they fit.
 * Returns 0; -1 refused (err[0] = record, err[1] = kind); -2 coverage >= 65 536 (err[0] = the coverage seen); -3 no memory. */
int ora_build_piles(const uint32_t* cols, uint64_t n, const uint32_t* read_len, uint32_t n_reads, uint32_t* piles, uint16_t* medians,
                    uint64_t* stats, uint32_t* run_off, uint32_t* run_begin, uint16_t* run_cov, uint64_t run_cap, uint64_t* err) {
    const uint32_t *ca = cols, *cb = cols + n, *cab = cols + 2 * n, *cae = cols + 3 * n, *cbb = cols + 4 * n, *cbe = cols + 5 * n;
    memset(stats, 0, 6 * sizeof(uint64_t));
    uint64_t* cnt = calloc((size_t) n_reads + 1, sizeof(uint64_t));
    if (!cnt) return -3;
    for (uint64_t i = 0; i < n; ++i) {
        if (ca[i] >> 31) continue;
        const uint32_t a = ca[i], b = cb[i] & 0x7FFFFFFFu;
        const uint32_t k = check(a, b, cab[i], cae[i], cbb[i], cbe[i], read_len, n_reads);
        if (k) {
            err[0] = i;
            err[1] = k;
            free(cnt);
            return -1;
        }
        cnt[a] += 2;
        cnt[b] += 2;
        stats[0]++;
    }
    /* the bound lists, read by read (CSR) */
    uint64_t total = 0;
    for (uint32_t r = 0; r < n_reads; ++r) {
        const uint64_t c = cnt[r];
        cnt[r] = total;
        total += c;
    }
    cnt[n_reads] = total;
    uint32_t* bounds = malloc((total + 1) * sizeof(uint32_t));
    uint64_t* fill = malloc(((size_t) n_reads + 1) * sizeof(uint64_t));
    uint32_t max_len = 0;
    for (uint32_t r = 0; r < n_reads; ++r) max_len = read_len[r] > max_len ? read_len[r] : max_len;
    uint16_t* data = malloc(((size_t) max_len + 1) * sizeof(uint16_t));
    uint32_t* hist = malloc(65536 * sizeof(uint32_t));
    if (!bounds || !fill || !data || !hist) {
        free(cnt); free(bounds); free(fill); free(data); free(hist);
        return -3;
    }
    memcpy(fill, cnt, ((size_t) n_reads + 1) * sizeof(uint64_t));
    for (uint64_t i = 0; i < n; ++i) {
        if (ca[i] >> 31) continue;
        const uint32_t a = ca[i], b = cb[i] & 0x7FFFFFFFu;
        bounds[fill[a]++] = (cab[i] + 15) << 1;
        bounds[fill[a]++] = (cae[i] - 15) << 1 | 1;
        bounds[fill[b]++] = (cbb[i] + 15) << 1;
        bounds[fill[b]++] = (cbe[i] - 15) << 1 | 1;
    }
    free(fill);
    uint64_t runs = 0;
    int rc = 0;
    for (uint32_t r = 0; r < n_reads && !rc; ++r) {
        const uint32_t len = read_len[r];
        uint32_t* bd = bounds + cnt[r];
        const uint64_t nb = cnt[r + 1] - cnt[r];
        memset(data, 0, (size_t) len * sizeof(uint16_t));
        /* add_layers */
        qsort(bd, nb, sizeof(uint32_t), cmp_u32);
        uint32_t coverage = 0, last = 0;
        for (uint64_t j = 0; j < nb; ++j) {
            const uint32_t pos = bd[j] >> 1;
            if (coverage > 0) {
                if (coverage >= 65536 && pos > last) {
                    err[0] = coverage;
                    rc = -2;
                    break;
                }
                for (uint32_t x = last; x < pos; ++x) data[x] += (uint16_t) coverage;
            }
            last = pos;
            if (bd[j] & 1) --coverage; else ++coverage;
        }
        if (rc) break;
        /* runs and the largest value */
        if (run_off) run_off[r] = (uint32_t) runs;
        for (uint32_t x = 0; x < len; ++x) {
            if (data[x] > stats[2]) stats[2] = data[x];
            if (x == 0 || data[x] != data[x - 1]) {
                if (run_begin && runs < run_cap) {
                    run_begin[runs] = x;
                    run_cov[runs] = data[x];
                }
                ++runs;
            }
        }
        /* find_valid_region */
        uint32_t nbeg = 0, nend = 0, cur = 0, n_best = 0;
        int found = 0;
        for (uint32_t x = 0; x <= len; ++x) {
            const int hi = x < len && data[x] >= 4;
            if (!found && hi) {
                cur = x;
                found = 1;
            } else if (found && !hi) {
                if (x - cur > nend - nbeg) {
                    nbeg = cur;
                    nend = x;
                    n_best = 1;
                } else if (x - cur == nend - nbeg) {
                    ++n_best;
                }
                found = 0;
            }
        }
        const int alive = nend - nbeg >= 1260;
        piles[2 * r] = alive ? nbeg : 0;
        piles[2 * r + 1] = alive ? nend : 0;
        medians[r] = 0;
        if (alive) {
            /* find_median: the element nth_element puts at size / 2 */
            uint32_t lo = 65535, hi = 0;
            for (uint32_t x = nbeg; x < nend; ++x) {
                lo = data[x] < lo ? data[x] : lo;
                hi = data[x] > hi ? data[x] : hi;
            }
            memset(hist + lo, 0, (size_t) (hi - lo + 1) * sizeof(uint32_t));
            for (uint32_t x = nbeg; x < nend; ++x) hist[data[x]]++;
            const uint32_t kth = (nend - nbeg) / 2;
            uint32_t seen = 0, v = lo;
            for (; v <= hi; ++v) {
                seen += hist[v];
                if (seen > kth) break;
            }
            medians[r] = (uint16_t) v;
            stats[3]++;
            if (n_best > 1) stats[4]++;
            if (nend - nbeg == 1260) stats[5]++;
        }
    }
    if (run_off && !rc) run_off[n_reads] = (uint32_t) runs;
    stats[1] = runs;
    free(cnt); free(bounds); free(data); free(hist);
    return rc;
}
