/* rala_b200.h — C ABI of the B200-native assembly-graph hot path (librala_b200.so).
 *
 * The reference (rvaser/rala) has no plugin / FFI interface: `rala` is one executable and the state
 * of rala::Graph is private.  The boundary is therefore cut at the two member functions its CLI
 * already calls (SURVEY.md 8b):
 *     Graph::construct               /root/reference/src/graph.cpp:427-640   (main.cpp:74)
 *     Graph::remove_transitive_edges /root/reference/src/graph.cpp:1281-1335 (via simplify, graph.cpp:646)
 * Each entry point below names the reference lines it replaces.  INTEGRATION.md shows the
 * reference-side patch (plain C++ calls; no binding layer is needed since the reference is C++).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no CUDA, torch or C++ types in any signature.
 *   - every function returns 0 on success or a negative rala_b200_status; the message is available
 *     from rala_b200_last_error().  The host shim keeps the reference's own convention on top of
 *     that: fprintf(stderr, "[rala::Graph::construct] error: %s!\n", ...); exit(1);  (cf. graph.cpp:418-421)
 *   - called from one host thread at a time per context (the reference drives this path from its
 *     main thread only, SURVEY.md finding 1).
 *   - there is NO CPU fallback: without a CUDA device rala_b200_create() fails.
 *
 * Limits: ids, coordinates and counts are 32-bit (SURVEY.md appendix D); read lengths < 2^30;
 * overlap records per context < 2^31.  Transitive reduction: a node with more than 1024 out-edges is
 * split by destination into ceil(degree / 768) hash chunks of at most 2048 distinct destinations each
 * (destination d goes to chunk ((d * 0x85EBCA6B mod 2^32) >> 12) mod chunks); more, or more than 2^32
 * block work items in one pass, is refused with RALA_B200_ERR_LIMIT.  Random ids put ~768 in a chunk.
 */
#ifndef RALA_B200_H
#define RALA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RALA_B200_ABI_VERSION 2

/* One PAF/MHAP overlap after name->id translation; replaces the numeric members of rala::Overlap
 * (overlap.hpp:104-116).  Records are passed in FILE ORDER: the position of a record is its
 * processing time in the reference's order-dependent containment removal (graph.cpp:448-480). */
typedef struct {
    uint32_t a_id, b_id;       /* sequence ids (Overlap::a_id_/b_id_ after transmute, overlap.cpp:36-82) */
    uint32_t a_begin, a_end;   /* on a's forward strand */
    uint32_t b_begin, b_end;   /* on b's forward strand */
    uint32_t flags;            /* bit0: orientation_ (overlap.cpp:18, 29); bit1: record is invalid —
                                  is_valid_overlap_ false (graph.cpp:450) or a name that is not in name_to_id_ */
} rala_ovl_t;
#define RALA_OVL_RC       1u
#define RALA_OVL_INVALID  2u

/* Valid region [begin, end) of one read's pile (Pile::begin()/end(), pile.hpp:33-42).
 * end == 0 means the pile is dead (piles_[i] == nullptr in the reference). */
typedef struct { uint32_t begin, end; } rala_pile_t;

/* per-pile flag byte */
#define RALA_PILE_HAS_HILL    1u   /* Pile::has_chimeric_hill()   (pile.hpp:107) */
#define RALA_PILE_HAS_REGION  2u   /* Pile::has_chimeric_region() (pile.hpp:121) */

/* One chimeric hill (Pile::chimeric_hills_[k]); rows grouped by ascending pile id, in the pile's own order. */
typedef struct { uint32_t pile, begin, end; } rala_hill_t;

/* One directed edge; row index = edge id, pair(e) = e ^ 1, pair(node) = node ^ 1 (graph.cpp:553-632). */
typedef struct { uint32_t src, dst, len; } rala_edge_t;

/* Overlap::type() values (overlap.hpp:27-33) + 255 for "rejected by trim / dead pile / invalid". */
enum { RALA_KX = 0, RALA_KA = 1, RALA_KB = 2, RALA_KAB = 3, RALA_KBA = 4, RALA_REJECTED = 255 };

typedef enum {
    RALA_B200_OK = 0,
    RALA_B200_ERR_CUDA = -1,        /* a CUDA call failed (message has the CUDA error string) */
    RALA_B200_ERR_ARG = -2,         /* bad argument */
    RALA_B200_ERR_STATE = -3,       /* stage called out of order */
    RALA_B200_ERR_NO_DEVICE = -4,   /* no sm_100 device: there is no CPU fallback */
    RALA_B200_ERR_LIMIT = -5        /* a documented limit was exceeded */
} rala_b200_status;

typedef struct rala_b200_ctx rala_b200_ctx;      /* one CUDA device + stream + scratch arena */
typedef struct rala_b200_graph rala_b200_graph;  /* device-resident state of one construct + reduce */

int rala_b200_abi_version(void);
int rala_b200_create(rala_b200_ctx** out, int device);
void rala_b200_destroy(rala_b200_ctx* ctx);
const char* rala_b200_last_error(const rala_b200_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t rala_b200_launch_count(const rala_b200_ctx* ctx);
/* CUDA events on the context's stream: record(0) ... record(1), then elapsed_ms waits for event 1. */
int rala_b200_event_record(rala_b200_ctx* ctx, int which);
int rala_b200_event_elapsed_ms(rala_b200_ctx* ctx, float* ms);
int rala_b200_synchronize(rala_b200_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * Stateless stages on HOST buffers (copies inside): the unit-level boundary.
 * ---------------------------------------------------------------------------------------------- */

/* Overlap::trim + Overlap::type (overlap.cpp:117-259) for n independent records: coordinates are
 * trimmed in place, type_out[i] is RALA_K* or RALA_REJECTED. */
int rala_b200_trim_classify(rala_b200_ctx* ctx, rala_ovl_t* ovl, uint64_t n,
                            const rala_pile_t* piles, uint32_t n_piles, uint8_t* type_out);

/* Graph::remove_transitive_edges (graph.cpp:1281-1318) on an arbitrary edge list:
 * marked_out[e] = 1 for every edge the reference removes; *n_pairs = its return value.
 * RALA_B200_ERR_LIMIT: the hash-chunk limit above. */
int rala_b200_transitive_reduce(rala_b200_ctx* ctx, uint32_t n_nodes, uint64_t n_edges,
                                const rala_edge_t* edges, uint8_t* marked_out, uint64_t* n_pairs);

/* The duplicate filter of the front end: Graph::initialize's remove_duplicate_overlaps (graph.cpp:273-303) as driven by
 * the grouping loop (:340-361), for n records in file order.  a_id[i] with bit 31 set (RALA_OVL_INVALID) = the record's
 * names did not resolve (the reference holds nullptr: skipped wherever it stands); bit 31 of b_id[i] (orientation) is
 * ignored; length[i] = Overlap::length() as parsed (PAF column 11, MHAP: the longer span).  valid_out[i] = what
 * is_valid_overlap_[i] holds after the pass: 0 for unresolved records, self overlaps and every record of a query group but
 * the last longest one per target.  device_ms (nullable) receives the kernel time.  SURVEY.md 8(f) row 1, first half; the
 * coverage accumulation of the same pass (:305-321, pile.cpp:274-297) is rala_b200_build_piles. */
int rala_b200_filter_duplicates(rala_b200_ctx* ctx, const uint32_t* a_id, const uint32_t* b_id, const uint32_t* length,
                                uint64_t n, uint8_t* valid_out, float* device_ms);

/* PAF text on the device (SURVEY.md 8(f) row 2): bioparser's PafParser (overlap.cpp:22-31 builds the records) and the
 * name -> id lookup of Overlap::transmute (overlap.cpp:36-82 against Graph::initialize's name_to_id_).
 * Reads: names = the read names back to back, read i = names[name_end[i-1], name_end[i]) (name_end[-1] = 0), id = i;
 * read_len[i] = its sequence length.  A name listed twice is refused (RALA_B200_ERR_ARG): which of the two name_to_id_
 * keeps is not pinned, so the library does not guess.
 * Text contract (anything else is refused with RALA_B200_ERR_ARG and a message naming the 1-based line and column; the
 * smallest offending line is reported): lines end in '\n' (the last one may lack it), fields are separated by tabs, at
 * least 12 of them; columns 2, 3, 4, 7, 8, 9, 11 are plain decimal numbers below 2^32 (leading zeros allowed); columns
 * 1 and 6 are the names, byte for byte; orientation = first byte of column 5 != '+'; columns 10, 12 and every extra
 * column (minimap2 tags, CIGARs) are never read, so a '\r' before '\n' needs no handling.  An empty line, fewer than 12
 * fields, a non-digit or a value >= 2^32 in a parsed column is refused.  Overlap::length() = column 11.
 * The text crosses PCIe in chunks of RALA_B200_PAF_CHUNK_BYTES cut behind their last '\n' (a longer line is refused with
 * RALA_B200_ERR_LIMIT); caller memory that is page-locked is uploaded in place, other memory through a pinned staging
 * pair, and the upload of one chunk overlaps the parse of the one before.  Text beyond 4 GiB is fine; records < 2^31. */
#define RALA_B200_PAF_CHUNK_BYTES (32u << 20)
typedef struct {
    uint64_t n_records;              /* lines = records, file order */
    uint64_t n_unresolved;           /* records with a name that is not among the reads (INVALID) */
    uint64_t n_length_mismatch;      /* records whose resolved name has a PAF length (column 2 or 7) other than read_len */
    uint64_t first_length_mismatch;  /* index of the first of them; UINT64_MAX when there is none */
    uint64_t n_bytes;                /* text bytes */
    uint64_t n_chunks;               /* upload chunks the text took */
} rala_b200_paf_stats_t;
/* Stateless form, like rala_b200_filter_duplicates: parse + lookup, no duplicate filter.  cols_out holds 7 columns of cap
 * words: a_id | INVALID << 31, b_id | orientation << 31, a_begin, a_end, b_begin, b_end, length (column 11).  An unresolved
 * name has id 0x7FFFFFFF and sets INVALID (bit 31 of a_id).  Length mismatches are only counted.  device_ms (nullable)
 * receives the kernel time of the line scan and the parse (name table and uploads excluded). */
int rala_b200_parse_paf(rala_b200_ctx* ctx, const char* names, const uint64_t* name_end, const uint32_t* read_len, uint32_t n_reads,
                        const char* text, uint64_t n_bytes, uint32_t* cols_out, uint64_t cap, rala_b200_paf_stats_t* stats,
                        float* device_ms);

/* MHAP text on the device (SURVEY.md 8(f) row 2): bioparser's MhapParser and the reference's MHAP Overlap constructor
 * (overlap.cpp:12-20, SURVEY.md 8(a) row a1).  Reads: read_len[i] = the sequence length of read i, in the order given to set_reads; MHAP
 * names reads by number, so no name table is built.
 * Text contract (anything else is refused with RALA_B200_ERR_ARG and a message naming the 1-based line and field; the
 * smallest offending line is reported and, within it, the smallest field):
 *   - lines end in '\n' (the last one may lack it); an empty line is refused;
 *   - fields are separated by single spaces (0x20), at least 12 of them; fields after the 12th are never read;
 *   - a '\r' that ends field 12 at the end of the line is dropped (CRLF files); anywhere else it is an ordinary byte;
 *   - fields 3 (error) and 4 (shared minmers) are never read and may be empty;
 *   - fields 1 and 2 are read ids, plain decimal with 1 <= id <= n_reads: a_id = field 1 - 1, b_id = field 2 - 1.  Id 0 or
 *     an id above n_reads is refused as "not a read id" (the reference indexes its sequences with it), so an MHAP
 *     record is never unresolved;
 *   - fields 5 (a_rc) and 9 (b_rc) are exactly "0" or "1", anything else is refused; orientation = a_rc != b_rc;
 *   - fields 6, 7, 10, 11 (a_begin, a_end, b_begin, b_end) and 8, 12 (the read lengths) are plain decimal below 2^32,
 *     leading zeros allowed; a non-digit or a value >= 2^32 is refused as in the PAF contract;
 *   - coordinates are stored as given, on either strand (no flip when a_rc = 1).  Restated from SURVEY a1, NOT pinned by
 *     a golden: n_query_rc counts the records this rule decided;
 *   - Overlap::length() = max(a_end - a_begin, b_end - b_begin), each difference mod 2^32 (the constructor's uint32_t
 *     arithmetic); the duplicate filter reads it;
 *   - fields 8 and 12 are checked against read_len as PAF columns 2 and 7 are.
 * Upload as for PAF: chunks of RALA_B200_PAF_CHUNK_BYTES cut behind their last '\n' (a longer line: RALA_B200_ERR_LIMIT),
 * page-locked caller memory in place.  No valid line is shorter than 22 bytes (ten one-byte fields, two empty ones,
 * eleven spaces, '\n'), which sizes the record buffers. */
typedef struct {
    uint64_t n_records;              /* lines = records, file order */
    uint64_t n_length_mismatch;      /* records whose field 8 or 12 differs from read_len */
    uint64_t first_length_mismatch;  /* index of the first of them; UINT64_MAX when there is none */
    uint64_t n_query_rc;             /* records with a_rc = 1: their coordinates were taken as given */
    uint64_t n_bytes;                /* text bytes */
    uint64_t n_chunks;               /* upload chunks the text took */
} rala_b200_mhap_stats_t;
/* Stateless form: parse only, no duplicate filter.  cols_out holds 7 columns of cap words: a_id (INVALID never set),
 * b_id | orientation << 31, a_begin, a_end, b_begin, b_end, length.  Length mismatches are only counted.  device_ms
 * (nullable) receives the kernel time of the line scan and the parse (uploads excluded). */
int rala_b200_parse_mhap(rala_b200_ctx* ctx, const uint32_t* read_len, uint32_t n_reads, const char* text, uint64_t n_bytes,
                         uint32_t* cols_out, uint64_t cap, rala_b200_mhap_stats_t* stats, float* device_ms);

/* The pile table from the overlap records (SURVEY.md 8(f) row 1, second half): the coverage half of Graph::initialize
 * (store_overlap_bounds + Pile::add_layers, graph.cpp:305-321, pile.cpp:274-297), the valid region and pile liveness
 * (Pile::find_valid_region, pile.cpp:307, 329) and the median (Pile::find_median).  The rule, as restated from the
 * reference's goldens (begin, end and median of every pile of tests/golden/g_*):
 *   - every record whose two names resolved counts, also those the duplicate filter drops;
 *   - it adds [a_begin + 15, a_end - 15) to read a and [b_begin + 15, b_end - 15) to read b (forward-strand coordinates as
 *     parsed, orientation ignored); coverage[x] = number of intervals containing x, x in [0, read_len);
 *   - the valid region is the longest maximal run of positions with coverage >= 4; the pile is dead (end == 0) when there
 *     is none or it is shorter than 1 260;
 *   - the median of a live pile is element size / 2 (0-based) of the sorted coverage over [begin, end) (nth_element).
 * Restated, NOT pinned (no golden has such a case), so decided here and counted in the stats:
 *   - ties between equally long runs: the first one wins (strict > of a left-to-right scan);
 *   - a run of exactly 1 260 lives.
 * Refused rather than guessed (RALA_B200_ERR_ARG; the message names the smallest offending record, 0-based, or its 1-based
 * PAF line in the session form): a self overlap, an interval that is empty or inverted after the shrink
 * (begin + 15 >= end - 15), an end beyond the read's length, a read id >= n_reads.  Coverage >= 65 536 (Pile keeps it in
 * 16 bits) is refused with RALA_B200_ERR_LIMIT.  Records < 2^29, read lengths < 2^30. */
typedef struct {
    uint64_t n_counted;      /* records that added coverage (both names resolved) */
    uint64_t n_runs;         /* constant-coverage runs over all reads (rala_b200_graph_get_coverage_runs) */
    uint32_t max_coverage;
    uint32_t n_live;         /* piles with a valid region */
    uint32_t n_tied;         /* live piles whose longest region is not unique: the first-wins rule decided them */
    uint32_t n_exact_min;    /* live piles whose region is exactly 1 260 long: the >= 1 260 rule decided them */
} rala_b200_pile_stats_t;
/* Stateless form on HOST columns in the rala_b200_graph_set_overlaps_columns layout: bit 31 of a_id marks an unresolved
 * record (it adds nothing), bit 31 of b_id is ignored.  piles_out: n_reads rows, dead = {0, 0}; medians_out (nullable):
 * n_reads values, 0 for a dead pile; stats (nullable); device_ms (nullable) = kernel time, uploads excluded. */
int rala_b200_build_piles(rala_b200_ctx* ctx, const uint32_t* a_id, const uint32_t* b_id, const uint32_t* a_begin, const uint32_t* a_end,
                          const uint32_t* b_begin, const uint32_t* b_end, uint64_t n, const uint32_t* read_len, uint32_t n_reads,
                          rala_pile_t* piles_out, uint16_t* medians_out, rala_b200_pile_stats_t* stats, float* device_ms);

/* ------------------------------------------------------------------------------------------------
 * Graph session: the drop-in for Graph::construct's hot loops and Graph::remove_transitive_edges.
 * Call order (what the patched Graph::construct does, INTEGRATION.md):
 *   set_piles, set_hills, set_overlaps        inputs produced by the unchanged Graph::initialize
 *   classify                                  graph.cpp:443-518
 *   get_hill_coverage, [host: Pile::break_over_chimeric_hills], set_piles      :704-720
 *   retrim                                    :722-736
 *   loop { get_connections, [host: components, medians, Pile::break_over_chimeric_pits], set_piles,
 *          retrim_promote(&changed) } until !changed                           :738-829
 *   finalize                                  :831-877
 *   get_piles                                 pile liveness for Sequence trimming / node creation (:527-574)
 *   build                                     :552-632 (ids, edge list, adjacency)
 *   get_edges, get_seq_to_node                re-materialise Node/Edge objects on the host
 *   transitive                                :1281-1318
 *   get_marked                                then the unchanged :1320-1334 on the host
 * rala_b200_graph_run() chains classify..transitive with the pile table frozen and no host
 * synchronisation in between (clean data: no hills, no pits).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t n_records;      /* as set */
    uint64_t n_overlaps;     /* current `overlaps` list */
    uint64_t n_internals;    /* current `internals` list */
    uint64_t n_candidates;   /* containment events of the first pass (graph.cpp:469-480) */
    uint32_t n_rounds;       /* fixed-point rounds their resolution took */
    uint32_t n_piles, n_alive_piles;
    uint32_t n_nodes;        /* nodes_.size() */
    uint64_t n_edges;        /* edges_.size() */
    uint64_t n_two_hop;      /* H = sum over edges (a->b) of outdegree(b): two-hop visits of the transitive pass */
    uint64_t n_transitive_pairs; /* return value of remove_transitive_edges */
    uint32_t n_heavy_items;  /* block-per-node work items of the last transitive pass */
    uint32_t n_final_rounds; /* fixed-point rounds of the final containment pass (graph.cpp:831-866) */
    uint64_t n_final_candidates; /* containment events of the final pass */
} rala_b200_counts_t;

int rala_b200_graph_create(rala_b200_ctx* ctx, rala_b200_graph** out);
void rala_b200_graph_destroy(rala_b200_graph* g);

int rala_b200_graph_set_overlaps(rala_b200_graph* g, const rala_ovl_t* ovl, uint64_t n);
/* The same records as six HOST COLUMNS in the layout the kernels read (replaces the same members of rala::Overlap,
 * overlap.hpp:104-116, marshalled column-wise by the host shim): 24 bytes per record cross PCIe instead of 28 and
 * land in place, with no staging copy and no transpose kernel.  Bit 31 of a_id[i] marks an INVALID record
 * (RALA_OVL_INVALID), bit 31 of b_id[i] is the orientation (RALA_OVL_RC); ids are < 2^31.  File order as above. */
int rala_b200_graph_set_overlaps_columns(rala_b200_graph* g, const uint32_t* a_id, const uint32_t* b_id,
                                         const uint32_t* a_begin, const uint32_t* a_end, const uint32_t* b_begin,
                                         const uint32_t* b_end, uint64_t n);
/* The same records in a COMPACT host form for the PCIe link: 12 bytes per record instead of 24 (the upload is 85 % of an
 * end-to-end step).  It relies on two properties of the data the reference consumes: a PAF / MHAP lists the overlaps
 * of one query together (graph.cpp:343-350 assumes the same grouping), and read coordinates of today's long reads fit
 * 16 bits (the caller checks: every coordinate < 65 536, otherwise it uses the column form).
 *   group k = records [group_end[k-1], group_end[k]) (group_end[-1] = 0), all with a_id = query_id[k] (< 2^31)
 *   b_id[i]   as in the column form (bit 31 = orientation)
 *   a_span[i] = a_begin | a_end << 16,   b_span[i] = b_begin | b_end << 16
 * An INVALID record (RALA_OVL_INVALID) is passed with both spans 0: Overlap::trim rejects it in every pass
 * (overlap.cpp:139-142), which is all "invalid" means on this path.  Expanded on the device into the column layout. */
int rala_b200_graph_set_overlaps_packed(rala_b200_graph* g, const uint32_t* query_id, const uint32_t* group_end, uint32_t n_groups,
                                        const uint32_t* b_id, const uint32_t* a_span, const uint32_t* b_span, uint64_t n);
int rala_b200_graph_set_piles(rala_b200_graph* g, const rala_pile_t* piles, const uint8_t* flags /* nullable */,
                              uint32_t n_piles);
/* The read names and lengths the PAF text is resolved against (name_to_id_ of Graph::initialize, graph.cpp:253-271, and
 * the sequence lengths transmute checks, overlap.cpp:54-59, 73-78); once per session.  Layout and refusals as
 * rala_b200_parse_paf.  The name table stays on the device.  MHAP text uses only the lengths and their order. */
int rala_b200_graph_set_reads(rala_b200_graph* g, const char* names, const uint64_t* name_end, const uint32_t* read_len, uint32_t n_reads);
/* The same from the sequence file: FASTA or FASTQ text in host memory -> the read names and lengths, parsed on the device
 * (the first half of Graph::initialize, graph.cpp:249-264).  After success every later call behaves exactly as after
 * set_reads(names, name_end, read_len) with the names and lengths the text holds, read ids in file order.  After a
 * refusal the session holds no reads (set_overlaps_paf / _mhap: RALA_B200_ERR_STATE) and no upload is in flight.
 * Text contract (anything else is refused with RALA_B200_ERR_ARG and a message naming the 1-based line and column; the
 * smallest offending line is reported, within it the smallest column):
 *   - the first byte picks the format: '>' FASTA, '@' FASTQ, anything else is refused; empty text = 0 reads;
 *   - lines end in '\n' (the last one may lack it); an empty line is refused; a '\r' anywhere is refused (CRLF handling
 *     is not pinned);
 *   - header line ('>' in FASTA, '@' in FASTQ): the name is the bytes after the marker up to the first space (0x20) or tab
 *     (0x09) or the line's end; the rest, the description, is never read.  An empty name, or a name byte < 0x20 or 0x7F,
 *     is refused.  Restated, NOT pinned: the cut at the first space or tab (the token minimap2 writes into PAF column 1);
 *     n_described counts the headers it cut;
 *   - FASTA: a line starting with '>' starts a read, every other line is a sequence line of the current read; a read's
 *     length is the sum of its sequence lines' lengths (any wrapping width); sequence bytes lie in 0x21..0x7E, each one
 *     base (case and IUPAC codes are never interpreted; a '>' inside a line is a base); a read without sequence is refused
 *     at its header line;
 *   - FASTQ: exactly four lines per read: '@' header, sequence (the FASTA byte rule, not empty), a line starting with '+'
 *     (the rest never read), quality with exactly as many bytes as the sequence (content never read, so it may start with
 *     '@' or '+').  Text that ends inside a read is refused at that read's header line; multi-line FASTQ is refused;
 *   - a name listed twice is refused as set_reads refuses it ("same name"); a read of 2^32 bases or more and a count of
 *     reads >= 2^31 are refused at the read's header line.
 * Upload as for PAF: chunks of RALA_B200_PAF_CHUNK_BYTES cut behind their last '\n' (a longer line, an unwrapped read
 * above 32 Mbp, is refused with RALA_B200_ERR_LIMIT), page-locked caller memory in place.  The text is below 2^34 bytes
 * (RALA_B200_ERR_LIMIT).  Device memory kept after the call is set_reads' (names, ends, lengths, table) plus the upload
 * staging shared with the overlap readers.  stats: nullable. */
typedef struct {
    uint32_t format;         /* 1 FASTA, 2 FASTQ, 0 empty text */
    uint32_t n_reads;
    uint64_t n_lines, n_bases, name_bytes;
    uint32_t max_len, n_described;   /* headers whose name was cut at a space / tab (restated, not pinned) */
    uint64_t n_bytes, n_chunks;
    float device_ms;         /* kernels of the call (line scan, roles, byte rules, lengths, name table); uploads excluded */
} rala_b200_reads_stats_t;
int rala_b200_graph_set_reads_text(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_reads_stats_t* stats);
/* After set_reads or set_reads_text: the session's reads in the set_reads layout (names back to back, u64 name ends,
 * u32 lengths).  *n_reads and *name_bytes (nullable) receive the sizes; each NULL buffer is skipped, so a call with NULL
 * buffers only returns the sizes.  RALA_B200_ERR_STATE when the session holds no reads. */
int rala_b200_graph_get_reads(rala_b200_graph* g, char* names_out, uint64_t* name_end_out, uint32_t* read_len_out,
                              uint32_t* n_reads, uint64_t* name_bytes);
/* PAF text in FILE ORDER -> the session's records, replacing the host parse and transmute of graph.cpp:443-451 and the
 * records set_overlaps* would receive: the text is parsed as rala_b200_parse_paf does, the duplicate filter of
 * Graph::initialize (graph.cpp:273-303, :340-361) runs on the parsed columns, and a record leaves INVALID when a name did
 * not resolve or the filter drops it.  A record that stays valid while its PAF read length (column 2 or 7) differs from
 * set_reads' length is refused (RALA_B200_ERR_ARG, naming its line): the reference exits on such a record when transmute
 * reaches it (overlap.cpp:54-59, 73-78); the library is stricter and also refuses one whose pile is already dead.  After
 * a refused call the session holds no records (classify needs a new set_overlaps*).  stats: nullable. */
int rala_b200_graph_set_overlaps_paf(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_paf_stats_t* stats);
/* MHAP text in FILE ORDER -> the session's records, as set_overlaps_paf does for PAF: parsed as rala_b200_parse_mhap,
 * then the duplicate filter, whose drops leave INVALID.  Needs set_reads first; only its lengths and count are used (ids
 * are numbers).  A record that stays valid while field 8 or 12 differs from set_reads' length is refused, naming its line.
 * After a refused call the session holds no records.  stats: nullable. */
int rala_b200_graph_set_overlaps_mhap(rala_b200_graph* g, const char* text, uint64_t n_bytes, rala_b200_mhap_stats_t* stats);
/* BGZF input: the readers above on a BGZF file (htslib's bgzip output, the usual form of indexed FASTA / FASTQ), inflated on
 * the device.  BGZF contract: the input is a series of gzip members, each with ID1 ID2 CM = 1f 8b 08, FLG = FEXTRA only,
 * and a `BC` extra subfield of SLEN 2 (other subfields may stand before or after it) holding BSIZE - 1, the member's
 * size; the members tile the input exactly; each member's trailer holds the CRC32 and ISIZE <= 65536 of its raw DEFLATE
 * stream (RFC 1951: stored, fixed and dynamic Huffman blocks), which is decoded on its own (no distance reaches into the
 * member before it).  Empty members and the end-of-file marker may stand anywhere.  The text is the concatenation of the
 * inflated members.  Refusals (RALA_B200_ERR_ARG unless noted), all worded "BGZF block N (byte offset O): <reason>" with N
 * the 0-based member and O its first byte; the smallest failing member is reported:
 *   - the input ends inside a member header; the magic is not 1f 8b 08;
 *   - a member without a BC subfield, e.g. plain `gzip` output: "the gzip member has no BC extra subfield: the input is
 *     not BGZF (blocked gzip); compress it with bgzip";
 *   - header flags other than FEXTRA; BSIZE smaller than the header and trailer, or past the end of the input;
 *     ISIZE above 65536;
 *   - in the DEFLATE stream: reading past BSIZE; BTYPE 3; a stored block whose LEN is not ~NLEN; more than 286
 *     literal/length or 30 distance codes; an over-subscribed or incomplete code (one code of length 1 is accepted); a bad
 *     code-length repeat; no end-of-block code; literal/length symbol 286 / 287 or a code not in the code; distance code
 *     30 / 31 or a code not in the code; a distance before the start of the member; more or fewer bytes than ISIZE;
 *     bytes between the end of the stream and the trailer; a CRC32 that differs from the trailer's.
 * An inflated text of 2^34 bytes or more is refused with RALA_B200_ERR_LIMIT from the headers, before any upload.  The
 * inflated text is then read exactly as the plain call reads the same text: the same chunks (RALA_B200_PAF_CHUNK_BYTES
 * cut behind their last '\n', found on the device), the same stats (n_bytes = inflated bytes; device_ms of the reads
 * stats covers the reader's kernels only), the same refusals with the same line and column, the same session afterwards.
 * Device memory kept by the session after a _bgzf call, beside the plain reader's: the compressed input, the block table
 * (40 B per member) and the inflated text, each grown to the largest call so far and freed with the session.
 * rala_b200_inflate_bgzf is stateless: with out == NULL it only walks the headers and fills stats (inflate_ms 0);
 * otherwise out receives the inflated bytes (cap smaller than the text: RALA_B200_ERR_ARG before any upload) and the
 * device memory is freed before it returns.  stats / bgzf: nullable, filled when the call succeeds. */
typedef struct {
    uint64_t n_blocks;        /* BGZF members, empty ones and the end-of-file marker included */
    uint64_t n_compressed;    /* input bytes */
    uint64_t n_bytes;         /* inflated bytes = the text the reader parsed */
    float inflate_ms;         /* device time of the inflate + CRC kernels; uploads excluded */
} rala_b200_bgzf_stats_t;
int rala_b200_inflate_bgzf(rala_b200_ctx* ctx, const uint8_t* data, uint64_t n, uint8_t* out, uint64_t cap,
                           rala_b200_bgzf_stats_t* stats);
int rala_b200_graph_set_reads_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_reads_stats_t* stats,
                                   rala_b200_bgzf_stats_t* bgzf);
int rala_b200_graph_set_overlaps_paf_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_paf_stats_t* stats,
                                          rala_b200_bgzf_stats_t* bgzf);
int rala_b200_graph_set_overlaps_mhap_bgzf(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_mhap_stats_t* stats,
                                           rala_b200_bgzf_stats_t* bgzf);
/* Plain gzip input (what gzip, pigz and `cat a.gz b.gz` write), inflated on the device.  The input is one or more gzip
 * members (RFC 1952): header 1f 8b 08 with FTEXT / FHCRC / FEXTRA / FNAME / FCOMMENT (FHCRC checked, reserved flags
 * refused), a raw DEFLATE stream whose distances never reach before the member's start, then CRC32 and ISIZE (mod 2^32),
 * both checked.  Zero bytes between and after members are skipped, as gzip.decompress does; the empty input is the empty
 * text.  An input that is BGZF throughout (the BGZF header walk succeeds) takes the BGZF path (stats bgzf = 1).
 * Refusals are RALA_B200_ERR_ARG, worded "gzip member M (byte offset O): <reason>" with M the 0-based member and O the
 * failing header or trailer, or the first byte of the failing DEFLATE block; the error earliest in the stream is reported:
 *   - bad magic or compression method; reserved flags; the input ends inside a header, a DEFLATE stream or a trailer;
 *   - every DEFLATE refusal of the BGZF path; a distance before the member's start;
 *   - header CRC; CRC32; ISIZE; non-zero bytes after the last member that start no member.
 * An inflated text of 2^34 bytes or more: RALA_B200_ERR_LIMIT.  The BGZF path refuses as the _bgzf calls do.
 * The stream is cut into chunks of chunk_bytes compressed bytes; each chunk's decode starts at the first block or member
 * boundary the finder proposes inside it and is accepted only when the decode of the chunk before it stops exactly there
 * (chunk 0 starts at the stream's start), so the output never depends on the finder being right.
 * The readers' _gzip calls read the inflated text exactly as the _bgzf calls do.  Device memory kept by the session
 * beside the BGZF path's: the per-chunk table, the decoded symbols of at most 1 GiB of text or of the longest chunk
 * (2 bytes per byte) and the member trailers, each grown to the largest call so far and freed with the session.
 * rala_b200_inflate_gzip is stateless: with out == NULL it runs the finder and the counting pass only and fills stats
 * (a stream they find malformed is decoded in full, to refuse it as the filling call does); otherwise out receives the
 * text (cap smaller than the text: RALA_B200_ERR_ARG before any of
 * it is written).  stats / gzip: nullable, filled when the call succeeds. */
typedef struct {
    uint64_t n_members;       /* gzip members (BGZF path: BGZF blocks) */
    uint64_t n_compressed;    /* input bytes */
    uint64_t n_bytes;         /* inflated bytes = the text the reader parsed */
    uint64_t n_chunks;        /* decode chunks (0 when the BGZF path ran) */
    uint64_t n_corrected;     /* chunk decodes redone because the chunk's proposed entry was not where its predecessor stopped */
    uint64_t chunk_bytes;     /* compressed bytes per chunk */
    uint32_t rounds;          /* counting rounds */
    uint32_t bgzf;            /* 1: the input was BGZF and took the block-table path */
    float inflate_ms;         /* device time of every inflate kernel; uploads excluded */
    float stage_ms[5];        /* of which: finder, counting, symbols, window chain, resolve + CRC32 */
} rala_b200_gzip_stats_t;
int rala_b200_inflate_gzip(rala_b200_ctx* ctx, const uint8_t* data, uint64_t n, uint8_t* out, uint64_t cap,
                           rala_b200_gzip_stats_t* stats);
int rala_b200_graph_set_reads_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_reads_stats_t* stats,
                                   rala_b200_gzip_stats_t* gzip);
int rala_b200_graph_set_overlaps_paf_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_paf_stats_t* stats,
                                          rala_b200_gzip_stats_t* gzip);
int rala_b200_graph_set_overlaps_mhap_gzip(rala_b200_graph* g, const uint8_t* data, uint64_t n, rala_b200_mhap_stats_t* stats,
                                           rala_b200_gzip_stats_t* gzip);
/* The pile table of the reads given to set_reads, built on the device (rule and refusals as rala_b200_build_piles) from
 * the records of the last successful set_overlaps_paf or set_overlaps_mhap, counted as parsed: before the duplicate
 * filter.  A refused record is named by its line in that text ("PAF line N" / "MHAP line N").  It is installed as
 * set_piles(piles, NULL, n_reads) would (flags 0; the hills are left as they are) and the next classify / run uses it.
 * RALA_B200_ERR_STATE after set_overlaps / _columns / _packed (their records have the filter folded in) or set_reads.
 * A refused call changes nothing in the session.  stats: nullable. */
int rala_b200_graph_build_piles(rala_b200_graph* g, rala_b200_pile_stats_t* stats);
/* After build_piles: the median of every pile it built (n_reads values of set_reads, 0 = dead pile), what Pile::find_median
 * leaves.  The medians and runs below belong to the last successful build_piles, whatever set_piles did since. */
int rala_b200_graph_get_medians(rala_b200_graph* g, uint16_t* out);
/* After build_piles: the constant-coverage runs of every read over [0, read_len), for the host's chimeric pit and hill
 * detection (Pile::find_chimeric_pits / find_chimeric_hills expand them into Pile::data_).  Runs are maximal (the coverage
 * changes at every run start); read r has the runs [run_off[r], run_off[r + 1]), run k covers [run_begin[k], run_begin[k + 1])
 * or up to read_len for the read's last one, with coverage run_cov[k].  run_off (n_reads + 1 words) is always written;
 * run_begin and run_cov are written when both are given and cap >= run_off[n_piles] (RALA_B200_ERR_ARG when cap is smaller),
 * so a first call with NULL buffers asks for the size. */
int rala_b200_graph_get_coverage_runs(rala_b200_graph* g, uint32_t* run_off, uint32_t* run_begin, uint16_t* run_cov, uint64_t cap);
/* Optional: have build / transitive / run write their results STRAIGHT into caller memory the GPU can address
 * (cudaHostAlloc / cudaHostRegister'ed host memory, or device memory): the rala_edge_t rows (graph.cpp:576-632)
 * leave as soon as the edge list exists, on a forked stream beside the CSR build and the transitive pass, and the
 * removed-edge marks (graph.cpp:1305-1309) as they are finalised.  Nothing beyond the given capacities (in edges)
 * is written; the counts come from rala_b200_graph_counts.  The buffers hold valid data once the stream has been
 * synchronised (rala_b200_graph_counts / rala_b200_synchronize).  NULL switches an output off again; pageable
 * memory is refused (RALA_B200_ERR_ARG): use get_edges / get_marked for it.  The caller keeps the buffers alive
 * (and pinned) until it has switched them off or destroyed the session: every later build / run writes into them. */
int rala_b200_graph_set_outputs(rala_b200_graph* g, rala_edge_t* edges_out, uint64_t edges_cap, uint8_t* marked_out,
                                uint64_t marked_cap);
int rala_b200_graph_set_hills(rala_b200_graph* g, const rala_hill_t* hills, uint32_t n_hills);

int rala_b200_graph_classify(rala_b200_graph* g);
int rala_b200_graph_retrim(rala_b200_graph* g);
int rala_b200_graph_retrim_promote(rala_b200_graph* g, int* is_changed);
int rala_b200_graph_finalize(rala_b200_graph* g);
int rala_b200_graph_build(rala_b200_graph* g);
int rala_b200_graph_transitive(rala_b200_graph* g);
int rala_b200_graph_run(rala_b200_graph* g);
/* rala_b200_graph_run() replays a captured CUDA graph of the whole chain once it has run a session shape (buffers,
 * sizes, first run after set_piles or not) eagerly: one launch instead of ~45 dependent stream operations.  The
 * per-stage timers of rala_b200_graph_stage_ms() are not recorded inside a graph: pass enabled = 0 before the
 * runs you want stage times for.  Default: enabled. */
int rala_b200_graph_use_cuda_graph(rala_b200_graph* g, int enabled);

/* synchronises the stream and reads the device-side counters */
int rala_b200_graph_counts(rala_b200_graph* g, rala_b200_counts_t* out);

int rala_b200_graph_get_hill_coverage(rala_b200_graph* g, uint32_t* cov_out /* n_hills */);
int rala_b200_graph_get_piles(rala_b200_graph* g, rala_pile_t* piles_out /* n_piles */);
/* (a_id, b_id) of every entry of `overlaps`, for the host's component search (graph.cpp:740-744) */
int rala_b200_graph_get_connections(rala_b200_graph* g, uint32_t* ab_out /* 2 * n_overlaps */);
int rala_b200_graph_get_lists(rala_b200_graph* g, rala_ovl_t* overlaps_out /* nullable */,
                              rala_ovl_t* internals_out /* nullable */);
/* Replaces the device `overlaps` list after finalize by a host-filtered copy of it, same order: what
 * Graph::preprocess(overlaps, sensitive_overlaps_path) (graph.cpp:523, 882-1054, the -s option) leaves. */
int rala_b200_graph_set_kept_overlaps(rala_b200_graph* g, const rala_ovl_t* kept, uint64_t n);
int rala_b200_graph_get_seq_to_node(rala_b200_graph* g, uint32_t* out /* n_piles; 0xFFFFFFFF = dead */);
int rala_b200_graph_get_edges(rala_b200_graph* g, rala_edge_t* out /* n_edges */);
int rala_b200_graph_get_marked(rala_b200_graph* g, uint8_t* out /* n_edges */);
/* The CSR adjacency build writes for the transitive pass (read-only there, so the same after transitive): node v's out-edges
 * are slots row_ptr_out[v] .. row_ptr_out[v + 1] of col_out (pairs {destination node, length}) and col_eid_out (their edge
 * ids), in no particular order inside a row.  row_ptr_out: n_nodes + 1 words, col_out: 2 x n_edges, col_eid_out: n_edges.
 * After build (RALA_B200_ERR_STATE before); synchronises the session's stream. */
int rala_b200_graph_get_csr(rala_b200_graph* g, uint32_t* row_ptr_out, uint32_t* col_out, uint32_t* col_eid_out);
/* Adjacency VIEW, built on the device: off_out[v] .. off_out[v + 1] delimit, in ids_out, the ids of node v's out-edges (which = 0:
 * suffix_edges_, graph.cpp:603 / 625) or in-edges (which = 1: prefix_edges_, :605-606 / 622-624) in ascending edge id, as the
 * reference keeps them; with skip_marked != 0 (after transitive) without the removed edges: the adjacency
 * Graph::remove_marked_objects leaves (graph.cpp:2118-2151).  off_out: n_nodes + 1 words, ids_out: n_edges words. */
int rala_b200_graph_get_adjacency(rala_b200_graph* g, int which, int skip_marked, uint32_t* off_out, uint32_t* ids_out, uint64_t* n_ids_out);

/* Device time of the last run of each stage, CUDA events on the context's stream (ms).
 * Order: classify, retrim, finalize, build, transitive (whole stages), then single kernels:
 * K1 events kernel (first pass over the records), K1b containment fixed point, K3 transitive kernels
 * (light + heavy), K1 survivors kernel (second pass over the records).  For bench.py's roofline object. */
#define RALA_B200_N_STAGES 9
int rala_b200_graph_stage_ms(rala_b200_graph* g, float* ms_out /* RALA_B200_N_STAGES */);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU phases: one process per GPU, records sharded by contiguous FILE RANGE (shard r holds
 * records [t0_r, t0_r + n_r)), pile table replicated.  The reference has no distributed code; this
 * is the partition BASELINE.json's north_star asks for: work split by overlap range (classify) and
 * by source-node range (transitive), the event lists and the edge list all-gathered, the marks
 * merged with an all-reduce(max) (= OR on 0/1 bytes).  The collectives are the caller's
 * (rala_b200/multi.py uses torch.distributed / NCCL); every pointer below is a DEVICE pointer of
 * the caller's exchange buffer.  No call synchronises with the host: element counts travel inside the
 * exchange blocks and the time bases of the final pass are computed on the device.
 *
 *   set_shard; set_piles; set_overlaps(local records)
 *   phase_events              -> export_padded(0), [all-gather], import_gathered(0) (all ranks' blocks)
 *   phase_resolve(1)          ordered containment of graph.cpp:469-480 on the union of the events (replicated)
 *   phase_survivors           -> export_list_counts, [all-gather]
 *   phase_final_events_gathered   time = global position in overlaps ++ internals (graph.cpp:831-866)
 *                             -> export_padded(0), [all-gather], import_gathered(0)
 *   phase_resolve(0)
 *   phase_emit_edges          -> export_padded(1), [all-gather], import_gathered(1) (global edge-id order = rank order)
 *   phase_csr                 CSR of the whole graph, replicated (two-hop lookups cross shards)
 *   phase_transitive          T(e) for candidate edges whose source node this rank owns
 *   export_marks, [all-reduce(max)], phase_marks     marked(e) = T(e) | T(e^1)
 *
 * Exchange blocks (rala_b200_exchange_block_words(kind, cap) = 3 * cap + 4 words):
 *   kind 0, containment events: [n clamped to cap | overflow flag | n | 0 | victim [cap] | container [cap] | time [cap]]
 *   kind 1, edges: the same layout with src | dst | len
 * n is the exporting rank's element count.  d_gathered = the `world` blocks of an all-gather, in rank order.  A count
 * beyond `cap` raises the session's overflow flag (reported by rala_b200_graph_counts); the largest word 2 of the
 * gathered blocks is the smallest `cap` that fits.
 * ---------------------------------------------------------------------------------------------- */
/* a context that enqueues on the caller's CUDA stream (cudaStream_t), e.g. torch's current stream */
int rala_b200_create_on_stream(rala_b200_ctx** out, int device, void* cuda_stream);
/* After set_shard with world > 1 the session holds one rank's share of a step: rala_b200_graph_build, _transitive and
 * _run return RALA_B200_ERR_STATE (they would give a partial edge list or marks); use the phase calls below, or the
 * multi-GPU session.  set_shard(g, 0, 0, 1) makes it a whole session again. */
int rala_b200_graph_set_shard(rala_b200_graph* g, uint32_t t0, int rank, int world);
int rala_b200_graph_phase_events(rala_b200_graph* g);
int rala_b200_graph_phase_resolve(rala_b200_graph* g, int first_pass);
int rala_b200_graph_phase_survivors(rala_b200_graph* g);
int rala_b200_graph_phase_emit_edges(rala_b200_graph* g);
int rala_b200_graph_phase_csr(rala_b200_graph* g);
uint64_t rala_b200_exchange_block_words(int kind, uint32_t cap);
int rala_b200_graph_export_padded(rala_b200_graph* g, int kind, uint32_t* d_block, uint32_t cap);
int rala_b200_graph_import_gathered(rala_b200_graph* g, int kind, const uint32_t* d_gathered, uint32_t cap, int world);
int rala_b200_graph_export_list_counts(rala_b200_graph* g, uint32_t* d_pair /* n_overlaps, n_internals */);
int rala_b200_graph_phase_final_events_gathered(rala_b200_graph* g, const uint32_t* d_counts /* world x 2 */, int world);
int rala_b200_graph_phase_transitive(rala_b200_graph* g);
int rala_b200_graph_export_marks(rala_b200_graph* g, uint8_t* d_T, uint32_t n);
int rala_b200_graph_phase_marks(rala_b200_graph* g, const uint8_t* d_T, uint32_t n);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU session (ABI version 2): Graph::construct's hot loops + Graph::remove_transitive_edges on `world` ranks,
 * one rank per GPU, with the whole orchestration INSIDE the library.  The reference has no distributed code
 * (rvaser/rala is one process); this is the partition BASELINE.json's north_star names: overlap records by
 * contiguous FILE RANGE (classification), piles / nodes by id range (ordered containment of graph.cpp:469-480 and
 * 831-866, adjacency rows of :576-632, the two-hop test of :1281-1318), CSR of the whole graph replicated.
 *
 * Exchange steps are kernels that write straight into the peer GPUs' memory over NVLink (peer access inside one
 * process, CUDA IPC between processes) separated by device-side flag barriers: one step enqueues kernels only, has
 * no host synchronisation and no library collective, and is replayed as one CUDA graph per rank.
 *
 *   single process, n GPUs (the drop-in CLI, host/graph_b200.cpp):
 *       rala_b200_multi_create(&m, devices, n, 0, n); set_piles; set_overlaps(k, shard k) for every k;
 *       rala_b200_multi_plan(m);  rala_b200_multi_run(m);  get_* ...
 *   one process per GPU (torch.distributed / MPI launchers; rala_b200/multi.py):
 *       rala_b200_multi_create(&m, &device, 1, rank, world); set_piles; set_overlaps(0, own shard);
 *       default_caps -> [max over ranks] -> reserve -> export_handle -> [all-gather handles] -> import_handles;
 *       run; synchronize; demand -> [max over ranks]: re-reserve with larger capacities if something did not fit.
 *
 * A device id may be listed more than once (several ranks share a GPU): that is how the parity tests cover
 * world > 1 on a one-GPU box.  rala_b200_multi_run is the frozen-pile chain (no hills, no host pile breaking between
 * the passes: what rala_b200_graph_run executes).  Pile tables that change between the passes (hill counters, pile
 * breaking, promoted internals) take the STAGED calls below, the same boundaries as the single session's:
 *
 *   set_piles, set_hills, set_overlaps(k, shard k) ...; plan (or reserve + handles)
 *   classify                                  graph.cpp:443-518; hill counters summed over the ranks on the device
 *   get_hill_coverage, [host: break_over_chimeric_hills], set_piles           :704-720
 *   retrim                                    :722-736
 *   loop { get_lists (connections), [host: pits], set_piles, retrim_promote(&changed) } until !changed   :738-829
 *   finish                                    :831-877, 552-632, 1281-1318
 *   synchronize, demand                       the capacities were planned from a frozen step: if the staged passes
 *                                             needed more (fits = 0, or counts fails), the results are incomplete;
 *                                             reserve with the reported capacities and construct again
 *   get_lists, edge_runs, get_edges, get_marked, get_seq_to_node ...
 *
 * Every staged call is made by every process with the same arguments and synchronises with the host; the counts it
 * needs from other ranks (hill totals, list counts, is_changed) arrive through the exchange arenas, so all processes
 * see the same values without a host collective.  Promotions go to the END of the global `overlaps` (graph.cpp:818):
 * with shards in rank order that list is segment-major (segment 0: every rank's entries of the first pass in rank
 * order; segment k: what the k-th round that promoted anything promoted, in rank order), and a rank's edges are one run
 * of global ids per segment.  Read ids, coordinates and counts 32-bit as above.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rala_b200_multi rala_b200_multi;

#define RALA_B200_MAX_RANKS 16
/* segments of the staged `overlaps` list: the first pass plus at most 63 pit rounds that promote something
 * (rala_b200_multi_retrim_promote fails with RALA_B200_ERR_LIMIT beyond, and the session's lists are void) */
#define RALA_B200_MAX_SEGMENTS 64
/* capacities of the exchange buffers (identical on every rank) */
enum { RALA_B200_CAP_EVENTS = 0,   /* containment events one rank sends to one owner */
       RALA_B200_CAP_EDGES,        /* edges one rank sends to one owner */
       RALA_B200_CAP_SLICE,        /* edges of one rank's CSR slice */
       RALA_B200_CAP_ROUNDS,       /* sweeps after which the resolution of the first containment pass gives up (it ends by itself) */
       RALA_B200_CAP_FINAL_ROUNDS, /* the same for the final containment pass */
       RALA_B200_CAP_LOCAL_EDGES,  /* edges one rank emits */
       RALA_B200_N_CAPS };

typedef struct {
    int world, n_local;
    uint64_t n_records;            /* records of the local ranks */
    uint32_t n_piles, n_alive_piles, n_nodes;
    uint64_t n_edges;              /* edges_.size(): all ranks (every rank knows the total) */
    uint64_t n_local_edges;        /* edges emitted by the local ranks */
    uint64_t n_candidates, n_final_candidates;   /* containment events emitted by the local ranks */
    uint32_t n_rounds, n_final_rounds;           /* resolution rounds needed (same on every rank) */
    uint64_t n_two_hop, n_transitive_pairs;      /* local ranks' share (sum over all ranks = the reference's values) */
    uint32_t n_heavy_items;
    uint32_t fabric_error;         /* 0, or bits: 1 barrier timeout, 2 rounds exhausted, 4 exchange buffer too small */
} rala_b200_multi_counts_t;

/* ranks [first_rank, first_rank + n_local) of `world` live in this process, local rank k on devices[k] */
int rala_b200_multi_create(rala_b200_multi** out, const int* devices, int n_local, int first_rank, int world);
void rala_b200_multi_destroy(rala_b200_multi* m);
const char* rala_b200_multi_last_error(const rala_b200_multi* m);
/* replicated pile table (every local rank gets a copy); as rala_b200_graph_set_piles: called after classify it replaces
 * the table every later staged pass trims against */
int rala_b200_multi_set_piles(rala_b200_multi* m, const rala_pile_t* piles, const uint8_t* flags, uint32_t n_piles);
/* replicated hill rows, as rala_b200_graph_set_hills; only the staged classify counts them (rala_b200_multi_run ignores
 * them).  More hills than the exchange arenas were reserved for: reserve again. */
int rala_b200_multi_set_hills(rala_b200_multi* m, const rala_hill_t* hills, uint32_t n_hills);
/* shard of local rank k: records [t0, t0 + n) of the file, in file order */
int rala_b200_multi_set_overlaps(rala_b200_multi* m, int k, const rala_ovl_t* ovl, uint64_t n, uint64_t t0);
int rala_b200_multi_set_overlaps_columns(rala_b200_multi* m, int k, const uint32_t* a_id, const uint32_t* b_id, const uint32_t* a_begin,
                                         const uint32_t* a_end, const uint32_t* b_begin, const uint32_t* b_end, uint64_t n, uint64_t t0);
int rala_b200_multi_set_overlaps_packed(rala_b200_multi* m, int k, const uint32_t* query_id, const uint32_t* group_end, uint32_t n_groups,
                                        const uint32_t* b_id, const uint32_t* a_span, const uint32_t* b_span, uint64_t n, uint64_t t0);
/* as rala_b200_graph_set_outputs, for the edges local rank k emits (edge ids rala_b200_multi_edge_range) and their marks */
int rala_b200_multi_set_outputs(rala_b200_multi* m, int k, rala_edge_t* edges_out, uint64_t edges_cap, uint8_t* marked_out,
                                uint64_t marked_cap);
/* capacities this process would choose for its own shards (take the maximum over all processes) */
int rala_b200_multi_default_caps(rala_b200_multi* m, uint64_t* caps /* RALA_B200_N_CAPS */);
/* (re)allocate the exchange arenas; with all ranks in one process this also connects them */
int rala_b200_multi_reserve(rala_b200_multi* m, const uint64_t* caps /* RALA_B200_N_CAPS */);
/* change the sweep limits of the two containment resolutions without touching the arenas */
int rala_b200_multi_set_rounds(rala_b200_multi* m, uint32_t rounds, uint32_t final_rounds);
/* one process per GPU: 64-byte CUDA IPC handle of local rank k's arena / the handles of all `world` ranks in rank order */
int rala_b200_multi_export_handle(rala_b200_multi* m, int k, void* handle64);
int rala_b200_multi_import_handles(rala_b200_multi* m, const void* handles /* world x 64 bytes */);
/* one step on every local rank: classify .. transitive.  Enqueues only (replays one CUDA graph per rank from the
 * third call with the same inputs on). */
int rala_b200_multi_run(rala_b200_multi* m);
int rala_b200_multi_use_cuda_graph(rala_b200_multi* m, int enabled);
/* How long a rank waits for its peers at a device-side barrier before it gives up (default 10 000 ms).  After a timeout
 * the step's results are void, no later barrier waits, and demand / counts report RALA_B200_ERR_CUDA. */
int rala_b200_multi_set_barrier_timeout_ms(rala_b200_multi* m, uint32_t ms);
int rala_b200_multi_synchronize(rala_b200_multi* m);
/* after synchronize: what the last step needed (per capacity; rounds: rounds needed) and whether everything fit */
int rala_b200_multi_demand(rala_b200_multi* m, uint64_t* need /* RALA_B200_N_CAPS */, int* fits);
/* all ranks in one process: reserve with the default capacities, run, grow what did not fit, until a step fits */
int rala_b200_multi_plan(rala_b200_multi* m);
int rala_b200_multi_counts(rala_b200_multi* m, rala_b200_multi_counts_t* out);
/* results of local rank k: the edges it emitted are edge ids [*first_edge, *first_edge + *n) (rows in id order).  After a
 * staged construct whose promotions gave rank k more than one run of ids: RALA_B200_ERR_STATE (use edge_runs). */
int rala_b200_multi_edge_range(rala_b200_multi* m, int k, uint64_t* first_edge, uint64_t* n);
/* the global id runs of the rows get_edges(k) / get_marked(k) return, in that order: (first id, count) pairs, adjacent
 * runs merged; first_and_count_out (nullable: count only) holds 2 x RALA_B200_MAX_SEGMENTS values */
int rala_b200_multi_edge_runs(rala_b200_multi* m, int k, uint64_t* first_and_count_out, uint32_t* n_runs_out);

/* staged construct (see above); each call runs on every local rank and returns when they are done */
int rala_b200_multi_classify(rala_b200_multi* m);
int rala_b200_multi_retrim(rala_b200_multi* m);
/* *is_changed (nullable): did the retrim of `overlaps` drop an entry on any rank (graph.cpp:801-807), the same on every rank */
int rala_b200_multi_retrim_promote(rala_b200_multi* m, int* is_changed);
int rala_b200_multi_finish(rala_b200_multi* m);
/* hill counters of the first pass summed over all ranks (n_hills), as local rank k holds them */
int rala_b200_multi_get_hill_coverage(rala_b200_multi* m, int k, uint32_t* cov_out);
/* local rank k's entries of `overlaps` / `internals` (nullable) with their positions in the global lists (nullable);
 * counts[0], counts[1] = how many (always written).  After finish: the final lists of graph.cpp:867-877. */
int rala_b200_multi_get_lists(rala_b200_multi* m, int k, rala_ovl_t* ovl_out, uint64_t* ovl_pos_out, rala_ovl_t* int_out,
                              uint64_t* int_pos_out, uint64_t* counts);
int rala_b200_multi_get_edges(rala_b200_multi* m, int k, rala_edge_t* out);
int rala_b200_multi_get_marked(rala_b200_multi* m, int k, uint8_t* out);
int rala_b200_multi_get_seq_to_node(rala_b200_multi* m, uint32_t* out /* n_piles */);
int rala_b200_multi_get_piles(rala_b200_multi* m, rala_pile_t* out /* n_piles */);
/* CUDA events on every local rank's stream; elapsed = max over the local ranks */
int rala_b200_multi_event_record(rala_b200_multi* m, int which);
int rala_b200_multi_event_elapsed_ms(rala_b200_multi* m, float* ms);
uint64_t rala_b200_multi_launch_count(const rala_b200_multi* m);
/* Diagnostics: device timestamps (ns) of the last barriers of local rank k, oldest first, as pairs (barrier kernel started,
 * every peer had arrived); out holds 2 x 128 values, *n_out = number of valid pairs.  Synchronises. */
int rala_b200_multi_barrier_log(rala_b200_multi* m, int k, uint64_t* out, uint32_t* n_out);
/* Diagnostics: the sweeps of the last containment resolution (pass 0 first, 1 final) of local rank k as pairs (victims still
 * open when the sweep started, ns since the kernel started when it ended); out holds 2 x 48 values. Synchronises. */
int rala_b200_multi_sweep_log(rala_b200_multi* m, int k, int pass, uint64_t* out, uint32_t* n_out);
/* device time of the stages of the last EAGER step of local rank k (as rala_b200_graph_stage_ms) */
int rala_b200_multi_stage_ms(rala_b200_multi* m, int k, float* ms_out /* RALA_B200_N_STAGES */);

#ifdef __cplusplus
}
#endif
#endif
