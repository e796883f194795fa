/*
 * gxalign.h -- C ABI of libgxalign: B200-native (sm_100a) affine-gap global (NW) / local (SW)
 * alignment, the drop-in for the one hot path of nlaha/genomics-rs:
 *
 *     alignment_table(&SequenceContainer,&Scores,is_local,reverse) -> (Array2<AlignmentCell>, usize)
 *                                                        /root/reference/src/alignment/algo.rs:151-156
 *     retrace(&SequenceContainer, Array2<AlignmentCell>, is_local) -> AlignedSequences
 *                                                        /root/reference/src/alignment/algo.rs:287-291
 *
 * The reference joins the two with an owned 48-byte-per-cell table (main.rs:143-150).  That table
 * cannot exist on a GPU design, so this boundary fuses the two calls: inputs are the first two
 * sequences as bytes + Scores + is_local, the output is the content of AlignedSequences
 * (algo.rs:135-146).  Results are bit-identical to the reference for every input that satisfies
 * the preconditions checked by gx_check_scores() -- including the reference's non-textbook
 * tie-breaks (SURVEY.md 3.3).  There is no CPU fallback: every entry point fails with
 * GX_ERR_NO_DEVICE / GX_ERR_CUDA when no sm_100 device is usable.
 *
 * Plain C, plain pointers and sizes; the library owns all device memory and pinned staging.
 * Calls on one context are serialised internally; callers may be multi-threaded.
 * The library never writes to stdout/stderr and never throws or aborts across the ABI.
 */
#ifndef GXALIGN_H
#define GXALIGN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (replace the reference's panic!/exit(1): algo.rs:168-169,407-408; config.rs:26,34) */
enum {
    GX_OK = 0,
    GX_ERR_ARG = 1,           /* null pointer / inconsistent sizes */
    GX_ERR_SCORES = 2,        /* precondition violated: need h <= 0, g < 0, h+g < 0 (SURVEY.md 3.3) */
    GX_ERR_RANGE = 3,         /* (m+n+2)*max|score| + |h| >= 2^29: int32 cell state would overflow */
    GX_ERR_OPS_CAP = 4,       /* ops buffer too small (need >= m+n+1) */
    GX_ERR_NO_DEVICE = 5,     /* no CUDA device of compute capability 10.x; there is no CPU path */
    GX_ERR_CUDA = 6,          /* CUDA runtime error, see gx_last_error() */
    GX_ERR_NOMEM = 7,         /* device or host allocation failed / traceback storage would not fit.  A traceback plan
                               * whose direction codes do not fit for every tile keeps them for the tiles of the code
                               * band only (DESIGN.md 2: global plans around the table's diagonal, local plans around
                               * the slope-1 line that ends at the start cell); it fails when even those do not fit,
                               * also after the band was moved to a new start cell or widened for a path that left it
                               * (gx_last_error names the pair -- "local pair" for a local plan --, the half-width and
                               * the bytes).  With GX_CODE_BAND=0 there is no band: codes must fit for every tile. */
    GX_ERR_NOT_INIT = 8,      /* gx_init() has not been called */
    GX_ERR_UNSUPPORTED = 9,   /* flag or mode not implemented */
    GX_ERR_INTERNAL = 10      /* impossible traceback state (the reference panics: algo.rs:407-408) */
};

/* ---- Scores: /root/reference/src/config.rs:6-13 (i64 there; int32 here, range-checked) */
typedef struct gx_scores {
    int32_t s_match;
    int32_t s_mismatch;
    int32_t g;   /* gap extension, per gap column (negative) */
    int32_t h;   /* gap opening (non-positive) */
} gx_scores;

/* ---- AlignmentChoice discriminants: algo.rs:124-133 (#[repr(u8)]) */
enum {
    GX_MATCH = 0, GX_MISMATCH = 1, GX_INSERT = 2, GX_DELETE = 3, GX_OPEN_INSERT = 4, GX_OPEN_DELETE = 5
};

/* ---- flags */
enum {
    GX_FLAG_TRACEBACK = 1,    /* fill direction codes and walk them (retrace, algo.rs:287-441) */
    GX_FLAG_LCS_AT_MAX = 2,   /* also return alignment_table's 2nd value (algo.rs:279-281): max_matches at the first max cell */
    GX_FLAG_START_CELL = 4    /* score-only local: also report the start cell (last argmax, algo.rs:311-322); read plans
                               * (>= 1024 pairs of <= 640 bp, s_mismatch < 0) compute it in the read kernels */
};

/* ---- AlignedSequences minus the sequence clones: algo.rs:135-146.
 * ops[k] is the AlignmentChoice discriminant of alignment[k] (walk order, start cell first,
 * algo.rs:357-396); the (i,j) of each entry follows by replaying the moves from (start_i,start_j)
 * with the checked_sub rules of algo.rs:412-417 (gx_replay_ops does it). */
typedef struct gx_result {
    int64_t score;            /* AlignedSequences.score, algo.rs:331 */
    uint64_t start_i, start_j;/* first walked cell: (m,n) global; last-argmax local (algo.rs:306-323) */
    uint64_t end_i, end_j;    /* last emitted cell */
    uint64_t n_ops;           /* alignment.len() */
    uint64_t matches, mismatches, gap_extensions, opening_gaps; /* algo.rs:141-145 */
    uint64_t lcs_at_first_max;/* GX_FLAG_LCS_AT_MAX only */
    double fill_ms, walk_ms;  /* device time of the fill / walk kernels of the call (shared by a batch) */
} gx_result;

/* ---- lifecycle.  One context per process, bound to one device (one process per GPU). */
int gx_init(int device);            /* device ordinal, or -1 for the current device */
void gx_shutdown(void);
int gx_device_count(void);          /* number of usable sm_100 devices, 0 if none / no driver */
const char *gx_strerror(int status);
const char *gx_last_error(void);    /* detail of the last GX_ERR_CUDA on this thread's context */
const char *gx_version(void);

/* GX_OK iff the reference's results can be reproduced in int32 for these lengths (SURVEY.md 3.3). */
int gx_check_scores(gx_scores sc, uint64_t m, uint64_t n);

/* ---- one pair, host buffers in, host buffers out.   replaces alignment_table + retrace.
 * s1 = sequences[0] (rows, i), s2 = sequences[1] (columns, j); any byte values.
 * ops may be NULL when GX_FLAG_TRACEBACK is not set; otherwise ops_cap >= m+n+1. */
int gx_align_pair(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n,
                  gx_scores sc, int is_local, int flags,
                  gx_result *out, uint8_t *ops, uint64_t ops_cap);

/* ---- many independent pairs in one call (pairs scattered over the SMs of this context's GPU).
 * Pair p is seq_blob[off1[p] .. off1[p]+len1[p]) vs seq_blob[off2[p] .. off2[p]+len2[p]).
 * With GX_FLAG_TRACEBACK pair p's ops go to ops_blob[ops_off[p] ..] and ops_off must have n_pairs+1
 * entries with ops_off[p+1]-ops_off[p] >= len1[p]+len2[p]+1.
 * The one-shot calls (gx_align_pair / gx_align_batch / gx_score_batch / gx_nw_score_banded) keep the plan of their
 * previous call and reuse it when the next call has the same lengths, scores, mode and flags (a stream of equally
 * shaped batches pays for plan creation once); another shape replaces it, gx_shutdown releases it. */
int gx_align_batch(const uint8_t *seq_blob, uint64_t blob_len,
                   const uint64_t *off1, const uint64_t *len1,
                   const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs,
                   gx_scores sc, int is_local, int flags,
                   gx_result *out, uint8_t *ops_blob, const uint64_t *ops_off);

/* ---- score-only batch (no traceback, no start cell): the form the short-read workload uses
 * (BASELINE config 4: 10M x 150 bp local).  Pairs of up to 640 bp run on the inter-task kernel. */
int gx_score_batch(const uint8_t *seq_blob, uint64_t blob_len,
                   const uint64_t *off1, const uint64_t *len1,
                   const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs,
                   gx_scores sc, int is_local, int64_t *scores);

/* gx_score_batch plus each pair's start cell: local = the last argmax (algo.rs:306-323), (m,n) when the maximum is 0;
 * global = (m,n).  Same inputs, routing, checks and status codes as gx_score_batch; start_i / start_j must not be NULL
 * when n_pairs > 0.  Read batches carry 8 bytes per pair back from the GPU (score and packed start cell). */
int gx_score_batch_cells(const uint8_t *seq_blob, uint64_t blob_len,
                         const uint64_t *off1, const uint64_t *len1,
                         const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs,
                         gx_scores sc, int is_local,
                         int64_t *scores, uint64_t *start_i, uint64_t *start_j);

/* ---- traceback for short-read sets (BASELINE config 4 with alignments): for every pair exactly the gx_result and op
 * bytes of gx_align_batch(..., GX_FLAG_TRACEBACK), computed by the inter-task read kernel (fill, direction codes in a
 * per-warp scratch slot, walk by the lane group that filled the pair) and streamed in chunks of 2^18 pairs like
 * gx_score_batch, for any n_pairs (0 included).  Device memory does not grow with n_pairs.  Arguments and the ops_off
 * contract are gx_align_batch's.  Differences: lcs_at_first_max is 0, fill_ms is the summed device time of the call's
 * read kernels, walk_ms is 0 (the walk runs inside them).  20 bytes per pair plus len1 + len2 + 1 op bytes come back.
 * Status: GX_ERR_UNSUPPORTED when a pair is longer than 640 bp, when the batch is local with s_mismatch >= 0, or when a
 * chunk's bytes are too scattered in seq_blob for one span copy (gx_align_batch handles those batches);
 * GX_ERR_OPS_CAP when ops_off[p+1] - ops_off[p] < len1[p] + len2[p] + 1; GX_ERR_ARG for null pointers or a sequence
 * outside seq_blob; GX_ERR_SCORES / GX_ERR_RANGE as gx_check_scores for 640 x 640 (local: also
 * 640 * max(s_match, 0) < 2^26).  After an error the contents of out and ops_blob are unspecified. */
int gx_align_reads(const uint8_t *seq_blob, uint64_t blob_len,
                   const uint64_t *off1, const uint64_t *len1,
                   const uint64_t *off2, const uint64_t *len2, uint64_t n_pairs,
                   gx_scores sc, int is_local,
                   gx_result *out, uint8_t *ops_blob, const uint64_t *ops_off);

/* ---- the same, split into phases so that callers can keep inputs resident in HBM, overlap
 * copies, and time the kernels alone.  gx_align_batch == create + upload + execute + fetch (+ destroy, deferred).
 * gx_plan_execute never returns a wrong result for speed's sake: a resident-strips fill that gives up waiting is
 * repeated in ticket mode, and a global traceback plan that writes direction codes only near the table's diagonal
 * (the "code band", DESIGN.md 2) is repeated if any path leaves the band: with codes everywhere, or -- when the plan
 * keeps codes for the band's tiles only (compact storage, stat 27 = 2) -- with the band of each pair whose path left
 * at least doubled and wide enough for where it left, until no path leaves.  The widths stay for the plan's life.
 * A local traceback plan with compact storage runs in two phases: a score-only pass finds every pair's start cell
 * (stat 29), each pair whose start cell moved gets a band of the default half-width around the slope-1 line that ends
 * there, then the traceback fill and walk run, repeated as above while a path leaves its band.  If the moved or
 * widened codes do not fit it returns GX_ERR_NOMEM, and so does every later execute of that plan. */
typedef struct gx_plan gx_plan;
int gx_plan_create(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs,
                   gx_scores sc, int is_local, int flags, gx_plan **plan);
int gx_plan_upload(gx_plan *plan, const uint8_t *seq_blob, uint64_t blob_len,
                   const uint64_t *off1, const uint64_t *off2);            /* host -> HBM */
int gx_plan_execute(gx_plan *plan);                                        /* kernels only, synchronous */
int gx_plan_fetch(gx_plan *plan, gx_result *out, uint8_t *ops_blob, const uint64_t *ops_off); /* HBM -> host */
int gx_plan_fetch_scores(gx_plan *plan, int64_t *scores);   /* scores only: 4 B per pair on the wire for read batches */
void gx_plan_destroy(gx_plan *plan);
/* introspection for benchmarks: what==0 fill ms, 1 walk ms, 2 kernels launched by the last execute,
 * 3 cells (sum (m+1)(n+1)), 4 bytes of the traceback codes buffer, 5 device bytes held by the plan,
 * 6 h2d bytes per upload, 7 d2h bytes per fetch, 8 tiles, 9 kernel family (0 wavefront, 1 read batch),
 * 15 K, 17 recurrence form (1 = CHAIN1), 18 ms of the GX_FLAG_LCS_AT_MAX passes, 20 ticket-mode retries,
 * 21 resident strips (1) or tickets (0), 22 steps per hand-off batch, 23 share of the cells in code-writing tiles,
 * 24 executes repeated because a path left the code band, 25 fill scores through the one-hot IDP.4A path (1; set at upload),
 * 26 read plans: lane width of the read kernel the last execute ran (16 = s16x2, 32; 0 before),
 * 27 code storage (0 codes in every tile or none, 1 dense with a code band, 2 compact: codes for the band's tiles only),
 * 28 widest code-band half-width in columns of the last execute (0 without a code band),
 * 29 ms of the start-cell pass of the last execute of a compact local plan (0 for other plans; included in stat 0).
 * Any other number returns -1. */
double gx_plan_stat(const gx_plan *plan, int what);

/* ---- one very long pair, global, score only, cut into column bands (BASELINE config 5; SURVEY.md 8e).
 * Replaces alignment_table (algo.rs:151-282) for tables whose 48-byte cells could never exist (1 Mbp x 1 Mbp).
 * The (m+1) x (n+1) table is cut into n_bands column bands (gx_band_range).  Band b hands the (E,I) of its last
 * column, 8 bytes per row, to band b+1 with the same flag-less 64-bit protocol the strips inside a band use.
 * A process owns the contiguous bands [first_band, last_band) on its GPU:
 *   all bands in one process      -> one kernel, nothing to connect (also the way to test N ranks on one GPU);
 *   one band (or range) per GPU   -> each process exports a 64-byte handle of its link block (CUDA IPC), the
 *                                    handles are exchanged by the caller (any transport; the Python host uses
 *                                    torch.distributed), and gx_band_connect maps the neighbours' blocks: the fill
 *                                    kernel of band b then stores its boundary rows straight into GPU b+1's HBM
 *                                    over NVLink and GPU b+1's kernel polls its own memory.  No host round trip,
 *                                    no collective call on the data path.
 * All processes must call gx_band_execute the same number of times; the score lives on the owner of the last band. */
#define GX_BAND_HANDLE_BYTES 64
typedef struct gx_band gx_band;
int gx_band_range(uint64_t n_total, int n_bands, int band, uint64_t *col0, uint64_t *width);   /* pure host arithmetic */
int gx_band_create(uint64_t m, uint64_t n_total, int n_bands, int first_band, int last_band, gx_scores sc, gx_band **band);
int gx_band_export(gx_band *band, void *handle, uint64_t handle_cap);     /* handle_cap >= GX_BAND_HANDLE_BYTES */
int gx_band_connect(gx_band *band, const void *left_handle, const void *right_handle);  /* NULL where there is no neighbour */
int gx_band_upload(gx_band *band, const uint8_t *s1, const uint8_t *s2);  /* full s1 (m bytes), full s2 (n_total bytes) */
int gx_band_execute(gx_band *band);                                       /* synchronous; device time in gx_band_stat(b,0) */
int gx_band_score(gx_band *band, int64_t *score, int *valid);             /* valid = 1 on the owner of the last band */
double gx_band_stat(const gx_band *band, int what);                       /* as gx_plan_stat; 16 = executes finished */
void gx_band_destroy(gx_band *band);
/* all bands on this process's GPU: create + upload + execute + score + destroy */
int gx_nw_score_banded(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n, gx_scores sc, int n_bands, int64_t *score);

/* ---- small-table visualiser support (display.rs:131-220, called at algo.rs:438): the insert / delete / sub score planes
 * of the table exactly as alignment_table stores them (algo.rs:195-248), row-major (m+1) x (n+1) int64 each, boundary
 * "minus infinity" = INT64_MIN + |g+h| (algo.rs:166).  Like the reference, only for m < 200 and n < 2000 (GX_ERR_RANGE). */
int gx_debug_planes(const uint8_t *s1, uint64_t m, const uint8_t *s2, uint64_t n, gx_scores sc, int is_local,
                    int64_t *insert_scores, int64_t *delete_scores, int64_t *sub_scores);

/* debug, pure host arithmetic (works without a GPU): the order in which the fill kernel hands out the tiles of these pairs
 * at register blocking K in {4,8,16} (bands != 0: the pairs are consecutive column bands of one table).  out receives
 * {pair, panel, strip} per tile (cap_tiles >= *n_tiles; out may be NULL to query the count).  Invariant (tested): the
 * tiles a tile depends on -- (panel, strip-1), (panel-1, strip), and for bands the last strip of the band to the left
 * -- always come earlier, which is what makes the persistent kernel deadlock-free. */
int gx_debug_tile_order(const uint64_t *len1, const uint64_t *len2, uint64_t n_pairs, int K, int bands, uint32_t *out,
                        uint64_t cap_tiles, uint64_t *n_tiles);

/* ---- replay helper: expands ops into (i,j) per entry exactly as algo.rs:412-417 would have pushed them. */
int gx_replay_ops(const uint8_t *ops, uint64_t n_ops, uint64_t start_i, uint64_t start_j,
                  uint32_t *ops_i, uint32_t *ops_j);

/* ---- INT32 / DPX issue-rate micro-benchmark (roofline denominator, SURVEY.md 8d "K0").
 * Fills out[0..n) with warp-instructions per clock per SM for:
 * 0 IADD3, 1 VIADDMNMX, 2 VIMNMX3, 3 ISETP+SEL, 4 IMAD, 5 the 7-op NW cell mix (cells/clk/SM),
 * 6 SM clock MHz observed, 7 SM count.  Returns the number of entries written or a negative status. */
int gx_k0_measure(double *out, int n);

#ifdef __cplusplus
}
#endif
#endif /* GXALIGN_H */
