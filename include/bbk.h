/* bbk.h - C ABI of libbbk.so, the B200 (sm_100a) kernels behind blueberry's Fit-Hi-C
 * significance pass.
 *
 * The reference (jmschrei/blueberry) has no FFI or plugin interface: its boundary is a set of
 * Python entry points in blueberry/fithic.py and blueberry/blueberry.pyx.  Each entry point below
 * names the reference code it replaces (paths relative to the reference root).  The Python host
 * in blueberry_b200/ keeps the reference's names and argument order and calls these functions
 * through ctypes; INTEGRATION.md shows the binding a maintainer would add to the reference.
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory owned by the caller; the library never allocates,
 *     frees or keeps caller buffers.  Scratch is caller-provided after a *_workspace_bytes query.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), returns 0 on
 *     success or a negative BBK_E_* code, and leaves a message for bbk_last_error().
 *   - no hidden global state: two calls never interact (the reference's module globals,
 *     fithic.py:25-42, accumulate across calls - a documented deviation).
 *   - results that later stages need (S, spline range, ...) stay on the device in BbkFitResult, so
 *     the whole pass can be enqueued without a host synchronisation.
 */
#ifndef BBK_H
#define BBK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BBK_VERSION 200 /* 0.2.0 */

/* error codes */
#define BBK_OK 0
#define BBK_E_INVALID (-1)      /* bad argument */
#define BBK_E_CUDA (-2)         /* a CUDA runtime call failed; see bbk_last_error */
#define BBK_E_WORKSPACE (-3)    /* workspace too small */
#define BBK_E_UNSUPPORTED (-4)
/* status codes the fit kernel leaves in BbkFitResult.status (see blueberry_b200/csrc/fit_stage.h) */
#define BBK_FIT_OK 0
#define BBK_FIT_ZERO_PAIRS_BIN (-11)   /* reference: ZeroDivisionError at fithic.py:216 */
#define BBK_FIT_TOO_FEW_BINS (-12)     /* scipy: "m > k must hold" */
#define BBK_FIT_TOO_MANY_BINS (-13)
#define BBK_FIT_S_ZERO (-14)           /* reference: ZeroDivisionError at fithic.py:216 */
#define BBK_FIT_X_NOT_INCREASING (-15)
#define BBK_FIT_EMPTY_GRID (-16)       /* no distance key inside [min(x), max(x)] */
#define BBK_FIT_BAD_PROBLEM (-17)      /* bbk_fit_batched: a problem's sizes, pointers or workspace do not allow the fit */
#define BBK_FIT_S_GIVEN 7777            /* INPUT value of BbkFitResult.status: use BbkFitResult.smoothing as s (see bbk_fit) */

int bbk_version(void);
/* copies the calling thread's last error message (NUL terminated) into buf; returns its length */
int bbk_last_error(char* buf, size_t buflen);
/* number of SMs of the current device (grid sizing is a multiple of it) */
int bbk_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  contact histogram by genomic distance            replaces read_interactions, fithic.py:229-270
 *
 * totals[8] (int64): 0 observedIntraInRangeSum (S)   1 observedIntraInRangeCount
 *                    2 observedIntraAllSum            3 observedIntraAllCount
 *                    4 observedInterAllSum            5 observedInterAllCount
 *                    6 minObservedGenomicDist         7 maxObservedGenomicDist
 * bbk_hist_init sets obs_sum to 0 and totals to the reference's initial values (fithic.py:25-41);
 * bbk_hist_pairs ACCUMULATES, so several shards (chromosomes, diagonal bands, ranks after an
 * allreduce) can feed one table.  d_chr1/d_chr2 may both be NULL: all records intra-chromosomal.
 * obs_sum[k] is mainDic[k*resolution][1]; nkeys = len(mainDic).
 * ------------------------------------------------------------------------------------------- */
int bbk_hist_init(int64_t* d_obs_sum, int32_t nkeys, int64_t* d_totals, void* stream);
int bbk_hist_pairs(const int32_t* d_chr1, const int32_t* d_chr2, const int32_t* d_mid1, const int32_t* d_mid2,
                   const int32_t* d_count, int64_t n_pairs, int64_t resolution, int64_t min_dist,
                   int64_t max_dist, int32_t nkeys, int64_t* d_obs_sum, int64_t* d_totals, void* stream);

/* Multi-GPU: one SUM all-reduce carries K1's whole output when the distance table, the totals and 2*world extra slots are
 * one contiguous int64 buffer [obs_sum (nkeys) | totals (8) | ext (2*world)]: bbk_stats_pack puts this rank's min / max
 * observed distance into its own slots of ext (zero elsewhere) before the all-reduce, bbk_stats_unpack folds the slots back
 * into totals[6] / totals[7] after it (fithic.py:258-259 over all ranks).  Integer sums: the result is independent of the
 * reduction order, so every rank holds bit-identical tables. */
int bbk_stats_pack(const int64_t* d_totals, int64_t* d_ext, int32_t world, int32_t rank, void* stream);
int bbk_stats_unpack(int64_t* d_totals, const int64_t* d_ext, int32_t world, void* stream);

/* Second pass (BASELINE config 4): the same histogram over the records that are NOT first-pass outliers,
 * i.e. skipping record i when d_p[i] <= p_outlier (NaN never compares true: unscored rows stay in).  The
 * reference has no second pass (n_passes is ignored, fithic.py:121-133); the definition follows SURVEY.md
 * section 8c: outliers are rows with p <= 1 / possibleIntraInRangeCount, the refit uses the reference's own
 * read_interactions / calculate_probabilities / fit_spline on the filtered records and scores ALL records. */
int bbk_hist_pairs_excluding(const int32_t* d_chr1, const int32_t* d_chr2, const int32_t* d_mid1, const int32_t* d_mid2,
                             const int32_t* d_count, const double* d_p, double p_outlier, int64_t n_pairs,
                             int64_t resolution, int64_t min_dist, int64_t max_dist, int32_t nkeys,
                             int64_t* d_obs_sum, int64_t* d_totals, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2a possible pairs per distance                      replaces generate_FragPairs, fithic.py:302-311
 * d_n_frags[c] = number of distinct fragment mids of chromosome c, d_max_frag[c] = max(mid) - R/2.
 * possible[k] = sum_c (k*R <= max_frag[c] ? n_frags[c] - k : 0)        (goes negative like the
 * reference when the fragment list is sparse).
 * ------------------------------------------------------------------------------------------- */
int bbk_possible_pairs(const int64_t* d_n_frags, const int64_t* d_max_frag, int32_t n_chrom, int64_t resolution,
                       int32_t nkeys, int64_t* d_possible, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2b+K3  equal-occupancy binning, smoothing spline, antitonic regression
 *         replaces calculate_probabilities (fithic.py:160-227) and the fit part of fit_spline
 *         (fithic.py:340-374: UnivariateSpline(x, y, s=min(y)**2), ius(splineX),
 *         IsotonicRegression(increasing=False)).
 * ------------------------------------------------------------------------------------------- */
typedef struct BbkFitResult {
    int32_t status;      /* BBK_FIT_* */
    int32_t n_out;       /* number of bins emitted (len(x)) */
    int32_t k0;          /* splineX[0] / resolution */
    int32_t L;           /* len(splineX) */
    int32_t n_knots;     /* knots of the spline (incl. the 2*4 boundary knots) */
    int32_t ier;         /* FITPACK-style status of the spline search */
    int64_t S;           /* observedIntraInRangeSum used */
    double min_x, max_x; /* min(x), max(x) */
    double residual;     /* sum((y - ius(x))**2), fithic.py:374 */
    double fp;           /* weighted sum of squared residuals of the smoothing spline */
    double smoothing;    /* s.  The reference passes s = min(y)**2 on Python floats, i.e. libm's pow(ymin, 2.0), which is NOT always
                            the correctly rounded ymin*ymin (glibc 2.39: one ulp off for ~0.09 % of inputs); the kernel computes
                            ymin*ymin.  A host that wants the reference's bits checks this field against its own min(y)**2 and, when
                            they differ, calls bbk_fit again with status = BBK_FIT_S_GIVEN and smoothing = its value on input. */
    int64_t phase_cycles[6]; /* SM clock cycles: staging+binning, bin stats, spline search, grid evaluation,
                                antitonic regression + residual, total */
    int64_t spline_diag[8];  /* LSQ fits, smoothing iterations, then SM cycles: B-spline rows, row QR + back
                                substitution, residuals + knot insertion, Givens sweep, f(p) evaluation */
    double y_min;            /* min(y): what the host needs to form the reference's own s = min(y)**2 for the check above */
} BbkFitResult;

/* bytes of scratch bbk_fit needs for up to max_bins bins and nkeys distances */
size_t bbk_fit_workspace_bytes(int32_t max_bins, int32_t nkeys);
/* d_totals: the table K1 filled (S is read from d_totals[0] on the device).
 * outputs: d_result (1 struct), d_x/d_y [max_bins], d_bin_of_key [nkeys] (-1 = none),
 *          d_spline_y [nkeys] (entries 0..L-1 = newSplineY), d_spline_raw [nkeys] (ius(splineX)),
 *          d_knots/d_coefs [max_bins+4]. */
int bbk_fit(const int64_t* d_possible, const int64_t* d_obs_sum, int32_t nkeys, const int64_t* d_totals,
            int32_t n_bins, int64_t resolution, int64_t min_dist, int64_t max_dist, int32_t max_bins,
            BbkFitResult* d_result, double* d_x, double* d_y, int32_t* d_bin_of_key, double* d_spline_y,
            double* d_spline_raw, double* d_knots, double* d_coefs, void* d_workspace, size_t workspace_bytes,
            void* stream);
/* Many independent fits in ONE launch (one CTA each, grid = n_problems), e.g. one per chromosome: the authors ran Fit-Hi-C
 * once per chromosome (datatypes.pyx:26), each run with its own calculate_probabilities (fithic.py:160-227) and fit_spline
 * (fithic.py:340-374).  Problem i is exactly bbk_fit with the tables and outputs of d_problems[i] and the shared n_bins,
 * resolution, min_dist and max_dist; each result struct carries its own BBK_FIT_S_GIVEN input.  d_problems: a DEVICE array
 * of n_problems descriptors owned by the caller.  A problem whose sizes, pointers or workspace (below
 * bbk_fit_workspace_bytes(max_bins, nkeys)) do not allow the fit gets status BBK_FIT_BAD_PROBLEM and writes nothing else;
 * the other problems are not affected. */
typedef struct BbkFitProblem {
    const int64_t* d_possible;
    const int64_t* d_obs_sum;
    const int64_t* d_totals;
    BbkFitResult* d_result;
    double* d_x;
    double* d_y;
    int32_t* d_bin_of_key;
    double* d_spline_y;
    double* d_spline_raw;
    double* d_knots;
    double* d_coefs;
    void* d_workspace;
    uint64_t workspace_bytes;
    int32_t nkeys;
    int32_t max_bins;
} BbkFitProblem;
int bbk_fit_batched(const BbkFitProblem* d_problems, int32_t n_problems, int32_t n_bins, int64_t resolution, int64_t min_dist,
                    int64_t max_dist, void* stream);
/* stage-injection entry for tests: the spline + antitonic part alone on given bin means x, y */
int bbk_fit_from_bins(const double* d_x_in, const double* d_y_in, int32_t m, int32_t nkeys, int64_t resolution,
                      BbkFitResult* d_result, double* d_spline_y, double* d_spline_raw, double* d_knots,
                      double* d_coefs, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4  per-pair binomial survival p-values              replaces the scoring loop, fithic.py:413-435
 *     p = bdtrc(count-1, S, newSplineY[i] * (bias1*bias2)),  i = min(bisect_left(splineX, clamp(d)), L-1)
 * Rows the reference does not score (d outside [min_dist, max_dist], :427) or drops (p_val <= 1
 * false, :434: negative prior from a -1 bias, prior > 1) get p = NaN.
 * Bias lookup (biasDic[chr][mid], default 1.0, :418-425) is a dense per-chromosome table:
 *   bias = d_bias[chrom_base[c] + (mid - mid0[c]) / resolution]  when (mid - mid0[c]) is a
 *   non-negative multiple of resolution below the table end and the entry is not NaN; else 1.0.
 * d_chr1/d_chr2 NULL: every record is on chromosome `shard_chrom`.
 * d_p_hist (nullable, int64[BBK_PHIST_LEN]): K4 adds the coarse p-value histogram the BH step uses
 * for pruning, saving BH one pass over p.  Bucket of a p in [0, 1) = (IEEE bits >> 51) & 4095
 * (exponent + top mantissa bit); entry [4096] counts p == 1.0 exactly, entry [4097] counts NaN.
 * ------------------------------------------------------------------------------------------- */
#define BBK_PHIST_BINS 4096
#define BBK_PHIST_LEN (BBK_PHIST_BINS + 2)
typedef struct BbkBiasTable {
    const double* d_bias;        /* concatenated per-chromosome tables (NaN = locus absent), NULL = no biases */
    const int64_t* d_chrom_base; /* [n_chrom + 1] offsets into d_bias */
    const int64_t* d_mid0;       /* [n_chrom] mid of entry 0 of each chromosome */
    int32_t n_chrom;
    int64_t step;                /* distance between neighbouring entries; 0 = the resolution of the pass (bias loci on the fragment grid) */
} BbkBiasTable;

int bbk_pvalues(const int32_t* d_chr1, const int32_t* d_chr2, const int32_t* d_mid1, const int32_t* d_mid2,
                const int32_t* d_count, int64_t n_pairs, int32_t shard_chrom, int64_t resolution, int64_t min_dist,
                int64_t max_dist, const BbkFitResult* d_fit, const double* d_spline_y, const BbkBiasTable* bias,
                double* d_p, int64_t* d_p_hist, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4 as one streaming pass + a patch pass       replaces the scoring loop of fit_spline, fithic.py:413-435
 *
 * Most records need no arithmetic (count <= 0: p = 1.0, or NaN when bdtrc rejects the prior), most of the rest have a count
 * of 1..8 (a handful of FP64 operations in the lower-tail form), a few per cent need a long tail sum.  bbk_score_pairs
 * streams the records of one shard once - tiles of BBK_TILE_ROWS rows staged in shared memory by bulk asynchronous copies -
 * finishes everything but that last kind and writes EVERY row's p (and q = 1.0 / NaN, the value of a row that is not a
 * q-value candidate) with full coalesced stores; the rows it cannot finish (count > 8, prior outside (0, 2^-10), a
 * lower-tail result below 1e-4, S < 64) are appended as (row, count, prior) to `deferred` and get a placeholder.
 * bbk_score_deferred then scores that list with the arithmetic and edge semantics of bbk_pvalues and patches p in place.
 * Both fill d_p_hist and append (key, row) of every p < 2^-5 to `cands` for bbk_bh_qvalues_listed.
 * count <= 0 rows are taken as p = 1.0 without looking at their prior when neither locus carries a flag bit
 * (bbk_bias_flags: bias < 0 or > 4) - which is right iff 0 <= splineY and 16 max(splineY) <= 1; bbk_score_guard (after the
 * fit) checks that and raises BbkScoreState.exact otherwise: every in-range row then goes through its prior.
 * Rows are positions in the rank-local p / q buffers: record i of a call is row out_base + i (out_base a multiple of 4,
 * rows < 2^32), so several shards share one pair of buffers, one deferred list, one candidate list and one q-value step.
 * p / q need (n_pairs + 3) & ~3 rows per shard.  No chromosome columns: a shard is one chromosome (shard_chrom).
 * Needs 0 <= min_dist <= max_dist and max_dist + resolution < 2^31; otherwise use bbk_pvalues.
 * A deferred list with capacity >= the number of records cannot overflow; a smaller one sets BbkScoreState.overflow when
 * it does (bbk_score_deferred then does nothing; the caller repeats the pass with a larger list).
 * Sequence:  bbk_score_begin -> K1, bbk_fit -> bbk_score_guard -> bbk_score_pairs per shard -> bbk_score_deferred
 *            -> [bbk_bh_qvalues_listed]
 * ------------------------------------------------------------------------------------------- */
#define BBK_TILE_ROWS 2048
typedef struct BbkScoreState {
    uint64_t n_list;         /* deferred rows appended so far */
    uint64_t n_cand;         /* candidates appended so far */
    int32_t overflow;        /* the deferred list was too small */
    int32_t cand_overflow;   /* the candidate list was too small (the q-value step then takes its full pass: still exact) */
    int32_t exact;           /* the guard failed: no count <= 0 shortcut in this pass */
    int32_t reserved;
} BbkScoreState;
typedef struct BbkDeferredList {
    uint32_t* d_row;         /* rank-local row */
    int32_t* d_count;
    double* d_prior;         /* newSplineY[i] * (bias1 * bias2), fithic.py:431 */
    int64_t capacity;        /* entries */
} BbkDeferredList;
typedef struct BbkCandidates {
    uint64_t* d_keys;        /* order-preserving key of p */
    uint32_t* d_rows;        /* rank-local row */
    int64_t capacity;
} BbkCandidates;

int bbk_score_begin(BbkScoreState* d_state, int64_t* d_p_hist, void* stream);     /* zeroes the state and the histogram */
/* one flag bit per entry of the concatenated bias table (bit j of word j / 32): value < 0 or > 4.  d_flags holds
 * bbk_bias_flags_bytes(n_entries) bytes, ZEROED by the caller before bbk_bias_flags (the size includes a spare word). */
size_t bbk_bias_flags_bytes(int64_t n_entries);
int bbk_bias_flags(const double* d_bias, int64_t n_entries, uint32_t* d_flags, void* stream);
int bbk_score_guard(const BbkFitResult* d_fit, const double* d_spline_y, BbkScoreState* d_state, void* stream);
int bbk_score_pairs(const int32_t* d_mid1, const int32_t* d_mid2, const int32_t* d_count, int64_t n_pairs,
                    int32_t shard_chrom, int64_t resolution, int64_t min_dist, int64_t max_dist,
                    const BbkFitResult* d_fit, const double* d_spline_y, const BbkBiasTable* bias,
                    const uint32_t* d_bias_flags, int64_t out_base, double* d_p, double* d_q, int64_t* d_p_hist,
                    const BbkCandidates* cands, const BbkDeferredList* deferred, BbkScoreState* d_state, void* stream);
int bbk_score_deferred(const BbkDeferredList* deferred, const BbkFitResult* d_fit, double* d_p, double* d_q,
                       int64_t* d_p_hist, const BbkCandidates* cands, BbkScoreState* d_state, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gather for the genome-wide q-value step               replaces utils.extract_contacts, utils.py:31-90
 *
 * d_map: a Fit-Hi-C result table, (n, 5) float64 rows (mid1, mid2, contactCount, p, q) = FithicContactMap.map
 * (datatypes.pyx:314).  Keeps, in order, the rows with p <= alpha (use_alpha != 0; utils.py:72-73) and
 * low <= mid2 - mid1 <= high (:80-83; the reference's LOW_/HIGH_FITHIC_CUTOFF), written as
 * (chromosome, mid1, mid2, contactCount, p) (:76-77) to d_out (capacity rows; rows beyond it are counted, not written).
 * d_n_out receives the number of rows kept.  Workspace: bbk_extract_workspace_bytes(n).
 * ------------------------------------------------------------------------------------------- */
size_t bbk_extract_workspace_bytes(int64_t n);
int bbk_extract_contacts(const double* d_map, int64_t n, double chromosome, double alpha, int32_t use_alpha, double low,
                         double high, double* d_out, int64_t capacity, int64_t* d_n_out, void* d_workspace,
                         size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Output packing                                         the output side of fithic.py:410-435, for the host link
 *
 * Most rows carry no information in their numbers (zero-count pairs: p = 1.0, q = 1.0; rows the reference does not emit:
 * NaN; q = 1.0 for all but the significant rows), and the end-to-end call is bound by the host link.  bbk_pack_scores turns
 * the dense p / q columns into two bits per row + the values that are not implied:
 *     code 0  p = 1.0, q = 1.0     code 1  p = NaN, q = NaN     code 2  p in d_values_p, q = 1.0     code 3  p and q in the lists
 * d_codes: one uint32 per 16 rows (row r: bits 2 (r % 16) of word r / 16), bbk_pack_code_words(m) words.
 * d_chunks: one record per BBK_PACK_CHUNK rows, bbk_pack_chunks(m) records: where the chunk's packed values start in
 * each list and how many there are (chunks land in the lists in no particular order; rows inside a chunk keep theirs).
 * d_q may be NULL (no q-values: codes 0..2).  A list that is too small sets BbkPackState.overflow (values beyond the
 * capacity are dropped; the caller falls back to the dense columns).  Lossless: bbkio_unpack_scores (bbk_io.h) rebuilds
 * the dense columns bit for bit.
 * ------------------------------------------------------------------------------------------- */
#define BBK_PACK_CHUNK 4096
typedef struct BbkPackChunk {
    uint64_t base_p;         /* first packed p of the chunk in d_values_p */
    uint64_t base_q;         /* first packed q of the chunk in d_values_q */
    uint32_t n_p;            /* rows of the chunk with code >= 2 */
    uint32_t n_q;            /* rows of the chunk with code 3 */
} BbkPackChunk;
typedef struct BbkPackState {
    uint64_t n_p;            /* values in d_values_p */
    uint64_t n_q;            /* values in d_values_q */
    int32_t overflow;
    int32_t reserved;
} BbkPackState;
int64_t bbk_pack_chunks(int64_t m);
int64_t bbk_pack_code_words(int64_t m);
int bbk_pack_scores(const double* d_p, const double* d_q, int64_t m, uint32_t* d_codes, BbkPackChunk* d_chunks,
                    double* d_values_p, int64_t capacity_p, double* d_values_q, int64_t capacity_q,
                    BbkPackState* d_state, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Packed contact records                                 the input side of the host link
 *
 * The int32 record columns (mid1, mid2, count) of a pass cost 12 B/row to move in, but carry far fewer bits: mid1 is nearly
 * constant over a block of rows, mid2 - mid1 is a multiple of the resolution, counts are small.  The packed form is a
 * frame-of-reference code per BBK_REC_CHUNK rows of the pass layout (layout_rows: shard i at starts[i], the padding rows
 * between shards encoded as zeros).  Buffer:
 *     BbkRecHeader | BbkRecChunk[ceil(rows / BBK_REC_CHUNK)] | chunk payloads
 * Chunk c holds rows [c * BBK_REC_CHUNK, min(rows, (c + 1) * BBK_REC_CHUNK)).  Its three columns j are
 *     j = 0: mid1    j = 1: e = mid2 - mid1 (in 64 bits)    j = 2: count
 * each stored as v = base[j] + step[j] * u, base = the chunk minimum, step = gcd(v - base) (1 when all values are equal),
 * u in bits[j] bits (0..32; 0..33 for e), packed little-endian into 64-bit words: row i of the chunk is bits
 * [i * bits, (i + 1) * bits) of the column's words.  Column j's block is BBK_REC_COL_BYTES(n, bits[j]) bytes (a multiple of
 * 16); the three blocks follow each other from `offset` (bytes from the buffer start, a multiple of 16).  Chunks are laid
 * out in order.  Lossless for every int32 input; the bytes depend on the records only (bbkio_pack_records in bbk_io.h
 * writes them on the host, bbkio_check_records validates them).
 * bbk_unpack_records decodes rows [0, rows) into three int32 device columns (16-byte aligned).  It trusts its buffer: the
 * caller passes only buffers that bbkio_check_records accepted for the same `rows` and `bytes`.
 * ------------------------------------------------------------------------------------------- */
#define BBK_REC_MAGIC 0x31434552u       /* "REC1" */
#define BBK_REC_VERSION 1
#define BBK_REC_CHUNK 4096
#define BBK_REC_COL_BYTES(n, bits) ((((uint64_t)(n) * (uint64_t)(bits) + 127u) / 128u) * 16u)
typedef struct BbkRecHeader {
    uint32_t magic;          /* BBK_REC_MAGIC */
    uint32_t version;        /* BBK_REC_VERSION */
    int64_t rows;            /* rows of the pass layout */
    uint64_t bytes;          /* bytes of the whole buffer */
    uint64_t reserved;
} BbkRecHeader;
typedef struct BbkRecChunk {
    int64_t base[3];
    uint64_t step[3];
    uint64_t offset;         /* first byte of column 0's block */
    uint8_t bits[3];
    uint8_t reserved[5];
} BbkRecChunk;
int bbk_unpack_records(const void* d_buf, int64_t bytes, int64_t rows, int32_t* d_mid1, int32_t* d_mid2, int32_t* d_count,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5  Benjamini-Hochberg q-values as the reference computes them: a FORWARD running max of
 *     min(p * N / rank, 1)   (fithic.py:466-487, blueberry.pyx:40-75) - not the textbook reverse
 *     cumulative minimum.  q comes back in input order; NaN p (dropped rows) -> NaN q, not ranked.
 * mode BBK_BH_UNSORTED   : benjamini_hochberg_correction(p_values, N)   (fithic.py:466)
 * mode BBK_BH_POSITIONAL : benjamini_hochberg(p_values, n) of blueberry.pyx:40 - the input is taken
 *                          as already sorted, rank = position + 1, no tie handling.
 * d_p_hist: optional coarse histogram from bbk_pvalues (NULL: computed here).
 * d_rank (nullable, int64[m]): 1 + number of strictly smaller p among the ranked rows.
 * ------------------------------------------------------------------------------------------- */
#define BBK_BH_UNSORTED 0
#define BBK_BH_POSITIONAL 1
size_t bbk_bh_workspace_bytes(int64_t m);
int bbk_bh_qvalues(const double* d_p, int64_t m, int64_t n_tests, int32_t mode, const int64_t* d_p_hist,
                   double* d_q, int64_t* d_rank, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5, genome-wide across ranks: the reference's q-value step ranks the p-values of ALL chromosomes
 * together (utils.py:31-90 gathers them per chromosome for blueberry.pyx:40).  Shards live on different
 * GPUs, so the ranking is split around two host-side collectives (NCCL through torch.distributed), with no
 * candidate count ever reaching the host:
 *   K4's d_p_hist        ->  all-reduce(sum) of the histogram
 *   bbk_bh_select[_listed] : common saturation bucket from the GLOBAL histogram; writes q = 1.0 / NaN for
 *                          everything that is not a candidate, candidates' keys / row indices to d_keys /
 *                          d_idx, d_state[4] = {n_candidates, tau_key, N, n_ones}
 *   bbk_bh_pack_count    : puts n_candidates in front of the keys (d_keys = d_send + 1)
 *   all-gather of the fixed-capacity blocks (order: rank 0's, rank 1's, ...)
 *   bbk_bh_rank_gathered_padded : ranks all gathered keys, scatters this rank's q-values back
 *   bbk_bh_fix_ones_dev  : only when q of the p == 1.0 group is below 1: q = q_ones wherever p == 1.0
 * Workspace of select: bbk_bh_workspace_bytes(0).  With one rank this reproduces bbk_bh_qvalues bit for bit.
 * d_keys / d_idx hold keys_capacity entries (a fixed-capacity send block); candidates beyond it are counted in
 * d_state[0] but not stored - bbk_bh_rank_gathered_padded then reports the overflow.
 * ------------------------------------------------------------------------------------------- */
int bbk_bh_select(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist_global, double* d_q,
                  uint64_t* d_keys, uint32_t* d_idx, int64_t keys_capacity, uint64_t* d_state, void* d_workspace,
                  size_t workspace_bytes, void* stream);
/* q = d_q_ones[0] wherever p == 1.0, decided on the device from d_q_ones[2] of bbk_bh_rank_gathered_padded (nothing to do
 * when d_q_ones[1] == 0) */
int bbk_bh_fix_ones_dev(const double* d_p, int64_t m, const double* d_q_ones, double* d_q, void* stream);

/* listed mode: after bbk_score_pairs / bbk_score_deferred on the same d_p / d_p_hist / d_q, ranking from their candidate list */
int bbk_bh_qvalues_listed(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist, double* d_q,
                          const BbkCandidates* cands, const BbkScoreState* d_state, void* d_workspace, size_t workspace_bytes,
                          void* stream);
/* Per-chromosome q-values in one step: the authors ran Fit-Hi-C once per chromosome, so each chromosome's q-values come from its
 * own benjamini_hochberg_correction (fithic.py:466-487) over its own p-values.  Segment s is rows [d_offsets[s], d_offsets[s+1])
 * of d_p / d_q (d_offsets: DEVICE int64[n_segments + 1], non-decreasing, every start a multiple of 4 as layout_rows gives, the
 * last <= m) scored by bbk_score_pairs / bbk_score_deferred with the segment's own histogram, candidate list and score state,
 * given in d_segments (a DEVICE array of complete descriptors; candidate rows are rows of d_p).  q of every segment equals
 * bbk_bh_qvalues_listed run on that segment alone, bit for bit, including segments that need the pass over p (saturation at or
 * above 2^-5, or an overflowed candidate list: decided on the device, and only those segments' rows are read).  The number of
 * launches does not depend on n_segments (<= 65536).  Workspace: bbk_bh_segmented_workspace_bytes(m, n_segments). */
typedef struct BbkBhSegment {
    const int64_t* d_p_hist;         /* BBK_PHIST_LEN: the segment's K4 histogram */
    const BbkScoreState* d_state;    /* the segment's score state */
    BbkCandidates cands;             /* the segment's candidate list */
    int64_t n_tests;                 /* N of the segment; -1 = its number of non-NaN p */
} BbkBhSegment;
size_t bbk_bh_segmented_workspace_bytes(int64_t m, int32_t n_segments);
int bbk_bh_qvalues_segmented(const double* d_p, int64_t m, const int64_t* d_offsets, const BbkBhSegment* d_segments,
                             int32_t n_segments, double* d_q, void* d_workspace, size_t workspace_bytes, void* stream);
/* bbk_bh_select from that candidate list */
int bbk_bh_select_listed(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist_global, double* d_q,
                         const BbkCandidates* cands, const BbkScoreState* d_score, uint64_t* d_keys, uint32_t* d_idx,
                         int64_t keys_capacity, uint64_t* d_state, void* d_workspace, size_t workspace_bytes, void* stream);

/* Genome-wide ranking with the gather left on the device (no candidate count ever reaches the host): every rank sends a
 * fixed-capacity block [count | keys[0 .. cap)] - d_keys of bbk_bh_select* written at send + 1, the count put in front by
 * bbk_bh_pack_count - and one all-gather delivers `world` such blocks (d_recv: world * (cap + 1) u64).
 * bbk_bh_rank_gathered_padded prefixes the counts, compacts the blocks, ranks them (forward running max) and scatters
 * THIS rank's slice back: d_q_dst[d_idx_local[i]] = q of this rank's candidate i.
 * A count above cap puts the largest count of any rank into *d_overflow (int32, never cleared here); the host checks it when it reads the results and repeats
 * the q-value step with a larger capacity.  d_q_ones[2] = {q of the p == 1.0 group, 1.0 if it is below 1}.  Workspace:
 * bbk_bh_gathered_workspace_bytes(world, cap). */
size_t bbk_bh_gathered_workspace_bytes(int32_t world, int64_t cap);
int bbk_bh_pack_count(const uint64_t* d_state, uint64_t* d_send, void* stream);
int bbk_bh_rank_gathered_padded(const uint64_t* d_recv, int32_t world, int64_t cap, int32_t rank, const uint64_t* d_state,
                                const uint32_t* d_idx_local, double* d_q_dst, double* d_q_ones, int32_t* d_overflow,
                                void* d_workspace, size_t workspace_bytes, void* stream);
/* The same ranking without the per-rank scatter, for one GPU that plays every rank itself (row blocks of a pass larger than
 * the device, distributed.BlockedPass): all gathered keys are sorted once and d_q_all[r * cap + i] receives the q of block
 * r's candidate i, for i below that block's count (the other places are left as they are).  d_q_all: world * cap doubles;
 * d_q_ones and d_overflow as above; world * cap < 2^32.  Workspace: bbk_bh_gathered_workspace_bytes(world, cap). */
int bbk_bh_rank_gathered_all(const uint64_t* d_recv, int32_t world, int64_t cap, const uint64_t* d_state, double* d_q_all,
                             double* d_q_ones, int32_t* d_overflow, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6  count_band_regions                               replaces blueberry.pyx:77-91
 *     t = #{(i, j) : j < i, low <= regions[i] - regions[j] <= high}
 * d_result: TWO int64 (device): [0] the count, [1] scratch.  Exact for sorted and unsorted input.
 * ------------------------------------------------------------------------------------------- */
int bbk_count_band(const double* d_regions, int64_t n, double low, double high, int64_t* d_result, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K7  FithicContactMap.decimate                        replaces datatypes.pyx:317-339  (SURVEY.md 8f, row 1)
 *     mid' = (int(mid) + r) / r * r - r/2 (Python-2 integer division) for both midpoints of every row, then rows with
 *     equal (mid1', mid2') are folded in file order: count = count_i + count, p = p_i * p, q = min(q_i, q) from (0, 1, 1).
 * d_map: the reference's own layout, (n, 5) float64 row-major rows (mid1, mid2, contactCount, p, q); d_out_map: the
 * decimated map in the same layout (capacity n rows), groups in the order of their first row in the file.
 * *d_n_out: number of groups, or -1 when a coordinate is outside [0, 2^31).
 * The sum and the product are folded by one thread per group, member by member, so they round like the reference's loop.
 * ------------------------------------------------------------------------------------------- */
size_t bbk_decimate_workspace_bytes(int64_t n);
int bbk_decimate(const double* d_map, int64_t n, int64_t resolution, double* d_out_map, int64_t* d_n_out, void* d_workspace,
                 size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K8  ContactMap ingest + normalize on band records    replaces datatypes.pyx:99-120 and :143-171  (SURVEY.md 8f, row 3)
 * The reference holds the map as a dense (n_bins+1)^2 float64 matrix; here the RAWobserved rows stay records.
 * ingest:    bin = int(nan_to_num(pos) / resolution) for both positions (:104, :111-112), stored as bin1 <= bin2 (the
 *            reference writes both triangles, :115-116); value = nan_to_num(count).  *d_bad != 0 afterwards when a
 *            bin is negative or > n_bins (outside the reference's matrix).
 * normalize: value / (KRnorm[bin1] * KRnorm[bin2] * KRexpected[bin2 - bin1]) for bin2 < n_bins (:166-168; the loop
 *            never reaches row / column n_bins), then nan_to_num (:171).  d_out may alias d_value.  *d_bad != 0 when a
 *            divisor is exactly 0.0: the reference's (Cython, checked) division raises ZeroDivisionError there.
 * Scattering the records into a zero matrix gives the reference's matrix when no (bin1, bin2) repeats (for repeats
 * the reference keeps the last row of the file; records keep them all).
 * ------------------------------------------------------------------------------------------- */
int bbk_contact_band_ingest(const double* d_pos1, const double* d_pos2, const double* d_count, int64_t n, int64_t resolution,
                            int32_t n_bins, int32_t* d_bin1, int32_t* d_bin2, double* d_value, int32_t* d_bad, void* stream);
int bbk_contact_band_normalize(const int32_t* d_bin1, const int32_t* d_bin2, const double* d_value, int64_t n,
                               const double* d_kr_norm, const double* d_kr_expected, int32_t n_bins, double* d_out,
                               int32_t* d_bad, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Synthetic contact records of the BASELINE shapes, generated on the device (bench only).
 * Fills mid1/mid2/count for one chromosome of n_bins bins: all (i, i+d), 0 <= d <= K, row-major.
 * d_bias (nullable): per-bin visibility multiplying the Poisson mean.  Returns records written
 * through *n_written (host).
 * ------------------------------------------------------------------------------------------- */
int64_t bbk_synth_n_pairs(int64_t n_bins, int64_t K);
int bbk_synth_contacts(int64_t n_bins, int64_t K, int64_t resolution, double depth, double decay, uint64_t seed,
                       const double* d_bias, int32_t* d_mid1, int32_t* d_mid2, int32_t* d_count, void* stream);
/* records first_record .. first_record + n_records - 1 of the same chromosome (a row block for one rank) */
int bbk_synth_contacts_range(int64_t n_bins, int64_t K, int64_t resolution, double depth, double decay, uint64_t seed,
                             const double* d_bias, int64_t first_record, int64_t n_records, int32_t* d_mid1, int32_t* d_mid2,
                             int32_t* d_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BBK_H */
