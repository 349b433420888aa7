/* bbk_io.h - host-side file formats either side of the Fit-Hi-C pass (SURVEY.md section 8f, row 1).
 *
 * Plain C ABI of libbbkio.so (host code only: g++, zlib, pthreads; no CUDA).  The reference writes its result as
 * gzip text one Python `write` per row (fithic.py:410-435, ~14 us/row of format + zlib); this is the same file -
 * same header, same rows, same number formatting - produced by all host cores as independent gzip members
 * (a concatenation of gzip members is a valid gzip file: gzip.open / zcat / pandas read it as one stream).
 */
#ifndef BBK_IO_H
#define BBK_IO_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define BBKIO_OK 0
#define BBKIO_E_INVALID (-1)
#define BBKIO_E_IO (-2)
#define BBKIO_E_ZLIB (-3)

/* message of the last failing call on this thread */
void bbkio_last_error(char* buf, size_t len);

/* replaces fithic.py:410-435.
 * Line 1: "chr1\tfragmentMid1\tchr2\tfragmentMid2\tcontactCount\tp-value\tq-value" (fithic.py:411).
 * Then, for every record i with p[i] <= 1 (fithic.py:434; NaN rows are the ones the reference never emits), in input order:
 *   chrom_names[chr1[i]] \t mid1[i] \t chrom_names[chr2[i]] \t mid2[i] \t count[i] \t p[i] \t q[i]   (fithic.py:435)
 * with the doubles formatted as Python's "{}".format(float64): shortest digits that round-trip, positional for
 * 1e-4 <= |x| < 1e16, otherwise d.ddde-XX with at least two exponent digits.  q == NULL writes the literal -1 the
 * reference writes (it never computes q).  chr1/chr2 == NULL: every record is on chrom_names[0].
 * threads <= 0: all online cores.  level: zlib level 1..9 (the reference's gzip.open default is 9; 1 is ~4x faster).
 * rows_written (nullable) receives the number of data rows. */
int bbkio_write_significances(const char* path, const char* const* chrom_names, int32_t n_chrom, const int32_t* chr1,
                              const int64_t* mid1, const int32_t* chr2, const int64_t* mid2, const int64_t* count,
                              const double* p, const double* q, int64_t n, int32_t threads, int32_t level,
                              int64_t* rows_written);

/* replaces the read loop of fithic.py:243-247 (`chr1, mid1, chr2, mid2, contactCount = line.rstrip().split()`).
 * Reads a gzip (or plain) text file of whitespace-separated rows into columns: one thread inflates, `threads` parse.
 * Chromosome names become small ids in order of first appearance (bbkio_table_chrom_name gives them back).
 * Errors like the reference's unpack / int(): a row with fewer or more than 5 fields, or a non-integer mid / count,
 * fails the call (BBKIO_E_PARSE; bbkio_last_error names the line).  Blank lines fail too (zero fields), as in the reference.
 * The table is owned by the library until bbkio_table_free. */
#define BBKIO_E_PARSE (-4)
typedef struct BbkioTable BbkioTable;
int bbkio_read_interactions(const char* path, int32_t threads, BbkioTable** out);
int64_t bbkio_table_rows(const BbkioTable* t);
int32_t bbkio_table_n_chrom(const BbkioTable* t);
const char* bbkio_table_chrom_name(const BbkioTable* t, int32_t id);
/* copies the five columns out (each pointer may be NULL to skip that column) */
int bbkio_table_copy(const BbkioTable* t, int32_t* chr1, int64_t* mid1, int32_t* chr2, int64_t* mid2, int64_t* count);
void bbkio_table_free(BbkioTable* t);

/* The packed form of a pass' p / q columns (bbk_pack_scores, bbk.h: two bits per row + the values that are not 1.0 / NaN)
 * back into dense columns, bit for bit.  codes: one uint32 per 16 rows; chunks: 24-byte records {uint64 base_p, uint64 base_q,
 * uint32 n_p, uint32 n_q}, one per 4096 rows; q may be NULL.  threads <= 0: all online cores. */
int bbkio_unpack_scores(const uint32_t* codes, const void* chunks, const double* values_p, const double* values_q,
                        int64_t m, double* p, double* q, int32_t threads);
/* the same, and keep[i] = (p[i] <= 1): the rows the reference emits (fithic.py:434) */
int bbkio_unpack_scores_keep(const uint32_t* codes, const void* chunks, const double* values_p, const double* values_q,
                             int64_t m, double* p, double* q, uint8_t* keep, int32_t threads);
/* a large host copy by `threads` cores (<= 0: all): numpy columns into pinned staging memory and back */
int bbkio_copy_bytes(void* dst, const void* src, size_t n, int32_t threads);

/* The packed contact records of a pass (format: bbk.h, BbkRecHeader), written from the shards' own int32 columns (any host
 * memory) straight into the pass layout: shard i of sizes[i] rows starts at row starts[i] of layout_rows(sizes) (every start
 * a multiple of 4), the padding rows between shards are zeros.  Two phases over the chunks by all cores (frames of
 * reference, then bits); the bytes do not depend on `threads` (<= 0: all online cores).  *bytes receives the size; a
 * capacity below it fails the call (BBKIO_E_INVALID, *bytes still set).  bbkio_pack_records_bound(rows) is the largest
 * size `rows` layout rows can take. */
uint64_t bbkio_pack_records_bound(int64_t rows);
int bbkio_pack_records(const int32_t* const* mid1, const int32_t* const* mid2, const int32_t* const* count, const int64_t* sizes,
                       int32_t n_shards, void* out, uint64_t capacity, uint64_t* bytes, int32_t threads);
/* BBKIO_OK when buf[0 .. bytes) is a packed record buffer of `rows` rows that bbk_unpack_records may read: header, chunk
 * offsets in bounds, aligned and increasing, bits within their limits, every payload ending within the buffer.
 * BBKIO_E_INVALID otherwise (bbkio_last_error says why). */
int bbkio_check_records(const void* buf, uint64_t bytes, int64_t rows);

/* "{}".format(float64) into buf (at least 32 bytes); returns the length.  Exposed for the parity tests. */
int bbkio_format_double(double x, char* buf);

#ifdef __cplusplus
}
#endif
#endif
