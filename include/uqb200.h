/* uqb200.h - C ABI of libuqb200.so: the B200 (sm_100a) device path of uQ's FASTQ->uQ encode and
 * uQ->FASTQ decode hot path.
 *
 * The reference (JohnLonginotto/uq, uq.py) has no FFI for this path: it is inline Python.  Each
 * entry point below replaces the reference code region cited beside it; INTEGRATION.md shows the
 * ctypes stub a maintainer would splice into uq.py at that region.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns 0 on success, non-zero on error
 *     (text via uqb_last_error); nothing throws, nothing calls exit().
 *   - one uqb_ctx per host thread; calls are synchronous with respect to the host unless stated.
 *   - device objects are opaque handles released with the matching *_free.
 *   - all integer table data is little-endian on the host side, exactly as numpy stores it.
 *   - there is NO CPU fallback: every entry point runs CUDA kernels on the context's device.
 */
#ifndef UQB200_H
#define UQB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UQB_VERSION 101
#define UQB_HDR_MAX 1024          /* longest first/last QNAME line the analysis reports on */
#define UQB_MAX_COLS 64           /* QNAME columns (separators + 1) */
#define UQB_MAX_CHECKPOINTS 40    /* Pass-2 checkpoints 10000*2^k (uq.py:572, 634-636) */
#define UQB_NONE_I64 INT64_MAX

typedef struct uqb_ctx uqb_ctx;
typedef struct uqb_fastq uqb_fastq;   /* device-resident FASTQ bytes + line offsets + QNAME scan results */
typedef struct uqb_array uqb_array;   /* device array: n rows x width bytes */

/* ---- context ------------------------------------------------------------------------------- */
int         uqb_version(void);
/* `stream` is a cudaStream_t (or NULL for a private stream); kernels of this context are launched
 * on it so that callers can time the path with events recorded on the same stream. */
int         uqb_ctx_create(int device, void* stream, uqb_ctx** out);
void        uqb_ctx_destroy(uqb_ctx* ctx);
const char* uqb_last_error(const uqb_ctx* ctx);
int         uqb_ctx_sync(uqb_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t    uqb_ctx_launch_count(const uqb_ctx* ctx);
/* per-kernel device timing (CUDA events around every launch on the context's stream).
 * report: writes up to cap entries "name\0" packed in names (each UQB_TIMER_NAME bytes),
 * launches[i], ms[i], algorithmic_bytes[i] (compulsory reads+writes summed over the launches; 0 for
 * kernels that are not annotated); returns the number of distinct kernels through *n. */
#define UQB_TIMER_NAME 48
int         uqb_ctx_timing(uqb_ctx* ctx, int enable);
int         uqb_ctx_timing_report(uqb_ctx* ctx, char* names, uint64_t* launches, double* ms, uint64_t* algorithmic_bytes, int cap, int* n);
int         uqb_ctx_timing_reset(uqb_ctx* ctx);
/* CUDA-event time between two points of the context's stream (device timeline, host gaps included) */
int         uqb_ctx_span_begin(uqb_ctx* ctx);
int         uqb_ctx_span_end(uqb_ctx* ctx, double* ms);
/* pinned host memory for end-to-end paths (cudaHostAlloc / cudaFreeHost) */
int         uqb_host_alloc(uqb_ctx* ctx, uint64_t nbytes, void** out);
int         uqb_host_free(uqb_ctx* ctx, void* p);
/* bytes currently allocated on the device by this context / free device memory */
int         uqb_mem_info(uqb_ctx* ctx, uint64_t* in_use, uint64_t* dev_free, uint64_t* dev_total);

/* ---- arrays -------------------------------------------------------------------------------- */
int uqb_array_info(const uqb_array* a, uint64_t* n, uint32_t* width);
int uqb_array_alloc(uqb_ctx* ctx, uint64_t n, uint32_t width, uqb_array** out);      /* uninitialised */
int uqb_array_upload(uqb_ctx* ctx, const void* host, uint64_t n, uint32_t width, uqb_array** out);
int uqb_array_download(uqb_ctx* ctx, const uqb_array* a, void* host, uint64_t nbytes);
/* D2H on the copy stream, ordered after all work queued so far on the compute stream.  `host` should be
 * pinned; the array must stay allocated until uqb_ctx_copy_sync returns. */
int uqb_array_download_async(uqb_ctx* ctx, const uqb_array* a, void* host, uint64_t nbytes);
int uqb_ctx_copy_sync(uqb_ctx* ctx);
/* index of the first differing byte of two device arrays, -1 if identical (round-trip checks at full size) */
int uqb_array_first_difference(uqb_ctx* ctx, const uqb_array* a, const uqb_array* b, int64_t* first);
int uqb_array_free(uqb_ctx* ctx, uqb_array* a);
void* uqb_array_device_ptr(const uqb_array* a);   /* for benches/tests that adopt device memory */
/* non-owning view of device memory (a peer GPU's window, another context's array): uqb_array_free releases the view only */
int uqb_array_wrap(uqb_ctx* ctx, void* dev, uint64_t n, uint32_t width, uqb_array** out);
/* device -> device copy of nbytes from src_dev (any device pointer this process can address, peer memory included)
 * into dst at byte offset dst_offset, on the context's stream */
int uqb_array_copy_in(uqb_ctx* ctx, uqb_array* dst, uint64_t dst_offset, const void* src_dev, uint64_t nbytes);

/* ---- stage 1: load + record splitting  (replaces open()/next(f) uq.py:339-342, 378-385 and the
 *      `wc -l` record count uq.py:85-87) -------------------------------------------------------- */
typedef struct {
    uint64_t n_bytes;
    uint64_t n_lines;      /* number of '\n' bytes */
    uint64_t n_reads;      /* n_lines / 4 */
    int32_t  status;       /* 0 ok, 1 = line count not divisible by 4 (uq.py:86-87) */
    int32_t  _pad;
} uqb_split_info;

int uqb_fastq_load(uqb_ctx* ctx, const uint8_t* host, uint64_t nbytes, uqb_fastq** out);      /* H2D */
/* adopt bytes already in HBM (not copied, not freed): used when inputs are device-resident */
int uqb_fastq_adopt(uqb_ctx* ctx, const uint8_t* dev, uint64_t nbytes, uqb_fastq** out);
/* H2D in chunks on a second stream while the compute stream splits and analyses every chunk that has
 * landed: when the call returns, uqb_split / uqb_analyze on the handle only return the cached results.
 * `host` should be pinned (uqb_host_alloc) for the copies to overlap; chunk_bytes 0 = 256 MiB.
 * ref / ref_len / rbase: a multi-GPU shard, as uqb_fastq_set_reference (rbase > 0 = this shard does not start the
 * file); ref NULL, ref_len 0, rbase 0 = the handle is the whole file. */
int uqb_fastq_load_streamed(uqb_ctx* ctx, const uint8_t* host, uint64_t nbytes, uint64_t chunk_bytes,
                            const uint8_t* ref, uint32_t ref_len, uint64_t rbase, uqb_fastq** out);
int uqb_fastq_free(uqb_ctx* ctx, uqb_fastq* fq);
int uqb_fastq_download(uqb_ctx* ctx, const uqb_fastq* fq, uint64_t offset, uint8_t* host, uint64_t nbytes);
int uqb_split(uqb_ctx* ctx, uqb_fastq* fq, uqb_split_info* info);
/* line offsets (uint64[n_lines+1], offset of the first byte of every line) for tests */
int uqb_fastq_line_offsets(uqb_ctx* ctx, const uqb_fastq* fq, uint64_t first, uint64_t count, uint64_t* host);

/* ---- stage 1: Pass-1 statistics  (replaces uq.py:342-425; the decisions uq.py:427-545 stay in
 *      host Python and consume this struct) --------------------------------------------------- */
typedef struct {
    uint64_t base_count[256];        /* base_graph, uq.py:448-451 */
    uint64_t qual_count[256];        /* qual_graph, uq.py:452 */
    /* static_qualities (uq.py:369-375, 420-425) reduced to what the N-trick reads (uq.py:480-494):
     * -1 base byte absent, 0..255 the only quality byte this base ever has, 256 = two or more */
    int32_t  base_single_qual[256];
    uint64_t dna_min, dna_max;       /* uq.py:356-357, 416-417 */
    int64_t  bad_first_char;         /* 0 if line 1 does not start with '@' (uq.py:346), else -1 */
    int64_t  bad_plus_record;        /* first record whose 3rd line does not start with '+' (uq.py:360, 382), -1 none */
    int64_t  bad_len_record;         /* first record with len(SEQ) != len(QUAL) (uq.py:366, 388), -1 none */
    uint32_t first_len, last_len;    /* QNAME line lengths (no newline) of the first / last record */
    uint8_t  first_name[UQB_HDR_MAX];
    uint8_t  last_name[UQB_HDR_MAX];
    uint32_t max_name_len;           /* longest QNAME line */
    uint32_t prefix_len, suffix_len; /* common prefix / suffix of all QNAME lines (uq.py:395-408) */
    /* last record whose count of byte c differs from the first QNAME's count of c; -1 none.
     * With first_lcp_eq this reproduces the order-dependent separator survival of uq.py:395-413. */
    int64_t  last_count_mismatch[256];
    int64_t  first_lcp_eq[UQB_HDR_MAX + 1];   /* first record k>=1 whose common prefix with line 1 has length j */
    int64_t  first_lcs_eq[UQB_HDR_MAX + 1];   /* same for the common suffix */
    int64_t  first_short_prefix[UQB_HDR_MAX + 1]; /* first record that IS a proper prefix of line 1, by its length (Q8) */
    int64_t  first_short_suffix[UQB_HDR_MAX + 1];
} uqb_stats;

int uqb_analyze(uqb_ctx* ctx, uqb_fastq* fq, uqb_stats* out);
/* multi-GPU shards: the handle holds records [rbase, rbase+n) of a larger file whose first QNAME line is
 * `name`; uqb_analyze then measures prefixes / suffixes / byte counts against that line (indices stay local) */
int uqb_fastq_set_reference(uqb_ctx* ctx, uqb_fastq* fq, const uint8_t* name, uint32_t len, uint64_t rbase);

/* ---- stage 1b: QNAME tokenisation + Pass-2 column statistics (replaces qname_reader and the
 *      Pass-2 loop uq.py:557-638; the typing decisions uq.py:586-602, 641-676 stay in Python) -- */
typedef struct {
    uint8_t  all_int;          /* every token matches [+-]?[0-9]+ */
    uint8_t  all_canonical;    /* every token equals str(int(token)) */
    uint8_t  overflow;         /* some integer token does not fit int64 */
    uint8_t  _pad[5];
    int64_t  min_val, max_val; /* over integer tokens */
    uint32_t min_len, max_len; /* token byte lengths */
    uint64_t n_distinct;       /* distinct tokens over all records */
    uint32_t n_checkpoints;    /* number of k with 10000*2^k <= n_reads-1 */
    uint32_t _pad2;
    uint64_t distinct_at[UQB_MAX_CHECKPOINTS]; /* distinct tokens among records [0 .. 10000*2^k] */
} uqb_colstats;

/* seps: the ordered separator string (uq.py:438-439).  bad_record: first record whose separator
 * sequence differs (the reference falls back / exits at uq.py:609-613, 637), -1 if none.
 * col_mode: one mode per column (NULL = all 0): 0 automatic, 1 no dictionary wanted (the column is known to
 * leave 'mapping'), 2 dictionary forced (skip the checkpoint-0 shortcut) - used by multi-GPU merges */
int uqb_qname_scan(uqb_ctx* ctx, uqb_fastq* fq, uint32_t prefix_len, uint32_t suffix_len,
                   const uint8_t* seps, uint32_t nseps, const uint8_t* col_mode, uqb_colstats* cols, int64_t* bad_record);
/* first record (local index) holding each dictionary entry, uint32[count] */
int uqb_qname_dict_first(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint32_t* host, uint64_t count);
/* sorted dictionary of a column (uq.py:659-661): count rows x width bytes, zero padded */
int uqb_qname_dict_info(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint64_t* count, uint32_t* width);
int uqb_qname_dict(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint8_t* host, uint64_t nbytes);

typedef struct {
    uint8_t  format;     /* 0 mapping (bisect_left rank, uq.py:724), 1 integers (uq.py:725-726),
                            2 strings (declared extension E1: the token's bytes, left-aligned, zero padded) */
    uint8_t  itemsize;   /* 1, 2, 4, 8; for strings the width W (1..255): at least the longest token */
    uint8_t  offset;     /* subtract min (uq.py:725) */
    uint8_t  _pad[5];
    int64_t  min_val;
} uqb_colspec;
/* Pass 4 (uq.py:717-735): one little-endian array per column, width = itemsize (strings: W bytes per record) */
int uqb_qname_encode(uqb_ctx* ctx, uqb_fastq* fq, uint32_t ncols, const uqb_colspec* spec, uqb_array** cols);

/* ---- stage 2: symbol mapping + bit packing (replaces encoder_fixed uq.py:108-182 and
 *      encoder_variable uq.py:188-254; call site uq.py:707-708) ------------------------------- */
typedef struct {
    uint8_t  base_code[256];   /* bases.index(ch); tricked bases -> 0 (N_base, uq.py:130, 152) */
    uint8_t  qual_code[256];   /* qualities.index(ch) */
    int16_t  trick_qual[256];  /* N_qual[base] for tricked base bytes (uq.py:153), -1 otherwise */
    uint32_t bits_per_base, bits_per_quality;
    uint32_t dna_bytes, qual_bytes;     /* row widths, uq.py:514-515, 543-544 */
    uint32_t variable;                  /* variable_read_lengths: marker bit (uq.py:242-243) */
    uint32_t dna_max;
} uqb_pack_params;
int uqb_pack(uqb_ctx* ctx, uqb_fastq* fq, const uqb_pack_params* p, uqb_array** dna, uqb_array** qual);

/* ---- stage 3: sort / unique (replaces numpy.argsort / numpy.unique / fancy indexing in
 *      encode_dna_qual uq.py:765-805 and encode_qname uq.py:808-851) -------------------------- */
/* Stable sort of the rows of `table` in memcmp order.  Any of the outputs may be NULL.
 *   perm       : uint32[n]  stable argsort                        (numpy.argsort(kind='stable'))
 *   key        : uint32[n]  index of each row in the unique table  (numpy.unique return_inverse)
 *   key_sorted : uint32[n]  key[perm], i.e. the key in sorted order (key[argsort(key)], uq.py:796-798)
 *   uniq       : [n_unique][width] distinct rows ascending         (numpy.unique)               */
int uqb_sort_rows(uqb_ctx* ctx, const uqb_array* table, uqb_array** perm, uqb_array** key,
                  uqb_array** key_sorted, uqb_array** uniq, uint64_t* n_unique);
int uqb_gather_rows(uqb_ctx* ctx, const uqb_array* table, const uqb_array* perm, uqb_array** out); /* out[i] = table[perm[i]] */
int uqb_add_scalar_u32(uqb_ctx* ctx, uqb_array* a, uint32_t value);   /* a[i] += value, uint32 array */
/* lower_bound of k host rows in a table sorted in memcmp order (splitter search of the multi-GPU sample sort) */
int uqb_rows_lower_bound(uqb_ctx* ctx, const uqb_array* sorted_table, const uint8_t* probes_host, uint32_t k, uint64_t* out_host);
/* partition-first sample sort (multi-GPU, replaces nothing in uq.py: the reference is single process): rows are sent
 * to rank d = number of splitter keys <= big-endian first 8 bytes of the row.  The table is read once, sequentially.
 * pos = uint32[n], pos[i] = index of row i in the destination-grouped, stable order; counts_host[0..nsplit] = rows per
 * destination */
int uqb_partition_positions(uqb_ctx* ctx, const uqb_array* table, const uint64_t* split_keys_host, uint32_t nsplit,
                            uqb_array** pos, uint64_t* counts_host);
/* exchange buffers of the sample sort: byte arrays in which every segment starts at a multiple of `align` bytes (NCCL
 * moves 16 bytes per thread only between 16-byte aligned pointers); seg_offsets_host receives the byte offset of every
 * segment.  uqb_scatter_rows_segmented: row i of `table` (the partitioned table itself, or any per-record payload that
 * has to follow it) lands at byte seg_offsets[d] + (pos[i] - first row of d) * width; rows of up to 224 bytes.
 * uqb_gather_rows_segmented: the same buffer from order = pos^-1 (rows of any width): the rows of segment d are
 * table[order[first_d .. first_d + seg_counts[d])). */
int uqb_scatter_rows_segmented(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, uint32_t nseg,
                               const uint64_t* seg_counts_host, uint32_t align, uqb_array** out, uint64_t* seg_offsets_host);
int uqb_gather_rows_segmented(uqb_ctx* ctx, const uqb_array* table, const uqb_array* order, uint32_t nseg,
                              const uint64_t* seg_counts_host, uint32_t align, uqb_array** out, uint64_t* seg_offsets_host);
/* device-initiated exchange: the rows of segment d go straight to the device address dst_addrs_host[d] (dense, in position
 * order) - normally the receive buffer of rank d mapped into this process (peer memory over NVLink).  The caller brackets
 * the call with its own barriers. */
int uqb_scatter_rows_to(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, uint32_t nseg,
                        const uint64_t* seg_counts_host, const uint64_t* dst_addrs_host);
/* the inverse on the receiving side: byte array with aligned segments -> dense table of `width`-byte rows */
int uqb_compact_segments(uqb_ctx* ctx, const uqb_array* padded, uint32_t nseg, const uint64_t* seg_offsets_host,
                         const uint64_t* seg_counts_host, uint32_t width, uqb_array** out);
/* out[idx[j]] = src[j], uint32 arrays, idx a permutation (inverse of uqb_gather_rows) */
int uqb_scatter_u32(uqb_ctx* ctx, const uqb_array* src, const uqb_array* idx, uqb_array** out);
/* the inverse on the decode side: an index member read from a container (itemsize 1/2/4/8, uq.py:953, 957, 973) widened to
 * uint32 and checked: first_bad = first position whose value is >= bound (rows of the table it indexes), -1 if none */
int uqb_index_u32(uqb_ctx* ctx, const uqb_array* a, uint64_t bound, uqb_array** out, int64_t* first_bad);
/* uint32 -> little-endian integer of itemsize bytes (key.astype(min_scalar_type(max)), uq.py:790) */
int uqb_narrow_u32(uqb_ctx* ctx, const uqb_array* a, uint32_t itemsize, uqb_array** out);
/* QNAME columns <-> rows in sort-key form: columns concatenated at their own widths, which makes memcmp order equal
 * numpy's field-by-field comparison (uq.py:814-816, 828-830).  kinds: one kind per column (NULL = all 0): 0 little-endian
 * integer (stored big-endian in the row: unsigned comparison), 1 bytes copied in order ('strings' columns, E1: memcmp of
 * zero-padded bytes is numpy's order of S values) */
int uqb_columns_to_rows(uqb_ctx* ctx, uint32_t ncols, uqb_array* const* cols, const uint8_t* kinds, uqb_array** rows);
int uqb_rows_to_columns(uqb_ctx* ctx, const uqb_array* rows, uint32_t ncols, const uint32_t* itemsizes, const uint8_t* kinds,
                        uqb_array** cols);
/* integer columns (itemsize 1/2/4/8) whose value ranges fit 64 bits together -> one packed sort key per row:
 * key = sum over c of (cols[c][i] - bases[c]) << shifts[c], field c `bits[c]` wide (0: a constant column), the first column
 * in the highest bits.  Its numeric order is the memcmp order of the rows of uqb_columns_to_rows.  `table` is a table of
 * 8-byte rows for uqb_sort_rows only, which sorts it by the key alone: its row bytes are the key itself (little-endian),
 * not memcmp rows.  The unique table uqb_sort_rows returns for it holds the distinct keys as 8 big-endian bytes;
 * uqb_key_to_columns unpacks such rows into columns of itemsizes[c] bytes: (field c) + bases[c]. */
int uqb_columns_to_key(uqb_ctx* ctx, uint32_t ncols, uqb_array* const* cols, const uint32_t* shifts, const uint32_t* bits,
                       const uint64_t* bases, uqb_array** table);
int uqb_key_to_columns(uqb_ctx* ctx, const uqb_array* keys, uint32_t ncols, const uint32_t* itemsizes, const uint32_t* shifts,
                       const uint32_t* bits, const uint64_t* bases, uqb_array** cols);

/* ---- stage 4: physical layouts (replaces write_pattern uq.py:257-270) ------------------------ */
/* pattern ids: 0='0.1' 1='1.1' 2='2.1' 3='3.1' 4='0.2' 5='1.2' 6='2.2' 7='3.2'.  Produces the exact
 * byte stream numpy.save writes after the NPY header (n*width bytes). */
int uqb_layout(uqb_ctx* ctx, const uqb_array* table, int pattern, uqb_array** stream);
/* inverse (load_from_tar uq.py:943-945): stream bytes -> logical table [n][width] */
int uqb_unlayout(uqb_ctx* ctx, const uqb_array* stream, uint64_t n, uint32_t width, int pattern, uqb_array** table);

/* ---- stage 5: decode (replaces uq.py:1002-1058) -------------------------------------------- */
typedef struct {
    uint8_t  format, itemsize, offset, _pad[5];   /* format and itemsize as in uqb_colspec; strings: text = bytes up to the first NUL */
    int64_t  min_val;
    const uint8_t* dict;       /* host: mapping strings, dict_count rows x dict_width bytes zero padded */
    uint64_t dict_count;
    uint32_t dict_width, _pad2;
} uqb_decode_col;
typedef struct {
    uint8_t  base_char[256];   /* bases[code] */
    uint8_t  qual_char[256];   /* qualities[code] */
    int16_t  qual_to_base[256];/* qual_N: quality code -> restored base byte (uq.py:999, 1036), -1 none */
    uint32_t bits_per_base, bits_per_quality, variable, dna_max;
    const uint8_t* prefix; uint32_t prefix_len, _p0;
    const uint8_t* suffix; uint32_t suffix_len, _p1;
    const uint8_t* seps;   uint32_t nseps, ncols;
    const uqb_decode_col* cols;
} uqb_decode_params;
/* dna/qual: logical tables [n][bytes] (already expanded through their keys with uqb_gather_rows),
 * cols: ncols arrays [n][itemsize].  Output: device byte array holding the FASTQ text. */
int uqb_decode(uqb_ctx* ctx, const uqb_array* dna, const uqb_array* qual, uqb_array* const* cols,
               const uqb_decode_params* p, uqb_array** fastq);

/* ---- verification of an encode (no reference counterpart: uq.py never reads back what it wrote) ----------- */
typedef struct {
    uint64_t records;        /* container rows compared */
    uint64_t differ[4];      /* rows whose line k differs: 0 name, 1 sequence, 2 '+' line, 3 quality */
    int64_t  first_row[4];   /* smallest such container row, -1 none */
    int64_t  first_src[4];   /* its input record number */
} uqb_verify_report;
/* src: the encoded FASTQ; text: decoded rows [first_row, first_row + k) as a uqb_fastq (adopted + split, k = its records);
 * order: uint32[n] container row -> input record, NULL = identity.  Compares the four lines of decoded record i - first_row
 * with those of input record order[i], lengths first, then bytes; an order value >= the input's record count is a
 * difference in all four fields and is not dereferenced.  Accumulates into *report, whose first_row entries the caller
 * starts at -1. */
int uqb_verify_records(uqb_ctx* ctx, const uqb_fastq* src, const uqb_fastq* text, uint64_t first_row,
                       const uqb_array* order, uqb_verify_report* report);
/* missing = smallest value in [0, n) that order does not hold, -1 if order (of length n) is a permutation of [0, n) */
int uqb_check_permutation(uqb_ctx* ctx, const uqb_array* order, uint64_t n, int64_t* missing);

/* ---- synthetic inputs for bench/tests (same generator as oracle/synth.py, oracle/synth_umi.py) - */
typedef struct {
    uint32_t kind;        /* 0 illumina, 1 genome, 2 casava, 3 ont, 4 umi (illumina header + '_' + 6-12 of ACGTN),
                             5 renamed (@SRR0000001.<record+1>), 6 mixed (blocks of 1024 records alternate between the
                             casava header and the pre-1.8 @HWI-D00123:<lane>:<tile>:<x>:<y>#0/1) */
    uint32_t length;      /* read length (kinds 0-2, 4-6) */
    uint32_t len_lo, len_hi; /* kind 3 */
    uint64_t seed, first, n; /* records first .. first+n-1 */
    uint64_t genome, pool;   /* kind 1 */
} uqb_synth_params;
int uqb_synth(uqb_ctx* ctx, const uqb_synth_params* p, const int64_t* ont_len_table /*4096 or NULL*/, uqb_array** bytes);

#ifdef __cplusplus
}
#endif
#endif
