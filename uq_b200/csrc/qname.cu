// Stage 1b: QNAME tokenisation, Pass-2 column statistics and Pass-4 column encoding.
// Replaces qname_reader (uq.py:557-570), the Pass-2 loop (uq.py:604-638) and Pass 4 (uq.py:717-735).
// The typing *decisions* (check_format uq.py:586-602, final typing uq.py:641-676) stay in host Python
// and consume uqb_colstats.
//
// Tokenising: for well-formed input re.split('(.*)'.join(separators), middle) equals "cut the middle
// part at every separator character, which must appear in exactly the order of `separators`"
// (SURVEY A.5); any record that violates the order is reported through bad_record and the host
// raises the reference's error.
//
// Distinct-token counts (len(column['map']) at the checkpoints 10000*2^k and at the end) and the
// sorted dictionary of a mapping column come from the stable row sort of sort.cu applied to the
// zero-padded token bytes: memcmp order of zero-padded rows is Python's str ordering as long as no
// token contains a NUL byte (rejected).
#include "common.cuh"

#define QN 256
#define SPAN_LEN_BITS 14
#define SPAN_MAXLEN ((1u << SPAN_LEN_BITS) - 1u)
#define FLAG_NONINT (1u << 28)
#define FLAG_NONCANON (1u << 29)
#define FLAG_OVERFLOW (1u << 30)
#define FLAG_TOOLONG (1u << 31)

struct qn_params {
    uint32_t prefix_len, suffix_len, nseps;
    uint8_t seps[UQB_MAX_COLS];
    uint32_t sepmask[8];
    int64_t* val[UQB_MAX_COLS];
    uint32_t* span[UQB_MAX_COLS];
};

struct qn_flags { long long bad_record; unsigned int has_nul; unsigned int pad; };

__global__ void __launch_bounds__(QN) k_qname_tokens(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off, uint64_t n_reads,
                                                    qn_params P, qn_flags* __restrict__ flags,
                                                    const uint8_t* __restrict__ names, uint32_t name_pitch) {
    const uint64_t r = (uint64_t)blockIdx.x * QN + threadIdx.x;
    if (r >= n_reads) return;
    // names != nullptr: QNAME lines from the compact side array (uqb_fastq::names, row r: length byte + text)
    uint64_t n;
    const uint8_t* name;
    if (names) {
        name = names + r * name_pitch + 1;
        n = name[-1];
    } else {
        const uint64_t o0 = line_off[4 * r];
        n = line_off[4 * r + 1] - o0 - 1;
        name = d + o0;
    }
    uint64_t mid_start = P.prefix_len;
    uint64_t mid_end = n > P.suffix_len ? n - P.suffix_len : 0;
    if (mid_end < mid_start) mid_end = mid_start;
    if (mid_start > n) { mid_start = n; mid_end = n; }

    uint32_t col = 0;
    uint64_t tok_start = mid_start;
    bool neg = false, sign = false, nonint = false, lead_zero = false, overflow = false, bad = false;
    uint32_t ndig = 0;
    unsigned long long val = 0;
    for (uint64_t i = mid_start; i <= mid_end; i++) {
        const bool at_end = i == mid_end;
        unsigned ch = at_end ? 0u : __ldg(name + i);
        const bool is_sep = !at_end && ((P.sepmask[ch >> 5] >> (ch & 31u)) & 1u);
        if (at_end || is_sep) {
            if (is_sep && (col >= P.nseps || ch != P.seps[col])) { bad = true; break; }
            // ---- finalise token `col` = name[tok_start, i) ----
            const uint64_t len = i - tok_start;
            const bool is_int = !nonint && ndig >= 1;
            if (neg ? val > 9223372036854775808ull : val > 9223372036854775807ull) overflow = true;
            const bool canonical = is_int && !(sign && !neg) && !(lead_zero && ndig > 1) && !(neg && val == 0);
            uint32_t sp;
            const uint64_t rel = tok_start - mid_start;
            if (len > SPAN_MAXLEN || rel > SPAN_MAXLEN) sp = FLAG_TOOLONG;
            else sp = (uint32_t)len | ((uint32_t)rel << SPAN_LEN_BITS);
            if (!is_int) sp |= FLAG_NONINT;
            if (!canonical) sp |= FLAG_NONCANON;
            if (overflow) sp |= FLAG_OVERFLOW;
            if (col <= P.nseps) {
                P.val[col][r] = is_int ? (neg ? -(long long)val : (long long)val) : 0ll;
                P.span[col][r] = sp;
            }
            col++;
            tok_start = i + 1;
            neg = sign = nonint = lead_zero = overflow = false;
            ndig = 0; val = 0;
        } else {
            if (ch == 0u) atomicOr(&flags->has_nul, 1u);
            if (ch >= '0' && ch <= '9') {
                const unsigned dgt = ch - '0';
                if (ndig == 0 && dgt == 0) lead_zero = true;
                if (val > 922337203685477580ull || (val == 922337203685477580ull && dgt > 8)) overflow = true;
                else val = val * 10ull + dgt;
                ndig++;
            } else if ((ch == '+' || ch == '-') && i == tok_start) {
                sign = true;
                neg = ch == '-';
            } else {
                nonint = true;
            }
        }
    }
    if (bad || col != P.nseps + 1) atomicMin(&flags->bad_record, (long long)r);
}

struct col_red {
    long long min_val, max_val;
    unsigned int min_len, max_len;
    unsigned int any_flags;     // OR of the flag bits over all tokens
    unsigned int pad;
};

__global__ void k_col_red_init(col_red* c, int ncols) {
    int i = threadIdx.x;
    if (i < ncols) { c[i].min_val = LLONG_MAX; c[i].max_val = LLONG_MIN; c[i].min_len = 0xFFFFFFFFu; c[i].max_len = 0; c[i].any_flags = 0; c[i].pad = 0; }
}

__global__ void __launch_bounds__(QN) k_col_reduce(const int64_t* __restrict__ val, const uint32_t* __restrict__ span, uint64_t n,
                                                  col_red* __restrict__ out) {
    long long mn = LLONG_MAX, mx = LLONG_MIN;
    unsigned lmin = 0xFFFFFFFFu, lmax = 0, fl = 0;
    // the value is loaded next to the span, not behind it (it is simply not used for a non-integer token): two independent
    // loads per item and four items in flight per thread instead of a chain of two dependent loads
#pragma unroll 4
    for (uint64_t i = (uint64_t)blockIdx.x * QN + threadIdx.x; i < n; i += (uint64_t)gridDim.x * QN) {
        const uint32_t sp = __ldg(span + i);
        const long long v = __ldg(val + i);
        fl |= sp & 0xF0000000u;
        if (!(sp & FLAG_NONINT)) {
            mn = v < mn ? v : mn; mx = v > mx ? v : mx;
        }
        const unsigned len = sp & SPAN_MAXLEN;
        lmin = len < lmin ? len : lmin; lmax = len > lmax ? len : lmax;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        unsigned c = __shfl_xor_sync(0xffffffffu, lmin, o), e = __shfl_xor_sync(0xffffffffu, lmax, o);
        fl |= __shfl_xor_sync(0xffffffffu, fl, o);
        mn = a < mn ? a : mn; mx = b > mx ? b : mx; lmin = c < lmin ? c : lmin; lmax = e > lmax ? e : lmax;
    }
    if (lane_id() == 0) {
        atomicMin(&out->min_val, mn);
        atomicMax(&out->max_val, mx);
        atomicMin(&out->min_len, lmin);
        atomicMax(&out->max_len, lmax);
        atomicOr(&out->any_flags, fl);
    }
}

// zero-padded token bytes of records [0, n) as rows of `w` bytes
__global__ void __launch_bounds__(QN) k_token_rows(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                  const uint32_t* __restrict__ span, uint32_t prefix_len, uint32_t w, uint64_t n,
                                                  uint8_t* __restrict__ rows, const uint8_t* __restrict__ names, uint32_t name_pitch) {
    const uint64_t r = (uint64_t)blockIdx.x * QN + threadIdx.x;
    if (r >= n) return;
    const uint32_t sp = span[r];
    const uint32_t len = sp & SPAN_MAXLEN, rel = (sp >> SPAN_LEN_BITS) & SPAN_MAXLEN;
    const uint8_t* src = (names ? names + r * name_pitch + 1 : d + line_off[4 * r]) + prefix_len + rel;
    uint8_t* dst = rows + r * w;
    for (uint32_t i = 0; i < w; i++) dst[i] = i < len ? __ldg(src + i) : (uint8_t)0;
}

__global__ void __launch_bounds__(QN) k_rank_and_first(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ gid, uint64_t n,
                                                      uint32_t* __restrict__ rank, uint32_t* __restrict__ first_row) {
    const uint64_t p = (uint64_t)blockIdx.x * QN + threadIdx.x;
    if (p >= n) return;
    const uint32_t g = gid[p], row = perm[p];
    rank[row] = g;
    if (p == 0 || gid[p - 1] != g) first_row[g] = row;    // stable sort: the group's first row is its first occurrence
}

// hist[k] = number of distinct tokens whose first occurrence lies in (T_{k-1}, T_k], T_k = 10000 * 2^k;
// hist[ncheck] collects the rest
__global__ void __launch_bounds__(QN) k_first_occ_hist(const uint32_t* __restrict__ first_row, uint64_t u, uint32_t ncheck,
                                                      unsigned long long* __restrict__ hist) {
    __shared__ unsigned sh[UQB_MAX_CHECKPOINTS + 1];
    if (threadIdx.x <= UQB_MAX_CHECKPOINTS) sh[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t g = (uint64_t)blockIdx.x * QN + threadIdx.x; g < u; g += (uint64_t)gridDim.x * QN) {
        const uint64_t f = first_row[g];
        uint32_t k = 0;
        uint64_t t = 10000;
        while (k < ncheck && f > t) { k++; t *= 2; }
        atomicAdd(&sh[k], 1u);
    }
    __syncthreads();
    if (threadIdx.x <= ncheck && sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}

__global__ void __launch_bounds__(QN) k_dict_rows(const uint8_t* __restrict__ rows, uint32_t w, const uint32_t* __restrict__ first_row,
                                                 uint64_t u, uint8_t* __restrict__ dict) {
    for (uint64_t t = (uint64_t)blockIdx.x * QN + threadIdx.x; t < u * w; t += (uint64_t)gridDim.x * QN) {
        const uint64_t g = t / w;
        const uint32_t b = (uint32_t)(t - g * w);
        dict[t] = rows[(uint64_t)first_row[g] * w + b];
    }
}

int uqb_fastq_free_qcols(uqb_ctx* ctx, uqb_fastq* fq);

static int distinct_of_prefix(uqb_ctx* ctx, uqb_fastq* fq, const uqb_qcol& qc, uint32_t w, uint64_t n, uint64_t* distinct) {
    uint8_t* rows;
    UQB_TRY(uqb_dalloc(ctx, (void**)&rows, n * w + 64));
    if (w) UQB_LAUNCH(k_token_rows, uqb_blocks(n, QN), QN, 0, fq->d, fq->line_off, qc.span, fq->prefix_len, w, n, rows, (const uint8_t*)fq->names, fq->name_pitch);
    uint32_t *perm, *gid;
    UQB_TRY(uqb_sort_rows_impl(ctx, rows, n, w, &perm, &gid, distinct));
    UQB_TRY(uqb_dfree(ctx, perm, n * 4));
    UQB_TRY(uqb_dfree(ctx, gid, n * 4));
    UQB_TRY(uqb_dfree(ctx, rows, n * w + 64));
    return 0;
}

extern "C" int uqb_qname_scan(uqb_ctx* ctx, uqb_fastq* fq, uint32_t prefix_len, uint32_t suffix_len,
                              const uint8_t* seps, uint32_t nseps, uqb_colstats* cols, int64_t* bad_record) {
    return uqb_qname_scan_ex(ctx, fq, prefix_len, suffix_len, seps, nseps, nullptr, cols, bad_record);
}

extern "C" int uqb_qname_scan_ex(uqb_ctx* ctx, uqb_fastq* fq, uint32_t prefix_len, uint32_t suffix_len,
                                 const uint8_t* seps, uint32_t nseps, const uint8_t* col_mode,
                                 uqb_colstats* cols, int64_t* bad_record) {
    if (!fq->line_off) return uqb_fail(ctx, "uqb_qname_scan: call uqb_split first");
    if (nseps + 1 > UQB_MAX_COLS) return uqb_fail(ctx, "uqb_qname_scan: more than %d QNAME columns", UQB_MAX_COLS);
    const uint64_t N = fq->n_reads;
    if (N == 0) return uqb_fail(ctx, "uqb_qname_scan: no records");
    UQB_TRY(uqb_fastq_free_qcols(ctx, fq));
    const uint32_t ncols = nseps + 1;
    fq->prefix_len = prefix_len; fq->suffix_len = suffix_len; fq->ncols = ncols;
    fq->qcols.resize(ncols);
    qn_params P;
    memset(&P, 0, sizeof(P));
    P.prefix_len = prefix_len; P.suffix_len = suffix_len; P.nseps = nseps;
    for (uint32_t i = 0; i < nseps; i++) { P.seps[i] = seps[i]; P.sepmask[seps[i] >> 5] |= 1u << (seps[i] & 31u); }
    for (uint32_t c = 0; c < ncols; c++) {
        UQB_TRY(uqb_dalloc_t(ctx, &fq->qcols[c].val, N));
        UQB_TRY(uqb_dalloc_t(ctx, &fq->qcols[c].span, N));
        P.val[c] = fq->qcols[c].val; P.span[c] = fq->qcols[c].span;
    }
    qn_flags hf = {LLONG_MAX, 0u, 0u};
    qn_flags* dflags;
    UQB_TRY(uqb_dalloc_t(ctx, &dflags, 1));
    UQB_CUDA(cudaMemcpyAsync(dflags, &hf, sizeof(hf), cudaMemcpyHostToDevice, ctx->stream));
    UQB_LAUNCH_B(fq->names ? N * fq->name_pitch + 12 * N * ncols : 0, k_qname_tokens, uqb_blocks(N, QN), QN, 0, fq->d, fq->line_off, N, P, dflags,
                 (const uint8_t*)fq->names, fq->name_pitch);
    col_red* dred;
    UQB_TRY(uqb_dalloc_t(ctx, &dred, ncols));
    UQB_LAUNCH(k_col_red_init, 1, UQB_MAX_COLS, 0, dred, (int)ncols);
    for (uint32_t c = 0; c < ncols; c++)
        UQB_LAUNCH(k_col_reduce, uqb_grid(ctx, N, QN * 4, 8), QN, 0, fq->qcols[c].val, fq->qcols[c].span, N, dred + c);
    UQB_TRY(uqb_readback(ctx, &hf, dflags, sizeof(hf)));
    std::vector<col_red> red(ncols);
    UQB_TRY(uqb_readback(ctx, red.data(), dred, sizeof(col_red) * ncols));
    UQB_TRY(uqb_dfree(ctx, dflags, sizeof(qn_flags)));
    UQB_TRY(uqb_dfree(ctx, dred, sizeof(col_red) * ncols));
    *bad_record = hf.bad_record == LLONG_MAX ? -1 : hf.bad_record;
    memset(cols, 0, sizeof(uqb_colstats) * ncols);
    if (*bad_record >= 0) return 0;          // the host raises the reference's error
    if (hf.has_nul) return uqb_fail(ctx, "uqb_qname_scan: NUL byte inside a QNAME");

    uint32_t ncheck = 0;
    for (uint64_t t = 10000; t <= N - 1 && ncheck < UQB_MAX_CHECKPOINTS; t *= 2) ncheck++;
    for (uint32_t c = 0; c < ncols; c++) {
        uqb_colstats& cs = cols[c];
        uqb_qcol& qc = fq->qcols[c];
        if (red[c].any_flags & FLAG_TOOLONG) return uqb_fail(ctx, "uqb_qname_scan: QNAME token longer than %u bytes", SPAN_MAXLEN);
        cs.all_int = (red[c].any_flags & FLAG_NONINT) ? 0 : 1;
        cs.all_canonical = (red[c].any_flags & FLAG_NONCANON) ? 0 : 1;
        cs.overflow = (red[c].any_flags & FLAG_OVERFLOW) ? 1 : 0;
        cs.min_val = red[c].min_val; cs.max_val = red[c].max_val;
        cs.min_len = red[c].min_len; cs.max_len = red[c].max_len;
        cs.n_checkpoints = ncheck;
        const uint32_t w = red[c].max_len;
        bool demoted_early = false;
        const uint8_t mode = col_mode ? col_mode[c] : 0;      // 0 auto, 1 no dictionary wanted, 2 dictionary forced
        if (mode == 1) {
            for (uint32_t k = 0; k < UQB_MAX_CHECKPOINTS; k++) cs.distinct_at[k] = UINT64_MAX;
            cs.n_distinct = UINT64_MAX;
            continue;
        }
        if (ncheck >= 1 && mode == 0) {
            // checkpoint 0 on its own: high-cardinality columns leave 'mapping' here (uq.py:634-636)
            uint64_t d0 = 0;
            UQB_TRY(distinct_of_prefix(ctx, fq, qc, w, 10001, &d0));
            cs.distinct_at[0] = d0;
            if (d0 > 10000 / 10) {
                demoted_early = true;
                for (uint32_t k = 1; k < UQB_MAX_CHECKPOINTS; k++) cs.distinct_at[k] = UINT64_MAX;   // not computed
                cs.n_distinct = UINT64_MAX;
            }
        }
        if (demoted_early) continue;
        // full dictionary: ranks, first occurrences, distinct counts at every checkpoint
        uint8_t* rows;
        UQB_TRY(uqb_dalloc(ctx, (void**)&rows, N * w + 64));
        if (w) UQB_LAUNCH(k_token_rows, uqb_blocks(N, QN), QN, 0, fq->d, fq->line_off, qc.span, prefix_len, w, N, rows, (const uint8_t*)fq->names, fq->name_pitch);
        uint32_t *perm, *gid;
        uint64_t u = 0;
        UQB_TRY(uqb_sort_rows_impl(ctx, rows, N, w, &perm, &gid, &u));
        uint32_t* first_row;
        UQB_TRY(uqb_dalloc_t(ctx, &qc.rank, N));
        UQB_TRY(uqb_dalloc_t(ctx, &first_row, u));
        UQB_LAUNCH(k_rank_and_first, uqb_blocks(N, QN), QN, 0, perm, gid, N, qc.rank, first_row);
        unsigned long long* dhist;
        UQB_TRY(uqb_dalloc_t(ctx, &dhist, UQB_MAX_CHECKPOINTS + 1));
        UQB_CUDA(cudaMemsetAsync(dhist, 0, 8 * (UQB_MAX_CHECKPOINTS + 1), ctx->stream));
        UQB_LAUNCH(k_first_occ_hist, uqb_grid(ctx, u, QN, 4), QN, 0, first_row, u, ncheck, dhist);
        qc.dict_count = u; qc.dict_width = w;
        UQB_TRY(uqb_dalloc(ctx, (void**)&qc.dict, u * w + 64));
        if (w) UQB_LAUNCH(k_dict_rows, uqb_grid(ctx, u * w, QN, 8), QN, 0, rows, w, first_row, u, qc.dict);
        unsigned long long hist[UQB_MAX_CHECKPOINTS + 1];
        UQB_TRY(uqb_readback(ctx, hist, dhist, sizeof(hist)));
        uint64_t run = 0;
        for (uint32_t k = 0; k < ncheck; k++) { run += hist[k]; cs.distinct_at[k] = run; }
        cs.n_distinct = u;
        UQB_TRY(uqb_dfree(ctx, dhist, 8 * (UQB_MAX_CHECKPOINTS + 1)));
        qc.first_occ = first_row;                 // first record of every dictionary entry (multi-GPU merges need it)
        UQB_TRY(uqb_dfree(ctx, perm, N * 4));
        UQB_TRY(uqb_dfree(ctx, gid, N * 4));
        UQB_TRY(uqb_dfree(ctx, rows, N * w + 64));
    }
    return 0;
}

extern "C" int uqb_qname_dict_info(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint64_t* count, uint32_t* width) {
    if (col >= fq->qcols.size()) return uqb_fail(ctx, "qname_dict: column %u out of range", col);
    if (!fq->qcols[col].rank) return uqb_fail(ctx, "qname_dict: column %u has no dictionary (it left 'mapping' at the first checkpoint)", col);
    *count = fq->qcols[col].dict_count;
    *width = fq->qcols[col].dict_width;
    return 0;
}

extern "C" int uqb_qname_dict_first(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint32_t* host, uint64_t count) {
    if (col >= fq->qcols.size() || !fq->qcols[col].rank) return uqb_fail(ctx, "qname_dict_first: column %u has no dictionary", col);
    const uqb_qcol& qc = fq->qcols[col];
    if (count != qc.dict_count) return uqb_fail(ctx, "qname_dict_first: buffer size mismatch");
    if (count) UQB_CUDA(cudaMemcpyAsync(host, qc.first_occ, count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int uqb_qname_dict(uqb_ctx* ctx, uqb_fastq* fq, uint32_t col, uint8_t* host, uint64_t nbytes) {
    if (col >= fq->qcols.size() || !fq->qcols[col].rank) return uqb_fail(ctx, "qname_dict: column %u has no dictionary", col);
    const uqb_qcol& qc = fq->qcols[col];
    if (nbytes != qc.dict_count * qc.dict_width) return uqb_fail(ctx, "qname_dict: buffer size mismatch");
    if (nbytes) UQB_CUDA(cudaMemcpyAsync(host, qc.dict, nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

template <typename T>
__global__ void __launch_bounds__(QN) k_encode_int(const int64_t* __restrict__ val, long long sub, uint64_t n, T* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * QN + threadIdx.x; i < n; i += (uint64_t)gridDim.x * QN)
        out[i] = (T)(unsigned long long)(val[i] - sub);
}
template <typename T>
__global__ void __launch_bounds__(QN) k_encode_rank(const uint32_t* __restrict__ rank, uint64_t n, T* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * QN + threadIdx.x; i < n; i += (uint64_t)gridDim.x * QN) out[i] = (T)rank[i];
}

// 'strings' column (format 2, declared extension E1): every record's token, left-aligned and zero padded to w bytes.
// A CTA takes QS_R consecutive records, whose output is ONE contiguous range of QS_R * w bytes: the token bytes are
// gathered into shared memory (all threads over the flat range, so narrow columns keep every thread busy) and the
// range leaves as aligned 16-byte stores.
#define QS_R 128
__global__ void __launch_bounds__(QN) k_encode_str(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                  const uint32_t* __restrict__ span, uint32_t prefix_len, uint32_t w, uint64_t n,
                                                  uint8_t* __restrict__ out, const uint8_t* __restrict__ names, uint32_t name_pitch) {
    __shared__ __align__(16) uint8_t stage[QS_R * 255 + 16];
    __shared__ const uint8_t* src[QS_R];
    __shared__ uint32_t len[QS_R];
    const uint64_t ntiles = (n + QS_R - 1) / QS_R;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t r0 = t * QS_R;
        const uint32_t nr = (uint32_t)(n - r0 < QS_R ? n - r0 : QS_R);
        __syncthreads();                                             // previous tile stored
        if (threadIdx.x < nr) {
            const uint64_t r = r0 + threadIdx.x;
            const uint32_t sp = __ldg(span + r);
            const uint32_t rel = (sp >> SPAN_LEN_BITS) & SPAN_MAXLEN;
            src[threadIdx.x] = (names ? names + r * name_pitch + 1 : d + __ldg(line_off + 4 * r)) + prefix_len + rel;
            len[threadIdx.x] = sp & SPAN_MAXLEN;
        }
        __syncthreads();
        const uint32_t total = nr * w;
        for (uint32_t k = threadIdx.x; k < total; k += QN) {
            const uint32_t i = k / w, b = k - i * w;
            stage[k] = b < len[i] ? __ldg(src[i] + b) : (uint8_t)0;
        }
        __syncthreads();
        uint8_t* o = out + r0 * w;                                   // QS_R * w bytes per tile: a multiple of 16
        const uint32_t nvec = (reinterpret_cast<uintptr_t>(out) & 15u) ? 0u : total >> 4;
        for (uint32_t v = threadIdx.x; v < nvec; v += QN) reinterpret_cast<uint4*>(o)[v] = reinterpret_cast<const uint4*>(stage)[v];
        for (uint32_t k = 16u * nvec + threadIdx.x; k < total; k += QN) o[k] = stage[k];
    }
}

template <typename T>
static int encode_col(uqb_ctx* ctx, const uqb_qcol& qc, const uqb_colspec& sp, uint64_t n, void* out) {
    unsigned g = uqb_grid(ctx, n, QN * 4, 8);
    if (sp.format == 0) UQB_LAUNCH(k_encode_rank<T>, g, QN, 0, qc.rank, n, (T*)out);
    else                UQB_LAUNCH(k_encode_int<T>, g, QN, 0, qc.val, (long long)(sp.offset ? sp.min_val : 0), n, (T*)out);
    return 0;
}

extern "C" int uqb_qname_encode(uqb_ctx* ctx, uqb_fastq* fq, uint32_t ncols, const uqb_colspec* spec, uqb_array** cols) {
    if (ncols != fq->qcols.size()) return uqb_fail(ctx, "qname_encode: %u columns given, scan produced %zu", ncols, fq->qcols.size());
    const uint64_t N = fq->n_reads;
    for (uint32_t c = 0; c < ncols; c++) {
        const uqb_qcol& qc = fq->qcols[c];
        if (spec[c].format == 0 && !qc.rank) return uqb_fail(ctx, "qname_encode: column %u has no dictionary ranks", c);
        if (spec[c].format > 2) return uqb_fail(ctx, "qname_encode: column %u has format %u", c, spec[c].format);
        if (spec[c].format == 2 && spec[c].itemsize == 0) return uqb_fail(ctx, "qname_encode: string column %u has width 0", c);
        UQB_TRY(uqb_new_array(ctx, N, spec[c].itemsize, &cols[c]));
        if (spec[c].format == 2) {          // token bytes, zero padded to itemsize (the host sizes it to the longest token)
            const uint32_t w = spec[c].itemsize;
            const uint64_t src_bytes = N * 4 + N * w + (fq->names ? 0 : 8 * N);
            if (N) UQB_LAUNCH_B(src_bytes + N * w, k_encode_str, uqb_grid(ctx, N, QS_R, 16), QN, 0, fq->d, fq->line_off, qc.span,
                                fq->prefix_len, w, N, (uint8_t*)cols[c]->d, (const uint8_t*)fq->names, fq->name_pitch);
            continue;
        }
        switch (spec[c].itemsize) {
            case 1: UQB_TRY(encode_col<uint8_t>(ctx, qc, spec[c], N, cols[c]->d)); break;
            case 2: UQB_TRY(encode_col<uint16_t>(ctx, qc, spec[c], N, cols[c]->d)); break;
            case 4: UQB_TRY(encode_col<uint32_t>(ctx, qc, spec[c], N, cols[c]->d)); break;
            case 8: UQB_TRY(encode_col<uint64_t>(ctx, qc, spec[c], N, cols[c]->d)); break;
            default: return uqb_fail(ctx, "qname_encode: itemsize %u", spec[c].itemsize);
        }
    }
    return 0;
}
