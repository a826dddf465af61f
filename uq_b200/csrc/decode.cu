// Stage 5: uQ tables -> FASTQ text (replaces split_bits uq.py:1002-1007, convert_qname
// uq.py:1010-1026 and the emit loop uq.py:1030-1058).
//
// Two phases: (1) one thread per record computes the byte length of its four lines (QNAME text
// length from the column values, read length from the marker bit for variable-length files);
// an exclusive scan turns lengths into output offsets; (2) one warp per record writes the text:
// lane 0 formats the QNAME, all lanes unpack DNA / QUAL symbols.
#include "common.cuh"

#define DC 256

struct dec_col {
    const uint8_t* data;       // column values [n][itemsize], little endian
    const uint8_t* dict;       // mapping strings, zero padded rows (device)
    const uint32_t* dict_len;  // strlen of every dictionary row (device)
    uint64_t dict_count;
    uint32_t dict_width;
    uint32_t itemsize;
    uint32_t format, offset;
    long long min_val;
};

struct dec_params {
    uint8_t base_char[256];
    uint8_t qual_char[256];
    int16_t qual_to_base[256];
    uint32_t bb, bq, variable, dna_max, wd, wq;
    uint32_t prefix_len, suffix_len, nseps, ncols;
    uint8_t prefix[UQB_HDR_MAX];
    uint8_t suffix[UQB_HDR_MAX];
    uint8_t seps[UQB_MAX_COLS];
    dec_col cols[UQB_MAX_COLS];
};

__device__ __forceinline__ unsigned long long load_le(const uint8_t* p, uint32_t size) {
    unsigned long long v = 0;
    for (uint32_t i = 0; i < size; i++) v |= (unsigned long long)p[i] << (8 * i);
    return v;
}

// 'strings' column (format 2, E1): the token is the value's bytes up to the first NUL
__device__ __forceinline__ uint32_t str_len(const uint8_t* p, uint32_t w) {
    uint32_t n = 0;
    while (n < w && p[n]) n++;
    return n;
}

__device__ __forceinline__ uint32_t dec_digits(long long v) {
    uint32_t n = v < 0 ? 1u : 0u;
    unsigned long long a = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
    if (a < (1ull << 32)) {                     // the usual case: no 64-bit divisions
        const uint32_t x = (uint32_t)a;
        return n + 1u + (x >= 10u) + (x >= 100u) + (x >= 1000u) + (x >= 10000u) + (x >= 100000u) + (x >= 1000000u) +
               (x >= 10000000u) + (x >= 100000000u) + (x >= 1000000000u);
    }
    do { n++; a /= 10ull; } while (a);
    return n;
}

// decimal digits of a (nd of them) -> w[0 .. nd)
__device__ __forceinline__ void dec_write(uint8_t* w, unsigned long long a, uint32_t nd) {
    uint32_t i = nd;
    while (a >= (1ull << 32)) { w[--i] = (uint8_t)('0' + a % 10ull); a /= 10ull; }
    uint32_t x = (uint32_t)a;
    while (i) { w[--i] = (uint8_t)('0' + x % 10u); x /= 10u; }
}

// read length of a variable-length row: the first set bit is the marker's (SURVEY A.2).  A row of a malformed
// container may carry bits in front of the widest legal marker position: the length is clamped to dna_max (so that
// no symbol index can leave the row) and *bad is set; uqb_decode then fails instead of emitting garbage.
__device__ __forceinline__ uint32_t row_read_len(const uint8_t* row, uint32_t w, uint32_t bits, uint32_t dna_max, uint32_t variable, bool* bad) {
    if (!variable) return dna_max;
    for (uint32_t j = 0; j < w; j++) {
        unsigned b = row[j];
        if (b) {
            uint32_t p = 8 * j + (__clz(b) - 24);
            uint32_t len = (8 * w - 1 - p) / bits;
            if (len > dna_max) { *bad = true; len = dna_max; }
            return len;
        }
    }
    *bad = true;                 // no marker at all
    return 0;
}

template <bool STR>
__device__ __forceinline__ uint32_t qname_text_len(const dec_params& P, uint64_t r) {
    uint32_t n = P.prefix_len + P.suffix_len;
    for (uint32_t c = 0; c < P.ncols; c++) {
        const dec_col& dc = P.cols[c];
        const uint8_t* p = dc.data + r * dc.itemsize;
        if (STR && dc.format == 2) { n += str_len(p, dc.itemsize); if (c < P.nseps) n += 1; continue; }
        unsigned long long raw = load_le(p, dc.itemsize);
        if (dc.format == 0) n += raw < dc.dict_count ? dc.dict_len[raw] : 0u;
        else n += dec_digits((long long)raw + (dc.offset ? dc.min_val : 0ll));
        if (c < P.nseps) n += 1;
    }
    return n;
}

template <bool STR>
__device__ __forceinline__ void decode_len_body(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna, uint64_t n,
                                                  uint32_t* __restrict__ rec_len, unsigned long long* __restrict__ bad_row) {
    const uint64_t r = (uint64_t)blockIdx.x * DC + threadIdx.x;
    if (r >= n) return;
    const dec_params& P = *Pp;
    bool bad = false;
    const uint32_t len = row_read_len(dna + r * P.wd, P.wd, P.bb, P.dna_max, P.variable, &bad);
    if (bad) atomicMin(bad_row, (unsigned long long)r);
    rec_len[r] = qname_text_len<STR>(P, r) + 1 + len + 1 + 2 + len + 1;
}

__device__ __forceinline__ unsigned row_symbol(const uint8_t* row, uint32_t w, uint32_t bits, uint32_t pos) {
    const uint32_t j = pos >> 3;
    unsigned v = (unsigned)row[j] << 8;
    if (j + 1 < w) v |= row[j + 1];
    return (v >> (16 - (pos & 7u) - bits)) & ((1u << bits) - 1u);
}

template <bool STR>
__device__ __forceinline__ void decode_write_body(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                    const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                    uint8_t* __restrict__ out) {
    __shared__ uint8_t base_char[256], qual_char[256];
    __shared__ int16_t qual_to_base[256];
    const dec_params& P = *Pp;
    for (unsigned i = threadIdx.x; i < 256; i += DC) { base_char[i] = P.base_char[i]; qual_char[i] = P.qual_char[i]; qual_to_base[i] = P.qual_to_base[i]; }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    const uint64_t wstride = (uint64_t)gridDim.x * (DC / 32);
    const uint32_t nsym_row = P.dna_max + P.variable;
    const uint32_t pad_d = 8 * P.wd - P.bb * nsym_row, pad_q = 8 * P.wq - P.bq * nsym_row;
    for (uint64_t r = (uint64_t)blockIdx.x * (DC / 32) + (threadIdx.x >> 5); r < n; r += wstride) {
        const uint8_t* drow = dna + r * P.wd;
        const uint8_t* qrow = qual + r * P.wq;
        uint8_t* o = out + rec_off[r];
        // ---- QNAME: prefix + sum(column text + separator) + suffix (uq.py:1010-1024) ----
        // lane c formats column c: text length -> warp prefix sum over the columns -> every lane writes
        // its own column text (and the separator behind it) straight to its place in the output line
        uint32_t run = P.prefix_len;                // offset of the next column's text within the line
        for (uint32_t c0 = 0; c0 < P.ncols; c0 += 32) {
            const uint32_t c = c0 + lane;
            uint32_t tl = 0;
            unsigned long long raw = 0;
            long long v = 0;
            if (c < P.ncols) {
                const dec_col& dc = P.cols[c];
                if (STR && dc.format == 2) {
                    tl = str_len(dc.data + r * dc.itemsize, dc.itemsize);
                } else if (dc.format == 0) {
                    raw = load_le(dc.data + r * dc.itemsize, dc.itemsize);
                    tl = raw < dc.dict_count ? dc.dict_len[raw] : 0u;
                } else {
                    raw = load_le(dc.data + r * dc.itemsize, dc.itemsize);
                    v = (long long)raw + (dc.offset ? dc.min_val : 0ll);
                    tl = dec_digits(v);
                }
                if (c < P.nseps) tl += 1;           // the separator that follows this column
            }
            uint32_t incl = tl;
#pragma unroll
            for (int sh = 1; sh < 32; sh <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, sh);
                if (lane >= (unsigned)sh) incl += t;
            }
            if (c < P.ncols) {
                const dec_col& dc = P.cols[c];
                uint8_t* w = o + run + incl - tl;
                uint32_t body = tl - (c < P.nseps ? 1u : 0u);
                if (STR && dc.format == 2) {
                    const uint8_t* sp = dc.data + r * dc.itemsize;
                    for (uint32_t i = 0; i < body; i++) w[i] = sp[i];
                } else if (dc.format == 0) {
                    if (raw < dc.dict_count) {
                        const uint8_t* sp = dc.dict + raw * dc.dict_width;
                        for (uint32_t i = 0; i < body; i++) w[i] = sp[i];
                    }
                } else {
                    unsigned long long a = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
                    if (v < 0) w[0] = '-';
                    dec_write(w + (v < 0 ? 1u : 0u), a, body - (v < 0 ? 1u : 0u));
                }
                if (c < P.nseps) w[body] = P.seps[c];
            }
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        for (uint32_t i = lane; i < P.prefix_len; i += 32) o[i] = P.prefix[i];
        for (uint32_t i = lane; i < P.suffix_len; i += 32) o[run + i] = P.suffix[i];
        if (lane == 0) o[run + P.suffix_len] = '\n';
        const uint32_t hl = run + P.suffix_len + 1;
        uint32_t len = 0;
        bool bad_unused = false;
        if (lane == 0) len = row_read_len(drow, P.wd, P.bb, P.dna_max, P.variable, &bad_unused);
        len = __shfl_sync(0xffffffffu, len, 0);
        uint8_t* od = o + hl;                  // DNA line
        uint8_t* oq = od + len + 3;            // after "\n+\n"
        const uint32_t s_first = nsym_row - len;     // skips the padding symbols and the marker
        for (uint32_t i = lane; i < len; i += 32) {
            const uint32_t s = s_first + i;
            const unsigned dcode = row_symbol(drow, P.wd, P.bb, pad_d + P.bb * s);
            const unsigned qcode = row_symbol(qrow, P.wq, P.bq, pad_q + P.bq * s);
            const int restored = qual_to_base[qcode];          // qual_N (uq.py:1036)
            od[i] = restored >= 0 ? (uint8_t)restored : base_char[dcode];
            oq[i] = qual_char[qcode];
        }
        if (lane == 0) { od[len] = '\n'; od[len + 1] = '+'; od[len + 2] = '\n'; oq[len] = '\n'; }
    }
}

// ---- tiled decode of fixed-length reads -----------------------------------------------------------
// A CTA takes DT_R consecutive records.  Their packed rows are two contiguous byte ranges (coalesced 16-byte
// loads into shared memory, stored as big-endian words) and their text is ONE contiguous range of the output,
// which is assembled in shared memory and leaves as aligned 16-byte stores.  Work items are chunks of 16
// positions (record index fastest, so that the byte stores of a warp fall into different banks): the codes of
// a chunk are cut out of the bit string with compile-time shifts (the mirror image of pack.cu's
// place_chunk16), mapped through the LUTs and written to the DNA and QUAL lines; one thread per record
// formats the QNAME.
#define DT_R 64
#define DT_THREADS 256
#define DT_TEXT_CAP (28 * 1024)
#define DT_IN_CAP (24 * 1024)
#define DT_FIX_CAP 512

template <int BITS>
__device__ __forceinline__ void extract_chunk16(const uint32_t* __restrict__ words, uint32_t gbit, uint32_t (&code)[16]) {
    constexpr int NW = (16 * BITS + 31) / 32;
    const uint32_t sh = gbit & 31u, w0 = gbit >> 5;
    uint32_t x[NW + 1], w[NW];
#pragma unroll
    for (int k = 0; k <= NW; k++) x[k] = words[w0 + k];
#pragma unroll
    for (int k = 0; k < NW; k++) w[k] = __funnelshift_l(x[k + 1], x[k], sh);      // bits gbit + 32k .. of the big-endian string
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int off = k * BITS, wi = off >> 5, o = off & 31;
        uint32_t v;
        if (o + BITS <= 32) v = w[wi] >> (32 - o - BITS);
        else v = (w[wi] << (o + BITS - 32)) | (w[wi + 1 < NW ? wi + 1 : wi] >> (64 - o - BITS));
        code[k] = v & ((1u << BITS) - 1u);
    }
}

__device__ __forceinline__ void extract_chunk16_any(uint32_t bits, const uint32_t* words, uint32_t gbit, uint32_t (&code)[16]) {
    switch (bits) {          // warp-uniform
        case 1: extract_chunk16<1>(words, gbit, code); break;
        case 2: extract_chunk16<2>(words, gbit, code); break;
        case 3: extract_chunk16<3>(words, gbit, code); break;
        case 4: extract_chunk16<4>(words, gbit, code); break;
        case 5: extract_chunk16<5>(words, gbit, code); break;
        case 6: extract_chunk16<6>(words, gbit, code); break;
        case 7: extract_chunk16<7>(words, gbit, code); break;
        default: extract_chunk16<8>(words, gbit, code); break;
    }
}

// QNAME text of record r -> w (prefix, columns with separators, suffix, newline); returns its length
template <bool STR>
__device__ __forceinline__ uint32_t qname_write(const dec_params& P, uint64_t r, uint8_t* w) {
    uint32_t n = 0;
    for (uint32_t i = 0; i < P.prefix_len; i++) w[n++] = P.prefix[i];
    for (uint32_t c = 0; c < P.ncols; c++) {
        const dec_col& dc = P.cols[c];
        if (STR && dc.format == 2) {
            const uint8_t* sp = dc.data + r * dc.itemsize;
            for (uint32_t i = 0; i < dc.itemsize && sp[i]; i++) w[n++] = sp[i];
            if (c < P.nseps) w[n++] = P.seps[c];
            continue;
        }
        const unsigned long long raw = load_le(dc.data + r * dc.itemsize, dc.itemsize);
        if (dc.format == 0) {
            if (raw < dc.dict_count) {
                const uint32_t tl = dc.dict_len[raw];
                const uint8_t* sp = dc.dict + raw * dc.dict_width;
                for (uint32_t i = 0; i < tl; i++) w[n++] = sp[i];
            }
        } else {
            const long long v = (long long)raw + (dc.offset ? dc.min_val : 0ll);
            unsigned long long a = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
            const uint32_t nd = dec_digits(v);
            if (v < 0) w[n] = '-';
            dec_write(w + n + (v < 0 ? 1u : 0u), a, nd - (v < 0 ? 1u : 0u));
            n += nd;
        }
        if (c < P.nseps) w[n++] = P.seps[c];
    }
    for (uint32_t i = 0; i < P.suffix_len; i++) w[n++] = P.suffix[i];
    w[n++] = '\n';
    return n;
}

// One QNAME column of record r -> text at w + (offset of that column inside the line): every (record, column) pair is a
// work item of its own, so the QNAME lines of a tile are formatted by all threads instead of one thread per record.
// The item recomputes the text lengths of the columns in front of it (a few compares each) to find its place.
template <bool STR>
__device__ __forceinline__ uint32_t col_text_len(const dec_col& dc, uint64_t r, unsigned long long* raw_out, long long* v_out) {
    if (STR && dc.format == 2) { *raw_out = 0; *v_out = 0; return str_len(dc.data + r * dc.itemsize, dc.itemsize); }
    const unsigned long long raw = load_le(dc.data + r * dc.itemsize, dc.itemsize);
    *raw_out = raw;
    if (dc.format == 0) { *v_out = 0; return raw < dc.dict_count ? dc.dict_len[raw] : 0u; }
    const long long v = (long long)raw + (dc.offset ? dc.min_val : 0ll);
    *v_out = v;
    return dec_digits(v);
}

template <bool STR>
__device__ __forceinline__ void qname_write_col(const dec_params& P, uint64_t r, uint32_t c, uint8_t* w) {
    uint32_t at = P.prefix_len;
    unsigned long long raw = 0;
    long long v = 0;
    for (uint32_t k = 0; k < c; k++) at += col_text_len<STR>(P.cols[k], r, &raw, &v) + 1u;      // + separator (k < nseps since k < c <= ncols - 1)
    const dec_col& dc = P.cols[c];
    const uint32_t tl = col_text_len<STR>(dc, r, &raw, &v);
    uint8_t* o = w + at;
    if (STR && dc.format == 2) {
        const uint8_t* sp = dc.data + r * dc.itemsize;
        for (uint32_t i = 0; i < tl; i++) o[i] = sp[i];
    } else if (dc.format == 0) {
        if (raw < dc.dict_count) {
            const uint8_t* sp = dc.dict + raw * dc.dict_width;
            for (uint32_t i = 0; i < tl; i++) o[i] = sp[i];
        }
    } else {
        const unsigned long long a = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
        if (v < 0) o[0] = '-';
        dec_write(o + (v < 0 ? 1u : 0u), a, tl - (v < 0 ? 1u : 0u));
    }
    if (c < P.nseps) o[tl] = P.seps[c];
    if (c == 0) for (uint32_t i = 0; i < P.prefix_len; i++) w[i] = P.prefix[i];
    if (c + 1 == P.ncols) {
        uint8_t* e = o + tl + (c < P.nseps ? 1u : 0u);
        for (uint32_t i = 0; i < P.suffix_len; i++) e[i] = P.suffix[i];
        e[P.suffix_len] = '\n';
    }
}

struct dt_smem {
    alignas(16) uint8_t text[DT_TEXT_CAP + 32];
    alignas(16) uint32_t in_d[DT_IN_CAP / 4 + 8];
    uint8_t base_char[256];
    uint16_t qual_lut[256];             // quality character | (restored base + 1) << 8
    uint32_t toff[DT_R + 1];            // text offset of every record relative to the staged range
    uint16_t sel_lut[256];              // four 2-bit codes (one byte of the DNA bit string) -> PRMT selector of their four characters
    uint32_t fix_n;                     // N restorations of this tile: (text offset << 8) | base character
    uint32_t fix[DT_FIX_CAP];
};

template <bool STR>
__device__ __forceinline__ void decode_tiles_body(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                            const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                            uint64_t total, uint8_t* __restrict__ out, unsigned int* __restrict__ fallback) {
    extern __shared__ __align__(16) uint8_t dt_raw[];
    dt_smem* S = reinterpret_cast<dt_smem*>(dt_raw);
    const dec_params& P = *Pp;
    const unsigned tid = threadIdx.x;
    for (unsigned i = tid; i < 256; i += DT_THREADS) {
        S->base_char[i] = P.base_char[i];
        const int rb = P.qual_to_base[i];
        S->qual_lut[i] = (uint16_t)(P.qual_char[i] | ((rb >= 0 ? (unsigned)rb + 1u : 0u) << 8));
        S->sel_lut[i] = (uint16_t)(((i >> 6) & 3u) | (((i >> 4) & 3u) << 4) | (((i >> 2) & 3u) << 8) | ((i & 3u) << 12));
    }
    // Two bits per base (the usual case): the characters of four positions are ONE byte permute of the 4-entry alphabet held
    // in a register, selected by a byte of the bit string, and leave as aligned 32-bit words.  The DNA lines are then written
    // by work items of their own (16 positions that start at a 4-byte aligned text address); the bases that a quality code
    // restores (N with its own quality, uq.py:1036) are rare and patched in afterwards from a per-tile list.
    const bool fast_dna = P.bb == 2u;
    const uint32_t tbl = (uint32_t)P.base_char[0] | ((uint32_t)P.base_char[1] << 8) | ((uint32_t)P.base_char[2] << 16) | ((uint32_t)P.base_char[3] << 24);
    const uint32_t L = P.dna_max, wd = P.wd, wq = P.wq;
    const uint32_t pad_d = 8 * wd - P.bb * L, pad_q = 8 * wq - P.bq * L;
    const uint32_t words_d = (DT_R * wd + 3) / 4 + 4;                     // QUAL words start behind the DNA words
    uint32_t* in_q = S->in_d + ((words_d + 3) & ~3u);
    const uint32_t chunks = (L + 15) / 16;
    const uint64_t ntiles = (n + DT_R - 1) / DT_R;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t r0 = t * DT_R, r1 = (r0 + DT_R < n) ? r0 + DT_R : n;
        const uint32_t nrec = (uint32_t)(r1 - r0);
        const uint64_t o0 = rec_off[r0], o1 = r1 < n ? rec_off[r1] : total;
        const uint64_t a0 = o0 & ~15ull;
        if (tid == 0) { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); S->fix_n = 0; }   // the bulk store of the previous tile has read its text
        __syncthreads();                                                   // previous tile fully stored
        if (o1 - a0 > DT_TEXT_CAP) { if (tid == 0) atomicOr(fallback, 1u); continue; }
        // ---- packed rows -> shared memory (big-endian words) ----
        {
            const uint4* gd = reinterpret_cast<const uint4*>(dna + r0 * wd);      // r0 * width is a multiple of 64
            const uint4* gq = reinterpret_cast<const uint4*>(qual + r0 * wq);
            const uint32_t vd = (nrec * wd + 15) / 16, vq = (nrec * wq + 15) / 16;   // tables carry 64 bytes of slack
            for (uint32_t v = tid; v < vd; v += DT_THREADS) {
                const uint4 x = __ldg(gd + v);
                uint32_t* dst = S->in_d + 4 * v;
                dst[0] = __byte_perm(x.x, 0, 0x0123); dst[1] = __byte_perm(x.y, 0, 0x0123); dst[2] = __byte_perm(x.z, 0, 0x0123); dst[3] = __byte_perm(x.w, 0, 0x0123);
            }
            for (uint32_t v = tid; v < vq; v += DT_THREADS) {
                const uint4 x = __ldg(gq + v);
                uint32_t* dst = in_q + 4 * v;
                dst[0] = __byte_perm(x.x, 0, 0x0123); dst[1] = __byte_perm(x.y, 0, 0x0123); dst[2] = __byte_perm(x.z, 0, 0x0123); dst[3] = __byte_perm(x.w, 0, 0x0123);
            }
            for (uint32_t i = tid; i <= nrec; i += DT_THREADS) S->toff[i] = (uint32_t)((i < nrec ? rec_off[r0 + i] : o1) - a0);
        }
        __syncthreads();
        // ---- work items: chunks of 16 positions (record index fastest), then one QNAME line per item ----
        const uint32_t nsymitems = nrec * chunks;
        const uint32_t ncol = P.ncols ? P.ncols : 1u;
        const uint32_t cmax = L / 16;                                       // full DNA chunks a line can hold
        const uint32_t ndnaitems = fast_dna ? nrec * (cmax + 1u) : 0u;      // + one item per record for the unaligned head and the tail
        for (uint32_t item = tid; item < nsymitems + ndnaitems + nrec * ncol; item += DT_THREADS) {
            if (item >= nsymitems && item < nsymitems + ndnaitems) {
                const uint32_t di = item - nsymitems, c = di / nrec, i = di - c * nrec;
                const uint32_t hl = S->toff[i + 1] - S->toff[i] - 2u * L - 4u;
                const uint32_t line = S->toff[i] + hl;                      // text offset of the DNA line
                uint32_t h = (4u - (line & 3u)) & 3u;                       // positions in front of the first aligned word
                if (h > L) h = L;
                const uint32_t nfull = (L - h) / 16;
                const uint32_t bit0 = (i * wd) * 8u + pad_d;
                if (c < cmax) {
                    if (c < nfull) {
                        const uint32_t p = h + 16u * c, g = bit0 + 2u * p;
                        const uint32_t x = __funnelshift_l(S->in_d[(g >> 5) + 1], S->in_d[g >> 5], g & 31u);   // 16 codes, first one on top
                        uint32_t* o = reinterpret_cast<uint32_t*>(S->text + line + p);
#pragma unroll
                        for (int m = 0; m < 4; m++) o[m] = __byte_perm(tbl, 0u, S->sel_lut[(x >> (24 - 8 * m)) & 255u]);
                    }
                } else {
                    for (uint32_t p = 0; p < L; p++) {
                        if (p == h) { p += 16u * nfull; if (p >= L) break; }
                        const uint32_t g = bit0 + 2u * p;
                        const uint32_t code = (S->in_d[g >> 5] >> (30u - (g & 31u))) & 3u;
                        S->text[line + p] = (uint8_t)(tbl >> (8u * code));
                    }
                }
                continue;
            }
            if (item >= nsymitems) {
                const uint32_t qi = item - nsymitems - ndnaitems, c = qi / nrec, i = qi - c * nrec;       // record index fastest
                uint8_t* w = S->text + S->toff[i];
                if (P.ncols == 0) {
                    qname_write<STR>(P, r0 + i, w);
                } else {
                    qname_write_col<STR>(P, r0 + i, c, w);
                }
                if (c == 0) {
                    const uint32_t hl = S->toff[i + 1] - S->toff[i] - 2u * L - 4u;             // record length - (2 L + 4) = QNAME line length
                    w[hl + L] = '\n'; w[hl + L + 1] = '+'; w[hl + L + 2] = '\n'; w[hl + 2 * L + 3] = '\n';
                }
                continue;
            }
            const uint32_t c = item / nrec, i = item - c * nrec;
            const uint32_t p0 = c * 16, nsym = (p0 + 16 <= L) ? 16u : L - p0;
            uint32_t cd[16], cq[16];
            extract_chunk16_any(P.bq, in_q, (i * wq) * 8u + pad_q + p0 * P.bq, cq);
            const uint32_t hl = S->toff[i + 1] - S->toff[i] - 2u * L - 4u;      // record length - (2 L + 4) = QNAME line length
            const uint32_t od_off = S->toff[i] + hl + p0;
            uint8_t* od = S->text + od_off;
            uint8_t* oq = od + L + 3;
            if (fast_dna) {
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    if ((uint32_t)k < nsym) {
                        const uint32_t ql = S->qual_lut[cq[k]];
                        oq[k] = (uint8_t)ql;
                        if (ql >> 8) {                                          // qual_N (uq.py:1036): patched in after the DNA items
                            const uint32_t slot = atomicAdd(&S->fix_n, 1u);
                            if (slot < DT_FIX_CAP) S->fix[slot] = ((od_off + (uint32_t)k) << 8) | ((ql >> 8) - 1u);
                        }
                    }
                }
                continue;
            }
            extract_chunk16_any(P.bb, S->in_d, (i * wd) * 8u + pad_d + p0 * P.bb, cd);
#pragma unroll
            for (int k = 0; k < 16; k++) {
                if ((uint32_t)k < nsym) {
                    const uint32_t ql = S->qual_lut[cq[k]];
                    od[k] = (ql >> 8) ? (uint8_t)((ql >> 8) - 1u) : S->base_char[cd[k]];       // qual_N (uq.py:1036)
                    oq[k] = (uint8_t)ql;
                }
            }
        }
        __syncthreads();
        if (fast_dna && S->fix_n) {                                         // uniform: written before the barrier
            const uint32_t nf = S->fix_n;
            if (nf <= DT_FIX_CAP) {
                for (uint32_t j = tid; j < nf; j += DT_THREADS) { const uint32_t e = S->fix[j]; S->text[e >> 8] = (uint8_t)e; }
            } else {
                // more restorations than the list holds (reads full of N): walk the quality codes again
                for (uint32_t item = tid; item < nsymitems; item += DT_THREADS) {
                    const uint32_t c = item / nrec, i = item - c * nrec;
                    const uint32_t p0 = c * 16, nsym = (p0 + 16 <= L) ? 16u : L - p0;
                    uint32_t cq[16];
                    extract_chunk16_any(P.bq, in_q, (i * wq) * 8u + pad_q + p0 * P.bq, cq);
                    const uint32_t hl = S->toff[i + 1] - S->toff[i] - 2u * L - 4u;
                    uint8_t* od = S->text + S->toff[i] + hl + p0;
#pragma unroll
                    for (int k = 0; k < 16; k++) {
                        if ((uint32_t)k < nsym) {
                            const uint32_t ql = S->qual_lut[cq[k]];
                            if (ql >> 8) od[k] = (uint8_t)((ql >> 8) - 1u);
                        }
                    }
                }
            }
            __syncthreads();
        }
        // ---- text out: aligned 16-byte units inside [o0, o1), bytes at the two edges ----
        {
            const uint32_t lo = (uint32_t)(o0 - a0), hi = (uint32_t)(o1 - a0);
            const uint32_t v0 = (lo + 15) / 16, v1 = hi / 16;
            // the aligned interior of the tile's text leaves as ONE TMA bulk store (shared -> global); the next tile
            // waits for its read side (wait_group.read) before it touches the text buffer again
            if (tid == 0 && v1 > v0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out + a0 + 16ull * v0),
                             "r"((uint32_t)__cvta_generic_to_shared(S->text + 16u * v0)), "r"(16u * (v1 - v0))
                             : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            if (v0 <= v1) {
                for (uint32_t b = lo + tid; b < v0 * 16 && b < hi; b += DT_THREADS) out[a0 + b] = S->text[b];
                for (uint32_t b = v1 * 16 + tid; b < hi; b += DT_THREADS) if (b >= lo) out[a0 + b] = S->text[b];
            } else {
                for (uint32_t b = lo + tid; b < hi; b += DT_THREADS) out[a0 + b] = S->text[b];
            }
        }
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // the last bulk store has landed
}

// The decode kernels: the plain ones for containers without 'strings' QNAME columns (exactly the kernels those always
// ran), the _str ones when a column holds strings (E1).
__global__ void __launch_bounds__(DC) k_decode_len(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna, uint64_t n,
                                                  uint32_t* __restrict__ rec_len, unsigned long long* __restrict__ bad_row) { decode_len_body<false>(Pp, dna, n, rec_len, bad_row); }
__global__ void __launch_bounds__(DC) k_decode_len_str(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna, uint64_t n,
                                                  uint32_t* __restrict__ rec_len, unsigned long long* __restrict__ bad_row) { decode_len_body<true>(Pp, dna, n, rec_len, bad_row); }
__global__ void __launch_bounds__(DC) k_decode_write(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                    const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                    uint8_t* __restrict__ out) { decode_write_body<false>(Pp, dna, qual, n, rec_off, out); }
__global__ void __launch_bounds__(DC) k_decode_write_str(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                    const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                    uint8_t* __restrict__ out) { decode_write_body<true>(Pp, dna, qual, n, rec_off, out); }
__global__ void __launch_bounds__(DT_THREADS) k_decode_tiles(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                            const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                            uint64_t total, uint8_t* __restrict__ out, unsigned int* __restrict__ fallback) { decode_tiles_body<false>(Pp, dna, qual, n, rec_off, total, out, fallback); }
__global__ void __launch_bounds__(DT_THREADS) k_decode_tiles_str(const dec_params* __restrict__ Pp, const uint8_t* __restrict__ dna,
                                                            const uint8_t* __restrict__ qual, uint64_t n, const uint64_t* __restrict__ rec_off,
                                                            uint64_t total, uint8_t* __restrict__ out, unsigned int* __restrict__ fallback) { decode_tiles_body<true>(Pp, dna, qual, n, rec_off, total, out, fallback); }

extern "C" int uqb_decode(uqb_ctx* ctx, const uqb_array* dna, const uqb_array* qual, uqb_array* const* cols,
                          const uqb_decode_params* p, uqb_array** fastq) {
    const uint64_t n = dna->n;
    if (qual->n != n) return uqb_fail(ctx, "decode: DNA has %llu rows, QUAL %llu", (unsigned long long)n, (unsigned long long)qual->n);
    if (p->ncols > UQB_MAX_COLS || p->nseps > UQB_MAX_COLS) return uqb_fail(ctx, "decode: too many QNAME columns");
    if (p->prefix_len > UQB_HDR_MAX || p->suffix_len > UQB_HDR_MAX) return uqb_fail(ctx, "decode: prefix/suffix too long");
    if (p->bits_per_base < 1 || p->bits_per_base > 8 || p->bits_per_quality < 1 || p->bits_per_quality > 8) return uqb_fail(ctx, "decode: bad bit widths");
    const uint64_t nsym = (uint64_t)p->dna_max + p->variable;
    if ((uint64_t)dna->width * 8 < nsym * p->bits_per_base || (uint64_t)qual->width * 8 < nsym * p->bits_per_quality)
        return uqb_fail(ctx, "decode: rows too narrow for dna_max");
    dec_params* hp = new dec_params();
    memset(hp, 0, sizeof(*hp));
    memcpy(hp->base_char, p->base_char, 256);
    memcpy(hp->qual_char, p->qual_char, 256);
    memcpy(hp->qual_to_base, p->qual_to_base, 512);
    hp->bb = p->bits_per_base; hp->bq = p->bits_per_quality; hp->variable = p->variable; hp->dna_max = p->dna_max;
    hp->wd = dna->width; hp->wq = qual->width;
    hp->prefix_len = p->prefix_len; hp->suffix_len = p->suffix_len; hp->nseps = p->nseps; hp->ncols = p->ncols;
    if (p->prefix_len) memcpy(hp->prefix, p->prefix, p->prefix_len);
    if (p->suffix_len) memcpy(hp->suffix, p->suffix, p->suffix_len);
    if (p->nseps) memcpy(hp->seps, p->seps, p->nseps);
    std::vector<void*> temps;
    std::vector<size_t> temp_sizes;
    int rc = 0;
    for (uint32_t c = 0; c < p->ncols && rc == 0; c++) {
        const uqb_decode_col& sc = p->cols[c];
        dec_col& dc = hp->cols[c];
        if (cols[c]->n != n || cols[c]->width != sc.itemsize) { rc = uqb_fail(ctx, "decode: column %u shape mismatch", c); break; }
        if (sc.format > 2 || (sc.format == 2 && sc.itemsize == 0)) { rc = uqb_fail(ctx, "decode: column %u has format %u, width %u", c, sc.format, sc.itemsize); break; }
        dc.data = (const uint8_t*)cols[c]->d;
        dc.itemsize = sc.itemsize; dc.format = sc.format; dc.offset = sc.offset; dc.min_val = sc.min_val;
        dc.dict_count = sc.dict_count; dc.dict_width = sc.dict_width;
        if (sc.format == 0) {
            const size_t nb = (size_t)sc.dict_count * sc.dict_width;
            std::vector<uint32_t> lens(sc.dict_count ? sc.dict_count : 1);
            for (uint64_t k = 0; k < sc.dict_count; k++) {
                uint32_t l = 0;
                while (l < sc.dict_width && sc.dict[k * sc.dict_width + l]) l++;
                lens[k] = l;
            }
            void *dd, *dl;
            if ((rc = uqb_dalloc(ctx, &dd, nb + 16))) break;
            temps.push_back(dd); temp_sizes.push_back(nb + 16);
            if ((rc = uqb_dalloc(ctx, &dl, lens.size() * 4))) break;
            temps.push_back(dl); temp_sizes.push_back(lens.size() * 4);
            if (nb) cudaMemcpyAsync(dd, sc.dict, nb, cudaMemcpyHostToDevice, ctx->stream);
            cudaMemcpyAsync(dl, lens.data(), lens.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
            cudaStreamSynchronize(ctx->stream);
            dc.dict = (const uint8_t*)dd; dc.dict_len = (const uint32_t*)dl;
        }
    }
    dec_params* dp = nullptr;
    uint32_t* rec_len = nullptr;
    uint64_t* rec_off = nullptr;
    uint64_t* d_total = nullptr;
    uint64_t total = 0;
    if (rc == 0) rc = uqb_dalloc_t(ctx, &dp, 1);
    if (rc == 0) {
        cudaMemcpyAsync(dp, hp, sizeof(dec_params), cudaMemcpyHostToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    }
    delete hp;
    if (rc) return rc;
    UQB_TRY(uqb_dalloc_t(ctx, &rec_len, n));
    UQB_TRY(uqb_dalloc_t(ctx, &rec_off, n));
    UQB_TRY(uqb_dalloc_t(ctx, &d_total, 1));
    unsigned long long* d_bad;
    UQB_TRY(uqb_dalloc_t(ctx, &d_bad, 1));
    UQB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 8, ctx->stream));
    bool has_str = false;
    for (uint32_t c = 0; c < p->ncols; c++) has_str |= p->cols[c].format == 2;
    if (n && has_str) UQB_LAUNCH(k_decode_len_str, uqb_blocks(n, DC), DC, 0, dp, (const uint8_t*)dna->d, n, rec_len, d_bad);
    else if (n) UQB_LAUNCH(k_decode_len, uqb_blocks(n, DC), DC, 0, dp, (const uint8_t*)dna->d, n, rec_len, d_bad);
    UQB_TRY(uqb_scan_u32_to_u64(ctx, rec_len, rec_off, n, d_total));
    UQB_TRY(uqb_readback(ctx, &total, d_total, 8));
    unsigned long long bad_row = ~0ull;
    UQB_TRY(uqb_readback(ctx, &bad_row, d_bad, 8));
    UQB_TRY(uqb_dfree(ctx, d_bad, 8));
    if (bad_row != ~0ull) {
        UQB_TRY(uqb_dfree(ctx, rec_len, n * 4));
        UQB_TRY(uqb_dfree(ctx, rec_off, n * 8));
        UQB_TRY(uqb_dfree(ctx, d_total, 8));
        UQB_TRY(uqb_dfree(ctx, dp, sizeof(dec_params)));
        for (size_t i = 0; i < temps.size(); i++) UQB_TRY(uqb_dfree(ctx, temps[i], temp_sizes[i]));
        return uqb_fail(ctx, "decode: DNA row %llu has no valid length marker (malformed variable-length table)", bad_row);
    }
    UQB_TRY(uqb_new_array(ctx, total, 1, fastq));
    bool done = false;
    const uint32_t in_words = ((DT_R * dna->width + 3) / 4 + 4 + 3) / 4 * 4 + (DT_R * qual->width + 3) / 4 + 8;
    if (n && !p->variable && (size_t)in_words * 4 <= DT_IN_CAP && total / n < DT_TEXT_CAP / DT_R - 16 && (((uintptr_t)(*fastq)->d) & 15) == 0) {
        // fixed-length reads whose tiles fit shared memory
        unsigned int* d_fb;
        UQB_TRY(uqb_dalloc_t(ctx, &d_fb, 1));
        UQB_CUDA(cudaMemsetAsync(d_fb, 0, 4, ctx->stream));
        uint64_t tab = 0;
        for (uint32_t c = 0; c < p->ncols; c++) tab += n * cols[c]->width;
        if (has_str) {
            UQB_CUDA(cudaFuncSetAttribute(k_decode_tiles_str, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(dt_smem)));
            UQB_LAUNCH_B(n * ((uint64_t)dna->width + qual->width + 8) + tab + total, k_decode_tiles_str, uqb_grid(ctx, n, DT_R, 4), DT_THREADS, sizeof(dt_smem), dp,
                         (const uint8_t*)dna->d, (const uint8_t*)qual->d, n, rec_off, total, (uint8_t*)(*fastq)->d, d_fb);
        } else {
            UQB_CUDA(cudaFuncSetAttribute(k_decode_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(dt_smem)));
            UQB_LAUNCH_B(n * ((uint64_t)dna->width + qual->width + 8) + tab + total, k_decode_tiles, uqb_grid(ctx, n, DT_R, 4), DT_THREADS, sizeof(dt_smem), dp,
                         (const uint8_t*)dna->d, (const uint8_t*)qual->d, n, rec_off, total, (uint8_t*)(*fastq)->d, d_fb);
        }
        unsigned int fb = 0;
        UQB_TRY(uqb_readback(ctx, &fb, d_fb, 4));
        UQB_TRY(uqb_dfree(ctx, d_fb, 4));
        done = fb == 0;
    }
    if (n && !done && has_str) UQB_LAUNCH(k_decode_write_str, uqb_grid(ctx, n, DC / 32, 16), DC, 0, dp, (const uint8_t*)dna->d, (const uint8_t*)qual->d, n, rec_off, (uint8_t*)(*fastq)->d);
    else if (n && !done) UQB_LAUNCH(k_decode_write, uqb_grid(ctx, n, DC / 32, 16), DC, 0, dp, (const uint8_t*)dna->d, (const uint8_t*)qual->d, n, rec_off, (uint8_t*)(*fastq)->d);
    UQB_TRY(uqb_dfree(ctx, rec_len, n * 4));
    UQB_TRY(uqb_dfree(ctx, rec_off, n * 8));
    UQB_TRY(uqb_dfree(ctx, d_total, 8));
    UQB_TRY(uqb_dfree(ctx, dp, sizeof(dec_params)));
    for (size_t i = 0; i < temps.size(); i++) UQB_TRY(uqb_dfree(ctx, temps[i], temp_sizes[i]));
    return 0;
}
