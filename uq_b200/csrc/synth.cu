// Synthetic FASTQ generator on the device (bench / tests only): the same counter-based generator as
// oracle/synth.py (kind 4 'umi': oracle/synth_umi.py), so bench.py can create the 100 M-read inputs of BASELINE.json directly in HBM.
#include "common.cuh"

#define SY 256
#define GOLD 0x9E3779B97F4A7C15ull
#define IDXK 0x632BE59BD9B4E019ull

enum { ST_LANE = 1, ST_TILE = 2, ST_X = 3, ST_Y = 4, ST_NPOS = 5, ST_BASE = 6, ST_QA = 7, ST_QB = 8, ST_FLAG = 9, ST_EVEN = 10,
       ST_BARCODE = 11, ST_OFF = 12, ST_SUB = 13, ST_SUBV = 14, ST_POOL = 15, ST_LEN = 16, ST_RUN = 17, ST_CH = 18,
       ST_UMI_LEN = 20, ST_UMI = 21, ST_GENOME = 100 };

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}
__device__ __forceinline__ unsigned long long rnd(unsigned long long seed, unsigned long long stream, unsigned long long idx) {
    return mix64((seed + stream * GOLD) ^ mix64(idx + IDXK));
}
__device__ __forceinline__ unsigned skew(unsigned long long a, unsigned long long b, unsigned nsym) {
    unsigned long long m = nsym + 1;
    unsigned long long v = ((a % m) * (b % m)) / m;
    return v < nsym - 1 ? (unsigned)v : nsym - 1;
}
__device__ __forceinline__ unsigned put_uint(uint8_t* w, unsigned long long v) {     // decimal, no padding; returns digits
    unsigned n = 0;
    unsigned long long a = v;
    do { n++; a /= 10; } while (a);
    if (w) { a = v; for (unsigned i = 0; i < n; i++) { w[n - 1 - i] = (uint8_t)('0' + a % 10); a /= 10; } }
    return n;
}
__device__ __forceinline__ unsigned put_str(uint8_t* w, const char* s) {
    unsigned n = 0;
    while (s[n]) { if (w) w[n] = (uint8_t)s[n]; n++; }
    return n;
}

__constant__ char c_barcodes[4][8] = {"ATCACG", "CGATGT", "TTAGGC", "TGACCA"};

// header text of record r (global index); w == nullptr only measures
__device__ unsigned synth_header(uint8_t* w, const uqb_synth_params& p, unsigned long long r) {
    const unsigned long long lane = 1 + rnd(p.seed, ST_LANE, r) % 8, tile = 1101 + rnd(p.seed, ST_TILE, r) % 1578;
    const unsigned long long x = 1000 + rnd(p.seed, ST_X, r) % 29000, y = 1000 + rnd(p.seed, ST_Y, r) % 199000;
    unsigned n = 0;
#define W (w ? w + n : nullptr)
    if (p.kind == 0 || p.kind == 1 || p.kind == 4) {
        n += put_str(W, "@SIM001:1:FCX123:");
        n += put_uint(W, lane); n += put_str(W, ":"); n += put_uint(W, tile); n += put_str(W, ":");
        n += put_uint(W, x); n += put_str(W, ":"); n += put_uint(W, y);
        if (p.kind == 4) {          // umi: '_' + 6-12 symbols of ACGTN, as UMI extraction tools append them
            const unsigned ulen = 6 + (unsigned)(rnd(p.seed, ST_UMI_LEN, r) % 7);
            n += put_str(W, "_");
            for (unsigned j = 0; j < ulen; j++) {
                if (w) w[n] = (uint8_t)"ACGTN"[rnd(p.seed, ST_UMI, r * 16 + j) % 5];
                n++;
            }
        }
    } else if (p.kind == 2) {
        const bool flag = rnd(p.seed, ST_FLAG, r) % 8 == 0;
        const unsigned long long even = 2 * (rnd(p.seed, ST_EVEN, r) % 20), bc = rnd(p.seed, ST_BARCODE, r) % 4;
        n += put_str(W, "@EAS139:136:FC706VJ:");
        n += put_uint(W, lane); n += put_str(W, ":"); n += put_uint(W, tile); n += put_str(W, ":");
        n += put_uint(W, x); n += put_str(W, ":"); n += put_uint(W, y);
        n += put_str(W, " 1:"); n += put_str(W, flag ? "Y" : "N"); n += put_str(W, ":");
        n += put_uint(W, even); n += put_str(W, ":"); n += put_str(W, c_barcodes[bc]);
    } else {
        const unsigned long long run = 1 + rnd(p.seed, ST_RUN, r) % 4, ch = 1 + rnd(p.seed, ST_CH, r) % 512;
        n += put_str(W, "@ONT7:");
        n += put_uint(W, run); n += put_str(W, ":"); n += put_uint(W, r + 1); n += put_str(W, ":"); n += put_uint(W, ch);
    }
#undef W
    return n;
}

__device__ __forceinline__ unsigned synth_read_len(const uqb_synth_params& p, const long long* __restrict__ len_table, unsigned long long r) {
    if (p.kind != 3) return p.length;
    return (unsigned)len_table[rnd(p.seed, ST_LEN, r) >> 52];
}

__global__ void __launch_bounds__(SY) k_synth_len(uqb_synth_params p, const long long* __restrict__ len_table, uint32_t* __restrict__ rec_len) {
    const unsigned long long i = (unsigned long long)blockIdx.x * SY + threadIdx.x;
    if (i >= p.n) return;
    const unsigned long long r = p.first + i;
    const unsigned L = synth_read_len(p, len_table, r);
    rec_len[i] = synth_header(nullptr, p, r) + 1 + L + 3 + L + 1;
}

__global__ void __launch_bounds__(SY) k_synth_write(uqb_synth_params p, const long long* __restrict__ len_table,
                                                   const uint64_t* __restrict__ rec_off, uint8_t* __restrict__ out) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned long long wstride = (unsigned long long)gridDim.x * (SY / 32);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (SY / 32) + (threadIdx.x >> 5); i < p.n; i += wstride) {
        const unsigned long long r = p.first + i;
        uint8_t* o = out + rec_off[i];
        const unsigned L = synth_read_len(p, len_table, r);
        unsigned hl = 0;
        if (lane == 0) { hl = synth_header(o, p, r); o[hl] = '\n'; }
        hl = __shfl_sync(0xffffffffu, hl, 0);
        uint8_t* od = o + hl + 1;
        uint8_t* oq = od + L + 3;
        unsigned long long off = 0, pidx = 0;
        if (p.kind == 1) {
            off = rnd(p.seed, ST_OFF, r) % (p.genome - L);
            pidx = rnd(p.seed, ST_POOL, r) % p.pool;
        }
        for (unsigned pos = lane; pos < L; pos += 32) {
            const unsigned long long gidx = (p.kind == 3 ? r * (1ull << 24) : r * (1ull << 20)) + pos;
            unsigned b, qidx;
            if (p.kind == 1) {
                b = (unsigned)(rnd(p.seed, ST_GENOME, off + pos) & 3ull);
                if (rnd(p.seed, ST_SUB, gidx) % 1000 == 0) b = (b + 1 + (unsigned)(rnd(p.seed, ST_SUBV, gidx) % 3)) & 3u;
                const unsigned long long qi = pidx * L + pos;
                qidx = skew(rnd(p.seed, ST_QA, qi), rnd(p.seed, ST_QB, qi), 38);
            } else {
                b = (unsigned)(rnd(p.seed, ST_BASE, gidx) & 3ull);
                qidx = skew(rnd(p.seed, ST_QA, gidx), rnd(p.seed, ST_QB, gidx), p.kind == 3 ? 70 : 38);
            }
            uint8_t dch = "ACGT"[b], qch;
            if (p.kind == 3) {
                qch = (uint8_t)(33 + qidx);
            } else {
                qch = (uint8_t)(74 - qidx);
                if (rnd(p.seed, ST_NPOS, gidx) % 200 == 0) { dch = 'N'; qch = '#'; }
            }
            od[pos] = dch;
            oq[pos] = qch;
        }
        if (lane == 0) { od[L] = '\n'; od[L + 1] = '+'; od[L + 2] = '\n'; oq[L] = '\n'; }
    }
}

extern "C" int uqb_synth(uqb_ctx* ctx, const uqb_synth_params* p, const int64_t* ont_len_table, uqb_array** bytes) {
    if (p->kind > 4) return uqb_fail(ctx, "synth: kind %u", p->kind);
    if (p->kind == 3 && !ont_len_table) return uqb_fail(ctx, "synth: ont needs a length table");
    if (p->kind == 1 && (p->genome <= p->length || p->pool == 0)) return uqb_fail(ctx, "synth: genome/pool too small");
    if (p->n >= (1ull << 32)) return uqb_fail(ctx, "synth: too many records");
    long long* dtab = nullptr;
    if (p->kind == 3) {
        UQB_TRY(uqb_dalloc_t(ctx, &dtab, 4096));
        UQB_CUDA(cudaMemcpyAsync(dtab, ont_len_table, 4096 * 8, cudaMemcpyHostToDevice, ctx->stream));
        UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    uint32_t* rec_len;
    uint64_t *rec_off, *d_total;
    UQB_TRY(uqb_dalloc_t(ctx, &rec_len, p->n));
    UQB_TRY(uqb_dalloc_t(ctx, &rec_off, p->n));
    UQB_TRY(uqb_dalloc_t(ctx, &d_total, 1));
    if (p->n) UQB_LAUNCH(k_synth_len, uqb_blocks(p->n, SY), SY, 0, *p, dtab, rec_len);
    UQB_TRY(uqb_scan_u32_to_u64(ctx, rec_len, rec_off, p->n, d_total));
    uint64_t total = 0;
    UQB_TRY(uqb_readback(ctx, &total, d_total, 8));
    UQB_TRY(uqb_new_array(ctx, total, 1, bytes));
    if (p->n) UQB_LAUNCH(k_synth_write, uqb_grid(ctx, p->n, SY / 32, 16), SY, 0, *p, dtab, rec_off, (uint8_t*)(*bytes)->d);
    UQB_TRY(uqb_dfree(ctx, rec_len, p->n * 4));
    UQB_TRY(uqb_dfree(ctx, rec_off, p->n * 8));
    UQB_TRY(uqb_dfree(ctx, d_total, 8));
    if (dtab) UQB_TRY(uqb_dfree(ctx, dtab, 4096 * 8));
    return 0;
}
