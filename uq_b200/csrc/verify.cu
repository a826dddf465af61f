// Encode verification (uq.py has no counterpart): the container's decoded text is compared, record by record, with the
// FASTQ it was encoded from, under the order that links container row i to its input record, and that order is checked
// to be a permutation.  Both run on data that is already in HBM at the end of the encode.
#include "common.cuh"

#define VT 256                      // threads per CTA: 8 warps, each on 32 consecutive rows at a time

// chunk c (8 bytes) of a byte range that starts at `s`: aligned 64-bit words w[c], w[c + 1] of the range's aligned base,
// joined by a funnel shift.  Lane l holds word l + 32 * it, takes word + 1 from lane l + 1 and lane 31 loads it itself.
// A word is loaded only if it holds at least one byte of the range, so nothing past the range's last aligned word is read.
__device__ __forceinline__ uint64_t range_chunk(const uint8_t* s, uint64_t len, uint64_t c0, unsigned lane) {
    const uintptr_t a = (uintptr_t)s & ~(uintptr_t)7;
    const uint32_t sh = (uint32_t)((uintptr_t)s & 7u) * 8u;
    const uintptr_t end = (uintptr_t)s + len;
    const uintptr_t p0 = a + 8 * (c0 + lane);
    const uint64_t w0 = p0 < end ? __ldg(reinterpret_cast<const unsigned long long*>(p0)) : 0ull;
    uint64_t w1 = __shfl_down_sync(0xffffffffu, w0, 1);
    if (lane == 31) w1 = p0 + 8 < end ? __ldg(reinterpret_cast<const unsigned long long*>(p0 + 8)) : 0ull;
    return sh ? (w0 >> sh) | (w1 << (64u - sh)) : w0;
}

// bytes [0, k) of an 8-byte chunk as a mask, k in [0, 8]
__device__ __forceinline__ uint64_t bytes_below(int64_t k) {
    return k <= 0 ? 0ull : k >= 8 ? ~0ull : (1ull << (8 * k)) - 1ull;
}

__device__ __forceinline__ void mark_fields(uint64_t x, int64_t p, uint64_t len, const uint64_t b[5], unsigned& flags) {
    // 0x80 in every byte of x that is not zero (exact: no carry crosses a byte)
    uint64_t nz = (((x & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | x) & 0x8080808080808080ull;
    nz &= bytes_below((int64_t)len - p);
    if (nz) {
#pragma unroll
        for (int f = 0; f < 4; f++)
            if (nz & bytes_below((int64_t)b[f + 1] - p) & ~bytes_below((int64_t)b[f] - p)) flags |= 1u << f;
    }
}

// bytes [0, len) at sa and sb compared by the whole warp, 512 bytes (two chunks a lane, four loads in flight) per step;
// field f owns the bytes [b[f], b[f + 1]) (b[0] = 0, b[4] = len).  -> this lane's mask of fields with a differing byte
__device__ __forceinline__ unsigned diff_fields(const uint8_t* sa, const uint8_t* sb, uint64_t len, const uint64_t b[5], unsigned lane) {
    unsigned flags = 0;
    for (uint64_t c0 = 0; c0 * 8 < len; c0 += 64) {
        const bool two = (c0 + 32) * 8 < len;                             // warp-uniform
        const uint64_t x0 = range_chunk(sa, len, c0, lane) ^ range_chunk(sb, len, c0, lane);
        const uint64_t x1 = two ? range_chunk(sa, len, c0 + 32, lane) ^ range_chunk(sb, len, c0 + 32, lane) : 0ull;
        mark_fields(x0, (int64_t)(8 * (c0 + lane)), len, b, flags);
        mark_fields(x1, (int64_t)(8 * (c0 + 32 + lane)), len, b, flags);
    }
    return flags;
}

// Container rows [row0, row0 + k): decoded record t = row - row0 (text) against input record order[row] (src, identity
// without an order).  A warp takes 32 consecutive rows: each lane loads the order entry and the ten line offsets of one
// of them into shared memory (all independent loads, in flight together), then the warp compares the 32 records one
// after the other - the four line lengths first, then the bytes: the whole record as one range when every length
// agrees, otherwise each line whose length agrees on its own.  An input record number >= n_src is a difference in all
// four fields and is never dereferenced.  Per warp, one atomicAdd per field for the count and one atomicMin per field for
// (row << 32 | input record) of the first difference.
__global__ void __launch_bounds__(VT, 4) k_verify_records(const uint8_t* __restrict__ src, const uint64_t* __restrict__ src_off, uint64_t n_src,
                                                      const uint8_t* __restrict__ txt, const uint64_t* __restrict__ txt_off, uint64_t k,
                                                      uint64_t row0, const uint32_t* __restrict__ order,
                                                      unsigned long long* __restrict__ count, unsigned long long* __restrict__ first) {
    __shared__ uint64_t s_off[VT / 32][32][10];  // per row: 5 input line offsets, 5 decoded line offsets
    __shared__ uint64_t s_rec[VT / 32][32];
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint64_t nwarps = (uint64_t)gridDim.x * (VT / 32);
    uint64_t my_count = 0;                       // lane f < 4: rows of this warp whose field f differs
    unsigned long long my_first = ~0ull;
    for (uint64_t t0 = ((uint64_t)blockIdx.x * (VT / 32) + w) * 32; t0 < k; t0 += nwarps * 32) {
        const uint32_t nr = (uint32_t)(k - t0 < 32 ? k - t0 : 32);
        __syncwarp();
        if (lane < nr) {
            const uint64_t t = t0 + lane, row = row0 + t;
            const uint64_t r = order ? (uint64_t)__ldg(order + row) : row;
            s_rec[w][lane] = r;
            if (r < n_src) {
#pragma unroll
                for (int j = 0; j < 5; j++) s_off[w][lane][j] = __ldg(src_off + 4 * r + j);
            }
#pragma unroll
            for (int j = 0; j < 5; j++) s_off[w][lane][5 + j] = __ldg(txt_off + 4 * t + j);
        }
        __syncwarp();
        for (uint32_t i = 0; i < nr; i++) {
            const uint64_t r = s_rec[w][i];
            unsigned m = 0xFu;
            if (r < n_src) {
                const uint64_t* so = s_off[w][i];
                const uint64_t* to = so + 5;
                unsigned lenmask = 0;
#pragma unroll
                for (int f = 0; f < 4; f++) lenmask |= (so[f + 1] - so[f] != to[f + 1] - to[f]) ? 1u << f : 0u;
                unsigned flags;
                if (!lenmask) {
                    const uint64_t b[5] = {0, so[1] - so[0], so[2] - so[0], so[3] - so[0], so[4] - so[0]};
                    flags = diff_fields(src + so[0], txt + to[0], so[4] - so[0], b, lane);
                } else {
                    flags = lenmask;
                    for (int f = 0; f < 4; f++) {
                        if (lenmask & (1u << f)) continue;
                        const uint64_t len = so[f + 1] - so[f];
                        uint64_t b[5];
#pragma unroll
                        for (int j = 0; j < 5; j++) b[j] = j <= f ? 0 : len;
                        flags |= diff_fields(src + so[f], txt + to[f], len, b, lane);
                    }
                }
                m = 0;
#pragma unroll
                for (int f = 0; f < 4; f++) m |= __ballot_sync(0xffffffffu, flags & (1u << f)) ? 1u << f : 0u;
            }
            if (lane < 4 && (m & (1u << lane))) {
                my_count++;
                if (my_first == ~0ull) my_first = ((row0 + t0 + i) << 32) | r;     // rows of a warp ascend
            }
        }
    }
    if (lane < 4 && my_count) {
        atomicAdd(count + lane, (unsigned long long)my_count);
        atomicMin(first + lane, my_first);
    }
}

// one bit per value of order that lies in [0, n)
__global__ void __launch_bounds__(VT) k_perm_mark(const uint32_t* __restrict__ order, uint64_t m, uint64_t n, uint32_t* __restrict__ bits) {
    for (uint64_t i = (uint64_t)blockIdx.x * VT + threadIdx.x; i < m; i += (uint64_t)gridDim.x * VT) {
        const uint32_t v = __ldg(order + i);
        if (v < n) atomicOr(bits + (v >> 5), 1u << (v & 31u));
    }
}

// smallest value in [0, n) whose bit is clear
__global__ void __launch_bounds__(VT) k_perm_missing(const uint32_t* __restrict__ bits, uint64_t n, unsigned long long* __restrict__ missing) {
    const uint64_t nw = (n + 31) / 32;
    unsigned long long best = ~0ull;
    for (uint64_t w = (uint64_t)blockIdx.x * VT + threadIdx.x; w < nw; w += (uint64_t)gridDim.x * VT) {
        const uint32_t want = (w + 1 < nw || (n & 31u) == 0) ? ~0u : (1u << (n & 31u)) - 1u;
        const uint32_t clear = ~__ldg(bits + w) & want;
        if (clear && best == ~0ull) best = 32 * w + (uint64_t)(__ffs((int)clear) - 1);
    }
    best = __reduce_min_sync(0xffffffffu, (unsigned)(best == ~0ull ? 0xFFFFFFFFu : best)) == 0xFFFFFFFFu ? ~0ull : best;
    if (best != ~0ull) atomicMin(missing, best);
}

extern "C" int uqb_verify_records(uqb_ctx* ctx, const uqb_fastq* src, const uqb_fastq* text, uint64_t first_row,
                                  const uqb_array* order, uqb_verify_report* report) {
    if (!src->line_off || !text->line_off) return uqb_fail(ctx, "verify_records: split both FASTQ handles first (uqb_split)");
    if (src->n_lines % 4 || text->n_lines % 4) return uqb_fail(ctx, "verify_records: a line count is not divisible by 4");
    const uint64_t k = text->n_reads;
    if (first_row + k > (1ull << 32)) return uqb_fail(ctx, "verify_records: container rows beyond 2^32");
    if (order && (order->width != 4 || first_row + k > order->n))
        return uqb_fail(ctx, "verify_records: order must be uint32 and hold rows [%llu, %llu)", (unsigned long long)first_row,
                        (unsigned long long)(first_row + k));
    report->records += k;
    if (k == 0) return 0;
    unsigned long long* d;                       // [0..4) counts, [4..8) first (row << 32 | input record)
    UQB_TRY(uqb_dalloc_t(ctx, &d, 8));
    UQB_CUDA(cudaMemsetAsync(d, 0, 32, ctx->stream));
    UQB_CUDA(cudaMemsetAsync(d + 4, 0xFF, 32, ctx->stream));
    // compulsory bytes: both texts once (equal in size when the records agree), five line offsets a side, the order
    const uint64_t ab = 2 * text->n + k * (80 + (order ? 4 : 0));
    UQB_LAUNCH_B(ab, k_verify_records, uqb_grid(ctx, k, VT, 8), VT, 0, src->d, src->line_off, src->n_reads, text->d, text->line_off, k,
                 first_row, order ? (const uint32_t*)order->d : nullptr, d, d + 4);
    unsigned long long h[8];
    UQB_TRY(uqb_readback(ctx, h, d, 64));
    UQB_TRY(uqb_dfree(ctx, d, 64));
    for (int f = 0; f < 4; f++) {
        report->differ[f] += h[f];
        if (h[4 + f] == ~0ull) continue;
        const int64_t row = (int64_t)(h[4 + f] >> 32), rec = (int64_t)(h[4 + f] & 0xFFFFFFFFull);
        if (report->first_row[f] < 0 || row < report->first_row[f]) { report->first_row[f] = row; report->first_src[f] = rec; }
    }
    return 0;
}

extern "C" int uqb_check_permutation(uqb_ctx* ctx, const uqb_array* order, uint64_t n, int64_t* missing) {
    if (order->width != 4) return uqb_fail(ctx, "check_permutation: order must be uint32");
    if (n >= (1ull << 32)) return uqb_fail(ctx, "check_permutation: n must be below 2^32");
    *missing = -1;
    if (n == 0) return 0;
    const uint64_t nw = (n + 31) / 32;
    uint32_t* bits;
    unsigned long long* d;
    UQB_TRY(uqb_dalloc_t(ctx, &bits, nw));
    UQB_TRY(uqb_dalloc_t(ctx, &d, 1));
    UQB_CUDA(cudaMemsetAsync(bits, 0, nw * 4, ctx->stream));
    UQB_CUDA(cudaMemsetAsync(d, 0xFF, 8, ctx->stream));
    if (order->n) UQB_LAUNCH_B(order->n * 4 + nw * 4, k_perm_mark, uqb_grid(ctx, order->n, VT, 16), VT, 0, (const uint32_t*)order->d, order->n, n, bits);
    UQB_LAUNCH_B(nw * 4, k_perm_missing, uqb_grid(ctx, nw, VT, 8), VT, 0, bits, n, d);
    unsigned long long h = ~0ull;
    UQB_TRY(uqb_readback(ctx, &h, d, 8));
    UQB_TRY(uqb_dfree(ctx, bits, nw * 4));
    UQB_TRY(uqb_dfree(ctx, d, 8));
    *missing = h == ~0ull ? -1 : (int64_t)h;
    return 0;
}
