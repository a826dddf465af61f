// Stage 1a: record splitting.  Newline scan over the raw FASTQ byte stream -> uint64 line offsets.
// Replaces the four `for line in file` sweeps of the reference (uq.py:132-139, 205-211, 378-385,
// 563-569) and its `wc -l` record count (uq.py:85-87).
//
// HBM traffic: the byte stream is read twice (count, then write) with 128-bit loads; line
// offsets (8 B per line) are written once.  Each thread owns 64 consecutive bytes so that the
// rank of a newline inside the tile follows byte order.
#include "common.cuh"

#define SP_THREADS 256
#define SP_BYTES_PER_THREAD 64
#define SP_TILE (SP_THREADS * SP_BYTES_PER_THREAD)
#define SP_STAGE 1024          // line offsets staged per tile (a 16 KB tile of FASTQ holds ~200)

// 0x01 in every byte of w that is '\n'.  Exact SIMD-in-register zero-byte test of w ^ 0x0A0A0A0A (the add cannot carry
// across bytes because bit 7 is masked off first): four integer instructions per word, where __vcmpeq4 is emulated byte
// by byte on this architecture (the newline-write kernel was bound by exactly those instructions).
__device__ __forceinline__ unsigned nl_bits(unsigned w) {
    const unsigned x = w ^ 0x0A0A0A0Au;
    const unsigned t = ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x;              // bit 7 of a byte set <=> the byte is non-zero
    return (~t & 0x80808080u) >> 7;
}

// load the 16 words of this thread's 64-byte chunk; bytes at or beyond `n` read as zero
__device__ __forceinline__ void load_chunk(const uint8_t* __restrict__ d, uint64_t n, uint64_t pos, unsigned (&w)[16]) {
    if (pos + SP_BYTES_PER_THREAD <= n) {
        const uint4* p = reinterpret_cast<const uint4*>(d + pos);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            uint4 q = __ldg(p + i);
            w[4 * i] = q.x; w[4 * i + 1] = q.y; w[4 * i + 2] = q.z; w[4 * i + 3] = q.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; i++) {
            unsigned x = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                uint64_t q = pos + 4 * i + b;
                if (q < n) x |= (unsigned)d[q] << (8 * b);
            }
            w[i] = x;
        }
    }
}

__global__ void __launch_bounds__(SP_THREADS) k_newline_count(const uint8_t* __restrict__ d, uint64_t n, uint64_t tile0, uint32_t* __restrict__ tile_counts) {
    uint64_t pos = (tile0 + blockIdx.x) * SP_TILE + (uint64_t)threadIdx.x * SP_BYTES_PER_THREAD;
    unsigned c = 0;
    if (pos < n) {
        unsigned w[16];
        load_chunk(d, n, pos, w);
#pragma unroll
        for (int i = 0; i < 16; i++) c += __popc(nl_bits(w[i]));
    }
    // block reduce
    __shared__ unsigned ws[SP_THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane_id() == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
#pragma unroll
        for (int i = 0; i < SP_THREADS / 32; i++) t += ws[i];
        tile_counts[tile0 + blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(SP_THREADS) k_newline_write(const uint8_t* __restrict__ d, uint64_t n, uint64_t tile0, uint64_t line_base,
                                                            const uint64_t* __restrict__ tile_base, uint64_t* __restrict__ line_off) {
    uint64_t pos = (tile0 + blockIdx.x) * SP_TILE + (uint64_t)threadIdx.x * SP_BYTES_PER_THREAD;
    // bit b of `nl` = byte b of this thread's 64-byte chunk is a newline: four mask bits per word, gathered with
    // one multiply (the 0x01 bits of the byte mask land in bits 24..27)
    unsigned long long nl = 0;
    if (pos < n) {
        unsigned w[16];
        load_chunk(d, n, pos, w);
        unsigned lo = 0, hi = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            lo |= ((nl_bits(w[i]) * 0x01020408u) >> 24) << (4 * i);
            hi |= ((nl_bits(w[8 + i]) * 0x01020408u) >> 24) << (4 * i);
        }
        nl = ((unsigned long long)hi << 32) | lo;
    }
    const unsigned c = __popcll(nl);
    // exclusive scan of c over the CTA
    __shared__ unsigned ws[SP_THREADS / 32];
    unsigned lane = lane_id(), wid = threadIdx.x >> 5;
    unsigned incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) ws[wid] = incl;
    __syncthreads();
    unsigned wbase = 0;
#pragma unroll
    for (int i = 0; i < SP_THREADS / 32; i++)
        if ((unsigned)i < wid) wbase += ws[i];
    // the tile's offsets are staged in shared memory in order and stored as one contiguous run
    __shared__ uint64_t stage[SP_STAGE];
    __shared__ unsigned tile_total;
    if (threadIdx.x == SP_THREADS - 1) tile_total = wbase + incl;
    __syncthreads();
    const unsigned total = tile_total;
    const uint64_t out0 = line_base + tile_base[tile0 + blockIdx.x] + 1;      // +1: line_off[0] = 0 is the first line
    unsigned k = wbase + incl - c;
    const bool staged = total <= SP_STAGE;
    while (nl) {
        const int b = __ffsll((long long)nl) - 1;
        nl &= nl - 1;
        const uint64_t v = pos + b + 1;                                      // the next line starts after the newline
        if (staged) stage[k] = v; else line_off[out0 + k] = v;
        k++;
    }
    if (staged) {
        __syncthreads();
        for (unsigned i = threadIdx.x; i < total; i += SP_THREADS) line_off[out0 + i] = stage[i];
    }
}

__global__ void k_set_u64(uint64_t* p, uint64_t v) { *p = v; }

// ---- one pass: count, number and write in the same sweep ------------------------------------------
// k_newline_count + scan + k_newline_write read the byte stream twice.  Here a CTA takes SP1_SUB consecutive 16 KB tiles
// (a "span", in blockIdx order), counts the newlines of the span while it keeps the 64-bit newline masks of all sub-tiles in
// registers, learns the number of newlines in front of the span from a decoupled look-back over one 64-bit status word per
// span (flag 1 = the span's own count, flag 2 = inclusive prefix; Merrill & Garland), and writes the offsets from the kept
// masks.  The stream is read once; the only serial dependence between CTAs is the status word.
// The number of lines is not known before the pass: the caller sizes line_off from the newline density of the head of
// the file; a span that would write past `cap` raises *overflow and writes nothing (the caller falls back to two passes).
#ifndef SP1_SUB
#define SP1_SUB 4
#endif
struct sp1_smem {
    uint64_t stage[SP_STAGE];
    unsigned ws[SP1_SUB][SP_THREADS / 32];
    unsigned sub_total[SP1_SUB];
    unsigned span;
    unsigned long long prefix;
};

__device__ __forceinline__ unsigned long long sp1_ld(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void sp1_st(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(SP_THREADS, 8) k_newline_scan1(const uint8_t* __restrict__ d, uint64_t n, uint64_t nspans,
                                                             unsigned int* __restrict__ ticket, unsigned long long* __restrict__ status,
                                                             uint64_t* __restrict__ line_off, uint64_t cap,
                                                             unsigned long long* __restrict__ total_out, unsigned int* __restrict__ overflow) {
    __shared__ sp1_smem S;
    const unsigned tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    // Spans are taken in blockIdx order, which is the order the hardware dispatches the CTAs of a 1-D grid in (the
    // assumption every blockIdx-ordered decoupled look-back makes): a ticket counter serialised the launch at ~18 ns per
    // CTA.  Should a predecessor ever fail to show up, the wait below is bounded: the CTA raises *overflow (bit 1) and the
    // caller runs the two-pass path.
    const uint64_t span = blockIdx.x;
    (void)ticket;
    if (span >= nspans) return;
    unsigned long long nl[SP1_SUB];
    unsigned incl[SP1_SUB];
    // the tiles of a span are taken one after the other: issuing their loads together (32 or 64 data registers) costs
    // more in occupancy than it gains in bytes in flight (measured: 12.9 / 13.7 ms against 10.7 ms)
#pragma unroll
    for (int q = 0; q < SP1_SUB; q++) {
        const uint64_t pos = (span * SP1_SUB + q) * SP_TILE + (uint64_t)tid * SP_BYTES_PER_THREAD;
        nl[q] = 0;
        if (pos < n) {
            unsigned w[16];
            load_chunk(d, n, pos, w);
            unsigned lo = 0, hi = 0;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                lo |= ((nl_bits(w[i]) * 0x01020408u) >> 24) << (4 * i);
                hi |= ((nl_bits(w[8 + i]) * 0x01020408u) >> 24) << (4 * i);
            }
            nl[q] = ((unsigned long long)hi << 32) | lo;
        }
        unsigned x = __popcll(nl[q]);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (unsigned)o) x += t;
        }
        incl[q] = x;
        if (lane == 31) S.ws[q][wid] = x;
    }
    __syncthreads();
    if (tid < SP1_SUB) {
        unsigned t = 0;
#pragma unroll
        for (int i = 0; i < SP_THREADS / 32; i++) t += S.ws[tid][i];
        S.sub_total[tid] = t;
    }
    __syncthreads();
    unsigned own = 0;
#pragma unroll
    for (int q = 0; q < SP1_SUB; q++) own += S.sub_total[q];
    // ---- look-back (warp 0) ----
    if (wid == 0) {
        unsigned long long run = 0;
        bool gave_up = false;
        if (span == 0) {
            if (lane == 0) { __threadfence(); sp1_st(status, (2ull << 62) | own); }
        } else {
            if (lane == 0) { __threadfence(); sp1_st(status + span, (1ull << 62) | own); }
            long long at = (long long)span - 1;                       // lane l looks at span at - l
            while (true) {
                const long long my = at - (long long)lane;
                unsigned long long v = my >= 0 ? sp1_ld(status + my) : (2ull << 62);
                unsigned spins = 0;
                while (__any_sync(0xffffffffu, (v >> 62) == 0)) {
                    if ((v >> 62) == 0) { __nanosleep(20); v = sp1_ld(status + my); }
                    if ((++spins & 1023u) == 0 && (spins > (1u << 20) || *(volatile unsigned int*)overflow)) { gave_up = true; break; }
                }
                if (gave_up) break;
                const unsigned incl_mask = __ballot_sync(0xffffffffu, (v >> 62) == 2);
                const unsigned upto = incl_mask ? (unsigned)__ffs((int)incl_mask) - 1u : 31u;      // nearest inclusive prefix
                unsigned long long part = lane <= upto ? (v & ((1ull << 62) - 1ull)) : 0ull;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                run += part;
                if (incl_mask) break;
                at -= 32;
            }
            if (lane == 0 && !gave_up) { __threadfence(); sp1_st(status + span, (2ull << 62) | (run + own)); }
        }
        if (lane == 0) {
            if (gave_up) { atomicOr(overflow, 2u); run = ~0ull >> 2; }        // far beyond any capacity: nothing is written
            S.prefix = run;
            if (span == nspans - 1) *total_out = run + own;
        }
    }
    __syncthreads();
    uint64_t out0 = 1 + S.prefix;                                      // line_off[0] = 0 is the first line
    if (out0 + own > cap) {
        if (tid == 0) atomicOr(overflow, 1u);
        return;
    }
    // ---- offsets of the kept masks, one sub-tile at a time through the staging buffer ----
#pragma unroll
    for (int q = 0; q < SP1_SUB; q++) {
        const unsigned total = S.sub_total[q];
        if (total) {
            unsigned wbase = 0;
#pragma unroll
            for (int i = 0; i < SP_THREADS / 32; i++)
                if ((unsigned)i < wid) wbase += S.ws[q][i];
            const unsigned c = __popcll(nl[q]);
            unsigned k = wbase + incl[q] - c;
            const bool staged = total <= SP_STAGE;
            const uint64_t pos = (span * SP1_SUB + q) * SP_TILE + (uint64_t)tid * SP_BYTES_PER_THREAD;
            unsigned long long m = nl[q];
            while (m) {
                const int b = __ffsll((long long)m) - 1;
                m &= m - 1;
                const uint64_t v = pos + b + 1;
                if (staged) S.stage[k] = v; else line_off[out0 + k] = v;
                k++;
            }
            if (staged) {
                __syncthreads();
                for (unsigned i = tid; i < total; i += SP_THREADS) line_off[out0 + i] = S.stage[i];
                __syncthreads();
            }
            out0 += total;
        }
    }
}

extern "C" int uqb_fastq_load(uqb_ctx* ctx, const uint8_t* host, uint64_t nbytes, uqb_fastq** out) {
    uqb_fastq* fq = new uqb_fastq();
    uint8_t* d;
    int r = uqb_dalloc(ctx, (void**)&d, nbytes + 64);
    if (r) { delete fq; return r; }
    fq->d = d;
    fq->n = nbytes;
    fq->owned = true;
    UQB_CUDA(cudaMemsetAsync(d + nbytes, 0, 64, ctx->stream));
    if (nbytes) UQB_CUDA(cudaMemcpyAsync(d, host, nbytes, cudaMemcpyHostToDevice, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = fq;
    return 0;
}

extern "C" int uqb_fastq_adopt(uqb_ctx* ctx, const uint8_t* dev, uint64_t nbytes, uqb_fastq** out) {
    if (((uintptr_t)dev) & 15) return uqb_fail(ctx, "adopted FASTQ buffer must be 16-byte aligned");
    uqb_fastq* fq = new uqb_fastq();
    fq->d = dev;
    fq->n = nbytes;
    fq->owned = false;
    *out = fq;
    return 0;
}

static int free_qcols(uqb_ctx* ctx, uqb_fastq* fq) {
    for (auto& c : fq->qcols) {
        UQB_TRY(uqb_dfree(ctx, c.val, fq->n_reads * 8));
        UQB_TRY(uqb_dfree(ctx, c.span, fq->n_reads * 4));
        UQB_TRY(uqb_dfree(ctx, c.rank, fq->n_reads * 4));
        UQB_TRY(uqb_dfree(ctx, c.first_occ, 0));
        UQB_TRY(uqb_dfree(ctx, c.dict, c.dict_count * c.dict_width + 64));
    }
    fq->qcols.clear();
    return 0;
}

int uqb_fastq_free_qcols(uqb_ctx* ctx, uqb_fastq* fq) { return free_qcols(ctx, fq); }

extern "C" int uqb_fastq_free(uqb_ctx* ctx, uqb_fastq* fq) {
    if (!fq) return 0;
    UQB_TRY(free_qcols(ctx, fq));
    UQB_TRY(uqb_names_release(ctx, fq));
    if (fq->line_off) UQB_TRY(uqb_dfree(ctx, fq->line_off, (fq->n_lines + 1) * 8));
    delete fq->cached_stats;
    if (fq->ref_name) UQB_TRY(uqb_dfree(ctx, fq->ref_name, 0));
    if (fq->owned) UQB_TRY(uqb_dfree(ctx, (void*)fq->d, fq->n + 64));
    delete fq;
    return 0;
}

extern "C" int uqb_fastq_download(uqb_ctx* ctx, const uqb_fastq* fq, uint64_t offset, uint8_t* host, uint64_t nbytes) {
    if (offset + nbytes > fq->n) return uqb_fail(ctx, "fastq download out of range");
    if (nbytes) UQB_CUDA(cudaMemcpyAsync(host, fq->d + offset, nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// chunk-wise building blocks for the streamed load (analyze.cu)
int uqb_split_count_tiles(uqb_ctx* ctx, const uint8_t* d, uint64_t n_end, uint64_t tile0, uint64_t ntiles, uint32_t* counts) {
    UQB_LAUNCH_B(ntiles * SP_TILE, k_newline_count, (unsigned)ntiles, SP_THREADS, 0, d, n_end, tile0, counts);
    return 0;
}
int uqb_split_write_tiles(uqb_ctx* ctx, const uint8_t* d, uint64_t n_end, uint64_t tile0, uint64_t ntiles, uint64_t line_base,
                          const uint64_t* bases, uint64_t* line_off) {
    UQB_LAUNCH_B(ntiles * SP_TILE, k_newline_write, (unsigned)ntiles, SP_THREADS, 0, d, n_end, tile0, line_base, bases, line_off);
    return 0;
}
int uqb_split_set_first(uqb_ctx* ctx, uint64_t* line_off) {
    UQB_LAUNCH(k_set_u64, 1, 1, 0, line_off, 0ull);
    return 0;
}

extern "C" int uqb_split(uqb_ctx* ctx, uqb_fastq* fq, uqb_split_info* info) {
    memset(info, 0, sizeof(*info));
    if (fq->streamed && fq->line_off) {          // already split while the bytes were streaming in
        info->n_bytes = fq->n; info->n_lines = fq->n_lines; info->n_reads = fq->n_reads;
        info->status = (fq->n_lines % 4 == 0) ? 0 : 1;
        return 0;
    }
    info->n_bytes = fq->n;
    if (fq->line_off) { UQB_TRY(uqb_dfree(ctx, fq->line_off, (fq->n_lines + 1) * 8)); fq->line_off = nullptr; }
    UQB_TRY(uqb_names_release(ctx, fq));
    uint64_t ntiles = (fq->n + SP_TILE - 1) / SP_TILE;
    uint64_t total = 0;
    if (ntiles >= 64) {
        // one pass (k_newline_scan1).  line_off is sized from the newline density of the first 64 MB (or the whole file) plus 2 % and 1 M lines;
        // if the rest of the file is denser than that, the pass reports it and the two-pass path below runs instead.
        const uint64_t head_tiles = ntiles < 4096 ? ntiles : 4096;
        uint32_t* hc;
        uint64_t *hb, *hd;
        UQB_TRY(uqb_dalloc_t(ctx, &hc, head_tiles));
        UQB_TRY(uqb_dalloc_t(ctx, &hb, head_tiles));
        UQB_TRY(uqb_dalloc_t(ctx, &hd, 1));
        UQB_LAUNCH_B(head_tiles * SP_TILE, k_newline_count, (unsigned)head_tiles, SP_THREADS, 0, fq->d, fq->n, 0ull, hc);
        UQB_TRY(uqb_scan_u32_to_u64(ctx, hc, hb, head_tiles, hd));
        uint64_t head_lines = 0;
        UQB_TRY(uqb_readback(ctx, &head_lines, hd, 8));
        UQB_TRY(uqb_dfree(ctx, hc, 0)); UQB_TRY(uqb_dfree(ctx, hb, 0)); UQB_TRY(uqb_dfree(ctx, hd, 0));
        const double density = (double)head_lines / (double)(head_tiles * SP_TILE);
        const uint64_t cap = (uint64_t)(density * 1.02 * (double)fq->n) + (1u << 20);
        const uint64_t nspans = (ntiles + SP1_SUB - 1) / SP1_SUB;
        uint64_t* lo;
        unsigned long long* status;
        UQB_TRY(uqb_dalloc_t(ctx, &lo, cap + 1));
        UQB_TRY(uqb_dalloc_t(ctx, &status, nspans + 4));
        UQB_CUDA(cudaMemsetAsync(status, 0, (nspans + 4) * 8, ctx->stream));      // [nspans] ticket, [+1] total, [+2] overflow
        UQB_LAUNCH(k_set_u64, 1, 1, 0, lo, 0ull);
        UQB_LAUNCH_B(fq->n + 8 * (uint64_t)(density * (double)fq->n), k_newline_scan1, (unsigned)nspans, SP_THREADS, 0, fq->d, fq->n, nspans,
                     (unsigned int*)(status + nspans), status, lo, cap + 1, status + nspans + 1, (unsigned int*)(status + nspans + 2));
        unsigned long long res[2] = {0, 0};
        UQB_TRY(uqb_readback(ctx, res, status + nspans + 1, 16));
        UQB_TRY(uqb_dfree(ctx, status, 0));
        if ((unsigned int)res[1] == 0) {
            fq->line_off = lo;
            fq->n_lines = res[0];
            fq->n_reads = res[0] / 4;
            info->n_lines = fq->n_lines;
            info->n_reads = fq->n_reads;
            info->status = (fq->n_lines % 4 == 0) ? 0 : 1;
            return 0;
        }
        UQB_TRY(uqb_dfree(ctx, lo, 0));
    }
    uint32_t* counts = nullptr;
    uint64_t* bases = nullptr;
    uint64_t* d_total = nullptr;
    if (ntiles) {
        UQB_TRY(uqb_dalloc_t(ctx, &counts, ntiles));
        UQB_TRY(uqb_dalloc_t(ctx, &bases, ntiles));
        UQB_TRY(uqb_dalloc_t(ctx, &d_total, 1));
        UQB_LAUNCH_B(fq->n, k_newline_count, (unsigned)ntiles, SP_THREADS, 0, fq->d, fq->n, 0ull, counts);
        UQB_TRY(uqb_scan_u32_to_u64(ctx, counts, bases, ntiles, d_total));
        UQB_TRY(uqb_readback(ctx, &total, d_total, 8));
    }
    fq->n_lines = total;
    fq->n_reads = total / 4;
    UQB_TRY(uqb_dalloc_t(ctx, &fq->line_off, total + 1));
    UQB_LAUNCH(k_set_u64, 1, 1, 0, fq->line_off, 0ull);
    if (ntiles) {
        UQB_LAUNCH_B(fq->n + 8 * total, k_newline_write, (unsigned)ntiles, SP_THREADS, 0, fq->d, fq->n, 0ull, 0ull, bases, fq->line_off);
        UQB_TRY(uqb_dfree(ctx, counts, ntiles * 4));
        UQB_TRY(uqb_dfree(ctx, bases, ntiles * 8));
        UQB_TRY(uqb_dfree(ctx, d_total, 8));
    }
    info->n_lines = total;
    info->n_reads = total / 4;
    info->status = (total % 4 == 0) ? 0 : 1;
    return 0;
}

extern "C" int uqb_fastq_line_offsets(uqb_ctx* ctx, const uqb_fastq* fq, uint64_t first, uint64_t count, uint64_t* host) {
    if (!fq->line_off || first + count > fq->n_lines + 1) return uqb_fail(ctx, "line offset range out of bounds");
    if (count) UQB_CUDA(cudaMemcpyAsync(host, fq->line_off + first, count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}
