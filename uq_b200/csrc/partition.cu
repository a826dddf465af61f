// Multi-GPU sample sort, streaming partition (SURVEY section 8e): rows leave for the rank whose key range holds their first
// 8 bytes, so rows that agree in those bytes (identical rows in particular) meet on one rank, and the ranks' ranges are
// ordered like the rows: each rank sorts / uniques what it receives on its own.  A stable radix pass over (destination,
// index) followed by a gather of table[order] segment by segment would read every W-th row of the table per segment, i.e.
// whole 128-byte lines for a 113-byte row.  Here the table is read ONCE, sequentially, and written as W sequential streams:
//   k_pp_count   destination of every row (from the round-0 sort keys the packer wrote, or from the row) + per-tile counts
//   k_pp_scan    per destination: exclusive scan of the tile counts, totals
//   k_pp_pos     pos[i] = index of row i in the destination-grouped, stable order (first[d] + rows of d before i)
//   k_scatter_rows_runs / k_scatter_items_by_pos   row i -> byte offset seg_off[d] + (pos[i] - first[d]) * width of a byte
//                buffer whose segments start at multiples of `align` bytes (what the exchange sends); the tile of rows is
//                staged in shared memory with 16-byte loads and leaves in one contiguous run per destination.
// The same pos moves every per-record payload of global_order, and brings the global ids back with a gather.
#include "common.cuh"

#define PP_THREADS 256
#define PP_TILE 2048
#define PP_MAXW 64                       // destinations (ranks)
struct pp_split { uint64_t key[PP_MAXW]; uint32_t n; };
struct pp_segs { uint64_t first[PP_MAXW + 1]; uint64_t off[PP_MAXW]; uint32_t n; };   // first row index / byte offset per segment

__global__ void __launch_bounds__(PP_THREADS) k_pp_count(const uint8_t* __restrict__ rows, const uint64_t* __restrict__ key0, uint64_t n,
                                                         uint32_t width, pp_split sp, uint8_t* __restrict__ dest,
                                                         uint32_t* __restrict__ tile_counts, uint32_t ntiles) {
    __shared__ unsigned int cnt[PP_MAXW];
    if (threadIdx.x < PP_MAXW) cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t tile0 = (uint64_t)blockIdx.x * PP_TILE;
#pragma unroll 4
    for (int j = 0; j < PP_TILE / PP_THREADS; j++) {
        const uint64_t i = tile0 + (uint64_t)j * PP_THREADS + threadIdx.x;
        if (i < n) {
            const uint64_t k = key0 ? key0[i] : load_be64(rows + i * width, width < 8 ? width : 8);
            uint32_t d = 0;
            for (uint32_t s = 0; s < sp.n; s++) d += sp.key[s] <= k ? 1u : 0u;
            dest[i] = (uint8_t)d;
            atomicAdd(&cnt[d], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x <= sp.n) tile_counts[(uint64_t)threadIdx.x * ntiles + blockIdx.x] = cnt[threadIdx.x];
}

// one CTA per destination: exclusive scan of its tile counts in place, total -> totals[d]
__global__ void __launch_bounds__(1024) k_pp_scan(uint32_t* __restrict__ tile_counts, uint32_t ntiles, unsigned long long* __restrict__ totals) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry_s;
    uint32_t* c = tile_counts + (uint64_t)blockIdx.x * ntiles;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    for (uint32_t start = 0; start < ntiles; start += 1024) {
        const uint32_t i = start + threadIdx.x;
        const uint32_t v = i < ntiles ? c[i] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += t;
        }
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        uint32_t wbase = 0, tot = 0;
        for (int k = 0; k < 32; k++) {
            const uint32_t t = warp_tot[k];
            if ((unsigned)k < w) wbase += t;
            tot += t;
        }
        const uint32_t carry = carry_s;
        if (i < ntiles) c[i] = carry + wbase + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = carry_s;
}

// pos[i] = first[d] + (rows of destination d before row i); rows are ranked in index order, so the order inside a
// destination is the input order (stable)
__global__ void __launch_bounds__(PP_THREADS) k_pp_pos(const uint8_t* __restrict__ dest, uint64_t n, const uint32_t* __restrict__ tile_off,
                                                       uint32_t ntiles, const unsigned long long* __restrict__ totals, uint32_t ndest,
                                                       uint32_t* __restrict__ pos) {
    __shared__ uint32_t base[PP_MAXW];
    __shared__ uint32_t wcnt[PP_THREADS / 32][PP_MAXW];
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    if (tid < ndest) {
        unsigned long long f = 0;
        for (uint32_t d = 0; d < tid; d++) f += totals[d];
        base[tid] = (uint32_t)f + tile_off[(uint64_t)tid * ntiles + blockIdx.x];
    }
    const uint64_t tile0 = (uint64_t)blockIdx.x * PP_TILE;
    for (int j = 0; j < PP_TILE / PP_THREADS; j++) {
        for (unsigned k = tid; k < (PP_THREADS / 32) * PP_MAXW; k += PP_THREADS) (&wcnt[0][0])[k] = 0;
        __syncthreads();
        const uint64_t i = tile0 + (uint64_t)j * PP_THREADS + tid;
        const bool valid = i < n;
        const uint32_t d = valid ? dest[i] : 0xFFu;
        const unsigned m = __match_any_sync(0xffffffffu, d);
        const uint32_t r = __popc(m & ((1u << lane) - 1u));
        if (valid && r == 0) wcnt[w][d] = __popc(m);
        __syncthreads();
        if (valid) {
            uint32_t before = 0;
            for (unsigned w2 = 0; w2 < w; w2++) before += wcnt[w2][d];
            pos[i] = base[d] + before + r;
        }
        __syncthreads();
        if (tid < ndest) {
            uint32_t tot = 0;
#pragma unroll
            for (unsigned w2 = 0; w2 < PP_THREADS / 32; w2++) tot += wcnt[w2][tid];
            base[tid] += tot;
        }
    }
}

extern "C" int uqb_partition_positions(uqb_ctx* ctx, const uqb_array* table, const uint64_t* split_keys_host, uint32_t nsplit,
                                       uqb_array** pos, uint64_t* counts_host) {
    if (nsplit >= PP_MAXW) return uqb_fail(ctx, "partition_positions: more than %d destinations", PP_MAXW);
    const uint64_t n = table->n;
    if (n >= (1ull << 32)) return uqb_fail(ctx, "partition_positions: %llu rows exceed the 32-bit index range", (unsigned long long)n);
    UQB_TRY(uqb_new_array(ctx, n, 4, pos));
    for (uint32_t d = 0; d <= nsplit; d++) counts_host[d] = 0;
    if (n == 0) return 0;
    pp_split sp;
    sp.n = nsplit;
    for (uint32_t j = 0; j < nsplit; j++) sp.key[j] = split_keys_host[j];
    const uint32_t ntiles = (uint32_t)((n + PP_TILE - 1) / PP_TILE), ndest = nsplit + 1;
    uint8_t* dest;
    uint32_t* tile_counts;
    unsigned long long* totals;
    UQB_TRY(uqb_dalloc(ctx, (void**)&dest, n + 16));
    UQB_TRY(uqb_dalloc_t(ctx, &tile_counts, (uint64_t)ndest * ntiles));
    UQB_TRY(uqb_dalloc_t(ctx, &totals, PP_MAXW));
    const uint64_t* key0 = table->width >= 8 ? table->key0 : nullptr;
    UQB_LAUNCH_B(n * ((key0 || table->width >= 8 ? 8 : table->width) + 1), k_pp_count, ntiles, PP_THREADS, 0, (const uint8_t*)table->d, key0, n, table->width, sp,
                 dest, tile_counts, ntiles);
    UQB_LAUNCH(k_pp_scan, ndest, 1024, 0, tile_counts, ntiles, totals);
    UQB_LAUNCH_B(n * 5, k_pp_pos, ntiles, PP_THREADS, 0, dest, n, tile_counts, ntiles, totals, ndest, (uint32_t*)(*pos)->d);
    unsigned long long hc[PP_MAXW];
    UQB_TRY(uqb_readback(ctx, hc, totals, ndest * 8));
    for (uint32_t d = 0; d < ndest; d++) counts_host[d] = hc[d];
    UQB_TRY(uqb_dfree(ctx, dest, n + 16));
    UQB_TRY(uqb_dfree(ctx, tile_counts, (uint64_t)ndest * ntiles * 4));
    UQB_TRY(uqb_dfree(ctx, totals, PP_MAXW * 8));
    return 0;
}

// ---- rows -> their place in the segmented byte buffer ---------------------------------------------
#define SR_THREADS 256
#define SR_MAXW 224                      // widest row staged (256 rows per tile in shared memory)

__device__ __forceinline__ uint32_t pp_seg_of(const pp_segs& S, uint64_t j) {
    uint32_t d = 0;
    for (uint32_t s = 1; s < S.n; s++) d += S.first[s] <= j ? 1u : 0u;
    return d;
}

// Rows -> place with CONTIGUOUS RUNS on the output side.  The rows of one tile that go to destination d are consecutive in
// d's stream (pos is stable), so the CTA first regroups the tile by destination inside shared memory - the run of d starts
// at an image offset with the same 16-byte phase as its global address - and then writes every run with aligned 16-byte
// stores (only the first / last few bytes of a run go one by one).  Rows written one at a time leave as unaligned 4-byte
// words: fine for local memory, but over NVLink (peer windows) that is a packet per sector - measured 240 GB/s against
// 770 GB/s for large aligned stores.  SUB lanes move one row into the image (32 / SUB rows per warp step): 8 lanes for
// rows of up to 32 bytes, 16 up to 64, 32 beyond.
#define SRR_MAXD 64
template <int SUB>
__global__ void __launch_bounds__(SR_THREADS) k_scatter_rows_runs(const uint8_t* __restrict__ rows, uint64_t n, uint32_t width,
                                                                 const uint32_t* __restrict__ pos, pp_segs segs, uint8_t* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t srr_smem[];                 // [input tile | output image]
    __shared__ uint32_t cnt[SRR_MAXD], minpos[SRR_MAXD], ioff[SRR_MAXD], rowdst[SR_THREADS];
    __shared__ uint64_t gaddr[SRR_MAXD];
    constexpr uint32_t NP = 32u / SUB;
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    const unsigned sg = lane / SUB, sl = lane % SUB;
    const uint32_t in_bytes = (SR_THREADS * width + 32u + 15u) & ~15u;
    uint8_t* in = srr_smem;
    uint8_t* img = srr_smem + in_bytes;
    const uint32_t* in32 = reinterpret_cast<const uint32_t*>(in);
    const uint64_t ntiles = (n + SR_THREADS - 1) / SR_THREADS;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t r0 = t * SR_THREADS;
        const uint32_t nr = (uint32_t)(n - r0 < SR_THREADS ? n - r0 : SR_THREADS);
        __syncthreads();
        if (tid < segs.n) { cnt[tid] = 0; minpos[tid] = 0xFFFFFFFFu; }
        const uint4* src = reinterpret_cast<const uint4*>(rows + r0 * width);
        const uint32_t nvec = (nr * width + 15u) / 16u;
        uint32_t j = 0, d = 0;
        if (tid < nr) { j = __ldg(pos + r0 + tid); d = pp_seg_of(segs, j); }
#pragma unroll 4
        for (uint32_t v = tid; v < nvec; v += SR_THREADS) reinterpret_cast<uint4*>(in)[v] = __ldg(src + v);
        __syncthreads();
        if (tid < nr) { atomicAdd(&cnt[d], 1u); atomicMin(&minpos[d], j); }
        __syncthreads();
        if (tid == 0) {
            uint32_t at = 0;
            for (uint32_t k = 0; k < segs.n; k++) {
                if (!cnt[k]) continue;
                const uint64_t g = segs.off[k] + (uint64_t)(minpos[k] - segs.first[k]) * width + (uint64_t)(uintptr_t)out;
                gaddr[k] = g;
                at = ((at + 15u) & ~15u) + ((uint32_t)g & 15u);          // same 16-byte phase as the global address
                ioff[k] = at;
                at += cnt[k] * width;
            }
        }
        __syncthreads();
        if (tid < nr) rowdst[tid] = ioff[d] + (j - minpos[d]) * width;
        __syncthreads();
        // rows -> image (shared to shared), NP rows per warp step
#pragma unroll 2
        for (uint32_t k = 0; k < 32; k += NP) {
            const uint32_t r = w * 32 + k + sg;
            if (r < nr) {
                uint8_t* D = img + rowdst[r];
                const uint32_t so = r * width;
                uint32_t head = (4u - (rowdst[r] & 3u)) & 3u;
                head = head < width ? head : width;
                if (sl < head) D[sl] = in[so + sl];
                const uint32_t nwords = (width - head) >> 2;
                uint32_t* Dw = reinterpret_cast<uint32_t*>(D + head);
                for (uint32_t q = sl; q < nwords; q += SUB) {
                    const uint32_t b = so + head + 4u * q;
                    Dw[q] = __funnelshift_r(in32[b >> 2], in32[(b >> 2) + 1], (b & 3u) * 8u);
                }
                const uint32_t fin = head + 4u * nwords;
                if (sl < width - fin) D[fin + sl] = in[so + fin + sl];
            }
        }
        __syncthreads();
        // image runs -> global
        for (uint32_t k = 0; k < segs.n; k++) {
            if (!cnt[k]) continue;
            const uint32_t i0 = ioff[k], i1 = i0 + cnt[k] * width;
            const uint32_t a = (i0 + 15u) & ~15u, b = i1 & ~15u;
            uint8_t* G = reinterpret_cast<uint8_t*>((uintptr_t)gaddr[k]) - i0;     // image offset x <-> G + x
            if (a <= b) {
                for (uint32_t x = a + 16u * tid; x < b; x += 16u * SR_THREADS)
                    *reinterpret_cast<uint4*>(G + x) = *reinterpret_cast<const uint4*>(img + x);
                if (tid < a - i0) G[i0 + tid] = img[i0 + tid];
                if (tid < i1 - b) G[b + tid] = img[b + tid];
            } else {
                for (uint32_t x = i0 + tid; x < i1; x += SR_THREADS) G[x] = img[x];
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(SR_THREADS) k_scatter_items_by_pos(const T* __restrict__ in, uint64_t n, const uint32_t* __restrict__ pos,
                                                                    pp_segs segs, uint8_t* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * SR_THREADS + threadIdx.x; i < n; i += (uint64_t)gridDim.x * SR_THREADS) {
        const uint64_t j = pos[i];
        const uint32_t d = pp_seg_of(segs, j);
        *reinterpret_cast<T*>(out + segs.off[d] + (j - segs.first[d]) * sizeof(T)) = in[i];
    }
}

static inline uint64_t pp_round(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// rows -> place: S.off[d] is either a byte offset into `out` or, with out == nullptr, an absolute device address
static int scatter_rows_impl(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, const pp_segs& S, uint8_t* o) {
    const uint32_t w = table->width;
    const uint64_t n = table->n;
    if (n == 0) return 0;
    if ((reinterpret_cast<uintptr_t>(table->d) & 15u) != 0) return uqb_fail(ctx, "scatter_rows: the table must be 16-byte aligned");
    const uint64_t ab = n * (2ull * w + 4);
    if (w == 4) {
        UQB_LAUNCH_B(ab, k_scatter_items_by_pos<uint32_t>, uqb_grid(ctx, n, SR_THREADS, 8), SR_THREADS, 0, (const uint32_t*)table->d, n, (const uint32_t*)pos->d, S, o);
    } else if (w == 8) {
        UQB_LAUNCH_B(ab, k_scatter_items_by_pos<uint64_t>, uqb_grid(ctx, n, SR_THREADS, 8), SR_THREADS, 0, (const uint64_t*)table->d, n, (const uint32_t*)pos->d, S, o);
    } else if (w == 2) {
        UQB_LAUNCH_B(ab, k_scatter_items_by_pos<uint16_t>, uqb_grid(ctx, n, SR_THREADS, 8), SR_THREADS, 0, (const uint16_t*)table->d, n, (const uint32_t*)pos->d, S, o);
    } else if (w == 1) {
        UQB_LAUNCH_B(ab, k_scatter_items_by_pos<uint8_t>, uqb_grid(ctx, n, SR_THREADS, 8), SR_THREADS, 0, (const uint8_t*)table->d, n, (const uint32_t*)pos->d, S, o);
    } else {
        // contiguous runs per destination, regrouped in shared memory
        const size_t in_bytes = ((size_t)SR_THREADS * w + 32 + 15) & ~(size_t)15;
        const size_t smem = in_bytes + (size_t)SR_THREADS * w + 32 * (size_t)S.n + 64;
        const unsigned per_sm = (unsigned)(200 * 1024 / (smem + 5 * 1024)) ? (unsigned)(200 * 1024 / (smem + 5 * 1024)) : 1u;
        const unsigned ctas = per_sm > 8 ? 8 : per_sm;
        const uint64_t ntiles = (n + SR_THREADS - 1) / SR_THREADS, cap = (uint64_t)ctx->sm_count * ctas;
        const unsigned grid = (unsigned)(ntiles < cap ? ntiles : cap);
        if (w <= 32) {
            auto k_scatter_rows_runs_8 = k_scatter_rows_runs<8>;
            UQB_CUDA(cudaFuncSetAttribute(k_scatter_rows_runs_8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            UQB_LAUNCH_B(ab, k_scatter_rows_runs_8, grid, SR_THREADS, smem, (const uint8_t*)table->d, n, w, (const uint32_t*)pos->d, S, o);
        } else if (w <= 64) {
            auto k_scatter_rows_runs_16 = k_scatter_rows_runs<16>;
            UQB_CUDA(cudaFuncSetAttribute(k_scatter_rows_runs_16, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            UQB_LAUNCH_B(ab, k_scatter_rows_runs_16, grid, SR_THREADS, smem, (const uint8_t*)table->d, n, w, (const uint32_t*)pos->d, S, o);
        } else {
            auto k_scatter_rows_runs_32 = k_scatter_rows_runs<32>;
            UQB_CUDA(cudaFuncSetAttribute(k_scatter_rows_runs_32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            UQB_LAUNCH_B(ab, k_scatter_rows_runs_32, grid, SR_THREADS, smem, (const uint8_t*)table->d, n, w, (const uint32_t*)pos->d, S, o);
        }
    }
    return 0;
}

static int scatter_check(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, uint32_t nseg, const char* who) {
    if (pos->width != 4 || pos->n != table->n) return uqb_fail(ctx, "%s: one uint32 position per row expected", who);
    if (nseg == 0 || nseg > PP_MAXW) return uqb_fail(ctx, "%s: 1..%d segments", who, PP_MAXW);
    if (table->width == 0 || table->width > SR_MAXW) return uqb_fail(ctx, "%s: rows of 1..%d bytes (use uqb_gather_rows_segmented for wider ones)", who, SR_MAXW);
    return 0;
}

extern "C" int uqb_scatter_rows_segmented(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, uint32_t nseg,
                                          const uint64_t* seg_counts_host, uint32_t align, uqb_array** out, uint64_t* seg_offsets_host) {
    UQB_TRY(scatter_check(ctx, table, pos, nseg, "scatter_rows_segmented"));
    if (align == 0 || (align & 15u)) return uqb_fail(ctx, "scatter_rows_segmented: alignment must be a multiple of 16");
    const uint32_t w = table->width;
    pp_segs S;
    S.n = nseg;
    uint64_t total = 0, rows = 0;
    for (uint32_t d = 0; d < nseg; d++) {
        S.first[d] = rows;
        S.off[d] = total;
        seg_offsets_host[d] = total;
        total = pp_round(total + seg_counts_host[d] * w, align);
        rows += seg_counts_host[d];
    }
    S.first[nseg] = rows;
    if (rows != table->n) return uqb_fail(ctx, "scatter_rows_segmented: the segments hold %llu rows, the table %llu",
                                          (unsigned long long)rows, (unsigned long long)table->n);
    UQB_TRY(uqb_new_array(ctx, total, 1, out));
    return scatter_rows_impl(ctx, table, pos, S, (uint8_t*)(*out)->d);
}

// The device-initiated form of the exchange: the rows of segment d are written straight to the device address dst_addrs_host[d]
// (dense, in position order) - the receive buffer of rank d, mapped into this process (peer memory over NVLink), at the
// place this rank's rows have in it.  No send buffer, no collective, no compaction on the other side; the caller brackets
// the call with its barriers.
extern "C" int uqb_scatter_rows_to(uqb_ctx* ctx, const uqb_array* table, const uqb_array* pos, uint32_t nseg,
                                   const uint64_t* seg_counts_host, const uint64_t* dst_addrs_host) {
    UQB_TRY(scatter_check(ctx, table, pos, nseg, "scatter_rows_to"));
    pp_segs S;
    S.n = nseg;
    uint64_t rows = 0;
    for (uint32_t d = 0; d < nseg; d++) {
        S.first[d] = rows;
        S.off[d] = dst_addrs_host[d];
        rows += seg_counts_host[d];
    }
    S.first[nseg] = rows;
    if (rows != table->n) return uqb_fail(ctx, "scatter_rows_to: the segments hold %llu rows, the table %llu",
                                          (unsigned long long)rows, (unsigned long long)table->n);
    return scatter_rows_impl(ctx, table, pos, S, nullptr);
}
