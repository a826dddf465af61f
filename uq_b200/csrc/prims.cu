// Device-wide primitives: exclusive scan and a stable LSD radix sort of (key64, aux32, val32) records.
//
// Both are HBM-bound streaming kernels.  Layout: SoA arrays, 16 items per thread, 256 threads per
// CTA (4096-item tiles) so that every warp-level access is a run of 128/256 contiguous bytes.
#include "common.cuh"

#define PR_THREADS 256
#define PR_ITEMS 16
#define PR_TILE (PR_THREADS * PR_ITEMS)

// ================================================================================================
// scan
// ================================================================================================
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* total_out) {
    // exclusive scan of one value per thread across a 256-thread CTA
    __shared__ T warp_tot[PR_THREADS / 32];
    unsigned lane = lane_id(), w = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    T wbase = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < PR_THREADS / 32; i++) {
        T t = warp_tot[i];
        if ((unsigned)i < w) wbase += t;
        tot += t;
    }
    __syncthreads();
    if (total_out) *total_out = tot;
    return wbase + incl - v;
}

template <typename Tout>
__global__ void __launch_bounds__(PR_THREADS) k_scan_reduce(const uint32_t* __restrict__ in, uint64_t n, Tout* __restrict__ block_sums) {
    uint64_t base = (uint64_t)blockIdx.x * PR_TILE + (uint64_t)threadIdx.x * PR_ITEMS;
    Tout s = 0;
    if (base + PR_ITEMS <= n) {
        const uint4* p = reinterpret_cast<const uint4*>(in + base);
#pragma unroll
        for (int i = 0; i < PR_ITEMS / 4; i++) {
            uint4 q = __ldg(p + i);
            s += (Tout)q.x + (Tout)q.y + (Tout)q.z + (Tout)q.w;
        }
    } else {
        for (int i = 0; i < PR_ITEMS; i++)
            if (base + i < n) s += (Tout)in[base + i];
    }
    Tout tot;
    block_exclusive_scan<Tout>(s, &tot);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}

template <typename Tout>
__global__ void __launch_bounds__(1024) k_scan_block_sums(Tout* __restrict__ sums, uint64_t nblocks, Tout* __restrict__ total) {
    // single CTA: exclusive scan of the per-tile sums, 1024 at a time with a running carry
    __shared__ Tout warp_tot[32];
    __shared__ Tout carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    unsigned lane = lane_id(), w = threadIdx.x >> 5;
    for (uint64_t start = 0; start < nblocks; start += 1024) {
        uint64_t i = start + threadIdx.x;
        Tout v = i < nblocks ? sums[i] : (Tout)0;
        Tout incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            Tout t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += t;
        }
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        Tout wbase = 0, tot = 0;
        for (int k = 0; k < 32; k++) {
            Tout t = warp_tot[k];
            if ((unsigned)k < w) wbase += t;
            tot += t;
        }
        Tout carry = carry_s;
        if (i < nblocks) sums[i] = carry + wbase + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total) *total = carry_s;
}

template <typename Tout>
__global__ void __launch_bounds__(PR_THREADS) k_scan_apply(const uint32_t* in, Tout* out, uint64_t n,
                                                          const Tout* __restrict__ block_offsets) {   // in may alias out
    uint64_t base = (uint64_t)blockIdx.x * PR_TILE + (uint64_t)threadIdx.x * PR_ITEMS;
    uint32_t v[PR_ITEMS];
    Tout s = 0;
    // full threads move their 16 items as 128-bit words (the radix passes scan 256 x tiles counters forty times per encode)
    const bool full = base + PR_ITEMS <= n && ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    if (full) {
        const uint4* p = reinterpret_cast<const uint4*>(in + base);       // plain loads: `in` may alias `out`
#pragma unroll
        for (int i = 0; i < PR_ITEMS / 4; i++) {
            const uint4 q = p[i];
            v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
        }
#pragma unroll
        for (int i = 0; i < PR_ITEMS; i++) s += (Tout)v[i];
    } else {
#pragma unroll
        for (int i = 0; i < PR_ITEMS; i++) {
            v[i] = (base + i < n) ? in[base + i] : 0u;
            s += (Tout)v[i];
        }
    }
    Tout ex = block_exclusive_scan<Tout>(s, nullptr) + block_offsets[blockIdx.x];
    if (full && sizeof(Tout) == 4) {
        uint4* o = reinterpret_cast<uint4*>(out + base);
#pragma unroll
        for (int i = 0; i < PR_ITEMS / 4; i++) {
            uint4 q;
            q.x = (uint32_t)ex; ex += (Tout)v[4 * i];
            q.y = (uint32_t)ex; ex += (Tout)v[4 * i + 1];
            q.z = (uint32_t)ex; ex += (Tout)v[4 * i + 2];
            q.w = (uint32_t)ex; ex += (Tout)v[4 * i + 3];
            o[i] = q;
        }
    } else {
#pragma unroll
        for (int i = 0; i < PR_ITEMS; i++) {
            if (base + i < n) out[base + i] = ex;
            ex += (Tout)v[i];
        }
    }
}

template <typename Tout>
static int scan_impl(uqb_ctx* ctx, const uint32_t* d_in, Tout* d_out, uint64_t n, Tout* d_total) {
    if (n == 0) {
        if (d_total) UQB_CUDA(cudaMemsetAsync(d_total, 0, sizeof(Tout), ctx->stream));
        return 0;
    }
    uint64_t nblocks = (n + PR_TILE - 1) / PR_TILE;
    Tout* sums;
    UQB_TRY(uqb_dalloc_t(ctx, &sums, nblocks));
    UQB_LAUNCH_B(n * 4, k_scan_reduce<Tout>, (unsigned)nblocks, PR_THREADS, 0, d_in, n, sums);
    UQB_LAUNCH(k_scan_block_sums<Tout>, 1, 1024, 0, sums, nblocks, d_total);
    UQB_LAUNCH_B(n * (4 + sizeof(Tout)), k_scan_apply<Tout>, (unsigned)nblocks, PR_THREADS, 0, d_in, d_out, n, sums);
    UQB_TRY(uqb_dfree(ctx, sums, nblocks * sizeof(Tout)));
    return 0;
}

int uqb_scan_u32(uqb_ctx* ctx, const uint32_t* d_in, uint32_t* d_out, uint64_t n, uint32_t* d_total) {
    return scan_impl<uint32_t>(ctx, d_in, d_out, n, d_total);
}
int uqb_scan_u32_to_u64(uqb_ctx* ctx, const uint32_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total) {
    return scan_impl<unsigned long long>(ctx, d_in, (unsigned long long*)d_out, n, (unsigned long long*)d_total);
}

// ================================================================================================
// radix sort
// ================================================================================================
struct bits_summary { unsigned long long or64, and64; unsigned int or32, and32; };

__global__ void __launch_bounds__(256) k_bits_reduce(const uint64_t* __restrict__ key, const uint32_t* __restrict__ aux, uint64_t n,
                                                     bits_summary* __restrict__ out) {
    unsigned long long o64 = 0, a64 = ~0ull;
    unsigned int o32 = 0, a32 = ~0u;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long k = key[i];
        o64 |= k; a64 &= k;
        if (aux) { unsigned int a = aux[i]; o32 |= a; a32 &= a; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        o64 |= __shfl_xor_sync(0xffffffffu, o64, o);
        a64 &= __shfl_xor_sync(0xffffffffu, a64, o);
        o32 |= __shfl_xor_sync(0xffffffffu, o32, o);
        a32 &= __shfl_xor_sync(0xffffffffu, a32, o);
    }
    if (lane_id() == 0) {
        atomicOr(&out->or64, o64);
        atomicAnd(&out->and64, a64);
        atomicOr(&out->or32, o32);
        atomicAnd(&out->and32, a32);
    }
}

// Bucket of the MSD sort below: items [start, start + size) of the array; its tiles are t0 .. t0 + nt - 1 of the pass and
// the counters of its tile t are ghist[t0 * 256 + digit * nt + t] (digit-major inside the bucket, so that one exclusive scan
// of all counters yields every bucket's digit runs in order).
struct msd_bucket { uint32_t start, size, t0, nt; };

// SEG = false: tile blockIdx.x of [0, n), counters ghist[digit * nblk + tile].  SEG = true: the tile belongs to bucket
// tile_bucket[blockIdx.x] (see msd_bucket).
template <bool SEG>
struct radix_tile {
    uint64_t tile0, end;        // items [tile0, min(end, tile0 + PR_TILE))
    uint64_t hbase, hstride;    // counter of digit d: hbase + d * hstride
    uint32_t bstart, hfirst;    // SEG: first item and first counter of the bucket
    __device__ __forceinline__ radix_tile(uint64_t n, uint32_t nblk, const uint32_t* tile_bucket, const msd_bucket* buckets) {
        if (SEG) {
            const msd_bucket b = buckets[tile_bucket[blockIdx.x]];
            const uint32_t t = blockIdx.x - b.t0;
            tile0 = (uint64_t)b.start + (uint64_t)t * PR_TILE;
            end = (uint64_t)b.start + b.size;
            hbase = (uint64_t)b.t0 * 256 + t;
            hstride = b.nt;
            bstart = b.start;
            hfirst = b.t0 * 256;
        } else {
            tile0 = (uint64_t)blockIdx.x * PR_TILE;
            end = n;
            hbase = blockIdx.x;
            hstride = nblk;
            bstart = hfirst = 0;
        }
    }
};

template <bool AUXDIGIT, bool SEG = false>
__global__ void __launch_bounds__(PR_THREADS) k_radix_hist(const uint64_t* __restrict__ key, const uint32_t* __restrict__ aux, uint64_t n,
                                                          int shift, uint32_t* __restrict__ ghist, uint32_t nblk,
                                                          const uint32_t* __restrict__ tile_bucket = nullptr,
                                                          const msd_bucket* __restrict__ buckets = nullptr) {
    __shared__ uint32_t hist[256];
    hist[threadIdx.x] = 0;
    const radix_tile<SEG> T(n, nblk, tile_bucket, buckets);
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < PR_ITEMS; j++) {
        uint64_t idx = T.tile0 + (uint64_t)j * PR_THREADS + threadIdx.x;
        if (idx < T.end) {
            uint32_t d = AUXDIGIT ? ((aux[idx] >> shift) & 255u) : (uint32_t)((key[idx] >> shift) & 255ull);
            atomicAdd(&hist[d], 1u);
        }
    }
    __syncthreads();
    ghist[T.hbase + (uint64_t)threadIdx.x * T.hstride] = hist[threadIdx.x];
}

// Stable scatter.  512 threads take one tile of PR_TILE items; every warp owns 256 consecutive items and
// ranks them 32 at a time with match_any, so the order inside a digit bucket is (CTA, warp, round, lane) =
// input order.  Keys, values (and aux words) are loaded ONCE, up front, and stay in registers through the
// ranking; the tile is then re-ordered by digit in shared memory and written out as one contiguous run per
// digit, which turns 4096 scattered 8/4-byte stores into ~256 coalesced runs.
#define RS_THREADS 512
#define RS_ITEMS (PR_TILE / RS_THREADS)
#define RS_WARPS (RS_THREADS / 32)
struct rs_stage {
    uint32_t whist[RS_WARPS][256];            // per-warp digit counts, then per-warp exclusive prefix
    uint32_t dstart[256];                     // first tile-local slot of every digit
    uint32_t gbase[256];                      // first global slot of this CTA's run of every digit
    uint32_t wtot[8];
    uint64_t key[PR_TILE];
    uint32_t val[PR_TILE];
    uint32_t aux[PR_TILE];
};

// SEG: the tile and its counters come from the MSD bucket lists (radix_tile); a bucket's items are scattered inside its own
// range, goff[first counter of the bucket] being the exclusive scan up to the bucket.
template <bool AUXDIGIT, bool HASAUX, bool SEG = false>
__global__ void __launch_bounds__(RS_THREADS, 2) k_radix_scatter(const uint64_t* __restrict__ kin, const uint32_t* __restrict__ ain,
                                                                const uint32_t* __restrict__ vin, uint64_t* __restrict__ kout,
                                                                uint32_t* __restrict__ aout, uint32_t* __restrict__ vout, uint64_t n_,
                                                                int shift, const uint32_t* __restrict__ goff, uint32_t nblk,
                                                                const uint32_t* __restrict__ tile_bucket = nullptr,
                                                                const msd_bucket* __restrict__ buckets = nullptr) {
    extern __shared__ __align__(16) uint8_t rs_raw[];
    rs_stage* S = reinterpret_cast<rs_stage*>(rs_raw);
    const unsigned tid = threadIdx.x, w = tid >> 5, lane = tid & 31u;
    const radix_tile<SEG> T(n_, nblk, tile_bucket, buckets);
    const uint64_t tile0 = T.tile0, n = T.end;
    const uint64_t warp0 = tile0 + (uint64_t)w * (32 * RS_ITEMS);
    const uint32_t ntile = (uint32_t)((n - tile0 < PR_TILE) ? (n - tile0) : PR_TILE);
    uint64_t key[RS_ITEMS];
    uint32_t val[RS_ITEMS], aux[RS_ITEMS];
#pragma unroll
    for (int j = 0; j < RS_ITEMS; j++) {
        const uint64_t idx = warp0 + (uint64_t)j * 32 + lane;
        key[j] = 0; val[j] = 0; aux[j] = 0;
        if (idx < n) {
            key[j] = kin[idx];
            val[j] = vin ? vin[idx] : (uint32_t)idx;          // first pass over producer-written keys: value = row index
            if (HASAUX) aux[j] = ain[idx];
        }
    }
    for (unsigned i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&S->whist[0][0])[i] = 0;
    __syncthreads();
    uint32_t rk[RS_ITEMS];
#pragma unroll
    for (int j = 0; j < RS_ITEMS; j++) {
        const uint64_t idx = warp0 + (uint64_t)j * 32 + lane;
        const bool valid = idx < n;
        uint32_t d = 256u;    // sentinel digit for lanes beyond the end
        if (valid) d = AUXDIGIT ? ((aux[j] >> shift) & 255u) : (uint32_t)((key[j] >> shift) & 255ull);
        const unsigned m = __match_any_sync(0xffffffffu, d);
        const unsigned r = __popc(m & ((1u << lane) - 1u));
        const int leader = __ffs(m) - 1;
        uint32_t old = 0;
        if (valid && (int)lane == leader) {
            old = S->whist[w][d];
            S->whist[w][d] = old + __popc(m);
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        rk[j] = (d << 16) | (old + r);     // old + r < 256
        __syncwarp();
    }
    __syncthreads();
    // digit totals -> per-warp exclusive prefixes, tile-local digit starts (256-wide scan), global bases
    uint32_t tot = 0, incl = 0;
    if (tid < 256) {
#pragma unroll
        for (int w2 = 0; w2 < RS_WARPS; w2++) {
            const uint32_t c = S->whist[w2][tid];
            S->whist[w2][tid] = tot;
            tot += c;
        }
        incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += t;
        }
        if (lane == 31) S->wtot[w] = incl;
    }
    __syncthreads();
    if (tid < 256) {
        uint32_t wb = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) if ((unsigned)i < w) wb += S->wtot[i];
        const uint32_t start = wb + incl - tot;
        S->dstart[tid] = start;
        uint32_t g = goff[T.hbase + (uint64_t)tid * T.hstride];
        if (SEG) g += T.bstart - goff[T.hfirst];
        S->gbase[tid] = g - start;      // global slot = gbase[d] + tile-local slot
    }
    __syncthreads();
    // stage the tile in digit order
#pragma unroll
    for (int j = 0; j < RS_ITEMS; j++) {
        const uint64_t idx = warp0 + (uint64_t)j * 32 + lane;
        if (idx < n) {
            const uint32_t d = rk[j] >> 16;
            const uint32_t slot = S->dstart[d] + S->whist[w][d] + (rk[j] & 0xffffu);
            S->key[slot] = key[j];
            S->val[slot] = val[j];
            if (HASAUX) S->aux[slot] = aux[j];
        }
    }
    __syncthreads();
    // contiguous runs out
    for (uint32_t i = tid; i < ntile; i += RS_THREADS) {
        const uint64_t k = S->key[i];
        const uint32_t a = HASAUX ? S->aux[i] : 0u;
        const uint32_t d = AUXDIGIT ? ((a >> shift) & 255u) : (uint32_t)((k >> shift) & 255ull);
        const uint32_t pos = S->gbase[d] + i;
        kout[pos] = k;
        if (HASAUX) aout[pos] = a;
        vout[pos] = S->val[i];
    }
}

// ---- out[idx[p]] = val[p] for arrays much larger than the L2 --------------------------------------
// A plain scatter of 4-byte items over 400 MB costs a sector fill and a write-back per element.  Here the (idx, val) pairs
// are first grouped by destination WINDOW (idx >> wshift: 32 MB of `out` per window) with one counting pass and one
// regrouping pass (tile-local order inside a window is free: idx is a permutation, no two pairs meet), then applied in
// that order: the stores of a window meet in the L2 and leave as full lines.  Three sequential sweeps over 8 bytes per
// pair instead of one sweep per window.
#define PW_THREADS 512
#define PW_ITEMS (PR_TILE / PW_THREADS)

__global__ void __launch_bounds__(PW_THREADS) k_pairs_hist(const uint32_t* __restrict__ idx, uint64_t n, uint32_t wshift, uint32_t nwin,
                                                          uint32_t* __restrict__ ghist, uint32_t nblk) {
    __shared__ uint32_t hist[256];
    if (threadIdx.x < 256) hist[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t tile0 = (uint64_t)blockIdx.x * PR_TILE;
#pragma unroll
    for (int j = 0; j < PW_ITEMS; j++) {
        const uint64_t i = tile0 + (uint64_t)j * PW_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&hist[__ldg(idx + i) >> wshift], 1u);
    }
    __syncthreads();
    if (threadIdx.x < nwin) ghist[(uint64_t)threadIdx.x * nblk + blockIdx.x] = hist[threadIdx.x];
}

struct pw_stage {
    uint32_t cnt[256], dstart[256], gbase[256], wtot[8];
    uint32_t idx[PR_TILE], val[PR_TILE];
};

__global__ void __launch_bounds__(PW_THREADS) k_pairs_regroup(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ val, uint64_t n,
                                                             uint32_t wshift, uint32_t nwin, const uint32_t* __restrict__ goff, uint32_t nblk,
                                                             uint32_t* __restrict__ idx_out, uint32_t* __restrict__ val_out) {
    extern __shared__ __align__(16) uint8_t pw_raw[];
    pw_stage* S = reinterpret_cast<pw_stage*>(pw_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    if (tid < 256) S->cnt[tid] = 0;
    __syncthreads();
    const uint64_t tile0 = (uint64_t)blockIdx.x * PR_TILE;
    const uint32_t ntile = (uint32_t)((n - tile0 < PR_TILE) ? (n - tile0) : PR_TILE);
    uint32_t ix[PW_ITEMS], vx[PW_ITEMS], rk[PW_ITEMS];
#pragma unroll
    for (int j = 0; j < PW_ITEMS; j++) {
        const uint64_t i = tile0 + (uint64_t)j * PW_THREADS + tid;
        ix[j] = 0; vx[j] = 0; rk[j] = 0;
        if (i < n) { ix[j] = __ldg(idx + i); vx[j] = __ldg(val + i); }
    }
#pragma unroll
    for (int j = 0; j < PW_ITEMS; j++) {
        const uint64_t i = tile0 + (uint64_t)j * PW_THREADS + tid;
        // warp-aggregated: the lanes of one window take consecutive places behind one shared-memory atomic
        const uint32_t d = i < n ? (ix[j] >> wshift) : 0xFFFFFFFFu;
        const unsigned m = __match_any_sync(0xffffffffu, d);
        const int leader = __ffs(m) - 1;
        uint32_t base = 0;
        if (i < n && (int)lane == leader) base = atomicAdd(&S->cnt[d], (uint32_t)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        rk[j] = base + __popc(m & ((1u << lane) - 1u));
    }
    __syncthreads();
    uint32_t tot = 0, incl = 0;
    if (tid < 256) {
        tot = tid < nwin ? S->cnt[tid] : 0u;
        incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += t;
        }
        if (lane == 31) S->wtot[w] = incl;
    }
    __syncthreads();
    if (tid < 256) {
        uint32_t wb = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) if ((unsigned)i < w) wb += S->wtot[i];
        const uint32_t start = wb + incl - tot;
        S->dstart[tid] = start;
        if (tid < nwin) S->gbase[tid] = goff[(uint64_t)tid * nblk + blockIdx.x] - start;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PW_ITEMS; j++) {
        const uint64_t i = tile0 + (uint64_t)j * PW_THREADS + tid;
        if (i < n) {
            const uint32_t slot = S->dstart[ix[j] >> wshift] + rk[j];
            S->idx[slot] = ix[j];
            S->val[slot] = vx[j];
        }
    }
    __syncthreads();
    for (uint32_t i = tid; i < ntile; i += PW_THREADS) {
        const uint32_t x = S->idx[i];
        const uint32_t pos = S->gbase[x >> wshift] + i;
        idx_out[pos] = x;
        val_out[pos] = S->val[i];
    }
}

__global__ void __launch_bounds__(256) k_pairs_apply(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ val, uint64_t n,
                                                    uint32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * 256 * 4;
    for (uint64_t p0 = ((uint64_t)blockIdx.x * 256 + threadIdx.x) * 4; p0 < n; p0 += stride) {
        if (p0 + 4 <= n) {
            const uint4 d = __ldg(reinterpret_cast<const uint4*>(idx + p0));
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(val + p0));
            out[d.x] = v.x; out[d.y] = v.y; out[d.z] = v.z; out[d.w] = v.w;
        } else {
            for (uint64_t p = p0; p < n; p++) out[idx[p]] = val[p];
        }
    }
}

// out[idx[p]] = val[p]; idx must be a permutation of 0..n-1 (n < 2^32).  Small arrays are scattered directly.
int uqb_scatter_pairs_u32(uqb_ctx* ctx, const uint32_t* idx, const uint32_t* val, uint64_t n, uint32_t* out) {
    if (n == 0) return 0;
    uint32_t wshift = 23;                                          // 2^23 entries = 32 MB of `out` per window
    while (((n + (1ull << wshift) - 1) >> wshift) > 256) wshift++;
    const uint32_t nwin = (uint32_t)((n + (1ull << wshift) - 1) >> wshift);
    const uint32_t nblk = (uint32_t)((n + PR_TILE - 1) / PR_TILE);
    uint32_t *ghist, *idx2, *val2;
    const uint64_t hist_n = (uint64_t)nwin * nblk;
    UQB_TRY(uqb_dalloc_t(ctx, &ghist, hist_n));
    UQB_TRY(uqb_dalloc_t(ctx, &idx2, n + 16));
    UQB_TRY(uqb_dalloc_t(ctx, &val2, n + 16));
    UQB_LAUNCH_B(n * 4, k_pairs_hist, nblk, PW_THREADS, 0, idx, n, wshift, nwin, ghist, nblk);
    UQB_TRY(uqb_scan_u32(ctx, ghist, ghist, hist_n, nullptr));
    UQB_CUDA(cudaFuncSetAttribute(k_pairs_regroup, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(pw_stage)));
    UQB_LAUNCH_B(n * 16, k_pairs_regroup, nblk, PW_THREADS, sizeof(pw_stage), idx, val, n, wshift, nwin, ghist, nblk, idx2, val2);
    UQB_LAUNCH_B(n * 12, k_pairs_apply, uqb_grid(ctx, n, 256 * 4, 4), 256, 0, idx2, val2, n, out);
    UQB_TRY(uqb_dfree(ctx, ghist, 0));
    UQB_TRY(uqb_dfree(ctx, idx2, 0));
    UQB_TRY(uqb_dfree(ctx, val2, 0));
    return 0;
}

int uqb_sortbuf_alloc(uqb_ctx* ctx, uqb_sortbuf* sb, uint64_t n, bool with_aux) {
    sb->cap = n;
    sb->cur = 0;
    for (int i = 0; i < 2; i++) {
        UQB_TRY(uqb_dalloc_t(ctx, &sb->key[i], n));
        UQB_TRY(uqb_dalloc_t(ctx, &sb->val[i], n + 16));          // slack: uqb_sort_rows hands the sorted values out as an array
        if (with_aux) UQB_TRY(uqb_dalloc_t(ctx, &sb->aux[i], n));
    }
    return 0;
}

int uqb_sortbuf_free(uqb_ctx* ctx, uqb_sortbuf* sb) {
    for (int i = 0; i < 2; i++) {
        UQB_TRY(uqb_dfree(ctx, sb->key[i], sb->cap * 8)); sb->key[i] = nullptr;
        UQB_TRY(uqb_dfree(ctx, sb->val[i], sb->cap * 4)); sb->val[i] = nullptr;
        if (sb->aux[i]) { UQB_TRY(uqb_dfree(ctx, sb->aux[i], sb->cap * 4)); sb->aux[i] = nullptr; }
    }
    return 0;
}

// digit windows: 8-bit windows that start at the lowest still-uncovered varying bit
static int plan_windows(uint64_t varying, int nbits, int* shifts) {
    int cnt = 0;
    int b = 0;
    while (b < nbits) {
        if ((varying >> b) & 1ull) {
            shifts[cnt++] = b;
            b += 8;
        } else {
            b++;
        }
    }
    return cnt;
}

__global__ void __launch_bounds__(256) k_key_iota(const uint64_t* __restrict__ kin, uint64_t* __restrict__ kout, uint32_t* __restrict__ vout, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) { kout[i] = kin[i]; vout[i] = (uint32_t)i; }
}

// ---- MSD sort of large key-only inputs ----------------------------------------------------------------------------
// Round 0 of a row sort is a stable sort of 100 M (key64, row index) records.  LSD needs one global pass per varying byte
// (8 for packed DNA / QUAL rows); here each global pass splits every still-large bucket by its next 8 varying bits
// (k_radix_hist / k_radix_scatter in their SEG form, each tile inside one bucket), and a bucket - or a run of
// consecutive small buckets - of at most PR_TILE items is finished by one CTA in shared memory (k_bucket_sort: stable LSD
// over the bits that vary inside it).  Uniform keys take 2 global passes and one read/write sweep; skewed keys
// (quality strings) keep splitting only their large buckets.  Every step is stable, so the result is the stable sort.
#define MSD_MIN_N (1u << 20)          // smaller sorts keep the LSD passes (not tuned: the bench sorts 100 M keys)

struct msd_counts { uint32_t nseg, nbuck, ntiles, pad; };

struct bs_stage {
    uint32_t whist[RS_WARPS][256];
    uint32_t dstart[256];
    uint32_t wtot[8];
    unsigned long long or64, and64;
    uint64_t key[PR_TILE];
    uint32_t val[PR_TILE];
};

// one segment (start, size <= PR_TILE) per CTA: load, stable LSD on the segment's varying bits in shared memory, store
__global__ void __launch_bounds__(RS_THREADS, 2) k_bucket_sort(const uint64_t* __restrict__ kin, const uint32_t* __restrict__ vin,
                                                              uint64_t* __restrict__ kout, uint32_t* __restrict__ vout,
                                                              const uint2* __restrict__ segs) {
    extern __shared__ __align__(16) uint8_t bs_raw[];
    bs_stage* S = reinterpret_cast<bs_stage*>(bs_raw);
    const unsigned tid = threadIdx.x, w = tid >> 5, lane = tid & 31u;
    const uint2 seg = segs[blockIdx.x];
    const uint64_t base = seg.x;
    const uint32_t m = seg.y;
    if (tid == 0) { S->or64 = 0ull; S->and64 = ~0ull; }
    __syncthreads();
    unsigned long long o64 = 0ull, a64 = ~0ull;
    for (uint32_t i = tid; i < m; i += RS_THREADS) {
        const uint64_t k = kin[base + i];
        S->key[i] = k;
        S->val[i] = vin[base + i];
        o64 |= k; a64 &= k;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        o64 |= __shfl_xor_sync(0xffffffffu, o64, o);
        a64 &= __shfl_xor_sync(0xffffffffu, a64, o);
    }
    if (lane == 0) { atomicOr(&S->or64, o64); atomicAnd(&S->and64, a64); }
    __syncthreads();
    uint64_t vary = S->or64 ^ S->and64;
    while (vary) {                                   // 8-bit windows from the lowest varying bit up (plan_windows)
        const int shift = __ffsll((long long)vary) - 1;
        vary = shift + 8 >= 64 ? 0ull : vary & (~0ull << (shift + 8));
        uint64_t key[RS_ITEMS];
        uint32_t val[RS_ITEMS], rk[RS_ITEMS];
#pragma unroll
        for (int j = 0; j < RS_ITEMS; j++) {
            const uint32_t i = w * (32 * RS_ITEMS) + j * 32 + lane;
            key[j] = i < m ? S->key[i] : 0ull;
            val[j] = i < m ? S->val[i] : 0u;
        }
        for (unsigned i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&S->whist[0][0])[i] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < RS_ITEMS; j++) {
            const uint32_t i = w * (32 * RS_ITEMS) + j * 32 + lane;
            const bool valid = i < m;
            const uint32_t d = valid ? (uint32_t)((key[j] >> shift) & 255ull) : 256u;
            const unsigned mm = __match_any_sync(0xffffffffu, d);
            const unsigned r = __popc(mm & ((1u << lane) - 1u));
            const int leader = __ffs(mm) - 1;
            uint32_t old = 0;
            if (valid && (int)lane == leader) {
                old = S->whist[w][d];
                S->whist[w][d] = old + __popc(mm);
            }
            old = __shfl_sync(0xffffffffu, old, leader);
            rk[j] = (d << 16) | (old + r);
            __syncwarp();
        }
        __syncthreads();
        uint32_t tot = 0, incl = 0;
        if (tid < 256) {
#pragma unroll
            for (int w2 = 0; w2 < RS_WARPS; w2++) {
                const uint32_t c = S->whist[w2][tid];
                S->whist[w2][tid] = tot;
                tot += c;
            }
            incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (unsigned)o) incl += t;
            }
            if (lane == 31) S->wtot[w] = incl;
        }
        __syncthreads();
        if (tid < 256) {
            uint32_t wb = 0;
#pragma unroll
            for (int i = 0; i < 8; i++) if ((unsigned)i < w) wb += S->wtot[i];
            S->dstart[tid] = wb + incl - tot;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < RS_ITEMS; j++) {
            const uint32_t i = w * (32 * RS_ITEMS) + j * 32 + lane;
            if (i < m) {
                const uint32_t d = rk[j] >> 16;
                const uint32_t slot = S->dstart[d] + S->whist[w][d] + (rk[j] & 0xffffu);
                S->key[slot] = key[j];
                S->val[slot] = val[j];
            }
        }
        __syncthreads();
    }
    for (uint32_t i = tid; i < m; i += RS_THREADS) {
        kout[base + i] = S->key[i];
        vout[base + i] = S->val[i];
    }
}

// One CTA per bucket split by the pass just made: its 256 digit runs (from the scanned counters) are packed greedily, in
// order, into segments of at most PR_TILE items for k_bucket_sort; larger runs become the buckets of the next pass, with
// their tiles.  last: no varying bit is left below the digit, every run is a run of equal keys, cut into segments (copies).
__global__ void __launch_bounds__(256) k_msd_plan(const uint32_t* __restrict__ goff, const msd_bucket* __restrict__ buckets, int last,
                                                 msd_counts* __restrict__ cnt, uint2* __restrict__ segs, msd_bucket* __restrict__ next,
                                                 uint32_t* __restrict__ next_tile_bucket) {
    __shared__ uint32_t st[257];
    __shared__ uint2 lseg[256], lover[256];
    __shared__ uint32_t nls, nlo, sbase, obase, t0s;
    const unsigned tid = threadIdx.x;
    const msd_bucket b = buckets[blockIdx.x];
    const uint64_t h0 = (uint64_t)b.t0 * 256;
    st[tid] = b.start + (goff[h0 + (uint64_t)tid * b.nt] - goff[h0]);
    if (tid == 0) st[256] = b.start + b.size;
    __syncthreads();
    if (last) {
        const uint32_t s = st[tid + 1] - st[tid], nch = (s + PR_TILE - 1) / PR_TILE;
        if (nch) {
            const uint32_t at = atomicAdd(&cnt->nseg, nch);
            for (uint32_t k = 0; k < nch; k++) segs[at + k] = make_uint2(st[tid] + k * PR_TILE, min((uint32_t)PR_TILE, s - k * PR_TILE));
        }
        return;
    }
    if (tid == 0) {
        uint32_t ns = 0, no = 0, cs = 0, cn = 0;
        for (int d = 0; d < 256; d++) {
            const uint32_t s = st[d + 1] - st[d];
            if (s == 0) continue;
            if (s > PR_TILE) {
                if (cn) { lseg[ns++] = make_uint2(cs, cn); cn = 0; }
                lover[no++] = make_uint2(st[d], s);
            } else {
                if (cn + s > PR_TILE) { lseg[ns++] = make_uint2(cs, cn); cn = 0; }
                if (cn == 0) cs = st[d];
                cn += s;
            }
        }
        if (cn) lseg[ns++] = make_uint2(cs, cn);
        nls = ns; nlo = no;
        sbase = ns ? atomicAdd(&cnt->nseg, ns) : 0u;
        obase = no ? atomicAdd(&cnt->nbuck, no) : 0u;
    }
    __syncthreads();
    for (uint32_t i = tid; i < nls; i += 256) segs[sbase + i] = lseg[i];
    for (uint32_t k = 0; k < nlo; k++) {
        const uint2 o = lover[k];
        const uint32_t nt = (o.y + PR_TILE - 1) / PR_TILE;
        if (tid == 0) {
            t0s = atomicAdd(&cnt->ntiles, nt);
            next[obase + k] = msd_bucket{o.x, o.y, t0s, nt};
        }
        __syncthreads();
        for (uint32_t t = tid; t < nt; t += 256) next_tile_bucket[t0s + t] = obase + k;
        __syncthreads();
    }
}

// highest 8-bit window below bit `below` that holds a varying bit (-1: none)
static int msd_shift(uint64_t vary, int below) {
    const uint64_t v = below >= 64 ? vary : vary & ((1ull << below) - 1);
    if (!v) return -1;
    const int hi = 63 - __builtin_clzll(v);
    return hi >= 7 ? hi - 7 : 0;
}

static int msd_sort(uqb_ctx* ctx, uqb_sortbuf* sb, uint64_t n, const uint64_t* key_first, uint64_t vary) {
    const uint32_t nblk = (uint32_t)((n + PR_TILE - 1) / PR_TILE);
    const uint64_t cap_b = n / PR_TILE + 1, cap_t = nblk + cap_b;     // every bucket of a later pass holds > PR_TILE items
    const int fin = sb->cur ^ 1;                                       // k_bucket_sort writes every segment here
    msd_bucket* bk[2];
    uint32_t* tb[2];
    msd_counts* cnt;
    UQB_TRY(uqb_dalloc_t(ctx, &bk[0], cap_b));
    UQB_TRY(uqb_dalloc_t(ctx, &bk[1], cap_b));
    UQB_TRY(uqb_dalloc_t(ctx, &tb[0], cap_t));
    UQB_TRY(uqb_dalloc_t(ctx, &tb[1], cap_t));
    UQB_TRY(uqb_dalloc_t(ctx, &cnt, 1));
    const msd_bucket all = {0u, (uint32_t)n, 0u, nblk};
    UQB_CUDA(cudaMemcpyAsync(bk[0], &all, sizeof(all), cudaMemcpyHostToDevice, ctx->stream));
    UQB_CUDA(cudaMemsetAsync(tb[0], 0, (uint64_t)nblk * 4, ctx->stream));
    auto k_radix_hist_seg = k_radix_hist<false, true>;
    auto k_radix_scatter_seg = k_radix_scatter<false, false, true>;
    UQB_CUDA(cudaFuncSetAttribute(k_radix_scatter_seg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(rs_stage)));
    UQB_CUDA(cudaFuncSetAttribute(k_bucket_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(bs_stage)));
    uint32_t nbuck = 1, ntiles = nblk;
    uint64_t items = n;
    int c = sb->cur, shift = msd_shift(vary, 64), lv = 0;
    while (nbuck) {
        const int o = c ^ 1, nxt = msd_shift(vary, shift);
        const uint64_t* kin = (lv == 0 && key_first) ? key_first : sb->key[c];
        const uint32_t* vin = (lv == 0 && key_first) ? nullptr : sb->val[c];
        uint32_t* ghist;
        const uint64_t hist_n = (uint64_t)256 * ntiles;
        UQB_TRY(uqb_dalloc_t(ctx, &ghist, hist_n));
        UQB_LAUNCH_B((uint64_t)items * 8, k_radix_hist_seg, ntiles, PR_THREADS, 0, kin, nullptr, n, shift, ghist, 0u, tb[lv & 1], bk[lv & 1]);
        UQB_TRY(uqb_scan_u32(ctx, ghist, ghist, hist_n, nullptr));
        UQB_LAUNCH_B((uint64_t)items * 24, k_radix_scatter_seg, ntiles, RS_THREADS, sizeof(rs_stage), kin, nullptr, vin, sb->key[o], nullptr,
                     sb->val[o], n, shift, ghist, 0u, tb[lv & 1], bk[lv & 1]);
        uint2* segs;
        const uint64_t cap_s = (uint64_t)256 * nbuck + n / PR_TILE + 1;
        UQB_TRY(uqb_dalloc_t(ctx, &segs, cap_s));
        UQB_CUDA(cudaMemsetAsync(cnt, 0, sizeof(msd_counts), ctx->stream));
        UQB_LAUNCH(k_msd_plan, nbuck, 256, 0, ghist, bk[lv & 1], nxt < 0 ? 1 : 0, cnt, segs, bk[(lv + 1) & 1], tb[(lv + 1) & 1]);
        msd_counts got;
        UQB_TRY(uqb_readback(ctx, &got, cnt, sizeof(got)));
        if (got.nseg) UQB_LAUNCH_B(0, k_bucket_sort, got.nseg, RS_THREADS, sizeof(bs_stage), sb->key[o], sb->val[o], sb->key[fin], sb->val[fin], segs);
        UQB_TRY(uqb_dfree(ctx, segs, cap_s * 8));
        UQB_TRY(uqb_dfree(ctx, ghist, hist_n * 4));
        nbuck = got.nbuck;
        ntiles = got.ntiles;
        items = (uint64_t)ntiles * PR_TILE;                // upper bound, for the byte count only
        c = o;
        shift = nxt;
        lv++;
    }
    sb->cur = fin;
    UQB_TRY(uqb_dfree(ctx, bk[0], cap_b * sizeof(msd_bucket)));
    UQB_TRY(uqb_dfree(ctx, bk[1], cap_b * sizeof(msd_bucket)));
    UQB_TRY(uqb_dfree(ctx, tb[0], cap_t * 4));
    UQB_TRY(uqb_dfree(ctx, tb[1], cap_t * 4));
    UQB_TRY(uqb_dfree(ctx, cnt, sizeof(msd_counts)));
    return 0;
}

int uqb_radix_sort(uqb_ctx* ctx, uqb_sortbuf* sb, uint64_t n, bool use_aux, const uint64_t* key_first) {
    if (key_first && (use_aux || n < 2)) {            // plain path: materialise (key, index) in buffer 0
        if (n) UQB_LAUNCH_B(n * 20, k_key_iota, uqb_grid(ctx, n, 256 * 8), 256, 0, key_first, sb->key[sb->cur], sb->val[sb->cur], n);
        key_first = nullptr;
    }
    if (n < 2) return 0;
    if (n >= (1ull << 32)) return uqb_fail(ctx, "radix sort: %llu items exceed the 32-bit index range", (unsigned long long)n);
    bits_summary init = {0ull, ~0ull, 0u, ~0u}, got;
    bits_summary* d_bits;
    UQB_TRY(uqb_dalloc_t(ctx, &d_bits, 1));
    UQB_CUDA(cudaMemcpyAsync(d_bits, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    UQB_LAUNCH_B(n * (use_aux ? 12 : 8), k_bits_reduce, uqb_grid(ctx, n, 256 * 8), 256, 0, key_first ? key_first : sb->key[sb->cur], use_aux ? sb->aux[sb->cur] : nullptr, n, d_bits);
    UQB_TRY(uqb_readback(ctx, &got, d_bits, sizeof(got)));
    UQB_TRY(uqb_dfree(ctx, d_bits, sizeof(bits_summary)));

    int kshift[16], ashift[8];
    int nk = plan_windows(got.or64 ^ got.and64, 64, kshift);
    int na = use_aux ? plan_windows((uint64_t)(got.or32 ^ got.and32), 32, ashift) : 0;
    if (nk + na == 0) {
        if (key_first) UQB_LAUNCH_B(n * 20, k_key_iota, uqb_grid(ctx, n, 256 * 8), 256, 0, key_first, sb->key[sb->cur], sb->val[sb->cur], n);
        return 0;
    }

    const bool has_aux = sb->aux[0] != nullptr;
    if (!use_aux && !has_aux && n >= MSD_MIN_N && nk >= 3) return msd_sort(ctx, sb, n, key_first, got.or64 ^ got.and64);
    uint32_t nblk = (uint32_t)((n + PR_TILE - 1) / PR_TILE);
    uint32_t* ghist;
    uint64_t hist_n = (uint64_t)256 * nblk;
    UQB_TRY(uqb_dalloc_t(ctx, &ghist, hist_n));
    for (int p = 0; p < nk + na; p++) {
        bool auxd = p >= nk;
        int shift = auxd ? ashift[p - nk] : kshift[p];
        int c = sb->cur, o = c ^ 1;
        const uint64_t* kin = (p == 0 && key_first) ? key_first : sb->key[c];
        const uint32_t* vin = (p == 0 && key_first) ? nullptr : sb->val[c];
        if (auxd) UQB_LAUNCH_B(n * 4, k_radix_hist<true>, nblk, PR_THREADS, 0, kin, sb->aux[c], n, shift, ghist, nblk);
        else      UQB_LAUNCH_B(n * 8, k_radix_hist<false>, nblk, PR_THREADS, 0, kin, sb->aux[c], n, shift, ghist, nblk);
        UQB_TRY(uqb_scan_u32(ctx, ghist, ghist, hist_n, nullptr));
        auto k_radix_scatter_aux = k_radix_scatter<true, true>;
        auto k_radix_scatter_key_aux = k_radix_scatter<false, true>;
        auto k_radix_scatter_key = k_radix_scatter<false, false>;
        const size_t rs_smem = sizeof(rs_stage);
        UQB_CUDA(cudaFuncSetAttribute(k_radix_scatter_aux, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem));
        UQB_CUDA(cudaFuncSetAttribute(k_radix_scatter_key_aux, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem));
        UQB_CUDA(cudaFuncSetAttribute(k_radix_scatter_key, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem));
        if (auxd)         UQB_LAUNCH_B(n * 32, k_radix_scatter_aux, nblk, RS_THREADS, rs_smem, kin, sb->aux[c], vin, sb->key[o], sb->aux[o], sb->val[o], n, shift, ghist, nblk, nullptr, nullptr);
        else if (has_aux) UQB_LAUNCH_B(n * 32, k_radix_scatter_key_aux, nblk, RS_THREADS, rs_smem, kin, sb->aux[c], vin, sb->key[o], sb->aux[o], sb->val[o], n, shift, ghist, nblk, nullptr, nullptr);
        else              UQB_LAUNCH_B(n * 24, k_radix_scatter_key, nblk, RS_THREADS, rs_smem, kin, sb->aux[c], vin, sb->key[o], sb->aux[o], sb->val[o], n, shift, ghist, nblk, nullptr, nullptr);
        sb->cur = o;
    }
    UQB_TRY(uqb_dfree(ctx, ghist, hist_n * 4));
    return 0;
}
