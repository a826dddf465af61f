// Record tiles: the common front end of the record-oriented kernels (analysis, pack).
//
// A CTA takes TL_R consecutive records.  Their bytes are ONE contiguous range of the FASTQ stream, so
// the whole range is brought into shared memory by a single TMA bulk copy (cp.async.bulk, SASS UBLKCP)
// whose completion is signalled on an mbarrier, while the other threads convert the tile's line
// offsets into 32-bit smem-relative offsets.  All further accesses are shared-memory accesses: the
// unaligned, byte-granular record structure never touches L1/L2 again.
//
// The copy preserves the 16-byte phase of the global address (smem byte k holds global byte a0 + k
// with a0 = b0 & ~15), so that bulk-copy alignment rules are met without touching the data.
#pragma once
#include "common.cuh"

#define TL_R 128                    // records per tile
#define TL_CAP (48 * 1024)          // staged FASTQ bytes per tile (128 records of up to ~380 bytes)

struct tile_smem {
    alignas(128) uint8_t bytes[TL_CAP + 32];
    uint32_t loff[4 * TL_R + 4];    // line offsets relative to a0
    alignas(8) uint64_t bar;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// explicit shared-space accesses on 32-bit addresses: the hot loops of the tile kernels index the staged
// bytes and their private counters with these instead of generic pointers (no generic->shared window
// arithmetic per access).
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds_u64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8m(uint32_t a) {        // with memory clobber: the private counters are read back
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned phase) {
    unsigned ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(phase)
                     : "memory");
    } while (!ok);
}

// One-time set-up per CTA (call before the tile loop, followed by __syncthreads()).
__device__ __forceinline__ void tile_init(tile_smem* T) {
    if (threadIdx.x == 0) {
        mbar_init(&T->bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
}

// Loads records [r0, r1) into T.  Returns the number of records, or 0 when the tile does not fit TL_CAP
// (the caller reports it; the host then uses the direct-from-global kernels).  `phase` is the mbarrier
// parity of this use (0, 1, 0, ... per CTA).  Must be called by every thread of the CTA; ends with a
// __syncthreads().
__device__ __forceinline__ uint32_t tile_load(tile_smem* T, const uint8_t* __restrict__ d, uint64_t n_bytes,
                                              const uint64_t* __restrict__ line_off, uint64_t r0, uint64_t r1, unsigned phase,
                                              uint64_t* a0_out) {
    __syncthreads();                                     // every thread is done with the previous tile
    const uint32_t nrec = (uint32_t)(r1 - r0);
    const uint64_t b0 = line_off[4 * r0], b1 = line_off[4 * r1];
    const uint64_t a0 = b0 & ~15ull;
    *a0_out = a0;
    if (b1 - a0 > TL_CAP) return 0;
    uint64_t a1 = (b1 + 15) & ~15ull;                    // bulk copies move multiples of 16 bytes
    const uint64_t lim = n_bytes & ~15ull;               // never read past the last full 16-byte unit of the buffer
    if (a1 > lim) a1 = lim;
    if (a1 < a0) a1 = a0;
    const uint32_t bulk = (uint32_t)(a1 - a0);
    if (threadIdx.x == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // earlier generic reads of the buffer are done
        mbar_expect_tx(&T->bar, bulk);
        if (bulk) bulk_g2s(T->bytes, d + a0, bulk, &T->bar);
    }
    for (uint32_t i = threadIdx.x; i <= 4 * nrec; i += blockDim.x) T->loff[i] = (uint32_t)(line_off[4 * r0 + i] - a0);
    // tail of the stream that is not a full 16-byte unit
    for (uint64_t q = a1 + threadIdx.x; q < b1; q += blockDim.x) T->bytes[q - a0] = d[q];
    mbar_wait(&T->bar, phase);
    __syncthreads();
    return nrec;
}
