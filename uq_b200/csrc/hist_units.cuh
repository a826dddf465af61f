// k_pair_hist_pipe: base / quality byte histograms and "does this base always carry one single quality"
// (static_qualities, uq.py:369-375, 420-425, read at uq.py:480-494) over shared-memory record tiles, sixteen
// positions per work item.
//
// A tile is 128 records (TMA bulk copies, see the pipeline below).  The 1024 threads of the CTA are bound to the
// 256 DNA / QUAL lines of the tile: thread t owns line (t & 255) - lines 0..127 are the DNA lines, 128..255 the QUAL
// lines of records 0..127 - and walks the ALIGNED 16-byte units k = t >> 8, +4, +8, ... of that line (one
// ld.shared.v4 each; units are warp-uniform, so the masked first / last units of the lines gather in few warps).
//
// Qualities: private 8-bit counters in shared memory, one column per QUAL thread ([value - 33][512 threads], bank =
// lane: no conflicts, no atomics), bumped with byte loads / stores; a word is range-checked with SIMD-in-register
// arithmetic (33..126, anything else raises `fallback` and the host runs the generic kernel).  The columns are
// summed by the whole CTA before any counter can pass 255 (the tile-end barrier carries the vote).
//
// Bases: no memory traffic at all in the common case.  Every CTA learns up to four HINT bytes - bases that have
// already been seen with more than one quality, one per value of the 2-bit code (byte >> 1) & 3, e.g. A C T G - from
// its own first tile.  A word of four bases is validated against the hints with two byte permutes (the codes select
// the expected bytes, which must equal the word), and counted by adding its code bit planes to three packed 8-bit
// accumulators in registers (code bit 0, code bit 1, both); the four hint counts follow from them and the number of
// words.  Bytes that are not hints ("offenders": N, IUPAC codes, anything while the hints are still unknown) are
// handled one by one: count in the CTA histogram, compare the quality of that very position with the base's single
// quality so far.  They stay in the accumulators (under their code) and are subtracted at the flush.
#pragma once
#include "tile.cuh"

#define H2_THREADS 1024
#define H2_QLO 33u
#define H2_ROWS 95               // quality values 33..126, row 94 (value 127) takes the masked-out bytes of edge units
#define H2_COLS 512              // QUAL threads per CTA
#define H2_NOHINT 0x00060402u    // slot c holds a byte whose code is c + 1: nothing validates

struct h2_core {                    // CTA-wide results
    unsigned hist_b[256];
    unsigned hist_q[H2_ROWS + 1];
    int state[256];                 // per base byte: -1 unseen, 0..255 its only quality so far, 256 = several
    unsigned hints, dirty, oor, qmax;
};

__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
// bit b of the result = byte b of the 16-byte unit lies in [lo, hi) (both may lie outside 0..16)
__device__ __forceinline__ uint32_t h2_unitmask(int lo, int hi) {
    const uint32_t l = lo < 0 ? 0u : (uint32_t)lo, h = hi > 16 ? 16u : (uint32_t)hi;
    return h > l ? (((1u << h) - 1u) & ~((1u << l) - 1u)) : 0u;
}
// four mask bits -> 0xFF in the bytes whose bit is set (the partial products of the multiply do not overlap)
__device__ __forceinline__ uint32_t h2_nibble_bytes(uint32_t nib) {
    return (((nib & 15u) * 0x00204081u) & 0x01010101u) * 0xFFu;
}

__device__ __forceinline__ unsigned h2_bytesum(unsigned x) {
    const unsigned y = (x & 0x00FF00FFu) + ((x >> 8) & 0x00FF00FFu);
    return (y & 0xFFFFu) + (y >> 16);
}

// one base that is not a hint: CTA histogram + single-quality state
__device__ __forceinline__ void h2_slow_byte(h2_core* S, unsigned b, unsigned q) {
    atomicAdd(&S->hist_b[b], 1u);
    int f = S->state[b];
    if (f != (int)q && f != 256) {
        if (f < 0) {
            const int old = atomicCAS(&S->state[b], -1, (int)q);
            if (old >= 0 && old != (int)q) { S->state[b] = 256; S->dirty = 1u; }
        } else {
            S->state[b] = 256; S->dirty = 1u;
        }
    }
}

struct h2_dna_acc {
    unsigned p0, p1, p01;        // packed 8-bit sums of code bit 0, 2 * code bit 1, both bits
    unsigned ocnt;               // offenders per code (packed 8-bit)
    unsigned words, zeroed, noff;
};

// thread-private flush of the base accumulators (H = the hints they were collected under); by value, so that the
// accumulators stay in registers
__device__ __noinline__ void h2_dna_flush_vals(h2_core* S, unsigned p0, unsigned p1, unsigned p01, unsigned ocnt, unsigned words,
                                               unsigned zeroed, unsigned H) {
    const unsigned s0 = h2_bytesum(p0), s1 = h2_bytesum(p1) >> 1, s01 = h2_bytesum(p01);
    const unsigned n3 = s01, n1 = s0 - s01, n2 = s1 - s01, n0 = 4u * words - zeroed - n1 - n2 - n3;
    const unsigned v0 = n0 - (ocnt & 255u), v1 = n1 - ((ocnt >> 8) & 255u), v2 = n2 - ((ocnt >> 16) & 255u), v3 = n3 - (ocnt >> 24);
    if (v0) atomicAdd(&S->hist_b[H & 255u], v0);
    if (v1) atomicAdd(&S->hist_b[(H >> 8) & 255u], v1);
    if (v2) atomicAdd(&S->hist_b[(H >> 16) & 255u], v2);
    if (v3) atomicAdd(&S->hist_b[H >> 24], v3);
}
__device__ __forceinline__ void h2_dna_flush(h2_core* S, h2_dna_acc& A, unsigned H) {
    h2_dna_flush_vals(S, A.p0, A.p1, A.p01, A.ocnt, A.words, A.zeroed, H);
    A.p0 = A.p1 = A.p01 = A.ocnt = A.words = A.zeroed = A.noff = 0;
}

// the same for a whole warp (all 32 lanes call it): shuffle reductions, lane 0 adds
__device__ __forceinline__ void h2_dna_flush_warp(h2_core* S, h2_dna_acc& A, unsigned H, unsigned lane) {
    unsigned s0 = h2_bytesum(A.p0), s1 = h2_bytesum(A.p1) >> 1, s01 = h2_bytesum(A.p01);
    unsigned nw = A.words, nz = A.zeroed;
    unsigned oc[4];
#pragma unroll
    for (unsigned c = 0; c < 4; c++) oc[c] = (A.ocnt >> (8 * c)) & 255u;
    s0 = __reduce_add_sync(0xffffffffu, s0); s1 = __reduce_add_sync(0xffffffffu, s1); s01 = __reduce_add_sync(0xffffffffu, s01);
    nw = __reduce_add_sync(0xffffffffu, nw); nz = __reduce_add_sync(0xffffffffu, nz);
#pragma unroll
    for (unsigned c = 0; c < 4; c++) oc[c] = __reduce_add_sync(0xffffffffu, oc[c]);
    if (lane == 0 && nw) {
        unsigned n[4];
        n[3] = s01; n[1] = s0 - s01; n[2] = s1 - s01;
        n[0] = 4u * nw - nz - n[1] - n[2] - n[3];
#pragma unroll
        for (unsigned c = 0; c < 4; c++) {
            const unsigned v = n[c] - oc[c];
            if (v) atomicAdd(&S->hist_b[(H >> (8 * c)) & 255u], v);
        }
    }
    A.p0 = A.p1 = A.p01 = A.ocnt = A.words = A.zeroed = A.noff = 0;
}

// sixteen bases: v = the unit's four words, ua = its shared-memory address, delta = distance to the quality of the same
// position, [lo, hi) = valid bytes of the unit
__device__ __forceinline__ void h2_dna_unit(h2_core* S, const uint4 v, uint32_t ua, uint32_t delta, int lo, int hi, unsigned H,
                                            h2_dna_acc& A) {
    unsigned w[4] = {v.x, v.y, v.z, v.w}, t[4], bad[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        t[k] = (w[k] >> 1) & 0x03030303u;
        const unsigned u2 = t[k] | (t[k] >> 4);
        const unsigned sel = __byte_perm(u2, 0u, 0x4420);                // nibble i = code of byte i
        unsigned ex;                                                     // the codes never set bit 3 of a nibble: plain prmt
        asm("prmt.b32 %0, %1, %2, %3;" : "=r"(ex) : "r"(H), "r"(0u), "r"(sel));
        bad[k] = ex ^ w[k];
    }
    if (lo > 0 || hi < 16) {                                             // edge unit: bytes outside the line count as zeroed
        const uint32_t vb = h2_unitmask(lo, hi);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned vm = h2_nibble_bytes(vb >> (4 * k));
            bad[k] &= vm;
            t[k] &= vm;
        }
        A.zeroed += 16u - __popc(vb);
    }
    if (bad[0] | bad[1] | bad[2] | bad[3]) {
        // offender map: bit 8 j + k <-> byte j of word k
        unsigned m = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned z = (((bad[k] & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | bad[k]) & 0x80808080u;
            m |= z >> (7 - k);
        }
        A.noff += __popc(m);
        do {
            const unsigned i = (unsigned)__ffs((int)m) - 1u;
            m &= m - 1u;
            const unsigned pos = 4u * (i & 7u) + (i >> 3);
            const unsigned b = lds_u8(ua + pos), q = lds_u8(ua + pos + delta);
            A.ocnt += 1u << (8u * ((b >> 1) & 3u));
            h2_slow_byte(S, b, q);
        } while (m);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        A.p0 += t[k] & 0x01010101u;
        A.p1 += t[k] & 0x02020202u;
        A.p01 += t[k] & (t[k] >> 1) & 0x01010101u;
    }
    A.words += 4u;
}

// sixteen qualities into the thread's counter column (qcol = column address - 33 rows).  Returns false when a byte
// outside 33..126 was met (nothing is counted then).
__device__ __forceinline__ bool h2_qual_unit(const uint4 v, int lo, int hi, uint32_t qcol) {
    unsigned w[4] = {v.x, v.y, v.z, v.w};
    unsigned bad = 0;
    if (lo > 0 || hi < 16) {
        const uint32_t vb = h2_unitmask(lo, hi);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned vm = h2_nibble_bytes(vb >> (4 * k));
            const unsigned chk = (w[k] & vm) | (0x21212121u & ~vm);
            bad |= ((chk | (chk + 0x01010101u)) | ~((chk & 0x7F7F7F7Fu) + 0x5F5F5F5Fu)) & 0x80808080u;
            w[k] = (w[k] & vm) | (0x7F7F7F7Fu & ~vm);                    // masked-out bytes go to the spare row
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++)
            bad |= ((w[k] | (w[k] + 0x01010101u)) | ~((w[k] & 0x7F7F7F7Fu) + 0x5F5F5F5Fu)) & 0x80808080u;
    }
    if (bad) return false;
#pragma unroll
    for (int k = 0; k < 4; k++) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t a = qcol + (__byte_perm(w[k], 0u, 0x4440 | j) << 9);
            sts_u8(a, lds_u8m(a) + 1u);
        }
    }
    return true;
}

// thread-private flush of one counter column (only when a single tile gives a thread more than ~240 qualities)
__device__ __noinline__ void h2_qual_flush(h2_core* S, uint32_t qcol) {
    for (unsigned r = 0; r < H2_ROWS; r++) {
        const uint32_t a = qcol + ((r + H2_QLO) << 9);
        const unsigned c = lds_u8m(a);
        if (c) { atomicAdd(&S->hist_q[r], c); sts_u8(a, 0u); }
    }
}

// ---- three-stage, barrier-free tile pipeline ----------------------------------------------------------------
// A barrier of the whole CTA at the end of every tile (2 us of work) would make the warps that own the short last units
// wait for the others and every thread pay the line-offset conversion of the next tile.  Instead the tiles flow through
// THREE buffers guarded by mbarriers:
//   full[s]    32 arrivals + the transaction count of the TMA bulk copy of the tile's bytes: every warp has converted its 17
//              of the tile's 513 line offsets (their low 32 bits are enough inside a tile), warp 31 has issued the copy;
//   empty[s]   32 arrivals: every warp is done with the tile that used the buffer.
// A warp waits for nothing but these two, so the warps drift apart by up to two tiles and the per-tile work imbalance
// averages out.  The CTA meets at a real barrier only every F tiles, F adapted so that the 8-bit
// quality counters reach about 200 between two flushes.
#define H3_STAGES 3
struct h3_smem {
    alignas(128) uint8_t front_pad[128];                      // the name copy reads the word in front of a tile's first byte
    alignas(128) uint8_t bytes[H3_STAGES][TL_CAP + 32];
    uint32_t loff[H3_STAGES][4 * TL_R + 4];
    alignas(8) uint64_t full[H3_STAGES];
    alignas(8) uint64_t empty[H3_STAGES];
    uint32_t ok[H3_STAGES];
    alignas(16) uint8_t qcnt[H2_ROWS * H2_COLS];
    h2_core C;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(H2_THREADS, 1) k_pair_hist_pipe(const uint8_t* __restrict__ d, uint64_t n_bytes,
                                                                 const uint64_t* __restrict__ line_off, uint64_t r_begin, uint64_t n_reads,
                                                                 an_dev* __restrict__ s, unsigned int* __restrict__ fallback,
                                                                 uint8_t* __restrict__ names, uint32_t name_pitch) {
    // names (optional): compact side array of the QNAME lines, row r = length byte + text in name_pitch (multiple of 16)
    // bytes.  The name statistics, the tokeniser and the dictionary rows then read 48 bytes per record instead of the
    // 128-byte lines of the FASTQ that hold the names.  A name that does not fit raises bit 2 of `fallback`.
    static_assert(TL_R == 128, "thread <-> line binding assumes 128 records per tile");
    extern __shared__ __align__(128) uint8_t h3_raw[];
    h3_smem* S = reinterpret_cast<h3_smem*>(h3_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    for (unsigned i = tid; i < H2_ROWS * H2_COLS / 4; i += H2_THREADS) reinterpret_cast<uint32_t*>(S->qcnt)[i] = 0;
    for (unsigned i = tid; i <= H2_ROWS; i += H2_THREADS) S->C.hist_q[i] = 0;
    if (tid < 256) { S->C.hist_b[tid] = 0; S->C.state[tid] = -1; }
    if (tid == 0) {
        S->C.hints = H2_NOHINT; S->C.dirty = 0; S->C.oor = 0; S->C.qmax = 0;
        for (int st = 0; st < H3_STAGES; st++) { mbar_init(&S->full[st], H2_THREADS / 32); mbar_init(&S->empty[st], H2_THREADS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const unsigned line = tid & 255u, rec = line & 127u, k0 = tid >> 8;
    const bool isq = (line >> 7) != 0;
    const bool producer = wid == H2_THREADS / 32 - 1;
    const unsigned cw = ((wid >> 3) << 2) | (wid & 3u);
    const uint32_t qcol = smem_u32(S->qcnt) + lane * 4u + (cw & 3u) + 128u * (cw >> 2) - (H2_QLO << 9);
    unsigned qsym = 0;
    h2_dna_acc A;
    A.p0 = A.p1 = A.p01 = A.ocnt = A.words = A.zeroed = A.noff = 0;
    unsigned H = H2_NOHINT;
    unsigned long long len_min = ~0ull, len_max = 0ull;
    long long bad_plus = LLONG_MAX, bad_len = LLONG_MAX;

    const uint64_t ntiles = (n_reads - r_begin + TL_R - 1) / TL_R;
    const uint32_t K = blockIdx.x < ntiles ? (uint32_t)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0u;   // tiles of this CTA

    // Tile k of this CTA -> buffer k % 3.  Every warp converts 17 of the tile's 513 line offsets (one global load per lane,
    // issued two tiles ahead and consumed at the end of the current tile, so its latency is never exposed); warp 31 also
    // issues the bulk copy.  full[s] therefore takes one arrival per warp plus the copy's transaction count.
    constexpr uint32_t OPW = (4 * TL_R + 1 + H2_THREADS / 32 - 1) / (H2_THREADS / 32);        // offsets per warp: 17
    uint64_t pend_off = 0, pend_b0 = 0, pend_b1 = 0;      // loads in flight for the tile that is being prepared
    // tile k of this CTA starts at record r_begin + (blockIdx.x + k * gridDim.x) * TL_R; the loop below carries that record
    // number, the buffer index k % 3 and the barrier parity (k / 3) & 1 along instead of recomputing them per call
    const uint64_t rstride = (uint64_t)gridDim.x * TL_R;
    const uint32_t my_off = wid * OPW + lane;
    auto nrec_at = [&](uint64_t r0) { return (uint32_t)(n_reads - r0 < TL_R ? n_reads - r0 : TL_R); };
    auto prep_load = [&](uint64_t r0, uint32_t nrec) {    // start the loads for the tile at r0
        const uint64_t* lo = line_off + 4 * r0;
        if (lane < OPW && my_off <= 4 * nrec) pend_off = __ldg(lo + my_off);
        if (producer && lane == 0) { pend_b0 = __ldg(lo); pend_b1 = __ldg(lo + 4 * nrec); }
    };
    // finish them: offsets into buffer st, bulk copy, arrivals.  wait_empty: the buffer held an earlier tile (parity given)
    auto prep_store = [&](uint32_t nrec, uint32_t st, bool wait_empty, uint32_t empty_par) {
        if (wait_empty) mbar_wait(&S->empty[st], empty_par);                              // every warp has left the previous tile of this buffer
        const uint32_t i = my_off;
        if (lane < OPW && i <= 4 * nrec) S->loff[st][i] = (uint32_t)pend_off;
        if (producer) {
            const uint64_t b0 = __shfl_sync(0xffffffffu, pend_b0, 0), b1 = __shfl_sync(0xffffffffu, pend_b1, 0);
            const uint64_t a0 = b0 & ~15ull;
            const bool fits = b1 - a0 <= TL_CAP;
            uint64_t a1 = (b1 + 15) & ~15ull;
            const uint64_t lim = n_bytes & ~15ull;         // never read past the last full 16-byte unit of the buffer
            if (a1 > lim) a1 = lim;
            if (a1 < a0) a1 = a0;
            if (fits) for (uint64_t q = a1 + lane; q < b1; q += 32) S->bytes[st][q - a0] = d[q];   // tail of the stream (last tile only)
            __syncwarp();
            if (lane == 0) {
                S->ok[st] = fits ? 1u : 0u;
                const uint32_t bulk = fits ? (uint32_t)(a1 - a0) : 0u;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(&S->full[st], bulk);        // this warp's arrival
                if (bulk) bulk_g2s(S->bytes[st], d + a0, bulk, &S->full[st]);
            }
        } else {
            __syncwarp();
            if (lane == 0) mbar_arrive(&S->full[st]);
        }
    };

    {
        uint64_t r0p = r_begin + (uint64_t)blockIdx.x * TL_R;
        for (uint32_t k = 0; k < K && k < H3_STAGES - 1; k++, r0p += rstride) { const uint32_t nr = nrec_at(r0p); prep_load(r0p, nr); prep_store(nr, k, false, 0u); }
    }
    uint32_t F = 1, next_flush = 1;
    uint64_t r0 = r_begin + (uint64_t)blockIdx.x * TL_R;   // first record of tile k
    uint32_t st = 0, par = 0;                              // k % 3, (k / 3) & 1
    for (uint32_t k = 0; k < K; k++) {
        const bool ahead = k + H3_STAGES - 1 < K;
        // tile k + 2: buffer (st + 2) % 3; it follows tile k - 1 there, whose round was (k - 1) / 3
        const uint64_t r0a = r0 + 2 * rstride;
        const uint32_t nrec_a = ahead ? nrec_at(r0a) : 0u;
        const uint32_t st_a = st ? st - 1u : 2u;
        const uint32_t par_a = st ? par : par ^ 1u;        // parity of round (k - 1) / 3
        if (ahead) prep_load(r0a, nrec_a);
        mbar_wait(&S->full[st], par);
        const uint32_t nrec = nrec_at(r0);
        if (S->ok[st] && names && wid < TL_R / 8) {        // warps 0..15: four lanes copy one name, 16 bytes each
            const uint32_t bytes_a = smem_u32(S->bytes[st]);
            const uint32_t* loff = S->loff[st];
            const uint32_t base32 = loff[0] & ~15u;
            const uint32_t nr = 8u * wid + (lane >> 2);
            if (nr < nrec) {
                const uint32_t n0 = loff[4 * nr] - base32, nlen = loff[4 * nr + 1] - base32 - n0 - 1u;
                if (nlen + 1u > name_pitch || nlen > 255u) {
                    if ((lane & 3u) == 0) atomicOr(&S->C.oor, 2u);
                } else {
                    uint4* dst = reinterpret_cast<uint4*>(names + (r0 + nr) * name_pitch);
                    // image byte 0 is the length, byte b > 0 is text byte b - 1: chunk c = image bytes 16 c .. 16 c + 15 starts one
                    // byte in front of text byte 16 c (for c = 0 that is the byte before the name, replaced by the length)
                    for (uint32_t c = lane & 3u; 16u * c <= nlen; c += 4) {
                        const uint32_t at = n0 + 16u * c - 1u, al = bytes_a + (at & ~3u), sh = (at & 3u) * 8u;
                        const uint32_t x0 = lds_u32(al), x1 = lds_u32(al + 4u), x2 = lds_u32(al + 8u), x3 = lds_u32(al + 12u), x4 = lds_u32(al + 16u);
                        uint4 v;
                        v.x = __funnelshift_r(x0, x1, sh); v.y = __funnelshift_r(x1, x2, sh);
                        v.z = __funnelshift_r(x2, x3, sh); v.w = __funnelshift_r(x3, x4, sh);
                        if (c == 0) v.x = (v.x & 0xFFFFFF00u) | nlen;
                        dst[c] = v;
                    }
                }
            }
        }
        if (!S->ok[st]) {
            if (tid == 0) atomicOr(fallback, 1u);
        } else if (rec < nrec) {
            const uint32_t bytes_a = smem_u32(S->bytes[st]);
            const uint32_t* loff = S->loff[st];
            const uint32_t base32 = loff[0] & ~15u;
            const uint32_t o1 = loff[4 * rec + 1] - base32, o2 = loff[4 * rec + 2] - base32, o3 = loff[4 * rec + 3] - base32,
                           o4 = loff[4 * rec + 4] - base32;
            uint32_t len = o2 - o1 - 1;
            const uint32_t qlen = o4 - o3 - 1;
            if (tid < TL_R) {                          // DNA thread of unit 0: the record's checks
                const long long r = (long long)(r0 + rec);
                if (len != qlen && r < bad_len) bad_len = r;
                len_min = len < len_min ? len : len_min; len_max = len > len_max ? len : len_max;
                const unsigned plus = o3 - o2 < 2u ? 0u : lds_u8(bytes_a + o2);
                if (plus != '+' && r < bad_plus) bad_plus = r;
            }
            if (qlen < len) len = qlen;
            const uint32_t sb = isq ? o3 : o1, eb = sb + len;
            for (uint32_t u = (sb & ~15u) + 16u * k0; u < eb; u += 64u) {
                const uint4 v = lds_v4(bytes_a + u);
                const int lo = (int)sb - (int)u, hi = (int)eb - (int)u;
                if (isq) {
                    if (qsym > 255u - 16u) { h2_qual_flush(&S->C, qcol); qsym = 0; }
                    if (!h2_qual_unit(v, lo, hi, qcol)) atomicOr(&S->C.oor, 1u);
                    qsym += 16u;
                } else {
                    if (A.words > 120u || A.noff > 224u) h2_dna_flush(&S->C, A, H);
                    h2_dna_unit(&S->C, v, bytes_a + u, o3 - o1, lo, hi, H, A);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&S->empty[st]);
        if (ahead) prep_store(nrec_a, st_a, k >= 1, par_a);
        r0 += rstride;
        if (++st == H3_STAGES) { st = 0; par ^= 1u; }
        if (k + 1 == next_flush || k + 1 == K) {
            // ---- the CTA meets: counter columns -> CTA histograms, hints ----
            const unsigned wq = __reduce_max_sync(0xffffffffu, isq ? qsym : 0u);
            if (lane == 0 && wq) atomicMax(&S->C.qmax, wq);
            __syncthreads();
            for (unsigned r = wid; r < H2_ROWS; r += H2_THREADS / 32) {
                uint32_t* row = reinterpret_cast<uint32_t*>(S->qcnt + r * H2_COLS);
                unsigned e = 0, o = 0;
#pragma unroll
                for (int j = 0; j < H2_COLS / 128; j++) {
                    const unsigned x = row[lane + 32 * j];
                    row[lane + 32 * j] = 0;
                    e += x & 0x00FF00FFu; o += (x >> 8) & 0x00FF00FFu;
                }
                unsigned tot = (e & 0xFFFFu) + (e >> 16) + (o & 0xFFFFu) + (o >> 16);
                tot = __reduce_add_sync(0xffffffffu, tot);
                if (lane == 0) S->C.hist_q[r] += tot;
            }
            qsym = 0;
            h2_dna_flush_warp(&S->C, A, H, lane);
            const unsigned m = S->C.qmax;                                     // read by every thread before it is reset
            __syncthreads();
            if (S->C.dirty && wid == 0) {
                unsigned best[4] = {0, 0, 0, 0};
#pragma unroll
                for (unsigned j = 0; j < 8; j++) {
                    const unsigned b = lane + 32u * j;
                    if (S->C.state[b] == 256) {
                        const unsigned cnt = S->C.hist_b[b] < 0xFFFFFFu ? S->C.hist_b[b] : 0xFFFFFFu;
                        const unsigned key = ((cnt + 1u) << 8) | b;
                        const unsigned c = (b >> 1) & 3u;
#pragma unroll
                        for (unsigned cc = 0; cc < 4; cc++) if (c == cc && key > best[cc]) best[cc] = key;
                    }
                }
                unsigned h = 0;
#pragma unroll
                for (unsigned c = 0; c < 4; c++) {
                    const unsigned mx = __reduce_max_sync(0xffffffffu, best[c]);
                    h |= (mx ? (mx & 255u) : ((H2_NOHINT >> (8 * c)) & 255u)) << (8 * c);
                }
                if (lane == 0) { S->C.hints = h; S->C.dirty = 0; }
            }
            if (tid == 0) S->C.qmax = 0;
            __syncthreads();
            H = S->C.hints;
            // next meeting: the busiest column should reach about 200 increments
            const unsigned rate = max(m / F, 16u);
            F = min(max(208u / rate, 1u), 32u);
            next_flush = k + 1 + F;
        }
    }
    // ---- results ----
    if (tid < TL_R) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long a = __shfl_xor_sync(0xffffffffu, len_min, o), b = __shfl_xor_sync(0xffffffffu, len_max, o);
            const long long e = __shfl_xor_sync(0xffffffffu, bad_plus, o), f = __shfl_xor_sync(0xffffffffu, bad_len, o);
            len_min = a < len_min ? a : len_min; len_max = b > len_max ? b : len_max;
            bad_plus = e < bad_plus ? e : bad_plus; bad_len = f < bad_len ? f : bad_len;
        }
        if (lane == 0) {
            if (len_min != ~0ull) atomicMin(&s->dna_min, len_min);
            atomicMax(&s->dna_max, len_max);
            if (bad_plus != LLONG_MAX) atomicMin(&s->bad_plus, bad_plus);
            if (bad_len != LLONG_MAX) atomicMin(&s->bad_len, bad_len);
        }
    }
    __syncthreads();
    if (tid < 256) {
        if (S->C.hist_b[tid]) atomicAdd(&s->base_count[tid], (unsigned long long)S->C.hist_b[tid]);
        if (tid < H2_ROWS - 1 && S->C.hist_q[tid]) atomicAdd(&s->qual_count[tid + H2_QLO], (unsigned long long)S->C.hist_q[tid]);
        if (tid == 0 && (S->C.oor & 1u)) atomicOr(fallback, 1u);
        if (tid == 0 && (S->C.oor & 2u)) atomicOr(fallback, 4u);
        const int f = S->C.state[tid];
        if (f >= 0) {
            if (f == 256) {
                s->multi[tid] = 1;
                atomicCAS(&s->first_q[tid], -1, 0);                 // mark the base as present
            } else {
                const int old = atomicCAS(&s->first_q[tid], -1, f);
                if (old >= 0 && old != f) s->multi[tid] = 1;
            }
        }
    }
}
