// Stage 3: stable sort / unique of fixed-width byte rows in memcmp order.
// Replaces numpy.argsort / numpy.unique(return_inverse) / fancy-index gathers in
// encode_dna_qual (uq.py:765-805) and encode_qname (uq.py:808-851).
//
// Algorithm: MSD refinement in 8-byte chunks on top of the stable LSD radix sort of prims.cu.
//   round 0   sort (be64(row[0:8]), row index) over all rows; mark group heads.  Rows wider than 256 bytes are
//             taken from their first non-zero byte: the key is (significant length, first 8 significant bytes).
//   finisher  tie groups of 2..32 rows are completed by one warp each (k_small_groups: three-way quicksort on rows
//             staged in shared memory); for typical data nothing is left after it.
//   round c   (groups of more than 32 rows) only rows that are still tied with a neighbour AND whose tie group is not made of
//             identical rows ("all-equal finisher": one compare of the remaining bytes against the
//             group's first row) stay active; they are compacted, keyed by (group id, be64(row[8c:8c+8]))
//             and sorted again; results are written back in place.  Groups are contiguous, so a
//             sort by (group id, chunk) never moves a row out of its group's position range.
// Stability: the radix sort is stable and every round keeps the previous order for equal keys, so
// equal rows end in input order (numpy kind='stable', SURVEY D1).
#include "common.cuh"

#define ST 256

__global__ void __launch_bounds__(ST) k_chunk0_keys(const uint8_t* __restrict__ rows, uint64_t n, uint32_t width,
                                                   uint64_t* __restrict__ key, uint32_t* __restrict__ val) {
    uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (i >= n) return;
    key[i] = load_be64(rows + i * width, width < 8 ? width : 8);
    val[i] = (uint32_t)i;
}

// Wide rows (variable-length reads are right aligned: a read of half the maximum length starts with thousands of zero
// bytes) are compared from their first non-zero byte: zoff[i] = number of leading zero bytes of row i (one warp per
// row, 16-byte loads when the row is aligned).  memcmp order = fewer significant bytes first, then the significant
// bytes, so round 0 sorts by (significant length, first 8 significant bytes) and the refinement rounds take their
// 8-byte chunks relative to zoff; rows of one tie group always share their zoff.
#define SORT_ZOFF_MIN_WIDTH 256
__global__ void __launch_bounds__(ST) k_leading_zero_bytes(const uint8_t* __restrict__ rows, uint64_t n, uint32_t width,
                                                          uint32_t* __restrict__ zoff) {
    const unsigned lane = threadIdx.x & 31u;
    const uint64_t wstride = (uint64_t)gridDim.x * (ST / 32);
    for (uint64_t i = (uint64_t)blockIdx.x * (ST / 32) + (threadIdx.x >> 5); i < n; i += wstride) {
        const uint8_t* row = rows + i * width;
        uint32_t z = width;
        const uint32_t head = (uint32_t)((16u - ((uintptr_t)row & 15u)) & 15u);          // bytes before the first aligned unit
        // unaligned head, byte by byte
        for (uint32_t b0 = 0; b0 < head && b0 < width && z == width; b0 += 32) {
            const uint32_t b = b0 + lane;
            const bool nz = b < head && b < width && row[b] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, nz);
            if (m) z = b0 + (__ffs(m) - 1);
        }
        // aligned body, 16 bytes per lane
        for (uint32_t b0 = head; b0 < width && z == width; b0 += 512) {
            const uint32_t b = b0 + lane * 16;
            uint32_t first = 16;
            if (b + 16 <= width) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(row + b));
                if (v.x) first = (__ffs(v.x) - 1) >> 3;
                else if (v.y) first = 4 + ((__ffs(v.y) - 1) >> 3);
                else if (v.z) first = 8 + ((__ffs(v.z) - 1) >> 3);
                else if (v.w) first = 12 + ((__ffs(v.w) - 1) >> 3);
            } else if (b < width) {
                for (uint32_t k = 0; k < width - b; k++) if (row[b + k] != 0) { first = k; break; }
            }
            const unsigned m = __ballot_sync(0xffffffffu, first < 16);
            if (m) {
                const int src = __ffs(m) - 1;
                z = b0 + src * 16 + __shfl_sync(0xffffffffu, first, src);
            }
        }
        if (lane == 0) zoff[i] = z;
    }
}

__global__ void __launch_bounds__(ST) k_chunk0_keys_z(const uint8_t* __restrict__ rows, uint64_t n, uint32_t width, const uint32_t* __restrict__ zoff,
                                                     uint64_t* __restrict__ key, uint32_t* __restrict__ aux, uint32_t* __restrict__ val) {
    uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (i >= n) return;
    const uint32_t z = zoff[i], sig = width - z;
    key[i] = load_be64(rows + i * width + z, sig < 8 ? sig : 8);
    aux[i] = sig;                       // fewer significant bytes = more leading zeros = smaller row
    val[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(ST) k_mark_heads(const uint64_t* __restrict__ key, const uint32_t* __restrict__ aux, uint64_t n,
                                                  uint32_t* __restrict__ head) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    head[p] = (p == 0 || key[p] != key[p - 1] || (aux && aux[p] != aux[p - 1])) ? 1u : 0u;
}

// gid[p] = excl[p] + head[p] - 1 ; headpos[gid] = p for heads
#define GLCP_EQUAL 0xFFFFFFFFu       // glcp[g]: every row of group g equals the group's first row
__global__ void __launch_bounds__(ST) k_headpos(const uint32_t* __restrict__ head, const uint32_t* __restrict__ excl, uint64_t n,
                                               uint32_t* __restrict__ headpos, uint32_t* __restrict__ glcp) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    if (head[p]) { headpos[excl[p]] = (uint32_t)p; glcp[excl[p]] = GLCP_EQUAL; }
    if (p == n - 1) headpos[excl[p] + head[p]] = (uint32_t)n;      // sentinel: headpos[number of groups] = n
}

// Common prefix of every tie group with its first row: glcp[g] = min over the members of the first byte offset (>= off,
// relative to the row's first significant byte) at which a member differs from the group's first row; stays
// GLCP_EQUAL when all members are identical.  One pass with every row read exactly once by SUB lanes (aligned 32-bit
// words, funnel shifted to the row's byte phase; 32 / SUB rows per warp step, four steps in flight), the first rows
// come from the caches.  Identical-row groups - the bulk of duplicated reads / qualities - are finished by this
// pass alone; the others continue, each from ITS OWN common prefix, so a table whose rows share long prefixes does
// not pay one refinement round per 8 bytes.
template <int SUB>
__global__ void __launch_bounds__(ST) k_group_lcp(const uint8_t* __restrict__ rows, uint32_t width, uint32_t off, const uint32_t* __restrict__ zoff,
                                                 const uint32_t* __restrict__ perm, const uint32_t* __restrict__ head,
                                                 const uint32_t* __restrict__ excl, const uint32_t* __restrict__ headpos,
                                                 const uint8_t* __restrict__ done, uint64_t n, uint32_t* __restrict__ glcp) {
    constexpr uint32_t NP = 32u / SUB;
    constexpr int UN = 4;
    const unsigned lane = threadIdx.x & 31u, sg = lane / SUB, sl = lane % SUB;
    const uint64_t nblk = (n + 31) / 32, wstride = (uint64_t)gridDim.x * (ST / 32);
    for (uint64_t blk = (uint64_t)blockIdx.x * (ST / 32) + (threadIdx.x >> 5); blk < nblk; blk += wstride) {
        const uint64_t p = blk * 32 + lane;
        uint32_t ra = 0, rb = 0, g = 0, z = 0;
        bool live = false;
        if (p < n && !head[p] && !done[p]) {
            live = true;
            g = excl[p] - 1;                           // exclusive scan of the head flags; head[p] == 0
            ra = perm[p];
            rb = perm[headpos[g]];
            if (zoff) z = zoff[ra];                    // the rows of a group share their leading-zero count
        }
        unsigned todo = __ballot_sync(0xffffffffu, live);
        if (!todo) continue;
        uint32_t mine = GLCP_EQUAL;                    // result of the row at this lane's position
        for (uint32_t j0 = 0; j0 < 32; j0 += NP * UN) {
            if (!((todo >> j0) & ((NP * UN >= 32) ? 0xffffffffu : ((1u << (NP * UN)) - 1u)))) continue;
            uint32_t res[UN];
#pragma unroll
            for (int u = 0; u < UN; u++) res[u] = GLCP_EQUAL;
            // rows of this batch
            uint32_t a_r[UN], b_r[UN], zz[UN];
            bool lv[UN];
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const uint32_t j = j0 + u * NP + sg;
                a_r[u] = __shfl_sync(0xffffffffu, ra, j & 31u);
                b_r[u] = __shfl_sync(0xffffffffu, rb, j & 31u);
                zz[u] = __shfl_sync(0xffffffffu, z, j & 31u);
                lv[u] = j < 32u && ((todo >> (j & 31u)) & 1u);
            }
            const uint32_t maxrem = width - off;       // upper bound of the bytes to compare (z only shortens it)
            for (uint32_t w0 = 0; 4u * w0 < maxrem; w0 += SUB) {
                const uint32_t wd = w0 + sl;
                uint32_t xa[UN], xb[UN];
#pragma unroll
                for (int u = 0; u < UN; u++) {
                    xa[u] = 0; xb[u] = 0;
                    const uint32_t start = zz[u] + off;
                    if (lv[u] && start + 4u * wd < width) {
                        const uint64_t A = (uint64_t)(uintptr_t)rows + (uint64_t)a_r[u] * width + start;
                        const uint64_t B = (uint64_t)(uintptr_t)rows + (uint64_t)b_r[u] * width + start;
                        const uint32_t pa = (uint32_t)A & 3u, pb = (uint32_t)B & 3u;
                        const uint32_t* wa = reinterpret_cast<const uint32_t*>(A - pa) + wd;
                        const uint32_t* wb = reinterpret_cast<const uint32_t*>(B - pb) + wd;
                        // the word after the row's last one may be read (never used): every table has >= 8 bytes of slack
                        xa[u] = __funnelshift_r(__ldg(wa), __ldg(wa + 1), pa * 8u);
                        xb[u] = __funnelshift_r(__ldg(wb), __ldg(wb + 1), pb * 8u);
                    }
                }
                bool any_live = false;
#pragma unroll
                for (int u = 0; u < UN; u++) {
                    const uint32_t start = zz[u] + off;
                    uint32_t d = xa[u] ^ xb[u];
                    const uint32_t left = (lv[u] && start + 4u * wd < width) ? width - start - 4u * wd : 0u;   // valid bytes of this word
                    if (left < 4u) d &= left ? (0xffffffffu >> (8u * (4u - left))) : 0u;
                    uint32_t m = d ? 4u * wd + (((uint32_t)__ffs((int)d) - 1u) >> 3) : GLCP_EQUAL;
#pragma unroll
                    for (int o = SUB / 2; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
                    if (res[u] == GLCP_EQUAL && m != GLCP_EQUAL) { res[u] = off + m; lv[u] = false; }
                    any_live |= lv[u];
                }
                if (!__any_sync(0xffffffffu, any_live)) break;
            }
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const uint32_t j = j0 + u * NP;       // rows j .. j + NP - 1: sub-group s holds row j + s
                // hand the result to the lane that owns the position
#pragma unroll
                for (uint32_t s2 = 0; s2 < NP; s2++) {
                    const uint32_t v = __shfl_sync(0xffffffffu, res[u], s2 * SUB);
                    if (lane == j + s2) mine = v;
                }
            }
        }
        // one atomic per warp when its rows share a group (a giant group would otherwise serialise millions of them), and
        // none when the group's value is already as small
        const uint32_t g0 = __shfl_sync(0xffffffffu, g, __ffs((int)todo) - 1);
        if (__all_sync(0xffffffffu, !live || g == g0)) {
            const uint32_t m = __reduce_min_sync(0xffffffffu, live ? mine : GLCP_EQUAL);
            if (lane == 0 && m != GLCP_EQUAL && m < *((volatile uint32_t*)&glcp[g0])) atomicMin(&glcp[g0], m);
        } else if (live && mine != GLCP_EQUAL && mine < *((volatile uint32_t*)&glcp[g])) {
            atomicMin(&glcp[g], mine);
        }
    }
}

// rows that go into the next radix round: members of groups whose rows are not all identical and that the small-group
// finisher has not completed.  Members of identical-row groups are marked done (nothing more to compare).
__global__ void __launch_bounds__(ST) k_active_flags(const uint32_t* __restrict__ head, const uint32_t* __restrict__ excl,
                                                    const uint32_t* __restrict__ glcp, uint8_t* __restrict__ done,
                                                    uint64_t n, uint32_t* __restrict__ act) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    if (done[p]) { act[p] = 0u; return; }       // finished by k_small_groups (its excl / head may be stale)
    uint32_t g = excl[p] + head[p] - 1;
    bool single = head[p] && (p + 1 == n || head[p + 1]);
    const bool differ = glcp[g] != GLCP_EQUAL;
    if (!single && !differ) done[p] = 1;
    act[p] = (!single && differ) ? 1u : 0u;
}

// ---- small tie groups: finished in one pass ------------------------------------------------------
// After round 0 almost every tie group is small.  A group of 2..32 rows is sorted completely by one
// warp: lane i holds row i of the group, the remaining bytes [off, width) of the rows are staged in
// shared memory as big-endian words (so an unsigned word compare is memcmp order), every lane ranks
// its row against the others (ties keep the current = input order), and the permutation and the
// group heads are rewritten in place.  Rows wider than SG_STAGE_BYTES are compared straight from
// global memory instead.  Groups larger than 32 rows are left to the radix rounds; their total row
// count is returned so that the host can stop as soon as there are none.
#define SG_MAX 32
#define SG_STAGE_BYTES 256

// Staged variant.  SUB lanes work on one row (SUB = 8, 16 or 32; 32 / SUB rows at a time).
//   staging   the remaining bytes of every row are fetched as ALIGNED 32-bit words (two per lane, funnel
//             shifted to the row's byte phase) and stored big-endian, zero padded, `pitch` words per row;
//   sorting   three-way quicksort with warp-uniform control: the first row of the first unresolved segment
//             is the pivot, every other row of the segment is compared with it word-parallel (ballots give
//             the first differing word), and a STABLE partition (ballot + popc) moves the rows to
//             less | equal | greater.  The equal range is final; ranges of one row are final.  A group of
//             identical rows costs size-1 compares (the common case for duplicated reads / qualities), a
//             group of distinct rows O(size log size) instead of all size(size-1)/2 pairs.
// Stable partitions keep equal rows in their current (= input) order.
// The first pass (pivot = first row of the group) is fused with the staging: the pivot's words stay in
// registers and every row is compared with them the moment it arrives, so a group of identical rows is
// finished without reading shared memory at all.
// all lanes: request the rows of the group held by the lane of the lowest set bit of `mask` (none when mask == 0)
__device__ __forceinline__ void sg_prefetch(const uint8_t* __restrict__ rows, uint32_t width, uint32_t off, const uint32_t* __restrict__ perm,
                                            uint32_t start, uint32_t size, unsigned mask, unsigned lane) {
    if (!mask) return;
    const int src = __ffs((int)mask) - 1;
    const uint32_t s = __shfl_sync(0xffffffffu, start, src), sz = __shfl_sync(0xffffffffu, size, src);
    if (lane < sz) {
        const uint8_t* a = rows + (uint64_t)__ldg(perm + s + lane) * width;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(a + off));
        if ((((uintptr_t)(a + off)) ^ ((uintptr_t)(a + width - 1))) >> 7) asm volatile("prefetch.global.L2 [%0];" ::"l"(a + width - 1));
    }
}

template <int SUB, int TRIPS>      // TRIPS = ceil(pitch / SUB): 1, or 2 for SUB == 32 and 33..64 words
__global__ void __launch_bounds__(ST) k_small_groups(const uint8_t* __restrict__ rows, uint32_t width, uint32_t off,
                                                    uint32_t* __restrict__ perm, uint32_t* __restrict__ head, uint8_t* __restrict__ done,
                                                    const uint32_t* __restrict__ headpos, const uint32_t* __restrict__ d_ngroups,
                                                    uint32_t pitch, unsigned long long* __restrict__ large_rows) {
    extern __shared__ uint32_t sg_smem[];
    constexpr uint32_t NP = 32u / SUB;
    constexpr uint32_t SUBMASK = SUB == 32 ? 0xffffffffu : ((1u << (SUB & 31)) - 1u);
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const unsigned sg = lane / SUB, sl = lane % SUB;
    uint32_t* srows = sg_smem + (size_t)w * (SG_MAX * pitch + 64);
    uint32_t* sord = srows + SG_MAX * pitch;
    const uint32_t G = *d_ngroups;
    const uint32_t rem = width - off;
    const uint64_t warps_total = (uint64_t)gridDim.x * (ST / 32);
    const uint32_t ltm = (1u << lane) - 1u;
    // per-lane constants of the staging: word index, validity, mask of the row's last (partial) word
    uint32_t tailmask[TRIPS];
    bool wvalid[TRIPS];
#pragma unroll
    for (int t = 0; t < TRIPS; t++) {
        const uint32_t wd = t * SUB + sl;
        wvalid[t] = wd < pitch;
        const uint32_t nvalid = wvalid[t] ? rem - 4u * wd : 0u;
        tailmask[t] = nvalid >= 4u ? 0xffffffffu : (nvalid ? 0xffffffffu << ((4u - nvalid) * 8u) : 0u);
    }
    unsigned long long my_large = 0;
    for (uint64_t g0 = ((uint64_t)blockIdx.x * (ST / 32) + w) * 32; g0 < G; g0 += warps_total * 32) {
        const uint64_t g = g0 + lane;
        uint32_t start = 0, size = 0;
        if (g < G) { start = headpos[g]; size = headpos[g + 1] - start; }
        const bool fin = size < 2 || done[start];
        if (size > SG_MAX && !fin) my_large += size;
        unsigned need = __ballot_sync(0xffffffffu, size <= SG_MAX && !fin);
        // the rows of the next two groups are requested (L2 prefetch) while the current one is staged and sorted: one group
        // alone keeps only a handful of random row reads in flight per warp
        sg_prefetch(rows, width, off, perm, start, size, need & (need - 1u), lane);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            sg_prefetch(rows, width, off, perm, start, size, need & (need - 1u), lane);
            const uint32_t s = __shfl_sync(0xffffffffu, start, src), sz = __shfl_sync(0xffffffffu, size, src);
            const uint32_t r = lane < sz ? perm[s + lane] : 0u;
            // ---- stage, and compare with the first row ----
            uint32_t pvw[TRIPS];                                           // the pivot's words of this lane
            int c = 0;                                                     // memcmp(row at my position, pivot)
#pragma unroll 2
            for (uint32_t j0 = 0; j0 < sz; j0 += NP) {
                const uint32_t j = j0 + sg;
                const uint32_t rj = __shfl_sync(0xffffffffu, r, j & 31u);
                const uint64_t A = (uint64_t)(uintptr_t)rows + (uint64_t)rj * width + off;
                const uint32_t ph = (uint32_t)A & 3u;
                const uint32_t* base = reinterpret_cast<const uint32_t*>(A - ph) + sl;
                const bool jv = j < sz;
                uint32_t v[TRIPS];
#pragma unroll
                for (int t = 0; t < TRIPS; t++) {
                    uint32_t lo = 0, hi = 0;
                    // the word after the row's last one may be read (never used): every table has >= 8 bytes of slack
                    if (jv && wvalid[t]) { lo = __ldg(base + t * SUB); hi = __ldg(base + t * SUB + 1); }
                    v[t] = __byte_perm(__funnelshift_r(lo, hi, ph * 8u), 0u, 0x0123) & tailmask[t];
                    if (jv && wvalid[t]) srows[j * pitch + t * SUB + sl] = v[t];
                }
                if (j0 == 0) {
#pragma unroll
                    for (int t = 0; t < TRIPS; t++) pvw[t] = NP == 1 ? v[t] : __shfl_sync(0xffffffffu, v[t], sl);
                }
                int cc = 0;
#pragma unroll
                for (int t = 0; t < TRIPS; t++) {
                    const unsigned ne = (__ballot_sync(0xffffffffu, jv && v[t] != pvw[t]) >> (sg * SUB)) & SUBMASK;
                    const unsigned lt = (__ballot_sync(0xffffffffu, v[t] < pvw[t]) >> (sg * SUB)) & SUBMASK;
                    if (cc == 0 && ne) cc = ((lt >> (__ffs((int)ne) - 1)) & 1u) ? -1 : 1;
                }
                if (NP == 1) {
                    if (lane == j0) c = cc;
                } else {
                    const int got = __shfl_sync(0xffffffffu, cc, ((lane - j0) * SUB) & 31u);
                    if (lane >= j0 && lane < j0 + NP) c = got;
                }
            }
            __syncwarp();
            // ---- sort ----
            uint32_t ord = lane;                                           // staged row at position `lane`
            uint32_t B = 1u;                                               // segment starts (finally: distinct-row starts)
            uint32_t R = sz < 32u ? ~((1u << sz) - 1u) : 0u;               // resolved positions
            bool have_c = true;
            while (~R) {
                const uint32_t lo = (uint32_t)__ffs((int)~R) - 1u;
                const uint32_t above = B & ~((2u << lo) - 1u);
                const uint32_t hi = above ? (uint32_t)__ffs((int)above) - 1u : sz;
                if (!have_c) {
                    const uint32_t piv = __shfl_sync(0xffffffffu, ord, lo);
                    uint32_t y[TRIPS];
#pragma unroll
                    for (int t = 0; t < TRIPS; t++) y[t] = wvalid[t] ? srows[piv * pitch + t * SUB + sl] : 0u;
                    c = 0;
                    for (uint32_t q0 = lo + 1; q0 < hi; q0 += NP) {
                        const uint32_t pp = q0 + sg;
                        const bool pv = pp < hi;
                        const uint32_t a = __shfl_sync(0xffffffffu, ord, pp & 31u);
                        int cc = 0;
#pragma unroll
                        for (int t = 0; t < TRIPS; t++) {
                            const uint32_t x = (pv && wvalid[t]) ? srows[a * pitch + t * SUB + sl] : y[t];
                            const unsigned ne = (__ballot_sync(0xffffffffu, x != y[t]) >> (sg * SUB)) & SUBMASK;
                            const unsigned lt = (__ballot_sync(0xffffffffu, x < y[t]) >> (sg * SUB)) & SUBMASK;
                            if (cc == 0 && ne) cc = ((lt >> (__ffs((int)ne) - 1)) & 1u) ? -1 : 1;
                        }
                        if (NP == 1) {
                            if (lane == q0) c = cc;
                        } else {
                            const int got = __shfl_sync(0xffffffffu, cc, ((lane - q0) * SUB) & 31u);
                            if (lane >= q0 && lane < q0 + NP && lane < hi) c = got;
                        }
                    }
                }
                have_c = false;
                const bool inr = lane >= lo && lane < hi;
                const unsigned less = __ballot_sync(0xffffffffu, inr && c < 0);
                const unsigned eq = __ballot_sync(0xffffffffu, inr && c == 0);
                const uint32_t nl = __popc(less), neq = __popc(eq);
                const uint32_t e0 = lo + nl, h0 = e0 + neq;                // equal range [e0, h0), greater range [h0, hi)
                if (nl | (hi - h0)) {                                      // anything to move?
                    const unsigned gt = ((hi < 32u ? (1u << hi) : 0u) - (1u << lo)) & ~(less | eq);
                    uint32_t np = lane;
                    if (inr) np = c < 0 ? lo + __popc(less & ltm) : (c == 0 ? e0 + __popc(eq & ltm) : h0 + __popc(gt & ltm));
                    sord[np] = ord;
                    __syncwarp();
                    ord = sord[lane];
                    __syncwarp();
                }
                B |= 1u << e0;
                if (h0 < hi) B |= 1u << h0;
                R |= (uint32_t)((1ull << h0) - (1ull << e0));
                if (nl == 1u) R |= 1u << lo;
                if (hi - h0 == 1u) R |= 1u << h0;
            }
            const uint32_t rfin = __shfl_sync(0xffffffffu, r, ord & 31u);
            if (lane < sz) {
                perm[s + lane] = rfin;
                if (lane > 0) head[s + lane] = (B >> lane) & 1u;
                done[s + lane] = 1;
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_large += __shfl_xor_sync(0xffffffffu, my_large, o);
    if (lane == 0 && my_large) atomicAdd(large_rows, my_large);
}

// ---- first refinement pass: several small tie groups per warp -------------------------------------
// Right after round 0 nothing is done yet, group sizes are small (duplicated reads / qualities come in handfuls) and a
// warp that takes ONE group at a time leaves most of its lanes idle and keeps a handful of random row reads in flight.
// Here a warp walks its chunk of sorted positions and packs as many WHOLE groups as fit into 32 rows: the group
// boundaries come straight from ballots over the head flags of the next 64 positions (no scan, no head-position array).
//   staging   every row of a group of 2+ rows is fetched once as aligned 32-bit words (SUB lanes per row, funnel shifted to
//             the row's byte phase, big-endian in shared memory), up to 32 rows in flight per warp;
//   masks     d[j] = set of words in which row j differs from the first row of its group (one ballot per row);
//   ranking   lane j compares its row with every other row i of its group, looking only at the words of d[i] | d[j] in
//             increasing order (rows that both equal the first row in a word equal each other there): typically one
//             or two word compares per pair.  rank = rows before it (ties keep their current = input order);
//   output    permutation, heads of the distinct rows and done flags, in place.
// Groups of more than 32 rows are skipped and reported; the caller then runs the general rounds for them.
#define SGP_CHUNK 2048
template <int SUB>
__global__ void __launch_bounds__(ST) k_small_groups_packed(const uint8_t* __restrict__ rows, uint32_t width, uint32_t off,
                                                           uint32_t* __restrict__ perm, const uint32_t* __restrict__ head, uint32_t* __restrict__ head_out,
                                                           uint8_t* __restrict__ done, uint64_t n, uint32_t pitch,
                                                           unsigned long long* __restrict__ large_rows) {
    // head: the group starts of round 0, read only (neighbouring warps look at each other's positions to find their
    // first group); head_out: a copy of it, in which the starts of the distinct rows are added
    extern __shared__ uint32_t sg_smem[];
    constexpr uint32_t NP = 32u / SUB;
    constexpr uint32_t SUBMASK = SUB == 32 ? 0xffffffffu : ((1u << (SUB & 31)) - 1u);
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const unsigned sg = lane / SUB, sl = lane % SUB;
    uint32_t* srows = sg_smem + (size_t)w * (32 * pitch);
    const uint32_t rem = width - off;
    const bool wvalid = sl < pitch;
    const uint32_t nvalid = wvalid ? rem - 4u * sl : 0u;
    const uint32_t tailmask = nvalid >= 4u ? 0xffffffffu : (nvalid ? 0xffffffffu << ((4u - nvalid) * 8u) : 0u);
    const uint64_t nchunks = (n + SGP_CHUNK - 1) / SGP_CHUNK, warps_total = (uint64_t)gridDim.x * (ST / 32);
    unsigned long long my_large = 0;
    for (uint64_t ck = (uint64_t)blockIdx.x * (ST / 32) + w; ck < nchunks; ck += warps_total) {
        const uint64_t c0 = ck * SGP_CHUNK, c1 = (c0 + SGP_CHUNK < n) ? c0 + SGP_CHUNK : n;
        uint64_t cur = c0;
        // the first group that STARTS in this chunk
        while (cur < c1) {
            const unsigned hb = __ballot_sync(0xffffffffu, cur + lane < n ? head[cur + lane] != 0u : true);
            if (hb) { cur += (unsigned)__ffs((int)hb) - 1u; break; }
            cur += 32;
        }
        while (cur < c1) {
            // the row index of position cur + lane is requested together with the head flags: the rows can then be fetched
            // as soon as the window is known (two dependent round trips per window instead of three)
            const uint32_t r_spec = cur + lane < n ? perm[cur + lane] : 0u;
            const unsigned h1 = __ballot_sync(0xffffffffu, cur + lane < n ? head[cur + lane] != 0u : true);             // bit 0 is set
            const unsigned h2 = __ballot_sync(0xffffffffu, cur + 32 + lane < n ? head[cur + 32 + lane] != 0u : true);
            const unsigned hi = (h1 >> 1) | (h2 << 31);            // bit k: a group starts at cur + 1 + k
            if (!hi) {
                // more than 32 rows: report it and skip to the next group that starts inside this chunk (the rest of a group
                // that runs past the chunk belongs to nobody: the warps of the following chunks start at their first head)
                uint64_t nxt = c1;
                if (h2 >> 1) nxt = cur + 32 + ((unsigned)__ffs((int)(h2 >> 1)));
                else {
                    for (uint64_t q = cur + 64; q < c1; q += 32) {
                        const unsigned hb = __ballot_sync(0xffffffffu, q + lane < n ? head[q + lane] != 0u : true);
                        if (hb) { nxt = q + (unsigned)__ffs((int)hb) - 1u; break; }
                    }
                }
                if (lane == 0) my_large += 33;                       // only "any large group" matters to the caller
                cur = nxt;
                continue;
            }
            const uint32_t cnt = 32u - (uint32_t)__clz((int)hi);   // rows cur .. cur + cnt - 1 are whole groups, cnt <= 32
            const unsigned live = cnt == 32u ? 0xffffffffu : ((1u << cnt) - 1u);
            const unsigned hm = h1 & live;
            if (hm == live) { cur += cnt; continue; }              // single rows only
            const uint32_t r = lane < cnt ? r_spec : 0u;
            const unsigned upto = (2u << lane) - 1u;               // lanes 0 .. lane
            const uint32_t gs = 31u - (uint32_t)__clz((int)(hm & upto));
            const unsigned above = hm & ~upto;
            const uint32_t ge = above ? (uint32_t)__ffs((int)above) - 1u : cnt;
            const bool multi = lane < cnt && ge - gs > 1u;
            const unsigned need = __ballot_sync(0xffffffffu, multi);
            // ---- stage ----
#pragma unroll 4
            for (uint32_t j0 = 0; j0 < cnt; j0 += NP) {
                const uint32_t j = j0 + sg;
                const uint32_t rj = __shfl_sync(0xffffffffu, r, j & 31u);
                if (j < cnt && ((need >> j) & 1u) && wvalid) {
                    const uint64_t A = (uint64_t)(uintptr_t)rows + (uint64_t)rj * width + off;
                    const uint32_t ph = (uint32_t)A & 3u;
                    const uint32_t* base = reinterpret_cast<const uint32_t*>(A - ph) + sl;
                    // the word after the row's last one may be read (never used): every table has >= 8 bytes of slack
                    const uint32_t lo = __ldg(base), hi2 = __ldg(base + 1);
                    srows[j * pitch + sl] = __byte_perm(__funnelshift_r(lo, hi2, ph * 8u), 0u, 0x0123) & tailmask;
                }
            }
            __syncwarp();
            // ---- difference masks against the first row of the group ----
            const uint32_t maxsz = __reduce_max_sync(0xffffffffu, multi ? ge - gs : 0u);
            unsigned dmask = 0;
            for (uint32_t j0 = 0; j0 < cnt; j0 += NP) {
                const uint32_t j = j0 + sg;
                const uint32_t sj = __shfl_sync(0xffffffffu, gs, j & 31u);
                bool ne = false;
                if (j < cnt && ((need >> j) & 1u) && wvalid) ne = srows[j * pitch + sl] != srows[sj * pitch + sl];
                const unsigned b = __ballot_sync(0xffffffffu, ne);
#pragma unroll
                for (uint32_t s2 = 0; s2 < NP; s2++) if (lane == j0 + s2) dmask = (b >> (s2 * SUB)) & SUBMASK;
            }
            // ---- rank inside the group ----
            uint32_t rank = 0;
            bool eq_before = false;
            for (uint32_t t = 0; t < maxsz; t++) {
                const uint32_t i = gs + t;
                const bool act = multi && i < ge && i != lane;
                const unsigned di = __shfl_sync(0xffffffffu, dmask, act ? i : lane);
                if (act) {
                    unsigned m = di | dmask;
                    int c = 0;          // memcmp(row i, row lane)
                    while (m) {
                        const uint32_t wd = (uint32_t)__ffs((int)m) - 1u;
                        m &= m - 1u;
                        const uint32_t a = srows[i * pitch + wd], b = srows[lane * pitch + wd];
                        if (a != b) { c = a < b ? -1 : 1; break; }
                    }
                    if (c < 0 || (c == 0 && i < lane)) rank++;
                    if (c == 0 && i < lane) eq_before = true;
                }
            }
            __syncwarp();
            if (multi) {
                perm[cur + gs + rank] = r;
                if (rank > 0) head_out[cur + gs + rank] = eq_before ? 0u : 1u;
                done[cur + lane] = 1;
            }
            cur += cnt;
        }
    }
    if (lane == 0 && my_large) atomicAdd(large_rows, my_large);
}

// Rows whose remainder is wider than SG_STAGE_BYTES: lane i ranks row i against the others straight from
// global memory (rare: only very long variable-length reads get here).
__global__ void __launch_bounds__(ST) k_small_groups_gmem(const uint8_t* __restrict__ rows, uint32_t width, uint32_t off,
                                                         const uint32_t* __restrict__ zoff, uint32_t* __restrict__ perm, uint32_t* __restrict__ head, uint8_t* __restrict__ done,
                                                         const uint32_t* __restrict__ headpos, const uint32_t* __restrict__ d_ngroups,
                                                         unsigned long long* __restrict__ large_rows) {
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t G = *d_ngroups;
    const uint64_t warps_total = (uint64_t)gridDim.x * (ST / 32);
    unsigned long long my_large = 0;
    for (uint64_t g0 = ((uint64_t)blockIdx.x * (ST / 32) + w) * 32; g0 < G; g0 += warps_total * 32) {
        const uint64_t g = g0 + lane;
        uint32_t start = 0, size = 0;
        if (g < G) { start = headpos[g]; size = headpos[g + 1] - start; }
        const bool fin = size < 2 || done[start];
        if (size > SG_MAX && !fin) my_large += size;
        unsigned need = __ballot_sync(0xffffffffu, size <= SG_MAX && !fin);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const uint32_t s = __shfl_sync(0xffffffffu, start, src), sz = __shfl_sync(0xffffffffu, size, src);
            const uint32_t r = lane < sz ? perm[s + lane] : 0u;
            // the rows of a group share their leading-zero count: compare from zoff + off
            const uint32_t z = __shfl_sync(0xffffffffu, (zoff && lane < sz) ? zoff[r] : 0u, 0);
            const uint32_t rem = z + off < width ? width - z - off : 0u;
            uint32_t rank = 0;
            bool eq_before = false;
            for (uint32_t j = 0; j < sz; j++) {
                const uint32_t rj = __shfl_sync(0xffffffffu, r, j);
                if (lane < sz && j != lane) {
                    int c = 0;       // memcmp(row_j, row_lane)
                    const uint8_t* pa = rows + (uint64_t)rj * width + z + off;
                    const uint8_t* pb = rows + (uint64_t)r * width + z + off;
                    for (uint32_t i = 0; i < rem; i++) {
                        const unsigned a = __ldg(pa + i), b = __ldg(pb + i);
                        if (a != b) { c = a < b ? -1 : 1; break; }
                    }
                    if (c < 0 || (c == 0 && j < lane)) rank++;
                    if (c == 0 && j < lane) eq_before = true;
                }
            }
            __syncwarp();
            if (lane < sz) {
                perm[s + rank] = r;
                if (rank > 0) head[s + rank] = eq_before ? 0u : 1u;
                done[s + lane] = 1;
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_large += __shfl_xor_sync(0xffffffffu, my_large, o);
    if (lane == 0 && my_large) atomicAdd(large_rows, my_large);
}

__global__ void __launch_bounds__(ST) k_compact_active(const uint8_t* __restrict__ rows, uint32_t width, const uint32_t* __restrict__ glcp,
                                                      const uint32_t* __restrict__ zoff, const uint32_t* __restrict__ act, const uint32_t* __restrict__ apos,
                                                      const uint32_t* __restrict__ head, const uint32_t* __restrict__ excl,
                                                      const uint32_t* __restrict__ perm, uint64_t n, uint32_t* __restrict__ pos_list,
                                                      uint64_t* __restrict__ key, uint32_t* __restrict__ aux, uint32_t* __restrict__ val) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n || !act[p]) return;
    uint32_t j = apos[p];
    uint32_t row = perm[p];
    pos_list[j] = (uint32_t)p;
    const uint32_t z = zoff ? zoff[row] : 0u;
    const uint32_t g = excl[p] + head[p] - 1;
    const uint32_t off = glcp[g];                     // the group's rows agree before this offset: the next 8 bytes decide
    const uint32_t rem = z + off < width ? width - z - off : 0u;
    key[j] = load_be64(rows + (uint64_t)row * width + z + off, rem < 8 ? rem : 8);
    aux[j] = g;
    val[j] = row;
}

__global__ void __launch_bounds__(ST) k_write_back(const uint64_t* __restrict__ key, const uint32_t* __restrict__ aux,
                                                  const uint32_t* __restrict__ val, const uint32_t* __restrict__ pos_list, uint64_t m,
                                                  uint32_t* __restrict__ perm, uint32_t* __restrict__ head) {
    uint64_t j = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (j >= m) return;
    uint32_t p = pos_list[j];
    perm[p] = val[j];
    head[p] = (j == 0 || aux[j] != aux[j - 1] || key[j] != key[j - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(ST) k_gid_from_scan(const uint32_t* __restrict__ head, uint32_t* __restrict__ excl_inout, uint64_t n) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    excl_inout[p] = excl_inout[p] + head[p] - 1;
}

__global__ void __launch_bounds__(ST) k_iota_zero(uint32_t* __restrict__ perm, uint32_t* __restrict__ gid, uint64_t n) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    perm[p] = (uint32_t)p;
    gid[p] = 0;
}

// d_perm / d_gid_sorted: arena blocks of n + 16 words (the callers turn them into arrays without a copy).
// sorted_keys (optional): for rows of up to 8 bytes the sorted round-0 keys ARE the sorted rows (big-endian, zero padded);
// the buffer is handed over instead of being freed, and the unique table is cut out of it without touching the rows.
int uqb_sort_rows_impl(uqb_ctx* ctx, const uint8_t* rows, uint64_t n, uint32_t width,
                       uint32_t** d_perm, uint32_t** d_gid_sorted, uint64_t* n_unique, const uint64_t* key0, uint64_t** sorted_keys) {
    *d_perm = nullptr; *d_gid_sorted = nullptr; *n_unique = 0;
    if (sorted_keys) *sorted_keys = nullptr;
    if (n >= (1ull << 32)) return uqb_fail(ctx, "sort_rows: %llu rows exceed the 32-bit index range", (unsigned long long)n);
    uint32_t *perm = nullptr, *head, *excl;
    UQB_TRY(uqb_dalloc_t(ctx, &excl, n + 16));
    if (n == 0 || width == 0) UQB_TRY(uqb_dalloc_t(ctx, &perm, n + 16));
    if (n == 0) { *d_perm = perm; *d_gid_sorted = excl; return 0; }
    const unsigned nb = uqb_blocks(n, ST);
    if (width == 0) {
        UQB_LAUNCH(k_iota_zero, nb, ST, 0, perm, excl, n);
        *d_perm = perm; *d_gid_sorted = excl; *n_unique = 1;
        return 0;
    }
    UQB_TRY(uqb_dalloc_t(ctx, &head, n));
    uint32_t* d_tot;
    UQB_TRY(uqb_dalloc_t(ctx, &d_tot, 2));

    // ---- round 0 ----
    uint32_t* zoff = nullptr;
    if (width > SORT_ZOFF_MIN_WIDTH) {
        UQB_TRY(uqb_dalloc_t(ctx, &zoff, n));
        UQB_LAUNCH_B(n * 4, k_leading_zero_bytes, uqb_grid(ctx, n, ST / 32, 16), ST, 0, rows, n, width, zoff);
    }
    {
        uqb_sortbuf sb;
        UQB_TRY(uqb_sortbuf_alloc(ctx, &sb, n, zoff != nullptr));
        const uint64_t* kf = (!zoff && width >= 8) ? key0 : nullptr;        // keys written by the table's producer
        if (zoff) UQB_LAUNCH_B(n * 24, k_chunk0_keys_z, nb, ST, 0, rows, n, width, zoff, sb.key[0], sb.aux[0], sb.val[0]);
        else if (!kf) UQB_LAUNCH_B(n * ((width < 8 ? width : 8) + 12), k_chunk0_keys, nb, ST, 0, rows, n, width, sb.key[0], sb.val[0]);
        UQB_TRY(uqb_radix_sort(ctx, &sb, n, zoff != nullptr, kf));
        UQB_LAUNCH(k_mark_heads, nb, ST, 0, sb.key[sb.cur], zoff ? sb.aux[sb.cur] : (const uint32_t*)nullptr, n, head);
        perm = sb.val[sb.cur];                                 // the sorted values are the permutation: the buffer is kept
        sb.val[sb.cur] = nullptr;
        if (sorted_keys && width <= 8 && !zoff) { *sorted_keys = sb.key[sb.cur]; sb.key[sb.cur] = nullptr; }
        UQB_TRY(uqb_sortbuf_free(ctx, &sb));
    }
    // ---- refinement ----
    // Every round: group heads -> per-group common prefix with the first row (k_group_lcp: identical-row groups end here)
    // -> groups of up to 32 rows are completed by one warp each -> the rows of larger groups are sorted by (group, the
    // 8 bytes at the group's common prefix) and the loop repeats for what is still tied.
    if (width > 8) {
        const uint32_t off = 8;                  // after round 0 the rows of a group agree in their first 8 (significant) bytes
        uint32_t *headpos, *glcp, *act = nullptr, *apos = nullptr;
        uint8_t* done;
        unsigned long long* d_large;
        UQB_TRY(uqb_dalloc_t(ctx, &headpos, n + 1));
        UQB_TRY(uqb_dalloc_t(ctx, &glcp, n));
        UQB_TRY(uqb_dalloc_t(ctx, &done, n));
        UQB_TRY(uqb_dalloc_t(ctx, &d_large, 1));
        UQB_CUDA(cudaMemsetAsync(done, 0, n, ctx->stream));
        const uint32_t max_rounds = (width + 7) / 8 + 1;
        bool finished = false;
        if (width - off <= 128 && !zoff) {
            // first pass: whole small groups packed 32 rows to a warp, boundaries straight from the head flags
            const uint32_t rem = width - off, pitch = (rem + 3) / 4;
            uint32_t* head2;
            UQB_TRY(uqb_dalloc_t(ctx, &head2, n));
            UQB_CUDA(cudaMemcpyAsync(head2, head, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            UQB_CUDA(cudaMemsetAsync(d_large, 0, 8, ctx->stream));
            const size_t smem = (size_t)(ST / 32) * 32 * pitch * 4;
            const unsigned grid = uqb_grid(ctx, (n + SGP_CHUNK - 1) / SGP_CHUNK, ST / 32, 16);
            const uint64_t ab = n * ((uint64_t)rem + 13);
            if (pitch <= 8) {
                auto k_small_groups_packed_8 = k_small_groups_packed<8>;
                UQB_LAUNCH_B(ab, k_small_groups_packed_8, grid, ST, smem, rows, width, off, perm, head, head2, done, n, pitch, d_large);
            } else if (pitch <= 16) {
                auto k_small_groups_packed_16 = k_small_groups_packed<16>;
                UQB_LAUNCH_B(ab, k_small_groups_packed_16, grid, ST, smem, rows, width, off, perm, head, head2, done, n, pitch, d_large);
            } else {
                auto k_small_groups_packed_32 = k_small_groups_packed<32>;
                UQB_LAUNCH_B(ab, k_small_groups_packed_32, grid, ST, smem, rows, width, off, perm, head, head2, done, n, pitch, d_large);
            }
            UQB_TRY(uqb_dfree(ctx, head, n * 4));
            head = head2;
            unsigned long long large = 0;
            UQB_TRY(uqb_readback(ctx, &large, d_large, 8));
            finished = large == 0;
        }
        for (uint32_t round = 0; round < max_rounds && !finished; round++) {
            UQB_TRY(uqb_scan_u32(ctx, head, excl, n, d_tot));
            UQB_LAUNCH(k_headpos, nb, ST, 0, head, excl, n, headpos, glcp);
            const uint32_t rem = width - off;
            // tie groups of up to 32 rows are finished right here
            UQB_CUDA(cudaMemsetAsync(d_large, 0, 8, ctx->stream));
            const unsigned sg_grid = uqb_grid(ctx, n, ST, 16);
            if (rem <= SG_STAGE_BYTES && !zoff) {
                const uint32_t pitch = (rem + 3) / 4;
                const size_t smem = (size_t)(ST / 32) * (SG_MAX * pitch + 64) * 4;
                if (pitch <= 8) {
                    auto k_small_groups_8 = k_small_groups<8, 1>;
                    UQB_LAUNCH(k_small_groups_8, sg_grid, ST, smem, rows, width, off, perm, head, done, headpos, d_tot, pitch, d_large);
                } else if (pitch <= 16) {
                    auto k_small_groups_16 = k_small_groups<16, 1>;
                    UQB_LAUNCH(k_small_groups_16, sg_grid, ST, smem, rows, width, off, perm, head, done, headpos, d_tot, pitch, d_large);
                } else if (pitch <= 32) {
                    auto k_small_groups_32 = k_small_groups<32, 1>;
                    UQB_CUDA(cudaFuncSetAttribute(k_small_groups_32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                    UQB_LAUNCH(k_small_groups_32, sg_grid, ST, smem, rows, width, off, perm, head, done, headpos, d_tot, pitch, d_large);
                } else {
                    auto k_small_groups_64 = k_small_groups<32, 2>;
                    UQB_CUDA(cudaFuncSetAttribute(k_small_groups_64, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                    UQB_LAUNCH(k_small_groups_64, sg_grid, ST, smem, rows, width, off, perm, head, done, headpos, d_tot, pitch, d_large);
                }
            } else {
                UQB_LAUNCH(k_small_groups_gmem, sg_grid, ST, 0, rows, width, off, zoff, perm, head, done, headpos, d_tot, d_large);
            }
            unsigned long long large = 0;
            UQB_TRY(uqb_readback(ctx, &large, d_large, 8));
            if (large == 0) break;                                 // no tie group of more than 32 rows is left
            // large tie groups: common prefix with the group's first row (identical-row groups end here), then one 8-byte
            // radix round at each group's own common prefix over the still active rows
            const uint64_t ab_lcp = n * ((uint64_t)rem + 16);
            if (rem <= 32) {
                auto k_group_lcp_8 = k_group_lcp<8>;
                UQB_LAUNCH_B(ab_lcp, k_group_lcp_8, uqb_grid(ctx, n, ST, 16), ST, 0, rows, width, off, zoff, perm, head, excl, headpos, done, n, glcp);
            } else {
                auto k_group_lcp_32 = k_group_lcp<32>;
                UQB_LAUNCH_B(ab_lcp, k_group_lcp_32, uqb_grid(ctx, n, ST, 16), ST, 0, rows, width, off, zoff, perm, head, excl, headpos, done, n, glcp);
            }
            if (!act) {
                UQB_TRY(uqb_dalloc_t(ctx, &act, n));
                UQB_TRY(uqb_dalloc_t(ctx, &apos, n));
            }
            UQB_LAUNCH(k_active_flags, nb, ST, 0, head, excl, glcp, done, n, act);
            UQB_TRY(uqb_scan_u32(ctx, act, apos, n, d_tot + 1));
            uint32_t tot[2];
            UQB_TRY(uqb_readback(ctx, tot, d_tot, 8));
            const uint64_t m = tot[1];
            if (m == 0) break;
            uqb_sortbuf sb;
            uint32_t* pos_list;
            UQB_TRY(uqb_sortbuf_alloc(ctx, &sb, m, true));
            UQB_TRY(uqb_dalloc_t(ctx, &pos_list, m));
            UQB_LAUNCH_B(n * 8 + m * 32, k_compact_active, nb, ST, 0, rows, width, glcp, zoff, act, apos, head, excl, perm, n, pos_list, sb.key[0], sb.aux[0], sb.val[0]);
            UQB_TRY(uqb_radix_sort(ctx, &sb, m, true));
            UQB_LAUNCH_B(m * 28, k_write_back, uqb_blocks(m, ST), ST, 0, sb.key[sb.cur], sb.aux[sb.cur], sb.val[sb.cur], pos_list, m, perm, head);
            UQB_TRY(uqb_dfree(ctx, pos_list, m * 4));
            UQB_TRY(uqb_sortbuf_free(ctx, &sb));
        }
        UQB_TRY(uqb_dfree(ctx, headpos, (n + 1) * 4));
        UQB_TRY(uqb_dfree(ctx, glcp, n * 4));
        if (act) { UQB_TRY(uqb_dfree(ctx, act, n * 4)); UQB_TRY(uqb_dfree(ctx, apos, n * 4)); }
        UQB_TRY(uqb_dfree(ctx, done, n));
        UQB_TRY(uqb_dfree(ctx, d_large, 8));
    }
    if (zoff) UQB_TRY(uqb_dfree(ctx, zoff, n * 4));
    // ---- group ids in sorted order ----
    UQB_TRY(uqb_scan_u32(ctx, head, excl, n, d_tot));
    UQB_LAUNCH(k_gid_from_scan, nb, ST, 0, head, excl, n);
    uint32_t u;
    UQB_TRY(uqb_readback(ctx, &u, d_tot, 4));
    UQB_TRY(uqb_dfree(ctx, d_tot, 8));
    UQB_TRY(uqb_dfree(ctx, head, n * 4));
    *d_perm = perm;
    *d_gid_sorted = excl;
    *n_unique = u;
    return 0;
}

// ---- public entry points -----------------------------------------------------------------------
__global__ void __launch_bounds__(ST) k_scatter_key(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ gid, uint64_t n,
                                                   uint32_t* __restrict__ key) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    key[perm[p]] = gid[p];
}

// key[perm[p]] = gid[p] for all p
static int scatter_key(uqb_ctx* ctx, const uint32_t* perm, const uint32_t* gid, uint64_t n, uint32_t* key) {
    if (n == 0) return 0;
    const uint32_t wshift = 23;                                    // 8 M entries = 32 MB per window
    if (n <= (3ull << wshift)) {
        UQB_LAUNCH_B(n * 12, k_scatter_key, uqb_blocks(n, ST), ST, 0, perm, gid, n, key);
        return 0;
    }
    return uqb_scatter_pairs_u32(ctx, perm, gid, n, key);          // regrouped by window first: 3 sweeps instead of one per window
}

__global__ void __launch_bounds__(ST) k_first_of_group(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ gid, uint64_t n,
                                                      uint32_t* __restrict__ first_row) {
    uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x;
    if (p >= n) return;
    if (p == 0 || gid[p] != gid[p - 1]) first_row[gid[p]] = perm[p];
}

// rows of up to 8 bytes: unique row g = the leading `width` bytes of the (big-endian) sorted key at the first position of
// group g.  Sequential reads, stores that advance with the positions.
__global__ void __launch_bounds__(ST) k_uniq_from_keys(const uint64_t* __restrict__ skey, const uint32_t* __restrict__ gid, uint64_t n,
                                                      uint32_t width, uint8_t* __restrict__ out) {
    for (uint64_t p = (uint64_t)blockIdx.x * ST + threadIdx.x; p < n; p += (uint64_t)gridDim.x * ST) {
        const uint32_t g = gid[p];
        if (p && gid[p - 1] == g) continue;
        const uint64_t k = skey[p];
        uint8_t* o = out + (uint64_t)g * width;
        for (uint32_t b = 0; b < width; b++) o[b] = (uint8_t)(k >> (56 - 8 * b));
    }
}

// out[i][:] = table[idx[i]][:]; one warp per row: the index is read once per row, the row bytes are
// contiguous loads and the output rows are contiguous stores
__global__ void __launch_bounds__(ST) k_gather_rows(const uint8_t* __restrict__ table, uint32_t width, const uint32_t* __restrict__ idx,
                                                   uint64_t nrows, uint8_t* __restrict__ out) {
    const unsigned lane = threadIdx.x & 31u;
    const uint64_t wstride = (uint64_t)gridDim.x * (ST / 32);
    for (uint64_t i = (uint64_t)blockIdx.x * (ST / 32) + (threadIdx.x >> 5); i < nrows; i += wstride) {
        const uint8_t* src = table + (uint64_t)__ldg(idx + i) * width;
        uint8_t* dst = out + i * width;
        for (uint32_t b = lane; b < width; b += 32) dst[b] = __ldg(src + b);
    }
}

// rows of 17..GR_MAXW bytes: a warp produces the output of 32 consecutive rows, which is ONE contiguous,
// 32-byte aligned range.  Lanes walk that range in 32-bit words (coalesced word stores); the four bytes of
// a word come from one source row or, at a row seam, from two.  Several words per lane are in flight
// (unrolled), so the random row reads overlap.
#define GR_MAXW 1024
__global__ void __launch_bounds__(ST) k_gather_rows32(const uint8_t* __restrict__ table, uint32_t width, uint32_t q128, uint32_t m128,
                                                     const uint32_t* __restrict__ idx, uint64_t nrows, uint8_t* __restrict__ out) {
    __shared__ uint32_t sidx[ST / 32][32];
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint64_t nblk = (nrows + 31) / 32, wstride = (uint64_t)gridDim.x * (ST / 32);
    for (uint64_t blk = (uint64_t)blockIdx.x * (ST / 32) + w; blk < nblk; blk += wstride) {
        const uint64_t i0 = blk * 32;
        const uint32_t nr = (uint32_t)(nrows - i0 < 32 ? nrows - i0 : 32);
        __syncwarp();
        sidx[w][lane] = lane < nr ? __ldg(idx + i0 + lane) : 0u;
        __syncwarp();
        const uint32_t total = nr * width, nwords = total >> 2;
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + i0 * width);
        uint32_t r = (4u * lane) / width, o = 4u * lane - r * width;
#pragma unroll 8
        for (uint32_t k = lane; k < nwords; k += 32) {
            const uint8_t* s = table + (uint64_t)sidx[w][r] * width + o;
            uint32_t v;
            if (o + 4u <= width) {
                // two aligned words + funnel shift (the second one may reach up to 3 bytes past the row: table slack)
                const uint32_t ph = (uint32_t)(uintptr_t)s & 3u;
                const uint32_t* a = reinterpret_cast<const uint32_t*>(s - ph);
                v = __funnelshift_r(__ldg(a), __ldg(a + 1), ph * 8u);
            } else {
                const uint32_t n0 = width - o;                                  // 1..3 bytes from row r, the rest from row r + 1
                const uint8_t* s2 = table + (uint64_t)sidx[w][(r + 1) & 31u] * width;
                v = 0;
#pragma unroll
                for (uint32_t b = 0; b < 4; b++) v |= (uint32_t)(b < n0 ? __ldg(s + b) : __ldg(s2 + (b - n0))) << (8 * b);
            }
            dst[k] = v;
            o += m128; r += q128;
            if (o >= width) { o -= width; r++; }
        }
        if (lane < (total & 3u)) {                                            // last partial word (last block only)
            const uint32_t bo = (nwords << 2) + lane, rr = bo / width;
            out[i0 * width + bo] = __ldg(table + (uint64_t)sidx[w][rr] * width + (bo - rr * width));
        }
    }
}

// rows of 3..16 bytes (not 1, 2, 4, 8): one thread per row reads its row, the CTA's 256 rows are staged in
// shared memory and leave as coalesced 32-bit words
__global__ void __launch_bounds__(ST) k_gather_narrow(const uint8_t* __restrict__ table, uint32_t width, const uint32_t* __restrict__ idx,
                                                     uint64_t nrows, uint8_t* __restrict__ out) {
    __shared__ __align__(16) uint8_t stage[ST * 16];
    const uint64_t nblk = (nrows + ST - 1) / ST;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t i0 = blk * ST, i = i0 + threadIdx.x;
        const uint32_t nr = (uint32_t)(nrows - i0 < ST ? nrows - i0 : ST);
        __syncthreads();
        if (i < nrows) {
            const uint8_t* s = table + (uint64_t)__ldg(idx + i) * width;
            for (uint32_t b = 0; b < width; b++) stage[threadIdx.x * width + b] = __ldg(s + b);
        }
        __syncthreads();
        const uint32_t total = nr * width;
        uint8_t* dst = out + i0 * width;                                      // ST * width bytes per block: 4-byte aligned
        for (uint32_t k = threadIdx.x; k < (total >> 2); k += ST) reinterpret_cast<uint32_t*>(dst)[k] = reinterpret_cast<const uint32_t*>(stage)[k];
        if (threadIdx.x < (total & 3u)) dst[(total & ~3u) + threadIdx.x] = stage[(total & ~3u) + threadIdx.x];
    }
}

// narrow rows (1, 2, 4, 8 bytes): one thread per row, typed loads
template <typename T>
__global__ void __launch_bounds__(ST) k_gather_items(const T* __restrict__ table, const uint32_t* __restrict__ idx, uint64_t n, T* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x; i < n; i += (uint64_t)gridDim.x * ST) out[i] = table[idx[i]];
}

static int gather_rows_impl(uqb_ctx* ctx, const void* table, uint32_t width, const uint32_t* idx, uint64_t n, void* out) {
    if (n == 0 || width == 0) return 0;
    const uint64_t ab = n * (2 * (uint64_t)width + 4);
    const unsigned g = uqb_grid(ctx, n, ST, 16);
    switch (width) {
        case 1: UQB_LAUNCH_B(ab, k_gather_items<uint8_t>, g, ST, 0, (const uint8_t*)table, idx, n, (uint8_t*)out); return 0;
        case 2: UQB_LAUNCH_B(ab, k_gather_items<uint16_t>, g, ST, 0, (const uint16_t*)table, idx, n, (uint16_t*)out); return 0;
        case 4: UQB_LAUNCH_B(ab, k_gather_items<uint32_t>, g, ST, 0, (const uint32_t*)table, idx, n, (uint32_t*)out); return 0;
        case 8: UQB_LAUNCH_B(ab, k_gather_items<uint64_t>, g, ST, 0, (const uint64_t*)table, idx, n, (uint64_t*)out); return 0;
    }
    if ((reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
        if (width <= 16) {
            UQB_LAUNCH_B(ab, k_gather_narrow, uqb_grid(ctx, n, ST, 16), ST, 0, (const uint8_t*)table, width, idx, n, (uint8_t*)out);
            return 0;
        }
        if (width <= GR_MAXW) {
            UQB_LAUNCH_B(ab, k_gather_rows32, uqb_grid(ctx, n, ST, 16), ST, 0, (const uint8_t*)table, width, 128u / width, 128u % width, idx, n, (uint8_t*)out);
            return 0;
        }
    }
    UQB_LAUNCH_B(ab, k_gather_rows, uqb_grid(ctx, n, ST / 32, 16), ST, 0, (const uint8_t*)table, width, idx, n, (uint8_t*)out);
    return 0;
}

extern "C" int uqb_sort_rows(uqb_ctx* ctx, const uqb_array* table, uqb_array** perm, uqb_array** key,
                             uqb_array** key_sorted, uqb_array** uniq, uint64_t* n_unique) {
    uint32_t *d_perm, *d_gid;
    uint64_t u = 0;
    const uint64_t n = table->n;
    uint64_t* skeys = nullptr;
    UQB_TRY(uqb_sort_rows_impl(ctx, (const uint8_t*)table->d, n, table->width, &d_perm, &d_gid, &u, table->key0, uniq ? &skeys : nullptr));
    if (n_unique) *n_unique = u;
    const unsigned nb = uqb_blocks(n, ST);
    if (key) {
        UQB_TRY(uqb_new_array(ctx, n, 4, key));
        UQB_TRY(scatter_key(ctx, d_perm, d_gid, n, (uint32_t*)(*key)->d));
    }
    if (uniq) {
        UQB_TRY(uqb_new_array(ctx, u, table->width, uniq));
        if (skeys) {
            UQB_LAUNCH_B(n * 12 + u * table->width, k_uniq_from_keys, uqb_grid(ctx, n, ST, 16), ST, 0, skeys, d_gid, n, table->width, (uint8_t*)(*uniq)->d);
            UQB_TRY(uqb_dfree(ctx, skeys, n * 8));
        } else if (n && table->width) {
            uint32_t* first_row;
            UQB_TRY(uqb_dalloc_t(ctx, &first_row, u));
            UQB_LAUNCH(k_first_of_group, nb, ST, 0, d_perm, d_gid, n, first_row);
            UQB_TRY(gather_rows_impl(ctx, table->d, table->width, first_row, u, (*uniq)->d));
            UQB_TRY(uqb_dfree(ctx, first_row, u * 4));
        }
    }
    // the two work arrays become the results (no copies)
    if (key_sorted) UQB_TRY(uqb_adopt_array(ctx, d_gid, n, 4, key_sorted));
    else UQB_TRY(uqb_dfree(ctx, d_gid, n * 4));
    if (perm) UQB_TRY(uqb_adopt_array(ctx, d_perm, n, 4, perm));
    else UQB_TRY(uqb_dfree(ctx, d_perm, n * 4));
    return 0;
}

extern "C" int uqb_gather_rows(uqb_ctx* ctx, const uqb_array* table, const uqb_array* perm, uqb_array** out) {
    if (perm->width != 4) return uqb_fail(ctx, "gather_rows: index array must be uint32");
    UQB_TRY(uqb_new_array(ctx, perm->n, table->width, out));
    UQB_TRY(gather_rows_impl(ctx, table->d, table->width, (const uint32_t*)perm->d, perm->n, (*out)->d));
    return 0;
}

template <typename T>
__global__ void __launch_bounds__(ST) k_narrow(const uint32_t* __restrict__ in, uint64_t n, T* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x; i < n; i += (uint64_t)gridDim.x * ST) out[i] = (T)in[i];
}

extern "C" int uqb_narrow_u32(uqb_ctx* ctx, const uqb_array* a, uint32_t itemsize, uqb_array** out) {
    if (a->width != 4) return uqb_fail(ctx, "narrow: input must be uint32");
    UQB_TRY(uqb_new_array(ctx, a->n, itemsize, out));
    if (a->n == 0) return 0;
    unsigned g = uqb_grid(ctx, a->n, ST, 16);
    const uint32_t* in = (const uint32_t*)a->d;
    switch (itemsize) {
        case 1: UQB_LAUNCH(k_narrow<uint8_t>, g, ST, 0, in, a->n, (uint8_t*)(*out)->d); break;
        case 2: UQB_LAUNCH(k_narrow<uint16_t>, g, ST, 0, in, a->n, (uint16_t*)(*out)->d); break;
        case 4: UQB_LAUNCH(k_narrow<uint32_t>, g, ST, 0, in, a->n, (uint32_t*)(*out)->d); break;
        case 8: UQB_LAUNCH(k_narrow<uint64_t>, g, ST, 0, in, a->n, (uint64_t*)(*out)->d); break;
        default: return uqb_fail(ctx, "narrow: itemsize %u", itemsize);
    }
    return 0;
}

// Index arrays read from a container (DNA.key / QUAL.key / QNAME.key, uq.py:953, 957, 973) are widened to uint32 and
// checked against the size of the table they index: a malformed file must not turn into an out-of-bounds gather.
template <typename T>
__global__ void __launch_bounds__(ST) k_index_u32(const T* __restrict__ in, uint64_t n, uint64_t bound, uint32_t* __restrict__ out,
                                                 unsigned long long* __restrict__ first_bad) {
    unsigned long long bad = ~0ull;
    for (uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x; i < n; i += (uint64_t)gridDim.x * ST) {
        const unsigned long long v = (unsigned long long)in[i];
        if (v >= bound) { if (i < bad) bad = i; out[i] = 0u; }
        else out[i] = (uint32_t)v;
    }
    if (bad != ~0ull) atomicMin(first_bad, bad);
}

extern "C" int uqb_index_u32(uqb_ctx* ctx, const uqb_array* a, uint64_t bound, uqb_array** out, int64_t* first_bad) {
    if (bound > (1ull << 32)) return uqb_fail(ctx, "index_u32: tables of more than 2^32 rows are not supported");
    UQB_TRY(uqb_new_array(ctx, a->n, 4, out));
    *first_bad = -1;
    if (a->n == 0) return 0;
    unsigned long long* d_bad;
    UQB_TRY(uqb_dalloc_t(ctx, &d_bad, 1));
    UQB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 8, ctx->stream));
    const unsigned g = uqb_grid(ctx, a->n, ST, 16);
    uint32_t* o = (uint32_t*)(*out)->d;
    switch (a->width) {
        case 1: UQB_LAUNCH_B(a->n * 5, k_index_u32<uint8_t>, g, ST, 0, (const uint8_t*)a->d, a->n, bound, o, d_bad); break;
        case 2: UQB_LAUNCH_B(a->n * 6, k_index_u32<uint16_t>, g, ST, 0, (const uint16_t*)a->d, a->n, bound, o, d_bad); break;
        case 4: UQB_LAUNCH_B(a->n * 8, k_index_u32<uint32_t>, g, ST, 0, (const uint32_t*)a->d, a->n, bound, o, d_bad); break;
        case 8: UQB_LAUNCH_B(a->n * 12, k_index_u32<uint64_t>, g, ST, 0, (const uint64_t*)a->d, a->n, bound, o, d_bad); break;
        default: UQB_TRY(uqb_dfree(ctx, d_bad, 8)); return uqb_fail(ctx, "index_u32: itemsize %u", a->width);
    }
    unsigned long long h = 0;
    UQB_TRY(uqb_readback(ctx, &h, d_bad, 8));
    UQB_TRY(uqb_dfree(ctx, d_bad, 8));
    if (h != ~0ull) *first_bad = (int64_t)h;
    return 0;
}

// ---- QNAME columns <-> big-endian key rows -------------------------------------------------------
struct col_desc { const uint8_t* p[UQB_MAX_COLS]; uint32_t size[UQB_MAX_COLS]; uint32_t off[UQB_MAX_COLS]; uint32_t ncols; uint32_t width; };
struct col_desc_out { uint8_t* p[UQB_MAX_COLS]; uint32_t size[UQB_MAX_COLS]; uint32_t off[UQB_MAX_COLS]; uint32_t ncols; uint32_t width; };

__global__ void __launch_bounds__(ST) k_cols_to_rows(col_desc cd, uint64_t n, uint8_t* __restrict__ rows) {
    for (uint64_t t = (uint64_t)blockIdx.x * ST + threadIdx.x; t < n * cd.ncols; t += (uint64_t)gridDim.x * ST) {
        uint64_t r = t / cd.ncols;
        uint32_t c = (uint32_t)(t - r * cd.ncols);
        uint32_t sz = cd.size[c];
        const uint8_t* src = cd.p[c] + r * sz;
        uint8_t* dst = rows + r * cd.width + cd.off[c];
        for (uint32_t b = 0; b < sz; b++) dst[b] = src[sz - 1 - b];      // little-endian value -> big-endian key bytes
    }
}

__global__ void __launch_bounds__(ST) k_rows_to_cols(col_desc_out cd, uint64_t n, const uint8_t* __restrict__ rows) {
    for (uint64_t t = (uint64_t)blockIdx.x * ST + threadIdx.x; t < n * cd.ncols; t += (uint64_t)gridDim.x * ST) {
        uint64_t r = t / cd.ncols;
        uint32_t c = (uint32_t)(t - r * cd.ncols);
        uint32_t sz = cd.size[c];
        uint8_t* dst = cd.p[c] + r * sz;
        const uint8_t* src = rows + r * cd.width + cd.off[c];
        for (uint32_t b = 0; b < sz; b++) dst[b] = src[sz - 1 - b];
    }
}

// Rows of up to CR_MAXW bytes: one thread per ROW.  Column values are read / written with typed, coalesced
// accesses, the rows of the CTA pass through shared memory, and the row table side is one contiguous range moved
// as 32-bit words.
#define CR_MAXW 64
template <typename T>
__device__ __forceinline__ unsigned long long cr_load(const uint8_t* p, uint64_t r) { return (unsigned long long)reinterpret_cast<const T*>(p)[r]; }

__global__ void __launch_bounds__(ST) k_cols_to_rows_staged(col_desc cd, uint64_t n, uint8_t* __restrict__ rows) {
    __shared__ __align__(16) uint8_t stage[ST * CR_MAXW];
    const uint64_t nblk = (n + ST - 1) / ST;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t r0 = blk * ST, r = r0 + threadIdx.x;
        const uint32_t nr = (uint32_t)(n - r0 < ST ? n - r0 : ST);
        __syncthreads();
        if (r < n) {
            uint8_t* dst = stage + threadIdx.x * cd.width;
            for (uint32_t c = 0; c < cd.ncols; c++) {
                const uint32_t sz = cd.size[c];
                const unsigned long long v = sz == 1 ? cr_load<uint8_t>(cd.p[c], r) : sz == 2 ? cr_load<uint16_t>(cd.p[c], r)
                                           : sz == 4 ? cr_load<uint32_t>(cd.p[c], r) : cr_load<uint64_t>(cd.p[c], r);
                for (uint32_t b = 0; b < sz; b++) dst[cd.off[c] + b] = (uint8_t)(v >> (8 * (sz - 1 - b)));   // big-endian key bytes
            }
        }
        __syncthreads();
        const uint32_t total = nr * cd.width;
        uint8_t* out = rows + r0 * cd.width;                                  // ST * width bytes per block: 4-byte aligned
        for (uint32_t k = threadIdx.x; k < (total >> 2); k += ST) reinterpret_cast<uint32_t*>(out)[k] = reinterpret_cast<const uint32_t*>(stage)[k];
        if (threadIdx.x < (total & 3u)) out[(total & ~3u) + threadIdx.x] = stage[(total & ~3u) + threadIdx.x];
    }
}

__global__ void __launch_bounds__(ST) k_rows_to_cols_staged(col_desc_out cd, uint64_t n, const uint8_t* __restrict__ rows) {
    __shared__ __align__(16) uint8_t stage[ST * CR_MAXW];
    const uint64_t nblk = (n + ST - 1) / ST;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t r0 = blk * ST, r = r0 + threadIdx.x;
        const uint32_t nr = (uint32_t)(n - r0 < ST ? n - r0 : ST);
        const uint32_t total = nr * cd.width;
        const uint8_t* in = rows + r0 * cd.width;
        __syncthreads();
        for (uint32_t k = threadIdx.x; k < (total >> 2); k += ST) reinterpret_cast<uint32_t*>(stage)[k] = reinterpret_cast<const uint32_t*>(in)[k];
        if (threadIdx.x < (total & 3u)) stage[(total & ~3u) + threadIdx.x] = in[(total & ~3u) + threadIdx.x];
        __syncthreads();
        if (r < n) {
            const uint8_t* src = stage + threadIdx.x * cd.width;
            for (uint32_t c = 0; c < cd.ncols; c++) {
                const uint32_t sz = cd.size[c];
                unsigned long long v = 0;
                for (uint32_t b = 0; b < sz; b++) v = (v << 8) | src[cd.off[c] + b];
                if (sz == 1) reinterpret_cast<uint8_t*>(cd.p[c])[r] = (uint8_t)v;
                else if (sz == 2) reinterpret_cast<uint16_t*>(cd.p[c])[r] = (uint16_t)v;
                else if (sz == 4) reinterpret_cast<uint32_t*>(cd.p[c])[r] = (uint32_t)v;
                else reinterpret_cast<uint64_t*>(cd.p[c])[r] = v;
            }
        }
    }
}

// ---- the same transforms with byte columns (kind 1: 'strings' QNAME columns, E1) -------------------------------
// A byte column enters the row as it is: memcmp of its zero-padded bytes is numpy's order of S values.  Bit c of
// `bytes_mask` marks column c as such a column.  These kernels are separate from the ones above so that tables of
// integer columns only keep exactly the kernels they always had.
__global__ void __launch_bounds__(ST) k_cols_to_rows_mixed(col_desc cd, uint64_t bytes_mask, uint64_t n, uint8_t* __restrict__ rows) {
    for (uint64_t t = (uint64_t)blockIdx.x * ST + threadIdx.x; t < n * cd.ncols; t += (uint64_t)gridDim.x * ST) {
        uint64_t r = t / cd.ncols;
        uint32_t c = (uint32_t)(t - r * cd.ncols);
        uint32_t sz = cd.size[c];
        const uint8_t* src = cd.p[c] + r * sz;
        uint8_t* dst = rows + r * cd.width + cd.off[c];
        if ((bytes_mask >> c) & 1ull) for (uint32_t b = 0; b < sz; b++) dst[b] = src[b];
        else                          for (uint32_t b = 0; b < sz; b++) dst[b] = src[sz - 1 - b];
    }
}

__global__ void __launch_bounds__(ST) k_rows_to_cols_mixed(col_desc_out cd, uint64_t bytes_mask, uint64_t n, const uint8_t* __restrict__ rows) {
    for (uint64_t t = (uint64_t)blockIdx.x * ST + threadIdx.x; t < n * cd.ncols; t += (uint64_t)gridDim.x * ST) {
        uint64_t r = t / cd.ncols;
        uint32_t c = (uint32_t)(t - r * cd.ncols);
        uint32_t sz = cd.size[c];
        uint8_t* dst = cd.p[c] + r * sz;
        const uint8_t* src = rows + r * cd.width + cd.off[c];
        if ((bytes_mask >> c) & 1ull) for (uint32_t b = 0; b < sz; b++) dst[b] = src[b];
        else                          for (uint32_t b = 0; b < sz; b++) dst[b] = src[sz - 1 - b];
    }
}

// Staged form: integer columns as in k_cols_to_rows_staged (one thread per row, typed loads); a byte column's values of
// the CTA's rows are one contiguous range of nr * size bytes, which all threads copy together (coalesced) into the rows.
__global__ void __launch_bounds__(ST) k_cols_to_rows_staged_mixed(col_desc cd, uint64_t bytes_mask, uint64_t n, uint8_t* __restrict__ rows) {
    __shared__ __align__(16) uint8_t stage[ST * CR_MAXW];
    const uint64_t nblk = (n + ST - 1) / ST;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t r0 = blk * ST, r = r0 + threadIdx.x;
        const uint32_t nr = (uint32_t)(n - r0 < ST ? n - r0 : ST);
        __syncthreads();
        for (uint32_t c = 0; c < cd.ncols; c++) {
            const uint32_t sz = cd.size[c];
            if ((bytes_mask >> c) & 1ull) {
                const uint8_t* src = cd.p[c] + r0 * sz;
                for (uint32_t k = threadIdx.x; k < nr * sz; k += ST) {
                    const uint32_t i = k / sz;
                    stage[i * cd.width + cd.off[c] + (k - i * sz)] = src[k];
                }
            } else if (r < n) {
                uint8_t* dst = stage + threadIdx.x * cd.width;
                const unsigned long long v = sz == 1 ? cr_load<uint8_t>(cd.p[c], r) : sz == 2 ? cr_load<uint16_t>(cd.p[c], r)
                                           : sz == 4 ? cr_load<uint32_t>(cd.p[c], r) : cr_load<uint64_t>(cd.p[c], r);
                for (uint32_t b = 0; b < sz; b++) dst[cd.off[c] + b] = (uint8_t)(v >> (8 * (sz - 1 - b)));   // big-endian key bytes
            }
        }
        __syncthreads();
        const uint32_t total = nr * cd.width;
        uint8_t* out = rows + r0 * cd.width;                                  // ST * width bytes per block: 4-byte aligned
        for (uint32_t k = threadIdx.x; k < (total >> 2); k += ST) reinterpret_cast<uint32_t*>(out)[k] = reinterpret_cast<const uint32_t*>(stage)[k];
        if (threadIdx.x < (total & 3u)) out[(total & ~3u) + threadIdx.x] = stage[(total & ~3u) + threadIdx.x];
    }
}

__global__ void __launch_bounds__(ST) k_rows_to_cols_staged_mixed(col_desc_out cd, uint64_t bytes_mask, uint64_t n, const uint8_t* __restrict__ rows) {
    __shared__ __align__(16) uint8_t stage[ST * CR_MAXW];
    const uint64_t nblk = (n + ST - 1) / ST;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t r0 = blk * ST, r = r0 + threadIdx.x;
        const uint32_t nr = (uint32_t)(n - r0 < ST ? n - r0 : ST);
        const uint32_t total = nr * cd.width;
        const uint8_t* in = rows + r0 * cd.width;
        __syncthreads();
        for (uint32_t k = threadIdx.x; k < (total >> 2); k += ST) reinterpret_cast<uint32_t*>(stage)[k] = reinterpret_cast<const uint32_t*>(in)[k];
        if (threadIdx.x < (total & 3u)) stage[(total & ~3u) + threadIdx.x] = in[(total & ~3u) + threadIdx.x];
        __syncthreads();
        for (uint32_t c = 0; c < cd.ncols; c++) {
            const uint32_t sz = cd.size[c];
            if ((bytes_mask >> c) & 1ull) {
                uint8_t* dst = cd.p[c] + r0 * sz;
                for (uint32_t k = threadIdx.x; k < nr * sz; k += ST) {
                    const uint32_t i = k / sz;
                    dst[k] = stage[i * cd.width + cd.off[c] + (k - i * sz)];
                }
            } else if (r < n) {
                const uint8_t* src = stage + threadIdx.x * cd.width;
                unsigned long long v = 0;
                for (uint32_t b = 0; b < sz; b++) v = (v << 8) | src[cd.off[c] + b];
                if (sz == 1) reinterpret_cast<uint8_t*>(cd.p[c])[r] = (uint8_t)v;
                else if (sz == 2) reinterpret_cast<uint16_t*>(cd.p[c])[r] = (uint16_t)v;
                else if (sz == 4) reinterpret_cast<uint32_t*>(cd.p[c])[r] = (uint32_t)v;
                else reinterpret_cast<uint64_t*>(cd.p[c])[r] = v;
            }
        }
    }
}

// kinds == NULL or all 0: integer columns only
static int cr_bytes_mask(uqb_ctx* ctx, const uint8_t* kinds, uint32_t ncols, uint64_t* mask) {
    *mask = 0;
    if (!kinds) return 0;
    for (uint32_t c = 0; c < ncols; c++) {
        if (kinds[c] > 1) return uqb_fail(ctx, "columns/rows: column %u has kind %u (0 integer, 1 bytes)", c, kinds[c]);
        if (kinds[c]) *mask |= 1ull << c;
    }
    return 0;
}

static bool cr_staged_ok(const uint32_t* sizes, uint32_t ncols, uint32_t width, const void* rows, uint64_t bytes_mask = 0) {
    if (width > CR_MAXW || (reinterpret_cast<uintptr_t>(rows) & 3u)) return false;
    for (uint32_t c = 0; c < ncols; c++)
        if (!((bytes_mask >> c) & 1ull) && sizes[c] != 1 && sizes[c] != 2 && sizes[c] != 4 && sizes[c] != 8) return false;
    return true;
}

extern "C" int uqb_columns_to_rows(uqb_ctx* ctx, uint32_t ncols, uqb_array* const* cols, uqb_array** rows) {
    return uqb_columns_to_rows_ex(ctx, ncols, cols, nullptr, rows);
}

extern "C" int uqb_columns_to_rows_ex(uqb_ctx* ctx, uint32_t ncols, uqb_array* const* cols, const uint8_t* kinds, uqb_array** rows) {
    if (ncols == 0 || ncols > UQB_MAX_COLS) return uqb_fail(ctx, "columns_to_rows: bad column count %u", ncols);
    uint64_t bm;
    UQB_TRY(cr_bytes_mask(ctx, kinds, ncols, &bm));
    col_desc cd;
    cd.ncols = ncols;
    uint32_t w = 0;
    uint64_t n = cols[0]->n;
    for (uint32_t c = 0; c < ncols; c++) {
        if (cols[c]->n != n) return uqb_fail(ctx, "columns_to_rows: ragged columns");
        cd.p[c] = (const uint8_t*)cols[c]->d; cd.size[c] = cols[c]->width; cd.off[c] = w; w += cols[c]->width;
    }
    cd.width = w;
    UQB_TRY(uqb_new_array(ctx, n, w, rows));
    if (bm) {
        if (n && cr_staged_ok(cd.size, ncols, w, (*rows)->d, bm)) UQB_LAUNCH_B(2 * n * w, k_cols_to_rows_staged_mixed, uqb_grid(ctx, n, ST, 16), ST, 0, cd, bm, n, (uint8_t*)(*rows)->d);
        else if (n) UQB_LAUNCH_B(2 * n * w, k_cols_to_rows_mixed, uqb_grid(ctx, n * ncols, ST, 16), ST, 0, cd, bm, n, (uint8_t*)(*rows)->d);
        return 0;
    }
    if (n && cr_staged_ok(cd.size, ncols, w, (*rows)->d)) UQB_LAUNCH_B(2 * n * w, k_cols_to_rows_staged, uqb_grid(ctx, n, ST, 16), ST, 0, cd, n, (uint8_t*)(*rows)->d);
    else if (n) UQB_LAUNCH(k_cols_to_rows, uqb_grid(ctx, n * ncols, ST, 16), ST, 0, cd, n, (uint8_t*)(*rows)->d);
    return 0;
}

extern "C" int uqb_rows_to_columns(uqb_ctx* ctx, const uqb_array* rows, uint32_t ncols, const uint32_t* itemsizes, uqb_array** cols) {
    return uqb_rows_to_columns_ex(ctx, rows, ncols, itemsizes, nullptr, cols);
}

extern "C" int uqb_rows_to_columns_ex(uqb_ctx* ctx, const uqb_array* rows, uint32_t ncols, const uint32_t* itemsizes, const uint8_t* kinds,
                                      uqb_array** cols) {
    if (ncols == 0 || ncols > UQB_MAX_COLS) return uqb_fail(ctx, "rows_to_columns: bad column count %u", ncols);
    uint64_t bm;
    UQB_TRY(cr_bytes_mask(ctx, kinds, ncols, &bm));
    col_desc_out cd;
    cd.ncols = ncols;
    uint32_t w = 0;
    for (uint32_t c = 0; c < ncols; c++) {
        UQB_TRY(uqb_new_array(ctx, rows->n, itemsizes[c], &cols[c]));
        cd.p[c] = (uint8_t*)cols[c]->d; cd.size[c] = itemsizes[c]; cd.off[c] = w; w += itemsizes[c];
    }
    cd.width = w;
    if (w != rows->width) return uqb_fail(ctx, "rows_to_columns: widths sum to %u, rows are %u wide", w, rows->width);
    if (bm) {
        if (rows->n && cr_staged_ok(cd.size, ncols, w, rows->d, bm)) UQB_LAUNCH_B(2 * rows->n * w, k_rows_to_cols_staged_mixed, uqb_grid(ctx, rows->n, ST, 16), ST, 0, cd, bm, rows->n, (const uint8_t*)rows->d);
        else if (rows->n) UQB_LAUNCH_B(2 * rows->n * w, k_rows_to_cols_mixed, uqb_grid(ctx, rows->n * ncols, ST, 16), ST, 0, cd, bm, rows->n, (const uint8_t*)rows->d);
        return 0;
    }
    if (rows->n && cr_staged_ok(cd.size, ncols, w, rows->d)) UQB_LAUNCH_B(2 * rows->n * w, k_rows_to_cols_staged, uqb_grid(ctx, rows->n, ST, 16), ST, 0, cd, rows->n, (const uint8_t*)rows->d);
    else if (rows->n) UQB_LAUNCH(k_rows_to_cols, uqb_grid(ctx, rows->n * ncols, ST, 16), ST, 0, cd, rows->n, (const uint8_t*)rows->d);
    return 0;
}

// ---- multi-GPU sample sort support ---------------------------------------------------------------
// lower_bound of k probe rows in a table sorted in memcmp order: out[j] = first i with table[i] >= probe[j]
__global__ void k_rows_lower_bound(const uint8_t* __restrict__ table, uint64_t n, uint32_t width, const uint8_t* __restrict__ probes,
                                   uint32_t k, uint64_t* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const uint8_t* p = probes + (uint64_t)j * width;
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        const uint8_t* row = table + mid * width;
        int c = 0;
        for (uint32_t b = 0; b < width; b++) {
            const unsigned x = row[b], y = p[b];
            if (x != y) { c = x < y ? -1 : 1; break; }
        }
        if (c < 0) lo = mid + 1; else hi = mid;
    }
    out[j] = lo;
}

extern "C" int uqb_rows_lower_bound(uqb_ctx* ctx, const uqb_array* sorted_table, const uint8_t* probes_host, uint32_t k, uint64_t* out_host) {
    if (k == 0) return 0;
    const uint32_t w = sorted_table->width;
    uint8_t* dp;
    uint64_t* dout;
    UQB_TRY(uqb_dalloc(ctx, (void**)&dp, (size_t)k * w + 16));
    UQB_TRY(uqb_dalloc_t(ctx, &dout, k));
    UQB_CUDA(cudaMemcpyAsync(dp, probes_host, (size_t)k * w, cudaMemcpyHostToDevice, ctx->stream));
    UQB_LAUNCH(k_rows_lower_bound, (k + 63) / 64, 64, 0, (const uint8_t*)sorted_table->d, sorted_table->n, w, dp, k, dout);
    UQB_TRY(uqb_readback(ctx, out_host, dout, (size_t)k * 8));
    UQB_TRY(uqb_dfree(ctx, dp, 0));
    UQB_TRY(uqb_dfree(ctx, dout, 0));
    return 0;
}

// ---- multi-GPU sample sort: exchange buffers (the partition is uqb_partition_positions, partition.cu) ------------
// Row exchange buffers: NCCL's send/recv path only moves 16 bytes per thread when both user pointers are 16-byte
// aligned, and the per-peer segments of a table of 113-byte rows start anywhere.  The rows of segment d
// (order[first_d .. first_d + count_d)) are therefore gathered into a byte buffer in which every segment starts at a
// multiple of `align` bytes; the receiver uses the same layout and closes the gaps afterwards (uqb_compact_segments).
static inline uint64_t seg_round(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

extern "C" int uqb_gather_rows_segmented(uqb_ctx* ctx, const uqb_array* table, const uqb_array* order, uint32_t nseg,
                                         const uint64_t* seg_counts_host, uint32_t align, uqb_array** out, uint64_t* seg_offsets_host) {
    if (order->width != 4) return uqb_fail(ctx, "gather_rows_segmented: index array must be uint32");
    if (align == 0 || (align & 3u)) return uqb_fail(ctx, "gather_rows_segmented: alignment must be a multiple of 4");
    const uint32_t w = table->width;
    uint64_t total = 0, rows = 0;
    for (uint32_t d = 0; d < nseg; d++) {
        seg_offsets_host[d] = total;
        total = seg_round(total + seg_counts_host[d] * w, align);
        rows += seg_counts_host[d];
    }
    if (rows != order->n) return uqb_fail(ctx, "gather_rows_segmented: the segments hold %llu rows, the index array %llu",
                                          (unsigned long long)rows, (unsigned long long)order->n);
    UQB_TRY(uqb_new_array(ctx, total, 1, out));
    uint64_t first = 0;
    for (uint32_t d = 0; d < nseg; d++) {
        UQB_TRY(gather_rows_impl(ctx, table->d, w, (const uint32_t*)order->d + first, seg_counts_host[d], (uint8_t*)(*out)->d + seg_offsets_host[d]));
        first += seg_counts_host[d];
    }
    return 0;
}

// byte buffer with aligned segments (seg_offsets, seg_counts rows of `width` bytes each) -> dense table
extern "C" int uqb_compact_segments(uqb_ctx* ctx, const uqb_array* padded, uint32_t nseg, const uint64_t* seg_offsets_host,
                                    const uint64_t* seg_counts_host, uint32_t width, uqb_array** out) {
    uint64_t rows = 0;
    for (uint32_t d = 0; d < nseg; d++) rows += seg_counts_host[d];
    UQB_TRY(uqb_new_array(ctx, rows, width, out));
    uint64_t first = 0;
    for (uint32_t d = 0; d < nseg; d++) {
        const uint64_t nb = seg_counts_host[d] * width;
        if (seg_offsets_host[d] + nb > padded->nbytes()) return uqb_fail(ctx, "compact_segments: segment %u exceeds the buffer", d);
        if (nb) UQB_CUDA(cudaMemcpyAsync((uint8_t*)(*out)->d + first * width, (const uint8_t*)padded->d + seg_offsets_host[d], nb,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
        first += seg_counts_host[d];
    }
    return 0;
}

__global__ void __launch_bounds__(ST) k_scatter_u32(const uint32_t* __restrict__ src, const uint32_t* __restrict__ idx, uint64_t n,
                                                   uint32_t* __restrict__ out) {
    for (uint64_t j = (uint64_t)blockIdx.x * ST + threadIdx.x; j < n; j += (uint64_t)gridDim.x * ST) out[idx[j]] = src[j];
}

// out[idx[j]] = src[j] (uint32 arrays; idx must be a permutation of 0..n-1): the inverse of uqb_gather_rows
extern "C" int uqb_scatter_u32(uqb_ctx* ctx, const uqb_array* src, const uqb_array* idx, uqb_array** out) {
    if (src->width != 4 || idx->width != 4 || src->n != idx->n) return uqb_fail(ctx, "scatter_u32: two uint32 arrays of one length expected");
    UQB_TRY(uqb_new_array(ctx, src->n, 4, out));
    if (src->n > (3ull << 23)) return uqb_scatter_pairs_u32(ctx, (const uint32_t*)idx->d, (const uint32_t*)src->d, src->n, (uint32_t*)(*out)->d);
    if (src->n) UQB_LAUNCH_B(src->n * 12, k_scatter_u32, uqb_grid(ctx, src->n, ST, 16), ST, 0, (const uint32_t*)src->d, (const uint32_t*)idx->d, src->n,
                             (uint32_t*)(*out)->d);
    return 0;
}

__global__ void __launch_bounds__(ST) k_add_u32(uint32_t* __restrict__ a, uint64_t n, uint32_t v) {
    for (uint64_t i = (uint64_t)blockIdx.x * ST + threadIdx.x; i < n; i += (uint64_t)gridDim.x * ST) a[i] += v;
}

// a[i] += value for a uint32 array (global unique ids = range offset + local id)
extern "C" int uqb_add_scalar_u32(uqb_ctx* ctx, uqb_array* a, uint32_t value) {
    if (a->width != 4) return uqb_fail(ctx, "add_scalar_u32: array must be uint32");
    if (a->n && value) UQB_LAUNCH_B(a->n * 8, k_add_u32, uqb_grid(ctx, a->n, ST, 16), ST, 0, (uint32_t*)a->d, a->n, value);
    return 0;
}
