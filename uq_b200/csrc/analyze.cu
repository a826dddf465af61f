// Stage 1: the Pass-1 statistics of the reference (uq.py:342-425) as device reductions.
//
// Per-record statistics (FASTQ shape checks, read-length min/max, and the QNAME statistics against line 1 from which
// the host reproduces the order-dependent prefix / suffix / separator logic of uq.py:395-413 exactly, see host.py):
//   k_record_stats_names   the product kernel: thread per record, reads offsets + name + '+' only
//   k_record_stats         generic fallback (names longer than 255 bytes, more than 64 distinct bytes in line 1)
// Base and quality byte histograms plus "does this base always carry one single quality" (static_qualities,
// uq.py:369-375, 420-425, read at uq.py:480-494):
//   k_pair_hist_pipe       records that fit shared-memory tiles (TMA tiles in a three-stage pipeline, hist_units.cuh)
//   k_pair_hist_long       long reads, straight from global memory
//   k_pair_hist            generic fallback (bytes outside 32..127)
// Counters are private per thread (packed 8-bit fields in shared memory or registers, flushed before they can
// overflow), so the hot loops have no atomics.
#include "common.cuh"
#include "tile.cuh"

#define AN_THREADS 256
#define MAXCH 128            // distinct byte values of line 1 tracked for separator counting

struct an_dev {
    unsigned long long base_count[256];
    unsigned long long qual_count[256];
    int first_q[256];
    int multi[256];
    unsigned long long dna_min, dna_max;
    long long bad_plus, bad_len;
    unsigned int max_name_len;
    long long last_count_mismatch[256];
    long long first_lcp_eq[UQB_HDR_MAX + 1];
    long long first_lcs_eq[UQB_HDR_MAX + 1];
    long long first_short_prefix[UQB_HDR_MAX + 1];
    long long first_short_suffix[UQB_HDR_MAX + 1];
};

__global__ void k_an_init(an_dev* s) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        s->base_count[i] = 0; s->qual_count[i] = 0; s->first_q[i] = -1; s->multi[i] = 0;
        s->last_count_mismatch[i] = -1;
    }
    for (int i = threadIdx.x; i <= UQB_HDR_MAX; i += blockDim.x) {
        s->first_lcp_eq[i] = LLONG_MAX; s->first_lcs_eq[i] = LLONG_MAX;
        s->first_short_prefix[i] = LLONG_MAX; s->first_short_suffix[i] = LLONG_MAX;
    }
    if (threadIdx.x == 0) {
        s->dna_min = ~0ull; s->dna_max = 0; s->bad_plus = LLONG_MAX; s->bad_len = LLONG_MAX; s->max_name_len = 0;
    }
}

__global__ void __launch_bounds__(AN_THREADS) k_record_stats(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                           uint64_t n_reads, const uint8_t* __restrict__ ref, uint64_t rbase,
                                                           uint32_t first_len, an_dev* __restrict__ s) {
    __shared__ uint8_t first[UQB_HDR_MAX];
    __shared__ uint8_t slot_of[256];          // byte value -> slot in the distinct-char list of line 1
    __shared__ uint8_t slot_char[MAXCH];
    __shared__ uint16_t first_cnt[MAXCH];
    __shared__ int nslots_s;
    __shared__ long long blk_last[MAXCH];
    const unsigned tid = threadIdx.x;
    for (unsigned i = tid; i < first_len; i += AN_THREADS) first[i] = ref[i];
    slot_of[tid] = 255;
    if (tid < MAXCH) { first_cnt[tid] = 0; blk_last[tid] = -1; }
    __syncthreads();
    if (tid == 0) {
        int ns = 0;
        for (unsigned i = 0; i < first_len; i++) {
            uint8_t c = first[i];
            if (slot_of[c] == 255 && ns < MAXCH) { slot_of[c] = (uint8_t)ns; slot_char[ns] = c; ns++; }
            if (slot_of[c] != 255) first_cnt[slot_of[c]]++;
        }
        nslots_s = ns;
    }
    __syncthreads();
    const int nslots = nslots_s;

    const uint64_t r = (uint64_t)blockIdx.x * AN_THREADS + tid;
    const bool active = r < n_reads;
    uint64_t dlen = 0;
    uint16_t cnt[MAXCH];
    unsigned name_len = 0;
    if (active) {
        const uint64_t o0 = line_off[4 * r], o1 = line_off[4 * r + 1], o2 = line_off[4 * r + 2];
        const uint64_t o3 = line_off[4 * r + 3], o4 = line_off[4 * r + 4];
        dlen = o2 - o1 - 1;
        const uint64_t qlen = o4 - o3 - 1;
        if (o3 - o2 < 2 || d[o2] != '+') atomicMin(&s->bad_plus, (long long)r);     // uq.py:360, 382
        if (dlen != qlen) atomicMin(&s->bad_len, (long long)r);                     // uq.py:366, 388
        // ---- QNAME line against line 1 ----
        const uint8_t* name = d + o0;
        const uint64_t nl64 = o1 - o0 - 1;
        name_len = nl64 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (unsigned)nl64;
        for (int i = 0; i < nslots; i++) cnt[i] = 0;
        const unsigned lim = name_len < first_len ? name_len : first_len;
        unsigned lcp = 0;
        bool run = true;
        for (unsigned i = 0; i < name_len; i++) {
            uint8_t c = __ldg(name + i);
            if (run && i < lim && c == first[i]) lcp = i + 1; else run = false;
            uint8_t sl = slot_of[c];
            if (sl != 255) cnt[sl]++;
        }
        unsigned lcs = 0;
        while (lcs < lim && __ldg(name + name_len - 1 - lcs) == first[first_len - 1 - lcs]) lcs++;
        if (r + rbase >= 1) {
            atomicMin(&s->first_lcp_eq[lcp], (long long)r);
            atomicMin(&s->first_lcs_eq[lcs], (long long)r);
            if (lcp == name_len && name_len < first_len) atomicMin(&s->first_short_prefix[name_len], (long long)r);
            if (lcs == name_len && name_len < first_len) atomicMin(&s->first_short_suffix[name_len], (long long)r);
        }
    }
    // last record (highest index) whose count of a tracked byte differs from line 1's count
    for (int i = 0; i < nslots; i++) {
        bool mis = active && cnt[i] != first_cnt[i];
        unsigned m = __ballot_sync(0xffffffffu, mis);
        if (m && lane_id() == 0) {
            long long rr = (long long)((uint64_t)blockIdx.x * AN_THREADS + (tid & ~31u) + (31 - __clz(m)));
            atomicMax(&blk_last[i], rr);
        }
    }
    // block reductions of min / max read length and max name length
    unsigned long long mn = active ? dlen : ~0ull, mx = active ? dlen : 0ull;
    unsigned nm = active ? name_len : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        unsigned c = __shfl_xor_sync(0xffffffffu, nm, o);
        mn = a < mn ? a : mn; mx = b > mx ? b : mx; nm = c > nm ? c : nm;
    }
    if (lane_id() == 0) {
        atomicMin(&s->dna_min, mn);
        atomicMax(&s->dna_max, mx);
        atomicMax(&s->max_name_len, nm);
    }
    __syncthreads();
    if (tid < (unsigned)nslots && blk_last[tid] >= 0) atomicMax(&s->last_count_mismatch[slot_char[tid]], blk_last[tid]);
}

// ---- base / quality histograms -------------------------------------------------------------------
// Private counters: word (v >> 2) of a thread holds four 8-bit counters for byte values 4*(v>>2)..+3.
// Layout priv[word][thread] keeps every access bank-conflict free.  Byte values >= 128 (never seen in
// real FASTQ) take a slow global-atomic path.
#define PH_THREADS 256
#define PH_WORDS 32

__device__ __forceinline__ void ph_flush(unsigned* priv, unsigned* blk_hist, unsigned tid) {
#pragma unroll 4
    for (int w = 0; w < PH_WORDS; w++) {
        unsigned x = priv[w * PH_THREADS + tid];
        if (x) {
            priv[w * PH_THREADS + tid] = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                unsigned c = (x >> (8 * b)) & 255u;
                if (c) atomicAdd(&blk_hist[4 * w + b], c);
            }
        }
    }
}

__global__ void __launch_bounds__(PH_THREADS) k_pair_hist(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                         uint64_t n_reads, an_dev* __restrict__ s) {
    extern __shared__ unsigned ph_smem[];
    unsigned* priv_b = ph_smem;                               // [PH_WORDS][PH_THREADS]
    unsigned* priv_q = ph_smem + PH_WORDS * PH_THREADS;
    unsigned* hist_b = priv_q + PH_WORDS * PH_THREADS;        // [256]
    unsigned* hist_q = hist_b + 256;
    int* first_q = (int*)(hist_q + 256);                      // [256]
    int* multi = first_q + 256;
    const unsigned tid = threadIdx.x, lane = tid & 31u;
    for (unsigned i = tid; i < 2 * PH_WORDS * PH_THREADS; i += PH_THREADS) ph_smem[i] = 0;
    hist_b[tid] = 0; hist_q[tid] = 0; first_q[tid] = -1; multi[tid] = 0;
    __syncthreads();

    const uint64_t warps_total = (uint64_t)gridDim.x * (PH_THREADS / 32);
    const uint64_t warp_global = (uint64_t)blockIdx.x * (PH_THREADS / 32) + (tid >> 5);
    unsigned since_flush = 0;
    for (uint64_t r = warp_global; r < n_reads; r += warps_total) {
        const uint64_t o1 = line_off[4 * r + 1], o2 = line_off[4 * r + 2], o3 = line_off[4 * r + 3], o4 = line_off[4 * r + 4];
        uint64_t len = o2 - o1 - 1;
        const uint64_t qlen = o4 - o3 - 1;
        if (qlen < len) len = qlen;            // malformed records are reported by k_record_stats
        const uint8_t* dna = d + o1;
        const uint8_t* qual = d + o3;
        for (uint64_t i = lane; i < len; i += 32) {
            const unsigned b = __ldg(dna + i), q = __ldg(qual + i);
            if (b < 128u) priv_b[(b >> 2) * PH_THREADS + tid] += 1u << (8 * (b & 3u));
            else atomicAdd(&s->base_count[b], 1ull);
            if (q < 128u) priv_q[(q >> 2) * PH_THREADS + tid] += 1u << (8 * (q & 3u));
            else atomicAdd(&s->qual_count[q], 1ull);
            const int f = first_q[b];
            if (f != (int)q) {
                if (f < 0) {
                    int old = atomicCAS(&first_q[b], -1, (int)q);
                    if (old >= 0 && old != (int)q) multi[b] = 1;
                } else {
                    multi[b] = 1;
                }
            }
            if (++since_flush == 255u) {
                ph_flush(priv_b, hist_b, tid);
                ph_flush(priv_q, hist_q, tid);
                since_flush = 0;
            }
        }
    }
    ph_flush(priv_b, hist_b, tid);
    ph_flush(priv_q, hist_q, tid);
    __syncthreads();
    if (hist_b[tid]) atomicAdd(&s->base_count[tid], (unsigned long long)hist_b[tid]);
    if (hist_q[tid]) atomicAdd(&s->qual_count[tid], (unsigned long long)hist_q[tid]);
    const int f = first_q[tid];
    if (f >= 0) {
        int old = atomicCAS(&s->first_q[tid], -1, f);
        if (old >= 0 && old != f) s->multi[tid] = 1;
    }
    if (multi[tid]) s->multi[tid] = 1;
}

// ================================================================================================
// The product kernels.  The generic kernels above remain the path for QNAME lines that defeat the packed
// counters (more than 64 distinct bytes in line 1 or a QNAME longer than 255 bytes) and for bytes outside
// 32..127 - the kernels report that through `fallback` and the host runs the generic pair.
// ================================================================================================
#define RS_SLOTS 64

// ---- record statistics, names only ----------------------------------------------------------------
// The per-record statistics need the line offsets, the QNAME line and the first byte of line 3 - not the
// bases and qualities - so this kernel does not stage whole records: one thread per record reads its
// name in aligned 8-byte words (about 100 of the 340 bytes of a record cross the memory system: its
// offsets, the sectors of the name and of the '+').  Per name byte: one compare with line 1 (while the
// common prefix still runs) and one read-modify-write of a private packed 8-bit counter in shared
// memory ([word][thread] layout, conflict free; the LUT gives word and increment, bytes that do not
// occur in line 1 add zero).  Needs <= 64 distinct bytes in line 1 and names of <= 255 bytes, else
// `fallback` is raised and the host uses the generic kernel.
#define RD_THREADS 256
#define RD_WORDS (RS_SLOTS / 4)

struct rd_smem {
    uint8_t first[UQB_HDR_MAX];
    uint8_t slot_of[256];
    uint8_t slot_char[RS_SLOTS];
    uint32_t lut[256];                  // byte -> (byte offset of its counter word row) << 16 | PRMT selector of its field
    uint32_t first_words[RD_WORDS];     // packed counts of line 1
    uint32_t cnt[RD_WORDS * RD_THREADS];
    uint32_t lcp_first[UQB_HDR_MAX + 1], lcs_first[UQB_HDR_MAX + 1], sp_first[UQB_HDR_MAX + 1], ss_first[UQB_HDR_MAX + 1];
    uint32_t last_mis[RS_SLOTS];        // record index + 1 of the last mismatch, 0 = none
    int nslots;
};

__global__ void __launch_bounds__(RD_THREADS) k_record_stats_names(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                                  uint64_t r_begin, uint64_t n_reads, const uint8_t* __restrict__ ref,
                                                                  uint64_t rbase, uint32_t first_len, an_dev* __restrict__ s,
                                                                  unsigned int* __restrict__ fallback,
                                                                  const uint8_t* __restrict__ names, uint32_t name_pitch, int checks) {
    // checks == 0: the FASTQ shape checks and the read lengths are produced by the histogram kernel, which has the whole
    // record in shared memory anyway; this kernel then touches the first two line offsets and the name only
    // names != nullptr: the QNAME lines come from the compact side array written by k_pair_hist_pipe (row r: length byte +
    // text); the per-record FASTQ checks and read lengths were done there, only the name statistics are produced here
    extern __shared__ __align__(16) uint8_t rd_raw[];
    rd_smem* S = reinterpret_cast<rd_smem*>(rd_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31u;
    for (unsigned i = tid; i < first_len && i < UQB_HDR_MAX; i += RD_THREADS) S->first[i] = ref[i];
    S->slot_of[tid] = 255;
    S->lut[tid] = 0x1111u;                                   // word 0, increment 0
    for (unsigned i = tid; i <= UQB_HDR_MAX; i += RD_THREADS) { S->lcp_first[i] = S->lcs_first[i] = S->sp_first[i] = S->ss_first[i] = 0xFFFFFFFFu; }
    if (tid < RS_SLOTS) S->last_mis[tid] = 0;
    if (tid < RD_WORDS) S->first_words[tid] = 0;
    for (unsigned i = tid; i < RD_WORDS * RD_THREADS; i += RD_THREADS) S->cnt[i] = 0;
    __syncthreads();
    if (tid == 0) {
        int ns = 0;
        bool over = false;
        for (unsigned i = 0; i < first_len && i < UQB_HDR_MAX; i++) {
            const uint8_t c = S->first[i];
            if (S->slot_of[c] == 255) {
                if (ns < RS_SLOTS) {
                    S->slot_of[c] = (uint8_t)ns; S->slot_char[ns] = c;
                    S->lut[c] = (((unsigned)(ns >> 2) * RD_THREADS * 4u) << 16) | (0x1111u ^ (1u << (4u * (ns & 3))));
                    ns++;
                } else over = true;
            }
            const uint8_t sl = S->slot_of[c];
            if (sl != 255) S->first_words[sl >> 2] += 1u << ((sl & 3) * 8);
        }
        if (over || first_len > 255) atomicOr(fallback, 1u);
        S->nslots = ns;
    }
    __syncthreads();
    const int nslots = S->nslots;
    const int nwords = (nslots + 3) >> 2;
    const uint32_t cnt_a = smem_u32(S->cnt + tid), lut_a = smem_u32(S->lut), first_a = smem_u32(S->first);

    unsigned long long mn = ~0ull, mx = 0ull;
    unsigned nm = 0;
    long long bad_plus = LLONG_MAX, bad_len = LLONG_MAX;
    const uint64_t nblk = (n_reads - r_begin + RD_THREADS - 1) / RD_THREADS;
    for (uint64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const uint64_t r = r_begin + blk * RD_THREADS + tid;
        const bool active = r < n_reads;
        unsigned lcp = 0, lcs = 0, name_len = 0;
        if (active) {
            unsigned plus = '+';
            const uint8_t* name;
            if (names) {
                name = names + r * name_pitch + 1;
                name_len = __ldg(name - 1);
            } else if (!checks) {
                const ulonglong2 oa = __ldg(reinterpret_cast<const ulonglong2*>(line_off + 4 * r));
                const uint64_t nl64 = oa.y - oa.x - 1;
                name_len = nl64 > 0xFFFFu ? 0xFFFFu : (unsigned)nl64;
                name = d + oa.x;
            } else {
                const ulonglong2 oa = __ldg(reinterpret_cast<const ulonglong2*>(line_off + 4 * r));
                const ulonglong2 ob = __ldg(reinterpret_cast<const ulonglong2*>(line_off + 4 * r + 2));
                const uint64_t o0 = oa.x, o1 = oa.y, o2 = ob.x, o3 = ob.y, o4 = __ldg(line_off + 4 * r + 4);
                const uint64_t dlen = o2 - o1 - 1, qlen = o4 - o3 - 1;
                plus = o3 - o2 < 2 ? 0u : (unsigned)__ldg(d + o2);           // used after the name loop
                if (dlen != qlen) bad_len = bad_len < (long long)r ? bad_len : (long long)r;
                mn = dlen < mn ? dlen : mn; mx = dlen > mx ? dlen : mx;
                const uint64_t nl64 = o1 - o0 - 1;
                name_len = nl64 > 0xFFFFu ? 0xFFFFu : (unsigned)nl64;
                name = d + o0;
            }
            nm = name_len > nm ? name_len : nm;
            if (name_len > 255) {
                atomicOr(fallback, 1u);                      // 8-bit packed counters could wrap
            } else {
                const unsigned lim = name_len < first_len ? name_len : first_len;
                const uint64_t addr = (uint64_t)(uintptr_t)name;
                const uint64_t* q = reinterpret_cast<const uint64_t*>(addr & ~7ull);
                const unsigned ph = (unsigned)(addr & 7ull);
                // the first 64 bytes of the aligned window are fetched at once (independent loads), then consumed
                // from registers; longer names continue word by word
                const unsigned nw8 = (ph + name_len + 7u) >> 3;
                uint64_t W[8];
#pragma unroll
                for (int k = 0; k < 8; k++) W[k] = (unsigned)k < nw8 ? __ldg(q + k) : 0ull;
                bool run = true;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if ((unsigned)k < nw8) {
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const unsigned i = (unsigned)(8 * k + j) - ph;             // wraps for window bytes before the name
                            if (i < name_len) {
                                const unsigned c = (unsigned)(W[k] >> (8 * j)) & 255u;
                                if (run) { if (i < lim && c == lds_u8(first_a + i)) lcp = i + 1; else run = false; }
                                const uint32_t e = lds_u32(lut_a + (c << 2));
                                const uint32_t wa = cnt_a + (e >> 16);
                                sts_u32(wa, lds_u32(wa) + __byte_perm(1u, 0u, e));
                            }
                        }
                    }
                }
                if (nw8 > 8) {
                    q += 8;
                    unsigned avail = 0;
                    uint64_t w = 0;
                    for (unsigned i = 64u - ph; i < name_len; i++) {
                        if (avail == 0) { w = __ldg(q++); avail = 8; }
                        const unsigned c = (unsigned)w & 255u;
                        w >>= 8; avail--;
                        if (run) { if (i < lim && c == lds_u8(first_a + i)) lcp = i + 1; else run = false; }
                        const uint32_t e = lds_u32(lut_a + (c << 2));
                        const uint32_t wa = cnt_a + (e >> 16);
                        sts_u32(wa, lds_u32(wa) + __byte_perm(1u, 0u, e));
                    }
                }
                while (lcs < lim && __ldg(name + name_len - 1 - lcs) == S->first[first_len - 1 - lcs]) lcs++;
            }
            if (plus != '+') bad_plus = bad_plus < (long long)r ? bad_plus : (long long)r;
        }
        // first record per lcp / lcs value: the lowest lane of each match group is the lowest record
        {
            const bool part = active && name_len <= 255 && r + rbase >= 1;
            const unsigned key1 = part ? lcp : 0xFFFFu, key2 = part ? lcs : 0xFFFFu;
            const unsigned m1 = __match_any_sync(0xffffffffu, key1), m2 = __match_any_sync(0xffffffffu, key2);
            if (part && (int)lane == __ffs(m1) - 1) atomicMin(&S->lcp_first[lcp], (uint32_t)r);
            if (part && (int)lane == __ffs(m2) - 1) atomicMin(&S->lcs_first[lcs], (uint32_t)r);
            if (part && lcp == name_len && name_len < first_len) atomicMin(&S->sp_first[name_len], (uint32_t)r);
            if (part && lcs == name_len && name_len < first_len) atomicMin(&S->ss_first[name_len], (uint32_t)r);
        }
        // last record whose count of a tracked byte differs from line 1's
        const uint64_t rw = r_begin + blk * RD_THREADS + (tid & ~31u);            // record of lane 0
        for (int wd = 0; wd < nwords; wd++) {
            const uint32_t x = S->cnt[wd * RD_THREADS + tid];
            S->cnt[wd * RD_THREADS + tid] = 0;
            const uint32_t diff = (active && name_len <= 255) ? (x ^ S->first_words[wd]) : 0u;
            if (__any_sync(0xffffffffu, diff != 0u)) {
#pragma unroll
                for (int f = 0; f < 4; f++) {
                    const unsigned m = __ballot_sync(0xffffffffu, ((diff >> (8 * f)) & 255u) != 0u);
                    if (m && lane == 0) atomicMax(&S->last_mis[wd * 4 + f], (uint32_t)(rw + (31 - __clz(m))) + 1u);
                }
            }
        }
    }
    // ---- CTA results -> global ----
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        unsigned c = __shfl_xor_sync(0xffffffffu, nm, o);
        long long e = __shfl_xor_sync(0xffffffffu, bad_plus, o), f = __shfl_xor_sync(0xffffffffu, bad_len, o);
        mn = a < mn ? a : mn; mx = b > mx ? b : mx; nm = c > nm ? c : nm;
        bad_plus = e < bad_plus ? e : bad_plus; bad_len = f < bad_len ? f : bad_len;
    }
    if (lane == 0) {
        if (mn != ~0ull) atomicMin(&s->dna_min, mn);
        atomicMax(&s->dna_max, mx);
        atomicMax(&s->max_name_len, nm);
        if (bad_plus != LLONG_MAX) atomicMin(&s->bad_plus, bad_plus);
        if (bad_len != LLONG_MAX) atomicMin(&s->bad_len, bad_len);
    }
    __syncthreads();
    for (unsigned j = tid; j <= first_len && j <= UQB_HDR_MAX; j += RD_THREADS) {
        if (S->lcp_first[j] != 0xFFFFFFFFu) atomicMin(&s->first_lcp_eq[j], (long long)S->lcp_first[j]);
        if (S->lcs_first[j] != 0xFFFFFFFFu) atomicMin(&s->first_lcs_eq[j], (long long)S->lcs_first[j]);
        if (S->sp_first[j] != 0xFFFFFFFFu) atomicMin(&s->first_short_prefix[j], (long long)S->sp_first[j]);
        if (S->ss_first[j] != 0xFFFFFFFFu) atomicMin(&s->first_short_suffix[j], (long long)S->ss_first[j]);
    }
    if (tid < (unsigned)nslots && S->last_mis[tid]) atomicMax(&s->last_count_mismatch[S->slot_char[tid]], (long long)S->last_mis[tid] - 1);
}

// base / quality histograms of long reads (k_pair_hist_long below).
//
// Qualities: private packed 8-bit counters per thread in shared memory ([word][thread] layout, bank-conflict
// free), addressed through a LUT that puts neighbouring byte values into different words, flushed through a
// warp-shuffle reduction before a counter can wrap (pt_flush).  Bytes outside 32..127 go to a dummy counter
// that the host reads as "use the generic kernels".
//
// Bases: a thread sees very few distinct base bytes, so its counters stay in REGISTERS: the LUT maps a byte to
// a group of seven byte values (A C G T N U . share one group) and to the increment of its 8-bit field in a
// 56-bit pending counter (two registers; the top byte of the second one carries the group id in the LUT and is
// ignored in the counter); only when a thread meets a byte of another group (or the fields could wrap) are the
// pending counts added to the CTA histogram.  The common case costs a LUT load, a compare and two adds per base.
//
// "Does this base always carry one single quality?" (the N-trick): state[b] = -1 unseen, 0..255 its only quality
// so far, 256 several.  A base whose state is not yet 256 carries a CHECK bit in its LUT group, which never
// equals the current group, so exactly those bases take the slow path that compares the quality.
#define PT_THREADS 1024
#define PT_WORDS 25
#define PT_LO 32u
#define PT_OOR 96u           // clamped index of out-of-range quality bytes -> histogram slot 128
#define PT_ROW (PT_THREADS * 4)
#define PT_GROUPS 40         // base groups: 1, 2 special, 3 + v / 7 generic
#define PT_CHECK 0x80000000u
#define PT_GMASK 0xff000000u
#define PT_NONE 0x7f000000u  // "no pending group yet"

struct pt_smem {
    unsigned priv_q[PT_WORDS * PT_THREADS];
    unsigned hist_b[256], hist_q[PT_LO + 4 * PT_WORDS];
    int state[256];                 // per base byte: -1 unseen, 0..255 its only quality so far, 256 = several
    uint2 lutb[256];                // base byte -> {increment of fields 0-3, (group | CHECK) << 24 | increment of fields 4-6}
    uint2 lutq[256];                // quality byte -> {byte offset of its counter word row, increment}
    uint8_t rev[PT_GROUPS * 8];     // (group, field) -> base byte
};

__device__ __forceinline__ void pt_base_group(unsigned v, unsigned* grp, unsigned* field) {
    const char* g1 = "ACGTNU.";
    const char* g2 = "acgtnu-";
    *grp = 3u + v / 7u; *field = v % 7u;
#pragma unroll
    for (unsigned f = 0; f < 7; f++) {
        if (v == (unsigned)(unsigned char)g1[f]) { *grp = 1u; *field = f; }
        if (v == (unsigned)(unsigned char)g2[f]) { *grp = 2u; *field = f; }
    }
}

// Flush of the private quality counters of one warp: the four 8-bit fields of a word are widened to two words
// of two 16-bit fields (32 lanes x 255 < 65536), summed across the warp with shuffles, and lane 0 adds
// the four sums to the CTA histogram.  Must be called by all 32 lanes.
__device__ __forceinline__ void pt_flush(unsigned* priv, unsigned* blk_hist, unsigned tid) {
    const unsigned lane = tid & 31u;
#pragma unroll 5
    for (int w = 0; w < PT_WORDS; w++) {
        const unsigned x = priv[w * PT_THREADS + tid];
        priv[w * PT_THREADS + tid] = 0;
        unsigned e = x & 0x00FF00FFu, o = (x >> 8) & 0x00FF00FFu;       // fields 0,2 and 1,3
        if (__any_sync(0xffffffffu, x != 0u)) {
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) {
                e += __shfl_xor_sync(0xffffffffu, e, sh);
                o += __shfl_xor_sync(0xffffffffu, o, sh);
            }
            if (lane == 0) {
                // counter (word w, field f) belongs to byte value 32 + f*24 + w (w < 24); word 24 holds the dummy
                const unsigned i0 = w < 24 ? PT_LO + w : PT_LO + 96u, st = w < 24 ? 24u : 1u;
                if (e & 0xFFFFu) atomicAdd(&blk_hist[i0], e & 0xFFFFu);
                if (o & 0xFFFFu) atomicAdd(&blk_hist[i0 + st], o & 0xFFFFu);
                if (e >> 16) atomicAdd(&blk_hist[i0 + 2 * st], e >> 16);
                if (o >> 16) atomicAdd(&blk_hist[i0 + 3 * st], o >> 16);
            }
        }
    }
}

// pending base counters of one thread -> CTA histogram (cur = group << 24)
__device__ __noinline__ void pt_base_flush(pt_smem* S, unsigned cur, unsigned pa, unsigned pb) {
    const unsigned g = cur >> 24;
    if (g >= PT_GROUPS) return;
#pragma unroll
    for (unsigned f = 0; f < 4; f++) {
        const unsigned ca = (pa >> (8 * f)) & 255u;
        if (ca) atomicAdd(&S->hist_b[S->rev[g * 8 + f]], ca);
    }
#pragma unroll
    for (unsigned f = 0; f < 3; f++) {
        const unsigned cb = (pb >> (8 * f)) & 255u;
        if (cb) atomicAdd(&S->hist_b[S->rev[g * 8 + 4 + f]], cb);
    }
}

// the same for a whole warp (all 32 lanes call it): one shuffle reduction when every lane is in the same group
__device__ __forceinline__ void pt_base_flush_warp(pt_smem* S, unsigned cur, unsigned& pa, unsigned& pb, unsigned lane) {
    const unsigned cur0 = __shfl_sync(0xffffffffu, cur, 0);
    if (__all_sync(0xffffffffu, cur == cur0)) {
        const unsigned g = cur0 >> 24;
        if (g < PT_GROUPS) {
            unsigned v[4] = {pa & 0x00FF00FFu, (pa >> 8) & 0x00FF00FFu, pb & 0x00FF00FFu, (pb >> 8) & 0x000000FFu};
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) {
#pragma unroll
                for (int k = 0; k < 4; k++) v[k] += __shfl_xor_sync(0xffffffffu, v[k], sh);
            }
            if (lane == 0) {
#pragma unroll
                for (unsigned k = 0; k < 4; k++) {           // v[k]: fields (k&1) and (k&1)+2 of half k>>1
                    const unsigned f0 = (k >> 1) * 4 + (k & 1u);
                    if (v[k] & 0xFFFFu) atomicAdd(&S->hist_b[S->rev[g * 8 + f0]], v[k] & 0xFFFFu);
                    if (v[k] >> 16) atomicAdd(&S->hist_b[S->rev[g * 8 + f0 + 2]], v[k] >> 16);
                }
            }
        }
    } else {
        pt_base_flush(S, cur, pa, pb);
    }
    pa = 0; pb = 0;
}

// slow path of one base: single-quality state, change of the pending group
__device__ __noinline__ uint3 pt_base_slow(pt_smem* S, unsigned b, unsigned q, unsigned ey, unsigned cur, unsigned pa, unsigned pb) {
    if (ey & PT_CHECK) {
        int f = S->state[b];
        if (f != 256 && f != (int)q) {
            if (f < 0) {
                const int old = atomicCAS(&S->state[b], -1, (int)q);
                if (old >= 0 && old != (int)q) { S->state[b] = 256; f = 256; }
            } else {
                S->state[b] = 256; f = 256;
            }
        }
        if (f == 256) S->lutb[b].y = ey & ~PT_CHECK;             // several qualities: no more checks for this base
    }
    const unsigned grp = ey & (PT_GMASK & ~PT_CHECK);
    if (grp != cur) {
        pt_base_flush(S, cur, pa, pb);
        cur = grp; pa = 0; pb = 0;
    }
    return make_uint3(cur, pa, pb);
}

#include "hist_units.cuh"

// Long reads (records that do not fit a tile): the counters above, fed straight from global memory.  One warp per
// record; a lane takes aligned 16-byte units of the DNA line and, separately, of the QUAL line (the two lines have
// different alignments, and counting does not need them paired).  Only a base that still carries the CHECK bit needs
// its own quality: that single byte is fetched on the spot.  At most 15 units (240 increments of one 8-bit field)
// between flushes.
__device__ __forceinline__ void pt_long_base(pt_smem* S, const uint8_t* __restrict__ d, uint64_t qbase, uint64_t pos0, unsigned b, unsigned k,
                                             uint32_t lutb_a, uint32_t state_a, unsigned& cur, unsigned& pa, unsigned& pb) {
    const uint2 e = lds_u64(lutb_a + (b << 3));
    const unsigned dd = (e.y ^ cur) & PT_GMASK;
    if (dd) {
        unsigned q = 0;
        if (e.y & PT_CHECK) q = __ldg(d + qbase + pos0 + k);                 // quality of this very position
        if (dd != PT_CHECK || lds_u32(state_a + (b << 2)) != q) {
            const uint3 r = pt_base_slow(S, b, q, e.y, cur, pa, pb);
            cur = r.x; pa = r.y; pb = r.z;
        }
    }
    pa += e.x;
    pb += e.y;
}

__global__ void __launch_bounds__(PT_THREADS, 1) k_pair_hist_long(const uint8_t* __restrict__ d, const uint64_t* __restrict__ line_off,
                                                                 uint64_t r_begin, uint64_t n_reads, an_dev* __restrict__ s,
                                                                 unsigned int* __restrict__ fallback) {
    extern __shared__ __align__(128) uint8_t pt_raw[];
    pt_smem* S = reinterpret_cast<pt_smem*>(pt_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    for (unsigned i = tid; i < PT_WORDS * PT_THREADS; i += PT_THREADS) S->priv_q[i] = 0;
    for (unsigned i = tid; i < PT_LO + 4 * PT_WORDS; i += PT_THREADS) S->hist_q[i] = 0;
    for (unsigned i = tid; i < PT_GROUPS * 8; i += PT_THREADS) S->rev[i] = 0;
    if (tid < 256) { S->hist_b[tid] = 0; S->state[tid] = -1; }
    __syncthreads();
    if (tid < 256) {
        const unsigned v = tid;
        unsigned grp, field;
        pt_base_group(v, &grp, &field);
        S->lutb[v] = make_uint2(field < 4 ? 1u << (8 * field) : 0u, ((grp << 24) | PT_CHECK) | (field >= 4 ? 1u << (8 * (field - 4)) : 0u));
        S->rev[grp * 8 + field] = (uint8_t)v;
        const unsigned idx = min(v - PT_LO, PT_OOR);
        const unsigned word = idx < 96u ? idx % 24u : 24u, qf = idx < 96u ? idx / 24u : 0u;
        S->lutq[v] = make_uint2(word * PT_ROW, 1u << (8 * qf));
    }
    __syncthreads();
    const uint32_t pq_a = smem_u32(S->priv_q + tid);
    const uint32_t lutb_a = smem_u32(S->lutb), lutq_a = smem_u32(S->lutq), state_a = smem_u32(S->state);
    unsigned cur = PT_NONE, pa = 0, pb = 0, since_flush = 0;
    const uint64_t nwarps = (uint64_t)gridDim.x * (PT_THREADS / 32);
    for (uint64_t r = r_begin + (uint64_t)blockIdx.x * (PT_THREADS / 32) + wid; r < n_reads; r += nwarps) {
        const uint64_t o1 = line_off[4 * r + 1], o2 = line_off[4 * r + 2], o3 = line_off[4 * r + 3], o4 = line_off[4 * r + 4];
        uint64_t len = o2 - o1 - 1;
        const uint64_t qlen = o4 - o3 - 1;
        if (qlen < len) len = qlen;                  // malformed records are reported by the record-stats kernel
        // the two lines as ranges of aligned 16-byte units
        for (int line = 0; line < 2; line++) {
            const uint64_t b0 = line == 0 ? o1 : o3, b1 = b0 + len;
            const uint64_t u0 = b0 >> 4, u1 = (b1 + 15) >> 4;
            for (uint64_t ub = u0; ub < u1; ub += 32) {              // warp-uniform trip count
                if (since_flush >= 15u) {
                    pt_flush(S->priv_q, S->hist_q, tid);
                    pt_base_flush_warp(S, cur, pa, pb, lane);
                    since_flush = 0;
                }
                since_flush++;
                const uint64_t u = ub + lane;
                if (u < u1) {
                    const uint4 x = __ldg(reinterpret_cast<const uint4*>(d) + u);
                    const uint32_t w[4] = {x.x, x.y, x.z, x.w};
                    const uint64_t p0 = u << 4;
                    const bool inner = p0 >= b0 && p0 + 16 <= b1;
#pragma unroll
                    for (int k = 0; k < 16; k++) {
                        if (inner || (p0 + k >= b0 && p0 + k < b1)) {
                            const unsigned c = (w[k >> 2] >> (8 * (k & 3))) & 255u;
                            if (line == 0) {
                                pt_long_base(S, d, o3, p0 - o1, c, (unsigned)k, lutb_a, state_a, cur, pa, pb);
                            } else {
                                const uint2 e = lds_u64(lutq_a + (c << 3));
                                const uint32_t wq = pq_a + e.x;
                                sts_u32(wq, lds_u32(wq) + e.y);
                            }
                        }
                    }
                }
            }
        }
    }
    pt_flush(S->priv_q, S->hist_q, tid);
    pt_base_flush(S, cur, pa, pb);
    __syncthreads();
    if (tid < 256) {
        if (S->hist_b[tid]) atomicAdd(&s->base_count[tid], (unsigned long long)S->hist_b[tid]);
        if (tid < 128 && S->hist_q[tid]) atomicAdd(&s->qual_count[tid], (unsigned long long)S->hist_q[tid]);
        if (tid == 0 && S->hist_q[PT_LO + PT_OOR]) atomicOr(fallback, 1u);
        const int f = S->state[tid];
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

// long reads: names-only record statistics + the direct histogram above
static int stats_long_range(uqb_ctx* ctx, const uqb_fastq* fq, an_dev* s, unsigned int* d_fb, uint32_t flen, uint64_t r0, uint64_t r1) {
    if (r1 <= r0) return 0;
    static_assert(sizeof(pt_smem) <= 227 * 1024, "pair histogram shared memory");
    UQB_CUDA(cudaFuncSetAttribute(k_pair_hist_long, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(pt_smem)));
    UQB_LAUNCH_B((r1 - r0) * 128, k_record_stats_names, uqb_grid(ctx, r1 - r0, RD_THREADS, 8), RD_THREADS, sizeof(rd_smem), fq->d, fq->line_off, r0, r1,
                 fq->ref_name ? fq->ref_name : fq->d, fq->rbase, flen, s, d_fb, (const uint8_t*)nullptr, 0u, 1);
    const uint64_t ab = (uint64_t)((double)fq->n * (double)(r1 - r0) / (double)(fq->n_reads ? fq->n_reads : 1)) + 32 * (r1 - r0);
    const uint64_t warps = (r1 - r0 + 0) ;
    const unsigned g = (unsigned)((warps + PT_THREADS / 32 - 1) / (PT_THREADS / 32) < (uint64_t)ctx->sm_count ? (warps + PT_THREADS / 32 - 1) / (PT_THREADS / 32)
                                                                                                           : (uint64_t)ctx->sm_count);
    UQB_LAUNCH_B(ab, k_pair_hist_long, g, PT_THREADS, sizeof(pt_smem), fq->d, fq->line_off, r0, r1, s, d_fb);
    return 0;
}

// launches the two tile kernels over records [r0, r1)
static int stats_tiles_range(uqb_ctx* ctx, const uqb_fastq* fq, an_dev* s, unsigned int* d_fb, uint32_t flen, uint64_t r0, uint64_t r1) {
    if (r1 <= r0) return 0;
    const uint64_t ntiles = (r1 - r0 + TL_R - 1) / TL_R;
    const unsigned g2 = (unsigned)(ntiles < (uint64_t)ctx->sm_count ? ntiles : (uint64_t)ctx->sm_count);      // one 1024-thread CTA per SM
    const uint64_t ab = (uint64_t)((double)fq->n * (double)(r1 - r0) / (double)(fq->n_reads ? fq->n_reads : 1)) + 32 * (r1 - r0);
    // names only: 32 B of offsets and the name's sectors per record
    UQB_LAUNCH_B((r1 - r0) * 96, k_record_stats_names, uqb_grid(ctx, r1 - r0, RD_THREADS, 8), RD_THREADS, sizeof(rd_smem), fq->d, fq->line_off, r0, r1,
                 fq->ref_name ? fq->ref_name : fq->d, fq->rbase, flen, s, d_fb, (const uint8_t*)nullptr, 0u, 0);
    static_assert(sizeof(h3_smem) <= 227 * 1024, "pipelined unit histogram shared memory");
    UQB_CUDA(cudaFuncSetAttribute(k_pair_hist_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(h3_smem)));
    UQB_LAUNCH_B(ab, k_pair_hist_pipe, g2, H2_THREADS, sizeof(h3_smem), fq->d, fq->n, fq->line_off, r0, r1, s, d_fb, (uint8_t*)nullptr, 0u);
    return 0;
}

// The whole file is resident (uqb_analyze): the histogram kernel also writes the compact QNAME array (fq->names), and the
// name statistics - like the tokeniser and the dictionary rows later - read that instead of the FASTQ.
// *fb_out: bit 0 = use the generic kernels, bit 2 = a name did not fit the compact rows (they are dropped)
static int stats_tiles_resident(uqb_ctx* ctx, uqb_fastq* fq, an_dev* s, unsigned int* d_fb, uint32_t flen, uint32_t own_first_len,
                                unsigned int* fb_out) {
    const uint64_t N = fq->n_reads;
    uint32_t pitch = (own_first_len + 1 + 24 + 15) / 16 * 16;
    if (pitch < 32) pitch = 32;
    if (pitch > 256 || fq->names) {
        UQB_TRY(stats_tiles_range(ctx, fq, s, d_fb, flen, 0, N));
        UQB_TRY(uqb_readback(ctx, fb_out, d_fb, 4));
        return 0;
    }
    uint8_t* names;
    UQB_TRY(uqb_dalloc(ctx, (void**)&names, N * pitch + 64));
    const uint64_t ntiles = (N + TL_R - 1) / TL_R;
    const unsigned g2 = (unsigned)(ntiles < (uint64_t)ctx->sm_count ? ntiles : (uint64_t)ctx->sm_count);
    UQB_CUDA(cudaFuncSetAttribute(k_pair_hist_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(h3_smem)));
    UQB_LAUNCH_B(fq->n + 32 * N + N * pitch, k_pair_hist_pipe, g2, H2_THREADS, sizeof(h3_smem), fq->d, fq->n, fq->line_off, 0ull, N, s, d_fb, names, pitch);
    UQB_TRY(uqb_readback(ctx, fb_out, d_fb, 4));
    if (*fb_out & 5u) {                                  // generic kernels, or a long name: no compact array
        UQB_TRY(uqb_dfree(ctx, names, 0));
        if (!(*fb_out & 1u))
            UQB_LAUNCH_B(N * 96, k_record_stats_names, uqb_grid(ctx, N, RD_THREADS, 8), RD_THREADS, sizeof(rd_smem), fq->d, fq->line_off, 0ull, N,
                         fq->ref_name ? fq->ref_name : fq->d, fq->rbase, flen, s, d_fb, (const uint8_t*)nullptr, 0u, 0);
    } else {
        fq->names = names; fq->name_pitch = pitch; fq->names_cap = N;
        UQB_LAUNCH_B(N * pitch, k_record_stats_names, uqb_grid(ctx, N, RD_THREADS, 8), RD_THREADS, sizeof(rd_smem), fq->d, fq->line_off, 0ull, N,
                     fq->ref_name ? fq->ref_name : fq->d, fq->rbase, flen, s, d_fb, (const uint8_t*)names, pitch, 0);
    }
    UQB_TRY(uqb_readback(ctx, fb_out, d_fb, 4));         // the name statistics may ask for the generic kernels, too
    return 0;
}

static int stats_generic(uqb_ctx* ctx, const uqb_fastq* fq, an_dev* s, uint32_t flen) {
    const uint64_t N = fq->n_reads;
    UQB_LAUNCH(k_an_init, 1, 256, 0, s);
    UQB_LAUNCH(k_record_stats, uqb_blocks(N, AN_THREADS), AN_THREADS, 0, fq->d, fq->line_off, N,
               fq->ref_name ? fq->ref_name : fq->d, fq->rbase, flen, s);
    const size_t smem = (2 * PH_WORDS * PH_THREADS + 4 * 256) * sizeof(unsigned);
    UQB_CUDA(cudaFuncSetAttribute(k_pair_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    UQB_LAUNCH(k_pair_hist, uqb_grid(ctx, N, PH_THREADS / 32, 3), PH_THREADS, smem, fq->d, fq->line_off, N, s);
    return 0;
}

// first / last QNAME lines -> out; returns their lengths
static int stats_names(uqb_ctx* ctx, const uqb_fastq* fq, uqb_stats* out, uint64_t* flen_out) {
    const uint64_t N = fq->n_reads;
    uint64_t offs[2], offl[2];
    UQB_TRY(uqb_readback(ctx, offs, fq->line_off, 16));
    UQB_TRY(uqb_readback(ctx, offl, fq->line_off + 4 * (N - 1), 16));
    const uint64_t flen = offs[1] - offs[0] - 1, llen = offl[1] - offl[0] - 1;
    if (flen > UQB_HDR_MAX || llen > UQB_HDR_MAX)
        return uqb_fail(ctx, "QNAME line longer than %d bytes is not supported by the device path", UQB_HDR_MAX);
    out->first_len = (uint32_t)flen;
    out->last_len = (uint32_t)llen;
    if (flen) UQB_TRY(uqb_readback(ctx, out->first_name, fq->d + offs[0], flen));
    if (llen) UQB_TRY(uqb_readback(ctx, out->last_name, fq->d + offl[0], llen));
    out->bad_first_char = (flen >= 1 && out->first_name[0] == '@') ? -1 : 0;
    *flen_out = flen;
    return 0;
}

// device accumulators -> uqb_stats
static int stats_finish(uqb_ctx* ctx, uqb_fastq* fq, an_dev* s, uqb_stats* out, uint64_t flen) {
    an_dev* h = new an_dev();
    int rc = uqb_readback(ctx, h, s, sizeof(an_dev));
    if (rc) { delete h; return rc; }
    fq->total_bases = 0;
    for (int i = 0; i < 256; i++) fq->total_bases += h->base_count[i];
    for (int i = 0; i < 256; i++) {
        out->base_count[i] = h->base_count[i];
        out->qual_count[i] = h->qual_count[i];
        out->base_single_qual[i] = h->first_q[i] < 0 ? -1 : (h->multi[i] ? 256 : h->first_q[i]);
        out->last_count_mismatch[i] = h->last_count_mismatch[i];
    }
    out->dna_min = h->dna_min;
    out->dna_max = h->dna_max;
    out->bad_plus_record = h->bad_plus == LLONG_MAX ? -1 : h->bad_plus;
    out->bad_len_record = h->bad_len == LLONG_MAX ? -1 : h->bad_len;
    out->max_name_len = h->max_name_len;
    uint32_t pl = (uint32_t)flen, sl = (uint32_t)flen;
    for (uint32_t j = 0; j <= UQB_HDR_MAX; j++) {
        out->first_lcp_eq[j] = h->first_lcp_eq[j];
        out->first_lcs_eq[j] = h->first_lcs_eq[j];
        out->first_short_prefix[j] = h->first_short_prefix[j];
        out->first_short_suffix[j] = h->first_short_suffix[j];
        if (h->first_lcp_eq[j] != LLONG_MAX && j < pl) pl = j;
        if (h->first_lcs_eq[j] != LLONG_MAX && j < sl) sl = j;
    }
    out->prefix_len = pl;
    out->suffix_len = sl;
    delete h;
    return 0;
}

int uqb_names_release(uqb_ctx* ctx, uqb_fastq* fq) {
    if (fq->names) { UQB_TRY(uqb_dfree(ctx, fq->names, 0)); fq->names = nullptr; }
    fq->name_pitch = 0; fq->names_cap = 0;
    return 0;
}

// Multi-GPU: this handle holds records [rbase, rbase + n) of a larger file whose first QNAME line is `name`.
// uqb_analyze then reports prefix/suffix/separator statistics against that line (record indices stay local).
extern "C" int uqb_fastq_set_reference(uqb_ctx* ctx, uqb_fastq* fq, const uint8_t* name, uint32_t len, uint64_t rbase) {
    if (len > UQB_HDR_MAX) return uqb_fail(ctx, "reference QNAME longer than %d bytes", UQB_HDR_MAX);
    if (fq->ref_name) { UQB_TRY(uqb_dfree(ctx, fq->ref_name, 0)); fq->ref_name = nullptr; }
    UQB_TRY(uqb_dalloc(ctx, (void**)&fq->ref_name, len + 16));
    if (len) UQB_CUDA(cudaMemcpyAsync(fq->ref_name, name, len, cudaMemcpyHostToDevice, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    fq->ref_len = len;
    fq->rbase = rbase;
    delete fq->cached_stats;
    fq->cached_stats = nullptr;
    return 0;
}

extern "C" int uqb_analyze(uqb_ctx* ctx, uqb_fastq* fq, uqb_stats* out) {
    if (!fq->line_off) return uqb_fail(ctx, "uqb_analyze: call uqb_split first");
    if (fq->n_reads == 0) return uqb_fail(ctx, "uqb_analyze: no records");
    if (fq->cached_stats) { memcpy(out, fq->cached_stats, sizeof(*out)); return 0; }     // produced by the streamed load
    memset(out, 0, sizeof(*out));
    const uint64_t N = fq->n_reads;
    uint64_t flen = 0;
    UQB_TRY(stats_names(ctx, fq, out, &flen));
    if (fq->ref_name) flen = fq->ref_len;        // multi-GPU shard: everything is measured against the global line 1
    an_dev* s;
    UQB_TRY(uqb_dalloc_t(ctx, &s, 1));
    bool done_fast = false;
    if (fq->n / N <= (TL_CAP - 64) / TL_R) {
        // v2: shared-memory record tiles
        unsigned int* d_fb;
        UQB_TRY(uqb_dalloc_t(ctx, &d_fb, 1));
        UQB_CUDA(cudaMemsetAsync(d_fb, 0, 4, ctx->stream));
        UQB_LAUNCH(k_an_init, 1, 256, 0, s);
        unsigned int fb = 0;
        UQB_TRY(stats_tiles_resident(ctx, fq, s, d_fb, (uint32_t)flen, out->first_len, &fb));
        UQB_TRY(uqb_dfree(ctx, d_fb, 4));
        done_fast = (fb & 3u) == 0;
    } else if ((((uintptr_t)fq->d) & 15) == 0) {
        // long reads: the same counters straight from global memory
        unsigned int* d_fb;
        UQB_TRY(uqb_dalloc_t(ctx, &d_fb, 1));
        UQB_CUDA(cudaMemsetAsync(d_fb, 0, 4, ctx->stream));
        UQB_LAUNCH(k_an_init, 1, 256, 0, s);
        UQB_TRY(stats_long_range(ctx, fq, s, d_fb, (uint32_t)flen, 0, N));
        unsigned int fb = 0;
        UQB_TRY(uqb_readback(ctx, &fb, d_fb, 4));
        UQB_TRY(uqb_dfree(ctx, d_fb, 4));
        done_fast = fb == 0;
    }
    if (!done_fast) UQB_TRY(stats_generic(ctx, fq, s, (uint32_t)flen));
    UQB_TRY(stats_finish(ctx, fq, s, out, flen));
    UQB_TRY(uqb_dfree(ctx, s, sizeof(an_dev)));
    return 0;
}

// ================================================================================================
// Streamed load: H2D copy of the FASTQ in chunks on the copy stream while the compute stream splits and
// analyses every chunk as soon as it has landed (newline count -> line offsets -> record tiles of the
// records completed so far).  When the last chunk arrives the split and the Pass-1 statistics are
// done; uqb_split / uqb_analyze on the returned handle return them without touching the data again.
// ================================================================================================
extern "C" int uqb_fastq_load_streamed(uqb_ctx* ctx, const uint8_t* host, uint64_t nbytes, uint64_t chunk_bytes, uqb_fastq** out_fq) {
    return uqb_fastq_load_streamed_ref(ctx, host, nbytes, chunk_bytes, nullptr, 0, 0, out_fq);
}

// as above for a multi-GPU shard: statistics are measured against the global first QNAME line `ref`; rbase > 0
// says that this shard does not start the file (its first record takes part in the prefix/suffix statistics)
extern "C" int uqb_fastq_load_streamed_ref(uqb_ctx* ctx, const uint8_t* host, uint64_t nbytes, uint64_t chunk_bytes,
                                           const uint8_t* ref, uint32_t ref_len, uint64_t rbase, uqb_fastq** out_fq) {
    if (chunk_bytes == 0) chunk_bytes = 256ull << 20;
    chunk_bytes = (chunk_bytes + UQB_SPLIT_TILE - 1) / UQB_SPLIT_TILE * UQB_SPLIT_TILE;
    cudaStream_t cs;
    UQB_TRY(uqb_copy_stream(ctx, &cs));
    uqb_fastq* fq = new uqb_fastq();
    *out_fq = fq;
    uint8_t* d;
    UQB_TRY(uqb_dalloc(ctx, (void**)&d, nbytes + 64));
    fq->d = d; fq->n = nbytes; fq->owned = true; fq->streamed = true;
    UQB_CUDA(cudaMemsetAsync(d + nbytes, 0, 64, ctx->stream));
    if (ref) UQB_TRY(uqb_fastq_set_reference(ctx, fq, ref, ref_len, rbase));
    const uint64_t nchunks = (nbytes + chunk_bytes - 1) / chunk_bytes;
    // all copies are queued up front; one event per chunk gates the compute stream
    std::vector<cudaEvent_t> ev(nchunks);
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));        // the destination buffer may be recycled arena memory still in use
    for (uint64_t c = 0; c < nchunks; c++) {
        const uint64_t off = c * chunk_bytes, len = (off + chunk_bytes <= nbytes) ? chunk_bytes : nbytes - off;
        UQB_CUDA(cudaMemcpyAsync(d + off, host + off, len, cudaMemcpyHostToDevice, cs));
        UQB_CUDA(cudaEventCreateWithFlags(&ev[c], cudaEventDisableTiming));
        UQB_CUDA(cudaEventRecord(ev[c], cs));
    }
    const uint64_t ntiles = (nbytes + UQB_SPLIT_TILE - 1) / UQB_SPLIT_TILE;
    uint32_t* counts = nullptr;
    uint64_t *bases = nullptr, *d_total = nullptr;
    an_dev* s = nullptr;
    unsigned int* d_fb = nullptr;
    if (ntiles) {
        UQB_TRY(uqb_dalloc_t(ctx, &counts, ntiles));
        UQB_TRY(uqb_dalloc_t(ctx, &bases, ntiles));
    }
    UQB_TRY(uqb_dalloc_t(ctx, &d_total, 1));
    UQB_TRY(uqb_dalloc_t(ctx, &s, 1));
    UQB_TRY(uqb_dalloc_t(ctx, &d_fb, 1));
    UQB_CUDA(cudaMemsetAsync(d_fb, 0, 4, ctx->stream));
    UQB_LAUNCH(k_an_init, 1, 256, 0, s);
    uint64_t lines_done = 0, cap = 0, recs_done = 0, flen = 0;
    bool tiles_ok = true, have_first = false;
    uqb_stats* st = new uqb_stats();
    memset(st, 0, sizeof(*st));
    fq->cached_stats = st;
    for (uint64_t c = 0; c < nchunks; c++) {
        const uint64_t off = c * chunk_bytes, end = (off + chunk_bytes <= nbytes) ? off + chunk_bytes : nbytes;
        const uint64_t t0 = off / UQB_SPLIT_TILE, t1 = (end + UQB_SPLIT_TILE - 1) / UQB_SPLIT_TILE;
        UQB_CUDA(cudaStreamWaitEvent(ctx->stream, ev[c], 0));
        UQB_TRY(uqb_split_count_tiles(ctx, d, end, t0, t1 - t0, counts));
        UQB_TRY(uqb_scan_u32_to_u64(ctx, counts + t0, bases + t0, t1 - t0, d_total));
        uint64_t chunk_lines = 0;
        UQB_TRY(uqb_readback(ctx, &chunk_lines, d_total, 8));
        if (lines_done + chunk_lines + 1 > cap) {        // (re)size the line-offset array from the density seen so far
            const double density = (double)(lines_done + chunk_lines + 1) / (double)end;
            uint64_t want = (uint64_t)(density * (double)nbytes * 1.05) + 4096;
            if (want < lines_done + chunk_lines + 1) want = lines_done + chunk_lines + 1;
            uint64_t* nl;
            UQB_TRY(uqb_dalloc_t(ctx, &nl, want));
            if (fq->line_off) {
                UQB_CUDA(cudaMemcpyAsync(nl, fq->line_off, (lines_done + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
                UQB_TRY(uqb_dfree(ctx, fq->line_off, 0));
            } else {
                UQB_TRY(uqb_split_set_first(ctx, nl));
            }
            fq->line_off = nl;
            cap = want;
        }
        UQB_TRY(uqb_split_write_tiles(ctx, d, end, t0, t1 - t0, lines_done, bases, fq->line_off));
        lines_done += chunk_lines;
        fq->n_lines = lines_done;
        fq->n_reads = lines_done / 4;
        // Pass-1 statistics of the records that are complete now
        const uint64_t recs_now = lines_done / 4;
        if (recs_now > 0 && !have_first) {
            uint64_t offs[2];
            UQB_TRY(uqb_readback(ctx, offs, fq->line_off, 16));
            flen = offs[1] - offs[0] - 1;
            if (flen > UQB_HDR_MAX) return uqb_fail(ctx, "QNAME line longer than %d bytes is not supported by the device path", UQB_HDR_MAX);
            if (fq->ref_name) flen = fq->ref_len;
            have_first = true;
            // records of typical short-read files fit the tiles; otherwise the generic kernels run at the end
            tiles_ok = true;
        }
        if (have_first && tiles_ok && recs_now > recs_done) {
            if ((double)end / (double)recs_now > (double)((TL_CAP - 64) / TL_R)) tiles_ok = false;
            else UQB_TRY(stats_tiles_range(ctx, fq, s, d_fb, (uint32_t)flen, recs_done, recs_now));
            recs_done = recs_now;
        }
    }
    for (auto e : ev) cudaEventDestroy(e);
    if (counts) { UQB_TRY(uqb_dfree(ctx, counts, 0)); UQB_TRY(uqb_dfree(ctx, bases, 0)); }
    UQB_TRY(uqb_dfree(ctx, d_total, 0));
    if (!fq->line_off) { UQB_TRY(uqb_dalloc_t(ctx, &fq->line_off, 1)); UQB_TRY(uqb_split_set_first(ctx, fq->line_off)); }
    int rc = 0;
    if (fq->n_reads > 0) {
        unsigned int fb = 0;
        UQB_TRY(uqb_readback(ctx, &fb, d_fb, 4));
        uint64_t fl2 = 0;
        UQB_TRY(stats_names(ctx, fq, st, &fl2));
        if (fq->ref_name) fl2 = fq->ref_len;
        if (!tiles_ok || fb != 0) UQB_TRY(stats_generic(ctx, fq, s, (uint32_t)fl2));
        rc = stats_finish(ctx, fq, s, st, fl2);
    } else {
        delete st;
        fq->cached_stats = nullptr;
    }
    UQB_TRY(uqb_dfree(ctx, s, 0));
    UQB_TRY(uqb_dfree(ctx, d_fb, 0));
    return rc;
}
