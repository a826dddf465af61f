// Internal definitions shared by the translation units of libuqb200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/uqb200.h"

#define UQB_SM_COUNT 148   // B200: 2 dies x 74 SMs; persistent grids are sized in multiples of this

struct uqb_timer_rec { const char* name; cudaEvent_t a, b; uint64_t bytes; };
struct uqb_timer_tot { uint64_t launches = 0; double ms = 0; uint64_t bytes = 0; };

// Device memory arena: ONE contiguous virtual address range per context, backed on demand by physical
// chunks (CUDA virtual memory management), with a first-fit free list on top.  All work of a context is
// on one stream, so a freed block may be handed out again immediately (stream order = program order).
// Sized for a 180 GB part: nothing is ever returned to the driver before the context dies, so the
// steady-state cost of an allocation is a map lookup instead of a driver call.
struct uqb_arena {
    unsigned long long base = 0;      // CUdeviceptr
    uint64_t reserved = 0;            // bytes of virtual address space
    uint64_t mapped = 0;              // bytes backed by physical memory, [base, base + mapped)
    uint64_t granularity = 0;
    std::map<uint64_t, uint64_t> free_by_off;           // offset -> size
    std::map<uint64_t, uint64_t> used;                  // offset -> size
    std::vector<unsigned long long> handles;            // CUmemGenericAllocationHandle per chunk
    std::vector<std::pair<uint64_t, uint64_t>> chunks;  // (offset, size) per chunk
};

struct uqb_ctx {
    int device = 0;
    uqb_arena arena;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;      // H2D / D2H copies that overlap the compute stream
    char err[512] = {0};
    uint64_t launches = 0;
    uint64_t bytes_in_use = 0;
    int sm_count = UQB_SM_COUNT;
    std::vector<const void*> copies_in_flight;   // sources of async device->host copies queued since the last copy sync
    // pinned scratch for small device->host read-backs
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    // optional per-kernel timing
    bool timing = false;
    std::vector<uqb_timer_rec> pending;
    std::vector<cudaEvent_t> free_events;
    std::map<std::string, uqb_timer_tot> totals;
    cudaEvent_t span_a = nullptr, span_b = nullptr;   // uqb_ctx_span_begin / _end
};

struct uqb_array {
    void* d = nullptr;
    uint64_t n = 0;
    uint32_t width = 0;
    bool owned = true;
    uint64_t* key0 = nullptr;     // optional (owned): be64 of the first 8 bytes of every row, written by the producer of the table
    uint64_t nbytes() const { return n * (uint64_t)width; }
};

struct uqb_qcol {                 // per QNAME column device state produced by uqb_qname_scan
    int64_t* val = nullptr;       // parsed integer value per record (valid where the token is an integer)
    uint32_t* span = nullptr;     // (start<<16 | len) of the token inside the QNAME middle part
    uint32_t* rank = nullptr;     // rank of the token in the sorted dictionary (filled lazily)
    uint32_t* first_occ = nullptr;// first record holding each dictionary entry
    uint8_t* dict = nullptr;      // sorted distinct tokens, zero padded rows
    uint64_t dict_count = 0;
    uint32_t dict_width = 0;
};

struct uqb_fastq {
    const uint8_t* d = nullptr;   // FASTQ bytes (readable up to n + 64 when owned)
    uint64_t n = 0;
    bool owned = false;
    uint64_t* line_off = nullptr; // uint64[n_lines + 1]
    uint64_t n_lines = 0, n_reads = 0;
    uint64_t total_bases = 0;     // sum of read lengths (set by uqb_analyze; bookkeeping for byte counts)
    // multi-GPU: a shard compares its QNAME lines with the GLOBAL first line and knows its first global record
    uint8_t* ref_name = nullptr;
    uint32_t ref_len = 0;
    uint64_t rbase = 0;
    // QNAME lines in a compact side array (row r: length byte + text, name_pitch bytes), written by the histogram kernel
    // of uqb_analyze (k_pair_hist_pipe) - it stays with the handle
    uint8_t* names = nullptr;
    uint32_t name_pitch = 0;
    uint64_t names_cap = 0;
    bool streamed = false;        // split + Pass-1 statistics were produced while the bytes streamed in
    uqb_stats* cached_stats = nullptr;
    uint32_t prefix_len = 0, suffix_len = 0, ncols = 0;
    std::vector<uqb_qcol> qcols;
};

// ---- error handling ---------------------------------------------------------------------------
int uqb_fail(uqb_ctx* ctx, const char* fmt, ...);

#define UQB_CUDA(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            return uqb_fail(ctx, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
    } while (0)

#define UQB_TRY(expr)                                                                        \
    do {                                                                                     \
        int _r = (expr);                                                                     \
        if (_r != 0) return _r;                                                              \
    } while (0)

// ---- memory ------------------------------------------------------------------------------------
int uqb_dalloc(uqb_ctx* ctx, void** p, size_t nbytes);            // stream-ordered
int uqb_dfree(uqb_ctx* ctx, void* p, size_t nbytes);
int uqb_new_array(uqb_ctx* ctx, uint64_t n, uint32_t width, uqb_array** out);
int uqb_adopt_array(uqb_ctx* ctx, void* d, uint64_t n, uint32_t width, uqb_array** out);   // d: arena block of >= n * width + 64 bytes
int uqb_pinned(uqb_ctx* ctx, size_t nbytes, void** out);          // ctx-owned scratch, grows
int uqb_readback(uqb_ctx* ctx, void* host, const void* dev, size_t nbytes);   // D2H + sync

template <typename T>
static inline int uqb_dalloc_t(uqb_ctx* ctx, T** p, size_t count) {
    return uqb_dalloc(ctx, (void**)p, count * sizeof(T));
}

// ---- launches ----------------------------------------------------------------------------------
void uqb_timer_begin(uqb_ctx* ctx, const char* name, uint64_t bytes);
void uqb_timer_end(uqb_ctx* ctx);
void uqb_timer_add_bytes(uqb_ctx* ctx, uint64_t bytes);   // adds to the most recent launch record (when the size is known late)

// Launch a kernel on the context stream, count it, optionally time it, and check the launch.
// UQB_LAUNCH_B additionally records the kernel's ALGORITHMIC bytes (compulsory reads + writes) so that
// bench.py can report achieved bandwidth per kernel from the event timings.
#define UQB_LAUNCH(kernel, grid, block, smem, ...) UQB_LAUNCH_B(0, kernel, grid, block, smem, __VA_ARGS__)
#define UQB_LAUNCH_B(abytes, kernel, grid, block, smem, ...)                                 \
    do {                                                                                     \
        uqb_timer_begin(ctx, #kernel, (uint64_t)(abytes));                                   \
        kernel<<<(grid), (block), (smem), ctx->stream>>>(__VA_ARGS__);                       \
        uqb_timer_end(ctx);                                                                  \
        ctx->launches++;                                                                     \
        UQB_CUDA(cudaGetLastError());                                                        \
    } while (0)

static inline unsigned uqb_blocks(uint64_t n, unsigned per_block) {
    uint64_t b = (n + per_block - 1) / per_block;
    if (b == 0) b = 1;
    return (unsigned)b;
}

// grid for grid-stride kernels: enough CTAs to fill the machine several times, capped by the work
static inline unsigned uqb_grid(uqb_ctx* ctx, uint64_t n, unsigned per_block, unsigned waves = 8) {
    uint64_t need = (n + per_block - 1) / per_block;
    uint64_t cap = (uint64_t)ctx->sm_count * waves;
    if (need < 1) need = 1;
    return (unsigned)(need < cap ? need : cap);
}

// ---- device helpers ----------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

// 8 bytes starting at an arbitrary address, big-endian, zero padded beyond `avail` bytes
__device__ __forceinline__ uint64_t load_be64(const uint8_t* p, uint32_t avail) {
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t b = (uint32_t)i < avail ? (uint64_t)__ldg(p + i) : 0ull;
        v = (v << 8) | b;
    }
    return v;
}

__device__ __forceinline__ void atomic_min_i64(int64_t* addr, int64_t v) {
    atomicMin((long long*)addr, (long long)v);
}
__device__ __forceinline__ void atomic_max_i64(int64_t* addr, int64_t v) {
    atomicMax((long long*)addr, (long long)v);
}
#endif

// ---- split building blocks (split.cu) ------------------------------------------------------------
#define UQB_SPLIT_TILE (256 * 64)
int uqb_split_count_tiles(uqb_ctx* ctx, const uint8_t* d, uint64_t n_end, uint64_t tile0, uint64_t ntiles, uint32_t* counts);
int uqb_split_write_tiles(uqb_ctx* ctx, const uint8_t* d, uint64_t n_end, uint64_t tile0, uint64_t ntiles, uint64_t line_base,
                          const uint64_t* bases, uint64_t* line_off);
int uqb_split_set_first(uqb_ctx* ctx, uint64_t* line_off);
int uqb_copy_stream(uqb_ctx* ctx, cudaStream_t* out);
// frees the compact QNAME array of the handle (analyze.cu)
int uqb_names_release(uqb_ctx* ctx, uqb_fastq* fq);

// ---- primitives (prims.cu) ---------------------------------------------------------------------
// exclusive prefix sum of n uint32 values into uint32 / uint64; total written to *d_total (device)
int uqb_scan_u32(uqb_ctx* ctx, const uint32_t* d_in, uint32_t* d_out, uint64_t n, uint32_t* d_total);
int uqb_scan_u32_to_u64(uqb_ctx* ctx, const uint32_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total);

// Stable LSD radix sort of n records (key64, aux32, val32) by (aux32 major, key64 minor).
// Only the byte positions whose digit is not constant over the input are processed.
// On return *k, *a, *v point at the buffers holding the result (either the primary or alternate).
struct uqb_sortbuf {
    uint64_t* key[2] = {nullptr, nullptr};
    uint32_t* aux[2] = {nullptr, nullptr};   // may be null when unused
    uint32_t* val[2] = {nullptr, nullptr};
    int cur = 0;
    uint64_t cap = 0;
};
int uqb_sortbuf_alloc(uqb_ctx* ctx, uqb_sortbuf* sb, uint64_t n, bool with_aux);
int uqb_sortbuf_free(uqb_ctx* ctx, uqb_sortbuf* sb);
// key_first != nullptr: the input of the first pass is (key_first[i], i) - buffer 0 of sb is scratch then
int uqb_radix_sort(uqb_ctx* ctx, uqb_sortbuf* sb, uint64_t n, bool use_aux, const uint64_t* key_first = nullptr);
// out[idx[p]] = val[p] through destination windows that fit the L2 (idx: a permutation of 0..n-1)
int uqb_scatter_pairs_u32(uqb_ctx* ctx, const uint32_t* idx, const uint32_t* val, uint64_t n, uint32_t* out);

// rows (sort.cu)
int uqb_sort_rows_impl(uqb_ctx* ctx, const uint8_t* rows, uint64_t n, uint32_t width,
                       uint32_t** d_perm, uint32_t** d_gid_sorted, uint64_t* n_unique, const uint64_t* key0 = nullptr,
                       uint64_t** sorted_keys = nullptr);
