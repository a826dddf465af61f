// Context, memory, arrays and the per-kernel timing facility of libuqb200.so.
#include "common.cuh"
#include <cstdlib>
#include <cuda.h>
#include <stdarg.h>
#include <new>

// ---- driver entry points for the VMM arena (resolved at run time: libuqb200.so does not link libcuda) ----
struct drv_api {
    CUresult (*GetGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*AddressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*Create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*Map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*SetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*Unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*Release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*AddressFree)(CUdeviceptr, size_t) = nullptr;
    bool ok = false;
};
static drv_api g_drv;

static int load_driver(uqb_ctx* ctx) {
    if (g_drv.ok) return 0;
    struct { const char* name; void** fn; } tab[] = {
        {"cuMemGetAllocationGranularity", (void**)&g_drv.GetGranularity}, {"cuMemAddressReserve", (void**)&g_drv.AddressReserve},
        {"cuMemCreate", (void**)&g_drv.Create}, {"cuMemMap", (void**)&g_drv.Map}, {"cuMemSetAccess", (void**)&g_drv.SetAccess},
        {"cuMemUnmap", (void**)&g_drv.Unmap}, {"cuMemRelease", (void**)&g_drv.Release}, {"cuMemAddressFree", (void**)&g_drv.AddressFree}};
    for (auto& t : tab) {
        cudaDriverEntryPointQueryResult st;
        cudaError_t e = cudaGetDriverEntryPoint(t.name, t.fn, cudaEnableDefault, &st);
        if (e != cudaSuccess || st != cudaDriverEntryPointSuccess || !*t.fn)
            return uqb_fail(ctx, "cannot resolve driver entry point %s", t.name);
    }
    g_drv.ok = true;
    return 0;
}

static inline uint64_t round_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

static int arena_init(uqb_ctx* ctx) {
    UQB_TRY(load_driver(ctx));
    uqb_arena& A = ctx->arena;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = ctx->device;
    size_t gran = 0;
    if (g_drv.GetGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0)
        return uqb_fail(ctx, "cuMemGetAllocationGranularity failed");
    A.granularity = gran;
    size_t f = 0, t = 0;
    UQB_CUDA(cudaMemGetInfo(&f, &t));
    A.reserved = round_up((uint64_t)t, gran);
    CUdeviceptr base = 0;
    if (g_drv.AddressReserve(&base, A.reserved, 0, 0, 0) != CUDA_SUCCESS)
        return uqb_fail(ctx, "cuMemAddressReserve of %llu bytes failed", (unsigned long long)A.reserved);
    A.base = base;
    A.mapped = 0;
    return 0;
}

static void arena_destroy(uqb_ctx* ctx) {
    uqb_arena& A = ctx->arena;
    if (!g_drv.ok || !A.base) return;
    for (size_t i = 0; i < A.handles.size(); i++) {
        g_drv.Unmap(A.base + A.chunks[i].first, A.chunks[i].second);
        g_drv.Release(A.handles[i]);
    }
    g_drv.AddressFree(A.base, A.reserved);
    A = uqb_arena();
}

// back [mapped, mapped + at_least) with physical memory
static int arena_grow(uqb_ctx* ctx, uint64_t at_least) {
    uqb_arena& A = ctx->arena;
    const uint64_t min_chunk = 1ull << 30;
    uint64_t chunk = round_up(at_least > min_chunk ? at_least : min_chunk, A.granularity);
    if (A.mapped + chunk > A.reserved) chunk = round_up(at_least, A.granularity);
    if (A.mapped + chunk > A.reserved)
        return uqb_fail(ctx, "device arena exhausted: %llu bytes mapped, %llu more requested", (unsigned long long)A.mapped, (unsigned long long)at_least);
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = ctx->device;
    CUmemGenericAllocationHandle h;
    CUresult r = g_drv.Create(&h, chunk, &prop, 0);
    if (r != CUDA_SUCCESS && chunk > round_up(at_least, A.granularity)) {
        chunk = round_up(at_least, A.granularity);
        r = g_drv.Create(&h, chunk, &prop, 0);
    }
    if (r != CUDA_SUCCESS) return uqb_fail(ctx, "out of device memory: cuMemCreate(%llu) failed (%d) with %llu bytes already mapped", (unsigned long long)chunk, (int)r, (unsigned long long)A.mapped);
    if (g_drv.Map(A.base + A.mapped, chunk, 0, h, 0) != CUDA_SUCCESS) { g_drv.Release(h); return uqb_fail(ctx, "cuMemMap failed"); }
    CUmemAccessDesc acc = {};
    acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    acc.location.id = ctx->device;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (g_drv.SetAccess(A.base + A.mapped, chunk, &acc, 1) != CUDA_SUCCESS) return uqb_fail(ctx, "cuMemSetAccess failed");
    A.handles.push_back(h);
    A.chunks.push_back({A.mapped, chunk});
    // append to the free list, merging with a free block that ends at the old frontier
    uint64_t off = A.mapped, size = chunk;
    if (!A.free_by_off.empty()) {
        auto last = std::prev(A.free_by_off.end());
        if (last->first + last->second == A.mapped) { off = last->first; size += last->second; A.free_by_off.erase(last); }
    }
    A.free_by_off[off] = size;
    A.mapped += chunk;
    return 0;
}

int uqb_fail(uqb_ctx* ctx, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    if (ctx) vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
    va_end(ap);
    return 1;
}

extern "C" int uqb_version(void) { return UQB_VERSION; }

extern "C" int uqb_ctx_create(int device, void* stream, uqb_ctx** out) {
    if (!out) return 1;
    *out = nullptr;
    uqb_ctx* ctx = new (std::nothrow) uqb_ctx();
    if (!ctx) return 1;
    *out = ctx;       // returned even on failure so that the caller can read the error text
    ctx->device = device;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return uqb_fail(ctx, "no CUDA device available (%s); libuqb200 has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= count) return uqb_fail(ctx, "device %d out of range (%d devices)", device, count);
    UQB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    UQB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return uqb_fail(ctx, "device %d is sm_%d%d; libuqb200 is built for sm_100a (B200) only", device, prop.major, prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    if (stream) {
        ctx->stream = (cudaStream_t)stream;
        ctx->own_stream = false;
    } else {
        UQB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    UQB_CUDA(cudaFree(0));            // make sure the primary context exists before driver-level calls
    UQB_TRY(arena_init(ctx));
    return 0;
}

extern "C" void uqb_ctx_destroy(uqb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& r : ctx->pending) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : ctx->free_events) cudaEventDestroy(e);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->span_a) { cudaEventDestroy(ctx->span_a); cudaEventDestroy(ctx->span_b); }
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    arena_destroy(ctx);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* uqb_last_error(const uqb_ctx* ctx) { return ctx ? ctx->err : "null context"; }

extern "C" int uqb_ctx_sync(uqb_ctx* ctx) {
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" uint64_t uqb_ctx_launch_count(const uqb_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---- timing ------------------------------------------------------------------------------------
static cudaEvent_t get_event(uqb_ctx* ctx) {
    if (!ctx->free_events.empty()) {
        cudaEvent_t e = ctx->free_events.back();
        ctx->free_events.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void uqb_timer_begin(uqb_ctx* ctx, const char* name, uint64_t bytes) {
    if (!ctx->timing) return;
    uqb_timer_rec r;
    r.name = name;
    r.bytes = bytes;
    r.a = get_event(ctx);
    r.b = get_event(ctx);
    cudaEventRecord(r.a, ctx->stream);
    ctx->pending.push_back(r);
}

void uqb_timer_end(uqb_ctx* ctx) {
    if (!ctx->timing) return;
    cudaEventRecord(ctx->pending.back().b, ctx->stream);
}

void uqb_timer_add_bytes(uqb_ctx* ctx, uint64_t bytes) {
    if (!ctx->timing || ctx->pending.empty()) return;
    ctx->pending.back().bytes += bytes;
}

static void drain_timers(uqb_ctx* ctx) {
    if (ctx->pending.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (auto& r : ctx->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
            auto& t = ctx->totals[r.name];
            t.launches += 1;
            t.ms += ms;
            t.bytes += r.bytes;
        }
        ctx->free_events.push_back(r.a);
        ctx->free_events.push_back(r.b);
    }
    ctx->pending.clear();
}

extern "C" int uqb_ctx_timing(uqb_ctx* ctx, int enable) {
    drain_timers(ctx);
    ctx->timing = enable != 0;
    return 0;
}

extern "C" int uqb_ctx_timing_reset(uqb_ctx* ctx) {
    drain_timers(ctx);
    ctx->totals.clear();
    return 0;
}

extern "C" int uqb_ctx_timing_report(uqb_ctx* ctx, char* names, uint64_t* launches, double* ms, uint64_t* bytes, int cap, int* n) {
    drain_timers(ctx);
    int i = 0;
    for (auto& kv : ctx->totals) {
        if (i >= cap) break;
        snprintf(names + (size_t)i * UQB_TIMER_NAME, UQB_TIMER_NAME, "%s", kv.first.c_str());
        launches[i] = kv.second.launches;
        ms[i] = kv.second.ms;
        bytes[i] = kv.second.bytes;
        i++;
    }
    *n = i;
    return 0;
}

// device time between two points of the context's stream (includes host gaps in between)
extern "C" int uqb_ctx_span_begin(uqb_ctx* ctx) {
    if (!ctx->span_a) { UQB_CUDA(cudaEventCreate(&ctx->span_a)); UQB_CUDA(cudaEventCreate(&ctx->span_b)); }
    UQB_CUDA(cudaEventRecord(ctx->span_a, ctx->stream));
    return 0;
}
extern "C" int uqb_ctx_span_end(uqb_ctx* ctx, double* ms) {
    if (!ctx->span_a) return uqb_fail(ctx, "span_end without span_begin");
    UQB_CUDA(cudaEventRecord(ctx->span_b, ctx->stream));
    UQB_CUDA(cudaEventSynchronize(ctx->span_b));
    float f = 0.f;
    UQB_CUDA(cudaEventElapsedTime(&f, ctx->span_a, ctx->span_b));
    *ms = f;
    return 0;
}

// ---- memory ------------------------------------------------------------------------------------
int uqb_dalloc(uqb_ctx* ctx, void** p, size_t nbytes) {
    *p = nullptr;
    uqb_arena& A = ctx->arena;
    const uint64_t want = round_up(nbytes ? nbytes : 1, 256);
    // best fit over the free list (a few hundred blocks at most)
    auto best = A.free_by_off.end();
    for (auto it = A.free_by_off.begin(); it != A.free_by_off.end(); ++it)
        if (it->second >= want && (best == A.free_by_off.end() || it->second < best->second)) best = it;
    if (best == A.free_by_off.end()) {
        uint64_t tail = 0;
        if (!A.free_by_off.empty()) {
            auto last = std::prev(A.free_by_off.end());
            if (last->first + last->second == A.mapped) tail = last->second;
        }
        UQB_TRY(arena_grow(ctx, want - tail));
        best = std::prev(A.free_by_off.end());
        if (best->second < want) return uqb_fail(ctx, "device arena: internal error after growth");
    }
    const uint64_t off = best->first, size = best->second;
    A.free_by_off.erase(best);
    if (size > want) A.free_by_off[off + want] = size - want;
    A.used[off] = want;
    ctx->bytes_in_use += want;
    *p = (void*)(uintptr_t)(A.base + off);
    return 0;
}

int uqb_dfree(uqb_ctx* ctx, void* p, size_t /*nbytes*/) {
    if (!p) return 0;
    // a block that an async device->host copy still reads (an array dropped without uqb_ctx_copy_sync, e.g. by an error
    // path or a garbage collector) must not be recycled under the DMA engine: wait for the copy stream first
    if (!ctx->copies_in_flight.empty()) {
        for (const void* q : ctx->copies_in_flight)
            if (q == p) {
                if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
                ctx->copies_in_flight.clear();
                break;
            }
    }
    uqb_arena& A = ctx->arena;
    const uint64_t off = (uint64_t)(uintptr_t)p - A.base;
    auto u = A.used.find(off);
    if (u == A.used.end()) return uqb_fail(ctx, "device arena: free of an unknown pointer");
    uint64_t size = u->second, start = off;
    A.used.erase(u);
    ctx->bytes_in_use -= size;
    auto next = A.free_by_off.lower_bound(start);
    if (next != A.free_by_off.end() && start + size == next->first) { size += next->second; next = A.free_by_off.erase(next); }
    if (next != A.free_by_off.begin()) {
        auto prev = std::prev(next);
        if (prev->first + prev->second == start) { start = prev->first; size += prev->second; A.free_by_off.erase(prev); }
    }
    A.free_by_off[start] = size;
    return 0;
}

int uqb_new_array(uqb_ctx* ctx, uint64_t n, uint32_t width, uqb_array** out) {
    uqb_array* a = new (std::nothrow) uqb_array();
    if (!a) return uqb_fail(ctx, "out of host memory");
    a->n = n;
    a->width = width;
    a->owned = true;
    // +64 slack so that vectorised tails may over-read/over-write safely
    int r = uqb_dalloc(ctx, &a->d, a->nbytes() + 64);
    if (r) { delete a; return r; }
    *out = a;
    return 0;
}

// an arena block (at least n * width + 64 bytes) becomes an owned array
int uqb_adopt_array(uqb_ctx* ctx, void* d, uint64_t n, uint32_t width, uqb_array** out) {
    uqb_array* a = new (std::nothrow) uqb_array();
    if (!a) return uqb_fail(ctx, "out of host memory");
    a->n = n;
    a->width = width;
    a->owned = true;
    a->d = d;
    *out = a;
    return 0;
}

int uqb_pinned(uqb_ctx* ctx, size_t nbytes, void** out) {
    if (ctx->pinned_bytes < nbytes) {
        if (ctx->pinned) { cudaStreamSynchronize(ctx->stream); cudaFreeHost(ctx->pinned); ctx->pinned = nullptr; ctx->pinned_bytes = 0; }
        size_t want = nbytes < (1u << 20) ? (1u << 20) : nbytes;
        UQB_CUDA(cudaHostAlloc(&ctx->pinned, want, cudaHostAllocMapped));
        ctx->pinned_bytes = want;
    }
    *out = ctx->pinned;
    return 0;
}

// Small device->host read-backs go through a copy KERNEL into mapped pinned memory, not through the
// DMA engine: a bulk D2H of finished output arrays may be in flight on the copy stream, and a tiny
// cudaMemcpy queued behind it would stall the control flow of the sort for the whole transfer.
__global__ void k_readback(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

int uqb_readback(uqb_ctx* ctx, void* host, const void* dev, size_t nbytes) {
    if (nbytes == 0) return 0;
    void* stage;
    UQB_TRY(uqb_pinned(ctx, nbytes, &stage));
    if (nbytes <= (1u << 20)) {
        void* dstage = nullptr;
        UQB_CUDA(cudaHostGetDevicePointer(&dstage, stage, 0));
        const unsigned blocks = (unsigned)((nbytes + 255) / 256 < 64 ? (nbytes + 255) / 256 : 64);
        k_readback<<<blocks, 256, 0, ctx->stream>>>((uint8_t*)dstage, (const uint8_t*)dev, nbytes);
        UQB_CUDA(cudaGetLastError());
    } else {
        UQB_CUDA(cudaMemcpyAsync(stage, dev, nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(host, stage, nbytes);
    return 0;
}

extern "C" int uqb_host_alloc(uqb_ctx* ctx, uint64_t nbytes, void** out) {
    UQB_CUDA(cudaHostAlloc(out, nbytes ? nbytes : 1, cudaHostAllocDefault));
    return 0;
}

extern "C" int uqb_host_free(uqb_ctx* ctx, void* p) {
    UQB_CUDA(cudaFreeHost(p));
    return 0;
}

extern "C" int uqb_mem_info(uqb_ctx* ctx, uint64_t* in_use, uint64_t* dev_free, uint64_t* dev_total) {
    size_t f = 0, t = 0;
    UQB_CUDA(cudaMemGetInfo(&f, &t));
    if (in_use) *in_use = ctx->bytes_in_use;
    if (dev_free) *dev_free = f;
    if (dev_total) *dev_total = t;
    return 0;
}

// ---- arrays ------------------------------------------------------------------------------------
extern "C" int uqb_array_info(const uqb_array* a, uint64_t* n, uint32_t* width) {
    if (!a) return 1;
    if (n) *n = a->n;
    if (width) *width = a->width;
    return 0;
}

extern "C" void* uqb_array_device_ptr(const uqb_array* a) { return a ? a->d : nullptr; }

extern "C" int uqb_array_alloc(uqb_ctx* ctx, uint64_t n, uint32_t width, uqb_array** out) {
    return uqb_new_array(ctx, n, width, out);
}

// view of device memory the caller owns (a peer's window, another context's array on the same device): never freed here
extern "C" int uqb_array_wrap(uqb_ctx* ctx, void* dev, uint64_t n, uint32_t width, uqb_array** out) {
    uqb_array* a = new (std::nothrow) uqb_array();
    if (!a) return uqb_fail(ctx, "out of host memory");
    a->d = dev; a->n = n; a->width = width; a->owned = false;
    *out = a;
    return 0;
}

// device -> device copy on the context's stream; `src_dev` may live in a peer GPU's memory (unified addressing)
extern "C" int uqb_array_copy_in(uqb_ctx* ctx, uqb_array* dst, uint64_t dst_offset, const void* src_dev, uint64_t nbytes) {
    if (dst_offset + nbytes > dst->nbytes()) return uqb_fail(ctx, "copy_in: %llu bytes at offset %llu exceed an array of %llu",
                                                                (unsigned long long)nbytes, (unsigned long long)dst_offset, (unsigned long long)dst->nbytes());
    if (nbytes) UQB_CUDA(cudaMemcpyAsync((uint8_t*)dst->d + dst_offset, src_dev, nbytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}

extern "C" int uqb_array_upload(uqb_ctx* ctx, const void* host, uint64_t n, uint32_t width, uqb_array** out) {
    uqb_array* a;
    UQB_TRY(uqb_new_array(ctx, n, width, &a));
    if (a->nbytes()) {
        UQB_CUDA(cudaMemcpyAsync(a->d, host, a->nbytes(), cudaMemcpyHostToDevice, ctx->stream));
        UQB_CUDA(cudaStreamSynchronize(ctx->stream));   // the host buffer may be pageable
    }
    *out = a;
    return 0;
}

extern "C" int uqb_array_download(uqb_ctx* ctx, const uqb_array* a, void* host, uint64_t nbytes) {
    if (nbytes > a->nbytes()) return uqb_fail(ctx, "download of %llu bytes from an array of %llu", (unsigned long long)nbytes, (unsigned long long)a->nbytes());
    if (nbytes) UQB_CUDA(cudaMemcpyAsync(host, a->d, nbytes, cudaMemcpyDeviceToHost, ctx->stream));
    UQB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int uqb_copy_stream(uqb_ctx* ctx, cudaStream_t* out) {
    if (!ctx->copy_stream) UQB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    *out = ctx->copy_stream;
    return 0;
}

// D2H on the copy stream, ordered after everything enqueued so far on the compute stream; the array must
// stay allocated until uqb_ctx_copy_sync() returns.
extern "C" int uqb_array_download_async(uqb_ctx* ctx, const uqb_array* a, void* host, uint64_t nbytes) {
    if (nbytes > a->nbytes()) return uqb_fail(ctx, "async download of %llu bytes from an array of %llu", (unsigned long long)nbytes, (unsigned long long)a->nbytes());
    cudaStream_t cs;
    UQB_TRY(uqb_copy_stream(ctx, &cs));
    cudaEvent_t ev;
    UQB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    UQB_CUDA(cudaEventRecord(ev, ctx->stream));
    UQB_CUDA(cudaStreamWaitEvent(cs, ev, 0));
    UQB_CUDA(cudaEventDestroy(ev));                      // released once the wait has consumed it
    if (nbytes) {
        UQB_CUDA(cudaMemcpyAsync(host, a->d, nbytes, cudaMemcpyDeviceToHost, cs));
        ctx->copies_in_flight.push_back(a->d);           // uqb_dfree waits for the copy before it recycles the block
    }
    return 0;
}

extern "C" int uqb_ctx_copy_sync(uqb_ctx* ctx) {
    if (ctx->copy_stream) UQB_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    ctx->copies_in_flight.clear();
    return 0;
}

// byte-wise comparison of two device arrays (full-size round-trip checks without a 34 GB host copy)
__global__ void k_first_diff(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint64_t n, unsigned long long* __restrict__ first) {
    unsigned long long best = ~0ull;
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; i < n; i += (uint64_t)gridDim.x * blockDim.x * 16) {
        if (i + 16 <= n) {
            const uint4 x = *reinterpret_cast<const uint4*>(a + i), y = *reinterpret_cast<const uint4*>(b + i);
            if (x.x != y.x || x.y != y.y || x.z != y.z || x.w != y.w) {
                for (int k = 0; k < 16; k++) if (a[i + k] != b[i + k]) { if (i + k < best) best = i + k; break; }
            }
        } else {
            for (uint64_t k = i; k < n; k++) if (a[k] != b[k]) { if (k < best) best = k; break; }
        }
    }
    if (best != ~0ull) atomicMin(first, best);
}

extern "C" int uqb_array_first_difference(uqb_ctx* ctx, const uqb_array* a, const uqb_array* b, int64_t* first) {
    if (a->nbytes() != b->nbytes()) { *first = (int64_t)(a->nbytes() < b->nbytes() ? a->nbytes() : b->nbytes()); return 0; }
    unsigned long long* d;
    UQB_TRY(uqb_dalloc_t(ctx, &d, 1));
    UQB_CUDA(cudaMemsetAsync(d, 0xFF, 8, ctx->stream));
    const uint64_t n = a->nbytes();
    if (n) UQB_LAUNCH_B(2 * n, k_first_diff, uqb_grid(ctx, n, 256 * 16, 16), 256, 0, (const uint8_t*)a->d, (const uint8_t*)b->d, n, d);
    unsigned long long h = 0;
    UQB_TRY(uqb_readback(ctx, &h, d, 8));
    UQB_TRY(uqb_dfree(ctx, d, 8));
    *first = h == ~0ull ? -1 : (int64_t)h;
    return 0;
}

extern "C" int uqb_array_free(uqb_ctx* ctx, uqb_array* a) {
    if (!a) return 0;
    int r = 0;
    if (a->owned) r = uqb_dfree(ctx, a->d, a->nbytes() + 64);
    if (a->key0) { const int r2 = uqb_dfree(ctx, a->key0, a->n * 8); if (!r) r = r2; }
    delete a;
    return r;
}
