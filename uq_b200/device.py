"""Thin object wrappers over the C ABI (include/uqb200.h).  No computation happens here: every method
is one call into libuqb200.so; numpy is used only as host memory."""
import ctypes as C

import numpy as np

from . import _lib as L

PATTERN_ID = {'0.1': 0, '1.1': 1, '2.1': 2, '3.1': 3, '0.2': 4, '1.2': 5, '2.2': 6, '3.2': 7}


class DeviceError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _plan_arrays(plan):
    n = len(plan)
    return ((C.c_uint32 * n)(*[int(s) for s, _, _ in plan]), (C.c_uint32 * n)(*[int(b) for _, b, _ in plan]),
            (C.c_uint64 * n)(*[int(a) for _, _, a in plan]))


class Context:
    """One per host thread.  `stream` may be a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""

    def __init__(self, device=0, stream=None):
        self.lib = L.load()
        self.h = C.c_void_p()
        rc = self.lib.uqb_ctx_create(int(device), C.c_void_p(stream or 0), C.byref(self.h))
        if rc:
            msg = self.lib.uqb_last_error(self.h).decode() if self.h else "context allocation failed"
            if self.h:
                self.lib.uqb_ctx_destroy(self.h)
                self.h = C.c_void_p()
            raise DeviceError("uq_b200: cannot create a CUDA context on device %d: %s" % (device, msg))
        self.device = device

    def close(self):
        if self.h:
            self.lib.uqb_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc:
            raise DeviceError(self.lib.uqb_last_error(self.h).decode())

    def sync(self):
        self.check(self.lib.uqb_ctx_sync(self.h))

    @property
    def launches(self):
        return int(self.lib.uqb_ctx_launch_count(self.h))

    def timing(self, enable):
        self.check(self.lib.uqb_ctx_timing(self.h, 1 if enable else 0))

    def timing_reset(self):
        self.check(self.lib.uqb_ctx_timing_reset(self.h))

    def timing_report(self):
        cap = 256
        names = C.create_string_buffer(cap * L.TIMER_NAME)
        cnt = (C.c_uint64 * cap)()
        ms = (C.c_double * cap)()
        nb = (C.c_uint64 * cap)()
        n = C.c_int()
        self.check(self.lib.uqb_ctx_timing_report(self.h, names, cnt, ms, nb, cap, C.byref(n)))
        out = {}
        for i in range(n.value):
            nm = names.raw[i * L.TIMER_NAME:(i + 1) * L.TIMER_NAME].split(b"\0")[0].decode()
            out[nm] = (int(cnt[i]), float(ms[i]), int(nb[i]))
        return out

    def span_begin(self):
        self.check(self.lib.uqb_ctx_span_begin(self.h))

    def span_end(self):
        ms = C.c_double()
        self.check(self.lib.uqb_ctx_span_end(self.h, C.byref(ms)))
        return float(ms.value)

    def mem_info(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self.check(self.lib.uqb_mem_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    # ---- pinned host memory ----
    def pinned_empty(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.uqb_host_alloc(self.h, int(nbytes), C.byref(p)))
        buf = (C.c_uint8 * max(int(nbytes), 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8, count=int(nbytes))
        return PinnedBuffer(self, p, arr)

    # ---- arrays ----
    def upload(self, arr, width=None):
        arr = np.ascontiguousarray(arr)
        if width is None:
            width = arr.dtype.itemsize if arr.ndim == 1 else arr.shape[1] * arr.dtype.itemsize
        n = arr.nbytes // width if width else arr.shape[0]
        h = C.c_void_p()
        self.check(self.lib.uqb_array_upload(self.h, _ptr(arr), int(n), int(width), C.byref(h)))
        return DeviceArray(self, h)

    def alloc(self, n, width):
        """uninitialised device array of n rows x width bytes"""
        h = C.c_void_p()
        self.check(self.lib.uqb_array_alloc(self.h, int(n), int(width), C.byref(h)))
        return DeviceArray(self, h)

    def wrap(self, dev_ptr, n, width):
        """non-owning DeviceArray over device memory somebody else owns (a peer's window, another context's array)"""
        h = C.c_void_p()
        self.check(self.lib.uqb_array_wrap(self.h, C.c_void_p(int(dev_ptr)), int(n), int(width), C.byref(h)))
        return DeviceArray(self, h)

    def copy_in(self, dst, dst_offset, src_ptr, nbytes):
        """device -> device copy from a raw device pointer (peer memory included) on this context's stream"""
        self.check(self.lib.uqb_array_copy_in(self.h, dst.h, int(dst_offset), C.c_void_p(int(src_ptr)), int(nbytes)))

    def index_u32(self, arr, bound):
        """index member of a container (uint8/16/32/64) -> (uint32 DeviceArray, first position with value >= bound or -1)"""
        h, bad = C.c_void_p(), C.c_int64()
        self.check(self.lib.uqb_index_u32(self.h, arr.h, int(bound), C.byref(h), C.byref(bad)))
        return DeviceArray(self, h), int(bad.value)

    def add_scalar_u32(self, arr, value):
        self.check(self.lib.uqb_add_scalar_u32(self.h, arr.h, int(value)))

    def gather_rows_segmented(self, table, order, seg_counts, align=128):
        """rows table[order[...]] gathered segment by segment into a byte array whose segments start at multiples of
        `align` bytes -> (DeviceArray of bytes, byte offset of every segment)"""
        counts = np.ascontiguousarray(seg_counts, dtype=np.uint64)
        offs = np.zeros(len(counts), dtype=np.uint64)
        h = C.c_void_p()
        self.check(self.lib.uqb_gather_rows_segmented(self.h, table.h, order.h, len(counts), _ptr(counts), int(align), C.byref(h), _ptr(offs)))
        return DeviceArray(self, h), [int(o) for o in offs]

    SCATTER_MAX_WIDTH = 224

    def partition_positions(self, table, split_keys):
        """rows -> destination ranks by their big-endian first 8 bytes (dest = number of split_keys <= key).
        -> (pos: uint32[n], pos[i] = index of row i in the destination-grouped stable order; counts per destination)"""
        keys = np.ascontiguousarray(split_keys, dtype=np.uint64)
        counts = np.zeros(len(keys) + 1, dtype=np.uint64)
        h = C.c_void_p()
        self.check(self.lib.uqb_partition_positions(self.h, table.h, _ptr(keys), len(keys), C.byref(h), _ptr(counts)))
        return DeviceArray(self, h), [int(c) for c in counts]

    def scatter_rows_segmented(self, table, pos, seg_counts, align=128):
        """row i of `table` -> its place pos[i] in a byte array whose segments start at multiples of `align` bytes
        -> (DeviceArray of bytes, byte offset of every segment); same layout as gather_rows_segmented"""
        counts = np.ascontiguousarray(seg_counts, dtype=np.uint64)
        offs = np.zeros(len(counts), dtype=np.uint64)
        h = C.c_void_p()
        self.check(self.lib.uqb_scatter_rows_segmented(self.h, table.h, pos.h, len(counts), _ptr(counts), int(align), C.byref(h), _ptr(offs)))
        return DeviceArray(self, h), [int(o) for o in offs]

    def scatter_rows_to(self, table, pos, seg_counts, dst_addrs):
        """row i of `table` -> device address dst_addrs[d] + (pos[i] - first row of d) * width (peer memory included)"""
        counts = np.ascontiguousarray(seg_counts, dtype=np.uint64)
        addrs = np.ascontiguousarray(dst_addrs, dtype=np.uint64)
        self.check(self.lib.uqb_scatter_rows_to(self.h, table.h, pos.h, len(counts), _ptr(counts), _ptr(addrs)))

    def compact_segments(self, padded, seg_offsets, seg_counts, width):
        """byte array with aligned segments -> dense table [sum(seg_counts)][width]"""
        offs = np.ascontiguousarray(seg_offsets, dtype=np.uint64)
        counts = np.ascontiguousarray(seg_counts, dtype=np.uint64)
        h = C.c_void_p()
        self.check(self.lib.uqb_compact_segments(self.h, padded.h, len(counts), _ptr(offs), _ptr(counts), int(width), C.byref(h)))
        return DeviceArray(self, h)

    def scatter_u32(self, src, idx):
        """out[idx[j]] = src[j] (uint32 arrays, idx a permutation)"""
        h = C.c_void_p()
        self.check(self.lib.uqb_scatter_u32(self.h, src.h, idx.h, C.byref(h)))
        return DeviceArray(self, h)

    def rows_lower_bound(self, sorted_table, probes):
        """lower_bound of every row of `probes` (uint8 [k][width], host) in a device table sorted in memcmp order"""
        probes = np.ascontiguousarray(probes, dtype=np.uint8)
        k = probes.shape[0]
        out = np.zeros(k, dtype=np.uint64)
        if k:
            self.check(self.lib.uqb_rows_lower_bound(self.h, sorted_table.h, _ptr(probes), int(k), _ptr(out)))
        return out

    def load_fastq(self, data):
        """H2D copy of FASTQ bytes (bytes / bytearray / uint8 ndarray / PinnedBuffer)."""
        if isinstance(data, PinnedBuffer):
            arr = data.array
        elif isinstance(data, np.ndarray):
            arr = np.ascontiguousarray(data, dtype=np.uint8)
        else:
            arr = np.frombuffer(data, dtype=np.uint8)
        h = C.c_void_p()
        self.check(self.lib.uqb_fastq_load(self.h, _ptr(arr) if arr.size else None, int(arr.size), C.byref(h)))
        return Fastq(self, h, int(arr.size))

    def load_fastq_streamed(self, data, chunk_bytes=0, ref=None, rbase=0):
        """H2D in chunks overlapped with record splitting and the Pass-1 statistics (data: PinnedBuffer or ndarray).
        ref / rbase: multi-GPU shard measured against the global first QNAME line (rbase > 0: not the first shard)."""
        arr = data.array if isinstance(data, PinnedBuffer) else np.ascontiguousarray(data, dtype=np.uint8)
        h = C.c_void_p()
        rb = np.frombuffer(b"" if ref is None else ref, dtype=np.uint8)
        rc = self.lib.uqb_fastq_load_streamed(self.h, _ptr(arr) if arr.size else None, int(arr.size), int(chunk_bytes),
                                              _ptr(rb) if rb.size else None, int(rb.size), int(rbase), C.byref(h))
        if rc:
            msg = self.lib.uqb_last_error(self.h).decode()
            if h:
                self.lib.uqb_fastq_free(self.h, h)
            raise DeviceError(msg)
        fq = Fastq(self, h, int(arr.size))
        fq.reference = ref
        return fq

    def copy_sync(self):
        self.check(self.lib.uqb_ctx_copy_sync(self.h))

    def adopt_fastq(self, device_array):
        """Wrap FASTQ bytes that already live in HBM (no copy); the array must outlive the Fastq."""
        h = C.c_void_p()
        self.check(self.lib.uqb_fastq_adopt(self.h, device_array.device_ptr, int(device_array.nbytes), C.byref(h)))
        fq = Fastq(self, h, int(device_array.nbytes))
        fq._keep = device_array
        return fq

    def synth(self, kind, n, length, seed, first=0, genome=0, pool=0, len_table=None):
        kinds = {"illumina": 0, "genome": 1, "casava": 2, "ont": 3, "umi": 4, "renamed": 5, "mixed": 6}
        p = L.SynthParams()
        p.kind = kinds[kind]
        if kind == "ont":
            p.len_lo, p.len_hi = int(length[0]), int(length[1])
            tab = np.ascontiguousarray(len_table, dtype=np.int64)
            assert tab.size == 4096
            tp = _ptr(tab)
        else:
            p.length = int(length)
            tp = None
        p.seed, p.first, p.n, p.genome, p.pool = int(seed), int(first), int(n), int(genome), int(pool)
        h = C.c_void_p()
        self.check(self.lib.uqb_synth(self.h, C.byref(p), tp, C.byref(h)))
        return DeviceArray(self, h)

    # ---- stage 3 / 4 ----
    def sort_rows(self, table, want_perm=False, want_key=False, want_uniq=False, want_key_sorted=False):
        """-> (perm, key, uniq, n_unique[, key_sorted])"""
        perm, key, uniq, ks = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        nu = C.c_uint64()
        self.check(self.lib.uqb_sort_rows(self.h, table.h, C.byref(perm) if want_perm else None,
                                          C.byref(key) if want_key else None, C.byref(ks) if want_key_sorted else None,
                                          C.byref(uniq) if want_uniq else None, C.byref(nu)))
        out = (DeviceArray(self, perm) if want_perm else None, DeviceArray(self, key) if want_key else None,
               DeviceArray(self, uniq) if want_uniq else None, int(nu.value))
        if want_key_sorted:
            out = out + (DeviceArray(self, ks),)
        return out

    def gather_rows(self, table, perm):
        h = C.c_void_p()
        self.check(self.lib.uqb_gather_rows(self.h, table.h, perm.h, C.byref(h)))
        return DeviceArray(self, h)

    def narrow_u32(self, a, itemsize):
        h = C.c_void_p()
        self.check(self.lib.uqb_narrow_u32(self.h, a.h, int(itemsize), C.byref(h)))
        return DeviceArray(self, h)

    def columns_to_rows(self, cols, kinds=None):
        """columns -> sort rows; kinds[c]: 0 little-endian integer (big-endian in the row), 1 bytes as they are"""
        arr = (C.c_void_p * len(cols))(*[c.h for c in cols])
        h = C.c_void_p()
        k = None if kinds is None else np.ascontiguousarray(kinds, dtype=np.uint8)
        self.check(self.lib.uqb_columns_to_rows(self.h, len(cols), arr, _ptr(k) if k is not None else None, C.byref(h)))
        return DeviceArray(self, h)

    def rows_to_columns(self, rows, itemsizes, kinds=None):
        n = len(itemsizes)
        sizes = (C.c_uint32 * n)(*[int(s) for s in itemsizes])
        outs = (C.c_void_p * n)()
        k = None if kinds is None else np.ascontiguousarray(kinds, dtype=np.uint8)
        self.check(self.lib.uqb_rows_to_columns(self.h, rows.h, n, sizes, _ptr(k) if k is not None else None, outs))
        return [DeviceArray(self, C.c_void_p(outs[i])) for i in range(n)]

    def columns_to_key(self, cols, plan):
        """integer columns -> table of packed 64-bit sort keys; plan = [(shift, bits, base)] per column"""
        arr = (C.c_void_p * len(cols))(*[c.h for c in cols])
        shifts, bits, bases = _plan_arrays(plan)
        h = C.c_void_p()
        self.check(self.lib.uqb_columns_to_key(self.h, len(cols), arr, shifts, bits, bases, C.byref(h)))
        return DeviceArray(self, h)

    def key_to_columns(self, keys, itemsizes, plan):
        """unique rows of a packed-key table (8 big-endian bytes) -> columns of the given itemsizes"""
        n = len(itemsizes)
        sizes = (C.c_uint32 * n)(*[int(s) for s in itemsizes])
        shifts, bits, bases = _plan_arrays(plan)
        outs = (C.c_void_p * n)()
        self.check(self.lib.uqb_key_to_columns(self.h, keys.h, n, sizes, shifts, bits, bases, outs))
        return [DeviceArray(self, C.c_void_p(outs[i])) for i in range(n)]

    def verify_records(self, src, text, first_row, order, report):
        """decoded records (text: split Fastq of container rows first_row..) against the encoded FASTQ src, under order
        (uint32 DeviceArray, container row -> input record; None = identity); accumulates into report (L.VerifyReport)"""
        self.check(self.lib.uqb_verify_records(self.h, src.h, text.h, int(first_row), order.h if order is not None else None,
                                               C.byref(report)))

    def check_permutation(self, order, n):
        """-> smallest value in [0, n) that order does not hold, -1 if it is a permutation of [0, n)"""
        m = C.c_int64()
        self.check(self.lib.uqb_check_permutation(self.h, order.h, int(n), C.byref(m)))
        return int(m.value)

    def layout(self, table, pattern):
        h = C.c_void_p()
        self.check(self.lib.uqb_layout(self.h, table.h, PATTERN_ID[pattern], C.byref(h)))
        return DeviceArray(self, h)

    def unlayout(self, stream, n, width, pattern):
        h = C.c_void_p()
        self.check(self.lib.uqb_unlayout(self.h, stream.h, int(n), int(width), PATTERN_ID[pattern], C.byref(h)))
        return DeviceArray(self, h)


class _PinnedArray(np.ndarray):
    """ndarray over pinned host memory that keeps its PinnedBuffer (and so the allocation) alive."""
    _pin = None


class PinnedBuffer:
    def __init__(self, ctx, ptr, array):
        self.ctx, self.ptr, self.array = ctx, ptr, array

    def owned_view(self, nbytes=None):
        """uint8 ndarray over the buffer; the pinned allocation is released when the last view dies."""
        a = (self.array if nbytes is None else self.array[:nbytes]).view(_PinnedArray)
        a._pin = self
        return a

    def __del__(self):
        try:
            if self.ptr and self.ctx.h:
                self.free()
        except Exception:
            pass

    def free(self):
        if self.ptr:
            self.array = None
            self.ctx.check(self.ctx.lib.uqb_host_free(self.ctx.h, self.ptr))
            self.ptr = None


class DeviceArray:
    """n rows x width bytes in HBM."""

    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle
        n, w = C.c_uint64(), C.c_uint32()
        ctx.lib.uqb_array_info(handle, C.byref(n), C.byref(w))
        self.n, self.width = int(n.value), int(w.value)

    @property
    def nbytes(self):
        return self.n * self.width

    @property
    def device_ptr(self):
        return C.c_void_p(self.ctx.lib.uqb_array_device_ptr(self.h))

    def download(self, dtype=np.uint8, out=None):
        """-> ndarray: 1-D of `dtype` when itemsize == width, else uint8 [n][width]."""
        dtype = np.dtype(dtype)
        if out is None:
            out = np.empty(self.nbytes, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.uqb_array_download(self.ctx.h, self.h, _ptr(out), self.nbytes))
        if dtype.itemsize == self.width and dtype != np.uint8:
            return out[:self.nbytes].view(dtype)
        if dtype == np.uint8 and self.width == 1:
            return out[:self.nbytes]
        return out[:self.nbytes].reshape(self.n, self.width)

    @property
    def __cuda_array_interface__(self):
        """zero-copy view for torch.as_tensor(...) (NCCL collectives of the multi-GPU path): flat uint8"""
        return {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.device_ptr.value or 0, False), "version": 3, "strides": None}

    def first_difference(self, other):
        """index of the first differing byte, -1 if the two device arrays are identical"""
        r = C.c_int64()
        self.ctx.check(self.ctx.lib.uqb_array_first_difference(self.ctx.h, self.h, other.h, C.byref(r)))
        return int(r.value)

    def download_async(self, out):
        """Queue the D2H copy into `out` (uint8 ndarray over pinned memory) on the copy stream; call ctx.copy_sync()."""
        self.ctx.check(self.ctx.lib.uqb_array_download_async(self.ctx.h, self.h, _ptr(out), self.nbytes))

    def free(self):
        if self.h:
            self.ctx.check(self.ctx.lib.uqb_array_free(self.ctx.h, self.h))
            self.h = C.c_void_p()

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.free()
        except Exception:
            pass


class Fastq:
    """Device-resident FASTQ bytes plus everything later stages cache on it (line offsets, QNAME scan)."""

    def __init__(self, ctx, handle, nbytes):
        self.ctx, self.h, self.nbytes = ctx, handle, nbytes
        self.n_reads = None
        self._keep = None
        self.reference = None

    def free(self):
        if self.h:
            self.ctx.check(self.ctx.lib.uqb_fastq_free(self.ctx.h, self.h))
            self.h = C.c_void_p()
            self._keep = None

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.free()
        except Exception:
            pass

    def download(self, offset=0, nbytes=None):
        nbytes = self.nbytes - offset if nbytes is None else nbytes
        out = np.empty(nbytes, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.uqb_fastq_download(self.ctx.h, self.h, int(offset), _ptr(out), int(nbytes)))
        return out

    def split(self):
        info = L.SplitInfo()
        self.ctx.check(self.ctx.lib.uqb_split(self.ctx.h, self.h, C.byref(info)))
        self.n_reads = int(info.n_reads)
        self.n_lines = int(info.n_lines)
        return info

    def line_offsets(self, first=0, count=None):
        count = self.n_lines + 1 - first if count is None else count
        out = np.empty(count, dtype=np.uint64)
        self.ctx.check(self.ctx.lib.uqb_fastq_line_offsets(self.ctx.h, self.h, int(first), int(count), _ptr(out)))
        return out

    def analyze(self):
        st = L.Stats()
        self.ctx.check(self.ctx.lib.uqb_analyze(self.ctx.h, self.h, C.byref(st)))
        return st

    def set_reference(self, name, rbase):
        """multi-GPU shard: measure QNAME statistics against the global first line; rbase = first global record"""
        b = np.frombuffer(name, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.uqb_fastq_set_reference(self.ctx.h, self.h, _ptr(b) if b.size else None, int(b.size), int(rbase)))
        self.reference = name

    def qname_scan(self, prefix_len, suffix_len, separators, col_mode=None):
        seps = np.frombuffer(separators.encode('latin-1'), dtype=np.uint8)
        ncols = len(seps) + 1
        cols = (L.ColStats * ncols)()
        bad = C.c_int64()
        mode = None if col_mode is None else np.ascontiguousarray(col_mode, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.uqb_qname_scan(self.ctx.h, self.h, int(prefix_len), int(suffix_len),
                                                   _ptr(seps) if len(seps) else None, len(seps),
                                                   _ptr(mode) if mode is not None else None, cols, C.byref(bad)))
        return cols, int(bad.value)

    def qname_dict_first(self, col):
        cnt, w = C.c_uint64(), C.c_uint32()
        self.ctx.check(self.ctx.lib.uqb_qname_dict_info(self.ctx.h, self.h, int(col), C.byref(cnt), C.byref(w)))
        out = np.zeros(max(cnt.value, 1), dtype=np.uint32)
        self.ctx.check(self.ctx.lib.uqb_qname_dict_first(self.ctx.h, self.h, int(col), _ptr(out), cnt.value))
        return out[:cnt.value]

    def qname_dict(self, col):
        cnt, w = C.c_uint64(), C.c_uint32()
        self.ctx.check(self.ctx.lib.uqb_qname_dict_info(self.ctx.h, self.h, int(col), C.byref(cnt), C.byref(w)))
        buf = np.zeros(max(cnt.value * w.value, 1), dtype=np.uint8)
        self.ctx.check(self.ctx.lib.uqb_qname_dict(self.ctx.h, self.h, int(col), _ptr(buf), cnt.value * w.value))
        rows = buf[:cnt.value * w.value].reshape(cnt.value, w.value) if w.value else np.zeros((cnt.value, 0), np.uint8)
        return [bytes(r).rstrip(b"\0").decode('latin-1') for r in rows]

    def qname_encode(self, specs):
        n = len(specs)
        arr = (L.ColSpec * n)()
        for i, (fmt, itemsize, offset, mn) in enumerate(specs):
            arr[i].format, arr[i].itemsize, arr[i].offset, arr[i].min_val = fmt, itemsize, 1 if offset else 0, int(mn)
        outs = (C.c_void_p * n)()
        self.ctx.check(self.ctx.lib.uqb_qname_encode(self.ctx.h, self.h, n, arr, outs))
        return [DeviceArray(self.ctx, C.c_void_p(outs[i])) for i in range(n)]

    def pack(self, params):
        d, q = C.c_void_p(), C.c_void_p()
        self.ctx.check(self.ctx.lib.uqb_pack(self.ctx.h, self.h, C.byref(params), C.byref(d), C.byref(q)))
        return DeviceArray(self.ctx, d), DeviceArray(self.ctx, q)
