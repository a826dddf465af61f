"""ctypes binding of libuqb200.so (include/uqb200.h).  Loading fails loudly: there is no CPU path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libuqb200.so")

HDR_MAX = 1024
MAX_COLS = 64
MAX_CHECKPOINTS = 40
TIMER_NAME = 48
NONE_I64 = 2 ** 63 - 1
U64_MAX = 2 ** 64 - 1


class SplitInfo(C.Structure):
    _fields_ = [("n_bytes", C.c_uint64), ("n_lines", C.c_uint64), ("n_reads", C.c_uint64),
                ("status", C.c_int32), ("_pad", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("base_count", C.c_uint64 * 256), ("qual_count", C.c_uint64 * 256),
                ("base_single_qual", C.c_int32 * 256),
                ("dna_min", C.c_uint64), ("dna_max", C.c_uint64),
                ("bad_first_char", C.c_int64), ("bad_plus_record", C.c_int64), ("bad_len_record", C.c_int64),
                ("first_len", C.c_uint32), ("last_len", C.c_uint32),
                ("first_name", C.c_uint8 * HDR_MAX), ("last_name", C.c_uint8 * HDR_MAX),
                ("max_name_len", C.c_uint32), ("prefix_len", C.c_uint32), ("suffix_len", C.c_uint32),
                ("last_count_mismatch", C.c_int64 * 256),
                ("first_lcp_eq", C.c_int64 * (HDR_MAX + 1)), ("first_lcs_eq", C.c_int64 * (HDR_MAX + 1)),
                ("first_short_prefix", C.c_int64 * (HDR_MAX + 1)), ("first_short_suffix", C.c_int64 * (HDR_MAX + 1))]


class ColStats(C.Structure):
    _fields_ = [("all_int", C.c_uint8), ("all_canonical", C.c_uint8), ("overflow", C.c_uint8), ("_pad", C.c_uint8 * 5),
                ("min_val", C.c_int64), ("max_val", C.c_int64), ("min_len", C.c_uint32), ("max_len", C.c_uint32),
                ("n_distinct", C.c_uint64), ("n_checkpoints", C.c_uint32), ("_pad2", C.c_uint32),
                ("distinct_at", C.c_uint64 * MAX_CHECKPOINTS)]


class ColSpec(C.Structure):
    _fields_ = [("format", C.c_uint8), ("itemsize", C.c_uint8), ("offset", C.c_uint8), ("_pad", C.c_uint8 * 5),
                ("min_val", C.c_int64)]


class PackParams(C.Structure):
    _fields_ = [("base_code", C.c_uint8 * 256), ("qual_code", C.c_uint8 * 256), ("trick_qual", C.c_int16 * 256),
                ("bits_per_base", C.c_uint32), ("bits_per_quality", C.c_uint32),
                ("dna_bytes", C.c_uint32), ("qual_bytes", C.c_uint32), ("variable", C.c_uint32), ("dna_max", C.c_uint32)]


class DecodeCol(C.Structure):
    _fields_ = [("format", C.c_uint8), ("itemsize", C.c_uint8), ("offset", C.c_uint8), ("_pad", C.c_uint8 * 5),
                ("min_val", C.c_int64), ("dict", C.c_void_p), ("dict_count", C.c_uint64),
                ("dict_width", C.c_uint32), ("_pad2", C.c_uint32)]


class DecodeParams(C.Structure):
    _fields_ = [("base_char", C.c_uint8 * 256), ("qual_char", C.c_uint8 * 256), ("qual_to_base", C.c_int16 * 256),
                ("bits_per_base", C.c_uint32), ("bits_per_quality", C.c_uint32), ("variable", C.c_uint32), ("dna_max", C.c_uint32),
                ("prefix", C.c_void_p), ("prefix_len", C.c_uint32), ("_p0", C.c_uint32),
                ("suffix", C.c_void_p), ("suffix_len", C.c_uint32), ("_p1", C.c_uint32),
                ("seps", C.c_void_p), ("nseps", C.c_uint32), ("ncols", C.c_uint32),
                ("cols", C.POINTER(DecodeCol))]


class SynthParams(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("length", C.c_uint32), ("len_lo", C.c_uint32), ("len_hi", C.c_uint32),
                ("seed", C.c_uint64), ("first", C.c_uint64), ("n", C.c_uint64), ("genome", C.c_uint64), ("pool", C.c_uint64)]


# name -> (restype, argtypes); every symbol include/uqb200.h declares
P = C.c_void_p
PP = C.POINTER(C.c_void_p)
SIGNATURES = {
    "uqb_version": (C.c_int, []),
    "uqb_ctx_create": (C.c_int, [C.c_int, P, PP]),
    "uqb_ctx_destroy": (None, [P]),
    "uqb_last_error": (C.c_char_p, [P]),
    "uqb_ctx_sync": (C.c_int, [P]),
    "uqb_ctx_launch_count": (C.c_uint64, [P]),
    "uqb_ctx_timing": (C.c_int, [P, C.c_int]),
    "uqb_ctx_timing_report": (C.c_int, [P, C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int, C.POINTER(C.c_int)]),
    "uqb_ctx_span_begin": (C.c_int, [P]),
    "uqb_ctx_span_end": (C.c_int, [P, C.POINTER(C.c_double)]),
    "uqb_ctx_timing_reset": (C.c_int, [P]),
    "uqb_host_alloc": (C.c_int, [P, C.c_uint64, PP]),
    "uqb_host_free": (C.c_int, [P, P]),
    "uqb_mem_info": (C.c_int, [P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "uqb_array_info": (C.c_int, [P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "uqb_array_alloc": (C.c_int, [P, C.c_uint64, C.c_uint32, PP]),
    "uqb_array_upload": (C.c_int, [P, P, C.c_uint64, C.c_uint32, PP]),
    "uqb_array_download": (C.c_int, [P, P, P, C.c_uint64]),
    "uqb_array_first_difference": (C.c_int, [P, P, P, C.POINTER(C.c_int64)]),
    "uqb_array_free": (C.c_int, [P, P]),
    "uqb_array_device_ptr": (C.c_void_p, [P]),
    "uqb_array_wrap": (C.c_int, [P, P, C.c_uint64, C.c_uint32, PP]),
    "uqb_array_copy_in": (C.c_int, [P, P, C.c_uint64, P, C.c_uint64]),
    "uqb_index_u32": (C.c_int, [P, P, C.c_uint64, PP, C.POINTER(C.c_int64)]),
    "uqb_fastq_load": (C.c_int, [P, P, C.c_uint64, PP]),
    "uqb_fastq_adopt": (C.c_int, [P, P, C.c_uint64, PP]),
    "uqb_fastq_load_streamed": (C.c_int, [P, P, C.c_uint64, C.c_uint64, PP]),
    "uqb_fastq_load_streamed_ref": (C.c_int, [P, P, C.c_uint64, C.c_uint64, P, C.c_uint32, C.c_uint64, PP]),
    "uqb_array_download_async": (C.c_int, [P, P, P, C.c_uint64]),
    "uqb_ctx_copy_sync": (C.c_int, [P]),
    "uqb_fastq_free": (C.c_int, [P, P]),
    "uqb_fastq_download": (C.c_int, [P, P, C.c_uint64, P, C.c_uint64]),
    "uqb_split": (C.c_int, [P, P, C.POINTER(SplitInfo)]),
    "uqb_fastq_line_offsets": (C.c_int, [P, P, C.c_uint64, C.c_uint64, P]),
    "uqb_analyze": (C.c_int, [P, P, C.POINTER(Stats)]),
    "uqb_fastq_set_reference": (C.c_int, [P, P, P, C.c_uint32, C.c_uint64]),
    "uqb_qname_scan_ex": (C.c_int, [P, P, C.c_uint32, C.c_uint32, P, C.c_uint32, P, C.POINTER(ColStats), C.POINTER(C.c_int64)]),
    "uqb_qname_dict_first": (C.c_int, [P, P, C.c_uint32, P, C.c_uint64]),
    "uqb_rows_lower_bound": (C.c_int, [P, P, P, C.c_uint32, P]),
    "uqb_add_scalar_u32": (C.c_int, [P, P, C.c_uint32]),
    "uqb_scatter_u32": (C.c_int, [P, P, P, PP]),
    "uqb_gather_rows_segmented": (C.c_int, [P, P, P, C.c_uint32, P, C.c_uint32, PP, P]),
    "uqb_compact_segments": (C.c_int, [P, P, C.c_uint32, P, P, C.c_uint32, PP]),
    "uqb_partition_positions": (C.c_int, [P, P, P, C.c_uint32, PP, P]),
    "uqb_scatter_rows_segmented": (C.c_int, [P, P, P, C.c_uint32, P, C.c_uint32, PP, P]),
    "uqb_scatter_rows_to": (C.c_int, [P, P, P, C.c_uint32, P, P]),
    "uqb_qname_scan": (C.c_int, [P, P, C.c_uint32, C.c_uint32, P, C.c_uint32, C.POINTER(ColStats), C.POINTER(C.c_int64)]),
    "uqb_qname_dict_info": (C.c_int, [P, P, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "uqb_qname_dict": (C.c_int, [P, P, C.c_uint32, P, C.c_uint64]),
    "uqb_qname_encode": (C.c_int, [P, P, C.c_uint32, C.POINTER(ColSpec), PP]),
    "uqb_pack": (C.c_int, [P, P, C.POINTER(PackParams), PP, PP]),
    "uqb_sort_rows": (C.c_int, [P, P, PP, PP, PP, PP, C.POINTER(C.c_uint64)]),
    "uqb_gather_rows": (C.c_int, [P, P, P, PP]),
    "uqb_narrow_u32": (C.c_int, [P, P, C.c_uint32, PP]),
    "uqb_columns_to_rows": (C.c_int, [P, C.c_uint32, PP, PP]),
    "uqb_rows_to_columns": (C.c_int, [P, P, C.c_uint32, C.POINTER(C.c_uint32), PP]),
    "uqb_columns_to_rows_ex": (C.c_int, [P, C.c_uint32, PP, P, PP]),
    "uqb_rows_to_columns_ex": (C.c_int, [P, P, C.c_uint32, C.POINTER(C.c_uint32), P, PP]),
    "uqb_layout": (C.c_int, [P, P, C.c_int, PP]),
    "uqb_unlayout": (C.c_int, [P, P, C.c_uint64, C.c_uint32, C.c_int, PP]),
    "uqb_decode": (C.c_int, [P, P, P, PP, C.POINTER(DecodeParams), PP]),
    "uqb_synth": (C.c_int, [P, C.POINTER(SynthParams), P, PP]),
}

_lib = None


def load():
    """Load libuqb200.so and declare every entry point.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError("uq_b200: %s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(make -C uq_b200/csrc).  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.uqb_version() != 100:
        raise RuntimeError("uq_b200: libuqb200.so version %d does not match the binding" % lib.uqb_version())
    _lib = lib
    return lib
