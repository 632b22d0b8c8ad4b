"""ctypes / numpy mirror of include/fplgpu.h (the C ABI).  Layout-only; no logic."""
import ctypes as C
import numpy as np

ABI_VERSION = 6
COMM_ID_BYTES = 128        # FPL_COMM_ID_BYTES == sizeof(ncclUniqueId)
MAX_ADAPTER_LEN = 1024
MAX_ADAPTERS = 1024
INLINE_EVENTS = 4

PASS_FILTER, FAIL_POLY_X, FAIL_OVERLAP, FAIL_N_BASE = 0, 4, 8, 12
FAIL_LENGTH, FAIL_TOO_LONG, FAIL_QUALITY, FAIL_COMPLEXITY = 16, 17, 20, 24
# src/common.h:55-64
FAILED_TYPES = {0: "passed", 4: "failed_polyx_filter", 8: "failed_bad_overlap", 12: "failed_too_many_n_bases",
                16: "failed_too_short", 17: "failed_too_long", 20: "failed_quality_filter",
                24: "failed_low_complexity"}

FLAG_DROPPED_BY_CUT, FLAG_POLYX, FLAG_MIDDLE_ADAPTER, FLAG_SEG0_IS_RIGHT = 1, 2, 4, 8

STATS_PRE, STATS_POST = 0, 1
STATS_KMER, STATS_QUALHIST, STATS_MEDHIST, STATS_MEDBASES = 0, 1024, 1152, 1280
STATS_READS, STATS_LENSUM, STATS_TAIL = 1408, 1409, 1536
CNT_FILTER, CNT_ADAPTER_READS, CNT_ADAPTER_BASES = 0, 32, 33
CNT_POLYX_READS, CNT_POLYX_BASES, CNT_DROPPED, CNT_SPLIT, CNT_FIXED = 34, 38, 42, 43, 64


def stats_words(cycles):
    return 16 * int(cycles) + STATS_TAIL


def counter_words(n_adapters):
    return CNT_FIXED + int(n_adapters) * 2 * (MAX_ADAPTER_LEN + 1)

GZIP_SEGMENT = 65536       # FPL_GZIP_SEGMENT


def gzip_bound(n_bytes, n_pieces):
    """FPL_GZIP_BOUND: the most bytes fpl_gzip_host writes for n_bytes in n_pieces pieces."""
    return int(n_bytes) + 28 * (int(n_bytes) // GZIP_SEGMENT + int(n_pieces))


def event_unpack(e):
    e = int(e)
    return e & 0xFFFF, (e >> 16) & 1, e >> 17


class FplOptions(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "struct_size", "device", "trim_front", "trim_tail",
        "cut_front_enabled", "cut_front_window", "cut_front_quality",
        "cut_tail_enabled", "cut_tail_window", "cut_tail_quality",
        "polyx_enabled", "polyx_min_len", "adapter_enabled", "trimming_extension")] + [
        ("ed_max", C.c_double)] + [(n, C.c_int32) for n in (
            "qual_filter_enabled", "qualified_qual", "unqualified_percent_limit", "avg_qual_req",
            "n_base_percent_limit", "n_base_limit", "length_filter_enabled", "length_required", "length_max",
            "complexity_enabled", "complexity_threshold_pct", "mask_enabled", "mask_window", "mask_quality",
            "break_enabled", "break_window", "break_quality")] + [("reserved", C.c_int32 * 3)]


class FplAdapters(C.Structure):
    _fields_ = [("start", C.c_char_p), ("end", C.c_char_p), ("n_fasta", C.c_int32),
                ("fasta", C.POINTER(C.c_char_p))]


class FplBatch(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("qual", C.c_void_p), ("offsets", C.c_void_p), ("lens", C.c_void_p),
                ("n_reads", C.c_int64), ("n_bytes", C.c_int64)]


RESULT_DTYPE = np.dtype([
    ("flags", "<u4"), ("n_segments", "<i4"), ("trim_lo", "<i4"), ("trim_len", "<i4"),
    ("seg_lo", "<i4", (2,)), ("seg_len", "<i4", (2,)),
    ("seg_result", "u1", (2,)), ("seg_median_qual", "u1", (2,)),
    ("pre_median_qual", "u1"), ("polyx_base", "u1"), ("n_events", "<u2"),
    ("polyx_len", "<i4"), ("adapter_trimmed_bases", "<i4"), ("events", "<u4", (INLINE_EVENTS,))], align=False)
assert RESULT_DTYPE.itemsize == 64
FASTQ_RECORD_DTYPE = np.dtype([("name_off", "<i8"), ("seq_off", "<i8"), ("plus_off", "<i8"), ("qual_off", "<i8"),
                               ("name_len", "<i4"), ("seq_len", "<i4"), ("plus_len", "<i4"), ("reserved", "<i4")])
assert FASTQ_RECORD_DTYPE.itemsize == 48
SEGMENT_DTYPE = np.dtype([("read", "<i4"), ("lo", "<i4"), ("len", "<i4"), ("result", "u1"), ("median_qual", "u1"),
                          ("split_side", "u1"), ("is_r1", "u1"), ("break_index", "<i4")])
assert SEGMENT_DTYPE.itemsize == 20
REGION_DTYPE = np.dtype([("read", "<i4"), ("lo", "<i4"), ("len", "<i4")])
assert C.sizeof(FplOptions) == 144, C.sizeof(FplOptions)


def make_adapters(start, end, fasta=()):
    """Build an FplAdapters plus the keep-alive objects it points into."""
    fasta = [s.encode() if isinstance(s, str) else s for s in fasta]
    arr = (C.c_char_p * max(1, len(fasta)))(*fasta) if fasta else (C.c_char_p * 1)()
    ad = FplAdapters((start or "").encode() if isinstance(start, str) or start is None else start,
                     (end or "").encode() if isinstance(end, str) or end is None else end,
                     len(fasta), C.cast(arr, C.POINTER(C.c_char_p)))
    return ad, (arr, fasta)
