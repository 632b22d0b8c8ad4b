"""ctypes binding of libfplgpu.so (include/fplgpu.h) — the product path used by tests, bench.py and the multi-GPU
driver.  There is no fallback: if the CUDA library is missing or no device is usable, construction raises."""
import ctypes as C
import os

import numpy as np

from . import abi
from .abi import FplAdapters, FplBatch, FplOptions, RESULT_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfplgpu.so")

_lib = None


class FplError(RuntimeError):
    pass


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FplError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback for the hot path)")
    lib = C.CDLL(LIB_PATH)
    lib.fpl_last_error.restype = C.c_char_p
    lib.fpl_abi_version.restype = C.c_int
    lib.fpl_create.argtypes = [C.POINTER(FplOptions), C.POINTER(FplAdapters), C.POINTER(C.c_void_p)]
    lib.fpl_destroy.argtypes = [C.c_void_p]
    lib.fpl_destroy.restype = None
    lib.fpl_process_host.argtypes = [C.c_void_p, C.POINTER(FplBatch), C.c_void_p]
    lib.fpl_process_device.argtypes = [C.c_void_p, C.POINTER(FplBatch), C.c_void_p]
    lib.fpl_sync.argtypes = [C.c_void_p]
    lib.fpl_process_fastq_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.fpl_emit_fastq_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.c_void_p, C.c_int64,
                                        C.POINTER(C.c_int64)]
    lib.fpl_gzip_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.fpl_emit_fastq_gzip_host.argtypes = lib.fpl_emit_fastq_host.argtypes
    lib.fpl_stream.argtypes = [C.c_void_p]
    lib.fpl_stream.restype = C.c_void_p
    lib.fpl_fetch_results.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.fpl_last_segments.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.fpl_last_mask_regions.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.fpl_stats_cycles.argtypes = [C.c_void_p]
    lib.fpl_stats_cycles.restype = C.c_int64
    lib.fpl_stats_reserve.argtypes = [C.c_void_p, C.c_int64]
    lib.fpl_stats_download.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]
    lib.fpl_stats_device_ptr.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    lib.fpl_counter_words.argtypes = [C.c_void_p]
    lib.fpl_counter_words.restype = C.c_int64
    lib.fpl_counters_download.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.fpl_counters_device_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    lib.fpl_comm_unique_id.argtypes = [C.c_void_p]
    lib.fpl_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.fpl_comm_destroy.argtypes = [C.c_void_p]
    lib.fpl_comm_size.argtypes = [C.c_void_p]
    lib.fpl_comm_agree_cycles.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    lib.fpl_allreduce_stats.argtypes = [C.c_void_p, C.c_int64]
    lib.fpl_eval_adapter_kmers.argtypes = [C.c_int, C.POINTER(FplBatch), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                           C.POINTER(C.c_int64)]
    lib.fpl_eval_pick_adapter.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_char_p, C.c_int32]
    lib.fpl_reset.argtypes = [C.c_void_p]
    lib.fpl_last_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_float),
                                          C.POINTER(C.c_int64), C.c_int]
    lib.fpl_launch_count.argtypes = [C.c_void_p]
    lib.fpl_launch_count.restype = C.c_int64
    lib.fpl_set_timing.argtypes = [C.c_void_p, C.c_int]
    if lib.fpl_abi_version() != abi.ABI_VERSION:
        raise FplError("libfplgpu.so ABI version mismatch")
    _lib = lib
    return lib


EXPORTS = ["fpl_last_error", "fpl_abi_version", "fpl_create", "fpl_destroy", "fpl_process_host", "fpl_process_device", "fpl_process_fastq_host", "fpl_emit_fastq_host",
           "fpl_gzip_host", "fpl_emit_fastq_gzip_host", "fpl_sync", "fpl_stream", "fpl_last_segments", "fpl_last_mask_regions", "fpl_fetch_results", "fpl_stats_cycles", "fpl_stats_reserve", "fpl_stats_download",
           "fpl_stats_device_ptr", "fpl_counter_words", "fpl_counters_download", "fpl_counters_device_ptr",
           "fpl_comm_unique_id", "fpl_comm_init", "fpl_comm_destroy", "fpl_comm_size", "fpl_comm_agree_cycles", "fpl_allreduce_stats",
           "fpl_eval_adapter_kmers", "fpl_eval_pick_adapter", "fpl_reset", "fpl_last_kernel_times", "fpl_launch_count", "fpl_set_timing"]


class _DeviceArray:
    """Wraps a raw device pointer for torch.as_tensor via __cuda_array_interface__ (int64 vector)."""

    def __init__(self, ptr, n_words, owner):
        self.__cuda_array_interface__ = {"shape": (int(n_words),), "typestr": "<i8", "data": (int(ptr), False),
                                         "version": 2}
        self._owner = owner


class Engine:
    """One context = one worker's state (2 Stats + FilterResult accumulators) on one GPU."""

    def __init__(self, options):
        self.lib = load_library()
        self.options = options
        o, ad, keep = options.to_abi()
        self._keep = (o, ad, keep)
        self.n_adapters = 2 + len(options.adapter_fasta)
        h = C.c_void_p()
        if self.lib.fpl_create(C.byref(o), C.byref(ad), C.byref(h)) != 0:
            raise FplError(self.lib.fpl_last_error().decode())
        self.h = h

    def _check(self, rc):
        if rc != 0:
            raise FplError(self.lib.fpl_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.fpl_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- processSingleEnd over a packed batch ---
    def process(self, batch, out=None):
        """Host batch (numpy / pinned buffers) -> per-read records (numpy structured array)."""
        res = out if out is not None else np.zeros(batch.n_reads, dtype=RESULT_DTYPE)
        if res.shape[0] < batch.n_reads or res.dtype != RESULT_DTYPE:
            raise FplError(f"process: `out` holds {res.shape[0]} records, the batch has {batch.n_reads} reads")
        b = batch.to_abi()
        self._check(self.lib.fpl_process_host(self.h, C.byref(b), res.ctypes.data))
        return res

    def process_fastq(self, text, is_last=True, max_records=None):
        """A chunk of plain FASTQ text (bytes / uint8 array) -> (record table, per-read results, bytes consumed), or None
        if the chunk is not in the strict layout (the caller then uses the reference reader)."""
        from .abi import FASTQ_RECORD_DTYPE
        buf = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else text
        cap = int(max_records if max_records is not None else max(16, buf.size // 8))
        recs = np.zeros(cap, dtype=FASTQ_RECORD_DTYPE)
        res = np.zeros(cap, dtype=RESULT_DTYPE)
        n, used = C.c_int64(), C.c_int64()
        rc = self.lib.fpl_process_fastq_host(self.h, buf.ctypes.data if buf.size else None, buf.size, int(is_last),
                                             recs.ctypes.data, res.ctypes.data, cap, C.byref(n), C.byref(used))
        if rc == 1:
            return None
        self._check(rc)
        return recs[:n.value], res[:n.value], used.value

    def emit_fastq(self, want_failed=True):
        """The --out / --failed_out text of the chunk the last process_fastq() call processed, assembled on the device
        (fpl_emit_fastq_host): (out_bytes, failed_bytes).  First call sizes, second call copies."""
        return self._emit(self.lib.fpl_emit_fastq_host, want_failed)

    def _emit(self, fn, want_failed):
        n_out, n_failed = C.c_int64(), C.c_int64()
        rc = fn(self.h, int(want_failed), None, 0, C.byref(n_out), None, 0, C.byref(n_failed))
        if rc < 0:
            self._check(rc)
        out = np.empty(n_out.value, dtype=np.uint8)
        failed = np.empty(n_failed.value, dtype=np.uint8)
        self._check(fn(self.h, int(want_failed), out.ctypes.data if out.size else None, out.size, C.byref(n_out),
                       failed.ctypes.data if failed.size else None, failed.size, C.byref(n_failed)))
        return out.tobytes(), failed.tobytes()

    def emit_fastq_gzip(self, want_failed=True):
        """emit_fastq() with both texts compressed on the device (fpl_emit_fastq_gzip_host): (out_gz, failed_gz), each a
        multi-member gzip stream."""
        return self._emit(self.lib.fpl_emit_fastq_gzip_host, want_failed)

    def gzip(self, pieces):
        """Each piece (bytes-like) compressed on the device into gzip members (fpl_gzip_host) -> list of bytes."""
        bufs = [bytes(p) for p in pieces]
        text = np.frombuffer(b"".join(bufs), dtype=np.uint8)
        sizes = np.array([len(b) for b in bufs], dtype=np.int64)
        cap = abi.gzip_bound(text.size, len(bufs))
        out = np.empty(max(cap, 1), dtype=np.uint8)
        out_sizes = np.zeros(max(len(bufs), 1), dtype=np.int64)
        self._check(self.lib.fpl_gzip_host(self.h, text.ctypes.data if text.size else None, sizes.ctypes.data, len(bufs),
                                           out.ctypes.data, cap, out_sizes.ctypes.data))
        ends = np.cumsum(out_sizes[:len(bufs)])
        return [out[e - k:e].tobytes() for e, k in zip(ends, out_sizes[:len(bufs)])]

    def process_device(self, seq_ptr, qual_ptr, offsets_ptr, lens_ptr, n_reads, n_bytes, results_ptr=None):
        b = FplBatch(seq_ptr, qual_ptr, offsets_ptr, lens_ptr, n_reads, n_bytes)
        self._check(self.lib.fpl_process_device(self.h, C.byref(b), results_ptr))

    def sync(self):
        self._check(self.lib.fpl_sync(self.h))

    @property
    def stream_ptr(self):
        """cudaStream_t of the context (wrap with torch.cuda.ExternalStream to record events / order collectives)."""
        return int(self.lib.fpl_stream(self.h) or 0)

    def _list(self, fn, dtype):
        n = C.c_int64()
        # ask for the count first (a call with cap 0 fails only when there are entries)
        fn(self.h, None, 0, C.byref(n))
        out = np.zeros(n.value, dtype=dtype)
        if n.value:
            self._check(fn(self.h, out.ctypes.data, n.value, C.byref(n)))
        return out

    def segments(self):
        """--mask/--break: every output read of the last process() call (abi.SEGMENT_DTYPE)."""
        return self._list(self.lib.fpl_last_segments, abi.SEGMENT_DTYPE)

    def mask_regions(self):
        return self._list(self.lib.fpl_last_mask_regions, abi.REGION_DTYPE)

    def fetch_results(self, n):
        res = np.zeros(n, dtype=RESULT_DTYPE)
        self._check(self.lib.fpl_fetch_results(self.h, res.ctypes.data, n))
        return res

    # --- accumulators ---
    @property
    def cycles(self):
        return int(self.lib.fpl_stats_cycles(self.h))

    def reserve_cycles(self, cycles):
        self._check(self.lib.fpl_stats_reserve(self.h, int(cycles)))

    def stats(self, which, cycles=None):
        """The FPL_STATS_WORDS block, re-laid out to `cycles` columns if given (must cover every non-zero cycle)."""
        cap = self.cycles
        raw = np.zeros(abi.stats_words(cap), dtype=np.int64)
        self._check(self.lib.fpl_stats_download(self.h, which, raw.ctypes.data, raw.shape[0]))
        if cycles is None or cycles == cap:
            return raw
        return relayout_stats(raw, cap, int(cycles))

    def counters(self):
        n = int(self.lib.fpl_counter_words(self.h))
        out = np.zeros(n, dtype=np.int64)
        self._check(self.lib.fpl_counters_download(self.h, out.ctypes.data, n))
        return out

    def stats_device(self, which):
        p, n = C.c_void_p(), C.c_int64()
        self._check(self.lib.fpl_stats_device_ptr(self.h, which, C.byref(p), C.byref(n)))
        return _DeviceArray(p.value, n.value, self)

    def counters_device(self):
        p, n = C.c_void_p(), C.c_int64()
        self._check(self.lib.fpl_counters_device_ptr(self.h, C.byref(p), C.byref(n)))
        return _DeviceArray(p.value, n.value, self)

    def reset(self):
        self._check(self.lib.fpl_reset(self.h))

    # --- multi-GPU merge (one process per GPU): Stats::merge / FilterResult::merge as NCCL all-reduces ---
    @staticmethod
    def comm_unique_id():
        """Rank 0: the FPL_COMM_ID_BYTES rendezvous id to hand to every rank."""
        lib = load_library()
        buf = (C.c_uint8 * abi.COMM_ID_BYTES)()
        if lib.fpl_comm_unique_id(buf) != 0:
            raise FplError(lib.fpl_last_error().decode())
        return bytes(buf)

    def comm_init(self, unique_id, rank, n_ranks):
        buf = (C.c_uint8 * abi.COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self.lib.fpl_comm_init(self.h, buf, int(rank), int(n_ranks)))

    def agree_cycles(self):
        n = C.c_int64()
        self._check(self.lib.fpl_comm_agree_cycles(self.h, C.byref(n)))
        return int(n.value)

    def allreduce_stats(self, cycles=0):
        """In-place sum over the ranks of both Stats blocks and the counters, on the context's stream (asynchronous).
        cycles = 0: agree on the number of cycles first (synchronous)."""
        self._check(self.lib.fpl_allreduce_stats(self.h, int(cycles)))

    # --- measurement ---
    def set_timing(self, on=True):
        self._check(self.lib.fpl_set_timing(self.h, int(on)))

    def kernel_times(self):
        """{kernel name: (total device ms, timed launches)} since set_timing(True)."""
        names = (C.c_char_p * 16)()
        ms = (C.c_float * 16)()
        cnt = (C.c_int64 * 16)()
        k = self.lib.fpl_last_kernel_times(self.h, names, ms, cnt, 16)
        return {names[i].decode(): (float(ms[i]), int(cnt[i])) for i in range(k)}

    @property
    def launch_count(self):
        return int(self.lib.fpl_launch_count(self.h))


def eval_adapter_kmers(batch, side, shift_tail=1, device=0):
    """Device half of Evaluator::evalAdapterAndReadNum: (counts uint32[1<<20], position_acc uint64[1<<20], total)."""
    lib = load_library()
    counts = np.zeros(1 << 20, dtype=np.uint32)
    acc = np.zeros(1 << 20, dtype=np.uint64)
    total = C.c_int64()
    b = batch.to_abi()
    rc = lib.fpl_eval_adapter_kmers(int(device), C.byref(b), int(shift_tail), int(side), counts.ctypes.data, acc.ctypes.data,
                                    C.byref(total))
    if rc != 0:
        raise FplError(f"fpl_eval_adapter_kmers failed ({rc})")
    return counts, acc, int(total.value)


def eval_pick_adapter(counts, position_acc, total, is_rna=False):
    """Table half of Evaluator::evalAdapterAndReadNum for one side (host only, fpl_eval_pick_adapter): the adapter string,
    or None when nothing is detected."""
    lib = load_library()
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    acc = np.ascontiguousarray(position_acc, dtype=np.uint64)
    if counts.shape != (1 << 20,) or acc.shape != (1 << 20,):
        raise FplError("eval_pick_adapter: the tables have 1 << 20 entries")
    buf = C.create_string_buffer(80)
    n = lib.fpl_eval_pick_adapter(counts.ctypes.data, acc.ctypes.data, int(total), int(bool(is_rna)), buf, 80)
    if n < 0:
        raise FplError(f"fpl_eval_pick_adapter failed ({n})")
    return buf.value.decode() if n > 0 else None


def relayout_stats(raw, cap, cycles):
    """[16][cap] + tail  ->  [16][cycles] + tail; raises if a dropped column is non-zero."""
    rows = raw[:16 * cap].reshape(16, cap)
    out = np.zeros(abi.stats_words(cycles), dtype=np.int64)
    n = min(cap, cycles)
    out[:16 * cycles].reshape(16, cycles)[:, :n] = rows[:, :n]
    if cap > cycles and rows[:, cycles:].any():
        raise ValueError("stats block has non-zero cycles beyond the requested width")
    out[16 * cycles:] = raw[16 * cap:]
    return out
