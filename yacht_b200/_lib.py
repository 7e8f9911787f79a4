"""ctypes binding of libyachtgpu.so (the C ABI declared in include/yacht_gpu.h).

This is the only place the Python host layer touches device code.  There is no CPU fallback:
if the shared library is missing, or no B200 is visible, the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libyachtgpu.so")

# every symbol include/yacht_gpu.h declares (tests check the library exports each of them)
ABI_SYMBOLS = [
    "ygpu_device_count", "ygpu_ctx_create", "ygpu_ctx_destroy", "ygpu_last_error", "ygpu_free",
    "ygpu_host_alloc", "ygpu_host_free", "ygpu_read_signatures", "ygpu_read_signatures_ksize", "ygpu_sketch_set_free", "ygpu_alt_mut_rate", "ygpu_reset_timers", "ygpu_get_timings", "ygpu_load_sketches", "ygpu_load_sketch_blocks", "ygpu_load_sketches_device",
    "ygpu_build_index", "ygpu_pairwise_flag", "ygpu_pairwise_flag_device", "ygpu_pairs_copy", "ygpu_row_partition",
    "ygpu_mark", "ygpu_elapsed_ms", "ygpu_set_option", "ygpu_get_option", "ygpu_exclusive_hashes",
    "ygpu_hyp_test",
    "ygpu_upload_begin", "ygpu_upload_block", "ygpu_upload_finish", "ygpu_greedy_select",
    "ygpu_comm_get_unique_id", "ygpu_comm_init", "ygpu_comm_destroy", "ygpu_load_sketches_sharded", "ygpu_load_sketches_sharded_device",
    "ygpu_train_step_sharded", "ygpu_upload_finish_sharded", "ygpu_load_sketches_hashrange", "ygpu_load_sketches_hashrange_device",
    "ygpu_train_step_replicated", "ygpu_sketch_sequences", "ygpu_sketch_result_free",
    "ygpu_stream_begin", "ygpu_stream_feed", "ygpu_stream_end_file", "ygpu_stream_finish",
]
STREAM_WHOLE, STREAM_PER_RECORD = 0, 1
COMM_ID_BYTES = 128


class YgpuError(RuntimeError):
    pass


class IndexStats(ctypes.Structure):
    _fields_ = [("n_hashes", ctypes.c_uint64), ("n_distinct", ctypes.c_uint64), ("n_singleton", ctypes.c_uint64),
                ("n_index", ctypes.c_uint64), ("n_postings", ctypes.c_uint64), ("n_increments", ctypes.c_uint64),
                ("n_row_items", ctypes.c_uint64), ("max_sketch", ctypes.c_uint32), ("has_duplicates", ctypes.c_uint32),
                ("index_path", ctypes.c_uint32), ("big_buckets", ctypes.c_uint32)]

    def as_dict(self) -> dict:
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class Timings(ctypes.Structure):
    _fields_ = [("ms_h2d", ctypes.c_double), ("ms_sort", ctypes.c_double), ("ms_index", ctypes.c_double),
                ("ms_count", ctypes.c_double), ("ms_pairsort", ctypes.c_double), ("ms_d2h", ctypes.c_double), ("ms_sample", ctypes.c_double),
                ("ms_stats", ctypes.c_double), ("n_count_launches", ctypes.c_uint64),
                ("n_kernel_launches", ctypes.c_uint64), ("n_library_launches", ctypes.c_uint64),
                ("ms_hist1", ctypes.c_double), ("ms_scatter1", ctypes.c_double), ("ms_hist2", ctypes.c_double),
                ("ms_scatter2", ctypes.c_double), ("ms_group", ctypes.c_double), ("ms_sample_kernels", ctypes.c_double),
                ("ms_items", ctypes.c_double), ("ms_sync", ctypes.c_double), ("ms_gather", ctypes.c_double),
                ("ms_sketch", ctypes.c_double)]

    def as_dict(self) -> dict:
        return {k: (float(getattr(self, k)) if t is ctypes.c_double else int(getattr(self, k))) for k, t in self._fields_}


class SketchResult(ctypes.Structure):
    _fields_ = [("hashes", ctypes.POINTER(ctypes.c_uint64)), ("abundances", ctypes.POINTER(ctypes.c_uint32)),
                ("offsets", ctypes.POINTER(ctypes.c_uint64)), ("n_sketches", ctypes.c_uint32), ("_pad", ctypes.c_uint32),
                ("n_kmers", ctypes.c_uint64)]


class StreamStats(ctypes.Structure):
    _fields_ = [("n_bytes", ctypes.c_uint64), ("n_bases", ctypes.c_uint64), ("n_records", ctypes.c_uint64),
                ("n_kmers", ctypes.c_uint64), ("n_chunks", ctypes.c_uint64), ("ms_h2d", ctypes.c_double),
                ("ms_parse", ctypes.c_double), ("ms_hash", ctypes.c_double), ("ms_merge", ctypes.c_double)]

    def as_dict(self) -> dict:
        return {k: (float(getattr(self, k)) if t is ctypes.c_double else int(getattr(self, k))) for k, t in self._fields_}


class SketchSet(ctypes.Structure):
    _fields_ = [("hashes", ctypes.POINTER(ctypes.c_uint64)), ("offsets", ctypes.POINTER(ctypes.c_uint64)),
                ("n_genomes", ctypes.c_uint32), ("n_unreadable", ctypes.c_uint32), ("pinned", ctypes.c_int32),
                ("_pad", ctypes.c_int32)]


PAIR_DTYPE = np.dtype([("i", "<i4"), ("j", "<i4"), ("count", "<i4")])
GENOME_COUNTS_DTYPE = np.dtype([("n_overlap", "<u4"), ("nontrivial", "<u4"), ("n_exclusive", "<u4"), ("n_match", "<u4")])
HYP_ROW_DTYPE = np.dtype([
    ("in_sample_est", "<i4"), ("_pad", "<i4"), ("p_val", "<f8"), ("num_exclusive_kmers", "<i8"),
    ("num_exclusive_kmers_coverage", "<i8"), ("num_matches", "<i8"),
    ("acceptance_threshold_with_coverage", "<f8"), ("actual_confidence_with_coverage", "<f8"),
    ("alt_confidence_mut_rate_with_coverage", "<f8"),
])

_lib = None


def load_library() -> ctypes.CDLL:
    """dlopen libyachtgpu.so from the package directory (built in-tree by __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise YgpuError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C yacht_b200/csrc). There is no CPU fallback for the hot path.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    lib.ygpu_device_count.restype = ctypes.c_int
    lib.ygpu_ctx_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int]
    lib.ygpu_ctx_destroy.argtypes = [vp]
    lib.ygpu_ctx_destroy.restype = None
    lib.ygpu_last_error.argtypes = [vp]
    lib.ygpu_last_error.restype = ctypes.c_char_p
    lib.ygpu_free.argtypes = [vp]
    lib.ygpu_free.restype = None
    lib.ygpu_host_alloc.argtypes = [u64]
    lib.ygpu_host_alloc.restype = vp
    lib.ygpu_host_free.argtypes = [vp]
    lib.ygpu_host_free.restype = None
    lib.ygpu_read_signatures.argtypes = [ctypes.POINTER(ctypes.c_char_p), u32, ctypes.c_int, ctypes.POINTER(SketchSet),
                                         ctypes.c_char_p, u64]
    lib.ygpu_read_signatures_ksize.argtypes = [ctypes.POINTER(ctypes.c_char_p), u32, ctypes.c_int, ctypes.c_int, ctypes.POINTER(SketchSet),
                                               ctypes.c_char_p, u64]
    lib.ygpu_sketch_set_free.argtypes = [ctypes.POINTER(SketchSet)]
    lib.ygpu_sketch_set_free.restype = None
    lib.ygpu_alt_mut_rate.argtypes = [vp, vp, vp, u64, ctypes.c_int, ctypes.c_double, vp]
    lib.ygpu_reset_timers.argtypes = [vp]
    lib.ygpu_get_timings.argtypes = [vp, ctypes.POINTER(Timings)]
    lib.ygpu_load_sketches.argtypes = [vp, vp, vp, u32]
    lib.ygpu_load_sketches_device.argtypes = [vp, vp, vp, u32]
    lib.ygpu_load_sketch_blocks.argtypes = [vp, vp, vp, u32, vp, u32]
    lib.ygpu_build_index.argtypes = [vp, ctypes.POINTER(IndexStats)]
    lib.ygpu_pairwise_flag.argtypes = [vp, ctypes.c_double, u32, u32, ctypes.POINTER(vp), ctypes.POINTER(u64)]
    lib.ygpu_row_partition.argtypes = [vp, u32, vp]
    lib.ygpu_upload_begin.argtypes = [vp]
    lib.ygpu_upload_block.argtypes = [vp, u32, vp, u64]
    lib.ygpu_upload_finish.argtypes = [vp, vp, u32, vp, u32]
    lib.ygpu_pairwise_flag_device.argtypes = [vp, ctypes.c_double, u32, u32, ctypes.POINTER(u64)]
    lib.ygpu_pairs_copy.argtypes = [vp, vp, ctypes.c_int]
    lib.ygpu_mark.argtypes = [vp, ctypes.c_int]
    lib.ygpu_elapsed_ms.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    lib.ygpu_set_option.argtypes = [vp, ctypes.c_char_p, ctypes.c_int64]
    lib.ygpu_get_option.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64)]
    lib.ygpu_exclusive_hashes.argtypes = [vp, vp, u64, vp, vp]
    lib.ygpu_hyp_test.argtypes = [vp, vp, vp, u64, ctypes.c_int, ctypes.c_double, ctypes.c_double, vp, ctypes.c_int, vp]
    lib.ygpu_greedy_select.argtypes = [vp, u32, vp, u64, vp, ctypes.POINTER(u32)]
    lib.ygpu_comm_get_unique_id.argtypes = [vp]
    lib.ygpu_comm_init.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp]
    lib.ygpu_comm_destroy.argtypes = [vp]
    lib.ygpu_load_sketches_sharded.argtypes = [vp, vp, vp, u32, u32, u32]
    lib.ygpu_load_sketches_sharded_device.argtypes = [vp, vp, vp, u32, u32, u32]
    lib.ygpu_load_sketches_hashrange.argtypes = [vp, vp, vp, vp, u32, u32, u32]
    lib.ygpu_load_sketches_hashrange_device.argtypes = [vp, vp, vp, vp, u32, u32, u32]
    lib.ygpu_upload_finish_sharded.argtypes = [vp, vp, u32, vp, u32, u32, u32]
    lib.ygpu_train_step_replicated.argtypes = [vp, ctypes.c_double, ctypes.POINTER(IndexStats), ctypes.POINTER(u64)]
    lib.ygpu_train_step_sharded.argtypes = [vp, ctypes.c_double, ctypes.POINTER(IndexStats), ctypes.POINTER(u64)]
    lib.ygpu_sketch_sequences.argtypes = [vp, vp, u64, vp, u32, ctypes.c_int, u64, u32, ctypes.POINTER(SketchResult)]
    lib.ygpu_sketch_result_free.argtypes = [ctypes.POINTER(SketchResult)]
    lib.ygpu_sketch_result_free.restype = None
    lib.ygpu_stream_begin.argtypes = [vp, ctypes.c_int, u64, u32, ctypes.c_int]
    lib.ygpu_stream_feed.argtypes = [vp, vp, u64]
    lib.ygpu_stream_end_file.argtypes = [vp]
    lib.ygpu_stream_finish.argtypes = [vp, ctypes.POINTER(SketchResult), ctypes.POINTER(StreamStats), ctypes.POINTER(vp),
                                       ctypes.POINTER(vp), ctypes.POINTER(u64)]
    for name in ABI_SYMBOLS:
        getattr(lib, name)  # AttributeError here means the .so does not match include/yacht_gpu.h
    _lib = lib
    return lib


class GpuContext:
    """One GPU's worth of the hot path: resident sketches, inverted index, pair flagging, run stats."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.ygpu_ctx_create(ctypes.byref(h), int(device))
        if rc != 0:
            msg = self.lib.ygpu_last_error(None)
            raise YgpuError(f"ygpu_ctx_create(device={device}) failed ({rc}): {msg.decode() if msg else ''}")
        self.h = h
        self.device = device
        self.n = 0
        self._keep = None

    # -- plumbing -----------------------------------------------------------------------------
    def _check(self, rc: int, what: str) -> None:
        if rc != 0:
            msg = self.lib.ygpu_last_error(self.h)
            raise YgpuError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.ygpu_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset_timers(self) -> None:
        self._check(self.lib.ygpu_reset_timers(self.h), "ygpu_reset_timers")

    def timings(self) -> dict:
        t = Timings()
        self._check(self.lib.ygpu_get_timings(self.h, ctypes.byref(t)), "ygpu_get_timings")
        return t.as_dict()

    # -- train path ---------------------------------------------------------------------------
    def load_sketches(self, hashes: np.ndarray, offsets: np.ndarray) -> None:
        """Host arrays (numpy uint64) -> device.  hashes[offsets[g]:offsets[g+1]] is sketch g."""
        hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offsets.shape[0] - 1
        self._check(self.lib.ygpu_load_sketches(self.h, hashes.ctypes.data, offsets.ctypes.data, n), "ygpu_load_sketches")
        self.n = n

    def load_sketches_streamed(self, hashes: np.ndarray, offsets: np.ndarray, genomes_per_block: int = 32) -> None:
        """The streaming ingest ABI (ygpu_upload_begin / _block / _finish) driven from one thread: blocks of
        `genomes_per_block` consecutive sketches, uploaded in REVERSE order (any order must work)."""
        hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = int(offsets.shape[0]) - 1
        nblocks = (n + genomes_per_block - 1) // genomes_per_block
        dst = np.array([int(offsets[min(b * genomes_per_block, n)]) for b in range(nblocks)] + [int(offsets[n])], dtype=np.uint64)
        self._check(self.lib.ygpu_upload_begin(self.h), "ygpu_upload_begin")
        for b in reversed(range(nblocks)):
            lo, hi = int(dst[b]), int(dst[b + 1])
            if hi > lo:
                blk = hashes[lo:hi]
                self._check(self.lib.ygpu_upload_block(self.h, b, blk.ctypes.data, hi - lo), "ygpu_upload_block")
        self._check(self.lib.ygpu_upload_finish(self.h, dst.ctypes.data, nblocks, offsets.ctypes.data, n), "ygpu_upload_finish")
        self.n = n

    def load_sketches_device(self, d_hashes_ptr: int, d_offsets_ptr: int, n: int) -> None:
        """Device pointers (e.g. torch tensors' data_ptr() on this context's device)."""
        self._check(self.lib.ygpu_load_sketches_device(self.h, d_hashes_ptr, d_offsets_ptr, n), "ygpu_load_sketches_device")
        self.n = n

    def build_index(self) -> dict:
        st = IndexStats()
        self._check(self.lib.ygpu_build_index(self.h, ctypes.byref(st)), "ygpu_build_index")
        return st.as_dict()

    # -- hash-range sharded build (multi-GPU; the exchange between the calls is the caller's) ------------
    def pairwise_flag(self, threshold: float, row_begin: int = 0, row_end: Optional[int] = None) -> np.ndarray:
        """Flagged ordered pairs (structured array i, j, count), sorted by (i, j)."""
        if row_end is None:
            row_end = self.n
        out = ctypes.c_void_p()
        n_out = ctypes.c_uint64()
        self._check(self.lib.ygpu_pairwise_flag(self.h, float(threshold), int(row_begin), int(row_end),
                                                ctypes.byref(out), ctypes.byref(n_out)), "ygpu_pairwise_flag")
        try:
            k = int(n_out.value)
            if k == 0:
                return np.zeros(0, dtype=PAIR_DTYPE)
            buf = ctypes.string_at(out, k * PAIR_DTYPE.itemsize)
            return np.frombuffer(buf, dtype=PAIR_DTYPE).copy()
        finally:
            self.lib.ygpu_free(out)

    def pairwise_flag_device(self, threshold: float, row_begin: int = 0, row_end: Optional[int] = None) -> int:
        """Same as pairwise_flag but the pairs stay on the device; returns how many there are."""
        if row_end is None:
            row_end = self.n
        n_out = ctypes.c_uint64()
        self._check(self.lib.ygpu_pairwise_flag_device(self.h, float(threshold), int(row_begin), int(row_end),
                                                       ctypes.byref(n_out)), "ygpu_pairwise_flag_device")
        return int(n_out.value)

    # ---- sharded train step: one rank per GPU (include/yacht_gpu.h) ----------------------------------------
    def comm_init(self, rank: int, nranks: int, unique_id: bytes) -> None:
        buf = ctypes.create_string_buffer(bytes(unique_id), COMM_ID_BYTES)
        self._check(self.lib.ygpu_comm_init(self.h, int(rank), int(nranks), ctypes.cast(buf, ctypes.c_void_p)), "ygpu_comm_init")

    def load_sketches_sharded(self, hashes_slice: np.ndarray, offsets: np.ndarray, g_begin: int, g_end: int) -> None:
        """hashes_slice = hashes[offsets[g_begin]:offsets[g_end]] (HOST); offsets = the offsets of ALL genomes."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        hashes_slice = np.ascontiguousarray(hashes_slice, dtype=np.uint64)
        self._check(self.lib.ygpu_load_sketches_sharded(self.h, hashes_slice.ctypes.data if hashes_slice.size else None, offsets.ctypes.data,
                                                        int(offsets.shape[0]) - 1, int(g_begin), int(g_end)), "ygpu_load_sketches_sharded")

    def load_sketches_sharded_ptr(self, slice_ptr: int, on_device: bool, offsets: np.ndarray, g_begin: int, g_end: int) -> None:
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        fn = self.lib.ygpu_load_sketches_sharded_device if on_device else self.lib.ygpu_load_sketches_sharded
        self._check(fn(self.h, ctypes.c_void_p(slice_ptr), offsets.ctypes.data, int(offsets.shape[0]) - 1, int(g_begin), int(g_end)),
                    "ygpu_load_sketches_sharded")

    def load_sketches_hashrange(self, part_hashes, part_offsets: np.ndarray, sizes: np.ndarray, row_begin: int, row_end: int,
                                on_device: bool = False) -> None:
        """Hash-range residency: part_hashes (numpy array, or a raw pointer when on_device) = of every sketch the hashes inside
        this rank's hash range; part_offsets = CSR over that share; sizes = the full sketch sizes."""
        part_offsets = np.ascontiguousarray(part_offsets, dtype=np.uint64)
        sizes = np.ascontiguousarray(sizes, dtype=np.uint32)
        n = int(sizes.shape[0])
        if isinstance(part_hashes, np.ndarray):
            part_hashes = np.ascontiguousarray(part_hashes, dtype=np.uint64)
            ptr = part_hashes.ctypes.data if part_hashes.size else None
        else:
            ptr = ctypes.c_void_p(int(part_hashes))
        fn = self.lib.ygpu_load_sketches_hashrange_device if on_device else self.lib.ygpu_load_sketches_hashrange
        self._check(fn(self.h, ptr, part_offsets.ctypes.data, sizes.ctypes.data, n, int(row_begin), int(row_end)), "ygpu_load_sketches_hashrange")

    def train_step_sharded(self, threshold: float) -> Tuple[dict, int]:
        """Index build + pairwise count/flag over all ranks; afterwards pairs_copy()/pairs_host() give the COMPLETE sorted pair list."""
        st = IndexStats()
        n_out = ctypes.c_uint64(0)
        self._check(self.lib.ygpu_train_step_sharded(self.h, float(threshold), ctypes.byref(st), ctypes.byref(n_out)), "ygpu_train_step_sharded")
        return st.as_dict(), int(n_out.value)

    def train_step_replicated(self, threshold: float) -> Tuple[dict, int]:
        """Replicated index (every rank holds all sketches: load_sketches), rows split by work, pair lists gathered."""
        st = IndexStats()
        n_out = ctypes.c_uint64(0)
        self._check(self.lib.ygpu_train_step_replicated(self.h, float(threshold), ctypes.byref(st), ctypes.byref(n_out)), "ygpu_train_step_replicated")
        return st.as_dict(), int(n_out.value)

    def pairs_host(self, n_pairs: int) -> np.ndarray:
        buf = np.empty(n_pairs, dtype=PAIR_DTYPE)
        if n_pairs:
            self.pairs_copy(buf.ctypes.data, False)
        return buf

    def pairs_copy(self, dst_ptr: int, dst_is_device: bool) -> None:
        self._check(self.lib.ygpu_pairs_copy(self.h, dst_ptr, 1 if dst_is_device else 0), "ygpu_pairs_copy")

    def mark(self, slot: int) -> None:
        self._check(self.lib.ygpu_mark(self.h, slot), "ygpu_mark")

    def elapsed_ms(self, a: int, b: int) -> float:
        ms = ctypes.c_double()
        self._check(self.lib.ygpu_elapsed_ms(self.h, a, b, ctypes.byref(ms)), "ygpu_elapsed_ms")
        return float(ms.value)

    def set_option(self, name: str, value: int) -> None:
        self._check(self.lib.ygpu_set_option(self.h, name.encode(), int(value)), "ygpu_set_option")

    def get_option(self, name: str) -> int:
        """Read-only state of the last count call (include/yacht_gpu.h: ygpu_get_option)."""
        v = ctypes.c_int64(0)
        self._check(self.lib.ygpu_get_option(self.h, name.encode(), ctypes.byref(v)), "ygpu_get_option")
        return int(v.value)

    def row_partition(self, nparts: int) -> np.ndarray:
        b = np.zeros(nparts + 1, dtype=np.uint32)
        self._check(self.lib.ygpu_row_partition(self.h, int(nparts), b.ctypes.data), "ygpu_row_partition")
        return b

    # -- sketching ----------------------------------------------------------------------------
    def sketch_sequences(self, bases, sketch_offsets: Sequence[int], ksize: int, max_hash: int, seed: int = 42):
        """FracMinHash sketches of bases[sketch_offsets[s]:sketch_offsets[s+1]] (bytes / uint8 array; anything that is not
        A/C/G/T, e.g. the '\\n' between two records, breaks the windows).  Returns (hashes, abundances, offsets, n_kmers):
        per sketch the distinct kept hashes ascending and how often each occurred."""
        arr = np.frombuffer(bases, dtype=np.uint8) if isinstance(bases, (bytes, bytearray, memoryview)) else np.ascontiguousarray(bases, dtype=np.uint8)
        off = np.ascontiguousarray(sketch_offsets, dtype=np.uint64)
        res = SketchResult()
        self._check(self.lib.ygpu_sketch_sequences(self.h, arr.ctypes.data if arr.size else None, arr.size, off.ctypes.data, off.shape[0] - 1,
                                                   int(ksize), int(max_hash), int(seed), ctypes.byref(res)), "ygpu_sketch_sequences")
        try:
            ns = int(res.n_sketches)
            offsets = np.ctypeslib.as_array(res.offsets, shape=(ns + 1,)).copy()
            total = int(offsets[-1])
            if total:
                hashes = np.ctypeslib.as_array(res.hashes, shape=(total,)).copy()
                abund = np.ctypeslib.as_array(res.abundances, shape=(total,)).copy()
            else:
                hashes, abund = np.zeros(0, np.uint64), np.zeros(0, np.uint32)
            return hashes, abund, offsets, int(res.n_kmers)
        finally:
            self.lib.ygpu_sketch_result_free(ctypes.byref(res))

    # -- streamed sketching (ygpu_stream_*) ------------------------------------------------------
    def _stream_error(self, rc: int, what: str, path: Optional[str]) -> None:
        if rc == 0:
            return
        msg = self.lib.ygpu_last_error(self.h)
        text = msg.decode(errors="replace") if msg else ""
        if rc == -3 and path is not None:           # YGPU_ERR_ARG: the input is not a FASTA / FASTQ file the reader accepts
            raise ValueError(f"{path}: {text}")
        raise YgpuError(f"{what} failed ({rc}): {text}")

    def host_buffer(self, nbytes: int):
        """A page-locked host buffer (ygpu_host_alloc) -> (writable memoryview, address, release function)."""
        ptr = self.lib.ygpu_host_alloc(int(nbytes))
        if not ptr:
            raise YgpuError(f"ygpu_host_alloc({nbytes}) failed")
        mv = memoryview((ctypes.c_uint8 * int(nbytes)).from_address(ptr)).cast("B")
        return mv, int(ptr), lambda: self.lib.ygpu_host_free(ctypes.c_void_p(ptr))

    def stream_begin(self, ksize: int, max_hash: int, seed: int = 42, per_record: bool = False) -> None:
        self._check(self.lib.ygpu_stream_begin(self.h, int(ksize), int(max_hash), int(seed),
                                               STREAM_PER_RECORD if per_record else STREAM_WHOLE), "ygpu_stream_begin")

    def stream_feed(self, ptr: int, n: int, path: Optional[str] = None) -> None:
        """The next n bytes of the current file at host address ptr (free to reuse when this returns)."""
        self._stream_error(self.lib.ygpu_stream_feed(self.h, ctypes.c_void_p(ptr), int(n)), "ygpu_stream_feed", path)

    def stream_end_file(self, path: Optional[str] = None) -> None:
        self._stream_error(self.lib.ygpu_stream_end_file(self.h), "ygpu_stream_end_file", path)

    def stream_finish(self, path: Optional[str] = None):
        """-> (hashes, abundances, offsets, names or None, stats dict); names are bytes, one per record that kept its name."""
        res, st = SketchResult(), StreamStats()
        names, name_off, n_names = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_uint64()
        self._stream_error(self.lib.ygpu_stream_finish(self.h, ctypes.byref(res), ctypes.byref(st), ctypes.byref(names),
                                                       ctypes.byref(name_off), ctypes.byref(n_names)), "ygpu_stream_finish", path)
        try:
            ns = int(res.n_sketches)
            offsets = np.ctypeslib.as_array(res.offsets, shape=(ns + 1,)).copy()
            total = int(offsets[-1])
            if total:
                hashes = np.ctypeslib.as_array(res.hashes, shape=(total,)).copy()
                abund = np.ctypeslib.as_array(res.abundances, shape=(total,)).copy()
            else:
                hashes, abund = np.zeros(0, np.uint64), np.zeros(0, np.uint32)
            out_names = None
            nn = int(n_names.value)
            if nn:
                off = np.ctypeslib.as_array(ctypes.cast(name_off, ctypes.POINTER(ctypes.c_uint64)), shape=(nn + 1,)).copy()
                blob = ctypes.string_at(names, int(off[-1])) if int(off[-1]) else b""
                out_names = [blob[int(off[i]):int(off[i + 1])] for i in range(nn)]
            return hashes, abund, offsets, out_names, st.as_dict()
        finally:
            self.lib.ygpu_sketch_result_free(ctypes.byref(res))
            self.lib.ygpu_free(names)
            self.lib.ygpu_free(name_off)

    # -- run path -----------------------------------------------------------------------------
    def exclusive_hashes(self, sample: np.ndarray, mask: Optional[np.ndarray] = None) -> np.ndarray:
        sample = np.ascontiguousarray(sample, dtype=np.uint64)
        counts = np.zeros(self.n, dtype=GENOME_COUNTS_DTYPE)
        mptr = None
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
            if mask.shape[0] != self.n:
                raise ValueError("mask must have one entry per loaded genome")
            mptr = mask.ctypes.data
        self._check(self.lib.ygpu_exclusive_hashes(self.h, sample.ctypes.data, sample.shape[0], mptr,
                                                   counts.ctypes.data), "ygpu_exclusive_hashes")
        return counts

    def hyp_test(self, n_exclusive: Sequence[int], n_match: Sequence[int], ksize: int, significance: float,
                 ani_thresh: float, min_coverage: Sequence[float]) -> np.ndarray:
        """rows[c, r] = single_hyp_test((n_exclusive[r], n_match[r]), ksize, significance, ani, cov[c])."""
        ne = np.ascontiguousarray(n_exclusive, dtype=np.int64)
        nm = np.ascontiguousarray(n_match, dtype=np.int64)
        cov = np.ascontiguousarray(min_coverage, dtype=np.float64)
        rows = np.zeros((cov.shape[0], ne.shape[0]), dtype=HYP_ROW_DTYPE)
        self._check(self.lib.ygpu_hyp_test(self.h, ne.ctypes.data, nm.ctypes.data, ne.shape[0], int(ksize),
                                           float(significance), float(ani_thresh), cov.ctypes.data, cov.shape[0],
                                           rows.ctypes.data), "ygpu_hyp_test")
        return rows


    def alt_mut_rate(self, nu: Sequence[int], thresh: Sequence[int], ksize: int, significance: float = 0.99) -> np.ndarray:
        a = np.ascontiguousarray(nu, dtype=np.int64)
        b = np.ascontiguousarray(thresh, dtype=np.int64)
        out = np.zeros(a.shape[0], dtype=np.float64)
        self._check(self.lib.ygpu_alt_mut_rate(self.h, a.ctypes.data, b.ctypes.data, a.shape[0], int(ksize),
                                               float(significance), out.ctypes.data), "ygpu_alt_mut_rate")
        return out


def read_signatures(paths: Sequence[str], threads: int = 1, ksize: int = 0) -> Tuple[np.ndarray, np.ndarray, int]:
    """Multi-threaded native ingest of uncompressed .sig files -> (hashes, offsets, n_unreadable).
    ksize = 0 mirrors the reference core's reader (main.cpp:62-124): first record, first sub-signature.  ksize > 0 mirrors
    load_signature_with_ksize (utils.py:31-51): exactly one sub-signature of that k-mer size per file, else an error."""
    lib = load_library()
    n = len(paths)
    arr = (ctypes.c_char_p * max(n, 1))(*[os.fsencode(p) for p in paths])
    ss = SketchSet()
    err = ctypes.create_string_buffer(2048)
    if ksize > 0:
        rc = lib.ygpu_read_signatures_ksize(arr, n, int(threads), int(ksize), ctypes.byref(ss), err, 2048)
    else:
        rc = lib.ygpu_read_signatures(arr, n, int(threads), ctypes.byref(ss), err, 2048)
    if rc != 0:
        raise YgpuError(f"ygpu_read_signatures failed ({rc}): {err.value.decode(errors='replace')}")
    try:
        offsets = np.ctypeslib.as_array(ss.offsets, shape=(n + 1,)).copy()
        T = int(offsets[-1])
        hashes = np.ctypeslib.as_array(ss.hashes, shape=(max(T, 1),))[:T].copy() if T else np.zeros(0, dtype=np.uint64)
        return hashes, offsets, int(ss.n_unreadable)
    finally:
        lib.ygpu_sketch_set_free(ctypes.byref(ss))


def greedy_select(offsets: np.ndarray, pairs: np.ndarray) -> np.ndarray:
    """do_yacht_train (reference main.cpp:371-420) over the flagged pairs of the whole database: the retained genome
    ids in the reference's visit order (host code inside the library: the same std::sort call as the reference)."""
    lib = load_library()
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    pairs = np.ascontiguousarray(pairs, dtype=PAIR_DTYPE)
    n = int(offsets.shape[0]) - 1
    out = np.zeros(max(n, 1), dtype=np.int32)
    ns = ctypes.c_uint32(0)
    rc = lib.ygpu_greedy_select(offsets.ctypes.data, n, pairs.ctypes.data if len(pairs) else None, len(pairs), out.ctypes.data,
                                ctypes.byref(ns))
    if rc != 0:
        raise YgpuError(f"ygpu_greedy_select failed ({rc})")
    return out[: int(ns.value)].copy()


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the library (rank 0 calls it and hands the bytes to every rank)."""
    lib = load_library()
    buf = ctypes.create_string_buffer(COMM_ID_BYTES)
    rc = lib.ygpu_comm_get_unique_id(ctypes.cast(buf, ctypes.c_void_p))
    if rc != 0:
        msg = lib.ygpu_last_error(None)
        raise YgpuError(f"ygpu_comm_get_unique_id failed ({rc}): {msg.decode() if msg else ''}")
    return buf.raw


def device_count() -> int:
    return int(load_library().ygpu_device_count())
