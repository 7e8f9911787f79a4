"""TEST INFRASTRUCTURE ONLY -- Python handle on the CPU oracles of the train path.

* :func:`oracle_train`  calls the C++ restatement (oracle/train_oracle.cpp) through ctypes;
  :func:`oracle_train_sparse` the same restatement with a sparse row accumulator, for large databases.
* :func:`reference_train` runs the UNMODIFIED reference core (oracle/_ref/run_yacht_train_core_ref,
  compiled from /root/reference/src/cpp by oracle/Makefile) on signature files written to a
  scratch directory, and parses what it wrote.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  Parity status: pinned (see the header of train_oracle.cpp).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys
import time
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libtrain_oracle.so")
PORT_BIN = os.path.join(HERE, "_build", "train_oracle")
REF_BIN = os.path.join(HERE, "_ref", "run_yacht_train_core_ref")


class _YoPair(ctypes.Structure):
    _fields_ = [("i", ctypes.c_int32), ("j", ctypes.c_int32), ("count", ctypes.c_int32),
                ("_pad", ctypes.c_int32), ("jaccard", ctypes.c_double), ("c_ij", ctypes.c_double),
                ("c_ji", ctypes.c_double)]


class _YoResult(ctypes.Structure):
    _fields_ = [("pairs", ctypes.POINTER(_YoPair)), ("n_pairs", ctypes.c_uint64),
                ("selected", ctypes.POINTER(ctypes.c_int32)), ("n_selected", ctypes.c_uint32),
                ("n_distinct", ctypes.c_uint64), ("n_singleton", ctypes.c_uint64),
                ("n_index", ctypes.c_uint64), ("n_postings", ctypes.c_uint64),
                ("n_increments", ctypes.c_uint64)]


PAIR_DTYPE = np.dtype([("i", "<i4"), ("j", "<i4"), ("count", "<i4"), ("_pad", "<i4"),
                       ("jaccard", "<f8"), ("c_ij", "<f8"), ("c_ji", "<f8")])


@dataclass
class TrainResult:
    pairs: np.ndarray           # structured PAIR_DTYPE, (i, j) ascending
    selected: np.ndarray        # int32 genome ids, greedy visit order
    n_distinct: int
    n_singleton: int
    n_index: int
    n_postings: int = 0
    n_increments: int = 0
    _lines: Optional[List[str]] = None

    @property
    def lines(self) -> List[str]:
        """Pair-file lines, sorted (formatted on first use: a threshold-0 run can hold tens of millions of pairs)."""
        if self._lines is None:
            self._lines = sorted(format_pairs(self.pairs))
        return self._lines

    @lines.setter
    def lines(self, value: List[str]) -> None:
        self._lines = value


def build(quiet: bool = True) -> None:
    """(Re)build the oracle artefacts via oracle/Makefile (g++ only)."""
    cmd = ["make", "-C", HERE, "all"]
    subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL if quiet else None)


_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        lib = ctypes.CDLL(LIB_PATH)
        lib.yo_train.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_double,
                                 ctypes.POINTER(_YoResult)]
        lib.yo_train.restype = ctypes.c_int
        lib.yo_train_sparse.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_double, ctypes.c_uint32,
                                        ctypes.c_uint32, ctypes.POINTER(_YoResult)]
        lib.yo_train_sparse.restype = ctypes.c_int
        lib.yo_free_result.argtypes = [ctypes.POINTER(_YoResult)]
        lib.yo_format_pair.argtypes = [ctypes.POINTER(_YoPair), ctypes.c_char_p, ctypes.c_int]
        lib.yo_format_pair.restype = ctypes.c_int
        _lib = lib
    return _lib


def format_pairs(pairs: np.ndarray) -> List[str]:
    """Pair-file lines "i,j,jaccard,c_ij,c_ji" with %g doubles (reference main.cpp:305)."""
    return ["%d,%d,%g,%g,%g" % (int(p["i"]), int(p["j"]), float(p["jaccard"]), float(p["c_ij"]), float(p["c_ji"]))
            for p in pairs]


def oracle_train(hashes: np.ndarray, offsets: np.ndarray, thr: float) -> TrainResult:
    lib = _load()
    hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = offsets.shape[0] - 1
    res = _YoResult()
    rc = lib.yo_train(hashes.ctypes.data, offsets.ctypes.data, n, float(thr), ctypes.byref(res))
    if rc != 0:
        raise RuntimeError(f"yo_train failed rc={rc}")
    return _take(lib, res)


def oracle_train_sparse(hashes: np.ndarray, offsets: np.ndarray, thr: float, row_begin: int = 0,
                        row_end: Optional[int] = None) -> TrainResult:
    """oracle_train with a sparse row accumulator (yo_train_sparse): O(sum of L^2) instead of O(n^2), so databases of
    millions of genomes can be checked.  A row range returns what GpuContext.pairwise_flag does for it: both ordered pairs
    of every {i, j} whose smaller genome lies in [row_begin, row_end).  `selected` is the greedy order over the returned
    pairs (the reference's when the range is the whole database)."""
    lib = _load()
    hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = offsets.shape[0] - 1
    res = _YoResult()
    rc = lib.yo_train_sparse(hashes.ctypes.data, offsets.ctypes.data, n, float(thr), int(row_begin),
                             n if row_end is None else int(row_end), ctypes.byref(res))
    if rc != 0:
        raise RuntimeError(f"yo_train_sparse failed rc={rc}")
    return _take(lib, res)


def _take(lib, res: _YoResult) -> TrainResult:
    """Copy a yo_result into numpy and release it."""
    try:
        npairs = int(res.n_pairs)
        if npairs:
            buf = ctypes.string_at(res.pairs, npairs * PAIR_DTYPE.itemsize)
            pairs = np.frombuffer(buf, dtype=PAIR_DTYPE).copy()
        else:
            pairs = np.zeros(0, dtype=PAIR_DTYPE)
        nsel = int(res.n_selected)
        sel = np.ctypeslib.as_array(res.selected, shape=(max(nsel, 1),))[:nsel].copy() if nsel else np.zeros(0, np.int32)
        out = TrainResult(pairs=pairs, selected=sel.astype(np.int32), n_distinct=int(res.n_distinct),
                          n_singleton=int(res.n_singleton), n_index=int(res.n_index),
                          n_postings=int(res.n_postings), n_increments=int(res.n_increments))
    finally:
        lib.yo_free_result(ctypes.byref(res))
    return out


def write_sig_dir(hashes: np.ndarray, offsets: np.ndarray, workdir: str, names: Optional[List[str]] = None) -> List[str]:
    """Write one sourmash-shaped .sig per sketch plus the file list; returns the paths (id order)."""
    sys.path.insert(0, os.path.dirname(HERE))
    from yacht_b200 import sigio  # plain file writer, no device code
    os.makedirs(os.path.join(workdir, "signatures"), exist_ok=True)
    paths = []
    n = offsets.shape[0] - 1
    for g in range(n):
        mins = hashes[int(offsets[g]):int(offsets[g + 1])]
        p = os.path.join(workdir, "signatures", f"g{g:07d}.sig")
        sigio.write_signature(p, names[g] if names else f"genome_{g}", mins)
        paths.append(p)
    with open(os.path.join(workdir, "training_sig_files.tsv"), "w") as f:
        for p in paths:
            f.write(p + "\n")
    return paths


_par_db = None
_par_paths = None


def _par_write(rng):
    from yacht_b200 import sigio
    for g in range(rng[0], rng[1]):
        sigio.write_signature(_par_paths[g], f"genome_{g}", _par_db.hashes[int(_par_db.offsets[g]):int(_par_db.offsets[g + 1])])
    return rng[1] - rng[0]


def write_sig_dir_parallel(db, workdir: str, threads: Optional[int] = None) -> List[str]:
    """write_sig_dir on all host cores (forked workers see `db` -- anything with .hashes / .offsets / .n -- without
    copying it): 85 205 signature files (7.5 GB of JSON) take ~15 s instead of minutes."""
    global _par_db, _par_paths
    from multiprocessing import Pool
    sys.path.insert(0, os.path.dirname(HERE))
    threads = threads or os.cpu_count() or 8
    n = int(db.n)
    os.makedirs(os.path.join(workdir, "signatures"), exist_ok=True)
    _par_db = db
    _par_paths = [os.path.join(workdir, "signatures", f"g{g:07d}.sig") for g in range(n)]
    if n < 2000:
        _par_write((0, n))
    else:
        step = max(1, n // (4 * threads))
        with Pool(threads) as pool:
            pool.map(_par_write, [(a, min(n, a + step)) for a in range(0, n, step)])
    with open(os.path.join(workdir, "training_sig_files.tsv"), "w") as f:
        for q in _par_paths:
            f.write(q + "\n")
    paths, _par_db, _par_paths = _par_paths, None, None
    return paths


def parse_core_outputs(workdir: str, paths: List[str], selected_file: str, stdout: str) -> TrainResult:
    import glob
    lines: List[str] = []
    for fn in glob.glob(os.path.join(workdir, "*_*.txt")):
        with open(fn) as f:
            lines.extend(l.rstrip("\n") for l in f if l.strip())
    with open(selected_file) as f:
        sel_paths = [l.rstrip("\n") for l in f if l.strip()]
    idx = {p: g for g, p in enumerate(paths)}
    stats = {"distinct": 0, "single": 0, "index": 0}
    for l in stdout.splitlines():
        if l.startswith("Total number of distinct hashes that appear in only one sketch:"):
            stats["single"] = int(l.rsplit(":", 1)[1])
        elif l.startswith("Total number of distinct hashes:"):
            stats["distinct"] = int(l.rsplit(":", 1)[1])
        elif l.startswith("Size of the index:"):
            stats["index"] = int(l.rsplit(":", 1)[1])
    return TrainResult(pairs=np.zeros(0, dtype=PAIR_DTYPE),
                       selected=np.array([idx[p] for p in sel_paths], dtype=np.int32),
                       n_distinct=stats["distinct"], n_singleton=stats["single"], n_index=stats["index"],
                       _lines=sorted(lines))


def run_core_binary(binary: str, filelist: str, workdir: str, thr: float, threads: int = 1, passes: int = 1,
                    timeout: Optional[float] = None) -> Tuple[str, float]:
    """Run a train-core executable with the reference CLI; returns (stdout, wall seconds)."""
    sel = os.path.join(workdir, "selected_result.tsv")
    cmd = [binary, "-t", str(threads), "-c", repr(float(thr)), "-p", str(passes), filelist, workdir, sel]
    t0 = time.perf_counter()
    cp = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    dt = time.perf_counter() - t0
    if cp.returncode != 0:
        raise RuntimeError(f"{binary} exited {cp.returncode}: {cp.stderr[-2000:]}")
    return cp.stdout, dt


def reference_available() -> bool:
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def reference_train(hashes: np.ndarray, offsets: np.ndarray, thr: float, workdir: str, threads: int = 1,
                    passes: int = 1) -> TrainResult:
    """The compiled reference core on the same sketches (written as .sig JSON into workdir)."""
    if not reference_available():
        raise FileNotFoundError(REF_BIN)
    paths = write_sig_dir(hashes, offsets, workdir)
    out, _ = run_core_binary(REF_BIN, os.path.join(workdir, "training_sig_files.tsv"), workdir, thr, threads, passes)
    return parse_core_outputs(workdir, paths, os.path.join(workdir, "selected_result.tsv"), out)


def parse_phase_times(stdout: str) -> dict:
    """The four self-reported phase timers of the reference core (main.cpp:458,471,483,495), ms."""
    keys = {"Time taken to read all sketches": "read_ms", "Time taken to build index": "index_ms",
            "Time taken to compute intersection matrix": "matrix_ms", "Time taken to do yacht train": "greedy_ms"}
    out = {}
    for l in stdout.splitlines():
        for k, v in keys.items():
            if l.startswith(k):
                out[v] = int(l.split(":")[1].strip().split()[0])
    return out
