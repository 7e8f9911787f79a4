"""The train step past 2^20 genomes and on the count kernel's automatically chosen tiled accumulators, bit-exact against the
sparse reference (oracle_train_sparse, itself checked against the pinned dense one in tests/test_sparse_oracle.py).

Branches that only large databases take, each case asserting which one answered:

* N = 2^20, hash width 55 (scaled 1000): MSD index path, genome ids of 20 bits inline in work items at their widest;
* N = 2^20 + 1, width 55: ids of 21 bits do not pack beside 55 hash bits: the general sort path (index and run);
* N = 2^20 + 1, width 54 (scaled 2000): MSD path with no inline ids, every item a posting slice; in-sketch duplicates,
  so 32-bit counters and the per-pair fp64 containment test;
* the first N whose packed 16-bit row no longer fits shared memory (103 393 at a 227 KiB opt-in limit): two u16 column
  tiles, a pair sharing 65 535 hashes (a counter at 0xFFFF), and with 65 536 shared hashes 32-bit tiles.

The expected tile geometry is recomputed here from the device's opt-in shared-memory limit.
"""
import ctypes

import numpy as np
import pytest

from harness import large_n
from oracle import run_oracle as ro
from oracle import sketch_oracle as so
from oracle import train_oracle as to
from yacht_b200 import _lib

pytestmark = pytest.mark.gpu

THR = 0.95 ** 31
N20 = 2 ** 20
H55 = so.max_hash_for_scaled(1000)      # hashes of 55 bits
H54 = so.max_hash_for_scaled(2000)      # below 2^54
K3_FIXED = 4096 * 4 + 1024 * 8 + 64     # touched list + long-segment queue + alignment (yacht_gpu.cu: pairwise_device)


def _budget():
    """The count kernel's shared-memory budget, from the device's opt-in limit read through the CUDA runtime the library
    links (already loaded by load_library, so dlopen by soname returns that very runtime)."""
    _lib.load_library()
    rt = ctypes.CDLL("libcudart.so.12")
    optin = ctypes.c_int(0)
    assert rt.cudaDeviceGetAttribute(ctypes.byref(optin), 97, 0) == 0      # cudaDevAttrMaxSharedMemoryPerBlockOptin
    return optin.value - K3_FIXED - 1024


def geometry(n, u16_ok, budget):
    """(tile_w, n_tiles, u16) the count kernel picks for n genomes."""
    tile_w, u16 = n, False
    if n * 4 > budget:
        if u16_ok and n * 2 <= budget:
            u16 = True
        elif u16_ok:
            u16, tile_w = True, (budget // 2) & ~1
        else:
            tile_w = budget // 4
    return tile_w, -(-n // tile_w), u16


class _Pairs:
    def __init__(self, p):
        self.t = np.stack([np.asarray(p[f], dtype=np.int64) for f in ("i", "j", "count")], axis=1) if len(p) else np.zeros((0, 3), np.int64)

    def __eq__(self, other):
        return self.t.shape == other.t.shape and bool(np.array_equal(self.t, other.t))

    def __repr__(self):
        return f"<{len(self.t)} pairs, first {self.t[:5].tolist()}>"


@pytest.fixture(scope="module")
def budget():
    return _budget()


@pytest.fixture(scope="module")
def dbs(budget):
    """Each database, built once for the module on first use."""
    n16 = budget // 2 + 1                                  # first N whose packed u16 row needs two tiles
    tws = (geometry(2 * N20, True, budget)[0], geometry(2 * N20, False, budget)[0])
    spec = {
        "n2^20_h55": dict(n=N20, max_hash=H55, seed=1, tile_ws=tws),
        "n2^20+1_h55": dict(n=N20 + 1, max_hash=H55, seed=2, tile_ws=tws),
        "n2^20+1_h54_dup": dict(n=N20 + 1, max_hash=H54, seed=3, tile_ws=tws, dup=True),
        "n2^20+1_h54_small": dict(n=N20 + 1, max_hash=H54, seed=4, tile_ws=tws, wide=False, big=False),
        f"n{n16}_twin65535": dict(n=n16, max_hash=H55, seed=5, tile_ws=tws, twin=65535),
        f"n{n16}_twin65536": dict(n=n16, max_hash=H55, seed=6, tile_ws=tws, twin=65536),
    }
    cache = {}

    def get(name):
        if name not in cache:
            kw = dict(spec[name])
            cache[name] = large_n.make_large_db(kw.pop("n"), kw.pop("max_hash"), kw.pop("seed"), **kw)
        return cache[name]
    get.n16 = n16
    return get


def _on_value_thresholds(ref, x):
    """Two thresholds that equal the containment of flagged pairs of planted groups: those pairs pass only through !(c < thr)."""
    p = ref.pairs
    planted = np.isin(p["i"], np.concatenate(x.groups)) & (p["c_ij"] < 1.0) & (p["c_ij"] > THR)
    vals = np.unique(p["c_ij"][planted])
    return [float(vals[len(vals) // 2]), float(vals[-1])] if len(vals) else []


def _narrow_ranges(x, n):
    lo = [0, N20 - 8, 2 ** 19 - 8, n - 16] + [r - 4 for r in x.wide_rows] + [int(m) for m in x.big_members[:1]]
    return sorted({(max(0, a), min(n, a + 20)) for a in lo if a < n})


def _check_train(ctx, x, budget, *, msd, u16, big):
    db = x.db
    n = db.n
    refs = {THR: to.oracle_train_sparse(db.hashes, db.offsets, THR)}
    for t in _on_value_thresholds(refs[THR], x):
        refs[t] = to.oracle_train_sparse(db.hashes, db.offsets, t)
    ranges = {r: to.oracle_train_sparse(db.hashes, db.offsets, 0.0, *r) for r in _narrow_ranges(x, n)}
    ref = refs[THR]
    assert 0 < len(ref.pairs) < 10 ** 7
    for t, r in refs.items():
        if t != THR:
            assert np.any(r.pairs["c_ij"] == t), t                  # a pair sits exactly on the threshold
    full = None
    try:
        for path in (1, 0):
            ctx.set_option("index_path", path)
            ctx.load_sketches(db.hashes, db.offsets)
            st = ctx.build_index()
            for f in ("n_distinct", "n_singleton", "n_index", "n_postings", "n_increments"):
                assert st[f] == getattr(ref, f), (path, f, st)
            assert st["index_path"] == (1 if path == 1 and msd else 0), (path, st)
            assert (st["big_buckets"] >= 1) == (path == 1 and msd and big), (path, st)
            u16_ok = not st["has_duplicates"] and st["max_sketch"] <= 65535
            tile_w, n_tiles, use_u16 = geometry(n, u16_ok, budget)
            assert use_u16 == u16 and n_tiles > 1
            for thr, r in refs.items():
                for ck in (1, 2):
                    ctx.set_option("count_kernel", ck)
                    got = ctx.pairwise_flag(thr)
                    assert _Pairs(got) == _Pairs(r.pairs), (path, ck, thr)
                    geo = {k: ctx.get_option("last_count_" + k) for k in ("kernel", "tile_w", "n_tiles", "u16", "overflow_rows")}
                    assert (geo["kernel"], geo["tile_w"], geo["n_tiles"], geo["u16"]) == (ck, tile_w, n_tiles, int(use_u16)), geo
                    if ck == 2 and (x.wide_rows or big):
                        assert geo["overflow_rows"] > 0, geo             # rows deferred to the dense kernel over many tiles
                    print(f"n={n} index_path={st['index_path']} big_buckets={st['big_buckets']} thr={thr:.6g} {geo} pairs={len(got)}")
                    if thr == THR and ck == 1 and path == 1:
                        full = got
                ctx.set_option("count_kernel", 0)
                ctx.set_option("count_thresholds", 0)
                try:
                    assert _Pairs(ctx.pairwise_flag(thr)) == _Pairs(r.pairs), (path, "fp64 per pair", thr)
                finally:
                    ctx.set_option("count_thresholds", 1)
            for (lo, hi), r in ranges.items():                 # every ordered pair's count of these rows
                for ck in (1, 2):
                    ctx.set_option("count_kernel", ck)
                    assert _Pairs(ctx.pairwise_flag(0.0, lo, hi)) == _Pairs(r.pairs), (path, ck, lo, hi)
                ctx.set_option("count_kernel", 0)
            b = ctx.row_partition(4)
            assert b[0] == 0 and b[-1] == n and all(b[k] <= b[k + 1] for k in range(4))
            parts = [ctx.pairwise_flag(THR, int(b[k]), int(b[k + 1])) for k in range(4)]
            assert _Pairs(np.sort(np.concatenate(parts), order=["i", "j"])) == _Pairs(ref.pairs), path
    finally:
        ctx.set_option("index_path", 1)
        ctx.set_option("count_kernel", 0)
    assert _lib.greedy_select(db.offsets, full).tolist() == ref.selected.tolist()
    return full


def test_n_2pow20_msd_inline_ids_at_their_widest(gpu_ctx, dbs, budget):
    x = dbs("n2^20_h55")
    assert int(x.db.hashes.max()).bit_length() == 55
    _check_train(gpu_ctx, x, budget, msd=True, u16=True, big=True)


def test_n_2pow20_plus1_h55_takes_the_general_path(gpu_ctx, dbs, budget):
    x = dbs("n2^20+1_h55")
    assert int(x.db.hashes.max()).bit_length() == 55
    _check_train(gpu_ctx, x, budget, msd=False, u16=True, big=True)


def test_n_2pow20_plus1_h54_msd_without_inline_ids(gpu_ctx, dbs, budget):
    x = dbs("n2^20+1_h54_dup")
    assert int(x.db.hashes.max()).bit_length() == 54
    _check_train(gpu_ctx, x, budget, msd=True, u16=False, big=True)


@pytest.mark.parametrize("twin,u16", [(65535, True), (65536, False)])
def test_first_u16_tiled_n(gpu_ctx, dbs, budget, twin, u16):
    x = dbs(f"n{dbs.n16}_twin{twin}")
    full = _check_train(gpu_ctx, x, budget, msd=True, u16=u16, big=True)
    a, b = x.twins
    hit = full[(full["i"] == a) & (full["j"] == b)]
    assert len(hit) == 1 and int(hit["count"][0]) == twin
    assert geometry(x.db.n, True, budget)[1] == 2


@pytest.mark.parametrize("name,probe", [("n2^20+1_h55", False), ("n2^20+1_h54_small", True)])
def test_run_counts_past_2pow20(gpu_ctx, dbs, name, probe):
    """exclusive_hashes on run_path 1 and 0 against the numpy reference.  At width 55 the partition does not pack 21-bit
    ids, so run_path 1 falls back to the sort path; at width 54 without heavy hashes the bucket probe answers."""
    db = dbs(name).db
    rng = np.random.default_rng(11)
    gid = np.repeat(np.arange(db.n), db.sizes)
    present = rng.choice(db.n, size=2000, replace=False)
    take = np.isin(gid, present) & (rng.random(len(gid)) < 0.7)
    sample = np.concatenate([db.hashes[take], rng.integers(1, int(db.hashes.max()), size=50000, dtype=np.uint64)])
    gpu_ctx.load_sketches(db.hashes, db.offsets)
    for mask in (None, (rng.random(db.n) < 0.01).astype(np.uint8)):
        exp = ro.exclusive_counts_np(db.hashes, db.offsets, sample, mask)
        for path in (1, 0):
            gpu_ctx.set_option("run_path", path)
            try:
                gpu_ctx.reset_timers()
                got = gpu_ctx.exclusive_hashes(sample, mask)
                took_probe = gpu_ctx.timings()["ms_sample_kernels"] > 0.0
            finally:
                gpu_ctx.set_option("run_path", 1)
            print(f"{name} run_path={path} probe={took_probe}")
            assert took_probe == (probe and path == 1), (path, took_probe)
            for f in ("n_overlap", "nontrivial", "n_exclusive", "n_match"):
                assert np.array_equal(got[f], exp[f]), (path, f)


def test_sharded_step_past_2pow20(dbs):
    """Two ranks, both residencies, with no inline ids: every group travels as a posting stream.  The oversized-bucket
    variant is refused by the sharded step, so it runs replicated."""
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_sharded_step_gpu import _run_ranks
    for name, residencies in (("n2^20+1_h54_small", ("hashes", "genomes")), ("n2^20+1_h54_dup", ("replicated",))):
        db = dbs(name).db
        ref = to.oracle_train_sparse(db.hashes, db.offsets, THR)
        for residency in residencies:
            for st, pairs in _run_ranks(db, 2, THR, residency):
                assert (st["n_distinct"], st["n_singleton"], st["n_index"], st["n_postings"], st["n_increments"]) == \
                    (ref.n_distinct, ref.n_singleton, ref.n_index, ref.n_postings, ref.n_increments), residency
                assert _Pairs(pairs) == _Pairs(ref.pairs), (name, residency)


def test_get_option_rejects_unknown_names(gpu_ctx):
    with pytest.raises(_lib.YgpuError, match=r"\(-3\)"):
        gpu_ctx.get_option("count_kernel")
