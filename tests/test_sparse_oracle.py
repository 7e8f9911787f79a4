"""The references of the large-N tests (tests/test_train_large_n_gpu.py) against the pinned ones (CPU only, no GPU needed).

* oracle_train_sparse (yo_train_sparse) against oracle_train (yo_train, pinned to the reference binary by
  tests/test_oracle_pinned.py) field for field: pairs, the three banner statistics, P, W and the greedy order, and its row
  ranges against the matching pairs of the whole.
* run_oracle.exclusive_counts_np against the set restatement run_oracle.exclusive_counts.
* the large-N generator plants what its tests rely on.
"""
import numpy as np
import pytest

from harness import large_n
from oracle import run_oracle as ro
from oracle import sketch_oracle as so
from oracle import train_oracle as to
from yacht_b200 import synth

THR = 0.95 ** 31


def _same(a, b, ctx=None):
    assert a.pairs.tobytes() == b.pairs.tobytes(), ctx
    assert (a.n_distinct, a.n_singleton, a.n_index, a.n_postings, a.n_increments) == \
        (b.n_distinct, b.n_singleton, b.n_index, b.n_postings, b.n_increments), ctx
    assert a.selected.tolist() == b.selected.tolist(), ctx


def _fuzz_db(rng):
    """The generator of test_random_small_databases: a small hash universe, so that ties, twins, subsets, in-sketch
    duplicates, empty sketches and thresholds exactly on a containment value all occur."""
    n = int(rng.integers(1, 14))
    universe = rng.integers(1, 2 ** 63, size=int(rng.integers(3, 40)), dtype=np.uint64)
    parts = []
    for g in range(n):
        k = int(rng.integers(0, min(len(universe), 12) + 1))
        s = rng.choice(universe, size=k, replace=False) if k else np.zeros(0, dtype=np.uint64)
        if k and rng.random() < 0.2:
            s = np.concatenate([s, s[: int(rng.integers(1, k + 1))]])
        if g and rng.random() < 0.25:
            src = parts[int(rng.integers(0, g))]
            s = src.copy() if rng.random() < 0.5 else src[: len(src) // 2]
        parts.append(np.asarray(s, dtype=np.uint64))
    sizes = [len(p) for p in parts if len(p)]
    thr = float(rng.choice([0.0, 1.0, 0.5, 1 / 3, THR] + ([1.0 * int(rng.integers(1, max(sizes) + 1)) / max(sizes)] if sizes else [])))
    return synth.from_sketches(parts), thr


def test_sparse_equals_dense_on_random_small_databases():
    rng = np.random.default_rng(20260103)
    for case in range(240):
        db, thr = _fuzz_db(rng)
        _same(to.oracle_train_sparse(db.hashes, db.offsets, thr), to.oracle_train(db.hashes, db.offsets, thr), (case, thr))


def test_sparse_equals_dense_on_edge_set():
    parts = [np.arange(1, 11), np.arange(1, 11), np.zeros(0), np.array([1, 2, 3, 4, 5] + list(range(100, 107))),
             np.array([7, 7, 7, 200])]
    db = synth.from_sketches([np.asarray(p, dtype=np.uint64) for p in parts])
    for thr in (0.0, 0.4, 0.5, 1.0, THR):
        _same(to.oracle_train_sparse(db.hashes, db.offsets, thr), to.oracle_train(db.hashes, db.offsets, thr), thr)
    empty = synth.from_sketches([])
    _same(to.oracle_train_sparse(empty.hashes, empty.offsets, 0.5), to.oracle_train(empty.hashes, empty.offsets, 0.5))


@pytest.mark.parametrize("n,seed,dups", [(800, 3, False), (3000, 9, False), (3000, 23, True)])
def test_sparse_equals_dense_on_synthetic(n, seed, dups):
    db = synth.make_reference_db(n, seed, mean_size=300, sd_size=100, min_size=20, core_hashes=4, core_lo=0.2, core_hi=0.5)
    if dups:
        parts = [db.sketch(g) for g in range(db.n)]
        for g in range(0, n, 7):
            parts[g] = np.concatenate([parts[g], parts[g][: 1 + g % 5]])
        db = synth.from_sketches(parts)
    for thr in (THR, 0.0, 0.5):
        dense = to.oracle_train(db.hashes, db.offsets, thr)
        _same(to.oracle_train_sparse(db.hashes, db.offsets, thr), dense, (n, thr))
        for lo, hi in [(0, 1), (n // 3, n // 3 + 57), (n - 5, n), (n, n)]:
            part = to.oracle_train_sparse(db.hashes, db.offsets, thr, lo, hi)
            low = np.minimum(dense.pairs["i"], dense.pairs["j"])     # pairwise_flag's range: the smaller genome's row
            rows = dense.pairs[(low >= lo) & (low < hi)]
            assert part.pairs.tobytes() == rows.tobytes(), (thr, lo, hi)


def test_sparse_rejects_bad_row_range():
    db = synth.make_reference_db(50, 1, mean_size=30, sd_size=5)
    with pytest.raises(RuntimeError):
        to.oracle_train_sparse(db.hashes, db.offsets, THR, 10, 5)
    with pytest.raises(RuntimeError):
        to.oracle_train_sparse(db.hashes, db.offsets, THR, 0, 51)


@pytest.mark.parametrize("n,seed", [(300, 1), (1200, 2)])
def test_numpy_run_reference_equals_set_restatement(n, seed):
    db = synth.make_reference_db(n, seed, mean_size=200, sd_size=60)
    parts = [db.sketch(g) for g in range(db.n)]
    parts[4] = np.concatenate([parts[4], parts[4][:9]])          # in-sketch duplicates count once
    parts[9] = np.zeros(0, dtype=np.uint64)
    db = synth.from_sketches(parts)
    sample, _, _ = synth.make_sample(db, seed + 100, n_present=n // 5, total_hashes=20000)
    rng = np.random.default_rng(seed)
    for s, mask in [(sample, None), (np.concatenate([sample, sample[::10]]), None), (sample, np.zeros(n, np.uint8)),
                    (sample, np.ones(n, np.uint8)), (sample, (rng.random(n) < 0.3).astype(np.uint8)),
                    (np.zeros(0, np.uint64), None)]:
        exp = ro.exclusive_counts(db.hashes, db.offsets, s, mask)
        got = ro.exclusive_counts_np(db.hashes, db.offsets, s, mask)
        for f in ("n_overlap", "nontrivial", "n_exclusive", "n_match"):
            assert np.array_equal(got[f], exp[f]), f


def test_large_n_generator_plants_its_edges():
    """At a small N the generator's promises can be checked with the dense reference too."""
    n, w = 100000, 45000
    x = large_n.make_large_db(n, so.max_hash_for_scaled(1000), 5, dup=True, tile_ws=(w,))
    db = x.db
    assert int(db.hashes.max()).bit_length() == 55
    sizes = db.sizes
    assert sizes[n // 3] == 0
    assert x.wide_rows == [3, w + 3]
    for r in x.wide_rows:                                         # > 4 096 distinct columns above r inside r's column tile
        p = to.oracle_train_sparse(db.hashes, db.offsets, 0.0, r, r + 1).pairs
        j = p["j"][p["i"] == r]
        assert np.count_nonzero((j > r) & (j // w == r // w)) > 4096
    lens = {len(g) for g in x.groups}
    assert {2, 3, 4, 5, 65, 66} <= lens
    assert len(x.big_members) == large_n.BIG_HOLDERS
    # every special id follows 0, 1, 2 smaller members in some planted group (where that many smaller ids exist)
    for s in large_n.special_ids(n):
        for e in range(3):
            if s >= e + 1:
                assert any(len(g) > e + 1 and g[e + 1] == s for g in x.groups), (s, e)
    t = large_n.make_large_db(5000, so.max_hash_for_scaled(1000), 6, wide=False, big=False, twin=65535)
    a, b = t.twins
    assert t.db.sizes[a] == t.db.sizes[b] == 65535 and np.array_equal(t.db.sketch(a), t.db.sketch(b))
