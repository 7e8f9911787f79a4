"""GPU parity of the run hot path (K5 sample membership / exclusive hashes, K6 statistics).

Bars: integer outputs bit-exact; floating-point outputs within 1e-9 relative of the reference's
scipy values (sentinels 0 / 1 / -1 exact; subnormal p-values to the nearest representable value).
All calls go through the C ABI.
"""
import gzip
import json
import os

import numpy as np
import pytest

from oracle import run_oracle as ro
from yacht_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 1e-9   # north_star: "within a stated tolerance (e.g. 1e-9 relative)"


def test_hyp_test_matches_every_workbook_row(gpu_ctx):
    gold = json.loads(gzip.open(os.path.join(GOLD, "run_golden.json.gz"), "rb").read().decode())
    total = 0
    for book in gold["books"]:
        rows = book["rows"]
        covs = sorted({r[1] for r in rows}, reverse=True)
        by_cov = {c: [r for r in rows if r[1] == c] for c in covs}
        for cov, rs in by_cov.items():
            ne = np.array([r[0] for r in rs], dtype=np.int64)
            nm = np.array([r[2] for r in rs], dtype=np.int64)
            got = gpu_ctx.hyp_test(ne, nm, book["ksize"], book["significance"], book["ani_thresh"], [cov])[0]
            for g, r in zip(got, rs):
                _, _, _, nc, thr, conf, alt, p, ins, p_ok = r
                ctxt = f"{book['source']} {r} got {g}"
                assert int(g["num_exclusive_kmers_coverage"]) == nc, ctxt
                assert float(g["acceptance_threshold_with_coverage"]) == thr, ctxt
                assert bool(g["in_sample_est"]) == bool(ins), ctxt
                assert ro.float_close(float(g["actual_confidence_with_coverage"]), conf, REL_TOL), ctxt
                assert ro.float_close(float(g["alt_confidence_mut_rate_with_coverage"]), alt, REL_TOL), ctxt
                if p_ok:
                    assert ro.float_close(float(g["p_val"]), p, REL_TOL), ctxt
                total += 1
    assert total == 29457


def test_hyp_test_vs_scipy_random(gpu_ctx):
    rng = np.random.default_rng(5)
    ne = np.concatenate([rng.integers(0, 40, 60), rng.integers(40, 20000, 200), rng.integers(20000, 300000, 12)]).astype(np.int64)
    nm = (ne * rng.random(len(ne)) * rng.choice([0.0, 0.05, 0.3, 1.0, 1.2], len(ne))).astype(np.int64)
    for k, sig, ani in [(31, 0.99, 0.95), (21, 0.999, 0.9), (51, 0.95, 0.97)]:
        covs = [1.0, 0.6, 0.2, 0.1, 0.001]
        rows = gpu_ctx.hyp_test(ne, nm, k, sig, ani, covs)
        ro.assert_rows_close(rows, ne, nm, k, sig, ani, covs, REL_TOL)


def test_reference_known_answers_on_gpu(gpu_ctx):
    # the fixture known answer of reference tests/test_workflow.py:58-66 (values: SURVEY.md appendix B)
    rows = gpu_ctx.hyp_test([3741], [2], 31, 0.99, 0.95, [1.0, 0.001])
    r1, r2 = rows[0, 0], rows[1, 0]
    assert r1["acceptance_threshold_with_coverage"] == 706 and not r1["in_sample_est"]
    assert ro.float_close(float(r1["actual_confidence_with_coverage"]), 0.9893565463905609, REL_TOL)
    assert ro.float_close(float(r1["alt_confidence_mut_rate_with_coverage"]), 0.054795863080029594, REL_TOL)
    assert float(r1["p_val"]) < 1e-300
    assert r2["acceptance_threshold_with_coverage"] == 0 and r2["in_sample_est"] and r2["num_exclusive_kmers_coverage"] == 3
    assert ro.float_close(float(r2["p_val"]), 0.9915219633070561, REL_TOL)
    assert ro.float_close(float(r2["actual_confidence_with_coverage"]), 0.49546453317314254, REL_TOL)
    assert ro.float_close(float(r2["alt_confidence_mut_rate_with_coverage"]), 0.16796854767978497, REL_TOL)
    # n_c == 0 sentinels (thr 0, conf 0, alt -1, p 1)
    r0 = gpu_ctx.hyp_test([5, 3], [0, 2], 31, 0.99, 0.95, [0.1])[0]
    assert (int(r0[0]["num_exclusive_kmers_coverage"]), float(r0[0]["acceptance_threshold_with_coverage"]),
            float(r0[0]["actual_confidence_with_coverage"]), float(r0[0]["alt_confidence_mut_rate_with_coverage"]),
            float(r0[0]["p_val"]), int(r0[0]["in_sample_est"])) == (0, 0.0, 0.0, -1.0, 1.0, 0)
    assert r0[1]["in_sample_est"] == 1 and r0[1]["p_val"] == 1.0


def test_alt_mut_rate_reference_kats_on_gpu(gpu_ctx):
    # reference tests/test_unit.py:11-20: get_alt_mut_rate(nu, thresh, k).  Through the ABI the pair
    # (nu, thresh) arises as (n_c, binom.ppf(...)); choose significance/ani so that ppf == thresh.
    # (10, 0, k): any ani with ppf 0 -> alt = 1 - (1 - 0.99**(1/10)) ** (1/k)
    for k, exp in [(21, 0.28015945851802826), (31, 0.19963312102481723)]:
        row = gpu_ctx.hyp_test([10], [0], k, 0.99, 0.5, [1.0])[0, 0]
        assert row["acceptance_threshold_with_coverage"] == 0
        assert np.isclose(float(row["alt_confidence_mut_rate_with_coverage"]), exp)


COUNT_FIELDS = ("n_overlap", "nontrivial", "n_exclusive", "n_match")


def _check_counts(ctx, db, sample, mask=None, *, probe):
    """Both run paths against the set oracle: run_path 1 (the bucket probe of run_buckets.cuh, when the input qualifies) and
    run_path 0 (the general sort path).  `probe`: whether run_path 1 is expected to take the probe.  Which path answered is
    read from the timers: ms_sample_kernels grows only when the probe ran."""
    exp = ro.exclusive_counts(db.hashes, db.offsets, sample, mask)
    ctx.load_sketches(db.hashes, db.offsets)
    res = {}
    for path in (1, 0):
        ctx.set_option("run_path", path)
        try:
            ctx.reset_timers()
            got = ctx.exclusive_hashes(sample, mask)
            took_probe = ctx.timings()["ms_sample_kernels"] > 0.0
        finally:
            ctx.set_option("run_path", 1)
        assert took_probe == (probe and path == 1), f"run_path {path}: probe expected {probe and path == 1}, taken {took_probe}"
        for f in COUNT_FIELDS:
            assert np.array_equal(got[f], exp[f]), f"run_path {path}: {f}"
        res[path] = got
    return res[1]


def test_fixture20_known_answer(gpu_ctx):
    z = np.load(os.path.join(GOLD, "fixture20.npz"))
    db = synth.SketchDB(hashes=z["hashes"], offsets=z["offsets"], cluster=np.full(20, -1))
    got = _check_counts(gpu_ctx, db, z["sample_hashes"], probe=True)
    nt = np.flatnonzero(got["nontrivial"])
    assert len(nt) == 1 and str(z["names"][nt[0]]).startswith("CP032507.1")
    assert (int(got["n_exclusive"][nt[0]]), int(got["n_match"][nt[0]])) == (3741, 2)


@pytest.mark.parametrize("n,seed", [(300, 1), (1200, 2)])
def test_exclusive_counts_synthetic(gpu_ctx, n, seed):
    db = synth.make_reference_db(n, seed, mean_size=400, sd_size=100)
    sample, present, cov = synth.make_sample(db, seed + 100, n_present=n // 5, total_hashes=60000)
    got = _check_counts(gpu_ctx, db, sample, probe=True)
    # the sample shuffled, with every tenth hash three times: membership is a set question
    rng = np.random.default_rng(seed + 200)
    _check_counts(gpu_ctx, db, rng.permutation(np.concatenate([sample, np.repeat(sample[::10], 2)])), probe=True)
    # masks: nothing nontrivial, everything nontrivial, and only genomes that share no hash with the sample
    _check_counts(gpu_ctx, db, sample, mask=np.zeros(n, np.uint8), probe=True)
    _check_counts(gpu_ctx, db, sample, mask=np.ones(n, np.uint8), probe=True)
    none = (got["n_overlap"] == 0).astype(np.uint8)
    assert 0 < none.sum() < n
    _check_counts(gpu_ctx, db, sample, mask=none, probe=True)
    # also after the index has been built on the same context (shared sorted array)
    gpu_ctx.build_index()
    got = gpu_ctx.exclusive_hashes(sample)
    exp = ro.exclusive_counts(db.hashes, db.offsets, sample)
    assert np.array_equal(got["n_exclusive"], exp["n_exclusive"]) and np.array_equal(got["n_match"], exp["n_match"])


def test_exclusive_counts_edge_cases(gpu_ctx):
    parts = [np.array([1, 2, 3, 4], np.uint64), np.array([3, 4, 5, 5, 5], np.uint64), np.zeros(0, np.uint64),
             np.array([2**64 - 1, 7, 7], np.uint64), np.array([100, 200], np.uint64)]
    db = synth.from_sketches(parts)
    _check_counts(gpu_ctx, db, np.array([5, 7, 2**64 - 1, 3, 3, 999], dtype=np.uint64), probe=True)
    _check_counts(gpu_ctx, db, np.zeros(0, dtype=np.uint64), probe=True)                       # empty sample: nothing nontrivial
    _check_counts(gpu_ctx, db, np.array([424242], dtype=np.uint64), probe=True)                # no overlap at all
    _check_counts(gpu_ctx, db, np.array([1], dtype=np.uint64), mask=np.array([1, 1, 1, 0, 1], np.uint8), probe=True)  # explicit mask
    _check_counts(gpu_ctx, db, np.array([0, 1, 2**63], dtype=np.uint64), mask=np.ones(5, np.uint8), probe=True)
    _check_counts(gpu_ctx, db, np.array([7, 3, 100], dtype=np.uint64), mask=np.zeros(5, np.uint8), probe=True)   # nothing nontrivial
    # mask marking only genomes without overlap (0, 2, 4 share nothing with {7}): their hashes count as exclusive, no match
    _check_counts(gpu_ctx, db, np.array([7], dtype=np.uint64), mask=np.array([1, 0, 1, 0, 1], np.uint8), probe=True)


def test_exclusive_counts_small_edges(gpu_ctx):
    # one genome: the probe needs two (the partition packs genome ids beside the hash), so the sort path answers
    one = synth.from_sketches([np.array([1, 2, 3, 3, 9], np.uint64)])
    _check_counts(gpu_ctx, one, np.array([3, 9, 9, 11], dtype=np.uint64), probe=False)
    _check_counts(gpu_ctx, one, np.array([3], dtype=np.uint64), mask=np.zeros(1, np.uint8), probe=False)
    # every sketch empty (T = 0): no hash to hold, the mask alone decides what is nontrivial
    empty = synth.from_sketches([np.zeros(0, np.uint64)] * 3)
    _check_counts(gpu_ctx, empty, np.array([1, 2], dtype=np.uint64), probe=False)
    _check_counts(gpu_ctx, empty, np.array([1, 2], dtype=np.uint64), mask=np.ones(3, np.uint8), probe=False)
    # a 10-bit reference (largest hash 1000): 1010 and 1023 are above the largest hash but inside the hash width, 1024 and
    # 2^63 beyond it; the sample is shuffled and repeats hashes
    narrow = synth.from_sketches([np.array([1, 5, 900, 1000], np.uint64), np.array([5, 7, 7, 1000], np.uint64), np.zeros(0, np.uint64),
                                  np.array([3, 900, 950], np.uint64)])
    for sample in ([1010, 1023, 1024, 2**63, 5000], [7, 1010, 5, 7, 1024, 5, 3, 1023], [1000, 1000, 2**64 - 1]):
        _check_counts(gpu_ctx, narrow, np.array(sample, dtype=np.uint64), probe=True)
    _check_counts(gpu_ctx, narrow, np.array([1023, 1], dtype=np.uint64), mask=np.array([0, 1, 1, 1], np.uint8), probe=True)
