"""K6 on the GPU (k6_hyp_test, k6_alt_mut_rate through ygpu_hyp_test / ygpu_alt_mut_rate) against scipy and the exact
reference oracle/binom_exact.py: dense threshold sweeps, exact ties, deep tails, large counts, the alternative mutation
rate on its own and degenerate parameters.  The checks and their acceptance rules are in tests/harness/k6_checks.py;
tests/test_binom_stats_exact.py runs the same checks on the host build of binom_stats.cuh."""
import numpy as np
import pytest

from harness import k6_checks as kc

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("k,sig,ani", kc.SWEEP_SETS)
def test_dense_threshold_sweep(gpu_ctx, k, sig, ani):
    kc.dense_sweep(gpu_ctx, k, sig, ani)


def test_exact_ties(gpu_ctx):
    n_ties, scipy_off = kc.check_ties(gpu_ctx)
    assert n_ties > 1000 and 0 < scipy_off < n_ties
    # how often the device's own fp64 cdf at the tie falls below q, i.e. how often the tie rule decided: for q >= 1/2,
    # 1 - confidence is that cdf exactly.  Which way a tie rounds depends on the code nvcc generates (it contracts to
    # FMA), so the count is reported, not asserted; the thresholds above are asserted whatever it is.
    below = 0
    by = {}
    for ani, k, s, n, kk in kc.exact_ties():
        if 1.0 - s >= 0.5:
            by.setdefault((ani, k, s), []).append((n, kk))
    for (ani, k, s), nks in by.items():
        rows = gpu_ctx.hyp_test([n for n, _ in nks], [kk for _, kk in nks], k, s, ani, [1.0])[0]
        below += int(np.count_nonzero(1.0 - rows["actual_confidence_with_coverage"] < 1.0 - s))
    print(f"{n_ties} exact ties; scipy resolves {scipy_off} differently; "
          f"the device's fp64 cdf falls below q at {below} of the ties with q >= 1/2")


def test_exact_tie_example(gpu_ctx):
    """ani 0.5, k 1, significance 0.5, n_c 5: cdf(2; 5, 1/2) = 1/2 = q exactly, so the threshold is 2 (scipy: 2) and the
    confidence 1/2.  The host build's fp64 cdf gives 0.49999999999999994 here, which without the tie rule meant a
    threshold of 3 and a confidence of 0.1875."""
    r = gpu_ctx.hyp_test([5], [2], 1, 0.5, 0.5, [1.0])[0, 0]
    assert r["acceptance_threshold_with_coverage"] == 2 and r["in_sample_est"] == 1
    assert abs(float(r["actual_confidence_with_coverage"]) - 0.5) <= 2.0 ** -52


def test_exact_tie_at_large_odd_n(gpu_ctx):
    """p = 1/2: cdf((n-1)/2) = 1/2 for every odd n, so the threshold at significance 1/2 is (n-1)/2."""
    ne = np.array([5, 4097, 10 ** 6 + 1, 718102475, 2 ** 31 + 1, 4 * 10 ** 9 + 1], np.int64)
    rows = gpu_ctx.hyp_test(ne, ne // 2, 1, 0.5, 0.5, [1.0])[0]
    assert np.array_equal(rows["acceptance_threshold_with_coverage"], (ne - 1) // 2)
    # one ulp above the tie (q = 1/2 + 2^-53) the answer moves up; decidable in fp64 only where n is small
    r = gpu_ctx.hyp_test([5], [2], 1, 0.5 - 2.0 ** -53, 0.5, [1.0])[0, 0]
    assert r["acceptance_threshold_with_coverage"] == 3


@pytest.mark.parametrize("k,sig,ani", [(31, .5, .95), (21, .01, .9)])
def test_own_cdf_as_q(gpu_ctx, k, sig, ani):
    assert kc.check_own_cdf_as_q(gpu_ctx, k, sig, ani, np.arange(1, 1500, 3)) > 400


def test_deep_tails(gpu_ctx):
    kc.check_deep_tails(gpu_ctx)


@pytest.mark.parametrize("k,sig,ani", [(31, .99, .95), (21, .999, .99)])
def test_large_counts(gpu_ctx, k, sig, ani):
    kc.check_large_counts(gpu_ctx, k, sig, ani)


@pytest.mark.parametrize("sig", kc.ALT_SIGS)
def test_alt_mut_rate(gpu_ctx, sig):
    kc.check_alt_mut_rate(gpu_ctx, sig)


def test_degenerate_parameters(gpu_ctx):
    assert kc.check_degenerate(gpu_ctx) == 960
