"""K6's arithmetic (yacht_b200/csrc/binom_stats.cuh) compiled for the host and checked against scipy and the exact
reference oracle/binom_exact.py -- the same checks tests/test_hyp_stats_exact_gpu.py runs on the CUDA kernels, so they
also run where there is no GPU.  tests/harness/stats_host_harness.cpp exports the header's functions and the bodies of
k6_hyp_test / k6_alt_mut_rate with the C ABI's signatures."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import binom_exact as be
from harness import k6_checks as kc
from yacht_b200._lib import HYP_ROW_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))


class HostK6:
    """The two ABI calls of GpuContext, evaluated by the host build of binom_stats.cuh."""

    def __init__(self, lib):
        self.lib = lib

    def hyp_test(self, n_exclusive, n_match, ksize, significance, ani_thresh, min_coverage):
        ne = np.ascontiguousarray(n_exclusive, dtype=np.int64)
        nm = np.ascontiguousarray(n_match, dtype=np.int64)
        cov = np.ascontiguousarray(min_coverage, dtype=np.float64)
        rows = np.zeros((cov.shape[0], ne.shape[0]), dtype=HYP_ROW_DTYPE)
        self.lib.sh_hyp_test(ne.ctypes.data, nm.ctypes.data, ne.shape[0], int(ksize), float(significance),
                             float(ani_thresh), cov.ctypes.data, cov.shape[0], rows.ctypes.data)
        return rows

    def alt_mut_rate(self, nu, thresh, ksize, significance=0.99):
        a = np.ascontiguousarray(nu, dtype=np.int64)
        b = np.ascontiguousarray(thresh, dtype=np.int64)
        out = np.zeros(a.shape[0], dtype=np.float64)
        self.lib.sh_alt_mut_rate(a.ctypes.data, b.ctypes.data, a.shape[0], int(ksize), float(significance),
                                 out.ctypes.data)
        return out


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("k6") / "libstats_host.so"
    src = os.path.join(HERE, "harness", "stats_host_harness.cpp")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-o", str(out), src], check=True)
    lib = ctypes.CDLL(str(out))
    d, vp, ll = ctypes.c_double, ctypes.c_void_p, ctypes.c_longlong
    for name in ("sh_binom_cdf", "sh_binom_ppf", "sh_betaincinv_int"):
        getattr(lib, name).argtypes = [d, d, d]
        getattr(lib, name).restype = d
    lib.sh_cdf_sf.argtypes = [d, d, d, vp]
    lib.sh_alt_mut_rate.argtypes = [vp, vp, ll, ctypes.c_int, d, vp]
    lib.sh_hyp_test.argtypes = [vp, vp, ll, ctypes.c_int, d, d, vp, ctypes.c_int, vp]
    return lib


@pytest.fixture(scope="module")
def host(host_lib):
    return HostK6(host_lib)


@pytest.mark.parametrize("k,sig,ani", kc.SWEEP_SETS)
def test_dense_threshold_sweep(host, k, sig, ani):
    kc.dense_sweep(host, k, sig, ani)


def test_exact_ties(host, host_lib):
    n_ties, scipy_off = kc.check_ties(host)
    assert n_ties > 1000 and 0 < scipy_off < n_ties
    # without the tie rule the fp64 cdf decides: it falls below q at many ties, e.g. cdf(2; 5, 1/2) = 1/2
    assert host_lib.sh_binom_cdf(2.0, 5.0, 0.5) < 0.5
    assert host_lib.sh_binom_ppf(0.5, 5.0, 0.5) == 2.0
    below = sum(host_lib.sh_binom_cdf(float(kk), float(n), ani ** k) < 1.0 - s for ani, k, s, n, kk in kc.exact_ties())
    assert below > 100
    print(f"{n_ties} exact ties; scipy resolves {scipy_off} differently; the fp64 cdf falls below q at {below}")


def test_exact_tie_at_large_odd_n(host_lib):
    """p = 1/2: cdf((n-1)/2) = 1/2 for every odd n, so ppf(1/2) = (n-1)/2."""
    for n in (5, 4097, 10 ** 6 + 1, 718102475, 2 ** 31 + 1, 4 * 10 ** 9 + 1):
        assert host_lib.sh_binom_ppf(0.5, float(n), 0.5) == (n - 1) // 2, n
    # one ulp above the tie the answer moves up; decidable in fp64 only where n is small
    assert host_lib.sh_binom_ppf(0.5 + 2.0 ** -53, 5.0, 0.5) == 3.0



@pytest.mark.parametrize("k,sig,ani", [(31, .5, .95), (21, .01, .9)])
def test_own_cdf_as_q(host, k, sig, ani):
    assert kc.check_own_cdf_as_q(host, k, sig, ani, np.arange(1, 1500, 3)) > 400


def test_deep_tails(host):
    kc.check_deep_tails(host)


@pytest.mark.parametrize("k,sig,ani", [(31, .99, .95), (21, .999, .99)])
def test_large_counts(host, k, sig, ani):
    kc.check_large_counts(host, k, sig, ani)


@pytest.mark.parametrize("sig", kc.ALT_SIGS)
def test_alt_mut_rate(host, sig):
    kc.check_alt_mut_rate(host, sig)


def test_degenerate_parameters(host):
    assert kc.check_degenerate(host) == 960


def test_cdf_against_exact(host_lib):
    """The fp64 cdf and sf within 1e-12 relative of the exact value on their summed side, from 1e-9 to 0.999 and +-40 sd."""
    out = (ctypes.c_double * 4)()
    for p in (0.204, 0.81, 1.14e-5, 0.989, 0.999, 0.5, 1e-9):
        for n in (10, 1000, 100000, 10 ** 7):
            mu, sd = n * p, (n * p * (1 - p)) ** 0.5
            for kk in sorted({int(min(max(mu + z * sd, 0), n - 1)) for z in (-40, -10, -3, -1, 0, 0.5, 1, 3, 10, 40)}):
                host_lib.sh_cdf_sf(float(kk), float(n), p, out)
                c, s = be.cdf_sf(kk, n, p)
                got, exact = (out[0], c) if out[3] else (out[1], s)
                assert abs(got - float(exact)) <= 1e-12 * float(exact) + kc.TINY, (p, n, kk, got, exact)


def test_scipy_restatement_matches_run_oracle():
    """k6_checks.scipy_rows is run_oracle.single_hyp_test, vectorised."""
    from oracle import run_oracle as ro
    ne = np.array([0, 1, 5, 100, 3741, 20000, 123457], np.int64)
    nm = np.array([0, 1, 2, 90, 2, 4000, 100000], np.int64)
    for k, sig, ani, cov in [(31, .99, .95, 1.0), (21, .01, .9, 0.5), (1, .5, .5, 1.5)]:
        nc, thr, conf, alt, pv, ins = kc.scipy_rows(ne, nm, k, sig, ani, cov)
        for i in range(ne.size):
            e = ro.single_hyp_test((int(ne[i]), int(nm[i])), k, sig, ani, cov)
            assert (bool(ins[i]), float(pv[i]), int(nc[i]), float(thr[i]), float(conf[i]), float(alt[i])) == \
                (e[0], e[1], e[3], e[5], e[6], e[7])
