"""Checks of the K6 statistics (yacht_b200/csrc/binom_stats.cuh) against scipy and the exact reference
(oracle/binom_exact.py), shared by tests/test_binom_stats_exact.py (the header compiled for the host) and
tests/test_hyp_stats_exact_gpu.py (the CUDA kernels through the C ABI).

`ev` is anything with the two ABI calls of yacht_b200._lib.GpuContext:
    ev.hyp_test(n_exclusive, n_match, ksize, significance, ani_thresh, min_coverage) -> rows[c, r] (HYP_ROW_DTYPE)
    ev.alt_mut_rate(nu, thresh, ksize, significance) -> float64[n]

Acceptance rules (DESIGN.md, K6):
  * thresholds equal scipy's; where they differ, the kernel's equals the exact ppf, or every cdf(k) >= q decision
    that separates the two answers lies in the ambiguity band (binom_exact.ambiguity_band);
  * exact ties cdf(k) == q resolve as cdf >= q;
  * confidence and p-value within 1e-9 relative of scipy (both below 1e-250 counts as equal: scipy underflows there),
    and within 1e-9 * max(|exact|, 2^-1022) of the exact value;
  * the alternative mutation rate within 1e-9 * |exp| + 4 * 2^-52 * c of scipy and of the exact value: it is formed as
    1 - pow(1 - x, 1/k) from an x with an absolute error of about ulp(1), and c (close_alt) is how much that pow
    amplifies it; the -1 sentinel exactly.
"""
from __future__ import annotations

import functools
import math
from fractions import Fraction

import numpy as np
from scipy.special import betaincinv
from scipy.stats import binom

from oracle import binom_exact as be
from oracle import run_oracle as ro

TINY = 2.0 ** -1022
ALT_ABS = 4 * 2.0 ** -52

SWEEP_SETS = [(31, .99, .95), (21, .999, .99), (51, .95, .8), (11, .99, .999), (15, .99, .9999), (31, .5, .95),
              (21, .01, .9), (1, .5, .5)]
SWEEP_N = np.concatenate([np.arange(20000), np.unique(np.geomspace(20000, 4e9, 200).astype(np.int64))]).astype(np.int64)
LARGE_N = [10 ** 5, 10 ** 6, 10 ** 7, 10 ** 8, 2 ** 31 - 1, 2 ** 31 + 1, 4 * 10 ** 9]


# ---- scipy, vectorised: the formulas of run_oracle.single_hyp_test / get_alt_mut_rate -------------------------------

def scipy_alt(nu, thresh, k, sig):
    with np.errstate(all="ignore"):
        x = betaincinv(np.asarray(nu, float) - thresh, 1.0 + np.asarray(thresh, float), sig)
        mut = 1 - (1 - x) ** (1 / k)
    return np.where(np.isnan(mut), -1.0, mut)


def scipy_rows(ne, nm, k, sig, ani, cov):
    """(n_c, thr, conf, alt, p_val, in_sample) as arrays."""
    ne, nm = np.asarray(ne, np.int64), np.asarray(nm, np.int64)
    p0 = ani ** k
    nc = (ne.astype(np.float64) * cov).astype(np.int64)
    with np.errstate(all="ignore"):
        thr = binom.ppf(1 - sig, nc, p0)
        conf = 1 - binom.cdf(thr, nc, p0)
        pv = np.where(nm <= nc, binom.cdf(nm, nc, p0), 1.0)
    return nc, thr, conf, scipy_alt(nc, thr, k, sig), pv, (nm >= thr) & (nm != 0)


def close_scipy(a, b, rel=ro.REL_TOL):
    """run_oracle.float_close, vectorised."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    return (a == b) | (np.isnan(a) & np.isnan(b)) | ((np.abs(a) < ro.UNDERFLOW_FLOOR) & (np.abs(b) < ro.UNDERFLOW_FLOOR)) \
        | (np.abs(a - b) <= rel * np.abs(b))


def close_exact(got: float, exact) -> bool:
    return abs(got - float(exact)) <= 1e-9 * max(abs(float(exact)), TINY)


def close_alt(got, exp, k):
    """|got - exp| <= 1e-9 |exp| + 4 ulp(1) * c, the -1 sentinel exactly.  c = max(1, d(1 - w^(1/k))/dw), w = 1 - x:
    x = betaincinv(...) carries an absolute error of an ulp(1) or so, which 1 - (1 - x)^(1/k) amplifies by c where
    w is tiny (thresh = 0 at large nu: w ~ 1e-9, c ~ 1e7 at k = 51)."""
    got, exp = np.asarray(got, float), np.asarray(exp, float)
    sentinel = (exp == -1.0) | (got == -1.0)
    with np.errstate(all="ignore"):
        w = (1 - exp) ** k
        c = np.where(w > 0, np.maximum(1.0, (1 - exp) / (k * w)), np.inf)
    return np.where(sentinel, got == exp, np.abs(got - exp) <= 1e-9 * np.abs(exp) + ALT_ABS * c)


def exact_conf(thr: int, n: int, p: float):
    return be.cdf_sf(int(thr), int(n), p)[1]


def exact_alt(n: int, thr: int, k: int, sig: float) -> float:
    return be.alt_mut_rate(int(n), int(thr), k, sig)


# ---- checks --------------------------------------------------------------------------------------------------------

def check_rows(rows, ne, nm, k, sig, ani, cov, what=""):
    """One hyp_test result (rows for one coverage) against scipy; disagreements adjudicated by the exact reference.
    Returns the number of thresholds that differ from scipy's (all of them acceptable)."""
    ne, nm = np.asarray(ne, np.int64), np.asarray(nm, np.int64)
    p0 = ani ** k
    q = 1 - sig
    nc, thr, conf, alt, pv, ins = scipy_rows(ne, nm, k, sig, ani, cov)
    g_thr = rows["acceptance_threshold_with_coverage"].astype(float)
    ctx = lambda i: (f"{what} k={k} sig={sig} ani={ani} cov={cov} n_excl={ne[i]} n_c={nc[i]} m={nm[i]}: "  # noqa: E731
                     f"got {rows[i]} scipy thr={thr[i]} conf={conf[i]!r} alt={alt[i]!r} p={pv[i]!r}")
    assert np.array_equal(rows["num_exclusive_kmers"], ne) and np.array_equal(rows["num_matches"], nm), what
    bad = np.flatnonzero(rows["num_exclusive_kmers_coverage"] != nc)
    assert bad.size == 0, ctx(bad[0])
    differ = np.flatnonzero(g_thr != thr)
    for i in differ:
        exact = be.ppf(q, int(nc[i]), p0, int(g_thr[i]))
        assert be.ppf_acceptable(int(g_thr[i]), q, int(nc[i]), p0, exact), ctx(i) + f" exact ppf {exact}"
    if differ.size:   # the downstream outputs follow the kernel's threshold: compare them with scipy at that threshold
        d_nc = nc[differ]
        with np.errstate(all="ignore"):
            conf[differ] = 1 - binom.cdf(g_thr[differ], d_nc, p0)
        alt[differ] = scipy_alt(d_nc, g_thr[differ], k, sig)
        ins[differ] = (nm[differ] >= g_thr[differ]) & (nm[differ] != 0)
    bad = np.flatnonzero(rows["in_sample_est"].astype(bool) != ins)
    assert bad.size == 0, ctx(bad[0])
    g_conf, g_pv = rows["actual_confidence_with_coverage"], rows["p_val"]
    g_alt = rows["alt_confidence_mut_rate_with_coverage"]
    for i in np.flatnonzero(~close_scipy(g_conf, conf)):
        assert close_exact(float(g_conf[i]), exact_conf(g_thr[i], nc[i], p0)), ctx(i)
    for i in np.flatnonzero(~close_scipy(g_pv, pv)):
        assert nm[i] <= nc[i] and close_exact(float(g_pv[i]), be.cdf(int(nm[i]), int(nc[i]), p0)), ctx(i)
    for i in np.flatnonzero(~close_alt(g_alt, alt, k)):
        assert close_alt(g_alt[i], exact_alt(nc[i], g_thr[i], k, sig), k), ctx(i) + f" exact alt {exact_alt(nc[i], g_thr[i], k, sig)!r}"
    return int(differ.size)


def dense_sweep(ev, k, sig, ani):
    """Returns the number of thresholds that differ from scipy's."""
    nm = (SWEEP_N.astype(np.float64) * (ani ** k)).astype(np.int64)
    rows = ev.hyp_test(SWEEP_N, nm, k, sig, ani, [1.0])[0]
    return check_rows(rows, SWEEP_N, nm, k, sig, ani, 1.0, "sweep")


@functools.lru_cache(maxsize=None)
def exact_ties(nmax: int = 60):
    """Every (ani, k, significance, n, kk) with ani in {.5, .75, .25}, k in {1, 2, 3}, n <= nmax and an exact tie
    cdf(kk; n, ani**k) == 1 - significance, for the double significances whose q = 1 - significance is that cdf."""
    out = []
    for ani in (0.5, 0.75, 0.25):
        for k in (1, 2, 3):
            p0 = ani ** k
            pf = Fraction(p0)
            for n in range(1, nmax + 1):
                c = Fraction(0)
                for kk in range(n):
                    c += math.comb(n, kk) * pf ** kk * (1 - pf) ** (n - kk)
                    qd = float(c)
                    if Fraction(qd) != c:
                        continue
                    sig = 1.0 - qd
                    for s in {sig, math.nextafter(sig, 0.0), math.nextafter(sig, 1.0)}:
                        if 0.0 < s < 1.0 and 1.0 - s == qd:
                            out.append((ani, k, s, n, kk))
    return tuple(sorted(set(out)))


def check_ties(ev):
    """Thresholds at exact ties equal the exact answer kk (cdf(kk) == q >= q).  Returns (ties, ties scipy resolves
    differently)."""
    ties = exact_ties()
    by = {}
    for ani, k, s, n, kk in ties:
        by.setdefault((ani, k, s), []).append((n, kk))
    scipy_off = 0
    for (ani, k, s), nks in by.items():
        ns = np.array([a for a, _ in nks], np.int64)
        kks = np.array([b for _, b in nks], np.int64)
        rows = ev.hyp_test(ns, kks, k, s, ani, [1.0])[0]
        thr = rows["acceptance_threshold_with_coverage"]
        bad = np.flatnonzero(thr != kks)
        assert bad.size == 0, f"ani={ani} k={k} sig={s!r} n={ns[bad[0]]}: threshold {thr[bad[0]]}, exact tie at {kks[bad[0]]}"
        assert np.array_equal(rows["in_sample_est"].astype(bool), kks != 0)
        scipy_off += int(np.count_nonzero(binom.ppf(1 - s, ns, ani ** k) != kks))
        # ppf stays non-decreasing in q (non-increasing in significance) across the tie
        sigs = [s]
        for _ in range(3):
            sigs = [math.nextafter(sigs[0], 0.0)] + sigs + [math.nextafter(sigs[-1], 1.0)]
        ts = np.stack([ev.hyp_test(ns, kks, k, x, ani, [1.0])[0]["acceptance_threshold_with_coverage"] for x in sigs])
        assert np.all(np.diff(ts, axis=0) <= 0), f"ani={ani} k={k} sig={s!r}: threshold not monotone in significance"
    return len(ties), scipy_off


def check_own_cdf_as_q(ev, k, sig, ani, ns):
    """ppf is the smallest k with cdf(k) >= q in the kernel's own arithmetic: with q set to the fp64 cdf at a threshold,
    the same threshold comes back.  For a cdf c >= 1/2, 1 - c is exact, so c = 1 - confidence and significance =
    confidence gives q = c exactly."""
    ns = np.asarray(ns, np.int64)
    first = ev.hyp_test(ns, np.zeros_like(ns), k, sig, ani, [1.0])[0]
    checked = 0
    for n, r in zip(ns, first):
        conf = float(r["actual_confidence_with_coverage"])
        if not 0.0 < conf <= 0.5:
            continue
        again = ev.hyp_test([n], [0], k, conf, ani, [1.0])[0, 0]
        assert again["acceptance_threshold_with_coverage"] == r["acceptance_threshold_with_coverage"], (n, conf, again, r)
        checked += 1
    return checked


def deep_tail_cases():
    """(k, ani, n_c, n_match list) with exact p-values from ~1e-190 through the subnormals to underflow."""
    out = []
    for k, ani, n in [(31, .95, 3243), (31, .95, 100000), (21, .99, 2000), (11, .999, 10 ** 6)]:
        p0 = ani ** k
        lo, hi = 0, int(n * p0)
        # smallest m with p-value > 1e-190, then walk down until the exact value is below 1e-330
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if be.cdf(mid, n, p0) > 1e-190:
                hi = mid
            else:
                lo = mid
        ms = []
        m = hi
        while m >= 0:
            ms.append(m)
            if be.cdf(m, n, p0) < be.mpmath.mpf("1e-330"):
                break
            m -= 1 if hi - m < 40 or m % 7 == 0 else 7
        out.append((k, ani, n, sorted(ms)))
    return out


def check_deep_tails(ev):
    seen_sub = seen_zero = 0
    for k, ani, n, ms in deep_tail_cases():
        p0 = ani ** k
        nm = np.array(ms, np.int64)
        rows = ev.hyp_test(np.full(nm.size, n, np.int64), nm, k, 0.99, ani, [1.0])[0]
        for m, g in zip(ms, rows["p_val"]):
            e = be.cdf(m, n, p0)
            assert close_exact(float(g), e), f"k={k} ani={ani} n_c={n} m={m}: p {g!r}, exact {e}"
            seen_sub += 0 < float(e) < TINY
            seen_zero += float(e) == 0.0
    assert seen_sub > 0 and seen_zero > 0


def check_large_counts(ev, k, sig, ani):
    ne = np.array(LARGE_N, np.int64)
    p0 = ani ** k
    for cov in (1.0, 1.5, 1e-9):
        first = ev.hyp_test(ne, np.zeros_like(ne), k, sig, ani, [cov])[0]
        check_rows(first, ne, np.zeros_like(ne), k, sig, ani, cov, "large")
        thr = first["acceptance_threshold_with_coverage"].astype(np.int64)
        nc = first["num_exclusive_kmers_coverage"]
        for i in range(ne.size):   # confidence against the exact value whatever scipy says
            assert close_exact(float(first["actual_confidence_with_coverage"][i]), exact_conf(thr[i], nc[i], p0)), (cov, ne[i])
        for d in (-1, 0, 1):
            nm = np.maximum(thr + d, 0)
            rows = ev.hyp_test(ne, nm, k, sig, ani, [cov])[0]
            check_rows(rows, ne, nm, k, sig, ani, cov, f"large thr{d:+d}")
            assert np.array_equal(rows["in_sample_est"].astype(bool), (nm >= thr) & (nm != 0))
            for i in range(ne.size):
                if nm[i] <= nc[i]:
                    assert close_exact(float(rows["p_val"][i]), be.cdf(int(nm[i]), int(nc[i]), p0)), (cov, ne[i], nm[i])


ALT_SIGS = (0.99, 0.95, 0.5, 0.999999, 0.01)
ALT_KS = (1, 21, 31, 51)
ALT_BIG_NU = (300, 1000, 10 ** 4, 10 ** 5, 10 ** 6, 10 ** 7)


def alt_grid():
    nu, th = [], []
    for n in range(300):
        nu += [n] * (n + 3)
        th += list(range(-1, n + 2))
    for n in ALT_BIG_NU:
        t = sorted({0, 1, n // 2, n - 2, n - 1, n, n + 1})
        nu += [n] * len(t)
        th += t
    return np.array(nu, np.int64), np.array(th, np.int64)


def check_alt_mut_rate(ev, sig):
    nu, th = alt_grid()
    exact_pick = np.flatnonzero((nu <= 24) | (nu >= 300))
    exact_x = {}
    for k in ALT_KS:
        got = ev.alt_mut_rate(nu, th, k, sig)
        exp = scipy_alt(nu, th, k, sig)
        sentinel = (th < 0) | (th >= nu)
        assert np.all(got[sentinel] == -1.0), "the -1 sentinel for thresh = -1 or thresh >= nu"
        bad = np.flatnonzero(~close_alt(got, exp, k))
        assert bad.size == 0, f"k={k} sig={sig} nu={nu[bad[0]]} thresh={th[bad[0]]}: got {got[bad[0]]!r} scipy {exp[bad[0]]!r}"
        for i in exact_pick:
            if sentinel[i]:
                continue
            key = (int(nu[i]), int(th[i]))
            if key not in exact_x:
                exact_x[key] = be.betaincinv_int(key[0], key[1], sig)
            e = float(1 - (1 - exact_x[key]) ** (be.mpmath.mpf(1) / k))
            assert close_alt(got[i], e, k), f"k={k} sig={sig} nu={key[0]} thresh={key[1]}: got {got[i]!r} exact {e!r}"


def check_degenerate(ev):
    """Significance 0 and 1, ani 0 and 1, n_c = 0: every output equal to run_oracle.single_hyp_test's."""
    pairs = [(0, 0), (1, 0), (1, 1), (2, 1), (10, 10), (10, 11), (1000, 0), (1000, 999), (1000, 1000), (123457, 100000)]
    ne = np.array([a for a, _ in pairs], np.int64)
    nm = np.array([b for _, b in pairs], np.int64)
    covs = [1.0, 0.5, 1.5, 1e-9]
    n = 0
    for sig in (0.0, 1.0, 0.5, 0.99):
        for ani in (0.0, 1.0, 0.95):
            for k in (1, 31):
                rows = ev.hyp_test(ne, nm, k, sig, ani, covs)
                for c, cov in enumerate(covs):
                    for r in range(ne.size):
                        e = ro.single_hyp_test((int(ne[r]), int(nm[r])), k, sig, ani, cov)
                        g = rows[c, r]
                        ctx = f"sig={sig} ani={ani} k={k} cov={cov} ({ne[r]}, {nm[r]}): got {g} exp {e}"
                        assert (bool(g["in_sample_est"]), int(g["num_exclusive_kmers_coverage"]),
                                float(g["acceptance_threshold_with_coverage"])) == (e[0], e[3], e[5]), ctx
                        assert ro.float_close(float(g["p_val"]), e[1]), ctx
                        assert ro.float_close(float(g["actual_confidence_with_coverage"]), e[6]), ctx
                        assert close_alt(float(g["alt_confidence_mut_rate_with_coverage"]), e[7], k), ctx
                        n += 1
    return n
