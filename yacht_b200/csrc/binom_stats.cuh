// binom_stats.cuh -- fp64 binomial statistics for the hypothesis test of `yacht run` (K6).
//
// Reference behaviour (KoslickiLab/YACHT src/yacht/hypothesis_recovery_src.py):
//   single_hyp_test  :233-306   thr  = binom.ppf(1 - significance, n_c, p0)
//                               conf = 1 - binom.cdf(thr, n_c, p0)
//                               p    = binom.cdf(m, n_c, p0) if m <= n_c else 1.0
//   get_alt_mut_rate :209-230   1 - (1 - betaincinv(n_c - thr, 1 + thr, significance))**(1/k); NaN -> -1
// There the numbers come from scipy, i.e. Boost.Math's incomplete-beta code.  That code is not
// restated here; the same mathematical quantities are evaluated with a different method that
// suits one GPU thread per (genome, coverage) pair:
//   * log pmf by the saddle-point expansion (Loader 2000: Stirling-error term + deviance terms),
//     accurate to ~1e-15 relative in the exponent;
//   * cdf as a one-sided sum of pmf ratios started at the boundary term and running AWAY from the
//     mode (every ratio < 1, geometric convergence, no cancellation); the side that is < 1/2 is
//     summed, the other is its complement -- the same choice an incomplete-beta evaluation makes;
//   * ppf as "the smallest k with cdf(k) >= q" (SURVEY.md appendix B: equals scipy's binom.ppf),
//     exact ties cdf(k) == q settled as >= (see cdf_ge_tie);
//   * betaincinv(n-k, k+1, y) through the identity I_x(n-k, k+1) = P[Bin(n, 1-x) <= k], solved
//     for w = 1-x by safeguarded Newton iterations on the log of the small tail.
// Target: integers exact, floats within 1e-9 relative of scipy (tests/test_run_parity_gpu.py).
//
// The functions are __host__ __device__ so the arithmetic can be exercised by a g++-compiled
// harness during development; the product only ever calls them from the CUDA kernel k6_hyp_test.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define YS_HD __host__ __device__ __forceinline__
#else
#define YS_HD inline
#endif

namespace ystats {

// ln(n!) - [(n + 1/2) ln n - n + ln(2 pi)/2] for integer n >= 0
YS_HD double stirlerr(double n) {
    const double sfe[16] = {
        0.0,
        0.0810614667953272582196702635943823601386, 0.0413406959554092940938220814071175080254,
        0.0276779256849983391487892927462446665954, 0.0207906721037650931115227717678486563331,
        0.0166446911898211921631948653735933911474, 0.0138761288230707479987457270237629085617,
        0.0118967099458917700950557241176594386201, 0.0104112652619720964974785671325346291995,
        0.0092554621827127329177286366331001361174, 0.0083305634333628712564693186596285522093,
        0.0075736754879518407949720242115950838929, 0.0069428401072095298656641526634753626599,
        0.0064089941880042070684396310829783125752, 0.0059513701127588477356244160464694583264,
        0.0055547335519628013710386899597922846491};
    if (n < 16.0) return sfe[(int)n];
    const double nn = n * n;
    // 1/(12n) - 1/(360n^3) + 1/(1260n^5) - 1/(1680n^7) + 1/(1188n^9)
    return (1.0 / 12.0 - (1.0 / 360.0 - (1.0 / 1260.0 - (1.0 / 1680.0 - (1.0 / 1188.0) / nn) / nn) / nn) / nn) / n;
}

// deviance part: x ln(x/np) + np - x, without cancellation when x ~ np
YS_HD double bd0(double x, double np) {
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        double ej = 2.0 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; j++) {
            ej *= v;
            const double s1 = s + ej / (double)(2 * j + 1);
            if (s1 == s) return s1;
            s = s1;
        }
        return s;
    }
    return x * log(x / np) + np - x;
}

// ln P[Bin(n, p) = x], 0 <= x <= n, 0 < p < 1
YS_HD double log_pmf(double x, double n, double p) {
    const double q = 1.0 - p;
    if (x == 0.0) return n * log1p(-p);
    if (x == n) return n * log(p);
    const double lc = stirlerr(n) - stirlerr(x) - stirlerr(n - x) - bd0(x, n * p) - bd0(n - x, n * q);
    // 0.5 * ln(n / (2 pi x (n - x)))
    return lc + 0.5 * log(n / (6.283185307179586476925286766559 * x * (n - x)));
}

// sum_{i <= k} pmf(i) / pmf(k): 1 + r_k + r_k r_{k-1} + ...,  r_i = pmf(i-1)/pmf(i) = i q / ((n-i+1) p)
YS_HD double ratio_sum_down(double k, double n, double p) {
    const double qp = (1.0 - p) / p;
    double term = 1.0, sum = 1.0;
    for (double i = k; i >= 1.0; i -= 1.0) {
        term *= i * qp / (n - i + 1.0);
        sum += term;
        if (term < sum * 1e-18 && i * qp < (n - i + 1.0)) break;
    }
    return sum;
}

// sum_{i >= k} pmf(i) / pmf(k): 1 + u_k + u_k u_{k+1} + ...,  u_i = pmf(i+1)/pmf(i) = (n-i) p / ((i+1) q)
YS_HD double ratio_sum_up(double k, double n, double p) {
    const double pq = p / (1.0 - p);
    double term = 1.0, sum = 1.0;
    for (double i = k; i < n; i += 1.0) {
        term *= (n - i) * pq / (i + 1.0);
        sum += term;
        if (term < sum * 1e-18 && (n - i) * pq < (i + 1.0)) break;
    }
    return sum;
}

// cdf = P[X <= k], sf = P[X > k] for X ~ Bin(n, p); the smaller one is summed directly.
// log_small receives ln(min(cdf, sf)) (usable when that side underflows), lower_side says which.
YS_HD void cdf_sf(double k, double n, double p, double* cdf, double* sf, double* log_small, bool* lower_side) {
    if (k < 0.0) { *cdf = 0.0; *sf = 1.0; if (log_small) *log_small = -INFINITY; if (lower_side) *lower_side = true; return; }
    if (k >= n) { *cdf = 1.0; *sf = 0.0; if (log_small) *log_small = -INFINITY; if (lower_side) *lower_side = false; return; }
    if (p <= 0.0) { *cdf = 1.0; *sf = 0.0; if (log_small) *log_small = -INFINITY; if (lower_side) *lower_side = false; return; }
    if (p >= 1.0) { *cdf = 0.0; *sf = 1.0; if (log_small) *log_small = -INFINITY; if (lower_side) *lower_side = true; return; }
    const double mode_edge = (n + 1.0) * p;
    if (k + 1.0 <= mode_edge) {
        // k is left of the mode: the lower tail is the small side
        const double l = log_pmf(k, n, p) + log(ratio_sum_down(k, n, p));
        const double c = exp(l);
        *cdf = c; *sf = 1.0 - c;
        if (log_small) *log_small = l;
        if (lower_side) *lower_side = true;
    } else {
        const double l = log_pmf(k + 1.0, n, p) + log(ratio_sum_up(k + 1.0, n, p));
        const double s = exp(l);
        *sf = s; *cdf = 1.0 - s;
        if (log_small) *log_small = l;
        if (lower_side) *lower_side = false;
    }
}

YS_HD double binom_cdf(double k, double n, double p) {
    double c, s;
    cdf_sf(k, n, p, &c, &s, nullptr, nullptr);
    return c;
}

// standard normal quantile (Acklam's rational approximation, ~1e-9): only an initial guess
YS_HD double norm_ppf_guess(double p) {
    const double a[6] = {-3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02,
                         1.383577518672690e+02, -3.066479806614716e+01, 2.506628277459239e+00};
    const double b[5] = {-5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02,
                         6.680131188771972e+01, -1.328068155288572e+01};
    const double c[6] = {-7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00,
                         -2.549732539343734e+00, 4.374664141464968e+00, 2.938163982698783e+00};
    const double d[4] = {7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00, 3.754408661907416e+00};
    if (p <= 0.0) return -40.0;
    if (p >= 1.0) return 40.0;
    if (p < 0.02425) {
        const double q = sqrt(-2.0 * log(p));
        return (((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
               ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1.0);
    }
    if (p > 1.0 - 0.02425) {
        const double q = sqrt(-2.0 * log(1.0 - p));
        return -(((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
               ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1.0);
    }
    const double q = p - 0.5, r = q * q;
    return (((((a[0] * r + a[1]) * r + a[2]) * r + a[3]) * r + a[4]) * r + a[5]) * q /
           (((((b[0] * r + b[1]) * r + b[2]) * r + b[3]) * r + b[4]) * r + 1.0);
}

// ---- exact ties cdf(k) == q --------------------------------------------------------------------
// cdf(k) can equal a double q exactly only when p has few significant bits (p = a / 2^m, so the cdf is a
// dyadic rational) and n is small -- or, for p = 1/2 and any odd n, at k = (n - 1) / 2 where it is 1/2 by
// symmetry.  The fp64 cdf above is good to ~1e-15 relative and rounds such a tie to either side, so
// binom_ppf re-decides the comparison that fixed its answer with the sum below, in double-double.
struct DD { double hi, lo; };
YS_HD DD dd_two_sum(double a, double b) { const double s = a + b, bb = s - a; return {s, (a - (s - bb)) + (b - bb)}; }
YS_HD DD dd_add(DD a, DD b) { DD s = dd_two_sum(a.hi, b.hi); s.lo += a.lo + b.lo; return dd_two_sum(s.hi, s.lo); }
YS_HD DD dd_mul(DD a, double b) { const double h = a.hi * b; return dd_two_sum(h, fma(a.hi, b, -h) + a.lo * b); }
YS_HD DD dd_div(DD a, double b) {
    const double q1 = a.hi / b, h = q1 * b;
    const double r = ((a.hi - h) - fma(q1, b, -h)) + a.lo;   // a - q1 b, exactly up to a.lo's rounding
    return dd_two_sum(q1, r / b);
}

constexpr double TIE_NMAX = 4096.0;

// whether cdf(k; n, p) == q is possible for a double q: p a multiple of 2^-32, and n small (or p = 1/2)
YS_HD bool tie_possible(double n, double p) {
    const double s = p * 4294967296.0;
    return s == floor(s) && (n <= TIE_NMAX || p == 0.5);
}

// P[Bin(n, p) <= k] >= q, settled to ~1e-27 and counting a cdf within that of q as equal (ties -> true).
// For tie_possible(n, p) with n <= TIE_NMAX only: (n - i + 1) p and i (1 - p) are then exact doubles.
YS_HD bool cdf_ge_tie(double k, double n, double p, double q) {
    // t_i = C(n, i) (p/q)^i relative to t_0; S = sum_{i<=k} t_i, T = sum_{i<=n} t_i, both rescaled by 2^-600
    // together whenever a term grows past 2^600 (a power of two: exact)
    const double pq = 1.0 - p;
    DD t = {1.0, 0.0}, S = {1.0, 0.0}, T = {1.0, 0.0};
    for (double i = 1.0; i <= n; i += 1.0) {
        t = dd_div(dd_mul(t, (n - i + 1.0) * p), i * pq);
        T = dd_add(T, t);
        if (i <= k) S = T;
        if (t.hi > 0x1p600) {
            const double sc = 0x1p-600;
            t = {t.hi * sc, t.lo * sc}; S = {S.hi * sc, S.lo * sc}; T = {T.hi * sc, T.lo * sc};
        }
    }
    const DD qT = dd_mul(T, -q);
    const DD d = dd_add(S, qT);                               // S - q T: cdf >= q  <=>  d >= 0
    return d.hi + d.lo >= -1e-27 * T.hi;
}

// smallest integer k in [0, n] with P[Bin(n,p) <= k] >= q   (== scipy.stats.binom.ppf(q, n, p))
YS_HD double binom_ppf(double q, double n, double p) {
    if (isnan(q) || isnan(p) || q < 0.0 || q > 1.0 || p < 0.0 || p > 1.0) return NAN;
    if (q == 0.0) return -1.0;   // scipy: ppf(0) = a - 1
    if (q == 1.0) return n;
    if (n <= 0.0) return 0.0;
    if (p == 0.0) return 0.0;
    if (p == 1.0) return n;
    const double mu = n * p, sd = sqrt(n * p * (1.0 - p));
    double k = floor(mu + norm_ppf_guess(q) * sd);
    if (k < 0.0) k = 0.0;
    if (k > n) k = n;
    // bracket: lo has cdf(lo) < q (or lo = -1), hi has cdf(hi) >= q
    double lo, hi, step = 1.0;
    if (binom_cdf(k, n, p) >= q) {
        hi = k;
        lo = k - 1.0;
        while (lo >= 0.0 && binom_cdf(lo, n, p) >= q) { hi = lo; step *= 2.0; lo = hi - step; }
        if (lo < 0.0) lo = -1.0;
    } else {
        lo = k;
        hi = k + 1.0;
        while (hi < n && binom_cdf(hi, n, p) < q) { lo = hi; step *= 2.0; hi = lo + step; }
        if (hi > n) hi = n;
    }
    while (hi - lo > 1.0) {
        const double mid = floor(0.5 * (lo + hi));
        if (binom_cdf(mid, n, p) >= q) hi = mid; else lo = mid;
    }
    // cdf(lo) < q decided the answer; if that cdf may be an exact tie within fp64's reach of q, settle it
    if (lo >= 0.0 && tie_possible(n, p)) {
        if (n > TIE_NMAX) {
            if (2.0 * lo + 1.0 == n && 0.5 >= q) hi = lo;   // p = 1/2: only cdf((n-1)/2) = 1/2 can tie
        } else {
            const double c = binom_cdf(lo, n, p);
            const double tol = 4.0 * 0x1p-53 * fmax(q, 1.0 - q) + 1e-13 * fmin(q, 1.0 - q);
            if (q - c <= tol && cdf_ge_tie(lo, n, p, q)) hi = lo;
        }
    }
    return hi;
}

// x with I_x(a, b) = y for a = n - k, b = k + 1 (positive integers), 0 < y < 1.
// Works on w = 1 - x: P[Bin(n, w) <= k] = y.  Returns x = 1 - w.
YS_HD double betaincinv_int(double n, double k, double y) {
    if (isnan(y) || y < 0.0 || y > 1.0) return NAN;
    if (n - k <= 0.0 || k + 1.0 <= 0.0) return NAN;   // scipy: a <= 0 -> nan
    if (y == 0.0) return 0.0;
    if (y == 1.0) return 1.0;
    const double t = 1.0 - y;             // = P[Bin(n, w) > k], the target of the upper tail
    if (k == 0.0) {
        // I_x(n, 1) = x^n
        return exp(log(y) / n);
    }
    // initial guess: k = n w + z sqrt(n w (1-w)) with z = norm_ppf(y)
    const double z = norm_ppf_guess(y);
    double w;
    {
        const double ph = k / n;
        w = ph - z * sqrt(ph * (1.0 - ph) / n);
        for (int it = 0; it < 3; it++) {
            const double ww = w < 1e-12 ? 1e-12 : (w > 1.0 - 1e-12 ? 1.0 - 1e-12 : w);
            w = ph - z * sqrt(ww * (1.0 - ww) / n);
        }
    }
    double wlo = 0.0, whi = 1.0;          // cdf(k; n, w) is decreasing in w: cdf(wlo) = 1 > y > cdf(whi) = 0
    if (!(w > 0.0)) w = 0.5 * k / n;
    if (!(w < 1.0)) w = 0.5 * (1.0 + k / n);
    // work with the smaller of the two tails for the residual
    const bool use_upper = (t <= 0.5);
    const double target = use_upper ? t : y;
    const double log_target = log(target);
    for (int it = 0; it < 200; it++) {
        double c, s, lsmall;
        bool lower;
        cdf_sf(k, n, w, &c, &s, &lsmall, &lower);
        // ln of the tail we track
        double ltail;
        if (use_upper) ltail = lower ? log1p(-c) : lsmall;
        else ltail = lower ? lsmall : log1p(-s);
        const double g = ltail - log_target;        // monotone in w: increasing if use_upper, decreasing otherwise
        const bool w_too_big = use_upper ? (g > 0.0) : (g < 0.0);
        if (g == 0.0) break;
        if (w_too_big) whi = w; else wlo = w;
        // d/dw P[X > k] = (n - k) pmf(k; n, w) / (1 - w)
        const double dtail = (n - k) * exp(log_pmf(k, n, w) - ltail) / (1.0 - w);   // |d ln tail / dw|
        double wn = use_upper ? (w - g / dtail) : (w + g / dtail);
        if (!(wn > wlo && wn < whi) || isnan(wn)) wn = 0.5 * (wlo + whi);
        if (fabs(wn - w) <= 4e-16 * w || whi - wlo <= 2e-16 * w) { w = wn; break; }
        w = wn;
    }
    return 1.0 - w;
}

struct HypRow {
    int in_sample_est;
    double p_val;
    long long num_exclusive_kmers;
    long long num_exclusive_kmers_coverage;
    long long num_matches;
    double acceptance_threshold_with_coverage;
    double actual_confidence_with_coverage;
    double alt_confidence_mut_rate_with_coverage;
};

// single_hyp_test (hypothesis_recovery_src.py:233-306).  non_mut_p = ani_thresh ** ksize is
// computed once by the caller (pow in double, like Python's **).
YS_HD HypRow single_hyp_test(long long n_excl, long long n_match, int ksize, double significance, double non_mut_p,
                             double min_coverage) {
    HypRow r;
    r.num_exclusive_kmers = n_excl;
    // int(num_exclusive_kmers * min_coverage): double multiply, truncation toward zero
    const long long n_cov = (long long)((double)n_excl * min_coverage);
    r.num_exclusive_kmers_coverage = n_cov;
    r.num_matches = n_match;
    const double n = (double)n_cov;
    const double q = 1.0 - significance;
    const double thr = binom_ppf(q, n, non_mut_p);
    r.acceptance_threshold_with_coverage = thr;
    r.actual_confidence_with_coverage = 1.0 - binom_cdf(thr, n, non_mut_p);
    // get_alt_mut_rate(:229-230)
    const double x = betaincinv_int(n, thr, significance);
    double mut = 1.0 - pow(1.0 - x, 1.0 / (double)ksize);
    if (isnan(mut)) mut = -1.0;
    r.alt_confidence_mut_rate_with_coverage = mut;
    if (n_match <= n_cov) {
        double c, s, ls;
        bool lower;
        cdf_sf((double)n_match, n, non_mut_p, &c, &s, &ls, &lower);
        r.p_val = c;
    } else {
        r.p_val = 1.0;
    }
    r.in_sample_est = ((double)n_match >= thr && n_match != 0) ? 1 : 0;
    return r;
}

}  // namespace ystats
