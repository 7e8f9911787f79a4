// TEST-ONLY harness: evaluates the fp64 formulas of yacht_b200/csrc/binom_stats.cuh with g++ so
// their numerics can be checked against scipy and an exact reference on a box without a GPU.
// It is never built into, linked with or called by the product (which runs these formulas only
// inside the CUDA kernels k6_hyp_test and k6_alt_mut_rate).
// As an executable:   stdin lines "n_excl n_match ksize significance ani cov", stdout the 8 outputs per line.
// As a shared library (tests/test_binom_stats_exact.py): the sh_* functions below, the last two with the
// signatures of ygpu_alt_mut_rate / ygpu_hyp_test minus the context.
#include <cmath>
#include <cstdio>
#include "../../include/yacht_gpu.h"
#include "../../yacht_b200/csrc/binom_stats.cuh"

extern "C" {

double sh_binom_cdf(double k, double n, double p) { return ystats::binom_cdf(k, n, p); }

// out[0] = cdf, out[1] = sf, out[2] = ln(min(cdf, sf)), out[3] = 1 if the lower tail was summed
void sh_cdf_sf(double k, double n, double p, double* out) {
    double c, s, l;
    bool lower;
    ystats::cdf_sf(k, n, p, &c, &s, &l, &lower);
    out[0] = c; out[1] = s; out[2] = l; out[3] = lower ? 1.0 : 0.0;
}

double sh_binom_ppf(double q, double n, double p) { return ystats::binom_ppf(q, n, p); }

double sh_betaincinv_int(double n, double k, double y) { return ystats::betaincinv_int(n, k, y); }

// ygpu_alt_mut_rate: out[r] = k6_alt_mut_rate's body for (nu[r], thresh[r])
void sh_alt_mut_rate(const long long* nu, const long long* thresh, long long n, int ksize, double significance,
                     double* out) {
    for (long long r = 0; r < n; r++) {
        const double x = ystats::betaincinv_int((double)nu[r], (double)thresh[r], significance);
        const double mut = 1.0 - pow(1.0 - x, 1.0 / (double)ksize);
        out[r] = std::isnan(mut) ? -1.0 : mut;
    }
}

// ygpu_hyp_test: rows[c * n + r] = k6_hyp_test's body, with non_mut_p = ani ** ksize formed as the host API forms it
void sh_hyp_test(const long long* n_excl, const long long* n_match, long long n, int ksize, double significance,
                 double ani, const double* cov, int n_cov, ygpu_hyp_row* rows) {
    const double p0 = std::pow(ani, (double)ksize);
    for (int c = 0; c < n_cov; c++)
        for (long long r = 0; r < n; r++) {
            const ystats::HypRow h = ystats::single_hyp_test(n_excl[r], n_match[r], ksize, significance, p0, cov[c]);
            ygpu_hyp_row& o = rows[c * n + r];
            o.in_sample_est = h.in_sample_est;
            o._pad = 0;
            o.p_val = h.p_val;
            o.num_exclusive_kmers = h.num_exclusive_kmers;
            o.num_exclusive_kmers_coverage = h.num_exclusive_kmers_coverage;
            o.num_matches = h.num_matches;
            o.acceptance_threshold_with_coverage = h.acceptance_threshold_with_coverage;
            o.actual_confidence_with_coverage = h.actual_confidence_with_coverage;
            o.alt_confidence_mut_rate_with_coverage = h.alt_confidence_mut_rate_with_coverage;
        }
}

}  // extern "C"

int main() {
    long long ne, nm; int k; double sig, ani, cov;
    while (scanf("%lld %lld %d %lf %lf %lf", &ne, &nm, &k, &sig, &ani, &cov) == 6) {
        const double p0 = std::pow(ani, (double)k);
        ystats::HypRow r = ystats::single_hyp_test(ne, nm, k, sig, p0, cov);
        printf("%d %.17g %lld %lld %lld %.17g %.17g %.17g\n", r.in_sample_est, r.p_val, r.num_exclusive_kmers,
               r.num_exclusive_kmers_coverage, r.num_matches, r.acceptance_threshold_with_coverage,
               r.actual_confidence_with_coverage, r.alt_confidence_mut_rate_with_coverage);
    }
    return 0;
}
