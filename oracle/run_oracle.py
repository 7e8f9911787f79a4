"""TEST INFRASTRUCTURE ONLY -- CPU restatement ("port") of the reference's run-side compute.

Restates reference src/yacht/hypothesis_recovery_src.py:
  * get_organisms_with_nonzero_overlap (:30-113): the reference shells out to
    ``sourmash scripts multisearch ... -t 0`` (sourmash_plugin_branchwater, a third-party Rust
    package that is NOT in /root/reference and has no version pin: env/yacht_env.yml:8,23) and
    keeps the ``match_name`` column.  Its published behaviour for threshold 0 is "report every
    (query, match) pair whose containment is > 0", i.e. the reference genomes that share at least
    one hash with the sample -- the function's own docstring says the same (:40).  Restated as
    ``|S_g & sample| > 0``.  PARITY OF THIS STEP IS PINNED ONLY by the reference's end-to-end known
    answer (tests/test_workflow.py:58-66: one organism with non-zero overlap, num_matches == 2);
    beyond that, multisearch's threshold semantics are unpinned.
  * get_exclusive_hashes (:116-206): python-set semantics -- among the nontrivial organisms a hash
    is exclusive if it occurs in exactly one organism; per organism (n_exclusive, n_exclusive in
    sample), in sub-manifest order (:160-163).
    PINNED: tests/test_run_reference_golden.py checks it against 200 calls of the reference's OWN
    get_exclusive_hashes over 50 seeded databases (tests/golden/make_run_reference_golden.py imports
    the unmodified hypothesis_recovery_src.py + utils.py with a stand-in for the absent sourmash
    package and commits inputs + outputs as tests/golden/run_reference_golden.npz).
  * get_alt_mut_rate (:209-230) and single_hyp_test (:233-306): restated verbatim on top of scipy
    (``binom.ppf/cdf``, ``betaincinv``), the same library calls the reference makes.
    PINNED: tests/test_oracle_pinned.py checks this restatement against the golden rows extracted
    from the reference's checked-in result workbooks (tests/golden/make_run_golden.py) and the
    reference's own known-answer tests (tests/test_unit.py:11-20, tests/test_unittests.py:86-111),
    and tests/test_run_reference_golden.py against 24,340 evaluations of the reference's own
    single_hyp_test (same generator).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np

COUNTS_DTYPE = np.dtype([("n_overlap", "<u4"), ("nontrivial", "<u4"), ("n_exclusive", "<u4"), ("n_match", "<u4")])


def nonzero_overlap(hashes: np.ndarray, offsets: np.ndarray, sample: np.ndarray) -> np.ndarray:
    """n_overlap[g] = |set(S_g) & set(sample)| (multisearch -t 0 keeps the genomes where it is > 0)."""
    n = offsets.shape[0] - 1
    sample_set = np.unique(np.asarray(sample, dtype=np.uint64))
    out = np.zeros(n, dtype=np.uint32)
    for g in range(n):
        sk = np.unique(hashes[int(offsets[g]):int(offsets[g + 1])])
        if sk.size and sample_set.size:
            out[g] = np.count_nonzero(np.isin(sk, sample_set, assume_unique=True))
    return out


def exclusive_counts(hashes: np.ndarray, offsets: np.ndarray, sample: np.ndarray, mask: np.ndarray = None) -> np.ndarray:
    """Python-set restatement of hypothesis_recovery_src.py:165-204 over the nontrivial organisms
    (mask, or overlap > 0).  Deliberately written with the same set operations as the reference."""
    n = offsets.shape[0] - 1
    out = np.zeros(n, dtype=COUNTS_DTYPE)
    out["n_overlap"] = nonzero_overlap(hashes, offsets, sample)
    nontrivial = (out["n_overlap"] > 0) if mask is None else (np.asarray(mask) != 0)
    out["nontrivial"] = nontrivial.astype(np.uint32)
    ids = np.flatnonzero(nontrivial)
    single, multiple = set(), set()
    sketches = {}
    for g in ids:
        hs = set(int(h) for h in hashes[int(offsets[g]):int(offsets[g + 1])])   # sig.minhash.hashes is a dict: unique
        sketches[int(g)] = hs
        for h in hs:
            if h in multiple:
                continue
            elif h in single:
                single.remove(h)
                multiple.add(h)
            else:
                single.add(h)
    sample_hashes = set(int(h) for h in sample)
    for g in ids:
        excl = {h for h in sketches[int(g)] if h in single}
        out["n_exclusive"][g] = len(excl)
        out["n_match"][g] = len(excl.intersection(sample_hashes))
    return out


def exclusive_counts_np(hashes: np.ndarray, offsets: np.ndarray, sample: np.ndarray, mask: np.ndarray = None) -> np.ndarray:
    """exclusive_counts with whole-array numpy operations, for databases of millions of genomes (the set restatement
    loops in Python per genome).  tests/test_sparse_oracle.py checks that both agree."""
    n = offsets.shape[0] - 1
    out = np.zeros(n, dtype=COUNTS_DTYPE)
    gid = np.repeat(np.arange(n, dtype=np.int64), np.diff(np.asarray(offsets, dtype=np.int64)))
    h = np.asarray(hashes, dtype=np.uint64)
    order = np.lexsort((gid, h))                                   # by hash, then genome
    h, gid = h[order], gid[order]
    first = np.ones(h.shape[0], dtype=bool)                       # one entry per distinct (hash, genome): sketches are sets
    first[1:] = (h[1:] != h[:-1]) | (gid[1:] != gid[:-1])
    h, gid = h[first], gid[first]
    in_sample = np.isin(h, np.unique(np.asarray(sample, dtype=np.uint64)))
    out["n_overlap"] = np.bincount(gid[in_sample], minlength=n)
    nontrivial = (out["n_overlap"] > 0) if mask is None else (np.asarray(mask) != 0)
    out["nontrivial"] = nontrivial
    keep = nontrivial[gid]
    h, gid, in_sample = h[keep], gid[keep], in_sample[keep]
    head = np.ones(h.shape[0] + 1, dtype=bool)                    # runs of equal hashes among the nontrivial genomes
    head[1:-1] = h[1:] != h[:-1]
    starts = np.flatnonzero(head)
    run_len = np.diff(starts)
    excl = np.repeat(run_len == 1, run_len)
    out["n_exclusive"] = np.bincount(gid[excl], minlength=n)
    out["n_match"] = np.bincount(gid[excl & in_sample], minlength=n)
    return out


def get_alt_mut_rate(nu: int, thresh: int, ksize: int, significance: float = 0.99) -> float:
    """hypothesis_recovery_src.py:209-230."""
    from scipy.special import betaincinv
    mut = 1 - (1 - betaincinv(nu - thresh, 1 + thresh, significance)) ** (1 / ksize)
    return -1.0 if np.isnan(mut) else float(mut)


def single_hyp_test(exclusive_hashes_info_org: Tuple[int, int], ksize: int, significance: float = 0.99,
                    ani_thresh: float = 0.95, min_coverage: float = 1):
    """hypothesis_recovery_src.py:233-306 -> the 8-tuple in the column order of :377-391."""
    from scipy.stats import binom
    num_exclusive_kmers = int(exclusive_hashes_info_org[0])
    non_mut_p = (ani_thresh) ** ksize
    num_exclusive_kmers_coverage = int(num_exclusive_kmers * min_coverage)
    acceptance_threshold_with_coverage = binom.ppf(1 - significance, num_exclusive_kmers_coverage, non_mut_p)
    actual_confidence_with_coverage = 1 - binom.cdf(acceptance_threshold_with_coverage, num_exclusive_kmers_coverage, non_mut_p)
    alt_confidence_mut_rate_with_coverage = get_alt_mut_rate(num_exclusive_kmers_coverage, acceptance_threshold_with_coverage,
                                                             ksize, significance=significance)
    num_matches = int(exclusive_hashes_info_org[1])
    if num_matches <= num_exclusive_kmers_coverage:
        p_val = binom.cdf(num_matches, num_exclusive_kmers_coverage, non_mut_p)
    else:
        p_val = 1.0
    in_sample_est = bool((num_matches >= acceptance_threshold_with_coverage) and (num_matches != 0))
    return (in_sample_est, float(p_val), num_exclusive_kmers, num_exclusive_kmers_coverage, num_matches,
            float(acceptance_threshold_with_coverage), float(actual_confidence_with_coverage),
            float(alt_confidence_mut_rate_with_coverage))


HYP_FIELDS = ["in_sample_est", "p_val", "num_exclusive_kmers", "num_exclusive_kmers_coverage", "num_matches",
              "acceptance_threshold_with_coverage", "actual_confidence_with_coverage",
              "alt_confidence_mut_rate_with_coverage"]

# Tolerance of the floating-point outputs (north_star: 1e-9 relative against the reference's
# floats).  One carve-out, for p-values only: scipy/Boost evaluates binom.cdf through the
# regularised incomplete beta and loses the result to underflow of intermediate powers when the
# true value is tiny -- e.g. binom.cdf(30, 3243, 0.95**31) returns exactly 0.0 where the true
# value is 8.76e-267, and binom.cdf(5, 3243, 0.95**31) returns 3.79e-309 for a true 2.21e-309
# (scan in DESIGN.md: the largest true value with a deviating scipy result was 8.8e-267).  Such
# p-values are "zero" for every use the reference makes of them, so two values that are BOTH
# below UNDERFLOW_FLOOR are accepted as equal; everything else must agree to REL_TOL.
REL_TOL = 1e-9
UNDERFLOW_FLOOR = 1e-250


def float_close(a: float, b: float, rel: float = REL_TOL) -> bool:
    if a == b:
        return True
    if np.isnan(a) or np.isnan(b):
        return bool(np.isnan(a) and np.isnan(b))
    if abs(a) < UNDERFLOW_FLOOR and abs(b) < UNDERFLOW_FLOOR:
        return True
    return abs(a - b) <= rel * abs(b)


def assert_rows_close(rows: np.ndarray, n_exclusive: Sequence[int], n_match: Sequence[int], ksize: int, significance: float,
                      ani_thresh: float, coverages: Sequence[float], rel: float = REL_TOL) -> None:
    """rows[c, r] (ygpu_hyp_row records) against single_hyp_test: integers/booleans exact, floats
    within `rel` relative (exact for the 0 / 1 / -1 sentinels)."""
    cache = {}
    for c, cov in enumerate(coverages):
        for r in range(len(n_exclusive)):
            key = (int(n_exclusive[r]), int(n_match[r]), float(cov))
            if key not in cache:
                cache[key] = single_hyp_test((key[0], key[1]), ksize, significance, ani_thresh, cov)
            exp = cache[key]
            got = rows[c, r]
            ctxt = f"n_excl={key[0]} m={key[1]} cov={cov} k={ksize} sig={significance} ani={ani_thresh}: got {got} exp {exp}"
            assert bool(got["in_sample_est"]) == exp[0], ctxt
            assert int(got["num_exclusive_kmers"]) == exp[2], ctxt
            assert int(got["num_exclusive_kmers_coverage"]) == exp[3], ctxt
            assert int(got["num_matches"]) == exp[4], ctxt
            assert float(got["acceptance_threshold_with_coverage"]) == exp[5], ctxt
            assert float_close(float(got["p_val"]), exp[1], rel), ctxt
            assert float_close(float(got["actual_confidence_with_coverage"]), exp[6], rel), ctxt
            assert float_close(float(got["alt_confidence_mut_rate_with_coverage"]), exp[7], rel), ctxt
