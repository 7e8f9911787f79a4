"""Fixed-capacity bucket slots of the MSD partition (index_msd.cu, msd_build).  The scatters write every bucket into a slot whose
size comes from the plan alone; the histogram passes run only when a slot overflows: a level-2 overflow repeats level 2 on the
exact layout, a level-1 overflow the whole partition.  ms_hist1 / ms_hist2 are non-zero exactly when those passes ran.

Covered here: synthetic databases that take the slotted path end to end (train statistics, flagged pairs and the run path's
exclusive-hash counts against the CPU oracles); a final bucket that fills its slot exactly (slotted) and one a word over it (level-2
retry), with both grouping kernels; a top level-1 digit over its slot (full retry).  The crafted databases of
test_group2_edges_gpu.py overflow their level-2 slots, so they keep covering the exact layout's bucket boundaries."""
import math

import numpy as np
import pytest

from oracle import train_oracle as to
from test_group2_edges_gpu import A_TARGET, bucket_db
from yacht_b200 import synth

pytestmark = pytest.mark.gpu

THR = 0.95 ** 31
SC_TILE = 4096          # index_msd.cu: words per scatter tile


def plan(hashes, n):
    """msd_build's plan: (hb, d1, d2, C1, C2)."""
    T = len(hashes)
    maxkey = int(hashes.max())
    hb = max(1, maxkey.bit_length())
    D = 0
    while D < hb and D < 22 and T // ((maxkey >> (hb - D)) + 1 if D else 1) > A_TARGET:
        D += 1
    d1 = max(D if D <= 8 else (D + 1) // 2, hb + (n - 1).bit_length() - 64)      # packing: hb - d1 + gb <= 64
    d2 = max(0, D - d1)

    def cap(bits, f, add):       # f * (expected words of a full bucket) + add, rounded up to 16 words
        mean = float(T) * 2.0 ** (hb - bits) / (float(maxkey) + 1.0)
        return (math.ceil(f * mean + add) + 15) // 16 * 16

    return hb, d1, d2, cap(d1, 1.02, SC_TILE), cap(d1 + d2, 1.25, 64.0)


def build(ctx, hashes, offsets):
    ctx.load_sketches(hashes, offsets)
    ctx.reset_timers()
    st = ctx.build_index()
    tm = ctx.timings()
    assert st["index_path"] == 1
    return st, tm


def check_train(ctx, hashes, offsets, thr, kernels=(0,)):
    ref = to.oracle_train(hashes, offsets, thr)
    tms = []
    for kernel in kernels:
        ctx.set_option("group_kernel", kernel)
        try:
            st, tm = build(ctx, hashes, offsets)
            pairs = ctx.pairwise_flag(thr)
        finally:
            ctx.set_option("group_kernel", 0)
        assert (st["n_distinct"], st["n_singleton"], st["n_index"]) == (ref.n_distinct, ref.n_singleton, ref.n_index)
        assert np.array_equal(pairs["i"], ref.pairs["i"]) and np.array_equal(pairs["j"], ref.pairs["j"])
        assert np.array_equal(pairs["count"], ref.pairs["count"])
        tms.append(tm)
    return tms


@pytest.mark.parametrize("n,seed,mean_size", [(3000, 11, 5000.0), (10000, 12, 2000.0)])
def test_slotted_synthetic(gpu_ctx, n, seed, mean_size):
    db = synth.make_reference_db(n, seed=seed, mean_size=mean_size, sd_size=0.3 * mean_size)
    assert plan(db.hashes, n)[2] > 0                    # two partition levels
    (tm,) = check_train(gpu_ctx, db.hashes, db.offsets, THR)
    assert tm["ms_hist1"] == 0.0 and tm["ms_hist2"] == 0.0, tm


def test_run_path_after_slotted_build(gpu_ctx):
    from oracle import run_oracle
    db = synth.make_reference_db(3000, seed=13)
    _, tm = build(gpu_ctx, db.hashes, db.offsets)
    assert tm["ms_hist1"] == 0.0 and tm["ms_hist2"] == 0.0, tm
    sample, _, _ = synth.make_sample(db, seed=14, n_present=60, total_hashes=200000)
    counts = gpu_ctx.exclusive_hashes(sample)
    exp = run_oracle.exclusive_counts(db.hashes, db.offsets, sample)
    for k in ("n_overlap", "n_exclusive", "n_match"):
        assert np.array_equal(counts[k], exp[k]), k


def level2_db(extra, seed, base=850):
    """2 048 final buckets (hb 40, d1 6, d2 5) of `base` words, except bucket 700: C2 words, and bucket 1 500: C2 + extra.
    C2 depends on the word count, which depends on C2: iterate to the fixed point."""
    hb, D = 40, 11
    sizes = [base] * (1 << D)
    for _ in range(8):
        h, o = bucket_db(hb, D, sizes, seed)
        _, d1, d2, c1, c2 = plan(h, len(o) - 1)
        if sizes[700] == c2 and sizes[1500] == c2 + extra:
            assert (d1, d2) == (6, 5) and 30 * base + 2 * c2 + extra <= c1
            return h, o, c2
        sizes[700], sizes[1500] = c2, c2 + extra
    raise AssertionError("slot capacity did not settle")


@pytest.mark.parametrize("extra", [0, 1])
def test_level2_slot_boundary(gpu_ctx, extra):
    # extra 0: a bucket fills its slot exactly -- slotted; extra 1: one word over -- level 2 again on the exact layout
    h, o, c2 = level2_db(extra, seed=21)
    for tm in check_train(gpu_ctx, h, o, 0.0, kernels=(0, 1)):
        assert tm["ms_hist1"] == 0.0, tm
        assert (tm["ms_hist2"] > 0.0) == (extra == 1), (c2, tm)


def test_level1_overflow_full_retry(gpu_ctx):
    # 64 level-1 digits of 32 final buckets: the top digit holds 32 x 1 000 words, more than its slot (~27 k words), so the
    # whole partition is repeated on the exact layout
    hb, D = 40, 11
    sizes = [700] * ((1 << D) - 32) + [1000] * 32
    h, o = bucket_db(hb, D, sizes, seed=22)
    _, d1, d2, c1, _ = plan(h, len(o) - 1)
    assert (d1, d2) == (6, 5) and 32 * 1000 > c1
    for tm in check_train(gpu_ctx, h, o, 0.0, kernels=(0, 1)):
        assert tm["ms_hist1"] > 0.0 and tm["ms_hist2"] > 0.0, tm
