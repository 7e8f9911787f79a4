"""Edge cases of the bucket schedule of the shared-memory grouping kernel k2_group2, on databases whose final buckets are
laid out word by word: CTAs whose only bucket is empty, runs of empty buckets a CTA has to skip, buckets of exactly
G2_MAXM (1022) words -- the largest it takes, a full 1024-word window when the bucket starts at an odd word -- and
G2_MAXM + 1 words, which go to the general kernel, and in-sketch duplicates.  Each database is indexed with k2_group2
(group_kernel 0) and with the general kernel k2_group alone (group_kernel 1); statistics and flagged pairs must agree with
each other and with the CPU oracle.  (Many buckets per CTA, so that the ring of stage buffers wraps hundreds of times, is
the benchmarked 85 205-genome database of tests/test_config_digests_gpu.py.  The single-GPU launch never has more CTAs
than buckets -- its grid is min(buckets, SMs x CTAs per SM) -- so CTAs without work arise only from empty buckets here;
the sharded step's launch, whose grid is always SMs x CTAs per SM, is exercised by the multi-GPU tests.)"""
import numpy as np
import pytest

from oracle import train_oracle as to

pytestmark = pytest.mark.gpu

A_TARGET = 900          # index_msd.cu: the plan takes the fewest leading hash bits D with T / 2^D <= A_TARGET
N_GENOMES = 211         # prime: the members of a group, g0 + 7 k mod N, are distinct genomes


def bucket_db(hb, D, sizes, seed):
    """Sketches whose words fall into final bucket b = hash >> (hb - D) exactly sizes[b] times.  Inside a bucket, hashes
    are held by 1..12 genomes (mostly 1 or 2, as in real databases), and about 1 % of the words repeat their neighbour's
    (hash, genome): in-sketch duplicates."""
    assert len(sizes) == 1 << D and sizes[-1] > 0          # the last bucket sets the hash width hb
    T = int(sum(sizes))
    assert A_TARGET * (1 << D) >= T > A_TARGET * (1 << (D - 1)), "the plan would pick another bucket count"
    rng = np.random.default_rng(seed)
    shift = hb - D
    hs, gs = [], []
    for b, m in enumerate(sizes):
        if not m:
            continue
        L = rng.choice([1, 2, 3, 4, 6, 12], size=m, p=[0.60, 0.25, 0.08, 0.04, 0.02, 0.01])
        L = L[:np.searchsorted(np.cumsum(L), m) + 1]
        L[-1] -= int(L.sum()) - m
        grp = np.repeat(np.arange(len(L)), L)
        rank = np.arange(m) - np.repeat(np.cumsum(L) - L, L)
        h = (np.uint64(b) << np.uint64(shift)) + rng.integers(0, 1 << shift, size=len(L), dtype=np.uint64)[grp]
        g = (rng.integers(0, N_GENOMES, size=len(L))[grp] + 7 * rank) % N_GENOMES
        dup = np.flatnonzero(rng.random(m) < 0.01)
        dup = dup[dup > 0]
        h[dup], g[dup] = h[dup - 1], g[dup - 1]
        hs.append(h)
        gs.append(g)
    h, g = np.concatenate(hs), np.concatenate(gs)
    order = np.lexsort((h, g))
    offsets = np.zeros(N_GENOMES + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(np.bincount(g, minlength=N_GENOMES))
    return h[order], offsets


def check_both_kernels(ctx, hashes, offsets):
    res = []
    for kernel in (0, 1):
        ctx.set_option("group_kernel", kernel)
        try:
            ctx.load_sketches(hashes, offsets)
            st = ctx.build_index()
            pairs = ctx.pairwise_flag(0.0)
        finally:
            ctx.set_option("group_kernel", 0)
        assert st["index_path"] == 1 and st["big_buckets"] == 0
        res.append((st, pairs))
    (st0, p0), (st1, p1) = res
    assert st0 == st1
    assert p0.tobytes() == p1.tobytes()
    ref = to.oracle_train(hashes, offsets, 0.0)
    assert (st0["n_distinct"], st0["n_singleton"], st0["n_index"]) == (ref.n_distinct, ref.n_singleton, ref.n_index)
    assert np.array_equal(p0["i"], ref.pairs["i"]) and np.array_equal(p0["j"], ref.pairs["j"])
    assert np.array_equal(p0["count"], ref.pairs["count"])
    assert st0["has_duplicates"] == 1
    return st0


def test_ctas_without_a_bucket(gpu_ctx):
    # four final buckets, one CTA each: the CTAs of buckets 1 and 2 find nothing to group
    h, o = bucket_db(20, 2, [1000, 0, 0, 1000], seed=5)
    check_both_kernels(gpu_ctx, h, o)


def test_empty_runs_and_largest_buckets(gpu_ctx):
    # 2 048 final buckets over at most 4 CTAs per SM: each CTA takes several, with stride gridDim.x.  In every 16 buckets:
    # one of G2_MAXM words, one of G2_MAXM + 1 (left to the general kernel), a run of eight empty ones, six of 900
    # words; 1022 + 1023 is odd, so both word parities of a bucket's start occur
    pattern = [1022, 1023, 900, 900] + [0] * 8 + [900] * 4
    h, o = bucket_db(40, 11, pattern * 128, seed=6)
    check_both_kernels(gpu_ctx, h, o)
