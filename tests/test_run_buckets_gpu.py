"""Crafted bucket layouts for the run path's bucket probe (k5_bucket in run_buckets.cuh, driven by ygpu_run_counts_buckets in
index_msd.cu).  Every crafted input runs both run paths through test_run_parity_gpu._check_counts -- the probe and the
general sort path -- against the set oracle, and asserts which path answered; the residency test probes one context in turn.  Each builder's claimed shape (bucket sizes, survivors per
bucket, sample hashes per bucket, partition plan) is recomputed on the host from plan() before the GPU is asked, and
test_crafted_inputs_have_their_shape checks all of them without a GPU.

Covered: the probe's bucket schedule (CTAs whose only bucket is empty, runs of empty buckets, buckets of exactly G2_MAXM
words at odd starts -- a full 1 024-word window); the settlement boundary of each pass (exactly RB_SMALL = 192 survivors in a
bucket: the all-pairs scan; 193: the sub-bucket machinery, with shared hashes, in-sketch duplicates, survivors alone in their
sub-bucket in and out of the sample, one sub-bucket holding most survivors); the sample capacity (a sample bucket of exactly
RB_SCAP = 1 024 hashes, and 1 025, which sends the sample to the sort path; also reached through duplicates); the partition
layouts (one level, two levels slotted, a level-2 retry, a full level-1 retry, an oversized final bucket, full-range 64-bit
hashes, a narrow hash width whose sub-bucket digit is all that remains of the key); and residency on one context (the
partition a sample builds is not a train index, the train index's partition serves samples, scratch reuse over samples of
changing size, a new database replaces the partition).

The probe's other fallback, gb + rest_bits > 63, cannot occur: packing keeps hb - d1 + gb <= 64, and rest_bits = hb - d1 - d2
- sbits with sbits = min(11, hb - d1 - d2), so gb + rest_bits <= 53 when the remaining key has 11 bits or more and
gb + rest_bits = gb <= 32 when it has fewer."""
import numpy as np
import pytest

from oracle import run_oracle as ro
from oracle import train_oracle as to
from test_bucket_slots_gpu import level2_db, plan
from test_group2_edges_gpu import bucket_db
from test_run_parity_gpu import _check_counts
from yacht_b200 import synth
from yacht_b200._lib import YgpuError

G2_MAXM = 1022          # index_msd.cu: the largest final bucket the probe takes
RB_SCAP = 1024          # run_buckets.cuh: sample hashes of one bucket held in shared memory
RB_SMALL = 192          # run_buckets.cuh: survivors settled by the all-pairs scan
SUBBITS = 11            # sub-bucket digit: the next 11 hash bits below the final bucket's
THR = 0.95 ** 31


# ---- the host model of the partition and of the probe's choice ----------------------------------------------------------
def shr(x, s):
    return np.zeros_like(x) if s >= 64 else x >> np.uint64(s)


def layout(hashes, n):
    """msd_build's final buckets: dict of the plan, the final bucket of every word and the words per final bucket."""
    hb, d1, d2, c1, c2 = plan(hashes, n)
    maxkey = int(hashes.max())
    nb1 = (maxkey >> (hb - d1)) + 1 if d1 else 1
    key_bits = hb - d1 - d2
    sbits = max(0, min(SUBBITS, key_bits))
    b = shr(hashes, key_bits).astype(np.int64)
    return dict(hb=hb, d1=d1, d2=d2, c1=c1, c2=c2, nb1=nb1, nb=nb1 << d2, key_bits=key_bits, sbits=sbits,
                rest_bits=key_bits - sbits, bucket=b, sizes=np.bincount(b, minlength=nb1 << d2))


def sub_digit(hashes, L):
    return (shr(hashes, L["rest_bits"]) & np.uint64((1 << L["sbits"]) - 1)).astype(np.int64)


def sample_counts(sample, L):
    """Sample hashes (duplicates included) per final bucket; hashes beyond the hash width or the last level-1 digit are dropped."""
    s = np.asarray(sample, dtype=np.uint64)
    if L["hb"] < 64:
        s = s[shr(s, L["hb"]) == 0]
    if L["d1"]:
        s = s[shr(s, L["hb"] - L["d1"]) < np.uint64(L["nb1"])]
    return np.bincount(shr(s, L["key_bits"]).astype(np.int64), minlength=L["nb"])


def genome_of(offsets):
    return np.repeat(np.arange(len(offsets) - 1), np.diff(offsets.astype(np.int64)))


def survivors(hashes, offsets, sample, mask, L):
    """Boolean per word: pass 1 (hash in the sample), pass 2 (genome nontrivial: the mask, else overlap > 0)."""
    g = genome_of(offsets)
    p1 = np.isin(hashes, np.asarray(sample, dtype=np.uint64))
    nt = np.zeros(len(offsets) - 1, bool)
    nt[g[p1]] = True
    if mask is not None:
        nt = np.asarray(mask) != 0
    return p1, nt[g]


def expect_probe(hashes, offsets, sample):
    """Whether ygpu_exclusive_hashes takes the bucket probe (run_path 1) for this input."""
    n = len(offsets) - 1
    if len(hashes) < 2 or n < 2:
        return False
    L = layout(hashes, n)
    if L["d1"] > 11 or L["d1"] > L["hb"] or L["d2"] > 11 or L["nb1"] > 2048:
        return False                                    # does not pack: no partition
    if L["sizes"].max() > G2_MAXM:
        return False                                    # skewed database
    return sample_counts(sample, L).max(initial=0) <= RB_SCAP


def db_of(h, o):
    return synth.SketchDB(hashes=h, offsets=o, cluster=np.full(len(o) - 1, -1))


def csr(h, g, n):
    order = np.lexsort((h, g))
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(np.bincount(g, minlength=n))
    return h[order].astype(np.uint64), offsets


def probe_case(ctx, h, o, sample, mask=None):
    probe = expect_probe(h, o, sample)
    _check_counts(ctx, db_of(h, o), sample, mask, probe=probe)
    return probe


def some_sample(h, rng, k, extra=0, hb=40):
    """k distinct hashes of the reference plus `extra` hashes it does not hold, shuffled."""
    s = rng.choice(np.unique(h), size=k, replace=False)
    if extra:
        s = np.concatenate([s, rng.integers(0, 1 << hb, size=extra, dtype=np.uint64)])
    return rng.permutation(s)


# ---- builders ------------------------------------------------------------------------------------------------------------
def schedule_db():
    """2 048 final buckets (hb 40, d1 6, d2 5); in every 16: two of G2_MAXM words, two of 900 and 901, a run of eight empty
    ones, four of 900.  The level-2 slots (~1.25 x 465 + 64 words) overflow, so the exact layout is used: buckets start at
    prefix sums, and 7 445 words per 16 buckets is odd, so the G2_MAXM buckets start at both word parities."""
    pattern = [G2_MAXM, 901, G2_MAXM, 900] + [0] * 8 + [900] * 4
    return bucket_db(40, 11, pattern * 128, seed=31)


def boundary_db(target, seed):
    """hb 40, d1 2, d2 0: 4 final buckets, sub-bucket digit = hash bits 27..37.  Bucket 0 holds `target` core words of
    genomes 0..9, 500 filler words of genomes 100..210 and one more filler word Y; buckets 1..3 come from bucket_db.
    Core: sub-bucket 5 holds 40 hashes of two genomes each, 20 of one genome and one hash twice in genome 3's sketch (102
    words); hash A (genome 4) is alone in sub-bucket 7 and hash B (genome 6) alone in sub-bucket 9; the rest are single
    words scattered over sub-buckets 16.. .  The sample holds every core hash but B, and Y: pass 1 keeps target words of
    bucket 0, and pass 2 under the mask of genomes 0..9 keeps the target core words."""
    rng = np.random.default_rng(seed)
    h0, o0 = bucket_db(40, 2, [0, 900, 900, 900], seed=seed)
    g0 = genome_of(o0)
    sub = lambda s, r: (np.uint64(s) << np.uint64(27)) | np.asarray(r, dtype=np.uint64)
    r5 = rng.choice(1 << 27, size=61, replace=False)
    hs, gs = [], []
    for i in range(40):                                     # two genomes share a hash
        hs += [sub(5, r5[i])] * 2
        gs += [i % 10, (i + 1) % 10]
    for i in range(40, 60):
        hs.append(sub(5, r5[i]))
        gs.append(i % 10)
    hs += [sub(5, r5[60])] * 2                              # an in-sketch duplicate
    gs += [3, 3]
    A, B = sub(7, rng.integers(1 << 27)), sub(9, rng.integers(1 << 27))
    hs += [A, B]
    gs += [4, 6]
    rest = target - len(hs)
    hr = sub(rng.integers(16, 1 << SUBBITS, size=rest + 501), rng.choice(1 << 27, size=rest + 501, replace=False))
    hs += list(hr[:rest])
    gs += list(rng.integers(0, 10, size=rest))
    core_h = np.array(hs, dtype=np.uint64)
    fill_h = hr[rest:]                                      # distinct from the core hashes
    fill_g = rng.integers(100, 211, size=501)
    h = np.concatenate([h0, core_h, fill_h])
    g = np.concatenate([g0, np.array(gs), fill_g])
    hh, oo = csr(h, g, 211)
    Y = fill_h[-1]
    others = rng.choice(h0, size=60, replace=False)
    sample = rng.permutation(np.concatenate([np.unique(core_h[core_h != B]), [Y], others]).astype(np.uint64))
    mask = np.zeros(211, np.uint8)
    mask[:10] = 1
    return hh, oo, sample, mask


def capacity_case(count, dups, seed):
    """hb 40, d1 2, d2 0, 4 final buckets of 900 words; the sample has `count` hashes in bucket 3 (4 distinct reference hashes
    repeated when `dups`, else 300 reference hashes and hashes the reference does not hold) and 100 in each other bucket."""
    rng = np.random.default_rng(seed)
    h, o = bucket_db(40, 2, [900] * 4, seed=seed)
    top = np.unique(h[shr(h, 38) == np.uint64(3)])
    if dups:
        pick = rng.choice(top, size=4, replace=False)
        s3 = np.concatenate([np.repeat(pick, 256), pick[:count - 1024]]) if count > 1024 else np.repeat(pick, 256)[:count]
    else:
        s3 = rng.choice(top, size=300, replace=False)
        new = np.setdiff1d((np.uint64(3) << np.uint64(38)) + rng.choice(1 << 38, size=2 * count, replace=False).astype(np.uint64), top)
        s3 = np.concatenate([s3, new[:count - 300]])
    low = np.unique(h[shr(h, 38) < np.uint64(3)])
    rest = np.concatenate([rng.choice(low[shr(low, 38) == np.uint64(b)], size=100, replace=False) for b in range(3)])
    return h, o, rng.permutation(np.concatenate([s3, rest]).astype(np.uint64))


def level1_retry_db():
    """test_bucket_slots_gpu.test_level1_overflow_full_retry: the top level-1 digit holds 32 x 1 000 words, over its slot."""
    return bucket_db(40, 11, [700] * ((1 << 11) - 32) + [1000] * 32, seed=22)


def full_range_db(n, per, seed):
    """n genomes of `per` uniform 64-bit hashes (hb 64: packing needs d1 >= gb)."""
    rng = np.random.default_rng(seed)
    h = rng.integers(0, 2**64 - 1, size=n * per, dtype=np.uint64, endpoint=True)
    h[0] = np.uint64(2**64 - 1)
    h[1::97] = h[0::97][:len(h[1::97])]                     # repeated hashes, inside a sketch and across two
    return csr(h, np.repeat(np.arange(n), per), n)


def narrow_db(seed):
    """hb 13, d1 2, d2 0: 11 bits remain inside a final bucket -- all of them the sub-bucket digit (rest_bits 0)."""
    return bucket_db(13, 2, [900] * 4, seed=seed)


def some_layout_sample(h, seed, k, extra, hb=40):
    return some_sample(h, np.random.default_rng(seed), k, extra, hb)


# (name, builder -> (hashes, offsets, sample), expected: probe?, ms_hist1 > 0, ms_hist2 > 0)
LAYOUTS = [
    ("one level", lambda: (lambda h, o: (h, o, some_layout_sample(h, 41, 3000, 500, 30)))(*bucket_db(30, 8, [850] * 256, seed=42)),
     True, False, False),
    ("two levels, extra 0", lambda: (lambda h, o, _: (h, o, some_layout_sample(h, 41, 40000, 2000)))(*level2_db(0, seed=43, base=600)),
     True, False, False),
    ("two levels, extra 1", lambda: (lambda h, o, _: (h, o, some_layout_sample(h, 41, 40000, 2000)))(*level2_db(1, seed=43, base=600)),
     True, False, True),
    ("level-1 retry", lambda: (lambda h, o: (h, o, some_layout_sample(h, 41, 40000, 2000)))(*level1_retry_db()), True, True, True),
    ("oversized bucket", lambda: (lambda h, o, _: (h, o, some_layout_sample(h, 41, 40000, 2000)))(*level2_db(0, seed=44)),
     False, False, False),
    ("full range, 211 genomes", lambda: (lambda h, o: (h, o, some_layout_sample(h, 41, 800, 200, 64)))(*full_range_db(211, 17, seed=45)),
     True, False, False),
    ("full range, 5000 genomes", lambda: (lambda h, o: (h, o, some_layout_sample(h, 41, 3000, 200, 64)))(*full_range_db(5000, 3, seed=46)),
     False, False, False),
    ("narrow", lambda: (lambda h, o: (h, o, some_layout_sample(h, 41, 1000, 0, 13)))(*narrow_db(seed=47)), True, False, False),
]


def partition_timings(ctx, h, o, sample, mask=None):
    """Timers of a probe that builds the partition itself (a fresh load, so no partition is resident)."""
    ctx.load_sketches(h, o)
    ctx.reset_timers()
    ctx.exclusive_hashes(sample, mask)
    tm = ctx.timings()
    assert tm["ms_sort"] > 0.0 and tm["ms_sample_kernels"] > 0.0, tm
    return tm


# ---- shapes, without a GPU -------------------------------------------------------------------------------------------------
def check_schedule(h, o):
    L = layout(h, len(o) - 1)
    sizes = L["sizes"]
    assert (L["d1"], L["d2"], L["nb"]) == (6, 5, 2048) and sizes.max() > L["c2"]      # level-2 slots overflow: exact layout
    start = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    full = np.flatnonzero(sizes == G2_MAXM)
    assert (start[full] % 2 == 1).any() and (start[full] % 2 == 0).any()                 # a full 1024-word window occurs
    assert sizes.max() == G2_MAXM and (sizes == 0).sum() == 8 * 128
    assert all((r[4:12] == 0).all() for r in np.split(sizes, 128))
    return L


def check_boundary(h, o, sample, mask, target):
    L = layout(h, len(o) - 1)
    assert (L["d1"], L["d2"], L["nb"], L["rest_bits"]) == (2, 0, 4, 27)
    p1, p2 = survivors(h, o, sample, mask, L)
    in0 = L["bucket"] == 0
    assert (p1 & in0).sum() == target and (p2 & in0).sum() == target and L["sizes"].max() <= G2_MAXM
    g = genome_of(o)
    sub = sub_digit(h, L)
    sset = set(int(x) for x in sample)
    for keep in (p1 & in0, p2 & in0):
        kh, kg, ks = h[keep], g[keep], sub[keep]
        assert np.bincount(ks).max() > target // 2                                     # one sub-bucket holds most survivors
        pairs = set()
        dup = False
        for x, y in zip(kh.tolist(), kg.tolist()):
            dup |= (x, y) in pairs
            pairs.add((x, y))
        assert dup                                                                      # an in-sketch duplicate
        holders = {}
        for x, y in pairs:
            holders.setdefault(x, set()).add(y)
        assert max(len(v) for v in holders.values()) >= 2                              # two genomes share a hash
        alone = np.bincount(ks, minlength=1 << SUBBITS)[ks] == 1
        assert alone.any()
    kh, ks = h[p2 & in0], sub[p2 & in0]
    alone = np.bincount(ks, minlength=1 << SUBBITS)[ks] == 1
    ins = np.array([int(x) in sset for x in kh])
    assert (alone & ins).any() and (alone & ~ins).any()                               # singletons in and out of the sample
    return L


def test_crafted_inputs_have_their_shape():
    h, o = bucket_db(20, 2, [1000, 0, 0, 1000], seed=30)
    L = layout(h, len(o) - 1)
    assert L["nb"] == 4 and list(L["sizes"]) == [1000, 0, 0, 1000]
    check_schedule(*schedule_db())
    for target in (RB_SMALL, RB_SMALL + 1):
        check_boundary(*boundary_db(target, seed=32), target)
    for count, dups in ((RB_SCAP, False), (RB_SCAP + 1, False), (RB_SCAP, True), (RB_SCAP + 1, True)):
        h, o, s = capacity_case(count, dups, seed=33)
        L = layout(h, len(o) - 1)
        c = sample_counts(s, L)
        assert c[3] == count and c.max() == count and (len(np.unique(s[shr(s, 38) == np.uint64(3)])) == 4) == dups
        assert expect_probe(h, o, s) == (count <= RB_SCAP)
    for name, make, probe, _, _ in LAYOUTS:
        h, o, s = make()
        L = layout(h, len(o) - 1)
        assert expect_probe(h, o, s) == probe, name
        if name == "one level":
            assert L["d2"] == 0 and L["d1"] == 8
        elif name.startswith("two levels"):
            assert L["d2"] > 0 and L["sizes"].max() <= G2_MAXM and L["sizes"].max() - L["c2"] == int(name[-1])
        elif name == "level-1 retry":
            assert L["d2"] > 0 and L["sizes"].max() <= G2_MAXM
            assert np.split(L["sizes"], L["nb1"])[-1].sum() > L["c1"]
        elif name == "oversized bucket":
            assert L["sizes"].max() > G2_MAXM
        elif name.startswith("full range"):
            gb = (len(o) - 2).bit_length()
            assert L["hb"] == 64 and L["d1"] >= gb
            assert (L["d1"] <= 11) == probe
            assert gb + L["rest_bits"] <= 53
        elif name == "narrow":
            assert L["rest_bits"] == 0 and L["sbits"] == 11


# ---- on the GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_schedule(gpu_ctx):
    rng = np.random.default_rng(34)
    # four final buckets, one CTA each: the CTAs of buckets 1 and 2 have nothing to probe
    h, o = bucket_db(20, 2, [1000, 0, 0, 1000], seed=30)
    assert probe_case(gpu_ctx, h, o, some_sample(h, rng, 600, 100, 20))
    h, o = schedule_db()
    check_schedule(h, o)
    # ~50 and ~260 sample hashes per bucket: pass 1 settles by the all-pairs scan, then by sub-buckets; pass 2 keeps every word
    # of a full bucket unless the mask picks a few genomes
    small, large = some_sample(h, rng, 60000, 5000), some_sample(h, rng, 300000, 0)
    for s, mask in ((small, None), (large, None), (small, (rng.random(211) < 0.05).astype(np.uint8))):
        assert probe_case(gpu_ctx, h, o, s, mask)
    tm = partition_timings(gpu_ctx, h, o, small)
    assert tm["ms_hist1"] == 0.0 and tm["ms_hist2"] > 0.0, tm     # level 2 ran again on the exact layout


@pytest.mark.gpu
@pytest.mark.parametrize("target", [RB_SMALL, RB_SMALL + 1])
def test_settlement_boundary(gpu_ctx, target):
    h, o, sample, mask = boundary_db(target, seed=32)
    check_boundary(h, o, sample, mask, target)
    assert probe_case(gpu_ctx, h, o, sample, mask)
    assert probe_case(gpu_ctx, h, o, sample)


@pytest.mark.gpu
@pytest.mark.parametrize("count", [RB_SCAP, RB_SCAP + 1])
@pytest.mark.parametrize("dups", [False, True])
def test_sample_capacity(gpu_ctx, count, dups):
    h, o, s = capacity_case(count, dups, seed=33)
    assert probe_case(gpu_ctx, h, o, s) == (count <= RB_SCAP)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c[0] for c in LAYOUTS])
def test_layouts(gpu_ctx, case):
    _, make, probe, hist1, hist2 = next(c for c in LAYOUTS if c[0] == case)
    h, o, s = make()
    assert probe_case(gpu_ctx, h, o, s) == probe
    if probe:
        tm = partition_timings(gpu_ctx, h, o, s)
        assert (tm["ms_hist1"] > 0.0, tm["ms_hist2"] > 0.0) == (hist1, hist2), tm


@pytest.mark.gpu
def test_residency_and_call_order(gpu_ctx):
    db = synth.make_reference_db(2000, seed=51, mean_size=1000, sd_size=300)
    s1, _, _ = synth.make_sample(db, seed=52, n_present=40, total_hashes=30000)
    assert expect_probe(db.hashes, db.offsets, s1)
    ctx = gpu_ctx

    def probe(sample, mask=None, rebuilt=False):
        ctx.reset_timers()
        got = ctx.exclusive_hashes(sample, mask)
        tm = ctx.timings()
        assert tm["ms_sample_kernels"] > 0.0 and (tm["ms_sort"] > 0.0) == rebuilt, tm
        exp = ro.exclusive_counts(db.hashes, db.offsets, sample, mask)
        for f in ("n_overlap", "nontrivial", "n_exclusive", "n_match"):
            assert np.array_equal(got[f], exp[f]), f

    ctx.load_sketches(db.hashes, db.offsets)
    probe(s1, rebuilt=True)                                 # builds the partition only
    with pytest.raises(YgpuError, match="build_index first"):
        ctx.pairwise_flag(THR)                              # ... which is no train index
    ctx.build_index()
    ref = to.oracle_train(db.hashes, db.offsets, THR)
    pairs = ctx.pairwise_flag(THR)
    assert np.array_equal(pairs["i"], ref.pairs["i"]) and np.array_equal(pairs["j"], ref.pairs["j"])
    assert np.array_equal(pairs["count"], ref.pairs["count"])
    probe(s1)                                               # the train index's partition serves the sample
    # samples growing, then shrinking, with and without a mask: scratch buffers are reused
    rng = np.random.default_rng(53)
    big = rng.permutation(synth.make_sample(db, seed=55, n_present=150, total_hashes=200000)[0])
    for k, size in enumerate((1000, 30000, len(big), 5000, 0, 80000)):
        mask = (rng.random(db.n) < 0.05).astype(np.uint8) if k % 2 else None
        probe(big[:size], mask)
    # another database of the same shape on the same context: the old partition must not answer
    db = synth.make_reference_db(2000, seed=54, mean_size=1000, sd_size=300)
    ctx.load_sketches(db.hashes, db.offsets)
    probe(s1, rebuilt=True)
    probe(s1)
