"""The general grouping kernel k2_group and the oversized-bucket route (k2_big_*) of the index build at their edges, bit for bit
against the dense CPU oracle.  The databases come from tests/harness/group_routes.py; tests/test_group_routes.py checks
without a GPU that each has the plan, routes and plantings named here.

* A  hb 55, D 11, N 211 (rest_bits 33: k2_group groups every bucket, m_lo 0): buckets of 1 022-1 025, 2 048, 3 071-3 073 and
     ~5 000 words; wide-key twins (equal low 32 remaining bits, different high bits beside the genome id) in FAST, SLOW and
     oversized buckets, a 3 072-word bucket under one sub-bucket digit, every genome's hash in a FAST and a SLOW bucket.
     The CTA schedules recomputed from the launch's grid meet FAST -> FAST (staged, also at exactly 1 024 words),
     SLOW -> FAST, skipped -> FAST, FAST -> SLOW and a first FAST bucket.
* A' the same with every bucket <= G2_MAXM words, the small-reference production case; also the run path's bucket probe.
* B  hb 40, D 11: all three routes in one build (k2_group2 <= 1 022, k2_group 1 023..3 072 with m_lo 1 022, oversized
     beyond), and with group_kernel 1 (k2_group takes everything up to 3 072).
* C  hb 64, D 10 / 9: low_bits 62 / 63, so the oversized route sorts in chunks of ord_cap 4 / 2 buckets (tag in bit 63 and a
     64-bit sort at D 9); 2 ord_cap + 3 oversized buckets with identical words below the bucket digits.
* D  hb 64, D 8: low_bits 64, one oversized bucket sends the whole database to the general path.
* E  hb 55, N 2 039: a 1 024-word bucket that is one group, a 3 072-word bucket of one sub-bucket with a 2 039-member group.
* F  buckets of 1 023, 1 024, 1 025 and exactly C2 words inside their level-2 slots (no histogram pass).

Every build is compared on n_distinct, n_singleton, n_index, n_postings, n_increments and has_duplicates, and on the flagged
pairs at threshold 0 (every shared count) and at 0.95^31 with both count kernels; which kernels and routes ran is read back
through ygpu_get_option ("last_group2_grid", "last_group_grid", "last_big_chunks")."""
import numpy as np
import pytest

from harness import group_routes as gr
from oracle import train_oracle as to
from test_run_buckets_gpu import probe_case, some_sample

pytestmark = pytest.mark.gpu

THR = 0.95 ** 31
STATS = ("n_distinct", "n_singleton", "n_index", "n_postings", "n_increments")

_dbs, _refs = {}, {}


def db(name):
    if name not in _dbs:
        _dbs[name] = gr.databases()[name]()
    return _dbs[name]


def refs(name):
    if name not in _refs:
        x = db(name)
        _refs[name] = {t: to.oracle_train(x.hashes, x.offsets, t) for t in (0.0, THR)}
    return _refs[name]


def has_duplicates(x):
    g = np.repeat(np.arange(x.n), np.diff(x.offsets.astype(np.int64)))
    return bool(np.any((x.hashes[1:] == x.hashes[:-1]) & (g[1:] == g[:-1])))


def same_pairs(got, ref):
    return (len(got) == len(ref) and np.array_equal(got["i"], ref["i"]) and np.array_equal(got["j"], ref["j"])
            and np.array_equal(got["count"], ref["count"]))


def check(ctx, name, group_kernel=0):
    """Build `name` with `group_kernel`, compare everything with the oracle and the mirror; returns (stats, mirror, grids)."""
    x = db(name)
    r = gr.routes(x.hashes, x.n, group_kernel=group_kernel)
    ref = refs(name)
    ctx.set_option("group_kernel", group_kernel)
    try:
        ctx.load_sketches(x.hashes, x.offsets)
        ctx.reset_timers()
        st = ctx.build_index()
        tm = ctx.timings()
        hooks = {k: ctx.get_option("last_" + k) for k in ("group2_grid", "group_grid", "big_chunks")}
        for thr, rf in ref.items():
            for ck in (1, 2):
                ctx.set_option("count_kernel", ck)
                got = ctx.pairwise_flag(thr)
                assert ctx.get_option("last_count_kernel") == ck
                assert same_pairs(got, rf.pairs), (name, group_kernel, thr, ck, len(got), len(rf.pairs))
    finally:
        ctx.set_option("group_kernel", 0)
        ctx.set_option("count_kernel", 0)
    rf = ref[THR]
    assert {f: st[f] for f in STATS} == {f: getattr(rf, f) for f in STATS}, (name, group_kernel, st)
    assert st["has_duplicates"] == has_duplicates(x) == 1
    assert (st["index_path"], st["big_buckets"]) == (r["index_path"], r["big_buckets"]), (name, st)
    assert (hooks["group2_grid"] > 0) == r["group2_runs"] and (hooks["group_grid"] > 0) == r["group_runs"], (name, hooks)
    assert hooks["big_chunks"] == len(r["chunks"]), (name, hooks, r["chunks"])
    if r["index_path"]:
        assert 0 < max(hooks["group2_grid"], hooks["group_grid"]) <= r["nb"]
        assert (tm["ms_hist1"] > 0.0, tm["ms_hist2"] > 0.0) == (r["hist1"], r["hist2"]), (name, tm)
    print(f"{name} group_kernel={group_kernel} T={len(x.hashes)} N={x.n} {hooks} index_path={st['index_path']} "
          f"big_buckets={st['big_buckets']} pairs@0={len(ref[0.0].pairs)}")
    return st, r, hooks


def test_wide_keys_every_class(gpu_ctx):
    st, r, hooks = check(gpu_ctx, "A")
    assert hooks["group2_grid"] == 0 and r["m_lo"] == 0
    print(dict(gr.assert_transitions(r, hooks["group_grid"])))


def test_wide_keys_small_reference(gpu_ctx):
    st, r, hooks = check(gpu_ctx, "A1")
    assert hooks["group2_grid"] == 0 and r["largest"] <= gr.G2_MAXM
    x = db("A1")
    rng = np.random.default_rng(7)
    sample = some_sample(x.hashes, rng, 40000, extra=20000, hb=55)
    twins = [(b << (x.hb - x.D)) | ka for b, ka, _, _, _ in x.planted.twins]      # one hash of each twin pair
    sample = rng.permutation(np.concatenate([sample, np.array(twins, dtype=np.uint64)]))
    assert probe_case(gpu_ctx, x.hashes, x.offsets, sample)                    # the bucket probe answered


@pytest.mark.parametrize("group_kernel", [0, 1])
def test_three_routes(gpu_ctx, group_kernel):
    st, r, hooks = check(gpu_ctx, "B", group_kernel)
    assert r["m_lo"] == (1022 if group_kernel == 0 else 0)
    print(dict(gr.assert_transitions(r, hooks["group_grid"])))


def test_three_routes_kernels_agree(gpu_ctx):
    x = db("B")
    out = []
    for kernel in (0, 1):
        gpu_ctx.set_option("group_kernel", kernel)
        try:
            gpu_ctx.load_sketches(x.hashes, x.offsets)
            st = gpu_ctx.build_index()
            out.append((st, gpu_ctx.pairwise_flag(0.0), gpu_ctx.pairwise_flag(THR)))
        finally:
            gpu_ctx.set_option("group_kernel", 0)
    assert out[0][0] == out[1][0]
    assert out[0][1].tobytes() == out[1][1].tobytes() and out[0][2].tobytes() == out[1][2].tobytes()


@pytest.mark.parametrize("name", ["C10", "C9"])
def test_big_route_across_chunks(gpu_ctx, name):
    st, r, hooks = check(gpu_ctx, name)
    assert hooks["big_chunks"] >= 3 and st["big_buckets"] >= 2 * r["ord_cap"] + 1


def test_low_bits_64_takes_the_general_path(gpu_ctx):
    st, r, hooks = check(gpu_ctx, "D8")
    assert st["index_path"] == 0 and hooks == {"group2_grid": 0, "group_grid": 0, "big_chunks": 0}


def test_long_groups(gpu_ctx):
    st, r, hooks = check(gpu_ctx, "E")
    assert hooks["group2_grid"] == 0


@pytest.mark.parametrize("group_kernel", [0, 1])
def test_slotted_general_kernel_buckets(gpu_ctx, group_kernel):
    st, r, hooks = check(gpu_ctx, "F", group_kernel)
    assert not r["hist1"] and not r["hist2"]
