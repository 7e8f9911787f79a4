"""The databases of tests/test_group_routes_gpu.py have the shape they were built for (no GPU needed): plan values, the number
of final buckets on every grouping route, the bucket sizes at the kernels' class boundaries, the oversized route's chunks, the
CTA schedules k2_group meets, and every planting.  A GPU test that passed on a database that took another route than
intended would prove nothing about the route it names.

Also the plan's wide-key guard (msd_build: rest_bits > 32 and rest_bits - 32 + gb > 32 sends the database to the general
path) cannot fire: packing keeps hb - d1 + gb <= 64, and rest_bits > 32 needs key_bits >= 44, so sbits = 11 and
rest_bits = hb - d1 - d2 - 11 <= 53 - gb, i.e. rest_bits - 32 + gb <= 21."""
import numpy as np
import pytest

from harness import group_routes as gr

SMS = 148               # B200
GRIDS = (SMS * 4, SMS * 3, SMS * 2)     # k2_group: 4 CTAs per SM by its shared memory; fewer, should registers limit it

# name: (plan values, routes with group_kernel 0, routes with group_kernel 1 where they differ)
EXPECT = {
    "A": (dict(hb=55, gb=8, D=11, d1=6, d2=5, rest_bits=33, low_bits=52, index_path=1, m_lo=0, ord_cap=4096),
          dict(fast=924, slow=112, big=16, empty=996), None),
    "A1": (dict(hb=55, gb=8, D=11, d1=6, d2=5, rest_bits=33, low_bits=52, index_path=1, m_lo=0),
           dict(fast=1280, empty=768), None),
    "B": (dict(hb=40, gb=8, D=11, d1=6, d2=5, rest_bits=18, low_bits=37, index_path=1, m_lo=1022, ord_cap=1 << 27),
          dict(group2=600, fast=500, slow=140, big=8, empty=800), dict(fast=1100, slow=140, big=8, empty=800)),
    "C10": (dict(hb=64, gb=8, D=10, d1=8, d2=2, rest_bits=43, low_bits=62, index_path=1, m_lo=0, ord_cap=4),
            dict(fast=1012, big=11, empty=1), None),
    "C9": (dict(hb=64, gb=8, D=9, d1=8, d2=1, rest_bits=44, low_bits=63, index_path=1, m_lo=0, ord_cap=2),
           dict(fast=505, big=7), None),
    "D8": (dict(hb=64, gb=8, D=8, d1=8, d2=0, rest_bits=45, low_bits=64, index_path=0), None, None),
    "E": (dict(hb=55, gb=11, D=11, d1=6, d2=5, rest_bits=33, low_bits=55, index_path=1, m_lo=0),
          dict(fast=1100, slow=81, empty=867), None),
    "F": (dict(hb=40, gb=8, D=11, d1=6, d2=5, rest_bits=18, low_bits=37, index_path=1, m_lo=1022, hist1=False, hist2=False),
          dict(group2=2044, fast=2, slow=2), dict(fast=2046, slow=2)),
}
CHUNKS = {"A": [(0, 16)], "B": [(0, 8)], "C10": [(0, 4), (4, 8), (8, 11)], "C9": [(0, 2), (2, 4), (4, 6), (6, 7)]}
END_BITS = {"A": [56], "B": [40], "C10": [64, 64, 64], "C9": [64, 64, 64, 63]}

_cache = {}


def db(name):
    if name not in _cache:
        _cache[name] = gr.databases()[name]()
    return _cache[name]


def route_counts(r):
    return {k: int((r["route"] == k).sum()) for k in (gr.GROUP2, gr.FAST, gr.SLOW, gr.BIG, gr.EMPTY) if (r["route"] == k).any()}


def genome_of(x):
    return np.repeat(np.arange(x.n), np.diff(x.offsets.astype(np.int64)))


def test_plan_guard_never_fires():
    for hb in range(1, 65):
        for gb in range(22):
            for D in range(min(hb, 22) + 1):
                d1 = max(D if D <= 8 else (D + 1) // 2, hb + gb - 64)
                d2 = max(0, D - d1)
                if d1 > 11 or d1 > hb or d2 > 11:
                    continue
                key_bits = hb - d1 - d2
                rest_bits = key_bits - max(0, min(gr.SUBBITS, key_bits))
                assert rest_bits <= max(32, 53 - gb), (hb, gb, D)
                assert not (rest_bits > 32 and rest_bits - 32 + gb > 32), (hb, gb, D)
                assert gr.plan_bits(hb, gb, D) == (d1, d2, key_bits, key_bits - rest_bits, rest_bits)


def test_small_references_take_k2_group_with_wide_keys():
    # scaled 1 000 (hash width 55), N <= 2^20: every database of up to A_TARGET x 2^10 hashes plans D <= 11 and so leaves
    # 33+ remaining key bits: no bucket is k2_group2's
    for gb in range(21):
        for D in range(12):
            bits = gr.plan_bits(55, gb, D)
            assert bits is not None and bits[4] >= 33, (gb, D, bits)


@pytest.mark.parametrize("name", sorted(EXPECT))
def test_plan_and_routes(name):
    x = db(name)
    want, c0, c1 = EXPECT[name]
    assert (x.hb, x.D) == (want["hb"], want["D"])
    for kernel, counts in ((0, c0), (1, c1 or c0)):
        r = gr.routes(x.hashes, x.n, group_kernel=kernel)
        got = {k: r[k] for k in want if k != "m_lo" or kernel == 0}
        assert got == {k: v for k, v in want.items() if k != "m_lo" or kernel == 0}, (name, kernel)
        if want["index_path"] == 0:
            assert r["route"] is None and r["largest"] > gr.BK_CAP
            continue
        assert route_counts(r) == counts, (name, kernel)
        assert r["group_runs"] and r["group2_runs"] == (want["rest_bits"] <= 32 and kernel == 0)
        assert r["chunks"] == CHUNKS.get(name, []) and r["end_bits"] == END_BITS.get(name, [])
        assert r["big_buckets"] == sum(b - a for a, b in r["chunks"])
        if name not in ("F",):
            assert r["hist2"], name          # every database but F overflows its level-2 slots: the exact layout


def test_boundary_sizes_present():
    sizes = lambda name: set(gr.routes(db(name).hashes, db(name).n)["sizes"].tolist())
    for name in ("A", "B"):
        assert {1022, 1023, 1024, 1025, 3071, 3072, 3073} <= sizes(name), name
    assert {0, 1, 2, 900, 2048} <= sizes("A")
    f = gr.routes(db("F").hashes, db("F").n)
    assert [int(f["sizes"][b]) for b in sorted(gr.SLOT_BUCKETS)] == [gr.SLOT_BUCKETS[b] for b in sorted(gr.SLOT_BUCKETS)]
    assert f["sizes"][gr.SLOT_C2] == f["C2"] and f["sizes"].max() == f["C2"]
    assert len({b >> 5 for b in list(gr.SLOT_BUCKETS) + [gr.SLOT_C2]}) == 4        # four level-1 digits


@pytest.mark.parametrize("name,kernel", [("A", 0), ("B", 0), ("B", 1), ("E", 0)])
def test_cta_schedules(name, kernel):
    r = gr.routes(db(name).hashes, db(name).n, group_kernel=kernel)
    for grid in GRIDS:
        gr.assert_transitions(r, grid)


def test_twins():
    inverted = 0
    for name in ("A", "A1", "C10", "C9", "D8", "E"):
        x = db(name)
        r = gr.routes(x.hashes, x.n)
        kb, rb, gb = x.hb - x.D, r["rest_bits"], r["gb"]
        g = genome_of(x)
        routes = set()
        assert len(x.planted.twins) >= 4, name
        for b, ka, ga, kb_, gb_ in x.planted.twins:
            assert ka != kb_ and ka >> rb == kb_ >> rb                        # one sub-bucket
            assert ka & 0xFFFFFFFF == kb_ & 0xFFFFFFFF                        # equal low 32 remaining bits
            for k, gs in ((ka, ga), (kb_, gb_)):
                h = (b << kb) | k
                assert sorted(g[x.hashes == np.uint64(h)].tolist()) == gs, (name, hex(h))
            hi_a, hi_b = (ka & ((1 << rb) - 1)) >> 32, (kb_ & ((1 << rb) - 1)) >> 32
            inverted += any((p < q) != ((p | hi_a << gb) < (q | hi_b << gb)) for p in ga for q in gb_)
            if r["route"] is not None:
                routes.add(r["route"][b])
        if name == "A":
            assert routes == {gr.FAST, gr.SLOW, gr.BIG}
    assert inverted >= 6


def test_crowded_and_long_groups():
    for name in ("A", "A1", "B", "E", "F"):
        x = db(name)
        r = gr.routes(x.hashes, x.n)
        kb, rb = r["key_bits"], r["rest_bits"]
        b_of = gr.shr(x.hashes, kb).astype(np.int64)
        sub = ((x.hashes >> np.uint64(rb)) & np.uint64((1 << gr.SUBBITS) - 1)).astype(np.int64)
        for b, s, m in x.planted.crowded:
            assert ((b_of == b) & (sub == s)).sum() >= m, (name, b)
        g = genome_of(x)
        for b, k, gs in x.planted.long:
            assert sorted(g[x.hashes == np.uint64((b << kb) | k)].tolist()) == gs, (name, b)
    # A: a whole 3 072-word bucket under one digit, every genome's hash in a FAST and a SLOW bucket
    a = gr.routes(db("A").hashes, db("A").n)
    assert any(m == 3072 == a["sizes"][b] for b, _, m in db("A").planted.crowded)
    assert {a["route"][b] for b, _, gs in db("A").planted.long if len(gs) == 211} == {gr.FAST, gr.SLOW}
    # E: a 1 024-word bucket that is one group, and a group of all 2 039 genomes in a 3 072-word bucket of one digit
    e = gr.routes(db("E").hashes, db("E").n)
    lg = {len(gs): b for b, _, gs in db("E").planted.long}
    assert e["sizes"][lg[1024]] == 1024 and e["route"][lg[1024]] == gr.FAST
    assert e["sizes"][lg[2039]] == 3072 and e["route"][lg[2039]] == gr.SLOW
    assert (lg[2039], 3072 - 2039) in [(b, m) for b, _, m in db("E").planted.crowded]


@pytest.mark.parametrize("name", ["C10", "C9"])
def test_aliased_big_buckets(name):
    x = db(name)
    r = gr.routes(x.hashes, x.n)
    big = r["big_list"].tolist()
    assert sorted(x.planted.aliased) == big and len(big) >= 2 * r["ord_cap"] + 1
    ords = set(range(len(big)))
    assert {0, 1, r["ord_cap"] - 1, r["ord_cap"], r["ord_cap"] + 1, 2 * r["ord_cap"]} <= ords
    # identical words below the bucket digits: (remaining hash bits | genome id) multisets
    kmask = np.uint64((1 << r["key_bits"]) - 1)
    g = genome_of(x).astype(np.uint64)
    b_of = gr.shr(x.hashes, r["key_bits"]).astype(np.int64)
    words = [np.sort(((x.hashes[b_of == b] & kmask) << np.uint64(r["gb"])) | g[b_of == b]) for b in big]
    assert all(np.array_equal(words[0], w) for w in words[1:])


@pytest.mark.parametrize("name", sorted(EXPECT))
def test_in_sketch_duplicates_in_every_class(name):
    x = db(name)
    r = gr.routes(x.hashes, x.n)
    g = genome_of(x)
    dup = np.flatnonzero((x.hashes[1:] == x.hashes[:-1]) & (g[1:] == g[:-1]))
    assert len(dup), name
    if r["route"] is None:
        return
    b_of = gr.shr(x.hashes[dup], r["key_bits"]).astype(np.int64)
    classes = set(r["route"][b_of].tolist())
    present = set(r["route"].tolist()) - {gr.EMPTY}
    # buckets of 1 or 2 words hold no filler duplicate; every larger class does
    small = {gr.FAST} if name in ("F",) else set()
    assert present - small <= classes, (name, present, classes)
