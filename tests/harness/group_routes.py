"""msd_build's plan and grouping routes restated in plain Python (yacht_b200/csrc/index_msd.cu), and seeded databases whose
words fall into chosen final buckets, with plantings for the general grouping kernel k2_group and the oversized route.

The plan: hash width hb, genome-id width gb, the fewest leading hash bits D with T / used buckets <= A_TARGET, the two
partition levels d1 / d2 (packing: hb - d1 + gb <= 64), and below the final bucket's digits key_bits = hb - d1 - d2 hash
bits: an 11-bit sub-bucket digit (sbits) and rest_bits compared inside a sub-bucket.  A final bucket of m words goes to
  * k2_group2 when rest_bits <= 32 and 0 < m <= G2_MAXM (unless group_kernel = 1);
  * k2_group, GK_FAST (m <= 1 024, prefetched with cp.async when the CTA's previous bucket was grouped) or GK_SLOW
    (1 025 <= m <= BK_CAP), for every other bucket of 1..BK_CAP words;
  * the oversized route (k2_big_*) when m > BK_CAP: sorted in chunks of at most ord_cap = 2^(64 - low_bits) buckets,
    low_bits = key_bits + gb, unless low_bits = 64, which sends the whole database to the general sort path (index_path 0).
"""
from __future__ import annotations

import math
from collections import Counter
from dataclasses import dataclass, field
from typing import Dict, List

import numpy as np

A_TARGET = 900          # average words per used final bucket the plan aims at
N_GENOMES = 211         # prime: the members of a group, g0 + 7 k mod N, are distinct genomes
SC_TILE = 4096          # words per scatter tile
NB_MAX = 2048           # digits per partition level
SUBBITS = 11            # sub-bucket digit of the grouping kernels
G2_MAXM = 1022          # largest bucket k2_group2 takes
GK_FAST_M = 1024        # largest bucket of k2_group's GK_FAST class (GK_FAST x GK_THREADS words)
BK_CAP = 3072           # largest bucket that fits shared memory

# routes of a final bucket
EMPTY, GROUP2, FAST, SLOW, BIG = "empty", "group2", "fast", "slow", "big"


def shr(x, s):
    return np.zeros_like(x) if s >= 64 else x >> np.uint64(s)


def slot_cap(T, maxkey, hb, bits, f, add):
    """slot_capacity: f x (expected words of a full bucket of `bits` leading hash bits) + add, rounded up to 16 words."""
    mean = float(T) * 2.0 ** (hb - bits) / (float(maxkey) + 1.0)
    return (math.ceil(f * mean + add) + 15) // 16 * 16


def plan_bits(hb, gb, D):
    """(d1, d2, key_bits, sbits, rest_bits) of msd_build for these widths, or None where it leaves the database to the
    general path before looking at bucket sizes (no packing, or a sub-bucket key too wide for the candidate arrays)."""
    d1 = D if D <= 8 else (D + 1) // 2
    d1 = max(d1, hb + gb - 64)
    if d1 > 11 or d1 > hb:
        return None
    d2 = max(0, D - d1)
    if d2 > 11:
        return None
    key_bits = hb - d1 - d2
    sbits = max(0, min(SUBBITS, key_bits))
    rest_bits = key_bits - sbits
    if rest_bits > 32 and rest_bits - 32 + gb > 32:
        return None
    return d1, d2, key_bits, sbits, rest_bits


def plan(hashes, n):
    """msd_build's partition plan: (hb, d1, d2, C1, C2)."""
    T = len(hashes)
    maxkey = int(hashes.max())
    hb = max(1, maxkey.bit_length())
    D = 0
    while D < hb and D < 22 and T // ((maxkey >> (hb - D)) + 1 if D else 1) > A_TARGET:
        D += 1
    d1 = max(D if D <= 8 else (D + 1) // 2, hb + (n - 1).bit_length() - 64)      # packing: hb - d1 + gb <= 64
    d2 = max(0, D - d1)
    return hb, d1, d2, slot_cap(T, maxkey, hb, d1, 1.02, SC_TILE), slot_cap(T, maxkey, hb, d1 + d2, 1.25, 64.0)


def routes(hashes, n, group_kernel=0, big_buckets=1):
    """Everything msd_build decides for a database: the plan, the route of every final bucket, the oversized route's chunks,
    the layout (which histogram passes run) and the index path.  `route` is None when the general path builds the index."""
    T = len(hashes)
    hb, d1, d2, C1, C2 = plan(hashes, n)
    maxkey = int(hashes.max())
    gb = (n - 1).bit_length()
    D = 0
    while D < hb and D < 22 and T // ((maxkey >> (hb - D)) + 1 if D else 1) > A_TARGET:
        D += 1
    r = dict(T=T, hb=hb, gb=gb, D=D, d1=d1, d2=d2, C1=C1, C2=C2, index_path=0, big_buckets=0, route=None, chunks=[],
             ord_cap=0, end_bits=[], group2_runs=False, group_runs=False, m_lo=0)
    bits = plan_bits(hb, gb, D)
    nb1 = (maxkey >> (hb - d1)) + 1 if d1 else 1
    if T < 2 or n < 2 or bits is None or nb1 > NB_MAX:
        return r
    _, _, key_bits, sbits, rest_bits = bits
    nb = nb1 << d2
    sizes = np.bincount(shr(np.asarray(hashes, np.uint64), key_bits).astype(np.int64), minlength=nb)
    low_bits = key_bits + gb
    largest = int(sizes.max())
    r.update(nb1=nb1, nb=nb, key_bits=key_bits, sbits=sbits, rest_bits=rest_bits, low_bits=low_bits, sizes=sizes,
             largest=largest)
    # layout: slotted unless a slot overflows (or slot positions would not fit 32 bits)
    slots_fit = C1 * nb1 + T < 2 ** 32 and (not d2 or C2 * (nb1 << d2) + T < 2 ** 32)
    over1 = sizes.reshape(nb1, 1 << d2).sum(axis=1).max() > C1
    over2 = d2 and sizes.max() > C2
    r["hist1"] = not slots_fit or bool(over1)
    r["hist2"] = bool(d2) and (r["hist1"] or bool(over2))
    big = np.flatnonzero(sizes > BK_CAP)
    if len(big) and (not big_buckets or low_bits >= 64):
        return r
    fast2 = rest_bits <= 32 and group_kernel != 1
    m_lo = G2_MAXM if fast2 else 0
    route = np.full(nb, EMPTY, dtype=object)
    if fast2:
        route[(sizes > 0) & (sizes <= G2_MAXM)] = GROUP2
    route[(sizes > m_lo) & (sizes <= GK_FAST_M)] = FAST
    route[(sizes > max(m_lo, GK_FAST_M)) & (sizes <= BK_CAP)] = SLOW
    route[big] = BIG
    r.update(index_path=1, route=route, m_lo=m_lo, big_buckets=len(big), group2_runs=fast2,
             group_runs=not fast2 or largest > G2_MAXM)
    if len(big):
        ord_cap = 0x7FFFFFFF if 64 - low_bits >= 31 else 1 << (64 - low_bits)
        cstart = np.concatenate([[0], np.cumsum(sizes[big])])
        c0 = 0
        while c0 < len(big):
            c1 = c0
            while c1 < len(big) and c1 - c0 < ord_cap and cstart[c1 + 1] - cstart[c0] < 2 ** 30:
                c1 += 1
            c1 = max(c1, c0 + 1)
            r["chunks"].append((c0, c1))
            r["end_bits"].append(min(64, low_bits + (c1 - c0 - 1).bit_length()))
            c0 = c1
        r.update(ord_cap=ord_cap, big_list=big)
    return r


def transitions(r, grid):
    """k2_group's schedule: CTA c groups final buckets c, c + grid, ...  Counts of what a CTA meets, as k2_group sees its
    buckets: FAST, SLOW, or skipped (empty, oversized, or left to k2_group2).  A FAST bucket right after a bucket the CTA
    grouped was prefetched ("staged")."""
    cls = np.where(r["route"] == FAST, FAST, np.where(r["route"] == SLOW, SLOW, "skip"))
    sizes = r["sizes"]
    t = Counter()
    for c in range(min(grid, r["nb"])):
        seq = range(c, r["nb"], grid)
        t["first_" + cls[c]] += 1
        for p, b in zip(seq, seq[1:]):
            t[f"{cls[p]}>{cls[b]}"] += 1
            if cls[b] == FAST and cls[p] != "skip" and sizes[b] == GK_FAST_M:
                t["staged_1024"] += 1
    return t


def assert_transitions(r, grid, at_least=3):
    t = transitions(r, grid)
    for k in ("fast>fast", "slow>fast", "skip>fast", "fast>slow", "first_fast", "staged_1024"):
        assert t[k] >= at_least, (grid, k, dict(t))
    return t


# ---- databases ------------------------------------------------------------------------------------------------------------
def _fill(rng, b, m, shift, n):
    """m words of bucket b: hashes held by 1..12 genomes (mostly 1 or 2, as in real databases), about 1 % of the words
    repeating their neighbour's (hash, genome): in-sketch duplicates."""
    L = rng.choice([1, 2, 3, 4, 6, 12], size=m, p=[0.60, 0.25, 0.08, 0.04, 0.02, 0.01])
    L = L[:np.searchsorted(np.cumsum(L), m) + 1]
    L[-1] -= int(L.sum()) - m
    grp = np.repeat(np.arange(len(L)), L)
    rank = np.arange(m) - np.repeat(np.cumsum(L) - L, L)
    h = (np.uint64(b) << np.uint64(shift)) + rng.integers(0, 1 << shift, size=len(L), dtype=np.uint64)[grp]
    g = (rng.integers(0, n, size=len(L))[grp] + 7 * rank) % n
    dup = np.flatnonzero(rng.random(m) < 0.01)
    dup = dup[dup > 0]
    h[dup], g[dup] = h[dup - 1], g[dup - 1]
    return h, g


def csr(h, g, n):
    order = np.lexsort((h, g))
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(np.bincount(g, minlength=n))
    return np.asarray(h, np.uint64)[order], offsets


def bucket_db(hb, D, sizes, seed, n=N_GENOMES, plant=None):
    """Sketches whose words fall into final bucket b = hash >> (hb - D) exactly sizes[b] times.  plant: {bucket: (keys,
    genomes)}: words placed in that bucket, key = the hash bits below the bucket digits; the rest of the bucket is filler
    (_fill)."""
    assert len(sizes) == 1 << D and sizes[-1] > 0          # the last bucket sets the hash width hb
    T = int(sum(sizes))
    assert A_TARGET * (1 << D) >= T > A_TARGET * (1 << (D - 1)), "the plan would pick another bucket count"
    plant = plant or {}
    rng = np.random.default_rng(seed)
    shift = hb - D
    hs, gs = [], []
    for b, m in enumerate(sizes):
        if not m:
            continue
        keys, gen = plant.get(b, ((), ()))
        keys, gen = np.asarray(keys, np.uint64), np.asarray(gen, np.int64)
        assert len(keys) <= m and (shift == 64 or int(keys.max(initial=0)) >> shift == 0)
        if m > len(keys):
            h, g = _fill(rng, b, m - len(keys), shift, n)
            hs.append(h)
            gs.append(g)
        hs.append((np.uint64(b) << np.uint64(shift)) + keys if shift < 64 else keys)
        gs.append(gen)
    return csr(np.concatenate(hs), np.concatenate(gs), n)


@dataclass
class Planted:
    """What a database was built to contain (checked against the generated words by tests/test_group_routes.py)."""
    twins: List[tuple] = field(default_factory=list)     # (bucket, key A, genomes A, key B, genomes B)
    crowded: List[tuple] = field(default_factory=list)   # (bucket, sub-bucket digit, words)
    long: List[tuple] = field(default_factory=list)      # (bucket, key, genomes)
    aliased: List[int] = field(default_factory=list)     # oversized buckets with identical words below the bucket digits


class Plants:
    """Collects plantings per bucket (keys below the bucket digits, genomes) for bucket_db."""

    def __init__(self, rng, key_bits, n):
        self.rng, self.key_bits, self.n = rng, key_bits, n
        self.rest_bits = key_bits - SUBBITS
        self.by_bucket: Dict[int, tuple] = {}
        self.info = Planted()

    def add(self, b, keys, genomes):
        k0, g0 = self.by_bucket.get(b, (np.zeros(0, np.uint64), np.zeros(0, np.int64)))
        self.by_bucket[b] = (np.concatenate([k0, np.asarray(keys, np.uint64)]), np.concatenate([g0, np.asarray(genomes, np.int64)]))

    def words(self, b):
        return len(self.by_bucket.get(b, ((),))[0])

    def twins(self, b):
        """Four pairs of different hashes in one sub-bucket whose remaining keys agree in their low 32 bits and differ above:
        held by overlapping genome sets; by sets whose G2 words (genome | high bits << gb) order against the genome ids;
        by one genome each (both singletons); and by one genome that holds one of them twice (an in-sketch duplicate)."""
        assert self.rest_bits > 32
        rng, n = self.rng, self.n
        hi_max = 1 << (self.rest_bits - 32)
        for v in range(4):
            sub = int(rng.integers(0, 1 << SUBBITS))
            lo = int(rng.integers(0, 1 << 32))
            ha, hb_ = (1, 0) if hi_max == 2 else sorted(rng.choice(hi_max, size=2, replace=False).tolist(), reverse=True)
            base = int(rng.integers(0, n - 8))
            if v == 0:
                ga, gb_ = [base, base + 3, base + 5], [base + 3, base + 5, base + 7]
            elif v == 1:        # the key with the larger high bits is held by the smaller genome ids
                ga, gb_ = [0, 1, 2], [1, n - 2, n - 1]
            elif v == 2:
                ga, gb_ = [base], [base + 1]
            else:
                ga, gb_ = [base, base, base + 2], [base]
            ka = (sub << self.rest_bits) | (ha << 32) | lo
            kb = (sub << self.rest_bits) | (hb_ << 32) | lo
            self.add(b, [ka] * len(ga) + [kb] * len(gb_), ga + gb_)
            self.info.twins.append((b, ka, sorted(ga), kb, sorted(gb_)))

    def crowded(self, b, m, sub=None):
        """m filler words of one sub-bucket digit."""
        sub = int(self.rng.integers(0, 1 << SUBBITS)) if sub is None else sub
        h, g = _fill(self.rng, sub, m, self.rest_bits, self.n)
        self.add(b, h, g)
        self.info.crowded.append((b, sub, m))
        return sub

    def long(self, b, genomes, sub=None):
        """One hash held by every genome in `genomes`."""
        sub = int(self.rng.integers(0, 1 << SUBBITS)) if sub is None else sub
        k = (sub << self.rest_bits) | int(self.rng.integers(0, 1 << min(self.rest_bits, 62)))
        self.add(b, [k] * len(genomes), genomes)
        self.info.long.append((b, k, sorted(int(x) for x in genomes)))

    def aliased(self, buckets, m):
        """The same m words (filler below the bucket digits) in every bucket of `buckets`."""
        h, g = _fill(self.rng, 0, m, self.key_bits, self.n)
        for b in buckets:
            self.add(b, h, g)
        self.info.aliased.extend(int(b) for b in buckets)


@dataclass
class RouteDB:
    name: str
    hashes: np.ndarray
    offsets: np.ndarray
    n: int
    hb: int
    D: int
    planted: Planted


def _sizes(rng, D, counts, fill=0):
    """2^D bucket sizes: counts {size: buckets} in seeded random order, the rest `fill`; the last bucket is not empty."""
    sizes = [s for s, c in counts.items() for _ in range(c)]
    sizes += [fill] * ((1 << D) - len(sizes))
    sizes = rng.permutation(np.array(sizes, dtype=np.int64))
    if sizes[-1] == 0:
        j = int(np.flatnonzero(sizes)[-1])
        sizes[-1], sizes[j] = sizes[j], 0
    return sizes


def _first(sizes, m, k=0):
    """The k-th bucket of m words."""
    return int(np.flatnonzero(sizes == m)[k])


def _db(name, hb, D, n, sizes, P, seed):
    h, o = bucket_db(hb, D, [int(s) for s in sizes], seed=seed, n=n, plant=P.by_bucket)
    return RouteDB(name, h, o, n, hb, D, P.info)


def wide_every_class(seed=101):
    """A: hb 55, D 11 (key_bits 44, rest_bits 33: k2_group groups every bucket, m_lo 0), N 211.  Buckets of 0, 1, 2, 900,
    1 022-1 025, 2 048, 3 071-3 073 and 5 000 words in seeded random order; wide-key twins in FAST, SLOW and oversized
    buckets, a 3 072-word bucket under one sub-bucket digit, a crowded 1 024-word bucket, a hash of every genome in a FAST
    and in a SLOW bucket."""
    hb, D, n = 55, 11, N_GENOMES
    rng = np.random.default_rng(seed)
    sizes = _sizes(rng, D, {1: 100, 2: 100, 900: 500, 1022: 64, 1023: 64, 1024: 96, 1025: 48, 2048: 32, 3071: 16, 3072: 16,
                            3073: 8, 5000: 8})
    P = Plants(rng, hb - D, n)
    for m in (900, 1024, 1025, 3072, 5000):
        P.twins(_first(sizes, m))
    P.crowded(_first(sizes, 3072, 1), 3072)
    P.crowded(_first(sizes, 1024, 1), 1000)
    P.long(_first(sizes, 1023), range(n))
    P.long(_first(sizes, 3071), range(n))
    return _db("A", hb, D, n, sizes, P, seed)


def wide_small_reference(seed=102):
    """A': the same shape with every bucket <= G2_MAXM words, as every reference of up to ~945 000 hashes at scaled 1 000."""
    hb, D, n = 55, 11, N_GENOMES
    rng = np.random.default_rng(seed)
    sizes = _sizes(rng, D, {1: 100, 2: 100, 900: 1000, 1022: 80})
    P = Plants(rng, hb - D, n)
    P.twins(_first(sizes, 900))
    P.twins(_first(sizes, 1022))
    P.crowded(_first(sizes, 1022, 1), 1000)
    P.long(_first(sizes, 900, 1), range(n))
    return _db("A1", hb, D, n, sizes, P, seed)


def three_routes(seed=103):
    """B: hb 40, D 11 (rest_bits 18), N 211: k2_group2 takes <= 1 022 words, k2_group 1 023..3 072 (m_lo 1 022, a quarter
    of the buckets of 1 023 or 1 024 words), the oversized route the rest."""
    hb, D, n = 40, 11, N_GENOMES
    rng = np.random.default_rng(seed)
    sizes = _sizes(rng, D, {1: 100, 2: 100, 900: 300, 1022: 100, 1023: 250, 1024: 250, 1025: 60, 2048: 40, 3071: 20,
                            3072: 20, 3073: 4, 5000: 4})
    P = Plants(rng, hb - D, n)
    P.crowded(_first(sizes, 3072), 3072)
    P.crowded(_first(sizes, 1024), 1000)
    P.long(_first(sizes, 1023), range(n))
    P.long(_first(sizes, 1022), range(n))
    P.long(_first(sizes, 3073), range(n))
    return _db("B", hb, D, n, sizes, P, seed)


def big_chunks(D, seed):
    """C: hb 64, N 211 (d1 8 for packing), D 10 (low_bits 62, ord_cap 4) or D 9 (low_bits 63, ord_cap 2): 2 ord_cap + 3
    oversized buckets, all with the same words below the bucket digits, so ordinals 0, ord_cap, 2 ord_cap and their
    neighbours alias in any chunk one bucket too long; wide-key twins (rest_bits 43 / 44) and a hash of every genome in
    regular buckets."""
    hb, n = 64, N_GENOMES
    rng = np.random.default_rng(seed)
    nb = 1 << D
    ord_cap = 1 << (64 - (hb - D + (n - 1).bit_length()))
    sizes = rng.integers(0, 1001, size=nb)
    sizes[-1] = 500
    big = np.sort(rng.choice(np.arange(1, nb - 1), size=2 * ord_cap + 3, replace=False))
    sizes[big] = 3500
    P = Plants(rng, hb - D, n)
    P.aliased(big, 3500)
    reg = [b for b in range(nb - 1) if sizes[b] >= 600 and b not in set(big.tolist())]
    P.twins(reg[0])
    P.long(reg[1], range(n))
    return _db(f"C{D}", hb, D, n, sizes, P, seed)


def whole_fallback(seed=106):
    """D: hb 64, D 8, N 211: d2 0, low_bits 64 -- one oversized bucket sends the whole database to the general path."""
    hb, D, n = 64, 8, N_GENOMES
    rng = np.random.default_rng(seed)
    sizes = rng.integers(200, 1001, size=1 << D)
    sizes[int(rng.integers(0, 255))] = 4000
    P = Plants(rng, hb - D, n)
    P.twins(_first(sizes, 4000))
    return _db("D8", hb, D, n, sizes, P, seed)


N_LONG = 2039           # prime, gb 11: still packs at hb 55 (55 - 6 + 11 <= 64)


def long_groups(seed=107):
    """E: hb 55, D 11, N 2 039: a 1 024-word bucket that is one group of 1 024 genomes; a 3 072-word bucket that is one
    sub-bucket: a hash of all 2 039 genomes and 1 033 filler words; wide-key twins."""
    hb, D, n = 55, 11, N_LONG
    rng = np.random.default_rng(seed)
    sizes = _sizes(rng, D, {1: 100, 2: 100, 900: 600, 1022: 100, 1023: 100, 1024: 100, 1025: 50, 2048: 30, 3072: 1})
    P = Plants(rng, hb - D, n)
    P.long(_first(sizes, 1024), np.sort(rng.choice(n, size=1024, replace=False)))
    b = _first(sizes, 3072)
    sub = P.crowded(b, 3072 - n)
    P.long(b, range(n), sub=sub)
    P.twins(_first(sizes, 900))
    P.twins(_first(sizes, 1025))
    return _db("E", hb, D, n, sizes, P, seed)


SLOT_BUCKETS = {300: 1023, 900: 1024, 1100: 1025}      # in four different level-1 digits (32 final buckets each) ...
SLOT_C2 = 1700                                          # ... with the bucket of exactly C2 words


def slotted(seed=108, base=850):
    """F: hb 40, D 11 (d1 6, d2 5), N 211, buckets of `base` words and of 1 023, 1 024, 1 025 and exactly C2 words, all
    inside their level-2 slots.  C2 depends on the word count, which depends on C2: iterate to the fixed point."""
    hb, D, n = 40, 11, N_GENOMES
    sizes = np.full(1 << D, base)
    for b, m in SLOT_BUCKETS.items():
        sizes[b] = m
    sizes[SLOT_C2] = 1.25 * base + 64
    for _ in range(8):
        rng = np.random.default_rng(seed)
        P = Plants(rng, hb - D, n)
        P.long(900, range(n))
        P.crowded(SLOT_C2, 1000)
        x = _db("F", hb, D, n, sizes, P, seed)
        c2 = plan(x.hashes, n)[4]
        if sizes[SLOT_C2] == c2:
            return x
        sizes[SLOT_C2] = c2
    raise AssertionError("slot capacity did not settle")


def databases():
    """Every database of tests/test_group_routes_gpu.py, by name."""
    return {"A": wide_every_class, "A1": wide_small_reference, "B": three_routes, "C10": lambda: big_chunks(10, 104),
            "C9": lambda: big_chunks(9, 105), "D8": whole_fallback, "E": long_groups, "F": slotted}
