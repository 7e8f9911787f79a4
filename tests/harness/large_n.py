"""Seeded databases of up to millions of genomes for the train step's large-N branches, built with numpy alone.

`synth.from_sketches` loops in Python per genome; here the (genome, hash) entries are generated as flat arrays and
grouped once.  Every sketch has 0-16 random background hashes below `max_hash`; planted hashes shared by chosen
member sets give the index its structure:

* special ids 0, 1, 2^19 - 1, 2^19, 2^20 - 1, 2^20 and N - 1 as the owner of a work item and as the follower in each of
  the three inline slots (a follower in slot e needs e + 1 smaller members before it: 0 only leads, 1 fills slot 0);
* groups of 2, 3, 4, 5 members (the inline / posting boundary L > 4) and of 65, 66 (64 and 65 followers);
* groups across column-tile boundaries (`tile_ws`);
* `wide`: rows holding three hashes of 1 500 other genomes each, all inside one column tile: > 4 096 distinct columns;
* `big`: one hash held by 3 500 genomes, an oversized final bucket;
* `twin`: two genomes with the same sketch of exactly `twin` hashes (65 535: a packed u16 counter reaches 0xFFFF);
* `dup`: some sketches hold a hash twice, the specials' planted hashes among them.

Members of the wide and big hashes get at least 10 background hashes, so a single shared hash stays below the
default threshold and the flagged pairs of a whole database stay in the hundreds of thousands.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Sequence

import numpy as np

from yacht_b200 import synth

WIDE_HOLDERS = 1500
BIG_HOLDERS = 3500


def special_ids(n: int) -> List[int]:
    return sorted({g for g in (0, 1, 2 ** 19 - 1, 2 ** 19, 2 ** 20 - 1, 2 ** 20, n - 1) if 0 <= g < n})


@dataclass
class LargeDB:
    db: synth.SketchDB
    groups: List[np.ndarray] = field(default_factory=list)   # planted member sets (ascending ids)
    wide_rows: List[int] = field(default_factory=list)
    big_members: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int64))
    twins: List[int] = field(default_factory=list)


def make_large_db(n: int, max_hash: int, seed: int, *, wide: bool = True, big: bool = True, dup: bool = False,
                  twin: int = 0, tile_ws: Sequence[int] = ()) -> LargeDB:
    rng = np.random.default_rng(seed)
    out = LargeDB(db=None)
    groups: List[np.ndarray] = []

    def pick(lo, hi, k):
        lo, hi = max(0, lo), min(n, hi)
        return rng.choice(np.arange(lo, hi), size=min(k, hi - lo), replace=False) if hi > lo else np.zeros(0, np.int64)

    spec = special_ids(n)
    for x in spec:
        for e in range(3):                                  # x in inline slot e of the item of the first member
            if x < e + 1:
                continue
            before = pick(0, x, e + 1) if x > 64 else np.arange(x - e - 1, x)
            after = pick(x + 1, x + 1 + 1000, int(rng.integers(0, 3 - e)))
            groups.append(np.concatenate([before, [x], after]))
        if x < n - 1:                                       # x as the owner of an item with 1-3 followers
            groups.append(np.concatenate([[x], pick(x + 1, x + 1 + 1000, int(rng.integers(1, 4)))]))
    for k in range(0, len(spec), 3):                        # the specials next to each other
        if len(spec[k:k + 4]) >= 2:
            groups.append(np.array(spec[k:k + 4]))
    for size in (2, 3, 4, 5):
        for _ in range(40):
            lo = int(rng.integers(0, n))
            groups.append(pick(lo, lo + 5000, size) if rng.random() < 0.5 else rng.choice(n, size=size, replace=False))
    for size in (65, 66):
        for _ in range(3):
            groups.append(rng.choice(n, size=size, replace=False))
        groups.append(pick(n - 2000, n, size))
        groups.append(pick(2 ** 20 - 1000, 2 ** 20 + 1000, size) if n > 2 ** 20 - 1000 else pick(0, 1000, size))
    for w in tile_ws:                                       # across the first, a middle and the last tile boundary
        bounds = list(range(w, n, w))
        for b in sorted({bounds[0], bounds[len(bounds) // 2], bounds[-1]} if bounds else set()):
            groups.append(np.arange(max(0, b - 2), min(n, b + 2)))
            groups.append(pick(b - 40, b + 40, 65))
    groups = [np.unique(np.asarray(g, dtype=np.int64)) for g in groups]
    groups = [g for g in groups if g.size >= 2]

    heavy = []                                              # (members, 1): one hash each
    if wide:
        w_min = min(tile_ws) if tile_ws else n
        for r in (3, w_min + 3):
            if r + 10 + 40000 > n:
                continue
            mem = pick(r + 10, r + 10 + 40000, 3 * WIDE_HOLDERS)
            for k in range(3):
                heavy.append(np.unique(np.concatenate([[r], mem[k * WIDE_HOLDERS:(k + 1) * WIDE_HOLDERS]])))
            out.wide_rows.append(r)
    if big:
        out.big_members = np.sort(rng.choice(n, size=BIG_HOLDERS, replace=False))
        heavy.append(out.big_members)

    # ---- entries: background, planted groups (1-3 common hashes each), heavy hashes ---------------------------------------
    bg = rng.integers(0, 17, size=n)
    for m in heavy:
        bg[m] = np.maximum(bg[m], 10)
    n_common = rng.integers(1, 4, size=len(groups))
    fresh = rng.integers(1, max_hash, size=int(bg.sum() + n_common.sum()) + len(heavy), dtype=np.uint64)
    fresh[0] = np.uint64(max_hash - 1)                     # the largest hash sets the hash width of the partition plan
    gid_parts = [np.repeat(np.arange(n, dtype=np.int64), bg)]
    h_parts = [fresh[:int(bg.sum())]]
    pos = int(bg.sum())
    for g, s in zip(groups, n_common):
        gid_parts.append(np.repeat(g, s))
        h_parts.append(np.tile(fresh[pos:pos + s], len(g)))
        pos += s
    for m in heavy:
        gid_parts.append(m)
        h_parts.append(np.full(len(m), fresh[pos], dtype=np.uint64))
        pos += 1
    gid = np.concatenate(gid_parts)
    hs = np.concatenate(h_parts)

    if dup:                                                 # the same hash twice inside a sketch
        k = np.concatenate([rng.choice(len(gid), size=2000, replace=False),
                            np.flatnonzero(np.isin(gid, spec) & (np.arange(len(gid)) >= int(bg.sum())))])
        gid, hs = np.concatenate([gid, gid[k]]), np.concatenate([hs, hs[k]])
    if twin:
        out.twins = [17, n - 2]
        keep = ~np.isin(gid, out.twins)
        th = rng.integers(1, max_hash, size=twin, dtype=np.uint64)
        gid = np.concatenate([gid[keep], np.repeat(np.array(out.twins, np.int64), twin)])
        hs = np.concatenate([hs[keep], np.tile(th, 2)])
    empty = n // 3                                          # an empty sketch among the others
    keep = gid != empty
    gid, hs = gid[keep], hs[keep]

    order = np.argsort(gid, kind="stable")
    offsets = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.bincount(gid, minlength=n), out=offsets[1:])
    out.db = synth.SketchDB(hashes=hs[order], offsets=offsets, cluster=np.full(n, -1, dtype=np.int64))
    out.groups = groups
    return out
