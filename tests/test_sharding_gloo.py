"""N > 1 host logic on CPU: world_size-2 gloo run of the row sharding + pair-list gather
(the same code path bench.py and multi-GPU callers use with NCCL on device tensors)."""
import multiprocessing
import os
import socket

import numpy as np
import pytest

from yacht_b200 import sharding, synth
from yacht_b200._lib import PAIR_DTYPE


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import train_oracle as to
        db = synth.make_reference_db(300, 17, mean_size=200, sd_size=60)
        full = to.oracle_train(db.hashes, db.offsets, 0.3).pairs
        full3 = np.zeros(len(full), dtype=PAIR_DTYPE)
        for f in ("i", "j", "count"):
            full3[f] = full[f]
        bounds = sharding.split_rows_by_work(db.sizes.astype(np.float64), world)
        mine = sharding.owned_pairs(full3, int(bounds[rank]), int(bounds[rank + 1]))
        merged = sharding.all_gather_pairs(mine, len(mine), world)
        ok = merged.tobytes() == np.sort(full3, order=["i", "j"]).tobytes()
        # a rank with nothing to report must not break the exchange
        empty = sharding.all_gather_pairs(mine if rank == 0 else mine[:0], len(mine) if rank == 0 else 0, world)
        ok = ok and len(empty) == len(sharding.owned_pairs(full3, int(bounds[0]), int(bounds[1])))
        q.put((rank, bool(ok), len(mine), len(full3)))
    finally:
        dist.destroy_process_group()


def test_two_rank_gather_matches_single_rank():
    # torch is imported in the spawned workers only: after the library's multi-GPU calls this process holds the NCCL the
    # loader found first, which need not be the one torch was built against
    ctx = multiprocessing.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), res
    assert sum(r[2] for r in res) == res[0][3]      # the shards partition the pair list
    assert all(r[2] > 0 for r in res)


def test_split_rows_by_work_properties():
    rng = np.random.default_rng(0)
    for n, parts in [(1000, 8), (5, 8), (0, 3), (97, 1)]:
        w = rng.integers(0, 1000, size=n).astype(np.float64)
        b = sharding.split_rows_by_work(w, parts)
        assert b[0] == 0 and b[-1] == n and np.all(np.diff(b.astype(np.int64)) >= 0)
        if n >= 100 * parts:
            loads = [float((w[b[k]:b[k + 1]] + sharding.ROW_CONSTANT).sum()) for k in range(parts)]
            assert max(loads) < 1.3 * (sum(loads) / parts)


def test_slice_bounds_and_size_split():
    b = sharding.slice_bounds(10, 4)
    assert b.tolist() == [0, 3, 6, 9, 10]
    assert sharding.slice_bounds(0, 3).tolist() == [0, 0, 0, 0]
    assert sharding.slice_bounds(8, 1).tolist() == [0, 8]
    off = np.array([0, 10, 10, 30, 60, 100], dtype=np.uint64)   # sizes 10, 0, 20, 30, 40
    r = sharding.split_rows_by_size(off, 2)
    assert r[0] == 0 and r[-1] == 5 and 0 < r[1] < 5
    sizes = np.diff(off.astype(np.int64))
    assert abs(int(sizes[:r[1]].sum()) - int(sizes[r[1]:].sum())) <= int(sizes.max()) + 2 * int(sharding.ROW_CONSTANT)


# ---- the sharded index build's exchange plan (host mirror of csrc/index_msd.cu: k2s_prep) -------------------------------
D1 = 7          # leading hash bits of the toy exchange


def _digits(h):
    return (np.asarray(h, dtype=np.uint64) >> np.uint64(55 - D1)).astype(np.int64)


def _check_plan(db, world, hists, plan):
    nb = hists.shape[1]
    owner, start, count = plan["owner"], plan["start"], plan["count"]
    assert np.all(np.diff(owner) >= 0) and owner.min() >= 0 and owner.max() < world          # contiguous digit ranges, rank order
    assert count.sum() == int(db.offsets[-1])
    cap = sharding.exchange_capacity(int(db.offsets[-1]), world, nb)
    assert count.max() <= cap                                                                # the buffer bound the library allocates
    # the (source, digit) ranges tile every owner's buffer exactly once, digit-major and source-minor
    for o in range(world):
        segs = sorted((int(start[r, d]), int(hists[r, d])) for d in np.flatnonzero(owner == o) for r in range(world) if hists[r, d])
        pos = 0
        for st, ln in segs:
            assert st == pos
            pos += ln
        assert pos == count[o]


def _plan_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        db = synth.make_reference_db(400, 23, mean_size=300, sd_size=90)
        bounds = sharding.split_rows_by_size(db.offsets, world)
        lo, hi = int(db.offsets[bounds[rank]]), int(db.offsets[bounds[rank + 1]])
        mine = db.hashes[lo:hi]
        nb = int(_digits([synth.MAX_HASH - 1])[0]) + 1
        h = torch.from_numpy(np.bincount(_digits(mine), minlength=nb).astype(np.int64))
        allh = [torch.zeros_like(h) for _ in range(world)]
        dist.all_gather(allh, h)                                   # the library: ncclAllGather of the level-1 histograms
        hists = torch.stack(allh).numpy()
        plan = sharding.exchange_plan(hists)
        _check_plan(db, world, hists, plan)
        # carry the exchange out: every rank "stores" its words at plan positions; the owners end up with exactly the words
        # of their digits, grouped by digit
        sizes = [int(c) for c in plan["count"]]
        send = [np.zeros(0, dtype=np.uint64)] * world
        cursor = plan["start"][rank].copy()
        bufs_pos = [[] for _ in range(world)]
        bufs_val = [[] for _ in range(world)]
        for v, d in zip(mine.tolist(), _digits(mine).tolist()):
            o = int(plan["owner"][d])
            bufs_pos[o].append(int(cursor[d]))
            bufs_val[o].append(v)
            cursor[d] += 1
        gathered = [None] * world
        dist.all_gather_object(gathered, (bufs_pos, bufs_val))
        buf = np.zeros(sizes[rank], dtype=np.uint64)
        seen = np.zeros(sizes[rank], dtype=bool)
        for pos_r, val_r in gathered:
            p, v = np.array(pos_r[rank], dtype=np.int64), np.array(val_r[rank], dtype=np.uint64)
            assert not seen[p].any()
            buf[p] = v
            seen[p] = True
        ok = bool(seen.all()) and bool(np.all(np.diff(_digits(buf)) >= 0)) and bool(np.all(plan["owner"][_digits(buf)] == rank))
        want = np.sort(db.hashes[plan["owner"][_digits(db.hashes)] == rank])
        ok = ok and np.array_equal(np.sort(buf), want)
        q.put((rank, ok, sizes[rank]))
    finally:
        dist.destroy_process_group()


def test_exchange_plan_two_ranks():
    ctx = multiprocessing.get_context("spawn")           # torch only in the workers, as above
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_plan_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), res
    assert sum(r[2] for r in res) > 0


def test_exchange_plan_properties():
    rng = np.random.default_rng(9)
    for world in (1, 2, 3, 8):
        for nb in (1, 5, 64, 525):
            hists = rng.integers(0, 50, size=(world, nb))
            hists[:, rng.integers(0, nb)] += 400                      # one heavy digit
            if nb > 3:
                hists[:, 2] = 0                                       # an empty digit
            plan = sharding.exchange_plan(hists)

            class _Db:
                offsets = np.array([0, int(hists.sum())])
            _check_plan(_Db, world, hists, plan)
    z = sharding.exchange_plan(np.zeros((2, 4), dtype=np.int64))
    assert z["count"].tolist() == [0, 0] and z["total"] == 0


def test_hash_range_shares_partition_every_sketch():
    """hash-range residency (ygpu_load_sketches_hashrange): the ranks' shares are disjoint, cover every sketch, keep the order,
    and equal hashes land on one rank."""
    from yacht_b200 import sharding, synth
    db = synth.make_reference_db(300, 17, mean_size=400, sd_size=120)
    offsets = np.asarray(db.offsets)
    for nranks in (1, 2, 3, 8):
        cuts = sharding.hash_cuts(int(db.hashes.max()), nranks)
        assert len(cuts) == nranks + 1 and cuts[0] == 0 and int(cuts[-1]) == 2 ** 64 - 1
        assert all(int(cuts[r]) <= int(cuts[r + 1]) for r in range(nranks))
        shares = [sharding.hashrange_share(db.hashes, offsets, int(cuts[r]), int(cuts[r + 1]), last=r == nranks - 1) for r in range(nranks)]
        assert sum(len(h) for h, _ in shares) == len(db.hashes)
        for g in range(0, db.n, 7):
            pieces = [h[int(o[g]):int(o[g + 1])] for h, o in shares]
            whole = db.hashes[int(offsets[g]):int(offsets[g + 1])]
            assert np.array_equal(np.concatenate(pieces), whole)          # sketches are sorted: the pieces concatenate back
            for r, piece in enumerate(pieces):
                if len(piece):
                    assert int(piece.min()) >= int(cuts[r])
                    assert int(piece.max()) < int(cuts[r + 1]) or r == nranks - 1
        sizes = [len(h) for h, _ in shares]
        assert max(sizes) - min(sizes) <= 0.1 * len(db.hashes) / nranks + 50      # uniform hashes: equal-width ranges balance


def test_hash_range_share_keeps_the_largest_hash_on_the_last_rank():
    from yacht_b200 import sharding
    hashes = np.array([0, 5, 2 ** 64 - 1, 7, 2 ** 64 - 1], dtype=np.uint64)
    offsets = np.array([0, 3, 5], dtype=np.uint64)
    cuts = sharding.hash_cuts(2 ** 64 - 1, 2)
    a = sharding.hashrange_share(hashes, offsets, int(cuts[0]), int(cuts[1]))
    b = sharding.hashrange_share(hashes, offsets, int(cuts[1]), int(cuts[2]), last=True)
    assert a[0].tolist() == [0, 5, 7] and a[1].tolist() == [0, 2, 3]
    assert b[0].tolist() == [2 ** 64 - 1, 2 ** 64 - 1] and b[1].tolist() == [0, 1, 2]
