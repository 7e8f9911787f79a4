#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: genome-pair containments per second of the
`yacht train` hot path (inverted-index build + pairwise shared-hash count + threshold/compaction)
on a synthetic GTDB-representatives-shaped reference database (BASELINE.json configs[2]).

    python bench.py --gpus N --steps K --warmup W                  # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W # the reference's CPU core (oracle/_ref)
    torchrun ... bench.py --gpus N ...                             # N > 1: one rank per GPU (NCCL)
    python bench.py ... --dump-outputs DIR                         # + the last resident step's results as DIR/*.npy

One "step" = one pass of the hot path over the whole database:
  value : sketches already resident in HBM -> ygpu_build_index + ygpu_pairwise_flag (+ NCCL gather
          of the pair lists when N > 1); timed with CUDA events on the library's stream.
  e2e   : the same through the C ABI starting from pinned HOST buffers (H2D of all sketches inside
          the timed region) and ending with the flagged pair list on the host (D2H).
N > 1 is STRONG scaling: the same database, query rows sharded across ranks by work, index
replicated, compacted pair lists all-gathered over NCCL (north_star's partitioning).

Only the cpu_baseline leg and --impl reference execute anything under oracle/.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KSIZE = 31
ANI = 0.95
THR = ANI ** KSIZE
L2_BYTES = 126 * 1024 * 1024


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for l in self.proc.stdout:
            self.lines.append(l.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        self.sm, self.mx, self.reasons = sm, mx, reasons
        return self.summary(sm, mx, reasons)

    @staticmethod
    def summary(sm, mx, reasons) -> dict:
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(genomes: int, seed: int):
    from yacht_b200 import synth
    t0 = time.time()
    db = synth.make_reference_db(genomes, seed)
    return db, time.time() - t0


def independent_counts_torch(d_hashes, torch):
    """T, U2, P, W from the input alone (sort + run-length with torch ops, not with the library)."""
    s, _ = torch.sort(d_hashes)
    _, cnt = torch.unique_consecutive(s, return_counts=True)
    shared = cnt[cnt >= 2].to(torch.int64)
    return dict(T=int(d_hashes.numel()), U=int(cnt.numel()), U2=int(shared.numel()), P=int(shared.sum().item()),
                W=int((shared * shared).sum().item()))


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference core (oracle/_ref) -- or the oracle port when that binary is absent.
#   --impl reference : --steps runs of the unmodified reference executable on the FULL configuration (same genomes, same
#                      seed as the GPU arm): the database is written as signature files and the stock CLI is run with
#                      every host thread.  Throughput counts the phases that correspond to the GPU arm's e2e step (host
#                      buffers -> pair list + retained set): its own index + matrix + greedy timers; its JSON read
#                      phase is reported separately.
#   cpu_baseline     : (inside the GPU arm's line) a bounded sample of the same database, ~15 s of CPU work, labelled
#                      with the sample size -- a reported baseline, never used for a ratio.
# ------------------------------------------------------------------------------------------------
def cpu_arm_setup(db, n_sample: int):
    from oracle import train_oracle as to
    tmp = tempfile.mkdtemp(prefix="yacht_cpu_arm_")
    sub = db if n_sample >= db.n else db.subset(range(n_sample))
    to.write_sig_dir_parallel(sub, tmp)
    if to.reference_available():
        binary, kind = to.REF_BIN, "reference"
    else:
        to.build()
        binary, kind = to.PORT_BIN, "port"
    return tmp, binary, kind


def cpu_arm_step(tmp: str, binary: str, cores: int, passes: int = 1):
    from oracle import train_oracle as to
    for f in os.listdir(tmp):
        if f.endswith(".txt"):
            os.remove(os.path.join(tmp, f))
    out, wall = to.run_core_binary(binary, os.path.join(tmp, "training_sig_files.tsv"), tmp, THR, threads=cores, passes=passes)
    ph = to.parse_phase_times(out)
    return ph, wall


def choose_cpu_sample(db, budget_s: float) -> int:
    # measured (SURVEY.md section 6): ~8 ms of reference-core time per 5k-hash genome (index build
    # dominates: ~1.2-1.5 us per hash, single-threaded)
    per_genome = 8e-3 * (float(db.offsets[-1]) / max(db.n, 1)) / 5000.0
    return int(max(100, min(db.n, budget_s / max(per_genome, 1e-6))))


def mem_available_bytes() -> int:
    try:
        with open("/proc/meminfo") as f:
            for l in f:
                if l.startswith("MemAvailable:"):
                    return int(l.split()[1]) * 1024
    except Exception:
        pass
    return 0


def reference_plan(n: int, T: int):
    """Passes (-p) and the memory the reference core needs: ~100 B per distinct hash in its unordered_map of vectors plus a
    dense int matrix of ceil(n/p) x n (main.cpp:318-335).  Results do not depend on -p (SURVEY.md 8a)."""
    avail = mem_available_bytes()
    map_bytes = 110 * T
    passes = 1
    while passes < 64 and 4.0 * n * n / passes > max(0.15 * avail, 2e9):
        passes += 1
    need = map_bytes + 4.0 * n * n / passes + 8 * T
    return passes, need, avail


REF_CACHE = os.path.join(tempfile.gettempdir(), "yacht_b200_reference_arm_cache.json")


def reference_cache_key(args, binary: str, cores: int) -> str:
    try:
        stamp = f"{os.path.getsize(binary)}:{int(os.path.getmtime(binary))}"
    except OSError:
        stamp = "?"
    return (f"genomes={args.genomes} seed={args.seed} cpu_sample={args.cpu_sample} steps={args.steps} thr={THR!r} cores={cores} "
            f"binary={stamp}")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # The CPU arm does not depend on the number of GPUs, and one run of the reference core on the full configuration is ~7 minutes
    # of CPU: when the driver asks for it again on the same box (same configuration, same binary, same cores -- e.g. at every N of
    # a scaling run) the line of the first run is printed again, marked as such (--no-reference-cache measures again).
    from oracle import train_oracle as to
    binary0 = to.REF_BIN if to.reference_available() else to.PORT_BIN
    key = reference_cache_key(args, binary0, os.cpu_count() or 1)
    if not args.no_reference_cache and os.path.exists(REF_CACHE):
        try:
            with open(REF_CACHE) as f:
                cache = json.load(f)
            if key in cache:
                line = cache[key]
                line["n_gpus"] = args.gpus
                line["cached"] = {"from": line.get("measured_at"), "why": "same box, same configuration, same binary: the CPU arm does not depend on "
                                  "the GPU count; first measurement repeated verbatim (bench.py --no-reference-cache measures again)"}
                print(json.dumps(line), flush=True)
                return
        except Exception:
            pass
    db, gen_s = make_workload(args.genomes, args.seed)
    n, T = db.n, int(db.offsets[-1])
    cores = os.cpu_count() or 1
    passes, need, avail = reference_plan(n, T)
    full = not args.cpu_sample and (avail == 0 or need < 0.9 * avail)
    n_s = n if full else (args.cpu_sample or choose_cpu_sample(db, 120.0))
    t0 = time.time()
    tmp, binary, kind = cpu_arm_setup(db, n_s)
    write_s = time.time() - t0
    try:
        if not full:
            passes = 1
        # --steps timed runs (each minutes of CPU at full size), no warm-up; the phase timers are averaged over the runs
        runs = [cpu_arm_step(tmp, binary, cores, passes) for _ in range(args.steps)]
        ph = {k: sum(r[0].get(k, 0) for r in runs) / len(runs) for k in runs[-1][0]}
        wall = sum(r[1] for r in runs) / len(runs)
        per =(ph.get("index_ms", 0) + ph.get("matrix_ms", 0) + ph.get("greedy_ms", 0)) / 1e3 if ph else wall
        pairs = n_s * (n_s - 1)
        val = pairs / per if per > 0 else 0.0
        cfg = workload_config(args, db)
        sample = (f"{'ALL' if full else 'first'} {n_s} of {n} genomes (file order), all-vs-all, {os.path.basename(binary)} -t {cores} -p {passes}, "
                  f"{args.steps} run(s) (steps_run = {args.steps}, no warm-up: a run is minutes of CPU); time = the mean of its own "
                  f"index+matrix+greedy phase timers "
                  f"(JSON read phase {ph.get('read_ms', 0)} ms excluded: the GPU arm's e2e also starts from parsed arrays)")
        if not full:
            # not the same configuration: say so where the driver looks (config.genomes) and never publish a ratio from it
            cfg = dict(cfg, genomes=n_s, hashes=int(db.offsets[n_s]), same_config=False,
                       workload=cfg["workload"] + f" -- REFERENCE ARM RAN ONLY THE FIRST {n_s} GENOMES "
                                                    f"(host memory available {avail / 1e9:.0f} GB < {need / 1e9:.0f} GB needed)")
        line = {"impl": "reference", "metric": "ref-pair containments/s (yacht train hot path)", "value": val, "unit": "pairs/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_run": len(runs), "warmup_run": 0,
                "ms_per_step": per * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/int32 (+f64 threshold)",
                "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample,
                                 "phases_ms": ph, "wall_s": wall, "passes": passes, "write_sig_files_s": write_s,
                                 "generate_s": gen_s},
                "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if full:
            # the reference's own outputs of this very run against the committed digests (same check as the GPU arm)
            try:
                from oracle import train_oracle as to
                with open(os.path.join(tmp, "training_sig_files.tsv")) as f:
                    paths = [l.rstrip("\n") for l in f if l.strip()]
                got = to.parse_core_outputs(tmp, paths, os.path.join(tmp, "selected_result.tsv"), "")
                line["parity"] = check_digest(args, n, len(got.lines), lines=got.lines, selected=got.selected)
            except Exception as e:
                line["parity"] = {"error": repr(e)}
        line["measured_at"] = time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())
        print(json.dumps(line), flush=True)
        try:
            cache = {}
            if os.path.exists(REF_CACHE):
                with open(REF_CACHE) as f:
                    cache = json.load(f)
            cache[key] = line
            with open(REF_CACHE, "w") as f:
                json.dump(cache, f)
        except Exception:
            pass
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def find_digest(args, n: int):
    """The committed reference digest of this (genomes, seed) workload, if any (tests/golden/config_digests.json)."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "config_digests.json")) as f:
            digests = json.load(f)
    except Exception:
        return None, None
    for name, e in digests.items():
        g = e.get("generator", {})
        if set(g) == {"n", "seed"} and g["n"] == n and g["seed"] == args.seed and abs(e.get("threshold", -1) - THR) < 1e-15:
            return name, e
    return None, None


def check_digest(args, n, F, lines=None, pairs=None, sizes=None, selected=None):
    """Bit-exactness at the benchmarked size: F, sha256 of the sorted pair lines and of the retained ids against what the
    UNMODIFIED reference core produced for the same seeded database."""
    from yacht_b200 import pairfmt
    name, e = find_digest(args, n)
    if e is None:
        return {"parity_digest_ok": None, "why": "no committed reference digest for this (genomes, seed)"}
    if lines is None:
        lines = pairfmt.pair_lines(pairs, sizes)
    out = {"golden": f"tests/golden/config_digests.json[{name}] (unmodified reference core, {e.get('reference_cmd', '')})",
           "F": int(F), "F_ok": int(F) == e["F"], "pairs_sha256_ok": pairfmt.digest_lines(lines) == e["pairs_sha256"],
           "selected_sha256_ok": None if selected is None else pairfmt.digest_ids(selected) == e["selected_sha256"],
           "n_selected": None if selected is None else int(len(selected))}
    out["parity_digest_ok"] = bool(out["F_ok"] and out["pairs_sha256_ok"] and out["selected_sha256_ok"] is not False)
    return out


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir: str, stats: dict, pairs: np.ndarray) -> None:
    """What a caller of the train step receives, as float64 .npy files (every value is an integer below 2**53, so exact):
    index_stats = [n_distinct, n_singleton, n_index, flagged pairs]; pairs_i / pairs_j / pairs_count = the flagged ordered
    pairs in the library's (i, j) order.  A pair list over DUMP_BYTES is cut to a fixed, seeded sample of its rows, in order,
    so that two builds that flag the same pairs dump the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    cols = ("i", "j", "count")
    max_rows = (DUMP_BYTES - 4096) // (8 * len(cols))
    rows = slice(None)
    if len(pairs) > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(len(pairs), size=max_rows, replace=False))
    np.save(os.path.join(out_dir, "index_stats.npy"),
            np.array([stats["n_distinct"], stats["n_singleton"], stats["n_index"], len(pairs)], dtype=np.float64))
    for c in cols:
        np.save(os.path.join(out_dir, f"pairs_{c}.npy"), pairs[c][rows].astype(np.float64))


def workload_config(args, db):
    T = int(db.offsets[-1])
    return {"workload": f"synthetic GTDB-representatives-shaped reference DB (BASELINE.json configs[2]): {db.n} genomes, "
                        f"{T} hashes (mean {T / max(db.n, 1):.0f}/genome), planted ANI clusters, seed {args.seed}; "
                        f"all-vs-all train hot path, k={KSIZE}, ani_thresh={ANI}",
            "genomes": db.n, "hashes": T, "seed": args.seed, "containment_threshold": THR,
            "parallelism": "1 GPU" if args.gpus == 1 else
                           f"{args.gpus} GPUs, residency by {args.residency}: index build sharded by hash range, pairwise count sharded by query rows "
                           f"(work items stored into the row owners' buffers over NVLink by the grouping kernel), pair lists all-gathered (NCCL)",
            "l2": f"inputs {8 * T / 1e9:.2f} GB > L2 {L2_BYTES / 1e6:.0f} MB: no flush needed" if 8 * T > L2_BYTES
                  else "inputs fit L2: an L2 flush (write of 256 MB) runs before every timed step"}


# ------------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from yacht_b200 import _lib, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # stdout carries the one JSON line only (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    db, gen_s = make_workload(args.genomes, args.seed)
    n, T = db.n, int(db.offsets[-1])
    lib = _lib.load_library()
    ctx = _lib.GpuContext(local)

    offsets = np.ascontiguousarray(db.offsets, dtype=np.uint64)
    hp = pinned = d_hashes = d_offsets = None
    if world == 1:
        # pinned host staging for the e2e arm
        hp = lib.ygpu_host_alloc(max(T, 1) * 8)
        if not hp:
            raise SystemExit("ygpu_host_alloc failed")
        pinned = np.ctypeslib.as_array(ctypes.cast(hp, ctypes.POINTER(ctypes.c_uint64)), shape=(max(T, 1),))[:T]
        pinned[:] = db.hashes
    # device-resident copy (torch owns it; the library copies device-to-device once, outside the timed region); with N > 1
    # only rank 0 needs the whole array, for the implementation-independent workload counts, and drops it again
    counts = None
    if world == 1 or rank == 0:
        d_hashes = torch.from_numpy(db.hashes.view(np.int64)).to(dev)
        d_offsets = torch.from_numpy(offsets.view(np.int64)).to(dev)
        counts = independent_counts_torch(d_hashes, torch)
        if world > 1:
            d_hashes = d_offsets = None
            torch.cuda.empty_cache()
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if 8 * T <= L2_BYTES else None

    index_stats = {}
    mode = {"index": "single GPU"}
    row_bounds = sharding.split_rows_by_size(offsets, world)     # contiguous genome ranges of nearly equal hash counts
    g0, g1 = int(row_bounds[rank]), int(row_bounds[rank + 1])
    lo, hi = int(offsets[g0]), int(offsets[g1])
    pinned_slice = d_slice = None
    part_off = None
    sizes32 = db.sizes.astype(np.uint32)
    if world > 1:
        # N > 1: the library's own sharded step (C++ host layer + NCCL + stores into peer buffers over NVLink).
        #   residency "hashes" (default): every rank holds, of EVERY sketch, the hashes of its hash range -- the host cuts the sorted
        #     sketches at the same N - 1 values; equal hashes meet on one rank, so only work items ever cross NVLink;
        #   residency "genomes": every rank holds the sketches of its genome range; the level-1 scatter stores every packed word
        #     into the buffer of the rank that owns its hash range (an all-to-all over NVLink inside the kernel).
        # torch.distributed is used for the unique-id hand-over, the barrier around the timed region and the max over ranks,
        # nothing on the data path.
        uid = [_lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
        if args.residency == "hashes":
            cuts = sharding.hash_cuts(int(db.hashes.max()), world)
            mine, part_off = sharding.hashrange_share(db.hashes, offsets, int(cuts[rank]), int(cuts[rank + 1]), last=rank == world - 1)
            mode["index"] = ("hash-range residency (each rank holds its hash range of every sketch): partition and grouping are local, work items "
                             "go to the owners of the query rows over NVLink (stores from the grouping kernel); NCCL for lengths, statistics, pair lists")
        else:
            mine = db.hashes[lo:hi]
            mode["index"] = ("genome-range residency (each rank holds the sketches of its genomes): level-1 words and work items stored into the "
                             "owners' buffers over NVLink by the partition / grouping kernels; NCCL for histograms, lengths, statistics, pair lists")
        pinned_slice = torch.empty(max(len(mine), 1), dtype=torch.int64, pin_memory=True)
        pinned_slice.numpy()[: len(mine)] = mine.view(np.int64)
        d_slice = torch.from_numpy(np.ascontiguousarray(mine).view(np.int64)).to(dev)
        h2d_mine = 8 * len(mine)

    def load_sharded(ptr, on_device):
        if args.residency == "hashes":
            ctx.load_sketches_hashrange(ptr, part_off, sizes32, g0, g1, on_device=on_device)
        else:
            ctx.load_sketches_sharded_ptr(ptr, on_device, offsets, g0, g1)

    def step_resident():
        if world > 1:
            st, F = ctx.train_step_sharded(THR)
            index_stats.update(st)
            return F
        index_stats.update(ctx.build_index())
        return ctx.pairwise_flag_device(THR, 0, n)

    def step_e2e():
        if world > 1:
            load_sharded(pinned_slice.data_ptr(), False)
            st, F = ctx.train_step_sharded(THR)
            index_stats.update(st)
            return ctx.pairs_host(F)                       # every rank reads the complete, ordered pair list back
        ctx.load_sketches(pinned, offsets)
        index_stats.update(ctx.build_index())
        F = ctx.pairwise_flag_device(THR, 0, n)
        return ctx.pairs_host(F)

    clock_samples = []      # samplers of both timed regions (resident, e2e): the step is short, so their samples are pooled

    def timed(fn, reload_first: bool):
        if reload_first:
            if world > 1:
                load_sharded(d_slice.data_ptr(), True)
            else:
                ctx.load_sketches_device(d_hashes.data_ptr(), d_offsets.data_ptr(), n)
        for _ in range(args.warmup):
            if flush_buf is not None:
                flush_buf.fill_(1)
            fn()
        barrier()
        ctx.reset_timers()
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        total_ms = 0.0
        wall0 = time.perf_counter()
        res = None
        for _ in range(args.steps):
            if flush_buf is not None:
                flush_buf.fill_(1)
                torch.cuda.synchronize()
            ctx.mark(0)
            res = fn()
            ctx.mark(1)
            total_ms += ctx.elapsed_ms(0, 1)
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if sampler else None
        if sampler and getattr(sampler, "sm", None) is not None:
            clock_samples.append(sampler)
        tm = ctx.timings()
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / args.steps, tm, clocks, res, wall / args.steps

    ms_res, tm_res, clocks, n_flagged, wall_res = timed(step_resident, True)
    if args.dump_outputs:
        # the last resident step's results, read back outside the timed region; after the sharded step every rank holds the
        # whole list, so every rank reads it (as step_e2e does) and rank 0 writes it
        pairs_last = ctx.pairs_host(n_flagged)
        if rank == 0:
            dump_outputs(args.dump_outputs, index_stats, pairs_last)
    ms_e2e, tm_e2e, clocks_e2e, pairs_host, wall_e2e = timed(step_e2e, False)

    if rank == 0:
        pairs_total = n * (n - 1)
        F = int(len(pairs_host))
        peak, peak_src = load_peaks()
        # ---- rooflines (HBM): algorithmic bytes per launch / CUDA-event duration of that phase -----------
        launches = max(tm_res["n_count_launches"], 1)
        steps = args.steps
        share = 1.0 / world   # rows are split by work; a rank sees ~1/world of T and W in the count kernel
        st = index_stats
        k3_ms = tm_res["ms_count"] / launches
        part_ms = tm_res["ms_sort"] / steps
        bucket_ms = tm_res["ms_index"] / steps
        Tn, Wn, Pn, In = counts["T"], counts["W"], counts["P"], st["n_row_items"]
        msd = st["index_path"] == 1

        def rl(kernel, nbytes, ms, formula):
            ach = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            return {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": None, "algorithmic_bytes": nbytes, "formula": formula, "ms_per_launch": ms,
                    "share_of_step": ms / ms_res if ms_res else None, "peak_source": peak_src}

        rooflines = {
            "pairwise_count": rl("k3_count_flag (K3+K4: pairwise shared-hash count + threshold/compaction)",
                                 (8 * Tn + 4 * Wn + 12 * F) * share, k3_ms, "8*T + 4*W + 12*F (SURVEY.md 8d), x rank share"),
            "index_partition": rl("k2_hist1 + k2_scatter<1> + k2_hist2 + k2_scatter<2> (K2: MSD radix partition)" if msd
                                  else "CUB DeviceRadixSort of (hash, genome) pairs (general path)",
                                  48 * Tn / world if msd else 12 * Tn * 2 * 7, part_ms,
                                  ("8T + (8T+8T) + 8T + (8T+8T) = 48*T" + ("" if world == 1 else
                                   " /N: every rank partitions only its own slice; level-1 words are stored into the owners' buffers over NVLink")) if msd
                                  else "12*T*2*7 (SURVEY.md 8d)"),
            "index_grouping": rl("k2_group (K2: sub-bucket counting filter + dense candidate scan -> postings + per-genome work lists)" if msd
                                 else "k_flag_runs + scan + k_post_compact + k_items_scatter (general path)",
                                 (8 * Tn + 4 * Pn + 8 * In if world == 1 else (8 * Tn + 8 * In) / world + 12 * Pn) if msd
                                 else 12 * Tn + 4 * Pn + 16 * In, bucket_ms,
                                 ("8*T (words) + 4*P (postings) + 8*I (items)" if world == 1 else
                                  "this rank: 8*T/N words in, 6*P/N stream entries stored to each of N ranks (6*P out), 6*P complete stream in, "
                                  "8*I/N items (k2_group2<stream> + k2_items_regions + the control collectives)") if msd
                                 else "12*T + 4*P + 16*I"),
        }
        # DRAM traffic per launch from the committed `ncu --set full` captures (profiles/), when they were taken
        # on this very workload
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tr = json.load(f)
            if tr.get("genomes") == n and tr.get("seed") == args.seed and world == 1:
                for k in rooflines:
                    if k in tr.get("dram_bytes_per_launch", {}):
                        rooflines[k]["traffic"] = tr["dram_bytes_per_launch"][k]
                        rooflines[k]["traffic_source"] = tr.get("source")
        except Exception:
            pass
        rooflines["index_partition"]["kernels"] = 4          # a phase of four kernels: not a candidate for `roofline`
        if msd:
            # the partition phase kernel by kernel (CUDA events around each launch, ygpu_timings.ms_hist1 ...)
            wsh = 1.0 if world == 1 else 1.0 / world
            for key, kern, nbytes, formula in (
                    ("part_hist1", "k2_hist1 (level-1 digit histogram)", 8 * Tn * wsh, "8*T" + ("" if world == 1 else "/N")),
                    ("part_scatter1", "k2_scatter<1> (pack (hash, genome) words, scatter to level-1 buckets"
                                      + (")" if world == 1 else "; stores into the owner ranks' buffers over NVLink)"), 16 * Tn * wsh,
                     "8*T read + 8*T written" + ("" if world == 1 else ", /N")),
                    ("part_hist2", "k2_hist2 (level-2 digit histogram)", 8 * Tn * wsh, "8*T" + ("" if world == 1 else "/N")),
                    ("part_scatter2", "k2_scatter<2> (scatter to final buckets)", 16 * Tn * wsh, "16*T" + ("" if world == 1 else "/N"))):
                ms = tm_res["ms_" + key.split("_", 1)[1]] / steps
                if ms > 0:
                    rooflines[key] = rl(kern, nbytes, ms, formula)
            if tm_res.get("ms_group", 0) > 0 and world > 1:
                rooflines["index_grouping_k2_group"] = rl("k2_group2<stream> alone", 8 * Tn / world + 6 * Pn, tm_res["ms_group"] / steps,
                                                          "8*T/N words in + 6*P/N stream entries stored to each of the N ranks")
        dominant = max((r for r in rooflines.values() if r.get("kernels", 1) == 1), key=lambda r: r["ms_per_launch"])
        line = {
            "metric": "ref-pair containments/s (yacht train hot path)", "value": pairs_total / (ms_res * 1e-3), "unit": "pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/int32 (+f64 threshold)",
            "data": "synthetic", "config": workload_config(args, db),
            "e2e": {"value": pairs_total / (ms_e2e * 1e-3), "unit": "pairs/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": 8 * T + world * 8 * (n + 1), "d2h_bytes_per_step": 12 * F * world,
                    "ingest": "whole array from pinned host memory" if world == 1 else
                              f"each rank copies the sketches of its genome range (1/{world} of the hashes) over its own PCIe link; no raw all-gather",
                    "phases_ms": {k: tm_e2e[k] / steps for k in ("ms_h2d", "ms_sort", "ms_index", "ms_count", "ms_pairsort", "ms_d2h")}},
            "gpu_launches": int(tm_res["n_kernel_launches"]),
            "library_launches": int(tm_res["n_library_launches"]),
            "clocks": (dict(ClockSampler.summary([v for c in clock_samples for v in c.sm], [v for c in clock_samples for v in c.mx],
                                                 set().union(*[c.reasons for c in clock_samples])),
                            regions="resident + e2e timed regions pooled") if clock_samples else clocks),
            "roofline": dominant, "rooflines": rooflines, "index_path": "msd-partition" if msd else "general-sort",
            "index_mode": mode["index"],
            "phases_ms": {k: tm_res[k] / steps for k in ("ms_sort", "ms_index", "ms_count", "ms_pairsort", "ms_hist1", "ms_scatter1", "ms_hist2",
                                                           "ms_scatter2", "ms_group", "ms_items", "ms_sync", "ms_gather")},
            "workload_counts": dict(counts, F=F, genomes=n), "wall_ms_per_step": wall_res * 1e3, "gen_seconds": gen_s,
        }
        # ---- parity at the benchmarked size: the gathered pair list of the last e2e step against the reference digest ----
        try:
            sel = _lib.greedy_select(offsets, pairs_host)
            line["parity"] = check_digest(args, n, F, pairs=pairs_host, sizes=db.sizes, selected=sel)
            line["parity"]["n_flagged_resident_step"] = int(n_flagged)
        except Exception as e:
            line["parity"] = {"parity_digest_ok": False, "error": repr(e)}
        line["parity_digest_ok"] = line["parity"].get("parity_digest_ok")
        # ---- the run path (configs[4]) beside it: never allowed to take the train numbers down ------------
        if world == 1 and not args.no_run_path:
            try:
                if not ctx.n:
                    ctx.load_sketches(db.hashes, db.offsets)
                rp, rp_roof, rp_e2e = measure_run_path(ctx, lib, db, args, rl)
                line["run_path"], line["run_e2e"] = rp, rp_e2e
                rooflines["run_k5"] = rp_roof
            except Exception as e:
                line["run_path"] = {"error": repr(e)}
        # ---- CPU baseline: bounded sample on this box's host cores -------------------------------------
        if not args.no_cpu_baseline:
            try:
                cores = os.cpu_count() or 1
                n_s = args.cpu_sample or choose_cpu_sample(db, 15.0)
                tmp, binary, kind = cpu_arm_setup(db, n_s)
                try:
                    ph, wall = cpu_arm_step(tmp, binary, cores)
                finally:
                    shutil.rmtree(tmp, ignore_errors=True)
                t = (ph.get("index_ms", 0) + ph.get("matrix_ms", 0) + ph.get("greedy_ms", 0)) / 1e3 if ph else wall
                line["cpu_baseline"] = {"value": n_s * (n_s - 1) / max(t, 1e-9), "unit": "pairs/s", "cores": cores, "kind": kind,
                                        "sample": f"first {n_s} of {n} genomes (file order), all-vs-all, {os.path.basename(binary)} "
                                                  f"-t {cores} -p 1; time = its index+matrix+greedy phase timers",
                                        "sample_genomes": n_s, "same_config": n_s == n,
                                        "note": "pairs/s of the CPU core grows with N (its O(T) index build dominates): this bounded-sample figure is "
                                                "NOT comparable with the full-size GPU value; the same-config CPU number is the --impl reference arm",
                                        "phases_ms": ph, "wall_s": wall}
            except Exception as e:  # the baseline must never take the GPU numbers down with it
                line["cpu_baseline"] = {"value": None, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}
        print(json.dumps(line), flush=True)

    if hp:
        lib.ygpu_host_free(hp)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def measure_run_path(ctx, lib, db, args, rl):
    """BASELINE.json configs[4] beside the train step (N = 1 only): a synthetic 10 M-hash sample against the resident reference,
    min_coverage_list 1 0.6 0.2 0.1, significance 0.99 -- sample membership + exclusive hashes (K5, one call) and the hypothesis
    statistics (K6), through the C ABI from host buffers.  The CPU figure is the python-set RESTATEMENT of the reference's
    get_exclusive_hashes / single_hyp_test (oracle/run_oracle.py; sourmash's multisearch is not in this image) on a few genomes."""
    import ctypes
    from yacht_b200 import synth
    covs = [1.0, 0.6, 0.2, 0.1]
    n, T = db.n, int(db.offsets[-1])
    t0 = time.perf_counter()
    sample, _, _ = synth.make_sample(db, 5, n_present=min(2000, max(1, n // 4)), total_hashes=args.run_sample_hashes)
    gen_s = time.perf_counter() - t0
    hp = lib.ygpu_host_alloc(max(len(sample), 1) * 8)          # page-locked, as a host that read the sample from disk would stage it
    try:
        pinned = np.ctypeslib.as_array(ctypes.cast(hp, ctypes.POINTER(ctypes.c_uint64)), shape=(max(len(sample), 1),))[: len(sample)]
        pinned[:] = sample
        best = None
        for rep in range(4):                                     # the first call also builds what the run path keeps resident
            ctx.reset_timers()
            t0 = time.perf_counter()
            counts = ctx.exclusive_hashes(pinned)
            w5 = time.perf_counter() - t0
            nt = np.flatnonzero(counts["nontrivial"])
            t0 = time.perf_counter()
            rows = ctx.hyp_test(counts["n_exclusive"][nt], counts["n_match"][nt], 31, 0.99, 0.95, covs)
            w6 = time.perf_counter() - t0
            tm = ctx.timings()
            cur = {"k5_ms": tm["ms_sample"], "k5_kernels_ms": tm["ms_sample_kernels"], "k5_wall_ms": w5 * 1e3, "k6_ms": tm["ms_stats"],
                   "k6_wall_ms": w6 * 1e3, "first_call_setup_ms": tm["ms_sort"]}
            if rep and (best is None or cur["k5_wall_ms"] + cur["k6_wall_ms"] < best["k5_wall_ms"] + best["k6_wall_ms"]):
                best = cur
        nbytes = 12 * T + 8 * len(sample)
        roof = rl("k5s_hist + k5s_scatter + k5_bucket<0> + k5_bucket<1> (K5: sample membership + exclusive hashes on the partitioned reference)",
                  nbytes, best["k5_kernels_ms"], "8*T_ref + 4*T_ref + 8*T_sample (SURVEY.md 8d)")
        roof["share_of_step"] = None
        e2e_ms = best["k5_wall_ms"] + best["k6_wall_ms"]
        out = {"workload": f"BASELINE.json configs[4]: {len(sample)}-hash synthetic sample vs the {n} resident reference genomes ({T} hashes), "
                           f"min_coverage_list {covs}, significance 0.99, k=31, ani_thresh=0.95",
               "nontrivial_genomes": int(len(nt)), "in_sample_at_cov1": int(rows["in_sample_est"][0].sum()), "k6_evaluations": int(len(nt) * len(covs)),
               **best, "sample_gen_seconds": gen_s}
        run_e2e = {"value": n / (e2e_ms * 1e-3), "unit": "reference genomes tested/s", "ms_per_sample": e2e_ms,
                   "h2d_bytes_per_step": 8 * len(sample) + 16 * len(nt), "d2h_bytes_per_step": 16 * n + 64 * len(nt) * len(covs),
                   "what": "ygpu_exclusive_hashes + ygpu_hyp_test from host buffers, wall clock around the two C-ABI calls"}
        # CPU restatement on a bounded sample + parity of the GPU counts against it
        if not args.no_cpu_baseline:
            from oracle import run_oracle as ro
            ns = min(n, args.run_cpu_genomes)
            sub = db.subset(range(ns))
            t0 = time.perf_counter()
            exp = ro.exclusive_counts(sub.hashes, sub.offsets, sample)
            cpu5 = time.perf_counter() - t0
            ids = np.flatnonzero(exp["nontrivial"])[:64]
            t0 = time.perf_counter()
            for g in ids:
                for c in covs:
                    ro.single_hyp_test((int(exp["n_exclusive"][g]), int(exp["n_match"][g])), 31, 0.99, 0.95, c)
            cpu6 = time.perf_counter() - t0
            ctx.load_sketches(sub.hashes, sub.offsets)
            got = ctx.exclusive_hashes(pinned)
            out["cpu_restated"] = {"kind": "port (python sets / scipy, like the reference's get_exclusive_hashes and single_hyp_test)", "cores": 1,
                                   "sample": f"first {ns} reference genomes, {len(ids)} nontrivial x {len(covs)} coverages",
                                   "exclusive_genomes_per_s": ns / max(cpu5, 1e-9), "hyp_evals_per_s": len(ids) * len(covs) / max(cpu6, 1e-9),
                                   "parity_on_sample": bool(all(np.array_equal(got[f], exp[f]) for f in ("n_overlap", "n_exclusive", "n_match")))}
        return out, roof, run_e2e
    finally:
        lib.ygpu_host_free(hp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--genomes", type=int, default=85205, help="BASELINE.json configs[2]: GTDB-rs214-representatives shape")
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="genomes in the CPU sample (cpu_baseline: 0 = size for ~15 s; --impl reference: 0 = the FULL configuration)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-run-path", action="store_true", help="skip the yacht-run measurement (configs[4]) that follows the train step at N = 1")
    ap.add_argument("--run-sample-hashes", type=int, default=10_000_000, help="hashes in the synthetic sample of the run-path measurement")
    ap.add_argument("--run-cpu-genomes", type=int, default=24, help="reference genomes in the CPU restatement of the run path (~0.4 s each)")
    ap.add_argument("--no-reference-cache", action="store_true",
                    help="--impl reference: measure again even if this box already holds a measurement of the same configuration")
    ap.add_argument("--residency", default="hashes", choices=["hashes", "genomes"],
                    help="N > 1: what a rank holds -- its hash range of every sketch (default) or the sketches of its genome range")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the flagged pairs and index statistics of the last resident step to DIR/*.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
