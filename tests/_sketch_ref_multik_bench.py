"""Measure `sketch ref --kmer 21,31,51` against three single-size `sketch ref` runs on a folder of genomes (not a test; run
by hand on a GPU machine).

    python tests/_sketch_ref_multik_bench.py --genomes 3000 --mb 1.0 --out DIR

Generates a seeded folder of synthetic genomes (FASTA, 80-column lines, 1 to 4 contigs, every second file gzip) in a
temporary directory, then, each in a child process of its own:
  * host read alone: every file through sketch.read_records on the same host threads `sketch ref` uses;
  * one `sketch ref` run (sketch_ref_genomes.main, zip written) for each of k = 21, 31, 51, and one for the three together:
    wall time, time inside the device calls, and the device's ms_h2d (host -> device copy of the batch, pageable memory)
    and ms_sketch (hashing kernels) summed over the batches;
  * a digest of every size's manifest rows and signature files, which must be the same from the single-size and the
    multi-size runs.
Prints one JSON object (also written to DIR/sketch_ref_multik_bench.json) with the card's name and power limit."""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KS = [21, 31, 51]

CHILD = r"""
import argparse, csv, gzip, hashlib, io, json, os, sys, time, zipfile
sys.path.insert(0, sys.argv[1])
from yacht_b200 import sketch, sketch_ref_genomes
mode, ks, folder, out = sys.argv[2], [int(k) for k in sys.argv[3].split(",")], sys.argv[4], sys.argv[5]
res = {}
t0 = time.perf_counter()
if mode == "read":
    from concurrent.futures import ThreadPoolExecutor
    paths = [p for _, p in sketch_ref_genomes.sequence_files_below(folder)]
    with ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        res["bases"] = sum(len(s) for recs in pool.map(sketch.read_records, paths) for _, s in recs)
else:
    ctx = sketch._context()
    acc = {"device_call_s": 0.0, "ms_h2d": 0.0, "ms_sketch": 0.0, "calls": 0}
    def timed(fn):
        def call(*a, **kw):
            ctx.reset_timers()
            t = time.perf_counter()
            r = fn(*a, **kw)
            acc["device_call_s"] += time.perf_counter() - t
            tm = ctx.timings()
            acc["ms_h2d"] += tm["ms_h2d"]
            acc["ms_sketch"] += tm["ms_sketch"]
            acc["calls"] += 1
            return r
        return call
    ctx.sketch_sequences = timed(ctx.sketch_sequences)
    ctx.sketch_sequences_k = timed(ctx.sketch_sequences_k)
    t0 = time.perf_counter()
    sketch_ref_genomes.main(argparse.Namespace(infile=folder, kmer=ks, scaled=1000, outfile=out))
    res.update(acc)
    with zipfile.ZipFile(out) as z:
        rows = [r for r in csv.reader(io.StringIO(z.read("SOURMASH-MANIFEST.csv").decode())) if r and not r[0].startswith("#")][1:]
        dig = {}
        for r in rows:
            h = dig.setdefault(r[3], hashlib.sha256())
            h.update(",".join(r).encode())
            h.update(gzip.decompress(z.read(r[0])))            # the gzip header holds the write time
    res["digest"] = {k: h.hexdigest() for k, h in dig.items()}
    res["n_signatures"] = len(rows)
res["wall_s"] = time.perf_counter() - t0
print(json.dumps(res))
"""


def child(mode, ks, folder, out):
    cp = subprocess.run([sys.executable, "-c", CHILD, ROOT, mode, ",".join(map(str, ks)), folder, out], capture_output=True, text=True)
    if cp.returncode:
        raise RuntimeError(cp.stderr[-4000:])
    return json.loads(cp.stdout.strip().splitlines()[-1])


def write_genome(args):
    path, seed, n_bases = args
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    cuts = np.sort(rng.integers(1, n_bases, size=int(rng.integers(0, 4))))
    parts = []
    for c, seq in enumerate(np.split(acgt[rng.integers(0, 4, size=n_bases)], cuts)):
        full = len(seq) // 80 * 80
        lines = seq[:full].reshape(-1, 80)
        body = np.concatenate([lines, np.full((lines.shape[0], 1), ord("\n"), np.uint8)], axis=1).tobytes()
        tail = seq[full:].tobytes()
        parts.append(b">contig%d synthetic\n" % c + body + (tail + b"\n" if tail else b""))
    data = b"".join(parts)
    if path.endswith(".gz"):
        data = gzip.compress(data, compresslevel=1)
    with open(path, "wb") as f:
        f.write(data)
    return n_bases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=3000)
    ap.add_argument("--mb", type=float, default=1.0, help="mean genome size in millions of bases")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        gpu = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown"
    except FileNotFoundError:
        gpu = "unknown"
    res = {"gpu": gpu, "ks": KS, "scaled": 1000}
    work = tempfile.mkdtemp(prefix="sketch_ref_bench_")
    try:
        folder = os.path.join(work, "genomes")
        os.makedirs(folder)
        rng = np.random.default_rng(2026)
        sizes = np.maximum(1000, rng.normal(a.mb * 1e6, a.mb * 2.5e5, size=a.genomes)).astype(np.int64)
        jobs = [(os.path.join(folder, f"G{g:05d}" + (".fna.gz" if g % 2 else ".fna")), 1000 + g, int(n)) for g, n in enumerate(sizes)]
        t = time.perf_counter()
        with ThreadPoolExecutor(os.cpu_count() or 1) as pool:
            res["bases"] = int(sum(pool.map(write_genome, jobs)))
        res["generate_s"] = time.perf_counter() - t
        res["genomes"] = a.genomes
        res["bytes_on_disk"] = sum(os.path.getsize(p) for p, _, _ in jobs)
        res["host_read"] = child("read", KS, folder, "")
        runs = {}
        for ks in [[k] for k in KS] + [KS]:              # single sizes first, then the three together
            name = ",".join(map(str, ks))
            runs[name] = child("ref", ks, folder, os.path.join(work, f"ref_{name.replace(',', '_')}.sig.zip"))
        res["single"] = {str(k): runs[str(k)] for k in KS}
        res["multi"] = runs[",".join(map(str, KS))]
        three = {key: sum(runs[str(k)][key] for k in KS) for key in ("wall_s", "device_call_s", "ms_h2d", "ms_sketch")}
        res["three_singles_sum"] = three
        res["multi_over_three_singles_wall"] = res["multi"]["wall_s"] / three["wall_s"]
        res["h2d_ms_saved"] = three["ms_h2d"] - res["multi"]["ms_h2d"]
        res["digests_equal"] = all(res["multi"]["digest"][str(k)] == runs[str(k)]["digest"][str(k)] for k in KS)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    text = json.dumps(res, indent=1, sort_keys=True)
    with open(os.path.join(a.out, "sketch_ref_multik_bench.json"), "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
