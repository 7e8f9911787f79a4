"""Measure the streamed sketch of a large FASTQ against the record path (not a test; run by hand on a GPU machine).

    python tests/_sketch_stream_bench.py --gb 8 --record-gb 4 --out DIR

Generates seeded FASTQ (150 bp reads from 20 planted 5 Mbp genomes, 1 % substitutions, some N), plain and gzip, in DIR. Then,
each in a child process of its own (peak RSS = ru_maxrss of that child):
  * host read alone (readinto through the same reader), per GB, plain and gzip;
  * the stream (sketch.sketch_stream): wall time, device parse / hash / merge / H2D time per GB, peak RSS;
  * the record path (read_records + sketch_record_groups) on the --record-gb input, and parity with the stream there.
Prints one JSON object (also written to DIR/sketch_stream_bench.json) with the card's name and power limit."""
import argparse
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GB = 1e9

CHILD = r"""
import json, resource, sys, time
sys.path.insert(0, sys.argv[1])
from yacht_b200 import sketch
mode, paths = sys.argv[2], sys.argv[3:]
t0 = time.perf_counter()
out = {}
if mode == "read":
    text, raw = sketch._open_text(paths[0])
    buf = bytearray(sketch.STREAM_READ_BYTES)
    n = 0
    while True:
        m = text.readinto(buf)
        if not m:
            break
        n += m
    out["bytes"] = n
elif mode == "stream":
    st = {}
    [(mins, ab)], _ = sketch.sketch_stream(paths, 31, 1000, stats=st)
    out.update(st)
    out["n_mins"] = len(mins)
    out["digest"] = int(np.bitwise_xor.reduce(mins ^ (ab.astype(mins.dtype) << 40))) if len(mins) else 0
else:
    reads = [s for p in paths for _, s in sketch.read_records(p)]
    [(mins, ab)] = sketch.sketch_record_groups([reads], 31, 1000)
    out["n_mins"] = len(mins)
    out["digest"] = int(np.bitwise_xor.reduce(mins ^ (ab.astype(mins.dtype) << 40))) if len(mins) else 0
out["wall_s"] = time.perf_counter() - t0
out["peak_rss_mb"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024
print(json.dumps(out))
""".replace("import json,", "import numpy as np, json,")


def write_fastq(path, nbytes, seed, gz=False):
    rng = np.random.default_rng(seed)
    genomes = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=(20, 5_000_000))
    n = 50_000
    col = lambda b: np.frombuffer(b, np.uint8)[None, :].repeat(n, 0)
    f = gzip.open(path, "wb", compresslevel=1) if gz else open(path, "wb")
    with f:
        done = 0
        while done < nbytes:
            g = rng.integers(0, 20, size=n)
            s = rng.integers(0, 5_000_000 - 150, size=n)
            reads = genomes[g[:, None], s[:, None] + np.arange(150)]
            sub = rng.random(reads.shape) < 0.01
            reads = np.where(sub, rng.choice(np.frombuffer(b"ACGT", np.uint8), size=reads.shape), reads)
            reads = np.where(rng.random(reads.shape) < 0.001, ord("N"), reads).astype(np.uint8)
            block = np.concatenate([col(b"@read\n"), reads, col(b"\n+\n"), np.full((n, 150), ord("F"), np.uint8), col(b"\n")], axis=1).tobytes()
            f.write(block)
            done += len(block)
    return done


def child(mode, paths):
    cp = subprocess.run([sys.executable, "-c", CHILD, ROOT, mode] + list(paths), capture_output=True, text=True)
    if cp.returncode:
        raise RuntimeError(cp.stderr[-4000:])
    return json.loads(cp.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=8.0, help="size of the streamed input (plain text)")
    ap.add_argument("--record-gb", type=float, default=4.0, help="size of the input both routes sketch")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown"}
    big, big_gz = os.path.join(a.out, "big.fq"), os.path.join(a.out, "big.fq.gz")
    mid = os.path.join(a.out, "mid.fq")
    t = time.perf_counter()
    nb = write_fastq(big, int(a.gb * GB), 1)
    write_fastq(big_gz, int(a.gb * GB), 1, gz=True)
    nm = write_fastq(mid, int(a.record_gb * GB), 2)
    res["generate_s"] = time.perf_counter() - t
    res["big_text_gb"], res["mid_text_gb"] = nb / GB, nm / GB
    res["big_gz_gb_on_disk"] = os.path.getsize(big_gz) / GB
    for name, path in (("plain", big), ("gzip", big_gz)):
        r = child("read", [path])
        res[f"host_read_{name}_s_per_gb"] = r["wall_s"] / (nb / GB)
        s = child("stream", [path])
        res[f"stream_{name}"] = s
        res[f"stream_{name}_wall_s_per_gb"] = s["wall_s"] / (nb / GB)
        dev = s["ms_h2d"] + s["ms_parse"] + s["ms_hash"] + s["ms_merge"]
        res[f"stream_{name}_device_ms_per_gb"] = {k: s[k] / (nb / GB) for k in ("ms_h2d", "ms_parse", "ms_hash", "ms_merge")}
        res[f"stream_{name}_device_s_per_gb"] = dev / 1000 / (nb / GB)
    rec = child("record", [mid])
    st = child("stream", [mid])
    res["record_mid"], res["stream_mid"] = rec, st
    res["parity_mid"] = rec["digest"] == st["digest"] and rec["n_mins"] == st["n_mins"]
    res["parity_plain_gzip"] = res["stream_plain"]["digest"] == res["stream_gzip"]["digest"]
    for p in (big, big_gz, mid):
        os.remove(p)
    text = json.dumps(res, indent=1, sort_keys=True)
    with open(os.path.join(a.out, "sketch_stream_bench.json"), "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
