"""Measure one multi-k stream (`sketch sample --kmer 21 31 51`) against single-k streams (not a test; run by hand on a GPU
machine).

    python tests/_sketch_multik_bench.py --gb 3 --out DIR

Generates seeded FASTQ with _sketch_stream_bench.write_fastq, plain and gzip, in DIR.  Then, per input, each in a child
process of its own:
  * host read alone (readinto through the stream's reader);
  * one single-k stream (sketch.sketch_stream) for each of k = 21, 31, 51: wall time, device ms per phase;
  * one stream of k = 21, 31, 51 together: wall time, device ms per phase (ms_h2d, ms_parse, ms_hash, ms_merge);
  * a digest of every k's sketch, which must be the same from the single-k and the multi-k runs.
Prints one JSON object (also written to DIR/sketch_multik_bench.json) with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from _sketch_stream_bench import write_fastq  # noqa: E402

GB = 1e9
KS = [21, 31, 51]
PHASES = ("ms_h2d", "ms_parse", "ms_hash", "ms_merge")

CHILD = r"""
import json, sys, time
import numpy as np
sys.path.insert(0, sys.argv[1])
from yacht_b200 import sketch
mode, ks, path = sys.argv[2], [int(k) for k in sys.argv[3].split(",")], sys.argv[4]
digest = lambda mins, ab: int(np.bitwise_xor.reduce(mins ^ (ab.astype(mins.dtype) << 40))) if len(mins) else 0
t0 = time.perf_counter()
out = {}
if mode == "read":
    text, raw = sketch._open_text(path)
    buf = bytearray(sketch.STREAM_READ_BYTES)
    n = 0
    while True:
        m = text.readinto(buf)
        if not m:
            break
        n += m
    out["bytes"] = n
else:
    st = {}
    res, _ = sketch.sketch_stream([path], ks[0] if len(ks) == 1 else ks, 1000, stats=st)
    per_k = [res] if len(ks) == 1 else res
    out.update(st)
    out["digest"] = {str(k): digest(*r[0]) for k, r in zip(ks, per_k)}
    out["n_mins"] = {str(k): len(r[0][0]) for k, r in zip(ks, per_k)}
out["wall_s"] = time.perf_counter() - t0
print(json.dumps(out))
"""


def child(mode, ks, path):
    cp = subprocess.run([sys.executable, "-c", CHILD, ROOT, mode, ",".join(map(str, ks)), path], capture_output=True, text=True)
    if cp.returncode:
        raise RuntimeError(cp.stderr[-4000:])
    return json.loads(cp.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=3.0, help="size of the input (plain text)")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown", "ks": KS}
    plain, gz = os.path.join(a.out, "mk.fq"), os.path.join(a.out, "mk.fq.gz")
    t = time.perf_counter()
    nb = write_fastq(plain, int(a.gb * GB), 7)
    write_fastq(gz, int(a.gb * GB), 7, gz=True)
    res["generate_s"], res["text_gb"], res["gz_gb_on_disk"] = time.perf_counter() - t, nb / GB, os.path.getsize(gz) / GB
    for name, path in (("plain", plain), ("gzip", gz)):
        r = {"host_read_s": child("read", KS, path)["wall_s"]}
        singles = {k: child("stream", [k], path) for k in KS}
        multi = child("stream", KS, path)
        r["single"] = {str(k): {"wall_s": s["wall_s"], **{p: s[p] for p in PHASES}} for k, s in singles.items()}
        r["single_sum_wall_s"] = sum(s["wall_s"] for s in singles.values())
        r["multi"] = {"wall_s": multi["wall_s"], **{p: multi[p] for p in PHASES}}
        r["multi_over_one_single_wall"] = multi["wall_s"] / singles[31]["wall_s"]
        r["multi_over_three_singles_wall"] = multi["wall_s"] / r["single_sum_wall_s"]
        r["digests_equal"] = all(multi["digest"][str(k)] == singles[k]["digest"][str(k)] for k in KS)
        r["n_mins"] = multi["n_mins"]
        res[name] = r
    for p in (plain, gz):
        os.remove(p)
    text = json.dumps(res, indent=1, sort_keys=True)
    with open(os.path.join(a.out, "sketch_multik_bench.json"), "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
