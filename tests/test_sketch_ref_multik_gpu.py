"""Several k-mer sizes of one batch on the device (ygpu_sketch_sequences_k): every size's result is exactly the single-size
call's and the oracle's; bad size lists are refused.  `yacht sketch ref --kmer 21,31,51` writes, per size, the signatures a
single-size run writes (folder, multi-record file, streamed files); `yacht train --ksize K` on that zip trains what the
size-K zip trains, and `yacht run` with a multi-size sample answers as the single-size chain does."""
import argparse
import csv
import ctypes
import glob
import gzip
import io
import json
import os
import re
import subprocess
import sys
import zipfile

import numpy as np
import pytest

from oracle import sketch_oracle as so

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_SETS = [(21, 31, 51), (51, 21), (1, 2), (32, 33, 64), (31, 65, 256)]


@pytest.fixture(scope="module")
def ctx():
    from yacht_b200 import _lib
    c = _lib.GpuContext(0)
    yield c
    c.close()


def _random_sequence(rng, n, p_bad=0.01):
    seq = rng.choice(np.frombuffer(b"ACGTacgt", dtype=np.uint8), size=n)
    bad = rng.random(n) < p_bad
    return np.where(bad, ord("N"), seq).astype(np.uint8).tobytes()


def _batch(groups):
    """bases and sketch offsets as sketch.sketch_record_groups lays them out (a '\\n' behind every record)"""
    parts, offs = [], [0]
    for recs in groups:
        body = b"".join(r + b"\n" for r in recs)
        parts.append(body)
        offs.append(offs[-1] + len(body))
    return b"".join(parts), offs


def _groups(rng, ks):
    """Empty sketches, sketches shorter than the smallest size, between the smallest and the largest size, and long ones of
    several records (windows across record ends must not count)."""
    k_min, k_max = min(ks), max(ks)
    mid = (k_min + k_max) // 2
    return [[], [_random_sequence(rng, 30_000)], [_random_sequence(rng, max(k_min - 2, 0), 0.0)], [],
            [_random_sequence(rng, mid, 0.0)], [_random_sequence(rng, k_max - 1, 0.0), _random_sequence(rng, k_min, 0.0)],
            [_random_sequence(rng, int(rng.integers(100, 5_000))) for _ in range(5)], [_random_sequence(rng, 70_000, 0.001)], []]


def _split(h, a, off):
    return [(h[int(off[s]):int(off[s + 1])], a[int(off[s]):int(off[s + 1])]) for s in range(len(off) - 1)]


@pytest.mark.parametrize("ks", K_SETS, ids=lambda ks: "k" + "_".join(map(str, ks)))
def test_each_size_equals_its_single_size_call_and_the_oracle(ctx, ks):
    from yacht_b200 import sketch
    rng = np.random.default_rng(sum(ks))
    groups = _groups(rng, ks)
    batches = {"mixed": groups,
               "shorter than every size": [[b"ACG"[:max(min(ks) - 1, 0)]], []],
               "between the sizes": [[_random_sequence(rng, (min(ks) + max(ks)) // 2, 0.0)]],
               "nothing": [[]]}
    for scaled in (1, 100, 1000):
        max_hash = sketch.max_hash_for_scaled(scaled)
        for what, grp in batches.items():
            bases, offs = _batch(grp)
            if what == "nothing":
                bases = b""
                offs = [0, 0]
            per_k = ctx.sketch_sequences_k(bases, offs, list(ks), max_hash)
            assert len(per_k) == len(ks)
            for k, (h, a, off, nk) in zip(ks, per_k):
                sh, sa, soff, snk = ctx.sketch_sequences(bases, offs, k, max_hash)
                tag = f"{what} ks={ks} k={k} scaled={scaled}"
                assert h.dtype == sh.dtype and a.dtype == sa.dtype and off.dtype == soff.dtype, tag
                assert np.array_equal(off, soff) and np.array_equal(h, sh) and np.array_equal(a, sa) and nk == snk, tag
                for s, (m, ab) in enumerate(_split(h, a, off)):
                    em, ea = so.sketch_records(grp[s] if what != "nothing" else [], k, scaled)
                    assert np.array_equal(m, em) and np.array_equal(ab, ea), f"{tag} sketch {s}"
    # the copy is made once, and the hashing time covers every size
    bases, offs = _batch(groups)
    ctx.reset_timers()
    ctx.sketch_sequences_k(bases, offs, list(ks), sketch.max_hash_for_scaled(100))
    t = ctx.timings()
    assert t["ms_h2d"] > 0 and t["ms_sketch"] > 0


def test_sequences_k_refuses_bad_size_lists(ctx):
    from yacht_b200 import _lib
    bases = _random_sequence(np.random.default_rng(5), 5000) + b"\n"
    offs = np.array([0, len(bases)], np.uint64)
    bad = [([], "0 k-mer sizes (1 to 8)"), (list(range(21, 30)), "9 k-mer sizes (1 to 8)"), ([21, 31, 21], "ksize 21 given twice"),
           ([31, 0], "ksize 0 outside [1, 256]"), ([257], "ksize 257 outside [1, 256]")]
    buf = np.frombuffer(bases, np.uint8)
    for ks, text in bad:
        arr = (ctypes.c_int * max(1, len(ks)))(*ks)
        res = (_lib.SketchResult * max(1, len(ks)))()
        rc = ctx.lib.ygpu_sketch_sequences_k(ctx.h, buf.ctypes.data, buf.size, offs.ctypes.data, 1, arr, len(ks), 2 ** 64 - 1, 42, res)
        assert rc == -3, ks                                           # YGPU_ERR_ARG
        assert text in ctx.lib.ygpu_last_error(ctx.h).decode(), ks
        with pytest.raises(_lib.YgpuError, match=re.escape(text)):
            ctx.sketch_sequences_k(bases, offs, ks, 2 ** 64 - 1)
    per_k = ctx.sketch_sequences_k(bases, offs, [21, 31], 2 ** 64 - 1)      # the context still works
    for k, (h, a, off, nk) in zip((21, 31), per_k):
        sh, sa, soff, snk = ctx.sketch_sequences(bases, offs, k, 2 ** 64 - 1)
        assert len(h) > 3000 and np.array_equal(h, sh) and np.array_equal(a, sa) and nk == snk


# ---- command line -------------------------------------------------------------------------------------------------------

def _yacht(*argv):
    cp = subprocess.run([sys.executable, "-m", "yacht_b200", *argv], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert cp.returncode == 0, cp.stderr[-3000:]
    return cp


def _members(path):
    """manifest rows (header dropped) and decompressed member text by location"""
    with zipfile.ZipFile(path) as z:
        rows = [r for r in csv.reader(io.StringIO(z.read("SOURMASH-MANIFEST.csv").decode())) if r and not r[0].startswith("#")][1:]
        return rows, {r[0]: gzip.decompress(z.read(r[0])) for r in rows}


def _assert_per_size_equal(multi, singles, ks):
    rows, text = _members(multi)
    srows = {k: _members(singles[k]) for k in ks}
    n = len(srows[ks[0]][0])
    assert n and len(rows) == n * len(ks)
    for i, row in enumerate(rows):
        k = ks[i % len(ks)]
        want_rows, want_text = srows[k]
        assert row == want_rows[i // len(ks)], (i, k)
        assert text[row[0]] == want_text[row[0]], (i, k)


def _mutate(rng, seq, rate):
    out = seq.copy()
    pos = np.flatnonzero(rng.random(len(seq)) < rate)
    out[pos] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=len(pos))
    return out


def _write_genome(path, contigs):
    opener = gzip.open if str(path).endswith(".gz") else open
    with opener(path, "wb") as f:
        for c, s in enumerate(contigs):
            f.write(f">{os.path.basename(str(path)).split('.')[0]}_contig{c} synthetic\n".encode())
            for i in range(0, len(s), 80):
                f.write(s[i:i + 80] + b"\n")


def test_cli_ref_multi_size_equals_single_size_runs(tmp_path, monkeypatch):
    rng = np.random.default_rng(31)
    folder = tmp_path / "refs"
    folder.mkdir()
    for g in range(9):
        contigs = [_random_sequence(rng, int(rng.integers(20_000, 60_000)), 0.002) for _ in range(1 + g % 3)]
        if g == 4:
            contigs += [b"ACGTACGTACGTAC", _random_sequence(rng, 40, 0.0)]   # shorter than every size; between 21 and 51
        _write_genome(folder / (f"G{g}.fna.gz" if g % 2 else f"G{g}.fa"), contigs)
    multi_record = folder / "G4.fa"
    d = str(tmp_path)
    ks = (21, 31, 51)
    for label, infile in (("folder", folder), ("records", multi_record)):
        singles = {}
        for k in ks:
            singles[k] = os.path.join(d, f"{label}_k{k}.sig.zip")
            _yacht("sketch", "ref", "--infile", str(infile), "--kmer", str(k), "--scaled", "100", "--outfile", singles[k])
        multi = os.path.join(d, f"{label}_multi.sig.zip")
        _yacht("sketch", "ref", "--infile", str(infile), "--kmer", ",".join(map(str, ks)), "--scaled", "100", "--outfile", multi)
        _assert_per_size_equal(multi, singles, ks)

        # the streamed route: every file over the limit (folder: whole mode, --infile: per-record mode)
        from yacht_b200 import sketch, sketch_ref_genomes
        monkeypatch.setattr(sketch, "STREAM_FILE_BYTES", 1)
        streamed = os.path.join(d, f"{label}_streamed.sig.zip")
        sketch_ref_genomes.main(argparse.Namespace(infile=str(infile), kmer=list(ks), scaled=100, outfile=streamed))
        monkeypatch.undo()
        _assert_per_size_equal(streamed, singles, ks)


def test_multi_size_ref_trains_and_runs_as_single_size_chains(tmp_path):
    rng = np.random.default_rng(2025)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    folder = tmp_path / "ref_genomes"
    folder.mkdir()
    base = [rng.choice(acgt, size=int(rng.integers(90_000, 150_000))) for _ in range(10)]
    seqs = base + [_mutate(rng, base[0], 0.002), _mutate(rng, base[7], 0.002), _mutate(rng, base[3], 0.0005)]
    for g, seq in enumerate(seqs):
        cut = len(seq) // 3
        _write_genome(folder / (f"GCF_{g:06d}.1_genomic.fna.gz" if g % 2 else f"GCF_{g:06d}.1_genomic.fna"),
                      [seq[:cut].tobytes(), seq[cut:].tobytes()])
    reads = []
    for g in (3, 4, 5):
        for _ in range(int(3 * len(seqs[g]) / 150)):
            p = int(rng.integers(0, len(seqs[g]) - 150))
            reads.append(_mutate(rng, seqs[g][p:p + 150], 0.002).tobytes())
    d = str(tmp_path)
    fq = os.path.join(d, "sample.fq")
    with open(fq, "wb") as f:
        f.writelines(b"@r%d\n" % i + r + b"\n+\n" + b"F" * len(r) + b"\n" for i, r in enumerate(reads))
    ks = ("21", "31", "51")
    multi_ref, multi_sample = os.path.join(d, "ref_multi.sig.zip"), os.path.join(d, "sample_multi.sig.zip")
    _yacht("sketch", "ref", "--infile", str(folder), "--kmer", ",".join(ks), "--scaled", "100", "--outfile", multi_ref)
    _yacht("sketch", "sample", "--infile", fq, "--kmer", *ks, "--scaled", "100", "--outfile", multi_sample)
    for k in ("31", "51"):
        single_ref, single_sample = os.path.join(d, f"ref_k{k}.sig.zip"), os.path.join(d, f"sample_k{k}.sig.zip")
        _yacht("sketch", "ref", "--infile", str(folder), "--kmer", k, "--scaled", "100", "--outfile", single_ref)
        _yacht("sketch", "sample", "--infile", fq, "--kmer", k, "--scaled", "100", "--outfile", single_sample)
        out = {}
        for which, ref, sample in (("multi", multi_ref, multi_sample), ("single", single_ref, single_sample)):
            od = os.path.join(d, f"{which}_{k}")
            os.makedirs(od)
            cp = _yacht("train", "--force", "--ref_file", ref, "--ksize", k, "--prefix", "db", "--ani_thresh", "0.95", "--outdir", od,
                        "--num_threads", "4")
            inter = os.path.join(od, "db_intermediate_files")
            listed = open(os.path.join(inter, "training_sig_files.tsv")).read().splitlines()
            names = [os.path.basename(p) for p in listed]
            selected = [os.path.basename(p) for p in open(os.path.join(inter, "selected_result.tsv")).read().splitlines()]
            pairs = set()                                       # pair lines with the file-list indices replaced by file names
            for pf in glob.glob(os.path.join(inter, "comparison_files", "*.txt")):
                for line in open(pf).read().splitlines():
                    i, j, rest = line.split(",", 2)
                    pairs.add((names[int(i)], names[int(j)], rest))
            cfg = json.load(open(os.path.join(od, "db_config.json")))
            cfg = {key: (os.path.relpath(v, od) if key in ("manifest_file_path", "intermediate_files_dir") else v) for key, v in cfg.items()}
            run_dir = os.path.join(od, "run")
            os.makedirs(run_dir)
            _yacht("run", "--json", os.path.join(od, "db_config.json"), "--sample_file", sample, "--significance", "0.99",
                   "--min_coverage_list", "1", "0.5", "0.1", "--outdir", run_dir, "--show_all", "--num_threads", "4")
            out[which] = dict(
                listed=sorted(names), selected=sorted(selected), pairs=pairs, cfg=cfg,
                manifest=open(os.path.join(od, "db_processed_manifest.tsv")).read(),
                result=open(os.path.join(run_dir, "results", "result_all.txt")).read(), log=cp.stdout)
        m, s = out["multi"], out["single"]
        assert "Leaving out 26 signature files without a k-mer size %s sketch" % k in m["log"]
        assert "Leaving out" not in s["log"]
        for key in ("listed", "selected", "pairs", "cfg", "manifest", "result"):
            assert m[key] == s[key], (k, key)
        assert len(m["listed"]) == 13 and 10 <= len(m["selected"]) < 13 and m["pairs"], k
        assert "True" in m["result"], k
