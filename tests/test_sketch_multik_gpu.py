"""Several k-mer sizes in one streamed pass on the device (ygpu_stream_begin_k / _finish_k): every size's result is exactly
the single-size stream's and the oracle's, for windows across chunk edges, in both modes; `yacht sketch sample --kmer 21 31
51` writes, per size, the signature a single-size run writes; `yacht run` answers the same from either file; bad size lists
are refused."""
import csv
import gzip
import io
import os
import subprocess
import sys
import zipfile

import numpy as np
import pytest

from harness.stream_cases import accepted_cases
from oracle import sketch_oracle as so
from yacht_b200 import xlsx

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_SETS = [(21, 31, 51), (51, 21), (1, 2), (32, 33, 64), (31, 65, 256)]
CHUNKS = (4096, 4097, 64 << 20)


@pytest.fixture(scope="module")
def ctx():
    from yacht_b200 import _lib
    c = _lib.GpuContext(0)
    yield c
    c.close()


def _inputs(tmp_path):
    """name -> [decompressed text of each file]: one file, and a pair as `sketch sample` takes it."""
    c = accepted_cases()
    return {"fasta": [c["fasta_wrapped"] + c["fasta_short_records"] + c["fasta_empty_header_and_body"] + c["fasta_one_long_line"]],
            "paired_fastq": [c["fastq_plain"] * 3, c["fastq_crlf_no_final_newline"] + b"\n" + c["fastq_tricky_quality"]]}


def _feed(ctx, files, ks, scaled, per_record, chunk):
    from yacht_b200 import sketch
    ctx.set_option("stream_chunk_bytes", chunk)
    ctx.stream_begin(ks, sketch.max_hash_for_scaled(scaled), 42, per_record)
    for data in files:
        buf = np.frombuffer(data, np.uint8)
        for a in range(0, len(data), 1000):
            piece = np.ascontiguousarray(buf[a:a + 1000])
            ctx.stream_feed(piece.ctypes.data, piece.size, "in")
        ctx.stream_end_file("in")
    return ctx.stream_finish("in")


def _split(h, a, off):
    return [(h[int(off[s]):int(off[s + 1])], a[int(off[s]):int(off[s + 1])]) for s in range(len(off) - 1)]


def _same(got, want, what):
    assert len(got) == len(want), what
    for i, ((gm, ga), (wm, wa)) in enumerate(zip(got, want)):
        assert np.array_equal(gm, wm) and np.array_equal(ga, wa), f"{what} sketch {i}"


@pytest.mark.parametrize("ks", K_SETS, ids=lambda ks: "k" + "_".join(map(str, ks)))
def test_each_k_equals_its_single_k_stream_and_the_oracle(ctx, tmp_path, ks):
    from yacht_b200 import sketch
    for name, files in _inputs(tmp_path).items():
        recs = []
        for i, data in enumerate(files):
            p = tmp_path / f"{name}{i}"
            p.write_bytes(data)
            recs.extend(sketch.read_records(str(p)))
        for scaled in (1, 100):
            for per_record in (False, True):
                groups = [[s] for _, s in recs] if per_record else [[s for _, s in recs]]
                orc = {k: [so.sketch_records(g, k, scaled) for g in groups] for k in ks}
                for chunk in CHUNKS:
                    what = f"{name} ks={ks} scaled={scaled} per_record={per_record} chunk={chunk}"
                    per_k, names, st = _feed(ctx, files, ks, scaled, per_record, chunk)
                    assert len(per_k) == len(ks), what
                    assert st["n_kmers"] == sum(nk for _, _, _, nk in per_k), what
                    for k, (h, a, off, nk) in zip(ks, per_k):
                        sh, sa, soff, snames, sst = _feed(ctx, files, k, scaled, per_record, chunk)
                        assert np.array_equal(off, soff) and np.array_equal(h, sh) and np.array_equal(a, sa), f"{what} k={k}"
                        assert nk == sst["n_kmers"], f"{what} k={k}"
                        assert names == snames, f"{what} k={k}"
                        _same(_split(h, a, off), orc[k], f"oracle {what} k={k}")
                    if per_record:
                        assert [n.decode() for n in (names or [])] == [n for n, _ in recs], what


def test_begin_k_refuses_bad_size_lists(ctx):
    import ctypes
    from yacht_b200 import _lib
    bad = [([], "0 k-mer sizes (1 to 8)"), (list(range(21, 30)), "9 k-mer sizes (1 to 8)"), ([21, 31, 21], "ksize 21 given twice"),
           ([31, 0], "ksize 0 outside [1, 256]"), ([257], "ksize 257 outside [1, 256]")]
    for ks, text in bad:
        arr = (ctypes.c_int * max(1, len(ks)))(*ks)
        rc = ctx.lib.ygpu_stream_begin_k(ctx.h, arr, len(ks), 2 ** 64 - 1, 42, _lib.STREAM_WHOLE)
        assert rc == -3, ks                                       # YGPU_ERR_ARG
        assert text in ctx.lib.ygpu_last_error(ctx.h).decode(), ks
    # a stream of several sizes is not finished by the single-size call, and the next begin works
    ctx.stream_begin([21, 31], 2 ** 64 - 1)
    res, st = _lib.SketchResult(), _lib.StreamStats()
    vp = ctypes.c_void_p
    rc = ctx.lib.ygpu_stream_finish(ctx.h, ctypes.byref(res), ctypes.byref(st), ctypes.byref(vp()), ctypes.byref(vp()),
                                    ctypes.byref(ctypes.c_uint64()))
    assert rc == -3 and "ygpu_stream_finish_k" in ctx.lib.ygpu_last_error(ctx.h).decode()
    per_k, _, _ = _feed(ctx, [accepted_cases()["fastq_plain"]], [21, 31], 1, False, 4096)
    assert [len(h) > 0 for h, _, _, _ in per_k] == [True, True]


def _yacht(*argv):
    cp = subprocess.run([sys.executable, "-m", "yacht_b200", *argv], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert cp.returncode == 0, cp.stderr[-3000:]
    return cp


def _members(path):
    """manifest rows (header dropped) and decompressed member text by location"""
    with zipfile.ZipFile(path) as z:
        rows = [r for r in csv.reader(io.StringIO(z.read("SOURMASH-MANIFEST.csv").decode())) if r and not r[0].startswith("#")][1:]
        return rows, {r[0]: gzip.decompress(z.read(r[0])) for r in rows}


def _mutate(rng, seq, rate):
    out = seq.copy()
    pos = np.flatnonzero(rng.random(len(seq)) < rate)
    out[pos] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=len(pos))
    return out


def test_cli_multik_sample_equals_single_k_runs_and_run_agrees(tmp_path):
    rng = np.random.default_rng(77)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    folder = tmp_path / "refs"
    folder.mkdir()
    base = [rng.choice(acgt, size=int(rng.integers(60_000, 100_000))) for _ in range(8)]
    seqs = base + [_mutate(rng, base[2], 0.003)]
    for g, seq in enumerate(seqs):
        with gzip.open(folder / f"G{g:03d}.fna.gz", "wb") as f:
            f.write(f">G{g}\n".encode())
            for i in range(0, len(seq), 70):
                f.write(seq[i:i + 70].tobytes() + b"\n")
    reads = []
    for g in (1, 2, 5):
        for _ in range(int(2 * len(seqs[g]) / 150)):
            p = int(rng.integers(0, len(seqs[g]) - 150))
            reads.append(_mutate(rng, seqs[g][p:p + 150], 0.005).tobytes())
    half = len(reads) // 2
    r1, r2 = tmp_path / "r1.fq", tmp_path / "r2.fq.gz"
    r1.write_bytes(b"".join(b"@a%d\n" % i + r + b"\n+\n" + b"F" * len(r) + b"\n" for i, r in enumerate(reads[:half])))
    text2 = b"".join(b"@b%d\n" % i + r + b"\n+\n" + b"F" * len(r) + b"\n" for i, r in enumerate(reads[half:]))
    r2.write_bytes(gzip.compress(text2[:len(text2) // 3]) + gzip.compress(text2[len(text2) // 3:]))      # two gzip members
    d = str(tmp_path)
    ks = (21, 31, 51)
    multi = os.path.join(d, "m.sig.zip")
    _yacht("sketch", "sample", "--infile", str(r1), str(r2), "--kmer", *map(str, ks), "--scaled", "100", "--outfile", multi)
    _yacht("sketch", "sample", "--infile", str(r1), str(r2), "--kmer", *map(str, ks), "--scaled", "100", "--outfile", multi[:-4])
    rows, text = _members(multi)
    assert [int(r[3]) for r in rows] == list(ks)
    import json
    multi_json = json.loads(open(multi[:-4]).read())
    assert len(multi_json) == len(ks)
    for i, k in enumerate(ks):
        single = os.path.join(d, f"s{k}.sig.zip")
        _yacht("sketch", "sample", "--infile", str(r1), str(r2), "--kmer", str(k), "--scaled", "100", "--outfile", single)
        _yacht("sketch", "sample", "--infile", str(r1), str(r2), "--kmer", str(k), "--scaled", "100", "--outfile", single[:-4])
        srows, stext = _members(single)
        assert len(srows) == 1 and rows[i] == srows[0], k
        assert text[rows[i][0]] == stext[srows[0][0]], k
        assert multi_json[i] == json.loads(open(single[:-4]).read())[0], k

    # downstream: a database per k, run with the multi-k sample and with the single-k one
    for k, ani in ((31, 0.95), (51, 0.95)):
        ref = os.path.join(d, f"ref{k}.sig.zip")
        _yacht("sketch", "ref", "--infile", str(folder), "--kmer", str(k), "--scaled", "100", "--outfile", ref)
        _yacht("train", "--force", "--ref_file", ref, "--ksize", str(k), "--prefix", f"db{k}", "--ani_thresh", str(ani),
               "--outdir", d, "--num_threads", "4")
        out = {}
        for which, sample in (("multi", multi), ("single", os.path.join(d, f"s{k}.sig.zip"))):
            od = os.path.join(d, f"run_{k}_{which}")
            os.makedirs(od)
            _yacht("run", "--json", os.path.join(d, f"db{k}_config.json"), "--sample_file", sample, "--significance", "0.99",
                   "--min_coverage_list", "1", "0.5", "0.1", "--outdir", od, "--show_all", "--num_threads", "4")
            res = os.path.join(od, "results")
            out[which] = (open(os.path.join(res, "result_all.txt")).read(), xlsx.read_xlsx(os.path.join(res, "result.xlsx")))
        assert out["multi"][0] == out["single"][0], k
        assert list(out["multi"][1]) == list(out["single"][1]) == ["min_coverage1.0", "min_coverage0.5", "min_coverage0.1"]
        for sheet in out["multi"][1]:
            a, b = out["multi"][1][sheet], out["single"][1][sheet]
            assert a.equals(b), (k, sheet)
        df = out["multi"][1]["min_coverage0.5"]
        assert len(df) and df["in_sample_est"].astype(str).eq("True").sum() >= 2, k
