"""Streamed FASTA / FASTQ sketching on the device (ygpu_stream_*, seq_stream.cu): bit-identical to the record path
(sketch.read_records + ygpu_sketch_sequences) and to the oracle on every case of tests/harness/stream_cases.py, through all
three hashing kernels; the CLI files written through either route are the same; host memory does not grow with the input."""
import argparse
import gzip
import json
import os
import resource
import subprocess
import sys
import zipfile

import numpy as np
import pytest

from harness.stream_cases import accepted_cases, rejected_cases
from oracle import sketch_oracle as so

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def ctx():
    from yacht_b200 import _lib
    c = _lib.GpuContext(0)
    yield c
    c.close()


def _stream(ctx, files, k, scaled, per_record, chunk):
    """Feed every file in pieces of 1 000 bytes (any split must do) with device chunks of `chunk` bytes."""
    from yacht_b200 import sketch
    ctx.set_option("stream_chunk_bytes", chunk)
    ctx.stream_begin(k, sketch.max_hash_for_scaled(scaled), 42, per_record)
    for data in files:
        buf = np.frombuffer(data, np.uint8)
        for a in range(0, len(data), 1000):
            piece = np.ascontiguousarray(buf[a:a + 1000])
            ctx.stream_feed(piece.ctypes.data, piece.size, "in")
        ctx.stream_end_file("in")
    h, a, off, names, stats = ctx.stream_finish("in")
    return [(h[int(off[s]):int(off[s + 1])], a[int(off[s]):int(off[s + 1])]) for s in range(len(off) - 1)], names, stats


def _records(tmp_path, files):
    from yacht_b200 import sketch
    recs = []
    for i, data in enumerate(files):
        p = tmp_path / f"f{i}"
        p.write_bytes(data)
        recs.extend(sketch.read_records(str(p)))
    return recs


def _record_path(ctx, groups, k, scaled):
    from yacht_b200 import sketch
    if not groups:                    # no records, no sketches (sketch_record_groups([]) == [])
        return []
    parts, offs = [], [0]
    for g in groups:
        parts.extend(s + b"\n" for s in g)
        offs.append(offs[-1] + sum(len(s) + 1 for s in g))
    h, a, off, _ = ctx.sketch_sequences(b"".join(parts), offs, k, sketch.max_hash_for_scaled(scaled))
    return [(h[int(off[s]):int(off[s + 1])], a[int(off[s]):int(off[s + 1])]) for s in range(len(groups))]


def _same(got, want, what):
    assert len(got) == len(want), what
    for i, ((gm, ga), (wm, wa)) in enumerate(zip(got, want)):
        assert np.array_equal(gm, wm) and np.array_equal(ga, wa), f"{what} sketch {i}"


@pytest.mark.parametrize("k", [21, 31, 51, 64, 100])
def test_stream_equals_record_path_and_oracle(ctx, tmp_path, k):
    cases = accepted_cases()
    for name, data in sorted(cases.items()):
        recs = _records(tmp_path, [data])
        for scaled in (1, 100, 1000):
            chunks = (k - 1, 4097) if scaled == 1 else (4097,)
            for per_record in (False, True):
                groups = [[s] for _, s in recs] if per_record else [[s for _, s in recs]]
                want = _record_path(ctx, groups, k, scaled)
                orc = [so.sketch_records(g, k, scaled) for g in groups]
                _same(want, orc, f"record path vs oracle {name} k={k} scaled={scaled}")
                for chunk in chunks:
                    got, names, _ = _stream(ctx, [data], k, scaled, per_record, chunk)
                    _same(got, want, f"{name} k={k} scaled={scaled} per_record={per_record} chunk={chunk}")
                    if per_record:
                        assert [n.decode() for n in (names or [])] == [n for n, _ in recs], name


def test_stream_several_files_one_sketch(ctx, tmp_path):
    cases = accepted_cases()
    files = [cases["fastq_plain"], cases["fasta_no_final_newline"], cases["only_whitespace"], cases["fastq_crlf_no_final_newline"]]
    recs = _records(tmp_path, files)
    for k in (31, 51):
        want = _record_path(ctx, [[s for _, s in recs]], k, 1)
        for chunk in (k - 1, 333, 1 << 20):
            got, _, st = _stream(ctx, files, k, 1, False, chunk)
            _same(got, want, f"k={k} chunk={chunk}")
            assert st["n_records"] == len(recs)


def test_stream_rejects_what_the_record_path_rejects(ctx, tmp_path):
    from yacht_b200 import sketch
    for name, data in sorted(rejected_cases().items()):
        p = tmp_path / "bad"
        p.write_bytes(data)
        with pytest.raises(ValueError) as ei:
            sketch.read_records(str(p))
        want = str(ei.value)[len(str(p)) + 2:]
        for chunk in (5, 4096):
            with pytest.raises(ValueError) as e2:
                _stream(ctx, [data], 31, 1, False, chunk)
            assert str(e2.value) == f"in: {want}", name
    # a failed stream is over: the next calls need a new begin, which works
    with pytest.raises(Exception):
        ctx.stream_end_file("in")
    got, _, _ = _stream(ctx, [accepted_cases()["fastq_plain"]], 31, 1, False, 4096)
    assert len(got) == 1 and len(got[0][0]) > 0


def _zip_contents(path):
    with zipfile.ZipFile(path) as z:
        return {n: (gzip.decompress(z.read(n)) if n.endswith(".gz") else z.read(n)) for n in sorted(z.namelist())}


def test_cli_outputs_identical_through_both_routes(tmp_path, monkeypatch):
    """`yacht sketch sample` (single, paired, plain, gzip) and `yacht sketch ref` (folder, single file): the files written
    through the stream are the ones the record path writes (.sig byte for byte; .sig.zip entry by entry, whose zip and gzip
    headers carry the time of writing)."""
    from yacht_b200 import sketch, sketch_ref_genomes, sketch_sample
    cases = accepted_cases()
    fq1 = tmp_path / "r1.fq"
    fq1.write_bytes(cases["fastq_plain"] * 20)
    fq2 = tmp_path / "r2.fq.gz"
    fq2.write_bytes(gzip.compress(cases["fastq_crlf_no_final_newline"] + b"\n") + gzip.compress(cases["fastq_tricky_quality"] * 5))
    folder = tmp_path / "refs"
    folder.mkdir()
    (folder / "A.fna").write_bytes(cases["fasta_wrapped"] * 3)
    (folder / "B.fa.gz").write_bytes(gzip.compress(cases["fasta_one_long_line"] + cases["fasta_case_n_iupac"]))
    (folder / "C.fasta").write_bytes(cases["fasta_empty_header_and_body"])
    single = tmp_path / "multi.fna"
    single.write_bytes(cases["fasta_wrapped"] + cases["fasta_empty_header_and_body"] + cases["fasta_headers_gt_and_acgt"])
    runs = [("sample1", lambda o: sketch_sample.main(argparse.Namespace(infile=[str(fq1)], kmer=31, scaled=10, outfile=o))),
            ("sample_gz", lambda o: sketch_sample.main(argparse.Namespace(infile=[str(fq2)], kmer=21, scaled=1, outfile=o))),
            ("paired", lambda o: sketch_sample.main(argparse.Namespace(infile=[str(fq1), str(fq2)], kmer=51, scaled=10, outfile=o))),
            ("folder", lambda o: sketch_ref_genomes.main(argparse.Namespace(infile=str(folder), kmer=31, scaled=10, outfile=o))),
            ("single", lambda o: sketch_ref_genomes.main(argparse.Namespace(infile=str(single), kmer=31, scaled=1, outfile=o)))]
    for name, run in runs:
        out = {}
        for route, limit in (("record", 1 << 40), ("stream", 0)):
            monkeypatch.setattr(sketch, "STREAM_FILE_BYTES", limit)
            monkeypatch.setattr(sketch, "STREAM_READ_BYTES", 5000)
            run(str(tmp_path / f"{name}_{route}.sig"))
            run(str(tmp_path / f"{name}_{route}.sig.zip"))
            out[route] = ((tmp_path / f"{name}_{route}.sig").read_bytes(), _zip_contents(tmp_path / f"{name}_{route}.sig.zip"))
        assert out["stream"][0] == out["record"][0], name
        assert out["stream"][1] == out["record"][1], name
        assert json.loads(out["record"][0])[0]["signatures"][0]["mins"], name


_CHILD = r"""
import json, os, resource, sys
sys.path.insert(0, sys.argv[1])
from yacht_b200 import sketch
sketch.STREAM_READ_BYTES = 64 << 20
sketch_ctx = sketch._context()
sketch_ctx.set_option("stream_chunk_bytes", 64 << 20)
sketch.sketch_stream([sys.argv[2]], 31, 1000)            # warm-up: buffers, device scratch, library code
rss0 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
[(mins, ab)], _ = sketch.sketch_stream([sys.argv[3]], 31, 1000)
rss1 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
print(json.dumps({"rss0_kb": rss0, "rss1_kb": rss1, "n_mins": len(mins)}))
"""


def _write_fastq(path, nbytes, seed):
    """Reads of 150 bp from one planted 4 Mbp genome with 1 % errors, written block after block until `nbytes`."""
    rng = np.random.default_rng(seed)
    genome = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=4_000_000)
    n_reads = 20_000
    with open(path, "wb") as f:
        written = 0
        while written < nbytes:
            starts = rng.integers(0, genome.size - 150, size=n_reads)
            reads = genome[starts[:, None] + np.arange(150)]
            err = rng.random(reads.shape) < 0.01
            reads = np.where(err, rng.choice(np.frombuffer(b"ACGTN", np.uint8), size=reads.shape), reads).astype(np.uint8)
            col = lambda b: np.frombuffer(b, np.uint8)[None, :].repeat(n_reads, 0)
            rows = np.concatenate([col(b"@r\n"), reads, col(b"\n+\n"), np.full((n_reads, 150), ord("I"), np.uint8), col(b"\n")], axis=1)
            block = rows.tobytes()
            f.write(block)
            written += len(block)


def test_host_memory_stays_bounded(tmp_path):
    small, one, two = tmp_path / "w.fq", tmp_path / "g1.fq", tmp_path / "g2.fq"
    _write_fastq(small, 8 << 20, 1)
    _write_fastq(one, 1 << 30, 2)
    _write_fastq(two, 2 << 30, 3)
    res = {}
    for name, path in (("1g", one), ("2g", two)):
        cp = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(small), str(path)], capture_output=True, text=True, timeout=1200)
        assert cp.returncode == 0, cp.stderr[-3000:]
        res[name] = json.loads(cp.stdout.strip().splitlines()[-1])
    out_mb = 8 * res["2g"]["n_mins"] * 2 / 2 ** 20
    for r in res.values():
        grew_mb = (r["rss1_kb"] - r["rss0_kb"]) / 1024
        assert grew_mb < 3 * 64 + out_mb + 256, res
    assert abs(res["2g"]["rss1_kb"] - res["1g"]["rss1_kb"]) / 1024 < 64, res
    print("rss", res)
