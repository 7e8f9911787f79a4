"""CPU suite of sketching several k-mer sizes in one pass: the chunked parse of seq_stream.cu for a list of k-mer sizes
(tests/harness/seq_stream_multik_host.cpp: one carry of k_max - 1 bases, the window rule ysq_window_new) takes every window of
every size exactly once for any split of the input; signature files with several sizes round-trip; the CLI takes several
--kmer values for `sketch sample` only.  No GPU needed."""
import argparse
import csv
import gzip
import io
import json
import os
import subprocess
import zipfile
import zlib

import numpy as np
import pytest

from harness.stream_cases import accepted_cases

HERE = os.path.dirname(os.path.abspath(__file__))
K_SETS = [(21, 31, 51), (51, 21), (1, 2), (32, 33, 64), (31, 65, 256)]


@pytest.fixture(scope="module")
def walk(tmp_path_factory):
    out = tmp_path_factory.mktemp("mk") / "libseq_stream_multik_host.so"
    src = os.path.join(HERE, "harness", "seq_stream_multik_host.cpp")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-o", str(out), src], check=True)
    lib = __import__("ctypes").CDLL(str(out))
    import ctypes
    vp, u64 = ctypes.c_void_p, ctypes.c_uint64
    lib.mk_begin.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    lib.mk_file.argtypes = [vp, u64, vp, u64]
    lib.mk_error.restype = ctypes.c_char_p
    lib.mk_bases.argtypes = [ctypes.POINTER(vp)]
    lib.mk_bases.restype = u64
    lib.mk_windows.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    lib.mk_windows.restype = u64
    lib.mk_records.restype = u64
    return lib


def run_walk(lib, files, ks, cuts_of, want_names=1):
    import ctypes
    karr = np.asarray(ks, dtype=np.int32)
    assert lib.mk_begin(karr.ctypes.data, len(ks), want_names) == 0
    for data in files:
        buf = np.frombuffer(data, np.uint8) if data else np.zeros(1, np.uint8)
        cuts = np.asarray(cuts_of(data), dtype=np.uint64)
        if lib.mk_file(buf.ctypes.data, len(data), cuts.ctypes.data if cuts.size else None, cuts.size):
            return lib.mk_error().decode()
    p = ctypes.c_void_p()
    n = int(lib.mk_bases(ctypes.byref(p)))
    bases = ctypes.string_at(p, n) if n else b""
    windows = []
    for ki in range(len(ks)):
        n = int(lib.mk_windows(ki, ctypes.byref(p)))
        windows.append(np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint64)), shape=(n,)).copy() if n
                       else np.zeros(0, np.uint64))
    return dict(bases=bases, windows=windows, n_records=int(lib.mk_records()))


def expected(tmp_path, files, ks):
    from yacht_b200 import sketch
    recs = []
    for i, data in enumerate(files):
        p = tmp_path / f"in{i}"
        p.write_bytes(data)
        recs.extend(sketch.read_records(str(p)))
    bases = b"".join(b"\n" + s for _, s in recs)
    win = [np.array(sorted((r << 32) | j for r, (_, s) in enumerate(recs) for j in range(len(s) - k + 1)), dtype=np.uint64)
           for k in ks]
    return dict(bases=bases, windows=win, n_records=len(recs))


def splits(data, ks, seed):
    n = len(data)
    steps = {1, 2, 3, min(ks) - 1, min(ks), max(ks) - 1, max(ks), max(ks) + 1, 4095, 4096, 4097}
    out = {f"every_{c}": list(range(c, n, c)) for c in sorted(steps) if c >= 1 and (c > 3 or n <= 3000)}
    rng = np.random.default_rng(seed)
    for r in range(2):
        out[f"random_{r}"] = sorted(set(int(x) for x in rng.integers(1, max(n, 2), size=max(1, n // 40))) & set(range(1, n)))
    out["whole"] = []
    return out


def _check(got, exp, ks):
    assert isinstance(got, dict), got
    assert got["bases"] == exp["bases"]
    assert got["n_records"] == exp["n_records"]
    for ki, k in enumerate(ks):
        # a multiset: a window taken twice (double counting) or never (lost at a chunk edge) both differ
        assert np.array_equal(np.sort(got["windows"][ki]), exp["windows"][ki]), f"k={k}"


@pytest.mark.parametrize("ks", K_SETS, ids=lambda ks: "k" + "_".join(map(str, ks)))
@pytest.mark.parametrize("case", sorted(accepted_cases()))
def test_every_window_of_every_k_once(walk, tmp_path, case, ks):
    data = accepted_cases()[case]
    exp = expected(tmp_path, [data], ks)
    for split, cuts in splits(data, ks, zlib.crc32(case.encode())).items():
        got = run_walk(walk, [data], ks, lambda d: cuts)
        try:
            _check(got, exp, ks)
        except AssertionError as e:
            raise AssertionError(f"{case} ks={ks} split={split}") from e


def test_several_files_and_short_records(walk, tmp_path):
    cases = accepted_cases()
    files = [cases["fastq_plain"], cases["fasta_short_records"], cases["only_whitespace"], cases["fastq_crlf_no_final_newline"],
             cases["fasta_empty_header_and_body"]]
    for ks in K_SETS:
        exp = expected(tmp_path, files, ks)
        for step in (1, 7, min(ks), max(ks) - 1, 4096):
            _check(run_walk(walk, files, ks, lambda d: list(range(step, len(d), step))), exp, ks)


def test_harness_refuses_bad_k_counts(walk):
    karr = np.arange(1, 10, dtype=np.int32)
    assert walk.mk_begin(karr.ctypes.data, 9, 1) == 1
    assert walk.mk_begin(karr.ctypes.data, 0, 1) == 1


# ---- signature files holding several k-mer sizes ---------------------------------------------------------------------------

def _sketches():
    rng = np.random.default_rng(5)
    out = []
    for k in (21, 31, 51):
        mins = np.unique(rng.integers(0, 2 ** 60, size=50 + k, dtype=np.uint64))
        out.append(dict(name="", filename="r1.fq", mins=mins, abundances=rng.integers(1, 9, size=mins.size), ksize=k))
    return out


def test_sig_zip_round_trip_several_k(tmp_path):
    from yacht_b200 import sigio
    sks = _sketches()
    path = str(tmp_path / "m.sig.zip")
    sigio.write_sig_zip(path, sks, 31, sigio.MAX_HASH_SCALED_1000)
    sigs = sigio.read_sig_zip(path)
    assert [s.ksize for s in sigs] == [21, 31, 51]
    for s, sk in zip(sigs, sks):
        assert s.md5sum == sigio.compute_md5sum(sk["ksize"], sk["mins"])
        assert np.array_equal(s.mins, sk["mins"]) and np.array_equal(s.abundances, sk["abundances"])
        assert s.scaled == 1000
        one = sigio.load_signature_with_ksize(path, sk["ksize"])
        assert one.md5sum == s.md5sum
    with pytest.raises(ValueError, match="found 0"):
        sigio.load_signature_with_ksize(path, 41)
    with zipfile.ZipFile(path) as z:
        rows = list(csv.reader(io.StringIO(z.read(sigio.MANIFEST_NAME).decode())))
        assert rows[0] == ["# SOURMASH-MANIFEST-VERSION: 1.0"] and rows[1] == sigio.MANIFEST_COLUMNS
        body = rows[2:]
        assert len(body) == 3
        for r, sk in zip(body, sks):
            md5 = sigio.compute_md5sum(sk["ksize"], sk["mins"])
            assert r == [f"signatures/{md5}.sig.gz", md5, md5[:8], str(sk["ksize"]), "DNA", "0", "1000", str(sk["mins"].size),
                         "1", "", "r1.fq"]
            assert json.loads(gzip.decompress(z.read(r[0])))[0]["signatures"][0]["ksize"] == sk["ksize"]


def test_sig_json_round_trip_several_k(tmp_path):
    from yacht_b200 import sigio
    sks = _sketches()
    for name in ("m.sig", "m.sig.gz"):
        path = str(tmp_path / name)
        sigio.write_signatures(path, sks, 31, sigio.MAX_HASH_SCALED_1000)
        sigs = sigio.parse_signature_json(sigio._open_text(path), path)
        assert [s.ksize for s in sigs] == [21, 31, 51]
        for s, sk in zip(sigs, sks):
            assert s.md5sum == sigio.compute_md5sum(sk["ksize"], sk["mins"])
            assert np.array_equal(s.mins, sk["mins"])
            assert sigio.load_signature_with_ksize(path, sk["ksize"]).md5sum == s.md5sum


def test_single_k_files_do_not_change(tmp_path):
    """A sketch that names the default k itself, or names none, writes the same bytes."""
    from yacht_b200 import sigio
    sk = _sketches()[1]
    plain = {k: v for k, v in sk.items() if k != "ksize"}
    a, b = str(tmp_path / "a.sig"), str(tmp_path / "b.sig")
    sigio.write_signatures(a, [sk], 31, sigio.MAX_HASH_SCALED_1000)
    sigio.write_signatures(b, [plain], 31, sigio.MAX_HASH_SCALED_1000)
    assert open(a, "rb").read() == open(b, "rb").read()
    za, zb = str(tmp_path / "a.sig.zip"), str(tmp_path / "b.sig.zip")
    sigio.write_sig_zip(za, [sk], 31, sigio.MAX_HASH_SCALED_1000)
    sigio.write_sig_zip(zb, [plain], 31, sigio.MAX_HASH_SCALED_1000)
    read = lambda p: {n: zipfile.ZipFile(p).read(n) for n in zipfile.ZipFile(p).namelist()}
    ra, rb = read(za), read(zb)
    assert ra.keys() == rb.keys()
    for n in ra:
        assert (gzip.decompress(ra[n]) if n.endswith(".gz") else ra[n]) == (gzip.decompress(rb[n]) if n.endswith(".gz") else rb[n])


# ---- CLI ------------------------------------------------------------------------------------------------------------------

def test_cli_sample_takes_several_kmer_sizes():
    from yacht_b200 import sketch_sample
    p = argparse.ArgumentParser()
    sketch_sample.add_arguments(p)
    assert p.parse_args(["--infile", "r.fq", "--kmer", "21", "31", "51", "--outfile", "m.sig.zip"]).kmer == [21, 31, 51]
    assert p.parse_args(["--infile", "r.fq", "--kmer", "51", "--outfile", "m.sig.zip"]).kmer == [51]
    assert p.parse_args(["--infile", "r.fq", "--outfile", "m.sig.zip"]).kmer == [31]


def test_cli_sample_refuses_duplicate_sizes(tmp_path, capsys):
    from yacht_b200 import sketch_sample
    args = argparse.Namespace(infile=[str(tmp_path / "r.fq")], kmer=[21, 31, 21], scaled=1000, outfile=str(tmp_path / "o.sig.zip"))
    with pytest.raises(ValueError, match="21 given more than once"):
        sketch_sample.main(args)
    assert not (tmp_path / "o.sig.zip").exists()
    out = capsys.readouterr()
    assert "Starting sketching" not in out.out + out.err          # refused before anything is logged as started


def test_cli_ref_stays_single_k(capsys):
    from yacht_b200 import __main__ as cli
    with pytest.raises(SystemExit) as e:
        cli.main(["sketch", "ref", "--infile", "refs", "--kmer", "21", "31", "--outfile", "r.sig.zip"])
    assert e.value.code == 2
    assert "unrecognized arguments: 31" in capsys.readouterr().err
