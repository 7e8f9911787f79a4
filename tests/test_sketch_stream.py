"""CPU suite of the streamed FASTA / FASTQ parse: the chunked state machine of seq_stream.cu, compiled from its header for the
host (tests/harness/seq_stream_host.cpp), against sketch.read_records for every split of the input; and the Python reader
(gzip members, page-locked buffers, reader thread) behind a stand-in stream context.  No GPU needed."""
import ctypes
import gzip
import os
import subprocess
import zlib

import numpy as np
import pytest

from oracle import sketch_oracle as so
from harness.stream_cases import accepted_cases, rejected_cases

HERE = os.path.dirname(os.path.abspath(__file__))
KS = [21, 31, 51]


@pytest.fixture(scope="module")
def walk(tmp_path_factory):
    out = tmp_path_factory.mktemp("sq") / "libseq_stream_host.so"
    src = os.path.join(HERE, "harness", "seq_stream_host.cpp")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-o", str(out), src], check=True)
    lib = ctypes.CDLL(str(out))
    vp, u64 = ctypes.c_void_p, ctypes.c_uint64
    lib.sh_begin.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.sh_file.argtypes = [vp, u64, vp, u64]
    lib.sh_error.restype = ctypes.c_char_p
    for fn in (lib.sh_bases, lib.sh_names, lib.sh_name_offsets, lib.sh_windows):
        fn.argtypes = [ctypes.POINTER(vp)]
        fn.restype = u64
    lib.sh_records.restype = u64
    return lib


def _get(fn, dtype):
    p = ctypes.c_void_p()
    n = int(fn(ctypes.byref(p)))
    if n == 0:
        return np.zeros(0, dtype)
    return np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(np.ctypeslib.as_ctypes_type(dtype))), shape=(n,)).copy()


def run_walk(lib, files, k, cuts_of, want_names):
    """files: list of bytes; cuts_of(data) -> ascending cut positions.  Returns dict or the error text."""
    lib.sh_begin(k, want_names)
    for data in files:
        buf = np.frombuffer(data, np.uint8) if data else np.zeros(1, np.uint8)
        cuts = np.asarray(cuts_of(data), dtype=np.uint64)
        if lib.sh_file(buf.ctypes.data, len(data), cuts.ctypes.data if cuts.size else None, cuts.size):
            return lib.sh_error().decode()
    names_blob = _get(lib.sh_names, np.uint8).tobytes()
    name_off = list(_get(lib.sh_name_offsets, np.uint64)) + [len(names_blob)]
    return dict(bases=_get(lib.sh_bases, np.uint8).tobytes(), windows=_get(lib.sh_windows, np.uint64),
                names=[names_blob[int(name_off[i]):int(name_off[i + 1])] for i in range(len(name_off) - 1)],
                n_records=int(lib.sh_records()))


def expected(tmp_path, files, k, want_names):
    from yacht_b200 import sketch
    recs, names = [], []
    for i, data in enumerate(files):
        p = tmp_path / f"in{i}"
        p.write_bytes(data)
        rs = sketch.read_records(str(p))
        recs.extend(rs)
        fasta = data.lstrip()[:1] == b">"
        names.extend(n.encode() for n, _ in rs if want_names == 2 or fasta)
    bases = b"".join(b"\n" + s for _, s in recs)
    win = [(r << 32) | j for r, (_, s) in enumerate(recs) for j in range(len(s) - k + 1)]
    return dict(bases=bases, windows=np.array(sorted(win), dtype=np.uint64), names=names, n_records=len(recs))


def splits(data, k, seed):
    n = len(data)
    out = {f"every_{c}": list(range(c, n, c)) for c in (1, 2, 3, k - 1, k, k + 1, 4095, 4096, 4097)}
    rng = np.random.default_rng(seed)
    out["random"] = sorted(set(int(x) for x in rng.integers(1, max(n, 2), size=max(1, n // 50))) & set(range(1, n)))
    out["whole"] = []
    return out


def _check(got, exp):
    assert isinstance(got, dict), got
    assert got["bases"] == exp["bases"]
    assert got["n_records"] == exp["n_records"]
    assert np.array_equal(np.sort(got["windows"]), exp["windows"])          # every window once, in its record
    assert got["names"] == exp["names"]


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("case", sorted(accepted_cases()))
def test_chunked_parse_matches_record_path(walk, tmp_path, case, k):
    data = accepted_cases()[case]
    for want_names in (1, 2):
        exp = expected(tmp_path, [data], k, want_names)
        for split, cuts in splits(data, k, zlib.crc32(case.encode())).items():
            if split.startswith("every_1") and split != "every_1" or (split == "every_1" and len(data) > 3000):
                continue
            got = run_walk(walk, [data], k, lambda d: cuts, want_names)
            try:
                _check(got, exp)
            except AssertionError as e:
                raise AssertionError(f"{case} k={k} split={split} names={want_names}") from e


def test_chunked_parse_several_files(walk, tmp_path):
    cases = accepted_cases()
    files = [cases["fastq_plain"], cases["fasta_no_final_newline"], cases["only_whitespace"], cases["fastq_crlf_no_final_newline"]]
    for k in KS:
        exp = expected(tmp_path, files, k, 1)
        for step in (1, 7, k - 1, 4096):
            _check(run_walk(walk, files, k, lambda d: list(range(step, len(d), step)), 1), exp)


@pytest.mark.parametrize("case", sorted(rejected_cases()))
def test_chunked_parse_rejects_what_the_record_path_rejects(walk, tmp_path, case):
    from yacht_b200 import sketch
    data = rejected_cases()[case]
    p = tmp_path / "bad.fq"
    p.write_bytes(data)
    with pytest.raises(ValueError) as ei:
        sketch.read_records(str(p))
    want = str(ei.value)[len(str(p)) + 2:]
    for split, cuts in splits(data, 31, 5).items():
        assert run_walk(walk, [data], 31, lambda d: cuts, 2) == want, split


# ---- the Python reader behind a stand-in stream context -------------------------------------------------------------------

class _WalkContext:
    """Stands in for the GPU context: the stream calls go to the host walk of the parse, the sketch of its output is made by the
    oracle.  Records which byte ranges were fed, so that the reader's splitting is visible."""

    def __init__(self, lib):
        self.lib, self.feeds, self.files, self.cur = lib, [], [], bytearray()

    def host_buffer(self, n):
        buf = bytearray(n)
        arr = (ctypes.c_uint8 * n).from_buffer(buf)
        return memoryview(buf), ctypes.addressof(arr), lambda: None

    def stream_begin(self, ksize, max_hash, seed=42, per_record=False):
        self.k, self.max_hash, self.per_record = ksize, max_hash, per_record
        self.files, self.cur = [], bytearray()

    def stream_feed(self, ptr, n, path=None):
        self.feeds.append(n)
        self.cur += ctypes.string_at(ptr, n)

    def stream_end_file(self, path=None):
        self.files.append(bytes(self.cur))
        self.cur = bytearray()

    def stream_finish(self, path=None):
        got = run_walk(self.lib, self.files, self.k, lambda d: [], 2 if self.per_record else 1)
        if isinstance(got, str):
            raise ValueError(f"{path}: {got}")
        seqs = got["bases"].split(b"\n")[1:]
        groups = [[s] for s in seqs] if self.per_record else [seqs]
        hs, ab, off = [], [], [0]
        for g in groups:
            m, a = so.sketch_records(g, self.k, 100)
            hs.append(m); ab.append(a); off.append(off[-1] + len(m))
        cat = (lambda xs, t: np.concatenate(xs).astype(t) if xs else np.zeros(0, t))
        return cat(hs, np.uint64), cat(ab, np.uint32), np.array(off, np.uint64), got["names"] or None, {}


def _gzip_members(data, parts):
    cut = [len(data) * i // parts for i in range(parts + 1)]
    return b"".join(gzip.compress(data[cut[i]:cut[i + 1]]) for i in range(parts))


def test_stream_reader_matches_record_path(walk, tmp_path, monkeypatch):
    from yacht_b200 import sketch
    fake = _WalkContext(walk)
    monkeypatch.setattr(sketch, "_context", lambda: fake)
    monkeypatch.setattr(sketch, "STREAM_READ_BYTES", 4097)
    cases = accepted_cases()
    fq = tmp_path / "r.fq"
    fq.write_bytes(cases["fastq_plain"] * 3)
    fqgz = tmp_path / "r2.fq.gz"
    fqgz.write_bytes(_gzip_members(cases["fastq_plain"].replace(b"\n", b"\r\n") * 4, 3))          # three gzip members
    fa = tmp_path / "g.fa.gz"
    fa.write_bytes(_gzip_members(cases["fasta_wrapped"] + cases["fasta_empty_header_and_body"], 2))
    for paths, per_record in (([str(fq)], False), ([str(fq), str(fqgz)], False), ([str(fa)], True), ([str(fqgz)], True)):
        sketches, names = sketch.sketch_stream(paths, 31, 100, per_record=per_record)
        recs = [r for p in paths for r in sketch.read_records(p)]
        if per_record:
            assert names == [n for n, _ in recs]
            groups = [[s] for _, s in recs]
        else:
            groups = [[s for _, s in recs]]
        assert len(sketches) == len(groups)
        for (mins, ab), g in zip(sketches, groups):
            em, ea = so.sketch_records(g, 31, 100)
            assert np.array_equal(mins, em) and np.array_equal(ab, ea)
    assert max(fake.feeds) == 4097 and len(fake.feeds) > 10


def test_stream_reader_raises_reader_errors(walk, tmp_path, monkeypatch):
    from yacht_b200 import sketch
    monkeypatch.setattr(sketch, "_context", lambda: _WalkContext(walk))
    monkeypatch.setattr(sketch, "STREAM_READ_BYTES", 1000)
    data = gzip.compress(accepted_cases()["fastq_plain"] * 5)
    bad = tmp_path / "cut.fq.gz"
    bad.write_bytes(data[: len(data) // 2])                   # truncated gzip: the reader thread fails mid-file
    with pytest.raises(EOFError):
        sketch.sketch_stream([str(bad)], 31, 100)
    junk = tmp_path / "junk.fq"
    junk.write_bytes(rejected_cases()["fastq_bad_plus"])
    with pytest.raises(ValueError, match="malformed FASTQ record at line 5"):
        sketch.sketch_stream([str(junk)], 31, 100)


def test_small_inputs_keep_the_record_path(tmp_path, monkeypatch):
    from yacht_b200 import sketch
    p = tmp_path / "a.fa"
    p.write_bytes(accepted_cases()["fasta_wrapped"])
    assert not sketch.is_streamed(str(p))
    monkeypatch.setattr(sketch, "STREAM_FILE_BYTES", 100)
    assert sketch.is_streamed(str(p))
