"""`yacht sketch ref --kmer 21,31,51` and `yacht train --ksize K` on the zip it writes, host side (no GPU): the multi-size
batching and merging of yacht_b200/sketch.py behind an oracle-backed stand-in context, the command line, and the train
core's file list on zips that hold several k-mer sizes."""
import argparse
import csv
import gzip
import io
import json
import os
import zipfile

import numpy as np
import pandas as pd
import pytest

from oracle import sketch_oracle as so
from yacht_b200 import sigio, sketch, sketch_ref_genomes, utils


def _random_sequence(rng, n, p_bad=0.01):
    seq = rng.choice(np.frombuffer(b"ACGTacgt", dtype=np.uint8), size=n)
    bad = rng.random(n) < p_bad
    return np.where(bad, ord("N"), seq).astype(np.uint8).tobytes()


class _OracleBackedContext:
    """Stands in for the GPU context: every sketch is the C oracle's.  `uploads` counts device calls (one per batch, what
    ygpu_sketch_sequences_k copies once), `hashed` the (batch, k-mer size) pairs hashed."""
    def __init__(self):
        self.uploads = []
        self.hashed = []

    def _one(self, bases, offsets, ksize, max_hash, seed):
        hs, ab, off = [], [], [0]
        lib = so._load()
        for s in range(len(offsets) - 1):
            chunk = bases[int(offsets[s]):int(offsets[s + 1])]
            n = len(chunk)
            kept = np.empty(max(n, 1), dtype=np.uint64)
            buf = np.frombuffer(chunk, dtype=np.uint8) if n else np.zeros(1, np.uint8)
            got = lib.so_sketch_record(buf.ctypes.data, n, ksize, seed, max_hash, kept.ctypes.data, n) if n >= ksize else 0
            m, a = np.unique(kept[:got], return_counts=True)
            hs.append(m.astype(np.uint64)); ab.append(a.astype(np.uint32)); off.append(off[-1] + len(m))
        self.hashed.append((len(self.uploads) - 1, ksize))
        return np.concatenate(hs), np.concatenate(ab), np.array(off, np.uint64), 0

    def sketch_sequences(self, bases, offsets, ksize, max_hash, seed=42):
        self.uploads.append(len(bases))
        return self._one(bytes(bases), offsets, ksize, max_hash, seed)

    def sketch_sequences_k(self, bases, offsets, ksizes, max_hash, seed=42):
        assert 1 <= len(ksizes) <= 8 and len(set(ksizes)) == len(ksizes)
        self.uploads.append(len(bases))
        bases = bytes(bases)
        return [self._one(bases, offsets, k, max_hash, seed) for k in ksizes]


@pytest.fixture
def fake(monkeypatch):
    ctx = _OracleBackedContext()
    monkeypatch.setattr(sketch, "_context", lambda: ctx)
    return ctx


def _write_fasta(path, recs, gz=False):
    data = b"".join(b">" + n.encode() + b"\n" + b"\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + b"\n" for n, s in recs)
    with (gzip.open if gz else open)(path, "wb") as f:
        f.write(data)


@pytest.fixture
def genome_folder(tmp_path):
    """Genomes of several records, gzip and plain, of every suffix the reference globs for, one nested; plus a record
    shorter than 21 bases and one between 21 and 51 bases."""
    rng = np.random.default_rng(7)
    folder = tmp_path / "genomes"
    (folder / "sub").mkdir(parents=True)
    suffixes = [".fna.gz", ".fa", ".fasta", ".fas.gz", ".fna", "sub/.fa.gz"]
    for g, suf in enumerate(suffixes):
        d, ext = (folder / "sub", suf[4:]) if suf.startswith("sub/") else (folder, suf)
        recs = [(f"g{g}_c{c} contig", _random_sequence(rng, int(rng.integers(2_000, 9_000)))) for c in range(1 + g % 3)]
        if g == 2:
            recs += [("short", b"ACGTACGTAC"), ("mid", _random_sequence(rng, 40, p_bad=0.0))]
        _write_fasta(d / f"G{g}{ext}", recs, gz=ext.endswith(".gz"))
    return folder


def _manifest(zip_path):
    with zipfile.ZipFile(zip_path) as z:
        text = z.read(sigio.MANIFEST_NAME).decode()
    return [r for r in csv.reader(io.StringIO(text)) if r and not r[0].startswith("#")][1:]


def _members(zip_path):
    with zipfile.ZipFile(zip_path) as z:
        return {n: gzip.decompress(z.read(n)) for n in z.namelist() if n.startswith("signatures/")}


def _run_ref(infile, kmer, outfile, scaled=50):
    sketch_ref_genomes.main(argparse.Namespace(infile=str(infile), kmer=kmer, scaled=scaled, outfile=str(outfile)))


# ---- command line -------------------------------------------------------------------------------------------------------

def test_cli_ref_takes_several_kmer_sizes_comma_separated(capsys):
    p = argparse.ArgumentParser()
    sketch_ref_genomes.add_arguments(p)
    assert p.parse_args(["--infile", "refs", "--kmer", "21,31,51", "--outfile", "r.sig.zip"]).kmer == [21, 31, 51]
    assert p.parse_args(["--infile", "refs", "--kmer", "51,21", "--outfile", "r.sig.zip"]).kmer == [51, 21]
    one = p.parse_args(["--infile", "refs", "--kmer", "51", "--outfile", "r.sig.zip"]).kmer
    assert one == 51 and type(one) is int                               # one value: an int, as before
    assert p.parse_args(["--infile", "refs", "--outfile", "r.sig.zip"]).kmer == 31
    for bad in ("21,x", "21,,31", "", "21 31"):
        with pytest.raises(SystemExit):
            p.parse_args(["--infile", "refs", "--kmer", bad, "--outfile", "r.sig.zip"])
        assert "comma-separated list of sizes" in capsys.readouterr().err, bad


@pytest.mark.parametrize("kmer", [[31], 31])
def test_one_value_takes_the_single_size_path(tmp_path, monkeypatch, kmer):
    seen = []
    monkeypatch.setattr(sketch, "sketch_files", lambda paths, ksize, *a, **kw: seen.append(ksize) or [])
    monkeypatch.setattr(sketch, "write_sketches", lambda outfile, sketches, ksize, scaled: seen.append(("write", ksize)))
    (tmp_path / "g").mkdir()
    _run_ref(tmp_path / "g", kmer, tmp_path / "r.sig.zip")
    assert seen == [31, ("write", 31)] and type(seen[0]) is int


def test_ref_refuses_duplicate_sizes(tmp_path, capsys):
    folder = tmp_path / "g"
    folder.mkdir()
    with pytest.raises(ValueError, match="21 given more than once"):
        _run_ref(folder, [21, 31, 21], tmp_path / "o.sig.zip")
    assert not (tmp_path / "o.sig.zip").exists() and not (folder / "dataset.csv").exists()
    out = capsys.readouterr()
    assert "Sketching" not in out.out + out.err


def test_ref_and_sample_refuse_duplicates_with_the_same_message(tmp_path):
    from yacht_b200 import sketch_sample
    msgs = []
    for mod, infile in ((sketch_ref_genomes, str(tmp_path)), (sketch_sample, [str(tmp_path / "r.fq")])):
        with pytest.raises(ValueError) as e:
            mod.main(argparse.Namespace(infile=infile, kmer=[51, 21, 51, 21], scaled=1000, outfile=str(tmp_path / "o.sig.zip")))
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1] == "--kmer: k-mer size(s) 21, 51 given more than once."


# ---- multi-size output equals single-size output per size ----------------------------------------------------------------

def _assert_multi_equals_singles(multi_zip, single_zips, sizes):
    """multi_zip: genome- or record-major, sizes in the order of `sizes`; single_zips[k]: the run at size k alone."""
    rows = _manifest(multi_zip)
    members = _members(multi_zip)
    singles = {k: _manifest(single_zips[k]) for k in sizes}
    n = len(singles[sizes[0]])
    assert len(rows) == n * len(sizes)
    for k in sizes:
        assert len(singles[k]) == n
    for i, row in enumerate(rows):
        k = sizes[i % len(sizes)]
        assert row == singles[k][i // len(sizes)], (i, k)              # location, md5, ksize, scaled, n_hashes, name, filename
        assert int(row[3]) == k
    for k in sizes:                                                     # the signature files themselves, byte for byte
        single_members = _members(single_zips[k])
        for row in singles[k]:
            assert members[row[0]] == single_members[row[0]]
    by_k = {k: [s for s in sigio.read_sig_zip(str(multi_zip)) if s.ksize == k] for k in sizes}
    for k in sizes:
        want = sigio.read_sig_zip(str(single_zips[k]))
        assert [(s.name, s.filename, s.md5sum) for s in by_k[k]] == [(s.name, s.filename, s.md5sum) for s in want]
        for a, b in zip(by_k[k], want):
            assert np.array_equal(a.mins, b.mins) and np.array_equal(a.abundances, b.abundances)


@pytest.mark.parametrize("sizes", [[21, 31, 51], [51, 21]])
def test_folder_multi_size_equals_single_size_runs(tmp_path, fake, genome_folder, monkeypatch, sizes):
    monkeypatch.setattr(sketch, "CHUNK_FILE_BYTES", 12_000)          # several read-ahead chunks
    singles = {}
    for k in sizes:
        singles[k] = tmp_path / f"k{k}.sig.zip"
        _run_ref(genome_folder, k, singles[k])
    dataset_single = (genome_folder / "dataset.csv").read_text()
    n_single_uploads = len(fake.uploads)
    fake.uploads.clear()
    fake.hashed.clear()
    multi = tmp_path / "multi.sig.zip"
    _run_ref(genome_folder, list(sizes), multi)
    assert (genome_folder / "dataset.csv").read_text() == dataset_single
    _assert_multi_equals_singles(multi, singles, sizes)
    # every batch is uploaded once and hashed at every size
    assert len(fake.uploads) * len(sizes) == n_single_uploads
    assert fake.hashed == [(b, k) for b in range(len(fake.uploads)) for k in sizes]
    # and the sketches are the oracle's
    for s in sigio.read_sig_zip(str(multi)):
        path = next(p for p in genome_folder.rglob("*") if p.name.startswith(s.name + "."))
        em, ea = so.sketch_records([seq for _, seq in so.read_records(str(path))], s.ksize, 50)
        assert np.array_equal(s.mins, em) and np.array_equal(s.abundances, ea), (s.name, s.ksize)


def test_single_file_multi_size_equals_single_size_runs(tmp_path, fake, genome_folder):
    path = genome_folder / "G2.fasta"                                   # several records, one shorter than every size
    sizes = [21, 31, 51]
    singles = {}
    for k in sizes:
        singles[k] = tmp_path / f"k{k}.sig.zip"
        _run_ref(path, k, singles[k], scaled=1)
    multi = tmp_path / "multi.sig.zip"
    _run_ref(path, sizes, multi, scaled=1)
    _assert_multi_equals_singles(multi, singles, sizes)
    rows = _manifest(multi)                                             # (empty sketches of one size share a member)
    names = [r[9] for r in rows]
    assert names[:3] == ["g2_c0 contig"] * 3 and names[-6:] == ["short"] * 3 + ["mid"] * 3
    # the 10-base record has no window at any size, the 40-base record none at k = 51
    by = {(r[9], int(r[3])): int(r[7]) for r in rows}
    assert by[("short", 21)] == by[("short", 51)] == by[("mid", 51)] == 0 and by[("mid", 21)] > 0


def test_multi_size_sig_output(tmp_path, fake, genome_folder):
    """`--outfile x.sig`: one JSON record per (genome, size), in order, as the zip."""
    sizes = [31, 21]
    out = tmp_path / "multi.sig"
    _run_ref(genome_folder, sizes, out)
    recs = json.loads(out.read_text())
    assert [r["signatures"][0]["ksize"] for r in recs] == sizes * (len(recs) // 2)
    zipped = tmp_path / "multi.sig.zip"
    _run_ref(genome_folder, sizes, zipped)
    assert [(r["name"], r["signatures"][0]["md5sum"]) for r in recs] == [(s.name, s.md5sum) for s in sigio.read_sig_zip(str(zipped))]


def test_group_split_over_batches_is_merged_per_size(fake, monkeypatch):
    monkeypatch.setattr(sketch, "BATCH_BASES", 50_000)
    rng = np.random.default_rng(23)
    unit = _random_sequence(rng, 30_000, p_bad=0.0)
    groups = [[unit, unit[:10_000], _random_sequence(rng, 45_000), unit], [_random_sequence(rng, 5_000)], [], [_random_sequence(rng, 70_000)],
              [b"ACGT"], [_random_sequence(rng, 20_000), _random_sequence(rng, 20_000), _random_sequence(rng, 20_000)]]
    sizes = [51, 21, 31]
    got = sketch.sketch_record_groups(groups, sizes, 50)
    uploads = len(fake.uploads)
    assert uploads >= 4 and len(got) == len(sizes) and all(len(g) == len(groups) for g in got)
    for ki, k in enumerate(sizes):
        single = sketch.sketch_record_groups(groups, k, 50)
        for g, (mins, ab), (sm, sa) in zip(groups, got[ki], single):
            em, ea = so.sketch_records(g, k, 50)
            assert np.array_equal(mins, em) and np.array_equal(ab, ea), k
            assert np.array_equal(mins, sm) and np.array_equal(ab, sa) and mins.dtype == sm.dtype and ab.dtype == sa.dtype
    assert len(fake.uploads) == uploads * (1 + len(sizes))              # each single-size pass makes the same batches


# ---- `yacht train --ksize K` on a zip of several sizes: the train core's file list ------------------------------------

def _odd_members(z):
    """Members the train ingest meets besides signatures of the zip's sizes (tests/test_train_ingest.py): an empty sketch,
    an uncompressed .sig, a stray file in signatures/ and one elsewhere; plus a document without any sketch, a file that is
    not JSON, and one document holding sketches of 21 and 31 together."""
    z.writestr("signatures/empty.sig.gz", gzip.compress(sigio.signature_json("nothing", [], 31).encode()))
    z.writestr("signatures/plain.sig", sigio.signature_json("plain one", [5, 6, 7, 8], 31))
    z.writestr("signatures/README.txt", "not a signature")
    z.writestr("notes/extra.txt", "kept as is")
    z.writestr("signatures/no_sketch.sig", json.dumps([{"class": "sourmash_signature", "name": "none", "signatures": []}]))
    z.writestr("signatures/broken.sig.gz", gzip.compress(b"[{\"signatures\": [ {"))
    both = json.loads(sigio.signature_json("both", [9, 10], 21))
    both[0]["signatures"].append(json.loads(sigio.signature_json("both", [11, 12, 13], 31))[0]["signatures"][0])
    z.writestr("signatures/both.sig", json.dumps(both))


# k-mer sizes of each odd member's sketches (None: not a signature holding a sketch): listed unless it holds sketches and
# none of the trained size
ODD_SIZES = {"empty.sig": {31}, "plain.sig": {31}, "README.txt": None, "no_sketch.sig": None, "broken.sig": None, "both.sig": {21, 31}}


def _odd_listed(ksize, odd_sizes=ODD_SIZES):
    return {f for f, ks in odd_sizes.items() if ks is None or ksize in ks}


def _make_zip(path, sizes, n=12, extra=None):
    rng = np.random.default_rng(len(sizes) * 100 + n)
    sk = []
    for g in range(n):
        for k in sizes:
            mins = np.unique(rng.integers(1, 2 ** 63, size=int(rng.integers(20, 60)), dtype=np.uint64))
            sk.append(dict(name=f"genome {g}", mins=mins, abundances=(np.arange(len(mins)) % 5 + 1) if g % 3 == 0 else None, ksize=k))
    sigio.write_sig_zip(str(path), sk, sizes[0])
    with zipfile.ZipFile(str(path), "a") as z:
        _odd_members(z)
        if extra:
            extra(z)
    return sk


def _train_list(tmp_path, ref_zip, ksize, monkeypatch, name):
    """extract + run_yacht_train_core with the executable replaced by a stand-in that selects every listed file with an
    info tuple: returns the list the core was given, the info dict and the manifest frame."""
    d = str(tmp_path / name)
    os.makedirs(d)
    info, other = utils.extract_signatures(str(ref_zip), d, ksize, 1)
    paths = {v[-1] for v in info.values()}

    def fake_core(cmd):
        parts = cmd.split()
        listed = open(parts[-3]).read().splitlines()
        with open(parts[-1], "w") as f:
            f.writelines(p + "\n" for p in listed if p in paths)
        return 0

    monkeypatch.setattr(utils.os, "system", fake_core)
    manifest = utils.run_yacht_train_core(1, 0.95, ksize, d, info, other_size_files=other)
    listed = open(os.path.join(d, "training_sig_files.tsv")).read().splitlines()
    return d, listed, info, manifest


def test_single_size_zip_lists_every_file_as_before(tmp_path, monkeypatch, capsys):
    ref_zip = tmp_path / "k31.zip"
    _make_zip(ref_zip, [31])
    d, listed, info, manifest = _train_list(tmp_path, ref_zip, 31, monkeypatch, "t")
    sig_dir = os.path.join(d, "signatures")
    assert listed == [os.path.join(sig_dir, f) for f in os.listdir(sig_dir)]      # the parent's expression, same order
    assert len(listed) == 12 + len(ODD_SIZES) and len(info) == 12 + 2          # + "plain one", "both"
    assert len(manifest) == len(info)
    assert "Leaving out" not in capsys.readouterr().out


@pytest.mark.parametrize("ksize", [31, 51, 21])
def test_multi_size_zip_lists_only_the_trained_size_and_odd_members(tmp_path, monkeypatch, capsys, ksize):
    sizes = [21, 31, 51]
    multi = tmp_path / "multi.zip"
    empty_k51 = lambda z: z.writestr("signatures/empty_k51.sig.gz", gzip.compress(sigio.signature_json("nothing 51", [], 51).encode()))
    sk = _make_zip(multi, sizes, extra=empty_k51)
    d, listed, info, manifest = _train_list(tmp_path, multi, ksize, monkeypatch, "multi")
    log = capsys.readouterr().out
    sig_dir = os.path.join(d, "signatures")
    assert len(os.listdir(sig_dir)) == 12 * 3 + len(ODD_SIZES) + 1              # extraction unchanged: every member lands
    want_k = {sigio.compute_md5sum(ksize, s["mins"]) + ".sig" for s in sk if s["ksize"] == ksize}
    odd_sizes = dict(ODD_SIZES, **{"empty_k51.sig": {51}})
    odd = _odd_listed(ksize, odd_sizes)
    assert {os.path.basename(p) for p in listed} == want_k | odd
    assert listed == [os.path.join(sig_dir, f) for f in os.listdir(sig_dir) if f in want_k | odd]
    assert f"Leaving out {12 * 2 + len(odd_sizes) - len(odd)} signature files" in log
    warned = {os.path.basename(line.split(": ")[-1]) for line in log.splitlines() if "CANNOT extract" in line}
    assert warned and warned <= odd                                              # no warning for a file left out
    # the same genomes, infos and manifest as training a zip of that size alone
    single = tmp_path / f"k{ksize}.zip"
    sigio.write_sig_zip(str(single), [s for s in sk if s["ksize"] == ksize], ksize)
    with zipfile.ZipFile(str(single), "a") as z:
        _odd_members(z)
        empty_k51(z)
    _, single_listed, single_info, single_manifest = _train_list(tmp_path, single, ksize, monkeypatch, "single")
    rel = lambda dd: {k: v[:4] + (os.path.basename(v[4]),) for k, v in dd.items()}
    assert rel(info) == rel(single_info)
    assert sorted(map(os.path.basename, listed)) == sorted(map(os.path.basename, single_listed))
    pd.testing.assert_frame_equal(manifest.sort_values("organism_name").reset_index(drop=True),
                                  single_manifest.sort_values("organism_name").reset_index(drop=True))
