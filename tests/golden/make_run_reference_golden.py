"""Run-path golden vectors produced by the UNMODIFIED reference code (not by a restatement).

Run in the build container (needs /root/reference; the GPU box never runs this):
    python tests/golden/make_run_reference_golden.py

What executes here is the reference's own src/yacht/hypothesis_recovery_src.py and src/yacht/utils.py, imported as
they lie under /root/reference.  Two things they depend on are absent from this image and are supplied as stand-ins:

  * the ``sourmash`` Python package (module-top ``import sourmash`` of both files; the only call either file makes on
    this path is ``sourmash.load_file_as_signatures(filename, ksize=...)``, utils.py:42).  The stand-in below parses the
    signature JSON with the ``json`` module and serves objects carrying ``.minhash.hashes`` (a dict hash -> abundance,
    like sourmash's), ``.name`` and ``.md5sum()``; it yields only the sub-signatures of the requested k-mer size, as
    sourmash does.
  * the ``sourmash scripts multisearch`` command line (sourmash_plugin_branchwater, third-party Rust, not vendored;
    hypothesis_recovery_src.py:93).  Only part B needs it: a stand-in executable named ``sourmash`` is put on PATH that
    writes the ``match_name`` rows multisearch documents for ``-t 0`` (every query/match pair that shares a hash).
    That stand-in IS a restatement (row a10 stays "pinned by definition + the reference's workflow known answer");
    everything downstream of its CSV -- name filtering, the sub-manifest, get_exclusive_hashes, single_hyp_test via
    multiprocessing.Pool, the result frames -- is the reference's own code.

The package ``yacht`` is entered through a synthetic parent module (``__path__`` -> /root/reference/src/yacht) so that
the package's ``__init__`` (which imports the download/CLI modules) does not run; no reference file is modified or
copied.

Part A (50 seeded databases): get_exclusive_hashes(manifest, names, sample_sig, ksize, dir) for several name lists
per database, and single_hyp_test for every (n_exclusive, n_match) pair that came out, over a grid of
(ksize, significance, ani, min_coverage).
Part B (6 databases): the whole hypothesis_recovery(...) call, one frame per min_coverage.

Output: tests/golden/run_reference_golden.npz (the tests never need /root/reference).  It holds what the reference
returned; the inputs it was given -- the seeded databases and samples of make_case(), the single_hyp_test arguments -- are
made again from their seeds by load(), which checks them against checksums stored beside the outputs (pack()).
"""
import gzip
import hashlib
import importlib
import io
import json
import os
import shutil
import stat
import sys
import tempfile
import types
import zipfile

import numpy as np
import pandas as pd

REF = os.environ.get("YACHT_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "run_reference_golden.npz")
MAX_HASH = 18446744073709552          # scaled = 1000
N_CASES_A = 50
N_CASES_B = 6
HYP_GRID = [(31, 0.99, 0.95), (51, 0.95, 0.95), (21, 0.90, 0.90), (31, 0.99, 0.995)]
COVS = [1, 0.5, 0.1, 0.05, 0.01]


# ------------------------------------------------------------------------------------------------ stand-ins
class _MinHash:
    def __init__(self, sub):
        mins = sub["mins"]
        abund = sub.get("abundances")
        self.hashes = dict(zip(mins, abund if abund is not None else [1] * len(mins)))
        self.ksize = sub["ksize"]
        self.track_abundance = abund is not None
        self.scaled = int(round((2 ** 64 - 1) / sub["max_hash"])) if sub.get("max_hash") else 0
        self._md5 = sub.get("md5sum", "")

    def __len__(self):
        return len(self.hashes)


class _Signature:
    def __init__(self, rec, sub):
        self.name = rec.get("name", "")
        self.filename = rec.get("filename", "")
        self.minhash = _MinHash(sub)

    def md5sum(self):
        return self.minhash._md5


def _load_file_as_signatures(filename, ksize=None, **_):
    opener = gzip.open if filename.endswith(".gz") else open
    with opener(filename, "rt") as f:
        recs = json.load(f)
    for rec in recs:
        for sub in rec["signatures"]:
            if ksize is None or sub["ksize"] == ksize:
                yield _Signature(rec, sub)


FAKE_CLI = r'''#!%(python)s
# stand-in for `sourmash scripts multisearch QUERY_LIST AGAINST_LIST -s S -k K -c C -t 0 -o OUT` (see make_run_reference_golden.py)
import csv, json, sys
a = sys.argv[1:]
assert a[0] == "scripts" and a[1] == "multisearch", a
qlist, rlist = a[2], a[3]
opt = dict(zip(a[4::2], a[5::2]))
k, scaled, thr, out = int(opt["-k"]), int(opt["-s"]), float(opt["-t"]), opt["-o"]
assert thr == 0.0
def load(path):
    res = []
    for rec in json.load(open(path)):
        for sub in rec["signatures"]:
            sc = int(round((2 ** 64 - 1) / sub["max_hash"])) if sub.get("max_hash") else 0
            if sub["ksize"] == k and sc == scaled:
                res.append((rec.get("name", ""), sub.get("md5sum", ""), set(sub["mins"])))
    return res
queries = [s for p in open(qlist).read().split() for s in load(p)]
against = [s for p in open(rlist).read().split() for s in load(p)]
rows = []
for qn, qm, qs in queries:
    for rn, rm, rs in against:
        n = len(qs & rs)
        if n > 0 and qs:
            rows.append((qn, qm, rn, rm, n / len(qs), n))
with open(out, "w", newline="") as f:
    if rows:
        w = csv.writer(f)
        w.writerow(["query_name", "query_md5", "match_name", "match_md5", "containment", "intersect_hashes"])
        w.writerows(rows)
'''


def import_reference():
    sm = types.ModuleType("sourmash")
    sm.load_file_as_signatures = _load_file_as_signatures
    sm.SourmashSignature = _Signature
    sys.modules["sourmash"] = sm
    pkg = types.ModuleType("yacht")
    pkg.__path__ = [os.path.join(REF, "src", "yacht")]
    sys.modules["yacht"] = pkg
    hr = importlib.import_module("yacht.hypothesis_recovery_src")
    assert os.path.realpath(hr.__file__).startswith(os.path.realpath(REF)), hr.__file__
    assert os.path.realpath(sys.modules["yacht.utils"].__file__).startswith(os.path.realpath(REF))
    try:
        from loguru import logger
        logger.remove()
    except Exception:
        pass
    return hr


# ------------------------------------------------------------------------------------------------ inputs
def md5_of(ksize, mins):
    m = hashlib.md5()
    m.update(str(ksize).encode("ascii"))
    for h in mins:
        m.update(str(h).encode("ascii"))
    return m.hexdigest()


def sig_text(name, subs):
    """subs: [(ksize, sorted mins)] -- one file may carry several k-mer sizes."""
    return json.dumps([{
        "class": "sourmash_signature", "email": "", "hash_function": "0.murmur64", "filename": name + ".fa", "name": name,
        "license": "CC0", "version": 0.4,
        "signatures": [{"num": 0, "ksize": k, "seed": 42, "max_hash": MAX_HASH, "mins": [int(h) for h in mins],
                        "md5sum": md5_of(k, [int(h) for h in mins]), "molecule": "dna"} for k, mins in subs],
    }], separators=(",", ":"))


def make_case(seed):
    """A small database with every sharing pattern the exclusive-hash step distinguishes."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(1, 48))
    wide = seed % 3 == 0
    total_hint = n * 120
    universe = MAX_HASH if wide else max(64, int(total_hint * rng.choice([0.6, 1.5, 4.0])))
    core = rng.integers(0, universe, size=int(rng.integers(1, 60)), dtype=np.uint64)       # shared by many genomes
    sketches = []
    for g in range(n):
        kind = rng.integers(0, 10)
        size = int(rng.integers(1, 400))
        own = rng.integers(0, universe, size=size, dtype=np.uint64)
        if kind == 0 and sketches:                                  # exact duplicate of an earlier genome
            s = sketches[int(rng.integers(0, len(sketches)))].copy()
        elif kind == 1 and sketches:                                # strict subset of an earlier genome
            p = sketches[int(rng.integers(0, len(sketches)))]
            s = p[rng.random(p.size) < 0.5]
            if s.size == 0:
                s = p[:1].copy()
        elif kind == 2:                                             # a single hash
            s = own[:1]
        elif kind in (3, 4, 5):                                     # core + own
            s = np.concatenate([core[rng.random(core.size) < 0.7], own])
        else:
            s = own
        sketches.append(np.unique(s))
    allh = np.unique(np.concatenate(sketches))
    mode = seed % 5
    if mode == 0:
        sample = allh[rng.random(allh.size) < 0.3]
    elif mode == 1:                                                 # one genome entirely + noise
        sample = np.concatenate([sketches[int(rng.integers(0, n))], rng.integers(0, universe, size=200, dtype=np.uint64)])
    elif mode == 2:                                                 # touches few genomes
        pick = rng.choice(n, size=min(n, 3), replace=False)
        sample = np.concatenate([sketches[int(g)][: max(1, sketches[int(g)].size // 3)] for g in pick])
    elif mode == 3:
        sample = np.concatenate([allh[rng.random(allh.size) < 0.05], rng.integers(0, MAX_HASH, size=500, dtype=np.uint64)])
    else:
        sample = allh.copy()
    sample = np.unique(sample)
    if sample.size == 0:
        sample = allh[:1].copy()
    return sketches, sample


def case_b_inputs(c):
    """Part B database c: hypothesis_recovery keys files by md5, so exact duplicates are dropped and manifest rows and
    files are one to one."""
    sketches, sample = make_case(100 + c)
    seen, uniq = set(), []
    for s in sketches:
        key = s.tobytes()
        if key not in seen:
            seen.add(key)
            uniq.append(s)
    return uniq, sample


def _csr(sketches):
    offsets = np.zeros(len(sketches) + 1, np.int64)
    np.cumsum([len(s) for s in sketches], out=offsets[1:])
    return np.concatenate(sketches).astype(np.uint64), offsets


def _checksum(hashes, sample):
    return [int(len(hashes)), int(np.bitwise_xor.reduce(hashes)), int(len(sample)), int(np.bitwise_xor.reduce(sample))]


def _hyp_in(pairs, meta):
    """single_hyp_test arguments in the generator's order: for each (n_exclusive, n_match), each grid point, each coverage."""
    return np.array([(ne, nm, k, sig, ani, cov) for ne, nm in pairs for k, sig, ani in meta["hyp_grid"] for cov in meta["covs"]],
                    dtype=np.float64)


def pack(out, meta):
    """The committed layout: the reference's outputs, and checksums of the seeded inputs instead of the inputs."""
    keep = {}
    for case in meta["cases_a"]:
        c = case["id"]
        case["inputs"] = _checksum(out[f"a{c}_hashes"], out[f"a{c}_sample"])
        keep[f"a{c}_overlap"] = out[f"a{c}_overlap"]
        for v in range(case["variants"]):
            keep[f"a{c}_mask{v}"], keep[f"a{c}_info{v}"] = out[f"a{c}_mask{v}"], out[f"a{c}_info{v}"]
    for case in meta["cases_b"]:
        case["inputs"] = _checksum(out[f"b{case['id']}_hashes"], out[f"b{case['id']}_sample"])
    pairs = np.array(sorted({(int(a), int(b)) for a, b in out["hyp_in"][:, :2]}), dtype=np.int64)
    assert np.array_equal(_hyp_in(pairs, meta), out["hyp_in"])
    keep["hyp_pairs"] = pairs
    keep["hyp_out_t"] = np.ascontiguousarray(out["hyp_out"].T)      # column by column: compresses to half
    keep["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    return keep


def load(path=OUT):
    """(arrays, meta) with every input and output array main() produced, the inputs made again from their seeds."""
    with np.load(path) as f:
        z = dict(f)
    meta = json.loads(bytes(z.pop("meta")).decode())
    for part, cases, make in (("a", meta["cases_a"], make_case), ("b", meta["cases_b"], case_b_inputs)):
        for case in cases:
            c = case["id"]
            sketches, sample = make(c)
            hashes, offsets = _csr(sketches)
            sample = sample.astype(np.uint64)
            assert _checksum(hashes, sample) == case["inputs"], \
                f"make_case no longer reproduces the inputs of case {part}{c} the reference was run on"
            z[f"{part}{c}_hashes"], z[f"{part}{c}_offsets"], z[f"{part}{c}_sample"] = hashes, offsets, sample
    z["hyp_in"] = _hyp_in(z.pop("hyp_pairs"), meta)
    z["hyp_out"] = np.ascontiguousarray(z.pop("hyp_out_t").T)
    return z, meta


def write_db(root, sketches, ksize, extra_ksize=None, seed=0):
    """root/signatures/<md5>.sig per genome (the layout `yacht train` leaves); returns the manifest frame."""
    os.makedirs(os.path.join(root, "signatures"))
    rows = []
    rng = np.random.default_rng(77 + seed)
    for g, s in enumerate(sketches):
        name = f"org_{g:03d}"
        subs = [(ksize, s)]
        if extra_ksize is not None and g % 2 == 0:       # a second k-mer size FIRST in the file: must not be picked
            other = np.unique(rng.integers(0, MAX_HASH, size=int(rng.integers(1, 50)), dtype=np.uint64))
            subs = [(extra_ksize, other), (ksize, s)]
        md5 = md5_of(ksize, [int(h) for h in s])
        # two genomes with identical sketches share one md5 / one file, as in the reference's layout
        with open(os.path.join(root, "signatures", md5 + ".sig"), "w") as f:
            f.write(sig_text(name, subs))
        rows.append((name, md5, len(s), len(s), 1000))
    return pd.DataFrame(rows, columns=["organism_name", "md5sum", "num_unique_kmers_in_genome_sketch",
                                       "num_total_kmers_in_genome_sketch", "genome_scale_factor"])


def write_sample_zip(path, name, ksize, sample):
    text = sig_text(name, [(ksize, sample)])
    md5 = md5_of(ksize, [int(h) for h in sample])
    with zipfile.ZipFile(path, "w", zipfile.ZIP_STORED) as z:
        z.writestr(f"signatures/{md5}.sig.gz", gzip.compress(text.encode(), compresslevel=1))
        z.writestr("SOURMASH-MANIFEST.csv", "# SOURMASH-MANIFEST-VERSION: 1.0\n"
                   "internal_location,md5,md5short,ksize,moltype,num,scaled,n_hashes,with_abundance,name,filename\n"
                   f"signatures/{md5}.sig.gz,{md5},{md5[:8]},{ksize},DNA,0,1000,{len(sample)},0,{name},{name}.fa\n")
    return text


# ------------------------------------------------------------------------------------------------ main
def main():
    if not os.path.isdir(REF):
        sys.exit(f"{REF} not found: this generator only runs where the reference is checked out")
    hr = import_reference()
    out = {}
    meta = {"reference_files": ["src/yacht/hypothesis_recovery_src.py", "src/yacht/utils.py"],
            "hyp_grid": HYP_GRID, "covs": COVS, "cases_a": [], "cases_b": []}
    tmp = tempfile.mkdtemp(prefix="yacht_refgold_")
    infos = set()
    try:
        # ---- part A
        for c in range(N_CASES_A):
            sketches, sample = make_case(c)
            ksize = [21, 31, 51][c % 3]
            # identical sketches would collide on the md5-named file AND on nothing else; keep them (same file content)
            root = os.path.join(tmp, f"a{c}")
            manifest = write_db(root, sketches, ksize, extra_ksize=(31 if ksize != 31 else 21) if c % 7 == 3 else None, seed=c)
            sample_sig = _Signature({"name": "sample"}, {"mins": [int(h) for h in sample], "ksize": ksize, "max_hash": MAX_HASH})
            n = len(sketches)
            sset = set(int(h) for h in sample)
            overlap = np.array([len(sset.intersection(int(h) for h in s)) for s in sketches])
            rng = np.random.default_rng(5000 + c)
            masks = [overlap > 0, np.ones(n, bool), rng.random(n) < 0.5, (overlap > 0) & (rng.random(n) < 0.7)]
            offsets = np.zeros(n + 1, np.int64)
            np.cumsum([len(s) for s in sketches], out=offsets[1:])
            out[f"a{c}_hashes"] = np.concatenate(sketches).astype(np.uint64)
            out[f"a{c}_offsets"] = offsets
            out[f"a{c}_sample"] = sample.astype(np.uint64)
            out[f"a{c}_overlap"] = overlap.astype(np.int64)
            nv = 0
            for m in masks:
                names = [nm for nm, keep in zip(manifest["organism_name"], m) if keep]
                info, sub = hr.get_exclusive_hashes(manifest, names, sample_sig, ksize, root)
                assert list(sub["organism_name"]) == names
                out[f"a{c}_mask{nv}"] = m.astype(np.uint8)
                out[f"a{c}_info{nv}"] = np.array(info, dtype=np.int64).reshape(-1, 2)
                infos.update((int(a), int(b)) for a, b in info)
                nv += 1
            meta["cases_a"].append({"id": c, "n": n, "ksize": ksize, "variants": nv})
        # ---- single_hyp_test over everything part A produced (+ the boundary pairs the reference's own tests use)
        infos.update([(3741, 2), (0, 0), (1, 0), (1, 1), (10, 11), (100000, 90000), (250000, 30000)])
        hin, hout = [], []
        for (ne, nm) in sorted(infos):
            for (k, sig, ani) in HYP_GRID:
                for cov in COVS:
                    r = hr.single_hyp_test((ne, nm), k, sig, ani, cov)
                    hin.append((ne, nm, k, sig, ani, cov))
                    hout.append(tuple(float(x) for x in r))
        out["hyp_in"] = np.array(hin, dtype=np.float64)
        out["hyp_out"] = np.array(hout, dtype=np.float64)
        # ---- part B: the whole hypothesis_recovery() call
        bindir = os.path.join(tmp, "bin")
        os.makedirs(bindir)
        cli = os.path.join(bindir, "sourmash")
        with open(cli, "w") as f:
            f.write(FAKE_CLI % {"python": sys.executable})
        os.chmod(cli, os.stat(cli).st_mode | stat.S_IXUSR | stat.S_IXGRP | stat.S_IXOTH)
        os.environ["PATH"] = bindir + os.pathsep + os.environ["PATH"]
        for c in range(N_CASES_B):
            sketches, sample = case_b_inputs(c)
            ksize, sig, ani = HYP_GRID[c % len(HYP_GRID)]
            root = os.path.join(tmp, f"b{c}")
            manifest = write_db(root, sketches, ksize, extra_ksize=(21 if ksize != 21 else 31) if c % 2 == 1 else None, seed=100 + c)
            sdir = os.path.join(tmp, f"b{c}_sample")
            os.makedirs(sdir)
            sample_file = os.path.join(sdir, "sample.sig.zip")
            write_sample_zip(sample_file, "sample", ksize, sample)
            sample_sig = _Signature({"name": "sample"}, {"mins": [int(h) for h in sample], "ksize": ksize, "max_hash": MAX_HASH})
            covs = COVS[: 2 + c % 3]
            frames = hr.hypothesis_recovery(manifest.copy(), (sample_file, sample_sig), root, covs, 1000, ksize, sig, ani, 2)
            offsets = np.zeros(len(sketches) + 1, np.int64)
            np.cumsum([len(s) for s in sketches], out=offsets[1:])
            out[f"b{c}_hashes"] = np.concatenate(sketches).astype(np.uint64)
            out[f"b{c}_offsets"] = offsets
            out[f"b{c}_sample"] = sample.astype(np.uint64)
            meta["cases_b"].append({
                "id": c, "ksize": ksize, "significance": sig, "ani": ani, "covs": covs, "seed": 100 + c,
                "extra_ksize": (21 if ksize != 21 else 31) if c % 2 == 1 else None,
                "frames": [json.loads(fr.to_json(orient="split", double_precision=15)) for fr in frames],
                "frames_exact": [{col: [repr(float(v)) for v in fr[col]] for col in
                                  ("p_vals", "acceptance_threshold_with_coverage", "actual_confidence_with_coverage",
                                   "alt_confidence_mut_rate_with_coverage")} for fr in frames],
            })
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    buf = io.BytesIO()
    np.savez_compressed(buf, **pack(out, meta))
    with open(OUT, "wb") as f:
        f.write(buf.getvalue())
    print(f"wrote {OUT}: {len(buf.getvalue())} bytes, {N_CASES_A} databases / {sum(c['variants'] for c in meta['cases_a'])} "
          f"get_exclusive_hashes calls, {len(hin)} single_hyp_test rows, {N_CASES_B} hypothesis_recovery calls")


if __name__ == "__main__":
    main()
