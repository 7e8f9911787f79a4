"""Sourmash-free reading / writing of sourmash signature files (the on-disk boundary format).

The reference obtains everything it needs from a signature through sourmash
(reference src/yacht/utils.py:31-51 ``load_signature_with_ksize`` and :89-110
``get_info_from_single_sig``).  sourmash is a third-party Rust/Python package that is not part of
the reference tree, so this module restates the handful of fields the hot path consumes directly
from the JSON text (format: SURVEY.md Appendix A):

* ``name``                      -> organism name
* ``signatures[k].mins``        -> the FracMinHash hashes (uint64, sorted ascending, unique)
* ``signatures[k].abundances``  -> optional; ``mean_abundance`` is their arithmetic mean
* ``signatures[k].max_hash``    -> ``scaled = round((2**64 - 1) / max_hash)``
* ``signatures[k].md5sum``      -> ``md5(str(ksize) + "".join(str(h) for h in mins))``

All 20 rows of the reference's own fixture tests/unittests_data/test_collect_signature_info_data.json
are reproduced by :func:`sig_info` (tests/test_sigio.py).
"""
from __future__ import annotations

import csv
import gzip
import hashlib
import io
import json
import os
import zipfile
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

MAX_HASH_SCALED_1000 = 18446744073709552  # == int((2**64 - 1) / 1000) as sourmash writes it
MANIFEST_NAME = "SOURMASH-MANIFEST.csv"
MANIFEST_COLUMNS = [
    "internal_location", "md5", "md5short", "ksize", "moltype", "num", "scaled",
    "n_hashes", "with_abundance", "name", "filename",
]


@dataclass
class Signature:
    """One (name, ksize) sketch: the subset of a sourmash signature the hot path reads."""
    name: str
    ksize: int
    mins: np.ndarray                      # uint64, ascending
    abundances: Optional[np.ndarray]      # int64 or None
    max_hash: int
    md5sum: str
    filename: str = ""
    molecule: str = "dna"
    path: str = ""

    @property
    def scaled(self) -> int:
        if self.max_hash == 0:
            return 0
        return int(round((2 ** 64 - 1) / self.max_hash))

    @property
    def mean_abundance(self) -> Optional[float]:
        # sourmash: MinHash.mean_abundance is None when abundances are not tracked
        if self.abundances is None:
            return None
        if len(self.abundances) == 0:
            return None
        return float(np.mean(self.abundances))

    def __len__(self) -> int:
        return int(self.mins.shape[0])


def compute_md5sum(ksize: int, mins: Sequence[int]) -> str:
    """md5 of ``str(ksize)`` followed by the decimal text of every hash (sourmash's definition)."""
    h = hashlib.md5()
    h.update(str(int(ksize)).encode())
    h.update("".join(str(int(x)) for x in mins).encode())
    return h.hexdigest()


def _open_text(path: str) -> str:
    with open(path, "rb") as f:
        head = f.read(2)
    if head == b"\x1f\x8b":
        with gzip.open(path, "rb") as f:
            return f.read().decode()
    with open(path, "rb") as f:
        return f.read().decode()


def parse_signature_json(text: str, path: str = "") -> List[Signature]:
    """All (record, sub-signature) sketches of a signature JSON document, in file order."""
    doc = json.loads(text)
    if isinstance(doc, dict):
        doc = [doc]
    out: List[Signature] = []
    for rec in doc:
        for sub in rec.get("signatures", []):
            mins = np.array(sub.get("mins", []), dtype=np.uint64)
            ab = sub.get("abundances")
            out.append(Signature(
                name=rec.get("name") or "",          # sourmash: sig.name is '' when the record carries no name (it does not fall back to the filename)
                ksize=int(sub.get("ksize", 0)),
                mins=mins,
                abundances=None if ab is None else np.array(ab, dtype=np.int64),
                max_hash=int(sub.get("max_hash", 0)),
                # the stored md5sum is trusted (recomputing it over ~5 000 decimal strings per sketch costs minutes of Python at
                # GTDB size); a record without one gets sourmash's definition computed
                md5sum=sub.get("md5sum") or compute_md5sum(int(sub.get("ksize", 0)), mins),
                filename=rec.get("filename", ""),
                molecule=sub.get("molecule", "dna"),
                path=path,
            ))
    return out


def load_signature_with_ksize(filename: str, ksize: int) -> Signature:
    """Mirror of reference utils.py:31-51: exactly one sketch of that k-mer size, and not empty.

    Accepts ``.sig``, ``.sig.gz`` and ``.sig.zip`` (a zip holding SOURMASH-MANIFEST.csv and
    ``signatures/*.sig.gz``).  Raises the same ``ValueError`` messages as the reference.
    """
    if zipfile.is_zipfile(filename):
        sigs = [s for s in read_sig_zip(filename) if s.ksize == ksize]
    else:
        sigs = [s for s in parse_signature_json(_open_text(filename), filename) if s.ksize == ksize]
    if len(sigs) != 1:
        raise ValueError(
            f"Expected exactly one signature with ksize {ksize} in {filename}, found {len(sigs)}"
        )
    if len(sigs[0]) == 0:
        raise ValueError(
            "Empty sketch in signature. This may be due to too high of a scale factor, please reduce it, eg. --scaled=1, and try again."
        )
    return sigs[0]


def read_sig_zip(zip_path: str) -> List[Signature]:
    """Every sketch inside a sourmash zip database, in manifest order when a manifest exists."""
    out: List[Signature] = []
    with zipfile.ZipFile(zip_path, "r") as z:
        names = z.namelist()
        order = [n for n in names if n.startswith("signatures/") and not n.endswith("/")]
        if MANIFEST_NAME in names:
            rows = list(csv.reader(io.StringIO(z.read(MANIFEST_NAME).decode())))
            rows = [r for r in rows if r and not r[0].startswith("#")]
            if rows and rows[0][0] == "internal_location":
                rows = rows[1:]
            seen = []
            for r in rows:
                if r[0] in names and r[0] not in seen:
                    seen.append(r[0])
            if seen:
                order = seen
        for n in order:
            raw = z.read(n)
            if raw[:2] == b"\x1f\x8b":
                raw = gzip.decompress(raw)
            out.extend(parse_signature_json(raw.decode(), os.path.join(zip_path, n)))
    return out


def sig_info(sig_file: str, ksize: int):
    """Mirror of reference utils.py:89-110: (path, name, md5, mean abundance, n hashes, scaled)."""
    try:
        sig = load_signature_with_ksize(sig_file, ksize)
        return (sig_file, sig.name, sig.md5sum, sig.mean_abundance, len(sig), sig.scaled)
    except Exception:
        return None


def sig_info_from_signatures(signatures: Sequence[Signature], sig_file: str, ksize: int):
    """:func:`sig_info` for a signature document already parsed by :func:`parse_signature_json` (`sig_file` is the path
    it was, or is being, written to): same selection rule -- exactly one non-empty sketch of that k-mer size -- same tuple."""
    try:
        sigs = [s for s in signatures if s.ksize == ksize]
        if len(sigs) != 1 or len(sigs[0]) == 0:
            return None
        sig = sigs[0]
        return (sig_file, sig.name, sig.md5sum, sig.mean_abundance, len(sig), sig.scaled)
    except Exception:
        return None


def signature_json(name: str, mins: Sequence[int], ksize: int = 31,
                   abundances: Optional[Sequence[int]] = None,
                   max_hash: int = MAX_HASH_SCALED_1000, filename: str = "") -> str:
    """Text of a one-sketch signature file laid out like sourmash writes it (Appendix A)."""
    mins_list = [int(x) for x in mins]
    sub = {
        "num": 0, "ksize": int(ksize), "seed": 42, "max_hash": int(max_hash),
        "mins": mins_list, "md5sum": compute_md5sum(ksize, mins_list),
    }
    if abundances is not None:
        sub["abundances"] = [int(a) for a in abundances]
    sub["molecule"] = "dna"
    rec = {
        "class": "sourmash_signature", "email": "", "hash_function": "0.murmur64",
        "filename": filename, "name": name, "license": "CC0", "signatures": [sub], "version": 0.4,
    }
    return json.dumps([rec], separators=(",", ":"))


def write_signature(path: str, name: str, mins: Sequence[int], ksize: int = 31,
                    abundances: Optional[Sequence[int]] = None,
                    max_hash: int = MAX_HASH_SCALED_1000, filename: str = "") -> str:
    """Write ``path`` (gzip when it ends in .gz); returns the sketch md5sum."""
    text = signature_json(name, mins, ksize, abundances, max_hash, filename)
    data = text.encode()
    if path.endswith(".gz"):
        with gzip.open(path, "wb", compresslevel=1) as f:
            f.write(data)
    else:
        with open(path, "wb") as f:
            f.write(data)
    return compute_md5sum(ksize, [int(x) for x in mins])


def write_signatures(path: str, sketches: Sequence[dict], ksize: int = 31, max_hash: int = MAX_HASH_SCALED_1000) -> None:
    """One JSON signature file holding several sketches (what ``sourmash sketch dna -o x.sig`` writes for several
    records); gzip when ``path`` ends in .gz.  ``sketches``: dicts with ``name``, ``mins`` and optional ``abundances``,
    ``filename`` and ``ksize`` (default: the argument), one JSON record each, in order."""
    recs = []
    for sk in sketches:
        recs.extend(json.loads(signature_json(sk["name"], sk["mins"], sk.get("ksize", ksize), sk.get("abundances"), max_hash,
                                              sk.get("filename", ""))))
    data = json.dumps(recs, separators=(",", ":")).encode()
    if path.endswith(".gz"):
        with gzip.open(path, "wb", compresslevel=1) as f:
            f.write(data)
    else:
        with open(path, "wb") as f:
            f.write(data)


def write_sig_zip(zip_path: str, sketches: Sequence[dict], ksize: int = 31,
                  max_hash: int = MAX_HASH_SCALED_1000) -> None:
    """Write a sourmash-style zip database (manifest + signatures/<md5>.sig.gz).

    ``sketches``: dicts with ``name``, ``mins`` and optional ``abundances``, ``filename`` and ``ksize`` (default: the
    argument); one signature file and one manifest row each, in order.
    """
    scaled = int(round((2 ** 64 - 1) / max_hash)) if max_hash else 0
    with zipfile.ZipFile(zip_path, "w", zipfile.ZIP_STORED) as z:
        buf = io.StringIO()
        buf.write("# SOURMASH-MANIFEST-VERSION: 1.0\n")
        w = csv.writer(buf, lineterminator="\n")
        w.writerow(MANIFEST_COLUMNS)
        for sk in sketches:
            k = sk.get("ksize", ksize)
            text = signature_json(sk["name"], sk["mins"], k, sk.get("abundances"), max_hash,
                                  sk.get("filename", ""))
            md5 = compute_md5sum(k, [int(x) for x in sk["mins"]])
            loc = f"signatures/{md5}.sig.gz"
            z.writestr(loc, gzip.compress(text.encode(), compresslevel=1))
            w.writerow([loc, md5, md5[:8], k, "DNA", 0, scaled, len(sk["mins"]),
                        1 if sk.get("abundances") is not None else 0, sk["name"], sk.get("filename", "")])
        z.writestr(MANIFEST_NAME, buf.getvalue())
