"""Host-side mirror of the reference's helpers on the train hot path (reference src/yacht/utils.py).

Same names, argument meaning and error behaviour as the reference functions they mirror:

* :func:`load_signature_with_ksize`   utils.py:31-51   (sourmash-free, see sigio.py)
* :func:`get_num_kmers`               utils.py:54-75
* :func:`get_info_from_single_sig`    utils.py:89-110
* :func:`collect_signature_info`      utils.py:201-221
* :func:`run_yacht_train_core`        utils.py:112-197  -- launches ``<package dir>/run_yacht_train_core``,
  which here is the B200 executable built from csrc/train_core.cpp (same CLI, same files).
* :func:`decompress_all_sig_files`    utils.py:482-509
"""
from __future__ import annotations

import gzip
import zipfile
import os
import shutil
import sys
from glob import glob
from multiprocessing import Pool
from typing import Collection, Dict, List, Optional, Tuple

import numpy as np
import pandas as pd

from . import sigio
from .sigio import load_signature_with_ksize  # noqa: F401  (re-exported, reference name)

FILE_LOCATION = os.path.dirname(os.path.realpath(__file__))
__version__ = "1.4.0-b200"
COL_NOT_FOUND_ERROR = "Column not found: {}"


def _log(level: str, msg: str) -> None:
    import datetime
    print(f"{datetime.datetime.now():%Y-%m-%d %H:%M:%S} - {level} - {msg}", flush=True)


def get_num_kmers(minhash_mean_abundance: Optional[float], minhash_hashes_len: int, minhash_scaled: int,
                  scale: bool = True) -> int:
    """utils.py:54-75: estimated number of k-mers (mean abundance x hashes [x scaled])."""
    if minhash_mean_abundance:
        num_kmers = minhash_mean_abundance * minhash_hashes_len
    else:
        num_kmers = minhash_hashes_len
    if scale:
        num_kmers *= minhash_scaled
    return int(np.round(num_kmers))


def check_file_existence(file_path: str, error_description: str) -> None:
    if not os.path.exists(file_path):
        raise ValueError(error_description)


def get_info_from_single_sig(sig_file: str, ksize: int):
    """utils.py:89-110: (path, name, md5sum, mean abundance, number of hashes, scaled) or None."""
    info = sigio.sig_info(sig_file, ksize)
    if info is None:
        _log("WARNING", f"CANNOT extract the relevant info from the signature file: {sig_file}")
    return info


def collect_signature_info(num_threads: int, ksize: int, path_to_temp_dir: str) -> Dict[str, Tuple[str, float, int, int, str]]:
    """utils.py:201-221: {name: (md5sum, mean abundance, n hashes, scaled, path)} over signatures/."""
    files = [os.path.join(path_to_temp_dir, "signatures", f) for f in os.listdir(os.path.join(path_to_temp_dir, "signatures"))]
    if num_threads > 1 and len(files) > 64:
        with Pool(num_threads) as p:
            signatures = p.starmap(get_info_from_single_sig, [(f, ksize) for f in files], chunksize=64)
    else:
        signatures = [get_info_from_single_sig(f, ksize) for f in files]
    return {sig[1]: (sig[2], sig[3], sig[4], sig[5], sig[0]) for sig in signatures if sig}


# ---- `yacht train` ingest in one pass ----------------------------------------------------------------------------
# The reference unzips the database (make_training_data_from_sketches.py:109-111), gunzips every member in a pool
# (:115, utils.py:482-509) and then loads every file again through sourmash to collect its info (:119,
# utils.py:201-221): three passes over ~85k files.  Here each worker takes a slice of the zip members and does
# all of it while the bytes are in memory: read member -> gunzip -> write signatures/<name>.sig -> info tuple.
# The directory ends up exactly as the reference leaves it.
_zip_handle = None


def _extract_chunk(args):
    zip_path, members, dest, ksize = args
    global _zip_handle
    if _zip_handle is None or _zip_handle[0] != zip_path:
        _zip_handle = (zip_path, zipfile.ZipFile(zip_path, "r"))
    z = _zip_handle[1]
    out = []
    for m in members:
        raw = z.read(m)
        target = os.path.join(dest, m)
        if m.endswith(".sig.gz"):
            target = target[:-3]                                  # the reference gunzips in place and drops the .gz
            if raw[:2] == b"\x1f\x8b":
                raw = gzip.decompress(raw)
        with open(target, "wb") as f:
            f.write(raw)
        try:
            sigs = sigio.parse_signature_json(raw.decode(), target)
        except Exception:                                         # not text, not JSON, not a signature document
            sigs = None
        info = sigio.sig_info_from_signatures(sigs, target, ksize) if sigs is not None else None
        other_size = bool(sigs) and all(sig.ksize != ksize for sig in sigs)
        out.append((target, info, other_size))
    return out


def extract_signatures_and_info(ref_zip: str, path_to_temp_dir: str, ksize: int, num_threads: int) -> Dict[str, Tuple[str, float, int, int, str]]:
    """Unzip + gunzip + collect_signature_info in one parallel pass; returns what collect_signature_info returns."""
    return extract_signatures(ref_zip, path_to_temp_dir, ksize, num_threads)[0]


def extract_signatures(ref_zip: str, path_to_temp_dir: str, ksize: int, num_threads: int):
    """:func:`extract_signatures_and_info`, and the names (under signatures/) of the extracted files that are signatures
    of other k-mer sizes only: they parse, hold at least one sketch and none of size `ksize`.  A zip sketched at several
    sizes holds one such file per genome and extra size; :func:`run_yacht_train_core` leaves them out of the train core's
    file list, which would otherwise compare them too."""
    with zipfile.ZipFile(ref_zip, "r") as z:
        names = z.namelist()
        sig_members = [n for n in names if n.startswith("signatures/") and not n.endswith("/") and "/" not in n[len("signatures/"):]]
        taken = set(sig_members)
        for n in names:                                           # manifest and anything else: plain extraction
            if n not in taken:
                z.extract(n, path_to_temp_dir)
    os.makedirs(os.path.join(path_to_temp_dir, "signatures"), exist_ok=True)
    _log("INFO", f"Decompressing {sum(1 for n in sig_members if n.endswith('.sig.gz'))} .sig.gz files using {num_threads} threads.")
    _log("INFO", "Extracting signature information")
    nproc = max(1, int(num_threads))
    chunk = max(1, min(256, (len(sig_members) + 4 * nproc - 1) // (4 * nproc)))
    jobs = [(ref_zip, sig_members[a:a + chunk], path_to_temp_dir, ksize) for a in range(0, len(sig_members), chunk)]
    if nproc > 1 and len(sig_members) > 64:
        with Pool(nproc) as p:
            parts = p.map(_extract_chunk, jobs)
    else:
        parts = [_extract_chunk(j) for j in jobs]
    info = {}
    other_size = set()
    for part in parts:
        for target, sig, other in part:
            if sig:
                info[sig[1]] = (sig[2], sig[3], sig[4], sig[5], sig[0])
            elif other:
                other_size.add(os.path.basename(target))
            else:
                _log("WARNING", f"CANNOT extract the relevant info from the signature file: {target}")
    if other_size:
        _log("INFO", f"Leaving out {len(other_size)} signature files without a k-mer size {ksize} sketch (other k-mer sizes)")
    return info, other_size


def _gunzip_one(path: str) -> str:
    out = os.path.splitext(path)[0]
    with gzip.open(path, "rb") as f_in, open(out, "wb") as f_out:
        shutil.copyfileobj(f_in, f_out)
    os.remove(path)
    return out


def decompress_all_sig_files(sig_files: List[str], num_threads: int) -> None:
    """utils.py:499-509: gunzip every .sig.gz in place (the .gz is removed)."""
    if not sig_files:
        return
    if num_threads > 1 and len(sig_files) > 16:
        with Pool(num_threads) as p:
            p.map(_gunzip_one, sig_files, chunksize=16)
    else:
        for f in sig_files:
            _gunzip_one(f)


def run_yacht_train_core(num_threads: int, ani_thresh: float, ksize: int, path_to_temp_dir: str,
                         sig_info_dict: Dict[str, Tuple[str, float, int, int, str]],
                         num_genome_threshold: int = 1000000, other_size_files: Collection[str] = ()) -> pd.DataFrame:
    """utils.py:112-197, verbatim semantics: write the file list, convert ANI to containment, launch
    the core executable, move the pair files, keep the manifest rows of the selected genomes.
    `other_size_files` (names under signatures/, from :func:`extract_signatures`) stay out of the file list: the
    signatures of other k-mer sizes of a multi-size zip, which the reference lists too and then fails on."""
    sig_files = pd.DataFrame(
        [os.path.join(path_to_temp_dir, "signatures", file) for file in os.listdir(os.path.join(path_to_temp_dir, "signatures"))
         if file not in other_size_files]
    )
    sig_files_path = os.path.join(path_to_temp_dir, "training_sig_files.tsv")
    sig_files.to_csv(sig_files_path, header=False, index=False)

    containment_thresh = ani_thresh ** ksize
    total_sig_files = len(sig_files)
    # the GPU core indexes hash slots with 32 bits (include/yacht_gpu.h): say so here, before anything is launched
    total_hashes = sum(int(v[2]) for v in sig_info_dict.values())
    if total_hashes >= 2 ** 32:
        raise ValueError(f"The reference database holds {total_hashes} hashes; this build of run_yacht_train_core supports fewer than 2^32 "
                         f"(about 850 000 genomes at scaled=1000). Split the database or raise --scaled.")
    if total_sig_files <= num_genome_threshold:
        passes = 1
    else:
        passes = int(total_sig_files / num_genome_threshold) + 1
    cmd = (f"{FILE_LOCATION}/run_yacht_train_core -t {num_threads} -c {containment_thresh} -p {passes} "
           f"{sig_files_path} {path_to_temp_dir} {os.path.join(path_to_temp_dir, 'selected_result.tsv')}")
    _log("INFO", f"Running comparison algorithm with command: {cmd}")
    exit_code = os.system(cmd)
    if exit_code != 0:
        raise ValueError(f"Error running comparison algorithm with command: {cmd}")

    os.makedirs(os.path.join(path_to_temp_dir, "comparison_files"), exist_ok=True)
    for file in glob(os.path.join(path_to_temp_dir, "*.txt")):
        shutil.move(file, os.path.join(path_to_temp_dir, "comparison_files"))

    selected_sig_files = pd.read_csv(os.path.join(path_to_temp_dir, "selected_result.tsv"), sep="\t", header=None)
    selected_sig_files = selected_sig_files[0].to_list()
    mapping = {sig_info_dict[name][-1]: name for name in sig_info_dict}
    selected_genome_names_set = set([mapping[sig_file_path] for sig_file_path in selected_sig_files])

    manifest_df = []
    for sig_name, (md5sum, minhash_mean_abundance, minhash_hashes_len, minhash_scaled, _) in sig_info_dict.items():
        if sig_name in selected_genome_names_set:
            manifest_df.append((sig_name, md5sum, minhash_hashes_len,
                                get_num_kmers(minhash_mean_abundance, minhash_hashes_len, minhash_scaled, False),
                                minhash_scaled))
    return pd.DataFrame(manifest_df, columns=["organism_name", "md5sum", "num_unique_kmers_in_genome_sketch",
                                              "num_total_kmers_in_genome_sketch", "genome_scale_factor"])
