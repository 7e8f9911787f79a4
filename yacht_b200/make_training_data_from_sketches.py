"""`yacht train` orchestration (mirror of reference src/yacht/make_training_data_from_sketches.py:20-155):
same arguments, same checks and messages, same outputs (<prefix>_intermediate_files/,
<prefix>_processed_manifest.tsv, <prefix>_config.json).  The comparison itself is
utils.run_yacht_train_core -> the B200 executable."""
from __future__ import annotations

import argparse
import glob
import json
import os
import shutil
import zipfile
from pathlib import Path

from . import utils
from .utils import _log


def add_arguments(parser):
    parser.add_argument("--ref_file", required=True,
                        help="Location of the Sourmash signature database file. This is expected to be in Zipfile format (eg. *.zip) "
                             'that contains a manifest "SOURMASH-MANIFEST.csv" and a folder "signatures" with all Gzip-format '
                             "signature file (eg. *.sig.gz).")
    parser.add_argument("--ksize", type=int, required=True, help="Size of kmers in sketch since Zipfiles can contain multiple k-sizes.")
    parser.add_argument("--num_threads", type=int, required=False, default=16, help="Number of threads to use for parallelization.")
    parser.add_argument("--ani_thresh", type=float, required=False, default=0.95,
                        help='mutation cutoff for species equivalence. Organisms with this ANI or greater between them are considered "equivalent".')
    parser.add_argument("--prefix", required=False, default="yacht", help="Prefix name to identify this experiment.")
    parser.add_argument("--outdir", type=str, required=False, default=os.getcwd(), help="Path to output directory.")
    parser.add_argument("--force", action="store_true", help="Overwrite the output directory if it exists.")


def main(args):
    ref_file = str(Path(args.ref_file).absolute())
    ksize, num_threads, ani_thresh, prefix = args.ksize, args.num_threads, args.ani_thresh, args.prefix
    outdir = str(Path(args.outdir).absolute())

    _log("INFO", "Checking reference database file")
    if os.path.splitext(ref_file)[1] != ".zip":
        raise ValueError(f"Reference database file {ref_file} is not a zip file. Please a Sourmash signature database file with Zipfile format.")
    utils.check_file_existence(ref_file, f"Reference database zip file {ref_file} does not exist.")

    _log("INFO", "Creating a temporary directory")
    path_to_temp_dir = os.path.join(outdir, prefix + "_intermediate_files")
    if os.path.exists(path_to_temp_dir) and not args.force:
        raise ValueError(f"Temporary directory {path_to_temp_dir} already exists. Please remove it, use '--force', "
                         f"or given a new prefix name using parameter '--prefix'.")
    if os.path.exists(path_to_temp_dir):
        _log("WARNING", f"Temporary directory {path_to_temp_dir} already exists. Removing it.")
        shutil.rmtree(path_to_temp_dir)
    os.makedirs(path_to_temp_dir, exist_ok=True)

    _log("INFO", "Unzipping the sourmash signature file to the temporary directory")
    # reference :109-119 (extractall, gunzip pool, collect_signature_info) as ONE parallel pass over the zip members
    # signatures of other k-mer sizes (a zip sketched at several sizes) are extracted too but stay out of the comparison
    sig_info_dict, other_size_files = utils.extract_signatures(ref_file, path_to_temp_dir, ksize, num_threads)
    _log("INFO", "Checking if all signatures have the same scaled")
    scale_set = set([value[-2] for value in sig_info_dict.values()])
    if len(scale_set) != 1:
        raise ValueError("Not all signatures have the same scaled. Please check your input.")
    scale = scale_set.pop()

    _log("INFO", "Finding the closely related genomes with ANI > ani_thresh from the reference database, then remove them, "
                 "and generate a dataframe with the selected genomes.")
    manifest_df = utils.run_yacht_train_core(num_threads, ani_thresh, ksize, path_to_temp_dir, sig_info_dict,
                                             other_size_files=other_size_files)

    _log("INFO", "Writing out the manifest file")
    manifest_file_path = os.path.join(outdir, f"{prefix}_processed_manifest.tsv")
    manifest_df.to_csv(manifest_file_path, sep="\t", index=None)

    _log("INFO", "Saving the config file")
    json_file_path = os.path.join(outdir, f"{prefix}_config.json")
    with open(json_file_path, "w") as f:
        json.dump({"manifest_file_path": manifest_file_path, "intermediate_files_dir": path_to_temp_dir, "scale": scale,
                   "ksize": ksize, "ani_thresh": ani_thresh}, f, indent=4)


if __name__ == "__main__":
    parser = argparse.ArgumentParser(description="This script converts a collection of signature files into a reference database matrix.",
                                     formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    add_arguments(parser)
    main(parser.parse_args())
