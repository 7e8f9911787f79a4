#!/usr/bin/env python
"""``yacht sketch ref`` on the GPU.

Same command line and output kinds as the reference's wrapper (src/yacht/sketch_ref_genomes.py), which builds a
``sourmash sketch`` command line instead:
  * ``--infile`` names a file   -> every sequence record becomes its own sketch (the reference passes ``--singleton``, :25);
  * ``--infile`` names a folder -> every sequence file below it becomes one sketch, named after the file without its
    extension; like the reference (:31-67) a ``dataset.csv`` listing (name, path) is left in the folder.
Sketches are DNA FracMinHash with abundances; ``--outfile`` ending in ``.zip`` gives a sourmash zip database.
``--kmer`` may also name several k-mer sizes, comma-separated (``--kmer 21,31,51``): every file is then read once and the
output holds one signature per (genome or record, size), sizes in the order given, each what a run with that size alone
writes.
``yacht train --ksize K`` trains on the size-K signatures of such a zip.
"""
import argparse
import os
from pathlib import Path

from . import sketch
from .utils import _log

# sequence file suffixes the reference globs for, in its order (:32-41)
SEQUENCE_SUFFIXES = (".fasta", ".fna", ".fas", ".fa", ".fasta.gz", ".fna.gz", ".fas.gz", ".fa.gz")


def add_arguments(parser):
    sketch.add_cli_arguments(parser, infile_help="Input file or folder path.")


def sequence_files_below(folder):
    """[(sketch name, absolute path)]: suffix by suffix, recursive, as the reference enumerates them."""
    found = []
    for suffix in SEQUENCE_SUFFIXES:
        found.extend((p.name.replace(suffix, ""), str(p.absolute())) for p in Path(folder).glob(f"**/*{suffix}"))
    return found


def _k_text(kmer):
    return ",".join(map(str, kmer)) if isinstance(kmer, list) else str(kmer)


def sketch_folder(folder, kmer, scaled, outfile):
    """kmer: one size (int) or several (list): one signature per file and size."""
    listing = sequence_files_below(folder)
    with open(os.path.join(folder, "dataset.csv"), "w") as out:
        out.write("name,genome_filename,protein_filename\n")
        out.writelines(f"{name},{path},\n" for name, path in listing)
    _log("INFO", f"Sketching {len(listing)} sequence files below {folder} (k={_k_text(kmer)}, scaled={scaled})")
    sketches = sketch.sketch_files([path for _, path in listing], kmer, scaled, names=[name for name, _ in listing])
    sketch.write_sketches(outfile, sketches, kmer[0] if isinstance(kmer, list) else kmer, scaled)
    _log("SUCCESS", f"Successfully sketched files in: {folder}")


def sketch_records_of(infile, kmer, scaled, outfile):
    """kmer: one size (int) or several (list): one signature per record and size."""
    _log("INFO", f"Sketching every record of {infile} (k={_k_text(kmer)}, scaled={scaled})")
    sketch.write_sketches(outfile, sketch.sketch_files([infile], kmer, scaled, singleton=True), kmer[0] if isinstance(kmer, list) else kmer, scaled)
    _log("SUCCESS", "Successfully sketched!!")


def main(args):
    target = args.infile
    kmers = sketch.kmer_sizes(args.kmer)
    kmer = kmers[0] if len(kmers) == 1 else kmers        # one size: the single-size path, unchanged
    if os.path.isdir(target):
        sketch_folder(target, kmer, args.scaled, args.outfile)
    elif os.path.isfile(target):
        sketch_records_of(target, kmer, args.scaled, args.outfile)
    else:
        _log("ERROR", f"Input path {target} does not exist.")      # the reference logs this and returns (:70-80)


if __name__ == "__main__":
    cli = argparse.ArgumentParser(description="Sketch genomes on the GPU.", formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    add_arguments(cli)
    main(cli.parse_args())
