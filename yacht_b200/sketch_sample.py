#!/usr/bin/env python
"""``yacht sketch sample`` on the GPU.

Same command line as the reference's wrapper (src/yacht/sketch_sample.py): one or two FASTA/FASTQ files in, ONE sketch with
abundances out.  For paired-end input the reference first concatenates both files into a temporary file (:42-57); here the
records of both files simply go into the same sketch.  ``--kmer`` may also name several k-mer sizes (``--kmer 21 31 51``):
the input is then read once and the output holds one signature per size, in the order given, each what a run with that
size alone writes (``sourmash sketch dna -p k=21,k=31,k=51,...`` makes such files too).
"""
import argparse

from . import sketch
from .utils import _log


def add_arguments(parser):
    sketch.add_cli_arguments(parser, infile_help="Input FASTA/Q file(s). For paired-end reads, provide two files.", nargs="+",
                             multi_kmer=True)


def sketch_reads(infiles, kmer, scaled, outfile):
    """All records of `infiles` -> one sketch (name empty, filename = the first file, like `sourmash sketch dna`).
    When one of the files is larger than sketch.STREAM_FILE_BYTES, all of them are streamed through the device parser,
    file after file, into the one sketch; otherwise the records are read whole and batched."""
    if any(sketch.is_streamed(path) for path in infiles):
        [(mins, abundances)], _ = sketch.sketch_stream(list(infiles), kmer, scaled)
    else:
        reads = [seq for path in infiles for _, seq in sketch.read_records(path)]
        [(mins, abundances)] = sketch.sketch_record_groups([reads], kmer, scaled)
    sketch.write_sketches(outfile, [dict(name="", filename=infiles[0], mins=mins, abundances=abundances)], kmer, scaled)


def sketch_reads_multik(infiles, kmers, scaled, outfile):
    """`sketch_reads` at several k-mer sizes: the files are streamed through the device parser once, every size is hashed
    on the same parsed text, and `outfile` holds one signature per size, in the order of `kmers`."""
    per_k, _ = sketch.sketch_stream(list(infiles), list(kmers), scaled)
    sketches = [dict(name="", filename=infiles[0], mins=mins, abundances=abundances, ksize=k) for k, [(mins, abundances)] in zip(kmers, per_k)]
    sketch.write_sketches(outfile, sketches, kmers[0], scaled)


def main(args):
    files = list(args.infile)
    if len(files) not in (1, 2):
        raise ValueError("Please provide either one file for single-end reads or two files for paired-end reads.")
    kmers = sketch.kmer_sizes(args.kmer)
    kind = "a single-end FASTA/Q file" if len(files) == 1 else "paired-end FASTA/Q files"
    _log("INFO", f"Starting sketching {kind}: {' '.join(files)}")
    if len(kmers) == 1:
        sketch_reads(files, kmers[0], args.scaled, args.outfile)
    else:
        sketch_reads_multik(files, kmers, args.scaled, args.outfile)
    _log("SUCCESS", "Successfully sketched!!")


if __name__ == "__main__":
    cli = argparse.ArgumentParser(description="Sketch single-end or paired-end reads on the GPU.",
                                  formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    add_arguments(cli)
    main(cli.parse_args())
