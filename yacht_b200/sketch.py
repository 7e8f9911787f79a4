"""FracMinHash sketching of sequence files on the GPU (SURVEY 8 row f-4).

Host side of what the reference delegates to ``sourmash sketch dna -p k=K,scaled=S,abund`` (sketch_ref_genomes.py:25,61;
sketch_sample.py:32,49): read FASTA / FASTQ (plain or gzip), hand the bases to ``ygpu_sketch_sequences`` (k-mer hashing,
ordering and de-duplication run on the device), write sourmash-style ``.sig.zip`` / ``.sig`` files (yacht_b200/sigio.py).
There is no CPU hashing path: without the library and a GPU these functions raise.
"""
from __future__ import annotations

import argparse
import gzip
import os
import queue
import threading
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib, sigio

SEED = 42                       # "seed": 42 in every sourmash DNA signature
BATCH_BASES = 1 << 31           # bases per device call (2 GiB of sequence + separators)
CHUNK_FILE_BYTES = 1 << 29      # on-disk bytes of sequence files read ahead of the device (gzip expands ~3.5x)
STREAM_FILE_BYTES = 1 << 30     # a file larger than this on disk is streamed: its text is parsed on the device chunk by chunk
STREAM_READ_BYTES = 64 << 20    # bytes per read into one page-locked buffer (one device chunk at the library's default)
STREAM_BUFFERS = 3              # page-locked read buffers: the reader fills one while the device works on another
_ctx = None


def _context() -> _lib.GpuContext:
    global _ctx
    if _ctx is None:
        _ctx = _lib.GpuContext(int(os.environ.get("YACHT_DEVICE", "0")))
    return _ctx


def kmer_list(text: str):
    """Type of `sketch ref --kmer`: one k-mer size ("31" -> 31) or a comma-separated list of them ("21,31,51" ->
    [21, 31, 51]).  The option takes one command-line word, so `--kmer 21 31` stays an unrecognized argument."""
    try:
        sizes = [int(part) for part in text.split(",")]
    except ValueError:
        raise argparse.ArgumentTypeError(f"expected a k-mer size or a comma-separated list of sizes (21,31,51), got {text!r}")
    return sizes[0] if len(sizes) == 1 else sizes


def add_cli_arguments(parser, infile_help: str, nargs=None, multi_kmer: bool = False) -> None:
    """The four options both `yacht sketch` sub-commands take (names and defaults of the reference's wrappers).
    With `multi_kmer`, --kmer takes one or more values and is always a list (default [31]); without it, --kmer is one
    word, a size or a comma-separated list of sizes (`kmer_list`)."""
    kw = {"nargs": nargs} if nargs else {}
    parser.add_argument("--infile", help=infile_help, required=True, **kw)
    if multi_kmer:
        parser.add_argument("--kmer", type=int, nargs="+", default=[31],
                            help="K-mer size(s). Several distinct sizes are sketched in one pass into one output file.")
    else:
        parser.add_argument("--kmer", type=kmer_list, default=31,
                            help="K-mer size, or several comma-separated (21,31,51): every file is read once and sketched at "
                                 "each size into one output file.")
    parser.add_argument("--scaled", type=int, default=1000, help="Scaled factor.")
    parser.add_argument("--outfile", help="Output file name.", required=True)


def max_hash_for_scaled(scaled: int) -> int:
    """sourmash's rule: round((2^64 - 1) / scaled) in double arithmetic (18446744073709552 at scaled = 1000)."""
    if scaled == 0:
        return 0
    if scaled == 1:
        return 2 ** 64 - 1
    return min(int(round((2 ** 64 - 1) / scaled, 0)), 2 ** 64 - 1)


def read_records(path: str) -> List[Tuple[str, bytes]]:
    """[(name, sequence bytes)] of a FASTA or FASTQ file, gzip or plain (whole-buffer splitting, no per-line Python loop
    for the sequence data)."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] == b"\x1f\x8b":
        data = gzip.decompress(data)
    data = data.replace(b"\r", b"")
    stripped = data.lstrip()
    if not stripped:
        return []
    records: List[Tuple[str, bytes]] = []
    if stripped[:1] == b">":
        for chunk in (b"\n" + stripped).split(b"\n>")[1:]:
            head, _, body = chunk.partition(b"\n")
            records.append((head.decode(), body.replace(b"\n", b"")))
    elif stripped[:1] == b"@":
        lines = stripped.split(b"\n")
        while lines and not lines[-1]:
            lines.pop()
        if len(lines) % 4:
            raise ValueError(f"{path}: FASTQ with {len(lines)} lines (not a multiple of 4)")
        for i in range(0, len(lines), 4):
            if not lines[i].startswith(b"@") or not lines[i + 2].startswith(b"+"):
                raise ValueError(f"{path}: malformed FASTQ record at line {i + 1}")
            records.append((lines[i][1:].decode(), lines[i + 1]))
    else:
        raise ValueError(f"{path}: neither FASTA ('>') nor FASTQ ('@')")
    return records


def is_streamed(path: str) -> bool:
    """Whether `path` takes the streamed route (decided by its size on disk only)."""
    return os.path.getsize(path) > STREAM_FILE_BYTES


def _open_text(path: str):
    """The file's decompressed bytes as a stream: gzip (every member) when it starts with the gzip magic, else plain."""
    f = open(path, "rb")
    if f.read(2) == b"\x1f\x8b":
        f.seek(0)
        return gzip.GzipFile(fileobj=f, mode="rb"), f
    f.seek(0)
    return f, f


def _reader(path: str, bufs, free: "queue.Queue", full: "queue.Queue") -> None:
    """Reader thread: fills free buffers with the file's next bytes, hands them over as (index, n); (None, 0) at the end,
    (None, exception) on a read error.  A None taken from `free` asks it to stop."""
    try:
        text, raw = _open_text(path)
        try:
            while True:
                i = free.get()
                if i is None:
                    return
                n = text.readinto(bufs[i][0])
                if not n:
                    full.put((None, 0))
                    return
                full.put((i, n))
        finally:
            text.close()
            raw.close()
    except BaseException as e:          # handed to the feeding thread, which raises it
        full.put((None, e))


def sketch_stream(paths: Sequence[str], ksize, scaled: int, per_record: bool = False, seed: int = SEED,
                  stats: Optional[dict] = None):
    """Sketch the files one after another through the device stream (ygpu_stream_*): the text is read and gunzipped on a
    reader thread into STREAM_BUFFERS page-locked buffers and parsed, hashed and accumulated on the device, so host memory
    stays at a few buffers plus the sketch whatever the size of the input.
    Returns ([(mins, abundances)], names): one sketch of all records, or with `per_record` one per record with its name.
    With a sequence of k-mer sizes for `ksize` the input is still read and parsed once, and the result is
    ([[(mins, abundances)] per k, in the order given], names).
    `stats`, when given, receives the stream's counters and device times (ygpu_stream_stats)."""
    ctx = _context()
    ctx.stream_begin(ksize, max_hash_for_scaled(scaled), seed, per_record)
    bufs = [ctx.host_buffer(STREAM_READ_BYTES) for _ in range(STREAM_BUFFERS)]
    try:
        for path in paths:
            free: queue.Queue = queue.Queue()
            full: queue.Queue = queue.Queue()
            for i in range(len(bufs)):
                free.put(i)
            th = threading.Thread(target=_reader, args=(path, bufs, free, full), daemon=True)
            th.start()
            try:
                while True:
                    i, n = full.get()
                    if i is None:
                        if isinstance(n, BaseException):
                            raise n
                        break
                    ctx.stream_feed(bufs[i][1], n, path)
                    free.put(i)
            finally:
                free.put(None)
                th.join()
            ctx.stream_end_file(path)
        if isinstance(ksize, (int, np.integer)):
            hashes, abund, offsets, names, st = ctx.stream_finish(paths[-1] if paths else None)
            per_k = None
        else:
            per_k, names, st = ctx.stream_finish(paths[-1] if paths else None)
        if stats is not None:
            stats.update(st)
    finally:
        for _, _, release in bufs:
            release()
    # names come back as bytes; decoding them raises on invalid UTF-8 as the record path's reader does
    names = [b.decode() for b in names] if names else []
    split = lambda hashes, abund, offsets: [(hashes[int(offsets[s]):int(offsets[s + 1])], abund[int(offsets[s]):int(offsets[s + 1])])
                                            for s in range(len(offsets) - 1)]
    if per_k is None:
        return split(hashes, abund, offsets), names
    return [split(h, a, o) for h, a, o, _ in per_k], names


def kmer_sizes(kmer) -> List[int]:
    """--kmer as a list (the command line gives one; a caller that builds the namespace itself may pass one int).
    Refuses a size given twice."""
    kmers = [int(k) for k in kmer] if isinstance(kmer, (list, tuple)) else [int(kmer)]
    dup = sorted({k for k in kmers if kmers.count(k) > 1})
    if dup:
        raise ValueError(f"--kmer: k-mer size(s) {', '.join(map(str, dup))} given more than once.")
    return kmers


def sketch_record_groups(groups: Sequence[Sequence[bytes]], ksize, scaled: int, seed: int = SEED):
    """One sketch per group of records.  Returns [(mins uint64 ascending, abundances uint32)] in group order.
    Groups are packed into device calls of at most BATCH_BASES bytes; a group larger than that is split over calls and its
    partial sketches are merged (hashes united, abundances added).
    With a sequence of k-mer sizes for `ksize` every batch is joined and uploaded once and hashed at each size
    (ygpu_sketch_sequences_k); the result is then [[(mins, abundances)] per group] per k, in the order given."""
    ctx = _context()
    max_hash = max_hash_for_scaled(scaled)
    multi = not isinstance(ksize, (int, np.integer))
    ks = list(ksize) if multi else [ksize]
    out: List[List[Optional[Tuple[np.ndarray, np.ndarray]]]] = [[None] * len(groups) for _ in ks]

    def merge(ki, gi, mins, ab):
        if out[ki][gi] is None:
            out[ki][gi] = (mins, ab)
            return
        m0, a0 = out[ki][gi]
        allm = np.concatenate([m0, mins])
        alla = np.concatenate([a0, ab]).astype(np.uint64)
        um, inv = np.unique(allm, return_inverse=True)
        ua = np.zeros(um.shape[0], dtype=np.uint64)
        np.add.at(ua, inv, alla)
        out[ki][gi] = (um, ua.astype(np.uint32))

    batch_parts: List[bytes] = []
    batch_ids: List[int] = []          # group id of every sketch range of the batch
    batch_offs: List[int] = [0]
    size = 0

    def flush():
        nonlocal batch_parts, batch_ids, batch_offs, size
        if not batch_ids:
            return
        bases = b"".join(batch_parts)
        if multi:
            per_k = ctx.sketch_sequences_k(bases, batch_offs, ks, max_hash, seed)
        else:
            per_k = [ctx.sketch_sequences(bases, batch_offs, ksize, max_hash, seed)]
        for ki, (hashes, abund, offs, _) in enumerate(per_k):
            for j, gi in enumerate(batch_ids):
                lo, hi = int(offs[j]), int(offs[j + 1])
                merge(ki, gi, hashes[lo:hi], abund[lo:hi])
        batch_parts, batch_ids, batch_offs, size = [], [], [0], 0

    for gi, recs in enumerate(groups):
        cur: List[bytes] = []
        cur_len = 0
        for seq in recs:
            if cur_len + len(seq) + 1 > BATCH_BASES - size and (cur or batch_ids):
                if cur:                                   # close the part of this group gathered so far
                    batch_parts.extend(cur)
                    batch_ids.append(gi)
                    batch_offs.append(batch_offs[-1] + cur_len)
                    cur, cur_len = [], 0
                flush()
            cur.append(seq)
            cur.append(b"\n")                             # separator: breaks every window that would span two records
            cur_len += len(seq) + 1
        batch_parts.extend(cur)
        batch_ids.append(gi)
        batch_offs.append(batch_offs[-1] + cur_len)
        size = batch_offs[-1]
    flush()
    empty = (np.zeros(0, np.uint64), np.zeros(0, np.uint32))
    per_k = [[o if o is not None else empty for o in out_k] for out_k in out]
    return per_k if multi else per_k[0]


def sketch_files(paths: Sequence[str], ksize, scaled: int, singleton: bool = False, names: Optional[Sequence[str]] = None,
                 threads: Optional[int] = None):
    """Sketch dicts ({name, filename, mins, abundances}) ready for sigio.write_sig_zip: one per file (all records together,
    like ``sourmash sketch fromfile`` / ``sketch dna``) or, with ``singleton``, one per record (``--singleton``).
    Files are taken in chunks of ~CHUNK_FILE_BYTES on disk so that a large collection never sits in host memory at once.
    With a sequence of k-mer sizes for `ksize` every file is read once and there is one dict per (file or record, size),
    file- or record-major and sizes in the order given, each with its own ``"ksize"``."""
    threads = max(1, int(threads or os.cpu_count() or 1))
    multi = not isinstance(ksize, (int, np.integer))
    out: List[dict] = []

    def emit(name, filename, per_k):
        """per_k: [(mins, abundances)] per size (one entry for a single size)."""
        if not multi:
            [(mins, ab)] = per_k
            out.append({"name": name, "filename": filename, "mins": mins, "abundances": ab})
            return
        out.extend({"name": name, "filename": filename, "mins": mins, "abundances": ab, "ksize": k}
                   for k, (mins, ab) in zip(ksize, per_k))

    i = 0
    while i < len(paths):
        if is_streamed(paths[i]):       # a large file: parsed on the device, never held in host memory
            sketches, rec_names = sketch_stream([paths[i]], ksize, scaled, per_record=singleton)
            per_k = sketches if multi else [sketches]     # [[(mins, ab)] per sketch] per size
            if singleton:
                for r, name in enumerate(rec_names):
                    emit(name, paths[i], [sk[r] for sk in per_k])
            else:
                emit(names[i] if names is not None else "", paths[i], [sk[0] for sk in per_k])
            i += 1
            continue
        j, size = i, 0
        while j < len(paths) and (j == i or (size + os.path.getsize(paths[j]) <= CHUNK_FILE_BYTES and not is_streamed(paths[j]))):
            size += os.path.getsize(paths[j])
            j += 1
        chunk = list(paths[i:j])
        # gunzip + splitting release the GIL for most of their time: read the chunk's files on host threads, in order
        if threads > 1 and len(chunk) > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(min(threads, len(chunk))) as pool:
                all_recs = list(pool.map(read_records, chunk))
        else:
            all_recs = [read_records(p) for p in chunk]
        groups: List[List[bytes]] = []
        meta: List[Tuple[str, str]] = []
        for k, (path, recs) in enumerate(zip(chunk, all_recs)):
            if singleton:
                for name, seq in recs:
                    groups.append([seq])
                    meta.append((name, path))
            else:
                groups.append([seq for _, seq in recs])
                meta.append((names[i + k] if names is not None else "", path))
        del all_recs
        sketches = sketch_record_groups(groups, ksize, scaled)
        per_k = sketches if multi else [sketches]
        for g, (name, filename) in enumerate(meta):
            emit(name, filename, [sk[g] for sk in per_k])
        i = j
    return out


def write_sketches(outfile: str, sketches: Sequence[dict], ksize: int, scaled: int) -> None:
    """``.zip`` -> a sourmash zip database (manifest + signatures/<md5>.sig.gz); anything else -> one JSON signature file.
    A sketch dict's own ``"ksize"`` takes the place of `ksize`."""
    max_hash = max_hash_for_scaled(scaled)
    if outfile.endswith(".zip"):
        sigio.write_sig_zip(outfile, sketches, ksize, max_hash)
    else:
        sigio.write_signatures(outfile, sketches, ksize, max_hash)
