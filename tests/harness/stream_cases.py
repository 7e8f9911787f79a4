"""FASTA / FASTQ inputs for the streamed parse (tests/test_sketch_stream.py on the CPU, tests/test_sketch_stream_gpu.py on the
device): the record path (sketch.read_records) is the reference for every one of them."""
import numpy as np


def _seq(rng, n, alphabet=b"ACGT"):
    return rng.choice(np.frombuffer(alphabet, dtype=np.uint8), size=n).tobytes()


def _wrap(seq, width):
    return b"".join(seq[i:i + width] + b"\n" for i in range(0, len(seq), width)) if seq else b""


def accepted_cases():
    """name -> file bytes that read_records accepts."""
    rng = np.random.default_rng(11)
    c = {}
    recs = [(f"contig_{i} desc".encode(), _seq(rng, int(rng.integers(50, 900)))) for i in range(8)]
    c["fasta_wrapped"] = b"".join(b">" + n + b"\n" + _wrap(s, 60) for n, s in recs)
    c["fasta_one_long_line"] = b">chr\n" + _seq(rng, 9000) + b"\n>chr2\n" + _seq(rng, 5000) + b"\n"
    c["fasta_crlf"] = c["fasta_wrapped"].replace(b"\n", b"\r\n")
    c["fasta_stray_cr"] = b">a\nACGTACGTAC\rGTACGTACGTACGTACGTACGTACGTACGTAC\rGT\n>b\r\n\rACGTACGTACGTACGTACGTACGTACGTACGTACGTAAA\n"
    c["fasta_spaces_and_junk"] = b">a\nACGTACGTACGTACGTACGTAC  \nGTACGTACGTACGTACGTACGTACGTACG*TACGTACGT.ACGTACGTACGTAC\tGGG\n"
    c["fasta_blank_lines"] = b">a\n\nACGTACGTACGTACGTACGTACGTACGT\n\n\nACGTACGTACGTACGTACGTACGTACGTACGT\n\n>b\n\n" + _wrap(_seq(rng, 300), 70) + b"\n\n"
    c["fasta_case_n_iupac"] = b">a\n" + _wrap(_seq(rng, 2000, b"ACGTacgtNnRYKMSWBDHV"), 61) + b">b\n" + _wrap(_seq(rng, 700, b"acgt"), 50)
    c["fasta_no_final_newline"] = b">a\n" + _seq(rng, 200) + b"\n>b\n" + _seq(rng, 333)
    c["fasta_empty_header_and_body"] = b">\n" + _seq(rng, 120) + b"\n>empty\n>\n>x\n" + _seq(rng, 80) + b"\n>last empty"
    c["fasta_headers_gt_and_acgt"] = (b">x>y " + b"ACGT" * 30 + b"\n" + _seq(rng, 150) + b"\n>>>\n" + _seq(rng, 90)
                                      + b"\n> " + b"ACGTACGT" * 20 + b"\n" + _seq(rng, 64) + b"\n")
    c["fasta_short_records"] = b"".join(b">s%d\n" % i + _seq(rng, i) + b"\n" for i in range(0, 70, 3))
    c["fasta_leading_whitespace"] = b"\n\r\n  \t\x0b\x0c>a\n" + _seq(rng, 400) + b"\n"
    c["fasta_cr_before_gt"] = b">a\n" + _seq(rng, 100) + b"\n\r>b\n" + _seq(rng, 100) + b"\n\r\r\n" + _seq(rng, 40) + b"\n"
    reads = [(f"r{i}/1 x".encode(), _seq(rng, int(rng.integers(0, 160)), b"ACGT" * 10 + b"N")) for i in range(40)]
    c["fastq_plain"] = b"".join(b"@" + n + b"\n" + s + b"\n+\n" + b"I" * len(s) + b"\n" for n, s in reads)
    c["fastq_crlf_no_final_newline"] = c["fastq_plain"].replace(b"\n", b"\r\n")[:-2]
    quals = [b"@" + b"I" * 30, b"", b"+" + b"I" * 30, b"ACGT" * 8, b"@@@@", b"++"]
    c["fastq_tricky_quality"] = b"".join(b"@q%d\n" % i + _seq(rng, len(q)) + b"\n+q%d repeated\n" % i + q + b"\n"
                                         for i, q in enumerate(quals))
    c["fastq_blank_seq_and_trailing_blank_lines"] = b"@a\n\n+\n\n@b\n" + _seq(rng, 90) + b"\n+\n" + b"I" * 90 + b"\n\n\r\n\n"
    c["fastq_leading_whitespace"] = b"  \n\t@a\n" + _seq(rng, 50) + b"\n+\n" + b"I" * 50 + b"\n"
    c["fastq_stray_cr"] = b"@a\nACGTACGTACGTACGTACGT\rACGTACGTACGTACGTACGTACGTACGT\n+\n" + b"I" * 48 + b"\n"
    c["empty"] = b""
    c["only_whitespace"] = b" \n\r\n\t"
    return c


def rejected_cases():
    """name -> file bytes that read_records rejects (it raises ValueError)."""
    rng = np.random.default_rng(12)
    s = _seq(rng, 40)
    good = b"@r\n" + s + b"\n+\n" + b"I" * 40 + b"\n"
    return {
        "neither": b"  \nACGT\n",
        "neither_plus": b"+x\n",
        "fastq_5_lines": good + b"@x\n",
        "fastq_bad_plus": good + b"@r2\nACGT\nX\nIIII\n",
        "fastq_bad_at": good + b"r3\nACGT\n+\nIIII\n" + good,
        "fastq_empty_line_mid": good + b"\n\n\n\n" + good,
        "fastq_empty_plus_mid": b"@r\nACGT\n\nIIII\n" + good,
        "fastq_gt_header": good + b">r\nACGT\n+\nIIII\n",
        "fastq_cr_only_line": good + b"\r\nA\n+\nI\n" + good,
    }
