// Per-byte and per-line rules of the streamed FASTA / FASTQ parse (seq_stream.cu).  They restate what sketch.read_records does
// with whole-buffer operations -- drop every '\r', lstrip the text, split FASTA at "\n>", take FASTQ as groups of four lines --
// as decisions a thread can take about one byte, given its line's first byte and the line's number.
//
// A line's "first byte" is its first byte that is not '\r' (the record path removes '\r' before it looks at a line); a line
// made of '\r' only is empty.  Line numbers count from the first byte after the leading whitespace of the file, as the
// record path's lines of `data.lstrip()` do.
//
// __host__ __device__ like sketch_hash.cuh, so that tests/harness/seq_stream_host.cpp can walk the chunked parse on the CPU
// with exactly these rules.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define YSQ_HD __host__ __device__ __forceinline__
#else
#define YSQ_HD inline
#endif

enum { YSQ_FMT_NONE = 0, YSQ_FASTA = 1, YSQ_FASTQ = 2 };
enum { YSQ_ROLE_DROP = 0, YSQ_ROLE_SEQ = 1, YSQ_ROLE_HEADER = 2 };
// per-byte flags: the byte goes to the hashing buffer / starts a record (it is written as the '\n' separator) / is a name byte
enum { YSQ_F_SEQ = 1, YSQ_F_REC = 2, YSQ_F_NAME = 4 };
constexpr int YSQ_CARRY_MAX = 256;             // room for k - 1 bases at the largest k

// Carried from one chunk to the next (and from one file to the next): state, never partial lines.
struct ysq_state {
    uint64_t line;            // number of the open line (the one the next byte belongs to)
    uint64_t n_records;       // records started so far, all files of the stream
    uint64_t last_nonempty1;  // FASTQ: 1 + number of the last line that has a first byte (0: none)
    uint64_t first_bad;       // FASTQ: first line with a first byte that breaks the 4-line structure (~0: none)
    uint64_t first_bad_empty; // FASTQ: first empty line at a place where '@' or '+' is due (~0: none)
    uint32_t fmt;             // YSQ_FASTA / YSQ_FASTQ of the current file
    uint32_t open_first;      // first byte of the open line, 0 while it has none
    uint32_t n_carry;         // bases of the open record carried into the next chunk (<= k - 1)
    uint32_t _pad;
    uint8_t carry[YSQ_CARRY_MAX];
};

// bytes.lstrip()'s whitespace
YSQ_HD bool ysq_is_space(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == 0x0b || c == 0x0c; }
YSQ_HD int ysq_format_of(uint8_t first) { return first == '>' ? YSQ_FASTA : first == '@' ? YSQ_FASTQ : YSQ_FMT_NONE; }

// Byte c is its line's first byte.  prev = the nearest byte before it in the chunk that is not '\r' (-1: none), open_has_first =
// the line open at the chunk's start already had its first byte in an earlier chunk.
YSQ_HD bool ysq_is_first(uint8_t c, int prev, bool open_has_first) {
    if (c == '\r' || c == '\n') return false;
    return prev < 0 ? !open_has_first : prev == '\n';
}

// What a line is, from its first byte (0: none) and its number.
YSQ_HD int ysq_line_role(int fmt, uint32_t first, uint64_t line) {
    if (fmt == YSQ_FASTA) return first == '>' ? YSQ_ROLE_HEADER : YSQ_ROLE_SEQ;
    const uint32_t ph = (uint32_t)(line & 3);
    return ph == 0 ? YSQ_ROLE_HEADER : ph == 1 ? YSQ_ROLE_SEQ : YSQ_ROLE_DROP;
}

// FASTQ: a line whose first byte is not the '@' (line 4i) or '+' (line 4i + 2) due there; first = 0 for an empty line.
YSQ_HD bool ysq_fastq_bad(uint32_t first, uint64_t line) {
    const uint32_t ph = (uint32_t)(line & 3);
    return (ph == 0 && first != '@') || (ph == 2 && first != '+');
}

// Flags of byte c in a line of `role`; is_first = it is the line's first byte.  The first byte of a header line becomes the
// record separator ('\n', which breaks every window across two records) and opens the record; the rest of a header line is the
// record's name.  '\r' and '\n' are never kept: a FASTA record's inner line ends vanish, so windows run across wrapped lines.
YSQ_HD uint32_t ysq_byte_flags(uint8_t c, int role, bool is_first, bool want_names) {
    if (c == '\r' || c == '\n') return 0;
    if (role == YSQ_ROLE_SEQ) return YSQ_F_SEQ;
    if (role == YSQ_ROLE_HEADER) return is_first ? (YSQ_F_SEQ | YSQ_F_REC) : (want_names ? YSQ_F_NAME : 0u);
    return 0;
}
YSQ_HD uint8_t ysq_out_byte(uint8_t c, uint32_t flags) { return (flags & YSQ_F_REC) ? (uint8_t)'\n' : c; }

// The bases carried into the next chunk: the last min(k - 1, bases of the open record) bytes of the compacted buffer.
// open_begin = where the open record's bases start in it (just behind its separator; 0 when it began in an earlier chunk).
YSQ_HD uint64_t ysq_carry_begin(uint64_t n_out, uint64_t open_begin, int k) {
    const uint64_t keep = (uint64_t)(k - 1);
    const uint64_t b = n_out > keep ? n_out - keep : 0;
    return b > open_begin ? b : open_begin;
}

// End of a chunk: carry the state into the next one.  n_nl = '\n' bytes of the chunk, n_rec = records started in it,
// last_first = first byte of the line still open at its end (0: none), out[0, n_out) = its compacted buffer, open_begin as
// for ysq_carry_begin.
YSQ_HD void ysq_advance(ysq_state* s, uint64_t n_nl, uint64_t n_rec, uint32_t last_first, const uint8_t* out, uint64_t n_out,
                        uint64_t open_begin, int k) {
    const uint64_t cb = ysq_carry_begin(n_out, open_begin, k);
    for (uint64_t j = cb; j < n_out; j++) s->carry[j - cb] = out[j];
    s->n_carry = (uint32_t)(n_out - cb);
    s->open_first = last_first;
    s->line += n_nl;
    s->n_records += n_rec;
}

// End of a FASTQ file: 0 = fine; 1 = the line count (trailing empty lines dropped) is not a multiple of 4, *value = that
// count; 2 = a record breaks the structure, *value = the 1-based number of its first line.
YSQ_HD int ysq_fastq_end_check(const ysq_state* s, uint64_t* value) {
    const uint64_t n_lines = s->last_nonempty1;
    if (n_lines % 4) { *value = n_lines; return 1; }
    uint64_t bad = s->first_bad;
    if (s->first_bad_empty < n_lines && s->first_bad_empty < bad) bad = s->first_bad_empty;
    if (bad != ~0ull) { *value = bad / 4 * 4 + 1; return 2; }
    return 0;
}
