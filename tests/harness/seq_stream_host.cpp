// TEST HARNESS: compiles yacht_b200/csrc/seq_stream.cuh -- the per-byte and per-line rules and the chunk-to-chunk state the
// stream kernels use -- for the host and walks the chunked parse of seq_stream.cu serially, so that the CPU suite can hold it
// against sketch.read_records for any split of the input.  Only the scans and the thread loops are re-stated here; every
// decision goes through the header's functions.  Not part of the product.
#include <stdint.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../yacht_b200/csrc/seq_stream.cuh"

namespace {

struct Walk {
    ysq_state s{};
    int k = 0;
    int want_names = 0;           // 2: every record, 1: FASTA records
    bool file_started = false;
    int fmt = YSQ_FMT_NONE;
    // what the hashing kernels would see, mapped back onto the stream of records
    std::string bases;            // new bytes of every chunk, concatenated: '\n' + record 0 + '\n' + record 1 ...
    std::vector<uint64_t> windows;// (record << 32 | start in the record) of every '\n'-free window of k bytes, as hashed
    std::string names;
    std::vector<uint64_t> name_off;
    std::vector<uint64_t> rec_pos;// position of every record's separator in `bases`
    std::string err;
};

void chunk(Walk& w, const uint8_t* c, uint64_t n) {
    if (!n) return;
    ysq_state& s = w.s;
    const bool open_has = s.open_first != 0;
    std::vector<uint32_t> line(n);
    std::vector<int> prev(n);
    uint32_t L = 0;
    int64_t last = -1;
    for (uint64_t i = 0; i < n; i++) {                       // the two scans
        line[i] = L;
        prev[i] = last < 0 ? -1 : (int)c[last];
        if (c[i] == '\n') L++;
        if (c[i] != '\r') last = (int64_t)i;
    }
    const uint64_t n_nl = L;
    std::vector<uint32_t> first(n_nl + 1, 0);
    if (open_has) first[0] = s.open_first;
    for (uint64_t i = 0; i < n; i++)
        if (ysq_is_first(c[i], prev[i], open_has)) first[line[i]] = c[i];
    const bool names = w.want_names == 2 || (w.want_names == 1 && (int)s.fmt == YSQ_FASTA);
    std::vector<uint8_t> out(s.carry, s.carry + s.n_carry);
    std::vector<uint64_t> off(1, 0);
    const uint64_t base_rec = s.n_records;
    for (uint64_t i = 0; i < n; i++) {                       // classify + scatter
        const uint64_t G = s.line + line[i];
        const uint32_t f = first[line[i]];
        const bool is_first = ysq_is_first(c[i], prev[i], open_has);
        const uint32_t fl = ysq_byte_flags(c[i], ysq_line_role((int)s.fmt, f, G), is_first, names);
        if ((int)s.fmt == YSQ_FASTQ) {
            if (is_first) {
                if (G + 1 > s.last_nonempty1) s.last_nonempty1 = G + 1;
                if (ysq_fastq_bad(c[i], G) && G < s.first_bad) s.first_bad = G;
            } else if (c[i] == '\n' && f == 0 && ysq_fastq_bad(0, G) && G < s.first_bad_empty) {
                s.first_bad_empty = G;
            }
        }
        if (fl & YSQ_F_SEQ) {
            if (fl & YSQ_F_REC) {
                off.push_back(out.size());
                w.rec_pos.push_back(w.bases.size() + out.size() - s.n_carry);
                if (names) w.name_off.push_back(w.names.size());
            }
            out.push_back(ysq_out_byte(c[i], fl));
        }
        if (fl & YSQ_F_NAME) w.names.push_back((char)c[i]);
    }
    const uint64_t n_rec = off.size() - 1;
    // windows as the hashing kernel takes them: inside one sketch range [off[j], off[j + 1]), no separator inside
    off.push_back(out.size());
    for (uint64_t j = 0; j + 1 < off.size(); j++) {
        for (uint64_t p = off[j]; p + w.k <= off[j + 1]; p++) {
            bool ok = true;
            for (int q = 0; q < w.k && ok; q++) ok = out[p + q] != '\n';
            if (!ok) continue;
            const uint64_t rec = base_rec + j - 1;           // sketch 0 of a chunk is the record open at its start
            // the window's start inside its record: its position in `bases` minus the record's separator position - 1
            const uint64_t gpos = w.bases.size() + p - s.n_carry;
            w.windows.push_back((rec << 32) | (gpos - w.rec_pos[rec] - 1));
        }
    }
    w.bases.append((const char*)out.data() + s.n_carry, out.size() - s.n_carry);
    ysq_advance(&s, n_nl, n_rec, first[n_nl], out.data(), out.size(), n_rec ? off[n_rec] + 1 : 0, w.k);
}

void reset_file(Walk& w) {
    w.file_started = false;
    w.fmt = YSQ_FMT_NONE;
    w.s.line = 0;
    w.s.last_nonempty1 = 0;
    w.s.first_bad = ~0ull;
    w.s.first_bad_empty = ~0ull;
    w.s.fmt = YSQ_FMT_NONE;
    w.s.open_first = 0;
    w.s.n_carry = 0;
}

// one file, fed in pieces cut at cuts[0 .. n_cuts) (ascending positions), each piece one device chunk
bool feed_file(Walk& w, const uint8_t* data, uint64_t n, const uint64_t* cuts, uint64_t n_cuts) {
    uint64_t a = 0;
    for (uint64_t ci = 0; ci <= n_cuts; ci++) {
        const uint64_t b = ci < n_cuts ? cuts[ci] : n;
        const uint8_t* p = data + a;
        uint64_t m = b - a;
        a = b;
        if (!w.file_started) {
            while (m && ysq_is_space(*p)) { p++; m--; }
            if (!m) continue;
            w.fmt = ysq_format_of(*p);
            if (w.fmt == YSQ_FMT_NONE) { w.err = "neither FASTA ('>') nor FASTQ ('@')"; return false; }
            w.s.fmt = (uint32_t)w.fmt;
            w.file_started = true;
        }
        chunk(w, p, m);
    }
    if (w.fmt == YSQ_FASTQ) {
        uint64_t v = 0;
        const int bad = ysq_fastq_end_check(&w.s, &v);
        if (bad == 1) { w.err = "FASTQ with " + std::to_string(v) + " lines (not a multiple of 4)"; return false; }
        if (bad == 2) { w.err = "malformed FASTQ record at line " + std::to_string(v); return false; }
    }
    reset_file(w);
    return true;
}

Walk g_walk;

}  // namespace

extern "C" int sh_begin(int k, int want_names) {
    g_walk = Walk();
    g_walk.k = k;
    g_walk.want_names = want_names;
    reset_file(g_walk);
    return 0;
}
// 0 = the file parsed; 1 = an error, text in sh_error()
extern "C" int sh_file(const uint8_t* data, uint64_t n, const uint64_t* cuts, uint64_t n_cuts) {
    return feed_file(g_walk, data, n, cuts, n_cuts) ? 0 : 1;
}
extern "C" const char* sh_error() { return g_walk.err.c_str(); }
extern "C" uint64_t sh_bases(const uint8_t** p) { *p = (const uint8_t*)g_walk.bases.data(); return g_walk.bases.size(); }
extern "C" uint64_t sh_names(const uint8_t** p) { *p = (const uint8_t*)g_walk.names.data(); return g_walk.names.size(); }
extern "C" uint64_t sh_name_offsets(const uint64_t** p) { *p = g_walk.name_off.data(); return g_walk.name_off.size(); }
extern "C" uint64_t sh_windows(const uint64_t** p) { *p = g_walk.windows.data(); return g_walk.windows.size(); }
extern "C" uint64_t sh_records() { return g_walk.s.n_records; }
