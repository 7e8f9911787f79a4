// TEST HARNESS: the chunked parse of seq_stream.cu for a stream of several k-mer sizes, compiled from seq_stream.cuh for the
// host.  Each chunk is parsed once; the state carries min(k_max - 1, bases of the open record) into the next chunk; every k
// takes its windows from the same compacted buffer, and a window is taken only when ysq_window_new says the previous chunk
// has not hashed it.  The CPU suite holds the windows of every k against sketch.read_records for any split of the input.
// Only the scans and the thread loops are re-stated here; every decision goes through the header's functions.  Not part of
// the product.
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../yacht_b200/csrc/seq_stream.cuh"

namespace {

struct Walk {
    ysq_state s{};
    std::vector<int> ks;
    int k_max = 0;
    int want_names = 0;           // 2: every record, 1: FASTA records
    bool file_started = false;
    int fmt = YSQ_FMT_NONE;
    std::string bases;            // new bytes of every chunk, concatenated: '\n' + record 0 + '\n' + record 1 ...
    std::vector<std::vector<uint64_t>> windows;   // per k: (record << 32 | start in the record) of every window taken
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
    off.push_back(out.size());
    // every k on the same buffer, as the hashing kernels take it: inside one sketch range [off[j], off[j + 1]), no separator
    // inside, and new by the window rule
    for (size_t ki = 0; ki < w.ks.size(); ki++) {
        const int k = w.ks[ki];
        for (uint64_t j = 0; j + 1 < off.size(); j++) {
            for (uint64_t p = off[j]; p + k <= off[j + 1]; p++) {
                if (!ysq_window_new(p, k, s.n_carry)) continue;
                bool ok = true;
                for (int q = 0; q < k && ok; q++) ok = out[p + q] != '\n';
                if (!ok) continue;
                const uint64_t rec = base_rec + j - 1;       // sketch 0 of a chunk is the record open at its start
                const uint64_t gpos = w.bases.size() + p - s.n_carry;
                w.windows[ki].push_back((rec << 32) | (gpos - w.rec_pos[rec] - 1));
            }
        }
    }
    w.bases.append((const char*)out.data() + s.n_carry, out.size() - s.n_carry);
    ysq_advance(&s, n_nl, n_rec, first[n_nl], out.data(), out.size(), n_rec ? off[n_rec] + 1 : 0, w.k_max);
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

extern "C" int mk_begin(const int* ks, int n_k, int want_names) {
    if (n_k < 1 || n_k > YSQ_MAX_K) return 1;
    g_walk = Walk();
    g_walk.ks.assign(ks, ks + n_k);
    g_walk.k_max = *std::max_element(ks, ks + n_k);
    g_walk.windows.assign(n_k, {});
    g_walk.want_names = want_names;
    reset_file(g_walk);
    return 0;
}
// 0 = the file parsed; 1 = an error, text in mk_error()
extern "C" int mk_file(const uint8_t* data, uint64_t n, const uint64_t* cuts, uint64_t n_cuts) {
    return feed_file(g_walk, data, n, cuts, n_cuts) ? 0 : 1;
}
extern "C" const char* mk_error() { return g_walk.err.c_str(); }
extern "C" uint64_t mk_bases(const uint8_t** p) { *p = (const uint8_t*)g_walk.bases.data(); return g_walk.bases.size(); }
extern "C" uint64_t mk_names(const uint8_t** p) { *p = (const uint8_t*)g_walk.names.data(); return g_walk.names.size(); }
extern "C" uint64_t mk_windows(int ki, const uint64_t** p) { *p = g_walk.windows[ki].data(); return g_walk.windows[ki].size(); }
extern "C" uint64_t mk_records() { return g_walk.s.n_records; }
