// =====================================================================================
// TEST INFRASTRUCTURE ONLY.  CPU restatement ("port") of the reference train core.
//
// Nothing in the product path (yacht_b200/, include/) may include, link or execute this
// file.  It is imported only by tests/, __graft_entry__.smoke() and bench.py's
// cpu_baseline / --impl reference legs, as the checker.
//
// Parity status: PINNED.  tests/test_oracle_pinned.py checks this restatement against
//   (a) outputs of the unmodified reference core compiled from /root/reference/src/cpp
//       (oracle/_ref/run_yacht_train_core_ref, built by oracle/Makefile), on the
//       20-genome fixture of the reference's own tests, the hand-made edge set of
//       SURVEY.md Appendix B and seeded synthetic sets, and
//   (b) the committed golden vectors under tests/golden/ that were produced by that
//       same reference binary (tests/golden/make_train_golden.py).
//
// What is restated (reference file:line):
//   * genome id = line index of the file list            src/cpp/main.cpp:127-139
//   * sketch  = [0]["signatures"][0]["mins"] of the file  src/cpp/main.cpp:62-84
//     (missing file => empty sketch, :68-71)
//   * inverted index hash -> genome ids, one entry per occurrence, ascending id;
//     hashes with a single posting are dropped; three statistics
//                                                        src/cpp/main.cpp:215-246
//   * M[i][g] += 1 for every query hash of i and every posting g of that hash
//                                                        src/cpp/main.cpp:252-262
//   * per ordered pair (i,j): skip i==j, M==0, empty sketches, zero "union";
//     jaccard, c_ij, c_ji in double; keep iff !(c_ij < thr) src/cpp/main.cpp:274-308
//   * greedy selection: std::sort by size only, visit ascending, drop a genome iff one
//     of its similars that is not already dropped is at least as large
//                                                        src/cpp/main.cpp:371-420
//   * pair-file line format (ostream default precision == "%g") src/cpp/main.cpp:305
//
// The index here is a sort-grouped posting array instead of the reference's
// unordered_map; the counts it yields are identical (same multiset of (hash, id)).
//
// yo_train_sparse shares the index and greedy stages with yo_train and accumulates each row over
// the columns its postings touch instead of a dense row of n counters; tests/test_oracle_pinned.py
// checks it against yo_train field for field.
// =====================================================================================
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <numeric>
#include <sstream>
#include <string>
#include <utility>
#include <vector>

extern "C" {

struct yo_pair {
    int32_t i, j, count;
    int32_t _pad;
    double jaccard, c_ij, c_ji;
};

struct yo_result {
    yo_pair* pairs;        // row-major: i ascending, j ascending (reference emission order with -t 1 -p 1)
    uint64_t n_pairs;
    int32_t* selected;     // genome ids in greedy visit order (reference :403,412-418)
    uint32_t n_selected;
    uint64_t n_distinct;   // "Total number of distinct hashes"               (:242)
    uint64_t n_singleton;  // "... that appear in only one sketch"            (:243)
    uint64_t n_index;      // "Size of the index"                             (:244)
    uint64_t n_postings;   // P = sum of posting lengths with L >= 2
    uint64_t n_increments; // W = sum of L^2 over those postings (reference's ++ count)
};

void yo_free_result(yo_result* r) {
    if (!r) return;
    free(r->pairs);
    free(r->selected);
    r->pairs = nullptr;
    r->selected = nullptr;
}

}  // extern "C"

// The inverted index of main.cpp:215-246 and its statistics.
struct yo_index {
    std::vector<uint64_t> key;       // kept hashes (posting length >= 2), ascending
    std::vector<uint64_t> post_off;  // CSR offsets into post
    std::vector<int32_t> post;
};

static void build_index(const uint64_t* hashes, const uint64_t* offsets, uint32_t n, yo_index& ix, yo_result* out) {
    const uint64_t T = offsets[n];
    // entries are generated in ascending (genome, position) order; a stable sort by hash keeps
    // each posting list in ascending genome order with one entry per occurrence.
    std::vector<std::pair<uint64_t, int32_t>> ent;
    ent.reserve(T);
    for (uint32_t g = 0; g < n; g++)
        for (uint64_t p = offsets[g]; p < offsets[g + 1]; p++) ent.emplace_back(hashes[p], (int32_t)g);
    std::stable_sort(ent.begin(), ent.end(),
                     [](const std::pair<uint64_t, int32_t>& a, const std::pair<uint64_t, int32_t>& b) { return a.first < b.first; });

    ix.post_off.push_back(0);
    for (uint64_t s = 0; s < T;) {
        uint64_t e = s;
        while (e < T && ent[e].first == ent[s].first) e++;
        out->n_distinct++;
        if (e - s >= 2) {
            ix.key.push_back(ent[s].first);
            for (uint64_t q = s; q < e; q++) ix.post.push_back(ent[q].second);
            ix.post_off.push_back(ix.post.size());
            out->n_postings += e - s;
            out->n_increments += (e - s) * (e - s);
        } else {
            out->n_singleton++;
        }
        s = e;
    }
    out->n_index = ix.key.size();
}

// M[i][g] += 1 for every query hash of row i and every posting g of that hash (main.cpp:252-262)
template <class F>
static void for_each_posting(const uint64_t* hashes, const uint64_t* offsets, const yo_index& ix, uint32_t i, F&& f) {
    for (uint64_t p = offsets[i]; p < offsets[i + 1]; p++) {
        auto it = std::lower_bound(ix.key.begin(), ix.key.end(), hashes[p]);
        if (it == ix.key.end() || *it != hashes[p]) continue;
        const size_t r = it - ix.key.begin();
        for (uint64_t q = ix.post_off[r]; q < ix.post_off[r + 1]; q++) f(ix.post[q]);
    }
}

// the reference's test of one ordered pair (main.cpp:274-308); appends it when it is kept
static void test_pair(const uint64_t* offsets, uint32_t i, uint32_t j, int32_t m, double thr, std::vector<yo_pair>& pairs) {
    if (i == j) return;
    if (m == 0) return;
    const uint64_t ni = offsets[i + 1] - offsets[i];
    const uint64_t nj = offsets[j + 1] - offsets[j];
    if (ni == 0 || nj == 0) return;
    // the reference evaluates size_t + size_t - int, i.e. modulo 2^64 (main.cpp:292,296)
    const uint64_t uni = ni + nj - (uint64_t)(int64_t)m;
    if (uni == 0) return;
    const double jac = 1.0 * m / uni;
    const double cij = 1.0 * m / ni;
    const double cji = 1.0 * m / nj;
    if (cij < thr) return;
    yo_pair pr;
    pr.i = (int32_t)i; pr.j = (int32_t)j; pr.count = m; pr._pad = 0;
    pr.jaccard = jac; pr.c_ij = cij; pr.c_ji = cji;
    pairs.push_back(pr);
}

// greedy selection (main.cpp:371-420) over the kept pairs (row-major: each genome's similars in ascending j).
// Same container type, same initial order (file-list order), same comparator, same std::sort => the same
// permutation of equal-size genomes as the reference build.
static void greedy(const uint64_t* offsets, uint32_t n, const std::vector<yo_pair>& pairs, yo_result* out) {
    std::vector<uint64_t> sim_off(n + 1, 0);
    for (const yo_pair& pr : pairs) sim_off[pr.i + 1]++;
    for (uint32_t g = 0; g < n; g++) sim_off[g + 1] += sim_off[g];
    std::vector<std::pair<int, int>> id_size(n);
    for (uint32_t g = 0; g < n; g++) id_size[g] = {(int)g, (int)(offsets[g + 1] - offsets[g])};
    std::sort(id_size.begin(), id_size.end(),
              [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.second < b.second; });
    std::vector<bool> dropped(n, false);
    std::vector<int32_t> selected;
    for (uint32_t v = 0; v < n; v++) {
        const int g = id_size[v].first;
        const int sz = id_size[v].second;
        bool keep = true;
        for (uint64_t k = sim_off[g]; k < sim_off[g + 1]; k++) {
            const int32_t o = pairs[k].j;
            if (dropped[o]) continue;
            const int so = (int)(offsets[o + 1] - offsets[o]);
            if (so >= sz) { keep = false; break; }
        }
        if (keep) selected.push_back(g);
        else dropped[g] = true;
    }
    out->n_selected = (uint32_t)selected.size();
    out->selected = (int32_t*)malloc(sizeof(int32_t) * (selected.size() ? selected.size() : 1));
    if (!selected.empty()) memcpy(out->selected, selected.data(), sizeof(int32_t) * selected.size());
}

static void emit_pairs(const std::vector<yo_pair>& pairs, yo_result* out) {
    out->n_pairs = pairs.size();
    out->pairs = (yo_pair*)malloc(sizeof(yo_pair) * (pairs.size() ? pairs.size() : 1));
    if (!pairs.empty()) memcpy(out->pairs, pairs.data(), sizeof(yo_pair) * pairs.size());
}

extern "C" {

// hashes: concatenated sketches (any order inside a sketch, duplicates allowed);
// offsets: n+1 prefix offsets into hashes.
int yo_train(const uint64_t* hashes, const uint64_t* offsets, uint32_t n, double thr, yo_result* out) {
    memset(out, 0, sizeof(*out));
    yo_index ix;
    build_index(hashes, offsets, n, ix, out);

    // ---- counts + threshold (main.cpp:252-308): a dense row of n counters, scanned in full -----
    std::vector<yo_pair> pairs;
    std::vector<int32_t> row(n, 0);
    for (uint32_t i = 0; i < n; i++) {
        std::fill(row.begin(), row.end(), 0);
        for_each_posting(hashes, offsets, ix, i, [&](int32_t g) { row[g]++; });
        for (uint32_t j = 0; j < n; j++) test_pair(offsets, i, j, row[j], thr, pairs);
    }
    emit_pairs(pairs, out);
    greedy(offsets, n, pairs, out);
    return 0;
}

// The same result in O(sum of L^2) instead of O(n^2): per row, only the columns a posting touched are
// visited, so databases of millions of genomes can be checked.  With a row range [row_begin, row_end) it
// returns what ygpu_pairwise_flag does for that range: both ordered pairs of every {i, j} whose smaller
// genome i lies in the range (the counts are symmetric), ordered by (i, j); the full range is yo_train's
// pair list.  `selected` is the greedy order over the returned pairs (the reference's for the full range).
int yo_train_sparse(const uint64_t* hashes, const uint64_t* offsets, uint32_t n, double thr, uint32_t row_begin,
                    uint32_t row_end, yo_result* out) {
    memset(out, 0, sizeof(*out));
    if (row_begin > row_end || row_end > n) return 1;
    yo_index ix;
    build_index(hashes, offsets, n, ix, out);

    std::vector<yo_pair> pairs;
    std::vector<int32_t> row(n, 0);
    std::vector<int32_t> touched;
    for (uint32_t i = row_begin; i < row_end; i++) {
        touched.clear();
        for_each_posting(hashes, offsets, ix, i, [&](int32_t g) { if (row[g]++ == 0) touched.push_back(g); });
        std::sort(touched.begin(), touched.end());
        for (int32_t j : touched) {
            if ((uint32_t)j > i) {
                test_pair(offsets, i, (uint32_t)j, row[j], thr, pairs);
                test_pair(offsets, (uint32_t)j, i, row[j], thr, pairs);
            }
            row[j] = 0;
        }
    }
    std::sort(pairs.begin(), pairs.end(), [](const yo_pair& a, const yo_pair& b) { return a.i != b.i ? a.i < b.i : a.j < b.j; });
    emit_pairs(pairs, out);
    greedy(offsets, n, pairs, out);
    return 0;
}

// One pair-file line exactly as the reference prints it (main.cpp:305): ints, then three
// doubles at ostream default precision (6 significant digits, "%g").
int yo_format_pair(const yo_pair* p, char* buf, int buflen) {
    return snprintf(buf, buflen, "%d,%d,%g,%g,%g", p->i, p->j, p->jaccard, p->c_ij, p->c_ji);
}

}  // extern "C"

#ifdef YO_WITH_MAIN
// -------------------------------------------------------------------------------------
// The same restatement behind the reference's command line (main.cpp:142-184):
//   train_oracle [-t T] [-c C] [-p P] file_list working_directory output_filename
// -t / -p only change how the pair lines are split over <pass>_<tid>.txt files.
// The sketch reader is a deliberately naive text scan (first "signatures", then the
// first "mins" array after it) -- independent of the product's ingest code.
// -------------------------------------------------------------------------------------
static bool naive_read_mins(const std::string& path, std::vector<uint64_t>& out) {
    std::ifstream f(path, std::ios::binary);
    if (!f.is_open()) { fprintf(stderr, "Could not open the file!\n"); return false; }
    std::stringstream ss; ss << f.rdbuf();
    const std::string s = ss.str();
    size_t a = s.find("\"signatures\"");
    if (a == std::string::npos) return true;
    size_t b = s.find("\"mins\"", a);
    if (b == std::string::npos) return true;
    size_t c = s.find('[', b);
    size_t d = s.find(']', c);
    const char* p = s.c_str() + c + 1;
    const char* e = s.c_str() + d;
    while (p < e) {
        while (p < e && (*p < '0' || *p > '9')) p++;
        if (p >= e) break;
        char* q;
        out.push_back(strtoull(p, &q, 10));
        p = q;
    }
    return true;
}

int main(int argc, char** argv) {
    int T = 1, P = 1; double thr = 0.9;
    std::vector<std::string> pos;
    for (int a = 1; a < argc; a++) {
        std::string s = argv[a];
        if ((s == "-t" || s == "--threads") && a + 1 < argc) T = atoi(argv[++a]);
        else if ((s == "-p" || s == "--passes") && a + 1 < argc) P = atoi(argv[++a]);
        else if ((s == "-c" || s == "--containment_threshold") && a + 1 < argc) thr = strtod(argv[++a], nullptr);
        else pos.push_back(s);
    }
    if (pos.size() != 3 || T < 1 || P < 1 || thr < 0.0 || thr > 1.0) { fprintf(stderr, "bad arguments\n"); return 1; }
    std::vector<std::string> names;
    { std::ifstream fl(pos[0]); std::string line; while (std::getline(fl, line)) names.push_back(line); }
    const uint32_t n = (uint32_t)names.size();
    std::vector<uint64_t> hashes, offsets(1, 0);
    for (uint32_t g = 0; g < n; g++) {
        std::vector<uint64_t> m; naive_read_mins(names[g], m);
        hashes.insert(hashes.end(), m.begin(), m.end());
        offsets.push_back(hashes.size());
    }
    yo_result r;
    yo_train(hashes.data(), offsets.data(), n, thr, &r);
    printf("Total number of distinct hashes: %llu\n", (unsigned long long)r.n_distinct);
    printf("Total number of distinct hashes that appear in only one sketch: %llu\n", (unsigned long long)r.n_singleton);
    printf("Size of the index: %llu\n", (unsigned long long)r.n_index);
    // file partition of main.cpp:318,338-348 (rows per pass = ceil(n/P); rows per thread = floor)
    const int per_pass = (int)((n + P - 1) / P);
    uint64_t k = 0;
    for (int pass = 0; pass < P; pass++) {
        const int ps = pass * per_pass, pe = (pass == P - 1) ? (int)n : (pass + 1) * per_pass;
        const int chunk = (pe - ps) / T;
        for (int t = 0; t < T; t++) {
            const int re = (t == T - 1) ? pe : ps + (t + 1) * chunk;
            char fn[4096]; snprintf(fn, sizeof fn, "%s/%d_%03d.txt", pos[1].c_str(), pass, t);
            FILE* fo = fopen(fn, "w");
            if (!fo) { fprintf(stderr, "cannot write %s\n", fn); return 2; }
            while (k < r.n_pairs && r.pairs[k].i < re) {
                char buf[256]; yo_format_pair(&r.pairs[k], buf, sizeof buf);
                fprintf(fo, "%s\n", buf); k++;
            }
            fclose(fo);
        }
    }
    FILE* fs = fopen(pos[2].c_str(), "w");
    if (!fs) { fprintf(stderr, "cannot write %s\n", pos[2].c_str()); return 2; }
    for (uint32_t s = 0; s < r.n_selected; s++) fprintf(fs, "%s\n", names[r.selected[s]].c_str());
    fclose(fs);
    yo_free_result(&r);
    return 0;
}
#endif
