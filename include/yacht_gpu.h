/*
 * yacht_gpu.h -- C ABI of libyachtgpu: the B200 (sm_100a) replacement for YACHT's data-parallel
 * hot path.  Plain C types only: no CUDA, torch or C++ types cross this boundary.
 *
 * What each entry point replaces in the reference (KoslickiLab/YACHT, paths relative to the
 * reference root; the train core is src/cpp/main.cpp, the run-side compute is
 * src/yacht/hypothesis_recovery_src.py):
 *
 *   ygpu_read_signatures    read_min_hashes() / read_sketches()                main.cpp:62-124
 *   ygpu_read_signatures_ksize   load_signature_with_ksize() per manifest row  utils.py:31-51, hypothesis_recovery_src.py:154-172
 *   ygpu_load_sketches      the in-memory result of read_sketches()            main.cpp:89-124
 *   ygpu_upload_begin / _block / _finish   the same, streamed while parsing        main.cpp:89-124
 *                           (vector<vector<hash_t>> sketches, :51) as one flat
 *                           uint64 array + CSR offsets; genome id = file-list
 *                           line index (:127-139)
 *   ygpu_build_index        compute_index_from_sketches()                      main.cpp:215-246
 *   ygpu_pairwise_flag      compute_intersection_matrix[_by_sketches]()        main.cpp:249-366
 *                           counts (:252-262) fused with threshold/emit (:274-308)
 *   ygpu_greedy_select      do_yacht_train(): greedy near-duplicate removal    main.cpp:371-420
 *   ygpu_row_partition      the contiguous row chunks per thread / per pass    main.cpp:338-349
 *   ygpu_comm_init / ygpu_load_sketches_sharded / ygpu_train_step_sharded
 *                           the same three steps (:215-366) with one rank per GPU: index build split by hash
 *                           range, count by query rows (the reference's row chunks per thread / pass, :338-349)
 *   ygpu_exclusive_hashes   `sourmash scripts multisearch ... -t 0`            hypothesis_recovery_src.py:93-113
 *                           (which reference genomes share >= 1 hash with the
 *                           sample: counts[g].n_overlap > 0), followed by
 *                           get_exclusive_hashes()                             hypothesis_recovery_src.py:116-206
 *   ygpu_hyp_test           single_hyp_test() + get_alt_mut_rate()             hypothesis_recovery_src.py:209-306
 *   ygpu_alt_mut_rate       get_alt_mut_rate() on its own                      hypothesis_recovery_src.py:209-230
 *
 * Conventions: every function returns 0 on success and a negative ygpu_status otherwise; the
 * text of the last error is available from ygpu_last_error().  The caller owns every input
 * buffer; the library owns every output buffer until ygpu_free().  One context drives one GPU;
 * calls on one context are not re-entrant.  There is NO CPU fallback: without a CUDA device
 * ygpu_ctx_create fails with YGPU_ERR_NO_DEVICE.
 */
#ifndef YACHT_GPU_H
#define YACHT_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ygpu_ctx ygpu_ctx;

typedef enum {
    YGPU_OK = 0,
    YGPU_ERR_NO_DEVICE = -1,   /* no CUDA device / driver: the product path refuses to run   */
    YGPU_ERR_CUDA = -2,        /* a CUDA runtime call or kernel failed                       */
    YGPU_ERR_ARG = -3,         /* invalid argument                                           */
    YGPU_ERR_STATE = -4,       /* call order violated (e.g. pairwise before build_index)     */
    YGPU_ERR_NOMEM = -5        /* host or device allocation failed                           */
} ygpu_status;

/* One flagged ORDERED pair: genome i is contained in genome j with `count` shared hashes
 * (count == intersectionMatrix[i][j], main.cpp:258) and count / |S_i| >= threshold (:297-303). */
typedef struct {
    int32_t i;
    int32_t j;
    int32_t count;
} ygpu_pair;

/* The three banner statistics of main.cpp:242-244 plus the workload counts of SURVEY.md 8(d). */
typedef struct {
    uint64_t n_hashes;      /* T  = sum of sketch sizes                                        */
    uint64_t n_distinct;    /* U  = "Total number of distinct hashes"                          */
    uint64_t n_singleton;   /*      "... that appear in only one sketch"                       */
    uint64_t n_index;       /* U2 = "Size of the index"                                        */
    uint64_t n_postings;    /* P  = sum of posting lengths L over hashes with L >= 2           */
    uint64_t n_increments;  /* W  = sum of L^2 (the ++ operations the reference performs)      */
    uint64_t n_row_items;   /* entries of the per-genome work lists (implementation detail)    */
    uint32_t max_sketch;    /* largest sketch size                                             */
    uint32_t has_duplicates;/* 1 if some sketch holds the same hash twice                      */
    uint32_t index_path;    /* 1 = MSD partition + shared-memory grouping, 0 = general sort path */
    uint32_t big_buckets;   /* path 1: final buckets too large for shared memory, grouped by the sort-based side route */
} ygpu_index_stats;

/* Device timings (CUDA events on the context's stream) accumulated since ygpu_reset_timers(). */
typedef struct {
    double ms_h2d;          /* ygpu_load_sketches host->device copies                          */
    double ms_sort;         /* K2a: MSD partition (or the (hash, genome) radix sort of the general path) */
    double ms_index;        /* K2b: grouping -> postings + per-genome work lists                */
    double ms_count;        /* K3+K4: pairwise shared-hash count fused with threshold/compact  */
    double ms_pairsort;     /* ordering of the flagged pairs by (i, j)                         */
    double ms_d2h;          /* pair-list device->host copy                                     */
    double ms_sample;       /* K5: sample membership + exclusive-hash reduction                */
    double ms_stats;        /* K6: binomial statistics                                         */
    uint64_t n_count_launches;   /* launches of the K3+K4 kernel                               */
    uint64_t n_kernel_launches;  /* launches of this library's own hand-written kernels         */
    uint64_t n_library_launches; /* launches it asked CUB for (radix sort / scan / reduce passes) */
    /* partition path, per kernel (their sum + the small scans in between = ms_sort):              */
    double ms_hist1, ms_scatter1, ms_hist2, ms_scatter2;
    double ms_group;        /* k2_group alone (ms_index additionally holds k2_items when sharded)  */
    double ms_sample_kernels; /* K5: the two probe passes over the partitioned reference alone (inside ms_sample) */
    /* sharded step: work-list build from the complete stream (k2_items_regions), the control collectives + cross-rank
     * waits between the phases, and the gather of the pair lists (inside ms_index / ms_pairsort)            */
    double ms_items, ms_sync, ms_gather;
    double ms_sketch;       /* ygpu_sketch_sequences: the k-mer hashing kernel (_k: every size's)                 */
} ygpu_timings;

/* Per reference genome, from ygpu_exclusive_hashes (hypothesis_recovery_src.py:194-204). */
typedef struct {
    uint32_t n_overlap;     /* |S_g  intersect  sample|  (multisearch: containment > 0 <=> n_overlap > 0) */
    uint32_t nontrivial;    /* 1 if the genome takes part in the exclusive-hash computation    */
    uint32_t n_exclusive;   /* hashes of g found in no other nontrivial genome                 */
    uint32_t n_match;       /* ... of which are present in the sample                          */
} ygpu_genome_counts;

/* One row of single_hyp_test's 8-tuple (hypothesis_recovery_src.py:297-306). */
typedef struct {
    int32_t in_sample_est;
    int32_t _pad;
    double p_val;
    int64_t num_exclusive_kmers;
    int64_t num_exclusive_kmers_coverage;
    int64_t num_matches;
    double acceptance_threshold_with_coverage;
    double actual_confidence_with_coverage;
    double alt_confidence_mut_rate_with_coverage;
} ygpu_hyp_row;

/* A set of sketches on the host, as ygpu_read_signatures returns it. */
typedef struct {
    uint64_t* hashes;       /* [offsets[n_genomes]] page-locked when pinned != 0                */
    uint64_t* offsets;      /* [n_genomes + 1]                                                  */
    uint32_t n_genomes;
    uint32_t n_unreadable;  /* files that could not be opened (they yield empty sketches)       */
    int32_t pinned;
    int32_t _pad;
} ygpu_sketch_set;

/* ---- context ------------------------------------------------------------------------------ */
int ygpu_device_count(void);
int ygpu_ctx_create(ygpu_ctx** out, int device);
void ygpu_ctx_destroy(ygpu_ctx* ctx);
const char* ygpu_last_error(const ygpu_ctx* ctx);      /* ctx may be NULL: last create error   */
void ygpu_free(void* p);                               /* release a library-owned host buffer  */
/* Page-locked host staging buffers (cudaHostAlloc) so ygpu_load_sketches copies at full PCIe
 * rate; plain malloc'ed memory is accepted too, just slower.  NULL on failure.               */
void* ygpu_host_alloc(uint64_t bytes);
void ygpu_host_free(void* p);
int ygpu_reset_timers(ygpu_ctx* ctx);
int ygpu_get_timings(ygpu_ctx* ctx, ygpu_timings* out);
/* CUDA-event stopwatch on the context's stream (slots 0..3): time a whole step from outside.    */
int ygpu_mark(ygpu_ctx* ctx, int slot);
int ygpu_elapsed_ms(ygpu_ctx* ctx, int slot_a, int slot_b, double* ms);
/* Tuning / test hooks: "force_tile_w" caps the accumulator tile width of the count kernel and
 * "force_u16" = 1 selects its packed 16-bit counters (both are otherwise chosen from N);
 * "index_path" = 0 forces the general sort-based index build (1 = automatic choice, default);
 * "count_kernel" = 1 forces the dense-row count kernel, 2 the warp-per-row one (0 = automatic);
 * "big_buckets" = 0 sends a database with ANY oversized final bucket to the general path (default 1:
 * only those buckets leave the partition path); "group_kernel" = 1 forces the general grouping kernel;
 * "run_path" = 0 forces the general sort-based run path (default 1: probe the partitioned reference);
 * "count_thresholds" = 0 evaluates the containment expression per pair in fp64 inside the count kernel (default 1: the
 * smallest passing count per genome is found with that expression once, the kernel compares integers);
 * "sketch_kernel" = 2 forces the byte-wise sketching kernel for every k-mer size (default 0: k <= 64 uses packed words);
 * "stream_chunk_bytes" = raw bytes per device chunk of ygpu_stream_* (default 64 MiB, at most 1 GiB).                */
int ygpu_set_option(ygpu_ctx* ctx, const char* name, int64_t value);
/* Read-only state of the last count call (ygpu_pairwise_flag / _device): "last_count_kernel" (1 = dense row accumulator,
 * 2 = warp per row), "last_count_overflow_rows" (rows the warp kernel deferred to the dense kernel), and the dense kernel's
 * accumulator geometry "last_count_tile_w" (columns per tile), "last_count_n_tiles" and "last_count_u16" (1 = packed 16-bit
 * counters).  Read-only state of the last ygpu_build_index on the partition path: "last_group2_grid" and "last_group_grid"
 * (CTAs of the k2_group2 and of the general k2_group launch; CTA c groups final buckets c, c + grid, ...) and
 * "last_big_chunks" (sorted chunks of the oversized-bucket route); each is 0 when that kernel or route did not run.
 * An unknown name fails with YGPU_ERR_ARG.                                                                                 */
int ygpu_get_option(ygpu_ctx* ctx, const char* name, int64_t* out);

/* ---- ingest (host side of the path) ------------------------------------------------------------ */
/* Parse n sourmash signature files (uncompressed JSON) on `threads` host threads: sketch i =
 * document[0]["signatures"][0]["mins"] of paths[i] (main.cpp:78); a file that cannot be opened
 * yields an empty sketch (main.cpp:68-71); malformed JSON is an error (text in errbuf).          */
int ygpu_read_signatures(const char* const* paths, uint32_t n, int threads, ygpu_sketch_set* out,
                         char* errbuf, uint64_t errlen);
/* The run side's rule instead (load_signature_with_ksize, utils.py:31-51): all records and sub-signatures of a file are
 * candidates and exactly one must have k-mer size `ksize`; a file with none or several is an error ("Expected exactly one
 * signature with ksize ...", text in errbuf), like in the reference.                                                    */
int ygpu_read_signatures_ksize(const char* const* paths, uint32_t n, int threads, int ksize, ygpu_sketch_set* out,
                               char* errbuf, uint64_t errlen);
void ygpu_sketch_set_free(ygpu_sketch_set* s);

/* ---- train path ---------------------------------------------------------------------------- */
/* hashes[offsets[g] .. offsets[g+1]) is sketch g (any order, duplicates allowed).  HOST pointers;
 * copied to the device (pinned staging is the caller's choice).                                 */
int ygpu_load_sketches(ygpu_ctx* ctx, const uint64_t* hashes, const uint64_t* offsets, uint32_t n_genomes);
/* Same sketches given as `nblocks` separate HOST pieces that concatenate to the flat hash array
 * (what a multi-threaded parser leaves behind): copied piece by piece, no host-side assembly.   */
int ygpu_load_sketch_blocks(ygpu_ctx* ctx, const uint64_t* const* blocks, const uint64_t* block_lens, uint32_t nblocks,
                            const uint64_t* offsets, uint32_t n_genomes);
/* Streaming ingest for callers that parse files themselves (read_sketches(), main.cpp:89-124, parses while
 * nothing else happens): blocks of consecutive sketches are uploaded WHILE later files are still being parsed.
 * ygpu_upload_block is thread-safe (parser threads call it concurrently; the host block may be released when it
 * returns) and stages through page-locked bounce buffers; block ids are the caller's.  ygpu_upload_finish takes
 * the position of every block in the flat array (known once all sketch sizes are) and leaves the context in the
 * same state as ygpu_load_sketches.                                                                          */
int ygpu_upload_begin(ygpu_ctx* ctx);
int ygpu_upload_block(ygpu_ctx* ctx, uint32_t block_id, const uint64_t* hashes, uint64_t len);
int ygpu_upload_finish(ygpu_ctx* ctx, const uint64_t* block_dst, uint32_t nblocks, const uint64_t* offsets, uint32_t n_genomes);
/* Same, but DEVICE pointers on ctx's device; the arrays are copied device-to-device.            */
int ygpu_load_sketches_device(ygpu_ctx* ctx, const uint64_t* d_hashes, const uint64_t* d_offsets, uint32_t n_genomes);
int ygpu_build_index(ygpu_ctx* ctx, ygpu_index_stats* stats /* may be NULL */);
/* Flag ordered pairs whose query genome (member i) OR target lies in rows [row_begin,row_end):
 * the unordered pair {a<b} is evaluated once by the owner of row a, and both directions (a,b)
 * and (b,a) are tested against `threshold` exactly as main.cpp:296-303 does.  The union over a
 * partition of [0,n) into row ranges is the full pair list.  *out is sorted by (i,j).            */
int ygpu_pairwise_flag(ygpu_ctx* ctx, double threshold, uint32_t row_begin, uint32_t row_end,
                       ygpu_pair** out, uint64_t* n_out);
/* Same computation, but the sorted pair list stays on the device; ygpu_pairs_copy() then copies
 * n_out * sizeof(ygpu_pair) bytes to a host (dst_is_device = 0) or device (1) buffer -- the
 * multi-GPU gather hands NCCL the device copy.                                                   */
int ygpu_pairwise_flag_device(ygpu_ctx* ctx, double threshold, uint32_t row_begin, uint32_t row_end, uint64_t* n_out);
int ygpu_pairs_copy(ygpu_ctx* ctx, void* dst, int dst_is_device);
/* Host-side (sequential, milliseconds): the greedy selection of main.cpp:371-420 over the flagged pairs of the whole
 * database (sorted by (i, j) as ygpu_pairwise_flag returns them).  offsets: the CSR offsets the sketches were loaded
 * with (sketch sizes).  selected[0..*n_selected) = retained genome ids in the reference's visit order (ascending
 * sketch size, ties as the reference's std::sort leaves them); `selected` must hold n entries.                    */
int ygpu_greedy_select(const uint64_t* offsets, uint32_t n_genomes, const ygpu_pair* pairs, uint64_t n_pairs,
                       int32_t* selected, uint32_t* n_selected);
/* bounds[0..nparts] : contiguous row ranges of (nearly) equal pairwise-count work.               */
int ygpu_row_partition(ygpu_ctx* ctx, uint32_t nparts, uint32_t* bounds);

/* ---- sharded train step: one rank per GPU (threads of one process or one process per GPU, one node) ---------
 * The reference's only parallelism is its contiguous row chunks per thread / pass over ONE shared index
 * (main.cpp:338-349).  Across GPUs every rank holds the sketches of its own genome range only; the index build is
 * split by hash range and exchanged by the kernels themselves (stores into the peers' buffers over NVLink), the
 * pairwise count by query rows; NCCL (loaded on demand) carries the control data and the final pair lists.
 *   rank 0:      ygpu_comm_get_unique_id(id)  -> hand `id` to every rank (any transport)
 *   every rank:  ygpu_comm_init(ctx, rank, nranks, id)                              collective
 *                ygpu_load_sketches_sharded(ctx, my hashes, ALL offsets, n, g_begin, g_end)   collective
 *                ygpu_train_step_sharded(ctx, threshold, &stats, &n_pairs)          collective; then on every rank
 *                ygpu_pairs_copy(ctx, dst, 0)   copies the COMPLETE pair list (all ranks' rows), sorted by (i, j)
 * The genome ranges must be contiguous, in rank order, and cover [0, n).  Databases whose buckets outgrow shared
 * memory (extreme skew) are refused with YGPU_ERR_STATE: use the replicated ygpu_build_index + row ranges.      */
#define YGPU_COMM_ID_BYTES 128
int ygpu_comm_get_unique_id(uint8_t* id /* [YGPU_COMM_ID_BYTES] */);
int ygpu_comm_init(ygpu_ctx* ctx, int rank, int nranks, const uint8_t* id);
int ygpu_comm_destroy(ygpu_ctx* ctx);
int ygpu_load_sketches_sharded(ygpu_ctx* ctx, const uint64_t* hashes_slice, const uint64_t* offsets, uint32_t n_genomes,
                               uint32_t g_begin, uint32_t g_end);
/* same, the slice already on ctx's device (offsets stay a HOST pointer) */
int ygpu_load_sketches_sharded_device(ygpu_ctx* ctx, const uint64_t* d_hashes_slice, const uint64_t* offsets, uint32_t n_genomes,
                                      uint32_t g_begin, uint32_t g_end);
/* streaming ingest (ygpu_upload_begin / _block) into a sharded residency: only the blocks of genomes [g_begin, g_end)
 * were uploaded to this rank; block_dst[id] is relative to the first hash of genome g_begin                       */
int ygpu_upload_finish_sharded(ygpu_ctx* ctx, const uint64_t* block_dst, uint32_t nblocks, const uint64_t* offsets, uint32_t n_genomes,
                               uint32_t g_begin, uint32_t g_end);
/* Hash-range residency (the faster of the two): this rank holds, of EVERY sketch, the hashes inside its hash range -- the
 * host cuts every (sorted) sketch at the same nranks - 1 hash values, so a rank's share of a sketch is one contiguous
 * piece of it.  part_offsets[n + 1]: CSR over this rank's share; sizes[n]: the FULL sketch sizes (the containment
 * denominators); [row_begin, row_end): the query rows this rank counts (contiguous, in rank order, covering [0, n)).
 * Equal hashes meet on one rank by construction, so ygpu_train_step_sharded exchanges nothing but work items.
 * The caller guarantees that the ranks' hash ranges are disjoint.                                                     */
int ygpu_load_sketches_hashrange(ygpu_ctx* ctx, const uint64_t* part_hashes, const uint64_t* part_offsets, const uint32_t* sizes,
                                 uint32_t n_genomes, uint32_t row_begin, uint32_t row_end);
int ygpu_load_sketches_hashrange_device(ygpu_ctx* ctx, const uint64_t* d_part_hashes, const uint64_t* part_offsets, const uint32_t* sizes,
                                        uint32_t n_genomes, uint32_t row_begin, uint32_t row_end);
int ygpu_train_step_sharded(ygpu_ctx* ctx, double threshold, ygpu_index_stats* stats /* may be NULL */, uint64_t* n_pairs_total);

/* Replicated index, rows split by measured work (north_star's starting layout; the multi-GPU route for databases the
 * sharded step refuses): every rank holds ALL sketches (ygpu_load_sketches) and builds the full index, rank r counts the
 * rows of its work-balanced range, the pair lists are gathered.  Collective; afterwards ygpu_pairs_copy as above.    */
int ygpu_train_step_replicated(ygpu_ctx* ctx, double threshold, ygpu_index_stats* stats /* may be NULL */, uint64_t* n_pairs_total);

/* ---- run path ------------------------------------------------------------------------------ */
/* sample: HOST pointer to the sample sketch hashes (any order).  Fills counts[n_genomes].
 * Step 1 (multisearch -t 0): n_overlap.  Step 2 (get_exclusive_hashes): among the genomes with
 * n_overlap > 0 (or, if `mask` is not NULL, the genomes with mask[g] != 0), the number of hashes
 * exclusive to each genome and how many of those are in the sample.                              */
int ygpu_exclusive_hashes(ygpu_ctx* ctx, const uint64_t* sample, uint64_t n_sample,
                          const uint8_t* mask /* may be NULL */, ygpu_genome_counts* counts);
/* rows[c * n + r] = single_hyp_test((n_exclusive[r], n_match[r]), ksize, significance, ani, cov[c]) */
/* out[r] = get_alt_mut_rate(nu[r], thresh[r], ksize, significance)  (hypothesis_recovery_src.py:209-230),
 * -1.0 where scipy's betaincinv returns NaN.                                                      */
int ygpu_alt_mut_rate(ygpu_ctx* ctx, const int64_t* nu, const int64_t* thresh, uint64_t n, int ksize,
                      double significance, double* out);
int ygpu_hyp_test(ygpu_ctx* ctx, const int64_t* n_exclusive, const int64_t* n_match, uint64_t n,
                  int ksize, double significance, double ani_thresh, const double* min_coverage,
                  int n_cov, ygpu_hyp_row* rows);

/* ---- sketching (SURVEY 8 row f-4) --------------------------------------------------------------- */
/* What the reference delegates to `sourmash sketch dna -p k=K,scaled=S,abund` (src/yacht/sketch_ref_genomes.py:25,61;
 * src/yacht/sketch_sample.py:32,49): FracMinHash sketches of DNA sequences.
 * bases: HOST pointer, the records one after another, any case; whatever is not A/C/G/T (N, IUPAC codes, the separator
 * byte the caller puts between two records -- '\n' will do) invalidates the windows that contain it.  Sketch s is made
 * from bases[sketch_offsets[s] .. sketch_offsets[s+1]) (a window must lie inside one sketch's range).  Every window of
 * `ksize` valid bases -> canonical k-mer (the smaller of the window and its reverse complement) -> first 64 bits of
 * MurmurHash3_x64_128(k-mer, seed) -> kept when <= max_hash.  seed = 42 and max_hash = round((2^64 - 1) / scaled)
 * (18446744073709552 at scaled = 1000) give sourmash's "0.murmur64" sketches.
 * out: per sketch the distinct kept hashes, ascending (= "mins"), and how often each occurred (= "abundances");
 * library-owned, release with ygpu_sketch_result_free.                                                               */
typedef struct {
    uint64_t* hashes;       /* [offsets[n_sketches]]                                            */
    uint32_t* abundances;   /* [offsets[n_sketches]]                                            */
    uint64_t* offsets;      /* [n_sketches + 1]                                                 */
    uint32_t n_sketches;
    uint32_t _pad;
    uint64_t n_kmers;       /* valid windows hashed                                             */
} ygpu_sketch_result;
int ygpu_sketch_sequences(ygpu_ctx* ctx, const uint8_t* bases, uint64_t n_bases, const uint64_t* sketch_offsets,
                          uint32_t n_sketches, int ksize, uint64_t max_hash, uint32_t seed, ygpu_sketch_result* out);
/* Several k-mer sizes of one batch: 1 to 8 distinct sizes in [1, 256] (otherwise YGPU_ERR_ARG, as ygpu_stream_begin_k).
 * The batch is copied to the device once and every size is hashed and ordered on that copy; out[0 .. n_k), in the order
 * of ksizes, each exactly what ygpu_sketch_sequences returns for that size alone (n_kmers included).  ms_h2d times the
 * one copy, ms_sketch the sum of the sizes' hashing kernels.  ygpu_sketch_sequences is the n_k = 1 case.           */
int ygpu_sketch_sequences_k(ygpu_ctx* ctx, const uint8_t* bases, uint64_t n_bases, const uint64_t* sketch_offsets,
                            uint32_t n_sketches, const int* ksizes, int n_k, uint64_t max_hash, uint32_t seed,
                            ygpu_sketch_result* out /* [n_k], order of ksizes */);
void ygpu_sketch_result_free(ygpu_sketch_result* r);

/* Streamed sketching of FASTA / FASTQ text of any size.  The raw (decompressed) text goes to the device in chunks of
 * "stream_chunk_bytes" (ygpu_set_option; default 64 MiB); the device parses it, hashes it with the kernels of
 * ygpu_sketch_sequences and adds the result to a sketch kept on the device.  Host memory stays at a few chunks plus
 * the output.  The parse follows the records of a whole-file read exactly: '\r' is dropped everywhere, leading
 * whitespace of a file is skipped and the next byte chooses FASTA ('>') or FASTQ ('@'); a FASTA record's inner line
 * ends vanish; a FASTQ record is four lines, '@' name, sequence, '+', quality.
 *   ygpu_stream_begin(ctx, ksize, max_hash, seed, mode)   mode YGPU_STREAM_WHOLE: one sketch of everything fed;
 *                                                         YGPU_STREAM_PER_RECORD: one sketch per record, with names
 *   ygpu_stream_feed(ctx, bytes, n)      the next bytes of the current file, split anywhere.  HOST pointer, free to
 *                                        reuse when the call returns (page-locked memory from ygpu_host_alloc copies
 *                                        fastest); reading the next piece on another thread overlaps the device work
 *   ygpu_stream_end_file(ctx)            end of the current file and its checks; the next feed starts a new file
 *   ygpu_stream_finish(ctx, &result, &stats, &names, &name_offsets, &n_names)
 * Several k-mer sizes in one pass: ygpu_stream_begin_k(ctx, ksizes, n_k, ...) takes 1 to 8 distinct sizes in [1, 256]
 * (otherwise YGPU_ERR_ARG); the text is parsed once and every size is hashed on it.  ygpu_stream_finish_k fills
 * result[0 .. n_k), in the order of ksizes, each exactly the result of a stream begun with that size alone (n_kmers: that
 * size's valid windows); stats.n_kmers is their sum, ms_hash covers every size's kernel, the names are shared.  Per-record
 * mode needs records x n_k < 2^32.  ygpu_stream_begin / _finish are the n_k = 1 case; ygpu_stream_finish refuses a stream
 * of several sizes.
 * Malformed input fails with YGPU_ERR_ARG and one of "neither FASTA ('>') nor FASTQ ('@')", "malformed FASTQ record at
 * line N", "FASTQ with N lines (not a multiple of 4)" (lines counted from the first byte after the leading whitespace);
 * the stream must then be begun again.  Names (the header line without its first byte and without '\r') are kept for
 * every record in per-record mode and for FASTA records in whole mode; names[name_offsets[i] .. name_offsets[i + 1])
 * is name i; both arrays are library-owned, release them with ygpu_free (NULL when there are none).               */
#define YGPU_STREAM_WHOLE 0
#define YGPU_STREAM_PER_RECORD 1
typedef struct {
    uint64_t n_bytes;       /* bytes fed, leading whitespace of the files excluded                  */
    uint64_t n_bases;       /* bytes handed to the hashing kernels (sequence + one separator per record + carried bases) */
    uint64_t n_records;
    uint64_t n_kmers;       /* valid windows hashed                                                 */
    uint64_t n_chunks;      /* device chunks parsed                                                 */
    double ms_h2d;          /* host -> device copies of the raw text                                */
    double ms_parse;        /* line scan, classification, compaction                                */
    double ms_hash;         /* the K7 hashing kernel; with several k-mer sizes every size's kernel, and the packing of
                               each size's kept hashes but the last one's                                                  */
    double ms_merge;        /* sort + reduce of each chunk's kept hashes into the resident sketch   */
} ygpu_stream_stats;
int ygpu_stream_begin(ygpu_ctx* ctx, int ksize, uint64_t max_hash, uint32_t seed, int mode);
int ygpu_stream_feed(ygpu_ctx* ctx, const uint8_t* bytes, uint64_t n);
int ygpu_stream_end_file(ygpu_ctx* ctx);
int ygpu_stream_finish(ygpu_ctx* ctx, ygpu_sketch_result* out, ygpu_stream_stats* stats /* may be NULL */,
                       char** names, uint64_t** name_offsets, uint64_t* n_names);
int ygpu_stream_begin_k(ygpu_ctx* ctx, const int* ksizes, int n_k, uint64_t max_hash, uint32_t seed, int mode);
int ygpu_stream_finish_k(ygpu_ctx* ctx, ygpu_sketch_result* out /* [n_k], order of ksizes */, ygpu_stream_stats* stats /* may be NULL */,
                         char** names, uint64_t** name_offsets, uint64_t* n_names);

#ifdef __cplusplus
}
#endif
#endif /* YACHT_GPU_H */
