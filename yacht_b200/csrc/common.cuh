// Shared declarations of libyachtgpu (internal; the public boundary is include/yacht_gpu.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <unordered_map>
#include <algorithm>
#include "../../include/yacht_gpu.h"

struct ygpu_comm;
#define YG_MAX_RANKS 16

struct ygpu_ctx {
    int device = 0;
    int num_sms = 148;
    int smem_optin = 0;          // max dynamic shared memory per CTA (opt-in), bytes
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8] = {};
    cudaEvent_t evp[16] = {};     // per-kernel events of the partition path / the sharded step
    std::string err;

    // ---- sketches (flat, device resident) ---------------------------------------------------
    uint32_t n = 0;              // genomes
    uint64_t T = 0;              // total hashes
    uint64_t* d_hashes = nullptr;   // [T]   sketch hashes, genome-major (as loaded)
    uint64_t* d_offsets = nullptr;  // [n+1]
    uint32_t* d_sizes = nullptr;    // [n]   sketch sizes
    uint32_t* d_gid = nullptr;      // [T]   genome id of every hash slot
    bool loaded = false;
    bool maxkey_valid = false;      // largest resident hash: a property of the loaded sketches, computed once per load
    uint64_t maxkey = 0;

    // ---- inverted index (K2 output) ---------------------------------------------------------
    bool indexed = false;
    bool sorted = false;            // d_skey / d_sgid valid
    uint64_t* d_skey = nullptr;     // [T]   hashes sorted ascending
    uint32_t* d_sgid = nullptr;     // [T]   genome id of each sorted hash (ascending inside a run)
    uint8_t* d_flag = nullptr;      // [T]   1 if the sorted slot belongs to a run of length >= 2
    uint32_t* d_cpos = nullptr;     // [T]   exclusive scan of d_flag (slot in the compacted postings)
    uint64_t P = 0;                 // postings kept
    uint32_t* d_post = nullptr;     // [P]   compacted posting array (genome ids), runs contiguous (partition path: indexed by
                                    //       position in the final buffer, + the words of oversized buckets behind it)
    uint32_t* d_rem = nullptr;      // [P]   postings that follow slot c inside its run
    uint64_t n_items = 0;
    uint64_t* d_row_ptr = nullptr;  // [n+1] CSR over row_items (general path)
    const uint64_t* d_row_begin = nullptr;  // [n] start of row g's work list in d_row_items (d_row_ptr or d_offsets)
    uint64_t* d_row_items = nullptr;// [n_items] (first posting slot << 32) | count  -- per query genome
    uint64_t* d_row_work = nullptr; // [n]   increments row i performs (sum of counts); filled on demand
    bool row_work_valid = false;
    unsigned long long* d_row_cnt = nullptr;  // [n+1] build scratch
    // MSD-partition build (index_msd.cu)
    uint64_t* d_ent1 = nullptr;     // [max(T, slots x capacity)] packed (hash low bits | genome id) words, level-1 buckets
    uint64_t* d_ent2 = nullptr;     // [max(T, slots x capacity)] same, final buckets ([T] on the exact layout)
    uint32_t* d_msd_aux = nullptr;  // histograms / bases / cursors
    uint32_t* d_units = nullptr;    // level-2 tile descriptors (uint2 per tile)
    uint32_t* d_tile_g0 = nullptr;  // genome holding the first hash slot of every level-1 tile
    int group_ctas = 4;             // test hook: CTAs per SM the grouping kernel k2_group2 is compiled for (4 or 5; measured at 85k genomes on 1 x B200: 3.72 ms vs 4.21 ms, profiles/r03b_ab_group.txt)
    int group_kernel = 0;           // test hook: 1 = always the general grouping kernel k2_group (0: k2_group2 where it applies)
    // final buckets too large for shared memory (k2_big_*): their list, compact starts, gathered / sorted words
    uint32_t* d_big_list = nullptr;
    uint64_t* d_big_cstart = nullptr;
    uint64_t* d_big_a = nullptr;
    uint64_t* d_big_b = nullptr;
    int big_buckets = 1;            // option: 0 = any oversized bucket sends the whole database to the general path
    uint32_t msd_big_buckets = 0;   // oversized buckets of the last build
    int last_group2_grid = 0;       // grids of the last build's k2_group2 and k2_group launches, chunks of its oversized route (0: did not run)
    int last_group_grid = 0;
    uint32_t last_big_chunks = 0;
    uint16_t* d_st_rem = nullptr;   // [T] group stream of a hash-range sharded build: members of the same group that follow
    int index_path = 1;             // 1: MSD partition when the input qualifies, 0: always the general sort path
    int msd_fallbacks = 0;
    int last_index_path = 0;        // which path built the current index
    int count_kernel = 0;           // 0: automatic, 1: dense row accumulator per CTA, 2: one warp per row (hash table)
    int last_count_kernel = 0;
    unsigned long long last_count_overflow_rows = 0;
    uint32_t last_count_tile_w = 0; // accumulator geometry of the last dense count launch: columns per tile, tiles, packed u16
    uint32_t last_count_n_tiles = 0;
    int last_count_u16 = 0;
    uint32_t* d_ovf_rows = nullptr; // rows the warp kernel deferred to the dense kernel
    uint32_t* d_tc = nullptr;       // [n] smallest shared-hash count that passes the containment test of genome g
    bool skip_pair_sort = false;    // sharded step: the pair lists of all ranks are ordered once, after the gather
    int count_thresholds = 1;       // test hook: 0 = evaluate the fp64 expression per pair inside the count kernel
    ygpu_index_stats stats = {};

    // ---- scratch ------------------------------------------------------------------------------
    std::unordered_map<void*, size_t> caps;   // capacity (bytes) of every dev_alloc'ed buffer, keyed by member address
    void* d_temp = nullptr;         // CUB temp storage (grown on demand)
    size_t temp_bytes = 0;
    unsigned long long* d_scalars = nullptr;  // [16] device counters
    uint64_t* d_out_key = nullptr;  // pair compaction buffers
    uint32_t* d_out_cnt = nullptr;
    uint64_t* d_out_key2 = nullptr;
    uint32_t* d_out_cnt2 = nullptr;
    uint64_t out_cap = 0;
    ygpu_pair* d_pairs = nullptr;   // sorted flagged pairs of the last pairwise call
    uint64_t pairs_cap = 0;
    uint64_t n_pairs = 0;
    uint32_t force_tile_w = 0;      // test hook: cap the accumulator tile width (0 = automatic)
    int force_u16 = 0;              // test hook: packed 16-bit counters even when 32-bit ones fit

    // ---- sharded residency + multi-GPU train step (comm.cu, index_msd.cu: ygpu_train_step_sharded) ----------------
    ygpu_comm* comm = nullptr;
    bool sharded = false;           // this context holds only a share of the sketches (rank of a communicator)
    int shard_mode = 0;             // 0: the sketches of genomes [g_begin, g_end); 1: of EVERY sketch the hashes of this rank's hash range
    uint64_t sh_cap_req = 0;        // mode 1: largest share over the ranks (sizes the exchange buffers)
    unsigned long long* d_sh_flags = nullptr;
    uint32_t g_begin = 0, g_end = 0;
    uint64_t T_global = 0;
    uint32_t max_sketch_global = 0;
    uint64_t* d_offsets_local = nullptr;    // [g_end - g_begin + 1] offsets relative to the resident slice
    uint64_t* d_row_begin_local = nullptr;  // [n] start of row g's work list in d_row_items (rows of the slice only)
    uint64_t sh_cap = 0;            // per-rank capacity (words / stream entries) of the exchange buffers
    uint32_t* d_sh_hist_all = nullptr;      // [nranks][NB_MAX] level-1 histograms of every rank's slice
    uint32_t* d_sh_owner = nullptr;         // [NB_MAX] owner rank of every level-1 digit
    unsigned long long* d_sh_info = nullptr;// small device block: digit range, word count, stream lengths ...
    void* sh_peer_ent1[YG_MAX_RANKS] = {};  // peers' level-1 exchange buffers (d_ent1)
    void* sh_peer_gid[YG_MAX_RANKS] = {};   // peers' group-stream buffers (d_post / d_st_rem)
    void* sh_peer_rem[YG_MAX_RANKS] = {};
    void* sh_peer_item[YG_MAX_RANKS] = {};  // peers' item inboxes (d_inbox_item / d_inbox_row)
    void* sh_peer_row[YG_MAX_RANKS] = {};
    uint64_t* d_inbox_item = nullptr;       // [nranks][sh_cap] ready-made work items for this rank's rows, one region per sending rank
    uint32_t* d_inbox_row = nullptr;        // ... and their query rows
    void* sh_shared_item = nullptr;
    void* sh_shared_row = nullptr;
    uint32_t sh_row_bounds[YG_MAX_RANKS + 1] = {};   // rank q holds / counts the genomes [sh_row_bounds[q], sh_row_bounds[q + 1])
    uint64_t row_items_cap = 0, row_items_need = 0;
    void* sh_shared_ent1 = nullptr;         // which allocations the peer pointers above refer to (re-shared when they move)
    void* sh_shared_gid = nullptr;
    void* sh_shared_rem = nullptr;
    ygpu_pair* d_pairs_local = nullptr;     // this rank's pairs before the gather
    uint64_t pairs_local_cap = 0;

    void* part_state = nullptr;     // the MSD partition of the resident sketches (index_msd.cu: MsdPartState), reused by the run path
    bool part_valid = false;
    void* run_part_scratch = nullptr;   // sample buckets / nontrivial bitmap of the partition-probe run path
    int run_path = 1;               // 1: partition-probe run path when the database qualifies, 0: always the general sort-based one
    int last_run_path = 0;

    void* run_scratch = nullptr;    // run-path buffers (run_kernels.cu)
    void* upload = nullptr;         // streaming ingest state (yacht_gpu.cu: ygpu_upload_*)
    void* sketch_scratch = nullptr; // sketching buffers (sketch.cu)
    int sketch_kernel = 0;          // 0 = by k-mer size (packed words up to k = 64), 2 = always the byte-wise kernel (test hook)
    void* seq_stream = nullptr;     // streamed FASTA / FASTQ sketching (seq_stream.cu)
    uint64_t stream_chunk_bytes = 64ull << 20;   // raw bytes the stream parses per device chunk

    ygpu_timings tm = {};
};

int ygpu_fail(ygpu_ctx* ctx, int code, const char* fmt, ...);

#define YG_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return ygpu_fail((ctx), YGPU_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,     \
                             cudaGetErrorString(e__));                                            \
    } while (0)

#define YG_CHECK(expr)                 \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != 0) return rc__;    \
    } while (0)

int ygpu_temp_reserve(ygpu_ctx* ctx, size_t bytes);

// Capacity-tracked device buffers: a buffer is reused when it is already large enough, so that
// repeated steps (bench loops, multi-sample runs) do not pay cudaMalloc/cudaFree -- which
// synchronise the device and cost milliseconds per GB -- inside the hot path.
template <typename T>
static inline int dev_alloc(ygpu_ctx* ctx, T** p, uint64_t count) {
    if (count == 0) count = 1;
    const size_t bytes = count * sizeof(T);
    auto it = ctx->caps.find((void*)p);
    if (*p && it != ctx->caps.end() && it->second >= bytes) return 0;
    if (*p) { cudaFree(*p); *p = nullptr; }
    const size_t want = bytes + (bytes >> 4) + 256;
    cudaError_t e = cudaMalloc((void**)p, want);
    if (e != cudaSuccess) {
        *p = nullptr;
        ctx->caps.erase((void*)p);
        return ygpu_fail(ctx, YGPU_ERR_NOMEM, "cudaMalloc(%llu bytes): %s", (unsigned long long)want, cudaGetErrorString(e));
    }
    ctx->caps[(void*)p] = want;
    return 0;
}
// dev_alloc that keeps the first `keep` elements: a buffer too small for `count` is replaced by a larger one and the kept
// elements are copied over on `st` before the old buffer is freed (cudaFree waits for the copy).
template <typename T>
static inline int dev_grow_keep(ygpu_ctx* ctx, T** p, uint64_t count, uint64_t keep, cudaStream_t st) {
    auto it = ctx->caps.find((void*)p);
    if (!keep || !*p || it == ctx->caps.end() || it->second >= std::max<uint64_t>(count, 1) * sizeof(T)) return dev_alloc(ctx, p, count);
    T* old = *p;
    const size_t old_cap = it->second;
    *p = nullptr;                                   // dev_alloc makes a new buffer and leaves the old one alone
    ctx->caps.erase((void*)p);
    const int rc = dev_alloc(ctx, p, count);
    if (rc) {
        *p = old;
        ctx->caps[(void*)p] = old_cap;
        return rc;
    }
    const cudaError_t e = cudaMemcpyAsync(*p, old, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
    cudaFree(old);
    if (e != cudaSuccess) return ygpu_fail(ctx, YGPU_ERR_CUDA, "dev_grow_keep: %s", cudaGetErrorString(e));
    return 0;
}
template <typename T>
static inline void dev_free(ygpu_ctx* ctx, T** p) {
    if (*p) cudaFree(*p);
    *p = nullptr;
    ctx->caps.erase((void*)p);
}

static inline float elapsed(ygpu_ctx* ctx, int a, int b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]);
    return ms;
}

// ---- work item format v2 (one 64-bit word per (query genome, shared hash)) ------------------------
//   low 2 bits c = 0 : indirect -- the (item >> 2) & 0x3FFFFFFF postings starting at d_post[item >> 32] follow me
//   low 2 bits c = 1..3 : inline -- the c genome ids that follow me are in bits [21:2], [41:22], [61:42]
//                        (20 bits each: used only while genome ids fit 20 bits)
#define YG_ITEM_INLINE_BITS 20

// device scalar slots (ctx->d_scalars)
enum { SC_HEADS = 0, SC_SINGLE = 1, SC_DUPS = 2, SC_W = 3, SC_OUT = 4, SC_UNIT = 5, SC_MAXKEY = 6, SC_OVF = 7 };

template <int BS>
__device__ __forceinline__ unsigned long long block_sum(unsigned long long v) {
    __shared__ unsigned long long sh[BS / 32];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    v = 0;
    if (w == 0) {
        v = (l < BS / 32) ? sh[l] : 0ull;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    return v;  // valid in thread 0
}

static inline int grid_for(ygpu_ctx* ctx, uint64_t work, int bs, int per_sm = 8) {
    uint64_t blocks = (work + bs - 1) / bs;
    uint64_t cap = (uint64_t)ctx->num_sms * per_sm;
    return (int)std::max<uint64_t>(1, std::min(blocks, cap));
}


int ygpu_sort_sketches(ygpu_ctx* ctx);   // K2a (yacht_gpu.cu)
int ygpu_max_hash(ygpu_ctx* ctx, uint64_t* maxkey);   // largest resident hash (cached per load)
// MSD-partition index build (index_msd.cu): *used = 0 when the input does not qualify for it
int ygpu_build_index_msd(ygpu_ctx* ctx, ygpu_index_stats* S, int* used);

// run path on the partitioned reference (index_msd.cu): *used = 0 when the database / sample does not qualify
int ygpu_run_counts_buckets(ygpu_ctx* ctx, const uint64_t* d_sample, uint64_t n_sample, const uint8_t* d_mask, ygpu_genome_counts* d_counts, int* used);
void ygpu_part_release(ygpu_ctx* ctx);
// run path (run_kernels.cu)
void ygpu_run_release(ygpu_ctx* ctx);
// sketching (sketch.cu)
void ygpu_sketch_release(ygpu_ctx* ctx);
void ygpu_stream_release(ygpu_ctx* ctx);
// K7 on a device buffer (d_bases zero-padded by YG_SKETCH_PAD bytes behind n_bases); survivors stay in the sketch scratch
constexpr uint64_t YG_SKETCH_PAD = 4096 + 256 + 16;
constexpr uint64_t YG_STREAM_CHUNK_MAX = 1ull << 30;
int ygpu_sketch_hash_device(ygpu_ctx* ctx, const uint8_t* d_bases, uint64_t n_bases, uint64_t* d_off, uint32_t n_sketches,
                            int ksize, uint64_t max_hash, uint32_t seed, uint64_t first_new, cudaEvent_t ev_done, uint64_t* m,
                            uint64_t* n_kmers);
void ygpu_sketch_survivors(ygpu_ctx* ctx, uint64_t** d_key, uint32_t** d_sid);
void ygpu_upload_release(ygpu_ctx* ctx);
