// libyachtgpu -- FracMinHash sketching on the device (SURVEY 8 row f-4).
//
// Replaces what the reference delegates to `sourmash sketch dna -p k=K,scaled=S,abund` (src/yacht/sketch_ref_genomes.py:25,61,
// src/yacht/sketch_sample.py:32,49): every window of K valid bases of every record -> canonical k-mer -> murmur64(seed) ->
// kept when <= max_hash; per sketch the distinct kept hashes, ascending, with their abundances.
//
//   k_sketch_hash_packed (k <= 32) : the same tile as 2-bit codes; windows are 64-bit words, canonical choice and ASCII
//                   expansion are word operations (ysk_canonical_hash_packed).  Three conflict-free loads per 16 windows.
//   k_sketch_hash_packed2 (33 <= k <= 64, YACHT's k = 51) : the same with two-word windows.
//   k_sketch_hash (any k <= 256) : one CTA per tile of 4 096 window starts.  The tile (+ K - 1 bytes) is brought into shared memory with
//                   16-byte loads and reduced to 2-bit codes on the way; a thread walks 16 consecutive starts with a rolling
//                   "valid bases so far" counter, so a window costs one code load for validity, ~1.3 compares for the
//                   canonical choice and the hash itself.  Integer-ALU bound (a few hundred instructions per window,
//                   1 byte of HBM per window).  Survivors (1 in `scaled`) are appended with their sketch id.
//   then          : device radix sorts (by hash, then stably by sketch id), k_sketch_heads / k_sketch_emit collapse equal
//                   neighbours into (hash, first index); the host turns index differences into abundances.
#include "common.cuh"
#include "sketch_hash.cuh"

#include <cub/cub.cuh>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace {

constexpr int SK_NT = 256;
constexpr int SK_PER = 16;                      // consecutive window starts per thread
constexpr int SK_TILE = SK_NT * SK_PER;         // 4096
constexpr int SK_KMAX = 256;                    // largest supported k-mer size
static_assert(SK_PER == 16 && SK_NT == 256, "the packed kernel's span layout (sketch_hash.cuh) assumes 16 windows per thread");
constexpr int SK_PAD = SK_TILE + SK_KMAX + 16;  // zero bytes behind the bases: the last tile is loaded without bounds checks
static_assert(SK_PAD == YG_SKETCH_PAD, "the stream pads its hashing buffer by YG_SKETCH_PAD");

struct SketchScratch {
    uint8_t* d_bases = nullptr;
    uint64_t* d_off = nullptr;
    uint64_t* d_key = nullptr;     // survivors: hash
    uint64_t* d_key2 = nullptr;
    uint32_t* d_sid = nullptr;     // survivors: sketch id
    uint32_t* d_sid2 = nullptr;
    uint32_t* d_flag = nullptr;
    uint32_t* d_pos = nullptr;
    uint64_t* d_out_h = nullptr;
    uint32_t* d_out_start = nullptr;
    uint32_t* d_out_sid = nullptr;
    unsigned long long* d_cnt = nullptr;   // [0] survivors, [1] valid k-mers
};

SketchScratch* sk_scratch(ygpu_ctx* ctx) {
    if (!ctx->sketch_scratch) ctx->sketch_scratch = new SketchScratch();
    return (SketchScratch*)ctx->sketch_scratch;
}

__global__ void __launch_bounds__(SK_NT) k_sketch_hash(const uint8_t* __restrict__ bases, uint64_t n_bases,
                                                       const uint64_t* __restrict__ sk_off, uint32_t n_sketches, int k, uint32_t seed,
                                                       uint64_t max_hash, uint64_t* __restrict__ out_key, uint32_t* __restrict__ out_sid,
                                                       uint64_t cap, unsigned long long* __restrict__ cnt) {
    __shared__ __align__(16) uint8_t sm[SK_TILE + SK_KMAX + 16];
    const int tid = threadIdx.x;
    const uint64_t n_tiles = (n_bases + SK_TILE - 1) / SK_TILE;
    unsigned long long valid_kmers = 0;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t base = tile * SK_TILE;
        __syncthreads();                                     // the previous tile's readers are done
        {   // 16 bytes per thread for the tile body, the first threads also fetch the K - 1 (rounded up) bytes behind it;
            // the allocation is padded with zero bytes (invalid), so no load needs a bounds check
            const uint4* g = (const uint4*)(bases + base);
            for (int v = tid; v < (SK_TILE + SK_KMAX) / 16; v += SK_NT) {
                if (v >= SK_TILE / 16 && (v - SK_TILE / 16) * 16 >= k - 1) break;
                uint4 w = g[v];
                uint32_t x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint32_t y = 0;
#pragma unroll
                    for (int b = 0; b < 4; b++) y |= (uint32_t)ysk_code((uint8_t)(x[q] >> (8 * b))) << (8 * b);
                    x[q] = y;
                }
                ((uint4*)sm)[v] = make_uint4(x[0], x[1], x[2], x[3]);
            }
        }
        __syncthreads();
        const int l0 = tid * SK_PER;
        int run = 0;                                         // valid bases ending just before the window's last base
        for (int j = 0; j < k - 1; j++) run = (sm[l0 + j] < 4) ? run + 1 : 0;
        for (int i = 0; i < SK_PER; i++) {
            const int l = l0 + i;
            run = (sm[l + k - 1] < 4) ? run + 1 : 0;
            const uint64_t p = base + l;
            if (run < k || p + (uint64_t)k > n_bases) continue;
            valid_kmers++;
            const uint64_t h = ysk_canonical_hash(sm + l, k, seed);
            if (h > max_hash) continue;
            // survivor (1 in `scaled`): which sketch does the window belong to?  It must lie inside it entirely.
            uint32_t lo = 0, hi = n_sketches;                // sk_off[lo] <= p < sk_off[hi]
            while (hi - lo > 1) {
                const uint32_t mid = (lo + hi) >> 1;
                if (sk_off[mid] <= p) lo = mid; else hi = mid;
            }
            if (p < sk_off[lo] || p + (uint64_t)k > sk_off[lo + 1]) continue;
            const unsigned long long slot = atomicAdd(&cnt[0], 1ull);
            if (slot < cap) { out_key[slot] = h; out_sid[slot] = lo; }
        }
    }
    // statistics: valid windows hashed by this CTA
    for (int o = 16; o > 0; o >>= 1) valid_kmers += __shfl_down_sync(0xffffffffu, valid_kmers, o);
    if ((tid & 31) == 0 && valid_kmers) atomicAdd(&cnt[1], valid_kmers);
}

// k <= 32: the tile lives in shared memory as 2-bit codes (16 bases per word) plus one "not A/C/G/T" bit per base.  A thread
// reads its 48-base span with three conflict-free word loads, a window is one funnel shift away, and canonical choice and
// ASCII expansion work on whole words (bit reversal, PRMT) -- see ysk_canonical_hash_packed.
__global__ void __launch_bounds__(SK_NT) k_sketch_hash_packed(const uint8_t* __restrict__ bases, uint64_t n_bases,
                                                              const uint64_t* __restrict__ sk_off, uint32_t n_sketches, int k, uint32_t seed,
                                                              uint64_t max_hash, uint64_t* __restrict__ out_key, uint32_t* __restrict__ out_sid,
                                                              uint64_t cap, unsigned long long* __restrict__ cnt) {
    __shared__ uint32_t s_code[SK_TILE / 16 + 2];            // + 32 bases behind the tile (k - 1 <= 31 are needed)
    __shared__ uint32_t s_bad[SK_TILE / 32 + 2];
    const int tid = threadIdx.x;
    const uint64_t n_tiles = (n_bases + SK_TILE - 1) / SK_TILE;
    unsigned long long valid_kmers = 0;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t base = tile * SK_TILE;
        const uint4* g = (const uint4*)(bases + base);       // 16-byte aligned; the allocation is zero-padded behind n_bases
        __syncthreads();                                     // the previous tile's readers are done
        {
            uint32_t code, bad;
            const uint4 v = g[tid];
            ysk_pack16(v.x, v.y, v.z, v.w, code, bad);
            s_code[tid] = code;
            const uint32_t up = __shfl_down_sync(0xffffffffu, bad, 1);
            if (!(tid & 1)) s_bad[tid >> 1] = bad | (up << 16);
            if (tid == 0) {                                  // the 32 bases behind the tile
                uint32_t c0, b0, c1, b1;
                const uint4 t0 = g[SK_TILE / 16], t1 = g[SK_TILE / 16 + 1];
                ysk_pack16(t0.x, t0.y, t0.z, t0.w, c0, b0);
                ysk_pack16(t1.x, t1.y, t1.z, t1.w, c1, b1);
                s_code[SK_TILE / 16] = c0;
                s_code[SK_TILE / 16 + 1] = c1;
                s_bad[SK_TILE / 32] = b0 | (b1 << 16);
            }
        }
        __syncthreads();
        uint64_t lo, hi, badbits;
        ysk_thread_span(s_code, s_bad, tid, lo, hi, badbits);
        const uint64_t p0 = base + (uint64_t)tid * SK_PER;
#pragma unroll 1
        for (int i = 0; i < SK_PER; i++) {
            const uint64_t p = p0 + i;
            uint64_t w;
            if (!ysk_span_window(lo, hi, badbits, i, k, w) || p + (uint64_t)k > n_bases) continue;
            valid_kmers++;
            const uint64_t h = ysk_canonical_hash_packed(w, k, seed);
            if (h > max_hash) continue;
            uint32_t a = 0, b = n_sketches;                  // sk_off[a] <= p < sk_off[b]
            while (b - a > 1) {
                const uint32_t mid = (a + b) >> 1;
                if (sk_off[mid] <= p) a = mid; else b = mid;
            }
            if (p < sk_off[a] || p + (uint64_t)k > sk_off[a + 1]) continue;
            const unsigned long long slot = atomicAdd(&cnt[0], 1ull);
            if (slot < cap) { out_key[slot] = h; out_sid[slot] = a; }
        }
    }
    for (int o = 16; o > 0; o >>= 1) valid_kmers += __shfl_down_sync(0xffffffffu, valid_kmers, o);
    if ((tid & 31) == 0 && valid_kmers) atomicAdd(&cnt[1], valid_kmers);
}

// 33 <= k <= 64 (YACHT's k = 51): the same layout, a window is two 64-bit words, the span of a thread 80 bases.
__global__ void __launch_bounds__(SK_NT) k_sketch_hash_packed2(const uint8_t* __restrict__ bases, uint64_t n_bases,
                                                               const uint64_t* __restrict__ sk_off, uint32_t n_sketches, int k, uint32_t seed,
                                                               uint64_t max_hash, uint64_t* __restrict__ out_key, uint32_t* __restrict__ out_sid,
                                                               uint64_t cap, unsigned long long* __restrict__ cnt) {
    __shared__ uint32_t s_code[SK_TILE / 16 + 4];            // + 64 bases behind the tile (k - 1 <= 63 are needed)
    __shared__ uint32_t s_bad[SK_TILE / 32 + 4];
    const int tid = threadIdx.x;
    const uint64_t n_tiles = (n_bases + SK_TILE - 1) / SK_TILE;
    unsigned long long valid_kmers = 0;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t base = tile * SK_TILE;
        const uint4* g = (const uint4*)(bases + base);
        __syncthreads();
        {
            uint32_t code, bad;
            const uint4 v = g[tid];
            ysk_pack16(v.x, v.y, v.z, v.w, code, bad);
            s_code[tid] = code;
            const uint32_t up = __shfl_down_sync(0xffffffffu, bad, 1);
            if (!(tid & 1)) s_bad[tid >> 1] = bad | (up << 16);
            if (tid < 2) {                                   // the 64 bases behind the tile: two threads, 32 bases each
                uint32_t c0, b0, c1, b1;
                const uint4 t0 = g[SK_TILE / 16 + 2 * tid], t1 = g[SK_TILE / 16 + 2 * tid + 1];
                ysk_pack16(t0.x, t0.y, t0.z, t0.w, c0, b0);
                ysk_pack16(t1.x, t1.y, t1.z, t1.w, c1, b1);
                s_code[SK_TILE / 16 + 2 * tid] = c0;
                s_code[SK_TILE / 16 + 2 * tid + 1] = c1;
                s_bad[SK_TILE / 32 + tid] = b0 | (b1 << 16);
                s_bad[SK_TILE / 32 + 2 + tid] = 0;           // read by the last threads' spans, never used
            }
        }
        __syncthreads();
        uint64_t s0, s1, s2, b0, b1;
        ysk_thread_span2(s_code, s_bad, tid, s0, s1, s2, b0, b1);
        const uint64_t p0 = base + (uint64_t)tid * SK_PER;
#pragma unroll 1
        for (int i = 0; i < SK_PER; i++) {
            const uint64_t p = p0 + i;
            uint64_t w0, w1;
            if (!ysk_span_window2(s0, s1, s2, b0, b1, i, k, w0, w1) || p + (uint64_t)k > n_bases) continue;
            valid_kmers++;
            const uint64_t h = ysk_canonical_hash_packed2(w0, w1, k, seed);
            if (h > max_hash) continue;
            uint32_t a = 0, b = n_sketches;                  // sk_off[a] <= p < sk_off[b]
            while (b - a > 1) {
                const uint32_t mid = (a + b) >> 1;
                if (sk_off[mid] <= p) a = mid; else b = mid;
            }
            if (p < sk_off[a] || p + (uint64_t)k > sk_off[a + 1]) continue;
            const unsigned long long slot = atomicAdd(&cnt[0], 1ull);
            if (slot < cap) { out_key[slot] = h; out_sid[slot] = a; }
        }
    }
    for (int o = 16; o > 0; o >>= 1) valid_kmers += __shfl_down_sync(0xffffffffu, valid_kmers, o);
    if ((tid & 31) == 0 && valid_kmers) atomicAdd(&cnt[1], valid_kmers);
}

}  // namespace

// K7 on a device buffer: d_bases[0, n_bases) followed by SK_PAD zero bytes (16-byte aligned), d_off[0 .. n_sketches] on the
// device.  Leaves the m survivors in the context's scratch (sketch_survivors) and the valid windows in *n_kmers; records
// ev_done behind the hashing kernel.  ygpu_sketch_sequences and the stream (seq_stream.cu) both hash through here.
int ygpu_sketch_hash_device(ygpu_ctx* ctx, const uint8_t* d_bases, uint64_t n_bases, const uint64_t* d_off, uint32_t n_sketches,
                            int ksize, uint64_t max_hash, uint32_t seed, cudaEvent_t ev_done, uint64_t* m, uint64_t* n_kmers) {
    SketchScratch* S = sk_scratch(ctx);
    cudaStream_t st = ctx->stream;
    YG_CHECK(dev_alloc(ctx, &S->d_cnt, 2));
    // Expected survivors: windows x (max_hash + 1) / 2^64.  Twice that plus slack; a second pass with the exact count
    // follows in the (never observed) case that it does not suffice.
    const double frac = ((double)max_hash + 1.0) / 18446744073709551616.0;
    uint64_t cap = (uint64_t)std::min<double>((double)n_bases, (double)n_bases * frac * 2.0 + 65536.0);
    unsigned long long h_cnt[2] = {0, 0};
    const uint64_t n_tiles = (n_bases + SK_TILE - 1) / SK_TILE;
    const int grid = (int)std::min<uint64_t>(n_tiles, (uint64_t)ctx->num_sms * 8);
    for (int attempt = 0; attempt < 2; attempt++) {
        if (cap >= (1ull << 31)) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_sketch_sequences: more than 2^31 kept hashes in one call; split the batch");
        YG_CHECK(dev_alloc(ctx, &S->d_key, cap));
        YG_CHECK(dev_alloc(ctx, &S->d_sid, cap));
        YG_CUDA(ctx, cudaMemsetAsync(S->d_cnt, 0, 2 * sizeof(unsigned long long), st));
        if (ksize <= 32 && ctx->sketch_kernel != 2)
            k_sketch_hash_packed<<<grid, SK_NT, 0, st>>>(d_bases, n_bases, d_off, n_sketches, ksize, seed, max_hash, S->d_key, S->d_sid, cap, S->d_cnt);
        else if (ksize <= 64 && ctx->sketch_kernel != 2)
            k_sketch_hash_packed2<<<grid, SK_NT, 0, st>>>(d_bases, n_bases, d_off, n_sketches, ksize, seed, max_hash, S->d_key, S->d_sid, cap, S->d_cnt);
        else
            k_sketch_hash<<<grid, SK_NT, 0, st>>>(d_bases, n_bases, d_off, n_sketches, ksize, seed, max_hash, S->d_key, S->d_sid, cap, S->d_cnt);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
        YG_CUDA(ctx, cudaEventRecord(ev_done, st));
        YG_CUDA(ctx, cudaMemcpyAsync(h_cnt, S->d_cnt, sizeof h_cnt, cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        if (h_cnt[0] <= cap) break;
        if (attempt == 1) return ygpu_fail(ctx, YGPU_ERR_STATE, "ygpu_sketch_sequences: survivor count changed between passes");
        cap = h_cnt[0];
    }
    *m = h_cnt[0];
    *n_kmers = h_cnt[1];
    return 0;
}

void ygpu_sketch_survivors(ygpu_ctx* ctx, uint64_t** d_key, uint32_t** d_sid) {
    SketchScratch* S = sk_scratch(ctx);
    *d_key = S->d_key;
    *d_sid = S->d_sid;
}

namespace {

__global__ void __launch_bounds__(256) k_sketch_heads(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sid, uint64_t m,
                                                       uint32_t* __restrict__ flag) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x)
        flag[i] = (i == 0 || key[i] != key[i - 1] || sid[i] != sid[i - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_sketch_emit(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sid,
                                                      const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos, uint64_t m,
                                                      uint64_t* __restrict__ out_h, uint32_t* __restrict__ out_start, uint32_t* __restrict__ out_sid) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        if (!flag[i]) continue;
        const uint32_t d = pos[i];
        out_h[d] = key[i];
        out_start[d] = (uint32_t)i;
        out_sid[d] = sid[i];
    }
}

}  // namespace

void ygpu_sketch_release(ygpu_ctx* ctx) {
    SketchScratch* s = (SketchScratch*)ctx->sketch_scratch;
    if (!s) return;
    dev_free(ctx, &s->d_bases); dev_free(ctx, &s->d_off); dev_free(ctx, &s->d_key); dev_free(ctx, &s->d_key2);
    dev_free(ctx, &s->d_sid); dev_free(ctx, &s->d_sid2); dev_free(ctx, &s->d_flag); dev_free(ctx, &s->d_pos);
    dev_free(ctx, &s->d_out_h); dev_free(ctx, &s->d_out_start); dev_free(ctx, &s->d_out_sid); dev_free(ctx, &s->d_cnt);
    delete s;
    ctx->sketch_scratch = nullptr;
}

extern "C" void ygpu_sketch_result_free(ygpu_sketch_result* r) {
    if (!r) return;
    free(r->hashes); free(r->abundances); free(r->offsets);
    memset(r, 0, sizeof *r);
}

extern "C" int ygpu_sketch_sequences(ygpu_ctx* ctx, const uint8_t* bases, uint64_t n_bases, const uint64_t* sketch_offsets,
                                     uint32_t n_sketches, int ksize, uint64_t max_hash, uint32_t seed, ygpu_sketch_result* out) {
    if (!ctx || !out || (!bases && n_bases) || !sketch_offsets || n_sketches == 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_sketch_sequences: bad argument");
    if (ksize < 1 || ksize > SK_KMAX) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_sketch_sequences: ksize %d outside [1, %d]", ksize, SK_KMAX);
    if (sketch_offsets[0] != 0 || sketch_offsets[n_sketches] != n_bases) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_sketch_sequences: sketch_offsets must run from 0 to n_bases");
    for (uint32_t s = 0; s < n_sketches; s++)
        if (sketch_offsets[s] > sketch_offsets[s + 1]) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_sketch_sequences: sketch_offsets must not decrease");
    memset(out, 0, sizeof *out);
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    SketchScratch* S = sk_scratch(ctx);
    cudaStream_t st = ctx->stream;

    out->offsets = (uint64_t*)calloc((size_t)n_sketches + 1, sizeof(uint64_t));
    if (!out->offsets) return ygpu_fail(ctx, YGPU_ERR_NOMEM, "out of host memory");
    out->n_sketches = n_sketches;
    if (n_bases < (uint64_t)ksize) return 0;                 // nothing to hash: n_sketches empty sketches

    YG_CHECK(dev_alloc(ctx, &S->d_bases, n_bases + SK_PAD));
    YG_CHECK(dev_alloc(ctx, &S->d_off, (uint64_t)n_sketches + 1));
    YG_CHECK(dev_alloc(ctx, &S->d_cnt, 2));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    YG_CUDA(ctx, cudaMemcpyAsync(S->d_bases, bases, n_bases, cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaMemsetAsync(S->d_bases + n_bases, 0, SK_PAD, st));
    YG_CUDA(ctx, cudaMemcpyAsync(S->d_off, sketch_offsets, ((size_t)n_sketches + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));

    uint64_t m = 0, n_kmers = 0;
    YG_CHECK(ygpu_sketch_hash_device(ctx, S->d_bases, n_bases, S->d_off, n_sketches, ksize, max_hash, seed, ctx->ev[2], &m, &n_kmers));
    ctx->tm.ms_h2d = elapsed(ctx, 0, 1);
    ctx->tm.ms_sketch = elapsed(ctx, 1, 2);
    out->n_kmers = n_kmers;
    if (m == 0) return 0;

    // order by (sketch id, hash): LSD radix sort by hash, then -- stable -- by sketch id
    YG_CHECK(dev_alloc(ctx, &S->d_key2, m));
    YG_CHECK(dev_alloc(ctx, &S->d_sid2, m));
    int hash_bits = 64;
    while (hash_bits > 1 && !((max_hash >> (hash_bits - 1)) & 1)) hash_bits--;
    int sid_bits = 1;
    while (sid_bits < 32 && (1ull << sid_bits) < (uint64_t)n_sketches) sid_bits++;
    size_t tb1 = 0, tb2 = 0, tb3 = 0;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb1, S->d_key, S->d_key2, S->d_sid, S->d_sid2, (int64_t)m, 0, hash_bits, st));
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb2, S->d_sid2, S->d_sid, S->d_key2, S->d_key, (int64_t)m, 0, sid_bits, st));
    YG_CHECK(dev_alloc(ctx, &S->d_flag, m));
    YG_CHECK(dev_alloc(ctx, &S->d_pos, m));
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb3, S->d_flag, S->d_pos, (int64_t)m, st));
    YG_CHECK(ygpu_temp_reserve(ctx, std::max(tb1, std::max(tb2, tb3))));
    size_t tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, S->d_key, S->d_key2, S->d_sid, S->d_sid2, (int64_t)m, 0, hash_bits, st));
    const uint64_t* d_key = S->d_key2;
    const uint32_t* d_sid = S->d_sid2;
    ctx->tm.n_library_launches += 3;
    if (n_sketches > 1) {
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, S->d_sid2, S->d_sid, S->d_key2, S->d_key, (int64_t)m, 0, sid_bits, st));
        d_key = S->d_key;
        d_sid = S->d_sid;
        ctx->tm.n_library_launches += 3;
    }
    const int g2 = grid_for(ctx, m, 256);
    k_sketch_heads<<<g2, 256, 0, st>>>(d_key, d_sid, m, S->d_flag);
    YG_CUDA(ctx, cudaGetLastError());
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, S->d_flag, S->d_pos, (int64_t)m, st));
    ctx->tm.n_library_launches += 2;
    YG_CHECK(dev_alloc(ctx, &S->d_out_h, m));
    YG_CHECK(dev_alloc(ctx, &S->d_out_start, m + 1));
    YG_CHECK(dev_alloc(ctx, &S->d_out_sid, m));
    k_sketch_emit<<<g2, 256, 0, st>>>(d_key, d_sid, S->d_flag, S->d_pos, m, S->d_out_h, S->d_out_start, S->d_out_sid);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches += 2;
    uint32_t last_pos = 0, last_flag = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(&last_pos, S->d_pos + (m - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(&last_flag, S->d_flag + (m - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t nd = (uint64_t)last_pos + last_flag;       // distinct (sketch, hash)

    out->hashes = (uint64_t*)malloc(std::max<uint64_t>(nd, 1) * sizeof(uint64_t));
    out->abundances = (uint32_t*)malloc(std::max<uint64_t>(nd, 1) * sizeof(uint32_t));
    std::vector<uint32_t> start(nd + 1), sid(nd);
    if (!out->hashes || !out->abundances) { ygpu_sketch_result_free(out); return ygpu_fail(ctx, YGPU_ERR_NOMEM, "out of host memory"); }
    YG_CUDA(ctx, cudaMemcpyAsync(out->hashes, S->d_out_h, nd * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(start.data(), S->d_out_start, nd * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(sid.data(), S->d_out_sid, nd * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    start[nd] = (uint32_t)m;
    for (uint64_t i = 0; i < nd; i++) {
        out->abundances[i] = start[i + 1] - start[i];
        out->offsets[sid[i] + 1]++;
    }
    for (uint32_t s = 0; s < n_sketches; s++) out->offsets[s + 1] += out->offsets[s];
    return 0;
}
