// libyachtgpu -- train path: context, sketch residency, inverted index (K2), pairwise
// shared-hash count fused with threshold + compaction (K3+K4).  sm_100a only.
//
// Reference behaviour being replaced: KoslickiLab/YACHT src/cpp/main.cpp
//   compute_index_from_sketches            :215-246  -> ygpu_build_index
//   compute_intersection_matrix_by_sketches:249-312  -> ygpu_pairwise_flag
// This is a new design, not a translation: the reference walks an unordered_map per query hash
// and increments a dense N x N int matrix on the host; here the index is a radix-sorted
// (hash, genome) array whose equal-hash runs ARE the posting lists, every genome gets a compact
// list of "the postings that follow me in my run" (upper triangle only: M is symmetric), and one
// CTA per query genome accumulates its row in shared memory and emits only the pairs that pass
// the containment threshold.
#include "common.cuh"

#include <cub/cub.cuh>
#include <cstdarg>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <new>
#include <vector>

static std::string g_create_err;
static std::mutex g_err_mu;      // ygpu_upload_block is called from several threads at once: their failures must not race on the text

int ygpu_fail(ygpu_ctx* ctx, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    std::lock_guard<std::mutex> lk(g_err_mu);
    if (ctx) ctx->err = buf;
    else g_create_err = buf;
    return code;
}

int ygpu_temp_reserve(ygpu_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->temp_bytes) return 0;
    if (ctx->d_temp) cudaFree(ctx->d_temp);
    ctx->d_temp = nullptr;
    ctx->temp_bytes = 0;
    size_t want = bytes + (bytes >> 3) + 256;
    YG_CUDA(ctx, cudaMalloc(&ctx->d_temp, want));
    ctx->temp_bytes = want;
    return 0;
}

// ============================================================================================
// context
// ============================================================================================
extern "C" int ygpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int ygpu_ctx_create(ygpu_ctx** out, int device) {
    if (!out) return ygpu_fail(nullptr, YGPU_ERR_ARG, "ygpu_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return ygpu_fail(nullptr, YGPU_ERR_NO_DEVICE,
                         "no CUDA device available (%s); libyachtgpu has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= ndev)
        return ygpu_fail(nullptr, YGPU_ERR_ARG, "device %d out of range (have %d)", device, ndev);
    ygpu_ctx* ctx = new (std::nothrow) ygpu_ctx();
    if (!ctx) return ygpu_fail(nullptr, YGPU_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess) {
        delete ctx;
        return ygpu_fail(nullptr, YGPU_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        delete ctx;
        return ygpu_fail(nullptr, YGPU_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    }
    if (prop.major < 10) {
        delete ctx;
        return ygpu_fail(nullptr, YGPU_ERR_NO_DEVICE,
                         "device %d is sm_%d%d; libyachtgpu is built for sm_100a (B200) only", device,
                         prop.major, prop.minor);
    }
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        delete ctx;
        return ygpu_fail(nullptr, YGPU_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    for (auto& ev : ctx->evp) cudaEventCreate(&ev);
    if (cudaMalloc(&ctx->d_scalars, 64 * sizeof(unsigned long long)) != cudaSuccess) {
        ygpu_ctx_destroy(ctx);
        return ygpu_fail(nullptr, YGPU_ERR_NOMEM, "cudaMalloc(scalars) failed");
    }
    *out = ctx;
    return 0;
}

static void release_index(ygpu_ctx* ctx) {   // invalidate only: the buffers are kept for reuse
    ctx->row_work_valid = false;
    ctx->sorted = false;
    ctx->indexed = false;
    ctx->P = 0; ctx->n_items = 0;
}

static void release_sketches(ygpu_ctx* ctx) {
    release_index(ctx);
    ctx->loaded = false;
    ctx->sharded = false;
    ctx->part_valid = false;
    ctx->maxkey_valid = false;
    ctx->n = 0; ctx->T = 0;
}

static void free_all(ygpu_ctx* ctx) {
    dev_free(ctx, &ctx->d_skey); dev_free(ctx, &ctx->d_sgid); dev_free(ctx, &ctx->d_flag); dev_free(ctx, &ctx->d_cpos);
    dev_free(ctx, &ctx->d_post); dev_free(ctx, &ctx->d_rem); dev_free(ctx, &ctx->d_row_ptr); dev_free(ctx, &ctx->d_row_items);
    dev_free(ctx, &ctx->d_row_work); dev_free(ctx, &ctx->d_row_cnt);
    dev_free(ctx, &ctx->d_ovf_rows); dev_free(ctx, &ctx->d_st_rem); dev_free(ctx, &ctx->d_units); dev_free(ctx, &ctx->d_tile_g0);
    dev_free(ctx, &ctx->d_big_list); dev_free(ctx, &ctx->d_big_cstart); dev_free(ctx, &ctx->d_big_a); dev_free(ctx, &ctx->d_big_b);
    dev_free(ctx, &ctx->d_ent1); dev_free(ctx, &ctx->d_ent2); dev_free(ctx, &ctx->d_msd_aux);
    dev_free(ctx, &ctx->d_hashes); dev_free(ctx, &ctx->d_offsets); dev_free(ctx, &ctx->d_sizes); dev_free(ctx, &ctx->d_gid);
    dev_free(ctx, &ctx->d_offsets_local); dev_free(ctx, &ctx->d_row_begin_local); dev_free(ctx, &ctx->d_sh_hist_all);
    dev_free(ctx, &ctx->d_sh_owner); dev_free(ctx, &ctx->d_sh_info);
    dev_free(ctx, &ctx->d_tc);
    dev_free(ctx, &ctx->d_out_key); dev_free(ctx, &ctx->d_out_cnt); dev_free(ctx, &ctx->d_out_key2); dev_free(ctx, &ctx->d_out_cnt2);
}

extern "C" void ygpu_ctx_destroy(ygpu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    release_sketches(ctx);
    free_all(ctx);
    ygpu_run_release(ctx);
    ygpu_part_release(ctx);
    ygpu_sketch_release(ctx);
    ygpu_stream_release(ctx);
    ygpu_upload_release(ctx);
    ygpu_comm_destroy(ctx);
    if (ctx->d_pairs_local) cudaFree(ctx->d_pairs_local);
    if (ctx->d_pairs) cudaFree(ctx->d_pairs);
    if (ctx->d_temp) cudaFree(ctx->d_temp);
    if (ctx->d_scalars) cudaFree(ctx->d_scalars);
    for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->evp) if (ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* ygpu_last_error(const ygpu_ctx* ctx) {
    return ctx ? ctx->err.c_str() : g_create_err.c_str();
}

extern "C" void ygpu_free(void* p) { free(p); }

extern "C" void* ygpu_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void ygpu_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int ygpu_reset_timers(ygpu_ctx* ctx) {
    if (!ctx) return YGPU_ERR_ARG;
    ctx->tm = ygpu_timings{};
    return 0;
}

extern "C" int ygpu_get_timings(ygpu_ctx* ctx, ygpu_timings* out) {
    if (!ctx || !out) return YGPU_ERR_ARG;
    *out = ctx->tm;
    return 0;
}

// ============================================================================================
// sketch residency
// ============================================================================================
// one CTA per genome (grid-stride): genome id of every hash slot + sketch sizes
__global__ void __launch_bounds__(256) k_expand_gid(const uint64_t* __restrict__ offsets, uint32_t n,
                                                     uint32_t* __restrict__ gid, uint32_t* __restrict__ sizes) {
    for (uint32_t g = blockIdx.x; g < n; g += gridDim.x) {
        const uint64_t b = offsets[g], e = offsets[g + 1];
        if (threadIdx.x == 0) sizes[g] = (uint32_t)(e - b);
        for (uint64_t p = b + threadIdx.x; p < e; p += blockDim.x) gid[p] = g;
    }
}

static int finish_load(ygpu_ctx* ctx) {
    const uint32_t n = ctx->n;
    YG_CHECK(dev_alloc(ctx, &ctx->d_sizes, n));
    YG_CHECK(dev_alloc(ctx, &ctx->d_gid, ctx->T));
    if (n) {
        int grid = (int)std::min<uint32_t>(n, (uint32_t)ctx->num_sms * 16);
        k_expand_gid<<<grid, 256, 0, ctx->stream>>>(ctx->d_offsets, n, ctx->d_gid, ctx->d_sizes);
        ctx->tm.n_kernel_launches++;
        YG_CUDA(ctx, cudaGetLastError());
    }
    YG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->loaded = true;
    if (ctx->T) {           // the largest hash decides the partition plan: a property of the resident sketches, taken at load
        uint64_t mk = 0;
        YG_CHECK(ygpu_max_hash(ctx, &mk));
    }
    return 0;
}

static int load_common(ygpu_ctx* ctx, const uint64_t* hashes, const uint64_t* offsets, uint32_t n, bool from_device) {
    if (!ctx) return YGPU_ERR_ARG;
    if (!offsets || (n > 0 && !hashes && false)) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches: NULL offsets");
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    release_sketches(ctx);
    uint64_t T = 0;
    if (from_device) {
        YG_CUDA(ctx, cudaMemcpy(&T, offsets + n, sizeof(uint64_t), cudaMemcpyDeviceToHost));
    } else {
        T = offsets[n];
        for (uint32_t g = 0; g < n; g++)
            if (offsets[g + 1] < offsets[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets not monotone at genome %u", g);
        if (offsets[0] != 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets[0] must be 0");
    }
    if (T >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes %llu >= 2^32 not supported", (unsigned long long)T);
    if (n >= (1u << 31)) return ygpu_fail(ctx, YGPU_ERR_ARG, "too many genomes");
    if (T > 0 && !hashes) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches: NULL hashes");
    ctx->n = n;
    ctx->T = T;
    YG_CHECK(dev_alloc(ctx, &ctx->d_hashes, T));
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets, (uint64_t)n + 1));
    cudaMemcpyKind kind = from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    if (T) YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_hashes, hashes, T * sizeof(uint64_t), kind, ctx->stream));
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_offsets, offsets, ((uint64_t)n + 1) * sizeof(uint64_t), kind, ctx->stream));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
    YG_CHECK(finish_load(ctx));
    ctx->tm.ms_h2d += elapsed(ctx, 0, 1);
    return 0;
}

extern "C" int ygpu_load_sketches(ygpu_ctx* ctx, const uint64_t* hashes, const uint64_t* offsets, uint32_t n) {
    return load_common(ctx, hashes, offsets, n, false);
}
extern "C" int ygpu_load_sketch_blocks(ygpu_ctx* ctx, const uint64_t* const* blocks, const uint64_t* block_lens, uint32_t nblocks,
                                       const uint64_t* offsets, uint32_t n) {
    if (!ctx || !offsets || (nblocks && (!blocks || !block_lens))) return YGPU_ERR_ARG;
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    release_sketches(ctx);
    uint64_t T = 0;
    for (uint32_t b = 0; b < nblocks; b++) T += block_lens[b];
    if (T != offsets[n] || offsets[0] != 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketch_blocks: pieces hold %llu hashes, offsets say %llu",
                                                             (unsigned long long)T, (unsigned long long)offsets[n]);
    for (uint32_t g = 0; g < n; g++)
        if (offsets[g + 1] < offsets[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets not monotone at genome %u", g);
    if (T >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes %llu >= 2^32 not supported", (unsigned long long)T);
    ctx->n = n;
    ctx->T = T;
    YG_CHECK(dev_alloc(ctx, &ctx->d_hashes, T));
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets, (uint64_t)n + 1));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    uint64_t pos = 0;
    for (uint32_t b = 0; b < nblocks; b++) {
        if (block_lens[b]) YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_hashes + pos, blocks[b], block_lens[b] * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        pos += block_lens[b];
    }
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_offsets, offsets, ((uint64_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
    YG_CHECK(finish_load(ctx));
    ctx->tm.ms_h2d += elapsed(ctx, 0, 1);
    return 0;
}

// ---- streaming ingest: blocks of parsed sketches travel to the device while later files are still being
// parsed.  Their final position in the flat array is only known once every sketch size is (CSR offsets are a
// prefix sum), so a block is first uploaded to a staging chunk -- through a small pool of page-locked bounce
// buffers, filled by the calling threads in parallel, DMA'd asynchronously -- and ygpu_upload_finish moves all
// blocks to their places with one device-side copy kernel.
#include <atomic>
#include <condition_variable>
#include <mutex>

namespace {
struct UploadBlk { const uint64_t* src; uint64_t len; uint32_t id; };
struct UploadState {
    static constexpr int NB = 8;
    static constexpr uint64_t BOUNCE = 1ull << 20;        // hashes per bounce buffer (8 MB)
    static constexpr uint64_t CHUNK = 1ull << 25;         // hashes per device staging chunk (256 MB)
    std::mutex mu;
    std::condition_variable cv;
    std::vector<uint64_t*> chunks;
    uint64_t fill = CHUNK;                                // used part of the last chunk (CHUNK = none yet)
    std::vector<UploadBlk> blocks;
    uint64_t* bounce[NB] = {};
    cudaEvent_t bev[NB] = {};
    cudaStream_t bst[NB] = {};
    bool busy[NB] = {};
    uint64_t total = 0;
    std::atomic<int> failed{0};
};

struct PlaceDesc { const uint64_t* src; uint64_t dst; uint64_t len; };

__global__ void __launch_bounds__(256) k_place_blocks(const PlaceDesc* __restrict__ d, uint32_t nd, uint64_t* __restrict__ out) {
    for (uint32_t b = blockIdx.x; b < nd; b += gridDim.x) {
        const PlaceDesc p = d[b];
        for (uint64_t i = threadIdx.x; i < p.len; i += blockDim.x) out[p.dst + i] = p.src[i];
    }
}
}  // namespace

void ygpu_upload_release(ygpu_ctx* ctx) {
    UploadState* u = (UploadState*)ctx->upload;
    if (!u) return;
    for (int b = 0; b < UploadState::NB; b++) {
        if (u->bst[b]) { cudaStreamSynchronize(u->bst[b]); cudaStreamDestroy(u->bst[b]); }
        if (u->bev[b]) cudaEventDestroy(u->bev[b]);
        if (u->bounce[b]) cudaFreeHost(u->bounce[b]);
    }
    for (uint64_t* c : u->chunks) cudaFree(c);
    delete u;
    ctx->upload = nullptr;
}

extern "C" int ygpu_upload_begin(ygpu_ctx* ctx) {
    if (!ctx) return YGPU_ERR_ARG;
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    ygpu_upload_release(ctx);
    release_sketches(ctx);
    UploadState* u = new (std::nothrow) UploadState();
    if (!u) return ygpu_fail(ctx, YGPU_ERR_NOMEM, "out of host memory");
    ctx->upload = u;
    for (int b = 0; b < UploadState::NB; b++) {
        YG_CUDA(ctx, cudaHostAlloc((void**)&u->bounce[b], UploadState::BOUNCE * sizeof(uint64_t), cudaHostAllocDefault));
        YG_CUDA(ctx, cudaStreamCreateWithFlags(&u->bst[b], cudaStreamNonBlocking));
        YG_CUDA(ctx, cudaEventCreateWithFlags(&u->bev[b], cudaEventDisableTiming));
    }
    return 0;
}

// Thread-safe: parser / uploader threads call it concurrently.  `hashes` may be released when it returns.
extern "C" int ygpu_upload_block(ygpu_ctx* ctx, uint32_t block_id, const uint64_t* hashes, uint64_t len) {
    if (!ctx || (len && !hashes)) return YGPU_ERR_ARG;
    UploadState* u = (UploadState*)ctx->upload;
    if (!u) return ygpu_fail(ctx, YGPU_ERR_STATE, "upload_block: ygpu_upload_begin first");
    if (len == 0) return 0;
    if (cudaSetDevice(ctx->device) != cudaSuccess) { u->failed = 1; return YGPU_ERR_CUDA; }
    uint64_t done = 0;
    uint64_t* base = nullptr;      // where this block lives in the staging chunks
    while (done < len) {
        const uint64_t piece = std::min<uint64_t>(len - done, UploadState::BOUNCE);
        int b = -1;
        {
            std::unique_lock<std::mutex> lk(u->mu);
            if (done == 0) {          // reserve device space for the whole block (contiguous inside one chunk when it fits)
                if (len > UploadState::CHUNK) { u->failed = 1; return ygpu_fail(ctx, YGPU_ERR_ARG, "upload_block: block of %llu hashes exceeds the staging chunk", (unsigned long long)len); }
                if (u->fill + len > UploadState::CHUNK) {
                    uint64_t* c = nullptr;
                    if (cudaMalloc((void**)&c, UploadState::CHUNK * sizeof(uint64_t)) != cudaSuccess) { u->failed = 1; return ygpu_fail(ctx, YGPU_ERR_NOMEM, "upload_block: staging chunk"); }
                    u->chunks.push_back(c);
                    u->fill = 0;
                }
                base = u->chunks.back() + u->fill;
                u->blocks.push_back(UploadBlk{base, len, block_id});
                u->fill += len;
                u->total += len;
            }
            u->cv.wait(lk, [&] { for (int i = 0; i < UploadState::NB; i++) if (!u->busy[i]) return true; return false; });
            for (int i = 0; i < UploadState::NB; i++) if (!u->busy[i]) { b = i; break; }
            u->busy[b] = true;
        }
        cudaError_t e = cudaEventSynchronize(u->bev[b]);            // the previous DMA out of this bounce buffer
        if (e == cudaSuccess) {
            memcpy(u->bounce[b], hashes + done, piece * sizeof(uint64_t));
            e = cudaMemcpyAsync(base + done, u->bounce[b], piece * sizeof(uint64_t), cudaMemcpyHostToDevice, u->bst[b]);
        }
        if (e == cudaSuccess) e = cudaEventRecord(u->bev[b], u->bst[b]);
        {
            std::lock_guard<std::mutex> lk(u->mu);
            u->busy[b] = false;
            if (e != cudaSuccess) u->failed = 1;
        }
        u->cv.notify_one();
        if (e != cudaSuccess) return ygpu_fail(ctx, YGPU_ERR_CUDA, "upload_block: %s", cudaGetErrorString(e));
        done += piece;
    }
    return 0;
}

// Place the uploaded blocks: block_dst[id] = position of block `id` in the resident hash array of T hashes (the whole
// flat array, or -- sharded residency -- this rank's slice).  Leaves d_hashes filled; the caller finishes the load.
static int upload_place(ygpu_ctx* ctx, const uint64_t* block_dst, uint32_t nblocks, uint64_t T) {
    UploadState* u = (UploadState*)ctx->upload;
    if (!u) return ygpu_fail(ctx, YGPU_ERR_STATE, "upload_finish: ygpu_upload_begin first");
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int b = 0; b < UploadState::NB; b++) YG_CUDA(ctx, cudaStreamSynchronize(u->bst[b]));
    int rc = 0;
    if (u->failed) rc = ygpu_fail(ctx, YGPU_ERR_CUDA, "upload_finish: an upload failed");
    else if (u->total != T) rc = ygpu_fail(ctx, YGPU_ERR_ARG, "upload_finish: %llu hashes uploaded, offsets say %llu", (unsigned long long)u->total, (unsigned long long)T);
    else if (T >= (1ull << 32)) rc = ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes %llu >= 2^32 not supported", (unsigned long long)T);
    std::vector<PlaceDesc> desc;
    for (const UploadBlk& k : u->blocks) {
        if (rc) break;
        if (k.id >= nblocks || block_dst[k.id] + k.len > T) { rc = ygpu_fail(ctx, YGPU_ERR_ARG, "upload_finish: block %u does not fit", k.id); break; }
        desc.push_back(PlaceDesc{k.src, block_dst[k.id], k.len});
    }
    if (!rc) {
        rc = dev_alloc(ctx, &ctx->d_hashes, T + 2);
        if (!rc) rc = ygpu_temp_reserve(ctx, std::max<size_t>(desc.size(), 1) * sizeof(PlaceDesc));
    }
    if (!rc) {
        cudaStream_t st = ctx->stream;
        cudaError_t e = cudaEventRecord(ctx->ev[0], st);
        if (e == cudaSuccess && !desc.empty()) {
            e = cudaMemcpyAsync(ctx->d_temp, desc.data(), desc.size() * sizeof(PlaceDesc), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                k_place_blocks<<<(unsigned)std::min<size_t>(desc.size(), (size_t)ctx->num_sms * 16), 256, 0, st>>>((const PlaceDesc*)ctx->d_temp, (uint32_t)desc.size(), ctx->d_hashes);
                e = cudaGetLastError();
                ctx->tm.n_kernel_launches++;
            }
        }
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev[1], st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);      // desc is a host temporary
        if (e != cudaSuccess) rc = ygpu_fail(ctx, YGPU_ERR_CUDA, "upload_finish: %s", cudaGetErrorString(e));
    }
    if (!rc) ctx->tm.ms_h2d += elapsed(ctx, 0, 1);
    ygpu_upload_release(ctx);
    return rc;
}

// block_dst[id] = position of block `id` in the flat hash array; offsets / n as for ygpu_load_sketches.
extern "C" int ygpu_upload_finish(ygpu_ctx* ctx, const uint64_t* block_dst, uint32_t nblocks, const uint64_t* offsets, uint32_t n) {
    if (!ctx || !offsets || (nblocks && !block_dst)) return YGPU_ERR_ARG;
    if (offsets[0] != 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets[0] must be 0");
    for (uint32_t g = 0; g < n; g++)
        if (offsets[g + 1] < offsets[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets not monotone at genome %u", g);
    const uint64_t T = offsets[n];
    YG_CHECK(upload_place(ctx, block_dst, nblocks, T));
    ctx->n = n;
    ctx->T = T;
    ctx->sharded = false;
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets, (uint64_t)n + 1));
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_offsets, offsets, ((uint64_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    return finish_load(ctx);
}

int ygpu_sharded_finish(ygpu_ctx* ctx, const uint64_t* offsets, uint32_t n, uint32_t g_begin, uint32_t g_end);   // index_msd.cu

// Sharded residency: the uploaded blocks are the sketches of genomes [g_begin, g_end) only; block_dst is relative to
// the first hash of genome g_begin.  Collective over the communicator (like ygpu_load_sketches_sharded).
extern "C" int ygpu_upload_finish_sharded(ygpu_ctx* ctx, const uint64_t* block_dst, uint32_t nblocks, const uint64_t* offsets, uint32_t n,
                                          uint32_t g_begin, uint32_t g_end) {
    if (!ctx || !offsets || (nblocks && !block_dst)) return YGPU_ERR_ARG;
    if (g_begin > g_end || g_end > n) return ygpu_fail(ctx, YGPU_ERR_ARG, "bad genome range [%u,%u) of %u", g_begin, g_end, n);
    YG_CHECK(upload_place(ctx, block_dst, nblocks, offsets[g_end] - offsets[g_begin]));
    return ygpu_sharded_finish(ctx, offsets, n, g_begin, g_end);
}

extern "C" int ygpu_load_sketches_device(ygpu_ctx* ctx, const uint64_t* d_hashes, const uint64_t* d_offsets, uint32_t n) {
    return load_common(ctx, d_hashes, d_offsets, n, true);
}

// ============================================================================================
// K2: inverted index
// ============================================================================================
// flag[s] = 1 iff sorted slot s lies in a run (equal hashes) of length >= 2.  Also counts the
// distinct hashes, the singletons (the three banner lines of main.cpp:242-244) and in-sketch
// duplicates (same hash twice in one genome).
__global__ void __launch_bounds__(256) k_flag_runs(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sgid,
                                                    uint64_t T, uint8_t* __restrict__ flag,
                                                    unsigned long long* __restrict__ scal) {
    unsigned long long heads = 0, singles = 0, dups = 0;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < T; s += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = key[s];
        const bool peq = s > 0 && key[s - 1] == k;
        const bool neq = s + 1 < T && key[s + 1] == k;
        flag[s] = (peq || neq) ? 1 : 0;
        heads += !peq;
        singles += (!peq && !neq);
        if (peq && sgid[s - 1] == sgid[s]) dups++;
    }
    heads = block_sum<256>(heads);
    singles = block_sum<256>(singles);
    dups = block_sum<256>(dups);
    if (threadIdx.x == 0) {
        if (heads) atomicAdd(&scal[SC_HEADS], heads);
        if (singles) atomicAdd(&scal[SC_SINGLE], singles);
        if (dups) atomicAdd(&scal[SC_DUPS], dups);
    }
}

// first slot e > s with key[e] != key[s] (exponential probe, then bisection)
__device__ __forceinline__ uint64_t run_end(const uint64_t* __restrict__ key, uint64_t s, uint64_t T) {
    const uint64_t k = key[s];
    uint64_t lo = s, step = 1, hi = s + 1;
    while (hi < T && key[hi] == k) { lo = hi; step <<= 1; hi = lo + step; }
    if (hi > T) hi = T;
    while (hi - lo > 1) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (key[mid] == k) lo = mid; else hi = mid;
    }
    return hi;
}

struct FlagToU32 {
    __host__ __device__ __forceinline__ uint32_t operator()(const uint8_t& f) const { return (uint32_t)f; }
};

// every kept slot: copy its genome id into the compact posting array, record how many postings
// follow it in its run (that is the work row `g` does for this hash: upper triangle only), and
// histogram non-empty work items per genome.
__global__ void __launch_bounds__(256) k_post_compact(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sgid,
                                                       const uint8_t* __restrict__ flag, const uint32_t* __restrict__ cpos,
                                                       uint64_t T, uint32_t* __restrict__ post, uint32_t* __restrict__ rem,
                                                       unsigned long long* __restrict__ row_cnt,
                                                       unsigned long long* __restrict__ row_work,
                                                       unsigned long long* __restrict__ scal) {
    unsigned long long w = 0;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < T; s += (uint64_t)gridDim.x * blockDim.x) {
        if (!flag[s]) continue;
        const uint32_t g = sgid[s];
        const uint32_t c = cpos[s];
        const uint64_t e = run_end(key, s, T);
        const uint32_t r = (uint32_t)(e - s - 1);
        post[c] = g;
        rem[c] = r;
        w += 2ull * r + 1ull;  // sum over the members of a run of (2*rem+1) == L^2
        if (r) {
            atomicAdd(&row_cnt[g], 1ull);
            atomicAdd(&row_work[g], (unsigned long long)r);
        }
    }
    w = block_sum<256>(w);
    if (threadIdx.x == 0 && w) atomicAdd(&scal[SC_W], w);
}

__global__ void __launch_bounds__(256) k_items_scatter(const uint32_t* __restrict__ post, const uint32_t* __restrict__ rem,
                                                        uint64_t P, const uint64_t* __restrict__ row_ptr,
                                                        unsigned long long* __restrict__ row_fill,
                                                        uint64_t* __restrict__ row_items) {
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < P; c += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = rem[c];
        if (!r) continue;
        const uint32_t g = post[c];
        const unsigned long long k = atomicAdd(&row_fill[g], 1ull);
        row_items[row_ptr[g] + k] = ((uint64_t)(c + 1) << 32) | ((uint64_t)r << 2);   // item format v2, indirect
    }
}

int ygpu_max_hash(ygpu_ctx* ctx, uint64_t* maxkey) {
    if (!ctx->maxkey_valid) {
        cudaStream_t st = ctx->stream;
        uint64_t* d_max = (uint64_t*)&ctx->d_scalars[SC_MAXKEY];
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb, ctx->d_hashes, d_max, (int64_t)ctx->T, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, ctx->d_hashes, d_max, (int64_t)ctx->T, st));
        ctx->tm.n_library_launches += 2;
        YG_CUDA(ctx, cudaMemcpyAsync(&ctx->maxkey, d_max, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        ctx->maxkey_valid = true;
    }
    *maxkey = ctx->maxkey;
    return 0;
}

// K2a: stable radix sort of (hash, genome id); equal-hash runs become posting lists in ascending
// genome order (slots are generated genome-major and the sort is stable).  Kept resident: the
// run path (K5) walks the same sorted array.
int ygpu_sort_sketches(ygpu_ctx* ctx) {
    if (ctx->sorted) return 0;
    const uint64_t T = ctx->T;
    cudaStream_t st = ctx->stream;
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    YG_CHECK(dev_alloc(ctx, &ctx->d_skey, T));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sgid, T));
    if (T) {
        uint64_t maxkey = 0;
        YG_CHECK(ygpu_max_hash(ctx, &maxkey));
        int end_bit = 1;
        while (end_bit < 64 && (maxkey >> end_bit) != 0) end_bit++;
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_hashes, ctx->d_skey, ctx->d_gid, ctx->d_sgid,
                                                     (int64_t)T, 0, end_bit, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, ctx->d_hashes, ctx->d_skey, ctx->d_gid, ctx->d_sgid,
                                                     (int64_t)T, 0, end_bit, st));
        ctx->tm.n_library_launches += 2 + (end_bit + 7) / 8;
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->tm.ms_sort += elapsed(ctx, 2, 3);
    ctx->sorted = true;
    return 0;
}

extern "C" int ygpu_build_index(ygpu_ctx* ctx, ygpu_index_stats* stats) {
    if (!ctx) return YGPU_ERR_ARG;
    if (!ctx->loaded) return ygpu_fail(ctx, YGPU_ERR_STATE, "build_index: no sketches loaded");
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    release_index(ctx);
    ctx->last_group2_grid = 0;
    ctx->last_group_grid = 0;
    ctx->last_big_chunks = 0;
    const uint64_t T = ctx->T;
    const uint32_t n = ctx->n;
    cudaStream_t st = ctx->stream;
    ygpu_index_stats S{};
    S.n_hashes = T;

    YG_CHECK(dev_alloc(ctx, &ctx->d_row_ptr, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_work, n));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_row_ptr, 0, ((uint64_t)n + 1) * sizeof(uint64_t), st));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_row_work, 0, std::max<uint64_t>(n, 1) * sizeof(uint64_t), st));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_scalars, 0, 16 * sizeof(unsigned long long), st));

    if (T == 0 || n == 0) {
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        if (n) {
            std::vector<uint32_t> sz(n);
            YG_CUDA(ctx, cudaMemcpy(sz.data(), ctx->d_sizes, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        }
        ctx->stats = S;
        ctx->indexed = true;
        if (stats) *stats = S;
        return 0;
    }

    // ---- preferred: MSD partition + shared-memory grouping (index_msd.cu) -----------------------------
    if (ctx->index_path != 0) {
        int used = 0;
        YG_CHECK(ygpu_build_index_msd(ctx, &S, &used));
        if (used) {
            std::vector<uint32_t> sz(n);
            YG_CUDA(ctx, cudaMemcpy(sz.data(), ctx->d_sizes, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
            uint32_t mx = 0;
            for (uint32_t v : sz) mx = std::max(mx, v);
            S.max_sketch = mx;
            S.index_path = 1;
            S.big_buckets = ctx->msd_big_buckets;
            ctx->stats = S;
            ctx->indexed = true;
            ctx->last_index_path = 1;
            if (stats) *stats = S;
            return 0;
        }
        // not applicable (or skewed): the scalars the general path accumulates into start from zero again
        YG_CUDA(ctx, cudaMemsetAsync(ctx->d_scalars, 0, 16 * sizeof(unsigned long long), st));
        YG_CUDA(ctx, cudaMemsetAsync(ctx->d_row_work, 0, std::max<uint64_t>(n, 1) * sizeof(uint64_t), st));
    }
    ctx->last_index_path = 0;
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    // ---- K2a: stable radix sort of (hash, genome id)
    YG_CHECK(ygpu_sort_sketches(ctx));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));

    // ---- K2b: runs -> compact postings + per-genome work lists
    YG_CHECK(dev_alloc(ctx, &ctx->d_flag, T));
    YG_CHECK(dev_alloc(ctx, &ctx->d_cpos, T + 1));
    k_flag_runs<<<grid_for(ctx, T, 256), 256, 0, st>>>(ctx->d_skey, ctx->d_sgid, T, ctx->d_flag, ctx->d_scalars);
    YG_CUDA(ctx, cudaGetLastError());
    {
        cub::TransformInputIterator<uint32_t, FlagToU32, const uint8_t*> it(ctx->d_flag, FlagToU32());
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb, it, ctx->d_cpos, (int64_t)T, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, it, ctx->d_cpos, (int64_t)T, st));
        ctx->tm.n_library_launches += 2;
    }
    uint32_t last_cpos = 0;
    uint8_t last_flag = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(&last_cpos, ctx->d_cpos + (T - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(&last_flag, ctx->d_flag + (T - 1), sizeof(uint8_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t P = (uint64_t)last_cpos + last_flag;
    ctx->P = P;
    YG_CHECK(dev_alloc(ctx, &ctx->d_post, P));
    YG_CHECK(dev_alloc(ctx, &ctx->d_rem, P));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_cnt, (uint64_t)n + 1));
    unsigned long long* d_row_cnt = ctx->d_row_cnt;
    YG_CUDA(ctx, cudaMemsetAsync(d_row_cnt, 0, ((uint64_t)n + 1) * sizeof(unsigned long long), st));
    if (P) {
        k_post_compact<<<grid_for(ctx, T, 256), 256, 0, st>>>(ctx->d_skey, ctx->d_sgid, ctx->d_flag, ctx->d_cpos, T,
                                                              ctx->d_post, ctx->d_rem, d_row_cnt,
                                                              (unsigned long long*)ctx->d_row_work, ctx->d_scalars);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
    }
    {
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb, d_row_cnt, (unsigned long long*)ctx->d_row_ptr, (int64_t)n + 1, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, d_row_cnt, (unsigned long long*)ctx->d_row_ptr, (int64_t)n + 1, st));
        ctx->tm.n_library_launches += 2;
    }
    unsigned long long sc[16];
    uint64_t n_items = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(&n_items, ctx->d_row_ptr + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(sc, ctx->d_scalars, sizeof sc, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->n_items = n_items;
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_items, n_items));
    if (n_items) {
        YG_CUDA(ctx, cudaMemsetAsync(d_row_cnt, 0, ((uint64_t)n + 1) * sizeof(unsigned long long), st));
        k_items_scatter<<<grid_for(ctx, P, 256), 256, 0, st>>>(ctx->d_post, ctx->d_rem, P, ctx->d_row_ptr, d_row_cnt,
                                                               ctx->d_row_items);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->d_row_begin = ctx->d_row_ptr;   // d_row_cnt (the scatter's fill cursors) now holds each row's item count
    ctx->row_work_valid = true;          // k_post_compact accumulated it
    ctx->tm.n_kernel_launches += 1;  // k_flag_runs
    ctx->tm.ms_index += elapsed(ctx, 1, 2);

    // sorted keys / flags / scan are only needed while building (the run path re-sorts with its
    // own mask); release them so an 85k-genome index leaves HBM to the count kernel's output.
    // (d_flag / d_cpos / d_rem are scratch of the build; they stay allocated for the next build)

    std::vector<uint32_t> sz(n);
    YG_CUDA(ctx, cudaMemcpy(sz.data(), ctx->d_sizes, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    uint32_t mx = 0;
    for (uint32_t v : sz) mx = std::max(mx, v);

    S.n_distinct = sc[SC_HEADS];
    S.n_singleton = sc[SC_SINGLE];
    S.n_index = S.n_distinct - S.n_singleton;
    S.n_postings = P;
    S.n_increments = sc[SC_W];
    S.n_row_items = n_items;
    S.max_sketch = mx;
    S.has_duplicates = sc[SC_DUPS] ? 1u : 0u;
    ctx->stats = S;
    ctx->indexed = true;
    if (stats) *stats = S;
    return 0;
}

// ============================================================================================
// K3 + K4: pairwise shared-hash count (row-wise integer SpGEMM over the inverted index, upper
// triangle) fused with the containment threshold and compaction of the flagged ordered pairs.
// ============================================================================================
#define K3_THREADS 256
#define K3_TOUCH_CAP 4096      // distinct columns tracked per (row, tile) before falling back to a dense scan
#define K3_LONG_CAP 1024       // posting segments longer than K3_LONG_LEN are expanded by the whole CTA, chunk by chunk of the
                               // work list (a chunk = one item per thread, so the queue can never overflow)
#define K3_LONG_LEN 64

struct K3Params {
    const uint64_t* list_begin;         // [n] start of each row's work list
    const unsigned long long* row_n;    // [n] its length
    const uint64_t* row_items;
    const uint32_t* post;
    const uint32_t* sizes;
    uint32_t n;
    uint32_t row_begin, row_end;
    uint32_t tile_w;       // columns per tile
    uint32_t n_tiles;
    double thr;
    uint64_t* out_key;     // (i << key_shift) | j   (key_shift = bits of a genome id: the later sort only walks 2 * key_shift bits)
    int key_shift;
    uint32_t* out_cnt;
    uint64_t out_cap;
    unsigned long long* scal;  // SC_OUT = pairs emitted, SC_UNIT = work-unit ticket, SC_OVF = rows deferred to the dense kernel
    const uint32_t* row_list;  // dense kernel: explicit rows (the warp kernel's overflow list) instead of [row_begin, row_end)
    uint32_t n_list;
    uint32_t* ovf_rows;        // warp kernel: rows whose distinct columns overflow a warp's hash table
    const uint32_t* tc;        // [n] smallest count that passes the containment test for genome g (k4_thresholds), or NULL
};

// warp-aggregated append: one atomic per warp-instruction instead of one per lane
__device__ __forceinline__ void emit_pair(const K3Params& p, uint32_t i, uint32_t j, uint32_t cnt) {
    const unsigned m = __activemask();
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(&p.scal[SC_OUT], (unsigned long long)__popc(m));
    base = __shfl_sync(m, base, leader);
    const unsigned long long slot = base + __popc(m & ((1u << lane) - 1u));
    if (slot < p.out_cap) {
        p.out_key[slot] = ((uint64_t)i << p.key_shift) | (uint64_t)j;
        p.out_cnt[slot] = cnt;
    }
}

// the reference's test for one unordered pair {i<j} with `cnt` shared hashes, both directions
// (main.cpp:277-303).  The "union" is evaluated modulo 2^64 exactly as size_t + size_t - int is.
// The reference's comparison `1.0 * cnt / size < thr` (main.cpp:297-301) is monotone in cnt, so for every genome there is a
// smallest passing count; k4_thresholds finds it with that very fp64 expression, and the kernel compares integers.  Only
// valid without in-sketch duplicates (the reference's zero-union skip can then never fire: cnt <= min(ni, nj)).
__global__ void __launch_bounds__(256) k4_thresholds(const uint32_t* __restrict__ sizes, uint32_t n, double thr, uint32_t* __restrict__ tc) {
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) {
        const uint32_t ni = sizes[g];
        if (ni == 0) { tc[g] = 0xFFFFFFFFu; continue; }
        const double dn = (double)ni;
        long long c = (long long)ceil(thr * dn);
        if (c < 1) c = 1;
        while (c > 1 && !(1.0 * (double)(int32_t)(c - 1) / dn < thr)) c--;
        while (c < 0x7FFFFFFFll && (1.0 * (double)(int32_t)c / dn < thr)) c++;
        tc[g] = (uint32_t)c;
    }
}

__device__ __forceinline__ void test_pair(const K3Params& p, uint32_t i, uint32_t j, uint32_t cnt) {
    if (p.tc) {
        if (cnt >= p.tc[i]) emit_pair(p, i, j, cnt);
        if (cnt >= p.tc[j]) emit_pair(p, j, i, cnt);
        return;
    }
    const uint32_t ni = p.sizes[i], nj = p.sizes[j];
    if (ni == 0 || nj == 0) return;
    const uint64_t uni = (uint64_t)ni + (uint64_t)nj - (uint64_t)(int64_t)(int32_t)cnt;
    if (uni == 0) return;
    const double m = 1.0 * (double)(int32_t)cnt;
    const double cij = m / (double)ni;
    const double cji = m / (double)nj;
    if (!(cij < p.thr)) emit_pair(p, i, j, cnt);
    if (!(cji < p.thr)) emit_pair(p, j, i, cnt);
}

template <bool U16>
__device__ __forceinline__ uint32_t acc_add(uint32_t* acc, uint32_t col) {
    if (U16) {
        const uint32_t sh = (col & 1u) << 4;
        const uint32_t old = atomicAdd(&acc[col >> 1], 1u << sh);
        return (old >> sh) & 0xffffu;
    } else {
        return atomicAdd(&acc[col], 1u);
    }
}
template <bool U16>
__device__ __forceinline__ uint32_t acc_take(uint32_t* acc, uint32_t col) {
    if (U16) {
        const uint32_t sh = (col & 1u) << 4;
        const uint32_t old = atomicAnd(&acc[col >> 1], ~(0xffffu << sh));
        return (old >> sh) & 0xffffu;
    } else {
        const uint32_t v = acc[col];
        acc[col] = 0;
        return v;
    }
}

// Work units (row, column tile) come from a global ticket.  A row's critical path would otherwise be a chain of
// dependent global round trips (ticket -> row metadata -> first items), and with a 170 KB accumulator only one
// row is in flight per SM, so the chain is software-pipelined three deep: while unit k is accumulated, every
// thread already holds its first item of unit k+1 in a register, and thread 0 resolves the metadata of unit
// k+2 from a ticket drawn one iteration earlier.
template <bool U16>
__global__ void __launch_bounds__(1024) k3_count_flag(const K3Params p) {
    const uint32_t NT = blockDim.x;   // 256 when several accumulators share an SM, up to 1024 when one CTA owns it
    extern __shared__ uint32_t smem[];
    const uint32_t acc_words = U16 ? (p.tile_w + 1) / 2 : p.tile_w;
    uint32_t* acc = smem;                               // [acc_words] dense row accumulator
    uint32_t* touched = acc + acc_words;                // [K3_TOUCH_CAP]
    uint64_t* longq = (uint64_t*)(touched + K3_TOUCH_CAP + (acc_words & 1u));  // 8-byte aligned
    __shared__ uint32_t s_ntv[2], s_nlongv[2];          // double-buffered by iteration parity: no reset barrier
    __shared__ unsigned long long s_unit[3];            // pipeline slots: unit id, its row, work-list start, length
    __shared__ uint64_t s_ib[3];
    __shared__ uint32_t s_row[3], s_n[3];

    const unsigned long long n_units = (unsigned long long)(p.row_list ? p.n_list : (p.row_end - p.row_begin)) * p.n_tiles;
    // the first two units of a CTA are static; tickets continue from 2 * gridDim.x
    if (threadIdx.x < 2) {
        const unsigned long long u = (unsigned long long)blockIdx.x + (unsigned long long)threadIdx.x * gridDim.x;
        uint32_t row = 0, n = 0;
        uint64_t ib = 0;
        if (u < n_units) {
            const uint32_t ridx = p.n_tiles == 1 ? (uint32_t)u : (uint32_t)(u / p.n_tiles);
            row = p.row_list ? p.row_list[ridx] : p.row_begin + ridx;
            ib = p.list_begin[row];
            n = (uint32_t)p.row_n[row];
        }
        s_unit[threadIdx.x] = u; s_row[threadIdx.x] = row; s_ib[threadIdx.x] = ib; s_n[threadIdx.x] = n;
    }
    unsigned long long tick = 0;
    if (threadIdx.x == 0) {
        s_ntv[0] = 0; s_ntv[1] = 0; s_nlongv[0] = 0; s_nlongv[1] = 0;
        tick = 2ull * gridDim.x + atomicAdd(&p.scal[SC_UNIT], 1ull);
    }
    for (uint32_t c = threadIdx.x; c < acc_words; c += NT) acc[c] = 0;
    __syncthreads();
    uint64_t item_cur = 0;
    if (s_unit[0] < n_units && threadIdx.x < s_n[0]) item_cur = p.row_items[s_ib[0] + threadIdx.x];

    uint32_t cur = 0, par = 0;
    for (;;) {
        const unsigned long long unit = s_unit[cur];
        if (unit >= n_units) break;
        uint32_t& s_nt = s_ntv[par];
        uint32_t& s_nlong = s_nlongv[par];
        const uint32_t nxt = cur == 2 ? 0 : cur + 1, nx2 = nxt == 2 ? 0 : nxt + 1;
        const uint32_t row = s_row[cur];
        const uint64_t ib = s_ib[cur], ie = ib + s_n[cur];
        // this thread's first item of the next unit
        uint64_t item_next = 0;
        if (s_unit[nxt] < n_units && threadIdx.x < s_n[nxt]) item_next = p.row_items[s_ib[nxt] + threadIdx.x];
        // thread 0: metadata of the unit after next (loads issued here, consumed at the bottom of the iteration)
        unsigned long long u2 = 0;
        uint32_t r2 = 0, n2 = 0;
        uint64_t ib2 = 0;
        if (threadIdx.x == 0) {
            u2 = tick;
            s_ntv[par ^ 1] = 0; s_nlongv[par ^ 1] = 0;      // last read before the previous iteration's final barrier
            if (u2 < n_units) {
                const uint32_t ridx = p.n_tiles == 1 ? (uint32_t)u2 : (uint32_t)(u2 / p.n_tiles);
                r2 = p.row_list ? p.row_list[ridx] : p.row_begin + ridx;
                ib2 = p.list_begin[r2];
                n2 = (uint32_t)p.row_n[r2];
                tick = 2ull * gridDim.x + atomicAdd(&p.scal[SC_UNIT], 1ull);
            }
        }
        const uint32_t tile = p.n_tiles == 1 ? 0u : (uint32_t)(unit % p.n_tiles);
        const uint32_t c0 = tile * p.tile_w;
        const uint32_t c1 = min(p.n, c0 + p.tile_w);
        // upper triangle: only columns > row matter
        if (c1 > row + 1 && ie > ib) {
            // ---- accumulate -----------------------------------------------------------------
            // The work list is walked in chunks of one item per thread.  Short posting segments are expanded by the thread that
            // holds the item; long ones (a hash held by thousands of genomes: the dense clusters of a skewed database) are queued
            // and expanded by the whole CTA after every chunk -- a row of such a cluster carries thousands of long segments, and
            // a thread walking 5 000 postings alone is what made the count of config 4 take minutes.
            uint64_t item = item_cur;
            uint32_t long_done = 0;
            for (uint64_t base = ib; base < ie; base += NT) {
                const uint64_t it = base + threadIdx.x;
                if (it < ie) {
                    const uint32_t inl = (uint32_t)item & 3u;
                    if (inl) {                                         // the following genome ids are inside the item
                        for (uint32_t e = 0; e < inl; e++) {
                            const uint32_t g = (uint32_t)(item >> (2 + YG_ITEM_INLINE_BITS * e)) & ((1u << YG_ITEM_INLINE_BITS) - 1u);
                            if (g <= row || g < c0 || g >= c1) continue;
                            if (acc_add<U16>(acc, g - c0) == 0) {
                                const uint32_t k = atomicAdd(&s_nt, 1u);
                                if (k < K3_TOUCH_CAP) touched[k] = g;
                            }
                        }
                    } else {
                        const uint32_t start = (uint32_t)(item >> 32), len = (uint32_t)(item >> 2) & 0x3FFFFFFFu;
                        if (len > K3_LONG_LEN) {
                            longq[(atomicAdd(&s_nlong, 1u) - long_done) & (K3_LONG_CAP - 1)] = item;      // at most NT <= K3_LONG_CAP per chunk
                        } else {
                            for (uint32_t e = 0; e < len; e++) {
                                const uint32_t g = p.post[start + e];
                                if (g <= row || g < c0 || g >= c1) continue;   // g == row: duplicate hash inside the sketch
                                if (acc_add<U16>(acc, g - c0) == 0) {
                                    const uint32_t k = atomicAdd(&s_nt, 1u);
                                    if (k < K3_TOUCH_CAP) touched[k] = g;
                                }
                            }
                        }
                    }
                    if (it + NT < ie) item = p.row_items[it + NT];
                }
                __syncthreads();
                const uint32_t nlong = s_nlong - long_done;
                if (nlong) {                                           // uniform
                    for (uint32_t q = 0; q < nlong; q++) {
                        const uint64_t litem = longq[q];
                        const uint32_t start = (uint32_t)(litem >> 32), len = (uint32_t)(litem >> 2) & 0x3FFFFFFFu;
                        for (uint32_t e = threadIdx.x; e < len; e += NT) {
                            const uint32_t g = p.post[start + e];
                            if (g <= row || g < c0 || g >= c1) continue;
                            if (acc_add<U16>(acc, g - c0) == 0) {
                                const uint32_t k = atomicAdd(&s_nt, 1u);
                                if (k < K3_TOUCH_CAP) touched[k] = g;
                            }
                        }
                    }
                    long_done += nlong;
                    __syncthreads();                                   // the queue slots are reused by the next chunk
                }
            }
            // ---- threshold + compaction (K4), and reset of the accumulator ---------------------
            const uint32_t nt = s_nt;
            if (nt <= K3_TOUCH_CAP) {
                for (uint32_t k = threadIdx.x; k < nt; k += NT) {
                    const uint32_t g = touched[k];
                    const uint32_t cnt = acc_take<U16>(acc, g - c0);
                    test_pair(p, row, g, cnt);
                }
            } else {
                const uint32_t w = c1 - c0;
                for (uint32_t c = threadIdx.x; c < w; c += NT) {
                    const uint32_t cnt = acc_take<U16>(acc, c);
                    if (cnt) test_pair(p, row, c0 + c, cnt);
                }
            }
        }
        // slot nx2 was last read one iteration ago (a barrier lies in between); it is read again after the barrier below
        if (threadIdx.x == 0) { s_unit[nx2] = u2; s_row[nx2] = r2; s_ib[nx2] = ib2; s_n[nx2] = n2; }
        __syncthreads();
        item_cur = item_next;
        cur = nxt;
        par ^= 1;
    }
}

// ---- K3 for large N: one WARP per query row, counts in a small per-warp hash table ------------------
// A dense row accumulator needs N counters (170 KB at 85k genomes => one row in flight per SM, latency
// bound).  A row only ever touches the few genomes it shares hashes with, so each warp keeps
// (column, count) pairs in a 512-slot open-addressing table in shared memory: 48 rows in flight per SM,
// no block-level barrier anywhere.  Rows that touch more distinct columns than the table holds are
// deferred to the dense kernel through an overflow list.
#define K3W_THREADS 256
#define K3W_SLOTS 512
#define K3W_TOUCH 96
#define K3W_LONG 64
#define K3W_EMPTY 0xFFFFFFFFu
#define K3W_ROWS 8           // rows per ticket (a warp's unit of dynamic scheduling)

struct WarpTable {
    uint32_t* keys;     // [K3W_SLOTS]
    uint32_t* cnts;     // [K3W_SLOTS]
    uint32_t* touched;  // [K3W_TOUCH] slots in first-touch order
    uint32_t* ctl;      // [0] = distinct columns so far, [1] = overflow flag
};

__device__ __forceinline__ void wt_insert(const WarpTable& t, uint32_t g) {
    uint32_t slot = (g * 2654435761u) >> 23;
    for (int probe = 0; probe < K3W_SLOTS; probe++) {
        const uint32_t k = *((volatile uint32_t*)&t.keys[slot]);
        if (k == g) { atomicAdd(&t.cnts[slot], 1u); return; }
        if (k == K3W_EMPTY) {
            const uint32_t old = atomicCAS(&t.keys[slot], K3W_EMPTY, g);
            if (old == K3W_EMPTY) {
                const uint32_t idx = atomicAdd(&t.ctl[0], 1u);
                if (idx < K3W_TOUCH) t.touched[idx] = slot;
                if (idx >= (K3W_SLOTS * 3) / 4) t.ctl[1] = 1;
                atomicAdd(&t.cnts[slot], 1u);
                return;
            }
            if (old == g) { atomicAdd(&t.cnts[slot], 1u); return; }
        }
        slot = (slot + 1) & (K3W_SLOTS - 1);
    }
    t.ctl[1] = 1;   // table full
}

__global__ void __launch_bounds__(K3W_THREADS) k3w_count_flag(const K3Params p) {
    extern __shared__ uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int WORDS = 2 * K3W_SLOTS + K3W_TOUCH + 32;
    WarpTable t;
    t.keys = smem + warp * WORDS;
    t.cnts = t.keys + K3W_SLOTS;
    t.touched = t.cnts + K3W_SLOTS;
    t.ctl = t.touched + K3W_TOUCH;
    for (int i = lane; i < K3W_SLOTS; i += 32) { t.keys[i] = K3W_EMPTY; t.cnts[i] = 0; }
    if (lane == 0) { t.ctl[0] = 0; t.ctl[1] = 0; }
    __syncwarp();

    const uint32_t n_rows = p.row_end - p.row_begin;
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&p.scal[SC_UNIT], (unsigned long long)K3W_ROWS);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n_rows) break;
        const uint32_t my_idx = (uint32_t)base + lane;
        const uint32_t my_n = (lane < K3W_ROWS && my_idx < n_rows) ? (uint32_t)p.row_n[p.row_begin + my_idx] : 0u;
        const uint64_t my_ib = my_n ? p.list_begin[p.row_begin + my_idx] : 0ull;
        unsigned todo = __ballot_sync(0xffffffffu, my_n > 0);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t row = p.row_begin + (uint32_t)base + src;
            const uint32_t nit = __shfl_sync(0xffffffffu, my_n, src);
            const uint64_t ib = __shfl_sync(0xffffffffu, my_ib, src);
            // ---- accumulate --------------------------------------------------------------------------
            for (uint32_t it0 = 0; it0 < nit; it0 += 32) {
                const uint32_t it = it0 + lane;
                uint32_t start = 0, len = 0;
                if (it < nit) {
                    const uint64_t item = p.row_items[ib + it];
                    const uint32_t inl = (uint32_t)item & 3u;
                    if (inl) {                                     // ids inline in the item: no posting read at all
                        if (*((volatile uint32_t*)&t.ctl[1]) == 0)
                            for (uint32_t e = 0; e < inl; e++) {
                                const uint32_t g = (uint32_t)(item >> (2 + YG_ITEM_INLINE_BITS * e)) & ((1u << YG_ITEM_INLINE_BITS) - 1u);
                                if (g > row) wt_insert(t, g);
                            }
                    } else {
                        start = (uint32_t)(item >> 32);
                        len = (uint32_t)(item >> 2) & 0x3FFFFFFFu;
                    }
                }
                const bool is_long = len > K3W_LONG;
                if (!is_long && *((volatile uint32_t*)&t.ctl[1]) == 0)
                    for (uint32_t e = 0; e < len; e++) {
                        const uint32_t g = p.post[start + e];
                        if (g > row) wt_insert(t, g);      // g == row: the same hash twice inside the sketch
                    }
                unsigned lm = __ballot_sync(0xffffffffu, is_long);
                while (lm) {
                    const int s2 = __ffs(lm) - 1;
                    lm &= lm - 1;
                    const uint32_t st2 = __shfl_sync(0xffffffffu, start, s2);
                    const uint32_t ln2 = __shfl_sync(0xffffffffu, len, s2);
                    if (*((volatile uint32_t*)&t.ctl[1]) == 0)
                        for (uint32_t e = lane; e < ln2; e += 32) {
                            const uint32_t g = p.post[st2 + e];
                            if (g > row) wt_insert(t, g);
                        }
                }
            }
            __syncwarp();
            // ---- threshold + compaction, table reset -------------------------------------------------------
            const uint32_t nt = t.ctl[0];
            const bool ovf = t.ctl[1] != 0;
            __syncwarp();
            if (ovf) {
                if (lane == 0) p.ovf_rows[atomicAdd(&p.scal[SC_OVF], 1ull)] = row;
                for (int i = lane; i < K3W_SLOTS; i += 32) { t.keys[i] = K3W_EMPTY; t.cnts[i] = 0; }
            } else if (nt <= K3W_TOUCH) {
                for (uint32_t k = lane; k < nt; k += 32) {
                    const uint32_t slot = t.touched[k];
                    const uint32_t g = t.keys[slot], c = t.cnts[slot];
                    t.keys[slot] = K3W_EMPTY; t.cnts[slot] = 0;
                    test_pair(p, row, g, c);
                }
            } else {
                for (int slot = lane; slot < K3W_SLOTS; slot += 32) {
                    const uint32_t g = t.keys[slot];
                    if (g != K3W_EMPTY) {
                        const uint32_t c = t.cnts[slot];
                        t.keys[slot] = K3W_EMPTY; t.cnts[slot] = 0;
                        test_pair(p, row, g, c);
                    }
                }
            }
            if (lane == 0) { t.ctl[0] = 0; t.ctl[1] = 0; }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(256) k_pack_pairs(const uint64_t* __restrict__ key, const uint32_t* __restrict__ cnt,
                                                     uint64_t n, int shift, ygpu_pair* __restrict__ out) {
    const uint64_t jmask = (1ull << shift) - 1ull;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t kk = key[k];
        ygpu_pair pr;
        pr.i = (int32_t)(kk >> shift);
        pr.j = (int32_t)(kk & jmask);
        pr.count = (int32_t)cnt[k];
        out[k] = pr;
    }
}

__global__ void __launch_bounds__(256) k_unpack_pairs(const ygpu_pair* __restrict__ in, uint64_t n, int shift, uint64_t* __restrict__ key,
                                                       uint32_t* __restrict__ cnt) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const ygpu_pair pr = in[k];
        key[k] = ((uint64_t)(uint32_t)pr.i << shift) | (uint64_t)(uint32_t)pr.j;
        cnt[k] = (uint32_t)pr.count;
    }
}

static int ensure_out(ygpu_ctx* ctx, uint64_t cap);

static int pair_key_shift(const ygpu_ctx* ctx) {     // bits of a genome id (at least 1)
    int b = 1;
    while (b < 32 && ((uint64_t)ctx->n >> b) != 0) b++;
    return b;
}

// order a device-resident pair list by (i, j) in place (the gathered lists of several ranks interleave)
int ygpu_sort_pairs_device(ygpu_ctx* ctx, ygpu_pair* d_pairs, uint64_t n) {
    if (n < 2) return 0;
    cudaStream_t st = ctx->stream;
    YG_CHECK(ensure_out(ctx, std::max<uint64_t>(ctx->out_cap, n)));
    const int shift = pair_key_shift(ctx);
    k_unpack_pairs<<<grid_for(ctx, n, 256), 256, 0, st>>>(d_pairs, n, shift, ctx->d_out_key, ctx->d_out_cnt);
    YG_CUDA(ctx, cudaGetLastError());
    size_t tb = 0;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_out_key, ctx->d_out_key2, ctx->d_out_cnt, ctx->d_out_cnt2, (int64_t)n, 0, 2 * shift, st));
    YG_CHECK(ygpu_temp_reserve(ctx, tb));
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, ctx->d_out_key, ctx->d_out_key2, ctx->d_out_cnt, ctx->d_out_cnt2, (int64_t)n, 0, 2 * shift, st));
    k_pack_pairs<<<grid_for(ctx, n, 256), 256, 0, st>>>(ctx->d_out_key2, ctx->d_out_cnt2, n, shift, d_pairs);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches += 2;
    ctx->tm.n_library_launches += 2 + (2 * shift + 7) / 8;
    return 0;
}

static int ensure_out(ygpu_ctx* ctx, uint64_t cap) {
    if (cap <= ctx->out_cap) return 0;
    YG_CHECK(dev_alloc(ctx, &ctx->d_out_key, cap));
    YG_CHECK(dev_alloc(ctx, &ctx->d_out_cnt, cap));
    YG_CHECK(dev_alloc(ctx, &ctx->d_out_key2, cap));
    YG_CHECK(dev_alloc(ctx, &ctx->d_out_cnt2, cap));
    ctx->out_cap = cap;
    return 0;
}

// count + flag + sort on the device; the sorted pairs stay resident in ctx->d_pairs
static int pairwise_device(ygpu_ctx* ctx, double threshold, uint32_t row_begin, uint32_t row_end, uint64_t* n_out) {
    *n_out = 0;
    ctx->n_pairs = 0;
    if (!ctx->indexed) return ygpu_fail(ctx, YGPU_ERR_STATE, "pairwise_flag: build_index first");
    if (row_begin > row_end || row_end > ctx->n) return ygpu_fail(ctx, YGPU_ERR_ARG, "bad row range [%u,%u) of %u", row_begin, row_end, ctx->n);
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint32_t n = ctx->n;
    uint64_t npairs = 0;

    if (ctx->n_items && row_end > row_begin) {
        // ---- dense accumulator geometry ---------------------------------------------------------
        const uint32_t fixed = K3_TOUCH_CAP * 4 + K3_LONG_CAP * 8 + 64;
        const uint32_t budget = (uint32_t)ctx->smem_optin - fixed - 1024;
        const bool u16_ok = !ctx->stats.has_duplicates && ctx->stats.max_sketch <= 65535u;
        bool use_u16 = false;
        uint32_t tile_w = n;
        if ((uint64_t)n * 4 > budget) {
            if (u16_ok && (uint64_t)n * 2 <= budget) use_u16 = true;
            else if (u16_ok) { use_u16 = true; tile_w = (budget / 2) & ~1u; }
            else tile_w = budget / 4;
        }
        if (ctx->force_u16 && u16_ok) use_u16 = true;                                       // test hook
        if (ctx->force_tile_w && ctx->force_tile_w < tile_w) tile_w = ctx->force_tile_w;   // test hook
        if (tile_w < 2) tile_w = 2;
        const uint32_t n_tiles = (n + tile_w - 1) / tile_w;
        const uint32_t acc_words = use_u16 ? (tile_w + 1) / 2 : tile_w;
        const size_t smem = (size_t)(acc_words + (acc_words & 1u)) * 4 + fixed;
        auto kern = use_u16 ? k3_count_flag<true> : k3_count_flag<false>;
        YG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 0;
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, K3_THREADS, smem));
        if (occ < 1) return ygpu_fail(ctx, YGPU_ERR_CUDA, "k3_count_flag does not fit: smem %zu", smem);
        // threads per CTA: when shared memory allows only 1-2 row accumulators per SM, give each CTA more
        // warps so a row's work list is walked with more loads in flight
        const int k3_threads = occ >= 4 ? 256 : (occ >= 2 ? 512 : 1024);
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, k3_threads, smem));
        if (occ < 1) return ygpu_fail(ctx, YGPU_ERR_CUDA, "k3_count_flag does not fit: smem %zu", smem);
        // the warp-per-row kernel is selectable (option count_kernel = 2); measured slower than the dense
        // kernel on cluster-shaped databases (rows carry ~700 work items: one warp walks them too slowly)
        const bool use_warp = ctx->count_kernel == 2;
        const size_t smem_w = (size_t)(K3W_THREADS / 32) * (2 * K3W_SLOTS + K3W_TOUCH + 32) * 4;
        int occ_w = 0;
        if (use_warp) {
            YG_CUDA(ctx, cudaFuncSetAttribute(k3w_count_flag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
            YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_w, k3w_count_flag, K3W_THREADS, smem_w));
            if (occ_w < 1) return ygpu_fail(ctx, YGPU_ERR_CUDA, "k3w_count_flag does not fit");
            YG_CHECK(dev_alloc(ctx, &ctx->d_ovf_rows, (uint64_t)n + 1));
        }

        uint64_t cap = std::max<uint64_t>(ctx->out_cap, std::max<uint64_t>(1u << 20, 8ull * n));
        for (int attempt = 0; attempt < 2; attempt++) {
            YG_CHECK(ensure_out(ctx, cap));
            K3Params p{};
            p.list_begin = ctx->d_row_begin; p.row_n = ctx->d_row_cnt; p.row_items = ctx->d_row_items; p.post = ctx->d_post; p.sizes = ctx->d_sizes;
            p.n = n; p.row_begin = row_begin; p.row_end = row_end; p.tile_w = tile_w; p.n_tiles = n_tiles;
            p.thr = threshold; p.out_key = ctx->d_out_key; p.out_cnt = ctx->d_out_cnt; p.out_cap = ctx->out_cap;
            p.scal = ctx->d_scalars; p.row_list = nullptr; p.n_list = 0; p.ovf_rows = ctx->d_ovf_rows;
            p.key_shift = pair_key_shift(ctx);
            p.tc = nullptr;
            if (!ctx->stats.has_duplicates && ctx->count_thresholds != 0) {
                YG_CHECK(dev_alloc(ctx, &ctx->d_tc, n));
                k4_thresholds<<<grid_for(ctx, n, 256), 256, 0, st>>>(ctx->d_sizes, n, threshold, ctx->d_tc);
                YG_CUDA(ctx, cudaGetLastError());
                ctx->tm.n_kernel_launches++;
                p.tc = ctx->d_tc;
            }
            YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SC_OUT], 0, 2 * sizeof(unsigned long long), st));
            YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SC_OVF], 0, sizeof(unsigned long long), st));
            YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
            unsigned long long cnt = 0, novf = 0;
            if (use_warp) {
                const unsigned long long chunks = ((unsigned long long)(row_end - row_begin) + K3W_ROWS - 1) / K3W_ROWS;
                const int grid_w = (int)std::max<unsigned long long>(1, std::min<unsigned long long>((unsigned long long)ctx->num_sms * occ_w,
                                                                                                     (chunks + 7) / 8));
                k3w_count_flag<<<grid_w, K3W_THREADS, smem_w, st>>>(p);
                YG_CUDA(ctx, cudaGetLastError());
                ctx->tm.n_kernel_launches++;
                YG_CUDA(ctx, cudaMemcpyAsync(&novf, &ctx->d_scalars[SC_OVF], sizeof novf, cudaMemcpyDeviceToHost, st));
                YG_CUDA(ctx, cudaStreamSynchronize(st));
                if (novf) {       // rows with too many distinct columns for a warp table: dense kernel on that list
                    p.row_list = ctx->d_ovf_rows; p.n_list = (uint32_t)novf;
                    YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SC_UNIT], 0, sizeof(unsigned long long), st));
                    const int grid = (int)std::min<unsigned long long>((unsigned long long)ctx->num_sms * occ, novf * n_tiles);
                    kern<<<grid, k3_threads, smem, st>>>(p);
                    YG_CUDA(ctx, cudaGetLastError());
                    ctx->tm.n_kernel_launches++;
                }
            } else {
                const unsigned long long units = (unsigned long long)(row_end - row_begin) * n_tiles;
                const int grid = (int)std::min<unsigned long long>((unsigned long long)ctx->num_sms * occ, units);
                kern<<<grid, k3_threads, smem, st>>>(p);
                YG_CUDA(ctx, cudaGetLastError());
                ctx->tm.n_kernel_launches++;
            }
            YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));
            YG_CUDA(ctx, cudaMemcpyAsync(&cnt, &ctx->d_scalars[SC_OUT], sizeof cnt, cudaMemcpyDeviceToHost, st));
            YG_CUDA(ctx, cudaStreamSynchronize(st));
            ctx->tm.ms_count += elapsed(ctx, 0, 1);
            ctx->tm.n_count_launches++;
            ctx->last_count_kernel = use_warp ? 2 : 1;
            ctx->last_count_overflow_rows = novf;
            ctx->last_count_tile_w = tile_w;
            ctx->last_count_n_tiles = n_tiles;
            ctx->last_count_u16 = use_u16 ? 1 : 0;
            npairs = cnt;
            if (npairs <= ctx->out_cap) break;
            if (attempt == 1) return ygpu_fail(ctx, YGPU_ERR_CUDA, "pair buffer overflow after resize");
            cap = npairs + 1024;
        }
    }
    if (npairs) {
        // order by (i, j): the reference emits row-major (main.cpp:274-275).  The sharded step orders the gathered lists of
        // all ranks once instead (ctx->skip_pair_sort): here the records are only packed.
        YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
        const int shift = pair_key_shift(ctx);
        const uint64_t* keys = ctx->d_out_key;
        const uint32_t* cnts = ctx->d_out_cnt;
        if (!ctx->skip_pair_sort) {
            size_t tb = 0;
            YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_out_key, ctx->d_out_key2, ctx->d_out_cnt,
                                                         ctx->d_out_cnt2, (int64_t)npairs, 0, 2 * shift, st));
            YG_CHECK(ygpu_temp_reserve(ctx, tb));
            tb = ctx->temp_bytes;
            YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, ctx->d_out_key, ctx->d_out_key2, ctx->d_out_cnt,
                                                         ctx->d_out_cnt2, (int64_t)npairs, 0, 2 * shift, st));
            ctx->tm.n_library_launches += 2 + (2 * shift + 7) / 8;
            keys = ctx->d_out_key2;
            cnts = ctx->d_out_cnt2;
        }
        if (npairs > ctx->pairs_cap) {
            if (ctx->d_pairs) cudaFree(ctx->d_pairs);
            ctx->d_pairs = nullptr; ctx->pairs_cap = 0;
            YG_CUDA(ctx, cudaMalloc(&ctx->d_pairs, (npairs + 1024) * sizeof(ygpu_pair)));
            ctx->pairs_cap = npairs + 1024;
        }
        k_pack_pairs<<<grid_for(ctx, npairs, 256), 256, 0, st>>>(keys, cnts, npairs, shift, ctx->d_pairs);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
        YG_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        ctx->tm.ms_pairsort += elapsed(ctx, 2, 3);
    }
    ctx->n_pairs = npairs;
    *n_out = npairs;
    return 0;
}

extern "C" int ygpu_pairwise_flag_device(ygpu_ctx* ctx, double threshold, uint32_t row_begin, uint32_t row_end, uint64_t* n_out) {
    if (!ctx || !n_out) return YGPU_ERR_ARG;
    return pairwise_device(ctx, threshold, row_begin, row_end, n_out);
}

extern "C" int ygpu_pairs_copy(ygpu_ctx* ctx, void* dst, int dst_is_device) {
    if (!ctx || (!dst && ctx->n_pairs)) return YGPU_ERR_ARG;
    if (!ctx->n_pairs) return 0;
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    YG_CUDA(ctx, cudaMemcpyAsync(dst, ctx->d_pairs, ctx->n_pairs * sizeof(ygpu_pair),
                                 dst_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    if (!dst_is_device) ctx->tm.ms_d2h += elapsed(ctx, 2, 3);
    return 0;
}

extern "C" int ygpu_pairwise_flag(ygpu_ctx* ctx, double threshold, uint32_t row_begin, uint32_t row_end,
                                  ygpu_pair** out, uint64_t* n_out) {
    if (!ctx || !out || !n_out) return YGPU_ERR_ARG;
    *out = nullptr;
    *n_out = 0;
    uint64_t npairs = 0;
    YG_CHECK(pairwise_device(ctx, threshold, row_begin, row_end, &npairs));
    ygpu_pair* host = (ygpu_pair*)malloc(std::max<uint64_t>(npairs, 1) * sizeof(ygpu_pair));
    if (!host) return ygpu_fail(ctx, YGPU_ERR_NOMEM, "malloc(%llu pairs)", (unsigned long long)npairs);
    const int rc = ygpu_pairs_copy(ctx, host, 0);
    if (rc) { free(host); return rc; }
    *out = host;
    *n_out = npairs;
    return 0;
}

// CUDA-event stopwatch on the context's stream (the stream every kernel of this library is
// launched on), for callers that time whole steps from outside.
extern "C" int ygpu_mark(ygpu_ctx* ctx, int slot) {
    if (!ctx || slot < 0 || slot > 3) return YGPU_ERR_ARG;
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[4 + slot], ctx->stream));
    return 0;
}
extern "C" int ygpu_elapsed_ms(ygpu_ctx* ctx, int slot_a, int slot_b, double* ms) {
    if (!ctx || !ms || slot_a < 0 || slot_a > 3 || slot_b < 0 || slot_b > 3) return YGPU_ERR_ARG;
    YG_CUDA(ctx, cudaEventSynchronize(ctx->ev[4 + slot_b]));
    float f = 0.f;
    YG_CUDA(ctx, cudaEventElapsedTime(&f, ctx->ev[4 + slot_a], ctx->ev[4 + slot_b]));
    *ms = (double)f;
    return 0;
}
extern "C" int ygpu_set_option(ygpu_ctx* ctx, const char* name, int64_t value) {
    if (!ctx || !name) return YGPU_ERR_ARG;
    if (!strcmp(name, "force_tile_w")) { ctx->force_tile_w = (uint32_t)value; return 0; }
    if (!strcmp(name, "force_u16")) { ctx->force_u16 = (int)value; return 0; }
    if (!strcmp(name, "index_path")) { ctx->index_path = (int)value; return 0; }
    if (!strcmp(name, "count_kernel")) { ctx->count_kernel = (int)value; return 0; }
    if (!strcmp(name, "big_buckets")) { ctx->big_buckets = (int)value; return 0; }
    if (!strcmp(name, "group_kernel")) { ctx->group_kernel = (int)value; return 0; }
    if (!strcmp(name, "run_path")) { ctx->run_path = (int)value; return 0; }
    if (!strcmp(name, "sketch_kernel")) { ctx->sketch_kernel = (int)value; return 0; }
    if (!strcmp(name, "stream_chunk_bytes")) {
        if (value < 1 || value > (int64_t)YG_STREAM_CHUNK_MAX) return ygpu_fail(ctx, YGPU_ERR_ARG, "stream_chunk_bytes must lie in [1, %llu]", (unsigned long long)YG_STREAM_CHUNK_MAX);
        ctx->stream_chunk_bytes = (uint64_t)value;
        return 0;
    }
    if (!strcmp(name, "group_ctas")) { ctx->group_ctas = (int)value; return 0; }
    if (!strcmp(name, "count_thresholds")) { ctx->count_thresholds = (int)value; return 0; }
    return ygpu_fail(ctx, YGPU_ERR_ARG, "unknown option %s", name);
}

extern "C" int ygpu_get_option(ygpu_ctx* ctx, const char* name, int64_t* out) {
    if (!ctx || !name || !out) return YGPU_ERR_ARG;
    if (!strcmp(name, "last_count_kernel")) { *out = ctx->last_count_kernel; return 0; }
    if (!strcmp(name, "last_count_overflow_rows")) { *out = (int64_t)ctx->last_count_overflow_rows; return 0; }
    if (!strcmp(name, "last_count_tile_w")) { *out = ctx->last_count_tile_w; return 0; }
    if (!strcmp(name, "last_count_n_tiles")) { *out = ctx->last_count_n_tiles; return 0; }
    if (!strcmp(name, "last_count_u16")) { *out = ctx->last_count_u16; return 0; }
    if (!strcmp(name, "last_group2_grid")) { *out = ctx->last_group2_grid; return 0; }
    if (!strcmp(name, "last_group_grid")) { *out = ctx->last_group_grid; return 0; }
    if (!strcmp(name, "last_big_chunks")) { *out = ctx->last_big_chunks; return 0; }
    return ygpu_fail(ctx, YGPU_ERR_ARG, "unknown option %s", name);
}

// increments each row performs = sum over its work items of how many postings follow (one warp per row)
__global__ void __launch_bounds__(256) k_row_work(const uint64_t* __restrict__ list_begin, const unsigned long long* __restrict__ row_n,
                                                   const uint64_t* __restrict__ row_items, uint32_t n, uint64_t* __restrict__ row_work) {
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += (gridDim.x * blockDim.x) >> 5) {
        const uint64_t ib = list_begin[row];
        const uint64_t cnt = row_n[row];
        unsigned long long s = 0;
        for (uint64_t k = lane; k < cnt; k += 32) {
            const uint64_t item = row_items[ib + k];
            const uint32_t c = (uint32_t)item & 3u;
            s += c ? c : ((uint32_t)(item >> 2) & 0x3FFFFFFFu);
        }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
        if (lane == 0) row_work[row] = s;
    }
}

extern "C" int ygpu_row_partition(ygpu_ctx* ctx, uint32_t nparts, uint32_t* bounds) {
    if (!ctx || !bounds || nparts == 0) return YGPU_ERR_ARG;
    if (!ctx->indexed) return ygpu_fail(ctx, YGPU_ERR_STATE, "row_partition: build_index first");
    const uint32_t n = ctx->n;
    if (nparts == 1) { bounds[0] = 0; bounds[1] = n; return 0; }
    if (!ctx->row_work_valid && n && ctx->n_items) {
        YG_CUDA(ctx, cudaSetDevice(ctx->device));
        k_row_work<<<grid_for(ctx, (uint64_t)n * 32, 256), 256, 0, ctx->stream>>>(ctx->d_row_begin, ctx->d_row_cnt, ctx->d_row_items, n, ctx->d_row_work);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
        YG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->row_work_valid = true;
    }
    std::vector<uint64_t> work(n);
    if (n) YG_CUDA(ctx, cudaMemcpy(work.data(), ctx->d_row_work, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    // cost model: increments + a per-row constant (launching / scanning a row is not free)
    long double total = 0;
    for (uint32_t g = 0; g < n; g++) total += (long double)work[g] + 64.0L;
    bounds[0] = 0;
    long double acc = 0;
    uint32_t part = 1;
    for (uint32_t g = 0; g < n && part < nparts; g++) {
        acc += (long double)work[g] + 64.0L;
        while (part < nparts && acc >= total * part / nparts) bounds[part++] = g + 1;
    }
    while (part < nparts) bounds[part++] = n;
    bounds[nparts] = n;
    return 0;
}
