// libyachtgpu -- streamed FASTA / FASTQ sketching (DESIGN §3 K7, "stream").
//
// The raw text of a file goes to the device chunk by chunk; per chunk:
//   k_sq_pre      : per byte, '\n' flag and "index if not '\r'"
//   scans         : line number of every byte (exclusive sum of '\n'), nearest byte before it that is not '\r' (max scan)
//   k_sq_first    : the first byte of every line (seq_stream.cuh: ysq_is_first)
//   k_sq_classify : role of the byte's line, per-byte flags (sequence / record start / name); FASTQ structure checks
//   scans         : output positions of the sequence and name bytes, record ordinals
//   k_sq_scatter  : compacted hashing buffer = carried bases of the open record + this chunk's sequence bytes, one '\n'
//                   per record start; record start offsets; name bytes
//   k_sq_finish   : chunk totals, the carried state for the next chunk (line number, open line, last k - 1 bases)
// then the K7 hashing kernels (ygpu_sketch_hash_device) and a merge of the chunk's kept hashes into the resident sketch:
// radix sort of (resident + new) by hash, stably by record, and a reduction that adds the abundances.
#include "common.cuh"
#include "seq_stream.cuh"

#include <cub/cub.cuh>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr int SQ_NT = 256;

struct ysq_chunk {
    uint64_t n_out;     // bytes of the compacted buffer (carried bases included)
    uint64_t n_rec;     // records started in the chunk
    uint64_t n_name;    // name bytes of the chunk
    uint64_t n_nl;      // '\n' bytes of the chunk
};

struct StreamState {
    bool active = false;
    int ksize = 0;
    uint64_t max_hash = 0;
    uint32_t seed = 0;
    int mode = YGPU_STREAM_WHOLE;
    uint64_t cap = 0;                 // raw bytes per chunk
    bool file_started = false;        // the current file's format is known
    int fmt = YSQ_FMT_NONE;
    uint8_t* h_stage = nullptr;       // page-locked: a chunk gathered from small feeds
    uint64_t staged = 0;
    ysq_state* h_state = nullptr;     // page-locked mirror of the device state, current after every chunk
    ysq_chunk* h_chunk = nullptr;
    ysq_state* d_state = nullptr;
    ysq_chunk* d_chunk = nullptr;
    // per-chunk buffers
    uint8_t* d_raw = nullptr;
    uint32_t* d_nl = nullptr;
    uint32_t* d_line = nullptr;
    int32_t* d_nr = nullptr;
    int32_t* d_prev = nullptr;
    uint8_t* d_first = nullptr;
    uint8_t* d_flags = nullptr;
    uint64_t* d_val_a = nullptr;
    uint64_t* d_pos_a = nullptr;
    uint32_t* d_val_b = nullptr;
    uint32_t* d_pos_b = nullptr;
    uint8_t* d_out = nullptr;
    uint64_t* d_off = nullptr;
    uint8_t* d_names = nullptr;
    uint32_t* d_name_start = nullptr;
    // resident sketch: hash, (record << 32) | abundance, sorted by (record, hash)
    uint64_t* d_rh = nullptr;
    uint64_t* d_rv = nullptr;
    uint64_t n_res = 0;
    uint64_t* d_ah = nullptr;
    uint64_t* d_av = nullptr;
    uint64_t* d_bh = nullptr;
    uint64_t* d_bv = nullptr;
    uint32_t* d_mflag = nullptr;
    uint32_t* d_mpos = nullptr;
    // names on the host
    std::string names;
    std::vector<uint64_t> name_off;
    std::vector<uint32_t> h_name_start;
    ygpu_stream_stats st = {};
    cudaEvent_t ev[6] = {};
};

StreamState* sq_get(ygpu_ctx* ctx) {
    if (!ctx->seq_stream) ctx->seq_stream = new StreamState();
    return (StreamState*)ctx->seq_stream;
}

struct MaxI32 {
    __device__ __forceinline__ int32_t operator()(int32_t a, int32_t b) const { return a > b ? a : b; }
};

__global__ void __launch_bounds__(SQ_NT) k_sq_pre(const uint8_t* __restrict__ raw, uint64_t n, uint32_t* __restrict__ nl,
                                                   int32_t* __restrict__ nr) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t c = raw[i];
        nl[i] = c == '\n' ? 1u : 0u;
        nr[i] = c != '\r' ? (int32_t)i : -1;
    }
}

__device__ __forceinline__ int sq_prev_byte(const uint8_t* raw, const int32_t* prev_incl, uint64_t i) {
    if (i == 0) return -1;
    const int32_t q = prev_incl[i - 1];
    return q < 0 ? -1 : (int)raw[q];
}

__global__ void __launch_bounds__(SQ_NT) k_sq_first(const uint8_t* __restrict__ raw, uint64_t n, const uint32_t* __restrict__ line,
                                                     const int32_t* __restrict__ prev_incl, const ysq_state* __restrict__ s,
                                                     uint8_t* __restrict__ first) {
    const bool open_has = s->open_first != 0;
    if (blockIdx.x == 0 && threadIdx.x == 0 && open_has) first[0] = (uint8_t)s->open_first;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t c = raw[i];
        if (ysq_is_first(c, sq_prev_byte(raw, prev_incl, i), open_has)) first[line[i]] = c;
    }
}

__global__ void __launch_bounds__(SQ_NT) k_sq_classify(const uint8_t* __restrict__ raw, uint64_t n, const uint32_t* __restrict__ line,
                                                        const int32_t* __restrict__ prev_incl, const uint8_t* __restrict__ first,
                                                        ysq_state* s, int want_names, uint8_t* __restrict__ flags,
                                                        uint64_t* __restrict__ val_a, uint32_t* __restrict__ val_b) {
    const bool open_has = s->open_first != 0;
    const int fmt = (int)s->fmt;
    const uint64_t line0 = s->line;
    // names: every record in per-record mode (want_names = 2), FASTA records in whole mode (1)
    const bool names = want_names == 2 || (want_names == 1 && fmt == YSQ_FASTA);
    uint64_t last1 = 0, bad = ~0ull, bad_empty = ~0ull;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t c = raw[i];
        const uint32_t L = line[i];
        const uint64_t G = line0 + L;
        const uint32_t f = first[L];
        const bool is_first = ysq_is_first(c, sq_prev_byte(raw, prev_incl, i), open_has);
        const uint32_t fl = ysq_byte_flags(c, ysq_line_role(fmt, f, G), is_first, names);
        flags[i] = (uint8_t)fl;
        val_a[i] = (uint64_t)(fl & YSQ_F_SEQ) | ((fl & YSQ_F_REC) ? (1ull << 32) : 0ull);
        val_b[i] = (fl & YSQ_F_NAME) ? 1u : 0u;
        if (fmt == YSQ_FASTQ) {
            if (is_first) {
                last1 = G + 1 > last1 ? G + 1 : last1;
                if (ysq_fastq_bad(c, G) && G < bad) bad = G;
            } else if (c == '\n' && f == 0 && ysq_fastq_bad(0, G) && G < bad_empty) {
                bad_empty = G;
            }
        }
    }
    if (fmt == YSQ_FASTQ) {
        if (last1) atomicMax((unsigned long long*)&s->last_nonempty1, (unsigned long long)last1);
        if (bad != ~0ull) atomicMin((unsigned long long*)&s->first_bad, (unsigned long long)bad);
        if (bad_empty != ~0ull) atomicMin((unsigned long long*)&s->first_bad_empty, (unsigned long long)bad_empty);
    }
}

__global__ void __launch_bounds__(SQ_NT) k_sq_scatter(const uint8_t* __restrict__ raw, uint64_t n, const uint8_t* __restrict__ flags,
                                                       const uint64_t* __restrict__ pos_a, const uint32_t* __restrict__ pos_b,
                                                       const ysq_state* __restrict__ s, uint8_t* __restrict__ out, uint64_t* __restrict__ off,
                                                       uint8_t* __restrict__ names, uint32_t* __restrict__ name_start) {
    const uint64_t nc = s->n_carry;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t fl = flags[i];
        if (!fl) continue;
        const uint8_t c = raw[i];
        if (fl & YSQ_F_SEQ) {
            const uint64_t o = nc + (uint32_t)pos_a[i];
            out[o] = ysq_out_byte(c, fl);
            if (fl & YSQ_F_REC) {
                const uint32_t r = (uint32_t)(pos_a[i] >> 32);
                off[1 + r] = o;
                if (name_start) name_start[r] = pos_b[i];
            }
        }
        if (fl & YSQ_F_NAME) names[pos_b[i]] = c;
    }
}

// one thread: totals of the chunk and the state carried into the next one
__global__ void k_sq_finish(const uint8_t* __restrict__ raw, uint64_t n, const uint32_t* __restrict__ line,
                            const uint8_t* __restrict__ flags, const uint64_t* __restrict__ pos_a, const uint32_t* __restrict__ pos_b,
                            const uint8_t* __restrict__ first, const uint8_t* __restrict__ out, uint64_t* __restrict__ off,
                            ysq_state* s, ysq_chunk* ch, int k) {
    const uint64_t last = n - 1;
    const uint32_t fl = flags[last];
    const uint64_t n_nl = (uint64_t)line[last] + (raw[last] == '\n' ? 1 : 0);
    const uint64_t a = pos_a[last] + ((uint64_t)(fl & YSQ_F_SEQ) | ((fl & YSQ_F_REC) ? (1ull << 32) : 0ull));
    const uint64_t n_rec = a >> 32;
    const uint64_t n_out = s->n_carry + (uint32_t)a;
    ch->n_out = n_out;
    ch->n_rec = n_rec;
    ch->n_name = pos_b ? (uint64_t)pos_b[last] + ((fl & YSQ_F_NAME) ? 1 : 0) : 0;
    ch->n_nl = n_nl;
    off[0] = 0;
    off[n_rec + 1] = n_out;
    ysq_advance(s, n_nl, n_rec, first[n_nl], out, n_out, n_rec ? off[n_rec] + 1 : 0, k);
}

__global__ void __launch_bounds__(256) k_sq_pack(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sid, uint64_t m,
                                                  uint32_t sid_base, int whole, uint64_t* __restrict__ h, uint64_t* __restrict__ v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t rec = whole ? 0u : sid[i] + sid_base;      // local sketch 0 is the record open at the chunk's start
        h[i] = key[i];
        v[i] = ((uint64_t)rec << 32) | 1ull;
    }
}

__global__ void __launch_bounds__(256) k_sq_heads(const uint64_t* __restrict__ h, const uint64_t* __restrict__ v, uint64_t m,
                                                   uint32_t* __restrict__ flag) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x)
        flag[i] = (i == 0 || h[i] != h[i - 1] || (v[i] >> 32) != (v[i - 1] >> 32)) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_sq_reduce(const uint64_t* __restrict__ h, const uint64_t* __restrict__ v,
                                                    const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos_incl, uint64_t m,
                                                    uint64_t* __restrict__ rh, unsigned long long* rv) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t d = pos_incl[i] - 1;
        const uint64_t x = v[i];
        if (flag[i]) rh[d] = h[i];
        atomicAdd(&rv[d], (unsigned long long)((flag[i] ? (x & ~0xFFFFFFFFull) : 0ull) + (x & 0xFFFFFFFFull)));
    }
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

int sq_fail(ygpu_ctx* ctx, StreamState* S, int code, const char* msg) {
    S->active = false;
    return ygpu_fail(ctx, code, "%s", msg);
}

int sq_alloc_chunk(ygpu_ctx* ctx, StreamState* S) {
    const uint64_t n = S->cap;
    YG_CHECK(dev_alloc(ctx, &S->d_raw, n));
    YG_CHECK(dev_alloc(ctx, &S->d_nl, n));
    YG_CHECK(dev_alloc(ctx, &S->d_line, n));
    YG_CHECK(dev_alloc(ctx, &S->d_nr, n));
    YG_CHECK(dev_alloc(ctx, &S->d_prev, n));
    YG_CHECK(dev_alloc(ctx, &S->d_first, n + 1));
    YG_CHECK(dev_alloc(ctx, &S->d_flags, n));
    YG_CHECK(dev_alloc(ctx, &S->d_val_a, n));
    YG_CHECK(dev_alloc(ctx, &S->d_pos_a, n));
    YG_CHECK(dev_alloc(ctx, &S->d_val_b, n));
    YG_CHECK(dev_alloc(ctx, &S->d_pos_b, n));
    YG_CHECK(dev_alloc(ctx, &S->d_out, n + YSQ_CARRY_MAX + YG_SKETCH_PAD));
    YG_CHECK(dev_alloc(ctx, &S->d_off, n + 2));
    YG_CHECK(dev_alloc(ctx, &S->d_names, n));
    YG_CHECK(dev_alloc(ctx, &S->d_name_start, n));
    YG_CHECK(dev_alloc(ctx, &S->d_state, 1));
    YG_CHECK(dev_alloc(ctx, &S->d_chunk, 1));
    size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, t1, S->d_nl, S->d_line, (int64_t)n, ctx->stream));
    YG_CUDA(ctx, cub::DeviceScan::InclusiveScan(nullptr, t2, S->d_nr, S->d_prev, MaxI32(), (int64_t)n, ctx->stream));
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, t3, S->d_val_a, S->d_pos_a, (int64_t)n, ctx->stream));
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, t4, S->d_val_b, S->d_pos_b, (int64_t)n, ctx->stream));
    return ygpu_temp_reserve(ctx, std::max(std::max(t1, t2), std::max(t3, t4)));
}

// Kept hashes of the chunk (sketch scratch) -> resident sketch.
int sq_merge(ygpu_ctx* ctx, StreamState* S, uint64_t m, uint32_t sid_base) {
    cudaStream_t st = ctx->stream;
    uint64_t* d_key;
    uint32_t* d_sid;
    ygpu_sketch_survivors(ctx, &d_key, &d_sid);
    const uint64_t r = S->n_res, t = r + m;
    if (t >= (1ull << 32)) return sq_fail(ctx, S, YGPU_ERR_ARG, "ygpu_stream: more than 2^32 kept hashes");
    YG_CHECK(dev_alloc(ctx, &S->d_ah, t));
    YG_CHECK(dev_alloc(ctx, &S->d_av, t));
    YG_CHECK(dev_alloc(ctx, &S->d_bh, t));
    YG_CHECK(dev_alloc(ctx, &S->d_bv, t));
    YG_CHECK(dev_alloc(ctx, &S->d_mflag, t));
    YG_CHECK(dev_alloc(ctx, &S->d_mpos, t));
    if (r) {
        YG_CUDA(ctx, cudaMemcpyAsync(S->d_ah, S->d_rh, r * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
        YG_CUDA(ctx, cudaMemcpyAsync(S->d_av, S->d_rv, r * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    }
    const bool whole = S->mode == YGPU_STREAM_WHOLE;
    k_sq_pack<<<grid_for(ctx, m, 256), 256, 0, st>>>(d_key, d_sid, m, sid_base, whole ? 1 : 0, S->d_ah + r, S->d_av + r);
    YG_CUDA(ctx, cudaGetLastError());
    int hash_bits = 64;
    while (hash_bits > 1 && !((S->max_hash >> (hash_bits - 1)) & 1)) hash_bits--;
    int sid_bits = 1;
    while (sid_bits < 32 && (1ull << sid_bits) < S->h_state->n_records + 1) sid_bits++;
    size_t tb1 = 0, tb2 = 0, tb3 = 0;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb1, S->d_ah, S->d_bh, S->d_av, S->d_bv, (int64_t)t, 0, hash_bits, st));
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb2, S->d_bv, S->d_av, S->d_bh, S->d_ah, (int64_t)t, 32, 32 + sid_bits, st));
    YG_CUDA(ctx, cub::DeviceScan::InclusiveSum(nullptr, tb3, S->d_mflag, S->d_mpos, (int64_t)t, st));
    YG_CHECK(ygpu_temp_reserve(ctx, std::max(tb1, std::max(tb2, tb3))));
    size_t tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, S->d_ah, S->d_bh, S->d_av, S->d_bv, (int64_t)t, 0, hash_bits, st));
    const uint64_t* h = S->d_bh;
    const uint64_t* v = S->d_bv;
    ctx->tm.n_library_launches += 3;
    if (!whole) {       // stable by record: (record, hash) order
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_temp, tb, S->d_bv, S->d_av, S->d_bh, S->d_ah, (int64_t)t, 32, 32 + sid_bits, st));
        h = S->d_ah;
        v = S->d_av;
        ctx->tm.n_library_launches += 3;
    }
    const int g = grid_for(ctx, t, 256);
    k_sq_heads<<<g, 256, 0, st>>>(h, v, t, S->d_mflag);
    YG_CUDA(ctx, cudaGetLastError());
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::InclusiveSum(ctx->d_temp, tb, S->d_mflag, S->d_mpos, (int64_t)t, st));
    uint32_t nd = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(&nd, S->d_mpos + (t - 1), sizeof nd, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    YG_CHECK(dev_alloc(ctx, &S->d_rh, nd));
    YG_CHECK(dev_alloc(ctx, &S->d_rv, nd));
    YG_CUDA(ctx, cudaMemsetAsync(S->d_rv, 0, (size_t)nd * sizeof(uint64_t), st));
    k_sq_reduce<<<g, 256, 0, st>>>(h, v, S->d_mflag, S->d_mpos, t, S->d_rh, (unsigned long long*)S->d_rv);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches += 3;
    S->n_res = nd;
    return 0;
}

// One chunk of raw text: host bytes [p, p + n) of the current file, n <= cap.
int sq_chunk(ygpu_ctx* ctx, StreamState* S, const uint8_t* p, uint64_t n) {
    if (n == 0) return 0;
    cudaStream_t st = ctx->stream;
    const int g = grid_for(ctx, n, SQ_NT);
    const int want_names = S->mode == YGPU_STREAM_PER_RECORD ? 2 : 1;
    const uint64_t rec_before = S->h_state->n_records;
    YG_CUDA(ctx, cudaEventRecord(S->ev[0], st));
    YG_CUDA(ctx, cudaMemcpyAsync(S->d_raw, p, n, cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaEventRecord(S->ev[1], st));
    k_sq_pre<<<g, SQ_NT, 0, st>>>(S->d_raw, n, S->d_nl, S->d_nr);
    YG_CUDA(ctx, cudaGetLastError());
    size_t tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, S->d_nl, S->d_line, (int64_t)n, st));
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::InclusiveScan(ctx->d_temp, tb, S->d_nr, S->d_prev, MaxI32(), (int64_t)n, st));
    YG_CUDA(ctx, cudaMemsetAsync(S->d_first, 0, n + 1, st));
    k_sq_first<<<g, SQ_NT, 0, st>>>(S->d_raw, n, S->d_line, S->d_prev, S->d_state, S->d_first);
    YG_CUDA(ctx, cudaGetLastError());
    k_sq_classify<<<g, SQ_NT, 0, st>>>(S->d_raw, n, S->d_line, S->d_prev, S->d_first, S->d_state, want_names, S->d_flags,
                                       S->d_val_a, S->d_val_b);
    YG_CUDA(ctx, cudaGetLastError());
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, S->d_val_a, S->d_pos_a, (int64_t)n, st));
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, S->d_val_b, S->d_pos_b, (int64_t)n, st));
    // the carried bases of the open record lead the compacted buffer
    YG_CUDA(ctx, cudaMemcpyAsync(S->d_out, (const uint8_t*)S->d_state + offsetof(ysq_state, carry), YSQ_CARRY_MAX, cudaMemcpyDeviceToDevice, st));
    k_sq_scatter<<<g, SQ_NT, 0, st>>>(S->d_raw, n, S->d_flags, S->d_pos_a, S->d_pos_b, S->d_state, S->d_out, S->d_off, S->d_names,
                                      S->d_name_start);
    YG_CUDA(ctx, cudaGetLastError());
    k_sq_finish<<<1, 1, 0, st>>>(S->d_raw, n, S->d_line, S->d_flags, S->d_pos_a, S->d_pos_b, S->d_first, S->d_out, S->d_off,
                                 S->d_state, S->d_chunk, S->ksize);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches += 5;
    ctx->tm.n_library_launches += 4;
    YG_CUDA(ctx, cudaEventRecord(S->ev[2], st));
    YG_CUDA(ctx, cudaMemcpyAsync(S->h_chunk, S->d_chunk, sizeof(ysq_chunk), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(S->h_state, S->d_state, sizeof(ysq_state), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    const ysq_chunk c = *S->h_chunk;
    S->st.ms_h2d += ev_ms(S->ev[0], S->ev[1]);
    S->st.ms_parse += ev_ms(S->ev[1], S->ev[2]);
    S->st.n_chunks++;
    S->st.n_bytes += n;
    S->st.n_bases += c.n_out;

    if (c.n_name || (c.n_rec && (S->mode == YGPU_STREAM_PER_RECORD || S->fmt == YSQ_FASTA))) {
        const uint64_t base = S->names.size();
        S->names.resize(base + c.n_name);
        S->h_name_start.resize(c.n_rec);
        if (c.n_name) YG_CUDA(ctx, cudaMemcpyAsync(&S->names[base], S->d_names, c.n_name, cudaMemcpyDeviceToHost, st));
        if (c.n_rec) YG_CUDA(ctx, cudaMemcpyAsync(S->h_name_start.data(), S->d_name_start, c.n_rec * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        for (uint64_t r = 0; r < c.n_rec; r++) S->name_off.push_back(base + S->h_name_start[r]);
    }

    if (c.n_out < (uint64_t)S->ksize) return 0;
    YG_CUDA(ctx, cudaMemsetAsync(S->d_out + c.n_out, 0, YG_SKETCH_PAD, st));
    uint64_t m = 0, n_kmers = 0;
    YG_CHECK(ygpu_sketch_hash_device(ctx, S->d_out, c.n_out, S->d_off, (uint32_t)(c.n_rec + 1), S->ksize, S->max_hash, S->seed,
                                     S->ev[3], &m, &n_kmers));
    S->st.ms_hash += ev_ms(S->ev[2], S->ev[3]);
    S->st.n_kmers += n_kmers;
    if (m == 0) return 0;
    YG_CHECK(sq_merge(ctx, S, m, (uint32_t)(rec_before - 1)));
    YG_CUDA(ctx, cudaEventRecord(S->ev[4], st));
    YG_CUDA(ctx, cudaEventSynchronize(S->ev[4]));
    S->st.ms_merge += ev_ms(S->ev[3], S->ev[4]);
    return 0;
}

int sq_active(ygpu_ctx* ctx, StreamState** out, const char* what) {
    StreamState* S = ctx ? (StreamState*)ctx->seq_stream : nullptr;
    if (!S || !S->active) return ygpu_fail(ctx, YGPU_ERR_STATE, "%s: no stream begun (or it failed; begin again)", what);
    *out = S;
    return 0;
}

void sq_reset_file(StreamState* S) {
    S->file_started = false;
    S->fmt = YSQ_FMT_NONE;
    ysq_state& s = *S->h_state;
    s.line = 0;
    s.last_nonempty1 = 0;
    s.first_bad = ~0ull;
    s.first_bad_empty = ~0ull;
    s.fmt = YSQ_FMT_NONE;
    s.open_first = 0;
    s.n_carry = 0;
}

}  // namespace

void ygpu_stream_release(ygpu_ctx* ctx) {
    StreamState* S = (StreamState*)ctx->seq_stream;
    if (!S) return;
    dev_free(ctx, &S->d_raw); dev_free(ctx, &S->d_nl); dev_free(ctx, &S->d_line); dev_free(ctx, &S->d_nr); dev_free(ctx, &S->d_prev);
    dev_free(ctx, &S->d_first); dev_free(ctx, &S->d_flags); dev_free(ctx, &S->d_val_a); dev_free(ctx, &S->d_pos_a);
    dev_free(ctx, &S->d_val_b); dev_free(ctx, &S->d_pos_b); dev_free(ctx, &S->d_out); dev_free(ctx, &S->d_off);
    dev_free(ctx, &S->d_names); dev_free(ctx, &S->d_name_start); dev_free(ctx, &S->d_state); dev_free(ctx, &S->d_chunk);
    dev_free(ctx, &S->d_rh); dev_free(ctx, &S->d_rv); dev_free(ctx, &S->d_ah); dev_free(ctx, &S->d_av); dev_free(ctx, &S->d_bh);
    dev_free(ctx, &S->d_bv); dev_free(ctx, &S->d_mflag); dev_free(ctx, &S->d_mpos);
    if (S->h_stage) cudaFreeHost(S->h_stage);
    if (S->h_state) cudaFreeHost(S->h_state);
    if (S->h_chunk) cudaFreeHost(S->h_chunk);
    for (cudaEvent_t e : S->ev)
        if (e) cudaEventDestroy(e);
    delete S;
    ctx->seq_stream = nullptr;
}

extern "C" int ygpu_stream_begin(ygpu_ctx* ctx, int ksize, uint64_t max_hash, uint32_t seed, int mode) {
    if (!ctx) return YGPU_ERR_ARG;
    if (ksize < 1 || ksize > YSQ_CARRY_MAX) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_stream_begin: ksize %d outside [1, %d]", ksize, YSQ_CARRY_MAX);
    if (mode != YGPU_STREAM_WHOLE && mode != YGPU_STREAM_PER_RECORD) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_stream_begin: unknown mode %d", mode);
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    StreamState* S = sq_get(ctx);
    if (!S->h_state) {
        YG_CUDA(ctx, cudaHostAlloc((void**)&S->h_state, sizeof(ysq_state), cudaHostAllocDefault));
        YG_CUDA(ctx, cudaHostAlloc((void**)&S->h_chunk, sizeof(ysq_chunk), cudaHostAllocDefault));
        for (cudaEvent_t& e : S->ev) YG_CUDA(ctx, cudaEventCreate(&e));
    }
    if (S->h_stage && S->cap != ctx->stream_chunk_bytes) { cudaFreeHost(S->h_stage); S->h_stage = nullptr; }
    S->cap = ctx->stream_chunk_bytes;
    if (!S->h_stage) YG_CUDA(ctx, cudaHostAlloc((void**)&S->h_stage, S->cap, cudaHostAllocDefault));
    YG_CHECK(sq_alloc_chunk(ctx, S));
    S->ksize = ksize;
    S->max_hash = max_hash;
    S->seed = seed;
    S->mode = mode;
    S->staged = 0;
    S->n_res = 0;
    S->names.clear();
    S->name_off.clear();
    S->st = ygpu_stream_stats{};
    memset(S->h_state, 0, sizeof(ysq_state));
    sq_reset_file(S);
    S->h_state->n_records = 0;
    S->active = true;
    return 0;
}

extern "C" int ygpu_stream_feed(ygpu_ctx* ctx, const uint8_t* bytes, uint64_t n) {
    StreamState* S;
    YG_CHECK(sq_active(ctx, &S, "ygpu_stream_feed"));
    if (!bytes && n) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_stream_feed: bad argument");
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!S->file_started) {           // leading whitespace is skipped; the next byte chooses the format
        uint64_t i = 0;
        while (i < n && ysq_is_space(bytes[i])) i++;
        bytes += i;
        n -= i;
        if (n == 0) return 0;
        S->fmt = ysq_format_of(bytes[0]);
        if (S->fmt == YSQ_FMT_NONE) return sq_fail(ctx, S, YGPU_ERR_ARG, "neither FASTA ('>') nor FASTQ ('@')");
        S->h_state->fmt = (uint32_t)S->fmt;
        YG_CUDA(ctx, cudaMemcpyAsync(S->d_state, S->h_state, sizeof(ysq_state), cudaMemcpyHostToDevice, ctx->stream));
        S->file_started = true;
    }
    while (n) {
        if (S->staged == 0 && n >= S->cap) {        // a whole chunk: straight from the caller's buffer
            const int rc = sq_chunk(ctx, S, bytes, S->cap);
            if (rc) { S->active = false; return rc; }
            bytes += S->cap;
            n -= S->cap;
            continue;
        }
        const uint64_t take = std::min(S->cap - S->staged, n);
        memcpy(S->h_stage + S->staged, bytes, take);
        S->staged += take;
        bytes += take;
        n -= take;
        if (S->staged == S->cap) {
            const int rc = sq_chunk(ctx, S, S->h_stage, S->staged);
            S->staged = 0;
            if (rc) { S->active = false; return rc; }
        }
    }
    return 0;
}

extern "C" int ygpu_stream_end_file(ygpu_ctx* ctx) {
    StreamState* S;
    YG_CHECK(sq_active(ctx, &S, "ygpu_stream_end_file"));
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    if (S->staged) {
        const int rc = sq_chunk(ctx, S, S->h_stage, S->staged);
        S->staged = 0;
        if (rc) { S->active = false; return rc; }
    }
    if (S->fmt == YSQ_FASTQ) {
        uint64_t v = 0;
        const int bad = ysq_fastq_end_check(S->h_state, &v);
        char msg[96];
        if (bad == 1) snprintf(msg, sizeof msg, "FASTQ with %llu lines (not a multiple of 4)", (unsigned long long)v);
        if (bad == 2) snprintf(msg, sizeof msg, "malformed FASTQ record at line %llu", (unsigned long long)v);
        if (bad) return sq_fail(ctx, S, YGPU_ERR_ARG, msg);
    }
    sq_reset_file(S);
    YG_CUDA(ctx, cudaMemcpyAsync(S->d_state, S->h_state, sizeof(ysq_state), cudaMemcpyHostToDevice, ctx->stream));
    YG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int ygpu_stream_finish(ygpu_ctx* ctx, ygpu_sketch_result* out, ygpu_stream_stats* stats, char** names,
                                  uint64_t** name_offsets, uint64_t* n_names) {
    StreamState* S;
    YG_CHECK(sq_active(ctx, &S, "ygpu_stream_finish"));
    if (!out || !names || !name_offsets || !n_names) return ygpu_fail(ctx, YGPU_ERR_ARG, "ygpu_stream_finish: bad argument");
    if (S->file_started || S->staged) YG_CHECK(ygpu_stream_end_file(ctx));
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    memset(out, 0, sizeof *out);
    *names = nullptr;
    *name_offsets = nullptr;
    *n_names = 0;
    const uint64_t n_rec = S->h_state->n_records;
    const uint64_t ns = S->mode == YGPU_STREAM_WHOLE ? 1 : n_rec;
    if (ns >= (1ull << 32)) return sq_fail(ctx, S, YGPU_ERR_ARG, "ygpu_stream_finish: more than 2^32 records");
    const uint64_t nd = S->n_res;
    out->offsets = (uint64_t*)calloc(ns + 1, sizeof(uint64_t));
    out->hashes = (uint64_t*)malloc(std::max<uint64_t>(nd, 1) * sizeof(uint64_t));
    out->abundances = (uint32_t*)malloc(std::max<uint64_t>(nd, 1) * sizeof(uint32_t));
    std::vector<uint64_t> v(nd);
    if (!out->offsets || !out->hashes || !out->abundances) { ygpu_sketch_result_free(out); return sq_fail(ctx, S, YGPU_ERR_NOMEM, "out of host memory"); }
    out->n_sketches = (uint32_t)ns;
    out->n_kmers = S->st.n_kmers;
    if (nd) {
        YG_CUDA(ctx, cudaMemcpyAsync(out->hashes, S->d_rh, nd * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaMemcpyAsync(v.data(), S->d_rv, nd * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
    }
    for (uint64_t i = 0; i < nd; i++) {
        out->abundances[i] = (uint32_t)v[i];
        out->offsets[(v[i] >> 32) + 1]++;
    }
    for (uint64_t s = 0; s < ns; s++) out->offsets[s + 1] += out->offsets[s];
    const uint64_t nn = S->name_off.size();
    if (nn) {
        *names = (char*)malloc(std::max<size_t>(S->names.size(), 1));
        *name_offsets = (uint64_t*)malloc((nn + 1) * sizeof(uint64_t));
        if (!*names || !*name_offsets) {
            free(*names); free(*name_offsets); *names = nullptr; *name_offsets = nullptr;
            ygpu_sketch_result_free(out);
            return sq_fail(ctx, S, YGPU_ERR_NOMEM, "out of host memory");
        }
        memcpy(*names, S->names.data(), S->names.size());
        memcpy(*name_offsets, S->name_off.data(), nn * sizeof(uint64_t));
        (*name_offsets)[nn] = S->names.size();
        *n_names = nn;
    }
    S->st.n_records = n_rec;
    if (stats) *stats = S->st;
    S->active = false;
    S->n_res = 0;
    return 0;
}
