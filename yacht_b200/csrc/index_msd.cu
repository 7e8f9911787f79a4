// libyachtgpu -- K2 (inverted index) without a full sort: MSD radix partition + in-shared-memory
// hash grouping.  sm_100a only.
//
// Replaces compute_index_from_sketches() of the reference (src/cpp/main.cpp:215-246), which inserts
// every hash into one unordered_map on one host thread.  What the pairwise kernel needs is weaker
// than a sorted index: for every hash held by >= 2 genome slots, the list of those genomes
// (ascending), and for every genome the list of "postings that follow me".  So instead of sorting
// T (hash, genome) pairs by all 55 significant bits (7 radix passes over 12-byte pairs), this path
//   1. packs (hash low bits, genome id) into ONE 64-bit word -- the leading d1 hash bits are implied
//      by the level-1 bucket, so 55 - d1 + ceil(log2 N) bits fit; the genome id of a hash slot is derived from
//      the CSR offsets (a few genome boundaries per tile), not read from a per-slot array --
//   2. partitions the words by the leading d1 and then the next d2 hash bits into ~T/800 final
//      buckets (two scatter passes of 8 bytes per element; tiles arrive through the copy engine --
//      cp.async.bulk + mbarrier, double-buffered -- and are reordered in the buffer they arrived in),
//   3. groups equal hashes inside each bucket in shared memory (k2_group2; k2_group for buckets or key widths it does
//      not take: a counting filter over the next 11 hash bits drops the words that are alone in their sub-bucket,
//      the rest are scanned densely; no ordering of singleton hashes is ever computed), orders only the members of
//      shared groups by genome id, and emits compact postings + per-genome work items.
// Algorithmic HBM traffic: 8T + 8T (scatter 1) + 16T (scatter 2) + 8T (bucket read) + O(P) outputs ~= 40 bytes per hash,
// against ~176 for the 7-pass pair sort.  The buckets live in fixed-capacity slots sized from the plan (msd_build); only a
// database that overflows one pays the two histogram passes (8T each) of the exact layout.
//
// Skew: a final bucket that does not fit shared memory (a hash held by thousands of genomes) leaves this path
// alone -- its words are sorted device-wide (in chunks of buckets) and grouped by neighbour comparison (k2_big_*).
// The general path (yacht_gpu.cu, library radix sort of all pairs) remains only for inputs that do not pack (hash width +
// genome-id width).  The choice is made per database from the measured bucket histogram -- "chosen by measured
// posting-list skew".
//
// Across GPUs (ygpu_train_step_sharded, end of this file) every rank partitions only its own sketches and the level-1
// scatter stores each word straight into the buffer of the rank that owns its hash range (NVLink), the grouping kernel
// stores each bucket's groups into every rank's stream buffer: the exchanges are part of the kernels.
// The run path (`yacht run`) probes the same partition bucket by bucket (run_buckets.cuh).
#include "common.cuh"

#include <cub/cub.cuh>
#include <algorithm>
#include <cstdio>
#include <vector>

namespace {

constexpr int SC_TILE = 4096;       // elements per scatter tile (512 threads x 8)
constexpr int SC_THREADS = 512;
constexpr int SC_ITEMS = SC_TILE / SC_THREADS;
constexpr int SC_BUF = SC_TILE + 8; // words per tile buffer: the 16-byte aligned window around a tile may start one word early
constexpr int SC_BND = 16;          // level 1: genome boundaries per tile resolved from shared memory (more: binary search in L2)
constexpr int NB_MAX = 2048;        // digits per partition level
constexpr uint32_t A_TARGET = 900;  // average elements per used final bucket (k2_group2 takes buckets of <= 1022)

// extra slots of ctx->d_scalars (SCM_MAXB uses two; SCM_OVF1 / SCM_OVF2: a slot of that partition level overflowed)
enum { SCM_PCUR = 8, SCM_ICUR = 9, SCM_MAXB = 10, SCM_STREAM = 12, SCM_OVF1 = 13, SCM_OVF2 = 14 };
// sharded step: the first REP_WORDS slots of d_scalars are one rank's report to the others (statistics, largest bucket, posting-
// stream length, and from REP_ICUR the number of work items it sent to every rank); ONE all-gather after the grouping carries it
enum { REP_ICUR = 16, REP_WORDS = 32 };
static_assert(REP_ICUR + YG_MAX_RANKS <= REP_WORDS, "the report holds one item counter per rank");

struct MsdPlan {
    int hb, gb, d1, d2, kb1;
    uint32_t nb1;     // used level-1 buckets
    uint32_t nfb;     // final buckets (nb1 << d2)
    uint64_t T;
    // hash-range sharding (multi-GPU): this rank keeps level-1 digits [dlo, dhi) only, i.e. level-2 tiles [unit_lo, unit_hi)
    uint32_t dlo, dhi, unit_lo, unit_hi;
};

__device__ __forceinline__ uint32_t digit1_of(uint64_t key, const MsdPlan& p) {
    return p.d1 ? (uint32_t)(key >> (p.hb - p.d1)) : 0u;
}
__device__ __forceinline__ uint64_t pack_entry(uint64_t key, uint32_t gid, const MsdPlan& p) {
    const uint64_t low = (p.kb1 >= 64) ? key : (key & ((1ull << p.kb1) - 1ull));
    return (low << p.gb) | (uint64_t)gid;
}
__device__ __forceinline__ uint32_t digit2_of(uint64_t e, const MsdPlan& p) {
    return p.d2 ? (uint32_t)((e >> (p.gb + p.kb1 - p.d2)) & ((1u << p.d2) - 1u)) : 0u;
}

// ---- bulk asynchronous copies (TMA engine, cp.async.bulk) completing on a shared-memory mbarrier ---------------
// One elected thread asks the copy engine for a whole tile; no thread holds the tile in registers while it is in
// flight, so the next tile streams in behind the current one (SASS: UBLKCP + SYNCS).
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// dst / src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "W:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra D;\n"
        "bra W;\n"
        "D:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---- level-1 histogram ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k2_hist1(const uint64_t* __restrict__ hashes, const MsdPlan p, uint32_t* __restrict__ hist) {
    extern __shared__ uint32_t sh[];
    for (uint32_t i = threadIdx.x; i < p.nb1; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const int shift = p.hb - p.d1;
    const bool one = p.d1 == 0;
    // 16-byte loads, four in flight per thread
    const ulonglong2* h2 = reinterpret_cast<const ulonglong2*>(hashes);
    const uint64_t n2 = p.T >> 1;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n2; i += 4 * stride) {
        const ulonglong2 a = h2[i], b = h2[i + stride], c = h2[i + 2 * stride], d = h2[i + 3 * stride];
        atomicAdd(&sh[one ? 0u : (uint32_t)(a.x >> shift)], 1u); atomicAdd(&sh[one ? 0u : (uint32_t)(a.y >> shift)], 1u);
        atomicAdd(&sh[one ? 0u : (uint32_t)(b.x >> shift)], 1u); atomicAdd(&sh[one ? 0u : (uint32_t)(b.y >> shift)], 1u);
        atomicAdd(&sh[one ? 0u : (uint32_t)(c.x >> shift)], 1u); atomicAdd(&sh[one ? 0u : (uint32_t)(c.y >> shift)], 1u);
        atomicAdd(&sh[one ? 0u : (uint32_t)(d.x >> shift)], 1u); atomicAdd(&sh[one ? 0u : (uint32_t)(d.y >> shift)], 1u);
    }
    for (; i < n2; i += stride) {
        const ulonglong2 a = h2[i];
        atomicAdd(&sh[one ? 0u : (uint32_t)(a.x >> shift)], 1u); atomicAdd(&sh[one ? 0u : (uint32_t)(a.y >> shift)], 1u);
    }
    if ((p.T & 1ull) && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&sh[digit1_of(hashes[p.T - 1], p)], 1u);
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < p.nb1; k += blockDim.x)
        if (sh[k]) atomicAdd(&hist[k], sh[k]);
}

// one CTA: tile prefix (for level-2 work units) and largest bucket from the level-1 bucket sizes, plus either
//   end == NULL (exact layout, before the scatter): cnt is the histogram; begin = its exclusive scan, begin[nb] = total, and
//               the scatter's cursors start there;
//   end != NULL (slotted layout, after the scatter): cnt are the scatter's counters, clamped to cap (a slot that overflowed is
//               cut; the host redoes the partition on the exact layout); end = begin + size.
__global__ void __launch_bounds__(1024) k2_prep1(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ cap, uint32_t nb,
                                                  uint32_t* __restrict__ begin, uint32_t* __restrict__ end, uint32_t* __restrict__ cursor,
                                                  uint32_t* __restrict__ tile_start, unsigned long long* __restrict__ scal) {
    typedef cub::BlockScan<uint32_t, 1024> Scan;
    __shared__ typename Scan::TempStorage ts1, ts2;
    const int per = (NB_MAX + 1023) / 1024;
    uint32_t h[per], t[per], hs = 0, tsum = 0, mx = 0;
    for (int k = 0; k < per; k++) {
        const uint32_t i = threadIdx.x * per + k;
        h[k] = i < nb ? (end ? min(cnt[i], cap[i]) : cnt[i]) : 0u;
        t[k] = (h[k] + SC_TILE - 1) / SC_TILE;
        hs += h[k]; tsum += t[k]; mx = max(mx, h[k]);
    }
    uint32_t hoff, toff, htot, ttot;
    Scan(ts1).ExclusiveSum(hs, hoff, htot);
    Scan(ts2).ExclusiveSum(tsum, toff, ttot);
    for (int k = 0; k < per; k++) {
        const uint32_t i = threadIdx.x * per + k;
        if (i < nb) {
            if (end) end[i] = begin[i] + h[k];
            else { begin[i] = hoff; cursor[i] = hoff; }
            tile_start[i] = toff;
        }
        hoff += h[k]; toff += t[k];
    }
    if (threadIdx.x == 0) {
        if (!end) begin[nb] = htot;
        tile_start[nb] = ttot;
    }
    if (mx) atomicMax(&scal[SCM_MAXB], (unsigned long long)mx);
}

// slotted layout: bucket b owns words [b * c, (b + 1) * c) of the level's buffer
__global__ void __launch_bounds__(256) k2_slots(uint32_t nb, uint32_t c, uint32_t* __restrict__ begin, uint32_t* __restrict__ cap) {
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b <= nb; b += gridDim.x * blockDim.x) {
        begin[b] = b * c;
        cap[b] = c;
    }
}

// slotted layout, level 2: bucket extents from the scatter's counters (clamped to the slot) and the largest bucket
__global__ void __launch_bounds__(256) k2_ends(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ cap,
                                               const uint32_t* __restrict__ begin, uint32_t nb, uint32_t* __restrict__ end,
                                               unsigned long long* __restrict__ maxb) {
    uint32_t mx = 0;
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
        const uint32_t m = min(cnt[b], cap[b]);
        end[b] = begin[b] + m;
        mx = max(mx, m);
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(maxb, (unsigned long long)mx);
}

// ---- scatter (level 1: raw hashes -> packed words by leading digit; level 2: words -> final buckets)
struct ScatterArgs {
    const uint64_t* hashes;      // level 1 input
    const uint64_t* offsets;     // level 1: CSR offsets of the sketches [n + 1] (the genome id of a hash slot is derived from them)
    const uint32_t* tile_g0;     // level 1: genome holding the first hash of every tile [tiles + 1] (k2_tile_g0)
    uint32_t n;
    const uint64_t* in_ent;      // level 2 input
    uint64_t* out_ent;
    const uint32_t* tile_start;  // level 2: prefix of tiles per level-1 bucket ([nb1] = number of units)
    // Slotted layout (slot != 0): bucket b's words go to out_ent[b * slot + rank], rank counted from zero in cursor[b], so an
    // overshoot cannot wrap 32 bits; words of rank >= slot are dropped and raise *ovf.  Exact layout (slot == 0, sized by a
    // histogram, cannot overflow): cursor[b] starts at the bucket's first position (sharded step: where this rank's words go).
    // Neither needs a load per (tile, digit) run beside the cursor atomic.
    uint32_t slot;
    uint32_t* cursor;
    unsigned long long* ovf;
    uint32_t* hist2;             // hist2 kernel only
    const uint2* units;          // level 2: per tile {first word, words | level-1 bucket << 16} (k2_units)
    // sharded build across GPUs (level 1, PEER): a word goes to the rank that owns its leading digit, stored straight into
    // that rank's level-1 buffer over NVLink (peer_ent: the ranks' d_ent1 as mapped into this process)
    uint32_t gid_base;           // genome id of the first resident sketch (sharded residency: offsets are slice-relative)
    const uint32_t* owner;       // [nb1] owner rank of every level-1 digit
    uint64_t* peer_ent[YG_MAX_RANKS];
};

template <int LEVEL>
__device__ __forceinline__ bool unit_range(const ScatterArgs& a, const MsdPlan& p, uint32_t unit, uint32_t n_units, uint64_t& begin,
                                           uint32_t& m, uint32_t& b1) {
    if (unit >= n_units) return false;
    if (LEVEL == 1) {
        begin = (uint64_t)unit * SC_TILE;
        m = (uint32_t)min((uint64_t)SC_TILE, p.T - begin);
        b1 = 0;
        return true;
    }
    const uint2 u = a.units[unit];      // resolved once by k2_units: a per-tile binary search here would put ~10 dependent
    begin = u.x;                        // L2 round trips on the critical path of every tile
    m = u.y & 0xffffu;
    b1 = u.y >> 16;
    return true;
}

// one thread per level-2 tile: which level-1 bucket it belongs to and which words it covers (bucket b: [begin1[b], end1[b]))
__global__ void __launch_bounds__(256) k2_units(const uint32_t* __restrict__ tile_start, const uint32_t* __restrict__ begin1,
                                                const uint32_t* __restrict__ end1, uint32_t nb1, uint2* __restrict__ units) {
    const uint32_t n_units = tile_start[nb1];
    for (uint32_t unit = blockIdx.x * blockDim.x + threadIdx.x; unit < n_units; unit += gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = nb1;          // last bucket b with tile_start[b] <= unit
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (tile_start[mid] <= unit) lo = mid; else hi = mid;
        }
        const uint32_t k = unit - tile_start[lo];
        const uint64_t begin = (uint64_t)begin1[lo] + (uint64_t)k * SC_TILE;
        const uint32_t m = (uint32_t)min((uint64_t)SC_TILE, (uint64_t)end1[lo] - begin);
        units[unit] = make_uint2((uint32_t)begin, m | (lo << 16));
    }
}

// largest g with offsets[g] <= idx, searched in [lo, hi] (offsets[lo] <= idx)
__device__ __forceinline__ uint32_t genome_of(const uint64_t* __restrict__ offsets, uint32_t lo, uint32_t hi, uint64_t idx) {
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo + 1) >> 1);
        if (offsets[mid] <= idx) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// one thread per level-1 tile: the genome that holds the tile's first hash slot (the last one holding slot T - 1 for
// the entry behind the last tile).  Replaces a 4-byte genome id per hash slot read by the level-1 scatter.
__global__ void __launch_bounds__(256) k2_tile_g0(const uint64_t* __restrict__ offsets, uint32_t n, uint64_t T, uint32_t n_tiles,
                                                  uint32_t* __restrict__ tile_g0) {
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t <= n_tiles; t += gridDim.x * blockDim.x) {
        const uint64_t idx = t < n_tiles ? (uint64_t)t * SC_TILE : T - 1;
        tile_g0[t] = genome_of(offsets, 0, n - 1, idx);
    }
}

// Level-2 digit histogram.  A CTA walks a contiguous range of tiles, so its shared-memory counters are flushed only when
// the level-1 bucket changes (once or twice per CTA), not once per tile.
__global__ void __launch_bounds__(256) k2_hist2(const ScatterArgs a, const MsdPlan p, uint32_t unit_end) {
    extern __shared__ uint32_t sh[];
    const uint32_t nd = 1u << p.d2;
    unit_end = min(unit_end, a.tile_start[p.nb1]);
    const uint32_t total = unit_end > p.unit_lo ? unit_end - p.unit_lo : 0u;
    const uint32_t per = (total + gridDim.x - 1) / gridDim.x;
    const uint32_t u0 = p.unit_lo + blockIdx.x * per;
    const uint32_t u1 = min(unit_end, u0 + per);
    const int shift = p.gb + p.kb1 - p.d2;
    const uint32_t mask = nd - 1u;
    uint32_t cur = 0xFFFFFFFFu;
    for (uint32_t unit = u0; unit < u1; unit++) {
        const uint2 u = a.units[unit];
        const uint64_t begin = u.x;
        const uint32_t m = u.y & 0xffffu, b1 = u.y >> 16;
        if (b1 != cur) {                    // uniform per CTA
            __syncthreads();
            if (cur != 0xFFFFFFFFu)
                for (uint32_t i = threadIdx.x; i < nd; i += blockDim.x)
                    if (sh[i]) atomicAdd(&a.hist2[((uint64_t)cur << p.d2) + i], sh[i]);
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < nd; i += blockDim.x) sh[i] = 0;
            __syncthreads();
            cur = b1;
        }
        const uint64_t* src = a.in_ent + begin;
        for (uint32_t i = threadIdx.x; i < m; i += 4 * 256) {
            uint64_t e0 = 0, e1 = 0, e2 = 0, e3 = 0;
            const bool v1 = i + 256 < m, v2 = i + 512 < m, v3 = i + 768 < m;
            e0 = src[i];
            if (v1) e1 = src[i + 256];
            if (v2) e2 = src[i + 512];
            if (v3) e3 = src[i + 768];
            atomicAdd(&sh[(uint32_t)(e0 >> shift) & mask], 1u);
            if (v1) atomicAdd(&sh[(uint32_t)(e1 >> shift) & mask], 1u);
            if (v2) atomicAdd(&sh[(uint32_t)(e2 >> shift) & mask], 1u);
            if (v3) atomicAdd(&sh[(uint32_t)(e3 >> shift) & mask], 1u);
        }
    }
    __syncthreads();
    if (cur != 0xFFFFFFFFu)
        for (uint32_t i = threadIdx.x; i < nd; i += blockDim.x)
            if (sh[i]) atomicAdd(&a.hist2[((uint64_t)cur << p.d2) + i], sh[i]);
}

// Tile-staged scatter.  Tiles arrive through the copy engine (cp.async.bulk + mbarrier) into two ping-pong buffers:
// while tile k is ranked, reordered and written out, tile k+1 is already streaming into the other buffer.  The
// reordered words are staged in the buffer the tile came in (its words are in registers by then), so a CTA holds two
// tile buffers, not three.  Level 1 derives the genome id of every hash slot from the CSR offsets (a few boundaries
// per tile, kept in shared memory) instead of reading a 4-byte id per slot.
template <int LEVEL, bool PEER>
__global__ void __launch_bounds__(SC_THREADS, 2) k2_scatter(const ScatterArgs a, const MsdPlan p, uint32_t unit_first, uint32_t n_units) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* buf0 = (uint64_t*)smem_raw;                          // [2][SC_BUF]
    const uint32_t nd = LEVEL == 1 ? p.nb1 : (1u << p.d2);
    uint64_t** gptr = (uint64_t**)(buf0 + 2 * SC_BUF);             // [nd] PEER only: where this tile's run of digit d goes
    // [nd] {gbase, glim}: slot q of digit d's run goes to gbase + q if q < glim (beyond: past its bucket's cap) -- one 8-byte
    // shared load per word
    uint2* gdst = (uint2*)(gptr + (PEER ? nd : 0));
    uint32_t* cnt = (uint32_t*)(gdst + nd);                        // [nd]
    uint32_t* lbase = cnt + nd;                                    // [nd]
    uint16_t* sdig = (uint16_t*)(lbase + nd);                      // [SC_TILE]
    typedef cub::BlockScan<uint32_t, SC_THREADS> Scan;
    __shared__ typename Scan::TempStorage scan_ts;
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t bnd[2][SC_BND];       // level 1: genome boundaries inside a tile, relative to its first hash slot

    const uint32_t tid = threadIdx.x;
    if (LEVEL == 2) n_units = min(n_units, a.tile_start[p.nb1]);
    const uint64_t* src_all = LEVEL == 1 ? a.hashes : a.in_ent;
    // level 1: the genome boundaries of a tile are fetched one tile ahead (visible after the barrier that ends an iteration)
    auto fetch_bnd = [&](uint32_t unit, uint32_t slot) {
        if (LEVEL != 1 || unit >= n_units) return;
        const uint32_t g0 = a.tile_g0[unit], nb = a.tile_g0[unit + 1] - g0;
        if (nb <= SC_BND && tid < nb) bnd[slot][tid] = (uint32_t)min(a.offsets[g0 + 1 + tid] - (uint64_t)unit * SC_TILE, (uint64_t)SC_TILE);
    };
    auto issue = [&](uint32_t unit, uint32_t slot) {              // thread 0 only
        uint64_t begin; uint32_t m, b1;
        if (!unit_range<LEVEL>(a, p, unit, n_units, begin, m, b1)) return;
        const uint64_t w0 = begin & ~1ull, w1 = (begin + m + 1) & ~1ull;
        bulk_load(buf0 + slot * SC_BUF, src_all + w0, (uint32_t)(w1 - w0) * 8u, &mbar[slot]);
    };
    for (uint32_t i = tid; i < nd; i += SC_THREADS) cnt[i] = 0;
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        mbar_init_fence();
    }
    const uint32_t unit0 = unit_first + blockIdx.x;
    fetch_bnd(unit0, 0);
    __syncthreads();
    if (tid == 0) {
        issue(unit0, 0);
        issue(unit0 + gridDim.x, 1);
    }

    constexpr uint16_t SKIP = 0xFFFFu;     // not in the tile, or (level 1, sharded) a digit another rank owns
    uint32_t it = 0;
    for (uint32_t unit = unit0;; unit += gridDim.x, it++) {
        uint64_t begin; uint32_t m, b1;
        if (!unit_range<LEVEL>(a, p, unit, n_units, begin, m, b1)) break;
        const uint32_t slot = it & 1u;
        uint64_t* buf = buf0 + slot * SC_BUF;
        // level 1: genome boundaries inside this tile
        uint32_t g0 = 0, nbnd = 0;
        if (LEVEL == 1) {
            g0 = a.tile_g0[unit];
            nbnd = a.tile_g0[unit + 1] - g0;
        }
        mbar_wait(&mbar[slot], (it >> 1) & 1u);
        const uint32_t sh = (uint32_t)(begin & 1ull);
        uint64_t e[SC_ITEMS];
        uint16_t dg[SC_ITEMS], rk[SC_ITEMS];
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) {
            const uint32_t idx = k * SC_THREADS + tid;
            dg[k] = SKIP;
            if (idx < m) {
                e[k] = buf[sh + idx];
                if (LEVEL == 1) {
                    const uint32_t d = digit1_of(e[k], p);
                    if (d >= p.dlo && d < p.dhi) {
                        uint32_t g = g0;
                        if (nbnd <= SC_BND) {
                            for (uint32_t j = 0; j < nbnd; j++) g += bnd[slot][j] <= idx ? 1u : 0u;
                        } else {
                            g = genome_of(a.offsets, g0, g0 + nbnd, begin + idx);
                        }
                        dg[k] = (uint16_t)d;
                        e[k] = pack_entry(e[k], a.gid_base + g, p);
                    }
                } else {
                    dg[k] = (uint16_t)digit2_of(e[k], p);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++)
            if (dg[k] != SKIP) rk[k] = (uint16_t)atomicAdd(&cnt[dg[k]], 1u);
        __syncthreads();                   // every word of the tile is in registers: the buffer becomes the staging area
        uint32_t mv = 0;     // words of this tile that are kept
        // exclusive scan of cnt -> lbase; reserve room per digit in its bucket (the cursor atomics' answers are only needed for the
        // write-out: they travel while the tile is being reordered); counters back to zero
        constexpr uint32_t PER_MAX = (NB_MAX + SC_THREADS - 1) / SC_THREADS;
        uint32_t gb0[PER_MAX], has = 0;
        const uint32_t per = (nd + SC_THREADS - 1) / SC_THREADS;
        const uint32_t d0 = tid * per;
        {
            uint32_t s = 0;
            for (uint32_t k = 0; k < per; k++) if (d0 + k < nd) s += cnt[d0 + k];
            uint32_t off;
            Scan(scan_ts).ExclusiveSum(s, off, mv);
#pragma unroll
            for (uint32_t k = 0; k < PER_MAX; k++) {
                const uint32_t d = d0 + k;
                gb0[k] = 0;
                if (k < per && d < nd) {
                    const uint32_t c = cnt[d];
                    lbase[d] = off;
                    if (c) {
                        const uint64_t ci = LEVEL == 1 ? (uint64_t)d : (((uint64_t)b1 << p.d2) + d);
                        gb0[k] = atomicAdd(&a.cursor[ci], c);
                        has |= 1u << k;
                        cnt[d] = 0;
                    }
                    off += c;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) {
            if (dg[k] != SKIP) {
                const uint32_t q = lbase[dg[k]] + rk[k];
                buf[q] = e[k];
                sdig[q] = dg[k];
            }
        }
        // where the run of digit d goes: slot q of the reordered tile lands at gbase + q (PEER: in the owner's buffer), for
        // q < glim (the rest of the run is beyond the bucket's cap)
#pragma unroll
        for (uint32_t k = 0; k < PER_MAX; k++) {
            if (has & (1u << k)) {
                const uint32_t d = d0 + k;
                const uint32_t ci = LEVEL == 1 ? d : (b1 << p.d2) + d;
                const uint32_t bg = ci * a.slot;              // 0 on the exact layout: the cursor is a position there
                const uint32_t lb = lbase[d];
                if (PEER) gptr[d] = a.peer_ent[a.owner[d]] + bg + gb0[k] - lb;
                gdst[d] = make_uint2(bg + gb0[k] - lb,
                                     !a.slot ? (uint32_t)SC_TILE : lb + (gb0[k] < a.slot ? min(a.slot - gb0[k], (uint32_t)SC_TILE) : 0u));
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) {
            const uint32_t q = k * SC_THREADS + tid;
            if (q < mv) {
                const uint32_t d = sdig[q];
                const uint2 g = gdst[d];
                if (q >= g.y) *a.ovf = 1ull;                                 // the bucket's slot is full: the host re-partitions
                else if (PEER) gptr[d][q] = buf[q];                          // a store over NVLink when the owner is a peer
                else a.out_ent[(uint64_t)(uint32_t)(g.x + q)] = buf[q];
            }
        }
        fetch_bnd(unit + gridDim.x, slot ^ 1u);
        __syncthreads();                   // the buffer is free again: fetch the tile after next into it
        if (tid == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes (staging) before the async-proxy write
            issue(unit + 2 * gridDim.x, slot);
        }
    }
}

constexpr int BK_CAP = 3072;        // max words of a final bucket (shared-memory resident)

// ---- grouping kernel (k2_group): sub-bucket counting filter + dense candidate scan ------------------------
// (The first version of this kernel chained equal hashes through a CAS hash table; its chain walks were
// divergent -- 15 of 32 lanes active on average -- and barrier-bound.)  k2_group has uniform work per thread and
// spends almost nothing on the ~80 % of hashes nobody shares:
//   A  words -> registers; sub-bucket = next GK_SUBBITS hash bits; rank inside the sub-bucket from one
//      shared-memory atomicAdd.  A word alone in its sub-bucket is a singleton: it is only counted.
//   B  exclusive scan over the sizes of the sub-buckets holding >= 2 words (8 counters per thread, warp shuffles)
//   C  the words of those sub-buckets ("candidates", ~30 %) are scattered to a dense array, sub-bucket by
//      sub-bucket: 32 low bits of the remaining hash, genome id (+ remaining high hash bits), sub-bucket id
//   D  one thread per candidate scans its sub-bucket (2-3 words): group size L, own rank among the members by
//      genome id, first member's position; that first member claims L posting slots (shared-memory cursor)
//   E  members write (genome id, members that follow) at claimed offset + rank: the groups are now dense and
//      ordered by genome id in shared memory (aliasing the candidate arrays, which are dead)
//   F  one thread per staged posting: coalesced posting writes (only for groups some item points into) and
//      the member's work item, appended to the member's per-genome list.  The returning atomicAdd on the
//      per-genome counter is consumed one bucket later (software pipelining), so its latency never sits
//      between two barriers.
// This is the GENERAL grouping kernel: buckets of up to BK_CAP words and remaining-key widths beyond 32 bits.  The common
// case runs in k2_group2 (below), which is leaner; GroupArgs::m_lo tells this kernel which buckets that one already took.
constexpr int GK_THREADS = 256;
constexpr int GK_SUBBITS = 11;
constexpr int GK_NSUB = 1 << GK_SUBBITS;            // 2048 = 8 counters per thread
constexpr int GK_FAST = 4;                          // words per thread for buckets of <= 1024 words (all but skewed ones)
constexpr int GK_SLOW = BK_CAP / GK_THREADS;        // 12

struct GroupArgs {
    const uint64_t* ent;
    const uint32_t* begin;       // bucket b: words [begin[b], end[b]) of ent (exact layout: end = begin + 1)
    const uint32_t* end;
    uint32_t nb;
    uint32_t b_lo, b_hi;         // final buckets this launch covers (all, or one rank's hash range)
    uint32_t m_lo;               // k2_group: only buckets of more than m_lo words (the smaller ones went to k2_group2)
    int gb;
    int sub_shift;               // sub-bucket digit = (word >> sub_shift) & sub_mask
    uint32_t sub_mask;
    uint64_t rest_mask;          // (word >> gb) & rest_mask = hash bits below the sub-bucket digit
    uint32_t* post;              // [T]
    const uint64_t* row_off;     // [n] start of genome g's work list (= sketch offsets)
    unsigned long long* row_cnt; // [n] items appended so far
    uint64_t* row_items;         // [T]
    // sharded build (k2_group2<STREAM>): the groups leave as a compact stream instead of work items
    uint32_t* st_gid;            // genome ids, group by group, ascending inside a group
    unsigned short* st_rem;      // members of the same group that follow
    unsigned long long* scal;
    // sharded build across GPUs: the bucket range comes from device memory (k2s_prep), and k2_group2<STREAM> stores every
    // bucket's groups into ALL ranks' stream buffers (region of this rank) -- the exchange is part of the kernel
    const unsigned long long* range;   // {first bucket, end bucket} or NULL (then b_lo / b_hi)
    int n_peers;
    uint64_t region_base;              // first stream entry of this rank's region in every rank's buffer
    uint32_t* peer_gid[YG_MAX_RANKS];
    unsigned short* peer_rem[YG_MAX_RANKS];
    // ... except that the work items of small groups (<= IG_MAXL members: every database without extreme skew) travel alone,
    // self-contained (the following genome ids are inside the item), and only to the rank that owns the query row
    uint32_t row_bounds[YG_MAX_RANKS + 1];   // rank q owns query rows [row_bounds[q], row_bounds[q + 1])
    uint64_t* peer_item[YG_MAX_RANKS];       // rank q's item inbox; this rank writes region [rank * icap, (rank + 1) * icap)
    uint32_t* peer_row[YG_MAX_RANKS];        // ... the query row of every item
    uint64_t icap;
    uint64_t item_region;                    // rank * icap
    unsigned long long* icursor;             // [n_peers] items this rank has sent to every rank so far (local memory)
};

struct GroupStats { uint32_t heads, single, dups; unsigned long long w; };   // postings = T - singles, items = postings - shared groups
struct GroupPending { uint64_t item; uint32_t dst, slot; bool has; };         // T < 2^32: list positions fit 32 bits

struct GroupSmem {
    uint32_t* cnt;               // [GK_NSUB]      sub-bucket sizes (zero between buckets)
    unsigned short* start2;      // [GK_NSUB + 8]  candidate-array start of every sub-bucket
    uint32_t* K2;                // [BK_CAP]       candidates: low 32 bits of the remaining hash
    uint32_t* G2;                // [BK_CAP]       candidates: genome id | remaining high hash bits << gb
    unsigned short* SUB2;        // [BK_CAP]       candidates: sub-bucket id
    unsigned short* gbase;       // [BK_CAP]       posting offset claimed by the group whose first member sits here
    uint32_t* s_wsum;            // [8]
};

// `staged`: this bucket's words were prefetched into shared memory (cp.async issued during the previous bucket's
// phase E, into the start2|SUB2 region, dead by then); bb_next / m_next: the bucket to prefetch during this one.
template <int ITEMS>
__device__ __forceinline__ void group_bucket(const GroupArgs& a, const uint32_t bb, const uint32_t m, const GroupSmem& sm,
                                             uint32_t* s_pcur, uint32_t* s_gpos, GroupStats& st, GroupPending& pd,
                                             const bool staged, const uint32_t bb_next, const uint32_t m_next) {
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gmask = a.gb ? (uint32_t)((1ull << a.gb) - 1ull) : 0u;
    // ---- A: load, sub-bucket rank ------------------------------------------------------------------
    uint64_t e[ITEMS];
    uint32_t rk[ITEMS];
    uint64_t* stage = reinterpret_cast<uint64_t*>(sm.start2);      // [GK_FAST * GK_THREADS] words (start2 + SUB2: 10 KB)
    if (ITEMS == GK_FAST && staged) {
        asm volatile("cp.async.wait_all;" ::: "memory");           // each thread reads back exactly the words it copied
#pragma unroll
        for (int k = 0; k < ITEMS; k++)
            if (k * GK_THREADS + tid < m) e[k] = stage[k * GK_THREADS + tid];
    } else {
        const uint64_t* src = a.ent + bb + tid;
#pragma unroll
        for (int k = 0; k < ITEMS; k++)
            if (k * GK_THREADS + tid < m) e[k] = src[k * GK_THREADS];
    }
#pragma unroll
    for (int k = 0; k < ITEMS; k++)
        if (k * GK_THREADS + tid < m) rk[k] = atomicAdd(&sm.cnt[(uint32_t)(e[k] >> a.sub_shift) & a.sub_mask], 1u);
    if (tid == 0) *s_pcur = 0;
    __syncthreads();
    // ---- B: scan the sizes of sub-buckets with >= 2 words (and reset the counters for the next bucket) ----
    {
        uint4* c4 = reinterpret_cast<uint4*>(&sm.cnt[8 * tid]);
        uint4 c0 = c4[0], c1 = c4[1];
        c4[0] = make_uint4(0u, 0u, 0u, 0u);
        c4[1] = make_uint4(0u, 0u, 0u, 0u);
        c0.x = c0.x >= 2 ? c0.x : 0u; c0.y = c0.y >= 2 ? c0.y : 0u; c0.z = c0.z >= 2 ? c0.z : 0u; c0.w = c0.w >= 2 ? c0.w : 0u;
        c1.x = c1.x >= 2 ? c1.x : 0u; c1.y = c1.y >= 2 ? c1.y : 0u; c1.z = c1.z >= 2 ? c1.z : 0u; c1.w = c1.w >= 2 ? c1.w : 0u;
        const uint32_t sum = c0.x + c0.y + c0.z + c0.w + c1.x + c1.y + c1.z + c1.w;
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)lane >= o) inc += v;
        }
        if (lane == 31) sm.s_wsum[warp] = inc;
        __syncthreads();
        uint32_t wp = 0;
#pragma unroll
        for (int w = 0; w < GK_THREADS / 32 - 1; w++) wp += (w < (int)warp) ? sm.s_wsum[w] : 0u;
        const uint32_t p0 = wp + inc - sum;
        const uint32_t p1 = p0 + c0.x, p2 = p1 + c0.y, p3 = p2 + c0.z, p4 = p3 + c0.w, p5 = p4 + c1.x, p6 = p5 + c1.y, p7 = p6 + c1.z;
        *reinterpret_cast<uint4*>(&sm.start2[8 * tid]) = make_uint4(p0 | (p1 << 16), p2 | (p3 << 16), p4 | (p5 << 16), p6 | (p7 << 16));
        if (tid == GK_THREADS - 1) sm.start2[GK_NSUB] = (unsigned short)(p7 + c1.w);
    }
    __syncthreads();
    // ---- C: candidates -> dense array, sub-bucket by sub-bucket; everything else is a singleton ---------------
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
        if (k * GK_THREADS + tid < m) {
            const uint32_t s = (uint32_t)(e[k] >> a.sub_shift) & a.sub_mask;
            const uint32_t lo = sm.start2[s], hi = sm.start2[s + 1];
            if (hi > lo) {
                const uint64_t rest = (e[k] >> a.gb) & a.rest_mask;
                const uint32_t pos = lo + rk[k];
                sm.K2[pos] = (uint32_t)rest;
                sm.G2[pos] = ((uint32_t)e[k] & gmask) | ((uint32_t)(rest >> 32) << a.gb);
                sm.SUB2[pos] = (unsigned short)s;
            } else {
                st.heads++;
                st.single++;
            }
        }
    }
    __syncthreads();
    // ---- D: dense scan over the candidates -----------------------------------------------------------------------
    const uint32_t ncand = sm.start2[GK_NSUB];
    uint32_t lr[ITEMS];            // group size | rank << 16   (0 = not a member of a shared group)
    uint32_t gq[ITEMS];            // genome id of this thread's candidate
    unsigned short qf[ITEMS];      // candidate position of the group's first member
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
        const uint32_t q = k * GK_THREADS + tid;
        lr[k] = 0; qf[k] = 0; gq[k] = 0;
        if (q < ncand) {
            const uint32_t kq = sm.K2[q], xq = sm.G2[q], s = sm.SUB2[q];
            const uint32_t lo = sm.start2[s], hi = sm.start2[s + 1];
            const uint32_t g = xq & gmask;
            // branch-free: most candidates do have partners, found at different iterations by different lanes, so a
            // divergent match body would be executed by nearly every warp on nearly every iteration
            uint32_t L = 0, rank = 0, first = 0xFFFFFFFFu, dup = 0;
            const uint32_t hmask = ~gmask;
            for (uint32_t x = lo; x < hi; x++) {
                const uint32_t k2 = sm.K2[x], x2 = sm.G2[x];
                const bool same = (k2 == kq) & (((x2 ^ xq) & hmask) == 0u);      // same hash (this candidate included)
                const bool tie = same & (x2 == xq) & (x < q);                    // same genome too: in-sketch duplicate
                L += same ? 1u : 0u;
                rank += (same & ((x2 < xq) | tie)) ? 1u : 0u;                    // high bits agree: order of G2 = order of genome ids
                first = min(first, same ? x : 0xFFFFFFFFu);
                dup |= tie ? 1u : 0u;
            }
            st.heads += rank == 0;
            st.single += L == 1;
            if (L >= 2) {
                lr[k] = L | (rank << 16);
                qf[k] = (unsigned short)first;
                gq[k] = g;
                st.dups += dup;
                if (rank == 0) st.w += (unsigned long long)L * L;
                if (first == q) sm.gbase[q] = (unsigned short)atomicAdd(s_pcur, L);
            }
        }
    }
    __syncthreads();
    // ---- E: dense, ordered groups in shared memory (the candidate arrays are dead: alias them) ---------------
    uint32_t* stg_g = sm.K2;                                                     // [BK_CAP]
    unsigned short* stg_rem = reinterpret_cast<unsigned short*>(sm.G2);          // [BK_CAP]
    const bool can_inline = a.gb <= YG_ITEM_INLINE_BITS;
    if (m_next > a.m_lo && m_next <= GK_FAST * GK_THREADS) {      // start2 / SUB2 were last read in phase D: stage the next bucket there
        const uint64_t* nsrc = a.ent + bb_next + tid;
        const uint32_t sdst = (uint32_t)__cvta_generic_to_shared(stage + tid);
#pragma unroll
        for (int k = 0; k < GK_FAST; k++)
            if (k * GK_THREADS + tid < m_next)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sdst + k * GK_THREADS * 8), "l"(nsrc + k * GK_THREADS) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
        if (lr[k]) {
            const uint32_t L = lr[k] & 0xffffu, rank = lr[k] >> 16;
            const uint32_t x = (uint32_t)sm.gbase[qf[k]] + rank;
            stg_g[x] = gq[k];
            stg_rem[x] = (unsigned short)((L - 1 - rank) | ((!can_inline || L > 4) ? 0x8000u : 0u));
        }
    }
    __syncthreads();
    // ---- F: postings + work items -------------------------------------------------------------------------------
    const uint32_t np = *s_pcur;
    for (uint32_t x = tid; x < np; x += GK_THREADS) {
        const uint32_t g = stg_g[x];
        const uint32_t rr = stg_rem[x];
        const uint32_t rem = rr & 0x7fffu;
        if (rr & 0x8000u) a.post[(uint64_t)bb + x] = g;
        if (rem) {
            uint64_t item;
            if (can_inline && rem <= 3) {
                item = (uint64_t)rem | ((uint64_t)stg_g[x + 1] << 2);
                if (rem >= 2) item |= (uint64_t)stg_g[x + 2] << 22;
                if (rem >= 3) item |= (uint64_t)stg_g[x + 3] << 42;
            } else {
                item = (((uint64_t)bb + x + 1) << 32) | ((uint64_t)rem << 2);
            }
            const uint32_t slot = atomicAdd(reinterpret_cast<unsigned int*>(&a.row_cnt[g]), 1u);
            const uint32_t dst = (uint32_t)a.row_off[g];
            if (pd.has) a.row_items[(uint64_t)pd.dst + pd.slot] = pd.item;     // the append issued one bucket ago
            pd.item = item; pd.dst = dst; pd.slot = slot; pd.has = true;
        }
    }
}

__global__ void __launch_bounds__(GK_THREADS, 4) k2_group(const GroupArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GroupSmem sm;
    sm.cnt = (uint32_t*)smem_raw;                                    // 8 KB
    sm.K2 = sm.cnt + GK_NSUB;                                        // 12 KB
    sm.G2 = sm.K2 + BK_CAP;                                          // 12 KB
    sm.start2 = (unsigned short*)(sm.G2 + BK_CAP);                   // 4 KB + 16
    sm.SUB2 = sm.start2 + GK_NSUB + 8;                               // 6 KB
    sm.gbase = sm.SUB2 + BK_CAP;                                     // 6 KB
    __shared__ uint32_t s_wsum[GK_THREADS / 32];
    __shared__ uint32_t s_pcur[2], s_gpos[2];
    sm.s_wsum = s_wsum;

    for (uint32_t i = threadIdx.x; i < GK_NSUB; i += GK_THREADS) sm.cnt[i] = 0;
    __syncthreads();
    GroupStats st{0, 0, 0, 0ull};
    GroupPending pd{0ull, 0u, 0u, false};
    uint32_t par = 0;
    uint32_t b = a.b_lo + blockIdx.x;
    uint32_t bb = 0, m = 0;
    if (b < a.b_hi) { bb = a.begin[b]; m = a.end[b] - bb; }
    bool staged = false;
    while (b < a.b_hi) {
        // the next bucket's extent is fetched now and used in phase E, where its words are prefetched
        const uint32_t bn = b + gridDim.x;
        uint32_t bbn = 0, mn = 0;
        if (bn < a.b_hi) { bbn = a.begin[bn]; mn = a.end[bn] - bbn; }
        if (m > a.m_lo && m <= BK_CAP) {    // uniform per CTA (larger buckets: k2_big_*, below)
            if (m <= GK_FAST * GK_THREADS) group_bucket<GK_FAST>(a, bb, m, sm, &s_pcur[par], &s_gpos[par], st, pd, staged, bbn, mn);
            else group_bucket<GK_SLOW>(a, bb, m, sm, &s_pcur[par], &s_gpos[par], st, pd, false, bbn, mn);
            par ^= 1;
            staged = mn > a.m_lo && mn <= GK_FAST * GK_THREADS;
        } else {
            staged = false;
        }
        b = bn; bb = bbn; m = mn;
    }
    if (pd.has) a.row_items[(uint64_t)pd.dst + pd.slot] = pd.item;
    const unsigned long long heads = block_sum<GK_THREADS>(st.heads);
    const unsigned long long single = block_sum<GK_THREADS>(st.single);
    const unsigned long long w = block_sum<GK_THREADS>(st.w);
    const unsigned long long dups = block_sum<GK_THREADS>(st.dups);
    if (threadIdx.x == 0) {
        if (heads) atomicAdd(&a.scal[SC_HEADS], heads);
        if (single) atomicAdd(&a.scal[SC_SINGLE], single);
        if (w) atomicAdd(&a.scal[SC_W], w);
        if (dups) atomicAdd(&a.scal[SC_DUPS], dups);
    }
}

// ---- k2_group2: the grouping kernel for the common case ---------------------------------------------------------
// Buckets of <= G2_MAXM words whose remaining hash bits (below the sub-bucket digit) fit 32 bits -- every bucket of a
// database without extreme skew.  Same idea as k2_group (sub-bucket counting filter, dense candidate scan), rebuilt
// around the instruction count, which is what bounds this step (not HBM):
//   * the bucket's words arrive by ONE bulk asynchronous copy (cp.async.bulk + mbarrier) into a ring of two stage
//     buffers, requested two buckets ahead; every thread then picks its four words with two 16-byte loads;
//   * the candidate-array room of a sub-bucket is claimed by its first word (warp scan + one shared atomic per warp),
//     so a bucket costs four CTA barriers and no pass over the 2 048 sub-bucket counters.  The order of the sub-buckets
//     inside a region is therefore the order in which the warps' atomics land, and it varies from run to run; so do
//     the positions of a bucket's postings and the posting offsets inside indirect items.  Nothing depends on them:
//     items are order-free, k2_group allocates its group slots with atomics too, and the flagged pairs are sorted;
//   * a candidate is one 64-bit word (remaining hash << 32 | genome id) plus the extent of its sub-bucket, so the scan
//     of a sub-bucket is one load and three compares per word, branch-free and fixed-length (4) for sub-buckets of
//     <= 4 words (all but a few per bucket);
//   * no allocation of posting slots: a candidate's slot is its rank in the (hash, genome) order of its sub-bucket,
//     which the same scan yields.  Groups come out contiguous and ordered; candidates that turn out to be alone leave
//     a hole that the output phase skips.  One barrier and the per-group shared-memory atomics of k2_group disappear.
constexpr int G2_THREADS = 256;
constexpr int G2_WIN = 1024;                      // words of the 16-byte aligned window copied per bucket
constexpr uint32_t G2_MAXM = G2_WIN - 2;          // largest bucket this kernel takes
constexpr int G2_NSUB = 1 << GK_SUBBITS;          // 2048 sub-bucket counters = 8 per thread
constexpr uint32_t IG_MAXL = 16;                  // sharded build: groups up to this size travel as self-contained items
constexpr uint64_t IG_ROW_MUL = (IG_MAXL - 1 + 2) / 3;   // ... so one shared hash is worth at most this many items of a query row

struct __align__(16) G2Smem {
    uint64_t stage[2][G2_WIN];                    // ring of two bucket windows (bulk copy targets): the CTA's i-th bucket lands in stage[i & 1]
    uint64_t cand[G2_WIN + 4];                    // candidates, sub-bucket by sub-bucket: remaining hash << 32 | genome id
    uint32_t cnt[G2_NSUB];                        // sub-bucket sizes; after phase B: start in its region | size << 16 (zero between buckets)
    uint32_t ext[G2_WIN];                         // per candidate of a sub-bucket of >= 3 words: start of its sub-bucket | size << 16
    uint32_t stg_g[G2_WIN + 4];                   // ordered groups: genome id
    unsigned short stg_r[G2_WIN];                 // ordered groups: members that follow | 0x8000 posting wanted | 0x4000 hole
    uint32_t wsum[G2_THREADS / 32];
    uint32_t next[2][2];                          // {first word, words} of the CTA's i-th bucket in next[i & 1] (words = 0: none)
    uint32_t cur;                                 // phase B cursor: words claimed in the pair region | in the larger region << 16
    uint32_t dcnt[YG_MAX_RANKS];                  // STREAM: items of this bucket per destination rank
    uint32_t dbase[YG_MAX_RANKS];                 // STREAM: ... and where they start in that rank's inbox
    uint64_t mbar[2];                             // "full" barrier of each stage buffer
};

template <bool STREAM, int MIN_CTAS>
__global__ void __launch_bounds__(G2_THREADS, MIN_CTAS) k2_group2(const GroupArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    G2Smem& sm = *reinterpret_cast<G2Smem*>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gmask = a.gb ? (uint32_t)((1ull << a.gb) - 1ull) : 0u;
    const uint32_t kmask = (uint32_t)a.rest_mask;
    const bool can_inline = a.gb <= YG_ITEM_INLINE_BITS;

    // The scheduler is the last thread: its warp has the least phase-D work (candidates are dealt out from thread 0 up).
    // It picks the CTA's buckets (stride gridDim.x, skipping empty ones and those over G2_MAXM words) two ahead: while
    // bucket i is grouped, the words of bucket i + 1 are already in flight and those of bucket i + 2 are requested in
    // phase D of bucket i, into the stage buffer bucket i's phase A has released.  Unless it has to skip buckets, the
    // barrier after phase D never waits on its loads.
    constexpr uint32_t SCHED = G2_THREADS - 1;
    const uint32_t b_end = a.range ? (uint32_t)a.range[1] : a.b_hi;
    uint32_t b_next = (a.range ? (uint32_t)a.range[0] : a.b_lo) + blockIdx.x;       // scheduler only
    // the extent of bucket b_next is fetched one bucket before it is needed, so that its two dependent loads are not waited for
    uint32_t pre_lo = 0, pre_hi = 0;
    auto preload = [&]() {
        if (b_next < b_end) { pre_lo = a.begin[b_next]; pre_hi = a.end[b_next]; }
    };
    auto advance = [&](uint32_t slot) {
        uint32_t bb = 0, m = 0;
        while (b_next < b_end) {
            bb = pre_lo;
            m = pre_hi - pre_lo;
            b_next += gridDim.x;
            if (m && m <= G2_MAXM) break;
            m = 0;
            preload();
        }
        sm.next[slot][0] = bb;
        sm.next[slot][1] = m;
        if (m) {
            const uint32_t w0 = bb & ~1u, w1 = (bb + m + 1u) & ~1u;
            bulk_load(sm.stage[slot], a.ent + w0, (w1 - w0) * 8u, &sm.mbar[slot]);
        }
        preload();
    };
    for (uint32_t i = tid; i < G2_NSUB; i += G2_THREADS) sm.cnt[i] = 0;
    if (tid == SCHED) {
        mbar_init(&sm.mbar[0], 1);
        mbar_init(&sm.mbar[1], 1);
        mbar_init_fence();
        sm.cur = 0;
        preload();
        advance(0);
        advance(1);
    }
    __syncthreads();

    uint32_t n_heads = 0, n_single = 0, n_dups = 0;
    unsigned long long n_w = 0;
    GroupPending pd{0ull, 0u, 0u, false}, pd2{0ull, 0u, 0u, false};   // two appends in flight: the atomic's answer is consumed two items later
    for (uint32_t it = 0;; it++) {
        const uint32_t par = it & 1u;
        const uint32_t bb = sm.next[par][0], m = sm.next[par][1];
        if (!m) break;
        mbar_wait(&sm.mbar[par], (it >> 1) & 1u);
        // ---- A: four words per thread, sub-bucket rank -----------------------------------------------------------
        const uint32_t wlo = bb & 1u, whi = wlo + m;                 // the bucket inside the copied window
        uint64_t e[4];
        {
            const uint4* s4 = reinterpret_cast<const uint4*>(sm.stage[par]);
            const uint4 v0 = s4[tid], v1 = s4[G2_THREADS + tid];
            e[0] = (uint64_t)v0.x | ((uint64_t)v0.y << 32); e[1] = (uint64_t)v0.z | ((uint64_t)v0.w << 32);
            e[2] = (uint64_t)v1.x | ((uint64_t)v1.y << 32); e[3] = (uint64_t)v1.z | ((uint64_t)v1.w << 32);
        }
        uint32_t sr[4];                                              // sub-bucket | rank << 16, ~0 = not a word of the bucket
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t w = (k >> 1) * 512u + 2u * tid + (k & 1);
            sr[k] = 0xFFFFFFFFu;
            if (w >= wlo && w < whi) {
                const uint32_t s = (uint32_t)(e[k] >> a.sub_shift) & a.sub_mask;
                sr[k] = s | (atomicAdd(&sm.cnt[s], 1u) << 16);
            }
        }
        __syncthreads();                                             // stage[par] is free (refilled in phase D)
        // ---- B: candidate-array place of every sub-bucket with >= 2 words, in TWO regions: sub-buckets of exactly two words
        //      (most of them: two genomes sharing a hash, or two hashes that merely share 11 bits) come first, as aligned
        //      pairs; phase D settles those with one compare.  Larger sub-buckets follow.  The word of rank 0 claims its
        //      sub-bucket's room: one warp scan and one shared-memory atomic per warp on a cursor that packs both regions
        //      (16 bits each).  Only the ~824 words of the bucket are visited, not the 2 048 counters; the order of the
        //      sub-buckets inside a region is the order of the claims.  The counter of a claimed sub-bucket becomes
        //      start in its region | size << 16 (an unclaimed one keeps its size, 1).
        {
            uint32_t cl[4];                                          // size of the sub-bucket this word claims (0: none)
            uint32_t own = 0;                                        // words claimed in the pair region | in the larger region << 16
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t c = sr[k] < 0x10000u ? sm.cnt[sr[k]] : 0u;     // rank 0 of a word of the bucket
                cl[k] = c >= 2 ? c : 0u;
                own += c == 2 ? 2u : (c >= 3 ? (c << 16) : 0u);
            }
            uint32_t inc = own;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
                if ((int)lane >= o) inc += v;
            }
            uint32_t wbase = 0;
            if (lane == 31 && inc) wbase = atomicAdd(&sm.cur, inc);
            const uint32_t ex = __shfl_sync(0xffffffffu, wbase, 31) + inc - own;
            uint32_t px = ex & 0xffffu, py = ex >> 16;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (cl[k]) {
                    const bool two = cl[k] == 2;
                    sm.cnt[sr[k]] = (two ? px : py) | (cl[k] << 16);
                    px += two ? 2u : 0u;
                    py += two ? 0u : cl[k];
                }
            }
        }
        __syncthreads();
        const uint32_t cur = sm.cur;
        const uint32_t nx = cur & 0xffffu, ncand = nx + (cur >> 16);
        // ---- C: candidates -> dense array, sub-bucket by sub-bucket; a word alone in its sub-bucket is a singleton ----
        uint32_t solo = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (sr[k] != 0xFFFFFFFFu) {
                const uint32_t v = sm.cnt[sr[k] & 0xffffu];
                if (v >= (2u << 16)) {
                    const uint32_t start = v >= (3u << 16) ? v + nx : v;   // larger region: after the nx pair words
                    const uint32_t pos = (start & 0xffffu) + (sr[k] >> 16);
                    const uint32_t K = (uint32_t)(e[k] >> a.gb) & kmask;
                    const uint32_t G = (uint32_t)e[k] & gmask;
                    sm.cand[pos] = ((uint64_t)K << 32) | (uint64_t)G;
                    if (v >= (3u << 16)) sm.ext[pos] = start;
                } else {
                    solo++;
                }
            }
        }
        n_heads += solo;
        n_single += solo;
        __syncthreads();
        // the counters and the cursor are free again: zero for the next bucket (its phase A is behind the barrier after D)
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (sr[k] != 0xFFFFFFFFu) sm.cnt[sr[k] & 0xffffu] = 0u;
        if (tid == SCHED) sm.cur = 0;
        // ---- D: group size, rank in the group (by genome id), slot in the (hash, genome) order of the sub-bucket ------------
        // pairs: the partner is the other word of the aligned pair
        for (uint32_t q = tid; q < nx; q += G2_THREADS) {
            const uint64_t wq = sm.cand[q], wp = sm.cand[q ^ 1u];
            const bool same = (uint32_t)(wp >> 32) == (uint32_t)(wq >> 32);
            const bool tie = (wp == wq) & (q & 1u);                          // same genome too (in-sketch duplicate): the even slot goes first
            const bool before = (wp < wq) | tie;
            const uint32_t pos = (q & ~1u) + (before ? 1u : 0u);
            sm.stg_g[pos] = (uint32_t)wq;
            sm.stg_r[pos] = same ? (unsigned short)((before ? 0u : 1u) | (can_inline ? 0u : 0x8000u)) : (unsigned short)0x4000u;
            n_heads += !(same & before);
            n_single += !same;
            n_dups += tie;
            if (same & !before) n_w += 4ull;
        }
        // larger sub-buckets: every candidate scans its sub-bucket once
        for (uint32_t q = nx + tid; q < ncand; q += G2_THREADS) {
            const uint64_t wq = sm.cand[q];
            const uint32_t x = sm.ext[q];
            const uint32_t lo = x & 0xffffu, c = x >> 16;
            const uint32_t Kq = (uint32_t)(wq >> 32);
            uint32_t L = 0, rank = 0, rall = 0, dup = 0;
            // four words of the sub-bucket per trip, branch-free: nearly every sub-bucket is done after one trip, clusters of
            // 5..8 genomes after two; lanes only diverge on the trip count
            for (uint32_t j0 = 0; j0 < c; j0 += 4) {
#pragma unroll
                for (uint32_t j = 0; j < 4; j++) {
                    const uint32_t jj = j0 + j;
                    const uint64_t w = sm.cand[lo + jj];
                    const bool valid = jj < c;
                    const bool same = valid & ((uint32_t)(w >> 32) == Kq);
                    const bool tie = valid & (w == wq) & (lo + jj < q);          // same genome too: in-sketch duplicate
                    const bool before = (valid & (w < wq)) | tie;
                    L += same ? 1u : 0u;
                    rank += (same & before) ? 1u : 0u;
                    rall += before ? 1u : 0u;
                    dup |= tie ? 1u : 0u;
                }
            }
            const uint32_t pos = lo + rall;
            sm.stg_g[pos] = (uint32_t)wq;
            sm.stg_r[pos] = L >= 2 ? (unsigned short)((L - 1 - rank) | ((!can_inline || L > (STREAM ? IG_MAXL : 4u)) ? 0x8000u : 0u)) : (unsigned short)0x4000u;
            n_heads += rank == 0;
            n_single += L == 1;
            n_dups += dup;
            if (L >= 2 && rank == 0) n_w += (unsigned long long)L * L;
        }
        if (tid == SCHED) advance(par);                              // bucket i + 2 -> stage[par]
        __syncthreads();
        if (STREAM) {
            // ---- F' (sharded build): the groups leave this rank --------------------------------------------------------------
            // (1) small groups: every non-last member becomes ceil(followers / 3) self-contained items, stored straight into
            //     the inbox of the rank that owns the member's query row (NVLink for peers); slots are claimed once per
            //     (bucket, destination) from this rank's cursors
            if (tid < (uint32_t)a.n_peers) sm.dcnt[tid] = 0;
            __syncthreads();
            bool any_big = false;
            for (uint32_t x = tid; x < ncand; x += G2_THREADS) {
                const uint32_t rr = sm.stg_r[x];
                sm.ext[x] = 0xFFFFFFFFu;
                if (rr & 0x4000u) continue;
                if (rr & 0x8000u) { any_big = true; continue; }
                const uint32_t rem = rr & 0x3fffu;
                if (!rem) continue;
                const uint32_t g = sm.stg_g[x];
                uint32_t dest = 0;
                for (int q = 1; q < a.n_peers; q++) dest += g >= a.row_bounds[q] ? 1u : 0u;
                sm.ext[x] = atomicAdd(&sm.dcnt[dest], (rem + 2u) / 3u) | (dest << 24);
            }
            any_big = __syncthreads_or(any_big);
            if (tid < (uint32_t)a.n_peers) {
                const uint32_t c = sm.dcnt[tid];
                sm.dbase[tid] = c ? (uint32_t)atomicAdd(&a.icursor[tid], (unsigned long long)c) : 0u;
            }
            __syncthreads();
            for (uint32_t x = tid; x < ncand; x += G2_THREADS) {
                const uint32_t ex = sm.ext[x];
                if (ex == 0xFFFFFFFFu) continue;
                const uint32_t dest = ex >> 24, rem = sm.stg_r[x] & 0x3fffu, g = sm.stg_g[x];
                uint64_t pos = (uint64_t)sm.dbase[dest] + (ex & 0xFFFFFFu);
                uint64_t* di = a.peer_item[dest] + a.item_region;
                uint32_t* dr = a.peer_row[dest] + a.item_region;
                for (uint32_t k = 0; k < rem; k += 3, pos++) {
                    const uint32_t c = min(3u, rem - k);
                    uint64_t item = (uint64_t)c | ((uint64_t)sm.stg_g[x + 1 + k] << 2);
                    if (c >= 2) item |= (uint64_t)sm.stg_g[x + 2 + k] << 22;
                    if (c >= 3) item |= (uint64_t)sm.stg_g[x + 3 + k] << 42;
                    if (pos < a.icap) { di[pos] = item; dr[pos] = g; }       // (an overflow shows in the cursor; the host checks it)
                }
            }
            // (2) larger groups (rare): their genome ids go, holes squeezed out, to EVERY rank's posting stream; the owners of
            //     the query rows derive indirect items from it (k2_items_regions)
            if (any_big) {
                uint32_t* cg = reinterpret_cast<uint32_t*>(sm.cand);                     // the candidate array is dead: compact copy
                unsigned short* cr = reinterpret_cast<unsigned short*>(cg + G2_WIN);
                uint32_t np = 0;
                for (uint32_t x0 = 0; x0 < ncand; x0 += G2_THREADS) {
                    const uint32_t x = x0 + tid;
                    const uint32_t rr = x < ncand ? sm.stg_r[x] : 0x4000u;
                    const bool member = !(rr & 0x4000u) && (rr & 0x8000u);
                    const uint32_t bal = __ballot_sync(0xffffffffu, member);
                    if (lane == 0) sm.wsum[warp] = __popc(bal);
                    __syncthreads();
                    uint32_t off = np, tot = 0;
#pragma unroll
                    for (int w = 0; w < G2_THREADS / 32; w++) {
                        const uint32_t c = sm.wsum[w];
                        off += (w < (int)warp) ? c : 0u;
                        tot += c;
                    }
                    if (member) {
                        const uint32_t pos = off + __popc(bal & ((1u << lane) - 1u));
                        cg[pos] = sm.stg_g[x];
                        cr[pos] = (unsigned short)(rr & 0x3fffu);
                    }
                    np += tot;
                    __syncthreads();
                }
                if (tid == 0) sm.wsum[0] = np ? (uint32_t)atomicAdd(&a.scal[SCM_STREAM], (unsigned long long)np) : 0u;
                __syncthreads();
                const uint64_t gpos = a.region_base + sm.wsum[0];
                for (int q = 0; q < a.n_peers; q++) {
                    uint32_t* dg = a.peer_gid[q] + gpos;
                    unsigned short* dr = a.peer_rem[q] + gpos;
                    for (uint32_t i = tid; i < np; i += G2_THREADS) { dg[i] = cg[i]; dr[i] = cr[i]; }
                }
            }
            continue;          // (the next bucket's first barrier separates its phases from this one)
        }
        // ---- F: postings + work items, one thread per ordered slot ------------------------------------------------------
        for (uint32_t x = tid; x < ncand; x += G2_THREADS) {
            const uint32_t rr = sm.stg_r[x];
            if (rr & 0x4000u) continue;
            const uint32_t g = sm.stg_g[x];
            const uint32_t rem = rr & 0x3fffu;
            if (rr & 0x8000u) a.post[(uint64_t)bb + x] = g;
            if (rem) {
                uint64_t item;
                if (can_inline && rem <= 3) {
                    item = (uint64_t)rem | ((uint64_t)sm.stg_g[x + 1] << 2);
                    if (rem >= 2) item |= (uint64_t)sm.stg_g[x + 2] << 22;
                    if (rem >= 3) item |= (uint64_t)sm.stg_g[x + 3] << 42;
                } else {
                    item = (((uint64_t)bb + x + 1) << 32) | ((uint64_t)rem << 2);
                }
                const uint32_t slot = atomicAdd(reinterpret_cast<unsigned int*>(&a.row_cnt[g]), 1u);
                const uint32_t dst = (uint32_t)a.row_off[g];
                if (pd.has) a.row_items[(uint64_t)pd.dst + pd.slot] = pd.item;     // the append issued two items ago
                pd = pd2;
                pd2.item = item; pd2.dst = dst; pd2.slot = slot; pd2.has = true;
            }
        }
        // (the next bucket's phase A only touches stage / cnt; its barriers order everything else against this phase F)
    }
    if (pd.has) a.row_items[(uint64_t)pd.dst + pd.slot] = pd.item;
    if (pd2.has) a.row_items[(uint64_t)pd2.dst + pd2.slot] = pd2.item;
    const unsigned long long heads = block_sum<G2_THREADS>(n_heads);
    const unsigned long long single = block_sum<G2_THREADS>(n_single);
    const unsigned long long w = block_sum<G2_THREADS>(n_w);
    const unsigned long long dups = block_sum<G2_THREADS>(n_dups);
    if (threadIdx.x == 0) {
        if (heads) atomicAdd(&a.scal[SC_HEADS], heads);
        if (single) atomicAdd(&a.scal[SC_SINGLE], single);
        if (w) atomicAdd(&a.scal[SC_W], w);
        if (dups) atomicAdd(&a.scal[SC_DUPS], dups);
    }
}

// ---- final buckets that do not fit shared memory (hashes held by thousands of genomes) ----------------------
// Only their words leave the partition path: they are gathered into one compact array under the key
// (bucket ordinal | remaining hash bits | genome id), sorted by one device-wide radix sort, and grouped by
// neighbour comparison -- same outputs as k2_group (postings, work items appended to the genome lists, the
// statistics), postings stored behind the T regular slots of d_post.  Everything else stays on the fast path.

__global__ void __launch_bounds__(256) k2_big_list(const uint32_t* __restrict__ begin, const uint32_t* __restrict__ end, uint32_t b_lo,
                                                   uint32_t b_hi, uint32_t* __restrict__ list, uint32_t list_cap,
                                                   unsigned long long* __restrict__ scal) {
    for (uint32_t b = b_lo + blockIdx.x * blockDim.x + threadIdx.x; b < b_hi; b += gridDim.x * blockDim.x) {
        const uint32_t m = end[b] - begin[b];
        if (m > BK_CAP) {
            const unsigned long long k = atomicAdd(&scal[SCM_STREAM], 1ull);       // (slot unused outside stream mode)
            if (k < list_cap) list[k] = b;
        }
    }
}

__global__ void __launch_bounds__(256) k2_big_gather(const uint64_t* __restrict__ ent, const uint32_t* __restrict__ begin,
                                                     const uint32_t* __restrict__ end, const uint32_t* __restrict__ list, const uint64_t* __restrict__ cstart, uint32_t n_big,
                                                     int low_bits, uint64_t* __restrict__ out) {
    const uint64_t lowmask = low_bits >= 64 ? ~0ull : ((1ull << low_bits) - 1ull);
    for (uint32_t j = blockIdx.x; j < n_big; j += gridDim.x) {
        const uint32_t b = list[j];
        const uint64_t bb = begin[b], m = end[b] - begin[b], dst = cstart[j];
        const uint64_t tag = low_bits >= 64 ? 0ull : ((uint64_t)j << low_bits);
        for (uint64_t i = threadIdx.x; i < m; i += blockDim.x) out[dst + i] = tag | (ent[bb + i] & lowmask);
    }
}

// first slot e > s whose (word >> gb) differs (exponential probe, then bisection)
__device__ __forceinline__ uint64_t big_run_end(const uint64_t* __restrict__ S, uint64_t s, uint64_t n, int gb) {
    const uint64_t k = S[s] >> gb;
    uint64_t lo = s, step = 1, hi = s + 1;
    while (hi < n && (S[hi] >> gb) == k) { lo = hi; step <<= 1; hi = lo + step; }
    if (hi > n) hi = n;
    while (hi - lo > 1) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if ((S[mid] >> gb) == k) lo = mid; else hi = mid;
    }
    return hi;
}

__global__ void __launch_bounds__(256) k2_big_groups(const uint64_t* __restrict__ S, uint64_t n, int gb, uint64_t post_base, int can_inline,
                                                     uint32_t* __restrict__ post, const uint64_t* __restrict__ row_off,
                                                     unsigned long long* __restrict__ row_cnt, uint64_t* __restrict__ row_items,
                                                     unsigned long long* __restrict__ scal) {
    const uint64_t gmask = gb ? ((1ull << gb) - 1ull) : 0ull;
    unsigned long long heads = 0, singles = 0, dups = 0, w = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t x = S[i], k = x >> gb;
        const bool peq = i > 0 && (S[i - 1] >> gb) == k;
        const bool neq = i + 1 < n && (S[i + 1] >> gb) == k;
        heads += !peq;
        singles += !peq && !neq;
        if (!peq && !neq) continue;
        const uint32_t g = (uint32_t)(x & gmask);
        const uint64_t rem = big_run_end(S, i, n, gb) - i - 1;
        post[post_base + i] = g;
        w += 2ull * rem + 1ull;                       // summed over a run of L members: L^2
        if (peq && (uint32_t)(S[i - 1] & gmask) == g) dups++;
        if (rem) {
            uint64_t item;
            if (can_inline && rem <= 3) {
                item = rem | ((S[i + 1] & gmask) << 2);
                if (rem >= 2) item |= (S[i + 2] & gmask) << 22;
                if (rem >= 3) item |= (S[i + 3] & gmask) << 42;
            } else {
                item = ((post_base + i + 1) << 32) | (rem << 2);
            }
            const unsigned long long slot = atomicAdd(reinterpret_cast<unsigned int*>(&row_cnt[g]), 1u);   // (32-bit: twice the L2 atomic rate; T < 2^32)
            row_items[row_off[g] + slot] = item;
        }
    }
    heads = block_sum<256>(heads);
    singles = block_sum<256>(singles);
    dups = block_sum<256>(dups);
    w = block_sum<256>(w);
    if (threadIdx.x == 0) {
        if (heads) atomicAdd(&scal[SC_HEADS], heads);
        if (singles) atomicAdd(&scal[SC_SINGLE], singles);
        if (dups) atomicAdd(&scal[SC_DUPS], dups);
        if (w) atomicAdd(&scal[SC_W], w);
    }
}

// sharded build, receiving side.  Work items arrive (a) ready-made in the item inbox: region q holds ilens[q * n_regions + me]
// items of rank q for rows of this rank; (b) as the posting stream of the larger groups: N regions of `cap` slots, region q holding
// lens[q] entries, every rank holds all of it and derives the (indirect) items of its own rows.  Row g's list lives at
// row_ptr[g] with room for IG_ROW_MUL * |S_g| + 8 items (k2s_sizes), which cannot be exceeded without in-sketch duplicates; if it
// is, *overflow is raised and the step is refused -- callers then run the database on one GPU.
__global__ void __launch_bounds__(256) k2_inbox(const uint64_t* __restrict__ items, const uint32_t* __restrict__ rows,
                                                const unsigned long long* __restrict__ report, int n_regions, int me, uint64_t icap,
                                                const uint64_t* __restrict__ row_ptr, const uint32_t* __restrict__ sizes,
                                                unsigned long long* __restrict__ row_cnt, uint64_t* __restrict__ row_items,
                                                unsigned long long* __restrict__ overflow) {
    {
        const int q = blockIdx.y;                 // one grid row per sending rank: the regions are worked off side by side
        const uint64_t base = (uint64_t)q * icap;
        const uint64_t len = min((uint64_t)report[(size_t)q * REP_WORDS + REP_ICUR + me], icap);
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (uint64_t)gridDim.x * blockDim.x) {
            const uint32_t g = rows[base + i];
            const uint64_t item = items[base + i];
            const unsigned long long slot = atomicAdd(reinterpret_cast<unsigned int*>(&row_cnt[g]), 1u);   // (32-bit: twice the L2 atomic rate; T < 2^32)
            if (slot < IG_ROW_MUL * sizes[g] + 8ull) row_items[row_ptr[g] + slot] = item;
            else *overflow = 1ull;
        }
    }
}

__global__ void __launch_bounds__(256) k2_items_regions(const uint32_t* __restrict__ gid, const unsigned short* __restrict__ rem,
                                                        const unsigned long long* __restrict__ report, int n_regions, uint64_t cap,
                                                        uint32_t row_begin, uint32_t row_end, int can_inline, const uint64_t* __restrict__ row_ptr,
                                                        const uint32_t* __restrict__ sizes, unsigned long long* __restrict__ row_cnt,
                                                        uint64_t* __restrict__ row_items, unsigned long long* __restrict__ overflow) {
    {
        const int q = blockIdx.y;
        const uint64_t base = (uint64_t)q * cap, len = report[(size_t)q * REP_WORDS + SCM_STREAM];
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (uint64_t)gridDim.x * blockDim.x) {
            const uint64_t x = base + i;
            const uint32_t r = rem[x];
            if (!r) continue;
            const uint32_t g = gid[x];
            if (g < row_begin || g >= row_end) continue;
            uint64_t item;
            if (can_inline && r <= 3) {
                item = (uint64_t)r | ((uint64_t)gid[x + 1] << 2);
                if (r >= 2) item |= (uint64_t)gid[x + 2] << 22;
                if (r >= 3) item |= (uint64_t)gid[x + 3] << 42;
            } else {
                item = ((x + 1) << 32) | ((uint64_t)r << 2);
            }
            const unsigned long long slot = atomicAdd(reinterpret_cast<unsigned int*>(&row_cnt[g]), 1u);   // (32-bit: twice the L2 atomic rate; T < 2^32)
            if (slot < IG_ROW_MUL * sizes[g] + 8ull) row_items[row_ptr[g] + slot] = item;
            else *overflow = 1ull;
        }
    }
}

// ---- sharded build: one CTA turns the all-gathered level-1 histograms into the exchange plan --------------------------
// Every rank computes the same plan from the same table: digit d belongs to rank floor(N * hashes before d / T) (contiguous
// digit ranges of nearly equal hash counts); inside its owner's level-1 buffer the words of digit d lie at (hashes of the
// owner's earlier digits) + (words of digit d from lower ranks), so every source rank knows exactly where its words go and
// the level-1 scatter can store them there directly.  For the digits this rank owns it also lays out level 2 (bucket
// bases and tile prefix in the GLOBAL digit numbering: foreign digits are simply empty).
// slots of ctx->d_sh_info (LENS: [nranks] posting-stream lengths; ICUR: [nranks] items sent to every rank; ILENS: [nranks][nranks] all-gathered)
enum { SHI_DLO = 0, SHI_DHI = 1, SHI_TMINE = 2, SHI_BLO = 3, SHI_BHI = 4, SHI_TMAX = 5, SHI_LENS = 8, SHI_ICUR = 64, SHI_ILENS = 96, SHI_WORDS = 1024 };

__global__ void __launch_bounds__(1024) k2s_prep(const uint32_t* __restrict__ hist_all, uint32_t nb, int nranks, int rank, int d2,
                                                 uint32_t* __restrict__ owner, uint32_t* __restrict__ cursor, uint32_t* __restrict__ base,
                                                 uint32_t* __restrict__ tile_start, unsigned long long* __restrict__ info,
                                                 unsigned long long* __restrict__ scal) {
    typedef cub::BlockScan<unsigned long long, 1024> Scan64;
    typedef cub::BlockScan<uint32_t, 1024> Scan32;
    __shared__ typename Scan64::TempStorage ts0;
    __shared__ typename Scan32::TempStorage ts1, ts2;
    __shared__ unsigned char s_own[NB_MAX];
    __shared__ unsigned long long s_start[YG_MAX_RANKS], s_owned[YG_MAX_RANKS];
    __shared__ uint32_t s_lo, s_hi;
    constexpr int per = (NB_MAX + 1023) / 1024;
    unsigned long long g[per], pre[per], gs = 0;
    for (int k = 0; k < per; k++) {
        const uint32_t d = threadIdx.x * per + k;
        g[k] = 0; pre[k] = 0;
        if (d < nb)
            for (int q = 0; q < nranks; q++) {
                const uint32_t h = hist_all[(size_t)q * NB_MAX + d];
                g[k] += h;
                if (q < rank) pre[k] += h;
            }
        gs += g[k];
    }
    unsigned long long acc, total;
    Scan64(ts0).ExclusiveSum(gs, acc, total);
    if (threadIdx.x == 0) { s_lo = 0xFFFFFFFFu; s_hi = 0; }
    if (threadIdx.x < YG_MAX_RANKS) s_owned[threadIdx.x] = 0;
    unsigned long long ex[per];
    uint32_t own[per];
    for (int k = 0; k < per; k++) {
        const uint32_t d = threadIdx.x * per + k;
        ex[k] = acc;
        acc += g[k];
        own[k] = total ? (uint32_t)min((unsigned long long)(nranks - 1), ex[k] * (unsigned long long)nranks / total) : 0u;
        if (d < nb) s_own[d] = (unsigned char)own[k];
    }
    __syncthreads();
    for (int k = 0; k < per; k++) {
        const uint32_t d = threadIdx.x * per + k;
        if (d < nb && (d == 0 || s_own[d - 1] != own[k])) s_start[own[k]] = ex[k];
        if (d < nb && g[k]) atomicAdd(&s_owned[own[k]], g[k]);
    }
    __syncthreads();
    uint32_t hm[per], tl[per], hs = 0, tsum = 0, mx = 0;
    for (int k = 0; k < per; k++) {
        const uint32_t d = threadIdx.x * per + k;
        hm[k] = 0;
        if (d < nb) {
            owner[d] = own[k];
            cursor[d] = (uint32_t)(ex[k] - s_start[own[k]] + pre[k]);
            if ((int)own[k] == rank) {
                hm[k] = (uint32_t)g[k];
                atomicMin(&s_lo, d);
                atomicMax(&s_hi, d + 1);
            }
        }
        tl[k] = (hm[k] + SC_TILE - 1) / SC_TILE;
        hs += hm[k]; tsum += tl[k]; mx = max(mx, hm[k]);
    }
    uint32_t hoff, toff, htot, ttot;
    Scan32(ts1).ExclusiveSum(hs, hoff, htot);
    Scan32(ts2).ExclusiveSum(tsum, toff, ttot);
    for (int k = 0; k < per; k++) {
        const uint32_t d = threadIdx.x * per + k;
        if (d < nb) { base[d] = hoff; tile_start[d] = toff; }
        hoff += hm[k]; toff += tl[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        base[nb] = htot; tile_start[nb] = ttot;
        const uint32_t lo = s_lo == 0xFFFFFFFFu ? 0u : s_lo, hi = s_lo == 0xFFFFFFFFu ? 0u : s_hi;
        info[SHI_DLO] = lo; info[SHI_DHI] = hi; info[SHI_TMINE] = htot;
        info[SHI_BLO] = (unsigned long long)lo << d2; info[SHI_BHI] = (unsigned long long)hi << d2;
        unsigned long long tmax = 0;
        for (int q = 0; q < nranks; q++) tmax = max(tmax, s_owned[q]);
        info[SHI_TMAX] = tmax;          // the most words any rank owns: every rank knows whether the exchange buffers suffice
    }
    if (mx) atomicMax(&scal[SCM_MAXB], (unsigned long long)mx);
}

// sketch sizes of ALL genomes, the slice-relative offsets (genome-range residency) and the work-list starts of this rank's
// query rows [g_begin, g_end): row g has room for IG_ROW_MUL * |S_g| + 8 items (a shared hash is worth ceil(followers / 3) items,
// at most IG_ROW_MUL for a group of IG_MAXL; the indirect items of larger groups are one per hash)
__global__ void __launch_bounds__(256) k2s_sizes(const uint64_t* __restrict__ offsets, uint32_t n, uint32_t g_begin, uint32_t g_end,
                                                 uint32_t* __restrict__ sizes, uint64_t* __restrict__ row_begin_local,
                                                 uint64_t* __restrict__ offsets_local) {
    const uint64_t o0 = offsets[g_begin];
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g <= n; g += gridDim.x * blockDim.x) {
        if (g < n) {
            sizes[g] = (uint32_t)(offsets[g + 1] - offsets[g]);
            row_begin_local[g] = (g >= g_begin && g < g_end) ? IG_ROW_MUL * (offsets[g] - o0) + 8ull * (g - g_begin) : 0ull;
        }
        if (offsets_local && g >= g_begin && g <= g_end) offsets_local[g - g_begin] = offsets[g] - o0;
    }
}

// first / last level-1 digit this rank holds words of (hash-range residency: its hash range), as bucket range for the grouping
__global__ void __launch_bounds__(1024) k2s_range(const uint32_t* __restrict__ hist, uint32_t nb, int d2, unsigned long long T_mine,
                                                  unsigned long long* __restrict__ info) {
    __shared__ uint32_t s_lo, s_hi;
    if (threadIdx.x == 0) { s_lo = 0xFFFFFFFFu; s_hi = 0; }
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < nb; d += blockDim.x)
        if (hist[d]) { atomicMin(&s_lo, d); atomicMax(&s_hi, d + 1); }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t lo = s_lo == 0xFFFFFFFFu ? 0u : s_lo, hi = s_lo == 0xFFFFFFFFu ? 0u : s_hi;
        info[SHI_DLO] = lo; info[SHI_DHI] = hi; info[SHI_TMINE] = T_mine;
        info[SHI_BLO] = (unsigned long long)lo << d2; info[SHI_BHI] = (unsigned long long)hi << d2;
    }
}

// Views of ctx->d_msd_aux.  Per level and bucket b: begin, cap (exact layout: the histogram), the scatter's cursor (slotted:
// counts from zero; exact: a position, starting at begin) and, slotted layout only, end = begin + words.  Exact layout: bucket b
// spans [begin[b], begin[b + 1]), so its consumers take end = begin + 1.
struct MsdAux {
    uint32_t *begin1, *cap1, *cur1, *end1, *tile_start;            // [NB_MAX + 2] each
    uint32_t *begin2, *cap2, *cur2, *end2;                         // [nfb + 2] each (cap2 and cur2 adjacent: one memset)
    static uint64_t words(uint32_t nfb) { return 5ull * (NB_MAX + 2) + 4ull * ((uint64_t)nfb + 2); }
    MsdAux(uint32_t* x, uint32_t nfb) {
        const uint64_t s1 = NB_MAX + 2, s2 = (uint64_t)nfb + 2;
        begin1 = x; cap1 = begin1 + s1; cur1 = cap1 + s1; end1 = cur1 + s1; tile_start = end1 + s1;
        begin2 = tile_start + s1; cap2 = begin2 + s2; cur2 = cap2 + s2; end2 = cur2 + s2;
    }
};

// What the partition leaves behind (kept per context: `yacht run` probes many samples against one partitioned reference)
struct MsdPartState {
    MsdPlan p;
    int sbits = 0, rest_bits = 0;
    const uint64_t* final_ent = nullptr;
    const uint32_t* final_begin = nullptr;     // final bucket b: words [final_begin[b], final_end[b]) of final_ent
    const uint32_t* final_end = nullptr;
    uint32_t nbuckets = 0;
    uint64_t largest = 0;
};

int bitlen(uint64_t v) {
    int b = 0;
    while (b < 64 && (v >> b) != 0) b++;
    return b;
}

// Slot capacity of a bucket of the leading `bits` hash bits.  Sketch hashes are FracMinHash values, uniform in [0, maxkey], so a
// full bucket expects mean = T * 2^(hb - bits) / (maxkey + 1) words; the capacity is f * mean + add, rounded up to 16 words
// (every slot starts 16-byte aligned, as the bulk copies need).
uint64_t slot_capacity(uint64_t T, uint64_t maxkey, int hb, int bits, double f, double add) {
    const double mean = (double)T * std::ldexp(1.0, hb - bits) / ((double)maxkey + 1.0);
    const double c = std::ceil(f * mean + add);
    if (!(c < 4294967296.0)) return 1ull << 32;
    return ((uint64_t)c + 15ull) & ~15ull;
}

// Partition + grouping of the resident sketches on one GPU.  partition_only: stop after the partition (the run path probes
// it, run_buckets.cuh).  *used = 0 when the input does not qualify for this path.
//
// Bucket layout.  Slotted (the rule): bucket b of a level owns a fixed slot of C words at b * C, C from the plan alone
// (slot_capacity), so the scatters need no histogram; a (tile, digit) run that would pass its slot's end is cut and raises that
// level's overflow flag, which the host reads at the one synchronisation after the partition.  Exact (the fallback): a
// histogram pass sizes every bucket.  A level-2 overflow repeats level 2 on the exact layout; a level-1 overflow repeats the
// whole partition on it (level 2 ran on cut buckets).  Slot positions must fit 32 bits (work items address postings by
// position), otherwise the exact layout is taken from the start.
int msd_build(ygpu_ctx* ctx, ygpu_index_stats* S, int* used, bool partition_only = false) {
    *used = 0;
    ctx->part_valid = false;
    const uint64_t T = ctx->T;
    const uint32_t n = ctx->n;
    if (T < 2 || n < 2) return 0;
    cudaStream_t st = ctx->stream;

    // ---- plan -----------------------------------------------------------------------------------
    uint64_t maxkey = 0;
    YG_CHECK(ygpu_max_hash(ctx, &maxkey));
    MsdPlan p{};
    p.T = T;
    p.hb = std::max(1, bitlen(maxkey));
    p.gb = bitlen((uint64_t)n - 1);
    auto used_buckets = [&](int D) -> uint64_t { return D == 0 ? 1ull : (maxkey >> (p.hb - D)) + 1ull; };
    int D = 0;
    while (D < p.hb && D < 22 && T / used_buckets(D) > A_TARGET) D++;
    int d1 = D <= 8 ? D : (D + 1) / 2;
    const int need = p.hb + p.gb - 64;           // packing: hb - d1 + gb <= 64
    if (need > d1) d1 = need;
    if (d1 > 11 || d1 > p.hb) return 0;          // does not pack: general path
    int d2 = D - d1;
    if (d2 < 0) d2 = 0;
    if (d2 > 11) return 0;
    p.d1 = d1; p.d2 = d2; p.kb1 = p.hb - d1;
    p.nb1 = d1 ? (uint32_t)(maxkey >> (p.hb - d1)) + 1 : 1u;
    if (p.nb1 > NB_MAX) return 0;
    p.nfb = p.nb1 << d2;
    p.dlo = 0; p.dhi = p.nb1; p.unit_lo = 0; p.unit_hi = 0xFFFFFFFFu;
    // sub-bucket digit of the grouping kernel
    const int key_bits = p.kb1 - d2;                       // hash bits that still vary inside a final bucket
    const int sbits = std::max(0, std::min(GK_SUBBITS, key_bits));
    const int rest_bits = key_bits - sbits;                // compared inside a sub-bucket (32 low bits + the rest beside the genome id)
    if (!partition_only && rest_bits > 32 && rest_bits - 32 + p.gb > 32) return 0;     // does not fit the candidate arrays: general path
    // Slot capacities.  Level 1: 2 % over the mean plus one scatter tile -- at 85 205 genomes a full bucket averages 822 516 words
    // and the largest holds 827 327 (+0.6 %).  Level 2: 25 % over the mean plus 64 -- at 85 205 genomes the buckets average
    // 804 words with a standard deviation of 35.5 (Poisson: 28.4; clusters of related genomes widen it) and the largest holds
    // 984, against C2 = 1 072, 7.5 deviations over the mean.  A database that fills a slot anyway is re-partitioned exactly.
    const uint64_t C1 = slot_capacity(T, maxkey, p.hb, d1, 1.02, (double)SC_TILE);
    const uint64_t C2 = slot_capacity(T, maxkey, p.hb, d1 + d2, 1.25, 64.0);
    // Positions in a level's buffer, and behind the final one the postings of oversized buckets (at most T words), must fit 32
    // bits: slot space + T < 2^32.  (400 000 genomes, T = 2.1e9: the exact layout from the start.)
    const bool slots_fit = C1 * p.nb1 + T < (1ull << 32) && (!d2 || C2 * p.nfb + T < (1ull << 32));

    // ---- buffers ----------------------------------------------------------------------------------
    const uint64_t aux_words = MsdAux::words(p.nfb);
    YG_CHECK(dev_alloc(ctx, &ctx->d_msd_aux, aux_words));
    const MsdAux x(ctx->d_msd_aux, p.nfb);
    const uint32_t units1 = (uint32_t)((T + SC_TILE - 1) / SC_TILE);
    const uint64_t max_units = T / SC_TILE + p.nb1 + 1;
    YG_CHECK(dev_alloc(ctx, &ctx->d_tile_g0, (uint64_t)units1 + 1));
    if (d2) YG_CHECK(dev_alloc(ctx, &ctx->d_units, 2 * max_units));
    const uint64_t T_mine = T;
    ScatterArgs a{};
    a.hashes = ctx->d_hashes; a.offsets = ctx->d_offsets; a.n = n; a.tile_g0 = ctx->d_tile_g0;
    a.tile_start = x.tile_start; a.hist2 = x.cap2; a.units = (const uint2*)ctx->d_units;
    const size_t smem1 = (size_t)2 * SC_BUF * 8 + (size_t)p.nb1 * 16 + (size_t)SC_TILE * 2;
    const size_t smem2 = (size_t)2 * SC_BUF * 8 + (size_t)(1u << d2) * 16 + (size_t)SC_TILE * 2;
    int grid1 = 1, grid2 = 1;
    {
        int occ = 1;
        YG_CUDA(ctx, cudaFuncSetAttribute(k2_scatter<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k2_scatter<1, false>, SC_THREADS, smem1));
        grid1 = (int)std::min<uint64_t>(units1, (uint64_t)ctx->num_sms * std::max(occ, 1));
        if (d2) {
            YG_CUDA(ctx, cudaFuncSetAttribute(k2_scatter<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k2_scatter<2, false>, SC_THREADS, smem2));
            grid2 = ctx->num_sms * std::max(occ, 1);
        }
    }
    bool ran_hist1 = false, ran_hist2 = false;

    // level 1: raw hashes -> packed words in d_ent1, by leading digit
    auto level1 = [&](bool exact) -> int {
        YG_CUDA(ctx, cudaMemsetAsync(ctx->d_msd_aux, 0, aux_words * sizeof(uint32_t), st));
        YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SCM_PCUR], 0, (SCM_OVF2 + 1 - SCM_PCUR) * sizeof(unsigned long long), st));
        YG_CHECK(dev_alloc(ctx, &ctx->d_ent1, exact ? T : std::max<uint64_t>(T, C1 * p.nb1)));
        a.out_ent = ctx->d_ent1; a.cursor = x.cur1; a.ovf = &ctx->d_scalars[SCM_OVF1];
        a.slot = exact ? 0u : (uint32_t)C1;
        if (exact) {
            YG_CUDA(ctx, cudaEventRecord(ctx->evp[0], st));
            k2_hist1<<<ctx->num_sms * 8, 256, p.nb1 * sizeof(uint32_t), st>>>(ctx->d_hashes, p, x.cap1);
            YG_CUDA(ctx, cudaGetLastError());
            YG_CUDA(ctx, cudaEventRecord(ctx->evp[1], st));
            k2_prep1<<<1, 1024, 0, st>>>(x.cap1, nullptr, p.nb1, x.begin1, nullptr, x.cur1, x.tile_start, ctx->d_scalars);
            ran_hist1 = true;
        } else {
            k2_slots<<<grid_for(ctx, (uint64_t)p.nb1 + 1, 256, 8), 256, 0, st>>>(p.nb1, (uint32_t)C1, x.begin1, x.cap1);
        }
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[2], st));
        k2_scatter<1, false><<<grid1, SC_THREADS, smem1, st>>>(a, p, 0u, units1);
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[3], st));
        if (!exact) {
            k2_prep1<<<1, 1024, 0, st>>>(x.cur1, x.cap1, p.nb1, x.begin1, x.end1, nullptr, x.tile_start, ctx->d_scalars);
            YG_CUDA(ctx, cudaGetLastError());
        }
        ctx->tm.n_kernel_launches += 3;
        return 0;
    };
    // level 2: words -> final buckets in d_ent2, by the next d2 bits (the level-1 units are laid out once per level-1 pass)
    auto level2 = [&](bool exact, bool units) -> int {
        YG_CHECK(dev_alloc(ctx, &ctx->d_ent2, exact ? T : std::max<uint64_t>(T, C2 * p.nfb)));
        a.in_ent = ctx->d_ent1; a.out_ent = ctx->d_ent2;
        a.cursor = x.cur2; a.ovf = &ctx->d_scalars[SCM_OVF2];
        a.slot = exact ? 0u : (uint32_t)C2;
        if (units) {
            k2_units<<<grid_for(ctx, max_units, 256, 8), 256, 0, st>>>(x.tile_start, x.begin1, ran_hist1 ? x.begin1 + 1 : x.end1, p.nb1,
                                                                       (uint2*)ctx->d_units);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 1;
        }
        if (exact) {
            YG_CUDA(ctx, cudaEventRecord(ctx->evp[12], st));
            k2_hist2<<<ctx->num_sms * 8, 256, (size_t)(1u << d2) * sizeof(uint32_t), st>>>(a, p, p.unit_hi);
            YG_CUDA(ctx, cudaGetLastError());
            YG_CUDA(ctx, cudaEventRecord(ctx->evp[4], st));
            // final-bucket bases and the largest bucket
            size_t tb = 0, tb2 = 0;
            YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb, x.cap2, x.begin2, (int64_t)p.nfb + 1, st));
            YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb2, x.cap2, (uint32_t*)&ctx->d_scalars[SCM_MAXB + 1], (int64_t)p.nfb, st));
            YG_CHECK(ygpu_temp_reserve(ctx, std::max(tb, tb2)));
            tb = ctx->temp_bytes;
            YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, x.cap2, x.begin2, (int64_t)p.nfb + 1, st));
            tb = ctx->temp_bytes;
            YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, x.cap2, (uint32_t*)&ctx->d_scalars[SCM_MAXB + 1], (int64_t)p.nfb, st));
            ctx->tm.n_library_launches += 4;
            ctx->tm.n_kernel_launches += 1;
            YG_CUDA(ctx, cudaMemcpyAsync(x.cur2, x.begin2, (uint64_t)p.nfb * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
            ran_hist2 = true;
        } else {
            k2_slots<<<grid_for(ctx, (uint64_t)p.nfb + 1, 256, 8), 256, 0, st>>>(p.nfb, (uint32_t)C2, x.begin2, x.cap2);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 1;
        }
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[5], st));
        k2_scatter<2, false><<<grid2, SC_THREADS, smem2, st>>>(a, p, p.unit_lo, p.unit_hi);
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[6], st));
        ctx->tm.n_kernel_launches += 1;
        if (!exact) {
            k2_ends<<<grid_for(ctx, p.nfb, 256, 8), 256, 0, st>>>(x.cur2, x.cap2, x.begin2, p.nfb, x.end2, &ctx->d_scalars[SCM_MAXB + 1]);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 1;
        }
        return 0;
    };
    // largest buckets of both levels and the overflow flags, at the one synchronisation after the partition
    unsigned long long rb[SCM_OVF2 + 1 - SCM_MAXB] = {};
    auto read_back = [&]() -> int {
        YG_CUDA(ctx, cudaMemcpyAsync(rb, &ctx->d_scalars[SCM_MAXB], sizeof rb, cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        return 0;
    };

    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    // genome of the first hash slot of every level-1 tile (the scatter derives genome ids from the CSR offsets)
    k2_tile_g0<<<grid_for(ctx, (uint64_t)units1 + 1, 256, 8), 256, 0, st>>>(ctx->d_offsets, n, T, units1, ctx->d_tile_g0);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches += 1;
    bool exact1 = !slots_fit;
    YG_CHECK(level1(exact1));
    if (d2) YG_CHECK(level2(exact1, true));
    YG_CHECK(read_back());
    if (!exact1 && rb[SCM_OVF1 - SCM_MAXB]) {
        // a level-1 slot overflowed: everything after it ran on cut buckets -- the whole partition again, exactly
        exact1 = true;
        YG_CHECK(level1(true));
        if (d2) YG_CHECK(level2(true, true));
        YG_CHECK(read_back());
    } else if (d2 && !exact1 && rb[SCM_OVF2 - SCM_MAXB]) {
        YG_CUDA(ctx, cudaMemsetAsync(x.cap2, 0, 2 * ((uint64_t)p.nfb + 2) * sizeof(uint32_t), st));      // histogram + cursors
        YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SCM_MAXB + 1], 0, sizeof(unsigned long long), st));
        YG_CHECK(level2(true, false));
        YG_CHECK(read_back());
    }
    const uint64_t* final_ent = d2 ? ctx->d_ent2 : ctx->d_ent1;
    const uint32_t* final_begin = d2 ? x.begin2 : x.begin1;
    const uint32_t* final_end = d2 ? (ran_hist2 ? x.begin2 + 1 : x.end2) : (ran_hist1 ? x.begin1 + 1 : x.end1);
    // positions in the final buffer: the slot space, or T (exact layout)
    const uint64_t final_words = d2 ? (ran_hist2 ? T : std::max<uint64_t>(T, C2 * p.nfb)) : (ran_hist1 ? T : std::max<uint64_t>(T, C1 * p.nb1));
    // largest final bucket decides whether the shared-memory grouping applies
    const uint64_t largest = d2 ? (uint64_t)(uint32_t)rb[1] : (uint64_t)rb[0];   // (level-1 maximum: over all digits, a safe bound)
    const uint32_t nbuckets = d2 ? p.nfb : p.nb1;
    {
        if (!ctx->part_state) ctx->part_state = new MsdPartState();
        MsdPartState* ps = (MsdPartState*)ctx->part_state;
        ps->p = p; ps->sbits = sbits; ps->rest_bits = rest_bits; ps->final_ent = final_ent;
        ps->final_begin = final_begin; ps->final_end = final_end;
        ps->nbuckets = nbuckets; ps->largest = largest;
        ctx->part_valid = true;
    }
    auto record_phases = [&]() {
        auto el = [&](int x0, int y0) { float ms = 0.f; cudaEventElapsedTime(&ms, ctx->evp[x0], ctx->evp[y0]); return (double)ms; };
        // phase times of the partition that was kept (a discarded slotted attempt shows in ms_sort only)
        if (ran_hist1) ctx->tm.ms_hist1 += el(0, 1);
        ctx->tm.ms_scatter1 += el(2, 3);
        if (d2) {
            if (ran_hist2) ctx->tm.ms_hist2 += el(12, 4);
            ctx->tm.ms_scatter2 += el(5, 6);
        }
    };
    if (partition_only) {
        ctx->tm.ms_sort += elapsed(ctx, 0, 1);
        record_phases();            // the run path's own partition reports its phases (and a retry) like the index build's
        *used = 1;
        return 0;
    }
    uint32_t n_big = 0;
    uint64_t N_big = 0;
    std::vector<uint32_t> big_list;
    std::vector<uint64_t> big_cstart;
    const int low_bits = (p.kb1 - d2) + p.gb;          // what distinguishes two words of one final bucket
    if (largest > BK_CAP) {
        // some final buckets do not fit shared memory.  Sharded builds and option big_buckets = 0 leave the whole
        // database to the general (sort) path; otherwise only those buckets take the k2_big_* route.
        bool ok = ctx->big_buckets != 0;
        if (ok) {
            YG_CHECK(dev_alloc(ctx, &ctx->d_big_list, (uint64_t)nbuckets));
            YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SCM_STREAM], 0, sizeof(unsigned long long), st));
            k2_big_list<<<grid_for(ctx, nbuckets, 256, 8), 256, 0, st>>>(final_begin, final_end, 0, nbuckets, ctx->d_big_list, nbuckets,
                                                                        ctx->d_scalars);
            YG_CUDA(ctx, cudaGetLastError());
            unsigned long long nb = 0;
            YG_CUDA(ctx, cudaMemcpyAsync(&nb, &ctx->d_scalars[SCM_STREAM], sizeof nb, cudaMemcpyDeviceToHost, st));
            YG_CUDA(ctx, cudaStreamSynchronize(st));
            ok = nb >= 1 && nb <= nbuckets && low_bits < 64;
            if (ok) {
                n_big = (uint32_t)nb;
                big_list.resize(n_big);
                YG_CUDA(ctx, cudaMemcpy(big_list.data(), ctx->d_big_list, (size_t)n_big * sizeof(uint32_t), cudaMemcpyDeviceToHost));
                std::sort(big_list.begin(), big_list.end());          // deterministic ordinals
                std::vector<uint32_t> hb(nbuckets), he(nbuckets);
                YG_CUDA(ctx, cudaMemcpy(hb.data(), final_begin, (size_t)nbuckets * sizeof(uint32_t), cudaMemcpyDeviceToHost));
                YG_CUDA(ctx, cudaMemcpy(he.data(), final_end, (size_t)nbuckets * sizeof(uint32_t), cudaMemcpyDeviceToHost));
                big_cstart.assign((size_t)n_big + 1, 0);
                for (uint32_t j = 0; j < n_big; j++) big_cstart[j + 1] = big_cstart[j] + (he[big_list[j]] - hb[big_list[j]]);
                N_big = big_cstart[n_big];
                ok = final_words + N_big + 4 < (1ull << 32);
            }
            YG_CUDA(ctx, cudaMemsetAsync(&ctx->d_scalars[SCM_STREAM], 0, sizeof(unsigned long long), st));
        }
        if (!ok) {
            ctx->msd_fallbacks++;
            return 0;                               // the general (sort) path handles it
        }
    }

    // ---- buckets -> postings + per-genome work lists (or the group stream) ------------------------------
    YG_CHECK(dev_alloc(ctx, &ctx->d_post, final_words + N_big));      // postings of oversized buckets: behind the final buffer's positions
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_items, T));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_cnt, (uint64_t)n + 1));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_row_cnt, 0, ((uint64_t)n + 1) * sizeof(unsigned long long), st));
    {
        GroupArgs g{};
        g.ent = final_ent; g.begin = final_begin; g.end = final_end; g.gb = p.gb;
        g.nb = d2 ? p.nfb : p.nb1;
        g.b_lo = d2 ? (p.dlo << d2) : p.dlo;
        g.b_hi = d2 ? (p.dhi << d2) : p.dhi;
        g.sub_shift = p.gb + rest_bits;
        g.sub_mask = (1u << sbits) - 1u;
        g.rest_mask = rest_bits >= 64 ? ~0ull : ((1ull << rest_bits) - 1ull);
        if (g.sub_shift > 63) { g.sub_shift = 0; g.sub_mask = 0; }
        g.post = ctx->d_post; g.row_off = ctx->d_offsets; g.row_cnt = ctx->d_row_cnt; g.row_items = ctx->d_row_items;
        g.st_gid = ctx->d_post; g.st_rem = ctx->d_st_rem; g.scal = ctx->d_scalars;
        const uint64_t nbk = g.b_hi > g.b_lo ? g.b_hi - g.b_lo : 0;
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[7], st));
        // the common case (remaining hash bits fit 32, bucket <= G2_MAXM words) goes to k2_group2; k2_group takes the rest
        const bool fast2 = rest_bits <= 32 && ctx->group_kernel != 1;
        g.m_lo = 0;
        if (fast2 && nbk) {
            const size_t smem2 = sizeof(G2Smem);
            // 4 CTAs per SM (61 registers) against 5 (48 registers, spills 24 bytes; measured slower): test hook "group_ctas"
            auto kern2 = ctx->group_ctas == 5 ? k2_group2<false, 5> : k2_group2<false, 4>;
            YG_CUDA(ctx, cudaFuncSetAttribute(kern2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            int occ2 = 1;
            YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, kern2, G2_THREADS, smem2));
            const int grid2 = (int)std::min<uint64_t>(nbk, (uint64_t)ctx->num_sms * std::max(occ2, 1));
            kern2<<<grid2, G2_THREADS, smem2, st>>>(g);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 1;
            g.m_lo = G2_MAXM;
        }
        if (nbk && (!fast2 || largest > G2_MAXM)) {
            const size_t smem = (size_t)GK_NSUB * 4 + (size_t)BK_CAP * 8 + (size_t)(GK_NSUB + 8) * 2 + (size_t)BK_CAP * 4;
            auto kern = k2_group;
            YG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int occ = 1;
            YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, GK_THREADS, smem));
            const int grid = (int)std::min<uint64_t>(nbk, (uint64_t)ctx->num_sms * std::max(occ, 1));
            kern<<<grid, GK_THREADS, smem, st>>>(g);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 1;
        }
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[8], st));
    }
    if (n_big) {
        // oversized buckets: gather under (ordinal | remaining hash bits | genome id), a device-wide sort, neighbour grouping.
        // The ordinal must fit beside the low_bits that tell two words of a bucket apart, and a sort handles < 2^30 words:
        // the list is worked off in chunks of consecutive buckets that satisfy both.
        const uint32_t ord_cap = (64 - low_bits) >= 31 ? 0x7FFFFFFFu : (1u << (64 - low_bits));
        uint64_t chunk_words_max = 0;
        std::vector<std::pair<uint32_t, uint32_t>> chunks;
        for (uint32_t c0 = 0; c0 < n_big;) {
            uint32_t c1 = c0;
            while (c1 < n_big && c1 - c0 < ord_cap && big_cstart[c1 + 1] - big_cstart[c0] < (1ull << 30)) c1++;
            if (c1 == c0) c1 = c0 + 1;          // a single bucket of >= 2^30 words cannot occur (T < 2^32 is split over >= 2 buckets) -- keep going anyway
            chunks.emplace_back(c0, c1);
            chunk_words_max = std::max<uint64_t>(chunk_words_max, big_cstart[c1] - big_cstart[c0]);
            c0 = c1;
        }
        YG_CHECK(dev_alloc(ctx, &ctx->d_big_a, chunk_words_max));
        YG_CHECK(dev_alloc(ctx, &ctx->d_big_b, chunk_words_max));
        YG_CHECK(dev_alloc(ctx, &ctx->d_big_cstart, (uint64_t)n_big + 1));
        YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_big_list, big_list.data(), (size_t)n_big * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        std::vector<uint64_t> rel((size_t)n_big + 1);
        for (const auto& ch : chunks) {
            const uint32_t c0 = ch.first, c1 = ch.second, nc = c1 - c0;
            const uint64_t words = big_cstart[c1] - big_cstart[c0];
            for (uint32_t j = 0; j <= nc; j++) rel[j] = big_cstart[c0 + j] - big_cstart[c0];
            YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_big_cstart, rel.data(), ((size_t)nc + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
            k2_big_gather<<<(unsigned)std::min<uint32_t>(nc, (uint32_t)ctx->num_sms * 8), 256, 0, st>>>(final_ent, final_begin, final_end, ctx->d_big_list + c0, ctx->d_big_cstart,
                                                                                                     nc, low_bits, ctx->d_big_a);
            YG_CUDA(ctx, cudaGetLastError());
            const int end_bit = std::min(64, low_bits + bitlen((uint64_t)nc - 1));
            size_t tb = 0;
            YG_CUDA(ctx, cub::DeviceRadixSort::SortKeys(nullptr, tb, ctx->d_big_a, ctx->d_big_b, (int64_t)words, 0, std::max(end_bit, 1), st));
            YG_CHECK(ygpu_temp_reserve(ctx, tb));
            tb = ctx->temp_bytes;
            YG_CUDA(ctx, cub::DeviceRadixSort::SortKeys(ctx->d_temp, tb, ctx->d_big_a, ctx->d_big_b, (int64_t)words, 0, std::max(end_bit, 1), st));
            ctx->tm.n_library_launches += 2 + (std::max(end_bit, 1) + 7) / 8;
            k2_big_groups<<<grid_for(ctx, words, 256, 8), 256, 0, st>>>(ctx->d_big_b, words, p.gb, final_words + big_cstart[c0], p.gb <= YG_ITEM_INLINE_BITS ? 1 : 0, ctx->d_post,
                                                                        ctx->d_offsets, ctx->d_row_cnt, ctx->d_row_items, ctx->d_scalars);
            YG_CUDA(ctx, cudaGetLastError());
            ctx->tm.n_kernel_launches += 2;
            YG_CUDA(ctx, cudaStreamSynchronize(st));      // `rel` is reused by the next chunk
        }
        ctx->msd_big_buckets = n_big;
    } else {
        ctx->msd_big_buckets = 0;
    }
    unsigned long long sc[16];
    YG_CUDA(ctx, cudaMemcpyAsync(sc, ctx->d_scalars, sizeof sc, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    // every word is a singleton or a member of a shared group
    const uint64_t P = T_mine - sc[SC_SINGLE];
    const uint64_t I = P - (sc[SC_HEADS] - sc[SC_SINGLE]);
    ctx->tm.ms_sort += elapsed(ctx, 0, 1);
    ctx->tm.ms_index += elapsed(ctx, 1, 2);
    record_phases();
    {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->evp[7], ctx->evp[8]);
        ctx->tm.ms_group += ms;
    }
    ctx->P = P;
    ctx->n_items = I;
    ctx->d_row_begin = ctx->d_offsets;          // work list of row g: row_items[offsets[g] .. + row_cnt[g])
    S->n_hashes = T_mine;
    S->n_distinct = sc[SC_HEADS];
    S->n_singleton = sc[SC_SINGLE];
    S->n_index = S->n_distinct - S->n_singleton;
    S->n_postings = P;
    S->n_increments = sc[SC_W];
    S->n_row_items = I;
    S->has_duplicates = sc[SC_DUPS] ? 1u : 0u;
    *used = 1;
    return 0;
}

#include "run_buckets.cuh"

struct RunPartScratch {
    uint32_t* d_aux = nullptr;      // sample histogram | bases | cursors: 3 x (nb + 2)
    uint64_t aux_cap = 0;
    uint64_t* d_skeys = nullptr;
    uint64_t skeys_cap = 0;
    uint32_t* d_ntbits = nullptr;
    uint64_t nt_cap = 0;
};

}  // namespace

void ygpu_part_release(ygpu_ctx* ctx) {
    if (ctx->part_state) delete (MsdPartState*)ctx->part_state;
    ctx->part_state = nullptr;
    ctx->part_valid = false;
    RunPartScratch* r = (RunPartScratch*)ctx->run_part_scratch;
    if (r) {
        if (r->d_aux) cudaFree(r->d_aux);
        if (r->d_skeys) cudaFree(r->d_skeys);
        if (r->d_ntbits) cudaFree(r->d_ntbits);
        delete r;
    }
    ctx->run_part_scratch = nullptr;
}

// K5 on the partitioned reference (run_buckets.cuh).  d_sample: the sample hashes on the device (any order); d_mask: NULL or
// the caller's nontrivial genomes; d_counts: zeroed by the caller.  *used = 0: this database / sample takes the general path.
int ygpu_run_counts_buckets(ygpu_ctx* ctx, const uint64_t* d_sample, uint64_t n_sample, const uint8_t* d_mask, ygpu_genome_counts* d_counts,
                            int* used) {
    *used = 0;
    if (ctx->run_path == 0 || ctx->sharded || ctx->T < 2 || ctx->n < 2) return 0;
    cudaStream_t st = ctx->stream;
    if (!ctx->part_valid) {
        ygpu_index_stats S{};
        int u = 0;
        YG_CUDA(ctx, cudaMemsetAsync(ctx->d_scalars, 0, 16 * sizeof(unsigned long long), st));
        YG_CHECK(msd_build(ctx, &S, &u, /*partition_only=*/true));
        if (!u || !ctx->part_valid) return 0;
        ctx->indexed = false;           // the partition buffers are shared with the train index build: that index is gone
    }
    const MsdPartState& ps = *(const MsdPartState*)ctx->part_state;
    if (ps.largest > G2_MAXM) return 0;                     // skewed database: general path
    const MsdPlan& p = ps.p;
    const uint32_t nb = ps.nbuckets;
    const int key_bits = ps.sbits + ps.rest_bits;
    if (p.gb + ps.rest_bits > 63) return 0;
    if (!ctx->run_part_scratch) ctx->run_part_scratch = new RunPartScratch();
    RunPartScratch* r = (RunPartScratch*)ctx->run_part_scratch;
    const uint64_t aux = 3ull * ((uint64_t)nb + 2);
    if (aux > r->aux_cap) {
        if (r->d_aux) cudaFree(r->d_aux);
        r->d_aux = nullptr; r->aux_cap = 0;
        YG_CUDA(ctx, cudaMalloc(&r->d_aux, aux * sizeof(uint32_t)));
        r->aux_cap = aux;
    }
    if (n_sample + 1 > r->skeys_cap) {
        if (r->d_skeys) cudaFree(r->d_skeys);
        r->d_skeys = nullptr; r->skeys_cap = 0;
        YG_CUDA(ctx, cudaMalloc(&r->d_skeys, (n_sample + 1) * sizeof(uint64_t)));
        r->skeys_cap = n_sample + 1;
    }
    const uint64_t ntw = ((uint64_t)ctx->n + 31) / 32 + 1;
    if (ntw > r->nt_cap) {
        if (r->d_ntbits) cudaFree(r->d_ntbits);
        r->d_ntbits = nullptr; r->nt_cap = 0;
        YG_CUDA(ctx, cudaMalloc(&r->d_ntbits, ntw * sizeof(uint32_t)));
        r->nt_cap = ntw;
    }
    uint32_t* shist = r->d_aux;
    uint32_t* sbase = shist + ((uint64_t)nb + 2);
    uint32_t* scur = sbase + ((uint64_t)nb + 2);
    const uint64_t key_mask = key_bits >= 64 ? ~0ull : ((1ull << key_bits) - 1ull);
    // ---- the sample, bucketed like the reference ----
    YG_CUDA(ctx, cudaMemsetAsync(r->d_aux, 0, aux * sizeof(uint32_t), st));
    if (n_sample) {
        k5s_hist<<<grid_for(ctx, n_sample, 256), 256, 0, st>>>(d_sample, n_sample, p, shist);
        YG_CUDA(ctx, cudaGetLastError());
    }
    uint32_t* d_smax = (uint32_t*)&ctx->d_scalars[SCM_ICUR];
    size_t tb = 0, tb2 = 0;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb, shist, sbase, (int64_t)nb + 1, st));
    YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb2, shist, d_smax, (int64_t)nb, st));
    YG_CHECK(ygpu_temp_reserve(ctx, std::max(tb, tb2)));
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, shist, sbase, (int64_t)nb + 1, st));
    tb = ctx->temp_bytes;
    YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, shist, d_smax, (int64_t)nb, st));
    ctx->tm.n_library_launches += 4;
    uint32_t smax = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(&smax, d_smax, sizeof smax, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    if (smax > RB_SCAP) return 0;                           // a bucket's sample does not fit shared memory: general path
    YG_CUDA(ctx, cudaMemcpyAsync(scur, sbase, ((uint64_t)nb + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    if (n_sample) {
        k5s_scatter<<<grid_for(ctx, n_sample, 256), 256, 0, st>>>(d_sample, n_sample, p, key_mask, scur, r->d_skeys);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches += 2;
    }
    RunBucketArgs a{};
    a.ent = ps.final_ent; a.begin = ps.final_begin; a.end = ps.final_end; a.nb = nb; a.gb = p.gb;
    a.sub_shift = p.gb + ps.rest_bits; a.sub_mask = (1u << ps.sbits) - 1u; a.rest_bits = ps.rest_bits;
    a.key_mask = key_mask; a.skeys = r->d_skeys; a.sbase = sbase; a.ntbits = r->d_ntbits; a.counts = d_counts;
    const size_t smem = sizeof(RunSmem);
    YG_CUDA(ctx, cudaFuncSetAttribute(k5_bucket<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    YG_CUDA(ctx, cudaFuncSetAttribute(k5_bucket<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k5_bucket<1>, G2_THREADS, smem));
    const int grid = (int)std::min<uint64_t>(nb, (uint64_t)ctx->num_sms * std::max(occ, 1));
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[0], st));
    if (n_sample) {
        k5_bucket<0><<<grid, G2_THREADS, smem, st>>>(a);
        YG_CUDA(ctx, cudaGetLastError());
        ctx->tm.n_kernel_launches++;
    }
    k5_nontrivial_bits<<<grid_for(ctx, ntw, 256), 256, 0, st>>>(d_counts, d_mask, ctx->n, r->d_ntbits);
    YG_CUDA(ctx, cudaGetLastError());
    k5_bucket<1><<<grid, G2_THREADS, smem, st>>>(a);
    YG_CUDA(ctx, cudaGetLastError());
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[1], st));
    ctx->tm.n_kernel_launches += 2;
    ctx->last_run_path = 1;
    *used = 1;
    return 0;
}

int ygpu_build_index_msd(ygpu_ctx* ctx, ygpu_index_stats* S, int* used) {
    const uint64_t T = ctx->T;
    const int rc = msd_build(ctx, S, used);
    S->n_hashes = T;
    return rc;
}


// ============================================================================================================
// Sharded train step: one rank per GPU, every rank resident with the sketches of ITS genome range only.
//
//   reference: compute_index_from_sketches() builds ONE hash map on one thread and the row chunks of
//   compute_intersection_matrix() share it read-only (src/cpp/main.cpp:215-246, 338-349).  Here
//     1. every rank histograms and partitions (level 1) only its own sketches; the packed words go STRAIGHT into the
//        level-1 buffer of the rank that owns their hash range -- stores over NVLink from inside k2_scatter<1, PEER>,
//        at positions every rank derives from the all-gathered histograms (k2s_prep): no all-to-all collective, no
//        send buffer, no replicated read of the sketches;
//     2. every rank runs level 2 and the grouping on its 1/N of the hash space; k2_group2<STREAM> stores each bucket's
//        groups into ALL ranks' stream buffers while the next bucket is grouped (again plain stores, NVLink for peers);
//     3. every rank turns the complete stream into the work lists of its own query rows (k2_items_regions) and counts /
//        flags those rows (K3+K4); the per-rank pair lists are all-gathered (NCCL) and ordered.
//   NCCL carries only the control data (histograms, stream lengths, statistics, pair lists) and separates the phases.
//   The host does not wait for the device between the first kernel and the statistics read-back.
// ============================================================================================================
#include "comm.cuh"

int ygpu_sort_pairs_device(ygpu_ctx* ctx, ygpu_pair* d_pairs, uint64_t n);      // yacht_gpu.cu

// everything after the slice's hashes are in d_hashes: global offsets, sizes, slice-relative offsets, the global largest hash
int ygpu_sharded_finish(ygpu_ctx* ctx, const uint64_t* offsets, uint32_t n, uint32_t g_begin, uint32_t g_end) {
    if (!ctx->comm) return ygpu_fail(ctx, YGPU_ERR_STATE, "sharded load: ygpu_comm_init first");
    cudaStream_t st = ctx->stream;
    ctx->loaded = false; ctx->indexed = false; ctx->sorted = false; ctx->maxkey_valid = false; ctx->row_work_valid = false;
    ctx->P = 0; ctx->n_items = 0;
    const uint64_t Tg = offsets[n];
    if (offsets[0] != 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets[0] must be 0");
    uint32_t mx = 0;
    for (uint32_t g = 0; g < n; g++) {
        if (offsets[g + 1] < offsets[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets not monotone at genome %u", g);
        mx = std::max<uint32_t>(mx, (uint32_t)std::min<uint64_t>(offsets[g + 1] - offsets[g], 0xFFFFFFFFull));
    }
    if (Tg >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes %llu >= 2^32 not supported", (unsigned long long)Tg);
    const uint64_t T = offsets[g_end] - offsets[g_begin];
    ctx->n = n; ctx->T = T; ctx->T_global = Tg; ctx->g_begin = g_begin; ctx->g_end = g_end; ctx->sharded = true;
    ctx->shard_mode = 0;
    ctx->max_sketch_global = mx;
    ctx->row_items_need = IG_ROW_MUL * T + 8ull * (g_end - g_begin) + 16;
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sizes, n));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_begin_local, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets_local, (uint64_t)(g_end - g_begin) + 1));
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_offsets, offsets, ((uint64_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    k2s_sizes<<<grid_for(ctx, (uint64_t)n + 1, 256, 8), 256, 0, st>>>(ctx->d_offsets, n, g_begin, g_end, ctx->d_sizes, ctx->d_row_begin_local, ctx->d_offsets_local);
    YG_CUDA(ctx, cudaGetLastError());
    ctx->tm.n_kernel_launches++;
    // the largest hash over ALL ranks decides the partition plan
    uint64_t* d_max = (uint64_t*)&ctx->d_scalars[SC_MAXKEY];
    YG_CUDA(ctx, cudaMemsetAsync(d_max, 0, sizeof(uint64_t), st));
    if (T) {
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb, ctx->d_hashes, d_max, (int64_t)T, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, ctx->d_hashes, d_max, (int64_t)T, st));
        ctx->tm.n_library_launches += 2;
    }
    YG_CHECK(ygpu_comm_allreduce_u64(ctx, d_max, d_max, 1, true));
    YG_CUDA(ctx, cudaMemcpyAsync(&ctx->maxkey, d_max, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    // every rank's genome range (the query rows it counts): contiguous, in rank order, covering [0, n)
    const int N = ctx->comm->nranks;
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_info, (uint64_t)SHI_WORDS));
    unsigned long long gb0 = g_begin, all[YG_MAX_RANKS];
    YG_CUDA(ctx, cudaMemcpyAsync(&ctx->d_sh_info[SHI_ICUR], &gb0, sizeof gb0, cudaMemcpyHostToDevice, st));
    YG_CHECK(ygpu_comm_allgather(ctx, &ctx->d_sh_info[SHI_ICUR], &ctx->d_sh_info[SHI_ILENS], sizeof(unsigned long long)));
    YG_CUDA(ctx, cudaMemcpyAsync(all, &ctx->d_sh_info[SHI_ILENS], (size_t)N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    for (int q = 0; q < N; q++) ctx->sh_row_bounds[q] = (uint32_t)all[q];
    ctx->sh_row_bounds[N] = n;
    if (ctx->sh_row_bounds[0] != 0 || ctx->sh_row_bounds[ctx->comm->rank + 1] != g_end)
        return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches_sharded: the ranks' genome ranges must be contiguous, in rank order, and cover [0, n)");
    for (int q = 0; q < N; q++)
        if (ctx->sh_row_bounds[q] > ctx->sh_row_bounds[q + 1]) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches_sharded: genome ranges out of order at rank %d", q);
    ctx->maxkey_valid = true;
    ctx->loaded = true;
    return 0;
}

static int sharded_load(ygpu_ctx* ctx, const uint64_t* hashes_slice, const uint64_t* offsets, uint32_t n, uint32_t g_begin, uint32_t g_end,
                        bool from_device) {
    if (!ctx || !offsets) return YGPU_ERR_ARG;
    if (!ctx->comm) return ygpu_fail(ctx, YGPU_ERR_STATE, "load_sketches_sharded: ygpu_comm_init first");
    if (g_begin > g_end || g_end > n) return ygpu_fail(ctx, YGPU_ERR_ARG, "bad genome range [%u,%u) of %u", g_begin, g_end, n);
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint64_t T = offsets[g_end] - offsets[g_begin];
    if (T && !hashes_slice) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches_sharded: NULL hashes");
    if (T >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes >= 2^32 not supported");
    ctx->loaded = false;
    YG_CHECK(dev_alloc(ctx, &ctx->d_hashes, T + 2));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    if (T) YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_hashes, hashes_slice, T * sizeof(uint64_t), from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));
    YG_CHECK(ygpu_sharded_finish(ctx, offsets, n, g_begin, g_end));
    ctx->tm.ms_h2d += elapsed(ctx, 0, 1);
    return 0;
}

extern "C" int ygpu_load_sketches_sharded(ygpu_ctx* ctx, const uint64_t* hashes_slice, const uint64_t* offsets, uint32_t n_genomes,
                                          uint32_t g_begin, uint32_t g_end) {
    return sharded_load(ctx, hashes_slice, offsets, n_genomes, g_begin, g_end, false);
}
extern "C" int ygpu_load_sketches_sharded_device(ygpu_ctx* ctx, const uint64_t* d_hashes_slice, const uint64_t* offsets, uint32_t n_genomes,
                                                 uint32_t g_begin, uint32_t g_end) {
    return sharded_load(ctx, d_hashes_slice, offsets, n_genomes, g_begin, g_end, true);
}

// The per-rank pair lists (unsorted, in ctx->d_pairs) of all ranks on every rank, ordered by (i, j): all-gather of the counts
// (the same gather carries a per-rank refusal flag so that every rank stops or goes on together), padded all-gather of the
// lists, one sort on packed keys.  Leaves the complete list in ctx->d_pairs.
static int gather_pairs(ygpu_ctx* ctx, uint64_t n_r, unsigned long long my_ovf, uint64_t* n_total) {
    cudaStream_t st = ctx->stream;
    const int N = ctx->comm->nranks, rank = ctx->comm->rank;
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    unsigned long long mine[2] = {n_r, my_ovf}, both[2 * YG_MAX_RANKS], counts[YG_MAX_RANKS];
    unsigned long long* d_cnt = &ctx->d_sh_info[44];
    YG_CUDA(ctx, cudaMemcpyAsync(d_cnt, mine, sizeof mine, cudaMemcpyHostToDevice, st));
    YG_CHECK(ygpu_comm_allgather(ctx, d_cnt, d_cnt + 2, 2 * sizeof(unsigned long long)));
    YG_CUDA(ctx, cudaMemcpyAsync(both, d_cnt + 2, (size_t)N * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    uint64_t total = 0, mxc = 0;
    for (int q = 0; q < N; q++) {
        counts[q] = both[2 * q];
        if (both[2 * q + 1]) {
            ctx->indexed = false;
            return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: a query row of rank %d received more work items than its list holds (sketches with repeated hashes): run this database on one GPU", q);
        }
        total += counts[q]; mxc = std::max<uint64_t>(mxc, counts[q]);
    }
    if (total) {
        // padded all-gather, then the ranks' lists are squeezed together and ordered
        const uint64_t need_all = (uint64_t)N * mxc + total + 16;
        if (need_all > ctx->pairs_local_cap) {
            if (ctx->d_pairs_local) cudaFree(ctx->d_pairs_local);
            ctx->d_pairs_local = nullptr; ctx->pairs_local_cap = 0;
            YG_CUDA(ctx, cudaMalloc(&ctx->d_pairs_local, (need_all + need_all / 8 + 1024) * sizeof(ygpu_pair)));
            ctx->pairs_local_cap = need_all + need_all / 8 + 1024;
        }
        ygpu_pair* pad = ctx->d_pairs_local;                 // [N][mxc] gathered, then [total] compact behind it
        ygpu_pair* out = pad + (uint64_t)N * mxc;
        if (n_r) YG_CUDA(ctx, cudaMemcpyAsync(pad + (uint64_t)rank * mxc, ctx->d_pairs, n_r * sizeof(ygpu_pair), cudaMemcpyDeviceToDevice, st));
        YG_CHECK(ygpu_comm_allgather(ctx, pad + (uint64_t)rank * mxc, pad, (size_t)mxc * sizeof(ygpu_pair)));
        uint64_t pos = 0;
        for (int q = 0; q < N; q++) {
            if (counts[q]) YG_CUDA(ctx, cudaMemcpyAsync(out + pos, pad + (uint64_t)q * mxc, counts[q] * sizeof(ygpu_pair), cudaMemcpyDeviceToDevice, st));
            pos += counts[q];
        }
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[12], st));
        YG_CHECK(ygpu_sort_pairs_device(ctx, out, total));
        if (total > ctx->pairs_cap) {
            if (ctx->d_pairs) cudaFree(ctx->d_pairs);
            ctx->d_pairs = nullptr; ctx->pairs_cap = 0;
            YG_CUDA(ctx, cudaMalloc(&ctx->d_pairs, (total + 1024) * sizeof(ygpu_pair)));
            ctx->pairs_cap = total + 1024;
        }
        YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_pairs, out, total * sizeof(ygpu_pair), cudaMemcpyDeviceToDevice, st));
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->tm.ms_pairsort += elapsed(ctx, 2, 3);
    if (total) { float g = 0.f; cudaEventElapsedTime(&g, ctx->ev[2], ctx->evp[12]); ctx->tm.ms_gather += g; }
    ctx->n_pairs = total;
    *n_total = total;
    return 0;
}

// ---- hash-range residency: this rank holds, of EVERY sketch, the hashes that fall into its hash range ------------------------
// (a sketch is sorted, so that share is one contiguous piece of it: the host cuts every sketch at the same N - 1 hash values).
// Equal hashes then meet on one rank by construction: the index build needs no exchange at all before the grouping, and the
// only data that ever crosses NVLink are the work items the grouping kernel sends to the owners of the query rows.
static int hashrange_load(ygpu_ctx* ctx, const uint64_t* part_hashes, const uint64_t* part_offsets, const uint32_t* sizes, uint32_t n,
                          uint32_t row_begin, uint32_t row_end, bool from_device) {
    if (!ctx || !part_offsets || (n && !sizes)) return YGPU_ERR_ARG;
    if (!ctx->comm) return ygpu_fail(ctx, YGPU_ERR_STATE, "load_sketches_hashrange: ygpu_comm_init first");
    if (row_begin > row_end || row_end > n) return ygpu_fail(ctx, YGPU_ERR_ARG, "bad row range [%u,%u) of %u", row_begin, row_end, n);
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ctx->loaded = false; ctx->indexed = false; ctx->sorted = false; ctx->maxkey_valid = false; ctx->row_work_valid = false;
    ctx->part_valid = false; ctx->P = 0; ctx->n_items = 0;
    if (part_offsets[0] != 0) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets[0] must be 0");
    uint64_t Tg = 0;
    uint32_t mx = 0;
    for (uint32_t g = 0; g < n; g++) {
        if (part_offsets[g + 1] < part_offsets[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "offsets not monotone at genome %u", g);
        if (part_offsets[g + 1] - part_offsets[g] > sizes[g]) return ygpu_fail(ctx, YGPU_ERR_ARG, "genome %u: the resident share exceeds the sketch size", g);
        Tg += sizes[g];
        mx = std::max(mx, sizes[g]);
    }
    const uint64_t T = part_offsets[n];
    if (Tg >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "total hashes %llu >= 2^32 not supported", (unsigned long long)Tg);
    if (T && !part_hashes) return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches_hashrange: NULL hashes");
    // work-list starts of this rank's query rows: room for IG_ROW_MUL * |S_g| + 8 items per row (k2s_sizes has the same rule)
    std::vector<uint64_t> rb((size_t)n + 1, 0);
    uint64_t acc = 0;
    for (uint32_t g = row_begin; g < row_end; g++) { rb[g] = acc; acc += IG_ROW_MUL * sizes[g] + 8ull; }
    ctx->n = n; ctx->T = T; ctx->T_global = Tg; ctx->g_begin = row_begin; ctx->g_end = row_end; ctx->sharded = true;
    ctx->shard_mode = 1;
    ctx->max_sketch_global = mx;
    ctx->row_items_need = acc + 16;
    YG_CHECK(dev_alloc(ctx, &ctx->d_hashes, T + 2));
    YG_CHECK(dev_alloc(ctx, &ctx->d_offsets, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sizes, n));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_begin_local, (uint64_t)n + 1));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    if (T) YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_hashes, part_hashes, T * sizeof(uint64_t), from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_offsets, part_offsets, ((uint64_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    if (n) YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_sizes, sizes, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaMemcpyAsync(ctx->d_row_begin_local, rb.data(), ((size_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));
    // over ALL ranks: the largest hash (decides the partition plan), the largest share (sizes the exchange buffers), the row ranges
    const int N = ctx->comm->nranks;
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_info, (uint64_t)SHI_WORDS));
    unsigned long long* d_mx = &ctx->d_sh_info[SHI_ICUR];            // {largest hash, largest share}
    YG_CUDA(ctx, cudaMemsetAsync(d_mx, 0, 2 * sizeof(unsigned long long), st));
    if (T) {
        size_t tb = 0;
        YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb, ctx->d_hashes, (uint64_t*)d_mx, (int64_t)T, st));
        YG_CHECK(ygpu_temp_reserve(ctx, tb));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, ctx->d_hashes, (uint64_t*)d_mx, (int64_t)T, st));
        ctx->tm.n_library_launches += 2;
    }
    unsigned long long share = T, back[2], rb0 = row_begin, all[YG_MAX_RANKS];
    YG_CUDA(ctx, cudaMemcpyAsync(d_mx + 1, &share, sizeof share, cudaMemcpyHostToDevice, st));
    YG_CHECK(ygpu_comm_allreduce_u64(ctx, d_mx, d_mx, 2, true));
    YG_CUDA(ctx, cudaMemcpyAsync(back, d_mx, sizeof back, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(d_mx + 2, &rb0, sizeof rb0, cudaMemcpyHostToDevice, st));
    YG_CHECK(ygpu_comm_allgather(ctx, d_mx + 2, &ctx->d_sh_info[SHI_ILENS], sizeof(unsigned long long)));
    YG_CUDA(ctx, cudaMemcpyAsync(all, &ctx->d_sh_info[SHI_ILENS], (size_t)N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->maxkey = back[0];
    ctx->sh_cap_req = back[1];
    for (int q = 0; q < N; q++) ctx->sh_row_bounds[q] = (uint32_t)all[q];
    ctx->sh_row_bounds[N] = n;
    if (ctx->sh_row_bounds[0] != 0 || ctx->sh_row_bounds[ctx->comm->rank + 1] != row_end)
        return ygpu_fail(ctx, YGPU_ERR_ARG, "load_sketches_hashrange: the ranks' row ranges must be contiguous, in rank order, and cover [0, n)");
    ctx->maxkey_valid = true;
    ctx->loaded = true;
    ctx->tm.ms_h2d += elapsed(ctx, 0, 1);
    return 0;
}

extern "C" int ygpu_load_sketches_hashrange(ygpu_ctx* ctx, const uint64_t* part_hashes, const uint64_t* part_offsets, const uint32_t* sizes,
                                            uint32_t n_genomes, uint32_t row_begin, uint32_t row_end) {
    return hashrange_load(ctx, part_hashes, part_offsets, sizes, n_genomes, row_begin, row_end, false);
}
extern "C" int ygpu_load_sketches_hashrange_device(ygpu_ctx* ctx, const uint64_t* d_part_hashes, const uint64_t* part_offsets, const uint32_t* sizes,
                                                   uint32_t n_genomes, uint32_t row_begin, uint32_t row_end) {
    return hashrange_load(ctx, d_part_hashes, part_offsets, sizes, n_genomes, row_begin, row_end, true);
}

extern "C" int ygpu_train_step_sharded(ygpu_ctx* ctx, double threshold, ygpu_index_stats* stats, uint64_t* n_pairs_total) {
    if (!ctx || !n_pairs_total) return YGPU_ERR_ARG;
    *n_pairs_total = 0;
    if (!ctx->comm || !ctx->sharded || !ctx->loaded) return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: ygpu_comm_init and ygpu_load_sketches_sharded first");
    YG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ygpu_comm* C = ctx->comm;
    const int N = C->nranks, rank = C->rank;
    const uint64_t T = ctx->T, Tg = ctx->T_global;
    const uint32_t n = ctx->n;
    ctx->indexed = false; ctx->row_work_valid = false; ctx->n_pairs = 0; ctx->part_valid = false;
    ygpu_index_stats S{};
    S.n_hashes = Tg;
    S.max_sketch = ctx->max_sketch_global;
    S.index_path = 1;
    if (Tg < 2 || n < 2) {
        ctx->stats = S; ctx->indexed = true; ctx->n_items = 0;
        if (stats) *stats = S;
        return 0;
    }
    // ---- plan (same rules as msd_build, bucket sizes by the GLOBAL hash count) --------------------------------------
    const uint64_t maxkey = ctx->maxkey;
    MsdPlan p{};
    p.T = T;
    p.hb = std::max(1, bitlen(maxkey));
    p.gb = bitlen((uint64_t)n - 1);
    auto used_buckets = [&](int D) -> uint64_t { return D == 0 ? 1ull : (maxkey >> (p.hb - D)) + 1ull; };
    int D = 0;
    while (D < p.hb && D < 22 && Tg / used_buckets(D) > A_TARGET) D++;
    // level 1 is the exchange: its runs per (tile, digit) are what crosses NVLink, so it gets as FEW digits as the two levels
    // allow (level 2 takes up to 11 bits) -- 16-word runs are 128-byte packets, 4-word runs are 32-byte ones
    const bool hr = ctx->shard_mode == 1;     // hash-range residency: nothing is exchanged before the grouping
    int d1 = D <= 8 ? D : (hr ? (D + 1) / 2 : std::max(D - 11, std::min(8, D / 2)));
    const int need = p.hb + p.gb - 64;
    if (need > d1) d1 = need;
    int d2 = std::max(0, D - d1);
    const char* why = nullptr;
    if (d1 > 11 || d1 > p.hb || d2 > 11) why = "hash and genome-id width do not pack into 64-bit words";
    p.d1 = d1; p.d2 = d2; p.kb1 = p.hb - d1;
    p.nb1 = d1 ? (uint32_t)(maxkey >> (p.hb - d1)) + 1 : 1u;
    if (!why && p.nb1 > NB_MAX) why = "too many level-1 buckets";
    p.nfb = p.nb1 << d2;
    p.dlo = 0; p.dhi = p.nb1; p.unit_lo = 0; p.unit_hi = 0xFFFFFFFFu;
    const int key_bits = p.kb1 - d2;
    const int sbits = std::max(0, std::min(GK_SUBBITS, key_bits));
    const int rest_bits = key_bits - sbits;
    if (!why && rest_bits > 32) why = "remaining hash bits exceed 32 (database too small for its hash width)";
    if (why) return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: this database does not qualify for the sharded partition path: %s", why);

    // ---- buffers; the exchange targets are (re)shared with the peers when they move ------------------------------------
    // words a rank can own: its share + digit granularity (genome-range residency), the largest share (hash-range residency)
    const uint64_t cap = hr ? ctx->sh_cap_req + 3 * SC_TILE : Tg / N + 2 * (Tg / std::max<uint32_t>(p.nb1, 1)) + 3 * SC_TILE;
    if ((uint64_t)N * cap + 8 >= (1ull << 32)) return ygpu_fail(ctx, YGPU_ERR_ARG, "stream of %llu entries >= 2^32 not supported", (unsigned long long)N * cap);
    ctx->sh_cap = cap;
    YG_CHECK(dev_alloc(ctx, &ctx->d_ent1, cap + 2));
    if (d2) YG_CHECK(dev_alloc(ctx, &ctx->d_ent2, cap + 2));
    YG_CHECK(dev_alloc(ctx, &ctx->d_post, (uint64_t)N * cap + 8));
    YG_CHECK(dev_alloc(ctx, &ctx->d_st_rem, (uint64_t)N * cap + 8));
    ctx->row_items_cap = ctx->row_items_need;
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_items, ctx->row_items_cap));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_cnt, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_row_ptr, (uint64_t)n + 1));
    YG_CHECK(dev_alloc(ctx, &ctx->d_inbox_item, (uint64_t)N * cap + 8));
    YG_CHECK(dev_alloc(ctx, &ctx->d_inbox_row, (uint64_t)N * cap + 8));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_hist_all, (uint64_t)(N + 1) * NB_MAX));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_owner, (uint64_t)NB_MAX));
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_info, (uint64_t)SHI_WORDS));
    const uint64_t aux_words = MsdAux::words(p.nfb);
    YG_CHECK(dev_alloc(ctx, &ctx->d_msd_aux, aux_words));
    const uint32_t units1 = (uint32_t)((T + SC_TILE - 1) / SC_TILE);
    YG_CHECK(dev_alloc(ctx, &ctx->d_tile_g0, (uint64_t)units1 + 2));
    const uint64_t max_units = cap / SC_TILE + p.nb1 + 2;
    YG_CHECK(dev_alloc(ctx, &ctx->d_units, 2 * max_units));
    {
        // collective: every rank evaluates the same conditions in the same order (allocations move together or a rank re-shares alone
        // harmlessly -- the exchange is an all-gather every rank takes part in, so the decision must be global)
        unsigned long long moved = (ctx->sh_shared_ent1 != ctx->d_ent1) || (ctx->sh_shared_gid != ctx->d_post) || (ctx->sh_shared_rem != ctx->d_st_rem) ||
                                   (ctx->sh_shared_item != ctx->d_inbox_item) || (ctx->sh_shared_row != ctx->d_inbox_row);
        unsigned long long* d_flag = &ctx->d_sh_info[40];
        YG_CUDA(ctx, cudaMemcpyAsync(d_flag, &moved, sizeof moved, cudaMemcpyHostToDevice, st));
        YG_CHECK(ygpu_comm_allreduce_u64(ctx, d_flag, d_flag, 1, true));
        YG_CUDA(ctx, cudaMemcpyAsync(&moved, d_flag, sizeof moved, cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        if (moved) {
            YG_CHECK(ygpu_comm_share(ctx, ctx->d_ent1, ctx->sh_peer_ent1));
            YG_CHECK(ygpu_comm_share(ctx, ctx->d_post, ctx->sh_peer_gid));
            YG_CHECK(ygpu_comm_share(ctx, ctx->d_st_rem, ctx->sh_peer_rem));
            YG_CHECK(ygpu_comm_share(ctx, ctx->d_inbox_item, ctx->sh_peer_item));
            YG_CHECK(ygpu_comm_share(ctx, ctx->d_inbox_row, ctx->sh_peer_row));
            ctx->sh_shared_ent1 = ctx->d_ent1; ctx->sh_shared_gid = ctx->d_post; ctx->sh_shared_rem = ctx->d_st_rem;
            ctx->sh_shared_item = ctx->d_inbox_item; ctx->sh_shared_row = ctx->d_inbox_row;
        }
    }
    // exact layout (every rank's histograms are exchanged anyway): bucket b spans [begin[b], begin[b + 1]); the histograms are the caps
    const MsdAux x(ctx->d_msd_aux, p.nfb);
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[0], st));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_msd_aux, 0, aux_words * sizeof(uint32_t), st));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_scalars, 0, REP_WORDS * sizeof(unsigned long long), st));
    YG_CUDA(ctx, cudaMemsetAsync(ctx->d_row_cnt, 0, ((uint64_t)n + 1) * sizeof(unsigned long long), st));

    // ---- 1. level 1.  Genome-range residency: on the resident slice, every word stored into its owner's buffer (NVLink).
    //         Hash-range residency: purely local -- this rank already holds exactly the hashes of its range. ---------------------
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[0], st));
    if (T) {
        k2_hist1<<<ctx->num_sms * 8, 256, p.nb1 * sizeof(uint32_t), st>>>(ctx->d_hashes, p, x.cap1);
        YG_CUDA(ctx, cudaGetLastError());
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[1], st));
    ScatterArgs a{};
    a.hashes = ctx->d_hashes; a.out_ent = ctx->d_ent1; a.tile_start = x.tile_start; a.hist2 = x.cap2;
    a.cursor = x.cur1; a.ovf = &ctx->d_scalars[SCM_OVF1];
    if (hr) {
        k2_prep1<<<1, 1024, 0, st>>>(x.cap1, nullptr, p.nb1, x.begin1, nullptr, x.cur1, x.tile_start, ctx->d_scalars);
        YG_CUDA(ctx, cudaGetLastError());
        k2s_range<<<1, 1024, 0, st>>>(x.cap1, p.nb1, d2, (unsigned long long)T, ctx->d_sh_info);
        YG_CUDA(ctx, cudaGetLastError());
        a.offsets = ctx->d_offsets; a.n = n; a.gid_base = 0;           // the resident CSR spans all genomes
    } else {
        YG_CHECK(ygpu_comm_allgather(ctx, x.cap1, ctx->d_sh_hist_all, (size_t)NB_MAX * sizeof(uint32_t)));
        k2s_prep<<<1, 1024, 0, st>>>(ctx->d_sh_hist_all, p.nb1, N, rank, d2, ctx->d_sh_owner, x.cur1, x.begin1, x.tile_start, ctx->d_sh_info,
                                     ctx->d_scalars);
        YG_CUDA(ctx, cudaGetLastError());
        // the plan is the same on every rank, so every rank sees whether some rank would own more words than the exchange
        // buffers hold (a hash distribution far from uniform) and all of them stop here, before a single word is stored
        unsigned long long tmax = 0;
        YG_CUDA(ctx, cudaMemcpyAsync(&tmax, &ctx->d_sh_info[SHI_TMAX], sizeof tmax, cudaMemcpyDeviceToHost, st));
        YG_CUDA(ctx, cudaStreamSynchronize(st));
        if (tmax > cap) return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: a rank would own %llu words, the exchange buffers hold %llu", tmax, (unsigned long long)cap);
        a.offsets = ctx->d_offsets_local; a.n = ctx->g_end - ctx->g_begin; a.gid_base = ctx->g_begin;
        a.owner = ctx->d_sh_owner;
        for (int q = 0; q < N; q++) a.peer_ent[q] = (uint64_t*)ctx->sh_peer_ent1[q];
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[2], st));
    if (T) {
        k2_tile_g0<<<grid_for(ctx, (uint64_t)units1 + 1, 256, 8), 256, 0, st>>>(a.offsets, a.n, T, units1, ctx->d_tile_g0);
        YG_CUDA(ctx, cudaGetLastError());
        a.tile_g0 = ctx->d_tile_g0;
        const size_t smem = (size_t)2 * SC_BUF * 8 + (size_t)p.nb1 * (hr ? 16 : 24) + (size_t)SC_TILE * 2;
        auto kern = hr ? k2_scatter<1, false> : k2_scatter<1, true>;
        YG_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 1;
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SC_THREADS, smem));
        const int grid = (int)std::min<uint64_t>(units1, (uint64_t)ctx->num_sms * std::max(occ, 1));
        kern<<<grid, SC_THREADS, smem, st>>>(a, p, 0u, units1);
        YG_CUDA(ctx, cudaGetLastError());
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[3], st));
    if (!hr) {
        // every rank's words have landed once every rank has passed this point (the collective also orders the peer stores)
        unsigned long long* d_sync = &ctx->d_sh_info[41];
        YG_CHECK(ygpu_comm_allreduce_u64(ctx, d_sync, d_sync, 1, true));
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[9], st));
    ctx->tm.n_kernel_launches += 4;

    // ---- 2. level 2 + grouping on this rank's share of the hash space; groups stored into every rank's stream ---------
    const uint64_t* final_ent = ctx->d_ent1;
    const uint32_t* final_begin = x.begin1;
    if (d2) {
        a.in_ent = ctx->d_ent1; a.out_ent = ctx->d_ent2;
        k2_units<<<grid_for(ctx, max_units, 256, 8), 256, 0, st>>>(x.tile_start, x.begin1, x.begin1 + 1, p.nb1, (uint2*)ctx->d_units);
        YG_CUDA(ctx, cudaGetLastError());
        a.units = (const uint2*)ctx->d_units;
        k2_hist2<<<ctx->num_sms * 8, 256, (size_t)(1u << d2) * sizeof(uint32_t), st>>>(a, p, 0xFFFFFFFFu);
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[4], st));
        size_t tb = 0, tb2 = 0;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tb, x.cap2, x.begin2, (int64_t)p.nfb + 1, st));
        YG_CUDA(ctx, cub::DeviceReduce::Max(nullptr, tb2, x.cap2, (uint32_t*)&ctx->d_scalars[SCM_MAXB + 1], (int64_t)p.nfb, st));
        YG_CHECK(ygpu_temp_reserve(ctx, std::max(tb, tb2)));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceScan::ExclusiveSum(ctx->d_temp, tb, x.cap2, x.begin2, (int64_t)p.nfb + 1, st));
        tb = ctx->temp_bytes;
        YG_CUDA(ctx, cub::DeviceReduce::Max(ctx->d_temp, tb, x.cap2, (uint32_t*)&ctx->d_scalars[SCM_MAXB + 1], (int64_t)p.nfb, st));
        ctx->tm.n_library_launches += 4;
        YG_CUDA(ctx, cudaMemcpyAsync(x.cur2, x.begin2, (uint64_t)p.nfb * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        a.cursor = x.cur2; a.ovf = &ctx->d_scalars[SCM_OVF2];
        const size_t smem = (size_t)2 * SC_BUF * 8 + (size_t)(1u << d2) * 16 + (size_t)SC_TILE * 2;
        YG_CUDA(ctx, cudaFuncSetAttribute(k2_scatter<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 1;
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k2_scatter<2, false>, SC_THREADS, smem));
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[5], st));
        k2_scatter<2, false><<<ctx->num_sms * std::max(occ, 1), SC_THREADS, smem, st>>>(a, p, 0u, 0xFFFFFFFFu);
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[6], st));
        ctx->tm.n_kernel_launches += 3;
        final_ent = ctx->d_ent2;
        final_begin = x.begin2;
    }
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[1], st));
    {
        GroupArgs g{};
        g.ent = final_ent; g.begin = final_begin; g.end = final_begin + 1; g.gb = p.gb;
        g.nb = d2 ? p.nfb : p.nb1;
        g.b_lo = 0; g.b_hi = g.nb; g.m_lo = 0;
        g.range = d2 ? &ctx->d_sh_info[SHI_BLO] : &ctx->d_sh_info[SHI_DLO];
        g.sub_shift = p.gb + rest_bits;
        g.sub_mask = (1u << sbits) - 1u;
        g.rest_mask = rest_bits >= 64 ? ~0ull : ((1ull << rest_bits) - 1ull);
        if (g.sub_shift > 63) { g.sub_shift = 0; g.sub_mask = 0; }
        g.scal = ctx->d_scalars;
        g.n_peers = N;
        g.region_base = (uint64_t)rank * cap;
        for (int q = 0; q < N; q++) {
            g.peer_gid[q] = (uint32_t*)ctx->sh_peer_gid[q]; g.peer_rem[q] = (unsigned short*)ctx->sh_peer_rem[q];
            g.peer_item[q] = (uint64_t*)ctx->sh_peer_item[q]; g.peer_row[q] = (uint32_t*)ctx->sh_peer_row[q];
        }
        for (int q = 0; q <= N; q++) g.row_bounds[q] = ctx->sh_row_bounds[q];
        g.icap = cap; g.item_region = (uint64_t)rank * cap; g.icursor = &ctx->d_scalars[REP_ICUR];
        const size_t smem2 = sizeof(G2Smem);
        YG_CUDA(ctx, cudaFuncSetAttribute(k2_group2<true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
        int occ2 = 1;
        YG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, k2_group2<true, 4>, G2_THREADS, smem2));
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[7], st));
        k2_group2<true, 4><<<ctx->num_sms * std::max(occ2, 1), G2_THREADS, smem2, st>>>(g);
        YG_CUDA(ctx, cudaGetLastError());
        YG_CUDA(ctx, cudaEventRecord(ctx->evp[8], st));
        ctx->tm.n_kernel_launches += 1;
    }
    // ONE all-gather of every rank's report (statistics, largest bucket, posting-stream length, items sent to every rank): it is
    // also the barrier behind the item / stream stores of the grouping kernels
    unsigned long long* d_rep = &ctx->d_sh_info[SHI_ILENS];         // [N][REP_WORDS]
    YG_CHECK(ygpu_comm_allgather(ctx, ctx->d_scalars, d_rep, (size_t)REP_WORDS * sizeof(unsigned long long)));
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[10], st));

    // ---- 3. work lists of this rank's rows: the items the ranks sent (+ those derived from the posting stream of the larger
    //         groups) are appended to the rows' lists -------------------------------------------------------------------------------
    const int can_inl = p.gb <= YG_ITEM_INLINE_BITS ? 1 : 0;
    const dim3 grid_in((unsigned)std::max(1, grid_for(ctx, std::max<uint64_t>(Tg / (4ull * N * N), 1), 256, 16) / 1), (unsigned)N);
    unsigned long long* d_ovf = &ctx->d_sh_info[42];
    YG_CUDA(ctx, cudaMemsetAsync(d_ovf, 0, sizeof(unsigned long long), st));
    k2_inbox<<<grid_in, 256, 0, st>>>(ctx->d_inbox_item, ctx->d_inbox_row, d_rep, N, rank, cap, ctx->d_row_begin_local, ctx->d_sizes, ctx->d_row_cnt,
                                      ctx->d_row_items, d_ovf);
    YG_CUDA(ctx, cudaGetLastError());
    k2_items_regions<<<grid_in, 256, 0, st>>>(ctx->d_post, ctx->d_st_rem, d_rep, N, cap, ctx->g_begin, ctx->g_end, can_inl, ctx->d_row_begin_local,
                                              ctx->d_sizes, ctx->d_row_cnt, ctx->d_row_items, d_ovf);
    YG_CUDA(ctx, cudaGetLastError());
    YG_CUDA(ctx, cudaEventRecord(ctx->evp[11], st));
    ctx->tm.n_kernel_launches += 2;
    unsigned long long tot[6] = {0, 0, 0, 0, 0, 0}, rep[YG_MAX_RANKS * REP_WORDS], my_ovf = 0;
    YG_CUDA(ctx, cudaMemcpyAsync(rep, d_rep, (size_t)N * REP_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaMemcpyAsync(&my_ovf, d_ovf, sizeof my_ovf, cudaMemcpyDeviceToHost, st));
    YG_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    YG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->tm.ms_sort += elapsed(ctx, 0, 1);
    ctx->tm.ms_index += elapsed(ctx, 1, 2);
    {
        auto el = [&](int x, int y) { float ms = 0.f; cudaEventElapsedTime(&ms, ctx->evp[x], ctx->evp[y]); return (double)ms; };
        ctx->tm.ms_hist1 += el(0, 1);
        ctx->tm.ms_scatter1 += el(2, 3);
        if (d2) { ctx->tm.ms_hist2 += el(3, 4); ctx->tm.ms_scatter2 += el(5, 6); }
        ctx->tm.ms_group += el(7, 8);
        ctx->tm.ms_items += el(10, 11);
        ctx->tm.ms_sync += el(3, 9) + el(8, 10);       // waiting for the peers behind the two exchanges (+ the collectives themselves)
    }
    // every rank holds every report: sums / maxima and all refusals below are unanimous
    for (int q = 0; q < N; q++) {
        const unsigned long long* r = rep + (size_t)q * REP_WORDS;
        tot[SC_HEADS] += r[SC_HEADS]; tot[SC_SINGLE] += r[SC_SINGLE]; tot[SC_DUPS] += r[SC_DUPS]; tot[SC_W] += r[SC_W];
        tot[4] = std::max(tot[4], r[SCM_MAXB]); tot[5] = std::max<unsigned long long>(tot[5], (uint32_t)r[SCM_MAXB + 1]);
        for (int d = 0; d < N; d++)
            if (r[REP_ICUR + d] > cap)
                return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: rank %d sent %llu work items to rank %d, the inbox region holds %llu", q, r[REP_ICUR + d], d, (unsigned long long)cap);
        if (r[SCM_STREAM] > cap) return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: the posting stream of rank %d overflows", q);
    }
    const uint64_t largest = d2 ? (uint64_t)(uint32_t)tot[5] : tot[4];
    if (largest > G2_MAXM)
        return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_sharded: a final bucket holds %llu words (> %u): skewed databases take the replicated build (ygpu_build_index)",
                         (unsigned long long)largest, G2_MAXM);
    S.n_distinct = tot[SC_HEADS];
    S.n_singleton = tot[SC_SINGLE];
    S.n_index = S.n_distinct - S.n_singleton;
    S.n_postings = Tg - tot[SC_SINGLE];
    S.n_increments = tot[SC_W];
    S.n_row_items = S.n_postings - S.n_index;
    S.has_duplicates = tot[SC_DUPS] ? 1u : 0u;
    ctx->stats = S;
    ctx->P = (uint64_t)N * cap;
    ctx->n_items = S.n_row_items;
    ctx->d_row_begin = ctx->d_row_begin_local;
    ctx->last_index_path = 1;
    ctx->indexed = true;
    if (stats) *stats = S;

    // ---- 4. K3 + K4 on this rank's rows, then the pair lists of all ranks on every rank, ordered by (i, j) ---------------
    uint64_t n_r = 0;
    ctx->skip_pair_sort = true;
    const int rc_pw = ygpu_pairwise_flag_device(ctx, threshold, ctx->g_begin, ctx->g_end, &n_r);
    ctx->skip_pair_sort = false;
    YG_CHECK(rc_pw);
    uint64_t total = 0;
    YG_CHECK(gather_pairs(ctx, n_r, my_ovf, &total));
    ctx->n_pairs = total;
    *n_pairs_total = total;
    return 0;
}

// ---- replicated index, rows split by measured work: the layout north_star starts from, and the multi-GPU route for databases the
// sharded step refuses (extreme skew: there the pairwise count dominates and splits cleanly by rows) --------------------------------
// Every rank holds ALL sketches (ygpu_load_sketches) and builds the full index; rank r counts / flags the rows of its
// work-balanced range; the pair lists are gathered like in the sharded step.
extern "C" int ygpu_train_step_replicated(ygpu_ctx* ctx, double threshold, ygpu_index_stats* stats, uint64_t* n_pairs_total) {
    if (!ctx || !n_pairs_total) return YGPU_ERR_ARG;
    *n_pairs_total = 0;
    if (!ctx->comm || ctx->sharded || !ctx->loaded) return ygpu_fail(ctx, YGPU_ERR_STATE, "train_step_replicated: ygpu_comm_init and ygpu_load_sketches (all sketches) first");
    const int N = ctx->comm->nranks, rank = ctx->comm->rank;
    ygpu_index_stats S{};
    YG_CHECK(ygpu_build_index(ctx, &S));
    if (stats) *stats = S;
    std::vector<uint32_t> bounds((size_t)N + 1, 0);
    YG_CHECK(ygpu_row_partition(ctx, (uint32_t)N, bounds.data()));      // same index on every rank => same bounds on every rank
    uint64_t n_r = 0;
    ctx->skip_pair_sort = true;
    const int rc = ygpu_pairwise_flag_device(ctx, threshold, bounds[rank], bounds[rank + 1], &n_r);
    ctx->skip_pair_sort = false;
    YG_CHECK(rc);
    YG_CHECK(dev_alloc(ctx, &ctx->d_sh_info, (uint64_t)SHI_WORDS));
    uint64_t total = 0;
    YG_CHECK(gather_pairs(ctx, n_r, 0ull, &total));
    *n_pairs_total = total;
    return 0;
}
