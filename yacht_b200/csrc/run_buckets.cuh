// libyachtgpu -- K5 on the partitioned reference (included by index_msd.cu, inside its anonymous namespace).
//
// Replaces, for `yacht run` (reference src/yacht/hypothesis_recovery_src.py):
//   get_organisms_with_nonzero_overlap :30-113   (`sourmash scripts multisearch ... -t 0`: genomes sharing >= 1 hash with the sample)
//   get_exclusive_hashes               :116-206  (hashes held by exactly one nontrivial genome, and how many of them the sample has)
//
// The first version sorted all (hash, genome) pairs and the sample with a library radix sort and walked equal-hash runs
// with one thread per run head (0.06 of the HBM roofline).  The train path already knows how to bring equal hashes
// together without a sort: the two-level MSD partition.  The run path reuses it -- the partitioned reference words stay
// resident across samples -- and probes bucket by bucket:
//   * the sample is bucketed by the same leading hash bits (a counting scatter: ~20 hashes per bucket at 10 M sample
//     hashes), so a bucket's sample fits shared memory together with a 2048-bit filter over its next 11 hash bits;
//   * pass 1 (overlap):   a reference word survives iff its hash is in the bucket's sample (filter bit, then exact compare);
//   * pass 2 (exclusive): a reference word survives iff its genome is nontrivial (bitmap over the genomes);
//   * survivors -- a few per cent of the words -- are grouped exactly as k2_group2 groups a bucket (sub-bucket counting
//     filter, dense candidates, one scan of the sub-bucket per candidate) and the first copy of every distinct
//     (hash, genome) credits n_overlap / the single holder of a hash gets n_exclusive (+ n_match when the sample has it).
// Each pass streams the packed words once (8 bytes per hash slot) through bulk asynchronous copies.
struct RunBucketArgs {
    const uint64_t* ent;            // partitioned reference words (remaining hash bits << gb | genome id)
    const uint32_t* begin;          // final bucket b: words [begin[b], end[b]) of ent
    const uint32_t* end;
    uint32_t nb;
    int gb;
    int sub_shift;                  // sub-bucket digit = (word >> sub_shift) & sub_mask
    uint32_t sub_mask;
    int rest_bits;                  // hash bits below the sub-bucket digit
    uint64_t key_mask;              // (word >> gb) & key_mask = all hash bits that vary inside a final bucket
    const uint64_t* skeys;          // bucketed sample: the same bits of every sample hash
    const uint32_t* sbase;          // [nb + 1]
    const uint32_t* ntbits;         // pass 2: bitmap of the nontrivial genomes
    ygpu_genome_counts* counts;
};

constexpr int RB_SCAP = 1024;       // sample hashes of one bucket held in shared memory (more: the general path takes the sample)
constexpr int RB_SMALL = 192;       // up to this many survivors per bucket are settled by a direct all-pairs scan (no sub-bucket machinery)

struct __align__(16) RunSmem {
    uint64_t stage[G2_WIN];         // the bucket's reference words (bulk copy target)
    uint64_t candK[G2_WIN + 4];     // surviving words, sub-bucket by sub-bucket: hash bits below the sub-bucket digit
    uint64_t skey[RB_SCAP];         // the bucket's sample hashes
    uint32_t candG[G2_WIN + 4];     // ... their genome ids
    uint32_t cnt[G2_NSUB];
    uint32_t ext[G2_WIN];           // per candidate: sub-bucket start | size << 10 | sub-bucket digit << 20
    uint32_t sbits[G2_NSUB / 32];   // filter over the sub-bucket digits of the bucket's sample
    unsigned short start2[G2_NSUB + 8];
    uint64_t lk[RB_SMALL];          // the survivors of a bucket with few of them: full key (sub-bucket digit and the bits below it) ...
    uint32_t lg[RB_SMALL];          // ... and genome id
    uint32_t wsum[G2_THREADS / 32];
    uint32_t next[2][4];            // [parity]{first word, words, bucket id}
    uint32_t nsurv;
    uint64_t mbar;
};

// MODE 0: overlap (survivor = hash in the sample), MODE 1: exclusive (survivor = nontrivial genome)
template <int MODE>
__global__ void __launch_bounds__(G2_THREADS, 4) k5_bucket(const RunBucketArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RunSmem& sm = *reinterpret_cast<RunSmem*>(smem_raw);
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t gmask = a.gb ? (uint32_t)((1ull << a.gb) - 1ull) : 0u;
    const uint64_t rest_mask = a.rest_bits >= 64 ? ~0ull : ((1ull << a.rest_bits) - 1ull);

    uint32_t b_next = blockIdx.x;                 // thread 0 only
    uint32_t pre_lo = 0, pre_hi = 0;
    auto preload = [&]() {
        if (b_next < a.nb) { pre_lo = a.begin[b_next]; pre_hi = a.end[b_next]; }
    };
    auto advance = [&](uint32_t par) {
        uint32_t bb = 0, m = 0, b = 0;
        while (b_next < a.nb) {
            bb = pre_lo;
            m = pre_hi - pre_lo;
            b = b_next;
            b_next += gridDim.x;
            if (m) break;                         // (the host checked that every bucket fits)
            preload();
        }
        sm.next[par][0] = bb;
        sm.next[par][1] = m;
        sm.next[par][2] = b;
        if (m) {
            const uint32_t w0 = bb & ~1u, w1 = (bb + m + 1u) & ~1u;
            bulk_load(sm.stage, a.ent + w0, (w1 - w0) * 8u, &sm.mbar);
        }
        preload();          // the extent of the bucket after that one: in flight during phases B..F, consumed after the next phase A
    };
    for (uint32_t i = tid; i < G2_NSUB; i += G2_THREADS) sm.cnt[i] = 0;
    if (tid < G2_NSUB / 32) sm.sbits[tid] = 0;
    if (tid == 0) sm.nsurv = 0;
    if (tid == 0) {
        mbar_init(&sm.mbar, 1);
        mbar_init_fence();
        preload();
        advance(0);
    }
    __syncthreads();

    // is the hash of word `e` in the bucket's sample?  (filter bit over the sub-bucket digit, then the exact keys)
    auto in_sample = [&](uint64_t kfull, uint32_t sub, uint32_t ns) -> bool {
        if (!((sm.sbits[sub >> 5] >> (sub & 31u)) & 1u)) return false;
        bool hit = false;
        for (uint32_t i = 0; i < ns; i++) hit |= sm.skey[i] == kfull;
        return hit;
    };

    uint32_t par = 0, phase = 0;
    for (;;) {
        const uint32_t bb = sm.next[par][0], m = sm.next[par][1], b = sm.next[par][2];
        if (!m) break;
        // ---- the bucket's sample: keys + filter over their sub-bucket digits -----------------------------------------------
        const uint32_t s0 = a.sbase[b], ns = a.sbase[b + 1] - s0;
        for (uint32_t i = tid; i < ns; i += G2_THREADS) {
            const uint64_t k = a.skeys[s0 + i];
            sm.skey[i] = k;
            const uint32_t sub = (uint32_t)(k >> a.rest_bits) & a.sub_mask;
            atomicOr(&sm.sbits[sub >> 5], 1u << (sub & 31u));
        }
        __syncthreads();
        mbar_wait(&sm.mbar, phase);
        phase ^= 1u;
        // ---- A: four words per thread; survivors take a rank in their sub-bucket --------------------------------------------
        const uint32_t wlo = bb & 1u, whi = wlo + m;
        uint64_t e[4];
        {
            const uint4* s4 = reinterpret_cast<const uint4*>(sm.stage);
            const uint4 v0 = s4[tid], v1 = s4[G2_THREADS + tid];
            e[0] = (uint64_t)v0.x | ((uint64_t)v0.y << 32); e[1] = (uint64_t)v0.z | ((uint64_t)v0.w << 32);
            e[2] = (uint64_t)v1.x | ((uint64_t)v1.y << 32); e[3] = (uint64_t)v1.z | ((uint64_t)v1.w << 32);
        }
        uint32_t keepm = 0;                 // which of the four words survive
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t w = (k >> 1) * 512u + 2u * tid + (k & 1);
            if (w >= wlo && w < whi) {
                const uint32_t s = (uint32_t)(e[k] >> a.sub_shift) & a.sub_mask;
                bool keep;
                if (MODE == 0) {
                    keep = ns && in_sample((e[k] >> a.gb) & a.key_mask, s, ns);
                } else {
                    const uint32_t g = (uint32_t)e[k] & gmask;
                    keep = (a.ntbits[g >> 5] >> (g & 31u)) & 1u;
                }
                if (keep) {
                    keepm |= 1u << k;
                    const uint32_t pos = atomicAdd(&sm.nsurv, 1u);
                    if (pos < RB_SMALL) { sm.lk[pos] = (e[k] >> a.gb) & a.key_mask; sm.lg[pos] = (uint32_t)e[k] & gmask; }
                }
            }
        }
        __syncthreads();
        if (tid == 0) advance(par ^ 1u);
        const uint32_t nsv = sm.nsurv;
        if (nsv <= RB_SMALL) {
            // ---- few survivors (the rule: a sample overlaps a few hashes of a bucket, nontrivial genomes are a few per cent): one
            //      thread per survivor scans them all -- no sub-bucket counting, no scan, three barriers less
            if (tid < nsv) {
                const uint64_t Kq = sm.lk[tid];
                const uint32_t Gq = sm.lg[tid];
                bool copy_before = false, same_before = false, other_genome = false;
                for (uint32_t j = 0; j < nsv; j++) {
                    const bool same = sm.lk[j] == Kq;
                    const bool sameg = sm.lg[j] == Gq;
                    // "before": the slot order is arbitrary but fixed for this bucket, which is all the first-copy rule needs
                    copy_before |= same & sameg & (j < tid);
                    same_before |= same & (j < tid);
                    other_genome |= same & !sameg;
                }
                if (MODE == 0) {
                    if (!copy_before) atomicAdd(&a.counts[Gq].n_overlap, 1u);
                } else if (!same_before && !other_genome) {
                    atomicAdd(&a.counts[Gq].n_exclusive, 1u);
                    if (ns && in_sample(Kq, (uint32_t)(Kq >> a.rest_bits) & a.sub_mask, ns)) atomicAdd(&a.counts[Gq].n_match, 1u);
                }
            }
            __syncthreads();
            for (uint32_t i = tid; i < ns; i += G2_THREADS) {
                const uint32_t sub = (uint32_t)(sm.skey[i] >> a.rest_bits) & a.sub_mask;
                sm.sbits[sub >> 5] = 0;
            }
            if (tid == 0) sm.nsurv = 0;
            __syncthreads();
            par ^= 1u;
            continue;
        }
        // ---- many survivors: the sub-bucket machinery of k2_group2 -------------------------------------------------------------
        uint32_t sr[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            sr[k] = 0xFFFFFFFFu;
            if (keepm & (1u << k)) {
                const uint32_t s = (uint32_t)(e[k] >> a.sub_shift) & a.sub_mask;
                sr[k] = s | (atomicAdd(&sm.cnt[s], 1u) << 16);
            }
        }
        __syncthreads();
        // ---- B: scan the sizes of sub-buckets with >= 2 survivors (counters back to zero) ----------------------------------
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
            if (lane == 31) sm.wsum[warp] = inc;
            __syncthreads();
            const uint4 wa = *reinterpret_cast<const uint4*>(&sm.wsum[0]), wb = *reinterpret_cast<const uint4*>(&sm.wsum[4]);
            const uint32_t wp = (warp > 0 ? wa.x : 0u) + (warp > 1 ? wa.y : 0u) + (warp > 2 ? wa.z : 0u) + (warp > 3 ? wa.w : 0u) +
                                (warp > 4 ? wb.x : 0u) + (warp > 5 ? wb.y : 0u) + (warp > 6 ? wb.z : 0u);
            const uint32_t p0 = wp + inc - sum;
            const uint32_t p1 = p0 + c0.x, p2 = p1 + c0.y, p3 = p2 + c0.z, p4 = p3 + c0.w, p5 = p4 + c1.x, p6 = p5 + c1.y, p7 = p6 + c1.z;
            *reinterpret_cast<uint4*>(&sm.start2[8 * tid]) = make_uint4(p0 | (p1 << 16), p2 | (p3 << 16), p4 | (p5 << 16), p6 | (p7 << 16));
            if (tid == G2_THREADS - 1) sm.start2[G2_NSUB] = (unsigned short)(p7 + c1.w);
        }
        __syncthreads();
        // ---- C: a survivor alone in its sub-bucket is a hash nobody else (that survived) holds: credit it right away ---------
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (sr[k] != 0xFFFFFFFFu) {
                const uint32_t s = sr[k] & 0xffffu;
                const uint32_t lo = sm.start2[s], hi = sm.start2[s + 1];
                const uint32_t G = (uint32_t)e[k] & gmask;
                if (hi > lo) {
                    const uint32_t pos = lo + (sr[k] >> 16);
                    sm.candK[pos] = (e[k] >> a.gb) & rest_mask;
                    sm.candG[pos] = G;
                    sm.ext[pos] = lo | ((hi - lo) << 10) | (s << 20);
                } else if (MODE == 0) {
                    atomicAdd(&a.counts[G].n_overlap, 1u);
                } else {
                    atomicAdd(&a.counts[G].n_exclusive, 1u);
                    if (ns && in_sample((e[k] >> a.gb) & a.key_mask, s, ns)) atomicAdd(&a.counts[G].n_match, 1u);
                }
            }
        }
        __syncthreads();
        // ---- D: every candidate scans its sub-bucket once ------------------------------------------------------------------
        const uint32_t ncand = sm.start2[G2_NSUB];
        for (uint32_t q = tid; q < ncand; q += G2_THREADS) {
            const uint64_t Kq = sm.candK[q];
            const uint32_t Gq = sm.candG[q];
            const uint32_t x = sm.ext[q];
            const uint32_t lo = x & 0x3ffu, c = (x >> 10) & 0x3ffu, s = x >> 20;
            bool copy_before = false;        // an identical (hash, genome) word earlier in the bucket: in-sketch duplicate
            bool same_before = false;        // the same hash earlier in the bucket (any genome)
            bool other_genome = false;       // the same hash in another (surviving) genome
            for (uint32_t j = 0; j < c; j++) {
                const bool same = sm.candK[lo + j] == Kq;
                const bool sameg = sm.candG[lo + j] == Gq;
                copy_before |= same & sameg & (lo + j < q);
                same_before |= same & (lo + j < q);
                other_genome |= same & !sameg;
            }
            if (MODE == 0) {
                if (!copy_before) atomicAdd(&a.counts[Gq].n_overlap, 1u);         // sets: once per (hash, genome)
            } else if (!same_before && !other_genome) {                           // one credit per hash held by exactly one nontrivial genome
                atomicAdd(&a.counts[Gq].n_exclusive, 1u);
                if (ns && in_sample(((uint64_t)s << a.rest_bits) | Kq, s, ns)) atomicAdd(&a.counts[Gq].n_match, 1u);
            }
        }
        __syncthreads();
        // the bucket's filter bits back to zero (the next bucket fills them after the barrier below)
        for (uint32_t i = tid; i < ns; i += G2_THREADS) {
            const uint32_t sub = (uint32_t)(sm.skey[i] >> a.rest_bits) & a.sub_mask;
            sm.sbits[sub >> 5] = 0;
        }
        if (tid == 0) sm.nsurv = 0;
        __syncthreads();
        par ^= 1u;
    }
}

// ---- the sample, bucketed like the reference -------------------------------------------------------------------------------
// bucket of a hash = its leading d1 + d2 bits (below hb); hashes beyond the reference's range cannot match and are dropped
__device__ __forceinline__ bool sample_bucket(uint64_t h, const MsdPlan& p, uint32_t& b) {
    if (p.hb < 64 && (h >> p.hb) != 0) return false;
    const uint32_t b1 = p.d1 ? (uint32_t)(h >> (p.hb - p.d1)) : 0u;
    if (b1 >= p.nb1) return false;
    const uint32_t b2 = p.d2 ? (uint32_t)((h >> (p.hb - p.d1 - p.d2)) & ((1u << p.d2) - 1u)) : 0u;
    b = (b1 << p.d2) | b2;
    return true;
}
__global__ void __launch_bounds__(256) k5s_hist(const uint64_t* __restrict__ samp, uint64_t ns, const MsdPlan p, uint32_t* __restrict__ hist) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t b;
        if (sample_bucket(samp[i], p, b)) atomicAdd(&hist[b], 1u);
    }
}
__global__ void __launch_bounds__(256) k5s_scatter(const uint64_t* __restrict__ samp, uint64_t ns, const MsdPlan p, uint64_t key_mask,
                                                   uint32_t* __restrict__ cursor, uint64_t* __restrict__ skeys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t b;
        const uint64_t h = samp[i];
        if (sample_bucket(h, p, b)) skeys[atomicAdd(&cursor[b], 1u)] = h & key_mask;
    }
}
// nontrivial genomes as a bitmap: mask[g] != 0 when the caller chose them, else n_overlap > 0
__global__ void __launch_bounds__(256) k5_nontrivial_bits(ygpu_genome_counts* __restrict__ counts, const uint8_t* __restrict__ mask, uint32_t n,
                                                          uint32_t* __restrict__ bits) {
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < (n + 31) / 32; w += gridDim.x * blockDim.x) {
        uint32_t v = 0;
        for (uint32_t k = 0; k < 32; k++) {
            const uint32_t g = w * 32 + k;
            if (g < n) {
                const uint32_t nt = mask ? (mask[g] ? 1u : 0u) : (counts[g].n_overlap > 0 ? 1u : 0u);
                counts[g].nontrivial = nt;
                v |= nt << k;
            }
        }
        bits[w] = v;
    }
}
