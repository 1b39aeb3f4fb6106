// Selection of the kc best candidate keys out of what the CTAs of the streaming kernel kept (gemv_topk.cu), shared by the
// streaming kernel's own last-CTA merge (rebert_gemv_topk) and the cluster kernel of the request path (finalize.cu).
#pragma once

#include "common.cuh"

namespace rebert {

__device__ __forceinline__ uint64_t ldcg_u64(const uint64_t* p) { return __ldcg((const unsigned long long*)p); }

constexpr int kPubRegions = 16;             // compaction regions (CTA b publishes into region b % 16: 16x less contention on a cursor)

// What the CTAs of the streaming kernel publish (all pointers into the launch workspace).
struct PublishedKeys {
    const uint64_t* keys;      // [kPubRegions][region_cap] kept keys, compacted per region in arrival order
    const unsigned* cursors;   // [kPubRegions] keys in each region (= the compaction cursors)
    const uint64_t* heads;     // [lists, P] the P = ceil(kc / lists) best keys of every CTA list (zero padded)
    const uint64_t* tails;     // [lists] the kc-th key of a CTA list that is full, else 0
    int lists, P, kc, region_cap;
};

// The kc best published keys -> out[kc] (sorted best first, zero padded; shared or global memory).  Every global load this needs —
// region sizes, list heads and tails, and the keys themselves — is issued in ONE round before the first is used (each
// L2 round trip here sits on the critical path of the request); keys are then filtered against the pruning threshold
//   T0 = max over lists of their kc-th key            (that one list alone holds kc keys >= T0)
//   T1 = kc-th largest key among the first P keys of every list
// and the few survivors are ordered by rank counting (one pass, no barriers) or, beyond 512 of them, a bitonic sort.
// buf: `cap` keys of scratch (power of two >= max(2 kc, kc + lists)); all threads call.

// Mass ties (more keys within the threshold than any buffer holds): merge everything that was published, region by region,
// into the running best kc.  Correct for any input, slow.  rtot: keys per region (shared memory); all threads call.
static __device__ void merge_all_regions(const PublishedKeys& pub, const unsigned* rtot, int cap, uint64_t* buf, uint64_t* out) {
    const int kc = pub.kc;
    for (int i = threadIdx.x; i < kc; i += blockDim.x) out[i] = 0;
    __syncthreads();
    for (int r = 0; r < kPubRegions; ++r) {
        int tot = (int)rtot[r];
        if (tot > pub.region_cap) tot = pub.region_cap;
        // merge region r into the running best kc: buf = [out (kc) | region chunk]
        int done = 0;
        while (done < tot) {
            int take = tot - done;
            if (take > cap - kc) take = cap - kc;
            for (int i = threadIdx.x; i < kc; i += blockDim.x) buf[i] = out[i];
            for (int i = threadIdx.x; i < take; i += blockDim.x) buf[kc + i] = ldcg_u64(pub.keys + (size_t)r * pub.region_cap + done + i);
            int p2 = 2;
            while (p2 < kc + take) p2 <<= 1;
            for (int i = kc + take + threadIdx.x; i < p2; i += blockDim.x) buf[i] = 0;
            __syncthreads();
            block_bitonic_sort_desc(buf, p2);
            for (int i = threadIdx.x; i < kc; i += blockDim.x) out[i] = buf[i];
            __syncthreads();
            done += take;
        }
    }
}

// More than 512 survivors (rare): pad to a power of two, bitonic sort, keep the best kc.  Out of line: cold code.
static __device__ void sort_survivors(uint64_t* buf, int cnt, int kc, uint64_t* out) {
    int p2 = 2;
    while (p2 < cnt || p2 < kc) p2 <<= 1;
    for (int i = cnt + threadIdx.x; i < p2; i += blockDim.x) buf[i] = 0;
    __syncthreads();
    block_bitonic_sort_desc(buf, p2);
    for (int i = threadIdx.x; i < kc; i += blockDim.x) out[i] = buf[i];
    __syncthreads();
}

// THREADS: the block size when the caller knows it at compile time (the slot arithmetic below then folds into shifts and masks —
// a third of this function's instructions otherwise), 0 = read blockDim.x.
template <int INFLIGHT, int THREADS = 0>
__device__ inline void select_winners(const PublishedKeys& pub, int cap, uint64_t* buf, uint64_t* out) {
    __shared__ unsigned long long s_t0, s_t1;
    __shared__ int s_cnt;
    __shared__ unsigned s_rtot[kPubRegions];
    const int nthr = THREADS ? THREADS : (int)blockDim.x;
    const int kc = pub.kc, lists = pub.lists;
    const int S = pub.P * lists;                    // kc <= S < kc + lists <= cap
    if (threadIdx.x == 0) { s_t0 = 0; s_t1 = 0; s_cnt = 0; }
    if (threadIdx.x < kPubRegions) s_rtot[threadIdx.x] = __ldcg(pub.cursors + threadIdx.x);
    // ---- round 1 of loads: tails, heads, and an optimistic first batch of keys (region sizes are not known yet, so the
    // batch reads slots [0, INFLIGHT * blockDim) of the flattened regions and sorts out validity afterwards)
    unsigned long long t0 = 0;
    for (int l = threadIdx.x; l < lists; l += blockDim.x) {
        const unsigned long long v = ldcg_u64(pub.tails + l);
        t0 = v > t0 ? v : t0;
    }
    for (int e = threadIdx.x; e < S; e += blockDim.x) buf[e] = ldcg_u64(pub.heads + e);
    // Flattened view of the regions: slot s = entry (s / 512) * 32 + s % 32 of region (s / 32) % 16 — a warp reads 32
    // consecutive keys of ONE region (coalesced), the warps rotate through the regions, and every region's first entries
    // (the only ones that exist when lists are short) come first.
    uint64_t kk[INFLIGHT];
    const int per_round = INFLIGHT * nthr;
#pragma unroll
    for (int j = 0; j < INFLIGHT; ++j) {
        const int sidx = (int)threadIdx.x + j * nthr;
        const int r = (sidx >> 5) % kPubRegions, e = (sidx / (32 * kPubRegions)) * 32 + (sidx & 31);
        kk[j] = e < pub.region_cap ? ldcg_u64(pub.keys + (size_t)r * pub.region_cap + e) : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long v = __shfl_xor_sync(0xffffffffu, t0, o);
        t0 = v > t0 ? v : t0;
    }
    if ((threadIdx.x & 31) == 0 && t0) atomicMax(&s_t0, t0);
    __syncthreads();
    for (int e = threadIdx.x; e < S; e += blockDim.x) {
        const uint64_t key = buf[e];
        if (key == 0) continue;
        int rank = 0;
        for (int j = 0; j < S; ++j) rank += buf[j] > key;
        if (rank == kc - 1) s_t1 = key;            // keys are distinct, so exactly one thread can hit this
    }
    __syncthreads();
    const uint64_t T = s_t0 > s_t1 ? s_t0 : s_t1;
    unsigned max_tot = 0;
#pragma unroll
    for (int r = 0; r < kPubRegions; ++r) max_tot = max(max_tot, s_rtot[r]);
    if ((int)max_tot > pub.region_cap) max_tot = (unsigned)pub.region_cap;
    const int slots = (((int)max_tot + 31) / 32) * 32 * kPubRegions;   // flattened slots that can hold a key
    __syncthreads();                                // everybody is past the T1 count: buf may now be reused for the survivors
    for (int base = 0; base < slots; base += per_round) {
        if (base > 0) {
#pragma unroll
            for (int j = 0; j < INFLIGHT; ++j) {
                const int sidx = base + (int)threadIdx.x + j * nthr;
                const int r = (sidx >> 5) % kPubRegions, e = (sidx / (32 * kPubRegions)) * 32 + (sidx & 31);
                kk[j] = (sidx < slots && e < (int)s_rtot[r]) ? ldcg_u64(pub.keys + (size_t)r * pub.region_cap + e) : 0;
            }
        }
#pragma unroll
        for (int j = 0; j < INFLIGHT; ++j) {
            const int sidx = base + (int)threadIdx.x + j * nthr;
            const int r = (sidx >> 5) % kPubRegions, e = (sidx / (32 * kPubRegions)) * 32 + (sidx & 31);
            // first batch: stale slots beyond the region size are dropped here.  One shared-memory atomic per WARP (ballot +
            // prefix count): a hundred survivors appending one by one would queue on the counter for microseconds.
            const bool keep = e < (int)s_rtot[r] && e < pub.region_cap && kk[j] >= T && kk[j] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (m) {
                const int lane_ = threadIdx.x & 31;
                int wbase = 0;
                if (lane_ == 0) wbase = atomicAdd(&s_cnt, __popc(m));
                wbase = __shfl_sync(0xffffffffu, wbase, 0);
                const int idx = wbase + __popc(m & ((1u << lane_) - 1u));
                REBERT_ASSERT(idx >= 0);
                if (keep && idx < cap) buf[idx] = kk[j];
            }
        }
    }
    __syncthreads();
    const int cnt = s_cnt;
    if (cnt > cap) {                               // mass ties: correct but slow path over everything that was published
        merge_all_regions(pub, s_rtot, cap, buf, out);
        return;
    }
    if (cnt <= 512) {
        // rank counting: survivor i goes to slot (number of survivors greater than it); distinct keys => a permutation
        for (int i = cnt + threadIdx.x; i < kc; i += blockDim.x) out[i] = 0;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const uint64_t key = buf[i];
            int rank = 0;
            for (int j = 0; j < cnt; ++j) rank += buf[j] > key;
            REBERT_ASSERT(key != 0 && rank < cnt);
            if (rank < kc) out[rank] = key;
        }
        __syncthreads();
        return;
    }
    sort_survivors(buf, cnt, kc, out);
}

// The same selection spread over the CTAs of a thread-block cluster (the request path's exact-pass kernel, long candidate
// lists).  With kc = 128 / 256 the streaming kernel publishes 19k / 38k keys; every CTA scanning all of them took 7 rounds of
// L2 loads (25 us at kc = 256) and the survivors (> 512) a block-wide bitonic sort (9 us).  Here
//   (1) every CTA finds the threshold T from the list heads and tails (redundant: ~300 keys),
//   (2) CTA c scans only its kPubRegions / CSIZE regions — one round of loads — and keeps the keys >= T,
//   (3) pushes its survivors into EVERY CTA's `buf` through distributed shared memory (one remote atomic per target reserves
//       the range), cluster barrier,
//   (4) ranks its 1/CSIZE slice of the survivors against all of them (4 threads per survivor) and stores each winner at its
//       rank into every CTA's `out`, cluster barrier.
// stage: stage_cap >= max(3 kc, kc + lists) keys of scratch that nothing else uses until the winners are known (heads first, then
// the local survivors); `out` may be its first kc entries.  s_total: one int per CTA, zero before a cluster barrier that precedes this call.
// Falls back to merge_all_regions (every CTA, redundantly) when the survivors overflow `buf` or a CTA's stage.
template <int CSIZE, int THREADS, typename Cluster>
__device__ inline void select_winners_cluster(Cluster& cluster, const PublishedKeys& pub, int cap, uint64_t* buf, uint64_t* stage, int stage_cap,
                                              uint64_t* out, int* s_total) {
    static_assert(kPubRegions % CSIZE == 0, "regions must divide over the cluster");
    constexpr int RPC = kPubRegions / CSIZE;        // regions scanned by one CTA
    constexpr int INFLIGHT = 24;                    // key loads in flight per thread
    __shared__ unsigned long long s_t0, s_t1;
    __shared__ int s_cnt;
    __shared__ unsigned s_rtot[kPubRegions];
    __shared__ int s_base[CSIZE];
    const int crank = (int)cluster.block_rank();
    const int kc = pub.kc, lists = pub.lists;
    const int S = pub.P * lists;                    // kc <= S < kc + lists <= stage_cap (the caller sizes the stage for it)
    if (threadIdx.x == 0) { s_t0 = 0; s_t1 = 0; s_cnt = 0; }
    if (threadIdx.x < kPubRegions) s_rtot[threadIdx.x] = __ldcg(pub.cursors + threadIdx.x);
    unsigned long long t0 = 0;
    for (int l = threadIdx.x; l < lists; l += blockDim.x) {
        const unsigned long long v = ldcg_u64(pub.tails + l);
        t0 = v > t0 ? v : t0;
    }
    for (int e = threadIdx.x; e < S; e += blockDim.x) stage[e] = ldcg_u64(pub.heads + e);
    // optimistic batch over this CTA's regions, flattened like select_winners: slot s = entry (s / (32 RPC)) * 32 + s % 32 of
    // region crank * RPC + (s / 32) % RPC
    uint64_t kk[INFLIGHT];
    constexpr int nthr = THREADS;
    const int per_round = INFLIGHT * nthr;
#pragma unroll
    for (int j = 0; j < INFLIGHT; ++j) {
        const int sidx = (int)threadIdx.x + j * nthr;
        const int r = crank * RPC + (sidx >> 5) % RPC, e = (sidx / (32 * RPC)) * 32 + (sidx & 31);
        kk[j] = e < pub.region_cap ? ldcg_u64(pub.keys + (size_t)r * pub.region_cap + e) : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long v = __shfl_xor_sync(0xffffffffu, t0, o);
        t0 = v > t0 ? v : t0;
    }
    if ((threadIdx.x & 31) == 0 && t0) atomicMax(&s_t0, t0);
    __syncthreads();
    for (int e = threadIdx.x; e < S; e += blockDim.x) {
        const uint64_t key = stage[e];
        if (key == 0) continue;
        int rank = 0;
        for (int j = 0; j < S; ++j) rank += stage[j] > key;
        if (rank == kc - 1) s_t1 = key;
    }
    __syncthreads();
    const uint64_t T = s_t0 > s_t1 ? s_t0 : s_t1;
    unsigned max_tot = 0;
#pragma unroll
    for (int r = 0; r < RPC; ++r) max_tot = max(max_tot, s_rtot[crank * RPC + r]);
    if ((int)max_tot > pub.region_cap) max_tot = (unsigned)pub.region_cap;
    const int slots = (((int)max_tot + 31) / 32) * 32 * RPC;
    __syncthreads();                                // the heads are dead: `stage` now collects this CTA's survivors
    for (int base = 0; base < slots; base += per_round) {
        if (base > 0) {
#pragma unroll
            for (int j = 0; j < INFLIGHT; ++j) {
                const int sidx = base + (int)threadIdx.x + j * nthr;
                const int r = crank * RPC + (sidx >> 5) % RPC, e = (sidx / (32 * RPC)) * 32 + (sidx & 31);
                kk[j] = (sidx < slots && e < (int)s_rtot[r]) ? ldcg_u64(pub.keys + (size_t)r * pub.region_cap + e) : 0;
            }
        }
#pragma unroll
        for (int j = 0; j < INFLIGHT; ++j) {
            const int sidx = base + (int)threadIdx.x + j * nthr;
            const int r = crank * RPC + (sidx >> 5) % RPC, e = (sidx / (32 * RPC)) * 32 + (sidx & 31);
            const bool keep = e < (int)s_rtot[r] && e < pub.region_cap && kk[j] >= T && kk[j] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (m) {
                const int lane_ = threadIdx.x & 31;
                int wbase = 0;
                if (lane_ == 0) wbase = atomicAdd(&s_cnt, __popc(m));
                wbase = __shfl_sync(0xffffffffu, wbase, 0);
                const int idx = wbase + __popc(m & ((1u << lane_) - 1u));
                if (keep && idx < stage_cap) stage[idx] = kk[j];
            }
        }
    }
    __syncthreads();
    const int mine = s_cnt;
    const bool overflow = mine > stage_cap;
    // reserve this CTA's range in every CTA's buf (an overflowing CTA poisons the totals: everybody takes the slow path)
    if (threadIdx.x < CSIZE) s_base[threadIdx.x] = atomicAdd(cluster.map_shared_rank(s_total, threadIdx.x), overflow ? cap + 1 : mine);
    __syncthreads();
    if (!overflow) {
        for (int t = 0; t < CSIZE; ++t) {
            uint64_t* rbuf = cluster.map_shared_rank(buf, t);
            const int b0 = s_base[t];
            for (int i = threadIdx.x; i < mine; i += blockDim.x)
                if (b0 + i < cap) rbuf[b0 + i] = stage[i];
        }
    }
    cluster.sync();                                 // every CTA's survivors are in every CTA's buf (and every stage is dead)
    const int total = *s_total;
    if (total > cap) {
        merge_all_regions(pub, s_rtot, cap, buf, out);
        return;
    }
    for (int i = total + threadIdx.x; i < kc; i += blockDim.x) out[i] = 0;
    // rank counting, 4 threads per survivor (keys are distinct: ranks are a permutation).  Each CTA ranks the survivors it
    // gathered itself — the range it reserved in its OWN buf.  (The arrival order of the pushes differs from CTA to CTA, so a
    // position-based split of buf would not partition the survivors.)
    const int lo = s_base[crank];
    const int len = mine;
    const int g = threadIdx.x >> 2, sub = threadIdx.x & 3, groups = (int)blockDim.x >> 2;
    for (int b0 = 0; b0 < len; b0 += groups) {      // trip count uniform over the CTA: the shuffles below need whole warps
        const int ii = b0 + g;
        const bool live = ii < len;
        const uint64_t key = live ? buf[lo + ii] : ~0ull;
        int rank = 0;
        for (int j = sub; j < total; j += 4) rank += buf[j] > key;
        rank += __shfl_xor_sync(0xffffffffu, rank, 1);
        rank += __shfl_xor_sync(0xffffffffu, rank, 2);
        if (live && sub == 0 && rank < kc) {
            REBERT_ASSERT(key != 0);
#pragma unroll
            for (int t = 0; t < CSIZE; ++t) cluster.map_shared_rank(out, t)[rank] = key;
        }
    }
    cluster.sync();                                 // the winners are in every CTA's out
}

}  // namespace rebert
