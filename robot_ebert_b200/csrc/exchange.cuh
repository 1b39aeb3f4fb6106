// Exchange steps of the row-sharded single-request path over NVLink peer memory (SURVEY.md §8e: the path shards by
// catalog rows and has exactly one exchange of per-rank results, plus one of partial profiles when the request is a
// liked-rows list).  No NCCL on the request path: a rank stores its block straight into every peer's symmetric buffer
// (P2P stores through NVSwitch), fences at system scope, publishes a sequence-number flag in every peer, acquire-spins on
// its own flags and then combines the blocks in fixed rank order, so every rank computes the same bits.
//
// One symmetric buffer per rank holds `channels` independent channels (one per concurrent request stream: FastAPI serves
// from a threadpool, api/users.py:151), each laid out in 64-bit words as
//     gather [2][world][2 * words_cap]   packed results (rows k | fp64 scores k | count + tag | margin) in "LL" form: every
//                                        32-bit half of a word travels in its own 8-byte store together with the call's
//                                        sequence number, so data and flag arrive atomically — no fence, no separate flag
//     flags  [2][world]                  (unused by the LL form; kept so the layout has one shape)
//     prof   [2][world][prof_cap]    fp64 partial profile sums (ld values) + the weight sum
//     pflags [2][world]
// The leading [2] is the parity of the channel's call sequence number.  Parity double-buffering suffices because a rank
// can be at most one call ahead of a peer: it needs that peer's flag of the current call to finish it.
#pragma once

#include "exact.cuh"
#include "merge.cuh"

namespace rebert {

constexpr int kMaxPeers = 16;

struct Exchange {
    unsigned long long* peer[kMaxPeers];   // this channel's base inside every rank's buffer, as this process maps it
    int world, rank;
    int words_cap, prof_cap;               // 2 * k_max + 2, prof_len + 1
    unsigned seq;                          // call number on this channel (same on every rank), never 0
    long long timeout_cycles;
    int* err;                              // int32, device or device-addressable pinned: 1 + rank = result not delivered, 51 + rank = partial
                                           // profile not delivered, 101 + rank = tag mismatch
};

__host__ __device__ __forceinline__ size_t xchg_channel_words(int world, int words_cap, int prof_cap) {
    return (size_t)4 * world * words_cap + (size_t)2 * world + (size_t)2 * world * prof_cap + (size_t)2 * world;
}
__device__ __forceinline__ size_t xchg_gather_off(const Exchange& x, int parity, int r) { return ((size_t)parity * x.world + r) * 2 * x.words_cap; }
__device__ __forceinline__ size_t xchg_prof_off(const Exchange& x, int parity, int r) {
    return (size_t)4 * x.world * x.words_cap + (size_t)2 * x.world + ((size_t)parity * x.world + r) * x.prof_cap;
}
__device__ __forceinline__ size_t xchg_pflag_off(const Exchange& x, int parity, int r) {
    return (size_t)4 * x.world * x.words_cap + (size_t)2 * x.world + (size_t)2 * x.world * x.prof_cap + (size_t)parity * x.world + r;
}

// publish `seq` in every peer's flag slot for my rank, then wait until every rank's flag in MY buffer shows `seq`.
// Called by all threads of the CTA after the payload stores (and a __threadfence_system + __syncthreads by the caller).
__device__ __forceinline__ void xchg_publish_and_wait(const Exchange& x, size_t my_flag_off_in_peer, size_t flag0_off_in_mine, int err_base = 1) {
    if ((int)threadIdx.x < x.world) {
        unsigned long long* f = x.peer[threadIdx.x] + my_flag_off_in_peer;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"((unsigned long long)x.seq) : "memory");
        const unsigned long long* w = x.peer[x.rank] + flag0_off_in_mine + threadIdx.x;
        const long long t0 = clock64();
        unsigned long long v;
        while (true) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(w) : "memory");
            if (v == (unsigned long long)x.seq) break;
            if (clock64() - t0 > x.timeout_cycles) { *(volatile int*)x.err = err_base + threadIdx.x; break; }   // plain store: err may live in pinned host memory
            __nanosleep(64);
        }
    }
    __syncthreads();
}

// Result exchange + merge, LL protocol (as in NCCL's low-latency path): half h (32 bits) of word w of my block goes to
// every peer as ONE 8-byte store {half, seq}; 8-byte stores are atomic over NVLink, so a reader that sees `seq` in the upper
// half has the data in the lower half — no system-scope fence and no separate flag round trip, which together cost ~10 us
// per request in the fenced form.  A stale word (the slot's previous use was call seq - 2) can never carry `seq`.
// `local` = this rank's packed block of 2k+2 words (shared or global memory); `out` receives the merged block (global or
// pinned host memory); s_all = world * (2k + 2) words of shared scratch.  All threads of the CTA call.
__device__ __forceinline__ void exchange_results(const Exchange& x, int k, const unsigned long long* local, unsigned long long* out,
                                                 unsigned long long* s_all) {
    const int words = 2 * k + 2;
    const int halves = 2 * words;
    const int parity = (int)(x.seq & 1u);
    REBERT_ASSERT(words <= x.words_cap && x.rank < x.world && x.world <= kMaxPeers);
    const unsigned long long tagged = (unsigned long long)x.seq << 32;
    for (int i = threadIdx.x; i < x.world * halves; i += blockDim.x) {
        const int pr = i / halves, h = i - pr * halves;
        const unsigned long long wv = local[h >> 1];
        const unsigned long long half = (h & 1) ? (wv >> 32) : (wv & 0xFFFFFFFFull);
        unsigned long long* dst = x.peer[pr] + xchg_gather_off(x, parity, x.rank) + h;
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(tagged | half) : "memory");
    }
    // collect every rank's block from MY buffer: poll each LL word until it carries this call's sequence number
    const unsigned long long* g = x.peer[x.rank] + xchg_gather_off(x, parity, 0);
    const long long t0 = clock64();
    for (int i = threadIdx.x; i < x.world * halves; i += blockDim.x) {
        const int l = i / halves, h = i - l * halves;
        const unsigned long long* src = g + (size_t)l * 2 * x.words_cap + h;
        unsigned long long v;
        while (true) {
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
            if ((unsigned)(v >> 32) == x.seq) break;
            if (clock64() - t0 > x.timeout_cycles) { *(volatile int*)x.err = 1 + l; v = 0; break; }   // plain store: err may live in pinned host memory
            __nanosleep(32);
        }
        ((unsigned*)s_all)[(size_t)l * halves + h] = (unsigned)v;             // little endian: half h of word h >> 1
    }
    __syncthreads();
    int total = 0;
    double margin = INFINITY;
    const unsigned my_tag = (unsigned)(local[2 * k] >> 32);
    for (int l = 0; l < x.world; ++l) {
        const unsigned long long* L = s_all + (size_t)l * words;
        total += min((int)(unsigned)L[2 * k], k);
        margin = fmin(margin, __longlong_as_double((long long)L[2 * k + 1]));
        // every rank must be serving the SAME request on this channel: a differing tag means the callers' request order diverged
        // (a peer that never delivered has already been reported and leaves a stale block here: do not relabel that)
        if ((unsigned)(L[2 * k] >> 32) != my_tag && threadIdx.x == 0 && *(volatile int*)x.err == 0) *(volatile int*)x.err = 101 + l;
    }
    const int nout = total < k ? total : k;
    for (int i = threadIdx.x; i < x.world * k; i += blockDim.x) {
        const int l = i / k, e = i - l * k;
        const unsigned long long* L = s_all + (size_t)l * words;
        if (e >= (int)(unsigned)L[2 * k]) continue;
        const int64_t r = (int64_t)L[e];
        const double sc = __longlong_as_double((long long)L[k + e]);
        int rank = e;
        for (int o = 0; o < x.world; ++o) {
            if (o == l) continue;
            const unsigned long long* O = s_all + (size_t)o * words;
            int lo = 0, hi = min((int)(unsigned)O[2 * k], k);
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (better(__longlong_as_double((long long)O[k + mid]), (int64_t)O[mid], sc, r)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < k) {
            out[rank] = (unsigned long long)r;
            out[k + rank] = (unsigned long long)__double_as_longlong(sc);
        }
    }
    for (int i = nout + threadIdx.x; i < k; i += blockDim.x) {
        out[i] = (unsigned long long)(-1ll);
        out[k + i] = (unsigned long long)__double_as_longlong(-INFINITY);
    }
    if (threadIdx.x == 0) {
        out[2 * k] = (unsigned long long)(unsigned)nout | ((unsigned long long)my_tag << 32);
        out[2 * k + 1] = (unsigned long long)__double_as_longlong(margin);
    }
}

// Partial-profile exchange (lib.py:51-52 with the liked rows scattered over the shards): every rank contributes the fp64
// sum of ITS liked rows' unit vectors (len values) ; total[c] = sum over ranks in rank order 0..world-1, so all ranks hold
// identical bits.  The weight sum is the same on every rank already (profile_accumulate counts every entry).
__device__ __forceinline__ void exchange_profile(const Exchange& x, int len, const double* local, double* total) {   // total may alias local
    const int parity = (int)(x.seq & 1u);
    REBERT_ASSERT(len < x.prof_cap + 1 && x.rank < x.world);
    for (int i = threadIdx.x; i < x.world * len; i += blockDim.x) {
        const int pr = i / len, c = i - pr * len;
        x.peer[pr][xchg_prof_off(x, parity, x.rank) + c] = (unsigned long long)__double_as_longlong(local[c]);
    }
    __threadfence_system();
    __syncthreads();
    xchg_publish_and_wait(x, xchg_pflag_off(x, parity, x.rank), xchg_pflag_off(x, parity, 0), 51);
    const unsigned long long* g = x.peer[x.rank] + xchg_prof_off(x, parity, 0);
    for (int c = threadIdx.x; c < len; c += blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < x.world; ++r) s += __longlong_as_double((long long)__ldcg(g + (size_t)r * x.prof_cap + c));
        total[c] = s;
    }
}

// host side: fill an Exchange from the C-ABI description (defined in finalize.cu)
int make_exchange(const rebert_exchange_t* ex, int32_t* err_flag, Exchange* out);

// ---- internal launchers shared by gemv_topk.cu / finalize.cu / catalog.cu / host_api.cu ----------------------------
// Request form of the single-query path: the streaming kernel publishes its pruned candidate keys, and a cluster kernel
// placed behind it by programmatic dependent launch selects the kc winners, re-scores them in fp64, ranks them and writes
// the packed result (and runs the exchange on a row shard).  fused == nullptr: the streaming kernel alone, kc candidate
// keys to cand_keys (the last CTA merges).
struct GemvFused {
    const rebert_catalog_t* exact_cat;   // catalog of record (the streamed catalog may be its int8 shadow)
    const double* q64;
    int k;
    unsigned long long* out_packed;
    uint32_t tag;
    const Exchange* xchg;                // nullptr on a single GPU
    uint32_t* done_flag;                 // device-addressable pinned host word that receives done_token after the result (or nullptr)
    uint32_t done_token;
};
// What the streaming kernel leaves in the workspace for the cluster kernel.
struct Published {
    PublishedKeys keys;
    unsigned* ctl;             // 32 control words (ticket, hint, tile claims, compaction cursors): the cluster kernel leaves them zero
};
int finalize_published_launch(const Published& pub, const GemvFused& f, int64_t row_base, cudaStream_t st);
int gemv_launch(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, int32_t kc, void* workspace,
                size_t workspace_bytes, uint64_t* cand_keys, const GemvFused* fused, cudaStream_t st);
// false for an int8 shadow whose rows no streaming kernel takes (gemv_launch would return REBERT_ERR_UNSUPPORTED)
bool gemv_streams(const rebert_catalog_t* cat);
int stage_profile_launch(const rebert_catalog_t* cat, const int32_t* liked_host, const float* w_host, int n_liked, const int32_t* excl_host,
                         int n_excl, int32_t* excl_dev, double* sum64, double* wsum, float* qn32, double* qn64, const Exchange* x,
                         cudaStream_t st);
}  // namespace rebert
