// Exact pass and merges.
//   rebert_finalize_topk : fp64 re-score of the fast pass's candidates with the oracle's formula
//                          (sklearn cosine_similarity: x/||x||, y/||y||, dot — lib.py:51), then the
//                          (score desc, row asc) order of lib.py:55,63, best k out.
//   rebert_merge_topk    : the same order across per-shard result lists (row-sharded catalogs).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "exchange.cuh"

namespace rebert {

namespace cg = cooperative_groups;

constexpr int kFinalThreads = 512;        // two CTAs per SM: one query's ranking overlaps the next one's row gather
constexpr int kMaxKc = 1024;

// grid = (b); one CTA per query.  cand_keys [b, kc], q64 [b, ld], outputs [b, k].
// The fp64 query is staged in shared memory once; every warp re-scores candidates with 16-byte row loads
// (exact_score_row, exact.cuh — the same function the fused single-request kernel uses, so both give the same bits).
template <typename T, bool DIV>
__global__ void __launch_bounds__(kFinalThreads, 2)
finalize_topk_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t row_base, int ld,
                     const double* __restrict__ q64, const uint64_t* __restrict__ cand_keys, int kc, int k,
                     int64_t* __restrict__ out_rows, double* __restrict__ out_scores, int32_t* __restrict__ out_count,
                     double* __restrict__ out_margin, double err_mult) {
    constexpr int EPC = ChunkDot<T>::EPC;
    extern __shared__ __align__(16) double s_q[];   // [ld]
    __shared__ double s_score[kMaxKc];
    __shared__ int64_t s_row[kMaxKc];
    __shared__ unsigned long long s_maxerr;      // bits of a non-negative double: integer order == numeric order
    __shared__ int s_tmp[2];
    __shared__ double s_kth;
    const int u = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    pdl_trigger();
    pdl_wait();                                      // the candidates come from the kernel launched just before
    const uint64_t* keys = cand_keys + (size_t)u * kc;
    stage_query_planes(q64 + (size_t)u * ld, ld, EPC, s_q);
    if (threadIdx.x == 0) { s_maxerr = 0ull; s_tmp[0] = 0; s_tmp[1] = 0; }
    __syncthreads();
    const QueryPlanes qsrc{s_q, ld / EPC};

    for (int c = warp; c < kc; c += nwarps) {
        const uint64_t key = keys[c];
        double sc = -INFINITY;
        int64_t gr = -1;
        if (key != 0) {
            const uint32_t lr = key_row(key);
            sc = exact_score_row<T, DIV>(rows, ld, norm64, lr, qsrc, lane);
            gr = row_base + lr;
        }
        if (lane == 0) {
            s_score[c] = sc;
            s_row[c] = gr;
            if (key != 0) atomicMax(&s_maxerr, (unsigned long long)__double_as_longlong(fabs(sc - (double)key_score(key))));
        }
    }
    __syncthreads();
    // list full => rows outside it have fast score <= key_score(last); the margin compares that against the exact k-th
    // minus 4x the largest fast-vs-exact deviation seen on the candidates themselves, which calibrates whatever
    // rounding the fast pass had (fp32 accumulation, bf16 queries on the tensor-core path)
    const uint64_t last = keys[kc - 1];
    rank_candidates<!DIV>(s_score, s_row, kc, k, last != 0, last ? (double)key_score(last) : 0.0,
                          __longlong_as_double((long long)s_maxerr), out_rows + (size_t)u * k,
                          out_scores + (size_t)u * k, out_count + u, out_margin ? out_margin + u : nullptr, s_tmp, &s_kth, err_mult);
}

// Long lists of the batched path (k > 240, kc <= 4096).  The re-score is finalize_topk_kernel's (exact_score_row<T, false>:
// the same bits); the ranking is a bitonic sort of (orderable fp64 score, local row) pairs in shared memory — kc log^2 kc
// steps instead of rank_candidates' kc x kc count, which at kc = 4096 would be 16 M compares per query.  Results, margin and
// the 4-ulp near-tie rule are those of rank_candidates<true>: in sorted order two distinct scores within 4 ulp of each other
// are adjacent, and the pair counts when the higher score's first position is at or above place k, i.e. ord[k] <= ord[i].
// Dynamic shared memory: [ld] query planes, [p2] keys, [p2] rows (p2 = the power of two >= kc).
__device__ __forceinline__ bool pair_before(unsigned long long ka, uint32_t ra, unsigned long long kb, uint32_t rb) {
    return ka > kb || (ka == kb && ra < rb);
}

template <typename T>
__global__ void __launch_bounds__(kFinalThreads, 2)
finalize_large_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t row_base, int64_t n, int ld,
                      const double* __restrict__ q64, const uint64_t* __restrict__ cand_keys, int kc, int p2, int k,
                      int64_t* __restrict__ out_rows, double* __restrict__ out_scores, int32_t* __restrict__ out_count,
                      double* __restrict__ out_margin, double err_mult) {
    constexpr int EPC = ChunkDot<T>::EPC;
    extern __shared__ __align__(16) double s_q[];
    unsigned long long* s_ord = (unsigned long long*)(s_q + ld);
    uint32_t* s_lr = (uint32_t*)(s_ord + p2);
    __shared__ unsigned long long s_maxerr;
    __shared__ int s_valid, s_near;
    const int u = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    pdl_trigger();
    pdl_wait();                                      // the candidates come from the kernel launched just before
    const uint64_t* keys = cand_keys + (size_t)u * kc;
    stage_query_planes(q64 + (size_t)u * ld, ld, EPC, s_q);
    if (threadIdx.x == 0) { s_maxerr = 0ull; s_valid = 0; s_near = 0; }
    for (int c = kc + threadIdx.x; c < p2; c += blockDim.x) { s_ord[c] = 0ull; s_lr[c] = 0xFFFFFFFFu; }
    __syncthreads();
    const QueryPlanes qsrc{s_q, ld / EPC};
    for (int c = warp; c < kc; c += nwarps) {
        const uint64_t key = keys[c];
        unsigned long long ord = 0ull;
        uint32_t lr = 0xFFFFFFFFu;
        if (key != 0) {
            lr = key_row(key);
            REBERT_ASSERT((int64_t)lr < n);
            const double sc = exact_score_row<T, false>(rows, ld, norm64, lr, qsrc, lane);
            ord = f64_orderable(sc);
            if (lane == 0) atomicMax(&s_maxerr, (unsigned long long)__double_as_longlong(fabs(sc - (double)key_score(key))));
        }
        if (lane == 0) {
            REBERT_ASSERT(c < p2);
            s_ord[c] = ord;
            s_lr[c] = lr;
        }
    }
    __syncthreads();
    for (int w = 2; w <= p2; w <<= 1) {
        for (int j = w >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < p2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long x = s_ord[i], y = s_ord[ixj];
                    const uint32_t rx = s_lr[i], ry = s_lr[ixj];
                    const bool desc = (i & w) == 0;
                    if (desc ? pair_before(y, ry, x, rx) : pair_before(x, rx, y, ry)) {
                        s_ord[i] = y; s_ord[ixj] = x;
                        s_lr[i] = ry; s_lr[ixj] = rx;
                    }
                }
            }
            __syncthreads();
        }
    }
    const unsigned long long ord_k = s_ord[k];       // k < kc <= p2; 0 when fewer than k + 1 candidates are valid
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        const unsigned long long a = s_ord[i];
        if (a == 0ull) continue;
        const unsigned long long nb = i + 1 < p2 ? s_ord[i + 1] : 0ull;
        if (nb == 0ull) s_valid = i + 1;             // the last valid entry: exactly one thread
        else if (a != nb && a - nb <= 4ull && ord_k <= a) s_near = 1;
    }
    __syncthreads();
    const int valid = s_valid;
    const int nout = valid < k ? valid : k;
    int64_t* o_rows = out_rows + (size_t)u * k;
    double* o_scores = out_scores + (size_t)u * k;
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        REBERT_ASSERT(i < p2);
        o_rows[i] = i < nout ? row_base + s_lr[i] : -1;
        o_scores[i] = i < nout ? f64_from_orderable(s_ord[i]) : -INFINITY;
    }
    if (threadIdx.x == 0) {
        out_count[u] = nout;
        if (out_margin) {
            const uint64_t last = keys[kc - 1];
            double mg = (last != 0 && valid >= k) ? f64_from_orderable(s_ord[k - 1]) - (double)key_score(last) -
                                                        err_mult * __longlong_as_double((long long)s_maxerr)
                                                  : INFINITY;
            if (s_near) mg = -INFINITY;
            out_margin[u] = mg;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Request path, second (and last) launch: a CLUSTER of 8 CTAs placed behind the streaming kernel by programmatic dependent
// launch.  The streaming kernel's CTAs have published their pruned candidate keys (gemv_topk.cu); here
//   (1) the kc winners are selected from them: short lists (kc < 128) by every CTA redundantly — <= 38 KB of keys, one round of
//       loads, cheaper than any cross-CTA step —, long lists by the cluster together (select_winners_cluster, merge.cuh),
//   (2) the winners are dealt out over the 8 x 8 warps of the cluster for the fp64 exact pass — one row per warp, on 8 SMs,
//       instead of a queue of rows behind one SM's fp64 unit — and each warp stores its score straight into CTA 0's shared
//       memory (distributed shared memory),
//   (3) CTA 0 ranks by (score desc, row asc), writes the packed result (device or pinned host memory) and, on a row shard,
//       runs the NVLink exchange + merge; it leaves the streaming kernel's control words zero for the next request.
// 256 threads, <= 128 registers and ~30 KB of shared memory per CTA: small enough to be resident beside the streaming
// kernel's CTAs, so the cluster is already waiting in griddepcontrol.wait when the stream ends.
// ---------------------------------------------------------------------------------------------------------
constexpr int kFinalCluster = 8;
constexpr int kFinalClusterThreads = 256;

struct FinalizeParams {
    Published pub;
    const void* x_rows;
    const double* x_norm64;
    const double* q64;
    int x_ld, x_dtype;
    int64_t row_base, x_n;
    int k, cap;
    int stage_words;           // words from fk on that are free until the winners are known: max(3 kc, heads of every list)
    unsigned long long* out_packed;
    uint32_t tag;
    uint32_t* done_flag;       // pinned host word the host polls instead of synchronising the stream (or nullptr)
    uint32_t done_token;
    Exchange xchg;
};

// SPLIT: winner selection spread over the cluster (kc >= 128, long candidate lists); XCHG: row shard, NVLink exchange + merge at the end.
// Eight instantiations (with the element type) instead of run-time branches: this kernel runs once per request with a cold instruction cache, and
// every variant it does not need (each one thousands of unrolled instructions) would sit between the ones it does.
// T: element type of the catalog of record — the exact pass carries one row function instead of both.
template <int SPLIT, bool XCHG, typename T>
__global__ void __launch_bounds__(kFinalClusterThreads, 2) finalize_published_kernel(const FinalizeParams p) {
    extern __shared__ __align__(16) unsigned char fsm[];
    const int kc = p.pub.keys.kc, k = p.k;
    double* s_q = (double*)fsm;                                        // [x_ld] fp64 query, pair planes
    uint64_t* buf = (uint64_t*)(s_q + p.x_ld);                         // [cap]
    uint64_t* fk = buf + p.cap;                                        // [kc] winners, best fast score first
    double* s_score = (double*)(fk + kc);                              // [kc]   (filled remotely in CTA 0)
    int64_t* s_row = (int64_t*)(s_score + kc);                         // [kc]
    unsigned long long* s_werr = (unsigned long long*)(fk + p.stage_words);   // [cluster warps] largest |fast - exact| per warp
    unsigned long long* s_block = s_werr + kFinalCluster * (kFinalClusterThreads / 32);   // [2 k + 2] local result (row shards)
    unsigned long long* s_all = s_block + 2 * k + 2;                   // [world][2 k + 2] every rank's result (row shards)
    __shared__ int s_tmp[2];
    __shared__ int s_total;                          // survivors pushed into this CTA's buf (select_winners_cluster)
    __shared__ double s_kth;
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = kFinalClusterThreads / 32;
    // Programmatic dependent launch lets the NEXT kernel of the stream place its CTAs early.  A kernel that will wait for
    // a PEER must not do that before the wait is over: the next request's streaming CTAs would sit resident on every SM,
    // blocked behind this kernel, while the peer — in the mirrored state on another channel — needs exactly those SMs to
    // produce what this kernel waits for (deadlock across ranks with concurrent channels).  So on a row shard the trigger
    // comes after the exchange.
    constexpr bool exchange = XCHG;
    if (!exchange) pdl_trigger();
    if (threadIdx.x == 0) { s_tmp[0] = 0; s_tmp[1] = 0; s_total = 0; }
    cluster.sync();                                  // every CTA of the cluster is running: its shared memory may be addressed.
                                                     // Done HERE, while the stream is still running, it costs nothing.
    pdl_wait();                                      // the keys come from the streaming kernel launched just before
    // (Waiting on the CTAs' publish counter instead would start 1-3 us earlier, but a cluster placed early by programmatic
    // launch could then mistake the PREVIOUS request's count for its own; stream order is the simple, safe hand-off.)
    constexpr int epc = ChunkDot<T>::EPC;
    // the fp64 query: its loads are issued here, ahead of the ones select_winners issues, and consumed only afterwards —
    // one L2 round trip for everything this kernel reads before the candidate rows
    constexpr int kQPre = 8;
    double qv[kQPre];
#pragma unroll
    for (int j = 0; j < kQPre; ++j) {
        const int i = threadIdx.x + j * kFinalClusterThreads;
        qv[j] = i < p.x_ld ? __ldg(p.q64 + i) : 0.0;
    }
    if (SPLIT)     // fk | s_score | s_row = 3 kc words that are free until the winners are known
        select_winners_cluster<kFinalCluster, kFinalClusterThreads>(cluster, p.pub.keys, p.cap, buf, fk, p.stage_words, fk, &s_total);
    else
        select_winners<24, kFinalClusterThreads>(p.pub.keys, p.cap, buf, fk);
    {
        const int chunks = p.x_ld / epc;
#pragma unroll
        for (int j = 0; j < kQPre; ++j) {
            const int i = threadIdx.x + j * kFinalClusterThreads;
            if (i < p.x_ld) {
                const int ch = i / epc, e = i - ch * epc;
                s_q[((size_t)(e >> 1) * chunks + ch) * 2 + (e & 1)] = qv[j];
            }
        }
        for (int i = kQPre * kFinalClusterThreads + threadIdx.x; i < p.x_ld; i += kFinalClusterThreads) {   // rows beyond 2048 elements
            const int ch = i / epc, e = i - ch * epc;
            s_q[((size_t)(e >> 1) * chunks + ch) * 2 + (e & 1)] = __ldg(p.q64 + i);
        }
    }
    __syncthreads();
    double* r_score = cluster.map_shared_rank(s_score, 0);
    int64_t* r_row = cluster.map_shared_rank(s_row, 0);
    unsigned long long* r_werr = cluster.map_shared_rank(s_werr, 0);
    const QueryPlanes qsrc{s_q, p.x_ld / epc};
    double werr = 0.0;
    for (int c = crank * nwarps + warp; c < kc; c += kFinalCluster * nwarps) {
        const uint64_t key = fk[c];
        double sc = -INFINITY;
        int64_t gr = -1;
        if (key != 0) {
            const uint32_t lr = key_row(key);
            REBERT_ASSERT((int64_t)lr < p.x_n && c < kc);
            sc = exact_score_row<T, true>((const T*)p.x_rows, p.x_ld, p.x_norm64, lr, qsrc, lane);
            gr = p.row_base + lr;
            werr = fmax(werr, fabs(sc - (double)key_score(key)));
        }
        if (lane == 0) { r_score[c] = sc; r_row[c] = gr; }
    }
    if (lane == 0) r_werr[crank * nwarps + warp] = (unsigned long long)__double_as_longlong(werr);
    cluster.sync();                                  // all scores have landed in CTA 0
    if (crank != 0) return;
    unsigned long long me = 0;                       // bits of non-negative doubles: integer order == numeric order
    for (int i = lane; i < kFinalCluster * nwarps; i += 32) me = s_werr[i] > me ? s_werr[i] : me;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, me, o); me = v > me ? v : me; }
    const uint64_t last = fk[kc - 1];
    unsigned long long* blk = exchange ? s_block : p.out_packed;
    rank_candidates<false>(s_score, s_row, kc, k, last != 0, last ? (double)key_score(last) : 0.0, __longlong_as_double((long long)me),
                           (int64_t*)blk, (double*)(blk + k), (int32_t*)(blk + 2 * k), (double*)(blk + 2 * k + 1), s_tmp, &s_kth);
    if (threadIdx.x == 0) ((uint32_t*)(blk + 2 * k))[1] = p.tag;
    if (exchange) {
        __syncthreads();
        exchange_results(p.xchg, k, s_block, p.out_packed, s_all);
        pdl_trigger();
    }
    if (threadIdx.x < 32 && !ctl_survives_merge(threadIdx.x)) p.pub.ctl[threadIdx.x] = 0u;   // ticket, hint, tile claims, cursors
    if (p.done_flag) {
        __syncthreads();                                     // every thread's result stores are ordered before the flag
        if (threadIdx.x == 0) {
            __threadfence_system();
            *(volatile uint32_t*)p.done_flag = p.done_token;
        }
    }
}

using PublishedKernel = void (*)(const FinalizeParams);
template <typename T>
static PublishedKernel published_kernel(bool split, bool xchg) {
    return split ? (xchg ? finalize_published_kernel<1, true, T> : finalize_published_kernel<1, false, T>)
                 : (xchg ? finalize_published_kernel<0, true, T> : finalize_published_kernel<0, false, T>);
}

int finalize_published_launch(const Published& pub, const GemvFused& f, int64_t row_base, cudaStream_t st) {
    FinalizeParams p;
    memset(&p, 0, sizeof(p));
    p.pub = pub;
    p.x_rows = f.exact_cat->rows;
    p.x_norm64 = f.exact_cat->norm64;
    p.q64 = f.q64;
    p.x_ld = f.exact_cat->ld;
    p.x_dtype = f.exact_cat->dtype;
    p.row_base = row_base;
    p.x_n = f.exact_cat->n;
    p.k = f.k;
    int need = 2 * pub.keys.kc > pub.keys.kc + pub.keys.lists ? 2 * pub.keys.kc : pub.keys.kc + pub.keys.lists;
    int cap = 1024;
    while (cap < need) cap <<= 1;
    p.cap = cap;
    // Long candidate lists (kc >= 128: k > 16, the int8 shadow, a widened retry) publish tens of thousands of keys: the cluster
    // shares the scan and the ordering (merge.cuh).  Short lists fit one round of loads per CTA and skip the two extra
    // cluster barriers.
    const bool split = pub.keys.kc >= 128;
    p.stage_words = 3 * pub.keys.kc > pub.keys.kc + pub.keys.lists ? 3 * pub.keys.kc : pub.keys.kc + pub.keys.lists;
    p.out_packed = f.out_packed;
    p.tag = f.tag;
    p.done_flag = f.done_flag;
    p.done_token = f.done_token;
    if (f.xchg) p.xchg = *f.xchg;
    const size_t smem = (size_t)p.x_ld * 8 + (size_t)cap * 8 + (size_t)p.stage_words * 8 + (size_t)kFinalCluster * (kFinalClusterThreads / 32) * 8 +
                        (size_t)(2 * f.k + 2) * 8 * (1 + (f.xchg ? f.xchg->world : 0));
    const bool xchg = p.xchg.world > 1;
    const PublishedKernel kern =
        p.x_dtype == REBERT_F32 ? published_kernel<float>(split, xchg) : published_kernel<__nv_bfloat16>(split, xchg);
    { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(kFinalCluster);
    cfg.blockDim = dim3(kFinalClusterThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kFinalCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    REBERT_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

// One CTA per query: rank-merge `lists` sorted lists of up to k entries each.  List l of query u lives at
// rows[l * rows_stride + u * k + e], scores[l * scores_stride + u * k + e], counts[l * counts_stride + u]
// (strides in elements), which covers both a dense [lists, b, k] layout and the packed per-rank buffers an
// all-gather produces.
__global__ void merge_topk_kernel(const int64_t* __restrict__ rows, const double* __restrict__ scores,
                                  const int32_t* __restrict__ counts, int64_t rows_stride, int64_t scores_stride,
                                  int64_t counts_stride, int lists, int k, int64_t* __restrict__ out_rows,
                                  double* __restrict__ out_scores, int32_t* __restrict__ out_count) {
    const int u = blockIdx.x;
    int total = 0;
    for (int l = 0; l < lists; ++l) total += min(counts[l * counts_stride + u], k);
    const int nout = total < k ? total : k;
    for (int i = threadIdx.x; i < lists * k; i += blockDim.x) {
        const int l = i / k, e = i - l * k;
        if (e >= counts[l * counts_stride + u]) continue;
        const double sc = scores[l * scores_stride + (int64_t)u * k + e];
        const int64_t r = rows[l * rows_stride + (int64_t)u * k + e];
        int rank = e;
        for (int o = 0; o < lists; ++o) {
            if (o == l) continue;
            const int64_t* orow = rows + o * rows_stride + (int64_t)u * k;
            const double* osc = scores + o * scores_stride + (int64_t)u * k;
            int lo = 0, hi = min(counts[o * counts_stride + u], k);      // entries of list o better than (sc, r)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (better(osc[mid], orow[mid], sc, r)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < k) {
            out_rows[(size_t)u * k + rank] = r;
            out_scores[(size_t)u * k + rank] = sc;
        }
    }
    for (int i = nout + threadIdx.x; i < k; i += blockDim.x) {
        out_rows[(size_t)u * k + i] = -1;
        out_scores[(size_t)u * k + i] = -INFINITY;
    }
    if (threadIdx.x == 0) out_count[u] = nout;
}


// Stand-alone forms of the two exchange steps (exchange.cuh).  The single-request kernel runs the result exchange in its
// own tail (gemv_topk.cu); these kernels serve callers that hold a packed local result / a partial profile already.
__global__ void __launch_bounds__(256) exchange_merge_kernel(Exchange x, int k, const unsigned long long* __restrict__ local,
                                                             unsigned long long* __restrict__ out) {
    extern __shared__ __align__(16) unsigned long long s_xall[];    // [world][2 k + 2]
    pdl_wait();                                      // `local` is written by the kernel launched just before
    exchange_results(x, k, local, out, s_xall);
    pdl_trigger();                                   // only now: see finalize_published_kernel
}

// sum64 [ld] partial -> exchanged, summed in rank order, divided by wsum: p32 / p64 (profile_finalize fused in).
__global__ void __launch_bounds__(256) profile_exchange_kernel(Exchange x, int ld, double* __restrict__ sum64, const double* __restrict__ wsum,
                                                               float* __restrict__ p32, double* __restrict__ p64) {
    pdl_wait();
    exchange_profile(x, ld, sum64, sum64);           // every element is read (pushed) before the barrier inside, written after it
    pdl_trigger();                                   // only now: see finalize_published_kernel
    __syncthreads();
    const double ws = wsum[0];
    for (int c = threadIdx.x; c < ld; c += blockDim.x) {
        const double v = ws != 0.0 ? sum64[c] / ws : 0.0;
        p64[c] = v;
        p32[c] = (float)v;
    }
}

int make_exchange(const rebert_exchange_t* ex, int32_t* err_flag, Exchange* out) {
    REBERT_REQUIRE(ex && ex->peer_buffers && err_flag, "exchange: null argument");
    REBERT_REQUIRE(ex->world > 0 && ex->world <= kMaxPeers && ex->rank >= 0 && ex->rank < ex->world, "exchange: world=%d rank=%d",
                   ex->world, ex->rank);
    REBERT_REQUIRE(ex->k_max > 0 && ex->prof_len >= 0 && ex->channels > 0 && ex->channel >= 0 && ex->channel < ex->channels && ex->seq != 0,
                   "exchange: k_max=%d prof_len=%d channel=%d/%d seq=%u", ex->k_max, ex->prof_len, ex->channel, ex->channels, ex->seq);
    memset(out, 0, sizeof(*out));
    out->world = ex->world;
    out->rank = ex->rank;
    out->words_cap = 2 * ex->k_max + 2;
    out->prof_cap = ex->prof_len + 1;
    out->seq = ex->seq;
    // ~10 s of SM clocks at 2 GHz: only a dead peer gets here.  (A constant: querying the clock rate is a slow driver
    // call and this function sits on the per-request path.)  REBERT_EXCHANGE_TIMEOUT_MS overrides it (read once; tests).
    static const long long timeout_cycles = [] {
        const char* e = getenv("REBERT_EXCHANGE_TIMEOUT_MS");
        const long long ms = e ? atoll(e) : 0;
        return ms > 0 ? ms * 2000000ll : 20000000000ll;
    }();
    out->timeout_cycles = timeout_cycles;
    out->err = err_flag;
    const size_t ch_words = xchg_channel_words(ex->world, out->words_cap, out->prof_cap);
    for (int i = 0; i < ex->world; ++i)
        out->peer[i] = (unsigned long long*)(uintptr_t)ex->peer_buffers[i] + (size_t)ex->channel * ch_words;
    return REBERT_OK;
}

template <typename T, bool DIV>
static int finalize_launch_t(const rebert_catalog_t* cat, const double* q64, const uint64_t* cand_keys, int b, int kc, int k,
                             int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin, cudaStream_t st, double err_mult) {
    const size_t smem = (size_t)cat->ld * sizeof(double);
    auto kern = finalize_topk_kernel<T, DIV>;
    { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
    REBERT_CUDA(launch_pdl(kern, dim3(b), dim3(kFinalThreads), smem, st, (const T*)cat->rows, cat->norm64, cat->row_base, cat->ld, q64,
                           cand_keys, kc, k, out_rows, out_scores, out_count, out_margin, err_mult));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

// exact_order = true: sklearn's operation order (element-wise division first) — the single-request path.
// exact_order = false: one division after the dot (within 1 ulp), near-ties flagged through the margin — the batched path.
int finalize_launch(const rebert_catalog_t* cat, const double* q64, const uint64_t* cand_keys, int b, int kc, int k,
                    int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin, cudaStream_t st,
                    bool exact_order, double err_mult = 4.0) {
    if (cat->dtype == REBERT_F32)
        return exact_order ? finalize_launch_t<float, true>(cat, q64, cand_keys, b, kc, k, out_rows, out_scores, out_count, out_margin, st, err_mult)
                           : finalize_launch_t<float, false>(cat, q64, cand_keys, b, kc, k, out_rows, out_scores, out_count, out_margin, st, err_mult);
    return exact_order ? finalize_launch_t<__nv_bfloat16, true>(cat, q64, cand_keys, b, kc, k, out_rows, out_scores, out_count, out_margin, st, err_mult)
                       : finalize_launch_t<__nv_bfloat16, false>(cat, q64, cand_keys, b, kc, k, out_rows, out_scores, out_count, out_margin, st, err_mult);
}

// Exact pass of the batched path's long lists (finalize_large_kernel): divide-after formula, near-ties flagged via the margin.
int finalize_large_launch(const rebert_catalog_t* cat, const double* q64, const uint64_t* cand_keys, int b, int kc, int k,
                          int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin, cudaStream_t st, double err_mult) {
    REBERT_REQUIRE(kc > 0 && k > 0 && k < kc, "finalize_large: k=%d kc=%d", k, kc);
    int p2 = 2;
    while (p2 < kc) p2 <<= 1;
    const size_t smem = (size_t)cat->ld * sizeof(double) + (size_t)p2 * (sizeof(unsigned long long) + sizeof(uint32_t));
    if (cat->dtype == REBERT_F32) {
        auto kern = finalize_large_kernel<float>;
        { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
        REBERT_CUDA(launch_pdl(kern, dim3(b), dim3(kFinalThreads), smem, st, (const float*)cat->rows, cat->norm64, cat->row_base, cat->n,
                               cat->ld, q64, cand_keys, kc, p2, k, out_rows, out_scores, out_count, out_margin, err_mult));
    } else {
        auto kern = finalize_large_kernel<__nv_bfloat16>;
        { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
        REBERT_CUDA(launch_pdl(kern, dim3(b), dim3(kFinalThreads), smem, st, (const __nv_bfloat16*)cat->rows, cat->norm64, cat->row_base,
                               cat->n, cat->ld, q64, cand_keys, kc, p2, k, out_rows, out_scores, out_count, out_margin, err_mult));
    }
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

}  // namespace rebert

using namespace rebert;

extern "C" {

REBERT_API int rebert_finalize_topk(const rebert_catalog_t* cat, const double* qn64, const uint64_t* cand_keys, int32_t kc,
                         int32_t k, int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin,
                         rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && cat->norm64 && qn64 && cand_keys && out_rows && out_scores && out_count,
                   "finalize_topk: null argument");
    REBERT_REQUIRE(kc > 0 && kc <= kMaxKc && k > 0 && k <= kc, "finalize_topk: k=%d kc=%d", k, kc);
    return finalize_launch(cat, qn64, cand_keys, 1, kc, k, out_rows, out_scores, out_count, out_margin,
                           (cudaStream_t)stream, /*exact_order=*/true);
}

REBERT_API int rebert_merge_topk(const int64_t* rows, const double* scores, const int32_t* counts, int64_t rows_stride,
                      int64_t scores_stride, int64_t counts_stride, int32_t lists, int32_t b, int32_t k,
                      int64_t* out_rows, double* out_scores, int32_t* out_count, rebert_stream stream) {
    REBERT_REQUIRE(rows && scores && counts && out_rows && out_scores && out_count, "merge_topk: null argument");
    REBERT_REQUIRE(lists > 0 && b > 0 && k > 0, "merge_topk: lists=%d b=%d k=%d", lists, b, k);
    merge_topk_kernel<<<b, 256, 0, (cudaStream_t)stream>>>(rows, scores, counts, rows_stride, scores_stride, counts_stride,
                                                           lists, k, out_rows, out_scores, out_count);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API size_t rebert_exchange_buffer_bytes(int32_t world, int32_t k_max, int32_t prof_len, int32_t channels) {
    if (world <= 0 || world > kMaxPeers || k_max <= 0 || prof_len < 0 || channels <= 0) return 0;
    return xchg_channel_words(world, 2 * k_max + 2, prof_len + 1) * 8 * (size_t)channels;
}

REBERT_API int rebert_exchange_merge(const rebert_exchange_t* ex, int32_t k, const int64_t* local_packed, int64_t* out_packed,
                                     int32_t* err_flag, rebert_stream stream) {
    REBERT_REQUIRE(local_packed && out_packed, "exchange_merge: null argument");
    Exchange x;
    int rc = make_exchange(ex, err_flag, &x);
    if (rc != REBERT_OK) return rc;
    REBERT_REQUIRE(k > 0 && k <= ex->k_max, "exchange_merge: k=%d k_max=%d", k, ex->k_max);
    REBERT_CUDA(launch_pdl(exchange_merge_kernel, dim3(1), dim3(256), (size_t)ex->world * (2 * k + 2) * 8, (cudaStream_t)stream, x, k,
                           (const unsigned long long*)local_packed, (unsigned long long*)out_packed));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_profile_exchange(const rebert_exchange_t* ex, int32_t ld, double* sum64, const double* wsum, float* p32,
                                       double* p64, int32_t* err_flag, rebert_stream stream) {
    REBERT_REQUIRE(sum64 && wsum && p32 && p64 && ld > 0, "profile_exchange: bad arguments");
    Exchange x;
    int rc = make_exchange(ex, err_flag, &x);
    if (rc != REBERT_OK) return rc;
    REBERT_REQUIRE(ld <= ex->prof_len, "profile_exchange: ld=%d exceeds the buffer's prof_len=%d", ld, ex->prof_len);
    REBERT_CUDA(launch_pdl(profile_exchange_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, x, ld, sum64, wsum, p32, p64));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

}  // extern "C"
