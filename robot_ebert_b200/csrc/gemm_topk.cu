// Batched queries on the 5th-gen tensor cores  (reference: lib.py:51-55 for many users at once).
//
// scores[q, j] = <Q[q, :], rows[j, :]> * inv_norm[j]  is a genuine dense contraction (B x N x D), so it runs as a
// bf16 tcgen05 GEMM with fp32 accumulators in TMEM; the B x N score matrix is NEVER written.  Pipeline of
// rebert_gemm_topk (everything enqueued on the caller's stream):
//
//   1. gemm<STORE>  over a strided SAMPLE of row tiles  -> sample scores [B, S]            (~1.5 % of the flops)
//   2. select_threshold: per query, knock out excluded / predicate-filtered sample rows, take the 16-th largest
//      (thread-maxima pruning, radix select as fallback) -> tau[q]: a lower bound of the query's k-th best that leaves
//      ~max(8 kc, 1024) rows above it in expectation
//   3. gemm<FILTER> over ALL row tiles: the epilogue scales by inv_norm (NaN for rows the batch predicate drops), compares
//      a whole 32-column chunk with tau[q] through a max tree (one compare per chunk), stages the rare winners in smem
//      and appends (score,row) keys to cand[q] with one atomicAdd per thread per tile
//   4. select_candidates: per query, drop excluded rows, bucket-select + small bitonic sort -> best kc keys
//   5. finalize_topk (csrc/finalize.cu): fp64 re-score, (score desc, row asc), best k, proof margin
//   Long lists (241 <= k <= 2048, kc up to 4096) use sample rank 64 with ~3 kc survivors, and their own stages 4 and 5:
//   select_candidates_large (histogram over the global buffer, gather + sort) and finalize_large (bitonic ranking).
//   status[q] != 0 tells the caller to re-run that query through the single-query kernel (threshold too optimistic,
//   staging / buffer overflow, margin below eps or a sub-4-ulp gap) — exactness never depends on the sample being lucky.
//
// Two GEMM kernels share the epilogue (epilogue_tile):
//   gemm2_kernel (B > 128, the normal case): cluster of 2 CTAs = one SM pair per 256-query x 256-row tile,
//     tcgen05.mma.cta_group::2 M=256 N=256 K=16, each CTA stages its 128-query half of A and its 128-row half of B
//     (32 KB / stage, 6 stages) with cp.async.bulk.tensor.2d.cta_group::2 completing on the leader's mbarrier; commits
//     are multicast to both CTAs; the peer's epilogue releases the accumulator with a remote mbarrier.arrive.
//   gemm_kernel (B <= 128): one CTA per SM, cta_group::1 M=128 N=256, 4 stages of 48 KB.
//   Both: 192 threads = warp 0 TMA producer (one lane), warp 1 MMA issuer (one lane) + TMEM allocator, warps 2-5
//   epilogue (thread = query row; tcgen05.ld 32x32b.x32 software-pipelined against the previous chunk's math);
//   fp32 accumulators double-buffered in TMEM (2 x 256 columns); K-major SWIZZLE_128B smem descriptors.
//   Tile order is row-tile-major so the CTAs of a wave share catalog tiles in L2 (the catalog streams from HBM about
//   once) and Q (12.6 MB at B = 4096) stays L2-resident (evict_last).
//   Measured (profiles/r01_gemm2_filter_1M_ncu_summary.md): tensor pipe 97 % active, 1607 TFLOP/s.
#include <cuda.h>

#include "common.cuh"

namespace rebert {

int finalize_launch(const rebert_catalog_t* cat, const double* q64, const uint64_t* cand_keys, int b, int kc, int k,
                    int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin, cudaStream_t st,
                    bool exact_order, double err_mult = 4.0);
int finalize_large_launch(const rebert_catalog_t* cat, const double* q64, const uint64_t* cand_keys, int b, int kc, int k,
                          int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin, cudaStream_t st, double err_mult);

constexpr int BM = 128, BN = 256, BK = 64, UK = 16;
constexpr int GEMM_STAGES = 4;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int EPI_WARPS = 4, GEMM_THREADS = 32 * (2 + EPI_WARPS);
constexpr int STAGE_SLOTS = 24;                                 // per-thread staged candidates per tile
constexpr int SMEM_STAGING = STAGE_SLOTS * 128 * 8;
constexpr int SMEM_INV = 2 * BN * 4;
constexpr int GEMM_SMEM = GEMM_STAGES * STAGE_BYTES + SMEM_STAGING + SMEM_INV + 256 + 1024;   // + alignment slack
// per-query filters only: the tile's genre_bits [2][BN] and year [2][BN], behind the barriers (227,584 B of 232,448 B in all)
constexpr int SMEM_QF = 2 * BN * 4 + 2 * BN * 2;
constexpr uint32_t TMEM_COLS = 512;
// k above kLargeK0 (the single-query kernel's limit) takes the long-list stages; kLargeKMax bounds kc at 4096 (int8 plans)
constexpr int kLargeK0 = 240, kLargeKMax = 2048, kLargeRank = 64, kLargeKcMax = 4096;

enum { MODE_STORE = 0, MODE_FILTER = 1 };

// Per-query genre / year predicate of a batch (rebert_query_filter_t).  A null pair switches that test off for every query.
struct QueryFilter {
    const uint32_t* genre_bits;   // [n] local
    const uint16_t* year;         // [n] local
    const uint32_t* genre_any;    // [b]
    const uint16_t* year_lo;      // [b]
    const uint16_t* year_hi;      // [b]
};
// One query's test: keep a row iff (genre_any == 0 or genre_bits & genre_any) and year_lo <= year <= year_hi
struct QueryTest { uint32_t genre_any, year_lo, year_hi; };
__device__ __forceinline__ QueryTest load_query_test(const QueryFilter& f, int q) {
    QueryTest t{0u, 0u, 0xFFFFu};
    if (f.genre_any) t.genre_any = __ldg(f.genre_any + q);
    if (f.year_lo) { t.year_lo = __ldg(f.year_lo + q); t.year_hi = __ldg(f.year_hi + q); }
    return t;
}
__device__ __forceinline__ bool query_allows(const QueryTest& t, uint32_t genre_bits, uint32_t year) {
    return (t.genre_any == 0u || (genre_bits & t.genre_any) != 0u) && year >= t.year_lo && year <= t.year_hi;
}

struct GemmParams {
    int b;                  // queries
    int num_qt;             // query tiles (ceil(b / 128))
    int num_rt;             // row tiles in this launch
    int64_t tile0;          // first global row tile
    int64_t tile_stride;    // global row-tile stride between consecutive launch tiles (1 = contiguous)
    int64_t n;              // shard rows
    int kblocks;            // ld / 64
    const float* inv_norm;
    DevFilter pred;         // per-row predicate (bitmap / genre / year); n_exclude is always 0 here
    int has_pred;
    // MODE_STORE
    float* out;             // [b, out_ld], column = launch tile index * 256 + c
    int64_t out_ld;
    // MODE_FILTER
    const float* qscale;    // [b] int8 operand path: dequantisation step of query q (scores = acc * factor[row] * qscale[q]); else nullptr
    const float* tau;       // [b]
    uint64_t* cand;         // [b, cand_cap]
    unsigned* cand_count;   // [b]
    int cand_cap;
    int* status;            // [b]
    QueryFilter qf;         // MODE_FILTER with the QF template flag: per-query genre / year tests
};

// ---------------------------------------------------------------- PTX wrappers ------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accum)
        : "memory");
}
// int8 operands, int32 accumulators (sm_100a has kind::i8 at twice the bf16 rate; the shadow catalog of the prefilter supplies the rows)
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in
// bits [0,14), LBO unused for swizzled K-major (0), SBO = 1024 B (8 rows x 128 B) >> 4 in bits [32,46),
// version 1 in bits [46,48), layout SWIZZLE_128B (2) in bits [61,64).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (1<<4), A=B=bf16 (1<<7, 1<<10), both K-major,
// N>>3 at bit 17, M>>4 at bit 24.
constexpr uint32_t kInstrDesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
// kind::i8: D = s32 (2 << 4), A = B = signed 8 bit (1 << 7, 1 << 10), both K-major, K = 32 per instruction
constexpr uint32_t kInstrDescI8 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// ---------------------------------------------------------------------------------------------------------
// Epilogue of one 128 x 256 accumulator (shared by the 1-CTA and 2-CTA kernels).  Thread = one query row.
// Per 32-column chunk: tcgen05.ld (software-pipelined against the previous chunk's math), 8 x LDS.128 of inv_norm,
// 32 independent FMULs, a max tree and ONE compare against the query's threshold; only a chunk that holds a winner
// (2.5 % of thread-chunks) builds the pass mask and stages keys.  No per-element branches, no per-element LDS.
// ---------------------------------------------------------------------------------------------------------
// I8: the accumulators are int32 (kind::i8) and a score is acc * factor[row] * qs, qs = the query's dequantisation step.  The
// filter compares acc * factor[row] against tau / qs (the caller passes that as `tau`), so the hot loop gains one I2F per
// element and nothing else; only stored samples and staged winners are multiplied by qs.
template <bool I8> __device__ __forceinline__ float acc_f32(uint32_t v) { return I8 ? __int2float_rn((int)v) : __uint_as_float(v); }
// (Tried and measured slower, same box: replacing the I2FP — it issues on the XU pipe, which ncu showed 88 % busy — by an integer add
// onto the bit pattern of 1.5 * 2^23 plus an FADD, which run on the main pipes: 7.44 vs 7.21 ms at 4096 x 1M.  The kernel sits at the
// board's power limit, where two instructions on the main pipes cost more than one on an idle pipe saves.  DESIGN.md 4.3.)

// QF (per-query filters): the rare path drops each winner the query's own genre / year test rejects before it is staged or
// counted; the tile's genre_bits / year sit in shared memory (gb_chunk / yr_chunk), so the test is two LDS per winner.
template <int MODE, bool I8, bool QF>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, const uint32_t* v, const float* inv_chunk, float tau, float qs, int q,
                                               float* out_row, uint32_t row_chunk0, uint64_t* staging, int et, int& cnt,
                                               const uint32_t* gb_chunk, const uint16_t* yr_chunk, const QueryTest& qt) {
    float s[32];
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
        const float4 iv = ((const float4*)inv_chunk)[c4];
        s[c4 * 4 + 0] = acc_f32<I8>(v[c4 * 4 + 0]) * iv.x;
        s[c4 * 4 + 1] = acc_f32<I8>(v[c4 * 4 + 1]) * iv.y;
        s[c4 * 4 + 2] = acc_f32<I8>(v[c4 * 4 + 2]) * iv.z;
        s[c4 * 4 + 3] = acc_f32<I8>(v[c4 * 4 + 3]) * iv.w;
    }
    if (MODE == MODE_STORE) {
        if (q < p.b) {
#pragma unroll
            for (int c = 0; c < 32; c += 4)
                *(float4*)(out_row + c) = I8 ? make_float4(s[c] * qs, s[c + 1] * qs, s[c + 2] * qs, s[c + 3] * qs)
                                             : make_float4(s[c], s[c + 1], s[c + 2], s[c + 3]);
        }
    } else {
        float m[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) m[i] = fmaxf(s[2 * i], s[2 * i + 1]);       // fmaxf drops NaN (padding rows)
#pragma unroll
        for (int w = 8; w > 0; w >>= 1)
#pragma unroll
            for (int i = 0; i < w; ++i) m[i] = fmaxf(m[i], m[i + w]);
        if (m[0] > tau) {                                                       // rare: this chunk holds a candidate
            uint32_t mask = 0;
#pragma unroll
            for (int c = 0; c < 32; ++c) mask |= (s[c] > tau) ? (1u << c) : 0u;
            while (mask) {
                const int c = __ffs(mask) - 1;
                mask &= mask - 1;
                if (QF && !query_allows(qt, gb_chunk[c], yr_chunk[c])) continue;
                float val = s[0];
#pragma unroll
                for (int j = 1; j < 32; ++j) val = (c == j) ? s[j] : val;       // register select, no local memory
                REBERT_ASSERT(et >= 0 && et < 128 && (int64_t)(row_chunk0 + (uint32_t)c) < p.n);
                if (cnt < STAGE_SLOTS) staging[cnt * 128 + et] = make_key(I8 ? val * qs : val, row_chunk0 + (uint32_t)c);
                ++cnt;
            }
        }
    }
}

template <int MODE, bool I8, bool QF>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, uint32_t taddr, const float* inv, float tau, float qs, int q, int64_t row0,
                                              int64_t rt, uint64_t* staging, int et, int& cnt, const uint32_t* gb, const uint16_t* yr,
                                              const QueryTest& qt) {
    float* out_row = nullptr;
    if (MODE == MODE_STORE) out_row = p.out + (int64_t)q * p.out_ld + rt * BN;
    uint32_t va[32], vb[32];
    tc_ld32(taddr, va);
    tc_wait_ld();
#pragma unroll
    for (int ch = 0; ch < BN / 32; ch += 2) {
        tc_ld32(taddr + (ch + 1) * 32, vb);                                     // in flight while chunk ch is processed
        epilogue_chunk<MODE, I8, QF>(p, va, inv + ch * 32, tau, qs, q, out_row + ch * 32, (uint32_t)(row0 + ch * 32), staging, et, cnt,
                                     gb + ch * 32, yr + ch * 32, qt);
        tc_wait_ld();
        if (ch + 2 < BN / 32) tc_ld32(taddr + (ch + 2) * 32, va);
        epilogue_chunk<MODE, I8, QF>(p, vb, inv + (ch + 1) * 32, tau, qs, q, out_row + (ch + 1) * 32, (uint32_t)(row0 + (ch + 1) * 32), staging,
                                     et, cnt, gb + (ch + 1) * 32, yr + (ch + 1) * 32, qt);
        if (ch + 2 < BN / 32) tc_wait_ld();
    }
}

// Shared by both kernels' epilogue warps: stage the tile's inv_norm (NaN marks rows beyond the shard and rows the batch
// predicate filters out: they can never pass tau) and, with per-query filters, its genre_bits / year.
template <bool QF>
__device__ __forceinline__ void stage_tile_columns(const GemmParams& p, int64_t row0, int et, float* inv, uint32_t* gb, uint16_t* yr) {
    for (int c = et; c < BN; c += 128) {
        const int64_t r = row0 + c;
        inv[c] = (r < p.n && (!p.has_pred || row_allowed(p.pred, (uint32_t)r))) ? __ldg(p.inv_norm + r) : __int_as_float(0x7FC00000);
        if (QF) {
            gb[c] = (r < p.n && p.qf.genre_bits) ? __ldg(p.qf.genre_bits + r) : 0u;
            yr[c] = (r < p.n && p.qf.year) ? __ldg(p.qf.year + r) : (uint16_t)0;
        }
    }
}

template <int MODE, bool I8, bool QF = false>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_rows, const GemmParams p) {
    constexpr int BKE = I8 ? 2 * BK : BK;             // elements per 128-byte k-block
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* stages = smem;
    uint64_t* staging = (uint64_t*)(smem + GEMM_STAGES * STAGE_BYTES);               // [STAGE_SLOTS][128]
    float* s_inv = (float*)(smem + GEMM_STAGES * STAGE_BYTES + SMEM_STAGING);         // [2][BN]
    uint64_t* bars = (uint64_t*)(smem + GEMM_STAGES * STAGE_BYTES + SMEM_STAGING + SMEM_INV);
    uint64_t* full_bar = bars;                       // [GEMM_STAGES]
    uint64_t* empty_bar = bars + GEMM_STAGES;        // [GEMM_STAGES]
    uint64_t* tfull_bar = bars + 2 * GEMM_STAGES;    // [2]
    uint64_t* tempty_bar = bars + 2 * GEMM_STAGES + 2;   // [2]
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * GEMM_STAGES + 4);
    uint32_t* s_gb = (uint32_t*)((unsigned char*)bars + 256);                        // [2][BN]  QF only
    uint16_t* s_yr = (uint16_t*)(s_gb + 2 * BN);                                       // [2][BN]  QF only

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t total_tiles = (int64_t)p.num_rt * p.num_qt;

    if (threadIdx.x == 0) {
        prefetch_tmap(&map_q);
        prefetch_tmap(&map_rows);
        for (int s = 0; s < GEMM_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], EPI_WARPS); }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ============================ TMA producer ============================
        if (lane == 0) {
            const uint64_t pol_rows = l2_policy_evict_normal();  // catalog tiles: re-read from L2 by the other query tiles of the wave
            const uint64_t pol_q = l2_policy_evict_last();       // query tiles: reused by every row tile
            uint32_t it = 0;
            for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int64_t rt = t / p.num_qt;
                const int qt = (int)(t - rt * p.num_qt);
                const int row0 = (int)((p.tile0 + rt * p.tile_stride) * BN);
                for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
                    const int s = it % GEMM_STAGES;
                    mbar_wait(&empty_bar[s], ((it / GEMM_STAGES) & 1u) ^ 1u);
                    unsigned char* sa = stages + s * STAGE_BYTES;
                    mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                    tma_load_2d(sa, &map_q, kb * BKE, qt * BM, &full_bar[s], pol_q);
                    tma_load_2d(sa + A_BYTES, &map_rows, kb * BKE, row0, &full_bar[s], pol_rows);
                }
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ============================
        if (lane == 0) {
            uint32_t it = 0, tile_i = 0;
            for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x, ++tile_i) {
                const int acc = tile_i & 1;
                mbar_wait(&tempty_bar[acc], ((tile_i >> 1) & 1u) ^ 1u);     // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
                    const int s = it % GEMM_STAGES;
                    mbar_wait(&full_bar[s], (it / GEMM_STAGES) & 1u);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(stages + s * STAGE_BYTES);
                    const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + A_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UK; ++k) {
                        // advancing K by 16 bf16 (32 int8) = 32 B inside the 128-B swizzle atom: +2 in the (>>4) address field
                        if (I8) tc_mma_i8(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), kInstrDescI8, (kb | k) ? 1u : 0u);
                        else tc_mma_bf16(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), kInstrDesc, (kb | k) ? 1u : 0u);
                    }
                    tc_commit(&empty_bar[s]);            // smem stage reusable once these MMAs have read it
                }
                tc_commit(&tfull_bar[acc]);              // accumulator complete
            }
        }
    } else {
        // ============================ epilogue warps ============================
        const int ew = warp - 2;                          // 0..3
        const int quarter = warp & 3;                     // TMEM lane quarter this warp may access
        const int et = ew * 32 + lane;                    // 0..127 epilogue thread id
        const int qrow = quarter * 32 + lane;             // accumulator row (query within the tile)
        uint32_t tile_i = 0;
        for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x, ++tile_i) {
            const int64_t rt = t / p.num_qt;
            const int qt = (int)(t - rt * p.num_qt);
            const int64_t row0 = (p.tile0 + rt * p.tile_stride) * BN;
            const int acc = tile_i & 1;
            const int q = qt * BM + qrow;
            // inv_norm slice of this row tile -> smem (NaN marks rows beyond the shard so they never pass / are skipped)
            float* inv = s_inv + (tile_i & 1) * BN;
            uint32_t* gb = s_gb + (tile_i & 1) * BN;
            uint16_t* yr = s_yr + (tile_i & 1) * BN;
            stage_tile_columns<QF>(p, row0, et, inv, gb, yr);
            float tau = INFINITY, qs = 1.f;
            if (I8 && q < p.b) qs = __ldg(p.qscale + q);
            if (MODE == MODE_FILTER && q < p.b) tau = I8 ? __ldg(p.tau + q) / qs : __ldg(p.tau + q);
            QueryTest qtest{0u, 0u, 0xFFFFu};
            if (QF && q < p.b) qtest = load_query_test(p.qf, q);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(&tfull_bar[acc], (tile_i >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN);
            int cnt = 0;
            epilogue_tile<MODE, I8, QF>(p, taddr, inv, tau, qs, q, row0, rt, staging, et, cnt, gb, yr, qtest);
            // accumulator drained: hand it back to the MMA warp before the (slow) global appends
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (MODE == MODE_FILTER && cnt > 0) {
                if (cnt > STAGE_SLOTS) { p.status[q] = 1; cnt = STAGE_SLOTS; }    // tau far too low for this query
                const unsigned base = atomicAdd(p.cand_count + q, (unsigned)cnt);
                uint64_t* dst = p.cand + (size_t)q * p.cand_cap;
                for (int i = 0; i < cnt; ++i)
                    if (base + i < (unsigned)p.cand_cap) dst[base + i] = staging[i * 128 + et];
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");   // s_inv / staging of this parity are free again
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

// =========================================================================================================
// cta_group::2 variant: a cluster of two CTAs (one SM pair) computes a 256-query x 256-row tile.  CTA r stages its own
// 128 query rows (A half) and its own 128 catalog rows (B half) per k-block — 32 KB per stage instead of 48 KB, and the
// MMA reads each operand byte from shared memory once per PAIR, which is what lifts the shared-memory-bandwidth cap
// of the 1-CTA kernel.  The leader CTA (rank 0) owns the full barriers and issues tcgen05.mma.cta_group::2 (M=256,
// N=256, K=16); its commits are multicast to both CTAs' empty / tmem-full barriers; both CTAs' epilogue warps drain
// their own 128 x 256 accumulator half and arrive on the leader's tmem-empty barrier (the peer remotely).
// =========================================================================================================
constexpr int G2_STAGES = 6;
constexpr int G2_A_BYTES = 128 * BK * 2, G2_B_BYTES = 128 * BK * 2, G2_STAGE_BYTES = G2_A_BYTES + G2_B_BYTES;
constexpr int G2_SMEM = G2_STAGES * G2_STAGE_BYTES + SMEM_STAGING + SMEM_INV + 256 + 1024;
constexpr uint32_t kInstrDesc2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
constexpr uint32_t kInstrDesc2I8 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank)); return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(leader_bar), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accum)
        : "memory");
}

__device__ __forceinline__ void tc_mma_i8_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accum)
        : "memory");
}

template <int MODE, bool I8, bool QF = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_rows, const GemmParams p) {
    constexpr int BKE = I8 ? 2 * BK : BK;             // elements per 128-byte k-block
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* stages = smem;
    uint64_t* staging = (uint64_t*)(smem + G2_STAGES * G2_STAGE_BYTES);
    float* s_inv = (float*)(smem + G2_STAGES * G2_STAGE_BYTES + SMEM_STAGING);
    uint64_t* bars = (uint64_t*)(smem + G2_STAGES * G2_STAGE_BYTES + SMEM_STAGING + SMEM_INV);
    uint64_t* full_bar = bars;                         // [G2_STAGES]  used in the leader CTA only
    uint64_t* empty_bar = bars + G2_STAGES;            // [G2_STAGES]  per CTA, arrived by the multicast commit
    uint64_t* tfull_bar = bars + 2 * G2_STAGES;        // [2]          per CTA, arrived by the multicast commit
    uint64_t* tempty_bar = bars + 2 * G2_STAGES + 2;   // [2]          leader only: 2 x EPI_WARPS arrivals
    uint32_t* tmem_slot = (uint32_t*)(bars + 2 * G2_STAGES + 4);
    uint32_t* s_gb = (uint32_t*)((unsigned char*)bars + 256);   // [2][BN]  QF only
    uint16_t* s_yr = (uint16_t*)(s_gb + 2 * BN);                  // [2][BN]  QF only

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    const int num_qt2 = (p.b + 255) / 256;                                     // 256-query tiles
    const int64_t total_tiles = (int64_t)p.num_rt * num_qt2;
    const int64_t cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        prefetch_tmap(&map_q);
        prefetch_tmap(&map_rows);
        for (int s = 0; s < G2_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 2 * EPI_WARPS); }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    tc_fence_before();
    cluster_sync_all();                                 // both CTAs' barriers are initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ============================ TMA producer (both CTAs, each for its own halves) ============================
        if (lane == 0) {
            const uint64_t pol_rows = l2_policy_evict_normal();
            const uint64_t pol_q = l2_policy_evict_last();
            uint32_t it = 0;
            for (int64_t t = cluster_id; t < total_tiles; t += num_clusters) {
                const int64_t rt = t / num_qt2;
                const int qt = (int)(t - rt * num_qt2);
                const int row0 = (int)((p.tile0 + rt * p.tile_stride) * BN) + (int)cta_rank * 128;
                const int q0 = qt * 256 + (int)cta_rank * 128;
                for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
                    const int s = it % G2_STAGES;
                    mbar_wait(&empty_bar[s], ((it / G2_STAGES) & 1u) ^ 1u);
                    unsigned char* sa = stages + s * G2_STAGE_BYTES;
                    const uint32_t lbar = mapa_u32(smem_u32(&full_bar[s]), 0);        // the leader's full barrier
                    if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * G2_STAGE_BYTES); // bytes of BOTH CTAs land on it
                    tma_load_2d_2sm(sa, &map_q, kb * BKE, q0, lbar, pol_q);
                    tma_load_2d_2sm(sa + G2_A_BYTES, &map_rows, kb * BKE, row0, lbar, pol_rows);
                }
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer (leader CTA only) ============================
        if (leader && lane == 0) {
            uint32_t it = 0, tile_i = 0;
            for (int64_t t = cluster_id; t < total_tiles; t += num_clusters, ++tile_i) {
                const int acc = tile_i & 1;
                mbar_wait(&tempty_bar[acc], ((tile_i >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
                    const int s = it % G2_STAGES;
                    mbar_wait(&full_bar[s], (it / G2_STAGES) & 1u);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(stages + s * G2_STAGE_BYTES);
                    const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + G2_A_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UK; ++k) {
                        if (I8) tc_mma_i8_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), kInstrDesc2I8, (kb | k) ? 1u : 0u);
                        else tc_mma_bf16_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), kInstrDesc2, (kb | k) ? 1u : 0u);
                    }
                    tc_commit_2sm(&empty_bar[s]);
                }
                tc_commit_2sm(&tfull_bar[acc]);
            }
        }
    } else {
        // ============================ epilogue warps (both CTAs, own 128 queries x 256 rows) ============================
        const int ew = warp - 2;
        const int quarter = warp & 3;
        const int et = ew * 32 + lane;
        const int qrow = quarter * 32 + lane;
        const uint32_t leader_tempty0 = mapa_u32(smem_u32(&tempty_bar[0]), 0);
        const uint32_t leader_tempty1 = mapa_u32(smem_u32(&tempty_bar[1]), 0);
        uint32_t tile_i = 0;
        for (int64_t t = cluster_id; t < total_tiles; t += num_clusters, ++tile_i) {
            const int64_t rt = t / num_qt2;
            const int qt = (int)(t - rt * num_qt2);
            const int64_t row0 = (p.tile0 + rt * p.tile_stride) * BN;
            const int acc = tile_i & 1;
            const int q = qt * 256 + (int)cta_rank * 128 + qrow;
            float* inv = s_inv + (tile_i & 1) * BN;
            uint32_t* gb = s_gb + (tile_i & 1) * BN;
            uint16_t* yr = s_yr + (tile_i & 1) * BN;
            stage_tile_columns<QF>(p, row0, et, inv, gb, yr);
            float tau = INFINITY, qs = 1.f;
            if (I8 && q < p.b) qs = __ldg(p.qscale + q);
            if (MODE == MODE_FILTER && q < p.b) tau = I8 ? __ldg(p.tau + q) / qs : __ldg(p.tau + q);
            QueryTest qtest{0u, 0u, 0xFFFFu};
            if (QF && q < p.b) qtest = load_query_test(p.qf, q);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(&tfull_bar[acc], (tile_i >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN);
            int cnt = 0;
            epilogue_tile<MODE, I8, QF>(p, taddr, inv, tau, qs, q, row0, rt, staging, et, cnt, gb, yr, qtest);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(acc ? leader_tempty1 : leader_tempty0);
            if (MODE == MODE_FILTER && cnt > 0) {
                if (cnt > STAGE_SLOTS) { p.status[q] = 1; cnt = STAGE_SLOTS; }
                const unsigned base = atomicAdd(p.cand_count + q, (unsigned)cnt);
                uint64_t* dst = p.cand + (size_t)q * p.cand_cap;
                for (int i = 0; i < cnt; ++i)
                    if (base + i < (unsigned)p.cand_cap) dst[base + i] = staging[i * 128 + et];
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
    }

    tc_fence_before();
    cluster_sync_all();                                 // nobody leaves while the peer may still touch its smem / TMEM
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

// ---------------------------------------------------------------------------------------------------------
// Per query: r-th largest sample score after masking excluded rows (4-pass radix select on orderable keys).
// Sample column j*256 + c is catalog row (tile0 + j*stride)*256 + c.
// Per-query filters (has_qf): rows the query's own genre / year test rejects are masked like excluded rows, so the rank-th best
// of the allowed sampled rows estimates the same quantile of the allowed population and the survivor count stays at the plan's
// figure.  Fewer than `rank` allowed sampled rows give tau = -inf: every allowed row survives (an overflow sets status bit 2).
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) select_threshold_kernel(float* sample, int keys_in_smem, int64_t s_cols, int64_t n,
                                                               int64_t row_base, int64_t tile0, int64_t tile_stride, int rank,
                                                               DevFilter pred, int has_pred, QueryFilter qf, int has_qf,
                                                               const int64_t* __restrict__ excl_ptr,
                                                               const int32_t* __restrict__ excl_col, float* __restrict__ tau) {
    extern __shared__ uint32_t smem_keys[];        // [s_cols] when it fits, else the sample row is rewritten in place
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix, s_rank;
    const int q = blockIdx.x;
    float* src = sample + (int64_t)q * s_cols;
    uint32_t* keys = keys_in_smem ? smem_keys : (uint32_t*)src;
    const int32_t* ex = nullptr;
    int nex = 0;
    if (excl_ptr) { ex = excl_col + excl_ptr[q]; nex = (int)(excl_ptr[q + 1] - excl_ptr[q]); }
    const QueryTest qt = has_qf ? load_query_test(qf, q) : QueryTest{0u, 0u, 0xFFFFu};
    for (int64_t j = threadIdx.x; j < s_cols; j += blockDim.x) {
        const int64_t row = (tile0 + (j / BN) * tile_stride) * BN + (j % BN);
        const float v = src[j];
        bool keep = row < n && v == v && (!has_pred || row_allowed(pred, (uint32_t)row));
        if (keep && has_qf)
            keep = query_allows(qt, qf.genre_bits ? __ldg(qf.genre_bits + row) : 0u, qf.year ? (uint32_t)__ldg(qf.year + row) : 0u);
        keys[j] = keep ? f32_orderable(v) : 0u;
    }
    __syncthreads();
    // knock out excluded rows that fall inside the sample: ~|excluded| scattered stores instead of a search per key
    for (int e = threadIdx.x; e < nex; e += blockDim.x) {
        const int64_t row = (int64_t)ex[e] - row_base;
        if (row < 0 || row >= n) continue;
        const int64_t tile = row / BN - tile0;
        if (tile < 0 || tile % tile_stride != 0) continue;
        const int64_t j = (tile / tile_stride) * BN + row % BN;
        if (j < s_cols) keys[j] = 0u;
    }
    // ---- fast path: prune with the rank-th largest of the per-thread maxima (a lower bound of the answer, because
    // `rank` distinct keys are >= it), gather the handful of keys above it, rank-count exactly.  No histogram atomics.
    __shared__ uint32_t s_max[256];
    __shared__ uint32_t s_buf[1024];
    __shared__ uint32_t s_low, s_ans;
    __shared__ int s_n, s_found;
    {
        uint32_t mx = 0;
        for (int64_t j = threadIdx.x; j < s_cols; j += blockDim.x) mx = max(mx, keys[j]);
        s_max[threadIdx.x] = mx;
        if (threadIdx.x == 0) { s_low = 0; s_n = 0; s_found = 0; s_ans = 0; }
        __syncthreads();
        if (rank <= (int)blockDim.x) {
            int c = 0;
            for (int t = 0; t < (int)blockDim.x; ++t) c += (s_max[t] > mx) || (s_max[t] == mx && t < (int)threadIdx.x);
            if (c == rank - 1) s_low = mx;                      // exactly one thread has this position
        }
        __syncthreads();
        const uint32_t low = s_low;
        if (low != 0) {
            for (int64_t j = threadIdx.x; j < s_cols; j += blockDim.x) {
                const uint32_t kk = keys[j];
                if (kk >= low) {
                    const int idx = atomicAdd(&s_n, 1);
                    if (idx < 1024) s_buf[idx] = kk;
                }
            }
        }
        __syncthreads();
        const int nb = s_n;
        if (low != 0 && nb >= rank && nb <= 1024) {
            for (int t = threadIdx.x; t < nb; t += blockDim.x) {
                const uint32_t kk = s_buf[t];
                int c = 0;
                for (int i = 0; i < nb; ++i) c += (s_buf[i] > kk) || (s_buf[i] == kk && i < t);
                if (c == rank - 1) { s_ans = kk; s_found = 1; }
            }
        }
        __syncthreads();
        if (s_found) {
            if (threadIdx.x == 0) tau[q] = orderable_f32(s_ans);
            return;
        }
    }
    // ---- general path (tiny samples, mass ties): 4-pass radix select
    if (threadIdx.x == 0) { s_prefix = 0; s_rank = (unsigned)rank; }
    __syncthreads();
    for (int pass = 3; pass >= 0; --pass) {
        hist[threadIdx.x] = 0;
        __syncthreads();
        const unsigned prefix = s_prefix;
        const unsigned himask = pass == 3 ? 0u : (0xFFFFFFFFu << (8 * (pass + 1)));
        for (int64_t j = threadIdx.x; j < s_cols; j += blockDim.x) {
            const uint32_t k = keys[j];
            if (k != 0 && (k & himask) == prefix) atomicAdd(&hist[(k >> (8 * pass)) & 0xFF], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned need = s_rank, cum = 0;
            int bin = 255;
            for (; bin >= 0; --bin) {
                if (cum + hist[bin] >= need) break;
                cum += hist[bin];
            }
            if (bin < 0) { s_prefix = 0; s_rank = 0xFFFFFFFFu; }     // fewer than `rank` valid samples
            else { s_prefix = prefix | ((unsigned)bin << (8 * pass)); s_rank = need - cum; }
        }
        __syncthreads();
        if (s_rank == 0xFFFFFFFFu) break;
    }
    if (threadIdx.x == 0) tau[q] = (s_rank == 0xFFFFFFFFu || s_prefix == 0) ? -INFINITY : orderable_f32(s_prefix);
}

// Per query: survivors of the filter -> drop excluded rows -> best kc keys, sorted (zero padded).
// With many more survivors than kc a full sort is wasted work: the scores' range [lo, hi] is cut into 1024 linear
// buckets, a histogram finds the bucket holding the kc-th best, and only the keys from that bucket upwards (kc + a
// few) are sorted.  Small or degenerate inputs (few survivors, mass ties) take the plain bitonic sort.
__global__ void __launch_bounds__(512) select_candidates_kernel(const uint64_t* __restrict__ cand, const unsigned* __restrict__ cand_count,
                                                                int cand_cap, int kc, int64_t row_base,
                                                                const int64_t* __restrict__ excl_ptr, const int32_t* __restrict__ excl_col,
                                                                const float* __restrict__ tau, uint64_t* __restrict__ out_keys,
                                                                int* __restrict__ status) {
    extern __shared__ __align__(16) uint64_t buf[];        // [pow2 >= cand_cap] survivors, then [1024] top set
    __shared__ unsigned hist[1024];
    __shared__ int s_valid, s_m, s_bstar;
    __shared__ unsigned s_lo, s_hi;
    const int q = blockIdx.x;
    const unsigned cnt_raw = cand_count[q];
    const int cnt = cnt_raw < (unsigned)cand_cap ? (int)cnt_raw : cand_cap;
    const int32_t* ex = nullptr;
    int nex = 0;
    if (excl_ptr) { ex = excl_col + excl_ptr[q]; nex = (int)(excl_ptr[q + 1] - excl_ptr[q]); }
    int p2 = 2;
    while (p2 < cnt || p2 < kc) p2 <<= 1;
    if (threadIdx.x == 0) { s_valid = 0; s_m = 0; s_lo = 0xFFFFFFFFu; s_hi = 0; s_bstar = 0; }
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    int mine = 0;
    unsigned lo = 0xFFFFFFFFu, hi = 0;
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        uint64_t key = i < cnt ? cand[(size_t)q * cand_cap + i] : 0;
        if (key && nex && sorted_contains(ex, nex, (int32_t)(row_base + key_row(key)))) key = 0;
        buf[i] = key;
        if (key) {
            ++mine;
            const unsigned v = (unsigned)(key >> 32);
            lo = min(lo, v);
            hi = max(hi, v);
        }
    }
    if (mine) { atomicAdd(&s_valid, mine); atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    const int valid = s_valid;
    bool sorted_in_place = true;
    if (valid > 2 * kc && s_hi > s_lo) {
        // ---- bucket select
        const unsigned blo = s_lo;
        const unsigned long long range = (unsigned long long)(s_hi - blo) + 1ull;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const uint64_t key = buf[i];
            if (key) atomicAdd(&hist[(unsigned)(((unsigned long long)((unsigned)(key >> 32) - blo) * 1023ull) / range)], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int cum = 0, b = 1023;
            for (; b > 0; --b) { cum += (int)hist[b]; if (cum >= kc) break; }
            if (b == 0) cum += (int)hist[0];
            s_bstar = b;
            s_m = cum >= kc ? cum : -1;            // keys in buckets >= b*
        }
        __syncthreads();
        const int m = s_m, bstar = s_bstar;
        if (m >= kc && m <= 1024) {
            uint64_t* top = buf + p2;              // second region of the dynamic smem
            __syncthreads();
            if (threadIdx.x == 0) s_m = 0;
            __syncthreads();
            for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
                const uint64_t key = buf[i];
                if (key && (int)(((unsigned long long)((unsigned)(key >> 32) - blo) * 1023ull) / range) >= bstar)
                    top[atomicAdd(&s_m, 1)] = key;
            }
            __syncthreads();
            int t2 = 2;
            while (t2 < m) t2 <<= 1;
            for (int i = m + threadIdx.x; i < t2; i += blockDim.x) top[i] = 0;
            __syncthreads();
            block_bitonic_sort_desc(top, t2);
            for (int i = threadIdx.x; i < kc; i += blockDim.x) out_keys[(size_t)q * kc + i] = top[i];
            sorted_in_place = false;
        }
    }
    if (sorted_in_place) {
        __syncthreads();
        block_bitonic_sort_desc(buf, p2);
        for (int i = threadIdx.x; i < kc; i += blockDim.x) out_keys[(size_t)q * kc + i] = buf[i];
    }
    if (threadIdx.x == 0) {
        int st = status[q];
        if (cnt_raw > (unsigned)cand_cap) st |= 2;                         // buffer overflow: some survivors were dropped
        if (valid < kc && tau[q] != -INFINITY) st |= 4;                    // threshold too optimistic: not enough candidates
        status[q] = st;
    }
}

// Long lists (k > 240, kc up to 4096): the survivors (~3 kc, up to cand_cap = 64 Ki keys) stay in global memory.  Per query:
//   pass 1  drop excluded rows (zeroed in place, so later passes skip the search) and find the score range [lo, hi];
//   pass 2  only when more than gather_cap keys are valid: histogram of the scores over 2048 linear buckets of [lo, hi], and
//           the bucket b* that holds the kc-th best (suffix sums: one lane per 64 buckets, then one lane walks its 64);
//   pass 3  gather every key from bucket b* upwards (kc plus part of one bucket) into shared memory, bitonic sort, write the
//           best kc.
// gather_cap = the power of two >= 2 kc.  A gathered set larger than that (mass ties inside one bucket) sets status bit 16 and
// writes no keys: the caller re-runs the query, nothing is dropped silently.  Bits 2 and 4 as in select_candidates_kernel.
constexpr int kSelLargeThreads = 512, kSelLargeBuckets = 2048;

__device__ __forceinline__ int large_bucket(uint64_t key, unsigned lo, unsigned long long range) {
    return (int)(((unsigned long long)((unsigned)(key >> 32) - lo) * (unsigned long long)kSelLargeBuckets) / range);
}

__global__ void __launch_bounds__(kSelLargeThreads) select_candidates_large_kernel(uint64_t* __restrict__ cand, const unsigned* __restrict__ cand_count,
                                                                              int cand_cap, int kc, int gather_cap, int64_t row_base,
                                                                              const int64_t* __restrict__ excl_ptr,
                                                                              const int32_t* __restrict__ excl_col,
                                                                              const float* __restrict__ tau, uint64_t* __restrict__ out_keys,
                                                                              int* __restrict__ status) {
    extern __shared__ __align__(16) uint64_t top[];        // [gather_cap]
    __shared__ unsigned hist[kSelLargeBuckets];
    __shared__ int s_valid, s_m, s_bstar, s_n;
    __shared__ unsigned s_lo, s_hi;
    const int q = blockIdx.x;
    const unsigned cnt_raw = cand_count[q];
    const int cnt = cnt_raw < (unsigned)cand_cap ? (int)cnt_raw : cand_cap;
    uint64_t* src = cand + (size_t)q * cand_cap;
    const int32_t* ex = nullptr;
    int nex = 0;
    if (excl_ptr) { ex = excl_col + excl_ptr[q]; nex = (int)(excl_ptr[q + 1] - excl_ptr[q]); }
    if (threadIdx.x == 0) { s_valid = 0; s_n = 0; s_lo = 0xFFFFFFFFu; s_hi = 0; s_bstar = 0; }
    for (int i = threadIdx.x; i < kSelLargeBuckets; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    int mine = 0;
    unsigned lo = 0xFFFFFFFFu, hi = 0;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const uint64_t key = src[i];
        if (!key) continue;
        if (nex && sorted_contains(ex, nex, (int32_t)(row_base + key_row(key)))) { src[i] = 0; continue; }
        ++mine;
        lo = min(lo, (unsigned)(key >> 32));
        hi = max(hi, (unsigned)(key >> 32));
    }
    if (mine) { atomicAdd(&s_valid, mine); atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    const int valid = s_valid;
    const unsigned blo = s_lo;
    const unsigned long long range = (unsigned long long)(s_hi - blo) + 1ull;   // only used when valid > 0
    int m = valid, bstar = 0;                                // few enough valid keys: gather them all
    if (valid > gather_cap && s_hi > blo) {
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const uint64_t key = src[i];
            if (key) atomicAdd(&hist[large_bucket(key, blo, range)], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            constexpr int PER = kSelLargeBuckets / 32;
            const int lane = threadIdx.x;
            const int top_b = kSelLargeBuckets - lane * PER;  // lane 0 owns the best buckets [B - 64, B)
            unsigned sum = 0;
            for (int j = 1; j <= PER; ++j) sum += hist[top_b - j];
            unsigned incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned ballot = __ballot_sync(0xffffffffu, incl >= (unsigned)kc);   // != 0: valid > gather_cap > kc
            if (lane == __ffs(ballot) - 1) {
                unsigned cum = incl - sum;
                int bb = top_b - 1;
                for (; bb > top_b - PER; --bb) {
                    cum += hist[bb];
                    if (cum >= (unsigned)kc) break;
                }
                if (cum < (unsigned)kc) cum += hist[bb];      // the walk ended on the lane's lowest bucket
                s_bstar = bb;
                s_m = (int)cum;
            }
        }
        __syncthreads();
        m = s_m;
        bstar = s_bstar;
    } else if (valid > gather_cap) {
        m = valid;                                           // every valid key has the same score: cannot split
    }
    const bool fits = m <= gather_cap;
    if (fits) {
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const uint64_t key = src[i];
            if (key && large_bucket(key, blo, range) >= bstar) {
                const int idx = atomicAdd(&s_n, 1);
                REBERT_ASSERT(idx >= 0 && idx < gather_cap);
                top[idx] = key;
            }
        }
        int t2 = 2;
        while (t2 < m || t2 < kc) t2 <<= 1;
        for (int i = m + threadIdx.x; i < t2; i += blockDim.x) top[i] = 0;
        __syncthreads();
        block_bitonic_sort_desc(top, t2);
    }
    for (int i = threadIdx.x; i < kc; i += blockDim.x) {
        REBERT_ASSERT(i < gather_cap);
        out_keys[(size_t)q * kc + i] = fits ? top[i] : 0ull;
    }
    if (threadIdx.x == 0) {
        int st = status[q];
        if (cnt_raw > (unsigned)cand_cap) st |= 2;                         // buffer overflow: some survivors were dropped
        if (valid < kc && tau[q] != -INFINITY) st |= 4;                    // threshold too optimistic: not enough candidates
        if (!fits) st |= 16;                                               // mass ties: the kc best could not be isolated
        status[q] = st;
    }
}

__global__ void margin_status_kernel(const double* __restrict__ margin, double eps, int b, int* __restrict__ status) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < b && !(margin[q] > eps)) status[q] |= 8;
}

// ---------------------------------------------------------------- host side ----------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)sym;
    }
    return fn;
}

// 2-D tensor map over a row-major [rows, ld] matrix of bf16 (or int8: `i8`), box = [box_rows x 128 bytes], 128-byte swizzle.
static int make_tmap(CUtensorMap* map, const void* base, int64_t rows, int ld, int box_rows, bool i8 = false) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled unavailable from the driver"); return REBERT_ERR_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * (i8 ? 1 : 2)};
    cuuint32_t box[2] = {(cuuint32_t)(i8 ? 2 * BK : BK), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, i8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld ld=%d", (int)r, (long long)rows, ld); return REBERT_ERR_CUDA; }
    return REBERT_OK;
}

static int check_gemm_catalog(const rebert_catalog_t* cat, const char* who) {
    REBERT_REQUIRE(cat && cat->rows && cat->inv_norm, "%s: null catalog", who);
    if (cat->dtype != REBERT_BF16 && cat->dtype != REBERT_I8) {
        set_error("%s: the tensor-core path needs a bf16 catalog (or its int8 shadow)", who);
        return REBERT_ERR_UNSUPPORTED;
    }
    const int kblock = cat->dtype == REBERT_I8 ? 2 * BK : BK;        // elements per 128-byte k-block
    if (cat->ld % kblock != 0) { set_error("%s: ld=%d is not a multiple of %d", who, cat->ld, kblock); return REBERT_ERR_UNSUPPORTED; }
    REBERT_REQUIRE(cat->n > 0 && cat->n < (1ll << 31) - BN, "%s: shard rows %lld out of range", who, (long long)cat->n);
    REBERT_REQUIRE(((uintptr_t)cat->rows & 127) == 0, "%s: catalog rows must be 128-byte aligned", who);
    return REBERT_OK;
}

static void set_pred(GemmParams& p, const rebert_catalog_t* cat, const rebert_filter_t* filter) {
    rebert_filter_t f;
    memset(&f, 0, sizeof(f));
    if (filter) { f = *filter; f.exclude_rows = nullptr; f.n_exclude = 0; }       // per-query exclusions travel as CSR
    p.pred = make_filter(&f, cat->row_base);
    p.has_pred = (f.exclude_bitmap || f.genre_bits || f.year) ? 1 : 0;
}

// `cat` is the operand catalog the tensor cores stream: the bf16 catalog of record, or its int8 shadow (then qmat is int8
// [b, ld8] and p.qscale holds the queries' dequantisation steps).
template <int MODE, bool I8, bool QF>
static int launch_gemm_t(const rebert_catalog_t* cat, const void* qmat, GemmParams& p, cudaStream_t st) {
    static_assert(!QF || MODE == MODE_FILTER, "per-query filters apply to the filter pass only");
    constexpr int extra_smem = QF ? SMEM_QF : 0;
    const bool pair = p.b > BM;   // cta_group::2 needs >= 2 query tiles to pay off
    CUtensorMap map_q, map_rows;
    int rc = make_tmap(&map_q, qmat, p.b, cat->ld, BM, I8);
    if (rc != REBERT_OK) return rc;
    rc = make_tmap(&map_rows, cat->rows, cat->n, cat->ld, pair ? 128 : BN, I8);
    if (rc != REBERT_OK) return rc;
    p.kblocks = cat->ld / (I8 ? 2 * BK : BK);
    p.n = cat->n;
    p.inv_norm = cat->inv_norm;
    p.num_qt = (p.b + BM - 1) / BM;
    if (pair) {
        const int64_t tiles = (int64_t)p.num_rt * ((p.b + 255) / 256);
        int grid = num_sms() & ~1;
        if (tiles * 2 < grid) grid = (int)(tiles * 2);
        auto kern = gemm2_kernel<MODE, I8, QF>;
        { int rc__ = raise_smem_limit(kern); if (rc__ != REBERT_OK) return rc__; }
        kern<<<grid, GEMM_THREADS, G2_SMEM + extra_smem, st>>>(map_q, map_rows, p);
    } else {
        const int64_t tiles = (int64_t)p.num_rt * p.num_qt;
        int grid = num_sms();
        if (tiles < grid) grid = (int)tiles;
        auto kern = gemm_kernel<MODE, I8, QF>;
        { int rc__ = raise_smem_limit(kern); if (rc__ != REBERT_OK) return rc__; }
        kern<<<grid, GEMM_THREADS, GEMM_SMEM + extra_smem, st>>>(map_q, map_rows, p);
    }
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}
template <int MODE, bool QF = false>
static int launch_gemm(const rebert_catalog_t* cat, const void* qmat, GemmParams& p, cudaStream_t st) {
    return cat->dtype == REBERT_I8 ? launch_gemm_t<MODE, true, QF>(cat, qmat, p, st) : launch_gemm_t<MODE, false, QF>(cat, qmat, p, st);
}

// Queries for the int8 operand path: q8[u, c] = rint(qn32[u, c] / step_u), step_u = max|qn32[u, :]| / 127 (1 for an all-zero
// query), zero padded to ld8.  eps[u] = the margin a result of query u must clear to count as proven on this path:
// 6 standard deviations of the score error under the random-direction model — the quantisation error vectors of row
// and query, of relative norms row_err (the shadow's measured worst) and rho_u (measured here), are not aligned with the
// vectors they meet, so the dot-product error has standard deviation sqrt(row_err^2 + rho_u^2) / sqrt(d) — plus fp32 noise.
__global__ void __launch_bounds__(256) query_quantize_i8_kernel(const float* __restrict__ qn32, int d, int ld, int ld8, double row_err,
                                                                int8_t* __restrict__ q8, float* __restrict__ qscale, double* __restrict__ eps) {
    __shared__ float s_max[8];
    __shared__ double s_e2[8], s_n2[8];
    const int u = blockIdx.x;
    const float* q = qn32 + (size_t)u * ld;
    float m = 0.f;
    for (int c = threadIdx.x; c < d; c += blockDim.x) m = fmaxf(m, fabsf(q[c]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
    __syncthreads();
    m = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) m = fmaxf(m, s_max[w]);
    const float step = m > 0.f ? m / 127.f : 1.f;
    double e2 = 0.0, n2 = 0.0;
    for (int c = threadIdx.x; c < ld8; c += blockDim.x) {
        int v = 0;
        if (c < d) {
            const float x = q[c];
            v = __float2int_rn(x / step);
            v = max(-127, min(127, v));
            const double e = (double)x - (double)v * (double)step;
            e2 = fma(e, e, e2);
            n2 = fma((double)x, (double)x, n2);
        }
        q8[(size_t)u * ld8 + c] = (int8_t)v;
    }
    e2 = warp_sum(e2);
    n2 = warp_sum(n2);
    if ((threadIdx.x & 31) == 0) { s_e2[threadIdx.x >> 5] = e2; s_n2[threadIdx.x >> 5] = n2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double E = 0.0, N = 0.0;
        for (int w = 0; w < 8; ++w) { E += s_e2[w]; N += s_n2[w]; }
        const double rho = N > 0.0 ? sqrt(E / N) : 0.0;                 // relative quantisation error of this query
        qscale[u] = step;
        // scores scale with ||q|| (a profile is shorter than a unit vector), and so does their error
        eps[u] = 6.0 * sqrt(row_err * row_err + rho * rho) / sqrt((double)d) * fmax(sqrt(N), 1e-30) + 64.0 * 5.96e-8;
    }
}

__global__ void margin_status_eps_kernel(const double* __restrict__ margin, const double* __restrict__ eps, int b, int* __restrict__ status) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < b && !(margin[q] > eps[q])) status[q] |= 8;
}

struct GemmWorkspace {
    float* sample;        // [b, sample_rows]
    float* tau;           // [b]
    unsigned* cand_count; // [b]
    uint64_t* cand;       // [b, cand_cap]
    uint64_t* cand_keys;  // [b, kc]
    double* margin;       // [b]
    size_t bytes;
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static GemmWorkspace carve(void* base, const rebert_gemm_plan_t* pl) {
    GemmWorkspace w;
    size_t off = 0;
    unsigned char* b0 = (unsigned char*)align_up((uintptr_t)base, 256);
    auto take = [&](size_t bytes) { void* ptr = b0 ? b0 + off : nullptr; off += align_up(bytes, 256); return ptr; };
    w.sample = (float*)take((size_t)pl->b * pl->sample_rows * 4);
    w.tau = (float*)take((size_t)pl->b * 4);
    w.cand_count = (unsigned*)take((size_t)pl->b * 4);
    w.cand = (uint64_t*)take((size_t)pl->b * pl->cand_cap * 8);
    w.cand_keys = (uint64_t*)take((size_t)pl->b * pl->kc * 8);
    w.margin = (double*)take((size_t)pl->b * 8);
    w.bytes = off + 256;
    return w;
}

}  // namespace rebert

using namespace rebert;

extern "C" {

static int gemm_plan_impl(int64_t n, int32_t b, int32_t k, bool shadow, rebert_gemm_plan_t* plan) {
    REBERT_REQUIRE(plan && n > 0 && b > 0 && k > 0, "gemm_plan: bad arguments");
    // Candidates for the exact pass.  The proof margin here must absorb the bf16 rounding of the query (sigma ~ 3e-5 at
    // d = 1536), so the list keeps >= 25 % more than k (the gap between the k-th and the 1.25k-th best of a large catalog
    // is ~1e-3); k itself must stay within what the single-query re-run path can serve.
    // int8 operands (shadow): the score error is ~10x larger (sigma ~ 0.009 / sqrt(d) per unit of row and query error), and
    // the margin has to clear 6 sigma plus twice the largest error seen on the candidates — ~0.16 standard deviations of the
    // score distribution, i.e. ~0.7 k more rows at the densities of a 1M..10M catalog (k z rows per unit z): the list doubles.
    if (k > kLargeKMax || (k <= kLargeK0 && rebert_candidates_for_k(k) == 0)) {
        set_error("gemm_plan: k=%d unsupported", k);
        return REBERT_ERR_UNSUPPORTED;
    }
    int need = k + 16 > k + (k + 3) / 4 ? k + 16 : k + (k + 3) / 4;
    if (shadow) need = k + (k > 64 ? k : 64);
    const int kc = (need + 31) / 32 * 32;
    if (k > kLargeK0) {
        // Long lists (k > 240, served by select_candidates_large_kernel + finalize_large_kernel).  The sample rank is 64 and
        // the survivor target E = max(3 kc, 50 x 64): P(Gamma(64) < 64 / 3) = 7e-14 that fewer than kc rows pass, and the
        // sample is rank / E <= 2 % of the rows (sample tiles round down, which only raises E).  E <= n / 64 as below.
        const int rank = kLargeRank;
        double e = 3.0 * kc;
        if (e < 50.0 * rank) e = 50.0 * rank;
        if (e > (double)n / 64.0) {
            set_error("gemm_plan: catalog of %lld rows is too small for the batched path at k=%d (needs >= %lld rows); "
                      "use the single-query path", (long long)n, k, (long long)(64.0 * e));
            return REBERT_ERR_UNSUPPORTED;
        }
        int64_t st = (int64_t)((double)n * rank / e / BN);
        if (st < 1) st = 1;
        plan->b = b;
        plan->k = k;
        plan->kc = kc;
        plan->sample_rows = (int32_t)(st * BN);
        plan->sample_rank = rank;
        int cap = 2 * kc;
        while (cap < 4.0 * e) cap <<= 1;
        plan->cand_cap = cap;
        return REBERT_OK;
    }
    // Expected survivors per query E = rank * n / sample_rows.  Want E >= 8 kc (the kc best are then inside with
    // overwhelming probability: the survivor count is Gamma(rank)-distributed around E) plus headroom for excluded
    // rows, which tend to score high; and E <= n / 64 so a thread stages ~4 keys per tile on average (24 slots).
    double e = 8.0 * kc;
    double head = (double)n / 64.0 < 1024.0 ? (double)n / 64.0 : 1024.0;
    if (head > e) e = head;
    if (e > (double)n / 64.0) {
        set_error("gemm_plan: catalog of %lld rows is too small for the batched path at k=%d (needs >= %d rows); "
                  "use the single-query path", (long long)n, k, 512 * kc);
        return REBERT_ERR_UNSUPPORTED;
    }
    const int rank = 16;                                    // order statistic of the sample used as threshold
    const int64_t tiles = (n + BN - 1) / BN;
    int64_t st = (int64_t)((double)n * rank / e / BN + 0.5); // sample tiles so that rank * n / sample_rows ~= e
    if (st < 1) st = 1;
    if (st > tiles) st = tiles;
    plan->b = b;
    plan->k = k;
    plan->kc = kc;
    plan->sample_rows = (int32_t)(st * BN);
    plan->sample_rank = rank;
    int cap = 2 * kc;
    while (cap < 4.0 * e) cap <<= 1;
    plan->cand_cap = cap;
    return REBERT_OK;
}

REBERT_API int rebert_gemm_plan(int64_t n, int32_t b, int32_t k, rebert_gemm_plan_t* plan) { return gemm_plan_impl(n, b, k, false, plan); }
REBERT_API int rebert_gemm_plan_i8(int64_t n, int32_t b, int32_t k, rebert_gemm_plan_t* plan) { return gemm_plan_impl(n, b, k, true, plan); }

REBERT_API int rebert_query_quantize_i8(const float* qn32, int32_t b, int32_t d, int32_t ld, int32_t ld8, double row_err, void* q8,
                                        float* qscale, double* eps, rebert_stream stream) {
    REBERT_REQUIRE(qn32 && q8 && qscale && eps && b > 0 && d > 0 && ld >= d && ld8 >= d, "query_quantize_i8: bad arguments");
    query_quantize_i8_kernel<<<b, 256, 0, (cudaStream_t)stream>>>(qn32, d, ld, ld8, row_err, (int8_t*)q8, qscale, eps);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API size_t rebert_gemm_workspace_bytes(const rebert_catalog_t* cat, const rebert_gemm_plan_t* plan) {
    (void)cat;
    if (!plan) return 0;
    return carve(nullptr, plan).bytes;
}

REBERT_API int rebert_gemm_scores(const rebert_catalog_t* cat, const void* qbf16, int32_t b, int64_t row0, int64_t nrows,
                                  float* out, rebert_stream stream) {
    int rc = check_gemm_catalog(cat, "gemm_scores");
    if (rc != REBERT_OK) return rc;
    REBERT_REQUIRE(cat->dtype == REBERT_BF16 && qbf16 && out && b > 0 && nrows > 0, "gemm_scores: bad arguments");
    REBERT_REQUIRE(row0 % BN == 0 && nrows % BN == 0 && row0 >= 0, "gemm_scores: row0 and nrows must be multiples of %d", BN);
    REBERT_REQUIRE(((uintptr_t)out & 15) == 0, "gemm_scores: out must be 16-byte aligned");
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.b = b;
    p.num_rt = (int)(nrows / BN);
    p.tile0 = row0 / BN;
    p.tile_stride = 1;
    p.out = out;
    p.out_ld = nrows;
    set_pred(p, cat, nullptr);
    return launch_gemm<MODE_STORE>(cat, qbf16, p, (cudaStream_t)stream);
}

}  // extern "C"

// `op` = the operand catalog the tensor cores stream (cat itself, or its int8 shadow with qmat = int8 queries, qscale / qeps
// from rebert_query_quantize_i8); the exact pass always reads `cat`.
static int gemm_topk_impl(const rebert_catalog_t* cat, const rebert_catalog_t* op, const void* qbf16, const float* qscale,
                          const double* qeps, const double* q64, const int64_t* excl_row_ptr,
                          const int32_t* excl_col, const rebert_filter_t* row_filter, const rebert_query_filter_t* query_filter,
                          const rebert_gemm_plan_t* plan, void* workspace, size_t workspace_bytes,
                          int64_t* out_rows, double* out_scores, int32_t* out_count, int32_t* out_status,
                          rebert_stream stream) {
    int rc = check_gemm_catalog(op, "gemm_topk");
    if (rc != REBERT_OK) return rc;
    QueryFilter qf;
    memset(&qf, 0, sizeof(qf));
    if (query_filter) {
        qf = QueryFilter{query_filter->genre_bits, query_filter->year, query_filter->genre_any, query_filter->year_lo, query_filter->year_hi};
        REBERT_REQUIRE((qf.genre_any == nullptr) == (qf.genre_bits == nullptr),
                       "gemm_topk: a per-query genre test needs both genre_any [b] and the catalog's genre_bits [n]");
        REBERT_REQUIRE((qf.year_lo == nullptr) == (qf.year_hi == nullptr) && (qf.year_lo == nullptr) == (qf.year == nullptr),
                       "gemm_topk: a per-query year test needs year_lo and year_hi [b] and the catalog's year [n]");
    }
    const bool has_qf = qf.genre_any || qf.year_lo;
    REBERT_REQUIRE(cat && cat->rows && (cat->dtype == REBERT_BF16 || cat->dtype == REBERT_F32), "gemm_topk: the catalog of record must be fp32 or bf16");
    REBERT_REQUIRE(qbf16 && q64 && plan && workspace && out_rows && out_scores && out_count && out_status && cat->norm64,
                   "gemm_topk: null argument");
    const bool shadow = op->dtype == REBERT_I8;
    REBERT_REQUIRE(!shadow || (qscale && qeps && op->n == cat->n && op->d == cat->d && op->row_base == cat->row_base),
                   "gemm_topk: int8 operands need query scales / bounds and a shadow of the same shape as the catalog");
    REBERT_REQUIRE((excl_row_ptr == nullptr) == (excl_col == nullptr), "gemm_topk: exclusion CSR needs both arrays");
    const bool large = plan->k > kLargeK0;                   // long lists: their own selection and exact-pass kernels
    REBERT_REQUIRE(!large || (plan->k < plan->kc && plan->kc <= kLargeKcMax && plan->cand_cap > 0),
                   "gemm_topk: plan k=%d kc=%d is not a long-list plan", plan->k, plan->kc);
    GemmWorkspace w = carve(workspace, plan);
    if (workspace_bytes < w.bytes) { set_error("gemm_topk: workspace %zu < %zu", workspace_bytes, w.bytes); return REBERT_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int b = plan->b;
    const int64_t tiles = (cat->n + BN - 1) / BN;
    const int64_t s_tiles = plan->sample_rows / BN;
    const int64_t stride = tiles / s_tiles;                  // sample tile j = global tile j * stride

    REBERT_CUDA(cudaMemsetAsync(w.cand_count, 0, (size_t)b * 4, st));
    REBERT_CUDA(cudaMemsetAsync(out_status, 0, (size_t)b * 4, st));

    // 1. sample scores
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.b = b;
    p.num_rt = (int)s_tiles;
    p.tile0 = 0;
    p.tile_stride = stride;
    p.out = w.sample;
    p.out_ld = plan->sample_rows;
    p.qscale = qscale;
    set_pred(p, cat, nullptr);                   // the sample keeps every row; the predicate is applied by the selector
    rc = launch_gemm<MODE_STORE>(op, qbf16, p, st);
    if (rc != REBERT_OK) return rc;
    // 2. thresholds
    const int keys_in_smem = plan->sample_rows <= 48 * 1024;
    const size_t tsmem = keys_in_smem ? (size_t)plan->sample_rows * 4 : 16;
    { int rc__ = raise_smem_limit(select_threshold_kernel); if (rc__ != REBERT_OK) return rc__; }
    GemmParams pf;
    memset(&pf, 0, sizeof(pf));
    set_pred(pf, cat, row_filter);
    select_threshold_kernel<<<b, 256, tsmem, st>>>(w.sample, keys_in_smem, plan->sample_rows, cat->n, cat->row_base, 0, stride,
                                                   plan->sample_rank, pf.pred, pf.has_pred, qf, has_qf ? 1 : 0, excl_row_ptr, excl_col,
                                                   w.tau);
    REBERT_CUDA(cudaGetLastError());
    // 3. full pass with fused filter
    memset(&p, 0, sizeof(p));
    p.b = b;
    p.num_rt = (int)tiles;
    p.tile0 = 0;
    p.tile_stride = 1;
    p.tau = w.tau;
    p.cand = w.cand;
    p.cand_count = w.cand_count;
    p.cand_cap = plan->cand_cap;
    p.status = out_status;
    p.qscale = qscale;
    set_pred(p, cat, row_filter);
    p.qf = qf;
    rc = has_qf ? launch_gemm<MODE_FILTER, true>(op, qbf16, p, st) : launch_gemm<MODE_FILTER>(op, qbf16, p, st);
    if (rc != REBERT_OK) return rc;
    // 4. per-query candidate selection
    if (large) {
        int gcap = 2;
        while (gcap < 2 * plan->kc) gcap <<= 1;
        { int rc__ = raise_smem_limit(select_candidates_large_kernel); if (rc__ != REBERT_OK) return rc__; }
        select_candidates_large_kernel<<<b, kSelLargeThreads, (size_t)gcap * 8, st>>>(w.cand, w.cand_count, plan->cand_cap, plan->kc, gcap,
                                                                                      cat->row_base, excl_row_ptr, excl_col, w.tau,
                                                                                      w.cand_keys, out_status);
    } else {
        int p2 = 2;
        while (p2 < plan->cand_cap) p2 <<= 1;
        const size_t csmem = (size_t)(p2 + 1024) * 8;        // survivors + the bucket-selected top set
        { int rc__ = raise_smem_limit(select_candidates_kernel); if (rc__ != REBERT_OK) return rc__; }
        select_candidates_kernel<<<b, 512, csmem, st>>>(w.cand, w.cand_count, plan->cand_cap, plan->kc, cat->row_base, excl_row_ptr,
                                                        excl_col, w.tau, w.cand_keys, out_status);
    }
    REBERT_CUDA(cudaGetLastError());
    // 5. exact pass; near-ties come back as margin = -inf and are re-run by the caller
    if (large)
        rc = finalize_large_launch(cat, q64, w.cand_keys, b, plan->kc, plan->k, out_rows, out_scores, out_count, w.margin, st,
                                   shadow ? 2.0 : 4.0);
    else
        rc = finalize_launch(cat, q64, w.cand_keys, b, plan->kc, plan->k, out_rows, out_scores, out_count, w.margin, st,
                             /*exact_order=*/false, shadow ? 2.0 : 4.0);
    if (rc != REBERT_OK) return rc;
    if (shadow) {
        // int8 operands: the margin (exact k-th - fast score of the worst kept candidate - 2 x the largest |fast - exact| seen on
        // the candidates) must clear the query's own 6-sigma model bound (rebert_query_quantize_i8)
        margin_status_eps_kernel<<<(b + 255) / 256, 256, 0, st>>>(w.margin, qeps, b, out_status);
        REBERT_CUDA(cudaGetLastError());
        return REBERT_OK;
    }
    // The margin already has 4 x (largest observed |fast - exact| over the kc candidates) subtracted (finalize.cu), which
    // calibrates the bf16 rounding of the query; on top require the model bound for that rounding, 3 sigma with
    // sigma = 2^-9 / sqrt(3 d) for a spread-out unit vector, plus the fp32 accumulation term.
    const double eps = 3.0 * 0.001953125 / sqrt(3.0 * (double)cat->d) + 64.0 * 5.96e-8;
    margin_status_kernel<<<(b + 255) / 256, 256, 0, st>>>(w.margin, eps, b, out_status);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}


extern "C" {

REBERT_API int rebert_gemm_scores_i8(const rebert_catalog_t* shadow, const void* q8, const float* qscale, int32_t b, int64_t row0,
                                     int64_t nrows, float* out, rebert_stream stream) {
    int rc = check_gemm_catalog(shadow, "gemm_scores_i8");
    if (rc != REBERT_OK) return rc;
    REBERT_REQUIRE(shadow->dtype == REBERT_I8 && q8 && qscale && out && b > 0 && nrows > 0, "gemm_scores_i8: bad arguments");
    REBERT_REQUIRE(row0 % BN == 0 && nrows % BN == 0 && row0 >= 0, "gemm_scores_i8: row0 and nrows must be multiples of %d", BN);
    REBERT_REQUIRE(((uintptr_t)out & 15) == 0, "gemm_scores_i8: out must be 16-byte aligned");
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.b = b;
    p.num_rt = (int)(nrows / BN);
    p.tile0 = row0 / BN;
    p.tile_stride = 1;
    p.out = out;
    p.out_ld = nrows;
    p.qscale = qscale;
    set_pred(p, shadow, nullptr);
    return launch_gemm<MODE_STORE>(shadow, q8, p, (cudaStream_t)stream);
}

REBERT_API int rebert_gemm_topk_filtered(const rebert_catalog_t* cat, const void* qbf16, const double* q64, const int64_t* excl_row_ptr,
                                         const int32_t* excl_col, const rebert_filter_t* row_filter,
                                         const rebert_query_filter_t* query_filter, const rebert_gemm_plan_t* plan, void* workspace,
                                         size_t workspace_bytes, int64_t* out_rows, double* out_scores, int32_t* out_count,
                                         int32_t* out_status, rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->dtype == REBERT_BF16, "gemm_topk: the bf16 tensor-core path needs a bf16 catalog");
    return gemm_topk_impl(cat, cat, qbf16, nullptr, nullptr, q64, excl_row_ptr, excl_col, row_filter, query_filter, plan, workspace,
                          workspace_bytes, out_rows, out_scores, out_count, out_status, stream);
}

REBERT_API int rebert_gemm_topk(const rebert_catalog_t* cat, const void* qbf16, const double* q64, const int64_t* excl_row_ptr,
                                const int32_t* excl_col, const rebert_filter_t* row_filter, const rebert_gemm_plan_t* plan,
                                void* workspace, size_t workspace_bytes,
                                int64_t* out_rows, double* out_scores, int32_t* out_count, int32_t* out_status,
                                rebert_stream stream) {
    return rebert_gemm_topk_filtered(cat, qbf16, q64, excl_row_ptr, excl_col, row_filter, nullptr, plan, workspace, workspace_bytes,
                                     out_rows, out_scores, out_count, out_status, stream);
}

REBERT_API int rebert_gemm_topk_i8_filtered(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const void* q8, const float* qscale,
                                            const double* qeps, const double* q64, const int64_t* excl_row_ptr, const int32_t* excl_col,
                                            const rebert_filter_t* row_filter, const rebert_query_filter_t* query_filter,
                                            const rebert_gemm_plan_t* plan, void* workspace, size_t workspace_bytes, int64_t* out_rows,
                                            double* out_scores, int32_t* out_count, int32_t* out_status, rebert_stream stream) {
    REBERT_REQUIRE(shadow && shadow->dtype == REBERT_I8, "gemm_topk_i8: shadow must be an int8 prefilter shadow");
    return gemm_topk_impl(cat, shadow, q8, qscale, qeps, q64, excl_row_ptr, excl_col, row_filter, query_filter, plan, workspace,
                          workspace_bytes, out_rows, out_scores, out_count, out_status, stream);
}

REBERT_API int rebert_gemm_topk_i8(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const void* q8, const float* qscale,
                                   const double* qeps, const double* q64, const int64_t* excl_row_ptr, const int32_t* excl_col,
                                   const rebert_filter_t* row_filter, const rebert_gemm_plan_t* plan, void* workspace,
                                   size_t workspace_bytes, int64_t* out_rows, double* out_scores, int32_t* out_count,
                                   int32_t* out_status, rebert_stream stream) {
    return rebert_gemm_topk_i8_filtered(cat, shadow, q8, qscale, qeps, q64, excl_row_ptr, excl_col, row_filter, nullptr, plan, workspace,
                                        workspace_bytes, out_rows, out_scores, out_count, out_status, stream);
}

}  // extern "C"
