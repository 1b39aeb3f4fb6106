// Single-query fused score + mask + top-k  (reference: lib.py:51-55 with one query / one profile).
//
// HBM-bound: every catalog byte is read exactly once.  Design (see DESIGN.md §kernels):
//   * persistent grid, one CTA per SM, 8 consumer warps + 1 producer warp;
//   * the producer streams contiguous row tiles (and the matching inv_norm slice) into a ring of shared-memory
//     stages with 1-D TMA bulk copies (cp.async.bulk, SASS UBLKCP) completing on mbarriers, L2 evict-first;
//   * a row is LANES*CPL 16-byte chunks; the LANES lanes that share a row each keep their CPL chunks of the query in
//     registers, so the inner loop is conflict-free LDS.128 + FFMA and never touches global memory;
//   * every warp keeps its running top-kc as packed 64-bit keys in registers (kc/32 per lane); a row is looked at
//     again only if it beats the warp's threshold (one FSETP per row), and only then is the filter evaluated;
//   * lower bounds of the kc-th best score ("hints") are shared inside the CTA and, sparsely, across the grid, so rows
//     that cannot make the final list are dropped before the insert path: a full warp list's threshold, and the much
//     tighter CTA-wide bound min over the 8 warps of their (kc/8)-th best score;
//   * tiles: static rounds for the first 88 %, then the tail is claimed from a grid-wide counter (four claims in
//     flight per producer), because SMs stream at unequal speeds and equal static shares finish up to 10 % apart;
//   * at the end the 8 warp lists are rank-merged through shared memory into one sorted list per CTA, and the last
//     CTA to finish (atomic ticket) merges the per-CTA lists behind two pruning thresholds — one launch per query.
//     The N-long score vector never exists;
//   * REQUEST PATH (rebert_recommend_device): the CTAs only PUBLISH their pruned keys (compacted through one atomic cursor)
//     plus the heads / tails of their lists; a cluster of 8 small CTAs (finalize.cu), placed behind this kernel by
//     programmatic dependent launch and already waiting when the stream ends, selects the kc winners, re-scores them in
//     fp64 on 8 SMs, ranks them, writes the result and runs the NVLink exchange on a row shard;
//   * launched with programmatic stream serialization: no access to memory an earlier kernel of the stream writes before
//     griddepcontrol.wait.  The catalog is immutable, so the producer starts streaming the first tiles BEFORE that wait:
//     the first TMA round trip overlaps the previous kernel's tail (query staging / the previous request's merge).
#include <type_traits>

#include "exchange.cuh"

namespace rebert {

constexpr int kConsumerWarps = 8;
constexpr int kThreads = (kConsumerWarps + 1) * 32;
constexpr int kStageBytes = 48 * 1024;
constexpr int kStages = 4;           // pipeline depth (lowered when shared memory is short); 48 KB x 4 is within 0.3 % of the best
constexpr int kDynTailPct = 12;      // share of the tiles claimed dynamically at the end (balances SMs of unequal speed)
constexpr int kMaxExclSmem = 4096;   // exclusion rows staged in shared memory (larger lists are searched in global memory)

struct GemvParams {
    const void*  rows;
    const float* inv_norm;
    const float* q;        // [ld] fp32
    int64_t      n;
    int64_t      num_tiles;
    int          ld;
    int          d;         // logical columns (int8 shadow: query elements beyond d are zero)
    int          cpl;       // runtime chunks per lane (generic kernel)
    int          tile_rows;
    int          stages;
    int          kc;
    DevFilter    filter;
    uint64_t*    pub_keys;  // [kPubRegions][region_cap] kept keys of all CTAs: CTA b compacts into region b % kPubRegions
    uint64_t*    pub_heads; // [grid, pub_P] the pub_P = ceil(kc / grid) best keys of every CTA (zero padded)
    uint64_t*    pub_tails; // [grid] kc-th key of a CTA whose list is full, else 0
    unsigned*    cursors;   // [kPubRegions] compaction cursors (zero before launch; reset by whoever merges)
    int          pub_P, region_cap;
    uint64_t*    cand_keys; // [kc] final output (rebert_gemv_topk: the last CTA merges)
    unsigned*    counter;   // CTAs finished (zero before launch; the last CTA resets it)
    unsigned*    ghint;     // grid-wide threshold hint, orderable fp32 bits (zero before launch; reset with the counter)
    unsigned*    tile_ctr;  // tail tiles claimed so far (zero before launch; reset with the counter)
    int64_t      static_rounds;  // every CTA takes tiles blockIdx.x + i * grid for i < static_rounds, the rest are claimed
    int          merge_cap; // keys the final merge may hold in shared memory (power of two)
    int          publish_only;  // request path: no ticket, no merge here — the cluster kernel behind this launch takes over
    // gated kernel only (rows / inv_norm above are the int8 gate): the catalog of record a gated row is fetched from
    const void*  xrows;     // [n, x_ld] bf16 / fp32
    const float* xinv;      // [n] its inv_norm
    int          x_ld, x_cpl;   // its padded row length and chunks per lane (32-lane layout)
    double       gate_err;  // max relative row error of the int8 gate rows (rebert_catalog_quantize_i8)
    // the gate's seed: rows i * seed_stride (i < seed_m) are sampled; every CTA publishes its seed_P best into seed_keys
    int64_t      seed_m, seed_stride;
    int          seed_P;
    uint64_t*    seed_keys; // [grid * seed_P]
    int          seed_fold; // gated kernel: run the seed as its prologue (else gate_seed_kernel ran ahead of it)
};

template <typename T> struct Elem;
template <> struct Elem<float> {
    static constexpr int EPC = 4;
    __device__ static __forceinline__ void dot(const uint4& v, const float* q, float& acc) {
        acc = fmaf(__uint_as_float(v.x), q[0], acc);
        acc = fmaf(__uint_as_float(v.y), q[1], acc);
        acc = fmaf(__uint_as_float(v.z), q[2], acc);
        acc = fmaf(__uint_as_float(v.w), q[3], acc);
    }
};
template <> struct Elem<__nv_bfloat16> {
    static constexpr int EPC = 8;
    __device__ static __forceinline__ void dot(const uint4& v, const float* q, float& acc) {
        acc = fmaf(bf16lo(v.x), q[0], acc);
        acc = fmaf(bf16hi(v.x), q[1], acc);
        acc = fmaf(bf16lo(v.y), q[2], acc);
        acc = fmaf(bf16hi(v.y), q[3], acc);
        acc = fmaf(bf16lo(v.z), q[4], acc);
        acc = fmaf(bf16hi(v.z), q[5], acc);
        acc = fmaf(bf16lo(v.w), q[6], acc);
        acc = fmaf(bf16hi(v.w), q[7], acc);
    }
};

// int8 prefilter shadow (rebert_catalog_quantize_i8): 16 elements per chunk, integer dot products (dp4a) against the query
// split into two int8 planes (q ~ dh * hi + dl * lo, dl = dh / 254), exact int32 accumulation.
template <> struct Elem<int8_t> {
    static constexpr int EPC = 16;
    __device__ static __forceinline__ void dot(const uint4&, const float*, float&) {}   // unused: the int8 path has its own loop
    __device__ static __forceinline__ void dot2(const uint4& v, const uint32_t* q, int& hi, int& lo) {
        hi = __dp4a((int)v.x, (int)q[0], hi); lo = __dp4a((int)v.x, (int)q[4], lo);
        hi = __dp4a((int)v.y, (int)q[1], hi); lo = __dp4a((int)v.y, (int)q[5], lo);
        hi = __dp4a((int)v.z, (int)q[2], hi); lo = __dp4a((int)v.z, (int)q[6], lo);
        hi = __dp4a((int)v.w, (int)q[3], hi); lo = __dp4a((int)v.w, (int)q[7], lo);
    }
};

// The fast score of one row, the same arithmetic wherever it is formed (the plain kernels and the gated kernel's fetch):
// lane cl holds the row's chunks j * LANES + cl; chunk j accumulates into a0 (j even) or a1 (j odd) in element order
// with fmaf; then a0 + a1, the xor-shuffle tree over the row's LANES lanes, and the caller's multiply by inv_norm.
template <typename T>
__device__ __forceinline__ void chunk_dot(const uint4& v, const float* q, int j, float& a0, float& a1) {
    if (j & 1) Elem<T>::dot(v, q, a1);
    else       Elem<T>::dot(v, q, a0);
}
template <int LANES>
__device__ __forceinline__ float row_sum(float a0, float a1) {
    float s = a0 + a1;
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

// Gated kernel: <q, row> of one row of record (32-lane layout, cpl chunks per lane) read straight from global memory,
// the query from shared memory.  Every lane returns the full sum.  Up to 12 chunks per lane are in flight at once.
template <typename TX>
__device__ __forceinline__ float fetch_row_dot(const uint4* __restrict__ row, const float* q_smem, int cpl, int lane) {
    constexpr int EPC = Elem<TX>::EPC;
    constexpr int kBatch = 12;
    float a0 = 0.f, a1 = 0.f;
    for (int j0 = 0; j0 < cpl; j0 += kBatch) {
        uint4 v[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u)
            if (j0 + u < cpl) v[u] = __ldg(row + (j0 + u) * 32 + lane);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
            if (j0 + u < cpl) {
                const int j = j0 + u;
                float qq[EPC];
                const float4* qs = (const float4*)(q_smem + (j * 32 + lane) * EPC);
#pragma unroll
                for (int e = 0; e < EPC / 4; ++e) {
                    const float4 f = qs[e];
                    qq[e * 4 + 0] = f.x; qq[e * 4 + 1] = f.y; qq[e * 4 + 2] = f.z; qq[e * 4 + 3] = f.w;
                }
                chunk_dot<TX>(v[u], qq, j, a0, a1);
            }
        }
    }
    return row_sum<32>(a0, a1);
}

// One element of the int8 query planes: qv ~ dh * h + dl * l (the consumers' registers and the gate's delta use this).
// The residual qv - h * dh is rounded once (fmaf), so the planes do not depend on whether the compiler contracts it; the
// tests' exact model of S (tests/int8_score_model.py) rounds it the same way.
__device__ __forceinline__ void quant_planes(float qv, float dh, float dl, int& h, int& l) {
    h = __float2int_rn(qv / dh);
    h = max(-127, min(127, h));
    l = __float2int_rn(fmaf(-dh, (float)h, qv) / dl);
    l = max(-127, min(127, l));
}

// The int8 arithmetic, one definition for the streaming kernel and the gate's seed (gate_seed_kernel).
// Plane steps from max |q|: dh = max|q| / 127, dl = dh / 254.
__device__ __forceinline__ void i8_steps(float qmax, float& dh, float& dl) {
    dh = qmax > 0.f ? qmax / 127.f : 1.f;
    dl = dh / 254.f;
}
// Lane cl's query registers: per chunk j (elements (j * LANES + cl) * 16 ...), 4 words of the hi plane, then 4 of the lo plane.
template <int CPL, int LANES>
__device__ __forceinline__ void i8_query_regs(const float* __restrict__ q, int d, int cl, float dh, float dl, uint32_t* qi) {
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            uint32_t ph = 0, pl = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int idx = (j * LANES + cl) * 16 + w * 4 + b;
                const float qv = idx < d ? __ldg(q + idx) : 0.f;
                int h, l;
                quant_planes(qv, dh, dl, h, l);
                ph |= (uint32_t)(h & 0xFF) << (8 * b);
                pl |= (uint32_t)(l & 0xFF) << (8 * b);
            }
            qi[j * 8 + w] = ph;
            qi[j * 8 + 4 + w] = pl;
        }
    }
}
// Four rows at once (8 independent dp4a chains): pr[u] points at row u's first chunk of this lane; on return this lane's
// partial int32 sums against both planes.
template <int CPL, int LANES>
__device__ __forceinline__ void i8_partial4(const uint4* const (&pr)[4], const uint32_t* qi, int (&hs)[4], int (&ls)[4]) {
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        uint4 x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) x[u] = pr[u][j * LANES];
#pragma unroll
        for (int u = 0; u < 4; ++u) Elem<int8_t>::dot2(x[u], qi + j * 8, hs[u], ls[u]);
    }
}
// Rows narrower than 32 lanes: 8 shuffle reductions over the row's LANES lanes; every lane of the row holds its exact sums.
template <int CPL, int LANES>
__device__ __forceinline__ void i8_dot4(const uint4* const (&pr)[4], const uint32_t* qi, int (&hs)[4], int (&ls)[4]) {
    i8_partial4<CPL, LANES>(pr, qi, hs, ls);
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            hs[u] += __shfl_xor_sync(0xffffffffu, hs[u], o);
            ls[u] += __shfl_xor_sync(0xffffffffu, ls[u], o);
        }
    }
}
// 32-lane rows: the 8 partial sums are reduced by a transposing butterfly instead of 8 separate 5-level trees (10 shuffles
// instead of 40).  At each of the first three levels a lane keeps half of its sums and adds its partner's copy of them, so
// afterwards lane L holds sum 4 b4 + 2 b3 + b2 (its lane bits) over the 8 lanes that share those bits; two more levels
// complete it over the warp, and one swap across lane bit 4 pairs each row's hi sum with its lo sum.  On return lane L holds
// the exact sums (hs, ls) of row i8_row(L).  Integer sums are exact, so they equal the trees' bit for bit.
__device__ __forceinline__ int i8_row(int lane) { return (lane >> 2) & 3; }
template <int CPL>
__device__ __forceinline__ void i8_dot4_32(const uint4* const (&pr)[4], const uint32_t* qi, int lane, int& hs, int& ls) {
    int h[4] = {0, 0, 0, 0}, l[4] = {0, 0, 0, 0};
    i8_partial4<CPL, 32>(pr, qi, h, l);
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
    int w[4];                                            // sums j + 4 b4: hi plane (b4 = 0) or lo plane (b4 = 1) of row j
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = (b4 ? l[j] : h[j]) + __shfl_xor_sync(0xffffffffu, b4 ? h[j] : l[j], 16);
    int x[2];                                            // rows 2 b3 + j
#pragma unroll
    for (int j = 0; j < 2; ++j) x[j] = (b3 ? w[j + 2] : w[j]) + __shfl_xor_sync(0xffffffffu, b3 ? w[j] : w[j + 2], 8);
    int y = (b2 ? x[1] : x[0]) + __shfl_xor_sync(0xffffffffu, b2 ? x[0] : x[1], 4);   // row 2 b3 + b2
    y += __shfl_xor_sync(0xffffffffu, y, 2);
    y += __shfl_xor_sync(0xffffffffu, y, 1);
    const int other = __shfl_xor_sync(0xffffffffu, y, 16);
    hs = b4 ? other : y;
    ls = b4 ? y : other;
}
// The int8 score S of a row from its sums and its factor (gate_factor / the shadow's inv_norm).
__device__ __forceinline__ float i8_score(float dh, float dl, int hs, int ls, float factor) {
    return fmaf(dh, (float)hs, dl * (float)ls) * factor;
}

// The gate's delta for the query actually passed (DESIGN.md §4.5), rounded up to fp32.  With S the int8 score, F the
// fp32 fast score and T = <x, q> / ||x||:
//   |S - T| <= row_err (||q|| + e_q) + e_q      (rows: Cauchy-Schwarz against the planes q~; query: e_q = ||q - q~||)
//   |F - T| <= (elements per lane + 12) 2^-24 ||q||      (CatalogStore.fast_eps, scaled by ||q||)
// plus 32 ulp of (||q|| + e_q)(1 + row_err) for S's own fp32 steps, and 1e-6 ||q|| for forming L - delta in fp32.
__device__ __forceinline__ float gate_delta(double q2, double e2, double row_err, int x_epl) {
    const double qn = sqrt(q2), eq = sqrt(e2);
    const double shadow = row_err * (qn + eq) + eq + 32.0 * 0x1p-24 * (1.0 + row_err) * (qn + eq);
    const double fast = (double)(x_epl + 12) * 0x1p-24 * qn;
    return __double2float_ru((shadow + fast) * (1.0 + 1e-6) + 1e-6 * qn + 1e-30);
}

// Warp-distributed sorted list of M*32 keys: entry e = m*32 + lane, best first.
template <int M>
struct WarpTopK {
    uint64_t keys[M];
    float    thr;   // score of the worst kept entry once the list is full, else -inf

    __device__ __forceinline__ void init() {
#pragma unroll
        for (int m = 0; m < M; ++m) keys[m] = 0;
        thr = -INFINITY;
    }
    // All lanes call with the same (warp-uniform) key.  Rows arrive in ascending order per warp, so a new key
    // never ties-and-wins against a kept one: strict "greater" decides the slot.
    __device__ __forceinline__ void insert(uint64_t key, int lane) {
        int pos = 0;
#pragma unroll
        for (int m = 0; m < M; ++m) pos += __popc(__ballot_sync(0xffffffffu, keys[m] > key));
#pragma unroll
        for (int m = M - 1; m >= 0; --m) {
            uint64_t up = __shfl_up_sync(0xffffffffu, keys[m], 1);
            if (m > 0) {
                uint64_t prev_last = __shfl_sync(0xffffffffu, keys[m - 1], 31);
                if (lane == 0) up = prev_last;
            }
            int e = m * 32 + lane;
            keys[m] = e < pos ? keys[m] : (e == pos ? key : up);
        }
        uint64_t last = __shfl_sync(0xffffffffu, keys[M - 1], 31);
        thr = last ? key_score(last) : -INFINITY;
    }
};

// After an insert: publish the two lower bounds of the kc-th best score this warp can now vouch for (see the kernel).
//   * its own threshold, once its list is full (kc rows of this warp reach it);
//   * the CTA-wide quantile bound: min over the 8 warps of their (kc/8)-th best score (kc rows of this CTA reach it).
// s_wq entries only grow, so a stale read only yields a smaller, still valid bound.
template <int QLANE>
__device__ __forceinline__ void publish_hints(uint64_t key0, float thr, int warp, int lane, unsigned* s_hint, unsigned* s_wq) {
    if (lane == 0 && thr > -INFINITY) atomicMax(s_hint, f32_orderable(thr));
    if (lane == QLANE && key0 != 0) {
        const unsigned mine = (unsigned)(key0 >> 32);
        ((volatile unsigned*)s_wq)[warp] = mine;
        unsigned mn = mine;
#pragma unroll
        for (int w = 0; w < kConsumerWarps; ++w) mn = min(mn, ((volatile unsigned*)s_wq)[w]);
        if (mn) atomicMax(s_hint, mn);
    }
}

// Seed of the gated kernel's grid-wide bound (DESIGN §4.5).  Until a warp's list is full its threshold is -inf, and until
// the CTA's warps hold kc/8 keys each its hint is too, so without a seed the gated kernel reads the row of record of almost
// every row it meets first (~38k rows at kc = 32 on 148 SMs) and later only the kc-th best of the rows ONE CTA has seen.
// The seed runs on 8 warps of every CTA of a grid of one CTA per SM: as the prologue of the gated kernel's consumer warps
// (seed_fold), or as gate_seed_kernel ahead of a gated grid of another size.
//   1. seed_sample: it scores a strided sample of seed_m int8 rows with the streaming kernel's arithmetic (i8_dot4_32 /
//      i8_score); warp w of CTA c takes samples c * 8 + w + t * 8 * grid;
//   2. each warp keeps its seed_P best allowed rows by S (the request's whole filter), each CTA the seed_P best of its warps;
//   3. seed_bound, in the last CTA (ticket): it takes the kc best of those, reads their rows of record, scores them exactly as
//      the gated kernel does (fetch_row_dot, xinv) and writes L0 = the smallest of these kc fast scores into the grid-wide
//      hint and control word 21, then resets the ticket, which tells the other CTAs that the seed is done (seed_wait).
// kc distinct allowed rows have F >= L0, so L0 is a lower bound of the final kc-th best fast score: the meaning the hint
// already has.  Nothing is inserted into any list, so the candidates stay the plain kernel's.  Fewer than kc published keys:
// no bound.  seed_P = 2 ceil(kc / grid) per CTA loses a row of the sample's best kc only where one CTA holds more than that.
constexpr int kSeedWarps = kConsumerWarps;
// The fold is compiled for int8 rows of up to 4 chunks per lane (d <= 2048): at 6 the prologue would make the gated kernel
// spill, so those rows keep gate_seed_kernel.
constexpr int kSeedFoldMaxCpl = 4;
constexpr int kSeedThreads = kSeedWarps * 32;
// shared memory of the seed: [kSeedWarps * 32] each warp's seed_P best (then the kc selected keys), [32] the CTA's seed_P best
constexpr int kSeedSmemKeys = kSeedWarps * 32 + 32;
// barrier of the 8 seed warps alone (the gated kernel's producer warp keeps issuing its first tiles meanwhile)
__device__ __forceinline__ void seed_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kSeedThreads) : "memory"); }

// Steps 1 and 2, then the ticket: true in the last CTA to publish.  Threads 0 .. kSeedThreads - 1; qi / dh / dl are the
// streaming kernel's query planes.
template <int CPL>
__device__ __forceinline__ bool seed_sample(const GemvParams& p, const uint32_t* qi, float dh, float dl, const int32_t* excl_s,
                                            uint64_t* s_keys, int* s_last) {
    uint64_t* s_best = s_keys + kSeedWarps * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int P = p.seed_P;
    if (threadIdx.x < 32) s_best[threadIdx.x] = 0;
    WarpTopK<1> top;
    top.init();
    uint64_t pth = 0;                                              // this warp's seed_P-th best key (0 while it has fewer)
    const int64_t W = (int64_t)gridDim.x * kSeedWarps;
    const int ul = i8_row(lane);
    for (int64_t i0 = (int64_t)blockIdx.x * kSeedWarps + warp; i0 < p.seed_m; i0 += 4 * W) {
        int64_t rr[4];
        const uint4* pr[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t i = i0 + u * W;
            rr[u] = i < p.seed_m ? i * p.seed_stride : -1;
            pr[u] = (const uint4*)p.rows + (size_t)(rr[u] < 0 ? 0 : rr[u]) * (CPL * 32) + lane;
        }
        const int64_t rl = i0 + ul * W < p.seed_m ? (i0 + ul * W) * p.seed_stride : 0;   // this lane's row
        const float fac = __ldg(p.inv_norm + rl);
        int hs, ls;
        i8_dot4_32<CPL>(pr, qi, lane, hs, ls);
        const float s_lane = i8_score(dh, dl, hs, ls, fac);
#pragma unroll
        for (int u = 0; u < 4; ++u) {                              // warp-uniform
            if (rr[u] < 0) continue;
            const float s = __shfl_sync(0xffffffffu, s_lane, 4 * u);
            const uint64_t key = make_key(s, (uint32_t)rr[u]);
            if (key > pth && row_allowed(p.filter, (uint32_t)rr[u], excl_s)) {
                top.insert(key, lane);
                pth = __shfl_sync(0xffffffffu, top.keys[0], P - 1);
            }
        }
    }
    if (lane < P) s_keys[warp * P + lane] = top.keys[0];
    seed_sync();
    // the CTA's seed_P best of its warps' keys (distinct: every sampled row belongs to one warp), by rank counting
    for (int i = threadIdx.x; i < kSeedWarps * P; i += kSeedThreads) {
        const uint64_t key = s_keys[i];
        if (!key) continue;
        int rank = 0;
        for (int j = 0; j < kSeedWarps * P; ++j) rank += s_keys[j] > key;
        if (rank < P) s_best[rank] = key;
    }
    seed_sync();
    if (threadIdx.x < P) p.seed_keys[(size_t)blockIdx.x * P + threadIdx.x] = s_best[threadIdx.x];
    __threadfence();
    seed_sync();
    if (threadIdx.x == 0) *s_last = (atomicAdd(p.counter + kCtlSeedTicket, 1u) == gridDim.x - 1);
    seed_sync();
    return *s_last != 0;
}

// Step 3, in the last CTA: q_smem holds the query [x_ld], buf has room for grid * seed_P keys.
template <typename TX>
__device__ __forceinline__ void seed_bound(const GemvParams& p, const float* q_smem, uint64_t* s_keys, uint64_t* buf, int* s_cnt,
                                           unsigned* s_min) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kc = p.kc;
    __threadfence();
    const int total = (int)gridDim.x * p.seed_P;
    for (int i = threadIdx.x; i < total; i += kSeedThreads) buf[i] = ldcg_u64(p.seed_keys + i);
    if (threadIdx.x == 0) { *s_cnt = 0; *s_min = ~0u; }
    seed_sync();
    uint64_t* sel = s_keys;                                        // [kc <= 256]
    for (int i = threadIdx.x; i < total; i += kSeedThreads) {
        const uint64_t key = buf[i];
        if (!key) continue;
        int rank = 0;
        for (int j = 0; j < total; ++j) rank += buf[j] > key;
        if (rank < kc) { sel[rank] = key; atomicAdd(s_cnt, 1); }
    }
    seed_sync();
    unsigned bound = 0;
    if (*s_cnt == kc) {
        for (int j = warp; j < kc; j += kSeedWarps) {
            const uint32_t lr = key_row(sel[j]);
            const uint4* xr = (const uint4*)((const TX*)p.xrows + (size_t)lr * p.x_ld);
            const float sc = fetch_row_dot<TX>(xr, q_smem, p.x_cpl, lane) * __ldg(p.xinv + lr);
            if (lane == 0) atomicMin(s_min, f32_orderable(sc));
        }
        seed_sync();
        bound = *s_min;
    }
    if (threadIdx.x == 0) {
        if (bound) {
            atomicMax(p.ghint, bound);
            atomicAdd(p.counter + kCtlGateFetches, (unsigned)kc);
        }
        p.counter[kCtlSeedBound] = bound;
        __threadfence();                                           // the bound is visible before the ticket says "done"
        *(volatile unsigned*)(p.counter + kCtlSeedTicket) = 0u;
    }
}

// The other CTAs of a folded seed wait (each warp on its own) until the last CTA has reset the ticket; their own increment
// came first, so a zero ticket cannot be the state before the seed.  The wait is bounded: a CTA that is not co-resident
// with the rest of its grid (another stream's kernel holds SMs) streams on after kSeedWaitNs without the bound, which is
// only slower; a bound that lands later reaches it through the grid-wide hint.
constexpr unsigned long long kSeedWaitNs = 200000;
__device__ __forceinline__ void seed_wait(const GemvParams& p) {
    if ((threadIdx.x & 31) == 0) {
        unsigned long long t0, t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            unsigned v;
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p.counter + kCtlSeedTicket) : "memory");
            if (v == 0u) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > kSeedWaitNs) break;
            __nanosleep(256);
        }
    }
    __syncwarp();
}

// TX = void: the plain kernel (T = the streamed rows' type).  TX = bf16 / float: the GATED kernel — T = int8_t streams the
// catalog's int8 gate, and a row whose int8 score reaches L - delta (L = the warp's pruning bound) is read from the bf16 /
// fp32 catalog of record and scored with the plain kernel's arithmetic, so the keys are the plain kernel's (DESIGN §4.5).
template <typename T, int CPL, int LANES, int M, typename TX = void>
__global__ void __launch_bounds__(kThreads, 1) gemv_topk_kernel(const GemvParams p) {
    constexpr int EPC = Elem<T>::EPC;
    constexpr int RPW = 32 / LANES;              // rows a warp scores at once
    constexpr bool kRegQ = CPL > 0;              // query chunks live in registers
    constexpr bool kI8 = std::is_same<T, int8_t>::value;   // int8 prefilter shadow (register-query variants only)
    constexpr bool kGate = !std::is_void<TX>::value;
    static_assert(!kGate || (kI8 && kRegQ && LANES == 32), "the gated kernel streams 32-lane int8 rows");
    constexpr int QREGS = (kRegQ && !kI8) ? CPL * EPC : 1;
    constexpr int QIREGS = kI8 ? CPL * 8 : 1;    // per chunk: 4 words of the hi plane + 4 of the lo plane
    constexpr int kQuantLane = 4 * M - 1;        // list entry kc/8 - 1 lives in keys[0] of this lane (kc = 32 M)

    extern __shared__ __align__(128) unsigned char smem[];
    const int row_bytes = p.ld * (int)sizeof(T);
    const int tile_bytes = p.tile_rows * row_bytes;
    const int inv_bytes = p.tile_rows * 4;                       // tile_rows is a multiple of 4
    const int stage_stride = tile_bytes + ((inv_bytes + 127) & ~127);
    unsigned char* stage_base = smem;
    uint64_t* full_bar = (uint64_t*)(smem + (size_t)p.stages * stage_stride);
    uint64_t* empty_bar = full_bar + kStages;
    float* q_smem = (float*)(empty_bar + kStages);               // generic kernel: [ld]; gated kernel: [x_ld]
    int32_t* excl_smem = (int32_t*)(q_smem + (kGate ? p.x_ld : (kRegQ ? 0 : p.ld)));
    const bool excl_staged = p.filter.n_exclude > 0 && p.filter.n_exclude <= kMaxExclSmem;
    const int32_t* excl_s = excl_staged ? excl_smem : nullptr;
    // seed_fold: the seed's keys after the staged exclusion list (seed_smem_bytes)
    uint64_t* seed_smem = (uint64_t*)(((uintptr_t)(excl_smem + (excl_staged ? p.filter.n_exclude : 0)) + 7) & ~(uintptr_t)7);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    __shared__ int s_tile[kStages];             // tile held by each stage, written by the producer before it arms the barrier
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kConsumerWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    // Programmatic dependent launch: let the next kernel of the stream place its CTAs as ours retire.
    pdl_trigger();
    // The catalog (rows, inv_norm) is immutable, so the first tiles can be requested BEFORE waiting for the previous kernel
    // of the stream (query staging / profile build / the previous request's merge): the first TMA round trip and the
    // pipeline fill overlap that kernel's tail.  Everything an earlier kernel writes — the query, the exclusion list, the
    // workspace counters — is touched only after pdl_wait().
    const int row_bytes_e = p.ld * (int)sizeof(T);
    int early = 0;                                     // tiles issued before pdl_wait (producer lane only)
    auto issue_tile = [&](int it, int64_t t, uint64_t policy) {
        const int s = it % p.stages;
        s_tile[s] = (int)t;
        const int64_t row0 = t * p.tile_rows;
        const int64_t left = p.n - row0;
        const int nrows = left < p.tile_rows ? (int)left : p.tile_rows;
        const uint32_t bytes = (uint32_t)nrows * (uint32_t)row_bytes_e;
        const uint32_t ibytes = (uint32_t)(nrows & ~3) * 4u;   // tail (<4 rows) is read through __ldg
        unsigned char* dst = stage_base + (size_t)s * stage_stride;
        mbar_arrive_expect_tx(&full_bar[s], bytes + ibytes);
        bulk_g2s(dst, (const unsigned char*)p.rows + row0 * row_bytes_e, bytes, &full_bar[s], policy);
        if (ibytes) bulk_g2s(dst + tile_bytes, p.inv_norm + row0, ibytes, &full_bar[s], policy);
    };
    if (warp == kConsumerWarps && lane == 0) {
        const uint64_t policy = l2_policy_evict_first();
        for (; early < p.stages && early < p.static_rounds; ++early) {
            const int64_t t = blockIdx.x + early * (int64_t)gridDim.x;
            if (t >= p.num_tiles) break;
            issue_tile(early, t, policy);
        }
    }
    pdl_wait();
    if (!kRegQ || kGate) {
        const int qlen = kGate ? p.x_ld : p.ld;
        for (int c = threadIdx.x; c < qlen; c += blockDim.x) q_smem[c] = p.q[c];
    }
    if (excl_staged) {
        for (int c = threadIdx.x; c < p.filter.n_exclude; c += blockDim.x) excl_smem[c] = __ldg(p.filter.exclude_rows + c);
    }
    __shared__ float s_qmax[kConsumerWarps + 1];
    if (kI8) {                                   // max |q| sets the quantisation step of the query planes
        float m = 0.f;
        for (int c = threadIdx.x; c < p.d; c += blockDim.x) m = fmaxf(m, fabsf(__ldg(p.q + c)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) s_qmax[threadIdx.x >> 5] = m;
    }

    WarpTopK<M> top;
    top.init();
    // Threshold hints.  A warp whose list is full has kc rows scoring >= its threshold, so that value bounds the global
    // kc-th best from below and every other warp may drop rows strictly below it (>= keeps equal scores, whose row
    // order is decided later).  Best value per CTA in shared memory, and sparsely grid-wide through one global word.
    // A second, much tighter bound feeds the same word: once every consumer warp holds kc/8 keys, the smallest of the
    // warps' (kc/8)-th best scores is reached by 8 * kc/8 = kc distinct allowed rows of this CTA, so it too bounds the
    // kc-th best from below — and it tracks the kc-th best of ALL rows the CTA has seen, not of one warp's eighth of them.
    // It is recomputed only by a warp that has just inserted (the rare path); the per-tile cost stays one shared load.
    __shared__ unsigned s_hint;
    __shared__ unsigned s_wq[kConsumerWarps];   // orderable score of warp w's (kc/8)-th best key, 0 = not there yet
    __shared__ float s_delta;
    if constexpr (kGate) {
        // delta from the query's own norm and the real error of its two int8 planes (the consumers form the same planes)
        __shared__ double s_red[2][kConsumerWarps + 1];
        __syncthreads();
        float qmax = 0.f;
#pragma unroll
        for (int w = 0; w <= kConsumerWarps; ++w) qmax = fmaxf(qmax, s_qmax[w]);
        const float gdh = qmax > 0.f ? qmax / 127.f : 1.f;
        const float gdl = gdh / 254.f;
        double e2 = 0.0, q2 = 0.0;
        for (int c = threadIdx.x; c < p.d; c += blockDim.x) {
            const float qv = __ldg(p.q + c);
            int h, l;
            quant_planes(qv, gdh, gdl, h, l);
            const double r = (double)qv - ((double)gdh * h + (double)gdl * l);
            e2 = fma(r, r, e2);
            q2 = fma((double)qv, (double)qv, q2);
        }
        e2 = warp_sum(e2);
        q2 = warp_sum(q2);
        if (lane == 0) { s_red[0][warp] = e2; s_red[1][warp] = q2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double se = 0.0, sq = 0.0;
            for (int w = 0; w <= kConsumerWarps; ++w) { se += s_red[0][w]; sq += s_red[1][w]; }
            s_delta = gate_delta(sq, se, p.gate_err, p.x_cpl * Elem<TX>::EPC);
        }
    }
    if (threadIdx.x == 0) s_hint = 0u;
    if (threadIdx.x < kConsumerWarps) s_wq[threadIdx.x] = 0u;
    __syncthreads();

    if (warp == kConsumerWarps) {
        // ===================== producer warp: one elected lane issues the bulk copies =====================
        if (lane == 0) {
            const uint64_t policy = l2_policy_evict_first();
            // SMs do not stream at the same speed (measured: equal shares finish up to 10 % apart), so only the first
            // `static_rounds` rounds are dealt out statically (tile = blockIdx.x + i * grid); the tail tiles are claimed
            // one by one from a grid-wide counter.  Four claims are kept in flight — the first four issued right here —
            // so a claim's L2 round trip is never waited for.  A CTA's tiles still ascend (WarpTopK::insert relies on it).
            const int64_t tail0 = p.static_rounds * (int64_t)gridDim.x;      // first dynamically claimed tile
            const bool has_tail = tail0 < p.num_tiles;
            unsigned c0 = 0, c1 = 0, c2 = 0, c3 = 0;
            if (has_tail) {
                c0 = atomicAdd(p.tile_ctr, 1u); c1 = atomicAdd(p.tile_ctr, 1u);
                c2 = atomicAdd(p.tile_ctr, 1u); c3 = atomicAdd(p.tile_ctr, 1u);
            }
            int it = early;                                                  // stages [0, early) were armed before pdl_wait
            auto issue = [&](int64_t t) {
                const int s = it % p.stages;
                const uint32_t round = (uint32_t)(it / p.stages);
                mbar_wait(&empty_bar[s], (round & 1u) ^ 1u);
                if (t >= p.num_tiles) {                                      // tell the consumers there is nothing more
                    s_tile[s] = -1;
                    mbar_arrive(&full_bar[s]);
                    ++it;
                    return false;
                }
                issue_tile(it, t, policy);
                ++it;
                return true;
            };
            bool more = true;
            for (int64_t i = early; i < p.static_rounds && more; ++i) more = issue(blockIdx.x + i * (int64_t)gridDim.x);
            if (more && !has_tail) more = issue(p.num_tiles);                // static only: post the end marker
            while (more) {
                if (!(more = issue(tail0 + c0))) break;
                c0 = atomicAdd(p.tile_ctr, 1u);
                if (!(more = issue(tail0 + c1))) break;
                c1 = atomicAdd(p.tile_ctr, 1u);
                if (!(more = issue(tail0 + c2))) break;
                c2 = atomicAdd(p.tile_ctr, 1u);
                if (!(more = issue(tail0 + c3))) break;
                c3 = atomicAdd(p.tile_ctr, 1u);
            }
        }
    } else {
        // ===================== consumer warps =====================
        const int sub = lane / LANES;            // which of the warp's RPW rows this lane works on
        const int cl = lane % LANES;             // chunk lane within the row
        float q[QREGS];
        uint32_t qi[QIREGS];
        float dh = 1.f, dl = 1.f;
        if constexpr (kI8) {
            float qmax = 0.f;
#pragma unroll
            for (int w = 0; w <= kConsumerWarps; ++w) qmax = fmaxf(qmax, s_qmax[w]);
            i8_steps(qmax, dh, dl);
            i8_query_regs<CPL, LANES>(p.q, p.d, cl, dh, dl, qi);
        } else if (kRegQ) {
#pragma unroll
            for (int j = 0; j < (kRegQ ? CPL : 0); ++j)
#pragma unroll
                for (int e = 0; e < EPC; ++e) q[j * EPC + e] = __ldg(p.q + (j * LANES + cl) * EPC + e);
        }
        const int cpl = kRegQ ? CPL : p.cpl;
        const int row_chunks = cpl * LANES;
        const float delta = kGate ? s_delta : 0.f;
        unsigned fetched = 0;                    // gated kernel: rows read from the catalog of record (warp-uniform)
        if constexpr (kGate && CPL <= kSeedFoldMaxCpl) {
            if (p.seed_fold) {
                // the seed, while the producer's first tiles are in flight; the last CTA forms the bound, the others wait
                // for it (bounded) and every CTA then streams with it from its first tile
                __shared__ int s_last, s_cnt;
                __shared__ unsigned s_min;
                if (seed_sample<CPL>(p, qi, dh, dl, excl_s, seed_smem, &s_last))
                    seed_bound<TX>(p, q_smem, seed_smem, seed_smem + kSeedSmemKeys, &s_cnt, &s_min);
                else
                    seed_wait(p);
            }
        }

        for (int it = 0;; ++it) {
            const int s = it % p.stages;
            const uint32_t round = (uint32_t)(it / p.stages);
            const unsigned char* st = stage_base + (size_t)s * stage_stride;
            const uint4* tile = (const uint4*)st;
            const float* inv_s = (const float*)(st + tile_bytes);

            // hint for this tile: CTA value, refreshed from / published to the grid-wide word every 8th tile by warp 0
            unsigned hb = *(volatile unsigned*)&s_hint;
            if ((it & 7) == 0) {
                const unsigned g = __ldcg(p.ghint);
                if (g > hb) { hb = g; if (lane == 0) atomicMax(&s_hint, g); }
                else if (warp == 0 && lane == 0 && hb > g) atomicMax(p.ghint, hb);
            }
            const float hint = hb ? orderable_f32(hb) : -INFINITY;

            mbar_wait(&full_bar[s], round & 1u);
            const int64_t t = s_tile[s];               // which tile the producer put into this stage (-1: none left)
            if (t < 0) break;
            const int64_t row0 = t * p.tile_rows;
            const int64_t left = p.n - row0;
            const int nrows = left < p.tile_rows ? (int)left : p.tile_rows;
            const int nrows4 = nrows & ~3;

            if constexpr (kI8 && LANES == 32) {
                // int8 rows are half as long, so a warp has to turn rows around twice as fast to keep up with HBM: FOUR rows
                // per step (8 independent dp4a chains, one butterfly reduction) hide the per-step latency.  Lane L scores
                // row i8_row(L); lanes 0, 4, 8, 12 vote for rows 0..3 in one ballot, whose bits ascend with the rows (which
                // WarpTopK::insert relies on).  Each candidate is re-tested against the list as it stands when its turn comes.
                const int ul = i8_row(lane);
                for (int base = warp; base < nrows; base += 4 * kConsumerWarps) {
                    const uint4* pr[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int r = base + u * kConsumerWarps;
                        pr[u] = tile + (size_t)(r < nrows ? r : 0) * row_chunks + lane;
                    }
                    const int rl = base + ul * kConsumerWarps;     // this lane's row
                    const bool vl = rl < nrows;
                    const float inv = vl ? (rl < nrows4 ? inv_s[rl] : __ldg(p.inv_norm + row0 + rl)) : 0.f;
                    int hs, ls;
                    i8_dot4_32<CPL>(pr, qi, lane, hs, ls);
                    const float sc_lane = i8_score(dh, dl, hs, ls, inv);
                    const bool voter = vl && (lane & 19) == 0;
                    if constexpr (kGate) {
                        // a row of the final list has F >= L, so S >= L - delta: rows below cannot get there
                        unsigned mm = __ballot_sync(0xffffffffu, voter && sc_lane >= fmaxf(top.thr, hint) - delta);
                        while (mm) {
                            const int src = __ffs(mm) - 1;
                            mm &= mm - 1;
                            const float sv = __shfl_sync(0xffffffffu, sc_lane, src);
                            const uint32_t lr = (uint32_t)(row0 + base + i8_row(src) * kConsumerWarps);
                            if (sv >= fmaxf(top.thr, hint) - delta && row_allowed(p.filter, lr, excl_s)) {
                                ++fetched;
                                const uint4* xr = (const uint4*)((const TX*)p.xrows + (size_t)lr * p.x_ld);
                                const float sc = fetch_row_dot<TX>(xr, q_smem, p.x_cpl, lane) * __ldg(p.xinv + lr);
                                if (sc > top.thr && sc >= hint) {
                                    top.insert(make_key(sc, lr), lane);
                                    publish_hints<kQuantLane>(top.keys[0], top.thr, warp, lane, &s_hint, s_wq);
                                }
                            }
                        }
                    } else {
                        unsigned mm = __ballot_sync(0xffffffffu, voter && sc_lane > top.thr && sc_lane >= hint);
                        while (mm) {
                            const int src = __ffs(mm) - 1;
                            mm &= mm - 1;
                            const float sc = __shfl_sync(0xffffffffu, sc_lane, src);
                            const uint32_t lr = (uint32_t)(row0 + base + i8_row(src) * kConsumerWarps);
                            if (sc > top.thr && row_allowed(p.filter, lr, excl_s)) {
                                top.insert(make_key(sc, lr), lane);
                                publish_hints<kQuantLane>(top.keys[0], top.thr, warp, lane, &s_hint, s_wq);
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);
                continue;
            } else if constexpr (kI8) {
                // int8 shadow rows narrower than 32 lanes: RPW rows per lane group, four groups per step
                for (int base = warp * RPW; base < nrows; base += 4 * kConsumerWarps * RPW) {
                    int rr[4];
                    bool vv[4];
                    const uint4* pr[4];
                    int hs[4] = {0, 0, 0, 0}, ls[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        rr[u] = base + sub + u * kConsumerWarps * RPW;
                        vv[u] = rr[u] < nrows;
                        pr[u] = tile + (size_t)(vv[u] ? rr[u] : 0) * row_chunks + cl;
                    }
                    i8_dot4<CPL, LANES>(pr, qi, hs, ls);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {          // u ascending = rows ascending, which WarpTopK::insert relies on
                        const float inv = vv[u] ? (rr[u] < nrows4 ? inv_s[rr[u]] : __ldg(p.inv_norm + row0 + rr[u])) : 0.f;
                        const float sc_lane = i8_score(dh, dl, hs[u], ls[u], inv);
                        unsigned mm = __ballot_sync(0xffffffffu, vv[u] && cl == 0 && sc_lane > top.thr && sc_lane >= hint);
                        while (mm) {
                            const int src = __ffs(mm) - 1;
                            mm &= mm - 1;
                            const float sc = __shfl_sync(0xffffffffu, sc_lane, src);
                            const uint32_t lr = (uint32_t)(row0 + base + u * kConsumerWarps * RPW + src / LANES);
                            if (sc > top.thr && row_allowed(p.filter, lr, excl_s)) {
                                top.insert(make_key(sc, lr), lane);
                                publish_hints<kQuantLane>(top.keys[0], top.thr, warp, lane, &s_hint, s_wq);
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);
                continue;
            }
            // two row groups per step for ILP: rows rA and rB = rA + kConsumerWarps*RPW
            for (int base = warp * RPW; base < nrows; base += 2 * kConsumerWarps * RPW) {
                const int rA = base + sub;
                const int rB = rA + kConsumerWarps * RPW;
                const bool vA = rA < nrows, vB = rB < nrows;
                float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
                const uint4* pa = tile + (size_t)(vA ? rA : 0) * row_chunks + cl;
                const uint4* pb = tile + (size_t)(vB ? rB : 0) * row_chunks + cl;
                if (kRegQ) {                 // (the int8 shadow has its own loop above and never gets here)
#pragma unroll
                    for (int j = 0; j < (kRegQ ? CPL : 0); ++j) {
                        const uint4 va = pa[j * LANES];
                        const uint4 vb = pb[j * LANES];
                        chunk_dot<T>(va, q + j * EPC, j, a0, a1);
                        chunk_dot<T>(vb, q + j * EPC, j, b0, b1);
                    }
                } else {
                    for (int j = 0; j < cpl; ++j) {
                        const uint4 va = pa[j * LANES];
                        const uint4 vb = pb[j * LANES];
                        float qq[EPC];
                        const float4* qs = (const float4*)(q_smem + (j * LANES + cl) * EPC);
#pragma unroll
                        for (int e = 0; e < EPC / 4; ++e) {
                            float4 f = qs[e];
                            qq[e * 4 + 0] = f.x; qq[e * 4 + 1] = f.y; qq[e * 4 + 2] = f.z; qq[e * 4 + 3] = f.w;
                        }
                        chunk_dot<T>(va, qq, j, a0, a1);
                        chunk_dot<T>(vb, qq, j, b0, b1);
                    }
                }
                float sa = row_sum<LANES>(a0, a1), sb = row_sum<LANES>(b0, b1);
                const float ia = vA ? (rA < nrows4 ? inv_s[rA] : __ldg(p.inv_norm + row0 + rA)) : 0.f;
                const float ib = vB ? (rB < nrows4 ? inv_s[rB] : __ldg(p.inv_norm + row0 + rB)) : 0.f;
                sa *= ia;
                sb *= ib;

                // rare path: some row of this step beats the warp threshold.  Row order A(sub 0..), then B(sub 0..)
                // is ascending, which WarpTopK::insert relies on.
                unsigned ma = __ballot_sync(0xffffffffu, vA && cl == 0 && sa > top.thr && sa >= hint);
                while (ma) {
                    const int src = __ffs(ma) - 1;
                    ma &= ma - 1;
                    const float sc = __shfl_sync(0xffffffffu, sa, src);
                    const uint32_t lr = (uint32_t)(row0 + base + src / LANES);
                    REBERT_ASSERT((int64_t)lr < p.n);
                    if (sc > top.thr && row_allowed(p.filter, lr, excl_s)) {
                        top.insert(make_key(sc, lr), lane);
                        publish_hints<kQuantLane>(top.keys[0], top.thr, warp, lane, &s_hint, s_wq);
                    }
                }
                unsigned mb = __ballot_sync(0xffffffffu, vB && cl == 0 && sb > top.thr && sb >= hint);
                while (mb) {
                    const int src = __ffs(mb) - 1;
                    mb &= mb - 1;
                    const float sc = __shfl_sync(0xffffffffu, sb, src);
                    const uint32_t lr = (uint32_t)(row0 + base + kConsumerWarps * RPW + src / LANES);
                    if (sc > top.thr && row_allowed(p.filter, lr, excl_s)) {
                        top.insert(make_key(sc, lr), lane);
                        publish_hints<kQuantLane>(top.keys[0], top.thr, warp, lane, &s_hint, s_wq);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);
        }
        if (kGate && lane == 0 && fetched) atomicAdd(p.counter + kCtlGateFetches, fetched);
    }

    // ===================== CTA merge: 8 sorted warp lists -> one sorted list of kc keys =====================
    __syncthreads();   // every stage has been consumed; the pipeline memory is free to reuse
    uint64_t* lists = (uint64_t*)smem;           // [kConsumerWarps][kc]
    const int kc = p.kc;
    __shared__ int s_kept[kConsumerWarps];       // entries of each warp list that can still matter
    if (warp < kConsumerWarps) {
        // Keys scoring below the best lower bound of the global kc-th best (CTA hint, or the grid-wide word) cannot be in
        // the result: drop them here, so only ~kc of the CTA's 8 kc keys go through the rank merge and reach the final
        // merge.  The lists are sorted, so the dropped keys are a tail and the zero-terminated-list convention holds.
        const unsigned hb = max(*(volatile unsigned*)&s_hint, __ldcg(p.ghint));
        int kept = 0;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const uint64_t key = ((unsigned)(top.keys[m] >> 32) >= hb) ? top.keys[m] : 0;
            lists[warp * kc + m * 32 + lane] = key;
            kept += __popc(__ballot_sync(0xffffffffu, key != 0));
        }
        if (lane == 0) s_kept[warp] = kept;
    }
    __syncthreads();
    uint64_t* merged = lists + kConsumerWarps * kc;      // [kc] this CTA's kept keys, best first, zero padded
    __shared__ unsigned s_base;
    int total = 0;
#pragma unroll
    for (int w = 0; w < kConsumerWarps; ++w) total += s_kept[w];
    const int nkeep = total < kc ? total : kc;
    const int region = blockIdx.x % kPubRegions;
    if (threadIdx.x == 0) s_base = atomicAdd(p.cursors + region, (unsigned)nkeep);      // its round trip overlaps the rank merge below
    for (int i = total + threadIdx.x; i < kc; i += blockDim.x) merged[i] = 0;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        int w = 0, e = i;                        // i-th kept key overall = entry e of warp list w
        while (e >= s_kept[w]) { e -= s_kept[w]; ++w; }
        const uint64_t key = lists[w * kc + e];
        int rank = e;
        for (int o = 0; o < kConsumerWarps; ++o) {
            if (o == w) continue;
            const uint64_t* L = lists + o * kc;
            int lo = 0, hi = s_kept[o];          // count of keys in L greater than key
            while (lo < hi) { int mid = (lo + hi) >> 1; if (L[mid] > key) lo = mid + 1; else hi = mid; }
            rank += lo;
        }
        REBERT_ASSERT(rank >= 0 && w < kConsumerWarps);
        if (rank < kc) merged[rank] = key;
    }
    __syncthreads();
    // publish: the kept keys into the compacted array, the list's head (first pub_P keys) and tail (kc-th key if full)
    {
        REBERT_ASSERT((int)s_base + nkeep <= p.region_cap && p.pub_P * (int)gridDim.x <= kc + 256);
        uint64_t* dst = p.pub_keys + (size_t)region * p.region_cap + s_base;
        for (int i = threadIdx.x; i < nkeep; i += blockDim.x) dst[i] = merged[i];
        for (int j = threadIdx.x; j < p.pub_P; j += blockDim.x) p.pub_heads[(size_t)blockIdx.x * p.pub_P + j] = j < kc ? merged[j] : 0;
        if (threadIdx.x == 0) p.pub_tails[blockIdx.x] = nkeep == kc ? merged[kc - 1] : 0;
    }
    if (p.publish_only) return;                        // request path: the cluster kernel behind this launch merges

    // ===================== rebert_gemv_topk: the last CTA to finish merges what all CTAs kept (no second launch) =========
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    {
        PublishedKeys pub;
        pub.keys = p.pub_keys; pub.cursors = p.cursors; pub.heads = p.pub_heads; pub.tails = p.pub_tails;
        pub.lists = (int)gridDim.x; pub.P = p.pub_P; pub.kc = kc; pub.region_cap = p.region_cap;
        select_winners<16>(pub, p.merge_cap, (uint64_t*)smem, p.cand_keys);
        __syncthreads();
    }
    if (threadIdx.x < 32 && !ctl_survives_merge(threadIdx.x)) p.counter[threadIdx.x] = 0u;   // ticket, hint, tile claims, cursors
}

// The seed ahead of a gated grid that is not one CTA per SM (small catalogs), or whose seed keys do not fit beside the
// pipeline: one CTA per SM, 8 warps, the same seed functions.
template <int CPL, typename TX>
__global__ void __launch_bounds__(kSeedThreads, 1) gate_seed_kernel(const GemvParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    float* q_smem = (float*)smem;                                  // [x_ld] the query, last CTA
    uint64_t* buf = (uint64_t*)(smem + (((size_t)p.x_ld * 4 + 15) & ~(size_t)15));   // [grid * seed_P] published keys, last CTA
    int32_t* excl_smem = (int32_t*)(buf + (size_t)gridDim.x * p.seed_P);
    const bool excl_staged = p.filter.n_exclude > 0 && p.filter.n_exclude <= kMaxExclSmem;
    const int32_t* excl_s = excl_staged ? excl_smem : nullptr;   // a filter test is a chain of dependent loads: keep it on chip
    __shared__ float s_qmax[kSeedWarps];
    __shared__ uint64_t s_keys[kSeedSmemKeys];
    __shared__ int s_last, s_cnt;
    __shared__ unsigned s_min;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();                   // the gated kernel may place its CTAs and start its early TMA as these retire
    pdl_wait();
    if (excl_staged) {
        for (int c = threadIdx.x; c < p.filter.n_exclude; c += blockDim.x) excl_smem[c] = __ldg(p.filter.exclude_rows + c);
    }

    float m = 0.f;
    for (int c = threadIdx.x; c < p.d; c += blockDim.x) m = fmaxf(m, fabsf(__ldg(p.q + c)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_qmax[warp] = m;
    __syncthreads();
    float qmax = 0.f, dh, dl;
#pragma unroll
    for (int w = 0; w < kSeedWarps; ++w) qmax = fmaxf(qmax, s_qmax[w]);
    i8_steps(qmax, dh, dl);
    uint32_t qi[CPL * 8];
    i8_query_regs<CPL, 32>(p.q, p.d, lane, dh, dl, qi);
    if (!seed_sample<CPL>(p, qi, dh, dl, excl_s, s_keys, &s_last)) return;
    for (int c = threadIdx.x; c < p.x_ld; c += blockDim.x) q_smem[c] = p.q[c];
    seed_bound<TX>(p, q_smem, s_keys, buf, &s_cnt, &s_min);
}

// ---------------------------------------------------------------- host side ----------------------------------
// The pipeline shape, the L2 policy, the dynamic tail share, the CTA-wide hint, merge pruning and the early TMA issue are
// fixed: each is the setting measured fastest on the B200 (DESIGN.md §4.1, "Tuning record").
struct GemvLaunch {
    int grid, stages, tile_rows, merge_cap;
    size_t smem;
};

// q_floats: query elements staged in shared memory (generic kernel: ld; gated kernel: the catalog of record's ld);
// seed_bytes: the folded seed's keys (seed_smem_bytes), 0 without
static GemvLaunch plan_gemv(const RowLayout& L, int64_t n, int kc, int q_floats, int n_exclude, size_t seed_bytes = 0) {
    GemvLaunch g;
    const int row_bytes = L.ld * L.esize;
    const int rpw = 32 / L.lanes;
    int tr = kStageBytes / row_bytes;
    const int unit = kConsumerWarps * rpw;           // rows one step of all warps covers
    if (tr >= 2 * unit) tr = (tr / (2 * unit)) * (2 * unit);
    else if (tr >= unit) tr = unit;
    tr &= ~3;
    if (tr < 4) tr = 4;
    // small catalogs: shrink the tile (down to one step of all warps) so the rows spread over more SMs
    const int sms = num_sms();
    while (tr >= 2 * unit && (n + tr - 1) / tr < sms && ((tr / 2) & 3) == 0) tr /= 2;
    g.tile_rows = tr;
    const int tile_bytes = tr * row_bytes;
    const int stage_stride = tile_bytes + ((tr * 4 + 127) & ~127);
    const size_t excl_bytes = (n_exclude > 0 && n_exclude <= kMaxExclSmem) ? (size_t)n_exclude * 4 : 0;
    const size_t fixed = 2 * kStages * sizeof(uint64_t) + (size_t)q_floats * 4 + excl_bytes + 128 + seed_bytes;
    int stages = kStages;
    while (stages > 1 && (size_t)stages * stage_stride + fixed > 220 * 1024) --stages;
    g.stages = stages;
    g.smem = (size_t)stages * stage_stride + fixed;
    size_t merge_bytes = (size_t)(kConsumerWarps + 1) * kc * sizeof(uint64_t);   // 8 warp lists + the CTA's merged list
    if (g.smem < merge_bytes) g.smem = merge_bytes;
    // last-CTA merge buffer (rebert_gemv_topk): a power of two >= max(2 kc, kc + grid), as large as the pipeline memory
    // allows (<= 16384 keys)
    int need = 2 * kc > kc + num_sms() ? 2 * kc : kc + num_sms();
    int cap = 2;
    while (cap < need) cap <<= 1;
    while (cap < 16384 && (size_t)cap * 2 * sizeof(uint64_t) <= g.smem) cap <<= 1;
    if (g.smem < (size_t)cap * sizeof(uint64_t)) g.smem = (size_t)cap * sizeof(uint64_t);
    g.merge_cap = cap;
    const int64_t tiles = (n + tr - 1) / tr;
    int grid = num_sms();
    if (tiles < grid) grid = (int)(tiles > 0 ? tiles : 1);
    g.grid = grid;
    return g;
}

template <typename T, int CPL, int LANES, typename TX = void>
static int launch_gemv_m(const GemvParams& p, const GemvLaunch& g, int kc, cudaStream_t st) {
#define REBERT_LAUNCH_M(MM)                                                                                      \
    {                                                                                                            \
        auto kern = gemv_topk_kernel<T, CPL, LANES, MM, TX>;                                                         \
        { int rc__ = raise_smem_limit(kern); if (rc__ != REBERT_OK) return rc__; }       \
        REBERT_CUDA(launch_pdl(kern, dim3(g.grid), dim3(kThreads), g.smem, st, p));                             \
    }
    switch (kc) {
        case 32: REBERT_LAUNCH_M(1); break;
        case 64: REBERT_LAUNCH_M(2); break;
        case 128: REBERT_LAUNCH_M(4); break;
        case 256: REBERT_LAUNCH_M(8); break;
        default: set_error("gemv_topk: kc=%d is not one of 32/64/128/256", kc); return REBERT_ERR_UNSUPPORTED;
    }
#undef REBERT_LAUNCH_M
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

// int8 prefilter shadow: register-query variants, kc = 256 only (the candidate list must absorb the quantisation error)
template <int CPL, int LANES>
static int launch_gemv_i8_one(const GemvParams& p, const GemvLaunch& g, cudaStream_t st) {
    auto kern = gemv_topk_kernel<int8_t, CPL, LANES, 8>;
    { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
    REBERT_CUDA(launch_pdl(kern, dim3(g.grid), dim3(kThreads), g.smem, st, p));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}
static int launch_gemv_i8(const RowLayout& L, const GemvParams& p, const GemvLaunch& g, cudaStream_t st) {
    if (L.lanes < 32) {
        switch (L.lanes) {
            case 2: return launch_gemv_i8_one<1, 2>(p, g, st);
            case 4: return launch_gemv_i8_one<1, 4>(p, g, st);
            case 8: return launch_gemv_i8_one<1, 8>(p, g, st);
            case 16: return launch_gemv_i8_one<1, 16>(p, g, st);
        }
    }
    switch (L.cpl) {
        case 1: return launch_gemv_i8_one<1, 32>(p, g, st);
        case 2: return launch_gemv_i8_one<2, 32>(p, g, st);
        case 3: return launch_gemv_i8_one<3, 32>(p, g, st);
        case 4: return launch_gemv_i8_one<4, 32>(p, g, st);
        case 6: return launch_gemv_i8_one<6, 32>(p, g, st);
        case 12: return launch_gemv_i8_one<12, 32>(p, g, st);
    }
    set_error("gemv_topk: no int8 kernel for rows of %d chunks per lane", L.cpl);
    return REBERT_ERR_UNSUPPORTED;
}

template <typename T>
static int launch_gemv(const RowLayout& L, const GemvParams& p, const GemvLaunch& g, int kc, cudaStream_t st) {
    if (L.lanes < 32) {
        switch (L.lanes) {
            case 2: return launch_gemv_m<T, 1, 2>(p, g, kc, st);
            case 4: return launch_gemv_m<T, 1, 4>(p, g, kc, st);
            case 8: return launch_gemv_m<T, 1, 8>(p, g, kc, st);
            case 16: return launch_gemv_m<T, 1, 16>(p, g, kc, st);
        }
    }
    switch (L.cpl) {
        case 1: return launch_gemv_m<T, 1, 32>(p, g, kc, st);
        case 2: return launch_gemv_m<T, 2, 32>(p, g, kc, st);
        case 3: return launch_gemv_m<T, 3, 32>(p, g, kc, st);
        case 4: return launch_gemv_m<T, 4, 32>(p, g, kc, st);
        case 6: return launch_gemv_m<T, 6, 32>(p, g, kc, st);
        case 12: return launch_gemv_m<T, 12, 32>(p, g, kc, st);
        default: return launch_gemv_m<T, 0, 32>(p, g, kc, st);
    }
}

static bool use_generic(const RowLayout& L) {
    if (L.lanes < 32) return false;
    switch (L.cpl) { case 1: case 2: case 3: case 4: case 6: case 12: return false; }
    return true;
}

// Gated kernels: the int8 gate streamed by its 32-lane register-query layout, rows of record fetched by 32 lanes.
template <typename TX>
static int launch_gemv_gated(const RowLayout& L8, const GemvParams& p, const GemvLaunch& g, int kc, cudaStream_t st) {
    switch (L8.cpl) {
        case 1: return launch_gemv_m<int8_t, 1, 32, TX>(p, g, kc, st);
        case 2: return launch_gemv_m<int8_t, 2, 32, TX>(p, g, kc, st);
        case 3: return launch_gemv_m<int8_t, 3, 32, TX>(p, g, kc, st);
        case 4: return launch_gemv_m<int8_t, 4, 32, TX>(p, g, kc, st);
        case 6: return launch_gemv_m<int8_t, 6, 32, TX>(p, g, kc, st);
    }
    set_error("gemv_topk: no gated kernel for int8 rows of %d chunks per lane", L8.cpl);
    return REBERT_ERR_UNSUPPORTED;
}

// Rows the gate's seed samples: 1/64 of the catalog, at least 16k and at most 128k (measured on the B200, DESIGN §4.5).
constexpr int64_t kSeedRowsMin = 16384, kSeedRowsMax = 131072, kSeedShare = 64;
static int64_t seed_rows(int64_t n) {
    int64_t m = n / kSeedShare;
    m = m < kSeedRowsMin ? kSeedRowsMin : (m > kSeedRowsMax ? kSeedRowsMax : m);
    return m < n ? m : n;
}
// Keys each seed CTA publishes: twice its share of kc, at most 32.
static int seed_P_for(int kc) {
    const int per = (kc + num_sms() - 1) / num_sms();
    return 2 * per < 32 ? 2 * per : 32;
}
// Shared memory of the folded seed (gemv_topk_kernel's seed_smem): its warps' and CTA's keys, the last CTA's copy of all
// CTAs' keys, 8 bytes of alignment.
static size_t seed_smem_bytes(int kc) { return ((size_t)kSeedSmemKeys + (size_t)num_sms() * seed_P_for(kc)) * sizeof(uint64_t) + 8; }

template <int CPL, typename TX>
static int launch_gate_seed_one(const GemvParams& p, cudaStream_t st) {
    auto kern = gate_seed_kernel<CPL, TX>;
    const int n_excl = p.filter.n_exclude > 0 && p.filter.n_exclude <= kMaxExclSmem ? p.filter.n_exclude : 0;
    const size_t smem = (((size_t)p.x_ld * 4 + 15) & ~(size_t)15) + (size_t)num_sms() * p.seed_P * sizeof(uint64_t) + (size_t)n_excl * 4;
    { int rc = raise_smem_limit(kern); if (rc != REBERT_OK) return rc; }
    REBERT_CUDA(launch_pdl(kern, dim3(num_sms()), dim3(kSeedThreads), smem, st, p));
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}
template <typename TX>
static int launch_gate_seed(const RowLayout& L8, const GemvParams& p, cudaStream_t st) {
    switch (L8.cpl) {
        case 1: return launch_gate_seed_one<1, TX>(p, st);
        case 2: return launch_gate_seed_one<2, TX>(p, st);
        case 3: return launch_gate_seed_one<3, TX>(p, st);
        case 4: return launch_gate_seed_one<4, TX>(p, st);
        case 6: return launch_gate_seed_one<6, TX>(p, st);
    }
    set_error("gemv_topk: no gate seed kernel for int8 rows of %d chunks per lane", L8.cpl);
    return REBERT_ERR_UNSUPPORTED;
}

// The catalog's gate is taken when both its int8 rows and its rows of record are 32-lane layouts and the int8 rows have a
// register-query kernel of at most 6 chunks per lane (d <= 3072; at 12 the gated kernel spills); any other catalog streams
// its own rows (the gate changes which rows are read, never the result).
static bool gate_applies(const rebert_catalog_t* cat) {
    if (cat->dtype == REBERT_I8 || !cat->gate_rows || !cat->gate_factor) return false;
    const RowLayout L8 = row_layout(cat->d, REBERT_I8), L = row_layout(cat->d, cat->dtype);
    return L8.lanes == 32 && L.lanes == 32 && !use_generic(L8) && L8.cpl <= 6;
}

// The int8 shadow has register-query kernels only (launch_gemv_i8): rows of 5 or 7-11 chunks per lane (d = 2049-2560,
// 3073-5632) have none, and such a shadow serves only the batched int8 GEMM.
bool gemv_streams(const rebert_catalog_t* cat) {
    return cat->dtype != REBERT_I8 || !use_generic(row_layout(cat->d, cat->dtype));
}

}  // namespace rebert

using namespace rebert;

extern "C" {

REBERT_API int32_t rebert_candidates_for_k(int32_t k) {
    if (k <= 0) return 0;
    int need = k + 16;                 // margin for the fp32 -> fp64 re-ranking (DESIGN.md §exactness)
    if (need <= 32) return 32;
    if (need <= 64) return 64;
    if (need <= 128) return 128;
    if (need <= 256) return 256;
    return 0;
}

// Workspace layout (kc-INDEPENDENT control words first, so one zero-filled-once workspace serves every kc a thread uses):
//   [0, 128)       32 control words: ticket counter, grid-wide hint, tile-claim counter, -, 16 compaction cursors  (zero
//                  before a launch; whoever merges — the last CTA, or the cluster kernel of the request path — zeroes them)
//   [128, 2176)    tail key of every CTA list (u64 x 256)
//   [2176, ...)    kept keys of all CTAs [16 regions][region_cap] u64; then the list heads [kc + 256] u64; then the keys the
//                  gate's seed CTAs publish [SMs * 32] u64 (their own region: with a folded seed, a CTA may publish its list
//                  while the last seed CTA still reads them)
constexpr size_t kWsCtl = 128, kWsTails = 8 * 256;
static inline int region_cap_for(int kc) { return ((num_sms() + kPubRegions - 1) / kPubRegions) * kc; }
static inline size_t ws_pub_keys(int kc) { return (size_t)kPubRegions * region_cap_for(kc) + (size_t)kc + 256; }

REBERT_API size_t rebert_gemv_workspace_bytes(int64_t n, int32_t kc) {
    (void)n;
    return 128 + kWsCtl + kWsTails + (ws_pub_keys(kc) + (size_t)num_sms() * 32) * sizeof(uint64_t) + 256;
}

REBERT_API int rebert_workspace_reset(void* workspace, size_t workspace_bytes, rebert_stream stream) {
    REBERT_REQUIRE(workspace && workspace_bytes >= 128 + kWsCtl, "workspace_reset: bad arguments");
    REBERT_CUDA(cudaMemsetAsync(workspace, 0, 128 + kWsCtl, (cudaStream_t)stream));
    return REBERT_OK;
}

REBERT_API int rebert_gate_fetches(const void* workspace, size_t workspace_bytes, uint32_t* out_count, rebert_stream stream) {
    REBERT_REQUIRE(workspace && out_count && workspace_bytes >= 128 + kWsCtl, "gate_fetches: bad arguments");
    const unsigned* ctl = (const unsigned*)(((uintptr_t)workspace + 127) & ~(uintptr_t)127);
    REBERT_CUDA(cudaMemcpyAsync(out_count, ctl + kCtlGateFetches, sizeof(uint32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    REBERT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return REBERT_OK;
}

}  // extern "C"

namespace rebert {

int gemv_launch(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, int32_t kc, void* workspace,
                size_t workspace_bytes, uint64_t* cand_keys, const GemvFused* fused, cudaStream_t st) {
    REBERT_REQUIRE(cat && cat->rows && cat->inv_norm && qn32 && workspace && (cand_keys || fused), "gemv_topk: null argument");
    REBERT_REQUIRE(cat->n >= 0 && cat->n < (1ll << 31), "gemv_topk: shard rows %lld out of range", (long long)cat->n);
    REBERT_REQUIRE(cat->dtype == REBERT_F32 || cat->dtype == REBERT_BF16 || cat->dtype == REBERT_I8, "gemv_topk: dtype %d", cat->dtype);
    REBERT_REQUIRE(cat->dtype != REBERT_I8 || kc == 256, "gemv_topk: the int8 prefilter shadow needs kc = 256 (got %d)", kc);
    REBERT_REQUIRE(((uintptr_t)cat->rows & 127) == 0 && ((uintptr_t)cat->inv_norm & 15) == 0,
                   "gemv_topk: catalog rows must be 128-byte and inv_norm 16-byte aligned");
    RowLayout L = row_layout(cat->d, cat->dtype);
    REBERT_REQUIRE(L.ld == cat->ld, "gemv_topk: ld=%d does not match rebert_catalog_layout (%d)", cat->ld, L.ld);
    if (L.ld * L.esize > kStageBytes / 4) {
        set_error("gemv_topk: rows of %d bytes exceed the %d-byte staging limit", L.ld * L.esize, kStageBytes / 4);
        return REBERT_ERR_UNSUPPORTED;
    }
    if (workspace_bytes < rebert_gemv_workspace_bytes(cat->n, kc)) {
        set_error("gemv_topk: workspace %zu < %zu", workspace_bytes, rebert_gemv_workspace_bytes(cat->n, kc));
        return REBERT_ERR_WORKSPACE;
    }
    REBERT_REQUIRE(num_sms() <= 256, "gemv_topk: device has %d SMs, the workspace holds the tails of at most 256 CTA lists", num_sms());
    if (fused) {
        const rebert_catalog_t* xc = fused->exact_cat;
        REBERT_REQUIRE(xc && xc->rows && xc->norm64 && fused->q64 && fused->out_packed, "recommend_device: null argument");
        REBERT_REQUIRE(xc->dtype == REBERT_F32 || xc->dtype == REBERT_BF16, "recommend_device: the catalog of record must be fp32 or bf16");
        REBERT_REQUIRE(xc->n == cat->n && xc->d == cat->d && xc->row_base == cat->row_base, "recommend_device: shadow and catalog differ in shape");
        REBERT_REQUIRE(fused->k > 0 && fused->k <= kc, "recommend_device: k=%d kc=%d", fused->k, kc);
    }
    if (cat->n == 0) {
        if (!fused) {
            REBERT_CUDA(cudaMemsetAsync(cand_keys, 0, (size_t)kc * sizeof(uint64_t), st));
            return REBERT_OK;
        }
        // an empty shard still has to answer (and, on a row shard, to take part in the exchange): run one empty tile
    }
    const bool gated = gate_applies(cat);
    const RowLayout LS = gated ? row_layout(cat->d, REBERT_I8) : L;     // layout of the rows the kernel streams
    if (gated)
        REBERT_REQUIRE(((uintptr_t)cat->gate_rows & 127) == 0 && ((uintptr_t)cat->gate_factor & 15) == 0,
                       "gemv_topk: gate rows must be 128-byte and gate factors 16-byte aligned");
    const int n_excl = (filter && filter->exclude_rows && filter->n_exclude > 0) ? filter->n_exclude : 0;
    GemvLaunch g = plan_gemv(LS, cat->n, kc, gated ? L.ld : (use_generic(L) ? L.ld : 0), n_excl);
    // The seed runs as the gated kernel's prologue when the gated grid is one CTA per SM (the seed's sample-to-CTA mapping),
    // the kernel has the prologue (kSeedFoldMaxCpl) and its keys fit beside the pipeline without a shallower ring; else
    // gate_seed_kernel runs ahead of the gated kernel.
    bool fold = false;
    if (gated && cat->n > 0 && g.grid == num_sms() && LS.cpl <= kSeedFoldMaxCpl) {
        const GemvLaunch gf = plan_gemv(LS, cat->n, kc, L.ld, n_excl, seed_smem_bytes(kc));
        if (gf.stages == g.stages) { g = gf; fold = true; }
    }
    GemvParams p;
    memset(&p, 0, sizeof(p));
    p.rows = gated ? cat->gate_rows : cat->rows;
    p.inv_norm = gated ? cat->gate_factor : cat->inv_norm;
    p.q = qn32;
    p.n = cat->n;
    p.ld = LS.ld;
    p.d = cat->d;
    p.cpl = LS.cpl;
    if (gated) {
        p.xrows = cat->rows;
        p.xinv = cat->inv_norm;
        p.x_ld = L.ld;
        p.x_cpl = L.cpl;
        p.gate_err = cat->gate_err;
    }
    p.tile_rows = g.tile_rows;
    p.num_tiles = (cat->n + g.tile_rows - 1) / g.tile_rows;
    p.stages = g.stages;
    p.kc = kc;
    p.filter = make_filter(filter, cat->row_base);
    unsigned char* ws = (unsigned char*)(((uintptr_t)workspace + 127) & ~(uintptr_t)127);
    p.counter = (unsigned*)ws;
    p.ghint = p.counter + 1;
    p.tile_ctr = p.counter + 2;
    p.cursors = p.counter + 4;
    p.region_cap = region_cap_for(kc);
    p.pub_tails = (uint64_t*)(ws + kWsCtl);
    p.pub_keys = (uint64_t*)(ws + kWsCtl + kWsTails);
    p.pub_heads = p.pub_keys + (size_t)kPubRegions * p.region_cap;
    p.pub_P = (kc + g.grid - 1) / g.grid;
    {
        const int64_t rounds = (p.num_tiles + g.grid - 1) / g.grid;       // static schedule would need this many
        int64_t sr = rounds - (rounds * kDynTailPct + 99) / 100;
        // Each CTA keeps four claims in flight from its first instruction on, so a dynamic tail shorter than a few rounds is
        // swallowed by the CTAs that start first (2264 x 1536: 34 CTAs took all 136 tail tiles and finished 5 us after the
        // rest).  Short launches are dealt out statically.
        if (rounds - sr < 8) sr = rounds;
        if (sr < 1) sr = 1;                                               // the first tile is always blockIdx.x
        p.static_rounds = sr;
    }
    p.cand_keys = cand_keys;
    p.merge_cap = g.merge_cap;
    p.publish_only = fused ? 1 : 0;

    int rc;
    if (gated && cat->n > 0) {                       // the seed's bound in the grid-wide hint
        p.seed_m = seed_rows(cat->n);
        p.seed_stride = cat->n / p.seed_m;
        p.seed_P = seed_P_for(kc);
        p.seed_keys = p.pub_keys + ws_pub_keys(kc);
        p.seed_fold = fold ? 1 : 0;
        if (!fold) {
            rc = cat->dtype == REBERT_F32 ? launch_gate_seed<float>(LS, p, st) : launch_gate_seed<__nv_bfloat16>(LS, p, st);
            if (rc != REBERT_OK) return rc;
        }
    }
    if (cat->dtype == REBERT_I8) rc = launch_gemv_i8(L, p, g, st);
    else if (gated) rc = cat->dtype == REBERT_F32 ? launch_gemv_gated<float>(LS, p, g, kc, st) : launch_gemv_gated<__nv_bfloat16>(LS, p, g, kc, st);
    else rc = cat->dtype == REBERT_F32 ? launch_gemv<float>(L, p, g, kc, st) : launch_gemv<__nv_bfloat16>(L, p, g, kc, st);
    if (rc != REBERT_OK || !fused) return rc;
    // request path: the cluster kernel that selects the winners, runs the exact pass, ranks, writes the result (and exchanges)
    Published pub;
    memset(&pub, 0, sizeof(pub));
    pub.keys.keys = p.pub_keys;
    pub.keys.cursors = p.cursors;
    pub.keys.heads = p.pub_heads;
    pub.keys.tails = p.pub_tails;
    pub.keys.lists = g.grid;
    pub.keys.P = p.pub_P;
    pub.keys.kc = kc;
    pub.keys.region_cap = p.region_cap;
    pub.ctl = p.counter;
    return finalize_published_launch(pub, *fused, cat->row_base, st);
}

}  // namespace rebert

extern "C" {

REBERT_API int rebert_gemv_topk(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, int32_t kc,
                     void* workspace, size_t workspace_bytes, uint64_t* cand_keys, rebert_stream stream) {
    REBERT_REQUIRE(cand_keys, "gemv_topk: null argument");
    return gemv_launch(cat, qn32, filter, kc, workspace, workspace_bytes, cand_keys, nullptr, (cudaStream_t)stream);
}

REBERT_API int rebert_recommend_device(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const float* qn32, const double* qn64,
                                       const rebert_filter_t* filter, int32_t k, int32_t kc, void* workspace, size_t workspace_bytes,
                                       int64_t* out_packed, uint32_t tag, const rebert_exchange_t* exchange, int32_t* err_flag,
                                       rebert_stream stream) {
    REBERT_REQUIRE(cat && qn64 && out_packed, "recommend_device: null argument");
    GemvFused f;
    f.exact_cat = cat;
    f.q64 = qn64;
    f.k = k;
    f.out_packed = (unsigned long long*)out_packed;
    f.tag = tag;
    f.done_flag = nullptr;
    f.done_token = 0;
    Exchange x;
    f.xchg = nullptr;
    if (exchange && exchange->world > 1) {
        int rc = make_exchange(exchange, err_flag, &x);
        if (rc != REBERT_OK) return rc;
        REBERT_REQUIRE(k <= exchange->k_max, "recommend_device: k=%d exceeds the exchange buffer's k_max=%d", k, exchange->k_max);
        f.xchg = &x;
    }
    return gemv_launch(shadow ? shadow : cat, qn32, filter, kc, workspace, workspace_bytes, nullptr, &f, (cudaStream_t)stream);
}

}  // extern "C"
