// Shared host/device helpers for the rebert_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/rebert_b200.h"

namespace rebert {

// ---------------------------------------------------------------- errors (host) -------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);

#define REBERT_CUDA(call)                                                   \
    do {                                                                    \
        cudaError_t e__ = (call);                                           \
        if (e__ != cudaSuccess) return ::rebert::cuda_fail(e__, #call);     \
    } while (0)

#define REBERT_REQUIRE(cond, ...)                                           \
    do {                                                                    \
        if (!(cond)) { ::rebert::set_error(__VA_ARGS__); return REBERT_ERR_INVALID; } \
    } while (0)

int num_sms();
int max_optin_smem();
// Raise a kernel's dynamic shared-memory limit to the device ceiling (opt-in max minus the kernel's static shared
// memory), once per kernel.  Always the same constant, so concurrent callers cannot race each other's launches.
int raise_smem_limit_impl(const void* kern);
template <typename K> static inline int raise_smem_limit(K kern) { return raise_smem_limit_impl((const void*)kern); }
// host_api.cu -> catalog.cu / finalize.cu (internal launchers)
int stage_query_launch(const float* q_host, int d, int ld, float* qn32, double* qn64, const int32_t* excl_host, int n_excl,
                       int32_t* excl_dev, cudaStream_t st);   // launched with programmatic dependent launch, like every kernel of a request

// ---------------------------------------------------------------- layout --------------------
// A stored row is LANES * CPL chunks of 16 bytes: LANES lanes of a warp each own CPL chunks.
struct RowLayout {
    int esize;   // bytes per element
    int epc;     // elements per 16-byte chunk
    int lanes;   // lanes per row (2..32, power of two)
    int cpl;     // chunks per lane
    int ld;      // padded row stride in elements
};
RowLayout row_layout(int d, int dtype);

// ---------------------------------------------------------------- candidate keys ------------
// key = (orderable(score) << 32) | (0xFFFFFFFF - local_row): a larger key is a better candidate under
// (score desc, row asc).  0 is "empty" and sorts below every real key (NaN scores are never packed).
__host__ __device__ __forceinline__ uint32_t f32_orderable(float f) {
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    uint32_t b; memcpy(&b, &f, 4);
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float orderable_f32(uint32_t o) {
    uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t row) {
    return ((uint64_t)f32_orderable(score) << 32) | (uint64_t)(0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ float key_score(uint64_t k) { return orderable_f32((uint32_t)(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_row(uint64_t k) { return 0xFFFFFFFFu - (uint32_t)k; }

// Control word 3 of a streaming workspace: rows the gated fast pass fetched from the catalog of record, summed over
// launches.  The merge that zeroes the other control words after every launch leaves it alone (rebert_gate_fetches).
constexpr int kCtlGateFetches = 3;
// Control words 20 and 21: the ticket of the gate's seed kernel (its last CTA resets it), and the bound that kernel wrote
// into the grid-wide hint at the last gated launch (orderable fp32 bits, 0 = none).  The merges leave word 21 alone too, so
// it can be read after the request (tests/test_gpu_gate_seed.py).
constexpr int kCtlSeedTicket = 20, kCtlSeedBound = 21;
__host__ __device__ __forceinline__ bool ctl_survives_merge(int w) { return w == kCtlGateFetches || w == kCtlSeedBound; }

// ---------------------------------------------------------------- debug build ---------------
// -DREBERT_DEBUG (robot_ebert_b200/build.py --debug -> librebert_b200_debug.so, loaded when REBERT_DEBUG=1) turns on
// device-side bounds assertions at every computed index the kernels write through; compute-sanitizer is not available on
// the GPU pool this was developed on, so tools/sanitize_small.py drives the debug library over small and ragged cases.
#if defined(REBERT_DEBUG) && defined(__CUDACC__)
#define REBERT_ASSERT(cond)                                                                                              \
    do {                                                                                                                 \
        if (!(cond)) {                                                                                                   \
            printf("REBERT_ASSERT failed: %s  at %s:%d  (block %d, thread %d)\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
                   (int)threadIdx.x);                                                                                    \
            __trap();                                                                                                    \
        }                                                                                                                \
    } while (0)
#else
#define REBERT_ASSERT(cond) do { } while (0)
#endif

#ifdef __CUDACC__
// ---------------------------------------------------------------- device: filter ------------
struct DevFilter {
    const uint32_t* exclude_bitmap;
    const int32_t*  exclude_rows;
    const uint32_t* genre_bits;
    const uint16_t* year;
    int32_t  n_exclude;
    uint32_t genre_any;
    uint32_t year_lo, year_hi;
    int64_t  row_base;
};
DevFilter make_filter(const rebert_filter_t* f, int64_t row_base);

// true iff a sorted int32 list contains v
__device__ __forceinline__ bool sorted_contains(const int32_t* __restrict__ a, int n, int32_t v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        int32_t x = __ldg(a + mid);
        if (x < v) lo = mid + 1; else hi = mid;
    }
    return lo < n && __ldg(a + lo) == v;
}

// same search on a list staged in shared memory (plain loads, ~30-cycle steps instead of L2 round trips)
__device__ __forceinline__ bool sorted_contains_smem(const int32_t* a, int n, int32_t v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo < n && a[lo] == v;
}

// Evaluated only for rows that beat the running threshold, so its cost is off the streaming path.
// excl_s: the exclusion list staged in shared memory by the caller, or nullptr to search the global copy.
__device__ __forceinline__ bool row_allowed(const DevFilter& f, uint32_t local_row, const int32_t* excl_s = nullptr) {
    if (f.exclude_bitmap && ((__ldg(f.exclude_bitmap + (local_row >> 5)) >> (local_row & 31)) & 1u)) return false;
    if (f.n_exclude > 0) {
        const int32_t g = (int32_t)(f.row_base + local_row);
        if (excl_s ? sorted_contains_smem(excl_s, f.n_exclude, g) : sorted_contains(f.exclude_rows, f.n_exclude, g)) return false;
    }
    if (f.genre_bits && (__ldg(f.genre_bits + local_row) & f.genre_any) == 0) return false;
    if (f.year) {
        uint32_t y = __ldg(f.year + local_row);
        if (y < f.year_lo || y > f.year_hi) return false;
    }
    return true;
}

// ---------------------------------------------------------------- device: misc --------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// bf16 pair packed in a 32-bit word -> two fp32 (exact)
__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// element c of a stored row as double
template <typename T> __device__ __forceinline__ double elem_f64(const T* row, int c);
template <> __device__ __forceinline__ double elem_f64<float>(const float* row, int c) { return (double)row[c]; }
template <> __device__ __forceinline__ double elem_f64<__nv_bfloat16>(const __nv_bfloat16* row, int c) {
    return (double)__bfloat162float(row[c]);
}

// ---------------------------------------------------------------- programmatic dependent launch
// The kernels of one request (normalize -> gemv_topk -> finalize -> exchange) run back to back on one stream.  Launched
// with the programmatic-serialization attribute, a kernel's CTAs are placed and run their global-memory-free preamble
// while the previous kernel drains; pdl_wait() then blocks until that kernel has completed and its writes are visible.
// Rule kept by every kernel here: NO global memory access before pdl_wait().  pdl_trigger() lets the next kernel in.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- device: mbarrier / bulk copy
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst_smem)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// Block-wide bitonic sort, descending, of a power-of-two array of u64 keys in shared memory.
__device__ __forceinline__ void block_bitonic_sort_desc(uint64_t* a, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                int ixj = i ^ j;
                if (ixj > i) {
                    uint64_t x = a[i], y = a[ixj];
                    bool desc = (i & k) == 0;
                    if (desc ? (x < y) : (x > y)) { a[i] = y; a[ixj] = x; }
                }
            }
            __syncthreads();
        }
    }
}
#endif  // __CUDACC__

#ifdef __CUDACC__
// Launch `kern` so that it may start while the previous kernel of the stream is still draining (see pdl_wait above).
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#endif

}  // namespace rebert
