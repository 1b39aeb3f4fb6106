// Catalog store, query / profile preparation, subset + dense scoring, synthetic generator.
// Reference sites: src/backend/app/constants.py:55-56 (catalog), lib.py:51-52 (profile = mean of unit rows),
// lib.py:105-106 (subset scoring).  All of these are one-pass HBM-bound or tiny kernels.
#include <stdarg.h>

#include <mutex>
#include <unordered_set>

#include "exchange.cuh"
#include "request.cuh"

namespace rebert {

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return REBERT_ERR_CUDA;
}
// Opt-in shared-memory ceiling of the device.  Kernels always raise their limit to THIS constant: the attribute is a
// per-function global, so setting a per-call size would race between concurrent callers.
int max_optin_smem() {
    static int cached = 0;                       // one process drives one GPU model; benign if two threads race to fill it
    if (cached) return cached;
    int dev = 0, v = 227 * 1024;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cached = v;
    return v;
}
int raise_smem_limit_impl(const void* kern) {
    static std::mutex mu;
    static std::unordered_set<const void*> done;
    std::lock_guard<std::mutex> lock(mu);
    if (done.count(kern)) return REBERT_OK;
    cudaFuncAttributes a;
    REBERT_CUDA(cudaFuncGetAttributes(&a, kern));
    REBERT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin_smem() - (int)a.sharedSizeBytes));
    done.insert(kern);
    return REBERT_OK;
}
int num_sms() {
    static int cached = 0;
    if (cached) return cached;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cached = sms;
    return sms;
}

RowLayout row_layout(int d, int dtype) {
    RowLayout L;
    L.esize = dtype == REBERT_BF16 ? 2 : (dtype == REBERT_I8 ? 1 : 4);
    L.epc = 16 / L.esize;
    int chunks = (d * L.esize + 15) / 16;
    if (chunks <= 16) {
        int lanes = 2;
        while (lanes < chunks) lanes <<= 1;
        L.lanes = lanes;
        L.cpl = 1;
    } else {
        L.lanes = 32;
        L.cpl = (chunks + 31) / 32;
    }
    L.ld = L.lanes * L.cpl * L.epc;
    return L;
}

DevFilter make_filter(const rebert_filter_t* f, int64_t row_base) {
    DevFilter d;
    memset(&d, 0, sizeof(d));
    d.row_base = row_base;
    if (f) {
        d.exclude_bitmap = f->exclude_bitmap;
        d.exclude_rows = f->n_exclude > 0 ? f->exclude_rows : nullptr;
        d.n_exclude = f->exclude_rows ? f->n_exclude : 0;
        d.genre_bits = f->genre_bits;
        d.genre_any = f->genre_any;
        d.year = f->year;
        d.year_lo = f->year_lo;
        d.year_hi = f->year_hi;
    }
    return d;
}

// ------------------------------------------------------------------------------------------------
// device side of the synthetic generator: must stay bit-identical to robot_ebert_b200/synth.py
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ float synth_value(uint64_t seed, uint64_t row, uint32_t d, uint32_t c, int scale_rows) {
    uint64_t h = splitmix64(seed * 0xD6E8FEB86659FD93ull + row * (uint64_t)d + c);
    int s = (int)(h & 0xFFFF) + (int)((h >> 16) & 0xFFFF) + (int)((h >> 32) & 0xFFFF) + (int)(h >> 48);
    float v = __fmul_rn((float)(s - 131070), (float)(1.0 / 37837.2273));
    if (scale_rows) {
        int e = (int)(splitmix64((seed ^ 0xA0761D6478BD642Full) + row) % 9ull) - 4;
        v = __fmul_rn(v, __int_as_float((127 + e) << 23));
    }
    return v;
}
__device__ __forceinline__ uint16_t f32_to_bf16_rne(float f) {
    uint32_t b = __float_as_uint(f);
    return (uint16_t)((b + 0x7FFFu + ((b >> 16) & 1u)) >> 16);
}

template <typename T> __device__ __forceinline__ T store_cvt(float v);
template <> __device__ __forceinline__ float store_cvt<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 store_cvt<__nv_bfloat16>(float v) {
    return __ushort_as_bfloat16(f32_to_bf16_rne(v));
}

template <typename T>
__global__ void synth_rows_kernel(uint64_t seed, int64_t row0, int64_t n, int d, int ld, int scale_rows, T* __restrict__ rows) {
    int64_t total = n * (int64_t)ld;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = i / ld;
        int c = (int)(i - r * ld);
        float v = c < d ? synth_value(seed, (uint64_t)(row0 + r), (uint32_t)d, (uint32_t)c, scale_rows) : 0.0f;
        rows[i] = store_cvt<T>(v);
    }
}

template <typename T>
__global__ void store_rows_kernel(const float* __restrict__ src, int64_t n, int d, int ld, T* __restrict__ rows) {
    int64_t total = n * (int64_t)ld;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = i / ld;
        int c = (int)(i - r * ld);
        rows[i] = store_cvt<T>(c < d ? src[r * d + c] : 0.0f);
    }
}

// One warp per row: fp64 sum of squares of the stored values (sklearn row_norms, zero -> 1).
template <typename T>
__global__ void norms_kernel(const T* __restrict__ rows, int64_t n, int ld, float* __restrict__ inv_norm,
                             double* __restrict__ norm64) {
    int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += nwarps) {
        const T* row = rows + r * ld;
        double acc = 0.0;
        for (int c = lane; c < ld; c += 32) {
            double x = elem_f64<T>(row, c);
            acc = fma(x, x, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) {
            double nrm = sqrt(acc);
            if (nrm == 0.0) nrm = 1.0;
            norm64[r] = nrm;
            inv_norm[r] = (float)(1.0 / nrm);
        }
    }
}

// One CTA per query.
__global__ void query_normalize_kernel(const float* __restrict__ q, int d, int ld, float* __restrict__ qn32,
                                       double* __restrict__ qn64, __nv_bfloat16* __restrict__ qnbf16) {
    __shared__ double red[32];
    pdl_trigger();                                   // the scoring kernel may place its CTAs; it waits for our results
    const float* src = q + (int64_t)blockIdx.x * d;
    double acc = 0.0;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        double x = (double)src[c];
        acc = fma(x, x, acc);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
        v = warp_sum(v);
        if (threadIdx.x == 0) red[0] = v;
    }
    __syncthreads();
    double nrm = sqrt(red[0]);
    if (nrm == 0.0) nrm = 1.0;
    for (int c = threadIdx.x; c < ld; c += blockDim.x) {
        double v = c < d ? (double)src[c] / nrm : 0.0;
        if (qn64) qn64[(int64_t)blockIdx.x * ld + c] = v;
        if (qn32) qn32[(int64_t)blockIdx.x * ld + c] = (float)v;
        if (qnbf16) qnbf16[(int64_t)blockIdx.x * ld + c] = __ushort_as_bfloat16(f32_to_bf16_rne((float)v));
    }
}

// int8 prefilter shadow: one warp per row, two passes over the (cache-resident) row: max|x| -> scale, then quantise,
// accumulate the squared quantisation error in fp64 and fold max_r err_r / ||x_r|| into one device double.
template <typename T>
__global__ void quantize_i8_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t n, int d, int ld,
                                   int ld8, int8_t* __restrict__ out, float* __restrict__ factor,
                                   unsigned long long* __restrict__ max_err_bits) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double worst = 0.0;
    for (int64_t r = warp0; r < n; r += nwarps) {
        const T* row = rows + r * ld;
        float mx = 0.f;
        for (int c = lane; c < d; c += 32) mx = fmaxf(mx, fabsf((float)elem_f64<T>(row, c)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float scale = mx > 0.f ? mx / 127.f : 1.f;
        double err2 = 0.0;
        for (int c = lane; c < ld8; c += 32) {
            int q = 0;
            if (c < d) {
                const float x = (float)elem_f64<T>(row, c);
                q = __float2int_rn(x / scale);
                q = max(-127, min(127, q));
                const double e = (double)x - (double)q * (double)scale;
                err2 = fma(e, e, err2);
            }
            out[r * ld8 + c] = (int8_t)q;
        }
        err2 = warp_sum(err2);
        if (lane == 0) {
            const double nrm = norm64[r];
            factor[r] = (float)((double)scale / nrm);
            worst = fmax(worst, sqrt(err2) / nrm);
        }
    }
    if (lane == 0 && worst > 0.0) atomicMax(max_err_bits, (unsigned long long)__double_as_longlong(worst));   // >= 0: bit order == numeric order
}

// Request staging for the host-buffer entry point: ONE CTA reads the raw query and the exclusion list straight from
// the caller's pinned host block (zero-copy over PCIe, no copy-engine operation in front of the kernels), normalises the
// query exactly as query_normalize_kernel does (same per-thread and reduction order => same bits) and drops the
// exclusion list into device scratch for the scoring kernel.  (Helpers in request.cuh.)
__global__ void __launch_bounds__(256) stage_query_kernel(const float* __restrict__ q_host, int d, int ld, float* __restrict__ qn32,
                                                          double* __restrict__ qn64, const int32_t* __restrict__ excl_host,
                                                          int n_excl, int32_t* __restrict__ excl_dev) {
    extern __shared__ __align__(16) float s_src[];   // [d]
    __shared__ double red[32];
    pdl_trigger();
    pdl_wait();
    fetch_query_zero_copy(q_host, d, s_src);
    copy_list_zero_copy(excl_host, n_excl, excl_dev);
    __syncthreads();
    const double nrm = query_norm_256(s_src, d, red);
    for (int c = threadIdx.x; c < ld; c += blockDim.x) {
        double v = c < d ? (double)s_src[c] / nrm : 0.0;
        qn64[c] = v;
        qn32[c] = (float)v;
    }
}

int stage_query_launch(const float* q_host, int d, int ld, float* qn32, double* qn64, const int32_t* excl_host, int n_excl,
                       int32_t* excl_dev, cudaStream_t st) {
    REBERT_CUDA(launch_pdl(stage_query_kernel, dim3(1), dim3(256), (size_t)d * sizeof(float), st, q_host, d, ld, qn32, qn64,
                           excl_host, n_excl, excl_dev));
    return REBERT_OK;
}

// One CTA per user (profile_accumulate_cta, request.cuh): the user's entries (local row, weight, row norm) are staged in
// shared memory in blocks; each thread owns 16-byte chunks of the row with fp64 accumulators and walks the entries in CSR
// order — a fixed summation order, so the profile is deterministic — with four row loads in flight.
// Entries outside this shard are skipped (their partial sums come from the owning rank through the exchange).
template <typename T, bool DIV>
__global__ void __launch_bounds__(256) profile_accumulate_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t n,
                                                                 int64_t row_base, int ld, const int64_t* __restrict__ row_ptr,
                                                                 const int32_t* __restrict__ col, const float* __restrict__ w,
                                                                 double* __restrict__ sum64, double* __restrict__ wsum) {
    const int u = blockIdx.x;
    const int64_t e0 = row_ptr[u], e1 = row_ptr[u + 1];
    profile_accumulate_cta<T, DIV>(rows, norm64, n, row_base, ld, col + e0, w ? w + e0 : nullptr, (int)(e1 - e0),
                                   sum64 + (int64_t)u * ld, wsum + u);
}

// Single liked-rows request (host-buffer entry point): ONE CTA reads the liked rows (+ weights) and the exclusion list
// zero-copy from the caller's pinned block, builds this shard's fp64 partial profile with the very arithmetic of
// profile_accumulate_kernel<T, true> (sklearn's divide-first order), on a row shard exchanges the partials with the peers
// (exchange.cuh, summed in rank order) and divides by the weight sum: qn32 / qn64 are ready for the scoring kernel.
// Replaces an H2D copy + accumulate + (all-reduce) + finalize.
template <typename T>
__global__ void __launch_bounds__(256) stage_profile_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t n,
                                                            int64_t row_base, int ld, const int32_t* __restrict__ liked_host,
                                                            const float* __restrict__ w_host, int n_liked,
                                                            const int32_t* __restrict__ excl_host, int n_excl, int32_t* __restrict__ excl_dev,
                                                            double* __restrict__ sum64, double* __restrict__ wsum,
                                                            float* __restrict__ qn32, double* __restrict__ qn64, Exchange x) {
    // a kernel that waits for a peer lets its dependents in only after that wait (see finalize_published_kernel)
    if (x.world <= 1) pdl_trigger();
    pdl_wait();
    // One GPU: the grid splits the row's 16-byte column chunks (one SM's fp64 unit made an 82-row profile a 20 us step); every
    // CTA owns its columns from the accumulation to the division.  Row shard: one CTA, the exchange needs the whole vector.
    constexpr int EPC = RowChunk<T>::EPC;
    const int chunks = ld / EPC;
    const int lo = (int)((int64_t)chunks * blockIdx.x / gridDim.x), hi = (int)((int64_t)chunks * (blockIdx.x + 1) / gridDim.x);
    if (blockIdx.x == 0) copy_list_zero_copy(excl_host, n_excl, excl_dev);
    profile_accumulate_cta<T, true, 16>(rows, norm64, n, row_base, ld, liked_host, w_host, n_liked, sum64, wsum, lo, hi);
    __syncthreads();
    if (x.world > 1) {
        exchange_profile(x, ld, sum64, sum64);
        pdl_trigger();
        __syncthreads();
    }
    const double ws = wsum[0];
    for (int c = lo * EPC + threadIdx.x; c < hi * EPC; c += blockDim.x) {
        const double v = ws != 0.0 ? sum64[c] / ws : 0.0;
        qn64[c] = v;
        qn32[c] = (float)v;
    }
}

int stage_profile_launch(const rebert_catalog_t* cat, const int32_t* liked_host, const float* w_host, int n_liked, const int32_t* excl_host,
                         int n_excl, int32_t* excl_dev, double* sum64, double* wsum, float* qn32, double* qn64, const Exchange* x,
                         cudaStream_t st) {
    Exchange xe;
    memset(&xe, 0, sizeof(xe));
    if (x) xe = *x;
    const int chunks = cat->ld * (cat->dtype == REBERT_F32 ? 4 : 2) / 16;
    int grid = (x && x->world > 1) ? 1 : (chunks + 31) / 32;                 // a warp's worth of column chunks per CTA
    if (grid > 16) grid = 16;
    if (grid < 1) grid = 1;
    if (cat->dtype == REBERT_F32)
        REBERT_CUDA(launch_pdl(stage_profile_kernel<float>, dim3(grid), dim3(256), 0, st, (const float*)cat->rows, cat->norm64, cat->n,
                               cat->row_base, cat->ld, liked_host, w_host, n_liked, excl_host, n_excl, excl_dev, sum64, wsum, qn32, qn64, xe));
    else
        REBERT_CUDA(launch_pdl(stage_profile_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, st, (const __nv_bfloat16*)cat->rows, cat->norm64,
                               cat->n, cat->row_base, cat->ld, liked_host, w_host, n_liked, excl_host, n_excl, excl_dev, sum64, wsum, qn32,
                               qn64, xe));
    return REBERT_OK;
}

__global__ void profile_finalize_kernel(const double* __restrict__ sum64, const double* __restrict__ wsum, int ld,
                                        float* __restrict__ p32, double* __restrict__ p64,
                                        __nv_bfloat16* __restrict__ pbf16) {
    int u = blockIdx.x;
    double ws = wsum[u];
    for (int c = threadIdx.x; c < ld; c += blockDim.x) {
        int64_t i = (int64_t)u * ld + c;
        double v = ws != 0.0 ? sum64[i] / ws : 0.0;
        if (p64) p64[i] = v;
        if (p32) p32[i] = (float)v;
        if (pbf16) pbf16[i] = __ushort_as_bfloat16(f32_to_bf16_rne((float)v));
    }
}

// One warp per (user, candidate): fp64 dot / norm64.
template <typename T>
__global__ void score_subset_kernel(const T* __restrict__ rows, const double* __restrict__ norm64, int64_t n,
                                    int64_t row_base, int ld, const double* __restrict__ p64, int b,
                                    const int32_t* __restrict__ sub_rows, int m, double* __restrict__ out) {
    int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (warp >= (int64_t)b * m) return;
    int u = (int)(warp / m), j = (int)(warp % m);
    int64_t r = (int64_t)sub_rows[j] - row_base;
    double acc = 0.0;
    if (r >= 0 && r < n) {
        const T* row = rows + r * ld;
        const double* p = p64 + (int64_t)u * ld;
        const double nrm = norm64[r];
        for (int c = lane; c < ld; c += 32) acc = fma(p[c], elem_f64<T>(row, c) / nrm, acc);   // sklearn's order: unit row first
        acc = warp_sum(acc);
    } else {
        acc = nan("");
    }
    if (lane == 0) out[(int64_t)u * m + j] = acc;
}

// One warp per catalog row, looping over the (few) queries: the materialised score matrix of lib.py:51 in fp32.
template <typename T>
__global__ void scores_dense_kernel(const T* __restrict__ rows, const float* __restrict__ inv_norm, int64_t n, int ld,
                                    const float* __restrict__ q32, int b, float* __restrict__ out) {
    int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += nwarps) {
        const T* row = rows + r * ld;
        float inv = inv_norm[r];
        for (int u = 0; u < b; ++u) {
            const float* q = q32 + (int64_t)u * ld;
            float acc = 0.0f;
            for (int c = lane; c < ld; c += 32) acc = fmaf(q[c], (float)elem_f64<T>(row, c), acc);
            acc = warp_sum(acc);
            if (lane == 0) out[(int64_t)u * n + r] = acc * inv;
        }
    }
}

// Exact-fallback sweep: every allowed row whose fast fp32 score reaches `threshold` is appended (unordered) to out_rows.
// Only used when a candidate list could not prove the result (mass ties in fp64 that fp32 rounding breaks).
template <typename T>
__global__ void collect_above_kernel(const T* __restrict__ rows, const float* __restrict__ inv_norm, int64_t n, int ld,
                                     const float* __restrict__ q32, DevFilter filter, float threshold,
                                     int32_t* __restrict__ out_rows, int cap, int32_t* __restrict__ out_count) {
    int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += nwarps) {
        const T* row = rows + r * ld;
        float acc = 0.0f;
        for (int c = lane; c < ld; c += 32) acc = fmaf(q32[c], (float)elem_f64<T>(row, c), acc);
        acc = warp_sum(acc) * inv_norm[r];
        if (lane == 0 && acc >= threshold && row_allowed(filter, (uint32_t)r)) {
            const int idx = atomicAdd(out_count, 1);
            if (idx < cap) out_rows[idx] = (int32_t)(filter.row_base + r);
        }
    }
}

static int grid_for(int64_t work_items, int block) {
    int64_t g = (work_items + block - 1) / block;
    int64_t cap = (int64_t)num_sms() * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace rebert

using namespace rebert;

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

REBERT_API int rebert_abi_version(void) { return REBERT_ABI_VERSION; }
REBERT_API const char* rebert_last_error(void) { return g_err; }

REBERT_API int rebert_check_device(void) {
    int dev = 0, major = 0;
    REBERT_CUDA(cudaGetDevice(&dev));
    REBERT_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) {
        set_error("device %d has compute capability %d.x; this library carries sm_100a code only", dev, major);
        return REBERT_ERR_DEVICE;
    }
    return REBERT_OK;
}

REBERT_API int rebert_catalog_layout(int64_t n, int32_t d, int32_t dtype, int32_t* ld, size_t* rows_bytes) {
    REBERT_REQUIRE(n >= 0 && d > 0, "catalog_layout: n=%lld d=%d", (long long)n, d);
    REBERT_REQUIRE(dtype == REBERT_F32 || dtype == REBERT_BF16 || dtype == REBERT_I8, "catalog_layout: dtype %d", dtype);
    RowLayout L = row_layout(d, dtype);
    if (ld) *ld = L.ld;
    if (rows_bytes) *rows_bytes = (size_t)n * L.ld * L.esize;
    return REBERT_OK;
}

REBERT_API int rebert_catalog_store_rows(const float* src, int64_t n, int32_t d, int32_t dtype, void* rows, int32_t ld,
                              rebert_stream stream) {
    REBERT_REQUIRE(src && rows && n >= 0 && d > 0 && ld >= d, "catalog_store_rows: bad arguments");
    if (n == 0) return REBERT_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int g = grid_for(n * ld, 256);
    if (dtype == REBERT_F32) store_rows_kernel<float><<<g, 256, 0, st>>>(src, n, d, ld, (float*)rows);
    else if (dtype == REBERT_BF16) store_rows_kernel<__nv_bfloat16><<<g, 256, 0, st>>>(src, n, d, ld, (__nv_bfloat16*)rows);
    else REBERT_REQUIRE(false, "catalog_store_rows: dtype %d", dtype);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_catalog_norms(const void* rows, int64_t n, int32_t ld, int32_t dtype, float* inv_norm, double* norm64,
                         rebert_stream stream) {
    REBERT_REQUIRE(rows && inv_norm && norm64 && n >= 0 && ld > 0, "catalog_norms: bad arguments");
    if (n == 0) return REBERT_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int g = grid_for(n * 32, 256);
    if (dtype == REBERT_F32) norms_kernel<float><<<g, 256, 0, st>>>((const float*)rows, n, ld, inv_norm, norm64);
    else if (dtype == REBERT_BF16) norms_kernel<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)rows, n, ld, inv_norm, norm64);
    else REBERT_REQUIRE(false, "catalog_norms: dtype %d", dtype);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_catalog_quantize_i8(const rebert_catalog_t* src, void* out_rows, int32_t ld8, float* out_factor,
                                          double* out_max_err, rebert_stream stream) {
    REBERT_REQUIRE(src && src->rows && src->norm64 && out_rows && out_factor && out_max_err, "catalog_quantize_i8: null argument");
    REBERT_REQUIRE(src->dtype == REBERT_F32 || src->dtype == REBERT_BF16, "catalog_quantize_i8: source dtype %d", src->dtype);
    RowLayout L8 = row_layout(src->d, REBERT_I8);
    REBERT_REQUIRE(ld8 == L8.ld, "catalog_quantize_i8: ld8=%d does not match rebert_catalog_layout (%d)", ld8, L8.ld);
    cudaStream_t st = (cudaStream_t)stream;
    REBERT_CUDA(cudaMemsetAsync(out_max_err, 0, sizeof(double), st));
    if (src->n == 0) return REBERT_OK;
    const int g = grid_for(src->n * 32, 256);
    if (src->dtype == REBERT_F32)
        quantize_i8_kernel<float><<<g, 256, 0, st>>>((const float*)src->rows, src->norm64, src->n, src->d, src->ld, ld8,
                                                     (int8_t*)out_rows, out_factor, (unsigned long long*)out_max_err);
    else
        quantize_i8_kernel<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)src->rows, src->norm64, src->n, src->d, src->ld,
                                                             ld8, (int8_t*)out_rows, out_factor, (unsigned long long*)out_max_err);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_query_normalize(const float* q, int32_t b, int32_t d, int32_t ld, float* qn32, double* qn64,
                           void* qnbf16, rebert_stream stream) {
    REBERT_REQUIRE(q && b > 0 && d > 0 && ld >= d && (qn32 || qn64 || qnbf16), "query_normalize: bad arguments");
    query_normalize_kernel<<<b, 256, 0, (cudaStream_t)stream>>>(q, d, ld, qn32, qn64, (__nv_bfloat16*)qnbf16);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_profile_accumulate(const rebert_catalog_t* cat, const int64_t* row_ptr, const int32_t* col, const float* w,
                              int32_t b, double* sum64, double* wsum, rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && cat->norm64 && row_ptr && col && sum64 && wsum && b > 0,
                   "profile_accumulate: bad arguments");
    REBERT_REQUIRE(cat->ld * (cat->dtype == REBERT_BF16 ? 2 : 4) <= kProfMaxIter * 256 * 16, "profile_accumulate: rows of %d elements are too long",
                   cat->ld);
    cudaStream_t st = (cudaStream_t)stream;
    // few users: element-wise division like sklearn's normalize(); large batches: one reciprocal per liked row (1 ulp apart)
    const bool div = b <= 8;
#define REBERT_PROFILE_LAUNCH(TT, DD)                                                                                  \
    profile_accumulate_kernel<TT, DD><<<b, 256, 0, st>>>((const TT*)cat->rows, cat->norm64, cat->n, cat->row_base, cat->ld, \
                                                         row_ptr, col, w, sum64, wsum)
    if (cat->dtype == REBERT_F32) { if (div) REBERT_PROFILE_LAUNCH(float, true); else REBERT_PROFILE_LAUNCH(float, false); }
    else { if (div) REBERT_PROFILE_LAUNCH(__nv_bfloat16, true); else REBERT_PROFILE_LAUNCH(__nv_bfloat16, false); }
#undef REBERT_PROFILE_LAUNCH
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_profile_finalize(const double* sum64, const double* wsum, int32_t b, int32_t ld, float* p32, double* p64,
                            void* pbf16, rebert_stream stream) {
    REBERT_REQUIRE(sum64 && wsum && b > 0 && ld > 0, "profile_finalize: bad arguments");
    profile_finalize_kernel<<<b, 256, 0, (cudaStream_t)stream>>>(sum64, wsum, ld, p32, p64, (__nv_bfloat16*)pbf16);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_score_subset(const rebert_catalog_t* cat, const double* p64, int32_t b, const int32_t* sub_rows, int32_t m,
                        double* out, rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && cat->norm64 && p64 && sub_rows && out && b > 0 && m > 0, "score_subset: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t warps = (int64_t)b * m;
    int g = (int)((warps * 32 + 255) / 256);
    if (cat->dtype == REBERT_F32)
        score_subset_kernel<float><<<g, 256, 0, st>>>((const float*)cat->rows, cat->norm64, cat->n, cat->row_base, cat->ld,
                                                      p64, b, sub_rows, m, out);
    else
        score_subset_kernel<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)cat->rows, cat->norm64, cat->n,
                                                              cat->row_base, cat->ld, p64, b, sub_rows, m, out);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_scores_dense(const rebert_catalog_t* cat, const float* q32, int32_t b, float* out, rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && cat->inv_norm && q32 && out && b > 0, "scores_dense: bad arguments");
    if (cat->n == 0) return REBERT_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int g = grid_for(cat->n * 32, 256);
    if (cat->dtype == REBERT_F32)
        scores_dense_kernel<float><<<g, 256, 0, st>>>((const float*)cat->rows, cat->inv_norm, cat->n, cat->ld, q32, b, out);
    else
        scores_dense_kernel<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)cat->rows, cat->inv_norm, cat->n, cat->ld,
                                                              q32, b, out);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_collect_above(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, float threshold,
                                    int32_t* out_rows, int32_t cap, int32_t* out_count, rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && cat->inv_norm && qn32 && out_rows && out_count && cap > 0, "collect_above: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    REBERT_CUDA(cudaMemsetAsync(out_count, 0, sizeof(int32_t), st));
    if (cat->n == 0) return REBERT_OK;
    DevFilter f = make_filter(filter, cat->row_base);
    int g = grid_for(cat->n * 32, 256);
    if (cat->dtype == REBERT_F32)
        collect_above_kernel<float><<<g, 256, 0, st>>>((const float*)cat->rows, cat->inv_norm, cat->n, cat->ld, qn32, f, threshold,
                                                       out_rows, cap, out_count);
    else
        collect_above_kernel<__nv_bfloat16><<<g, 256, 0, st>>>((const __nv_bfloat16*)cat->rows, cat->inv_norm, cat->n, cat->ld, qn32,
                                                               f, threshold, out_rows, cap, out_count);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

REBERT_API int rebert_synth_rows(uint64_t seed, int64_t row0, int64_t n, int32_t d, int32_t scale_rows, int32_t dtype, void* rows,
                      int32_t ld, rebert_stream stream) {
    REBERT_REQUIRE(rows && n >= 0 && d > 0 && ld >= d, "synth_rows: bad arguments");
    if (n == 0) return REBERT_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int g = grid_for(n * ld, 256);
    if (dtype == REBERT_F32) synth_rows_kernel<float><<<g, 256, 0, st>>>(seed, row0, n, d, ld, scale_rows, (float*)rows);
    else if (dtype == REBERT_BF16)
        synth_rows_kernel<__nv_bfloat16><<<g, 256, 0, st>>>(seed, row0, n, d, ld, scale_rows, (__nv_bfloat16*)rows);
    else REBERT_REQUIRE(false, "synth_rows: dtype %d", dtype);
    REBERT_CUDA(cudaGetLastError());
    return REBERT_OK;
}

}  // extern "C"
