// Host-buffer entry point: one C call = one request of the reference's hot path (lib.py:43-55) end to end.
// Host pointers in, host pointers out.  The request is packed into the caller's pinned block and read from there by the
// first kernel (zero-copy: no copy-engine operation at all); a staging kernel normalises the query or builds the
// profile; the streaming kernel does score + mask + top-k and a cluster of 8 CTAs placed behind it by programmatic
// dependent launch does the fp64 exact pass, the ranking (+ the NVLink exchange and merge on a row shard) and writes the
// packed result straight into the pinned block; a stream synchronisation ends the call.  The proof loop lives here too: int8
// shadow first when the caller has one, then the plain fast pass with 4x more candidates until the margin proves the ids.
// Scratch (pinned host + device) is provided by the caller, so the library still allocates nothing and concurrent
// callers only need their own scratch + stream (+ their own exchange channel on a row shard).
#include <algorithm>
#include <chrono>

#include "exchange.cuh"

namespace rebert {

// The result block lives in pinned host memory and the exact-pass kernel stores a completion token behind it, so the host
// waits by polling that word instead of synchronising the stream (saves the driver's completion path, a few us per
// request).  true when *flag == token arrived; false after ~20 s (a faulted kernel or a dead peer: the caller then
// synchronises the stream, which reports the error)
static bool poll_done(const volatile uint32_t* flag, uint32_t token) {
    for (int spin = 0; spin < 4096; ++spin) {
        if (*flag == token) return true;
        __builtin_ia32_pause();
    }
    const auto t0 = std::chrono::steady_clock::now();
    while (true) {
        for (int spin = 0; spin < 2048; ++spin) {
            if (*flag == token) return true;
            __builtin_ia32_pause();
        }
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(20)) return false;
    }
}

static double now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static size_t al16(size_t x) { return (x + 15) & ~(size_t)15; }
static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

struct HostLayout {
    // pinned block: request (query | exclusions | liked rows | weights), then the result block, the error word and the
    // in-flight marker
    size_t off_q, off_excl, off_col, off_w, in_bytes, pin_out, out_bytes, pin_err, pin_bytes;
    // device scratch
    size_t off_dexcl, off_qn32, off_qn64, off_sum64, off_wsum, off_ws, ws_bytes, dev_bytes;
};

static HostLayout host_layout(int ld, int d, int n_liked_cap, int n_excl_cap, int k, int kc, int64_t n) {
    HostLayout L;
    L.off_q = 0;
    L.off_excl = al16((size_t)d * 4);
    L.off_col = L.off_excl + al16((size_t)n_excl_cap * 4);
    L.off_w = L.off_col + al16((size_t)n_liked_cap * 4);
    L.in_bytes = L.off_w + al16((size_t)n_liked_cap * 4);
    L.pin_out = al256(L.in_bytes);
    L.out_bytes = (size_t)(2 * k + 2) * 8;
    L.pin_err = L.pin_out + al16(L.out_bytes);
    L.pin_bytes = L.pin_err + 256;
    size_t o = 0;
    L.ws_bytes = rebert_gemv_workspace_bytes(n, kc);
    L.off_ws = o; o += al256(L.ws_bytes);                  // first: its control words are what "zero-filled once" is about
    L.off_dexcl = o; o += al256((size_t)n_excl_cap * 4);
    L.off_qn32 = o; o += al256((size_t)ld * 4);
    L.off_qn64 = o; o += al256((size_t)ld * 8);
    L.off_sum64 = o; o += al256((size_t)ld * 8);
    L.off_wsum = o; o += 256;
    L.dev_bytes = o;
    return L;
}

// 32-bit tag of a request (FNV-1a over 64-bit words): travels with every rank's result so the merge can refuse to combine
// answers to different requests.
static uint32_t request_tag(const void* a, size_t na, const void* b, size_t nb, const void* c, size_t nc, uint64_t salt) {
    uint64_t h = 0xcbf29ce484222325ull ^ salt;
    auto mix = [&](const void* p, size_t nbytes) {
        const unsigned char* s = (const unsigned char*)p;
        size_t i = 0;
        for (; i + 8 <= nbytes; i += 8) { uint64_t v; memcpy(&v, s + i, 8); h = (h ^ v) * 0x100000001b3ull; h ^= h >> 29; }
        for (; i < nbytes; ++i) h = (h ^ s[i]) * 0x100000001b3ull;
    };
    if (a) mix(a, na);
    if (b) mix(b, nb);
    if (c) mix(c, nc);
    uint32_t t = (uint32_t)(h ^ (h >> 32));
    return t ? t : 1u;
}

}  // namespace rebert

using namespace rebert;

extern "C" {

REBERT_API int rebert_recommend_host_scratch(const rebert_catalog_t* cat, int32_t n_liked_cap, int32_t n_exclude_cap, int32_t k,
                                             size_t* pinned_bytes, size_t* device_bytes) {
    REBERT_REQUIRE(cat && k > 0 && n_liked_cap >= 0 && n_exclude_cap >= 0, "recommend_host_scratch: bad arguments");
    HostLayout L = host_layout(cat->ld, cat->d, n_liked_cap, n_exclude_cap, k, 256, cat->n);
    if (pinned_bytes) *pinned_bytes = L.pin_bytes;
    if (device_bytes) *device_bytes = L.dev_bytes;
    return REBERT_OK;
}

REBERT_API int rebert_recommend_host(const rebert_catalog_t* cat, const float* query, const int32_t* liked_rows,
                                     const float* liked_w, int32_t n_liked, const int32_t* exclude_rows, int32_t n_exclude,
                                     const rebert_filter_t* device_filter, int32_t k, int32_t kc, int32_t n_liked_cap,
                                     int32_t n_exclude_cap, void* pinned, size_t pinned_bytes, void* device_scratch,
                                     size_t device_bytes, const rebert_proof_t* proof, const rebert_exchange_t* exchange,
                                     int64_t* out_rows, double* out_scores, int32_t* out_count, rebert_request_info_t* info,
                                     rebert_stream stream) {
    REBERT_REQUIRE(cat && cat->rows && pinned && device_scratch && out_rows && out_scores && out_count, "recommend_host: null argument");
    REBERT_REQUIRE((query != nullptr) != (liked_rows != nullptr), "recommend_host: pass exactly one of query / liked_rows");
    REBERT_REQUIRE(k > 0 && kc >= k && kc <= 256, "recommend_host: k=%d kc=%d", k, kc);
    REBERT_REQUIRE(n_liked >= 0 && n_liked <= n_liked_cap && n_exclude >= 0 && n_exclude <= n_exclude_cap,
                   "recommend_host: list longer than the scratch capacity");
    if (liked_rows && n_liked == 0) {
        // what sklearn's check_array raises in the reference when no rated movie is liked (lib.py:47,51)
        set_error("Found array with 0 sample(s): user has no liked movies in the catalog");
        return REBERT_ERR_INVALID;
    }
    const bool sharded = exchange && exchange->world > 1;
    if (sharded) REBERT_REQUIRE(!liked_rows || cat->ld <= exchange->prof_len, "recommend_host: ld=%d exceeds the exchange buffer's prof_len=%d",
                                cat->ld, exchange->prof_len);
    const HostLayout L = host_layout(cat->ld, cat->d, n_liked_cap, n_exclude_cap, k, 256, cat->n);
    if (pinned_bytes < L.pin_bytes || device_bytes < L.dev_bytes) {
        set_error("recommend_host: scratch too small (pinned %zu < %zu or device %zu < %zu)", pinned_bytes, L.pin_bytes,
                  device_bytes, L.dev_bytes);
        return REBERT_ERR_WORKSPACE;
    }
    const double t_entry = now_us();
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* h = (unsigned char*)pinned;
    unsigned char* dv = (unsigned char*)device_scratch;
    float* qn32 = (float*)(dv + L.off_qn32);
    double* qn64 = (double*)(dv + L.off_qn64);
    int32_t* excl_dev = (int32_t*)(dv + L.off_dexcl);
    int32_t* err_word = (int32_t*)(h + L.pin_err);
    int32_t* in_flight = err_word + 1;
    volatile uint32_t* done_flag = (volatile uint32_t*)(err_word + 2);
    uint32_t* token_ctr = (uint32_t*)(err_word + 3);
    unsigned long long* res = (unsigned long long*)(h + L.pin_out);
    int rc;
    // A previous call on this scratch that never completed (a fault between launch and synchronisation) may have left the
    // scoring kernel's control words non-zero: clear them before they poison this request.
    if (*in_flight == 0x5EBE47) {
        rc = rebert_workspace_reset(dv + L.off_ws, L.ws_bytes, stream);
        if (rc != REBERT_OK) return rc;
    }
    *in_flight = 0x5EBE47;
    *err_word = 0;

    // ---- the request goes into the pinned block; the kernels read it from there
    if (n_exclude) {
        // the kernels binary-search the exclusions: the pinned copy is made strictly increasing here if it is not already
        int32_t* e = (int32_t*)(h + L.off_excl);
        memcpy(e, exclude_rows, (size_t)n_exclude * 4);
        bool increasing = true;
        for (int32_t i = 1; i < n_exclude; ++i)
            if (e[i] <= e[i - 1]) { increasing = false; break; }
        if (!increasing) {
            std::sort(e, e + n_exclude);
            n_exclude = (int32_t)(std::unique(e, e + n_exclude) - e);
        }
    }
    if (query) {
        memcpy(h + L.off_q, query, (size_t)cat->d * 4);
    } else {
        memcpy(h + L.off_col, liked_rows, (size_t)n_liked * 4);
        if (liked_w) memcpy(h + L.off_w, liked_w, (size_t)n_liked * 4);
    }
    const float* q_host = query ? (const float*)(h + L.off_q) : nullptr;
    const int32_t* liked_host = query ? nullptr : (const int32_t*)(h + L.off_col);
    const float* w_host = (!query && liked_w) ? (const float*)(h + L.off_w) : nullptr;
    const int32_t* excl_host = (const int32_t*)(h + L.off_excl);

    rebert_request_info_t inf;
    memset(&inf, 0, sizeof(inf));
    auto finish = [&]() {
        const double t_u = now_us();
        const int32_t cnt = (int32_t)(uint32_t)res[2 * (size_t)k];
        memcpy(out_rows, res, (size_t)k * 8);
        memcpy(out_scores, res + k, (size_t)k * 8);
        *out_count = cnt;
        memcpy(&inf.margin, res + 2 * (size_t)k + 1, 8);
        *in_flight = 0;
        inf.host_unpack_us = now_us() - t_u;
        if (info) *info = inf;
    };

    double t_mark = now_us();
    inf.host_pack_us = t_mark - t_entry;
    // ---- staging kernel: normalised query, or the profile (with the partial-profile exchange on a row shard)
    uint32_t seq = sharded ? exchange->seq : 0;
    Exchange x;
    rebert_exchange_t ex;
    if (sharded) {
        ex = *exchange;
        rc = make_exchange(&ex, err_word, &x);
        if (rc != REBERT_OK) return rc;
    }
    if (query) {
        rc = stage_query_launch(q_host, cat->d, cat->ld, qn32, qn64, excl_host, n_exclude, excl_dev, st);
    } else {
        rc = stage_profile_launch(cat, liked_host, w_host, n_liked, excl_host, n_exclude, excl_dev, (double*)(dv + L.off_sum64),
                                  (double*)(dv + L.off_wsum), qn32, qn64, sharded ? &x : nullptr, st);
    }
    if (rc != REBERT_OK) return rc;

    rebert_filter_t f;
    memset(&f, 0, sizeof(f));
    if (device_filter) f = *device_filter;
    f.exclude_rows = n_exclude ? excl_dev : nullptr;
    f.n_exclude = n_exclude;
    const uint32_t tag = sharded ? request_tag(query ? (const void*)query : (const void*)liked_rows,
                                               query ? (size_t)cat->d * 4 : (size_t)n_liked * 4, excl_host, (size_t)n_exclude * 4,
                                               liked_w, liked_w ? (size_t)n_liked * 4 : 0, ((uint64_t)k << 32) | (uint32_t)n_liked)
                                 : 0u;

    // ---- proof loop: each attempt is the streaming launch + its cluster kernel + one synchronisation
    // a shadow without a streaming kernel for its rows cannot help: the plain pass answers, as when its bound proves nothing
    const bool try_shadow = proof && proof->shadow && k <= proof->shadow_max_k && proof->shadow_eps > 0.0 && gemv_streams(proof->shadow);
    int cur_kc = kc;
    bool shadow_turn = try_shadow;
    while (true) {
        GemvFused gf;
        gf.exact_cat = cat;
        gf.q64 = qn64;
        gf.k = k;
        gf.out_packed = res;
        gf.tag = tag;
        gf.xchg = nullptr;
        uint32_t token = *token_ctr + 1u;
        if (token == 0u) token = 1u;
        *token_ctr = token;
        *done_flag = 0u;
        gf.done_flag = (uint32_t*)done_flag;
        gf.done_token = token;
        if (sharded) {
            x.seq = seq ? seq : 1u;
            gf.xchg = &x;
        }
        const int use_kc = shadow_turn ? 256 : cur_kc;
        rc = gemv_launch(shadow_turn ? proof->shadow : cat, qn32, &f, use_kc, dv + L.off_ws, L.ws_bytes, nullptr, &gf, st);
        if (rc != REBERT_OK) return rc;
        const double t_enq = now_us();
        inf.host_enqueue_us += t_enq - t_mark;
        if (!poll_done(done_flag, token)) REBERT_CUDA(cudaStreamSynchronize(st));
        t_mark = now_us();
        inf.host_wait_us += t_mark - t_enq;
        ++inf.attempts;
        ++seq;
        if (*err_word != 0) {
            if (*err_word > 100) set_error("recommend_host: rank %d answered a different request on this channel (request order diverged)", *err_word - 101);
            else if (*err_word > 50) set_error("recommend_host: peer %d did not deliver its partial profile to the exchange", *err_word - 51);
            else set_error("recommend_host: peer %d did not deliver its result to the exchange", *err_word - 1);
            *in_flight = 0;
            if (info) *info = inf;               // attempts = exchange sequence numbers this call consumed, the failed one included
            return REBERT_ERR_CUDA;
        }
        double margin;
        memcpy(&margin, res + 2 * (size_t)k + 1, 8);
        inf.kc = use_kc;
        inf.used_shadow = shadow_turn ? 1 : 0;
        if (!proof) { inf.proven = 0; break; }
        const double eps = shadow_turn ? proof->shadow_eps : proof->fast_eps;
        inf.proven = margin > eps ? 1 : 0;
        if (inf.proven) break;
        if (shadow_turn) { shadow_turn = false; continue; }     // not provable on the shadow: take the plain pass
        if (!proof->widen || cur_kc >= 256) break;
        cur_kc = cur_kc * 4 < 256 ? cur_kc * 4 : 256;            // candidate set not provably exact: widen and redo
    }
    finish();
    return REBERT_OK;
}

}  // extern "C"
