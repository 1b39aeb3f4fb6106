/*
 * rebert_b200.h — C ABI of the B200-native recommendation scoring path.
 *
 * This is the drop-in boundary for robot-ebert's scoring code.  The reference has no FFI of its
 * own (it is pure Python); the entry points below replace, one for one, the pandas / scikit-learn
 * expressions on its hot path.  Citations are into the reference tree (src/backend/app/...):
 *
 *   catalog load          constants.py:55-56   -> rebert_catalog_store_rows, rebert_catalog_norms
 *   E.loc[liked] + mean   lib.py:51-52         -> rebert_profile_accumulate, rebert_profile_finalize
 *   cosine_similarity     lib.py:51, :105      -> rebert_query_normalize + rebert_gemv_topk (one query),
 *                                                 rebert_gemm_* (batched), rebert_score_subset (:105 subset form)
 *   .loc[unrated]         lib.py:48,55         -> rebert_filter_t (applied inside the scoring kernels)
 *   sort_values()[:k]     lib.py:55            -> fused in rebert_gemv_topk / rebert_gemm_filter,
 *                                                 finished by rebert_finalize_topk / rebert_merge_topk
 *
 * Conventions
 *   - Plain C: pointers, sizes, POD structs.  No torch types, no exceptions across the boundary.
 *   - Every function returns REBERT_OK (0) or a negative rebert_status; rebert_last_error() gives a
 *     thread-local message for the last failure on the calling thread.
 *   - Unless a parameter says "host", pointers are DEVICE pointers owned by the caller.  The
 *     library allocates no device memory: scratch space is a caller-provided workspace whose size
 *     comes from the matching *_workspace_bytes function.
 *   - All work is enqueued on the caller's stream; functions return without synchronising, except
 *     the *_host convenience entry points, which say so.
 *   - Re-entrant: no global mutable state; concurrent calls on one immutable catalog are safe as
 *     long as each call has its own stream + workspace + outputs.
 *   - Row ids: "local" = index into this shard's arrays; "global" = local + row_base.
 *   - Result order everywhere: (score descending, global row ascending).  With catalog rows stored
 *     in tmdb_id-string order this is the order lib.py:55,63 guarantees.
 */
#ifndef REBERT_B200_H
#define REBERT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REBERT_ABI_VERSION 5

#if defined(__GNUC__)
#define REBERT_API __attribute__((visibility("default")))
#else
#define REBERT_API
#endif

typedef enum {
    REBERT_OK = 0,
    REBERT_ERR_INVALID = -1,      /* bad argument (null pointer, size, alignment, k out of range) */
    REBERT_ERR_UNSUPPORTED = -2,  /* shape / dtype combination this build has no kernel for */
    REBERT_ERR_WORKSPACE = -3,    /* workspace too small */
    REBERT_ERR_CUDA = -4,         /* a CUDA runtime call failed; message holds cudaGetErrorString */
    REBERT_ERR_DEVICE = -5        /* not an sm_100 device */
} rebert_status;

/* REBERT_I8 is the dtype of a PREFILTER SHADOW only (rebert_catalog_quantize_i8): never the catalog of record. */
typedef enum { REBERT_F32 = 0, REBERT_BF16 = 1, REBERT_I8 = 2 } rebert_dtype;

typedef void* rebert_stream;      /* a cudaStream_t */

/* One HBM-resident catalog shard (replaces the DataFrame at constants.py:55-56).
 * rows is row-major [n, ld]; ld >= d is the padded row stride from rebert_catalog_layout, padding
 * columns are zero.  inv_norm / norm64 follow sklearn's normalize(): zero-norm rows use 1.
 *
 * Optional GATE (gate_rows != NULL; a zero-filled struct has none): the int8 rows and factors of
 * rebert_catalog_quantize_i8 over THESE rows, and its *out_max_err as gate_err.  The single-query fast pass
 * (rebert_gemv_topk, rebert_recommend_device, rebert_recommend_host) then streams the int8 rows and reads a bf16 / fp32
 * row only when its int8 score can still reach the candidate list: shadow(r) >= L - delta, L a lower bound of the kc-th
 * best fast score, delta the per-query bound of DESIGN.md §4.5.  The candidates, and so every result, margin and kc, are
 * the ones the plain pass produces, bit for bit; only the bytes read change.  Taken for rows of more than 256 bytes in
 * int8 and in the catalog's own dtype whose int8 layout has a streaming kernel (the others ignore the gate).  The gate
 * must be rebuilt after ANY write to rows / inv_norm: a stale gate can hide rows. */
typedef struct {
    const void*   rows;       /* [n, ld] of dtype */
    const float*  inv_norm;   /* [n] fp32 1 / ||row||2 */
    const double* norm64;     /* [n] fp64 ||row||2 (1 where the row is all zero) */
    int64_t       n;          /* rows in this shard */
    int64_t       row_base;   /* global row index of local row 0 */
    int32_t       d;          /* logical columns */
    int32_t       ld;         /* padded columns (elements) */
    int32_t       dtype;      /* rebert_dtype */
    int32_t       reserved;
    const void*   gate_rows;  /* [n, ld8] int8 (128-byte aligned), or NULL = no gate */
    const float*  gate_factor;/* [n] (16-byte aligned) */
    double        gate_err;   /* max_r ||x_r - dequant(q8_r)|| / ||x_r|| of the gate rows */
} rebert_catalog_t;

/* Rows that may NOT be returned (lib.py:48,55 `unrated`), plus the optional C5 genre/year predicate.
 * Any member may be NULL / 0.  A row is allowed iff it passes every non-null test. */
typedef struct {
    const uint32_t* exclude_bitmap;  /* [ceil(n/32)], local row r excluded iff bit (r & 31) of word r >> 5 is set */
    const int32_t*  exclude_rows;    /* GLOBAL row ids, sorted ascending, unique */
    int32_t         n_exclude;
    uint32_t        genre_any;       /* keep rows with (genre_bits & genre_any) != 0 */
    const uint32_t* genre_bits;      /* [n] local, or NULL */
    const uint16_t* year;            /* [n] local, or NULL */
    uint16_t        year_lo, year_hi;/* keep year_lo <= year <= year_hi */
    uint32_t        reserved;
} rebert_filter_t;

/* Per-QUERY genre / year predicate of a batch (rebert_gemm_topk_filtered): query u keeps local row r iff
 *   (genre_any[u] == 0 || (genre_bits[r] & genre_any[u]) != 0) && year_lo[u] <= year[r] <= year_hi[u].
 * Each test comes as a pair of the catalog's column and the per-query arrays: genre_bits + genre_any, year + year_lo /
 * year_hi.  A NULL pair switches that test off for every query; half a pair is REBERT_ERR_INVALID.  A query with
 * (0, 0, 65535) is unrestricted. */
typedef struct {
    const uint32_t* genre_bits;      /* [n] local, per row */
    const uint16_t* year;            /* [n] local, per row */
    const uint32_t* genre_any;       /* [b], device */
    const uint16_t* year_lo;         /* [b], device */
    const uint16_t* year_hi;         /* [b], device */
} rebert_query_filter_t;

/* How ONE RANK of a row-sharded catalog reaches its peers: NVLink peer memory, no NCCL on the request path.
 * Every rank owns a peer-mapped buffer of rebert_exchange_buffer_bytes(world, k_max, prof_len, channels) bytes,
 * ZERO-FILLED once; peer_buffers is a HOST array of the `world` device addresses under which THIS process sees the
 * ranks' buffers (e.g. torch symmetric memory's buffer_ptrs).  The buffer holds `channels` independent channels, one per
 * concurrent request stream (the reference serves from a threadpool, api/users.py:151): calls on one channel must be
 * issued in the same order by every rank, calls on different channels are independent.  seq is the call number on the
 * channel, starting at 1, the same on every rank.  A 32-bit tag of the request travels with every result; the merge
 * refuses (error) to combine results whose tags differ, i.e. when the ranks' request order on a channel diverged. */
typedef struct {
    const uint64_t* peer_buffers;
    int32_t  world, rank;
    int32_t  k_max;      /* largest k the buffers were sized for */
    int32_t  prof_len;   /* largest padded row length (ld) of a liked-rows request; 0 = query requests only */
    int32_t  channels, channel;
    uint32_t seq;
    uint32_t reserved;
} rebert_exchange_t;

/* Proof policy of rebert_recommend_host: which fast passes to try and what their error bounds are.  A result is PROVEN
 * (ids bit-exact, DESIGN.md §4.2) when the exact pass's margin exceeds the bound of the fast pass that produced the
 * candidates. */
typedef struct {
    const rebert_catalog_t* shadow;  /* int8 prefilter shadow (rebert_catalog_quantize_i8) or NULL */
    double  shadow_eps;              /* proven bound on |shadow score - true score| (rows + query planes) */
    double  fast_eps;                /* proven bound of the plain fp32 fast pass */
    int32_t shadow_max_k;            /* try the shadow only for k <= this */
    int32_t widen;                   /* 1: while the margin does not clear the bound, retry with 4x candidates (<= 256) */
} rebert_proof_t;

typedef struct {
    int32_t kc;          /* candidates of the attempt that produced the result */
    int32_t attempts;    /* fast passes run (each one consumed one exchange sequence number on a row shard) */
    int32_t proven;      /* 1: margin > bound; 0: not proven — the caller must take an exhaustive route (rebert_collect_above) */
    int32_t used_shadow; /* 1: the result came from the int8 shadow's candidates */
    double  margin;
    /* where the call's wall time went (host clock, microseconds): packing the request into the pinned block, enqueueing the
     * kernels, waiting for the completion token (all attempts summed), unpacking the result */
    double  host_pack_us, host_enqueue_us, host_wait_us, host_unpack_us;
} rebert_request_info_t;

/* ---- library ------------------------------------------------------------------------------ */
REBERT_API int         rebert_abi_version(void);
REBERT_API const char* rebert_last_error(void);
/* REBERT_OK iff the current device is compute capability 10.x. */
REBERT_API int         rebert_check_device(void);

/* ---- catalog store (constants.py:55-56) --------------------------------------------------- */
/* Padded row stride (elements) and bytes for an [n, d] catalog of `dtype`. */
REBERT_API int rebert_catalog_layout(int64_t n, int32_t d, int32_t dtype, int32_t* ld, size_t* rows_bytes);
/* Convert src fp32 [n, d] (dense, device) into stored rows [n, ld] of `dtype` (bf16: round-to-nearest-even),
 * zero-filling the padding.  May be called per chunk with offset pointers. */
REBERT_API int rebert_catalog_store_rows(const float* src, int64_t n, int32_t d, int32_t dtype, void* rows, int32_t ld,
                              rebert_stream stream);
/* Row norms of the STORED values: norm64[r] = sqrt(sum x^2) in fp64 (0 -> 1), inv_norm[r] = (float)(1/norm64[r]). */
REBERT_API int rebert_catalog_norms(const void* rows, int64_t n, int32_t ld, int32_t dtype, float* inv_norm, double* norm64,
                         rebert_stream stream);

/* Optional int8 PREFILTER SHADOW of a catalog: halves (bf16) or quarters (fp32) the bytes the single-query fast pass
 * streams.  Row r is stored as q8[r, c] = rint(x[r, c] / s_r) with s_r = max|x[r, :]| / 127, and
 * factor[r] = (float)(s_r / ||x_r||), so that  score~(r) = factor[r] * sum_c q8[r, c] * q_c  approximates the cosine.
 * *out_max_err (device double) receives max_r ||x_r - s_r q8_r|| / ||x_r||: by Cauchy-Schwarz |score~ - score| <= that
 * value for ANY unit query, a rigorous bound the caller adds to its proof margin.  The shadow is described by its own
 * rebert_catalog_t {rows = out_rows, inv_norm = out_factor, norm64 = src->norm64, dtype = REBERT_I8, ld = layout of
 * (d, REBERT_I8)} and is accepted by rebert_gemv_topk ONLY; candidates are always re-scored from the catalog of
 * record by rebert_finalize_topk, so results never depend on the shadow's precision. */
REBERT_API int rebert_catalog_quantize_i8(const rebert_catalog_t* src, void* out_rows, int32_t ld8, float* out_factor,
                                          double* out_max_err, rebert_stream stream);

/* ---- query / profile (lib.py:51-52) ------------------------------------------------------- */
/* b queries q[b, d] fp32 -> unit vectors: qn64 = q / ||q|| (fp64, zero norm -> 1), qn32 = (float) qn64,
 * qnbf16 = bf16(qn32) for the tensor-core path; all [b, ld], any output may be NULL. */
REBERT_API int rebert_query_normalize(const float* q, int32_t b, int32_t d, int32_t ld, float* qn32, double* qn64,
                           void* qnbf16, rebert_stream stream);
/* Ragged CSR gather-sum over THIS shard's rows: for user u, sum64[u, :] += w * row / norm64[row] for every
 * entry whose global row `col` lies in [row_base, row_base + n); wsum[u] += w for EVERY entry (so it is the
 * same on all shards).  w == NULL means weight 1 (the reference's 1[rating >= 3.5]).  Outputs are overwritten. */
REBERT_API int rebert_profile_accumulate(const rebert_catalog_t* cat, const int64_t* row_ptr, const int32_t* col, const float* w,
                              int32_t b, double* sum64 /* [b, ld] */, double* wsum /* [b] */, rebert_stream stream);
/* p64 = sum64 / wsum (the mean of unit rows, NOT re-normalised: lib.py:52), p32 = (float) p64, pbf16 optional. */
REBERT_API int rebert_profile_finalize(const double* sum64, const double* wsum, int32_t b, int32_t ld, float* p32, double* p64,
                            void* pbf16 /* [b, ld] bf16 or NULL */, rebert_stream stream);

/* ---- single query: fused score + mask + top-k (lib.py:51-55, L = 1 or a prebuilt profile) -- */
/* Candidate count the fast pass keeps for a request of k: a multiple of 32 >= k + margin; 0 if k is unsupported. */
REBERT_API int32_t rebert_candidates_for_k(int32_t k);
/* The workspace must be ZERO-FILLED once before its first use (it holds a ticket counter, a tile-claim counter and a
 * threshold word that every launch leaves at zero again); after that it can be reused by consecutive calls on the
 * same stream without further clearing. */
REBERT_API size_t  rebert_gemv_workspace_bytes(int64_t n, int32_t kc);
/* Zero the control words again after a launch that did not run to completion (a fault): they sit at a kc-independent
 * place at the start of the workspace, so one workspace serves every kc. */
REBERT_API int     rebert_workspace_reset(void* workspace, size_t workspace_bytes, rebert_stream stream);
/* Diagnostics: rows the gated fast pass has read from the catalog of record on this workspace since it was zero-filled
 * or reset (a wrapping 32-bit count, summed over launches).  Synchronises the stream. */
REBERT_API int     rebert_gate_fetches(const void* workspace, size_t workspace_bytes, uint32_t* out_count, rebert_stream stream);
/* Fast pass.  score(r) = <qn32, row r> * inv_norm[r] in fp32; keeps the kc best allowed rows of the shard.
 * Output: cand_keys[kc] sorted best-first (packed (score, local row) keys; unused slots are 0). */
REBERT_API int rebert_gemv_topk(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, int32_t kc,
                     void* workspace, size_t workspace_bytes, uint64_t* cand_keys, rebert_stream stream);
/* Exact pass over the kc candidates: fp64 re-score with the oracle's formula (x/||x||, y/||y||, dot), order by
 * (score desc, global row asc), write the best k.  out_count[0] = results written (<= k).
 * out_margin[0] = (exact k-th score) - (fast score of the worst kept candidate) - 4 max|fast - exact| when the list was
 * full, else +inf: a caller proves the set exact by margin > eps (see DESIGN.md) and retries with more candidates otherwise. */
REBERT_API int rebert_finalize_topk(const rebert_catalog_t* cat, const double* qn64, const uint64_t* cand_keys, int32_t kc,
                         int32_t k, int64_t* out_rows, double* out_scores, int32_t* out_count, double* out_margin,
                         rebert_stream stream);

/* ---- device-resident request (lib.py:51-55 for a prepared query / profile) -------------------------------------- */
/* Fast pass + exact pass + ranking as two chained launches without host involvement: the streaming kernel publishes its
 * pruned candidate keys, and a cluster of 8 CTAs placed behind it by programmatic dependent launch selects the kc winners,
 * re-scores them in fp64 from `cat` (the catalog of record), orders them and writes the packed result
 *     out_packed[0..k) rows | [k..2k) fp64 score bits | [2k] count (low 32 bits) + tag (high 32 bits) | [2k+1] margin
 * (device memory or device-addressable pinned host memory).  shadow != NULL: the fast pass streams the int8 shadow
 * (kc must be 256).  exchange != NULL with world > 1: the cluster kernel also runs the NVLink exchange + merge, so that
 * out_packed is the merged result a single GPU would return (margin = the smallest over the ranks); *err_flag (int32,
 * device or pinned) becomes 1 + rank if a peer did not deliver within ~10 s, 101 + rank if its request tag differs. */
REBERT_API int rebert_recommend_device(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const float* qn32, const double* qn64,
                                       const rebert_filter_t* filter, int32_t k, int32_t kc, void* workspace, size_t workspace_bytes,
                                       int64_t* out_packed, uint32_t tag, const rebert_exchange_t* exchange, int32_t* err_flag,
                                       rebert_stream stream);

/* ---- host-buffer entry point: one call = one request, end to end -------------------------- */
/* Scratch sizes for rebert_recommend_host with lists of at most n_liked_cap / n_exclude_cap entries and results of k.
 * pinned: page-locked host memory (cudaHostAlloc / pinned torch tensor); device: device memory, ZERO-FILLED once. */
REBERT_API int rebert_recommend_host_scratch(const rebert_catalog_t* cat, int32_t n_liked_cap, int32_t n_exclude_cap, int32_t k,
                                             size_t* pinned_bytes, size_t* device_bytes);
/* lib.py:43-55 for one request with HOST buffers: pass `query` [d] fp32 (not normalised) OR `liked_rows` (+ optional
 * weights), plus the GLOBAL `exclude_rows` (any order, duplicates allowed: the call sorts and de-duplicates its pinned copy
 * when the list is not already strictly increasing); device_filter may add device-resident bitmap / genre / year tests.  The request is packed into the pinned block and read from there by the first kernel (zero-copy, no copy-engine
 * operation): a staging kernel normalises the query or builds the profile (mean of the liked rows' unit vectors), then
 * rebert_recommend_device's two chained launches do fused score + mask + top-k and the fp64 exact pass, whose packed
 * result the kernel writes straight into the pinned block; a stream synchronisation ends the call.
 * `pinned` must therefore be page-locked memory the device can address.  out_rows / out_scores are host [k]
 * (-1 / -inf padded), *out_count <= k.
 * proof  (may be NULL = one attempt with `kc`, info->proven = 0): see rebert_proof_t — int8 shadow first, then the plain
 *        fast pass with kc, 4 kc, ... 256 candidates until the margin proves the id set.
 * exchange (may be NULL = single GPU): this rank's view of a row-sharded catalog.  Every rank calls with the same
 *        request; liked rows owned by other shards are summed there and the fp64 partial profiles are exchanged and
 *        added in rank order; the local results are exchanged and merged by the exact-pass kernel.  Each attempt uses
 *        sequence numbers exchange->seq, seq + 1, ... (info->attempts of them).
 * Returns REBERT_ERR_INVALID with "Found array with 0 sample(s)" when liked_rows is given but empty (the reference's
 * own failure for a user without liked movies). */
REBERT_API int rebert_recommend_host(const rebert_catalog_t* cat, const float* query, const int32_t* liked_rows,
                                     const float* liked_w, int32_t n_liked, const int32_t* exclude_rows, int32_t n_exclude,
                                     const rebert_filter_t* device_filter, int32_t k, int32_t kc, int32_t n_liked_cap,
                                     int32_t n_exclude_cap, void* pinned, size_t pinned_bytes, void* device_scratch,
                                     size_t device_bytes, const rebert_proof_t* proof, const rebert_exchange_t* exchange,
                                     int64_t* out_rows, double* out_scores, int32_t* out_count, rebert_request_info_t* info,
                                     rebert_stream stream);

/* ---- merge of per-shard results (lib.py:55 across shards) --------------------------------- */
/* For each of b queries merge `lists` sorted result lists into the best k.  List l of query u is at
 * rows[l*rows_stride + u*k ..], scores[l*scores_stride + u*k ..], counts[l*counts_stride + u] (strides in elements):
 * a dense [lists, b, k] layout has strides (b*k, b*k, b); the packed per-rank buffers of an all-gather have one
 * common byte stride expressed in each array's element size. */
REBERT_API int rebert_merge_topk(const int64_t* rows, const double* scores, const int32_t* counts, int64_t rows_stride,
                      int64_t scores_stride, int64_t counts_stride, int32_t lists, int32_t b, int32_t k,
                      int64_t* out_rows, double* out_scores, int32_t* out_count, rebert_stream stream);

/* Stand-alone forms of the two exchange steps over NVLink peer memory (rebert_exchange_t above).
 * rebert_exchange_merge: local_packed / out_packed are packed result blocks of 2k+2 64-bit words (layout as in
 * rebert_recommend_device).  The kernel stores the local block into every peer, publishes a flag, waits for all peers'
 * flags and merges under (score desc, row asc); out_packed / err_flag may point into pinned host memory.
 * rebert_profile_exchange: sum64 [ld] = this rank's fp64 partial profile (rebert_profile_accumulate); the partials are
 * exchanged, added in rank order and divided by wsum[0]: p32 / p64 [ld] receive the profile, identical on every rank. */
REBERT_API size_t rebert_exchange_buffer_bytes(int32_t world, int32_t k_max, int32_t prof_len, int32_t channels);
REBERT_API int rebert_exchange_merge(const rebert_exchange_t* exchange, int32_t k, const int64_t* local_packed, int64_t* out_packed,
                                     int32_t* err_flag, rebert_stream stream);
REBERT_API int rebert_profile_exchange(const rebert_exchange_t* exchange, int32_t ld, double* sum64, const double* wsum, float* p32,
                                       double* p64, int32_t* err_flag, rebert_stream stream);

/* ---- subset scoring for the search re-rank (lib.py:105-106) ------------------------------- */
/* out[u, j] = <p64[u], row sub_rows[j]> / norm64 in fp64 for m candidate GLOBAL rows (all must be in this shard). */
REBERT_API int rebert_score_subset(const rebert_catalog_t* cat, const double* p64, int32_t b, const int32_t* sub_rows, int32_t m,
                        double* out /* [b, m] */, rebert_stream stream);

/* ---- exact fallback for unprovable results (mass ties in fp64 that fp32 rounding breaks) ---- */
/* Appends (unordered) the GLOBAL row id of every allowed row whose fast score <qn32,row>*inv_norm >= threshold to
 * out_rows[cap]; *out_count (device int32) receives the number found (may exceed cap: then only cap were stored).
 * With threshold = (exact k-th score so far) - 2 eps this set provably contains the true top-k; the caller re-scores
 * it in fp64 with rebert_score_subset and orders it.  A plain one-warp-per-row kernel: correctness path, not the hot path. */
REBERT_API int rebert_collect_above(const rebert_catalog_t* cat, const float* qn32, const rebert_filter_t* filter, float threshold,
                                    int32_t* out_rows, int32_t cap, int32_t* out_count, rebert_stream stream);

/* ---- dense scores (test / diagnostics: the materialised matrix of lib.py:51) --------------- */
/* out[u, r] = <q32[u], row r> * inv_norm[r], fp32, plain CUDA-core kernel independent of the fused paths. */
REBERT_API int rebert_scores_dense(const rebert_catalog_t* cat, const float* q32, int32_t b, float* out /* [b, n] */,
                        rebert_stream stream);

/* ---- batched queries: tcgen05 bf16 GEMM with fused threshold filter (lib.py:51-55, many users) ---- */
typedef struct {
    int32_t b;            /* queries */
    int32_t k;            /* results per query */
    int32_t kc;           /* exact-pass candidates per query */
    int32_t sample_rows;  /* catalog rows in the threshold sample (multiple of 256) */
    int32_t sample_rank;  /* order statistic of the sample used as the threshold */
    int32_t cand_cap;     /* per-query capacity of the filtered candidate buffer */
} rebert_gemm_plan_t;
/* Plan for b queries of top-k over an n-row catalog (shard).  k <= 240: kc = round32(max(k + 16, 1.25 k)), sample rank 16,
 * ~max(8 kc, 1024) survivors.  241 <= k <= 2048 (long lists, their own selection and exact-pass kernels): the same kc (up
 * to 2560), sample rank 64, max(3 kc, 3200) survivors, so the sample is <= 2 % of the GEMM.  k > 2048: REBERT_ERR_UNSUPPORTED.
 * A catalog with fewer than 64 x survivors rows is REBERT_ERR_UNSUPPORTED ("too small"): serve it one query at a time. */
REBERT_API int    rebert_gemm_plan(int64_t n, int32_t b, int32_t k, rebert_gemm_plan_t* plan);
REBERT_API size_t rebert_gemm_workspace_bytes(const rebert_catalog_t* cat, const rebert_gemm_plan_t* plan);
/* Whole batched path: sample -> per-query threshold -> full GEMM with fused scale + threshold filter -> per-query
 * select -> fp64 re-score -> ordered top-k.  qbf16 [b, ld] bf16 (fast pass), q64 [b, ld] (exact pass).
 * excl_row_ptr / excl_col: per-query CSR of excluded GLOBAL rows, sorted within a query (may be NULL).
 * row_filter: optional per-ROW predicate shared by the whole batch (exclude_bitmap / genre_bits+genre_any / year range;
 * its exclude_rows member is ignored — per-query exclusions are the CSR).  Filtered rows are dropped inside the GEMM
 * epilogue at no extra cost and are left out of the threshold sample.
 * out_rows / out_scores are [b, k]; out_count[b]; out_status[b] is 0 when the query's result is proven exact and
 * non-zero when the caller must re-run that query through the single-query path (threshold sample too optimistic,
 * candidate buffer overflow, or margin below eps). */
REBERT_API int rebert_gemm_topk(const rebert_catalog_t* cat, const void* qbf16, const double* q64, const int64_t* excl_row_ptr,
                     const int32_t* excl_col, const rebert_filter_t* row_filter, const rebert_gemm_plan_t* plan, void* workspace,
                     size_t workspace_bytes,
                     int64_t* out_rows, double* out_scores, int32_t* out_count, int32_t* out_status,
                     rebert_stream stream);
/* rebert_gemm_topk with a per-query predicate on top of the shared row_filter (query_filter NULL = rebert_gemm_topk).  The
 * threshold sample leaves out the rows each query's test rejects, so its survivor count stays at the plan's figure; the
 * filter GEMM's epilogue drops the rejected winners.  A query with fewer than sample_rank allowed sampled rows gets no
 * threshold: every allowed row survives, and an overflowing candidate buffer sets its status. */
REBERT_API int rebert_gemm_topk_filtered(const rebert_catalog_t* cat, const void* qbf16, const double* q64, const int64_t* excl_row_ptr,
                                         const int32_t* excl_col, const rebert_filter_t* row_filter,
                                         const rebert_query_filter_t* query_filter, const rebert_gemm_plan_t* plan, void* workspace,
                                         size_t workspace_bytes, int64_t* out_rows, double* out_scores, int32_t* out_count,
                                         int32_t* out_status, rebert_stream stream);
/* ---- the same batched path with INT8 OPERANDS: the filter GEMM streams the prefilter shadow (rebert_catalog_quantize_i8)
 * with tcgen05 kind::i8 — half the bytes and twice the tensor rate of bf16 — and int8 queries; exact integer accumulation.
 * Only the FILTER is approximate: candidates are re-scored in fp64 from the catalog of record exactly as in
 * rebert_gemm_topk, and a query whose proof margin does not clear its bound gets out_status != 0 and is re-run by the
 * caller on the single-query path, whose bound is rigorous.
 *   rebert_gemm_plan_i8       as rebert_gemm_plan, with the wider candidate list the larger filter error needs
 *                             (kc = round32(k + max(k, 64)), up to 4096 at k = 2048)
 *   rebert_query_quantize_i8  qn32 [b, ld] unit queries / profiles -> q8 [b, ld8] int8, qscale [b] (dequantisation step),
 *                             qeps [b] = the margin a result of that query must clear: 6 sigma of the score error under the
 *                             random-direction model, sigma = sqrt(row_err^2 + rho_q^2) / sqrt(d) with row_err the shadow's
 *                             measured worst relative row error (*out_max_err of rebert_catalog_quantize_i8) and rho_q
 *                             the query's own, measured here.  The batched proof is statistical (as on the bf16 path, whose
 *                             query rounding has no useful worst-case bound either); the margin is additionally reduced by
 *                             2 x the largest |filter score - exact score| observed on the candidates.
 *   rebert_gemm_topk_i8       cat = catalog of record (exact pass), shadow = its int8 shadow (operands of the GEMM);
 *                             needs ld8 % 128 == 0. */
REBERT_API int rebert_gemm_plan_i8(int64_t n, int32_t b, int32_t k, rebert_gemm_plan_t* plan);
REBERT_API int rebert_query_quantize_i8(const float* qn32, int32_t b, int32_t d, int32_t ld, int32_t ld8, double row_err, void* q8,
                                        float* qscale, double* qeps, rebert_stream stream);
REBERT_API int rebert_gemm_topk_i8(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const void* q8, const float* qscale,
                                   const double* qeps, const double* q64, const int64_t* excl_row_ptr, const int32_t* excl_col,
                                   const rebert_filter_t* row_filter, const rebert_gemm_plan_t* plan, void* workspace,
                                   size_t workspace_bytes, int64_t* out_rows, double* out_scores, int32_t* out_count,
                                   int32_t* out_status, rebert_stream stream);
/* rebert_gemm_topk_i8 with a per-query predicate, as rebert_gemm_topk_filtered (query_filter NULL = rebert_gemm_topk_i8). */
REBERT_API int rebert_gemm_topk_i8_filtered(const rebert_catalog_t* cat, const rebert_catalog_t* shadow, const void* q8, const float* qscale,
                                            const double* qeps, const double* q64, const int64_t* excl_row_ptr, const int32_t* excl_col,
                                            const rebert_filter_t* row_filter, const rebert_query_filter_t* query_filter,
                                            const rebert_gemm_plan_t* plan, void* workspace, size_t workspace_bytes, int64_t* out_rows,
                                            double* out_scores, int32_t* out_count, int32_t* out_status, rebert_stream stream);
/* out[u, j] = (sum_c q8[u, c] * shadow[j, c]) * factor[j] * qscale[u] for rows [row0, row0 + nrows), fp32 [b, nrows]. */
REBERT_API int rebert_gemm_scores_i8(const rebert_catalog_t* shadow, const void* q8, const float* qscale, int32_t b, int64_t row0,
                                     int64_t nrows, float* out, rebert_stream stream);
/* Building block, also used by tests: out[u, j] = <q[u], row j> * inv_norm[j] for rows [row0, row0 + nrows) on the
 * tensor cores (bf16 catalog only), fp32 [b, nrows]. */
REBERT_API int rebert_gemm_scores(const rebert_catalog_t* cat, const void* qbf16, int32_t b, int64_t row0, int64_t nrows,
                       float* out, rebert_stream stream);

/* ---- synthetic inputs (bench / tests; bit-identical twin of robot_ebert_b200/synth.py) ----- */
REBERT_API int rebert_synth_rows(uint64_t seed, int64_t row0, int64_t n, int32_t d, int32_t scale_rows, int32_t dtype, void* rows,
                      int32_t ld, rebert_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* REBERT_B200_H */
