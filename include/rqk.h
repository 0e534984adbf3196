/*
 * rqk.h - C ABI of librqk_sm100a.so: the semantic-ID hot path of zeehu/generative_ranking_recommender
 * (hierarchical residual-quantisation balanced K-Means) as hand-written CUDA for sm_100a (B200).
 *
 * The reference (100 % Python, /root/reference) has no FFI layer; its hot path is a chain of torch
 * library calls.  Each entry point below replaces the calls cited next to it (paths relative to
 * src/semantic_id_generator/).  The Python host side that mirrors the reference's classes
 * (generative_ranking_recommender_b200/{balancekmeans,hierarchical_rq_kmeans}) binds these with ctypes;
 * INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked HOST
 *   - the library never allocates or frees: the caller owns all buffers and passes a workspace whose
 *     size comes from the matching *_workspace_bytes()
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation
 *     except the functions documented as returning host scalars
 *   - return 0 on success, a negative code on failure (-1 argument, -2 CUDA, -3 workspace too small,
 *     -4 unsupported size, -5 internal); rqk_last_error() holds a thread-local message.  No exceptions.
 *   - "fp16 key": fp16 bit pattern mapped monotonically onto uint16 (sign-flip, -0 folded on +0)
 */
#ifndef RQK_H_
#define RQK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int rqk_version(void);
const char* rqk_last_error(void);
/* 0 iff CUDA device `device` is an sm_100 part */
int rqk_device_check(int device);

/* ---- score pass ----------------------------------------------------------------------------
 * balancekmeans/__init__.py:576-603 pairwise_distance_full (torch.cdist :596), fused with its
 * consumers: (-D).half() + transpose (:29,:40), max/min for eps (:33), argmin (:312,:328,:528),
 * bincount (:329).  tcgen05 3xTF32, TMA-staged; the N x K fp32 matrix is never written unless
 * `dist` is given.  x [n][dim] fp32, centers [k][dim] fp32, 1 <= k <= 4096, dim % 32 == 0.
 * k > 256 is scored in phases of 256 centres (same outputs; bit1 takes k <= 256 only).
 *   scores_t    [k][ld] fp16 = half(-dist), ld multiple of 128 >= n, columns >= n set to -inf   (or NULL)
 *   argmin      int32 [n]                                                                      (or NULL)
 *   best2       fp32 [n][2] smallest and second-smallest distance                              (or NULL)
 *   counts      int32 [k], += bincount(argmin)  (caller zeroes)                                (or NULL)
 *   minmax_keys uint32 [2] = {max, min} fp16 key of scores_t (only with scores_t)              (or NULL)
 *   dist        fp32 [n][k]                                                                    (or NULL)
 *   flags       bit0: argmax instead of argmin (auction_lap_half's n < k quirk, :24-26)
 *               bit1: CUDA-core cross-check kernel instead of the tensor-core kernel (tests only)
 */
size_t rqk_score_workspace_bytes(int64_t n, int32_t k, int32_t dim);
int rqk_score_pass(const float* x, int64_t n, int32_t dim, const float* centers, int32_t k, void* scores_t,
                   int64_t ld, int32_t* argmin, float* best2, int32_t* counts, uint32_t* minmax_keys,
                   float* dist, int32_t flags, void* workspace, size_t workspace_bytes, void* stream);

/* ---- balanced assignment --------------------------------------------------------------------
 * balancekmeans/__init__.py:12-140 auction_lap_half on the worker-major fp16 score matrix, 1 <= k <= 512 workers
 * (every auction entry point returns -4 for any other k before it reads a pointer).
 * Canonical tie rule (the reference leaves it to torch.topk's heap order): among jobs whose value
 * equals a worker's threshold, lowest job index first.  n >= k required (the n < k quirk is the
 * score pass with flags bit0).  rqk_auction() is the single-GPU driver and SYNCHRONISES the stream
 * (it returns host scalars); the step functions let a multi-GPU host sum the int32 "reduce block"
 * between pass and resolve when the jobs are sharded over ranks.
 */
typedef struct rqk_auction_info {
    int32_t done;
    int32_t rounds;        /* rounds the reference loop would have executed (1002 in the n % k != 0 regime) */
    int32_t passes;        /* passes over the score matrix actually made */
    int32_t cold_passes;   /* of which histogram-only (cold start, window miss, after a fast-forward) */
    int32_t window_misses;
    int32_t frozen_exit;   /* 1: finished through the frozen-state fast-forward (DESIGN.md) */
    int32_t counter;
    uint16_t eps_bits;     /* fp16 eps of :33-34 */
    uint16_t list_passes;    /* bidding rounds served from the HIST pass's survivor lists (no second read of S) */
} rqk_auction_info;

typedef struct rqk_auction_layout {
    int64_t total_bytes;       /* workspace size */
    int64_t reduce_offset;     /* byte offset of the int32 reduce block */
    int64_t reduce_count;      /* its length: k*256 + 2k + 2 */
    int64_t tie_total_offset;  /* byte offset of int32[k]: local number of values equal to the threshold */
} rqk_auction_layout;

/* Host only.  np.random.choice(n, k, replace=False) of NumPy's legacy MT19937 RandomState, state in/out
 * (KMeans.initialize, balancekmeans/__init__.py:247-253): key uint32[624], *pos from np.random.get_state();
 * scratch int64[n], out int64[k], all host memory. */
int rqk_legacy_choice(uint32_t* key, int32_t* pos, int64_t n, int64_t k, int64_t* scratch, int64_t* out);

size_t rqk_auction_workspace_bytes(int64_t n, int32_t k);
int rqk_auction_layout_query(int64_t n, int32_t k, rqk_auction_layout* out /*HOST*/);
int rqk_auction(const void* scores_t, int64_t ld, int64_t n, int32_t k, const void* minmax_keys, int32_t* assign,
                void* workspace, size_t workspace_bytes, rqk_auction_info* info /*HOST*/, void* stream);
int rqk_auction_init(int64_t n, int64_t ld, int32_t k, const void* minmax_keys, void* workspace,
                     size_t workspace_bytes, void* stream);
int rqk_auction_pass(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, int32_t which,
                     void* workspace, size_t workspace_bytes, void* stream);
/* which: 0 = sample + HIST + BID; else bit0 window sampling, bit1 HIST, bit2 BID.  Followed by rqk_auction_resolve
 * this is the step-by-step flow (the HIST pass merges its histograms into the reduce block).
 * bit4 (unsharded jobs): the kernels exactly as rqk_auction chains them - the HIST pass dumps its histograms per CTA,
 * bit3 is the merge kernel (one CTA per worker: sum of the dumps, threshold, tie prefix, state transition) and the
 * bidding kernel's last CTA resolves the round; no rqk_auction_resolve calls in that flow.  bit3 requires bit4. */
/* sharded jobs: every rank samples `count` of its jobs per worker (uint16 fp16 keys, [k][count]); the host
 * all-gathers them into [k][world*count] (<= 8192) and every rank places identical windows from the union */
int rqk_auction_sample_collect(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, void* out,
                               int32_t count, void* workspace, size_t workspace_bytes, void* stream);
int rqk_auction_sample_window(int64_t n, int64_t ld, int32_t k, int64_t n_global, const void* keys, int32_t count,
                              int32_t parts, void* workspace, size_t workspace_bytes, void* stream);   /* keys [parts][k][count] */
int rqk_auction_resolve(int64_t n, int64_t ld, int32_t k, int64_t n_global, int32_t expect, void* workspace,
                        size_t workspace_bytes, void* stream);   /* expect: -1 any, 0 after a HIST pass, 1 after a BID pass */
int rqk_auction_tie_offset(int64_t n, int64_t ld, int32_t k, const int32_t* totals /*[world][k]*/, int32_t rank,
                           void* workspace, size_t workspace_bytes, void* stream);
/* Jobs sharded over GPUs, exchange through peer memory instead of NCCL (DESIGN.md section 4).  peers: HOST array
 * of `world` (<= 8) device pointers, peers[r] = rank r's exchange block of rqk_auction_peer_bytes(k_max) bytes of
 * symmetric memory (zeroed once) as mapped into this process; seq0: increased by 3 per call by every rank. */
size_t rqk_auction_peer_bytes(int32_t k);
int rqk_auction_peer_round(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, int32_t count,
                           const void* const* peers, int32_t world, int32_t rank, int32_t seq0, void* workspace,
                           size_t workspace_bytes, void* stream);   /* a whole round (7 launches): seq0 = the previous round's bid counters, seq0+1 samples, seq0+2 histograms */
int rqk_auction_poll(int64_t n, int64_t ld, int32_t k, void* workspace, size_t workspace_bytes,
                     rqk_auction_info* info /*HOST*/, void* stream);   /* synchronises */
int rqk_auction_finalize(int64_t n, int64_t ld, int32_t k, void* workspace, size_t workspace_bytes, int32_t* assign,
                         void* stream);

/* ---- centroid update -------------------------------------------------------------------------
 * balancekmeans/__init__.py:314-324 (K x nonzero/index_select/mean) and :343-346 (centre shift) as
 * one deterministic segmented reduction.  accumulate: sums [k][dim] fp32, counts [k] int64 (what
 * ranks all-reduce when rows are sharded).  finalize: centers <- sums/counts IN PLACE (centers holds
 * the previous centroids), shift_out[0] = sum_k |move_k|_2, shift_out[1] = number of empty clusters
 * (left untouched, flagged in empty_mask; the host redraws them, :321-322).
 */
size_t rqk_centroid_workspace_bytes(int64_t n, int32_t k, int32_t dim);
int rqk_centroid_accumulate(const float* x, int64_t n, int32_t dim, const int32_t* assign, int32_t k, float* sums,
                            int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);
int rqk_centroid_finalize(const float* sums, const int64_t* counts, int32_t k, int32_t dim, float* centers,
                          float* shift_out, int32_t* empty_mask, void* stream);

/* ---- residual / weights / init ------------------------------------------------------------------
 * hierarchical_rq_kmeans.py:1088-1128 (_compute_residuals_with_centers), :583-604 (_apply_weights),
 * balancekmeans/__init__.py:255 (X[indices]).  out may alias x.  group_end: int32 [ngroups] exclusive
 * end dims.
 */
int rqk_residual_normalise(const float* x, int64_t n, int32_t dim, const int32_t* ids, const float* centers,
                           const int32_t* group_end, int32_t ngroups, float* out, void* stream);
int rqk_scale_dims(const float* x, int64_t n, int32_t dim, const float* w, float* out, void* stream);
/* simplified_semantic_id_generator.py:78-96, :160-164 (`batch - centers[cluster_ids]`, NOT normalised) and :317-331
 * (`dist[match == 0] = inf; argmin`): group int32 [n] selects the row's line of allow uint8 [ngroups][k]; first index
 * on ties, 0 if no candidate is allowed.  penalty = 1: a disallowed candidate competes with fl32(d + 10000) instead of
 * +inf, hierarchical_rq_kmeans.py:953 / :1288 (`distance.add_(10000.0 * (1 - match_matrix_batch))`). */
int rqk_residual_plain(const float* x, int64_t n, int32_t dim, const int32_t* ids, const float* centers, float* out,
                       void* stream);
int rqk_masked_argmin(const float* dist, int64_t n, int32_t k, const int32_t* group, const uint8_t* allow,
                      int32_t ngroups, int32_t penalty, int32_t* ids, void* stream);
int rqk_gather_rows(const float* x, int32_t dim, const int64_t* rows, int32_t nrows, float* out, void* stream);

/* ---- multi-level encode ----------------------------------------------------------------------
 * hierarchical_rq_kmeans.py:539-581 predict (mode 1, incl. the +10000 masking of :1210-1219) and the
 * id chain train() emits (mode 0: :654 + :660 per level).  Mode 1 requires ks[l] == needs[l] at the
 * masked levels 0 < l < levels-1, where the reference's id % need (:1231) is the identity; other shapes
 * (a recursive middle layer) return RQK_ERR_UNSUPPORTED.
 * centers / weights: HOST arrays [levels] of device pointers (weights[l] NULL = all ones);
 * ks / needs: HOST int32 [levels]; ids: int32 [levels][n].
 */
size_t rqk_encode_workspace_bytes(int64_t n, int32_t dim, int32_t kmax);
int rqk_encode(const float* x, int64_t n, int32_t dim, int32_t levels, const void* const* centers /*HOST*/,
               const void* const* weights /*HOST*/, const int32_t* ks /*HOST*/, const int32_t* needs /*HOST*/,
               const int32_t* group_end, int32_t ngroups, int32_t* ids, int32_t mode, int32_t flags, void* workspace,
               size_t workspace_bytes, void* stream);

/* ---- multi-level encode in one tensor-core kernel (csrc/encode_fused.cu) ----------------------
 * Same ids as rqk_encode for unit weights and one dim-group (the shape train_semantic_ids.py runs:
 * hierarchical_rq_kmeans.py:539-581, :1111-1122), but X is read from HBM once and the per-level
 * residual is never materialised: level l's scores are x . C_l^T corrected by gathered rows of the
 * Gram tables C_m C_l^T (m < l) and the running scales.  Rows whose top-2 gap is inside the error
 * budget of that algebra are re-evaluated through the literal chain by a second small kernel.
 * rqk_encode_fused_supported: 1 if the shape is taken (1..4 levels, cluster counts multiples of 32
 * in [32,256], dim a multiple of 32; mode 1 needs needs[l] == ks[l] at the masked levels), else 0 -
 * callers then use rqk_encode.  workspace[0] (int32) = number of re-evaluated rows of the call.
 */
int rqk_encode_fused_supported(int32_t dim, int32_t levels, const int32_t* ks /*HOST*/, const int32_t* needs /*HOST*/,
                               int32_t mode);
size_t rqk_encode_fused_workspace_bytes(int64_t n, int32_t dim, int32_t levels, const int32_t* ks /*HOST*/);
int rqk_encode_fused(const float* x, int64_t n, int32_t dim, int32_t levels, const void* const* centers /*HOST*/,
                     const int32_t* ks /*HOST*/, const int32_t* needs /*HOST*/, int32_t* ids, int32_t mode,
                     void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RQK_H_ */
