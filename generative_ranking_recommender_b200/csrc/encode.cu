// Multi-level encode (hierarchical_rq_kmeans.py:539-581 `predict`, and the id chain `train` emits,
// :654-660): per level  weight -> nearest centre -> normalised residual, for a model whose layers
// were trained directly (layer_clusters == need_clusters).
//
//   mode 0  "train chain": ids = KMeans.predict on the weighted data, residual of the WEIGHTED data
//           (:428, :654, :660).  These are the ids train() returns and the jsonl holds.
//   mode 1  "predict()":   as the reference's predict(): middle levels add fl32(+10000) to every
//           centre outside the block of the previous id (:1210-1219; with directly trained centres
//           that is every centre unless the previous id is 0 - SURVEY.md F8), and the residual comes
//           from the UNWEIGHTED running data (:577).  The reference's id % need (:1231) is the identity
//           when ks[l] == needs[l], which mode 1 requires at the masked levels (else RQK_ERR_UNSUPPORTED).
//
// This is the general path: a row-chunked chain of the tcgen05 score pass (argmin only, no score matrix) and the
// residual kernel per level; the running residual lives in a chunk-sized scratch so X itself is read once per level.
// It takes per-group weights, several dim-groups and any cluster count <= 4096 (the score pass's limit).  Unit weights + one dim-group (what
// train_semantic_ids.py runs) go through the single tensor-core kernel of encode_fused.cu instead (rqk_encode_fused),
// which reads X once and never materialises a residual; the two are compared with each other and with the oracle in
// tests/test_gpu_parity.py::test_fused_encode_matches_oracle_chain.
#include "common.cuh"

namespace rqk {
// Rows per chunk of the level chain (bounds the workspace: two chunk x dim fp32 buffers).  Measured on B200 at
// 1 M x 512, [128,128,256] (tools/encode_probe.py): 1 Mi rows 4.09 ms, 151 552 rows 4.44 ms, 37 888 rows (residual
// L2-resident between levels) 5.46 ms - the chain is bound by its three score passes, not by the residual's HBM
// traffic, so small L2-sized chunks only add pipeline fill.  RQK_ENC_CHUNK overrides (tuning).
constexpr long long ENC_CHUNK_DEFAULT = 1 << 20;
static long long enc_chunk() {
    static long long v = 0;
    if (!v) {
        const char* e = getenv("RQK_ENC_CHUNK");
        v = (e && atoll(e) >= 128) ? atoll(e) : ENC_CHUNK_DEFAULT;
    }
    return v;
}
}

extern "C" {

size_t rqk_encode_workspace_bytes(int64_t n, int32_t dim, int32_t kmax) {
    using namespace rqk;
    long long chunk = n < enc_chunk() ? n : enc_chunk();
    return 2 * align256((size_t)chunk * dim * 4) + score_workspace_bytes(chunk, kmax, dim) + 256;
}

// centers/weights: HOST arrays [levels] of DEVICE pointers (weights[l] may be null = all ones);
// ks/needs: HOST int32[levels]; group_end: DEVICE int32[ngroups]; ids: DEVICE int32 [levels][n].
int rqk_encode(const float* x, int64_t n, int32_t dim, int32_t levels, const void* const* centers,
               const void* const* weights, const int32_t* ks, const int32_t* needs, const int32_t* group_end,
               int32_t ngroups, int32_t* ids, int32_t mode, int32_t flags, void* workspace, size_t workspace_bytes,
               void* stream_) {
    using namespace rqk;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!x || !centers || !ks || !needs || !group_end || !ids || !workspace) return fail(RQK_ERR_ARG, "rqk_encode: null pointer%s");
    if (levels < 1 || levels > 16) return fail(RQK_ERR_UNSUPPORTED, "rqk_encode: levels=%s%lld outside [1,16]", "", levels);
    if (mode != 0 && mode != 1) return fail(RQK_ERR_ARG, "rqk_encode: mode=%s%lld must be 0 or 1", "", mode);
    // predict()'s id % need (:1231) is not applied by the score epilogues, so a masked level must have ks == needs
    // (a recursive middle layer goes through the host's block-by-block chain instead)
    if (mode == 1)
        for (int l = 1; l < levels - 1; ++l)
            if (needs[l] != ks[l])
                return fail(RQK_ERR_UNSUPPORTED, "rqk_encode: mode 1 needs ks[l] == needs[l] at masked level l=%s%lld", "", l);
    int kmax = 1;
    for (int l = 0; l < levels; ++l) kmax = ks[l] > kmax ? ks[l] : kmax;
    if (workspace_bytes < rqk_encode_workspace_bytes(n, dim, kmax))
        return fail(RQK_ERR_WORKSPACE, "rqk_encode: workspace %s%lld too small", "", (long long)workspace_bytes);
    if (n == 0) return 0;
    const long long chunk = n < enc_chunk() ? n : enc_chunk();
    char* w = (char*)workspace;
    float* cur = (float*)w; w += align256((size_t)chunk * dim * 4);     // running (unweighted) data
    float* wtd = (float*)w; w += align256((size_t)chunk * dim * 4);     // weighted view when weights != 1
    void* sws = w;
    const size_t sws_bytes = score_workspace_bytes(chunk, kmax, dim);
    for (long long r0 = 0; r0 < n; r0 += chunk) {
        const long long m = (n - r0) < chunk ? (n - r0) : chunk;
        const float* src = x + r0 * dim;                                   // level-0 input is X itself
        for (int l = 0; l < levels; ++l) {
            const float* lvl_in = src;
            if (weights && weights[l]) {
                int rc = scale_dims_launch(src, m, dim, (const float*)weights[l], wtd, stream);
                if (rc) return rc;
                lvl_in = wtd;
            }
            int* out_ids = ids + (long long)l * n + r0;
            ScoreOut o{nullptr, 0, out_ids, nullptr, nullptr, nullptr, 0, nullptr, 0};
            if (mode == 1 && l > 0 && l < levels - 1) {
                o.mask_ids = ids + (long long)(l - 1) * n + r0;
                o.mask_block = needs[l];
            }
            int rc = score_pass_dispatch(lvl_in, m, dim, (const float*)centers[l], ks[l], o, flags & 2, sws, sws_bytes, stream);
            if (rc) return rc;
            if (l < levels - 1) {
                // train chain subtracts in the weighted space (:660); predict() from the unweighted data (:577)
                const float* rin = (mode == 0) ? lvl_in : src;
                rc = residual_launch(rin, m, dim, out_ids, (const float*)centers[l], group_end, ngroups, cur, stream);
                if (rc) return rc;
                src = cur;
            }
        }
    }
    return 0;
}

}  // extern "C"
