// C ABI of librqk_sm100a.so: version / error plumbing and the score-pass entry point.
// The other entry points live next to their kernels (auction.cu, centroid.cu, residual.cu, encode.cu).
#include "common.cuh"

namespace rqk {
thread_local char g_last_error[512] = {0};
__global__ void score_pad_kernel(__half* s, long long n, long long ld, int K);
__global__ void minmax_init_kernel(unsigned int* mm);

size_t score_workspace_bytes(long long n, int K, int dim) {
    return align256((size_t)n * 4) + 2 * align256((size_t)K * dim * 4) + align256((size_t)K * 4);
}

// flags: bit 0 = farthest, bit 1 = CUDA-core cross-check kernel instead of tcgen05
int score_pass_dispatch(const float* x, long long n, int dim, const float* centers, int k, const ScoreOut& o_in,
                        int flags, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    if (!x || !centers || !workspace) return fail(RQK_ERR_ARG, "rqk_score_pass: null pointer%s");
    if (n < 0 || n > 0x7fffffffLL) return fail(RQK_ERR_ARG, "rqk_score_pass: n=%s%lld outside [0,2^31)", "", n);
    if (k < 1 || k > 4096) return fail(RQK_ERR_UNSUPPORTED, "rqk_score_pass: k=%s%lld outside [1,4096]", "", k);
    if (dim < 32 || dim % 32 != 0 || dim > 4096) return fail(RQK_ERR_UNSUPPORTED, "rqk_score_pass: dim=%s%lld must be a multiple of 32 in [32,4096]", "", dim);
    if (o_in.scores_t && (o_in.ld < n || o_in.ld % 128 != 0)) return fail(RQK_ERR_ARG, "rqk_score_pass: ld=%s%lld must be a multiple of 128 and >= n", "", o_in.ld);
    if (((uintptr_t)x & 15) || ((uintptr_t)centers & 15)) return fail(RQK_ERR_ARG, "rqk_score_pass: x and centers must be 16-byte aligned%s");
    size_t need = score_workspace_bytes(n, k, dim);
    if (workspace_bytes < need) return fail(RQK_ERR_WORKSPACE, "rqk_score_pass: workspace %s%lld < %lld bytes", "", (long long)workspace_bytes, (long long)need);
    if (n == 0) return 0;
    ScoreOut o = o_in;
    o.farthest = flags & 1;
    char* w = (char*)workspace;
    float* x2 = (float*)w; w += align256((size_t)n * 4);
    float* chi = (float*)w; w += align256((size_t)k * dim * 4);
    float* clo = (float*)w; w += align256((size_t)k * dim * 4);
    float* c2 = (float*)w;
    if (o.scores_t) {
        if (o.minmax_keys) minmax_init_kernel<<<1, 1, 0, stream>>>(o.minmax_keys);
        long long padn = (o.ld - n) * k;
        if (padn > 0) score_pad_kernel<<<(unsigned)ceil_div<long long>(padn, 256), 256, 0, stream>>>(o.scores_t, n, o.ld, k);
        RQK_LAUNCH_OK();
    }
    if (flags & 2) return score_pass_simt(x, n, dim, centers, k, x2, c2, o, stream);
    int dev = 0, sms = 148;
    RQK_CUDA_OK(cudaGetDevice(&dev));
    RQK_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    return score_pass_tc(x, n, dim, centers, k, chi, clo, c2, o, sms, stream);
}
}  // namespace rqk

extern "C" {

int rqk_version(void) { return 100; }

const char* rqk_last_error(void) { return rqk::g_last_error; }

// 0 if `device` is an sm_100 part this library can run on.
int rqk_device_check(int device) {
    using namespace rqk;
    cudaDeviceProp prop;
    RQK_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0)      // the binary holds sm_100a code only (no PTX for other sm_10x parts)
        return fail(RQK_ERR_UNSUPPORTED, "rqk: device is sm_%s%lld%lld, this library is built for sm_100a only", "",
                    (long long)prop.major, (long long)prop.minor);
    return 0;
}

size_t rqk_score_workspace_bytes(int64_t n, int32_t k, int32_t dim) { return rqk::score_workspace_bytes(n, k, dim); }

// flags: bit 0 = farthest (argmax; the N<K quirk of auction_lap_half), bit 1 = CUDA-core cross-check kernel
int rqk_score_pass(const float* x, int64_t n, int32_t dim, const float* centers, int32_t k, void* scores_t,
                   int64_t ld, int32_t* argmin, float* best2, int32_t* counts, uint32_t* minmax_keys,
                   float* dist, int32_t flags, void* workspace, size_t workspace_bytes, void* stream_) {
    rqk::ScoreOut o{(__half*)scores_t, ld, argmin, best2, counts, minmax_keys, flags & 1, nullptr, 0, dist};
    return rqk::score_pass_dispatch(x, n, dim, centers, k, o, flags, workspace, workspace_bytes, (cudaStream_t)stream_);
}

}  // extern "C"
