// Bring-up / cross-check score pass on CUDA cores (plain fp32 FFMA).  The production score pass is
// the tcgen05 3xTF32 kernel in score_tc.cu; this one exists so that every other stage can be
// validated independently of the tensor-core path and so that tests can compare the two.
//
// Computes what `pairwise_distance_full` + the consumers of its result compute
// (balancekmeans/__init__.py:576-603, :29, :40, :312, :328-329):
//   d[n][k]   = sqrt(max(|x_n|^2 + |c_k|^2 - 2 x_n.c_k, 0))      (ATen _euclidean_dist)
//   S[k][n]   = half(-d[n][k])                                    fp16, transposed, -inf padded
//   argmin[n] = first k minimising d ; best2[n] = {d_min, d_second}
//   counts[k] += #{n : argmin[n] == k} ; minmax = extrema of S as monotone keys
#include "common.cuh"

namespace rqk {

// row norms: one warp per row
__global__ void row_sqnorm_kernel(const float* __restrict__ x, long long n, int dim, float* __restrict__ out) {
    long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (row >= n) return;
    const float* r = x + row * dim;
    float s = 0.f;
    for (int d = lane * 4; d < dim; d += 128) {
        float4 v = *reinterpret_cast<const float4*>(r + d);
        s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row] = s;
}

constexpr int SS_BM = 64;    // rows per CTA
constexpr int SS_BK = 32;    // dims per step
constexpr int SS_THREADS = 256;

template <int KT>   // centroids per thread (K <= 16*KT)
__global__ void __launch_bounds__(SS_THREADS)
score_simt_kernel(const float* __restrict__ x, long long n, int dim, const float* __restrict__ c, int K,
                  const float* __restrict__ x2, const float* __restrict__ c2, ScoreOut o) {
    __shared__ float xs[SS_BM][SS_BK + 1];
    extern __shared__ float cs_dyn[];   // [K][SS_BK+1]
    float (*cs)[SS_BK + 1] = reinterpret_cast<float (*)[SS_BK + 1]>(cs_dyn);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long long row0 = (long long)blockIdx.x * SS_BM;
    float acc[4][KT];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int j = 0; j < KT; ++j) acc[r][j] = 0.f;

    for (int d0 = 0; d0 < dim; d0 += SS_BK) {
        for (int i = tid; i < SS_BM * SS_BK; i += SS_THREADS) {
            int r = i / SS_BK, d = i % SS_BK;
            long long row = row0 + r;
            xs[r][d] = (row < n) ? x[row * dim + d0 + d] : 0.f;
        }
        for (int i = tid; i < K * SS_BK; i += SS_THREADS) {
            int k = i / SS_BK, d = i % SS_BK;
            cs[k][d] = c[(long long)k * dim + d0 + d];
        }
        __syncthreads();
#pragma unroll 8
        for (int d = 0; d < SS_BK; ++d) {
            float xv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) xv[r] = xs[ty * 4 + r][d];
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                int k = tx + 16 * j;
                float cv = (k < K) ? cs[k][d] : 0.f;
#pragma unroll
                for (int r = 0; r < 4; ++r) acc[r][j] = fmaf(xv[r], cv, acc[r][j]);
            }
        }
        __syncthreads();
    }

    unsigned int kmax = 0, kmin = 0xffffu;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        long long row = row0 + ty * 4 + r;
        bool rv = row < n;
        float xn = rv ? x2[row] : 0.f;
        const int pid = (rv && o.mask_ids) ? o.mask_ids[row] : -1;
        float b1 = INFINITY, b2 = INFINITY;
        int bi = 0x7fffffff;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            int k = tx + 16 * j;
            if (k < K) {
                float d2 = fmaf(-2.f, acc[r][j], xn + c2[k]);
                float d = sqrtf(fmaxf(d2, 0.f));
                if (rv && o.dist) o.dist[row * K + k] = d;
                if (rv && o.scores_t) {
                    __half h = __float2half_rn(-d);
                    o.scores_t[(long long)k * o.ld + row] = h;
                    unsigned int key = h2key(h2bits(h));
                    kmax = max(kmax, key);
                    kmin = min(kmin, key);
                }
                float dd = o.farthest ? -d : d;
                if (pid >= 0 && (k < pid * o.mask_block || k >= (pid + 1) * o.mask_block)) dd = d + 10000.0f;
                if (dd < b1) { b2 = b1; b1 = dd; bi = k; }
                else if (dd < b2) b2 = dd;
            }
        }
        // reduce over the 16 threads (tx) that share this row: lexicographic (dist, index) min
#pragma unroll
        for (int off = 8; off; off >>= 1) {
            float ob1 = __shfl_xor_sync(0xffffffffu, b1, off);
            float ob2 = __shfl_xor_sync(0xffffffffu, b2, off);
            int obi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (ob1 < b1 || (ob1 == b1 && obi < bi)) {
                b2 = fminf(b1, ob2);
                b1 = ob1;
                bi = obi;
            } else {
                b2 = fminf(b2, ob1);
            }
        }
        if (rv && tx == 0) {
            if (o.argmin) o.argmin[row] = bi;
            if (o.best2) { o.best2[row * 2] = o.farthest ? -b1 : b1; o.best2[row * 2 + 1] = o.farthest ? -b2 : b2; }
            if (o.counts) atomicAdd(&o.counts[bi], 1);
        }
    }
    if (o.scores_t && o.minmax_keys) {
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, off));
            kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, off));
        }
        if ((tid & 31) == 0) {
            atomicMax(&o.minmax_keys[0], kmax);
            atomicMin(&o.minmax_keys[1], kmin);
        }
    }
}

// -inf padding of the columns [n, ld) of the transposed score matrix
__global__ void score_pad_kernel(__half* s, long long n, long long ld, int K) {
    long long pad = ld - n;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < pad * K) {
        long long k = i / pad, j = n + i % pad;
        s[k * ld + j] = __ushort_as_half(0xFC00);
    }
}

__global__ void minmax_init_kernel(unsigned int* mm) {
    mm[0] = 0u;
    mm[1] = 0xffffu;
}

int score_pass_simt(const float* x, long long n, int dim, const float* c, int K, float* x2, float* c2,
                    const ScoreOut& o, cudaStream_t stream) {
    // the whole centroid block of a k-step sits in shared memory and a thread holds 16 columns per row
    if (K > 256) return fail(RQK_ERR_UNSUPPORTED, "score_pass_simt: the CUDA-core cross-check takes k <= 256, got %s%lld", "", K);
    if (n == 0) return 0;
    row_sqnorm_kernel<<<(unsigned)ceil_div<long long>(n * 32, 256), 256, 0, stream>>>(x, n, dim, x2);
    row_sqnorm_kernel<<<(unsigned)ceil_div<long long>((long long)K * 32, 256), 256, 0, stream>>>(c, K, dim, c2);
    RQK_LAUNCH_OK();
    unsigned grid = (unsigned)ceil_div<long long>(n, SS_BM);
    size_t smem = (size_t)K * (SS_BK + 1) * 4;
    if (K <= 64) {
        score_simt_kernel<4><<<grid, SS_THREADS, smem, stream>>>(x, n, dim, c, K, x2, c2, o);
    } else if (K <= 128) {
        score_simt_kernel<8><<<grid, SS_THREADS, smem, stream>>>(x, n, dim, c, K, x2, c2, o);
    } else {
        score_simt_kernel<16><<<grid, SS_THREADS, smem, stream>>>(x, n, dim, c, K, x2, c2, o);
    }
    RQK_LAUNCH_OK();
    return 0;
}

}  // namespace rqk
