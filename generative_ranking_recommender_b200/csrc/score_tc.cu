// Score pass on the 5th-generation tensor cores: X[n,dim] . C[K,dim]^T as 3xTF32 on tcgen05 with
// TMA-staged tiles and TMEM accumulators, and everything that consumes the N x K distance matrix in
// the reference fused into the epilogue so that matrix never exists in HBM:
//   pairwise_distance_full (balancekmeans/__init__.py:576-603 over torch.cdist :596)
//     d = sqrt(max(|x|^2 + |c|^2 - 2 x.c, 0))
//   (-d).half() transposed to worker-major            (:29, :40)     -> scores_t [K][ld] fp16
//   max / min of that matrix for eps                    (:33)          -> minmax_keys
//   argmin (first index) and the runner-up              (:312, :328)   -> argmin, best2
//   bincount of the argmin                              (:329)         -> counts
//
// Shape of the kernel (one CTA per SM, persistent over 128-row tiles of X):
//   warp 8      TMA producer: per 32-float k-block, X tile [128 x 32] and the centroid hi/lo blocks
//               [KC x 32] (128-byte swizzle, zero fill outside the tensors) into a smem ring.
//   warps 4-7   transform: split the landed fp32 X block into tf32 hi = rna(x) (in place) and
//               lo = rna(x - hi) (second buffer, same swizzled offsets - the map is elementwise), and
//               accumulate |x|^2 per row in fp32; one thread per row.
//   warp 9      one elected thread issues, per k-block, 4 x {hi.hi, hi.lo, lo.hi} tcgen05.mma
//               kind::tf32 (M=128, N=KC, K=8) into a TMEM accumulator [128 lanes x KC columns];
//               tcgen05.commit frees the ring slot / publishes the accumulator.
//   warps 0-3   epilogue: tcgen05.ld 32 columns at a time (thread = row), distance, fp16 store,
//               running best/second/argmin in registers; accumulators are double-buffered in TMEM so
//               the epilogue of tile i overlaps the MMAs of tile i+1.
// The lo.lo product is dropped (<= 2^-22 |x||c| per term), which leaves the dot products at fp32
// accuracy (~1e-7 relative on d): far below the fp16 rounding of the scores and the 1e-5 near-tie gate.
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc_common.cuh"

namespace rqk {

struct ScoreTcParams {
    long long n;
    int dim, K, KC;          // KC = K rounded up to 16 (UMMA N)
    int tmem_cols;           // columns per accumulator stage (power of two >= 32, >= KC)
    int stages;
    int raw;                 // depth of the raw X ring
    int tmem_alloc;          // TMEM columns allocated (power of two)
    int a_col0;              // ATMEM kernel: first TMEM column of the A-operand stages (64 columns each: hi | lo)
    const float* c2;         // [K] |c|^2
    ScoreOut o;
    int debug;               // timing attribution only (RQK_SCORE_DEBUG): 1 = skip epilogue math, 2 = hi.hi MMA only, 4 = no transform
    int phases;              // WIDE kernel: ceil(K / 256) column phases (KC = 256); 1 otherwise
    int kc_last;             // WIDE kernel: UMMA N of the last phase, round_up(K - 256 (phases - 1), 16)
};

constexpr int TC_PHASE_COLS = 256;   // columns per phase of the WIDE kernel: the TMA box limit and one accumulator

// |c|^2 of 32 consecutive columns from global memory; every thread of a warp reads the same address (WIDE epilogue).
// The phase's last chunk may read up to round_up(K, 32) entries: inside the align256(K * 4) bytes the workspace
// reserves for |c|^2, and masked out by k < K.
__device__ __forceinline__ void load_c2_32(const float* c2, float (&cw)[32]) {
    const float4* c4 = reinterpret_cast<const float4*>(c2);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 t = __ldg(c4 + i);
        cw[4 * i + 0] = t.x; cw[4 * i + 1] = t.y; cw[4 * i + 2] = t.z; cw[4 * i + 3] = t.w;
    }
}

// ATMEM (K <= 128, where two accumulators leave TMEM columns free): the transform warps write the hi / lo split of an
// X block straight into TENSOR MEMORY (tcgen05.st, thread = row = TMEM lane) and the MMAs take their A operand from
// there (tcgen05.mma [d], [a_tmem], b_desc).  The A operand then costs no shared-memory bandwidth at all - neither the
// 32 KB written per k-block nor the 48 KB the three MMAs read back - which is what bounds the smem-operand kernel at
// K = 128 (DESIGN.md section 6); the operand stages in shared memory hold the centroid blocks only.
//
// WIDE (256 < K <= 4096, shared-memory A operand only): the centres are scored in phases of 256 columns, the TMA box
// limit and the size of one of the two accumulators.  Each (tile, phase) runs the tile's k-loop once into the next
// accumulator, so the epilogue of phase p overlaps the MMAs of phase p + 1 exactly as the epilogue of one tile overlaps
// the next tile's MMAs in the narrow kernel.  Phase p TMA-loads centroid rows [256 p, 256 p + 256) (rows past K
// zero-filled, masked by the epilogue) and the last phase runs the MMAs at N = kc_last.  The X blocks of phases >= 1 are
// re-streamed through the raw ring; a tile is 128 x dim x 4 bytes (256 KB at dim 512), so with one tile per SM in
// flight L2 serves them.  |x|^2 is summed in phase 0 only, in the narrow kernel's chunk order, so a row's norm is
// bit-identical to the narrow pass.  The epilogue thread of a row carries b1 / b2 / bi and the extrema across the
// phases with global column indices 256 p + j, so the first index still wins a tie across a phase boundary.
// Shared memory: two operand stages of 96 KB (A hi/lo 32 KB + centroid hi/lo 64 KB) and one raw X block, as at
// K = 256, leave no room for K-sized tables.  |c|^2 is read with warp-uniform __ldg (every thread of a warp reads the
// same column, one L1 broadcast per 32 columns and 128 rows) instead of staging slices, which would need a barrier
// among the epilogue warps per phase; the counts go to global atomics once per row (16 KB of per-CTA table at
// K = 4096 does not fit).
template <bool ATMEM, bool WIDE = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_chi,
                const __grid_constant__ CUtensorMap map_clo, const ScoreTcParams P) {
    extern __shared__ __align__(1024) unsigned char smem_dyn[];
    // SWIZZLE_128B tiles need 1024-byte alignment; do not rely on the attribute alone
    unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KC = P.KC, stages = P.stages, nraw = P.raw;
    const int kblocks = P.dim / TC_BK;
    const long long ntiles = (P.n + TC_BM - 1) / TC_BM;
    const int nph = WIDE ? P.phases : 1;

    // ---- smem carve-up: per stage {A hi 16K, A lo 16K, B hi KC*128, B lo KC*128}, all 1024-aligned ----
    const uint32_t a_bytes = TC_BM * TC_BK * 4;           // 16384
    const uint32_t b_bytes = (uint32_t)KC * TC_BK * 4;    // KC*128, multiple of 2048
    const uint32_t b_off = ATMEM ? 0u : 2 * a_bytes;     // centroid blocks inside an operand stage
    const uint32_t stage_bytes = b_off + 2 * b_bytes;
    // raw X ring: the X stream from HBM runs up to `nraw` k-blocks ahead of the operand stages, so that the HBM
    // latency is covered by bytes in flight instead of by stage occupancy (a stage is held from its centroid
    // load until its MMAs retire)
    unsigned char* raw0 = smem + (size_t)stages * stage_bytes;
    unsigned char* tail = raw0 + (size_t)nraw * a_bytes;
    uint64_t* full_bar = (uint64_t*)tail;          // [stages]
    uint64_t* xf_bar = full_bar + 8;               // [stages]
    uint64_t* empty_bar = xf_bar + 8;              // [stages]
    uint64_t* tmem_full = empty_bar + 8;           // [2]
    uint64_t* tmem_empty = tmem_full + 2;          // [2]
    uint64_t* x2_full = tmem_empty + 2;            // [2]
    uint64_t* raw_full = x2_full + 2;              // [TC_MAX_RAW]
    uint64_t* raw_empty = raw_full + TC_MAX_RAW;   // [TC_MAX_RAW]
    uint32_t* tmem_base_slot = (uint32_t*)(raw_empty + TC_MAX_RAW);
    float* x2s = (float*)(tmem_base_slot + 4);     // [2][128]
    float* c2s = x2s + 2 * TC_BM;                  // [KC]
    int* cnt_s = (int*)(c2s + 256);                // [256]

    if (!WIDE)
        for (int i = threadIdx.x; i < 256; i += TC_THREADS) {
            c2s[i] = (i < P.K) ? P.c2[i] : 0.f;
            cnt_s[i] = 0;
        }
    if (warp == TC_TMA_WARP && lane == 0) {
        tma_prefetch_desc(&map_x);
        tma_prefetch_desc(&map_chi);
        tma_prefetch_desc(&map_clo);
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&xf_bar[s], 128);
            mbar_init(&empty_bar[s], 1);
        }
        for (int i = 0; i < nraw; ++i) {
            mbar_init(&raw_full[i], 1);
            mbar_init(&raw_empty[i], 128);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full[a], 1);
            mbar_init(&tmem_empty[a], 128);
            mbar_init(&x2_full[a], 128);
        }
        fence_barrier_init();
    }
    if (warp == TC_MMA_WARP) {
        uint32_t ncols = (uint32_t)P.tmem_alloc;
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;

    if (warp == TC_XLOAD_WARP) {
        // ===================== TMA producer: X blocks into the raw ring =====================
        if (lane == 0) {
            int rs = 0; uint32_t rph = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int row0 = (int)(tile * TC_BM);
                for (int kbp = 0; kbp < nph * kblocks; ++kbp) {   // WIDE: phases >= 1 re-read the tile (from L2)
                    const int kb = WIDE ? kbp % kblocks : kbp;
                    mbar_wait(&raw_empty[rs], rph ^ 1);
                    mbar_expect_tx(&raw_full[rs], a_bytes);
                    tma_load_2d(raw0 + (size_t)rs * a_bytes, &map_x, &raw_full[rs], kb * TC_BK, row0);
                    if (++rs == nraw) { rs = 0; rph ^= 1; }
                }
            }
        }
    } else if (warp == TC_TMA_WARP) {
        // ===================== TMA producer: centroid hi / lo blocks into the operand stages =====================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int kbp = 0; kbp < nph * kblocks; ++kbp) {
                    const int kb = WIDE ? kbp % kblocks : kbp;
                    const int c1 = WIDE ? kbp / kblocks * TC_PHASE_COLS : 0;   // phase p: centroid rows from 256 p
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    unsigned char* st = smem + (size_t)s * stage_bytes;
                    mbar_expect_tx(&full_bar[s], 2 * b_bytes);
                    tma_load_2d(st + b_off, &map_chi, &full_bar[s], kb * TC_BK, c1);
                    tma_load_2d(st + b_off + b_bytes, &map_clo, &full_bar[s], kb * TC_BK, c1);
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == TC_MMA_WARP) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc_full = make_idesc_tf32(TC_BM, KC);
            const uint32_t idesc_last = WIDE ? make_idesc_tf32(TC_BM, P.kc_last) : idesc_full;
            int s = 0; uint32_t ph = 0;
            int a = 0; uint32_t aph = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
            for (int p = 0; p < nph; ++p) {
                const uint32_t idesc = (p == nph - 1) ? idesc_last : idesc_full;
                mbar_wait(&tmem_empty[a], aph ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(a * P.tmem_cols);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full_bar[s], ph);    // centroid blocks landed (TMA)
                    mbar_wait(&xf_bar[s], ph);      // hi/lo of the X block written by the transform warps
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + (size_t)s * stage_bytes);
                    const uint64_t a_hi = make_sw128_desc(st);
                    const uint64_t a_lo = make_sw128_desc(st + a_bytes);
                    const uint64_t b_hi = make_sw128_desc(st + b_off);
                    const uint64_t b_lo = make_sw128_desc(st + b_off + b_bytes);
                    const uint32_t at_hi = tmem_base + (uint32_t)(P.a_col0 + s * 2 * TC_BK);   // ATMEM: A stage in TMEM
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k) {
                        const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);   // +32 B along K inside the swizzle row
                        if (ATMEM) {                                         // 8 tf32 = 8 TMEM columns per k-step
                            umma_tf32_ts(d_tmem, at_hi + TC_BK + k * 8, b_hi + adv, idesc, (kb | k) != 0);
                            umma_tf32_ts(d_tmem, at_hi + k * 8, b_lo + adv, idesc, 1);
                            umma_tf32_ts(d_tmem, at_hi + k * 8, b_hi + adv, idesc, 1);
                        } else if (!(P.debug & 2)) {
                            umma_tf32(d_tmem, a_lo + adv, b_hi + adv, idesc, (kb | k) != 0);
                            umma_tf32(d_tmem, a_hi + adv, b_lo + adv, idesc, 1);
                            umma_tf32(d_tmem, a_hi + adv, b_hi + adv, idesc, 1);
                        } else {
                            umma_tf32(d_tmem, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
                        }
                    }
                    umma_commit(&empty_bar[s]);      // frees the ring slot when these MMAs retire
                    if (kb == kblocks - 1) umma_commit(&tmem_full[a]);
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
                if (++a == 2) { a = 0; aph ^= 1; }
            }
        }
    } else if (warp >= TC_XF_WARP0 && warp < TC_XF_WARP0 + 4) {
        // ===================== transform: hi/lo split + row norms =====================
        const int r = (warp - TC_XF_WARP0) * 32 + lane;     // row of the tile owned by this thread
        int s = 0; uint32_t ph = 0;
        int rs = 0; uint32_t rph = 0;
        int a = 0; uint32_t aph = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            float nrm = 0.f;
            for (int p = 0; p < nph; ++p) {                  // WIDE: each phase re-splits the tile's X blocks
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&raw_full[rs], rph);               // the raw X block has landed
                    mbar_wait(&empty_bar[s], ph ^ 1);            // the operand stage is free (its last MMAs retired)
                    if (P.debug & 4) {
                        fence_proxy_async();
                        mbar_arrive(&xf_bar[s]);
                        mbar_arrive(&raw_empty[rs]);
                        if (++s == stages) { s = 0; ph ^= 1; }
                        if (++rs == nraw) { rs = 0; rph ^= 1; }
                        continue;
                    }
                    unsigned char* st = smem + (size_t)s * stage_bytes;
                    const float4* raw = reinterpret_cast<const float4*>(raw0 + (size_t)rs * a_bytes + (size_t)r * 128);
                    if (ATMEM) {
                        // the row's 32 floats in LOGICAL order (chunk c sits at physical chunk c ^ (row & 7)), split, and stored
                        // to this thread's TMEM lane: columns [0,32) of the stage = hi, [32,64) = lo
                        uint32_t hv[TC_BK], lv[TC_BK];
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const float4 v = raw[c ^ (lane & 7)];
                            nrm = fmaf(v.x, v.x, nrm); nrm = fmaf(v.y, v.y, nrm);
                            nrm = fmaf(v.z, v.z, nrm); nrm = fmaf(v.w, v.w, nrm);
                            const float hx = to_tf32_rna(v.x), hy = to_tf32_rna(v.y), hz = to_tf32_rna(v.z), hw = to_tf32_rna(v.w);
                            hv[4 * c + 0] = __float_as_uint(hx); hv[4 * c + 1] = __float_as_uint(hy);
                            hv[4 * c + 2] = __float_as_uint(hz); hv[4 * c + 3] = __float_as_uint(hw);
                            lv[4 * c + 0] = __float_as_uint(to_tf32_rna(v.x - hx)); lv[4 * c + 1] = __float_as_uint(to_tf32_rna(v.y - hy));
                            lv[4 * c + 2] = __float_as_uint(to_tf32_rna(v.z - hz)); lv[4 * c + 3] = __float_as_uint(to_tf32_rna(v.w - hw));
                        }
                        const uint32_t ta = tmem_base + ((uint32_t)((warp - TC_XF_WARP0) * 32) << 16) + (uint32_t)(P.a_col0 + s * 2 * TC_BK);
                        tmem_st32(ta, hv);
                        tmem_st32(ta + TC_BK, lv);
                        tmem_st_wait();
                        tc_fence_before();                           // tcgen05.st -> visible to the MMAs issued after the barrier
                        mbar_arrive(&xf_bar[s]);
                        mbar_arrive(&raw_empty[rs]);
                        if (++s == stages) { s = 0; ph ^= 1; }
                        if (++rs == nraw) { rs = 0; rph ^= 1; }
                        continue;
                    }
                    float4* hi = reinterpret_cast<float4*>(st + (size_t)r * 128);
                    float4* lo = reinterpret_cast<float4*>(st + a_bytes + (size_t)r * 128);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        // logical 16-byte chunk c of the row sits at physical chunk c ^ (row & 7) (SWIZZLE_128B), which
                        // is also conflict-free; summing in LOGICAL order keeps a row's norm independent of where
                        // the row lands in a tile, so row-sharded runs reproduce the unsharded scores bit for bit
                        const int ch = c ^ (lane & 7);
                        float4 v = raw[ch];                       // same swizzled position in the raw block and in the operand tile
                        if (!WIDE || p == 0) {                    // WIDE: the row norm comes from phase 0 alone
                            nrm = fmaf(v.x, v.x, nrm); nrm = fmaf(v.y, v.y, nrm);
                            nrm = fmaf(v.z, v.z, nrm); nrm = fmaf(v.w, v.w, nrm);
                        }
                        float4 h, l;
                        h.x = to_tf32_rna(v.x); h.y = to_tf32_rna(v.y); h.z = to_tf32_rna(v.z); h.w = to_tf32_rna(v.w);
                        l.x = to_tf32_rna(v.x - h.x); l.y = to_tf32_rna(v.y - h.y);
                        l.z = to_tf32_rna(v.z - h.z); l.w = to_tf32_rna(v.w - h.w);
                        hi[ch] = h;
                        lo[ch] = l;
                    }
                    fence_proxy_async();                         // generic-proxy writes -> visible to the UMMA reads
                    mbar_arrive(&xf_bar[s]);
                    mbar_arrive(&raw_empty[rs]);                 // the raw slot can be refilled
                    if (++s == stages) { s = 0; ph ^= 1; }
                    if (++rs == nraw) { rs = 0; rph ^= 1; }
                }
                mbar_wait(&tmem_empty[a], aph ^ 1);              // x2s[a] is free once the epilogue two units back is done
                x2s[a * TC_BM + r] = nrm;
                mbar_arrive(&x2_full[a]);
                if (++a == 2) { a = 0; aph ^= 1; }
            }
        }
    } else if (warp < 4) {
        // ===================== epilogue =====================
        const int q = warp;                                  // TMEM lane quarter = warp % 4
        const int r = q * 32 + lane;
        int a = 0; uint32_t aph = 0;
        // fast path: no fp32 distance matrix, no predict()-mode masking, nearest (not farthest) centre
        const bool fast = !P.o.dist && !P.o.mask_ids && !P.o.farthest;
        unsigned int kmax = 0, kmin = 0xffffu;               // generic path: extrema as fp16 keys
        float dmin2 = INFINITY, dmax2 = 0.f;                 // fast path: extrema of d^2 over valid rows
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const long long row = tile * TC_BM + r;
            const bool rv = row < P.n;
            float b1 = INFINITY, b2 = INFINITY;              // carried across the phases of a WIDE tile
            int bi = 0;
            float mx = 0.f;
            for (int p = 0; p < nph; ++p) {
                const bool last = p == nph - 1;
                const int kp = p * TC_PHASE_COLS;            // global index of the phase's first column
                const int ncol = WIDE ? (last ? P.kc_last : TC_PHASE_COLS) : KC;
                mbar_wait(&x2_full[a], aph);
                const float xn = x2s[a * TC_BM + r];
                mbar_wait(&tmem_full[a], aph);
                tc_fence_after();
                if (fast) {
                    // argmin / runner-up on d^2 (sqrt is monotone; identical d^2 keep the first index like
                    // torch.argmin); sqrt only where the fp16 score is actually stored
                    __half* sp = (P.o.scores_t && rv) ? P.o.scores_t + row : nullptr;
                    const long long ld = P.o.ld;
                    for (int c0 = 0; c0 < ncol; c0 += 32) {
                        if (P.debug & 1) break;
                        uint32_t v[32];
                        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * P.tmem_cols + c0), v);
                        float cw[32];
                        if (WIDE) load_c2_32(P.c2 + kp + c0, cw);
                        tmem_ld_wait();
                        const bool whole = (kp + c0 + 32 <= P.K);
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int k = kp + c0 + j;
                            if (whole || k < P.K) {
                                const float d2 = fmaxf(fmaf(-2.f, __uint_as_float(v[j]), xn + (WIDE ? cw[j] : c2s[k])), 0.f);
                                if (d2 < b1) { b2 = b1; b1 = d2; bi = k; }
                                else if (d2 < b2) b2 = d2;
                                mx = fmaxf(mx, d2);
                                // one 2-byte store per entry, 64 contiguous bytes per warp.  (Staging the tile through shared
                                // memory for 16-byte stores was measured on B200: slower, 0.86 vs 0.82 ms at K = 128 and 1.70 vs
                                // 1.43 ms at K = 256 per 1 M rows - the barriers and the lost raw-ring slot cost more.)
                                if (sp) sp[(long long)k * ld] = __float2half_rn(-sqrtf(d2));
                            }
                        }
                    }
                    if (last) {
                        if (rv) { dmin2 = fminf(dmin2, b1); dmax2 = fmaxf(dmax2, mx); }
                        b1 = sqrtf(b1);
                        b2 = sqrtf(b2);
                    }
                } else {
                    const int pid = (rv && P.o.mask_ids) ? P.o.mask_ids[row] : -1;
                    const int mlo = pid * P.o.mask_block, mhi = mlo + P.o.mask_block;
                    for (int c0 = 0; c0 < ncol; c0 += 32) {
                        if (P.debug & 1) break;
                        uint32_t v[32];
                        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * P.tmem_cols + c0), v);
                        float cw[32];
                        if (WIDE) load_c2_32(P.c2 + kp + c0, cw);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int k = kp + c0 + j;
                            if (k < P.K) {
                                float d2 = fmaf(-2.f, __uint_as_float(v[j]), xn + (WIDE ? cw[j] : c2s[k]));
                                float d = sqrtf(fmaxf(d2, 0.f));
                                if (P.o.dist && rv) P.o.dist[row * P.K + k] = d;
                                if (P.o.scores_t && rv) {
                                    __half h = __float2half_rn(-d);
                                    P.o.scores_t[(long long)k * P.o.ld + row] = h;
                                    unsigned int key = h2key(h2bits(h));
                                    kmax = max(kmax, key);
                                    kmin = min(kmin, key);
                                }
                                float dd = P.o.farthest ? -d : d;
                                if (pid >= 0 && (k < mlo || k >= mhi)) dd = d + 10000.0f;
                                if (dd < b1) { b2 = b1; b1 = dd; bi = k; }
                                else if (dd < b2) b2 = dd;
                            }
                        }
                    }
                    if (last && P.o.farthest) { b1 = -b1; b2 = -b2; }
                }
                tc_fence_before();
                mbar_arrive(&tmem_empty[a]);
                if (last && rv) {
                    if (P.o.argmin) P.o.argmin[row] = bi;
                    if (P.o.best2) { P.o.best2[row * 2] = b1; P.o.best2[row * 2 + 1] = b2; }
                    if (P.o.counts) atomicAdd(WIDE ? &P.o.counts[bi] : &cnt_s[bi], 1);
                }
                if (++a == 2) { a = 0; aph ^= 1; }
            }
        }
        if (P.o.scores_t && P.o.minmax_keys) {
            if (fast && dmin2 <= dmax2) {                    // rounding is monotone: extrema of half(-d) from those of d^2
                kmax = h2key(h2bits(__float2half_rn(-sqrtf(dmin2))));
                kmin = h2key(h2bits(__float2half_rn(-sqrtf(dmax2))));
            }
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, off));
                kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, off));
            }
            if (lane == 0 && kmin <= kmax) {
                atomicMax(&P.o.minmax_keys[0], kmax);
                atomicMin(&P.o.minmax_keys[1], kmin);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (!WIDE && P.o.counts)
        for (int i = threadIdx.x; i < P.K; i += TC_THREADS)
            if (cnt_s[i]) atomicAdd(&P.o.counts[i], cnt_s[i]);
    if (warp == TC_MMA_WARP) {
        uint32_t ncols = (uint32_t)P.tmem_alloc;
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// centroid preparation: hi = rna_tf32(c), lo = rna_tf32(c - hi), |c|^2
__global__ void centroid_split_kernel(const float* __restrict__ c, int K, int dim, float* __restrict__ chi,
                                      float* __restrict__ clo, float* __restrict__ c2) {
    const int k = blockIdx.x;
    float s = 0.f;
    for (int d = threadIdx.x; d < dim; d += blockDim.x) {
        float v = c[(long long)k * dim + d];
        float h = to_tf32_rna(v);
        chi[(long long)k * dim + d] = h;
        clo[(long long)k * dim + d] = to_tf32_rna(v - h);
        s = fmaf(v, v, s);
    }
    __shared__ float red[32];
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < (blockDim.x + 31) / 32; ++i) t += red[i];
        c2[k] = t;
    }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

int make_map_2d(CUtensorMap* m, const float* base, long long rows, int dim, int box_rows, CUtensorMapL2promotion l2) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return fail(RQK_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver%s");
    cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)dim * 4};
    cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(RQK_ERR_CUDA, "cuTensorMapEncodeTiled failed (%s%lld)", "", (long long)r);
    return 0;
}

// workspace: chi [K][dim], clo [K][dim], c2 [K]
int score_pass_tc(const float* x, long long n, int dim, const float* c, int K, float* chi, float* clo, float* c2,
                  const ScoreOut& o, int num_sms, cudaStream_t stream) {
    if (n == 0) return 0;
    // K > 256: phases of 256 columns (WIDE kernel); the operand stages, TMA box and accumulators are those of K = 256
    const bool wide = K > TC_PHASE_COLS;
    const int KC = wide ? TC_PHASE_COLS : round_up(K, 16);
    int tcols = 32;
    while (tcols < KC) tcols <<= 1;
    ScoreTcParams P;
    P.n = n; P.dim = dim; P.K = K; P.KC = KC; P.tmem_cols = tcols;
    P.c2 = c2; P.o = o;
    P.phases = wide ? ceil_div(K, TC_PHASE_COLS) : 1;
    P.kc_last = wide ? round_up(K - TC_PHASE_COLS * (P.phases - 1), 16) : KC;
    {
        const char* dbg = getenv("RQK_SCORE_DEBUG");
        P.debug = dbg ? atoi(dbg) : 0;
    }
    // K <= 128: two accumulators leave at least 256 TMEM columns, enough for four 64-column A-operand stages
    static const bool no_atmem = [] { const char* e = getenv("RQK_SCORE_A_SMEM"); return e && e[0] == '1'; }();
    const bool atmem = !no_atmem && 2 * tcols + 4 * 2 * TC_BK <= 512;
    const size_t stage_bytes = (atmem ? 0 : 2 * (size_t)TC_BM * TC_BK * 4) + 2 * (size_t)KC * TC_BK * 4;
    const size_t tail = 8 * 8 * 3 + 2 * 8 * 3 + 2 * 8 * TC_MAX_RAW + 16 + 2 * TC_BM * 4 + 256 * 4 + 256 * 4 + 64;
    const size_t raw_bytes = (size_t)TC_BM * TC_BK * 4;
    const long long room = 225 * 1024 - (long long)tail - 1024;
    // two operand stages (A hi/lo + centroid hi/lo blocks); the rest of shared memory is the raw X ring
    int stages = 2;
    int raw;
    if (atmem) {
        stages = 4;                                  // centroid blocks in smem + A blocks in TMEM, stage for stage
        raw = (int)((room - (long long)(stages * stage_bytes)) / (long long)raw_bytes);
        if (raw > TC_MAX_RAW) raw = TC_MAX_RAW;
        if (raw < 2) return fail(RQK_ERR_INTERNAL, "score_pass_tc: no room for the raw ring%s");
        P.a_col0 = 2 * tcols;
        int need = 2 * tcols + stages * 2 * TC_BK, alloc = 32;
        while (alloc < need) alloc <<= 1;
        P.tmem_alloc = alloc;
    } else {
        if (room < (long long)(stages * stage_bytes + raw_bytes))
            return fail(RQK_ERR_UNSUPPORTED, "score_pass_tc: K=%s%lld does not fit two pipeline stages", "", K);
        raw = (int)((room - (long long)(stages * stage_bytes)) / (long long)raw_bytes);
        if (raw > TC_MAX_RAW) {                      // small K: spend the surplus on a third operand stage
            if (room >= (long long)(3 * stage_bytes + 4 * raw_bytes)) {
                stages = 3;
                raw = (int)((room - (long long)(stages * stage_bytes)) / (long long)raw_bytes);
            }
            if (raw > TC_MAX_RAW) raw = TC_MAX_RAW;
        }
        P.a_col0 = 0;
        P.tmem_alloc = 2 * tcols;
    }
    P.stages = stages;
    P.raw = raw;
    const size_t smem = (size_t)stages * stage_bytes + (size_t)raw * raw_bytes + tail + 1024;

    centroid_split_kernel<<<K, 128, 0, stream>>>(c, K, dim, chi, clo, c2);
    RQK_LAUNCH_OK();
    CUtensorMap mx, mhi, mlo;
    int rc;
    if ((rc = make_map_2d(&mx, x, n, dim, TC_BM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B))) return rc;
    if ((rc = make_map_2d(&mhi, chi, K, dim, KC, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))) return rc;
    if ((rc = make_map_2d(&mlo, clo, K, dim, KC, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))) return rc;
    auto kern = wide ? score_tc_kernel<false, true> : atmem ? score_tc_kernel<true> : score_tc_kernel<false>;
    RQK_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long ntiles = ceil_div<long long>(n, TC_BM);
    int grid = (int)(ntiles < num_sms ? ntiles : num_sms);
    kern<<<grid, TC_THREADS, smem, stream>>>(mx, mhi, mlo, P);
    RQK_LAUNCH_OK();
    return 0;
}

}  // namespace rqk
