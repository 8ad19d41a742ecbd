// Whiten-colour transform (ops.py:24-140) and AdaIN (ops.py:282-294) for one relu level,
// batched over frames.
//
// Stage A  channel sums / covariance        HBM-bound streaming kernels (fp32 FFMA, fp64 combine)
// Stage B  C x C symmetric eigendecomposition: one-sided (Hestenes) Jacobi, one pair per warp,
//          columns staged in shared memory, a thread-block CLUSTER of C/64 CTAs per matrix
// Stage C  W_c = E_c D_c^-1/2 E_c^T, C_s = E_s D_s^1/2 E_s^T, T = C_s W_c, M = aT + (1-a)I, bias
// Stage D  out = M x + bias : the 1-tap mode of the tcgen05 conv kernel (conv_tc.cu) with a
//          per-frame weight set, so the apply GEMM runs on the tensor cores.
#include <cooperative_groups.h>

#include "common.cuh"
#include "jacobi_common.cuh"

namespace cg = cooperative_groups;

namespace wctb {

// ---------------------------------------------------------------------------
// Stage A.1: per-channel sums (and sums of squares) over the interior pixels
//   grid (chunks, problems); 256 threads; thread = (row lane, 8-channel group)
// ---------------------------------------------------------------------------
template <bool SQ>
__global__ void __launch_bounds__(256)
k_chan_sums(const __half* __restrict__ act, ActGeom g, int chunk_pix, double* __restrict__ sum, double* __restrict__ sumsq,
            const uint8_t* __restrict__ labels = nullptr) {
    // labels (optional, [N][H][W]): grid.z = R regions, sums of the pixels labelled blockIdx.z into item n * R + region
    __shared__ float red[256 * 8];
    __shared__ float red2[SQ ? 256 * 8 : 8];
    const int cgs = g.C / 8;
    const int rows = 256 / cgs;                 // pixel rows handled per iteration (C <= 2048)
    const int grp = threadIdx.x % cgs;
    const int rl = threadIdx.x / cgs;
    const int n = blockIdx.y;
    const int region = blockIdx.z;
    const long long item = (long long)n * gridDim.z + region;
    const long long HW = (long long)g.H * g.W;
    const long long q0 = (long long)blockIdx.x * chunk_pix;
    const long long q1 = min(q0 + chunk_pix, HW);
    float s[8], s2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] = 0.f; s2[j] = 0.f; }
    if (rl < rows) {
        for (long long q = q0 + rl; q < q1; q += rows) {
            if (labels && labels[(long long)n * HW + q] != region) continue;
            const int y = (int)((unsigned)q / (unsigned)g.W), x = (int)((unsigned)q - (unsigned)y * (unsigned)g.W);
            float v[8];
            load8(act, g, ((long long)n * g.Hp + y + 1) * g.Wp + x + 1, grp * 8, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                s[j] += v[j];
                if (SQ) s2[j] = fmaf(v[j], v[j], s2[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        red[threadIdx.x * 8 + j] = s[j];
        if (SQ) red2[threadIdx.x * 8 + j] = s2[j];
    }
    __syncthreads();
    // thread t < C reduces channel t over the row lanes
    for (int c = threadIdx.x; c < g.C; c += 256) {
        const int gq = c / 8, j = c % 8;
        float a = 0.f, a2 = 0.f;
        for (int r = 0; r < rows; ++r) {
            a += red[(r * cgs + gq) * 8 + j];
            if (SQ) a2 += red2[(r * cgs + gq) * 8 + j];
        }
        atomicAdd(&sum[item * g.C + c], (double)a);
        if (SQ) atomicAdd(&sumsq[item * g.C + c], (double)a2);
    }
}

__global__ void k_mean_finalize(const double* __restrict__ sum, const double* __restrict__ sumsq, long long HW0, int total,
                                float* __restrict__ mean, float* __restrict__ var, const int* __restrict__ counts = nullptr,
                                int C = 1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long HW = counts ? (counts[i / C] > 0 ? counts[i / C] : 1) : HW0;   // regions: pixels of item i / C
    const double m = sum[i] / (double)HW;
    mean[i] = (float)m;
    if (var) var[i] = (float)fmax(sumsq[i] / (double)HW - m * m, 0.0);   // biased variance (tf.nn.moments)
}

// ---------------------------------------------------------------------------
// Stage B: one-sided Jacobi.  Matrix n x n (n = 64*P), columns contiguous
//   (symmetric input, so row-major == column-major).  A cluster of P CTAs owns one
//   matrix; the 2P column blocks (32 columns each) are paired by a round-robin
//   tournament; a CTA stages its two blocks in shared memory, orthogonalises
//   all 32x32 cross pairs (one pair per warp, 32 warps), writes them back, and
//   the cluster barriers.  On convergence column i = sigma_i * u_i.
// ---------------------------------------------------------------------------
template <int NN>
struct JacobiCfg {
    static constexpr int P = NN / 64;
    static constexpr int VEC = NN >= 128 ? 4 : 2;        // floats per lane per load
    static constexpr int NV = NN / (32 * VEC);           // vector loads per lane per column
    static constexpr int SMEM_BYTES = 64 * NN * 4 + 64;
};

// Two INDEPENDENT rotations (x0,y0) and (x1,y1) fused and branch-free so their long
// dependency chains (dot -> 5-step shuffle reduction -> MUFU chain -> rotation) interleave:
// the kernel is latency bound (ncu: 38 % issue utilisation with 16 warps per SM).
template <int HP>
__device__ __forceinline__ void rot_regs2(f32x2 (&x0)[HP], f32x2 (&y0)[HP], float& a0, float& b0, f32x2 (&x1)[HP],
                                          f32x2 (&y1)[HP], float& a1, float& b1, float tol2, float tolq2, float null2,
                                          float& flag) {
    f32x2 d00 = 0ull, d01 = 0ull, d10 = 0ull, d11 = 0ull;
#pragma unroll
    for (int i = 0; i < HP; ++i) {
        if (i & 1) { d01 = fma2(x0[i], y0[i], d01); d11 = fma2(x1[i], y1[i], d11); }
        else { d00 = fma2(x0[i], y0[i], d00); d10 = fma2(x1[i], y1[i], d10); }
    }
    float p0, p1, p2, p3, q0, q1, q2, q3;
    unpack2(d00, p0, p1); unpack2(d01, p2, p3);
    unpack2(d10, q0, q1); unpack2(d11, q2, q3);
    float g0 = (p0 + p1) + (p2 + p3);
    float g1 = (q0 + q1) + (q2 + q3);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        g0 += __shfl_xor_sync(0xffffffffu, g0, o);
        g1 += __shfl_xor_sync(0xffffffffu, g1, o);
    }
    float t0, s0, c0, t1, s1, c1;
    rot_scalars(g0, a0, b0, tol2, tolq2, null2, flag, t0, s0, c0);
    rot_scalars(g1, a1, b1, tol2, tolq2, null2, flag, t1, s1, c1);
    if (t0 != 0.f || t1 != 0.f) {          // warp-uniform: skip the FMAs only when BOTH pairs are already orthogonal
        const f32x2 s20 = pack2(s0, s0), ns20 = pack2(-s0, -s0), c20 = pack2(c0, c0);
        const f32x2 s21 = pack2(s1, s1), ns21 = pack2(-s1, -s1), c21 = pack2(c1, c1);
#pragma unroll
        for (int i = 0; i < HP; ++i) {
            const f32x2 xa = x0[i], ya = y0[i], xb = x1[i], yb = y1[i];
            x0[i] = fma2(c20, xa, fma2(ns20, ya, xa));       // x' = x + cm1*x - s*y
            y0[i] = fma2(c20, ya, fma2(s20, xa, ya));        // y' = y + cm1*y + s*x
            x1[i] = fma2(c21, xb, fma2(ns21, yb, xb));
            y1[i] = fma2(c21, yb, fma2(s21, xb, yb));
        }
        a0 = fmaxf(fmaf(-t0, g0, a0), 0.f); b0 = fmaxf(fmaf(t0, g0, b0), 0.f);   // |x'|^2 = |x|^2 - t g , |y'|^2 = |y|^2 + t g
        a1 = fmaxf(fmaf(-t1, g1, a1), 0.f); b1 = fmaxf(fmaf(t1, g1, b1), 0.f);
    }
}

template <int NN>
__device__ __forceinline__ void load_col(const float* __restrict__ c, int lane, f32x2 (&r)[NN / 64]) {
    using Cfg = JacobiCfg<NN>;
#pragma unroll
    for (int v = 0; v < Cfg::NV; ++v) {
        const int off = (v * 32 + lane) * Cfg::VEC;
        if (Cfg::VEC == 4) {
            const ulonglong2 a = *reinterpret_cast<const ulonglong2*>(c + off);
            r[v * 2] = a.x;
            r[v * 2 + 1] = a.y;
        } else {
            r[v] = *reinterpret_cast<const unsigned long long*>(c + off);
        }
    }
}
template <int NN>
__device__ __forceinline__ void store_col(float* __restrict__ c, int lane, const f32x2 (&r)[NN / 64]) {
    using Cfg = JacobiCfg<NN>;
#pragma unroll
    for (int v = 0; v < Cfg::NV; ++v) {
        const int off = (v * 32 + lane) * Cfg::VEC;
        if (Cfg::VEC == 4) *reinterpret_cast<ulonglong2*>(c + off) = make_ulonglong2(r[v * 2], r[v * 2 + 1]);
        else *reinterpret_cast<unsigned long long*>(c + off) = r[v];
    }
}

__device__ __forceinline__ void group_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// All pairs between the two columns x0,x1 held in REGISTERS by this warp (cached squared norms a0,a1) and the
// `npairs` column pairs of the shared-memory sub-block starting at bot0: npairs steps x 4 rotations.  Each bottom
// pair is loaded/stored once per 4 rotations, column norms are cached in nrm[] and updated analytically, so a
// rotation costs one dot product instead of three.  The `npairs` warps that share the sub-block form a ring
// (warp wsub starts at pair wsub) and synchronise on their own named barrier `bar` (32*npairs threads): groups
// working on disjoint sub-blocks run out of phase, so one group's FMA bursts fill the other's latency chains.
template <int NN>
__device__ __forceinline__ void ring_steps(float* cols, float* nrm, f32x2 (&x0)[NN / 64], f32x2 (&x1)[NN / 64], float& a0,
                                           float& a1, int bot0, int npairs, int wsub, int bar, int lane, float tol2,
                                           float tolq2, float null2, float& flag) {
    constexpr int HP = NN / 64;
    for (int s = 0; s < npairs; ++s) {
        const int j = bot0 + 2 * ((wsub + s) & (npairs - 1));
        float* cy0 = cols + j * NN;
        float* cy1 = cy0 + NN;
        f32x2 y0[HP], y1[HP];
        load_col<NN>(cy0, lane, y0);
        load_col<NN>(cy1, lane, y1);
        float b0 = nrm[j], b1 = nrm[j + 1];
        rot_regs2<HP>(x0, y0, a0, b0, x1, y1, a1, b1, tol2, tolq2, null2, flag);
        rot_regs2<HP>(x0, y1, a0, b1, x1, y0, a1, b0, tol2, tolq2, null2, flag);
        store_col<NN>(cy0, lane, y0);
        store_col<NN>(cy1, lane, y1);
        if (lane == 0) { nrm[j] = b0; nrm[j + 1] = b1; }
        if (npairs > 1) group_bar(bar, 32 * npairs);
        else __syncwarp();
    }
}

// tops (top, top+1) from shared memory, one ring pass, tops back to shared memory (the pairs INSIDE a block)
template <int NN>
__device__ __forceinline__ void cross_steps(float* cols, float* nrm, int top, int bot0, int npairs, int wsub, int bar,
                                            int lane, float tol2, float tolq2, float null2, float& flag) {
    constexpr int HP = NN / 64;
    f32x2 x0[HP], x1[HP];
    load_col<NN>(cols + top * NN, lane, x0);
    load_col<NN>(cols + (top + 1) * NN, lane, x1);
    float a0 = nrm[top], a1 = nrm[top + 1];
    ring_steps<NN>(cols, nrm, x0, x1, a0, a1, bot0, npairs, wsub, bar, lane, tol2, tolq2, null2, flag);
    store_col<NN>(cols + top * NN, lane, x0);
    store_col<NN>(cols + (top + 1) * NN, lane, x1);
    if (lane == 0) { nrm[top] = a0; nrm[top + 1] = a1; }
}

// 512 threads = 16 warps, 64 columns (a "top" and a "bottom" block of 32) in shared memory.
//   every round : the 32x32 cross pairs: warp w keeps top columns 2w,2w+1 in registers; the warps split into
//                 2^lg groups, group g walks bottom sub-block g^h in sub-round h (ring of 16>>lg warps on a named
//                 barrier), groups start `stagger` cycles apart so that they stay out of phase;
//   round 0     : additionally the pairs INSIDE both blocks, by recursive halving with the same register-blocked
//                 step (16|16 -> 8|8 -> 4|4 -> 2|2 -> 1|1 : 8+4+2+1+1 steps instead of 62 one-pair-per-warp steps).
__device__ float g_jacobi_tolq = 1e-4f;   // predicted-convergence level (see k_jacobi); device global so a probe can vary it

template <int NN>
__global__ void __launch_bounds__(512, 1)
k_jacobi(float* __restrict__ Gall, float* __restrict__ conv_ws, int* __restrict__ sweeps_out, int max_sweeps, float tol,
         int lg, int stagger, const int* __restrict__ skip) {
    if (skip && skip[blockIdx.y]) {          // matrix handled by the matrix-function fast path (matfun_tc.cu): whole cluster leaves
        if (blockIdx.x == 0 && threadIdx.x == 0 && sweeps_out) sweeps_out[blockIdx.y] = 0;
        return;
    }
    using Cfg = JacobiCfg<NN>;
    constexpr int P = Cfg::P;
    constexpr int NB = 2 * P;
    constexpr int M = NB - 1;
    constexpr int HP = NN / 64;
    extern __shared__ __align__(16) float cols[];          // [64][NN]
    __shared__ float nrm[64];
    __shared__ unsigned int s_max, s_amax;

    const int rank = blockIdx.x;
    const int prob = blockIdx.y;
    float* G = Gall + (long long)prob * NN * NN;
    float* cw = conv_ws + (long long)prob * 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    cg::cluster_group cluster = cg::this_cluster();

    // Every pair is rotated, including columns that have collapsed to rounding noise: keeping the noise
    // columns orthogonal to the large ones is what makes their Rayleigh quotients (k_rayleigh) second-order
    // small.  (A variant that left columns below 4*eps*max|column| alone was measured: the untouched columns
    // keep large range-space components and their Rayleigh quotients are O(lambda).)
    const float tol2 = tol * tol;
    // Quadratic convergence: a sweep whose largest cosine was rho leaves ~rho^2 behind.  When a sweep saw
    // nothing above tol_q = 1e-4 (rho^2 = 1e-8 << tol ~ 2.7e-6) its own rotations already finished the job and
    // the verification sweep (no rotations, ~60 % of a sweep's cost) is skipped.
    const float tolq2 = g_jacobi_tolq * g_jacobi_tolq;

    float null2 = 0.f;                                 // noise floor of the previous sweep (0: every pair is live)
    int sweep = 0;
    for (; sweep < max_sweeps; ++sweep) {
        if (threadIdx.x == 0) { s_max = 0u; s_amax = 0u; }
        float flag = 0.f, amax = 0.f;
        for (int r = 0; r < (P == 1 ? 1 : M); ++r) {
            int bt, bb;
            if (P == 1) { bt = 0; bb = 1; }
            else if (rank == 0) { bt = NB - 1; bb = r; }
            else { bt = (r + rank) % M; bb = (r - rank + M) % M; }
            if (P > 1 || sweep == 0) {
                const float4* s0 = reinterpret_cast<const float4*>(G + (long long)bt * 32 * NN);
                const float4* s1 = reinterpret_cast<const float4*>(G + (long long)bb * 32 * NN);
                float4* d = reinterpret_cast<float4*>(cols);
                for (int i = threadIdx.x; i < 32 * NN / 4; i += 512) {
                    d[i] = __ldcg(s0 + i);                 // L2 (peers of the cluster wrote these columns)
                    d[32 * NN / 4 + i] = __ldcg(s1 + i);
                }
            }
            __syncthreads();
            // ---- column norms (fresh every round: the cached values never drift far)
            for (int c = warp * 4; c < warp * 4 + 4; ++c) {
                f32x2 v[HP];
                load_col<NN>(cols + c * NN, lane, v);
                f32x2 q = 0ull;
#pragma unroll
                for (int i = 0; i < HP; ++i) q = fma2(v[i], v[i], q);
                float q0, q1;
                unpack2(q, q0, q1);
                float ss = q0 + q1;
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                if (lane == 0) nrm[c] = ss;
                amax = fmaxf(amax, ss);
            }
            __syncthreads();
            // ---- pairs inside each 32-column block: once per sweep
            if (r == 0) {
                for (int lv = 3; lv >= 0; --lv) {          // sub-block halves of 16, 8, 4, 2 columns
                    const int wpg = 1 << lv;               // warps per sub-block pair = column pairs per half
                    const int base = (warp >> lv) * (4 << lv);
                    cross_steps<NN>(cols, nrm, base + 2 * (warp & (wpg - 1)), base + (2 << lv), wpg, warp & (wpg - 1),
                                    1 + (warp >> lv), lane, tol2, tolq2, null2, flag);
                    __syncthreads();
                }
                {   // 1|1 : columns (4w,4w+1) and (4w+2,4w+3)
                    f32x2 x0[HP], y0[HP], x1[HP], y1[HP];
                    float* c0 = cols + 4 * warp * NN;
                    load_col<NN>(c0, lane, x0);
                    load_col<NN>(c0 + NN, lane, y0);
                    load_col<NN>(c0 + 2 * NN, lane, x1);
                    load_col<NN>(c0 + 3 * NN, lane, y1);
                    float a0 = nrm[4 * warp], b0 = nrm[4 * warp + 1], a1 = nrm[4 * warp + 2], b1 = nrm[4 * warp + 3];
                    rot_regs2<HP>(x0, y0, a0, b0, x1, y1, a1, b1, tol2, tolq2, null2, flag);
                    store_col<NN>(c0, lane, x0);
                    store_col<NN>(c0 + NN, lane, y0);
                    store_col<NN>(c0 + 2 * NN, lane, x1);
                    store_col<NN>(c0 + 3 * NN, lane, y1);
                    if (lane == 0) { nrm[4 * warp] = a0; nrm[4 * warp + 1] = b0; nrm[4 * warp + 2] = a1; nrm[4 * warp + 3] = b1; }
                    __syncthreads();
                }
            }
            // ---- cross pairs: 16 steps x 4 rotations per warp
            {
                f32x2 x0[HP], x1[HP];
                load_col<NN>(cols + 2 * warp * NN, lane, x0);
                load_col<NN>(cols + (2 * warp + 1) * NN, lane, x1);
                float a0 = nrm[2 * warp], a1 = nrm[2 * warp + 1];
                const int ring = 16 >> lg;                         // warps per group = bottom pairs per sub-block
                const int grp = warp / ring, wsub = warp & (ring - 1);
                for (int h = 0; h < (1 << lg); ++h) {
                    if (stagger > 0 && grp > 0) {
                        const long long t0 = clock64();
                        while (clock64() - t0 < (long long)grp * stagger) {}
                    }
                    ring_steps<NN>(cols, nrm, x0, x1, a0, a1, 32 + 2 * ring * (grp ^ h), ring, wsub, 1 + grp, lane, tol2,
                                   tolq2, null2, flag);
                    __syncthreads();
                }
                store_col<NN>(cols + 2 * warp * NN, lane, x0);
                store_col<NN>(cols + (2 * warp + 1) * NN, lane, x1);
                __syncthreads();
            }
            if (P > 1) {
                float4* d0 = reinterpret_cast<float4*>(G + (long long)bt * 32 * NN);
                float4* d1 = reinterpret_cast<float4*>(G + (long long)bb * 32 * NN);
                const float4* sc = reinterpret_cast<const float4*>(cols);
                for (int i = threadIdx.x; i < 32 * NN / 4; i += 512) {
                    d0[i] = sc[i];
                    d1[i] = sc[32 * NN / 4 + i];
                }
                __threadfence();
                cluster.sync();   // release/acquire: next round reads what the peers just wrote
            }
        }
        // ---- convergence: worst pair class seen in this sweep (0 / 1 / 2), agreed across the cluster
        if (lane == 0) { atomicMax(&s_max, __float_as_uint(flag)); atomicMax(&s_amax, __float_as_uint(amax)); }
        __syncthreads();
        float gmax = __uint_as_float(s_max);
        float amx = __uint_as_float(s_amax);
        if (P > 1) {
            if (threadIdx.x == 0) {
                reinterpret_cast<volatile float*>(cw)[rank] = gmax;
                reinterpret_cast<volatile float*>(cw)[8 + rank] = amx;
                __threadfence();
            }
            cluster.sync();
            gmax = 0.f;
            amx = 0.f;
            for (int i = 0; i < P; ++i) {
                gmax = fmaxf(gmax, reinterpret_cast<volatile float*>(cw)[i]);
                amx = fmaxf(amx, reinterpret_cast<volatile float*>(cw)[8 + i]);
            }
            cluster.sync();   // everyone has read before the next sweep overwrites
        }
        null2 = 1e-11f * amx;                          // |column| < 3e-6 of the largest column: below what fp32 resolves in A
        __syncthreads();
        if (gmax < 2.f) { ++sweep; break; }
    }
    if (P == 1) {
        float4* d = reinterpret_cast<float4*>(G);
        const float4* sc = reinterpret_cast<const float4*>(cols);
        for (int i = threadIdx.x; i < 64 * NN / 4; i += 512) d[i] = sc[i];
    }
    if (rank == 0 && threadIdx.x == 0 && sweeps_out) sweeps_out[prob] = sweep;
}

// Rayleigh quotients  lambda_i = g_i^T A g_i / |g_i|^2  of the converged columns against the ORIGINAL matrix.
// The column norm |g_i| is a first-order eigenvalue estimate: on a rank-deficient map the null columns
// keep the rounding noise of the cancellations that created them (measured 4e-7*lambda_max, i.e. above
// the 1e-5 cut for lambda_max > 25; LAPACK: 4e-8*lambda_max).  The Rayleigh quotient is second order in
// that noise: the same null columns give ~1e-8.   grid (C/16, problems), C threads.
__global__ void __launch_bounds__(512)
k_rayleigh(const float* __restrict__ A0all, const float* __restrict__ Gall, int C, float* __restrict__ lam,
           const int* __restrict__ skip) {
    if (skip && skip[blockIdx.y]) return;
    __shared__ __align__(16) float gs[512 * 16];
    __shared__ float red_q[16][17], red_s[16][17];     // [warp][column]: fixed-order (deterministic) reduction
    const int prob = blockIdx.y, j0 = blockIdx.x * 16, r = threadIdx.x;
    const float* A0 = A0all + (long long)prob * C * C;
    const float* G = Gall + (long long)prob * C * C;
    float mine[16];
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) {
        mine[jj] = G[(long long)(j0 + jj) * C + r];          // column j0+jj, row r (coalesced over r)
        gs[r * 16 + jj] = mine[jj];
    }
    __syncthreads();
    float acc[16];
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) acc[jj] = 0.f;
    // 8 rows of A in flight per thread: the loop is a chain of dependent L2 loads otherwise (measured 311 us per launch
    // of 16 matrices at C = 512 for 33 MB of traffic)
#pragma unroll 1
    for (int k8 = 0; k8 < C; k8 += 8) {
        float av[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) av[u] = __ldg(A0 + (long long)(k8 + u) * C + r);   // A symmetric: row k read as column k, coalesced over r
#pragma unroll
        for (int u = 0; u < 8; ++u) {
        const int k = k8 + u;
        const float a = av[u];
        const float4* g4 = reinterpret_cast<const float4*>(gs + k * 16);
        const float4 g0 = g4[0], g1 = g4[1], g2 = g4[2], g3 = g4[3];
        acc[0] = fmaf(a, g0.x, acc[0]); acc[1] = fmaf(a, g0.y, acc[1]); acc[2] = fmaf(a, g0.z, acc[2]); acc[3] = fmaf(a, g0.w, acc[3]);
        acc[4] = fmaf(a, g1.x, acc[4]); acc[5] = fmaf(a, g1.y, acc[5]); acc[6] = fmaf(a, g1.z, acc[6]); acc[7] = fmaf(a, g1.w, acc[7]);
        acc[8] = fmaf(a, g2.x, acc[8]); acc[9] = fmaf(a, g2.y, acc[9]); acc[10] = fmaf(a, g2.z, acc[10]); acc[11] = fmaf(a, g2.w, acc[11]);
        acc[12] = fmaf(a, g3.x, acc[12]); acc[13] = fmaf(a, g3.y, acc[13]); acc[14] = fmaf(a, g3.z, acc[14]); acc[15] = fmaf(a, g3.w, acc[15]);
        }
    }
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) {
        float q = mine[jj] * acc[jj], ss = mine[jj] * mine[jj];
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            q += __shfl_xor_sync(0xffffffffu, q, o);
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
        }
        if (lane == 0) { red_q[threadIdx.x >> 5][jj] = q; red_s[threadIdx.x >> 5][jj] = ss; }
    }
    __syncthreads();
    if (r < 16) {
        float q = 0.f, ss = 0.f;
        for (int w = 0; w < (C >> 5); ++w) { q += red_q[w][r]; ss += red_s[w][r]; }
        lam[(long long)prob * C + j0 + r] = ss > 0.f ? q / ss : 0.f;
    }
}

// eigenvalue estimate (Rayleigh quotient when `lam` is given, else |column i|); per-problem kept count;
// scaling d_i of the rank-k reconstruction
//   mode 0 (content, whitening): d = (sigma+eps_eig)^-1/2 / sigma^2
//   mode 1 (style, colouring)  : d = (sigma+eps_eig)^+1/2 / sigma^2
//   so that  E_k f(S_k) E_k^T = G diag(d) G^T  with G's columns = sigma_i u_i.
__global__ void k_eig_post(const float* __restrict__ Gall, const float* __restrict__ lam, int C, float thresh, float eps_eig,
                           int n_content, float* __restrict__ sigma, float* __restrict__ dvec, int* __restrict__ kcount,
                           const int* __restrict__ skip) {
    const int prob = blockIdx.y;
    if (skip && skip[prob]) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int col = blockIdx.x * (blockDim.x >> 5) + warp;
    if (col >= C) return;
    const float* g = Gall + ((long long)prob * C + col) * C;
    float ss = 0.f;
    for (int i = lane; i < C; i += 32) ss = fmaf(g[i], g[i], ss);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (lane == 0) {
        const float sg = lam ? fabsf(lam[(long long)prob * C + col]) : sqrtf(ss);   // |lambda| like the SVD of ops.py:54,110
        sigma[(long long)prob * C + col] = sg;
        float d = 0.f;
        if (sg > thresh) {                                       // ops.py:68-69,112,125
            const float f = (prob < n_content) ? rsqrtf(sg + eps_eig) : sqrtf(sg + eps_eig);
            d = f / ss;
            if (kcount) atomicAdd(&kcount[prob], 1);
        }
        if (dvec) dvec[(long long)prob * C + col] = d;
    }
}

// ---------------------------------------------------------------------------
// Stage C: small dense products  Cm[i][j] = sum_k A[k][i] * d[k] * B[k][j]   (all n x n, k-major)
//   grid (n/64, n/64, batch); 256 threads, 4x4 per thread
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_outer_gemm(const float* __restrict__ A, long long sa, const float* __restrict__ B, long long sb,
             const float* __restrict__ d, long long sd, float* __restrict__ Cm, long long sc, int n,
             const int* __restrict__ skip = nullptr) {
    if (skip && skip[blockIdx.z]) return;      // this output was produced by the matrix-function fast path
    __shared__ __align__(16) float As[16][64];
    __shared__ __align__(16) float Bs[16][64];
    const int z = blockIdx.z;
    const float* a = A + (long long)z * sa;
    const float* b = B + (long long)z * sb;
    const float* dd = d ? d + (long long)z * sd : nullptr;
    const int i0 = blockIdx.x * 64, j0 = blockIdx.y * 64;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    const int lk = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;   // loader: 16 k-rows x 64 cols
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
    for (int k0 = 0; k0 < n; k0 += 16) {
        float4 av = *reinterpret_cast<const float4*>(a + (long long)(k0 + lk) * n + i0 + lc);
        const float4 bv = *reinterpret_cast<const float4*>(b + (long long)(k0 + lk) * n + j0 + lc);
        if (dd) {
            const float s = dd[k0 + lk];
            av.x *= s; av.y *= s; av.z *= s; av.w *= s;
        }
        __syncthreads();
        *reinterpret_cast<float4*>(&As[lk][lc]) = av;
        *reinterpret_cast<float4*>(&Bs[lk][lc]) = bv;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            const float4 x = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 y = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float xv[4] = {x.x, x.y, x.z, x.w};
            const float yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(xv[r], yv[c], acc[r][c]);
        }
    }
    float* cm = Cm + (long long)z * sc;
#pragma unroll
    for (int r = 0; r < 4; ++r)
        *reinterpret_cast<float4*>(cm + (long long)(i0 + ty * 4 + r) * n + j0 + tx * 4) =
            make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
}

// M = alpha*T + (1-alpha)*I  -> split-fp16 GEMM operand [frame][2][C][C] (row = output channel)
// bias = alpha*ms - M*mc + (1-alpha)*readd*mc                       (ops.py:80-83 / 131-133)
//   one warp per (frame, output channel)
__global__ void k_finalize_transform(const float* __restrict__ T, int C, int Nc, int Ns, float alpha, int readd,
                                     const float* __restrict__ mean_c, const float* __restrict__ mean_s,
                                     __half* __restrict__ Msplit, float* __restrict__ bias) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + warp;
    const int z = blockIdx.y;
    if (row >= C) return;
    const float* t = T + ((long long)z * C + row) * C;
    const float* mc = mean_c + (long long)z * C;
    const float* ms = mean_s + (long long)(z % Ns) * C;          // Ns = 1 (shared), Nc (per frame) or R (item z = frame*R + region)
    __half* mh = Msplit + (((long long)z * 2 + 0) * C + row) * C;
    __half* ml = Msplit + (((long long)z * 2 + 1) * C + row) * C;
    float dot = 0.f;
    for (int j = lane; j < C; j += 32) {
        const float m = alpha * t[j] + (j == row ? 1.f - alpha : 0.f);
        __half hi, lo;
        split_f32(m, hi, lo);
        mh[j] = hi;
        ml[j] = lo;
        dot = fmaf(m, mc[j], dot);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    if (lane == 0) bias[(long long)z * C + row] = alpha * ms[row] - dot + (readd ? (1.f - alpha) * mc[row] : 0.f);
}

// ---------------------------------------------------------------------------
// AdaIN (ops.py:282-294): per-(frame,channel) affine map
// ---------------------------------------------------------------------------
__global__ void k_adain_coeffs(const float* __restrict__ mean_c, const float* __restrict__ var_c,
                               const float* __restrict__ mean_s, const float* __restrict__ var_s, int C, int Nc, int Ns,
                               float alpha, float eps, float* __restrict__ scale, float* __restrict__ shift) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Nc * C) return;
    const int z = i / C, c = i % C;
    const int si = (z % Ns) * C + c;                                // Ns = 1, Nc, or R (item z = frame*R + region)
    const float inv = rsqrtf(var_c[i] + eps) * sqrtf(var_s[si]);   // batch_normalization(scale=sqrt(style_var))
    // y = (x - mc)*inv + ms ; out = alpha*y + (1-alpha)*x
    scale[i] = alpha * inv + (1.f - alpha);
    shift[i] = alpha * (mean_s[si] - mean_c[i] * inv);
}
__global__ void k_affine_apply(const __half* __restrict__ in, ActGeom g, const float* __restrict__ scale,
                               const float* __restrict__ shift, __half* __restrict__ out) {
    const int cgs = g.C / 8;
    const long long total = (long long)g.N * g.H * g.W * cgs;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < (unsigned)total; i += gridDim.x * blockDim.x) {
        const int c0 = (int)(i % (unsigned)cgs) * 8;
        unsigned pix = i / (unsigned)cgs;
        const int x = (int)(pix % (unsigned)g.W); pix /= (unsigned)g.W;
        const int y = (int)(pix % (unsigned)g.H);
        const int n = (int)(pix / (unsigned)g.H);
        float v[8];
        load8(in, g, ((long long)n * g.Hp + y + 1) * g.Wp + x + 1, c0, v);
        const float* sc = scale + (long long)n * g.C + c0;
        const float* sh = shift + (long long)n * g.C + c0;
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
        Half8 hi, lo;
        split8(v, hi, lo);
        store8_with_halo(out, g, n, y, x, c0, hi, lo);
    }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WctWs {
    size_t sum, sumsq, dsum, mean, var, G, A0, lam, sigma, dvec, Wc, Cs, T, Msplit, bias, conv, kcount, ok, scale, shift, total;
};
static WctWs wct_layout(int C, int Nc, int Ns) {
    WctWs w;
    const size_t np = (size_t)Nc + Ns;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    w.sum = take(np * C * 8);          // AdaIN: fp64 sums / sums of squares (contiguous: one memset clears both)
    w.sumsq = take(np * C * 8);
    w.dsum = take(np * C * 8);         // WCT: fp64 sums of the shifted features (cov_tc.cu)
    w.mean = take(np * C * 4);
    w.var = take(np * C * 4);
    w.G = take(np * C * C * 4);
    w.A0 = take(np * C * C * 4);
    w.lam = take(np * C * 4);
    w.sigma = take(np * C * 4);
    w.dvec = take(np * C * 4);
    w.Wc = take((size_t)Nc * C * C * 4);
    w.Cs = take((size_t)Ns * C * C * 4);
    w.T = take((size_t)Nc * C * C * 4);
    w.Msplit = take((size_t)Nc * 2 * C * C * 2);
    w.bias = take((size_t)Nc * C * 4);
    w.conv = take(np * 16 * 4);
    w.kcount = take(np * 2 * 4);
    w.ok = take(np * 4);               // matrices whose W / C_s came from the matrix-function fast path (matfun_tc.cu)
    w.scale = take((size_t)Nc * C * 4);
    w.shift = take((size_t)Nc * C * 4);
    w.total = o;
    return w;
}
size_t wct_workspace_bytes(int C, int Nc, int Ns) { return wct_layout(C, Nc, Ns).total; }

template <bool SQ>
static int launch_sums(const __half* act, ActGeom g, double* sum, double* sumsq, cudaStream_t st) {
    const long long HW = (long long)g.H * g.W;
    // enough blocks to fill the chip (~4 per SM) even for small feature maps, at most 1024 px per block
    long long chunk = (HW * g.N + 591) / 592;
    const int rows = 256 / (g.C / 8) > 0 ? 256 / (g.C / 8) : 1;
    chunk = (chunk + rows - 1) / rows * rows;
    if (chunk < rows) chunk = rows;
    if (chunk > 1024) chunk = 1024;
    dim3 grid((unsigned)cdiv(HW, chunk), (unsigned)g.N);
    k_chan_sums<SQ><<<grid, 256, 0, st>>>(act, g, chunk, sum, sumsq);
    WCTB_CHECK_LAUNCH("k_chan_sums");
    return 0;
}

// cross-phase schedule of k_jacobi: 2^lg warp groups, started `stagger` cycles apart (wctb200_debug_set_jacobi)
// -1 = auto: measured best on B200 (tools/jacobi_bench.py): C=512 -> 4 groups 300 cycles apart (6.76 ms vs 7.80 ms for
// one group), smaller matrices -> 2 groups 600 cycles apart.
int g_jacobi_lg = -1;
int g_jacobi_stagger = -1;
int set_jacobi_tolq(float v) {
    return cudaMemcpyToSymbol(g_jacobi_tolq, &v, sizeof(float)) == cudaSuccess ? 0 : -1;
}

int launch_jacobi(float* G, int C, int count, float* conv_ws, int* sweeps, cudaStream_t st, const int* skip) {
    const float tol = 2.f * sqrtf((float)C) * 5.96e-8f;
    const int max_sweeps = 40;
    const int lg = g_jacobi_lg >= 0 ? g_jacobi_lg : (C >= 512 ? 2 : 1);
    const int stagger = g_jacobi_stagger >= 0 ? g_jacobi_stagger : (C >= 512 ? 300 : 600);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(C / 64), (unsigned)count, 1);
    cfg.blockDim = dim3(512, 1, 1);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)(C / 64);
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
#define WCTB_JACOBI_CASE(NN)                                                                                         \
    case NN: {                                                                                                       \
        WCTB_ENSURE_SMEM(k_jacobi<NN>, JacobiCfg<NN>::SMEM_BYTES);                                                   \
        cfg.dynamicSmemBytes = JacobiCfg<NN>::SMEM_BYTES;                                                            \
        WCTB_CUDA(cudaLaunchKernelEx(&cfg, k_jacobi<NN>, G, conv_ws, sweeps, max_sweeps, tol, lg, stagger, skip));         \
        break;                                                                                                       \
    }
    switch (C) {
        WCTB_JACOBI_CASE(64)
        WCTB_JACOBI_CASE(128)
        WCTB_JACOBI_CASE(256)
        WCTB_JACOBI_CASE(512)
        default:
            set_error("jacobi: C=%d not in {64,128,256,512}", C);
            return WCTB200_EINVAL;
    }
#undef WCTB_JACOBI_CASE
    return 0;
}

int launch_eig_post(const float* G, const float* A0, float* lam, int C, int count, float thresh, float eps_eig,
                    int n_content, float* sigma, float* dvec, int* kcount, cudaStream_t st, const int* skip = nullptr) {
    if (A0 && lam) {
        dim3 gr((unsigned)(C / 16), (unsigned)count);
        k_rayleigh<<<gr, C, 0, st>>>(A0, G, C, lam, skip);
        WCTB_CHECK_LAUNCH("k_rayleigh");
    } else {
        lam = nullptr;
    }
    dim3 grid((unsigned)cdiv(C, 8), (unsigned)count);
    k_eig_post<<<grid, 256, 0, st>>>(G, lam, C, thresh, eps_eig, n_content, sigma, dvec, kcount, skip);
    WCTB_CHECK_LAUNCH("k_eig_post");
    return 0;
}

// matfun_tc.cu: A^-1/2 / A^+1/2 by coupled Newton-Schulz on the tensor cores where every eigenvalue is kept; ok[b] = 1 there
int launch_matfun_ns(const float* A, int C, int count, int n_first, float thresh, float eps_eig, float* out, int* ok, int* kcount,
                     cudaStream_t st, float* info = nullptr);
// cov_tc.cu: per-channel means and covariance (+ eps_cov I) in one pass over the features
int launch_mean_cov(const __half* act, ActGeom g, float eps_cov, float* mean, float* G, float* A0, double* dsum, cudaStream_t st,
                    const uint8_t* labels = nullptr, int R = 1, const int* counts = nullptr);

int launch_wct_level(const __half* content, int Nc, int Hc, int Wc, const __half* style, int Ns, int Hs, int Ws, int C,
                     float alpha, float eps_cov, float eps_eig, float thresh, int readd, __half* out, int32_t* k_out,
                     void* ws, size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "wct_level: C=%d not in {64,128,256,512}", C);
    WCTB_REQUIRE(Ns == 1 || Ns == Nc, "wct_level: Ns must be 1 or Nc");
    WCTB_REQUIRE(Hc >= 2 && Wc >= 2 && Hs >= 2 && Ws >= 2 && (long long)Hc * Wc >= 2 && (long long)Hs * Ws >= 2, "wct_level: bad geometry");
    const WctWs L = wct_layout(C, Nc, Ns);
    if (ws_bytes < L.total) {
        set_error("wct_level: workspace %zu < %zu bytes", ws_bytes, L.total);
        return WCTB200_EWS;
    }
    uint8_t* w = static_cast<uint8_t*>(ws);
    const int np = Nc + Ns;
    double* dsum = reinterpret_cast<double*>(w + L.dsum);
    float* mean = reinterpret_cast<float*>(w + L.mean);
    float* G = reinterpret_cast<float*>(w + L.G);
    float* sigma = reinterpret_cast<float*>(w + L.sigma);
    float* dvec = reinterpret_cast<float*>(w + L.dvec);
    float* Wcm = reinterpret_cast<float*>(w + L.Wc);
    float* Csm = reinterpret_cast<float*>(w + L.Cs);
    float* T = reinterpret_cast<float*>(w + L.T);
    __half* Msplit = reinterpret_cast<__half*>(w + L.Msplit);
    float* bias = reinterpret_cast<float*>(w + L.bias);
    float* conv = reinterpret_cast<float*>(w + L.conv);
    int* kc = reinterpret_cast<int*>(w + L.kcount);
    const long long CC = (long long)C * C;

    WCTB_CUDA(cudaMemsetAsync(kc, 0, (size_t)np * 2 * 4, st));
    ActGeom gc(Nc, Hc, Wc, C), gs(Ns, Hs, Ws, C);
    float* A0 = reinterpret_cast<float*>(w + L.A0);
    float* lam = reinterpret_cast<float*>(w + L.lam);
    int rc = launch_mean_cov(content, gc, eps_cov, mean, G, A0, dsum, st);
    if (rc) return rc;
    rc = launch_mean_cov(style, gs, eps_cov, mean + (long long)Nc * C, G + Nc * CC, A0 + Nc * CC, dsum + (long long)Nc * C, st);
    if (rc) return rc;
    // fast path first: W_c = A^-1/2, C_s = A^+1/2 straight from the covariances where the threshold keeps every eigenvalue
    int* ok = reinterpret_cast<int*>(w + L.ok);
    rc = launch_matfun_ns(A0, C, np, Nc, thresh, eps_eig, Wcm, ok, kc, st);        // Wc and Cs are contiguous in ws (Wc then Cs)
    if (rc < 0) return rc;
    rc = launch_jacobi(G, C, np, conv, kc + np, st, ok);
    if (rc) return rc;
    rc = launch_eig_post(G, A0, lam, C, np, thresh, eps_eig, Nc, sigma, dvec, kc, st, ok);
    if (rc) return rc;
    // W_c (whitening) per content frame, C_s (colouring) per style
    dim3 gg((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)np);
    k_outer_gemm<<<gg, 256, 0, st>>>(G, CC, G, CC, dvec, C, Wcm, CC, C, ok);
    WCTB_CHECK_LAUNCH("k_outer_gemm(W)");
    dim3 gt((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)Nc);
    k_outer_gemm<<<gt, 256, 0, st>>>(Csm, Ns == 1 ? 0 : CC, Wcm, CC, nullptr, 0, T, CC, C);   // T = C_s W_c (C_s symmetric)
    WCTB_CHECK_LAUNCH("k_outer_gemm(T)");
    dim3 gf((unsigned)cdiv(C, 8), (unsigned)Nc);
    k_finalize_transform<<<gf, 256, 0, st>>>(T, C, Nc, Ns, alpha, readd, mean, mean + (long long)Nc * C, Msplit, bias);
    WCTB_CHECK_LAUNCH("k_finalize_transform");
    // out = M x + bias on the tensor cores (1-tap conv, per-frame weight set)
    rc = launch_conv_tc(CONV_APPLY, content, Nc, Hc, Wc, C, Msplit, Nc, nullptr, bias, C, 0, out, st);
    if (rc) return rc;
    if (k_out) WCTB_CUDA(cudaMemcpyAsync(k_out, kc, (size_t)np * 2 * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

// ---------------------------------------------------------------------------
// Split form of the level transform: the style side (means, covariance, eigendecomposition,
// colouring matrix C_s) depends only on the style features, so the host runs it on a second
// stream where it overlaps the content encoder/decoder convolutions (the Jacobi kernel is
// latency bound and leaves the tensor cores idle), and caches it when a batch shares a style.
//   state layout: [Ns][C] mean_s | [Ns][C][C] C_s | [2*Ns] int32 (k_s, sweeps)
// ---------------------------------------------------------------------------
static size_t style_state_offsets(int C, int Ns, size_t* off_cs, size_t* off_k) {
    size_t o = align_up((size_t)Ns * C * 4, 256);
    *off_cs = o;
    o = align_up(o + (size_t)Ns * C * C * 4, 256);
    *off_k = o;
    return align_up(o + (size_t)Ns * 2 * 4, 256);
}
size_t wct_style_state_bytes(int C, int Ns) {
    size_t a, b;
    return style_state_offsets(C, Ns, &a, &b);
}

int launch_wct_style_prepare(const __half* style, int Ns, int Hs, int Ws, int C, float eps_cov, float eps_eig, float thresh,
                             void* state, void* ws, size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "wct_style_prepare: C=%d not in {64,128,256,512}", C);
    const WctWs L = wct_layout(C, 0, Ns);
    if (ws_bytes < L.total) {
        set_error("wct_style_prepare: workspace %zu < %zu bytes", ws_bytes, L.total);
        return WCTB200_EWS;
    }
    uint8_t* w = static_cast<uint8_t*>(ws);
    size_t off_cs, off_k;
    style_state_offsets(C, Ns, &off_cs, &off_k);
    uint8_t* sp = static_cast<uint8_t*>(state);
    float* mean_s = reinterpret_cast<float*>(sp);
    float* Cs = reinterpret_cast<float*>(sp + off_cs);
    int* kc = reinterpret_cast<int*>(sp + off_k);
    double* dsum = reinterpret_cast<double*>(w + L.dsum);
    float* G = reinterpret_cast<float*>(w + L.G);
    float* sigma = reinterpret_cast<float*>(w + L.sigma);
    float* dvec = reinterpret_cast<float*>(w + L.dvec);
    float* conv = reinterpret_cast<float*>(w + L.conv);
    const long long CC = (long long)C * C;
    WCTB_CUDA(cudaMemsetAsync(kc, 0, (size_t)Ns * 2 * 4, st));
    float* A0 = reinterpret_cast<float*>(w + L.A0);
    float* lam = reinterpret_cast<float*>(w + L.lam);
    int rc = launch_mean_cov(style, ActGeom(Ns, Hs, Ws, C), eps_cov, mean_s, G, A0, dsum, st);
    if (rc) return rc;
    int* ok = reinterpret_cast<int*>(w + L.ok);
    rc = launch_matfun_ns(A0, C, Ns, /*n_first=*/0, thresh, eps_eig, Cs, ok, kc, st);     // C_s = A^+1/2 where every eigenvalue is kept
    if (rc < 0) return rc;
    rc = launch_jacobi(G, C, Ns, conv, kc + Ns, st, ok);
    if (rc) return rc;
    rc = launch_eig_post(G, A0, lam, C, Ns, thresh, eps_eig, /*n_content=*/0, sigma, dvec, kc, st, ok);
    if (rc) return rc;
    dim3 gg((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)Ns);
    k_outer_gemm<<<gg, 256, 0, st>>>(G, CC, G, CC, dvec, C, Cs, CC, C, ok);
    WCTB_CHECK_LAUNCH("k_outer_gemm(Cs)");
    return 0;
}

int launch_wct_apply(const __half* content, int Nc, int Hc, int Wc, int C, const void* state, int Ns, float alpha,
                     float eps_cov, float eps_eig, float thresh, int readd, __half* out, int32_t* k_out, void* ws,
                     size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "wct_apply: C=%d not in {64,128,256,512}", C);
    WCTB_REQUIRE(Ns == 1 || Ns == Nc, "wct_apply: Ns must be 1 or Nc");
    const WctWs L = wct_layout(C, Nc, 0);
    if (ws_bytes < L.total) {
        set_error("wct_apply: workspace %zu < %zu bytes", ws_bytes, L.total);
        return WCTB200_EWS;
    }
    uint8_t* w = static_cast<uint8_t*>(ws);
    size_t off_cs, off_k;
    style_state_offsets(C, Ns, &off_cs, &off_k);
    const uint8_t* sp = static_cast<const uint8_t*>(state);
    const float* mean_s = reinterpret_cast<const float*>(sp);
    const float* Cs = reinterpret_cast<const float*>(sp + off_cs);
    const int* ks = reinterpret_cast<const int*>(sp + off_k);
    double* dsum = reinterpret_cast<double*>(w + L.dsum);
    float* mean = reinterpret_cast<float*>(w + L.mean);
    float* G = reinterpret_cast<float*>(w + L.G);
    float* sigma = reinterpret_cast<float*>(w + L.sigma);
    float* dvec = reinterpret_cast<float*>(w + L.dvec);
    float* Wcm = reinterpret_cast<float*>(w + L.Wc);
    float* T = reinterpret_cast<float*>(w + L.T);
    __half* Msplit = reinterpret_cast<__half*>(w + L.Msplit);
    float* bias = reinterpret_cast<float*>(w + L.bias);
    float* conv = reinterpret_cast<float*>(w + L.conv);
    int* kc = reinterpret_cast<int*>(w + L.kcount);
    const long long CC = (long long)C * C;
    WCTB_CUDA(cudaMemsetAsync(kc, 0, (size_t)Nc * 2 * 4, st));
    float* A0 = reinterpret_cast<float*>(w + L.A0);
    float* lam = reinterpret_cast<float*>(w + L.lam);
    int rc = launch_mean_cov(content, ActGeom(Nc, Hc, Wc, C), eps_cov, mean, G, A0, dsum, st);
    if (rc) return rc;
    int* ok = reinterpret_cast<int*>(w + L.ok);
    rc = launch_matfun_ns(A0, C, Nc, /*n_first=*/Nc, thresh, eps_eig, Wcm, ok, kc, st);   // W_c = A^-1/2 where every eigenvalue is kept
    if (rc < 0) return rc;
    rc = launch_jacobi(G, C, Nc, conv, kc + Nc, st, ok);
    if (rc) return rc;
    rc = launch_eig_post(G, A0, lam, C, Nc, thresh, eps_eig, Nc, sigma, dvec, kc, st, ok);
    if (rc) return rc;
    dim3 gg((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)Nc);
    k_outer_gemm<<<gg, 256, 0, st>>>(G, CC, G, CC, dvec, C, Wcm, CC, C, ok);
    WCTB_CHECK_LAUNCH("k_outer_gemm(Wc)");
    k_outer_gemm<<<gg, 256, 0, st>>>(Cs, Ns == 1 ? 0 : CC, Wcm, CC, nullptr, 0, T, CC, C);   // T = C_s W_c
    WCTB_CHECK_LAUNCH("k_outer_gemm(T)");
    dim3 gf((unsigned)cdiv(C, 8), (unsigned)Nc);
    k_finalize_transform<<<gf, 256, 0, st>>>(T, C, Nc, Ns, alpha, readd, mean, mean_s, Msplit, bias);
    WCTB_CHECK_LAUNCH("k_finalize_transform");
    rc = launch_conv_tc(CONV_APPLY, content, Nc, Hc, Wc, C, Msplit, Nc, nullptr, bias, C, 0, out, st);
    if (rc) return rc;
    if (k_out) {
        // k_out: [k_c x Nc | k_s x Ns | sweeps_c x Nc | sweeps_s x Ns]  (same order as wct_level)
        WCTB_CUDA(cudaMemcpyAsync(k_out, kc, (size_t)Nc * 4, cudaMemcpyDeviceToDevice, st));
        WCTB_CUDA(cudaMemcpyAsync(k_out + Nc, ks, (size_t)Ns * 4, cudaMemcpyDeviceToDevice, st));
        WCTB_CUDA(cudaMemcpyAsync(k_out + Nc + Ns, kc + Nc, (size_t)Nc * 4, cudaMemcpyDeviceToDevice, st));
        WCTB_CUDA(cudaMemcpyAsync(k_out + 2 * Nc + Ns, ks + Ns, (size_t)Ns * 4, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

// test / profiling hook: means and covariance of a feature batch (stage A of the transform)
int launch_covariance(const __half* act, int N, int H, int W, int C, float eps_cov, float* mean_out, float* cov_out,
                      cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || (C % 128 == 0 && C >= 128), "covariance: C=%d must be 64 or a multiple of 128", C);
    double* dsum = nullptr;
    { int rc0 = scratch_alloc(reinterpret_cast<void**>(&dsum), (size_t)N * C * sizeof(double), st, 1); if (rc0) return rc0; }
    return launch_mean_cov(act, ActGeom(N, H, W, C), eps_cov, mean_out, cov_out, nullptr, dsum, st);
}

int launch_adain_level(const __half* content, int Nc, int Hc, int Wc, const __half* style, int Ns, int Hs, int Ws, int C,
                       float alpha, float eps, __half* out, void* ws, size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C % 8 == 0 && C <= 2048, "adain_level: C=%d must be a multiple of 8 (<= 2048)", C);
    WCTB_REQUIRE(Ns == 1 || Ns == Nc, "adain_level: Ns must be 1 or Nc");
    const WctWs L = wct_layout(C, Nc, Ns);
    if (ws_bytes < L.total) {
        set_error("adain_level: workspace %zu < %zu bytes", ws_bytes, L.total);
        return WCTB200_EWS;
    }
    uint8_t* w = static_cast<uint8_t*>(ws);
    double* sum = reinterpret_cast<double*>(w + L.sum);
    double* sumsq = reinterpret_cast<double*>(w + L.sumsq);
    float* mean = reinterpret_cast<float*>(w + L.mean);
    float* var = reinterpret_cast<float*>(w + L.var);
    float* scale = reinterpret_cast<float*>(w + L.scale);
    float* shift = reinterpret_cast<float*>(w + L.shift);
    WCTB_CUDA(cudaMemsetAsync(w + L.sum, 0, L.dsum - L.sum, st));
    ActGeom gc(Nc, Hc, Wc, C), gs(Ns, Hs, Ws, C);
    int rc = launch_sums<true>(content, gc, sum, sumsq, st);
    if (rc) return rc;
    rc = launch_sums<true>(style, gs, sum + (long long)Nc * C, sumsq + (long long)Nc * C, st);
    if (rc) return rc;
    k_mean_finalize<<<cdiv((long long)Nc * C, 256), 256, 0, st>>>(sum, sumsq, (long long)Hc * Wc, Nc * C, mean, var);
    WCTB_CHECK_LAUNCH("k_mean_finalize(c)");
    k_mean_finalize<<<cdiv((long long)Ns * C, 256), 256, 0, st>>>(sum + (long long)Nc * C, sumsq + (long long)Nc * C,
                                                                  (long long)Hs * Ws, Ns * C, mean + (long long)Nc * C,
                                                                  var + (long long)Nc * C);
    WCTB_CHECK_LAUNCH("k_mean_finalize(s)");
    k_adain_coeffs<<<cdiv((long long)Nc * C, 256), 256, 0, st>>>(mean, var, mean + (long long)Nc * C, var + (long long)Nc * C, C,
                                                                 Nc, Ns, alpha, eps, scale, shift);
    WCTB_CHECK_LAUNCH("k_adain_coeffs");
    const long long total = (long long)Nc * Hc * Wc * (C / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > device_sm_count() * 16) blocks = device_sm_count() * 16;
    k_affine_apply<<<(unsigned)blocks, 256, 0, st>>>(content, gc, scale, shift, out);
    WCTB_CHECK_LAUNCH("k_affine_apply");
    return 0;
}

// ---------------------------------------------------------------------------
// Style swap at one level (ops.py:145-278: wct_style_swap + style_swap), ONE content/style pair, 3x3 patches, stride 1.
//   whiten content and style (same eigensolver as the WCT level; whitening on BOTH sides, ops.py:187-196)
//   -> every 3x3 patch of the whitened style becomes a conv filter, normalised per filter TAP across patches
//      (tf.nn.l2_normalize(style_patches, dim=3), ops.py:233) -> cross-correlation with the whitened content on the
//      tensor cores (the patches are just a weight tensor for the 3x3 conv kernel; VALID = the interior of the SAME conv)
//   -> first arg-max per position (ops.py:242) -> paste the un-normalised patch back and average the overlaps
//      (conv2d_transpose / counting, ops.py:255-276 = a gather of <= 9 style pixels per output pixel)
//   -> colour with the style (S^+1/2), add the style mean, blend with the content (ops.py:203-210).
// ---------------------------------------------------------------------------
static inline int swap_grid(long long total, int block) {
    long long b = (total + block - 1) / block;
    return (int)(b < 1 ? 1 : (b > device_sm_count() * 32ll ? device_sm_count() * 32ll : b));
}

struct SwapWs {
    size_t base, zeros, dvec2, sigma2, mats, msplit, bias3, norms, idx, wc_feat, ws_feat, ss_feat, tmp, scores, wsplit, total;
    int cout_pad, n_patches, prow, pcol, ho, wo;   // style patch grid prow x pcol, content score grid ho x wo
};
static SwapWs swap_layout(int C, int Hc, int Wc, int Hs, int Ws, int P, int S) {
    SwapWs L;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    L.prow = (Hs - P) / S + 1;                                    // tf.extract_image_patches, VALID (ops.py:226)
    L.pcol = (Ws - P) / S + 1;
    L.ho = (Hc - P) / S + 1;                                      // tf.nn.conv2d VALID with the same stride (ops.py:236-239)
    L.wo = (Wc - P) / S + 1;
    L.n_patches = L.prow * L.pcol;
    L.cout_pad = (L.n_patches + 63) / 64 * 64;
    L.base = take(wct_layout(C, 1, 1).total);
    L.zeros = take((size_t)C * 4);
    L.dvec2 = take((size_t)C * 4);
    L.sigma2 = take((size_t)C * 4);
    L.mats = take((size_t)3 * C * C * 4);                         // W_c, W_s (whitening), C_s (colouring)
    L.msplit = take((size_t)3 * 2 * C * C * 2);
    L.bias3 = take((size_t)3 * C * 4);
    L.norms = take((size_t)P * P * C * 4);
    L.idx = take((size_t)L.ho * L.wo * 4);
    const size_t fc = (size_t)ActGeom(1, Hc, Wc, C).plane * 2 * sizeof(__half), fs = (size_t)ActGeom(1, Hs, Ws, C).plane * 2 * sizeof(__half);
    L.wc_feat = take(fc);
    L.ws_feat = take(fs);
    L.ss_feat = take(fc);
    L.tmp = take(fc);
    L.scores = take((size_t)ActGeom(1, Hc, Wc, L.cout_pad).plane * 2 * sizeof(__half));
    L.wsplit = take((size_t)2 * P * P * C * L.cout_pad * sizeof(__half));
    L.total = o;
    return L;
}
size_t style_swap_workspace_bytes(int C, int Hc, int Wc, int Hs, int Ws, int P, int S) { return swap_layout(C, Hc, Wc, Hs, Ws, P, S).total; }

// patch geometry of the swap: P x P patches taken every S pixels (ops.py:219-278: --ss-patch-size, --ss-stride)
struct SwapGeom { int P, S, prow, pcol, ho, wo; };

// 1 / ||patch tap||: for every (tap, channel) the l2 norm ACROSS all patches (ops.py:233); block = (tap, 256 channels)
__global__ void k_swap_tap_norms(const __half* __restrict__ feat, ActGeom g, SwapGeom q, float* __restrict__ inv_norm) {
    const int tap = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= g.C) return;
    const int ky = tap / q.P, kx = tap % q.P;
    float s = 0.f;
    for (int py = 0; py < q.prow; ++py)
        for (int px = 0; px < q.pcol; ++px) {
            const long long pos = ((long long)(py * q.S + ky + 1)) * g.Wp + (px * q.S + kx + 1);      // interior pixel -> padded position
            const float v = merge_f32(feat[pos * g.C + c], feat[g.plane + pos * g.C + c]);
            s = fmaf(v, v, s);
        }
    inv_norm[tap * g.C + c] = rsqrtf(fmaxf(s, 1e-12f));
}
// conv weights of the correlation: [plane][patch n][tap*C + c] = whitened_style[py*S+ky][px*S+kx][c] * inv_norm[tap][c]; rows >= n_patches zero
__global__ void k_swap_patch_weights(const __half* __restrict__ feat, ActGeom g, SwapGeom q, const float* __restrict__ inv_norm,
                                     int n_patches, int cout_pad, __half* __restrict__ wsplit) {
    const long long K = (long long)q.P * q.P * g.C, total = K * cout_pad;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i / K);
        const int k = (int)(i - (long long)n * K);
        float v = 0.f;
        if (n < n_patches) {
            const int tap = k / g.C, c = k - tap * g.C;
            const int py = n / q.pcol, px = n - py * q.pcol;
            const long long pos = ((long long)(py * q.S + tap / q.P + 1)) * g.Wp + (px * q.S + tap % q.P + 1);
            v = merge_f32(feat[pos * g.C + c], feat[g.plane + pos * g.C + c]) * inv_norm[k];
        }
        __half hi, lo;
        split_f32(v, hi, lo);
        wsplit[i] = hi;
        wsplit[total + i] = lo;
    }
}
// first arg-max over the patch axis for every VALID strided position (y,x): the top-left-anchored P x P correlation
// at interior pixel (y*S, x*S), which the conv kernel stored at that pixel's own padded cell
__global__ void k_swap_argmax(const __half* __restrict__ scores, ActGeom g, SwapGeom q, int n_patches, int* __restrict__ idx) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= q.ho * q.wo) return;
    const int y = warp / q.wo, x = warp - y * q.wo;
    const long long pos = ((long long)(y * q.S + 1)) * g.Wp + (x * q.S + 1);
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int n = lane; n < n_patches; n += 32) {
        const float v = merge_f32(scores[pos * g.C + n], scores[g.plane + pos * g.C + n]);
        if (v > best) { best = v; bi = n; }                       // strictly greater: keeps the first maximum of this lane
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (lane == 0) idx[warp] = bi;
}
// conv2d_transpose of the one-hot map with the raw patches, divided by the overlap count (ops.py:255-276): output pixel
// (Y,X) averages, over the <= P*P patch positions (py,px) with py*S + dy = Y, px*S + dx = X that cover it, the style
// pixel (sy*S + dy, sx*S + dx) of the matched patch.  The caller guarantees (ho-1)*S + P == H (wct.py:84-90 refits).
__global__ void k_swap_gather(const __half* __restrict__ sfeat, ActGeom gs, SwapGeom q, const int* __restrict__ idx, ActGeom gc,
                              __half* __restrict__ out) {
    const int cg = gc.C / 8;
    const long long total = (long long)gc.H * gc.W * cg;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c0 = (int)(i % cg) * 8;
        const int pix = (int)(i / cg);
        const int Y = pix / gc.W, X = pix - Y * gc.W;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        int cnt = 0;
        for (int dy = 0; dy < q.P; ++dy) {
            const int ty = Y - dy;
            if (ty < 0 || ty % q.S != 0 || ty / q.S >= q.ho) continue;
            for (int dx = 0; dx < q.P; ++dx) {
                const int tx = X - dx;
                if (tx < 0 || tx % q.S != 0 || tx / q.S >= q.wo) continue;
                const int n = idx[(ty / q.S) * q.wo + tx / q.S];
                const int sy = n / q.pcol, sx = n - sy * q.pcol;
                float v[8];
                load8(sfeat, gs, ((long long)(sy * q.S + dy + 1)) * gs.Wp + (sx * q.S + dx + 1), c0, v);
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[j] += v[j];
                ++cnt;
            }
        }
        const float inv = cnt > 0 ? 1.f / (float)cnt : 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] *= inv;
        Half8 hi, lo;
        split8(acc, hi, lo);
        store8_with_halo(out, gc, 0, Y, X, c0, hi, lo);
    }
}
// out = a*x + b*y on SPF16 interiors (+ halos)
__global__ void k_blend2(const __half* __restrict__ x, const __half* __restrict__ y, ActGeom g, float a, float b,
                         __half* __restrict__ out) {
    const int cg = g.C / 8;
    const long long total = (long long)g.N * g.H * g.W * cg;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c0 = (int)(i % cg) * 8;
        long long pix = i / cg;
        const int X = (int)(pix % g.W); pix /= g.W;
        const int Y = (int)(pix % g.H);
        const int n = (int)(pix / g.H);
        const long long pos = ((long long)n * g.Hp + Y + 1) * g.Wp + X + 1;
        float u[8], v[8];
        load8(x, g, pos, c0, u);
        load8(y, g, pos, c0, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) u[j] = fmaf(a, u[j], b * v[j]);
        Half8 hi, lo;
        split8(u, hi, lo);
        store8_with_halo(out, g, n, Y, X, c0, hi, lo);
    }
}

int launch_style_swap_level(const __half* content, int Hc, int Wc, const __half* style, int Hs, int Ws, int C, int patch, int stride,
                            float alpha, float eps_cov, float thresh, __half* out, int32_t* k_out, void* ws, size_t ws_bytes,
                            cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "style_swap: C=%d not in {64,128,256,512}", C);
    WCTB_REQUIRE(patch >= 1 && patch <= 16 && stride >= 1 && stride <= 16, "style_swap: patch %d / stride %d out of range", patch, stride);
    WCTB_REQUIRE(Hc >= patch && Wc >= patch && Hs >= patch && Ws >= patch && Hc >= 2 && Wc >= 2 && Hs >= 2 && Ws >= 2,
                 "style_swap: maps must be at least %dx%d (content %dx%d, style %dx%d)", patch, patch, Hc, Wc, Hs, Ws);
    const SwapWs S = swap_layout(C, Hc, Wc, Hs, Ws, patch, stride);
    // the swapped encoding must have the content's size (ops.py:199 reshapes it to [Hc*Wc, C]); wct.py:84-90 crops the content
    // image beforehand when the stride makes the filter not fit (utils.swap_filter_fit)
    WCTB_REQUIRE((S.ho - 1) * stride + patch == Hc && (S.wo - 1) * stride + patch == Wc,
                 "style_swap: patch %d / stride %d does not tile a %dx%d encoding (refit the content: swap_filter_fit, wct.py:84-90)",
                 patch, stride, Hc, Wc);
    const SwapGeom q = {patch, stride, S.prow, S.pcol, S.ho, S.wo};
    if (ws_bytes < S.total) {
        set_error("style_swap: workspace %zu < %zu bytes", ws_bytes, S.total);
        return WCTB200_EWS;
    }
    uint8_t* sw = static_cast<uint8_t*>(ws);
    const WctWs L = wct_layout(C, 1, 1);
    uint8_t* w = sw + S.base;
    double* dsum = reinterpret_cast<double*>(w + L.dsum);
    float* mean = reinterpret_cast<float*>(w + L.mean);          // [mc, ms]
    float* G = reinterpret_cast<float*>(w + L.G);
    float* A0 = reinterpret_cast<float*>(w + L.A0);
    float* lam = reinterpret_cast<float*>(w + L.lam);
    float* sigma = reinterpret_cast<float*>(w + L.sigma);
    float* dvec = reinterpret_cast<float*>(w + L.dvec);          // whitening scalings of content and style
    float* conv = reinterpret_cast<float*>(w + L.conv);
    int* kc = reinterpret_cast<int*>(w + L.kcount);
    float* zeros = reinterpret_cast<float*>(sw + S.zeros);
    float* dvec2 = reinterpret_cast<float*>(sw + S.dvec2);       // colouring scaling of the style
    float* sigma2 = reinterpret_cast<float*>(sw + S.sigma2);
    float* mats = reinterpret_cast<float*>(sw + S.mats);
    __half* msplit = reinterpret_cast<__half*>(sw + S.msplit);
    float* bias3 = reinterpret_cast<float*>(sw + S.bias3);
    float* norms = reinterpret_cast<float*>(sw + S.norms);
    int* idx = reinterpret_cast<int*>(sw + S.idx);
    __half* wc_feat = reinterpret_cast<__half*>(sw + S.wc_feat);
    __half* ws_feat = reinterpret_cast<__half*>(sw + S.ws_feat);
    __half* ss_feat = reinterpret_cast<__half*>(sw + S.ss_feat);
    __half* tmp = reinterpret_cast<__half*>(sw + S.tmp);
    __half* scores = reinterpret_cast<__half*>(sw + S.scores);
    __half* wsplit = reinterpret_cast<__half*>(sw + S.wsplit);
    const long long CC = (long long)C * C;

    WCTB_CUDA(cudaMemsetAsync(kc, 0, 4 * 4, st));
    WCTB_CUDA(cudaMemsetAsync(zeros, 0, (size_t)C * 4, st));
    ActGeom gc(1, Hc, Wc, C), gs(1, Hs, Ws, C);
    int rc = launch_mean_cov(content, gc, eps_cov, mean, G, A0, dsum, st);
    if (rc) return rc;
    rc = launch_mean_cov(style, gs, eps_cov, mean + C, G + CC, A0 + CC, dsum + C, st);
    if (rc) return rc;
    rc = launch_jacobi(G, C, 2, conv, kc + 2, st, nullptr);
    if (rc) return rc;
    rc = launch_eig_post(G, A0, lam, C, 2, thresh, 0.f, 2, sigma, dvec, kc, st);          // S^-1/2 for BOTH (ops.py:187,193)
    if (rc) return rc;
    k_eig_post<<<dim3((unsigned)cdiv(C, 8), 1), 256, 0, st>>>(G + CC, lam + C, C, thresh, 0.f, 0, sigma2, dvec2, nullptr, nullptr);   // S^+1/2 (ops.py:203)
    WCTB_CHECK_LAUNCH("k_eig_post(colour)");
    dim3 g2((unsigned)(C / 64), (unsigned)(C / 64), 2), g1((unsigned)(C / 64), (unsigned)(C / 64), 1);
    k_outer_gemm<<<g2, 256, 0, st>>>(G, CC, G, CC, dvec, C, mats, CC, C);                   // W_c, W_s
    WCTB_CHECK_LAUNCH("k_outer_gemm(whiten)");
    k_outer_gemm<<<g1, 256, 0, st>>>(G + CC, CC, G + CC, CC, dvec2, C, mats + 2 * CC, CC, C);   // C_s
    WCTB_CHECK_LAUNCH("k_outer_gemm(colour)");
    // operand 0/1: x -> W (x - m)   (alpha = 1, "style mean" = 0);  operand 2: x -> C_s x + m_s  ("content mean" = 0)
    k_finalize_transform<<<dim3((unsigned)cdiv(C, 8), 2), 256, 0, st>>>(mats, C, 2, 1, 1.f, 0, mean, zeros, msplit, bias3);
    WCTB_CHECK_LAUNCH("k_finalize_transform(whiten)");
    k_finalize_transform<<<dim3((unsigned)cdiv(C, 8), 1), 256, 0, st>>>(mats + 2 * CC, C, 1, 1, 1.f, 0, zeros, mean + C, msplit + 4 * CC,
                                                                         bias3 + 2 * C);
    WCTB_CHECK_LAUNCH("k_finalize_transform(colour)");
    rc = launch_conv_tc(CONV_APPLY, content, 1, Hc, Wc, C, msplit, 1, nullptr, bias3, C, 0, wc_feat, st);
    if (rc) return rc;
    rc = launch_conv_tc(CONV_APPLY, style, 1, Hs, Ws, C, msplit + 2 * CC, 1, nullptr, bias3 + C, C, 0, ws_feat, st);
    if (rc) return rc;
    k_swap_tap_norms<<<dim3((unsigned)cdiv(C, 256), (unsigned)(patch * patch)), 256, 0, st>>>(ws_feat, gs, q, norms);
    WCTB_CHECK_LAUNCH("k_swap_tap_norms");
    k_swap_patch_weights<<<swap_grid((long long)patch * patch * C * S.cout_pad, 256), 256, 0, st>>>(ws_feat, gs, q, norms, S.n_patches,
                                                                                                  S.cout_pad, wsplit);
    WCTB_CHECK_LAUNCH("k_swap_patch_weights");
    // every style patch is a filter: the P x P correlation (top-left anchored, all positions; the strided VALID subset is
    // read by the arg-max) runs on the tensor-core conv kernel
    rc = launch_conv_tc(CONV_TAPS, wc_feat, 1, Hc, Wc, C, wsplit, 1, nullptr, nullptr, S.cout_pad, 0, scores, st, patch);
    if (rc) return rc;
    const int npos = S.ho * S.wo;
    k_swap_argmax<<<(unsigned)cdiv((long long)npos * 32, 256), 256, 0, st>>>(scores, ActGeom(1, Hc, Wc, S.cout_pad), q, S.n_patches, idx);
    WCTB_CHECK_LAUNCH("k_swap_argmax");
    k_swap_gather<<<swap_grid((long long)Hc * Wc * (C / 8), 256), 256, 0, st>>>(ws_feat, gs, q, idx, gc, ss_feat);
    WCTB_CHECK_LAUNCH("k_swap_gather");
    rc = launch_conv_tc(CONV_APPLY, ss_feat, 1, Hc, Wc, C, msplit + 4 * CC, 1, nullptr, bias3 + 2 * C, C, 0, tmp, st);
    if (rc) return rc;
    k_blend2<<<swap_grid((long long)Hc * Wc * (C / 8), 256), 256, 0, st>>>(tmp, content, gc, alpha, 1.f - alpha, out);   // ops.py:210
    WCTB_CHECK_LAUNCH("k_blend2");
    if (k_out) WCTB_CUDA(cudaMemcpyAsync(k_out, kc, 2 * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

// ---------------------------------------------------------------------------
// Spatial control (Li et al. 2017, sec. 4): a uint8 label map splits every frame into regions; region r < R is whitened
// with its OWN statistics and coloured with style r, labels >= R ("keep") and regions of < 2 pixels leave the level equal
// by value to its input.  Item i = frame * R + region runs through the unchanged content chain of launch_wct_apply
// (means / covariance over the region's pixels, A^-1/2, W_c, T = C_s[r] W_c[i], M, bias); the tcgen05 apply multiplies
// (tile, region) pairs and stores only the region's pixels; k_copy_keep writes the rest.
// ---------------------------------------------------------------------------

// nearest-neighbour label resize in exact integer arithmetic: dst[n][y][x] = src[n][(y*Hs) div Hd][(x*Ws) div Wd]
__global__ void k_labels_nearest(const uint8_t* __restrict__ src, int N, int Hs, int Ws, int Hd, int Wd, uint8_t* __restrict__ dst) {
    const long long total = (long long)N * Hd * Wd;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % Wd);
        const long long r = i / Wd;
        const int y = (int)(r % Hd);
        const long long n = r / Hd;
        const int sy = (int)(((long long)y * Hs) / Hd), sx = (int)(((long long)x * Ws) / Wd);
        dst[i] = src[(n * Hs + sy) * Ws + sx];
    }
}
int launch_labels_nearest(const uint8_t* src, int N, int Hs, int Ws, int Hd, int Wd, uint8_t* dst, cudaStream_t st) {
    const long long total = (long long)N * Hd * Wd;
    long long blocks = (total + 255) / 256;
    if (blocks > device_sm_count() * 16ll) blocks = device_sm_count() * 16ll;
    k_labels_nearest<<<(unsigned)blocks, 256, 0, st>>>(src, N, Hs, Ws, Hd, Wd, dst);
    WCTB_CHECK_LAUNCH("k_labels_nearest");
    return 0;
}

// counts[n*R + r] = pixels of frame n labelled r (integer sums in a fixed order: deterministic).  grid N, 256 threads.
__global__ void __launch_bounds__(256) k_region_counts(const uint8_t* __restrict__ labels, long long HW, int R, int* __restrict__ counts) {
    __shared__ int red[8][256];
    const int n = blockIdx.x;
    int c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint8_t* lab = labels + (long long)n * HW;
    for (long long q = threadIdx.x; q < HW; q += 256) {
        const int l = lab[q];
#pragma unroll
        for (int r = 0; r < 8; ++r) c[r] += (l == r) ? 1 : 0;
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) red[r][threadIdx.x] = c[r];
    __syncthreads();
    if (threadIdx.x < R) {
        int a = 0;
        for (int t = 0; t < 256; ++t) a += red[threadIdx.x][t];
        counts[n * R + threadIdx.x] = a;
    }
}

// tilemask[n][t] bit r: the 128 padded positions [t*128, t*128+128) of frame n's plane hold an interior pixel of region r
// with >= 2 pixels (those are transformed by the apply; everything else is copied).  One warp per tile.
__global__ void k_tile_mask(const uint8_t* __restrict__ labels, ActGeom g, int R, const int* __restrict__ counts, int tiles_per_image,
                            uint32_t* __restrict__ tilemask) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= g.N * tiles_per_image) return;
    const int n = warp / tiles_per_image, t = warp - n * tiles_per_image;
    const int HpWp = g.Hp * g.Wp;
    uint32_t bits = 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int pos = t * 128 + k * 32 + lane;
        if (pos >= HpWp) continue;
        const int yy = pos / g.Wp, xx = pos - yy * g.Wp;
        if (yy < 1 || yy > g.H || xx < 1 || xx > g.W) continue;
        const int l = labels[((long long)n * g.H + yy - 1) * g.W + xx - 1];
        if (l < R && counts[n * R + l] >= 2) bits |= 1u << l;
    }
    bits = __reduce_or_sync(0xffffffffu, bits);
    if (lane == 0) tilemask[warp] = bits;
}

// pixels the transform leaves alone (label >= R, or a region of < 2 pixels): copy both fp16 planes (+ the halo cells that
// mirror them) -- equal by value to the input
__global__ void k_copy_keep(const __half* __restrict__ in, ActGeom g, const uint8_t* __restrict__ labels, int R,
                            const int* __restrict__ counts, __half* __restrict__ out) {
    const int cgs = g.C / 8;
    const long long total = (long long)g.N * g.H * g.W * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pix = i / cgs;
        const int c0 = (int)(i - pix * cgs) * 8;
        const int l = labels[pix];
        const int x = (int)(pix % g.W);
        const long long r = pix / g.W;
        const int y = (int)(r % g.H);
        const int n = (int)(r / g.H);
        if (l < R && counts[n * R + l] >= 2) continue;
        const long long off = (((long long)n * g.Hp + y + 1) * g.Wp + x + 1) * g.C + c0;
        const Half8 hi = *reinterpret_cast<const Half8*>(in + off);
        const Half8 lo = *reinterpret_cast<const Half8*>(in + g.plane + off);
        store8_with_halo(out, g, n, y, x, c0, hi, lo);
    }
}

// AdaIN per region: item n*R + label's affine map; keep pixels copied
__global__ void k_affine_apply_regions(const __half* __restrict__ in, ActGeom g, const uint8_t* __restrict__ labels, int R,
                                       const int* __restrict__ counts, const float* __restrict__ scale, const float* __restrict__ shift,
                                       __half* __restrict__ out) {
    const int cgs = g.C / 8;
    const long long total = (long long)g.N * g.H * g.W * cgs;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pix = i / cgs;
        const int c0 = (int)(i - pix * cgs) * 8;
        const int l = labels[pix];
        const int x = (int)(pix % g.W);
        const long long r = pix / g.W;
        const int y = (int)(r % g.H);
        const int n = (int)(r / g.H);
        const long long off = (((long long)n * g.Hp + y + 1) * g.Wp + x + 1) * g.C + c0;
        Half8 hi = *reinterpret_cast<const Half8*>(in + off);
        Half8 lo = *reinterpret_cast<const Half8*>(in + g.plane + off);
        if (l < R && counts[n * R + l] >= 2) {
            float v[8];
            merge8(hi, lo, v);
            const float* sc = scale + ((long long)n * R + l) * g.C + c0;
            const float* sh = shift + ((long long)n * R + l) * g.C + c0;
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
            split8(v, hi, lo);
        }
        store8_with_halo(out, g, n, y, x, c0, hi, lo);
    }
}

// workspace: the content chain of Nc*R items (wct_layout(C, Nc*R, 0)) | style means [R][C] | pixel counts [Nc*R] |
// AdaIN style sums [2][R][C] fp64 and style mean / variance [2][R][C]
struct RegionWs {
    WctWs base;
    size_t ms, counts, ssum, smv, total;
};
static RegionWs regions_layout(int C, int Nc, int R) {
    RegionWs L;
    L.base = wct_layout(C, Nc * R, 0);
    size_t o = L.base.total;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    L.ms = take((size_t)R * C * 4);
    L.counts = take((size_t)Nc * R * 4);
    L.ssum = take((size_t)2 * R * C * 8);
    L.smv = take((size_t)2 * R * C * 4);
    L.total = o;
    return L;
}
size_t wct_regions_workspace_bytes(int C, int Nc, int R) { return regions_layout(C, Nc, R).total; }

static int launch_region_counts(const uint8_t* labels, int Nc, int Hc, int Wc, int R, int* counts, cudaStream_t st) {
    k_region_counts<<<(unsigned)Nc, 256, 0, st>>>(labels, (long long)Hc * Wc, R, counts);
    WCTB_CHECK_LAUNCH("k_region_counts");
    return 0;
}

static int launch_copy_keep(const __half* content, ActGeom gc, const uint8_t* labels, int R, const int* counts, __half* out,
                            cudaStream_t st) {
    const long long total = (long long)gc.N * gc.H * gc.W * (gc.C / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > device_sm_count() * 16ll) blocks = device_sm_count() * 16ll;
    k_copy_keep<<<(unsigned)blocks, 256, 0, st>>>(content, gc, labels, R, counts, out);
    WCTB_CHECK_LAUNCH("k_copy_keep");
    return 0;
}

int launch_wct_apply_regions(const __half* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                             const void* const* states, float alpha, float eps_cov, float eps_eig, float thresh, int readd,
                             __half* out, int32_t* k_out, void* ws, size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "wct_apply_regions: C=%d not in {64,128,256,512}", C);
    WCTB_REQUIRE(R >= 1 && R <= 8, "wct_apply_regions: R=%d not in 1..8", R);
    for (int r = 0; r < R; ++r) WCTB_REQUIRE(states[r] != nullptr, "wct_apply_regions: style state %d is NULL", r);
    const RegionWs RL = regions_layout(C, Nc, R);
    if (ws_bytes < RL.total) {
        set_error("wct_apply_regions: workspace %zu < %zu bytes", ws_bytes, RL.total);
        return WCTB200_EWS;
    }
    const WctWs& L = RL.base;
    const int NR = Nc * R;
    uint8_t* w = static_cast<uint8_t*>(ws);
    size_t off_cs, off_k;
    style_state_offsets(C, 1, &off_cs, &off_k);
    double* dsum = reinterpret_cast<double*>(w + L.dsum);
    float* mean = reinterpret_cast<float*>(w + L.mean);
    float* G = reinterpret_cast<float*>(w + L.G);
    float* A0 = reinterpret_cast<float*>(w + L.A0);
    float* lam = reinterpret_cast<float*>(w + L.lam);
    float* sigma = reinterpret_cast<float*>(w + L.sigma);
    float* dvec = reinterpret_cast<float*>(w + L.dvec);
    float* Wcm = reinterpret_cast<float*>(w + L.Wc);
    float* T = reinterpret_cast<float*>(w + L.T);
    __half* Msplit = reinterpret_cast<__half*>(w + L.Msplit);
    float* bias = reinterpret_cast<float*>(w + L.bias);
    float* conv = reinterpret_cast<float*>(w + L.conv);
    int* kc = reinterpret_cast<int*>(w + L.kcount);
    int* ok = reinterpret_cast<int*>(w + L.ok);
    float* ms_all = reinterpret_cast<float*>(w + RL.ms);
    int* counts = reinterpret_cast<int*>(w + RL.counts);
    const long long CC = (long long)C * C;
    const ActGeom gc(Nc, Hc, Wc, C);
    const int tpi = cdiv((long long)gc.Hp * gc.Wp, 128);
    uint32_t* tilemask = nullptr;
    { int rc0 = scratch_alloc(reinterpret_cast<void**>(&tilemask), (size_t)Nc * tpi * 4, st, 3); if (rc0) return rc0; }

    WCTB_CUDA(cudaMemsetAsync(kc, 0, (size_t)NR * 2 * 4, st));
    int rc = launch_region_counts(labels, Nc, Hc, Wc, R, counts, st);
    if (rc) return rc;
    rc = launch_mean_cov(content, gc, eps_cov, mean, G, A0, dsum, st, labels, R, counts);
    if (rc) return rc;
    rc = launch_matfun_ns(A0, C, NR, /*n_first=*/NR, thresh, eps_eig, Wcm, ok, kc, st);   // W_c = A^-1/2 where every eigenvalue is kept
    if (rc < 0) return rc;
    rc = launch_jacobi(G, C, NR, conv, kc + NR, st, ok);
    if (rc) return rc;
    rc = launch_eig_post(G, A0, lam, C, NR, thresh, eps_eig, NR, sigma, dvec, kc, st, ok);
    if (rc) return rc;
    dim3 gg((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)NR);
    k_outer_gemm<<<gg, 256, 0, st>>>(G, CC, G, CC, dvec, C, Wcm, CC, C, ok);
    WCTB_CHECK_LAUNCH("k_outer_gemm(Wc)");
    // T[n*R + r] = C_s[r] W_c[n*R + r]: one launch per region (strides R*C*C over the frames)
    dim3 gt((unsigned)(C / 64), (unsigned)(C / 64), (unsigned)Nc);
    for (int r = 0; r < R; ++r) {
        const uint8_t* sp = static_cast<const uint8_t*>(states[r]);
        WCTB_CUDA(cudaMemcpyAsync(ms_all + (long long)r * C, sp, (size_t)C * 4, cudaMemcpyDeviceToDevice, st));
        k_outer_gemm<<<gt, 256, 0, st>>>(reinterpret_cast<const float*>(sp + off_cs), 0, Wcm + r * CC, R * CC, nullptr, 0,
                                         T + r * CC, R * CC, C);
        WCTB_CHECK_LAUNCH("k_outer_gemm(T)");
    }
    dim3 gf((unsigned)cdiv(C, 8), (unsigned)NR);
    k_finalize_transform<<<gf, 256, 0, st>>>(T, C, NR, R, alpha, readd, mean, ms_all, Msplit, bias);
    WCTB_CHECK_LAUNCH("k_finalize_transform");
    k_tile_mask<<<(unsigned)cdiv((long long)Nc * tpi * 32, 256), 256, 0, st>>>(labels, gc, R, counts, tpi, tilemask);
    WCTB_CHECK_LAUNCH("k_tile_mask");
    rc = launch_conv_tc(CONV_APPLY, content, Nc, Hc, Wc, C, Msplit, NR, nullptr, bias, C, 0, out, st, 3, labels, R, tilemask);
    if (rc) return rc;
    rc = launch_copy_keep(content, gc, labels, R, counts, out, st);
    if (rc) return rc;
    if (k_out) {
        // k_out: [k_c x Nc*R | n_r x Nc*R], frame-major
        WCTB_CUDA(cudaMemcpyAsync(k_out, kc, (size_t)NR * 4, cudaMemcpyDeviceToDevice, st));
        WCTB_CUDA(cudaMemcpyAsync(k_out + NR, counts, (size_t)NR * 4, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

int launch_adain_regions(const __half* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                         const __half* const* styles, const int* style_hw, float alpha, float eps, __half* out, void* ws,
                         size_t ws_bytes, cudaStream_t st) {
    WCTB_REQUIRE(C % 8 == 0 && C <= 2048, "adain_regions: C=%d must be a multiple of 8 (<= 2048)", C);
    WCTB_REQUIRE(R >= 1 && R <= 8, "adain_regions: R=%d not in 1..8", R);
    for (int r = 0; r < R; ++r)
        WCTB_REQUIRE(styles[r] != nullptr && style_hw[2 * r] >= 2 && style_hw[2 * r + 1] >= 2, "adain_regions: bad style %d", r);
    const RegionWs RL = regions_layout(C, Nc, R);
    if (ws_bytes < RL.total) {
        set_error("adain_regions: workspace %zu < %zu bytes", ws_bytes, RL.total);
        return WCTB200_EWS;
    }
    const WctWs& L = RL.base;
    const int NR = Nc * R;
    uint8_t* w = static_cast<uint8_t*>(ws);
    double* sum = reinterpret_cast<double*>(w + L.sum);
    double* sumsq = reinterpret_cast<double*>(w + L.sumsq);
    float* mean = reinterpret_cast<float*>(w + L.mean);
    float* var = reinterpret_cast<float*>(w + L.var);
    float* scale = reinterpret_cast<float*>(w + L.scale);
    float* shift = reinterpret_cast<float*>(w + L.shift);
    int* counts = reinterpret_cast<int*>(w + RL.counts);
    double* ssum = reinterpret_cast<double*>(w + RL.ssum);
    float* smean = reinterpret_cast<float*>(w + RL.smv);
    float* svar = smean + (long long)R * C;
    WCTB_CUDA(cudaMemsetAsync(w + L.sum, 0, L.dsum - L.sum, st));
    WCTB_CUDA(cudaMemsetAsync(ssum, 0, (size_t)2 * R * C * 8, st));
    int rc = launch_region_counts(labels, Nc, Hc, Wc, R, counts, st);
    if (rc) return rc;
    const ActGeom gc(Nc, Hc, Wc, C);
    {
        // the chunking of launch_sums, one grid layer per region
        const long long HW = (long long)Hc * Wc;
        long long chunk = (HW * Nc + 591) / 592;
        const int rows = 256 / (C / 8) > 0 ? 256 / (C / 8) : 1;
        chunk = (chunk + rows - 1) / rows * rows;
        if (chunk < rows) chunk = rows;
        if (chunk > 1024) chunk = 1024;
        dim3 grid((unsigned)cdiv(HW, chunk), (unsigned)Nc, (unsigned)R);
        k_chan_sums<true><<<grid, 256, 0, st>>>(content, gc, (int)chunk, sum, sumsq, labels);
        WCTB_CHECK_LAUNCH("k_chan_sums(regions)");
    }
    for (int r = 0; r < R; ++r) {
        const ActGeom gs(1, style_hw[2 * r], style_hw[2 * r + 1], C);
        rc = launch_sums<true>(styles[r], gs, ssum + (long long)r * C, ssum + (long long)(R + r) * C, st);
        if (rc) return rc;
        k_mean_finalize<<<cdiv(C, 256), 256, 0, st>>>(ssum + (long long)r * C, ssum + (long long)(R + r) * C, (long long)gs.H * gs.W,
                                                       C, smean + (long long)r * C, svar + (long long)r * C);
        WCTB_CHECK_LAUNCH("k_mean_finalize(s)");
    }
    k_mean_finalize<<<cdiv((long long)NR * C, 256), 256, 0, st>>>(sum, sumsq, 1, NR * C, mean, var, counts, C);
    WCTB_CHECK_LAUNCH("k_mean_finalize(c)");
    k_adain_coeffs<<<cdiv((long long)NR * C, 256), 256, 0, st>>>(mean, var, smean, svar, C, NR, R, alpha, eps, scale, shift);
    WCTB_CHECK_LAUNCH("k_adain_coeffs");
    const long long total = (long long)Nc * Hc * Wc * (C / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > device_sm_count() * 16) blocks = device_sm_count() * 16;
    k_affine_apply_regions<<<(unsigned)blocks, 256, 0, st>>>(content, gc, labels, R, counts, scale, shift, out);
    WCTB_CHECK_LAUNCH("k_affine_apply_regions");
    return 0;
}

}  // namespace wctb
