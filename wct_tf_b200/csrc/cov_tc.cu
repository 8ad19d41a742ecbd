// Covariance GEMM  S = sum_p (x_p - t)(x_p - t)^T  (C x HW . HW x C, ops.py:43-45,48-50,105-108) on the tensor cores,
// with the centring and the per-channel sums fused in: ONE pass over the features.
//
// The features are SPF16 [pixel][channel]: for the product X^T X the contraction index K is the
// PIXEL, so both operands are "MN-major" (for a fixed k the 64 channels of a slice are the 128
// contiguous bytes of a row).  A TMA box of 64 pixels x 64 channels lands as the canonical
// MN-major SWIZZLE_128B tile (8-pixel groups of 1024 B), and tcgen05.mma reads A and B from the
// same staged tiles with a_major = b_major = MN.  The tensor map is built over the INTERIOR of the
// reflect-padded plane (base pointer at pixel (0,0), padded strides, dims W x H): boxes that stick
// out at a ragged edge are zero-filled by TMA and add nothing to the sums, halo cells are never read.
//
// Centring (ops.py:44,49,106: fc = f - mean BEFORE the product).  Round 1 ran three extra passes for it (channel sums,
// a centred SPF16 copy written to HBM, the product over the copy).  Now a tiny pre-kernel estimates a per-channel SHIFT t
// (the mean of <= 1024 strided pixels; the exact mean when HW <= 1024), eight worker warps subtract t from every staged
// tile IN SHARED MEMORY (hi+lo -> fp32 -> minus t -> re-split, zero-filled out-of-range pixels stay zero) before the MMA warp
// may read it, and accumulate s = sum_p (x_p - t) on the way.  The finalize kernel forms
//     cov = (S - s s^T / HW) / (HW - 1),   mean = t + s / HW
// in fp64: exact algebra for ANY t, and with t within sigma/32 of the mean the subtracted term is ~1e-3 of S, so nothing
// cancels (the fully uncentred form, t = 0, was measured in round 1: it produced a spurious eigenvalue above the 1e-5 cut).
//
// Determinism.  Products in fp32 (split-fp16 x3), drained from TMEM every 128 pixels into registers (the tensor core
// accumulates with truncation and the diagonals are all-positive sums).  Every CTA writes its partial block and partial sums
// to its OWN slot; the finalize kernel adds the slots in a fixed order.  The split of an image into CTAs depends on (C, H, W)
// only -- not on the batch size or the SM count -- so a frame's covariance is bit-identical whatever batch or GPU it is in
// (tests: 2-GPU shards == 1 GPU, batch == single frames).
//
// One CTA = one 128 x 128 block pair (bi <= bj) of the C x C matrix x one range of pixel tiles.
#include "common.cuh"

namespace wctb {

struct CovParams {
    int C, W, H, N;
    int tiles_x, tiles_y;        // 32 x 2 pixel tiles per image
    int ksplit, tiles_per_split;
    int nb;                      // 128-channel blocks (C=64: 1 block, rows duplicated)
    int nslots;                  // partial slots per image: ksplit (C=64: 4*ksplit)
    int max_stages;              // cap on the ring depth (probe knob; 12 = no cap)
    const float* shift;          // [N][C]
    float* part;                 // [N][nslots][C][C] fp32 partial products (upper block triangle)
    float* psum;                 // [N][ksplit][C] fp32 partial sums of (x - shift)
    unsigned int* err;
    // per-region statistics (wctb200_wct_apply_regions): item i = frame * R + region reads frame i / R; pixels whose label
    // [frame][y][x] is not the item's region are zeroed in the centring step like TMA's out-of-range pixels
    const uint8_t* labels;       // [N][H][W] or nullptr
    int R;                       // regions per frame (1 without labels)
};

struct CovCfg {
    static constexpr int SLICE = 64 * 128;                  // 64 pixels x 64 channels fp16 = 8 KB
    static constexpr int OPER = 4 * SLICE;                  // 2 channel slices x 2 planes
    static constexpr int STAGE = 2 * OPER;                  // A + B (off-diagonal block pair); a diagonal pair uses OPER, C = 64 two SLICEs
    static constexpr int RING_BYTES = 3 * STAGE;            // 192 KB of tiles in flight whatever the stage size: 3 / 6 / 12 stages
    static constexpr int STAGES = 12;                       // barrier slots (the deepest ring)
    static constexpr int NBUF = 4;
    static constexpr int CH = 2;                            // 64-pixel tiles per TMEM accumulation chunk (24 truncating adds)
    static constexpr int THREADS = 320;                     // producer, MMA, 8 worker warps (centring + TMEM drains)
    static constexpr int RED_BYTES = 32 * 128 * 4;          // worker warps: [32 row groups][128 channels] partial sums
    static constexpr int SMEM_BYTES = RING_BYTES + 512 + RED_BYTES + 1024;
};

__device__ __forceinline__ void tma_load_5d_cov(void* smem_dst, const void* map, uint64_t* bar, int c0, int c1, int c2,
                                                int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
        : "memory");
}

// REG: statistics per (frame, region) item (CovParams::labels); a template parameter so that the plain covariance compiles as before
template <bool REG>
__global__ void __launch_bounds__(CovCfg::THREADS, 1)
cov_tc_kernel(const __grid_constant__ CUtensorMap mapX, const CovParams p) {
    using Cfg = CovCfg;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* aux = smem + Cfg::RING_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(aux);
    uint64_t* empty = full + Cfg::STAGES;
    uint64_t* ready = empty + Cfg::STAGES;
    uint64_t* tfull = ready + Cfg::STAGES;
    uint64_t* tempty = tfull + Cfg::NBUF;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + Cfg::NBUF);
    volatile int* abort_flag = reinterpret_cast<volatile int*>(tmem_slot + 1);
    float* red = reinterpret_cast<float*>(aux + 512);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // block pair / k-split / image of this CTA
    const int npairs = p.nb * (p.nb + 1) / 2;
    const int pair = blockIdx.x % npairs;
    const int split = blockIdx.x / npairs;
    int bi = 0, rem = pair;
    while (rem >= p.nb - bi) { rem -= p.nb - bi; ++bi; }
    const int bj = bi + rem;
    const bool diag = (bi == bj);
    const int img = blockIdx.y;                  // item: output slots
    const int frame = REG ? img / p.R : img;     // image the tiles are read from
    const int region = REG ? img - frame * p.R : 0;
    const int tiles_img = p.tiles_x * p.tiles_y;
    const int t0 = split * p.tiles_per_split;
    const int t1 = min(t0 + p.tiles_per_split, tiles_img);
    const int ntiles = max(t1 - t0, 0);
    // C = 64: a single 64-channel slice.  The 128-row operand is [hi plane | lo plane] of that slice and is used as BOTH
    // A and B: ONE MMA per 16 pixels yields hi.hi, hi.lo, lo.hi (and lo.lo) as the four 64x64 quadrants of the 128x128
    // accumulator; the epilogue adds the quadrants.
    const bool dup = (p.C == 64);

    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&ready[s], 8); }
        for (int b = 0; b < Cfg::NBUF; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 8); }
        *abort_flag = 0;
        fence_barrier_init();
        tma_prefetch_desc(&mapX);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int nchunks = (ntiles + Cfg::CH - 1) / Cfg::CH;
    // One stage holds exactly what one tile needs, so the ring is 3 (off-diagonal pair), 6 (diagonal pair) or 12 (C = 64)
    // stages deep: the C <= 128 levels are HBM-latency bound, with 3 stages of 16 KB in flight a CTA could not pull more than
    // ~27 GB/s (measured 0.34 of the HBM rate)
    const uint32_t stage_bytes = dup ? 2 * Cfg::SLICE : (diag ? Cfg::OPER : Cfg::STAGE);
    const int nst = min(Cfg::RING_BYTES / (int)stage_bytes, p.max_stages);

    if (warp == 0) {
        if (lane == 0) {
            // (stage index, barrier phase and tile coordinates advance incrementally: runtime div/mod cost ~40 instructions each)
            int s = 0, ty = t0 / p.tiles_x, tx = t0 - ty * p.tiles_x;
            uint32_t ph = 0;
            for (int it = 0; it < ntiles; ++it, ++s, ++tx) {
                if (s == nst) { s = 0; ph ^= 1u; }
                if (tx == p.tiles_x) { tx = 0; ++ty; }
                mbar_wait(&empty[s], ph ^ 1u, abort_flag, p.err, 0x510u + s);
                uint8_t* st = smem + s * stage_bytes;
                mbar_arrive_expect_tx(&full[s], stage_bytes);
                if (dup) {
                    tma_load_5d_cov(st, &mapX, &full[s], 0, tx * 32, ty * 2, frame, 0);                  // rows 0..63   : hi
                    tma_load_5d_cov(st + Cfg::SLICE, &mapX, &full[s], 0, tx * 32, ty * 2, frame, 1);     // rows 64..127 : lo
                    continue;
                }
                for (int op = 0; op < (diag ? 1 : 2); ++op) {
                    const int blk = op == 0 ? bi : bj;
                    for (int sl = 0; sl < 2; ++sl) {
                        const int ch = blk * 128 + sl * 64;
                        for (int pl = 0; pl < 2; ++pl)
                            tma_load_5d_cov(st + op * Cfg::OPER + (pl * 2 + sl) * Cfg::SLICE, &mapX, &full[s], ch, tx * 32,
                                            ty * 2, frame, pl);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16_mn(128, 128);
            int it = 0, s = 0;
            uint32_t ph = 0;
            for (int c = 0; c < nchunks; ++c) {
                const int b = c % Cfg::NBUF;
                mbar_wait(&tempty[b], ((c / Cfg::NBUF) & 1) ^ 1u, abort_flag, p.err, 0x540u + b);
                tc_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)(b * 128);
                const int it_end = min(ntiles, (c + 1) * Cfg::CH);
                for (; it < it_end; ++it, ++s) {
                    if (s == nst) { s = 0; ph ^= 1u; }
                    mbar_wait(&ready[s], ph, abort_flag, p.err, 0x520u + s);   // tile landed AND centred
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(smem + s * stage_bytes);
                    const uint32_t b0 = diag ? a0 : a0 + Cfg::OPER;
                    const bool first = (it == c * Cfg::CH);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {           // 64 pixels = 4 x UMMA_K(16): 16 rows of 128 B = 2048 B per step
                        const uint32_t ko = k * 2048;
                        if (dup) {
                            const uint64_t d = umma_desc_mn_sw128(a0 + ko);   // [hi | lo] x [hi | lo]^T
                            umma_f16(tacc, d, d, idesc, (first && k == 0) ? 0u : 1u);
                            continue;
                        }
                        const uint64_t a_hi = umma_desc_mn_sw128(a0 + ko);
                        const uint64_t a_lo = umma_desc_mn_sw128(a0 + 2 * Cfg::SLICE + ko);
                        const uint64_t b_hi = umma_desc_mn_sw128(b0 + ko);
                        const uint64_t b_lo = umma_desc_mn_sw128(b0 + 2 * Cfg::SLICE + ko);
                        umma_f16(tacc, a_hi, b_lo, idesc, (first && k == 0) ? 0u : 1u);
                        umma_f16(tacc, a_lo, b_hi, idesc, 1u);
                        umma_f16(tacc, a_hi, b_hi, idesc, 1u);
                    }
                    umma_commit(&empty[s]);
                }
                umma_commit(&tfull[b]);
            }
        }
        __syncwarp();
    } else {
        // ---- 8 worker warps (2..9).  All of them centre the staged tiles (x -> x - shift in place, sums of the shifted
        // values); in between they drain the finished TMEM chunks into registers: warps 2-5 own accumulator columns 0..63,
        // warps 6-9 columns 64..127 (a warp may only read the TMEM lanes of its quadrant, warp & 3).  One warp per
        // scheduler for the centring (the first version: warps 6-9 only) ran at the latency of its own instruction chain
        // and capped the kernel at 0.34 of the HBM rate.
        const int ct = threadIdx.x - 64;      // 0..255
        const int chunk = ct & 7;             // logical 16-byte chunk of a 128-byte row = channels chunk*8 .. +7 of the slice
        const int rg = ct >> 3;               // rows rg and rg+32 of every 64-pixel slice
        const int pchunk = (chunk ^ (rg & 7)) << 4;      // SWIZZLE_128B: physical chunk = logical ^ (row & 7); row & 7 == rg & 7
        const int nops = dup ? 1 : (diag ? 1 : 2);
        const int nsl = dup ? 1 : 2;
        const bool want_sums = dup || diag;   // every channel block has exactly one diagonal pair
        const int g = warp & 3;               // TMEM lane quadrant
        const int chalf = warp >= 6 ? 1 : 0;  // accumulator column half drained by this warp
        float sh[2][2][8], sums[2][8], acc[64];
#pragma unroll
        for (int op = 0; op < 2; ++op)
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                const int blk = op == 0 ? bi : bj;
                const int c0 = dup ? chunk * 8 : blk * 128 + sl * 64 + chunk * 8;
#pragma unroll
                for (int j = 0; j < 8; ++j) sh[op][sl][j] = (op < nops && sl < nsl) ? __ldg(p.shift + (long long)img * p.C + c0 + j) : 0.f;
            }
#pragma unroll
        for (int sl = 0; sl < 2; ++sl)
#pragma unroll
            for (int j = 0; j < 8; ++j) sums[sl][j] = 0.f;
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] = 0.f;
        int drained = 0;
        auto drain = [&](int c) {
            const int b = c % Cfg::NBUF;
            mbar_wait(&tfull[b], (c / Cfg::NBUF) & 1, abort_flag, p.err, 0x530u + b);
            tc_fence_after();
            const uint32_t tsrc = tmem_base + ((uint32_t)(g * 32) << 16) + (uint32_t)(b * 128 + chalf * 64);
            uint32_t r0[32], r1[32];
            tmem_ld32(tsrc, r0);
            tmem_ld32(tsrc + 32, r1);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r0[j]);
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[32 + j] += __uint_as_float(r1[j]);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[b]);
        };
        // fence.proxy.async (generic-proxy writes -> visible to the tensor core) is expensive: measured ~2100 cycles per tile
        // whatever the number of centring warps or the ring depth (ncu: tensor pipe 13 % active, 2.2 TB/s).  The workers
        // therefore centre a GROUP of tiles per fence: 4 when the ring is 12 deep, 2 when 6, 1 when 3.
        const int T = nst >= 12 ? 4 : (nst >= 6 ? 2 : 1);
        int s = 0, ty = t0 / p.tiles_x, tx = t0 - ty * p.tiles_x;
        uint32_t ph = 0;
        for (int it0 = 0; it0 < ntiles; it0 += T) {
            const int it1 = min(it0 + T, ntiles);
            const int s_first = s;
            for (int it = it0; it < it1; ++it, ++s, ++tx) {
                if (s == nst) { s = 0; ph ^= 1u; }
                if (tx == p.tiles_x) { tx = 0; ++ty; }
                mbar_wait(&full[s], ph, abort_flag, p.err, 0x550u + s);
                uint8_t* st = smem + s * stage_bytes;
#pragma unroll
                for (int op = 0; op < 2; ++op) {
                    if (op >= nops) break;
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl) {
                        if (sl >= nsl) break;
                        uint8_t* hi_base = dup ? st : st + op * Cfg::OPER + sl * Cfg::SLICE;
                        uint8_t* lo_base = dup ? st + Cfg::SLICE : st + op * Cfg::OPER + (2 + sl) * Cfg::SLICE;
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const int r = rg + 32 * k;
                            const int x = tx * 32 + (r & 31), y = ty * 2 + (r >> 5);
                            const int off = r * 128 + pchunk;
                            if (REG && x < p.W && y < p.H && p.labels[((long long)frame * p.H + y) * p.W + x] != region) {
                                // another region's pixel: zero, so that it adds nothing to S or s
                                Half8 z;
#pragma unroll
                                for (int j = 0; j < 4; ++j) z.v[j] = __float2half2_rn(0.f);
                                *reinterpret_cast<Half8*>(hi_base + off) = z;
                                *reinterpret_cast<Half8*>(lo_base + off) = z;
                            } else if (x < p.W && y < p.H) {    // out-of-range pixels were zero-filled by TMA and must stay zero
                                const Half8 h = *reinterpret_cast<const Half8*>(hi_base + off);
                                const Half8 l = *reinterpret_cast<const Half8*>(lo_base + off);
                                float v[8];
                                merge8(h, l, v);
#pragma unroll
                                for (int j = 0; j < 8; ++j) v[j] -= sh[op][sl][j];
                                if (op == 0) {
#pragma unroll
                                    for (int j = 0; j < 8; ++j) sums[sl][j] += v[j];
                                }
                                Half8 nh, nl;
                                split8(v, nh, nl);
                                *reinterpret_cast<Half8*>(hi_base + off) = nh;
                                *reinterpret_cast<Half8*>(lo_base + off) = nl;
                            }
                        }
                    }
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                int sa = s_first == nst ? 0 : s_first;
                for (int it = it0; it < it1; ++it) {
                    mbar_arrive(&ready[sa]);
                    if (++sa == nst) sa = 0;
                }
            }
            // every tile of the chunks up to (it1-1) / CH is centred now: drain the chunks BEFORE that one
            {
                const int cdone = (it1 - 1) / Cfg::CH;
                while (drained < cdone) drain(drained++);
            }
        }
        while (drained < nchunks) drain(drained++);
        // ---- this CTA's partial block -> its own slot ----
        const int m = g * 32 + lane;          // accumulator row
        if (!*abort_flag) {
            if (dup) {
                // accumulator rows m and m+64 both belong to channel m & 63, columns j and 64+j to channel j: the four
                // (row half, column half) quadrants go to four slots, the finalize kernel adds them
                float* dst = p.part + (((long long)img * p.nslots + split * 4 + (m >> 6) * 2 + chalf) * p.C + (m & 63)) * p.C;
#pragma unroll
                for (int j = 0; j < 64; j += 4)
                    *reinterpret_cast<float4*>(dst + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
            } else {
                float* dst = p.part + (((long long)img * p.nslots + split) * p.C + bi * 128 + m) * p.C + bj * 128 + chalf * 64;
#pragma unroll
                for (int j = 0; j < 64; j += 4)
                    *reinterpret_cast<float4*>(dst + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
            }
        }
        if (want_sums) {
            // fixed-order reduction over the 32 row groups, then one partial per (image, split, channel)
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
#pragma unroll
                for (int j = 0; j < 8; ++j) red[rg * 128 + sl * 64 + chunk * 8 + j] = sums[sl][j];
        }
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (want_sums) {
            const int nch = dup ? 64 : 128;
            if (ct < nch && !*abort_flag) {
                float a = 0.f;
#pragma unroll
                for (int r = 0; r < 32; ++r) a += red[r * 128 + ct];
                p.psum[((long long)img * p.ksplit + split) * p.C + (dup ? 0 : bi * 128) + ct] = a;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Region form of k_sample_shift: item n = frame * R + region; the mean of the sampled pixels OF THE REGION.  A region the
// sample misses (a few pixels) takes the mean of all its pixels (stride 1); an empty region gets t = 0.
__device__ __noinline__ void k_sample_shift_region(const __half* __restrict__ act, const ActGeom& g, int stride,
                                                   float* __restrict__ shift, const uint8_t* __restrict__ labels, int R,
                                                   float (*red)[64]) {
    __shared__ int cnt_red[32];
    const int grp = threadIdx.x & 7, rl = threadIdx.x >> 3;
    const int c0 = blockIdx.x * 64 + grp * 8;
    const int item = blockIdx.y, frame = item / R, region = item - frame * R;
    const long long HW = (long long)g.H * g.W;
    const uint8_t* lab = labels + (long long)frame * HW;
    float s[8];
    int cnt = 0;
    for (int pass = 0; pass < 2; ++pass) {
        const int str = pass == 0 ? stride : 1;
        const long long ns = (HW + str - 1) / str;
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] = 0.f;
        int c = 0;
        for (long long k = rl; k < ns; k += 32) {
            const long long q = k * str;
            if (lab[q] != region) continue;
            const int y = (int)(q / g.W), x = (int)(q - (long long)y * g.W);
            float v[8];
            load8(act, g, ((long long)frame * g.Hp + y + 1) * g.Wp + x + 1, c0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) s[j] += v[j];
            ++c;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) red[rl][grp * 8 + j] = s[j];
        if (grp == 0) cnt_red[rl] = c;
        __syncthreads();
        cnt = 0;
        for (int r = 0; r < 32; ++r) cnt += cnt_red[r];
        if (cnt > 0 || str == 1) break;
        __syncthreads();
    }
    if (threadIdx.x < 64) {
        float a = 0.f;
#pragma unroll
        for (int r = 0; r < 32; ++r) a += red[r][threadIdx.x];
        shift[(long long)item * g.C + blockIdx.x * 64 + threadIdx.x] = cnt > 0 ? a / (float)cnt : 0.f;
    }
}

// shift[n][c] = mean of <= ~1024 strided interior pixels (all pixels when HW <= 1024): fixed-order reduction.
// grid (C/64, N): one CTA per 64 channels of an image (a single CTA per image took 180 us at C = 512);
// 256 threads = 8 channel groups x 32 pixel lanes
__global__ void __launch_bounds__(256)
k_sample_shift(const __half* __restrict__ act, ActGeom g, int stride, float* __restrict__ shift, const uint8_t* __restrict__ labels,
               int R) {
    __shared__ float red[32][64];
    const int grp = threadIdx.x & 7, rl = threadIdx.x >> 3;
    const int c0 = blockIdx.x * 64 + grp * 8;
    const int n = blockIdx.y;
    if (labels) {
        k_sample_shift_region(act, g, stride, shift, labels, R, red);
        return;
    }
    const long long HW = (long long)g.H * g.W;
    const long long ns = (HW + stride - 1) / stride;
    float s[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = 0.f;
#pragma unroll 4
    for (long long k = rl; k < ns; k += 32) {
        const long long q = k * stride;
        const int y = (int)(q / g.W), x = (int)(q - (long long)y * g.W);
        float v[8];
        load8(act, g, ((long long)n * g.Hp + y + 1) * g.Wp + x + 1, c0, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += v[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[rl][grp * 8 + j] = s[j];
    __syncthreads();
    if (threadIdx.x < 64) {
        float a = 0.f;
#pragma unroll
        for (int r = 0; r < 32; ++r) a += red[r][threadIdx.x];
        shift[(long long)n * g.C + blockIdx.x * 64 + threadIdx.x] = a / (float)ns;
    }
}

// dsum[n][c] = sum over splits of psum (fp64, fixed order); mean = shift + dsum / HW
__global__ void k_cov_sums(const float* __restrict__ psum, const float* __restrict__ shift, int C, int ksplit, long long HW,
                           int total, double* __restrict__ dsum, float* __restrict__ mean, const int* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int n = i / C, c = i - n * C;
    double a = 0.0;
    for (int s = 0; s < ksplit; ++s) a += (double)psum[((long long)n * ksplit + s) * C + c];
    dsum[i] = a;
    const long long cnt = counts ? (long long)counts[n] : HW;      // regions: the pixels of the item's region
    mean[i] = cnt > 0 ? (float)((double)shift[i] + a / (double)cnt) : shift[i];
}

// G = (sum_slots part - s s^T / HW) / (HW - 1) + eps_cov * I   (ops.py:45,50,108,121), exactly symmetric
__global__ void k_cov_finalize(const float* __restrict__ part, const double* __restrict__ dsum, int C, int nslots, long long HW0,
                               float eps_cov, int count, float* __restrict__ G, float* __restrict__ A0, const int* __restrict__ counts) {
    const long long total = (long long)count * C * C;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(t % C);
        const int i = (int)((t / C) % C);
        const long long n = t / ((long long)C * C);
        const long long HW = counts ? (long long)counts[n] : HW0;
        if (HW < 2) {                 // a region of < 2 pixels: 1/(n-1) is undefined; its pixels are copied, never transformed
            G[t] = 0.f;
            if (A0) A0[t] = 0.f;
            continue;
        }
        // every (min,max) entry lies in a stored upper block: reading it for both (i,j) and (j,i) makes G exactly symmetric
        const long long e = (i <= j) ? (long long)i * C + j : (long long)j * C + i;
        const float* pp = part + n * nslots * (long long)C * C + e;
        // four interleaved partial sums (a fixed order all the same): the serial fp64 chain over up to 256 slots took 73-85 us
        double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
        const long long cc = (long long)C * C;
        int s = 0;
        for (; s + 4 <= nslots; s += 4) {
            v0 += (double)pp[(long long)s * cc];
            v1 += (double)pp[(long long)(s + 1) * cc];
            v2 += (double)pp[(long long)(s + 2) * cc];
            v3 += (double)pp[(long long)(s + 3) * cc];
        }
        for (; s < nslots; ++s) v0 += (double)pp[(long long)s * cc];
        double v = (v0 + v1) + (v2 + v3);
        v -= dsum[n * C + i] * dsum[n * C + j] / (double)HW;
        float r = (float)(v / (double)(HW - 1));
        if (i == j) r += eps_cov;
        G[t] = r;
        if (A0) A0[t] = r;          // pristine copy: the Jacobi kernel overwrites G, the Rayleigh quotients need A
    }
}

// ---------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiledC)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int g_cov_max_stages = 12;   // probe knob (wctb200_debug_set_cov_stages)

// Means and covariance (+ eps_cov I) of a feature batch: mean [N][C], G [N][C][C] (and a copy A0 if not null), fp32.
// dsum: [N][C] fp64 scratch (caller's workspace); partial products live in the per-stream scratch cache.
// labels / R / counts (optional): statistics per (frame, region) item, n = frame * R + region, over the pixels whose label
// [frame][y][x] is the region; counts [N*R] = those pixel counts (k_region_counts); outputs are [N*R][...].
int launch_mean_cov(const __half* act, ActGeom g, float eps_cov, float* mean, float* G, float* A0, double* dsum, cudaStream_t st,
                    const uint8_t* labels, int R, const int* counts) {
    static PFN_encodeTiledC enc = nullptr;
    if (!enc) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            set_error("cuTensorMapEncodeTiled entry point not available");
            return WCTB200_ECUDA;
        }
        enc = reinterpret_cast<PFN_encodeTiledC>(ptr);
    }
    WCTB_REQUIRE(g.C == 64 || (g.C % 128 == 0 && g.C <= 2048), "covariance: C=%d must be 64 or a multiple of 128 (<= 2048)", g.C);
    const long long HW = (long long)g.H * g.W;
    if (!labels) R = 1;
    const int items = g.N * R;
    CovParams p;
    p.C = g.C; p.W = g.W; p.H = g.H; p.N = g.N;
    p.labels = labels;
    p.R = R;
    p.tiles_x = (g.W + 31) / 32;
    p.tiles_y = (g.H + 1) / 2;
    p.nb = g.C == 64 ? 1 : g.C / 128;
    const int npairs = p.nb * (p.nb + 1) / 2;
    const int tiles_img = p.tiles_x * p.tiles_y;
    // Split of one image into CTAs: a function of (C, H, W) ONLY (batch- and device-invariant results).  Up to 64 tiles
    // (4096 pixels) per CTA keeps the ~5 us of TMEM/barrier set-up per CTA below 20 % and still gives a single
    // 512x512 frame 64 CTAs per block pair.
    int tps = 64;
    if (tiles_img < 64 * 8) tps = (tiles_img + 7) / 8;        // small maps: 8 splits
    if (tps < 8) tps = 8;
    p.tiles_per_split = tps;
    p.ksplit = (tiles_img + tps - 1) / tps;
    p.nslots = g.C == 64 ? 4 * p.ksplit : p.ksplit;
    // scratch: shift [N][C] | psum [N][ksplit][C] | part [N][nslots][C][C]
    const size_t n_shift = (size_t)items * g.C, n_psum = (size_t)items * p.ksplit * g.C;
    const size_t n_part = (size_t)items * p.nslots * g.C * g.C;
    float* scratch = nullptr;
    { int rc0 = scratch_alloc(reinterpret_cast<void**>(&scratch), (n_shift + n_psum + n_part + 64) * sizeof(float), st, 0); if (rc0) return rc0; }
    float* shift = scratch;
    float* psum = shift + ((n_shift + 3) & ~(size_t)3);
    float* part = psum + ((n_psum + 3) & ~(size_t)3);
    p.shift = shift; p.psum = psum; p.part = part;
    p.err = device_error_word();
    p.max_stages = g_cov_max_stages;
    // (blocks below the diagonal are never written -- and never read: k_cov_finalize only touches (min,max) entries)

    const int stride = HW <= 1024 ? 1 : (int)(HW / 1024);
    k_sample_shift<<<dim3((unsigned)(g.C / 64), (unsigned)items), 256, 0, st>>>(act, g, stride, shift, labels, R);
    WCTB_CHECK_LAUNCH("k_sample_shift");

    // tensor map over the interior pixels only (see header comment)
    CUtensorMap mX;
    const __half* base = act + ((long long)g.Wp + 1) * g.C;
    cuuint64_t dims[5] = {(cuuint64_t)g.C, (cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)g.N, 2};
    cuuint64_t strides[4] = {(cuuint64_t)g.C * 2, (cuuint64_t)g.Wp * g.C * 2, (cuuint64_t)g.Hp * g.Wp * g.C * 2,
                             (cuuint64_t)g.plane * 2};
    cuuint32_t box[5] = {64, 32, 2, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&mX, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<__half*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cov_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return WCTB200_ECUDA;
    }
    dim3 grid((unsigned)(npairs * p.ksplit), (unsigned)items);
    if (labels) {
        WCTB_ENSURE_SMEM(cov_tc_kernel<true>, CovCfg::SMEM_BYTES);
        cov_tc_kernel<true><<<grid, CovCfg::THREADS, CovCfg::SMEM_BYTES, st>>>(mX, p);
    } else {
        WCTB_ENSURE_SMEM(cov_tc_kernel<false>, CovCfg::SMEM_BYTES);
        cov_tc_kernel<false><<<grid, CovCfg::THREADS, CovCfg::SMEM_BYTES, st>>>(mX, p);
    }
    WCTB_CHECK_LAUNCH("cov_tc_kernel");
    k_cov_sums<<<cdiv((long long)items * g.C, 256), 256, 0, st>>>(psum, shift, g.C, p.ksplit, HW, items * g.C, dsum, mean,
                                                                   labels ? counts : nullptr);
    WCTB_CHECK_LAUNCH("k_cov_sums");
    const long long tot = (long long)items * g.C * g.C;
    k_cov_finalize<<<(unsigned)(cdiv(tot, 256) > 4096 ? 4096 : cdiv(tot, 256)), 256, 0, st>>>(part, dsum, g.C, p.nslots, HW,
                                                                                               eps_cov, items, G, A0,
                                                                                               labels ? counts : nullptr);
    WCTB_CHECK_LAUNCH("k_cov_finalize");
    return 0;
}

}  // namespace wctb
