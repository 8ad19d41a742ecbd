// Conv2DReflect 3x3, the 1x1 "apply" of the feature transform, and UpSampling2D+Conv2DReflect as ONE conv,
// all as an implicit GEMM on the 5th-gen tensor cores.
//
//   reference: Lambda(pad_reflect) -> Conv2D(valid) (+ReLU)   ops.py:12-19,
//              vgg_normalised.py:28-40, model.py:291; the whitening/colouring
//              apply  M * fc  of ops.py:73,77 (mode APPLY); and
//              UpSampling2D() -> Conv2DReflect of model.py:291-293 (mode UP2).
//
// Formulation.  Activations are SPF16: two fp16 planes (hi, lo) of the padded
// NHWC tensor, viewed as a 2-D matrix [P = N*(H+2)*(W+2) padded positions][C].  For an
// output position p (padded coordinates) and filter tap (ky,kx) the input row is simply
// p + (ky-1)*(W+2) + (kx-1): each tap of a 128-position output tile is ONE dense
// 128 x 64 TMA box at a shifted row coordinate (rows outside [0,P) are zero-filled by
// TMA and only feed halo/junk outputs, which the epilogue never stores).
//
//   D[128 pos][BN cout] = sum_{tap, cin-slice}  A_tap[128][64] * W_tap[BN][64]^T
//
// UP2 (nearest x2 upsampling folded into the conv that follows it).  Output pixel (2i+a, 2j+b) of
// conv3x3(reflect_pad(upsample2(L))) only ever reads the 2x2 low-resolution neighbourhood
// rows {i-1+a, i+a} x cols {j-1+b, j+b} of L, because two of the three filter rows (columns) land on the same
// low-resolution row (column): a = 0 -> {w[-1]} on row i-1 and {w[0]+w[1]} on row i; a = 1 -> {w[-1]+w[0]} on
// row i and {w[1]} on row i+1.  So each of the 4 output parities is a 2x2-tap conv over L with pre-summed
// weights (wctb200_prep_conv_weights_up2): 16 instead of 36 tap-products per low-resolution pixel (4/9 of the
// MACs), and the 4x larger upsampled tensor is never written or read.  At the border the reflect padding of the
// UPSAMPLED image mirrors onto the same low-resolution pixel (u[-1] = u[1] = L[0]), i.e. L needs an EDGE-replicated
// halo: its producer is launched with WCTB200_HALO_EDGE.
//
// Precision.  fp32-class accuracy from fp16 tensor-core inputs: x = x_hi + x_lo,
//   x*w ~= x_hi*w_hi + x_hi*w_lo + x_lo*w_hi     (3 x tcgen05.mma kind::f16, fp32 accumulate in TMEM)
// the dropped lo*lo term is 2^-22 relative.  Weights are stored SCALED by a per-layer power of two
// (max|w| -> [512,1024), undone exactly in the epilogue): He-initialised / trained conv weights are ~1e-2, so the
// unscaled lo plane (~5e-6) fell into the fp16 subnormals and kept only ~16 bits of the weight -- measured as
// 8x the reference's own fp32 noise on the free-running 5-level image (profiles/r02_noise_split.txt).
//
// Structure (persistent CTAs, 192 threads):
//   warp 0   : TMA producer   (cp.async.bulk.tensor 3-D, 128B swizzle, mbarrier complete_tx)
//   warp 1   : MMA issuer     (one elected thread, tcgen05.mma / tcgen05.commit), owns TMEM alloc
//   warps 2-5: epilogue       (tcgen05.ld 32x32b -> *scale +bias, ReLU -> split fp16 -> 16-byte stores
//                              of the interior pixel AND the halo cells that mirror it)
#include "common.cuh"

namespace wctb {

extern int g_conv_bn_override;

struct ConvParams {
    int N, H, W, Cin, Cout, Hp, Wp;   // INPUT geometry (UP2: the low-resolution tensor)
    long long P;
    int mode;             // ConvMode
    int taps;             // 9 (3x3), 1 (apply), 4 (up2: per output parity), kw*kw (taps)
    int kw;               // CONV_TAPS: filter width (top-left anchored kw x kw correlation, style-swap patches)
    int products;         // 3 (default): a_hi b_hi + a_hi b_lo + a_lo b_hi; 2: without a_lo b_hi; 1: a_hi b_hi only (experiment knob)
    int per_image;        // tiles never straddle images; weight/bias set = image index (APPLY with nsets > 1)
    int pool;             // CONV_3X3 + WCTB200_POOL2: M tile = 2 image rows x 64 columns, 2x2 max-pool in the epilogue
    int pool_tx, pool_ho; // pool: column segments per row pair, row pairs per image
    int nsets;
    int tiles_per_image;
    int flags;
    const float* bias;    // [nsets][Cout] or nullptr
    const float* wscale;  // device scalar: 1 / (power-of-two scale the weights were stored with), or nullptr (= 1)
    __half* out;          // SPF16, Cout channels; UP2: [N, 2H, 2W, Cout]
    unsigned int* err;
    // APPLY per region (wctb200_wct_apply_regions): work items are (tile, region) pairs, weight / bias set image*R + region;
    // tilemask[image][tile] bit r = the tile holds a pixel of region r that is transformed, the epilogue stores only those
    const uint8_t* labels;      // [N][H][W] or nullptr
    const uint32_t* tilemask;   // [N][tiles_per_image]
    int R;
};

// ===========================================================================
// v2: persistent CTAs + chunked accumulation drained into registers
//
//   * grid = #SMs, every CTA walks a static tile list (cout tile fastest, so CTAs running
//     together share activation tiles in L2 and the whole weight tensor stays L2 resident);
//   * the accumulator ring: TMEM holds NBUF buffers of BN fp32 columns.  The MMA warp
//     accumulates CH k-iterations (CH*4*3 tcgen05.mma) into one buffer starting from zero,
//     commits it, and moves on to the next buffer; the epilogue warps drain each finished
//     buffer with tcgen05.ld and ADD IT INTO REGISTERS with round-to-nearest FADDs.
//     The tensor core adds into its fp32 accumulator with truncation (measured: -1.2e-5
//     relative bias at K=4608 when everything is accumulated in TMEM); short chunks summed
//     in registers bring the conv back to fp32-class error, and the drain of chunk i
//     overlaps the MMAs of chunk i+1 (also across tiles: the epilogue of tile t overlaps
//     the main loop of tile t+1).
// ===========================================================================
template <int BN, bool FUSE_>
struct Conv2Cfg {
    static constexpr int BM = 128;
    static constexpr int BK = 64;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int STAGES = BN == 64 ? 4 : (BN == 128 ? 3 : 2);
    // FUSE: the products a_hi*b_hi and a_hi*b_lo share the A operand, and the two weight planes sit back to back in a
    // stage, so ONE tcgen05.mma with N = 2*BN computes both into adjacent accumulator column ranges (summed when the
    // chunk is drained); a_lo*b_hi follows with N = BN into the first range.  8 instead of 12 MMAs per k-iteration and
    // half the A-operand shared-memory reads per flop (timeline probe: ~80 cycles per MMA regardless of N <= 128).
    static constexpr bool FUSE = FUSE_ && BN <= 128;
    static constexpr int ACC_COLS = FUSE ? 2 * BN : BN;         // TMEM columns of one accumulation buffer
    static constexpr int NBUF = 512 / ACC_COLS >= 4 ? 4 : 2;
    static constexpr int TMEM_COLS = NBUF * ACC_COLS;           // 512 / 512 / 512
    static constexpr int CH = 4;                                // k-iterations per accumulation chunk
    // (8 epilogue warps -- two per TMEM lane quadrant, 32-channel staging, 64-byte stores -- were measured in round 2:
    //  slower on every short-K layer, e.g. UP2 64->64 841 -> 1002 us; profiles/r02_conv_layer_bench.txt)
    static constexpr int EPI_WARPS = BN == 256 ? 8 : 4;
    static constexpr int THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int NACC = BN / (EPI_WARPS / 4);           // accumulators per epilogue thread (<= 128)
    static constexpr int AUX_BYTES = 256 + BN * 4;
    static constexpr int STG_BYTES = BN <= 128 ? 4 * 8192 : 0;  // per-epilogue-warp store staging (coalesced stores)
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + AUX_BYTES + STG_BYTES + 1024;
};

struct TileCoord {
    long long p0, p_end;
    int n0, set;
    int cls;              // UP2: output parity class a*2+b
    int region;           // APPLY per region: the region this work item stores
    bool skip;            // APPLY per region: the tile holds no pixel of the region (every role skips the item)
};

template <bool REG>
__device__ __forceinline__ TileCoord tile_coord(const ConvParams& p, int tile, int n_tiles, int BN) {
    TileCoord t;
    const int nt = tile % n_tiles;
    int mt = tile / n_tiles;
    const long long HpWp = (long long)p.Hp * p.Wp;
    t.n0 = nt * BN;
    t.cls = 0;
    t.region = 0;
    t.skip = false;
    if (REG) {
        // region fastest after the cout tile: the R items of one position tile run together and share its A tiles in L2
        t.region = mt % p.R;
        mt /= p.R;
        const int img = mt / p.tiles_per_image;
        const int r = mt - img * p.tiles_per_image;
        t.p0 = img * HpWp + (long long)r * 128;
        t.p_end = (img + 1) * HpWp;
        t.set = img * p.R + t.region;
        t.skip = ((__ldg(p.tilemask + mt) >> t.region) & 1u) == 0u;
    } else if (p.pool) {
        // mt = (image * row pairs + pair i) * column segments + t; rows 2i, 2i+1, interior columns [64t, 64t + 64)
        const int t_ = mt % p.pool_tx;
        const int r_ = mt / p.pool_tx;
        const int i_ = r_ % p.pool_ho;
        const int img = r_ / p.pool_ho;
        t.p0 = img * HpWp + (long long)(2 * i_ + 1) * p.Wp + 1 + 64 * t_;     // first position of the UPPER row segment
        t.p_end = p.P;
        t.set = 0;
        t.cls = t_;                          // (reused: column segment; the row pair is recovered from p0)
    } else if (p.mode == CONV_UP2) {
        // cout tile fastest, then the 4 parity classes: CTAs running together share one activation tile in L2
        t.cls = mt & 3;
        mt >>= 2;
        t.p0 = (long long)mt * 128;
        t.p_end = p.P;
        t.set = t.cls;                       // weight set = parity class
    } else if (p.per_image) {
        const int img = mt / p.tiles_per_image;
        const int r = mt - img * p.tiles_per_image;
        t.p0 = img * HpWp + (long long)r * 128;
        t.p_end = (img + 1) * HpWp;
        t.set = p.nsets > 1 ? img : 0;
    } else {
        t.p0 = (long long)mt * 128;
        t.p_end = p.P;
        t.set = 0;
    }
    return t;
}

// REG: the per-region apply (ConvParams::labels); a template parameter so that every other conv compiles as before
template <int BN, bool FUSE_, bool REG>
__global__ void __launch_bounds__(Conv2Cfg<BN, FUSE_>::THREADS, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const __grid_constant__ CUtensorMap mapA64, const ConvParams p, const int total_tiles, const int n_tiles) {
    using Cfg = Conv2Cfg<BN, FUSE_>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* aux = smem + Cfg::STAGES * Cfg::STAGE_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(aux);
    uint64_t* empty = full + Cfg::STAGES;
    uint64_t* tfull = empty + Cfg::STAGES;
    uint64_t* tempty = tfull + Cfg::NBUF;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + Cfg::NBUF);
    volatile int* abort_flag = reinterpret_cast<volatile int*>(tmem_slot + 1);
    float* sbias = reinterpret_cast<float*>(aux + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    {
        __shared__ unsigned int s_prev_err;
        if (threadIdx.x == 0) s_prev_err = *reinterpret_cast<volatile unsigned int*>(p.err);
        __syncthreads();
        if (s_prev_err != 0u) return;
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < Cfg::NBUF; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], Cfg::EPI_WARPS);
        }
        *abort_flag = 0;
        fence_barrier_init();
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int ksl = p.Cin / Cfg::BK;
    const int kiters = p.taps * ksl;
    const int nchunks = (kiters + Cfg::CH - 1) / Cfg::CH;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t itg = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const TileCoord tc = tile_coord<REG>(p, tile, n_tiles, BN);
                if (REG && tc.skip) continue;        // the MMA and epilogue warps skip the same items (same tile_coord)
                for (int it = 0; it < kiters; ++it, ++itg) {
                    const int s = itg % Cfg::STAGES;
                    const uint32_t ph = (itg / Cfg::STAGES) & 1;
                    mbar_wait(&empty[s], ph ^ 1u, abort_flag, p.err, 0x100u + s);
                    const int tap = it / ksl;
                    const int ks = it - tap * ksl;
                    int off = 0;
                    if (p.mode == CONV_3X3) off = (tap / 3 - 1) * p.Wp + (tap % 3 - 1);
                    else if (p.mode == CONV_TAPS) off = (tap / p.kw) * p.Wp + (tap % p.kw);
                    else if (p.mode == CONV_UP2) off = ((tap >> 1) - 1 + (tc.cls >> 1)) * p.Wp + ((tap & 1) - 1 + (tc.cls & 1));
                    const int row = (int)(tc.p0 + off);
                    uint8_t* st = smem + s * Cfg::STAGE_BYTES;
                    mbar_arrive_expect_tx(&full[s], Cfg::STAGE_BYTES);
                    if (p.pool) {
                        // two 64-position boxes per plane: the segment of image row 2i and the one below it
                        tma_load_3d(st, &mapA64, &full[s], ks * Cfg::BK, row, 0);
                        tma_load_3d(st + Cfg::A_BYTES / 2, &mapA64, &full[s], ks * Cfg::BK, row + p.Wp, 0);
                        tma_load_3d(st + Cfg::A_BYTES, &mapA64, &full[s], ks * Cfg::BK, row, 1);
                        tma_load_3d(st + Cfg::A_BYTES + Cfg::A_BYTES / 2, &mapA64, &full[s], ks * Cfg::BK, row + p.Wp, 1);
                    } else {
                        tma_load_3d(st, &mapA, &full[s], ks * Cfg::BK, row, 0);
                        tma_load_3d(st + Cfg::A_BYTES, &mapA, &full[s], ks * Cfg::BK, row, 1);
                    }
                    tma_load_3d(st + 2 * Cfg::A_BYTES, &mapB, &full[s], tap * p.Cin + ks * Cfg::BK, tc.n0, tc.set * 2);
                    tma_load_3d(st + 2 * Cfg::A_BYTES + Cfg::B_BYTES, &mapB, &full[s], tap * p.Cin + ks * Cfg::BK,
                                tc.n0, tc.set * 2 + 1);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(Cfg::BM, BN);
            constexpr uint32_t idesc2 = umma_idesc_f16(Cfg::BM, Cfg::FUSE ? 2 * BN : BN);
            uint32_t itg = 0, cg_ = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                if (REG && tile_coord<REG>(p, tile, n_tiles, BN).skip) continue;
                for (int c = 0; c < nchunks; ++c, ++cg_) {
                    const int b = cg_ % Cfg::NBUF;
                    const uint32_t bph = (cg_ / Cfg::NBUF) & 1;
                    mbar_wait(&tempty[b], bph ^ 1u, abort_flag, p.err, 0x400u + b);   // epilogue drained this buffer
                    tc_fence_after();
                    const uint32_t tacc = tmem_base + (uint32_t)(b * Cfg::ACC_COLS);
                    const int it_end = min(kiters, (c + 1) * Cfg::CH);
                    for (int it = c * Cfg::CH; it < it_end; ++it, ++itg) {
                        const int s = itg % Cfg::STAGES;
                        const uint32_t ph = (itg / Cfg::STAGES) & 1;
                        mbar_wait(&full[s], ph, abort_flag, p.err, 0x200u + s);
                        tc_fence_after();
                        const uint32_t st = smem_u32(smem + s * Cfg::STAGE_BYTES);
                        const uint64_t a_hi = umma_desc_sw128(st);
                        const uint64_t a_lo = umma_desc_sw128(st + Cfg::A_BYTES);
                        const uint64_t b_hi = umma_desc_sw128(st + 2 * Cfg::A_BYTES);
                        const uint64_t b_lo = umma_desc_sw128(st + 2 * Cfg::A_BYTES + Cfg::B_BYTES);
                        const bool first = (it == c * Cfg::CH);
#pragma unroll
                        for (int k = 0; k < Cfg::BK / 16; ++k) {
                            const uint64_t ko = (uint64_t)(k * 32 >> 4);
                            if (Cfg::FUSE) {
                                // [b_hi | b_lo] is one 2*BN-row K-major tile: columns [0,BN) += a_hi b_hi, [BN,2BN) += a_hi b_lo
                                umma_f16(tacc, a_hi + ko, b_hi + ko, idesc2, (first && k == 0) ? 0u : 1u);
                                if (p.products >= 3) umma_f16(tacc, a_lo + ko, b_hi + ko, idesc, 1u);
                            } else {
                                umma_f16(tacc, a_hi + ko, b_hi + ko, idesc, (first && k == 0) ? 0u : 1u);
                                if (p.products >= 2) umma_f16(tacc, a_hi + ko, b_lo + ko, idesc, 1u);
                                if (p.products >= 3) umma_f16(tacc, a_lo + ko, b_hi + ko, idesc, 1u);
                            }
                        }
                        umma_commit(&empty[s]);
                    }
                    umma_commit(&tfull[b]);
                }
            }
        }
        __syncwarp();
    } else {
        // ---- epilogue warps: drain chunks into registers, then bias/ReLU/split/store ----
        const int e = warp - 2;
        const int g = warp & 3;                              // TMEM lane quadrant of this warp
        const int colbase = (e >> 2) * Cfg::NACC;            // BN=256: warps 6..9 take the upper half
        const int et = threadIdx.x - 64;                     // 0 .. 32*EPI_WARPS-1
        constexpr int ETHREADS = 32 * Cfg::EPI_WARPS;
        const bool up2 = p.mode == CONV_UP2;
        ActGeom go(p.N, up2 ? 2 * p.H : (p.pool ? (p.H + 1) / 2 : p.H), up2 ? 2 * p.W : (p.pool ? (p.W + 1) / 2 : p.W), p.Cout);
        go.edge = (p.flags & WCTB200_HALO_EDGE) ? 1 : 0;
        const bool relu = (p.flags & WCTB200_RELU) != 0;
        const float wsc = p.wscale ? __ldg(p.wscale) : 1.f;
        uint32_t cg_ = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const TileCoord tc = tile_coord<REG>(p, tile, n_tiles, BN);
            if (REG && tc.skip) continue;
            // stage this tile's bias slice (named barrier 1: epilogue warps only)
            asm volatile("bar.sync 1, %0;" ::"r"(ETHREADS) : "memory");
            for (int i = et; i < BN; i += ETHREADS) sbias[i] = p.bias ? p.bias[(long long)(p.mode == CONV_APPLY ? tc.set : 0) * p.Cout + tc.n0 + i] : 0.f;   // UP2: set = weight parity class, ONE bias
            asm volatile("bar.sync 1, %0;" ::"r"(ETHREADS) : "memory");

            float acc[Cfg::NACC];
#pragma unroll
            for (int i = 0; i < Cfg::NACC; ++i) acc[i] = 0.f;
            for (int c = 0; c < nchunks; ++c, ++cg_) {
                const int b = cg_ % Cfg::NBUF;
                const uint32_t bph = (cg_ / Cfg::NBUF) & 1;
                mbar_wait(&tfull[b], bph, abort_flag, p.err, 0x300u + b);
                tc_fence_after();
                const uint32_t tsrc = tmem_base + ((uint32_t)(g * 32) << 16) + (uint32_t)(b * Cfg::ACC_COLS + colbase);
                if (Cfg::FUSE) {
#pragma unroll
                    for (int c0 = 0; c0 < Cfg::NACC; c0 += 32) {
                        uint32_t r0[32], r1[32];
                        tmem_ld32(tsrc + c0, r0);               // a_hi b_hi + a_lo b_hi
                        tmem_ld32(tsrc + BN + c0, r1);          // a_hi b_lo
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[c0 + j] += __uint_as_float(r0[j]) + __uint_as_float(r1[j]);
                    }
                } else {
#pragma unroll
                    for (int c0 = 0; c0 < Cfg::NACC; c0 += 64) {
                        uint32_t r0[32], r1[32];
                        tmem_ld32(tsrc + c0, r0);
                        if (c0 + 32 < Cfg::NACC) tmem_ld32(tsrc + c0 + 32, r1);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[c0 + j] += __uint_as_float(r0[j]);
                        if (c0 + 32 < Cfg::NACC) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) acc[c0 + 32 + j] += __uint_as_float(r1[j]);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[b]);      // buffer may be overwritten
            }
            if (Cfg::STG_BYTES > 0 && p.pool) {
                // ---- MaxPooling2D 2x2/2 'same' (vgg_normalised.py:41-42) on the raw accumulators: max commutes with the
                // monotone  *scale + bias -> ReLU -> split  that follows.  Tile rows 0..63 = image row 2i, 64..127 = row 2i+1.
                // Work split: the two lanes of a horizontal pixel pair share the pooled pixel's channels (16-channel blocks:
                // lane parity l owns channels 8l..8l+7 of each block), and the warps of the two image rows share them by halves
                // (upper-row warps keep the lower half of the channel range, lower-row warps the upper half), so every lane of
                // all four warps finishes and stores NACC/4 channels of one pooled pixel.
                constexpr int NH = Cfg::NACC / 2;            // channels per half
                constexpr int Q = Cfg::NACC / 4;             // channels a lane finishes
                const int tpos = g * 32 + lane;
                const int xloc = tpos & 63;
                const int hv = tpos >> 6;                    // 0: image row 2i, 1: row 2i+1
                const int lp = lane & 1;
                const unsigned int hpwp = (unsigned int)(p.Hp * p.Wp);
                const unsigned int n = (unsigned int)tc.p0 / hpwp;
                const int yy0 = (int)(((unsigned int)tc.p0 - n * hpwp) / (unsigned int)p.Wp);   // padded row of image row 2i
                const int x = 64 * tc.cls + xloc;
                const bool valid = (yy0 - 1 + hv) < p.H && x < p.W;
                if (__any_sync(0xffffffffu, !valid)) {       // ragged right / bottom edge only
                    const float ninf = __int_as_float(0xff800000);
#pragma unroll
                    for (int j = 0; j < Cfg::NACC; ++j) acc[j] = valid ? acc[j] : ninf;
                }
                // horizontal: m[h][k] = max over the pixel pair of channel  h*NH + (k>>3)*16 + lp*8 + (k&7)
                float keep[Q], send[Q];
#pragma unroll
                for (int k = 0; k < Q; ++k) {
                    const int c0 = (k >> 3) * 16 + (k & 7);
                    float mh[2];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const float a0 = acc[h * NH + c0], a1 = acc[h * NH + c0 + 8];
                        const float mine = lp ? a1 : a0;
                        const float other = lp ? a0 : a1;    // the neighbour lane's channel, this lane's pixel
                        mh[h] = fmaxf(mine, __shfl_xor_sync(0xffffffffu, other, 1));
                    }
                    keep[k] = hv ? mh[1] : mh[0];
                    send[k] = hv ? mh[0] : mh[1];
                }
                // vertical: hand the other half over to the warp of the other image row (same lane = same pixel column)
                uint8_t* stg_all = aux + Cfg::AUX_BYTES;
                {
                    float* xb = reinterpret_cast<float*>(stg_all + e * 8192) + lane;
#pragma unroll
                    for (int k = 0; k < Q; ++k) xb[k * 32] = send[k];
                }
                asm volatile("bar.sync 1, %0;" ::"r"(ETHREADS) : "memory");
                {
                    const float* pb = reinterpret_cast<const float*>(stg_all + (e ^ 2) * 8192) + lane;   // TMEM quadrant g ^ 2
#pragma unroll
                    for (int k = 0; k < Q; ++k) keep[k] = fmaxf(keep[k], pb[k * 32]);
                }
                const int xe = x & ~1;                       // the even column of the pair
                if (xe < p.W && yy0 - 1 < p.H && !*abort_flag) {
                    const int yo = (yy0 - 1) >> 1, xo = xe >> 1;
                    const int flags = halo_flags(go, yo, xo);
                    const unsigned int ppos = (n * (unsigned int)go.Hp + (unsigned int)(yo + 1)) * (unsigned int)go.Wp + (unsigned int)(xo + 1);
                    const int cb = colbase + hv * NH + lp * 8;   // first channel this lane stores
#pragma unroll
                    for (int q = 0; q < Q / 8; ++q) {
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float t = fmaf(keep[q * 8 + j], wsc, sbias[cb + q * 16 + j]);
                            v[j] = relu ? fmaxf(t, 0.f) : t;
                        }
                        Half8 hi, lo;
                        split8(v, hi, lo);
                        store8_at(p.out, go, ppos, flags, tc.n0 + cb + q * 16, hi, lo);
                    }
                }
                continue;
            }
            // ---- store: interior pixel + the halo cells that mirror it ----
            // (32-bit position arithmetic: P < 2^31 is checked by the launcher; 64-bit divisions cost ~60 instructions each)
            const unsigned int pos = (unsigned int)tc.p0 + (unsigned int)(g * 32 + lane);
            int flags = -1;                                      // < 0: nothing to store for this row
            unsigned int ppos = 0;
            if (pos < (unsigned int)tc.p_end) {
                const unsigned int hpwp = (unsigned int)(p.Hp * p.Wp);
                const unsigned int n = pos / hpwp;
                const unsigned int r = pos - n * hpwp;
                const int yy = (int)(r / (unsigned int)p.Wp);
                const int xx = (int)(r - (unsigned int)yy * (unsigned int)p.Wp);
                if (yy >= 1 && yy <= p.H && xx >= 1 && xx <= p.W && !*abort_flag &&
                    (!REG || p.labels[((long long)n * p.H + (yy - 1)) * p.W + (xx - 1)] == tc.region)) {
                    int y = yy - 1, x = xx - 1;
                    if (up2) { y = 2 * y + (tc.cls >> 1); x = 2 * x + (tc.cls & 1); }
                    flags = halo_flags(go, y, x);
                    ppos = ((unsigned int)n * (unsigned int)go.Hp + (unsigned int)(y + 1)) * (unsigned int)go.Wp + (unsigned int)(x + 1);
                }
            }
            if (Cfg::STG_BYTES > 0) {
                uint8_t* stg = aux + Cfg::AUX_BYTES + e * 8192;
                store_tile_rows<Cfg::NACC>(acc, wsc, sbias + colbase, relu, stg, lane, ppos, flags, p.out, go, tc.n0 + colbase);
            } else if (flags >= 0) {
#pragma unroll
                for (int q = 0; q < Cfg::NACC / 8; ++q) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float t = fmaf(acc[q * 8 + j], wsc, sbias[colbase + q * 8 + j]);
                        v[j] = relu ? fmaxf(t, 0.f) : t;
                    }
                    Half8 hi, lo;
                    split8(v, hi, lo);
                    store8_at(p.out, go, ppos, flags, tc.n0 + colbase + q * 8, hi, lo);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    }
    return fn;
}

// 3-D fp16 tensor map [d2][d1][d0] (d0 contiguous), box {64, box1, 1}, 128B swizzle, zero OOB fill
int make_tensor_map_3d(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                    uint64_t stride2_bytes, uint32_t box1) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled entry point not available");
        return WCTB200_ECUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {64, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): dims %llu %llu %llu strides %llu %llu box1 %u", (int)r,
                  (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, box1);
        return WCTB200_ECUDA;
    }
    return 0;
}

int g_conv_oversub = 4;

template <int BN, bool FUSE_, bool REG = false>
static int launch2_bn(const CUtensorMap& mA, const CUtensorMap& mB, const CUtensorMap& mA64, const ConvParams& p, int total_tiles,
                      int n_tiles, cudaStream_t st) {
    using Cfg = Conv2Cfg<BN, FUSE_>;
    WCTB_ENSURE_SMEM((conv_tc2_kernel<BN, FUSE_, REG>), Cfg::SMEM_BYTES);
    // Over-subscribed persistent grid: with g_conv_oversub x #SMs CTAs (1 resident per SM) the
    // hardware block scheduler hands queued CTAs to whichever SMs are free, so a conv launched
    // while the Jacobi clusters of the other stream hold half the SMs still balances its tiles
    // (a grid of exactly #SMs would run as two unbalanced waves).
    int grid = device_sm_count() * (g_conv_oversub > 0 ? g_conv_oversub : 1);
    if (grid > total_tiles) grid = total_tiles;
    conv_tc2_kernel<BN, FUSE_, REG><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(mA, mB, mA64, p, total_tiles, n_tiles);
    WCTB_CHECK_LAUNCH("conv_tc2_kernel");
    return 0;
}

int g_conv_products = 3;     // experiment knob (wctb200_debug_set_conv_products): split-fp16 products per MAC
int g_conv_fuse = -1;        // -1 auto, 0 never, 1 whenever the tile allows (wctb200_debug_set_conv_fuse)
int g_conv_bn_override = 0;  // test/tuning hook: force the N tile (64/128/256)

// mode CONV_3X3  : in [N,H,W,Cin], w_split [2][Cout][9*Cin],          out [N,H,W,Cout]
// mode CONV_APPLY: in [N,H,W,Cin], w_split [nsets][2][Cout][Cin],     out [N,H,W,Cout]   (per-image weight sets)
// mode CONV_UP2  : in [N,H,W,Cin] (edge halo), w_split [4][2][Cout][4*Cin], out [N,2H,2W,Cout]
// mode CONV_TAPS : in [N,H,W,Cin], w_split [2][Cout][kw*kw*Cin],      out [N,H,W,Cout]: top-left anchored kw x kw correlation
// APPLY with labels: nsets = N*R weight sets (image-major), work items (tile, region) skipped where tilemask says so
int launch_conv_tc(int mode, const __half* in, int N, int H, int W, int Cin, const __half* w_split, int nsets,
                   const float* wscale, const float* bias, int Cout, int flags, __half* out, cudaStream_t st, int kw,
                   const uint8_t* labels, int R, const uint32_t* tilemask) {
    WCTB_REQUIRE(N >= 1 && H >= 2 && W >= 2, "conv: bad geometry N=%d H=%d W=%d", N, H, W);
    WCTB_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0 && Cin >= 64 && Cout >= 64, "conv: Cin=%d Cout=%d must be multiples of 64", Cin, Cout);
    WCTB_REQUIRE(mode == CONV_3X3 || mode == CONV_APPLY || mode == CONV_UP2 || mode == CONV_TAPS, "conv: bad mode %d", mode);
    WCTB_REQUIRE(mode != CONV_TAPS || (kw >= 1 && kw <= 16), "conv: bad filter width %d", kw);
    if (!labels) R = 1;
    WCTB_REQUIRE(!labels || (mode == CONV_APPLY && tilemask && R >= 1 && R <= 32 && nsets == N * R && !(flags & WCTB200_POOL2)),
                 "conv: per-region apply needs the apply mode, a tile mask and N*R weight sets");
    WCTB_REQUIRE(labels || nsets == 1 || (mode == CONV_APPLY && nsets == N), "conv: nsets must be 1 (or N in apply mode)");
    ActGeom gi(N, H, W, Cin);
    WCTB_REQUIRE(gi.P < (1ll << 31) - 4096, "conv: too many padded positions (%lld)", gi.P);
    WCTB_REQUIRE(mode != CONV_UP2 || ActGeom(N, 2 * H, 2 * W, Cout).P < (1ll << 31), "conv: too many output positions");
    const int taps = mode == CONV_3X3 ? 9 : (mode == CONV_UP2 ? 4 : (mode == CONV_TAPS ? kw * kw : 1));
    const int wsets = mode == CONV_UP2 ? 4 : nsets;

    const bool pool = (flags & WCTB200_POOL2) != 0;
    WCTB_REQUIRE(!pool || (mode == CONV_3X3 && (H + 1) / 2 >= 2 && (W + 1) / 2 >= 2), "conv: POOL2 needs the 3x3 mode and a pooled output >= 2x2");
    int BN = Cout % 128 == 0 ? 128 : 64;   // 256-wide tiles leave only 2 pipeline stages: measured slower
    if (g_conv_bn_override && Cout % g_conv_bn_override == 0) BN = g_conv_bn_override;
    if ((pool || labels) && BN > 128) BN = 128;   // the pooling / per-region epilogues work on the 4-warp layouts

    CUtensorMap mA, mB;
    int rc = make_tensor_map_3d(&mA, in, (uint64_t)Cin, (uint64_t)gi.P, 2, (uint64_t)Cin * 2, (uint64_t)gi.plane * 2, 128);
    if (rc) return rc;
    const uint64_t K = (uint64_t)taps * Cin;
    rc = make_tensor_map_3d(&mB, w_split, K, (uint64_t)Cout, (uint64_t)2 * wsets, K * 2, K * Cout * 2, (uint32_t)BN);
    if (rc) return rc;
    CUtensorMap mA64 = mA;
    if (pool) {
        rc = make_tensor_map_3d(&mA64, in, (uint64_t)Cin, (uint64_t)gi.P, 2, (uint64_t)Cin * 2, (uint64_t)gi.plane * 2, 64);
        if (rc) return rc;
    }

    ConvParams p;
    p.N = N; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout; p.Hp = gi.Hp; p.Wp = gi.Wp; p.P = gi.P;
    p.mode = mode;
    p.taps = taps;
    p.kw = kw;
    p.products = (mode == CONV_3X3 || mode == CONV_UP2) ? g_conv_products : 3;    // the knob only touches the encoder / decoder convs
    p.nsets = nsets;
    p.per_image = (nsets > 1 || labels) ? 1 : 0;
    p.labels = labels;
    p.tilemask = tilemask;
    p.R = R;
    p.tiles_per_image = cdiv((long long)gi.Hp * gi.Wp, 128);
    p.pool = pool ? 1 : 0;
    p.pool_tx = cdiv(W, 64);
    p.pool_ho = (H + 1) / 2;
    p.flags = flags;
    p.bias = bias;
    p.wscale = wscale;
    p.out = out;
    p.err = device_error_word();
    const int m_tiles = pool ? N * p.pool_ho * p.pool_tx : (p.per_image ? N * p.tiles_per_image * R : cdiv(gi.P, 128));
    const int n_tiles = Cout / BN;
    const int total = m_tiles * n_tiles * (mode == CONV_UP2 ? 4 : 1);
    if (labels) {   // per-region apply: the same tile / fusion choice as the plain apply, so one region computes bit-identically
        if (BN == 64) return g_conv_fuse == 0 ? launch2_bn<64, false, true>(mA, mB, mA64, p, total, n_tiles, st)
                                              : launch2_bn<64, true, true>(mA, mB, mA64, p, total, n_tiles, st);
        return (g_conv_fuse == 1 || (g_conv_fuse < 0 && (long long)taps * Cin >= 9 * 256))
                   ? launch2_bn<128, true, true>(mA, mB, mA64, p, total, n_tiles, st)
                   : launch2_bn<128, false, true>(mA, mB, mA64, p, total, n_tiles, st);
    }
    switch (BN) {
        // fused [b_hi|b_lo] MMAs (Conv2Cfg::FUSE): always at BN=64 (4 TMEM buffers stay); at BN=128 the ring shrinks to 2
        // buffers, which only pays for long K loops (measured: Cin=128 -9 %, Cin>=256 +3..5 %)
        case 64: return g_conv_fuse == 0 ? launch2_bn<64, false>(mA, mB, mA64, p, total, n_tiles, st)
                                         : launch2_bn<64, true>(mA, mB, mA64, p, total, n_tiles, st);
        case 128: return (g_conv_fuse == 1 || (g_conv_fuse < 0 && (long long)taps * Cin >= 9 * 256))
                             ? launch2_bn<128, true>(mA, mB, mA64, p, total, n_tiles, st)
                             : launch2_bn<128, false>(mA, mB, mA64, p, total, n_tiles, st);
        default: return launch2_bn<256, false>(mA, mB, mA64, p, total, n_tiles, st);
    }
}

}  // namespace wctb
