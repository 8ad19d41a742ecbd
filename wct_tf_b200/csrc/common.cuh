// Shared device/host helpers for libwctb200 (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/wctb200.h"

namespace wctb {

// ---------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
// device error word (set by kernels on pipeline time-outs)
unsigned int* device_error_word();

#define WCTB_CUDA(call)                                        \
    do {                                                       \
        cudaError_t _e = (call);                               \
        if (_e != cudaSuccess) return ::wctb::cuda_fail(_e, #call); \
    } while (0)

#define WCTB_CHECK_LAUNCH(name)                                \
    do {                                                       \
        cudaError_t _e = cudaGetLastError();                   \
        if (_e != cudaSuccess) return ::wctb::cuda_fail(_e, name); \
    } while (0)

#define WCTB_REQUIRE(cond, ...)                                \
    do {                                                       \
        if (!(cond)) {                                         \
            ::wctb::set_error(__VA_ARGS__);                    \
            return WCTB200_EINVAL;                             \
        }                                                      \
    } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Per-DEVICE one-time kernel attribute: cudaFuncSetAttribute applies to the current device only, so the
// "already done" state is one bit per device ordinal (a process may drive several GPUs: WCT(device='/gpu:1')
// after '/gpu:0').  The kernel argument may contain commas: wrap it in parentheses.
#define WCTB_ENSURE_SMEM(kernel, bytes)                                                                  \
    do {                                                                                                 \
        static std::atomic<unsigned long long> _done{0ull};                                              \
        int _dev = 0;                                                                                    \
        WCTB_CUDA(cudaGetDevice(&_dev));                                                                 \
        const unsigned long long _bit = 1ull << (_dev & 63);                                             \
        if (!(_done.load(std::memory_order_acquire) & _bit)) {                                           \
            WCTB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
            _done.fetch_or(_bit, std::memory_order_release);                                             \
        }                                                                                                \
    } while (0)
// SM count of the CURRENT device (cached per device ordinal)
int device_sm_count();

// ---------------------------------------------------------------------------
// SPF16 geometry
// ---------------------------------------------------------------------------
struct ActGeom {
    int N, H, W, C;
    int Hp, Wp;          // H+2, W+2
    int edge;            // halo written by a producer: 0 = REFLECT (ops.py:12-15), 1 = EDGE-replicated (input of an UP2 conv)
    long long P;         // N*Hp*Wp padded positions
    long long plane;     // P*C elements per plane
    __host__ __device__ ActGeom() {}
    __host__ __device__ ActGeom(int n, int h, int w, int c)
        : N(n), H(h), W(w), C(c), Hp(h + 2), Wp(w + 2), edge(0) {
        P = (long long)N * Hp * Wp;
        plane = P * C;
    }
};

#ifdef __CUDACC__
// ---------------------------------------------------------------------------
// split-pair fp16
// ---------------------------------------------------------------------------
__device__ __forceinline__ void split_f32(float x, __half& hi, __half& lo) {
    x = fminf(fmaxf(x, -65000.f), 65000.f);   // keep hi finite
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ float merge_f32(__half hi, __half lo) { return __half2float(hi) + __half2float(lo); }

// 8 channels = one 16-byte vector per plane
struct alignas(16) Half8 { __half2 v[4]; };

// two fp32 -> (hi pair, lo pair).  cvt.rn.satfinite.f16x2.f32 (F2FP.SATFINITE.F16.F32.PACK_AB) converts, saturates to
// +-65504 and packs two values in ONE instruction: 6 instructions per pair instead of the 11 of two clamped scalar splits
// (the conv epilogue is instruction bound on every short-K layer, profiles/r02_ncu_conv_epilogue.txt)
__device__ __forceinline__ void split2(float a, float b, __half2& hi, __half2& lo) {
    unsigned int h, l;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(b), "f"(a));       // a -> low half, b -> high half
    hi = *reinterpret_cast<__half2*>(&h);
    const float2 hf = __half22float2(hi);
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(b - hf.y), "f"(a - hf.x));
    lo = *reinterpret_cast<__half2*>(&l);
}
__device__ __forceinline__ void split8(const float* x, Half8& hi, Half8& lo) {
#pragma unroll
    for (int i = 0; i < 4; ++i) split2(x[2 * i], x[2 * i + 1], hi.v[i], lo.v[i]);
}
__device__ __forceinline__ void merge8(const Half8& hi, const Half8& lo, float* x) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 a = __half22float2(hi.v[i]);
        float2 b = __half22float2(lo.v[i]);
        x[2 * i] = a.x + b.x;
        x[2 * i + 1] = a.y + b.y;
    }
}

// Destinations of interior pixel (y,x) in the reflect-padded plane (ops.py:12-15):
// the pixel itself at (y+1,x+1) plus the halo cells that mirror it.
// rows[] / cols[] receive padded coordinates; returns counts.
__device__ __forceinline__ int halo_rows(int y, int H, int* rows) {
    int n = 0;
    rows[n++] = y + 1;
    if (y == 1) rows[n++] = 0;
    if (y == H - 2) rows[n++] = H + 1;
    return n;
}

// store one 8-channel group (hi+lo) of pixel (n,y,x) to every padded cell that holds it.
// Interior pixels (the overwhelming majority) take the fast path: one address, two 16-byte stores.  (The first version
// evaluated all 9 candidate cells with predicated stores for EVERY pixel: 18 STG + ~26 IMAD per call, which made the
// epilogue of the 64-channel convs -- not their operand traffic -- the bound: 9.4k cycles per 128x64 tile, measured
// identical for 9 and for 4 k-iterations per tile.)
__device__ __forceinline__ void store8_with_halo(__half* __restrict__ act, const ActGeom& g, int n, int y, int x,
                                                 int c0, const Half8& hi, const Half8& lo) {
    // reflect: padded row 0 mirrors interior row 1, row H+1 mirrors row H-2; edge: they replicate rows 0 and H-1
    const int m = g.edge ? 0 : 1;
    __half* p0 = act + (((long long)n * g.Hp + y + 1) * g.Wp + x + 1) * g.C + c0;
    *reinterpret_cast<Half8*>(p0) = hi;
    *reinterpret_cast<Half8*>(p0 + g.plane) = lo;
    const bool yt = (y == m), yb = (y == g.H - 1 - m), xl = (x == m), xr = (x == g.W - 1 - m);
    if (!(yt | yb | xl | xr)) return;
    const long long pitch = (long long)g.Wp * g.C;
    // element offsets from the pixel's own cell to the halo row / column that mirrors it (0 = none)
    const long long dy[3] = {0, yt ? -(long long)(y + 1) * pitch : 0, yb ? (long long)(g.H - y) * pitch : 0};
    const long long dx[3] = {0, xl ? -(long long)(x + 1) * g.C : 0, xr ? (long long)(g.W - x) * g.C : 0};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (a && dy[a] == 0) continue;
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            if ((b && dx[b] == 0) || (a == 0 && b == 0)) continue;
            __half* q = p0 + dy[a] + dx[b];
            *reinterpret_cast<Half8*>(q) = hi;
            *reinterpret_cast<Half8*>(q + g.plane) = lo;
        }
    }
}

// Epilogue variant: the pixel's padded position `ppos` = (n*Hp + y+1)*Wp + x+1 (fits 31 bits) and its border flags
// (bit0: the pixel mirrors into padded row 0, bit1: into row H+1, bit2: into column 0, bit3: into column W+1) were computed
// ONCE by the thread that owns the pixel; the 8 lanes that store its channels only add the channel offset.
__device__ __forceinline__ int halo_flags(const ActGeom& g, int y, int x) {
    const int m = g.edge ? 0 : 1;
    return (y == m ? 1 : 0) | (y == g.H - 1 - m ? 2 : 0) | (x == m ? 4 : 0) | (x == g.W - 1 - m ? 8 : 0);
}
__device__ __forceinline__ void store8_at(__half* __restrict__ act, const ActGeom& g, unsigned int ppos, int flags, int c0,
                                          const Half8& hi, const Half8& lo) {
    __half* p0 = act + (long long)ppos * g.C + c0;
    *reinterpret_cast<Half8*>(p0) = hi;
    *reinterpret_cast<Half8*>(p0 + g.plane) = lo;
    if (flags == 0) return;
    // a mirrored cell sits (m+1) rows / columns beyond the pixel: reflect m = 1 -> 2 away, edge m = 0 -> 1 away
    const int d = g.edge ? 1 : 2;
    const long long pitch = (long long)g.Wp * g.C;
    const long long dy[3] = {0, (flags & 1) ? -d * pitch : 0, (flags & 2) ? d * pitch : 0};
    const long long dx[3] = {0, (flags & 4) ? -(long long)d * g.C : 0, (flags & 8) ? (long long)d * g.C : 0};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (a && dy[a] == 0) continue;
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            if ((b && dx[b] == 0) || (a == 0 && b == 0)) continue;
            __half* q = p0 + dy[a] + dx[b];
            *reinterpret_cast<Half8*>(q) = hi;
            *reinterpret_cast<Half8*>(q + g.plane) = lo;
        }
    }
}

__device__ __forceinline__ void load8(const __half* __restrict__ act, const ActGeom& g, long long pos, int c0,
                                      float* x) {
    long long off = pos * g.C + c0;
    Half8 hi = *reinterpret_cast<const Half8*>(act + off);
    Half8 lo = *reinterpret_cast<const Half8*>(act + g.plane + off);
    merge8(hi, lo, x);
}

// ---------------------------------------------------------------------------
// Coalesced tile store for the GEMM epilogues.  Each epilogue thread owns one output
// position (row) and NACC consecutive channels in registers.  Writing them directly puts
// 16-byte fragments 128+ bytes apart (ncu: 27 half-filled sectors per store request, the
// 64-channel convs were bound by L2 write requests).  Instead every warp transposes
// 64 channels at a time through an 8 KB shared-memory staging buffer (XOR-swizzled, conflict
// free) so that 8 consecutive lanes write one position's 128 contiguous bytes per plane.
//   stg: this warp's private 8 KB buffer; value = acc*oscale + sbias (oscale undoes the power-of-two weight scale);
//   sbias: bias of acc[0..NACC); cbase: channel of acc[0]
// ---------------------------------------------------------------------------
template <int NACC>
__device__ __forceinline__ void store_tile_rows(const float (&acc)[NACC], const float oscale, const float* __restrict__ sbias, bool relu,
                                                uint8_t* __restrict__ stg, int lane, unsigned int ppos, int flags,
                                                __half* __restrict__ out, const ActGeom& go, int cbase) {
    // flags < 0: this thread's position is not an interior pixel (halo / junk row of the padded tiling): nothing is stored
#pragma unroll
    for (int h = 0; h < NACC / 64; ++h) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float t = fmaf(acc[h * 64 + q * 8 + j], oscale, sbias[h * 64 + q * 8 + j]);
                v[j] = relu ? fmaxf(t, 0.f) : t;
            }
            Half8 hi, lo;
            split8(v, hi, lo);
            const int slot = q ^ (lane & 7);
            *reinterpret_cast<Half8*>(stg + (lane * 8 + slot) * 16) = hi;
            *reinterpret_cast<Half8*>(stg + 4096 + (lane * 8 + slot) * 16) = lo;
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int row = j * 4 + (lane >> 3);
            const int c = lane & 7;
            const unsigned int pp = __shfl_sync(0xffffffffu, ppos, row);
            const int fl = __shfl_sync(0xffffffffu, flags, row);
            const int slot = c ^ (row & 7);
            const Half8 hi = *reinterpret_cast<const Half8*>(stg + (row * 8 + slot) * 16);
            const Half8 lo = *reinterpret_cast<const Half8*>(stg + 4096 + (row * 8 + slot) * 16);
            if (fl >= 0) store8_at(out, go, pp, fl, cbase + h * 64 + c * 8, hi, lo);
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------
// packed fp32 pairs: fma.rn.f32x2 does two FMAs per instruction on sm_100 (same FMA-pipe time, half the issue slots)
// ---------------------------------------------------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// ---------------------------------------------------------------------------
// PTX wrappers: mbarrier / TMA / tcgen05 (sm_100a)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
#ifdef WCTB_MBAR_TEST_WAIT
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#else
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#endif
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must not hang the GPU.  After ~2 s the CTA-wide abort
// flag is raised (all later waits fall through) and the global error word is set.
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, volatile int* abort_flag,
                                          unsigned int* err_word, unsigned int code) {
    if (mbar_try_wait(bar, parity)) return;
    // The time-out clock is the SM cycle counter: reading %globaltimer costs ~0.5 us (measured: every wait that
    // missed its first poll paid it, which capped the tap-reuse conv pipelines at ~1 us per k-iteration).
    const long long t0 = clock64();
    for (unsigned int it = 1;; ++it) {
        if (mbar_try_wait(bar, parity)) return;
        if ((it & 255u) == 0u) {
            if (*abort_flag) return;
            if (*reinterpret_cast<volatile unsigned int*>(err_word)) { *abort_flag = 1; return; }
            if (clock64() - t0 > 4000000000ll) break;            // >= 2 s at <= 2 GHz
        }
    }
    *abort_flag = 1;
    atomicExch(err_word, code);
}

__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], kind::f16 (fp16 inputs, fp32 accumulate), issued by ONE thread
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread retire
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled shared-memory operand descriptor (tile rows are 128 bytes =
// 64 fp16 of K; 8-row groups 1024 B apart).  Bit layout: cute::UMMA::SmemDescriptor.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);   // start address  [0,14)
    d |= (uint64_t)1 << 16;                       // LBO (unused for swizzled K-major) [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;             // SBO = 1024 B   [32,46)
    d |= (uint64_t)1 << 46;                       // descriptor version = 1 (sm_100)
    d |= (uint64_t)2 << 61;                       // layout type = SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: fp16 x fp16 -> fp32, K-major A and B, M x N tile.
// Bit layout: cute::UMMA::InstrDescriptor.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
    return (1u << 4)                      // c_format = F32
           | (0u << 7) | (0u << 10)       // a_format = b_format = F16
           | (0u << 15) | (0u << 16)      // a_major = b_major = K
           | ((uint32_t)(N >> 3) << 17)   // n_dim
           | ((uint32_t)(M >> 4) << 24);  // m_dim
}
// MN-major SWIZZLE_128B operand (used when the contraction index is the slow one: covariance X^T X, Gram G^T G):
// 64 MN elements (128 B) per row, rows = K; LBO = stride between 64-wide MN groups (8 KB: the next slice / the lo plane),
// SBO = stride between 8-row K groups (1 KB)  (cute::UMMA canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte
// units; strides probed on B200, profiles/r01_cov_mn_major_probe.txt)
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((8192 >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((1024 >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__host__ __device__ constexpr uint32_t umma_idesc_f16_mn(int M, int N) {
    return (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
#endif  // __CUDACC__

// per-(device, stream, slot) grow-only scratch buffer (capi.cu); valid until the next call with the same key
int scratch_alloc(void** ptr, size_t bytes, cudaStream_t st, int slot);

// ---------------------------------------------------------------------------
// kernel launchers implemented in the .cu files (host API used by capi.cu)
// ---------------------------------------------------------------------------
enum ConvMode { CONV_3X3 = 0, CONV_APPLY = 1, CONV_UP2 = 2, CONV_TAPS = 3 };
int launch_conv_tc(int mode, const __half* in, int N, int H, int W, int Cin, const __half* w_split, int nsets,
                   const float* wscale, const float* bias, int Cout, int flags, __half* out, cudaStream_t st, int kw = 3,
                   const uint8_t* labels = nullptr, int R = 1, const uint32_t* tilemask = nullptr);
// trailer of a prepared weight buffer: [0] = 1/scale (float), see wctb200_prep_conv_weights
static inline const float* weight_scale_ptr(const __half* w_split, int taps_total, int Cin, int Cout) {
    return reinterpret_cast<const float*>(w_split + (size_t)2 * taps_total * Cin * Cout);
}

}  // namespace wctb
