// extern "C" surface of libwctb200 (declared in include/wctb200.h).
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "wctb200_debug.h"

namespace wctb {

static thread_local char t_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return WCTB200_ECUDA;
}

// Per-stream scratch cache.  Work on one stream is ordered, so a stream can reuse ONE grow-only buffer per slot for every
// call it serves.  (The first version used cudaMallocAsync/cudaFreeAsync: the stream-ordered pool only re-uses a block
// across streams once a dependency exists, so with 8 streams it kept growing at unpredictable moments AFTER the warm-up
// steps -- each growth maps hundreds of MB and showed up as a one-off 75..500 ms step in some bench runs.)
int scratch_alloc(void** ptr, size_t bytes, cudaStream_t st, int slot) {
    struct Entry { void* p; size_t cap; };
    static std::mutex mu;
    static std::map<std::tuple<int, cudaStream_t, int>, Entry> cache;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    Entry& e = cache[std::make_tuple(dev, st, slot)];
    if (e.cap < bytes) {
        if (e.p) {
            WCTB_CUDA(cudaStreamSynchronize(st));
            WCTB_CUDA(cudaFree(e.p));
            e.p = nullptr;
            e.cap = 0;
        }
        const size_t cap = bytes + bytes / 8 + 256;
        WCTB_CUDA(cudaMalloc(&e.p, cap));
        e.cap = cap;
    }
    *ptr = e.p;
    return 0;
}

__device__ unsigned int g_device_error = 0;

unsigned int* device_error_word() {
    static unsigned int* ptr[64] = {nullptr};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!ptr[dev]) {
        void* p = nullptr;
        if (cudaGetSymbolAddress(&p, g_device_error) == cudaSuccess) ptr[dev] = static_cast<unsigned int*>(p);
    }
    return ptr[dev];
}

int device_sm_count() {
    static std::atomic<int> sms[64];
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    int v = sms[dev].load(std::memory_order_relaxed);
    if (v <= 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        sms[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

// launchers (layers.cu / wct.cu)
int launch_u8_to_f32(const uint8_t*, size_t, float*, cudaStream_t);
int launch_f32_to_u8(const float*, size_t, uint8_t*, cudaStream_t);
size_t resize_workspace_bytes(int N, int Hs, int Ws, int C, int Hd, int Wd, int Wout);
int launch_resize_u8(const uint8_t* src, int N, int Hs, int Ws, int C, int Hd, int Wd, int y0, int x0, int Hout, int Wout,
                     uint8_t* dst, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_rgb_moments(const uint8_t* img, long long npix, unsigned long long* sums, cudaStream_t st);
int launch_coral_apply(const uint8_t* src, long long npix, const double* A, const double* sm, const double* ss, const double* tm,
                       const double* ts, uint8_t* dst, cudaStream_t st);
int launch_act_from_f32(const float*, ActGeom, __half*, cudaStream_t);
int launch_act_to_f32(const __half*, ActGeom, float*, cudaStream_t);
int launch_prep_weights(const float*, int, int, int, __half*, cudaStream_t);
int launch_prep_weights_up2(const float*, int, int, __half*, cudaStream_t);
size_t style_swap_workspace_bytes(int C, int Hc, int Wc, int Hs, int Ws, int P, int S);
int launch_style_swap_level(const __half* content, int Hc, int Wc, const __half* style, int Hs, int Ws, int C, int patch, int stride,
                            float alpha, float eps_cov, float thresh, __half* out, int32_t* k_out, void* ws, size_t ws_bytes,
                            cudaStream_t st);
int launch_conv3x3_ref(const __half*, ActGeom, const float*, const float*, int, int, __half*, cudaStream_t);
int launch_conv_head(const float*, int, int, int, const float*, const float*, __half*, cudaStream_t);
int launch_conv_tail(const __half*, ActGeom, const float*, const float*, int, float*, cudaStream_t);
int launch_maxpool2(const __half*, ActGeom, __half*, cudaStream_t);
int launch_upsample2(const __half*, ActGeom, __half*, cudaStream_t);
size_t wct_workspace_bytes(int, int, int);
int launch_wct_level(const __half*, int, int, int, const __half*, int, int, int, int, float, float, float, float, int,
                     __half*, int32_t*, void*, size_t, cudaStream_t);
int launch_adain_level(const __half*, int, int, int, const __half*, int, int, int, int, float, float, __half*, void*,
                       size_t, cudaStream_t);
size_t wct_style_state_bytes(int, int);
int launch_wct_style_prepare(const __half*, int, int, int, int, float, float, float, void*, void*, size_t, cudaStream_t);
int launch_wct_apply(const __half*, int, int, int, int, const void*, int, float, float, float, float, int, __half*, int32_t*,
                     void*, size_t, cudaStream_t);
int launch_covariance(const __half*, int, int, int, int, float, float*, float*, cudaStream_t);
int launch_labels_nearest(const uint8_t* src, int N, int Hs, int Ws, int Hd, int Wd, uint8_t* dst, cudaStream_t st);
size_t wct_regions_workspace_bytes(int C, int Nc, int R);
int launch_wct_apply_regions(const __half* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                             const void* const* states, float alpha, float eps_cov, float eps_eig, float thresh, int readd,
                             __half* out, int32_t* k_out, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_adain_regions(const __half* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                         const __half* const* styles, const int* style_hw, float alpha, float eps, __half* out, void* ws,
                         size_t ws_bytes, cudaStream_t st);
int launch_jacobi(float*, int, int, float*, int*, cudaStream_t, const int* skip);
int launch_eig_post(const float*, const float*, float*, int, int, float, float, int, float*, float*, int*, cudaStream_t, const int* skip);
extern int g_conv_bn_override;
extern int g_conv_oversub;
extern int g_conv_fuse;
extern int g_conv_products;
extern int g_conv_tail_tc;
extern int g_conv_head_tc;
int launch_matfun_ns(const float* A, int C, int count, int n_first, float thresh, float eps_eig, float* out, int* ok, int* kcount,
                     cudaStream_t st, float* info);
extern int g_matfun;
extern int g_matfun_max_it;
extern int g_cov_max_stages;
int set_jacobi_tolq(float v);
extern int g_jacobi_lg;
extern int g_jacobi_stagger;

// kernels index elements with 32-bit arithmetic: keep every element count (incl. a 2x upsampled output) below 2^32
static bool geom_ok(int N, int H, int W, int C) {
    return N >= 1 && H >= 2 && W >= 2 && C >= 8 && C % 8 == 0 &&
           (long long)N * (2ll * H + 2) * (2ll * W + 2) * (C / 8) < (1ll << 32) && (long long)H * W < (1ll << 31);
}

}  // namespace wctb

using namespace wctb;

#define ST(s) static_cast<cudaStream_t>(s)
#define HP(p) static_cast<__half*>(p)
#define HCP(p) static_cast<const __half*>(p)

extern "C" {

int wctb200_abi_version(void) { return WCTB200_ABI_VERSION; }
const char* wctb200_last_error(void) { return t_err; }

int wctb200_check_device(void* stream) {
    WCTB_CUDA(cudaStreamSynchronize(ST(stream)));
    unsigned int* w = device_error_word();
    if (!w) {
        set_error("device error word unavailable (no CUDA device?)");
        return WCTB200_ECUDA;
    }
    unsigned int v = 0;
    WCTB_CUDA(cudaMemcpy(&v, w, sizeof(v), cudaMemcpyDeviceToHost));
    if (v != 0) {
        unsigned int zero = 0;
        cudaMemcpy(w, &zero, sizeof(zero), cudaMemcpyHostToDevice);
        set_error("device-side pipeline time-out, code 0x%x (0x1xx producer wait, 0x2xx MMA wait, 0x3xx epilogue wait)", v);
        return WCTB200_EDEVICE;
    }
    return 0;
}

size_t wctb200_act_bytes(int N, int H, int W, int C) {
    if (!geom_ok(N, H, W, C)) return 0;
    ActGeom g(N, H, W, C);
    return (size_t)g.plane * 2 * sizeof(__half);
}

int wctb200_act_from_f32(const float* nhwc, int N, int H, int W, int C, void* act, void* stream) {
    WCTB_REQUIRE(geom_ok(N, H, W, C) && nhwc && act, "act_from_f32: bad arguments");
    return launch_act_from_f32(nhwc, ActGeom(N, H, W, C), HP(act), ST(stream));
}
int wctb200_act_to_f32(const void* act, int N, int H, int W, int C, float* nhwc, void* stream) {
    WCTB_REQUIRE(geom_ok(N, H, W, C) && nhwc && act, "act_to_f32: bad arguments");
    return launch_act_to_f32(HCP(act), ActGeom(N, H, W, C), nhwc, ST(stream));
}

int wctb200_image_u8_to_f32(const uint8_t* img, size_t count, float* out, void* stream) {
    WCTB_REQUIRE(img && out, "image_u8_to_f32: null pointer");
    if (count == 0) return 0;
    return launch_u8_to_f32(img, count, out, ST(stream));
}
int wctb200_image_f32_to_u8(const float* img, size_t count, uint8_t* out, void* stream) {
    WCTB_REQUIRE(img && out, "image_f32_to_u8: null pointer");
    if (count == 0) return 0;
    return launch_f32_to_u8(img, count, out, ST(stream));
}

static bool resize_args_ok(int N, int Hs, int Ws, int C, int Hd, int Wd) {
    return N >= 1 && Hs >= 1 && Ws >= 1 && C >= 1 && C <= 4 && Hd >= 1 && Wd >= 1 && Hs <= (1 << 15) && Ws <= (1 << 15) &&
           Hd <= (1 << 15) && Wd <= (1 << 15);
}
size_t wctb200_resize_workspace_bytes(int N, int Hs, int Ws, int C, int Hd, int Wd, int Wout) {
    if (!resize_args_ok(N, Hs, Ws, C, Hd, Wd) || Wout < 1 || Wout > Wd) return 0;
    return resize_workspace_bytes(N, Hs, Ws, C, Hd, Wd, Wout);
}
int wctb200_resize_bilinear_u8(const uint8_t* src, int N, int Hs, int Ws, int C, int Hd, int Wd, int y0, int x0, int Hout,
                               int Wout, uint8_t* dst, void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(src && dst && ws, "resize_bilinear_u8: null pointer");
    WCTB_REQUIRE(resize_args_ok(N, Hs, Ws, C, Hd, Wd), "resize_bilinear_u8: bad geometry N=%d %dx%dx%d -> %dx%d", N, Hs, Ws, C, Hd, Wd);
    WCTB_REQUIRE(y0 >= 0 && x0 >= 0 && Hout >= 1 && Wout >= 1 && y0 + Hout <= Hd && x0 + Wout <= Wd,
                 "resize_bilinear_u8: window [%d,%d)x[%d,%d) outside %dx%d", y0, y0 + Hout, x0, x0 + Wout, Hd, Wd);
    return launch_resize_u8(src, N, Hs, Ws, C, Hd, Wd, y0, x0, Hout, Wout, dst, ws, ws_bytes, ST(stream));
}
int wctb200_rgb_moments_u8(const uint8_t* img, long long npix, unsigned long long* sums, void* stream) {
    WCTB_REQUIRE(img && sums && npix >= 1 && npix < (1ll << 40), "rgb_moments_u8: bad arguments");
    return launch_rgb_moments(img, npix, sums, ST(stream));
}
int wctb200_coral_apply_u8(const uint8_t* src, long long npix, const double* A, const double* src_mean, const double* src_std,
                           const double* tgt_mean, const double* tgt_std, uint8_t* dst, void* stream) {
    WCTB_REQUIRE(src && dst && A && src_mean && src_std && tgt_mean && tgt_std && npix >= 1, "coral_apply_u8: bad arguments");
    return launch_coral_apply(src, npix, A, src_mean, src_std, tgt_mean, tgt_std, dst, ST(stream));
}

size_t wctb200_conv_weight_bytes(int taps, int Cin, int Cout) {
    if (taps < 1 || Cin < 1 || Cout < 1) return 0;
    return (size_t)2 * taps * Cin * Cout * sizeof(__half) + 256;     // + trailer: the power-of-two scale (layers.cu)
}
int wctb200_prep_conv_weights(const float* w_hwio, int taps, int Cin, int Cout, void* w_split, void* stream) {
    WCTB_REQUIRE(w_hwio && w_split && (taps == 9 || taps == 1) && Cin >= 1 && Cout >= 1, "prep_conv_weights: bad arguments");
    return launch_prep_weights(w_hwio, taps, Cin, Cout, HP(w_split), ST(stream));
}

int wctb200_prep_conv_weights_up2(const float* w_hwio, int Cin, int Cout, void* w_up2, void* stream) {
    WCTB_REQUIRE(w_hwio && w_up2 && Cin >= 1 && Cout >= 1, "prep_conv_weights_up2: bad arguments");
    return launch_prep_weights_up2(w_hwio, Cin, Cout, HP(w_up2), ST(stream));
}

int wctb200_conv3x3(const void* act_in, int N, int H, int W, int Cin, const void* w_split, const float* bias, int Cout,
                    int flags, void* act_out, void* stream) {
    WCTB_REQUIRE(act_in && w_split && act_out, "conv3x3: null pointer");
    WCTB_REQUIRE((flags & ~(WCTB200_RELU | WCTB200_HALO_EDGE | WCTB200_POOL2)) == 0, "conv3x3: unknown flag bits 0x%x", flags);
    return launch_conv_tc(CONV_3X3, HCP(act_in), N, H, W, Cin, HCP(w_split), 1, weight_scale_ptr(HCP(w_split), 9, Cin, Cout),
                          bias, Cout, flags, HP(act_out), ST(stream));
}
int wctb200_conv3x3_up2(const void* act_in, int N, int H, int W, int Cin, const void* w_up2, const float* bias, int Cout,
                        int flags, void* act_out, void* stream) {
    WCTB_REQUIRE(act_in && w_up2 && act_out, "conv3x3_up2: null pointer");
    WCTB_REQUIRE((flags & ~WCTB200_RELU) == 0, "conv3x3_up2: unknown flag bits 0x%x", flags);
    WCTB_REQUIRE(geom_ok(N, 2 * H, 2 * W, Cout), "conv3x3_up2: output geometry too large");
    return launch_conv_tc(CONV_UP2, HCP(act_in), N, H, W, Cin, HCP(w_up2), 1, weight_scale_ptr(HCP(w_up2), 16, Cin, Cout),
                          bias, Cout, flags, HP(act_out), ST(stream));
}
int wctb200_conv3x3_ref(const void* act_in, int N, int H, int W, int Cin, const float* w_hwio, const float* bias, int Cout,
                        int flags, void* act_out, void* stream) {
    WCTB_REQUIRE(act_in && w_hwio && act_out && geom_ok(N, H, W, Cin) && Cout >= 1, "conv3x3_ref: bad arguments");
    return launch_conv3x3_ref(HCP(act_in), ActGeom(N, H, W, Cin), w_hwio, bias, Cout, flags, HP(act_out), ST(stream));
}
int wctb200_conv_head(const float* img, int N, int H, int W, const float* w, const float* b, void* act_out, void* stream) {
    WCTB_REQUIRE(img && w && b && act_out && geom_ok(N, H, W, 64), "conv_head: bad arguments");
    return launch_conv_head(img, N, H, W, w, b, HP(act_out), ST(stream));
}
int wctb200_conv_tail(const void* act_in, int N, int H, int W, int Cin, const float* w, const float* b, int flags,
                      float* img_out, void* stream) {
    WCTB_REQUIRE(act_in && w && b && img_out && geom_ok(N, H, W, Cin) && Cin <= 1024, "conv_tail: bad arguments");
    return launch_conv_tail(HCP(act_in), ActGeom(N, H, W, Cin), w, b, flags, img_out, ST(stream));
}
int wctb200_maxpool2(const void* act_in, int N, int H, int W, int C, void* act_out, void* stream) {
    WCTB_REQUIRE(act_in && act_out && geom_ok(N, H, W, C) && (H + 1) / 2 >= 2 && (W + 1) / 2 >= 2, "maxpool2: bad arguments (output must be >= 2x2)");
    return launch_maxpool2(HCP(act_in), ActGeom(N, H, W, C), HP(act_out), ST(stream));
}
int wctb200_upsample2(const void* act_in, int N, int H, int W, int C, void* act_out, void* stream) {
    WCTB_REQUIRE(act_in && act_out && geom_ok(N, H, W, C), "upsample2: bad arguments");
    return launch_upsample2(HCP(act_in), ActGeom(N, H, W, C), HP(act_out), ST(stream));
}

size_t wctb200_wct_workspace_bytes(int C, int Nc, int Ns) {
    if (C < 8 || Nc < 0 || Ns < 0 || Nc + Ns < 1) return 0;     // Nc = 0 / Ns = 0: style-only / content-only calls
    return wct_workspace_bytes(C, Nc, Ns);
}
int wctb200_wct_level(const void* content, int Nc, int Hc, int Wc, const void* style, int Ns, int Hs, int Ws, int C,
                      float alpha, float eps_cov, float eps_eig, float thresh, int readd_content_mean, void* out,
                      int32_t* k_out, void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(content && style && out && ws, "wct_level: null pointer");
    WCTB_REQUIRE(geom_ok(Nc, Hc, Wc, C) && geom_ok(Ns, Hs, Ws, C), "wct_level: bad geometry");
    return launch_wct_level(HCP(content), Nc, Hc, Wc, HCP(style), Ns, Hs, Ws, C, alpha, eps_cov, eps_eig, thresh,
                            readd_content_mean, HP(out), k_out, ws, ws_bytes, ST(stream));
}
size_t wctb200_wct_style_state_bytes(int C, int Ns) {
    if (C < 8 || Ns < 1) return 0;
    return wct_style_state_bytes(C, Ns);
}
int wctb200_wct_style_prepare(const void* style, int Ns, int Hs, int Ws, int C, float eps_cov, float eps_eig, float thresh,
                              void* state, void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(style && state && ws, "wct_style_prepare: null pointer");
    WCTB_REQUIRE(geom_ok(Ns, Hs, Ws, C), "wct_style_prepare: bad geometry");
    return launch_wct_style_prepare(HCP(style), Ns, Hs, Ws, C, eps_cov, eps_eig, thresh, state, ws, ws_bytes, ST(stream));
}
int wctb200_wct_apply(const void* content, int Nc, int Hc, int Wc, int C, const void* state, int Ns, float alpha,
                      float eps_cov, float eps_eig, float thresh, int readd_content_mean, void* out, int32_t* k_out,
                      void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(content && state && out && ws, "wct_apply: null pointer");
    WCTB_REQUIRE(geom_ok(Nc, Hc, Wc, C), "wct_apply: bad geometry");
    return launch_wct_apply(HCP(content), Nc, Hc, Wc, C, state, Ns, alpha, eps_cov, eps_eig, thresh, readd_content_mean,
                            HP(out), k_out, ws, ws_bytes, ST(stream));
}
int wctb200_adain_level(const void* content, int Nc, int Hc, int Wc, const void* style, int Ns, int Hs, int Ws, int C,
                        float alpha, float eps, void* out, void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(content && style && out && ws, "adain_level: null pointer");
    WCTB_REQUIRE(geom_ok(Nc, Hc, Wc, C) && geom_ok(Ns, Hs, Ws, C), "adain_level: bad geometry");
    return launch_adain_level(HCP(content), Nc, Hc, Wc, HCP(style), Ns, Hs, Ws, C, alpha, eps, HP(out), ws, ws_bytes,
                              ST(stream));
}

int wctb200_labels_resize_nearest(const uint8_t* src, int N, int Hs, int Ws, int Hd, int Wd, uint8_t* dst, void* stream) {
    WCTB_REQUIRE(src && dst, "labels_resize_nearest: null pointer");
    WCTB_REQUIRE(N >= 1 && Hs >= 1 && Ws >= 1 && Hd >= 1 && Wd >= 1 && Hs <= (1 << 15) && Ws <= (1 << 15) && Hd <= (1 << 15) &&
                     Wd <= (1 << 15) && (long long)N * Hd * Wd < (1ll << 40),
                 "labels_resize_nearest: bad geometry N=%d %dx%d -> %dx%d", N, Hs, Ws, Hd, Wd);
    return launch_labels_nearest(src, N, Hs, Ws, Hd, Wd, dst, ST(stream));
}
size_t wctb200_wct_regions_workspace_bytes(int C, int Nc, int R) {
    if (C < 8 || Nc < 1 || R < 1 || R > 8) return 0;
    return wct_regions_workspace_bytes(C, Nc, R);
}
int wctb200_wct_apply_regions(const void* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                              const void* const* states, float alpha, float eps_cov, float eps_eig, float thresh,
                              int readd_content_mean, void* out, int32_t* k_out, void* ws, size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(content && labels && states && out && ws, "wct_apply_regions: null pointer");
    WCTB_REQUIRE(R >= 1 && R <= 8, "wct_apply_regions: R=%d not in 1..8", R);
    WCTB_REQUIRE(geom_ok(Nc, Hc, Wc, C), "wct_apply_regions: bad geometry");
    return launch_wct_apply_regions(HCP(content), Nc, Hc, Wc, C, labels, R, states, alpha, eps_cov, eps_eig, thresh,
                                    readd_content_mean, HP(out), k_out, ws, ws_bytes, ST(stream));
}
int wctb200_adain_regions(const void* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                          const void* const* styles, const int* style_hw, float alpha, float eps, void* out, void* ws,
                          size_t ws_bytes, void* stream) {
    WCTB_REQUIRE(content && labels && styles && style_hw && out && ws, "adain_regions: null pointer");
    WCTB_REQUIRE(R >= 1 && R <= 8, "adain_regions: R=%d not in 1..8", R);
    WCTB_REQUIRE(geom_ok(Nc, Hc, Wc, C), "adain_regions: bad geometry");
    for (int r = 0; r < R; ++r)
        WCTB_REQUIRE(geom_ok(1, style_hw[2 * r], style_hw[2 * r + 1], C), "adain_regions: bad geometry of style %d", r);
    return launch_adain_regions(HCP(content), Nc, Hc, Wc, C, labels, R, reinterpret_cast<const __half* const*>(styles), style_hw,
                                alpha, eps, HP(out), ws, ws_bytes, ST(stream));
}

int wctb200_covariance(const void* act, int N, int H, int W, int C, float eps_cov, float* mean, float* cov, void* stream) {
    WCTB_REQUIRE(act && mean && cov && geom_ok(N, H, W, C), "covariance: bad arguments");
    return launch_covariance(HCP(act), N, H, W, C, eps_cov, mean, cov, ST(stream));
}

int wctb200_jacobi_eigh(float* a, int C, int count, float* sigma, int32_t* sweeps, void* stream) {
    WCTB_REQUIRE(a && sigma && count >= 1, "jacobi_eigh: bad arguments");
    WCTB_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, "jacobi_eigh: C=%d not in {64,128,256,512}", C);
    // scratch: convergence words (16 floats per matrix), a pristine copy of the input (Rayleigh quotients), lambda
    const size_t nmat = (size_t)count * C * C;
    float* scratch = nullptr;
    {
        int rc0 = scratch_alloc(reinterpret_cast<void**>(&scratch), ((size_t)count * 16 + nmat + (size_t)count * C) * sizeof(float), ST(stream), 2);
        if (rc0) return rc0;
    }
    float* conv = scratch;
    float* a0 = scratch + (size_t)count * 16;
    float* lam = a0 + nmat;
    cudaError_t ce = cudaMemcpyAsync(a0, a, nmat * sizeof(float), cudaMemcpyDeviceToDevice, ST(stream));
    int rc = ce == cudaSuccess ? launch_jacobi(a, C, count, conv, sweeps, ST(stream), nullptr) : cuda_fail(ce, "cudaMemcpyAsync");
    if (!rc) rc = launch_eig_post(a, a0, lam, C, count, 0.f, 0.f, count, sigma, nullptr, nullptr, ST(stream), nullptr);
    return rc;
}

size_t wctb200_style_swap_workspace_bytes(int C, int Hc, int Wc, int Hs, int Ws, int patch, int stride) {
    if (!geom_ok(1, Hc, Wc, C) || !geom_ok(1, Hs, Ws, C) || patch < 1 || patch > 16 || stride < 1 || stride > 16 || Hc < patch ||
        Wc < patch || Hs < patch || Ws < patch)
        return 0;
    return style_swap_workspace_bytes(C, Hc, Wc, Hs, Ws, patch, stride);
}
int wctb200_style_swap_level(const void* content, int Hc, int Wc, const void* style, int Hs, int Ws, int C, int patch, int stride,
                             float alpha, float eps_cov, float thresh, void* out, int32_t* k_out, void* ws, size_t ws_bytes,
                             void* stream) {
    WCTB_REQUIRE(content && style && out && ws, "style_swap_level: null pointer");
    WCTB_REQUIRE(geom_ok(1, Hc, Wc, C) && geom_ok(1, Hs, Ws, C), "style_swap_level: bad geometry");
    return launch_style_swap_level(HCP(content), Hc, Wc, HCP(style), Hs, Ws, C, patch, stride, alpha, eps_cov, thresh, HP(out), k_out, ws,
                                   ws_bytes, ST(stream));
}
// tuning hooks (wctb200_debug.h; not part of the stable ABI)
int wctb200_debug_set_conv_bn(int bn) {
    g_conv_bn_override = bn;
    return 0;
}
int wctb200_debug_set_conv_oversub(int k) {
    g_conv_oversub = k < 1 ? 1 : (k > 16 ? 16 : k);
    return g_conv_oversub;
}
int wctb200_debug_set_conv_fuse(int mode) {
    g_conv_fuse = mode < 0 ? -1 : (mode ? 1 : 0);
    return g_conv_fuse;
}
int wctb200_debug_set_jacobi_tolq(float tolq) { return set_jacobi_tolq(tolq); }
int wctb200_debug_set_cov_stages(int n) {
    if (n >= 1 && n <= 12) g_cov_max_stages = n;
    return g_cov_max_stages;
}
int wctb200_debug_matfun(const float* A, int C, int count, int n_first, float thresh, float eps_eig, float* out, int* ok,
                         float* info, void* stream) {
    WCTB_REQUIRE(A && out && ok && count >= 1 && n_first >= 0 && n_first <= count, "debug_matfun: bad arguments");
    const int rc = launch_matfun_ns(A, C, count, n_first, thresh, eps_eig, out, ok, nullptr, ST(stream), info);
    return rc < 0 ? rc : 0;
}
int wctb200_debug_set_matfun(int mode, int max_it) {
    if (mode == 0 || mode == 1) g_matfun = mode;
    if (max_it >= 1 && max_it <= 64) g_matfun_max_it = max_it;
    return g_matfun;
}
int wctb200_debug_set_conv_head_tc(int on) {
    if (on == 0 || on == 1) g_conv_head_tc = on;
    return g_conv_head_tc;
}
int wctb200_debug_set_conv_tail_tc(int on) {
    if (on == 0 || on == 1) g_conv_tail_tc = on;
    return g_conv_tail_tc;
}
int wctb200_debug_set_conv_products(int n) {
    if (n >= 1 && n <= 3) g_conv_products = n;
    return g_conv_products;
}

int wctb200_debug_set_jacobi(int lg_groups, int stagger_cycles) {
    if (lg_groups <= 4) g_jacobi_lg = lg_groups < 0 ? -1 : lg_groups;              // negative: back to the per-size default
    g_jacobi_stagger = stagger_cycles < 0 ? -1 : stagger_cycles;
    return g_jacobi_lg;
}

}  // extern "C"
