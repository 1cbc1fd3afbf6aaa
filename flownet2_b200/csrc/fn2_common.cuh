// Shared device/host helpers for libfn2.so kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <mutex>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/fn2.h"

namespace fn2 {

// Thread-local last error + launch counter (fn2_last_error / fn2_launch_count).
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define FN2_CHECK_ARG(cond, ...)                     \
    do {                                             \
        if (!(cond)) {                               \
            ::fn2::set_error(__VA_ARGS__);           \
            return FN2_ERR_INVALID;                  \
        }                                            \
    } while (0)

#define FN2_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) {                                                   \
            ::fn2::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                   \
            return FN2_ERR_CUDA;                                                    \
        }                                                                           \
    } while (0)

#define FN2_LAUNCH_CHECK()                                                          \
    do {                                                                            \
        ::fn2::count_launch();                                                      \
        cudaError_t e__ = cudaGetLastError();                                       \
        if (e__ != cudaSuccess) {                                                   \
            ::fn2::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                             __FILE__, __LINE__);                                   \
            return FN2_ERR_CUDA;                                                    \
        }                                                                           \
    } while (0)

// Device-side view of fn2_tensor (passed by value to kernels).
struct T4 {
    float* p;
    int n, c, h, w;
    long long sn, sc, sh, sw;
    __host__ __device__ __forceinline__ long long off(int in, int ic, int ih, int iw) const {
        return in * sn + ic * sc + ih * sh + iw * sw;
    }
    __host__ __device__ __forceinline__ long long count() const { return (long long)n * c * h * w; }
    __host__ __device__ bool is_nchw() const {
        return sw == 1 && sh == w && sc == (long long)h * w && sn == (long long)c * h * w;
    }
    // channel-contiguous ("NHWC") with arbitrary pixel stride sw >= c
    __host__ __device__ bool is_nhwc() const {
        return sc == 1 && sh == (long long)w * sw && sn == (long long)h * w * sw;
    }
};

inline T4 view(const fn2_tensor* t) {
    T4 v;
    v.p = t->data; v.n = t->n; v.c = t->c; v.h = t->h; v.w = t->w;
    v.sn = t->sn; v.sc = t->sc; v.sh = t->sh; v.sw = t->sw;
    return v;
}
inline bool same_dims(const T4& a, const T4& b) {
    return a.n == b.n && a.c == b.c && a.h == b.h && a.w == b.w;
}
inline bool valid(const fn2_tensor* t) {
    return t && t->data && t->n > 0 && t->c > 0 && t->h > 0 && t->w > 0;
}

inline int num_sms() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}
// cuTensorMapEncodeTiled, looked up once from the driver (the runtime API has no wrapper); nullptr if the driver lacks it.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    });
    return fn;
}
// Grid for grid-stride elementwise kernels: enough CTAs to cover, capped at a multiple of the
// SM count (148 SMs x 8 resident 256-thread CTAs).
inline int ew_grid(long long total, int block) {
    long long need = (total + block - 1) / block;
    long long cap = (long long)num_sms() * 8;
    return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

}  // namespace fn2
