// Convolution / Deconvolution forward with fused bias + leaky ReLU -- FP32 SIMT engine.
//
// Reference: ConvolutionLayer::Forward_gpu conv_layer.cu:8-23 (per-sample im2col + cublasSgemm,
// base_conv_layer.cpp:326-349, separate bias GEMM :351-356), DeconvolutionLayer::Forward_gpu
// deconv_layer.cu:8-23 (GEMM + col2im), ReLUForward relu_layer.cu:9-14.
//
// Here: one implicit-GEMM kernel over the whole batch (M = N*Ho*Wo output pixels, N = Co,
// K = kh*kw*Ci), no materialised col buffer, bias and ReLU applied in the epilogue.  This is the
// exact-FP32 engine (`engine: CAFFE` in the prototxt, fn2_conv_desc.engine == 1) and the fallback
// for shapes the tcgen05 engine (fn2_conv_tc.cu) does not take (tiny Ci / Co).
//
// Packed weight layout (built once at load time by fn2_conv_pack_weights):
//   Wp[k][co], k = (r*kw + s)*ci_stride + ci, rows for padded channels ci >= Ci are zero.
#include "fn2_common.cuh"

namespace fn2 {

int conv_tc_eligible(const fn2_conv_desc* d, const T4& in, const T4& out);
int conv_tc_forward(const fn2_conv_desc* d, const T4& in, const float* wp, const float* bias,
                    const T4& out, float* ws, size_t ws_floats, cudaStream_t st);
size_t conv_tc_workspace_floats(const fn2_conv_desc* d, int N, int Ho, int Wo);
int conv_tc_plan(const fn2_conv_desc* d, int N, int Ho, int Wo, int ci_stride, int* out8);
int conv_tc_packed_floats(const fn2_conv_desc* d, int ci_stride, size_t* floats);
int conv_tc_pack(const fn2_conv_desc* d, int ci_stride, const float* w, float* wp, cudaStream_t st);
int conv_nhwc_eligible(const fn2_conv_desc* d, const T4& in, const T4& out);
size_t conv_nhwc_workspace_floats(const fn2_conv_desc* d, int N, int Ho, int Wo);
int conv_nhwc_forward(const fn2_conv_desc* d, const T4& in, const float* wp, const float* bias, const T4& out,
                      float* ws, size_t ws_floats, cudaStream_t st);

struct ConvP {
    int Ci, Co, kh, kw, sh, sw, ph, pw;
    int H, W, Ho, Wo, N;
    int cis;          // ci_stride used in the packed-weight k index
    int K;            // kh*kw*cis
    int relu, has_bias;
    float slope;
};

// k -> (r, s, ci); returns false when the k row is a padded channel or beyond K
__device__ __forceinline__ bool decode_k(const ConvP& p, int k, int& r, int& s, int& ci) {
    if (k >= p.K) return false;
    ci = k % p.cis;
    const int rs = k / p.cis;
    s = rs % p.kw;
    r = rs / p.kw;
    return ci < p.Ci;
}

// Input coordinate for output (oy, ox) and tap (r, s).  Convolution: iy = oy*sh - ph + r.
// Deconvolution (gather form of col2im, util/im2col.cpp:158-190): oy = iy*sh - ph + r, so
// iy = (oy + ph - r)/sh when divisible.
template <bool DECONV>
__device__ __forceinline__ bool in_coord(const ConvP& p, int oy, int ox, int r, int s, int& iy, int& ix) {
    if (!DECONV) {
        iy = oy * p.sh - p.ph + r;
        ix = ox * p.sw - p.pw + s;
    } else {
        const int ty = oy + p.ph - r, tx = ox + p.pw - s;
        if (ty < 0 || tx < 0 || (ty % p.sh) || (tx % p.sw)) return false;
        iy = ty / p.sh;
        ix = tx / p.sw;
    }
    return iy >= 0 && iy < p.H && ix >= 0 && ix < p.W;
}

constexpr int BM = 128, BN = 128, BK = 16;

// 256 threads, 8x8 outputs per thread arranged as 2x2 blocks of 4x4 (rows ty*4 + {0,64},
// cols tx*4 + {0,64}) so that shared-memory float4 reads are conflict free.
template <bool DECONV>
__global__ void __launch_bounds__(256) conv_igemm_kernel(T4 in, const float* __restrict__ wp,
                                                         const float* __restrict__ bias, T4 out, ConvP p) {
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Bs[2][BK][BN];
    const int tid = threadIdx.x;
    const long long M = (long long)p.N * p.Ho * p.Wo;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;

    // A loader: thread owns k_local = tid % 16 and rows m_local = tid/16 + 16*i
    const int a_k = tid & 15;
    const int a_m = tid >> 4;
    int a_n[8], a_oy[8], a_ox[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const long long m = m0 + a_m + 16 * i;
        if (m < M) {
            a_ox[i] = (int)(m % p.Wo);
            a_oy[i] = (int)((m / p.Wo) % p.Ho);
            a_n[i] = (int)(m / ((long long)p.Wo * p.Ho));
        } else {
            a_n[i] = -1; a_oy[i] = 0; a_ox[i] = 0;
        }
    }
    // B loader: rows k = tid/32 + 8*i (i=0,1), cols (tid%32)*4 .. +3
    const int b_k = tid >> 5;
    const int b_n = (tid & 31) * 4;

    float a_reg[8];
    float4 b_reg[2];
    auto load_tiles = [&](int k0) {
        int r, s, ci;
        const bool kv = decode_k(p, k0 + a_k, r, s, ci);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            float v = 0.f;
            int iy, ix;
            if (kv && a_n[i] >= 0 && in_coord<DECONV>(p, a_oy[i], a_ox[i], r, s, iy, ix))
                v = __ldg(in.p + in.off(a_n[i], ci, iy, ix));
            a_reg[i] = v;
        }
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const int k = k0 + b_k + 8 * i;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < p.K) {
                const float* src = wp + (long long)k * p.Co + n0 + b_n;
                if (n0 + b_n + 3 < p.Co && ((p.Co & 3) == 0)) {
                    v = __ldg(reinterpret_cast<const float4*>(src));
                } else {
                    if (n0 + b_n + 0 < p.Co) v.x = __ldg(src + 0);
                    if (n0 + b_n + 1 < p.Co) v.y = __ldg(src + 1);
                    if (n0 + b_n + 2 < p.Co) v.z = __ldg(src + 2);
                    if (n0 + b_n + 3 < p.Co) v.w = __ldg(src + 3);
                }
            }
            b_reg[i] = v;
        }
    };
    auto store_tiles = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 8; i++) As[buf][a_k][a_m + 16 * i] = a_reg[i];
#pragma unroll
        for (int i = 0; i < 2; i++) *reinterpret_cast<float4*>(&Bs[buf][b_k + 8 * i][b_n]) = b_reg[i];
    };

    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

    const int ktiles = (p.K + BK - 1) / BK;
    load_tiles(0);
    store_tiles(0);
    __syncthreads();
    for (int kt = 0; kt < ktiles; kt++) {
        const int buf = kt & 1;
        if (kt + 1 < ktiles) load_tiles((kt + 1) * BK);
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4 + 64]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4 + 64]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 8; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kt + 1 < ktiles) {
            store_tiles(buf ^ 1);
            __syncthreads();
        }
    }

    // epilogue: bias (base_conv_layer.cpp:351-356) + ReLU (relu_layer.cu:9-14)
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const long long m = m0 + ty * 4 + (i & 3) + (i >> 2) * 64;
        if (m >= M) continue;
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float* orow = out.p + out.off(n, 0, oy, ox);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int co = n0 + tx * 4 + (j & 3) + (j >> 2) * 64;
            if (co >= p.Co) continue;
            float v = acc[i][j];
            if (p.has_bias) v += __ldg(bias + co);
            if (p.relu) v = v > 0 ? v : v * p.slope;
            orow[co * out.sc] = v;
        }
    }
}

// Small-Co path (flow predictors: Co = 2): one warp per output pixel, lanes stride K, shuffle
// reduce.  Avoids padding Co to a 128-wide tile.
template <bool DECONV, int CO>
__global__ void __launch_bounds__(256) conv_smallco_kernel(T4 in, const float* __restrict__ wp,
                                                           const float* __restrict__ bias, T4 out, ConvP p) {
    const long long M = (long long)p.N * p.Ho * p.Wo;
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long m = warp0; m < M; m += nwarps) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float acc[CO];
#pragma unroll
        for (int j = 0; j < CO; j++) acc[j] = 0.f;
        for (int rs = 0; rs < p.kh * p.kw; rs++) {
            const int r = rs / p.kw, s = rs % p.kw;
            int iy, ix;
            if (!in_coord<DECONV>(p, oy, ox, r, s, iy, ix)) continue;
            const float* ip = in.p + in.off(n, 0, iy, ix);
            const float* wr = wp + (long long)rs * p.cis * p.Co;
            for (int ci = lane; ci < p.Ci; ci += 32) {
                const float a = __ldg(ip + ci * in.sc);
#pragma unroll
                for (int j = 0; j < CO; j++)
                    if (j < p.Co) acc[j] = fmaf(a, __ldg(wr + (long long)ci * p.Co + j), acc[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < CO; j++)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < CO; j++) {
                if (j >= p.Co) break;
                float v = acc[j];
                if (p.has_bias) v += __ldg(bias + j);
                if (p.relu) v = v > 0 ? v : v * p.slope;
                out.p[out.off(n, j, oy, ox)] = v;
            }
        }
    }
}

// Tiny path (Co <= 4 and Ci <= 32: flow upsamplers 2->2, full-resolution flow predictors): one thread per
// output pixel, all weights staged in shared memory.
template <bool DECONV>
__global__ void __launch_bounds__(256) conv_tiny_kernel(T4 in, const float* __restrict__ wp,
                                                        const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float wsm[];                    // [kh*kw][Ci][Co]
    const int nw = p.kh * p.kw * p.Ci * p.Co;
    for (int i = threadIdx.x; i < nw; i += blockDim.x) wsm[i] = wp[i];
    __syncthreads();
    const long long M = (long long)p.N * p.Ho * p.Wo;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int r = 0; r < p.kh; r++)
            for (int s = 0; s < p.kw; s++) {
                int iy, ix;
                if (!in_coord<DECONV>(p, oy, ox, r, s, iy, ix)) continue;
                const float* ip = in.p + in.off(n, 0, iy, ix);
                const float* w = wsm + (r * p.kw + s) * p.Ci * p.Co;
                for (int ci = 0; ci < p.Ci; ci++) {
                    const float a = __ldg(ip + ci * in.sc);
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (j < p.Co) acc[j] = fmaf(a, w[ci * p.Co + j], acc[j]);
                }
            }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j >= p.Co) break;
            float v = acc[j];
            if (p.has_bias) v += __ldg(bias + j);
            if (p.relu) v = v > 0 ? v : v * p.slope;
            out.p[out.off(n, j, oy, ox)] = v;
        }
    }
}

// Flow predictors (Co == 2, NHWC input): the layers are memory bound (a few MFLOP per MB), so the kernels below read
// every input pixel as float4 vectors and keep the [tap][ci] weight pairs in shared memory.
//   conv_pf_thread_kernel: Ci <= 32 (full-resolution fusion predictors) -- one thread per output pixel
//   conv_pf_warp_kernel:   larger Ci -- one warp per output pixel, lanes stride the channel vectors, shuffle reduce
// Channels [Ci, 4*C4) are blob padding: their weights are zero (the padding itself is finite, the arena is zero-filled).
__device__ __forceinline__ void pf_stage_weights(float2* wsm, const float* __restrict__ wp, int taps, int Ci, int C4) {
    const int cp = C4 * 4;
    for (int i = threadIdx.x; i < taps * cp; i += blockDim.x) {
        const int ci = i % cp, t = i / cp;
        wsm[i] = ci < Ci ? make_float2(wp[((long long)t * Ci + ci) * 2], wp[((long long)t * Ci + ci) * 2 + 1]) : make_float2(0.f, 0.f);
    }
    __syncthreads();
}
__device__ __forceinline__ void pf_store(const T4& out, const ConvP& p, const float* __restrict__ bias, int n, int oy, int ox, float a0, float a1) {
    if (p.has_bias) { a0 += __ldg(bias); a1 += __ldg(bias + 1); }
    if (p.relu) { a0 = a0 > 0 ? a0 : a0 * p.slope; a1 = a1 > 0 ? a1 : a1 * p.slope; }
    out.p[out.off(n, 0, oy, ox)] = a0;
    out.p[out.off(n, 1, oy, ox)] = a1;
}
template <int C4>
__global__ void __launch_bounds__(256) conv_pf_thread_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float2 pf_wsm[];
    pf_stage_weights(pf_wsm, wp, p.kh * p.kw, p.Ci, C4);
    const long long M = (long long)p.N * p.Ho * p.Wo;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float a0 = 0.f, a1 = 0.f;
        for (int r = 0; r < p.kh; r++) {
            const int iy = oy * p.sh - p.ph + r;
            if (iy < 0 || iy >= p.H) continue;
            for (int s = 0; s < p.kw; s++) {
                const int ix = ox * p.sw - p.pw + s;
                if (ix < 0 || ix >= p.W) continue;
                const float4* ip = reinterpret_cast<const float4*>(in.p + in.off(n, 0, iy, ix));
                const float4* w = reinterpret_cast<const float4*>(pf_wsm + (r * p.kw + s) * C4 * 4);
#pragma unroll
                for (int q = 0; q < C4; q++) {
                    const float4 a = __ldg(ip + q);
                    const float4 w01 = w[2 * q], w23 = w[2 * q + 1];       // (c0.o0, c0.o1, c1.o0, c1.o1), (c2.., c3..)
                    a0 = fmaf(a.x, w01.x, a0); a1 = fmaf(a.x, w01.y, a1);
                    a0 = fmaf(a.y, w01.z, a0); a1 = fmaf(a.y, w01.w, a1);
                    a0 = fmaf(a.z, w23.x, a0); a1 = fmaf(a.z, w23.y, a1);
                    a0 = fmaf(a.w, w23.z, a0); a1 = fmaf(a.w, w23.w, a1);
                }
            }
        }
        pf_store(out, p, bias, n, oy, ox, a0, a1);
    }
}
__global__ void __launch_bounds__(256) conv_pf_warp_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p, int C4) {
    extern __shared__ float2 pf_wsm[];
    pf_stage_weights(pf_wsm, wp, p.kh * p.kw, p.Ci, C4);
    const long long M = (long long)p.N * p.Ho * p.Wo;
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long m = warp0; m < M; m += nwarps) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float a0 = 0.f, a1 = 0.f;
        for (int r = 0; r < p.kh; r++) {
            const int iy = oy * p.sh - p.ph + r;
            if (iy < 0 || iy >= p.H) continue;
            for (int s = 0; s < p.kw; s++) {
                const int ix = ox * p.sw - p.pw + s;
                if (ix < 0 || ix >= p.W) continue;
                const float4* ip = reinterpret_cast<const float4*>(in.p + in.off(n, 0, iy, ix));
                const float4* w = reinterpret_cast<const float4*>(pf_wsm + (long long)(r * p.kw + s) * C4 * 4);
#pragma unroll 2
                for (int q = lane; q < C4; q += 32) {
                    const float4 a = __ldg(ip + q);
                    const float4 w01 = w[2 * q], w23 = w[2 * q + 1];
                    a0 = fmaf(a.x, w01.x, a0); a1 = fmaf(a.x, w01.y, a1);
                    a0 = fmaf(a.y, w01.z, a0); a1 = fmaf(a.y, w01.w, a1);
                    a0 = fmaf(a.z, w23.x, a0); a1 = fmaf(a.z, w23.y, a1);
                    a0 = fmaf(a.w, w23.z, a0); a1 = fmaf(a.w, w23.w, a1);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a0 += __shfl_xor_sync(0xffffffffu, a0, o);
            a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        }
        if (lane == 0) pf_store(out, p, bias, n, oy, ox, a0, a1);
    }
}

// 3x3 / stride 1 specialisations of the two flow-predictor kernels (every predict_flow layer of FlowNet2): compile-time tap
// loops so that the loads of a kernel row are in flight together.
template <int C4>
__global__ void __launch_bounds__(256) conv_pf3_thread_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float2 pf_wsm[];
    pf_stage_weights(pf_wsm, wp, 9, p.Ci, C4);
    const long long M = (long long)p.N * p.Ho * p.Wo;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const int iy = oy - p.ph + r;
            if (iy < 0 || iy >= p.H) continue;
            float4 a[3][C4];
#pragma unroll
            for (int s = 0; s < 3; s++) {
                const int ix = ox - p.pw + s;
                const bool ok = ix >= 0 && ix < p.W;
                const float4* ip = reinterpret_cast<const float4*>(in.p + in.off(n, 0, iy, ok ? ix : ox));
#pragma unroll
                for (int q = 0; q < C4; q++) a[s][q] = ok ? __ldg(ip + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int s = 0; s < 3; s++) {
                const float4* w = reinterpret_cast<const float4*>(pf_wsm + (r * 3 + s) * C4 * 4);
#pragma unroll
                for (int q = 0; q < C4; q++) {
                    const float4 w01 = w[2 * q], w23 = w[2 * q + 1];
                    a0 = fmaf(a[s][q].x, w01.x, a0); a1 = fmaf(a[s][q].x, w01.y, a1);
                    a0 = fmaf(a[s][q].y, w01.z, a0); a1 = fmaf(a[s][q].y, w01.w, a1);
                    a0 = fmaf(a[s][q].z, w23.x, a0); a1 = fmaf(a[s][q].z, w23.y, a1);
                    a0 = fmaf(a[s][q].w, w23.z, a0); a1 = fmaf(a[s][q].w, w23.w, a1);
                }
            }
        }
        pf_store(out, p, bias, n, oy, ox, a0, a1);
    }
}
// Shared-memory tiled variant of the thread-per-pixel predictor for Ci <= 32: a block of 256 threads produces a 32 x 8 output
// tile from a 34 x 10 input halo that is fetched with fully coalesced 128-bit loads (the direct version reads 64..128-byte
// pixels at a 64..128-byte lane stride: 16 L1 wavefronts per load instruction).  Same accumulation order, bit-identical.
template <int C4>
__global__ void __launch_bounds__(256) conv_pf3_tile_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float2 pf_wsm[];
    constexpr int TW = 32, TH = 8, HW = TW + 2, HH = TH + 2, PS = C4 + 1;         // PS: pixel stride in float4 (odd: no bank conflicts)
    float4* tile = reinterpret_cast<float4*>(pf_wsm + 9 * C4 * 4);                 // [HH][HW][PS]
    pf_stage_weights(pf_wsm, wp, 9, p.Ci, C4);
    const int tiles_x = (p.Wo + TW - 1) / TW, tiles_y = (p.Ho + TH - 1) / TH;
    const int ntiles = p.N * tiles_x * tiles_y;
    const int tx = threadIdx.x % TW, ty = threadIdx.x / TW;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int bx = t % tiles_x, by = (t / tiles_x) % tiles_y, n = t / (tiles_x * tiles_y);
        const int x0 = bx * TW - p.pw, y0 = by * TH - p.ph;
        __syncthreads();                                                             // previous tile fully consumed
        for (int i = threadIdx.x; i < HH * HW * C4; i += 256) {
            const int q = i % C4, px_ = (i / C4) % HW, py_ = i / (C4 * HW);
            const int ix = x0 + px_, iy = y0 + py_;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ix >= 0 && ix < p.W && iy >= 0 && iy < p.H) v = __ldg(reinterpret_cast<const float4*>(in.p + in.off(n, 0, iy, ix)) + q);
            tile[(py_ * HW + px_) * PS + q] = v;
        }
        __syncthreads();
        const int ox = bx * TW + tx, oy = by * TH + ty;
        if (ox >= p.Wo || oy >= p.Ho) continue;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int r = 0; r < 3; r++) {
            if (oy - p.ph + r < 0 || oy - p.ph + r >= p.H) continue;                 // same skipping as the direct kernel
#pragma unroll
            for (int s_ = 0; s_ < 3; s_++) {
                const float4* a = tile + ((ty + r) * HW + tx + s_) * PS;
                const float4* w = reinterpret_cast<const float4*>(pf_wsm + (r * 3 + s_) * C4 * 4);
#pragma unroll
                for (int q = 0; q < C4; q++) {
                    const float4 v = a[q];
                    const float4 w01 = w[2 * q], w23 = w[2 * q + 1];
                    a0 = fmaf(v.x, w01.x, a0); a1 = fmaf(v.x, w01.y, a1);
                    a0 = fmaf(v.y, w01.z, a0); a1 = fmaf(v.y, w01.w, a1);
                    a0 = fmaf(v.z, w23.x, a0); a1 = fmaf(v.z, w23.y, a1);
                    a0 = fmaf(v.w, w23.z, a0); a1 = fmaf(v.w, w23.w, a1);
                }
            }
        }
        pf_store(out, p, bias, n, oy, ox, a0, a1);
    }
}

// one warp per PX = 4 consecutive output pixels of a row: the 6 input columns and the weights of a kernel row are loaded
// once for the four of them (shared memory bandwidth for the weights was the limit of the one-pixel version)
__global__ void __launch_bounds__(256) conv_pf3_warp_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p, int C4) {
    extern __shared__ float2 pf_wsm[];
    pf_stage_weights(pf_wsm, wp, 9, p.Ci, C4);
    constexpr int PX = 4;
    const int gx = (p.Wo + PX - 1) / PX;
    const long long G = (long long)p.N * p.Ho * gx;
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long g = warp0; g < G; g += nwarps) {
        const int ox0 = (int)(g % gx) * PX;
        const int oy = (int)((g / gx) % p.Ho);
        const int n = (int)(g / ((long long)gx * p.Ho));
        float acc[PX][2];
#pragma unroll
        for (int j = 0; j < PX; j++) { acc[j][0] = 0.f; acc[j][1] = 0.f; }
        // per-row base pointers and column validity once per group (the address arithmetic used to be repeated per load)
        const float4* rowp[3];
        bool rowok[3], colok[PX + 2];
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const int iy = oy - p.ph + r;
            rowok[r] = iy >= 0 && iy < p.H;
            rowp[r] = reinterpret_cast<const float4*>(in.p + in.off(n, 0, rowok[r] ? iy : 0, 0));
        }
#pragma unroll
        for (int c = 0; c < PX + 2; c++) { const int ix = ox0 - p.pw + c; colok[c] = ix >= 0 && ix < p.W; }
        const long long px4 = in.sw / 4;                                   // pixel stride in float4
        const long long col0 = (long long)(ox0 - p.pw) * px4;
        for (int q = lane; q < C4; q += 32) {
#pragma unroll
            for (int r = 0; r < 3; r++) {
                if (!rowok[r]) continue;
                float4 a[PX + 2];
#pragma unroll
                for (int c = 0; c < PX + 2; c++)
                    a[c] = colok[c] ? __ldg(rowp[r] + col0 + c * px4 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int s = 0; s < 3; s++) {
                    const float4* w = reinterpret_cast<const float4*>(pf_wsm + (long long)(r * 3 + s) * C4 * 4);
                    const float4 w01 = w[2 * q], w23 = w[2 * q + 1];
#pragma unroll
                    for (int j = 0; j < PX; j++) {
                        const float4 v = a[j + s];
                        acc[j][0] = fmaf(v.x, w01.x, acc[j][0]); acc[j][1] = fmaf(v.x, w01.y, acc[j][1]);
                        acc[j][0] = fmaf(v.y, w01.z, acc[j][0]); acc[j][1] = fmaf(v.y, w01.w, acc[j][1]);
                        acc[j][0] = fmaf(v.z, w23.x, acc[j][0]); acc[j][1] = fmaf(v.z, w23.y, acc[j][1]);
                        acc[j][0] = fmaf(v.w, w23.z, acc[j][0]); acc[j][1] = fmaf(v.w, w23.w, acc[j][1]);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < PX; j++)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                acc[j][0] += __shfl_xor_sync(0xffffffffu, acc[j][0], o);
                acc[j][1] += __shfl_xor_sync(0xffffffffu, acc[j][1], o);
            }
        if (lane < PX && ox0 + lane < p.Wo) {
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int j = 0; j < PX; j++) if (lane == j) { a0 = acc[j][0]; a1 = acc[j][1]; }
            pf_store(out, p, bias, n, oy, ox0 + lane, a0, a1);
        }
    }
}

// Flow upsamplers (Deconvolution 4x4, stride 2, Ci, Co <= 4): an output pixel is reached by exactly the 2x2 taps whose parity
// matches, so only those are visited (conv_tiny_kernel<true> tests all 16).  Same tap and channel order as the generic kernel,
// hence bit-identical results.
__global__ void __launch_bounds__(256) deconv_s2_tiny_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float wsm[];                    // [kh*kw][Ci][Co]
    const int nw = p.kh * p.kw * p.Ci * p.Co;
    for (int i = threadIdx.x; i < nw; i += blockDim.x) wsm[i] = wp[i];
    __syncthreads();
    const long long M = (long long)p.N * p.Ho * p.Wo;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(m % p.Wo);
        const int oy = (int)((m / p.Wo) % p.Ho);
        const int n = (int)(m / ((long long)p.Wo * p.Ho));
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const int ty = oy + p.ph, tx = ox + p.pw;
        for (int r = ty & 1; r < p.kh; r += 2) {
            const int iy = (ty - r) >> 1;
            if (ty - r < 0 || iy >= p.H) continue;
            for (int s_ = tx & 1; s_ < p.kw; s_ += 2) {
                const int ix = (tx - s_) >> 1;
                if (tx - s_ < 0 || ix >= p.W) continue;
                const float* ip = in.p + in.off(n, 0, iy, ix);
                const float* w = wsm + (r * p.kw + s_) * p.Ci * p.Co;
                for (int ci = 0; ci < p.Ci; ci++) {
                    const float a = __ldg(ip + ci * in.sc);
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (j < p.Co) acc[j] = fmaf(a, w[ci * p.Co + j], acc[j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j >= p.Co) break;
            float v = acc[j];
            if (p.has_bias) v += __ldg(bias + j);
            if (p.relu) v = v > 0 ? v : v * p.slope;
            out.p[out.off(n, j, oy, ox)] = v;
        }
    }
}

// Caffe weights -> packed [k][co].  conv: w[co][ci][r][s]; deconv: w[ci][co][r][s].
__global__ void pack_weights_kernel(const float* __restrict__ w, float* __restrict__ wp, int Ci, int Co,
                                    int kh, int kw, int cis, int deconv) {
    const long long total = (long long)kh * kw * cis * Co;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int co = (int)(idx % Co);
        const long long k = idx / Co;
        const int ci = (int)(k % cis);
        const int rs = (int)(k / cis);
        const int s = rs % kw, r = rs / kw;
        float v = 0.f;
        if (ci < Ci)
            v = deconv ? w[(((long long)ci * Co + co) * kh + r) * kw + s]
                       : w[(((long long)co * Ci + ci) * kh + r) * kw + s];
        wp[idx] = v;
    }
}

// Few input channels, many output channels (the gradient operator of the 2-channel predict_flow convolutions: 2 -> 194 .. 1026):
// K = taps * Ci is tiny, the layer is a pure store stream.  Lanes = output channels (coalesced weight reads and stores), the
// input patch of FEW_PX consecutive output pixels sits in shared memory and is broadcast.
constexpr int FEW_PX = 16;
__global__ void __launch_bounds__(256) conv_fewci_kernel(T4 in, const float* __restrict__ wp, const float* __restrict__ bias, T4 out, ConvP p) {
    extern __shared__ float sIn[];                            // [FEW_PX][K]
    const int K = p.kh * p.kw * p.Ci;
    const int xt = (p.Wo + FEW_PX - 1) / FEW_PX;
    const int ox0 = (blockIdx.x % xt) * FEW_PX;
    const int oy = (blockIdx.x / xt) % p.Ho, n = blockIdx.x / (xt * p.Ho);
    for (int e = threadIdx.x; e < FEW_PX * K; e += blockDim.x) {
        const int px = e / K, k = e % K;
        const int ci = k % p.Ci, tap = k / p.Ci;
        const int iy = oy * p.sh + tap / p.kw - p.ph, ix = (ox0 + px) * p.sw + tap % p.kw - p.pw;
        sIn[e] = (ox0 + px < p.Wo && iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) ? in.p[in.off(n, ci, iy, ix)] : 0.f;
    }
    __syncthreads();
    for (int co = threadIdx.x; co < p.Co; co += blockDim.x) {
        float acc[FEW_PX];
        const float b = p.has_bias ? bias[co] : 0.f;
#pragma unroll
        for (int px = 0; px < FEW_PX; px++) acc[px] = b;
        for (int k = 0; k < K; k++) {
            const float w = __ldg(wp + (long long)k * p.Co + co);
#pragma unroll
            for (int px = 0; px < FEW_PX; px++) acc[px] = fmaf(w, sIn[px * K + k], acc[px]);
        }
#pragma unroll
        for (int px = 0; px < FEW_PX; px++)
            if (ox0 + px < p.Wo) {
                float v = acc[px];
                if (p.relu) v = v > 0.f ? v : v * p.slope;
                out.p[out.off(n, co, oy, ox0 + px)] = v;
            }
    }
}

static int make_params(const fn2_conv_desc* d, const T4& in, const T4& out, ConvP* p) {
    FN2_CHECK_ARG(d->ci > 0 && d->co > 0 && d->kh > 0 && d->kw > 0 && d->stride_h > 0 && d->stride_w > 0 &&
                  d->pad_h >= 0 && d->pad_w >= 0 && d->out_pad_h >= 0 && d->out_pad_w >= 0 && (d->deconv || (!d->out_pad_h && !d->out_pad_w)),
                  "conv: bad descriptor");
    FN2_CHECK_ARG(in.c == d->ci, "conv: bottom has %d channels, descriptor says %d", in.c, d->ci);
    int Ho, Wo;
    int rc = fn2_conv_out_shape(d, in.h, in.w, &Ho, &Wo);
    if (rc) return rc;
    FN2_CHECK_ARG(out.n == in.n && out.c == d->co && out.h == Ho && out.w == Wo,
                  "conv: top must be (%d,%d,%d,%d), got (%d,%d,%d,%d)", in.n, d->co, Ho, Wo, out.n, out.c, out.h, out.w);
    p->Ci = d->ci; p->Co = d->co; p->kh = d->kh; p->kw = d->kw; p->sh = d->stride_h; p->sw = d->stride_w;
    p->ph = d->pad_h; p->pw = d->pad_w; p->H = in.h; p->W = in.w; p->Ho = Ho; p->Wo = Wo; p->N = in.n;
    p->relu = d->relu; p->has_bias = d->has_bias; p->slope = d->negative_slope;
    return FN2_OK;
}

}  // namespace fn2

using namespace fn2;

extern "C" {

int fn2_conv_out_shape(const fn2_conv_desc* d, int H, int W, int* Ho, int* Wo) {
    FN2_CHECK_ARG(d && Ho && Wo, "conv_out_shape: null argument");
    if (!d->deconv) {
        *Ho = (H + 2 * d->pad_h - d->kh) / d->stride_h + 1;      // conv_layer.cpp:8-22 (dilation 1)
        *Wo = (W + 2 * d->pad_w - d->kw) / d->stride_w + 1;
    } else {
        *Ho = d->stride_h * (H - 1) + d->kh - 2 * d->pad_h + d->out_pad_h;      // deconv_layer.cpp:18-19 (+ 0 there)
        *Wo = d->stride_w * (W - 1) + d->kw - 2 * d->pad_w + d->out_pad_w;
    }
    FN2_CHECK_ARG(*Ho >= 1 && *Wo >= 1, "conv: empty output (%d x %d)", *Ho, *Wo);
    return FN2_OK;
}

// ci_stride: for the SIMT engine the k index uses the real Ci (no padded rows); the argument is
// what the tcgen05 engine needs (padded channel count of the bottom tensor).
int fn2_conv_packed_floats(const fn2_conv_desc* d, int ci_stride, size_t* floats) {
    FN2_CHECK_ARG(d && floats, "conv_packed_floats: null argument");
    size_t simt = (size_t)d->kh * d->kw * d->ci * d->co;
    size_t tc = 0;
    int rc = conv_tc_packed_floats(d, ci_stride, &tc);
    if (rc) return rc;
    *floats = simt + tc;
    return FN2_OK;
}

int fn2_conv_pack_weights(const fn2_conv_desc* d, int ci_stride, const float* caffe_weights_dev,
                          float* packed_dev, void* stream) {
    FN2_CHECK_ARG(d && caffe_weights_dev && packed_dev, "conv_pack_weights: null argument");
    const long long total = (long long)d->kh * d->kw * d->ci * d->co;
    pack_weights_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)stream>>>(
        caffe_weights_dev, packed_dev, d->ci, d->co, d->kh, d->kw, d->ci, d->deconv);
    FN2_LAUNCH_CHECK();
    return conv_tc_pack(d, ci_stride, caffe_weights_dev, packed_dev + total, (cudaStream_t)stream);
}

int fn2_conv_plan(const fn2_conv_desc* d, int N, int H, int W, int ci_stride, int32_t* plan8) {
    FN2_CHECK_ARG(d && plan8, "conv_plan: null argument");
    int Ho, Wo;
    int rc = fn2_conv_out_shape(d, H, W, &Ho, &Wo);
    if (rc) return rc;
    conv_tc_plan(d, N, Ho, Wo, ci_stride, plan8);
    return FN2_OK;
}

int fn2_conv_workspace_bytes(const fn2_conv_desc* d, int N, int H, int W, size_t* bytes) {
    FN2_CHECK_ARG(d && bytes, "conv_workspace_bytes: null argument");
    int Ho, Wo;
    int rc = fn2_conv_out_shape(d, H, W, &Ho, &Wo);
    if (rc) return rc;
    *bytes = max(conv_nhwc_workspace_floats(d, N, Ho, Wo), conv_tc_workspace_floats(d, N, Ho, Wo)) * sizeof(float);
    return FN2_OK;
}

int fn2_conv_forward(const fn2_conv_desc* d, const fn2_tensor* bottom, const float* packed_weights_dev,
                     const float* bias_dev, const fn2_tensor* top, void* workspace, size_t workspace_bytes,
                     void* stream) {
    FN2_CHECK_ARG(d && valid(bottom) && valid(top) && packed_weights_dev, "conv: null argument");
    FN2_CHECK_ARG(!d->has_bias || bias_dev, "conv: bias_term set but no bias given");
    T4 in = view(bottom), out = view(top);
    ConvP p;
    int rc = make_params(d, in, out, &p);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const long long simt_floats = (long long)d->kh * d->kw * d->ci * d->co;
    if (d->engine != 1 && conv_tc_eligible(d, in, out))
        return conv_tc_forward(d, in, packed_weights_dev + simt_floats, bias_dev, out, (float*)workspace, workspace_bytes / sizeof(float), st);
    FN2_CHECK_ARG(d->engine != 2, "conv: tcgen05 engine requested but the shape/layout is not eligible");
    if (!d->deconv && d->ci <= 4 && d->co >= 32 && out.sc == 1 && d->kh * d->kw * d->ci <= 200) {
        p.cis = d->ci;
        const int xt = (p.Wo + FEW_PX - 1) / FEW_PX;
        const size_t smem = (size_t)FEW_PX * d->kh * d->kw * d->ci * sizeof(float);
        conv_fewci_kernel<<<(unsigned)(p.N * p.Ho * xt), 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);
        FN2_LAUNCH_CHECK();
        return FN2_OK;
    }
    if (conv_nhwc_eligible(d, in, out))
        return conv_nhwc_forward(d, in, packed_weights_dev, bias_dev, out, (float*)workspace, workspace_bytes / sizeof(float), st);
    p.cis = d->ci;
    p.K = d->kh * d->kw * p.cis;
    const long long M = (long long)p.N * p.Ho * p.Wo;
    const int C4 = (d->ci + 3) / 4;
    const bool pf_ok = !d->deconv && d->co == 2 && in.sc == 1 && in.sw >= 4 * C4 && !((uintptr_t)in.p & 15) && !(in.sw & 3) &&
                       !(in.sh & 3) && !(in.sn & 3) && (size_t)d->kh * d->kw * C4 * 4 * sizeof(float2) <= 200 * 1024;
    if (pf_ok) {
        const size_t smem = (size_t)d->kh * d->kw * C4 * 4 * sizeof(float2);
        const bool k3 = d->kh == 3 && d->kw == 3 && d->stride_h == 1 && d->stride_w == 1;
        if (C4 <= 8) {
            const int grid = (int)min((long long)num_sms() * 8, (M + 255) / 256);
#define FN2_PF_THREAD(C)                                                                                                   \
            case C: if (k3 && d->pad_h == 1 && d->pad_w == 1) {                                                            \
                        const size_t tsm = smem + (size_t)10 * 34 * (C + 1) * sizeof(float4);                               \
                        const int tgrid = (int)min((long long)num_sms() * 4, (long long)p.N * ((p.Wo + 31) / 32) * ((p.Ho + 7) / 8)); \
                        if (tsm > 48 * 1024) FN2_CUDA(cudaFuncSetAttribute(conv_pf3_tile_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm)); \
                        conv_pf3_tile_kernel<C><<<tgrid, 256, tsm, st>>>(in, packed_weights_dev, bias_dev, out, p);            \
                    } else if (k3) conv_pf3_thread_kernel<C><<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);  \
                    else conv_pf_thread_kernel<C><<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);      \
                    break;
            switch (C4) { FN2_PF_THREAD(1) FN2_PF_THREAD(2) FN2_PF_THREAD(3) FN2_PF_THREAD(4) FN2_PF_THREAD(5) FN2_PF_THREAD(6)
                          FN2_PF_THREAD(7) FN2_PF_THREAD(8) }
#undef FN2_PF_THREAD
        } else {
            static size_t smem_set = 0;
            if (smem > 48 * 1024 && smem > smem_set) {
                FN2_CUDA(cudaFuncSetAttribute(conv_pf_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
                FN2_CUDA(cudaFuncSetAttribute(conv_pf3_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
                smem_set = 200 * 1024;
            }
            const int per_sm = (int)max((size_t)1, min((size_t)8, (size_t)(220 * 1024) / (smem + 1024)));
            if (k3) {
                const long long groups = (long long)p.N * p.Ho * ((p.Wo + 3) / 4);
                const int grid = (int)min((long long)num_sms() * per_sm, (groups + 7) / 8);
                conv_pf3_warp_kernel<<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p, C4);
            } else {
                const int grid = (int)min((long long)num_sms() * per_sm, (M + 7) / 8);
                conv_pf_warp_kernel<<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p, C4);
            }
        }
    } else if (d->co <= 4 && d->ci <= 32) {
        const size_t smem = (size_t)p.K * p.Co * sizeof(float);
        const int grid = ew_grid(M, 256);
        if (d->deconv && d->stride_h == 2 && d->stride_w == 2) deconv_s2_tiny_kernel<<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);
        else if (d->deconv) conv_tiny_kernel<true><<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);
        else           conv_tiny_kernel<false><<<grid, 256, smem, st>>>(in, packed_weights_dev, bias_dev, out, p);
    } else if (d->co <= 4) {
        const int grid = ew_grid(M * 32, 256);
        if (d->deconv) conv_smallco_kernel<true, 4><<<grid, 256, 0, st>>>(in, packed_weights_dev, bias_dev, out, p);
        else           conv_smallco_kernel<false, 4><<<grid, 256, 0, st>>>(in, packed_weights_dev, bias_dev, out, p);
    } else {
        dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((d->co + BN - 1) / BN));
        if (d->deconv) conv_igemm_kernel<true><<<grid, 256, 0, st>>>(in, packed_weights_dev, bias_dev, out, p);
        else           conv_igemm_kernel<false><<<grid, 256, 0, st>>>(in, packed_weights_dev, bias_dev, out, p);
    }
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

}  // extern "C"
