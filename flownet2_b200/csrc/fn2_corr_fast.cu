// Fast Correlation path for the FlowNet2 parameter class: MULTIPLY, kernel_size 1, stride_1 1,
// pad == max_displacement, stride_2 | max_displacement  (FlowNet2-C: pad 20, md 20, s2 2 -> 21x21 = 441
// displacements).  Reference: CorrelateData, correlation_layer.cu:46-114 (+ rearrange :24-42).
//
// Design (B200, FP32 SIMT -- the north_star forbids tensor cores for this gather-reduce):
//   * stride_2 = S samples only displacements that are multiples of S, so an output pixel only ever
//     meets map-1 pixels of its own (x mod S, y mod S) parity class.  The problem therefore splits into
//     S*S independent DENSE correlations (radius R = md/S) on the parity sub-grids.  A cheap rearrange
//     pass writes both maps parity-planar:  ws[n][plane][c][ys][xs]   (the reference also rearranges,
//     into zero-padded NHWC, 3.4x larger; here nothing is padded -- TMA zero-fills out-of-bounds).
//   * main kernel: one CTA per (sample, plane, 8x10 sub-grid tile).  A producer warp streams 8-channel
//     chunks of the map-0 tile (8x10) and the map-1 halo tile (28x30) through a 5-stage TMA/mbarrier
//     pipeline.  220 consumer threads (7 warps + the producer warp = 8 warps, 2 per SM sub-partition, so
//     each thread may use up to 255 registers): thread = (4x2 pixel group, halo row j).  For its halo row the
//     thread owns the 21 x-displacements of 8 pixels = 168 FP32 accumulators in registers; per channel it
//     issues 8 LDS.128 (map-0 loads are warp broadcasts) for 168 FFMA, i.e. 5.25 FMA per shared-memory
//     float, which keeps the FMA pipe -- not shared memory -- the limiter.  No cross-thread reduction is
//     needed at all: every (pixel, displacement) sum lives in exactly one thread.
//   * epilogue: divide by C (sumelems, :106-108) and store straight into the strided top view (NCHW for
//     drop-in use, NHWC/concat view inside the engine).
#include <cuda.h>
#include <unordered_map>

#include "fn2_common.cuh"

namespace fn2 {

namespace {

constexpr int TW = 8, TH = 10;      // output tile in sub-grid pixels
constexpr int CC = 8;               // channels per pipeline stage
constexpr int NST = 5;              // pipeline stages
constexpr int PGX = TW / 4, PGY = TH / 2, NPG = PGX * PGY;

template <int R> struct Geo {
    static constexpr int D = 2 * R + 1;
    static constexpr int WIN = ((4 + 2 * R + 3) / 4) * 4;          // map-1 window floats per thread (mult. of 4)
    static constexpr int BW = ((TW + 2 * R + 3) / 4) * 4;          // halo tile width (36 for R=10)
    static constexpr int BH = TH + 2 * R;                          // halo tile height (26)
    static constexpr int ROWS = 2 * R + 2;                         // halo rows (threads) per pixel group
    static constexpr int CONSUMERS = NPG * ROWS;                   // 264
    static constexpr int THREADS = ((CONSUMERS + 31) / 32) * 32 + 32;   // + producer warp
    static constexpr int A_STAGE = CC * TH * TW;                   // floats
    static constexpr int B_STAGE = CC * BH * BW;
    static constexpr int STAGE_BYTES = (A_STAGE + B_STAGE) * 4;
    static constexpr int SMEM = NST * STAGE_BYTES + 1024;
};

// ---- PTX helpers (mbarrier + TMA), see blackwell_cuda_programming.md Guideline 15 ----------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) break;
        if (++spins > (1u << 24)) __trap();       // never hang the GPU: a lost arrival becomes a launch error
    }
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

struct FastP {
    int N, C, H, W;          // bottoms
    int S;                   // stride_2
    int Hs, Ws;              // sub-grid extent (ceil(H/S), ceil(W/S))
    int tiles_x, tiles_y;
};

template <int R>
__global__ void __launch_bounds__(Geo<R>::THREADS, 1)
corr_fast_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, T4 top, FastP p) {
    using G = Geo<R>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* stage_mem = reinterpret_cast<float*>(smem_raw);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + NST * G::STAGE_BYTES);
    uint64_t* empty_bar = full_bar + NST;

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    // tile decode: blockIdx.x = ((n*S*S + plane) * tiles_y + ty) * tiles_x + tx
    int bid = blockIdx.x;
    const int tx = bid % p.tiles_x; bid /= p.tiles_x;
    const int ty = bid % p.tiles_y; bid /= p.tiles_y;
    const int nplane = bid;                      // n*S*S + plane
    const int plane = nplane % (p.S * p.S);
    const int n = nplane / (p.S * p.S);
    const int py = plane / p.S, px = plane % p.S;
    const int xs0 = tx * TW, ys0 = ty * TH;

    constexpr int NCW = (G::CONSUMERS + 31) / 32;          // consumer warps
    if (tid == 0) {
        for (int s = 0; s < NST; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], NCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int nchunks = p.C / CC;
    if (warp == NCW) {
        // ===== producer warp: one elected lane issues the TMA loads =====
        if ((tid & 31) == 0) {
            for (int it = 0; it < nchunks; it++) {
                const int s = it % NST;
                const uint32_t ph = (uint32_t)(it / NST) & 1u;
                mbar_wait(&empty_bar[s], ph ^ 1u);
                float* a_dst = stage_mem + (size_t)s * (G::A_STAGE + G::B_STAGE);
                float* b_dst = a_dst + G::A_STAGE;
                mbar_expect_tx(&full_bar[s], (uint32_t)G::STAGE_BYTES);
                tma_load_4d(a_dst, &mapA, &full_bar[s], xs0, ys0, it * CC, nplane);
                tma_load_4d(b_dst, &mapB, &full_bar[s], xs0 - R + (R % 4), ys0 - R, it * CC, nplane);
            }
        }
        return;
    }
    // ===== consumers =====  (the few padding lanes of the last consumer warp run the same code on a
    // non-existent pixel group -- all their shared-memory reads stay inside the stage -- and store nothing)
    const bool real_thread = tid < G::CONSUMERS;
    const int pg = tid / G::ROWS;                 // pixel group
    const int jj = tid % G::ROWS;                 // halo row relative to the group's first pixel row
    const int xg = pg % PGX, yp = pg / PGX;
    const int y0 = yp * 2;                        // tile-local pixel rows y0, y0+1
    const int j = y0 + jj;                        // tile-local halo row (0 .. BH-1)

    float acc0[4][G::D], acc1[4][G::D];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int d = 0; d < G::D; d++) { acc0[i][d] = 0.f; acc1[i][d] = 0.f; }

    const int a_off0 = y0 * TW + 4 * xg;
    const int b_off = j * G::BW + 4 * xg;

    for (int it = 0; it < nchunks; it++) {
        const int s = it % NST;
        const uint32_t ph = (uint32_t)(it / NST) & 1u;
        mbar_wait(&full_bar[s], ph);
        const float* as = stage_mem + (size_t)s * (G::A_STAGE + G::B_STAGE);
        const float* bs = as + G::A_STAGE;
#pragma unroll 2
        for (int c = 0; c < CC; c++) {
            const float4 a0v = *reinterpret_cast<const float4*>(as + c * (TH * TW) + a_off0);
            const float4 a1v = *reinterpret_cast<const float4*>(as + c * (TH * TW) + a_off0 + TW);
            const float a0[4] = {a0v.x, a0v.y, a0v.z, a0v.w};
            const float a1[4] = {a1v.x, a1v.y, a1v.z, a1v.w};
            const float4* brow = reinterpret_cast<const float4*>(bs + c * (G::BH * G::BW) + b_off);
#pragma unroll
            for (int q = 0; q < G::WIN / 4; q++) {
                const float4 bq = brow[q];
                const float bv[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int w = 4 * q + e;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int d = w - i;
                        if (d >= 0 && d < G::D) {
                            acc0[i][d] = fmaf(a0[i], bv[e], acc0[i][d]);
                            acc1[i][d] = fmaf(a1[i], bv[e], acc1[i][d]);
                        }
                    }
                }
            }
        }
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&empty_bar[s]);
    }

    // ===== epilogue =====
    const float sumelems = (float)p.C;                       // kernel_size == 1 (correlation_layer.cu:106)
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const int pr = jj - r;                               // p + R for pixel row y0 + r
        if (!real_thread || pr < 0 || pr >= G::D) continue;
        const int ys = ys0 + y0 + r;
        const int y = ys * p.S + py;
        if (ys >= p.Hs || y >= p.H) continue;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int xs = xs0 + 4 * xg + i;
            const int x = xs * p.S + px;
            if (xs >= p.Ws || x >= p.W) continue;
            float* o = top.p + top.off(n, pr * G::D, y, x);
#pragma unroll
            for (int d = 0; d < G::D; d++) o[d * top.sc] = (r == 0 ? acc0[i][d] : acc1[i][d]) / sumelems;
        }
    }
}

// ---- rearrange: strided (n,c,h,w) view -> parity-planar ws[n][plane][c][Hs][Ws] ------------------------
// `shift` empty columns precede every row of the map-1 planes: TMA needs the innermost start coordinate
// of a box to be 16-byte aligned (measured: tools/tma_probe.cu), and the halo starts at xs0 - R, so the
// planes are stored shifted by R mod 4 columns and the halo box starts at xs0 - R + shift = 0 (mod 4).
// channel-fast (NHWC) source: 32 channels x 32 pixels tiles through shared memory (writes real pixels
// only; corr_zero_pads_kernel clears the pad columns/rows).
__global__ void corr_zero_pads_kernel(float* __restrict__ ws, int rows_total, int S, int C, int Hs, int Ws, int shift,
                                      int H, int W) {
    // one thread per plane row
    for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < rows_total; row += gridDim.x * blockDim.x) {
        const int ys = row % Hs;
        const int plane = (row / (Hs * C)) % (S * S);
        const int py = plane / S, px = plane % S;
        const int w_true = (W - px + S - 1) / S;                 // real pixels of this parity class per row
        const bool row_real = ys * S + py < H;
        float* r = ws + (size_t)row * Ws;
        for (int x = 0; x < Ws; x++)
            if (!row_real || x < shift || x >= shift + w_true) r[x] = 0.f;
    }
}
__global__ void corr_rearrange_cfast_kernel(T4 in, float* __restrict__ ws, int S, int Hs, int Ws, int shift) {
    __shared__ float tile[32][33];                           // [x][c]
    const int n = blockIdx.z / in.h, y = blockIdx.z % in.h;
    const int x0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x;
    for (int jx = threadIdx.y; jx < 32; jx += blockDim.y)
        if (x0 + jx < in.w && c0 + tx < in.c) tile[jx][tx] = in.p[in.off(n, c0 + tx, y, x0 + jx)];
    __syncthreads();
    const int x = x0 + tx;
    if (x >= in.w) return;
    const int plane = (y % S) * S + (x % S);
    const size_t plane_sz = (size_t)Hs * Ws;
    float* dst = ws + (((size_t)n * S * S + plane) * in.c) * plane_sz + (size_t)(y / S) * Ws + (x / S) + shift;
    for (int jc = threadIdx.y; jc < 32; jc += blockDim.y)
        if (c0 + jc < in.c) dst[(size_t)(c0 + jc) * plane_sz] = tile[tx][jc];
}
// any other layout (NCHW drop-in): one thread per workspace element, x fastest.
__global__ void corr_rearrange_generic_kernel(T4 in, float* __restrict__ ws, int S, int Hs, int Ws, int shift) {
    const long long total = (long long)in.n * S * S * in.c * Hs * Ws;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int xs = (int)(idx % Ws);
        long long r = idx / Ws;
        const int ys = (int)(r % Hs); r /= Hs;
        const int c = (int)(r % in.c); r /= in.c;
        const int plane = (int)(r % (S * S));
        const int n = (int)(r / (S * S));
        const int y = ys * S + plane / S, x = (xs - shift) * S + plane % S;
        ws[idx] = (xs >= shift && y < in.h && x < in.w) ? in.p[in.off(n, c, y, x)] : 0.f;
    }
}

int make_map(CUtensorMap* m, float* base, int Ws, int Hs, int C, int NP, int bw, int bh) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return FN2_ERR_CUDA; }
    cuuint64_t dims[4] = {(cuuint64_t)Ws, (cuuint64_t)Hs, (cuuint64_t)C, (cuuint64_t)NP};
    cuuint64_t strides[3] = {(cuuint64_t)Ws * 4, (cuuint64_t)Ws * Hs * 4, (cuuint64_t)Ws * Hs * C * 4};
    cuuint32_t box[4] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)CC, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return FN2_ERR_CUDA; }
    return FN2_OK;
}

int sub_extent(int v, int S) { return (v + S - 1) / S; }
int ws_width(int W, int S, int shift) { return (sub_extent(W, S) + shift + 3) / 4 * 4; }     // 16-byte row pitch for TMA

template <int R>
int launch(const T4& b0, const T4& b1, const T4& top, int S, float* ws, cudaStream_t st) {
    using G = Geo<R>;
    FastP p;
    p.N = b0.n; p.C = b0.c; p.H = b0.h; p.W = b0.w; p.S = S;
    constexpr int SHIFT = R % 4;                    // see corr_zero_pads_kernel
    p.Hs = sub_extent(b0.h, S); p.Ws = sub_extent(b0.w, S);
    p.tiles_x = (p.Ws + TW - 1) / TW;
    p.tiles_y = (p.Hs + TH - 1) / TH;
    const int pitch[2] = {ws_width(b0.w, S, 0), ws_width(b0.w, S, SHIFT)};
    const int shift[2] = {0, SHIFT};
    const size_t rows = (size_t)p.N * S * S * p.C * p.Hs;
    float* dst[2] = {ws, ws + rows * pitch[0]};
    const T4* src[2] = {&b0, &b1};
    for (int k = 0; k < 2; k++) {
        const bool pads = (b0.w % S) || (b0.h % S) || pitch[k] != p.Ws;
        if (src[k]->sc == 1) {
            if (pads) {
                corr_zero_pads_kernel<<<ew_grid((long long)rows, 256), 256, 0, st>>>(dst[k], (int)rows, S, p.C, p.Hs, pitch[k],
                                                                                   shift[k], b0.h, b0.w);
                FN2_LAUNCH_CHECK();
            }
            dim3 grid((src[k]->w + 31) / 32, (src[k]->c + 31) / 32, src[k]->n * src[k]->h);
            corr_rearrange_cfast_kernel<<<grid, dim3(32, 8), 0, st>>>(*src[k], dst[k], S, p.Hs, pitch[k], shift[k]);
        } else {
            corr_rearrange_generic_kernel<<<ew_grid((long long)(rows * pitch[k]), 256), 256, 0, st>>>(*src[k], dst[k], S, p.Hs,
                                                                                                     pitch[k], shift[k]);
        }
        FN2_LAUNCH_CHECK();
    }
    CUtensorMap mapA, mapB;
    int rc = make_map(&mapA, dst[0], pitch[0], p.Hs, p.C, p.N * S * S, TW, TH);
    if (rc) return rc;
    rc = make_map(&mapB, dst[1], pitch[1], p.Hs, p.C, p.N * S * S, G::BW, G::BH);
    if (rc) return rc;
    static bool attr_set = false;
    if (!attr_set) {
        FN2_CUDA(cudaFuncSetAttribute(corr_fast_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM));
        attr_set = true;
    }
    const int grid = p.N * S * S * p.tiles_x * p.tiles_y;
    corr_fast_kernel<R><<<grid, G::THREADS, G::SMEM, st>>>(mapA, mapB, top, p);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

}  // namespace

int corr_fast_eligible(const T4& b0, const T4& b1, const T4& top, int pad, int k, int md, int s1, int s2, int type) {
    if (type != 0 || k != 1 || s1 != 1 || pad != md || s2 < 1 || md % s2) return 0;
    const int R = md / s2;
    if (R != 10 && R != 4) return 0;                   // instantiated radii
    if (b0.c % CC) return 0;
    if ((long long)b0.n * s2 * s2 > 65535LL * 1024) return 0;
    (void)b1; (void)top;
    return 1;
}

int corr_fast_workspace(int N, int C, int H, int W, int md, int s2, size_t* bytes) {
    const int R = md / s2;
    *bytes = (size_t)N * s2 * s2 * C * sub_extent(H, s2) * (ws_width(W, s2, 0) + ws_width(W, s2, R % 4)) * sizeof(float);
    return FN2_OK;
}

int corr_fast_forward(const T4& b0, const T4& b1, const T4& top, int md, int s2, void* ws, size_t ws_bytes, cudaStream_t st) {
    size_t need = 0;
    corr_fast_workspace(b0.n, b0.c, b0.h, b0.w, md, s2, &need);
    if (ws_bytes < need) { set_error("correlation: workspace too small"); return FN2_ERR_WORKSPACE; }
    if (((uintptr_t)ws & 127) != 0) { set_error("correlation: workspace must be 128-byte aligned"); return FN2_ERR_INVALID; }
    const int R = md / s2;
    if (R == 10) return launch<10>(b0, b1, top, s2, (float*)ws, st);
    if (R == 4) return launch<4>(b0, b1, top, s2, (float*)ws, st);
    set_error("corr_fast: radius %d not instantiated", R);
    return FN2_ERR_INVALID;
}

}  // namespace fn2
