// Correlation backward (2-D and 1-D, MULTIPLY and SUBTRACT) and the Correlation1D forward.
//
// Reference: CorrelateDataBackward0/1 (correlation_layer.cu:118-249), ...Subtract (:298-427), correlation_layer1d.cu:48-420.
// The reference launches one thread per bottom element that walks all displacements and, inside, the range of top positions
// whose patch covers the element.  Here the adjoint is FACTORISED instead (the patch walk does not depend on the channel):
//
//   G[n, d, q]   = sum over the k x k patch taps (j, i) with (q - tap - (md - pad)) divisible by stride_1 and inside the top
//                  of topdiff[n, d, y, x]                                  -- "patch sum", bottom resolution, channel-free
//   d bottom0[q] = 1/(k*k*C) * sum_d G[d, q]          * M[q + disp(d)]     M = bottom1            (MULTIPLY)
//   d bottom1[q] = 1/(k*k*C) * sum_d G[d, q - disp(d)] * M'[q - disp(d)]   M' = bottom0           (MULTIPLY)
//   SUBTRACT uses the reference's sign map in place of M / M': s(q) = (bottom0[q] >= bottom1[q]) ? +1 : -1 evaluated AT THE
//   DISPLACED position for both gradients (:327-329, :397-399), +s for bottom0 and -s for bottom1, and +-1 (not 0) outside
//   the image, because the reference compares its two zero-padded copies there.
// For FlowNet2-C's layer (k = 1, stride_1 = 1, pad = md) G is topdiff itself.  The apply step is one shared-memory tiled kernel:
// an 8 x 8 pixel tile keeps its G rows (64 x D floats) resident and streams the (8 + 2*reach)^2 halo of M in 8-channel chunks;
// thread = (pixel, 2 channels), D fused multiply-adds per chunk and channel, fixed summation order (no atomics).
#include "fn2_common.cuh"

namespace fn2 {

namespace {

constexpr int CB_TILE = 8;                 // tile edge (pixels)
constexpr int CB_CH = 8;                   // channels per chunk

struct CbP {
    int N, C, H, W;                        // bottom shape
    int D;                                 // displacements (top channels)
    int topH, topW;
    int k, s1, md, pad;                    // patch walk
    int ypatch_off;                        // (md - pad) vertically; 0 for Correlation1D rows (no vertical displacement border)
    int reach_y, reach_x;                  // max |dy|, |dx| over the displacement table
    int identity_g;                        // G == topdiff (k == 1, s1 == 1, offsets 0, top size == bottom size)
    float scale, oob;                      // 1 / (k*k*C); value of M outside the image
    short dy[441], dx[441];
};

// patch sum: G[n][q][d] (d fastest) = sum of topdiff[n][d][y][x] over the top positions whose patch covers q
__global__ void corr_patchsum_kernel(T4 td, float* __restrict__ g, CbP p) {
    const long long total = (long long)p.N * p.H * p.W * p.D;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int d = (int)(idx % p.D);
        long long r = idx / p.D;
        const int xx = (int)(r % p.W); r /= p.W;
        const int yy = (int)(r % p.H);
        const int n = (int)(r / p.H);
        float acc = 0.f;
        for (int j = 0; j < p.k; j++) {
            const int ty = yy - j - p.ypatch_off;                      // = y * s1
            if (ty < 0 || ty % p.s1) continue;
            const int y = ty / p.s1;
            if (y >= p.topH) continue;
            for (int i = 0; i < p.k; i++) {
                const int tx = xx - i - (p.md - p.pad);
                if (tx < 0 || tx % p.s1) continue;
                const int x = tx / p.s1;
                if (x >= p.topW) continue;
                acc += td.p[td.off(n, d, y, x)];
            }
        }
        g[idx] = acc;
    }
}

// sign map of the SUBTRACT gradients
__global__ void corr_sign_kernel(T4 a, T4 b, float* __restrict__ s) {
    const long long total = a.count();
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % a.c);
        long long r = idx / a.c;
        const int x = (int)(r % a.w); r /= a.w;
        const int y = (int)(r % a.h);
        const int n = (int)(r / a.h);
        s[idx] = a.p[a.off(n, c, y, x)] >= b.p[b.off(n, c, y, x)] ? 1.f : -1.f;
    }
}

// MODE 0: out[q] = scale * sum_d G[q][d] * M[q + disp(d)]        (gradient w.r.t. bottom0)
// MODE 1: out[q] = scale * sum_d G[q - disp(d)][d] * M[q - disp(d)]   (gradient w.r.t. bottom1), M already carries its sign
// G: dense [N][H][W][D] or (identity_g) the top diff tensor itself; M: strided view, channel-fast or not.
template <int MODE>
__global__ void __launch_bounds__(256) corr_apply_kernel(const float* __restrict__ gdense, T4 td, T4 m, T4 out, CbP p, float msign) {
    extern __shared__ float sm[];
    const int hw = CB_TILE + 2 * p.reach_x, hh = CB_TILE + 2 * p.reach_y;
    float* gs = sm;                                        // [64][D]
    float* hs = sm + 64 * p.D;                             // [hh][hw][CB_CH]
    const int tiles_x = (p.W + CB_TILE - 1) / CB_TILE, tiles_y = (p.H + CB_TILE - 1) / CB_TILE;
    const int tid = threadIdx.x;
    const int px = tid >> 2, cg = tid & 3;                 // pixel 0..63, channel pair 0..3
    const int ty_ = px >> 3, tx_ = px & 7;
    for (int tile = blockIdx.x; tile < p.N * tiles_y * tiles_x; tile += gridDim.x) {
        const int n = tile / (tiles_y * tiles_x);
        const int t2 = tile - n * tiles_y * tiles_x;
        const int y0 = (t2 / tiles_x) * CB_TILE, x0 = (t2 % tiles_x) * CB_TILE;
        __syncthreads();
        // G rows of the tile: gs[pixel][d]
        for (int idx = tid; idx < 64 * p.D; idx += 256) {
            const int q = idx / p.D, d = idx - q * p.D;
            int y = y0 + (q >> 3), x = x0 + (q & 7);
            if (MODE == 1) { y -= p.dy[d]; x -= p.dx[d]; }
            float v = 0.f;
            if (y >= 0 && y < p.H && x >= 0 && x < p.W) {
                if (y0 + (q >> 3) < p.H && x0 + (q & 7) < p.W)
                    v = p.identity_g ? td.p[td.off(n, d, y, x)] : gdense[(((long long)n * p.H + y) * p.W + x) * p.D + d];
            }
            gs[idx] = v;
        }
        const int y = y0 + ty_, x = x0 + tx_;
        for (int c0 = 0; c0 < p.C; c0 += CB_CH) {
            __syncthreads();
            for (int idx = tid; idx < hh * hw * CB_CH; idx += 256) {
                const int c = idx % CB_CH, hpix = idx / CB_CH;
                const int hy = hpix / hw, hx = hpix - hy * hw;
                const int yy = y0 - p.reach_y + hy, xx = x0 - p.reach_x + hx;
                float v = 0.f;
                if (c0 + c < p.C) v = (yy >= 0 && yy < p.H && xx >= 0 && xx < p.W) ? msign * m.p[m.off(n, c0 + c, yy, xx)] : p.oob * msign;
                hs[idx] = v;
            }
            __syncthreads();
            float a0 = 0.f, a1 = 0.f;
            const float* grow = gs + px * p.D;
            const float* hbase = hs + ((ty_ + p.reach_y) * hw + (tx_ + p.reach_x)) * CB_CH + 2 * cg;
#pragma unroll 4
            for (int d = 0; d < p.D; d++) {
                const int off = (MODE == 0 ? 1 : -1) * ((int)p.dy[d] * hw + (int)p.dx[d]) * CB_CH;
                const float g = grow[d];
                const float2 v = *reinterpret_cast<const float2*>(hbase + off);
                a0 = fmaf(g, v.x, a0);
                a1 = fmaf(g, v.y, a1);
            }
            if (y < p.H && x < p.W) {
                const int c = c0 + 2 * cg;
                if (c < p.C) out.p[out.off(n, c, y, x)] = a0 * p.scale;
                if (c + 1 < p.C) out.p[out.off(n, c + 1, y, x)] = a1 * p.scale;
            }
        }
    }
}

// Correlation1D forward (correlation_layer1d.cu:48-112): displacement in x only, rows are not padded; one warp per output
// pixel and displacement group, lanes over channels, shuffle reduction (fixed order).
__global__ void __launch_bounds__(128) corr1d_fwd_kernel(T4 b0, T4 b1, T4 top, int pad, int k, int md, int s1, int s2, int x_shift, int type) {
    extern __shared__ float patch[];                  // [k*k][C]
    const int x = blockIdx.x, y = blockIdx.y, n = blockIdx.z;
    const int C = b0.c, H = b0.h, W = b0.w;
    const int x1 = x * s1 + md - pad, y1 = y * s1;     // upper-left of the patch, unpadded coordinates (:56-57)
    for (int idx = threadIdx.x; idx < k * k * C; idx += blockDim.x) {
        const int ch = idx % C, ji = idx / C;
        const int yy = y1 + ji / k, xx = x1 + ji % k;
        patch[idx] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? b0.p[b0.off(n, ch, yy, xx)] : 0.f;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sumelems = k * k * C;
    for (int tc = warp; tc < top.c; tc += 4) {
        const int s2o = (tc + x_shift) * s2;             // :83
        float acc = 0.f;
        for (int j = 0; j < k; j++) {
            const int yy = y1 + j;
            for (int i = 0; i < k; i++) {
                const int xx = x1 + s2o + i;
                const bool inb = yy >= 0 && yy < H && xx >= 0 && xx < W;
                const float* ap = patch + (j * k + i) * C;
                for (int ch = lane; ch < C; ch += 32) {
                    const float b = inb ? b1.p[b1.off(n, ch, yy, xx)] : 0.f;
                    acc += type == 0 ? ap[ch] * b : fabsf(ap[ch] - b);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) top.p[top.off(n, tc, y, x)] = acc / (float)sumelems;
    }
}

// ---- fast path: FlowNet2-C's layer (MULTIPLY, k = 1, stride_1 = 1, pad = md, R = md / stride_2 = 10, C % 32 == 0) ----------------
// out[q][c] = scale * sum over (dj, di) of Gx[q][dj][di] * M[q + SGN * (dj - R, di - R) * stride_2][c]
//   bottom0 gradient: Gx = top diff, M = bottom1, SGN = +1
//   bottom1 gradient: Gx = the top diff SHIFTED per displacement (corr_shift_kernel: Gx[q][d] = topdiff[q - disp(d)][d]), M = bottom0, SGN = -1
// A displacement only connects pixels of the same stride_2 parity class, so a work unit is (sample, parity class, 8 x 16 tile of
// that class's plane, 32 channels): the (8 + 2R) x (16 + 2R) plane-pixel halo of M sits in shared memory (129 KB), the tile's Gx
// values of one displacement row (128 x 21) are re-staged per dj.  Thread = 4 consecutive pixels x 4 channels: a halo float4 is
// loaded once and feeds up to 4 pixels (pixel i meets it with di = t - i), the pixel's 21 Gx values of the row live in registers:
// 336 FMAs per 24 + 24 128-bit shared loads.  Fixed summation order (dj, then the halo column), no atomics.
constexpr int CF_R = 10, CF_DW = 2 * CF_R + 1, CF_TH = 8, CF_TW = 16, CF_HH = CF_TH + 2 * CF_R, CF_HW = CF_TW + 2 * CF_R, CF_GROW = 24;
constexpr int CF_GB = 3;                                  // displacement rows staged per step (Gx values prefetched one step ahead)
constexpr int CF_GSTAGE = CF_GB * CF_TH * CF_TW * CF_GROW; // floats per stage
constexpr int CF_SMEM = (CF_HH * CF_HW * 32 + CF_GSTAGE) * (int)sizeof(float);
static_assert(CF_DW % CF_GB == 0 && CF_GSTAGE % 256 == 0, "stage shape");

struct CfP { int N, C, H, W, S, tiles_x, tiles_y, cchunks; float scale; };

template <int SGN>
__global__ void __launch_bounds__(256, 1) corr_bwd_fast_kernel(T4 g, T4 m, T4 out, CfP p) {
    extern __shared__ __align__(16) float cfsm[];
    float* halo = cfsm;                                   // [HH * HW][32]
    float* gs = cfsm + CF_HH * CF_HW * 32;                // [128][GROW]
    const int tid = threadIdx.x;
    const int cg = tid & 7, pg = tid >> 3;                // channel float4 0..7, pixel group 0..31
    const int row = pg >> 2, xg = pg & 3;                 // tile row 0..7, group of 4 pixels 0..3
    const int units = p.N * p.S * p.S * p.tiles_y * p.tiles_x * p.cchunks;
    for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
        int r = unit;
        const int cc = r % p.cchunks; r /= p.cchunks;
        const int tx = r % p.tiles_x; r /= p.tiles_x;
        const int ty = r % p.tiles_y; r /= p.tiles_y;
        const int cls = r % (p.S * p.S), n = r / (p.S * p.S);
        const int py = cls / p.S, px = cls % p.S;
        const int u0 = ty * CF_TH, v0 = tx * CF_TW, c0 = cc * 32;
        __syncthreads();
        for (int idx = tid; idx < CF_HH * CF_HW * 8; idx += 256) {
            const int hp = idx >> 3, c4 = idx & 7;
            const int hy = hp / CF_HW, hx = hp - hy * CF_HW;
            const int y = (u0 - CF_R + hy) * p.S + py, x = (v0 - CF_R + hx) * p.S + px;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (y >= 0 && y < p.H && x >= 0 && x < p.W) v = *reinterpret_cast<const float4*>(m.p + m.off(n, c0 + 4 * c4, y, x));
            *reinterpret_cast<float4*>(halo + hp * 32 + 4 * c4) = v;
        }
        float4 acc[4];
#pragma unroll
        for (int i = 0; i < 4; i++) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        // Gx values of CF_GB displacement rows per step; the next step's values are fetched into registers while this one computes
        float pre[CF_GSTAGE / 256];
        auto gfetch = [&](int dj0) {
#pragma unroll
            for (int j = 0; j < CF_GSTAGE / 256; j++) {
                const int idx = tid + 256 * j;
                const int b = idx / (CF_TH * CF_TW * CF_GROW), rem = idx - b * (CF_TH * CF_TW * CF_GROW);
                const int q = rem / CF_GROW, di = rem - q * CF_GROW;
                const int y = (u0 + (q >> 4)) * p.S + py, x = (v0 + (q & 15)) * p.S + px;
                pre[j] = (di < CF_DW && y < p.H && x < p.W) ? g.p[g.off(n, (dj0 + b) * CF_DW + di, y, x)] : 0.f;
            }
        };
        gfetch(0);
#pragma unroll 1
        for (int dj = 0; dj < CF_DW; dj++) {
            if (dj % CF_GB == 0) {
                __syncthreads();
#pragma unroll
                for (int j = 0; j < CF_GSTAGE / 256; j++) gs[tid + 256 * j] = pre[j];
                __syncthreads();
                if (dj + CF_GB < CF_DW) gfetch(dj + CF_GB);
            }
            const float* gsr = gs + (dj % CF_GB) * (CF_TH * CF_TW * CF_GROW);
            float gr[4][CF_GROW];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int k4 = 0; k4 < CF_GROW / 4; k4++) {
                    const float4 t = *reinterpret_cast<const float4*>(gsr + (row * CF_TW + xg * 4 + i) * CF_GROW + 4 * k4);
                    gr[i][4 * k4] = t.x; gr[i][4 * k4 + 1] = t.y; gr[i][4 * k4 + 2] = t.z; gr[i][4 * k4 + 3] = t.w;
                }
            // halo row / first halo column of this thread for displacement row dj
            const int hrow = SGN > 0 ? row + dj : row + 2 * CF_R - dj;
            const float* hb = halo + (hrow * CF_HW + xg * 4) * 32 + 4 * cg;
#pragma unroll
            for (int t = 0; t < CF_DW + 3; t++) {
                const float4 mv = *reinterpret_cast<const float4*>(hb + t * 32);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    // halo column xg*4 + t is pixel i's column + di (SGN > 0) resp. + 2R - di (SGN < 0)
                    const int e = t - i;
                    if (e >= 0 && e < CF_DW) {
                        const float gv = gr[i][SGN > 0 ? e : 2 * CF_R - e];
                        acc[i].x = fmaf(gv, mv.x, acc[i].x); acc[i].y = fmaf(gv, mv.y, acc[i].y);
                        acc[i].z = fmaf(gv, mv.z, acc[i].z); acc[i].w = fmaf(gv, mv.w, acc[i].w);
                    }
                }
            }
        }
        const int y = (u0 + row) * p.S + py;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = (v0 + xg * 4 + i) * p.S + px;
            if (y < p.H && x < p.W)
                *reinterpret_cast<float4*>(out.p + out.off(n, c0 + 4 * cg, y, x)) =
                    make_float4(acc[i].x * p.scale, acc[i].y * p.scale, acc[i].z * p.scale, acc[i].w * p.scale);
        }
    }
}

// Gx[n][y][x][d] = topdiff[n][d][y - dy(d)][x - dx(d)] (0 outside): the bottom1 gradient then has the bottom0 gradient's form
__global__ void corr_shift_kernel(T4 td, float* __restrict__ gx, int R, int S) {
    const int Dw = 2 * R + 1, D = Dw * Dw;
    const long long total = (long long)td.n * td.h * td.w * D;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int d = (int)(idx % D);
        long long r = idx / D;
        const int x = (int)(r % td.w); r /= td.w;
        const int y = (int)(r % td.h);
        const int n = (int)(r / td.h);
        const int yy = y - (d / Dw - R) * S, xx = x - (d % Dw - R) * S;
        gx[idx] = (yy >= 0 && yy < td.h && xx >= 0 && xx < td.w) ? td.p[td.off(n, d, yy, xx)] : 0.f;
    }
}

static bool corr_fast_ok(const T4& b0, const T4& b1, const T4& td, const T4& d0, const T4& d1, const CbP& p, int corr_type, int s2) {
    if (corr_type != 0 || !p.identity_g || p.D != CF_DW * CF_DW || s2 < 1 || s2 > 2 || p.reach_x != CF_R * s2 || p.C % 32) return false;
    const T4* ts[4] = {&b0, &b1, &d0, &d1};
    for (const T4* t : ts)
        if (t->sc != 1 || ((uintptr_t)t->p & 15) || (t->sw & 3) || (t->sh & 3) || (t->sn & 3)) return false;
    return true;
}

static int corr_fast_run(const T4& b0, const T4& b1, const T4& td, const T4& d0, const T4& d1, const CbP& p, int s2, float* ws, cudaStream_t st) {
    CfP f;
    f.N = p.N; f.C = p.C; f.H = p.H; f.W = p.W; f.S = s2; f.scale = p.scale; f.cchunks = p.C / 32;
    const int Hp = (p.H + s2 - 1) / s2, Wp = (p.W + s2 - 1) / s2;
    f.tiles_y = (Hp + CF_TH - 1) / CF_TH; f.tiles_x = (Wp + CF_TW - 1) / CF_TW;
    const int units = f.N * s2 * s2 * f.tiles_y * f.tiles_x * f.cchunks;
    static bool attr = false;
    if (!attr) {
        FN2_CUDA(cudaFuncSetAttribute(corr_bwd_fast_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, CF_SMEM));
        FN2_CUDA(cudaFuncSetAttribute(corr_bwd_fast_kernel<-1>, cudaFuncAttributeMaxDynamicSharedMemorySize, CF_SMEM));
        attr = true;
    }
    const int grid = min(units, num_sms());
    corr_bwd_fast_kernel<1><<<grid, 256, CF_SMEM, st>>>(td, b1, d0, f);
    FN2_LAUNCH_CHECK();
    corr_shift_kernel<<<ew_grid((long long)p.N * p.H * p.W * p.D, 256), 256, 0, st>>>(td, ws, CF_R, s2);
    FN2_LAUNCH_CHECK();
    T4 gx;
    gx.p = ws; gx.n = p.N; gx.c = p.D; gx.h = p.H; gx.w = p.W;
    gx.sc = 1; gx.sw = p.D; gx.sh = (long long)p.W * p.D; gx.sn = (long long)p.H * p.W * p.D;
    corr_bwd_fast_kernel<-1><<<grid, 256, CF_SMEM, st>>>(gx, b0, d1, f);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

int corr_bwd_run(const T4& b0, const T4& b1, const T4& td, const T4& d0, const T4& d1, CbP& p, int corr_type, float* ws, size_t ws_floats,
                 cudaStream_t st, int s2_2d = 0) {
    if (s2_2d > 0 && corr_fast_ok(b0, b1, td, d0, d1, p, corr_type, s2_2d)) {
        if (!ws || ws_floats < (size_t)p.N * p.H * p.W * p.D) { set_error("correlation_backward: workspace too small"); return FN2_ERR_WORKSPACE; }
        return corr_fast_run(b0, b1, td, d0, d1, p, s2_2d, ws, st);
    }
    const size_t gfloats = p.identity_g ? 0 : (size_t)p.N * p.H * p.W * p.D;
    const size_t sfloats = corr_type == 1 ? (size_t)p.N * p.H * p.W * p.C : 0;
    if (gfloats + sfloats > ws_floats || (!ws && gfloats + sfloats)) { set_error("correlation_backward: workspace too small (%zu floats needed)", gfloats + sfloats); return FN2_ERR_WORKSPACE; }
    float* g = ws;
    float* sgn = ws + gfloats;
    if (!p.identity_g) {
        corr_patchsum_kernel<<<ew_grid((long long)gfloats, 256), 256, 0, st>>>(td, g, p);
        FN2_LAUNCH_CHECK();
    }
    T4 m0 = b1, m1 = b0;
    float s0 = 1.f, s1 = 1.f;
    p.oob = 0.f;
    if (corr_type == 1) {
        corr_sign_kernel<<<ew_grid(b0.count(), 256), 256, 0, st>>>(b0, b1, sgn);
        FN2_LAUNCH_CHECK();
        T4 sv; sv.p = sgn; sv.n = p.N; sv.c = p.C; sv.h = p.H; sv.w = p.W;
        sv.sc = 1; sv.sw = p.C; sv.sh = (long long)p.W * p.C; sv.sn = (long long)p.H * p.W * p.C;
        m0 = sv; m1 = sv; s0 = 1.f; s1 = -1.f; p.oob = 1.f;
    }
    const int hw = CB_TILE + 2 * p.reach_x, hh = CB_TILE + 2 * p.reach_y;
    const size_t smem = ((size_t)64 * p.D + (size_t)hh * hw * CB_CH) * sizeof(float);
    if (smem > 220 * 1024) { set_error("correlation_backward: displacement window too large for the tiled kernel (%zu B)", smem); return FN2_ERR_INVALID; }
    static size_t set0 = 0, set1 = 0;
    if (smem > set0) { FN2_CUDA(cudaFuncSetAttribute(corr_apply_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); set0 = smem; }
    if (smem > set1) { FN2_CUDA(cudaFuncSetAttribute(corr_apply_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); set1 = smem; }
    const int tiles = p.N * ((p.H + CB_TILE - 1) / CB_TILE) * ((p.W + CB_TILE - 1) / CB_TILE);
    const int grid = min(tiles, num_sms());
    corr_apply_kernel<0><<<grid, 256, smem, st>>>(g, td, m0, d0, p, s0);
    FN2_LAUNCH_CHECK();
    corr_apply_kernel<1><<<grid, 256, smem, st>>>(g, td, m1, d1, p, s1);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

}  // namespace

size_t corr_bwd_workspace_floats(int N, int C, int H, int W, int D, int k, int s1, int pad, int md, int topH, int topW, int corr_type, int one_d) {
    const bool ident = k == 1 && s1 == 1 && pad == md && topH == H && topW == W;
    // (the identity case of the 2-D MULTIPLY layer may take the fast path, which stages the shifted top diff there)
    return ((ident && (one_d || corr_type == 1)) ? 0 : (size_t)N * H * W * D) + (corr_type == 1 ? (size_t)N * H * W * C : 0);
}

// 2-D layer: top channel tc <-> displacement ((tc / Dw - R) * s2, (tc % Dw - R) * s2)   (correlation_layer.cu:81-82)
int corr_bwd_2d(const T4& b0, const T4& b1, const T4& td, const T4& d0, const T4& d1, int pad, int k, int md, int s1, int s2, int corr_type,
                float* ws, size_t ws_floats, cudaStream_t st) {
    CbP p;
    memset(&p, 0, sizeof(p));
    p.N = b0.n; p.C = b0.c; p.H = b0.h; p.W = b0.w;
    const int R = md / s2, Dw = 2 * R + 1;
    p.D = Dw * Dw;
    if (p.D > 441) { set_error("correlation_backward: more than 441 displacements"); return FN2_ERR_INVALID; }
    p.topH = td.h; p.topW = td.w; p.k = k; p.s1 = s1; p.md = md; p.pad = pad; p.ypatch_off = md - pad;
    for (int tc = 0; tc < p.D; tc++) { p.dy[tc] = (short)((tc / Dw - R) * s2); p.dx[tc] = (short)((tc % Dw - R) * s2); }
    p.reach_y = p.reach_x = R * s2;
    p.identity_g = (k == 1 && s1 == 1 && pad == md && td.h == b0.h && td.w == b0.w) ? 1 : 0;
    p.scale = 1.f / (float)(k * k * p.C);
    return corr_bwd_run(b0, b1, td, d0, d1, p, corr_type, ws, ws_floats, st, s2);
}

// 1-D layer: tc <-> (0, (tc + x_shift) * s2), x_shift = -R (both directions or left only) or 0 (right only)
static int corr1d_geometry(int md, int s2, int single_direction, int* D, int* x_shift) {
    const int R = md / s2;
    *D = single_direction != 0 ? R + 1 : 2 * R + 1;          // correlation_layer1d.cpp:64-68
    // correlation_layer1d.cu Forward_gpu: -R, "to the left" -grid_width (sic: one stride_2 step beyond -max_displacement), "to the right" 0
    *x_shift = single_direction == 1 ? 0 : (single_direction == -1 ? -(R + 1) : -R);
    return R;
}

int corr1d_shape(int H, int W, int pad, int k, int md, int s1, int s2, int single_direction, int* tc, int* th, int* tw) {
    if (k < 1 || k % 2 == 0) { set_error("Odd kernel size required (correlation_layer1d.cpp:22)"); return FN2_ERR_INVALID; }
    if (s1 < 1 || s2 < 1 || md < 0 || pad < 0) { set_error("correlation1d: bad stride/displacement/pad"); return FN2_ERR_INVALID; }
    if (single_direction < -1 || single_direction > 1) { set_error("single_direction must be -1 (left), 0 (off), or 1 (right)"); return FN2_ERR_INVALID; }
    const int kr = (k - 1) / 2, border = md + kr;
    const int w = (int)ceilf((float)(W + 2 * pad - border * 2) / (float)s1);     // :55
    const int h = (int)ceilf((float)(H - kr * 2) / (float)s1);                   // :56 (rows are not padded)
    if (w < 1 || h < 1) { set_error("Correlation cannot be done with current settings. Neighborhood and kernel don't fit in blob"); return FN2_ERR_INVALID; }
    int D, xs;
    corr1d_geometry(md, s2, single_direction, &D, &xs);
    *tc = D; *th = h; *tw = w;
    return FN2_OK;
}

int corr1d_forward(const T4& b0, const T4& b1, const T4& top, int pad, int k, int md, int s1, int s2, int single_direction, int corr_type,
                   cudaStream_t st) {
    int D, xs;
    corr1d_geometry(md, s2, single_direction, &D, &xs);
    const size_t smem = (size_t)k * k * b0.c * sizeof(float);
    if (smem > 200 * 1024) { set_error("correlation1d: k*k*C patch does not fit in shared memory"); return FN2_ERR_INVALID; }
    if (smem > 48 * 1024) FN2_CUDA(cudaFuncSetAttribute(corr1d_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(top.w, top.h, b0.n);
    corr1d_fwd_kernel<<<grid, 128, smem, st>>>(b0, b1, top, pad, k, md, s1, s2, xs, corr_type);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

int corr_bwd_1d(const T4& b0, const T4& b1, const T4& td, const T4& d0, const T4& d1, int pad, int k, int md, int s1, int s2,
                int single_direction, int corr_type, float* ws, size_t ws_floats, cudaStream_t st) {
    CbP p;
    memset(&p, 0, sizeof(p));
    p.N = b0.n; p.C = b0.c; p.H = b0.h; p.W = b0.w;
    int xs;
    const int R = corr1d_geometry(md, s2, single_direction, &p.D, &xs);
    p.topH = td.h; p.topW = td.w; p.k = k; p.s1 = s1; p.md = md; p.pad = pad; p.ypatch_off = 0;
    for (int tc = 0; tc < p.D; tc++) { p.dy[tc] = 0; p.dx[tc] = (short)((tc + xs) * s2); }
    p.reach_y = 0; p.reach_x = (single_direction == -1 ? R + 1 : R) * s2;
    p.identity_g = (k == 1 && s1 == 1 && pad == md && td.h == b0.h && td.w == b0.w) ? 1 : 0;
    p.scale = 1.f / (float)(k * k * p.C);
    return corr_bwd_run(b0, b1, td, d0, d1, p, corr_type, ws, ws_floats, st);
}

}  // namespace fn2
