// "Taps on N" tcgen05 convolution / deconvolution for layers with FEW output channels at high resolution (sm_100a).
//
// The fusion tail of FlowNet2 (fuse_interconv0 82->16, fuse_deconv0 162->16, fuse_interconv1 162->32, fuse_deconv1 128->32 at
// full / half resolution) is 18 % of the forward pass on the per-tap engine (fn2_conv_tc.cu): with NT = 16 / 32 output channels
// on the MMA's N side every tcgen05.mma is bound by the fetch of its 128 x 8 A operand (64 cycles however small N is), and the
// A tile is re-fetched and re-split for each of the 9 / 4 taps (profiles/r01_prof_tc16_*: L2->SM traffic 10x the DRAM bytes).
//
// Here the GEMM is turned around the way Caffe's own deconvolution is (col = W^T x, then col2im -- base_conv_layer.cpp:283-298),
// for convolutions as well ("kn2row"):
//     D[128 input pixels x (taps * Co)] = X[128 x Ci] * Wt[(taps * Co) x Ci]^T          K = Ci only
//     out[pixel + shift(tap)][co] += D[pixel][tap][co]                                   scatter-add ("col2im")
// Every input pixel is loaded and TF32-split ONCE per K block (not once per tap), N = taps*Co is 128..192 so the tensor core
// is busy for >= 64 cycles per A fetch, and no tap multiplies structural zeros (deconvolution: each input pixel meets all
// kh*kw taps, each belonging to exactly one output parity).
//   * 3xTF32 as in fn2_conv_tc.cu (a_hi*w_hi + a_hi*w_lo + a_lo*w_hi), A split by converter warps into tensor memory, W
//     pre-split at pack time.  K is short here (Ci <= 256: <= 8 K blocks), so all three products chain into ONE accumulator per
//     pass (n = 12 * cblocks MMAs) and the calibrated mean round-toward-zero loss of a chain of that length is added back
//     when the accumulator is drained (profiles/r01_tc_calibration.txt); accumulators are double-buffered in tensor memory.
//   * A CTA walks DOWN a strip of tw input columns, tile (th x tw = 128 pixels) by tile.  The scatter-add target is a ring
//     of output rows in shared memory, laid out [ring row][co][column] so that the 32 lanes of a warp (consecutive input
//     columns) hit consecutive banks.  One kernel row per phase: within a phase different warps (different input rows) hit
//     different output rows, within a warp the kw taps are applied in program order -- no atomics, fixed summation order.
//     Output rows leave the ring (bias, leaky ReLU, 128-bit NHWC stores) as soon as no later tile can touch them; only
//     the strip borders (kw-1 columns) and the segment borders are recomputed: 30 of 32 columns are useful for a 3x3.
//   * Taps are cut into passes of <= 192 accumulator columns (tensor memory: 2 x 192 accumulator + 2 x 64 A-slot columns).
// Warp roles, barrier rings and PDL as in fn2_conv_tc.cu.  Reference ops replaced: conv_layer.cu:8-23, deconv_layer.cu:8-23.
#include <cuda.h>

#include "fn2_common.cuh"
#include "fn2_tc_ptx.cuh"

namespace fn2 {

namespace {

constexpr int TN_THREADS = 512;
constexpr int TN_DRAIN = 256;                    // drain threads (warps 8-15)
constexpr int TN_A_BYTES = 128 * 128;            // 128 pixels x 32 fp32
constexpr int TN_ACC_COLS = 192;                 // tensor-memory columns per accumulator buffer
constexpr int TN_COL_A = 384;                    // A slots: hi at 384 + 64*s, lo at +32
constexpr int TN_MAXPASS = 6;

struct TnParams {
    int N, Hin, Win, Ho, Wo, Co, cblocks;
    int S, kh, kw;                               // S: output step per input pixel (1 conv, 2 deconv)
    int oy[4], ox[4];                            // output row / column offset of kernel row r / column s
    int oy_min, oy_max, ox_min;
    int tw, th;
    int stepx, cshift, xa;                       // strip b: input cols [b*stepx + cshift, +tw); complete outputs x = S*c0 + xa + [0, S*stepx)
    int nstrips, nseg, seg_rows;                 // segment g: output rows [g*seg_rows, min(Ho, (g+1)*seg_rows))
    int RR, CW, F;                               // ring rows; columns per (ring row, co); tiles between two flushes of the ring
    int npass, pass_tap0[TN_MAXPASS], pass_ntaps[TN_MAXPASS];
    // scatter plan: every pass is a list of groups = runs of taps of ONE kernel row; inside a group, taps whose column offsets
    // differ by a multiple of S are summed across lanes first (class cls: leader tap + partners with their lane shifts)
    int ngrp[TN_MAXPASS];
    struct Grp { short tl0, nrow, oyr, ncls; short ox0[2], np[2]; short ps[2][3], sh[2][3]; } grp[TN_MAXPASS][4];
    int ngmax;                                   // W tile rows in shared memory (max taps per pass * Co)
    int RA, RW, wres;                            // raw-A ring depth, W ring depth, 1 = all W stages resident in shared memory
    int total;                                   // units = N * nstrips * nseg
    float comp;                                  // mean RZ shrink of the 12*cblocks-MMA chain
    int relu, has_bias;
    float slope;
    long long out_sn, out_sh, out_sw;
    FastDiv d_nseg, d_nstrips;
};

struct TnUnit { int n, c0, R0, R1, i_lo, ntiles; };

__device__ __forceinline__ int floordiv_d(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
__device__ __forceinline__ int ceildiv_d(int a, int b) { return -floordiv_d(-a, b); }

__device__ __forceinline__ TnUnit tn_decode(const TnParams& p, int u) {
    TnUnit U;
    int q, g, b;
    p.d_nseg.divmod(u, q, g);
    p.d_nstrips.divmod(q, U.n, b);
    U.c0 = b * p.stepx + p.cshift;
    U.R0 = g * p.seg_rows;
    U.R1 = min(p.Ho, U.R0 + p.seg_rows);
    int lo = 1 << 30, hi = -(1 << 30);
    for (int r = 0; r < p.kh; r++) {
        lo = min(lo, ceildiv_d(U.R0 - p.oy[r], p.S));
        hi = max(hi, floordiv_d(U.R1 - 1 - p.oy[r], p.S));
    }
    U.i_lo = lo;
    U.ntiles = (hi - lo + 1 + p.th - 1) / p.th;
    return U;
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(taddr) : "memory");
}

// named barrier of one channel half of the drain group (4 warps)
__device__ __forceinline__ void tn_group_sync(int h) {
    if (h) asm volatile("bar.sync 2, 128;" ::: "memory");
    else asm volatile("bar.sync 1, 128;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}

// Warps: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4-7 converters, 8-15 drain (two warps per TMEM lane quarter, each
// taking half of the output channels of every tap).  512 threads x 128 registers = the whole register file.
template <int CO, int S>
__global__ void __launch_bounds__(TN_THREADS, 1)
conv_tn_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const float* __restrict__ bias,
               float* __restrict__ out, const TnParams p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    // shared memory: [A ring: RA raw 16 KB tiles][W ring: RW stages of (hi, lo) tiles -- or, when the layer's whole packed weight
    // matrix fits, all npass*cblocks stages resident for the lifetime of the CTA][barriers][output ring]
    const int wstage = 2 * p.ngmax * 128;
    const int nw = p.wres ? p.npass * p.cblocks : p.RW;
    unsigned char* smemW = smem + (size_t)p.RA * TN_A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smemW + (size_t)nw * wstage);
    uint64_t* fullA = bars;                        // [RA] TMA bytes of the raw A tile have landed
    uint64_t* freeA = bars + 4;                    // [RA] the 128 converter threads have read the raw tile
    uint64_t* fullW = bars + 8;                    // [RW] W stage landed  (resident mode: fullW[0] = everything landed)
    uint64_t* a_ready = bars + 12;                 // [2]  converters have written A slot (hi, lo) in tensor memory
    uint64_t* sdone = bars + 14;                   // [6]  MMAs of step it (it % 6) have retired: frees W stage it % RW and A slot it & 1
    uint64_t* acc_full = bars + 20;                // [2]
    uint64_t* acc_free = bars + 22;                // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);
    float* obuf = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bars) + 256);       // [RR][CO][CW]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid == 0) {
        for (int s = 0; s < 4; s++) { mbar_init(&fullA[s], 1); mbar_init(&freeA[s], 128); mbar_init(&fullW[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&a_ready[s], 128); mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], TN_DRAIN); }
        for (int s = 0; s < 6; s++) mbar_init(&sdone[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(su32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < p.RR * CO * p.CW; i += TN_THREADS) obuf[i] = 0.f;
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp < 4) {
        if (warp == 0 && lane == 0) {
            // ===== TMA producer: raw A tiles run RA steps ahead (released by the converters), W stages RW steps ahead
            // (released by the MMAs) =====
            if (p.wres) {
                mbar_expect_tx(&fullW[0], (uint32_t)(nw * wstage));
                for (int b = 0; b < nw; b++) {
                    tma_load_4d(smemW + (size_t)b * wstage, &mapW, &fullW[0], 0, 0, b, 0);
                    tma_load_4d(smemW + (size_t)b * wstage + p.ngmax * 128, &mapW, &fullW[0], 0, 0, b, 1);
                }
            }
            int sa = 0, sw = 0, it = 0; uint32_t pha = 1u;
            for (int u = blockIdx.x; u < p.total; u += gridDim.x) {
                const TnUnit U = tn_decode(p, u);
                for (int k = 0; k < U.ntiles; k++) {
                    const int i0 = U.i_lo + k * p.th;
                    for (int ps = 0; ps < p.npass; ps++) {
#pragma unroll 1
                        for (int cb = 0; cb < p.cblocks; cb++, it++) {
                            if (!p.wres) {
                                if (it >= p.RW) { const int j = it - p.RW; mbar_wait(&sdone[j % 6], (uint32_t)(j / 6) & 1u); }
                                unsigned char* st = smemW + (size_t)sw * wstage;
                                mbar_expect_tx(&fullW[sw], (uint32_t)wstage);
                                tma_load_4d(st, &mapW, &fullW[sw], 0, 0, ps * p.cblocks + cb, 0);
                                tma_load_4d(st + p.ngmax * 128, &mapW, &fullW[sw], 0, 0, ps * p.cblocks + cb, 1);
                                if (++sw == p.RW) sw = 0;
                            }
                            mbar_wait(&freeA[sa], pha);
                            mbar_expect_tx(&fullA[sa], (uint32_t)TN_A_BYTES);
                            tma_load_4d(smem + (size_t)sa * TN_A_BYTES, &mapA, &fullA[sa], cb * 32, U.c0, i0, U.n);
                            if (++sa == p.RA) { sa = 0; pha ^= 1u; }
                        }
                    }
                }
            }
        } else if (warp == 1) {
            // ===== MMA issuer (convergent warp, one elected lane issues) =====
            int sw = 0, buf = 0, it = 0;
            uint32_t phw = 0, pacc = 1u;
            if (p.wres) mbar_wait(&fullW[0], 0);
            for (int u = blockIdx.x; u < p.total; u += gridDim.x) {
                const TnUnit U = tn_decode(p, u);
                for (int k = 0; k < U.ntiles; k++) {
                    for (int ps = 0; ps < p.npass; ps++) {
                        const uint32_t idesc = make_idesc_tf32(128, p.pass_ntaps[ps] * CO);
                        mbar_wait(&acc_free[buf], pacc);
                        const uint32_t d = tmem + (uint32_t)(buf * TN_ACC_COLS);
#pragma unroll 1
                        for (int cb = 0; cb < p.cblocks; cb++, it++) {
                            uint32_t bh;
                            if (p.wres) bh = su32(smemW + (size_t)(ps * p.cblocks + cb) * wstage);
                            else { mbar_wait(&fullW[sw], phw); bh = su32(smemW + (size_t)sw * wstage); }
                            mbar_wait(&a_ready[it & 1], (uint32_t)(it >> 1) & 1u);
                            fence_after();
                            const uint64_t dbh0 = make_desc_sw128(bh), dbl0 = make_desc_sw128(bh + (uint32_t)p.ngmax * 128u);
                            const uint32_t a_hi = tmem + TN_COL_A + 64 * (it & 1), a_lo = a_hi + 32;
                            if (elect_one()) {
#pragma unroll
                                for (int kk = 0; kk < 4; kk++) {
                                    mma_tf32_ts(d, a_hi + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc, (cb | kk) != 0);
                                    mma_tf32_ts(d, a_hi + kk * 8, dbl0 + (uint64_t)(2 * kk), idesc, 1);
                                    mma_tf32_ts(d, a_lo + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc, 1);
                                }
                                mma_commit(&sdone[it % 6]);
                                if (cb == p.cblocks - 1) mma_commit(&acc_full[buf]);
                            }
                            __syncwarp();
                            if (!p.wres && ++sw == p.RW) { sw = 0; phw ^= 1u; }
                        }
                        if (buf) pacc ^= 1u;
                        buf ^= 1;
                    }
                }
            }
        }
    } else if (warp < 8) {
        // ===== converters: raw FP32 tile (smem, swizzled) -> a_hi / a_lo in tensor memory (two halves of 16 channels) =====
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        int sa = 0, it = 0;
        uint32_t pha = 0;
        for (int u = blockIdx.x; u < p.total; u += gridDim.x) {
            const TnUnit U = tn_decode(p, u);
            const int steps = U.ntiles * p.npass * p.cblocks;
#pragma unroll 1
            for (int i = 0; i < steps; i++, it++) {
                mbar_wait(&fullA[sa], pha);
                const float4* row = reinterpret_cast<const float4*>(smem + (size_t)sa * TN_A_BYTES + m * 128);
                float4 raw[8];
#pragma unroll
                for (int j = 0; j < 8; j++) raw[j] = row[j ^ (m & 7)];
                mbar_arrive(&freeA[sa]);           // the raw tile may be overwritten (values are in registers)
                // A slot (it & 1) was last read by the MMAs of step it-2
                if (it >= 2) { const int j = it - 2; mbar_wait(&sdone[j % 6], (uint32_t)(j / 6) & 1u); }
                fence_after();
                const uint32_t slot = lane_addr + TN_COL_A + 64 * (it & 1);
#pragma unroll
                for (int half = 0; half < 2; half++) {
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const float4 v4 = raw[4 * half + j];
                        const float f[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const uint32_t h = to_tf32(f[e]);
                            hi[4 * j + e] = h;
                            lo[4 * j + e] = to_tf32(f[e] - __uint_as_float(h));
                        }
                    }
                    tmem_st16(slot + 16 * half, hi);
                    tmem_st16(slot + 32 + 16 * half, lo);
                }
                tmem_wait_st();
                fence_before();
                mbar_arrive(&a_ready[it & 1]);
                if (++sa == p.RA) { sa = 0; pha ^= 1u; }
            }
        }
    } else {
        // ===== drain + scatter-add + write-out: 8 warps; warp (q, h) owns TMEM lanes 32q.. and channels [h*CO/2, (h+1)*CO/2) =====
        constexpr int CH = CO / 2;                 // channels per drain thread
        const int q = warp & 3, h = (warp - 8) >> 2;
        const int m = q * 32 + lane;               // tile pixel == TMEM lane
        const int dt = tid - 256;                  // 0..255 within the drain group
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const int it_ = m / p.tw, jt = m % p.tw;   // tile row / column of this lane's input pixel
        const int rowstride = CO * p.CW;
        const int col0 = jt * p.S - p.ox_min + h * CH * p.CW;     // + ox[sx]: this thread's first element inside a ring row
        const int advance = p.th * p.S;            // output rows that leave the ring per tile
        float bv[4] = {0.f, 0.f, 0.f, 0.f};        // bias of the 4 channels this thread writes out
        if (p.has_bias) {
            const int cb_ = h * CH + 4 * ((dt & 127) % (CH / 4));
            bv[0] = __ldg(bias + cb_); bv[1] = __ldg(bias + cb_ + 1); bv[2] = __ldg(bias + cb_ + 2); bv[3] = __ldg(bias + cb_ + 3);
        }
        int buf = 0; uint32_t pfull = 0;
        for (int u = blockIdx.x; u < p.total; u += gridDim.x) {
            const TnUnit U = tn_decode(p, u);
            const int x_base = p.S * U.c0 + p.ox_min;                 // output column of ring column 0
            const int xc_lo = max(0, p.S * U.c0 + p.xa), xc_hi = min(p.Wo, p.S * U.c0 + p.xa + p.S * p.stepx);   // complete output columns
            const int ncol = xc_hi - xc_lo;
            int rb = 0;                            // ring slot of the first row the current tile can touch
            int flush_lo = 0, since_flush = 0;     // first row still in the ring; tiles since the last flush
            for (int k = 0; k < U.ntiles; k++) {
                const int i0 = U.i_lo + k * p.th;
                const int touched_lo = i0 * p.S + p.oy_min;
                const int yrel0 = it_ * p.S - p.oy_min;            // + oy[r]: row of this lane's contribution relative to touched_lo
                for (int ps = 0; ps < p.npass; ps++) {
                    mbar_wait(&acc_full[buf], pfull);
                    fence_after();
                    const uint32_t src = lane_addr + (uint32_t)(buf * TN_ACC_COLS + h * CH);
                    // Taps of one kernel row land in the same output row, a few columns apart: taps whose column offsets differ
                    // by a multiple of S hit the column of a NEIGHBOURING lane's tap, so they are first summed across lanes with
                    // shuffles (lane L collects what belongs to its own column) and only one read-modify-write per group reaches
                    // shared memory.  Lanes whose neighbour lies outside the warp (= outside the tile row) produce an incomplete
                    // sum for a column outside the strip's complete range, which is never written out.
                    const int ng = p.ngrp[ps];
#pragma unroll 1
                    for (int gi = 0; gi < ng; gi++) {
                        const int tl0 = p.grp[ps][gi].tl0, nrow = p.grp[ps][gi].nrow, oyr = p.grp[ps][gi].oyr;
                        if (gi) tn_group_sync(h);                      // the other 3 warps of this channel half may still add into the rows we now target
                        int ring = rb + yrel0 + oyr;
                        if (ring >= p.RR) ring -= p.RR;
                        float* rowp = obuf + ring * rowstride + col0;
                        const int ox0 = p.grp[ps][gi].ox0[0], ox1 = p.grp[ps][gi].ox0[1];
#pragma unroll 1
                        for (int c0 = 0; c0 < CH; c0 += 8) {
                            // straight-line code per (S, number of taps of this kernel row in the pass): the taps' values of lane L,
                            // RZ-compensated; conv (S = 1): tap sa+d of lane L+d belongs to lane L's column -> shuffle down by d;
                            // deconv (S = 2): tap sa+2 (sa+3) of lane L-1 belongs to the column of lane L's tap sa (sa+1) -> shuffle
                            // up by 1.  Lanes without that neighbour add garbage to a column outside the strip's complete range.
                            float a0[8], a1[8];
                            uint32_t v0[8], v1[8], v2[8], v3[8];
                            const uint32_t tsrc = src + (uint32_t)(tl0 * CO + c0);
                            tmem_ld8(tsrc, v0);
                            if (nrow > 1) tmem_ld8(tsrc + CO, v1);
                            if (nrow > 2) tmem_ld8(tsrc + 2 * CO, v2);
                            if (nrow > 3) tmem_ld8(tsrc + 3 * CO, v3);
                            tmem_wait_ld();
#define FN2_TN_COMP(x) fmaf(__uint_as_float(x), p.comp, __uint_as_float(x))
#pragma unroll
                            for (int c = 0; c < 8; c++) a0[c] = FN2_TN_COMP(v0[c]);
                            if constexpr (S == 1) {
                                if (nrow > 1) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a0[c] += __shfl_down_sync(0xffffffffu, FN2_TN_COMP(v1[c]), 1);
                                }
                                if (nrow > 2) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a0[c] += __shfl_down_sync(0xffffffffu, FN2_TN_COMP(v2[c]), 2);
                                }
                                if (nrow > 3) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a0[c] += __shfl_down_sync(0xffffffffu, FN2_TN_COMP(v3[c]), 3);
                                }
                            } else {
                                if (nrow > 1) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a1[c] = FN2_TN_COMP(v1[c]);
                                }
                                if (nrow > 2) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a0[c] += __shfl_up_sync(0xffffffffu, FN2_TN_COMP(v2[c]), 1);
                                }
                                if (nrow > 3) {
#pragma unroll
                                    for (int c = 0; c < 8; c++) a1[c] += __shfl_up_sync(0xffffffffu, FN2_TN_COMP(v3[c]), 1);
                                }
                            }
#undef FN2_TN_COMP
                            // read-modify-write of 8 different channel planes: all loads first (the compiler must otherwise assume that
                            // the store of plane c aliases the load of plane c+1 and serialises 8 shared-memory round trips)
                            float* o = rowp + c0 * p.CW + ox0;
                            float t_[8];
#pragma unroll
                            for (int c = 0; c < 8; c++) t_[c] = o[c * p.CW];
#pragma unroll
                            for (int c = 0; c < 8; c++) o[c * p.CW] = t_[c] + a0[c];
                            if (S == 2 && nrow > 1) {
                                __syncwarp();
                                float* o1 = rowp + c0 * p.CW + ox1;
#pragma unroll
                                for (int c = 0; c < 8; c++) t_[c] = o1[c * p.CW];
#pragma unroll
                                for (int c = 0; c < 8; c++) o1[c * p.CW] = t_[c] + a1[c];
                            }
                            __syncwarp();
                        }
                    }
                    fence_before();
                    mbar_arrive(&acc_free[buf]);
                    if (buf) pfull ^= 1u;
                    buf ^= 1;
                    tn_group_sync(h);
                }
                // rows no later tile of this unit can touch: write them out (inside the segment / image) and clear them.  The two
                // channel halves never meet in the ring, so each group of 4 warps flushes its own half on its own barrier.
                const int hi_row = (k == U.ntiles - 1) ? (i0 + p.th - 1) * p.S + p.oy_max + 1 : (i0 + p.th) * p.S + p.oy_min;
                if (k == 0) flush_lo = touched_lo;
                const bool do_flush = (k == U.ntiles - 1) || (++since_flush == p.F);
                if (do_flush) {
                    const int lo_row = flush_lo;
                    since_flush = 0; flush_lo = hi_row;
                    constexpr int CG = CH / 4;                 // float4 groups per pixel in this half
                    constexpr int XPI = 128 / CG;              // columns per iteration
                    const int d128 = dt & 127;
                    const int cg = d128 % CG, xi0 = d128 / CG;
                    const int cbase = h * CH + 4 * cg;
                    for (int y = max(lo_row, U.R0); y < min(hi_row, U.R1); y++) {
                        int ring = rb + (y - touched_lo);
                        if (ring >= p.RR) ring -= p.RR;
                        if (ring < 0) ring += p.RR;
                        const float* src_o = obuf + ring * rowstride + cbase * p.CW + (xc_lo - x_base);
                        float* dst = out + U.n * p.out_sn + (long long)y * p.out_sh + (long long)xc_lo * p.out_sw + cbase;
                        for (int xi = xi0; xi < ncol; xi += XPI) {
                            float rv[4];
#pragma unroll
                            for (int e = 0; e < 4; e++) {
                                float xv = src_o[e * p.CW + xi] + bv[e];
                                if (p.relu) xv = xv > 0 ? xv : xv * p.slope;
                                rv[e] = xv;
                            }
                            *reinterpret_cast<float4*>(dst + (long long)xi * p.out_sw) = make_float4(rv[0], rv[1], rv[2], rv[3]);
                        }
                    }
                    tn_group_sync(h);
                    const int n4 = (CH * p.CW) >> 2;           // this half of a ring row, a multiple of 4 floats (CW even)
                    for (int y = lo_row; y < hi_row; y++) {
                        int ring = rb + (y - touched_lo);
                        if (ring >= p.RR) ring -= p.RR;
                        if (ring < 0) ring += p.RR;
                        float4* z = reinterpret_cast<float4*>(obuf + ring * rowstride + h * CH * p.CW);
                        for (int e = d128; e < n4; e += 128) z[e] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    tn_group_sync(h);
                }
                rb += advance;
                while (rb >= p.RR) rb -= p.RR;
            }
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}



// ---- host ---------------------------------------------------------------------------------------------------------------
// packed weights: [hi|lo][pass * cblocks + cb][ngmax rows = (tap in pass, co)][32 channels of K block cb]
__global__ void tn_pack_kernel(const float* __restrict__ w, float* __restrict__ wp, int Ci, int Co, int kh, int kw, int deconv,
                               int cblocks, int ngmax, TnParams p) {
    const long long per = (long long)p.npass * cblocks * ngmax * 32;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(idx % 32);
        long long r_ = idx / 32;
        const int row = (int)(r_ % ngmax); r_ /= ngmax;
        const int cb = (int)(r_ % cblocks);
        const int ps = (int)(r_ / cblocks);
        const int tl = row / Co, co = row - tl * Co;
        const int ci = cb * 32 + k;
        float v = 0.f;
        if (tl < p.pass_ntaps[ps] && ci < Ci) {
            const int t = p.pass_tap0[ps] + tl;
            const int r = t / kw, s = t - r * kw;
            v = deconv ? w[(((long long)ci * Co + co) * kh + r) * kw + s] : w[(((long long)co * Ci + ci) * kh + r) * kw + s];
        }
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
        const float hi = __uint_as_float(h);
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - hi));
        wp[idx] = hi;
        wp[per + idx] = __uint_as_float(l);
    }
}

int tn_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("FN2_TN"); v = (e && e[0] == '0') ? 0 : 1; }
    return v;
}

// Everything that depends on the layer alone (not on the image size): taps, passes, tile shape, strip geometry, ring.
static bool tn_layer_plan(const fn2_conv_desc* d, TnParams* p) {
    if (d->out_pad_h || d->out_pad_w) return false;               // gradient operators of strided convolutions: general engine
    if (!tn_enabled()) return false;
    if (d->co != 16 && d->co != 32) return false;
    if (d->ci <= 16 || d->ci > 256) return false;
    if (d->kh > 4 || d->kw > 4 || d->kh * d->kw < 4) return false;
    if (!d->deconv && (d->stride_h != 1 || d->stride_w != 1 || d->pad_h >= d->kh || d->pad_w >= d->kw)) return false;
    if (d->deconv && (d->stride_h != 2 || d->stride_w != 2 || d->pad_h >= d->kh || d->pad_w >= d->kw)) return false;
    memset(p, 0, sizeof(*p));
    p->Co = d->co; p->cblocks = (d->ci + 31) / 32;
    p->kh = d->kh; p->kw = d->kw; p->S = d->deconv ? 2 : 1;
    p->oy_min = 1 << 30; p->oy_max = -(1 << 30); p->ox_min = 1 << 30;
    int ox_max = -(1 << 30);
    for (int r = 0; r < d->kh; r++) { p->oy[r] = d->deconv ? r - d->pad_h : d->pad_h - r; p->oy_min = min(p->oy_min, p->oy[r]); p->oy_max = max(p->oy_max, p->oy[r]); }
    for (int s = 0; s < d->kw; s++) { p->ox[s] = d->deconv ? s - d->pad_w : d->pad_w - s; p->ox_min = min(p->ox_min, p->ox[s]); ox_max = max(ox_max, p->ox[s]); }
    // passes: balanced chunks of consecutive taps with at most TN_ACC_COLS accumulator columns
    const int ntaps = d->kh * d->kw, maxt = TN_ACC_COLS / d->co;
    p->npass = (ntaps + maxt - 1) / maxt;
    if (p->npass > TN_MAXPASS) return false;
    const int per = (ntaps + p->npass - 1) / p->npass;
    int t0 = 0;
    p->ngmax = 0;
    for (int i = 0; i < p->npass; i++) {
        p->pass_tap0[i] = t0;
        p->pass_ntaps[i] = min(per, ntaps - t0);
        t0 += p->pass_ntaps[i];
        p->ngmax = max(p->ngmax, p->pass_ntaps[i] * d->co);
    }
    // scatter plan per pass
    for (int i = 0; i < p->npass; i++) {
        int tl = 0, ng = 0;
        while (tl < p->pass_ntaps[i]) {
            const int t = p->pass_tap0[i] + tl, r = t / d->kw, sa = t - r * d->kw;
            const int nrow = min(d->kw - sa, p->pass_ntaps[i] - tl);
            if (ng >= 4) return false;
            TnParams::Grp& G = p->grp[i][ng++];
            G.tl0 = (short)tl; G.nrow = (short)nrow; G.oyr = (short)p->oy[r]; G.ncls = (short)min(p->S, nrow);
            for (int cls = 0; cls < G.ncls; cls++) {
                G.ox0[cls] = (short)p->ox[sa + cls]; G.np[cls] = 0;
                for (int s_ = cls + p->S; s_ < nrow; s_ += p->S) {
                    const int k = G.np[cls]++;
                    G.ps[cls][k] = (short)s_;
                    G.sh[cls][k] = (short)((p->ox[sa + s_] - p->ox[sa + cls]) / p->S);
                }
            }
            tl += nrow;
        }
        p->ngrp[i] = ng;
    }
    // tile: one warp of the drain group = one (tw = 32) or two (tw = 16) input rows
    p->tw = 32; p->th = 4;
    p->CW = p->S * (p->tw - 1) + (ox_max - p->ox_min) + 1;
    const int span = (p->th - 1) * p->S + (p->oy_max - p->oy_min) + 1;       // output rows one tile can touch
    p->F = 1; p->RR = span;
    // complete output columns of a strip at c0 = 0: x such that every input column that contributes lies in [0, tw)
    int xa = 1 << 30, xb = -(1 << 30);
    for (int x = -64; x < p->S * p->tw + 64; x++) {
        bool any = false, all_in = true;
        for (int j = -40; j < p->tw + 40; j++)
            for (int s = 0; s < d->kw; s++)
                if (j * p->S + p->ox[s] == x) { any = true; if (j < 0 || j >= p->tw) all_in = false; }
        if (any && all_in) { xa = min(xa, x); xb = max(xb, x); }
    }
    if (xb < xa || (xb - xa + 1) % p->S) return false;
    p->stepx = (xb - xa + 1) / p->S;
    p->xa = xa;
    // shift the strips so that strip 0's complete range starts at or just before output column 0
    p->cshift = -((xa + p->S - 1) / p->S);
    if (p->S * p->cshift + xa > 0) p->cshift -= 1;
    // mean round-toward-zero loss of the accumulation chain: every MMA that adds a non-zero product truncates the accumulator
    // (1.67e-8 of its magnitude on average, tools/tc_calibrate2.py) -- the two cross-term MMAs of a K=8 slice as much as the
    // a_hi*w_hi one, while slices beyond the last real channel add exact zeros and lose nothing.  Checked by the mean signed error
    // of tests/test_ops_gpu.py::test_conv_taps_on_n_engine (< 1e-7 of the output scale for Ci = 40 .. 162).
    const char* nocomp = getenv("FN2_TC_COMP");
    p->comp = (nocomp && nocomp[0] == '0') ? 0.f : (RZ_COMP_A + 3.f * RZ_COMP_B * (float)((d->ci + 7) / 8));
    // shared memory: raw-A ring + W (resident if it all fits, else a ring of 2..3 stages) + barriers + output ring.  The ring is
    // flushed (written out + cleared, two barriers) every F tiles; a larger F needs (F-1) * th * S more ring rows.
    const int wstage = 2 * p->ngmax * 128;
    const int nwall = p->npass * p->cblocks;
    for (int F = 4; F >= 1; F--) {
        p->F = F; p->RR = span + (F - 1) * p->th * p->S;
        const int ring = p->RR * d->co * p->CW * 4;
        const int budget = 227 * 1024 - ring - 1024 - 256;
        p->RA = 4;
        if (p->RA * TN_A_BYTES + nwall * wstage <= budget) { p->wres = 1; p->RW = 0; return true; }
        p->wres = 0;
        p->RW = min(3, (budget - p->RA * TN_A_BYTES) / wstage);
        if (p->RW >= 3) return true;                 // a 2-deep W ring costs more than the rarer flush saves (measured)
        if (F == 1 && p->RW >= 2) return true;
        if (F == 1) { p->RA = 2; p->RW = min(3, (budget - p->RA * TN_A_BYTES) / wstage); return p->RW >= 2; }
    }
    return false;
}
static int tn_smem_bytes(const TnParams& p) {
    const int wstage = 2 * p.ngmax * 128;
    return p.RA * TN_A_BYTES + (p.wres ? p.npass * p.cblocks : p.RW) * wstage + 256 + p.RR * p.Co * p.CW * 4 + 1024;
}

}  // namespace

int conv_tn_applicable(const fn2_conv_desc* d) {
    TnParams p;
    return tn_layer_plan(d, &p) ? 1 : 0;
}

size_t conv_tn_packed_floats(const fn2_conv_desc* d) {
    TnParams p;
    if (!tn_layer_plan(d, &p)) return 0;
    return (size_t)2 * p.npass * p.cblocks * p.ngmax * 32;
}

int conv_tn_pack(const fn2_conv_desc* d, const float* w, float* wp, cudaStream_t st) {
    TnParams p;
    if (!tn_layer_plan(d, &p)) return FN2_OK;
    const long long per = (long long)p.npass * p.cblocks * p.ngmax * 32;
    tn_pack_kernel<<<ew_grid(per, 256), 256, 0, st>>>(w, wp, d->ci, d->co, d->kh, d->kw, d->deconv, p.cblocks, p.ngmax, p);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

// plan8 (fn2_conv_plan): {NT = -(accumulator columns of the widest pass), units, K blocks, mode 3 = taps on N, passes, strips, segments, 0}
int conv_tn_plan(const fn2_conv_desc* d, int N, int Ho, int Wo, int* out8) {
    TnParams p;
    if (!tn_layer_plan(d, &p)) return 0;
    const int nstrips = (Wo - (p.S * p.cshift + p.xa) + p.S * p.stepx - 1) / (p.S * p.stepx);
    out8[0] = -p.ngmax; out8[2] = p.cblocks; out8[3] = 3; out8[4] = p.npass; out8[5] = nstrips;
    return 1;
}

int conv_tn_forward(const fn2_conv_desc* d, const T4& in, const float* wp, const float* bias, const T4& out, cudaStream_t st) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("conv_tn: cuTensorMapEncodeTiled unavailable"); return FN2_ERR_CUDA; }
    TnParams p;
    if (!tn_layer_plan(d, &p)) { set_error("conv_tn: layer not eligible"); return FN2_ERR_INVALID; }
    p.N = in.n; p.Hin = in.h; p.Win = in.w; p.Ho = out.h; p.Wo = out.w;
    p.relu = d->relu; p.has_bias = d->has_bias; p.slope = d->negative_slope;
    p.out_sn = out.sn; p.out_sh = out.sh; p.out_sw = out.sw;
    p.nstrips = (p.Wo - (p.S * p.cshift + p.xa) + p.S * p.stepx - 1) / (p.S * p.stepx);
    // vertical segments: enough units to fill the SMs in (almost) whole rounds; every segment recomputes its halo rows
    const int nsm = num_sms();
    const long long cols = (long long)p.N * p.nstrips;
    int best_seg = 1; double best_cost = 1e30;
    const int halo = (p.oy_max - p.oy_min + p.S - 1) / p.S;            // extra input rows per segment
    for (int nseg = 1; nseg <= 64 && nseg * 8 <= p.Ho; nseg++) {
        const int rows_out = (p.Ho + nseg - 1) / nseg;
        const int tiles = (rows_out / p.S + halo + p.th - 1) / p.th + 1;
        const long long units = cols * nseg;
        const double cost = (double)((units + nsm - 1) / nsm) * tiles;
        if (cost < best_cost * 0.97) { best_cost = cost; best_seg = nseg; }
    }
    p.nseg = best_seg;
    p.seg_rows = (p.Ho + p.nseg - 1) / p.nseg;
    p.nseg = (p.Ho + p.seg_rows - 1) / p.seg_rows;
    p.total = p.N * p.nstrips * p.nseg;
    p.d_nseg.init(p.nseg); p.d_nstrips.init(p.nstrips);
    CUtensorMap mapA, mapW;
    {
        cuuint64_t dims[4] = {(cuuint64_t)in.c, (cuuint64_t)in.w, (cuuint64_t)in.h, (cuuint64_t)in.n};
        cuuint64_t strides[3] = {(cuuint64_t)in.sw * 4, (cuuint64_t)in.sh * 4, (cuuint64_t)in.sn * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)p.tw, (cuuint32_t)p.th, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&mapA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)in.p, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tn: activation tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    {
        const int nblk = p.npass * p.cblocks;
        cuuint64_t dims[4] = {32, (cuuint64_t)p.ngmax, (cuuint64_t)nblk, 2};
        cuuint64_t strides[3] = {32 * 4, (cuuint64_t)32 * p.ngmax * 4, (cuuint64_t)32 * p.ngmax * nblk * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)p.ngmax, 1, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&mapW, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)wp, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tn: weight tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    const int smem_bytes = tn_smem_bytes(p);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)min(p.total, nsm), 1, 1);
    cfg.blockDim = dim3(TN_THREADS);
    cfg.stream = st;
    cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
#define FN2_TN_LAUNCH(COV, SV)                                                                                          \
    {                                                                                                                   \
        static int set_ = 0;                                                                                            \
        if (set_ < smem_bytes) { FN2_CUDA(cudaFuncSetAttribute(conv_tn_kernel<COV, SV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes)); set_ = smem_bytes; } \
        FN2_CUDA(cudaLaunchKernelEx(&cfg, conv_tn_kernel<COV, SV>, mapA, mapW, bias, out.p, p));                        \
    }
    if (d->co == 16 && p.S == 1) FN2_TN_LAUNCH(16, 1)
    else if (d->co == 16) FN2_TN_LAUNCH(16, 2)
    else if (p.S == 1) FN2_TN_LAUNCH(32, 1)
    else FN2_TN_LAUNCH(32, 2)
#undef FN2_TN_LAUNCH
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

}  // namespace fn2
