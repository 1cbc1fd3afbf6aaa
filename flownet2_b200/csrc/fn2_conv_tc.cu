// tcgen05 / TMEM implicit-GEMM convolution + deconvolution engine (sm_100a), FP32-faithful.
//
// GEMM view per CTA: D[128 pixels x NT outputs] = sum over (kernel tap, 32-channel block) A_tap[128 x 32] * W_tap[NT x 32]^T
//   * A (activations, NHWC) : one TMA box per step straight from the activation tensor -- {32 ch, tw, th} with element
//     strides = conv stride and out-of-bounds zero fill, so padding, stride and the channel tail cost nothing and no
//     im2col buffer exists.  Lands as a K-major SWIZZLE_128B tile of raw FP32.
//   * W (weights) : packed once as [hi|lo][tap][Co][Ci32] (TF32 split), TMA boxes {32, NT}, K-major SWIZZLE_128B.
//   * 3xTF32: a = a_hi + a_lo, w = w_hi + w_lo (each rounded to TF32), D = a_hi*w_hi + a_hi*w_lo + a_lo*w_hi.
//     The activation split is done in-kernel by 4 converter warps that read the raw tile from shared memory and write
//     a_hi / a_lo into TENSOR MEMORY (tcgen05.st); the MMAs take A from TMEM (kind::tf32, "TS" form), which also keeps
//     shared-memory traffic (W reads + TMA writes) near the 128 B/clk budget.
//   * Accumulation: the B200 tensor core rounds its FP32 accumulator TOWARD ZERO (tools/tc_probe.cu: -1.7e-8 relative
//     per chained MMA), which over K up to 9216 and ~60 layers would shrink the flow by 1e-3.  Therefore the dominant
//     a_hi*w_hi term is accumulated in the tensor core only over short chains (kd K steps = 4*kd MMAs) into a
//     double-buffered TMEM accumulator that 4 drain warps pull out (tcgen05.ld) and add into FP32 REGISTERS with
//     round-to-nearest, applying the measured mean RZ loss of a chain of that length as a correction.  The two cross
//     terms (2^-11 smaller) accumulate in their own TMEM columns for the whole K loop of a tile (TcGeo).
//   * Epilogue from registers: + bias, leaky ReLU, 128-bit stores into the strided NHWC output view (or raw partials
//     into the workspace when the K loop is split over SMs).
// Persistent kernel, one CTA per SM walking the tile list (pixel tile x Co tile x deconv parity class x K split).
// Warp roles (384 threads, setmaxnreg re-balances registers): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM
// allocator, warps 4-7 converters, warps 8-11 drain + epilogue.  Small-Ci inputs use kernel-row or tap-group packing of
// the K blocks (tc_small_ci).  DESIGN.md section 3 has the measurements behind each of these choices.
#include <cuda.h>

#include "fn2_common.cuh"
#include "fn2_tc_ptx.cuh"

namespace fn2 {

namespace {

constexpr int TC_THREADS = 384;
constexpr int CORR_TR_STRIDE = 57;             // floats per pixel row of the correlation epilogue's transpose buffer (odd: no bank conflicts)
constexpr int A_TILE_BYTES = 128 * 128;          // 128 pixels x 32 fp32

struct TcParams {
    int N, su, sv, ou, ov;                        // sub-grid / mapping (see fn2_conv_nhwc.cu)
    int ncls;                                     // output parity classes handled by this launch (grid.z)
    int cls_Hu[4], cls_Wu[4], cls_oy0[4], cls_ox0[4], cls_tap0[4], cls_ntaps[4];
    int Co, cblocks;                              // cblocks = ceil(Ci / 32)
    long long out_sn, out_sh, out_sw;
    int relu, has_bias;
    float slope;
    int tw, th, tiles_x, tiles_y;
    int kd;                                       // channel blocks per tensor-core accumulation chain
    int splits, Ho, Wo;                           // split-K: K ranges per tile (partials go to the workspace), output size
    // tail split: the tiles of the last, partial wave [tail_first, ntotal) are cut into tail_z K ranges each so that they
    // spread over all SMs (448 tiles on 148 SMs: 3 + 1/8 rounds instead of 4); their partials are summed by a fix-up kernel
    int tail_first, tail_z, ntotal;
    FastDiv d_ntiles, d_cotiles, d_tiles_x, d_tiles_y, d_splits, d_tail_z;
    // Correlation on the same pipeline (corr_tc_forward): a unit = (sample, parity plane, 128-pixel tile of map 0, block of
    // cbw x cbh halo pixels of map 1); D[pixel][halo pixel] = <a, b> over C channels; the epilogue keeps the band that
    // lies inside the (2R+1)^2 displacement window.  W tiles are halo-pixel tiles of the pre-split map 1.
    int corr, cR, cS, cD, cbw, cbh, cnx, cnt;
    float cscale;
    int ntiles, cotiles, total;                   // pixel tiles, Co tiles, all tiles
    float comp_a, comp_b;                         // RZ bias model: shrink(n MMAs) = comp_a + comp_b * n
    int gcs;                                      // tap-group packing for Ci <= 16: padded channels per tap (4/8/12/16), 0 = off
    // kernel-row packing for Ci <= 16 on a dense input (pixel stride == rcs floats, guard band around the blob): the kw taps
    // of one kernel row are CONTIGUOUS in memory for every output pixel, so one K block = 32 consecutive floats of that run.
    int rowmode, rcs, rblocks, rsteps, rkw, rpad, rW;   // rblocks = ceil(kw*rcs/32) K blocks per kernel row, rsteps = kh*rblocks
    // Weight gradient on the same pipeline (conv_tc_wgrad): a unit = (kernel tap, 128 channels of the shifted map, NT channels of
    // the unshifted map, range of 32-pixel K segments); D[big channel][small channel] = sum over the segments' pixels.
    // Maps with few channels (wg_G = 8 .. 64 rows per tap) put 128 / wg_G taps side by side in one 128-row tile (wg_TPT).
    int wg_S, wg_ST, wg_BT, wg_segs, wg_segs_x, wg_sx, wg_G, wg_TPT, wg_taps;
    short dy[49], dx[49], widx[49];
};

// Tap-group packing (Ci <= 16): the stage holds up to 32/CS dense boxes [128 pixels][CS floats] (one per kernel tap);
// row m of K block = concatenation of its CS-channel slices, zero beyond the taps present.
template <int CS>
__device__ __forceinline__ void gather_taps(const unsigned char* base, int m, int nt, uint32_t* hi, uint32_t* lo) {
    constexpr int GS = 32 / CS;
#pragma unroll
    for (int j = 0; j < 32; j++) { hi[j] = 0; lo[j] = 0; }
#pragma unroll
    for (int j = 0; j < GS; j++) {
        if (j < nt) {
            const float4* row = reinterpret_cast<const float4*>(base + (size_t)j * (128 * CS * 4) + (size_t)m * (CS * 4));
#pragma unroll
            for (int q4 = 0; q4 < CS / 4; q4++) {
                const float4 v = row[q4];
                const float f[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const uint32_t h = to_tf32(f[e]);
                    hi[j * CS + 4 * q4 + e] = h;
                    lo[j * CS + 4 * q4 + e] = to_tf32(f[e] - __uint_as_float(h));
                }
            }
        }
    }
}

template <int NT> struct TcGeo {
    static constexpr int B_TILE_BYTES = NT * 128;
    static constexpr int STAGE_BYTES = A_TILE_BYTES + 2 * B_TILE_BYTES;
    // One ring of R entries: entry s = shared-memory stage s (raw A tile + W hi/lo tiles) + tensor-memory A slot s.
    // A single tcgen05.commit per step (done[s]) releases both: the MMAs of a step cannot start before the converters
    // have read the raw tile, so "MMAs of the step retired" also means the raw tile is free.  (Every tcgen05 op -- MMA
    // or commit -- costs the issuing thread ~64-78 cycles once the queue is full, see profiles/r01_prof_tc128_*.)
    static constexpr int R = NT >= 64 ? 4 : 6;
    static constexpr int SMEM = R * STAGE_BYTES + 1024;
    // tensor-memory columns.  Two chunk accumulators (double-buffered against the drain warps), then (NT == 128 only) the
    // cross-term accumulator, then the A slots.  The tensor core truncates on every accumulation, proportionally to the
    // accumulator's magnitude, so the dominant a_hi*w_hi chain is kept short (a chunk of kd steps, 4 MMAs per step) and
    // drained to FP32 registers, while the small cross terms a_hi*w_lo + a_lo*w_hi may chain over the whole tile.
    // NT == 128 (SEPX): cross terms in their own 128 columns (drained once per tile); only two A slots fit, which is
    //   enough because a converter only needs the MMAs of step i-2 retired before it stores step i.
    // NT <= 64 (WIDE): the W stage holds [w_hi rows ; w_lo rows] back to back, so ONE MMA with N = 2*NT computes
    //   a_hi*[w_hi|w_lo] into 2*NT columns and a second one adds a_lo*w_hi onto the last NT of them: 2 MMAs per K=8
    //   slice instead of 3 (with A in tensor memory an MMA costs >= 64 cycles however small N is).
    static constexpr bool WIDE = NT <= 64;
    static constexpr bool SEPX = !WIDE;
    static constexpr int ACCW = WIDE ? 2 * NT : NT;
    static constexpr int MMAS_PER_STEP = 4;                                        // length of the RZ chain per step
    static constexpr int COL_HH0 = 0, COL_HH1 = ACCW;
    static constexpr int COL_X = 2 * ACCW;                                         // SEPX only
    static constexpr int NSLOTS = SEPX ? 2 : R;                                    // must divide R
    static constexpr int COL_A = 512 - 64 * NSLOTS;                                // slot a: hi at COL_A + 64*a, lo at +32
    static_assert(2 * ACCW + (SEPX ? NT : 0) <= COL_A, "tensor memory overflow");
    static_assert(R % NSLOTS == 0, "slot ring must divide the stage ring");
};

// one output tile: 128 pixels (th x tw) of one sample and parity class, NT output channels
struct TcTile {
    int n, u0, v0, co0, cls, tap0, ntaps, steps;
    int k0, split;                                // first K step of this unit, split index
    int slot;                                     // >= 0: raw partial sums go to workspace slot `slot` (tail split)
    bool valid;
};
// MODE (compile time, so that each instantiation's role loops stay small -- the all-in-one kernel had ~1900 SASS instructions in
// the converter loop and stalled on instruction fetch): 0 plain K blocks, 1 tap groups, 2 kernel rows, 3 correlation
enum { TC_PLAIN = 0, TC_GROUP = 1, TC_ROW = 2, TC_CORR = 3, TC_WGRAD = 4 };

template <int NT, int MODE>
__device__ __forceinline__ TcTile tc_decode_tile(const TcParams& p, int tile) {
    TcTile t;
    t.split = 0; t.slot = -1;
    if constexpr (MODE == TC_CORR) {
        // unit -> (halo block, tile x, tile y, plane, sample); co0 carries the halo block, cls the parity plane
        int r = tile / p.cnt;
        t.co0 = tile - r * p.cnt;
        int q = r / p.tiles_x;
        const int tx = r - q * p.tiles_x;
        r = q / p.tiles_y;
        const int ty = q - r * p.tiles_y;
        const int planes = p.cS * p.cS;
        t.n = r / planes;
        t.cls = r - t.n * planes;
        t.u0 = ty * p.th; t.v0 = tx * p.tw;
        t.tap0 = 0; t.ntaps = 1; t.k0 = 0;
        t.steps = p.cblocks;
        const int py = t.cls / p.cS, px = t.cls % p.cS;
        t.valid = t.u0 * p.cS + py < p.Ho && t.v0 * p.cS + px < p.Wo;
        return t;
    }
    if constexpr (MODE == TC_WGRAD) {
        // unit -> (K range, small-channel tile, big-channel tile, tap); u0 carries the first big channel, slot the unit itself
        int q = tile / p.wg_S;
        t.split = tile - q * p.wg_S;
        const int q2 = q / p.wg_ST;
        t.co0 = (q - q2 * p.wg_ST) * NT;
        t.tap0 = q2 / p.wg_BT;
        t.u0 = (q2 - t.tap0 * p.wg_BT) * 128;
        t.tap0 *= p.wg_TPT;                                        // first tap of the group
        t.n = 0; t.v0 = 0; t.cls = 0; t.ntaps = 1; t.slot = tile; t.valid = true;
        const int per = (p.wg_segs + p.wg_S - 1) / p.wg_S;
        t.k0 = min(p.wg_segs, t.split * per);
        t.steps = min(p.wg_segs, t.k0 + per) - t.k0;
        return t;
    }
    int tseg = 0;
    if (p.tail_z > 1 && tile >= p.tail_first) {
        t.slot = tile - p.tail_first;
        int q;
        p.d_tail_z.divmod(t.slot, q, tseg);
        tile = p.tail_first + q;
    }
    if (p.splits > 1) { int q; p.d_splits.divmod(tile, q, t.split); tile = q; }   // splits of a tile run side by side (shared A tiles in L2)
    int pix, r, cot = 0;
    p.d_ntiles.divmod(tile, r, pix);
    t.cls = 0;
    if (r) p.d_cotiles.divmod(r, t.cls, cot);
    int tx, ty, q2;
    p.d_tiles_x.divmod(pix, q2, tx);
    p.d_tiles_y.divmod(q2, t.n, ty);
    t.u0 = ty * p.th; t.v0 = tx * p.tw;
    t.co0 = cot * NT;
    t.tap0 = p.cls_tap0[t.cls]; t.ntaps = p.cls_ntaps[t.cls];
    t.valid = t.u0 < p.cls_Hu[t.cls] && t.v0 < p.cls_Wu[t.cls];       // false: tile outside this (smaller) parity class
    const int gsz = MODE == TC_GROUP ? 32 / p.gcs : 1;
    t.steps = MODE == TC_ROW ? p.rsteps : (MODE == TC_GROUP ? (t.ntaps + gsz - 1) / gsz : t.ntaps * p.cblocks);
    t.k0 = 0;
    if (p.splits > 1) {
        const int per = (t.steps + p.splits - 1) / p.splits;
        t.k0 = min(t.steps, t.split * per);
        t.steps = min(t.steps, t.k0 + per) - t.k0;
    }
    if (t.slot >= 0) {
        const int per = (t.steps + p.tail_z - 1) / p.tail_z;
        t.k0 = min(t.steps, tseg * per);
        t.steps = min(t.steps, t.k0 + per) - t.k0;
    }
    return t;
}

// Persistent kernel: gridDim.x CTAs (one per SM) walk the tile list with stride gridDim.x; the barrier rings and the two
// accumulator buffers run straight through tile boundaries, so the loads / conversions / MMAs of the next tile overlap
// the drain + epilogue of the current one.
template <int NT, int MODE>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW, const float* __restrict__ bias,
               float* __restrict__ out, float* __restrict__ ws, const TcParams p) {
    using G = TcGeo<NT>;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + G::R * G::STAGE_BYTES);
    uint64_t* full = bars;                         // [R]  TMA bytes of the stage have landed
    uint64_t* a_ready = bars + G::R;               // [R]  converters have written the A slot
    uint64_t* done = bars + 2 * G::R;              // [R]  MMAs of the step have retired: stage + slot are free
    uint64_t* acc_full = bars + 3 * G::R;          // [2]
    uint64_t* acc_free = acc_full + 2;             // [2]
    uint64_t* x_free = acc_free + 2;               // [1]  drain has read the cross-term accumulator of the previous tile
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x_free + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // Programmatic dependent launch: let the next kernel of the stream be scheduled as soon as every CTA of this one is
    // running, so that its CTAs take over SMs the moment ours exit and run their prologue (barrier init, TMEM allocation)
    // there; it blocks in griddepcontrol.wait (below, before its first global access) until this grid has completed.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int gsz = MODE == TC_GROUP ? 32 / p.gcs : 1;   // taps per K block when packing

    if (tid == 0) {
        for (int s = 0; s < G::R; s++) { mbar_init(&full[s], 1); mbar_init(&a_ready[s], 128); mbar_init(&done[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], 128); }
        mbar_init(x_free, 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(su32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    asm volatile("griddepcontrol.wait;" ::: "memory");      // no-op unless launched with programmatic stream serialization

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");
        if (warp == 0 && lane == 0) {
            // ===== TMA producer (running counters instead of per-step divisions: this single thread's instruction chain
            // paces the whole pipeline) =====
            const int cblocks = p.cblocks, gcs = p.gcs;
            int s = 0; uint32_t ph = 1u;                // ph: parity to wait on done[s]
            for (int tile = blockIdx.x; tile < p.total; tile += gridDim.x) {
                const TcTile T = tc_decode_tile<NT, MODE>(p, tile);
                if (!T.valid) continue;
                const int cx0 = T.v0 * p.su, cy0 = T.u0 * p.sv;
                auto load_w = [&](unsigned char* st, uint64_t* bar, int c0, int blk) {
                    tma_load_4d(st + A_TILE_BYTES, &mapW, bar, c0, T.co0, blk, 0);
                    tma_load_4d(st + A_TILE_BYTES + G::B_TILE_BYTES, &mapW, bar, c0, T.co0, blk, 1);
                };
                if constexpr (MODE == TC_CORR) {
                    const int py = T.cls / p.cS, px = T.cls % p.cS;
                    const int ax = T.v0 * p.cS + px, ay = T.u0 * p.cS + py;
                    const int bx = (T.v0 - p.cR) * p.cS + px, by = (T.u0 - p.cR + T.co0 * p.cbh) * p.cS + py;
                    const uint32_t bbytes = (uint32_t)(p.cbw * p.cbh * 128);
#pragma unroll 1
                    for (int i = 0; i < T.steps; i++) {
                        mbar_wait(&done[s], ph);
                        unsigned char* st = smem + (size_t)s * G::STAGE_BYTES;
                        mbar_expect_tx(&full[s], (uint32_t)A_TILE_BYTES + 2u * bbytes);
                        tma_load_4d(st, &mapA, &full[s], i * 32, ax, ay, T.n);
                        tma_load_4d(st + A_TILE_BYTES, &mapW, &full[s], i * 32, bx, by, T.n);
                        tma_load_4d(st + A_TILE_BYTES + G::B_TILE_BYTES, &mapW, &full[s], i * 32, bx, by, p.N + T.n);
                        if (++s == G::R) { s = 0; ph ^= 1u; }
                    }
                } else if constexpr (MODE == TC_WGRAD) {
                    // K segment = 32 consecutive output columns of one output row of one sample.  A: the tap's shifted window of
                    // the big map, 128 channel rows x 32 pixels (column-parity plane widx[tap], so that a strided convolution
                    // still reads consecutive floats); B: the same 32 pixels of the small map's hi and lo planes.
                    // (TMA needs the innermost coordinate on a 16-byte boundary: the big map is stored in 4 copies delayed by 0..3
                    // columns, widx[tap] >> 4 picks the copy that makes the tap's column shift a multiple of 4.)
                    int xs = T.k0 % p.wg_segs_x, r = T.k0 / p.wg_segs_x;
                    int oy = r % p.Ho, n = r / p.Ho;
                    const int tpt = p.wg_TPT, gbytes = p.wg_G * 128;
#pragma unroll 1
                    for (int i = 0; i < T.steps; i++) {
                        mbar_wait(&done[s], ph);
                        unsigned char* st = smem + (size_t)s * G::STAGE_BYTES;
                        mbar_expect_tx(&full[s], (uint32_t)G::STAGE_BYTES);
                        for (int j = 0; j < tpt; j++) {
                            // a group past the last tap repeats tap 0 (its rows are never read back)
                            const int tap = T.tap0 + j < p.wg_taps ? T.tap0 + j : 0;
                            tma_load_4d(st + j * gbytes, &mapA, &full[s], xs * 32 + p.dx[tap], (oy * p.sv + p.dy[tap]) * p.wg_sx + (p.widx[tap] & 15),
                                        T.u0, (p.widx[tap] >> 4) * p.N + n);
                        }
                        tma_load_4d(st + A_TILE_BYTES, &mapW, &full[s], xs * 32, oy, T.co0, n);
                        tma_load_4d(st + A_TILE_BYTES + G::B_TILE_BYTES, &mapW, &full[s], xs * 32, oy, T.co0, p.N + n);
                        if (++xs == p.wg_segs_x) { xs = 0; if (++oy == p.Ho) { oy = 0; ++n; } }
                        if (++s == G::R) { s = 0; ph ^= 1u; }
                    }
                } else if constexpr (MODE == TC_ROW) {
                    // one box per step: {32 floats of the kernel-row run, tw output pixels (stride su pixels), th rows}
                    int r = 0, kb = 0;
#pragma unroll 1
                    for (int i = 0; i < T.steps; i++) {
                        mbar_wait(&done[s], ph);
                        unsigned char* st = smem + (size_t)s * G::STAGE_BYTES;
                        mbar_expect_tx(&full[s], (uint32_t)G::STAGE_BYTES);
                        tma_load_4d(st, &mapA, &full[s], kb * 32, T.v0, cy0 + p.dy[r * p.rkw], T.n);
                        load_w(st, &full[s], 0, i);
                        if (++kb == p.rblocks) { kb = 0; ++r; }
                        if (++s == G::R) { s = 0; ph ^= 1u; }
                    }
                } else if constexpr (MODE == TC_GROUP) {
                    // several taps share one 32-wide K block: one small box {gcs channels, tw, th} per tap
                    const int box_bytes = 128 * gcs * 4;
                    for (int i = 0, t0 = 0; i < T.steps; i++, t0 += gsz) {
                        mbar_wait(&done[s], ph);
                        unsigned char* st = smem + (size_t)s * G::STAGE_BYTES;
                        const int nt = min(gsz, T.ntaps - t0);
                        mbar_expect_tx(&full[s], (uint32_t)(nt * box_bytes + 2 * G::B_TILE_BYTES));
                        for (int j = 0; j < nt; j++) {
                            const int t = T.tap0 + t0 + j;
                            tma_load_4d(st + j * box_bytes, &mapA, &full[s], 0, cx0 + p.dx[t], cy0 + p.dy[t], T.n);
                        }
                        load_w(st, &full[s], 0, i);
                        if (++s == G::R) { s = 0; ph ^= 1u; }
                    }
                } else {
                    int t = T.tap0 + T.k0 / cblocks, cb = T.k0 % cblocks;
                    int cx = cx0 + p.dx[t], cy = cy0 + p.dy[t], wi = p.widx[t];
#pragma unroll 1
                    for (int i = 0; i < T.steps; i++) {
                        mbar_wait(&done[s], ph);
                        unsigned char* st = smem + (size_t)s * G::STAGE_BYTES;
                        mbar_expect_tx(&full[s], (uint32_t)G::STAGE_BYTES);
                        tma_load_4d(st, &mapA, &full[s], cb * 32, cx, cy, T.n);
                        load_w(st, &full[s], cb * 32, wi);
                        if (++cb == cblocks && i + 1 < T.steps) { cb = 0; ++t; cx = cx0 + p.dx[t]; cy = cy0 + p.dy[t]; wi = p.widx[t]; }
                        if (++s == G::R) { s = 0; ph ^= 1u; }
                    }
                }
            }
        } else if (warp == 1) {
            // ===== MMA issuer: the whole warp runs the loop convergently (so descriptors live in uniform registers),
            // one elected lane issues the tcgen05 instructions =====
            // correlation: N = the halo block's pixel count (a multiple of 16), not the full NT
            const uint32_t idesc = make_idesc_tf32(128, MODE == TC_CORR ? p.cbw * p.cbh : NT), idesc_w = make_idesc_tf32(128, G::ACCW);
            const int kd = p.kd;
            int s = 0, buf = 0;
            uint32_t ph = 0, pacc = 1u;                 // pacc: parity to wait on acc_free[buf] (flips every second chunk)
            uint32_t px = 1u;                           // parity to wait on x_free (one phase per tile)
            for (int tile = blockIdx.x; tile < p.total; tile += gridDim.x) {
                const TcTile T = tc_decode_tile<NT, MODE>(p, tile);
                if (!T.valid) continue;
                int in_chunk = 0;
                if (G::SEPX && T.steps > 0) { mbar_wait(x_free, px); px ^= 1u; }
#pragma unroll 1
                for (int i = 0; i < T.steps; i++) {
                    if (in_chunk == 0) mbar_wait(&acc_free[buf], pacc);
                    mbar_wait(&full[s], ph);
                    mbar_wait(&a_ready[s], ph);
                    fence_after();
                    const uint32_t bh = su32(smem + (size_t)s * G::STAGE_BYTES + A_TILE_BYTES);
                    const uint64_t dbh0 = make_desc_sw128(bh), dbl0 = make_desc_sw128(bh + G::B_TILE_BYTES);
                    const uint32_t a_hi = tmem + G::COL_A + 64 * (s % G::NSLOTS), a_lo = a_hi + 32;
                    const uint32_t d = tmem + (buf ? G::COL_HH1 : G::COL_HH0);
                    const bool chunk_end = (in_chunk == kd - 1) || (i == T.steps - 1);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; kk++) {
                            // +2 in the start-address field = +32 bytes = the next 8 TF32 columns of the swizzled tile
                            if constexpr (G::WIDE) {
                                mma_tf32_ts(d, a_hi + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc_w, (in_chunk | kk) != 0);
                                mma_tf32_ts(d + NT, a_lo + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc, 1);
                            } else {
                                mma_tf32_ts(d, a_hi + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc, (in_chunk | kk) != 0);
                                mma_tf32_ts(tmem + G::COL_X, a_hi + kk * 8, dbl0 + (uint64_t)(2 * kk), idesc, (i | kk) != 0);
                                mma_tf32_ts(tmem + G::COL_X, a_lo + kk * 8, dbh0 + (uint64_t)(2 * kk), idesc, 1);
                            }
                        }
                        mma_commit(&done[s]);
                        if (chunk_end) mma_commit(&acc_full[buf]);
                    }
                    __syncwarp();
                    if (++s == G::R) { s = 0; ph ^= 1u; }
                    if (chunk_end) { in_chunk = 0; if (buf) pacc ^= 1u; buf ^= 1; } else ++in_chunk;
                }
            }
        }
    } else if (warp < 8) {
        // ===== converters: raw FP32 tile (smem, swizzled) -> a_hi / a_lo in tensor memory =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 136;" ::: "memory");
        const int q = warp & 3;
        const int m = q * 32 + lane;               // tile row == TMEM lane
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        int s = 0, s_prev = -1;
        uint32_t ph = 0;                           // full[s] parity; done[s] is waited with ph ^ 1
        for (int tile = blockIdx.x; tile < p.total; tile += gridDim.x) {
            const TcTile T = tc_decode_tile<NT, MODE>(p, tile);
            if (!T.valid) continue;
#pragma unroll 1
            for (int i = 0; i < T.steps; i++) {
                mbar_wait(&full[s], ph);
                const float4* row = reinterpret_cast<const float4*>(smem + (size_t)s * G::STAGE_BYTES + m * 128);
                uint32_t hi[32], lo[32];
                float4 raw[8];
                if constexpr (MODE != TC_GROUP) {
#pragma unroll
                    for (int j = 0; j < 8; j++) raw[j] = row[j ^ (m & 7)];
                }
                if (s_prev >= 0) {
                    // publish the previous step's slot: its TMEM stores had the barrier wait + the loads above to land
                    tmem_wait_st();
                    fence_before();
                    mbar_arrive(&a_ready[s_prev]);
                }
                if constexpr (MODE == TC_GROUP) {
                    const int nt = min(gsz, T.ntaps - i * gsz);
                    const unsigned char* base = smem + (size_t)s * G::STAGE_BYTES;
                    if (p.gcs == 4) gather_taps<4>(base, m, nt, hi, lo);
                    else if (p.gcs == 8) gather_taps<8>(base, m, nt, hi, lo);
                    else if (p.gcs == 12) gather_taps<12>(base, m, nt, hi, lo);
                    else gather_taps<16>(base, m, nt, hi, lo);
                } else if constexpr (MODE == TC_ROW) {
                    // row mode: taps that fall outside the image row (and the K padding) hold whatever follows in memory
                    const int x0 = (T.v0 + m % p.tw) * p.su - p.rpad;            // input column of tap 0
                    const int kb32 = (i % p.rblocks) * 32;
                    const int k_lo = max(0, -x0) * p.rcs - kb32;
                    const int k_hi = min(p.rkw, p.rW - x0) * p.rcs - kb32;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const bool keep = 4 * j >= k_lo && 4 * j < k_hi;
                        const float f[4] = {raw[j].x, raw[j].y, raw[j].z, raw[j].w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const uint32_t h = keep ? to_tf32(f[e]) : 0u;
                            hi[4 * j + e] = h;
                            lo[4 * j + e] = keep ? to_tf32(f[e] - __uint_as_float(h)) : 0u;
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float f[4] = {raw[j].x, raw[j].y, raw[j].z, raw[j].w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const uint32_t h = to_tf32(f[e]);
                            hi[4 * j + e] = h;
                            lo[4 * j + e] = to_tf32(f[e] - __uint_as_float(h));
                        }
                    }
                }
                // the MMAs that read this A slot NSLOTS steps ago must have retired
                if (s >= G::NSLOTS) mbar_wait(&done[s - G::NSLOTS], ph);
                else mbar_wait(&done[s - G::NSLOTS + G::R], ph ^ 1u);
                fence_after();
                tmem_st32(lane_addr + G::COL_A + 64 * (s % G::NSLOTS), hi);
                tmem_st32(lane_addr + G::COL_A + 64 * (s % G::NSLOTS) + 32, lo);
                s_prev = s;
                if (++s == G::R) { s = 0; ph ^= 1u; }
            }
        }
        if (s_prev >= 0) {
            tmem_wait_st();
            fence_before();
            mbar_arrive(&a_ready[s_prev]);
        }
    } else {
        // ===== drain + epilogue: TMEM accumulators -> FP32 registers (round to nearest) -> global =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const int yy = m / p.tw, xx = m % p.tw;
        int buf = 0; uint32_t pfull = 0;           // pfull: parity to wait on acc_full[buf]
        for (int tile = blockIdx.x; tile < p.total; tile += gridDim.x) {
            const TcTile T = tc_decode_tile<NT, MODE>(p, tile);
            if (!T.valid) continue;
            float acc[NT];
#pragma unroll
            for (int j = 0; j < NT; j++) acc[j] = 0.f;
            const int chunks = (T.steps + p.kd - 1) / p.kd;
#pragma unroll 1
            for (int c = 0; c < chunks; c++) {
                const int nsteps = min(p.kd, T.steps - c * p.kd);
                // mean RZ shrink of the accumulation chain of this chunk
                const float comp = p.comp_a + p.comp_b * (float)(G::MMAS_PER_STEP * nsteps);
                mbar_wait(&acc_full[buf], pfull);
                fence_after();
                const uint32_t src = lane_addr + (buf ? G::COL_HH1 : G::COL_HH0);
                if constexpr (NT == 128) {
#pragma unroll
                    for (int j0 = 0; j0 < NT; j0 += 64) {
                        uint32_t v0[32], v1[32];
                        tmem_ld32(src + j0, v0);
                        tmem_ld32(src + j0 + 32, v1);
                        tmem_wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const float a = __uint_as_float(v0[j]), b = __uint_as_float(v1[j]);
                            acc[j0 + j] += fmaf(a, comp, a);
                            acc[j0 + 32 + j] += fmaf(b, comp, b);
                        }
                    }
                } else if constexpr (NT == 64) {
                    // columns [0,64): a_hi*w_hi, columns [64,128): a_hi*w_lo + a_lo*w_hi
#pragma unroll
                    for (int j0 = 0; j0 < 64; j0 += 32) {
                        uint32_t v0[32], v1[32];
                        tmem_ld32(src + j0, v0);
                        tmem_ld32(src + 64 + j0, v1);
                        tmem_wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const float a = __uint_as_float(v0[j]);
                            acc[j0 + j] += fmaf(a, comp, a) + __uint_as_float(v1[j]);
                        }
                    }
                } else if constexpr (NT == 32) {
                    uint32_t v0[32], v1[32];
                    tmem_ld32(src, v0);
                    tmem_ld32(src + 32, v1);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const float a = __uint_as_float(v0[j]);
                        acc[j] += fmaf(a, comp, a) + __uint_as_float(v1[j]);
                    }
                } else {
                    uint32_t v0[32];
                    tmem_ld32(src, v0);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const float a = __uint_as_float(v0[j]);
                        acc[j] += fmaf(a, comp, a) + __uint_as_float(v0[16 + j]);
                    }
                }
                fence_before();
                mbar_arrive(&acc_free[buf]);
                if (buf) pfull ^= 1u;
                buf ^= 1;
            }
            if constexpr (G::SEPX) {
                // cross terms of the whole tile (the last chunk's commit also covers them)
                if (T.steps > 0) {
#pragma unroll
                    for (int j0 = 0; j0 < NT; j0 += 64) {
                        uint32_t v0[32], v1[32];
                        tmem_ld32(lane_addr + G::COL_X + j0, v0);
                        tmem_ld32(lane_addr + G::COL_X + j0 + 32, v1);
                        tmem_wait_ld();
#pragma unroll
                        for (int j = 0; j < 32; j++) { acc[j0 + j] += __uint_as_float(v0[j]); acc[j0 + 32 + j] += __uint_as_float(v1[j]); }
                    }
                    fence_before();
                    mbar_arrive(x_free);
                }
            }
            // epilogue
            if constexpr (MODE == TC_CORR) {
                // A halo block = cbh full halo rows (cbw = tw + 2R pixels each): for every tile pixel it holds cbh
                // displacement rows dy with all D = 2R+1 values of dx, i.e. runs of D consecutive output channels.  Lanes
                // are pixels after tcgen05.ld, so the block goes through shared memory (two halves of cbh/2 halo rows) and
                // is written with lanes = channels: one coalesced run per (pixel, dy).
                if constexpr (NT == 128) {
                    float* tr = reinterpret_cast<float*>(smem + G::SMEM);            // [128 pixels][CORR_TR_STRIDE]
                    const int py = T.cls / p.cS, px = T.cls % p.cS;
                    const int wq = warp & 3;
                    const bool lane_on = lane < p.cD;
#pragma unroll
                    for (int h = 0; h < 2; h++) {
#pragma unroll
                        for (int j = 0; j < 56; j++) tr[m * CORR_TR_STRIDE + j] = acc[h * 56 + j] * p.cscale;
                        asm volatile("bar.sync 1, 128;" ::: "memory");
                        // warp wq stores tile rows qy = wq, wq+4, ...: 8 pixels x 2 displacement rows each, lanes = dx
                        const int dy_base = T.co0 * 4 + h * 2 - p.cR;
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const int qy = wq + 4 * k;
                            const int y = (T.u0 + qy) * p.cS + py;
                            const int dy0 = dy_base - qy, dy1 = dy0 + 1;
                            const bool ok0 = lane_on && y < p.Ho && dy0 >= -p.cR && dy0 <= p.cR;
                            const bool ok1 = lane_on && y < p.Ho && dy1 >= -p.cR && dy1 <= p.cR;
                            float* o = out + T.n * p.out_sn + (long long)y * p.out_sh + (long long)(T.v0 * p.cS + px) * p.out_sw + lane;
                            const float* t = tr + (qy * 8) * CORR_TR_STRIDE + lane;
                            const int c0 = (dy0 + p.cR) * p.cD, c1 = (dy1 + p.cR) * p.cD;
#pragma unroll
                            for (int qx = 0; qx < 8; qx++) {
                                const bool inx = (T.v0 + qx) * p.cS + px < p.Wo;
                                const float v0 = lane_on ? t[qx * CORR_TR_STRIDE + qx] : 0.f, v1 = lane_on ? t[qx * CORR_TR_STRIDE + 28 + qx] : 0.f;
                                if (ok0 && inx) o[(long long)qx * p.cS * p.out_sw + c0] = v0;
                                if (ok1 && inx) o[(long long)qx * p.cS * p.out_sw + c1] = v1;
                            }
                        }
                        asm volatile("bar.sync 1, 128;" ::: "memory");
                    }
                }
                continue;
            }
            if constexpr (MODE == TC_WGRAD) {
                // raw partial sums of this unit, [unit][128 big channels][NT small channels]; conv_tc_wgrad's reduction sums the
                // K ranges in a fixed order and scatters into the Caffe weight layout
                float* o = ws + ((long long)T.slot * 128 + m) * NT;
#pragma unroll
                for (int j = 0; j < NT; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
                continue;
            }
            const int u = T.u0 + yy, v = T.v0 + xx;
            if (T.valid && u < p.cls_Hu[T.cls] && v < p.cls_Wu[T.cls]) {
                const int oy = u * p.ou + p.cls_oy0[T.cls], ox = v * p.ov + p.cls_ox0[T.cls];
                if (T.slot >= 0) {
                    // tail split: raw partial sums of this K range, [slot][128 pixels][NT]
                    float* o = ws + ((long long)T.slot * 128 + m) * NT;
#pragma unroll
                    for (int j = 0; j < NT; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
                } else if (p.splits > 1) {
                    // raw partial sums, dense [split][n][oy][ox][Co]; bias / ReLU are applied by the fixed-order reduction
                    float* o = ws + ((((long long)T.split * p.N + T.n) * p.Ho + oy) * p.Wo + ox) * p.Co + T.co0;
#pragma unroll
                    for (int j = 0; j < NT; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
                } else {
                    float* o = out + T.n * p.out_sn + (long long)oy * p.out_sh + (long long)ox * p.out_sw + T.co0;
#pragma unroll
                    for (int j = 0; j < NT; j += 4) {
                        float r[4];
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            float x = acc[j + e];
                            if (p.has_bias) x += __ldg(bias + T.co0 + j + e);
                            if (p.relu) x = x > 0 ? x : x * p.slope;
                            r[e] = x;
                        }
                        *reinterpret_cast<float4*>(o + j) = make_float4(r[0], r[1], r[2], r[3]);
                    }
                }
            }
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

// ---- weight packing: Caffe layout -> [hi|lo][tap][Co][Ci32] with the TF32 split -------------------------------------
__global__ void tc_pack_kernel(const float* __restrict__ w, float* __restrict__ wp, int Ci, int Co, int kh, int kw, int cip, int deconv) {
    const long long per = (long long)kh * kw * Co * cip;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int ci = (int)(idx % cip);
        long long r_ = idx / cip;
        const int co = (int)(r_ % Co);
        const int t = (int)(r_ / Co);
        const int r = t / kw, s = t % kw;
        float v = 0.f;
        if (ci < Ci) v = deconv ? w[(((long long)ci * Co + co) * kh + r) * kw + s] : w[(((long long)co * Ci + ci) * kh + r) * kw + s];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
        const float hi = __uint_as_float(h);
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - hi));
        wp[idx] = hi;
        wp[per + idx] = __uint_as_float(l);
    }
}

// group-packed weights for Ci <= 16: [hi|lo][group][Co][32], K index = j*CS + ci for tap = group*(32/CS) + j
__global__ void tc_pack_group_kernel(const float* __restrict__ w, float* __restrict__ wp, int Ci, int Co, int kh, int kw, int cs, int ngroups) {
    const long long per = (long long)ngroups * Co * 32;
    const int gs = 32 / cs;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(idx % 32);
        long long r_ = idx / 32;
        const int co = (int)(r_ % Co);
        const int g = (int)(r_ / Co);
        const int j = k / cs, ci = k % cs;
        const int t = g * gs + j;
        float v = 0.f;
        if (j < gs && t < kh * kw && ci < Ci) v = w[(((long long)co * Ci + ci) * kh + t / kw) * kw + t % kw];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
        const float hi = __uint_as_float(h);
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - hi));
        wp[idx] = hi;
        wp[per + idx] = __uint_as_float(l);
    }
}

// row-packed weights for Ci <= 16: [hi|lo][r*rblocks + kb][Co][32], K index kb*32 + k = s*cs + ci of kernel row r
__global__ void tc_pack_row_kernel(const float* __restrict__ w, float* __restrict__ wp, int Ci, int Co, int kh, int kw, int cs, int rblocks) {
    const long long per = (long long)kh * rblocks * Co * 32;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(idx % 32);
        long long r_ = idx / 32;
        const int co = (int)(r_ % Co);
        const int blk = (int)(r_ / Co);
        const int r = blk / rblocks, kk = (blk % rblocks) * 32 + k;
        const int sx = kk / cs, ci = kk % cs;
        float v = 0.f;
        if (sx < kw && ci < Ci) v = w[(((long long)co * Ci + ci) * kh + r) * kw + sx];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
        const float hi = __uint_as_float(h);
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(v - hi));
        wp[idx] = hi;
        wp[per + idx] = __uint_as_float(l);
    }
}

// fixed-order sum of the split-K partials + bias + ReLU (4 channels per thread)
__global__ void tc_splitk_reduce_kernel(const float* __restrict__ ws, const float* __restrict__ bias, float* __restrict__ out, TcParams p) {
    const int c4 = p.Co / 4;
    const long long per = (long long)p.N * p.Ho * p.Wo * c4;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % c4) * 4;
        long long m = idx / c4;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int z = 0; z < p.splits; z++) {
            const float4 v = *reinterpret_cast<const float4*>(ws + ((long long)z * p.N * p.Ho * p.Wo + m) * p.Co + c);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        if (p.has_bias) { a.x += __ldg(bias + c); a.y += __ldg(bias + c + 1); a.z += __ldg(bias + c + 2); a.w += __ldg(bias + c + 3); }
        if (p.relu) {
            a.x = a.x > 0 ? a.x : a.x * p.slope; a.y = a.y > 0 ? a.y : a.y * p.slope;
            a.z = a.z > 0 ? a.z : a.z * p.slope; a.w = a.w > 0 ? a.w : a.w * p.slope;
        }
        const int ox = (int)(m % p.Wo); m /= p.Wo;
        const int oy = (int)(m % p.Ho);
        const int n = (int)(m / p.Ho);
        *reinterpret_cast<float4*>(out + n * p.out_sn + (long long)oy * p.out_sh + (long long)ox * p.out_sw + c) = a;
    }
}

// fix-up of the tail split: fixed-order sum of the tail_z partial tiles + bias + ReLU, one thread per (tile row, 4 channels)
template <int NT>
__global__ void tc_tail_reduce_kernel(const float* __restrict__ ws, const float* __restrict__ bias, float* __restrict__ out, TcParams p) {
    const int ntail = p.ntotal - p.tail_first;
    const long long per = (long long)ntail * 128 * (NT / 4);
    TcParams q = p;
    q.tail_z = 1;                                  // decode whole tiles
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < per; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % (NT / 4)) * 4;
        const int m = (int)((idx / (NT / 4)) % 128);
        const int t = (int)(idx / ((NT / 4) * 128));
        const TcTile T = tc_decode_tile<NT, TC_PLAIN>(q, p.tail_first + t);     // the tail split only exists in plain mode
        const int u = T.u0 + m / p.tw, v = T.v0 + m % p.tw;
        if (!T.valid || u >= p.cls_Hu[T.cls] || v >= p.cls_Wu[T.cls]) continue;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int z = 0; z < p.tail_z; z++) {
            const float4 x = *reinterpret_cast<const float4*>(ws + (((long long)t * p.tail_z + z) * 128 + m) * NT + c);
            a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w;
        }
        const int co = T.co0 + c;
        if (p.has_bias) { a.x += __ldg(bias + co); a.y += __ldg(bias + co + 1); a.z += __ldg(bias + co + 2); a.w += __ldg(bias + co + 3); }
        if (p.relu) {
            a.x = a.x > 0 ? a.x : a.x * p.slope; a.y = a.y > 0 ? a.y : a.y * p.slope;
            a.z = a.z > 0 ? a.z : a.z * p.slope; a.w = a.w > 0 ? a.w : a.w * p.slope;
        }
        const int oy = u * p.ou + p.cls_oy0[T.cls], ox = v * p.ov + p.cls_ox0[T.cls];
        *reinterpret_cast<float4*>(out + T.n * p.out_sn + (long long)oy * p.out_sh + (long long)ox * p.out_sw + co) = a;
    }
}

int tc_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("FN2_TC");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v;
}

// Accumulation chains of the conv forward and weight gradient (tiles of NT columns) and of the correlation (corr).  The
// a_hi*w_hi product is chained in the tensor core over kd K steps (4 MMAs each) and then drained to FP32 registers: 24 (NT =
// 128) or 16 MMAs per chain keep the end-to-end flow error equal to the FP32 SIMT engine's; the correlation chains a whole
// unit (4 * C/32 MMAs).  The drain adds back the mean round-toward-zero loss of the chain, comp_a + comp_b * n for n MMAs
// (tools/tc_probe.cu test3, tools/tc_calibrate2.py); a per-binade (ulp) model was measured too and is no better, and the
// residual after removing the mean (~half the loss, growing linearly with n) is what bounds kd.
// FN2_TC_KD (NT = 128, correlation) / FN2_TC_KDW (narrower tiles) override kd; FN2_TC_COMP=0 turns the compensation off.
void tc_chain_model(TcParams& p, int NT, bool corr) {
    p.kd = corr ? p.cblocks : (NT == 128 ? 6 : 4);
    if (const char* e = getenv(NT == 128 ? "FN2_TC_KD" : "FN2_TC_KDW")) { const int v = atoi(e); if (v >= 1 && v <= 1024) p.kd = v; }
    const char* nocomp = getenv("FN2_TC_COMP");
    const bool off = nocomp && nocomp[0] == '0';
    p.comp_a = off ? 0.f : RZ_COMP_A;
    p.comp_b = off ? 0.f : RZ_COMP_B;
}

}  // namespace

// Small-Ci packing (plain convolutions with at most 16 input channels): mode 1 = tap groups (several taps share a 32-wide
// K block, one small TMA box per tap), mode 2 = kernel rows (needs a dense input whose pixel stride equals the padded
// channel count, and a guard band around the tensor because the row runs of the edge pixels reach a little outside it).
struct TcSmallCi { int mode, cs, gs, ngroups, rblocks; };
static TcSmallCi tc_small_ci(const fn2_conv_desc* d, int ci_stride) {
    TcSmallCi m = {0, 0, 0, 0, 0};
    if (d->deconv || d->ci > 16 || d->kh * d->kw < 2) return m;
    m.cs = (d->ci + 3) / 4 * 4;
    m.gs = 32 / m.cs;
    m.ngroups = (d->kh * d->kw + m.gs - 1) / m.gs;
    m.rblocks = (d->kw * m.cs + 31) / 32;
    m.mode = 1;
    if (d->input_guard_bytes >= 512 && ci_stride == m.cs && d->kh * m.rblocks <= m.ngroups) m.mode = 2;
    return m;
}

// Split-K plan: layers whose tile list cannot fill the GPU (the 7x16 .. 14x32 maps of conv5/conv6/deconv5 with
// K = 9 * 1024) cut every tile's K loop into `z` ranges that run on different SMs.
// tail split plan for a layer with `tiles` tile units of `steps` K steps each: returns z (1 = off) and the first tail tile
static int tc_tail_plan(long long tiles, int steps, int* first, int NT = 128) {
    *first = (int)tiles;
    const int nsm = num_sms();
    if (steps < 16) return 1;                       // (tiles <= nsm: everything is "tail" -- 112 tiles become 560 fifths on 148 SMs)
    const long long full = tiles / nsm * nsm, r = tiles - full;
    if (r == 0) return 1;
    // cost model in units of one tile's time: rounds of whole tiles + rounds of 1/z tiles + the fix-up kernel reading r*z
    // partial tiles (128 x NT floats each at ~3 TB/s; a tile takes ~1400 cycles per K step at 1.9 GHz)
    const double tile_s = steps * 1400.0 / 1.9e9, part_s = 128.0 * NT * 4 / 3e12 + 2e-9;
    const double now = (double)((tiles + nsm - 1) / nsm);
    double best = now * 0.94;
    int bz = 1;
    for (int z = 2; z <= min(8, steps / 8); z++) {
        const double then = (double)(full / nsm) + (double)((r * z + nsm - 1) / nsm) / z + (r * z * part_s + 4e-6) / tile_s;
        if (then < best) { best = then; bz = z; }
    }
    if (bz < 2) return 1;
    *first = (int)full;
    return bz;
}
// tile count / K steps of a layer (same tiling rules as conv_tc_forward)
static void tc_layer_geometry(const fn2_conv_desc* d, int N, int Ho, int Wo, int* NTo, long long* tiles, int* steps) {
    const int NT = (d->co % 128 == 0) ? 128 : (d->co % 64 == 0 ? 64 : (d->co % 32 == 0 ? 32 : 16));
    const int sh = d->deconv ? d->stride_h : 1, sw = d->deconv ? d->stride_w : 1;
    const int Hu = (Ho + sh - 1) / sh, Wu = (Wo + sw - 1) / sw, ncls = min(sh, Ho) * min(sw, Wo);
    int tw = 8;
    while (tw < Wu && tw < 128) tw *= 2;
    const int th = 128 / tw;
    *tiles = (long long)N * ((Wu + tw - 1) / tw) * ((Hu + th - 1) / th) * (d->co / NT) * ncls;
    const int ntaps = d->deconv ? max(1, d->kh / sh) * max(1, d->kw / sw) : d->kh * d->kw;
    *steps = ntaps * ((d->ci + 31) / 32);
    *NTo = NT;
}

static int tc_split_plan(const fn2_conv_desc* d, int N, int Ho, int Wo) {
    if (!d->deconv && d->ci <= 16) return 1;                       // small-Ci packing modes do not split
    if (d->co % 16) return 1;
    const int NT = (d->co % 128 == 0) ? 128 : (d->co % 64 == 0 ? 64 : (d->co % 32 == 0 ? 32 : 16));
    const int sh = d->deconv ? d->stride_h : 1, sw = d->deconv ? d->stride_w : 1;
    const int Hu = (Ho + sh - 1) / sh, Wu = (Wo + sw - 1) / sw, ncls = min(sh, Ho) * min(sw, Wo);
    int tw = 8;
    while (tw < Wu && tw < 128) tw *= 2;
    const int th = 128 / tw;
    const long long tiles = (long long)N * ((Wu + tw - 1) / tw) * ((Hu + th - 1) / th) * (d->co / NT) * ncls;
    const int ntaps = d->deconv ? max(1, d->kh / sh) * max(1, d->kw / sw) : d->kh * d->kw;
    const int steps = ntaps * ((d->ci + 31) / 32);
    const int nsm = num_sms();
    if (tiles * 2 > nsm || steps < 32) return 1;
    int z = (int)(nsm / tiles);
    z = min(z, steps / 16);
    z = min(z, 8);
    return z < 2 ? 1 : z;
}

// taps-on-N engine for few output channels at high resolution (fn2_conv_tn.cu)
int conv_tn_applicable(const fn2_conv_desc* d);
size_t conv_tn_packed_floats(const fn2_conv_desc* d);
int conv_tn_pack(const fn2_conv_desc* d, const float* w, float* wp, cudaStream_t st);
int conv_tn_plan(const fn2_conv_desc* d, int N, int Ho, int Wo, int* out8);
int conv_tn_forward(const fn2_conv_desc* d, const T4& in, const float* wp, const float* bias, const T4& out, cudaStream_t st);

size_t conv_tc_workspace_floats(const fn2_conv_desc* d, int N, int Ho, int Wo) {
    if (conv_tn_applicable(d)) return 0;
    const int z = tc_split_plan(d, N, Ho, Wo);
    if (z > 1) return (size_t)z * N * Ho * Wo * d->co;
    if (d->co % 16 || (!d->deconv && d->ci <= 16)) return 0;
    int NT, steps, first; long long tiles;
    tc_layer_geometry(d, N, Ho, Wo, &NT, &tiles, &steps);
    const int tz = tc_tail_plan(tiles, steps, &first, NT);
    return tz > 1 ? (size_t)(tiles - first) * tz * 128 * NT : 0;
}

// Host-side plan of the tcgen05 engine for one layer shape (introspection for tests and tools; needs no GPU):
// out = {NT, tile units, K steps per tile, small-Ci mode (0 plain, 1 tap groups, 2 kernel rows), uniform K splits,
//        first tail tile, tail K ranges, 0}
int conv_tc_plan(const fn2_conv_desc* d, int N, int Ho, int Wo, int ci_stride, int* out8) {
    for (int i = 0; i < 8; i++) out8[i] = 0;
    if (d->co % 16) return 0;
    if (conv_tn_applicable(d)) return conv_tn_plan(d, N, Ho, Wo, out8);
    int NT, steps; long long tiles;
    tc_layer_geometry(d, N, Ho, Wo, &NT, &tiles, &steps);
    const TcSmallCi sm = tc_small_ci(d, ci_stride);
    if (sm.mode == 1) steps = sm.ngroups;
    if (sm.mode == 2) steps = d->kh * sm.rblocks;
    out8[0] = NT; out8[1] = (int)tiles; out8[2] = steps; out8[3] = sm.mode;
    out8[4] = tc_split_plan(d, N, Ho, Wo);
    out8[5] = (int)tiles; out8[6] = 1;
    if (out8[4] == 1 && !sm.mode) { int first = 0; out8[6] = tc_tail_plan(tiles, steps, &first, NT); out8[5] = first; }
    return 1;
}

int conv_tc_eligible(const fn2_conv_desc* d, const T4& in, const T4& out) {
    if (!tc_enabled()) return 0;
    if (in.sc != 1 || out.sc != 1) return 0;
    if (d->co % 16) return 0;
    if (d->deconv && (d->stride_h != 2 || d->stride_w != 2) && (d->stride_h != 1 || d->stride_w != 1)) return 0;
    if (d->kh * d->kw > 49) return 0;
    if (d->stride_h > 2 || d->stride_w > 2) return 0;
    if (((uintptr_t)in.p & 15) || (in.sw & 3) || (in.sh & 3) || (in.sn & 3)) return 0;
    if (((uintptr_t)out.p & 15) || (out.sw & 3) || (out.sh & 3) || (out.sn & 3)) return 0;
    if (!encode_tiled_fn()) return 0;
    return 1;
}

int conv_tc_packed_floats(const fn2_conv_desc* d, int ci_stride, size_t* floats) {
    if (conv_tn_applicable(d)) { *floats = conv_tn_packed_floats(d); return FN2_OK; }
    const int cip = (d->ci + 31) / 32 * 32;
    const TcSmallCi sm = tc_small_ci(d, ci_stride);
    if (sm.mode) {
        const int nblk = sm.mode == 2 ? d->kh * sm.rblocks : sm.ngroups;
        *floats = (d->co % 16 == 0) ? (size_t)2 * nblk * d->co * 32 : 0;
        return FN2_OK;
    }
    *floats = (d->co % 16 == 0) ? (size_t)2 * d->kh * d->kw * d->co * cip : 0;
    return FN2_OK;
}

int conv_tc_pack(const fn2_conv_desc* d, int ci_stride, const float* w, float* wp, cudaStream_t st) {
    if (conv_tn_applicable(d)) return conv_tn_pack(d, w, wp, st);
    size_t floats = 0;
    conv_tc_packed_floats(d, ci_stride, &floats);
    if (!floats) return FN2_OK;
    const int cip = (d->ci + 31) / 32 * 32;
    const TcSmallCi sm = tc_small_ci(d, ci_stride);
    if (sm.mode) {
        if (sm.mode == 2) tc_pack_row_kernel<<<ew_grid((long long)floats / 2, 256), 256, 0, st>>>(w, wp, d->ci, d->co, d->kh, d->kw, sm.cs, sm.rblocks);
        else tc_pack_group_kernel<<<ew_grid((long long)floats / 2, 256), 256, 0, st>>>(w, wp, d->ci, d->co, d->kh, d->kw, sm.cs, sm.ngroups);
        FN2_LAUNCH_CHECK();
        return FN2_OK;
    }
    tc_pack_kernel<<<ew_grid((long long)floats / 2, 256), 256, 0, st>>>(w, wp, d->ci, d->co, d->kh, d->kw, cip, d->deconv);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

static inline int floordiv_i(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

int conv_tc_forward(const fn2_conv_desc* d, const T4& in, const float* wp, const float* bias, const T4& out, float* ws, size_t ws_floats,
                    cudaStream_t st) {
    if (conv_tn_applicable(d)) return conv_tn_forward(d, in, wp, bias, out, st);
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("conv_tc: cuTensorMapEncodeTiled unavailable"); return FN2_ERR_CUDA; }
    const int NT = (d->co % 128 == 0) ? 128 : (d->co % 64 == 0 ? 64 : (d->co % 32 == 0 ? 32 : 16));
    const int cip = (d->ci + 31) / 32 * 32;
    TcParams p;
    p.corr = 0;
    p.N = in.n; p.Co = d->co; p.cblocks = cip / 32;
    p.Ho = out.h; p.Wo = out.w;
    p.splits = tc_split_plan(d, in.n, out.h, out.w);
    if (p.splits > 1 && (!ws || ws_floats < (size_t)p.splits * in.n * out.h * out.w * d->co)) p.splits = 1;
    p.out_sn = out.sn; p.out_sh = out.sh; p.out_sw = out.sw;
    p.relu = d->relu; p.has_bias = d->has_bias; p.slope = d->negative_slope;
    tc_chain_model(p, NT, false);

    const TcSmallCi sm = tc_small_ci(d, (int)in.sw);
    p.gcs = sm.mode == 1 ? sm.cs : 0;
    p.rowmode = sm.mode == 2; p.rcs = sm.cs; p.rblocks = sm.rblocks; p.rsteps = d->kh * sm.rblocks; p.rkw = d->kw; p.rpad = d->pad_w; p.rW = in.w;
    // weights: [2][taps][Co][cip]   (group mode: [2][groups][Co][32])
    CUtensorMap mapW;
    {
        const int kin = sm.mode ? 32 : cip;
        const int nblk = sm.mode == 2 ? p.rsteps : (sm.mode == 1 ? sm.ngroups : d->kh * d->kw);
        cuuint64_t dims[4] = {(cuuint64_t)kin, (cuuint64_t)d->co, (cuuint64_t)nblk, 2};
        cuuint64_t strides[3] = {(cuuint64_t)kin * 4, (cuuint64_t)kin * d->co * 4, (cuuint64_t)kin * d->co * nblk * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)NT, 1, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&mapW, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)wp, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tc: weight tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    auto run = [&](int su, int sv) -> int {
        // tile shape: widest power of two covering the (largest) row, 128 pixels per tile
        int Wmax = 0, Hmax = 0;
        for (int c = 0; c < p.ncls; c++) { Wmax = max(Wmax, p.cls_Wu[c]); Hmax = max(Hmax, p.cls_Hu[c]); }
        int tw = 8;
        while (tw < Wmax && tw < 128) tw *= 2;
        p.tw = tw; p.th = 128 / tw;
        p.tiles_x = (Wmax + p.tw - 1) / p.tw; p.tiles_y = (Hmax + p.th - 1) / p.th;
        p.su = su; p.sv = sv;
        CUtensorMap mapA;
        cuuint64_t dims[4] = {(cuuint64_t)in.c, (cuuint64_t)in.w, (cuuint64_t)in.h, (cuuint64_t)in.n};
        cuuint64_t strides[3] = {(cuuint64_t)in.sw * 4, (cuuint64_t)in.sh * 4, (cuuint64_t)in.sn * 4};
        cuuint32_t box[4] = {(cuuint32_t)(p.gcs ? p.gcs : 32), (cuuint32_t)(p.tw * su), (cuuint32_t)(p.th * sv), 1};
        cuuint32_t es[4] = {1, (cuuint32_t)su, (cuuint32_t)sv, 1};
        const float* baseA = in.p;
        if (p.rowmode) {
            // dim0: the run of kw*cs floats that starts pad_w pixels left of the output pixel's first tap column;
            // dim1: output column (consecutive runs overlap: stride = su pixels); dim2: input row; dim3: sample
            dims[0] = (cuuint64_t)p.rblocks * 32; dims[1] = (cuuint64_t)p.cls_Wu[0];
            strides[0] = (cuuint64_t)su * p.rcs * 4;
            box[1] = (cuuint32_t)p.tw; es[1] = 1;
            baseA = in.p - (long long)p.rpad * p.rcs;
        }
        CUresult r = enc(&mapA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)baseA, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         p.gcs ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tc: activation tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
        p.ntiles = p.N * p.tiles_x * p.tiles_y;
        p.cotiles = d->co / NT;
        p.total = p.ntiles * p.cotiles * p.ncls * p.splits;
        p.ntotal = p.total; p.tail_first = p.total; p.tail_z = 1;
        p.d_ntiles.init(p.ntiles); p.d_cotiles.init(p.cotiles); p.d_tiles_x.init(p.tiles_x); p.d_tiles_y.init(p.tiles_y);
        p.d_splits.init(max(1, p.splits)); p.d_tail_z.init(1);
        if (p.splits == 1 && !sm.mode && ws) {
            int first = 0, steps_min = 1 << 30;
            for (int c = 0; c < p.ncls; c++) steps_min = min(steps_min, p.cls_ntaps[c] * p.cblocks);
            const int tz = tc_tail_plan(p.total, steps_min, &first, NT);
            if (tz > 1 && ws_floats >= (size_t)(p.total - first) * tz * 128 * NT) {
                p.tail_first = first; p.tail_z = tz; p.d_tail_z.init(tz);
                p.total = first + (p.ntotal - first) * tz;
            }
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)min(p.total, num_sms()), 1, 1);
        cfg.blockDim = dim3(TC_THREADS);
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
#define FN2_TC_LAUNCH(NTV, MODEV)                                                                                       \
        {                                                                                                               \
            static bool attr_set = false;                                                                               \
            if (!attr_set) {                                                                                            \
                FN2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<NTV, MODEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGeo<NTV>::SMEM)); \
                attr_set = true;                                                                                        \
            }                                                                                                           \
            cfg.dynamicSmemBytes = TcGeo<NTV>::SMEM;                                                                    \
            FN2_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<NTV, MODEV>, mapA, mapW, bias, out.p, ws, p));                \
        }
#define FN2_TC_LAUNCH_NT(MODEV)                                                                                         \
        if (NT == 128) FN2_TC_LAUNCH(128, MODEV)                                                                        \
        else if (NT == 64) FN2_TC_LAUNCH(64, MODEV)                                                                     \
        else if (NT == 32) FN2_TC_LAUNCH(32, MODEV)                                                                     \
        else FN2_TC_LAUNCH(16, MODEV)
        if (sm.mode == 2) { FN2_TC_LAUNCH_NT(TC_ROW) }
        else if (sm.mode == 1) { FN2_TC_LAUNCH_NT(TC_GROUP) }
        else { FN2_TC_LAUNCH_NT(TC_PLAIN) }
#undef FN2_TC_LAUNCH_NT
#undef FN2_TC_LAUNCH
        FN2_LAUNCH_CHECK();
        if (p.tail_z > 1) {
            const long long work = (long long)(p.ntotal - p.tail_first) * 128 * (NT / 4);
            if (NT == 128) tc_tail_reduce_kernel<128><<<ew_grid(work, 256), 256, 0, st>>>(ws, bias, out.p, p);
            else if (NT == 64) tc_tail_reduce_kernel<64><<<ew_grid(work, 256), 256, 0, st>>>(ws, bias, out.p, p);
            else if (NT == 32) tc_tail_reduce_kernel<32><<<ew_grid(work, 256), 256, 0, st>>>(ws, bias, out.p, p);
            else tc_tail_reduce_kernel<16><<<ew_grid(work, 256), 256, 0, st>>>(ws, bias, out.p, p);
            FN2_LAUNCH_CHECK();
        }
        if (p.splits > 1) {
            tc_splitk_reduce_kernel<<<ew_grid((long long)p.N * p.Ho * p.Wo * (p.Co / 4), 256), 256, 0, st>>>(ws, bias, out.p, p);
            FN2_LAUNCH_CHECK();
        }
        return FN2_OK;
    };
    if (!d->deconv) {
        p.ncls = 1;
        p.cls_Hu[0] = out.h; p.cls_Wu[0] = out.w; p.ou = p.ov = 1; p.cls_oy0[0] = p.cls_ox0[0] = 0;
        p.cls_tap0[0] = 0; p.cls_ntaps[0] = d->kh * d->kw;
        for (int r = 0; r < d->kh; r++)
            for (int s = 0; s < d->kw; s++) {
                const int t = r * d->kw + s;
                p.dy[t] = (short)(r - d->pad_h); p.dx[t] = (short)(s - d->pad_w); p.widx[t] = (short)t;
            }
        return run(d->stride_w, d->stride_h);
    }
    // deconvolution: all output parity classes in one launch (grid.z); every kernel tap belongs to exactly one class
    const int sh = d->stride_h, sw = d->stride_w;
    p.ou = sh; p.ov = sw; p.ncls = 0;
    int nt = 0;
    for (int py = 0; py < sh; py++)
        for (int px = 0; px < sw; px++) {
            if (py >= out.h || px >= out.w) continue;
            const int c = p.ncls++;
            p.cls_Hu[c] = (out.h - py + sh - 1) / sh; p.cls_Wu[c] = (out.w - px + sw - 1) / sw;
            p.cls_oy0[c] = py; p.cls_ox0[c] = px; p.cls_tap0[c] = nt;
            for (int r = 0; r < d->kh; r++) {
                if (((py + d->pad_h - r) % sh + sh) % sh) continue;
                for (int s = 0; s < d->kw; s++) {
                    if (((px + d->pad_w - s) % sw + sw) % sw) continue;
                    p.dy[nt] = (short)floordiv_i(py + d->pad_h - r, sh);
                    p.dx[nt] = (short)floordiv_i(px + d->pad_w - s, sw);
                    p.widx[nt] = (short)(r * d->kw + s);
                    nt++;
                }
            }
            p.cls_ntaps[c] = nt - p.cls_tap0[c];
            if (p.cls_ntaps[c] == 0) { set_error("conv_tc: deconvolution parity class without taps"); return FN2_ERR_INVALID; }
        }
    return run(1, 1);
}

// ---------------------------------------------------------------------------------------------------------------------
// Correlation (MULTIPLY, kernel 1, stride_1 1, pad == max_displacement) on the tensor cores.
// stride_2 = S samples displacements that are multiples of S, so a pixel only meets map-1 pixels of its own parity plane;
// within a plane the op is "every pixel against its (2R+1)^2 neighbours", R = md / S.  Per 8x16-pixel tile the neighbours are
// the (8+2R) x (16+2R) halo; the kernel computes ALL tile-pixel x halo-pixel dot products as 3xTF32 GEMMs
// D[128 x 112] = A[128 x C] * B[112 x C]^T (one unit per block of 4 full halo rows: 9 blocks for R = 10) and keeps the 441 of the
// 1008 that lie in the window (2.3x redundant MMA work, which still beats the FP32 FMA pipe by a wide margin).
// Map 1 is split into TF32 hi / lo once per call (workspace [2][N][H][W][C]); both maps are read through element-strided
// TMA boxes, so the parity planes are never materialised and out-of-image neighbours are zero fill.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void corr_split_kernel(const float* __restrict__ b, long long sn, long long sh, long long sw, int N, int H, int W, int C,
                                  float* __restrict__ hi, float* __restrict__ lo) {
    const long long total = (long long)N * H * W * (C / 4);
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % (C / 4)) * 4;
        long long r = idx / (C / 4);
        const int x = (int)(r % W); r /= W;
        const int y = (int)(r % H);
        const int n = (int)(r / H);
        const float4 v = *reinterpret_cast<const float4*>(b + n * sn + y * sh + x * sw + c);
        const float f[4] = {v.x, v.y, v.z, v.w};
        float h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const uint32_t hb = to_tf32(f[e]);
            h[e] = __uint_as_float(hb);
            l[e] = __uint_as_float(to_tf32(f[e] - h[e]));
        }
        const long long o = (((long long)n * H + y) * W + x) * C + c;
        *reinterpret_cast<float4*>(hi + o) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(lo + o) = make_float4(l[0], l[1], l[2], l[3]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Weight gradient of Convolution / Deconvolution on the tensor cores (base_conv_layer.cpp:352-372 weight_gpu_gemm).
//   dW[a][b][ky][kx] = sum over (n, u, v) small[n, a, u, v] * big[n, b, u*s + ky - pad, v*s + kx - pad]
// with (small, big) = (top diff, bottom) for a convolution and (bottom, top diff) for a deconvolution: in both cases the Caffe
// blob is [small channels][big channels][kh][kw].  Per kernel tap this is a GEMM D[big ch x small ch] over K = pixels, and with
// both maps transposed to channel-major planes (pixels contiguous) its operands are K-major tiles exactly like the forward
// engine's: A = 128 channel rows x 32 consecutive pixels of the big map (raw FP32, split into TF32 hi/lo by the converter warps),
// B = NT channel rows x the same 32 pixels of the small map, pre-split once by the transposition pass.  The tap's shift is a TMA
// coordinate offset (zero fill = the convolution's padding); a strided layer reads the column-parity plane the tap falls into.
// Same FP32-faithful accumulation as the forward pass (short RZ chains drained to FP32 registers).
// ---------------------------------------------------------------------------------------------------------------------
struct WgPlan {
    int Cb, Cs, Hb, Wb, Hs, Ws, N, sx, sy;
    int NT, BT, ST, S, segs_x, segs, taps, G, TPT, TG;   // G rows per tap, TPT taps per 128-row tile, TG tap groups
    int Wq, Wq_p, Ws_p;                           // columns per parity plane (and its padded pitch), padded pitch of the small map
    size_t big_floats, small_floats, part_floats; // workspace pieces (each a multiple of 64 floats)
    size_t bias_floats;                           // per-block channel sums of the top diff (bias gradient, fused into its transposition)
    int bias_blocks;
};
static size_t up64(size_t x) { return (x + 63) / 64 * 64; }

static WgPlan wg_plan(const fn2_conv_desc* d, int N, int H, int W) {
    WgPlan g;
    int Ho = 0, Wo = 0;
    fn2_conv_out_shape(d, H, W, &Ho, &Wo);
    g.N = N; g.sx = d->stride_w; g.sy = d->stride_h; g.taps = d->kh * d->kw;
    if (!d->deconv) { g.Cb = d->ci; g.Cs = d->co; g.Hb = H; g.Wb = W; g.Hs = Ho; g.Ws = Wo; }
    else            { g.Cb = d->co; g.Cs = d->ci; g.Hb = Ho; g.Wb = Wo; g.Hs = H; g.Ws = W; }
    g.NT = g.Cs >= 128 ? 128 : (g.Cs >= 64 ? 64 : (g.Cs >= 32 ? 32 : 16));
    g.BT = (g.Cb + 127) / 128; g.ST = (g.Cs + g.NT - 1) / g.NT;
    g.G = 128;
    if (g.Cb <= 64) { g.G = 8; while (g.G < g.Cb) g.G *= 2; }
    g.TPT = 128 / g.G; g.TG = (g.taps + g.TPT - 1) / g.TPT;
    g.segs_x = (g.Ws + 31) / 32; g.segs = N * g.Hs * g.segs_x;
    const int base = g.TG * g.BT * g.ST;
    int S = (3 * num_sms() + base - 1) / base;
    S = max(1, min(S, g.segs / 8));
    g.S = S;
    g.Wq = (g.Wb + g.sx - 1) / g.sx + 3;          // + 3: room for the column delay of the 4 copies
    g.Wq_p = (g.Wq + 3) / 4 * 4; g.Ws_p = (g.Ws + 3) / 4 * 4;
    g.big_floats = up64((size_t)4 * N * g.Cb * g.Hb * g.sx * g.Wq_p);          // 4 copies, delayed by 0..3 columns
    g.small_floats = up64((size_t)2 * N * g.Cs * g.Hs * g.Ws_p);
    g.part_floats = up64((size_t)base * S * 128 * g.NT);
    // the top diff is the small map of a convolution and the big map of a deconvolution
    g.bias_blocks = d->deconv ? ((g.Wq_p + 127) / 128) * (N * g.Hb * g.sx) : ((g.Ws_p + 127) / 128) * (N * g.Hs);
    g.bias_floats = d->has_bias ? up64((size_t)g.bias_blocks * d->co) : 0;
    return g;
}

// channel-major planes: dst[dl][((n*C + c)*H + h)*sx + par][j] = src[n, c, h, (j - dl)*sx + par] (zero outside the row) for
// dl < nadv column delays; SPLIT writes the TF32 hi plane there and the lo plane `lo_off` floats further
// `dlmask`: which of the 4 delays are written (bit dl); the source is read once per block: 32 channels x (WG_TW + 3) columns.
// bias_part != nullptr: also the per-block channel sums of src, [block (x, z)][C] (the bias gradient when src is the top diff).
constexpr int WG_TW = 128;                        // columns per block (4 x the 32 threads of a row)
template <bool SPLIT>
__global__ void __launch_bounds__(256) wg_transpose_kernel(T4 src, float* __restrict__ dst, int sx, int Wq, int Wq_p, long long lo_off, int dlmask,
                                                           float* __restrict__ bias_part) {
    __shared__ float tile[WG_TW + 3][33];
    __shared__ float red[8][33];
    // grid: x = (sample, row, parity) -- the long dimension --, y = channel tile, z = column tile
    const int wq0 = blockIdx.z * WG_TW, c0 = blockIdx.y * 32;
    const int rp = blockIdx.x % (src.h * sx), n = blockIdx.x / (src.h * sx);
    const int h = rp / sx, par = rp % sx;
    const int halo = SPLIT ? 0 : 3;
    const int cols = min(WG_TW, Wq_p - wq0);                         // columns of this block that exist in the destination row
    for (int j = threadIdx.y; j < cols + halo; j += 8) {
        const int wq = wq0 + j - halo, w = wq * sx + par, c = c0 + threadIdx.x;       // tile row j = column wq0 + j - halo
        tile[j][threadIdx.x] = (c < src.c && wq >= 0 && w < src.w) ? src.p[src.off(n, c, h, w)] : 0.f;
    }
    __syncthreads();
    if (bias_part) {
        float a = 0.f;
        for (int j = threadIdx.y; j < cols; j += 8) a += tile[j + halo][threadIdx.x];           // the core columns, fixed order
        red[threadIdx.y][threadIdx.x] = a;
        __syncthreads();
        if (threadIdx.y == 0 && c0 + threadIdx.x < src.c) {
            float t = 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) t += red[k][threadIdx.x];
            bias_part[((long long)blockIdx.z * gridDim.x + blockIdx.x) * src.c + c0 + threadIdx.x] = t;
        }
    }
    const long long copy = (long long)src.n * src.c * src.h * sx * Wq_p;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j;
        if (c >= src.c) continue;
        float* row = dst + (((long long)n * src.c + c) * src.h * sx + rp) * Wq_p + wq0;
        for (int x = threadIdx.x; x < cols; x += 32) {
            if (SPLIT) {
                const float v = tile[x][j];
                const float hi = __uint_as_float(to_tf32(v));
                row[x] = hi;
                row[x + lo_off] = __uint_as_float(to_tf32(v - hi));
            } else {
#pragma unroll
                for (int dl = 0; dl < 4; dl++)
                    if (dlmask >> dl & 1) row[x + dl * copy] = tile[x + 3 - dl][j];       // index wq holds column wq - dl
            }
        }
    }
}

// db[c] (+)= sum over the blocks' partial sums, fixed order: 8 strided groups per channel, then the 8 group sums
__global__ void wg_bias_final_kernel(const float* __restrict__ part, float* __restrict__ db, int C, int blocks, int accumulate) {
    __shared__ float red[32][33];
    const int c = blockIdx.x * 32 + threadIdx.x;
    float a = 0.f;
    if (c < C)
        for (int k = threadIdx.y; k < blocks; k += 32) a += part[(long long)k * C + c];
    red[threadIdx.y][threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 32; k++) t += red[k][threadIdx.x];
        db[c] = accumulate ? db[c] + t : t;
    }
}

// dW[a][b][tap] (+)= sum over the K ranges of part[unit][row = (tap % TPT) * G + b % 128][col = a % NT]; threads run along the
// Caffe layout (coalesced read-modify-write of the diff; the strided partial reads hit L2).  A variant with coalesced partial reads
// and scattered diff updates measured 2.3x slower.
__global__ void wg_reduce_kernel(const float* __restrict__ part, float* __restrict__ dw, WgPlan g, int accumulate) {
    const long long total = (long long)g.Cs * g.Cb * g.taps;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int tap = (int)(idx % g.taps);
        const long long r = idx / g.taps;
        const int b = (int)(r % g.Cb), a = (int)(r / g.Cb);
        const long long unit0 = ((long long)((tap / g.TPT) * g.BT + b / 128) * g.ST + a / g.NT) * g.S;
        const float* src = part + (unit0 * 128 + (tap % g.TPT) * g.G + (b % 128)) * g.NT + (a % g.NT);
        float acc = 0.f;
        for (int k = 0; k < g.S; k++) acc += src[(long long)k * 128 * g.NT];
        dw[idx] = accumulate ? dw[idx] + acc : acc;
    }
}

int conv_tc_wgrad_eligible(const fn2_conv_desc* d) {
    if (!tc_enabled() || d->engine == 1) return 0;      // engine 1 = `engine: CAFFE`: exact-FP32 SIMT everywhere
    if (d->kh * d->kw > 49 || d->stride_w > 8 || d->stride_h > 8) return 0;
    if (!encode_tiled_fn()) return 0;
    return 1;
}
size_t conv_tc_wgrad_workspace_floats(const fn2_conv_desc* d, int N, int H, int W) {
    const WgPlan g = wg_plan(d, N, H, W);
    return g.big_floats + g.small_floats + g.part_floats + g.bias_floats + 64;
}

int conv_tc_wgrad(const fn2_conv_desc* d, const T4& bottom, const T4& top_diff, float* dw, float* db, int accumulate, float* ws,
                  size_t ws_floats, cudaStream_t st) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("conv_tc_wgrad: cuTensorMapEncodeTiled unavailable"); return FN2_ERR_CUDA; }
    const WgPlan g = wg_plan(d, bottom.n, bottom.h, bottom.w);
    if (!ws || ws_floats < conv_tc_wgrad_workspace_floats(d, bottom.n, bottom.h, bottom.w)) { set_error("conv_tc_wgrad: workspace too small"); return FN2_ERR_WORKSPACE; }
    const T4& big = d->deconv ? top_diff : bottom;
    const T4& small = d->deconv ? bottom : top_diff;
    if (big.h != g.Hb || big.w != g.Wb || small.h != g.Hs || small.w != g.Ws || big.c != g.Cb || small.c != g.Cs) {
        set_error("conv_tc_wgrad: tensor shapes do not match the descriptor"); return FN2_ERR_INVALID;
    }
    ws = reinterpret_cast<float*>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    float* bigT = ws; float* smallT = ws + g.big_floats; float* part = smallT + g.small_floats;
    float* bias_part = (d->has_bias && db) ? part + g.part_floats : nullptr;
    {
        dim3 blk(32, 8);
        int dlmask = 0;                                     // column delays the layer's taps actually use
        for (int kx = 0; kx < d->kw; kx++) {
            const int q = kx - d->pad_w, par = ((q % g.sx) + g.sx) % g.sx, shift = (q - par) / g.sx;
            dlmask |= 1 << ((((-shift) % 4) + 4) % 4);
        }
        dim3 gb((unsigned)(g.N * g.Hb * g.sx), (unsigned)((g.Cb + 31) / 32), (unsigned)((g.Wq_p + WG_TW - 1) / WG_TW));
        wg_transpose_kernel<false><<<gb, blk, 0, st>>>(big, bigT, g.sx, g.Wq, g.Wq_p, 0, dlmask, d->deconv ? bias_part : nullptr);
        FN2_LAUNCH_CHECK();
        dim3 gs((unsigned)(g.N * g.Hs), (unsigned)((g.Cs + 31) / 32), (unsigned)((g.Ws_p + WG_TW - 1) / WG_TW));
        wg_transpose_kernel<true><<<gs, blk, 0, st>>>(small, smallT, 1, g.Ws, g.Ws_p, (long long)g.N * g.Cs * g.Hs * g.Ws_p, 1,
                                                      d->deconv ? nullptr : bias_part);
        FN2_LAUNCH_CHECK();
        if (bias_part) {
            wg_bias_final_kernel<<<(unsigned)((d->co + 31) / 32), dim3(32, 32), 0, st>>>(bias_part, db, d->co, g.bias_blocks, accumulate);
            FN2_LAUNCH_CHECK();
        }
    }
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.N = g.N; p.Co = g.Cs; p.cblocks = 1;
    p.Ho = g.Hs; p.Wo = g.Ws;
    p.splits = 1; p.tail_z = 1; p.su = g.sx; p.sv = g.sy; p.ou = p.ov = 1; p.ncls = 1;
    p.tw = 128; p.th = 1; p.tiles_x = p.tiles_y = 1;
    p.wg_S = g.S; p.wg_ST = g.ST; p.wg_BT = g.BT; p.wg_segs = g.segs; p.wg_segs_x = g.segs_x; p.wg_sx = g.sx;
    p.wg_G = g.G; p.wg_TPT = g.TPT; p.wg_taps = g.taps;
    tc_chain_model(p, g.NT, false);
    for (int ky = 0; ky < d->kh; ky++)
        for (int kx = 0; kx < d->kw; kx++) {
            const int t = ky * d->kw + kx, q = kx - d->pad_w;
            const int par = ((q % g.sx) + g.sx) % g.sx;
            const int shift = (q - par) / g.sx, dl = (((-shift) % 4) + 4) % 4;    // copy `dl` holds column j - dl at index j
            p.dy[t] = (short)(ky - d->pad_h); p.dx[t] = (short)(shift + dl); p.widx[t] = (short)(par | (dl << 4));
        }
    p.total = g.TG * g.BT * g.ST * g.S;
    p.ntotal = p.total; p.tail_first = p.total;
    CUtensorMap mapA, mapB;
    {
        cuuint64_t dims[4] = {(cuuint64_t)g.Wq, (cuuint64_t)g.Hb * g.sx, (cuuint64_t)g.Cb, (cuuint64_t)4 * g.N};
        cuuint64_t strides[3] = {(cuuint64_t)g.Wq_p * 4, (cuuint64_t)g.Hb * g.sx * g.Wq_p * 4, (cuuint64_t)g.Cb * g.Hb * g.sx * g.Wq_p * 4};
        cuuint32_t box[4] = {32, 1, (cuuint32_t)g.G, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&mapA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)bigT, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tc_wgrad: big-map tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)g.Ws, (cuuint64_t)g.Hs, (cuuint64_t)g.Cs, (cuuint64_t)2 * g.N};
        cuuint64_t strides[3] = {(cuuint64_t)g.Ws_p * 4, (cuuint64_t)g.Hs * g.Ws_p * 4, (cuuint64_t)g.Cs * g.Hs * g.Ws_p * 4};
        cuuint32_t box[4] = {32, 1, (cuuint32_t)g.NT, 1};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&mapB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)smallT, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("conv_tc_wgrad: small-map tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)min(p.total, num_sms()), 1, 1);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.stream = st;
#define FN2_WG_LAUNCH(NTV)                                                                                              \
    {                                                                                                                   \
        static bool attr_set = false;                                                                                   \
        if (!attr_set) {                                                                                                \
            FN2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<NTV, TC_WGRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGeo<NTV>::SMEM)); \
            attr_set = true;                                                                                            \
        }                                                                                                               \
        cfg.dynamicSmemBytes = TcGeo<NTV>::SMEM;                                                                        \
        FN2_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<NTV, TC_WGRAD>, mapA, mapB, (const float*)nullptr, (float*)nullptr, part, p));                   \
    }
    if (g.NT == 128) FN2_WG_LAUNCH(128)
    else if (g.NT == 64) FN2_WG_LAUNCH(64)
    else if (g.NT == 32) FN2_WG_LAUNCH(32)
    else FN2_WG_LAUNCH(16)
#undef FN2_WG_LAUNCH
    FN2_LAUNCH_CHECK();
    wg_reduce_kernel<<<ew_grid((long long)g.Cs * g.Cb * g.taps, 256), 256, 0, st>>>(part, dw, g, accumulate);
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

int corr_tc_eligible(const T4& b0, const T4& b1, const T4& top, int md, int s2) {
    if (!tc_enabled() || getenv("FN2_CORR_NOTC")) return 0;
    if (s2 < 1 || s2 > 2 || md % s2 || md / s2 != 10) return 0;            // halo blocks are laid out for R = 10
    if (b0.c % 32 || b0.sc != 1 || b1.sc != 1 || top.sc != 1) return 0;
    if (((uintptr_t)b0.p & 15) || (b0.sw & 3) || (b0.sh & 3) || (b0.sn & 3)) return 0;
    if (((uintptr_t)b1.p & 15) || (b1.sw & 3) || (b1.sh & 3) || (b1.sn & 3)) return 0;
    if (!encode_tiled_fn()) return 0;
    return 1;
}
size_t corr_tc_workspace_floats(int N, int C, int H, int W) { return (size_t)2 * N * H * W * C; }

int corr_tc_forward(const T4& b0, const T4& b1, const T4& top, int md, int s2, float* ws, size_t ws_floats, cudaStream_t st) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("corr_tc: cuTensorMapEncodeTiled unavailable"); return FN2_ERR_CUDA; }
    const int N = b0.n, C = b0.c, H = b0.h, W = b0.w, S = s2, R = md / s2;
    if (!ws || ws_floats < corr_tc_workspace_floats(N, C, H, W)) { set_error("corr_tc: workspace too small"); return FN2_ERR_WORKSPACE; }
    float* hi = ws; float* lo = ws + (size_t)N * H * W * C;
    corr_split_kernel<<<ew_grid((long long)N * H * W * (C / 4), 256), 256, 0, st>>>(b1.p, b1.sn, b1.sh, b1.sw, N, H, W, C, hi, lo);
    FN2_LAUNCH_CHECK();
    constexpr int NT = 128;
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.corr = 1; p.cR = R; p.cS = S; p.cD = 2 * R + 1;
    p.tw = 8; p.th = 16;                                                   // halo 28 x 36
    p.cbw = p.tw + 2 * R; p.cbh = 4;                                       // block = 4 full halo rows = 112 pixels (MMA N = 112)
    p.cnx = 1; p.cnt = (p.th + 2 * R) / p.cbh;                             // 9 blocks
    p.cscale = 1.0f / (float)C;                                           // sumelems = k*k*C (correlation_layer.cu:108)
    p.N = N; p.Co = NT; p.cblocks = C / 32;
    p.Ho = H; p.Wo = W;
    p.out_sn = top.sn; p.out_sh = top.sh; p.out_sw = top.sw;
    p.splits = 1; p.tail_z = 1; p.su = S; p.sv = S; p.ou = p.ov = 1; p.ncls = 1;
    tc_chain_model(p, NT, true);
    const int Ws = (W + S - 1) / S, Hs = (H + S - 1) / S;
    p.tiles_x = (Ws + p.tw - 1) / p.tw; p.tiles_y = (Hs + p.th - 1) / p.th;
    p.total = N * S * S * p.tiles_x * p.tiles_y * p.cnt;
    p.ntotal = p.total; p.tail_first = p.total;
    CUtensorMap mapA, mapB;
    {
        cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)b0.sw * 4, (cuuint64_t)b0.sh * 4, (cuuint64_t)b0.sn * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)(p.tw * S), (cuuint32_t)(p.th * S), 1};
        cuuint32_t es[4] = {1, (cuuint32_t)S, (cuuint32_t)S, 1};
        CUresult r = enc(&mapA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)b0.p, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("corr_tc: map-0 tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)2 * N};
        cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)(p.cbw * S), (cuuint32_t)(p.cbh * S), 1};
        cuuint32_t es[4] = {1, (cuuint32_t)S, (cuuint32_t)S, 1};
        CUresult r = enc(&mapB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)hi, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("corr_tc: map-1 tensor map failed (%d)", (int)r); return FN2_ERR_CUDA; }
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)min(p.total, num_sms()), 1, 1);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.stream = st;
    const int smem_bytes = TcGeo<NT>::SMEM + 128 * CORR_TR_STRIDE * (int)sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        FN2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<NT, TC_CORR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        attr_set = true;
    }
    cfg.dynamicSmemBytes = smem_bytes;
    FN2_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<NT, TC_CORR>, mapA, mapB, (const float*)nullptr, top.p, (float*)nullptr, p));
    FN2_LAUNCH_CHECK();
    return FN2_OK;
}

}  // namespace fn2
