// detectorch_b200 -- implicit-GEMM convolution / GEMM on tcgen05 tensor cores (sm_100a).
//
// Replaces every Conv2d / Linear / ConvTranspose2d that the reference runs through
// torch+cuDNN/cuBLAS (reference lib/model/detector.py:17-27,58-59,71-74,89-90,119-121,
// 170-183,212-214; SURVEY.md 2.2 K1/K3/K4/K9/K11).
//
// Data layout: activations are NHWC fp32 in HBM (pixel-major rows of C channels), weights are
// [Cout][kh][kw][Cin] fp32 (K-major rows), both fetched by TMA into 128B-swizzled shared
// memory tiles; accumulators live in TMEM.
//
// Precision: the parity contract is fp32 (1e-4, BASELINE.json north_star), but tcgen05 has no
// fp32-input MMA.  We therefore run error-compensated 3xTF32:
//     D += A*B_hi + A*B_lo + A_lo*B_hi          (kind::tf32 reads only the top 19 bits of each
//                                                 fp32 word, so "A" and "B_hi" need no rounding pass)
// with A_lo = A - trunc_tf32(A) produced in shared memory by 4 converter warps while the
// previous stage's MMAs run, and B_lo precomputed once per weight tensor.  `passes`==1 runs the
// plain single-pass TF32 product (debug / speed-of-light reference).
//
// KIND_F16X3 (the engine default) runs the same three-term product on the kind::f16 pipe, which
// issues at twice the tf32 rate: A = A_h + A_l with A_h = fp16(A), A_l = fp16(A - A_h) (22 mantissa bits, the same as the two
// tf32 pieces), B_h / B_l likewise (precomputed, pre-scaled by a power of two so that B_l stays a normal fp16 number; the
// epilogue scale undoes it exactly).  The fp32 A tile still arrives by TMA; the converter warps write A_h / A_l as two
// 64-byte-row (SWIZZLE_64B) fp16 tiles -- unless the producing layer already wrote the activation as two fp16 planes
// (a_planes / out_planes: conv1 -> conv2 of a bottleneck), in which case TMA delivers the operand tiles directly.
// fp16 has a 5-bit exponent: |A| >= 65504 raises a device flag (the engine then reports it; the tf32 kind has no such limit).
//
// Tile: BLOCK_M = 128 output pixels (a wbox x hbox x nbox box of the NHWC output, so the same
// TMA box geometry loads A for any filter tap and stores D, with hardware zero-fill doing the
// padding and hardware clipping doing the edge masking), BLOCK_N = 64/128/256 output channels,
// BLOCK_K = 32 fp32 = one 128-byte swizzle row.
//
// Execution model (round-1 profile: the one-tile-per-CTA version lost ~20k cycles per tile to prologue +
// un-overlapped epilogue): PERSISTENT CTAs in 2-CTA clusters, 512 threads =
//   warp 0       TMA producer (A tile; its half of the weight k-block, multicast to both CTAs of the pair)
//   warp 1       TMEM owner + MMA issuer (one elected lane)
//   warps 2-5    operand converters (fp32 -> fp16 hi/lo, in place for most instantiations; pass-through for plane inputs)
//   warps 6-13   epilogue WORKERS, two independent groups of 4 warps: TMEM -> regs -> scale/shift [+residual] [ReLU|sigmoid] ->
//                swizzled staging slot, 32-channel chunks (even chunks group 0, odd chunks group 1); the staging slots are NOT
//                aliased with the pipeline, so the producer / converter / MMA warps run ahead into the next tile while a tile drains
//   warps 14-15  one STORE warp per group: TMA store of the staged chunk, tile bookkeeping, residual-ring refill, slot hand-back
//                (arrive/sync named-barrier pair with the workers)
// TMEM holds NMAIN rotating main-term accumulators + 1 cross-term accumulator per tile (NMAIN == 0: a single accumulator for
// both, used by the 256-wide layers up to K = 2304), double-buffered when two tiles fit in the 512 columns.
// Variants selected by the host per layer (conv_host.cuh): 1-SM MMA with multicast weights vs cta_group::2, a K-split over filter
// taps (tap0 / ntaps), RING > 0: a ring of residual tiles prefetched by TMA for the conv3 + residual layers, SLOTS: staging slots per
// epilogue group, HALO: 3x3 / stem forms that fetch one A box per filter row (row parity) and address the taps through shifted
// UMMA descriptors, WS: weights resident in shared memory (stem).  DT_CONV_WARPS_NARROW (8 converter warps) is a
// measured-and-rejected experiment switch; DT_INPLACE_NARROW / DT_INPLACE_RING are build switches kept for A/B.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace dt {

enum ConvResidualMode { RES_NONE = 0, RES_TILE = 1, RES_UPSAMPLE2X = 2 };
enum ConvKind { KIND_TF32X3 = 0, KIND_F16X3 = 1 };
#ifndef DT_INPLACE_RING
#define DT_INPLACE_RING 1
#endif
#ifndef DT_INPLACE_NARROW
#define DT_INPLACE_NARROW 1      // in-place fp16 split for the 64 / 128-wide fp32-input layers too (build switch kept for A/B)
#endif
#ifndef DT_CONV_WARPS_NARROW
#define DT_CONV_WARPS_NARROW 4
#endif


struct ConvParams {
    CUtensorMap tm_a;      // 4D {C, W, H, N} over the NHWC input (elementStrides carry the conv stride)
    CUtensorMap tm_bhi;    // 2D {K, Cout} weights (fp32; the MMA ignores the low 13 bits -> "hi"), box = BLOCK_N/2 rows
    CUtensorMap tm_blo;    // 2D {K, Cout} B - trunc_tf32(B)
    CUtensorMap tm_d;      // 4D {Cout, Wo, Ho, N} over the NHWC output, box {32, wbox, hbox, nbox}
    CUtensorMap tm_r;      // 4D residual, same geometry as tm_d (RES_TILE only)
    CUtensorMap tm_a2;     // a_planes: the fp16 LOW plane of the input (tm_a is then the fp16 HIGH plane), SWIZZLE_64B boxes of 32 channels
    CUtensorMap tm_d2;     // out_planes: the fp16 LOW plane of the output (tm_d the HIGH plane), SWIZZLE_64B boxes of 32 channels
    const float* scale;    // [Cout] per-channel scale (folded BN gain, or 1)
    const float* shift;    // [Cout] per-channel shift (folded BN bias, or conv bias)
    const float* up_src;   // RES_UPSAMPLE2X: coarser NHWC map [N, up_h, up_w, Cout]
    int up_h, up_w;
    int cin_blocks;        // Cin / 32
    int kh, kw;
    int tap0, ntaps;       // this launch covers filter taps [tap0, tap0 + ntaps) of the kh*kw (a K-split partial convolution; default all)
    int pad_w, pad_h, stride_w, stride_h;   // A-load coordinate = tile origin * stride + tap - pad, per axis
    int tiles_w, tiles_h, tiles_n;
    int m_pairs, n_tiles;  // work items = m_pairs * n_tiles; a CTA pair handles M-tiles (2*mp, 2*mp+1) of one N-tile
    int wbox, hbox, nbox;
    int wo, ho, nimg;      // output extents (for RES_UPSAMPLE2X bounds)
    int cout;              // true Cout (channels >= cout are never stored: TMA clips)
    int a_tile_bytes;      // wbox*hbox*nbox*128
    int relu;
    int sigmoid_ch;        // channels [0, sigmoid_ch) get a sigmoid (RPN objectness), after bias
    int res_mode;
    int passes;            // 3 = error-compensated three-term product (default), 1 = single pass
    int a_planes;          // KIND_F16X3: the input already is a pair of fp16 planes (hi, lo) written by the producing layer: the A_h / A_l
                           // operand tiles arrive by TMA and the converter warps have nothing to do
    int out_planes;        // KIND_F16X3: write the output as a pair of fp16 planes (hi = fp16(y), lo = fp16(y - hi)) instead of fp32
    int* range_flag;       // KIND_F16X3: set to 1 when an activation does not fit fp16 (|x| >= 65504 or NaN); may be null
    int pdl;               // launched with programmatic stream serialization: release the next launch early, wait for the previous one
    int a_halo_bytes;      // HALO variant: bytes of ONE fp16 plane of the (wbox + 2) x hbox x nbox halo box (rows of 64 B)
    float a_mult;          // KIND_F16X3, fp32 input: power of two the converters apply before the fp16 split (0 = none; the engine passes none)
};

// HALO (3x3, stride 1, fp16-plane input, tiles 8 pixels wide): one TMA box of (8 + 2) x hbox x nbox pixels per (filter row, 32-channel
// block) serves the THREE horizontal taps -- the A descriptor of tap dx starts dx rows into the box and steps 10 rows (640 B) from one
// 8-pixel group to the next -- so the A tile is fetched from L2 3 times per tile instead of 9 (the 64/128-channel 3x3 layers were bound by
// exactly that re-fetch: ncu 7.8 TB/s L2->SM at 23 % tensor-pipe activity).  A stage holds the halo planes + the weights of 3 taps.
// HALO == 2 (the 7-tap, stride-2 fused-window stem over fp16 planes, tiles 8 x 16 pixels of one image): a step is one PARITY of the filter
// rows -- the even rows ky = 0, 2, 4, 6 read input rows 2 (h + j), j = 0..3, the odd rows ky = 1, 3, 5 input rows 2 (h + j) + 1 -- so one
// stride-2 box of 16 + 3 row slabs serves the 4 (3) taps of a parity: tap j starts j slabs (j x 8 rows = j swizzle atoms) into the box.
// The A tile is fetched 2 times per tile instead of 7.
template <int BLOCK_N, int NMAIN, bool kTwoSM, int KIND, int RING = 0, int SLOTS = 1, int HALO = 0, bool WS = false>
struct ConvCfg {
    static constexpr int BLOCK_M = 128;
    static constexpr int BLOCK_K = 32;
    static constexpr int A_BYTES = BLOCK_M * 128;                    // 16 KB: the fp32 A tile as TMA delivers it
    // 1-SM MMA: every CTA holds the whole BLOCK_N-row weight tile (its half arrives by multicast from the peer).
    // 2-SM MMA (cta_group::2): every CTA holds only ITS half -> smaller stages, deeper pipeline, half the operand ingest per SM.
    static constexpr int B_ROW_BYTES = KIND == KIND_F16X3 ? 64 : 128; // 32 k-elements per row
    static constexpr int B_BYTES = (kTwoSM ? BLOCK_N / 2 : BLOCK_N) * B_ROW_BYTES;
    // tf32: A, A_lo (16 KB each), B_hi, B_lo.
    // f16 : A (fp32 staging, 16 KB), A_h | A_l (8 KB each), B_h, B_l -- or, INPLACE, ONE 16 KB A area: TMA delivers the fp32 tile into
    //       it; the converter warps read their rows into registers, meet at a named barrier and write A_h | A_l IN PLACE over the fp32
    //       data (the two fp16 tiles are exactly as large as the fp32 tile); with a_planes TMA delivers A_h | A_l there directly.  A stage
    //       is then 32 KB instead of 48 KB (5-6 pipeline stages instead of 3-4).  Used by every non-ring, non-halo kind::f16 instantiation
    //       but the 256-wide merged-accumulator ones with two staging slots.  History: with the round-2-start epilogue the deeper
    //       pipeline only paid on the long-K 256-wide layers (-4..7 %) and cost the 64-wide / short-K layers 4-7 % (the extra converter
    //       barrier sat on a chain the epilogue dominated); after the epilogue rewrite the 64 / 128-wide fp32-input layers (conv1 of
    //       layers 1-2, RPN heads, mask logits) turned out to be bound by BYTES IN FLIGHT -- 3 stages x 16 KB per SM = 7 MB against the
    //       ~10 MB that 6.5 TB/s x 1.5 us need -- and gained 6-12 % from the 6-deep in-place pipeline (profiles/r02_summary.md).
    static constexpr bool INPLACE = KIND == KIND_F16X3 && (RING == 0 || DT_INPLACE_RING != 0) && HALO == 0 &&
                                    (BLOCK_N == 256 ? (NMAIN == 1 || SLOTS == 1) : (DT_INPLACE_NARROW != 0 && DT_CONV_WARPS_NARROW == 4));
    static_assert(!HALO || (KIND == KIND_F16X3 && RING == 0 && !INPLACE), "the halo variant is a kind::f16, plane-input, no-ring kernel");
    static constexpr int HALO_ROWS = 160;                            // (8 + 2) x 16 pixel rows of 64 B per plane (HALO == 2: 8 x (16 + 3) = 152)
    static constexpr int HALO_PLANE_BYTES = HALO_ROWS * 64;          // 10 KB, a multiple of the 512-byte swizzle atom
    static constexpr int B_TAPS = HALO == 1 ? 3 : (HALO == 2 ? 4 : 1);   // weight tiles per stage
    static constexpr int A_STAGE_BYTES = HALO ? 2 * HALO_PLANE_BYTES : (INPLACE ? A_BYTES : 2 * A_BYTES);
    static constexpr int A_OP_OFF = (KIND == KIND_F16X3 && !INPLACE && !HALO) ? A_BYTES : 0;      // where A_h starts inside a stage (kind::f16)
    static constexpr int A_LO_OFF = A_OP_OFF + (HALO ? HALO_PLANE_BYTES : A_BYTES / 2);          // ... and A_l
    // WS (weight-stationary; halo variants, 64-wide, one N tile, 2-SM MMA so that each CTA keeps only 32 weight rows): the hi / lo weights of
    // ALL k-blocks are loaded once per CTA and stay resident; a stage then holds the A halo planes only.  After the halo cut the A
    // re-fetch, the per-tile weight fetch was more than half of the L2 -> SM traffic of the 64-channel 3x3 layers and of the stem (ncu: 7.8 TB/s).
    static_assert(!WS || (HALO != 0 && kTwoSM && BLOCK_N == 64), "weight-stationary: halo variants of the 64-wide 2-SM kernel only");
    static constexpr int BRES_KB = WS ? (HALO == 1 ? 18 : 7) : 0;   // resident k-blocks: 3x3 x 64 channels, or the stem's 7 filter rows
    static constexpr int BRES_BYTES = BRES_KB * 2 * B_BYTES;
    static constexpr int STAGE_BYTES = WS ? A_STAGE_BYTES : A_STAGE_BYTES + 2 * B_BYTES * B_TAPS;
    // epilogue staging: each of the two epilogue groups owns EPI_SLOTS 16 KB slots (128 rows x 32 channels).  With ONE slot the group's
    // per-chunk chain is  TMEM load -> scale/shift/residual -> staging -> TMA store -> wait until the store has READ the slot -> next chunk;
    // with TWO slots the store of chunk i drains while chunk i+1 is computed.  Measured per layer (profiles/r02_ab_epilogue_slots.md):
    // two slots cut the epilogue-bound launches by 10-16 % (K <= 256 at 256 channels: downsample 1x1, deconv GEMMs, the conv3 + residual
    // layers; every <= 128-wide layer, where the extra 32 KB do not cost a pipeline stage), but cost the long-K 256-wide layers their
    // fourth pipeline stage (+6-15 %): the host picks SLOTS per layer (conv_host.cuh).
    static constexpr int EPI_SLOTS = SLOTS;
    // RING > 0 (short-K residual layers, where the epilogue IS the kernel): a ring of RING residual tiles per epilogue group is
    // prefetched by TMA RING chunks ahead, so the HBM latency of the residual never sits in the per-chunk chain; the mainloop
    // (<= 16 k-blocks per tile) makes do with two pipeline stages.
    static constexpr int RING_BYTES = 2 * RING * A_BYTES;
    static constexpr int EPI_BYTES = 2 * EPI_SLOTS * A_BYTES;
    static constexpr int STAGES_FIT = (196608 + 2 * A_BYTES - EPI_BYTES - RING_BYTES - BRES_BYTES) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_FIT > 6 ? 6 : STAGES_FIT;
    static constexpr int BRES_OFF = STAGES * STAGE_BYTES;            // resident weights follow the pipeline stages
    static constexpr int PIPE_BYTES = STAGES * STAGE_BYTES + BRES_BYTES;
    static_assert(STAGES >= 2, "pipeline too shallow");
    static constexpr int TILE_COLS = (NMAIN + 1) * BLOCK_N;          // TMEM columns of one tile's accumulators
    static constexpr int NBUF = (2 * TILE_COLS <= 512) ? 2 : 1;      // double-buffer the accumulators when they fit
    static constexpr int TMEM_COLS = (NBUF * TILE_COLS > 256) ? 512 : (NBUF * TILE_COLS > 128 ? 256 : 128);
    static constexpr int NUM_BARS = 3 * STAGES + 2 * NBUF + 2 * EPI_SLOTS + 2 * RING + (WS ? 1 : 0);
    static constexpr int SMEM_BYTES = PIPE_BYTES + EPI_BYTES + RING_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
    // converter warps: the fp16 split of a 16 KB tile costs ~2x the tf32 residual and, for tiles up to 128 wide, more than the
    // MMAs of a k-block -> 8 warps there (two 16-byte pieces per thread), 4 otherwise
    static constexpr int CONV_WARPS = (KIND == KIND_F16X3 && BLOCK_N <= 128) ? DT_CONV_WARPS_NARROW : 4;
    static constexpr int CONV_THREADS = CONV_WARPS * 32;
    static constexpr int EPI_WARP0 = 2 + CONV_WARPS;                 // first epilogue warp
    static constexpr int STORE_WARP0 = EPI_WARP0 + 8;                // two store warps (one per epilogue group) follow the 8 epilogue warps
    static constexpr int THREADS = 64 + CONV_THREADS + 256 + 64;
    static_assert(TILE_COLS <= 512, "accumulators of one tile must fit TMEM");
    static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared-memory limit");
    static_assert(8 * (NUM_BARS + 1) <= 256, "barrier area");
};

template <int BLOCK_N, int NMAIN, bool kTwoSM, int KIND, int RING = 0, int SLOTS = 1, int HALO = 0, bool WS = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((ConvCfg<BLOCK_N, NMAIN, kTwoSM, KIND, RING, SLOTS, HALO, WS>::THREADS), 1) conv_tcgen05_kernel(const __grid_constant__ ConvParams p) {
    using Cfg = ConvCfg<BLOCK_N, NMAIN, kTwoSM, KIND, RING, SLOTS, HALO, WS>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int NBUF = Cfg::NBUF;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment is required by SWIZZLE_128B (TMA and UMMA descriptors)
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t epi_base = smem_base + Cfg::PIPE_BYTES;
    uint8_t* epi_gen = smem_gen + Cfg::PIPE_BYTES;
    const uint32_t ring_base = epi_base + Cfg::EPI_BYTES;          // residual prefetch ring (RING > 0)
    uint8_t* ring_gen = epi_gen + Cfg::EPI_BYTES;
    const uint32_t bar_base = ring_base + Cfg::RING_BYTES;
    // barrier slots (8 B each)
    auto bar_full = [&](int s) { return bar_base + 8u * s; };                            // TMA bytes landed
    auto bar_conv = [&](int s) { return bar_base + 8u * (STAGES + s); };                 // A_lo published
    auto bar_empty = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };            // both CTAs' MMAs retired
    auto bar_tfull = [&](int b) { return bar_base + 8u * (3 * STAGES + b); };            // a tile's accumulators complete
    auto bar_tempty = [&](int b) { return bar_base + 8u * (3 * STAGES + NBUF + b); };    // ... drained by the epilogue
    auto bar_res = [&](int b) { return bar_base + 8u * (3 * STAGES + 2 * NBUF + b); };   // residual chunk landed in epilogue slot b (group * EPI_SLOTS + slot)
    auto bar_ring = [&](int b) { return bar_base + 8u * (3 * STAGES + 2 * NBUF + 2 * Cfg::EPI_SLOTS + b); };   // ... in ring slot b (group * RING + r)
    const uint32_t bar_bres = bar_base + 8u * (Cfg::NUM_BARS - 1);      // WS: the resident weights landed (once per CTA)
    const uint32_t bres_base = smem_base + Cfg::BRES_OFF;
    const uint32_t tmem_slot = bar_base + 8u * Cfg::NUM_BARS;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(epi_gen + Cfg::EPI_BYTES + Cfg::RING_BYTES + 8 * Cfg::NUM_BARS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // pipeline steps per tile: one k-block (32 channels of one filter tap) -- or, HALO, one (filter row, 32-channel block) = 3 taps
    const int num_kb = HALO == 1 ? p.kh * p.cin_blocks : (HALO == 2 ? 2 : p.ntaps * p.cin_blocks);
    const int num_items = p.m_pairs * p.n_tiles;
    const int pair = blockIdx.x >> 1;
    const int num_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tm_a);
        tma_prefetch_desc(&p.tm_bhi);
        tma_prefetch_desc(&p.tm_blo);
        tma_prefetch_desc(&p.tm_d);
        if (p.res_mode == RES_TILE) tma_prefetch_desc(&p.tm_r);
        if (p.a_planes) tma_prefetch_desc(&p.tm_a2);
        if (p.out_planes) tma_prefetch_desc(&p.tm_d2);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_conv(s), (kTwoSM ? 2 : 1) * Cfg::CONV_THREADS);     // 2-SM: the leader's issuer also waits for the peer's converters
            mbar_init(bar_empty(s), kTwoSM ? 1 : 2);        // 1-SM: own MMA commit + the peer's (its multicast writes land in our stage too)
        }
        for (int b = 0; b < NBUF; ++b) {
            mbar_init(bar_tfull(b), 1);
            mbar_init(bar_tempty(b), kTwoSM ? 512 : 256);   // 2-SM: both CTAs' epilogues release the leader's issuer
        }
        for (int b = 0; b < 2 * Cfg::EPI_SLOTS; ++b) mbar_init(bar_res(b), 1);
        for (int b = 0; b < 2 * RING; ++b) mbar_init(bar_ring(b), 1);
        if constexpr (WS) mbar_init(bar_bres, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        if constexpr (kTwoSM) tmem_alloc_2sm<Cfg::TMEM_COLS>(tmem_slot); else tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();          // the peer's barriers must be initialised before any multicast / remote arrive
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot_gen;
    const uint32_t cta_rank = cluster_ctarank();
    if (p.pdl) {
        // Everything above (barrier init, TMEM allocation, descriptor prefetch, cluster handshake) touched no global data: with PDL it
        // overlaps the tail of the previous launch on the SMs that launch has already left.  The next launch in the stream may become
        // resident as soon as every CTA of this grid got here (it then parks in its own griddep_wait until this grid has completed).
        griddep_launch_dependents();
        griddep_wait();
    }

    // work item -> tile coordinates.  The N-tile varies fastest so that consecutive items re-read the same A tile from L2.
    auto tile_of = [&](int item, int& w0, int& h0, int& n0img, int& n0) {
        const int nt = item % p.n_tiles;
        int t = (item / p.n_tiles) * 2 + (int)cta_rank;       // this CTA's M-tile (may be the out-of-range surplus tile)
        const int tw = t % p.tiles_w; t /= p.tiles_w;
        const int th = t % p.tiles_h; t /= p.tiles_h;
        w0 = tw * p.wbox; h0 = th * p.hbox; n0img = t * p.nbox; n0 = nt * BLOCK_N;
    };

    if (warp == 0) {
        // ================================================================ TMA producer
        if (lane == 0) {
            const uint32_t tx_bytes = (uint32_t)p.a_tile_bytes + (p.passes == 3 ? 2u : 1u) * Cfg::B_BYTES;
            uint32_t it = 0;
            if constexpr (WS) {
                // this CTA's 32 rows of every k-block of the weight matrix (hi, lo), once
                const int nkb_all = HALO == 1 ? p.kh * p.kw * p.cin_blocks : 7;
                mbar_arrive_expect_tx(bar_bres, (uint32_t)nkb_all * 2u * Cfg::B_BYTES);
                for (int kbg = 0; kbg < nkb_all; ++kbg) {
                    tma_load_2d(bres_base + kbg * 2 * Cfg::B_BYTES, &p.tm_bhi, bar_bres, kbg * 32, (int)cta_rank * (BLOCK_N / 2));
                    tma_load_2d(bres_base + kbg * 2 * Cfg::B_BYTES + Cfg::B_BYTES, &p.tm_blo, bar_bres, kbg * 32, (int)cta_rank * (BLOCK_N / 2));
                }
            }
            for (int item = pair; item < num_items; item += num_pairs) {
                int w0, h0, n0img, n0;
                tile_of(item, w0, h0, n0img, n0);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1u;
                    mbar_wait(bar_empty(s), ph ^ 1u);
                    if constexpr (HALO == 2) {
                        // step = parity q of the filter rows: the two plane boxes (stride 2 in h from row 2 h0 + q) + the weights of its 4 - q taps
                        const int q = kb, ntq = 4 - q;
                        const uint32_t st = smem_base + s * Cfg::STAGE_BYTES;
                        mbar_arrive_expect_tx(bar_full(s), 2u * (uint32_t)p.a_halo_bytes + (WS ? 0u : (uint32_t)ntq * 2u * Cfg::B_BYTES));
                        tma_load_4d(st, &p.tm_a, bar_full(s), 0, w0, 2 * h0 + q, n0img);
                        tma_load_4d(st + Cfg::HALO_PLANE_BYTES, &p.tm_a2, bar_full(s), 0, w0, 2 * h0 + q, n0img);
                        const int nrow = n0 + (int)cta_rank * (BLOCK_N / 2);
                        for (int j = 0; j < ntq && !WS; ++j) {
                            const int kbg = 2 * j + q;         // filter row = k-block of the weight matrix
                            const uint32_t bh = st + Cfg::A_STAGE_BYTES + j * 2 * Cfg::B_BYTES, bl = bh + Cfg::B_BYTES;
                            if constexpr (kTwoSM) {
                                tma_load_2d(bh, &p.tm_bhi, bar_full(s), kbg * 32, nrow);
                                tma_load_2d(bl, &p.tm_blo, bar_full(s), kbg * 32, nrow);
                            } else {
                                const uint32_t half = cta_rank * (Cfg::B_BYTES / 2);
                                tma_load_2d_mcast(bh + half, &p.tm_bhi, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                                tma_load_2d_mcast(bl + half, &p.tm_blo, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                            }
                        }
                        continue;
                    }
                    if constexpr (HALO == 1) {
                        // step = (filter row fy, channel block cb): the two halo planes + the hi / lo weights of the row's three taps
                        const int fy = kb / p.cin_blocks;
                        const int cb = kb - fy * p.cin_blocks;
                        const uint32_t st = smem_base + s * Cfg::STAGE_BYTES;
                        mbar_arrive_expect_tx(bar_full(s), 2u * (uint32_t)p.a_halo_bytes + (WS ? 0u : 6u * Cfg::B_BYTES));
                        tma_load_4d(st, &p.tm_a, bar_full(s), cb * 32, w0 - 1, h0 + fy - 1, n0img);
                        tma_load_4d(st + Cfg::HALO_PLANE_BYTES, &p.tm_a2, bar_full(s), cb * 32, w0 - 1, h0 + fy - 1, n0img);
                        const int nrow = n0 + (int)cta_rank * (BLOCK_N / 2);
#pragma unroll
                        for (int dx = 0; dx < 3 && !WS; ++dx) {
                            const int kbg = (fy * 3 + dx) * p.cin_blocks + cb;
                            const uint32_t bh = st + Cfg::A_STAGE_BYTES + dx * 2 * Cfg::B_BYTES, bl = bh + Cfg::B_BYTES;
                            if constexpr (kTwoSM) {
                                tma_load_2d(bh, &p.tm_bhi, bar_full(s), kbg * 32, nrow);
                                tma_load_2d(bl, &p.tm_blo, bar_full(s), kbg * 32, nrow);
                            } else {
                                const uint32_t half = cta_rank * (Cfg::B_BYTES / 2);
                                tma_load_2d_mcast(bh + half, &p.tm_bhi, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                                tma_load_2d_mcast(bl + half, &p.tm_blo, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                            }
                        }
                        continue;
                    }
                    const int tap_l = kb / p.cin_blocks;
                    const int cb = kb - tap_l * p.cin_blocks;
                    const int tap = p.tap0 + tap_l;
                    const int kbg = tap * p.cin_blocks + cb;        // k-block index into the full weight row
                    const int fy = tap / p.kw, fx = tap - fy * p.kw;
                    const uint32_t st = smem_base + s * Cfg::STAGE_BYTES;
                    mbar_arrive_expect_tx(bar_full(s), tx_bytes);
                    if (KIND == KIND_F16X3 && p.a_planes) {
                        // fp16 planes: the two operand tiles land where the converters would have written them
                        tma_load_4d(st + Cfg::A_OP_OFF, &p.tm_a, bar_full(s), cb * 32, w0 * p.stride_w + fx - p.pad_w, h0 * p.stride_h + fy - p.pad_h, n0img);
                        tma_load_4d(st + Cfg::A_OP_OFF + Cfg::A_BYTES / 2, &p.tm_a2, bar_full(s), cb * 32, w0 * p.stride_w + fx - p.pad_w,
                                    h0 * p.stride_h + fy - p.pad_h, n0img);
                    } else {
                        tma_load_4d(st, &p.tm_a, bar_full(s), cb * 32, w0 * p.stride_w + fx - p.pad_w, h0 * p.stride_h + fy - p.pad_h, n0img);
                    }
                    // this CTA's half of the weight rows
                    const int nrow = n0 + (int)cta_rank * (BLOCK_N / 2);
                    if constexpr (kTwoSM) {
                        // 2-SM MMA: the half stays local (the pair's tensor cores read both halves in place)
                        tma_load_2d(st + Cfg::A_STAGE_BYTES, &p.tm_bhi, bar_full(s), kbg * 32, nrow);
                        if (p.passes == 3) tma_load_2d(st + Cfg::A_STAGE_BYTES + Cfg::B_BYTES, &p.tm_blo, bar_full(s), kbg * 32, nrow);
                    } else {
                        // 1-SM MMA: multicast to both CTAs of the pair
                        const uint32_t half = cta_rank * (Cfg::B_BYTES / 2);
                        tma_load_2d_mcast(st + Cfg::A_STAGE_BYTES + half, &p.tm_bhi, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                        if (p.passes == 3)
                            tma_load_2d_mcast(st + Cfg::A_STAGE_BYTES + Cfg::B_BYTES + half, &p.tm_blo, bar_full(s), kbg * 32, nrow, (uint16_t)3);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================================================================ MMA issuer (one elected lane; 2-SM: leader CTA only)
        constexpr uint32_t idesc_main = umma_idesc(KIND == KIND_F16X3 ? 0 : 2, kTwoSM ? 256 : 128, BLOCK_N);
        // one K step of the instruction = 32 bytes of a row: 8 tf32 or 16 fp16 elements -> 4 or 2 steps per 32-element k-block
        constexpr int KSTEPS = KIND == KIND_F16X3 ? 2 : 4;
        auto mma = [&](uint32_t acc, uint64_t da_, uint64_t db_, uint32_t flag) {
            constexpr uint32_t idesc = idesc_main;
            if constexpr (KIND == KIND_F16X3) {
                if constexpr (kTwoSM) umma_f16_2sm(acc, da_, db_, idesc, flag); else umma_f16(acc, da_, db_, idesc, flag);
            } else {
                if constexpr (kTwoSM) umma_tf32_2sm(acc, da_, db_, idesc, flag); else umma_tf32(acc, da_, db_, idesc, flag);
            }
        };
        uint32_t it = 0;
        int t = 0;
        for (int item = pair; item < num_items && (!kTwoSM || cta_rank == 0); item += num_pairs, ++t) {
            const int buf = t % NBUF;
            if constexpr (kTwoSM) mbar_wait_cluster(bar_tempty(buf), (((uint32_t)(t / NBUF)) & 1u) ^ 1u);
            else mbar_wait(bar_tempty(buf), (((uint32_t)(t / NBUF)) & 1u) ^ 1u);     // the epilogue drained this accumulator set
            tc_fence_after();
            const uint32_t acc0 = tmem_acc + (uint32_t)(buf * Cfg::TILE_COLS);
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1u;
                if constexpr (kTwoSM) mbar_wait_cluster(bar_conv(s), ph);   // both CTAs' TMA data landed and both converted A tiles are published
                else mbar_wait(bar_conv(s), ph);      // converters waited on full[s] and published their tiles
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t st = smem_base + s * Cfg::STAGE_BYTES;
                    if constexpr (HALO == 2) {
                        // tap j of this parity reads the box from row slab j on (8 rows = one swizzle atom per slab: plain descriptors)
                        constexpr int NM = NMAIN == 0 ? 1 : NMAIN;
                        const uint32_t acc_x = acc0 + (uint32_t)(NMAIN * BLOCK_N);
                        const int ntq = 4 - kb;
                        for (int j = 0; j < ntq; ++j) {
                            const uint64_t da = umma_desc_k_sw64(st + j * 512);
                            const uint64_t dal = umma_desc_k_sw64(st + Cfg::HALO_PLANE_BYTES + j * 512);
                            const uint32_t bsm = WS ? bres_base + (2 * j + kb) * 2 * Cfg::B_BYTES : st + Cfg::A_STAGE_BYTES + j * 2 * Cfg::B_BYTES;
                            const uint64_t dbh = umma_desc_k_sw64(bsm);
                            const uint64_t dbl = umma_desc_k_sw64(bsm + Cfg::B_BYTES);
                            const int idx = kb * 4 + j;
                            const uint32_t acc_main = acc0 + (uint32_t)((idx % NM) * BLOCK_N);
#pragma unroll
                            for (int k = 0; k < KSTEPS; ++k) {
                                const uint64_t koff = (uint64_t)(k * 32 >> 4);
                                const uint32_t main_flag = NMAIN == 0 ? 1u : ((idx >= NMAIN || k != 0) ? 1u : 0u);
                                mma(acc_x, dal + koff, dbh + koff, (idx | k) != 0);
                                mma(acc_x, da + koff, dbl + koff, 1u);
                                mma(acc_main, da + koff, dbh + koff, main_flag);
                            }
                        }
                    } else if constexpr (HALO == 1) {
                        // tap dx of this filter row reads the halo box from pixel column dx on: start + dx rows, 10 rows between 8-pixel groups
                        constexpr int NM = NMAIN == 0 ? 1 : NMAIN;
                        const uint32_t acc_x = acc0 + (uint32_t)(NMAIN * BLOCK_N);
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
                            const uint64_t da = umma_desc_k_sw64_sbo(st + dx * 64, 640);
                            const uint64_t dal = umma_desc_k_sw64_sbo(st + Cfg::HALO_PLANE_BYTES + dx * 64, 640);
                            // WS: k-block (fy, dx, cb) of the resident weights; this step is (fy, cb) = (kb / cin_blocks, kb % cin_blocks)
                            const uint32_t bsm = WS ? bres_base + (((kb / p.cin_blocks) * 3 + dx) * p.cin_blocks + kb % p.cin_blocks) * 2 * Cfg::B_BYTES
                                                    : st + Cfg::A_STAGE_BYTES + dx * 2 * Cfg::B_BYTES;
                            const uint64_t dbh = umma_desc_k_sw64(bsm);
                            const uint64_t dbl = umma_desc_k_sw64(bsm + Cfg::B_BYTES);
                            const int idx = kb * 3 + dx;       // the main term rotates over the accumulators by tap
                            const uint32_t acc_main = acc0 + (uint32_t)((idx % NM) * BLOCK_N);
#pragma unroll
                            for (int k = 0; k < KSTEPS; ++k) {
                                const uint64_t koff = (uint64_t)(k * 32 >> 4);
                                const uint32_t main_flag = NMAIN == 0 ? 1u : ((idx >= NMAIN || k != 0) ? 1u : 0u);
                                mma(acc_x, dal + koff, dbh + koff, (idx | k) != 0);
                                mma(acc_x, da + koff, dbl + koff, 1u);
                                mma(acc_main, da + koff, dbh + koff, main_flag);
                            }
                        }
                    } else {
                    uint64_t da, dal, dbh, dbl;      // "hi" A, "lo" A, "hi" B, "lo" B
                    if constexpr (KIND == KIND_F16X3) {
                        da = umma_desc_k_sw64(st + Cfg::A_OP_OFF);
                        dal = umma_desc_k_sw64(st + Cfg::A_LO_OFF);
                        dbh = umma_desc_k_sw64(st + Cfg::A_STAGE_BYTES);
                        dbl = umma_desc_k_sw64(st + Cfg::A_STAGE_BYTES + Cfg::B_BYTES);
                    } else {
                        da = umma_desc_k_sw128(st);
                        dal = umma_desc_k_sw128(st + Cfg::A_BYTES);
                        dbh = umma_desc_k_sw128(st + 2 * Cfg::A_BYTES);
                        dbl = umma_desc_k_sw128(st + 2 * Cfg::A_BYTES + Cfg::B_BYTES);
                    }
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                        const uint64_t koff = (uint64_t)(k * 32 >> 4);
                        // The tensor core accumulates in fp32 with truncation, so every accumulate step costs up to 1 ulp of
                        // the running sum (a systematic shrink of ~0.18 * steps * 2^-23).  Two measures keep the chains short:
                        //  * the two cross terms (~2^-11 of the main term) go to their own accumulator,
                        //  * the main term rotates over NMAIN accumulators by k-block (summed with RN adds in the epilogue).
                        // NMAIN == 0: short-K layers keep everything in ONE accumulator, which leaves room to double-buffer a
                        // 256-wide tile (the epilogue of tile i then overlaps the MMAs of tile i+1)
                        constexpr int NM = NMAIN == 0 ? 1 : NMAIN;
                        const uint32_t acc_main = acc0 + (uint32_t)((kb % NM) * BLOCK_N);
                        const uint32_t main_flag = NMAIN == 0 ? ((p.passes == 3 || (kb | k) != 0) ? 1u : 0u) : ((kb >= NMAIN || k != 0) ? 1u : 0u);
                        if (p.passes == 3) {
                            const uint32_t acc_x = acc0 + (uint32_t)(NMAIN * BLOCK_N);
                            mma(acc_x, dal + koff, dbh + koff, (kb | k) != 0);
                            mma(acc_x, da + koff, dbl + koff, 1u);
                        }
                        mma(acc_main, da + koff, dbh + koff, main_flag);
                    }
                    }
                    if constexpr (kTwoSM) {
                        umma_commit_2sm_mcast(bar_empty(s), (uint16_t)3);                        // frees this stage in both CTAs
                        if (kb == num_kb - 1) umma_commit_2sm_mcast(bar_tfull(buf), (uint16_t)3);  // both CTAs' accumulators are complete
                    } else {
                        umma_commit_mcast(bar_empty(s), (uint16_t)3);       // frees this stage in BOTH CTAs' producers when these MMAs retire
                        if (kb == num_kb - 1) umma_commit(bar_tfull(buf));  // this tile's accumulators are complete
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp < Cfg::EPI_WARP0) {
        // ================================================================ A_lo converters (128 threads)
        const int ct = threadIdx.x - 64;    // 0..CONV_THREADS-1
        uint32_t it = 0;
        // WS: a stage is passed on only after this CTA's resident weights have landed (2-SM: the leader's issuer waits for both CTAs' converters)
        if constexpr (WS) mbar_wait(bar_bres, 0u);
        for (int item = pair; item < num_items; item += num_pairs) {
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1u;
                mbar_wait(bar_full(s), ph);
                if (KIND == KIND_F16X3 && p.a_planes) {
                    // operand tiles were delivered by TMA (async proxy): nothing to convert, just pass the stage on
                } else if constexpr (KIND == KIND_F16X3) {
                    if constexpr (Cfg::INPLACE) {
                        // A_h = fp16(A), A_l = fp16(A - A_h), IN PLACE: a thread owns one row -- 8 x 16-byte pieces of the 128B-swizzled fp32 row in
                        // (registers), then, once every converter thread has read its row (named barrier: the fp16 tiles overlay other threads'
                        // fp32 rows), 4 x 16-byte pieces of each 64B-swizzled fp16 row out (both access patterns are conflict-free)
                        uint8_t* a32 = smem_gen + s * Cfg::STAGE_BYTES;
                        uint8_t* ah = a32;
                        uint8_t* al = ah + Cfg::A_BYTES / 2;
                        bool bad = false;
                        // rows past the TMA box (boxes smaller than 128 pixels) are never written: whatever they hold produces accumulator
                        // rows that are never stored, but it must not trip the range flag
                        const bool live_row = (ct & 127) * 128 < p.a_tile_bytes;
                        static_assert(Cfg::CONV_THREADS == 128, "the in-place split maps one converter thread to one tile row");
                        const int r = ct;
                        float4 fin[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) fin[i] = *reinterpret_cast<const float4*>(a32 + r * 128 + ((i ^ (r & 7)) << 4));
                        if (p.a_mult != 0.f) {
                            // exact (a power of two): lifts small activations out of the range where the low half is subnormal
#pragma unroll
                            for (int i = 0; i < 8; ++i) { fin[i].x *= p.a_mult; fin[i].y *= p.a_mult; fin[i].z *= p.a_mult; fin[i].w *= p.a_mult; }
                        }
                        named_bar_sync(3, Cfg::CONV_THREADS);          // ids 1, 2 belong to the epilogue groups
#pragma unroll
                        for (int c8 = 0; c8 < 4; ++c8) {
                            const float4 v0 = fin[2 * c8], v1 = fin[2 * c8 + 1];
                            const float f[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                            __half2 hh[4], ll[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const __half h0 = __float2half_rn(f[2 * j]), h1 = __float2half_rn(f[2 * j + 1]);
                                bad = bad || !(fabsf(f[2 * j]) < 65504.f) || !(fabsf(f[2 * j + 1]) < 65504.f);
                                hh[j] = __halves2half2(h0, h1);
                                ll[j] = __halves2half2(__float2half_rn(f[2 * j] - __half2float(h0)), __float2half_rn(f[2 * j + 1] - __half2float(h1)));
                            }
                            const int off = r * 64 + ((c8 ^ ((r >> 1) & 3)) << 4);
                            *reinterpret_cast<uint4*>(ah + off) = *reinterpret_cast<const uint4*>(hh);
                            if (p.passes == 3) *reinterpret_cast<uint4*>(al + off) = *reinterpret_cast<const uint4*>(ll);
                        }
                        if (bad && live_row && p.range_flag) *p.range_flag = 1;
                        fence_proxy_async_smem();
                    } else {
                        // A_h = fp16(A), A_l = fp16(A - A_h): thread -> (row, 8-channel group); two 16-byte pieces of the 128B-swizzled
                        // fp32 row in, one 16-byte piece of each 64B-swizzled fp16 row out (both access patterns are conflict-free)
                        const uint8_t* a32 = smem_gen + s * Cfg::STAGE_BYTES;
                        uint8_t* ah = smem_gen + s * Cfg::STAGE_BYTES + Cfg::A_BYTES;
                        uint8_t* al = ah + Cfg::A_BYTES / 2;
                        bool bad = false;
                        // rows past the TMA box (boxes smaller than 128 pixels) are never written: whatever they hold produces accumulator
                        // rows that are never stored, but it must not trip the range flag
                        const bool live_row = (ct & 127) * 128 < p.a_tile_bytes;
                        constexpr int PIECES = 4 * 128 / Cfg::CONV_THREADS;        // 16-byte fp16 pieces per thread (4 or 2)
#pragma unroll
                        for (int i = 0; i < PIECES; ++i) {
                            const int r = ct & 127, c8 = (ct >> 7) * PIECES + i;
                            const float4 v0 = *reinterpret_cast<const float4*>(a32 + r * 128 + (((2 * c8) ^ (r & 7)) << 4));
                            const float4 v1 = *reinterpret_cast<const float4*>(a32 + r * 128 + (((2 * c8 + 1) ^ (r & 7)) << 4));
                            float f[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                            if (p.a_mult != 0.f) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) f[j] *= p.a_mult;
                            }
                            __half2 hh[4], ll[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const __half h0 = __float2half_rn(f[2 * j]), h1 = __float2half_rn(f[2 * j + 1]);
                                bad = bad || !(fabsf(f[2 * j]) < 65504.f) || !(fabsf(f[2 * j + 1]) < 65504.f);
                                hh[j] = __halves2half2(h0, h1);
                                ll[j] = __halves2half2(__float2half_rn(f[2 * j] - __half2float(h0)), __float2half_rn(f[2 * j + 1] - __half2float(h1)));
                            }
                            const int off = r * 64 + ((c8 ^ ((r >> 1) & 3)) << 4);
                            *reinterpret_cast<uint4*>(ah + off) = *reinterpret_cast<const uint4*>(hh);
                            if (p.passes == 3) *reinterpret_cast<uint4*>(al + off) = *reinterpret_cast<const uint4*>(ll);
                        }
                        if (bad && live_row && p.range_flag) *p.range_flag = 1;
                        fence_proxy_async_smem();
                    }
                } else if (p.passes == 3) {
                    // A_lo = A - trunc_tf32(A), element-wise, so the swizzled placement is preserved verbatim
                    const float4* a = reinterpret_cast<const float4*>(smem_gen + s * Cfg::STAGE_BYTES);
                    float4* alo = reinterpret_cast<float4*>(smem_gen + s * Cfg::STAGE_BYTES + Cfg::A_BYTES);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 v = a[ct + i * 128];
                        float4 o;
                        o.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
                        o.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
                        o.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
                        o.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
                        alo[ct + i * 128] = o;
                    }
                    fence_proxy_async_smem();    // generic-proxy writes -> visible to the tensor core (async proxy)
                }
                if constexpr (kTwoSM) mbar_arrive_cluster(mapa_cluster(bar_conv(s), 0));   // the leader CTA's issuer collects both CTAs
                else mbar_arrive(bar_conv(s));
            }
        }
    } else {
        // ================================================================ epilogue: two independent groups of 4 warps (warps 6-9, 10-13)
        // Group g drains the live 32-channel chunks c with c % 2 == g through its own 16 KB staging slot, so two chunks are in
        // flight per tile and every SM sub-partition has two epilogue warps to hide TMEM / shared / global latencies.
        // Each group has a STORE WARP (warps STORE_WARP0 + g): it issues the chunk's TMA store, does the tile bookkeeping, refills the residual
        // ring and waits for the next staging slot to drain, while the 128 workers are already reading and summing the next chunk's
        // accumulators.  Two named barriers per group pair them: B2 (id 4 + g: workers arrive after writing + fencing the staging slot, the
        // store warp waits) and B1 (id 1 + g: the store warp arrives once the next chunk's slot is free, the workers wait right before
        // they write it).  With the store inside the worker group (thread 0) the other 127 threads idled through its bookkeeping: ncu
        // showed 31 % of the epilogue warps' samples on that barrier in the short-K layers.
        constexpr int NCHUNK = BLOCK_N / 32;
        const bool is_store = warp >= Cfg::STORE_WARP0;
        const int g = is_store ? warp - Cfg::STORE_WARP0 : (warp - Cfg::EPI_WARP0) >> 2;
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;          // accumulator row == pixel slot in the box
        constexpr int NS = Cfg::EPI_SLOTS;
        uint32_t gc = 0;                        // chunks this group has processed -> slot parity and residual-barrier phase
        auto nlive_of = [&](int item_) {
            int nl = (p.cout - (item_ % p.n_tiles) * BLOCK_N + 31) / 32;       // chunks past the true Cout are neither computed nor stored
            return nl < 0 ? 0 : (nl > NCHUNK ? NCHUNK : nl);
        };
        // A cursor over this group's live chunks in processing order.  The tile fields are recomputed only when the item changes: thread 0
        // advances two of these per chunk between the group's barriers (the other 127 threads wait for it), and the divisions of tile_of /
        // nlive_of per chunk were a quarter of the chunk time of the short-K layers (ncu source view: 31 % of the epilogue warps' samples
        // on the barrier that follows thread 0's bookkeeping).
        struct Cursor { int item, c, nlive, w0, h0, n0img, n0; };
        auto cur_init = [&](Cursor& k) {
            k.item = pair; k.c = g - 2;
            k.nlive = nlive_of(k.item);
            tile_of(k.item, k.w0, k.h0, k.n0img, k.n0);
        };
        auto cur_next = [&](Cursor& k) {        // -> the group's next live chunk (same tile, or the first live chunk of a later tile)
            k.c += 2;
            if (k.c < k.nlive) return true;
            do {
                k.item += num_pairs; k.c = g;
                if (k.item >= num_items) return false;
                k.nlive = nlive_of(k.item);
            } while (k.c >= k.nlive);
            tile_of(k.item, k.w0, k.h0, k.n0img, k.n0);
            return true;
        };
        auto issue_residual = [&](const Cursor& k, uint32_t gcn) {     // et == 0 only: residual tile chunk -> slot of chunk number gcn
            const uint32_t sl = (uint32_t)(g * NS) + (gcn % NS);
            mbar_arrive_expect_tx(bar_res(sl), (uint32_t)p.a_tile_bytes);
            tma_load_4d(epi_base + sl * Cfg::A_BYTES, &p.tm_r, bar_res(sl), k.n0 + k.c * 32, k.w0, k.h0, k.n0img);
        };
        if (is_store) {
            // ------------------------------------------------------------ store warp of group g (lane 0 issues; the warp stays convergent for the barriers)
            Cursor cur, pf;                         // the chunk being stored; the ring prefetch position (RING chunks ahead)
            cur_init(cur); cur_init(pf);
            bool live = cur_next(cur), pf_live = true;
            uint32_t pf_n = 0;                      // chunks whose residual load has been issued
            auto issue_ring = [&]() {               // lane 0 only
                if (!pf_live) return;
                pf_live = cur_next(pf);
                if (!pf_live) return;
                const uint32_t sl = (uint32_t)(g * RING) + (pf_n % (RING > 0 ? RING : 1));
                mbar_arrive_expect_tx(bar_ring(sl), (uint32_t)p.a_tile_bytes);
                tma_load_4d(ring_base + sl * Cfg::A_BYTES, &p.tm_r, bar_ring(sl), pf.n0 + pf.c * 32, pf.w0, pf.h0, pf.n0img);
                ++pf_n;
            };
            if (lane == 0 && p.res_mode == RES_TILE) {
                if constexpr (RING > 0) {
                    for (int r = 0; r < RING; ++r) issue_ring();
                } else if (live) {                     // residual of the group's very first chunk
                    issue_residual(cur, 0u);
                }
            }
            __syncwarp();
            if (live) named_bar_arrive(1 + g, 160);     // the first chunk's slot is free
            while (live) {
                named_bar_sync(4 + g, 160);             // the workers have written (and fenced) this chunk's staging slot
                if (lane == 0) {
                    const uint32_t sidx = (uint32_t)(g * NS) + (gc % NS);
                    const uint32_t slot = epi_base + sidx * Cfg::A_BYTES;
                    const int ch0 = cur.n0 + cur.c * 32;
                    if (KIND == KIND_F16X3 && p.out_planes) {
                        tma_store_4d(&p.tm_d, slot, ch0, cur.w0, cur.h0, cur.n0img);
                        tma_store_4d(&p.tm_d2, slot + Cfg::A_BYTES / 2, ch0, cur.w0, cur.h0, cur.n0img);
                    } else {
                        tma_store_4d(&p.tm_d, slot, ch0, cur.w0, cur.h0, cur.n0img);
                    }
                    tma_store_commit();
                }
                live = cur_next(cur);                   // (every lane keeps the cursor: the loop condition must stay warp-uniform)
                if (lane == 0) {
                    // free the slot the NEXT chunk will use (its last store must have finished reading shared memory) and start that
                    // chunk's residual load
                    if constexpr (RING > 0) {
                        // every worker is past its reads of this chunk's ring slot (it arrived on B2): refill it
                        if (p.res_mode == RES_TILE) issue_ring();
                        if (live) tma_store_wait_read<NS - 1>();
                    } else if (live) {
                        tma_store_wait_read<NS - 1>();
                        if (p.res_mode == RES_TILE) issue_residual(cur, gc + 1);
                    }
                }
                __syncwarp();
                if (live) named_bar_arrive(1 + g, 160);
                ++gc;
            }
            if (lane == 0) tma_store_wait0();      // all output bytes written before the CTA may exit
        } else {
        int t = 0;
        for (int item = pair; item < num_items; item += num_pairs, ++t) {
            int w0, h0, n0img, n0;
            tile_of(item, w0, h0, n0img, n0);
            const int buf = t % NBUF;
            const int nacc = HALO ? NMAIN : (num_kb < NMAIN ? num_kb : NMAIN);     // HALO: >= 3 taps per tile, NMAIN <= 3
            const int nlive = nlive_of(item);
            // pixel coordinates of this row (needed for the upsample operand)
            int pw_ = 0, ph_ = 0, pn_ = 0;
            bool row_valid = false;
            if (p.res_mode == RES_UPSAMPLE2X) {
                int r = row;
                pw_ = r % p.wbox; r /= p.wbox;
                ph_ = r % p.hbox; r /= p.hbox;
                pn_ = r;
                row_valid = (pn_ < p.nbox) && (w0 + pw_ < p.wo) && (h0 + ph_ < p.ho) && (n0img + pn_ < p.nimg);
            }
            mbar_wait(bar_tfull(buf), ((uint32_t)(t / NBUF)) & 1u);
            tc_fence_after();
            const uint32_t tbase0 = tmem_acc + (uint32_t)(buf * Cfg::TILE_COLS) + ((uint32_t)(q * 32) << 16);
            int last_c = -1;                             // this group's last live chunk of the tile
            for (int c = g; c < nlive; c += 2) last_c = c;
            if (last_c < 0) {
                tc_fence_before();
                if constexpr (kTwoSM) mbar_arrive_cluster(mapa_cluster(bar_tempty(buf), 0)); else mbar_arrive(bar_tempty(buf));
            }
#pragma unroll 1
            for (int c = g; c < nlive; c += 2, ++gc) {
                const int ch0 = n0 + c * 32;
                const uint32_t sidx = (uint32_t)(g * NS) + (gc % NS);
                const uint32_t slot = epi_base + sidx * Cfg::A_BYTES;
                uint8_t* slot_gen = epi_gen + sidx * Cfg::A_BYTES;
                // upsample operand of this chunk: requested from global BEFORE the TMEM reads (latency overlap)
                float4 rr[8];
                if (p.res_mode == RES_UPSAMPLE2X) {
                    const float* rp = nullptr;
                    if (row_valid) {
                        const int uy = min((h0 + ph_) >> 1, p.up_h - 1), ux = min((w0 + pw_) >> 1, p.up_w - 1);
                        rp = p.up_src + (((size_t)(n0img + pn_) * p.up_h + uy) * p.up_w + ux) * (size_t)p.cout + ch0;
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        rr[j] = (rp != nullptr && ch0 + j * 4 < p.cout) ? __ldg(reinterpret_cast<const float4*>(rp) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                // the accumulator read does not depend on the staging slot: request it BEFORE the group barrier, so that the TMEM latency
                // overlaps the wait for thread 0 (slot hand-over / residual issue) instead of following it
                const bool full_chunk = ch0 + 32 <= p.cout;
                uint32_t v[32];
                const uint32_t tbase = tbase0 + (uint32_t)(c * 32);
                tmem_ld_32x32(tbase, v);
                tmem_ld_wait();
#pragma unroll 1
                for (int a = 1; a <= NMAIN; ++a) {      // remaining main accumulators, then the cross accumulator
                    const bool is_cross = (a == NMAIN);
                    if (is_cross ? (p.passes != 3) : (a >= nacc)) continue;
                    uint32_t x[32];
                    tmem_ld_32x32(tbase + (uint32_t)(a * BLOCK_N), x);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(x[j]));
                }
                if (c == last_c) {
                    // this thread's last TMEM read of the tile: hand the accumulators back (256 arrivals release the MMA warp)
                    tc_fence_before();
                    if constexpr (kTwoSM) mbar_arrive_cluster(mapa_cluster(bar_tempty(buf), 0)); else mbar_arrive(bar_tempty(buf));
                }
                const float4* rsrc = nullptr;           // this row's residual line (ring variant)
                if (p.res_mode == RES_TILE) {
                    if constexpr (RING > 0) {
                        const uint32_t rs = (uint32_t)(g * RING) + (gc % RING);
                        mbar_wait(bar_ring(rs), (gc / RING) & 1u);
                        rsrc = reinterpret_cast<const float4*>(ring_gen + rs * Cfg::A_BYTES + row * 128);
                    } else {
                        mbar_wait(bar_res(sidx), (gc / NS) & 1u);
                    }
                }
                float* stg = reinterpret_cast<float*>(slot_gen + row * 128);
                // The chunk's arithmetic runs as PASSES over this row's 32 values with the (warp-uniform) mode branches BETWEEN the passes: inside
                // a pass the 8 pieces are straight-line code, so the 16 scale / shift loads and the shared-memory reads of a pass are all in
                // flight together.  (Per-piece branches serialised them: ncu source view of the stem, 820 executed instructions and ~7600
                // cycles per chunk, a third of the stall samples on the reconvergence points behind the per-piece loads.)
                // (Measured and rejected: fetching the scale / shift vectors ahead of the group barrier -- 64 more live registers spill.)
                float o[32];
                if (full_chunk) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 sc = __ldg(reinterpret_cast<const float4*>(p.scale + ch0) + j);
                        const float4 sh = __ldg(reinterpret_cast<const float4*>(p.shift + ch0) + j);
                        o[4 * j + 0] = fmaf(__uint_as_float(v[4 * j + 0]), sc.x, sh.x);
                        o[4 * j + 1] = fmaf(__uint_as_float(v[4 * j + 1]), sc.y, sh.y);
                        o[4 * j + 2] = fmaf(__uint_as_float(v[4 * j + 2]), sc.z, sh.z);
                        o[4 * j + 3] = fmaf(__uint_as_float(v[4 * j + 3]), sc.w, sh.w);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {       // the last, partial chunk of a Cout that is not a multiple of 32 (cout % 4 == 0: host pads)
                        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ch0 + j * 4 < p.cout) {
                            sc = __ldg(reinterpret_cast<const float4*>(p.scale + ch0) + j);
                            sh = __ldg(reinterpret_cast<const float4*>(p.shift + ch0) + j);
                        }
                        o[4 * j + 0] = fmaf(__uint_as_float(v[4 * j + 0]), sc.x, sh.x);
                        o[4 * j + 1] = fmaf(__uint_as_float(v[4 * j + 1]), sc.y, sh.y);
                        o[4 * j + 2] = fmaf(__uint_as_float(v[4 * j + 2]), sc.z, sh.z);
                        o[4 * j + 3] = fmaf(__uint_as_float(v[4 * j + 3]), sc.w, sh.w);
                    }
                }
                if (p.res_mode == RES_TILE) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int pj = j ^ (row & 7);      // SWIZZLE_128B: 16-byte piece index XOR (row mod 8)
                        const float4 r = (RING > 0) ? rsrc[pj] : reinterpret_cast<const float4*>(stg)[pj];
                        o[4 * j + 0] += r.x; o[4 * j + 1] += r.y; o[4 * j + 2] += r.z; o[4 * j + 3] += r.w;
                    }
                } else if (p.res_mode == RES_UPSAMPLE2X) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) { o[4 * j + 0] += rr[j].x; o[4 * j + 1] += rr[j].y; o[4 * j + 2] += rr[j].z; o[4 * j + 3] += rr[j].w; }
                }
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) o[j] = fmaxf(o[j], 0.f);
                }
                if (ch0 < p.sigmoid_ch) {
                    // torch.sigmoid on CPU evaluates 1/(1+exp(-x)); expf/div are IEEE-rounded here
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (ch0 + j < p.sigmoid_ch) o[j] = 1.f / (1.f + expf(-o[j]));
                }
                // B1: the store warp has seen the store that last used this slot finish reading it (non-ring RES_TILE: the residual tile was
                // loaded into the slot after that, and has been consumed above)
                named_bar_sync(1 + g, 160);
                if (KIND == KIND_F16X3 && p.out_planes) {
                    // two 64-byte-row fp16 tiles in the 16 KB slot (hi | lo), SWIZZLE_64B: this row's 8-byte piece j of the 64-byte line
                    bool bad = false;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float ox = o[4 * j + 0], oy = o[4 * j + 1], oz = o[4 * j + 2], ow = o[4 * j + 3];
                        bad = bad || !(fabsf(ox) < 65504.f) || !(fabsf(oy) < 65504.f) || !(fabsf(oz) < 65504.f) || !(fabsf(ow) < 65504.f);
                        const __half2 h01 = __floats2half2_rn(ox, oy), h23 = __floats2half2_rn(oz, ow);
                        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                        const __half2 l01 = __floats2half2_rn(ox - f01.x, oy - f01.y), l23 = __floats2half2_rn(oz - f23.x, ow - f23.y);
                        const int off = row * 64 + ((((j >> 1) ^ ((row >> 1) & 3)) << 4) | ((j & 1) << 3));
                        uint2 hv, lv;
                        hv.x = *reinterpret_cast<const uint32_t*>(&h01); hv.y = *reinterpret_cast<const uint32_t*>(&h23);
                        lv.x = *reinterpret_cast<const uint32_t*>(&l01); lv.y = *reinterpret_cast<const uint32_t*>(&l23);
                        *reinterpret_cast<uint2*>(slot_gen + off) = hv;
                        *reinterpret_cast<uint2*>(slot_gen + Cfg::A_BYTES / 2 + off) = lv;
                    }
                    // (out_planes layers have Cout % 32 == 0: every channel of the chunk is live)
                    if (bad && p.range_flag && row * 128 < p.a_tile_bytes) *p.range_flag = 1;
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        reinterpret_cast<float4*>(stg)[j ^ (row & 7)] = make_float4(o[4 * j + 0], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                }
                fence_proxy_async_smem();
                named_bar_arrive(4 + g, 160);           // B2: this row of the staging slot is written; the store warp takes it from here
            }
        }
        }
    }

    // ---- teardown: neither CTA may exit while the peer can still multicast into it or arrive on its barriers
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        if constexpr (kTwoSM) tmem_dealloc_2sm<Cfg::TMEM_COLS>(tmem_acc); else tmem_dealloc<Cfg::TMEM_COLS>(tmem_acc);
    }
}

}  // namespace dt
