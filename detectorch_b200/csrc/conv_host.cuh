// detectorch_b200 -- host side of the tcgen05 conv/GEMM engine: TMA descriptor construction,
// tile-geometry selection and launch.  No torch types; raw device pointers only.
#pragma once
#include <cudaTypedefs.h>
#include <stdlib.h>
#include <string.h>

#include "conv_tcgen05.cuh"

namespace dt {

// cuTensorMapEncodeTiled is a driver entry point; fetch it through the runtime so that the
// library links against cudart only (libcuda is resolved by the driver at load time).
inline PFN_cuTensorMapEncodeTiled_v12000 get_tmap_encode() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) {
            fprintf(stderr, "[detectorch_b200] cuTensorMapEncodeTiled unavailable (%s)\n", cudaGetErrorString(e));
            return nullptr;
        }
        fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
    }
    return fn;
}

// 4D fp32 tensor map {d0 (contiguous), d1, d2, d3} with byte strides s1,s2,s3, SWIZZLE_128B
inline bool make_tmap_4d(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint64_t s1,
                         uint64_t s2, uint64_t s3, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3, uint32_t e1 = 1,
                         uint32_t e2 = 1) {
    auto fn = get_tmap_encode();
    if (!fn) return false;
    cuuint64_t dims[4] = {d0, d1, d2, d3};
    cuuint64_t strides[3] = {s1, s2, s3};
    cuuint32_t box[4] = {b0, b1, b2, b3};
    cuuint32_t estr[4] = {1, e1, e2, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr,
                "[detectorch_b200] cuTensorMapEncodeTiled(4d) failed: %d dims=(%llu,%llu,%llu,%llu) strides=(%llu,%llu,%llu) "
                "box=(%u,%u,%u,%u) estr=(%u,%u)\n",
                (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, (unsigned long long)d3,
                (unsigned long long)s1, (unsigned long long)s2, (unsigned long long)s3, b0, b1, b2, b3, e1, e2);
        return false;
    }
    return true;
}

inline bool make_tmap_2d(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t s1, uint32_t b0, uint32_t b1) {
    auto fn = get_tmap_encode();
    if (!fn) return false;
    cuuint64_t dims[2] = {d0, d1};
    cuuint64_t strides[1] = {s1};
    cuuint32_t box[2] = {b0, b1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "[detectorch_b200] cuTensorMapEncodeTiled(2d) failed: %d dims=(%llu,%llu) stride=%llu box=(%u,%u)\n", (int)r,
                (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)s1, b0, b1);
        return false;
    }
    return true;
}

// 2D fp16 weight map {K (contiguous), rows}, box {32 elements = 64 bytes, rows}, SWIZZLE_64B (KIND_F16X3)
inline bool make_tmap_2d_f16(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t s1, uint32_t b0, uint32_t b1) {
    auto fn = get_tmap_encode();
    if (!fn) return false;
    cuuint64_t dims[2] = {d0, d1};
    cuuint64_t strides[1] = {s1};
    cuuint32_t box[2] = {b0, b1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "[detectorch_b200] cuTensorMapEncodeTiled(2d f16) failed: %d dims=(%llu,%llu) stride=%llu box=(%u,%u)\n", (int)r,
                (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)s1, b0, b1);
        return false;
    }
    return true;
}

// 4D fp16 plane map {C (contiguous), W, H, N}, box {32 channels = 64 bytes, ...}, SWIZZLE_64B (activations handed over as hi/lo planes)
inline bool make_tmap_4d_f16(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint64_t s1, uint64_t s2,
                             uint64_t s3, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3, uint32_t e1 = 1, uint32_t e2 = 1) {
    auto fn = get_tmap_encode();
    if (!fn) return false;
    cuuint64_t dims[4] = {d0, d1, d2, d3};
    cuuint64_t strides[3] = {s1, s2, s3};
    cuuint32_t box[4] = {b0, b1, b2, b3};
    cuuint32_t estr[4] = {1, e1, e2, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "[detectorch_b200] cuTensorMapEncodeTiled(4d f16) failed: %d dims=(%llu,%llu,%llu,%llu) box=(%u,%u,%u,%u)\n", (int)r,
                (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, (unsigned long long)d3, b0, b1, b2, b3);
        return false;
    }
    return true;
}

// A conv layer instance: everything needed to (re)launch it.  Built once per (layer, shape).
struct ConvLayer {
    ConvParams p;
    int block_n;
    int nmain = 1;      // rotating main-term accumulators (3 = precise: shorter truncating accumulation chains)
    bool two_sm = true; // cta_group::2 MMA (default) vs 1-SM MMA + multicast (DT_CONV_1SM=1)
    int kind = KIND_TF32X3;
    int ring = 0;       // residual prefetch ring (short-K RES_TILE layers)
    int slots = 1;      // epilogue staging slots per group (2 = the TMA store of a chunk drains while the next chunk is computed)
    bool ws = false;    // weight-stationary halo kernel (64-wide, one N tile): the whole weight matrix stays resident in shared memory
    int halo = 0;       // 1 = 3x3 halo variant: one (8 + 2)-pixel-wide A box per filter row serves its three taps; 2 = stem row-parity halo
    dim3 grid;
    bool valid = false;
};

// Logical description of one convolution over NHWC fp32 tensors.
struct ConvSpec {
    const float* x; int N, H, W, Cin;          // input  [N,H,W,Cin], Cin % 32 == 0
    int x_pix_stride;                          // floats between consecutive pixels of x (>= Cin; lets x be a channel slice)
    const void* w_hi; const void* w_lo;        // [Cout_rows][kh*kw*Cin] K-major: fp32 (w, w - trunc_tf32(w)) or fp16 (hi, lo) for KIND_F16X3
    int kind;                                  // ConvKind
    int* range_flag;                           // KIND_F16X3: device flag raised when an activation does not fit fp16
    int Cout;                                  // output channels, multiple of 4
    int kh, kw, pad, stride;
    const float* scale; const float* shift;    // [Cout]
    float* y; int y_pix_stride;                // output [N,Ho,Wo,*], y_pix_stride floats between pixels (>= Cout)
    // optional output remap (transposed conv): pixel (n,h,w) is written at y + ((n*Hy + h*ys + yo)*Wy + w*ys + xo)*y_pix_stride
    int out_h, out_w, out_step, out_y0, out_x0;   // out_step==0 -> plain [N,Ho,Wo]
    const float* residual; int res_pix_stride;    // RES_TILE: same geometry as the (plain) output
    const float* up_src; int up_h, up_w;          // RES_UPSAMPLE2X
    int res_mode, relu, sigmoid_ch, passes;
    // fp16 hi/lo plane hand-over between two KIND_F16X3 layers (dense channel stride only): x / y then point at the HIGH plane and
    // x_lo / y_lo at the LOW plane, each [N,H,W,C] fp16
    const void* x_lo; void* y_lo;
    int tap0, ntaps;                              // K-split: only filter taps [tap0, tap0+ntaps) (ntaps == 0: all kh*kw)
    int force_block_n;                            // 0 = auto
    int precise;                                  // BLOCK_N == 128 only: 3 rotating accumulators instead of TMEM double-buffering
    int no_merge;                                 // keep the cross terms in their own accumulator whatever K is (mask head: tightest parity bar)
    float x_mult;                                 // KIND_F16X3, fp32 input: power of two applied to x before the fp16 split (0 or 1: none);
                                                  // the caller folds 1 / x_mult into scale.  Keeps the low half of small activations normal.
};

inline void choose_box(int Wo, int Ho, int N, int max_w, int* wbox, int* hbox, int* nbox) {
    long best_tiles = -1;
    int bw = 1, bh = 1, bn = 1;
    for (int w = 1; w <= Wo && w <= 128 && w <= max_w; ++w) {
        for (int h = 1; h <= Ho && w * h <= 128; ++h) {
            int n = 128 / (w * h);
            if (n > N) n = N;
            if (n < 1) n = 1;
            long tiles = (long)ceil_div(Wo, w) * ceil_div(Ho, h) * ceil_div(N, n);
            if (best_tiles < 0 || tiles < best_tiles || (tiles == best_tiles && w > bw)) {
                best_tiles = tiles; bw = w; bh = h; bn = n;
            }
        }
    }
    *wbox = bw; *hbox = bh; *nbox = bn;
}

// MMA mode per layer.  cta_group::2 (each SM keeps half of the weight tile: smaller stages, half the B-operand ingest and shared-memory
// reads per SM) measured 1-22 % faster on every 128- and 256-wide layer once the cluster-scope fences were gone from the per-k-block
// signalling; the 64-wide layers (stem, 64-channel stage, RPN heads) are a wash or up to 5 % slower, so they stay on 1-SM MMAs with
// multicast weights.  DT_CONV_MMA=1sm|2sm forces one mode everywhere (tests exercise both).
inline bool conv_use_two_sm(int block_n, int num_kb) {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DT_CONV_MMA");
        v = (e && e[0] == '1') ? 1 : ((e && e[0] == '2') ? 2 : 0);
    }
    if (v == 1) return false;
    if (v == 2) return true;
    (void)num_kb;
    return block_n > 64;
}

inline bool conv_merge_acc(int num_kb) {
    static int thr = -1;
    if (thr < 0) { const char* e = getenv("DT_CONV_MERGE_KB"); thr = e ? atoi(e) : 72; }
    return num_kb <= thr;
}

// DT_CONV_HALO=0 switches the halo variant of the 64 / 128-wide 3x3 plane-input layers off (A/B, tests)
inline bool conv_use_halo() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("DT_CONV_HALO"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

// weight-stationary form of the 64-wide halo kernels: DT_CONV_WS=0 off, 1 (default) the stem only, 2 also the 64-channel 3x3 layers
inline int conv_ws_mode() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("DT_CONV_WS"); v = e ? atoi(e) : 1; }
    return v;
}

// DT_CONV_NARROW1=0: 64-wide short-K layers and the stem keep 3 rotating accumulators (A/B, tests)
inline bool conv_narrow_one_acc() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("DT_CONV_NARROW1"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

// Persistent launch geometry: work items = (pairs of M-tiles) x (N-tiles); one 2-CTA cluster per SM pair (74 on B200),
// each looping over items pair, pair + num_pairs, ...  An odd M-tile count gets one all-out-of-range surplus tile (TMA
// zero-fills its loads and clips its stores) so that both CTAs of a pair always run the same multicast protocol.
inline void finish_grid(ConvLayer* L, int n_tiles) {
    ConvParams& p = L->p;
    const int mtiles = p.tiles_w * p.tiles_h * p.tiles_n;
    p.m_pairs = (mtiles + 1) / 2;
    p.n_tiles = n_tiles;
    const int items = p.m_pairs * p.n_tiles;
    const int pairs = items < kNumSMs / 2 ? items : kNumSMs / 2;
    L->two_sm = conv_use_two_sm(L->block_n, p.kh * p.kw * p.cin_blocks);
    L->grid = dim3((unsigned)(2 * pairs), 1, 1);
    L->valid = true;
}

inline bool conv_build(const ConvSpec& s, ConvLayer* L) {
    memset(&L->p, 0, sizeof(ConvParams));
    ConvParams& p = L->p;
    if (s.Cin % 32 != 0 || s.Cout % 4 != 0) {
        fprintf(stderr, "[detectorch_b200] conv_build: Cin must be a multiple of 32 and Cout of 4 (got %d, %d)\n", s.Cin, s.Cout);
        return false;
    }
    const int Ho = (s.H + 2 * s.pad - s.kh) / s.stride + 1;
    const int Wo = (s.W + 2 * s.pad - s.kw) / s.stride + 1;
    int wbox, hbox, nbox;
    choose_box(Wo, Ho, s.N, 256 / s.stride, &wbox, &hbox, &nbox);
    int bn = s.force_block_n;
    if (bn == 0) bn = s.Cout > 128 ? 256 : (s.Cout > 64 ? 128 : 64);
    L->block_n = bn;
    // Halo variant (conv_tcgen05.cuh): 3x3 / stride 1 / pad 1 over fp16 planes, tiles up to 128 channels wide in the two instantiations
    // the engine uses for them (64: 1-SM MMA, 3 rotating accumulators; 128: 2-SM MMA, 1 accumulator).  Tiles are 8 pixels wide and
    // (hbox x nbox) = 16 rows high; the A box is 10 pixels wide.
    L->halo = conv_use_halo() && s.x_lo && s.kind == KIND_F16X3 && s.kh == 3 && s.kw == 3 && s.stride == 1 && s.pad == 1 && s.ntaps == 0 &&
              s.passes != 1 && s.W >= 10 && ((bn == 64 && !conv_use_two_sm(64, 0)) || (bn == 128 && conv_use_two_sm(128, 0) && !s.precise));
    if (L->halo) {
        long best = -1;
        for (int h = 16; h >= 1; h >>= 1) {
            const int n = 16 / h;
            if (h > s.H || n > s.N) continue;
            const long tiles = (long)ceil_div(Wo, 8) * ceil_div(Ho, h) * ceil_div(s.N, n);
            if (best < 0 || tiles < best) { best = tiles; hbox = h; nbox = n; }
        }
        if (best < 0) L->halo = 0; else wbox = 8;
    }
    if (s.x_mult != 0.f && s.x_mult != 1.f && (s.kind != KIND_F16X3 || s.x_lo)) {
        fprintf(stderr, "[detectorch_b200] conv_build: an input multiplier needs the f16 kind and an fp32 input\n");
        return false;
    }
    const int abox_w = L->halo ? wbox + 2 : wbox * s.stride;
    const int K = s.kh * s.kw * s.Cin;
    const uint64_t xs = (uint64_t)s.x_pix_stride * 4;
    if (s.x_lo) {
        if (s.kind != KIND_F16X3 || s.x_pix_stride != s.Cin) { fprintf(stderr, "[detectorch_b200] conv_build: fp16 input planes need the f16 kind and a dense layout\n"); return false; }
        const uint64_t hs = (uint64_t)s.Cin * 2;
        if (!make_tmap_4d_f16(&p.tm_a, s.x, s.Cin, s.W, s.H, s.N, hs, hs * s.W, hs * s.W * s.H, 32, abox_w, hbox * s.stride, nbox, s.stride, s.stride) ||
            !make_tmap_4d_f16(&p.tm_a2, s.x_lo, s.Cin, s.W, s.H, s.N, hs, hs * s.W, hs * s.W * s.H, 32, abox_w, hbox * s.stride, nbox, s.stride, s.stride))
            return false;
        p.a_planes = 1;
    } else if (!make_tmap_4d(&p.tm_a, s.x, s.Cin, s.W, s.H, s.N, xs, xs * s.W, xs * s.W * s.H, 32, wbox * s.stride, hbox * s.stride, nbox,
                             s.stride, s.stride))
        return false;
    // each CTA of a pair fetches half of the BLOCK_N weight rows and multicasts them
    if (s.kind == KIND_F16X3) {
        if (!make_tmap_2d_f16(&p.tm_bhi, s.w_hi, K, s.Cout, (uint64_t)K * 2, 32, bn / 2)) return false;
        if (!make_tmap_2d_f16(&p.tm_blo, s.w_lo ? s.w_lo : s.w_hi, K, s.Cout, (uint64_t)K * 2, 32, bn / 2)) return false;
    } else {
        if (!make_tmap_2d(&p.tm_bhi, s.w_hi, K, s.Cout, (uint64_t)K * 4, 32, bn / 2)) return false;
        if (!make_tmap_2d(&p.tm_blo, s.w_lo ? s.w_lo : s.w_hi, K, s.Cout, (uint64_t)K * 4, 32, bn / 2)) return false;
    }
    L->kind = s.kind == KIND_F16X3 ? KIND_F16X3 : KIND_TF32X3;
    p.range_flag = s.range_flag;
    p.a_mult = (s.x_mult != 1.f) ? s.x_mult : 0.f;
    const uint64_t ys = (uint64_t)s.y_pix_stride * 4;
    if (s.y_lo) {
        if (s.kind != KIND_F16X3 || s.out_step != 0 || s.y_pix_stride != s.Cout || s.res_mode != RES_NONE || (s.Cout % 32) != 0) {
            fprintf(stderr, "[detectorch_b200] conv_build: fp16 output planes need the f16 kind, a dense layout, Cout %% 32 == 0 and no residual\n");
            return false;
        }
        const uint64_t hs = (uint64_t)s.Cout * 2;
        if (!make_tmap_4d_f16(&p.tm_d, s.y, s.Cout, Wo, Ho, s.N, hs, hs * Wo, hs * Wo * Ho, 32, wbox, hbox, nbox) ||
            !make_tmap_4d_f16(&p.tm_d2, s.y_lo, s.Cout, Wo, Ho, s.N, hs, hs * Wo, hs * Wo * Ho, 32, wbox, hbox, nbox))
            return false;
        p.out_planes = 1;
    } else if (s.out_step == 0) {
        if (!make_tmap_4d(&p.tm_d, s.y, s.Cout, Wo, Ho, s.N, ys, ys * Wo, ys * Wo * Ho, 32, wbox, hbox, nbox)) return false;
    } else {
        if (s.out_step < 0 || s.out_y0 < 0 || s.out_x0 < 0 || (Ho - 1) * s.out_step + s.out_y0 >= s.out_h ||
            (Wo - 1) * s.out_step + s.out_x0 >= s.out_w) {
            fprintf(stderr, "[detectorch_b200] conv_build: the output remap scatters outside the [N,out_h,out_w] map\n");
            return false;
        }
        // strided scatter view: logical (w,h) -> physical (w*step + x0, h*step + y0) of an [N,out_h,out_w] map
        const float* base = s.y + ((size_t)s.out_y0 * s.out_w + s.out_x0) * s.y_pix_stride;
        if (!make_tmap_4d(&p.tm_d, base, s.Cout, Wo, Ho, s.N, ys * s.out_step, ys * s.out_w * s.out_step, ys * s.out_w * s.out_h, 32,
                          wbox, hbox, nbox))
            return false;
    }
    if (s.res_mode == RES_TILE) {
        const uint64_t rs = (uint64_t)s.res_pix_stride * 4;
        if (!make_tmap_4d(&p.tm_r, s.residual, s.Cout, Wo, Ho, s.N, rs, rs * Wo, rs * Wo * Ho, 32, wbox, hbox, nbox)) return false;
    }
    p.scale = s.scale; p.shift = s.shift;
    p.up_src = s.up_src; p.up_h = s.up_h; p.up_w = s.up_w;
    p.cin_blocks = s.Cin / 32;
    p.kh = s.kh; p.kw = s.kw; p.pad_w = p.pad_h = s.pad; p.stride_w = p.stride_h = s.stride;
    p.tap0 = s.ntaps > 0 ? s.tap0 : 0; p.ntaps = s.ntaps > 0 ? s.ntaps : s.kh * s.kw;
    if (p.tap0 < 0 || p.tap0 + p.ntaps > s.kh * s.kw) { fprintf(stderr, "[detectorch_b200] conv_build: bad tap range\n"); return false; }
    p.tiles_w = ceil_div(Wo, wbox); p.tiles_h = ceil_div(Ho, hbox); p.tiles_n = ceil_div(s.N, nbox);
    p.wbox = wbox; p.hbox = hbox; p.nbox = nbox;
    p.wo = Wo; p.ho = Ho; p.nimg = s.N;
    p.cout = s.Cout;
    p.a_tile_bytes = wbox * hbox * nbox * 128;
    p.a_halo_bytes = L->halo ? (wbox + 2) * hbox * nbox * 64 : 0;
    p.relu = s.relu; p.sigmoid_ch = s.sigmoid_ch; p.res_mode = s.res_mode;
    p.passes = s.passes == 1 ? 1 : 3;
    // 256-wide tiles: (main + cross) accumulators fill the 512 TMEM columns, so the epilogue cannot overlap the next tile's MMAs.  One
    // merged accumulator leaves room for two tiles (measured: -0.7 ms per step when applied to every layer up to K = 2304); the price is
    // a 3x longer truncating-accumulate chain (main and both cross terms in one accumulator), which the trunk / FPN / RPN / box-head
    // activations can afford (they sit at 1e-5 of their 1e-4 bar) and the mask-head layers cannot (no_merge).
    // 64-wide tiles rotate the main term over 3 accumulators (short truncating-accumulate chains at no TMEM cost) -- except at K <= 256, where
    // one accumulator already is a chain of at most 16 steps and the two extra TMEM reads + RN adds per chunk only lengthen the epilogue
    const bool narrow1 = bn == 64 && s.kind == KIND_F16X3 && !L->halo && p.ntaps * p.cin_blocks <= 8 && conv_narrow_one_acc();
    L->nmain = (bn == 64) ? (narrow1 ? 1 : 3) : ((bn == 128 && s.precise) ? 3 : ((bn == 256 && !s.no_merge && conv_merge_acc(p.ntaps * p.cin_blocks)) ? 0 : 1));
    finish_grid(L, ceil_div(s.Cout, bn));
    {
        // Residual prefetch ring for the conv3 + residual layers (K <= 512): -15..26 % at K <= 256 when it was introduced; K = 512 (16 k-blocks
        // per tile) was 11 % slower with it while a ring kernel had two 48 KB pipeline stages -- with in-place 32 KB stages it gains 15 %
        // with 3 ring tiles / 3 stages and 23 % with 2 ring tiles / 4 stages (same-box sweep over DT_CONV_RING_KB / DT_CONV_RING2_KB).
        static int use_ring = -1, ring_kb = 16, ring2_kb = 16;
        if (use_ring < 0) {
            const char* e = getenv("DT_CONV_RES_RING"); use_ring = e ? atoi(e) : 1;
            const char* e1 = getenv("DT_CONV_RING_KB"); if (e1) ring_kb = atoi(e1);             // ring for at most this many k-blocks per tile
            const char* e2 = getenv("DT_CONV_RING2_KB"); if (e2) ring2_kb = atoi(e2);           // from this many k-blocks on: 2 ring tiles (one more stage)
        }
        L->ring = (use_ring && L->nmain == 0 && L->two_sm && L->kind == KIND_F16X3 && s.res_mode == RES_TILE && p.ntaps * p.cin_blocks <= ring_kb) ? 1 : 0;
        if (L->ring && ring2_kb > 0 && p.ntaps * p.cin_blocks >= ring2_kb) L->ring = 2;
    }
    {
        // Two staging slots per epilogue group (the TMA store of a chunk drains while the next chunk is computed) for tiles up to 128 wide,
        // where the extra 32 KB do not cost a pipeline stage.  256-wide tiles take ONE slot = one more pipeline stage: since the store warps
        // decoupled the stores from the workers, the second slot no longer pays for itself there (same-box sweep, profiles/r02_summary.md:
        // short-K 256-wide layers -5..20 % with one slot, long-K +15 % with two; with the stores still issued by worker thread 0 the
        // short-K layers had been 10-16 % faster with two).  DT_CONV_SLOTS=1|2 forces one setting (A/B, tests).
        static int force = -1;
        if (force < 0) { const char* e = getenv("DT_CONV_SLOTS"); force = e ? atoi(e) : 0; }
        L->slots = bn <= 128 ? 2 : 1;
        if (force == 1 || force == 2) L->slots = force;
        if (L->halo) L->slots = 2;
    }
    // weight-stationary form of the 64-wide 3x3 halo layer (one N tile, all 18 k-blocks resident, 2-SM MMA): measured a wash to +4 % slower
    // than the streaming form (167 -> 175 us; the stem gains 17 %), so it is opt-in here (DT_CONV_WS=2)
    L->ws = L->halo == 1 && bn == 64 && conv_ws_mode() == 2 && s.Cout <= 64 && s.kh * s.kw * p.cin_blocks <= 18;
    if (L->ws) L->two_sm = true;
    if (L->nmain == 1 && bn == 64 && L->slots != 2) L->nmain = 3;       // the one-accumulator 64-wide kernel exists with two staging slots only
    if (L->halo && (L->nmain != (bn == 64 ? 3 : 1) || L->two_sm != (bn == 128 || L->ws) || L->ring)) {
        fprintf(stderr, "[detectorch_b200] conv_build: halo layer ended up in an instantiation the halo kernel does not cover\n");
        return false;
    }
    return true;
}

// The 7x7 stride-2 stem (3 input channels) as an implicit GEMM without an im2col buffer: the image is repacked once as
// zero-bordered NHWC4 [B, Hp, Wp, 4]; for filter row ky the 7 taps x 4 channels of an output pixel are 28 CONTIGUOUS floats
// starting at padded pixel 2*ow, so a TMA descriptor whose "pixel" dimension has an OVERLAPPING stride of 8 floats
// (2 pixels) delivers, per ky, one 32-float K-block per output pixel straight into the swizzled A tile (last 4 floats
// hit zero weights).  K = 7 x 32.  H uses elementStride 2.
inline bool conv_build_stem(const float* x4, int B, int Hp, int Wp, int H1, int W1, const void* w_hi, const void* w_lo, const float* scale,
                            const float* shift, float* y, int passes, ConvLayer* L, int kind = KIND_TF32X3, int* range_flag = nullptr,
                            bool x4_planes = false, float x_mult = 0.f) {
    memset(&L->p, 0, sizeof(ConvParams));
    ConvParams& p = L->p;
    int wbox, hbox, nbox;
    choose_box(W1, H1, B, 256, &wbox, &hbox, &nbox);
    const int bn = 64;
    L->block_n = bn;
    L->halo = 0;
    const uint64_t row = (uint64_t)Wp * 16;
    if (x4_planes) {
        // x4 holds two fp16 planes [B, Hp, Wp, 4] back to back (hi, lo): same overlapping-stride window, 16 bytes (2 pixels) per step
        if (kind != KIND_F16X3 || (Wp & 1)) return false;
        const __half* xh = reinterpret_cast<const __half*>(x4);
        const __half* xl = xh + (size_t)B * Hp * Wp * 4;
        const uint64_t rowh = (uint64_t)Wp * 8;
        // row-parity halo (conv_tcgen05.cuh, HALO == 2): tiles of 8 x 16 pixels of one image, A boxes of 16 + 3 stride-2 row slabs
        L->halo = (conv_use_halo() && H1 >= 16 && W1 >= 8 && !conv_use_two_sm(64, 0)) ? 2 : 0;
        if (L->halo) { wbox = 8; hbox = 16; nbox = 1; }
        const int abox_h = L->halo ? (hbox + 3) * 2 : hbox * 2;
        if (!make_tmap_4d_f16(&p.tm_a, xh, 32, W1, Hp, B, 16, rowh, rowh * Hp, 32, wbox, abox_h, nbox, 1, 2) ||
            !make_tmap_4d_f16(&p.tm_a2, xl, 32, W1, Hp, B, 16, rowh, rowh * Hp, 32, wbox, abox_h, nbox, 1, 2))
            return false;
        p.a_planes = 1;
        p.a_halo_bytes = L->halo ? wbox * (hbox + 3) * 64 : 0;
    } else if (!make_tmap_4d(&p.tm_a, x4, 32, W1, Hp, B, 32, row, row * Hp, 32, wbox, hbox * 2, nbox, 1, 2)) return false;
    if (kind == KIND_F16X3) {
        if (!make_tmap_2d_f16(&p.tm_bhi, w_hi, 224, 64, 224 * 2, 32, bn / 2)) return false;
        if (!make_tmap_2d_f16(&p.tm_blo, w_lo, 224, 64, 224 * 2, 32, bn / 2)) return false;
    } else {
        if (!make_tmap_2d(&p.tm_bhi, w_hi, 224, 64, 224 * 4, 32, bn / 2)) return false;
        if (!make_tmap_2d(&p.tm_blo, w_lo, 224, 64, 224 * 4, 32, bn / 2)) return false;
    }
    L->kind = kind == KIND_F16X3 ? KIND_F16X3 : KIND_TF32X3;
    p.range_flag = range_flag;
    if (x_mult != 0.f && x_mult != 1.f) {
        if (kind != KIND_F16X3 || x4_planes) return false;
        p.a_mult = x_mult;
    }
    const uint64_t ys = 64 * 4;
    if (!make_tmap_4d(&p.tm_d, y, 64, W1, H1, B, ys, ys * W1, ys * W1 * H1, 32, wbox, hbox, nbox)) return false;
    p.scale = scale; p.shift = shift;
    p.cin_blocks = 1; p.kh = 7; p.kw = 1; p.tap0 = 0; p.ntaps = 7;
    p.pad_w = 0; p.pad_h = 0; p.stride_w = 1; p.stride_h = 2;
    p.tiles_w = ceil_div(W1, wbox); p.tiles_h = ceil_div(H1, hbox); p.tiles_n = ceil_div(B, nbox);
    p.wbox = wbox; p.hbox = hbox; p.nbox = nbox;
    p.wo = W1; p.ho = H1; p.nimg = B; p.cout = 64;
    p.a_tile_bytes = wbox * hbox * nbox * 128;
    p.relu = 1; p.sigmoid_ch = 0; p.res_mode = RES_NONE; p.passes = passes == 1 ? 1 : 3;
    L->nmain = 3;
    L->slots = 2;
    finish_grid(L, 1);
    L->ws = L->halo == 2 && conv_ws_mode() >= 1;
    if (L->ws) L->two_sm = true;
    if (L->ws && conv_narrow_one_acc()) L->nmain = 1;       // K = 7 k-blocks: one main accumulator (see conv_build)
    return true;
}

// DT_CONV_PDL=1: conv launches carry the programmatic-stream-serialization attribute (see griddep_wait in common.cuh): the prologue of
// launch i+1 overlaps the tail of launch i.  Only conv launches take part; every other kernel keeps plain stream order.
inline bool conv_use_pdl() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("DT_CONV_PDL"); v = (e && e[0] == '1') ? 1 : 0; }
    return v == 1;
}

template <int BN, int NM, bool TWO, int KIND, int RING = 0, int SLOTS = 1, int HALO = 0, bool WS = false>
inline cudaError_t conv_launch_cfg(const ConvLayer& L, cudaStream_t stream) {
    using Cfg = ConvCfg<BN, NM, TWO, KIND, RING, SLOTS, HALO, WS>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(conv_tcgen05_kernel<BN, NM, TWO, KIND, RING, SLOTS, HALO, WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    if (conv_use_pdl()) {
        ConvParams prm = L.p;
        prm.pdl = 1;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = L.grid; cfg.blockDim = dim3(Cfg::THREADS, 1, 1); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, conv_tcgen05_kernel<BN, NM, TWO, KIND, RING, SLOTS, HALO, WS>, prm);
    }
    conv_tcgen05_kernel<BN, NM, TWO, KIND, RING, SLOTS, HALO, WS><<<L.grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(L.p);
    return cudaGetLastError();
}

// Every instantiation of conv_tcgen05_kernel, one row each.  conv_instance_of() maps a built layer to its row; the launcher and the
// plan report (dt_conv2d_spec) both go through it, and dt_conv_instantiation_info exports the table.
struct ConvInstance {
    int bn, nmain, two_sm, kind, ring, slots, halo, ws;
    cudaError_t (*launch)(const ConvLayer&, cudaStream_t);
};
#define DT_CONV_ROW(BN, NM, TWO, KIND, RING, SLOTS, HALO, WS) \
    { BN, NM, TWO, KIND, RING, SLOTS, HALO, WS, &conv_launch_cfg<BN, NM, (TWO != 0), KIND, RING, SLOTS, HALO, (WS != 0)> }
static const ConvInstance kConvInstances[] = {
    // halo forms (kind::f16, fp16-plane input): 3x3 (HALO 1) and the stem (HALO 2)
    DT_CONV_ROW(128, 1, 1, KIND_F16X3, 0, 2, 1, 0), DT_CONV_ROW(64, 3, 1, KIND_F16X3, 0, 2, 1, 1), DT_CONV_ROW(64, 1, 1, KIND_F16X3, 0, 2, 2, 1),
    DT_CONV_ROW(64, 3, 1, KIND_F16X3, 0, 2, 2, 1), DT_CONV_ROW(64, 3, 0, KIND_F16X3, 0, 2, 1, 0), DT_CONV_ROW(64, 3, 0, KIND_F16X3, 0, 2, 2, 0),
    // kind::f16, 2-SM MMA
    DT_CONV_ROW(64, 1, 1, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(64, 3, 1, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(64, 3, 1, KIND_F16X3, 0, 1, 0, 0),
    DT_CONV_ROW(128, 3, 1, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(128, 3, 1, KIND_F16X3, 0, 1, 0, 0), DT_CONV_ROW(128, 1, 1, KIND_F16X3, 0, 2, 0, 0),
    DT_CONV_ROW(128, 1, 1, KIND_F16X3, 0, 1, 0, 0),
    // residual prefetch ring: 2 tiles in flight per epilogue group with two staging slots (3 with one slot); ring 3 + 2 slots (possible with
    // 32 KB stages) measured 8-11 % slower than ring 2 + 2 slots
    DT_CONV_ROW(256, 0, 1, KIND_F16X3, 2, 1, 0, 0), DT_CONV_ROW(256, 0, 1, KIND_F16X3, 3, 1, 0, 0), DT_CONV_ROW(256, 0, 1, KIND_F16X3, 2, 2, 0, 0),
    DT_CONV_ROW(256, 0, 1, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(256, 0, 1, KIND_F16X3, 0, 1, 0, 0), DT_CONV_ROW(256, 1, 1, KIND_F16X3, 0, 2, 0, 0),
    DT_CONV_ROW(256, 1, 1, KIND_F16X3, 0, 1, 0, 0),
    // kind::f16, 1-SM MMA + multicast weights
    DT_CONV_ROW(64, 1, 0, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(64, 3, 0, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(64, 3, 0, KIND_F16X3, 0, 1, 0, 0),
    DT_CONV_ROW(128, 3, 0, KIND_F16X3, 0, 2, 0, 0), DT_CONV_ROW(128, 3, 0, KIND_F16X3, 0, 1, 0, 0), DT_CONV_ROW(128, 1, 0, KIND_F16X3, 0, 2, 0, 0),
    DT_CONV_ROW(128, 1, 0, KIND_F16X3, 0, 1, 0, 0), DT_CONV_ROW(256, 0, 0, KIND_F16X3, 0, 1, 0, 0), DT_CONV_ROW(256, 1, 0, KIND_F16X3, 0, 1, 0, 0),
    // 3xTF32 (one staging slot: the tf32 kind's stages are 64-96 KB)
    DT_CONV_ROW(64, 3, 1, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(128, 3, 1, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(128, 1, 1, KIND_TF32X3, 0, 1, 0, 0),
    DT_CONV_ROW(256, 0, 1, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(256, 1, 1, KIND_TF32X3, 0, 1, 0, 0),
    DT_CONV_ROW(64, 3, 0, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(128, 3, 0, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(128, 1, 0, KIND_TF32X3, 0, 1, 0, 0),
    DT_CONV_ROW(256, 0, 0, KIND_TF32X3, 0, 1, 0, 0), DT_CONV_ROW(256, 1, 0, KIND_TF32X3, 0, 1, 0, 0),
};
#undef DT_CONV_ROW
constexpr int kNumConvInstances = (int)(sizeof(kConvInstances) / sizeof(kConvInstances[0]));

// The row a built layer runs: its fields, with the combinations a kernel does not exist for folded onto the one that runs them
// (the tf32 kind and the 1-SM 256-wide tiles have one staging slot; ring layers are told apart by ring size and slots).  -1: none.
inline int conv_instance_of(const ConvLayer& L) {
    if (!L.valid) return -1;
    const bool f16 = L.kind == KIND_F16X3, two = L.two_sm;
    const bool s2 = f16 && L.slots == 2;
    int nm = L.nmain, ring = 0, slots = s2 ? 2 : 1;
    if (L.halo) {
        if (!f16) return -1;
        if (L.block_n == 64 && L.halo == 1 && !L.ws) nm = 3;
        if (L.block_n == 64 && L.halo == 2 && !L.ws) nm = 3;
        if (L.block_n == 64 && L.halo == 2 && L.ws && nm != 1) nm = 3;
        slots = 2;
    } else if (L.block_n == 64) {
        if (!(f16 && nm == 1 && s2)) nm = 3;
    } else if (L.block_n == 128) {
        if (nm != 3) nm = 1;
    } else if (L.block_n == 256) {
        if (nm == 0 && two && f16 && L.ring) { ring = (s2 || L.ring == 2) ? 2 : 3; }
        else if (!(two && f16)) slots = 1;
        if (nm != 0) nm = 1;
    }
    const int ws = L.ws ? 1 : 0;
    for (int i = 0; i < kNumConvInstances; ++i) {
        const ConvInstance& r = kConvInstances[i];
        if (r.bn == L.block_n && r.nmain == nm && r.two_sm == (two ? 1 : 0) && r.kind == L.kind && r.ring == ring && r.slots == slots &&
            r.halo == L.halo && r.ws == ws)
            return i;
    }
    return -1;
}

inline cudaError_t conv_launch(const ConvLayer& L, cudaStream_t stream) {
    const int i = conv_instance_of(L);
    if (i < 0) return cudaErrorInvalidValue;
    return kConvInstances[i].launch(L, stream);
}

}  // namespace dt
