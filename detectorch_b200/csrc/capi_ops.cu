// detectorch_b200 -- C-ABI entry points for the stand-alone operators (include/detectorch_b200.h).
#include <stdlib.h>

#include "../../include/detectorch_b200.h"
#include "conv_host.cuh"
#include "roi_align.cuh"
#include "roi_align_bwd.cuh"
#include "segm.cuh"
#include "sort_nms.cuh"

using namespace dt;

extern "C" const char* dt_version(void) { return "detectorch_b200 0.1 (sm_100a)"; }

// ================================================================================== RoIAlign
extern "C" int dt_roi_align_forward_nchw(const float* features, const float* rois, int64_t num_rois, int roi_cols, int channels,
                                         int height, int width, int pooled_height, int pooled_width, float spatial_scale,
                                         int sampling_ratio, float* out, dt_stream_t stream) {
    if (num_rois <= 0) return 1;
    if (roi_cols != 4 && roi_cols != 5) {
        fprintf(stderr, "[detectorch_b200] roi_align: rois must have 4 or 5 columns\n");
        return 0;
    }
    const int grid = (int)(num_rois < (int64_t)kNumSMs * 64 ? num_rois : (int64_t)kNumSMs * 64);
    roi_align_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(features, rois, (long long)num_rois, roi_cols, channels, height, width,
                                                                  pooled_height, pooled_width, spatial_scale, sampling_ratio, out);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

extern "C" int launch_roi_align_forward_cuda(const int outputElements, const float* bottom_data, const float* bottom_rois,
                                             const float spatial_scale, const int channels, const int height, const int width,
                                             const int pooled_height, const int pooled_width, const int sampling_ratio,
                                             float* top_data, dt_stream_t stream) {
    const int per_roi = channels * pooled_height * pooled_width;
    if (per_roi <= 0) return 1;
    return dt_roi_align_forward_nchw(bottom_data, bottom_rois, outputElements / per_roi, 5, channels, height, width, pooled_height,
                                     pooled_width, spatial_scale, sampling_ratio, top_data, stream);
}

// Replaces lib/cppcuda_cffi/src/cuda/roi_align_backward_cuda_kernel.h:7-21 (exact signature).  bottom_diff [B,C,H,W] is
// accumulated into (the caller zeroes it, lib/model/roi_align.py:117); nthreads = R*C*ph*pw.
extern "C" int launch_roi_align_backward_cuda(const int nthreads, const float* top_diff, const int num_rois, const float spatial_scale,
                                              const int channels, const int height, const int width, const int pooled_height,
                                              const int pooled_width, const int sampling_ratio, float* bottom_diff, const float* bottom_rois,
                                              int roi_cols, dt_stream_t stream) {
    (void)nthreads;
    if (num_rois <= 0 || channels <= 0) return 1;
    if (roi_cols != 4 && roi_cols != 5) { fprintf(stderr, "[detectorch_b200] roi_align backward: rois must have 4 or 5 columns\n"); return 0; }
    const int grid = num_rois < kNumSMs * 8 ? num_rois : kNumSMs * 8;
    roi_align_backward_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(top_diff, bottom_rois, (long long)num_rois, roi_cols, channels, height,
                                                                          width, pooled_height, pooled_width, spatial_scale, sampling_ratio,
                                                                          bottom_diff);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// ---- deterministic backward (roi_align_bwd.cuh) ------------------------------------------------------------------------------------
namespace {
struct BwdWs { int* counts; long long* offsets; long long* total; uint32_t *k0, *k1; int *v0, *v1, *src; float *wgt, *cnt; };
inline size_t bwd_align(size_t x) { return (x + 255) / 256 * 256; }
inline BwdWs bwd_carve(void* ws, int64_t num_rois, int64_t total) {
    uint8_t* p = reinterpret_cast<uint8_t*>(ws);
    BwdWs w;
    w.counts = reinterpret_cast<int*>(p); p += bwd_align((size_t)num_rois * 4);
    w.offsets = reinterpret_cast<long long*>(p); p += bwd_align((size_t)(num_rois + 1) * 8);
    w.total = reinterpret_cast<long long*>(p); p += 256;
    const size_t m = bwd_align((size_t)total * 4);
    w.k0 = reinterpret_cast<uint32_t*>(p); p += m; w.k1 = reinterpret_cast<uint32_t*>(p); p += m;
    w.v0 = reinterpret_cast<int*>(p); p += m; w.v1 = reinterpret_cast<int*>(p); p += m;
    w.src = reinterpret_cast<int*>(p); p += m; w.wgt = reinterpret_cast<float*>(p); p += m; w.cnt = reinterpret_cast<float*>(p);
    return w;
}
}  // namespace

extern "C" int64_t dt_roi_align_backward_det_workspace_bytes(int64_t num_rois, int64_t total_contributions) {
    return (int64_t)(bwd_align((size_t)num_rois * 4) + bwd_align((size_t)(num_rois + 1) * 8) + 256 + 7 * bwd_align((size_t)total_contributions * 4));
}

// total number of (sample, corner) contributions of this RoI set = the size the workspace must provide; written to *total_dev (device int64).
// scratch: device, >= dt_roi_align_backward_det_workspace_bytes(num_rois, 0) bytes.
extern "C" int dt_roi_align_backward_plan(const float* rois, int64_t num_rois, int roi_cols, float spatial_scale, int pooled_height, int pooled_width,
                                          int sampling_ratio, void* scratch, int64_t* total_dev, dt_stream_t stream) {
    if (roi_cols != 4 && roi_cols != 5) { fprintf(stderr, "[detectorch_b200] roi_align backward: rois must have 4 or 5 columns\n"); return 0; }
    cudaStream_t st = (cudaStream_t)stream;
    if (num_rois <= 0) { DT_CHECK_CUDA(cudaMemsetAsync(total_dev, 0, 8, st)); return 1; }
    BwdWs w = bwd_carve(scratch, num_rois, 0);
    roi_bwd_count_kernel<<<(unsigned)((num_rois + 255) / 256), 256, 0, st>>>(rois, (int)num_rois, roi_cols, spatial_scale, pooled_height, pooled_width,
                                                                            sampling_ratio, w.counts);
    roi_bwd_scan_kernel<<<1, 1024, 0, st>>>(w.counts, (int)num_rois, w.offsets, reinterpret_cast<long long*>(total_dev));
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// Deterministic, atomics-free twin of launch_roi_align_backward_cuda: bottom_diff [B,C,H,W] is accumulated into in exactly the order of the
// reference CPU loop (lib/cppcuda/roi_align_backward_cpu.cpp:79-186) => bit-identical to it and bit-reproducible.  total_contributions is the
// value dt_roi_align_backward_plan produced for these rois; workspace >= dt_roi_align_backward_det_workspace_bytes(num_rois, total).
extern "C" int dt_roi_align_backward_deterministic(const float* top_diff, const float* rois, int64_t num_rois, int roi_cols, int batch, int channels,
                                                   int height, int width, int pooled_height, int pooled_width, float spatial_scale,
                                                   int sampling_ratio, int64_t total_contributions, float* bottom_diff, void* workspace,
                                                   dt_stream_t stream) {
    if (num_rois <= 0 || channels <= 0 || total_contributions <= 0) return 1;
    if (roi_cols != 4 && roi_cols != 5) { fprintf(stderr, "[detectorch_b200] roi_align backward: rois must have 4 or 5 columns\n"); return 0; }
    if (total_contributions >= (1ll << 31) || (int64_t)batch * height * width >= 0xffffffffll) {
        fprintf(stderr, "[detectorch_b200] roi_align deterministic backward: problem too large for the 32-bit sort keys\n");
        return 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    BwdWs w = bwd_carve(workspace, num_rois, total_contributions);
    roi_bwd_count_kernel<<<(unsigned)((num_rois + 255) / 256), 256, 0, st>>>(rois, (int)num_rois, roi_cols, spatial_scale, pooled_height, pooled_width,
                                                                            sampling_ratio, w.counts);
    roi_bwd_scan_kernel<<<1, 1024, 0, st>>>(w.counts, (int)num_rois, w.offsets, w.total);
    const long long bins = (long long)num_rois * pooled_height * pooled_width;
    roi_bwd_emit_kernel<<<(unsigned)((bins + 255) / 256), 256, 0, st>>>(rois, (int)num_rois, roi_cols, spatial_scale, batch, height, width, pooled_height,
                                                                       pooled_width, sampling_ratio, w.offsets, (long long)total_contributions, w.k0,
                                                                       w.v0, w.src, w.wgt, w.cnt);
    roi_bwd_sort_kernel<<<1, 1024, 0, st>>>(w.k0, w.v0, w.k1, w.v1, (int)total_contributions);
    const long long cells = (long long)batch * height * width;
    const int grid = (int)(cells < (long long)kNumSMs * 16 ? cells : (long long)kNumSMs * 16);
    roi_bwd_reduce_kernel<<<grid, 256, 0, st>>>(w.k0, w.v0, (long long)total_contributions, w.src, w.wgt, w.cnt, top_diff, channels, height * width,
                                               cells, pooled_height * pooled_width, bottom_diff);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

extern "C" int dt_roi_align_forward_nhwc(const float* const* feats, const int* heights, const int* widths, const float* scales,
                                         int num_levels, const float* rois, const int* level, const int* num_rois_dev, int max_rois,
                                         int channels, int pooled_height, int pooled_width, int sampling_ratio, float* out,
                                         dt_stream_t stream) {
    if (max_rois <= 0) return 1;
    if (num_levels < 1 || num_levels > 5 || (channels & 3)) {
        fprintf(stderr, "[detectorch_b200] roi_align_nhwc: 1..5 levels and C %% 4 == 0 required\n");
        return 0;
    }
    RoiLevels lv;
    lv.num_levels = num_levels;
    for (int i = 0; i < num_levels; ++i) { lv.feat[i] = feats[i]; lv.H[i] = heights[i]; lv.W[i] = widths[i]; lv.scale[i] = scales[i]; }
    const int grid = max_rois < kNumSMs * 64 ? max_rois : kNumSMs * 64;
    roi_align_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(lv, rois, level, num_rois_dev, max_rois, channels, pooled_height,
                                                                  pooled_width, sampling_ratio, out);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// fast (separable, fused-multiply-add) variants for sampling_ratio == 2 -------------------------------------------------
namespace {
__global__ void nchw_to_nhwc_tr_kernel(const float* __restrict__ x, int HW, int C, float* __restrict__ y) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int c = c0 + r, p = p0 + threadIdx.x;
        tile[r][threadIdx.x] = (p < HW && c < C) ? x[((size_t)b * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int p = p0 + r, c = c0 + threadIdx.x;
        if (c < C && p < HW) y[((size_t)b * HW + p) * C + c] = tile[threadIdx.x][r];
    }
}
}  // namespace

namespace {
// shared-memory-resident map variant: geometry of the launch, or false if the map slab does not fit
struct SmemMapPlan { int group, nwarps, num_chunks, num_items; size_t smem; };
bool smem_map_plan(int batch, int channels, int height, int width, int64_t num_rois, int ph, int pw, SmemMapPlan* pl) {
    static int mode = -1;
    if (mode < 0) { const char* e = getenv("DT_ROI_SMEM_MAP"); mode = e ? atoi(e) : 1; }
    if (!mode) return false;
    if (!((ph == 7 && pw == 7) || (ph == 14 && pw == 14)) || channels % kSlabC) return false;
    const size_t hw = (size_t)height * width;
    if ((size_t)(height - 1) * width > 65535) return false;      // row offsets are packed as uint16
    const size_t map_bytes = ((hw + 7) / 8 * 8) * kSlabC * 4;
    static int nwarps = 0;
    if (!nwarps) { const char* e = getenv("DT_ROI_SMEM_WARPS"); nwarps = e ? atoi(e) : 24; if (nwarps < 4) nwarps = 4; if (nwarps > 24) nwarps = 24; }
    pl->nwarps = nwarps;
    pl->group = 3584 / ((ph + pw) * 32);
    pl->smem = map_bytes + (size_t)pl->nwarps * pl->group * (ph + pw) * 32;
    if (pl->smem > 227 * 1024) return false;
    const int slabs = batch * (channels / kSlabC);
    int a = kNumSMs, b = slabs;
    while (b) { const int t = a % b; a = b; b = t; }
    int chunks = kNumSMs / a;                                        // slabs * chunks is a multiple of the SM count
    const int64_t per_pass = (int64_t)pl->nwarps * pl->group;       // RoIs one CTA covers per sweep of its warps
    const int64_t max_chunks = (num_rois + per_pass - 1) / per_pass;
    if (chunks > max_chunks) chunks = (int)max_chunks;
    pl->num_chunks = chunks < 1 ? 1 : chunks;
    pl->num_items = slabs * pl->num_chunks;
    return true;
}
}  // namespace

extern "C" int64_t dt_roi_align_fast_workspace_bytes(int batch, int channels, int height, int width, int64_t num_rois, int pooled_height,
                                                     int pooled_width) {
    const int64_t nhwc = ((int64_t)batch * channels * height * width * 4 + 255) / 256 * 256;
    const int64_t tables = num_rois * (pooled_height + pooled_width) * (int64_t)sizeof(AxisBinPacked);
    return nhwc + tables;
}

extern "C" int dt_roi_align_forward_nchw_fast(const float* features, int batch, const float* rois, int64_t num_rois, int roi_cols, int channels,
                                              int height, int width, int pooled_height, int pooled_width, float spatial_scale,
                                              int sampling_ratio, float* out, void* workspace, dt_stream_t stream) {
    if (num_rois <= 0) return 1;
    // channel slab: the largest divisor of C (multiple of 4) whose [CS][ph*pw] fp32 tile fits ~50 KB of shared memory
    // smaller tiles = more resident CTAs and more L1 left for the gathers; measured on B200: 28 KB (128 channels x 49 bins)
    // beats 56 / 14 / 7 KB (tunable: DT_ROI_TILE_KB)
    static int tile_kb = 0;
    if (!tile_kb) { const char* e = getenv("DT_ROI_TILE_KB"); tile_kb = e ? atoi(e) : 28; if (tile_kb < 4) tile_kb = 4; if (tile_kb > 100) tile_kb = 100; }
    int cs = 0;
    for (int d = channels; d >= 4; --d)
        if (channels % d == 0 && (d & 3) == 0 && (size_t)d * pooled_height * pooled_width * 4 <= (size_t)tile_kb * 1024 && ((size_t)d * pooled_height * pooled_width * 4) % 16 == 0) { cs = d; break; }
    const size_t tile_bytes = (size_t)cs * pooled_height * pooled_width * 4;
    if (sampling_ratio != 2 || (channels & 3) || pooled_height > kMaxPooled || pooled_width > kMaxPooled || cs == 0) {
        // outside the fast path's envelope: the exact kernel handles every configuration
        return dt_roi_align_forward_nchw(features, rois, num_rois, roi_cols, channels, height, width, pooled_height, pooled_width, spatial_scale,
                                         sampling_ratio, out, stream);
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* nhwc = reinterpret_cast<float*>(workspace);
    const int HW = height * width;
    SmemMapPlan pl;
    if (smem_map_plan(batch, channels, height, width, num_rois, pooled_height, pooled_width, &pl)) {
        AxisBinPacked* tab = reinterpret_cast<AxisBinPacked*>(reinterpret_cast<uint8_t*>(workspace) +
                                                              ((size_t)batch * channels * HW * 4 + 255) / 256 * 256);
        const long long ents = (long long)num_rois * (pooled_height + pooled_width);
        roi_tables_kernel<<<(unsigned)((ents + 255) / 256), 256, 0, st>>>(rois, (long long)num_rois, roi_cols, spatial_scale, height, width,
                                                                         pooled_height, pooled_width, batch, tab);
        DT_CHECK_CUDA(cudaGetLastError());
        const int grid = pl.num_items < kNumSMs ? pl.num_items : kNumSMs;
#define DT_LAUNCH_SMEM_MAP(PHW, BATCHED)                                                                                                   \
    {                                                                                                                                      \
        static bool attr = false;                                                                                                          \
        if (!attr) {                                                                                                                       \
            DT_CHECK_CUDA(cudaFuncSetAttribute(roi_align_smem_map_kernel<PHW, PHW, BATCHED>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                               227 * 1024));                                                                              \
            attr = true;                                                                                                                   \
        }                                                                                                                                  \
        roi_align_smem_map_kernel<PHW, PHW, BATCHED><<<grid, pl.nwarps * 32, pl.smem, st>>>(features, tab, (long long)num_rois, channels,   \
                                                                                           HW, pl.num_items, pl.num_chunks, pl.group, out); \
    }
        if (pooled_height == 7 && batch == 1) DT_LAUNCH_SMEM_MAP(7, false)
        else if (pooled_height == 7) DT_LAUNCH_SMEM_MAP(7, true)
        else if (batch == 1) DT_LAUNCH_SMEM_MAP(14, false)
        else DT_LAUNCH_SMEM_MAP(14, true)
#undef DT_LAUNCH_SMEM_MAP
        DT_CHECK_CUDA(cudaGetLastError());
        return 1;
    }
    nchw_to_nhwc_tr_kernel<<<dim3((HW + 31) / 32, (channels + 31) / 32, batch), dim3(32, 8), 0, st>>>(features, HW, channels, nhwc);
    DT_CHECK_CUDA(cudaGetLastError());
    static bool attr_set = false;
    if (!attr_set) {
        DT_CHECK_CUDA(cudaFuncSetAttribute(roi_align_fast_nchw_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        attr_set = true;
    }
    const int per_sm = (int)(200 * 1024 / (tile_bytes + 2048)) < 8 ? (int)(200 * 1024 / (tile_bytes + 2048)) : 8;
    const int grid = (int)(num_rois < (int64_t)kNumSMs * per_sm ? num_rois : (int64_t)kNumSMs * per_sm);
    roi_align_fast_nchw_out_kernel<<<grid, 256, tile_bytes, st>>>(nhwc, rois, (long long)num_rois, roi_cols, channels, cs, height, width, pooled_height,
                                                                  pooled_width, spatial_scale, out);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// ================================================================================== NMS (single set, boxes.nms contract)
namespace {
struct NmsWs {
    uint32_t *k0, *k1;
    int *v0, *v1;
    float4* sorted;
    unsigned long long* removed;
    int* flags;
};
__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline NmsWs carve_nms_ws(void* ws, int64_t n) {
    NmsWs w;
    uint8_t* p = (uint8_t*)ws;
    const size_t n4 = align_up((size_t)n * 4, 256);
    w.k0 = (uint32_t*)p; p += n4;
    w.k1 = (uint32_t*)p; p += n4;
    w.v0 = (int*)p; p += n4;
    w.v1 = (int*)p; p += n4;
    w.flags = (int*)p; p += n4;
    w.sorted = (float4*)p; p += align_up((size_t)n * 16, 256);
    w.removed = (unsigned long long*)p;
    return w;
}

__global__ void __launch_bounds__(1024) nms_single_kernel(const float* __restrict__ dets, int n, float thresh, NmsWs w,
                                                         long long* __restrict__ keep_out, int* __restrict__ num_keep) {
    __shared__ uint32_t hist[32 * 256];
    __shared__ NmsSmem nsm;
    __shared__ int scan_warp[32];
    __shared__ int running;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        w.k0[i] = float_desc_key(dets[(size_t)i * 5 + 4]);
        w.v0[i] = i;
        w.flags[i] = 0;
    }
    __syncthreads();
    block_radix_sort_asc_u32(w.k0, w.v0, w.k1, w.v1, n, hist);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float* d = dets + (size_t)w.v0[i] * 5;
        w.sorted[i] = make_float4(d[0], d[1], d[2], d[3]);
    }
    __syncthreads();
    block_nms_sorted(w.sorted, n, thresh, 0, w.removed, &nsm);
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (!((w.removed[i >> 6] >> (i & 63)) & 1ull)) w.flags[w.v0[i]] = 1;
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    // ordered compaction of the flags -> ascending original indices
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int f = (i < n) ? w.flags[i] : 0;
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (lane == 0) scan_warp[warp] = __popc(b);
        __syncthreads();
        if (warp == 0) {
            int v = scan_warp[lane], inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
            scan_warp[lane] = inc - v;
            if (lane == 31) nsm.kcount = inc;   // block total (reuse a scratch int)
        }
        __syncthreads();
        if (f) keep_out[running + scan_warp[warp] + __popc(b & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (threadIdx.x == 0) running += nsm.kcount;
        __syncthreads();
    }
    if (threadIdx.x == 0) *num_keep = running;
}


// ---- large sets (n > kNmsSingleCtaMax): sort (1 CTA) -> 64x64 IoU bit-matrix (all SMs) -> chunked scan (1 CTA) -> compaction
static constexpr int kNmsSingleCtaMax = 4096;

__global__ void __launch_bounds__(1024) nms_big_sort_kernel(const float* __restrict__ dets, int n, NmsWs w) {
    __shared__ uint32_t hist[32 * 256];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        w.k0[i] = float_desc_key(dets[(size_t)i * 5 + 4]);
        w.v0[i] = i;
        w.flags[i] = 0;
    }
    __syncthreads();
    block_radix_sort_asc_u32(w.k0, w.v0, w.k1, w.v1, n, hist);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float* d = dets + (size_t)w.v0[i] * 5;
        w.sorted[i] = make_float4(d[0], d[1], d[2], d[3]);
    }
}

// grid (nchunks, nchunks), 64 threads: block (bj, bi) with bj >= bi fills mask[i][bj] for the 64 boxes i of chunk bi:
// bit b set  <=>  sorted box i suppresses sorted box bj*64 + b (only later boxes: index > i)
__global__ void __launch_bounds__(64) nms_big_mask_kernel(const float4* __restrict__ boxes, int n, int nchunks, float thresh,
                                                        unsigned long long* __restrict__ mask) {
    const int bj = blockIdx.x, bi = blockIdx.y;
    if (bj < bi) return;
    __shared__ float4 jb[64];
    __shared__ float ja[64];
    const int j0 = bj * 64, i = bi * 64 + threadIdx.x;
    const int jn = min(64, n - j0);
    if ((int)threadIdx.x < jn) { const float4 b = boxes[j0 + threadIdx.x]; jb[threadIdx.x] = b; ja[threadIdx.x] = box_area_p1(b); }
    __syncthreads();
    if (i >= n) return;
    const float4 me = boxes[i];
    const float ma = box_area_p1(me);
    unsigned long long bits = 0ull;
    for (int b = 0; b < jn; ++b)
        if (j0 + b > i && iou_suppresses(me, ma, jb[b], ja[b], thresh)) bits |= 1ull << b;
    mask[(size_t)i * nchunks + bj] = bits;
}

__global__ void __launch_bounds__(1024) nms_big_scan_kernel(const unsigned long long* __restrict__ mask, int n, int nchunks, NmsWs w) {
    extern __shared__ unsigned long long removed[];     // nchunks words
    __shared__ unsigned long long diag[64];
    __shared__ int kept_list[64];
    __shared__ int kcount;
    for (int i = threadIdx.x; i < nchunks; i += blockDim.x) removed[i] = 0ull;
    __syncthreads();
    for (int c = 0; c < nchunks; ++c) {
        const int cn = min(64, n - c * 64);
        if ((int)threadIdx.x < cn) diag[threadIdx.x] = mask[(size_t)(c * 64 + threadIdx.x) * nchunks + c];
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned long long valid = (cn == 64) ? ~0ull : ((1ull << cn) - 1ull);
            unsigned long long alive = ~removed[c] & valid;
            int kc = 0;
            while (alive) {
                const int b = __ffsll((long long)alive) - 1;
                kept_list[kc++] = c * 64 + b;
                w.flags[w.v0[c * 64 + b]] = 1;        // survivor, in original index space
                alive &= ~diag[b];
                alive &= ~(1ull << b);
            }
            kcount = kc;
        }
        __syncthreads();
        const int kc = kcount;
        for (int wd = c + 1 + threadIdx.x; wd < nchunks; wd += blockDim.x) {
            unsigned long long acc = 0ull;
            for (int k = 0; k < kc; ++k) acc |= mask[(size_t)kept_list[k] * nchunks + wd];
            removed[wd] |= acc;
        }
        __syncthreads();
    }
}

// flags (original index space) -> ascending kept indices
__global__ void __launch_bounds__(1024) nms_compact_kernel(const int* __restrict__ flags, int n, long long* __restrict__ keep_out, int* __restrict__ num_keep) {
    __shared__ int scan_warp[33];
    __shared__ int running;
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int f = (i < n) ? flags[i] : 0;
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (lane == 0) scan_warp[warp] = __popc(b);
        __syncthreads();
        if (warp == 0) {
            int v = scan_warp[lane], inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
            scan_warp[lane] = inc - v;
            if (lane == 31) scan_warp[32] = inc;
        }
        __syncthreads();
        if (f) keep_out[running + scan_warp[warp] + __popc(b & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (threadIdx.x == 0) running += scan_warp[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) *num_keep = running;
}
}  // namespace

extern "C" int64_t dt_nms_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    int64_t base = (int64_t)(5 * align_up((size_t)n * 4, 256) + align_up((size_t)n * 16, 256) + align_up(((size_t)n + 63) / 64 * 8, 256));
    if (n > kNmsSingleCtaMax) base += (int64_t)align_up((size_t)n * (((size_t)n + 63) / 64) * 8, 256);      // the 64-bit suppression matrix
    return base;
}

extern "C" int dt_nms(const float* dets, int n, float thresh, int64_t* keep_out, int* num_keep_out, void* workspace, dt_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n <= 0) {
        DT_CHECK_CUDA(cudaMemsetAsync(num_keep_out, 0, sizeof(int), st));
        return 1;
    }
    NmsWs w = carve_nms_ws(workspace, n);
    if (n <= kNmsSingleCtaMax) {
        nms_single_kernel<<<1, 1024, 0, st>>>(dets, n, thresh, w, (long long*)keep_out, num_keep_out);
        DT_CHECK_CUDA(cudaGetLastError());
        return 1;
    }
    const int nchunks = (n + 63) / 64;
    if ((size_t)nchunks * 8 > 200 * 1024) {
        fprintf(stderr, "[detectorch_b200] dt_nms: at most %d boxes per set\n", 200 * 1024 / 8 * 64);
        return 0;
    }
    unsigned long long* mask = reinterpret_cast<unsigned long long*>(reinterpret_cast<uint8_t*>(w.removed) + align_up((size_t)nchunks * 8, 256));
    nms_big_sort_kernel<<<1, 1024, 0, st>>>(dets, n, w);
    nms_big_mask_kernel<<<dim3(nchunks, nchunks), 64, 0, st>>>(w.sorted, n, nchunks, thresh, mask);
    static bool attr_set = false;
    if (!attr_set) {
        DT_CHECK_CUDA(cudaFuncSetAttribute(nms_big_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_set = true;
    }
    nms_big_scan_kernel<<<1, 1024, (size_t)nchunks * 8, st>>>(mask, n, nchunks, w);
    nms_compact_kernel<<<1, 1024, 0, st>>>(w.flags, n, (long long*)keep_out, num_keep_out);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// ================================================================================== conv / GEMM
namespace {
__global__ void tf32_residual_kernel(const float* __restrict__ w, float* __restrict__ lo, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = w[i];
        lo[i] = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    }
}
}  // namespace

extern "C" int dt_tf32_residual(const float* w, float* w_lo, int64_t n, dt_stream_t stream) {
    if (n <= 0) return 1;
    const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
    tf32_residual_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, w_lo, (long long)n);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

namespace {
__global__ void fp16_split_kernel(const float* __restrict__ w, float mult, __half* __restrict__ hi, __half* __restrict__ lo, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = w[i] * mult;          // mult is a power of two: exact
        const __half h = __float2half_rn(v);
        hi[i] = h;
        lo[i] = __float2half_rn(v - __half2float(h));
    }
}

void fill_plan(const ConvLayer& L, int inst, int num_kb, dt_conv_plan* o) {
    memset(o, 0, sizeof(*o));
    o->instantiation = inst;
    if (inst >= 0) {
        const ConvInstance& r = kConvInstances[inst];
        o->block_n = r.bn; o->nmain = r.nmain; o->two_sm = r.two_sm; o->kind = r.kind; o->ring = r.ring; o->slots = r.slots; o->halo = r.halo;
        o->ws = r.ws;
    }
    const ConvParams& p = L.p;
    o->wbox = p.wbox; o->hbox = p.hbox; o->nbox = p.nbox; o->tiles_w = p.tiles_w; o->tiles_h = p.tiles_h; o->tiles_n = p.tiles_n;
    o->m_pairs = p.m_pairs; o->n_tiles = p.n_tiles; o->grid = (int)L.grid.x; o->num_kb = num_kb; o->ho = p.ho; o->wo = p.wo;
}

// plan (and, launch != 0, run) a built layer
int plan_and_launch(const ConvLayer& L, int num_kb, dt_conv_plan* plan_out, int launch, dt_stream_t stream) {
    const int inst = conv_instance_of(L);
    if (plan_out) fill_plan(L, inst, num_kb, plan_out);
    if (inst < 0) { fprintf(stderr, "[detectorch_b200] conv: no kernel instantiation for this layer\n"); return 0; }
    if (launch) DT_CHECK_CUDA(kConvInstances[inst].launch(L, (cudaStream_t)stream));
    return 1;
}
}  // namespace

extern "C" int dt_conv2d_spec(const dt_conv_desc* d, dt_conv_plan* plan_out, int launch, dt_stream_t stream) {
    if (!d) return 0;
    ConvSpec s;
    memset(&s, 0, sizeof(s));
    s.kind = d->kind == 1 ? KIND_F16X3 : KIND_TF32X3;
    s.x = reinterpret_cast<const float*>(d->x); s.x_lo = d->x_lo; s.N = d->N; s.H = d->H; s.W = d->W; s.Cin = d->Cin;
    s.x_pix_stride = d->x_pix_stride > 0 ? d->x_pix_stride : d->Cin; s.x_mult = d->x_multiplier;
    s.w_hi = d->w_hi; s.w_lo = d->w_lo; s.range_flag = d->range_flag;
    s.Cout = d->Cout; s.kh = d->kh; s.kw = d->kw; s.pad = d->pad; s.stride = d->stride;
    s.scale = d->scale; s.shift = d->shift;
    s.y = reinterpret_cast<float*>(d->y); s.y_lo = d->y_lo; s.y_pix_stride = d->y_pix_stride > 0 ? d->y_pix_stride : d->Cout;
    s.out_h = d->out_h; s.out_w = d->out_w; s.out_step = d->out_step; s.out_y0 = d->out_y0; s.out_x0 = d->out_x0;
    s.residual = d->residual; s.res_pix_stride = d->res_pix_stride > 0 ? d->res_pix_stride : d->Cout;
    s.up_src = d->up_src; s.up_h = d->up_h; s.up_w = d->up_w;
    s.res_mode = d->res_mode; s.relu = d->relu; s.sigmoid_ch = d->sigmoid_ch; s.passes = d->passes;
    s.tap0 = d->tap0; s.ntaps = d->ntaps; s.force_block_n = d->force_block_n; s.precise = d->precise; s.no_merge = d->no_merge;
    ConvLayer L;
    if (!conv_build(s, &L)) return 0;
    const int num_kb = L.p.ntaps * L.p.cin_blocks;
    return plan_and_launch(L, num_kb, plan_out, launch, stream);
}

extern "C" int dt_conv2d_stem(const void* x4, int planes, int B, int Hp, int Wp, int H1, int W1, const void* w_hi, const void* w_lo, int kind,
                              const float* scale, const float* shift, float x_multiplier, int passes, int* range_flag, float* y,
                              dt_conv_plan* plan_out, int launch, dt_stream_t stream) {
    ConvLayer L;
    if (!conv_build_stem(reinterpret_cast<const float*>(x4), B, Hp, Wp, H1, W1, w_hi, w_lo, scale, shift, y, passes, &L,
                         kind == 1 ? KIND_F16X3 : KIND_TF32X3, range_flag, planes != 0, x_multiplier)) {
        fprintf(stderr, "[detectorch_b200] dt_conv2d_stem: the layer could not be built\n");
        return 0;
    }
    return plan_and_launch(L, 7, plan_out, launch, stream);
}

extern "C" int dt_conv_instantiation_count(void) { return kNumConvInstances; }

extern "C" int dt_conv_instantiation_info(int i, int* fields8) {
    if (i < 0 || i >= kNumConvInstances || !fields8) return 0;
    const ConvInstance& r = kConvInstances[i];
    const int f[8] = {r.bn, r.nmain, r.two_sm, r.kind, r.ring, r.slots, r.halo, r.ws};
    memcpy(fields8, f, sizeof(f));
    return 1;
}

namespace {
int conv2d_nhwc_impl(int kind, const float* x, int N, int H, int W, int Cin, int x_pix_stride, const void* w, const void* w_lo, int Cout, int kh,
                     int kw, int pad, int stride, const float* scale, const float* shift, const float* residual, int res_mode,
                     const float* up_src, int up_h, int up_w, int relu, int sigmoid_ch, int passes, int force_block_n, int* range_flag,
                     float* y, int y_pix_stride, dt_stream_t stream) {
    dt_conv_desc d;
    memset(&d, 0, sizeof(d));
    d.kind = kind == KIND_F16X3 ? 1 : 0;
    d.x = x; d.N = N; d.H = H; d.W = W; d.Cin = Cin; d.x_pix_stride = x_pix_stride;
    d.w_hi = w; d.w_lo = w_lo; d.range_flag = range_flag;
    d.Cout = Cout; d.kh = kh; d.kw = kw; d.pad = pad; d.stride = stride;
    d.scale = scale; d.shift = shift; d.y = y; d.y_pix_stride = y_pix_stride;
    d.residual = residual; d.res_pix_stride = Cout; d.up_src = up_src; d.up_h = up_h; d.up_w = up_w;
    d.res_mode = res_mode; d.relu = relu; d.sigmoid_ch = sigmoid_ch; d.passes = passes; d.force_block_n = force_block_n;
    d.precise = force_block_n < 0;
    if (force_block_n < 0) d.force_block_n = 128;        // -1: the precise 128-wide tile (3 rotating accumulators)
    return dt_conv2d_spec(&d, nullptr, 1, stream);
}
}  // namespace

extern "C" int dt_fp16_split(const float* w, int64_t n, float multiplier, void* w_hi16, void* w_lo16, dt_stream_t stream) {
    if (n <= 0) return 1;
    const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
    fp16_split_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, multiplier, reinterpret_cast<__half*>(w_hi16), reinterpret_cast<__half*>(w_lo16),
                                                             (long long)n);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

extern "C" int dt_conv2d_nhwc(const float* x, int N, int H, int W, int Cin, int x_pix_stride, const float* w, const float* w_lo, int Cout,
                              int kh, int kw, int pad, int stride, const float* scale, const float* shift, const float* residual,
                              int res_mode, const float* up_src, int up_h, int up_w, int relu, int sigmoid_ch, int passes,
                              int force_block_n, float* y, int y_pix_stride, dt_stream_t stream) {
    return conv2d_nhwc_impl(KIND_TF32X3, x, N, H, W, Cin, x_pix_stride, w, w_lo, Cout, kh, kw, pad, stride, scale, shift, residual, res_mode,
                            up_src, up_h, up_w, relu, sigmoid_ch, passes, force_block_n, nullptr, y, y_pix_stride, stream);
}

extern "C" int dt_conv2d_nhwc_f16x3(const float* x, int N, int H, int W, int Cin, int x_pix_stride, const void* w_hi16, const void* w_lo16,
                                    int Cout, int kh, int kw, int pad, int stride, const float* scale, const float* shift,
                                    const float* residual, int res_mode, const float* up_src, int up_h, int up_w, int relu, int sigmoid_ch,
                                    int passes, int force_block_n, int* range_flag, float* y, int y_pix_stride, dt_stream_t stream) {
    return conv2d_nhwc_impl(KIND_F16X3, x, N, H, W, Cin, x_pix_stride, w_hi16, w_lo16, Cout, kh, kw, pad, stride, scale, shift, residual,
                            res_mode, up_src, up_h, up_w, relu, sigmoid_ch, passes, force_block_n, range_flag, y, y_pix_stride, stream);
}

// ================================================================================== mask paste + COCO RLE (segm_results)
namespace {
constexpr int kSegmCharsPerRun = 4;     // staging bytes per run (maskApi's worst case is 7; typical masks need 1-2)
size_t segm_smem_bytes(int M, int im_h, int im_w) {
    const int S = M + 2;
    return (size_t)((S * S + 3) & ~3) * 4 + (size_t)im_h * sizeof(SegmRowCoef) + (size_t)(im_w + 2) * 4 + 40 * 4;
}
}  // namespace

extern "C" int64_t dt_segm_workspace_bytes(int max_dets, int runs_cap) {
    return (int64_t)max_dets * runs_cap * 4 + (int64_t)max_dets * runs_cap * kSegmCharsPerRun + (int64_t)max_dets * 4 + 256;
}

extern "C" int64_t dt_segm_strings_bytes(int max_dets, int runs_cap) { return (int64_t)max_dets * runs_cap * kSegmCharsPerRun; }

extern "C" int dt_segm_rle(const float* masks, const int* classes, int num_mask_classes, int mask_size, const float* ref_boxes,
                           const int* expanded_boxes, const int* num_dets_dev, int max_dets, int im_h, int im_w, float thresh_binarize,
                           uint32_t* counts, int* num_counts, int runs_cap, uint8_t* strings, int64_t* str_offsets, int* overflow,
                           void* workspace, dt_stream_t stream) {
    if (max_dets <= 0) return 1;
    if (!masks || (!ref_boxes && !expanded_boxes) || !counts || !num_counts || !strings || !str_offsets || !overflow || !workspace) {
        fprintf(stderr, "dt_segm_rle: null argument\n");
        return 0;
    }
    if (mask_size < 1 || mask_size > 126 || im_h < 1 || im_w < 1 || (int64_t)im_h * im_w >= (1ll << 32) || runs_cap < 2) {
        fprintf(stderr, "dt_segm_rle: unsupported size (mask %d, image %dx%d, runs_cap %d)\n", mask_size, im_h, im_w, runs_cap);
        return 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    uint32_t* positions = reinterpret_cast<uint32_t*>(ws);
    uint8_t* staging = ws + (size_t)max_dets * runs_cap * 4;
    int* str_len = reinterpret_cast<int*>(staging + (((size_t)max_dets * runs_cap * kSegmCharsPerRun + 15) / 16 * 16));
    const size_t smem = segm_smem_bytes(mask_size, im_h, im_w);
    if (smem > 200 * 1024) { fprintf(stderr, "dt_segm_rle: image too large for the row/column tables (%zu B)\n", smem); return 0; }
    static size_t smem_set = 48 * 1024;
    if (smem > smem_set) {
        DT_CHECK_CUDA(cudaFuncSetAttribute(segm_rle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        smem_set = 200 * 1024;
    }
    DT_CHECK_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int), st));
    segm_rle_kernel<<<max_dets, 256, smem, st>>>(masks, classes, classes ? num_mask_classes : 1, mask_size, ref_boxes, expanded_boxes,
                                                 num_dets_dev, im_h, im_w, thresh_binarize, positions, counts, num_counts, runs_cap,
                                                 staging, str_len, runs_cap * kSegmCharsPerRun, overflow);
    DT_CHECK_CUDA(cudaGetLastError());
    segm_compact_kernel<<<max_dets, 256, 0, st>>>(staging, str_len, max_dets, runs_cap * kSegmCharsPerRun, strings,
                                                  reinterpret_cast<long long*>(str_offsets));
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

extern "C" int dt_segm_paste(const float* masks, const int* classes, int num_mask_classes, int mask_size, const float* ref_boxes,
                             const int* expanded_boxes, const int* num_dets_dev, int max_dets, int im_h, int im_w, float thresh_binarize,
                             uint8_t* out, dt_stream_t stream) {
    if (max_dets <= 0) return 1;
    if (!masks || (!ref_boxes && !expanded_boxes) || !out || mask_size < 1 || mask_size > 126) {
        fprintf(stderr, "dt_segm_paste: bad argument\n");
        return 0;
    }
    const int S = mask_size + 2;
    segm_paste_kernel<<<max_dets, 256, (size_t)S * S * 4, (cudaStream_t)stream>>>(masks, classes, classes ? num_mask_classes : 1, mask_size,
                                                                                  ref_boxes, expanded_boxes, num_dets_dev, im_h, im_w,
                                                                                  thresh_binarize, out);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}

// ================================================================================== image pre-processing (prep_im_for_blob + im_list_to_blob)
extern "C" int dt_prep_image(const uint8_t* image_hwc, int height, int width, const double* pixel_means, double im_scale, int out_height,
                             int out_width, float* blob_chw, int blob_height, int blob_width, dt_stream_t stream) {
    if (!image_hwc || !pixel_means || !blob_chw || height < 1 || width < 1 || !(im_scale > 0.0) || out_height < 1 || out_width < 1 ||
        blob_height < out_height || blob_width < out_width) {
        fprintf(stderr, "dt_prep_image: bad argument\n");
        return 0;
    }
    const double inv_scale = 1.0 / im_scale;
    // cv::resize: INTER_LINEAR becomes the area-fast kernel when both scale factors are exactly 2
    const int area2 = (fabs(inv_scale - 2.0) < 2.220446049250313e-16 && out_height * 2 <= height && out_width * 2 <= width) ? 1 : 0;
    dim3 grid((blob_width + 255) / 256, blob_height);
    prep_image_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(image_hwc, height, width, pixel_means[0], pixel_means[1], pixel_means[2], inv_scale,
                                                             out_height, out_width, area2, blob_chw, blob_height, blob_width);
    DT_CHECK_CUDA(cudaGetLastError());
    return 1;
}
