/*
 * detectorch_b200 -- C ABI of the B200-native two-stage-detector inference hot path.
 *
 * Plain pointers and sizes only (no torch types).  Every pointer is a DEVICE pointer unless
 * stated otherwise; every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 * never synchronises, and returns 1 on success / 0 on failure (the reference's launcher
 * convention, lib/cppcuda_cffi/src/cuda/roi_align_forward_cuda_kernel.cu:161-199), printing the
 * reason to stderr.  Layouts are fp32 throughout.
 *
 * Each entry point names the reference interface it replaces (paths relative to the reference
 * repository root).  INTEGRATION.md shows the reference-side binding for each.
 */
#ifndef DETECTORCH_B200_H
#define DETECTORCH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dt_stream_t; /* cudaStream_t */

/* ---------------------------------------------------------------------------------------------
 * RoIAlign forward.
 * Replaces: lib/cppcuda_cffi/src/cuda/roi_align_forward_cuda_kernel.h:7-19 (exact signature kept:
 * this symbol is what lib/cppcuda_cffi/src/roi_align_forward_cuda.c:35-47 calls), and through it
 * lib/cppcuda/roi_align_cuda.h:4-11 / lib/model/roi_align.py:32-89.
 * bottom_data NCHW [B,C,H,W]; bottom_rois [R,5] (batch,x1,y1,x2,y2); top_data [R,C,ph,pw];
 * outputElements = R*C*ph*pw (int, as in the reference: < 2^31).
 */
int launch_roi_align_forward_cuda(const int outputElements, const float* bottom_data, const float* bottom_rois,
                                  const float spatial_scale, const int channels, const int height, const int width,
                                  const int pooled_height, const int pooled_width, const int sampling_ratio, float* top_data,
                                  dt_stream_t stream);

/* RoIAlign backward (gradient w.r.t. the features), the training-side caller of the same boundary.
 * Replaces: lib/cppcuda_cffi/src/cuda/roi_align_backward_cuda_kernel.h:7-21 (exact signature kept; called by
 * lib/cppcuda_cffi/src/roi_align_backward_cuda.c and lib/model/roi_align.py:91-147).  top_diff [R,C,ph,pw];
 * bottom_diff [B,C,H,W] is ACCUMULATED into (the caller zeroes it, roi_align.py:117); atomic fp32 scatter like the reference,
 * so the last bits depend on the summation order exactly as they do there. */
int launch_roi_align_backward_cuda(const int nthreads, const float* top_diff, const int num_rois, const float spatial_scale,
                                   const int channels, const int height, const int width, const int pooled_height,
                                   const int pooled_width, const int sampling_ratio, float* bottom_diff, const float* bottom_rois,
                                   int roi_cols, dt_stream_t stream);

/* Deterministic (atomics-free) backward: the contributions to every feature-map cell are summed in exactly the order of the reference's
 * single-threaded CPU loop (lib/cppcuda/roi_align_backward_cpu.cpp:79-186) => bit-identical to it and bit-reproducible run to run
 * (the atomic scatter above is neither).  Two calls: _plan writes the number of (sample, corner) contributions of the RoI set to *total_dev
 * (device int64; the grid is adaptive when sampling_ratio == 0, so only the device knows it); the caller reads it, allocates
 * dt_roi_align_backward_det_workspace_bytes(num_rois, total) bytes and calls _deterministic.  bottom_diff is accumulated into. */
int64_t dt_roi_align_backward_det_workspace_bytes(int64_t num_rois, int64_t total_contributions);
int dt_roi_align_backward_plan(const float* rois, int64_t num_rois, int roi_cols, float spatial_scale, int pooled_height, int pooled_width,
                               int sampling_ratio, void* scratch, int64_t* total_dev, dt_stream_t stream);
int dt_roi_align_backward_deterministic(const float* top_diff, const float* rois, int64_t num_rois, int roi_cols, int batch, int channels,
                                        int height, int width, int pooled_height, int pooled_width, float spatial_scale, int sampling_ratio,
                                        int64_t total_contributions, float* bottom_diff, void* workspace, dt_stream_t stream);

/* 64-bit-safe variant (R*C*ph*pw may exceed 2^31, e.g. 100k RoIs x 256 ch x 14 x 14); roi_cols is 4 or 5
 * like the reference CPU loop (lib/cppcuda_cffi/src/cpp/roi_align_cpu_loop.h:5-17). */
int dt_roi_align_forward_nchw(const float* features, const float* rois, int64_t num_rois, int roi_cols, int channels, int height,
                              int width, int pooled_height, int pooled_width, float spatial_scale, int sampling_ratio, float* out,
                              dt_stream_t stream);

/* Fast variant for sampling_ratio == 2 (the FPN configurations and the RoIAlign microbench): separable bilinear weights with
 * merged duplicate taps, fused multiply-adds, output tile assembled in shared memory and written by one bulk async copy per
 * RoI.  Same contract as dt_roi_align_forward_nchw (any other configuration is forwarded to it); results agree with the
 * exact kernel to fp32 re-association (~1e-7 relative).  Maps small enough for an 8-channel slab of the whole map to live in
 * shared memory (H*W <= ~3600 cells, 7x7 or 14x14 bins) take the shared-memory-resident variant: the gathers never leave
 * the SM.  workspace: dt_roi_align_fast_workspace_bytes() (an NHWC copy of the feature map + the per-RoI tap tables). */
int64_t dt_roi_align_fast_workspace_bytes(int batch, int channels, int height, int width, int64_t num_rois, int pooled_height,
                                          int pooled_width);
int dt_roi_align_forward_nchw_fast(const float* features, int batch, const float* rois, int64_t num_rois, int roi_cols, int channels, int height,
                                   int width, int pooled_height, int pooled_width, float spatial_scale, int sampling_ratio, float* out,
                                   void* workspace, dt_stream_t stream);

/* Multi-level NHWC variant used inside the fused detector (replaces the 4 per-level RoIAlign calls + cat +
 * index-restore of lib/model/detector.py:259-270 and :100-106).  feats[l] is an NHWC map [B,H[l],W[l],C];
 * rois [max_rois,5]; level[max_rois] (index into feats, NULL = all level 0); num_rois_dev: optional device int
 * (rows >= *num_rois_dev are written as zeros); out [max_rois, ph, pw, C]. */
int dt_roi_align_forward_nhwc(const float* const* feats_host_array, const int* heights, const int* widths, const float* scales,
                              int num_levels, const float* rois, const int* level, const int* num_rois_dev, int max_rois,
                              int channels, int pooled_height, int pooled_width, int sampling_ratio, float* out, dt_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Greedy hard NMS with the reference's exact fp32 semantics ("+1" widths, ovr >= thresh).
 * Replaces: lib/utils/boxes.py:332-336 -> lib/utils_cython/cython_nms.pyx:37-87.
 * dets [n,5] (x1,y1,x2,y2,score).  keep_out [n] int64 receives the ASCENDING ORIGINAL indices of the
 * survivors, *num_keep_out (device int) their count.  workspace: dt_nms_workspace_bytes(n) bytes.
 */
int64_t dt_nms_workspace_bytes(int64_t n);
int dt_nms(const float* dets, int n, float thresh, int64_t* keep_out, int* num_keep_out, void* workspace, dt_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Mask paste + COCO run-length encoding (the step right after the path, SURVEY.md 8f rank 1).
 * Replaces: lib/utils/result_utils.py:170-228 (segm_results): per detection zero-pad the MxM mask by one cell, expand the
 * reference box by (M+2)/M (lib/utils/boxes.py:245-261), truncate to int32, cv2.resize(float32, INTER_LINEAR) to the box,
 * threshold, paste into an im_h x im_w image, pycocotools rleEncode + rleToString -- without ever materialising the image.
 *   masks          [max_dets, num_mask_classes, M, M] with classes[d] selecting the plane, or [max_dets, M, M] (classes NULL)
 *   ref_boxes      [max_dets,4] fp32 image-space boxes (expanded on the device), or expanded_boxes [max_dets,4] int32
 *                  (already expanded and truncated by the caller); one of the two must be non-NULL
 *   num_dets_dev   optional device int: detections >= *num_dets_dev produce empty results
 *   counts         [max_dets, runs_cap] uint32 run lengths (column-major, zeros run first), num_counts[max_dets]
 *   strings        dt_segm_strings_bytes() bytes: the compressed RLE strings back to back; str_offsets[max_dets+1]
 *   overflow       device int: 0, or the number of runs a detection needed when runs_cap (or its string staging) was too small
 * dt_segm_paste writes the pasted binary masks themselves, uint8 [max_dets, im_h, im_w].
 */
int64_t dt_segm_workspace_bytes(int max_dets, int runs_cap);
int64_t dt_segm_strings_bytes(int max_dets, int runs_cap);
int dt_segm_rle(const float* masks, const int* classes, int num_mask_classes, int mask_size, const float* ref_boxes,
                const int* expanded_boxes, const int* num_dets_dev, int max_dets, int im_h, int im_w, float thresh_binarize,
                uint32_t* counts, int* num_counts, int runs_cap, uint8_t* strings, int64_t* str_offsets, int* overflow, void* workspace,
                dt_stream_t stream);
int dt_segm_paste(const float* masks, const int* classes, int num_mask_classes, int mask_size, const float* ref_boxes,
                  const int* expanded_boxes, const int* num_dets_dev, int max_dets, int im_h, int im_w, float thresh_binarize,
                  uint8_t* out, dt_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Image pre-processing (the step right before the path, SURVEY.md 8f rank 3).
 * Replaces: lib/utils/blob.py:57-87 prep_im_for_blob (float32, minus pixel_means, cv2.resize(fx=fy=im_scale, INTER_LINEAR)) fused
 * with blob.py:27-55 im_list_to_blob (zero-pad to a multiple of the coarsest FPN stride, HWC -> CHW).
 *   image_hwc    device uint8 [height, width, 3] (BGR, as cv2.imread returns it)
 *   pixel_means  HOST double[3]; im_scale: the factor prep_im_for_blob computes (target_size / min side, capped by max_size)
 *   out_height/out_width = cvRound(height * im_scale), cvRound(width * im_scale)  (the size cv2.resize produces)
 *   blob_chw     device fp32 [3, blob_height, blob_width], zero outside the resized image
 */
int dt_prep_image(const uint8_t* image_hwc, int height, int width, const double* pixel_means, double im_scale, int out_height, int out_width,
                  float* blob_chw, int blob_height, int blob_width, dt_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Convolution / GEMM on tcgen05 tensor cores (3xTF32, fp32-accurate), NHWC activations.
 * Replaces the torch.nn.Conv2d / Linear / ConvTranspose2d calls of lib/model/detector.py
 * (:17-27 FPN, :58-59 FC6/FC7, :71-74 mask convs, :89-90 deconv + mask logits, :119-121 RPN, :170-183 trunk).
 *   x        [N,H,W,Cin]   (Cin % 32 == 0), x_pix_stride floats between pixels
 *   w        [Cout][kh][kw][Cin] fp32, w_lo = w - trunc_tf32(w) (dt_tf32_residual)
 *   y        [N,Ho,Wo,Cout] (Cout % 4 == 0), y = act( conv(x,w)*scale[c] + shift[c] (+ residual) )
 *   res_mode 0 none | 1 residual [N,Ho,Wo,Cout] | 2 nearest-2x-upsampled up_src [N,up_h,up_w,Cout]
 *   relu     0/1 ; sigmoid_ch: channels [0,sigmoid_ch) get a sigmoid ; passes 3 (3xTF32) or 1 (TF32)
 *   force_block_n 0 = auto | 64 | 128 | 256 | -1 = 128 with 3 rotating accumulators (shortest truncating-accumulate chains)
 * dt_conv2d_nhwc_f16x3 is the same product on the kind::f16 pipe (twice the tf32 issue rate): w_hi16 / w_lo16 are the fp16 halves of
 * w * multiplier from dt_fp16_split (multiplier a power of two that keeps the low half a normal fp16 number; the caller folds
 * 1/multiplier into `scale`); the fp32 activations are split in shared memory.  *range_flag (device int, may be NULL) is set
 * to 1 if an activation does not fit fp16 (|x| >= 65504); the result is then not meaningful and the tf32 entry must be used.
 */
int dt_tf32_residual(const float* w, float* w_lo, int64_t n, dt_stream_t stream);
int dt_fp16_split(const float* w, int64_t n, float multiplier, void* w_hi16, void* w_lo16, dt_stream_t stream);
int dt_conv2d_nhwc_f16x3(const float* x, int N, int H, int W, int Cin, int x_pix_stride, const void* w_hi16, const void* w_lo16, int Cout,
                         int kh, int kw, int pad, int stride, const float* scale, const float* shift, const float* residual, int res_mode,
                         const float* up_src, int up_h, int up_w, int relu, int sigmoid_ch, int passes, int force_block_n, int* range_flag,
                         float* y, int y_pix_stride, dt_stream_t stream);
int dt_conv2d_nhwc(const float* x, int N, int H, int W, int Cin, int x_pix_stride, const float* w, const float* w_lo, int Cout,
                   int kh, int kw, int pad, int stride, const float* scale, const float* shift, const float* residual,
                   int res_mode, const float* up_src, int up_h, int up_w, int relu, int sigmoid_ch, int passes, int force_block_n,
                   float* y, int y_pix_stride, dt_stream_t stream);

/* Any single conv layer the engine can run, with every option of its layers: fp16 hi/lo plane input (x_lo) and output (y_lo, f16 kind,
 * dense layout, Cout % 32 == 0), the filter-tap range of a K-split (taps [tap0, tap0 + ntaps), ntaps 0 = all), the scattered output of a
 * transposed conv (out_step != 0: output pixel (n,h,w) is written at pixel (n, h*out_step + out_y0, w*out_step + out_x0) of an
 * [N,out_h,out_w] map), channel-slice input / wider output buffers (pixel strides; 0 = dense), the precise / unmerged accumulator forms.
 * kind 0 = 3xTF32 (w_hi fp32, w_lo = dt_tf32_residual), 1 = the kind::f16 product (w_hi / w_lo from dt_fp16_split).  x_multiplier
 * (f16 kind, fp32 input; 0 or 1 = none) is a power of two applied to x before the fp16 split: it keeps the low halves of small
 * activations normal fp16 numbers; the caller folds 1 / x_multiplier into scale like the weight multiplier.
 * plan_out (host, may be NULL) receives the tile geometry and the kernel instantiation the layer runs; launch 0 only plans. */
typedef struct dt_conv_desc {
    int kind;
    const void* x; const void* x_lo;
    int N, H, W, Cin, x_pix_stride;
    float x_multiplier;
    const void* w_hi; const void* w_lo;
    int Cout, kh, kw, pad, stride;
    const float* scale; const float* shift;
    void* y; void* y_lo; int y_pix_stride;
    int out_h, out_w, out_step, out_y0, out_x0;
    const float* residual; int res_pix_stride;
    const float* up_src; int up_h, up_w;
    int res_mode, relu, sigmoid_ch, passes;
    int tap0, ntaps;
    int force_block_n, precise, no_merge;
    int* range_flag;
} dt_conv_desc;

typedef struct dt_conv_plan {
    int instantiation;                                 /* row of the instantiation table below (-1: none) */
    int block_n, nmain, two_sm, kind, ring, slots, halo, ws;   /* that row; nmain 0 = one merged accumulator, 1, or 3 rotating */
    int wbox, hbox, nbox, tiles_w, tiles_h, tiles_n;   /* output tile box and tile counts */
    int m_pairs, n_tiles, grid;                        /* work items = m_pairs * n_tiles over `grid` CTAs (2 per cluster) */
    int num_kb;                                        /* 32-element k-blocks per tile */
    int ho, wo;
} dt_conv_plan;

int dt_conv2d_spec(const dt_conv_desc* desc, dt_conv_plan* plan_out, int launch, dt_stream_t stream);
/* The 7x7 stride-2 stem (3 input channels) over a zero-bordered NHWC4 image x4 [B,Hp,Wp,4] (3-pixel border, channel 3 = 0,
 * Hp >= 2*H1 + 5, Wp >= 2*W1 + 6), or (planes != 0, f16 kind, Wp even) its fp16 hi and lo planes back to back; weights [64][7 (ky)][32]
 * (element kx*4 + c, zero for kx = 7 or c = 3); y [B,H1,W1,64], ReLU applied. */
int dt_conv2d_stem(const void* x4, int planes, int B, int Hp, int Wp, int H1, int W1, const void* w_hi, const void* w_lo, int kind,
                   const float* scale, const float* shift, float x_multiplier, int passes, int* range_flag, float* y, dt_conv_plan* plan_out,
                   int launch, dt_stream_t stream);
/* the kernel instantiation table: fields8 = {block_n, nmain, two_sm, kind, ring, slots, halo, ws} of row i */
int dt_conv_instantiation_count(void);
int dt_conv_instantiation_info(int i, int* fields8);

/* ---------------------------------------------------------------------------------------------
 * Fused Mask R-CNN (ResNet-50/101 + FPN) inference engine: the whole of
 *   lib/model/detector.py:233-286 (detector.forward), lib/utils/result_utils.py:76-168
 *   (postprocess_output) and lib/model/detector.py:99-112 (mask_head.forward)
 * as one static, sync-free program of sm_100a kernels.  The caller owns two flat device buffers
 * (weights, workspace); named intermediate / output tensors are exposed as (offset, shape) into the
 * workspace so the host language wraps them without copies.
 */
typedef struct dt_engine_config {
    int arch_blocks[4];          /* bottlenecks per stage: {3,4,6,3} = ResNet-50, {3,4,23,3} = ResNet-101 */
    int batch, height, width;    /* network input [batch,3,height,width], height/width multiples of 32 */
    int pre_nms_top_n;           /* per-level RPN top-k before NMS (1000, detector.py:206)  */
    int post_nms_top_n;          /* per-level and collected RoI count (1000, detector.py:207) */
    float rpn_nms_thresh;        /* 0.7 (generate_proposals.py:28) */
    float rpn_min_size;          /* 0   (generate_proposals.py:17) */
    int num_classes;             /* 81 */
    float score_thresh;          /* 0.05 (result_utils.py:98) */
    float det_nms_thresh;        /* 0.5  (result_utils.py:99) */
    int max_dets;                /* 100  (result_utils.py:106) */
    int det_cap;                 /* padded detections per image in the fused outputs (>= max_dets) */
    int use_mask;                /* build the '1up4convs' mask head */
    int output_prob;             /* softmax / sigmoid on the outputs (detector.py:147) */
    int emit_full_masks;         /* also materialise masks_full [D,num_classes,28,28] (the public layout) */
    int passes;                  /* 3 = 3xTF32 (fp32-accurate, default), 1 = single-pass TF32 */
    int precise_mask;            /* mask-head 3x3 convs (K = 2304): 1 = K-split in two launches with an fp32 RN add between them (halves the
                                    truncating-accumulate error; default), 2 = 128-wide tiles with 3 rotating accumulators, 0 = plain */
    int stem_im2col;             /* 1 = force the im2col + GEMM stem instead of the fused TMA-window stem (debug) */
    int exact_roialign;          /* 1 = RoIAlign in the reference's exact fp32 operation order (bit-identical to its CPU loop);
                                    0 = separable / FMA fast path (fp32 re-association only, ~1e-7 relative) */
    int model_type;              /* 0 = R-50/101-FPN + RPN (+ '1up4convs' mask head); 1 = R-50/101-C4 (res5 head, 'upshare' mask head) */
    int use_rpn;                 /* 1 = Faster/Mask R-CNN (RPN head + proposal generation on the device), 0 = Fast R-CNN with pre-computed
                                    proposals (eval_fast.ipynb / eval_fast_FPN.ipynb): the caller fills `rois` (+ `roi_levels` for FPN), `roi_counts` */
    int conv_kind;               /* 0 = three-term product on the kind::f16 pipe (fp16 hi/lo halves, default: twice the tf32 issue rate; an
                                    activation >= 65504 raises the int32 buffer "range_flag", which every run that starts at the first stage clears
                                    before it launches anything), 1 = 3xTF32 (no range limit) */
    int plane_handover;          /* kind::f16 only: 1 = conv1 of every bottleneck writes its output as two fp16 planes (hi, lo) that conv2 (3x3)
                                    loads straight into its operand tiles (no per-tap re-conversion); 2 = conv2 -> conv3 as well; 3 = also the
                                    packed image -> stem (FPN engine); 4 = also the pooled map -> first bottleneck (no net gain measured:
                                    opt-in); 0 = fp32 hand-over */
} dt_engine_config;

typedef void* dt_engine_t;

dt_engine_t dt_engine_create(const dt_engine_config* cfg);
void dt_engine_destroy(dt_engine_t e);
int64_t dt_engine_weight_bytes(dt_engine_t e);
int64_t dt_engine_workspace_bytes(dt_engine_t e);
/* attach caller-owned device memory and build the launch program (TMA descriptors) */
int dt_engine_bind(dt_engine_t e, void* weights, void* workspace, dt_stream_t stream);
/* same, on a weight buffer that another engine with the same model configuration (all of dt_engine_config but batch/height/width)
 * has already loaded and finalised: packed weights are shape-independent, so engines for different image sizes share one copy */
int dt_engine_attach(dt_engine_t e, void* loaded_weights, void* workspace, dt_stream_t stream);
/* load one parameter by its reference state_dict name (torch layout, e.g. conv [Cout,Cin,kh,kw]); BN gains are
 * folded as g/sqrt(1+1e-5) (detector.py:231,301).  returns 1 loaded, 2 ignored (not on the hot path), 0 error */
int dt_engine_load_param(dt_engine_t e, const char* name, const float* src_dev, int64_t numel, dt_stream_t stream);
int dt_engine_finalize_weights(dt_engine_t e, dt_stream_t stream);
/* named buffer -> byte offset into the workspace, shape (<=5 dims), dtype (0 f32, 1 i32, 2 u8) */
int dt_engine_buffer(dt_engine_t e, const char* name, int64_t* byte_offset, int* ndim, int* dims5, int* dtype);
int dt_engine_num_stages(void);
/* the hot-path parameter table: reference state_dict names and element counts */
int dt_engine_param_count(dt_engine_t e);
int dt_engine_param_info(dt_engine_t e, int i, char* name_out, int name_cap, int64_t* numel);
/* original (un-scaled) image size used by the detection clip (result_utils.py:86); 0,0 = network size / scaling_factor */
int dt_engine_set_original_size(dt_engine_t e, float orig_h, float orig_w);
/* stages: 0 trunk, 1 FPN, 2 RPN convs, 3 proposals, 4 collect, 5 RoIAlign(box), 6 box head, 7 detect (decode+NMS+limit),
 *         8 mask RoIs, 9 RoIAlign(mask), 10 mask convs, 11 mask output */
int dt_engine_run(dt_engine_t e, const float* image_nchw, float scaling_factor, int first_stage, int last_stage, dt_stream_t stream);
int dt_engine_count_launches(dt_engine_t e, int first_stage, int last_stage);
/* measurement aid: one pass with a CUDA-event pair around every launch on `stream` (synchronises at the end);
 * per-op milliseconds, algorithmic FLOPs (0 for non-GEMM ops), stage id, BLOCK_N (0 for non-GEMM ops) */
int dt_engine_profile(dt_engine_t e, const float* image_nchw, float scaling_factor, int first_stage, int last_stage, dt_stream_t stream,
                      float* ms_out, double* flops_out, int* stage_out, int* block_n_out, int cap);

/* library / build info */
const char* dt_version(void);

#ifdef __cplusplus
}
#endif
#endif
