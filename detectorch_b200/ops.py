"""Torch-tensor front-ends of the C-ABI operators.  Torch is only plumbing here (device memory,
current stream); all compute happens in detectorch_b200/csrc.  Every function requires CUDA
tensors -- there is no CPU path."""
import ctypes
import math

import torch

from . import _lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise TypeError("detectorch_b200 operators run on CUDA tensors only (no CPU fallback)")


def roi_align_forward_nchw(features, rois, pooled_height, pooled_width, spatial_scale, sampling_ratio, out=None):
    """features [B,C,H,W] fp32 contiguous, rois [R,4|5] -> [R,C,ph,pw].  Mirrors
    roialign.roi_align_forward_cuda of the reference (lib/model/roi_align.py:46-63)."""
    _need_cuda(features, rois)
    if features.dim() != 4 or rois.dim() != 2 or rois.size(1) not in (4, 5):
        raise RuntimeError("roi_align: features must be [B,C,H,W] and rois [R,4|5]")
    if not (features.is_contiguous() and rois.is_contiguous()):
        raise RuntimeError("roi_align: features and rois must be contiguous")   # reference AT_CHECK, roi_align_forward_cuda.cu:189
    if features.dtype != torch.float32 or rois.dtype != torch.float32:
        raise RuntimeError("roi_align: fp32 only")
    R, C = rois.size(0), features.size(1)
    if out is None:
        out = torch.empty((R, C, pooled_height, pooled_width), device=features.device, dtype=torch.float32)
    ok = _lib.lib().dt_roi_align_forward_nchw(_p(features), _p(rois), R, rois.size(1), C, features.size(2), features.size(3),
                                              int(pooled_height), int(pooled_width), float(spatial_scale), int(sampling_ratio),
                                              _p(out), _stream())
    _lib.check(ok, "dt_roi_align_forward_nchw")
    return out


def roi_align_backward_nchw(rois, grad_output, features_size, pooled_height, pooled_width, spatial_scale, sampling_ratio):
    """grad_output [R,C,ph,pw], rois [R,4|5] -> gradient w.r.t. the NCHW features [B,C,H,W] (lib/model/roi_align.py:91-147)."""
    _need_cuda(rois, grad_output)
    B, C, H, W = [int(v) for v in features_size]
    R = rois.size(0)
    if grad_output.dim() != 4 or grad_output.size(0) != R or grad_output.size(1) != C:
        raise RuntimeError("roi_align backward: grad_output must be [R,C,ph,pw]")
    grad_input = torch.zeros((B, C, H, W), device=grad_output.device, dtype=torch.float32)
    ok = _lib.lib().launch_roi_align_backward_cuda(int(grad_output.numel() & 0x7fffffff), _p(grad_output), R, float(spatial_scale), C, H, W,
                                                   int(pooled_height), int(pooled_width), int(sampling_ratio), _p(grad_input), _p(rois),
                                                   rois.size(1), _stream())
    _lib.check(ok, "launch_roi_align_backward_cuda")
    return grad_input


def roi_align_backward_nchw_deterministic(rois, grad_output, features_size, pooled_height, pooled_width, spatial_scale, sampling_ratio, grad_input=None):
    """Same contract as roi_align_backward_nchw, without atomics: every feature-map cell sums its contributions in the order of the
    reference's single-threaded CPU backward (lib/cppcuda/roi_align_backward_cpu.cpp:79-186), so the result is bit-identical to that loop
    and bit-reproducible run to run.  One host read (the contribution count: the sampling grid is adaptive when sampling_ratio == 0)."""
    _need_cuda(rois, grad_output)
    B, C, H, W = [int(v) for v in features_size]
    R = rois.size(0)
    if grad_output.dim() != 4 or grad_output.size(0) != R or grad_output.size(1) != C:
        raise RuntimeError("roi_align backward: grad_output must be [R,C,ph,pw]")
    rois, grad_output = rois.contiguous().float(), grad_output.contiguous().float()
    if grad_input is None:
        grad_input = torch.zeros((B, C, H, W), device=grad_output.device, dtype=torch.float32)
    if R == 0:
        return grad_input
    L = _lib.lib()
    dev = grad_output.device
    with torch.cuda.device(dev):
        scratch = torch.empty((L.dt_roi_align_backward_det_workspace_bytes(R, 0),), dtype=torch.uint8, device=dev)
        total = torch.zeros((1,), dtype=torch.int64, device=dev)
        _lib.check(L.dt_roi_align_backward_plan(_p(rois), R, rois.size(1), float(spatial_scale), int(pooled_height), int(pooled_width),
                                                int(sampling_ratio), _p(scratch), _p(total), _stream()), "dt_roi_align_backward_plan")
        m = int(total.item())
        ws = torch.empty((L.dt_roi_align_backward_det_workspace_bytes(R, m),), dtype=torch.uint8, device=dev)
        _lib.check(L.dt_roi_align_backward_deterministic(_p(grad_output), _p(rois), R, rois.size(1), B, C, H, W, int(pooled_height), int(pooled_width),
                                                         float(spatial_scale), int(sampling_ratio), m, _p(grad_input), _p(ws), _stream()),
                   "dt_roi_align_backward_deterministic")
    return grad_input


def roi_align_forward_nchw_fast(features, rois, pooled_height, pooled_width, spatial_scale, sampling_ratio, out=None):
    """Same contract as roi_align_forward_nchw; sampling_ratio == 2 takes the separable / FMA fast path (fp32 re-association
    differences only), anything else is forwarded to the exact kernel."""
    _need_cuda(features, rois)
    if not (features.is_contiguous() and rois.is_contiguous()):
        raise RuntimeError("roi_align: features and rois must be contiguous")
    B, C, H, W = features.shape
    R = rois.size(0)
    if out is None:
        out = torch.empty((R, C, pooled_height, pooled_width), device=features.device, dtype=torch.float32)
    L = _lib.lib()
    ws = torch.empty((L.dt_roi_align_fast_workspace_bytes(B, C, H, W, R, int(pooled_height), int(pooled_width)),), dtype=torch.uint8, device=features.device)
    ok = L.dt_roi_align_forward_nchw_fast(_p(features), B, _p(rois), R, rois.size(1), C, H, W, int(pooled_height), int(pooled_width),
                                          float(spatial_scale), int(sampling_ratio), _p(out), _p(ws), _stream())
    _lib.check(ok, "dt_roi_align_forward_nchw_fast")
    return out


def roi_align_forward_nhwc(feats, scales, rois, level, pooled_height, pooled_width, sampling_ratio, num_rois=None):
    """feats: list of NHWC maps [B,H,W,C]; rois [R,5]; level int32 [R] or None -> out [R,ph,pw,C]."""
    _need_cuda(rois, *feats)
    n = len(feats)
    ptrs = (ctypes.c_void_p * n)(*[f.data_ptr() for f in feats])
    hs = (ctypes.c_int * n)(*[f.size(1) for f in feats])
    ws = (ctypes.c_int * n)(*[f.size(2) for f in feats])
    sc = (ctypes.c_float * n)(*[float(s) for s in scales])
    C = feats[0].size(3)
    R = rois.size(0)
    out = torch.empty((R, pooled_height, pooled_width, C), device=rois.device, dtype=torch.float32)
    ok = _lib.lib().dt_roi_align_forward_nhwc(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(hs, ctypes.c_void_p),
                                              ctypes.cast(ws, ctypes.c_void_p), ctypes.cast(sc, ctypes.c_void_p), n, _p(rois),
                                              _p(level), _p(num_rois), R, C, pooled_height, pooled_width, sampling_ratio, _p(out),
                                              _stream())
    _lib.check(ok, "dt_roi_align_forward_nhwc")
    return out


def nms(dets, thresh):
    """dets [N,5] fp32 CUDA (x1,y1,x2,y2,score) -> int64 CUDA tensor of ascending kept indices
    (the contract of lib/utils/boxes.py:332-336)."""
    _need_cuda(dets)
    n = dets.size(0)
    if n == 0:
        return torch.zeros((0,), dtype=torch.int64, device=dets.device)
    dets = dets.contiguous().float()
    L = _lib.lib()
    ws = torch.empty((L.dt_nms_workspace_bytes(n),), dtype=torch.uint8, device=dets.device)
    keep = torch.empty((n,), dtype=torch.int64, device=dets.device)
    cnt = torch.zeros((1,), dtype=torch.int32, device=dets.device)
    _lib.check(L.dt_nms(_p(dets), n, float(thresh), _p(keep), _p(cnt), _p(ws), _stream()), "dt_nms")
    return keep[:int(cnt.item())]


def segm_rle(masks, classes, boxes, im_h, im_w, thresh=0.5, expanded=False, num_dets=None, runs_cap=4096):
    """Mask paste + COCO RLE on the device (lib/utils/result_utils.py:170-228).
    masks [D,K,M,M] (classes int32 [D] selects the plane) or [D,M,M]; boxes [D,4] fp32 reference boxes, or int32 already
    expanded boxes when expanded=True.  Returns (counts list of uint32 arrays, strings list of bytes)."""
    _need_cuda(masks, boxes, classes)
    D = masks.size(0)
    if D == 0:
        return [], []
    masks = masks.contiguous().float()
    M = masks.size(-1)
    K = masks.size(1) if masks.dim() == 4 else 1
    boxes = boxes.contiguous()
    if expanded and boxes.dtype != torch.int32:
        raise TypeError("segm_rle: expanded boxes must be int32")
    if not expanded:
        boxes = boxes.float()
    if classes is not None:
        classes = classes.contiguous().to(torch.int32)
    L = _lib.lib()
    dev = masks.device
    while True:
        ws = torch.empty((L.dt_segm_workspace_bytes(D, runs_cap),), dtype=torch.uint8, device=dev)
        counts = torch.empty((D, runs_cap), dtype=torch.int32, device=dev)
        ncount = torch.empty((D,), dtype=torch.int32, device=dev)
        strings = torch.empty((L.dt_segm_strings_bytes(D, runs_cap),), dtype=torch.uint8, device=dev)
        offs = torch.empty((D + 1,), dtype=torch.int64, device=dev)
        over = torch.zeros((1,), dtype=torch.int32, device=dev)
        ok = L.dt_segm_rle(_p(masks), _p(classes), K, M, _p(None if expanded else boxes), _p(boxes if expanded else None), _p(num_dets), D,
                           int(im_h), int(im_w), float(thresh), _p(counts), _p(ncount), runs_cap, _p(strings), _p(offs), _p(over), _p(ws),
                           _stream())
        _lib.check(ok, "dt_segm_rle")
        need = int(over.item())
        if need == 0:
            break
        runs_cap = max(2 * runs_cap, need + 1)     # a detection needed more runs than provisioned: grow and redo
    offs_h = offs.cpu().numpy()
    str_h = strings[:int(offs_h[-1])].cpu().numpy().tobytes()
    n_h = ncount.cpu().numpy()
    nmax = int(n_h.max()) if D else 0
    cnt_h = counts[:, :max(nmax, 1)].cpu().numpy().view("uint32")
    return [cnt_h[d, :n_h[d]].copy() for d in range(D)], [str_h[offs_h[d]:offs_h[d + 1]] for d in range(D)]


def segm_paste(masks, classes, boxes, im_h, im_w, thresh=0.5, expanded=False, num_dets=None):
    """Pasted binary masks uint8 [D, im_h, im_w] (the im_mask of result_utils.py:203-217 for every detection)."""
    _need_cuda(masks, boxes, classes)
    D = masks.size(0)
    masks = masks.contiguous().float()
    M = masks.size(-1)
    K = masks.size(1) if masks.dim() == 4 else 1
    boxes = boxes.contiguous() if expanded else boxes.contiguous().float()
    if classes is not None:
        classes = classes.contiguous().to(torch.int32)
    out = torch.empty((D, int(im_h), int(im_w)), dtype=torch.uint8, device=masks.device)
    ok = _lib.lib().dt_segm_paste(_p(masks), _p(classes), K, M, _p(None if expanded else boxes), _p(boxes if expanded else None),
                                  _p(num_dets), D, int(im_h), int(im_w), float(thresh), _p(out), _stream())
    _lib.check(ok, "dt_segm_paste")
    return out


def tf32_residual(w):
    lo = torch.empty_like(w)
    _lib.check(_lib.lib().dt_tf32_residual(_p(w), _p(lo), w.numel(), _stream()), "dt_tf32_residual")
    return lo


def fp16_split(w, multiplier=1.0):
    """w fp32 -> (hi, lo) fp16 tensors of w * multiplier (multiplier must be a power of two)."""
    _need_cuda(w)
    hi = torch.empty(w.shape, dtype=torch.float16, device=w.device)
    lo = torch.empty_like(hi)
    _lib.check(_lib.lib().dt_fp16_split(_p(w.contiguous()), w.numel(), float(multiplier), _p(hi), _p(lo), _stream()), "dt_fp16_split")
    return hi, lo


def weight_multiplier(w):
    """Power of two that brings max|w| into [2^13, 2^14): the fp16 low half then stays a normal number for every weight
    within 2^-9 of the largest one."""
    m = float(w.abs().max())
    if not (m > 0.0):
        return 1.0
    import math
    return 2.0 ** (13 - math.floor(math.log2(m)))


def input_multiplier(x):
    """Power of two (>= 1) that brings max|x| up into [2^13, 2^14) for the kind::f16 split: the low half fp16(a - fp16(a)) of an
    activation below 2^-3 is a subnormal fp16 number with a fixed step of 2^-24, which costs inputs with a small scale their
    fp32 accuracy.  Never scales down, so activations >= 65504 still raise the range flag."""
    m = float(x.abs().max()) if x.numel() else 0.0
    if not (m > 0.0) or math.isinf(m):
        return 1.0
    return max(1.0, 2.0 ** (13 - math.floor(math.log2(m))))


def _pix_stride(t, C, what):
    """floats (or halves) between consecutive pixels of an NHWC view whose channels are contiguous"""
    if t.is_contiguous():
        return t.size(3)
    if t.dim() != 4 or t.stride(3) != 1 or t.stride(1) != t.stride(2) * t.size(2) or t.stride(0) != t.stride(1) * t.size(1) or t.stride(2) < C:
        raise RuntimeError("conv2d_nhwc: %s must be an NHWC tensor or a channel slice of one" % what)
    return t.stride(2)


def _plan_dict(plan):
    return {f: int(getattr(plan, f)) for f in _lib.PLAN_FIELDS}


class PreparedConv:
    """One conv layer with every host-side step done (weight split, multipliers, folded scale, descriptor): launch() only calls
    dt_conv2d_spec, so consecutive launch() calls put consecutive conv kernels on the stream with no other work between them."""

    def __init__(self, desc, keep, result):
        self.desc, self._keep, self.result = desc, keep, result

    def launch(self, launch=True):
        """-> the plan (tile geometry and kernel instantiation) as a dict; launch=False only plans"""
        plan = _lib.ConvPlan()
        _lib.check(_lib.lib().dt_conv2d_spec(ctypes.byref(self.desc), ctypes.byref(plan), int(bool(launch)), _stream()), "dt_conv2d_spec")
        return _plan_dict(plan)


def _need(cond, msg):
    if not cond:
        raise RuntimeError("conv2d_nhwc: " + msg)


def conv2d_prepare(x, w_kmajor, scale, shift, kh, kw, pad, stride, w_lo=None, residual=None, up_src=None, relu=False, sigmoid_ch=0,
                   passes=3, force_block_n=0, out=None, kind="tf32", range_flag=None, x_lo=None, out_lo=None, tap0=0, ntaps=0, out_map=None,
                   precise=False, no_merge=False, x_multiplier=None):
    """The arguments of conv2d_nhwc -> a PreparedConv.  With kind "f16" and an fp32 input, pass x_multiplier when x is not written yet
    (input_multiplier reads it)."""
    _need_cuda(x, w_kmajor)
    N, H, W, Cin = x.shape
    Cout = w_kmajor.size(0)
    Ho = (H + 2 * pad - kh) // stride + 1
    Wo = (W + 2 * pad - kw) // stride + 1
    planes_in, planes_out = x_lo is not None, out_lo is not None
    _need(kind == "f16" or not (planes_in or planes_out), "fp16 planes need kind 'f16'")
    _need(x.dtype == (torch.float16 if planes_in else torch.float32), "x must be fp16 (the high plane, with x_lo) or fp32")
    if planes_in:
        _need(x_lo.dtype == torch.float16 and x_lo.shape == x.shape and x.is_contiguous() and x_lo.is_contiguous(),
              "x / x_lo must be dense fp16 planes of the same shape")
    odt = torch.float16 if planes_out else torch.float32
    if out is None:
        _need(out_map is None, "out_map needs the output buffer")
        out = torch.empty((N, Ho, Wo, Cout), device=x.device, dtype=odt)
    _need(out.dtype == odt and out.dim() == 4 and out.size(3) == Cout and out.size(0) == N, "out must be [N,*,*,Cout] %s" % odt)
    if planes_out:
        _need(out_lo.dtype == torch.float16 and out_lo.shape == out.shape and out.is_contiguous() and out_lo.is_contiguous(),
              "out / out_lo must be dense fp16 planes of the same shape")
    if out_map is None:
        _need(tuple(out.shape[1:3]) == (Ho, Wo), "out must be [N,%d,%d,Cout]" % (Ho, Wo))
    else:
        oh, ow, step, y0, x0 = [int(v) for v in out_map]
        _need(not planes_out, "out_map writes fp32 outputs only")
        _need(tuple(out.shape[1:3]) == (oh, ow), "out must be [N,out_h,out_w,Cout] for out_map")
        _need(step > 0 and y0 >= 0 and x0 >= 0 and (Ho - 1) * step + y0 < oh and (Wo - 1) * step + x0 < ow,
              "out_map scatters outside the output buffer")
    for t, what in ((residual, "residual"), (up_src, "up_src")):
        if t is not None:
            _need(t.dtype == torch.float32 and t.dim() == 4 and t.size(0) == N and t.size(3) == Cout, "%s must be [N,*,*,Cout] fp32" % what)
    if residual is not None:
        _need(tuple(residual.shape[1:3]) == (Ho, Wo), "residual must be [N,Ho,Wo,Cout]")
    if up_src is not None:
        _need(up_src.is_contiguous() and up_src.size(1) * 2 >= Ho and up_src.size(2) * 2 >= Wo, "up_src must be a dense [N,ceil(Ho/2),ceil(Wo/2),Cout] map")
    res_mode = 1 if residual is not None else (2 if up_src is not None else 0)
    d = _lib.ConvDesc()
    d.kind = 1 if kind == "f16" else 0
    d.x, d.x_lo = _p(x).value, _p(x_lo).value
    d.N, d.H, d.W, d.Cin = N, H, W, Cin
    d.x_pix_stride = Cin if planes_in else _pix_stride(x, Cin, "x")
    d.Cout, d.kh, d.kw, d.pad, d.stride = Cout, kh, kw, pad, stride
    d.y, d.y_lo = _p(out).value, _p(out_lo).value
    d.y_pix_stride = Cout if planes_out else _pix_stride(out, Cout, "out")
    if out_map is not None:
        d.out_h, d.out_w, d.out_step, d.out_y0, d.out_x0 = oh, ow, step, y0, x0
    d.residual = _p(residual).value
    d.res_pix_stride = _pix_stride(residual, Cout, "residual") if residual is not None else 0
    d.up_src = _p(up_src).value
    d.up_h, d.up_w = (up_src.size(1), up_src.size(2)) if up_src is not None else (0, 0)
    d.res_mode, d.relu, d.sigmoid_ch, d.passes = res_mode, int(relu), int(sigmoid_ch), int(passes)
    d.tap0, d.ntaps, d.no_merge = int(tap0), int(ntaps), int(no_merge)
    d.precise = int(bool(precise) or force_block_n < 0)
    d.force_block_n = 128 if force_block_n < 0 else int(force_block_n)
    d.range_flag = _p(range_flag).value
    if kind == "f16":
        mult = weight_multiplier(w_kmajor)
        hi, lo = fp16_split(w_kmajor, mult)
        xm = 1.0
        if not planes_in:
            xm = float(x_multiplier) if x_multiplier is not None else input_multiplier(x)
        sc = (scale / (mult * xm)).contiguous()
        d.x_multiplier = xm
    else:
        if w_lo is None:
            w_lo = tf32_residual(w_kmajor)
        hi, lo, sc = w_kmajor, w_lo, scale
    d.w_hi, d.w_lo, d.scale, d.shift = _p(hi).value, _p(lo).value, _p(sc).value, _p(shift).value
    keep = (x, x_lo, hi, lo, sc, shift, out, out_lo, residual, up_src, range_flag)
    return PreparedConv(d, keep, out if out_lo is None else (out, out_lo))


def conv2d_nhwc(*args, return_plan=False, launch=True, **kw):
    """x [N,H,W,Cin] fp32 (channels-last memory, or a channel slice of a wider NHWC tensor), w_kmajor [Cout, kh*kw*Cin] -> y [N,Ho,Wo,Cout].
    Arguments: (x, w_kmajor, scale, shift, kh, kw, pad, stride, w_lo=None, residual=None, up_src=None, relu=False, sigmoid_ch=0, passes=3,
    force_block_n=0, out=None, kind="tf32", range_flag=None, x_lo=None, out_lo=None, tap0=0, ntaps=0, out_map=None, precise=False,
    no_merge=False, x_multiplier=None).
    kind "tf32": 3xTF32 (w_lo = tf32 residual); kind "f16": 3xFP16 on the kind::f16 pipe (weights split here; fp32 inputs are lifted by
    input_multiplier(x) unless x_multiplier is given).
    Layer options of the engine (dt_conv2d_spec): x_lo -- x and x_lo are the fp16 hi / lo planes of the input; out_lo -- write the output as
    fp16 planes into out / out_lo; taps [tap0, tap0 + ntaps) only (ntaps 0 = all); out_map = (out_h, out_w, step, y0, x0): output pixel
    (n,h,w) goes to pixel (n, h*step + y0, w*step + x0) of `out` [N,out_h,out_w,*]; `out` / `residual` may be channel slices of wider
    buffers; precise: 3 rotating accumulators (128-wide tiles); no_merge: cross terms in their own accumulator.
    return_plan: also return the plan (tile geometry and kernel instantiation) as a dict; launch=False only plans."""
    pc = conv2d_prepare(*args, **kw)
    plan = pc.launch(launch)
    return (pc.result, plan) if return_plan else pc.result


def conv_plan(*args, **kw):
    """The plan conv2d_nhwc(*args, **kw) would run -- tile geometry and kernel instantiation -- without launching it."""
    kw = dict(kw, return_plan=True, launch=False)
    return conv2d_nhwc(*args, **kw)[1]


def conv2d_stem(x4, w, scale, shift, H1, W1, kind="f16", passes=3, range_flag=None, out=None, x_multiplier=None, return_plan=False, launch=True):
    """The 7x7 stride-2 stem over a zero-bordered NHWC4 image: x4 fp32 [B,Hp,Wp,4], or (kind "f16") fp16 [2,B,Hp,Wp,4] holding its hi and
    lo planes; w [64, 7*32] fp32 (row ky, element kx*4 + c); -> relu(conv*scale + shift) [B,H1,W1,64]."""
    _need_cuda(x4, w)
    planes = x4.dtype == torch.float16
    B, Hp, Wp = x4.shape[-4:-1] if planes else x4.shape[:3]
    if out is None:
        out = torch.empty((B, H1, W1, 64), device=x4.device, dtype=torch.float32)
    xm = 1.0
    if kind == "f16":
        mult = weight_multiplier(w)
        hi, lo = fp16_split(w, mult)
        if not planes:
            xm = float(x_multiplier) if x_multiplier is not None else input_multiplier(x4)
        sc = (scale / (mult * xm)).contiguous()
    else:
        hi, lo, sc = w, tf32_residual(w), scale
    plan = _lib.ConvPlan()
    ok = _lib.lib().dt_conv2d_stem(_p(x4), int(planes), B, Hp, Wp, int(H1), int(W1), _p(hi), _p(lo), 1 if kind == "f16" else 0, _p(sc), _p(shift),
                                   float(xm), int(passes), _p(range_flag), _p(out), ctypes.byref(plan), int(bool(launch)), _stream())
    _lib.check(ok, "dt_conv2d_stem")
    return (out, _plan_dict(plan)) if return_plan else out


def conv_instantiations():
    """The conv kernel instantiation table: one (block_n, nmain, two_sm, kind, ring, slots, halo, ws) tuple per row."""
    L = _lib.lib()
    rows = []
    for i in range(L.dt_conv_instantiation_count()):
        f = (ctypes.c_int * 8)()
        _lib.check(L.dt_conv_instantiation_info(i, f), "dt_conv_instantiation_info")
        rows.append(tuple(int(v) for v in f))
    return rows
