"""ctypes binding of the C-ABI library (include/detectorch_b200.h).  There is NO fallback: if the
CUDA library is missing or fails to load, importing an operator raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DETECTORCH_B200_LIB selects another build of the same library (A/B experiments with compile-time kernel switches); default: the in-tree build
LIB_PATH = os.environ.get("DETECTORCH_B200_LIB") or os.path.join(_HERE, "csrc", "libdetectorch_b200.so")
_lib = None

c_void_p, c_int, c_int64, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float


class ConvDesc(ctypes.Structure):
    """struct dt_conv_desc"""
    _fields_ = [("kind", c_int), ("x", c_void_p), ("x_lo", c_void_p), ("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int),
                ("x_pix_stride", c_int), ("x_multiplier", c_float), ("w_hi", c_void_p), ("w_lo", c_void_p), ("Cout", c_int), ("kh", c_int),
                ("kw", c_int), ("pad", c_int), ("stride", c_int), ("scale", c_void_p), ("shift", c_void_p), ("y", c_void_p), ("y_lo", c_void_p),
                ("y_pix_stride", c_int), ("out_h", c_int), ("out_w", c_int), ("out_step", c_int), ("out_y0", c_int), ("out_x0", c_int),
                ("residual", c_void_p), ("res_pix_stride", c_int), ("up_src", c_void_p), ("up_h", c_int), ("up_w", c_int), ("res_mode", c_int),
                ("relu", c_int), ("sigmoid_ch", c_int), ("passes", c_int), ("tap0", c_int), ("ntaps", c_int), ("force_block_n", c_int),
                ("precise", c_int), ("no_merge", c_int), ("range_flag", c_void_p)]


PLAN_FIELDS = ("instantiation", "block_n", "nmain", "two_sm", "kind", "ring", "slots", "halo", "ws", "wbox", "hbox", "nbox", "tiles_w", "tiles_h",
               "tiles_n", "m_pairs", "n_tiles", "grid", "num_kb", "ho", "wo")


class ConvPlan(ctypes.Structure):
    """struct dt_conv_plan"""
    _fields_ = [(f, c_int) for f in PLAN_FIELDS]

# symbol -> (restype, argtypes); mirrors include/detectorch_b200.h
SIGNATURES = {
    "dt_version": (ctypes.c_char_p, []),
    "launch_roi_align_forward_cuda": (c_int, [c_int, c_void_p, c_void_p, c_float, c_int, c_int, c_int, c_int, c_int, c_int,
                                              c_void_p, c_void_p]),
    "launch_roi_align_backward_cuda": (c_int, [c_int, c_void_p, c_int, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                               c_int, c_void_p]),
    "dt_roi_align_forward_nchw": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                          c_void_p, c_void_p]),
    "dt_roi_align_fast_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int64, c_int, c_int]),
    "dt_roi_align_forward_nchw_fast": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                               c_void_p, c_void_p, c_void_p]),
    "dt_roi_align_forward_nhwc": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                          c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dt_nms_workspace_bytes": (c_int64, [c_int64]),
    "dt_nms": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dt_segm_workspace_bytes": (c_int64, [c_int, c_int]),
    "dt_segm_strings_bytes": (c_int64, [c_int, c_int]),
    "dt_segm_rle": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                            c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dt_segm_paste": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                              c_void_p, c_void_p]),
    "dt_roi_align_backward_det_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "dt_roi_align_backward_plan": (c_int, [c_void_p, c_int64, c_int, c_float, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dt_roi_align_backward_deterministic": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                                    c_int64, c_void_p, c_void_p, c_void_p]),
    "dt_prep_image": (c_int, [c_void_p, c_int, c_int, c_void_p, ctypes.c_double, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "dt_tf32_residual": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dt_fp16_split": (c_int, [c_void_p, c_int64, c_float, c_void_p, c_void_p, c_void_p]),
    "dt_conv2d_nhwc_f16x3": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                     c_void_p, c_int, c_void_p]),
    "dt_conv2d_spec": (c_int, [ctypes.POINTER(ConvDesc), ctypes.POINTER(ConvPlan), c_int, c_void_p]),
    "dt_conv2d_stem": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_float, c_int,
                               c_void_p, c_void_p, ctypes.POINTER(ConvPlan), c_int, c_void_p]),
    "dt_conv_instantiation_count": (c_int, []),
    "dt_conv_instantiation_info": (c_int, [c_int, ctypes.POINTER(c_int)]),
    "dt_conv2d_nhwc": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_int, c_void_p]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("detectorch_b200: %s not built. Run `python -m detectorch_b200.build` "
                               "(or __graft_entry__.build()). There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError if the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(ok, what):
    if ok != 1:
        raise RuntimeError("detectorch_b200: %s failed (see stderr)" % what)
