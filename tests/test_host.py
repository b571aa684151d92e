"""CPU tests of the host side: the C-ABI library builds for sm_100a without a GPU, loads, and exports
every symbol include/detectorch_b200.h declares; the engine's parameter table equals the reference's
state_dict names; the product path refuses to run without CUDA (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "detectorch_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dt_[a-z0-9_]+|launch_roi_align_[a-z]+_cuda)\s*\(", src)) - {"dt_engine_config"})


def test_library_exports_every_declared_symbol(built):
    from detectorch_b200 import _lib
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = header_functions()
    assert "launch_roi_align_forward_cuda" in names and "launch_roi_align_backward_cuda" in names and "dt_engine_run" in names
    assert "dt_segm_rle" in names and "dt_prep_image" in names and "dt_conv2d_nhwc_f16x3" in names and len(names) >= 33
    for n in names:
        assert hasattr(L, n), "library does not export %s" % n
    assert b"sm_100a" in _lib.lib().dt_version()


def test_ctypes_signatures_cover_operator_api(built):
    from detectorch_b200 import _lib
    for n in ("launch_roi_align_forward_cuda", "launch_roi_align_backward_cuda", "dt_roi_align_forward_nchw", "dt_roi_align_forward_nhwc", "dt_nms",
              "dt_conv2d_nhwc", "dt_conv2d_nhwc_f16x3", "dt_conv2d_spec", "dt_conv2d_stem", "dt_conv_instantiation_count",
              "dt_conv_instantiation_info", "dt_fp16_split", "dt_segm_rle", "dt_segm_paste", "dt_prep_image"):
        assert n in _lib.SIGNATURES


def test_conv_desc_and_plan_structs_match_header(built):
    """The ctypes mirrors of dt_conv_desc / dt_conv_plan list the header's fields in the header's order with the same C types, and the
    instantiation table is exported (39 rows of distinct kernel template arguments)."""
    from detectorch_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "detectorch_b200.h")).read(), flags=re.S)
    ctype = {"int": ctypes.c_int, "float": ctypes.c_float}
    for cname, py in (("dt_conv_desc", _lib.ConvDesc), ("dt_conv_plan", _lib.ConvPlan)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), src, re.S).group(1)
        fields = []
        for decl in body.split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            m = re.match(r"(const )?(int|float|void|char)\s*(\*?)\s*(.*)", decl)
            base, ptr = m.group(2), m.group(3)
            for name in m.group(4).split(","):
                name = name.strip()
                star = ptr or name.startswith("*")
                fields.append((name.lstrip("* "), ctypes.c_void_p if star else ctype[base]))
        assert [(f, t) for f, t in py._fields_] == fields, cname
    rows = __import__("detectorch_b200.ops", fromlist=["ops"]).conv_instantiations()
    assert len(rows) == 39 and len(set(rows)) == 39


def test_engine_param_table_matches_reference_names(built):
    from detectorch_b200 import engine
    from oracle import network as net
    for arch in ("resnet50", "resnet101"):
        t = engine.param_table(arch)
        s = {k: int(np.prod(v)) for k, v in net.param_shapes(arch).items()}
        assert t == s
        t4 = engine.param_table(arch, model="c4")
        assert t4 == {k: int(np.prod(v)) for k, v in net.param_shapes(arch, fpn=False).items()}


def test_mirror_detector_state_dict_names(built):
    """The drop-in detector exposes the reference's state_dict names (so pickles / checkpoints load unchanged)."""
    from detectorch_b200.model.detector import detector
    from oracle import network as net
    m = detector(arch='resnet50', conv_body_layers=['conv1', 'bn1', 'relu', 'maxpool', 'layer1', 'layer2', 'layer3', 'layer4'],
                 conv_head_layers='two_layer_mlp', fpn_layers=['layer1', 'layer2', 'layer3', 'layer4'], fpn_extra_lvl=True,
                 roi_height=7, roi_width=7, roi_spatial_scale=[0.25, 0.125, 0.0625, 0.03125], roi_sampling_ratio=2,
                 use_rpn_head=True, use_mask_head=True, mask_head_type='1up4convs')
    sd = m.state_dict()
    for k, shape in net.param_shapes('resnet50').items():
        assert k in sd and tuple(sd[k].shape) == tuple(shape), k
    for attr in ("model", "conv_body", "conv_head", "rpn", "bbox_head", "classif_head", "mask_head"):
        assert hasattr(m, attr)
    # the C4 family (defaults of the reference constructor) exposes the reference's names as well
    m4 = detector(arch='resnet50', use_rpn_head=True, use_mask_head=True, mask_head_type='upshare')
    sd4 = m4.state_dict()
    for k, shape in net.param_shapes('resnet50', fpn=False).items():
        assert k in sd4 and tuple(sd4[k].shape) == tuple(shape), k
    with pytest.raises(NotImplementedError):
        detector(arch='resnet50', roi_height=9)      # configurations the reference's notebooks never use: loud, not silent


def test_no_cpu_fallback(built):
    from detectorch_b200 import ops
    from detectorch_b200.model.roi_align import RoIAlignFunction, preprocess_rois
    f, r = torch.zeros(1, 4, 8, 8), torch.zeros(3, 5)
    with pytest.raises(TypeError):
        ops.roi_align_forward_nchw(f, r, 7, 7, 0.25, 2)
    with pytest.raises(TypeError):
        RoIAlignFunction.apply(f, r, 7, 7, 0.25, 2)
    with pytest.raises(TypeError):
        ops.nms(torch.zeros(4, 5), 0.5)
    # preprocess_rois keeps the reference's conventions (roi_align.py:172-188)
    assert preprocess_rois(torch.ones(5, 4)).shape == (5, 5) and float(preprocess_rois(torch.ones(5, 4))[:, 0].sum()) == 0.0
    assert preprocess_rois([torch.ones(2, 5), torch.ones(3, 5)]).shape == (5, 5)
    assert preprocess_rois(torch.ones(1, 6, 4)).shape == (6, 5)
    if not torch.cuda.is_available():
        from detectorch_b200.engine import Engine
        with pytest.raises(RuntimeError):
            Engine(batch=1, height=64, width=64)


def test_product_path_does_not_import_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "detectorch_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(root, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "oracle/" not in txt.replace("parity oracle", ""), f


def test_lib_overlay_imports(built):
    """The reference-facing overlay (lib/, INTEGRATION.md) resolves `cppcuda_cffi.roialign`, `model.detector`, `model.roi_align`,
    `utils.result_utils`, `utils.preprocess_sample` to this package (fresh interpreter: the names must not collide with anything)."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r + '/lib'); sys.path.insert(0, %r)\n"
            "import cppcuda_cffi.roialign as r, model.detector as d, model.roi_align as a, utils.result_utils as u, utils.preprocess_sample as p\n"
            "assert all(hasattr(r, n) for n in ('roi_align_forward_cuda', 'roi_align_backward_cuda', 'roi_align_forward_cpu'))\n"
            "assert hasattr(d, 'detector') and hasattr(a, 'RoIAlignFunction') and hasattr(u, 'postprocess_output') and hasattr(u, 'segm_results')\n"
            "assert hasattr(p, 'preprocess_sample'); print('OVERLAY IMPORTS OK')\n") % (ROOT, ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OVERLAY IMPORTS OK" in out.stdout, out.stderr[-1500:]


def test_host_side_helpers():
    """Host logic of the new entry points: the prep_im_for_blob scale rule (blob.py:67-76) and the power-of-two weight pre-scale
    of the kind::f16 convolutions."""
    from detectorch_b200.utils.blob import im_scale_for
    from detectorch_b200 import ops
    from oracle import ref
    rng = np.random.RandomState(0)
    for (h, w) in [(480, 640), (375, 1242), (1600, 2000), (64, 48), (800, 1216), (333, 500)]:
        im = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
        # the oracle restatement (pinned to the reference's blob.py) gives the scale; skip its resize for the big images
        want = ref.prep_im_for_blob(im, target_sizes=[800], max_size=1333)[1][0] if h * w < 400000 else None
        got = im_scale_for((h, w, 3), 800, 1333)
        if want is not None:
            assert got == want
        assert np.round(got * max(h, w)) <= 1333 + 1e-9 and (abs(got * min(h, w) - 800) < 1e-9 or abs(got * max(h, w) - 1333) < 1e-9)
    for m in (3e-4, 0.02, 0.7, 1.0, 5.5, 300.0):
        w_ = torch.tensor([m, -m / 3, 0.0])
        mult = ops.weight_multiplier(w_)
        assert 2.0 ** 13 <= m * mult < 2.0 ** 14 and np.log2(mult) == int(np.log2(mult))
    assert ops.weight_multiplier(torch.zeros(4)) == 1.0


@pytest.mark.parametrize("notebook", ["eval_fast.ipynb", "eval_faster.ipynb", "eval_mask.ipynb", "eval_fast_FPN.ipynb", "eval_faster_FPN.ipynb",
                                      "eval_mask_FPN.ipynb"])
def test_notebook_setup_cells_run_on_the_overlay(built, tmp_path, notebook):
    """CPU half of tests/test_gpu_notebooks.py: the reference notebook's import cell, paths cell, detector(...) constructor cell (with a
    synthetic Detectron pickle -> load_pretrained_weights for that configuration) and the empty_results cell execute verbatim against the
    lib/ overlay (the detection loop needs a GPU and runs in the gpu-marked test)."""
    import pickle
    import subprocess
    import sys
    from oracle import reference_shim as rs
    if not rs.staged_available():
        pytest.skip("oracle/_ref/reflib.zip not staged (oracle/build_ref.sh needs the reference tree once)")
    out = os.path.join(str(tmp_path), "res.pkl")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "notebook_harness.py"), notebook, out, "--cpu"], capture_output=True, text=True,
                       timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0 and "NOTEBOOK OK" in r.stdout, r.stderr[-3000:]
    res = pickle.load(open(out, "rb"))
    assert res["detector_module"] == "detectorch_b200.model.detector" and os.path.join(ROOT, "lib") in res["result_utils_file"]
    assert len(res["all_boxes"]) == 81 and len(res["all_boxes"][1]) == 2 and res["all_boxes"][1][0] == []
    assert res["all_boxes"][1] is not res["all_boxes"][2] and res["all_boxes"] is not res["all_segms"]


def test_result_containers_and_multilevel_rois():
    """empty_results / extend_results (result_utils.py:32-60) and the FPN level mapping used for pre-computed boxes
    (multilevel_rois.py:19-82) -- host helpers of the mirror, against the oracle restatement."""
    from detectorch_b200.utils import result_utils as ru
    from detectorch_b200.utils.multilevel_rois import add_multilevel_rois_for_test
    from oracle import ref
    a, b, c = ru.empty_results(5, 3)
    assert len(a) == 5 and all(len(x) == 3 for x in a) and a[1][0] == [] and a is not b and a[1] is not a[2] and a[1][0] is not a[1][1]
    ru.extend_results(2, a, [["bg"], ["c1"], ["c2"], ["c3"], ["c4"]])
    assert a[0][2] == [] and a[1][2] == ["c1"] and a[4][2] == ["c4"] and a[1][0] == []
    rng = np.random.RandomState(3)
    x1, y1 = rng.uniform(0, 900, 300), rng.uniform(0, 600, 300)
    r = np.stack([x1, y1, x1 + np.exp(rng.uniform(1, 6.5, 300)), y1 + np.exp(rng.uniform(1, 6.5, 300))], 1).astype(np.float32)
    blobs = add_multilevel_rois_for_test({'rois': r}, 'rois')
    per_level, restore = ref.multilevel_rois_for_test(r)
    for i, l in enumerate(range(2, 6)):
        assert np.array_equal(blobs['rois_fpn%d' % l], per_level[i])
    assert np.array_equal(blobs['rois_idx_restore_int32'], restore) and blobs['rois_idx_restore_int32'].dtype == np.int32
    assert np.array_equal(np.concatenate(per_level, 0)[restore], r)


def test_bn_running_stats_fold():
    """Engine.load_state_dict folds non-trivial BatchNorm running statistics into the (gamma, beta) pair the engine applies as
    gamma / sqrt(1 + eps), beta: the result must equal torch's eval-mode BatchNorm."""
    from detectorch_b200.engine import fold_bn_running_stats
    g = torch.Generator().manual_seed(0)
    sd = {"model.bn1.weight": torch.rand(64, generator=g) + 0.5, "model.bn1.bias": torch.randn(64, generator=g),
          "model.bn1.running_mean": torch.randn(64, generator=g), "model.bn1.running_var": torch.rand(64, generator=g) + 0.3,
          "model.layer1.0.bn1.weight": torch.rand(8, generator=g), "model.layer1.0.bn1.bias": torch.randn(8, generator=g),
          "model.layer1.0.bn1.running_mean": torch.zeros(8), "model.layer1.0.bn1.running_var": torch.ones(8)}
    out = fold_bn_running_stats(sd)
    x = torch.randn(2, 64, 5, 5, generator=g)
    want = torch.nn.functional.batch_norm(x, sd["model.bn1.running_mean"], sd["model.bn1.running_var"], sd["model.bn1.weight"], sd["model.bn1.bias"],
                                          False, 0.0, 1e-5)
    got = x * (out["model.bn1.weight"] / np.sqrt(1 + 1e-5)).view(1, -1, 1, 1) + out["model.bn1.bias"].view(1, -1, 1, 1)
    assert (got - want).abs().max().item() < 1e-5
    assert out["model.layer1.0.bn1.weight"] is sd["model.layer1.0.bn1.weight"]      # trivial stats (the reference's case): untouched, bit-identical
