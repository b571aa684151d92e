"""CPU test of the Detectron caffe2-pickle weight import (SURVEY.md 8f "next" row 2): a synthetic pickle written with the
reference's own blob names loads into the detectorch_b200 mirror exactly as it loads into the reference detector, for the
constructor kwargs of every eval_*.ipynb notebook (Fast / Faster / Mask R-CNN on the C4 and on the FPN body: the loader
branches on use_rpn_head / use_fpn_body / mask_head_type / two_layer_mlp exactly like detector.py:317-374).
The blob names (the reference's utils.utils.parse_th_to_caffe2) and what the reference's loader made of each pickle are stored in
tests/golden/pickle_golden.npz (tests/golden/make_crosscheck_golden.py runs the reference to produce them)."""
import hashlib
import os
import pickle

import numpy as np
import pytest
import torch

from oracle import network as net

FPN = dict(arch='resnet50', conv_body_layers=['conv1', 'bn1', 'relu', 'maxpool', 'layer1', 'layer2', 'layer3', 'layer4'],
           conv_head_layers='two_layer_mlp', fpn_layers=['layer1', 'layer2', 'layer3', 'layer4'],
           roi_height=7, roi_width=7, roi_spatial_scale=[0.25, 0.125, 0.0625, 0.03125], roi_sampling_ratio=2)
# name -> (constructor kwargs as the notebook passes them, oracle parameter-set flags)
CONFIGS = {
    "eval_fast": (dict(arch='resnet50'), dict(fpn=False, rpn=False, mask=False)),
    "eval_faster": (dict(arch='resnet50', use_rpn_head=True), dict(fpn=False, rpn=True, mask=False)),
    "eval_mask": (dict(arch='resnet50', use_rpn_head=True, use_mask_head=True), dict(fpn=False, rpn=True, mask=True)),
    "eval_fast_FPN": (dict(FPN), dict(fpn=True, rpn=False, mask=False)),
    "eval_faster_FPN": (dict(FPN, fpn_extra_lvl=True, use_rpn_head=True), dict(fpn=True, rpn=True, mask=False)),
    "eval_mask_FPN": (dict(FPN, fpn_extra_lvl=True, use_rpn_head=True, use_mask_head=True, mask_head_type='1up4convs'), dict(fpn=True, rpn=True, mask=True)),
}


GOLD = os.path.join(os.path.dirname(__file__), "golden", "pickle_golden.npz")


def sha1(t):
    return hashlib.sha1(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def write_detectron_pickle(path, G, name, P):
    """A pickle in the published checkpoints' format ({'blobs': {caffe2 name: ndarray}}), filled from the flat parameter dict P by the
    recipe stored for this configuration (blob name, parameter it holds or '' for a zero blob, BGR stem flag)."""
    blobs = {}
    for blob, src, bgr in zip(G[name + "_blob"], G[name + "_src"], G[name + "_bgr"]):
        w = P[str(src)].numpy() if src else np.zeros((), np.float32)
        blobs[str(blob)] = w[:, (2, 1, 0), :, :].copy() if bgr else w     # pickles hold BGR
    with open(path, "wb") as f:
        pickle.dump({'blobs': blobs}, f, protocol=2)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_detectron_pickle_loads_like_the_reference(tmp_path, built, name):
    from detectorch_b200.model.detector import detector as b200_detector
    G = np.load(GOLD)
    kw, flags = CONFIGS[name]
    P = net.synthetic_params("resnet50", **flags)
    pkl = os.path.join(str(tmp_path), "model_final.pkl")
    write_detectron_pickle(pkl, G, name, P)
    mine = b200_detector(detector_pkl_file=pkl, **kw)                    # exactly the notebook's cell 7
    sm = mine.state_dict()
    assert [str(k) for k in G[name + "_keys"]] == sorted(P)
    for k, want in zip(G[name + "_keys"], G[name + "_sha1"]):
        k = str(k)
        assert torch.equal(sm[k], P[k]), "mirror loader: " + k
        assert sha1(sm[k]) == str(want), "differs from the reference loader: " + k
    # and the engine's parameter table accepts exactly these names
    from detectorch_b200 import engine
    t = engine.param_table("resnet50", use_mask=flags["mask"], model="fpn" if flags["fpn"] else "c4", use_rpn=flags["rpn"])
    assert set(t) == set(P) and all(t[k] == int(np.prod(P[k].shape)) for k in P)


def test_caffe2_blob_names_match_the_reference_helper():
    """The mirror's own torchvision-name -> caffe2-blob-name mapping equals utils/utils.py:44-71 (parse_th_to_caffe2) on every trunk key."""
    from detectorch_b200.model.detector import caffe2_blob_name
    G = np.load(GOLD)
    for arch in ("resnet50", "resnet101"):
        keys, names = G["names_%s_keys" % arch], G["names_%s_blobs" % arch]
        assert len(keys) > 150 and len(keys) == len(names)
        for k, n in zip(keys, names):
            assert caffe2_blob_name(str(k)) == str(n), k
