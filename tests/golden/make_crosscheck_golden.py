"""Generates the fixtures of the cross-checks against the reference's own code, by RUNNING THE REFERENCE (imported unmodified through
oracle/reference_shim.py, its compiled RoIAlign loops and Cython NMS from oracle/_ref).  Only runnable where the reference tree exists;
the fixtures are committed so that the tests run anywhere.

  crosscheck_golden.npz  (tests/test_oracle.py)
    nms*         the reference's box_utils.nms on random boxes (n = 5, 333, 1500; thresholds 0.3, 0.7)
    roi*         the reference's RoIAlign CPU loop (4 x 13 x 19 map, 80 RoIs partly outside it; 7x7 sr 2 and 14x14 sr 0)
    prep*        the reference's blob.prep_im_for_blob + im_list_to_blob (real cv2 with IPP off): up-scale, portrait cap, exact 1/2
    segm*        the reference's segm_results, mask_util.encode replaced by a recorder of the pasted mask (pycocotools is not installed)
    bwd*         the reference's RoIAlign backward loop (libroialign_bwd_ref.so) on three random cases
  pickle_golden.npz  (tests/test_pickle_import.py)
    names_<arch>_{keys,blobs}   the reference's utils.utils.parse_th_to_caffe2 on every torchvision ResNet trunk key
    <config>_{blob,src,bgr}     a Detectron pickle in the published checkpoints' format: blob name, flat parameter it holds ('' = the
                                zero num_batches_tracked blob the reference's loader expects), BGR stem flag
    <config>_{keys,sha1}        sha1 of every parameter in the reference detector's state_dict after loading that pickle

    python tests/golden/make_crosscheck_golden.py
"""
import hashlib
import os
import pickle
import sys
import tempfile

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import network as net  # noqa: E402
from oracle import ref  # noqa: E402
from oracle import reference_shim as rs  # noqa: E402
from test_pickle_import import CONFIGS, FPN  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def sha1(t):
    return hashlib.sha1(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def crosscheck():
    import utils.blob as rb
    import utils.boxes as box_utils
    import utils.result_utils as ru
    G = {}
    rng = np.random.RandomState(7)
    for i, n in enumerate((5, 333, 1500)):
        x1 = rng.uniform(0, 900, n); y1 = rng.uniform(0, 600, n)
        d = np.stack([x1, y1, x1 + rng.uniform(2, 300, n), y1 + rng.uniform(2, 300, n), rng.uniform(0, 1, n)], 1).astype(np.float32)
        G["nms%d_dets" % i] = d
        for t in (0.3, 0.7):
            G["nms%d_t%d_keep" % (i, int(t * 10))] = np.asarray(box_utils.nms(d, t), dtype=np.int64)
    f = rng.randn(1, 4, 13, 19).astype(np.float32)
    x1 = rng.uniform(-40, 500, 80); y1 = rng.uniform(-40, 300, 80)
    r = np.stack([np.zeros(80), x1, y1, x1 + rng.uniform(1, 400, 80), y1 + rng.uniform(1, 300, 80)], 1).astype(np.float32)
    G["roi_feat"], G["roi_rois"] = f, r
    for (p, sr) in ((7, 2), (14, 0)):
        G["roi_out_p%d_sr%d" % (p, sr)] = ref.roi_align_forward_ref(f, r, p, p, 1 / 32., sr)

    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        rng = np.random.RandomState(123)
        cases = ((37, 52, 60, 100), (80, 41, 40, 1333), (64, 96, 32, 1333))
        G["prep_cases"] = np.array(cases, np.int64)
        for i, (h, w, ts, ms) in enumerate(cases):
            im = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
            ims, scales = rb.prep_im_for_blob(im.copy(), target_sizes=[ts], max_size=ms)
            G["prep_im%d" % i], G["prep_scale%d" % i], G["prep_blob%d" % i] = im, np.float64(scales[0]), rb.im_list_to_blob(ims, fpn_on=True)
        captured = []
        ru.mask_util.encode = lambda arr: (captured.append(np.ascontiguousarray(arr[:, :, 0])) or
                                           [{'size': list(arr.shape[:2]), 'counts': ref.rle_to_string(ref.rle_encode(arr[:, :, 0]))}])
        M, K, im_h, im_w = 28, 3, 120, 150
        boxes = np.array([[3.2, 4.1, 60.7, 80.3], [100, 20, 149, 119], [0, 0, 149, 119], [70, 70, 83, 83], [10, 90, 40, 119]], np.float32)
        cls = np.array([1, 1, 2, 2, 2])
        masks = rng.rand(5, K, M, M).astype(np.float32)
        cls_boxes = [[], np.hstack([boxes[cls == 1], np.ones((2, 1), np.float32)]), np.hstack([boxes[cls == 2], np.ones((3, 1), np.float32)])]
        segms = ru.segm_results(cls_boxes, masks, boxes, im_h, im_w, num_classes=K, M=M)
        assert len(captured) == 5
        G["segm_boxes"], G["segm_cls"], G["segm_masks"] = boxes, cls, masks
        G["segm_size"] = np.array([im_h, im_w], np.int64)
        G["segm_counts"] = np.array([s['counts'].decode() if isinstance(s['counts'], bytes) else s['counts'] for j in range(1, K) for s in segms[j]])
        G["segm_pasted_bits"] = np.packbits(np.stack(captured).reshape(5, -1), axis=1)
    finally:
        cv2.ipp.setUseIPP(ipp)

    rng = np.random.RandomState(5)
    for i, (PH, sr, scale) in enumerate(((7, 2, 0.25), (14, 0, 0.0625), (7, 0, 0.125))):
        B, C, H, W, R = 2, 3, 18, 26, 30
        x1, y1 = rng.uniform(-10, W / scale, R), rng.uniform(-10, H / scale, R)
        r = np.stack([rng.randint(0, B, R).astype(np.float32), x1, y1, x1 + rng.uniform(1, 300, R), y1 + rng.uniform(1, 300, R)], 1).astype(np.float32)
        top = rng.randn(R, C, PH, PH).astype(np.float32)
        G["bwd%d_rois" % i], G["bwd%d_top" % i] = r, top
        G["bwd%d_meta" % i] = np.array([PH, sr, B, C, H, W], np.int64)
        G["bwd%d_scale" % i] = np.float32(scale)
        G["bwd%d_grad" % i] = ref.roi_align_backward_ref(top, r, (B, C, H, W), PH, PH, scale, sr)
    return G


def pickle_recipe(ref_model, flags):
    """(blob name, flat parameter name or '' for a zero blob, BGR flag) of every blob of a Detectron pickle for this configuration."""
    from utils.utils import parse_th_to_caffe2
    rows = []
    for k in ref_model.model.state_dict().keys():                            # trunk: torchvision name -> caffe2 blob name
        if 'running' in k or 'fc' in k:
            continue
        if 'num_batches' in k:
            rows.append((parse_th_to_caffe2(k.split('.')), '', False))       # the reference's loader (detector.py:300-304) expects this blob
            continue
        rows.append((parse_th_to_caffe2(k.split('.')), "model." + k, k == 'conv1.weight'))

    def put(wn, bn, name):
        rows.extend([(wn, name + ".weight", False), (bn, name + ".bias", False)])
    put('bbox_pred_w', 'bbox_pred_b', 'bbox_head'); put('cls_score_w', 'cls_score_b', 'classif_head')
    if flags["rpn"]:
        sfx = '_fpn2' if flags["fpn"] else ''
        put('conv_rpn%s_w' % sfx, 'conv_rpn%s_b' % sfx, 'rpn.conv_rpn')
        put('rpn_cls_logits%s_w' % sfx, 'rpn_cls_logits%s_b' % sfx, 'rpn.rpn_cls_prob')
        put('rpn_bbox_pred%s_w' % sfx, 'rpn_bbox_pred%s_b' % sfx, 'rpn.rpn_bbox_pred')
    if flags["mask"]:
        put('conv5_mask_w', 'conv5_mask_b', 'mask_head.transposed_conv'); put('mask_fcn_logits_w', 'mask_fcn_logits_b', 'mask_head.classif_logits')
        if flags["fpn"]:
            for i in range(1, 5):
                put('_[mask]_fcn%d_w' % i, '_[mask]_fcn%d_b' % i, 'mask_head.conv_head.fcn%d' % i)
    if flags["fpn"]:
        for i, l in enumerate(FPN['fpn_layers']):
            kc = parse_th_to_caffe2((l + '.' + list(getattr(ref_model.model, l).state_dict().keys())[-1]).split('.'))
            kc = kc[:kc.rfind("_")]
            suffix = '_sum_lateral' if i < 3 else '_sum'
            put('fpn_inner_' + kc + suffix + '_w', 'fpn_inner_' + kc + suffix + '_b', 'conv_body.fpn_lateral.%d' % i)
            put('fpn_' + kc + '_sum_w', 'fpn_' + kc + '_sum_b', 'conv_body.fpn_output.%d' % i)
        put('fc6_w', 'fc6_b', 'conv_head.fc6'); put('fc7_w', 'fc7_b', 'conv_head.fc7')
    return rows


def pickle_golden():
    import torchvision.models as models
    from model.detector import detector as ref_detector
    from utils.utils import parse_th_to_caffe2
    G = {}
    for arch in ("resnet50", "resnet101"):
        keys = [k for k in getattr(models, arch)().state_dict().keys() if not ('running' in k or 'fc' in k or 'num_batches' in k)]
        G["names_%s_keys" % arch] = np.array(keys)
        G["names_%s_blobs" % arch] = np.array([parse_th_to_caffe2(k.split('.')) for k in keys])
    tmp = tempfile.mkdtemp()
    for name, (kw, flags) in sorted(CONFIGS.items()):
        P = net.synthetic_params("resnet50", **flags)
        ref_kw = dict(kw, roi_feature_channels=1024) if flags["fpn"] else kw   # the FPN notebooks rely on the pickle to resize the 2048-wide default heads
        rows = pickle_recipe(ref_detector(**ref_kw), flags)
        blobs = {}
        for blob, src, bgr in rows:
            w = P[src].numpy() if src else np.zeros((), np.float32)
            blobs[blob] = w[:, (2, 1, 0), :, :].copy() if bgr else w
        pkl = os.path.join(tmp, name + ".pkl")
        with open(pkl, "wb") as f:
            pickle.dump({'blobs': blobs}, f, protocol=2)
        sd = ref_detector(detector_pkl_file=pkl, **kw).state_dict()          # exactly the notebook's cell 7
        for k, v in P.items():
            assert torch.equal(sd[k], v), "reference loader: " + k           # the synthetic pickle round-trips through the reference
        G[name + "_blob"] = np.array([r[0] for r in rows])
        G[name + "_src"] = np.array([r[1] for r in rows])
        G[name + "_bgr"] = np.array([r[2] for r in rows])
        G[name + "_keys"] = np.array(sorted(P))
        G[name + "_sha1"] = np.array([sha1(sd[k]) for k in sorted(P)])
        os.remove(pkl)
    os.rmdir(tmp)
    return G


if __name__ == "__main__":
    rs.install()
    for fname, G in (("crosscheck_golden.npz", crosscheck()), ("pickle_golden.npz", pickle_golden())):
        np.savez_compressed(os.path.join(OUT, fname), **G)
        print(fname, os.path.getsize(os.path.join(OUT, fname)) // 1024, "KiB")
