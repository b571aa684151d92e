"""Generates tests/golden/*.npz by RUNNING THE REFERENCE ITSELF (imported unmodified from
/root/reference through oracle/reference_shim.py, RoIAlign through the reference's own compiled
loop, NMS through its own Cython module).  Only runnable where /root/reference exists; the
fixtures are committed so the GPU box (which has no reference tree) can pin against them.

    python tests/golden/make_golden.py
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import CPU_BITWISE_ENV  # noqa: E402
from oracle import reference_shim as rs  # noqa: E402
from oracle import network as net  # noqa: E402
from oracle import ref as oref  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def boxes(rng, n, W=1216, H=800):
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    w = np.exp(rng.uniform(np.log(16), np.log(600), n))
    a = np.exp(rng.uniform(-0.7, 0.7, n))
    bw, bh = w * np.sqrt(a), w / np.sqrt(a)
    b = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, W - 1)
    b[:, 1::2] = np.clip(b[:, 1::2], 0, H - 1)
    return b.astype(np.float32)


def main():
    rs.install()
    import utils.boxes as box_utils
    import utils.result_utils as ru
    from utils.generate_anchors import generate_anchors
    from utils.multilevel_rois import add_multilevel_rois_for_test
    from model.generate_proposals import GenerateProposals
    from model.collect_and_distribute_fpn_rpn_proposals import CollectAndDistributeFpnRpnProposals
    from model.detector import detector

    rng = np.random.RandomState(1234)
    G = {}
    # ---- anchors (generate_anchors.py known-answer: the comment table at :26-51 minus 1)
    for i in range(5):
        G["anchors_fpn%d" % (i + 2)] = generate_anchors(stride=4. * 2 ** i, sizes=(32 * 2 ** i,), aspect_ratios=(0.5, 1, 2))
    G["anchors_c4"] = generate_anchors(stride=16, sizes=(32, 64, 128, 256, 512), aspect_ratios=(0.5, 1, 2))
    G["anchors_matlab"] = generate_anchors(stride=16, sizes=(128, 256, 512), aspect_ratios=(0.5, 1, 2))
    # ---- NMS
    for k, (n, t) in enumerate([(1, 0.5), (50, 0.3), (300, 0.5), (1000, 0.7), (2000, 0.5)]):
        d = np.hstack([boxes(rng, n), rng.uniform(0, 1, (n, 1)).astype(np.float32)])
        if n == 300:                       # duplicates and nested boxes
            d[100:150, :4] = d[:50, :4]
            d[150:200, :4] = d[:50, :4] + 1.0
        G["nms%d_dets" % k] = d
        G["nms%d_thresh" % k] = np.float32(t)
        G["nms%d_keep" % k] = np.asarray(box_utils.nms(d, t), dtype=np.int64)
    # ---- RoIAlign through the reference's compiled CPU loop
    feat = rng.randn(2, 6, 25, 38).astype(np.float32)
    rois = np.hstack([rng.randint(0, 2, (60, 1)).astype(np.float32), boxes(rng, 60, 600, 400)])
    rois[0, 1:] = [-30, -30, -5, -5]          # fully outside
    rois[1, 1:] = [100, 100, 100, 100]        # degenerate -> forced 1x1
    rois[2, 1:] = [0, 0, 599, 399]            # whole map
    G["roi_feat"], G["roi_rois"] = feat, rois
    for (p, sr, sc) in [(7, 2, 1 / 16.), (14, 2, 1 / 16.), (14, 0, 1 / 16.), (7, 0, 1 / 32.)]:
        G["roi_out_p%d_sr%d_s%d" % (p, sr, int(1 / sc))] = oref.roi_align_forward_ref(feat, rois, p, p, sc, sr)
    G["roi_out_4col"] = oref.roi_align_forward_ref(feat[:1], rois[:, 1:], 7, 7, 1 / 16., 2)
    # ---- GenerateProposals (reference module) on synthetic RPN maps, two levels
    for k, (H, W, scale, size, pre) in enumerate([(25, 38, 1 / 32., 256, 1000), (50, 76, 1 / 16., 128, 600)]):
        cls = torch.sigmoid(2.0 * torch.from_numpy(rng.randn(1, 3, H, W).astype(np.float32)))
        box = torch.from_numpy((0.3 * rng.randn(1, 12, H, W)).astype(np.float32))
        gp = GenerateProposals(spatial_scale=scale, anchor_sizes=(size,), rpn_pre_nms_top_n=pre, rpn_post_nms_top_n=300)
        pr, sc = gp(cls, box, 800, 1216, 1.0)
        G["gp%d_cls" % k], G["gp%d_box" % k] = cls.numpy(), box.numpy()
        G["gp%d_cfg" % k] = np.array([H, W, 1 / scale, size, pre, 300], dtype=np.float64)
        G["gp%d_props" % k], G["gp%d_scores" % k] = pr.numpy(), sc.numpy()
    # ---- collect and distribute
    rl = [torch.from_numpy(boxes(rng, n)) for n in (300, 200, 100, 50, 7)]
    sl = [torch.from_numpy(rng.uniform(0, 1, (len(r), 1)).astype(np.float32)) for r in rl]
    cd = CollectAndDistributeFpnRpnProposals(spatial_scales=[0.25, 0.125, 0.0625, 0.03125])
    import model.collect_and_distribute_fpn_rpn_proposals as cdm
    cdm_collect = cdm.collect

    def collect400(a, b, train):        # exercise the top-N cut with a small N as well
        return cdm_collect(a, b, train)
    per, restore = cd(rl, sl)
    for i in range(5):
        G["cd_in_rois%d" % i], G["cd_in_scores%d" % i] = rl[i].numpy(), sl[i].numpy()
    for i in range(4):
        G["cd_out_rois%d" % i] = per[i].numpy()
    G["cd_restore"] = np.asarray(restore, dtype=np.int64)
    # ---- postprocess_output
    R = 400
    pr_rois = torch.from_numpy(boxes(rng, R))
    logits = 2.0 * rng.randn(R, 81).astype(np.float32)
    logits[:, 0] += 2.0
    cls_scores = torch.softmax(torch.from_numpy(logits), 1)
    deltas = torch.from_numpy((0.5 * rng.randn(R, 324)).astype(np.float32))
    sf, bf, cb = ru.postprocess_output(pr_rois, torch.tensor([1.0]), torch.tensor([[800., 1216.]]), cls_scores, deltas)
    G["pp_rois"], G["pp_cls"], G["pp_deltas"] = pr_rois.numpy(), cls_scores.numpy(), deltas.numpy()
    G["pp_scores_final"], G["pp_boxes_final"] = sf, bf
    G["pp_counts"] = np.array([len(cb[j]) for j in range(81)], dtype=np.int64)
    bm = add_multilevel_rois_for_test({'rois': bf.copy()}, 'rois')
    G["pp_mask_restore"] = bm['rois_idx_restore_int32']
    for l in range(2, 6):
        G["pp_mask_rois_fpn%d" % l] = bm['rois_fpn%d' % l]
    # the RoIAlign forward vectors go to a file of their own so that each fixture stays under 1 MB
    np.savez_compressed(os.path.join(OUT, "roialign_golden.npz"), **{k: v for k, v in G.items() if k.startswith("roi_")})
    np.savez_compressed(os.path.join(OUT, "ops_golden.npz"), **{k: v for k, v in G.items() if not k.startswith("roi_")})
    # the detector fixture is bit-exact only under the pinned torch-CPU configuration that tests/test_oracle.py checks it with
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--detector"], env=dict(os.environ, **CPU_BITWISE_ENV))
    for f in ("ops_golden.npz", "roialign_golden.npz", "net_golden_r50fpn_128x160.npz"):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")


def detector_golden():
    """The reference detector end to end (tiny image, synthetic weights shared by name)."""
    rs.install()
    import utils.result_utils as ru
    from utils.multilevel_rois import add_multilevel_rois_for_test
    from model.detector import detector
    torch.set_num_threads(1)
    m = detector(arch='resnet50', conv_body_layers=['conv1', 'bn1', 'relu', 'maxpool', 'layer1', 'layer2', 'layer3', 'layer4'],
                 conv_head_layers='two_layer_mlp', fpn_layers=['layer1', 'layer2', 'layer3', 'layer4'], fpn_extra_lvl=True,
                 roi_height=7, roi_width=7, roi_spatial_scale=[0.25, 0.125, 0.0625, 0.03125], roi_sampling_ratio=2,
                 use_rpn_head=True, use_mask_head=True, mask_head_type='1up4convs', roi_feature_channels=1024)
    P = net.synthetic_params('resnet50')
    sd = m.state_dict()
    for k, v in P.items():
        sd[k].copy_(v)
    img = net.synthetic_image(1, 128, 160)
    with torch.no_grad():
        cls, box, rois_o, feats = m(img, scaling_factor=1.0)
    sf, bf, cb = ru.postprocess_output(rois_o, torch.tensor(1.0), torch.tensor([[128., 160.]]), cls, box)
    bm = add_multilevel_rois_for_test({'rois': bf * 1.0}, 'rois')
    lst = [torch.FloatTensor(bm['rois_fpn%d' % l]) if len(bm['rois_fpn%d' % l]) > 0 else None for l in range(2, 6)]
    with torch.no_grad():
        masks = m.mask_head(feats, lst, torch.FloatTensor(bm['rois_idx_restore_int32']).long())
    N = {"cls_score": cls.numpy(), "bbox_pred": box.numpy(), "rois": rois_o.numpy(), "scores_final": sf, "boxes_final": bf,
         "counts": np.array([len(cb[j]) for j in range(81)], dtype=np.int64)}
    for i, f in enumerate(feats):
        N["P%d_sub" % (i + 2)] = f.numpy()[:, ::16, ::2, ::2].copy()       # channel / spatial subsample keeps the file small
        N["P%d_absmax" % (i + 2)] = np.float32(f.abs().max().item())
    cls_of_det = np.concatenate([np.full(len(cb[j]), j) for j in range(1, 81)])
    N["det_classes"] = cls_of_det.astype(np.int64)
    N["masks_own_class"] = masks.numpy()[np.arange(len(cls_of_det)), cls_of_det][:, ::2, ::2].copy()
    np.savez_compressed(os.path.join(OUT, "net_golden_r50fpn_128x160.npz"), **N)


if __name__ == "__main__":
    detector_golden() if "--detector" in sys.argv else main()
