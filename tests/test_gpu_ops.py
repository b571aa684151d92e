"""GPU parity tests of the stand-alone operators, called through the C ABI (detectorch_b200/_lib.py ->
include/detectorch_b200.h), against the oracle and the committed golden vectors."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def dev(built):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def G():
    g = dict(np.load(os.path.join(GOLD, "ops_golden.npz")))
    g.update(np.load(os.path.join(GOLD, "roialign_golden.npz")))
    return g


def _boxes(rng, n, W=1216, H=800):
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    w = np.exp(rng.uniform(np.log(16), np.log(600), n)); a = np.exp(rng.uniform(-0.7, 0.7, n))
    b = np.stack([cx - w * np.sqrt(a) / 2, cy - w / np.sqrt(a) / 2, cx + w * np.sqrt(a) / 2, cy + w / np.sqrt(a) / 2], 1)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, W - 1); b[:, 1::2] = np.clip(b[:, 1::2], 0, H - 1)
    return b.astype(np.float32)


# ------------------------------------------------------------------------------- RoIAlign
def test_roi_align_golden_bit_exact(dev, G):
    from detectorch_b200 import ops
    f, r = torch.from_numpy(G["roi_feat"]).to(dev), torch.from_numpy(G["roi_rois"]).to(dev)
    for (p, sr, s) in [(7, 2, 16), (14, 2, 16), (14, 0, 16), (7, 0, 32)]:
        out = ops.roi_align_forward_nchw(f, r, p, p, 1. / s, sr).cpu().numpy()
        assert np.array_equal(out, G["roi_out_p%d_sr%d_s%d" % (p, sr, s)]), (p, sr, s)
    out4 = ops.roi_align_forward_nchw(f[:1].contiguous(), r[:, 1:].contiguous(), 7, 7, 1 / 16., 2).cpu().numpy()
    assert np.array_equal(out4, G["roi_out_4col"])


def test_roi_align_reference_launcher_symbol(dev, G):
    """The exact extern "C" symbol of the reference (roi_align_forward_cuda_kernel.h:7-19), raw pointers + stream."""
    from detectorch_b200 import _lib
    f, r = torch.from_numpy(G["roi_feat"]).to(dev), torch.from_numpy(G["roi_rois"]).to(dev)
    out = torch.zeros((r.size(0), f.size(1), 7, 7), device=dev)
    ok = _lib.lib().launch_roi_align_forward_cuda(out.numel(), f.data_ptr(), r.data_ptr(), 1 / 16., f.size(1), f.size(2), f.size(3), 7, 7, 2,
                                                  out.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert ok == 1
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), G["roi_out_p7_sr2_s16"])


def test_roi_align_random_vs_oracle_and_layouts(dev):
    from detectorch_b200 import ops
    from oracle import ref
    rng = np.random.RandomState(3)
    f = rng.randn(2, 32, 50, 68).astype(np.float32)
    r = np.hstack([rng.randint(0, 2, (500, 1)).astype(np.float32), _boxes(rng, 500, 1088, 800)])
    r[:5, 1:] = [[-100, -100, -50, -50], [2000, 2000, 2100, 2100], [5, 5, 5, 5], [0, 0, 1087, 799], [500, 400, 499, 399]]
    for (p, sr) in ((7, 2), (14, 0), (14, 2)):
        want = ref.roi_align_forward(f, r, p, p, 1 / 16., sr)
        got = ops.roi_align_forward_nchw(torch.from_numpy(f).to(dev), torch.from_numpy(r).to(dev), p, p, 1 / 16., sr).cpu().numpy()
        assert np.array_equal(got, want)
        fn = torch.from_numpy(f).permute(0, 2, 3, 1).contiguous().to(dev)
        got2 = ops.roi_align_forward_nhwc([fn], [1 / 16.], torch.from_numpy(r).to(dev), None, p, p, sr).permute(0, 3, 1, 2).cpu().numpy()
        assert np.array_equal(got2, want)
    # empty input
    assert ops.roi_align_forward_nchw(torch.from_numpy(f).to(dev), torch.zeros((0, 5), device=dev), 7, 7, 1 / 16., 2).shape == (0, 32, 7, 7)


def test_roi_align_fast_path_matches_exact(dev, G):
    """The separable / FMA fast kernel (sampling_ratio 2) agrees with the bit-exact kernel within fp32 re-association;
    other sampling ratios are forwarded to the exact kernel."""
    from detectorch_b200 import ops
    rng = np.random.RandomState(11)
    f = torch.from_numpy(rng.randn(2, 64, 50, 68).astype(np.float32)).to(dev)
    r = np.hstack([rng.randint(0, 2, (3000, 1)).astype(np.float32), _boxes(rng, 3000, 1088, 800)])
    r[:4, 1:] = [[-100, -100, -50, -50], [5, 5, 5, 5], [0, 0, 1087, 799], [1080, 790, 1200, 900]]
    r = torch.from_numpy(r).to(dev)
    for p in (7, 14):
        exact = ops.roi_align_forward_nchw(f, r, p, p, 1 / 16., 2)
        fast = ops.roi_align_forward_nchw_fast(f, r, p, p, 1 / 16., 2)          # 50x68 map: shared-memory-resident variant
        assert float((exact - fast).abs().max()) < 2e-5
    # a map too large for the shared-memory-resident variant (100x136 cells) takes the gather variant; ragged RoI counts
    fb = torch.from_numpy(rng.randn(2, 16, 100, 136).astype(np.float32)).to(dev)
    for n in (1, 7, 129, 3000):
        for (ff, sc) in ((f, 1 / 16.), (fb, 1 / 8.)):
            exact = ops.roi_align_forward_nchw(ff, r[:n].contiguous(), 7, 7, sc, 2)
            fast = ops.roi_align_forward_nchw_fast(ff, r[:n].contiguous(), 7, 7, sc, 2)
            assert float((exact - fast).abs().max()) < 2e-5
    r4 = r[:, 1:].contiguous()                                                   # 4-column RoIs (batch index 0 implied)
    assert float((ops.roi_align_forward_nchw(f[:1], r4, 7, 7, 1 / 16., 2) - ops.roi_align_forward_nchw_fast(f[:1], r4, 7, 7, 1 / 16., 2)).abs().max()) < 2e-5
    assert torch.equal(ops.roi_align_forward_nchw_fast(f, r, 14, 14, 1 / 16., 0), ops.roi_align_forward_nchw(f, r, 14, 14, 1 / 16., 0))
    gf, gr = torch.from_numpy(G["roi_feat"]).to(dev), torch.from_numpy(G["roi_rois"]).to(dev)
    assert np.abs(ops.roi_align_forward_nchw_fast(gf[:, :4].contiguous(), gr, 7, 7, 1 / 16., 2).cpu().numpy() - G["roi_out_p7_sr2_s16"][:, :4]).max() < 1e-5


def test_roi_align_mirror_module_and_errors(dev):
    from detectorch_b200.model.roi_align import RoIAlign, RoIAlignFunction
    from oracle import ref
    rng = np.random.RandomState(4)
    f = rng.randn(1, 8, 20, 30).astype(np.float32)
    r4 = _boxes(rng, 40, 480, 320)
    out = RoIAlign(7, 7, 1 / 16., 2)(torch.from_numpy(f).to(dev), torch.from_numpy(r4).to(dev))
    assert np.array_equal(out.cpu().numpy(), ref.roi_align_forward(f, r4, 7, 7, 1 / 16., 2))
    with pytest.raises(TypeError):
        RoIAlignFunction.apply(torch.from_numpy(f).to(dev), torch.from_numpy(r4), 7, 7, 1 / 16., 2)     # device mismatch, roi_align.py:43-44


def test_roi_align_backward(dev):
    """launch_roi_align_backward_cuda (the reference's exported symbol) through the mirror's autograd Function: agrees with the
    gradient of torchvision's CPU roi_align (aligned=False, the same caffe2 algorithm; its forward is bit-identical to the
    reference loop) within fp32 atomic-summation noise, for adaptive and fixed sampling ratios."""
    tv = pytest.importorskip("torchvision")
    from torchvision.ops import roi_align as tv_roi_align
    from detectorch_b200.model.roi_align import RoIAlignFunction
    rng = np.random.RandomState(9)
    f = torch.from_numpy(rng.randn(2, 6, 25, 38).astype(np.float32))
    r = torch.from_numpy(np.hstack([rng.randint(0, 2, (60, 1)).astype(np.float32), _boxes(rng, 60, 600, 400)]))
    for (p, sr) in ((7, 2), (14, 0), (5, 3)):
        go = torch.from_numpy(rng.randn(60, 6, p, p).astype(np.float32))
        fc = f.clone().requires_grad_(True)
        tv_roi_align(fc, r, (p, p), 1 / 16., sr, aligned=False).backward(go)
        fg = f.clone().to(dev).requires_grad_(True)
        out = RoIAlignFunction.apply(fg, r.to(dev), p, p, 1 / 16., sr)
        out.backward(go.to(dev))
        want = fc.grad.numpy()
        assert np.abs(fg.grad.cpu().numpy() - want).max() <= 2e-5 * max(1.0, np.abs(want).max())
    r4 = r[:, 1:].contiguous()                                  # 4-column RoIs
    from detectorch_b200 import ops
    g4 = ops.roi_align_backward_nchw(r4.to(dev), go.to(dev), (1, 6, 25, 38), 5, 5, 1 / 16., 3)
    r5 = torch.cat([torch.zeros(60, 1), r4], 1)
    g5 = ops.roi_align_backward_nchw(r5.to(dev), go.to(dev), (1, 6, 25, 38), 5, 5, 1 / 16., 3)
    assert float((g4 - g5).abs().max()) <= 1e-4


def test_roi_align_backward_deterministic_bit_exact(dev):
    """The atomics-free backward (dt_roi_align_backward_deterministic) equals the reference's single-threaded CPU backward BIT FOR BIT
    (golden vectors produced by the reference loop itself + fresh random cases against the oracle restatement), is bit-reproducible run
    to run, and the atomic twin (the reference GPU kernel's semantics) agrees with it to fp32 re-association."""
    from detectorch_b200 import ops
    from oracle import ref
    G = np.load(os.path.join(os.path.dirname(__file__), "golden", "roialign_bwd_golden.npz"))
    for i in range(int(G["n"])):
        PH, sr, B, C, H, W = [int(v) for v in G["meta%d" % i]]
        r, t = torch.from_numpy(G["rois%d" % i]).to(dev), torch.from_numpy(G["top%d" % i]).to(dev)
        got = ops.roi_align_backward_nchw_deterministic(r, t, (B, C, H, W), PH, PH, float(G["scale%d" % i]), sr)
        assert np.array_equal(got.cpu().numpy(), G["grad%d" % i]), i
        again = ops.roi_align_backward_nchw_deterministic(r, t, (B, C, H, W), PH, PH, float(G["scale%d" % i]), sr)
        assert torch.equal(got, again)
        atomic = ops.roi_align_backward_nchw(r, t, (B, C, H, W), PH, PH, float(G["scale%d" % i]), sr)
        assert float((atomic - got).abs().max()) <= 1e-5 * max(1.0, float(got.abs().max()))
    # the shapes of a Fast R-CNN training step: 512 heavily overlapping RoIs on a 50x76 map, 64 channels (each cell receives hundreds of terms)
    rng = np.random.RandomState(3)
    for (PH, sr, scale, C, H, W, R) in ((7, 2, 0.0625, 64, 50, 76, 512), (14, 0, 0.0625, 16, 50, 76, 128)):
        cx, cy = rng.uniform(200, 1000, R), rng.uniform(150, 650, R)
        wd, ht = rng.uniform(30, 500, R), rng.uniform(30, 400, R)
        r = np.stack([np.zeros(R), cx - wd / 2, cy - ht / 2, cx + wd / 2, cy + ht / 2], 1).astype(np.float32)
        top = rng.randn(R, C, PH, PH).astype(np.float32)
        want = ref.roi_align_backward(top, r, (1, C, H, W), PH, PH, scale, sr)
        got = ops.roi_align_backward_nchw_deterministic(torch.from_numpy(r).to(dev), torch.from_numpy(top).to(dev), (1, C, H, W), PH, PH, scale, sr)
        assert np.array_equal(got.cpu().numpy(), want)


def test_roi_align_training_step_is_reproducible(dev):
    """The training-side caller of the boundary (train_fast.py:115-194 shape: features -> RoIAlignFunction -> head -> loss -> backward -> SGD):
    torch autograd drives the same RoIAlignFunction the reference uses; with the deterministic backward two runs of three optimisation steps
    give bit-identical parameters, and the RoIAlign gradient inside the step equals the oracle's."""
    from detectorch_b200.model.roi_align import RoIAlignFunction, preprocess_rois
    from oracle import ref

    def run():
        torch.manual_seed(0)
        conv = torch.nn.Conv2d(3, 16, 3, padding=1).to(dev)
        head = torch.nn.Linear(16 * 7 * 7, 5).to(dev)
        torch.backends.cudnn.deterministic = True
        opt = torch.optim.SGD(list(conv.parameters()) + list(head.parameters()), lr=0.05)
        g = torch.Generator().manual_seed(1)
        img = torch.randn((1, 3, 40, 56), generator=g).to(dev)
        rng = np.random.RandomState(2)
        x1, y1 = rng.uniform(0, 120, 64), rng.uniform(0, 80, 64)
        rois = torch.from_numpy(np.stack([x1, y1, x1 + rng.uniform(8, 100, 64), y1 + rng.uniform(8, 70, 64)], 1).astype(np.float32)).to(dev)
        labels = torch.from_numpy(rng.randint(0, 5, 64)).to(dev)
        losses, saved = [], {}
        for step in range(3):
            opt.zero_grad()
            feat = conv(img)
            feat.retain_grad()
            pooled = RoIAlignFunction.apply(feat, preprocess_rois(rois), 7, 7, 0.25, 2)
            pooled.retain_grad()
            loss = torch.nn.functional.cross_entropy(head(pooled.reshape(64, -1)), labels)
            loss.backward()
            if step == 0:
                saved = {"gfeat": feat.grad.clone(), "gpool": pooled.grad.clone(), "rois": preprocess_rois(rois).clone()}
            opt.step()
            losses.append(float(loss))
        return losses, [p.detach().clone() for p in list(conv.parameters()) + list(head.parameters())], saved

    l1, p1, s1 = run()
    l2, p2, s2 = run()
    assert l1 == l2 and all(torch.equal(a, b) for a, b in zip(p1, p2))
    assert l1[-1] < l1[0]                                           # it trains
    want = ref.roi_align_backward(s1["gpool"].cpu().numpy(), s1["rois"].cpu().numpy(), (1, 16, 40, 56), 7, 7, 0.25, 2)
    assert np.array_equal(s1["gfeat"].cpu().numpy(), want)          # d(loss)/d(features) through RoIAlign == the reference CPU backward, bit for bit


def test_roi_align_full_size_properties(dev):
    """BASELINE configs[4] size (100k RoIs x 256 ch, 50x68 map): constant map -> every in-map bin equals the constant;
    linearity in the features."""
    from detectorch_b200 import ops
    rng = np.random.RandomState(5)
    R = 100000
    rois = torch.from_numpy(np.hstack([np.zeros((R, 1), np.float32), _boxes(rng, R, 1088, 800)])).to(dev)
    ones = torch.full((1, 256, 50, 68), 3.0, device=dev)
    out = ops.roi_align_forward_nchw(ones, rois, 7, 7, 1 / 16., 2)
    assert out.shape == (R, 256, 7, 7)
    assert float(out.max()) <= 3.0 + 1e-5 and float(out[:, 0].min()) >= 0.0
    inside = (rois[:, 3] < 1087 - 16) & (rois[:, 4] < 799 - 16)
    assert torch.all((out[inside] - 3.0).abs() < 1e-5)
    a = torch.randn((1, 256, 50, 68), device=dev); b = torch.randn((1, 256, 50, 68), device=dev)
    sub = rois[:2000].contiguous()
    lhs = ops.roi_align_forward_nchw(a + b, sub, 7, 7, 1 / 16., 2)
    rhs = ops.roi_align_forward_nchw(a, sub, 7, 7, 1 / 16., 2) + ops.roi_align_forward_nchw(b, sub, 7, 7, 1 / 16., 2)
    assert float((lhs - rhs).abs().max()) < 1e-4


# ------------------------------------------------------------------------------- NMS
def test_nms_golden_bit_exact(dev, G):
    from detectorch_b200 import ops
    for k in range(5):
        keep = ops.nms(torch.from_numpy(G["nms%d_dets" % k]).to(dev), float(G["nms%d_thresh" % k])).cpu().numpy()
        assert np.array_equal(keep, G["nms%d_keep" % k]), k
    assert ops.nms(torch.zeros((0, 5), device=dev), 0.5).numel() == 0


def test_nms_random_vs_oracle(dev):
    from detectorch_b200 import ops
    from detectorch_b200.utils import boxes as mirror
    from oracle import ref
    rng = np.random.RandomState(6)
    for n in (1, 2, 63, 64, 65, 129, 1000, 4097, 6000):
        d = np.hstack([_boxes(rng, n), rng.permutation(n).astype(np.float32)[:, None] / n])     # unique scores
        for t in (0.3, 0.5, 0.7):
            assert np.array_equal(ops.nms(torch.from_numpy(d).to(dev), t).cpu().numpy(), ref.nms(d, t)), (n, t)
    d = np.hstack([_boxes(rng, 500), rng.uniform(0, 1, (500, 1)).astype(np.float32)])
    assert np.array_equal(np.asarray(mirror.nms(d, 0.5)), ref.nms(d, 0.5))       # numpy-in / numpy-out mirror of boxes.nms
    assert mirror.nms(np.zeros((0, 5), np.float32), 0.5) == []


def test_nms_large_properties(dev):
    """20k boxes: idempotence (NMS of the survivors keeps everything) and kept ids are sorted ascending."""
    from detectorch_b200 import ops
    rng = np.random.RandomState(8)
    n = 20000
    d = torch.from_numpy(np.hstack([_boxes(rng, n), rng.permutation(n).astype(np.float32)[:, None] / n])).to(dev)
    keep = ops.nms(d, 0.5)
    assert torch.all(keep[1:] > keep[:-1])
    again = ops.nms(d[keep].contiguous(), 0.5)
    assert again.numel() == keep.numel()


# ------------------------------------------------------------------------------- conv / GEMM (tcgen05, 3xTF32)
def _conv_case(dev, N, Hh, Ww, Cin, Cout, k, pad, stride, res=False, up=False, relu=False, sig=0, passes=3, kind="tf32", force_block_n=0):
    from detectorch_b200 import ops
    g = torch.Generator().manual_seed(N * 1000 + Hh * 10 + Cin + Cout + k)
    x = torch.randn((N, Hh, Ww, Cin), generator=g)
    w = torch.randn((Cout, k, k, Cin), generator=g) * (2.0 / (k * k * Cin)) ** 0.5
    sc, sh = 0.5 + torch.rand((Cout,), generator=g), 0.1 * torch.randn((Cout,), generator=g)
    Ho, Wo = (Hh + 2 * pad - k) // stride + 1, (Ww + 2 * pad - k) // stride + 1
    R = torch.randn((N, Ho, Wo, Cout), generator=g) if res else None
    U = torch.randn((N, (Ho + 1) // 2, (Wo + 1) // 2, Cout), generator=g) if up else None
    y = torch.nn.functional.conv2d(x.double().permute(0, 3, 1, 2), w.double().permute(0, 3, 1, 2), stride=stride, padding=pad)
    y = y * sc.double().view(1, -1, 1, 1) + sh.double().view(1, -1, 1, 1)
    if res:
        y = y + R.double().permute(0, 3, 1, 2)
    if up:
        y = y + torch.nn.functional.interpolate(U.double().permute(0, 3, 1, 2), scale_factor=2, mode="nearest")[:, :, :Ho, :Wo]
    if relu:
        y = torch.relu(y)
    y = y.permute(0, 2, 3, 1).contiguous()
    if sig:
        y[..., :sig] = torch.sigmoid(y[..., :sig])
    got = ops.conv2d_nhwc(x.to(dev), w.reshape(Cout, -1).contiguous().to(dev), sc.to(dev), sh.to(dev), k, k, pad, stride,
                          residual=R.to(dev) if res else None, up_src=U.to(dev) if up else None, relu=relu, sigmoid_ch=sig, passes=passes,
                          kind=kind, force_block_n=force_block_n)
    err = (got.cpu().double() - y).abs().max().item()
    return err / max(1.0, y.abs().max().item())


@pytest.mark.parametrize("case", [
    (1, 1, 128, 64, 64, 1, 0, 1), (1, 1, 1000, 1024, 408, 1, 0, 1), (1, 20, 30, 64, 128, 3, 1, 1), (2, 25, 38, 256, 256, 3, 1, 1),
    (1, 50, 76, 256, 128, 1, 0, 2), (2, 25, 38, 128, 64, 1, 0, 2), (5, 14, 14, 256, 256, 3, 1, 1), (1, 1, 300, 12544, 1024, 1, 0, 1)])
def test_conv_3xtf32_matches_fp64_within_1e4(dev, case):
    # tolerance: 1e-4 of the tensor's max-abs (BASELINE north_star fp32 parity bar); 3xTF32 measures ~1e-6..1e-5
    assert _conv_case(dev, *case) < 1e-4


_CONV_CASES = [(1, 1, 128, 64, 64, 1, 0, 1), (1, 1, 1000, 1024, 408, 1, 0, 1), (1, 20, 30, 64, 128, 3, 1, 1), (2, 25, 38, 256, 256, 3, 1, 1),
               (1, 50, 76, 256, 128, 1, 0, 2), (2, 25, 38, 128, 64, 1, 0, 2), (5, 14, 14, 256, 256, 3, 1, 1), (1, 1, 300, 12544, 1024, 1, 0, 1)]


@pytest.mark.parametrize("case", _CONV_CASES)
def test_conv_3xf16_matches_fp64_within_1e4(dev, case):
    """The kind::f16 three-term product (fp16 hi/lo halves of both operands, fp32 accumulate) meets the same fp32 parity bar."""
    assert _conv_case(dev, *case, kind="f16") < 1e-4


def test_conv_f16_epilogues_tiles_and_range_flag(dev):
    from detectorch_b200 import ops
    assert _conv_case(dev, 1, 20, 30, 64, 256, 1, 0, 1, res=True, relu=True, kind="f16") < 1e-4
    assert _conv_case(dev, 2, 13, 19, 128, 64, 3, 1, 1, res=True, relu=True, kind="f16") < 1e-4
    assert _conv_case(dev, 1, 26, 38, 64, 256, 1, 0, 1, up=True, kind="f16") < 1e-4
    assert _conv_case(dev, 1, 25, 38, 256, 16, 1, 0, 1, sig=3, kind="f16") < 1e-4
    assert _conv_case(dev, 5, 14, 14, 256, 256, 3, 1, 1, kind="f16", force_block_n=-1) < 1e-4      # precise 128-wide tile
    assert _conv_case(dev, 5, 14, 14, 256, 256, 3, 1, 1, kind="f16", force_block_n=128) < 1e-4
    assert _conv_case(dev, 1, 1, 512, 2048, 256, 1, 0, 1, kind="f16") < 1e-4                         # K = 2048: cta_group::2 variant
    assert 1e-5 < _conv_case(dev, 1, 1, 256, 1024, 128, 1, 0, 1, passes=1, kind="f16") < 5e-3       # single fp16 pass: not fp32-accurate
    # fp16 has a 5-bit exponent: an activation of 1e5 raises the range flag, ordinary data does not
    x = torch.randn((1, 4, 32, 64), device=dev)
    w = torch.randn((64, 64), device=dev) * 0.1
    one, zero = torch.ones(64, device=dev), torch.zeros(64, device=dev)
    flag = torch.zeros((1,), dtype=torch.int32, device=dev)
    ops.conv2d_nhwc(x, w, one, zero, 1, 1, 0, 1, kind="f16", range_flag=flag)
    assert int(flag.item()) == 0
    x[0, 1, 7, 3] = 1.0e5
    ops.conv2d_nhwc(x, w, one, zero, 1, 1, 0, 1, kind="f16", range_flag=flag)
    assert int(flag.item()) == 1


def test_conv_epilogues(dev):
    assert _conv_case(dev, 1, 20, 30, 64, 256, 1, 0, 1, res=True, relu=True) < 1e-4
    assert _conv_case(dev, 2, 13, 19, 128, 64, 3, 1, 1, res=True, relu=True) < 1e-4
    assert _conv_case(dev, 1, 26, 38, 64, 256, 1, 0, 1, up=True) < 1e-4
    assert _conv_case(dev, 1, 25, 38, 256, 16, 1, 0, 1, sig=3) < 1e-4
    # single-pass TF32 is NOT fp32-accurate: this is why the product path runs 3 passes
    assert 1e-4 < _conv_case(dev, 1, 1, 256, 1024, 128, 1, 0, 1, passes=1) < 5e-3


# ------------------------------------------------------------------------------------------------ mask paste + RLE (8f rank 1)
def _segm_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "segm_golden.npz"))


def test_segm_golden(dev):
    """dt_segm_paste / dt_segm_rle against the fixtures produced by the reference's own segm_results (real cv2.resize)."""
    from detectorch_b200 import ops
    from detectorch_b200.utils import result_utils as ru
    S = _segm_golden()
    for tag, M in (("m28", 28), ("m14", 14)):
        masks, boxes, cls = S[tag + "_masks"], S[tag + "_boxes"], S[tag + "_cls"]
        im_h, im_w = [int(v) for v in S[tag + "_size"]]
        D, K = masks.shape[:2]
        want_bits = np.unpackbits(S[tag + "_pasted_bits"], axis=1)[:, :im_h * im_w].reshape(D, im_h, im_w)
        tm, tb, tc = torch.from_numpy(masks).to(dev), torch.from_numpy(boxes).to(dev), torch.from_numpy(cls).to(dev)
        pasted = ops.segm_paste(tm, tc, tb, im_h, im_w).cpu().numpy()
        assert np.array_equal(pasted, want_bits)
        counts, strings = ops.segm_rle(tm, tc, tb, im_h, im_w)
        assert [s.decode() for s in strings] == [str(x) for x in S[tag + "_rle"]]
        for d in range(D):
            assert np.array_equal(counts[d], ref_mod().rle_encode(want_bits[d]))
        # the mirror of result_utils.segm_results returns the reference's structure (device masks, no host copy of them)
        cls_boxes = [[] for _ in range(K)]
        for j in range(1, K):
            cls_boxes[j] = np.hstack([boxes[cls == j], np.ones((int((cls == j).sum()), 1), np.float32)])
        got = ru.segm_results(cls_boxes, tm, boxes, im_h, im_w, num_classes=K, M=M)
        want = ref_mod().segm_results(cls_boxes, masks, boxes, im_h, im_w, num_classes=K, M=M)
        assert got == want
        assert ru.segm_results(cls_boxes, masks, boxes, im_h, im_w, num_classes=K, M=M) == want      # numpy masks are accepted too


def ref_mod():
    from oracle import ref
    return ref


def test_segm_full_size_and_edges(dev):
    """800x1216 image, 100 detections (BASELINE headline shape): bit-exact against the oracle on a sample, and for every
    detection decode(counts) == pasted mask and sum(counts) == H*W; tiny runs_cap exercises the grow-and-redo path; no
    detections; class-agnostic masks."""
    from detectorch_b200 import ops
    ref = ref_mod()
    rng = np.random.RandomState(21)
    im_h, im_w, D, M = 800, 1216, 100, 28
    b = _boxes(rng, D, im_w, im_h)
    b[:6] = [[0, 0, im_w - 1, im_h - 1], [0, 0, 3, 3], [im_w - 9, im_h - 9, im_w - 1, im_h - 1], [600, 0, 620, im_h - 1], [0, 400, im_w - 1, 410],
             [100, 100, 113, 113]]
    yy, xx = np.mgrid[0:M, 0:M].astype(np.float32) / M
    masks = np.stack([np.clip(1 / (1 + np.exp(((xx - rng.uniform(.3, .7)) ** 2 + (yy - rng.uniform(.3, .7)) ** 2 - rng.uniform(.05, .2)) * 40))
                              + 0.2 * rng.randn(M, M), 0, 1) for _ in range(D)]).astype(np.float32)
    masks[0] = 1.0                                                      # the whole image set: runs touch every border
    tm, tb = torch.from_numpy(masks).to(dev), torch.from_numpy(b).to(dev)
    pasted = ops.segm_paste(tm, None, tb, im_h, im_w)
    counts, strings = ops.segm_rle(tm, None, tb, im_h, im_w, runs_cap=64)          # forces at least one regrow
    exp = ref.expand_boxes(b, (M + 2.0) / M).astype(np.int32)
    for d in range(D):
        assert int(counts[d].astype(np.int64).sum()) == im_h * im_w
        if d < 12:
            want = ref.paste_mask(masks[d], exp[d], im_h, im_w)
            assert np.array_equal(pasted[d].cpu().numpy(), want)
            assert np.array_equal(counts[d], ref.rle_encode(want))
            assert strings[d] == ref.rle_to_string(ref.rle_encode(want))
    # decode on the device side of the comparison: cumulative run ends -> parity bit per pixel, column-major
    for d in (0, 1, 2, 3, 4, 5, 17, 99):
        ends = torch.from_numpy(np.cumsum(counts[d].astype(np.int64))).to(dev)
        pos = torch.arange(im_h * im_w, device=dev)
        bit = (torch.searchsorted(ends, pos, right=True) & 1).to(torch.uint8).reshape(im_w, im_h).t()
        assert torch.equal(bit, pasted[d])
    assert ops.segm_rle(tm[:0], None, tb[:0], im_h, im_w) == ([], [])
    nd = torch.tensor([3], dtype=torch.int32, device=dev)
    c3, s3 = ops.segm_rle(tm[:8], None, tb[:8], im_h, im_w, num_dets=nd)
    assert [len(c) for c in c3[3:]] == [0] * 5 and s3[:3] == strings[:3]


# ------------------------------------------------------------------------------------------------ image pre-processing (8f rank 3)
def test_prep_image_golden_and_full_size(dev):
    """dt_prep_image == the reference's prep_im_for_blob + im_list_to_blob bit for bit (fixtures generated by the reference with the
    real cv2), and at the headline size (a 480x640 image -> 3x800x1088 blob) against the oracle; mirror preprocess_sample."""
    from detectorch_b200.utils import blob as B
    from detectorch_b200.utils.preprocess_sample import preprocess_sample
    P = np.load(os.path.join(os.path.dirname(__file__), "golden", "prep_golden.npz"))
    for i, (h, w, ts, ms) in enumerate(P["cases"]):
        blob, s = B.image_to_blob(P["im%d" % i], target_size=int(ts), max_size=int(ms), fpn_on=True)
        assert s == float(P["scale%d" % i])
        assert np.array_equal(blob.cpu().numpy(), P["blob%d" % i])
        ims, scales = B.prep_im_for_blob(P["im%d" % i], target_sizes=[int(ts)], max_size=int(ms))
        assert np.array_equal(B.im_list_to_blob(ims, fpn_on=True).cpu().numpy(), P["blob%d" % i])
    ref = ref_mod()
    rng = np.random.RandomState(2)
    for (h, w) in ((480, 640), (375, 1242), (1600, 2000)):
        im = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
        ims, scales = ref.prep_im_for_blob(im)
        want = ref.im_list_to_blob(ims, fpn_on=True)
        sample = preprocess_sample(fpn_on=True)({'image': im, 'dbentry': {'boxes': np.zeros((0, 4), np.float32)}})
        assert sample['scaling_factors'] == scales[0] and tuple(sample['original_im_size'].tolist()) == (h, w, 3)
        assert sample['image'].is_cuda and np.array_equal(sample['image'].cpu().numpy(), want)


def test_lib_overlay_modules(built):
    """The lib/ overlay a reference maintainer puts ahead of the reference's lib/ on sys.path (INTEGRATION.md): `cppcuda_cffi.roialign`
    with the cffi calling convention (caller allocates and zeroes the output / grad_input), `model.detector`, `model.roi_align`,
    `utils.result_utils`, `utils.preprocess_sample` -- run in a fresh interpreter so the module names cannot collide."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import sys, numpy as np, torch
sys.path.insert(0, %r + "/lib")
sys.path.insert(0, %r)
import cppcuda_cffi.roialign as roialign
from model.detector import detector
from model.roi_align import RoIAlign
from utils.result_utils import postprocess_output, segm_results
from utils.preprocess_sample import preprocess_sample
from detectorch_b200 import ops
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
f = torch.randn((1, 8, 20, 30), generator=g).to(dev)
r = torch.tensor([[0, 10., 12., 200., 150.], [0, 50., 60., 90., 300.], [0, 0., 0., 479., 319.]]).to(dev)
out = torch.zeros((3, 8, 7, 7), device=dev)
assert roialign.roi_align_forward_cuda(f, r, out, 7, 7, 1 / 16., 2) == 1
assert torch.equal(out, ops.roi_align_forward_nchw(f, r, 7, 7, 1 / 16., 2))
go = torch.randn((3, 8, 7, 7), generator=g).to(dev)
gi = torch.zeros((1, 8, 20, 30), device=dev)
assert roialign.roi_align_backward_cuda(r, go, gi, 7, 7, 1 / 16., 2) == 1
want = ops.roi_align_backward_nchw(r, go, (1, 8, 20, 30), 7, 7, 1 / 16., 2)
assert float((gi - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
try:
    roialign.roi_align_forward_cpu(f.cpu(), r.cpu(), out.cpu(), 7, 7, 1 / 16., 2)
    raise SystemExit("the overlay must not have a CPU path")
except RuntimeError:
    pass
# the torch-0.4 flavour: a module named `roialign` with the pybind entry points (callee allocates; AT_CHECK -> RuntimeError)
sys.modules.pop("roialign", None)
import roialign as pyb
assert pyb.__file__.startswith(%r + "/lib")
o2 = pyb.roi_align_forward_cuda(f, r, 7, 7, 1 / 16., 2)
assert torch.equal(o2, out)
g2 = pyb.roi_align_backward_cuda(r, go, 1, 8, 20, 30, 7, 7, 1 / 16., 2)
assert float((g2 - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
for bad in (lambda: pyb.roi_align_forward_cuda(f[0], r, 7, 7, 1 / 16., 2), lambda: pyb.roi_align_forward_cuda(f, r[:, :4].contiguous(), 7, 7, 1 / 16., 2),
            lambda: pyb.roi_align_forward_cuda(f.permute(0, 1, 3, 2), r, 7, 7, 1 / 16., 2)):
    try:
        bad()
        raise SystemExit("AT_CHECK condition not enforced")
    except RuntimeError:
        pass
print("OVERLAY OK")
''' % (root, root, root)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OVERLAY OK" in out.stdout, out.stderr[-2000:]
