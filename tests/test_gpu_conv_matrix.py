"""Every instantiation of the tcgen05 conv kernel, driven one layer at a time through dt_conv2d_spec / dt_conv2d_stem, against an fp64
reference at the shapes where tiled TMA kernels go wrong: ragged output tiles, several images per box, work-item counts around the
74-pair persistent loop, channel counts that are not a multiple of the tile, K-split, transposed-conv scatter, fp16 plane input and
output, channel-slice input, wider output buffers, NaN sentinels around every output, and inputs of small magnitude.

Tolerance, per element, from the arithmetic of the three-term product with a truncating fp32 accumulate:

    |got - ref| <= |scale| * S * (C0 + C1 * L) * 2^-23  +  C2 * 2^-23 * (|ref| + |residual|)

S is the fp64 conv of |x| with |w|.  L is the truncating-accumulate chain length the plan implies: MMA steps per accumulator (2 per
32-element k-block on the f16 pipe, 4 on the tf32 pipe), times 3 for the merged accumulator, over 3 for rotating accumulators.  Every
truncating step costs at most one ulp of the running sum (<= S * 2^-23): C1 = 1.  C0 covers the split residuals and the dropped
lo x lo term of the operands and the RN adds of the epilogue: 3 * 2^-22 relative on the f16 pipe (fp16 hi / lo rounded to nearest), so
C0 = 8; 3 * 2^-20 on the tf32 pipe (the MMA truncates both pieces to 10 mantissa bits), so C0 = 24.  Single-pass products (passes=1)
keep only hi x hi: C0 = 2^15.  C2 covers the final roundings of the scale / shift / residual epilogue: C2 = 2.

test_bound_detects_kernel_mutations shows on the CPU that the bound catches a dropped cross term, a single pass, a skipped k-block and
tile-edge addressing mistakes by >= 10x at short K.  It stops catching a dropped cross term or a single pass where the chain term
C1 * L outgrows them: with the merged accumulator at K = 2304 they come to about 0.5 and 0.7 of the bound.  The long-K cases (the
K-split mask-head layers, K = 12544) rely on the plain `< 1e-4 of max-abs` parity bar for those, which every case asserts as well.

The kernel switches are read once per process, so the matrix runs again in one subprocess per setting (tests/conv_matrix_check.py);
every case asserts the plan it is meant to reach under the default settings."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 2.0 ** -23
C0_F16, C0_TF32, C0_ONE_PASS, C1, C2 = 8.0, 24.0, 2.0 ** 15, 1.0, 2.0
SWITCHES = ("DT_CONV_MMA", "DT_CONV_WS", "DT_CONV_SLOTS", "DT_CONV_NARROW1", "DT_CONV_HALO", "DT_CONV_RES_RING", "DT_CONV_PDL",
            "DT_CONV_MERGE_KB", "DT_CONV_RING_KB", "DT_CONV_RING2_KB")


def chain_length(plan, passes=3):
    """truncating-accumulate steps of the longest accumulator chain of a tile"""
    ksteps = 2 if plan["kind"] == 1 else 4
    kb = plan["num_kb"]
    if plan["nmain"] == 0:
        return 3 * kb * ksteps if passes == 3 else kb * ksteps
    if plan["nmain"] == 3:
        return -(-kb // 3) * ksteps
    return kb * ksteps


def c0_of(kind, passes=3):
    """kind: the plan's kind field (1 = f16 pipe, 0 = tf32 pipe)"""
    return C0_ONE_PASS if passes != 3 else (C0_F16 if kind == 1 else C0_TF32)


def bound(S, ref, scale, L, residual=None, c0=C0_F16):
    """elementwise bound (numpy / torch fp64, NHWC; scale broadcasts over the last axis)"""
    res = abs(residual) if residual is not None else 0.0
    return abs(scale) * S * (c0 + C1 * L) * EPS + C2 * EPS * (abs(ref) + res)


# ============================================================================================ CPU: the bound's own sensitivity
def _trunc32(v):
    """fp64 -> fp32 rounding toward zero (the tensor core's accumulate)"""
    f = v.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(v)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def _split16(a):
    h = a.astype(np.float16)
    return h, (a - h.astype(np.float32)).astype(np.float16)


def emulate_f16_gemm(A, B, nmain=1, passes=3, drop_lh=False, skip_kb=None):
    """A [M,K] fp32 x B [K,N] fp32 as the kind::f16 kernel computes it: fp16 hi/lo splits, one MMA = 16 k-elements with a truncating fp32
    accumulate, main term rotating over nmain accumulators by 32-element k-block (0: main and cross terms merged), RN adds at the end."""
    ah, al = _split16(A)
    bh, bl = _split16(B)
    M, K = A.shape
    nm = max(nmain, 1)
    acc = [np.zeros((M, B.shape[1]), np.float32) for _ in range(nm)]
    accx = np.zeros((M, B.shape[1]), np.float32)
    for k0 in range(0, K, 16):
        kb = k0 // 32
        if kb == skip_kb:
            continue
        s = slice(k0, k0 + 16)
        a_h, a_l, b_h, b_l = (t[s if t.shape[0] == K else (slice(None), s)].astype(np.float64) for t in (ah.T, al.T, bh, bl))
        main = a_h.T @ b_h
        cross = (0.0 if drop_lh else a_l.T @ b_h) + a_h.T @ b_l
        i = kb % nm
        if passes != 3:
            acc[i] = _trunc32(acc[i] + main)
        elif nmain == 0:
            acc[0] = _trunc32(_trunc32(_trunc32(acc[0] + (0.0 if drop_lh else a_l.T @ b_h)) + a_h.T @ b_l) + main)
        else:
            accx = _trunc32(accx + cross)
            acc[i] = _trunc32(acc[i] + main)
    out = acc[0]
    for a in acc[1:]:
        out = (out + a).astype(np.float32)
    if passes == 3 and nmain != 0:
        out = (out + accx).astype(np.float32)
    return out


def _im2col(x, k, pad):
    """x [N,H,W,C] -> [N*H*W, k*k*C] (stride 1, same padding), tap-major like the kernel's K"""
    N, H, W, C = x.shape
    xp = np.pad(x, ((0, 0), (pad, pad), (pad, pad), (0, 0)))
    cols = [xp[:, fy:fy + H, fx:fx + W, :] for fy in range(k) for fx in range(k)]
    return np.concatenate(cols, axis=3).reshape(N * H * W, k * k * C)


def _ratio(got, ref, S, L, residual=None):
    return float(np.max(np.abs(got.astype(np.float64) - ref) / bound(S, ref, 1.0, L, residual)))


@pytest.mark.parametrize("K,nmain", [(32, 1), (64, 0), (576, 3), (576, 1), (2304, 0), (2304, 1)])
def test_bound_holds_for_the_emulated_product(K, nmain):
    """A numpy emulation of the kind::f16 three-term product meets the bound on the matrix's shapes."""
    rng = np.random.RandomState(K + nmain)
    A = rng.randn(256, K).astype(np.float32)
    B = (rng.randn(K, 64) * np.sqrt(2.0 / K)).astype(np.float32)
    ref = A.astype(np.float64) @ B.astype(np.float64)
    S = np.abs(A).astype(np.float64) @ np.abs(B).astype(np.float64)
    L = chain_length({"kind": 1, "num_kb": K // 32, "nmain": nmain})
    r = _ratio(emulate_f16_gemm(A, B, nmain), ref, S, L)
    assert r < 0.5, r


def test_bound_detects_kernel_mutations():
    """Each plausible kernel mistake exceeds the bound by >= 10x on at least one case, so the GPU assertions can fail."""
    worst = {}
    for K in (32, 64, 576):
        rng = np.random.RandomState(K)
        A = rng.randn(256, K).astype(np.float32)
        B = (rng.randn(K, 64) * np.sqrt(2.0 / K)).astype(np.float32)
        ref = A.astype(np.float64) @ B.astype(np.float64)
        S = np.abs(A).astype(np.float64) @ np.abs(B).astype(np.float64)
        for nmain in (0, 1, 3):
            L = chain_length({"kind": 1, "num_kb": K // 32, "nmain": nmain})
            for name, kw in (("drop A_l*B_h", dict(drop_lh=True)), ("one pass", dict(passes=1)), ("skip a k-block", dict(skip_kb=K // 32 - 1))):
                worst[name] = max(worst.get(name, 0.0), _ratio(emulate_f16_gemm(A, B, nmain, **kw), ref, S, L))
    # tile-edge addressing on a 3x3 conv of a 2 x 12 x 20 map with 8-pixel-wide tiles: a tap read one pixel off at the tile's right edge,
    # and a residual pixel taken from the neighbouring tile
    rng = np.random.RandomState(7)
    N, H, W, C, Co, wbox = 2, 12, 20, 32, 64, 8
    x = rng.randn(N, H, W, C).astype(np.float32)
    w = (rng.randn(9 * C, Co) * np.sqrt(2.0 / (9 * C))).astype(np.float32)
    res = rng.randn(N, H, W, Co)
    cols = _im2col(x, 3, 1)
    ref = (cols.astype(np.float64) @ w.astype(np.float64)).reshape(N, H, W, Co)
    S = (np.abs(cols).astype(np.float64) @ np.abs(w).astype(np.float64)).reshape(N, H, W, Co)
    L = chain_length({"kind": 1, "num_kb": 9, "nmain": 1})
    got = emulate_f16_gemm(cols, w, 1).reshape(N, H, W, Co).astype(np.float64)
    assert _ratio(got, ref, S, L) < 0.5
    edge = np.arange(W) % wbox == wbox - 1
    shifted = np.concatenate([x[:, :, 1:], np.zeros_like(x[:, :, :1])], axis=2)
    tap = slice(5 * C, 6 * C)                         # filter tap (1, 2): the right-hand neighbour
    delta = (_im2col(shifted, 3, 1)[:, tap].astype(np.float64) - cols[:, tap]) @ w[tap].astype(np.float64)
    mut = got + np.where(edge[None, None, :, None], delta.reshape(N, H, W, Co), 0.0)
    worst["tap off at the right edge"] = _ratio(mut, ref, S, L)
    ref_r = ref + res
    got_r = got + res
    nb = np.concatenate([res[:, :, 1:], res[:, :, :1]], axis=2)
    mut_r = got_r + np.where(edge[None, None, :, None], nb - res, 0.0)
    assert _ratio(got_r, ref_r, S, L, res) < 0.5
    worst["residual from the neighbouring tile"] = _ratio(mut_r, ref_r, S, L, res)
    for name, r in worst.items():
        assert r > 10.0, (name, r)


# ============================================================================================ GPU matrix
def _default_switches():
    return not any(k in os.environ for k in SWITCHES)


def _rand(g, shape, scale=1.0):
    return torch.randn(shape, generator=g, dtype=torch.float32) * scale


def _sentinel_buffer(shape_nhwc, pix_stride, dev, dtype=torch.float32, margin_pix=37):
    """an output view [N,H,W,C] inside a NaN-filled allocation: margin_pix pixels before and after, pix_stride - C spare channels"""
    N, H, W, C = shape_nhwc
    npix = N * H * W
    buf = torch.full(((npix + 2 * margin_pix) * pix_stride,), float("nan"), dtype=dtype, device=dev)
    view = buf[margin_pix * pix_stride:(margin_pix + npix) * pix_stride].view(N, H, W, pix_stride)[..., :C]
    return buf, view


def _stray_free(buf, view):
    """every sentinel outside the view survived (the view itself holds no NaN: _check asserts it)"""
    return int(torch.isnan(buf).sum()) == buf.numel() - view.numel() and not bool(torch.isnan(view).any())


def _ref_conv(x, w, scale, shift, k, pad, stride, res=None, up=None, relu=False, sig=0):
    """fp64 reference (NHWC in/out) and S = conv(|x|, |w|)"""
    xd, wd = x.double().permute(0, 3, 1, 2), w.double().permute(0, 3, 1, 2)
    y = torch.nn.functional.conv2d(xd, wd, stride=stride, padding=pad)
    S = torch.nn.functional.conv2d(xd.abs(), wd.abs(), stride=stride, padding=pad).permute(0, 2, 3, 1)
    y = y * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1)
    addend = None
    if res is not None:
        addend = res.double()
    if up is not None:
        u = torch.nn.functional.interpolate(up.double().permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
        addend = u[:, :, :y.size(2), :y.size(3)].permute(0, 2, 3, 1)
    if addend is not None:
        y = y + addend.permute(0, 3, 1, 2)
    if relu:
        y = torch.relu(y)
    y = y.permute(0, 2, 3, 1).contiguous()
    if sig:
        y[..., :sig] = torch.sigmoid(y[..., :sig])
    return y, S, addend


def _check(got, ref, S, scale, plan, addend=None, sig=0, passes=3, L=None):
    """-> (max error / bound, max error / max(1, max|ref|)); sigmoid channels are checked against the bound of their argument"""
    got = got.double()
    L = chain_length(plan, passes) if L is None else L
    b = bound(S, ref, scale.double().view(1, 1, 1, -1), L, addend, c0_of(plan["kind"], passes))
    if sig:
        b[..., :sig] = b[..., :sig] * 0.25 + 8 * EPS        # sigmoid' <= 1/4, plus the rounding of expf and the division
    err = (got - ref).abs()
    assert not torch.isnan(got).any(), "NaN in the output"
    return float((err / b).max()), float(err.max() / max(1.0, float(ref.abs().max())))


def _rel_maxabs(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max())


# A case: dict(name, N, H, W, Cin, Cout, k, pad, stride, + options); `expect` = plan fields under the default switch settings.
def matrix_cases():
    C = []

    def add(name, **kw):
        kw.setdefault("kind", "f16")
        C.append(dict(name=name, **kw))
    # ---- ragged tiles / several images per box / channel counts (fp32 input, f16 and tf32 kinds)
    for kind in ("f16", "tf32"):
        add("1x1 cin32 cout4 7x7", kind=kind, N=3, H=7, W=7, Cin=32, Cout=4, k=1, pad=0, stride=1, ragged=True, expect=dict(block_n=64, num_kb=1))
        add("1x1 cout16 sig3 14x14", kind=kind, N=5, H=14, W=14, Cin=64, Cout=16, k=1, pad=0, stride=1, sig=3, ragged=True,
            expect=dict(block_n=64))
        add("3x3 cout76 13x19 relu", kind=kind, N=3, H=13, W=19, Cin=64, Cout=76, k=3, pad=1, stride=1, relu=True, ragged=True,
            expect=dict(block_n=128))
        add("3x3 cout84 precise", kind=kind, N=2, H=11, W=23, Cin=64, Cout=84, k=3, pad=1, stride=1, precise=True,
            expect=dict(block_n=128, nmain=3))
        add("1x1 s2 cout408 odd", kind=kind, N=2, H=25, W=39, Cin=128, Cout=408, k=1, pad=0, stride=2, sig=33, expect=dict(block_n=256))
        add("3x3 cout256 14x14 nomerge", kind=kind, N=5, H=14, W=14, Cin=256, Cout=256, k=3, pad=1, stride=1, no_merge=True, relu=True,
            expect=dict(block_n=256, nmain=1))
        add("3x3 cout256 merged res", kind=kind, N=2, H=13, W=19, Cin=64, Cout=256, k=3, pad=1, stride=1, res=True, relu=True,
            expect=dict(block_n=256, nmain=0))
        add("1x1 up2x odd crop", kind=kind, N=1, H=25, W=37, Cin=64, Cout=256, k=1, pad=0, stride=1, up=True, expect=dict(block_n=256))
        add("gemm K12544 cout1024", kind=kind, N=1, H=1, W=40, Cin=12544, Cout=1024, k=1, pad=0, stride=1,
            expect=dict(block_n=256, nmain=1, num_kb=392))
    # ---- the residual ring forms (K <= 16 k-blocks, 256 wide, RES_TILE): ring 3 with one slot, ring 2 with one slot
    add("ring3 res K256", N=2, H=13, W=19, Cin=256, Cout=256, k=1, pad=0, stride=1, res=True, relu=True, expect=dict(ring=3, slots=1))
    add("ring2 res K512 ragged", N=1, H=25, W=37, Cin=512, Cout=1024, k=1, pad=0, stride=1, res=True, relu=True, xslice=544,
        expect=dict(ring=2, slots=1))
    # ---- 64-wide: one accumulator at K <= 256, three rotating above; channel-slice input, wider output buffer
    add("64w K64 one acc", N=2, H=9, W=33, Cin=64, Cout=64, k=1, pad=0, stride=1, relu=True, expect=dict(block_n=64, nmain=1, two_sm=0))
    add("64w K576 xslice ywide", N=1, H=21, W=27, Cin=64, Cout=64, k=3, pad=1, stride=1, xslice=96, ywide=72, relu=True,
        expect=dict(block_n=64, nmain=3))
    # ---- work distribution: one M-tile (the surplus tile only), odd M-tile count, < 74 pairs, 74, 74 + 1 and 2 x 74 work items
    add("one M-tile", N=1, H=1, W=100, Cin=64, Cout=256, k=1, pad=0, stride=1, expect=dict(m_pairs=1, tiles_w=1))
    add("74 pairs", N=1, H=1, W=148 * 128, Cin=64, Cout=256, k=1, pad=0, stride=1, expect=dict(m_pairs=74, n_tiles=1, grid=148))
    add("75 pairs odd tiles", N=1, H=1, W=149 * 128, Cin=64, Cout=256, k=1, pad=0, stride=1, expect=dict(m_pairs=75, grid=148))
    add("148 items", N=1, H=1, W=148 * 128, Cin=32, Cout=512, k=1, pad=0, stride=1, expect=dict(m_pairs=74, n_tiles=2))
    add("149 items", N=1, H=1, W=297 * 128 + 10, Cin=32, Cout=256, k=1, pad=0, stride=1, sig=15, expect=dict(m_pairs=149, n_tiles=1))
    # ---- the persistent loop wrap per kernel family: 149 = 2 x 74 + 1 work items, so every CTA pair runs two or three items (TMEM
    #      accumulator buffers, pipeline / ring / staging barrier phases and resident weights carried from one item to the next)
    P149 = 297 * 128                              # 297 M-tiles of 128 pixels -> 149 pairs
    wrap = dict(m_pairs=149, n_tiles=1)
    add("ring3 149 items", N=1, H=1, W=P149, Cin=256, Cout=256, k=1, pad=0, stride=1, res=True, relu=True, expect=dict(wrap, ring=3))
    add("ring2 149 items", N=1, H=1, W=P149, Cin=512, Cout=256, k=1, pad=0, stride=1, res=True, relu=True, expect=dict(wrap, ring=2))
    for kind in ("f16", "tf32"):
        add("64w one acc 149 items", kind=kind, N=1, H=1, W=P149, Cin=64, Cout=64, k=1, pad=0, stride=1, relu=True, expect=dict(wrap, block_n=64))
        add("64w 3x3 rotating 149 items", kind=kind, N=1, H=1, W=P149, Cin=64, Cout=64, k=3, pad=1, stride=1,
            expect=dict(wrap, block_n=64, nmain=3))
        add("128w 149 items", kind=kind, N=1, H=1, W=P149, Cin=64, Cout=128, k=1, pad=0, stride=1, relu=True, expect=dict(wrap, block_n=128, nmain=1))
        add("128w precise 149 items", kind=kind, N=1, H=1, W=P149, Cin=64, Cout=128, k=1, pad=0, stride=1, precise=True,
            expect=dict(wrap, block_n=128, nmain=3))
        add("256w merged 149 items", kind=kind, N=1, H=1, W=P149, Cin=32, Cout=256, k=1, pad=0, stride=1, expect=dict(wrap, block_n=256, nmain=0))
    for cout in (64, 128):                        # 176 x 216 = 11 x 27 halo tiles of 8 x 16
        add("halo%d 149 items" % cout, N=1, H=176, W=216, Cin=64, Cout=cout, k=3, pad=1, stride=1, planes_in=True, relu=True,
            expect=dict(wrap, halo=1, hbox=16))
    add("stem planes 149 items", N=1, H=351, W=431, stem=True, planes_in=True, expect=dict(wrap, halo=2, ws=1))
    # ---- single-pass products (passes=1) and the op's automatic fp16 input multiplier
    for kind in ("f16", "tf32"):
        add("gemm passes1", kind=kind, N=1, H=1, W=300, Cin=1024, Cout=128, k=1, pad=0, stride=1, passes=1, expect=dict(block_n=128))
        add("64w passes1", kind=kind, N=2, H=13, W=19, Cin=64, Cout=64, k=3, pad=1, stride=1, passes=1, relu=True, expect=dict(block_n=64))
    add("1x1 auto multiplier", N=2, H=13, W=19, Cin=128, Cout=256, k=1, pad=0, stride=1, xm="auto", relu=True)
    add("stem fp32 auto multiplier", N=1, H=37, W=29, stem=True, xm="auto", expect=dict(halo=0))
    # ---- halo 3x3 over fp16 planes: W = 10 (the minimum), W = 9 (falls back to the per-tap form), Wo % 8 in {1, 4, 7}, H < 16
    for cout, bn in ((64, 64), (128, 128)):
        add("halo%d W10" % bn, N=2, H=20, W=10, Cin=64, Cout=cout, k=3, pad=1, stride=1, planes_in=True, relu=True, expect=dict(halo=1, wbox=8))
        add("halo%d W9 fallback" % bn, N=2, H=20, W=9, Cin=64, Cout=cout, k=3, pad=1, stride=1, planes_in=True, expect=dict(halo=0))
        for W in (17, 12, 15):
            add("halo%d W%d" % (bn, W), N=3, H=19, W=W, Cin=64, Cout=cout, k=3, pad=1, stride=1, planes_in=True, relu=True,
                expect=dict(halo=1, hbox=16))
        for H, hb in ((8, 8), (5, 4), (3, 2), (1, 1)):
            add("halo%d H%d" % (bn, H), N=16 // hb + 1, H=H, W=13, Cin=64, Cout=cout, k=3, pad=1, stride=1, planes_in=True, relu=True,
                expect=dict(halo=1, hbox=hb, nbox=16 // hb))
    # ---- plane output, plane-out -> plane-in chain, K-split, transposed conv
    add("plane out 1x1", N=2, H=13, W=19, Cin=64, Cout=64, k=1, pad=0, stride=1, relu=True, planes_out=True, expect=dict(block_n=64))
    add("plane out 256", N=1, H=11, W=29, Cin=128, Cout=256, k=1, pad=0, stride=1, relu=True, planes_out=True, expect=dict(block_n=256))
    add("chain planes", N=2, H=14, W=21, Cin=64, Cout=64, k=1, pad=0, stride=1, relu=True, chain=True)
    for kind in ("f16", "tf32"):
        add("ksplit 5+4", kind=kind, N=5, H=14, W=14, Cin=256, Cout=256, k=3, pad=1, stride=1, relu=True, ksplit=5,
            expect=dict(block_n=256, num_kb=40))
        add("ksplit 1+8", kind=kind, N=3, H=14, W=14, Cin=256, Cout=256, k=3, pad=1, stride=1, relu=True, ksplit=1, no_merge=True)
        add("deconv scatter", kind=kind, N=3, H=14, W=14, Cin=256, Cout=256, k=1, pad=0, stride=1, relu=True, deconv=True)
    # ---- the stem: HALO = 2 over fp16 planes (with and without WS, nmain 1 or 3), H1 / W1 not multiples of 16 / 8, H1 < 16 (no halo)
    add("stem planes ragged", N=2, H=45, W=51, stem=True, planes_in=True, expect=dict(halo=2, ws=1, nmain=1, wbox=8, hbox=16))
    add("stem planes H1<16", N=2, H=25, W=40, stem=True, planes_in=True, expect=dict(halo=0))
    add("stem fp32 ragged", N=3, H=37, W=29, stem=True, expect=dict(halo=0))
    add("stem tf32", kind="tf32", N=1, H=33, W=47, stem=True, expect=dict(halo=0))
    return C


def _split_planes(x):
    h = x.half()
    return h, (x - h.float()).half()


def _case_multiplier(c):
    """the fp16 input multiplier a case passes: 1 (what the engine runs) unless the case asks for the op's automatic choice"""
    xm = c.get("xm", 1.0)
    return None if xm == "auto" else xm


def run_case(c, dev, scale_exp=0):
    """-> dict(name, ratio, rel, plan, rows, ok, ...); raises AssertionError on a failed property other than the numeric bound"""
    from detectorch_b200 import ops
    g = torch.Generator().manual_seed(sum(map(ord, c["name"])) * 7 + c["N"])
    if c.get("stem"):
        return _run_stem(c, dev, g)
    N, H, W, Cin, Cout, k, pad, stride = (c[f] for f in ("N", "H", "W", "Cin", "Cout", "k", "pad", "stride"))
    kind, sig, relu = c["kind"], c.get("sig", 0), c.get("relu", False)
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    xs = 2.0 ** scale_exp
    xfull = _rand(g, (N, H, W, c.get("xslice", Cin)), xs)
    x = xfull[..., :Cin]
    w = _rand(g, (Cout, k, k, Cin), (2.0 / (k * k * Cin)) ** 0.5)
    sc, sh = 0.5 + torch.rand((Cout,), generator=g), 0.1 * torch.randn((Cout,), generator=g)
    if c.get("plain"):
        sc, sh = torch.ones((Cout,)), torch.zeros((Cout,))
    R = _rand(g, (N, Ho, Wo, Cout)) if c.get("res") else None
    U = _rand(g, (N, (Ho + 1) // 2, (Wo + 1) // 2, Cout)) if c.get("up") else None
    xh = xl = None
    if c.get("planes_in"):
        xh, xl = _split_planes(x.contiguous())
        x = xh.float() + xl.float()                  # what the kernel sees
    out = {"name": c["name"], "kind": kind}
    wk = w.reshape(Cout, -1).contiguous().to(dev)
    passes = c.get("passes", 3)
    common = dict(passes=passes, kind=kind, precise=c.get("precise", False), no_merge=c.get("no_merge", False), return_plan=True)
    xm = _case_multiplier(c)
    if xm is not None:
        common["x_multiplier"] = xm
    flag = torch.zeros((1,), dtype=torch.int32, device=dev)
    if c.get("deconv"):
        return _run_deconv(c, dev, g, x, xs, out)
    if c.get("chain"):
        return _run_chain(c, dev, g, x, out)
    if c.get("ksplit"):
        return _run_ksplit(c, dev, g, x, w, sc, sh, out, common)
    ref, S, addend = _ref_conv(x, w, sc, sh, k, pad, stride, R, U, relu, sig)
    xd = xfull.to(dev)[..., :Cin] if not c.get("planes_in") else xh.to(dev)
    kw = dict(common, residual=R.to(dev) if R is not None else None, up_src=U.to(dev) if U is not None else None, relu=relu, sigmoid_ch=sig,
              range_flag=flag, x_lo=xl.to(dev) if xl is not None else None)
    results = []
    for rep in range(2):                                  # determinism: the same launch twice is bit-identical
        if c.get("planes_out"):
            bh, yh = _sentinel_buffer((N, Ho, Wo, Cout), Cout, dev, torch.float16)
            bl, yl = _sentinel_buffer((N, Ho, Wo, Cout), Cout, dev, torch.float16)
            (_, _), plan = ops.conv2d_nhwc(xd, wk, sc.to(dev), sh.to(dev), k, k, pad, stride, out=yh, out_lo=yl, **kw)
            torch.cuda.synchronize()
            for b, v in ((bh, yh), (bl, yl)):
                assert _stray_free(b, v), "stray write outside a plane output"
            hi, lo = yh.cpu(), yl.cpu()
            got = hi.double() + lo.double()
            e = torch.frexp(hi.float())[1]
            ulp = torch.where(hi == 0, torch.full_like(hi, 2.0 ** -24, dtype=torch.float32), torch.ldexp(torch.ones_like(e, dtype=torch.float32), e - 11))
            ulp = ulp.clamp(min=2.0 ** -24)
            assert bool((lo.float().abs() <= ulp / 2).all()), "|lo| > ulp(hi) / 2"
            tie = lo.float().abs() == ulp / 2               # hi + lo exactly half-way: fp16 rounding goes to the even neighbour
            assert torch.equal(hi[~tie], got.float().half()[~tie]), "hi != fp16_rn(hi + lo)"
            results.append(torch.cat([hi.view(torch.int16).flatten(), lo.view(torch.int16).flatten()]))
        else:
            buf, y = _sentinel_buffer((N, Ho, Wo, Cout), c.get("ywide", Cout), dev)
            _, plan = ops.conv2d_nhwc(xd, wk, sc.to(dev), sh.to(dev), k, k, pad, stride, out=y, **kw)
            torch.cuda.synchronize()
            assert _stray_free(buf, y), "stray write outside the output view"
            got = y.cpu()
            results.append(got.contiguous().view(torch.int32).flatten())
    assert torch.equal(results[0], results[1]), "two identical launches differ"
    assert int(flag.item()) == 0, "range flag raised on ordinary data"
    out["ratio"], out["rel"] = _check(got, ref, S, sc, plan, addend, sig, passes)
    out["rel_maxabs"] = _rel_maxabs(got, ref)
    out["plan"] = plan
    return out


def _run_ksplit(c, dev, g, x, w, sc, sh, out, common):
    """taps [0, t) with scale / shift, then taps [t, 9) adding the first result through RES_TILE on its own output buffer (the engine's
    mask-head form): meets the bound of the unsplit conv"""
    from detectorch_b200 import ops
    N, H, W, Cin, Cout = (c[f] for f in ("N", "H", "W", "Cin", "Cout"))
    t = c["ksplit"]
    ref, S, _ = _ref_conv(x, w, sc, sh, 3, 1, 1, relu=True)
    buf, y = _sentinel_buffer((N, H, W, Cout), Cout, dev)
    wk = w.reshape(Cout, -1).contiguous().to(dev)
    xd, scd = x.to(dev), sc.to(dev)
    common = {k: v for k, v in common.items() if k != "return_plan"}
    # both layers prepared first (weight split, scale folding), then issued back to back: the second reads the first's output through
    # RES_TILE with no other work between the two kernels (under DT_CONV_PDL=1 it overlaps the first's tail)
    first = ops.conv2d_prepare(xd, wk, scd, sh.to(dev), 3, 3, 1, 1, out=y, tap0=0, ntaps=t, **common)
    second = ops.conv2d_prepare(xd, wk, scd, torch.zeros_like(scd), 3, 3, 1, 1, out=y, residual=y, relu=True, tap0=t, ntaps=9 - t, **common)
    p1 = first.launch()
    p2 = second.launch()
    torch.cuda.synchronize()
    assert _stray_free(buf, y)
    full = dict(p1, num_kb=p1["num_kb"] + p2["num_kb"], nmain=p1["nmain"])
    out["ratio"], out["rel"] = _check(y.cpu(), ref, S, sc, p1, L=chain_length(full))
    out["plan"] = p1
    out["rows2"] = p2["instantiation"]
    return out


def _run_deconv(c, dev, g, x, xs, out):
    """ConvTranspose2d(k=2, s=2) as 4 GEMMs, each scattered with out_step = 2 into the [N, 2H, 2W, Cout] map"""
    from detectorch_b200 import ops
    N, H, W, Cin, Cout, kind = (c[f] for f in ("N", "H", "W", "Cin", "Cout", "kind"))
    Wt = _rand(g, (Cin, Cout, 2, 2), (1.0 / Cin) ** 0.5)
    sc, sh = 0.5 + torch.rand((Cout,), generator=g), 0.1 * torch.randn((Cout,), generator=g)
    xd64 = x.double().permute(0, 3, 1, 2)
    ref = torch.nn.functional.conv_transpose2d(xd64, Wt.double(), stride=2)
    S = torch.nn.functional.conv_transpose2d(xd64.abs(), Wt.double().abs(), stride=2).permute(0, 2, 3, 1)
    ref = torch.relu(ref * sc.double().view(1, -1, 1, 1) + sh.double().view(1, -1, 1, 1)).permute(0, 2, 3, 1)
    buf, y = _sentinel_buffer((N, 2 * H, 2 * W, Cout), Cout, dev)
    xd = x.to(dev)
    gemms = [ops.conv2d_prepare(xd, Wt[:, :, ij // 2, ij % 2].t().contiguous().to(dev), sc.to(dev), sh.to(dev), 1, 1, 0, 1, out=y,
                                out_map=(2 * H, 2 * W, 2, ij // 2, ij % 2), relu=True, kind=kind, x_multiplier=1.0) for ij in range(4)]
    plan = [gm.launch() for gm in gemms][-1]
    torch.cuda.synchronize()
    assert _stray_free(buf, y)
    out["ratio"], out["rel"] = _check(y.cpu(), ref, S, sc, plan)
    out["plan"] = plan
    return out


def _run_chain(c, dev, g, x, out):
    """plane output of one layer -> plane input of a 3x3 halo layer (the bottleneck's conv1 -> conv2 hand-over)"""
    from detectorch_b200 import ops
    N, H, W, Cin, Cout = (c[f] for f in ("N", "H", "W", "Cin", "Cout"))
    w1 = _rand(g, (Cout, 1, 1, Cin), (2.0 / Cin) ** 0.5)
    w2 = _rand(g, (Cout, 3, 3, Cout), (2.0 / (9 * Cout)) ** 0.5)
    s1, b1 = 0.5 + torch.rand((Cout,), generator=g), 0.1 * torch.randn((Cout,), generator=g)
    s2, b2 = 0.5 + torch.rand((Cout,), generator=g), 0.1 * torch.randn((Cout,), generator=g)
    yh = torch.empty((N, H, W, Cout), dtype=torch.float16, device=dev)
    yl = torch.empty_like(yh)
    _, p1 = ops.conv2d_nhwc(x.to(dev), w1.reshape(Cout, -1).contiguous().to(dev), s1.to(dev), b1.to(dev), 1, 1, 0, 1, out=yh, out_lo=yl,
                            relu=True, kind="f16", return_plan=True, x_multiplier=1.0)
    y2, p2 = ops.conv2d_nhwc(yh, w2.reshape(Cout, -1).contiguous().to(dev), s2.to(dev), b2.to(dev), 3, 3, 1, 1, x_lo=yl, relu=True,
                             kind="f16", return_plan=True)
    torch.cuda.synchronize()
    mid = yh.cpu().double() + yl.cpu().double()
    ref1, S1, _ = _ref_conv(x, w1, s1, b1, 1, 0, 1, relu=True)
    r1, _ = _check(mid, ref1, S1, s1, p1)
    ref2, S2, _ = _ref_conv(mid.float(), w2, s2, b2, 3, 1, 1, relu=True)
    r2, rel2 = _check(y2.cpu(), ref2, S2, s2, p2)
    out["ratio"], out["rel"], out["plan"], out["rows2"] = max(r1, r2), rel2, p1, p2["instantiation"]
    assert p2["halo"] == 1 or not _default_switches()
    return out


def _pack_stem(img, planes):
    """NCHW image -> zero-bordered NHWC4 [B,Hp,Wp,4] (border 3, channel 3 = 0), or its fp16 hi / lo planes [2,B,Hp,Wp,4]"""
    B, _, H, W = img.shape
    H1, W1 = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    Hp, Wp = max(H + 6, 2 * H1 + 5), max(W + 6, 2 * W1 + 6)
    Wp += Wp % 2
    x4 = torch.zeros((B, Hp, Wp, 4))
    x4[:, 3:3 + H, 3:3 + W, :3] = img.permute(0, 2, 3, 1)
    if planes:
        h, l = _split_planes(x4)
        return torch.stack([h, l]), H1, W1
    return x4, H1, W1


def _run_stem(c, dev, g):
    from detectorch_b200 import ops
    B, H, W, kind = c["N"], c["H"], c["W"], c["kind"]
    img = _rand(g, (B, 3, H, W), 50.0)
    if c.get("planes_in"):
        h, l = _split_planes(img)
        img = h.float() + l.float()
    Wc = _rand(g, (64, 3, 7, 7), (2.0 / 147) ** 0.5)
    sc, sh = 0.5 + torch.rand((64,), generator=g), 0.1 * torch.randn((64,), generator=g)
    wm = torch.zeros((64, 7, 8, 4))
    wm[:, :, :7, :3] = Wc.permute(0, 2, 3, 1)
    wm = wm.reshape(64, 224).contiguous()
    x4, H1, W1 = _pack_stem(img, c.get("planes_in", False))
    ref = torch.nn.functional.conv2d(img.double(), Wc.double(), stride=2, padding=3)
    S = torch.nn.functional.conv2d(img.double().abs(), Wc.double().abs(), stride=2, padding=3).permute(0, 2, 3, 1)
    ref = torch.relu(ref * sc.double().view(1, -1, 1, 1) + sh.double().view(1, -1, 1, 1)).permute(0, 2, 3, 1)
    buf, y = _sentinel_buffer((B, H1, W1, 64), 64, dev)
    flag = torch.zeros((1,), dtype=torch.int32, device=dev)
    _, plan = ops.conv2d_stem(x4.to(dev), wm.to(dev), sc.to(dev), sh.to(dev), H1, W1, kind=kind, range_flag=flag, out=y, return_plan=True,
                              x_multiplier=_case_multiplier(c))
    torch.cuda.synchronize()
    assert _stray_free(buf, y)
    assert int(flag.item()) == 0
    out = {"name": c["name"], "kind": kind, "plan": plan}
    out["ratio"], out["rel"] = _check(y.cpu(), ref, S, sc, plan)
    return out


def check_result(c, r):
    assert r["ratio"] <= 1.0, "%s: error %.3g x the bound" % (c["name"], r["ratio"])
    bar = 5e-3 if c.get("passes", 3) == 1 else 1e-4          # a single pass is not fp32-accurate (why the product path runs 3)
    assert r["rel"] < bar, "%s: %.3g of max-abs" % (c["name"], r["rel"])
    assert r["plan"]["instantiation"] >= 0
    p = r["plan"]
    if c.get("ragged"):                 # several images per box with N, Ho or Wo not a multiple of the box
        assert p["nbox"] > 1 and (c["N"] % p["nbox"] or p["ho"] % p["hbox"] or p["wo"] % p["wbox"]), p
    if _default_switches():
        for f, v in c.get("expect", {}).items():
            assert r["plan"][f] == v, "%s: plan %s = %s, expected %s" % (c["name"], f, r["plan"][f], v)


def range_flag_checks(dev):
    """range_flag: raised by one |a| = 65504 or NaN input element in the last, partial tile and by a plane-output epilogue producing
    |y| >= 65504"""
    from detectorch_b200 import ops
    g = torch.Generator().manual_seed(5)
    N, H, W, Cin, Cout = 3, 7, 9, 64, 64
    w = _rand(g, (Cout, Cin), 0.1).to(dev)
    one, zero = torch.ones(Cout, device=dev), torch.zeros(Cout, device=dev)
    for bad in (65504.0, float("nan")):
        x = _rand(g, (N, H, W, Cin)).to(dev)
        x[N - 1, H - 1, W - 1, Cin - 1] = bad
        flag = torch.zeros((1,), dtype=torch.int32, device=dev)
        _, plan = ops.conv2d_nhwc(x, w, one, zero, 1, 1, 0, 1, kind="f16", range_flag=flag, return_plan=True)
        assert plan["tiles_w"] * plan["wbox"] > W or plan["tiles_h"] * plan["hbox"] > H or plan["tiles_n"] * plan["nbox"] > N
        assert int(flag.item()) == 1, bad
    x = _rand(g, (N, H, W, Cin)).to(dev)
    yh = torch.empty((N, H, W, Cout), dtype=torch.float16, device=dev)
    flag = torch.zeros((1,), dtype=torch.int32, device=dev)
    ops.conv2d_nhwc(x, w, one, zero, 1, 1, 0, 1, kind="f16", range_flag=flag, out=yh, out_lo=torch.empty_like(yh))
    assert int(flag.item()) == 0
    ops.conv2d_nhwc(x, w, one * 1e6, zero, 1, 1, 0, 1, kind="f16", range_flag=flag, out=yh, out_lo=torch.empty_like(yh))
    assert int(flag.item()) == 1


def pdl_chain_check(dev):
    """two dependent layers launched back to back, no sync between them (under DT_CONV_PDL=1 the second overlaps the first's tail)"""
    from detectorch_b200 import ops
    g = torch.Generator().manual_seed(11)
    x = _rand(g, (2, 13, 19, 64))
    w1, w2 = _rand(g, (256, 1, 1, 64), 0.17), _rand(g, (128, 3, 3, 256), 0.03)
    s, b = torch.ones(256), torch.zeros(256)
    y1 = torch.empty((2, 13, 19, 256), device=dev)
    # all host-side work (weight splits, scale folding) first; x_multiplier given, so nothing reads y1 before the second launch
    first = ops.conv2d_prepare(x.to(dev), w1.reshape(256, -1).contiguous().to(dev), s.to(dev), b.to(dev), 1, 1, 0, 1, relu=True, kind="f16",
                               out=y1, x_multiplier=1.0)
    second = ops.conv2d_prepare(y1, w2.reshape(128, -1).contiguous().to(dev), s[:128].to(dev), b[:128].to(dev), 3, 3, 1, 1, kind="f16",
                                x_multiplier=1.0)
    torch.cuda.synchronize()
    first.launch()
    second.launch()                      # consecutive conv kernels on the stream, no sync and no other kernel between them
    y2 = second.result
    torch.cuda.synchronize()
    r1, S1, _ = _ref_conv(x, w1, s, b, 1, 0, 1, relu=True)
    r2, S2, _ = _ref_conv(r1.float(), w2, s[:128], b[:128], 3, 1, 1)
    err = float((y2.cpu().double() - r2).abs().max() / max(1.0, float(r2.abs().max())))
    assert err < 1e-4, err


DYN_EXPS = (-16, -12, -8, 0, 8)


def dynamic_range(dev):
    """one representative 3x3 layer per kind with x scaled by 2^e: the tf32 kind and the f16 op (with its automatic input multiplier)
    meet the bound at every scale; the bare f16 split (x_multiplier = 1, the engine's form) meets it at e >= 0 and is measured below"""
    c = dict(name="dyn 3x3", N=2, H=13, W=19, Cin=64, Cout=128, k=3, pad=1, stride=1, plain=True)
    rows = []
    for e in DYN_EXPS:
        for kind, xm in (("tf32", "auto"), ("f16", "auto"), ("f16", 1.0)):
            r = run_case(dict(c, kind=kind, xm=xm), dev, scale_exp=e)
            r.update(exp=e, x_multiplier=xm)
            rows.append(r)
    return rows


@pytest.fixture(scope="module")
def dev(built):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("case", matrix_cases(), ids=lambda c: "%s-%s" % (c["kind"], c["name"].replace(" ", "_")))
def test_conv_matrix_case(dev, case):
    check_result(case, run_case(case, dev))


@pytest.mark.gpu
def test_conv_range_flag(dev):
    range_flag_checks(dev)


@pytest.mark.gpu
def test_conv_dynamic_range(dev):
    for r in dynamic_range(dev):
        if r["x_multiplier"] == "auto" or r["exp"] >= 0:
            assert r["ratio"] <= 1.0 and r["rel"] < 1e-4, (r["kind"], r["exp"], r["x_multiplier"], r["ratio"], r["rel"])


# the kernel switches, one process each (the default settings included); the combined settings reach the 1-slot forms of the tiles
# whose MMA mode they force
SETTINGS = [{}, {"DT_CONV_MMA": "1sm"}, {"DT_CONV_MMA": "2sm"}, {"DT_CONV_MMA": "1sm", "DT_CONV_SLOTS": "1"},
            {"DT_CONV_MMA": "2sm", "DT_CONV_SLOTS": "1"}, {"DT_CONV_WS": "0"}, {"DT_CONV_WS": "2"}, {"DT_CONV_SLOTS": "1"}, {"DT_CONV_SLOTS": "2"},
            {"DT_CONV_NARROW1": "0"}, {"DT_CONV_HALO": "0"}, {"DT_CONV_RES_RING": "0"}, {"DT_CONV_PDL": "1"}]


def _setting_id(s):
    return "+".join("%s=%s" % kv for kv in s.items()) or "default"


@pytest.fixture(scope="module")
def switch_runs(built):
    """the matrix once per setting, each in its own process: setting id -> (return code, summary or None, output tail)"""
    runs = {}
    for setting in SETTINGS:
        env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
        env.update(setting)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "conv_matrix_check.py")], env=env, capture_output=True, text=True,
                           timeout=600)
        lines = r.stdout.strip().splitlines()
        summary = json.loads(lines[-1]) if lines and lines[-1].startswith('{"rows"') else None
        runs[_setting_id(setting)] = (r.returncode, summary, r.stdout[-3000:] + r.stderr[-3000:])
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("setting", SETTINGS, ids=_setting_id)
def test_conv_matrix_under_switch(switch_runs, setting):
    code, summary, tail = switch_runs[_setting_id(setting)]
    assert summary is not None and code == 0, tail
    assert summary["failed"] == [], summary["failed"]


@pytest.mark.gpu
def test_every_instantiation_is_reached(switch_runs, built):
    """the union of the rows the settings reach (each setting in its own process) is the whole instantiation table"""
    from detectorch_b200 import ops
    reached = set()
    for _, summary, _ in switch_runs.values():
        reached.update(summary["rows"] if summary else [])
    table = ops.conv_instantiations()
    missing = [table[i] for i in range(len(table)) if i not in reached]
    assert not missing, "instantiations no case reaches: %s" % missing
