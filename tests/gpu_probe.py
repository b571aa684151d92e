"""GPU bring-up probe (not a pytest file): runs groups of operator checks against the oracle and
prints one line per case.  Used under gpurun with a per-group `timeout` so a hung kernel cannot
hang the box:   timeout 300 python tests/gpu_probe.py roialign nms
"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from detectorch_b200 import ops  # noqa: E402
from oracle import ref  # noqa: E402

dev = torch.device("cuda:0")


def group_roialign():
    rng = np.random.RandomState(0)
    f = rng.randn(2, 16, 25, 38).astype(np.float32)
    R = 300
    x1 = rng.uniform(-50, 600, R); y1 = rng.uniform(-50, 400, R); w = rng.uniform(1, 500, R); h = rng.uniform(1, 400, R)
    r = np.stack([rng.randint(0, 2, R), x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
    for (p, sr, sc) in [(7, 2, 1 / 16), (14, 0, 1 / 16), (14, 2, 1 / 8), (7, 0, 1 / 32)]:
        want = ref.roi_align_forward(f, r, p, p, sc, sr)
        got = ops.roi_align_forward_nchw(torch.from_numpy(f).to(dev), torch.from_numpy(r).to(dev), p, p, sc, sr).cpu().numpy()
        print("ROIALIGN nchw p%d sr%d : max_abs %.3e bit_exact %s" % (p, sr, np.abs(got - want).max(), np.array_equal(got, want)), flush=True)
        fn = torch.from_numpy(f).permute(0, 2, 3, 1).contiguous().to(dev)
        got2 = ops.roi_align_forward_nhwc([fn], [sc], torch.from_numpy(r).to(dev), None, p, p, sr).permute(0, 3, 1, 2).cpu().numpy()
        print("ROIALIGN nhwc p%d sr%d : max_abs %.3e bit_exact %s" % (p, sr, np.abs(got2 - want).max(), np.array_equal(got2, want)), flush=True)


def group_nms():
    rng = np.random.RandomState(1)
    for n in [1, 7, 64, 65, 100, 1000, 3000, 6000]:
        x1 = rng.uniform(0, 1000, n); y1 = rng.uniform(0, 700, n); w = rng.uniform(5, 300, n); h = rng.uniform(5, 300, n)
        d = np.stack([x1, y1, x1 + w, y1 + h, rng.uniform(0, 1, n)], 1).astype(np.float32)
        for t in (0.3, 0.5, 0.7):
            want = ref.nms(d, t)
            t0 = time.time()
            got = ops.nms(torch.from_numpy(d).to(dev), t).cpu().numpy()
            print("NMS n%d t%.1f : kept %d/%d equal %s  %.3fs" % (n, t, len(got), len(want), np.array_equal(got, want), time.time() - t0), flush=True)


if __name__ == "__main__":
    print("device:", torch.cuda.get_device_name(0), flush=True)
    for name in sys.argv[1:]:
        print("==== group", name, flush=True)
        globals()["group_" + name]()
    print("==== done", flush=True)
