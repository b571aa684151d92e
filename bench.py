#!/usr/bin/env python
"""bench.py -- images/sec of Mask R-CNN R-50-FPN inference @ 3x800x1216, 1000 proposals, 100 detections
(BASELINE.json `metric`, configs[2]: batch 8 per B200), one process per GPU.

  python bench.py --gpus 1 --steps 20 --warmup 3            # our arm (sm_100a engine)
  python bench.py --impl reference --steps 2 --warmup 1     # reference arm: the reference path on the host cores
  python bench.py --steps 20 --dump-outputs DIR            # also write the outputs of the last timed step as DIR/<name>.npy

A "step" = one pass of the whole hot path (trunk, FPN, RPN, proposals, RoIAlign, box head, per-class NMS,
mask head) over one batch of synthetic images.  `value` is timed with inputs resident in HBM (CUDA-graph replay of
dt_engine_run); `e2e` is the same metric through the public call `detector.detect(pinned host images)`: H2D copy of
the images and D2H read of the detections + masks inside the timed region; `e2e_reference_flow` is the batch-1
notebook-shaped flow (model(img) -> postprocess_output -> add_multilevel_rois_for_test -> mask_head -> segm_results,
host image in, COCO RLE strings out).  Extra keys: `roofline_roialign` (+ `microbench`) = BASELINE.json configs[4]
(100k RoIs x 256 ch x 50x68) with the reference's own CUDA kernel timed beside it.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec Mask R-CNN R-50-FPN @800x1216, 1k proposals"
WORKLOAD = "Mask R-CNN R-50-FPN inference, batch 8 per GPU, 3x800x1216 fp32, 1000 proposals/img, 100 dets/img (BASELINE.json configs[2])"
GFLOP_PER_IMAGE = 490.5          # SURVEY.md 8(a): algorithmic 2*MAC per image for this config
H, W, BATCH = 800, 1216, 8


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1400.0, "fallback"       # B200_PROFILING.md fallback figures


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2])


def cpu_reference_images_per_sec(steps, warmup, arch="resnet50"):
    """The reference's CPU path for this workload: its detector graph under torch-CPU fp32 + its RoIAlign loop +
    its greedy NMS + numpy post-processing, as restated in oracle/ (the reference tree does not exist on the GPU
    box; oracle/_ref holds its compiled RoIAlign loop when it was built here).  One step = one image (bounded sample).
    Threads = what this process may really use (affinity mask capped by the cgroup quota), not os.cpu_count(): a 128-thread pool
    inside a smaller quota was the 12x swing of the round-1 figure.  >= 1 warm-up, median of >= 3, per-stage break-out."""
    import torch
    from oracle import network as net
    from oracle import usable_cpus
    n = usable_cpus()
    torch.set_num_threads(n)
    P = net.synthetic_params(arch)
    img = net.synthetic_image(1, H, W)
    for _ in range(max(1, warmup)):
        net.detect_and_mask_fpn(img, P, arch=arch)
    times, stages = [], {}
    for _ in range(max(3, steps)):
        t = {}
        t0 = time.perf_counter()
        net.detect_and_mask_fpn(img, P, arch=arch, timers=t)
        times.append(time.perf_counter() - t0)
        for k, v in t.items():
            stages.setdefault(k, []).append(v)
    dt = _median(times)
    return 1.0 / dt, dt, n, {k: round(_median(v) * 1e3, 2) for k, v in stages.items()}, len(times), [round(x, 4) for x in times]


def cpu_fast_rcnn_c4(steps=3, warmup=1):
    """BASELINE.json configs[0] (BASELINE.md section 3): Fast R-CNN R-50-C4, 1 image 3x800x1216, 300 pre-computed proposals, on the host cores."""
    import numpy as np
    import torch
    from oracle import network as net
    from oracle import usable_cpus
    n = usable_cpus()
    torch.set_num_threads(n)
    P = net.synthetic_params("resnet50", fpn=False, rpn=False, mask=False)
    img = net.synthetic_image(1, H, W)
    rng = np.random.RandomState(0)
    cx, cy = rng.uniform(0, W, 300), rng.uniform(0, H, 300)
    wd = np.exp(rng.uniform(np.log(16), np.log(600), 300)); a = np.exp(rng.uniform(-0.7, 0.7, 300))
    pr = np.stack([cx - wd * np.sqrt(a) / 2, cy - wd / np.sqrt(a) / 2, cx + wd * np.sqrt(a) / 2, cy + wd / np.sqrt(a) / 2], 1)
    pr[:, 0::2] = np.clip(pr[:, 0::2], 0, W - 1); pr[:, 1::2] = np.clip(pr[:, 1::2], 0, H - 1)
    pr = pr.astype(np.float32)
    for _ in range(warmup):
        net.detect_and_mask_c4(img, P, proposals=pr, use_mask=False)
    times, stages = [], {}
    for _ in range(steps):
        t = {}
        t0 = time.perf_counter()
        net.detect_and_mask_c4(img, P, proposals=pr, use_mask=False, timers=t)
        times.append(time.perf_counter() - t0)
        for k, v in t.items():
            stages.setdefault(k, []).append(v)
    dt = _median(times)
    return {"workload": "Fast R-CNN R-50-C4, 1 image 3x800x1216, 300 pre-computed proposals (BASELINE.json configs[0])", "images_per_sec": 1.0 / dt,
            "ms_per_image": dt * 1e3, "cores": n, "runs": len(times), "stage_ms": {k: round(_median(v) * 1e3, 2) for k, v in stages.items()}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(3, min(args.steps, 5))
    warm = max(1, min(args.warmup, 2))
    ips, dt, n, stages, runs, raw = cpu_reference_images_per_sec(steps, warm, args.arch)
    line = {"impl": "reference", "metric": METRIC if args.arch == "resnet50" else METRIC.replace("R-50", "R-101"), "value": ips, "unit": "images/sec", "n_gpus": args.gpus,
            "steps": runs, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "reference CPU path (torch-CPU fp32 graph + reference RoIAlign loop + greedy NMS), 1 image per step "
                                                     "(bounded sample of the batch-8 workload); value = 1 / median step time", "threads": n,
                       "threads_rule": "len(sched_getaffinity) capped by the cgroup cpu.max quota", "step_seconds": raw},
            "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": n, "kind": "port", "sample": "median of %d x 1 image 3x800x1216 after %d warm-up" % (runs, warm),
                             "stage_ms": stages},
            "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_config1:
        line["cpu_config1_fast_rcnn_c4"] = cpu_fast_rcnn_c4()
    emit(line)


# ----------------------------------------------------------------------------- our arm
MIRROR_KW = dict(conv_body_layers=['conv1', 'bn1', 'relu', 'maxpool', 'layer1', 'layer2', 'layer3', 'layer4'], conv_head_layers='two_layer_mlp',
                 fpn_layers=['layer1', 'layer2', 'layer3', 'layer4'], fpn_extra_lvl=True, roi_height=7, roi_width=7,
                 roi_spatial_scale=[0.25, 0.125, 0.0625, 0.03125], roi_sampling_ratio=2, use_rpn_head=True, use_mask_head=True,
                 mask_head_type='1up4convs')       # eval_mask_FPN.ipynb cell 7


def pin_to_gpu_numa_node(local):
    """Bind this process (the launch thread and, by first touch, the pinned host buffers it allocates next) to the CPUs of the GPU's NUMA
    node: at N=8 eight processes otherwise share two sockets at random and the H2D streams / launch threads cross the socket link
    (round-1: device-side scaling 0.998 but end-to-end 0.973).  Best effort; returns a description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return {"numa_node": None}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus_bound": len(allowed)}
    except Exception as e:       # no sysfs entry / no permission: keep the default placement
        return {"numa_node": None, "note": type(e).__name__}


def time_cuda(fn, torch, warm=2, reps=5, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()               # > L2-sized write between timed iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return _median(ts)


def microbench_roialign(torch, dev, hbm_peak, which):
    """BASELINE.json configs[4]: 100 000 RoIs x 256 channels x 50x68 map, pooled 7x7 (and 14x14), sampling_ratio 2.  Algorithmic bytes =
    output write + map + RoIs (SURVEY.md 8d: 5 023 081 600 B for 7x7).  L2 is flushed between timed iterations.  The reference's own
    CUDA kernel (lib/cppcuda_cffi/src/cuda/roi_align_forward_cuda_kernel.cu compiled unmodified for sm_100a into oracle/_ref) is timed on the
    same inputs when that build exists."""
    import ctypes
    import numpy as np
    from detectorch_b200 import ops
    R, C, Hf, Wf = 100000, 256, 50, 68
    rng = np.random.RandomState(0)
    cx, cy = rng.uniform(0, 1088, R), rng.uniform(0, 800, R)
    wd = np.exp(rng.uniform(np.log(16), np.log(600), R)); a = np.exp(rng.uniform(-0.7, 0.7, R))
    b = np.stack([np.zeros(R), cx - wd * np.sqrt(a) / 2, cy - wd / np.sqrt(a) / 2, cx + wd * np.sqrt(a) / 2, cy + wd / np.sqrt(a) / 2], 1)
    b[:, 1::2] = np.clip(b[:, 1::2], 0, 1087); b[:, 2::2] = np.clip(b[:, 2::2], 0, 799)
    rois = torch.from_numpy(b.astype(np.float32)).to(dev)
    g = torch.Generator().manual_seed(0)
    feat = torch.randn((1, C, Hf, Wf), generator=g).to(dev)
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    refso = os.path.join(ROOT, "oracle", "_ref", "libroialign_ref_cuda.so")
    rows = {}
    for pooled in (7, 14):
        out = torch.empty((R, C, pooled, pooled), device=dev)
        alg = out.numel() * 4 + feat.numel() * 4 + rois.numel() * 4
        r = {"algorithmic_bytes": alg}
        r["fast_ms"] = time_cuda(lambda: ops.roi_align_forward_nchw_fast(feat, rois, pooled, pooled, 1 / 16., 2, out=out), torch, flush=flush)
        r["exact_ms"] = time_cuda(lambda: ops.roi_align_forward_nchw(feat, rois, pooled, pooled, 1 / 16., 2, out=out), torch, flush=flush)
        if os.path.exists(refso) and out.numel() < 2 ** 31:
            L = ctypes.CDLL(refso)
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            r["reference_cuda_kernel_ms"] = time_cuda(lambda: L.launch_roi_align_forward_cuda(
                ctypes.c_int(out.numel()), ctypes.c_void_p(feat.data_ptr()), ctypes.c_void_p(rois.data_ptr()), ctypes.c_float(1 / 16.), C, Hf, Wf,
                pooled, pooled, 2, ctypes.c_void_p(out.data_ptr()), st), torch, flush=flush)
        r["fast_gbs"] = alg / (r["fast_ms"] * 1e-3) / 1e9
        r["frac_hbm_peak"] = r["fast_gbs"] / hbm_peak
        rows["%dx%d" % (pooled, pooled)] = r
        del out
    r7 = rows["7x7"]
    roof = {"bound": "hbm", "kernel": "roi_align fast path (dt_roi_align_forward_nchw_fast), 100k RoIs x 256 ch x 50x68, 7x7 sr=2", "achieved": r7["fast_gbs"],
            "peak": hbm_peak, "unit": "GB/s", "frac": r7["frac_hbm_peak"], "traffic": None, "peak_source": which, "frac_14x14": rows["14x14"]["frac_hbm_peak"]}
    return roof, rows


def dump_outputs(out_dir, eng):
    """Writes what the last timed step computed, the arrays detector.detect() returns for that batch (boxes, scores, classes, counts,
    roi_idx, masks of the detected class, range_flag), to out_dir/<name>.npy as float32 (float64 for the integer arrays): about 3 MB at
    batch 8.  Slots past an image's detection count hold no result and are written as zeros, so that the outputs of two builds on the
    same (seeded) inputs can be compared array for array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    counts = eng.buffer("det_counts").cpu().numpy().astype(np.int64)
    B = len(counts)
    arrays = {"boxes": eng.buffer("det_boxes"), "scores": eng.buffer("det_scores"), "classes": eng.buffer("det_classes"),
              "roi_idx": eng.buffer("det_roi_idx"), "masks": eng.buffer("masks")}
    for name, t in arrays.items():
        a = t.cpu().numpy()
        a = a.reshape((B, -1) + a.shape[1:] if name == "masks" else a.shape)          # masks: [B * cap, 28, 28] -> [B, cap, 28, 28]
        a = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
        for b in range(B):
            a[b, counts[b]:] = 0
        np.save(os.path.join(out_dir, name + ".npy"), a)
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))
    np.save(os.path.join(out_dir, "range_flag.npy"), eng.buffer("range_flag").cpu().numpy().astype(np.float64))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from detectorch_b200.engine import ST_TRUNK, ST_MASK_OUT
    from detectorch_b200.model.detector import detector
    from detectorch_b200.utils import result_utils
    from detectorch_b200.utils.multilevel_rois import add_multilevel_rois_for_test
    from oracle import network as net      # synthetic weights / images only (shared seeded generator)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    steps, warmup = args.steps, max(args.warmup, 3)

    # the public object: the reference-shaped detector (eval_mask_FPN.ipynb kwargs) with the synthetic weights in its state_dict
    model = detector(arch=args.arch, **MIRROR_KW)
    model.load_state_dict(net.synthetic_params(args.arch), strict=False)
    model = model.cuda(dev)
    model.engine_defaults.update(det_cap=100, emit_full_masks=False)       # fused outputs only; model.mask_head (reference flow) uses its own engine below
    eng = model.engine_for(BATCH, H, W)
    # distinct images per rank (weak scaling: 8 images per GPU); two host batches alternate so no step re-reads a hot input
    host = [net.synthetic_image(BATCH, H, W, seed=10 * rank + i).pin_memory() for i in range(2)]
    dimg = [h.to(dev, non_blocking=True) for h in host]
    torch.cuda.synchronize()
    launches_per_step = eng.count_launches(ST_TRUNK, ST_MASK_OUT)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- capture the step in a CUDA graph (one per resident input buffer)
    graphs = []
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        for i in range(2):
            eng.run(dimg[i], 1.0)
        side.synchronize()
        for i in range(2):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                eng.run(dimg[i], 1.0)
            graphs.append(g)
    torch.cuda.synchronize()

    # ---- (A) device-resident throughput
    for i in range(warmup):
        graphs[i % 2].replay()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_region = os.environ.get("DT_NCU_REGION") == "1"      # `ncu --profile-from-start off`: profile exactly the timed steps
    if ncu_region:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
    ev0.record()
    for i in range(steps):
        graphs[i % 2].replay()
    ev1.record()
    if ncu_region:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    eng.check_range()      # the kind::f16 conv path raises a device flag if an activation left the fp16 range (never on this workload)
    rois_per_image = float(eng.buffer("roi_counts").float().mean().item())
    dets_per_image = float(eng.buffer("det_counts").float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)         # the engine buffers still hold the last timed step (batch (steps - 1) % 2)

    # ---- (B) end to end through the public call with HOST buffers: model.detect(pinned host batch) uploads through its two staging
    # buffers on a copy stream (H2D of step i+1 overlaps the compute of step i); every step's results are read back to pinned host memory
    res_keys = ["boxes", "scores", "classes", "counts", "masks", "range_flag"]
    probe = model.detect(host[0])
    res_host = [[torch.empty(probe[k].shape, dtype=probe[k].dtype).pin_memory() for k in res_keys] for _ in range(2)]
    h2d_bytes = host[0].numel() * 4
    d2h_bytes = sum(probe[k].numel() * probe[k].element_size() for k in res_keys)
    torch.cuda.synchronize()

    def e2e_loop(n):
        for i in range(n):
            out = model.detect(host[i % 2])
            for k, hbuf in zip(res_keys, res_host[i % 2]):
                hbuf.copy_(out[k], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_loop(max(warmup, 4))          # detect() captures its CUDA graphs (one per staging buffer) on the second use of each buffer
    barrier()
    t0 = time.perf_counter()
    e2e_loop(steps)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3            # wall clock around H2D + compute + D2H of all steps (device work is bracketed by syncs)
    assert int(res_host[0][res_keys.index("range_flag")].item()) == 0

    # ---- (C) the reference-shaped flow, one image at a time, host image in, RLE strings out (what a notebook user runs)
    flow = None
    if rank == 0 and not args.no_reference_flow:
        imgs1 = [net.synthetic_image(1, H, W, seed=100 + i).pin_memory() for i in range(4)]
        im_size = torch.tensor([[float(H), float(W), 3.0]])

        def one_image(x):
            cls, box, rois, feats = model(x.to(dev, non_blocking=True), scaling_factor=1.0)
            sf_, bf_, per_class = result_utils.postprocess_output(rois, 1.0, im_size, cls, box)
            if len(bf_) == 0:
                return 0
            ml = add_multilevel_rois_for_test({'rois': bf_ * 1.0}, 'rois')
            lst = [torch.from_numpy(ml['rois_fpn%d' % l]).to(dev) if len(ml['rois_fpn%d' % l]) else None for l in (2, 3, 4, 5)]
            masks = model.mask_head(feats, lst, torch.from_numpy(ml['rois_idx_restore_int32'].astype(np.int64)).to(dev))
            segms = result_utils.segm_results(per_class, masks, bf_, H, W, M=28)
            return sum(len(c) for c in segms)
        model.engine_defaults.update(det_cap=128, emit_full_masks=True)      # the reference layout [D,81,28,28] for model.mask_head
        for x in imgs1[:2]:
            one_image(x)
        torch.cuda.synchronize()
        n_flow = 16
        t0 = time.perf_counter()
        nseg = 0
        for i in range(n_flow):
            nseg += one_image(imgs1[i % 4])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        flow = {"value": n_flow / dt, "unit": "images/sec", "ms_per_image": dt / n_flow * 1e3, "images": n_flow, "rle_strings": nseg,
                "h2d_bytes_per_image": imgs1[0].numel() * 4,
                "note": "batch-1 reference-shaped flow: model(img) -> postprocess_output (.item() + D2H + numpy) -> add_multilevel_rois_for_test -> "
                        "model.mask_head -> segm_results (RLE strings on the host); wall clock, pinned host image in"}
        model.engine_defaults.update(det_cap=100, emit_full_masks=False)

    # ---- max over ranks
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = t.tolist()

    # ---- roofline of the dominant kernel family (conv_tcgen05_kernel), measured live with CUDA events on the launch stream
    roof, roi_roof, roi_engine, micro, cpu_base = None, None, None, None, None
    if rank == 0:
        hbm_peak, bf16_peak, which = peaks()
        prof = eng.profile(dimg[0], 1.0)
        conv = [(m, f) for (m, f, st, bn) in prof if bn > 0]
        conv_ms, conv_flops = sum(m for m, _ in conv), sum(f for _, f in conv)
        all_ms = sum(m for (m, _, _, _) in prof)
        stage_names = ["trunk", "fpn", "rpn_convs", "proposals", "collect", "roialign_box", "box_head", "detect_nms", "mask_rois", "roialign_mask",
                       "mask_head", "mask_out"]
        stage_ms = {}
        for (m, f, st, bn) in prof:
            stage_ms[stage_names[st]] = round(stage_ms.get(stage_names[st], 0.0) + m, 4)
        f16_kind = eng.cfg.conv_kind == 0
        # kind::f16 issues at the bf16 rate; kind::tf32 at half of it (B200_PROFILING.md nominal 2.25 vs 1.1 PF)
        mma_peak = bf16_peak if f16_kind else bf16_peak / 2.0
        ach = conv_flops / (conv_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_dram_bytes.json")
        if os.path.exists(tp):       # dram__bytes_read.sum + dram__bytes_write.sum of the conv launches of one step (an ncu pass of this very command)
            td = json.load(open(tp))
            traffic, traffic_src = td.get("conv_family_bytes_per_step"), td.get("source")
        roof = {"bound": "tensor", "kernel": "conv_tcgen05_kernel (%d launches/step)" % len(conv), "achieved": ach, "peak": mma_peak, "unit": "TFLOP/s",
                "frac": ach / mma_peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "%s bf16_tflops_sustained%s" % (which, " (kind::f16 MMA rate)" if f16_kind else "/2 (tf32 MMA rate is half of bf16)"),
                "executed_tflops": 3.0 * ach, "frac_executed": 3.0 * ach / mma_peak,
                "note": "achieved = algorithmic 2*MAC FLOPs of all conv/GEMM launches / their summed CUDA-event time; the kernel executes 3 %s MMAs "
                        "per algorithmic product (error-compensated hi/lo split, fp32-accurate), frac_executed counts those" % ("fp16" if f16_kind else "TF32"),
                "share_of_step": conv_ms / all_ms, "stage_ms": stage_ms}
        # RoIAlign inside the engine (box head, 7x7): algorithmic bytes = output write + RoIs (maps are L2 resident)
        roi = [m for (m, f, st, bn) in prof if st == 5]
        if roi:
            gbs = BATCH * 1000 * (49 * 256 * 4 + 20) / (roi[0] * 1e-3) / 1e9
            roi_engine = {"kernel": "roi_align_fast_nhwc_kernel (box head, 8000 RoIs over P2..P5)", "achieved": gbs, "unit": "GB/s", "frac": gbs / hbm_peak}
        if not args.no_microbench:
            roi_roof, micro = microbench_roialign(torch, dev, hbm_peak, which)
            roi_roof["in_engine"] = roi_engine
        if not args.no_cpu_baseline and world == 1:          # the CPU baseline is reported at N=1 only
            ips, dt, n, stages, runs, raw = cpu_reference_images_per_sec(3, 1)
            cpu_base = {"value": ips, "unit": "images/sec", "cores": n, "kind": "port",
                        "sample": "median of %d x 1 image 3x800x1216 (1/8 of one step) after 1 warm-up, oracle/network.py" % runs, "stage_ms": stages,
                        "step_seconds": raw}

    if rank == 0:
        total_images = BATCH * world * steps
        value = total_images / (ms * 1e-3)
        gflop_img = GFLOP_PER_IMAGE if args.arch == "resnet50" else 634.5
        line = {"metric": METRIC if args.arch == "resnet50" else METRIC.replace("R-50", "R-101"), "value": value, "unit": "images/sec", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (%s tensor-core products, fp32 accumulate)" % ("3xFP16 hi/lo" if eng.cfg.conv_kind == 0 else "3xTF32"),
                "data": "synthetic", "per_gpu_value": value / world,
                "config": {"workload": WORKLOAD if args.arch == "resnet50" else WORKLOAD.replace("R-50", "R-101").replace("configs[2]", "configs[3] model"), "global_batch": BATCH * world, "parallelism": "dp%d (images sharded, no data-path collective)" % world,
                           "l2": "inputs alternate between two 93 MB batches and every step streams ~11 GB of activations (>> 126 MB L2)",
                           "cuda_graph": True, "tflops_algorithmic": value * gflop_img / 1e3,
                           "rois_per_image": rois_per_image, "dets_per_image": dets_per_image, "numa": numa},
                "clocks": clocks,
                "e2e": {"value": total_images / (e2e_ms * 1e-3), "unit": "images/sec", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "ms_per_step": e2e_ms / steps, "per_gpu_value": total_images / (e2e_ms * 1e-3) / world,
                        "note": "detector.detect(pinned host batch): H2D through two staging buffers on a copy stream -> fused engine (CUDA-graph replay inside detect) -> D2H of "
                                "boxes/scores/classes/counts/masks into pinned memory; wall clock, max over ranks"},
                "e2e_reference_flow": flow,
                "gpu_launches": launches_per_step * steps,
                "roofline": roof, "roofline_roialign": roi_roof, "microbench": micro, "cpu_baseline": cpu_base}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_json_out = None


def emit(line):
    """The ONE JSON line goes to the process's original stdout; everything else that libraries write to fd 1 (e.g. NCCL's version
    banner on rank 0) was redirected to stderr in main()."""
    out = _json_out if _json_out is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _json_out
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-microbench", action="store_true", help="skip the configs[4] RoIAlign microbench keys")
    ap.add_argument("--no-reference-flow", action="store_true", help="skip the batch-1 notebook-shaped end-to-end figure")
    ap.add_argument("--no-config1", action="store_true", help="reference arm: skip the Fast R-CNN R-50-C4 (configs[0]) CPU timing")
    ap.add_argument("--arch", default="resnet50", choices=["resnet50", "resnet101"],
                    help="resnet101 = BASELINE.json configs[3] model (not the headline metric)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
