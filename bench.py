#!/usr/bin/env python
"""Benchmark of the B200-native proposal + NMS + RoI-layer hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload C1 (SURVEY.md 8d): ResNet-50 at 600x1000 -> 38x63 feature map, 9 anchors (scales 128/256/512),
21,546 anchors/image; top-k 8000, NMS 0.7 -> 300 RoIs, padded to 320 = 5x64 rows like the reference, RoI layer
(crop + bilinear resize to 7x7) on 1024-channel float32 features.  One "step" = this path over one batch of
`--images-per-gpu` synthetic images per GPU (weak scaling: images are independent, no collective on the path; the
only exchange is one NCCL all-gather of the final RoIs + counts per step).

Prints ONE JSON line (rank 0).  `value` = images/s with inputs resident in HBM; `e2e` = the same through the
public API (`ProposalRoiPipeline.__call__`) with pinned HOST inputs, H2D/D2H inside the timed region (plus
`e2e.device_features`: the same call when a GPU backbone hands the feature map over as a CUDA tensor);
`roofline` = RoI-forward kernel (the HBM-bound, dominant kernel) vs the measured copy peak, as a 20-step burst
(`frac`) and over a >= 2 s window under the power cap (`frac_sustained`);
`stages` = the other BASELINE.json configs timed live in the same run (C2 post-processing, C3 KITTI proposals,
C4 target assignment, C5 RoI forward + backward in both modes; per-GPU work is fixed, times are the max over ranks);
`cpu_baseline` / `--impl reference` = the reference's CPU algorithm (numpy port of the reference, pinned bit-exact
against it) on the host cores.  Both arms print the same `config`.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ROWS, COLS, CHANNELS = 38, 63, 1024
SCALES = [128, 256, 512]
STRIDE, TOPK, NMS_THRESH, MAX_BOXES, NUM_ROIS, POOL = 16, 8000, 0.7, 300, 64, 7
PADDED = -(-MAX_BOXES // NUM_ROIS) * NUM_ROIS          # 320
POOLED_SAMPLE = 128                                     # RoI rows of the pooled output kept by --dump-outputs
METRIC = "img/s proposal+NMS+RoIpool @600x1000"
UNIT = "img/s"
WORKLOAD = ("C1: ResNet-50 600x1000 -> 38x63x9 anchors (21546/img), top-k 8000, NMS 0.7->300, pad to 320 RoIs, "
            "RoI crop+bilinear 7x7 on 1024-ch f32 features")


def shared_config(batch, world):
    """`config` of BOTH arms (the driver compares them): the workload and how a step is cut, nothing arm-specific."""
    return {"workload": WORKLOAD, "images_per_gpu_per_step": batch, "global_images_per_step": world * batch,
            "parallelism": "image-sharded x%d, no hot-path collective, all-gather of final RoIs" % world,
            "l2": "inputs larger than L2 (%.0f MB of features + %.0f MB of pooled output per GPU and step vs 126 MB L2)"
                  % (batch * ROWS * COLS * CHANNELS * 4 / 1e6, batch * PADDED * POOL * POOL * CHANNELS * 4 / 1e6)}


def anchor_dims():
    from faster_rcnn_b200.util import get_anchors
    return get_anchors(SCALES)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port) on the host cores, image-parallel
# ------------------------------------------------------------------------------------------------
_cpu_inputs = None


def _cpu_init():
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)          # one image per worker process; no nested BLAS/OpenMP threads
    except Exception:
        pass


def _cpu_proposals(i):
    """one image through decode -> filter -> top-k -> NMS only (the part the reference itself runs on the CPU;
    its RoI layer lives in the TF graph)."""
    from oracle import frcnn_oracle as O
    cls, regr, _ = _cpu_inputs[i % len(_cpu_inputs)]
    dims = O.anchor_table(SCALES)
    boxes = O.proposals_from_rpn(regr.copy(), dims, STRIDE)
    b, p, _ = O.topk_proposals(boxes, cls.reshape(-1), TOPK)
    rois, _ = O.nms(b, p, NMS_THRESH, MAX_BOXES)
    return len(rois)


def check_decode(path):
    """cpu_baseline leg as the CHECKER: rows of the device's decoded boxes (saved by the GPU arm) that differ from the
    numpy port's decode of the same head outputs, per config."""
    from oracle import frcnn_oracle as O
    z = np.load(path)
    out = {}
    for tag, scales in (("C1", SCALES), ("C3", None)):
        dims = O.anchor_table(scales) if scales else O.anchor_table()
        regr, dense = z[tag + "_regr"], z[tag + "_dense"]
        flips = 0
        for i in range(len(regr)):
            want = O.proposals_from_rpn(regr[i:i + 1].copy(), dims, STRIDE)
            flips += int(np.sum(np.any(dense[i] != want, axis=1)))
        out[tag] = {"anchors_checked": int(dense.shape[0] * dense.shape[1]), "rows_differing": flips}
    return out


def _cpu_image(i):
    """one image through the reference's CPU path: decode -> filter -> top-k -> NMS -> pad -> RoI layer."""
    from oracle import frcnn_oracle as O
    from oracle import roi_oracle as R
    cls, regr, feat = _cpu_inputs[i % len(_cpu_inputs)]
    dims = O.anchor_table(SCALES)
    boxes = O.proposals_from_rpn(regr.copy(), dims, STRIDE)
    b, p, _ = O.topk_proposals(boxes, cls.reshape(-1), TOPK)
    rois, _ = O.nms(b, p, NMS_THRESH, MAX_BOXES)
    n = len(rois)
    rows = -(-n // NUM_ROIS) * NUM_ROIS
    if rows > n:
        rois = np.concatenate([rois, np.tile(rois[rows - NUM_ROIS], (rows - n, 1))])
    out = R.roi_resize_fwd(feat[0], rois, POOL)
    return float(out[0, 0, 0, 0])


class CpuArm:
    def __init__(self, cores=None, n_pre=8):
        global _cpu_inputs
        from faster_rcnn_b200 import synth
        self.cores = cores or len(os.sched_getaffinity(0))
        _cpu_inputs = []                                     # built before the fork: shared copy-on-write
        for i in range(n_pre):
            cls, regr = synth.rpn_outputs(ROWS, COLS, 9, 1000 + i)
            _cpu_inputs.append((cls, regr, synth.feature_map(ROWS, COLS, CHANNELS, 2000 + i)))
        ctx = mp.get_context("fork")
        self.pool = ctx.Pool(self.cores, initializer=_cpu_init)
        self.pool.map(_cpu_image, range(self.cores))          # warm every worker

    def run(self, n_images, fn=None):
        t0 = time.perf_counter()
        self.pool.map(fn or _cpu_image, range(n_images), chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (numpy port), all host cores.  One step =
    the same global batch as the GPU arm's step (world x images-per-gpu images); under torchrun rank 0 alone runs."""
    if rank != 0:
        return
    arm = CpuArm()
    batch = args.images_per_gpu
    per_step = world * batch
    for _ in range(args.warmup):
        arm.run(per_step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.run(per_step)
    dt = time.perf_counter() - t0
    value = args.steps * per_step / dt
    prop_s = arm.run(max(per_step, 2 * arm.cores), _cpu_proposals)
    prop_value = max(per_step, 2 * arm.cores) / prop_s
    arm.close()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": shared_config(batch, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": "port",
                         "sample": "%d steps x %d images, numpy port of the reference (pinned bit-exact against it), image-"
                                   "parallel fork pool, %s" % (args.steps, per_step, cpu_model()),
                         "proposals_nms_only": {"value": prop_value, "unit": UNIT,
                                                "note": "decode + top-k + NMS without the RoI layer: the part the reference "
                                                        "runs on the CPU itself (its RoI layer is a TF graph op); ~80 % of "
                                                        "the full figure's time is the numpy RoI-layer restatement"}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.check_decode:
        line["decode_check"] = check_decode(args.check_decode)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        ids = [v for v in vis.split(",") if v != ""]
        if local_rank < len(ids) and ids[local_rank].isdigit():
            return int(ids[local_rank])
    return local_rank


def measured_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def roi_traffic_bytes(batch):
    """dram bytes per RoI-forward launch from the committed `ncu --set full` capture (profiles/roi_fwd_traffic.json).
    The capture names the sha256 of the kernel source it was taken from: a number from another version of roi.cu is
    stale and is dropped (null) instead of being replayed."""
    try:
        import hashlib
        t = json.load(open(os.path.join(ROOT, "profiles", "roi_fwd_traffic.json")))
        src = open(os.path.join(ROOT, "faster_rcnn_b200", "csrc", "roi.cu"), "rb").read()
        if int(t["images_per_launch"]) == batch and t.get("roi_cu_sha256") == hashlib.sha256(src).hexdigest():
            return float(t["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def timeit(fn, min_ms=10.0, iters=5):
    """mean ms per call by CUDA events on the current stream; warm-up and measurement each cover >= min_ms."""
    import torch
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        fn()
    b.record()
    torch.cuda.synchronize()
    per = max(a.elapsed_time(b) / 3, 1e-3)
    n = max(iters, int(min_ms / per))
    for _ in range(n // 2):
        fn()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def measure_stages(ops, dev, rank, world, peak, want_dump):
    """BASELINE.json configs[1..4] on this rank's GPU (per-GPU work is fixed: weak scaling, no collective).  Returns
    ({stage: ms}, algorithmic bytes per stage, dump of decoded boxes for the CPU-side decode check)."""
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.util import get_anchors

    def d(x, dtype=None):
        return torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).to(dev)

    ms, nbytes, dump = {}, {}, {}
    voc, kitti = get_anchors(SCALES), get_anchors()
    # C3: KITTI 600x1500 -> 38x94, 18 anchors / location (64,296 anchors): 12000 -> NMS 2000 (training) and 8000 -> 300
    b3 = 16
    pairs = [synth.rpn_outputs(38, 94, len(kitti), 9000 + rank * b3 + i, clustered=True) for i in range(b3)]
    cls3, regr3 = d(np.concatenate([p[0] for p in pairs])), d(np.concatenate([p[1] for p in pairs]))
    ms["c3_kitti_proposals_12000_to_2000_b16"] = timeit(lambda: ops.proposals(regr3, cls3, kitti, STRIDE, 12000, 0.7, 2000))
    ms["c3_kitti_proposals_8000_to_300_b16"] = timeit(lambda: ops.proposals(regr3, cls3, kitti, STRIDE, 8000, 0.7, 300))
    ms["c3_kitti_proposals_12000_to_2000_b1"] = timeit(lambda: ops.proposals(regr3[:1], cls3[:1], kitti, STRIDE, 12000, 0.7, 2000))
    ms["c3_kitti_proposals_8000_to_300_b1"] = timeit(lambda: ops.proposals(regr3[:1], cls3[:1], kitti, STRIDE, 8000, 0.7, 300))
    if want_dump:
        dump["C3_regr"] = np.concatenate([p[1] for p in pairs[:2]])
        dump["C3_dense"] = ops.decode_topk(regr3[:2], cls3[:2], kitti, STRIDE, 12000, want_dense=True)[4].cpu().numpy()
    del cls3, regr3
    # C4: RPN labelling + packing + RoI labelling, 50 GT per image, batch 128 (16 per GPU at 8 GPUs)
    b4 = 128 // world if world > 1 else 128
    gts = np.stack([np.array([g[1:] for g in synth.gt_boxes(50, 1000, 600, 300 + rank * b4 + i)], np.float32) for i in range(b4)])
    gt, n_gt = d(gts), d(np.full(b4, 50, np.int32))
    wh = d(np.tile(np.array([[1000, 600]], np.int32), (b4, 1)))
    n_anch = ROWS * COLS * 9
    ms["c4_label_anchors"] = timeit(lambda: ops.label_anchors(gt, n_gt, wh, ROWS, COLS, voc, STRIDE))
    nbytes["c4_label_anchors"] = b4 * (16 * 50 + n_anch * 18)
    cu, ip, bb, _ = ops.label_anchors(gt, n_gt, wh, ROWS, COLS, voc, STRIDE)
    ms["c4_pack_rpn_targets"] = timeit(lambda: ops.pack_rpn_targets(cu, ip, bb, ROWS, COLS, 9))
    nbytes["c4_pack_rpn_targets"] = b4 * (n_anch * 18 + ROWS * COLS * (18 + 72 * 4))
    rois4 = d(np.stack([synth.random_rois(2000, ROWS, COLS, 400 + rank * b4 + i) for i in range(b4)]))
    gt64, gcls = d(gts.astype(np.float64) / 16), d(np.tile(np.arange(50, dtype=np.int32) % 20, (b4, 1)))
    ms["c4_label_rois_2000"] = timeit(lambda: ops.label_rois(rois4, gt64, gcls, n_gt, 21))
    nbytes["c4_label_rois_2000"] = b4 * 2000 * (8 + 8 + 84 + 640 + 4)
    del cu, ip, bb, rois4
    # C2: VGG16 detector post-processing, 21 classes, 320 rows per image, batch 64 (8 per GPU at 8 GPUs)
    b2 = 64 // world if world > 1 else 64
    rois2 = d(np.stack([synth.random_rois(320, 37, 62, 500 + rank * b2 + i) for i in range(b2)]))
    outs = [synth.detector_outputs(320, 21, 600 + rank * b2 + i) for i in range(b2)]
    oc, orr = d(np.stack([o[0] for o in outs])), d(np.stack([o[1] for o in outs]))
    ratio = d(np.full(b2, 1.6))
    ms["c2_det_postprocess"] = timeit(lambda: ops.det_postprocess(rois2, oc, orr, ratio, 20))
    # C5: ResNet-101 RoI layer forward + backward, 1024-ch stride-16 features, 2000 RoIs per image; 1 image per GPU
    # per launch (the curve of configs[4]) and, for the throughput figure, 8 images per GPU per launch
    n5 = 2000
    for b5 in (1, 8):
        feat = torch.randn((b5, ROWS, COLS, CHANNELS), device=dev)
        rois5 = d(np.stack([synth.random_rois(n5, ROWS, COLS, 7 + rank * 8 + i) for i in range(b5)]))
        gout = torch.randn((b5, n5, POOL, POOL, CHANNELS), device=dev)
        io = 4 * b5 * ROWS * COLS * CHANNELS + 8 * b5 * n5
        pooled = 4 * b5 * n5 * POOL * POOL * CHANNELS
        for mode in ("resize", "max"):
            arg = ops.roi_forward(feat, rois5, POOL, "max")[1] if mode == "max" else None
            k = "c5_roi_%s_b%d" % (mode, b5)
            ms[k + "_fwd"] = timeit(lambda: ops.roi_forward(feat, rois5, POOL, mode))
            ms[k + "_bwd"] = timeit(lambda: ops.roi_backward(gout, rois5, (b5, ROWS, COLS, CHANNELS), mode, arg))
            nbytes[k + "_fwd"] = nbytes[k + "_bwd"] = io + pooled * (2 if mode == "max" else 1)
            del arg
        # max mode with the one-byte arg-max (5 instead of 8 bytes per pooled element)
        code = ops.roi_forward(feat, rois5, POOL, "max", compact=True)[1]
        k = "c5_roi_max_u8arg_b%d" % b5
        ms[k + "_fwd"] = timeit(lambda: ops.roi_forward(feat, rois5, POOL, "max", compact=True))
        ms[k + "_bwd"] = timeit(lambda: ops.roi_backward(gout, rois5, (b5, ROWS, COLS, CHANNELS), "max", code))
        nbytes[k + "_fwd"] = nbytes[k + "_bwd"] = io + pooled + pooled // 4
        del code
        del feat, gout
    # SURVEY 8f-4: input pipeline on the device: 16 decoded 375x500 BGR images -> bicubic 600x800 + mirror + mean subtraction
    raw = torch.randint(0, 256, (16, 375, 500, 3), dtype=torch.uint8, device=dev)
    ms["f4_image_resize_preprocess_b16"] = timeit(lambda: ops.image_resize_cubic(raw, 600, 800, flip=True, mean=ops.IMAGENET_MEAN_BGR))
    nbytes["f4_image_resize_preprocess_b16"] = 16 * (375 * 500 * 3 + 600 * 800 * 3 * (1 + 4))
    del raw
    if want_dump:
        pairs = [synth.rpn_outputs(ROWS, COLS, len(voc), 1000 + i) for i in range(2)]
        regr1, cls1 = np.concatenate([p[1] for p in pairs]), np.concatenate([p[0] for p in pairs])
        dump["C1_regr"] = regr1
        dump["C1_dense"] = ops.decode_topk(d(regr1), d(cls1), voc, STRIDE, TOPK, want_dense=True)[4].cpu().numpy()
    sizes = {"c3_images": b3, "c4_images": b4, "c2_images": b2}
    return ms, nbytes, sizes, dump


def output_arrays(rois, scores, count, pooled):
    """What one step of the timed path returned, as float32 host arrays for --dump-outputs, so that two builds can be
    compared output for output on the same seeded inputs.  RoIs, scores and counts are kept whole (rows past an image's
    count are zero); the pooled features (4.1 GB at 64 images) as a fixed, seeded sample of POOLED_SAMPLE (image, RoI
    row) pairs, 25.7 MB, with the pairs in `pooled_sample_index`."""
    import torch
    b, m = pooled.shape[:2]
    pick = np.sort(np.random.default_rng(0).choice(b * m, size=min(POOLED_SAMPLE, b * m), replace=False))
    sample = pooled.reshape((b * m,) + tuple(pooled.shape[2:]))[torch.from_numpy(pick).to(pooled.device)]
    arrays = {"rois": rois, "scores": scores, "count": count, "pooled_sample": sample}
    arrays = {k: v.cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    arrays["pooled_sample_index"] = np.stack([pick // m, pick % m], axis=1).astype(np.float32)
    return arrays


def run_ours(args, rank, world, local_rank):
    import tempfile

    import torch
    import torch.distributed as dist
    from faster_rcnn_b200 import parallel, synth
    from faster_rcnn_b200.pipeline import ProposalRoiPipeline
    from faster_rcnn_b200.runtime import get_context

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (sm_100a); there is no CPU fallback. "
                         "Use --impl reference for the CPU arm.")
    torch.cuda.set_device(local_rank)
    numa_cores = parallel.bind_to_gpu_numa(physical_gpu_index(local_rank)) if world > 1 else None
    parallel.init_from_env("nccl")
    dev = torch.device("cuda", local_rank)
    ctx = get_context(local_rank)
    batch = args.images_per_gpu
    dims = anchor_dims()
    pipe = ProposalRoiPipeline(dims, STRIDE, TOPK, NMS_THRESH, MAX_BOXES, NUM_ROIS, POOL, "resize", device=local_rank)

    # synthetic inputs (seeded per global image index), resident in HBM, plus pinned host copies for e2e
    first = rank * batch
    pairs = [synth.rpn_outputs(ROWS, COLS, len(dims), 1000 + first + i) for i in range(batch)]
    cls_h = torch.from_numpy(np.concatenate([p[0] for p in pairs])).pin_memory()
    regr_h = torch.from_numpy(np.concatenate([p[1] for p in pairs])).pin_memory()
    gen = torch.Generator(device=dev).manual_seed(2000 + rank)
    feat = torch.randn((batch, ROWS, COLS, CHANNELS), generator=gen, device=dev, dtype=torch.float32)
    feat_h = torch.empty(feat.shape, dtype=torch.float32).pin_memory()
    feat_h.copy_(feat)
    cls, regr = cls_h.to(dev), regr_h.to(dev)
    ctx.reserve(256 << 20)

    gathered = {}

    def step(events=None):
        rois, scores, count = pipe_ops.proposals(regr, cls, dims, STRIDE, TOPK, NMS_THRESH, MAX_BOXES)
        padded, _ = pipe_ops.pad_rois(rois, count, NUM_ROIS)
        pending = None
        if world > 1:      # the path's only exchange: final RoIs + counts, one all-gather each per step, issued
            #                before the RoI layer (which needs only the local RoIs) so that NCCL runs next to it
            if "rois" not in gathered:
                gathered["rois"] = torch.empty((world * batch, MAX_BOXES, 4), dtype=torch.int16, device=dev)
                gathered["count"] = torch.empty((world * batch,), dtype=torch.int32, device=dev)
            _, _, pending = parallel.all_gather_rois(rois, count, gathered["rois"], gathered["count"], async_op=True)
        if events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        pooled = pipe_ops.roi_forward(feat, padded, POOL, "resize")
        if events is not None:
            e1.record()
            events.append((e0, e1))
        if pending is not None:
            pending.wait()
        return rois, scores, count, pooled

    from faster_rcnn_b200 import ops as pipe_ops

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput -------------------------------------------------------------------
    for _ in range(args.warmup):
        out = step()
    fence()
    count0 = out[2].cpu().numpy()
    sampler = ClockSampler(physical_gpu_index(local_rank)) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = ctx.launches
    events = []
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    start.record()
    for _ in range(args.steps):
        out = step(events)
    stop.record()
    fence()
    launches = ctx.launches - launches0
    ms = start.elapsed_time(stop)
    roi_ms = float(np.mean([a.elapsed_time(b) for a, b in events]))
    # with several GPUs only rank 0's own images are kept
    dumped = output_arrays(*out) if args.dump_outputs and rank == 0 else None
    del out

    # ---- end to end through the public API: pinned host inputs, H2D + compute + D2H every step -----------------
    for _ in range(max(1, min(args.warmup, 3))):
        res = pipe(cls_h, regr_h, feat_h)
    fence()
    e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    def exchange(rois, scores, count):
        if world > 1:
            parallel.all_gather_rois(rois, count, gathered["rois"], gathered["count"])

    e_start.record()
    for _ in range(args.steps):
        res = pipe(cls_h, regr_h, feat_h, on_device=exchange)
    e_stop.record()
    fence()
    e2e_ms = e_start.elapsed_time(e_stop)
    assert np.array_equal(res[2], count0), "e2e path and device path disagree"
    # the same public call when the backbone runs on this GPU and hands its feature map over as a CUDA tensor: only
    # the RPN head outputs (28 MB per 64 images instead of 655 MB) cross PCIe
    for _ in range(2):
        res = pipe(cls_h, regr_h, feat)
    fence()
    e_start.record()
    for _ in range(args.steps):
        res = pipe(cls_h, regr_h, feat, on_device=exchange)
    e_stop.record()
    fence()
    e2e_dev_ms = e_start.elapsed_time(e_stop)
    assert np.array_equal(res[2], count0), "device-feature e2e path and device path disagree"
    del res
    clocks = sampler.stop() if sampler else None
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        del dumped

    # ---- sustained window: >= 2 s of back-to-back steps (the GPU reaches its power cap), RoI kernel timed every 8th step
    sus_sampler = ClockSampler(physical_gpu_index(local_rank)) if rank == 0 else None
    if sus_sampler:
        sus_sampler.start()
    # every rank runs the SAME number of steps (each step holds a collective when world > 1): agree on it first
    per_step = torch.tensor([ms / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(per_step, op=dist.ReduceOp.MAX)
    sus_total = max(64, int(np.ceil(args.sustained_seconds * 1e3 / float(per_step.item()) / 64.0)) * 64)
    sus_events, sus_steps = [], 0
    fence()
    s_start, s_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_start.record()
    while sus_steps < sus_total:
        for i in range(64):
            step(sus_events if i % 8 == 0 else None)
        sus_steps += 64
    s_stop.record()
    fence()
    sus_ms = s_start.elapsed_time(s_stop)
    sus_roi_ms = float(np.mean([a.elapsed_time(b) for a, b in sus_events])) if sus_events else float("nan")
    sus_clocks = sus_sampler.stop() if sus_sampler else None

    # ---- the other BASELINE.json configs, timed live on every rank ------------------------------------------------------
    peak, peak_src = measured_peak()
    st_ms, st_bytes, st_sizes, dump = measure_stages(pipe_ops, dev, rank, world, peak, want_dump=(rank == 0 and world == 1))

    if world > 1:
        keys = sorted(st_ms)
        t = torch.tensor([ms, e2e_ms, roi_ms, e2e_dev_ms, sus_ms / max(sus_steps, 1), sus_roi_ms] + [st_ms[k] for k in keys],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = [float(v) for v in t.cpu()]
        ms, e2e_ms, roi_ms, e2e_dev_ms, sus_step_ms, sus_roi_ms = vals[:6]
        st_ms = dict(zip(keys, vals[6:]))
    else:
        sus_step_ms = sus_ms / max(sus_steps, 1)

    if rank == 0:
        total_images = world * batch * args.steps
        value = total_images / (ms / 1e3)
        e2e_value = total_images / (e2e_ms / 1e3)
        algo_bytes = batch * (4 * ROWS * COLS * CHANNELS + 8 * PADDED + 4 * PADDED * POOL * POOL * CHANNELS)
        achieved = algo_bytes / (roi_ms / 1e3) / 1e9
        achieved_sus = algo_bytes / (sus_roi_ms / 1e3) / 1e9
        stages = {}
        for k in sorted(st_ms):
            row = {"ms": round(st_ms[k], 5)}
            if k in st_bytes:
                row.update(algorithmic_bytes=int(st_bytes[k]), frac=round(st_bytes[k] / st_ms[k] / 1e6 / peak, 4))
            stages[k] = row
        stages["_sizes"] = dict(st_sizes, c5="1 and 8 images x 2000 RoIs per GPU and launch, 38x63x1024 f32 features",
                                note="per-GPU work (weak scaling); ms = max over ranks; frac = algorithmic bytes / ms / measured "
                                     "HBM copy peak for the HBM-bound stages; max-mode bytes count the int32 arg-max, the max_u8arg rows the one-byte one")
        stages["c5_img_per_s_fwd_bwd_resize"] = round(world * 1e3 / (st_ms["c5_roi_resize_b1_fwd"] + st_ms["c5_roi_resize_b1_bwd"]), 1)
        stages["c5_img_per_s_fwd_bwd_max"] = round(world * 1e3 / (st_ms["c5_roi_max_b1_fwd"] + st_ms["c5_roi_max_b1_bwd"]), 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": shared_config(batch, world),
            "notes": {"rois_per_image": int(count0[0]),
                      "timing": "CUDA events around K back-to-back steps after W warm-up steps (burst); `sustained` is the "
                                "same step repeated for >= %.1f s, where the GPU reaches its 1000 W power cap" % args.sustained_seconds,
                      "host_affinity": ("rank 0 bound to %d GPU-local cores" % len(numa_cores)) if numa_cores else "unbound"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": pipe.h2d_bytes(cls_h, regr_h, feat_h), "d2h_bytes_per_step": pipe.d2h_bytes(batch),
                    "note": "ProposalRoiPipeline.__call__ on pinned host arrays; RoIs/scores/counts return to the host, "
                            "pooled features stay on the device for the detector head as in the reference's TF graph",
                    "device_features": {"value": total_images / (e2e_dev_ms / 1e3), "unit": UNIT,
                                        "ms_per_step": e2e_dev_ms / args.steps,
                                        "h2d_bytes_per_step": pipe.h2d_bytes(cls_h, regr_h, feat),
                                        "d2h_bytes_per_step": pipe.d2h_bytes(batch),
                                        "note": "same call, feature map already on the device (GPU backbone): removes the "
                                                "9.8 MB/image copy of det_util.py:48-51"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "roi_fwd_kernel<RESIZE>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": roi_traffic_bytes(batch),
                         "algorithmic_bytes_per_launch": algo_bytes, "launch_ms": roi_ms, "peak_source": peak_src,
                         "kernel_share_of_step": roi_ms / (ms / args.steps),
                         "frac_sustained": achieved_sus / peak, "achieved_sustained": achieved_sus,
                         "launch_ms_sustained": sus_roi_ms},
            "sustained": {"seconds": sus_ms / 1e3, "steps": sus_steps, "value": world * batch / (sus_step_ms / 1e3),
                          "unit": UNIT, "ms_per_step": sus_step_ms, "clocks": sus_clocks},
            "stages": stages,
        }
        if world == 1 and not args.no_cpu_baseline:
            # separate process: never fork a process that holds a CUDA context
            dump_path = os.path.join(tempfile.gettempdir(), "frcnn_bench_decode_%d.npz" % os.getpid())
            np.savez(dump_path, **dump)
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                  "--warmup", "0", "--images-per-gpu", str(args.cpu_images), "--check-decode", dump_path],
                                 capture_output=True, text=True)
            try:
                os.unlink(dump_path)
            except OSError:
                pass
            try:
                ref = json.loads(res.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = dict(ref["cpu_baseline"], sample="%d images of the same workload, image-parallel "
                                            "fork pool of the numpy port of the reference (RoI layer = numpy restatement "
                                            "of TF-1.3 bilinear), %s" % (args.cpu_images, cpu_model()))
                line["stages"]["decode_check"] = ref.get("decode_check")
            except Exception as exc:      # the GPU line must still be printed
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                        "sample": "failed: %r %s" % (exc, res.stderr[-300:])}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--images-per-gpu", type=int, default=64)
    ap.add_argument("--cpu-images", type=int, default=128, help="bounded sample for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sustained-seconds", type=float, default=2.2, help="length of the power-capped window")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="--impl ours: after the timed steps, write the last step's RoIs, scores, counts and a seeded "
                         "sample of the pooled features to DIR/<name>.npy (float32); with several GPUs, those of "
                         "rank 0's own images")
    ap.add_argument("--check-decode", default="", help=argparse.SUPPRESS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours only")
        run_reference(args, rank, world if world == args.gpus else args.gpus)
        return
    if world != args.gpus:
        if args.gpus > 1 and world == 1:
            # convenience: re-launch under torchrun, one rank per GPU
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
            raise SystemExit(subprocess.call(cmd))
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
