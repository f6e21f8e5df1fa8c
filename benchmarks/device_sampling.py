"""Training mini-batch draws on the device (ops.sample_rpn_ / ops.sample_det) against the host draws that replay the
reference's RNG streams.

  det_targets   DetTrainingPipeline.targets, 128 images at C4 shapes (38 x 63 x 9 anchors, 12000 -> NMS 2000 -> 64 RoIs),
                host draw (default) vs device draw (state=).
  rpn_targets   64 VOC-shaped mixed-size images (img_wh of tests/golden/voc_gt_200.npz): rpn_y_true_ragged (host draw +
                pack + D2H of the Keras targets) vs rpn_targets_device (device draw, targets stay on the device); and
                the cost of labelling through the ragged entry on a uniform batch (64 images at 38 x 63).
  kernels       each sampler kernel next to the labelling kernel it follows, for the same batch.

Every number is the median over `--reps` repetitions of CUDA events around `--iters` back-to-back calls (host work and
enqueue included; each call of the host-draw paths ends in its own synchronisation).  Prints one JSON line with the card
name, power limit and clocks read in the same run.

    python benchmarks/device_sampling.py [--iters 20] [--reps 7]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu_record():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return dict(zip(q.split(","), (v.strip() for v in out[0].split(",")))) if out else {}
    except (OSError, subprocess.SubprocessError):
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()

    import torch
    from faster_rcnn_b200 import _build, ops, rpn_util, synth
    from faster_rcnn_b200.pipeline import DetTrainingPipeline
    from faster_rcnn_b200.util import get_bbox_coords
    from helpers import FakeImage
    from oracle import frcnn_oracle as O
    if not torch.cuda.is_available():
        raise SystemExit("device_sampling.py measures on the GPU; no CUDA device found")
    _build.build()
    dims = O.anchor_table([128, 256, 512])
    a = len(dims)

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.iters):
                fn()
            t1.record()
            t1.synchronize()
            ms.append(t0.elapsed_time(t1) / args.iters)
        return float(np.median(ms))

    res = {}
    # ---- detector targets at C4: 128 images, 50 GT each
    b = 128
    heads = [synth.rpn_outputs(38, 63, a, 500 + i, clustered=True) for i in range(b)]
    cls = torch.from_numpy(np.concatenate([h[0] for h in heads])).cuda()
    regr = torch.from_numpy(np.concatenate([h[1] for h in heads])).cuda()
    images = [FakeImage("c4_%d" % i, 1000, 600, synth.gt_boxes(50, 1000, 600, 600 + i)) for i in range(b)]
    pipe = DetTrainingPipeline(synth.VOC_CLASS_MAPPING, dims)
    gt = pipe.ground_truth(images)
    state = ops.sampler_state(0)
    host_ms = timed(lambda: pipe.targets(cls, regr, *gt))
    dev_ms = timed(lambda: pipe.targets(cls, regr, *gt, state=state))
    host_ms2 = timed(lambda: pipe.targets(cls, regr, *gt))
    dev_ms2 = timed(lambda: pipe.targets(cls, regr, *gt, state=state))
    res["det_targets_c4_128"] = {"host_draw_ms": [host_ms, host_ms2], "device_draw_ms": [dev_ms, dev_ms2]}

    # kernels of the same batch: label_rois vs sample_det, label_anchors vs sample_rpn_
    rois, _, count = ops.proposals(regr, cls, dims, 16, 12000, 0.7, 2000)
    l_rois, y_cls, y_tr, _, m = ops.label_rois(rois, *gt, 21, n_roi=count)
    found = (y_cls[:, :, -1] == 0).to(torch.uint8)
    gt_px = np.stack([get_bbox_coords(img.gt_boxes) for img in images]).astype(np.float32)
    gt_px, n_gt = torch.from_numpy(gt_px).cuda(), torch.full((b,), 50, dtype=torch.int32, device="cuda")
    wh = torch.tensor([[1000, 600]] * b, dtype=torch.int32, device="cuda")
    cu, ip, bb, counts = ops.label_anchors(gt_px, n_gt, wh, 38, 63, dims, 16)
    cu_work = cu.clone()
    res["kernels_128_images"] = {
        "label_rois_ms": timed(lambda: ops.label_rois(rois, *gt, 21, n_roi=count)),
        "sample_det_ms": timed(lambda: ops.sample_det(found, m, 64, state)),
        "label_anchors_ms": timed(lambda: ops.label_anchors(gt_px, n_gt, wh, 38, 63, dims, 16)),
        "sample_rpn_ms": timed(lambda: ops.sample_rpn_(cu_work.copy_(cu), ip, counts, state)),
        "copy_can_use_ms": timed(lambda: cu_work.copy_(cu)),
        "usable_per_image_mean": float(counts.sum(dim=1).float().mean()),
    }

    # ---- RPN targets of 64 VOC-shaped mixed-size images
    g = np.load(os.path.join(ROOT, "tests", "golden", "voc_gt_200.npz"))
    rng = np.random.default_rng(0)
    draw = rng.integers(0, len(g["img_wh"]), 64)
    voc = [FakeImage("v%d" % i, int(g["img_wh"][j][0]), int(g["img_wh"][j][1]),
                     synth.gt_boxes(int(rng.integers(1, 8)), int(g["img_wh"][j][0]), int(g["img_wh"][j][1]), 700 + i))
           for i, j in enumerate(draw)]
    mgr = rpn_util.RpnTrainingManager(O.conv_dims_resnet, 16, preprocess_func=None, anchor_dims=dims)
    rag_host = timed(lambda: mgr.rpn_y_true_ragged(voc))
    rag_dev = timed(lambda: mgr.rpn_targets_device(voc, state))
    rag_host2 = timed(lambda: mgr.rpn_y_true_ragged(voc))
    rag_dev2 = timed(lambda: mgr.rpn_targets_device(voc, state))
    res["rpn_targets_voc_mixed_64"] = {"rpn_y_true_ragged_ms": [rag_host, rag_host2],
                                       "rpn_targets_device_ms": [rag_dev, rag_dev2],
                                       "distinct_shapes": len({tuple(O.conv_dims_resnet(i.height, i.width)) for i in voc})}
    # ragged labelling on a uniform batch: 64 images at 38 x 63
    uni = [FakeImage("u%d" % i, 1000, 600, synth.gt_boxes(5, 1000, 600, 800 + i)) for i in range(64)]
    ext_u = torch.tensor([[38, 63]] * 64, dtype=torch.int32, device="cuda")

    def uniform_then_sample():
        c_, i_, _, k_ = mgr._label_batch(uni)
        ops.sample_rpn_(c_, i_, k_, state)

    def ragged_then_sample():
        c_, i_, _, k_ = mgr._label_batch(uni, ext_u, (38, 63))
        ops.sample_rpn_(c_, i_, k_, state, extents=ext_u, padded_shape=(38, 63), n_anchors=a)
    u1, r1, u2, r2 = timed(uniform_then_sample), timed(ragged_then_sample), timed(uniform_then_sample), timed(ragged_then_sample)
    res["rpn_label_sample_uniform_64_c1"] = {"uniform_entry_ms": [u1, u2], "ragged_entry_ms": [r1, r2],
                                             "rpn_targets_device_ms": timed(lambda: mgr.rpn_targets_device(uni, state))}
    print(json.dumps({"metric": "device_sampling", "iters": args.iters, "reps": args.reps, "results": res,
                      "gpu": _gpu_record()}))


if __name__ == "__main__":
    main()
