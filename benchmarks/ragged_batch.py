"""Mixed-size batches: one padded launch with per-image extents against one launch per shape group.

64 images are drawn from the VOC shape distribution (img_wh of tests/golden/voc_gt_200.npz -> conv_dims_resnet), with
synthetic RPN heads (9 anchors) and 1024-channel features, and timed three ways:
  (a) ragged   one call on the batch padded to its largest extents, with `extents`;
  (b) grouped  one call per distinct conv shape (what the single-shape entry points need);
  (c) overhead the ragged entry with every extent full against the single-shape entry, 64 images at C1 (38 x 63).
Stages: proposals (k 8000 -> 300 and 12000 -> 2000), anchor labelling + packing of the RPN targets, and
ProposalRoiPipeline.run_device.  Each number is the median over `--reps` timed repetitions of CUDA events around
`--iters` back-to-back calls (host enqueue included, which is what a grouped batch pays for).  Prints one JSON line.

    python benchmarks/ragged_batch.py [--batch 64] [--iters 20] [--reps 7] [--seed 0]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()

    import torch
    from faster_rcnn_b200 import _build, ops, synth
    from faster_rcnn_b200.pipeline import ProposalRoiPipeline
    from oracle import frcnn_oracle as O
    if not torch.cuda.is_available():
        raise SystemExit("ragged_batch.py measures on the GPU; no CUDA device found")
    _build.build()
    dev = torch.device("cuda")
    g = np.load(os.path.join(ROOT, "tests", "golden", "voc_gt_200.npz"))
    rng = np.random.default_rng(args.seed)
    draw = rng.integers(0, len(g["img_wh"]), args.batch)
    wh = g["img_wh"][draw].astype(np.int32)
    shapes = [tuple(O.conv_dims_resnet(int(h), int(w))) for w, h in wh]
    ext_h = np.array(shapes, np.int32)
    rows, cols = (int(v) for v in ext_h.max(axis=0))
    dims = O.anchor_table([128, 256, 512])
    a = len(dims)

    cls = torch.zeros((args.batch, rows, cols, a), device=dev)
    regr = torch.zeros((args.batch, rows, cols, 4 * a), device=dev)
    for b, (r, c) in enumerate(shapes):
        pc, pr = synth.rpn_outputs(r, c, a, 1000 + b)
        cls[b, :r, :c], regr[b, :r, :c] = torch.from_numpy(pc[0]), torch.from_numpy(pr[0])
    feat = torch.randn((args.batch, rows, cols, 1024), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    ext = torch.from_numpy(ext_h).to(dev)
    gts = [synth.gt_boxes(int(rng.integers(1, 8)), int(w), int(h), 2000 + b) for b, (w, h) in enumerate(wh)]
    g_max = max(len(x) for x in gts)
    gt = np.zeros((args.batch, g_max, 4), np.float32)
    for b, x in enumerate(gts):
        gt[b, :len(x)] = np.array([v[1:] for v in x], np.float32)
    gt, n_gt = torch.from_numpy(gt).to(dev), torch.tensor([len(x) for x in gts], dtype=torch.int32, device=dev)
    wh_d = torch.from_numpy(wh).to(dev)

    groups = {}
    for b, s in enumerate(shapes):
        groups.setdefault(s, []).append(b)
    grouped = []
    for (r, c), idx in groups.items():
        ii = torch.tensor(idx, device=dev)
        grouped.append((r, c, cls[ii, :r, :c].contiguous(), regr[ii, :r, :c].contiguous(), feat[ii, :r, :c].contiguous(),
                        gt[ii].contiguous(), n_gt[ii].contiguous(), wh_d[ii].contiguous()))
    pipe = ProposalRoiPipeline(anchor_dims=dims)

    def label_pack(gt_, n_, wh_, r, c, e=None):
        cu, ip, bb, _ = ops.label_anchors(gt_, n_, wh_, r, c, dims, 16, extents=e)
        return ops.pack_rpn_targets(cu, ip, bb, r, c, a)

    work = {
        "proposals_8000_300": (lambda: ops.proposals(regr, cls, dims, 16, 8000, 0.7, 300, extents=ext),
                               lambda: [ops.proposals(q[3], q[2], dims, 16, 8000, 0.7, 300) for q in grouped]),
        "proposals_12000_2000": (lambda: ops.proposals(regr, cls, dims, 16, 12000, 0.7, 2000, extents=ext),
                                 lambda: [ops.proposals(q[3], q[2], dims, 16, 12000, 0.7, 2000) for q in grouped]),
        "label_pack": (lambda: label_pack(gt, n_gt, wh_d, rows, cols, ext),
                       lambda: [label_pack(q[5], q[6], q[7], q[0], q[1]) for q in grouped]),
        "run_device": (lambda: pipe.run_device(cls, regr, feat, extents=ext),
                       lambda: [pipe.run_device(q[2], q[3], q[4]) for q in grouped]),
    }

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
        return float(np.median(ms)), float(min(ms)), float(max(ms))

    res = {}
    for name, (rag, grp) in work.items():
        r_ms, g_ms = timed(rag), timed(grp)
        res[name] = {"ragged_ms": r_ms, "grouped_ms": g_ms, "grouped_over_ragged": g_ms[0] / r_ms[0]}

    # (c) full extents against the single-shape entry at C1
    c1 = (38, 63)
    p = [synth.rpn_outputs(c1[0], c1[1], a, 3000 + b) for b in range(args.batch)]
    cls1 = torch.from_numpy(np.concatenate([x[0] for x in p])).to(dev)
    regr1 = torch.from_numpy(np.concatenate([x[1] for x in p])).to(dev)
    feat1 = torch.randn((args.batch, c1[0], c1[1], 1024), device=dev)
    ext1 = torch.tensor([c1] * args.batch, dtype=torch.int32, device=dev)
    overhead = {
        "proposals_8000_300": (lambda: ops.proposals(regr1, cls1, dims, 16, 8000, 0.7, 300, extents=ext1),
                               lambda: ops.proposals(regr1, cls1, dims, 16, 8000, 0.7, 300)),
        "proposals_12000_2000": (lambda: ops.proposals(regr1, cls1, dims, 16, 12000, 0.7, 2000, extents=ext1),
                                 lambda: ops.proposals(regr1, cls1, dims, 16, 12000, 0.7, 2000)),
        "run_device": (lambda: pipe.run_device(cls1, regr1, feat1, extents=ext1),
                       lambda: pipe.run_device(cls1, regr1, feat1)),
    }
    res_c = {}
    for name, (rag, uni) in overhead.items():
        u1, r1 = timed(uni), timed(rag)
        u2, r2 = timed(uni), timed(rag)                # alternated twice: the spread of either is the noise floor
        res_c[name] = {"uniform_ms": [u1[0], u2[0]], "ragged_full_ms": [r1[0], r2[0]]}
    print(json.dumps({"metric": "ragged_batch", "batch": args.batch, "padded_map": [rows, cols],
                      "distinct_shapes": len(groups), "valid_cell_share": float(ext_h.prod(axis=1).sum()) / (args.batch * rows * cols),
                      "iters": args.iters, "reps": args.reps, "a_vs_b": res, "c_full_extents_at_C1": res_c,
                      "gpu": _gpu_record()}))


if __name__ == "__main__":
    main()
