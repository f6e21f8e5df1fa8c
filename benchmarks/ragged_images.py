"""Mixed-size batches at both ends of an RPN step: one ragged call against one call per image.

  preprocess   64 images whose resized sizes are drawn from img_wh of tests/golden/voc_gt_200.npz; their raw sizes have a
               long side of 500 (VOC's raw size) and their pixels are synthetic natural images.  Bicubic resize + mirror
               (every other image) + mean subtraction to float32:
                 ragged      one `image_resize_cubic_ragged` call into the padded batch;
                 per_image   one `image_resize_cubic` call per image;
                 per_pair    one `image_resize_cubic` call per distinct (source size, target size, mirror).
               Kernel time is timed on sources already on the device.  The host-to-device upload is timed on its own:
               `pack_images` (one pinned buffer, one copy) against one upload per image.
  rpn_losses   loss + gradients on 64 padded RPN maps of the same VOC sizes (conv_dims_resnet): one
               `rpn_losses(..., extents=)` call against one call per image on the cropped inputs.
  overhead     every extent full against the uniform entry at equal sizes (375 x 500 -> 600 x 800, map 38 x 50).
Each number is the median over `--reps` timed repetitions of CUDA events around `--iters` back-to-back calls (host
enqueue included, which is what a per-image loop pays for).  Prints one JSON line.

    python benchmarks/ragged_images.py [--batch 64] [--iters 20] [--reps 7] [--seed 0]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def _natural(h, w, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 127 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 23.0) + 30 * np.sin((xx + yy) / 5.0)
    return np.clip(base[:, :, None] + rng.normal(0, 12, (h, w, 3)) + np.array([10, -20, 5]), 0, 255).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()

    import torch
    from faster_rcnn_b200 import _build, ops
    from faster_rcnn_b200.runtime import get_context
    from oracle import frcnn_oracle as O
    from ragged_batch import _gpu_record
    if not torch.cuda.is_available():
        raise SystemExit("ragged_images.py measures on the GPU; no CUDA device found")
    _build.build()
    dev = torch.device("cuda")
    ctx = get_context()
    mean = ops.IMAGENET_MEAN_BGR
    g = np.load(os.path.join(ROOT, "tests", "golden", "voc_gt_200.npz"))
    rng = np.random.default_rng(args.seed)
    wh = g["img_wh"][rng.integers(0, len(g["img_wh"]), args.batch)].astype(np.int64)
    dst = [(int(h), int(w)) for w, h in wh]
    raw = [(int(round(h * 500 / max(h, w))), int(round(w * 500 / max(h, w)))) for h, w in dst]
    flips = [b % 2 == 1 for b in range(args.batch)]
    srcs = [_natural(r[0], r[1], b) for b, r in enumerate(raw)]
    height, width = max(d[0] for d in dst), max(d[1] for d in dst)

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

    # ---- preprocess -------------------------------------------------------------------------------------------------
    packed, offsets, sizes = ops.pack_images(srcs)
    geom = torch.cat([sizes, torch.tensor(dst, dtype=torch.int32, device=dev)], dim=1).contiguous()
    flip_d = torch.tensor(flips, dtype=torch.uint8, device=dev)
    out = (None, torch.empty((args.batch, height, width, 3), dtype=torch.float32, device=dev))
    per_src = [torch.from_numpy(s[None]).to(dev) for s in srcs]
    pairs = {}
    for b, key in enumerate(zip(raw, dst, flips)):
        pairs.setdefault(key, []).append(b)
    pair_src = [(k, torch.cat([per_src[b] for b in idx])) for k, idx in pairs.items()]

    def ragged():
        ops.image_resize_cubic_ragged(packed, offsets, geom, height, width, flip=flip_d, mean=mean, want_u8=False, out=out)

    def per_image():
        for b in range(args.batch):
            ops.image_resize_cubic(per_src[b], dst[b][0], dst[b][1], flip=flips[b], mean=mean, want_u8=False)

    def per_pair():
        for (_, d, f), s in pair_src:
            ops.image_resize_cubic(s, d[0], d[1], flip=f, mean=mean, want_u8=False)

    valid_bytes = sum(h * w for h, w in dst) * 3 * 4
    pre = {"ragged_ms": timed(ragged), "per_image_ms": timed(per_image), "per_pair_ms": timed(per_pair),
           "h2d_pack_images_ms": timed(lambda: ops.pack_images(srcs)),
           "h2d_per_image_ms": timed(lambda: [ctx.to_device(s[None]) for s in srcs]),
           "distinct_pairs": len(pairs), "padded_shape": [height, width],
           "source_bytes": int(sum(s.nbytes for s in srcs)), "f32_valid_bytes": valid_bytes,
           "f32_padded_bytes": args.batch * height * width * 3 * 4}
    pre["per_image_over_ragged"] = pre["per_image_ms"][0] / pre["ragged_ms"][0]
    pre["per_pair_over_ragged"] = pre["per_pair_ms"][0] / pre["ragged_ms"][0]

    # ---- rpn_losses + gradients -------------------------------------------------------------------------------------
    a = 9
    ext_h = np.array([O.conv_dims_resnet(h, w) for h, w in dst], np.int32)
    rows, cols = (int(v) for v in ext_h.max(axis=0))
    n = rows * cols * a

    def rpn_inputs(b, r, c):
        q = np.random.default_rng(100 + b)
        return [q.integers(0, 2, (b, r * c * a), dtype=np.uint8), q.integers(0, 2, (b, r * c * a), dtype=np.uint8),
                q.standard_normal((b, r * c * a, 4)).astype(np.float32), q.uniform(0.01, 0.99, (b, r * c * a)).astype(np.float32),
                q.standard_normal((b, r * c * a, 4)).astype(np.float32)]

    padded = [torch.from_numpy(x).to(dev) for x in rpn_inputs(args.batch, rows, cols)]
    ext = torch.from_numpy(ext_h).to(dev)
    crops = []
    for b, (r, c) in enumerate(ext_h):
        crops.append([t[b:b + 1].reshape((1, rows, cols, a) + t.shape[2:])[:, :r, :c].reshape((1, -1) + t.shape[2:]).contiguous()
                      for t in padded])
    losses = {"ragged_ms": timed(lambda: ops.rpn_losses(*padded, want_grad=True, extents=ext, padded_shape=(rows, cols))),
              "per_image_ms": timed(lambda: [ops.rpn_losses(*x, want_grad=True) for x in crops]),
              "padded_map": [rows, cols], "valid_anchor_share": float(ext_h.prod(axis=1).sum()) / (args.batch * rows * cols)}
    losses["per_image_over_ragged"] = losses["per_image_ms"][0] / losses["ragged_ms"][0]

    # ---- overhead: full extents against the uniform entry -----------------------------------------------------------
    imgs = np.stack([_natural(375, 500, 300 + b) for b in range(args.batch)])
    imgs_d = torch.from_numpy(imgs).to(dev)
    p1, o1, s1 = ops.pack_images([imgs_d[b] for b in range(args.batch)])
    g1 = torch.cat([s1, torch.tensor([[600, 800]] * args.batch, dtype=torch.int32, device=dev)], dim=1).contiguous()
    f1 = torch.ones((args.batch,), dtype=torch.uint8, device=dev)
    out1 = (None, torch.empty((args.batch, 600, 800, 3), dtype=torch.float32, device=dev))
    l1 = [torch.from_numpy(x).to(dev) for x in rpn_inputs(args.batch, 38, 50)]
    e1 = torch.tensor([[38, 50]] * args.batch, dtype=torch.int32, device=dev)
    work = {
        "preprocess": (lambda: ops.image_resize_cubic(imgs_d, 600, 800, flip=True, mean=mean, want_u8=False),
                       lambda: ops.image_resize_cubic_ragged(p1, o1, g1, 600, 800, flip=f1, mean=mean, want_u8=False, out=out1)),
        "rpn_losses": (lambda: ops.rpn_losses(*l1, want_grad=True),
                       lambda: ops.rpn_losses(*l1, want_grad=True, extents=e1, padded_shape=(38, 50))),
    }
    overhead = {}
    for name, (uni, rag) in work.items():
        u1, r1 = timed(uni), timed(rag)
        u2, r2 = timed(uni), timed(rag)                # alternated twice: the spread of either is the noise floor
        overhead[name] = {"uniform_ms": [u1[0], u2[0]], "ragged_full_ms": [r1[0], r2[0]]}
    print(json.dumps({"metric": "ragged_images", "batch": args.batch, "iters": args.iters, "reps": args.reps,
                      "preprocess": pre, "rpn_losses_grad": losses, "full_extents_overhead": overhead,
                      "gpu": _gpu_record()}))


if __name__ == "__main__":
    main()
