#!/usr/bin/env python
"""Randomised GPU-vs-oracle parity sweep (not part of pytest; run on the GPU box):

    python benchmarks/fuzz_parity.py [--cases 300] [--seed 0]

Draws shapes / thresholds / limits the fixed test parametrisations do not cover (NMS stopping inside a tile, 1-box
inputs, heavy ties, thresholds at 0 and 1 and off the p/q ratios, NMS boxes with negative, invalid or near-16000
coordinates, odd channel counts and pool sizes, ragged batches, RoI labelling at K up to 128 and 256 GT boxes,
detector post-processing at K up to 128, M up to 1024, any max_boxes and 'bg' first, last or in the middle) and
compares every result bit for bit with the oracle (resize-mode RoI backward: 1e-5 relative; log()-based regression
targets: 1 float32 ulp).  Prints one JSON summary line."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from faster_rcnn_b200 import ops, synth          # noqa: E402
from oracle import frcnn_oracle as O             # noqa: E402
from oracle import roi_oracle as R               # noqa: E402


def dev(x, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).cuda()


def host(t):
    return t.cpu().numpy()


def case_nms(rng):
    n = int(rng.choice([1, 2, 63, 64, 65, 200, 1000, 3000]))
    span = int(rng.choice([20, 60, 200]))
    # offsets: non-negative (16-bit packed pair test), negative, or around 16000 (both leave the packed test)
    dx, dy = (int(rng.choice([0, 0, -int(rng.integers(1, 60)), 16000 - span - int(rng.integers(0, 60))])) for _ in range(2))
    x1, y1 = dx + rng.integers(0, span, n), dy + rng.integers(0, span, n)
    w, h = rng.integers(1, 41, n), rng.integers(1, 41, n)
    if rng.random() < 0.3:                                      # invalid boxes: a side in [-11, 0], areas <= 0
        bad = np.where(rng.random(n) < 0.05 + rng.random() * 0.3)[0]
        side, in_x = rng.integers(-11, 1, len(bad)), rng.random(len(bad)) < 0.5
        w[bad[in_x]], h[bad[~in_x]] = side[in_x], side[~in_x]
    # every area, intersection and pairwise area sum stays far inside int16: the oracle's arithmetic does not wrap
    boxes = np.stack([x1, y1, x1 + w - 1, y1 + h - 1], 1).astype(np.int16)
    if rng.random() < 0.3:                                      # heavy duplicates -> many exact-threshold / IoU 1 pairs
        boxes = boxes[rng.integers(0, max(1, n // 4), n)]
    probs = rng.permutation(n).astype(np.float32) / n if rng.random() < 0.7 else rng.integers(0, 5, n).astype(np.float32)
    # ratios p/q take the integer pair tests, the others the fixed-point screen (0 < t < 1) or the exact predicate
    thresh = float(rng.choice([0.0, 0.3, 0.5, 0.7, 0.999, 1.0, 0.65432, 0.71234, np.nextafter(0.7, 1.0),
                               np.nextafter(0.7, 0.0), 0.3141, 1e-7, -0.5, 1.5]))
    max_boxes = int(rng.choice([1, 2, 7, 64, 65, 300, 2000]))
    pick = O.greedy_nms(boxes, probs, thresh, max_boxes)
    ki, kc, kb, ks = ops.nms_i16(dev(boxes[None]), dev(probs[None]), None, thresh, max_boxes)
    m = int(host(kc)[0])
    ok = m == len(pick) and np.array_equal(host(ki)[0, :m], pick) and np.array_equal(host(kb)[0, :m], boxes[pick])
    return ok, dict(kind="nms", n=n, thresh=thresh, max_boxes=max_boxes)


def _scores(rng, shape):
    """objectness of many shapes: the rank-uniform synthetic ones, and arrays that stress proposals_kernel's bucket window
    ([2^-32, 1), 64 buckets per octave): logits, saturated sigmoids, tiny values, few distinct values, narrow bands."""
    n = int(np.prod(shape))
    u = (rng.permutation(n).astype(np.float64) + 0.5) / n
    kind = int(rng.integers(0, 8))
    if kind == 0:
        v = (u - rng.random()) * float(rng.choice([4.0, 30.0, 200.0]))                    # logits
    elif kind == 1:
        v = 1.0 / (1.0 + np.exp(-(u - rng.random()) * float(rng.choice([10.0, 40.0, 120.0]))))   # sigmoid, saturating
    elif kind == 2:
        v = u * float(rng.choice([1e-12, 1e-6, 1e-3]))
    elif kind == 3:
        v = np.minimum(u * float(rng.choice([1.2, 2.0, 8.0])), 1.0)                       # many exact 1.0
    elif kind == 4:
        v = float(rng.choice([0.3, 0.75, 0.999])) + u * float(rng.choice([1e-6, 1e-4, 1e-2]))   # one or two buckets
    elif kind == 5:
        v = np.round(u * int(rng.choice([1, 2, 7, 100]))) / 100.0                          # few distinct values incl. 0
    elif kind == 6:
        v = np.exp(-u * float(rng.choice([5.0, 30.0, 80.0])))                             # log-uniform over many octaves
    else:
        v = u
    return v.astype(np.float32).reshape(shape)


def case_proposals(rng):
    rows, cols = int(rng.integers(1, 40)), int(rng.integers(1, 70))
    scales = [128, 256, 512] if rng.random() < 0.6 else [16, 32, 64, 128, 256, 512]
    dims = O.anchor_table(scales)
    b = int(rng.choice([1, 1, 1, 2, 5, 20]))
    pairs = [synth.rpn_outputs(rows, cols, len(dims), int(rng.integers(1 << 30)), clustered=bool(rng.random() < 0.5)) for _ in range(b)]
    cls, regr = np.concatenate([p[0] for p in pairs]), np.concatenate([p[1] for p in pairs])
    if rng.random() < 0.6:
        cls = np.stack([_scores(rng, cls.shape[1:]) for _ in range(b)])
    k = int(rng.choice([1, 50, 1024, 2049, 8000, 12000, 16384]))
    max_boxes = int(rng.choice([1, 10, 300, 2000]))
    boxes, scores_k, index, cnt, dense = [host(t) for t in ops.decode_topk(dev(regr), dev(cls), dims, 16, k, want_dense=True)]
    rois, scores, count = ops.proposals(dev(regr), dev(cls), dims, 16, k, 0.7, max_boxes)
    rois, scores, count = host(rois), host(scores), host(count)
    ok = True
    for i in range(b):
        wb, wp, widx = O.topk_proposals(dense[i].copy(), cls[i].reshape(-1), k)
        n = int(cnt[i])
        ok = ok and n == len(wb) and np.array_equal(index[i, :n], widx) and np.array_equal(boxes[i, :n], wb) \
            and np.array_equal(scores_k[i, :n], wp) and bool(np.all(index[i, n:] == -1))
        pick = O.greedy_nms(wb, wp, 0.7, max_boxes) if len(wb) else np.zeros(0, np.int64)
        m = int(count[i])
        ok = ok and m == len(pick) and np.array_equal(rois[i, :m], wb[pick]) and np.array_equal(scores[i, :m], wp[pick])
    return ok, dict(kind="proposals", rows=rows, cols=cols, a=len(dims), k=k, max_boxes=max_boxes, batch=b)


def case_roi(rng):
    h, w = int(rng.integers(1, 40)), int(rng.integers(1, 64))
    c = int(rng.choice([4, 20, 64, 128, 260, 384, 512, 1024]))
    n, b = int(rng.choice([1, 3, 33, 64, 300])), int(rng.choice([1, 2, 5]))
    pool = int(rng.choice([1, 3, 7, 7, 7, 9, 14]))
    if n * b * pool * pool * c > 40e6:
        n = max(1, int(40e6 // (b * pool * pool * c)))
    feat = rng.standard_normal((b, h, w, c), dtype=np.float32)
    if rng.random() < 0.5:
        feat = np.round(feat)                                   # ties for the max mode
    x1, y1 = rng.integers(0, w, (b, n)), rng.integers(0, h, (b, n))
    rois = np.stack([x1, y1, np.minimum(w, x1 + 1 + rng.integers(0, w, (b, n))), np.minimum(h, y1 + 1 + rng.integers(0, h, (b, n)))], 2).astype(np.int16)
    gout = rng.standard_normal((b, n, pool, pool, c), dtype=np.float32)
    out = host(ops.roi_forward(dev(feat), dev(rois), pool, "resize"))
    g = host(ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "resize"))
    mo, ma = ops.roi_forward(dev(feat), dev(rois), pool, "max")
    gm = host(ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "max", argmax=ma))
    ok = True
    for i in range(b):
        ok &= np.array_equal(out[i], R.roi_resize_fwd(feat[i], rois[i], pool))
        want = R.roi_resize_bwd(gout[i], rois[i], (h, w, c))
        ok &= bool(np.abs(g[i] - want).max() <= 1e-5 * max(np.abs(want).max(), 1e-30))
        wo, wa = R.roi_max_fwd(feat[i], rois[i], pool)
        ok &= np.array_equal(host(mo)[i], wo) and np.array_equal(host(ma)[i], wa)
        wm = R.roi_max_bwd(gout[i], wa, (h, w, c))
        if n < 256:                                             # one warp per block list: the oracle's order, bit for bit
            ok &= np.array_equal(gm[i], wm)
        else:                                                   # sliced lists: re-associated (fixed order)
            ok &= bool(np.abs(gm[i] - wm).max() <= 1e-5 * max(np.abs(wm).max(), 1e-30))
    if ops.roi_compact_supported(h, w, c, pool):                # one-byte arg-max: same outputs, same gradient
        co, cc = ops.roi_forward(dev(feat), dev(rois), pool, "max", compact=True)
        g8 = ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "max", argmax=cc)
        ok &= bool(torch.equal(co, mo))
        ok &= bool((g8 - torch.from_numpy(gm).cuda()).abs().max().item() <= 1e-5 * max(float(np.abs(gm).max()), 1e-30))
        dy, dx = host(cc).astype(np.int64) >> 4, host(cc).astype(np.int64) & 15
        for i in range(b):
            x1r, y1r = rois[i, :, 0].astype(np.int64), rois[i, :, 1].astype(np.int64)
            hr, wr = rois[i, :, 3].astype(np.int64) - y1r, rois[i, :, 2].astype(np.int64) - x1r
            ya = y1r[:, None] + (np.arange(pool)[None, :] * hr[:, None]) // pool
            xa = x1r[:, None] + (np.arange(pool)[None, :] * wr[:, None]) // pool
            flat = (ya[:, :, None, None] + dy[i]) * w + xa[:, None, :, None] + dx[i]
            ok &= np.array_equal(flat, host(ma)[i])
    return bool(ok), dict(kind="roi", h=h, w=w, c=c, n=n, b=b, pool=pool)


def case_image(rng):
    from oracle import image_oracle as IO
    sh, sw = int(rng.integers(1, 120)), int(rng.integers(1, 160))
    dh, dw = int(rng.integers(1, 200)), int(rng.integers(1, 260))
    cn, b, flip = int(rng.choice([1, 3, 3, 4])), int(rng.choice([1, 2])), bool(rng.random() < 0.5)
    imgs = rng.integers(0, 256, (b, sh, sw, cn), dtype=np.uint8)
    mean = [103.939, 116.779, 123.68, 1.5][:cn]
    u8, f32 = ops.image_resize_cubic(dev(imgs), dh, dw, flip=flip, mean=mean)
    ok = True
    for i in range(b):
        want = IO.resize_cubic_u8(imgs[i], dw, dh, flip=flip)
        ok &= np.array_equal(host(u8)[i], want) and np.array_equal(host(f32)[i], IO.preprocess_bgr(want, mean).astype(np.float32))
    return bool(ok), dict(kind="image", src=(sh, sw), dst=(dh, dw), cn=cn, flip=flip)


def case_labels(rng):
    rows, cols = int(rng.integers(2, 40)), int(rng.integers(2, 64))
    dims = O.anchor_table([128, 256, 512])
    W, H = cols * 16, rows * 16
    g = int(rng.choice([1, 2, 7, 50]))
    gts = np.array([x[1:] for x in synth.gt_boxes(g, max(W, 64), max(H, 64), int(rng.integers(1 << 30)))], np.float32)
    cu, ip, bb, _ = ops.label_anchors(dev(gts[None]), dev(np.array([g], np.int32)), dev(np.array([[W, H]], np.int32)), rows, cols, dims, 16)
    wc, wp, wb = O.label_anchors(W, H, gts, rows, cols, dims, 16)
    ok = np.array_equal(host(cu)[0] == 1, wc) and np.array_equal(host(ip)[0] == 1, wp)
    diff = np.abs(host(bb)[0] - wb)
    ok &= bool(np.all(diff <= 2e-6 * np.maximum(np.abs(wb), 1.0)))       # log() in the targets: <= 1 ulp after the f32 store
    return bool(ok), dict(kind="labels", rows=rows, cols=cols, g=g)


def _ulp_close(got, want, max_ulp=1):
    gi, wi = np.ascontiguousarray(got, np.float32).view(np.int32).astype(np.int64), np.ascontiguousarray(want, np.float32).view(np.int32).astype(np.int64)
    gi = np.where(gi < 0, -(gi & 0x7fffffff), gi)
    wi = np.where(wi < 0, -(wi & 0x7fffffff), wi)
    return got.shape == want.shape and (got.size == 0 or int(np.abs(gi - wi).max()) <= max_ulp)


def case_label_rois(rng):
    rows, cols = int(rng.integers(4, 40)), int(rng.integers(4, 64))
    n, g = int(rng.choice([1, 17, 300, 1023, 1025, 2000])), int(rng.choice([1, 3, 12, 50, 256]))
    k = int(rng.choice([2, 21, 81, 128]))
    rois = synth.random_rois(n, rows, cols, int(rng.integers(1 << 30)))
    gts = synth.gt_boxes(g, cols * 16, rows * 16, int(rng.integers(1 << 30)))
    gt64 = np.array([[v * (1 / 16) for v in x[1:]] for x in gts], np.float64)
    gidx = (rng.permutation(g) % (k - 1)).astype(np.int32)     # GT classes covering 0..K-2
    out = ops.label_rois(dev(rois[None]), dev(gt64[None]), dev(gidx[None]), dev(np.array([g], np.int32)), k)
    e_rois, w_cls, w_tr = O.label_rois(rois, gt64, gidx, k)
    m = int(host(out[4])[0])
    ok = m == len(e_rois) and np.array_equal(host(out[0])[0, :m], e_rois) and np.array_equal(host(out[1])[0, :m], w_cls)
    ok = ok and _ulp_close(host(out[2])[0, :m], w_tr)           # log() in the targets: <= 1 ulp after the f32 store
    return bool(ok), dict(kind="label_rois", n=n, g=g, k=k)


def case_postprocess(rng):
    k = int(rng.choice([21, 33, 81, 128]))
    m = int(rng.choice([64, 128, 320, 1000, 1024, int(rng.integers(1, 1025))]))
    bg = int(rng.choice([k - 1, k - 1, 0, k // 2]))
    max_boxes = int(rng.choice([1, 2, 7, 300, 2000]))
    rois = synth.random_rois(m, 37, 62, int(rng.integers(1 << 30)))
    oc, orr = synth.detector_outputs(m, k, int(rng.integers(1 << 30)))
    ratio, thr = float(rng.choice([0.75, 1.0, 1.6, 2.2])), float(rng.choice([0.0, 0.2, 0.5]))
    boxes, probs, dcls, count = ops.det_postprocess(dev(rois[None]), dev(oc[None]), dev(orr[None]), dev(np.array([ratio])), bg,
                                                    16, thr, max_boxes=max_boxes)
    ocl = oc.copy()
    if bg != k - 1:                                             # class K-1 has no regression columns: dropped like 'bg'
        drop = np.argmax(ocl, axis=1) == k - 1
        ocl[drop] = 0.0
        ocl[drop, bg] = 1.0
    want = O.det_postprocess(rois, ocl, orr, bg, 16, ratio, det_threshold=thr, max_boxes=max_boxes)
    c = int(host(count)[0])
    ok = c == len(want)
    for i, (wc, wbox, wp) in enumerate(want if ok else []):
        ok &= int(host(dcls)[0, i]) == wc and host(boxes)[0, i].tolist() == wbox.tolist() and float(host(probs)[0, i]) == float(wp)
    return bool(ok), dict(kind="postprocess", m=m, k=k, bg=bg, max_boxes=max_boxes, ratio=ratio, thr=thr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=300)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--only", default="", help="comma-separated case kinds, e.g. proposals,nms")
    args = ap.parse_args()
    rng = np.random.default_rng(args.seed)
    kinds = [case_nms, case_proposals, case_roi, case_labels, case_label_rois, case_postprocess, case_image]
    if args.only:
        kinds = [f for f in kinds if f.__name__[5:] in args.only.split(",")]
    counts, failures = {}, []
    for i in range(args.cases):
        fn = kinds[i % len(kinds)]
        ok, info = fn(rng)
        counts[info["kind"]] = counts.get(info["kind"], 0) + 1
        if not ok:
            failures.append(info)
            print("FAIL", json.dumps(info), flush=True)
    print(json.dumps({"cases": args.cases, "seed": args.seed, "per_kind": counts, "failures": len(failures)}))
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
