"""Device-resident functional API: torch CUDA tensors in, torch CUDA tensors out.

One function per C-ABI entry point (include/frcnn_b200.h).  Everything is enqueued on torch's
current stream and nothing here synchronises; the numpy drop-in modules (`det_util`, `rpn_util`,
`util`, `custom_layers`, `voc_dets`) sit on top of these.  A leading batch dimension = independent
images.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .runtime import get_context, ptr

_ROI_DTYPES = {torch.int16: _lib.ROI_I16, torch.int32: _lib.ROI_I32, torch.float32: _lib.ROI_F32}
_MODES = {"resize": _lib.ROI_RESIZE, "max": _lib.ROI_MAX}


def _chk(t, dtype, name, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor" % name)
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if ndim is not None and t.dim() != ndim:
        raise ValueError("%s must have %d dimensions, got shape %s" % (name, ndim, tuple(t.shape)))
    return t.contiguous()


def _chk_out(t, dtype, name, ndim):
    if not t.is_contiguous():
        raise ValueError("%s is written in place and must be contiguous" % name)
    return _chk(t, dtype, name, ndim)


def _chk_extents(extents, b):
    """extents (B,2) i32 (rows, cols) per image of a padded batch, a CUDA tensor: the call stays asynchronous."""
    extents = _chk(extents, torch.int32, "extents", 2)
    if extents.shape != (b, 2):
        raise ValueError("extents must be (B, 2) = (%d, 2), got %s" % (b, tuple(extents.shape)))
    return extents


def decode_topk(regr, cls, anchor_dims, stride, k, want_dense=False, extents=None):
    """K-a.  regr (B,R,C,4A) f32, cls (B,R,C,A) f32 -> boxes (B,k,4) i16, scores (B,k) f32,
    index (B,k) i32, count (B,) i32 [, dense (B,R*C*A,4) f32].  det_util.py:63-76,145-155,370-380.
    `extents` (B,2) i32 (rows, cols) on the device: a padded batch of differently sized maps, see `pad_batch`; each
    image's result is that of the call on its own map, `index` counts in that map, no dense boxes."""
    regr, cls = _chk(regr, torch.float32, "regr", 4), _chk(cls, torch.float32, "cls", 4)
    ctx = get_context(regr.device)
    b, rows, cols, a = cls.shape
    if regr.shape != (b, rows, cols, 4 * a):
        raise ValueError("regr shape %s does not match cls shape %s" % (tuple(regr.shape), tuple(cls.shape)))
    anc, n_anc = ctx.anchors(anchor_dims)
    if n_anc != a:
        raise ValueError("cls has %d anchors per cell, anchor_dims has %d" % (a, n_anc))
    if extents is not None:
        if want_dense:
            raise ValueError("dense boxes are not available for a padded batch (extents given)")
        extents = _chk_extents(extents, b)
    k = int(min(k, rows * cols * a))
    boxes, scores = ctx.empty((b, k, 4), torch.int16), ctx.empty((b, k), torch.float32)
    index, count = ctx.empty((b, k), torch.int32), ctx.empty((b,), torch.int32)
    if extents is not None:
        ctx.call("frcnn_decode_topk_ragged", ptr(regr), ptr(cls), anc, rows, cols, a, int(stride), k, b, ptr(extents),
                 ptr(boxes), ptr(scores), ptr(index), ptr(count), None)
        return boxes, scores, index, count
    dense = ctx.empty((b, rows * cols * a, 4), torch.float32) if want_dense else None
    ctx.call("frcnn_decode_topk", ptr(regr), ptr(cls), anc, rows, cols, a, int(stride), k, b, ptr(boxes),
             ptr(scores), ptr(index), ptr(count), ptr(dense))
    return (boxes, scores, index, count, dense) if want_dense else (boxes, scores, index, count)


def nms_i16(boxes, scores, n=None, overlap_thresh=0.7, max_boxes=300):
    """K-b.  boxes (B,n_max,4) i16, scores (B,n_max) f32, n (B,) i32 or None ->
    keep_index (B,max_boxes) i32 (-1 padded), keep_count (B,), keep_boxes, keep_scores.
    det_util.py:209-256.  Areas, intersections and unions are exact integers while every side x2 - x1 + 1, y2 - y1 + 1 is at most 32767 in magnitude, so the result
    equals the reference's int16 numpy arithmetic wherever that does not wrap (|area|, intersection and
    |area_i + area_j| < 32768), and that of the same boxes as int64 everywhere else."""
    boxes, scores = _chk(boxes, torch.int16, "boxes", 3), _chk(scores, torch.float32, "scores", 2)
    ctx = get_context(boxes.device)
    b, n_max, _ = boxes.shape
    if n is not None:
        n = _chk(n, torch.int32, "n", 1)
    max_boxes = int(max_boxes)
    ki, kc = ctx.empty((b, max_boxes), torch.int32), ctx.empty((b,), torch.int32)
    kb, ks = ctx.empty((b, max_boxes, 4), torch.int16), ctx.empty((b, max_boxes), torch.float32)
    ctx.call("frcnn_nms_i16", ptr(boxes), ptr(scores), ptr(n), n_max, b, float(overlap_thresh), max_boxes,
             ptr(ki), ptr(kc), ptr(kb), ptr(ks))
    return ki, kc, kb, ks


def nms_f64(boxes, scores, seg_offsets, max_seg_len, overlap_thresh=0.5, max_boxes=2000):
    """K-b'.  boxes (T,4) f64, scores (T,) f32, seg_offsets (S+1,) i32 -> keep_index (S,stride) i32
    relative to the segment start, keep_count (S,).  det_util.py:209-256 as called at voc_dets.py:76."""
    boxes, scores = _chk(boxes, torch.float64, "boxes", 2), _chk(scores, torch.float32, "scores", 1)
    seg_offsets = _chk(seg_offsets, torch.int32, "seg_offsets", 1)
    ctx = get_context(boxes.device)
    n_seg = seg_offsets.numel() - 1
    out_stride = int(min(max_boxes, max_seg_len))
    ki, kc = ctx.empty((n_seg, out_stride), torch.int32), ctx.empty((n_seg,), torch.int32)
    ctx.call("frcnn_nms_f64", ptr(boxes), ptr(scores), ptr(seg_offsets), n_seg, int(max_seg_len),
             float(overlap_thresh), int(max_boxes), out_stride, ptr(ki), ptr(kc))
    return ki, kc


def proposals(regr, cls, anchor_dims, stride, k, overlap_thresh=0.7, max_boxes=300, out=None, extents=None):
    """K-a -> K-b fused on the device.  Returns rois (B,max_boxes,4) i16, scores (B,max_boxes) f32,
    count (B,) i32 (written into `out` = (rois, scores, count) when given).
    det_util.py:63-77 (k=12000, 2000) / :136-158 (k=8000, 300).
    `extents` (B,2) i32 (rows, cols) on the device: a padded batch of differently sized maps (see `pad_batch`); each
    image's proposals are those of the call on its own map."""
    regr, cls = _chk(regr, torch.float32, "regr", 4), _chk(cls, torch.float32, "cls", 4)
    ctx = get_context(regr.device)
    b, rows, cols, a = cls.shape
    if regr.shape != (b, rows, cols, 4 * a):
        raise ValueError("regr shape %s does not match cls shape %s" % (tuple(regr.shape), tuple(cls.shape)))
    anc, n_anc = ctx.anchors(anchor_dims)
    if n_anc != a:
        raise ValueError("cls has %d anchors per cell, anchor_dims has %d" % (a, n_anc))
    max_boxes = int(max_boxes)
    if out is not None:
        rois, scores, count = (_chk_out(out[0], torch.int16, "out rois", 3), _chk_out(out[1], torch.float32, "out scores", 2),
                               _chk_out(out[2], torch.int32, "out count", 1))
        if rois.shape != (b, max_boxes, 4) or scores.shape != (b, max_boxes) or count.shape != (b,):
            raise ValueError("out buffers have the wrong shape")
    else:
        rois, scores = ctx.empty((b, max_boxes, 4), torch.int16), ctx.empty((b, max_boxes), torch.float32)
        count = ctx.empty((b,), torch.int32)
    if extents is not None:
        ctx.call("frcnn_proposals_ragged", ptr(regr), ptr(cls), anc, rows, cols, a, int(stride), int(k),
                 float(overlap_thresh), max_boxes, b, ptr(_chk_extents(extents, b)), ptr(rois), ptr(scores), ptr(count))
        return rois, scores, count
    ctx.call("frcnn_proposals", ptr(regr), ptr(cls), anc, rows, cols, a, int(stride), int(k), float(overlap_thresh),
             max_boxes, b, ptr(rois), ptr(scores), ptr(count))
    return rois, scores, count


def label_anchors(gt, n_gt, img_wh, rows, cols, anchor_dims, stride, extents=None):
    """K-c.  gt (B,Gmax,4) f32 pixel corners, n_gt (B,) i32, img_wh (B,2) i32 (width,height) ->
    can_use (B,N) u8, is_pos (B,N) u8, bbreg (B,N,4) f32, counts (B,2) i32.  rpn_util.py:54-103.
    `extents` (B,2) i32 (rows_b, cols_b) on the device: images of different conv shapes padded to rows x cols; each
    image's labels are those of the call on its own map, laid into the padded (R,C,A) layout, padding cells zero."""
    gt, n_gt = _chk(gt, torch.float32, "gt", 3), _chk(n_gt, torch.int32, "n_gt", 1)
    img_wh = _chk(img_wh, torch.int32, "img_wh", 2)
    ctx = get_context(gt.device)
    b, g_max, _ = gt.shape
    anc, a = ctx.anchors(anchor_dims)
    n = rows * cols * a
    can_use, is_pos = ctx.empty((b, n), torch.uint8), ctx.empty((b, n), torch.uint8)
    bbreg, counts = ctx.empty((b, n, 4), torch.float32), ctx.empty((b, 2), torch.int32)
    if extents is not None:
        ctx.call("frcnn_label_anchors_ragged", ptr(gt), ptr(n_gt), ptr(img_wh), g_max, int(rows), int(cols), a, anc,
                 int(stride), b, ptr(_chk_extents(extents, b)), ptr(can_use), ptr(is_pos), ptr(bbreg), ptr(counts))
        return can_use, is_pos, bbreg, counts
    ctx.call("frcnn_label_anchors", ptr(gt), ptr(n_gt), ptr(img_wh), g_max, int(rows), int(cols), a, anc, int(stride),
             b, ptr(can_use), ptr(is_pos), ptr(bbreg), ptr(counts))
    return can_use, is_pos, bbreg, counts


def pack_rpn_targets(can_use, is_pos, bbreg, rows, cols, n_anchors, off_pos=None, off_neg=None):
    """T6/T7.  off_pos / off_neg = (ranks (T,) i32, offsets (B+1,) i32) of the host-drawn
    random.sample switch-offs (rpn_util.py:324-350) or None.  Clears can_use at those ranks IN
    PLACE (can_use must be contiguous), then packs y_class (B,R,C,2A) u8 and y_bbreg (B,R,C,8A)
    f32 (rpn_util.py:124-140)."""
    is_pos, bbreg = _chk(is_pos, torch.uint8, "is_pos", 2), _chk(bbreg, torch.float32, "bbreg", 3)
    if not can_use.is_contiguous():
        raise ValueError("can_use is updated in place and must be contiguous")
    can_use = _chk(can_use, torch.uint8, "can_use", 2)
    ctx = get_context(can_use.device)
    b = can_use.shape[0]
    args = []
    for pair, name in ((off_pos, "off_pos"), (off_neg, "off_neg")):
        if pair is None or pair[0].numel() == 0:
            args += [None, None]
            continue
        ranks, offs = _chk(pair[0], torch.int32, name, 1), _chk(pair[1], torch.int32, name + " offsets", 1)
        if offs.numel() != b + 1:
            raise ValueError("%s offsets must have batch+1 entries" % name)
        args += [ptr(ranks), ptr(offs)]
    y_class = ctx.empty((b, rows, cols, 2 * n_anchors), torch.uint8)
    y_bbreg = ctx.empty((b, rows, cols, 8 * n_anchors), torch.float32)
    ctx.call("frcnn_pack_rpn_targets", ptr(can_use), ptr(is_pos), ptr(bbreg), *args, int(rows), int(cols),
             int(n_anchors), b, ptr(y_class), ptr(y_bbreg))
    return y_class, y_bbreg


def sampler_state(seed, device=None):
    """The device RNG state of `sample_rpn_` / `sample_det`: a CUDA int64 tensor [seed, offset = 0].  The kernels read it
    on the device and the calls advance the offset by the batch size, so a captured CUDA graph draws new samples on
    every replay.  `seed` is taken modulo 2^64 (stored as its two's complement int64)."""
    s = int(seed) & 0xffffffffffffffff
    return torch.tensor([s - (1 << 64) if s >= 1 << 63 else s, 0], dtype=torch.int64, device=get_context(device).device)


def _chk_state(state):
    state = _chk_out(state, torch.int64, "state", 1)
    if state.shape != (2,):
        raise ValueError("state must be the (2,) int64 tensor of sampler_state(), got shape %s" % (tuple(state.shape),))
    return state


def sample_rpn_(can_use, is_pos, counts, state, extents=None, padded_shape=None, n_anchors=None, max_pos=128,
                sample_size=256):
    """rpn_util.py:324-350 drawn on the device: in each image keeps min(#pos, max_pos) usable positives and
    min(#neg, sample_size - kept positives) usable negatives, a uniformly random subset of each chosen with the
    counter-based RNG of `state` (sampler_state), and clears can_use of the others IN PLACE.  can_use / is_pos (B,N) u8
    and counts (B,2) i32 as label_anchors returns them.  `extents` (B,2) i32 with `padded_shape` = (rows, cols) and
    `n_anchors`: the padded layout of label_anchors(..., extents=); each image's draw equals the call on its own map.
    Advances state[1] by B (stream-ordered).  Returns can_use."""
    can_use = _chk_out(can_use, torch.uint8, "can_use", 2)
    is_pos, counts = _chk(is_pos, torch.uint8, "is_pos", 2), _chk(counts, torch.int32, "counts", 2)
    state = _chk_state(state)
    ctx = get_context(can_use.device)
    b, n = can_use.shape
    if is_pos.shape != (b, n) or counts.shape != (b, 2):
        raise ValueError("sample_rpn_: shapes must be (B,N), (B,N), (B,2)")
    if extents is not None:
        if padded_shape is None or n_anchors is None:
            raise ValueError("sample_rpn_: extents need padded_shape and n_anchors")
        rows, cols = (int(v) for v in padded_shape)
        if rows * cols * int(n_anchors) != n:
            raise ValueError("sample_rpn_: N = %d is not rows * cols * n_anchors" % n)
        ctx.call("frcnn_sample_rpn_ragged", ptr(can_use), ptr(is_pos), ptr(counts), rows, cols, int(n_anchors),
                 ptr(_chk_extents(extents, b)), int(max_pos), int(sample_size), ptr(state), b)
    else:
        ctx.call("frcnn_sample_rpn", ptr(can_use), ptr(is_pos), ptr(counts), n, int(max_pos), int(sample_size), ptr(state), b)
    state[1:].add_(b)
    return can_use


def sample_det(is_pos, n_rows, n_samples, state):
    """det_util.py:260-306 drawn on the device with the counter-based RNG of `state` (sampler_state).  is_pos (B,n_max)
    u8 flags of label_rois's rows, n_rows (B,) i32 its count -> index (B,S) i32 (the input of gather_det_samples,
    positives first; -1 rows for an image without an eligible row), has (B,) bool.  Advances state[1] by B."""
    is_pos, n_rows = _chk(is_pos, torch.uint8, "is_pos", 2), _chk(n_rows, torch.int32, "n_rows", 1)
    state = _chk_state(state)
    ctx = get_context(is_pos.device)
    b, n_max = is_pos.shape
    if n_rows.shape != (b,):
        raise ValueError("sample_det: n_rows must be (B,)")
    s = int(n_samples)
    index, has = ctx.empty((b, s), torch.int32), ctx.empty((b,), torch.bool)
    ctx.call("frcnn_sample_det", ptr(is_pos), ptr(n_rows), n_max, s, ptr(state), b, ptr(index), ptr(has))
    state[1:].add_(b)
    return index, has


def label_rois(rois, gt, gt_cls, n_gt, n_classes, n_roi=None):
    """K-c'.  rois (B,n_max,4) i16, gt (B,Gmax,4) f64 feature units, gt_cls (B,Gmax) i32, n_gt (B,) ->
    out_rois (B,n_max,4) i16, y_class (B,n_max,K) i32, y_transform (B,n_max,8(K-1)) f32,
    src (B,n_max) i32, count (B,) i32 (rows >= count are undefined).  det_util.py:310-366."""
    rois = _chk(rois, torch.int16, "rois", 3)
    gt, gt_cls = _chk(gt, torch.float64, "gt", 3), _chk(gt_cls, torch.int32, "gt_cls", 2)
    n_gt = _chk(n_gt, torch.int32, "n_gt", 1)
    if n_roi is not None:
        n_roi = _chk(n_roi, torch.int32, "n_roi", 1)
    ctx = get_context(rois.device)
    b, n_max, _ = rois.shape
    g_max, k = gt.shape[1], int(n_classes)
    out_rois, out_cls = ctx.empty((b, n_max, 4), torch.int16), ctx.empty((b, n_max, k), torch.int32)
    out_bbreg = ctx.empty((b, n_max, 8 * (k - 1)), torch.float32)
    src, count = ctx.empty((b, n_max), torch.int32), ctx.empty((b,), torch.int32)
    ctx.call("frcnn_label_rois", ptr(rois), ptr(n_roi), n_max, ptr(gt), ptr(gt_cls), ptr(n_gt), g_max, k, b,
             ptr(out_rois), ptr(out_cls), ptr(out_bbreg), ptr(src), ptr(count))
    return out_rois, out_cls, out_bbreg, src, count


def clip_rois(rois, extents):
    """rois (B,N,4) i16/i32/f32 of a padded batch -> a new tensor of the same dtype, truncated to int like the RoI layer
    and clamped to each image's own map (x1, y1 >= 0, x2 <= cols_b, y2 <= rows_b; extents (B,2) i32 on the device).  The
    RoI layer on the padded features then takes the crops of the call on the image's own map and reads no padding."""
    if rois.dtype not in _ROI_DTYPES:
        raise TypeError("rois must be int16, int32 or float32")
    rois = _chk(rois, rois.dtype, "rois", 3)
    extents = _chk_extents(extents, rois.shape[0])
    ctx = get_context(rois.device)
    out = ctx.empty(tuple(rois.shape), rois.dtype)
    ctx.call("frcnn_clip_rois", ptr(rois), _ROI_DTYPES[rois.dtype], rois.shape[1], rois.shape[0], ptr(extents), ptr(out))
    return out


def pad_batch(arrays, pad_to=None):
    """A list of per-image (R_b, C_b, X) arrays (numpy or torch, one dtype) -> (padded (B,R,C,X), extents (B,2) i32), both
    CUDA tensors.  (R, C) = the largest extents, or `pad_to` (which must hold every image).  Only each image's valid
    region is copied; the padding is zero, and the ragged entry points never read it."""
    if not isinstance(arrays, (list, tuple)) or len(arrays) == 0:
        raise ValueError("pad_batch needs a non-empty list of (R_b, C_b, X) arrays")
    shapes = [tuple(x.shape) for x in arrays]
    if any(len(s) != 3 for s in shapes):
        raise ValueError("every array must have 3 dimensions (R_b, C_b, X), got %s" % (shapes,))
    if len({s[2] for s in shapes}) != 1:
        raise ValueError("arrays disagree in their last dimension: %s" % (shapes,))
    dtypes = {str(x.dtype).replace("torch.", "") for x in arrays}
    if len(dtypes) != 1:
        raise ValueError("arrays must share one dtype, got %s" % sorted(dtypes))
    rows, cols = max(s[0] for s in shapes), max(s[1] for s in shapes)
    if pad_to is not None:
        pr, pc = (int(v) for v in pad_to)
        if pr < rows or pc < cols:
            raise ValueError("pad_to %s is smaller than the largest extents (%d, %d)" % ((pr, pc), rows, cols))
        rows, cols = pr, pc
    if rows <= 0 or cols <= 0:
        raise ValueError("the padded map is empty")
    first = arrays[0] if isinstance(arrays[0], torch.Tensor) else torch.from_numpy(np.ascontiguousarray(arrays[0]))
    ctx = get_context(first.device if first.is_cuda else None)
    padded = torch.zeros((len(arrays), rows, cols, shapes[0][2]), dtype=first.dtype, device=ctx.device)
    for b, x in enumerate(arrays):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        padded[b, :t.shape[0], :t.shape[1]].copy_(t, non_blocking=t.is_cuda)
    extents = ctx.to_device(np.array([s[:2] for s in shapes], np.int32).reshape(-1, 2))
    return padded, extents


def roi_compact_supported(height, width, channels, pool):
    """True when max mode can use the one-byte arg-max (every bin fits 16 x 16 cells, C % 4 == 0, pool <= 8)."""
    return bool(_lib.load().frcnn_roi_compact_supported(int(height), int(width), int(channels), int(pool)))


def roi_forward(feat, rois, pool, mode="resize", out=None, argmax_out=None, compact=False):
    """K-d forward.  feat (B,H,W,C) f32 channels-last, rois (B,N,4) i16/i32/f32 ->
    out (B,N,P,P,C) f32 [, argmax (B,N,P,P,C) in max mode: i32 flat cell index y*W+x, or with `compact=True` u8
    (dy << 4) | dx relative to the bin's first cell (training fast path, see include/frcnn_b200.h)].
    custom_layers.py:35-56.  `out` / `argmax_out`: caller-owned result buffers (e.g. slices of a batch buffer)."""
    feat = _chk(feat, torch.float32, "feat", 4)
    if rois.dtype not in _ROI_DTYPES:
        raise TypeError("rois must be int16, int32 or float32")
    rois = _chk(rois, rois.dtype, "rois", 3)
    ctx = get_context(feat.device)
    b, h, w, c = feat.shape
    n, p = rois.shape[1], int(pool)
    if out is not None:
        out = _chk_out(out, torch.float32, "out", 5)
        if out.shape != (b, n, p, p, c):
            raise ValueError("out buffer has the wrong shape")
    else:
        out = ctx.empty((b, n, p, p, c), torch.float32)
    argmax = None
    if compact and mode != "max":
        raise ValueError("compact arg-max exists in max mode only")
    if mode == "max":
        adt = torch.uint8 if compact else torch.int32
        if argmax_out is not None:
            argmax = _chk_out(argmax_out, adt, "argmax_out", 5)
            if argmax.shape != (b, n, p, p, c):
                raise ValueError("argmax_out buffer has the wrong shape")
        else:
            argmax = ctx.empty((b, n, p, p, c), adt)
    if compact:
        ctx.call("frcnn_roi_max_fwd_compact", ptr(feat), h, w, c, ptr(rois), _ROI_DTYPES[rois.dtype], n, p, b, ptr(out),
                 ptr(argmax))
        return out, argmax
    ctx.call("frcnn_roi_fwd", _MODES[mode], ptr(feat), h, w, c, ptr(rois), _ROI_DTYPES[rois.dtype], n, p, b,
             ptr(out), ptr(argmax))
    return (out, argmax) if mode == "max" else out


def roi_backward(grad_out, rois, feat_shape, mode="resize", argmax=None):
    """K-d backward.  grad_out (B,N,P,P,C) f32 -> grad_feat (B,H,W,C) f32 (atomic-free).  Max mode takes the forward's
    arg-max in either format (int32 flat index or the one-byte compact code)."""
    grad_out = _chk(grad_out, torch.float32, "grad_out", 5)
    rois = _chk(rois, rois.dtype, "rois", 3)
    ctx = get_context(grad_out.device)
    b, h, w, c = feat_shape
    n, p = grad_out.shape[1], grad_out.shape[2]
    gfeat = ctx.empty((b, h, w, c), torch.float32)
    if mode == "max" and isinstance(argmax, torch.Tensor) and argmax.dtype == torch.uint8:      # one-byte arg-max
        argmax = _chk(argmax, torch.uint8, "argmax", 5)
        ctx.call("frcnn_roi_max_bwd_compact", ptr(grad_out), ptr(rois), _ROI_DTYPES[rois.dtype], ptr(argmax), h, w, c, n, p,
                 b, ptr(gfeat))
        return gfeat
    if mode == "max":
        argmax = _chk(argmax, torch.int32, "argmax", 5)
    ctx.call("frcnn_roi_bwd", _MODES[mode], ptr(grad_out), ptr(rois), _ROI_DTYPES[rois.dtype],
             ptr(argmax) if mode == "max" else None, h, w, c, n, p, b, ptr(gfeat))
    return gfeat


def det_postprocess(rois, out_cls, out_reg, resize_ratio, bg_index, stride=16, det_threshold=0.0, nms_thresh=0.5,
                    max_boxes=2000, n_rows=None):
    """K-e.  rois (B,M,4) i16, out_cls (B,M,K) f32, out_reg (B,M,4(K-1)) f32, resize_ratio (B,) f64 ->
    det_boxes (B,M,4) i32, det_probs (B,M) f32, det_cls (B,M) i32, det_count (B,) i32.
    voc_dets.py:51-86."""
    rois = _chk(rois, torch.int16, "rois", 3)
    out_cls, out_reg = _chk(out_cls, torch.float32, "out_cls", 3), _chk(out_reg, torch.float32, "out_reg", 3)
    resize_ratio = _chk(resize_ratio, torch.float64, "resize_ratio", 1)
    if n_rows is not None:
        n_rows = _chk(n_rows, torch.int32, "n_rows", 1)
    ctx = get_context(rois.device)
    b, m, _ = rois.shape
    k = out_cls.shape[2]
    if out_reg.shape != (b, m, 4 * (k - 1)):
        raise ValueError("out_reg must be (B, M, 4*(K-1))")
    boxes, probs = ctx.empty((b, m, 4), torch.int32), ctx.empty((b, m), torch.float32)
    cls, count = ctx.empty((b, m), torch.int32), ctx.empty((b,), torch.int32)
    ctx.call("frcnn_det_postprocess", ptr(rois), ptr(out_cls), ptr(out_reg), ptr(resize_ratio), ptr(n_rows), m, k, int(bg_index),
             int(stride), float(det_threshold), float(nms_thresh), int(max_boxes), b, ptr(boxes), ptr(probs),
             ptr(cls), ptr(count))
    return boxes, probs, cls, count


def gather_det_samples(rois, y_cls, y_tr, index):
    """det_util.py:119-125 batched: rows `index` (B,S) i32 of label_rois's outputs -> rois (B,S,4) i16,
    y_class_num (B,S,K) i32, y_transform (B,S,8(K-1)) f32; index -1 gives zero rows."""
    rois, y_cls = _chk(rois, torch.int16, "rois", 3), _chk(y_cls, torch.int32, "y_cls", 3)
    y_tr, index = _chk(y_tr, torch.float32, "y_tr", 3), _chk(index, torch.int32, "index", 2)
    ctx = get_context(rois.device)
    b, n_max, _ = rois.shape
    k, s = y_cls.shape[2], index.shape[1]
    if y_cls.shape != (b, n_max, k) or y_tr.shape != (b, n_max, 8 * (k - 1)) or index.shape[0] != b:
        raise ValueError("gather_det_samples: inconsistent shapes")
    out_rois, out_cls = ctx.empty((b, s, 4), torch.int16), ctx.empty((b, s, k), torch.int32)
    out_tr = ctx.empty((b, s, 8 * (k - 1)), torch.float32)
    ctx.call("frcnn_gather_det_samples", ptr(rois), ptr(y_cls), ptr(y_tr), ptr(index), n_max, k, s, b, ptr(out_rois),
             ptr(out_cls), ptr(out_tr))
    return out_rois, out_cls, out_tr


def cross_ious(boxes, gt):
    """util.cross_ious (util.py:146-177).  boxes (N,4) i16 or f32, gt (G,4) f32 -> (N,G) f32."""
    if boxes.dtype not in (torch.int16, torch.float32):
        raise TypeError("boxes must be int16 or float32")
    boxes, gt = _chk(boxes, boxes.dtype, "boxes", 2), _chk(gt, torch.float32, "gt", 2)
    ctx = get_context(boxes.device)
    out = ctx.empty((boxes.shape[0], gt.shape[0]), torch.float32)
    ctx.call("frcnn_cross_ious", ptr(boxes), _ROI_DTYPES[boxes.dtype], boxes.shape[0], ptr(gt), gt.shape[0], ptr(out))
    return out


def box_transform_(boxes, deltas=None, sanitize=None):
    """In place: util.transform_np_inplace (deltas given) and/or det_util._sanitize_boxes_inplace
    (sanitize=(cols, rows)).  boxes (N,4) f32."""
    boxes = _chk(boxes, torch.float32, "boxes", 2)
    if deltas is not None:
        deltas = _chk(deltas, torch.float32, "deltas", 2)
    cols, rows = sanitize if sanitize is not None else (0, 0)
    get_context(boxes.device).call("frcnn_box_transform", ptr(boxes), ptr(deltas), boxes.shape[0],
                                   1 if deltas is not None else 0, int(cols), int(rows))
    return boxes


def anchor_grid(anchor_dims, rows, cols, stride=1, pixel_space=False, device=None):
    """(rows*cols*A, 4) f32 anchors; feature space (det_util.py:162-175) or pixel space
    (rpn_util.py:276-298)."""
    ctx = get_context(device)
    anc, a = ctx.anchors(anchor_dims)
    out = ctx.empty((rows * cols * a, 4), torch.float32)
    ctx.call("frcnn_anchor_grid", anc, a, int(rows), int(cols), int(stride), 1 if pixel_space else 0, ptr(out))
    return out


def valid_boxes(boxes):
    """det_util._get_valid_box_idxs (det_util.py:196-205): index (N,) i32 + count (1,) i32."""
    boxes = _chk(boxes, torch.float32, "boxes", 2)
    ctx = get_context(boxes.device)
    index, count = ctx.empty((max(boxes.shape[0], 1),), torch.int32), ctx.empty((1,), torch.int32)
    ctx.call("frcnn_valid_boxes", ptr(boxes), boxes.shape[0], ptr(index), ptr(count))
    return index, count


def pad_rois(rois, count, group=64, out=None):
    """voc_dets.py:37-46 on the device: rois (B,n_max,4) i16 + count (B,) -> padded (B,M,4) i16 with
    M = n_max rounded up to `group` (last detector batch filled with copies of its first RoI, unused
    rows = empty box) and rows (B,) i32 = count rounded up."""
    rois, count = _chk(rois, torch.int16, "rois", 3), _chk(count, torch.int32, "count", 1)
    ctx = get_context(rois.device)
    b, n_max, _ = rois.shape
    m = -(-n_max // group) * group
    if out is not None:
        out, rows = _chk_out(out[0], torch.int16, "out rois", 3), _chk_out(out[1], torch.int32, "out rows", 1)
        if out.shape != (b, m, 4) or rows.shape != (b,):
            raise ValueError("out buffers have the wrong shape")
    else:
        out, rows = ctx.empty((b, m, 4), torch.int16), ctx.empty((b,), torch.int32)
    ctx.call("frcnn_pad_rois", ptr(rois), ptr(count), n_max, int(group), m, b, ptr(out), ptr(rows))
    return out, rows


def rpn_losses(can_use, is_pos, bbreg, cls_pred, reg_pred, want_grad=False, extents=None, padded_shape=None):
    """loss_functions.py:15-48 fused with the unpacked RPN labels.  can_use/is_pos (B,N) u8, bbreg (B,N,4) f32,
    cls_pred (B,N) f32, reg_pred (B,N,4) f32 -> loss (B,2) f32 = (class, box) [, grad_cls (B,N), grad_reg (B,N,4)].
    `extents` (B,2) i32 (rows_b, cols_b) on the device with `padded_shape` = (rows, cols): N = rows*cols*A in the padded
    (R,C,A) layout of `label_anchors(..., extents=)`; each image's loss and gradients are those of the call on its own
    map (its box loss averages over its own anchors), the padding is never read and gets zero gradients."""
    can_use, is_pos = _chk(can_use, torch.uint8, "can_use", 2), _chk(is_pos, torch.uint8, "is_pos", 2)
    bbreg, reg_pred = _chk(bbreg, torch.float32, "bbreg", 3), _chk(reg_pred, torch.float32, "reg_pred", 3)
    cls_pred = _chk(cls_pred, torch.float32, "cls_pred", 2)
    ctx = get_context(can_use.device)
    b, n = can_use.shape
    if cls_pred.shape != (b, n) or bbreg.shape != (b, n, 4) or reg_pred.shape != (b, n, 4):
        raise ValueError("rpn_losses: shapes must be (B,N), (B,N), (B,N,4), (B,N), (B,N,4)")
    if (extents is None) != (padded_shape is None):
        raise ValueError("rpn_losses: give extents and padded_shape together")
    if extents is not None:
        rows, cols = (int(v) for v in padded_shape)
        if rows <= 0 or cols <= 0 or n % (rows * cols) != 0:
            raise ValueError("rpn_losses: N = %d is not rows * cols * A for padded_shape %s" % (n, (rows, cols)))
        extents = _chk_extents(extents, b)
    loss = ctx.empty((b, 2), torch.float32)
    g_cls = ctx.empty((b, n), torch.float32) if want_grad else None
    g_reg = ctx.empty((b, n, 4), torch.float32) if want_grad else None
    if extents is not None:
        ctx.call("frcnn_rpn_losses_ragged", ptr(can_use), ptr(is_pos), ptr(bbreg), ptr(cls_pred), ptr(reg_pred), rows, cols,
                 n // (rows * cols), b, ptr(extents), ptr(loss), ptr(g_cls), ptr(g_reg))
    else:
        ctx.call("frcnn_rpn_losses", ptr(can_use), ptr(is_pos), ptr(bbreg), ptr(cls_pred), ptr(reg_pred), n, b, ptr(loss),
                 ptr(g_cls), ptr(g_reg))
    return (loss, g_cls, g_reg) if want_grad else loss


def det_losses(y_class, y_transform, cls_pred, reg_pred, want_grad=False):
    """loss_functions.py:51-76 on label_rois' targets.  y_class (B,M,K) i32, y_transform (B,M,8(K-1)) f32,
    cls_pred (B,M,K) f32, reg_pred (B,M,4(K-1)) f32 -> loss (B,2) f32 = (class, box) [, grad_cls, grad_reg]."""
    y_class, y_transform = _chk(y_class, torch.int32, "y_class", 3), _chk(y_transform, torch.float32, "y_transform", 3)
    cls_pred, reg_pred = _chk(cls_pred, torch.float32, "cls_pred", 3), _chk(reg_pred, torch.float32, "reg_pred", 3)
    ctx = get_context(y_class.device)
    b, m, k = y_class.shape
    if y_transform.shape != (b, m, 8 * (k - 1)) or cls_pred.shape != (b, m, k) or reg_pred.shape != (b, m, 4 * (k - 1)):
        raise ValueError("det_losses: shapes must be (B,M,K), (B,M,8(K-1)), (B,M,K), (B,M,4(K-1))")
    loss = ctx.empty((b, 2), torch.float32)
    g_cls = ctx.empty((b, m, k), torch.float32) if want_grad else None
    g_reg = ctx.empty((b, m, 4 * (k - 1)), torch.float32) if want_grad else None
    ctx.call("frcnn_det_losses", ptr(y_class), ptr(y_transform), ptr(cls_pred), ptr(reg_pred), m, k, b, ptr(loss),
             ptr(g_cls), ptr(g_reg))
    return (loss, g_cls, g_reg) if want_grad else loss


def voc_match(det_boxes, img_det_offsets, img_det_rank, gt_boxes, gt_difficult, img_gt_offsets, ovthresh=0.5):
    """eval_dets.py:75-116 for one class.  det_boxes (nd,4) f64 sorted by descending confidence, CSR of detection
    ranks per image, gt (ng,4) f64 + difficult (ng,) u8 grouped by image -> tp (nd,) f64, fp (nd,) f64."""
    det_boxes, gt_boxes = _chk(det_boxes, torch.float64, "det_boxes", 2), _chk(gt_boxes, torch.float64, "gt_boxes", 2)
    img_det_offsets, img_det_rank = _chk(img_det_offsets, torch.int32, "img_det_offsets", 1), _chk(img_det_rank, torch.int32, "img_det_rank", 1)
    gt_difficult, img_gt_offsets = _chk(gt_difficult, torch.uint8, "gt_difficult", 1), _chk(img_gt_offsets, torch.int32, "img_gt_offsets", 1)
    ctx = get_context(det_boxes.device)
    nd, ng, n_img = det_boxes.shape[0], gt_boxes.shape[0], img_det_offsets.numel() - 1
    tp, fp = ctx.empty((nd,), torch.float64), ctx.empty((nd,), torch.float64)
    ctx.call("frcnn_voc_match", ptr(det_boxes), ptr(img_det_offsets), ptr(img_det_rank), ptr(gt_boxes), ptr(gt_difficult),
             ptr(img_gt_offsets), n_img, nd, ng, float(ovthresh), ptr(tp), ptr(fp))
    return tp, fp


def voc_pr_ap(tp, fp, npos, thresholds):
    """eval_dets.py:118-125 + the 11-point voc_ap (:8-19): -> rec (nd,), prec (nd,), ap (1,) all f64."""
    tp, fp = _chk(tp, torch.float64, "tp", 1), _chk(fp, torch.float64, "fp", 1)
    thresholds = _chk(thresholds, torch.float64, "thresholds", 1)
    ctx = get_context(tp.device)
    nd = tp.shape[0]
    rec, prec, ap = ctx.empty((nd,), torch.float64), ctx.empty((nd,), torch.float64), ctx.empty((1,), torch.float64)
    ctx.call("frcnn_voc_pr_ap", ptr(tp), ptr(fp), nd, float(npos), ptr(thresholds), thresholds.numel(), ptr(rec), ptr(prec),
             ptr(ap))
    return rec, prec, ap


# ---- SURVEY 8f-4: host-side input pipeline on the device -------------------------------------------------------------
IMAGENET_MEAN_BGR = (103.939, 116.779, 123.68)     # keras.applications.imagenet_utils.preprocess_input ('caffe' mode)


def image_resize_cubic(images, dst_height, dst_width, flip=False, mean=None, want_u8=True):
    """shapes.py:19-29 on the device: images (B,H,W,C) u8 (BGR, as cv2.imread) -> cv2.resize(INTER_CUBIC) [+ cv2.flip(.., 1)].
    Returns u8 (B,dst_h,dst_w,C) when `want_u8`, and additionally float32 pixels minus `mean` (C floats, the subtraction
    of resnet.preprocess, resnet.py:64-75) when `mean` is given: u8, (u8, f32) or f32."""
    images = _chk(images, torch.uint8, "images", 4)
    ctx = get_context(images.device)
    b, h, w, c = images.shape
    if not want_u8 and mean is None:
        raise ValueError("nothing to compute: want_u8=False and no mean")
    out_u8 = ctx.empty((b, int(dst_height), int(dst_width), c), torch.uint8) if want_u8 else None
    out_f = ctx.empty((b, int(dst_height), int(dst_width), c), torch.float32) if mean is not None else None
    mean_arr = None
    if mean is not None:
        mean_arr = np.ascontiguousarray(np.asarray(mean, dtype=np.float64).reshape(-1))
        if mean_arr.shape[0] != c:
            raise ValueError("mean must have one entry per channel")
    ctx.call("frcnn_image_resize_cubic", ptr(images), h, w, c, int(dst_height), int(dst_width), int(bool(flip)), b,
             None if mean_arr is None else mean_arr.ctypes.data_as(C.c_void_p), ptr(out_u8), ptr(out_f))
    if out_u8 is not None and out_f is not None:
        return out_u8, out_f
    return out_u8 if out_u8 is not None else out_f


def pack_images(sources):
    """A list of (h_b, w_b, C) uint8 images (numpy or torch, one channel count) -> (packed (T,) u8, offsets (B,) i64 byte
    offsets, sizes (B,2) i32 (h_b, w_b)), all CUDA tensors: the source layout of `image_resize_cubic_ragged`.  Host images
    are staged in one pinned buffer and uploaded with one asynchronous copy."""
    if not isinstance(sources, (list, tuple)) or len(sources) == 0:
        raise ValueError("pack_images needs a non-empty list of (h, w, C) uint8 images")
    for x in sources:
        if not isinstance(x, (np.ndarray, torch.Tensor)):
            raise TypeError("pack_images takes numpy arrays or torch tensors, got %s" % type(x).__name__)
        if x.dtype not in (np.uint8, torch.uint8):
            raise TypeError("pack_images needs uint8 images, got %s" % x.dtype)
    shapes = [tuple(x.shape) for x in sources]
    if any(len(s) != 3 for s in shapes):
        raise ValueError("every image must have 3 dimensions (h, w, C), got %s" % (shapes,))
    if len({s[2] for s in shapes}) != 1:
        raise ValueError("images disagree in their channel count: %s" % (shapes,))
    nbytes = np.array([s[0] * s[1] * s[2] for s in shapes], np.int64)
    offsets = np.concatenate([[0], np.cumsum(nbytes)[:-1]]).astype(np.int64)
    cuda = [x for x in sources if isinstance(x, torch.Tensor) and x.is_cuda]
    ctx = get_context(cuda[0].device if cuda else None)
    total = max(int(nbytes.sum()), 1)
    if cuda:
        packed = ctx.empty((total,), torch.uint8)
        for x, o, n in zip(sources, offsets.tolist(), nbytes.tolist()):
            t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
            packed[o:o + n].copy_(t.reshape(-1), non_blocking=True)
    else:
        packed = _stage_pinned([x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x) for x in sources], offsets,
                               total).to(ctx.device, non_blocking=True)
    sizes = np.array([s[:2] for s in shapes], np.int32).reshape(-1, 2)
    return packed, ctx.to_device(offsets), ctx.to_device(sizes)


def _stage_pinned(arrays, offsets, total):
    """The host arrays written back to back at `offsets` into one pinned (total,) u8 buffer (one upload's source)."""
    pinned = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
    view = pinned.numpy()
    for x, o in zip(arrays, offsets.tolist()):
        flat = x.reshape(-1).view(np.uint8)
        view[o:o + flat.size] = flat
    return pinned


def _jpeg_bytes(data):
    if isinstance(data, (bytes, bytearray, memoryview)):
        return np.frombuffer(data, np.uint8)
    if isinstance(data, np.ndarray) and data.dtype == np.uint8 and data.ndim == 1:
        return np.ascontiguousarray(data)
    raise TypeError("a JPEG file must be bytes or a 1-D uint8 array, got %s" % type(data).__name__)


def jpeg_supported(data):
    """(height, width) when the device decoder takes this JPEG file (frcnn_jpeg_inspect: baseline Huffman, 8-bit,
    greyscale or YCbCr 4:4:4 / 4:2:2 / 4:4:0 / 4:2:0 / 4:1:1, no Exif rotation), else None.  Runs on the CPU."""
    a = _jpeg_bytes(data)
    hw = np.zeros(2, np.int32)
    rc = _lib.load().frcnn_jpeg_inspect(a.ctypes.data_as(C.c_void_p), a.size, hw.ctypes.data_as(C.c_void_p))
    return (int(hw[0]), int(hw[1])) if rc == _lib.OK else None


def jpeg_decode(files):
    """cv2.imdecode(file, IMREAD_COLOR) of every file on the device, bit for bit: files = list of bytes or 1-D uint8
    arrays, each `jpeg_supported`.  Returns (packed (T,) u8, offsets (B,) i64, sizes (B,2) i32 (h, w), status (B,) i32),
    CUDA tensors: `pack_images`' layout of the (h, w, 3) BGR images plus a status per image (0, or < 0 when the file's
    entropy-coded data is corrupt: that image's pixels are zero).  The files are staged in one pinned buffer and uploaded
    with one copy."""
    if not isinstance(files, (list, tuple)) or len(files) == 0:
        raise ValueError("jpeg_decode needs a non-empty list of JPEG files")
    arrays = [_jpeg_bytes(f) for f in files]
    hw = [jpeg_supported(a) for a in arrays]
    bad = [i for i, x in enumerate(hw) if x is None]
    if bad:
        raise ValueError("files %s are not JPEG files the device decoder supports (check with jpeg_supported)" % bad)
    nbytes = np.array([a.size for a in arrays], np.int64)
    offsets = np.concatenate([[0], np.cumsum(nbytes)[:-1]]).astype(np.int64)
    sizes = np.array(hw, np.int32).reshape(-1, 2)
    out_n = sizes[:, 0].astype(np.int64) * sizes[:, 1] * 3
    out_off = np.concatenate([[0], np.cumsum(out_n)[:-1]]).astype(np.int64)
    ctx = get_context()
    pinned = _stage_pinned(arrays, offsets, int(nbytes.sum()))
    files_dev = pinned.to(ctx.device, non_blocking=True)
    out = ctx.empty((max(int(out_n.sum()), 1),), torch.uint8)
    out_offsets = ctx.to_device(out_off)
    status = ctx.empty((len(arrays),), torch.int32)
    ctx.call("frcnn_jpeg_decode", C.c_void_p(pinned.data_ptr()), ptr(files_dev), offsets.ctypes.data_as(C.c_void_p),
             nbytes.ctypes.data_as(C.c_void_p), len(arrays), ptr(out), ptr(out_offsets), out.numel(), ptr(status))
    return out, out_offsets, ctx.to_device(sizes), status


def image_resize_cubic_ragged(src, src_offsets, geom, dst_height, dst_width, flip=None, mean=None, want_u8=True, out=None,
                              channels=3):
    """`image_resize_cubic` for differently sized sources in one launch.  src (T,) u8 = the images packed back to back
    (`pack_images`), src_offsets (B,) i64, geom (B,4) i32 = (src_h, src_w, dst_h, dst_w) per image, flip (B,) u8 or None,
    all CUDA tensors (never read on the host: the call can be captured in a graph).  Image b is resized to its own
    (dst_h, dst_w) [and mirrored within that width] into the padded (B,dst_height,dst_width,C) output; every padding
    element is written as zero.  Returns u8, (u8, f32) or f32 as `image_resize_cubic`; `out` = (u8 or None, f32 or None)
    takes preallocated buffers of that shape."""
    src, src_offsets = _chk(src, torch.uint8, "src", 1), _chk(src_offsets, torch.int64, "src_offsets", 1)
    geom = _chk(geom, torch.int32, "geom", 2)
    b, c, h, w = src_offsets.shape[0], int(channels), int(dst_height), int(dst_width)
    if geom.shape != (b, 4):
        raise ValueError("geom must be (B, 4) = (%d, 4), got %s" % (b, tuple(geom.shape)))
    if flip is not None:
        flip = _chk(flip, torch.uint8, "flip", 1)
        if flip.shape != (b,):
            raise ValueError("flip must be (B,) = (%d,)" % b)
    if not want_u8 and mean is None:
        raise ValueError("nothing to compute: want_u8=False and no mean")
    ctx = get_context(src.device)
    shape = (b, h, w, c)
    if out is not None:
        if len(out) != 2 or (want_u8 and out[0] is None) or (mean is not None and out[1] is None):
            raise ValueError("out must be (u8, f32) with a u8 buffer when want_u8 and a f32 buffer when mean is given")
        out_u8 = _chk_out(out[0], torch.uint8, "out u8", 4) if want_u8 else None
        out_f = _chk_out(out[1], torch.float32, "out f32", 4) if mean is not None else None
        if any(t is not None and tuple(t.shape) != shape for t in (out_u8, out_f)):
            raise ValueError("out buffers must be %s" % (shape,))
    else:
        out_u8 = ctx.empty(shape, torch.uint8) if want_u8 else None
        out_f = ctx.empty(shape, torch.float32) if mean is not None else None
    mean_arr = None
    if mean is not None:
        mean_arr = np.ascontiguousarray(np.asarray(mean, dtype=np.float64).reshape(-1))
        if mean_arr.shape[0] != c:
            raise ValueError("mean must have one entry per channel")
    ctx.call("frcnn_image_resize_cubic_ragged", ptr(src), ptr(src_offsets), src.numel(), ptr(geom), ptr(flip), c, h, w, b,
             None if mean_arr is None else mean_arr.ctypes.data_as(C.c_void_p), ptr(out_u8), ptr(out_f))
    if out_u8 is not None and out_f is not None:
        return out_u8, out_f
    return out_u8 if out_u8 is not None else out_f


def gt_transform(boxes, ratio, flip_width=None, n_box=None):
    """shapes.py:93-101 / 292-300 on the device: boxes (B,G,4) f64 corners * ratio (B,) f64, then mirrored about
    flip_width (B,) f64 where it is >= 0 -> (B,G,4) f64 (rows >= n_box zeroed)."""
    boxes, ratio = _chk(boxes, torch.float64, "boxes", 3), _chk(ratio, torch.float64, "ratio", 1)
    if flip_width is not None:
        flip_width = _chk(flip_width, torch.float64, "flip_width", 1)
    if n_box is not None:
        n_box = _chk(n_box, torch.int32, "n_box", 1)
    ctx = get_context(boxes.device)
    b, g, _ = boxes.shape
    out = ctx.empty((b, g, 4), torch.float64)
    ctx.call("frcnn_gt_transform", ptr(boxes), ptr(n_box), g, b, ptr(ratio), ptr(flip_width), ptr(out))
    return out
