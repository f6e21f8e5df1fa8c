"""GPU parity of the detector half of the hot path at its limits: RoI labelling (label.cu), the detector and RPN losses
(losses.cu), post-processing (postproc.cu) and RoI padding / mini-batch gather (boxes.cu) at COCO-sized class counts
(K up to 128), post-processing rows up to PP_MAX_ROWS = 1024, 256 GT boxes, RoI counts around the 1024-row chunks, and
the exact float32 / float64 threshold boundaries.

Labels, indices, classes, integer boxes and probabilities are bit-exact against oracle.frcnn_oracle; float32
regression targets within 1 ulp (DESIGN.md section 2, exception 2); loss values within 1e-5 relative and gradients
within rtol 1e-4 of a float64 torch restatement of the Keras formulas; every image of a batch bit-identical to its
single-image call."""
import numpy as np
import pytest

from helpers import dev, host
from oracle import frcnn_oracle as O
from test_gpu_targets import assert_f32_ulp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import ops as _ops
    return _ops


# ------------------------------------------------------------------------------------------------
# det_postprocess (postproc.cu)
# ------------------------------------------------------------------------------------------------
def _softmax_rows(rng, shape, scale=2.0):
    logits = scale * rng.standard_normal(shape)
    e = np.exp(logits - logits.max(axis=-1, keepdims=True))
    return (e / e.sum(axis=-1, keepdims=True)).astype(np.float32)


def _pp_inputs(seed, b, m, k):
    from faster_rcnn_b200 import synth
    rng = np.random.default_rng(seed)
    rois = np.stack([synth.random_rois(m, 37, 62, seed * 100 + i) for i in range(b)])
    return rois, _softmax_rows(rng, (b, m, k)), rng.standard_normal((b, m, 4 * (k - 1))).astype(np.float32)


def _oracle_rows(out_cls, bg):
    """The oracle on the rows the kernel reads: with 'bg' not last, out_reg has no columns for class K-1 (its slice in
    the reference is empty), and the kernel drops rows whose arg-max is K-1 like 'bg' rows.  Those rows are handed to
    the oracle as one-hot 'bg' rows, which keeps every other row at its position (positions decide tie order)."""
    k = out_cls.shape[-1]
    if bg == k - 1:
        return out_cls
    out = out_cls.copy()
    drop = np.argmax(out, axis=-1) == k - 1
    out[drop] = 0.0
    out[drop, bg] = 1.0
    return out


def _check_postprocess(ops, rois, out_cls, out_reg, ratios, bg, stride=16, det_threshold=0.0, nms_thresh=0.5,
                       max_boxes=2000, n_rows=None):
    """One launch over the batch; image b must equal the oracle on rows[:clamp(n_rows[b], 0, M)].  Returns the host
    outputs (boxes, probs, cls, count)."""
    b, m, k = out_cls.shape
    out = ops.det_postprocess(dev(rois), dev(out_cls), dev(out_reg), dev(np.asarray(ratios, np.float64)), bg, stride,
                              det_threshold, nms_thresh, max_boxes,
                              None if n_rows is None else dev(np.asarray(n_rows, np.int32)))
    boxes, probs, cls, count = (host(t) for t in out)
    ocls = _oracle_rows(out_cls, bg)
    for i in range(b):
        live = m if n_rows is None else min(max(int(n_rows[i]), 0), m)
        want = O.det_postprocess(rois[i, :live], ocls[i, :live], out_reg[i, :live], bg, stride, ratios[i],
                                 det_threshold=det_threshold, nms_thresh=nms_thresh, max_boxes=max_boxes)
        n = int(count[i])
        assert n == len(want), "image %d: %d detections, oracle %d" % (i, n, len(want))
        assert cls[i, :n].tolist() == [w[0] for w in want]
        assert np.array_equal(boxes[i, :n], np.array([w[1] for w in want], np.int64).reshape(-1, 4))
        assert np.array_equal(probs[i, :n], np.array([w[2] for w in want], np.float32))
        assert np.all(cls[i, n:] == -1) and np.all(boxes[i, n:] == 0) and np.all(probs[i, n:] == 0)
    return boxes, probs, cls, count


@pytest.mark.parametrize("bg_where", ["last", "first", "middle"])
@pytest.mark.parametrize("k", [21, 33, 81, 128])
def test_postprocess_class_counts_and_bg_index(ops, k, bg_where):
    """K up to PP_MAX_CLASSES with 1000 rows per image: at K >= 81 more than 32 classes are present, so warps run NMS
    for several classes (ci += 32) and warp 0 orders the classes over several 32-class rounds."""
    bg = {"last": k - 1, "first": 0, "middle": k // 2}[bg_where]
    rois, oc, orr = _pp_inputs(k * 10 + len(bg_where), 3, 1000, k)
    _, _, cls, count = _check_postprocess(ops, rois, oc, orr, [1.6, 1.0, 0.75], bg)
    present = max(len(set(cls[i, :int(count[i])].tolist())) for i in range(3))
    if k >= 81:
        assert present > 32
    if bg != k - 1:                                      # the rows without regression columns were there to drop
        assert np.any(np.argmax(oc, axis=-1) == k - 1) and not np.any(cls == k - 1)


@pytest.mark.parametrize("m", [1, 63, 320, 1000, 1024])
def test_postprocess_row_counts_and_n_rows(ops, m):
    """M up to PP_MAX_ROWS (M = 1024 takes about 60 KB of opt-in shared memory), six images with different ratios, and
    n_rows of 0, 1, M/2, M, M + 5 and -3.  Rows at and past n_rows hold confident detections that must not show."""
    rois, oc, orr = _pp_inputs(m, 6, m, 21)
    n_rows = [0, 1, m // 2, m, m + 5, -3]
    for i, n in enumerate(n_rows):
        live = min(max(n, 0), m)
        oc[i, live:] = 0.0
        oc[i, live:, 1] = 1.0
    _check_postprocess(ops, rois, oc, orr, [1.6, 1.0, 0.75, 2.2, 1.3, 0.5], 20, n_rows=n_rows)


@pytest.mark.parametrize("max_boxes", [1, 2, 7, 2000])
def test_postprocess_max_boxes_inside_a_class(ops, max_boxes):
    """Image 0: all 1024 rows pick class 5, so one warp runs NMS over 1024 candidates; image 1: 81 classes with per-class
    lists longer than the small caps.  max_boxes cuts inside each class list."""
    rois, oc, orr = _pp_inputs(7, 2, 1024, 81)
    oc[0] = _softmax_rows(np.random.default_rng(8), (1024, 81), 0.5)
    oc[0, :, 5] += 1.0
    oc[0] /= oc[0].sum(axis=-1, keepdims=True)
    assert np.all(np.argmax(oc[0], axis=-1) == 5)
    _, _, cls, count = _check_postprocess(ops, rois, oc, orr, [1.6, 0.75], 80, max_boxes=max_boxes)
    per_class = np.bincount(cls[1, :int(count[1])], minlength=81)
    if max_boxes < 2000:
        assert int(count[0]) == max_boxes and per_class.max() == max_boxes
    else:
        assert int(count[0]) > 7


def test_postprocess_tied_probabilities(ops):
    """Quantised probabilities: many rows of a class share one probability, and duplicated RoIs with different deltas
    overlap, so which tied row NMS keeps depends on the visit order (prob desc, position desc; the oracle's
    stable=True).  Some rows hold two equal maxima: the first one is the class."""
    from faster_rcnn_b200 import synth
    rng = np.random.default_rng(11)
    b, m, k = 2, 1024, 33
    base = synth.random_rois(40, 37, 62, 12)
    rois = np.stack([base[rng.integers(0, 40, m)] for _ in range(b)])
    c = rng.integers(0, 4, (b, m))
    v = rng.choice([0.5, 0.625, 0.75, 0.875], (b, m))
    oc = np.repeat(((1.0 - v) / (k - 1))[..., None], k, axis=-1)
    np.put_along_axis(oc, c[..., None], v[..., None], axis=-1)
    two = rng.random((b, m)) < 0.2                       # two equal maxima at c and c + 5
    oc[two] = 0.1 / (k - 2)
    bi, ri = np.nonzero(two)
    oc[bi, ri, c[two]] = 0.45
    oc[bi, ri, c[two] + 5] = 0.45
    oc = oc.astype(np.float32)
    orr = (0.5 * rng.standard_normal((b, m, 4 * (k - 1)))).astype(np.float32)
    _check_postprocess(ops, rois, oc, orr, [1.6, 1.0], k - 1)


def test_postprocess_nms_threshold_is_inclusive_in_float64(ops):
    """Zero deltas decode to exactly stride * roi in float64.  With nms_thresh equal to the pair's +1 IoU (computed in
    the kernel's order of operations) both boxes survive (`ratio <= thresh`); one float64 step below, the later box
    is suppressed."""
    m, k, stride = 64, 21, 16
    rois = np.zeros((1, m, 4), np.int16)
    rois[0, :, 2:] = 1
    rois[0, 0], rois[0, 1] = [2, 3, 10, 12], [4, 5, 13, 11]
    oc = np.zeros((1, m, k), np.float32)
    oc[0, :, k - 1] = 1.0                                # every other row is 'bg'
    oc[0, 0, 3], oc[0, 0, k - 1] = 0.9, 0.1
    oc[0, 1, 3], oc[0, 1, k - 1] = 0.8, 0.2
    orr = np.zeros((1, m, 4 * (k - 1)), np.float32)
    a, c = (stride * rois[0, 0].astype(np.float64)), (stride * rois[0, 1].astype(np.float64))
    area = lambda q: (q[2] - q[0] + 1.0) * (q[3] - q[1] + 1.0)       # noqa: E731
    iw = max(0.0, min(a[2], c[2]) - max(a[0], c[0]) + 1.0)
    ih = max(0.0, min(a[3], c[3]) - max(a[1], c[1]) + 1.0)
    t = (iw * ih) / (area(a) + area(c) - iw * ih)
    assert 0.0 < t < 1.0
    _, _, _, count = _check_postprocess(ops, rois, oc, orr, [1.0], k - 1, stride, nms_thresh=t)
    assert int(count[0]) == 2
    _, _, _, count = _check_postprocess(ops, rois, oc, orr, [1.0], k - 1, stride, nms_thresh=float(np.nextafter(t, 0.0)))
    assert int(count[0]) == 1


def test_postprocess_detection_threshold_in_float32(ops):
    """`conf < det_threshold` drops a row.  A threshold equal to a row's float32 probability keeps the row; the next
    float32 above drops it.  A threshold float32 cannot represent is rounded to float32 by the kernel (the C ABI takes
    a double, the kernel compares floats), and numpy >= 2 (NEP 50) compares a float32 scalar with a Python float in
    float32 as well, so the oracle agrees: float(conf) plus a quarter ulp rounds to conf and keeps the row, although it
    is larger than conf in float64."""
    rois, oc, orr = _pp_inputs(21, 1, 320, 21)
    top = oc[0].max(axis=-1)
    top[np.argmax(oc[0], axis=-1) == 20] = 0.0           # 'bg' rows never pass
    conf = top.max()                                     # the one row at or above this threshold: NMS never drops it
    assert np.count_nonzero(top == conf) == 1
    up = float(np.nextafter(conf, np.float32(np.inf)))
    quarter = float(conf) + (up - float(conf)) / 4
    assert np.float32(quarter) == conf and quarter > float(conf)
    for thr, n in ((float(conf), 1), (quarter, 1), (up, 0)):
        _, probs, _, count = _check_postprocess(ops, rois, oc, orr, [1.0], 20, det_threshold=thr)
        assert int(count[0]) == n and (n == 0 or probs[0, 0] == conf)


def test_postprocess_rescale_rounds_half_to_even(ops):
    """stride 16 and ratio 32 with zero deltas put v / ratio = roi / 2: odd coordinates land exactly on .5, where
    rint (half to even, Python's round) and round (half away from zero) differ."""
    m, k = 64, 21
    x = np.arange(-7, 57, dtype=np.int16)                # 64 RoIs, x1 and y1 odd and even, some negative
    rois = np.stack([x, x + 1, x + 3, x + 6], axis=1)[None].astype(np.int16)
    oc = np.zeros((1, m, k), np.float32)
    oc[0, np.arange(m), np.arange(m) % (k - 1)] = 0.9    # rows spread over the classes; NMS at 1.0 keeps every row
    oc[0, :, k - 1] = 0.1
    orr = np.zeros((1, m, 4 * (k - 1)), np.float32)
    halves = rois[0].astype(np.float64) / 2.0
    away = np.sign(halves) * np.floor(np.abs(halves) + 0.5)                        # C round(): half away from zero
    assert np.count_nonzero(np.rint(halves) != away) >= 32
    boxes, _, _, count = _check_postprocess(ops, rois, oc, orr, [32.0], k - 1, 16, nms_thresh=1.0)
    assert int(count[0]) == m
    assert np.array_equal(np.sort(boxes[0].reshape(-1)), np.sort(np.rint(halves).astype(np.int64).reshape(-1)))


def test_postprocess_rejects_rows_or_classes_beyond_limits(ops):
    from faster_rcnn_b200 import _lib
    for m, k in ((1025, 21), (64, 129)):
        rois, oc, orr = _pp_inputs(3, 1, m, k)
        with pytest.raises(_lib.FrcnnError) as e:
            ops.det_postprocess(dev(rois), dev(oc), dev(orr), dev(np.array([1.0])), k - 1)
        assert e.value.code == _lib.ERR_UNSUPPORTED


# ------------------------------------------------------------------------------------------------
# label_rois (label.cu)
# ------------------------------------------------------------------------------------------------
def _check_label_rois(ops, rois, gt64, gcls, n_gt, k, n_roi=None):
    """One launch; image b must equal the oracle on rois[:n_roi[b]] x gt[:n_gt[b]] (an image without RoIs or GTs gives
    count 0; the oracle needs a non-empty IoU matrix).  `src` must be the eligible input rows in order."""
    b, n_max, _ = rois.shape
    out = ops.label_rois(dev(rois), dev(gt64), dev(gcls), dev(np.asarray(n_gt, np.int32)), k,
                         None if n_roi is None else dev(np.asarray(n_roi, np.int32)))
    o_rois, o_cls, o_tr, src, count = (host(t) for t in out)
    for i in range(b):
        n = n_max if n_roi is None else min(max(int(n_roi[i]), 0), n_max)
        g = min(max(int(n_gt[i]), 0), gt64.shape[1])
        m = int(count[i])
        if n == 0 or g == 0:
            assert m == 0
            continue
        e_rois, w_cls, w_tr = O.label_rois(rois[i, :n], gt64[i, :g], gcls[i, :g], k)
        best = np.amax(O.iou_matrix(rois[i, :n], gt64[i, :g].astype(np.float32)), axis=1)
        assert m == len(e_rois)
        assert np.array_equal(src[i, :m], np.where(best >= O.DET_MIN_IOU)[0])
        assert np.array_equal(o_rois[i, :m], e_rois) and np.array_equal(o_cls[i, :m], w_cls)
        assert_f32_ulp(o_tr[i, :m], w_tr)
    return o_rois, o_cls, o_tr, src, count


def _gt_set(g, seed, k, g_max):
    from faster_rcnn_b200 import synth
    gt = np.zeros((g_max, 4), np.float64)
    if g:
        gt[:g] = [[v * (1 / 16) for v in x[1:]] for x in synth.gt_boxes(g, 62 * 16, 37 * 16, seed)]
    return gt, (np.arange(g_max) % (k - 1)).astype(np.int32)


@pytest.mark.parametrize("k", [2, 21, 81, 128])
def test_label_rois_gt_and_roi_counts(ops, k):
    """Per image (n_roi, n_gt) through one launch with n_max = 3000 and g_max = FRCNN_MAX_GT = 256: RoI counts around the
    1024-row chunks (0, 1, 1023, 1024, 1025, 3000), GT counts 0, 1, 50 and 256, GT classes covering 0..K-2."""
    from faster_rcnn_b200 import synth
    pairs = [(3000, 256), (1025, 50), (1024, 1), (1023, 0), (1, 50), (0, 50), (3000, 50), (1023, 256)]
    n_max, g_max = 3000, 256
    rois = np.stack([synth.random_rois(n_max, 37, 62, 300 + i) for i in range(len(pairs))])
    gts = [_gt_set(g, 400 + i, k, g_max) for i, (_, g) in enumerate(pairs)]
    gt64, gcls = np.stack([g[0] for g in gts]), np.stack([g[1] for g in gts])
    *_, count = _check_label_rois(ops, rois, gt64, gcls, [p[1] for p in pairs], k, [p[0] for p in pairs])
    assert int(count[0]) > 2048 and int(count[3]) == 0 and int(count[5]) == 0


def test_label_rois_exact_thresholds(ops):
    """RoI [0,0,10,10]: GT [0,0,10,5] gives IoU exactly 0.5 (positive), GT [0,0,10,1] exactly float32(0.1) (eligible,
    'bg'); the float64 corner just below 5 and 1 (below after the float32 copy too) lands on the other side."""
    below5 = float(np.nextafter(np.float32(5), np.float32(0)))
    below1 = float(np.nextafter(np.float32(1), np.float32(0)))
    y2 = [5.0, below5, 1.0, below1]
    rois = np.tile(np.array([0, 0, 10, 10], np.int16), (4, 1, 1))
    gt64 = np.array([[[0.0, 0.0, 10.0, v]] for v in y2])
    gcls = np.full((4, 1), 3, np.int32)
    _, o_cls, _, _, count = _check_label_rois(ops, rois, gt64, gcls, [1] * 4, 21)
    assert count.tolist() == [1, 1, 1, 0]
    assert [int(np.argmax(o_cls[i, 0])) for i in range(3)] == [3, 20, 20]


def test_label_rois_first_gt_wins_ties(ops):
    """Two GTs of different classes with bit-identical IoU against a RoI: the first GT's class and regression target
    win (strict `>` over the GTs, numpy's first arg-max).  Image 1 lists the GTs in the other order."""
    rois = np.array([[0, 0, 10, 10], [0, 0, 10, 20], [2, 0, 12, 10]], np.int16)
    gts = np.array([[0, 0, 10, 5], [0, 5, 10, 10]], np.float64)
    cls = np.array([3, 7], np.int32)
    iou = O.iou_matrix(rois, gts.astype(np.float32))
    assert np.all(iou[:, 0] == iou[:, 1]) and np.all(iou[:, 0] >= 0.1)
    _, o_cls, o_tr, _, count = _check_label_rois(ops, np.stack([rois, rois]), np.stack([gts, gts[::-1]]),
                                                 np.stack([cls, cls[::-1]]), [2, 2], 21)
    assert count.tolist() == [3, 3]
    assert int(np.argmax(o_cls[0, 0])) == 3 and int(np.argmax(o_cls[1, 0])) == 7
    assert o_tr[0, 0, 80 + 13] == -2.5 and o_tr[1, 0, 80 + 29] == 2.5              # ty of the winning GT


def test_label_rois_degenerate_rois(ops):
    """Zero-width and zero-height RoIs (area 0, IoU 0) and RoIs of 182..255 cells a side, whose int16 area wraps in the
    kernel as in numpy (int16 * int16).  The GTs keep every float32 union away from 0 (a 0/0 IoU is not tested)."""
    rng = np.random.default_rng(5)
    n = 600
    x1, y1 = rng.integers(-20, 60, n), rng.integers(-20, 40, n)
    side = rng.choice([0, 1, 5, 150, 181, 182, 200, 255], (n, 2))
    rois = np.stack([x1, y1, x1 + side[:, 0], y1 + side[:, 1]], axis=1).astype(np.int16)
    gt64, gcls = _gt_set(40, 6, 21, 40)
    gt64 = gt64 * 4.0                                    # GTs of up to 100 cells: overlaps with the wrapped RoIs
    gt32 = gt64.astype(np.float32)
    a1 = ((rois[:, 2] - rois[:, 0]) * (rois[:, 3] - rois[:, 1]))                  # int16, wraps like the reference
    assert np.any(a1 < 0) and np.any(a1 == 0)
    a2 = (gt32[:, 2] - gt32[:, 0]) * (gt32[:, 3] - gt32[:, 1])
    w = np.maximum(0, np.minimum(rois[:, None, 2], gt32[None, :, 2]) - np.maximum(rois[:, None, 0], gt32[None, :, 0]))
    h = np.maximum(0, np.minimum(rois[:, None, 3], gt32[None, :, 3]) - np.maximum(rois[:, None, 1], gt32[None, :, 1]))
    assert np.all((a1[:, None] + a2[None, :]) - w * h != 0)
    *_, count = _check_label_rois(ops, rois[None], gt64[None], gcls[None], [40], 21)
    assert int(count[0]) > 0


def test_label_rois_unaligned_bbreg_takes_the_scalar_store(ops):
    """out_bbreg one float past a 16-byte boundary (reachable through the C ABI only) takes the scalar store branch;
    every output equals the aligned call."""
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.runtime import get_context, ptr
    k, n_max, g_max, b = 21, 1500, 50, 2
    rois = np.stack([synth.random_rois(n_max, 37, 62, 70 + i) for i in range(b)])
    gts = [_gt_set(g_max, 80 + i, k, g_max) for i in range(b)]
    gt64, gcls = np.stack([g[0] for g in gts]), np.stack([g[1] for g in gts])
    n_gt = np.array([g_max, 17], np.int32)
    want = [host(t) for t in ops.label_rois(dev(rois), dev(gt64), dev(gcls), dev(n_gt), k)]
    ctx = get_context()
    d_rois, d_gt, d_gcls, d_ngt = dev(rois), dev(gt64), dev(gcls), dev(n_gt)
    o_rois, o_cls = torch.empty((b, n_max, 4), dtype=torch.int16, device="cuda"), torch.empty((b, n_max, k), dtype=torch.int32, device="cuda")
    flat = torch.empty(b * n_max * 8 * (k - 1) + 4, dtype=torch.float32, device="cuda")
    o_tr = flat[1:1 + b * n_max * 8 * (k - 1)]
    assert o_tr.data_ptr() % 16 == 4
    src, count = torch.empty((b, n_max), dtype=torch.int32, device="cuda"), torch.empty((b,), dtype=torch.int32, device="cuda")
    ctx.call("frcnn_label_rois", ptr(d_rois), None, n_max, ptr(d_gt), ptr(d_gcls), ptr(d_ngt), g_max, k, b,
             ptr(o_rois), ptr(o_cls), ptr(o_tr), ptr(src), ptr(count))
    got = [host(o_rois), host(o_cls), host(o_tr).reshape(b, n_max, 8 * (k - 1)), host(src), host(count)]
    assert np.array_equal(got[4], want[4]) and int(want[4].min()) > 0
    for i in range(b):
        m = int(want[4][i])
        for g_, w_ in zip(got[:4], want[:4]):
            assert np.array_equal(g_[i, :m], w_[i, :m])


# ------------------------------------------------------------------------------------------------
# losses (losses.cu)
# ------------------------------------------------------------------------------------------------
# Keras clips with float32 constants: 1 - 1e-7 is 1 - 2^-23 there, 19 % further from 1 than in float64.  The float64
# restatements clip at the same two values, so a clipped output contributes the same term on both sides.
EPS = float(np.float32(1e-7))
ONE_M_EPS = float(np.float32(1.0) - np.float32(1e-7))

def _det_targets(rng, m, k, kind):
    """One-hot y_class (M,K) i32 and y_transform (M,8(K-1)) f32 = [labels | targets] as label_rois writes them:
    'mixed' classes, 'bg' = every row background, 'pos' = no background row."""
    kf = k - 1
    c = {"mixed": rng.integers(0, k, m), "bg": np.full(m, kf), "pos": rng.integers(0, kf, m)}[kind]
    y_cls = np.zeros((m, k), np.int32)
    y_cls[np.arange(m), c] = 1
    y_tr = np.zeros((m, 8 * kf), np.float32)
    for r in np.nonzero(c < kf)[0]:
        y_tr[r, 4 * c[r]:4 * c[r] + 4] = 1.0
        y_tr[r, 4 * kf + 4 * c[r]:4 * kf + 4 * c[r] + 4] = 1.5 * rng.standard_normal(4)
    return y_cls, y_tr


def _det_preds(rng, m, k, y_cls):
    """Softmax-like rows (not renormalised in float32), with rows holding exact 0 and 1 entries: the clip boundaries
    of categorical_crossentropy, where clip_by_value passes the gradient inclusively."""
    cp = _softmax_rows(rng, (m, k))
    true = np.argmax(y_cls, axis=1)
    if m > 0:
        cp[0] = 0.0
        cp[0, true[0]] = 1.0                              # normalised output exactly 1: clipped
    if m > 1:
        cp[1] = 0.0
        cp[1, (true[1] + 1) % k] = 1.0                   # the true class exactly 0: clipped
    if m > 2:
        cp[2, (true[2] + 1) % k] = 0.0                   # one exact 0 elsewhere
    rp = (1.5 * rng.standard_normal((m, 4 * (k - 1)))).astype(np.float32)
    return cp, rp


def _det_losses_f64(y_cls, y_tr, cp, rp):
    """float64 torch restatement of loss_functions.py:51-76 (categorical cross entropy after normalisation and clip;
    smooth L1 over the labelled columns / sum(1e-4 + mask)) -> (cls, box, d cls / d cp, d box / d rp)."""
    import torch
    kf4 = rp.shape[-1]
    a = torch.tensor(cp, dtype=torch.float64, device="cuda", requires_grad=True)
    b = torch.tensor(rp, dtype=torch.float64, device="cuda", requires_grad=True)
    t = torch.tensor(y_cls, dtype=torch.float64, device="cuda")
    mask = torch.tensor(y_tr[..., :kf4], dtype=torch.float64, device="cuda")
    tgt = torch.tensor(y_tr[..., kf4:], dtype=torch.float64, device="cuda")
    yn = (a / a.sum(dim=-1, keepdim=True)).clamp(EPS, ONE_M_EPS)
    l_c = (-(t * torch.log(yn)).sum(dim=-1)).mean()
    x = tgt - b
    l_b = (mask * torch.where(x.abs() <= 1, 0.5 * x * x, x.abs() - 0.5)).sum() / (1e-4 + mask).sum()
    (l_c + l_b).backward()
    return l_c.item(), l_b.item(), a.grad.cpu().numpy(), b.grad.cpu().numpy()


def _check_det_losses(ops, y_cls, y_tr, cp, rp):
    loss, g_cls, g_reg = (host(t) for t in ops.det_losses(dev(y_cls[None]), dev(y_tr[None]), dev(cp[None]),
                                                          dev(rp[None]), want_grad=True))
    w_c, w_b, w_gc, w_gr = _det_losses_f64(y_cls, y_tr, cp, rp)
    assert abs(loss[0, 0] - w_c) <= 1e-5 * abs(w_c) and abs(loss[0, 1] - w_b) <= 1e-5 * abs(w_b)
    assert np.allclose(g_cls[0], w_gc, rtol=1e-4, atol=1e-9) and np.allclose(g_reg[0], w_gr, rtol=1e-4, atol=1e-12)
    return loss[0], g_cls[0], g_reg[0]


@pytest.mark.parametrize("k", [2, 21, 81, 128])
@pytest.mark.parametrize("m", [1, 64, 1023, 1025, 4096])
def test_det_losses_shapes(ops, m, k):
    """Rows past the CTA's 1024 threads (every thread walks several rows) and K from 2 to 128."""
    rng = np.random.default_rng(m * 1000 + k)
    y_cls, y_tr = _det_targets(rng, m, k, "mixed")
    cp, rp = _det_preds(rng, m, k, y_cls)
    _check_det_losses(ops, y_cls, y_tr, cp, rp)


@pytest.mark.parametrize("kind", ["bg", "pos"])
def test_det_losses_all_background_or_all_positive(ops, kind):
    """All background: the box loss is exactly 0 over a denominator of only 1e-4 * M * 4(K-1), and its gradient is a
    finite 0.  All positive: every row contributes a box term."""
    rng = np.random.default_rng(41 if kind == "bg" else 42)
    y_cls, y_tr = _det_targets(rng, 1025, 81, kind)
    cp, rp = _det_preds(rng, 1025, 81, y_cls)
    loss, _, g_reg = _check_det_losses(ops, y_cls, y_tr, cp, rp)
    if kind == "bg":
        assert loss[1] == 0.0 and np.all(g_reg == 0.0)
    else:
        assert loss[1] > 0.0 and np.count_nonzero(np.any(g_reg != 0.0, axis=1)) == 1025


def test_det_losses_batch_on_label_rois_targets(ops):
    """label_rois' own outputs at K = 81 as targets; each image of a B = 3 batch gets the bits of its single-image call
    (the float64 fixed-tree reductions do not depend on the other images)."""
    from faster_rcnn_b200 import synth
    k, n_max, b = 81, 2500, 3
    rois = np.stack([synth.random_rois(n_max, 37, 62, 90 + i) for i in range(b)])
    gts = [_gt_set(50, 95 + i, k, 50) for i in range(b)]
    gt64, gcls = np.stack([g[0] for g in gts]), np.stack([g[1] for g in gts])
    _, y_cls, y_tr, _, count = (host(t) for t in ops.label_rois(dev(rois), dev(gt64), dev(gcls), dev(np.full(b, 50, np.int32)), k))
    m = int(count.min())
    assert m > 1024
    y_cls, y_tr = np.ascontiguousarray(y_cls[:, :m]), np.ascontiguousarray(y_tr[:, :m])
    assert 0 < int(y_cls[..., -1].sum()) < b * m
    rng = np.random.default_rng(96)
    preds = [_det_preds(rng, m, k, y_cls[i]) for i in range(b)]
    cp, rp = np.stack([p[0] for p in preds]), np.stack([p[1] for p in preds])
    batch = [host(t) for t in ops.det_losses(dev(y_cls), dev(y_tr), dev(cp), dev(rp), want_grad=True)]
    for i in range(b):
        single = _check_det_losses(ops, y_cls[i], y_tr[i], cp[i], rp[i])
        for got, want in zip(batch, single):
            assert np.array_equal(got[i], want)


def _rpn_case(rng, n, kind):
    """Unpacked RPN labels of one image: 256 usable anchors (at most 128 positive) plus positives that are not usable
    (out of bounds); 'no_use' = no usable anchor, 'no_pos' = no positive."""
    can_use, is_pos = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    idx = rng.permutation(n)
    if kind != "no_use":
        can_use[idx[:256]] = 1
    if kind != "no_pos":
        is_pos[idx[:100]] = 1
        is_pos[idx[300:340]] = 1
    bbreg = (2.0 * rng.standard_normal((n, 4))).astype(np.float32)
    cls_pred = np.clip(rng.uniform(0, 1, n), 1e-4, 1 - 1e-4).astype(np.float32)
    cls_pred[idx[:8]] = [0.0, 1.0, 0.0, 1.0, 1e-9, 1 - 1e-9, 0.5, 0.25]          # usable anchors at the clip range
    reg_pred = (1.5 * rng.standard_normal((n, 4))).astype(np.float32)
    return can_use, is_pos, bbreg, cls_pred, reg_pred


def _rpn_losses_f64(can_use, is_pos, bbreg, cls_pred, reg_pred):
    """float64 torch restatement of loss_functions.py:15-48 (the box mask applied outside the sum, Keras' mean)."""
    import torch
    d = lambda x: torch.tensor(x, dtype=torch.float64, device="cuda")            # noqa: E731
    p, q = d(cls_pred).requires_grad_(True), d(reg_pred).requires_grad_(True)
    sel, z = d(can_use), d(is_pos)
    pc = p.clamp(EPS, ONE_M_EPS)
    x = torch.log(pc / (1 - pc))
    # softplus(x) - x*z is max(x,0) - x*z + log1p(exp(-|x|)) without the kinks at x = 0 (p = 0.5), where autograd's
    # subgradients of max and abs would give 1 - z instead of the derivative sigmoid(0) - z
    l_cls = (sel * (torch.nn.functional.softplus(x) - x * z)).sum() / 256
    dd = (d(bbreg) - q).abs()
    s = torch.where(dd <= 1, 0.5 * dd * dd, dd - 0.5).sum()
    l_reg = ((sel * z).unsqueeze(-1).expand(-1, 4) * (10 * s / 2400)).mean()
    (l_cls + l_reg).backward()
    return l_cls.item(), l_reg.item(), p.grad.cpu().numpy(), q.grad.cpu().numpy()


@pytest.mark.parametrize("n", [38 * 94 * 18, 5000])
def test_rpn_losses_batch_and_empty_images(ops, n):
    """rpn_losses (uniform entry) at KITTI's 38 x 94 x 18 anchors and at a size that is not a multiple of 1024, B = 4:
    image 1 has no usable anchor (class loss 0), image 2 no positive (box loss 0, zero box gradient).  Every image
    equals its single-image call bit for bit and the float64 restatement within tolerance."""
    rng = np.random.default_rng(n)
    cases = [_rpn_case(rng, n, kind) for kind in ("mixed", "no_use", "no_pos", "mixed")]
    stacked = [np.stack([c[j] for c in cases]) for j in range(5)]
    batch = [host(t) for t in ops.rpn_losses(*(dev(x) for x in stacked), want_grad=True)]
    for i, c in enumerate(cases):
        single = [host(t) for t in ops.rpn_losses(*(dev(x[None]) for x in c), want_grad=True)]
        for got, want in zip(batch, single):
            assert np.array_equal(got[i], want[0])
        w_c, w_r, w_gc, w_gr = _rpn_losses_f64(*c)
        loss = single[0][0]
        assert abs(loss[0] - w_c) <= 1e-5 * abs(w_c) and abs(loss[1] - w_r) <= 1e-5 * abs(w_r)
        assert np.allclose(single[1][0], w_gc, rtol=1e-4, atol=1e-9)
        assert np.allclose(single[2][0], w_gr, rtol=1e-4, atol=1e-12)
    assert batch[0][1].tolist() == [0.0, 0.0] and np.all(batch[1][1] == 0.0)      # nothing usable: nothing selected
    assert batch[0][2, 1] == 0.0 and np.all(batch[2][2] == 0.0) and batch[0][2, 0] > 0.0


# ------------------------------------------------------------------------------------------------
# pad_rois and gather_det_samples (boxes.cu)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("group", [1, 64, 300])
def test_pad_rois_counts(ops, group):
    """voc_dets' batching rule on rois[:clamp(count, 0, n_max)]: rows up to the count rounded up to `group` (padding
    = copies of the last group's first RoI), zero rows after; a negative count is an empty list (rows 0)."""
    from faster_rcnn_b200 import synth, voc_dets
    n_max = 700
    counts = [0, 1, group, group + 1, n_max, n_max + 7, -1, -(2 * group + 1)]
    rois = np.stack([synth.random_rois(n_max, 37, 62, 500 + i) for i in range(len(counts))])
    out, rows = (host(t) for t in ops.pad_rois(dev(rois), dev(np.array(counts, np.int32)), group))
    m = -(-n_max // group) * group
    assert out.shape == (len(counts), m, 4)
    for i, c in enumerate(counts):
        n = min(max(c, 0), n_max)
        want = voc_dets.pad_roi_batches(rois[i, :n], group)
        assert int(rows[i]) == len(want) == -(-n // group) * group
        assert np.array_equal(out[i, :len(want)], want) and np.all(out[i, len(want):] == 0)


@pytest.mark.parametrize("k", [2, 81, 128])
def test_gather_det_samples_class_counts(ops, k):
    """K class words and 8(K-1) target words per row (8 at K = 2, 1016 = eight rounds of 128 threads at K = 128);
    indices -1, n_max and beyond give zero rows, repeats copy the row again."""
    rng = np.random.default_rng(k)
    b, n_max = 2, 50
    rois = rng.integers(-100, 100, (b, n_max, 4)).astype(np.int16)
    y_cls = rng.integers(-5, 5, (b, n_max, k)).astype(np.int32)
    y_tr = rng.standard_normal((b, n_max, 8 * (k - 1))).astype(np.float32)
    index = np.array([[0, -1, n_max, n_max - 1, 3, 3, 3, n_max + 9, -7, 17, 0, 49],
                      [5, 5, -1, -1, 48, n_max, 1, 2, 3, 4, 1, 1]], np.int32)
    o_rois, o_cls, o_tr = (host(t) for t in ops.gather_det_samples(dev(rois), dev(y_cls), dev(y_tr), dev(index)))
    valid = (index >= 0) & (index < n_max)
    safe = np.where(valid, index, 0)
    for arr, got in ((rois, o_rois), (y_cls, o_cls), (y_tr, o_tr)):
        want = np.take_along_axis(arr, safe[..., None], axis=1) * valid[..., None]
        assert np.array_equal(got, want.astype(arr.dtype))
