"""Pins the numpy oracle against the UNMODIFIED reference, imported live.

Runs only where a reference checkout is present (oracle/_ref/ or
FRCNN_REFERENCE_DIR, see oracle/ref_loader.py); everywhere else the committed fixtures under
tests/golden/ (made by make_golden.py from the same reference) take over --
see test_oracle_golden.py and test_oracle_eval.py.
"""
import random

import numpy as np
import pytest

from oracle import frcnn_oracle as O
from oracle import ref_loader
from faster_rcnn_b200 import synth

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="reference checkout not present")


@pytest.fixture(scope="module")
def ref():
    return ref_loader.load()


def _ref_image(ref, name, w, h, gts):
    S = ref.shapes
    boxes = [S.GroundTruthBox(c, False, S.Box(x1, y1, x2, y2)) for c, x1, y1, x2, y2 in gts]
    return S.Image(S.Metadata(name, w, h, boxes, '/nonexistent.jpg'))


def test_anchor_tables(ref):
    for scales in ([128, 256, 512], [16, 32, 64, 128, 256, 512]):
        assert np.array_equal(O.anchor_table(scales), ref.util.get_anchors(scales))
    assert np.array_equal(O.anchor_table(), ref.shared_constants.DEFAULT_ANCHORS)


@pytest.mark.parametrize("rows,cols,scales,seed", [(38, 63, [128, 256, 512], 1), (38, 94, None, 2), (5, 7, [128, 256, 512], 3)])
def test_proposals_and_topk(ref, rows, cols, scales, seed):
    dims = O.anchor_table(scales) if scales else O.anchor_table()
    cls, regr = synth.rpn_outputs(rows, cols, len(dims), seed)
    with ref_loader.quiet():
        want = ref.det_util._get_rois(regr.copy(), dims, 16)
        v = ref.det_util._get_valid_box_idxs(want)
    got = O.proposals_from_rpn(regr.copy(), dims, 16)
    assert got.dtype == want.dtype and np.array_equal(got, want)
    assert np.array_equal(O.valid_box_indices(got), v)
    probs = cls.reshape(-1)
    order = probs[v].argsort()[::-1][:8000]                       # det_util.py:151-153 (tie-free input)
    b, p, idx = O.topk_proposals(got, probs, 8000)
    assert np.array_equal(b, want[v][order].astype('int16')) and np.array_equal(p, probs[v][order])
    assert np.array_equal(idx, v[order])


@pytest.mark.parametrize("k,max_boxes,clustered", [(8000, 300, False), (8000, 300, True), (3000, 2000, True)])
def test_nms_int16(ref, k, max_boxes, clustered):
    dims = O.anchor_table([128, 256, 512])
    cls, regr = synth.rpn_outputs(38, 63, 9, 11, clustered=clustered)
    b, p, _ = O.topk_proposals(O.proposals_from_rpn(regr, dims, 16), cls.reshape(-1), k)
    with ref_loader.quiet():
        wb, wp = ref.det_util.nms(b, p, overlap_thresh=0.7, max_boxes=max_boxes)
    pick = O.greedy_nms(b, p, 0.7, max_boxes)
    assert np.array_equal(b[pick], wb) and np.array_equal(p[pick], wp)
    for stable in (True, False):                                   # tie-free: both orders agree
        gb, gp = O.nms(b, p, 0.7, max_boxes, stable=stable)
        assert np.array_equal(gb, wb) and np.array_equal(gp, wp)


def test_nms_float64_and_empty(ref):
    rng = np.random.default_rng(5)
    xy = rng.uniform(0, 500, (400, 2))
    wh = rng.uniform(5, 200, (400, 2))
    boxes = np.concatenate([xy, xy + wh], axis=1)
    probs = rng.permutation(400).astype(np.float32) / 400
    with ref_loader.quiet():
        wb, wp = ref.det_util.nms(boxes, probs, overlap_thresh=0.5, max_boxes=2000)
        assert ref.det_util.nms(boxes[:0], probs[:0]) == []
    gb, gp = O.nms(boxes, probs, 0.5, 2000)
    assert np.array_equal(gb, wb) and np.array_equal(gp, wp)
    assert O.nms(boxes[:0], probs[:0]) == []


def test_iou_and_regression_params(ref):
    rng = np.random.default_rng(9)
    anc = O.pixel_anchors(38, 63, O.anchor_table([128, 256, 512]), 16)
    with ref_loader.quiet():
        assert np.array_equal(anc, ref.rpn_util._get_all_anchor_coords(38, 63, O.anchor_table([128, 256, 512]), 16))
    gt = np.array([[g[1], g[2], g[3], g[4]] for g in synth.gt_boxes(50, 1000, 600, 4)], dtype=np.float32)
    with ref_loader.quiet():
        want = ref.util.cross_ious(anc, gt)
    got = O.iou_matrix(anc, gt)
    assert got.dtype == np.float32 and np.array_equal(got, want)
    rois = synth.random_rois(300, 38, 63, 2)
    with ref_loader.quiet():
        assert np.array_equal(O.iou_matrix(rois, gt / 16), ref.util.cross_ious(rois, gt / 16))
    for _ in range(20):
        a = np.array([10, 20, 138, 148]) + rng.integers(0, 5, 4)
        assert O.regression_params(a, gt[3]) == ref.util.get_reg_params(a, gt[3])


@pytest.mark.parametrize("n_gt,seed", [(50, 1), (3, 2), (1, 3)])
def test_rpn_labels(ref, n_gt, seed):
    dims = O.anchor_table([128, 256, 512])
    gts = synth.gt_boxes(n_gt, 1000, 600, seed)
    img = _ref_image(ref, 'synth%d' % seed, 1000, 600, gts)
    mgr = ref.rpn_util.RpnTrainingManager(O.conv_dims_resnet, 16, preprocess_func=None, anchor_dims=dims)
    with ref_loader.quiet():
        mgr._process(img)
    want = mgr._cache[img.cache_key]
    gt = np.array([g[1:] for g in gts], dtype=np.float32)
    rows, cols = O.conv_dims_resnet(600, 1000)
    cu, ip, bb = O.label_anchors(1000, 600, gt, rows, cols, dims, 16)
    assert np.array_equal(cu, want['can_use']) and np.array_equal(ip, want['is_pos'])
    assert np.array_equal(bb, want['bbreg_targets'])
    random.seed(1)
    with ref_loader.quiet():
        y_cls, y_reg = mgr.rpn_y_true(img)
    random.seed(1)
    cu2 = O.sample_rpn(ip, cu.copy())
    g_cls, g_reg = O.pack_rpn_targets(cu2, ip, bb, rows, cols, len(dims))
    assert g_cls.dtype == y_cls.dtype and np.array_equal(g_cls, y_cls)
    assert g_reg.dtype == y_reg.dtype and np.array_equal(g_reg, y_reg)


@pytest.mark.parametrize("seed", [1, 2])
def test_det_labels_and_sampling(ref, seed):
    gts = synth.gt_boxes(50, 1000, 600, seed)
    img = _ref_image(ref, 'synth%d' % seed, 1000, 600, gts)
    rois = synth.random_rois(2000, 38, 63, seed)
    mapping = synth.VOC_CLASS_MAPPING
    with ref_loader.quiet():
        w_rois, w_cls, w_tr = ref.det_util._rois_to_truth(rois, img, mapping, stride=16)
    gt64 = np.array([[v * (1 / 16) for v in g[1:]] for g in gts], dtype=np.float64)
    gidx = np.array([mapping[g[0]] for g in gts])
    g_rois, g_cls, g_tr = O.label_rois(rois, gt64, gidx, len(mapping))
    assert np.array_equal(g_rois, w_rois) and g_cls.dtype == w_cls.dtype and np.array_equal(g_cls, w_cls)
    assert g_tr.dtype == w_tr.dtype and np.array_equal(g_tr, w_tr)
    found = w_cls[:, -1] == 0
    for flags in (found, np.zeros_like(found), np.ones_like(found), found & (np.arange(len(found)) < 40)):
        np.random.seed(1337)
        with ref_loader.quiet():
            want = ref.det_util._get_det_samples(flags, 64)
        np.random.seed(1337)
        assert O.sample_det(flags, 64) == want


def test_det_postprocess(ref):
    """voc_dets.py cannot be imported (Keras), so its loop (voc_dets.py:51-86) is
    replayed here around the reference's own nms/transform."""
    mapping = synth.VOC_CLASS_MAPPING
    rev = {v: k for k, v in mapping.items()}
    rois = synth.random_rois(320, 37, 62, 3)
    out_cls, out_reg = synth.detector_outputs(320, 21, 3)
    ratio, stride = 1.6, 16
    bb, pp = {}, {}
    for r in range(320):
        c = np.argmax(out_cls[r])
        if c == mapping['bg']:
            continue
        x1, y1, x2, y2 = rois[r]
        t = out_reg[r, c * 4:(c + 1) * 4] / ref.shared_constants.BBREG_MULTIPLIERS
        px = ref.util.transform([x1, y1, x2, y2], t)
        bb.setdefault(rev[c], []).append([stride * v for v in px])
        pp.setdefault(rev[c], []).append(out_cls[r, c])
    want = []
    for name in bb:
        with ref_loader.quiet():
            nb, npb = ref.det_util.nms(np.array(bb[name]), np.array(pp[name]), overlap_thresh=0.5, max_boxes=2000)
        for i in range(nb.shape[0]):
            want.append((mapping[name], [int(round(v / ratio)) for v in nb[i]], npb[i]))
    got = O.det_postprocess(rois, out_cls, out_reg, mapping['bg'], stride, ratio)
    assert len(got) == len(want) > 50
    for (gc, gb, gp), (wc, wb, wp) in zip(got, want):
        assert gc == wc and list(gb) == wb and gp == wp


def test_known_answer_000005(ref):
    """SURVEY.md section 8c (ii): labelling known-answer on the one shipped VOC image."""
    img = ref.voc.extract_img_data(ref_loader.VOC_DIR, '000005').resize_within_bounds(600, 1000)[0]
    assert (img.width, img.height) == (800, 600)
    dims = O.anchor_table([128, 256, 512])
    gt = ref.util.get_bbox_coords(img.gt_boxes)
    rows, cols = O.conv_dims_resnet(img.height, img.width)
    cu, ip, bb = O.label_anchors(img.width, img.height, gt, rows, cols, dims, 16)
    assert (rows, cols) == (38, 50)
    assert np.where(ip)[0].tolist() == [7454, 10586, 11036, 11486, 11963, 12413, 12863, 13079, 13529, 13680, 13979]
    assert int(cu.sum()) == 5287
    assert abs(float(np.abs(bb).sum()) - 33.408202) < 1e-4


def test_voc_eval_live(ref, tmp_path):
    """eval_dets.voc_eval (imports without Keras) run live on the reference's own annotations vs the eval oracle."""
    import contextlib
    import io
    import sys
    from oracle import eval_oracle as E
    sys.path.insert(0, ref_loader.REF_DIR)
    import eval_dets as ref_eval
    root = ref_loader.VOC_DIR
    names = [l.strip() for l in open(root + '/ImageSets/Main/trainval.txt')][400:520]
    rng = np.random.default_rng(11)
    iset = tmp_path / 'set.txt'
    iset.write_text('\n'.join(names) + '\n')
    lines, gt = [], {}
    for nm in names:
        objs = [b for b in ref.voc.extract_img_data(root, nm).gt_boxes if b.obj_cls == 'person']
        gt[nm] = (np.array([b.corners for b in objs]).reshape(-1, 4), np.array([b.difficult for b in objs], dtype=bool))
        for b in objs:
            for _ in range(rng.integers(0, 3)):
                lines.append((nm, np.round(np.asarray(b.corners, float) + rng.normal(0, 8, 4), 1)))
        lines.append((nm, np.array([5., 5., 60., 80.])))
    conf = rng.permutation(len(lines)) / len(lines)
    det_file = tmp_path / 'comp3_det_test_person.txt'
    det_file.write_text(''.join("%s %r %r %r %r %r\n" % (n, float(c), *[float(v) for v in b]) for (n, b), c in zip(lines, conf)))
    with contextlib.redirect_stdout(io.StringIO()):
        rec, prec, ap = ref_eval.voc_eval(root, str(det_file), str(iset), 'person', ovthresh=0.5)
    r, p, a = E.voc_match([l[0] for l in lines], conf, np.array([l[1] for l in lines]), gt)
    assert np.array_equal(r, rec) and np.array_equal(p, prec) and a == ap and ap > 0.05
    assert E.voc_ap(rec, prec, False) == ref_eval.voc_ap(rec, prec, False)


def test_shapes_value_objects_match_the_reference(ref):
    """faster_rcnn_b200.shapes (Box / GroundTruthBox / Image geometry: dims, centres, resize, resize_within_bounds,
    horizontal_flip, cache_key) against the reference's shapes.py on the VOC 000005 boxes and synthetic ones."""
    from faster_rcnn_b200 import shapes as M
    S = ref.shapes
    gts = [("chair", 262, 210, 323, 338), ("chair", 164, 263, 252, 371), ("chair", 4, 243, 66, 373)] + synth.gt_boxes(9, 500, 375, 4)
    mine = M.Image("000005", 500, 375, [M.GroundTruthBox(c, False, M.Box(*b)) for c, *b in gts])
    theirs = _ref_image(ref, "000005", 500, 375, gts)

    def same(a, b):
        assert (a.width, a.height, a.cache_key, a.num_gt_boxes) == (b.width, b.height, b.cache_key, b.num_gt_boxes)
        for ga, gb in zip(a.gt_boxes, b.gt_boxes):
            assert ga.obj_cls == gb.obj_cls and ga.difficult == gb.difficult
            for attr in ("corners", "corner_dims", "center_dims"):
                assert np.array_equal(getattr(ga, attr), getattr(gb, attr))
            assert (ga.x1, ga.y1, ga.x2, ga.y2, ga.width, ga.height, ga.x_center, ga.y_center) == \
                   (gb.x1, gb.y1, gb.x2, gb.y2, gb.width, gb.height, gb.x_center, gb.y_center)

    same(mine, theirs)
    (m2, r_m), (t2, r_t) = mine.resize_within_bounds(600, 1000), theirs.resize_within_bounds(600, 1000)
    assert r_m == r_t == 1.6
    same(m2, t2)
    same(m2.horizontal_flip(), t2.horizontal_flip())
    same(m2.horizontal_flip().horizontal_flip(), t2.horizontal_flip().horizontal_flip())
    same(mine.resize(0.37), theirs.resize(0.37))
    for args in ((456, 264, 128, 128), (8, 8, 91, 181), (0, 0, 5, 11)):
        assert np.array_equal(M.Box.from_center_dims_int(*args).corners, S.Box.from_center_dims_int(*args).corners)
    assert np.array_equal(M.Box.from_corners([1, 2, 3, 4]).corners, S.Box.from_corners([1, 2, 3, 4]).corners)


def test_oracle_equals_reference_on_drawn_inputs(ref):
    """hypothesis-drawn boxes, scores, ground truth and image sizes: NMS picks, IoU matrices and RPN labels of the oracle
    equal the live reference bit for bit (tie-free scores: the reference's argsort is only defined there)."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st

    @settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])
    @given(st.integers(0, 2 ** 31 - 1), st.integers(1, 300), st.sampled_from([0.3, 0.5, 0.7]), st.integers(1, 64),
           st.integers(1, 12), st.sampled_from([(1000, 600), (800, 600), (600, 904), (333, 500)]))
    def run(seed, n, thresh, max_boxes, n_gt, wh):
        rng = np.random.default_rng(seed)
        xy = rng.integers(0, 60, (n, 2))
        boxes = np.concatenate([xy, xy + rng.integers(0, 40, (n, 2))], axis=1).astype(np.int16)
        probs = ((rng.permutation(n) + 0.5) / n).astype(np.float32)
        with ref_loader.quiet():
            wb, wp = ref.det_util.nms(boxes, probs, overlap_thresh=thresh, max_boxes=max_boxes)
        pick = O.greedy_nms(boxes, probs, thresh, max_boxes)
        assert np.array_equal(boxes[pick], wb) and np.array_equal(probs[pick], wp)
        a = (rng.integers(0, 200, (n, 4)) + np.array([0, 0, 200, 200])).astype(np.float32)
        g = (rng.integers(0, 200, (n_gt, 4)) + np.array([0, 0, 200, 200])).astype(np.float32)
        assert np.array_equal(O.iou_matrix(a, g), ref.util.cross_ious(a, g))
        w, h = wh
        gts = synth.gt_boxes(n_gt, w, h, seed % 100000)
        img = _ref_image(ref, 'drawn', w, h, gts)
        dims = O.anchor_table([128, 256, 512])
        mgr = ref.rpn_util.RpnTrainingManager(O.conv_dims_resnet, 16, preprocess_func=None, anchor_dims=dims)
        with ref_loader.quiet():
            mgr._process(img)
        want = mgr._cache[img.cache_key]
        rows, cols = O.conv_dims_resnet(h, w)
        cu, ip, bb = O.label_anchors(w, h, np.array([x[1:] for x in gts], np.float32), rows, cols, dims, 16)
        assert np.array_equal(cu, want['can_use']) and np.array_equal(ip, want['is_pos']) and np.array_equal(bb, want['bbreg_targets'])

    run()
