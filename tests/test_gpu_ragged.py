"""Mixed-size batches: a padded (B,R,C,.) batch with per-image extents (rows, cols) must give, image by image, what the
single-shape entry points give on the cropped inputs [:rows_b, :cols_b], with zero padding in every output and without
reading the padding of any input.  The argument checks of ops.pad_batch need no GPU."""
import random

import numpy as np
import pytest

from helpers import FakeImage, dev, golden, host
from oracle import frcnn_oracle as O

GARBAGE = (np.nan, np.inf, -np.inf, 1e30)


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import _build, ops as ops_mod
    _build.build()
    return ops_mod


def _voc_shapes():
    g = golden("voc_gt_200")
    return [tuple(O.conv_dims_resnet(int(h), int(w))) for w, h in g["img_wh"]]


def _padded_heads(shapes, n_anchors, seed, fill=0.0, scores=None):
    """per-image synthetic heads laid into one padded batch whose padding holds `fill` (cycled through GARBAGE when
    fill is None)"""
    from faster_rcnn_b200 import synth
    rows, cols = max(s[0] for s in shapes), max(s[1] for s in shapes)
    cls = np.empty((len(shapes), rows, cols, n_anchors), np.float32)
    regr = np.empty((len(shapes), rows, cols, 4 * n_anchors), np.float32)
    per = []
    for b, (r, c) in enumerate(shapes):
        v = GARBAGE[b % len(GARBAGE)] if fill is None else fill
        cls[b], regr[b] = v, v
        if r and c:
            pc, pr = synth.rpn_outputs(r, c, n_anchors, seed + b)
            if scores is not None:
                pc = scores(pc)
            cls[b, :r, :c], regr[b, :r, :c] = pc[0], pr[0]
            per.append((pc, pr))
        else:
            per.append(None)
    return cls, regr, per, np.array(shapes, np.int32).reshape(-1, 2)


MIXES = {
    "voc_all_30_shapes": (sorted(set(_voc_shapes())), [128, 256, 512], 8000, 300),
    "kitti_anchors": ([(20, 40), (24, 31), (17, 44)], None, 12000, 2000),
    "tiny_and_empty": ([(1, 1), (0, 5), (3, 0), (2, 3), (9, 14)], [128, 256, 512], 8000, 300),
    "k_above_anchor_count": ([(4, 6), (10, 12), (7, 3)], [128, 256, 512], 900, 300),
}


def _check_ragged_topk(ops, shapes, dims, k, max_boxes, scores=None):
    a = len(dims)
    cls, regr, per, ext = _padded_heads(shapes, a, 300, scores=scores)
    boxes, sc, index, count = (host(t) for t in ops.decode_topk(dev(regr), dev(cls), dims, 16, k, extents=dev(ext)))
    rois, rsc, rcount = (host(t) for t in ops.proposals(dev(regr), dev(cls), dims, 16, k, 0.7, max_boxes,
                                                         extents=dev(ext)))
    # the padding of the inputs is never read
    g_cls, g_regr, _, _ = _padded_heads(shapes, a, 300, fill=None, scores=scores)
    again = [host(t) for t in ops.decode_topk(dev(g_regr), dev(g_cls), dims, 16, k, extents=dev(ext))]
    again += [host(t) for t in ops.proposals(dev(g_regr), dev(g_cls), dims, 16, k, 0.7, max_boxes, extents=dev(ext))]
    for x, y in zip((boxes, sc, index, count, rois, rsc, rcount), again):
        assert np.array_equal(x, y, equal_nan=False)
    for b, p in enumerate(per):
        if p is None:
            assert count[b] == 0 and rcount[b] == 0
            assert not boxes[b].any() and not sc[b].any() and (index[b] == -1).all()
            assert not rois[b].any() and not rsc[b].any()
            continue
        wb, ws, wi, wc = (host(t)[0] for t in ops.decode_topk(dev(p[1]), dev(p[0]), dims, 16, k))
        kb = wb.shape[0]
        assert count[b] == wc
        assert np.array_equal(boxes[b, :kb], wb) and np.array_equal(sc[b, :kb], ws) and np.array_equal(index[b, :kb], wi)
        assert not boxes[b, kb:].any() and not sc[b, kb:].any() and (index[b, kb:] == -1).all()
        pr, ps, pn = (host(t)[0] for t in ops.proposals(dev(p[1]), dev(p[0]), dims, 16, k, 0.7, max_boxes))
        assert rcount[b] == pn and np.array_equal(rois[b], pr) and np.array_equal(rsc[b], ps)


@pytest.mark.gpu
@pytest.mark.parametrize("mix", sorted(MIXES))
def test_ragged_proposals_equal_cropped_calls(ops, mix):
    shapes, scales, k, max_boxes = MIXES[mix]
    dims = O.anchor_table(scales) if scales else O.anchor_table()
    _check_ragged_topk(ops, shapes, dims, k, max_boxes)


@pytest.mark.gpu
def test_ragged_proposals_with_tied_scores(ops):
    """a few score levels: the sort position (padded index) must order ties like the image's own index"""
    dims = O.anchor_table([128, 256, 512])
    _check_ragged_topk(ops, [(38, 50), (38, 57), (50, 38)], dims, 8000, 300,
                       scores=lambda c: (np.floor(c * 7) / 7 + 0.01).astype(np.float32))


@pytest.mark.gpu
def test_ragged_proposals_with_full_extents_equal_the_uniform_entry(ops):
    from faster_rcnn_b200 import synth
    dims = O.anchor_table([128, 256, 512])
    pairs = [synth.rpn_outputs(38, 63, 9, 40 + i) for i in range(4)]
    cls, regr = dev(np.concatenate([p[0] for p in pairs])), dev(np.concatenate([p[1] for p in pairs]))
    ext = dev(np.tile(np.array([[38, 63]], np.int32), (4, 1)))
    for got, want in zip(ops.decode_topk(regr, cls, dims, 16, 8000, extents=ext), ops.decode_topk(regr, cls, dims, 16, 8000)):
        assert np.array_equal(host(got), host(want))
    for got, want in zip(ops.proposals(regr, cls, dims, 16, 12000, 0.7, 2000, extents=ext),
                         ops.proposals(regr, cls, dims, 16, 12000, 0.7, 2000)):
        assert np.array_equal(host(got), host(want))
    # extents beyond the map are clamped to it
    big = dev(np.full((4, 2), 10000, np.int32))
    for got, want in zip(ops.decode_topk(regr, cls, dims, 16, 8000, extents=big), ops.decode_topk(regr, cls, dims, 16, 8000)):
        assert np.array_equal(host(got), host(want))


@pytest.mark.gpu
def test_ragged_decode_topk_rejects_dense_boxes(ops):
    from faster_rcnn_b200 import _lib, synth
    dims = O.anchor_table([128, 256, 512])
    cls, regr = (dev(x) for x in synth.rpn_outputs(5, 6, 9, 1))
    ext = dev(np.array([[5, 6]], np.int32))
    with pytest.raises(ValueError):
        ops.decode_topk(regr, cls, dims, 16, 100, want_dense=True, extents=ext)
    import torch
    from faster_rcnn_b200.runtime import get_context, ptr
    ctx = get_context()
    anc, a = ctx.anchors(dims)
    outs = [torch.empty(s, dtype=d, device="cuda") for s, d in (((1, 100, 4), torch.int16), ((1, 100), torch.float32),
                                                                  ((1, 100), torch.int32), ((1,), torch.int32),
                                                                  ((1, 270, 4), torch.float32))]
    with pytest.raises(_lib.FrcnnError) as e:
        ctx.call("frcnn_decode_topk_ragged", ptr(regr), ptr(cls), anc, 5, 6, a, 16, 100, 1, ptr(ext), *map(ptr, outs))
    assert e.value.code == _lib.ERR_INVALID


def _voc_gt():
    g = golden("voc_gt_200")
    gts = [g["gt"][g["offsets"][i]:g["offsets"][i + 1]] for i in range(len(g["names"]))]
    return g, gts


@pytest.mark.gpu
def test_ragged_labels_on_real_voc_ground_truth_in_one_launch(ops):
    """all 200 VOC GT sets (30 conv shapes) as ONE padded launch: every crop hashes to the reference digests"""
    import hashlib
    g, gts = _voc_gt()
    dims = O.anchor_table([128, 256, 512])
    ext = np.array(_voc_shapes(), np.int32)
    rows, cols = (int(v) for v in ext.max(axis=0))
    g_max = max(len(x) for x in gts)
    gt = np.zeros((len(gts), g_max, 4), np.float32)
    for b, x in enumerate(gts):
        gt[b, :len(x)] = x
    n_gt = np.array([len(x) for x in gts], np.int32)
    cu, ip, bb, counts = (host(t) for t in ops.label_anchors(dev(gt), dev(n_gt), dev(g["img_wh"], np.int32), rows, cols,
                                                             dims, 16, extents=dev(ext)))
    a = len(dims)
    cu, ip, bb = cu.reshape(-1, rows, cols, a), ip.reshape(-1, rows, cols, a), bb.reshape(-1, rows, cols, a, 4)
    for b in range(len(gts)):
        r, c = ext[b]
        cub, ipb = cu[b, :r, :c].reshape(-1).view(np.bool_), ip[b, :r, :c].reshape(-1).view(np.bool_)
        assert hashlib.sha1(cub.tobytes() + ipb.tobytes()).hexdigest()[:16] == str(g["label_sha1"][b]), g["names"][b]
        assert int(ipb.sum()) == int(g["n_pos"][b]) and int(cub.sum()) == int(g["n_use"][b])
        assert counts[b].tolist() == [int((cub & ipb).sum()), int((cub & ~ipb).sum())]
        pad = np.ones((rows, cols), bool)
        pad[:r, :c] = False
        assert not cu[b][pad].any() and not ip[b][pad].any() and not bb[b][pad].any()
    # bbreg of the crops equals the single-shape call (one of the shape groups)
    idx = [i for i in range(len(gts)) if tuple(ext[i]) == tuple(ext[0])][:8]
    wcu, wip, wbb, _ = (host(t) for t in ops.label_anchors(dev(gt[idx]), dev(n_gt[idx]), dev(g["img_wh"][idx], np.int32),
                                                           int(ext[0][0]), int(ext[0][1]), dims, 16))
    r, c = ext[0]
    for j, i in enumerate(idx):
        assert np.array_equal(bb[i, :r, :c].reshape(-1, 4), wbb[j])


def _voc_images(n):
    g, gts = _voc_gt()
    names = g["names"]
    return [FakeImage(str(names[i]), int(g["img_wh"][i][0]), int(g["img_wh"][i][1]),
                      [("chair", *row) for row in gts[i].tolist()]) for i in range(n)]


@pytest.mark.gpu
def test_rpn_y_true_ragged_equals_per_image_targets(ops):
    from faster_rcnn_b200 import rpn_util
    dims = O.anchor_table([128, 256, 512])
    a = len(dims)
    images = _voc_images(24)
    mgr = rpn_util.RpnTrainingManager(lambda h, w: O.conv_dims_resnet(h, w), 16, preprocess_func=None, anchor_dims=dims)
    rows, cols = (int(v) + 2 for v in np.array(_voc_shapes()[:24]).max(axis=0))
    random.seed(11)
    y_cls, y_reg, ext = mgr.rpn_y_true_ragged(images, pad_to=(rows, cols))
    assert y_cls.shape == (24, rows, cols, 2 * a) and y_reg.shape == (24, rows, cols, 8 * a)
    assert len({tuple(e) for e in ext}) > 1
    random.seed(11)
    want = [mgr.rpn_y_true(img) for img in images]
    for b, (wc, wr) in enumerate(want):
        r, c = ext[b]
        assert wc.shape[1:3] == (r, c)
        assert np.array_equal(y_cls[b, :r, :c], wc[0]) and np.array_equal(y_reg[b, :r, :c], wr[0])
        pad = np.ones((rows, cols), bool)
        pad[:r, :c] = False
        assert not y_cls[b][pad].any() and not y_reg[b][pad].any()
    # class loss of the padded targets = per-image class loss; no class gradient reaches the padding
    rng = np.random.default_rng(3)
    pred = rng.uniform(0.02, 0.98, (24, rows, cols, a)).astype(np.float32)
    rpred = rng.standard_normal((24, rows, cols, a, 4)).astype(np.float32)
    cu, ip = y_cls[..., :a].astype(np.uint8), y_cls[..., a:].astype(np.uint8)
    tg = y_reg[..., 4 * a:].reshape(24, rows, cols, a, 4)
    loss, gcls, _ = ops.rpn_losses(dev(cu.reshape(24, -1)), dev(ip.reshape(24, -1)), dev(tg.reshape(24, -1, 4)),
                                   dev(pred.reshape(24, -1)), dev(rpred.reshape(24, -1, 4)), want_grad=True)
    loss, gcls = host(loss), host(gcls).reshape(24, rows, cols, a)
    for b in range(24):
        r, c = ext[b]
        wl = host(ops.rpn_losses(dev(cu[b:b + 1, :r, :c].reshape(1, -1)), dev(ip[b:b + 1, :r, :c].reshape(1, -1)),
                                 dev(tg[b:b + 1, :r, :c].reshape(1, -1, 4)), dev(pred[b:b + 1, :r, :c].reshape(1, -1)),
                                 dev(rpred[b:b + 1, :r, :c].reshape(1, -1, 4))))
        assert abs(loss[b, 0] - wl[0, 0]) <= 2e-6 * max(1.0, abs(wl[0, 0]))
        pad = np.ones((rows, cols), bool)
        pad[:r, :c] = False
        assert (gcls[b][pad] == 0).all()


def _roi_case(seed):
    """padded features (garbage in the padding) + RoIs that cross their image's extent"""
    rng = np.random.default_rng(seed)
    shapes = [(38, 50), (50, 38), (23, 61), (38, 57)]
    rows, cols = max(s[0] for s in shapes), max(s[1] for s in shapes)
    feat = np.empty((len(shapes), rows, cols, 64), np.float32)
    per_feat, rois = [], np.zeros((len(shapes), 96, 4), np.int32)
    for b, (r, c) in enumerate(shapes):
        feat[b] = GARBAGE[b % len(GARBAGE)]
        f = rng.standard_normal((r, c, 64)).astype(np.float32)
        feat[b, :r, :c] = f
        per_feat.append(f)
        x1, y1 = rng.integers(-3, c, 96), rng.integers(-3, r, 96)
        rois[b] = np.stack([x1, y1, x1 + rng.integers(1, 30, 96), y1 + rng.integers(1, 30, 96)], axis=1)
    return feat, per_feat, rois, np.array(shapes, np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["resize", "max"])
@pytest.mark.parametrize("roi_dtype", [np.int16, np.float32])
def test_ragged_roi_pool_equals_cropped_calls(ops, mode, roi_dtype):
    import torch
    from faster_rcnn_b200.custom_layers import roi_pool
    feat, per_feat, rois, ext = _roi_case(7)
    rois = rois.astype(roi_dtype) + (0.7 if roi_dtype == np.float32 else 0)
    x = dev(feat).requires_grad_(True)
    out = roi_pool(x, dev(rois), 7, mode, extents=dev(ext))
    w = torch.randn(out.shape, generator=torch.Generator(device="cuda").manual_seed(1), device="cuda")
    (out * w).sum().backward()
    got, grad = host(out.detach()), host(x.grad)
    for b, f in enumerate(per_feat):
        r, c = ext[b]
        xb = dev(f[None]).requires_grad_(True)
        ob = roi_pool(xb, dev(rois[b:b + 1]), 7, mode)
        (ob * w[b:b + 1]).sum().backward()
        assert np.array_equal(got[b], host(ob.detach())[0])
        np.testing.assert_allclose(grad[b, :r, :c], host(xb.grad)[0], rtol=1e-5, atol=1e-5)
        pad = np.ones(grad.shape[1:3], bool)
        pad[:r, :c] = False
        assert (grad[b][pad] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("compact", [False, True])
def test_ragged_roi_max_argmax_refers_to_the_padded_width(ops, compact):
    feat, per_feat, rois, ext = _roi_case(8)
    clipped = ops.clip_rois(dev(rois), dev(ext))
    out, am = (host(t) for t in ops.roi_forward(dev(feat), clipped, 7, "max", compact=compact))
    width = feat.shape[2]
    for b, f in enumerate(per_feat):
        r, c = ext[b]
        ob, ab = (host(t)[0] for t in ops.roi_forward(dev(f[None]), dev(rois[b:b + 1]), 7, "max", compact=compact))
        assert np.array_equal(out[b], ob)
        if compact:
            assert np.array_equal(am[b], ab)
        else:
            assert np.array_equal((am[b] // width) * c + am[b] % width, ab)


@pytest.mark.gpu
def test_clip_rois_truncates_like_the_roi_layer(ops):
    import torch
    rois = np.array([[[-2.9, -0.5, 70.9, 12.2], [3.7, 4.2, 5.1, 9.9]], [[1, 2, 3, 4], [0, 0, 99, 99]]], np.float32)
    ext = np.array([[10, 20], [0, 5]], np.int32)
    got = host(ops.clip_rois(dev(rois), dev(ext)))
    want = np.array([[[0, 0, 20, 10], [3, 4, 5, 9]], [[1, 2, 3, 0], [0, 0, 5, 0]]], np.float32)
    assert np.array_equal(got, want)
    for dt in (torch.int16, torch.int32):
        assert np.array_equal(host(ops.clip_rois(dev(rois).to(dt), dev(ext))), want.astype(np.int32))


def _pipeline_inputs(shapes, n_anchors=9, channels=32, seed=500):
    from faster_rcnn_b200 import synth
    cls, regr, feat = [], [], []
    for i, (r, c) in enumerate(shapes):
        pc, pr = synth.rpn_outputs(r, c, n_anchors, seed + i, clustered=bool(i % 2))
        cls.append(pc[0])
        regr.append(pr[0])
        feat.append(synth.feature_map(r, c, channels, seed + 50 + i)[0])
    return cls, regr, feat


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["resize", "max"])
def test_proposal_pipeline_on_a_list_of_sizes(ops, mode):
    from faster_rcnn_b200.pipeline import ProposalRoiPipeline
    dims = O.anchor_table([128, 256, 512])
    shapes = [(38, 50), (38, 57), (50, 38), (38, 56), (12, 20)]
    cls, regr, feat = _pipeline_inputs(shapes)
    pipe = ProposalRoiPipeline(anchor_dims=dims, mode=mode, h2d_chunk=2)
    rois, scores, count, pooled = pipe(cls, regr, feat)
    pooled = pooled if mode == "resize" else pooled[0]
    for b in range(len(shapes)):
        w = ProposalRoiPipeline(anchor_dims=dims, mode=mode).run_device(dev(cls[b][None]), dev(regr[b][None]),
                                                                         dev(feat[b][None]))
        assert np.array_equal(rois[b], host(w[0])[0]) and np.array_equal(scores[b], host(w[1])[0])
        assert count[b] == host(w[2])[0]
        wp = w[4] if mode == "resize" else w[4][0]
        assert np.array_equal(host(pooled[b]), host(wp)[0])


@pytest.mark.gpu
def test_graph_captured_with_extents_replays_other_extents(ops):
    from faster_rcnn_b200.pipeline import ProposalRoiPipeline
    dims = O.anchor_table([128, 256, 512])
    shapes_a = [(38, 50), (38, 57), (50, 38)]
    shapes_b = [(50, 57), (20, 11), (0, 0)]
    pipe = ProposalRoiPipeline(anchor_dims=dims)
    ca, ra, fa = (ops.pad_batch(x, pad_to=(50, 57)) for x in _pipeline_inputs(shapes_a))
    cb, rb, fb = (ops.pad_batch(x, pad_to=(50, 57)) for x in _pipeline_inputs([(50, 57), (20, 11), (1, 1)], seed=900))
    ext_b = dev(np.array(shapes_b, np.int32))
    g = pipe.capture(ca[0], ra[0], fa[0], ca[1])
    got = [host(t).copy() for t in g(cb[0], rb[0], fb[0], ext_b)]
    want = pipe.run_device(cb[0], rb[0], fb[0], extents=ext_b)
    for x, y in zip(got, want):
        assert np.array_equal(x, host(y))
    assert got[2][2] == 0
    got_a = [host(t).copy() for t in g(ca[0], ra[0], fa[0], ca[1])]
    for x, y in zip(got_a, pipe.run_device(ca[0], ra[0], fa[0], extents=ca[1])):
        assert np.array_equal(x, host(y))


@pytest.mark.gpu
def test_detection_pipeline_on_a_list_of_sizes(ops):
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.pipeline import DetectionPipeline
    dims = O.anchor_table([128, 256, 512])
    shapes = [(37, 62), (38, 50), (50, 38), (20, 33)]
    cls, regr, feat = _pipeline_inputs(shapes, channels=16)
    gen = torch.Generator(device="cuda").manual_seed(5)
    w_cls = torch.randn((16, 21), generator=gen, device="cuda")
    w_reg = torch.randn((16, 80), generator=gen, device="cuda")

    def head(pooled, rois):
        x = pooled.mean(dim=(2, 3)) + rois.to(torch.float32).sum(dim=2, keepdim=True) * 0.01
        return torch.softmax(x @ w_cls, dim=2), x @ w_reg

    ratios = [1.6, 1.0, 2.0, 1.2]
    pipe = DetectionPipeline(head, synth.VOC_CLASS_MAPPING, anchor_dims=dims)
    got = pipe.detect(cls, regr, feat, ratios)
    for b in range(len(shapes)):
        want = pipe.detect(cls[b][None], regr[b][None], feat[b][None], ratios[b:b + 1])[0]
        assert len(got[b]) == len(want) > 0
        for g, w in zip(got[b], want):
            assert np.array_equal(g['bbox'], w['bbox']) and g['cls_name'] == w['cls_name'] and g['prob'] == w['prob']


@pytest.mark.gpu
def test_det_training_pipeline_on_a_list_of_sizes(ops):
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.pipeline import DetTrainingPipeline
    dims = O.anchor_table([128, 256, 512])
    shapes = [(37, 62), (38, 50), (50, 38)]
    cls, regr, feat = _pipeline_inputs(shapes, channels=16)
    images = [FakeImage("t%d" % b, c * 16, r * 16, synth.gt_boxes(6, c * 16, r * 16, 70 + b)) for b, (r, c) in
              enumerate(shapes)]
    pipe = DetTrainingPipeline(synth.VOC_CLASS_MAPPING, anchor_dims=dims)
    np.random.seed(4)
    got = pipe(cls, regr, feat, images)
    np.random.seed(4)
    for b in range(len(shapes)):
        want = pipe(cls[b][None], regr[b][None], feat[b][None], images[b:b + 1])
        for x, y in zip(got[:4], want[:4]):
            assert np.array_equal(host(x[b]), host(y[0]))
        assert got[4][b] == want[4][0]


@pytest.mark.gpu
def test_pad_batch_copies_the_valid_regions(ops):
    import torch
    arrays = [np.arange(2 * 3 * 4, dtype=np.float32).reshape(2, 3, 4), np.ones((4, 1, 4), np.float32),
              np.zeros((0, 2, 4), np.float32)]
    padded, ext = ops.pad_batch(arrays, pad_to=(5, 3))
    assert padded.shape == (3, 5, 3, 4) and ext.dtype == torch.int32 and ext.is_cuda
    assert host(ext).tolist() == [[2, 3], [4, 1], [0, 2]]
    p = host(padded)
    assert np.array_equal(p[0, :2, :3], arrays[0]) and np.array_equal(p[1, :4, :1], arrays[1])
    assert p[0, 2:].sum() == 0 and p[1, :, 1:].sum() == 0 and p[2].sum() == 0
    t_padded, t_ext = ops.pad_batch([dev(a) for a in arrays])
    assert np.array_equal(host(t_padded), p[:, :4]) and np.array_equal(host(t_ext), host(ext))


# ---- argument checks (no GPU) ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("arrays,pad_to,match", [
    ([], None, "non-empty"),
    ([np.zeros((2, 3), np.float32)], None, "3 dimensions"),
    ([np.zeros((2, 3, 4), np.float32), np.zeros((2, 3, 5), np.float32)], None, "last dimension"),
    ([np.zeros((2, 3, 4), np.float32), np.zeros((2, 3, 4), np.float64)], None, "one dtype"),
    ([np.zeros((2, 3, 4), np.float32), np.zeros((5, 1, 4), np.float32)], (4, 3), "smaller"),
    ([np.zeros((0, 0, 4), np.float32)], None, "empty"),
])
def test_pad_batch_validates_its_arguments(arrays, pad_to, match):
    from faster_rcnn_b200 import ops
    with pytest.raises(ValueError, match=match):
        ops.pad_batch(arrays, pad_to)
