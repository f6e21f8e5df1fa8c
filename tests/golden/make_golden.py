"""Generates tests/golden/*.npz by running the UNMODIFIED reference (a checkout of
Kelicious/faster_rcnn, see oracle/ref_loader.py) on seeded synthetic inputs and on the
one VOC image it ships:

    python tests/golden/make_golden.py     # reference checked out at oracle/_ref/, or
    FRCNN_REFERENCE_DIR=<checkout>/faster_rcnn python tests/golden/make_golden.py

Every fixture stores the inputs next to the reference's outputs, so the tests do not depend on
regenerating the inputs bit-for-bit.  Sizes are kept small (a few hundred KB compressed in total).
voc_dets.py cannot be imported (Keras), so its post-processing loop (voc_dets.py:51-86) is replayed
here around the reference's own `nms` / `transform`, as in tests/test_oracle_vs_reference.py.
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from faster_rcnn_b200 import synth          # noqa: E402
from oracle import ref_loader               # noqa: E402
from oracle import frcnn_oracle as O        # noqa: E402  (only conv_dims helpers: resnet.py needs Keras)


def ref_image(ref, name, w, h, gts):
    S = ref.shapes
    boxes = [S.GroundTruthBox(c, False, S.Box(x1, y1, x2, y2)) for c, x1, y1, x2, y2 in gts]
    return S.Image(S.Metadata(name, w, h, boxes, '/nonexistent.jpg'))


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("%-28s %7d bytes" % (name + ".npz", os.path.getsize(path)))


def proposals_case(ref, tag, rows, cols, scales, seed, k, max_boxes, clustered):
    dims = ref.util.get_anchors(scales) if scales else ref.shared_constants.DEFAULT_ANCHORS
    cls, regr = synth.rpn_outputs(rows, cols, len(dims), seed, clustered=clustered)
    with ref_loader.quiet():
        dense = ref.det_util._get_rois(regr.copy(), dims, 16)
        valid = ref.det_util._get_valid_box_idxs(dense)
    probs = cls.reshape(-1)
    order = probs[valid].argsort()[::-1][:k]              # det_util.py:151-153 (tie-free scores)
    tb, tp = dense[valid][order].astype('int16'), probs[valid][order]
    with ref_loader.quiet():
        nb, npb = ref.det_util.nms(tb, tp, max_boxes=max_boxes, overlap_thresh=0.7)
    save("proposals_" + tag, anchor_dims=dims, cls=cls, regr=regr, k=k, max_boxes=max_boxes, dense=dense,
         valid=valid, topk_boxes=tb, topk_probs=tp, topk_index=valid[order], nms_boxes=nb, nms_probs=npb)


def labels_case(ref, tag, img, dims, conv_dims):
    mgr = ref.rpn_util.RpnTrainingManager(conv_dims, 16, preprocess_func=None, anchor_dims=dims)
    with ref_loader.quiet():
        mgr._process(img)
    c = mgr._cache[img.cache_key]
    can_use, is_pos, bbreg = c['can_use'].copy(), c['is_pos'].copy(), c['bbreg_targets'].copy()
    random.seed(1)
    with ref_loader.quiet():
        y_class, y_bbreg = mgr.rpn_y_true(img)
    gt = ref.util.get_bbox_coords(img.gt_boxes)
    save("rpn_labels_" + tag, anchor_dims=dims, gt=gt, img_wh=np.array([img.width, img.height]),
         conv=np.array(conv_dims(img.height, img.width)), can_use=can_use, is_pos=is_pos, bbreg=bbreg,
         y_class=y_class, y_bbreg=y_bbreg, py_random_seed=1)


def voc_gt_case(ref, n_images=200):
    """Real ground truth: the first `n_images` VOC2007 trainval annotations the reference ships
    (test_data/VOC_test, XML only), resized like training (600/1000), with a digest of the reference's labels."""
    import hashlib
    root = ref_loader.VOC_DIR
    names = [l.strip() for l in open(root + '/ImageSets/Main/trainval.txt')][:n_images]
    dims = ref.util.get_anchors([128, 256, 512])
    rows, offs, whs, digests, npos, nuse = [], [0], [], [], [], []
    for nm in names:
        img = ref.voc.extract_img_data(root, nm).resize_within_bounds(600, 1000)[0]
        rows.append(ref.util.get_bbox_coords(img.gt_boxes))
        offs.append(offs[-1] + len(rows[-1]))
        whs.append([img.width, img.height])
        mgr = ref.rpn_util.RpnTrainingManager(O.conv_dims_resnet, 16, preprocess_func=None, anchor_dims=dims)
        with ref_loader.quiet():
            mgr._process(img)
        c = mgr._cache[img.cache_key]
        digests.append(hashlib.sha1(c['can_use'].tobytes() + c['is_pos'].tobytes()).hexdigest()[:16])
        npos.append(int(c['is_pos'].sum()))
        nuse.append(int(c['can_use'].sum()))
    save("voc_gt_200", gt=np.concatenate(rows).astype(np.float32), offsets=np.array(offs), img_wh=np.array(whs),
         names=np.array(names), label_sha1=np.array(digests), n_pos=np.array(npos), n_use=np.array(nuse))


def voc_eval_case(n_images=400):
    """eval_dets.voc_eval (unmodified reference) on its own VOC_test annotations and synthetic detection files:
    jittered copies of the ground truth (0-2 per object) plus random false positives, unique confidences."""
    import contextlib
    import io
    import tempfile
    sys.path.insert(0, ref_loader.REF_DIR)
    import eval_dets as ref_eval
    from data.voc_data_helpers import extract_img_data
    root = ref_loader.VOC_DIR
    names = [l.strip() for l in open(root + '/ImageSets/Main/trainval.txt')][:n_images]
    rng = np.random.default_rng(7)
    out = {'names': np.array(names)}
    with tempfile.TemporaryDirectory() as tmp:
        iset = os.path.join(tmp, 'set.txt')
        open(iset, 'w').write('\n'.join(names) + '\n')
        for cls in ('person', 'chair', 'car'):
            lines, gt = [], {}
            for nm in names:
                objs = [b for b in extract_img_data(root, nm).gt_boxes if b.obj_cls == cls]
                gt[nm] = (np.array([b.corners for b in objs]).reshape(-1, 4), np.array([b.difficult for b in objs], dtype=bool))
                for b in objs:
                    for _ in range(rng.integers(0, 3)):
                        lines.append((nm, np.asarray(b.corners, float) + rng.normal(0, 6, 4)))
                for _ in range(rng.integers(0, 3)):
                    x1, y1 = rng.uniform(0, 300, 2)
                    w, h = rng.uniform(10, 200, 2)
                    lines.append((nm, np.array([x1, y1, x1 + w, y1 + h])))
            conf = rng.permutation(len(lines)) / len(lines) + 1e-3
            order = rng.permutation(len(lines))
            det_file = os.path.join(tmp, 'comp3_det_test_%s.txt' % cls)
            with open(det_file, 'w') as f:
                for i in order:
                    f.write("%s %r %r %r %r %r\n" % (lines[i][0], float(conf[i]), *[float(round(v, 1)) for v in lines[i][1]]))
            with contextlib.redirect_stdout(io.StringIO()):
                rec, prec, ap = ref_eval.voc_eval(root, det_file, iset, cls, ovthresh=0.5)
            gnames = [n for n in names if len(gt[n][0])]
            out.update({cls + '_ids': np.array([lines[i][0] for i in order]), cls + '_conf': np.array([conf[i] for i in order]),
                        cls + '_boxes': np.array([np.round(lines[i][1], 1) for i in order]), cls + '_rec': rec,
                        cls + '_prec': prec, cls + '_ap': ap, cls + '_gt_names': np.array(gnames),
                        cls + '_gt_boxes': np.concatenate([gt[n][0] for n in gnames]).astype(np.float64),
                        cls + '_gt_difficult': np.concatenate([gt[n][1] for n in gnames]),
                        cls + '_gt_counts': np.array([len(gt[n][0]) for n in gnames])})
    save("voc_eval", **out)


def main():
    ref = ref_loader.load()
    voc_gt_case(ref)
    voc_eval_case()
    # P1: anchor tables
    save("anchors", voc=ref.util.get_anchors([128, 256, 512]), default=ref.shared_constants.DEFAULT_ANCHORS,
         scales_voc=np.array([128, 256, 512]))

    # P2-P8: proposal stage, small maps (full sizes are covered by the live oracle in the GPU tests)
    proposals_case(ref, "voc_small", 13, 17, [128, 256, 512], 101, 600, 100, False)
    proposals_case(ref, "voc_clustered", 19, 25, [128, 256, 512], 102, 2000, 300, True)
    proposals_case(ref, "kitti_small", 10, 24, None, 103, 3000, 500, True)

    # T1-T7: RPN labels.  (a) the one real VOC image, (b) synthetic 50 GT
    img = ref.voc.extract_img_data(ref_loader.VOC_DIR, '000005').resize_within_bounds(600, 1000)[0]
    dims = ref.util.get_anchors([128, 256, 512])
    labels_case(ref, "000005_resnet", img, dims, O.conv_dims_resnet)
    labels_case(ref, "000005_vgg", img, dims, O.conv_dims_vgg)
    gts = synth.gt_boxes(50, 1000, 600, 7)
    labels_case(ref, "synth50", ref_image(ref, 'synth50', 1000, 600, gts), dims, O.conv_dims_resnet)

    # D1-D4: detector labels + sampling
    rois = synth.random_rois(600, 38, 63, 5)
    mapping = synth.VOC_CLASS_MAPPING
    with ref_loader.quiet():
        e_rois, y_cls, y_tr = ref.det_util._rois_to_truth(rois, ref_image(ref, 'det', 1000, 600, gts), mapping, stride=16)
    np.random.seed(1337)
    with ref_loader.quiet():
        sampled = ref.det_util._get_det_samples(y_cls[:, -1] == 0, 64)
    save("det_labels", rois=rois, gt_pixels=np.array([g[1:] for g in gts], dtype=np.int64),
         gt_cls=np.array([mapping[g[0]] for g in gts]), eligible_rois=e_rois, y_class_num=y_cls, y_transform=y_tr,
         sampled=np.array(sampled), np_random_seed=1337)

    # V1-V3: detector post-processing (loop of voc_dets.py:51-86 replayed around ref nms/transform)
    rev = {v: k for k, v in mapping.items()}
    prois = synth.random_rois(320, 37, 62, 3)
    out_cls, out_reg = synth.detector_outputs(320, 21, 3)
    ratio, stride = 1.6, 16
    bb, pp = {}, {}
    for r in range(320):
        c = np.argmax(out_cls[r])
        if c == mapping['bg']:
            continue
        x1, y1, x2, y2 = prois[r]
        t = out_reg[r, c * 4:(c + 1) * 4] / ref.shared_constants.BBREG_MULTIPLIERS
        px = ref.util.transform([x1, y1, x2, y2], t)
        bb.setdefault(rev[c], []).append([stride * v for v in px])
        pp.setdefault(rev[c], []).append(out_cls[r, c])
    d_cls, d_box, d_prob = [], [], []
    for name in bb:
        with ref_loader.quiet():
            nb, npb = ref.det_util.nms(np.array(bb[name]), np.array(pp[name]), overlap_thresh=0.5, max_boxes=2000)
        for i in range(nb.shape[0]):
            d_cls.append(mapping[name])
            d_box.append([int(round(v / ratio)) for v in nb[i]])
            d_prob.append(npb[i])
    save("det_postprocess", rois=prois, out_cls=out_cls, out_reg=out_reg, resize_ratio=ratio, stride=stride,
         det_cls=np.array(d_cls), det_boxes=np.array(d_box), det_probs=np.array(d_prob, dtype=np.float32))

    # P8 float64 variant + cross_ious
    rng = np.random.default_rng(5)
    xy, wh = rng.uniform(0, 500, (400, 2)), rng.uniform(5, 200, (400, 2))
    fboxes = np.concatenate([xy, xy + wh], axis=1)
    fprobs = rng.permutation(400).astype(np.float32) / 400
    with ref_loader.quiet():
        nb, npb = ref.det_util.nms(fboxes, fprobs, overlap_thresh=0.5, max_boxes=2000)
        anc = ref.rpn_util._get_all_anchor_coords(6, 9, dims, 16)
        gt32 = np.array([g[1:] for g in gts[:7]], dtype=np.float32)
        iou_f = ref.util.cross_ious(anc, gt32)
        iou_i = ref.util.cross_ious(rois[:100], gt32 / 16)
    save("nms_f64_iou", boxes=fboxes, probs=fprobs, nms_boxes=nb, nms_probs=npb, anchors=anc, gt=gt32, iou_f32=iou_f,
         rois_i16=rois[:100], gt_feat=gt32 / 16, iou_i16=iou_i)


if __name__ == "__main__":
    main()
