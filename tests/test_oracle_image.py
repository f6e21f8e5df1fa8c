"""Pins oracle/image_oracle.py (SURVEY 8f-4) against the installed OpenCV and the data helpers against the reference.
CPU only."""
import os

import numpy as np
import pytest

from oracle import image_oracle as IO
from oracle import ref_loader

cv2 = pytest.importorskip("cv2")
REF_VOC = ref_loader.VOC_DIR


def _natural(h, w, seed):
    """smooth structure + texture + noise, closer to a photograph than white noise"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 127 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 23.0) + 30 * np.sin((xx + yy) / 5.0)
    img = base[:, :, None] + rng.normal(0, 12, (h, w, 3)) + np.array([10, -20, 5])
    return np.clip(img, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("src,dst", [((375, 500), (600, 800)), ((333, 500), (600, 901)), ((480, 640), (300, 400)),
                                     ((37, 53), (111, 97)), ((600, 800), (600, 800)), ((5, 4), (9, 13))])
def test_resize_oracle_is_opencv_generic_bicubic(src, dst):
    """cv2 with its SIMD dispatch switched off runs the generic fixed-point path the oracle restates: equal on all but
    <= 2e-4 of the pixels, never by more than one grey level.  The default (SIMD) path of the same binary is allowed one
    grey level on <= 8 % of the pixels -- it differs from its own generic path by exactly that."""
    for seed, make in ((0, _natural), (1, lambda h, w, s: np.random.default_rng(s).integers(0, 256, (h, w, 3), dtype=np.uint8))):
        img = make(src[0], src[1], seed)
        got = IO.resize_cubic_u8(img, dst[1], dst[0]).astype(int)
        try:
            cv2.setUseOptimized(False)
            generic = cv2.resize(img, (dst[1], dst[0]), interpolation=cv2.INTER_CUBIC).astype(int)
        finally:
            cv2.setUseOptimized(True)
        default = cv2.resize(img, (dst[1], dst[0]), interpolation=cv2.INTER_CUBIC).astype(int)
        assert np.abs(got - generic).max() <= 1 and np.mean(got != generic) <= 2e-4 + 2.0 / got.size
        assert np.abs(got - default).max() <= 1 and np.mean(got != default) <= 0.08
        assert np.abs(default - generic).max() <= 1                      # cv2 against itself: the same +-1
    assert np.array_equal(IO.resize_cubic_u8(img, dst[1], dst[0], flip=True), IO.resize_cubic_u8(img, dst[1], dst[0])[:, ::-1])


def test_preprocess_and_gt_transform_formulas():
    img = _natural(6, 7, 3)
    pre = IO.preprocess_bgr(img)
    assert pre.dtype == np.float64 and np.array_equal(pre[..., 1], img[..., 1].astype(np.float64) - 116.779)
    from faster_rcnn_b200.shapes import Box, GroundTruthBox, Image
    gts = [GroundTruthBox('cat', False, Box(3, 5, 40, 60)), GroundTruthBox('dog', True, Box(0, 0, 499, 374))]
    im = Image('x', 500, 375, gts)
    big, ratio = im.resize_within_bounds(600, 1000)
    want = IO.transform_gt([g.corners for g in gts], ratio)
    assert (big.width, big.height) == (800, 600) and np.array_equal(np.array([g.corners for g in big.gt_boxes]), want)
    flipped = big.horizontal_flip()
    want_f = IO.transform_gt([g.corners for g in gts], ratio, flip_width=big.width)
    assert flipped.flipped and flipped.cache_key == 'xTrue'
    assert np.array_equal(np.array([g.corners for g in flipped.gt_boxes]), want_f)


def _write_voc(root, name, w, h, objects, with_pixels=True):
    for d in ("Annotations", "JPEGImages", os.path.join("ImageSets", "Main")):
        os.makedirs(os.path.join(root, d), exist_ok=True)
    objs = "".join("<object><name>%s</name><difficult>%d</difficult><bndbox><xmin>%s</xmin><ymin>%s</ymin><xmax>%s</xmax>"
                   "<ymax>%s</ymax></bndbox></object>" % o for o in objects)
    open(os.path.join(root, "Annotations", name + ".xml"), "w").write(
        "<annotation><filename>%s.png</filename><size><width>%d</width><height>%d</height><depth>3</depth></size>%s"
        "</annotation>" % (name, w, h, objs))
    if with_pixels:
        cv2.imwrite(os.path.join(root, "JPEGImages", name + ".png"), _natural(h, w, 9))


def test_voc_loader_conventions(tmp_path):
    from faster_rcnn_b200 import args_util
    from faster_rcnn_b200.data import voc_data_helpers as V
    root = str(tmp_path)
    _write_voc(root, "a1", 60, 40, [("cat", 0, "3", "5", "41.0", "30"), ("person", 1, 1, 1, 60, 40)])
    _write_voc(root, "a2", 50, 50, [])
    open(os.path.join(root, "ImageSets", "Main", "trainval.txt"), "w").write("a1\na2\n")
    assert V.get_img_names_from_set(root, "trainval") == ["a1", "a2"]
    img = V.extract_img_data(root, "a1")
    assert (img.name, img.width, img.height, img.flipped, img.cache_key) == ("a1", 60, 40, False, "a1False")
    assert [g.corners.tolist() for g in img.gt_boxes] == [[2, 4, 40, 29], [0, 0, 59, 39]]      # 1-based -> 0-based
    assert [g.difficult for g in img.gt_boxes] == [False, True] and img.gt_boxes[0].obj_cls == "cat"
    assert V.VOC_CLASS_MAPPING["bg"] == 20 and V.KITTI_CLASS_MAPPING["bg"] == 9
    imgs = args_util.base_paths_to_imgs(root + "," + root, "trainval")
    assert len(imgs) == 8 and [i.flipped for i in imgs] == [False] * 4 + [True] * 4
    assert imgs[4].gt_boxes[0].corners.tolist() == [60 - 40, 4, 60 - 2, 29]
    # pixels: lazily read, resized and mirrored like shapes.py:19-29
    big, _ = imgs[4].resize_within_bounds(80, 200)
    raw = cv2.imread(os.path.join(root, "JPEGImages", "a1.png"))
    want = cv2.flip(cv2.resize(raw, (big.width, big.height), interpolation=cv2.INTER_CUBIC), 1)
    assert np.array_equal(big.data, want)


@pytest.mark.skipif(not (ref_loader.available() and os.path.isdir(REF_VOC)), reason="reference checkout not present")
def test_voc_loader_equals_the_reference_on_its_own_test_data():
    from faster_rcnn_b200.data import voc_data_helpers as V
    ref = ref_loader.load()
    from data import voc_data_helpers as RV                         # the reference's module (ref_loader set sys.path)
    names = RV.get_img_names_from_set(REF_VOC, "trainval")
    assert V.get_img_names_from_set(REF_VOC, "trainval") == names
    have = [n for n in names if os.path.exists(os.path.join(REF_VOC, "Annotations", n + ".xml"))][:40]
    assert have
    for n in have:
        a, b = V.extract_img_data(REF_VOC, n), RV.extract_img_data(REF_VOC, n)
        assert (a.name, a.width, a.height, a.cache_key, a.image_path) == (b.name, b.width, b.height, b.cache_key, b._image_path)
        assert [(g.obj_cls, g.difficult, g.corners.tolist()) for g in a.gt_boxes] == \
               [(g.obj_cls, g.difficult, g.corners.tolist()) for g in b.gt_boxes]
        ar, ra = a.resize_within_bounds(600, 1000)
        br, rb = b.resize_within_bounds(600, 1000)
        af, bf = ar.horizontal_flip(), br.horizontal_flip()
        assert ra == rb and (af.width, af.height, af.cache_key) == (bf.width, bf.height, bf.cache_key)
        assert [g.corners.tolist() for g in af.gt_boxes] == [g.corners.tolist() for g in bf.gt_boxes]
        if os.path.exists(a.image_path):
            assert np.array_equal(af.data, bf.data)                   # same cv2 calls -> same pixels
    assert ref is not None
