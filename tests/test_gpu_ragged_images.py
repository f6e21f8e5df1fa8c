"""Mixed-size batches at both ends of an RPN step: differently sized source images resized, mirrored and mean-subtracted
into one padded batch by one device call, and the RPN losses taken per image on padded targets.  Image by image, the
results must equal the single-image calls bit for bit, with zeros in all padding.  The argument checks of
ops.pack_images need no GPU."""
import os
import random

import numpy as np
import pytest

from helpers import dev, golden, host
from oracle import frcnn_oracle as O
from oracle import image_oracle as IO

GARBAGE = (np.nan, np.inf, -np.inf, 1e30)
MEAN4 = (103.939, 116.779, 123.68, 7.25)


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import _build, ops as ops_mod
    _build.build()
    return ops_mod


def _natural(h, w, cn, seed):
    """smooth structure + texture + noise, one white-noise channel"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 127 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 23.0) + 30 * np.sin((xx + yy) / 5.0)
    img = np.clip(base[:, :, None] + rng.normal(0, 12, (h, w, cn)), 0, 255).astype(np.uint8)
    img[..., -1] = rng.integers(0, 256, (h, w), dtype=np.uint8)
    return img


# (source (h, w), destination (h, w), flip)
MIX = [
    ((375, 500), (600, 800), True),      # VOC landscape enlargement
    ((500, 333), (901, 600), False),     # VOC portrait enlargement
    ((333, 500), (600, 901), True),
    ((120, 90), (120, 90), False),       # identity
    ((640, 480), (90, 70), True),        # 7x reduction: past the tile limit, per-pixel arithmetic
    ((1, 1), (5, 7), False),             # 1x1 source
    ((50, 60), (0, 40), True),           # zero destination extent: all padding
    ((37, 53), (111, 97), False),
]


def _mix_inputs(ops, mix, cn, seed=0):
    srcs = [_natural(s[0], s[1], cn, seed + i) for i, (s, _, _) in enumerate(mix)]
    packed, offsets, sizes = ops.pack_images(srcs)
    geom = np.array([(s[0], s[1], d[0], d[1]) for s, d, _ in mix], np.int32)
    flip = np.array([f for _, _, f in mix], np.uint8)
    assert np.array_equal(host(sizes), geom[:, :2])
    return srcs, packed, offsets, dev(geom), dev(flip)


def _check_against_oracle(srcs, mix, u8, f32, mean, height, width):
    for b, (src, (_, (h, w), flip)) in enumerate(zip(srcs, mix)):
        pad = np.ones((height, width), bool)
        pad[:h, :w] = False
        if h and w:
            want = IO.resize_cubic_u8(src, w, h, flip=flip)
            assert np.array_equal(u8[b, :h, :w], want), b
            assert np.array_equal(f32[b, :h, :w], IO.preprocess_bgr(want, mean).astype(np.float32)), b
        assert not u8[b][pad].any() and (f32[b][pad] == 0).all() and not np.signbit(f32[b][pad]).any(), b


@pytest.mark.gpu
@pytest.mark.parametrize("cn", [1, 2, 3, 4])
def test_ragged_resize_equals_oracle_image_by_image(ops, cn):
    """one batch of VOC enlargements, an identity, a 7x reduction, a 1x1 source and a zero extent, mirrored in part;
    2 channels run off the uniform entry's tile path"""
    import torch
    srcs, packed, offsets, geom, flip = _mix_inputs(ops, MIX, cn)
    height, width = max(d[0] for _, d, _ in MIX), max(d[1] for _, d, _ in MIX)
    mean = MEAN4[:cn]
    u8, f32 = ops.image_resize_cubic_ragged(packed, offsets, geom, height, width, flip=flip, mean=mean, channels=cn)
    assert u8.shape == (len(MIX), height, width, cn) and f32.shape == u8.shape
    _check_against_oracle(srcs, MIX, host(u8), host(f32), mean, height, width)
    # preallocated outputs full of garbage come back with zeros in all padding
    o8 = torch.full(tuple(u8.shape), 0xAB, dtype=torch.uint8, device="cuda")
    of = torch.full(tuple(u8.shape), float("nan"), dtype=torch.float32, device="cuda")
    g8, gf = ops.image_resize_cubic_ragged(packed, offsets, geom, height, width, flip=flip, mean=mean, out=(o8, of),
                                           channels=cn)
    assert g8.data_ptr() == o8.data_ptr() and gf.data_ptr() == of.data_ptr()
    assert np.array_equal(host(g8), host(u8)) and np.array_equal(host(gf), host(f32))
    only_f = ops.image_resize_cubic_ragged(packed, offsets, geom, height, width, flip=flip, mean=mean, want_u8=False,
                                           channels=cn)
    assert np.array_equal(host(only_f), host(f32))
    only_u8 = ops.image_resize_cubic_ragged(packed, offsets, geom, height, width, flip=flip, channels=cn)
    assert np.array_equal(host(only_u8), host(u8))


@pytest.mark.gpu
def test_ragged_resize_of_bad_sources_is_all_zero(ops):
    """a non-positive source size or bytes outside the buffer: the image is written as zeros and nothing is read;
    destination extents beyond the padded shape are clamped to it"""
    import torch
    srcs = [_natural(20, 30, 3, i) for i in range(4)]
    packed, offsets, _ = ops.pack_images(srcs)
    n = 20 * 30 * 3
    geom = np.array([(20, 30, 40, 50), (0, 30, 40, 50), (20, 30, 40, 50), (20, 30, 99, 99)], np.int32)
    offs = np.array([0, n, 3 * n + 1, 3 * n], np.int64)     # image 2 would end one byte past the buffer
    u8 = host(ops.image_resize_cubic_ragged(packed, dev(offs), dev(geom), 40, 50))
    assert np.array_equal(u8[0], IO.resize_cubic_u8(srcs[0], 50, 40))
    assert not u8[1].any() and not u8[2].any()
    assert np.array_equal(u8[3], IO.resize_cubic_u8(srcs[3], 50, 40))
    offs[0] = -1
    u8 = host(ops.image_resize_cubic_ragged(packed, dev(offs), dev(geom), 40, 50))
    assert not u8[0].any()
    assert packed.dtype == torch.uint8 and packed.numel() == 4 * n
    with pytest.raises(ValueError, match="out must be"):          # want_u8 without a u8 buffer
        ops.image_resize_cubic_ragged(packed, dev(offs), dev(geom), 40, 50, out=(None, torch.empty((4, 40, 50, 3),
                                                                                                   device="cuda")))


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst,flip", [((375, 500), (600, 800), True), ((480, 640), (160, 213), False),
                                          ((640, 480), (90, 70), True)])
def test_ragged_resize_with_full_extents_equals_the_uniform_entry(ops, src, dst, flip):
    import torch
    imgs = np.stack([_natural(src[0], src[1], 3, 40 + i) for i in range(3)])
    packed, offsets, sizes = ops.pack_images([dev(x) for x in imgs])
    geom = torch.cat([sizes, torch.tensor([dst] * 3, dtype=torch.int32, device="cuda")], dim=1).contiguous()
    flips = torch.full((3,), int(flip), dtype=torch.uint8, device="cuda")
    got = ops.image_resize_cubic_ragged(packed, offsets, geom, dst[0], dst[1], flip=flips, mean=MEAN4[:3])
    want = ops.image_resize_cubic(dev(imgs), dst[0], dst[1], flip=flip, mean=MEAN4[:3])
    for g, w in zip(got, want):
        assert np.array_equal(host(g), host(w))


@pytest.mark.gpu
def test_preprocessed_batch_device_equals_per_image_calls(ops, tmp_path):
    """shapes.Image objects from a VOC-layout directory, with their mirrored copies, at resize_within_bounds(600, 1000)"""
    pytest.importorskip("cv2")
    from test_oracle_image import _write_voc
    from faster_rcnn_b200 import args_util
    from faster_rcnn_b200.shapes import preprocessed_batch_device
    root = str(tmp_path)
    names = {"a1": (500, 375), "a2": (375, 500), "a3": (500, 333)}
    for name, (w, h) in names.items():
        _write_voc(root, name, w, h, [("cat", 0, 10, 20, 300, 200)])
    open(os.path.join(root, "ImageSets", "Main", "trainval.txt"), "w").write("\n".join(names) + "\n")
    images = [img.resize_within_bounds(600, 1000)[0] for img in args_util.base_paths_to_imgs(root, "trainval")]
    assert len(images) == 6 and sum(img.flipped for img in images) == 3
    padded, ext = preprocessed_batch_device(images, pad_to=(901, 905))
    assert padded.shape == (6, 901, 905, 3)
    ext = host(ext)
    got = host(padded)
    for b, img in enumerate(images):
        assert tuple(ext[b]) == (img.height, img.width)
        want = host(img.preprocessed_device())[0]
        assert np.array_equal(got[b, :img.height, :img.width], want), b
        assert not got[b, img.height:].any() and not got[b, :, img.width:].any()
    with pytest.raises(ValueError, match="smaller"):
        preprocessed_batch_device(images, pad_to=(600, 600))


@pytest.mark.gpu
def test_graph_replays_another_size_mix(ops):
    """one graph captured on a private handle (as pipeline.GraphedRun does) serves a second mix of sizes"""
    import torch
    from faster_rcnn_b200.runtime import Context, use_context
    mix_a = [((375, 500), (600, 800), False), ((500, 333), (600, 400), True), ((100, 100), (50, 60), False)]
    mix_b = [((333, 500), (450, 677), True), ((10, 12), (600, 800), False), ((200, 300), (0, 0), False)]
    height, width = 600, 800
    _, pa, oa, ga, fa = _mix_inputs(ops, mix_a, 3, seed=1)
    srcs_b, pb, ob, gb, fb = _mix_inputs(ops, mix_b, 3, seed=2)
    src = torch.zeros((max(pa.numel(), pb.numel()),), dtype=torch.uint8, device="cuda")
    src[:pa.numel()].copy_(pa)
    inputs = (src, oa.clone(), ga.clone(), fa.clone())
    ctx = Context(torch.cuda.current_device())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with use_context(ctx), torch.cuda.stream(side):
        for _ in range(2):
            ops.image_resize_cubic_ragged(*inputs[:3], height, width, flip=inputs[3], mean=MEAN4[:3])
        side.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            outs = ops.image_resize_cubic_ragged(*inputs[:3], height, width, flip=inputs[3], mean=MEAN4[:3])
    torch.cuda.current_stream().wait_stream(side)
    inputs[0][:pb.numel()].copy_(pb)
    for dst, s in zip(inputs[1:], (ob, gb, fb)):
        dst.copy_(s)
    graph.replay()
    got = [host(t).copy() for t in outs]
    want = ops.image_resize_cubic_ragged(pb, ob, gb, height, width, flip=fb, mean=MEAN4[:3])
    for g, w in zip(got, want):
        assert np.array_equal(g, host(w))
    _check_against_oracle(srcs_b, mix_b, got[0], got[1], MEAN4[:3], height, width)


def _voc_targets(n_images, zero_image):
    """RPN targets of `n_images` VOC GT sets from rpn_y_true_ragged, one extent set to zero"""
    from faster_rcnn_b200 import rpn_util
    from helpers import FakeImage
    g = golden("voc_gt_200")
    gts = [g["gt"][g["offsets"][i]:g["offsets"][i + 1]] for i in range(n_images)]
    images = [FakeImage(str(g["names"][i]), int(g["img_wh"][i][0]), int(g["img_wh"][i][1]),
                        [("chair", *row) for row in gts[i].tolist()]) for i in range(n_images)]
    dims = O.anchor_table([128, 256, 512])
    mgr = rpn_util.RpnTrainingManager(lambda h, w: O.conv_dims_resnet(h, w), 16, preprocess_func=None, anchor_dims=dims)
    shapes = np.array([O.conv_dims_resnet(int(h), int(w)) for w, h in g["img_wh"][:n_images]])
    rows, cols = (int(v) + 2 for v in shapes.max(axis=0))
    random.seed(5)
    y_cls, y_reg, ext = mgr.rpn_y_true_ragged(images, pad_to=(rows, cols))
    ext = np.array(ext, np.int32)
    assert len({tuple(e) for e in ext}) > 1
    ext[zero_image] = (0, ext[zero_image][1])
    return y_cls, y_reg, ext, len(dims), rows, cols


@pytest.mark.gpu
def test_rpn_losses_with_extents_equal_cropped_calls(ops):
    """loss, class and box gradients per image equal the uniform call on the crop bit for bit; NaN / inf / 1e30 in the
    padding of predictions and targets reach no output; a zero extent gives zero loss and gradients"""
    import torch
    from faster_rcnn_b200 import loss_functions
    n_img, zero = 24, 5
    y_cls, y_reg, ext, a, rows, cols = _voc_targets(n_img, zero)
    rng = np.random.default_rng(3)
    pred = rng.uniform(0.02, 0.98, (n_img, rows, cols, a)).astype(np.float32)
    pred[:, :2, :3] = 0.0                                            # clipped: no class gradient
    rpred = rng.standard_normal((n_img, rows, cols, a, 4)).astype(np.float32) * 2
    cu, ip = y_cls[..., :a].astype(np.uint8), y_cls[..., a:].astype(np.uint8)
    tg = y_reg[..., 4 * a:].reshape(n_img, rows, cols, a, 4).copy()
    for b in range(n_img):
        r, c = ext[b]
        pad = np.ones((rows, cols), bool)
        pad[:r, :c] = False
        v = GARBAGE[b % len(GARBAGE)]
        pred[b][pad], rpred[b][pad], tg[b][pad] = v, v, v
        cu[b][pad], ip[b][pad] = 1, 1
    args = [dev(cu.reshape(n_img, -1)), dev(ip.reshape(n_img, -1)), dev(tg.reshape(n_img, -1, 4)),
            dev(pred.reshape(n_img, -1)), dev(rpred.reshape(n_img, -1, 4))]
    loss, gcls, greg = ops.rpn_losses(*args, want_grad=True, extents=dev(ext), padded_shape=(rows, cols))
    only_loss = ops.rpn_losses(*args, extents=dev(ext), padded_shape=(rows, cols))
    assert np.array_equal(host(only_loss), host(loss))
    loss, gcls, greg = host(loss), host(gcls).reshape(n_img, rows, cols, a), host(greg).reshape(n_img, rows, cols, a, 4)
    box_losses = 0
    for b in range(n_img):
        r, c = ext[b]
        pad = np.ones((rows, cols), bool)
        pad[:r, :c] = False
        assert (gcls[b][pad] == 0).all() and (greg[b][pad] == 0).all() and not np.signbit(greg[b][pad]).any()
        if r == 0 or c == 0:
            assert b == zero and (loss[b] == 0).all() and (gcls[b] == 0).all() and (greg[b] == 0).all()
            continue
        crop = [dev(x[b:b + 1, :r, :c].reshape(1, -1)) for x in (cu, ip, pred)]
        wl, wc, wr = (host(t) for t in ops.rpn_losses(crop[0], crop[1], dev(tg[b:b + 1, :r, :c].reshape(1, -1, 4)), crop[2],
                                                      dev(rpred[b:b + 1, :r, :c].reshape(1, -1, 4)), want_grad=True))
        assert np.array_equal(loss[b], wl[0]), b
        box_losses += int(wl[0, 1] != 0)
        assert np.array_equal(gcls[b, :r, :c].reshape(-1), wc[0]) and np.array_equal(greg[b, :r, :c].reshape(-1, 4), wr[0]), b
    assert box_losses >= n_img // 2                                  # the box loss depends on the image's own map size
    # the autograd form
    cp = args[3].clone().requires_grad_(True)
    rp = args[4].clone().requires_grad_(True)
    lt = loss_functions.rpn_losses(cp, rp, args[0], args[1], args[2], extents=dev(ext), padded_shape=(rows, cols))
    w = torch.tensor(np.random.default_rng(4).uniform(0.5, 2.0, (n_img, 2)), dtype=torch.float32, device="cuda")
    (lt * w).sum().backward()
    assert np.array_equal(host(lt.detach()), loss)
    wh = host(w)
    assert np.array_equal(host(cp.grad), (gcls.reshape(n_img, -1) * wh[:, 0:1]))
    assert np.array_equal(host(rp.grad), (greg.reshape(n_img, -1, 4) * wh[:, 1].reshape(-1, 1, 1)))


@pytest.mark.gpu
def test_rpn_losses_with_full_extents_equal_the_uniform_entry(ops):
    rng = np.random.default_rng(8)
    b, rows, cols, a = 3, 17, 23, 9
    n = rows * cols * a
    cu, ip = rng.integers(0, 2, (b, n), dtype=np.uint8), rng.integers(0, 2, (b, n), dtype=np.uint8)
    args = [dev(cu), dev(ip), dev(rng.standard_normal((b, n, 4)).astype(np.float32)),
            dev(rng.uniform(0, 1, (b, n)).astype(np.float32)), dev(rng.standard_normal((b, n, 4)).astype(np.float32))]
    ext = dev(np.array([[rows, cols]] * b, np.int32))
    for got, want in zip(ops.rpn_losses(*args, want_grad=True, extents=ext, padded_shape=(rows, cols)),
                         ops.rpn_losses(*args, want_grad=True)):
        assert np.array_equal(host(got), host(want))
    with pytest.raises(ValueError, match="together"):
        ops.rpn_losses(*args, extents=ext)
    with pytest.raises(ValueError, match="rows \\* cols \\* A"):
        ops.rpn_losses(*args, extents=ext, padded_shape=(rows, cols + 1))


# ---- argument checks (no GPU) ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("sources,exc,match", [
    ([], ValueError, "non-empty"),
    ([np.zeros((2, 3, 3), np.uint8), np.zeros((2, 3, 4), np.uint8)], ValueError, "channel count"),
    ([np.zeros((2, 3, 3), np.uint8), np.zeros((2, 3, 3), np.float32)], TypeError, "uint8"),
    ([np.zeros((2, 3), np.uint8)], ValueError, "3 dimensions"),
    ([[[[1, 2, 3]]]], TypeError, "numpy arrays or torch tensors"),
])
def test_pack_images_validates_its_arguments(sources, exc, match):
    from faster_rcnn_b200 import ops
    with pytest.raises(exc, match=match):
        ops.pack_images(sources)
