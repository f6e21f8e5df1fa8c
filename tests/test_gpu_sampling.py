"""GPU: the device-side mini-batch draws (csrc/sample.cu) against oracle/sample_oracle.py bit for bit, their batching
and state semantics, the training pipelines built on them, and CUDA-graph capture without host synchronisation."""
import numpy as np
import pytest

from helpers import FakeImage, dev, host
from oracle import frcnn_oracle as O
from oracle import roi_oracle as R
from oracle import sample_oracle as S

pytestmark = pytest.mark.gpu

DIMS = O.anchor_table([128, 256, 512])
S_P = [0, 1, 15, 16, 17, 200]                                    # |P| and |Q| covering every branch of the detector rule
S_Q = [0, 1, 47, 48, 49, 1900]


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import ops as _ops
    return _ops


def _state(ops, seed, offset=0):
    s = ops.sampler_state(seed)
    s[1] = offset
    return s


def _counts(cu, ip):
    cu, ip = cu.astype(bool), ip.astype(bool)
    return np.stack([(cu & ip).sum(axis=1), (cu & ~ip).sum(axis=1)], axis=1).astype(np.int32)


def _c4_labels(ops, b, rows=38, cols=63):
    """128 images labelled from 50 GT boxes each, with special cases laid over the first four."""
    from faster_rcnn_b200 import synth
    gts = [np.array([g[1:] for g in synth.gt_boxes(50, 1000, 600, 300 + i)], np.float32) for i in range(b)]
    out = ops.label_anchors(dev(np.stack(gts)), dev(np.full(b, 50, np.int32)), dev(np.tile([1000, 600], (b, 1)), np.int32),
                            rows, cols, DIMS, 16)
    cu, ip = host(out[0]), host(out[1])
    rng = np.random.default_rng(1)
    n = cu.shape[1]
    ip[0] = 0                                                     # no positive
    ip[1] = 0
    ip[1, rng.choice(np.where(cu[1])[0], 128, replace=False)] = 1   # exactly 128 usable positives
    cu[2] = 0
    cu[2, rng.choice(n, 200, replace=False)] = 1                  # |P| + |Q| <= 256
    cu[3] = 0                                                     # nothing usable
    ip[4, rng.choice(np.where(cu[4])[0], 300, replace=False)] = 1   # more than 128 usable positives
    return cu, ip


@pytest.mark.parametrize("offset", [0, (1 << 32) - 50])
def test_sample_rpn_vs_oracle_c4_batch(ops, offset):
    b, seed = 128, 0xC0FFEE
    cu, ip = _c4_labels(ops, b)
    counts = _counts(cu, ip)
    assert counts[1, 0] == 128 and counts[2].sum() <= 256 and counts[3].sum() == 0 and counts[0, 0] == 0
    assert counts[4, 0] > 128
    state = _state(ops, seed, offset)
    got = ops.sample_rpn_(dev(cu), dev(ip), dev(counts), state)
    assert int(state[1]) == offset + b
    got = host(got)
    for i in range(b):
        want = S.rpn_keep(cu[i], ip[i], seed, offset + i)
        assert np.array_equal(got[i].astype(bool), want), i


def test_sample_rpn_kitti_anchors(ops):
    """64,296 anchors per image (38 x 94 x 18)."""
    rng = np.random.default_rng(2)
    b, n = 3, 38 * 94 * 18
    cu = (rng.random((b, n)) < 0.7).astype(np.uint8)
    ip = (rng.random((b, n)) < 0.01).astype(np.uint8)
    got = host(ops.sample_rpn_(dev(cu), dev(ip), dev(_counts(cu, ip)), _state(ops, 12)))
    for i in range(b):
        assert np.array_equal(got[i].astype(bool), S.rpn_keep(cu[i], ip[i], 12, i))


def test_sample_rpn_ragged_equals_cropped_uniform(ops):
    rng = np.random.default_rng(3)
    a, rows, cols = 9, 40, 60
    ext = np.array([[40, 60], [23, 37], [31, 60], [0, 0], [40, 11]], np.int32)
    b = len(ext)
    cu = np.zeros((b, rows, cols, a), np.uint8)
    ip = np.zeros((b, rows, cols, a), np.uint8)
    for i, (r, c) in enumerate(ext):
        cu[i, :r, :c] = rng.random((r, c, a)) < 0.6
        ip[i, :r, :c] = rng.random((r, c, a)) < 0.03
    flat_cu, flat_ip = cu.reshape(b, -1), ip.reshape(b, -1)
    state = _state(ops, 99, 1000)
    got = host(ops.sample_rpn_(dev(flat_cu), dev(flat_ip), dev(_counts(flat_cu, flat_ip)), state, extents=dev(ext),
                               padded_shape=(rows, cols), n_anchors=a)).reshape(b, rows, cols, a)
    assert int(state[1]) == 1000 + b
    for i, (r, c) in enumerate(ext):
        crop_cu = np.ascontiguousarray(cu[i, :r, :c]).reshape(1, -1)
        crop_ip = np.ascontiguousarray(ip[i, :r, :c]).reshape(1, -1)
        if crop_cu.size:
            want = host(ops.sample_rpn_(dev(crop_cu), dev(crop_ip), dev(_counts(crop_cu, crop_ip)), _state(ops, 99, 1000 + i)))
            assert np.array_equal(got[i, :r, :c].reshape(-1), want[0])
        pad = np.ones((rows, cols, a), bool)
        pad[:r, :c] = False
        assert not got[i][pad].any()


def _det_case(n_max, cases, rng):
    b = len(cases)
    is_pos = (rng.random((b, n_max)) < 0.5).astype(np.uint8)     # rows >= m hold junk that must be ignored
    n_rows = np.zeros(b, np.int32)
    for i, (p, q) in enumerate(cases):
        m = p + q
        flags = np.zeros(m, np.uint8)
        flags[rng.permutation(m)[:p]] = 1
        is_pos[i, :m] = flags
        n_rows[i] = m
    return is_pos, n_rows


def test_sample_det_vs_oracle_every_branch(ops):
    from faster_rcnn_b200 import _lib
    n_max, s, seed = 2000, 64, 2024
    cases = [(p, min(q, n_max - p)) for p in S_P for q in S_Q] + [(0, 0), (100, 1900)]   # m <= n_max
    is_pos, n_rows = _det_case(n_max, cases, np.random.default_rng(4))
    state = _state(ops, seed, 7)
    index, has = ops.sample_det(dev(is_pos), dev(n_rows), s, state)
    index, has = host(index), host(has)
    assert int(state[1]) == 7 + len(cases) and has.dtype == np.bool_
    for i, m in enumerate(n_rows.tolist()):
        want = S.det_samples(is_pos[i, :m], seed, 7 + i, s)
        assert np.array_equal(index[i], want), (i, cases[i])
        assert has[i] == (m > 0)
    with pytest.raises(_lib.FrcnnError) as e:
        ops.sample_det(dev(np.zeros((2, 4097), np.uint8)), dev(np.ones(2, np.int32)), s, state)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    from faster_rcnn_b200.runtime import get_context, ptr
    out, hs = dev(np.zeros((1, s), np.int32)), dev(np.zeros(1, np.uint8))
    with pytest.raises(_lib.FrcnnError) as e:
        get_context().call("frcnn_sample_det", ptr(dev(is_pos[:1])), ptr(dev(n_rows[:1])), n_max, s, None, 1, ptr(out), ptr(hs))
    assert e.value.code == _lib.ERR_INVALID


def test_state_batching_and_seeds(ops):
    rng = np.random.default_rng(5)
    is_pos, n_rows = _det_case(500, [(int(rng.integers(0, 40)), int(rng.integers(1, 400))) for _ in range(16)], rng)
    st = _state(ops, 31)
    a1, _ = ops.sample_det(dev(is_pos[:8]), dev(n_rows[:8]), 64, st)
    a2, _ = ops.sample_det(dev(is_pos[8:]), dev(n_rows[8:]), 64, st)
    assert int(st[1]) == 16
    whole, _ = ops.sample_det(dev(is_pos), dev(n_rows), 64, _state(ops, 31))
    assert np.array_equal(np.concatenate([host(a1), host(a2)]), host(whole))
    other, _ = ops.sample_det(dev(is_pos), dev(n_rows), 64, _state(ops, 32))
    assert not np.array_equal(host(other), host(whole))
    cu = (rng.random((16, 3000)) < 0.6).astype(np.uint8)
    ip = (rng.random((16, 3000)) < 0.1).astype(np.uint8)
    c = dev(_counts(cu, ip))
    st = _state(ops, 31)
    r1, r2 = ops.sample_rpn_(dev(cu[:8]), dev(ip[:8]), c[:8], st), ops.sample_rpn_(dev(cu[8:]), dev(ip[8:]), c[8:], st)
    assert int(st[1]) == 16
    whole = host(ops.sample_rpn_(dev(cu), dev(ip), c, _state(ops, 31)))
    assert np.array_equal(np.concatenate([host(r1), host(r2)]), whole)
    assert not np.array_equal(host(ops.sample_rpn_(dev(cu), dev(ip), c, _state(ops, 32))), whole)


def _det_batch(b, rows=19, cols=25, ch=16):
    from faster_rcnn_b200 import synth
    heads = [synth.rpn_outputs(rows, cols, 9, 170 + i, clustered=True) for i in range(b)]
    gts = [synth.gt_boxes(6, 400, 300, 180 + i) for i in range(b)]
    gts[2] = [("cat", 1, 1, 3, 3)]                                # no eligible RoI
    images = [FakeImage("d%d" % i, 400, 300, g, data=np.zeros((2, 2, 3), np.float32)) for i, g in enumerate(gts)]
    feat = np.random.default_rng(6).standard_normal((b, rows, cols, ch), dtype=np.float32)
    return np.concatenate([h[0] for h in heads]), np.concatenate([h[1] for h in heads]), feat, images


def test_det_training_pipeline_device_draw_vs_oracle(ops):
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.pipeline import DetTrainingPipeline
    b, seed = 40, 4242
    cls, regr, feat, images = _det_batch(b)
    mapping = synth.VOC_CLASS_MAPPING
    pipe = DetTrainingPipeline(mapping, DIMS)
    state = _state(ops, seed, 11)
    rois, y_cls, y_tr, pooled, has = pipe(cls, regr, feat, images, state=state)
    assert isinstance(has, torch.Tensor) and has.is_cuda and has.dtype == torch.bool
    assert int(state[1]) == 11 + b
    # oracle: label_rois's rows at the oracle's indices
    gt, gt_cls, n_gt = pipe.ground_truth(images)
    p_rois, _, count = ops.proposals(dev(regr), dev(cls), DIMS, 16, 12000, 0.7, 2000)
    l_rois, l_cls, l_tr, _, m = (host(t) for t in ops.label_rois(p_rois, gt, gt_cls, n_gt, len(mapping), n_roi=count))
    rois, y_cls, y_tr, pooled, has = host(rois), host(y_cls), host(y_tr), host(pooled), host(has)
    assert has.tolist() == [bool(v > 0) for v in m] and not has[2]
    for i in range(b):
        idx = S.det_samples(l_cls[i, :m[i], -1] == 0, seed, 11 + i, 64)
        if m[i] == 0:
            assert not rois[i].any() and not y_cls[i].any() and not y_tr[i].any()
            continue
        assert np.array_equal(rois[i], l_rois[i, idx]) and np.array_equal(y_cls[i], l_cls[i, idx])
        assert np.array_equal(y_tr[i], l_tr[i, idx])
        assert np.array_equal(pooled[i], R.roi_resize_fwd(feat[i], rois[i], 7))
    # chunking does not change the draw
    d_in = dev(cls), dev(regr)
    o32 = pipe.targets(*d_in, gt, gt_cls, n_gt, chunk=32, state=_state(ops, seed, 11))
    ob = pipe.targets(*d_in, gt, gt_cls, n_gt, chunk=b, state=_state(ops, seed, 11))
    for x, y, z in zip(o32, ob, (rois, y_cls, y_tr, has)):
        assert np.array_equal(host(x), host(y)) and np.array_equal(host(x), z)


def test_rpn_targets_device_feed_rpn_losses(ops):
    import torch
    from faster_rcnn_b200 import rpn_util, synth
    sizes = [(1000, 600), (800, 600), (600, 1000), (640, 480)]
    images = [FakeImage("r%d" % i, w, h, synth.gt_boxes(5 + 3 * i, w, h, 400 + i)) for i, (w, h) in enumerate(sizes)]
    mgr = rpn_util.RpnTrainingManager(O.conv_dims_resnet, 16, preprocess_func=None, anchor_dims=DIMS)
    state = _state(ops, 8, 3)
    cu, ip, bb, ext = mgr.rpn_targets_device(images, state)
    assert int(state[1]) == 3 + len(images)
    ext_h = host(ext)
    rows, cols = (int(v) for v in ext_h.max(axis=0))
    a = len(DIMS)
    assert cu.shape == (len(images), rows * cols * a) and bb.shape == (len(images), rows * cols * a, 4)
    # oracle-sampled targets from the same labels
    l_cu, l_ip, l_bb, _ = mgr._label_batch(images, ext_h, (rows, cols))
    want_cu = host(l_cu).reshape(len(images), rows, cols, a).copy()
    for i, (r, c) in enumerate(ext_h):
        crop_cu, crop_ip = (host(t).reshape(-1, rows, cols, a)[i, :r, :c].reshape(-1) for t in (l_cu, l_ip))
        want_cu[i, :r, :c] = S.rpn_keep(crop_cu, crop_ip, 8, 3 + i).reshape(r, c, a)
    assert np.array_equal(host(cu), want_cu.reshape(len(images), -1))
    assert np.array_equal(host(ip), host(l_ip)) and np.array_equal(host(bb), host(l_bb))
    g = torch.Generator(device="cuda").manual_seed(3)
    cls_pred = torch.rand(cu.shape, generator=g, device="cuda") * 0.98 + 0.01
    reg_pred = torch.randn(bb.shape, generator=g, device="cuda")
    got = ops.rpn_losses(cu, ip, bb, cls_pred, reg_pred, want_grad=True, extents=ext, padded_shape=(rows, cols))
    want = ops.rpn_losses(dev(want_cu.reshape(len(images), -1)), l_ip, l_bb, cls_pred, reg_pred, want_grad=True,
                          extents=ext, padded_shape=(rows, cols))
    for x, y in zip(got, want):
        assert torch.equal(x, y)


def test_device_draws_do_not_synchronise(ops):
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.pipeline import DetTrainingPipeline
    cls, regr, _, images = _det_batch(8)
    pipe = DetTrainingPipeline(synth.VOC_CLASS_MAPPING, DIMS)
    gt = pipe.ground_truth(images)
    d_cls, d_regr = dev(cls), dev(regr)
    rng = np.random.default_rng(7)
    cu = dev((rng.random((8, 5000)) < 0.6).astype(np.uint8))
    ip = dev((rng.random((8, 5000)) < 0.05).astype(np.uint8))
    counts = dev(_counts(host(cu), host(ip)))
    state = ops.sampler_state(1)
    pipe.targets(d_cls, d_regr, *gt, state=state)
    ops.sample_rpn_(cu, ip, counts, state)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pipe.targets(d_cls, d_regr, *gt, state=state)
        ops.sample_rpn_(cu, ip, counts, state)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert int(state[1]) == 32


def test_det_targets_graph_capture(ops):
    import torch
    from faster_rcnn_b200 import synth
    from faster_rcnn_b200.pipeline import DetTrainingPipeline
    from faster_rcnn_b200.runtime import Context, use_context
    cls, regr, _, images = _det_batch(8)
    pipe = DetTrainingPipeline(synth.VOC_CLASS_MAPPING, DIMS)
    gt = pipe.ground_truth(images)
    d_cls, d_regr = dev(cls), dev(regr)
    state = ops.sampler_state(77)
    ctx = Context(torch.cuda.current_device())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with use_context(ctx), torch.cuda.stream(side):
        for _ in range(2):
            pipe.targets(d_cls, d_regr, *gt, state=state)
        side.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            outs = pipe.targets(d_cls, d_regr, *gt, state=state)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert int(state[1]) == 16                                    # capture enqueues nothing
    graph.replay()
    first = [host(t) for t in outs]
    graph.replay()
    second = [host(t) for t in outs]
    assert int(state[1]) == 32
    assert not np.array_equal(first[0], second[0])
    eager = pipe.targets(d_cls, d_regr, *gt, state=_state(ops, 77, 16))
    for x, y in zip(eager, first):
        assert np.array_equal(host(x), y)
