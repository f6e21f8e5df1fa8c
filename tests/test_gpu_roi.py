"""GPU parity: RoI layer (K-d) forward / backward through the C ABI vs oracle/roi_oracle.py.

resize mode: forward bit-exact (same float32 op order, no FMA); backward within 1e-5 relative
(the oracle sums each RoI into a private crop first like TF's slice-gradient + AddN, the kernel adds
taps straight into the owned tile -- a different but fixed float32 summation order).
max mode: outputs and argmax bit-exact; backward bit-exact while one warp walks a block's list (fewer than 256 RoIs
per image, or launches large enough to need no slicing), 1e-5 relative (like the resize mode) when the list is sliced across warps."""
import numpy as np
import pytest

from helpers import dev, host
from oracle import roi_oracle as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import ops as _ops
    return _ops


def _rois(rng, n, rows, cols, dtype=np.int16):
    x1 = rng.integers(0, cols - 1, n)
    y1 = rng.integers(0, rows - 1, n)
    x2 = np.minimum(cols - 1, x1 + 1 + rng.integers(0, cols, n))
    y2 = np.minimum(rows - 1, y1 + 1 + rng.integers(0, rows, n))
    return np.stack([x1, y1, x2, y2], axis=1).astype(dtype)


@pytest.mark.parametrize("h,w,c,n,dtype", [
    (12, 17, 64, 40, np.int16), (38, 63, 128, 64, np.int16), (9, 9, 1024, 8, np.int32),
    (12, 17, 20, 16, np.float32), (7, 5, 6, 10, np.int16),      # C % 4 != 0 -> scalar-channel kernels
])
def test_roi_resize_forward_backward(ops, h, w, c, n, dtype):
    rng = np.random.default_rng(h * w + c)
    feat = rng.standard_normal((h, w, c), dtype=np.float32)
    rois = _rois(rng, n, h, w, dtype)
    out = ops.roi_forward(dev(feat[None]), dev(rois[None]), 7, "resize")
    want = R.roi_resize_fwd(feat, rois, 7)
    assert tuple(out.shape) == (1, n, 7, 7, c) and np.array_equal(host(out)[0], want)
    gout = rng.standard_normal((n, 7, 7, c), dtype=np.float32)
    gfeat = host(ops.roi_backward(dev(gout[None]), dev(rois[None]), (1, h, w, c), "resize"))[0]
    wgrad = R.roi_resize_bwd(gout, rois, (h, w, c))
    scale = np.abs(wgrad).max()
    assert np.abs(gfeat - wgrad).max() <= 1e-5 * scale            # tolerance: 1e-5 relative to the largest gradient


@pytest.mark.parametrize("h,w,c,n", [(12, 17, 64, 40), (38, 63, 128, 64), (7, 5, 6, 10)])
def test_roi_max_forward_backward(ops, h, w, c, n):
    rng = np.random.default_rng(h + w + c)
    feat = rng.standard_normal((h, w, c), dtype=np.float32)
    feat[::3, ::2] = feat[0, 0]                                    # plant ties: first maximum must win
    rois = _rois(rng, n, h, w)
    out, arg = ops.roi_forward(dev(feat[None]), dev(rois[None]), 7, "max")
    wout, warg = R.roi_max_fwd(feat, rois, 7)
    assert np.array_equal(host(out)[0], wout) and np.array_equal(host(arg)[0], warg)
    gout = rng.standard_normal((n, 7, 7, c), dtype=np.float32)
    gfeat = host(ops.roi_backward(dev(gout[None]), dev(rois[None]), (1, h, w, c), "max", argmax=arg))[0]
    assert np.array_equal(gfeat, R.roi_max_bwd(gout, warg, (h, w, c)))


def test_roi_small_and_edge_crops(ops):
    """1x1, 1xW, Hx1 crops (upsampling repeats cells), crops touching the border, x2 beyond the map."""
    rng = np.random.default_rng(0)
    h, w, c = 10, 13, 8
    feat = rng.standard_normal((h, w, c), dtype=np.float32)
    rois = np.array([[0, 0, 1, 1], [12, 9, 13, 10], [0, 0, 13, 1], [5, 0, 6, 10], [0, 0, 13, 10], [3, 2, 10, 9],
                     [11, 8, 13, 10], [2, 3, 4, 10]], np.int16)
    assert np.array_equal(host(ops.roi_forward(dev(feat[None]), dev(rois[None]), 7, "resize"))[0],
                          R.roi_resize_fwd(feat, rois, 7))
    out, arg = ops.roi_forward(dev(feat[None]), dev(rois[None]), 7, "max")
    wout, warg = R.roi_max_fwd(feat, rois, 7)
    assert np.array_equal(host(out)[0], wout) and np.array_equal(host(arg)[0], warg)
    # a 7x7 crop resized to 7x7 is the crop itself
    assert np.array_equal(host(ops.roi_forward(dev(feat[None]), dev(rois[5:6][None]), 7, "resize"))[0, 0], feat[2:9, 3:10])
    # x2/y2 beyond the map are clipped like a python slice
    far = np.array([[8, 6, 30, 30]], np.int16)
    assert np.array_equal(host(ops.roi_forward(dev(feat[None]), dev(far[None]), 7, "resize"))[0],
                          R.roi_resize_fwd(feat, np.array([[8, 6, 13, 10]]), 7))


def test_roi_batch_and_pool_sizes(ops):
    rng = np.random.default_rng(4)
    b, h, w, c, n = 3, 14, 15, 32, 9
    feat = rng.standard_normal((b, h, w, c), dtype=np.float32)
    rois = np.stack([_rois(rng, n, h, w) for _ in range(b)])
    for pool in (7, 3, 14):
        out = host(ops.roi_forward(dev(feat), dev(rois), pool, "resize"))
        for i in range(b):
            assert np.array_equal(out[i], R.roi_resize_fwd(feat[i], rois[i], pool))
    gout = rng.standard_normal((b, n, 7, 7, c), dtype=np.float32)
    g = host(ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "resize"))
    for i in range(b):
        want = R.roi_resize_bwd(gout[i], rois[i], (h, w, c))
        assert np.abs(g[i] - want).max() <= 1e-5 * np.abs(want).max()


@pytest.mark.parametrize("b,h,w,c,n,pool", [
    (4, 38, 63, 1024, 24, 7),     # 1024 channels: only full channel slabs (no channel guards), one plan warp per block
    (2, 14, 15, 384, 12, 7),      # 384 channels: resize mode's second 256-channel slab is partial
    (2, 14, 15, 32, 9, 3),        # pool 3, one 128-channel slab of which 32 channels exist
    (2, 14, 15, 64, 9, 14),       # pool 14 > 8: 32-bit masks and RoI records (wide plan)
    (1, 12, 17, 64, 40, 9),       # pool 9: the smallest pool of the wide plan
    (1, 38, 63, 128, 64, 32),     # pool 32: every bit of the 32-bit masks
    (1, 12, 17, 128, 300, 7),     # >= 256 RoIs in a small launch: every block's list sliced across warps
    (1, 9, 11, 1024, 257, 7),     # same with 1024 channels and a ragged last slice
    (1, 38, 63, 64, 1100, 14),    # > 1024 RoIs, pool 14: wide plan with 8-warp CTAs per block, sliced lists
])
def test_roi_backward_kernel_variants(ops, b, h, w, c, n, pool):
    """Variants of the work-list backward, both modes: channel slabs and guards of the streaming kernel, the narrow
    (pool <= 8) and wide plan, the plan's CTA shapes and the slicing of a block's list across warps."""
    rng = np.random.default_rng(b * h + c + pool)
    feat = rng.standard_normal((b, h, w, c), dtype=np.float32)
    feat[:, ::3, ::2] = feat[0, 0, 0]                              # ties for the max mode
    rois = np.stack([_rois(rng, n, h, w) for _ in range(b)])
    gout = rng.standard_normal((b, n, pool, pool, c), dtype=np.float32)
    g = host(ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "resize"))
    out, arg = ops.roi_forward(dev(feat), dev(rois), pool, "max")
    gm = host(ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "max", argmax=arg))
    for i in range(b):
        want = R.roi_resize_bwd(gout[i], rois[i], (h, w, c))
        assert np.abs(g[i] - want).max() <= 1e-5 * np.abs(want).max()
        wout, warg = R.roi_max_fwd(feat[i], rois[i], pool)
        assert np.array_equal(host(out)[i], wout) and np.array_equal(host(arg)[i], warg)
        wm = R.roi_max_bwd(gout[i], warg, (h, w, c))
        if n < 256:                       # one warp walks a block's whole list: the oracle's (roi, ph, pw) order, bit for bit
            assert np.array_equal(gm[i], wm)
        else:                             # sliced lists: partial sums are added in slice order (fixed, but re-associated)
            assert np.abs(gm[i] - wm).max() <= 1e-5 * np.abs(wm).max()


def test_roi_backward_ignores_environment(ops, monkeypatch):
    """The work-list backward picks its variant from the shape and the device: variables that once overrode the variant,
    the channels per lane or the list slices change neither the gradients nor whether the call succeeds."""
    import torch
    b, h, w, c, n, pool = 2, 14, 15, 256, 40, 7
    rng = np.random.default_rng(b * h + c + n)
    feat = rng.standard_normal((b, h, w, c), dtype=np.float32)
    rois = dev(np.stack([_rois(rng, n, h, w) for _ in range(b)]))
    gout = dev(rng.standard_normal((b, n, pool, pool, c), dtype=np.float32))
    _, arg = ops.roi_forward(dev(feat), rois, pool, "max")

    def grads():
        return (ops.roi_backward(gout, rois, (b, h, w, c), "resize"),
                ops.roi_backward(gout, rois, (b, h, w, c), "max", argmax=arg))

    first = grads()
    for name, value in (("FRCNN_BWD_PARTS", "3"), ("FRCNN_BWD_IMPL", "cell"), ("FRCNN_BWD_CPB", "1")):
        with monkeypatch.context() as m:
            m.setenv(name, value)
            for got, want in zip(grads(), first):
                assert torch.equal(got, want), name


def test_roi_full_size_properties(ops):
    """C5 shape (38x63x1024, 2000 RoIs): <dY, fwd(X)> == <bwd(dY), X> (the backward is the exact adjoint of
    the forward), linearity of the forward, and a spot check of 16 RoIs against the oracle."""
    import torch
    from faster_rcnn_b200 import synth
    h, w, c, n = 38, 63, 1024, 2000
    torch.manual_seed(0)
    feat = torch.randn((1, h, w, c), device="cuda")
    feat2 = torch.randn((1, h, w, c), device="cuda")
    rois_np = synth.random_rois(n, h, w, 3)
    rois = dev(rois_np[None])
    gout = torch.randn((1, n, 7, 7, c), device="cuda")
    out = ops.roi_forward(feat, rois, 7, "resize")
    gfeat = ops.roi_backward(gout, rois, (1, h, w, c), "resize")
    lhs = (out.double() * gout.double()).sum().item()
    rhs = (gfeat.double() * feat.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), abs(rhs), 1.0)
    out2 = ops.roi_forward(feat + feat2, rois, 7, "resize")
    ref2 = out + ops.roi_forward(feat2, rois, 7, "resize")
    assert (out2 - ref2).abs().max().item() <= 1e-4
    pick = np.arange(0, n, n // 16)[:16]
    assert np.array_equal(host(out)[0, pick], R.roi_resize_fwd(host(feat)[0], rois_np[pick], 7))
    # max mode: gradient mass is conserved (every dY element lands on exactly one cell)
    mout, marg = ops.roi_forward(feat, rois, 7, "max")
    mg = ops.roi_backward(gout, rois, (1, h, w, c), "max", argmax=marg)
    assert abs(mg.double().sum().item() - gout.double().sum().item()) <= 1e-6 * gout.double().abs().sum().item()
    gathered = torch.gather(feat.reshape(h * w, c), 0, marg.reshape(-1, c).long()).reshape(mout.shape)
    assert torch.equal(gathered, mout)


def test_roi_backward_65536_rois_properties(ops):
    """65536 RoIs of one image (pool 7) take the wide plan, whose queue keeps RoI indices beyond 16 bits.  Too many RoIs
    for the per-RoI oracle: <dY, fwd(X)> == <bwd(dY), X> in resize mode; in max mode gradient mass conservation and a
    float64 scatter-add of dY onto the arg-max cells."""
    import torch
    h, w, c, n = 12, 17, 16, 65536
    rng = np.random.default_rng(11)
    rois = dev(_rois(rng, n, h, w)[None])
    torch.manual_seed(2)
    feat = torch.rand((1, h, w, c), device="cuda")              # non-negative: the inner products do not cancel
    gout = torch.rand((1, n, 7, 7, c), device="cuda")
    out = ops.roi_forward(feat, rois, 7, "resize")
    gfeat = ops.roi_backward(gout, rois, (1, h, w, c), "resize")
    lhs = (out.double() * gout.double()).sum().item()
    rhs = (gfeat.double() * feat.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), abs(rhs), 1.0)
    gout = torch.randn((1, n, 7, 7, c), device="cuda")
    mout, marg = ops.roi_forward(feat, rois, 7, "max")
    mg = ops.roi_backward(gout, rois, (1, h, w, c), "max", argmax=marg)
    assert abs(mg.double().sum().item() - gout.double().sum().item()) <= 1e-6 * gout.double().abs().sum().item()
    gathered = torch.gather(feat.reshape(h * w, c), 0, marg.reshape(-1, c).long()).reshape(mout.shape)
    assert torch.equal(gathered, mout)
    # and every dY element lands on its arg-max cell (float32 sums of ~15000 terms per element against float64 ones)
    idx, g = marg.reshape(-1, c).long(), gout.reshape(-1, c).double()
    want = torch.zeros((h * w, c), dtype=torch.float64, device="cuda").scatter_add_(0, idx, g)
    mass = torch.zeros((h * w, c), dtype=torch.float64, device="cuda").scatter_add_(0, idx, g.abs())
    assert bool(((mg.reshape(h * w, c).double() - want).abs() <= 1e-6 * mass).all())


def test_roi_layer_dropin_and_autograd():
    """custom_layers.RoiResizeConv: Keras-style surface + torch autograd through the CUDA backward."""
    import torch
    from faster_rcnn_b200.custom_layers import RoiResizeConv
    rng = np.random.default_rng(6)
    h, w, c, n = 11, 12, 16, 5
    feat = rng.standard_normal((1, h, w, c), dtype=np.float32)
    rois = _rois(rng, n, h, w)[None]
    layer = RoiResizeConv(7, n)
    out = layer([feat, rois])
    assert isinstance(out, np.ndarray) and out.shape == (1, n, 7, 7, c)
    assert layer.nb_channels == c and layer.compute_output_shape(None) == (None, n, 7, 7, c)
    assert layer.get_config() == {'pool_size': 7, 'num_rois': n}
    assert np.array_equal(out[0], R.roi_resize_fwd(feat[0], rois[0], 7))
    x = dev(feat).requires_grad_(True)
    y = layer([x, dev(rois)])
    gout = rng.standard_normal((1, n, 7, 7, c), dtype=np.float32)
    (y * dev(gout)).sum().backward()
    want = R.roi_resize_bwd(gout[0], rois[0], (h, w, c))
    assert np.abs(host(x.grad)[0] - want).max() <= 1e-5 * np.abs(want).max()
    mlayer = RoiResizeConv(7, n, mode="max")
    assert mlayer.get_config() == {'pool_size': 7, 'num_rois': n, 'mode': 'max'}
    assert np.array_equal(mlayer([feat, rois])[0], R.roi_max_fwd(feat[0], rois[0], 7)[0])
    with pytest.raises(ValueError):
        layer([feat, rois[:, :3]])


def test_roi_max_full_size_equals_torchvision_roi_pool(ops):
    """C5 shape (38x63x1024, 2000 RoIs): the CUDA max-mode forward equals torchvision.ops.roi_pool's CUDA kernel bit for
    bit (an independent implementation of the same RoIPool spec), and the arg-max gathers those outputs."""
    import torch
    tv = pytest.importorskip("torchvision")
    from faster_rcnn_b200 import synth
    h, w, c, n = 38, 63, 1024, 2000
    torch.manual_seed(1)
    feat = torch.randn((1, h, w, c), device="cuda")
    rois_np = synth.random_rois(n, h, w, 5)
    out, arg = ops.roi_forward(feat, dev(rois_np[None]), 7, "max")
    boxes = torch.tensor(np.concatenate([np.zeros((n, 1)), rois_np[:, :2], rois_np[:, 2:] - 1], axis=1), dtype=torch.float32, device="cuda")
    want = tv.ops.roi_pool(feat.permute(0, 3, 1, 2).contiguous(), boxes, output_size=7, spatial_scale=1.0)     # (N, C, 7, 7)
    assert torch.equal(out[0], want.permute(0, 2, 3, 1))
    assert torch.equal(torch.gather(feat.reshape(h * w, c), 0, arg.reshape(-1, c).long()).reshape(out.shape), out)


def _decode_compact(code, rois, pool, width):
    """one-byte arg-max (dy << 4 | dx from the bin's first cell) -> flat cell index y*W + x (include/frcnn_b200.h)."""
    code = code.astype(np.int64)
    flat = np.zeros(code.shape, np.int64)
    for r, (x1, y1, x2, y2) in enumerate(np.asarray(rois).tolist()):
        h, w = y2 - y1, x2 - x1
        ya = y1 + (np.arange(pool) * h) // pool
        xa = x1 + (np.arange(pool) * w) // pool
        flat[r] = (ya[:, None, None] + (code[r] >> 4)) * width + xa[None, :, None] + (code[r] & 15)
    return flat


@pytest.mark.parametrize("b,h,w,c,n,pool", [
    (2, 12, 17, 64, 40, 7),        # one warp walks every list: backward in the oracle's order
    (1, 38, 63, 1024, 300, 7),     # C5 map, sliced lists
    (2, 14, 15, 384, 12, 3),       # pool 3 (bins up to 6 x 6), partial channel slab
    (1, 38, 94, 256, 64, 7),       # KITTI map: bins up to 7 x 15 cells
    (1, 10, 13, 8, 9, 8),
])
def test_roi_max_compact_argmax(ops, b, h, w, c, n, pool):
    """Max mode with the one-byte arg-max: same outputs, codes that decode to the oracle's flat arg-max, and the same
    gradient as the int32 path (bit for bit while one warp walks a block's list, 1e-5 when the lists are sliced)."""
    import torch
    assert ops.roi_compact_supported(h, w, c, pool)
    rng = np.random.default_rng(h * w + n)
    feat = rng.standard_normal((b, h, w, c), dtype=np.float32)
    feat[:, ::3, ::2] = feat[0, 0, 0]                              # ties: the first maximum must win
    rois = np.stack([_rois(rng, n, h, w) for _ in range(b)])
    rois[0, 0] = [0, 0, w, h]                                      # the largest bins the map allows
    rois[0, 1] = [w - 1, h - 1, w, h]                              # 1 x 1 crop: every bin repeats the same cell
    out, code = ops.roi_forward(dev(feat), dev(rois), pool, "max", compact=True)
    out32, arg32 = ops.roi_forward(dev(feat), dev(rois), pool, "max")
    assert code.dtype == torch.uint8 and torch.equal(out, out32)
    for i in range(b):
        wout, warg = R.roi_max_fwd(feat[i], rois[i], pool)
        assert np.array_equal(host(out)[i], wout)
        assert np.array_equal(_decode_compact(host(code)[i], rois[i], pool, w), warg)
    gout = rng.standard_normal((b, n, pool, pool, c), dtype=np.float32)
    g8 = ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "max", argmax=code)
    g32 = ops.roi_backward(dev(gout), dev(rois), (b, h, w, c), "max", argmax=arg32)
    if n < 256:                        # one warp per list in both paths: the same additions in the same order
        assert torch.equal(g8, g32)
    else:                              # sliced lists: the two paths cut the lists differently (fixed order, re-associated)
        assert (g8 - g32).abs().max().item() <= 1e-5 * g32.abs().max().item()
    # the layer picks the compact format by itself
    from faster_rcnn_b200.custom_layers import roi_pool
    x = dev(feat).requires_grad_(True)
    y = roi_pool(x, dev(rois), pool, "max")
    (y * dev(gout)).sum().backward()
    assert torch.equal(y.detach(), out) and torch.equal(x.grad, g8)


def test_roi_max_compact_unsupported_shapes_fail_loudly(ops):
    import torch
    from faster_rcnn_b200 import _lib
    assert not ops.roi_compact_supported(120, 40, 64, 7)           # bins up to 19 rows
    assert not ops.roi_compact_supported(38, 63, 6, 7)             # C % 4 != 0
    with pytest.raises(_lib.FrcnnError) as e:
        ops.roi_forward(torch.zeros((1, 120, 40, 64), device="cuda"), dev(np.array([[[0, 0, 40, 120]]], np.int16)), 7, "max",
                        compact=True)
    assert e.value.code == _lib.ERR_UNSUPPORTED
