"""Device JPEG decode (ops.jpeg_decode / frcnn_jpeg_decode) against cv2.imdecode(..., IMREAD_COLOR) and the oracle, bit for
bit, over sampling layouts, qualities, Huffman optimisation, restart intervals, sizes, content and spliced segments;
batches against single-file calls with canaries around every slot; corrupt entropy data confined to its image; and the
device-decode selection of shapes.Image.data_device / shapes.preprocessed_batch_device."""
import ctypes as C
import os

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from oracle import jpeg_oracle as J
from test_oracle_jpeg import SAMPLING, _content, encode, imdecode

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import _build, ops as ops_mod
    _build.build()
    return ops_mod


def _natural(h, w, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 127 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 23.0) + 30 * np.sin((xx + yy) / 5.0)
    return np.clip(base[:, :, None] + rng.normal(0, 12, (h, w, 3)) + np.array([10, -20, 5]), 0, 255).astype(np.uint8)


def decode_one(ops, data):
    packed, offsets, sizes, status = ops.jpeg_decode([data])
    h, w = (int(v) for v in sizes[0].cpu())
    assert int(status[0]) == 0
    return packed[:h * w * 3].cpu().numpy().reshape(h, w, 3)


def splice(data):
    """a COM and an APP9 segment and three 0xFF fill bytes in front of every marker segment after SOI"""
    out, pos = bytearray(data[:2]), 2
    scan = J.parse(data)["scan"]
    while pos < scan:
        ln = int.from_bytes(data[pos + 2:pos + 4], "big")
        out += b"\xff\xfe\x00\x06note" + b"\xff\xe9\x00\x04ab" + b"\xff\xff\xff" + data[pos:pos + 2 + ln]
        pos += 2 + ln
    return bytes(out) + data[scan:]


SIZES = [(1, 1), (1, 17), (17, 1), (8, 8), (15, 15), (16, 16), (17, 33)]
MATRIX = ([((h, w), s, q, "smooth", 0, False) for (h, w) in SIZES for s in list(SAMPLING) + ["grey"] for q in (1, 50, 90, 100)]
          + [((33, 47), s, q, kind, rst, opt) for s in list(SAMPLING) + ["grey"] for q, kind in
             [(100, "noise"), (90, "edges"), (50, "flat")] for rst, opt in [(0, True), (1, False), (3, True), (64, False)]])


@pytest.mark.parametrize("hw,sampling,quality,kind,rst,optimize", MATRIX)
def test_decode_equals_imdecode_and_oracle(ops, hw, sampling, quality, kind, rst, optimize):
    data = encode(_content(*hw, kind), sampling, quality, rst, optimize, grey=sampling == "grey")
    got = decode_one(ops, data)
    assert np.array_equal(got, imdecode(data))
    assert np.array_equal(got, J.decode(data))


@pytest.mark.parametrize("sampling", list(SAMPLING) + ["grey"])
def test_voc_sizes_qualities_and_restarts(ops, sampling):
    for i, (h, w) in enumerate([(375, 500), (500, 333)]):
        img = _natural(h, w, i)
        for kw in (dict(quality=90), dict(quality=100, rst=3, optimize=True), dict(quality=90, luma=95, chroma=30),
                   dict(quality=50, rst=64)):
            data = encode(img, sampling, grey=sampling == "grey", **kw)
            assert np.array_equal(decode_one(ops, data), imdecode(data)), (h, w, kw)


def test_large_images(ops):
    for (h, w), s in [((1000, 1500), "420"), ((4000, 6000), "420"), ((1000, 1500), "444")]:
        data = encode(_natural(h, w, 7), s, 90, rst=0 if h > 1000 else 7)
        assert np.array_equal(decode_one(ops, data), imdecode(data)), (h, w, s)


def test_long_codes_and_clamps(ops):
    """white noise at quality 100 uses Huffman codes longer than the device's 9-bit fast table; saturated content
    drives the IDCT's range limit and the colour clamps"""
    data = encode(_content(64, 64, "noise", 3), "444", 100)
    assert max(J.code_lengths(data)) > 9
    assert np.array_equal(decode_one(ops, data), imdecode(data))
    sat = np.zeros((48, 48, 3), np.uint8)
    sat[::2, :, 2] = 255
    sat[:, ::3, 0] = 255
    for s in SAMPLING:
        data = encode(sat, s, 100)
        assert np.array_equal(decode_one(ops, data), imdecode(data)), s


def test_spliced_segments_and_fill_bytes(ops):
    for s in ("420", "grey"):
        data = splice(encode(_content(29, 35, "smooth"), s, 90, rst=2, grey=s == "grey"))
        assert ops.jpeg_supported(data) == (29, 35)
        assert np.array_equal(decode_one(ops, data), imdecode(data))


# ---- batches, canaries, corrupt data ------------------------------------------------------------------------------------
CANARY = 0xA5


def decode_with_canaries(ops, files, gap=64):
    """frcnn_jpeg_decode into slots separated by `gap` canary bytes, with `gap` more after the last: -> (images, status,
    canaries intact)"""
    import torch
    from faster_rcnn_b200.runtime import get_context, ptr
    ctx = get_context()
    arrays = [np.frombuffer(f, np.uint8) for f in files]
    hw = [ops.jpeg_supported(a) for a in arrays]
    nb = np.array([a.size for a in arrays], np.int64)
    foff = np.concatenate([[0], np.cumsum(nb)[:-1]]).astype(np.int64)
    blob = np.concatenate(arrays)
    n = [h * w * 3 for h, w in hw]
    ooff = np.array([sum(n[:i]) + gap * (i + 1) for i in range(len(n))], np.int64)
    total = int(ooff[-1] + n[-1] + gap)
    out = torch.full((total,), CANARY, dtype=torch.uint8, device=ctx.device)
    status = torch.full((len(files),), 7, dtype=torch.int32, device=ctx.device)
    files_dev = torch.from_numpy(blob).to(ctx.device)
    ooff_dev = torch.from_numpy(ooff).to(ctx.device)
    ctx.call("frcnn_jpeg_decode", blob.ctypes.data_as(C.c_void_p), ptr(files_dev), foff.ctypes.data_as(C.c_void_p),
             nb.ctypes.data_as(C.c_void_p), len(files), ptr(out), ptr(ooff_dev), total, ptr(status))
    host = out.cpu().numpy()
    imgs = [host[o:o + k].reshape(h, w, 3) for o, k, (h, w) in zip(ooff, n, hw)]
    mask = np.ones(total, bool)
    for o, k in zip(ooff, n):
        mask[o:o + k] = False
    return imgs, status.cpu().numpy(), bool((host[mask] == CANARY).all())


def _mixed_files(count):
    rng = np.random.default_rng(11)
    files = []
    for i in range(count):
        h, w = [(375, 500), (500, 333), (333, 500), (17, 33), (1, 1), (64, 48)][i % 6]
        s = (list(SAMPLING) + ["grey"])[i % 6]
        files.append(encode(_natural(h, w, i), s, int(rng.choice([50, 75, 90, 95])), rst=int(rng.choice([0, 0, 1, 5])),
                            optimize=bool(i % 2), grey=s == "grey"))
    return files


def test_mixed_batch_equals_single_calls_with_canaries(ops):
    files = _mixed_files(64)
    imgs, status, canaries = decode_with_canaries(ops, files)
    assert canaries and (status == 0).all()
    for f, img in zip(files, imgs):
        assert np.array_equal(img, imdecode(f))
        assert np.array_equal(img, decode_one(ops, f))
    packed, offsets, sizes, st = ops.jpeg_decode(files)
    off, sz = offsets.cpu().numpy(), sizes.cpu().numpy()
    host = packed.cpu().numpy()
    for i, f in enumerate(files):
        h, w = sz[i]
        assert np.array_equal(host[off[i]:off[i] + h * w * 3].reshape(h, w, 3), imgs[i])


def _corrupt(data, want, seed):
    """flip bytes of the scan until the oracle reports `want` (deterministic in `seed`)"""
    scan = J.parse(data)["scan"]
    rng = np.random.default_rng(seed)
    for _ in range(4000):
        b = bytearray(data)
        for _ in range(2):
            i = int(rng.integers(scan, len(data) - 2))
            v = int(rng.integers(0, 256))
            if v == 0xFF or b[i] == 0xFF or b[i - 1] == 0xFF:
                continue
            b[i] = v
        try:
            J.decode_coefficients(bytes(b))
        except J.CorruptData as e:
            if want in str(e):
                return bytes(b)
    raise AssertionError("no corruption of kind %r found" % want)


def test_corrupt_entropy_data_is_confined_to_its_image(ops):
    good = _mixed_files(6)
    base = encode(_natural(40, 56, 3), "420", 75, optimize=True)
    scan = J.parse(base)["scan"]
    truncated = base[:scan + (len(base) - scan) // 2] + b"\xff\xd9"
    bad = [truncated, _corrupt(base, "past 63", 1), _corrupt(base, "not in table", 2)]
    for b in bad:
        files = good[:3] + [b] + good[3:]
        imgs, status, canaries = decode_with_canaries(ops, files)
        assert canaries
        assert status[3] < 0 and not imgs[3].any()
        for i in (0, 1, 2, 4, 5, 6):
            assert status[i] == 0 and np.array_equal(imgs[i], imdecode(files[i]))


# ---- shapes: selection of the device decoder ----------------------------------------------------------------------------
@pytest.fixture
def jpeg_dir(tmp_path):
    paths = []
    for i, (h, w) in enumerate([(375, 500), (500, 333), (281, 500), (500, 375)]):
        p = tmp_path / ("img%d.jpg" % i)
        p.write_bytes(encode(_natural(h, w, i), ("420", "444", "422", "grey")[i], 90, grey=i == 3))
        paths.append(str(p))
    return paths


def _images(paths, png=None):
    from faster_rcnn_b200.shapes import Image
    out = []
    for i, p in enumerate(paths):
        raw = cv2.imread(p)
        h, w = raw.shape[:2]
        img = Image("n%d" % i, int(w * 1.6), int(h * 1.6), image_path=p)
        out.append(img.horizontal_flip() if i % 2 else img)
    return out


def test_preprocessed_batch_device_uses_the_device_decoder_bit_exactly(ops, jpeg_dir, monkeypatch):
    from faster_rcnn_b200 import shapes
    images = _images(jpeg_dir)
    host_images = [shapes._host_decoded(img) for img in images]
    calls = []
    real = ops.jpeg_decode
    monkeypatch.setattr(ops, "jpeg_decode", lambda files: calls.append(len(files)) or real(files))
    got, ext = shapes.preprocessed_batch_device(images)
    assert calls == [len(images)]
    want, wext = shapes.preprocessed_batch_device(host_images)
    assert calls == [len(images)]
    assert np.array_equal(got.cpu().numpy(), want.cpu().numpy())
    assert np.array_equal(ext.cpu().numpy(), wext.cpu().numpy())
    for img, himg in zip(images, host_images):
        a, b = img.data_device(mean=ops.IMAGENET_MEAN_BGR), himg.data_device(mean=ops.IMAGENET_MEAN_BGR)
        assert all(np.array_equal(x.cpu().numpy(), y.cpu().numpy()) for x, y in zip(a, b))
    assert calls == [len(images)] + [1] * len(images)


def test_batch_with_an_unsupported_file_takes_the_host_path(ops, jpeg_dir, tmp_path, monkeypatch):
    from faster_rcnn_b200 import shapes
    prog = tmp_path / "prog.jpg"
    prog.write_bytes(cv2.imencode(".jpg", _natural(300, 400, 9), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes())
    images = _images(jpeg_dir + [str(prog)])
    calls = []
    monkeypatch.setattr(ops, "jpeg_decode", lambda files: calls.append(1))
    got, _ = shapes.preprocessed_batch_device(images)
    want, _ = shapes.preprocessed_batch_device([shapes._host_decoded(img) for img in images])
    assert not calls
    assert np.array_equal(got.cpu().numpy(), want.cpu().numpy())


def test_voc_files_decode_like_imread(ops):
    from oracle import ref_loader
    d = os.path.join(ref_loader.VOC_DIR, "JPEGImages")
    if not os.path.isdir(d):
        pytest.skip("reference checkout with VOC test images not present")
    names = sorted(os.listdir(d))
    assert names
    for i in range(0, len(names), 64):
        files = [open(os.path.join(d, n), "rb").read() for n in names[i:i + 64]]
        for n, f in zip(names[i:i + 64], files):
            p = J.parse(f)
            assert [(c["h"], c["v"]) for c in p["comps"]] == [(2, 2), (1, 1), (1, 1)], n    # baseline 4:2:0
            assert ops.jpeg_supported(f) is not None, n
        packed, offsets, sizes, status = ops.jpeg_decode(files)
        assert (status.cpu().numpy() == 0).all()
        host, off, sz = packed.cpu().numpy(), offsets.cpu().numpy(), sizes.cpu().numpy()
        for k, n in enumerate(names[i:i + 64]):
            h, w = sz[k]
            assert np.array_equal(host[off[k]:off[k] + h * w * 3].reshape(h, w, 3),
                                  cv2.imread(os.path.join(d, n))), n
