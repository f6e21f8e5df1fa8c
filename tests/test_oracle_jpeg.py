"""The JPEG oracle (oracle/jpeg_oracle.py) against cv2.imdecode(..., IMREAD_COLOR) bit for bit on small files of every
supported layout, its model of the self-synchronising Huffman decode against its sequential decode, and the header
inspection of the library (frcnn_jpeg_inspect, CPU only) on supported, unsupported and malformed files."""
import ctypes as C

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from oracle import jpeg_oracle as J

SAMPLING = {"444": 0x111111, "422": 0x211111, "440": 0x121111, "420": 0x221111, "411": 0x411111}


def _content(h, w, kind, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "flat":
        return np.full((h, w, 3), (40, 200, 90), np.uint8)
    if kind == "edges":
        yy, xx = np.mgrid[0:h, 0:w]
        img = np.repeat(np.where((xx // 3 + yy // 2) % 2 == 1, 255, 0)[:, :, None], 3, axis=2).astype(np.uint8)
        img[..., 1] = np.where(xx > w // 2, 255, 0)
        return img
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(xx * 7 + yy * 3) % 256, (xx * xx + yy) % 256, 128 + 100 * np.sin(xx / 5.0 + yy / 7.0)],
                    -1).astype(np.uint8)


def encode(img, sampling="420", quality=90, rst=0, optimize=False, luma=None, chroma=None, grey=False):
    p = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize), cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if luma is not None:
        p += [cv2.IMWRITE_JPEG_LUMA_QUALITY, luma, cv2.IMWRITE_JPEG_CHROMA_QUALITY, chroma]
    if grey:
        img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    else:
        p += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    ok, buf = cv2.imencode(".jpg", img, p)
    assert ok
    return buf.tobytes()


def imdecode(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


CASES = [((h, w), s, q, kind, rst) for (h, w) in [(1, 1), (1, 17), (17, 1), (8, 8), (15, 15), (16, 16), (17, 33)]
         for s in list(SAMPLING) + ["grey"] for q, kind, rst in [(1, "smooth", 0), (50, "noise", 3), (100, "edges", 1)]]


@pytest.mark.parametrize("hw,sampling,quality,kind,rst", CASES)
def test_oracle_equals_imdecode(hw, sampling, quality, kind, rst):
    data = encode(_content(*hw, kind), sampling, quality, rst, grey=sampling == "grey")
    assert np.array_equal(J.decode(data), imdecode(data))


@pytest.mark.parametrize("sampling", list(SAMPLING))
def test_oracle_equals_imdecode_larger(sampling):
    img = _content(40, 57, "smooth", 1)
    for kw in (dict(quality=90), dict(quality=75, optimize=True, rst=2), dict(luma=95, chroma=20, quality=90)):
        data = encode(img, sampling, **kw)
        assert np.array_equal(J.decode(data), imdecode(data)), kw


@pytest.mark.parametrize("sub_bits", [32, 64, 128, 256, 512, 1024])
def test_self_synchronising_decode_equals_sequential(sub_bits):
    for s, q, rst, kind, opt in [("420", 90, 0, "smooth", False), ("444", 100, 0, "noise", True),
                                 ("411", 50, 3, "smooth", True), ("grey", 95, 1, "noise", False)]:
        data = encode(_content(31, 42, kind, 2), s, q, rst, opt, grey=s == "grey")
        want = J.decode_coefficients(data)[0]
        assert np.array_equal(J.sync_decode(data, sub_bits), want), (s, q, rst)


# ---- frcnn_jpeg_inspect -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from faster_rcnn_b200 import _build, _lib
    _build.build()
    return _lib.load()


def inspect(lib, data):
    a = np.frombuffer(bytes(data), np.uint8)
    hw = np.zeros(2, np.int32)
    rc = lib.frcnn_jpeg_inspect(a.ctypes.data_as(C.c_void_p), a.size, hw.ctypes.data_as(C.c_void_p))
    return rc, (int(hw[0]), int(hw[1]))


def _segment(marker, payload):
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + payload


def _exif(orientation):
    tiff = b"II*\x00\x08\x00\x00\x00\x01\x00" + b"\x12\x01\x03\x00\x01\x00\x00\x00" + bytes([orientation, 0, 0, 0]) + \
        b"\x00\x00\x00\x00"
    return _segment(0xE1, b"Exif\x00\x00" + tiff)


def _strip_app0(data):
    i = data.index(b"\xff\xe0")
    return data[:i] + data[i + 2 + int.from_bytes(data[i + 2:i + 4], "big"):]


def test_inspect_accepts_every_supported_layout(lib):
    from faster_rcnn_b200 import _lib
    img = _content(23, 31, "smooth")
    for s in list(SAMPLING) + ["grey"]:
        for kw in (dict(), dict(rst=5, optimize=True)):
            data = encode(img, s, grey=s == "grey", **kw)
            assert inspect(lib, data) == (_lib.OK, (23, 31)), (s, kw)
    data = encode(img)
    assert inspect(lib, data[:2] + _exif(1) + data[2:])[0] == _lib.OK
    assert inspect(lib, _strip_app0(data))[0] == _lib.OK          # no JFIF, component IDs 1, 2, 3: YCbCr


def test_inspect_reports_unsupported(lib):
    from faster_rcnn_b200 import _lib
    img = _content(23, 31, "smooth")
    data = encode(img)
    ok, prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    assert inspect(lib, prog.tobytes())[0] == _lib.ERR_UNSUPPORTED
    i = data.index(b"\xff\xc0")
    assert inspect(lib, data[:i + 1] + b"\xc9" + data[i + 2:])[0] == _lib.ERR_UNSUPPORTED
    rotated = data[:2] + _exif(6) + data[2:]
    assert imdecode(rotated).shape == (31, 23, 3)                      # IMREAD_COLOR applies the rotation
    assert inspect(lib, rotated)[0] == _lib.ERR_UNSUPPORTED
    nojfif = _strip_app0(data)
    adobe = _segment(0xEE, b"Adobe" + bytes([0, 100, 0, 0, 0, 0, 0]))
    assert inspect(lib, nojfif[:2] + adobe + nojfif[2:])[0] == _lib.ERR_UNSUPPORTED
    # a 4-component frame (the SOF alone decides: CMYK / YCCK)
    ln = int.from_bytes(data[i + 2:i + 4], "big")
    sof = data[i + 4:i + 2 + ln]
    sof4 = sof[:5] + b"\x04" + sof[6:] + bytes([4, 0x11, 0])
    assert inspect(lib, data[:i] + _segment(0xC0, sof4) + data[i + 2 + ln:])[0] == _lib.ERR_UNSUPPORTED


def test_inspect_reports_invalid(lib):
    from faster_rcnn_b200 import _lib
    data = encode(_content(23, 31, "smooth"))
    scan = J.parse(data)["scan"]
    for n in (0, 1, 3, 4, 20, 100, scan - 1):
        assert inspect(lib, data[:n])[0] == _lib.ERR_INVALID, n
    bad = bytearray(data)
    bad[4:6] = b"\xff\xf0"                                             # APP0 length past the end of the file
    assert inspect(lib, bytes(bad))[0] == _lib.ERR_INVALID
    bad = bytearray(data)
    bad[4:6] = b"\x00\x01"                                             # length below 2
    assert inspect(lib, bytes(bad))[0] == _lib.ERR_INVALID
    i = data.index(b"\xff\xc0")
    zero = bytearray(data)
    zero[i + 5:i + 7] = b"\x00\x00"                                    # height 0
    assert inspect(lib, bytes(zero))[0] == _lib.ERR_INVALID
    j = data.index(b"\xff\xda")
    undef = bytearray(data)
    undef[j + 6] = 0x33                                                # scan references DC/AC table 3
    assert inspect(lib, bytes(undef))[0] == _lib.ERR_INVALID


def test_inspect_agrees_with_the_oracle_parser(lib):
    from faster_rcnn_b200 import _lib
    rng = np.random.default_rng(5)
    data = encode(_content(19, 27, "smooth"), "422", rst=2)
    scan = J.parse(data)["scan"]
    for _ in range(300):
        b = bytearray(data)
        for _ in range(int(rng.integers(1, 4))):
            b[int(rng.integers(2, scan))] = int(rng.integers(0, 256))
        try:
            J.parse(bytes(b))
            want = _lib.OK
        except J.Unsupported:
            want = _lib.ERR_UNSUPPORTED
        except J.Invalid:
            want = _lib.ERR_INVALID
        except Exception:
            continue
        assert inspect(lib, bytes(b))[0] == want
