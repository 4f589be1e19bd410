"""Baseline JPEG decode without a GPU: oracle/jpeg.py (the numpy restatement of libjpeg-turbo's default decode the GPU
route reproduces) against the installed Pillow bit for bit, and which files the host parser ma_jpeg_parse accepts."""
import io
import struct

import numpy as np
import PIL.Image
import pytest

from oracle import jpeg as oj

cv2 = pytest.importorskip("cv2")


def smooth(w, h, seed=0):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    base = np.stack([np.sin(x / 7 + c) * 90 + np.cos(y / 5 * c + 1) * 60 + 128 for c in range(3)], -1)
    return np.clip(base + rng.normal(0, 25, base.shape), 0, 255).astype(np.uint8)


def pil_jpeg(a, **kw):
    b = io.BytesIO()
    PIL.Image.fromarray(a).save(b, "JPEG", **kw)
    return b.getvalue()


def cv_jpeg(a, q, sampling, optimize=False, rst_interval=0):
    ok, enc = cv2.imencode(".jpg", a[:, :, ::-1], [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sampling,
                                                   cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize),
                                                   cv2.IMWRITE_JPEG_RST_INTERVAL, rst_interval])
    assert ok
    return enc.tobytes()


def pillow_rgb(data):
    return np.asarray(PIL.Image.open(io.BytesIO(data)).convert("RGB"))


SIZES = [(1, 1), (2, 1), (1, 2), (3, 3), (5, 7), (8, 8), (16, 16), (17, 9), (33, 31), (4, 9), (2, 17), (100, 70)]
OPTIONS = [{}, {"optimize": True}, {"restart_marker_blocks": 1}, {"restart_marker_rows": 1}]


@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("subsampling", [0, 1, 2])
def test_oracle_equals_pillow_pillow_encoded(w, h, subsampling):
    a = smooth(w, h, w * 131 + h)
    for q in (1, 50, 95, 100):
        for kw in OPTIONS:
            data = pil_jpeg(a, quality=q, subsampling=subsampling, **kw)
            np.testing.assert_array_equal(oj.decode(data), pillow_rgb(data), err_msg=f"q={q} {kw}")


@pytest.mark.parametrize("w,h", SIZES)
def test_oracle_equals_pillow_440_and_gray(w, h):
    a = smooth(w, h, w * 7 + h)
    for q in (1, 50, 95, 100):
        for opt, rst in ((False, 0), (True, 0), (False, 1), (True, 2 * -(-w // 8))):
            data = cv_jpeg(a, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, opt, rst)
            assert (b"\xff\xdd" in data) == (rst > 0)
            np.testing.assert_array_equal(oj.decode(data), pillow_rgb(data), err_msg=f"4:4:0 q={q} opt={opt} rst={rst}")
        for kw in OPTIONS:
            data = pil_jpeg(a[:, :, 1], quality=q, **kw)
            np.testing.assert_array_equal(oj.decode(data), pillow_rgb(data), err_msg=f"gray q={q} {kw}")


def test_oracle_equals_pillow_opencv_422():
    for w, h in SIZES:
        data = cv_jpeg(smooth(w, h, 3), 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422)
        np.testing.assert_array_equal(oj.decode(data), pillow_rgb(data))


# ------------------------------------------------------------------------------------------------ ma_jpeg_parse
def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib


def parse(data):
    import ctypes as C

    L = _lib()
    lib = L.load()
    info = L.JpegInfo()
    buf = np.frombuffer(data, np.uint8) if len(data) else np.zeros(1, np.uint8)
    rc = lib.ma_jpeg_parse(buf.ctypes.data, len(data), C.byref(info), None, 0)
    return rc, lib.ma_last_error().decode(), info


@pytest.mark.parametrize("subsampling,hv", [(0, (1, 1)), (1, (2, 1)), (2, (2, 2))])
def test_parse_accepts_baseline(subsampling, hv):
    data = pil_jpeg(smooth(37, 21), quality=90, subsampling=subsampling, restart_marker_rows=1)
    rc, msg, info = parse(data)
    assert rc == 0, msg
    assert (info.width, info.height, info.ncomp, info.h_samp, info.v_samp) == (37, 21, 3) + hv
    mcus = -(-37 // (8 * hv[0])) * -(-21 // (8 * hv[1]))
    assert info.nblocks == mcus * (hv[0] * hv[1] + 2)
    assert info.restart_interval == -(-37 // (8 * hv[0])) and info.nsegments == -(-21 // (8 * hv[1]))


def test_parse_accepts_gray_and_440():
    rc, msg, info = parse(pil_jpeg(smooth(19, 11)[:, :, 0], quality=80))
    assert rc == 0, msg
    assert (info.ncomp, info.nblocks) == (1, 3 * 2)
    rc, msg, info = parse(cv_jpeg(smooth(19, 11), 80, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440))
    assert rc == 0, msg
    assert (info.h_samp, info.v_samp) == (1, 2)


def test_parse_blob_holds_the_unstuffed_stream():
    data = pil_jpeg(smooth(64, 64), quality=100)
    j = oj.parse(data)
    from mapanything_b200.image import jpeg_parse

    info, blob = jpeg_parse(data)
    n = len(j["segs"][0])
    assert info.blob_bytes == blob.size and blob.size >= n + 16
    assert j["segs"][0] in blob.tobytes()


def _rejects(data, what):
    rc, msg, _ = parse(data)
    assert rc == -1, f"accepted {what}"
    assert msg.startswith("ma_jpeg_parse:")
    return msg


def test_parse_rejects_progressive_cmyk_and_non_baseline():
    a = smooth(40, 30)
    assert "SOF2" in _rejects(pil_jpeg(a, quality=80, progressive=True), "progressive")
    b = io.BytesIO()
    PIL.Image.fromarray(a).convert("CMYK").save(b, "JPEG", quality=80)
    _rejects(b.getvalue(), "CMYK")
    base = pil_jpeg(a, quality=80)
    i = base.index(b"\xff\xc0")
    _rejects(base[:i] + b"\xff\xc9" + base[i + 2:], "SOF9 arithmetic")
    twelve = bytearray(base)
    twelve[i + 4] = 12
    assert "12-bit" in _rejects(bytes(twelve), "12-bit")
    adobe = base[:2] + b"\xff\xee\x00\x0eAdobe\x00\x64\x00\x00\x00\x00\x00" + base[2:]
    jfif_free = adobe[:2] + adobe[2:].replace(b"JFIF\x00", b"JFXX\x00", 1)
    assert "YCbCr" in _rejects(jfif_free, "Adobe transform 0")


def test_parse_rejects_truncated_and_bad_tables():
    base = pil_jpeg(smooth(40, 30), quality=80)
    for cut in (0, 1, 3, 20, 200, len(base) // 2, len(base) - 2):
        _rejects(base[:cut], f"truncated at {cut}")
    i = base.index(b"\xff\xc4")
    bad = bytearray(base)
    bad[i + 5:i + 5 + 16] = bytes([2, 2, 2] + [0] * 13)   # 2 + 2 + 2 codes of length 1..3: all-ones code at length 1..2
    assert "prefix code" in _rejects(bytes(bad), "over-full Huffman table")
    bad = bytearray(base)
    bad[i + 4] = 0x05   # table index 5
    _rejects(bytes(bad), "Huffman table index 5")
    j = base.index(b"\xff\xdb")
    bad = bytearray(base)
    bad[j + 4] = 0x07   # quantisation table 7
    _rejects(bytes(bad), "quantisation table index 7")
    k = base.index(b"\xff\xda")
    bad = bytearray(base)
    bad[k + 4] = 1      # scan with one of three components
    assert "cover" in _rejects(bytes(bad), "partial scan")


def _dht(n_len1):
    """A DHT segment (DC table 0) with n_len1 codes of length 1: over-full from the second code on."""
    body = bytes([0x00, n_len1] + [0] * 15) + bytes(n_len1)
    return b"\xff\xc4" + (2 + len(body)).to_bytes(2, "big") + body


@pytest.mark.parametrize("n_len1", [2, 3, 16, 255])
def test_parse_rejects_over_full_huffman_table(n_len1):
    base = pil_jpeg(smooth(40, 30), quality=80)
    assert "prefix code" in _rejects(base[:2] + _dht(n_len1) + base[2:], f"{n_len1} codes of length 1")
    assert parse(base)[0] == 0   # the parser's tables are intact afterwards


def test_parse_short_jfif_app0_does_not_make_rgb_ids_ycbcr():
    """libjpeg-turbo takes a JFIF APP0 into account only with at least 14 data bytes (examine_app0); with 'R', 'G', 'B'
    component ids and no valid JFIF marker the frame is RGB, which the GPU route does not decode."""
    base = pil_jpeg(smooth(40, 30), quality=80)
    i = base.index(b"\xff\xc0")
    rgb = bytearray(base)
    for c, cid in enumerate(b"RGB"):
        rgb[i + 10 + 3 * c] = cid
    k = base.index(b"\xff\xda")
    for c, cid in enumerate(b"RGB"):
        rgb[k + 5 + 2 * c] = cid
    assert parse(bytes(rgb))[0] == 0                  # full JFIF APP0: YCbCr whatever the ids
    app0 = base.index(b"\xff\xe0")
    n = int.from_bytes(base[app0 + 2:app0 + 4], "big")
    short = bytes(rgb[:app0]) + b"\xff\xe0\x00\x0eJFIF\x00\x01\x01\x00\x00\x01\x00\x01" + bytes(rgb[app0 + 2 + n:])
    assert "YCbCr" in _rejects(short, "12-byte JFIF APP0 with R, G, B ids")


def test_parse_blob_capacity_one_pass_and_retry():
    """The blob is the same whether the file is parsed once into a roomy buffer or again into one of the exact size;
    a capacity below the blob's size fills the info and is refused."""
    import ctypes as C

    from mapanything_b200.image import jpeg_parse

    lib = _lib().load()
    for data in (pil_jpeg(smooth(300, 200), quality=95),
                 pil_jpeg(smooth(1600, 1600), quality=1, subsampling=0, restart_marker_blocks=1)):  # tables > file
        info, blob = jpeg_parse(data)
        buf = np.frombuffer(data, np.uint8)
        exact = np.empty(info.blob_bytes, np.uint8)
        info2 = _lib().JpegInfo()
        assert lib.ma_jpeg_parse(buf.ctypes.data, buf.size, C.byref(info2), exact.ctypes.data, exact.size - 1) == -1
        assert info2.blob_bytes == info.blob_bytes and "blob_capacity" in lib.ma_last_error().decode()
        assert lib.ma_jpeg_parse(buf.ctypes.data, buf.size, C.byref(info2), exact.ctypes.data, exact.size) == 0
        np.testing.assert_array_equal(blob, exact)
    assert info.blob_bytes > len(data) * 1.5 + (1 << 16)


def test_parse_rejects_bad_arguments():
    import ctypes as C

    L = _lib()
    lib = L.load()
    info = L.JpegInfo()
    data = np.frombuffer(pil_jpeg(smooth(8, 8), quality=50), np.uint8)
    assert lib.ma_jpeg_parse(None, data.size, C.byref(info), None, 0) == -1
    assert lib.ma_jpeg_parse(data.ctypes.data, data.size, None, None, 0) == -1
    assert lib.ma_jpeg_parse(data.ctypes.data, -1, C.byref(info), None, 0) == -1
    assert lib.ma_jpeg_parse(data.ctypes.data, data.size, C.byref(info), None, 0) == 0
    small = np.empty(int(info.blob_bytes) - 1, np.uint8)
    assert lib.ma_jpeg_parse(data.ctypes.data, data.size, C.byref(info), small.ctypes.data, small.size) == -1
    assert "blob_capacity" in lib.ma_last_error().decode()
    ws = C.c_int64(0)
    assert lib.ma_jpeg_workspace(C.byref(info), 1, C.byref(ws)) == 0 and ws.value > 0
    assert lib.ma_jpeg_workspace(None, 1, C.byref(ws)) == -1
