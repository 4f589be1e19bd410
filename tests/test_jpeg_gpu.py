"""GPU JPEG decoding (csrc/jpeg.cu through ma_jpeg_decode and load_images): every frame the decoder reports as decoded
must equal np.asarray(exif_transpose(PIL.Image.open(f)).convert("RGB")) byte for byte."""
import ctypes as C
import io

import numpy as np
import PIL.Image
import pytest
import torch
from PIL.ImageOps import exif_transpose

from test_jpeg_cpu import cv_jpeg, pil_jpeg, smooth

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def pillow_rgb(data):
    return np.asarray(exif_transpose(PIL.Image.open(io.BytesIO(data))).convert("RGB"))


def gpu_decode(files, orientations=None):
    """[bytes] -> [(status, (H', W', 3) uint8 array)] from ONE ma_jpeg_decode call over all files."""
    from mapanything_b200 import _lib
    from mapanything_b200.image import jpeg_parse

    lib = _lib.load()
    orientations = orientations or [1] * len(files)
    parsed = [jpeg_parse(f) for f in files]
    assert all(p is not None for p in parsed)
    n = len(files)
    offs = np.cumsum([0] + [p[1].size for p in parsed])
    cat = np.concatenate([p[1] for p in parsed])
    d_blobs = torch.from_numpy(cat).cuda()
    infos = (_lib.JpegInfo * n)(*[p[0] for p in parsed])
    outs = []
    for (info, _), o in zip(parsed, orientations):
        W, H = (info.height, info.width) if o >= 5 else (info.width, info.height)
        outs.append(torch.full((H, W, 3), 77, dtype=torch.uint8, device="cuda"))
    ws = C.c_int64(0)
    assert lib.ma_jpeg_workspace(infos, n, C.byref(ws)) == 0
    work = torch.empty(ws.value, dtype=torch.uint8, device="cuda")
    status = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    rc = lib.ma_jpeg_decode(d_blobs.data_ptr(), (C.c_int64 * n)(*[int(x) for x in offs[:-1]]), infos, n,
                            (C.c_void_p * n)(*[t.data_ptr() for t in outs]), (C.c_int32 * n)(*orientations),
                            work.data_ptr(), ws.value, status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.ma_last_error().decode()
    torch.cuda.synchronize()
    return list(zip(status.cpu().tolist(), [t.cpu().numpy() for t in outs]))


def check_all(files, orientations=None, what=""):
    res = gpu_decode(files, orientations)
    for i, (f, (st, got)) in enumerate(zip(files, res)):
        assert st == 0, f"{what} frame {i}: status {st}"
        ref = pillow_rgb(f)
        assert got.shape == ref.shape, f"{what} frame {i}"
        if not np.array_equal(got, ref):
            bad = np.argwhere((got != ref).any(-1))
            pytest.fail(f"{what} frame {i} {ref.shape}: {len(bad)} pixels differ, first {bad[:4].tolist()}")


SMALL = [(1, 1), (2, 2), (3, 1), (7, 5), (16, 8), (17, 9), (31, 33), (100, 70), (333, 211)]
LAYOUTS = ["444", "422", "420", "440", "gray"]


def encode(a, layout, q, optimize=False, restart=None):
    kw = {"quality": q, "optimize": optimize}
    if restart == "mcu":
        kw["restart_marker_blocks"] = 1
    elif restart == "rows":
        kw["restart_marker_rows"] = 3
    if layout == "gray":
        return pil_jpeg(a[:, :, 0], **kw)
    if layout == "440":   # 4:4:0 MCUs are 8 x 16: "rows" = 3 MCU rows
        rst = {None: 0, "mcu": 1, "rows": 3 * -(-a.shape[1] // 8)}[restart]
        return cv_jpeg(a, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, optimize, rst)
    return pil_jpeg(a, subsampling={"444": 0, "422": 1, "420": 2}[layout], **kw)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("restart", [None, "mcu", "rows"])
def test_small_frames_match_pillow(layout, restart):
    files = []
    for w, h in SMALL:
        a = smooth(w, h, w + 3 * h)
        for q in (5, 75, 95, 100):
            for opt in (False, True):
                try:
                    files.append(encode(a, layout, q, opt, restart))
                except OSError:   # Pillow's encoder refuses some optimised 4:4:4 frames written to memory
                    assert opt
    check_all(files, what=f"{layout} restart={restart}")   # one mixed-size batch


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("W,H", [(1920, 1080), (4032, 3024)])
def test_camera_frames_match_pillow(layout, W, H):
    a = smooth(W, H, 11)
    files = [encode(a, layout, 95), encode(a, layout, 75, True, "rows")]
    check_all(files, what=f"{layout} {W}x{H}")


def test_high_entropy_12mp_q100_syncs():
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, (3024, 4032, 3), dtype=np.uint8)
    f = pil_jpeg(a, quality=100, subsampling=0)
    assert len(f) > 20 << 20
    check_all([f], what="noise q100")


def with_orientation(data, o):
    im = PIL.Image.open(io.BytesIO(data))
    exif = PIL.Image.Exif()
    exif[0x0112] = o
    b = io.BytesIO()
    im.save(b, "JPEG", quality=100, subsampling=0, exif=exif.tobytes())
    return b.getvalue()


@pytest.mark.parametrize("layout", ["444", "420", "gray"])
def test_exif_orientations_match_exif_transpose(layout):
    from mapanything_b200.image import _open_for_gpu

    files, orients = [], []
    for w, h in [(37, 21), (64, 48)]:
        for o in range(1, 9):
            b = io.BytesIO()
            src = smooth(w, h, o)
            exif = PIL.Image.Exif()
            exif[0x0112] = o
            img = PIL.Image.fromarray(src[:, :, 0] if layout == "gray" else src)
            kw = {} if layout == "gray" else {"subsampling": {"444": 0, "420": 2}[layout]}
            img.save(b, "JPEG", quality=90, exif=exif.tobytes(), **kw)
            files.append(b.getvalue())
            orients.append(o)
    import tempfile, os
    with tempfile.TemporaryDirectory() as d:
        for i, f in enumerate(files):
            p = os.path.join(d, f"{i}.jpg")
            open(p, "wb").write(f)
            assert _open_for_gpu(p)[2] == orients[i]
    check_all(files, orients, what=f"orientation {layout}")


def test_flipped_bytes_flagged_or_equal():
    rng = np.random.default_rng(9)
    base = [encode(smooth(w, h, 1), lay, 90, restart=r) for (w, h) in [(64, 48), (333, 211)] for lay in ("420", "444", "gray")
            for r in (None, "rows")]
    from mapanything_b200.image import jpeg_parse

    files = []
    for f in base:
        sos = f.index(b"\xff\xda")
        for _ in range(6):
            g = bytearray(f)
            for _ in range(rng.integers(1, 4)):
                k = int(rng.integers(sos + 20, len(g) - 2))
                g[k] ^= 1 << int(rng.integers(0, 8))
            if jpeg_parse(bytes(g), with_blob=False) is not None:
                files.append(bytes(g))
    assert len(files) > 20
    res = gpu_decode(files)
    flagged = 0
    for f, (st, got) in zip(files, res):
        try:
            ref = pillow_rgb(f)
        except Exception:  # noqa: BLE001  (Pillow refuses it: the GPU route must not accept it)
            assert st != 0
            flagged += 1
            continue
        if st != 0:
            flagged += 1
        else:
            np.testing.assert_array_equal(got, ref)
    print(f"{flagged} of {len(files)} corrupted frames flagged")


def test_load_images_mixed_folder_routes(tmp_path):
    from mapanything_b200 import ops
    from mapanything_b200.image import load_images
    from oracle import image as OI

    a = smooth(300, 200, 4)
    n_gpu = 0
    for i, (lay, q) in enumerate([("420", 95), ("444", 90), ("422", 75), ("gray", 80), ("440", 95)]):
        (tmp_path / f"g{i}.jpg").write_bytes(encode(a, lay, q))
        n_gpu += 1
    (tmp_path / "r0.jpg").write_bytes(with_orientation(encode(a, "420", 95), 6))
    n_gpu += 1
    (tmp_path / "p0.jpg").write_bytes(pil_jpeg(a, quality=90, progressive=True))
    b = io.BytesIO()
    PIL.Image.fromarray(a).convert("CMYK").save(b, "JPEG", quality=90)
    (tmp_path / "c0.jpg").write_bytes(b.getvalue())
    PIL.Image.fromarray(smooth(200, 300, 6)).save(tmp_path / "n0.png")
    before = dict(ops.JPEG_ROUTES)
    views = load_images(str(tmp_path))
    ref = OI.load_images(str(tmp_path))
    assert len(views) == len(ref)
    for v, r in zip(views, ref):
        assert torch.equal(v["img"].cpu(), r["img"])
        np.testing.assert_array_equal(v["true_shape"], r["true_shape"])
    assert ops.JPEG_ROUTES["gpu"] - before["gpu"] == n_gpu
    assert ops.JPEG_ROUTES["pillow"] - before["pillow"] == 3
