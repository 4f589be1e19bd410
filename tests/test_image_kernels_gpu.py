"""Every kernel of csrc/image.cu, called through the C ABI, bit for bit against Pillow's integer arithmetic.

References
- Resampling (both passes): the arithmetic of oracle/image.py (Pillow's Resample.c) over exactly the sub-range the call asks
  for, with the tables of ma_resample_coeffs (pinned to Pillow by test_image_cpu.py): accumulate in int64 from 1 << 21,
  shift right by 22, clamp to a byte.  The restatement is checked against PIL.Image.resize once, on a full image.
- Normalisation: torch fp32 (u.float() / 255 - mean) / std, torchvision's rounding order.
- Depth gather: cv2.resize(INTER_NEAREST) and the crop, with the offsets of image._nearest_indices.
- Image conversion: the reference's expression (img * 255).clamp(0, 255).byte() or img.clamp(0, 255).byte(), on the same
  CUDA tensor and on its CPU copy.

Every output byte and every fp32 output bit is compared (fp32 through an int32 view).  Output buffers are pre-filled with
a sentinel and have margins on both sides; every element the call must not write must still hold it.  Source pixels outside
the rows and columns a call may read hold a value other than those inside, and source row / frame padding holds another.

Horizontal pass: each case asserts, with ma_last_resample_kernel(), which form and instantiation it ran -- every dp4a
instantiation (NW4 = 1 .. 16, packed coefficients passed), every word-load instantiation (KMAX = 4 .. 64, packed = NULL) and
the byte-load form (above 64 taps), each once with a staged row below 48 KB of shared memory and once above it.  Odd window
lengths reach every bucket: ksize = 4 NW4 - 1 or 4 NW4 - 3 (identity for NW4 = 1), from LANCZOS or BICUBIC downscaling or
BICUBIC enlargement.  test_every_horizontal_instantiation_ran, last in the file, checks that the whole set was reached.
"""
import ctypes as C
import functools
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

LANCZOS, BICUBIC = 1, 3
BIAS, SHIFT = 1 << 21, 22
SENT = 0xA7            # byte sentinel of the u8 outputs
FSENT = -77.0          # fp32 sentinel of out_chw / the gather output
OUTSIDE = 0x5A         # source pixels the call must not read
PAD = 0xE1             # source row / frame padding
MARGIN = 64            # sentinel bytes (u8) or elements (fp32) before and after each output
LARGE_SPAN = 17100     # staged pixels: above 48 KB of shared memory in every form
SMALL_SPAN_MAX = 11000  # staged pixels: below 48 KB in every form
DP4A, VEC, BYTE = "dp4a", "vec", "byte"


def _lib():
    from mapanything_b200 import _lib

    return _lib.load()


def _check(rc, what):
    from mapanything_b200._lib import check

    check(rc, what)


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------ tables
class Table:
    """Pillow's windows of one axis (ma_resample_coeffs / ma_resample_pack_coeffs) on the host and on `device`."""

    def __init__(self, in_size, out_size, filt, device):
        lib = _lib()
        ks = C.c_int(0)
        _check(lib.ma_resample_coeffs(in_size, out_size, filt, C.byref(ks), None, None), "ma_resample_coeffs")
        self.in_size, self.out_size, self.filt, self.ksize = in_size, out_size, filt, ks.value
        self.bounds = np.zeros((out_size, 2), np.int32)
        self.coeffs = np.zeros((self.ksize, out_size), np.int32)
        _check(lib.ma_resample_coeffs(in_size, out_size, filt, C.byref(ks), self.bounds.ctypes.data, self.coeffs.ctypes.data),
               "ma_resample_coeffs")
        packed = np.zeros((3, (self.ksize + 3) // 4, out_size), np.uint32)
        _check(lib.ma_resample_pack_coeffs(self.coeffs.ctypes.data, self.ksize, out_size, packed.ctypes.data),
               "ma_resample_pack_coeffs")
        self.d_bounds = torch.from_numpy(self.bounds).to(device)
        self.d_coeffs = torch.from_numpy(self.coeffs).to(device)
        self.d_packed = torch.from_numpy(packed.view(np.int32)).to(device)

    def span(self, x0, cols):
        """Source columns [sx0, sx1) the windows of outputs [x0, x0 + cols) cover."""
        b = self.bounds[x0:x0 + cols]
        return int(b[:, 0].min()), int((b[:, 0] + b[:, 1]).max())


@functools.lru_cache(maxsize=None)
def table(in_size, out_size, filt, device="cuda"):
    return Table(in_size, out_size, filt, device)


def _ksize(in_size, out_size, filt):
    ks = C.c_int(0)
    _check(_lib().ma_resample_coeffs(in_size, out_size, filt, C.byref(ks), None, None), "ma_resample_coeffs")
    return ks.value


def sizes_for(ksize, filt, out_size, odd_in=False):
    """(in_size, out_size) whose table for `filt` has `ksize` taps: ksize = 2 ceil(support * max(in / out, 1)) + 1."""
    if ksize == 1:
        return out_size, out_size
    support = 3.0 if filt == LANCZOS else 2.0
    c = (ksize - 1) // 2
    s = (c - 0.5) / support  # middle of the ratios that give c; below 1 means enlarging (5 / 7 taps)
    guess = s * out_size
    for in_size in sorted(range(max(1, int(guess) - 8), int(guess) + 9), key=lambda v: abs(v - guess)):
        if (not odd_in or in_size % 2 == 1) and in_size != out_size and _ksize(in_size, out_size, filt) == ksize:
            return in_size, out_size
    raise AssertionError(f"no table of {ksize} taps for {out_size} outputs")


# ------------------------------------------------------------------------------------------------ references
def ref_h(src, y0, rows, tab, x0, cols):
    """Horizontal pass of Pillow over source rows [y0, y0 + rows) and output columns [x0, x0 + cols) of src (n, H, W, 3) u8:
    (bytes (n, rows, cols, 3), unclamped accumulators >> 22)."""
    first = tab.bounds[x0:x0 + cols, 0].astype(np.int64)
    cnt = tab.bounds[x0:x0 + cols, 1]
    k = tab.coeffs[:, x0:x0 + cols].astype(np.int64)
    rowsrc = src[:, y0:y0 + rows].astype(np.int64)
    acc = np.full((src.shape[0], rows, cols, 3), BIAS, np.int64)
    for t in range(int(cnt.max())):
        live = t < cnt
        acc += rowsrc[:, :, np.where(live, first + t, first), :] * np.where(live, k[t], 0)[None, None, :, None]
    v = acc >> SHIFT
    return np.clip(v, 0, 255).astype(np.uint8), v


def ref_v(tmp, y0, tab, top, th):
    """Vertical pass over tmp (n, rows, cols, 3), whose row 0 is source row y0: output rows [top, top + th)."""
    first = tab.bounds[top:top + th, 0].astype(np.int64) - y0
    cnt = tab.bounds[top:top + th, 1]
    k = tab.coeffs[:, top:top + th].astype(np.int64)
    t8 = tmp.astype(np.int64)
    acc = np.full((tmp.shape[0], th, tmp.shape[2], 3), BIAS, np.int64)
    for t in range(int(cnt.max())):
        live = t < cnt
        acc += t8[:, np.where(live, first + t, first)] * np.where(live, k[t], 0)[None, :, None, None]
    return np.clip(acc >> SHIFT, 0, 255).astype(np.uint8)


def ref_normalize(u8, mean, std):
    """torchvision ToTensor + Normalize in fp32: (n, th, cols, 3) u8 -> (n, 3, th, cols)."""
    u = torch.from_numpy(u8).permute(0, 3, 1, 2).float()
    m = torch.tensor(mean, dtype=torch.float32).view(1, 3, 1, 1)
    s = torch.tensor(std, dtype=torch.float32).view(1, 3, 1, 1)
    return (u / 255 - m) / s


def test_reference_matches_pillow():
    """ref_h (and ref_v through the transpose) against PIL.Image.resize on full images, and against oracle/image.py."""
    import PIL.Image

    from oracle import image as OI

    rng = np.random.default_rng(5)
    for (W, H), (ow, oh), filt in [((1001, 7), (273, 7), LANCZOS), ((97, 5), (140, 5), BICUBIC), ((9, 611), (9, 100), LANCZOS)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        want = np.asarray(PIL.Image.fromarray(img).resize((ow, oh), resample=filt))
        if ow != W:
            got = ref_h(img[None], 0, H, table(W, ow, filt), 0, ow)[0][0]
            assert np.array_equal(got, OI.pil_resize_u8(img, (ow, oh), filt))
        else:
            got = ref_v(img[None], 0, table(H, oh, filt), 0, oh)[0]
        assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ horizontal pass
SEEN = set()  # (ma_last_resample_kernel(), "small" / "large") of every matrix case that ran


def fence(img, y0, rows, sx0, sx1):
    """img with every pixel outside rows [y0, y0 + rows) x columns [sx0, sx1) set to OUTSIDE."""
    out = np.full_like(img, OUTSIDE)
    out[:, y0:y0 + rows, sx0:sx1] = img[:, y0:y0 + rows, sx0:sx1]
    return out


def run_h(src, *, y0, rows, sx0, sx1, tab, x0, cols, packed=True, ptr_off=0, row_pad=0, frame_pad=0, device="cuda"):
    """Lays src (n, H, W, 3) u8 out on the device -- row stride 3 W + row_pad, frame stride H (3 W + row_pad) + frame_pad,
    first byte at ptr_off past a 16-byte aligned address, padding bytes PAD -- runs ma_resample_h_u8rgb into a
    sentinel-filled buffer and returns (bytes (n, rows, cols, 3), ma_last_resample_kernel(), staged-row misalignments)."""
    n, H, W, _ = src.shape
    rs = 3 * W + row_pad
    fs = H * rs + frame_pad
    host = np.full(ptr_off + n * fs + 64, PAD, np.uint8)
    np.lib.stride_tricks.as_strided(host[ptr_off:], shape=(n, H, 3 * W), strides=(fs, rs, 1))[...] = src.reshape(n, H, 3 * W)
    d_src = torch.from_numpy(host).to(device)
    assert d_src.data_ptr() % 16 == 0
    size = n * rows * cols * 3
    tmp = torch.full((size + 2 * MARGIN,), SENT, dtype=torch.uint8, device=device)
    lib = _lib()
    _check(lib.ma_resample_h_u8rgb(d_src.data_ptr() + ptr_off, rs, fs, n, y0, rows, sx0, sx1, tab.d_bounds.data_ptr(),
                                   tab.d_coeffs.data_ptr(), tab.d_packed.data_ptr() if packed else None, tab.ksize,
                                   tab.out_size, x0, cols, tmp.data_ptr() + MARGIN, _stream()), "ma_resample_h_u8rgb")
    code = lib.ma_last_resample_kernel()
    out = tmp.cpu().numpy()
    assert (out[:MARGIN] == SENT).all() and (out[MARGIN + size:] == SENT).all(), "wrote outside tmp"
    mis = {(d_src.data_ptr() + ptr_off + f * fs + (y0 + r) * rs + 3 * sx0) % 4 for f in range(n) for r in range(rows)}
    return out[MARGIN:MARGIN + size].reshape(n, rows, cols, 3), code, mis


def expected_code(form, ksize):
    nw = (ksize + 3) // 4
    return {DP4A: 2000 + nw, VEC: 1000 + 4 * nw, BYTE: 1}[form]


def form_case(form, ksize, filt, large, odd_in=False):
    """(Table, x0, cols) for a `ksize`-tap window whose staged span is above (large) or below 48 KB; x0 > 0, cols < out_size."""
    if not large:
        out_size = 97
    else:
        ratio = table(*sizes_for(ksize, filt, 1000), filt).in_size / 1000
        out_size = math.ceil(LARGE_SPAN / ratio) + 16
    tab = table(*sizes_for(ksize, filt, out_size, odd_in), filt)
    x0 = 3 if not large else 5
    return tab, x0, out_size - x0 - 4


def _matrix():
    cases = []
    for nw in range(1, 17):
        for large in (False, True):
            # alternate the two odd window lengths of the bucket and the two filters
            if nw == 1:
                ksize, filt = 1, LANCZOS  # identity
            else:  # nw = 2: BICUBIC and LANCZOS enlargement
                ksize = 4 * nw - 1 if large else 4 * nw - 3
                filt = LANCZOS if (nw + large) % 2 else BICUBIC
            for form in (DP4A, VEC):
                cases.append(pytest.param(form, ksize, filt, large, id=f"{form}-{4 * nw if form == VEC else nw}-k{ksize}-"
                                                                       f"{'large' if large else 'small'}"))
    for ksize, filt in ((67, LANCZOS), (129, BICUBIC), (233, LANCZOS)):
        for large in (False, True):
            cases.append(pytest.param(BYTE, ksize, filt, large, id=f"byte-k{ksize}-{'large' if large else 'small'}"))
    return cases


@pytest.mark.parametrize("form,ksize,filt,large", _matrix())
def test_horizontal_instantiation(form, ksize, filt, large):
    tab, x0, cols = form_case(form, ksize, filt, large)
    assert tab.ksize == ksize and 0 < x0 and x0 + cols < tab.out_size
    sx0, sx1 = tab.span(x0, cols)
    span = sx1 - sx0
    assert span >= 17000 if large else span <= SMALL_SPAN_MAX
    n, H, y0, rows = 1, 4, 1, 2
    rng = np.random.default_rng(ksize * 7 + large)
    src = fence(rng.integers(0, 256, (n, H, tab.in_size, 3), dtype=np.uint8), y0, rows, sx0, sx1)
    got, code, _ = run_h(src, y0=y0, rows=rows, sx0=sx0, sx1=sx1, tab=tab, x0=x0, cols=cols, packed=form != VEC)
    assert code == expected_code(form, ksize), f"ran {code}"
    want, _ = ref_h(src, y0, rows, tab, x0, cols)
    assert np.array_equal(got, want), f"{int((got != want).sum())} bytes differ"
    SEEN.add((code, "large" if large else "small"))


# Staged span (pixels) on both sides of each dispatch threshold, with packed coefficients and a 13-tap window.
@pytest.mark.parametrize("span,form", [(61098, DP4A), (61099, VEC), (68096, VEC), (68097, BYTE), (68264, BYTE)])
def test_dispatch_threshold(span, form):
    tab = table(68300, 34150, LANCZOS)
    assert tab.ksize == 13
    x0 = 7
    sx0 = tab.span(x0, 1)[0]
    cols = int(np.searchsorted((tab.bounds[:, 0] + tab.bounds[:, 1])[x0:], sx0 + span, side="right"))
    sx1 = sx0 + span  # the staged span reaches past the last window (unused pixels, still staged)
    assert tab.span(x0, cols)[1] <= sx1 <= tab.in_size
    rng = np.random.default_rng(span)
    src = fence(rng.integers(0, 256, (1, 1, tab.in_size, 3), dtype=np.uint8), 0, 1, sx0, sx1)
    got, code, _ = run_h(src, y0=0, rows=1, sx0=sx0, sx1=sx1, tab=tab, x0=x0, cols=cols, ptr_off=span % 4)
    assert code == expected_code(form, 13), f"ran {code}"
    assert np.array_equal(got, ref_h(src, 0, 1, tab, x0, cols)[0])


def test_span_above_shared_memory_is_refused():
    lib = _lib()
    tab = table(68300, 34150, LANCZOS)
    src = torch.zeros(68300 * 3, dtype=torch.uint8, device="cuda")
    tmp = torch.full((100 * 3,), SENT, dtype=torch.uint8, device="cuda")
    rc = lib.ma_resample_h_u8rgb(src.data_ptr(), 68300 * 3, 68300 * 3, 1, 0, 1, 0, 68265, tab.d_bounds.data_ptr(),
                                 tab.d_coeffs.data_ptr(), tab.d_packed.data_ptr(), tab.ksize, tab.out_size, 0, 100,
                                 tmp.data_ptr(), _stream())
    assert rc == -1 and "68265 pixels do not fit shared memory" in lib.ma_last_error().decode()
    torch.cuda.synchronize()
    assert (tmp == SENT).all()


def test_second_device_after_first():
    """The large-shared-memory opt-in is cached per device: a launch above 48 KB on device 1 after device 0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for dev in (0, 1):
        with torch.cuda.device(dev):
            tab = table(*sizes_for(25, LANCZOS, 4700), LANCZOS, device=f"cuda:{dev}")
            x0, cols = 2, 4690
            sx0, sx1 = tab.span(x0, cols)
            assert sx1 - sx0 >= 17000
            src = fence(np.random.default_rng(dev).integers(0, 256, (1, 2, tab.in_size, 3), dtype=np.uint8), 0, 2, sx0, sx1)
            got, code, _ = run_h(src, y0=0, rows=2, sx0=sx0, sx1=sx1, tab=tab, x0=x0, cols=cols, device=f"cuda:{dev}")
            assert code == expected_code(DP4A, 25)
            assert np.array_equal(got, ref_h(src, 0, 2, tab, x0, cols)[0])


# Geometry: pointer offset 0-3 (with odd widths and odd row strides every frame row has its own staged-row misalignment),
# y0 > 0, rows < H, padded row and frame strides, n up to 5, x0 > 0, and a staged span wider than the windows need.
GEOMETRY = [  # ptr_off, n, y0, rows, extra rows, row_pad, frame_pad, x0, cols short of out_size, widen left, widen right
    (0, 1, 0, 4, 0, 0, 0, 0, 0, 0, 0),
    (1, 3, 1, 4, 1, 2, 5, 5, 3, 0, 1),
    (2, 4, 3, 5, 2, 6, 13, 17, 9, 2, 0),
    (3, 5, 5, 4, 3, 66, 1001, 40, 1, 7, 5),
]
GEOMETRY_FORMS = [(DP4A, 25, LANCZOS), (DP4A, 5, BICUBIC), (VEC, 25, LANCZOS), (VEC, 63, BICUBIC), (BYTE, 71, LANCZOS)]


@pytest.mark.parametrize("form,ksize,filt", GEOMETRY_FORMS, ids=[f"{f}-k{k}" for f, k, _ in GEOMETRY_FORMS])
@pytest.mark.parametrize("geom", GEOMETRY, ids=[f"off{g[0]}-n{g[1]}" for g in GEOMETRY])
def test_horizontal_geometry(form, ksize, filt, geom):
    ptr_off, n, y0, rows, extra, row_pad, frame_pad, x0, short, wl, wr = geom
    tab = table(*sizes_for(ksize, filt, 151, odd_in=True), filt)
    assert tab.in_size % 2 == 1
    cols = tab.out_size - x0 - short
    sx0, sx1 = tab.span(x0, cols)
    sx0, sx1 = max(sx0 - wl, 0), min(sx1 + wr, tab.in_size)
    H = y0 + rows + extra
    rng = np.random.default_rng(ptr_off * 100 + ksize)
    src = fence(rng.integers(0, 256, (n, H, tab.in_size, 3), dtype=np.uint8), y0, rows, sx0, sx1)
    got, code, mis = run_h(src, y0=y0, rows=rows, sx0=sx0, sx1=sx1, tab=tab, x0=x0, cols=cols, packed=form != VEC,
                           ptr_off=ptr_off, row_pad=row_pad, frame_pad=frame_pad)
    assert code == expected_code(form, ksize)
    assert mis == {0, 1, 2, 3}
    want, _ = ref_h(src, y0, rows, tab, x0, cols)
    assert np.array_equal(got, want), f"{int((got != want).sum())} bytes differ"


def _pattern(name, tab, x0, cols, H, rng):
    W = tab.in_size
    if name == "random":
        return rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)
    if name in ("zeros", "full"):
        return np.full((1, H, W, 3), 0 if name == "zeros" else 255, np.uint8)
    # "clamps": row 0 sets the pixels under the positive taps of every few output columns (disjoint windows) to 255 and the
    # rest to 0, row 1 those under the negative taps: the accumulator goes above 255 and below 0.  Rows 2 and 3 hold binary
    # noise from {0, 255}; rows 4-7 square waves with periods of 2, 1.8, 2 and 2.2 output pixels (source pixels when
    # enlarging), near the spacing of the LANCZOS / BICUBIC lobes, each at its own phase.
    img = np.zeros((1, H, W, 3), np.uint8)
    ratio = W / tab.out_size
    step = math.ceil(tab.ksize / ratio) + 1
    for xx in range(x0, x0 + cols, step):
        first, cnt = tab.bounds[xx]
        k = tab.coeffs[:cnt, xx]
        img[0, 0, first:first + cnt] = np.where(k > 0, 255, 0)[:, None]
        img[0, 1, first:first + cnt] = np.where(k < 0, 255, 0)[:, None]
    img[0, 2:4] = rng.integers(0, 2, (2, W, 3)).astype(np.uint8) * 255
    x = np.arange(W)
    for r, period in zip(range(4, 8), (2.0, 1.8, 2.0, 2.2)):
        img[0, r] = (((x + r) / (period * max(ratio, 1.0) / 2)).astype(np.int64) % 2 * 255)[:, None].astype(np.uint8)
    return img


PATTERN_FORMS = [(DP4A, 25, LANCZOS), (DP4A, 5, BICUBIC), (VEC, 13, BICUBIC), (VEC, 49, LANCZOS), (BYTE, 71, LANCZOS),
                 (BYTE, 129, BICUBIC)]


@pytest.mark.parametrize("pattern", ["random", "zeros", "full", "clamps"])
@pytest.mark.parametrize("form,ksize,filt", PATTERN_FORMS, ids=[f"{f}-k{k}" for f, k, _ in PATTERN_FORMS])
def test_horizontal_pixel_patterns(form, ksize, filt, pattern):
    tab = table(*sizes_for(ksize, filt, 211), filt)
    x0, cols = 6, tab.out_size - 10
    sx0, sx1 = tab.span(x0, cols)
    H, y0, rows = 10, 1, 8
    rng = np.random.default_rng(ksize)
    img = _pattern(pattern, tab, x0, cols, rows, rng)
    src = np.full((1, H, tab.in_size, 3), 255 - int(img[0, 0, sx0, 0]) if pattern in ("zeros", "full") else OUTSIDE, np.uint8)
    src[:, y0:y0 + rows, sx0:sx1] = img[:, :, sx0:sx1]
    got, code, _ = run_h(src, y0=y0, rows=rows, sx0=sx0, sx1=sx1, tab=tab, x0=x0, cols=cols, packed=form != VEC, ptr_off=1)
    assert code == expected_code(form, ksize)
    want, acc = ref_h(src, y0, rows, tab, x0, cols)
    assert np.array_equal(got, want), f"{int((got != want).sum())} bytes differ"
    if pattern == "clamps":
        assert (acc < 0).any() and (acc > 255).any(), "the pattern reached neither or only one clamp"
        assert (acc[:, 0] > 255).any() and (acc[:, 1] < 0).any()


# ------------------------------------------------------------------------------------------------ vertical pass
V_TAPS = [(1, LANCZOS), (5, BICUBIC), (13, LANCZOS), (71, LANCZOS), (129, BICUBIC)]
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def run_v(tmp, y0, tab, top, th, want_chw, want_u8, mean=MEAN, std=STD, frame_rows=None):
    """tmp (n, rows, cols, 3) u8 -> (out_chw (n, 3, th, cols) fp32 or None, out_u8 (n, th, cols, 3) or None); frame_rows >=
    rows pads every tmp frame with PAD rows the call must not read."""
    n, rows, cols, _ = tmp.shape
    frame_rows = rows if frame_rows is None else frame_rows
    host = np.full((n, frame_rows, cols, 3), PAD, np.uint8)
    host[:, :rows] = tmp
    d_tmp = torch.from_numpy(host).cuda()
    chw = torch.full((n * 3 * th * cols + 2 * MARGIN,), FSENT, device="cuda") if want_chw else None
    u8 = torch.full((n * th * cols * 3 + 2 * MARGIN,), SENT, dtype=torch.uint8, device="cuda") if want_u8 else None
    m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    _check(_lib().ma_resample_v_norm_u8rgb(d_tmp.data_ptr(), n, frame_rows, cols, y0, tab.d_bounds.data_ptr(),
                                           tab.d_coeffs.data_ptr(), tab.ksize, tab.out_size, top, th, m3, s3,
                                           None if chw is None else chw.data_ptr() + 4 * MARGIN,
                                           None if u8 is None else u8.data_ptr() + MARGIN, _stream()),
           "ma_resample_v_norm_u8rgb")
    res = []
    for buf, sent, shape in ((chw, FSENT, (n, 3, th, cols)), (u8, SENT, (n, th, cols, 3))):
        if buf is None:
            res.append(None)
            continue
        b = buf.cpu()
        for edge in (b[:MARGIN], b[-MARGIN:]):
            assert torch.equal(edge, torch.full_like(edge, sent)), "wrote outside the output"
        res.append(b[MARGIN:-MARGIN].reshape(shape))
    return res


def _bits(t):
    return t.view(torch.int32).numpy() if t.dtype == torch.float32 else t.numpy()


@pytest.mark.parametrize("mode", ["both", "chw", "u8"])
@pytest.mark.parametrize("cols", [1, 127, 128, 129, 300])
@pytest.mark.parametrize("ksize,filt", V_TAPS, ids=[f"k{k}" for k, _ in V_TAPS])
def test_vertical_pass(ksize, filt, cols, mode):
    tab = table(*sizes_for(ksize, filt, 31), filt)
    assert tab.ksize == ksize
    top, th = 7, tab.out_size - 10  # far enough down that even the 129-tap window of row `top` starts below source row 0
    y0, y1 = tab.span(top, th)
    assert y0 > 0 and top + th < tab.out_size
    n = {"both": 5, "chw": 1, "u8": 3}[mode]
    rng = np.random.default_rng(ksize * 1000 + cols)
    tmp = rng.integers(0, 256, (n, y1 - y0, cols, 3), dtype=np.uint8)
    chw, u8 = run_v(tmp, y0, tab, top, th, mode != "u8", mode != "chw", frame_rows=y1 - y0 + 2)
    want8 = ref_v(tmp, y0, tab, top, th)
    if u8 is not None:
        assert np.array_equal(u8.numpy(), want8)
    if chw is not None:
        assert np.array_equal(_bits(chw), _bits(ref_normalize(want8, MEAN, STD)))


@pytest.mark.parametrize("norm", ["dinov2", "dust3r", "identity"])
def test_normalisation_of_every_byte(norm):
    from mapanything_b200.inference import IMAGE_NORMALIZATION_DICT

    assert sorted(IMAGE_NORMALIZATION_DICT) == ["dinov2", "dust3r", "identity"]
    mean, std = IMAGE_NORMALIZATION_DICT[norm]
    v = np.arange(256)
    tmp = np.stack([v, (v + 85) % 256, (255 - v)], -1).astype(np.uint8).reshape(1, 16, 16, 3)  # every byte in each channel
    tab = table(16, 16, LANCZOS)
    chw, u8 = run_v(tmp, 0, tab, 0, 16, True, True, mean, std)
    assert np.array_equal(u8.numpy(), tmp)
    assert np.array_equal(_bits(chw), _bits(ref_normalize(tmp, mean, std)))


# ------------------------------------------------------------------------------------------------ depth gather
SPECIAL_BITS = [0x7FC12345, 0x7F800001, 0xFFA00001, 0x7F800000, 0xFF800000, 0x80000000, 0x00000001, 0x80000003, 0x007FFFFF,
                0x00400000]  # NaNs with payloads (quiet, signalling, negative), +-inf, -0.0, subnormals


@pytest.mark.parametrize("H1,W1,rh,rw,top,left,th,tw,pad", [
    (50, 70, 120, 150, 5, 9, 100, 128, 0),       # enlarging
    (300, 411, 97, 133, 3, 2, 90, 129, 5),       # shrinking, padded source rows
    (64, 64, 64, 64, 0, 0, 64, 64, 3),           # same size
    (1080, 1920, 294, 522, 0, 2, 294, 518, 17),  # a camera depth map to 518 x 294
])
def test_gather_rows_cols(H1, W1, rh, rw, top, left, th, tw, pad):
    import cv2

    from mapanything_b200.image import _nearest_indices

    rng = np.random.default_rng(H1 + W1)
    src = rng.standard_normal((H1, W1)).astype(np.float32)
    flat = src.reshape(-1).view(np.uint32)
    pos = rng.choice(flat.size, 40 * len(SPECIAL_BITS), replace=False)
    flat[pos] = np.tile(np.array(SPECIAL_BITS, np.uint32), 40)
    want = cv2.resize(src, (rw, rh), interpolation=cv2.INTER_NEAREST)[top:top + th, left:left + tw]
    host = np.full((H1, W1 + pad), np.uint32(0x7FBADBAD), np.uint32).view(np.float32)  # NaN padding
    host[:, :W1] = src
    d_src = torch.from_numpy(host).cuda()
    yi = torch.from_numpy(_nearest_indices(H1, rh)[top:top + th].copy()).cuda()
    xi = torch.from_numpy(_nearest_indices(W1, rw)[left:left + tw].copy()).cuda()
    out = torch.full((th * tw + 2 * MARGIN,), FSENT, device="cuda")
    _check(_lib().ma_gather_rows_cols_f32(d_src.data_ptr(), W1 + pad, yi.data_ptr(), xi.data_ptr(), th, tw,
                                          out.data_ptr() + 4 * MARGIN, _stream()), "ma_gather_rows_cols_f32")
    got = out.cpu().view(torch.int32).numpy()
    sent = np.float32(FSENT).view(np.int32)
    assert (got[:MARGIN] == sent).all() and (got[-MARGIN:] == sent).all()
    assert np.array_equal(got[MARGIN:-MARGIN].reshape(th, tw), want.view(np.int32))
    assert np.isin(want.view(np.uint32), SPECIAL_BITS).sum() > 0  # the specials are in the crop


# ------------------------------------------------------------------------------------------------ image conversion
def _reference_u8(img):
    """The reference's conversion (image.py:503-506), in img's own dtype and on img's device."""
    if img.max() <= 1.0:
        return (img * 255).clamp(0, 255).byte()
    return img.clamp(0, 255).byte()


def _neighbours(x):
    """x and its two floating-point neighbours (positive x), through the integer view of the dtype."""
    it = {torch.float16: torch.int16, torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}[x.dtype]
    b = x.view(it)
    return torch.cat([x, (b - 1).view(x.dtype), (b + 1).view(x.dtype)])


def _conversion_values(dtype, kind):
    g = torch.Generator().manual_seed(11)
    u = torch.arange(256, dtype=torch.int64)
    if dtype == torch.uint8:
        return {"random": torch.randint(0, 256, (3000,), generator=g), "binary": torch.randint(0, 2, (3000,), generator=g),
                "zeros": torch.zeros(300, dtype=torch.int64)}[kind].to(dtype)
    if not dtype.is_floating_point:
        return {"random": torch.randint(-300, 600, (3000,), generator=g), "binary": torch.randint(0, 2, (3000,), generator=g),
                "unit_negative": torch.randint(-5, 2, (3000,), generator=g)}[kind].to(dtype)
    if kind == "k_over_255":
        return u.to(dtype) / 255
    if kind == "fp16_codes":
        return torch.arange(0, 0x3C01, dtype=torch.int16).view(torch.float16)
    if kind == "random_1e6":
        return torch.rand(10 ** 6, dtype=torch.float64, generator=g)
    if kind == "near_integers":  # max > 1: no scaling, truncation right below and above every integer up to 256
        ints = torch.arange(1, 257, dtype=torch.float64).to(dtype)
        halves = (torch.arange(0, 300, dtype=torch.float64) + 0.5).to(dtype)
        special = torch.tensor([math.inf, -math.inf, -0.0, -1.0, -0.4, -300.0, 1e30, -1e30, 255.5, 254.99999999999997,
                                0.9137254686570376], dtype=torch.float64).to(dtype)
        return torch.cat([_neighbours(ints), halves, special])
    if kind == "unit_with_negatives":  # max <= 1, so scaled, with negatives and -inf
        return torch.cat([u.to(dtype) / 255, torch.tensor([-0.0, -1e-3, -1.0, -math.inf], dtype=torch.float64).to(dtype)])
    raise KeyError(kind)


FLOATS = [torch.float16, torch.bfloat16, torch.float32, torch.float64]
CONVERSION_CASES = (
    [(torch.uint8, k) for k in ("random", "binary", "zeros")]
    + [(dt, k) for dt in (torch.int32, torch.int64) for k in ("random", "binary", "unit_negative")]
    + [(dt, k) for dt in FLOATS for k in ("k_over_255", "near_integers", "unit_with_negatives")]
    + [(torch.float16, "fp16_codes"), (torch.float64, "random_1e6")]
)


def _as_image(v):
    v = torch.cat([v, v[: (-v.numel()) % 3]])  # a multiple of 3 values
    return v.reshape(-1, 1, 3)


@pytest.mark.parametrize("dtype,kind", CONVERSION_CASES, ids=[f"{str(d)[6:]}-{k}" for d, k in CONVERSION_CASES])
def test_image_conversion_matches_reference(dtype, kind):
    from mapanything_b200.image import _image_to_device_u8, _Uploader
    from oracle.image import _to_u8

    img = _as_image(_conversion_values(dtype, kind))
    assert img.dtype == dtype and not img.isnan().any()
    dev = torch.device("cuda", torch.cuda.current_device())
    d_img = img.to(dev)
    got = _image_to_device_u8(d_img, 0, dev, _Uploader(dev))
    assert got.is_cuda and got.dtype == torch.uint8 and got.shape == img.shape and got.is_contiguous()
    want = _reference_u8(d_img)
    bad = got != want
    assert not bad.any(), f"{int(bad.sum())} of {bad.numel()} bytes differ, e.g. {d_img[bad][:4].tolist()} -> " \
                          f"{got[bad][:4].tolist()}, want {want[bad][:4].tolist()}"
    assert np.array_equal(got.cpu().numpy(), _to_u8(img, 0))  # the same expression on the CPU copy


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int32, torch.int64] + FLOATS, ids=lambda d: str(d)[6:])
def test_preprocess_inputs_of_cuda_images_matches_reference(dtype):
    """preprocess_inputs on a CUDA image of each dtype against oracle.image.preprocess_inputs on its CPU copy, bit for bit."""
    from mapanything_b200.image import preprocess_inputs
    from oracle import image as OI

    g = torch.Generator().manual_seed(3)
    u8 = torch.randint(0, 256, (45, 61, 3), dtype=torch.uint8, generator=g)
    if dtype == torch.uint8:
        img = torch.randint(0, 2, u8.shape, dtype=torch.uint8, generator=g)  # 0 / 1: scaled by 255
    elif dtype.is_floating_point:
        img = u8.to(dtype) / 255
        if dtype == torch.float64:
            img = img + (torch.rand(u8.shape, dtype=dtype, generator=g) - 0.5) * 1e-9
            img = img.clamp(0, 1)
    else:
        img = u8.to(dtype) * 3 - 200  # outside [0, 255] on both sides
    kw = dict(resize_mode="fixed_size", size=(56, 42))
    got = preprocess_inputs([{"img": img.cuda()}], **kw)[0]["img"]
    want = OI.preprocess_inputs([{"img": img}], **kw)[0]["img"]
    assert got.is_cuda and got.shape == want.shape
    assert torch.equal(got.cpu().view(torch.int32), want.view(torch.int32))


@pytest.mark.parametrize("n", [1, 255, 256, 257, 1_000_003])
@pytest.mark.parametrize("scale", [255.0, 1.0])
def test_f32_to_u8(n, scale):
    g = torch.Generator().manual_seed(n)
    base = torch.cat([torch.arange(256) / 255, _neighbours(torch.arange(1, 257, dtype=torch.float32)),
                      torch.tensor([math.inf, -math.inf, -0.0, -1.0, 255.5, 1e30, -1e30, 1.4e-45]),
                      torch.rand(n, generator=g) * 310 - 10])
    x = base[torch.randperm(base.numel(), generator=g)[:n]] if n < base.numel() else base[:n]
    buf = torch.zeros(n + 1, device="cuda")
    d_in = buf[1:]  # 4- but not 16-byte aligned
    d_in.copy_(x.cuda())
    out = torch.full((n + 2 * MARGIN,), SENT, dtype=torch.uint8, device="cuda")
    _check(_lib().ma_f32_to_u8(d_in.data_ptr(), n, scale, out.data_ptr() + MARGIN, _stream()), "ma_f32_to_u8")
    want = (d_in * scale).clamp(0, 255).byte()
    got = out.cpu()
    assert (got[:MARGIN] == SENT).all() and (got[-MARGIN:] == SENT).all()
    assert torch.equal(got[MARGIN:-MARGIN], want.cpu())


# ------------------------------------------------------------------------------------------------ coverage
def test_every_horizontal_instantiation_ran():
    """Last in the file: the matrix above reached every dp4a and word-load instantiation and the byte-load form, each with a
    staged row below and above 48 KB of shared memory."""
    want = {(c, size) for c in [1] + [1000 + 4 * w for w in range(1, 17)] + [2000 + w for w in range(1, 17)]
            for size in ("small", "large")}
    assert want - SEEN == set(), f"not reached: {sorted(want - SEEN)}"
