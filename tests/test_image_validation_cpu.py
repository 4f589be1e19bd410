"""Host-side argument checks of the image kernels (csrc/image.cu) that run before any CUDA call.

The horizontal resampling pass indexes its staged row from sx0 and its source rows from y0, and reads bounds, coeffs and
the packed coefficients as 32-bit words; the vertical pass reads bounds / coeffs as words and stores fp32 to out_chw; the
depth gather reads and writes fp32 and int32; the float -> byte conversion reads fp32.  th is gridDim.y of the vertical
pass and of the gather, so it is at most 65535.  A source row span that does not fit shared memory cannot be staged.  A
call that breaks one of these rules must be refused with MA_ERR_INVALID naming the operand instead of being launched.

The calls pass fake, never dereferenced device addresses.  They are made only where no CUDA device is visible: if a check
were missing, the call would go on to the launch, and on a GPU box that would run a kernel on those addresses."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device addresses; host-only check")

BASE = 1 << 32  # fake device addresses, 16-byte aligned
SRC, TMP, BOUNDS, COEFFS, PACKED, OUT, OUT8, YIDX, XIDX = (BASE + i * (1 << 28) for i in range(9))
MA_ERR_INVALID = -1
MAX_SPAN = 68264  # pixels of the widest source row span that fits the 200 KB of shared memory of the byte-load form


def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib.load()


def _call(fn, *args):
    lib = _lib()
    rc = getattr(lib, fn)(*args)
    return rc, lib.ma_last_error().decode()


def resample_h(*, src=SRC, y0=3, sx0=5, span=900, bounds=BOUNDS, coeffs=COEFFS, packed=PACKED, ksize=25, tmp=TMP):
    # 1920 -> 522 LANCZOS (25 taps): 200 output columns from column 40 over `span` source pixels, 2 frames of 12 rows
    return _call("ma_resample_h_u8rgb", src, 1920 * 3 + 5, 1081 * (1920 * 3 + 5), 2, y0, 12, sx0, sx0 + span, bounds, coeffs,
                 packed, ksize, 522, 40, 200, tmp, None)


MEAN, STD = (C.c_float * 3)(0.485, 0.456, 0.406), (C.c_float * 3)(0.229, 0.224, 0.225)


def resample_v(*, tmp=TMP, bounds=BOUNDS, coeffs=COEFFS, out_chw=OUT, out_u8=OUT8, top=2, th=294, out_size=300):
    return _call("ma_resample_v_norm_u8rgb", tmp, 2, 1080, 518, 0, bounds, coeffs, 25, out_size, top, th, MEAN, STD, out_chw,
                 out_u8, None)


def gather(*, src=SRC, y_idx=YIDX, x_idx=XIDX, out=OUT, th=294):
    return _call("ma_gather_rows_cols_f32", src, 1920, y_idx, x_idx, th, 518, out, None)


def f32_to_u8(*, inp=SRC, out=OUT8):
    return _call("ma_f32_to_u8", inp, 1080 * 1920 * 3, 255.0, out, None)


# (call, arguments, start of the error message).  Each case is legal except for the one bad operand.
REFUSED = {
    "resample_h_sx0_negative": (resample_h, dict(sx0=-1), "ma_resample_h_u8rgb: sx0=-1 is negative"),
    "resample_h_y0_negative": (resample_h, dict(y0=-2), "ma_resample_h_u8rgb: y0=-2 is negative"),
    "resample_h_bounds_off2": (resample_h, dict(bounds=BOUNDS + 2), "ma_resample_h_u8rgb: bounds not 4-byte aligned"),
    "resample_h_coeffs_off1": (resample_h, dict(coeffs=COEFFS + 1), "ma_resample_h_u8rgb: coeffs not 4-byte aligned"),
    "resample_h_packed_off2": (resample_h, dict(packed=PACKED + 2), "ma_resample_h_u8rgb: packed not 4-byte aligned"),
    "resample_h_span_68265": (resample_h, dict(span=MAX_SPAN + 1),
                              "ma_resample_h_u8rgb: source rows of 68265 pixels do not fit shared memory"),
    "resample_h_span_68265_no_packed": (resample_h, dict(span=MAX_SPAN + 1, packed=None),
                                        "ma_resample_h_u8rgb: source rows of 68265 pixels do not fit shared memory"),
    "resample_h_span_68265_71_taps": (resample_h, dict(span=MAX_SPAN + 1, ksize=71),
                                      "ma_resample_h_u8rgb: source rows of 68265 pixels do not fit shared memory"),
    "resample_v_bounds_off2": (resample_v, dict(bounds=BOUNDS + 2), "ma_resample_v_norm_u8rgb: bounds not 4-byte aligned"),
    "resample_v_coeffs_off1": (resample_v, dict(coeffs=COEFFS + 1), "ma_resample_v_norm_u8rgb: coeffs not 4-byte aligned"),
    "resample_v_out_chw_off2": (resample_v, dict(out_chw=OUT + 2), "ma_resample_v_norm_u8rgb: out_chw not 4-byte aligned"),
    "resample_v_th_65536": (resample_v, dict(top=0, th=65536, out_size=70000), "ma_resample_v_norm_u8rgb: th=65536"),
    "gather_src_off2": (gather, dict(src=SRC + 2), "ma_gather_rows_cols_f32: src not 4-byte aligned"),
    "gather_y_idx_off1": (gather, dict(y_idx=YIDX + 1), "ma_gather_rows_cols_f32: y_idx not 4-byte aligned"),
    "gather_x_idx_off2": (gather, dict(x_idx=XIDX + 2), "ma_gather_rows_cols_f32: x_idx not 4-byte aligned"),
    "gather_out_off3": (gather, dict(out=OUT + 3), "ma_gather_rows_cols_f32: out not 4-byte aligned"),
    "gather_th_65536": (gather, dict(th=65536), "ma_gather_rows_cols_f32: th=65536"),
    "f32_to_u8_in_off2": (f32_to_u8, dict(inp=SRC + 2), "ma_f32_to_u8: in not 4-byte aligned"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_refuses_bad_operand(case):
    call, kw, want = REFUSED[case]
    rc, msg = call(**kw)
    assert rc == MA_ERR_INVALID, f"{case}: accepted ({msg})"
    assert msg.startswith(want), msg


# Legal edge operands: each gets past the checks and then fails for want of a device, not of an argument.
ACCEPTED = {
    "resample_h_src_odd_tmp_odd": (resample_h, dict(src=SRC + 1, tmp=TMP + 3)),
    "resample_h_src_off2": (resample_h, dict(src=SRC + 2)),
    "resample_h_sx0_y0_zero": (resample_h, dict(sx0=0, y0=0)),
    "resample_h_no_packed": (resample_h, dict(packed=None)),
    "resample_h_span_61098_dp4a": (resample_h, dict(span=61098)),
    "resample_h_span_68096_word_loads": (resample_h, dict(span=68096)),
    "resample_h_span_68264_byte_loads": (resample_h, dict(span=MAX_SPAN)),
    "resample_h_span_68264_71_taps": (resample_h, dict(span=MAX_SPAN, ksize=71)),
    "resample_v_out_u8_odd_no_chw": (resample_v, dict(out_chw=None, out_u8=OUT8 + 1, tmp=TMP + 3)),
    "resample_v_out_chw_off4": (resample_v, dict(out_chw=OUT + 4, out_u8=None)),
    "resample_v_th_65535": (resample_v, dict(top=1, th=65535, out_size=65536)),
    "gather_off4": (gather, dict(src=SRC + 4, y_idx=YIDX + 4, x_idx=XIDX + 12, out=OUT + 4)),
    "gather_th_65535": (gather, dict(th=65535)),
    "f32_to_u8_in_off4_out_odd": (f32_to_u8, dict(inp=SRC + 4, out=OUT8 + 1)),
}


@pytest.mark.parametrize("case", sorted(ACCEPTED))
def test_legal_edge_operands_pass_the_checks(case):
    call, kw = ACCEPTED[case]
    rc, msg = call(**kw)
    assert rc != 0, f"{case}: launched without a device"
    for word in ("aligned", "negative", "above", "bad arguments", "do not fit", "missing"):
        assert word not in msg, msg
