"""Host-side argument checks of the HBM-bound stage kernels (csrc/elementwise.cu) that run before any CUDA call.

Those kernels move four or eight elements per access: LayerNorm loads fp32 rows as float4 and bf16 rows as uint2 (and stores
out the same way), gamma / beta as float4; im2col, pixel_shuffle and the bilinear resize load and store uint4; split3 loads
float4 and stores uint2; decode_dense loads each row as float4 + float2 when ld_raw % 4 == 0.  A row stride below the row
width makes rows overlap.  A call that breaks one of these rules must be refused with MA_ERR_INVALID naming the operand
instead of being launched.

The calls pass fake, never dereferenced device addresses.  They are made only where no CUDA device is visible: if a check
were missing, the call would go on to the launch, and on a GPU box that would run a kernel on those addresses."""
import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device addresses; host-only check")

BASE = 1 << 32  # fake device addresses, 16-byte aligned
IN, OUT, GAMMA, BETA, A, B, W, BIAS, POSE, SCALE = (BASE + i * (1 << 28) for i in range(10))
MA_BF16, MA_F32 = 0, 1
MA_ERR_INVALID = -1


def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib.load()


def _call(fn, *args):
    lib = _lib()
    rc = getattr(lib, fn)(*args)
    return rc, lib.ma_last_error().decode()


def layernorm(*, inp=IN, in_dtype=MA_F32, ld_in=None, out=OUT, out_dtype=MA_BF16, ld_out=None, gamma=GAMMA, beta=BETA,
              C=1024):
    return _call("ma_layernorm", inp, in_dtype, C if ld_in is None else ld_in, out, out_dtype, C if ld_out is None else ld_out,
                 gamma, beta, 4096, C, 1e-6, 0, 0, 0, 0, 0, None)


def im2col(*, inp=IN, out=OUT):
    return _call("ma_im2col3x3", inp, out, 2, 37, 21, 64, 1, None)


def pixel_shuffle(*, inp=IN, out=OUT):
    return _call("ma_pixel_shuffle", inp, out, 2, 37, 21, 256, 2, None)


def bilinear(*, inp=IN, out=OUT):
    return _call("ma_bilinear_align_corners", inp, out, 2, 19, 11, 256, 38, 22, 37, 21, None)


def split3(*, inp=IN, ld_in=120, out=OUT, C=120):
    return _call("ma_split_bf16x3", inp, ld_in, out, 300, C, None)


def decode(*, raw=IN, ld_raw=8):
    outs = [OUT + i * (1 << 24) for i in range(10)]
    return _call("ma_decode_dense", raw, ld_raw, POSE, SCALE, 3, 70 * 98, *outs, None)


def set_rows(*, dst=OUT, ld=1024, C=1024, b=B):
    return _call("ma_set_rows", dst, ld, 3, 1370, 0, A, b, C, None)


def head_linear(*, x=IN, ldx=128, w=W, ldw=128, ldo=8, K=128, N=6):
    return _call("ma_head_linear_small", x, ldx, w, ldw, BIAS, OUT, ldo, 3 * 518 * 518, N, K, None)


def linear_rows(*, x=IN, ldx=768, w=W, ldw=768, ldo=768, K=768, N=768):
    return _call("ma_linear_rows_f32", x, ldx, w, ldw, BIAS, 0, OUT, ldo, 8, N, K, None)


# (call, arguments, start of the error message).  Each case is legal except for the one bad operand.
REFUSED = {
    "layernorm_f32_in_off8": (layernorm, dict(inp=IN + 8), "ma_layernorm: in not 16-byte aligned"),
    "layernorm_f32_in_off8_c772": (layernorm, dict(inp=IN + 8, C=772), "ma_layernorm: in not 16-byte aligned"),
    "layernorm_bf16_in_off4": (layernorm, dict(inp=IN + 4, in_dtype=MA_BF16), "ma_layernorm: in not 8-byte aligned"),
    "layernorm_f32_out_off8": (layernorm, dict(out=OUT + 8, out_dtype=MA_F32), "ma_layernorm: out not 16-byte aligned"),
    "layernorm_bf16_out_off4": (layernorm, dict(out=OUT + 4, C=768), "ma_layernorm: out not 8-byte aligned"),
    "layernorm_gamma_off4": (layernorm, dict(gamma=GAMMA + 4), "ma_layernorm: gamma not 16-byte aligned"),
    "layernorm_beta_off4": (layernorm, dict(beta=BETA + 4, in_dtype=MA_BF16, C=128), "ma_layernorm: beta not 16-byte aligned"),
    "layernorm_ld_in_short": (layernorm, dict(ld_in=1020), "ma_layernorm: ld_in"),
    "layernorm_ld_out_short": (layernorm, dict(ld_out=1020), "ma_layernorm: ld_out"),
    "im2col_in_off2": (im2col, dict(inp=IN + 2), "ma_im2col3x3: in not 16-byte aligned"),
    "im2col_out_off8": (im2col, dict(out=OUT + 8), "ma_im2col3x3: out not 16-byte aligned"),
    "pixel_shuffle_in_off8": (pixel_shuffle, dict(inp=IN + 8), "ma_pixel_shuffle: in not 16-byte aligned"),
    "pixel_shuffle_out_off8": (pixel_shuffle, dict(out=OUT + 8), "ma_pixel_shuffle: out not 16-byte aligned"),
    "bilinear_in_off8": (bilinear, dict(inp=IN + 8), "ma_bilinear_align_corners: in not 16-byte aligned"),
    "bilinear_out_off2": (bilinear, dict(out=OUT + 2), "ma_bilinear_align_corners: out not 16-byte aligned"),
    "split3_in_off8": (split3, dict(inp=IN + 8), "ma_split_bf16x3: in not 16-byte aligned"),
    "split3_out_off4": (split3, dict(out=OUT + 4), "ma_split_bf16x3: out not 8-byte aligned"),
    "split3_ld_in_short": (split3, dict(ld_in=116), "ma_split_bf16x3: ld_in"),
    "decode_ld8_raw_off4": (decode, dict(raw=IN + 4), "ma_decode_dense: raw not 16-byte aligned"),
    "decode_ld12_raw_off8": (decode, dict(raw=IN + 8, ld_raw=12), "ma_decode_dense: raw not 16-byte aligned"),
    "set_rows_ld_short": (set_rows, dict(ld=1000), "ma_set_rows: ld"),
    "head_linear_ldx_short": (head_linear, dict(ldx=120), "ma_head_linear_small: ldx"),
    "head_linear_ldw_short": (head_linear, dict(ldw=127), "ma_head_linear_small: ldw"),
    "linear_rows_ldx_short": (linear_rows, dict(ldx=764), "ma_linear_rows_f32: ldx"),
    "linear_rows_ldw_short": (linear_rows, dict(ldw=764), "ma_linear_rows_f32: ldw"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_refuses_misaligned_or_overlapping_operand(case):
    call, kw, want = REFUSED[case]
    rc, msg = call(**kw)
    assert rc == MA_ERR_INVALID, f"{case}: accepted ({msg})"
    assert msg.startswith(want), msg


# Legal edge operands: each gets past the checks and then fails for want of a device, not of alignment or stride.
ACCEPTED = {
    "layernorm_bf16_out_off8_c1024": (layernorm, dict(out=OUT + 8)),               # generic kernel instead of the register one
    "layernorm_bf16_in_off8": (layernorm, dict(inp=IN + 8, in_dtype=MA_BF16, out_dtype=MA_F32)),
    "layernorm_ld_in_wider": (layernorm, dict(ld_in=1028, ld_out=1032, C=772)),
    "split3_out_off8": (split3, dict(out=OUT + 8, ld_in=136)),
    "decode_ld6_raw_off4": (decode, dict(raw=IN + 4, ld_raw=6)),
    "decode_ld7_raw_off4": (decode, dict(raw=IN + 4, ld_raw=7)),
    "set_rows_ld_wider_dst_off4": (set_rows, dict(dst=OUT + 4, ld=1030, b=None)),
    "head_linear_ldo11_w_off2": (head_linear, dict(ldo=11, ldx=136, ldw=133, w=W + 2)),
    "head_linear_thread_kernel": (head_linear, dict(K=200, ldx=200, ldw=200, N=8, ldo=8)),
    "linear_rows_ldo_wider": (linear_rows, dict(ldo=800, ldx=772, ldw=776)),
}


@pytest.mark.parametrize("case", sorted(ACCEPTED))
def test_legal_edge_operands_pass_the_checks(case):
    call, kw = ACCEPTED[case]
    rc, msg = call(**kw)
    assert rc != 0, f"{case}: launched without a device"
    assert "aligned" not in msg and "below" not in msg and "bad arguments" not in msg, msg
