"""Host-side argument checks of ma_gemm_bf16 / ma_conv3x3_bf16 that run before any CUDA call.

Every full 32-column chunk of an output row goes through the vector epilogue (16-byte loads of bias / colscale / residual,
16-byte stores of out / out_relu), also when N is not a multiple of 32 and a scalar chunk follows it.  So with N >= 32
every epilogue operand must be 16-byte aligned at each row, and a call that breaks that must be refused with
MA_ERR_INVALID naming the operand instead of being launched.

The calls pass fake, never dereferenced device addresses.  They are made only where no CUDA device is visible: if a
check were missing, the call would go on to the launch, and on a GPU box that would run a kernel on those addresses."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device addresses; host-only check")

BASE = 1 << 32  # fake device addresses, 16-byte aligned
X, W, OUT, RES, RELU, BIAS, CS = (BASE + i * (1 << 24) for i in range(7))
MA_BF16, MA_F32 = 0, 1


def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib


def _epi(N, *, out=OUT, ldo=None, out_dtype=MA_F32, residual=None, ldr=0, residual_dtype=MA_F32, out_relu=None, ldo_relu=0,
         bias=None, colscale=None):
    ep = _lib().GemmEpilogue()
    ep.out, ep.ldo, ep.out_dtype = out, N if ldo is None else ldo, out_dtype
    ep.residual, ep.ldr, ep.residual_dtype = residual, ldr, residual_dtype
    ep.out_relu, ep.ldo_relu = out_relu, ldo_relu
    ep.bias, ep.colscale = bias, colscale
    return ep


def _gemm(N, ep, M=256, K=64):
    lib = _lib().load()
    rc = lib.ma_gemm_bf16(X, K, W, K, M, N, K, ctypes.byref(ep), 0, None)
    return rc, lib.ma_last_error().decode()


def _conv(Cout, ep, n=1, H=8, W_=8, C=64):
    lib = _lib().load()
    rc = lib.ma_conv3x3_bf16(X, n, H, W_, C, W, 9 * C, Cout, ctypes.byref(ep), 0, None)
    return rc, lib.ma_last_error().decode()


# (N, epilogue, operand the error must name).  Each case is legal except for the one misaligned operand.
MISALIGNED = {
    "f32_residual_ldr34": (34, dict(ldo=36, residual=RES, ldr=34), "residual"),          # 136-byte rows
    "bf16_residual_ldr34": (34, dict(ldo=36, residual=RES, ldr=34, residual_dtype=MA_BF16), "residual"),
    "f32_residual_ldr42": (40, dict(ldo=40, residual=RES, ldr=42), "residual"),         # 168-byte rows
    "residual_ptr_off": (40, dict(ldo=40, residual=RES + 4, ldr=40), "residual"),
    "out_relu_ldo36": (40, dict(ldo=40, out_relu=RELU, ldo_relu=36), "out_relu"),        # 72-byte rows
    "out_relu_ptr_off": (40, dict(ldo=40, out_relu=RELU + 8, ldo_relu=40), "out_relu"),
    "bias_off4": (40, dict(ldo=40, bias=BIAS + 4), "bias"),
    "colscale_off4": (40, dict(ldo=40, colscale=CS + 4), "colscale"),
    "bias_off4_n100": (100, dict(ldo=100, bias=BIAS + 4), "bias"),
    "bf16_out_ldo36": (40, dict(ldo=36, out_dtype=MA_BF16), "output"),
    "f32_out_ldo34": (34, dict(ldo=34), "output"),
    "bias_off4_n64": (64, dict(ldo=64, bias=BIAS + 4), "bias"),                         # N % 32 == 0: refused before too
    "residual_ldr34_n64": (64, dict(ldo=64, residual=RES, ldr=34), "residual"),
}


@pytest.mark.parametrize("case", sorted(MISALIGNED))
def test_gemm_refuses_misaligned_epilogue_operand(case):
    N, kw, operand = MISALIGNED[case]
    rc, msg = _gemm(N, _epi(N, **kw))
    assert rc == -1, f"{case}: accepted ({msg})"
    assert msg.startswith("ma_gemm_bf16:") and f"{operand} not 16-byte aligned" in msg, msg


@pytest.mark.parametrize("case", sorted(c for c, (N, _, _) in MISALIGNED.items() if N == 40))
def test_conv_refuses_misaligned_epilogue_operand(case):
    """ma_conv3x3_bf16 shares the epilogue and its checks; Cout = 40 has one vector chunk and one scalar chunk per row."""
    Cout, kw, operand = MISALIGNED[case]
    rc, msg = _conv(Cout, _epi(Cout, **kw))
    assert rc == -1, f"{case}: accepted ({msg})"
    assert msg.startswith("ma_conv3x3_bf16:") and f"{operand} not 16-byte aligned" in msg, msg


@pytest.mark.parametrize("N,kw", [
    (34, dict(ldo=36, residual=RES, ldr=36, out_relu=RELU, ldo_relu=40, bias=BIAS, colscale=CS)),
    (100, dict(ldo=104, out_dtype=MA_BF16, residual=RES, ldr=104, residual_dtype=MA_BF16, bias=BIAS)),
    (6, dict(ldo=7, residual=RES + 4, ldr=6, out_relu=RELU + 2, ldo_relu=7, bias=BIAS + 4, colscale=CS + 4)),
])
def test_aligned_or_narrow_epilogue_passes_the_checks(N, kw):
    """Control: legal operands get past the epilogue checks (and then fail for want of a device, not of alignment).  N < 32
    has only the scalar chunk, so element alignment suffices there."""
    for rc, msg in (_gemm(N, _epi(N, **kw)), _conv(N, _epi(N, **kw))):
        assert rc != 0
        assert "aligned" not in msg, msg
