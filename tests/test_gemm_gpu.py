"""GPU parity tests for the tcgen05 GEMM (ma_gemm_bf16) against a plain fp32 PyTorch matmul."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref(x, w, bias=None, act=0, colscale=None, residual=None):
    y = x.float() @ w.float().t()
    if bias is not None:
        y = y + bias
    if act == 1:
        y = torch.nn.functional.gelu(y)
    elif act == 2:
        y = torch.relu(y)
    if colscale is not None:
        y = y * colscale
    if residual is not None:
        y = y + residual.float()
    return y


def _check(y, ref, tol=2e-2, what=""):
    err = (y.float() - ref).abs().max().item()
    scale = ref.abs().max().item() + 1e-6
    assert err <= tol * scale, f"{what}: max abs err {err:.4g} vs scale {scale:.4g}"


@pytest.mark.parametrize("bn", [0, 64, 128, 256, 2128, 2256])
@pytest.mark.parametrize("shape", [(128, 256, 64), (300, 512, 192), (2740, 1024, 1024), (1369, 96, 1024), (1000, 3072, 640)])
def test_gemm_plain(bn, shape):
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    M, N, K = shape
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    x = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) / K**0.5).bfloat16()
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float32)
    ops.gemm(x, w, out, block_n=bn)
    torch.cuda.synchronize()
    _check(out, _ref(x, w), 2e-3, f"plain {shape} bn={bn}")


def test_gemm_epilogues():
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    M, N, K = 1370 * 2, 1024, 1024
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) / K**0.5).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    gamma = torch.rand(N, device="cuda", generator=g) + 0.5
    res = torch.randn(M, N, device="cuda", generator=g)

    # bias + GELU -> bf16
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    ops.gemm(x, w, out, bias=bias, act=ops.MA_ACT_GELU)
    _check(out, _ref(x, w, bias, 1), 1e-2, "bias+gelu")

    # bias, layerscale, fp32 residual in place
    stream = res.clone()
    ops.gemm(x, w, stream, bias=bias, colscale=gamma, residual=stream)
    _check(stream, _ref(x, w, bias, 0, gamma, res), 2e-3, "bias+ls+residual(in place)")

    # relu + bf16 residual + second relu output
    resb = res.bfloat16()
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    out2 = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    ops.gemm(x, w, out, bias=bias, residual=resb, out_relu=out2)
    ref = _ref(x, w, bias, 0, None, resb)
    _check(out, ref, 1e-2, "bf16 residual")
    _check(out2, torch.relu(ref), 1e-2, "relu twin output")


@pytest.mark.parametrize("shape", [(10960, 1024, 4096), (10953, 768, 3072), (2740, 1024, 4096), (1370, 768, 3072),
                                   (26 * 1369 + 1, 768, 3072), (10960, 1024, 2048 + 40)])
def test_gemm_stream_k_residual(shape):
    """In-place fp32 residual GEMMs with K >= 2048 (fc2 of the transformer blocks): the K blocks of the last partial wave of
    tiles are split over all CTA pairs (stream-K) and joined by the reduce-add epilogue.  Same result as the whole-tile
    schedule up to the rounding of the partial-product sum (measured 2.6e-6 of the output scale at K = 4096: the tensor
    core's own fp32 accumulation over 4096 products differs by that much when the range is cut); bias added exactly once; the
    whole-tile schedule stays bit reproducible.  Shapes: 2 waves + 24 tiles, 1 wave + 55, fewer tiles than CTA pairs, ragged M and K."""
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    M, N, K = shape
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) / K**0.5).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    gamma = torch.rand(N, device="cuda", generator=g) + 0.5
    res = torch.randn(M, N, device="cuda", generator=g)
    ref = _ref(x, w, bias, 0, gamma, res)
    before = ops.set_stream_k(None)
    try:
        outs = {}
        for mode in (False, True):
            ops.set_stream_k(mode)
            runs = []
            for _ in range(2):
                y = res.clone()
                ops.gemm(x, w, y, bias=bias, colscale=gamma, residual=y)
                runs.append(y)
            outs[mode] = runs
            _check(runs[0], ref, 5e-4, f"stream_k={mode}")
        assert torch.equal(outs[False][0], outs[False][1]), "the whole-tile schedule is bit reproducible"
        _check(outs[True][0], outs[False][0].float(), 1e-5, "stream-K vs whole tiles")
        _check(outs[True][1], outs[True][0].float(), 1e-5, "stream-K run to run")
        e_sk = (outs[True][0] - ref).abs().max().item()
        e_dp = (outs[False][0] - ref).abs().max().item()
        print(f"\n{shape}: max abs err vs the fp32 product: whole tiles {e_dp:.3g}, stream-K {e_sk:.3g}")
        assert e_sk <= 2 * e_dp + 1e-5
        # without bias / LayerScale (plain x += X W^T)
        ops.set_stream_k(True)
        y = res.clone()
        ops.gemm(x, w, y, residual=y)
        _check(y, _ref(x, w, None, 0, None, res), 5e-4, "stream-K, no bias")
    finally:
        ops.set_stream_k(before)


def test_gemm_row_remap_and_strides():
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    n_img, P, K, N = 3, 1369, 640, 1024
    g = torch.Generator(device="cuda").manual_seed(2)
    xfull = torch.randn(n_img * P, K + 64, device="cuda", generator=g).bfloat16()
    x = xfull[:, :K]  # strided view, ld = K+64
    w = (torch.randn(N, K, device="cuda", generator=g) / K**0.5).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    pos = torch.randn(P + 1, N, device="cuda", generator=g)
    out = torch.zeros(n_img * (P + 1), N, device="cuda")
    ops.gemm(x, w, out, bias=bias, residual=pos[1:], residual_row_mod=P, rows_per_group_in=P,
             rows_per_group_out=P + 1, row_offset_out=1)
    ref = (_ref(x, w, bias).view(n_img, P, N) + pos[1:]).reshape(n_img, P, N)
    got = out.view(n_img, P + 1, N)
    _check(got[:, 1:], ref, 2e-3, "row remap")
    assert got[:, 0].abs().max().item() == 0.0

    # ragged N (scalar store path), N not a multiple of 32 and ldo padded
    N2 = 6
    w2 = (torch.randn(N2, 128, device="cuda", generator=g) / 11.0).bfloat16()
    x2 = torch.randn(777, 128, device="cuda", generator=g).bfloat16()
    b2 = torch.randn(N2, device="cuda", generator=g)
    out2 = torch.zeros(777, 8, device="cuda")
    ops.gemm(x2, w2, out2[:, :N2], bias=b2)
    _check(out2[:, :N2], _ref(x2, w2, b2), 2e-3, "ragged N")
    assert out2[:, N2:].abs().max().item() == 0.0


@pytest.mark.parametrize("n,H,W,C,Cout", [(2, 37, 37, 256, 256), (1, 19, 19, 768, 256), (3, 74, 74, 192, 256), (1, 148, 148, 96, 256),
                                          (2, 40, 56, 128, 128), (1, 5, 3, 64, 32), (1, 130, 70, 128, 6)])
@pytest.mark.parametrize("bn", [0, 64, 128, 256, 2128, 2256])
def test_conv3x3_implicit_gemm_matches_torch(n, H, W, C, Cout, bn):
    """Implicit-GEMM 3x3 conv (4-D TMA boxes, zero padding by out-of-bounds fill) vs F.conv2d on the same bf16 operands,
    incl. C not a multiple of 64, ragged pixel tiles, ragged Cout, bias + ReLU + residual + twin ReLU output, and the
    geometric-input encoders' bias + fp32 residual + GELU after the residual into bf16.  The fp32 output and the GELU case
    are also checked per element against an fp64 reference (the bound of test_gemm_epilogue_gpu.py)."""
    import torch.nn.functional as F

    from mapanything_b200 import _lib, ops
    from mapanything_b200.ops import MA_ACT_GELU, MA_ACT_RELU
    from test_gemm_epilogue_gpu import GELU_SLOPE, _bound, _check as _check_elementwise, _conv_f64, _gelu

    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(n * 1000 + H + W + C)
    x = torch.randn(n, H, W, C, device="cuda", generator=g).bfloat16()
    w4 = (torch.randn(Cout, C, 3, 3, device="cuda", generator=g) / (9 * C) ** 0.5).bfloat16()
    bias = torch.randn(Cout, device="cuda", generator=g)
    w = w4.permute(0, 2, 3, 1).reshape(Cout, 9 * C).contiguous()  # [Cout][(ky,kx),Cin]
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w4.float(), bias, padding=1).permute(0, 2, 3, 1).reshape(n * H * W, Cout)
    ref64 = _conv_f64(x, w4, bias)
    mag = _conv_f64(x.abs(), w4.abs(), bias.abs())

    out = torch.full((n * H * W, Cout), float("nan"), device="cuda")
    ops.conv3x3(x, w, out, bias=bias, block_n=bn)
    assert bn == 0 or _lib.load().ma_last_gemm_block() == bn
    _check(out, ref, 2e-3, "conv3x3 fp32 out")
    _check_elementwise(out, ref64, _bound(ref64, mag, None, False, True), f"conv3x3 fp32 out bn={bn}")

    # bias + fp32 residual, then GELU (geometric-input encoders), bf16 out
    res32 = torch.randn(n * H * W, Cout, device="cuda", generator=g)
    o4 = torch.full((n * H * W, Cout), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.conv3x3(x, w, o4, bias=bias, residual=res32, act=MA_ACT_GELU, act_after_residual=True, block_n=bn)
    pre = ref64 + res32.double()
    want = _gelu(pre)
    _check_elementwise(o4, want, _bound(want, (mag + res32.double().abs()) * GELU_SLOPE, (pre.abs(), 1.0), True, False),
                       f"conv3x3 + residual, GELU after it, bn={bn}")

    if Cout % 32 == 0:
        res = torch.randn(n * H * W, Cout, device="cuda", generator=g).bfloat16()
        o1 = torch.empty(n * H * W, Cout, device="cuda", dtype=torch.bfloat16)
        o2 = torch.empty(n * H * W, Cout, device="cuda", dtype=torch.bfloat16)
        ops.conv3x3(x, w, o1, bias=bias, residual=res, out_relu=o2, relu_out_before_residual=True, block_n=bn)
        _check(o1, ref + res.float(), 1e-2, "conv3x3 + residual")
        _check(o2, torch.relu(ref), 1e-2, "conv3x3 relu twin (before residual)")
        o3 = torch.empty(n * H * W, Cout, device="cuda", dtype=torch.bfloat16)
        ops.conv3x3(x, w, o3, bias=bias, act=MA_ACT_RELU, block_n=bn)
        _check(o3, torch.relu(ref), 1e-2, "conv3x3 + relu")


@pytest.mark.parametrize("n,H,W,C", [(2, 70, 70, 128), (1, 518, 301, 128), (3, 9, 5, 64)])
def test_conv3x3_fused_narrow_head_matches_torch(n, H, W, C):
    """ma_gemm_epilogue.head_*: conv3x3 (Cout = 128) + bias + ReLU consumed by a 128 -> 6 linear head in the epilogue (two
    64-column half-row warps combine through shared memory) vs F.conv2d -> relu -> F.linear in fp32 on the same bf16 operands.
    The hidden map is kept in fp32 here (the separate-kernel path rounds it to bf16 first)."""
    import torch.nn.functional as F

    from mapanything_b200 import ops
    from mapanything_b200.ops import MA_ACT_RELU

    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(H * 7 + W)
    x = torch.randn(n, H, W, C, device="cuda", generator=g).bfloat16()
    w4 = (torch.randn(128, C, 3, 3, device="cuda", generator=g) / (9 * C) ** 0.5).bfloat16()
    bias = torch.randn(128, device="cuda", generator=g)
    w = w4.permute(0, 2, 3, 1).reshape(128, 9 * C).contiguous()
    hw = torch.zeros(8, 128, device="cuda")
    hw[:6] = torch.randn(6, 128, device="cuda", generator=g) / 128 ** 0.5
    hb = torch.zeros(8, device="cuda")
    hb[:6] = torch.randn(6, device="cuda", generator=g)
    hidden = torch.relu(F.conv2d(x.float().permute(0, 3, 1, 2), w4.float(), bias, padding=1)).permute(0, 2, 3, 1).reshape(-1, 128)
    ref = hidden @ hw.t() + hb
    out = torch.full((n * H * W, 8), float("nan"), device="cuda")
    ops.conv3x3_head(x, w, bias, MA_ACT_RELU, hw, hb, out)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    _check(out[:, :6], ref[:, :6], 2e-3, "conv3x3 + fused head")
    assert out[:, 6:].abs().max().item() == 0.0
