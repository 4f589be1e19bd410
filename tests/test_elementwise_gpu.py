"""GPU parity of the HBM-bound stage kernels against plain PyTorch fp32 references."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("C", [1024, 768, 128, 588 * 0 + 256])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_layernorm_matches_torch(C, out_dtype):
    """Both code paths: register-resident rows (C = 768 / 1024, fp32 in) and the generic three-pass kernel."""
    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(C)
    rows = 3 * 1370
    x = torch.randn(rows, C, device="cuda", generator=g) * 3 + 0.5
    w = torch.rand(C, device="cuda", generator=g) + 0.5
    b = torch.randn(C, device="cuda", generator=g)
    out = torch.full((rows, C), float("nan"), device="cuda", dtype=out_dtype)
    ops.layernorm(x, out, w, b, eps=1e-6)
    ref = torch.nn.functional.layer_norm(x, (C,), w, b, 1e-6)
    tol = 2e-2 if out_dtype == torch.bfloat16 else 2e-5
    assert (out.float() - ref).abs().max().item() < tol * ref.abs().max().item()


def test_layernorm_row_remap_drops_cls_token():
    from mapanything_b200 import ops

    n, N, C = 3, 1369, 1024
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(n * (N + 1), C, device="cuda", generator=g)
    w = torch.rand(C, device="cuda", generator=g) + 0.5
    b = torch.randn(C, device="cuda", generator=g)
    out = torch.zeros(n * N, C, device="cuda")
    ops.layernorm(x, out, w, b, rows=n * N, rows_per_group=N, in_group_stride=N + 1, in_row_offset=1, out_group_stride=N,
                  out_row_offset=0)
    ref = torch.nn.functional.layer_norm(x.view(n, N + 1, C)[:, 1:], (C,), w, b, 1e-6).reshape(n * N, C)
    assert (out - ref).abs().max().item() < 2e-5 * ref.abs().max().item()


@pytest.mark.parametrize("N,K", [(6, 128), (7, 256), (1, 32), (8, 64)])
def test_head_linear_small_matches_torch(N, K):
    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(N * 100 + K)
    rows = 70 * 70 * 3 + 5
    x = torch.randn(rows, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device="cuda", generator=g)
    out = torch.full((rows, 8), 7.0, device="cuda")
    ops.head_linear_small(x, w, b, out)
    ref = x.float() @ w.float().t() + b
    assert (out[:, :N] - ref).abs().max().item() < 1e-4 * max(1.0, ref.abs().max().item())
    assert (out[:, N:] == 7.0).all()


@pytest.mark.parametrize("pct", [10, 50, 0, 100, 33.3])
def test_quantile_mask_matches_torch_quantile(pct):
    """apply_confidence_mask (reference inference.py:393-415): exact radix select + torch's float32 lerp."""
    from mapanything_b200.inference import quantile_mask

    g = torch.Generator().manual_seed(int(pct * 10))
    conf = 1.0 + torch.exp(torch.randn(3, 70, 70, generator=g) * 2)
    conf[1, :10] = 1.0          # many ties at the minimum
    conf[2] = conf[2].round()   # heavy ties everywhere
    thr = torch.quantile(conf.reshape(3, -1), pct / 100.0, dim=1).view(3, 1, 1)
    want = conf > thr
    got = quantile_mask(conf.cuda(), pct / 100.0).cpu()
    assert torch.equal(got, want), (got != want).sum().item()


@pytest.mark.parametrize("n,Hin,Win,C,Ho,Wo,virt", [(2, 19, 19, 256, 37, 37, (38, 38)), (1, 37, 37, 256, 74, 74, None),
                                                    (1, 40, 56, 128, 70, 98, None), (2, 5, 7, 64, 5, 7, None)])
def test_bilinear_align_corners_matches_torch(n, Hin, Win, C, Ho, Wo, virt):
    """F.interpolate(mode="bilinear", align_corners=True) over NHWC bf16, incl. the refinenet4 case (19 -> 38 cropped to 37)."""
    import torch.nn.functional as F

    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(Hin * 100 + Wo)
    x = torch.randn(n, Hin, Win, C, device="cuda", generator=g).bfloat16()
    out = torch.full((n, Ho, Wo, C), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.bilinear_ac(x, out, virtual_hw=virt)
    Hv, Wv = virt if virt else (Ho, Wo)
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), size=(Hv, Wv), mode="bilinear", align_corners=True)
    ref = ref[:, :, :Ho, :Wo].permute(0, 2, 3, 1)
    assert (out.float() - ref).abs().max().item() < 2e-2 * ref.abs().max().item()


LINEAR_ROWS = [(8, 768, 768, "relu"), (1, 768, 768, "gelu"), (8, 7, 768, None), (1, 1, 768, None), (16, 128, 8, "gelu"),
               (3, 1024, 512, None), (12, 77, 1024, "relu")]
# (rows, N, K, act, ldx - K, ldo - N, bias): row-strided x (NaN padding) and out (sentinel padding), no bias, K = 4, and
# rows * K = 16 * 768 floats, exactly the 48 KB of shared memory the kernel stages x in
LINEAR_ROWS_STRIDED = [(16, 40, 768, "gelu", 4, 3, True), (16, 9, 768, None, 8, 0, False), (5, 33, 4, "relu", 4, 1, False),
                       (3, 100, 256, None, 0, 5, False)]


@pytest.mark.parametrize("rows,N,K,act,ldx_pad,ldo_pad,bias", [
    *(pytest.param(*c, 0, 0, True, id="-".join(map(str, c))) for c in LINEAR_ROWS),
    *(pytest.param(*c, id="-".join(map(str, c[:4])) + f"-ldx+{c[4]}-ldo+{c[5]}" + ("" if c[6] else "-nobias"))
      for c in LINEAR_ROWS_STRIDED)])
def test_linear_rows_f32_matches_torch(rows, N, K, act, ldx_pad, ldo_pad, bias):
    """ma_linear_rows_f32 (the pooled MLPs of the pose / scale heads and the per-view global encoders): plain fp32 Linear on up
    to 16 rows against torch (float64 accumulation as the yardstick).  Per element: lanes stride over K in float4 steps, so
    each output is a chain of 4 ceil(K / 128) FMAs, 5 shuffle adds and the bias: D = 4 ceil(K / 128) + 7 and
    |y - ref| <= D u (|x| |w|^T + |b|) (x 1.13 through GELU) + 2e-7 |pre-GELU| (the erf approximation) + u |ref|."""
    import torch.nn.functional as F

    from mapanything_b200 import _lib, ops
    from mapanything_b200._lib import MA_ACT_GELU, MA_ACT_NONE, MA_ACT_RELU

    g = torch.Generator(device="cuda").manual_seed(rows * 1000 + N + K)
    xbuf = torch.full((rows + 1, K + ldx_pad), float("nan"), device="cuda")
    xbuf[:rows, :K] = torch.randn(rows, K, device="cuda", generator=g)
    x = xbuf[:rows, :K]
    w = torch.randn(N, K, device="cuda", generator=g) * K ** -0.5
    b = torch.randn(N, device="cuda", generator=g) if bias else None
    obuf = torch.full((rows, N + ldo_pad), -77.0, device="cuda")
    out = obuf[:, :N]
    code = {"relu": MA_ACT_RELU, "gelu": MA_ACT_GELU, None: MA_ACT_NONE}[act]
    if ldx_pad or ldo_pad:   # ops.linear_rows_f32 takes contiguous tensors only
        _lib.check(_lib.load().ma_linear_rows_f32(x.data_ptr(), x.stride(0), w.data_ptr(), w.stride(0), b.data_ptr() if bias else None,
                                                  code, out.data_ptr(), out.stride(0), rows, N, K,
                                                  torch.cuda.current_stream().cuda_stream), "ma_linear_rows_f32")
    else:
        ops.linear_rows_f32(x, w, b, out, code)
    pre = x.double() @ w.double().t() + (b.double() if bias else 0.0)
    mag = x.double().abs() @ w.double().abs().t() + (b.double().abs() if bias else 0.0)
    ref = F.relu(pre) if act == "relu" else F.gelu(pre) if act == "gelu" else pre
    assert torch.isfinite(out).all()
    assert (out.double() - ref).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())
    u = 2.0 ** -24
    bound = (4 * -(-K // 128) + 7) * u * mag * (1.13 if act == "gelu" else 1.0) + u * ref.abs()
    if act == "gelu":
        bound = bound + 2e-7 * pre.abs()
    ratio = ((out.double() - ref).abs() / bound).max().item()
    print(f"\n[linear_rows_f32] rows={rows} N={N} K={K} act={act}: worst err/bound {ratio:.3g}", end="")
    assert ratio <= 1.0, ratio
    assert (obuf[:, N:] == -77.0).all(), "ldo padding written"


def test_token_mean_f32_matches_torch():
    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(5)
    for n, T, C in ((8, 1369, 768), (2, 25, 96), (1, 70, 64)):
        x = torch.randn(n, T, C, device="cuda", generator=g) + 0.5
        out = torch.full((n, C), float("nan"), device="cuda")
        ops.token_mean_f32(x, out)
        assert (out.double() - x.double().mean(1)).abs().max().item() < 1e-5
