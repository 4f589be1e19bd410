"""Every HBM-bound stage kernel of csrc/elementwise.cu on each path it accepts, against an fp64 reference, element by element.

Copies and permutations (patchify, im2col3x3, pixel_shuffle, pixel_shuffle_f32, set_rows, fill_f32, the logits of
decode_dense) are compared bit for bit with the same data moved by PyTorch.  Arithmetic kernels are compared with an fp64
reference of their operation under an elementwise bound built from u = 2^-24 (fp32 rounding), the length D of the fp32
reduction chain the kernel runs, and ub = 2^-8 (bf16 output rounding).  No bound is relative to the tensor maximum.  With
|s| the sum of the magnitudes of the reduced terms, a reduction of depth D is off by at most D u |s| (first order); a bf16
output adds ub |ref| to the fp32 bound b32: b = b32 (1 + ub) + ub |ref|.

- layernorm (row of C, B = ceil(C / 128) float4 steps per lane, 5 shuffle levels):
    mean  D = B + 8:            |d_mu| <= (B + 8) u mean|x|
    var   D = 4B + 10 over (x - mean)^2, plus d_mu^2 from the mean error:  e_var = (4B + 10) u + d_mu^2 / (var + eps)
    rstd  rsqrtf (2 ulp):       e_r = e_var / 2 + 4 u
    y = ((x - mean) rstd) g + b:  b32 = |g| rstd (d_mu + |x - mean| (e_r + 3 u)) + u (|y| + |b|)
  A one-pass variance (E[x^2] - mean^2) is off by ~1 in the rows of mean 1e3 and std 0.1; a dropped eps by a factor
  sqrt(2) in the rows of variance eps: both are orders of magnitude above the bound.
- head_linear_small: exact bf16 x bf16 products, D = K + 1 (thread kernel) or 8 + log2(K / 8) + 1 (warp kernels),
  b = D u (|x| |w|^T + |b|).
- token_mean_f32: D = ceil(T / 64) + 22 (four accumulators, three remainder steps, 16 row lanes, the division);
  token_mean (bf16): D = ceil(T / 4) + 3 and the bf16 output rounding.  b32 = D u mean_t |x|.
- bilinear (align_corners): the kernel's source coordinate yo * ((Hin - 1) / (Hv - 1)) carries two fp32 roundings, at
  most 3 u (Hin - 1) in source rows (the same in x); the interpolant's slope is at most 2 max|x|; the two lerps add at most
  12 u max|tap|.  b32 = 3 u ((Hin - 1) + (Win - 1)) 2 max|x| + 12 u max|tap|, then the bf16 output rounding.
- decode_dense: expf is within 2 ulp (4 u), sqrtf and the division are correctly rounded.  Per component:
  rays 8 u; pts3d_cam 24 u |cam| scale; pts3d 128 u (|cam| + |t|) scale (about 70 u from the rotation built from the
  normalised quaternion, rounded up); depth 12 u |ref|; conf 6 u |ref|; cam_trans 6 u |ref|; cam_quats 8 u;
  the metric scale 6 u |ref|.  Logits are bit exact; the mask is exactly logit > 0 (logits are kept off |l| < 1e-3).

Each case prints its worst err / bound as "[family] ...".  Where a kernel has several dispatch branches (layernorm,
head_linear_small), each case asserts from a torch.profiler trace which kernel ran.  Outputs hold a sentinel wherever the
call must not write (padding columns, rows a remap skips, one row or element past the end), checked bit for bit; inputs
hold NaN in their padding columns, in rows the call must skip and one row or image past the end.
"""
import math
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SENTINEL = -77.0                 # exact in fp32 and bf16
F32, BF16 = torch.float32, torch.bfloat16
U = 2.0 ** -24                   # fp32 unit roundoff
UB = 2.0 ** -8                   # bf16 unit roundoff
NAN = float("nan")
DEV = "cuda"
TYPE_NAME = {F32: "float", BF16: "__nv_bfloat16"}


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _kernel_of(call):
    """Runs call() under torch.profiler and returns the one ma:: kernel it launched, as name<template args> without spaces."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    found = set()
    for e in prof.events():
        m = re.search(r"ma::(\w+)(<[^()]*>)?\(", e.name)
        if m:
            found.add((m.group(1) + (m.group(2) or "")).replace(" ", ""))
    assert len(found) == 1, f"expected one ma:: kernel, the profiler saw {sorted(found)}"
    return found.pop()


def _bits(t):
    return t.view({F32: torch.int32, BF16: torch.int16, torch.uint8: torch.uint8}[t.dtype])


def _assert_bits(got, want, what):
    bad = _bits(got) != _bits(want)
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ, first at {list(i)}: "
                             f"{got[i].item()!r}, want {want[i].item()!r}")


def _assert_sentinel(buf, written, what):
    """Bit-exact SENTINEL in buf wherever the bool mask `written` (buf's shape) is False."""
    bad = (_bits(buf) != _bits(torch.full_like(buf, SENTINEL))) & ~written
    if bad.any():
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the output were written, first at "
                             f"{bad.nonzero()[0].tolist()}")


def _check(family, got, ref, bound, what):
    err = (got.double() - ref).abs()
    ratio = torch.nan_to_num(torch.where(err == 0, torch.zeros_like(err), err / bound), nan=math.inf)
    worst = ratio.max().item()
    print(f"\n[{family}] {what}: worst err/bound {worst:.3g}", end="")
    if worst > 1.0:
        i = int(ratio.argmax())
        raise AssertionError(f"{what}: element {i} = {got.reshape(-1)[i].item()!r}, reference {ref.reshape(-1)[i].item()!r}, "
                             f"bound {bound.reshape(-1)[i].item():.3g} (worst err/bound {worst:.3g})")
    return worst


def _bf16_bound(b32, ref):
    return b32 * (1 + UB) + UB * ref.abs()


# ---- patchify -----------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("hp,wp", [(37, 37), (37, 21), (7, 5), (1, 1)])
@pytest.mark.parametrize("p,kpad", [(14, 592), (14, 640), (8, 192), (8, 256)])
def test_patchify(p, kpad, hp, wp, n):
    """Bit exact against unfold -> bf16 (k = c p^2 + ky p + kx, the Conv2d weight order), zero in the kpad columns."""
    from mapanything_b200 import ops

    g = _gen(p * 1000 + kpad + hp * 37 + wp * 3 + n)
    H, W = hp * p, wp * p
    ibuf = torch.full((n + 1, 3, H, W), NAN, device=DEV)
    ibuf[:n] = torch.randn(n, 3, H, W, device=DEV, generator=g) * 3
    img = ibuf[:n]
    rows = n * hp * wp
    obuf = torch.full((rows + 1, kpad), SENTINEL, device=DEV, dtype=BF16)
    ops.patchify(img, obuf[:rows], p)
    want = torch.full_like(obuf, SENTINEL)
    want[:rows] = 0.0
    want[:rows, :3 * p * p] = F.unfold(img, p, stride=p).transpose(1, 2).reshape(rows, 3 * p * p).to(BF16)
    _assert_bits(obuf, want, f"patchify p={p} kpad={kpad} grid {hp}x{wp} n={n}")


# ---- layernorm ----------------------------------------------------------------------------------------------------------


def _ln_expected_kernel(in_dt, out_dt, C, aligned16):
    if in_dt == F32 and aligned16 and C in (768, 1024):
        return f"layernorm_f32_reg_kernel<{C // 128},{TYPE_NAME[out_dt]}>"
    return f"layernorm_kernel<{TYPE_NAME[in_dt]},{TYPE_NAME[out_dt]}>"


def _ln_rows(R, C, in_dt, eps, g):
    """Rows by r % 8: 0-4 N(0.5, 3^2); 5 mean 1e3 (std 0.1 in fp32, 16 in bf16, whose spacing there is 4); 6 variance ~eps;
    7 N(0.5, 3^2) with one element 300."""
    z = torch.randn(R, C, device=DEV, generator=g)
    kind = (torch.arange(R, device=DEV) % 8)[:, None]
    x = z * 3 + 0.5
    x = torch.where(kind == 5, 1e3 + z * (0.1 if in_dt == F32 else 16.0), x)
    x = torch.where(kind == 6, z * eps ** 0.5, x)
    r7 = torch.arange(7, R, 8, device=DEV)
    x[r7, r7 % C] = 300.0
    return x.to(in_dt)


def _ln_ref(x, gamma, beta, eps, out_dt):
    """fp64 LayerNorm of the rows of x and the elementwise bound of the module docstring."""
    C = x.shape[1]
    x, g, b = x.double(), gamma.double(), beta.double()
    mu = x.mean(1, keepdim=True)
    d = x - mu
    var = (d * d).mean(1, keepdim=True)
    rstd = (var + eps).rsqrt()
    ref = d * rstd * g + b
    B = -(-C // 128)
    d_mu = (B + 8) * U * x.abs().mean(1, keepdim=True)
    e_r = ((4 * B + 10) * U + d_mu ** 2 / (var + eps)) / 2 + 4 * U
    bound = g.abs() * rstd * (d_mu + d.abs() * (e_r + 3 * U)) + U * (ref.abs() + b.abs())
    return ref, _bf16_bound(bound, ref) if out_dt == BF16 else bound


def _ln_remap(remap, n, N):
    """(rows, rows of x, rows of out, ops.layernorm remap kwargs).  n views of N patch tokens (+ a cls token)."""
    if remap == "identity":
        R = n * (N + 1) + 3
        return R, R, R, {}
    if remap == "drop_cls":       # the encoder's final norm: skip each view's cls token
        return n * N, n * (N + 1), n * N, dict(rows_per_group=N, in_group_stride=N + 1, in_row_offset=1, out_group_stride=N)
    if remap == "scatter":        # groups land N + 3 rows apart at offset 2: sentinel gaps of 3 rows
        return n * N, n * N, n * (N + 3), dict(rows_per_group=N, in_group_stride=N, out_group_stride=N + 3, out_row_offset=2)
    if remap == "skip_last":      # info sharing: the scale token after the n * N patch rows is not normalised
        return n * N, n * N + 1, n * N + 1, {}
    raise ValueError(remap)


def run_layernorm(in_dt, out_dt, C, eps, remap="identity", out_off=0, seed=0):
    from mapanything_b200 import ops

    g = _gen(seed * 7919 + C * 31 + (in_dt == BF16) * 2 + (out_dt == BF16) + int(eps * 1e7) + out_off)
    n, N = 2, 1369
    rows, x_rows, out_rows, kw = _ln_remap(remap, n, N)
    r = torch.arange(rows, device=DEV)
    rpg = kw.get("rows_per_group", 0)
    if rpg:
        in_idx = (r // rpg) * kw["in_group_stride"] + kw.get("in_row_offset", 0) + r % rpg
        out_idx = (r // rpg) * kw["out_group_stride"] + kw.get("out_row_offset", 0) + r % rpg
    else:
        in_idx = out_idx = r

    ld_in, ld_out = C + 4, C + 4          # NaN / sentinel padding columns
    xbuf = torch.full((x_rows, ld_in), NAN, device=DEV, dtype=in_dt)
    xbuf[in_idx, :C] = _ln_rows(rows, C, in_dt, eps, g)    # rows the call must skip stay NaN
    x = xbuf[:, :C]
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g)
    flat = torch.full((out_off + out_rows * ld_out + 8,), SENTINEL, device=DEV, dtype=out_dt)
    out2d = flat[out_off:out_off + out_rows * ld_out].view(out_rows, ld_out)
    out = out2d[:, :C]

    ran = _kernel_of(lambda: ops.layernorm(x, out, gamma, beta, rows=rows, eps=eps, **kw))
    assert ran == _ln_expected_kernel(in_dt, out_dt, C, out_off == 0), ran

    eps32 = torch.tensor(eps, dtype=F32).item()
    ref, bound = _ln_ref(x[in_idx], gamma, beta, eps32, out_dt)
    what = f"layernorm {TYPE_NAME[in_dt]}->{TYPE_NAME[out_dt]} C={C} eps={eps} {remap} out+{out_off}"
    _check("layernorm", out[out_idx], ref, bound, what)
    written = torch.zeros(flat.shape, dtype=torch.bool, device=DEV)
    w2d = torch.zeros(out_rows, ld_out, dtype=torch.bool, device=DEV)
    w2d[out_idx, :C] = True
    written[out_off:out_off + out_rows * ld_out] = w2d.reshape(-1)
    _assert_sentinel(flat, written, what)


@pytest.mark.parametrize("eps", [1e-6, 1e-5])
@pytest.mark.parametrize("C", [1024, 768, 128, 4, 772])
@pytest.mark.parametrize("out_dt", [F32, BF16], ids=["f32out", "bf16out"])
@pytest.mark.parametrize("in_dt", [F32, BF16], ids=["f32in", "bf16in"])
def test_layernorm(in_dt, out_dt, C, eps):
    """Every dispatch branch: the register kernel (fp32 in, C = 768 / 1024) and the generic kernel for each dtype pair,
    also at C = 772 (not a multiple of 128) and C = 4 (one lane)."""
    run_layernorm(in_dt, out_dt, C, eps)


@pytest.mark.parametrize("remap", ["drop_cls", "scatter", "skip_last"])
@pytest.mark.parametrize("in_dt,out_dt,C", [(F32, BF16, 1024), (F32, F32, 768), (BF16, BF16, 772), (F32, BF16, 128)],
                         ids=["reg_f32_bf16_1024", "reg_f32_f32_768", "gen_bf16_bf16_772", "gen_f32_bf16_128"])
def test_layernorm_row_remap(in_dt, out_dt, C, remap):
    run_layernorm(in_dt, out_dt, C, 1e-6, remap, seed=1)


@pytest.mark.parametrize("remap", ["identity", "scatter"])
def test_layernorm_bf16_out_8_byte_aligned(remap):
    """A bf16 output 8- but not 16-byte aligned is legal and takes the generic kernel (C = 1024, fp32 in)."""
    run_layernorm(F32, BF16, 1024, 1e-6, remap, out_off=4, seed=2)


# ---- set_rows / fill_f32 ------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("with_b", [True, False], ids=["a_plus_b", "a"])
@pytest.mark.parametrize("C,ld,groups,group_stride,row_offset", [(1024, 1030, 3, 1370, 0), (768, 772, 8, 1370, 1369),
                                                                 (100, 103, 5, 7, 3)])
def test_set_rows(C, ld, groups, group_stride, row_offset, with_b):
    from mapanything_b200 import ops

    g = _gen(C + ld + groups)
    dst = torch.full((groups * group_stride, ld), SENTINEL, device=DEV)
    a = torch.randn(C, device=DEV, generator=g)
    b = torch.randn(C, device=DEV, generator=g) if with_b else None
    ops.set_rows(dst[:, :C], a, b, groups=groups, group_stride=group_stride, row_offset=row_offset)
    want = torch.full_like(dst, SENTINEL)
    want[torch.arange(groups, device=DEV) * group_stride + row_offset, :C] = a + b if with_b else a
    _assert_bits(dst, want, f"set_rows C={C} ld={ld} groups={groups}")


@pytest.mark.parametrize("value", [-math.inf, NAN, 3.5], ids=["-inf", "nan", "3.5"])
@pytest.mark.parametrize("count", ["1", "255", "257", "grid_stride"])
def test_fill_f32(count, value):
    """The grid holds at most 8 blocks of 256 per SM: sms * 8 * 256 + 13 elements run the grid-stride loop."""
    from mapanything_b200 import ops

    n = _sms() * 8 * 256 + 13 if count == "grid_stride" else int(count)
    buf = torch.full((n + 1,), SENTINEL, device=DEV)
    ops.fill_f32(buf[:n], value)
    want = torch.full_like(buf, value)
    want[n] = SENTINEL
    _assert_bits(buf, want, f"fill_f32 n={n} value={value}")


# ---- im2col3x3 / pixel_shuffle ------------------------------------------------------------------------------------------


@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("H,W", [(37, 37), (37, 21), (8, 9), (2, 3), (1, 1)])
@pytest.mark.parametrize("C", [8, 64, 256])
def test_im2col3x3(C, H, W, stride):
    """Bit exact against F.pad + a gather of the 9 taps (out[(i, yo, xo)][(ky * 3 + kx) * C + c])."""
    from mapanything_b200 import ops

    n = 2
    g = _gen(C * 1000 + H * 37 + W + stride)
    xbuf = torch.full((n + 1, H, W, C), NAN, device=DEV, dtype=BF16)
    xbuf[:n] = torch.randn(n, H, W, C, device=DEV, generator=g).to(BF16)
    x = xbuf[:n]
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    M = n * Ho * Wo
    obuf = torch.full((M + 1, 9 * C), SENTINEL, device=DEV, dtype=BF16)
    ops.im2col3x3(x, obuf[:M], stride)
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    taps = [xp[:, ky:ky + (Ho - 1) * stride + 1:stride, kx:kx + (Wo - 1) * stride + 1:stride] for ky in range(3) for kx in range(3)]
    want = torch.full_like(obuf, SENTINEL)
    want[:M] = torch.stack(taps, dim=3).reshape(M, 9 * C)
    _assert_bits(obuf, want, f"im2col3x3 C={C} {H}x{W} stride={stride}")


@pytest.mark.parametrize("s", [2, 4])
@pytest.mark.parametrize("h,w", [(37, 21), (21, 37), (5, 3), (1, 1)])
@pytest.mark.parametrize("C", [8, 256])
def test_pixel_shuffle(C, h, w, s):
    """bf16, the DPT act_postprocess ConvTranspose2d (s = 4 / 2): bit exact, on landscape and portrait patch grids."""
    from mapanything_b200 import ops

    n = 2
    g = _gen(C * 100 + h * 7 + w + s)
    rows, M = n * h * w, n * h * w * s * s
    xbuf = torch.full((rows + 1, s * s * C), NAN, device=DEV, dtype=BF16)
    xbuf[:rows] = torch.randn(rows, s * s * C, device=DEV, generator=g).to(BF16)
    x = xbuf[:rows]
    obuf = torch.full((M + 1, C), SENTINEL, device=DEV, dtype=BF16)
    ops.pixel_shuffle(x, obuf[:M], n, h, w, C, s)
    want = torch.full_like(obuf, SENTINEL)
    want[:M] = x.view(n, h, w, s, s, C).permute(0, 1, 3, 2, 4, 5).reshape(M, C)
    _assert_bits(obuf, want, f"pixel_shuffle C={C} {h}x{w} s={s}")


@pytest.mark.parametrize("ld_out", ["C", 8])
@pytest.mark.parametrize("C", [1, 4, 6])
@pytest.mark.parametrize("s,h,w", [(14, 5, 3), (2, 37, 21)])
def test_pixel_shuffle_f32(s, h, w, C, ld_out):
    """fp32 with row strides (the `linear` prediction head, patch 14): NaN in the ld_in padding, sentinel in ld_out's."""
    from mapanything_b200 import ops

    n = 2
    g = _gen(s * 100 + C * 10 + h)
    ldo = C if ld_out == "C" else ld_out
    rows, M, K = n * h * w, n * h * w * s * s, s * s * C
    xbuf = torch.full((rows + 1, K + 3), NAN, device=DEV)
    xbuf[:rows, :K] = torch.randn(rows, K, device=DEV, generator=g)
    x = xbuf[:rows, :K]
    obuf = torch.full((M + 1, ldo), SENTINEL, device=DEV)
    ops.pixel_shuffle_f32(x, obuf[:M, :C], n, h, w, C, s)
    want = torch.full_like(obuf, SENTINEL)
    want[:M, :C] = x.reshape(n, h, w, s, s, C).permute(0, 1, 3, 2, 4, 5).reshape(M, C)
    _assert_bits(obuf, want, f"pixel_shuffle_f32 s={s} {h}x{w} C={C} ld_out={ldo}")


# ---- bilinear (align_corners) -------------------------------------------------------------------------------------------


def _taps(n_in, n_virtual, n_out, dev):
    s = (n_in - 1) / (n_virtual - 1) if n_virtual > 1 else 0.0
    f = torch.arange(n_out, dtype=torch.float64, device=dev) * s
    i0 = f.floor().long().clamp(max=n_in - 1)
    return i0, (i0 + 1).clamp(max=n_in - 1), f - i0


BILINEAR = {   # (Hin, Win, (Hv, Wv), (Ho, Wo))
    "refinenet4_19x11_crop_37x21": (19, 11, (38, 22), (37, 21)),
    "37x21_to_74x42": (37, 21, (74, 42), (74, 42)),
    "regressor_296x168_to_518x294": (296, 168, (518, 294), (518, 294)),
    "regressor_296x296_to_518x518": (296, 296, (518, 518), (518, 518)),
    "hin1_1x7_to_4x13": (1, 7, (4, 13), (4, 13)),
    "win1_6x1_to_11x3": (6, 1, (11, 3), (11, 3)),
}


@pytest.mark.parametrize("C", [8, 256])
@pytest.mark.parametrize("shape", sorted(BILINEAR))
def test_bilinear_align_corners(shape, C):
    from mapanything_b200 import ops

    Hin, Win, (Hv, Wv), (Ho, Wo) = BILINEAR[shape]
    n = 2
    g = _gen(Hin * 1000 + Win + C)
    xbuf = torch.full((n + 1, Hin, Win, C), NAN, device=DEV, dtype=BF16)
    xbuf[:n] = torch.randn(n, Hin, Win, C, device=DEV, generator=g).to(BF16)
    x = xbuf[:n]
    m = n * Ho * Wo * C
    obuf = torch.full((m + 8 * C,), SENTINEL, device=DEV, dtype=BF16)
    out = obuf[:m].view(n, Ho, Wo, C)
    ops.bilinear_ac(x, out, virtual_hw=(Hv, Wv))
    y0, y1, wy = _taps(Hin, Hv, Ho, x.device)
    x0, x1, wx = _taps(Win, Wv, Wo, x.device)
    wx, wy = wx.view(1, Wo, 1), wy.view(Ho, 1, 1)
    for i in range(n):   # one image at a time: the 518 x 518 x 256 fp64 reference is 0.5 GB per tensor
        xi = x[i].double()
        a, b, c, d = xi[y0][:, x0], xi[y0][:, x1], xi[y1][:, x0], xi[y1][:, x1]
        top, bot = a * (1 - wx) + b * wx, c * (1 - wx) + d * wx
        ref = top * (1 - wy) + bot * wy
        tap = torch.maximum(torch.maximum(a.abs(), b.abs()), torch.maximum(c.abs(), d.abs()))
        b32 = 3 * U * ((Hin - 1) + (Win - 1)) * 2 * xi.abs().max() + 12 * U * tap
        _check("bilinear", out[i], ref, _bf16_bound(b32, ref), f"bilinear {shape} C={C} image {i}")
    _assert_sentinel(obuf[m:], torch.zeros(8 * C, dtype=torch.bool, device=DEV), f"bilinear {shape} C={C} tail")


# ---- token means --------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("C", [8, 100, 1024])
@pytest.mark.parametrize("T", [1, 3, 15, 16, 17, 63, 64, 65, 1369])
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
def test_token_mean(dt, T, C):
    """ma_token_mean_f32 / ma_token_mean (bf16) on inputs offset by +10, so that every term has the same sign."""
    from mapanything_b200 import ops

    n = 2
    g = _gen(T * 10000 + C * 2 + (dt == BF16))
    xbuf = torch.full((n + 1, T, C), NAN, device=DEV, dtype=dt)
    xbuf[:n] = (torch.randn(n, T, C, device=DEV, generator=g) + 10).to(dt)
    x = xbuf[:n]
    obuf = torch.full((n * C + 8,), SENTINEL, device=DEV, dtype=dt)
    out = obuf[:n * C].view(n, C)
    (ops.token_mean_f32 if dt == F32 else ops.token_mean)(x, out)
    x64 = x.double()
    ref = x64.mean(1)
    if dt == F32:
        bound = (-(-T // 64) + 22) * U * x64.abs().mean(1)
    else:
        bound = _bf16_bound((-(-T // 4) + 3) * U * x64.abs().mean(1), ref)
    what = f"token_mean {TYPE_NAME[dt]} T={T} C={C}"
    _check("token_mean_f32" if dt == F32 else "token_mean_bf16", out, ref, bound, what)
    _assert_sentinel(obuf[n * C:], torch.zeros(8, dtype=torch.bool, device=DEV), what)


# ---- head_linear_small --------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("N", [1, 6, 8])
@pytest.mark.parametrize("K", [8, 24, 32, 48, 200, 64, 128, 256])
def test_head_linear_small(K, N):
    """K = 64 / 128 / 256 take the warp kernels with LPR = K / 8 lanes per row, every other K the thread-per-row kernel.
    Rows: 1, 17, the 3 x 70 x 70 + 5 pixels of a small batch and, for each warp kernel, one row past two whole rounds of
    the grid (RPW * 4 rows per warp iteration, 8 blocks of 8 warps per SM).  x and w carry NaN in their padding."""
    from mapanything_b200 import ops

    lpr = K // 8
    warp = lpr in (8, 16, 32)
    kernel = f"head_linear_small_warp_kernel<{lpr}>" if warp else "head_linear_small_kernel"
    depth = 8 + int(math.log2(lpr)) + 1 if warp else K + 1
    rows_list = [1, 17, 70 * 70 * 3 + 5]
    if warp:
        rows_list.append((32 // lpr) * 4 * (2 * _sms() * 64) + 1)
    g = _gen(K * 10 + N)
    wbuf = torch.full((N + 1, K + 3), NAN, device=DEV, dtype=BF16)
    wbuf[:N, :K] = (torch.randn(N, K, device=DEV, generator=g) / K ** 0.5).to(BF16)
    w = wbuf[:N, :K]
    for i, rows in enumerate(rows_list):
        ldo = (N, 8, 11)[i % 3]
        b = torch.randn(N, device=DEV, generator=g) if i % 2 == 0 else None
        xbuf = torch.full((rows + 1, K + 8), NAN, device=DEV, dtype=BF16)
        xbuf[:rows, :K] = torch.randn(rows, K, device=DEV, generator=g).to(BF16)
        x = xbuf[:rows, :K]
        obuf = torch.full((rows + 1, ldo), SENTINEL, device=DEV)
        ran = _kernel_of(lambda: ops.head_linear_small(x, w, b, obuf[:rows, :N]))
        assert ran == kernel, ran
        x64, w64 = x.double(), w.double()
        ref, mag = x64 @ w64.T, x64.abs() @ w64.abs().T
        if b is not None:
            ref, mag = ref + b.double(), mag + b.double().abs()
        what = f"head_linear_small K={K} N={N} rows={rows} ldo={ldo} bias={b is not None}"
        _check("head_linear_small", obuf[:rows, :N], ref, depth * U * mag, what)
        written = torch.zeros(obuf.shape, dtype=torch.bool, device=DEV)
        written[:rows, :N] = True
        _assert_sentinel(obuf, written, what)


# ---- decode_dense -------------------------------------------------------------------------------------------------------


def _quat_to_rot(q):
    qx, qy, qz, qw = q.unbind(-1)
    return torch.stack([
        1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qw * qz), 2 * (qx * qz + qw * qy),
        2 * (qx * qy + qw * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qw * qx),
        2 * (qx * qz - qw * qy), 2 * (qy * qz + qw * qx), 1 - 2 * (qx * qx + qy * qy),
    ], -1).view(*q.shape[:-1], 3, 3)


def _decode_dense(raw, pose, scale_raw, n, HW, outs):
    """ma_decode_dense on caller-owned outputs (ops.decode_dense allocates its own, uninitialised)."""
    from mapanything_b200 import _lib

    _lib.check(_lib.load().ma_decode_dense(raw.data_ptr(), raw.stride(0), pose.data_ptr(), scale_raw.data_ptr(), n, HW,
                                           *(t.data_ptr() for t in outs), torch.cuda.current_stream().cuda_stream),
               "ma_decode_dense")


@pytest.mark.parametrize("HW", [70 * 98, 518 * 518], ids=["70x98", "518x518"])
@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("ld_raw", [6, 7, 8, 12])
def test_decode_dense(ld_raw, n, HW):
    """ld_raw % 4 != 0 takes the scalar loads (raw then starts 4 bytes past a 16-byte boundary, which is legal), else the
    float4 + float2 loads.  The grid holds at most 1024 blocks of 256 per view: 518 x 518 runs the grid-stride loop."""
    g = _gen(ld_raw * 100 + n * 10 + (HW > 10000))
    P = n * HW
    off = 1 if ld_raw % 4 else 0
    flat = torch.full((off + (P + 1) * ld_raw,), NAN, device=DEV)
    raw = flat[off:off + P * ld_raw].view(P, ld_raw)
    ray = torch.randn(P, 3, device=DEV, generator=g)
    ray = ray / ray.norm(dim=1, keepdim=True) * (0.5 + torch.rand(P, 1, device=DEV, generator=g))
    logit = torch.randn(P, device=DEV, generator=g) * 3
    logit = torch.where(logit.abs() < 1e-3, torch.copysign(torch.full_like(logit, 1e-3), logit), logit)
    raw[:, :3] = ray
    raw[:, 3] = torch.randn(P, device=DEV, generator=g) * 1.5      # depth logit
    raw[:, 4] = torch.randn(P, device=DEV, generator=g) * 2        # confidence logit
    raw[:, 5] = logit                                                 # mask logit
    pose = torch.randn(n, 7, device=DEV, generator=g)
    scale_raw = torch.tensor([0.3], device=DEV)

    def buf(*shape, dtype=F32):   # output + one sentinel row past its end
        b = torch.full((shape[0] + 1, *shape[1:]), SENTINEL if dtype == F32 else 0xAB, device=DEV, dtype=dtype)
        return b, b[:shape[0]]

    names = ["pts3d", "pts3d_cam", "rays", "depth", "conf", "logits", "mask", "cam_trans", "cam_quats", "scale"]
    shapes = [(P, 3), (P, 3), (P, 3), (P,), (P,), (P,), (P,), (n, 3), (n, 4), (1,)]
    bufs = {k: buf(*s, dtype=torch.uint8 if k == "mask" else F32) for k, s in zip(names, shapes)}
    o = {k: v[1] for k, v in bufs.items()}
    _decode_dense(raw, pose, scale_raw, n, HW, [o[k] for k in names])
    torch.cuda.synchronize()

    a = raw.double()
    scale = max(math.exp(scale_raw.double().item()), 1e-8)
    q = pose[:, 3:].double()
    q = q / q.norm(dim=1, keepdim=True)
    t = pose[:, :3].double()
    R = _quat_to_rot(q).repeat_interleave(HW, 0)
    tv = t.repeat_interleave(HW, 0)
    rays = a[:, :3] / a[:, :3].norm(dim=1, keepdim=True)
    depth = a[:, 3].exp()
    cam = rays * depth[:, None]
    world = (R @ cam[:, :, None]).squeeze(2) + tv
    conf = 1 + a[:, 4].exp()
    tn = tv.norm(dim=1, keepdim=True)
    what = f"decode_dense ld_raw={ld_raw} n={n} HW={HW}"
    _check("decode_dense", o["rays"], rays, torch.full_like(rays, 8 * U), what + " rays")
    _check("decode_dense", o["pts3d_cam"], cam * scale, (24 * U * depth * scale)[:, None].expand_as(cam), what + " pts3d_cam")
    _check("decode_dense", o["pts3d"], world * scale, (128 * U * (depth[:, None] + tn) * scale).expand_as(cam), what + " pts3d")
    _check("decode_dense", o["depth"], depth * scale, 12 * U * depth * scale, what + " depth")
    _check("decode_dense", o["conf"], conf, 6 * U * conf, what + " conf")
    _check("decode_dense", o["cam_trans"], t * scale, 6 * U * (t * scale).abs(), what + " cam_trans")
    _check("decode_dense", o["cam_quats"], q, torch.full_like(q, 8 * U), what + " cam_quats")
    s64 = torch.tensor([scale], dtype=torch.float64, device=DEV)
    _check("decode_dense", o["scale"], s64, 6 * U * s64, what + " scale")
    _assert_bits(o["logits"], raw[:, 5], what + " logits")
    assert torch.equal(o["mask"], (raw[:, 5] > 0).to(torch.uint8)), what + " mask"
    for k, (b, _) in bufs.items():
        _assert_bits(b[-1:], torch.full_like(b[-1:], SENTINEL if b.dtype == F32 else 0xAB), f"{what} {k} past the end")
