"""Every tile instantiation of the tcgen05 GEMM with every fused epilogue route, against an fp64 reference, element by element.

gemm_bf16_kernel<CTAS, BN> has five instantiations (block codes 64 / 128 / 256 = one CTA per 128 x BN tile, 2128 / 2256 =
a CTA pair per 256 x BN tile) and three store routes: the TMA store (plain output rows), the TMA reduce-add (in-place fp32
residual, plus the stream-K tail on pairs) and the per-thread vector store with a scalar path for a ragged last 32-column
chunk.  pick_block_n can put any shape on any instantiation, so each route runs here on each of them (`block_n` forced,
checked with ma_last_gemm_block).

Reference: x.double() @ w.double().T on the bf16 operand values, then the epilogue in fp64 in the order
include/mapanything_b200.h states (bias, activation unless late, out_relu if early, colscale, residual, activation if late,
out, out_relu).  GELU is the erf form.

Bound, per element: with mag = (|x| @ |w|^T) |colscale| + |bias colscale| + |residual| (GELU slope 1.13 folded in),
  fp32 out:  |y - ref| <= 2^-19 mag + 2e-7 |pre-GELU|                (the second term: the A&S erf of gelu_erf)
  bf16 out:  the fp32 bound (1 + 2^-8) + 2^-8 |ref|  [+ 5e-4 + 2^-12 |pre-GELU| where the tanh GELU may run]
Rounding the accumulator to bf16 would cost 2^-9 |acc|, which is > 10x the fp32 bound at every shape here (|acc| / mag is
at least ~1/30 at K = 1024), so the fp32 checks tell an fp32 epilogue from a bf16 one, and the erf term tells erf GELU from
the tanh form (4.8e-4 apart at |x| ~ 2.7).  Every case prints its worst err / bound.  Measured on one NVIDIA B200 (1000 W
power limit): fp32 outputs <= 0.16 of the bound (GELU routes <= 0.09); bf16 outputs up to 0.994, the 2^-8 |ref| term being
the exact worst case of rounding to the nearest bf16 just above a power of two.

Outputs are NaN-filled where the kernel must write and hold a sentinel where it must not (ldo / ldo_relu padding columns,
rows the row remap skips), checked bit for bit.  x and w carry NaN in their ldx / ldw > K padding: TMA must read K columns.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

CODES = [64, 128, 256, 2128, 2256]
NONE, GELU, RELU = 0, 1, 2
SENTINEL = -77.0           # exact in fp32 and bf16
F32, BF16 = torch.float32, torch.bfloat16
GELU_SLOPE = 1.13          # max |GELU'(x)|


def _lib():
    from mapanything_b200 import _lib

    return _lib.load()


def _round_up(n, a):
    return (n + a - 1) // a * a


def _padded(rows, cols, dtype, align, fill, g=None, scale=1.0):
    """[rows, cols] view of a [rows, round_up(cols, align) + align] buffer whose padding columns hold `fill`."""
    buf = torch.full((rows, _round_up(cols, align) + align), fill, device="cuda", dtype=dtype)
    if g is not None:
        buf[:, :cols] = (torch.randn(rows, cols, device="cuda", generator=g) * scale).to(dtype)
    return buf, buf[:, :cols]


def _gelu(v):
    return 0.5 * v * (1.0 + torch.erf(v / math.sqrt(2.0)))


def _act(v, act):
    return _gelu(v) if act == GELU else (torch.relu(v) if act == RELU else v)


def _bound(ref, mag, pre, bf16_out, gelu_erf_ok):
    """Elementwise bound (module docstring).  pre: None, or (|pre-GELU value|, factor the GELU output was scaled by
    afterwards); gelu_erf_ok: only the erf form may have run."""
    b = 2.0 ** -19 * mag
    if pre is not None:
        b = b + 2e-7 * pre[0] * pre[1]
    if bf16_out:
        b = b * (1 + 2.0 ** -8) + 2.0 ** -8 * ref.abs()
        if pre is not None and not gelu_erf_ok:
            b = b + (5e-4 + 2.0 ** -12 * pre[0]) * pre[1]
    return b


def _check(got, ref, bound, what):
    err = (got.double() - ref).abs()
    ratio = torch.nan_to_num(err / bound, nan=float("inf"))
    worst = ratio.max().item()
    print(f"\n{what}: worst err/bound {worst:.3g}", end="")
    if worst > 1.0:
        r, c = divmod(int(ratio.argmax().item()), ratio.shape[1])
        raise AssertionError(f"{what}: element ({r}, {c}) = {got[r, c].item()!r}, reference {ref[r, c].item()!r}, "
                             f"bound {bound[r, c].item():.3g} (worst err/bound {worst:.3g})")
    return worst


def _check_untouched(buf, out_rows, N, what):
    """Bit-exact sentinel everywhere in buf except columns [0, N) of out_rows."""
    written = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    written[out_rows, :N] = True
    bits = buf.view(torch.int32 if buf.dtype == F32 else torch.int16)
    want = torch.tensor([SENTINEL], dtype=buf.dtype, device=buf.device).view(bits.dtype)
    bad = (bits != want) & ~written
    assert not bad.any(), f"{what}: {int(bad.sum())} elements outside the output were written, first at {bad.nonzero()[0].tolist()}"


def run_case(bn, M, N, K, *, out_dtype=F32, bias=False, act=NONE, colscale=False, residual=None, res_mod=0, out_relu=False,
             act_late=False, relu_early=False, remap=None, seed=0, what=""):
    """One ops.gemm call with the given epilogue, checked against the fp64 reference.  residual: None / F32 / BF16 /
    "inplace" (out is the fp32 residual).  remap: (rows_per_group_in, rows_per_group_out, row_offset_out)."""
    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(seed * 7919 + M * 31 + N * 7 + K + bn)
    _, x = _padded(M, K, BF16, 8, float("nan"), g)
    _, w = _padded(N, K, BF16, 8, float("nan"), g, 1.0 / K ** 0.5)
    b = torch.randn(N, device="cuda", generator=g) if bias else None
    cs = torch.randn(N, device="cuda", generator=g) if colscale else None   # signs and small columns included

    m = torch.arange(M, device="cuda")
    if remap:
        rin, rout, off = remap
        out_rows = (m // rin) * rout + off + m % rin
        rows_out = (M // rin) * rout
    else:
        out_rows, rows_out = m, M
    res_rows = m % res_mod if res_mod else out_rows

    oalign = 4 if out_dtype == F32 else 8
    obuf, out = _padded(rows_out, N, out_dtype, oalign, SENTINEL)
    r = None
    if residual == "inplace":
        out[out_rows] = torch.randn(M, N, device="cuda", generator=g)
        r = out
        res64 = out.double().clone()
    elif residual is not None:
        ralign = 4 if residual == F32 else 8
        _, r = _padded(res_mod or rows_out, N, residual, ralign, float("nan"), g)
        res64 = r.double()
        out[out_rows] = float("nan")
    else:
        out[out_rows] = float("nan")
    relu_buf = relu = None
    if out_relu:
        relu_buf, relu = _padded(rows_out, N, BF16, 8, SENTINEL)
        relu[out_rows] = float("nan")

    ops.gemm(x, w, out, bias=b, act=act, colscale=cs, residual=r, residual_row_mod=res_mod, out_relu=relu,
             rows_per_group_in=remap[0] if remap else 0, rows_per_group_out=remap[1] if remap else 0,
             row_offset_out=remap[2] if remap else 0, block_n=bn, act_after_residual=act_late,
             relu_out_before_residual=relu_early)
    torch.cuda.synchronize()
    assert _lib().ma_last_gemm_block() == bn

    # fp64 reference of the epilogue, rows in GEMM order m
    x64, w64 = x.double(), w.double()
    v = x64 @ w64.T
    mag = x64.abs() @ w64.abs().T
    if b is not None:
        v = v + b.double()
        mag = mag + b.double().abs()
    pre = None
    if not act_late and act != NONE:
        pre = (v.abs(), 1.0) if act == GELU else None
        v = _act(v, act)
        mag = mag * (GELU_SLOPE if act == GELU else 1.0)
    twin = (v, mag, pre) if relu_early else None
    if cs is not None:
        v = v * cs.double()
        mag = mag * cs.double().abs()
        pre = pre and (pre[0], cs.double().abs())
    if residual is not None:
        rr = res64[res_rows]
        v = v + rr
        mag = mag + rr.abs()
    if act_late and act != NONE:
        pre = (v.abs(), 1.0) if act == GELU else None
        v = _act(v, act)
        mag = mag * (GELU_SLOPE if act == GELU else 1.0)
    if twin is None:
        twin = (v, mag, pre)

    bf16_out = out_dtype == BF16
    tag = f"{what} bn={bn} M={M} N={N} K={K}"
    worst = _check(out[out_rows], v, _bound(v, mag, pre, bf16_out, not bf16_out), tag)
    _check_untouched(obuf, out_rows, N, tag + " out")
    if out_relu:
        tv, tmag, tpre = twin
        tref = torch.relu(tv)
        _check(relu[out_rows], tref, _bound(tref, tmag, tpre, True, not bf16_out), tag + " out_relu")
        _check_untouched(relu_buf, out_rows, N, tag + " out_relu")
    return out, worst


# route -> (epilogue, shapes (M, N, K)).  M: 1 (one tile), 129 (ragged second tile), 261 (3 row tiles: a CTA pair's second
# half of its last tile is empty); N: multiples of every BN, multiples of 32 that are not multiples of 64 / 128 / 256; K from
# one MMA (8) to 16 K blocks.
ROUTES = {
    "a_bias_colscale_f32_tma": (dict(bias=True, colscale=True), [(1, 256, 40), (261, 160, 1024), (129, 96, 8)]),
    "b_bias_gelu_bf16_tma": (dict(bias=True, act=GELU, out_dtype=BF16), [(129, 256, 200), (261, 96, 40)]),
    "c_bias_gelu_f32_erf": (dict(bias=True, act=GELU), [(261, 256, 200), (1, 160, 1024)]),
    "e_f32_residual_vector": (dict(bias=True, colscale=True, residual=F32), [(129, 256, 200), (261, 96, 1024)]),
    "f_bf16_residual_bf16_out": (dict(bias=True, residual=BF16, out_dtype=BF16), [(261, 160, 40), (1, 256, 200)]),
    "g_out_relu_after_residual": (dict(bias=True, residual=BF16, out_relu=True), [(129, 256, 40), (261, 96, 200)]),
    "h_relu_out_before_residual": (dict(bias=True, colscale=True, residual=F32, out_relu=True, relu_early=True),
                                   [(261, 256, 200), (129, 160, 8)]),
    "i_relu_after_residual_twin": (dict(bias=True, residual=F32, act=RELU, act_late=True, out_relu=True),
                                   [(261, 256, 1024), (129, 96, 40)]),
    "j_gelu_after_residual_f32": (dict(bias=True, residual=F32, act=GELU, act_late=True), [(129, 256, 200)]),
    "j_gelu_after_residual_bf16": (dict(bias=True, residual=F32, act=GELU, act_late=True, out_dtype=BF16), [(261, 160, 40)]),
    "k_row_remap_residual_row_mod": (dict(bias=True, residual=F32, res_mod=137, remap=(137, 138, 1)), [(3 * 137, 256, 200)]),
    "l_residual_row_mod_1": (dict(bias=True, residual=F32, res_mod=1), [(261, 160, 40)]),
}
ROUTE_CASES = [(r, s) for r, (_, shapes) in ROUTES.items() for s in shapes]


@pytest.mark.parametrize("bn", CODES)
@pytest.mark.parametrize("route,shape", ROUTE_CASES, ids=[f"{r}-{'x'.join(map(str, s))}" for r, s in ROUTE_CASES])
def test_epilogue_route(route, shape, bn):
    torch.backends.cuda.matmul.allow_tf32 = False
    epi, _ = ROUTES[route]
    run_case(bn, *shape, what=route, **epi)


# Route m: a ragged N (6: the scalar chunk alone; 40 / 100: vector chunks and a scalar chunk in one row) with each feature
# of the vector-store routes.
RAGGED = {
    "e": dict(bias=True, colscale=True, residual=F32),
    "f": dict(bias=True, residual=BF16, out_dtype=BF16),
    "g": dict(bias=True, residual=BF16, out_relu=True),
    "h": dict(bias=True, colscale=True, residual=F32, out_relu=True, relu_early=True),
    "i": dict(bias=True, residual=F32, act=RELU, act_late=True, out_relu=True),
    "j": dict(bias=True, colscale=True, residual=F32, act=GELU, act_late=True),
}


@pytest.mark.parametrize("bn", CODES)
@pytest.mark.parametrize("N", [6, 40, 100])
@pytest.mark.parametrize("feature", sorted(RAGGED))
def test_epilogue_ragged_n(feature, N, bn):
    torch.backends.cuda.matmul.allow_tf32 = False
    run_case(bn, 261, N, 200, what=f"m_ragged_{feature}", **RAGGED[feature])


def _multi_wave_m(bn, N):
    """M giving every CTA / CTA pair >= 3 tiles (both TMEM accumulators go around their phases more than once)."""
    ctas, BN = (2, bn - 2000) if bn > 2000 else (1, bn)
    workers = torch.cuda.get_device_properties(0).multi_processor_count // ctas
    tiles_n = -(-N // BN)
    row_tiles = -(-(3 * workers + 1) // tiles_n)   # per worker (CTA or pair)
    return row_tiles * ctas * 128 - 77             # ragged last tile


@pytest.mark.parametrize("bn", CODES)
@pytest.mark.parametrize("route", ["a_bias_colscale_f32_tma", "e_f32_residual_vector"])
def test_epilogue_multi_wave(route, bn):
    torch.backends.cuda.matmul.allow_tf32 = False
    run_case(bn, _multi_wave_m(bn, 256), 256, 40, what=route + "_multiwave", **ROUTES[route][0])


@pytest.mark.parametrize("bn", CODES)
@pytest.mark.parametrize("shape", [(261, 256, 1024), (129, 160, 40)])
def test_inplace_residual_reduce_add(shape, bn):
    """Route d: x += colscale * (x W^T + bias) through the TMA reduce-add.  The whole-tile schedule is bit reproducible; on
    one-CTA codes stream-K (a CTA-pair feature) changes nothing."""
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    before = ops.set_stream_k(None)
    try:
        outs = []
        for mode in (False, False, True):
            ops.set_stream_k(mode)
            y, _ = run_case(bn, *shape, bias=True, colscale=True, residual="inplace", what=f"d_inplace stream_k={mode}")
            outs.append(y.clone())
        assert torch.equal(outs[0], outs[1]), "whole-tile reduce-add not bit reproducible"
        if bn < 2000:
            assert torch.equal(outs[0], outs[2]), "stream-K changed a one-CTA launch"
    finally:
        ops.set_stream_k(before)


@pytest.mark.parametrize("bn", [2128, 2256])
def test_stream_k_tail_on_each_pair_tile(bn):
    """Route d with K = 2048 on 20 / 40 pair tiles (fewer than the 74 CTA pairs): the K blocks are split over all pairs and
    joined by the reduce-add; bias added once."""
    from mapanything_b200 import ops

    torch.backends.cuda.matmul.allow_tf32 = False
    before = ops.set_stream_k(None)
    try:
        ops.set_stream_k(True)
        run_case(bn, 5000, 256, 2048, bias=True, colscale=True, residual="inplace", what="d_stream_k")
    finally:
        ops.set_stream_k(before)


# ---- split-bf16 (~fp32) products: ops.split3 activations [hi | lo | hi] x engine.Lin3 weights [hi | hi | lo] ----------


def test_split3_bit_exact_on_strided_input():
    from mapanything_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(3)
    buf = torch.randn(300, 136, device="cuda", generator=g) * torch.exp(torch.randn(300, 136, device="cuda", generator=g) * 4)
    # rows 0-59: +-0, fp32 subnormals, magnitudes near 1e30 and exact bf16 rounding ties (low 16 bits 0x8000: halfway
    # between two bf16 values, with an even and an odd bf16 neighbour below) at normal, subnormal and ~1e30 magnitudes
    base = torch.tensor([1.0, -3.0, 1e30, -7e29, 1.5e-38, 2.5e-39, -1e-40, 0.1], device="cuda")
    bits = base.view(torch.int32)
    ties = torch.cat([((bits & -0x20000) | 0x8000).view(torch.float32), ((bits & -0x20000) | 0x18000).view(torch.float32)])
    special = torch.cat([torch.tensor([0.0, -0.0, 1e-45, -1e-45, 1e-40, -3e-39, 1.1e-38, 1e30, -1e30, 3.3e30, -9.9e29],
                                      device="cuda"), ties])
    buf[:60, :special.numel()] = special
    buf[:60, 60:60 + special.numel()] = special.flip(0)
    x = buf[:, :120]   # ld_in = 136 > C
    got = ops.split3(x)
    hi = x.bfloat16()
    lo = (x - hi.float()).bfloat16()
    want = torch.cat([hi, lo, hi], dim=1)
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


def _split_vs_plain(got_split, got_plain, ref, mag, what):
    """Worst |y - ref| / mag of the split and the plain bf16 product, with mag = |x| @ |w|^T + |b|: the split must stay
    within 2^-15 (3.1e-5; its missing lo x lo term and the rounding of lo are ~2^-18 each) and be >= 30x better than plain
    bf16.  Measured on one NVIDIA B200 (1000 W power limit): split 2.3e-6 (Linear) / 1.7e-6 (conv), plain bf16 1.1e-3 /
    8.6e-4, a ratio of ~490."""
    e_split = ((got_split.double() - ref).abs() / mag).max().item()
    e_plain = ((got_plain.double() - ref).abs() / mag).max().item()
    print(f"\n{what}: worst err/mag split {e_split:.3g}, plain bf16 {e_plain:.3g}, ratio {e_plain / max(e_split, 1e-300):.3g}",
          end="")
    assert e_split <= 2.0 ** -15, f"{what}: split-bf16 error {e_split:.3g} of the magnitude"
    assert e_plain >= 30 * e_split, f"{what}: plain bf16 ({e_plain:.3g}) not 30x worse than split ({e_split:.3g})"


@pytest.mark.parametrize("bn", [128, 2256])
def test_split_bf16_linear_matches_fp64(bn):
    """A Linear (group = K) in split-bf16: gemm(split3(x32), Lin3(w32).w) vs x32 @ w32^T in fp64."""
    from mapanything_b200 import ops
    from mapanything_b200.engine import Lin3

    torch.backends.cuda.matmul.allow_tf32 = False
    M, N, K = 517, 192, 200
    g = torch.Generator(device="cuda").manual_seed(11)
    x32 = torch.randn(M, K, device="cuda", generator=g)
    w32 = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    lin = Lin3(w32, b)
    out = torch.full((M, N), float("nan"), device="cuda")
    ops.gemm(ops.split3(x32), lin.w, out, bias=lin.b, block_n=bn)
    assert _lib().ma_last_gemm_block() == bn
    plain = torch.full((M, N), float("nan"), device="cuda")
    ops.gemm(x32.bfloat16(), w32.bfloat16(), plain, bias=b, block_n=bn)
    torch.cuda.synchronize()
    ref = x32.double() @ w32.double().T + b.double()
    mag = x32.double().abs() @ w32.double().abs().T + b.double().abs()
    _split_vs_plain(out, plain, ref, mag, f"split linear bn={bn}")


def _conv_f64(u, w4, b=None):
    """3x3 / pad 1 conv in fp64 as im2col + matmul: u (n,H,W,C), w4 (Cout,C,3,3) -> [n*H*W, Cout]."""
    n, H, W, C = u.shape
    cols = torch.nn.functional.unfold(u.double().permute(0, 3, 1, 2), 3, padding=1)   # (n, C*9, H*W), k = c*9 + ky*3 + kx
    y = cols.transpose(1, 2).reshape(n * H * W, C * 9) @ w4.double().reshape(w4.shape[0], -1).T
    return y + b.double() if b is not None else y


@pytest.mark.parametrize("bn", [64, 2128])
def test_split_bf16_conv3x3_matches_fp64(bn):
    """A 3x3 conv (group = Cin, the tap-major layout of the pose blocks): conv3x3(split3(u) as (n,h,w,3C), Lin3(w).w) vs the
    fp64 conv.  Ragged pixel tiles (13 x 11) and C = 40 (not a multiple of 64)."""
    from mapanything_b200 import ops
    from mapanything_b200.engine import Lin3

    n, H, W, C, Cout = 2, 13, 11, 40, 96
    g = torch.Generator(device="cuda").manual_seed(12)
    u = torch.randn(n, H, W, C, device="cuda", generator=g)
    w4 = torch.randn(Cout, C, 3, 3, device="cuda", generator=g) / (9 * C) ** 0.5
    b = torch.randn(Cout, device="cuda", generator=g)
    lin = Lin3(w4.permute(0, 2, 3, 1), b, group=C)
    out = torch.full((n * H * W, Cout), float("nan"), device="cuda")
    ops.conv3x3(ops.split3(u.reshape(-1, C)).view(n, H, W, 3 * C), lin.w, out, bias=lin.b, block_n=bn)
    assert _lib().ma_last_gemm_block() == bn
    plain = torch.full((n * H * W, Cout), float("nan"), device="cuda")
    ops.conv3x3(u.bfloat16(), w4.permute(0, 2, 3, 1).reshape(Cout, 9 * C).bfloat16().contiguous(), plain, bias=b, block_n=bn)
    torch.cuda.synchronize()
    ref = _conv_f64(u, w4, b)
    mag = _conv_f64(u.abs(), w4.abs(), b.abs())
    _split_vs_plain(out, plain, ref, mag, f"split conv3x3 bn={bn}")
