"""The geometric-input kernels (csrc/geometric_inputs.cu) and the infer() post-processing kernels (csrc/postprocess.cu),
each against a plain high-precision reference of the same operation, element by element.

Bounds use u = 2^-24 (one fp32 rounding) and follow the fp32 operation chain of each kernel.  No bound is relative to
the tensor maximum: each is per element, from the magnitudes of that element's own terms.

geometric_inputs.cu, against fp64:
- rays_from_intrinsics: xx = (x - cx) / fx is 2 roundings (2u relative), likewise yy; n = sqrt(xx^2 + yy^2 + 1) carries
  2 * 2u from the squared inputs, 3u from the sum and u from the sqrt (halved inside the root): 4.5u; the quotients
  xx / n add u.  b = 8u |ref|.
- normalize_rays: the sum of squares 3u, sqrt and the +1e-8f 2.5u, the quotient u: b = 6u |ref| (+ 2^-149 for
  subnormal squares of the near-zero rays, where 1e-8 dominates the norm).
- depth_z_to_along_ray: each d * (r / z) 2u; squares, sum and sqrt 4u more: b = 6u |ref|.
- pose_to_quat_trans: sq_best (3 additions of the diagonal, S = 1 + sum |m_ii|) is off by e_sq = 3u S; qa = sqrt(sq)
  by e_qa = u + e_sq / (2 sq_best); the candidate numerators by u (|m_a| + |m_b|) (one sum) or qa^2 (2 e_qa + u);
  the quotient adds e_qa + u relative.  b = 2 (e_num / den + |ref| (e_qa + u)).  The branch is checked explicitly:
  the float32 argmax of sq (first maximum, like torch.argmax) must equal the fp64 one on every case that is not an
  exact tie, and each of the four branches and the w < 0 flip is hit.  Translations are bit exact.
- unshuffle_split: mode 0 copies, so hi = bf16(v) and lo = bf16(v - hi) are bit exact on the input.  In mode 1 the
  kernel's fp32 v = (x * (1 / f)) / max(|.|, 1e-8) * log1pf(|.|) is recomputed with CUDA torch in the same operation
  order (torch.log1p calls the same log1pf); hi / lo are bit exact on it and it is within b = 8u |ref| + 2^-149 of
  fp64 (x / f: 2u, passed on at most fully by log1p; log1pf 1 ulp = 2u; below |v| = 1e-8 the quotient by 1e-8 and
  the product add u each and log1p(a) ~ a carries the 2u of a again).  hi + lo (what a split-bf16 GEMM sees) is also
  checked against fp64 with 2^-16 |ref| added: |v - hi| <= 2^-8 |v|, and lo rounds that to 2^-8 relative.
- depth_factor: 1024 threads each sum ceil(P / 1024) positive terms, then 5 shuffle levels and 32 warp partials:
  D = ceil(P / 1024) + 37; counts are exact integers.  factor: b = (D + 2) u |ref| (the sum, c + 1e-8f, the
  quotient).  log_factor: logf is 1 ulp: b = (D + 3) u f / (f + 1e-8) + 2u |ref|.
- pose_inputs: the inverse quaternion is within 5u per component (sum of squares and the quotient); the Hamilton
  product adds 4 roundings over its terms: b_q = 10u (|q0^-1| x |q_v|) with x the Hamilton product of the absolute
  values.  R(q0^-1) is within 16u per entry after normalisation, and R t adds 3u: e_t = 19u (|t_v|_1 + |t_0|_1) + u |t|.
  The normaliser f = sum |t| / count has D = ceil(V / 256) + 13 summation roundings over the norms (each off by e_t)
  and 2 more roundings: e_f = (D u sum|t| + sum e_t) / sum|t| + 2u; the output t / f: b = e_t / f + |ref| (e_f + u);
  log_scale: b = (e_f + 2u) + 2u |ref|.  Views without a pose are exactly (0, 0, 0, 1) / 0 and padding is exactly 0.
- fuse_add: gates are 0 or 1, so each term is added exactly in the kernel's order
  x = ((feat + a) + b) + (((g0 + g1) + g2) + g3): compared bit for bit with that order in torch, and with fp64
  under b = 6u sum|terms|.

postprocess.cu:
- denorm_image, apply_mask, mask_and: bit exact with torch float32 in the kernel's operation order.
- pose_matrices: normalised components within 4.5u; each product within 10u; the entry 1 - 2 (t1 + t2) or
  2 (t1 +- t2) within 22u (|t1| + |t2|) + u |ref|: b = 24u (|t1| + |t2|) + 2u |ref|.  Translations bit exact.
- depthmap_to_world: the camera frame is bit exact with oracle.geometry.depthmap_to_camera_frame (fp32, 3 roundings
  each); the world frame adds 3 products and 3 sums: b = sum_k |p_k| e_k + 4u sum_k |p_k c_k| with e = 3u |cam|.
- intrinsics_from_rays: the least-squares branch accumulates in double and only the fp32 ratios r = p[0] / p[2]
  (|dr| <= u |r|) matter: for x = c + f r the slope moves by f cov(dr, r) / var(r) <= u f A with
  A = mean(|r| |r - mean r|) / var(r), the intercept by |df| |mean r| + u f mean|r|; both doubled for second order, plus
  the final float rounding.  The five-pixel branch (H W > 1e6) is fp32: each term (q - c) / (l - r_c) carries
  u (|l| + |r_c|) / |l - r_c| + 2u, the mean u more; cx = cw - fx r_c adds |dfx r_c| + 3u (|cw| + |fx r_c|); doubled.
- quantile_mask: thr_out equals torch.quantile value for value (==, so -0.0 == +0.0) on CPU, and on CUDA wherever CUDA
  torch agrees with CPU torch; the mask is bit exact with conf > thr.  A row holding a NaN has a NaN threshold, as CPU
  torch.quantile gives; CUDA torch.quantile returns a finite value for a row whose only NaN has its sign bit set, which
  the test prints and allows (it fails if CPU and CUDA torch ever disagree on a row without NaN).
- edge_mask: each pass is checked against oracle.geometry: normals, normal mask and depth edge bit for bit; the angle
  map within ANGLE_ULPS ulp of numpy's (acosf is within 2 ulp in CUDA, numpy's float32 arccos within 4 ulp on its
  SIMD paths: the dot products it is applied to are bit exact; 2 ulp were measured, so the angle is not bit exact); the
  final mask bit for bit on every pixel whose pooled numpy angle is farther than that bound from the threshold.

Each case prints its worst err / bound as "[family] ...".  Outputs hold a sentinel wherever the call must not write,
including one element past the end, checked bit for bit; inputs hold NaN past the end.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENTINEL = -77.0                 # exact in fp32 and bf16
BYTE_SENTINEL = 0xA5
F32, BF16 = torch.float32, torch.bfloat16
U = 2.0 ** -24
NAN = float("nan")
TINY = 2.0 ** -149
DEV = "cuda"
ANGLE_ULPS = 6


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _lib():
    from mapanything_b200 import _lib

    return _lib.load()


def _call(fn, *args):
    from mapanything_b200 import ops

    lib = _lib()
    rc = getattr(lib, fn)(*args, ops._stream())
    assert rc == 0, f"{fn}: {lib.ma_last_error().decode()}"
    torch.cuda.synchronize()


def _p(t):
    return None if t is None else t.data_ptr()


def _bits(t):
    return t.view({F32: torch.int32, BF16: torch.int16, torch.uint8: torch.uint8, torch.bool: torch.uint8}[t.dtype])


def _assert_bits(got, want, what, nan_equal=False):
    bad = _bits(got) != _bits(want)
    if nan_equal and got.is_floating_point():
        bad &= ~(torch.isnan(got) & torch.isnan(want))
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ, first at {list(i)}: "
                             f"{got[i].item()!r}, want {want[i].item()!r}")


def _sentinel_like(t):
    return torch.full_like(t, BYTE_SENTINEL if t.dtype == torch.uint8 else SENTINEL)


def _assert_tail(buf, n, what):
    """Everything of buf past its first n elements (flattened) holds the sentinel, bit for bit."""
    tail = buf.reshape(-1)[n:]
    bad = _bits(tail) != _bits(_sentinel_like(tail))
    if bad.any():
        raise AssertionError(f"{what}: {int(bad.sum())} elements past the output were written")


def _out(n, dtype=F32, extra=1):
    """Output buffer of n elements plus `extra` sentinel elements; returns (buffer, view of the first n)."""
    buf = torch.full((n + extra,), BYTE_SENTINEL if dtype == torch.uint8 else SENTINEL, device=DEV, dtype=dtype)
    return buf, buf[:n]


def _in(t, extra=None):
    """Copy of t in a buffer followed by `extra` (default: one element, or one leading-dim slab) of NaN."""
    flat = t.reshape(-1)
    extra = extra if extra is not None else (t[0].numel() if t.dim() > 1 else 1)
    buf = torch.full((flat.numel() + extra,), NAN if t.is_floating_point() else BYTE_SENTINEL, device=DEV, dtype=t.dtype)
    buf[:flat.numel()] = flat
    return buf[:flat.numel()].view(t.shape)


def _check(family, got, ref, bound, what):
    err = (got.double() - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    ratio = torch.nan_to_num(ratio, nan=math.inf)
    worst = ratio.max().item() if ratio.numel() else 0.0
    print(f"\n[{family}] {what}: worst err/bound {worst:.3g}", end="")
    if worst > 1.0:
        i = int(ratio.reshape(-1).argmax())
        raise AssertionError(f"{what}: element {i} = {got.reshape(-1)[i].item()!r}, reference {ref.reshape(-1)[i].item()!r}, "
                             f"bound {bound.reshape(-1)[i].item():.3g} (worst err/bound {worst:.3g})")
    return worst


def _rand_K(B, H, W, g):
    f = torch.rand(B, 2, device=DEV, generator=g) * 0.8 + 0.6
    K = torch.zeros(B, 3, 3, device=DEV)
    K[:, 0, 0] = f[:, 0] * max(H, W)
    K[:, 1, 1] = f[:, 1] * max(H, W) * 1.1
    K[:, 0, 2] = W * (0.3 + 0.4 * torch.rand(B, device=DEV, generator=g))
    K[:, 1, 2] = H * (0.3 + 0.4 * torch.rand(B, device=DEV, generator=g))
    K[:, 2, 2] = 1.0
    return K


def _rays64(K, H, W):
    K = K.double()
    xs = torch.arange(W, device=DEV, dtype=torch.float64)[None, None, :]
    ys = torch.arange(H, device=DEV, dtype=torch.float64)[None, :, None]
    xx = ((xs - K[:, 0, 2, None, None]) / K[:, 0, 0, None, None]).expand(-1, H, W)
    yy = ((ys - K[:, 1, 2, None, None]) / K[:, 1, 1, None, None]).expand(-1, H, W)
    d = torch.stack([xx, yy, torch.ones_like(xx)], -1)
    return d / d.norm(dim=-1, keepdim=True)


# ---- rays_from_intrinsics / normalize_rays / depth_z_to_along_ray ------------------------------------------------------


@pytest.mark.parametrize("B", [1, 5])
@pytest.mark.parametrize("H,W", [(518, 518), (294, 518), (1, 518), (294, 1), (37, 61)])
def test_rays_from_intrinsics(B, H, W):
    g = _gen(B * 7 + H * 3 + W)
    K = _in(_rand_K(B, H, W, g))
    P = B * H * W
    buf, out = _out(P * 3)
    _call("ma_rays_from_intrinsics", K.data_ptr(), out.data_ptr(), B, H, W)
    ref = _rays64(K, H, W).reshape(-1)
    big = " (grid-stride)" if P > _sms() * 16 * 256 else ""
    _check("rays", out, ref, 8 * U * ref.abs(), f"rays_from_intrinsics B={B} {H}x{W}{big}")
    _assert_tail(buf, P * 3, "rays_from_intrinsics")


@pytest.mark.parametrize("P", [1, 1000, 3 * 518 * 518])
def test_normalize_rays(P):
    g = _gen(P)
    x = torch.randn(P, 3, device=DEV, generator=g)
    scale = 10.0 ** -torch.randint(0, 13, (P, 1), device=DEV, generator=g).float()  # 1 .. 1e-12: +1e-8 dominates below
    x = x * scale
    x[::97] = 0.0
    x = _in(x)
    buf, out = _out(P * 3)
    _call("ma_normalize_rays", x.data_ptr(), out.data_ptr(), P)
    x64 = x.double()
    ref = (x64 / (x64.norm(dim=-1, keepdim=True) + float(np.float32(1e-8)))).reshape(-1)
    _check("normalize_rays", out, ref, 6 * U * ref.abs() + TINY, f"normalize_rays P={P}")
    _assert_tail(buf, P * 3, "normalize_rays")


@pytest.mark.parametrize("B,H,W", [(1, 37, 61), (3, 518, 518)])
def test_depth_z_to_along_ray(B, H, W):
    g = _gen(H * W + B)
    rays = _in(_rays64(_rand_K(B, H, W, g), H, W).float())
    d = torch.rand(B, H, W, device=DEV, generator=g) * 20
    d.view(-1)[::13] = 0.0
    d = _in(d)
    P = B * H * W
    buf, out = _out(P)
    _call("ma_depth_z_to_along_ray", d.data_ptr(), rays.data_ptr(), out.data_ptr(), P)
    r64 = rays.double()
    ref = (d.double() * r64.norm(dim=-1) / r64[..., 2].abs()).reshape(-1)
    _check("depth_along_ray", out, ref, 6 * U * ref.abs(), f"depth_z_to_along_ray {B}x{H}x{W}")
    _assert_tail(buf, P, "depth_z_to_along_ray")


# ---- pose_to_quat_trans -------------------------------------------------------------------------------------------------


def _rot(axis, deg):
    t = math.radians(deg)
    c, s = math.cos(t), math.sin(t)
    m = np.eye(3)
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    m[i, i], m[i, j], m[j, i], m[j, j] = c, -s, s, c
    return m


def _pose_cases():
    """(4,4) float32 matrices: rotations near 0 and 180 degrees about x, y and z with both signs (every branch and the
    w < 0 flip), random rotations, and non-orthogonal matrices whose sq candidates tie exactly (dyadic diagonals)."""
    rng = np.random.default_rng(5)
    mats = []
    for axis in range(3):
        for deg in (0.5, -0.5, 1.0, 179.0, -179.0, 179.9, -179.9, 120.0, -150.0):
            mats.append(_rot(axis, deg))
    for _ in range(40):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        x, y, z, w = q
        mats.append(np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                              [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                              [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]]))
    off = np.array([[0, 0.2, 0.1], [0.05, 0, -0.1], [-0.2, 0.3, 0]])
    for diag in ((1, 0, 0), (0, 1, 0), (0, 0, 1), (0.5, 0.5, -0.5), (-0.5, -0.5, 0.5), (0, 0, 0), (1, 1, 1), (-1, -1, -1),
                 (0.25, -0.25, 0.25)):
        for sgn in (1, -1):
            mats.append(np.diag(diag) + sgn * off)
    out = np.zeros((len(mats), 4, 4), dtype=np.float32)
    for i, m in enumerate(mats):
        out[i, :3, :3] = m
        out[i, :3, 3] = rng.normal(size=3) * 5
        out[i, 3] = (0.5, -0.25, 0.125, 1.0)   # never read
    return out


def test_pose_to_quat_trans():
    P = _pose_cases()
    B = P.shape[0]
    m32 = P[:, :3, :3].reshape(B, 9)
    m = m32.astype(np.float64)
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = m.T
    one = np.float32(1)
    d32 = [m32[:, i] for i in (0, 4, 8)]
    sq32 = np.stack([one + d32[0] + d32[1] + d32[2], one + d32[0] - d32[1] - d32[2],
                     one - d32[0] + d32[1] - d32[2], one - d32[0] - d32[1] + d32[2]], 1)
    qa32 = np.where(sq32 > 0, np.sqrt(np.maximum(sq32, 0)), 0).astype(np.float32)
    best = qa32.argmax(1)                                    # first maximum, as the kernel and torch.argmax
    sq = np.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22, 1 - m00 - m11 + m22], 1)
    qa = np.sqrt(np.maximum(sq, 0))
    srt = np.sort(qa, 1)
    tie = srt[:, -1] == srt[:, -2]
    assert (qa.argmax(1)[~tie] == best[~tie]).all(), "test matrices: fp32 and fp64 branch choice differ"
    assert set(best.tolist()) == {0, 1, 2, 3} and tie.sum() >= 6
    cand = np.stack([
        np.stack([qa[:, 0] ** 2, m21 - m12, m02 - m20, m10 - m01], 1),
        np.stack([m21 - m12, qa[:, 1] ** 2, m10 + m01, m02 + m20], 1),
        np.stack([m02 - m20, m10 + m01, qa[:, 2] ** 2, m12 + m21], 1),
        np.stack([m10 - m01, m20 + m02, m21 + m12, qa[:, 3] ** 2], 1)], 1)
    absn = np.stack([
        np.stack([0 * m00, abs(m21) + abs(m12), abs(m02) + abs(m20), abs(m10) + abs(m01)], 1),
        np.stack([abs(m21) + abs(m12), 0 * m00, abs(m10) + abs(m01), abs(m02) + abs(m20)], 1),
        np.stack([abs(m02) + abs(m20), abs(m10) + abs(m01), 0 * m00, abs(m12) + abs(m21)], 1),
        np.stack([abs(m10) + abs(m01), abs(m20) + abs(m02), abs(m21) + abs(m12), 0 * m00], 1)], 1)
    r = np.arange(B)
    qb = qa[r, best]
    den = 2 * np.maximum(qb, 0.1)
    c = cand[r, best] / den[:, None]                          # (w, x, y, z)
    flip = c[:, 0] < 0
    assert flip.any() and (~flip).any()
    c = np.where(flip[:, None], -c, c)
    ref = c[:, [1, 2, 3, 0]]
    S = 1 + abs(m00) + abs(m11) + abs(m22)
    e_qa = U + 3 * U * S / (2 * sq[r, best])
    e_num = U * absn[r, best]
    e_num[r, best] = qb ** 2 * (2 * e_qa + U)
    bound = 2 * (e_num / den[:, None] + np.abs(c) * (e_qa + U)[:, None])[:, [1, 2, 3, 0]]
    assert (np.abs(ref[:, 3]) > bound[:, 3]).all(), "test matrices: the sign of w is not decidable"
    poses = _in(torch.from_numpy(P).to(DEV))
    qbuf, q = _out(B * 4)
    tbuf, t = _out(B * 3)
    _call("ma_pose_to_quat_trans", poses.data_ptr(), q.data_ptr(), t.data_ptr(), B)
    _check("pose_to_quat", q, torch.from_numpy(ref).to(DEV).reshape(-1), torch.from_numpy(bound).to(DEV).reshape(-1),
           f"pose_to_quat_trans B={B} branches {np.bincount(best, minlength=4).tolist()} ties {int(tie.sum())}")
    _assert_bits(t, torch.from_numpy(np.ascontiguousarray(P[:, :3, 3])).to(DEV).reshape(-1), "pose_to_quat_trans trans")
    _assert_tail(qbuf, B * 4, "pose_to_quat_trans quats")
    _assert_tail(tbuf, B * 3, "pose_to_quat_trans trans")


# ---- unshuffle_split ----------------------------------------------------------------------------------------------------


def _unshuffle_ref(x, p):
    """(n,H,W,cin) -> (n,H/p,W/p,cin*p*p), channel k = c*p*p + dy*p + dx (nn.PixelUnshuffle on the NCHW tensor)."""
    n, H, W, cin = x.shape
    t = x.reshape(n, H // p, p, W // p, p, cin).permute(0, 1, 3, 5, 2, 4)
    return t.reshape(n, H // p, W // p, cin * p * p)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("p,cin,extra_pad", [(14, 3, 0), (14, 1, 8), (8, 3, 0), (8, 1, 8), (14, 3, 16), (8, 1, 0)])
@pytest.mark.parametrize("n,hp,wp", [(1, 37, 37), (3, 5, 3)])
def test_unshuffle_split(mode, p, cin, extra_pad, n, hp, wp):
    """hi / lo / hi bit exact on the kernel's fp32 v; zero padding; several views with different factors."""
    g = _gen(mode * 1000 + p * 10 + cin + extra_pad + n * 77 + hp)
    H, W = hp * p, wp * p
    kk = cin * p * p
    cpad = (kk + 7) // 8 * 8 + extra_pad
    x = torch.randn(n, H, W, cin, device=DEV, generator=g) * 3
    factor = None
    if mode == 1:
        x = x.abs() * 4
        x.view(-1)[::11] = 0.0                                        # zero-depth pixels
        x.view(-1)[5::23] *= 1e-9                                     # |v| < 1e-8 after the division
        factor = _in(torch.rand(n, device=DEV, generator=g) * 5 + 0.25)
    x = _in(x)
    rows = n * hp * wp
    buf, out = _out(rows * 3 * cpad, dtype=BF16, extra=3 * cpad)
    _call("ma_unshuffle_split", x.data_ptr(), out.data_ptr(), n, H, W, cin, p, cpad, mode, _p(factor))
    out = out.view(rows, 3, cpad)
    v = _unshuffle_ref(x, p).reshape(rows, kk)
    if mode == 1:   # the kernel's fp32 chain, same operation order (torch.log1p is CUDA's log1pf)
        inv_f = (1.0 / factor).repeat_interleave(hp * wp)[:, None]
        v1 = v * inv_f
        a = v1.abs()
        v = v1 / a.clamp(min=1e-8) * torch.log1p(a)
        x64 = _unshuffle_ref(x.double(), p).reshape(rows, kk) / factor.double().repeat_interleave(hp * wp)[:, None]
        ref = x64 / x64.abs().clamp(min=1e-8) * torch.log1p(x64.abs())
        _check("unshuffle", v, ref, 8 * U * ref.abs() + TINY, f"unshuffle mode 1 fp32 chain p={p} cin={cin}")
    hi = v.to(BF16)
    lo = (v - hi.float()).to(BF16)
    want = torch.zeros(rows, 3, cpad, device=DEV, dtype=BF16)
    want[:, 0, :kk], want[:, 1, :kk], want[:, 2, :kk] = hi, lo, hi
    what = f"unshuffle mode {mode} p={p} cin={cin} cpad={cpad} n={n} {hp}x{wp}"
    _assert_bits(out, want, what)
    if mode == 1:
        got = out[:, 0, :kk].double() + out[:, 1, :kk].double()
        _check("unshuffle", got, ref, (8 * U + 2.0 ** -16) * ref.abs() + TINY, what + " hi + lo")
    _assert_tail(buf, rows * 3 * cpad, what)


# ---- depth_factor -------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("per_view", [1, 2, 1023, 1024, 1025, 4099, 518 * 518, 518 * 518 + 7])
def test_depth_factor(per_view):
    """Views: positive depths with zeros and negatives, all zero, all negative, one positive pixel at the end."""
    g = _gen(per_view)
    n = 5
    d = torch.rand(n, per_view, device=DEV, generator=g) * 10 + 0.1
    d[0, ::3] = 0.0
    d[0, 1::7] = -d[0, 1::7]
    d[1] = 0.0
    d[2] = -d[2]
    d[3, :-1] = 0.0
    d[4] = d[4] * 1e3
    d[4, ::2] = 0.0
    d = _in(d)
    fbuf, f = _out(n)
    lbuf, lf = _out(n * 8)
    _call("ma_depth_factor", d.data_ptr(), n, per_view, f.data_ptr(), lf.data_ptr())
    d64 = d.double()
    pos = d64 > 0
    f_ref = ((d64 * pos).sum(1) / (pos.sum(1) + 1e-8)).clamp(min=1e-8)
    D = -(-per_view // 1024) + 37
    _check("depth_factor", f, f_ref, (D + 2) * U * f_ref, f"depth_factor factor per_view={per_view}")
    lf = lf.view(n, 8)
    l_ref = torch.log(f_ref + 1e-8)
    _check("depth_factor", lf[:, 0], l_ref, (D + 3) * U * f_ref / (f_ref + 1e-8) + 2 * U * l_ref.abs(),
           f"depth_factor log per_view={per_view}")
    assert f[1].item() == np.float32(1e-8) and f[2].item() == np.float32(1e-8), "all-zero / all-negative views: clip to 1e-8"
    _assert_bits(lf[:, 1:], torch.zeros(n, 7, device=DEV), "depth_factor padding")
    _assert_tail(fbuf, n, "depth_factor factor")
    _assert_tail(lbuf, n * 8, "depth_factor log_factor8")


# ---- pose_inputs --------------------------------------------------------------------------------------------------------


def _qmul(a, b):
    x1, y1, z1, w1 = a.unbind(-1)
    x2, y2, z2, w2 = b.unbind(-1)
    return torch.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                        w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], -1)


def _qmul_abs(a, b):
    a, b = a.abs(), b.abs()
    x1, y1, z1, w1 = a.unbind(-1)
    x2, y2, z2, w2 = b.unbind(-1)
    return torch.stack([w1 * x2 + x1 * w2 + y1 * z2 + z1 * y2, w1 * y2 + x1 * z2 + y1 * w2 + z1 * x2,
                        w1 * z2 + x1 * y2 + y1 * x2 + z1 * w2, w1 * w2 + x1 * x2 + y1 * y2 + z1 * z2], -1)


@pytest.mark.parametrize("V", [1, 9, 256, 257, 1000])
def test_pose_inputs(V):
    """Against oracle.geometry.relative_pose_2_to_1 + normalize_pose_translations in fp64.  View 0's quaternion is not
    unit; some views have no pose; some repeat view 0's pose, whose zero translation must not count toward the mean."""
    from oracle.geometry import normalize_pose_translations, relative_pose_2_to_1

    g = _gen(V)
    q = torch.randn(V, 4, device=DEV, generator=g)
    q = q / q.norm(dim=1, keepdim=True) * (torch.rand(V, 1, device=DEV, generator=g) * 1.5 + 0.5)
    q[0] *= 1.7
    t = torch.randn(V, 3, device=DEV, generator=g) * 4
    has = (torch.rand(V, device=DEV, generator=g) > 0.25).to(torch.uint8)
    has[0] = 1
    if V > 2:
        q[2], t[2], has[2] = q[0], t[0], 1
    if V > 8:
        q[7], t[7], has[7] = q[0] * 2, t[0], 1
        has[8] = 0
    qi, ti, hi = _in(q), _in(t), _in(has)
    bufs = [_out(V * 8) for _ in range(3)]
    (qb, q8), (tb, t8), (sb, s8) = bufs
    _call("ma_pose_inputs", qi.data_ptr(), ti.data_ptr(), hi.data_ptr(), V, q8.data_ptr(), t8.data_ptr(), s8.data_ptr())
    q8, t8, s8 = q8.view(V, 8), t8.view(V, 8), s8.view(V, 8)
    q64, t64 = q.double(), t.double()
    q0, t0 = q64[:1].expand(V, 4), t64[:1].expand(V, 3)
    qr, tr = relative_pose_2_to_1(q0, t0, q64, t64)
    on = has.bool()[:, None]
    qr = torch.where(on, qr, torch.tensor([0.0, 0, 0, 1], device=DEV, dtype=torch.float64))
    tr = torch.where(on, tr, torch.zeros_like(tr))
    tn, f = normalize_pose_translations(tr[None])
    tn, f = tn[0], f[0]
    qinv = torch.cat([-q64[:1, :3], q64[:1, 3:]], 1) / (q64[:1] ** 2).sum()
    b_q = 10 * U * _qmul_abs(qinv.expand(V, 4), q64)
    e_t = 19 * U * (t64.abs().sum(1, keepdim=True) + t64[:1].abs().sum()) + U * tr.abs()
    e_t = torch.where(on, e_t, torch.zeros_like(e_t))
    dist = tr.norm(dim=1)
    D = -(-V // 256) + 13
    e_f = (D * U * dist.sum() + e_t.norm(dim=1).sum()) / dist.sum().clamp(min=1e-300) + 2 * U
    b_t = e_t / f + tn.abs() * (e_f + U)
    what = f"pose_inputs V={V} ({int(has.sum())} posed)"
    _check("pose_inputs", q8[:, :4], qr, b_q, what + " quats")
    _check("pose_inputs", t8[:, :3], tn, b_t, what + " trans")
    lf = torch.log(f + 1e-8)
    _check("pose_inputs", s8[:, 0], lf.expand(V), (e_f + 2 * U) + 2 * U * lf.abs(), what + " log scale")
    off = ~on[:, 0]
    _assert_bits(q8[off, :4], torch.tensor([0.0, 0, 0, 1], device=DEV).expand(int(off.sum()), 4), what + " unposed quats")
    _assert_bits(t8[off, :3], torch.zeros(int(off.sum()), 3, device=DEV), what + " unposed trans")
    _assert_bits(t8[0, :3], torch.zeros(3, device=DEV), what + " view 0 trans")
    if V > 8:
        _assert_bits(t8[[2, 7], :3], torch.zeros(2, 3, device=DEV), what + " trans of the repeated view-0 pose")
    _assert_bits(q8[:, 4:], torch.zeros(V, 4, device=DEV), what + " quats8 padding")
    _assert_bits(t8[:, 3:], torch.zeros(V, 5, device=DEV), what + " trans8 padding")
    _assert_bits(s8[:, 1:], torch.zeros(V, 7, device=DEV), what + " log_scale8 padding")
    for b, name in ((qb, "quats8"), (tb, "trans8"), (sb, "log_scale8")):
        _assert_tail(b, V * 8, what + " " + name)


# ---- fuse_add -----------------------------------------------------------------------------------------------------------


def _run_fuse(V, N, C, a_slot, b_slot, present, gates, seed, g_rows=None):
    """present: which of (dense_a, dense_b, g0, g1, g2, g3) are passed; gates [4][V] of 0 / 1."""
    g = _gen(seed)
    T = V * N
    fbuf = torch.full(((T + 1) * C,), SENTINEL, device=DEV)
    feat = fbuf[:T * C].view(T, C)
    feat.copy_(torch.randn(T, C, device=DEV, generator=g))
    feat[::5, ::7] = -0.0
    ref_feat = feat.clone()
    n_a = int((a_slot >= 0).sum()) if a_slot is not None else 0
    n_b = int((b_slot >= 0).sum()) if b_slot is not None else 0
    dense_a = _in(torch.randn(n_a * N, C, device=DEV, generator=g)) if present[0] else None
    dense_b = _in(torch.randn(n_b * N, C, device=DEV, generator=g) * 10) if present[1] else None
    G = []
    for j in range(4):
        rows = (n_b if j == 3 else V) if g_rows is None else g_rows[j]
        G.append(_in(torch.randn(rows, C, device=DEV, generator=g) * (j + 1), extra=V * C) if present[2 + j] else None)
    gw = _in(torch.tensor(gates, dtype=torch.float32, device=DEV))
    a_t = _in(a_slot.to(DEV)) if dense_a is not None else None
    b_t = _in(b_slot.to(DEV)) if (dense_b is not None or present[5]) and b_slot is not None else None
    _call("ma_fuse_add", feat.data_ptr(), V, N, C, _p(dense_a), _p(a_t), _p(dense_b), _p(b_t), *(_p(x) for x in G),
          gw.data_ptr() if any(x is not None for x in G) else None)
    # the kernel's order in fp32, and the fp64 sum with the magnitudes of its terms
    x = ref_feat.view(V, N, C)
    x64, mag = x.double(), x.double().abs()
    v = torch.arange(V, device=DEV)
    if dense_a is not None:
        use = (a_t >= 0)[:, None, None]
        add = dense_a.view(-1, N, C)[a_t.long().clamp(min=0)] if n_a else torch.zeros_like(x)
        x = torch.where(use, x + add, x)
        x64, mag = x64 + use * add.double(), mag + use * add.double().abs()
    if dense_b is not None:
        use = (b_t >= 0)[:, None, None]
        add = dense_b.view(-1, N, C)[b_t.long().clamp(min=0)] if n_b else torch.zeros_like(x)
        x = torch.where(use, x + add, x)
        x64, mag = x64 + use * add.double(), mag + use * add.double().abs()
    gs = torch.zeros(V, 1, C, device=DEV)
    anyg = torch.zeros(V, 1, 1, dtype=torch.bool, device=DEV)
    for j in range(4):
        if G[j] is None:
            continue
        gv = (b_t.long() if b_t is not None else torch.full_like(v, -1)) if j == 3 else v
        use = ((gw[j] != 0) & (gv >= 0))[:, None, None]
        rows = G[j][gv.clamp(min=0)][:, None, :]
        gs = torch.where(use, gs + gw[j][:, None, None] * rows, gs)
        anyg |= use
        x64, mag = x64 + use * rows.double(), mag + use * rows.double().abs()
    x = torch.where(anyg, x + gs, x)
    return fbuf, feat, x.reshape(T, C), x64.reshape(T, C), mag.reshape(T, C)


A_SLOT = torch.tensor([2, -1, 0, 1, -1], dtype=torch.int32)
B_SLOT = torch.tensor([-1, 1, 0, -1, 2], dtype=torch.int32)
GATES = [[1, 0, 1, 1, 1], [1, 1, 0, 1, 1], [0, 1, 1, 1, 0], [1, 1, 1, 1, 1]]


def _fuse_check(fbuf, feat, want, x64, mag, what):
    T, C = feat.shape
    _assert_bits(feat, want, what)
    _check("fuse_add", feat, x64, 6 * U * mag, what)
    _assert_tail(fbuf, T * C, what)


@pytest.mark.parametrize("combo", range(64))
def test_fuse_add_operand_combinations(combo):
    """Every subset of dense_a, dense_b, g0..g3; slot tables with -1 in non-monotone order; g3 read through b_slot."""
    present = [bool(combo >> i & 1) for i in range(6)]
    fbuf, feat, want, x64, mag = _run_fuse(5, 37, 64, A_SLOT, B_SLOT, present, GATES, combo)
    _fuse_check(fbuf, feat, want, x64, mag, f"fuse_add present={''.join('1' if p else '0' for p in present)}")


@pytest.mark.parametrize("V,N,C", [(3, 100, 64), (5, 1369, 1024)])
def test_fuse_add_grid_cap(V, N, C):
    """V N C / 4 below and above the SMs x 16 x 256 grid cap (the grid-stride loop)."""
    fbuf, feat, want, x64, mag = _run_fuse(V, N, C, A_SLOT[:V] if V == 5 else torch.tensor([1, -1, 0], dtype=torch.int32),
                                           B_SLOT[:V] if V == 5 else torch.tensor([0, 1, -1], dtype=torch.int32),
                                           [True] * 6, [r[:V] for r in GATES], V * 1000 + N)
    cap = " (above the grid cap)" if V * N * C // 4 > _sms() * 16 * 256 else ""
    _fuse_check(fbuf, feat, want, x64, mag, f"fuse_add V={V} N={N} C={C}{cap}")


@pytest.mark.parametrize("V", [2, 9])
def test_fuse_add_view_pe(V):
    """The view-index PE call of Engine.info_sharing: feat = y[:V N] (D = 1024), globals_ = [table rows, -, -, -],
    gate 1 for views with a PE row and 0 for the others; no dense addends, no slot tables."""
    N, C = 1369, 1024
    gates = [[1 if v % 3 != 1 else 0 for v in range(V)], [0] * V, [0] * V, [0] * V]
    fbuf, feat, want, x64, mag = _run_fuse(V, N, C, None, None, [False, False, True, False, False, False], gates, V,
                                           g_rows=[V, 0, 0, 0])
    _fuse_check(fbuf, feat, want, x64, mag, f"fuse_add view PE V={V}")


# ---- denorm_image / apply_mask / mask_and -------------------------------------------------------------------------------


MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


@pytest.mark.parametrize("n,H,W", [(2, 518, 518), (3, 294, 518), (1, 1, 7)])
def test_denorm_image(n, H, W):
    """Bit exact: clip(img * std + mean, 0, 1) with separate roundings, NCHW -> NHWC; 518x518 exceeds the 1024-block cap."""
    g = _gen(n * H * W)
    img = _in(torch.randn(n, 3, H, W, device=DEV, generator=g) * 3)
    buf, out = _out(n * H * W * 3)
    _call("ma_denorm_image", img.data_ptr(), out.data_ptr(), n, H, W, (C.c_float * 3)(*MEAN), (C.c_float * 3)(*STD))
    s = torch.tensor(STD, device=DEV).view(1, 3, 1, 1)
    m = torch.tensor(MEAN, device=DEV).view(1, 3, 1, 1)
    want = (img * s + m).clamp(0, 1).permute(0, 2, 3, 1).reshape(-1)
    _assert_bits(out, want, f"denorm_image {n}x{H}x{W}")
    _assert_tail(buf, n * H * W * 3, "denorm_image")


@pytest.mark.parametrize("stride,offset,width", [(3, 0, 3), (3, 2, 1), (1, 0, 1), (5, 1, 3), (4, 0, 4)])
@pytest.mark.parametrize("pixels", [1000, 2 * 518 * 518])
def test_apply_mask(stride, offset, width, pixels):
    """Bit exact in[px * stride + offset + c] * (mask ? 1 : 0) (so -x -> -0.0, inf -> NaN outside the mask)."""
    g = _gen(stride * 100 + offset * 10 + width + pixels)
    x = torch.randn(pixels, stride, device=DEV, generator=g) * 5
    x.view(-1)[::17] = math.inf
    x.view(-1)[3::29] = -0.0
    x = _in(x)
    mask = _in((torch.rand(pixels, device=DEV, generator=g) > 0.3).to(torch.uint8) * torch.randint(
        1, 256, (pixels,), device=DEV, generator=g, dtype=torch.uint8))
    buf, out = _out(pixels * width)
    _call("ma_apply_mask", x.data_ptr(), stride, offset, mask.data_ptr(), out.data_ptr(), pixels, width)
    want = (x[:, offset:offset + width] * (mask != 0).float()[:, None]).reshape(-1)
    cap = " (above the grid cap)" if pixels * width > 148 * 16 * 256 else ""
    _assert_bits(out, want, f"apply_mask stride={stride} offset={offset} width={width} pixels={pixels}{cap}", nan_equal=True)
    _assert_tail(buf, pixels * width, "apply_mask")


@pytest.mark.parametrize("n", [1, 1000, 3 * 518 * 518])
def test_mask_and(n):
    g = _gen(n)
    a = _in(torch.randint(0, 4, (n,), device=DEV, generator=g, dtype=torch.uint8) * 85)   # 0, 85, 170, 255
    b = _in(torch.randint(0, 3, (n,), device=DEV, generator=g, dtype=torch.uint8))
    buf, out = _out(n, dtype=torch.uint8)
    _call("ma_mask_and", a.data_ptr(), b.data_ptr(), out.data_ptr(), n)
    _assert_bits(out, ((a != 0) & (b != 0)).to(torch.uint8), f"mask_and n={n}")
    _assert_tail(buf, n, "mask_and")


# ---- pose_matrices / depthmap_to_world ----------------------------------------------------------------------------------


@pytest.mark.parametrize("n", [1, 129, 300])
def test_pose_matrices(n):
    g = _gen(n)
    q = torch.randn(n, 4, device=DEV, generator=g) * 10.0 ** torch.randint(-2, 3, (n, 1), device=DEV, generator=g).float()
    t = torch.randn(n, 3, device=DEV, generator=g) * 7
    qi, ti = _in(q), _in(t)
    buf, out = _out(n * 16)
    _call("ma_pose_matrices", qi.data_ptr(), ti.data_ptr(), out.data_ptr(), n)
    out = out.view(n, 4, 4)
    qn = q.double() / q.double().norm(dim=1, keepdim=True)
    x, y, z, w = qn.abs().unbind(1)
    terms = torch.stack([y * y + z * z, x * y + w * z, x * z + w * y,
                         x * y + w * z, x * x + z * z, y * z + w * x,
                         x * z + w * y, y * z + w * x, x * x + y * y], 1).view(n, 3, 3)
    from oracle.geometry import quat_to_rotmat

    R = quat_to_rotmat(q.double())
    _check("pose_matrices", out[:, :3, :3], R, 24 * U * terms + 2 * U * R.abs(), f"pose_matrices n={n}")
    _assert_bits(out[:, :3, 3], t, "pose_matrices translation")
    _assert_bits(out[:, 3], torch.tensor([0.0, 0, 0, 1], device=DEV).expand(n, 4), "pose_matrices last row")
    _assert_tail(buf, n * 16, "pose_matrices")


@pytest.mark.parametrize("with_pose", [True, False])
@pytest.mark.parametrize("with_valid", [True, False])
@pytest.mark.parametrize("n,H,W", [(3, 294, 518), (1, 1, 7), (2, 37, 1)])
def test_depthmap_to_world(n, H, W, with_pose, with_valid):
    from oracle.geometry import depthmap_to_camera_frame, quat_to_rotmat

    g = _gen(n * H * W + with_pose * 2 + with_valid)
    K = _in(_rand_K(n, H, W, g))
    depth = torch.rand(n, H, W, device=DEV, generator=g) * 30
    depth.view(-1)[::7] = 0.0
    depth.view(-1)[3::11] *= -1
    depth = _in(depth)
    pose = None
    if with_pose:
        P = torch.eye(4, device=DEV).repeat(n, 1, 1)
        P[:, :3, :3] = quat_to_rotmat(torch.randn(n, 4, device=DEV, generator=g))
        P[:, :3, 3] = torch.randn(n, 3, device=DEV, generator=g) * 10
        P[:, 3] = torch.tensor([0.5, -2.0, 3.0, 7.0], device=DEV)     # never read: the 3x4 part only
        pose = _in(P)
    pbuf, pts = _out(n * H * W * 3)
    vbuf, valid = _out(n * H * W, dtype=torch.uint8) if with_valid else (None, None)
    _call("ma_depthmap_to_world", depth.data_ptr(), K.data_ptr(), _p(pose), pts.data_ptr(), _p(valid), n, H, W)
    pts = pts.view(n, H, W, 3)
    cam, v_ref = depthmap_to_camera_frame(depth.cpu(), K.cpu())
    what = f"depthmap_to_world n={n} {H}x{W} pose={with_pose} valid={with_valid}"
    if not with_pose:
        _assert_bits(pts.cpu(), cam, what + " camera frame")
    else:
        c64 = torch.cat([cam.double(), torch.ones_like(cam[..., :1]).double()], -1).to(DEV)
        x64 = depth.double()
        xs = torch.arange(W, device=DEV, dtype=torch.float64)[None, None, :]
        ys = torch.arange(H, device=DEV, dtype=torch.float64)[None, :, None]
        K64 = K.double()
        exact = torch.stack([(xs - K64[:, 0, 2, None, None]) * x64 / K64[:, 0, 0, None, None],
                             (ys - K64[:, 1, 2, None, None]) * x64 / K64[:, 1, 1, None, None], x64,
                             torch.ones_like(x64)], -1)
        P64 = pose.double()[:, :3]
        ref = torch.einsum("bik,bhwk->bhwi", P64, exact)
        e_cam = torch.stack([3 * U * exact[..., 0].abs(), 3 * U * exact[..., 1].abs(), torch.zeros_like(x64),
                             torch.zeros_like(x64)], -1)
        bound = torch.einsum("bik,bhwk->bhwi", P64.abs(), e_cam) + 4 * U * torch.einsum("bik,bhwk->bhwi", P64.abs(), c64.abs())
        _check("depthmap_to_world", pts, ref, bound, what + " world frame")
    _assert_tail(pbuf, n * H * W * 3, what + " pts")
    if with_valid:
        _assert_bits(valid.view(n, H, W).cpu(), v_ref.to(torch.uint8), what + " valid")
        _assert_tail(vbuf, n * H * W, what + " valid")


# ---- intrinsics_from_rays -----------------------------------------------------------------------------------------------


def _ls_ref(rays, H, W):
    """fp64 solve of the sampled system and its bound (module docstring)."""
    sh, sw = max(1, H // 50), max(1, W // 50)
    hi = torch.arange(0, H, sh, device=DEV)
    wi = torch.arange(0, W, sw, device=DEV)
    s = rays.double()[:, hi[:, None], wi[None, :], :]
    n = rays.shape[0]
    out = []
    for ratio, coord in ((s[..., 0] / s[..., 2], wi.double()[None, None, :].expand(n, len(hi), len(wi))),
                         (s[..., 1] / s[..., 2], hi.double()[None, :, None].expand(n, len(hi), len(wi)))):
        r = ratio.reshape(n, -1)
        x = coord.reshape(n, -1)
        rm, xm = r.mean(1, keepdim=True), x.mean(1, keepdim=True)
        var = ((r - rm) ** 2).mean(1)
        f = ((r - rm) * (x - xm)).mean(1) / var
        c = xm[:, 0] - f * rm[:, 0]
        A = (r.abs() * (r - rm).abs()).mean(1) / var
        bf = 2 * U * A * f.abs() + U * f.abs()
        bc = 2 * (bf * rm[:, 0].abs() + f.abs() * U * r.abs().mean(1)) + U * c.abs()
        out.append((f, c, bf, bc))
    return out


def _five_ref(rays, H, W):
    ch, cw, qw, tqw, qh, tqh = H // 2, W // 2, W // 4, 3 * W // 4, H // 4, 3 * H // 4
    r = rays.double()

    def at(y, x, k):
        return r[:, y, x, k] / r[:, y, x, 2]

    out = []
    for k, cc, a, b, pts in ((0, cw, qw, tqw, ((ch, qw), (ch, tqw))), (1, ch, qh, tqh, ((qh, cw), (tqh, cw)))):
        rc = at(ch, cw, k)
        l1, l2 = at(*pts[0], k), at(*pts[1], k)
        t1, t2 = (a - cc) / (l1 - rc), (b - cc) / (l2 - rc)
        f = (t1 + t2) / 2
        c = cc - f * rc
        e1 = (U * (l1.abs() + rc.abs()) / (l1 - rc).abs() + 2 * U) * t1.abs()
        e2 = (U * (l2.abs() + rc.abs()) / (l2 - rc).abs() + 2 * U) * t2.abs()
        bf = 2 * ((e1 + e2) / 2 + U * f.abs())
        bc = 2 * (bf * rc.abs() + 3 * U * (cc + (f * rc).abs()))
        out.append((f, c, bf, bc))
    return out


@pytest.mark.parametrize("n,H,W", [(3, 37, 61), (2, 518, 294), (3, 101, 149), (1, 49, 50), (2, 294, 518), (2, 1024, 1024)])
def test_intrinsics_from_rays(n, H, W):
    """Least squares below 1 MP (H or W < 50, sizes not multiples of 50), the five-pixel closed form above; several views
    with different K each."""
    g = _gen(n * H + W)
    K = _rand_K(n, H, W, g)
    rays = _in(_rays64(K, H, W).float())
    buf, out = _out(n * 9)
    _call("ma_intrinsics_from_rays", rays.data_ptr(), out.data_ptr(), n, H, W)
    out = out.view(n, 3, 3)
    five = H * W > 1_000_000
    (fx, cx, bfx, bcx), (fy, cy, bfy, bcy) = (_five_ref if five else _ls_ref)(rays, H, W)
    what = f"intrinsics_from_rays n={n} {H}x{W} ({'five-pixel' if five else 'least squares'})"
    got = torch.stack([out[:, 0, 0], out[:, 0, 2], out[:, 1, 1], out[:, 1, 2]], 1)
    _check("intrinsics", got, torch.stack([fx, cx, fy, cy], 1), torch.stack([bfx, bcx, bfy, bcy], 1), what)
    fixed = out.clone()
    fixed[:, 0, 0] = fixed[:, 0, 2] = fixed[:, 1, 1] = fixed[:, 1, 2] = 0
    want = torch.zeros(n, 3, 3, device=DEV)
    want[:, 2, 2] = 1
    _assert_bits(fixed, want, what + " zeros and K[2][2]")
    _assert_tail(buf, n * 9, what)


# ---- quantile_mask ------------------------------------------------------------------------------------------------------


def _quantile_case(name):
    """(conf (images, per_image) fp32 on the GPU, q)."""
    g = _gen(sum(map(ord, name)))
    rn = lambda *s: torch.randn(*s, device=DEV, generator=g)  # noqa: E731
    if name.startswith("n1_"):
        return rn(4, 1), float(name[3:])
    if name.startswith("n2_"):
        return rn(8, 2), float(name[3:])
    if name.startswith("random_"):                            # 2 % of rows round differently with two roundings
        return rn(256, 257) * 10.0 ** torch.randint(-3, 4, (256, 1), device=DEV, generator=g).float(), float(name[7:])
    if name.startswith("ties_"):                              # the order statistics fall inside and across tie runs
        vals = torch.tensor([-1.0, -0.0, 0.0, 0.5, 0.5000001, 2.0], device=DEV)
        return vals[torch.randint(0, 6, (64, 1000), device=DEV, generator=g)], float(name[5:])
    if name.startswith("inf_"):
        x = rn(16, 100)
        x[:, ::9] = math.inf
        x[:, 4::13] = -math.inf
        x[0] = math.inf
        x[1] = -math.inf
        return x, float(name[4:])
    if name == "nan_rows":
        x = rn(6, 333)
        x[1, 17] = NAN
        x[3, 0] = -NAN
        x[4, :] = NAN
        return x, 0.75
    if name.startswith("big_"):                              # 518 x 518 per image, three kinds of content
        x = rn(3, 518 * 518)
        x[1] = torch.exp(x[1] * 3)
        x[2] = torch.round(x[2] * 4) / 4
        return x, float(name[4:])
    raise ValueError(name)


QUANTILE_CASES = ([f"n1_{q}" for q in (0.0, 0.5, 1.0)] + [f"n2_{q}" for q in (0.0, 0.3, 0.5, 0.7, 1.0)] +
                  [f"random_{q}" for q in (0.37, 0.9, 0.05)] + [f"ties_{q}" for q in (0.0, 0.37, 0.5, 0.81, 1.0)] +
                  [f"inf_{q}" for q in (0.0, 0.2, 0.5, 0.999, 1.0)] + ["nan_rows"] + [f"big_{q}" for q in (0.1, 0.9)])


def _same(a, b):
    return (a == b) | (torch.isnan(a) & torch.isnan(b))


@pytest.mark.parametrize("case", QUANTILE_CASES)
def test_quantile_mask(case):
    """thr_out equals torch.quantile value for value on CPU and on CUDA; mask = conf > thr bit for bit."""
    x, q = _quantile_case(case)
    n, per = x.shape
    xi = _in(x)
    mbuf, mask = _out(n * per, dtype=torch.uint8)
    tbuf, thr = _out(n)
    _call("ma_quantile_mask", xi.data_ptr(), mask.data_ptr(), thr.data_ptr(), n, per, q)
    got = thr.cpu()
    cpu = torch.quantile(x.cpu(), q, dim=1)
    cuda = torch.quantile(x, q, dim=1).cpu()
    torch_agree = _same(cpu, cuda)
    bad_cpu, bad_cuda = ~_same(got, cpu), ~_same(got, cuda) & torch_agree
    if bad_cpu.any() or bad_cuda.any():
        i = int((bad_cpu | bad_cuda).nonzero()[0])
        raise AssertionError(
            f"quantile {case}: thr_out differs from CPU torch.quantile in {int(bad_cpu.sum())} of {n} images and from "
            f"CUDA torch.quantile in {int((~_same(got, cuda)).sum())} (CPU and CUDA torch disagree in "
            f"{int((~torch_agree).sum())}); first at image {i}: {got[i].item()!r}, CPU {cpu[i].item()!r}, CUDA {cuda[i].item()!r}")
    for i in (~torch_agree).nonzero()[:, 0].tolist():   # the kernel equals CPU torch here: CUDA torch is the one that differs
        nan_sign = "a NaN with the sign bit set" if (torch.isnan(x[i]) & torch.signbit(x[i])).any() else "no negative NaN"
        print(f"\n[quantile] {case} image {i} ({nan_sign}): CUDA torch.quantile gives {cuda[i].item()!r}, CPU torch and the "
              f"kernel {cpu[i].item()!r}", end="")
        assert torch.isnan(x[i]).any(), f"quantile {case} image {i}: CPU and CUDA torch.quantile disagree on a row without NaN"
    want = (x > cpu.to(DEV)[:, None]).to(torch.uint8).reshape(-1)
    _assert_bits(mask, want, f"quantile {case} mask")
    if case == "nan_rows":
        assert not mask.view(n, per)[[1, 3, 4]].any()
    _assert_tail(mbuf, n * per, f"quantile {case} mask")
    _assert_tail(tbuf, n, f"quantile {case} thr_out")


# ---- edge_mask ----------------------------------------------------------------------------------------------------------


TOL_DEG, RTOL = 5.0, 0.03


def _edge_scene(n, H, W, seed):
    """Camera-frame point grids with creases of 4.9, 5.1, 9.8 and 10.2 degrees and a sweep from 2 to 14 degrees (row
    bands), depth steps of 2.9 % and 3.1 %, zero-depth pixels, and masks with random and rectangular holes.  The world
    points are a rigid motion of them in fp32."""
    g = torch.Generator().manual_seed(seed)
    ys = torch.arange(H, dtype=torch.float64)[:, None].expand(H, W)
    xs = torch.arange(W, dtype=torch.float64)[None, :].expand(H, W)
    band = (ys * 5 // max(H, 1)).long()
    sweep = 2.0 + 12.0 * ys / max(H - 1, 1)
    theta = torch.tensor([4.9, 5.1, 9.8, 10.2, 0.0], dtype=torch.float64)[band.clamp(max=4)]
    theta = torch.where(band >= 4, sweep, theta)
    s = 0.01
    X, Y = (xs - W / 2) * s, (ys - H / 2) * s
    x0 = W // 2
    pts, masks = [], []
    for v in range(n):
        Z = 2.0 + 0.3 * v + torch.tan(torch.deg2rad(theta)) * ((xs - x0).clamp(min=0) * s)
        Z = Z + torch.randn(H, W, generator=g, dtype=torch.float64) * 2e-5
        step = torch.where(ys.long() % 2 == 0, 0.029, 0.031)
        Z = torch.where(xs >= W // 4, Z * (1 + step), Z)
        zero = torch.rand(H, W, generator=g) < 0.01
        Z = torch.where(zero, torch.zeros_like(Z), Z)
        pts.append(torch.stack([X * Z / 2, Y * Z / 2, Z], -1).float())
        m = torch.rand(H, W, generator=g) > 0.05
        m[H // 3:H // 3 + 3, W // 5:W // 5 + 7] = False
        m &= ~zero | (torch.rand(H, W, generator=g) < 0.3)          # some zero-depth pixels stay in the mask
        masks.append(m)
    cam = torch.stack(pts)
    from oracle.geometry import quat_to_rotmat

    R = quat_to_rotmat(torch.tensor([0.1, -0.2, 0.3, 0.9])).float()
    world = cam @ R.T + torch.tensor([1.0, -2.0, 0.5])
    return world, cam, torch.stack(masks)


def _angle_np(normals, nmask):
    """oracle.geometry.normals_edge up to the per-pixel max angle (before the pool)."""
    from oracle.geometry import _windows3

    with np.errstate(all="ignore"):
        nn = normals / (np.linalg.norm(normals, axis=-1, keepdims=True) + 1e-12)
        npad = np.pad(nn, ((1, 1), (1, 1), (0, 0)), mode="edge")
        mpad = np.pad(nmask, ((1, 1), (1, 1)), mode="edge")
        dots = (_windows3(npad) * nn[None]).sum(axis=-1)
        mwin = _windows3(mpad).reshape(3, 3, *nmask.shape).transpose(1, 0, 2, 3).reshape(9, *nmask.shape)
        return np.where(mwin, np.arccos(dots), 0).max(axis=0)


@pytest.mark.parametrize("n,H,W", [(1, 518, 518), (3, 294, 518), (8, 37, 53), (1, 1, 64), (1, 64, 1), (1, 2, 2),
                                   (1, 1024, 600)])
def test_edge_mask(n, H, W):
    from oracle.geometry import _nanmax_pool3, depth_edge, points_to_normals

    world, cam, mask = _edge_scene(n, H, W, n * H + W)
    P = n * H * W
    pts = _in(world.to(DEV))
    camd = _in(cam.to(DEV))
    mk = _in(mask.to(torch.uint8).to(DEV))
    obuf, out = _out(P, dtype=torch.uint8)
    nbuf, ws_n = _out(P * 3)
    mbuf, ws_m = _out(P, dtype=torch.uint8)
    abuf, ws_a = _out(P)
    dbuf, ws_d = _out(P, dtype=torch.uint8)
    _call("ma_edge_mask", pts.data_ptr(), camd.data_ptr() + 8, 3, mk.data_ptr(), out.data_ptr(), ws_n.data_ptr(),
          ws_m.data_ptr(), ws_a.data_ptr(), ws_d.data_ptr(), n, H, W, TOL_DEG, RTOL)
    what = f"edge_mask n={n} {H}x{W}"
    for b, k in ((obuf, 1), (nbuf, 3), (mbuf, 1), (abuf, 1), (dbuf, 1)):
        _assert_tail(b, P * k, what)
    got_n = ws_n.view(n, H, W, 3).cpu().numpy()
    got_m, got_a = ws_m.view(n, H, W).cpu().numpy(), ws_a.view(n, H, W).cpu().numpy()
    got_d, got_o = ws_d.view(n, H, W).cpu().numpy(), out.view(n, H, W).cpu().numpy()
    tol = np.deg2rad(TOL_DEG)
    worst_ulp, skipped, removed = 0.0, 0, 0
    for v in range(n):
        pv, mv = world[v].numpy(), mask[v].numpy()
        normals, nmask = points_to_normals(pv, mv)
        assert np.array_equal(got_n[v].view(np.int32), normals.astype(np.float32).view(np.int32)), \
            f"{what} view {v}: normals differ in {int((got_n[v] != normals).any(-1).sum())} pixels"
        assert np.array_equal(got_m[v] != 0, nmask), f"{what} view {v}: normal mask"
        assert set(np.unique(got_m[v]).tolist()) <= {0, 1}
        de = depth_edge(np.ascontiguousarray(cam[v, ..., 2].numpy()), RTOL, mv)
        assert np.array_equal(got_d[v] != 0, de), f"{what} view {v}: depth edge differs in {int((got_d[v] != de).sum())} pixels"
        ang = _angle_np(normals.astype(np.float32), nmask)
        assert np.array_equal(np.isnan(got_a[v]), np.isnan(ang)), f"{what} view {v}: NaN angles differ"
        ok = ~np.isnan(ang)
        ulp = np.abs(got_a[v][ok].astype(np.float64) - ang[ok]) / np.spacing(np.abs(ang[ok]).astype(np.float32))
        worst_ulp = max(worst_ulp, float(ulp.max()) if ulp.size else 0.0)
        assert worst_ulp <= ANGLE_ULPS, f"{what} view {v}: angle {worst_ulp:.1f} ulp from numpy's"
        pooled = _nanmax_pool3(ang)
        with np.errstate(invalid="ignore"):
            ne = pooled > tol
            near = np.abs(pooled.astype(np.float64) - tol) <= ANGLE_ULPS * np.spacing(np.float32(tol))
        want = mv & ~(de & ne)
        bad = (got_o[v] != want) & ~near
        assert not bad.any(), f"{what} view {v}: final mask differs in {int(bad.sum())} pixels, first at {np.argwhere(bad)[0]}"
        assert set(np.unique(got_o[v]).tolist()) <= {0, 1}
        skipped += int(near.sum())
        removed += int((mv & ~want).sum())
    print(f"\n[edge_mask] {what}: worst angle {worst_ulp:.2f} ulp of numpy's (bound {ANGLE_ULPS}); {removed} pixels removed, "
          f"{skipped} within the bound of the threshold", end="")
    if H * W >= 4096:
        assert removed > 0, f"{what}: the scene removes nothing"
