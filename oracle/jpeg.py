"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the baseline JPEG decode Pillow runs through libjpeg-turbo with its
defaults: sequential Huffman entropy decoding (jdhuff.c), DC prediction, dequantisation + the `JDCT_ISLOW` integer IDCT
(jidctint.c) with the post-IDCT range-limit table (jdmaster.c prepare_range_limit_table), fancy upsampling
(jdsample.c h2v1 / h2v2 / h1v2, plain replication for chroma no wider than 2 samples) and the table-driven YCbCr -> RGB
conversion (jdcolor.c).  Written for clarity on small images; `decode(data)` returns the (H, W, 3) uint8 frame before
EXIF orientation, the same bytes as `np.asarray(PIL.Image.open(f).convert("RGB"))` for the baseline files the GPU route
accepts.  tests/test_jpeg_cpu.py checks it against the installed Pillow bit for bit.
"""
from __future__ import annotations

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63])   # jpeg_natural_order: zig-zag index -> natural index


class JpegError(ValueError):
    pass


def parse(data: bytes) -> dict:
    """Markers of a baseline file -> frame, tables, scan and the entropy-coded segments (restart intervals), stuffing
    removed.  Raises JpegError for anything outside baseline 8-bit 1- or 3-component sequential Huffman."""
    if data[:2] != b"\xff\xd8":
        raise JpegError("no SOI")
    q, dc, ac, frame, ri, p = {}, {}, {}, None, 0, 2
    while True:
        while p < len(data) and data[p] == 0xFF and p + 1 < len(data) and data[p + 1] == 0xFF:
            p += 1
        if p + 4 > len(data) or data[p] != 0xFF:
            raise JpegError("truncated or bad marker")
        m, L = data[p + 1], int.from_bytes(data[p + 2:p + 4], "big")
        seg = data[p + 4:p + 2 + L]
        if len(seg) != L - 2:
            raise JpegError("truncated segment")
        p += 2 + L
        if m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                n = 128 if pq else 64
                vals = np.frombuffer(seg[i + 1:i + 1 + n], ">u2" if pq else "u1").astype(np.int32)
                t = np.zeros(64, np.int32)
                t[ZIGZAG] = vals
                q[tq] = t
                i += 1 + n
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                tc, th = seg[i] >> 4, seg[i] & 15
                counts = list(seg[i + 1:i + 17])
                vals = list(seg[i + 17:i + 17 + sum(counts)])
                codes, code = {}, 0
                k = 0
                for ln in range(1, 17):
                    for _ in range(counts[ln - 1]):
                        codes[(ln, code)] = vals[k]
                        k += 1
                        code += 1
                    if code >= (1 << ln):   # jdhuff.c: no code may be all ones
                        raise JpegError("bad Huffman table")
                    code <<= 1
                if not tc and any(v > 15 for v in vals):
                    raise JpegError("DC symbol above 15")
                (ac if tc else dc)[th] = codes
                i += 17 + sum(counts)
        elif m == 0xDD:
            ri = int.from_bytes(seg[:2], "big")
        elif m in (0xC0, 0xC1):
            if seg[0] != 8:
                raise JpegError("not 8-bit")
            H, W, nc = int.from_bytes(seg[1:3], "big"), int.from_bytes(seg[3:5], "big"), seg[5]
            comps = [(seg[6 + 3 * c], seg[7 + 3 * c] >> 4, seg[7 + 3 * c] & 15, seg[8 + 3 * c]) for c in range(nc)]
            frame = (W, H, comps)
        elif 0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            raise JpegError("not baseline")
        elif m == 0xDA:
            ns = seg[0]
            sel = [(seg[1 + 2 * k], seg[2 + 2 * k] >> 4, seg[2 + 2 * k] & 15) for k in range(ns)]
            break
    # entropy-coded data up to the next non-RST marker, split at RSTn, stuffing removed
    segs, cur, n = [], bytearray(), len(data)
    while p < n:
        b = data[p]
        if b != 0xFF:
            cur.append(b)
            p += 1
            continue
        nxt = data[p + 1] if p + 1 < n else 0xD9
        if nxt == 0:
            cur.append(0xFF)
            p += 2
        elif 0xD0 <= nxt <= 0xD7:
            segs.append(bytes(cur))
            cur = bytearray()
            p += 2
        elif nxt == 0xFF:
            p += 1
        else:
            break
    segs.append(bytes(cur))
    W, H, comps = frame
    return dict(W=W, H=H, comps=comps, q=q, dc=dc, ac=ac, ri=ri, scan=sel, segs=segs)


class _Bits:
    def __init__(self, b: bytes):
        self.v, self.n, self.p = int.from_bytes(b, "big") if b else 0, len(b) * 8, 0

    def bit(self) -> int:
        if self.p >= self.n:
            raise JpegError("entropy data exhausted")
        self.p += 1
        return (self.v >> (self.n - self.p)) & 1

    def bits(self, k: int) -> int:
        r = 0
        for _ in range(k):
            r = (r << 1) | self.bit()
        return r

    def huff(self, codes: dict) -> int:
        code = 0
        for ln in range(1, 17):
            code = (code << 1) | self.bit()
            if (ln, code) in codes:
                return codes[(ln, code)]
        raise JpegError("bad Huffman code")


def _extend(r: int, s: int) -> int:
    return r - (1 << s) + 1 if s and r < (1 << (s - 1)) else r


def coefficients(j: dict) -> list:
    """Quantised coefficients per component, (blocks_h, blocks_w, 64) int32 in natural order, DC prediction applied."""
    W, H, comps = j["W"], j["H"], j["comps"]
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    mx, my = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    tabs = {cid: (dc, ac) for cid, dc, ac in j["scan"]}
    if len(comps) == 1:   # non-interleaved: one block per MCU, over the component's own block grid
        bw, bh = -(-W // 8), -(-H // 8)
        out = [np.zeros((bh, bw, 64), np.int32)]
        order = [(0, by, bx) for by in range(bh) for bx in range(bw)]
        per_mcu = 1
    else:
        out = [np.zeros((my * c[2], mx * c[1], 64), np.int32) for c in comps]
        per_mcu = sum(c[1] * c[2] for c in comps)
        order = []
        for m in range(mx * my):
            for ci, c in enumerate(comps):
                for v in range(c[2]):
                    for h in range(c[1]):
                        order.append((ci, (m // mx) * c[2] + v, (m % mx) * c[1] + h))
    ri = j["ri"]
    blocks_per_seg = ri * per_mcu if ri else len(order)
    k0 = 0
    for seg in j["segs"]:
        if k0 >= len(order):
            break
        bits, pred = _Bits(seg), [0] * len(comps)
        for ci, by, bx in order[k0:k0 + blocks_per_seg]:
            dct, act = tabs[comps[ci][0]]
            blk = out[ci][by, bx]
            s = bits.huff(j["dc"][dct])
            pred[ci] += _extend(bits.bits(s), s)
            blk[0] = np.int16(np.int32(pred[ci]).astype(np.int16))
            k = 1
            while k < 64:
                rs = bits.huff(j["ac"][act])
                r, s = rs >> 4, rs & 15
                if s:
                    k += r
                    blk[ZIGZAG[min(k, 63)]] = _extend(bits.bits(s), s)
                else:
                    if r != 15:
                        break
                    k += 15
                k += 1
        k0 += blocks_per_seg
    if k0 < len(order):
        raise JpegError("fewer restart intervals than MCUs")
    return out


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def idct_islow(coef: np.ndarray, qt: np.ndarray) -> np.ndarray:
    """jidctint.c jpeg_idct_islow on (..., 64) natural-order coefficients -> (..., 8, 8) samples via the range-limit
    table (x & 1023 indexes a table that clamps [-512, 511] + 128 and wraps outside it)."""
    CB, P1 = 13, 2
    F = {k: v for k, v in dict(f0298=2446, f0390=3196, f0541=4433, f0765=6270, f0899=7373, f1175=9633, f1501=12299,
                                 f1847=15137, f1961=16069, f2053=16819, f2562=20995, f3072=25172).items()}
    x = (coef.astype(np.int64) * qt.astype(np.int64)).reshape(coef.shape[:-1] + (8, 8))

    def one_d(v0, v1, v2, v3, v4, v5, v6, v7, shift_in, shift_out):
        z2, z3 = v2, v6
        z1 = (z2 + z3) * F["f0541"]
        tmp2 = z1 + z3 * -F["f1847"]
        tmp3 = z1 + z2 * F["f0765"]
        tmp0, tmp1 = (v0 + v4) << CB, (v0 - v4) << CB
        if shift_in:
            tmp0, tmp1 = tmp0 + shift_in, tmp1 + shift_in
        t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
        o0, o1, o2, o3 = v7, v5, v3, v1
        z1, z2, z3, z4 = o0 + o3, o1 + o2, o0 + o2, o1 + o3
        z5 = (z3 + z4) * F["f1175"]
        o0, o1, o2, o3 = o0 * F["f0298"], o1 * F["f2053"], o2 * F["f3072"], o3 * F["f1501"]
        z1, z2, z3, z4 = z1 * -F["f0899"], z2 * -F["f2562"], z3 * -F["f1961"] + z5, z4 * -F["f0390"] + z5
        o0, o1, o2, o3 = o0 + z1 + z3, o1 + z2 + z4, o2 + z2 + z3, o3 + z1 + z4
        r = [t10 + o3, t11 + o2, t12 + o1, t13 + o0, t13 - o0, t12 - o1, t11 - o2, t10 - o3]
        return [_descale(v, shift_out) for v in r]

    cols = one_d(*[x[..., i, :] for i in range(8)], 0, CB - P1)        # pass 1 over columns: (..., 8 cols) each
    ws = np.stack(cols, axis=-2)                                         # (..., row, col)
    rows = one_d(*[ws[..., :, i] for i in range(8)], 0, CB + P1 + 3)     # pass 2 over rows
    out = np.stack(rows, axis=-1)
    return range_limit_idct(out)


def range_limit_idct(x: np.ndarray) -> np.ndarray:
    v = x & 1023
    return np.where(v < 128, v + 128, np.where(v < 512, 255, np.where(v < 896, 0, v - 896))).astype(np.uint8)


def _planes(j: dict, coefs: list) -> list:
    planes = []
    for ci, c in enumerate(j["comps"]):
        qt = j["q"][c[3]]
        s = idct_islow(coefs[ci], qt)                       # (bh, bw, 8, 8)
        bh, bw = s.shape[:2]
        planes.append(s.transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8).astype(np.int32))
    return planes


def _h2(p: np.ndarray, w: int) -> np.ndarray:
    """h2v1_fancy_upsample over the first w columns: triangular filter, biases 1 / 2 alternating, edges replicated."""
    p = p[:, :w]
    out = np.empty((p.shape[0], 2 * w), np.int32)
    left = np.concatenate([p[:, :1], p[:, :-1]], 1)
    right = np.concatenate([p[:, 1:], p[:, -1:]], 1)
    out[:, 0::2] = (3 * p + left + 1) >> 2
    out[:, 1::2] = (3 * p + right + 2) >> 2
    out[:, 0], out[:, -1] = p[:, 0], p[:, -1]
    return out


def upsample(p: np.ndarray, h: int, v: int, dw: int, dh: int, do_fancy_h: bool) -> np.ndarray:
    """One chroma plane (the component's downsampled_width dw x downsampled_height dh samples) -> h x v times larger."""
    p = p[:dh, :dw]
    if h == 1 and v == 1:
        return p
    if h == 2 and v == 1:
        return _h2(p, dw) if do_fancy_h else np.repeat(p, 2, 1)
    if h == 2 and v == 2 and not do_fancy_h:
        return np.repeat(np.repeat(p, 2, 1), 2, 0)
    up = np.concatenate([p[:1], p[:-1]], 0)          # row above; the first row is its own neighbour
    dn = np.concatenate([p[1:], p[-1:]], 0)          # row below; the last real row is its own neighbour
    if h == 1:                                       # h1v2_fancy_upsample
        out = np.empty((2 * dh, dw), np.int32)
        out[0::2] = (3 * p + up + 1) >> 2
        out[1::2] = (3 * p + dn + 2) >> 2
        return out
    out = np.empty((2 * dh, 2 * dw), np.int32)       # h2v2_fancy_upsample on column sums
    for r, nb in ((0, up), (1, dn)):
        cs = 3 * p + nb
        last = np.concatenate([cs[:, :1], cs[:, :-1]], 1)
        nxt = np.concatenate([cs[:, 1:], cs[:, -1:]], 1)
        o = np.empty((dh, 2 * dw), np.int32)
        o[:, 0::2] = (3 * cs + last + 8) >> 4
        o[:, 1::2] = (3 * cs + nxt + 7) >> 4
        o[:, 0] = (cs[:, 0] * 4 + 8) >> 4
        o[:, -1] = (cs[:, -1] * 4 + 7) >> 4
        out[r::2] = o
    return out


def _color_tables():
    x = np.arange(256, dtype=np.int64) - 128
    S, half = 16, 1 << 15

    def fix(f):
        return int(f * (1 << S) + 0.5)

    cr_r = (fix(1.40200) * x + half) >> S
    cb_b = (fix(1.77200) * x + half) >> S
    cr_g = -fix(0.71414) * x
    cb_g = -fix(0.34414) * x + half
    return cr_r, cb_b, cr_g, cb_g


def ycc_to_rgb(y, cb, cr) -> np.ndarray:
    cr_r, cb_b, cr_g, cb_g = _color_tables()
    r = y + cr_r[cr]
    g = y + ((cb_g[cb] + cr_g[cr]) >> 16)
    b = y + cb_b[cb]
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(data: bytes) -> np.ndarray:
    j = parse(data)
    coefs = coefficients(j)
    planes = _planes(j, coefs)
    W, H, comps = j["W"], j["H"], j["comps"]
    if len(comps) == 1:
        g = planes[0][:H, :W].astype(np.uint8)
        return np.repeat(g[:, :, None], 3, 2)
    hmax, vmax = comps[0][1], comps[0][2]
    full = []
    for ci, c in enumerate(comps):
        dw, dh = -(-W * c[1] // hmax), -(-H * c[2] // vmax)
        hf, vf = hmax // c[1], vmax // c[2]
        full.append(upsample(planes[ci], hf, vf, dw, dh, dw > 2)[:H, :W])
    return ycc_to_rgb(*full)
