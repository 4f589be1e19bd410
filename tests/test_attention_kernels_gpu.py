"""Every attention forward kernel (v5, v3, v2) and the partial-state merge against an fp64 reference, on each path they accept.

ma_attention_fwd_ex picks the kernel from the call's shape: v5 for plain attention whose (128-row query tile, head, sequence)
items number at least 6 x SMs, v3 for other calls with up to 4096 keys and no kv split, v2 otherwise.  Every case asserts
the kernel it meant to reach (ma_last_attention_kernel) and compares every element the call writes -- for calls with more
than ~10^7 score entries a fixed sample of query rows holding the first and last row of every 128-row query tile -- with
softmax(scale q k^T) v computed in fp64 on the bf16 inputs.  Every element the call must not write (the columns of a wider
out beside the heads, rows between strided sequences, rows past the last sequence, unused partial slots) holds a sentinel
and is checked bit for bit.  The inputs are column slices of wider matrices whose other columns are NaN.

Inputs.  Channel 0 of every head is a per-key bias: q[:, 64 h] = 1 and k[j, 64 h] = b_j (a bf16-exact integer), so key j's
raw score is shifted by b_j exactly and the fp64 reference needs no special case.  Patterns: iid (randn x 1.5); needle
(b = +160 on the first and last key of every 64-key tile of every segment -- which includes every 128-key tile, every kv
split part and kv_len - 1 --, spread over heads and over the two parities of query rows by a +-40 selector in channel 1,
with |v| ~ 4 on those keys, so that a dropped, doubled or shifted key moves the output by O(|v|)); rise (b grows by 48 raw
per 64 keys: more than 8 log2 units per key tile at every scale here, so every tile rescales); rise_alt (the same for even
query rows only: lazy_rescale's warp vote with some lanes that need no rescale); fall (later tiles underflow); big (raw
scores ~ 10^3); uniform (q = 0: the output is the mean of V).  In every pattern the key rows inside the tensor that are not
in the key set (past kv_len, between sequences, between segments) are poison: bias 200 above the largest in-set bias and
V = +-1000 (finite: 0 x NaN in the P.V MMA would turn a correctly masked key into NaN), so a leaked key dominates.

Bound, per element, with A = sum_i p_i |v_i| / sum_i p_i (fp64), n keys, and ds = 2^-16 max_i sum_d |q_d k_id| the fp32
score error (64 exact bf16 products summed in fp32: 64 x 2^-23 = 2^-17, doubled for the fp32 rounding of the scale):
  bf16 out:       |got - ref| <= 2^-8 |ref| + A (2^-8 + 4 scale ds + n 2^-21 + 2^-17)
  fp32 state_o:   the same without 2^-8 |ref|
  state_m (raw score units, m' = logsumexp(scale s) / scale):  ds + (n 2^-23 + 2^-19) / scale + 2^-22 |m'|
2^-8 (the unit roundoff of bf16's 8 significant bits) |ref| is the rounding of the output to bf16; 2^-8 A bounds the
probabilities rounded to bf16 for P.V while l sums them in fp32; a score error shifts the output by at most 2 scale ds A,
and a merge weighs partials by m', which carries the same error again; n 2^-21 covers the fp32 sums of O and l (n 2^-23
each) and their effect through m'; 2^-17 the ex2 / log2 approximations.  Every case prints its worst err / bound, and the
largest per kernel is printed at the end of the module.  Measured on one NVIDIA B200 (1000 W power limit): v5 0.92, v3
0.89, v2 0.71, merge 0.80.  The largest are at kv_len = 1, where the one probability (2^x with |x| <= 0.5 against the
integer reference maximum) and the output are each rounded once: the exact worst case the first two terms allow.
"""

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32
SENTINEL = -77.0           # exact in bf16: every out element the call must not write
PAD = 8                    # bf16 columns of NaN left of the heads in every input / of sentinel around them in out
SCALES = [0.125, 0.125 * 1.37, 1.0]
PATTERNS = ["iid", "needle", "rise", "rise_alt", "fall", "big", "uniform"]
SAMPLE_ABOVE = 10 ** 7     # score entries above which the check samples query rows
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print("\n[attention kernels] worst err/bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(WORST.items())))


def _lib():
    from mapanything_b200 import _lib

    return _lib.load()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


class Geometry:
    """Query and key rows of one call: nseq sequences q_gap / kv_gap rows apart, the keys of a sequence being the segments
    (row0, len) in segment order, and rows past the last sequence inside the tensors (`tail`)."""

    def __init__(self, H, q_len, kv_len=None, *, nseq=1, q_gap=0, kv_gap=0, segs=None, tail=70):
        self.segs = segs or [(0, kv_len)]
        self.H, self.D, self.q_len, self.nseq = H, 64 * H, q_len, nseq
        self.kv_len = sum(n for _, n in self.segs)
        extent = max(r + n for r, n in self.segs)
        self.q_stride, self.kv_stride = q_len + q_gap, extent + kv_gap
        self.q_total = (nseq - 1) * self.q_stride + q_len + 5
        self.kv_total = (nseq - 1) * self.kv_stride + extent + tail
        self.qrows = torch.arange(nseq)[:, None] * self.q_stride + torch.arange(q_len)

    def keys(self, segs=None):
        """[nseq, n] key rows of `segs` (default: all segments), in segment order."""
        off = torch.cat([torch.arange(r, r + n) for r, n in (segs or self.segs)])
        return torch.arange(self.nseq)[:, None] * self.kv_stride + off

    def probes(self):
        """Positions (in key order) of the first and last key of every 64-key tile of every segment."""
        out, o = set(), 0
        for _, n in self.segs:
            for t in range(0, n, 64):
                out |= {o + t, o + min(t + 64, n) - 1}
            o += n
        return sorted(out)


def make_inputs(geo, pattern, seed):
    """q, k, v: column slices of NaN-padded bf16 matrices filled for `pattern` (module docstring)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    H, D, n = geo.H, geo.D, geo.kv_len
    qbuf = torch.full((geo.q_total, D + 2 * PAD), float("nan"), device="cuda", dtype=BF16)
    kvbuf = torch.full((geo.kv_total, 2 * D + 4 * PAD), float("nan"), device="cuda", dtype=BF16)
    qf = torch.randn(geo.q_total, H, 64, device="cuda", generator=g) * 1.5
    kf = torch.randn(geo.kv_total, H, 64, device="cuda", generator=g) * 1.5
    vf = torch.randn(geo.kv_total, H, 64, device="cuda", generator=g)
    j = torch.arange(n, device="cuda")
    bias = torch.zeros(n, H, device="cuda")
    sel = torch.zeros(n, H, device="cuda")
    vscale = torch.ones(n, H, device="cuda")
    qf[:, :, 0] = 1.0
    if pattern == "iid":
        bias = torch.randn(n, H, device="cuda", generator=g) * 1.5
    elif pattern == "needle":
        qf[:, :, 1:] *= 1.0 / 6
        qf[:, :, 1] = (1 - 2 * (torch.arange(geo.q_total, device="cuda") % 2)).float()[:, None]   # row parity selector
        for i, pos in enumerate(geo.probes()):
            h, grp = i % H, (i // H) % 2
            bias[pos, h], sel[pos, h], vscale[pos, h] = 160.0, 40.0 if grp == 0 else -40.0, 4.0
    elif pattern in ("rise", "rise_alt"):
        bias[:] = (48 * (j // 64)).float()[:, None]
        if pattern == "rise_alt":
            qf[1::2, :, 0] = 0.0
    elif pattern == "fall":
        bias[:] = (-48 * (j // 64)).float()[:, None]
    elif pattern == "big":
        bias = 960.0 + 4 * torch.randint(0, 16, (n, H), device="cuda", generator=g).float()
    elif pattern == "uniform":
        qf.zero_()
    else:
        raise ValueError(pattern)
    keys = geo.keys().cuda().flatten()   # every sequence gets the same per-key pattern
    kf[keys, :, 0] = bias.repeat(geo.nseq, 1)
    kf[keys, :, 1] = torch.where(sel != 0, sel, 0.0).repeat(geo.nseq, 1) + kf[keys, :, 1] * (sel == 0).repeat(geo.nseq, 1)
    vf[keys] *= vscale.repeat(geo.nseq, 1)[:, :, None]
    poison = torch.ones(geo.kv_total, dtype=torch.bool, device="cuda")
    poison[keys] = False
    kf[poison, :, 0] = float(bias.max()) + 200.0
    vf[poison] = 1000.0 * torch.sign(torch.randn(int(poison.sum()), H, 64, device="cuda", generator=g) + 0.1)
    q, k, v = qbuf[:, PAD:PAD + D], kvbuf[:, PAD:PAD + D], kvbuf[:, D + 3 * PAD:2 * D + 3 * PAD]
    q.copy_(qf.reshape(geo.q_total, D))
    k.copy_(kf.reshape(geo.kv_total, D))
    v.copy_(vf.reshape(geo.kv_total, D))
    return q, k, v


def sample_rows(geo, n_keys):
    """Query indices (within a sequence) the check compares: all, or the first and last row of every 128-row tile plus 32
    fixed random rows when the call has more than SAMPLE_ABOVE score entries."""
    if geo.nseq * geo.H * geo.q_len * n_keys <= SAMPLE_ABOVE:
        return torch.arange(geo.q_len)
    rows = {0, geo.q_len - 1}
    for t in range(0, geo.q_len, 128):
        rows |= {t, min(t + 128, geo.q_len) - 1}
    rows |= set(torch.randint(0, geo.q_len, (32,), generator=torch.Generator().manual_seed(geo.q_len)).tolist())
    return torch.tensor(sorted(rows))


def reference(q, k, v, geo, qidx, keys, scale):
    """fp64 softmax attention of query rows geo.qrows[:, qidx] over key rows keys [nseq, n].  Returns (o, A, ds, m') with
    o / A [nseq, R, H, 64] and ds / m' [nseq, R, H] (module docstring)."""
    H, R, n = geo.H, len(qidx), keys.shape[1]
    qr, kr = geo.qrows[:, qidx].cuda(), keys.cuda()
    q64 = q[qr.flatten()].double().view(geo.nseq, R, H, 64).transpose(1, 2)
    k64 = k[kr.flatten()].double().view(geo.nseq, n, H, 64).transpose(1, 2)
    v64 = v[kr.flatten()].double().view(geo.nseq, n, H, 64).transpose(1, 2)
    s = q64 @ k64.transpose(-1, -2)
    ds = 2.0 ** -16 * (q64.abs() @ k64.abs().transpose(-1, -2)).amax(-1)
    lse = torch.logsumexp(s * scale, -1)
    p = torch.exp(s * scale - lse[..., None])
    del s
    o, a = p @ v64, p @ v64.abs()
    return o.transpose(1, 2), a.transpose(1, 2), ds.transpose(1, 2), (lse / scale).transpose(1, 2)


def out_bound(ref, a, ds, n, scale, bf16):
    b = a * (2.0 ** -8 + 4 * scale * ds[..., None] + n * 2.0 ** -21 + 2.0 ** -17)
    return b + 2.0 ** -8 * ref.abs() if bf16 else b


def m_bound(m, ds, n, scale):
    return ds + (n * 2.0 ** -23 + 2.0 ** -19) / scale + 2.0 ** -22 * m.abs()


def check(got, ref, bound, what, kernel):
    err = (got.double() - ref).abs()
    ratio = torch.nan_to_num(err / bound, nan=float("inf"))
    worst = ratio.max().item()
    WORST[kernel] = max(WORST.get(kernel, 0.0), worst)
    print(f"\n{what}: worst err/bound {worst:.3g}", end="")
    if worst > 1.0:
        i = int(ratio.argmax().item())
        raise AssertionError(f"{what}: element {list(torch.unravel_index(torch.tensor(i), ratio.shape))} = "
                             f"{got.flatten()[i].item()!r}, reference {ref.flatten()[i].item()!r}, bound "
                             f"{bound.flatten()[i].item():.3g} (worst err/bound {worst:.3g})")


def check_untouched(buf, written, sentinel_bits, what):
    """Bit-exact sentinel in every element of buf outside the boolean mask `written`."""
    bits = buf.view(torch.int16 if buf.dtype == BF16 else torch.int32)
    bad = (bits != sentinel_bits) & ~written
    assert not bad.any(), f"{what}: {int(bad.sum())} elements outside the output were written, first at {bad.nonzero()[0].tolist()}"


def _bits(value, dtype):
    return torch.tensor([value], dtype=dtype).view(torch.int16 if dtype == BF16 else torch.int32).item()


class Out:
    """bf16 output: a column slice of a sentinel-filled matrix, NaN where the call is to write (row, head)."""

    def __init__(self, geo):
        self.geo = geo
        self.buf = torch.full((geo.q_total, geo.D + 2 * PAD), SENTINEL, device="cuda", dtype=BF16)
        self.t = self.buf[:, PAD:PAD + geo.D]
        self.written = torch.zeros(self.buf.shape, dtype=torch.bool, device="cuda")

    def expect(self, rows, heads):
        """The call writes (rows [nseq, q_len] or flat, heads) -- all heads when heads is None."""
        rows = rows.flatten().cuda()
        for h in range(self.geo.H) if heads is None else heads:
            self.t[rows, 64 * h:64 * h + 64] = float("nan")
            self.written[rows, PAD + 64 * h:PAD + 64 * h + 64] = True

    def check(self, what, kernel, ref, qidx, scale, n):
        o, a, ds, _ = ref
        geo = self.geo
        got = self.t[geo.qrows[:, qidx].flatten().cuda()].view(geo.nseq, len(qidx), geo.H, 64)
        check(got, o, out_bound(o, a, ds, n, scale, True), what + " out", kernel)
        assert torch.isfinite(self.t[self.written[:, PAD:PAD + geo.D]].float()).all(), f"{what}: out left unwritten"
        check_untouched(self.buf, self.written, _bits(SENTINEL, BF16), what + " out")


class State:
    """fp32 partial states (parts, q_total, ld) with the heads at a 16-byte column offset; state_o NaN and state_m -inf
    where nothing is written."""

    def __init__(self, geo, parts):
        self.geo, self.parts = geo, parts
        self.obuf = torch.full((parts, geo.q_total, geo.D + 8), float("nan"), device="cuda")
        self.o = self.obuf[:, :, 4:4 + geo.D]
        self.m = torch.full((parts, geo.q_total, geo.H), float("-inf"), device="cuda")
        self.written = torch.zeros(parts, geo.q_total, geo.H, dtype=torch.bool, device="cuda")

    def expect(self, part, rows, heads=None):
        for h in range(self.geo.H) if heads is None else heads:
            self.written[part, rows.flatten().cuda(), h] = True

    def check_part(self, part, what, kernel, ref, qidx, scale, n, mask=None):
        """Partial `part` against ref at the (row, head) pairs of mask [q_total, H] (default: all it was to write)."""
        o, a, ds, m = ref
        geo = self.geo
        rows = geo.qrows[:, qidx].flatten().cuda()
        sel = (self.written[part] if mask is None else mask)[rows].view(geo.nseq, len(qidx), geo.H)
        if not sel.any():
            return
        got_o = self.o[part, rows].view(geo.nseq, len(qidx), geo.H, 64)
        got_m = self.m[part, rows].view(geo.nseq, len(qidx), geo.H)
        check(got_o[sel], o[sel], out_bound(o, a, ds, n, scale, False)[sel], f"{what} state_o[{part}]", kernel)
        check(got_m[sel], m[sel], m_bound(m, ds, n, scale)[sel], f"{what} state_m[{part}]", kernel)

    def check_untouched(self, what):
        wo = self.written[..., None].expand(-1, -1, -1, 64).reshape(self.parts, self.geo.q_total, self.geo.D)
        assert torch.isfinite(self.o[wo]).all() and torch.isfinite(self.m[self.written]).all(), f"{what}: state left unwritten"
        wbuf = torch.zeros(self.obuf.shape, dtype=torch.bool, device="cuda")
        wbuf[:, :, 4:4 + self.geo.D] = wo
        check_untouched(self.obuf, wbuf, _bits(float("nan"), F32), what + " state_o")
        check_untouched(self.m, self.written, _bits(float("-inf"), F32), what + " state_m")


def attend(geo, q, k, v, out, kernel, scale, segs=None, **kw):
    """ops.attention over the key segments `segs` (None: the plain call over [0, kv_len)); asserts the kernel it ran."""
    from mapanything_b200 import ops

    n = geo.kv_len if segs is None else sum(l for _, l in segs)
    ops.attention(q, k, v, out, num_heads=geo.H, num_seqs=geo.nseq, q_len=geo.q_len, kv_len=n, q_seq_stride=geo.q_stride,
                  kv_seq_stride=geo.kv_stride, scale=scale, kv_segments=segs, **kw)
    torch.cuda.synchronize()
    ran = _lib().ma_last_attention_kernel()
    assert ran == kernel, f"ran v{ran}, meant for v{kernel}"


def run_plain(kernel, geo, pattern, scale, seed, what, segs=None):
    q, k, v = make_inputs(geo, pattern, seed)
    out = Out(geo)
    out.expect(geo.qrows, None)
    attend(geo, q, k, v, out.t, kernel, scale, segs)
    keys = geo.keys()
    qidx = sample_rows(geo, keys.shape[1])
    out.check(what, f"v{kernel}", reference(q, k, v, geo, qidx, keys, scale), qidx, scale, keys.shape[1])


# ---- v5: plain attention with >= 6 x SMs query-tile items ------------------------------------------------------------


def _v5_nseq(H, q_len, odd=True):
    """Sequences giving >= 6 x SMs items, an odd item count when `odd` and H and the tile count are odd."""
    per = -(-q_len // 128) * H
    n = -(-6 * _sms() // per)
    return n + 1 if odd and (n * per) % 2 == 0 and per % 2 == 1 else n


# (q_len, kv_len, gaps): q_len != kv_len, one to three query tiles, 1 / 63 / 127 / 128 / 129 / 1370 keys
V5_SHAPES = [(1, 1, True), (100, 63, True), (128, 127, False), (129, 128, True), (257, 129, True), (128, 1370, True),
             (129, 1370, False)]


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("shape", V5_SHAPES, ids=[f"q{a}-kv{b}{'-gaps' if c else ''}" for a, b, c in V5_SHAPES])
def test_v5(shape, pattern):
    """Three heads (odd item counts), q / k / v / out at column offsets, strided sequences with poisoned gap rows."""
    q_len, kv_len, gaps = shape
    i = V5_SHAPES.index(shape) + PATTERNS.index(pattern)
    H = 3
    geo = Geometry(H, q_len, kv_len, nseq=_v5_nseq(H, q_len), q_gap=3 if gaps else 0, kv_gap=5 if gaps else 0)
    run_plain(5, geo, pattern, SCALES[i % 3], i, f"v5 {shape} {pattern}")


# ---- v3: up to 4096 keys, below the v5 threshold or with segments / state ----------------------------------------------


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("kv_len", [1, 63, 64, 65, 4095, 4096])
def test_v3_plain(kv_len, pattern):
    """Two strided sequences of 200 query rows (a ragged second query tile)."""
    i = kv_len + PATTERNS.index(pattern)
    geo = Geometry(2, 200, kv_len, nseq=2, q_gap=7, kv_gap=9)
    run_plain(3, geo, pattern, SCALES[i % 3], i, f"v3 kv{kv_len} {pattern}")


def _segments(lens, gap, order=1):
    """Segments of the given lengths `gap` rows apart, listed in increasing (order=1) or decreasing row order."""
    segs, r = [], gap
    for n in lens:
        segs.append((r, n))
        r += n + gap
    return segs if order == 1 else segs[::-1]


SEG_SETS = {
    "1_to_129": [1, 63, 64, 65, 127, 128, 129],
    "16_segments": [37, 1, 200, 64, 129, 5, 300, 128, 63, 250, 65, 2, 190, 127, 44, 256],
}


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("order", [1, -1], ids=["increasing", "decreasing"])
@pytest.mark.parametrize("segset", sorted(SEG_SETS))
def test_v3_segments(segset, order, pattern):
    i = len(segset) + order + PATTERNS.index(pattern)
    segs = _segments(SEG_SETS[segset], 3, order)
    geo = Geometry(2, 150, nseq=2, kv_gap=11, segs=segs)
    run_plain(3, geo, pattern, SCALES[i % 3], i, f"v3 segments {segset} {order} {pattern}", segs=segs)


def run_state_out(kernel, geo, pattern, scale, seed, what):
    """STATE_OUT over every segment: state_o / state_m of every row checked directly."""
    q, k, v = make_inputs(geo, pattern, seed)
    st = State(geo, 1)
    st.expect(0, geo.qrows)
    attend(geo, q, k, v, None, kernel, scale, geo.segs, state=(st.o[0], st.m[0]), state_out=True)
    keys = geo.keys()
    qidx = sample_rows(geo, keys.shape[1])
    st.check_part(0, what, f"v{kernel}", reference(q, k, v, geo, qidx, keys, scale), qidx, scale, keys.shape[1])
    st.check_untouched(what)


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("kernel,lens", [(3, [1000, 65, 1]), (3, [4096]), (2, [4097]), (2, [3000, 1, 1500])],
                         ids=["v3-3segs", "v3-4096", "v2-4097", "v2-3segs"])
def test_state_out(kernel, lens, pattern):
    i = len(lens) + sum(lens) + PATTERNS.index(pattern)
    segs = _segments(lens, 5)
    geo = Geometry(2, 257, nseq=2, q_gap=2, kv_gap=3, segs=segs)
    run_state_out(kernel, geo, pattern, SCALES[i % 3], i, f"v{kernel} state_out {lens} {pattern}")


@pytest.mark.parametrize("pattern", ["iid", "needle", "rise", "fall"])
@pytest.mark.parametrize("first,second", [(2, 3), (3, 3), (3, 2), (2, 2)])
def test_state_in(first, second, pattern):
    """The keys in two launches: STATE_OUT over the first segments by kernel `first`, STATE_IN over the rest by `second`;
    the result must be one softmax over all keys."""
    lens = {2: [2500, 1700], 3: [1300, 77]}
    segs = _segments(lens[first] + lens[second], 4)
    a, b = segs[:len(lens[first])], segs[len(lens[first]):]
    i = first * 3 + second + PATTERNS.index(pattern)
    scale = SCALES[i % 3]
    geo = Geometry(2, 300, nseq=2, q_gap=1, kv_gap=6, segs=segs)
    q, k, v = make_inputs(geo, pattern, i)
    so = torch.full((geo.q_total, geo.D), float("nan"), device="cuda")
    sm = torch.full((geo.q_total, geo.H), float("nan"), device="cuda")
    attend(geo, q, k, v, None, first, scale, a, state=(so, sm), state_out=True)
    out = Out(geo)
    out.expect(geo.qrows, None)
    attend(geo, q, k, v, out.t, second, scale, b, state=(so, sm), state_in=True)
    keys = geo.keys()
    qidx = sample_rows(geo, keys.shape[1])
    out.check(f"state v{first} -> v{second} {pattern}", f"v{second}", reference(q, k, v, geo, qidx, keys, scale), qidx,
              scale, keys.shape[1])


# ---- v2: more than 4096 keys, kv split ------------------------------------------------------------------------------


V2_SHAPES = [(ql, kl) for kl in (4097, 4224, 5000) for ql in (1, 100, 128, 129, 256, 257)]


@pytest.mark.parametrize("shape", V2_SHAPES, ids=[f"q{a}-kv{b}" for a, b in V2_SHAPES])
def test_v2(shape):
    """Each shape with the needle and one more pattern; two strided sequences where q_len > 128 (query tile B present)."""
    q_len, kv_len = shape
    i = V2_SHAPES.index(shape)
    nseq = 2 if q_len > 128 else 1
    geo = Geometry(2, q_len, kv_len, nseq=nseq, q_gap=5 if nseq > 1 else 0, kv_gap=7 if nseq > 1 else 0)
    for j, pattern in enumerate(("needle", [p for p in PATTERNS if p != "needle"][i % 6])):
        run_plain(2, geo, pattern, SCALES[(i + j) % 3], i, f"v2 {shape} {pattern}")


@pytest.mark.parametrize("pattern", PATTERNS)
def test_v2_ragged_segments(pattern):
    segs = _segments([1370, 1369, 77, 1500], 9)
    geo = Geometry(2, 300, nseq=2, kv_gap=4, segs=segs)
    i = PATTERNS.index(pattern)
    run_plain(2, geo, pattern, SCALES[i % 3], i, f"v2 ragged segments {pattern}", segs=segs)


def _kv_tiles(segs):
    """Key positions (in key order) of each 128-key tile of the segment walk."""
    tiles, o = [], 0
    for _, n in segs:
        tiles += [torch.arange(o + t, o + min(t + 128, n)) for t in range(0, n, 128)]
        o += n
    return tiles


def _slot_rows(q_len, H):
    """(query block, head) slot of attention_fwd_v2_kernel -> (rows, head), single sequence: full 256-row blocks of every
    head first, then the ragged last blocks."""
    n_full, slots = q_len // 256, []
    for h in range(H):
        slots += [(torch.arange(qb * 256, qb * 256 + 256), h) for qb in range(n_full)]
    if q_len % 256:
        slots += [(torch.arange(n_full * 256, q_len), h) for h in range(H)]
    return slots


def run_split(geo, pattern, scale, seed, parts, split_from, state_out, what):
    """kv split over v2: every partial state checked against the softmax over its own key tiles, then the merge (only
    the split slots with first_slot, as Engine._attention_one_sequence does, without STATE_OUT) against the whole."""
    from mapanything_b200 import ops

    q, k, v = make_inputs(geo, pattern, seed)
    H = geo.H
    slots = _slot_rows(geo.q_len, H)
    first = {"0": 0, "mid": len(slots) // 2, "n_slots": len(slots)}[split_from]
    st = State(geo, parts)
    out = Out(geo)
    for s, (rows, h) in enumerate(slots):
        if s >= first:
            for part in range(parts):
                st.expect(part, rows, [h])
        elif state_out:
            st.expect(0, rows, [h])
        else:
            out.expect(rows, [h])
    attend(geo, q, k, v, None if state_out else out.t, 2, scale, geo.segs, state=(st.o, st.m), state_out=state_out,
           kv_split=parts, kv_split_from=first)
    st.check_untouched(what)
    if not state_out:
        check_untouched(out.buf, out.written, _bits(SENTINEL, BF16), what + " out before the merge")
    keys = geo.keys()
    qidx = sample_rows(geo, keys.shape[1])
    split = torch.zeros(geo.q_total, H, dtype=torch.bool, device="cuda")
    for s, (rows, h) in enumerate(slots):
        split[rows.cuda(), h] = s >= first
    tiles = _kv_tiles(geo.segs)
    for part in range(parts):
        pos = torch.cat(tiles[part * len(tiles) // parts:(part + 1) * len(tiles) // parts])
        st.check_part(part, what, "v2", reference(q, k, v, geo, qidx, keys[:, pos], scale), qidx, scale, len(pos), split)
    full = reference(q, k, v, geo, qidx, keys, scale)
    if state_out and first > 0:   # the unsplit slots hold the state over all keys in part 0
        unsplit = ~split
        unsplit[geo.q_len:] = False
        st.check_part(0, what + " unsplit slots", "v2", full, qidx, scale, keys.shape[1], unsplit)
    for s, (rows, h) in enumerate(slots):
        if s >= first or state_out:
            out.expect(rows, [h])
    L = geo.q_len
    ops.attention_merge((st.o[:, :L], st.m[:, :L]), out.t[:L], num_heads=H, scale=scale, first_slot=-1 if state_out else first)
    torch.cuda.synchronize()
    out.check(what + " merged", "merge", full, qidx, scale, keys.shape[1])


SPLITS = [(4224, 2), (4224, 3), (4224, "all"), (5000, 3), (1000, "all")]


@pytest.mark.parametrize("state_out", [False, True], ids=["out", "state_out"])
@pytest.mark.parametrize("split_from", ["0", "mid", "n_slots"])
@pytest.mark.parametrize("kv_len,parts", SPLITS, ids=[f"kv{a}-split{b}" for a, b in SPLITS])
def test_v2_kv_split(kv_len, parts, split_from, state_out):
    """kv_split in {2, 3, n_kv_tiles} (uneven parts: 33 and 40 tiles), on 643 query rows (two full 256-row blocks and a
    ragged one) of 3 heads; the needle marks the first key of every part."""
    i = kv_len + (parts if parts != "all" else 1) + len(split_from)
    geo = Geometry(3, 643, kv_len, tail=100)
    parts = len(_kv_tiles(geo.segs)) if parts == "all" else parts
    pattern = ["needle", "iid", "rise"][i % 3]
    run_split(geo, pattern, SCALES[i % 3], i, parts, split_from, state_out,
              f"v2 split {kv_len}/{parts} from {split_from} {'state_out' if state_out else 'out'} {pattern}")


# ---- merge -----------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("level", [40.0, -40.0])
@pytest.mark.parametrize("scale", SCALES)
def test_merge_levels_and_unused_slots(level, scale):
    """Two partial states over key ranges whose scores differ in level by `level` raw, in slots 1 and 3 of 5; slots 0, 2
    and 4 are unused (-inf / NaN)."""
    from mapanything_b200 import ops

    segs = _segments([700, 900], 3)
    geo = Geometry(2, 300, segs=segs)
    q, k, v = make_inputs(geo, "iid", int(level) + int(scale * 100))
    keys = geo.keys()
    k[keys[0, 700:].cuda(), 0::64] += level
    st = State(geo, 5)
    attend(geo, q, k, v, None, 3, scale, segs[:1], state=(st.o[1], st.m[1]), state_out=True)
    attend(geo, q, k, v, None, 3, scale, segs[1:], state=(st.o[3], st.m[3]), state_out=True)
    out = Out(geo)
    out.expect(geo.qrows, None)
    ops.attention_merge((st.o, st.m), out.t, num_heads=geo.H, scale=scale)
    torch.cuda.synchronize()
    qidx = sample_rows(geo, keys.shape[1])
    out.check(f"merge level {level} scale {scale}", "merge", reference(q, k, v, geo, qidx, keys, scale), qidx, scale,
              keys.shape[1])


@pytest.mark.parametrize("first_slot", [0, 1, 2, 3])
def test_merge_first_slot(first_slot):
    """q_len 257 (a one-row last block), 2 heads = 4 slots: only the rows of slots >= first_slot are written."""
    from mapanything_b200 import ops

    geo = Geometry(2, 257, 1500)
    q, k, v = make_inputs(geo, "needle", first_slot)
    st = State(geo, 2)
    attend(geo, q, k, v, None, 2, 0.125 * 1.37, None, state=(st.o, st.m), state_out=True, kv_split=2)
    out = Out(geo)
    for s, (rows, h) in enumerate(_slot_rows(geo.q_len, geo.H)):
        if s >= first_slot:
            out.expect(rows, [h])
    L = geo.q_len
    ops.attention_merge((st.o[:, :L], st.m[:, :L]), out.t[:L], num_heads=geo.H, scale=0.125 * 1.37, first_slot=first_slot)
    torch.cuda.synchronize()
    keys = geo.keys()
    qidx = torch.arange(geo.q_len)
    o, a, ds, m = reference(q, k, v, geo, qidx, keys, 0.125 * 1.37)
    sel = out.written[:, PAD:PAD + geo.D][geo.qrows.flatten().cuda()].view(1, geo.q_len, geo.H, 64)
    got = out.t[geo.qrows.flatten().cuda()].view(1, geo.q_len, geo.H, 64)
    check(got[sel], o[sel], out_bound(o, a, ds, keys.shape[1], 0.125 * 1.37, True)[sel], f"merge first_slot {first_slot}",
          "merge")
    check_untouched(out.buf, out.written, _bits(SENTINEL, BF16), f"merge first_slot {first_slot}")


@pytest.mark.parametrize("scale_factor", [1.0, 1.37])
def test_sharded_protocol_with_entropy_scale(scale_factor):
    """Engine._block_global_sharded at a softmax scale 64^-0.5 x factor: local keys (STATE_OUT, tail slots split in 2),
    remote segments (STATE_OUT), one merge at that scale."""
    from mapanything_b200 import ops

    segs = _segments([1369, 1370, 600, 1369], 31)
    geo = Geometry(3, 1369, segs=segs)
    scale = 0.125 * scale_factor
    q, k, v = make_inputs(geo, "needle", 7)
    st = State(geo, 3)
    attend(geo, q, k, v, None, 2, scale, segs[:1], state=(st.o[:2], st.m[:2]), state_out=True, kv_split=2, kv_split_from=9)
    attend(geo, q, k, v, None, 3, scale, segs[1:], state=(st.o[2:], st.m[2:]), state_out=True)
    out = Out(geo)
    out.expect(geo.qrows, None)
    ops.attention_merge((st.o, st.m), out.t, num_heads=geo.H, scale=scale)
    torch.cuda.synchronize()
    keys = geo.keys()
    qidx = sample_rows(geo, keys.shape[1])
    out.check(f"sharded protocol scale {scale:.4g}", "merge", reference(q, k, v, geo, qidx, keys, scale), qidx, scale,
              keys.shape[1])


# ---- kernel choice: both sides of every threshold ---------------------------------------------------------------------


def _threshold_cases():
    """(id, kernel, runner) pairs; the SM count is read at run time."""
    return ["items_below", "items_at", "items_above_odd", "kv4096", "kv4097", "seg_row0_0", "seg_row0_gt0", "plain_many",
            "state_out_many", "split_many"]


@pytest.mark.parametrize("case", _threshold_cases())
def test_kernel_choice(case):
    """n_items 6 x SMs - 1 / 6 x SMs / 6 x SMs + 1 (v3 / v5 / v5); kv_len 4096 / 4097 (v3 / v2); one segment starting at row
    0 / row 5 (v5 / v3); plain / STATE_OUT / kv split on the same many-item shape (v5 / v3 / v2)."""
    n = 6 * _sms()
    if case.startswith("items"):
        nseq = {"items_below": n - 1, "items_at": n, "items_above_odd": n + 1}[case]
        geo = Geometry(1, 100, 70, nseq=nseq, q_gap=1, kv_gap=2)
        run_plain(3 if case == "items_below" else 5, geo, "needle", 0.125, nseq, case)
    elif case.startswith("kv"):
        kv_len = int(case[2:])
        geo = Geometry(2, 130, kv_len)
        run_plain(3 if kv_len == 4096 else 2, geo, "needle", 0.125, kv_len, case)
    elif case.startswith("seg"):
        segs = [(0 if case == "seg_row0_0" else 5, 300)]
        geo = Geometry(4, 128, nseq=-(-n // 4), kv_gap=3, segs=segs)
        run_plain(5 if case == "seg_row0_0" else 3, geo, "needle", 0.125, 1, case, segs=segs)
    else:
        geo = Geometry(8, 128 * -(-n // 8), 200)
        if case == "plain_many":
            run_plain(5, geo, "needle", 0.125, 2, case)
        elif case == "state_out_many":
            run_state_out(3, geo, "needle", 0.125, 2, case)
        else:
            run_split(geo, "needle", 0.125, 2, 2, "0", False, case)
