"""Tensor-level wrappers over the C-ABI kernels.

PyTorch is used for device memory and streams only: every function here hands raw device pointers and
the current CUDA stream to `libmapanything_b200.so`.  `LAUNCHES` counts kernel launches issued through
this module (bench.py reports it as `gpu_launches`); when `PROFILE` is a list, every launch is bracketed by
CUDA events on the launching stream and appended as (family, algorithmic_flops, start_event, end_event, shape tag).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import (MA_ACT_GELU, MA_ACT_NONE, MA_ACT_RELU, MA_ATTN_MAX_SEGMENTS, MA_ATTN_STATE_IN,  # noqa: F401
                   MA_ATTN_STATE_OUT, MA_BF16, MA_F32, AttnExt, GemmEpilogue, check)

LAUNCHES = 0
# files load_images decoded on the GPU (ma_jpeg_decode) and with Pillow
JPEG_ROUTES = {"gpu": 0, "pillow": 0}
PROFILE = None
# weight data_ptr -> (algorithmic N, algorithmic K) for packed weights whose stored shape is larger than the reference layer's:
# K zero-padded for TMA alignment (patch embed 588 -> 640, conv channels to multiples of 8) or tripled by the split-bf16
# packing.  The roofline counts 2*M*N*K of the REFERENCE layer, not the executed MMA work.
ALGO_NK = {}


def register_algorithmic_shape(w: torch.Tensor, n: int, k: int) -> None:
    ALGO_NK[w.data_ptr()] = (int(n), int(k))


def _gemm_kernel_name() -> str:
    code = _lib.load().ma_last_gemm_block()
    return f"gemm_bf16_kernel<2, {code - 2000}>" if code > 2000 else f"gemm_bf16_kernel<1, {code}>"


class launch:
    """Context manager around one kernel launch: counts it and (optionally) times it with CUDA events."""

    __slots__ = ("name", "flops", "n", "s", "tag")

    def __init__(self, name: str, flops: float = 0.0, n: int = 1, tag: str = ""):
        self.name, self.flops, self.n, self.s, self.tag = name, flops, n, None, tag

    def __enter__(self):
        if PROFILE is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, et, ev, tb):
        global LAUNCHES
        if et is None:
            LAUNCHES += self.n
            if PROFILE is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                PROFILE.append((self.name, self.flops, self.s, e, self.tag))
        return False


def _count(n: int = 1) -> None:
    global LAUNCHES
    LAUNCHES += n


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def set_pdl(enabled: Optional[bool]) -> bool:
    """Programmatic dependent launch of the chained GEMM / attention / LayerNorm kernels (include/mapanything_b200.h:
    ma_set_pdl).  None queries.  Returns the previous setting."""
    return bool(_lib.load().ma_set_pdl(-1 if enabled is None else int(bool(enabled))))


def set_stream_k(enabled: Optional[bool]) -> bool:
    """Stream-K tail of the in-place fp32 residual GEMMs (include/mapanything_b200.h: ma_set_stream_k): faster, reproducible
    to fp32 rounding instead of bit for bit.  None queries.  Returns the previous setting."""
    return bool(_lib.load().ma_set_stream_k(-1 if enabled is None else int(bool(enabled))))


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.bfloat16:
        return MA_BF16
    if t.dtype == torch.float32:
        return MA_F32
    raise TypeError(f"unsupported dtype {t.dtype}")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _f32c(t: Optional[torch.Tensor], n: int, name: str) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n or not t.is_cuda:
        raise ValueError(f"{name} must be a contiguous CUDA float32 tensor with {n} elements")
    return t


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous CUDA {dtype} tensor")
    return t


def _epilogue(out, N, bias, act, colscale, residual, residual_row_mod, out_relu, rows_per_group_in, rows_per_group_out,
              row_offset_out, act_after_residual, relu_out_before_residual) -> GemmEpilogue:
    ep = GemmEpilogue()
    ep.out = out.data_ptr()
    ep.ldo = out.stride(-2)
    ep.out_dtype = _dt(out)
    ep.act = act
    ep.bias = _ptr(_f32c(bias, N, "bias"))
    ep.colscale = _ptr(_f32c(colscale, N, "colscale"))
    if residual is not None:
        ep.residual = residual.data_ptr()
        ep.ldr = residual.stride(-2)
        ep.residual_dtype = _dt(residual)
    ep.residual_row_mod = residual_row_mod
    if out_relu is not None:
        if out_relu.dtype != torch.bfloat16:
            raise TypeError("out_relu must be bfloat16")
        ep.out_relu = out_relu.data_ptr()
        ep.ldo_relu = out_relu.stride(-2)
    ep.rows_per_group_in = rows_per_group_in
    ep.rows_per_group_out = rows_per_group_out
    ep.row_offset_out = row_offset_out
    ep.flags = (1 if act_after_residual else 0) | (2 if relu_out_before_residual else 0)
    return ep


def gemm(
    x: torch.Tensor,
    w: torch.Tensor,
    out: torch.Tensor,
    *,
    bias: Optional[torch.Tensor] = None,
    act: int = MA_ACT_NONE,
    colscale: Optional[torch.Tensor] = None,
    residual: Optional[torch.Tensor] = None,
    residual_row_mod: int = 0,
    out_relu: Optional[torch.Tensor] = None,
    rows_per_group_in: int = 0,
    rows_per_group_out: int = 0,
    row_offset_out: int = 0,
    block_n: int = 0,
    act_after_residual: bool = False,
    relu_out_before_residual: bool = False,
) -> torch.Tensor:
    """out = epilogue(x @ w.T); x [M,K] bf16, w [N,K] bf16 (row strides may exceed K). See ma_gemm_bf16."""
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise TypeError("gemm operands must be bfloat16")
    if x.dim() != 2 or w.dim() != 2 or x.stride(1) != 1 or w.stride(1) != 1 or out.stride(-1) != 1:
        raise ValueError("gemm operands must be 2-D with contiguous rows")
    M, K = x.shape
    N, Kw = w.shape
    if K != Kw:
        raise ValueError(f"K mismatch: x {tuple(x.shape)} vs w {tuple(w.shape)}")
    ep = _epilogue(out, N, bias, act, colscale, residual, residual_row_mod, out_relu, rows_per_group_in, rows_per_group_out,
                   row_offset_out, act_after_residual, relu_out_before_residual)
    lib = _lib.load()
    n_alg, k_alg = ALGO_NK.get(w.data_ptr(), (N, K))
    with launch("gemm", 2.0 * M * n_alg * k_alg, tag=f"{M}x{N}x{K}") as rec:
        check(
            lib.ma_gemm_bf16(x.data_ptr(), x.stride(0), w.data_ptr(), w.stride(0), M, N, K, C.byref(ep), block_n, _stream()),
            "ma_gemm_bf16",
        )
        if PROFILE is not None:
            rec.tag = f"{M}x{N}x{K}|{_gemm_kernel_name()}"
    return out


def conv3x3_head(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: int, head_w: torch.Tensor,
                 head_bias: torch.Tensor, head_out: torch.Tensor) -> torch.Tensor:
    """3x3 conv (Cout = 128) whose output is consumed in the epilogue by a narrow linear head instead of being stored:
    head_out[pixel][j] = head_bias[j] + sum_c head_w[j][c] * act(conv(x)[pixel][c] + bias[c]), j < 8 (fp32, row stride 8).
    x NHWC bf16, w [128, 9*C] bf16, head_w fp32 [8][128], head_bias fp32 [8].  See ma_gemm_epilogue.head_*."""
    _req(x, torch.bfloat16, "x")
    n, H, W, C_ = x.shape
    Cout = w.shape[0]
    if Cout != 128 or w.shape[1] != 9 * C_ or head_w.shape != (8, 128) or head_out.shape[-1] != 8:
        raise ValueError("conv3x3_head: needs Cout == 128, head_w [8,128], head_out [..., 8]")
    _req(head_w, torch.float32, "head_w")
    _req(head_bias, torch.float32, "head_bias")
    _req(head_out, torch.float32, "head_out")
    ep = GemmEpilogue()
    ep.out_dtype = MA_BF16
    ep.act = act
    ep.bias = _ptr(_f32c(bias, Cout, "bias"))
    ep.head_w, ep.head_bias, ep.head_out = head_w.data_ptr(), head_bias.data_ptr(), head_out.data_ptr()
    n_alg, k_alg = ALGO_NK.get(w.data_ptr(), (Cout, 9 * C_))
    with launch("conv3x3", 2.0 * n * H * W * (n_alg * k_alg + 8 * Cout), tag=f"{n}x{H}x{W}x{C_}->{Cout}+head") as rec:
        check(_lib.load().ma_conv3x3_bf16(x.data_ptr(), n, H, W, C_, w.data_ptr(), w.stride(0), Cout, C.byref(ep), 0, _stream()),
              "ma_conv3x3_bf16")
        if PROFILE is not None:
            rec.tag = f"{n}x{H}x{W}x{C_}->{Cout}+head|{_gemm_kernel_name()}"
    return head_out


def conv3x3(
    x: torch.Tensor,
    w: torch.Tensor,
    out: torch.Tensor,
    *,
    bias: Optional[torch.Tensor] = None,
    act: int = MA_ACT_NONE,
    residual: Optional[torch.Tensor] = None,
    out_relu: Optional[torch.Tensor] = None,
    block_n: int = 0,
    act_after_residual: bool = False,
    relu_out_before_residual: bool = False,
) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 conv as implicit GEMM: x NHWC bf16 (n,H,W,C) contiguous, w [Cout, 9*C] bf16 (tap-major),
    out [n*H*W, Cout] (rows = pixels). See ma_conv3x3_bf16."""
    _req(x, torch.bfloat16, "x")
    if w.dtype != torch.bfloat16 or w.dim() != 2 or w.stride(1) != 1 or out.stride(-1) != 1:
        raise ValueError("conv3x3: w must be 2-D bf16 with contiguous rows")
    n, H, W, C_ = x.shape
    Cout = w.shape[0]
    if w.shape[1] != 9 * C_ or out.shape[-1] != Cout or out.numel() // Cout != n * H * W:
        raise ValueError(f"conv3x3: shape mismatch x {tuple(x.shape)} w {tuple(w.shape)} out {tuple(out.shape)}")
    ep = _epilogue(out, Cout, bias, act, None, residual, 0, out_relu, 0, 0, 0, act_after_residual, relu_out_before_residual)
    n_alg, k_alg = ALGO_NK.get(w.data_ptr(), (Cout, 9 * C_))
    with launch("conv3x3", 2.0 * n * H * W * n_alg * k_alg, tag=f"{n}x{H}x{W}x{C_}->{Cout}") as rec:
        check(_lib.load().ma_conv3x3_bf16(x.data_ptr(), n, H, W, C_, w.data_ptr(), w.stride(0), Cout, C.byref(ep), block_n,
                                          _stream()), "ma_conv3x3_bf16")
        if PROFILE is not None:
            rec.tag = f"{n}x{H}x{W}x{C_}->{Cout}|{_gemm_kernel_name()}"
    return out


def attention(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    out: torch.Tensor,
    *,
    num_heads: int,
    num_seqs: int,
    q_len: int,
    kv_len: int,
    q_seq_stride: Optional[int] = None,
    kv_seq_stride: Optional[int] = None,
    scale: Optional[float] = None,
    kv_segments=None,
    state=None,
    state_in: bool = False,
    state_out: bool = False,
    kv_split: int = 1,
    kv_split_from: int = 0,
) -> torch.Tensor:
    """softmax(q k^T * scale) v per (sequence, head), head_dim 64.

    q/k/v/out are 2-D token-major bf16 views whose rows may be strided column slices of a wider matrix
    (e.g. qkv[:, :D], qkv[:, D:2D], qkv[:, 2D:]); no head permutation is materialised. See ma_attention_fwd.

    kv_segments: optional list of (row0, length) key/value row ranges (sum of lengths == kv_len).
    state = (state_o fp32 [q_rows, heads*64], state_m fp32 [q_rows, heads]): with state_out the launch writes the
    online-softmax state instead of `out`; with state_in it resumes from it.  kv_split > 1 (with state_out): the key range
    is cut into kv_split parts, one CTA each, and `state` holds one partial per part: (fp32 [kv_split, q_rows, heads*64],
    fp32 [kv_split, q_rows, heads], the latter pre-filled with -inf); join them with attention_merge.  kv_split_from: only
    (query block, head) slots from that index on are split (the others write `out` / part 0).  See ma_attention_fwd_ex."""
    width = num_heads * 64
    for name, t in (("q", q), ("k", k), ("v", v), ("out", out)):
        if t is None:
            continue
        if t.dtype != torch.bfloat16 or t.dim() != 2 or t.stride(1) != 1:
            raise ValueError("attention operands must be 2-D bf16 with contiguous rows")
        # the library sees only the row stride: a narrower view would let the heads run into the parent's next columns
        if t.shape[1] < width:
            raise ValueError(f"attention: {name} has {t.shape[1]} columns, {num_heads} heads need {width}")
    if q_seq_stride is None:
        q_seq_stride = q_len
    if kv_seq_stride is None:
        kv_seq_stride = kv_len
    q_rows = (num_seqs - 1) * q_seq_stride + q_len   # query rows the call reads and writes
    if out is not None and out.shape[0] < q_rows:
        raise ValueError(f"attention: out has {out.shape[0]} rows, the call writes {q_rows}")
    if scale is None:
        scale = 64 ** -0.5
    lib = _lib.load()
    # Column offsets are folded into the base pointers; the tensor map width is the row stride, which
    # always covers [col0, col0 + heads*64) of the parent matrix when the view is a column slice of it.
    if kv_split > 1 and state is None:
        raise ValueError("kv_split > 1 writes partial states: pass state=...")
    ext = None
    if kv_segments is not None or state_in or state_out or kv_split > 1:
        ext = AttnExt()
        if kv_segments is not None:
            if len(kv_segments) > MA_ATTN_MAX_SEGMENTS:
                raise ValueError(f"at most {MA_ATTN_MAX_SEGMENTS} kv segments")
            ext.n_segments = len(kv_segments)
            for i, (r0, ln) in enumerate(kv_segments):
                ext.seg_row0[i], ext.seg_len[i] = int(r0), int(ln)
        if state_in or state_out or kv_split > 1:
            so, sm = state
            if so.dim() == 2:
                so, sm = so.unsqueeze(0), sm.unsqueeze(0)
            if (so.dtype != torch.float32 or sm.dtype != torch.float32 or so.stride(2) != 1 or sm.stride(2) != 1
                    or sm.stride(1) != num_heads or so.shape[1] < q.shape[0] or sm.shape[1:] != (so.shape[1], num_heads)
                    or so.shape[0] < kv_split or sm.shape[0] < kv_split):
                raise ValueError("attention state must be (fp32 [parts, q_rows, >=heads*64], fp32 [parts, q_rows, heads])")
            if so.shape[2] < width:
                raise ValueError(f"attention: state_o has {so.shape[2]} columns, {num_heads} heads need {width}")
            ext.flags = (MA_ATTN_STATE_IN if state_in else 0) | (MA_ATTN_STATE_OUT if state_out else 0)
            ext.state_o, ext.ld_state_o, ext.state_m = so.data_ptr(), so.stride(1), sm.data_ptr()
            ext.kv_split, ext.split_stride_o, ext.split_stride_m = kv_split, so.stride(0), sm.stride(0)
            ext.kv_split_from = kv_split_from
    with launch("attention", 4.0 * num_seqs * num_heads * q_len * kv_len * 64, tag=f"{num_seqs}x{num_heads}x{q_len}x{kv_len}"):
        check(
            lib.ma_attention_fwd_ex(
                q.data_ptr(), q.stride(0), q.shape[0], 0,
                k.data_ptr(), k.stride(0), k.shape[0], 0,
                v.data_ptr(), v.stride(0), 0,
                _ptr(out), out.stride(0) if out is not None else num_heads * 64, 0,
                num_seqs, num_heads, q_len, kv_len, q_seq_stride, kv_seq_stride, float(scale),
                C.byref(ext) if ext is not None else None, _stream(),
            ),
            "ma_attention_fwd_ex",
        )
    return out


def attention_merge(state, out: torch.Tensor, *, num_heads: int, scale: Optional[float] = None, first_slot: int = -1) -> torch.Tensor:
    """Joins partial softmax states (fp32 [parts, rows, heads*64], fp32 [parts, rows, heads]) into bf16 out [rows, heads*64]
    (ma_attention_merge)."""
    so, sm = state
    if so.dim() != 3 or sm.dim() != 3 or so.dtype != torch.float32 or sm.dtype != torch.float32 or so.stride(2) != 1:
        raise ValueError("attention_merge: state must be (fp32 [parts, rows, D], fp32 [parts, rows, heads])")
    if out.dtype != torch.bfloat16 or out.stride(1) != 1 or sm.stride(1) != num_heads or sm.stride(2) != 1:
        raise ValueError("attention_merge: out must be bf16 with contiguous rows")
    parts, rows = so.shape[0], out.shape[0]
    width = num_heads * 64
    if out.shape[1] < width:
        raise ValueError(f"attention_merge: out has {out.shape[1]} columns, {num_heads} heads need {width}")
    if so.shape[2] < width or so.shape[1] < rows:
        raise ValueError(f"attention_merge: state_o is [{so.shape[1]}, {so.shape[2]}] per part, out needs [{rows}, {width}]")
    if sm.shape[0] < parts or sm.shape[1] < rows:
        raise ValueError(f"attention_merge: state_m has {sm.shape[0]} parts of {sm.shape[1]} rows, state_o {parts} of {rows}")
    if scale is None:
        scale = 64 ** -0.5
    with launch("attention_merge"):
        check(_lib.load().ma_attention_merge(so.data_ptr(), so.stride(1), so.stride(0), sm.data_ptr(), sm.stride(0), parts, rows,
                                             num_heads, float(scale), out.data_ptr(), out.stride(0), first_slot, _stream()),
              "ma_attention_merge")
    return out


def patchify(img: torch.Tensor, out: torch.Tensor, patch: int) -> torch.Tensor:
    """(n,3,H,W) fp32 -> out [n*hp*wp, kpad] bf16 (ma_patchify)."""
    _req(img, torch.float32, "img")
    _req(out, torch.bfloat16, "out")
    n, c, H, W = img.shape
    assert c == 3 and out.shape[0] == n * (H // patch) * (W // patch)
    with launch("patchify"):
        check(_lib.load().ma_patchify(img.data_ptr(), out.data_ptr(), n, H, W, patch, out.shape[1], _stream()), "ma_patchify")
    return out


def layernorm(
    x: torch.Tensor,
    out: torch.Tensor,
    gamma: torch.Tensor,
    beta: torch.Tensor,
    *,
    rows: Optional[int] = None,
    eps: float = 1e-6,
    rows_per_group: int = 0,
    in_group_stride: int = 0,
    in_row_offset: int = 0,
    out_group_stride: int = 0,
    out_row_offset: int = 0,
) -> torch.Tensor:
    """LayerNorm over the last dim of 2-D row-major x -> out, with optional row remapping (ma_layernorm)."""
    C_ = x.shape[-1]
    if rows is None:
        rows = x.shape[0]
    if x.stride(-1) != 1 or out.stride(-1) != 1 or out.shape[-1] != C_:
        raise ValueError("layernorm: rows must be contiguous and widths must match")
    _f32c(gamma, C_, "gamma")
    _f32c(beta, C_, "beta")
    with launch("layernorm"):
        check(
            _lib.load().ma_layernorm(
                x.data_ptr(), _dt(x), x.stride(-2), out.data_ptr(), _dt(out), out.stride(-2), gamma.data_ptr(),
                beta.data_ptr(), rows, C_, float(eps), rows_per_group, in_group_stride, in_row_offset, out_group_stride,
                out_row_offset, _stream(),
            ),
            "ma_layernorm",
        )
    return out


def set_rows(dst: torch.Tensor, a: torch.Tensor, b: Optional[torch.Tensor], *, groups: int, group_stride: int,
             row_offset: int) -> torch.Tensor:
    C_ = dst.shape[-1]
    if dst.dtype != torch.float32 or dst.stride(-1) != 1:
        raise ValueError("set_rows: dst must be fp32 with contiguous rows")
    _f32c(a, C_, "a")
    _f32c(b, C_, "b")
    with launch("set_rows"):
        check(_lib.load().ma_set_rows(dst.data_ptr(), dst.stride(-2), groups, group_stride, row_offset, a.data_ptr(), _ptr(b),
                                      C_, _stream()), "ma_set_rows")
    return dst


def im2col3x3(x: torch.Tensor, out: torch.Tensor, stride: int = 1) -> torch.Tensor:
    """NHWC bf16 (n,H,W,C) -> out [n*Ho*Wo, 9*C] (ma_im2col3x3)."""
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    n, H, W, C_ = x.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    assert out.numel() == n * Ho * Wo * 9 * C_, "im2col3x3: bad output size"
    with launch("im2col"):
        check(_lib.load().ma_im2col3x3(x.data_ptr(), out.data_ptr(), n, H, W, C_, stride, _stream()), "ma_im2col3x3")
    return out


def fill_f32(x: torch.Tensor, value: float) -> torch.Tensor:
    """x[...] = value (contiguous fp32; ma_fill_f32)."""
    _req(x, torch.float32, "x")
    with launch("fill"):
        check(_lib.load().ma_fill_f32(x.data_ptr(), x.numel(), float(value), _stream()), "ma_fill_f32")
    return x


def pixel_shuffle(x: torch.Tensor, out: torch.Tensor, n: int, h: int, w: int, C_: int, s: int) -> torch.Tensor:
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    assert x.numel() == n * h * w * s * s * C_ == out.numel()
    with launch("pixel_shuffle"):
        check(_lib.load().ma_pixel_shuffle(x.data_ptr(), out.data_ptr(), n, h, w, C_, s, _stream()), "ma_pixel_shuffle")
    return out


def pixel_shuffle_f32(x: torch.Tensor, out: torch.Tensor, n: int, h: int, w: int, C_: int, s: int) -> torch.Tensor:
    """fp32 rows [(i,y,x)][(ky*s+kx)*C + c] (row stride x.stride(0)) -> out rows [(i, y*s+ky, x*s+kx)][0:C] (ma_pixel_shuffle_f32)."""
    if x.dtype != torch.float32 or out.dtype != torch.float32 or x.stride(-1) != 1 or out.stride(-1) != 1:
        raise ValueError("pixel_shuffle_f32: fp32 tensors with contiguous rows")
    if x.shape[0] != n * h * w or out.shape[0] != n * h * w * s * s:
        raise ValueError("pixel_shuffle_f32: row counts do not match (n, h, w, s)")
    with launch("pixel_shuffle"):
        check(_lib.load().ma_pixel_shuffle_f32(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), n, h, w, C_, s, _stream()),
              "ma_pixel_shuffle_f32")
    return out


def bilinear_ac(x: torch.Tensor, out: torch.Tensor, virtual_hw=None) -> torch.Tensor:
    """NHWC bf16 bilinear resize with align_corners=True; out (n,Ho,Wo,C); virtual_hw = uncropped output size."""
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    n, Hin, Win, C_ = x.shape
    _, Ho, Wo, _ = out.shape
    Hv, Wv = virtual_hw if virtual_hw is not None else (Ho, Wo)
    with launch("bilinear"):
        check(_lib.load().ma_bilinear_align_corners(x.data_ptr(), out.data_ptr(), n, Hin, Win, C_, Hv, Wv, Ho, Wo, _stream()),
              "ma_bilinear_align_corners")
    return out


def token_mean(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """bf16 (n,T,C) -> (n,C)."""
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    n, T, C_ = x.shape
    with launch("token_mean"):
        check(_lib.load().ma_token_mean(x.data_ptr(), out.data_ptr(), n, T, C_, _stream()), "ma_token_mean")
    return out


def head_linear_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor) -> torch.Tensor:
    """out[:, :N] = x @ w.T + bias for N <= 8, K <= 256: x bf16 [rows,K], w bf16 [N,K], out fp32 [rows, >=N] (ma_head_linear_small)."""
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16 or out.dtype != torch.float32 or x.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError("head_linear_small: bf16 x / w with contiguous rows, fp32 out")
    rows, K = x.shape
    N = w.shape[0]
    with launch("head_linear", 2.0 * rows * N * K):
        check(_lib.load().ma_head_linear_small(x.data_ptr(), x.stride(0), w.data_ptr(), w.stride(0), _ptr(_f32c(bias, N, "bias")),
                                               out.data_ptr(), out.stride(0), rows, N, K, _stream()), "ma_head_linear_small")
    return out


def split3(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 [rows][C] (any row stride) -> bf16 [rows][3C] = [hi | lo | hi] (ma_split_bf16x3)."""
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("split3: x must be 2-D fp32 with contiguous rows")
    rows, C_ = x.shape
    if out is None:
        out = torch.empty(rows, 3 * C_, device=x.device, dtype=torch.bfloat16)
    _req(out, torch.bfloat16, "out")
    with launch("split3"):
        check(_lib.load().ma_split_bf16x3(x.data_ptr(), x.stride(0), out.data_ptr(), rows, C_, _stream()), "ma_split_bf16x3")
    return out


def token_mean_f32(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """fp32 (n,T,C) -> (n,C)."""
    _req(x, torch.float32, "x")
    _req(out, torch.float32, "out")
    n, T, C_ = x.shape
    with launch("token_mean"):
        check(_lib.load().ma_token_mean_f32(x.data_ptr(), out.data_ptr(), n, T, C_, _stream()), "ma_token_mean_f32")
    return out


LINEAR_ROWS_MAX = 16


def linear_rows_f32(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor, act: int = MA_ACT_NONE):
    """out[r] = act(b + W x[r]) in plain fp32 for x of at most LINEAR_ROWS_MAX rows (ma_linear_rows_f32)."""
    _req(x, torch.float32, "x")
    _req(w, torch.float32, "w")
    _req(out, torch.float32, "out")
    rows, K = x.shape
    N = w.shape[0]
    if w.shape[1] != K or out.shape != (rows, N) or x.stride(1) != 1 or w.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError(f"linear_rows_f32: shape mismatch x {tuple(x.shape)} w {tuple(w.shape)} out {tuple(out.shape)}")
    with launch("linear_rows"):
        check(_lib.load().ma_linear_rows_f32(x.data_ptr(), x.stride(0), w.data_ptr(), w.stride(0),
                                             _ptr(_f32c(bias, N, "bias")) if bias is not None else None, act, out.data_ptr(),
                                             out.stride(0), rows, N, K, _stream()), "ma_linear_rows_f32")
    return out


def decode_dense(raw: torch.Tensor, pose_raw: torch.Tensor, scale_raw: torch.Tensor, n: int, H: int, W: int):
    """Fused adaptor + decode (ma_decode_dense). raw fp32 [n*H*W, ld>=6]; returns the dict of forward() tensors."""
    if raw.dtype != torch.float32 or raw.stride(-1) != 1:
        raise ValueError("decode_dense: raw must be fp32 with contiguous rows")
    _req(pose_raw, torch.float32, "pose_raw")
    _req(scale_raw, torch.float32, "scale_raw")
    dev = raw.device
    f32 = dict(device=dev, dtype=torch.float32)
    o = {
        "pts3d": torch.empty(n, H, W, 3, **f32), "pts3d_cam": torch.empty(n, H, W, 3, **f32),
        "ray_directions": torch.empty(n, H, W, 3, **f32), "depth_along_ray": torch.empty(n, H, W, 1, **f32),
        "conf": torch.empty(n, H, W, **f32), "non_ambiguous_mask_logits": torch.empty(n, H, W, **f32),
        "non_ambiguous_mask": torch.empty(n, H, W, device=dev, dtype=torch.bool),
        "cam_trans": torch.empty(n, 3, **f32), "cam_quats": torch.empty(n, 4, **f32),
        "metric_scaling_factor": torch.empty(1, 1, **f32),
    }
    with launch("decode"):
        check(
            _lib.load().ma_decode_dense(
                raw.data_ptr(), raw.stride(0), pose_raw.data_ptr(), scale_raw.data_ptr(), n, H * W, o["pts3d"].data_ptr(),
                o["pts3d_cam"].data_ptr(), o["ray_directions"].data_ptr(), o["depth_along_ray"].data_ptr(),
                o["conf"].data_ptr(), o["non_ambiguous_mask_logits"].data_ptr(), o["non_ambiguous_mask"].data_ptr(),
                o["cam_trans"].data_ptr(), o["cam_quats"].data_ptr(), o["metric_scaling_factor"].data_ptr(), _stream(),
            ),
            "ma_decode_dense",
        )
    return o


def decode_scene(raw: torch.Tensor, pose_raw: Optional[torch.Tensor], scale_raw: torch.Tensor, n: int, H: int, W: int, *,
                 rep: str, has_conf: bool, has_mask: bool, point_mode: str = "exp", use_factored: bool = False,
                 conf_vmin: float = 1.0):
    """ma_decode_scene: the fused adaptor + decode for every scene representation of reference model.py:407-587 / :1618-1907.
    raw fp32 [n*H*W, ld]; pose_raw fp32 [n, 7] for the posed representations, else None.  Returns the forward() tensors the
    representation defines (as [n, ...]) + metric_scaling_factor [1, 1]."""
    if raw.dtype != torch.float32 or raw.stride(-1) != 1:
        raise ValueError("decode_scene: raw must be fp32 with contiguous rows")
    if rep not in _lib.MA_REP or point_mode not in _lib.MA_PTS:
        raise ValueError(f"decode_scene: unknown representation {rep!r} / pointmap_mode {point_mode!r}")
    posed = "pose" in rep
    if posed != (pose_raw is not None):
        raise ValueError("decode_scene: pose_raw is given exactly for the posed representations")
    _req(scale_raw, torch.float32, "scale_raw")
    dev = raw.device
    f32 = dict(device=dev, dtype=torch.float32)
    o = {"pts3d": torch.empty(n, H, W, 3, **f32), "metric_scaling_factor": torch.empty(1, 1, **f32)}
    if posed:
        _req(pose_raw, torch.float32, "pose_raw")
        o.update(pts3d_cam=torch.empty(n, H, W, 3, **f32), cam_trans=torch.empty(n, 3, **f32), cam_quats=torch.empty(n, 4, **f32))
    if rep == "raymap+depth":
        o["ray_origins"] = torch.empty(n, H, W, 3, **f32)
    if rep != "pointmap":
        o.update(ray_directions=torch.empty(n, H, W, 3, **f32), depth_along_ray=torch.empty(n, H, W, 1, **f32))
    if has_conf:
        o["conf"] = torch.empty(n, H, W, **f32)
    if has_mask:
        o["non_ambiguous_mask_logits"] = torch.empty(n, H, W, **f32)
        o["non_ambiguous_mask"] = torch.empty(n, H, W, device=dev, dtype=torch.bool)
    spec = _lib.DecodeSpec(_lib.MA_REP[rep], int(has_conf), int(has_mask), _lib.MA_PTS[point_mode], int(use_factored),
                           float(conf_vmin))

    def ptr(key):
        return o[key].data_ptr() if key in o else None

    with launch("decode"):
        check(
            _lib.load().ma_decode_scene(
                C.byref(spec), raw.data_ptr(), raw.stride(0), _ptr(pose_raw), scale_raw.data_ptr(), n, H * W, ptr("pts3d"),
                ptr("pts3d_cam"), ptr("ray_directions"), ptr("ray_origins"), ptr("depth_along_ray"), ptr("conf"),
                ptr("non_ambiguous_mask_logits"), ptr("non_ambiguous_mask"), ptr("cam_trans"), ptr("cam_quats"),
                o["metric_scaling_factor"].data_ptr(), _stream(),
            ),
            "ma_decode_scene",
        )
    return o


# ------------------------------------------------------------------------------------------ geometric inputs
def unshuffle_split(x: torch.Tensor, patch: int, cpad: int, factor: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 NHWC (n,H,W,cin) -> bf16 (n,H/p,W/p,3*cpad) split layout (ma_unshuffle_split); factor -> depth mode."""
    _req(x, torch.float32, "x")
    n, H, W, cin = x.shape
    out = torch.empty(n, H // patch, W // patch, 3 * cpad, device=x.device, dtype=torch.bfloat16)
    with launch("unshuffle"):
        check(_lib.load().ma_unshuffle_split(x.data_ptr(), out.data_ptr(), n, H, W, cin, patch, cpad, 0 if factor is None else 1,
                                             _ptr(factor), _stream()), "ma_unshuffle_split")
    return out


def depth_factor(depth: torch.Tensor):
    """fp32 (n,H,W,1) -> (factor fp32 [n], log_factor8 fp32 [n,8]) (ma_depth_factor)."""
    _req(depth, torch.float32, "depth")
    n = depth.shape[0]
    f = torch.empty(n, device=depth.device, dtype=torch.float32)
    lf = torch.empty(n, 8, device=depth.device, dtype=torch.float32)
    with launch("depth_factor"):
        check(_lib.load().ma_depth_factor(depth.data_ptr(), n, depth.numel() // n, f.data_ptr(), lf.data_ptr(), _stream()),
              "ma_depth_factor")
    return f, lf


def pose_inputs(quats: torch.Tensor, trans: torch.Tensor, has_pose: torch.Tensor):
    """quats fp32 [V,4], trans fp32 [V,3], has_pose uint8 [V] -> (quats8, trans8, log_scale8) fp32 [V,8] (ma_pose_inputs)."""
    _req(quats, torch.float32, "quats")
    _req(trans, torch.float32, "trans")
    _req(has_pose, torch.uint8, "has_pose")
    V = quats.shape[0]
    q8, t8, s8 = (torch.empty(V, 8, device=quats.device, dtype=torch.float32) for _ in range(3))
    with launch("pose_inputs"):
        check(_lib.load().ma_pose_inputs(quats.data_ptr(), trans.data_ptr(), has_pose.data_ptr(), V, q8.data_ptr(),
                                         t8.data_ptr(), s8.data_ptr(), _stream()), "ma_pose_inputs")
    return q8, t8, s8


def fuse_add(feat: torch.Tensor, V: int, N: int, dense_a=None, a_slot=None, dense_b=None, b_slot=None, globals_=(), gw=None):
    """In place: feat fp32 [V*N,C] += dense / global geometric features (ma_fuse_add)."""
    _req(feat, torch.float32, "feat")
    g = [None] * 4
    for i, t in enumerate(globals_):
        g[i] = None if t is None else _req(t, torch.float32, "global feature")
    with launch("fuse_add"):
        check(_lib.load().ma_fuse_add(feat.data_ptr(), V, N, feat.shape[1], _ptr(dense_a), _ptr(a_slot), _ptr(dense_b),
                                      _ptr(b_slot), _ptr(g[0]), _ptr(g[1]), _ptr(g[2]), _ptr(g[3]), _ptr(gw), _stream()),
              "ma_fuse_add")
    return feat
