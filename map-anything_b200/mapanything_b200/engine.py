"""Execution engine: packs the parameter tree into kernel-ready device buffers and drives the CUDA kernels.

Data layout in HBM (B200-first, no NCHW anywhere inside):
  * activations are TOKEN-MAJOR / NHWC: row = (view, y, x), channels contiguous -- the ViT token layout, the
    GEMM row-major A operand, and the im2col-free layout of the DPT convolutions are the same thing, so the
    reference's permute().contiguous() and torch.cat copies (model.py:1245-1259, :1549-1572) never happen;
  * the residual streams of both transformers are fp32 (what the reference's bf16 autocast keeps them in),
    every GEMM/attention operand is bf16, accumulation is fp32 in TMEM;
  * weights are packed once: Linear/conv1x1 as [N][K] bf16, conv3x3 as [Cout][(ky,kx),Cin],
    ConvTranspose(k=s) as [(ky,kx),Cout][Cin]; biases / LayerNorm / LayerScale vectors stay fp32.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .ops import MA_ACT_GELU, MA_ACT_NONE, MA_ACT_RELU


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.bfloat16).contiguous()


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


class Lin:
    """Packed y = x W^T + b."""

    def __init__(self, w: torch.Tensor, b: Optional[torch.Tensor], kpad: int = 0, algo_nk=None):
        w2 = w.detach().reshape(w.shape[0], -1)
        k0 = w2.shape[1]
        if kpad and kpad > w2.shape[1]:
            w2 = torch.cat([w2, w2.new_zeros(w2.shape[0], kpad - w2.shape[1])], dim=1)
        self.w = _bf16(w2)
        self.b = _f32(b) if b is not None else None
        self.n, self.k = self.w.shape
        ops.register_algorithmic_shape(self.w, *(algo_nk or (self.n, k0)))   # zero padding is not algorithmic work


class Lin3:
    """y = x W^T + b evaluated to ~fp32 accuracy on the bf16 tensor cores (see ma_split_bf16x3): the weight is packed as
    [w_hi | w_hi | w_lo] per `group` input channels, matching activations split as [a_hi | a_lo | a_hi].
    group = K for a Linear / 1x1 conv; group = Cin for the (tap-major) im2col layout of a 3x3 conv."""

    def __init__(self, w2d: torch.Tensor, b: Optional[torch.Tensor], group: Optional[int] = None, algo_nk=None):
        w2d = w2d.detach().float().reshape(w2d.shape[0], -1)
        n, k = w2d.shape
        group = group or k
        w = w2d.view(n, k // group, group)
        hi = w.to(torch.bfloat16)
        lo = (w - hi.float()).to(torch.bfloat16)
        self.w = torch.cat([hi, hi, lo], dim=2).reshape(n, 3 * k).contiguous()
        self.w32 = w2d.contiguous() if group == k else None   # plain fp32 copy for the few-row kernel (ops.linear_rows_f32)
        self.b = _f32(b) if b is not None else None
        self.n, self.k = n, 3 * k
        ops.register_algorithmic_shape(self.w, *(algo_nk or (n, k)))   # the 3x of the split is not algorithmic work


def _conv3x3(conv: nn.Conv2d) -> Lin:
    return Lin(conv.weight.detach().permute(0, 2, 3, 1), conv.bias)  # [Cout][ky][kx][Cin]


def _conv1x1(conv: nn.Conv2d) -> Lin:
    return Lin(conv.weight, conv.bias)


def _convT(conv: nn.ConvTranspose2d) -> Lin:
    cin, cout, k, _ = conv.weight.shape
    w = conv.weight.detach().permute(2, 3, 1, 0).reshape(k * k * cout, cin)  # [(ky,kx,co)][ci]
    b = conv.bias.detach().repeat(k * k) if conv.bias is not None else None
    return Lin(w, b)


def _sinusoid_table(n_rows: int, dim: int, base: float = 10000.0) -> torch.Tensor:
    """MAE / CroCo-style fixed table (SURVEY App. A.3): angle[pos, j] = pos / base^(2 (j // 2) / dim), sin on even j, cos on odd."""
    pos = torch.arange(n_rows, dtype=torch.float64)[:, None]
    j = torch.arange(dim, dtype=torch.float64)[None, :]
    angle = pos / torch.pow(torch.tensor(base, dtype=torch.float64), 2 * torch.div(j, 2, rounding_mode="floor") / dim)
    return torch.where((torch.arange(dim) % 2 == 0)[None, :], torch.sin(angle), torch.cos(angle)).float()


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _conv3x3_padded(conv: nn.Conv2d, cin_pad: int, cout_pad: int, split: bool = False):
    """3x3 conv weight [Cout][Cin][3][3] -> tap-major [cout_pad][9*cin_pad] with zero padded channels (TMA needs
    channel counts that are multiples of 8; e.g. 588 -> 592).  split=True packs it for split-bf16 activations."""
    w = conv.weight.detach().float().permute(0, 2, 3, 1)  # [Cout][ky][kx][Cin]
    cout, _, _, cin = w.shape
    wp = w.new_zeros(cout_pad, 3, 3, cin_pad)
    wp[:cout, :, :, :cin] = w
    b = conv.bias.detach().float() if conv.bias is not None else w.new_zeros(cout)
    bp = b.new_zeros(cout_pad)
    bp[:cout] = b
    if split:
        return Lin3(wp.reshape(cout_pad, 9 * cin_pad), bp, group=cin_pad, algo_nk=(cout, 9 * cin))
    return Lin(wp.reshape(cout_pad, 9 * cin_pad), bp, algo_nk=(cout, 9 * cin))


def _linear_padded(w: torch.Tensor, b: Optional[torch.Tensor], kpad: int, npad: int) -> Lin:
    w = w.detach().float().reshape(w.shape[0], -1)
    wp = w.new_zeros(npad, kpad)
    wp[:w.shape[0], :w.shape[1]] = w
    bp = w.new_zeros(npad)
    if b is not None:
        bp[:w.shape[0]] = b.detach().float()
    return Lin(wp, bp, algo_nk=(w.shape[0], w.shape[1]))


class DenseEncW:
    """Packed `dense_rep_encoder` (SURVEY App. A.2): PixelUnshuffle -> conv3x3 -> 2 residual blocks -> conv1x1 -> LayerNorm."""

    def __init__(self, enc):
        self.patch, self.in_chans = enc.patch_size, enc.in_chans
        self.cpad0 = _pad8(enc.in_chans * enc.patch_size ** 2)
        d0 = enc.conv_in.out_channels
        # first conv in split-bf16 precision: its input is raw geometry (unit rays / log depth), fp32 in the reference
        self.conv_in = _conv3x3_padded(enc.conv_in, self.cpad0, _pad8(d0), split=True)
        self.blocks = []
        cin = d0
        for rb in (enc.encoder[0], enc.encoder[1]):
            cout = rb.conv1.out_channels
            sc = None if isinstance(rb.shortcut, nn.Identity) else \
                _linear_padded(rb.shortcut.weight, rb.shortcut.bias, _pad8(cin), _pad8(cout))
            self.blocks.append((_conv3x3_padded(rb.conv1, _pad8(cin), _pad8(cout)),
                                _conv3x3_padded(rb.conv2, _pad8(cout), _pad8(cout)), sc))
            cin = cout
        last = enc.encoder[2]
        self.out = _linear_padded(last.weight, last.bias, _pad8(cin), last.out_channels)
        self.nw, self.nb, self.eps = _f32(enc.norm_layer.weight), _f32(enc.norm_layer.bias), float(enc.norm_layer.eps)


class GlobalEncW:
    """Packed `global_rep_encoder` (App. A.2): MLP with GELU + LayerNorm, split-bf16 (~fp32) precision."""

    def __init__(self, enc):
        lins = [m for m in enc.encoder if isinstance(m, nn.Linear)]
        self.lins = []
        for i, m in enumerate(lins):
            w = m.weight.detach().float()
            if i == 0:  # K padded to 8 (inputs arrive as [V][8] rows)
                w = torch.cat([w, w.new_zeros(w.shape[0], 8 - w.shape[1])], dim=1)
            self.lins.append(Lin3(w, m.bias))
        self.nw, self.nb, self.eps = _f32(enc.norm_layer.weight), _f32(enc.norm_layer.bias), float(enc.norm_layer.eps)


class BlockW:
    def __init__(self, blk):
        self.n1w, self.n1b = _f32(blk.norm1.weight), _f32(blk.norm1.bias)
        self.n2w, self.n2b = _f32(blk.norm2.weight), _f32(blk.norm2.bias)
        self.qkv = Lin(blk.attn.qkv.weight, blk.attn.qkv.bias)
        self.proj = Lin(blk.attn.proj.weight, blk.attn.proj.bias)
        self.fc1 = Lin(blk.mlp.fc1.weight, blk.mlp.fc1.bias)
        self.fc2 = Lin(blk.mlp.fc2.weight, blk.mlp.fc2.bias)
        self.ls1 = _f32(blk.ls1.gamma) if hasattr(blk.ls1, "gamma") else None
        self.ls2 = _f32(blk.ls2.gamma) if hasattr(blk.ls2, "gamma") else None
        # row slices of the fused qkv weight (views, no copies): the view-sharded global blocks write Q and K|V to
        # different buffers (K|V goes straight into this rank's slot of the all-gather buffer)
        d = self.qkv.n // 3
        self.q_w, self.kv_w = self.qkv.w[:d], self.qkv.w[d:]
        self.q_b = self.qkv.b[:d] if self.qkv.b is not None else None
        self.kv_b = self.qkv.b[d:] if self.qkv.b is not None else None


class Engine:
    """Owns the packed weights of one MapAnything module on one CUDA device."""

    def __init__(self, model: nn.Module):
        self.device = next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("mapanything_b200 has no CPU path: move the module to a CUDA (sm_100a) device first")
        enc = model.encoder.model
        self.patch = enc.patch_size
        self.C = enc.embed_dim
        self.enc_heads = enc.num_heads
        self.kpad = (3 * self.patch * self.patch + 63) // 64 * 64
        self.patch_embed = Lin(enc.patch_embed.proj.weight, enc.patch_embed.proj.bias, kpad=self.kpad)
        self.cls = _f32(enc.cls_token.reshape(-1))
        self.pos_embed_param = enc.pos_embed.detach()
        self.interp_offset = enc.interpolate_offset
        self._pos_cache: Dict = {}
        self.enc_blocks = [BlockW(b) for b in enc.blocks]
        self.enc_nw, self.enc_nb = _f32(enc.norm.weight), _f32(enc.norm.bias)
        self.fus_w, self.fus_b = _f32(model.fusion_norm_layer.weight), _f32(model.fusion_norm_layer.bias)
        self.fus_eps = float(model.fusion_norm_layer.eps)

        self._model_ref = model  # geometric-input encoders are packed on first use (image-only scenes never need them)
        self._geo = None

        isx = model.info_sharing
        self.isx = isx   # wiring switches: is_global(i), view_pe_rows(V, first), softmax_scale_factor(n_keys)
        self._view_pe_table = None
        self.D, self.is_heads, self.indices = isx.dim, isx.num_heads, list(isx.indices)
        self.norm_intermediate = isx.norm_intermediate
        if isinstance(isx.proj_embed, nn.Linear):
            self.proj_embed = Lin(isx.proj_embed.weight, isx.proj_embed.bias)
        else:  # identity projection when dims match: expressed as an identity GEMM to keep one code path
            self.proj_embed = Lin(torch.eye(self.D, device=self.device), None)
        self.is_blocks = [BlockW(b) for b in isx.self_attention_blocks]
        self.is_nw, self.is_nb = _f32(isx.norm.weight), _f32(isx.norm.bias)
        self.use_ref_pe = isx.distinguish_ref_and_non_ref_views
        # sinusoid row 0 (position 0): sin(0)=0 on even channels, cos(0)=1 on odd channels
        pe0 = torch.zeros(1, self.D, device=self.device)
        pe0[0, 1::2] = 1.0
        self.pe0 = pe0
        # projected scale token is input independent: computed once with our own GEMM
        tok = _bf16(model.scale_token.reshape(1, -1))
        self.scale_tok_proj = torch.empty(1, self.D, device=self.device, dtype=torch.float32)
        ops.gemm(tok, self.proj_embed.w, self.scale_tok_proj, bias=self.proj_embed.b)

        # prediction heads (reference model.py:320-388): "dpt+pose" (released), "dpt" (no pose head), "linear"
        self.head_type = getattr(model, "pred_head_type", "dpt+pose")
        self.reg3_fused, self.linear_head = None, None
        if "dpt" in self.head_type:
            self._init_dpt(model)
            self.head_out_dim = self.reg3.n
        else:
            self._init_linear_head(model)
        self.raw_ld = 8 if self.head_out_dim <= 8 else (self.head_out_dim + 3) // 4 * 4
        self.scale_act = MA_ACT_GELU if getattr(model.scale_head, "activation", "relu") == "gelu" else MA_ACT_RELU
        if self.head_type == "dpt+pose":
            self._init_pose(model)
        self.scale_mlp = [Lin3(m.weight, m.bias) for m in model.scale_head.mlp if isinstance(m, nn.Linear)]
        import os

        # view groups of the encoder on separate CUDA streams: +1 % before programmatic dependent launch existed, equal with
        # it, and now slower than one stream (same-box A/B at 8 views: 327-328 views/s with two, 332 with one, 335 with one
        # and the persistent two-stream attention kernel, which wants all views in one launch)
        self.encoder_streams = max(1, int(os.environ.get("MA_ENCODER_STREAMS", "1")))
        self.sm_count = torch.cuda.get_device_properties(self.device).multi_processor_count
        # views per DPT pass (bounds the activation scratch: ~0.6 GB per view at 518 px).  8 instead of 4: same-box A/B at 8
        # views 311.1 vs 301.6 views/s (fewer, larger launches); MA_DPT_CHUNK overrides for A/B runs
        self.dpt_chunk_default = max(1, int(os.environ.get("MA_DPT_CHUNK", "8")))
        self.dpt_chunk = self.dpt_chunk_default
        self.proj_block_n = int(os.environ.get("MA_PROJ_BN", "0"))   # A/B knob: tile code of the attention-projection GEMMs
        # measurement aid (bench.py `strong` record): when a list, every sharded global block appends the CUDA events that
        # bracket its wait for the K/V all-gather on the compute stream
        self.ag_wait_events = None

    def _init_dpt(self, model):
        dpt = model.dpt_feature_head
        ap = dpt.act_postprocess
        self.feat = dpt.feature_dim
        self.ap0a, self.ap0b = _conv1x1(ap[0][0]), _convT(ap[0][1])
        self.ap1a, self.ap1b = _conv1x1(ap[1][0]), _convT(ap[1][1])
        self.ap2a = _conv1x1(ap[2][0])
        self.ap3a, self.ap3b = _conv1x1(ap[3][0]), _conv3x3(ap[3][1])
        self.ap0_s, self.ap1_s = ap[0][1].stride[0], ap[1][1].stride[0]
        self.layer_rn = [_conv3x3(c) for c in dpt.scratch.layer_rn]
        self.refine = []
        for name in ("refinenet1", "refinenet2", "refinenet3", "refinenet4"):
            r = getattr(dpt.scratch, name)
            self.refine.append({
                "r1c1": _conv3x3(r.resConfUnit1.conv1), "r1c2": _conv3x3(r.resConfUnit1.conv2),
                "r2c1": _conv3x3(r.resConfUnit2.conv1), "r2c2": _conv3x3(r.resConfUnit2.conv2),
                "out": _conv1x1(r.out_conv),
            })
        reg = model.dpt_regressor_head
        self.reg1, self.reg2, self.reg3 = _conv3x3(reg.conv1), _conv3x3(reg.conv2[0]), _conv1x1(reg.conv2[2])
        # the last 1x1 conv (hidden -> 6) as the epilogue of the 3x3 conv in front of it (ma_gemm_epilogue.head_*): fp32
        # weights [8][128] (the kernel form needs hidden = 128 and <= 8 outputs; MA_FUSED_HEAD=0 keeps the separate kernel)
        import os as _os2

        self.reg3_fused = None
        w3 = reg.conv2[2].weight.detach().reshape(reg.conv2[2].weight.shape[0], -1)
        if w3.shape[1] == 128 and w3.shape[0] <= 8 and self.reg2.n == 128 and _os2.environ.get("MA_FUSED_HEAD", "1") != "0":
            hw = torch.zeros(8, 128, device=self.device, dtype=torch.float32)
            hb = torch.zeros(8, device=self.device, dtype=torch.float32)
            hw[:w3.shape[0]] = w3.float()
            if reg.conv2[2].bias is not None:
                hb[:w3.shape[0]] = reg.conv2[2].bias.detach().float()
            self.reg3_fused = (hw.contiguous(), hb.contiguous())

    def _init_pose(self, model):
        ph = model.pose_head
        self.pose_relu_after_skip = bool(getattr(ph, "final_relu_after_skip", True))
        self.pose_blocks = []
        for rb in ph.res_conv:
            if not isinstance(rb.head_skip, nn.Identity):
                raise ValueError("pose head with a projecting skip is not part of the released config")
            # pose + scale heads run in split-bf16 (~fp32) precision: their outputs are normalised / exponentiated and
            # the reference computes them with autocast disabled (model.py:1599)
            cin = rb.res_conv2.weight.shape[1]
            self.pose_blocks.append((
                Lin3(rb.res_conv1.weight, rb.res_conv1.bias),
                Lin3(rb.res_conv2.weight.detach().permute(0, 2, 3, 1), rb.res_conv2.bias, group=cin),
                Lin3(rb.res_conv3.weight, rb.res_conv3.bias),
            ))
        # MA_POSE_HEAD=bf16 (default): the three convolutions of each ResConvBlock run with plain bf16 operands (fp32
        # accumulate, fp32 residual chain) -- they act on 1369 tokens per view whose average is what the MLPs see, so bf16
        # rounding averages out (measured: rotation / translation error vs the fp32 oracle unchanged, DESIGN.md section 4),
        # and the split-bf16 form cost 3x the MMA work (1.05 ms of a 26 ms step).  The pooled MLPs and the output layer,
        # whose results are normalised / exponentiated, stay in split-bf16 (~fp32).  MA_POSE_HEAD=split restores round 1.
        import os as _os

        self.pose_bf16 = _os.environ.get("MA_POSE_HEAD", "bf16") != "split"
        self.pose_blocks_bf16 = [(
            Lin(rb.res_conv1.weight, rb.res_conv1.bias), _conv3x3(rb.res_conv2), Lin(rb.res_conv3.weight, rb.res_conv3.bias),
        ) for rb in ph.res_conv]
        self.pose_mlp = [Lin3(ph.more_mlps[0].weight, ph.more_mlps[0].bias), Lin3(ph.more_mlps[2].weight, ph.more_mlps[2].bias)]
        self.pose_out = Lin3(torch.cat([ph.fc_t.weight, ph.fc_rot.weight], 0), torch.cat([ph.fc_t.bias, ph.fc_rot.bias], 0))

    def _init_linear_head(self, model):
        """pred_head_type "linear": the 1x1 conv as a split-bf16 (~fp32: the reference runs the heads with autocast disabled,
        model.py:1599) GEMM whose rows are reordered from F.pixel_shuffle's channel order (c, ky, kx) to (ky, kx, c), so that
        ma_pixel_shuffle_f32 scatters contiguous channel groups."""
        lf = model.dense_head
        p, od = lf.patch_size, lf.output_dim
        w = lf.proj.weight.detach().reshape(od, p * p, -1).permute(1, 0, 2).reshape(p * p * od, -1)
        b = lf.proj.bias.detach().reshape(od, p * p).t().reshape(-1) if lf.proj.bias is not None else None
        self.linear_head = Lin3(w, b)
        self.head_out_dim = od

    # ------------------------------------------------------------------------------------------ helpers
    def _empty(self, *shape, dtype=torch.bfloat16):
        return torch.empty(*shape, device=self.device, dtype=dtype)

    def _lin(self, x, lin: Lin, out=None, *, act=MA_ACT_NONE, out_dtype=torch.bfloat16, **kw):
        if out is None:
            out = self._empty(x.shape[0], lin.n, dtype=out_dtype)
        return ops.gemm(x, lin.w, out, bias=lin.b, act=act, **kw)

    def _conv3(self, x, lin: Lin, stride=1, *, act=MA_ACT_NONE, **kw):
        """x NHWC bf16 (n,H,W,C) -> (n,Ho,Wo,N): implicit GEMM (4-D TMA boxes, no im2col) for stride 1; the single
        stride-2 conv of the path (act_postprocess[3], 37 -> 19) goes through the explicit im2col."""
        n, H, W, C = x.shape
        if stride == 1:
            out = self._empty(n * H * W, lin.n)
            ops.conv3x3(x, lin.w, out, bias=lin.b, act=act, **kw)
            return out.view(n, H, W, lin.n)
        Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
        col = self._empty(n * Ho * Wo, 9 * C)
        ops.im2col3x3(x, col, stride)
        out = self._empty(n * Ho * Wo, lin.n)
        ops.gemm(col, lin.w, out, bias=lin.b, act=act, **kw)
        return out.view(n, Ho, Wo, lin.n)

    def _pos_embed(self, hp: int, wp: int, H: int, W: int) -> torch.Tensor:
        """pos_embed (1+hp*wp, C) fp32 for this resolution.  Interpolating the learned table for a non-native /
        non-square input (reference vision_transformer.py:208-242) is WEIGHT preparation: it is input independent,
        done once per resolution with torch's bicubic resampler and cached."""
        key = (hp, wp)
        if key in self._pos_cache:
            return self._pos_cache[key]
        pe = self.pos_embed_param.float()
        n0 = pe.shape[1] - 1
        if hp * wp == n0 and H == W:
            out = pe[0].contiguous()
        else:
            m = int(math.sqrt(n0))
            # the reference passes (w, h) = (x.shape[2], x.shape[3]) = (H, W): first grid axis follows image rows
            kw = {}
            if self.interp_offset:
                kw["scale_factor"] = (float(hp + self.interp_offset) / m, float(wp + self.interp_offset) / m)
            else:
                kw["size"] = (hp, wp)
            grid = torch.nn.functional.interpolate(pe[:, 1:].reshape(1, m, m, -1).permute(0, 3, 1, 2), mode="bicubic",
                                                   antialias=False, **kw)
            assert grid.shape[-2:] == (hp, wp)
            out = torch.cat([pe[0, :1], grid.permute(0, 2, 3, 1).reshape(hp * wp, -1)], 0).contiguous()
        self._pos_cache[key] = out
        return out

    def _pick_tail_split(self, q_len: int, kv_len: int, heads: int):
        """(first split slot, parts) for a long single-sequence attention, or None.  The (query block x head) CTAs have
        equal cost and fill the SMs in whole waves (8 views: 516 CTAs on 148 SMs = 3 full waves + 72 CTAs on half the
        chip).  Only the slots of that last partial wave are cut into `parts` CTAs, each with a share of the key range and
        a partial softmax state; ma_attention_merge joins them (touching those rows only).  With the ping-pong two-tile
        kernel this takes the 8-view global attention from 6.34 to 5.67 + 0.15 (merge) ms per step (same-box A/B on a B200,
        320 -> 332 views/s)."""
        sms = self.sm_count
        slots = -(-q_len // 256) * heads
        rem = slots % sms
        if slots <= sms or rem == 0 or rem > 0.7 * sms:
            return None
        parts = min(4, sms // rem, (-(-kv_len // 128)) // 8)
        return (slots - rem, parts) if parts >= 2 else None

    def _attention_one_sequence(self, q, k, v, out, heads: int, q_len: int, kv_len: int):
        """Global attention over one long sequence; the last partial wave of CTAs is split over the key range."""
        common = dict(num_heads=heads, num_seqs=1, q_len=q_len, kv_len=kv_len, q_seq_stride=q_len, kv_seq_stride=kv_len)
        pick = self._pick_tail_split(q_len, kv_len, heads)
        if pick is None:
            return ops.attention(q, k, v, out, **common)
        first, parts = pick
        so = self._empty(parts, q_len, heads * 64, dtype=torch.float32)
        sm = ops.fill_f32(self._empty(parts, q_len, heads, dtype=torch.float32), float("-inf"))
        ops.attention(q, k, v, out, state=(so, sm), kv_split=parts, kv_split_from=first, **common)
        return ops.attention_merge((so, sm), out, num_heads=heads, first_slot=first)

    def _block(self, x, bw: BlockW, rows: int, heads: int, num_seqs: int, seq_len: int, seq_stride: int,
               scale_factor: float = 1.0):
        """One pre-LN transformer block, in place on the fp32 residual stream x[:rows]."""
        dim = x.shape[1]
        scale = None if scale_factor == 1.0 else 64 ** -0.5 * scale_factor
        xr = x[:rows]
        h = self._empty(rows, dim)
        ops.layernorm(xr, h, bw.n1w, bw.n1b)
        qkv = self._lin(h, bw.qkv)
        a = self._empty(rows, dim)
        if num_seqs == 1 and seq_len >= 2048 and scale is None:
            self._attention_one_sequence(qkv[:, :dim], qkv[:, dim:2 * dim], qkv[:, 2 * dim:], a, heads, seq_len, seq_len)
        else:
            ops.attention(qkv[:, :dim], qkv[:, dim:2 * dim], qkv[:, 2 * dim:], a, num_heads=heads, num_seqs=num_seqs,
                          q_len=seq_len, kv_len=seq_len, q_seq_stride=seq_stride, kv_seq_stride=seq_stride, scale=scale)
        ops.gemm(a, bw.proj.w, xr, bias=bw.proj.b, colscale=bw.ls1, residual=xr, block_n=self.proj_block_n)
        ops.layernorm(xr, h, bw.n2w, bw.n2b)
        f = self._lin(h, bw.fc1, act=MA_ACT_GELU)
        ops.gemm(f, bw.fc2.w, xr, bias=bw.fc2.b, colscale=bw.ls2, residual=xr)

    def _block_global_sharded(self, x, bw: BlockW, plan, comm, bufs):
        """Global-attention block of the view-sharded stream (SURVEY 8e): local query rows, keys/values of every rank.
        K|V of the local rows are written by the GEMM epilogue into this rank's slot of the gather buffer; the NCCL
        all-gather of the slots runs while the attention over the local keys executes; a second launch resumes the
        online softmax over the remote slots."""
        dim, heads = x.shape[1], self.is_heads
        rows, slot = plan.rows(), plan.slot_rows
        kvbuf, state = bufs["kv"], bufs["state"]
        h = self._empty(rows, dim)
        ops.layernorm(x, h, bw.n1w, bw.n1b)
        mine = kvbuf[plan.rank * slot:plan.rank * slot + rows]
        ops.gemm(h, bw.kv_w, mine, bias=bw.kv_b)
        work = comm.all_gather_slots(kvbuf, slot)           # async: NCCL stream waits for the GEMM above
        q = self._empty(rows, dim)
        ops.gemm(h, bw.q_w, q, bias=bw.q_b)
        K, Vv = kvbuf[:, :dim], kvbuf[:, dim:]
        a = self._empty(rows, dim)
        remote = plan.remote_segments()
        sf = self.isx.softmax_scale_factor(plan.total_rows)
        common = dict(num_heads=heads, num_seqs=1, q_len=rows, kv_seq_stride=kvbuf.shape[0],
                      scale=None if sf == 1.0 else 64 ** -0.5 * sf)
        if remote:
            # partial softmax states: the local key range (runs while the all-gather is in flight) and the remote ranges
            # (after it landed), each cut into as many parts as fills the SMs; one merge pass joins them all
            kv_r = sum(l for _, l in remote)
            p_l, p_r = self._pick_tail_split(rows, rows, heads), self._pick_tail_split(rows, kv_r, heads)
            n_slots = -(-rows // 256) * heads
            f_l, s_l = p_l if p_l else (n_slots, 1)
            f_r, s_r = p_r if p_r else (n_slots, 1)
            so, sm = state
            if so.shape[0] < s_l + s_r:
                so = self._empty(s_l + s_r, rows, dim, dtype=torch.float32)
                sm = self._empty(s_l + s_r, rows, heads, dtype=torch.float32)
                bufs["state"] = (so, sm)
            ops.fill_f32(sm, float("-inf"))                  # unused partial slots are skipped by the merge
            ops.attention(q, K, Vv, None, kv_len=rows, kv_segments=plan.local_segment(), state=(so[:s_l], sm[:s_l]),
                          state_out=True, kv_split=s_l, kv_split_from=f_l, **common)
            if self.ag_wait_events is not None:
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record()
            work.wait()                                      # current stream waits for the gathered slots
            if self.ag_wait_events is not None:
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record()
                self.ag_wait_events.append((e0, e1))
            ops.attention(q, K, Vv, None, kv_len=kv_r, kv_segments=remote, state=(so[s_l:s_l + s_r], sm[s_l:s_l + s_r]),
                          state_out=True, kv_split=s_r, kv_split_from=f_r, **common)
            ops.attention_merge((so[:s_l + s_r], sm[:s_l + s_r]), a, num_heads=heads, scale=common["scale"])
        else:
            work.wait()
            ops.attention(q, K, Vv, a, kv_len=rows, kv_segments=plan.local_segment(), **common)
        ops.gemm(a, bw.proj.w, x, bias=bw.proj.b, colscale=bw.ls1, residual=x)
        ops.layernorm(x, h, bw.n2w, bw.n2b)
        f = self._lin(h, bw.fc1, act=MA_ACT_GELU)
        ops.gemm(f, bw.fc2.w, x, bias=bw.fc2.b, colscale=bw.ls2, residual=x)

    # ------------------------------------------------------------------------------------------ stage 1
    def encode(self, imgs: torch.Tensor) -> torch.Tensor:
        """(n,3,H,W) fp32 normalised images -> DINOv2 x_norm_patchtokens, fp32 [n*N][C] token-major."""
        n, _, H, W = imgs.shape
        p = self.patch
        hp, wp = H // p, W // p
        N = hp * wp
        pos = self._pos_embed(hp, wp, H, W)
        pos0 = pos[0].contiguous()
        imgs = imgs.contiguous()
        feat = self._empty(n * N, self.C, dtype=torch.float32)
        # The encoder is independent per view: run it as `groups` batches of views on separate CUDA streams, issued
        # block by block in turn.  Every kernel here is a persistent grid over all SMs whose last wave leaves SMs idle
        # (2.3 - 5.2 waves per launch at 8 views); the other group's next kernel fills that tail.
        groups = self.encoder_streams if n >= 2 * self.encoder_streams else 1
        main = torch.cuda.current_stream()
        bounds = [(g * n) // groups for g in range(groups + 1)]
        streams = [main] if groups == 1 else self._side_streams(groups)
        xs = []
        for g in range(groups):
            lo, ng = bounds[g], bounds[g + 1] - bounds[g]
            if groups > 1:
                streams[g].wait_stream(main)
            with torch.cuda.stream(streams[g]):
                a = self._empty(ng * N, self.kpad)
                ops.patchify(imgs[lo:lo + ng], a, p)
                x = self._empty(ng * (N + 1), self.C, dtype=torch.float32)
                ops.gemm(a, self.patch_embed.w, x, bias=self.patch_embed.b, residual=pos[1:], residual_row_mod=N,
                         rows_per_group_in=N, rows_per_group_out=N + 1, row_offset_out=1)
                ops.set_rows(x, self.cls, pos0, groups=ng, group_stride=N + 1, row_offset=0)
            xs.append(x)
        for bw in self.enc_blocks:
            for g in range(groups):
                ng = bounds[g + 1] - bounds[g]
                with torch.cuda.stream(streams[g]):
                    self._block(xs[g], bw, ng * (N + 1), self.enc_heads, ng, N + 1, N + 1)
        for g in range(groups):
            lo, ng = bounds[g], bounds[g + 1] - bounds[g]
            with torch.cuda.stream(streams[g]):
                ops.layernorm(xs[g], feat[lo * N:(lo + ng) * N], self.enc_nw, self.enc_nb, rows=ng * N, rows_per_group=N,
                              in_group_stride=N + 1, in_row_offset=1, out_group_stride=N, out_row_offset=0)
            if groups > 1:
                main.wait_stream(streams[g])
        return feat

    def _lin3(self, x32: torch.Tensor, lin: "Lin3", out: torch.Tensor, act: int = MA_ACT_NONE) -> torch.Tensor:
        """fp32-accurate Linear: the few-row fp32 kernel for up to 16 rows (pooled pose / scale MLPs, per-view global
        encoders), else the split-bf16 tensor-core GEMM."""
        rows, k = x32.shape
        if lin.w32 is not None and rows <= ops.LINEAR_ROWS_MAX and rows * k * 4 <= 48 * 1024 and k % 4 == 0:
            return ops.linear_rows_f32(x32, lin.w32, lin.b, out, act)
        return ops.gemm(ops.split3(x32), lin.w, out, bias=lin.b, act=act)

    def _side_streams(self, k: int):
        if len(getattr(self, "_streams", [])) < k:
            self._streams = [torch.cuda.Stream(device=self.device) for _ in range(k)]
        return self._streams[:k]

    # ------------------------------------------------------------------------------------------ stage 2
    def fuse_norm(self, feat: torch.Tensor) -> torch.Tensor:
        """fusion LayerNorm over channels (model.py:1245-1254): fp32 [n*N][C] -> bf16 (DPT tap 0 and proj_embed input)."""
        out = self._empty(*feat.shape)
        ops.layernorm(feat, out, self.fus_w, self.fus_b, eps=self.fus_eps)
        return out

    # ------------------------------------------------------------------------------------------ geometric inputs
    def _geo_weights(self):
        if self._geo is None:
            m = self._model_ref
            self._geo = {
                "ray": DenseEncW(m.ray_dirs_encoder), "depth": DenseEncW(m.depth_encoder),
                "depth_scale": GlobalEncW(m.depth_scale_encoder), "rot": GlobalEncW(m.cam_rot_encoder),
                "trans": GlobalEncW(m.cam_trans_encoder), "trans_scale": GlobalEncW(m.cam_trans_scale_encoder),
            }
        return self._geo

    def _dense_rep(self, w: DenseEncW, data: torch.Tensor, factor: Optional[torch.Tensor] = None) -> torch.Tensor:
        """fp32 NHWC (k,H,W,cin) -> fp32 [k*N][C] dense geometric features (reference model.py:812-814, :972-975)."""
        x = ops.unshuffle_split(data.contiguous(), w.patch, w.cpad0, factor)   # bf16 (k,hp,wp,3*cpad0)
        k, hp, wp, _ = x.shape
        M = k * hp * wp
        a = self._empty(M, w.conv_in.n)
        ops.conv3x3(x, w.conv_in.w, a, bias=w.conv_in.b)
        for c1, c2, sc in w.blocks:
            t = self._empty(M, c1.n)
            ops.conv3x3(a.view(k, hp, wp, -1), c1.w, t, bias=c1.b, act=MA_ACT_GELU)
            if sc is None:
                res = a
            else:
                res = self._empty(M, sc.n, dtype=torch.float32)
                ops.gemm(a, sc.w, res, bias=sc.b)
            o = self._empty(M, c2.n)
            ops.conv3x3(t.view(k, hp, wp, -1), c2.w, o, bias=c2.b, residual=res, act=MA_ACT_GELU, act_after_residual=True)
            a = o
        y = self._empty(M, w.out.n, dtype=torch.float32)
        ops.gemm(a, w.out.w, y, bias=w.out.b)
        f = self._empty(M, w.out.n, dtype=torch.float32)
        ops.layernorm(y, f, w.nw, w.nb, eps=w.eps)
        return f

    def _global_rep(self, w: GlobalEncW, x8: torch.Tensor) -> torch.Tensor:
        """fp32 [rows][8] (K-padded input) -> fp32 [rows][C] global geometric features (model.py:986-987, :1050-1110)."""
        g = x8
        for i, lin in enumerate(w.lins):
            o = self._empty(g.shape[0], lin.n, dtype=torch.float32)
            self._lin3(g, lin, o, MA_ACT_GELU if i + 1 < len(w.lins) else MA_ACT_NONE)
            g = o
        f = self._empty(g.shape[0], g.shape[1], dtype=torch.float32)
        ops.layernorm(g, f, w.nw, w.nb, eps=w.eps)
        return f

    def fuse_geometric(self, feat: torch.Tensor, V: int, N: int, ray=None, depth=None, pose=None):
        """Adds the encoded geometric inputs to the fp32 encoder features feat [V*N][C], in place
        (reference _encode_and_fuse_optional_geometric_inputs, model.py:1133-1244; the fusion LayerNorm follows).
          ray   = (view ids, fp32 (k,H,W,3) unit ray directions)
          depth = (view ids, fp32 (k,H,W,1) depth along ray, metric gates [k] of 0/1)
          pose  = (quats8, trans8, log_scale8 fp32 [V,8] from ops.pose_inputs, cam gates [V], metric gates [V])"""
        gw_ = self._geo_weights()
        dev = self.device

        def slots(ids):
            t = [-1] * V
            for j, i in enumerate(ids):
                t[i] = j
            return torch.tensor(t, dtype=torch.int32, device=dev)

        dense_a = a_slot = dense_b = b_slot = None
        g = [None, None, None, None]
        gates = [[0.0] * V for _ in range(4)]
        if ray is not None and len(ray[0]):
            dense_a, a_slot = self._dense_rep(gw_["ray"], ray[1]), slots(ray[0])
        if depth is not None and len(depth[0]):
            ids, d, metric = depth
            factor, logf8 = ops.depth_factor(d.contiguous())
            dense_b, b_slot = self._dense_rep(gw_["depth"], d, factor), slots(ids)
            g[3] = self._global_rep(gw_["depth_scale"], logf8)
            for j, i in enumerate(ids):
                gates[3][i] = float(metric[j])
        if pose is not None and any(pose[3]):
            q8, t8, s8, cam, metric = pose
            g[0] = self._global_rep(gw_["rot"], q8)
            g[1] = self._global_rep(gw_["trans"], t8)
            g[2] = self._global_rep(gw_["trans_scale"], s8)
            for i in range(V):
                gates[0][i] = gates[1][i] = float(cam[i])
                gates[2][i] = float(cam[i]) * float(metric[i])
        if dense_a is None and dense_b is None and all(x is None for x in g):
            return feat
        gw = torch.tensor(gates, dtype=torch.float32, device=dev)
        # the kernel walks g_0..g_3 positionally; absent ones are NULL
        return ops.fuse_add(feat, V, N, dense_a, a_slot, dense_b, b_slot, g, gw)

    def info_sharing(self, fused: torch.Tensor, V: int, N: int, plan=None, comm=None):
        """fused bf16 [V*N][C] -> taps (bf16 [V*N][D]) after blocks `indices`, final (bf16 [V*N][D]), and the fp32 final
        features [T][D] (row V*N = scale-token feature when this rank holds the scale token).

        With a ViewShardPlan, V is the number of LOCAL views, rank 0 holds the reference view and the scale token, and the
        global blocks attend over the keys of all ranks (_block_global_sharded)."""
        sharded = plan is not None and plan.world > 1
        has_tok = (not sharded) or plan.rank == 0
        has_ref = has_tok
        D, T = self.D, V * N + (1 if has_tok else 0)
        y = self._empty(T, D, dtype=torch.float32)
        pe_rows = self.isx.view_pe_rows(V, plan.view_offset if sharded else 0)
        ref_only = pe_rows is not None and pe_rows[0] == 0 and all(r is None for r in pe_rows[1:])
        if ref_only:   # released config: sinusoid row 0 on the reference view's tokens, folded into the GEMM epilogue
            ops.gemm(fused[:N], self.proj_embed.w, y[:N], bias=self.proj_embed.b, residual=self.pe0, residual_row_mod=1)
            if V > 1:
                ops.gemm(fused[N:], self.proj_embed.w, y[N:V * N], bias=self.proj_embed.b)
        else:
            ops.gemm(fused, self.proj_embed.w, y[:V * N], bias=self.proj_embed.b)
            if pe_rows is not None and any(r is not None for r in pe_rows):
                # per-view rows of the fixed sinusoid table (view-index PE, *_w_view_pe.yaml / gat_ifr_*.yaml): one
                # broadcast-add launch over all views
                if self._view_pe_table is None:
                    self._view_pe_table = _sinusoid_table(self.isx.max_views, D).to(self.device)
                idx = torch.tensor([r if r is not None else 0 for r in pe_rows], device=self.device)
                gw = torch.zeros(4, V, device=self.device)
                gw[0] = torch.tensor([1.0 if r is not None else 0.0 for r in pe_rows], device=self.device)
                ops.fuse_add(y[:V * N], V, N, globals_=[self._view_pe_table[idx].contiguous(), None, None, None], gw=gw)
        if has_tok:
            ops.set_rows(y, self.scale_tok_proj.reshape(-1), None, groups=1, group_stride=0, row_offset=V * N)
        bufs = None
        if sharded:
            assert plan.rows() == T and plan.tokens_per_view == N
            key = (plan.world * plan.slot_rows, T)
            if getattr(self, "_shard_bufs_key", None) != key:
                # zero-initialised once: slot padding rows are never written, so masked keys stay finite
                self._shard_bufs = {
                    "kv": torch.zeros(plan.world * plan.slot_rows, 2 * D, device=self.device, dtype=torch.bfloat16),
                    "state": (self._empty(2, T, D, dtype=torch.float32), self._empty(2, T, self.is_heads, dtype=torch.float32)),
                }
                self._shard_bufs_key = key
            bufs = self._shard_bufs
        taps: List[torch.Tensor] = []
        for i, bw in enumerate(self.is_blocks):
            if self.isx.is_global(i) and sharded:
                self._block_global_sharded(y, bw, plan, comm, bufs)
            elif self.isx.is_global(i):  # global: every token of every view + scale token
                self._block(y, bw, T, self.is_heads, 1, T, T, scale_factor=self.isx.softmax_scale_factor(T))
            else:  # frame: per view, scale token bypasses the block
                self._block(y, bw, V * N, self.is_heads, V, N, N, scale_factor=self.isx.softmax_scale_factor(N))
            if i in self.indices:
                tap = self._empty(V * N, D)
                if self.norm_intermediate:
                    ops.layernorm(y, tap, self.is_nw, self.is_nb, rows=V * N)
                else:
                    raise NotImplementedError("norm_intermediate=False is not part of the released config")
                taps.append(tap)
        final = self._empty(V * N, D)
        ops.layernorm(y, final, self.is_nw, self.is_nb, rows=V * N)      # bf16: DPT tap 3
        final32 = self._empty(T, D, dtype=torch.float32)
        ops.layernorm(y, final32, self.is_nw, self.is_nb)                 # fp32: pose head input + scale-token feature
        return taps, final, final32

    # ------------------------------------------------------------------------------------------ stage 3
    def _rcu(self, x_relu, x_skip, r, c1: str, c2: str, *, want_relu: bool):
        """ResidualConvUnit: conv2(relu(conv1(relu(x)))) + skip; returns (out, relu(out) or None)."""
        t = self._conv3(x_relu, r[c1], act=MA_ACT_RELU)
        n, H, W, _ = t.shape
        out = self._empty(n * H * W, r[c2].n)
        out_relu = self._empty(n * H * W, r[c2].n) if want_relu else None
        ops.conv3x3(t, r[c2].w, out, bias=r[c2].b, residual=x_skip.reshape(n * H * W, -1), out_relu=out_relu)
        return out.view(n, H, W, -1), (out_relu.view(n, H, W, -1) if want_relu else None)

    def _fusion(self, r, x0, lay_in, rn: Lin, up_virtual, up_out):
        """FeatureFusionBlock on NHWC bf16. x0: previous path (or None for refinenet4); lay_in: act_postprocess output."""
        n, H, W, _ = lay_in.shape
        M = n * H * W
        lay_in = lay_in.contiguous()
        lay = self._empty(M, rn.n)
        lay_relu = self._empty(M, rn.n)
        if x0 is None:
            ops.conv3x3(lay_in, rn.w, lay, out_relu=lay_relu)  # l4 and relu(l4)
            y, y_relu = lay.view(n, H, W, -1), lay_relu.view(n, H, W, -1)
        else:
            # one launch: lay = x0 + layer_rn(x)  (skip for RCU1's output),  lay_relu = relu(layer_rn(x))  (RCU1 input)
            ops.conv3x3(lay_in, rn.w, lay, residual=x0.reshape(M, -1), out_relu=lay_relu, relu_out_before_residual=True)
            y, y_relu = self._rcu(lay_relu.view(n, H, W, -1), lay.view(n, H, W, -1), r, "r1c1", "r1c2", want_relu=True)
        z, _ = self._rcu(y_relu, y, r, "r2c1", "r2c2", want_relu=False)
        # out_conv (1x1) commutes with the bilinear upsample (both linear, interpolation weights sum to 1):
        # apply it at the low resolution (4x fewer FLOPs), then upsample.
        o = self._lin(z.reshape(M, -1), r["out"]).view(n, H, W, -1)
        up = self._empty(n, up_out[0], up_out[1], o.shape[3])
        ops.bilinear_ac(o, up, virtual_hw=up_virtual)
        return up

    def pose_head(self, x32: torch.Tensor, n: int, hp: int, wp: int, out: torch.Tensor, x16: Optional[torch.Tensor] = None):
        """x32 fp32 [n*N][D] (final info-sharing features; x16 = the same in bf16) -> out fp32 [n][7] = (t | q)."""
        N = hp * wp
        D = x32.shape[1]
        if self.pose_bf16 and self.pose_relu_after_skip and x16 is not None:
            xb = x16
            for c1, c2, c3 in self.pose_blocks_bf16:
                u = self._lin(xb, c1, act=MA_ACT_RELU)
                u2 = self._conv3(u.view(n, hp, wp, c1.n), c2, act=MA_ACT_RELU).reshape(n * N, c2.n)
                xn = self._empty(n * N, c3.n, dtype=torch.float32)
                xb = self._empty(n * N, c3.n)   # bf16 copy of relu(x + y) = the next block's GEMM operand, same launch
                ops.gemm(u2, c3.w, xn, bias=c3.b, residual=x32, act=MA_ACT_RELU, act_after_residual=True, out_relu=xb)
                x32 = xn
        else:
            x32 = self._pose_blocks_split(x32, n, hp, wp)
        pooled = self._empty(n, D, dtype=torch.float32)
        ops.token_mean_f32(x32.view(n, N, D), pooled)
        g = pooled
        for lin in self.pose_mlp:
            gn = self._empty(n, lin.n, dtype=torch.float32)
            self._lin3(g, lin, gn, MA_ACT_RELU)
            g = gn
        self._lin3(g, self.pose_out, out)
        return out

    def _pose_blocks_split(self, x32: torch.Tensor, n: int, hp: int, wp: int) -> torch.Tensor:
        """ResConvBlocks in split-bf16 (~fp32) precision."""
        N = hp * wp
        for c1, c2, c3 in self.pose_blocks:
            u = self._empty(n * N, c1.n, dtype=torch.float32)
            ops.gemm(ops.split3(x32), c1.w, u, bias=c1.b, act=MA_ACT_RELU)
            us = ops.split3(u).view(n, hp, wp, 3 * c1.n)
            u2 = self._empty(n * N, c2.n, dtype=torch.float32)
            ops.conv3x3(us, c2.w, u2, bias=c2.b, act=MA_ACT_RELU)
            xn = self._empty(n * N, c3.n, dtype=torch.float32)
            ops.gemm(ops.split3(u2), c3.w, xn, bias=c3.b, residual=x32, act=MA_ACT_RELU,
                     act_after_residual=self.pose_relu_after_skip)
            x32 = xn
        return x32

    def dpt_and_pose(self, taps4: List[torch.Tensor], V: int, hp: int, wp: int, H: int, W: int,
                     final32: Optional[torch.Tensor] = None):
        """taps4: 4 x bf16 [V*N][C_i] (+ final32 fp32 [V*N][D] for the pose / linear head; defaults to taps4[-1] upcast)
        -> raw dense fp32 [V*H*W][raw_ld] (head_out_dim used), pose_raw fp32 [V][7] (None without a pose head)."""
        if final32 is None:
            final32 = taps4[-1].float()
        N = hp * wp
        raw = self._empty(V * H * W, self.raw_ld, dtype=torch.float32)
        if self.head_type == "linear":
            # reference model.py:1310-1320: the dense head sees the final features only; rows = tokens, fp32-accurate GEMM
            od, ps = self.head_out_dim, self.patch
            for s in range(0, V, self.dpt_chunk):
                n = min(self.dpt_chunk, V - s)
                y = self._empty(n * N, self.linear_head.n, dtype=torch.float32)
                self._lin3(final32[s * N:(s + n) * N], self.linear_head, y)
                ops.pixel_shuffle_f32(y, raw[s * H * W:(s + n) * H * W], n, hp, wp, od, ps)
            return raw, None
        with_pose = self.head_type == "dpt+pose"
        pose_raw = self._empty(V, 7, dtype=torch.float32) if with_pose else None
        for s in range(0, V, self.dpt_chunk):
            n = min(self.dpt_chunk, V - s)
            t = [x[s * N:(s + n) * N] for x in taps4]
            r1, r2, r3, r4 = self.refine
            # act_postprocess
            a0 = self._lin(self._lin(t[0], self.ap0a), self.ap0b)
            s0 = self.ap0_s
            l0 = self._empty(n, hp * s0, wp * s0, self.ap0a.n)
            ops.pixel_shuffle(a0, l0, n, hp, wp, self.ap0a.n, s0)
            a1 = self._lin(self._lin(t[1], self.ap1a), self.ap1b)
            s1 = self.ap1_s
            l1 = self._empty(n, hp * s1, wp * s1, self.ap1a.n)
            ops.pixel_shuffle(a1, l1, n, hp, wp, self.ap1a.n, s1)
            l2 = self._lin(t[2], self.ap2a).view(n, hp, wp, -1)
            l3 = self._conv3(self._lin(t[3], self.ap3a).view(n, hp, wp, -1), self.ap3b, stride=2)
            h3, w3 = l3.shape[1], l3.shape[2]
            # refinenets, bottom-up.  refinenet4 output is upsampled x2 then cropped to layer 3's grid.
            p4 = self._fusion(r4, None, l3, self.layer_rn[3], (2 * h3, 2 * w3), (hp, wp))
            p3 = self._fusion(r3, p4, l2, self.layer_rn[2], (2 * hp, 2 * wp), (2 * hp, 2 * wp))
            p2 = self._fusion(r2, p3, l1, self.layer_rn[1], (4 * hp, 4 * wp), (4 * hp, 4 * wp))
            p1 = self._fusion(r1, p2, l0, self.layer_rn[0], (8 * hp, 8 * wp), (8 * hp, 8 * wp))
            # regressor: conv3x3 -> bilinear to the image size -> conv3x3 + ReLU -> conv1x1 (fp32 out)
            g1 = self._conv3(p1, self.reg1)
            g1u = self._empty(n, H, W, g1.shape[3])
            ops.bilinear_ac(g1, g1u)
            rawv = raw[s * H * W:(s + n) * H * W]
            if self.reg3_fused is not None and raw.shape[1] == 8:
                ops.conv3x3_head(g1u, self.reg2.w, self.reg2.b, MA_ACT_RELU, self.reg3_fused[0], self.reg3_fused[1], rawv)
                if with_pose:
                    self.pose_head(final32[s * N:(s + n) * N], n, hp, wp, pose_raw[s:s + n], x16=t[3])
                continue
            g2 = self._conv3(g1u, self.reg2, act=MA_ACT_RELU)
            g2f = g2.reshape(n * H * W, -1)
            if self.reg3.n <= 8 and self.reg3.k <= 256 and self.reg3.k % 8 == 0:
                ops.head_linear_small(g2f, self.reg3.w, self.reg3.b, rawv)   # 128 -> 6 per pixel: streaming kernel
            else:
                ops.gemm(g2f, self.reg3.w, rawv[:, :self.reg3.n], bias=self.reg3.b)
            # pose head on the final info-sharing features (split-bf16 precision)
            if with_pose:
                self.pose_head(final32[s * N:(s + n) * N], n, hp, wp, pose_raw[s:s + n], x16=t[3])
        return raw, pose_raw

    def scale_head(self, tok_feat32: torch.Tensor) -> torch.Tensor:
        """scale-token feature fp32 [1][D] -> log metric scale fp32 [1] (split-bf16 precision)."""
        x = tok_feat32
        for lin in self.scale_mlp[:-1]:
            xn = self._empty(x.shape[0], lin.n, dtype=torch.float32)
            self._lin3(x, lin, xn, self.scale_act)
            x = xn
        out = self._empty(1, self.scale_mlp[-1].n, dtype=torch.float32)
        self._lin3(x, self.scale_mlp[-1], out)
        return out.reshape(-1)[:1].contiguous()
