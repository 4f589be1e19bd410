/*
 * mapanything_b200 -- C ABI of the B200-native (sm_100a) kernels behind the MapAnything
 * feed-forward inference hot path.
 *
 * The reference (etola/map-anything) is pure Python over PyTorch library kernels; it has no FFI of
 * its own.  The boundary a maintainer binds is therefore the Python surface
 * `MapAnything.forward / MapAnything.infer` (reference mapanything/models/mapanything/model.py:1477,
 * :1964); each entry point below replaces the PyTorch op(s) that a stage of that path dispatches
 * and cites the reference call site it stands in for.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - all functions return MA_OK (0) or a negative ma_status; the message for the calling thread is
 *    available from ma_last_error();
 *  - no C++ exceptions, no torch types, no ownership transfer: the caller owns every buffer;
 *  - bf16 tensors are `__nv_bfloat16` (uint16 storage), row-major, innermost dimension contiguous.
 */
#ifndef MAPANYTHING_B200_H_
#define MAPANYTHING_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MA_ABI_VERSION 1

typedef enum ma_status {
  MA_OK = 0,
  MA_ERR_INVALID = -1, /* bad argument (shape / alignment / dtype) */
  MA_ERR_CUDA = -2     /* CUDA runtime / driver error */
} ma_status;

typedef enum ma_dtype { MA_BF16 = 0, MA_F32 = 1 } ma_dtype;
typedef enum ma_act { MA_ACT_NONE = 0, MA_ACT_GELU = 1, MA_ACT_RELU = 2 } ma_act;

/* ---- library ------------------------------------------------------------------------------ */
const char* ma_last_error(void);
int ma_abi_version(void);
int ma_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Programmatic dependent launch of the chained GEMM / attention / LayerNorm kernels (the next kernel's prologue overlaps
 * the previous kernel's last wave; results are identical).  enabled: 0 / 1, or -1 to query only.  Returns the previous
 * setting.  Initial value: environment variable MA_PDL, else the build default.  The reference has no counterpart (it
 * relies on the PyTorch stream order, model.py:1477-1909). */
int ma_set_pdl(int enabled);
/* Stream-K tail of the in-place fp32 residual GEMMs (ma_gemm_bf16 with residual == out, fp32, K >= 2048: fc2 of every
 * transformer block): the K blocks of the last, partially filled wave of tiles are split evenly over all CTA pairs and the
 * partial products are joined by the same bulk reduce-add that applies the residual.  Shorter critical path (172 tiles on 74
 * pairs: 149 instead of 192 K blocks per pair; -11 % for such a launch alone, +0.2 - 0.7 % on the 8-view step), but the fp32
 * sum of an element's partial products is formed in arrival order, so such a GEMM is reproducible to fp32 rounding, not bit
 * for bit.  enabled: 0 / 1, or -1 to query only.  Returns the previous setting.  Initial value: environment variable
 * MA_GEMM_STREAMK, else on. */
int ma_set_stream_k(int enabled);
/* Which kernel the last ma_gemm_bf16 / ma_conv3x3_bf16 call of THIS thread launched, as a block_n code (64 / 128 / 256 = the
 * one-CTA instantiation gemm_bf16_kernel<1, block_n>, 2128 / 2256 = the CTA-pair instantiation
 * gemm_bf16_kernel<2, block_n - 2000>); 0 before the first call.  Measurement aid (bench.py names the dominant kernel from it); no reference counterpart. */
int ma_last_gemm_block(void);
/* Which kernel the last ma_attention_fwd / ma_attention_fwd_ex call of THIS thread launched: 5 = attention_fwd_v5_kernel
 * (plain attention over many short sequences), 3 = attention_fwd_v3_kernel (up to 4096 keys, no kv split), 2 =
 * attention_fwd_v2_kernel (longer key ranges, kv split); 0 before the first launch.  Lets tests and tools see which kernel
 * a shape reaches; no reference counterpart. */
int ma_last_attention_kernel(void);
/* Which form of the horizontal resampling pass the last ma_resample_h_u8rgb call of THIS thread launched: 1 =
 * resample_h_kernel (byte loads, any window length), 1000 + KMAX = resample_h_vec_kernel<KMAX> (word loads, windows up to
 * KMAX taps), 2000 + NW4 = resample_h_dp4a_kernel<NW4> (dp4a on packed coefficients, windows up to 4 * NW4 taps); 0 before
 * the first launch.  Lets tests see which instantiation a call reaches; no reference counterpart. */
int ma_last_resample_kernel(void);

/* ---- GEMM: Y = epilogue(X . W^T) ------------------------------------------------------------
 * Replaces every nn.Linear / 1x1 conv / im2col'ed conv on the path (cuBLASLt / cuDNN calls in the
 * reference: DINOv2 qkv/proj/fc1/fc2 mapanything/models/external/dinov2/layers/attention.py:53-70,
 * mlp.py:16-40; patch embed patch_embed.py:65-87; the uniception info-sharing / DPT / pose-head
 * layers invoked at model.py:1532-1542, :1302-1338, :1449-1457).
 *
 * X: [M,K] bf16 (row stride ldx), W: [N,K] bf16 (row stride ldw), fp32 accumulate in TMEM
 * (tcgen05.mma), operands staged by TMA.  K and the strides must be multiples of 8 elements.
 * Epilogue, applied per element in this order:
 *    v = acc + bias[n];  v = act(v);  v *= colscale[n];  v += residual[res_row, n]
 *    out[out_row, n] = v;  out_relu[out_row, n] = max(v, 0)   (optional second output, bf16)
 * (`flags` can move the activation after the residual add, or take out_relu before it.)
 * Row mapping (token assembly without copy kernels): when rows_per_group_in > 0,
 *    out_row = (m / rows_per_group_in) * rows_per_group_out + row_offset_out + m % rows_per_group_in
 * else out_row = m.  res_row = m % residual_row_mod when residual_row_mod > 0, else out_row.
 * Alignment: when N >= 32 (a multiple of 32 or not), out, residual, out_relu, bias and colscale must be 16-byte aligned and
 * ldo / ldr / ldo_relu multiples of 16 bytes (full 32-column chunks are loaded and stored as 16-byte vectors); otherwise
 * the call returns MA_ERR_INVALID.  With N < 32 they need only their element alignment. */
typedef struct ma_gemm_epilogue {
  void* out;
  int64_t ldo;
  int32_t out_dtype; /* ma_dtype */
  int32_t act;       /* ma_act */
  const float* bias;     /* [N] or NULL */
  const float* colscale; /* [N] or NULL (LayerScale gamma) */
  const void* residual;  /* or NULL */
  int64_t ldr;
  int32_t residual_dtype; /* ma_dtype */
  int32_t residual_row_mod;
  void* out_relu; /* bf16 or NULL */
  int64_t ldo_relu;
  int32_t rows_per_group_in;
  int32_t rows_per_group_out;
  int32_t row_offset_out;
  int32_t flags; /* MA_GEMM_* bits */
  /* Fused narrow head (optional; CTA-pair kernel, N = 128 only -- pass block_n = 2128): when head_out != NULL the tile
   * values y (after bias / activation) are NOT stored; instead head_out[row][j] = head_bias[j] + sum_n head_w[j][n] * y[n]
   * for j < 8 is written (fp32, row stride 8).  head_w: fp32 [8][N] (rows >= head_n zero), head_bias: fp32 [8].
   * Replaces the last 1x1 convolution of the DPT regressor (128 -> 6 channels on every pixel; reference
   * DPTRegressionProcessor.conv2[2], model.py:1326-1338) as the epilogue of the 3x3 convolution in front of it: the
   * 128-channel full-resolution map (69 MB per view in bf16) is never written or re-read. */
  const float* head_w;
  const float* head_bias;
  float* head_out;
} ma_gemm_epilogue;

/* act is applied after the residual add instead of before the column scale (ResConvBlock: relu(skip + y)). */
#define MA_GEMM_ACT_AFTER_RESIDUAL 1
/* out_relu receives relu(value BEFORE colscale/residual) instead of relu(final value) (DPT: the conv input
 * relu(x1) and the fused skip x0 + x1 come out of one launch). */
#define MA_GEMM_RELU_OUT_BEFORE_RESIDUAL 2

/* block_n: 0 = choose automatically (wave count x measured per-tile cost); 64 / 128 / 256 = one CTA per 128 x block_n
 * tile; 2128 / 2256 = a CTA pair (tcgen05 cta_group::2, cluster of 2) per 256 x 128 / 256 x 256 tile. */
int ma_gemm_bf16(const void* x, int64_t ldx, const void* w, int64_t ldw, int M, int N, int K,
                 const ma_gemm_epilogue* epi, int block_n, void* stream);

/* 3x3 / stride 1 / pad 1 convolution over NHWC bf16 (n,H,W,C) as an IMPLICIT GEMM on the same kernel: the A operand of
 * each (pixel tile, tap) is one 4-D TMA box of the input shifted by the tap, the zero padding is TMA out-of-bounds fill;
 * no im2col matrix exists.  w: [Cout][9*C] bf16, k = (ky*3+kx)*C + c (row stride ldw).  Output rows are pixel indices
 * (i*H + y)*W + x; the epilogue is the one of ma_gemm_bf16 (row remapping unsupported).  Replaces the cuDNN 3x3 convs of
 * the DPT feature head / regressor / pose head (reference model.py:1302-1338, :1449-1457; SURVEY App. A.4, A.6) and of
 * the dense geometric-input encoders (model.py:753-1010; App. A.2). */
int ma_conv3x3_bf16(const void* x, int n, int H, int W, int C, const void* w, int64_t ldw, int Cout,
                    const ma_gemm_epilogue* epi, int block_n, void* stream);

/* ---- Attention forward (head_dim 64, non-causal) ---------------------------------------------
 * Replaces the attention of the DINOv2 blocks (reference dinov2/layers/attention.py:53-90,
 * F.scaled_dot_product_attention / xformers there) and of the info-sharing frame / global blocks
 * (uniception, invoked at model.py:1532-1542; analog vggt/layers/attention.py:46-76).
 *
 * q/k/v are token-major bf16 matrices (typically three column slices of one fused-qkv GEMM output):
 * head h of q occupies columns [q_col0 + 64 h, q_col0 + 64 h + 64).  Sequence s uses query rows
 * [s*q_seq_stride, s*q_seq_stride + q_len) and key/value rows [s*kv_seq_stride, ... + kv_len).
 * out[row, o_col0 + 64 h ...] = softmax(q k^T * softmax_scale) v, bf16.  QK^T and PV run on tcgen05
 * with accumulators in TMEM; softmax statistics and the output accumulator are fp32. */
int ma_attention_fwd(const void* q, int64_t ldq, int64_t q_rows, int q_col0, const void* k, int64_t ldk,
                     int64_t kv_rows, int k_col0, const void* v, int64_t ldv, int v_col0, void* out, int64_t ldo,
                     int o_col0, int num_seqs, int num_heads, int q_len, int kv_len, int64_t q_seq_stride,
                     int64_t kv_seq_stride, float softmax_scale, void* stream);

/* Extended form for the view-sharded global attention (SURVEY 8e; the reference runs it as one SDPA call over all
 * views, uniception info-sharing invoked at model.py:1532-1542):
 *  - the keys/values of a sequence may be n_segments row ranges [seg_row0[i], seg_row0[i] + seg_len[i]) (relative to the
 *    sequence's first kv row, sum of seg_len == kv_len): one range per source rank of the all-gathered K/V buffer;
 *  - MA_ATTN_STATE_OUT: instead of `out`, write the online-softmax state after the last key: state_o = normalised
 *    output (fp32 [q_rows][ld_state_o], head h at column 64 h) and state_m [q_rows][num_heads] = running maximum
 *    (raw score units) + log2(running sum) / (softmax_scale * log2 e);
 *  - MA_ATTN_STATE_IN: resume from such a state (local keys first, remote keys when the all-gather has landed).
 * ext == NULL is ma_attention_fwd. */
#define MA_ATTN_MAX_SEGMENTS 16
#define MA_ATTN_STATE_IN 1
#define MA_ATTN_STATE_OUT 2
typedef struct ma_attn_ext {
  int32_t n_segments; /* 0 = single range [0, kv_len) */
  int32_t flags;      /* MA_ATTN_STATE_* */
  int32_t seg_row0[MA_ATTN_MAX_SEGMENTS];
  int32_t seg_len[MA_ATTN_MAX_SEGMENTS];
  float* state_o;
  int64_t ld_state_o;
  float* state_m;
  /* kv_split > 1: (query block, head) slots with index >= kv_split_from (slot order: full 256-row blocks of all heads
   * first, ragged last blocks after them) are cut into kv_split CTAs, each taking a share of the key range; part i
   * writes its state at state_o + i * split_stride_o, state_m + i * split_stride_m (state buffers required; state_m
   * pre-filled with -inf).  Slots below kv_split_from run as one CTA and write `out` (or part 0 with STATE_OUT).
   * Join with ma_attention_merge.  kv_split 0 / 1 = off. */
  int32_t kv_split;
  int32_t kv_split_from;
  int64_t split_stride_o;
  int64_t split_stride_m;
} ma_attn_ext;

/* Joins n_partials partial softmax states (kv_split parts and / or local + remote key ranges of the sharded global
 * attention) into the bf16 attention output: out = sum_p w_p o_p / sum_p w_p, w_p = exp((m'_p - max m') * softmax_scale).
 * first_slot >= 0 (single sequence): only the rows of the (query block, head) slots >= first_slot are visited (tail-only
 * splitting); -1 = every (row, head).  state_m must be pre-filled with -inf (unused partials are skipped). */
int ma_attention_merge(const float* state_o, int64_t ld_state_o, int64_t split_stride_o, const float* state_m,
                       int64_t split_stride_m, int n_partials, int64_t rows, int num_heads, float softmax_scale, void* out,
                       int64_t ldo, int first_slot, void* stream);
int ma_attention_fwd_ex(const void* q, int64_t ldq, int64_t q_rows, int q_col0, const void* k, int64_t ldk,
                        int64_t kv_rows, int k_col0, const void* v, int64_t ldv, int v_col0, void* out, int64_t ldo,
                        int o_col0, int num_seqs, int num_heads, int q_len, int kv_len, int64_t q_seq_stride,
                        int64_t kv_seq_stride, float softmax_scale, const ma_attn_ext* ext, void* stream);

/* ---- HBM-bound stage kernels ------------------------------------------------------------------ */

/* DINOv2 PatchEmbed im2col (reference dinov2/layers/patch_embed.py:65-87, Conv2d k=s=patch): fp32 NCHW image
 * (n,3,H,W) -> bf16 [n*(H/p)*(W/p)][kpad], k = c*p*p + ky*p + kx, zero padded to kpad (multiple of 8). */
int ma_patchify(const float* img, void* out, int n, int H, int W, int patch, int kpad, void* stream);

/* nn.LayerNorm over the last dim (reference: every norm1/norm2/norm of dinov2/layers/block.py:93-119, the
 * fusion_norm_layer model.py:1245-1254, the info-sharing norms).  in/out dtype are ma_dtype; the optional row
 * remap row(r) = (r / rows_per_group) * group_stride + row_offset + r % rows_per_group (separately for in and
 * out; rows_per_group = 0 -> identity) drops the cls token / skips the scale token without a copy.  C and the row
 * strides are multiples of 4 with ld_in, ld_out >= C; in and out are 16-byte aligned when fp32 and 8-byte aligned when bf16,
 * gamma and beta 16-byte aligned. */
int ma_layernorm(const void* in, int in_dtype, int64_t ld_in, void* out, int out_dtype, int64_t ld_out,
                 const float* gamma, const float* beta, int rows, int C, float eps, int rows_per_group,
                 int64_t in_group_stride, int64_t in_row_offset, int64_t out_group_stride, int64_t out_row_offset,
                 void* stream);

/* dst[0:n] = value, fp32 (initial -inf maxima of the partial softmax states joined by ma_attention_merge; keeps the step free
 * of library kernels).  No reference counterpart. */
int ma_fill_f32(float* dst, int64_t n, float value, void* stream);

/* dst[g*group_stride + row_offset][0:C] = a[0:C] + b[0:C] (b may be NULL) for g in [0, groups): cls token +
 * pos_embed[0] (reference vision_transformer.py:252-253), scale token row (model.py:1524-1535). fp32, ld >= C. */
int ma_set_rows(float* dst, int64_t ld, int groups, int64_t group_stride, int64_t row_offset, const float* a,
                const float* b, int C, void* stream);

/* im2col of a 3x3 / pad 1 / stride {1,2} convolution over NHWC bf16 (n,H,W,C): out[(i,yo,xo)][(ky*3+kx)*C + c].
 * With ma_gemm_bf16 this replaces the cuDNN convs of the DPT / pose heads (reference model.py:1302-1338).  C % 8 == 0;
 * in and out 16-byte aligned. */
int ma_im2col3x3(const void* in, void* out, int n, int H, int W, int C, int stride, void* stream);

/* ConvTranspose2d with kernel == stride == s as GEMM + this permutation: in[(i,y,x)][(ky*s+kx)*C + c] ->
 * NHWC out[(i, y*s+ky, x*s+kx)][c]  (DPT act_postprocess, SURVEY App. A.4). bf16, C % 8 == 0, in and out 16-byte aligned. */
int ma_pixel_shuffle(const void* in, void* out, int n, int h, int w, int C, int s, void* stream);

/* The same permutation in fp32 with row strides: the `linear` prediction head (reference model.py:339-343, a 1x1 conv
 * to output_dim * patch^2 channels + F.pixel_shuffle) as GEMM (weight rows reordered to [(ky,kx), c]) + this scatter
 * into the per-pixel rows [(i, y*s+ky, x*s+kx)][0:C] (row stride ld_out) that ma_decode_scene reads. */
int ma_pixel_shuffle_f32(const float* in, int64_t ld_in, float* out, int64_t ld_out, int n, int h, int w, int C, int s,
                         void* stream);

/* F.interpolate(mode="bilinear", align_corners=True) over NHWC bf16.  (Hv,Wv) is the full output size that
 * defines the scale; only the top-left (Ho,Wo) window is written (refinenet4 crop 38 -> 37).  C % 8 == 0; in and out
 * 16-byte aligned. */
int ma_bilinear_align_corners(const void* in, void* out, int n, int Hin, int Win, int C, int Hv, int Wv, int Ho, int Wo,
                              void* stream);

/* AdaptiveAvgPool2d(1) over tokens: bf16 [n][T][C] -> bf16 [n][C] (pose head, SURVEY App. A.6). */
int ma_token_mean(const void* in, void* out, int n, int T, int C, void* stream);

/* fp32 [rows][C] -> bf16 [rows][3C] = [hi | lo | hi] (hi = bf16(x), lo = bf16(x - hi)).  With weights packed
 * [w_hi | w_hi | w_lo] one ma_gemm_bf16 over K' = 3K evaluates the product to ~2^-16 relative accuracy: used for
 * the pose / scale heads, which the reference runs with autocast disabled (model.py:1599).  C and ld_in are multiples of 4
 * with ld_in >= C; in is 16-byte aligned, out 8-byte aligned. */
int ma_split_bf16x3(const float* in, int64_t ld_in, void* out, int rows, int C, void* stream);

/* Narrow linear head out[row][0:N] = W[N][K] . x[row] + b (N <= 8, K <= 256, bf16 in, fp32 out): the final 1x1 conv of
 * the DPT regressor (128 -> 6 channels per pixel, SURVEY App. A.4; reference model.py:1326-1332) as a streaming kernel.
 * K % 8 == 0, ldx % 8 == 0, ldx >= K, ldw >= K, ldo >= N; x 16-byte aligned. */
int ma_head_linear_small(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias, float* out, int64_t ldo,
                         int64_t rows, int N, int K, void* stream);

/* fp32 Linear on a handful of rows: out[r][0:N] = act(b + W[N][K] . x[r]), 1 <= rows <= 16, K % 4 == 0, rows * K * 4 <= 48 KB,
 * plain fp32 arithmetic (act: MA_ACT_NONE / MA_ACT_RELU / MA_ACT_GELU, exact erf).  The pooled MLPs of the pose head and the
 * scale head (uniception PoseHead.more_mlps / fc_t / fc_rot and MLPHead on the scale token, invoked at reference
 * model.py:1449-1469 with autocast disabled): 8 x 768 and 1 x 768 inputs.  ldx, ldw multiples of 4 and >= K, ldo >= N; x and w
 * 16-byte aligned. */
int ma_linear_rows_f32(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* bias, int act, float* out,
                       int64_t ldo, int rows, int N, int K, void* stream);

/* fp32 variant of ma_token_mean. */
int ma_token_mean_f32(const float* in, float* out, int n, int T, int C, void* stream);

/* Fused dense adaptor + pose/scale adaptors + factored-geometry decode + output packaging (reference
 * model.py:1683-1741, :1874-1907; geometry.py:855-907): raw [n*HW][ld_raw] fp32 = (ray xyz, depth logit,
 * confidence logit, mask logit); pose_raw [n][7] = (t, q xyzw); scale_raw [1] (log metric scale).
 * Writes pts3d, pts3d_cam, rays [n*HW][3]; depth, conf, logits [n*HW]; mask [n*HW] (1 byte bool);
 * cam_trans [n][3] (scaled), cam_quats [n][4] (unit), scale_out [1].  ld_raw >= 6; when ld_raw % 4 == 0 each row is read
 * as a float4 and a float2, so raw must then be 16-byte aligned. */
int ma_decode_dense(const float* raw, int ld_raw, const float* pose_raw, const float* scale_raw, int n, int HW,
                    float* pts3d, float* pts3d_cam, float* rays, float* depth, float* conf, float* logits, uint8_t* mask,
                    float* cam_trans, float* cam_quats, float* scale_out, void* stream);

/* The same decode for every scene representation the reference model can be configured with (model.py:407-587 adaptor
 * table, :1618-1907 decode branches).  Head-output channel order: [representation | confidence logit | mask logit].
 *   MA_REP_POINTMAP                    xyz                       -> pts3d
 *   MA_REP_RAYMAP_DEPTH                origin xyz, ray xyz, depth -> pts3d = o + r d, ray_origins, rays, depth
 *   MA_REP_RAYDIRS_DEPTH_POSE          ray xyz, depth   (+ pose)  -> what ma_decode_dense writes (the released model)
 *   MA_REP_CAMPOINTMAP_POSE            xyz camera frame (+ pose)  -> depth = |p|, rays = p / depth, pts3d = R (rays depth) + t
 *   MA_REP_POINTMAP_RAYDIRS_DEPTH_POSE xyz, ray xyz, depth (+ pose) -> pts3d predicted, or factored when use_factored != 0
 * point_mode (the three point channels): MA_PTS_LINEAR, MA_PTS_EXP (unit direction x expm1(norm)), MA_PTS_Z_EXP
 * ((x z, y z, z), z = exp(raw z)).  Rays are normalised to the unit sphere, depth = exp, confidence = conf_vmin + exp,
 * mask = sigmoid(logit) > 0.5.  Output pointers the representation does not produce (and conf / logits / mask without
 * has_conf / has_mask, pose_raw / cam_trans / cam_quats without a pose) must be NULL.  Metric scale as in ma_decode_dense. */
#define MA_REP_POINTMAP 0
#define MA_REP_RAYMAP_DEPTH 1
#define MA_REP_RAYDIRS_DEPTH_POSE 2
#define MA_REP_CAMPOINTMAP_POSE 3
#define MA_REP_POINTMAP_RAYDIRS_DEPTH_POSE 4
#define MA_PTS_LINEAR 0
#define MA_PTS_EXP 1
#define MA_PTS_Z_EXP 2
typedef struct ma_decode_spec {
  int rep;          /* MA_REP_* */
  int has_conf;     /* a confidence channel follows the representation */
  int has_mask;     /* a mask-logit channel follows (after the confidence channel when both) */
  int point_mode;   /* MA_PTS_*: activation of the point channels (reps 0, 3, 4) */
  int use_factored; /* rep 4: world points from rays, depth and pose instead of the predicted ones */
  float conf_vmin;  /* confidence = conf_vmin + exp(logit) */
} ma_decode_spec;
int ma_decode_scene(const ma_decode_spec* spec, const float* raw, int ld_raw, const float* pose_raw, const float* scale_raw,
                    int n, int HW, float* pts3d, float* pts3d_cam, float* rays, float* ray_origins, float* depth, float* conf,
                    float* logits, uint8_t* mask, float* cam_trans, float* cam_quats, float* scale_out, void* stream);

/* ---- infer() input preprocessing (reference mapanything/utils/inference.py:202-291; SURVEY 8a row a3) ------------ */

/* get_rays_in_camera_frame(normalize_to_unit_sphere=True) (geometry.py:186-241): K [B][3][3] -> unit rays (B,H,W,3). */
int ma_rays_from_intrinsics(const float* K, float* rays, int B, int H, int W, void* stream);
/* rays / (|rays| + 1e-8) (inference.py:238-241). */
int ma_normalize_rays(const float* in, float* out, int64_t pixels, void* stream);
/* depth_along_ray = |depth_z * ray / ray_z| (inference.py:243-251). */
int ma_depth_z_to_along_ray(const float* depth_z, const float* rays, float* out, int64_t pixels, void* stream);
/* (B,4,4) cam2world matrices -> quats (B,4; xyzw, w >= 0; geometry.py:655-742) and translations (B,3). */
int ma_pose_to_quat_trans(const float* poses, float* quats, float* trans, int B, void* stream);

/* ---- geometric-input fusion (reference model.py:647-1261; SURVEY 8a rows a8-a11) -------------------------- */

/* nn.PixelUnshuffle(patch) of an NHWC fp32 map (n,H,W,cin) (ray directions model.py:803-811 / depth :946-971) written as
 * the split-bf16 activation [hi | lo | hi] of an NHWC token map (n,H/p,W/p,3*cpad), channel k = c*p*p + dy*p + dx zero
 * padded to cpad (multiple of 8).  mode 1 (depth): v /= factor[i]; v = v/max(|v|,1e-8) * log1p(|v|) (geometry.py:1666-1679).
 * patch must be positive and divide H and W; cpad >= cin*patch*patch. */
int ma_unshuffle_split(const float* in, void* out, int n, int H, int W, int cin, int patch, int cpad, int mode,
                       const float* factor, void* stream);

/* normalize_depth_using_non_zero_pixels (geometry.py:1523-1555): factor[i] = mean of the positive depths of view i
 * (clipped at 1e-8); log_factor8[i] = (log(factor + 1e-8), 0 x 7): the K-padded input of the depth-scale encoder. */
int ma_depth_factor(const float* depth, int n, int64_t per_view, float* factor, float* log_factor8, void* stream);

/* Camera-pose inputs: poses relative to view 0 (model.py:647-751, geometry.py:814-852), identity for views without a
 * pose (has_pose[v] == 0), translations normalised by the mean non-zero norm across views (geometry.py:1558-1595).
 * quats [V][4] xyzw, trans [V][3]; outputs K-padded to 8 columns: quats8, trans8, log_scale8 (log(factor + 1e-8)). */
int ma_pose_inputs(const float* quats, const float* trans, const uint8_t* has_pose, int V, float* quats8, float* trans8,
                   float* log_scale8, void* stream);

/* In-place fusion adds on the fp32 encoder features feat [V*N][C] (model.py:820-825, :1003-1008, :1124-1129):
 * feat[v*N+t] += dense_a[a_slot[v]*N+t] + dense_b[b_slot[v]*N+t] + sum_j gw[j*V+v] * g_j[v]; slot -1 / NULL = absent;
 * g3 (depth-scale features) has one row per b_slot and is read at g3[b_slot[v]].  C % 4 == 0; the kernel moves float4, so
 * feat and each of dense_a, dense_b, g0..g3 that is present must be 16-byte aligned. */
int ma_fuse_add(float* feat, int V, int N, int C, const float* dense_a, const int* a_slot, const float* dense_b,
                const int* b_slot, const float* g0, const float* g1, const float* g2, const float* g3, const float* gw,
                void* stream);

/* ---- input side: load_images() (reference mapanything/utils/image.py:134-332) -------------------------------------
 * The reference resizes every decoded RGB image with PIL.Image.resize (LANCZOS when shrinking, BICUBIC when enlarging:
 * cropping.py:188-275), centre-crops it to the target resolution (cropping.py:385-467) and applies torchvision
 * ToTensor + Normalize (image.py:291-296, :312).  PIL's 8-bit resize is integer arithmetic (22-bit fixed-point
 * coefficients, byte-rounded horizontal pass feeding the vertical pass); these entry points reproduce it BIT-EXACTLY. */
#define MA_FILTER_LANCZOS 1 /* = PIL.Image.Resampling.LANCZOS */
#define MA_FILTER_BICUBIC 3 /* = PIL.Image.Resampling.BICUBIC */

/* HOST function (no CUDA): Pillow's resampling windows for one axis, in_size -> out_size.  bounds: int32 [out_size][2] =
 * (first source index, tap count); coeffs: int32 [ksize][out_size] (tap-major), 22-bit fixed point.  *ksize_out is always
 * written; pass bounds = coeffs = NULL to query it.  in_size == out_size gives identity taps (PIL skips that pass). */
int ma_resample_coeffs(int in_size, int out_size, int filter, int* ksize_out, int32_t* bounds, int32_t* coeffs);

/* Horizontal pass over n frames of the same size.  src: device u8 RGB, interleaved; row / frame strides in bytes;
 * source rows [y0, y0+rows) and source columns [sx0, sx1) are read (sx0/sx1 = the window span of output columns
 * [x0, x0+cols)); bounds / coeffs: device copies of the tables for the horizontal axis (ksize taps, out_size columns); packed: optional, see ma_resample_pack_coeffs.
 * tmp: device u8 [n][rows][cols][3].  src may sit at any byte address; y0 and sx0 must be >= 0 and bounds, coeffs and
 * packed 4-byte aligned.  The staged span sx1 - sx0 may be at most 68,264 pixels (a row of it lives in shared memory). */
int ma_resample_h_u8rgb(const uint8_t* src, int64_t src_row_stride, int64_t src_frame_stride, int n, int y0, int rows,
                        int sx0, int sx1, const int32_t* bounds, const int32_t* coeffs, const uint32_t* packed, int ksize,
                        int out_size, int x0, int cols, uint8_t* tmp, void* stream);

/* HOST function: the coefficients of ma_resample_coeffs split into bytes for the dp4a form of the horizontal pass.
 * packed: uint32 [3][ceil(ksize/4)][out_size]; plane 0 / 1 = bits 0-7 / 8-15 (unsigned), plane 2 = bits 16-23 (signed);
 * each word holds 4 consecutive taps.  Pass its device copy as `packed` above (NULL: plain 32-bit coefficients). */
int ma_resample_pack_coeffs(const int32_t* coeffs, int ksize, int out_size, uint32_t* packed);

/* Vertical pass + crop + normalise.  tmp: [n][rows][cols][3] u8 whose row 0 is source row y0; output rows
 * [top, top+th) of the resampled image (out_size rows; bounds / coeffs: the vertical axis' tables, ksize taps).  out_chw: fp32 (n, 3, th, cols) = ((u/255) - mean) / std in
 * torchvision's rounding order (mean / std: 3 HOST floats), may be NULL; out_u8: u8 [n][th][cols][3], may be NULL.
 * bounds, coeffs and out_chw must be 4-byte aligned; th and n at most 65535. */
int ma_resample_v_norm_u8rgb(const uint8_t* tmp, int n, int rows, int cols, int y0, const int32_t* bounds,
                             const int32_t* coeffs, int ksize, int out_size, int top, int th, const float* mean_host,
                             const float* std_host, float* out_chw, uint8_t* out_u8, void* stream);

/* preprocess_inputs() (image.py:335-675) resizes depth maps with cv2.resize(INTER_NEAREST) and slices the crop
 * (cropping.py:248-255, :339): out[y][x] = src[y_idx[y]][x_idx[x]], th x tw; y_idx / x_idx: device int32 source offsets
 * of the cropped window (OpenCV resizeNN: min(floor(i * (1 / (dst / src))), src - 1), computed on the host).
 * src, y_idx, x_idx and out must be 4-byte aligned; th at most 65535. */
int ma_gather_rows_cols_f32(const float* src, int64_t src_row_stride, const int32_t* y_idx, const int32_t* x_idx, int th,
                            int tw, float* out, void* stream);

/* Float image -> bytes as image.py:503-506 does with torch for an fp32 tensor: (in * scale).clamp(0, 255).byte(); n elements.
 * in must be 4-byte aligned. */
int ma_f32_to_u8(const float* in, int64_t n, float scale, uint8_t* out, void* stream);

/* ---- load_images(): baseline JPEG decoding on the GPU ------------------------------------------------------------
 * The reference decodes every file with exif_transpose(PIL.Image.open(f)).convert("RGB") (image.py:134-332), i.e.
 * libjpeg-turbo's default decode: JDCT_ISLOW integer IDCT, fancy upsampling, no merged upsampler, table-driven
 * YCbCr -> RGB.  These entry points reproduce that decode bit for bit for sequential Huffman 8-bit frames with one
 * component or three YCbCr components sampled 4:4:4, 4:2:2, 4:2:0 or 4:4:0; the caller decodes every other file, and
 * every frame ma_jpeg_decode reports, with Pillow. */
#define MA_JPEG_SUBSEQ_BYTES 128 /* entropy-coded bytes per subsequence of the parallel Huffman decode */

typedef struct ma_jpeg_info {
  int32_t width, height;       /* frame size before EXIF orientation */
  int32_t ncomp;               /* 1 (grayscale) or 3 (YCbCr) */
  int32_t h_samp, v_samp;      /* luma sampling factors (chroma is 1x1); 1x1 for grayscale */
  int32_t restart_interval;    /* MCUs per restart interval, 0 = none */
  int32_t nsegments;           /* restart intervals of the scan */
  int32_t nsubseq;             /* subsequences of MA_JPEG_SUBSEQ_BYTES */
  int64_t nblocks;             /* 8x8 coefficient blocks of the scan */
  int64_t plane_bytes;         /* bytes of the frame's sample planes in the workspace */
  int64_t blob_bytes;          /* size of the device blob ma_jpeg_parse writes */
} ma_jpeg_info;

/* HOST function (no CUDA): reads the markers of a JPEG file (file_host, size bytes): SOI, SOF0 / SOF1, DQT, DHT, DRI,
 * APP0 (JFIF), APP14 (Adobe), other APPn / COM skipped, one SOS, entropy-coded data, EOI.  Fills *info; with
 * blob_host != NULL also writes the self-contained device blob (header with the Huffman lookup + canonical tables, the
 * quantisation tables in natural order, restart-interval and subsequence tables, and the entropy-coded bytes with the
 * FF00 stuffing and RSTn markers removed), which needs blob_capacity >= info->blob_bytes; with a smaller capacity the
 * call still fills *info and returns MA_ERR_INVALID, so the caller can retry with info->blob_bytes.  With blob_capacity
 * >= size + 16384 the entropy-coded data is read once, straight into the blob.  Returns MA_ERR_INVALID with a
 * message for: no SOI; a truncated segment or a stream that does not end in EOI; any SOF other than SOF0 / SOF1
 * (progressive, lossless, arithmetic); precision other than 8; 2 or 4 or more components; three components that are not
 * YCbCr (Adobe transform != 1, or 'R','G','B' ids without JFIF) or not sampled as above; a zero frame height (DNL);
 * quantisation or Huffman table indices above 3, a table class above 1, or a scan that refers to a missing table; a
 * Huffman table that is not a valid prefix code (more codes of a length than fit, a code of all 1-bits, more than 256
 * symbols) or a DC symbol above 15;
 * a scan that does not cover every component in frame order, or that is not Ss = 0, Se = 63, Ah = Al = 0; restart
 * markers out of sequence, without DRI, or not one per restart interval; a second scan or any other marker. */
int ma_jpeg_parse(const uint8_t* file_host, int64_t size, ma_jpeg_info* info, uint8_t* blob_host, int64_t blob_capacity);

/* Device workspace ma_jpeg_decode needs for these n frames (infos: HOST array). */
int ma_jpeg_workspace(const ma_jpeg_info* infos, int n, int64_t* bytes);

/* Decodes n frames in one set of launches.  blobs: device copy of the blobs of ma_jpeg_parse, frame i at byte offset
 * blob_offsets_host[i] (16-byte aligned; blobs 16-byte aligned); infos_host: their infos.  out_host[i]: device pointer
 * of frame i's packed RGB output, (H', W', 3) bytes where (W', H') is the frame size after orientation_host[i] (EXIF
 * orientation 1-8; 5-8 swap width and height; other values = 1).  workspace: at least ma_jpeg_workspace bytes,
 * 256-byte aligned.  status: device int32[n], 4-byte aligned, written with 0 for a frame decoded exactly, else a
 * nonzero bit set (1: the entropy-coded data is invalid or holds the wrong number of blocks; 2: the parallel Huffman
 * decode did not synchronise; 4: coefficients outside the range in which every libjpeg-turbo islow IDCT agrees); the
 * output of such a frame is undefined.  n at most 65535. */
int ma_jpeg_decode(const uint8_t* blobs, const int64_t* blob_offsets_host, const ma_jpeg_info* infos_host, int n,
                   uint8_t* const* out_host, const int32_t* orientation_host, void* workspace, int64_t workspace_bytes,
                   int32_t* status, void* stream);

/* ---- infer() post-processing (reference mapanything/utils/inference.py:294-480, host numpy there) ---- */

/* img_no_norm: clip(img * std + mean, 0, 1), (n,3,H,W) -> (n,H,W,3) fp32 (image.py:93-131). mean/std: 3 HOST floats. */
int ma_denorm_image(const float* img, float* out, int n, int H, int W, const float* mean_host, const float* std_host,
                    void* stream);

/* Pinhole intrinsics (n,3,3) from unit ray directions (n,H,W,3) (geometry.py:304-447): 2x2 least squares over
 * the sampled grid for <= 1 MP images, five-pixel closed form above. */
int ma_intrinsics_from_rays(const float* rays, float* K, int n, int H, int W, void* stream);

/* camera_poses (n,4,4) from quats (n,4, xyzw) and translations (n,3) (inference.py:364-379). */
int ma_pose_matrices(const float* quats, const float* trans, float* out, int n, void* stream);

/* Edge mask (inference.py:418-454 + geometry.py:1717-1780, :2031-2072, :2129-2188): mask_out = mask_in & ~(depth_edge &
 * normal_edge).  Normals, normal mask and depth edge are float32-exact with numpy; the neighbour angles use CUDA's acosf,
 * which can differ from numpy's float32 arccos by a few ulp, so only a pixel whose pooled angle lies that close to the
 * threshold can differ from numpy.  depth_z is read with an element stride (pass pts3d_cam + 2,
 * stride 3).  Workspaces per pixel: ws_normals 3 floats, ws_nmask 1 byte, ws_angle 1 float, ws_depth_edge 1 byte. */
int ma_edge_mask(const float* pts3d, const float* depth_z, int depth_stride, const uint8_t* mask_in, uint8_t* mask_out,
                 float* ws_normals, uint8_t* ws_nmask, float* ws_angle, uint8_t* ws_depth_edge, int n, int H, int W,
                 float normal_tol_deg, float depth_rtol, void* stream);

/* out[px, c] = in[px*in_stride + in_offset + c] * mask[px], c < width (inference.py:457-476).  The columns read must lie
 * within one pixel: 0 <= in_offset and in_offset + width <= in_stride (depth_z from pts3d_cam: stride 3, offset 2, width 1). */
int ma_apply_mask(const float* in, int in_stride, int in_offset, const uint8_t* mask, float* out, int64_t pixels, int width,
                  void* stream);

/* Confidence mask (inference.py:393-415): per image thr = torch.quantile(conf, q) (linear interpolation, float32
 * arithmetic of torch: its lerp rounds once, as an FMA) by exact radix selection, mask = conf > thr (1 byte bool).
 * An image holding a NaN gets a NaN threshold and an all-False mask, as torch.quantile propagates NaN.  thr_out [n]
 * optional. */
int ma_quantile_mask(const float* conf, uint8_t* mask, float* thr_out, int n, int64_t per_image, float q, void* stream);

/* depthmap_to_camera_frame / depthmap_to_world_frame (geometry.py:18-114; what every demo calls on infer()'s depth_z,
 * intrinsics and camera_poses: scripts/demo_images_only_inference.py:179): depth (n,H,W), K (n,3,3), pose (n,4,4)
 * cam2world or NULL (camera frame) -> pts (n,H,W,3), valid (n,H,W) bytes = depth > 0 (may be NULL). */
int ma_depthmap_to_world(const float* depth, const float* K, const float* pose, float* pts, uint8_t* valid, int n, int H,
                         int W, void* stream);

/* out = a & b over n bool bytes. */
int ma_mask_and(const uint8_t* a, const uint8_t* b, uint8_t* out, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAPANYTHING_B200_H_ */
