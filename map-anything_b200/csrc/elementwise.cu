// HBM-bound kernels of the MapAnything hot path: coalesced, 16-byte vectorised, warp-primitive reductions.
// Everything between the tensor-core kernels lives here so that no permute().contiguous(), torch.cat or
// separate bias/activation pass is ever materialised (reference: model.py:1245-1259, :1549-1572, :1683-1741).
#include "host_common.h"
#include "ptx.cuh"

namespace ma {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffff, v, o);
  return v;
}

// ----------------------------------------------------------------------------------------------
// patchify: (n,3,H,W) fp32 NCHW image -> [n*hp*wp][kpad] bf16 rows, k = c*p*p + ky*p + kx (the Conv2d weight
// order of DINOv2's PatchEmbed, dinov2/layers/patch_embed.py:65-67), zero padded to kpad.
// ----------------------------------------------------------------------------------------------
__global__ void patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int H, int W, int hp,
                                int wp, int p, int kpad) {
  const int patch = blockIdx.x;  // n*hp*wp
  const int i = patch / (hp * wp);
  const int rem = patch - i * hp * wp;
  const int py = rem / wp, px = rem - py * wp;
  const int kk = 3 * p * p;
  for (int k = threadIdx.x; k < kpad; k += blockDim.x) {
    float v = 0.f;
    if (k < kk) {
      const int c = k / (p * p);
      const int r = k - c * p * p;
      const int ky = r / p, kx = r - ky * p;
      v = __ldg(img + (((size_t)i * 3 + c) * H + (py * p + ky)) * W + px * p + kx);
    }
    out[(size_t)patch * kpad + k] = __float2bfloat16(v);
  }
}

// ----------------------------------------------------------------------------------------------
// LayerNorm over the last dim (eps inside the sqrt, biased variance -- nn.LayerNorm), one warp per row.
// Row remap on both sides lets one launch drop the cls token / skip the scale token / scatter view-major
// rows into the info-sharing layout:   row(r) = (r / rpg) * group_stride + row_offset + r % rpg.
// ----------------------------------------------------------------------------------------------
struct LnParams {
  const void* in;
  void* out;
  const float* gamma;
  const float* beta;
  int64_t ld_in, ld_out;
  int rows, C;
  int rpg;  // rows per group (0 = identity mapping)
  int64_t in_group_stride, in_row_offset, out_group_stride, out_row_offset;
  float eps;
};

template <typename TIn, typename TOut>
__global__ void layernorm_kernel(const LnParams p) {
  const int warps_per_block = blockDim.x >> 5;
  const int r = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (r >= p.rows) return;
  const int lane = threadIdx.x & 31;
  int64_t rin = r, rout = r;
  if (p.rpg > 0) {
    const int g = r / p.rpg, o = r - g * p.rpg;
    rin = (int64_t)g * p.in_group_stride + p.in_row_offset + o;
    rout = (int64_t)g * p.out_group_stride + p.out_row_offset + o;
  }
  const TIn* x = static_cast<const TIn*>(p.in) + rin * p.ld_in;
  TOut* y = static_cast<TOut*>(p.out) + rout * p.ld_out;
  const int C = p.C;

  auto load4 = [&](int c, float (&v)[4]) {
    if constexpr (sizeof(TIn) == 4) {
      float4 t = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + c);
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
      uint2 t = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + c);
      v[0] = bf16_lo(t.x); v[1] = bf16_hi(t.x); v[2] = bf16_lo(t.y); v[3] = bf16_hi(t.y);
    }
  };

  float s = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    float v[4];
    load4(c, v);
    s += (v[0] + v[1]) + (v[2] + v[3]);
  }
  const float mean = warp_sum(s) / C;
  float ss = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    float v[4];
    load4(c, v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float d = v[i] - mean;
      ss = fmaf(d, d, ss);
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) / C + p.eps);
  for (int c = lane * 4; c < C; c += 128) {
    float v[4];
    load4(c, v);
    const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p.beta + c));
    const float o0 = (v[0] - mean) * rstd * g.x + b.x, o1 = (v[1] - mean) * rstd * g.y + b.y;
    const float o2 = (v[2] - mean) * rstd * g.z + b.z, o3 = (v[3] - mean) * rstd * g.w + b.w;
    if constexpr (sizeof(TOut) == 4) {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + c) = make_float4(o0, o1, o2, o3);
    } else {
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + c) = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
    }
  }
}

// Register-resident variant for fp32 rows with C = 128 * NV4 (768 / 1024 on this path): the row is read from global
// memory ONCE (NV4 float4 per lane, all loads in flight together), mean and variance are reduced from registers
// (two-pass, like nn.LayerNorm), the bf16 / fp32 result is written once: 4C B in + 2C (or 4C) B out per row.
template <int NV4, typename TOut>
__global__ void layernorm_f32_reg_kernel(const LnParams p) {
  pdl_sync();  // may be launched programmatically behind the GEMM that produced p.in
  const int warps_per_block = blockDim.x >> 5;
  const int r = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (r >= p.rows) return;
  const int lane = threadIdx.x & 31;
  int64_t rin = r, rout = r;
  if (p.rpg > 0) {
    const int g = r / p.rpg, o = r - g * p.rpg;
    rin = (int64_t)g * p.in_group_stride + p.in_row_offset + o;
    rout = (int64_t)g * p.out_group_stride + p.out_row_offset + o;
  }
  const float4* x = reinterpret_cast<const float4*>(static_cast<const float*>(p.in) + rin * p.ld_in) + lane;
  float4 v[NV4];
#pragma unroll
  for (int i = 0; i < NV4; ++i) v[i] = x[i * 32];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV4; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) / p.C;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    ss = fmaf(a, a, ss); ss = fmaf(b, b, ss); ss = fmaf(c, c, ss); ss = fmaf(d, d, ss);
  }
  const float rstd = rsqrtf(warp_sum(ss) / p.C + p.eps);
  TOut* y = static_cast<TOut*>(p.out) + rout * p.ld_out;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p.beta + c));
    const float o0 = (v[i].x - mean) * rstd * g.x + b.x, o1 = (v[i].y - mean) * rstd * g.y + b.y;
    const float o2 = (v[i].z - mean) * rstd * g.z + b.z, o3 = (v[i].w - mean) * rstd * g.w + b.w;
    if constexpr (sizeof(TOut) == 4) {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + c) = make_float4(o0, o1, o2, o3);
    } else {
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + c) = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
    }
  }
}

// ----------------------------------------------------------------------------------------------
// set_rows: dst[g*group_stride + row_offset][:] = a[:] (+ b[:]), fp32.  (cls token + pos_embed[0]; scale token.)
// ----------------------------------------------------------------------------------------------
__global__ void set_rows_kernel(float* __restrict__ dst, int64_t ld, int64_t group_stride, int64_t row_offset,
                                const float* __restrict__ a, const float* __restrict__ b, int C) {
  float* d = dst + ((int64_t)blockIdx.x * group_stride + row_offset) * ld;
  for (int c = threadIdx.x; c < C; c += blockDim.x) d[c] = a[c] + (b ? b[c] : 0.f);
}

// fill_f32: dst[0:n] = value (the -inf maxima of unused partial softmax states in front of ma_attention_merge).
__global__ void fill_f32_kernel(float* __restrict__ dst, int64_t n, float value) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = value;
}

// ----------------------------------------------------------------------------------------------
// im2col for 3x3 / pad 1 / stride s convolutions over NHWC bf16: out[(i,yo,xo)][tap*C + c], tap = ky*3+kx.
// One thread moves 8 channels (16 B); consecutive threads walk channels then taps -> coalesced both ways.
// ----------------------------------------------------------------------------------------------
__global__ void im2col3x3_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int n, int H,
                                 int W, int C, int Ho, int Wo, int stride) {
  const int c8 = C >> 3;
  const int64_t total = (int64_t)n * Ho * Wo * 9 * c8;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int cc = static_cast<int>(idx % c8);
    int64_t t = idx / c8;
    const int tap = static_cast<int>(t % 9);
    t /= 9;
    const int xo = static_cast<int>(t % Wo);
    t /= Wo;
    const int yo = static_cast<int>(t % Ho);
    const int i = static_cast<int>(t / Ho);
    const int y = yo * stride + tap / 3 - 1, x = xo * stride + tap % 3 - 1;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (y >= 0 && y < H && x >= 0 && x < W)
      v = __ldg(reinterpret_cast<const uint4*>(in + (((size_t)i * H + y) * W + x) * C) + cc);
    reinterpret_cast<uint4*>(out)[idx] = v;
  }
}

// ----------------------------------------------------------------------------------------------
// pixel_shuffle: GEMM output of a ConvTranspose2d with kernel == stride == s,
//   in[(i,y,x)][(ky*s+kx)*C + c]  ->  out NHWC [(i, y*s+ky, x*s+kx)][c]       (bias already added by the GEMM)
// ----------------------------------------------------------------------------------------------
__global__ void pixel_shuffle_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int n, int h,
                                     int w, int C, int s) {
  const int c8 = C >> 3;
  const int64_t total = (int64_t)n * h * w * s * s * c8;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int cc = static_cast<int>(idx % c8);
    int64_t t = idx / c8;
    const int kk = static_cast<int>(t % (s * s));
    t /= (s * s);
    const int x = static_cast<int>(t % w);
    t /= w;
    const int y = static_cast<int>(t % h);
    const int i = static_cast<int>(t / h);
    const int ky = kk / s, kx = kk - ky * s;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(in) + idx);
    reinterpret_cast<uint4*>(out + (((size_t)i * h * s + (y * s + ky)) * (w * s) + (x * s + kx)) * C)[cc] = v;
  }
}

// The same permutation in fp32 with row strides, for the `linear` prediction head (reference model.py:339-343: a 1x1
// conv to output_dim * patch^2 channels + F.pixel_shuffle): the GEMM writes [(i,y,x)][(ky*s+kx)*C + c] (weight rows
// reordered at pack time), this kernel scatters it to the per-pixel rows [(i, y*s+ky, x*s+kx)][0:C] the decode reads.
__global__ void pixel_shuffle_f32_kernel(const float* __restrict__ in, int64_t ld_in, float* __restrict__ out, int64_t ld_out,
                                         int n, int h, int w, int C, int s) {
  const int64_t total = (int64_t)n * h * w * s * s * C;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    int64_t t = idx / C;
    const int kk = static_cast<int>(t % (s * s));
    t /= (s * s);
    const int x = static_cast<int>(t % w);
    const int64_t row = t;   // (i*h + y)*w + x
    t /= w;
    const int y = static_cast<int>(t % h);
    const int i = static_cast<int>(t / h);
    const int ky = kk / s, kx = kk - ky * s;
    out[(((int64_t)i * h * s + (y * s + ky)) * (w * s) + (x * s + kx)) * ld_out + c] = __ldg(in + row * ld_in + kk * C + c);
  }
}

// ----------------------------------------------------------------------------------------------
// bilinear resize, align_corners=True, NHWC bf16.  The scale is defined by the VIRTUAL output size (Hv, Wv);
// only the top-left (Ho, Wo) window is produced (refinenet4: 19 -> 38, cropped to 37; SURVEY App. A.4).
// ----------------------------------------------------------------------------------------------
// One block per output row (image i, row yo): the vertical taps / weights are block constants, the horizontal ones
// come from one multiply per pixel, and consecutive threads walk (xo, 8-channel chunk) so that loads and stores are
// fully coalesced 16-byte accesses.
__global__ void bilinear_ac_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int n, int Hin,
                                   int Win, int C, int Hv, int Wv, int Ho, int Wo) {
  const int c8 = C >> 3;
  const int i = blockIdx.x / Ho, yo = blockIdx.x - i * Ho;
  const float sy = Hv > 1 ? (float)(Hin - 1) / (float)(Hv - 1) : 0.f;
  const float sx = Wv > 1 ? (float)(Win - 1) / (float)(Wv - 1) : 0.f;
  const float fy = yo * sy;
  const int y0 = min((int)fy, Hin - 1);
  const int y1 = min(y0 + 1, Hin - 1);
  const float wy = fy - y0;
  const uint4* row0 = reinterpret_cast<const uint4*>(in + ((size_t)i * Hin + y0) * Win * C);
  const uint4* row1 = reinterpret_cast<const uint4*>(in + ((size_t)i * Hin + y1) * Win * C);
  uint4* orow = reinterpret_cast<uint4*>(out + ((size_t)i * Ho + yo) * Wo * C);
  const int total = Wo * c8;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int xo = idx / c8, cc = idx - xo * c8;
    const float fx = xo * sx;
    const int x0 = min((int)fx, Win - 1), x1 = min(x0 + 1, Win - 1);
    const float wx = fx - x0;
    const uint4 a = __ldg(row0 + x0 * c8 + cc), b = __ldg(row0 + x1 * c8 + cc);
    const uint4 c = __ldg(row1 + x0 * c8 + cc), d = __ldg(row1 + x1 * c8 + cc);
    const uint32_t aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w};
    const uint32_t cw[4] = {c.x, c.y, c.z, c.w}, dd[4] = {d.x, d.y, d.z, d.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float t0 = bf16_lo(aa[j]) + wx * (bf16_lo(bb[j]) - bf16_lo(aa[j]));
      const float b0 = bf16_lo(cw[j]) + wx * (bf16_lo(dd[j]) - bf16_lo(cw[j]));
      const float t1 = bf16_hi(aa[j]) + wx * (bf16_hi(bb[j]) - bf16_hi(aa[j]));
      const float b1 = bf16_hi(cw[j]) + wx * (bf16_hi(dd[j]) - bf16_hi(cw[j]));
      o[j] = pack_bf16x2(t0 + wy * (b0 - t0), t1 + wy * (b1 - t1));
    }
    orow[idx] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ----------------------------------------------------------------------------------------------
// token mean: [n][T][C] bf16 -> [n][C] bf16 (AdaptiveAvgPool2d(1) of the pose head).  grid (C/64, n), block 256.
// ----------------------------------------------------------------------------------------------
__global__ void token_mean_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int T, int C) {
  __shared__ float red[8][64];
  const int c = blockIdx.x * 64 + (threadIdx.x & 63);
  const int rl = threadIdx.x >> 6;  // 0..3
  const __nv_bfloat16* base = in + (size_t)blockIdx.y * T * C;
  float s = 0.f;
  if (c < C)
    for (int t = rl; t < T; t += 4) s += __bfloat162float(base[(size_t)t * C + c]);
  red[rl][threadIdx.x & 63] = s;
  __syncthreads();
  if (rl == 0 && c < C) {
    const float tot = (red[0][threadIdx.x] + red[1][threadIdx.x]) + (red[2][threadIdx.x] + red[3][threadIdx.x]);
    out[(size_t)blockIdx.y * C + c] = __float2bfloat16(tot / T);
  }
}

// ----------------------------------------------------------------------------------------------
// Narrow linear head: out[row][0:N] = W[N][K] . x[row] + b, N <= 8, K <= 256 (the last 1x1 conv of the DPT regressor,
// 128 -> 6 channels on every 518 x 518 pixel).  Pure streaming read of x (2K bytes per row); a tensor-core tile would
// carry 6 useful columns of 64.  One thread per row, W broadcast from shared memory, fp32 accumulate.
// ----------------------------------------------------------------------------------------------
__global__ void head_linear_small_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const __nv_bfloat16* __restrict__ w,
                                         int64_t ldw, const float* __restrict__ bias, float* __restrict__ out, int64_t ldo,
                                         int64_t rows, int N, int K) {
  __shared__ __align__(16) float sw[8][256];
  for (int i = threadIdx.x; i < 8 * K; i += blockDim.x) {
    const int n = i / K, k = i - n * K;
    sw[n][k] = n < N ? __bfloat162float(w[(int64_t)n * ldw + k]) : 0.f;
  }
  __syncthreads();
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < rows; row += (int64_t)gridDim.x * blockDim.x) {
    float acc[8];
#pragma unroll
    for (int n = 0; n < 8; ++n) acc[n] = (bias && n < N) ? __ldg(bias + n) : 0.f;
    const uint4* xr = reinterpret_cast<const uint4*>(x + row * ldx);
#pragma unroll 4
    for (int k8 = 0; k8 < K / 8; ++k8) {
      const uint4 u = __ldcs(xr + k8);  // streamed once
      const float xv[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y), bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        const float4 w0 = *reinterpret_cast<const float4*>(&sw[n][k8 * 8]);
        const float4 w1 = *reinterpret_cast<const float4*>(&sw[n][k8 * 8 + 4]);
        acc[n] = fmaf(xv[0], w0.x, acc[n]); acc[n] = fmaf(xv[1], w0.y, acc[n]);
        acc[n] = fmaf(xv[2], w0.z, acc[n]); acc[n] = fmaf(xv[3], w0.w, acc[n]);
        acc[n] = fmaf(xv[4], w1.x, acc[n]); acc[n] = fmaf(xv[5], w1.y, acc[n]);
        acc[n] = fmaf(xv[6], w1.z, acc[n]); acc[n] = fmaf(xv[7], w1.w, acc[n]);
      }
    }
    float* o = out + row * ldo;
#pragma unroll
    for (int n = 0; n < 8; ++n)
      if (n < N) o[n] = acc[n];
  }
}

// Warp-cooperative form for K = 8 * LPR (LPR = lanes per row, a power of two <= 32): LPR consecutive lanes read one row
// as LPR 16-byte pieces -- every load instruction of a warp covers 32 / LPR whole rows, 512 contiguous bytes, instead of
// 32 different rows (the thread-per-row kernel above reached 0.26 of the HBM roofline: ncu / bench, 550 MB in 0.32 ms).
// Each lane keeps its 8 x N weights in registers, forms N partial dot products and the LPR lanes of a row combine them
// with a shuffle tree.  Output: N (<= 8) fp32 per row.
template <int LPR>
__global__ void head_linear_small_warp_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const __nv_bfloat16* __restrict__ w,
                                              int64_t ldw, const float* __restrict__ bias, float* __restrict__ out, int64_t ldo,
                                              int64_t rows, int N) {
  constexpr int RPW = 32 / LPR;  // rows per warp instruction
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR, rsel = lane / LPR;
  float wr[8][8];  // [n][j]: weights of this lane's 8 input channels
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int j = 0; j < 8; ++j) wr[n][j] = n < N ? __bfloat162float(w[(int64_t)n * ldw + sub * 8 + j]) : 0.f;
  float bv = 0.f;
  if (bias != nullptr && sub < N) bv = __ldg(bias + sub);
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  constexpr int U = 4;  // row groups in flight per warp: 4 x 512 B of loads issued before the first FMA
  for (int64_t r0 = warp * (RPW * U); r0 < rows; r0 += nwarps * (RPW * U)) {
    uint4 u[U];
#pragma unroll
    for (int t = 0; t < U; ++t) {
      const int64_t row = r0 + t * RPW + rsel;
      u[t] = make_uint4(0u, 0u, 0u, 0u);
      if (row < rows) u[t] = __ldcs(reinterpret_cast<const uint4*>(x + row * ldx) + sub);  // streamed once
    }
#pragma unroll
    for (int t = 0; t < U; ++t) {
      const int64_t row = r0 + t * RPW + rsel;
      const float xv[8] = {bf16_lo(u[t].x), bf16_hi(u[t].x), bf16_lo(u[t].y), bf16_hi(u[t].y),
                           bf16_lo(u[t].z), bf16_hi(u[t].z), bf16_lo(u[t].w), bf16_hi(u[t].w)};
      float acc[8];
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        acc[n] = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[n] = fmaf(xv[j], wr[n][j], acc[n]);
      }
      // shuffle tree over the LPR lanes of the row; afterwards every lane of the group holds all N sums
#pragma unroll
      for (int off = LPR / 2; off >= 1; off >>= 1)
#pragma unroll
        for (int n = 0; n < 8; ++n) acc[n] += __shfl_xor_sync(0xffffffffu, acc[n], off);
      // lane `sub` of the group writes output channel `sub`: N consecutive floats per row leave from N consecutive lanes
      if (row < rows && sub < N) {
        float v = acc[0];
#pragma unroll
        for (int n = 1; n < 8; ++n) v = sub == n ? acc[n] : v;
        out[row * ldo + sub] = v + bv;
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------
// Fused dense adaptor + factored-geometry decode + packaging (reference model.py:1683-1741, :1874-1907,
// geometry.py:855-907, adaptor semantics SURVEY App. A.5/A.6):
//   raw[pixel][0:3] ray (linear) -> /|ray| ; raw[3] -> depth = exp ; raw[4] -> conf = 1 + exp ; raw[5] -> mask logits
//   pose_raw[view] = (t, q) -> q/|q| -> R ; scale = clamp(exp(scale_raw), 1e-8)
//   pts3d_cam = ray*depth ; pts3d = R pts3d_cam + t ; metric scale on pts3d, pts3d_cam, depth, cam_trans.
// ----------------------------------------------------------------------------------------------
struct DecodeParams {
  const float* raw;  // [n*HW][ld_raw]
  int ld_raw;
  const float* pose_raw;   // [n][7]
  const float* scale_raw;  // [1]
  float* pts3d;            // [n*HW][3]
  float* pts3d_cam;        // [n*HW][3]
  float* rays;             // [n*HW][3]
  float* depth;            // [n*HW]
  float* conf;             // [n*HW]
  float* logits;           // [n*HW]
  uint8_t* mask;           // [n*HW] (bool)
  float* cam_trans;        // [n][3]
  float* cam_quats;        // [n][4]
  float* scale_out;        // [1]
  int n, HW;
};

__global__ void decode_dense_kernel(const DecodeParams p) {
  const int view = blockIdx.y;
  const float* pr = p.pose_raw + view * 7;
  const float scale = fmaxf(expf(p.scale_raw[0]), 1e-8f);
  float qx = pr[3], qy = pr[4], qz = pr[5], qw = pr[6];
  {
    // pose adaptor: q / |q|  (then geometry.py:883 and :621 re-normalise; idempotent up to rounding)
    const float inv = 1.0f / sqrtf(qx * qx + qy * qy + qz * qz + qw * qw);
    qx *= inv; qy *= inv; qz *= inv; qw *= inv;
  }
  const float tx = pr[0], ty = pr[1], tz = pr[2];
  const float r00 = 1 - 2 * (qy * qy + qz * qz), r01 = 2 * (qx * qy - qw * qz), r02 = 2 * (qx * qz + qw * qy);
  const float r10 = 2 * (qx * qy + qw * qz), r11 = 1 - 2 * (qx * qx + qz * qz), r12 = 2 * (qy * qz - qw * qx);
  const float r20 = 2 * (qx * qz - qw * qy), r21 = 2 * (qy * qz + qw * qx), r22 = 1 - 2 * (qx * qx + qy * qy);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    p.cam_trans[view * 3 + 0] = tx * scale;
    p.cam_trans[view * 3 + 1] = ty * scale;
    p.cam_trans[view * 3 + 2] = tz * scale;
    p.cam_quats[view * 4 + 0] = qx;
    p.cam_quats[view * 4 + 1] = qy;
    p.cam_quats[view * 4 + 2] = qz;
    p.cam_quats[view * 4 + 3] = qw;
    if (view == 0) p.scale_out[0] = scale;
  }
  for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < p.HW; px += gridDim.x * blockDim.x) {
    const size_t g = (size_t)view * p.HW + px;
    const float* r = p.raw + g * p.ld_raw;
    float a[6];
    if ((p.ld_raw & 3) == 0) {
      const float4 v0 = *reinterpret_cast<const float4*>(r);
      const float2 v1 = *reinterpret_cast<const float2*>(r + 4);
      a[0] = v0.x; a[1] = v0.y; a[2] = v0.z; a[3] = v0.w; a[4] = v1.x; a[5] = v1.y;
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) a[i] = r[i];
    }
    const float inv = 1.0f / sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    const float dx = a[0] * inv, dy = a[1] * inv, dz = a[2] * inv;
    const float depth = expf(a[3]);
    const float cx = dx * depth, cy = dy * depth, cz = dz * depth;
    const float wx = r00 * cx + r01 * cy + r02 * cz + tx;
    const float wy = r10 * cx + r11 * cy + r12 * cz + ty;
    const float wz = r20 * cx + r21 * cy + r22 * cz + tz;
    p.rays[g * 3 + 0] = dx; p.rays[g * 3 + 1] = dy; p.rays[g * 3 + 2] = dz;
    p.pts3d_cam[g * 3 + 0] = cx * scale; p.pts3d_cam[g * 3 + 1] = cy * scale; p.pts3d_cam[g * 3 + 2] = cz * scale;
    p.pts3d[g * 3 + 0] = wx * scale; p.pts3d[g * 3 + 1] = wy * scale; p.pts3d[g * 3 + 2] = wz * scale;
    p.depth[g] = depth * scale;
    p.conf[g] = 1.0f + expf(a[4]);
    p.logits[g] = a[5];
    p.mask[g] = (1.0f / (1.0f + expf(-a[5]))) > 0.5f ? 1 : 0;
  }
}

// ----------------------------------------------------------------------------------------------
// The same decode for the other scene representations of the reference (model.py:407-587, :1618-1907); the
// representation / activation selectors are uniform over the launch.  See ma_decode_scene in the header.
// ----------------------------------------------------------------------------------------------
struct DecodeSceneParams {
  ma_decode_spec spec;
  const float* raw;
  int ld_raw;
  const float* pose_raw;
  const float* scale_raw;
  float *pts3d, *pts3d_cam, *rays, *origins, *depth, *conf, *logits;
  uint8_t* mask;
  float *cam_trans, *cam_quats, *scale_out;
  int n, HW;
};

__device__ __forceinline__ void point_activation(int mode, float& x, float& y, float& z) {
  if (mode == MA_PTS_EXP) {  // unit direction x expm1(norm)
    const float d = sqrtf(x * x + y * y + z * z);
    const float f = expm1f(d) / fmaxf(d, 1e-8f);
    x *= f; y *= f; z *= f;
  } else if (mode == MA_PTS_Z_EXP) {
    z = expf(z);
    x *= z; y *= z;
  }
}

__device__ __forceinline__ void store3(float* p, size_t g, float x, float y, float z) {
  p[g * 3 + 0] = x; p[g * 3 + 1] = y; p[g * 3 + 2] = z;
}

__global__ void decode_scene_kernel(const DecodeSceneParams p) {
  const int view = blockIdx.y;
  const int rep = p.spec.rep;
  const float scale = fmaxf(expf(p.scale_raw[0]), 1e-8f);
  float tx = 0.f, ty = 0.f, tz = 0.f;
  float r00 = 1, r01 = 0, r02 = 0, r10 = 0, r11 = 1, r12 = 0, r20 = 0, r21 = 0, r22 = 1;
  if (p.pose_raw != nullptr) {
    const float* pr = p.pose_raw + view * 7;
    float qx = pr[3], qy = pr[4], qz = pr[5], qw = pr[6];
    const float inv = 1.0f / sqrtf(qx * qx + qy * qy + qz * qz + qw * qw);
    qx *= inv; qy *= inv; qz *= inv; qw *= inv;
    tx = pr[0]; ty = pr[1]; tz = pr[2];
    r00 = 1 - 2 * (qy * qy + qz * qz); r01 = 2 * (qx * qy - qw * qz); r02 = 2 * (qx * qz + qw * qy);
    r10 = 2 * (qx * qy + qw * qz); r11 = 1 - 2 * (qx * qx + qz * qz); r12 = 2 * (qy * qz - qw * qx);
    r20 = 2 * (qx * qz - qw * qy); r21 = 2 * (qy * qz + qw * qx); r22 = 1 - 2 * (qx * qx + qy * qy);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      store3(p.cam_trans, view, tx * scale, ty * scale, tz * scale);
      p.cam_quats[view * 4 + 0] = qx; p.cam_quats[view * 4 + 1] = qy;
      p.cam_quats[view * 4 + 2] = qz; p.cam_quats[view * 4 + 3] = qw;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && view == 0) p.scale_out[0] = scale;
  const int rep_ch = rep == MA_REP_POINTMAP || rep == MA_REP_CAMPOINTMAP_POSE ? 3 : rep == MA_REP_RAYDIRS_DEPTH_POSE ? 4 : 7;
  const int total_ch = rep_ch + (p.spec.has_conf ? 1 : 0) + (p.spec.has_mask ? 1 : 0);
  for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < p.HW; px += gridDim.x * blockDim.x) {
    const size_t g = (size_t)view * p.HW + px;
    const float* r = p.raw + g * p.ld_raw;
    float a[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) a[i] = i < total_ch ? r[i] : 0.f;
    if (rep == MA_REP_POINTMAP) {
      point_activation(p.spec.point_mode, a[0], a[1], a[2]);
      store3(p.pts3d, g, a[0] * scale, a[1] * scale, a[2] * scale);
    } else if (rep == MA_REP_RAYMAP_DEPTH) {
      const float inv = 1.0f / sqrtf(a[3] * a[3] + a[4] * a[4] + a[5] * a[5]);
      const float dx = a[3] * inv, dy = a[4] * inv, dz = a[5] * inv;
      const float depth = expf(a[6]);
      store3(p.origins, g, a[0] * scale, a[1] * scale, a[2] * scale);
      store3(p.rays, g, dx, dy, dz);
      store3(p.pts3d, g, (a[0] + dx * depth) * scale, (a[1] + dy * depth) * scale, (a[2] + dz * depth) * scale);
      p.depth[g] = depth * scale;
    } else {
      // the three posed representations: rays + depth (+ predicted world points), camera points = rays x depth
      float dx, dy, dz, depth, cx, cy, cz, wx = 0.f, wy = 0.f, wz = 0.f;
      bool world_predicted = false;
      if (rep == MA_REP_CAMPOINTMAP_POSE) {
        point_activation(p.spec.point_mode, a[0], a[1], a[2]);
        depth = sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
        dx = a[0] / depth; dy = a[1] / depth; dz = a[2] / depth;
        cx = a[0]; cy = a[1]; cz = a[2];   // pts3d_cam is the prediction itself (model.py:1751)
      } else {
        const int o = rep == MA_REP_RAYDIRS_DEPTH_POSE ? 0 : 3;
        const float inv = 1.0f / sqrtf(a[o] * a[o] + a[o + 1] * a[o + 1] + a[o + 2] * a[o + 2]);
        dx = a[o] * inv; dy = a[o + 1] * inv; dz = a[o + 2] * inv;
        depth = expf(a[o + 3]);
        cx = dx * depth; cy = dy * depth; cz = dz * depth;
        if (rep == MA_REP_POINTMAP_RAYDIRS_DEPTH_POSE && !p.spec.use_factored) {
          point_activation(p.spec.point_mode, a[0], a[1], a[2]);
          wx = a[0]; wy = a[1]; wz = a[2];
          world_predicted = true;
        }
      }
      if (!world_predicted) {  // geometry.py:855-907 on rays x depth
        const float fx = dx * depth, fy = dy * depth, fz = dz * depth;
        wx = r00 * fx + r01 * fy + r02 * fz + tx;
        wy = r10 * fx + r11 * fy + r12 * fz + ty;
        wz = r20 * fx + r21 * fy + r22 * fz + tz;
      }
      store3(p.rays, g, dx, dy, dz);
      store3(p.pts3d_cam, g, cx * scale, cy * scale, cz * scale);
      store3(p.pts3d, g, wx * scale, wy * scale, wz * scale);
      p.depth[g] = depth * scale;
    }
    int c = rep_ch;
    if (p.spec.has_conf) p.conf[g] = p.spec.conf_vmin + expf(a[c++]);
    if (p.spec.has_mask) {
      const float l = a[c];
      p.logits[g] = l;
      p.mask[g] = (1.0f / (1.0f + expf(-l))) > 0.5f ? 1 : 0;
    }
  }
}

// ----------------------------------------------------------------------------------------------
// split_bf16x3: fp32 [rows][C] -> bf16 [rows][3C] = [hi | lo | hi] per group of C channels, hi = bf16(x),
// lo = bf16(x - hi).  Against weights packed as [w_hi | w_hi | w_lo] one bf16 tensor-core GEMM over K' = 3K computes
// a_hi*w_hi + a_lo*w_hi + a_hi*w_lo with fp32 accumulation: ~2^-16 relative error per product instead of 2^-8.
// Used where the reference runs fp32 (autocast disabled, model.py:1599) and the output feeds a normalisation
// (pose quaternion, metric scale).
// ----------------------------------------------------------------------------------------------
__global__ void split_bf16x3_kernel(const float* __restrict__ in, int64_t ld_in, __nv_bfloat16* __restrict__ out, int rows,
                                    int C) {
  const int c4 = C >> 2;
  const int64_t total = (int64_t)rows * c4;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / c4;
    const int c = static_cast<int>(idx - r * c4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(in + r * ld_in + c);
    const float x[4] = {v.x, v.y, v.z, v.w};
    float hi[4], lo[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      hi[i] = __bfloat162float(__float2bfloat16(x[i]));
      lo[i] = x[i] - hi[i];
    }
    const uint2 h = make_uint2(pack_bf16x2(hi[0], hi[1]), pack_bf16x2(hi[2], hi[3]));
    const uint2 l = make_uint2(pack_bf16x2(lo[0], lo[1]), pack_bf16x2(lo[2], lo[3]));
    __nv_bfloat16* o = out + r * (3 * (int64_t)C) + c;
    *reinterpret_cast<uint2*>(o) = h;
    *reinterpret_cast<uint2*>(o + C) = l;
    *reinterpret_cast<uint2*>(o + 2 * C) = h;
  }
}

// fp32 token mean: [n][T][C] -> [n][C]
// block = 64 channels x 16 row lanes, four independent loads in flight per thread (the first form -- 4 row lanes, one load in
// flight -- took 58 us for 8 x 1369 x 768: 96 blocks cannot hide the latency of 342 dependent steps each)
__global__ void __launch_bounds__(1024) token_mean_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int T, int C) {
  __shared__ float red[16][64];
  const int c = blockIdx.x * 64 + (threadIdx.x & 63);
  const int rl = threadIdx.x >> 6;  // 0..15
  const float* base = in + (size_t)blockIdx.y * T * C;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (c < C) {
    int t = rl;
    for (; t + 48 < T; t += 64) {
      s0 += base[(size_t)t * C + c];
      s1 += base[(size_t)(t + 16) * C + c];
      s2 += base[(size_t)(t + 32) * C + c];
      s3 += base[(size_t)(t + 48) * C + c];
    }
    for (; t < T; t += 16) s0 += base[(size_t)t * C + c];
  }
  red[rl][threadIdx.x & 63] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (rl == 0 && c < C) {
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) tot += red[i][threadIdx.x];
    out[(size_t)blockIdx.y * C + c] = tot / T;
  }
}

// ----------------------------------------------------------------------------------------------
// fp32 Linear on a handful of rows: out[r][n] = act(b[n] + sum_k x[r][k] * w[n][k]), rows <= 16 (the pooled MLPs of the pose
// head and the scale head: 8 x 768 or 1 x 768 inputs).  A tensor-core tile would carry 8 useful rows of 128 and, in the
// split-bf16 form those layers otherwise use, a single CTA walks K' = 3K alone (23 - 37 us per launch).  Here x sits in shared
// memory, one warp owns an output column: lanes stride over k with float4 loads of the weight row, 16 accumulators, one
// shuffle reduction per row.  Plain fp32 FMAs.
// ----------------------------------------------------------------------------------------------
constexpr int LIN_ROWS_MAX = 16;
__global__ void __launch_bounds__(256) linear_rows_f32_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                                                              int64_t ldw, const float* __restrict__ bias, float* __restrict__ out,
                                                              int64_t ldo, int rows, int N, int K, int act) {
  extern __shared__ float sx[];  // [rows][K]
  for (int i = threadIdx.x; i < rows * (K >> 2); i += blockDim.x) {
    const int r = i / (K >> 2), q = i - r * (K >> 2);
    reinterpret_cast<float4*>(sx)[i] = *reinterpret_cast<const float4*>(x + r * ldx + 4 * q);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  float acc[LIN_ROWS_MAX];
#pragma unroll
  for (int r = 0; r < LIN_ROWS_MAX; ++r) acc[r] = 0.f;
  const float4* wr = reinterpret_cast<const float4*>(w + (int64_t)n * ldw);
  for (int q = lane; q < (K >> 2); q += 32) {
    const float4 wv = __ldg(wr + q);
#pragma unroll
    for (int r = 0; r < LIN_ROWS_MAX; ++r) {
      if (r < rows) {
        const float4 xv = reinterpret_cast<const float4*>(sx + r * K)[q];
        acc[r] = fmaf(xv.x, wv.x, acc[r]);
        acc[r] = fmaf(xv.y, wv.y, acc[r]);
        acc[r] = fmaf(xv.z, wv.z, acc[r]);
        acc[r] = fmaf(xv.w, wv.w, acc[r]);
      }
    }
  }
  const float b = bias ? bias[n] : 0.f;
#pragma unroll
  for (int r = 0; r < LIN_ROWS_MAX; ++r) {
    if (r < rows) {
      float v = warp_sum(acc[r]) + b;
      if (act == MA_ACT_RELU) v = fmaxf(v, 0.f);
      else if (act == MA_ACT_GELU) v = gelu_erf(v);
      if (lane == 0) out[r * ldo + n] = v;
    }
  }
}

static inline int grid_for(int64_t total, int block, int max_blocks) {
  int64_t g = (total + block - 1) / block;
  if (g > max_blocks) g = max_blocks;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace ma

using namespace ma;

extern "C" int ma_patchify(const float* img, void* out, int n, int H, int W, int patch, int kpad, void* stream) {
  MA_REQUIRE(img && out && n > 0 && patch > 0 && H % patch == 0 && W % patch == 0 && kpad >= 3 * patch * patch && kpad % 8 == 0,
             "ma_patchify: bad arguments (H=%d W=%d patch=%d kpad=%d)", H, W, patch, kpad);
  const int hp = H / patch, wp = W / patch;
  patchify_kernel<<<n * hp * wp, 128, 0, static_cast<cudaStream_t>(stream)>>>(img, static_cast<__nv_bfloat16*>(out), H, W,
                                                                               hp, wp, patch, kpad);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_layernorm(const void* in, int in_dtype, int64_t ld_in, void* out, int out_dtype, int64_t ld_out,
                            const float* gamma, const float* beta, int rows, int C, float eps, int rows_per_group,
                            int64_t in_group_stride, int64_t in_row_offset, int64_t out_group_stride,
                            int64_t out_row_offset, void* stream) {
  MA_REQUIRE(in && out && gamma && beta && rows > 0 && C > 0 && C % 4 == 0, "ma_layernorm: bad arguments (rows=%d C=%d)", rows, C);
  MA_REQUIRE(ld_in % 4 == 0 && ld_out % 4 == 0, "ma_layernorm: row strides must be multiples of 4 elements");
  MA_REQUIRE(ld_in >= C, "ma_layernorm: ld_in (%lld) below C = %d", (long long)ld_in, C);
  MA_REQUIRE(ld_out >= C, "ma_layernorm: ld_out (%lld) below C = %d", (long long)ld_out, C);
  // four elements per access: float4 / uint2 loads of in, stores of out, float4 loads of gamma and beta
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & (in_dtype == MA_F32 ? 15 : 7)) == 0, "ma_layernorm: in not %d-byte aligned",
             in_dtype == MA_F32 ? 16 : 8);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & (out_dtype == MA_F32 ? 15 : 7)) == 0, "ma_layernorm: out not %d-byte aligned",
             out_dtype == MA_F32 ? 16 : 8);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(gamma) & 15) == 0, "ma_layernorm: gamma not 16-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(beta) & 15) == 0, "ma_layernorm: beta not 16-byte aligned");
  LnParams p{in, out, gamma, beta, ld_in, ld_out, rows, C, rows_per_group, in_group_stride, in_row_offset,
             out_group_stride, out_row_offset, eps};
  const int wpb = 8;
  const int grid = (rows + wpb - 1) / wpb;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool vec_ok = in_dtype == MA_F32 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  if (vec_ok && C == 1024 && out_dtype == MA_BF16) MA_CHECK_CUDA(launch_kernel(layernorm_f32_reg_kernel<8, __nv_bfloat16>, dim3(grid), dim3(wpb * 32), 0, s, pdl_enabled(), p));
  else if (vec_ok && C == 768 && out_dtype == MA_BF16) MA_CHECK_CUDA(launch_kernel(layernorm_f32_reg_kernel<6, __nv_bfloat16>, dim3(grid), dim3(wpb * 32), 0, s, pdl_enabled(), p));
  else if (vec_ok && C == 1024 && out_dtype == MA_F32) MA_CHECK_CUDA(launch_kernel(layernorm_f32_reg_kernel<8, float>, dim3(grid), dim3(wpb * 32), 0, s, pdl_enabled(), p));
  else if (vec_ok && C == 768 && out_dtype == MA_F32) MA_CHECK_CUDA(launch_kernel(layernorm_f32_reg_kernel<6, float>, dim3(grid), dim3(wpb * 32), 0, s, pdl_enabled(), p));
  else if (in_dtype == MA_F32 && out_dtype == MA_BF16) layernorm_kernel<float, __nv_bfloat16><<<grid, wpb * 32, 0, s>>>(p);
  else if (in_dtype == MA_F32 && out_dtype == MA_F32) layernorm_kernel<float, float><<<grid, wpb * 32, 0, s>>>(p);
  else if (in_dtype == MA_BF16 && out_dtype == MA_BF16) layernorm_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, wpb * 32, 0, s>>>(p);
  else if (in_dtype == MA_BF16 && out_dtype == MA_F32) layernorm_kernel<__nv_bfloat16, float><<<grid, wpb * 32, 0, s>>>(p);
  else MA_REQUIRE(false, "ma_layernorm: unsupported dtypes %d -> %d", in_dtype, out_dtype);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_set_rows(float* dst, int64_t ld, int groups, int64_t group_stride, int64_t row_offset, const float* a,
                           const float* b, int C, void* stream) {
  MA_REQUIRE(dst && a && groups > 0 && C > 0, "ma_set_rows: bad arguments");
  MA_REQUIRE(ld >= C, "ma_set_rows: ld (%lld) below C = %d", (long long)ld, C);
  set_rows_kernel<<<groups, 256, 0, static_cast<cudaStream_t>(stream)>>>(dst, ld, group_stride, row_offset, a, b, C);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_fill_f32(float* dst, int64_t n, float value, void* stream) {
  MA_REQUIRE(dst && n > 0, "ma_fill_f32: bad arguments");
  fill_f32_kernel<<<grid_for(n, 256, device_sm_count() * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(dst, n, value);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_im2col3x3(const void* in, void* out, int n, int H, int W, int C, int stride, void* stream) {
  MA_REQUIRE(in && out && n > 0 && C % 8 == 0 && (stride == 1 || stride == 2), "ma_im2col3x3: bad arguments (C=%d stride=%d)", C, stride);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0, "ma_im2col3x3: in not 16-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "ma_im2col3x3: out not 16-byte aligned");
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  const int64_t total = (int64_t)n * Ho * Wo * 9 * (C / 8);
  im2col3x3_kernel<<<grid_for(total, 256, device_sm_count() * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in), static_cast<__nv_bfloat16*>(out), n, H, W, C, Ho, Wo, stride);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_pixel_shuffle(const void* in, void* out, int n, int h, int w, int C, int s, void* stream) {
  MA_REQUIRE(in && out && n > 0 && C % 8 == 0 && s > 0, "ma_pixel_shuffle: bad arguments");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0, "ma_pixel_shuffle: in not 16-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "ma_pixel_shuffle: out not 16-byte aligned");
  const int64_t total = (int64_t)n * h * w * s * s * (C / 8);
  pixel_shuffle_kernel<<<grid_for(total, 256, device_sm_count() * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in), static_cast<__nv_bfloat16*>(out), n, h, w, C, s);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_pixel_shuffle_f32(const float* in, int64_t ld_in, float* out, int64_t ld_out, int n, int h, int w, int C,
                                    int s, void* stream) {
  MA_REQUIRE(in && out && n > 0 && h > 0 && w > 0 && C > 0 && s > 0 && ld_in >= (int64_t)s * s * C && ld_out >= C,
             "ma_pixel_shuffle_f32: bad arguments");
  const int64_t total = (int64_t)n * h * w * s * s * C;
  pixel_shuffle_f32_kernel<<<grid_for(total, 256, device_sm_count() * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, ld_in, out, ld_out, n, h, w, C, s);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_bilinear_align_corners(const void* in, void* out, int n, int Hin, int Win, int C, int Hv, int Wv, int Ho,
                                         int Wo, void* stream) {
  MA_REQUIRE(in && out && n > 0 && C % 8 == 0 && Ho <= Hv && Wo <= Wv && Hin > 0 && Win > 0, "ma_bilinear_align_corners: bad arguments");
  MA_REQUIRE((int64_t)n * Ho < (1ll << 31), "ma_bilinear_align_corners: too many output rows");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0, "ma_bilinear_align_corners: in not 16-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "ma_bilinear_align_corners: out not 16-byte aligned");
  bilinear_ac_kernel<<<n * Ho, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in), static_cast<__nv_bfloat16*>(out), n, Hin, Win, C, Hv, Wv, Ho, Wo);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_token_mean(const void* in, void* out, int n, int T, int C, void* stream) {
  MA_REQUIRE(in && out && n > 0 && T > 0 && C > 0, "ma_token_mean: bad arguments");
  dim3 grid((C + 63) / 64, n);
  token_mean_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(in),
                                                                         static_cast<__nv_bfloat16*>(out), T, C);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_head_linear_small(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias, float* out,
                                    int64_t ldo, int64_t rows, int N, int K, void* stream) {
  MA_REQUIRE(x && w && out && rows > 0, "ma_head_linear_small: null pointer");
  MA_REQUIRE(N >= 1 && N <= 8 && K >= 8 && K <= 256 && K % 8 == 0 && ldx % 8 == 0 && ldo >= N,
             "ma_head_linear_small: needs N <= 8, K <= 256, K %% 8 == 0 (N=%d K=%d)", N, K);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "ma_head_linear_small: x not 16-byte aligned");
  MA_REQUIRE(ldx >= K, "ma_head_linear_small: ldx (%lld) below K = %d", (long long)ldx, K);
  MA_REQUIRE(ldw >= K, "ma_head_linear_small: ldw (%lld) below K = %d", (long long)ldw, K);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* wb = static_cast<const __nv_bfloat16*>(w);
  const int lpr = K / 8;
  if (lpr >= 8 && lpr <= 32 && (lpr & (lpr - 1)) == 0) {
    const int rpw = 32 / lpr;
    const unsigned grid = grid_for((rows + 4 * rpw - 1) / (4 * rpw) * 32, 256, device_sm_count() * 8);
    if (lpr == 8) head_linear_small_warp_kernel<8><<<grid, 256, 0, st>>>(xb, ldx, wb, ldw, bias, out, ldo, rows, N);
    else if (lpr == 16) head_linear_small_warp_kernel<16><<<grid, 256, 0, st>>>(xb, ldx, wb, ldw, bias, out, ldo, rows, N);
    else head_linear_small_warp_kernel<32><<<grid, 256, 0, st>>>(xb, ldx, wb, ldw, bias, out, ldo, rows, N);
  } else {
    head_linear_small_kernel<<<grid_for(rows, 128, device_sm_count() * 16), 128, 0, st>>>(xb, ldx, wb, ldw, bias, out, ldo, rows, N, K);
  }
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_split_bf16x3(const float* in, int64_t ld_in, void* out, int rows, int C, void* stream) {
  MA_REQUIRE(in && out && rows > 0 && C > 0 && C % 4 == 0 && ld_in % 4 == 0, "ma_split_bf16x3: bad arguments (C=%d)", C);
  MA_REQUIRE(ld_in >= C, "ma_split_bf16x3: ld_in (%lld) below C = %d", (long long)ld_in, C);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0, "ma_split_bf16x3: in not 16-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 7) == 0, "ma_split_bf16x3: out not 8-byte aligned");
  const int64_t total = (int64_t)rows * (C / 4);
  split_bf16x3_kernel<<<grid_for(total, 256, device_sm_count() * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, ld_in, static_cast<__nv_bfloat16*>(out), rows, C);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_token_mean_f32(const float* in, float* out, int n, int T, int C, void* stream) {
  MA_REQUIRE(in && out && n > 0 && T > 0 && C > 0, "ma_token_mean_f32: bad arguments");
  dim3 grid((C + 63) / 64, n);
  token_mean_f32_kernel<<<grid, 1024, 0, static_cast<cudaStream_t>(stream)>>>(in, out, T, C);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_linear_rows_f32(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* bias, int act, float* out,
                                  int64_t ldo, int rows, int N, int K, void* stream) {
  MA_REQUIRE(x && w && out && rows >= 1 && rows <= LIN_ROWS_MAX && N >= 1 && K >= 4 && K % 4 == 0 && ldx % 4 == 0 && ldw % 4 == 0 &&
                 ldo >= N, "ma_linear_rows_f32: needs 1 <= rows <= %d, K %% 4 == 0, strides %% 4 == 0 (rows=%d N=%d K=%d)",
             LIN_ROWS_MAX, rows, N, K);
  MA_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w)) & 15) == 0, "ma_linear_rows_f32: x / w not 16-byte aligned");
  MA_REQUIRE(ldx >= K, "ma_linear_rows_f32: ldx (%lld) below K = %d", (long long)ldx, K);
  MA_REQUIRE(ldw >= K, "ma_linear_rows_f32: ldw (%lld) below K = %d", (long long)ldw, K);
  MA_REQUIRE(act == MA_ACT_NONE || act == MA_ACT_RELU || act == MA_ACT_GELU, "ma_linear_rows_f32: bad activation %d", act);
  const size_t smem = (size_t)rows * K * sizeof(float);
  MA_REQUIRE(smem <= 48 * 1024, "ma_linear_rows_f32: rows * K = %d floats do not fit 48 KB of shared memory", rows * K);
  linear_rows_f32_kernel<<<(N + 7) / 8, 256, smem, static_cast<cudaStream_t>(stream)>>>(x, ldx, w, ldw, bias, out, ldo, rows, N, K, act);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_decode_dense(const float* raw, int ld_raw, const float* pose_raw, const float* scale_raw, int n, int HW,
                               float* pts3d, float* pts3d_cam, float* rays, float* depth, float* conf, float* logits,
                               uint8_t* mask, float* cam_trans, float* cam_quats, float* scale_out, void* stream) {
  MA_REQUIRE(raw && pose_raw && scale_raw && pts3d && pts3d_cam && rays && depth && conf && logits && mask && cam_trans &&
                 cam_quats && scale_out && n > 0 && HW > 0 && ld_raw >= 6,
             "ma_decode_dense: bad arguments");
  MA_REQUIRE(ld_raw % 4 != 0 || (reinterpret_cast<uintptr_t>(raw) & 15) == 0,
             "ma_decode_dense: raw not 16-byte aligned (ld_raw %% 4 == 0 takes the float4 loads)");
  DecodeParams p{raw, ld_raw, pose_raw, scale_raw, pts3d, pts3d_cam, rays, depth, conf, logits, mask, cam_trans, cam_quats,
                 scale_out, n, HW};
  dim3 grid(grid_for(HW, 256, 1024), n);
  decode_dense_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_decode_scene(const ma_decode_spec* spec, const float* raw, int ld_raw, const float* pose_raw,
                               const float* scale_raw, int n, int HW, float* pts3d, float* pts3d_cam, float* rays,
                               float* ray_origins, float* depth, float* conf, float* logits, uint8_t* mask, float* cam_trans,
                               float* cam_quats, float* scale_out, void* stream) {
  MA_REQUIRE(spec && raw && scale_raw && pts3d && scale_out && n > 0 && HW > 0, "ma_decode_scene: bad arguments");
  const int rep = spec->rep;
  MA_REQUIRE(rep >= MA_REP_POINTMAP && rep <= MA_REP_POINTMAP_RAYDIRS_DEPTH_POSE, "ma_decode_scene: unknown representation %d", rep);
  MA_REQUIRE(spec->point_mode >= MA_PTS_LINEAR && spec->point_mode <= MA_PTS_Z_EXP, "ma_decode_scene: unknown point_mode %d",
             spec->point_mode);
  const bool posed = rep >= MA_REP_RAYDIRS_DEPTH_POSE;
  const int rep_ch = rep == MA_REP_POINTMAP || rep == MA_REP_CAMPOINTMAP_POSE ? 3 : rep == MA_REP_RAYDIRS_DEPTH_POSE ? 4 : 7;
  MA_REQUIRE(ld_raw >= rep_ch + (spec->has_conf ? 1 : 0) + (spec->has_mask ? 1 : 0), "ma_decode_scene: ld_raw %d too small", ld_raw);
  MA_REQUIRE(posed == (pose_raw != nullptr) && posed == (cam_trans != nullptr) && posed == (cam_quats != nullptr) &&
                 posed == (pts3d_cam != nullptr),
             "ma_decode_scene: pose_raw / cam_trans / cam_quats / pts3d_cam are given exactly for the posed representations");
  MA_REQUIRE((rep == MA_REP_RAYMAP_DEPTH) == (ray_origins != nullptr), "ma_decode_scene: ray_origins is for MA_REP_RAYMAP_DEPTH");
  MA_REQUIRE((rep != MA_REP_POINTMAP) == (rays != nullptr) && (rep != MA_REP_POINTMAP) == (depth != nullptr),
             "ma_decode_scene: rays / depth are given for every representation but MA_REP_POINTMAP");
  MA_REQUIRE((spec->has_conf != 0) == (conf != nullptr), "ma_decode_scene: conf pointer vs has_conf");
  MA_REQUIRE((spec->has_mask != 0) == (logits != nullptr) && (spec->has_mask != 0) == (mask != nullptr),
             "ma_decode_scene: logits / mask pointers vs has_mask");
  DecodeSceneParams p{*spec, raw, ld_raw, pose_raw, scale_raw, pts3d, pts3d_cam, rays, ray_origins, depth, conf, logits, mask,
                      cam_trans, cam_quats, scale_out, n, HW};
  dim3 grid(grid_for(HW, 256, 1024), n);
  decode_scene_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
