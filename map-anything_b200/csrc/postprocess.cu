// infer() post-processing on the GPU: the reference does this per view in numpy on the host
// (mapanything/utils/inference.py:294-480, 0.42 s per 518x518 view measured in SURVEY.md F6) -- here it is
// four small HBM-bound kernels per scene.
//
// The edge-mask kernels reproduce numpy's float32 arithmetic operation by operation (separate multiply /
// add roundings via __fmul_rn/__fadd_rn/__fsub_rn so nvcc cannot contract them into FMAs, sequential
// ((a+b)+c) reductions, IEEE sqrt/div, NaN propagation of np.max vs NaN skipping of np.nanmax) because their
// OUTPUT IS BOOLEAN: any rounding difference can flip a pixel.  Reference functions:
//   points_to_normals geometry.py:1717-1780, normals_edge :2129-2188 (including its transposed mask window),
//   depth_edge :2031-2072, max_pool_2d :1905-2028, mask combination inference.py:418-476.
// The one exception is the neighbour angle: CUDA's acosf can differ from numpy's float32 arccos by a few ulp, so a pixel
// whose pooled angle lies within that distance of the threshold can differ from numpy.
#include <math_constants.h>

#include "host_common.h"
#include "ptx.cuh"

namespace ma {

// ---------------------------------------------------------------------------------------------
// img_no_norm = clip(img * std + mean, 0, 1), NCHW -> NHWC   (image.py:93-131 rgb())
// ---------------------------------------------------------------------------------------------
__global__ void denorm_image_kernel(const float* __restrict__ img, float* __restrict__ out, int HW, float m0, float m1,
                                    float m2, float s0, float s1, float s2) {
  const int i = blockIdx.y;
  const float* src = img + (size_t)i * 3 * HW;
  float* dst = out + (size_t)i * 3 * HW;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x) {
    const float r = __fadd_rn(__fmul_rn(src[p], s0), m0);
    const float g = __fadd_rn(__fmul_rn(src[HW + p], s1), m1);
    const float b = __fadd_rn(__fmul_rn(src[2 * HW + p], s2), m2);
    dst[3 * p + 0] = fminf(fmaxf(r, 0.f), 1.f);
    dst[3 * p + 1] = fminf(fmaxf(g, 0.f), 1.f);
    dst[3 * p + 2] = fminf(fmaxf(b, 0.f), 1.f);
  }
}

// ---------------------------------------------------------------------------------------------
// pinhole intrinsics from unit ray directions (geometry.py:304-447): one block per view.
// ---------------------------------------------------------------------------------------------
__global__ void intrinsics_from_rays_kernel(const float* __restrict__ rays, float* __restrict__ K, int H, int W) {
  const float* r = rays + (size_t)blockIdx.x * H * W * 3;
  float* k = K + blockIdx.x * 9;
  if ((long long)H * W > 1000000) {
    if (threadIdx.x == 0) {
      const int ch = H / 2, cw = W / 2, qw = W / 4, tqw = 3 * W / 4, qh = H / 4, tqh = 3 * H / 4;
      auto at = [&](int y, int x, float& rx, float& ry) {
        const float* p = r + ((size_t)y * W + x) * 3;
        rx = p[0] / p[2];
        ry = p[1] / p[2];
      };
      float cx_, cy_, lx, ly, rx, ry, tx, ty, bx, by;
      at(ch, cw, cx_, cy_);
      at(ch, qw, lx, ly);
      at(ch, tqw, rx, ry);
      at(qh, cw, tx, ty);
      at(tqh, cw, bx, by);
      const float fx = ((qw - cw) / (lx - cx_) + (tqw - cw) / (rx - cx_)) / 2;
      const float fy = ((qh - ch) / (ty - cy_) + (tqh - ch) / (by - cy_)) / 2;
      k[0] = fx; k[1] = 0; k[2] = cw - fx * cx_;
      k[3] = 0; k[4] = fy; k[5] = ch - fy * cy_;
      k[6] = 0; k[7] = 0; k[8] = 1;
    }
    return;
  }
  const int sh = max(1, H / 50), sw = max(1, W / 50);
  const int nh = (H + sh - 1) / sh, nw = (W + sw - 1) / sw;
  // normal equations of x = cx + fx*(dx/dz), y = cy + fy*(dy/dz), accumulated in double
  double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // n, Srx, Srx2, Sx, Srx*x, Sry, Sry2, (Sy, Sry*y packed below)
  double sy_ = 0, sryy = 0;
  for (int idx = threadIdx.x; idx < nh * nw; idx += blockDim.x) {
    const int y = (idx / nw) * sh, x = (idx % nw) * sw;
    const float* p = r + ((size_t)y * W + x) * 3;
    const double rx = (double)(p[0] / p[2]), ry = (double)(p[1] / p[2]);
    s[0] += 1.0; s[1] += rx; s[2] += rx * rx; s[3] += x; s[4] += rx * x;
    s[5] += ry; s[6] += ry * ry; sy_ += y; sryy += ry * y;
  }
  __shared__ double red[10][32];
  double vals[10] = {s[0], s[1], s[2], s[3], s[4], s[5], s[6], sy_, sryy, 0};
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    double v = vals[j];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffff, v, o);
    if ((threadIdx.x & 31) == 0) red[j][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t[9];
    for (int j = 0; j < 9; ++j) {
      t[j] = 0;
      for (int w = 0; w < (blockDim.x >> 5); ++w) t[j] += red[j][w];
    }
    const double n = t[0];
    const double detx = n * t[2] - t[1] * t[1];
    const double cx = (t[3] * t[2] - t[1] * t[4]) / detx, fx = (n * t[4] - t[1] * t[3]) / detx;
    const double dety = n * t[6] - t[5] * t[5];
    const double cy = (t[7] * t[6] - t[5] * t[8]) / dety, fy = (n * t[8] - t[5] * t[7]) / dety;
    k[0] = (float)fx; k[1] = 0; k[2] = (float)cx;
    k[3] = 0; k[4] = (float)fy; k[5] = (float)cy;
    k[6] = 0; k[7] = 0; k[8] = 1;
  }
}

// ---------------------------------------------------------------------------------------------
// 4x4 cam2world matrices from (unit) quaternions + translations (inference.py:364-379, geometry.py:601-652)
// ---------------------------------------------------------------------------------------------
__global__ void pose_matrix_kernel(const float* __restrict__ quats, const float* __restrict__ trans, float* __restrict__ out,
                                   int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x = quats[4 * i], y = quats[4 * i + 1], z = quats[4 * i + 2], w = quats[4 * i + 3];
  const float inv = 1.0f / sqrtf(x * x + y * y + z * z + w * w);
  x *= inv; y *= inv; z *= inv; w *= inv;
  float* m = out + 16 * i;
  m[0] = 1 - 2 * (y * y + z * z); m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y); m[3] = trans[3 * i];
  m[4] = 2 * (x * y + w * z); m[5] = 1 - 2 * (x * x + z * z); m[6] = 2 * (y * z - w * x); m[7] = trans[3 * i + 1];
  m[8] = 2 * (x * z - w * y); m[9] = 2 * (y * z + w * x); m[10] = 1 - 2 * (x * x + y * y); m[11] = trans[3 * i + 2];
  m[12] = 0; m[13] = 0; m[14] = 0; m[15] = 1;
}

// ---------------------------------------------------------------------------------------------
// edge masks
// ---------------------------------------------------------------------------------------------
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 sub3(V3 a, V3 b) { return {__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)}; }
// np.cross on the last axis: c0 = a1*b2 - a2*b1, c1 = a2*b0 - a0*b2, c2 = a0*b1 - a1*b0 (products rounded separately)
__device__ __forceinline__ V3 cross3(V3 a, V3 b) {
  return {__fsub_rn(__fmul_rn(a.y, b.z), __fmul_rn(a.z, b.y)), __fsub_rn(__fmul_rn(a.z, b.x), __fmul_rn(a.x, b.z)),
          __fsub_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x))};
}
// x / (np.linalg.norm(x) + 1e-12) in float32
__device__ __forceinline__ V3 normalize_np(V3 v) {
  const float ss = __fadd_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)), __fmul_rn(v.z, v.z));
  const float d = __fadd_rn(__fsqrt_rn(ss), 1e-12f);
  return {__fdiv_rn(v.x, d), __fdiv_rn(v.y, d), __fdiv_rn(v.z, d)};
}

// pass A: normals (H,W,3) + normal_mask from the point map and the validity mask (zero / False padded).
__global__ void edge_normals_kernel(const float* __restrict__ pts, const uint8_t* __restrict__ mask, float* __restrict__ normals,
                                    uint8_t* __restrict__ nmask, int H, int W) {
  const int view = blockIdx.y;
  pts += (size_t)view * H * W * 3;
  mask += (size_t)view * H * W;
  normals += (size_t)view * H * W * 3;
  nmask += (size_t)view * H * W;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < H * W; p += gridDim.x * blockDim.x) {
    const int y = p / W, x = p - y * W;
    auto P = [&](int yy, int xx) -> V3 {
      if (yy < 0 || yy >= H || xx < 0 || xx >= W) return {0.f, 0.f, 0.f};
      const float* q = pts + ((size_t)yy * W + xx) * 3;
      return {q[0], q[1], q[2]};
    };
    auto M = [&](int yy, int xx) -> bool { return yy >= 0 && yy < H && xx >= 0 && xx < W && mask[(size_t)yy * W + xx] != 0; };
    const V3 c = P(y, x);
    const V3 up = sub3(P(y - 1, x), c), left = sub3(P(y, x - 1), c), down = sub3(P(y + 1, x), c), right = sub3(P(y, x + 1), c);
    const V3 n0 = normalize_np(cross3(up, left)), n1 = normalize_np(cross3(left, down));
    const V3 n2 = normalize_np(cross3(down, right)), n3 = normalize_np(cross3(right, up));
    const bool mc = M(y, x), mu = M(y - 1, x), ml = M(y, x - 1), md = M(y + 1, x), mr = M(y, x + 1);
    const float v0 = (mu && ml && mc) ? 1.f : 0.f, v1 = (ml && md && mc) ? 1.f : 0.f;
    const float v2 = (md && mr && mc) ? 1.f : 0.f, v3 = (mr && mu && mc) ? 1.f : 0.f;
    V3 s;
    s.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(n0.x, v0), __fmul_rn(n1.x, v1)), __fmul_rn(n2.x, v2)), __fmul_rn(n3.x, v3));
    s.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(n0.y, v0), __fmul_rn(n1.y, v1)), __fmul_rn(n2.y, v2)), __fmul_rn(n3.y, v3));
    s.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(n0.z, v0), __fmul_rn(n1.z, v1)), __fmul_rn(n2.z, v2)), __fmul_rn(n3.z, v3));
    s = normalize_np(s);
    const bool any = (v0 + v1 + v2 + v3) > 0.f;
    if (!any) s = {0.f, 0.f, 0.f};
    normals[3 * (size_t)p + 0] = s.x; normals[3 * (size_t)p + 1] = s.y; normals[3 * (size_t)p + 2] = s.z;
    nmask[p] = any ? 1 : 0;
  }
}

// pass B: per pixel, max angle to the (edge padded) 3x3 neighbours gated by the reference's transposed mask
// window, with np.max NaN propagation; plus the depth edge.
__global__ void edge_angle_depth_kernel(const float* __restrict__ normals, const uint8_t* __restrict__ nmask,
                                        const float* __restrict__ depth, int depth_stride, const uint8_t* __restrict__ mask,
                                        float* __restrict__ angle, uint8_t* __restrict__ depth_edge, int H, int W, float rtol) {
  const int view = blockIdx.y;
  normals += (size_t)view * H * W * 3;
  nmask += (size_t)view * H * W;
  mask += (size_t)view * H * W;
  depth += (size_t)view * H * W * depth_stride;
  angle += (size_t)view * H * W;
  depth_edge += (size_t)view * H * W;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < H * W; p += gridDim.x * blockDim.x) {
    const int y = p / W, x = p - y * W;
    auto N = [&](int yy, int xx) -> V3 {
      yy = min(max(yy, 0), H - 1);
      xx = min(max(xx, 0), W - 1);
      const float* q = normals + ((size_t)yy * W + xx) * 3;
      return normalize_np({q[0], q[1], q[2]});
    };
    auto NM = [&](int yy, int xx) -> bool {
      yy = min(max(yy, 0), H - 1);
      xx = min(max(xx, 0), W - 1);
      return nmask[(size_t)yy * W + xx] != 0;
    };
    const V3 c = N(y, x);
    float amax = 0.f;
    bool nan = false;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        // angle to neighbour (dy,dx) is gated by the validity of neighbour (dx,dy) -- reference quirk, see oracle
        if (!NM(y + dx - 1, x + dy - 1)) continue;
        const V3 nb = N(y + dy - 1, x + dx - 1);
        const float dot = __fadd_rn(__fadd_rn(__fmul_rn(c.x, nb.x), __fmul_rn(c.y, nb.y)), __fmul_rn(c.z, nb.z));
        const float a = acosf(dot);
        if (a != a) nan = true;
        else amax = fmaxf(amax, a);
      }
    }
    angle[p] = nan ? CUDART_NAN_F : amax;

    // depth edge: (max - min over valid in-bounds 3x3) / depth > rtol, with -inf for invalid pixels
    float dmax = -CUDART_INF_F, nmin = -CUDART_INF_F;  // nmin = max of (-depth)
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        const int yy = y + dy, xx = x + dx;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;  // NaN padding is skipped by nanmax
        const bool m = mask[(size_t)yy * W + xx] != 0;
        const float d = depth[((size_t)yy * W + xx) * depth_stride];
        const float a = m ? d : -CUDART_INF_F, b = m ? -d : -CUDART_INF_F;
        // np.nanmax skips NaN inputs
        if (a == a) dmax = fmaxf(dmax, a);
        if (b == b) nmin = fmaxf(nmin, b);
      }
    const float diff = __fadd_rn(dmax, nmin);
    const float dc = depth[(size_t)p * depth_stride];
    depth_edge[p] = (__fdiv_rn(diff, dc) > rtol) ? 1 : 0;
  }
}

// pass C: 3x3 nanmax pool of the angle map -> normal edge; final = mask & ~(depth_edge & normal_edge)
__global__ void edge_combine_kernel(const float* __restrict__ angle, const uint8_t* __restrict__ depth_edge,
                                    const uint8_t* __restrict__ mask, uint8_t* __restrict__ out, int H, int W, double tol_rad) {
  const int view = blockIdx.y;
  angle += (size_t)view * H * W;
  depth_edge += (size_t)view * H * W;
  mask += (size_t)view * H * W;
  out += (size_t)view * H * W;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < H * W; p += gridDim.x * blockDim.x) {
    const int y = p / W, x = p - y * W;
    float m = 0.f;
    bool have = false;
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        const int yy = y + dy, xx = x + dx;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
        const float a = angle[(size_t)yy * W + xx];
        if (a == a) {
          m = have ? fmaxf(m, a) : a;
          have = true;
        }
      }
    const bool nedge = have && (static_cast<double>(m) > tol_rad);  // all-NaN window -> NaN > tol is False
    out[p] = (mask[p] != 0 && !(depth_edge[p] != 0 && nedge)) ? 1 : 0;
  }
}

// out[i] = in[i] * mask[i / width]  (dense geometry zeroing, inference.py:457-476).  width = channels per pixel.
__global__ void apply_mask_kernel(const float* __restrict__ in, int in_stride, int in_offset, const uint8_t* __restrict__ mask,
                                  float* __restrict__ out, int64_t pixels, int width) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pixels * width; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t px = i / width;
    const int c = static_cast<int>(i - px * width);
    out[i] = __fmul_rn(in[px * in_stride + in_offset + c], mask[px] ? 1.f : 0.f);
  }
}

// out = a & b (bool bytes)
__global__ void mask_and_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint8_t* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (a[i] != 0 && b[i] != 0) ? 1 : 0;
}


// ----------------------------------------------------------------------------------------------
// Per-image confidence quantile mask (reference inference.py:393-415): thr = torch.quantile(conf, q) with linear
// interpolation, mask = conf > thr.  One block per image: exact order statistics by a 4 x 8-bit radix select over the
// order-preserving integer image of the floats (no sort), then torch's lerp in float32, each branch one FMA rounding as
// in ATen's lerp:
//   rank = q * (n - 1) (float32), lo = floor(rank), w = rank - lo,
//   thr = w < 0.5 ? fma(w, b - a, a) : fma(w - 1, b - a, b)      with a, b = the lo-th / ceil(rank)-th smallest values
// (w - 1 is exact for w in [0.5, 1)).  As in torch.quantile, an image holding a NaN gets a NaN threshold (an all-False
// mask).
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t float_to_ordered(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__global__ void quantile_mask_kernel(const float* __restrict__ conf, uint8_t* __restrict__ mask, float* __restrict__ thr_out,
                                     int64_t per_image, float q) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_prefix, s_k, s_next, s_cnt_le, s_nan;
  const float* x = conf + (int64_t)blockIdx.x * per_image;
  const float rank = q * static_cast<float>(per_image - 1);  // float32 like torch (q and n - 1 as float32 tensors)
  const float lo_f = floorf(rank);
  const float w = rank - lo_f;
  const uint32_t k_lo = static_cast<uint32_t>(lo_f);
  const bool need_hi = ceilf(rank) != lo_f;

  if (threadIdx.x == 0) { s_prefix = 0u; s_k = k_lo; s_nan = 0u; }
  __syncthreads();
  uint32_t less_total = 0;  // (thread 0) number of elements strictly below the selected value so far
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    const uint32_t pmask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
    for (int64_t i = threadIdx.x; i < per_image; i += blockDim.x) {
      const float xi = x[i];
      if (pass == 0 && xi != xi) s_nan = 1u;
      const uint32_t u = float_to_ordered(xi);
      if ((u & pmask) == prefix) atomicAdd(&hist[(u >> shift) & 0xffu], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t k = s_k, acc = 0;
      int b = 0;
      for (; b < 256; ++b) {
        if (acc + hist[b] > k) break;
        acc += hist[b];
      }
      s_k = k - acc;
      less_total += acc;
      s_prefix = prefix | (static_cast<uint32_t>(b) << shift);
      if (pass == 3) s_cnt_le = less_total + hist[b];  // elements <= selected value
    }
    __syncthreads();
  }
  const uint32_t v_lo = s_prefix;
  float a = ordered_to_float(v_lo), b = a;
  if (need_hi) {
    if (k_lo + 1 >= s_cnt_le) {  // the next order statistic is the smallest value above v_lo
      if (threadIdx.x == 0) s_next = 0xffffffffu;
      __syncthreads();
      uint32_t mn = 0xffffffffu;
      for (int64_t i = threadIdx.x; i < per_image; i += blockDim.x) {
        const uint32_t u = float_to_ordered(x[i]);
        if (u > v_lo && u < mn) mn = u;
      }
      atomicMin(&s_next, mn);
      __syncthreads();
      b = ordered_to_float(s_next);
    }
  }
  const float diff = b - a;
  const float thr = s_nan ? CUDART_NAN_F : w < 0.5f ? __fmaf_rn(w, diff, a) : __fmaf_rn(w - 1.0f, diff, b);
  if (threadIdx.x == 0 && thr_out) thr_out[blockIdx.x] = thr;
  uint8_t* m = mask + (int64_t)blockIdx.x * per_image;
  for (int64_t i = threadIdx.x; i < per_image; i += blockDim.x) m[i] = x[i] > thr ? 1 : 0;
}

// depthmap_to_camera_frame / depthmap_to_world_frame (geometry.py:18-114): one thread per pixel.  The camera-frame point
// uses the reference's operation order ((x - cx) * z) / fx with IEEE roundings (bit-exact); the optional cam2world
// transform is the 3x4 part of the homogeneous product.
__global__ void depthmap_to_world_kernel(const float* __restrict__ depth, const float* __restrict__ K, const float* __restrict__ pose,
                                         float* __restrict__ pts, uint8_t* __restrict__ valid, int H, int W) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const float* k = K + b * 9;
  const float fx = k[0], fy = k[4], cx = k[2], cy = k[5];
  const float z = depth[static_cast<int64_t>(b) * H * W + i];
  const float xg = static_cast<float>(i % W), yg = static_cast<float>(i / W);
  float x = __fdiv_rn(__fmul_rn(__fsub_rn(xg, cx), z), fx);
  float y = __fdiv_rn(__fmul_rn(__fsub_rn(yg, cy), z), fy);
  float zz = z;
  if (pose) {
    const float* p = pose + b * 16;
    const float wx = p[0] * x + p[1] * y + p[2] * z + p[3];
    const float wy = p[4] * x + p[5] * y + p[6] * z + p[7];
    const float wz = p[8] * x + p[9] * y + p[10] * z + p[11];
    x = wx;
    y = wy;
    zz = wz;
  }
  float* o = pts + (static_cast<int64_t>(b) * H * W + i) * 3;
  o[0] = x;
  o[1] = y;
  o[2] = zz;
  if (valid) valid[static_cast<int64_t>(b) * H * W + i] = z > 0.0f ? 1 : 0;
}

}  // namespace ma

using namespace ma;

extern "C" int ma_depthmap_to_world(const float* depth, const float* K, const float* pose, float* pts, uint8_t* valid, int n,
                                    int H, int W, void* stream) {
  MA_REQUIRE(depth && K && pts && n > 0 && H > 0 && W > 0, "ma_depthmap_to_world: bad arguments");
  dim3 grid((H * W + 255) / 256, n);
  depthmap_to_world_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(depth, K, pose, pts, valid, H, W);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_denorm_image(const float* img, float* out, int n, int H, int W, const float* mean_host, const float* std_host,
                               void* stream) {
  MA_REQUIRE(img && out && mean_host && std_host && n > 0 && H > 0 && W > 0, "ma_denorm_image: bad arguments");
  dim3 grid((H * W + 255) / 256 > 1024 ? 1024 : (H * W + 255) / 256, n);
  denorm_image_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(img, out, H * W, mean_host[0], mean_host[1],
                                                                           mean_host[2], std_host[0], std_host[1], std_host[2]);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_intrinsics_from_rays(const float* rays, float* K, int n, int H, int W, void* stream) {
  MA_REQUIRE(rays && K && n > 0 && H > 0 && W > 0, "ma_intrinsics_from_rays: bad arguments");
  intrinsics_from_rays_kernel<<<n, 256, 0, static_cast<cudaStream_t>(stream)>>>(rays, K, H, W);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_pose_matrices(const float* quats, const float* trans, float* out, int n, void* stream) {
  MA_REQUIRE(quats && trans && out && n > 0, "ma_pose_matrices: bad arguments");
  pose_matrix_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(quats, trans, out, n);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_edge_mask(const float* pts3d, const float* depth_z, int depth_stride, const uint8_t* mask_in, uint8_t* mask_out,
                            float* ws_normals, uint8_t* ws_nmask, float* ws_angle, uint8_t* ws_depth_edge, int n, int H, int W,
                            float normal_tol_deg, float depth_rtol, void* stream) {
  MA_REQUIRE(pts3d && depth_z && mask_in && mask_out && ws_normals && ws_nmask && ws_angle && ws_depth_edge && n > 0 && H > 0 &&
                 W > 0 && depth_stride > 0,
             "ma_edge_mask: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int gx = (H * W + 255) / 256 > 2048 ? 2048 : (H * W + 255) / 256;
  dim3 grid(gx, n);
  edge_normals_kernel<<<grid, 256, 0, s>>>(pts3d, mask_in, ws_normals, ws_nmask, H, W);
  edge_angle_depth_kernel<<<grid, 256, 0, s>>>(ws_normals, ws_nmask, depth_z, depth_stride, mask_in, ws_angle, ws_depth_edge, H,
                                               W, depth_rtol);
  // np.deg2rad(tol) returns a float64 NumPy scalar (not a weak Python float), so `angle > tol` promotes the
  // float32 angles to float64: compare in double.
  const double tol_rad = static_cast<double>(normal_tol_deg) * (3.14159265358979323846 / 180.0);
  edge_combine_kernel<<<grid, 256, 0, s>>>(ws_angle, ws_depth_edge, mask_in, mask_out, H, W, tol_rad);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_apply_mask(const float* in, int in_stride, int in_offset, const uint8_t* mask, float* out, int64_t pixels,
                             int width, void* stream) {
  MA_REQUIRE(in && mask && out && pixels > 0 && width > 0 && in_stride >= width, "ma_apply_mask: bad arguments");
  MA_REQUIRE(in_offset >= 0 && in_offset <= in_stride - width,
             "ma_apply_mask: in_offset %d + width %d must lie in [0, in_stride %d]", in_offset, width, in_stride);
  const int64_t total = pixels * width;
  const int grid = static_cast<int>((total + 255) / 256 > 148 * 16 ? 148 * 16 : (total + 255) / 256);
  apply_mask_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(in, in_stride, in_offset, mask, out, pixels, width);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_mask_and(const uint8_t* a, const uint8_t* b, uint8_t* out, int64_t n, void* stream) {
  MA_REQUIRE(a && b && out && n > 0, "ma_mask_and: bad arguments");
  const int grid = static_cast<int>((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256);
  mask_and_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a, b, out, n);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_quantile_mask(const float* conf, uint8_t* mask, float* thr_out, int n, int64_t per_image, float q, void* stream) {
  using namespace ma;
  MA_REQUIRE(conf && mask && n > 0 && per_image > 0 && per_image < (1ll << 31), "ma_quantile_mask: bad arguments");
  MA_REQUIRE(q >= 0.f && q <= 1.f, "ma_quantile_mask: q must be in [0, 1], got %f", (double)q);
  quantile_mask_kernel<<<n, 1024, 0, static_cast<cudaStream_t>(stream)>>>(conf, mask, thr_out, per_image, q);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
