// Geometric-input side of the hot path (SURVEY 8a rows a8-a11): the small fp32 preparation steps around the encoders
// of ray directions / depth / camera pose, which the reference runs as chains of PyTorch elementwise ops with autocast
// disabled (model.py:647-1131).  The encoders themselves are ma_conv3x3_bf16 / ma_gemm_bf16 launches.
#include "host_common.h"
#include "ptx.cuh"

namespace ma {

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffff, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = 0.f;
  const int nw = (blockDim.x + 31) >> 5;
  for (int i = 0; i < nw; ++i) t += red[i];
  return t;
}

// ----------------------------------------------------------------------------------------------
// PixelUnshuffle(p) of an NHWC fp32 map (n,H,W,cin) + optional depth normalisation, emitted as the split-bf16
// activation layout [hi | lo | hi] (see ma_split_bf16x3) of an NHWC token map (n, H/p, W/p, 3*cpad):
//   channel k = c*p*p + dy*p + dx  (nn.PixelUnshuffle on the NCHW tensor the reference builds, model.py:803-811),
//   zero padded to cpad (multiple of 8, TMA alignment).
// mode 1 (depth, model.py:946-971): v = v / factor[i];  v = v/max(|v|,1e-8) * log1p(|v|)   (geometry.py:1666-1679)
// ----------------------------------------------------------------------------------------------
__global__ void unshuffle_split_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int H, int W, int cin,
                                       int hp, int wp, int p, int cpad, int mode, const float* __restrict__ factor) {
  const int tok = blockIdx.x;
  const int i = tok / (hp * wp);
  const int rem = tok - i * hp * wp;
  const int py = rem / wp, px = rem - py * wp;
  const int kk = cin * p * p;
  const float inv_f = mode == 1 ? 1.0f / factor[i] : 1.0f;
  __nv_bfloat16* o = out + (size_t)tok * 3 * cpad;
  for (int k = threadIdx.x; k < cpad; k += blockDim.x) {
    float v = 0.f;
    if (k < kk) {
      const int c = k / (p * p);
      const int r = k - c * p * p;
      const int dy = r / p, dx = r - dy * p;
      v = __ldg(in + (((size_t)i * H + py * p + dy) * W + px * p + dx) * cin + c);
      if (mode == 1) {
        v = v * inv_f;
        const float a = fabsf(v);
        v = v / fmaxf(a, 1e-8f) * log1pf(a);
      }
    }
    const __nv_bfloat16 hi = __float2bfloat16(v);
    const __nv_bfloat16 lo = __float2bfloat16(v - __bfloat162float(hi));
    o[k] = hi;
    o[cpad + k] = lo;
    o[2 * cpad + k] = hi;
  }
}

// ----------------------------------------------------------------------------------------------
// normalize_depth_using_non_zero_pixels (geometry.py:1523-1555): factor[i] = sum(d > 0 ? d : 0) / (count(d > 0) + 1e-8),
// clipped at 1e-8; log_factor[i][0] = log(factor + 1e-8), padded to 8 columns (K of the scale-encoder GEMM).
// ----------------------------------------------------------------------------------------------
__global__ void depth_factor_kernel(const float* __restrict__ depth, int64_t per_view, float* __restrict__ factor,
                                    float* __restrict__ log_factor8) {
  __shared__ float red[32];
  const float* d = depth + (int64_t)blockIdx.x * per_view;
  float s = 0.f, c = 0.f;
  for (int64_t j = threadIdx.x; j < per_view; j += blockDim.x) {
    const float v = d[j];
    if (v > 0.f) { s += v; c += 1.f; }
  }
  s = block_sum(s, red);
  c = block_sum(c, red);
  if (threadIdx.x == 0) {
    const float f = fmaxf(s / (c + 1e-8f), 1e-8f);
    factor[blockIdx.x] = f;
    float* o = log_factor8 + (int64_t)blockIdx.x * 8;
    o[0] = logf(f + 1e-8f);
#pragma unroll
    for (int j = 1; j < 8; ++j) o[j] = 0.f;
  }
}

// ----------------------------------------------------------------------------------------------
// Camera-pose inputs (model.py:647-751, :1012-1131): poses relative to view 0
//   q_rel = q0^-1 (x) q_v,  t_rel = R(q0^-1) (t_v - t0)          (geometry.py:814-852)
// identity / zero for views without a pose; translations divided by the mean norm of the non-zero ones across views
// (geometry.py:1558-1595).  Outputs padded to 8 columns: quats8 [V][8], trans8 [V][8], log_scale8 [V][8].
// One block; views strided over threads.
// ----------------------------------------------------------------------------------------------
__global__ void pose_inputs_kernel(const float* __restrict__ quats, const float* __restrict__ trans,
                                   const uint8_t* __restrict__ has_pose, int V, float* __restrict__ quats8,
                                   float* __restrict__ trans8, float* __restrict__ log_scale8) {
  __shared__ float red[32];
  const float q0x = quats[0], q0y = quats[1], q0z = quats[2], q0w = quats[3];
  const float n2 = q0x * q0x + q0y * q0y + q0z * q0z + q0w * q0w;
  // inverse quaternion, then its rotation matrix (normalised first, geometry.py:601-652)
  const float ix = -q0x / n2, iy = -q0y / n2, iz = -q0z / n2, iw = q0w / n2;
  const float inn = sqrtf(ix * ix + iy * iy + iz * iz + iw * iw);
  const float x = ix / inn, y = iy / inn, z = iz / inn, w = iw / inn;
  const float r00 = 1 - 2 * (y * y + z * z), r01 = 2 * (x * y - w * z), r02 = 2 * (x * z + w * y);
  const float r10 = 2 * (x * y + w * z), r11 = 1 - 2 * (x * x + z * z), r12 = 2 * (y * z - w * x);
  const float r20 = 2 * (x * z - w * y), r21 = 2 * (y * z + w * x), r22 = 1 - 2 * (x * x + y * y);
  // R t evaluated with ONE fixed operation order, so that R t_v - R t_0 is exactly 0 for v = 0 (the reference computes
  // einsum(R, t_v) + (-einsum(R, t_0)) with identical kernels; a zero translation must not count as "non-zero" below)
  auto rot_row = [](float a, float b, float c, float x_, float y_, float z_) {
    return __fmaf_rn(c, z_, __fmaf_rn(b, y_, __fmul_rn(a, x_)));
  };
  const float t0x = trans[0], t0y = trans[1], t0z = trans[2];
  const float tix = -rot_row(r00, r01, r02, t0x, t0y, t0z), tiy = -rot_row(r10, r11, r12, t0x, t0y, t0z),
              tiz = -rot_row(r20, r21, r22, t0x, t0y, t0z);
  float dsum = 0.f, dcnt = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float qx = 0.f, qy = 0.f, qz = 0.f, qw = 1.f, tx = 0.f, ty = 0.f, tz = 0.f;
    if (has_pose[v]) {
      const float ax = quats[4 * v], ay = quats[4 * v + 1], az = quats[4 * v + 2], aw = quats[4 * v + 3];
      // Hamilton product (inverse of q0) (x) q_v, scalar last (geometry.py:775-811)
      qx = iw * ax + ix * aw + iy * az - iz * ay;
      qy = iw * ay - ix * az + iy * aw + iz * ax;
      qz = iw * az + ix * ay - iy * ax + iz * aw;
      qw = iw * aw - ix * ax - iy * ay - iz * az;
      const float bx = trans[3 * v], by = trans[3 * v + 1], bz = trans[3 * v + 2];
      tx = __fadd_rn(rot_row(r00, r01, r02, bx, by, bz), tix);
      ty = __fadd_rn(rot_row(r10, r11, r12, bx, by, bz), tiy);
      tz = __fadd_rn(rot_row(r20, r21, r22, bx, by, bz), tiz);
    }
    float* q8 = quats8 + 8 * v;
    q8[0] = qx; q8[1] = qy; q8[2] = qz; q8[3] = qw; q8[4] = q8[5] = q8[6] = q8[7] = 0.f;
    float* t8 = trans8 + 8 * v;  // unscaled for now
    t8[0] = tx; t8[1] = ty; t8[2] = tz; t8[3] = t8[4] = t8[5] = t8[6] = t8[7] = 0.f;
    const float d = sqrtf(tx * tx + ty * ty + tz * tz);
    dsum += d;
    dcnt += d > 0.f ? 1.f : 0.f;
  }
  dsum = block_sum(dsum, red);
  dcnt = block_sum(dcnt, red);
  const float f = fmaxf(dsum / (dcnt + 1e-8f), 1e-8f);
  const float lf = logf(f + 1e-8f);
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float* t8 = trans8 + 8 * v;
    t8[0] /= f; t8[1] /= f; t8[2] /= f;
    float* s8 = log_scale8 + 8 * v;
    s8[0] = lf;
#pragma unroll
    for (int j = 1; j < 8; ++j) s8[j] = 0.f;
  }
}

// ----------------------------------------------------------------------------------------------
// Fusion adds (model.py:820-825, :1003-1008, :1124-1129), in place on the fp32 encoder features [V*N][C]:
//   feat[v*N + t] += dense_a[a_slot[v]*N + t] + dense_b[b_slot[v]*N + t] + sum_j gw[j][v] * g_j[v]
// a_slot / b_slot = index of view v among the views that provide the modality, or -1; g_j = global features
// (0 rotation, 1 translation, 2 pose scale: one row per view; 3 depth scale: one row per b_slot), gw = their 0/1 gates.  The fusion LayerNorm follows (ma_layernorm).
// ----------------------------------------------------------------------------------------------
struct FuseParams {
  float* feat;
  const float* dense_a;
  const int* a_slot;
  const float* dense_b;
  const int* b_slot;
  const float* g[4];
  const float* gw;  // [4][V]
  int V, N, C;
};

__global__ void fuse_add_kernel(const FuseParams p) {
  const int c4n = p.C >> 2;
  const int64_t total = (int64_t)p.V * p.N * c4n;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c4 = static_cast<int>(idx % c4n);
    const int64_t row = idx / c4n;
    const int v = static_cast<int>(row / p.N);
    const int t = static_cast<int>(row - (int64_t)v * p.N);
    float4* f = reinterpret_cast<float4*>(p.feat + row * p.C) + c4;
    float4 x = *f;
    if (p.dense_a && p.a_slot[v] >= 0) {
      const float4 a = *(reinterpret_cast<const float4*>(p.dense_a + ((int64_t)p.a_slot[v] * p.N + t) * p.C) + c4);
      x.x += a.x; x.y += a.y; x.z += a.z; x.w += a.w;
    }
    if (p.dense_b && p.b_slot[v] >= 0) {
      const float4 a = *(reinterpret_cast<const float4*>(p.dense_b + ((int64_t)p.b_slot[v] * p.N + t) * p.C) + c4);
      x.x += a.x; x.y += a.y; x.z += a.z; x.w += a.w;
    }
    float4 gs = make_float4(0.f, 0.f, 0.f, 0.f);
    bool any = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (!p.g[j]) continue;
      const float wj = p.gw[j * p.V + v];
      if (wj == 0.f) continue;
      // g_3 (depth scale) is stored per DEPTH view: indexed through the depth slot table
      const int gv = j == 3 ? (p.b_slot ? p.b_slot[v] : -1) : v;
      if (gv < 0) continue;
      const float4 a = *(reinterpret_cast<const float4*>(p.g[j] + (int64_t)gv * p.C) + c4);
      gs.x += wj * a.x; gs.y += wj * a.y; gs.z += wj * a.z; gs.w += wj * a.w;
      any = true;
    }
    if (any) { x.x += gs.x; x.y += gs.y; x.z += gs.z; x.w += gs.w; }
    *f = x;
  }
}

// ----------------------------------------------------------------------------------------------
// infer() input preprocessing (reference mapanything/utils/inference.py:202-291), one thread per pixel / per pose.
// ----------------------------------------------------------------------------------------------
// get_rays_in_camera_frame(normalize_to_unit_sphere=True) (geometry.py:186-241): ((x-cx)/fx, (y-cy)/fy, 1) / norm
__global__ void rays_from_intrinsics_kernel(const float* __restrict__ K, float* __restrict__ out, int H, int W, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int x = static_cast<int>(idx % W);
    const int64_t t = idx / W;
    const int y = static_cast<int>(t % H);
    const int b = static_cast<int>(t / H);
    const float* k = K + 9 * b;
    const float xx = (static_cast<float>(x) - k[2]) / k[0];
    const float yy = (static_cast<float>(y) - k[5]) / k[4];
    const float n = sqrtf(xx * xx + yy * yy + 1.0f);
    float* o = out + idx * 3;
    o[0] = xx / n; o[1] = yy / n; o[2] = 1.0f / n;
  }
}

// ray / (|ray| + 1e-8)   (inference.py:238-241)
__global__ void normalize_rays_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const float a = in[idx * 3], b = in[idx * 3 + 1], c = in[idx * 3 + 2];
    const float n = sqrtf(a * a + b * b + c * c) + 1e-8f;
    out[idx * 3] = a / n; out[idx * 3 + 1] = b / n; out[idx * 3 + 2] = c / n;
  }
}

// depth_along_ray = | depth_z * ray / ray_z |   (inference.py:243-251)
__global__ void depth_z_to_along_ray_kernel(const float* __restrict__ depth_z, const float* __restrict__ rays,
                                            float* __restrict__ out, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const float z = rays[idx * 3 + 2];
    const float d = depth_z[idx];
    const float px = d * (rays[idx * 3] / z), py = d * (rays[idx * 3 + 1] / z), pz = d * (z / z);
    out[idx] = sqrtf(px * px + py * py + pz * pz);
  }
}

// (B,4,4) cam2world -> quats (xyzw, w >= 0) + translations: rotation_matrix_to_quaternion (geometry.py:655-742)
__global__ void pose_to_quat_trans_kernel(const float* __restrict__ poses, float* __restrict__ quats, float* __restrict__ trans,
                                          int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* m = poses + 16 * b;
  const float m00 = m[0], m01 = m[1], m02 = m[2], m10 = m[4], m11 = m[5], m12 = m[6], m20 = m[8], m21 = m[9], m22 = m[10];
  trans[3 * b] = m[3]; trans[3 * b + 1] = m[7]; trans[3 * b + 2] = m[11];
  const float sq[4] = {1 + m00 + m11 + m22, 1 + m00 - m11 - m22, 1 - m00 + m11 - m22, 1 - m00 - m11 + m22};
  float qa[4];
  int best = 0;
  for (int i = 0; i < 4; ++i) {
    qa[i] = sq[i] > 0.f ? sqrtf(sq[i]) : 0.f;
    if (qa[i] > qa[best]) best = i;  // first maximum, like torch.argmax
  }
  float c[4];  // candidate `best`, order (w, x, y, z)
  if (best == 0) { c[0] = qa[0] * qa[0]; c[1] = m21 - m12; c[2] = m02 - m20; c[3] = m10 - m01; }
  else if (best == 1) { c[0] = m21 - m12; c[1] = qa[1] * qa[1]; c[2] = m10 + m01; c[3] = m02 + m20; }
  else if (best == 2) { c[0] = m02 - m20; c[1] = m10 + m01; c[2] = qa[2] * qa[2]; c[3] = m12 + m21; }
  else { c[0] = m10 - m01; c[1] = m20 + m02; c[2] = m21 + m12; c[3] = qa[3] * qa[3]; }
  const float den = 2.0f * fmaxf(qa[best], 0.1f);
  float w = c[0] / den, x = c[1] / den, y = c[2] / den, z = c[3] / den;
  if (w < 0.f) { w = -w; x = -x; y = -y; z = -z; }
  quats[4 * b] = x; quats[4 * b + 1] = y; quats[4 * b + 2] = z; quats[4 * b + 3] = w;
}

static inline int grid_for(int64_t total) {
  int64_t blocks = (total + 255) / 256;
  const int64_t cap = (int64_t)device_sm_count() * 16;
  return static_cast<int>(blocks > cap ? cap : blocks);
}

}  // namespace ma

extern "C" int ma_rays_from_intrinsics(const float* K, float* rays, int B, int H, int W, void* stream) {
  using namespace ma;
  MA_REQUIRE(K && rays && B > 0 && H > 0 && W > 0, "ma_rays_from_intrinsics: bad arguments");
  const int64_t total = (int64_t)B * H * W;
  rays_from_intrinsics_kernel<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(K, rays, H, W, total);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_normalize_rays(const float* in, float* out, int64_t pixels, void* stream) {
  using namespace ma;
  MA_REQUIRE(in && out && pixels > 0, "ma_normalize_rays: bad arguments");
  normalize_rays_kernel<<<grid_for(pixels), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, pixels);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_depth_z_to_along_ray(const float* depth_z, const float* rays, float* out, int64_t pixels, void* stream) {
  using namespace ma;
  MA_REQUIRE(depth_z && rays && out && pixels > 0, "ma_depth_z_to_along_ray: bad arguments");
  depth_z_to_along_ray_kernel<<<grid_for(pixels), 256, 0, static_cast<cudaStream_t>(stream)>>>(depth_z, rays, out, pixels);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_pose_to_quat_trans(const float* poses, float* quats, float* trans, int B, void* stream) {
  using namespace ma;
  MA_REQUIRE(poses && quats && trans && B > 0, "ma_pose_to_quat_trans: bad arguments");
  pose_to_quat_trans_kernel<<<(B + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(poses, quats, trans, B);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_unshuffle_split(const float* in, void* out, int n, int H, int W, int cin, int patch, int cpad, int mode,
                                  const float* factor, void* stream) {
  using namespace ma;
  MA_REQUIRE(in && out, "ma_unshuffle_split: null pointer");
  MA_REQUIRE(patch > 0, "ma_unshuffle_split: patch must be positive, got %d", patch);
  MA_REQUIRE(n > 0 && H % patch == 0 && W % patch == 0 && cin > 0, "ma_unshuffle_split: bad shape");
  MA_REQUIRE(cpad % 8 == 0 && cpad >= cin * patch * patch, "ma_unshuffle_split: cpad must be a multiple of 8 >= cin*p*p");
  MA_REQUIRE(mode == 0 || (mode == 1 && factor), "ma_unshuffle_split: mode 1 needs the per-view factor");
  const int hp = H / patch, wp = W / patch;
  unshuffle_split_kernel<<<n * hp * wp, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, static_cast<__nv_bfloat16*>(out), H, W, cin, hp, wp, patch, cpad, mode, factor);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_depth_factor(const float* depth, int n, int64_t per_view, float* factor, float* log_factor8, void* stream) {
  using namespace ma;
  MA_REQUIRE(depth && factor && log_factor8 && n > 0 && per_view > 0, "ma_depth_factor: bad arguments");
  depth_factor_kernel<<<n, 1024, 0, static_cast<cudaStream_t>(stream)>>>(depth, per_view, factor, log_factor8);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_pose_inputs(const float* quats, const float* trans, const uint8_t* has_pose, int V, float* quats8,
                              float* trans8, float* log_scale8, void* stream) {
  using namespace ma;
  MA_REQUIRE(quats && trans && has_pose && quats8 && trans8 && log_scale8 && V > 0, "ma_pose_inputs: bad arguments");
  pose_inputs_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(quats, trans, has_pose, V, quats8, trans8, log_scale8);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_fuse_add(float* feat, int V, int N, int C, const float* dense_a, const int* a_slot, const float* dense_b,
                           const int* b_slot, const float* g0, const float* g1, const float* g2, const float* g3,
                           const float* gw, void* stream) {
  using namespace ma;
  MA_REQUIRE(feat && V > 0 && N > 0 && C > 0 && C % 4 == 0, "ma_fuse_add: bad arguments");
  MA_REQUIRE((!dense_a || a_slot) && (!dense_b || b_slot), "ma_fuse_add: dense addend without its slot table");
  MA_REQUIRE(!(g0 || g1 || g2 || g3) || gw, "ma_fuse_add: global addends need their gate table");
  // float4 loads and stores: every row operand that is present must be 16-byte aligned (C % 4 == 0 keeps its rows so)
  const struct { const void* ptr; const char* name; } rows[] = {{feat, "feat"}, {dense_a, "dense_a"}, {dense_b, "dense_b"},
                                                               {g0, "g0"}, {g1, "g1"}, {g2, "g2"}, {g3, "g3"}};
  for (const auto& r : rows)
    MA_REQUIRE(reinterpret_cast<uintptr_t>(r.ptr) % 16 == 0, "ma_fuse_add: %s not 16-byte aligned", r.name);
  FuseParams p;
  p.feat = feat; p.dense_a = dense_a; p.a_slot = a_slot; p.dense_b = dense_b; p.b_slot = b_slot;
  p.g[0] = g0; p.g[1] = g1; p.g[2] = g2; p.g[3] = g3; p.gw = gw;
  p.V = V; p.N = N; p.C = C;
  const int64_t total = (int64_t)V * N * (C / 4);
  int blocks = static_cast<int>((total + 255) / 256);
  const int cap = device_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  fuse_add_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
