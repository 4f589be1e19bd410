// Input side of infer(): load_images() resize / crop / normalise (reference mapanything/utils/image.py:134-332 through
// cropping.py:385-467 crop_resize_if_necessary -> cropping.py:188-275 rescale_image_and_other_optional_info, which calls
// PIL.Image.resize with LANCZOS (down-scaling) or BICUBIC (up-scaling), then a centred crop, then torchvision
// ToTensor + Normalize, image.py:291-296, :312).
//
// PIL's 8-bit resize is INTEGER arithmetic (Pillow src/libImaging/Resample.c): per output coordinate a window of the
// separable filter is evaluated in double precision, normalised, rounded to 22-bit fixed point; each pass accumulates
// int32 products from 1 << 21, shifts right by 22 and clamps to a byte; the horizontal pass runs first and its 8-bit
// result feeds the vertical pass.  Restated here so that the GPU path is BIT-EXACT with the reference's images:
//   * ma_resample_coeffs / ma_resample_pack_coeffs (host, libm double precision like Pillow): window bounds, fixed-point
//                          coefficients and their byte planes
//   * resample_h_dp4a_kernel  one block per source row: the row is staged in shared memory with 4-byte coalesced loads and
//                          split into R / G / B byte planes; every thread produces output pixels of that row with dp4a on
//                          byte-split coefficients.  Runs when the caller passes the packed coefficients, the window has
//                          at most 64 taps and the staged span fits shared memory.  Otherwise resample_h_vec_kernel
//                          (32-bit loads + PRMT) runs for windows of at most 64 taps, and resample_h_kernel (byte loads,
//                          any window length) for longer windows or spans too wide for the other two
//   * resample_v_norm_kernel  thread per output pixel of the CROPPED target: vertical pass over the 8-bit
//                          intermediate (taps are row-contiguous across a warp), byte clamp, (u/255 - mean)/std in the
//                          rounding order of torchvision, planar fp32 (3,H,W) output = the model's `img` layout
//   * gather_rows_cols_f32_kernel / f32_to_u8_kernel  nearest-neighbour depth resize + crop, float image -> bytes
// By bytes this is HBM work (a 1920x1080 frame: 6.2 MB in, 1.7 MB intermediate, 1.8 MB out); in practice the integer
// pipes bound it (25-tap LANCZOS windows at this reduction), see DESIGN.md section 5 for the measured forms.
#include <math.h>

#include <vector>

#include "host_common.h"

namespace ma {

constexpr int RS_PRECISION_BITS = 32 - 8 - 2;  // Pillow Resample.c PRECISION_BITS

static inline double sinc_filter(double x) {
  if (x == 0.0) return 1.0;
  x = x * M_PI;
  return sin(x) / x;
}
static inline double lanczos_filter(double x) {  // truncated sinc, support 3
  if (-3.0 <= x && x < 3.0) return sinc_filter(x) * sinc_filter(x / 3);
  return 0.0;
}
static inline double bicubic_filter(double x) {  // Keys cubic, a = -0.5, support 2
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

__device__ __forceinline__ uint8_t clip8(int v) {
  v >>= RS_PRECISION_BITS;  // arithmetic shift, like Pillow's clip8 lookup
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// One block per source row [y0 + blockIdx.x] of frame blockIdx.y; output columns [x0, x0 + cols) of the resampled row.
__global__ void resample_h_kernel(const uint8_t* __restrict__ src, int64_t row_stride, int64_t frame_stride, int y0, int sx0,
                                  int sx1, const int32_t* __restrict__ bounds, const int32_t* __restrict__ coeffs, int out_size,
                                  int x0, int cols, uint8_t* __restrict__ tmp) {
  extern __shared__ __align__(16) uint8_t srow[];
  const uint8_t* row = src + blockIdx.y * frame_stride + (y0 + static_cast<int64_t>(blockIdx.x)) * row_stride +
                       static_cast<int64_t>(sx0) * 3;
  const int nbytes = (sx1 - sx0) * 3;
  // 4-byte coalesced loads from the enclosing aligned span; `mis` is the offset of the first wanted byte in it
  const int mis = static_cast<int>(reinterpret_cast<uintptr_t>(row) & 3);
  const uint32_t* row4 = reinterpret_cast<const uint32_t*>(row - mis);
  const int nwords = (mis + nbytes + 3) >> 2;
  uint32_t* s4 = reinterpret_cast<uint32_t*>(srow);
  for (int i = threadIdx.x; i < nwords; i += blockDim.x) s4[i] = __ldg(row4 + i);
  __syncthreads();
  const uint8_t* s = srow + mis;
  uint8_t* orow = tmp + (static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x) * cols * 3;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) {
    const int xx = x0 + i;
    const int first = bounds[2 * xx], cnt = bounds[2 * xx + 1];
    int a0 = 1 << (RS_PRECISION_BITS - 1), a1 = a0, a2 = a0;
    const uint8_t* p = s + (first - sx0) * 3;
    for (int t = 0; t < cnt; ++t) {
      const int k = coeffs[static_cast<int64_t>(t) * out_size + xx];  // tap-major: coalesced across the warp
      a0 += p[3 * t] * k;
      a1 += p[3 * t + 1] * k;
      a2 += p[3 * t + 2] * k;
    }
    orow[3 * i] = clip8(a0);
    orow[3 * i + 1] = clip8(a1);
    orow[3 * i + 2] = clip8(a2);
  }
}

// Word-load form of the horizontal pass (the default).  Same block <-> source row mapping as resample_h_kernel, but a
// thread fetches its whole window (3 * KMAX bytes at an arbitrary byte offset of the staged row) with 32-bit shared-memory
// loads, realigns it with funnel shifts and picks the bytes with PRMT: 3*KMAX/4 + 1 shared-memory instructions per output
// pixel instead of 3 * taps byte loads.  The byte loads were the bound of the first kernel: neighbouring lanes read
// windows ~11 bytes apart, every LDS.U8 is a 3-way bank conflict, and the shared-memory pipe -- not HBM, not the integer
// pipe -- set the time (14.8 us per 1920x1080 frame, 12 % of the HBM roofline).  A "strip" variant that kept the window
// coefficients in registers over 8 staged rows was measured SLOWER (23.9 us: same byte loads, half the occupancy).
// Absent taps (t >= cnt) carry a zero coefficient; the staged row is padded so their bytes are inside the block's smem.
template <int KMAX>
__global__ void __launch_bounds__(256)
resample_h_vec_kernel(const uint8_t* __restrict__ src, int64_t row_stride, int64_t frame_stride, int y0, int sx0, int sx1,
                      const int32_t* __restrict__ bounds, const int32_t* __restrict__ coeffs, int out_size, int x0, int cols,
                      uint8_t* __restrict__ tmp) {
  constexpr int NW = (3 * KMAX + 3) / 4;  // words holding the realigned window
  extern __shared__ __align__(16) uint8_t srow[];
  const uint8_t* row = src + blockIdx.y * frame_stride + (y0 + static_cast<int64_t>(blockIdx.x)) * row_stride +
                       static_cast<int64_t>(sx0) * 3;
  const int nbytes = (sx1 - sx0) * 3;
  const int mis = static_cast<int>(reinterpret_cast<uintptr_t>(row) & 3);
  const uint32_t* row4 = reinterpret_cast<const uint32_t*>(row - mis);
  const int nwords = (mis + nbytes + 3) >> 2;
  uint32_t* s4 = reinterpret_cast<uint32_t*>(srow);
  for (int i = threadIdx.x; i < nwords; i += blockDim.x) s4[i] = __ldg(row4 + i);
  __syncthreads();
  uint8_t* orow = tmp + (static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x) * cols * 3;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) {
    const int xx = x0 + i;
    const int first = bounds[2 * xx], cnt = bounds[2 * xx + 1];
    const int off = mis + (first - sx0) * 3;
    const uint32_t* w4 = s4 + (off >> 2);
    const int sh = (off & 3) * 8;
    uint32_t w[NW + 1];
#pragma unroll
    for (int j = 0; j <= NW; ++j) w[j] = w4[j];
#pragma unroll
    for (int j = 0; j < NW; ++j) w[j] = __funnelshift_r(w[j], w[j + 1], sh);  // window byte b is now byte (b & 3) of w[b >> 2]
    int a0 = 1 << (RS_PRECISION_BITS - 1), a1 = a0, a2 = a0;
#pragma unroll
    for (int t = 0; t < KMAX; ++t) {
      const int k = t < cnt ? __ldg(coeffs + static_cast<int64_t>(t) * out_size + xx) : 0;
      a0 += static_cast<int>(__byte_perm(w[(3 * t) >> 2], 0, 0x4440 | ((3 * t) & 3))) * k;
      a1 += static_cast<int>(__byte_perm(w[(3 * t + 1) >> 2], 0, 0x4440 | ((3 * t + 1) & 3))) * k;
      a2 += static_cast<int>(__byte_perm(w[(3 * t + 2) >> 2], 0, 0x4440 | ((3 * t + 2) & 3))) * k;
    }
    orow[3 * i] = clip8(a0);
    orow[3 * i + 1] = clip8(a1);
    orow[3 * i + 2] = clip8(a2);
  }
}

// dp4a form of the horizontal pass (used when the caller supplies byte-packed coefficients, ma_resample_pack_coeffs).
// While a row is staged, R, G and B are separated into three byte planes (12 bytes = 4 pixels per thread step: 4 aligned
// word loads, funnel shift, 6 PRMT, 3 word stores), so 4 consecutive taps of ONE channel sit in one 32-bit word.  The 22-bit
// signed coefficient k = k0 + 2^8 k1 + 2^16 k2 (k0, k1 unsigned bytes, k2 a signed byte) is applied as three dp4a per word:
// 3 integer instructions per 4 taps instead of 4 byte extractions + 4 multiply-adds; the three partial sums recombine
// exactly (two's-complement adds; the true accumulator fits 32 bits as it does in Pillow).
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {  // a: 4 unsigned bytes, b: 4 SIGNED bytes
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

template <int NW4>  // 32-bit words per channel window = ceil(window length / 4)
__global__ void __launch_bounds__(256)
resample_h_dp4a_kernel(const uint8_t* __restrict__ src, int64_t row_stride, int64_t frame_stride, int y0, int sx0, int sx1,
                       const int32_t* __restrict__ bounds, const uint32_t* __restrict__ packed, int out_size, int x0, int cols,
                       uint8_t* __restrict__ tmp, int plane_words) {
  extern __shared__ __align__(16) uint8_t srow[];
  uint32_t* plane = reinterpret_cast<uint32_t*>(srow);  // [3][plane_words]
  const uint8_t* row = src + blockIdx.y * frame_stride + (y0 + static_cast<int64_t>(blockIdx.x)) * row_stride +
                       static_cast<int64_t>(sx0) * 3;
  const int npx = sx1 - sx0;
  const int mis = static_cast<int>(reinterpret_cast<uintptr_t>(row) & 3);
  const uint32_t* row4 = reinterpret_cast<const uint32_t*>(row - mis);
  const int last_word = (mis + npx * 3 - 1) >> 2;  // last word holding a wanted byte: nothing beyond it is read
  const int sh0 = mis * 8;
  for (int g = threadIdx.x; g * 4 < npx; g += blockDim.x) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = __ldg(row4 + min(3 * g + j, last_word));
    const uint32_t b0 = __funnelshift_r(w[0], w[1], sh0);  // R0 G0 B0 R1
    const uint32_t b1 = __funnelshift_r(w[1], w[2], sh0);  // G1 B1 R2 G2
    const uint32_t b2 = __funnelshift_r(w[2], w[3], sh0);  // B2 R3 G3 B3
    plane[g] = __byte_perm(__byte_perm(b0, b1, 0x0630), b2, 0x5210);
    plane[plane_words + g] = __byte_perm(__byte_perm(b0, b1, 0x0741), b2, 0x6210);
    plane[2 * plane_words + g] = __byte_perm(__byte_perm(b0, b1, 0x0052), b2, 0x7410);
  }
  __syncthreads();
  uint8_t* orow = tmp + (static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x) * cols * 3;
  const int64_t pstride = static_cast<int64_t>(NW4) * out_size;  // words per coefficient byte plane
  for (int i = threadIdx.x; i < cols; i += blockDim.x) {
    const int xx = x0 + i;
    const int po = bounds[2 * xx] - sx0;  // first window pixel, relative to the staged span
    const uint32_t* wp = plane + (po >> 2);
    const int sh = (po & 3) * 8;
    uint32_t k0[NW4], k1[NW4], k2[NW4];
#pragma unroll
    for (int j = 0; j < NW4; ++j) {
      k0[j] = __ldg(packed + static_cast<int64_t>(j) * out_size + xx);
      k1[j] = __ldg(packed + pstride + static_cast<int64_t>(j) * out_size + xx);
      k2[j] = __ldg(packed + 2 * pstride + static_cast<int64_t>(j) * out_size + xx);
    }
    int acc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      uint32_t w[NW4 + 1];
#pragma unroll
      for (int j = 0; j <= NW4; ++j) w[j] = wp[c * plane_words + j];
      int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
      for (int j = 0; j < NW4; ++j) {
        const uint32_t px = __funnelshift_r(w[j], w[j + 1], sh);
        s0 = static_cast<int>(__dp4a(px, k0[j], static_cast<uint32_t>(s0)));
        s1 = static_cast<int>(__dp4a(px, k1[j], static_cast<uint32_t>(s1)));
        s2 = dp4a_us(px, k2[j], s2);
      }
      acc[c] = (1 << (RS_PRECISION_BITS - 1)) + s0 + s1 * 256 + s2 * 65536;
    }
    orow[3 * i] = clip8(acc[0]);
    orow[3 * i + 1] = clip8(acc[1]);
    orow[3 * i + 2] = clip8(acc[2]);
  }
}

// Thread per output pixel (x, yy = top + blockIdx.y) of the cropped target of frame blockIdx.z.
// (A fully unrolled tap loop -- all byte loads of a pixel in flight at once -- was measured slower: 11.7 vs 10.1 us per
// 1920x1080 frame for both passes together.)
__global__ void resample_v_norm_kernel(const uint8_t* __restrict__ tmp, int rows, int cols, int y0, const int32_t* __restrict__ bounds,
                                       const int32_t* __restrict__ coeffs, int out_size, int top, int th, float m0, float m1,
                                       float m2, float s0, float s1, float s2, float* __restrict__ out_chw,
                                       uint8_t* __restrict__ out_u8) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= cols) return;
  const int yy = top + y;
  const int first = bounds[2 * yy], cnt = bounds[2 * yy + 1];
  int a0 = 1 << (RS_PRECISION_BITS - 1), a1 = a0, a2 = a0;
  const uint8_t* p = tmp + ((static_cast<int64_t>(blockIdx.z) * rows + (first - y0)) * cols + x) * 3;
  const int64_t rs = static_cast<int64_t>(cols) * 3;
  for (int t = 0; t < cnt; ++t, p += rs) {
    const int k = __ldg(coeffs + static_cast<int64_t>(t) * out_size + yy);  // warp-uniform
    a0 += p[0] * k;
    a1 += p[1] * k;
    a2 += p[2] * k;
  }
  const uint8_t u0 = clip8(a0), u1 = clip8(a1), u2 = clip8(a2);
  if (out_u8) {
    uint8_t* o = out_u8 + ((static_cast<int64_t>(blockIdx.z) * th + y) * cols + x) * 3;
    o[0] = u0;
    o[1] = u1;
    o[2] = u2;
  }
  if (out_chw) {
    // torchvision: ToTensor = float(u) / 255, Normalize = (t - mean) / std; each step rounded to fp32
    const int64_t plane = static_cast<int64_t>(th) * cols;
    const int64_t o = 3 * plane * blockIdx.z + static_cast<int64_t>(y) * cols + x;
    out_chw[o] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(u0), 255.0f), m0), s0);
    out_chw[plane + o] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(u1), 255.0f), m1), s1);
    out_chw[2 * plane + o] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(u2), 255.0f), m2), s2);
  }
}

// out[y][x] = src[y_idx[y]][x_idx[x]]: cv2.resize(INTER_NEAREST) + crop of a float map as one gather (index arrays are
// OpenCV's resizeNN offsets of the cropped window, computed on the host in double precision).
__global__ void gather_rows_cols_f32_kernel(const float* __restrict__ src, int64_t row_stride, const int32_t* __restrict__ y_idx,
                                            const int32_t* __restrict__ x_idx, int tw, float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= tw) return;
  const int y = blockIdx.y;
  out[static_cast<int64_t>(y) * tw + x] = __ldg(src + static_cast<int64_t>(y_idx[y]) * row_stride + x_idx[x]);
}

// torch: (img * scale).clamp(0, 255).byte()  (image.py:503-506); scale = 255 for images in [0, 1], else 1
__global__ void f32_to_u8_kernel(const float* __restrict__ in, int64_t n, float scale, uint8_t* __restrict__ out) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = fminf(fmaxf(__fmul_rn(in[i], scale), 0.f), 255.f);
  out[i] = static_cast<uint8_t>(static_cast<int>(v));  // truncation, like the C cast behind .byte()
}

// Which form of the horizontal pass this thread launched last: 1 = resample_h_kernel, 1000 + KMAX = resample_h_vec_kernel<KMAX>,
// 2000 + NW4 = resample_h_dp4a_kernel<NW4>; 0 before the first launch.
thread_local int g_last_resample_kernel = 0;

}  // namespace ma

extern "C" int ma_last_resample_kernel(void) { return ma::g_last_resample_kernel; }

using namespace ma;

extern "C" int ma_gather_rows_cols_f32(const float* src, int64_t src_row_stride, const int32_t* y_idx, const int32_t* x_idx,
                                       int th, int tw, float* out, void* stream) {
  MA_REQUIRE(src && y_idx && x_idx && out && th > 0 && tw > 0, "ma_gather_rows_cols_f32: bad arguments (th=%d tw=%d)", th, tw);
  MA_REQUIRE(th <= 65535, "ma_gather_rows_cols_f32: th=%d above 65535 (one grid row per output row)", th);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(src) & 3) == 0, "ma_gather_rows_cols_f32: src not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(y_idx) & 3) == 0, "ma_gather_rows_cols_f32: y_idx not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(x_idx) & 3) == 0, "ma_gather_rows_cols_f32: x_idx not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0, "ma_gather_rows_cols_f32: out not 4-byte aligned");
  dim3 grid((tw + 127) / 128, th);
  gather_rows_cols_f32_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(src, src_row_stride, y_idx, x_idx, tw, out);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_f32_to_u8(const float* in, int64_t n, float scale, uint8_t* out, void* stream) {
  MA_REQUIRE(in && out && n > 0, "ma_f32_to_u8: bad arguments");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(in) & 3) == 0, "ma_f32_to_u8: in not 4-byte aligned");
  f32_to_u8_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, n, scale, out);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_resample_coeffs(int in_size, int out_size, int filter, int* ksize_out, int32_t* bounds, int32_t* coeffs) {
  MA_REQUIRE(in_size > 0 && out_size > 0 && ksize_out, "ma_resample_coeffs: bad sizes (%d -> %d)", in_size, out_size);
  MA_REQUIRE(filter == MA_FILTER_LANCZOS || filter == MA_FILTER_BICUBIC, "ma_resample_coeffs: unsupported filter %d", filter);
  if (in_size == out_size) {  // Pillow skips the pass (Resample.c need_horizontal / need_vertical): identity taps
    *ksize_out = 1;
    if (bounds && coeffs) {
      for (int i = 0; i < out_size; ++i) {
        bounds[2 * i] = i;
        bounds[2 * i + 1] = 1;
        coeffs[i] = 1 << RS_PRECISION_BITS;
      }
    }
    return MA_OK;
  }
  double (*f)(double) = filter == MA_FILTER_LANCZOS ? lanczos_filter : bicubic_filter;
  const double fsupport = filter == MA_FILTER_LANCZOS ? 3.0 : 2.0;
  // Resample.c precompute_coeffs with box = (0, in_size)
  const float in0 = 0.f, in1 = static_cast<float>(in_size);
  double scale = static_cast<double>(in1 - in0) / out_size, filterscale = scale;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = fsupport * filterscale;
  const int ksize = static_cast<int>(ceil(support)) * 2 + 1;
  *ksize_out = ksize;
  if (!bounds || !coeffs) return MA_OK;
  std::vector<double> k(ksize);
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = in0 + (xx + 0.5) * scale;
    double ww = 0.0;
    const double ss = 1.0 / filterscale;
    int xmin = static_cast<int>(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = static_cast<int>(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    int x = 0;
    for (; x < xmax; ++x) {
      const double w = f((x + xmin - center + 0.5) * ss);
      k[x] = w;
      ww += w;
    }
    for (x = 0; x < xmax; ++x)
      if (ww != 0.0) k[x] /= ww;
    for (; x < ksize; ++x) k[x] = 0;
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
    for (x = 0; x < ksize; ++x) {  // normalize_coeffs_8bpc; stored tap-major [ksize][out_size]
      const double v = k[x];
      coeffs[static_cast<int64_t>(x) * out_size + xx] =
          v < 0 ? static_cast<int>(-0.5 + v * (1 << RS_PRECISION_BITS)) : static_cast<int>(0.5 + v * (1 << RS_PRECISION_BITS));
    }
  }
  return MA_OK;
}

template <int KMAX>
static int launch_h_vec(const uint8_t* src, int64_t row_stride, int64_t frame_stride, int n, int y0, int rows, int sx0, int sx1,
                        const int32_t* bounds, const int32_t* coeffs, int out_size, int x0, int cols, uint8_t* tmp,
                        cudaStream_t stream) {
  // staged row + misalignment + the zero-coefficient taps' bytes + the funnel shift's extra word
  const size_t smem = (static_cast<size_t>(sx1 - sx0) * 3 + 3 + 3 * KMAX + 8 + 15) & ~static_cast<size_t>(15);
  static size_t configured_dev[MA_MAX_DEVICES] = {};
  size_t& configured = configured_dev[current_device()];
  if (smem > 48 * 1024 && smem > configured) {
    MA_CHECK_CUDA(cudaFuncSetAttribute(resample_h_vec_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = 200 * 1024;
  }
  g_last_resample_kernel = 1000 + KMAX;
  resample_h_vec_kernel<KMAX><<<dim3(rows, n), 256, smem, stream>>>(src, row_stride, frame_stride, y0, sx0, sx1, bounds, coeffs,
                                                                    out_size, x0, cols, tmp);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

template <int NW4>
static int launch_h_dp4a(const uint8_t* src, int64_t row_stride, int64_t frame_stride, int n, int y0, int rows, int sx0, int sx1,
                         const int32_t* bounds, const uint32_t* packed, int out_size, int x0, int cols, uint8_t* tmp,
                         cudaStream_t stream) {
  // per plane: the staged pixels + the window overhang of the last output (zero coefficients) + the funnel shift's word
  const int plane_words = ((sx1 - sx0 + 3) >> 2) + NW4 + 2;
  const size_t smem = static_cast<size_t>(3) * plane_words * 4;
  static size_t configured_dev[MA_MAX_DEVICES] = {};
  size_t& configured = configured_dev[current_device()];
  if (smem > 48 * 1024 && smem > configured) {
    MA_CHECK_CUDA(cudaFuncSetAttribute(resample_h_dp4a_kernel<NW4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = 200 * 1024;
  }
  g_last_resample_kernel = 2000 + NW4;
  resample_h_dp4a_kernel<NW4><<<dim3(rows, n), 256, smem, stream>>>(src, row_stride, frame_stride, y0, sx0, sx1, bounds, packed,
                                                                    out_size, x0, cols, tmp, plane_words);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_resample_pack_coeffs(const int32_t* coeffs, int ksize, int out_size, uint32_t* packed) {
  MA_REQUIRE(coeffs && packed && ksize > 0 && out_size > 0, "ma_resample_pack_coeffs: bad arguments");
  const int nw = (ksize + 3) / 4;
  for (int p = 0; p < 3; ++p)
    for (int j = 0; j < nw; ++j)
      for (int xx = 0; xx < out_size; ++xx) {
        uint32_t word = 0;
        for (int b = 0; b < 4; ++b) {
          const int t = 4 * j + b;
          const int32_t k = t < ksize ? coeffs[static_cast<int64_t>(t) * out_size + xx] : 0;
          const int32_t hi = k >> 16;  // arithmetic shift: k = (k & 255) + 256 * ((k >> 8) & 255) + 65536 * hi
          MA_REQUIRE(hi >= -128 && hi <= 127, "ma_resample_pack_coeffs: coefficient %d does not fit 24 signed bits", k);
          const uint32_t byte = p == 0 ? (k & 255) : p == 1 ? ((k >> 8) & 255) : (static_cast<uint32_t>(hi) & 255u);
          word |= byte << (8 * b);
        }
        packed[(static_cast<int64_t>(p) * nw + j) * out_size + xx] = word;
      }
  return MA_OK;
}

extern "C" int ma_resample_h_u8rgb(const uint8_t* src, int64_t src_row_stride, int64_t src_frame_stride, int n, int y0, int rows,
                                   int sx0, int sx1, const int32_t* bounds, const int32_t* coeffs, const uint32_t* packed,
                                   int ksize, int out_size, int x0, int cols, uint8_t* tmp, void* stream) {
  MA_REQUIRE(src && bounds && coeffs && tmp && n > 0 && n <= 65535 && rows > 0 && cols > 0 && sx1 > sx0 && x0 >= 0 &&
                 x0 + cols <= out_size && ksize > 0,
             "ma_resample_h_u8rgb: bad arguments (n=%d rows=%d cols=%d ksize=%d)", n, rows, cols, ksize);
  MA_REQUIRE(sx0 >= 0, "ma_resample_h_u8rgb: sx0=%d is negative", sx0);
  MA_REQUIRE(y0 >= 0, "ma_resample_h_u8rgb: y0=%d is negative", y0);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(bounds) & 3) == 0, "ma_resample_h_u8rgb: bounds not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(coeffs) & 3) == 0, "ma_resample_h_u8rgb: coeffs not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 3) == 0, "ma_resample_h_u8rgb: packed not 4-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t row_bytes = static_cast<int64_t>(sx1 - sx0) * 3;
  if (packed && ksize <= 64 && row_bytes + 1024 <= 180 * 1024) {
#define MA_H_DP4A(W) \
  case W:            \
    return launch_h_dp4a<W>(src, src_row_stride, src_frame_stride, n, y0, rows, sx0, sx1, bounds, packed, out_size, x0, cols, tmp, st)
    switch ((ksize + 3) / 4) {
      MA_H_DP4A(1); MA_H_DP4A(2); MA_H_DP4A(3); MA_H_DP4A(4); MA_H_DP4A(5); MA_H_DP4A(6); MA_H_DP4A(7); MA_H_DP4A(8);
      MA_H_DP4A(9); MA_H_DP4A(10); MA_H_DP4A(11); MA_H_DP4A(12); MA_H_DP4A(13); MA_H_DP4A(14); MA_H_DP4A(15); MA_H_DP4A(16);
      default: break;
    }
#undef MA_H_DP4A
  }
  if (ksize <= 64 && row_bytes + 512 <= 200 * 1024) {
#define MA_H_VEC(K) \
  case K / 4:       \
    return launch_h_vec<K>(src, src_row_stride, src_frame_stride, n, y0, rows, sx0, sx1, bounds, coeffs, out_size, x0, cols, tmp, st)
    switch ((ksize + 3) / 4) {  // unrolled tap count = the window length rounded up to a multiple of 4
      MA_H_VEC(4); MA_H_VEC(8); MA_H_VEC(12); MA_H_VEC(16); MA_H_VEC(20); MA_H_VEC(24); MA_H_VEC(28); MA_H_VEC(32);
      MA_H_VEC(36); MA_H_VEC(40); MA_H_VEC(44); MA_H_VEC(48); MA_H_VEC(52); MA_H_VEC(56); MA_H_VEC(60); MA_H_VEC(64);
      default: break;
    }
#undef MA_H_VEC
  }
  const size_t smem = static_cast<size_t>(row_bytes) + 8;
  MA_REQUIRE(smem <= 200 * 1024, "ma_resample_h_u8rgb: source rows of %d pixels do not fit shared memory", sx1 - sx0);
  if (smem > 48 * 1024) {
    static size_t configured_dev[MA_MAX_DEVICES] = {};
    size_t& configured = configured_dev[current_device()];
    if (smem > configured) {
      MA_CHECK_CUDA(cudaFuncSetAttribute(resample_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      configured = 200 * 1024;
    }
  }
  g_last_resample_kernel = 1;
  resample_h_kernel<<<dim3(rows, n), 256, smem, st>>>(src, src_row_stride, src_frame_stride, y0, sx0, sx1, bounds, coeffs, out_size,
                                                     x0, cols, tmp);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_resample_v_norm_u8rgb(const uint8_t* tmp, int n, int rows, int cols, int y0, const int32_t* bounds,
                                        const int32_t* coeffs, int ksize, int out_size, int top, int th, const float* mean_host,
                                        const float* std_host, float* out_chw, uint8_t* out_u8, void* stream) {
  MA_REQUIRE(tmp && bounds && coeffs && ksize > 0 && n > 0 && n <= 65535 && rows > 0 && cols > 0 && th > 0 && top >= 0 &&
                 top + th <= out_size && (out_chw || out_u8),
             "ma_resample_v_norm_u8rgb: bad arguments (n=%d cols=%d th=%d)", n, cols, th);
  MA_REQUIRE(!out_chw || (mean_host && std_host), "ma_resample_v_norm_u8rgb: mean / std missing");
  MA_REQUIRE(th <= 65535, "ma_resample_v_norm_u8rgb: th=%d above 65535 (one grid row per output row)", th);
  MA_REQUIRE((reinterpret_cast<uintptr_t>(bounds) & 3) == 0, "ma_resample_v_norm_u8rgb: bounds not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(coeffs) & 3) == 0, "ma_resample_v_norm_u8rgb: coeffs not 4-byte aligned");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out_chw) & 3) == 0, "ma_resample_v_norm_u8rgb: out_chw not 4-byte aligned");
  const float m0 = mean_host ? mean_host[0] : 0.f, m1 = mean_host ? mean_host[1] : 0.f, m2 = mean_host ? mean_host[2] : 0.f;
  const float s0 = std_host ? std_host[0] : 1.f, s1 = std_host ? std_host[1] : 1.f, s2 = std_host ? std_host[2] : 1.f;
  dim3 grid((cols + 127) / 128, th, n);
  resample_v_norm_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(tmp, rows, cols, y0, bounds, coeffs, out_size, top, th,
                                                                             m0, m1, m2, s0, s1, s2, out_chw, out_u8);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
