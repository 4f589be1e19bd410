// Persistent, warp-specialised bf16 GEMM / implicit 3x3 conv for sm_100a:  Y = epilogue(X . W^T)
//
// One kernel template, gemm_bf16_kernel<CTAS, BN>, computes a 128 x BN tile on one CTA (CTAS = 1, tcgen05 cta_group::1) or
// a 256 x BN tile on a CTA pair (CTAS = 2, cta_group::2, a cluster of the two SMs of a TPC).
//
//   warp 0      : TMA producer  (cp.async.bulk.tensor, 128B swizzle, STAGES-deep mbarrier ring)
//   warp 1      : MMA issuer    (one thread of the leader CTA, tcgen05.mma kind::f16, M = 128 x CTAS, N = BN, K = 16)
//   warp 2      : TMEM allocator / deallocator
//   warps 4..11 : epilogue      (tcgen05.ld TMEM -> registers -> fused bias/act/scale/residual -> global)
//
// Two fp32 accumulators (2*BN TMEM columns) are double-buffered so the epilogue of tile i overlaps the MMA main loop of
// tile i+1.  Ragged M / N / K edges are handled by TMA out-of-bounds zero fill on the load side and predicated stores on
// the store side.
//
// CTA pair: CTA r loads A rows [m0 + 128 r, +128) and B rows [n0 + BN/2 * r, + BN/2) of every K block; ONE thread of the
// leader CTA issues tcgen05.mma.cta_group::2 with M = 256, N = BN: each SM's tensor core multiplies its own 128 A rows with
// all BN columns, reading the other half of B from the peer SM's shared memory.  Per MMA an SM therefore reads 128x16 A +
// BN/2 x16 B instead of 128x16 + BNx16: at BN = 256 that is 8 KB instead of 12 KB per 128 tensor-core cycles, which is what
// keeps the one-CTA tile below the tensor pipe's rate (shared-memory operand bandwidth, B300_MICROARCH "tcgen05 floor").
// The transaction bytes of both CTAs are credited to the LEADER's full barrier, tcgen05.commit multicasts "stage free" /
// "accumulator ready" to both CTAs, and "accumulator drained" arrives on the leader's barrier from both CTAs.
//
// Stream-K tail (CTA pair; in-place fp32 residual GEMMs, i.e. the reduce-add epilogue, K >= 2048): the tiles of the last,
// partially filled wave are not handed out whole.  Their K blocks form one flattened range that is cut into equal
// contiguous pieces, one per cluster, so every cluster works until (nearly) the same K block: 10960 x 1024 x 4096 on 74
// clusters is 172 tiles = 2 full waves + 24 tiles; whole tiles cost 3 x 64 K blocks per cluster, stream-K 2 x 64 + 21.  A
// piece that covers part of a tile's K range is an ordinary work unit (tile, k0, k1): its partial product leaves through
// the same bulk tensor REDUCE-ADD as a whole tile (x += gamma * acc; the unit that holds K block 0 also adds gamma * bias),
// so no workspace and no fix-up pass exist.  The fp32 adds of one element's two or three partial products reach the L2 in
// arbitrary order: such a GEMM is reproducible to fp32 rounding of the sum (~1e-7 relative), not bit for bit
// (ma_set_stream_k(0) restores that).
#include "host_common.h"
#include "ptx.cuh"

namespace ma {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 384;
constexpr int GEMM_EPI_WARPS = 8;
constexpr int GEMM_SK_MIN_KBLOCKS = 32;  // stream-K only for K >= 2048 (fc2 of the transformer blocks)
constexpr int GEMM_SK_MIN_PIECE = 8;     // ... and pieces of at least 8 K blocks

// Implicit-GEMM geometry of a 3x3 / stride 1 / pad 1 convolution over an NHWC tensor (mode 1).  The A operand of the
// tile (bh x bw output pixels of one image) and of tap (ky,kx) is the input window shifted by (ky-1, kx-1): ONE 4-D TMA
// box {64 channels, bw, bh, 1} whose out-of-bounds pixels (the zero padding) and channels are zero-filled by the TMA
// unit -- no im2col matrix is ever written.  K runs over 9 taps x ceil(C/64) channel blocks.
struct ConvGeom {
  int mode;  // 0 = plain GEMM
  int H, W, C;
  int bw, bh;            // pixel box of one M tile (bw * bh <= 128)
  int tiles_x, tiles_y;  // per image
  int cblocks;           // ceil(C / 64)
};

// Tile raster of the persistent GEMMs: tile t of tiles_m x tiles_n -> (row tile, column tile).  Concurrently running
// workers (CTAs / CTA pairs) take consecutive t.  M-fastest order made every worker of a wave stream a DIFFERENT X row
// tile against the same W panel, so X was re-read once per column panel -- from DRAM when X + residual exceed the L2 (ncu,
// 10960 x 1024 x 4096: 260 MB read for 143 MB algorithmic).  Banded order: `band` row tiles x all column tiles are in flight
// together, column-fastest, so the tiles_n workers sharing an X row tile run at the same time (one DRAM read, L2 hits for
// the rest) while the W panels (a few MB) stay L2 resident.
__device__ __forceinline__ void raster_tile(int t, int tiles_n, int workers, int& tm, int& tn) {
  int band = workers / tiles_n;
  band = band < 1 ? 1 : band;
  const int per_band = band * tiles_n;
  const int b = t / per_band;
  const int r = t - b * per_band;  // the last band is shorter, but every earlier one is full: no special case
  tm = b * band + r / tiles_n;
  tn = r - (r / tiles_n) * tiles_n;
}

// Work units of one cluster: whole tiles t = cluster, cluster + W, ... below sk_lo, then the cluster's piece of the
// flattened (tile, K block) range of the tiles [sk_lo, total_tiles).  Every warp role walks the same sequence.  With
// sk_lo = total_tiles (every launch without a stream-K tail) these are the whole tiles t = cluster, cluster + W, ...
struct UnitWalk {
  int t, W, sk_lo, kblocks;
  int pos, end;  // stream-K piece, in K blocks from the start of tile sk_lo
  __device__ UnitWalk(int cluster, int W_, int total_tiles, int sk_lo_, int kblocks_) : t(cluster), W(W_), sk_lo(sk_lo_), kblocks(kblocks_) {
    const int total = (total_tiles - sk_lo) * kblocks;
    const int piece = (total + W - 1) / W;
    pos = cluster * piece;
    end = pos + piece < total ? pos + piece : total;
  }
  __device__ bool next(int& tile, int& k0, int& k1) {
    if (t < sk_lo) {
      tile = t; k0 = 0; k1 = kblocks;
      t += W;
      return true;
    }
    if (pos >= end) return false;
    const int j = pos / kblocks;
    tile = sk_lo + j;
    k0 = pos - j * kblocks;
    k1 = k0 + (end - pos) < kblocks ? k0 + (end - pos) : kblocks;
    pos += k1 - k0;
    return true;
  }
};

// ----------------------------------------------------------------------------------------------------------------
// Fused epilogue.  The vector path works on one thread's 32 consecutive columns [col0, col0 + 32) of its row; these are
// its steps (bias, column scale: 16-byte aligned [N] fp32 vectors).
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void epi_bias(float (&v)[32], const float* bias, int col0) {
  const float4* b4 = reinterpret_cast<const float4*>(bias + col0);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = __ldg(b4 + j);
    v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
  }
}

// GELU in the erf form when `erf`, else the tanh form (bf16 outputs, see DESIGN.md "GELU").
__device__ __forceinline__ void epi_act(float (&v)[32], int act, bool erf) {
  if (act == MA_ACT_GELU) {
    if (erf) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = gelu_tanh_fast(v[j]);
    }
  } else if (act == MA_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
  }
}

__device__ __forceinline__ void epi_colscale(float (&v)[32], const float* colscale, int col0) {
  const float4* s4 = reinterpret_cast<const float4*>(colscale + col0);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 s = __ldg(s4 + j);
    v[4 * j] *= s.x; v[4 * j + 1] *= s.y; v[4 * j + 2] *= s.z; v[4 * j + 3] *= s.w;
  }
}

// out_relu[out_row, col0 .. col0 + 32) = bf16(max(v, 0))
__device__ __forceinline__ void epi_store_relu(const float (&v)[32], const ma_gemm_epilogue& ep, int out_row, int col0) {
  uint4* o4 = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(ep.out_relu) + (size_t)out_row * ep.ldo_relu + col0);
#pragma unroll
  for (int j = 0; j < 4; ++j)
    o4[j] = make_uint4(pack_bf16x2(fmaxf(v[8 * j], 0.f), fmaxf(v[8 * j + 1], 0.f)),
                       pack_bf16x2(fmaxf(v[8 * j + 2], 0.f), fmaxf(v[8 * j + 3], 0.f)),
                       pack_bf16x2(fmaxf(v[8 * j + 4], 0.f), fmaxf(v[8 * j + 5], 0.f)),
                       pack_bf16x2(fmaxf(v[8 * j + 6], 0.f), fmaxf(v[8 * j + 7], 0.f)));
}

// 32 consecutive output columns of one row: fused epilogue + store.
__device__ __forceinline__ void epilogue_store_chunk(const ma_gemm_epilogue& ep, const uint32_t (&acc)[32], int m,
                                                     int col0, int N) {
  int out_row = m;
  if (ep.rows_per_group_in > 0) {
    int g = m / ep.rows_per_group_in;
    out_row = g * ep.rows_per_group_out + ep.row_offset_out + (m - g * ep.rows_per_group_in);
  }
  const int res_row = ep.residual_row_mod > 0 ? (m % ep.residual_row_mod) : out_row;
  const int nvalid = min(32, N - col0);

  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);

  if (nvalid == 32) {
    if (ep.bias) epi_bias(v, ep.bias, col0);
    const bool act_late = (ep.flags & MA_GEMM_ACT_AFTER_RESIDUAL) != 0;
    const bool relu_early = (ep.flags & MA_GEMM_RELU_OUT_BEFORE_RESIDUAL) != 0;
    if (!act_late) epi_act(v, ep.act, ep.out_dtype == MA_F32);
    if (ep.out_relu && relu_early) epi_store_relu(v, ep, out_row, col0);
    if (ep.colscale) epi_colscale(v, ep.colscale, col0);
    if (ep.residual) {
      if (ep.residual_dtype == MA_F32) {
        const float4* r4 =
            reinterpret_cast<const float4*>(static_cast<const float*>(ep.residual) + (size_t)res_row * ep.ldr + col0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 r = r4[j];
          v[4 * j + 0] += r.x; v[4 * j + 1] += r.y; v[4 * j + 2] += r.z; v[4 * j + 3] += r.w;
        }
      } else {
        const uint4* r4 = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(ep.residual) +
                                                         (size_t)res_row * ep.ldr + col0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 r = r4[j];
          v[8 * j + 0] += bf16_lo(r.x); v[8 * j + 1] += bf16_hi(r.x);
          v[8 * j + 2] += bf16_lo(r.y); v[8 * j + 3] += bf16_hi(r.y);
          v[8 * j + 4] += bf16_lo(r.z); v[8 * j + 5] += bf16_hi(r.z);
          v[8 * j + 6] += bf16_lo(r.w); v[8 * j + 7] += bf16_hi(r.w);
        }
      }
    }
    if (act_late) epi_act(v, ep.act, ep.out_dtype == MA_F32);
    if (ep.out_dtype == MA_F32) {
      float4* o4 = reinterpret_cast<float4*>(static_cast<float*>(ep.out) + (size_t)out_row * ep.ldo + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) o4[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    } else {
      uint4* o4 = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(ep.out) + (size_t)out_row * ep.ldo + col0);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        o4[j] = make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                           pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
    }
    if (ep.out_relu && !relu_early) epi_store_relu(v, ep, out_row, col0);
  } else {
    // ragged N edge: scalar path (fully unrolled + predicated so v[] stays in registers)
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j >= nvalid) continue;
      const int n = col0 + j;
      float x = v[j];
      const bool act_late = (ep.flags & MA_GEMM_ACT_AFTER_RESIDUAL) != 0;
      const bool relu_early = (ep.flags & MA_GEMM_RELU_OUT_BEFORE_RESIDUAL) != 0;
      if (ep.bias) x += __ldg(ep.bias + n);
      if (!act_late) {
        if (ep.act == MA_ACT_GELU) x = gelu_erf(x);
        else if (ep.act == MA_ACT_RELU) x = fmaxf(x, 0.0f);
      }
      if (ep.out_relu && relu_early)
        static_cast<__nv_bfloat16*>(ep.out_relu)[(size_t)out_row * ep.ldo_relu + n] = __float2bfloat16(fmaxf(x, 0.f));
      if (ep.colscale) x *= __ldg(ep.colscale + n);
      if (ep.residual) {
        if (ep.residual_dtype == MA_F32) x += static_cast<const float*>(ep.residual)[(size_t)res_row * ep.ldr + n];
        else x += __bfloat162float(static_cast<const __nv_bfloat16*>(ep.residual)[(size_t)res_row * ep.ldr + n]);
      }
      if (act_late) {
        if (ep.act == MA_ACT_GELU) x = gelu_erf(x);
        else if (ep.act == MA_ACT_RELU) x = fmaxf(x, 0.0f);
      }
      if (ep.out_dtype == MA_F32) static_cast<float*>(ep.out)[(size_t)out_row * ep.ldo + n] = x;
      else static_cast<__nv_bfloat16*>(ep.out)[(size_t)out_row * ep.ldo + n] = __float2bfloat16(x);
      if (ep.out_relu && !relu_early)
        static_cast<__nv_bfloat16*>(ep.out_relu)[(size_t)out_row * ep.ldo_relu + n] = __float2bfloat16(fmaxf(x, 0.f));
    }
  }
}

// Fused narrow head: this thread's 32 accumulator columns [col0, col0 + 32) of its row get bias + activation (GELU in the
// erf form for every output type) and are folded into 8 running dot products with the head weights (shared memory copy
// hw[8][N], read as broadcast float4).
__device__ __forceinline__ void epilogue_head_chunk(const ma_gemm_epilogue& ep, const uint32_t (&acc)[32], int col0, int N,
                                                    const float* __restrict__ hw, float (&h)[8]) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  if (ep.bias) epi_bias(v, ep.bias, col0);
  epi_act(v, ep.act, true);
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const float4* w4 = reinterpret_cast<const float4*>(hw + n * N + col0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 w = w4[j];
      h[n] = fmaf(v[4 * j], w.x, h[n]); h[n] = fmaf(v[4 * j + 1], w.y, h[n]);
      h[n] = fmaf(v[4 * j + 2], w.z, h[n]); h[n] = fmaf(v[4 * j + 3], w.w, h[n]);
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------
// TMA epilogue (plain GEMMs whose output rows are the GEMM rows): the warp's 32 x 32 accumulator chunk gets
// bias / activation / column scale applied per thread (thread = row), is written to a warp-private, hardware-swizzled
// shared-memory stage and leaves the SM as ONE asynchronous bulk tensor store -- or, for the in-place fp32 residual of a
// transformer block (x += gamma * (acc + b)), as a bulk tensor REDUCE-ADD executed at the L2, so the residual stream is
// never read by the SM.  No strided 16-byte stores, no exposed global-load latency in the epilogue warps, ragged
// M handled by TMA clipping.  mode: 1 = store, 2 = reduce-add.  All 32 lanes call; lane 0 issues the TMA.
// ----------------------------------------------------------------------------------------------------------------
constexpr int EPI_STAGE_BYTES = 32 * 32 * 4;

__device__ __forceinline__ void epilogue_tma_chunk(const CUtensorMap* tmap_out, int mode, const ma_gemm_epilogue& ep,
                                                   const uint32_t (&acc)[32], int row0, int col0, uint8_t* stage, int lane,
                                                   bool with_bias) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  if (ep.bias && with_bias) epi_bias(v, ep.bias, col0);
  epi_act(v, ep.act, ep.out_dtype == MA_F32);
  if (ep.colscale) epi_colscale(v, ep.colscale, col0);
  // the previous bulk store of this warp must have finished reading the stage
  if (lane == 0) tma_store_wait_read<0>();
  __syncwarp();
  if (ep.out_dtype == MA_F32) {
    // rows of 128 B, SWIZZLE_128B: 16-byte chunk q of row r lives at r*128 + ((q ^ (r & 7)) << 4)
    uint4* row = reinterpret_cast<uint4*>(stage + lane * 128);
#pragma unroll
    for (int q = 0; q < 8; ++q)
      row[q ^ (lane & 7)] = make_uint4(__float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]), __float_as_uint(v[4 * q + 2]),
                                       __float_as_uint(v[4 * q + 3]));
  } else {
    // rows of 64 B, SWIZZLE_64B: chunk q of row r lives at r*64 + ((q ^ ((r >> 1) & 3)) << 4)
    uint4* row = reinterpret_cast<uint4*>(stage + lane * 64);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      row[q ^ ((lane >> 1) & 3)] = make_uint4(pack_bf16x2(v[8 * q], v[8 * q + 1]), pack_bf16x2(v[8 * q + 2], v[8 * q + 3]),
                                              pack_bf16x2(v[8 * q + 4], v[8 * q + 5]), pack_bf16x2(v[8 * q + 6], v[8 * q + 7]));
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (mode == 2) tma_reduce_add_2d(tmap_out, stage, col0, row0);
    else tma_store_2d(tmap_out, stage, col0, row0);
    tma_store_commit();
  }
}

// Host side: can this launch use the TMA epilogue, and in which mode (0 = no)?
static int tma_epilogue_mode(const ma_gemm_epilogue& ep, int N) {
  if (ep.rows_per_group_in != 0 || ep.residual_row_mod != 0 || ep.out_relu != nullptr || N % 32 != 0) return 0;
  if ((ep.flags & (MA_GEMM_ACT_AFTER_RESIDUAL | MA_GEMM_RELU_OUT_BEFORE_RESIDUAL)) != 0) return 0;
  const int64_t esz = ep.out_dtype == MA_F32 ? 4 : 2;
  if ((ep.ldo * esz) % 16 != 0 || (reinterpret_cast<uintptr_t>(ep.out) & 15) != 0) return 0;
  if (ep.residual == nullptr) return 1;
  if (ep.residual == ep.out && ep.residual_dtype == MA_F32 && ep.out_dtype == MA_F32 && ep.ldr == ep.ldo) return 2;
  return 0;
}

// ----------------------------------------------------------------------------------------------------------------
// The kernel
// ----------------------------------------------------------------------------------------------------------------
template <int CTAS, int BN>
struct GemmCfg {
  static constexpr int STAGES = CTAS == 2 ? (BN == 256 ? 6 : 8) : (BN == 256 ? 4 : (BN == 128 ? 6 : 8));
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;       // this CTA's 128 rows
  static constexpr int B_BYTES = BN / CTAS * GEMM_BK * 2;     // this CTA's share of the BN rows
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_BYTES = 1024;  // barrier block, padded so that the epilogue stages stay 1024-byte aligned
  static constexpr int EPI_BYTES = GEMM_EPI_WARPS * EPI_STAGE_BYTES;  // fused head: reused as hw[8][128] + partial sums
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + EPI_BYTES + 1024;  // +1024: manual alignment slack
  static constexpr int TMEM_COLS = 2 * BN;                                   // 128 / 256 / 512: powers of two
};

template <int CTAS, int BN>
__global__ void __cluster_dims__(CTAS, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                 const __grid_constant__ CUtensorMap tmap_out, const ma_gemm_epilogue ep, const int M, const int N, const int K,
                 const ConvGeom cg, const int epi_mode, const int sk_lo) {
  using Cfg = GemmCfg<CTAS, BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* bar_empty = bar_full + STAGES;
  uint64_t* bar_tfull = bar_empty + STAGES;
  uint64_t* bar_tempty = bar_tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);
  uint8_t* sEpi = smem + STAGES * Cfg::STAGE_BYTES + Cfg::BAR_BYTES;  // 8 x 4 KB TMA-store stages (1024-byte aligned)

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = lane_id();
  const uint32_t cta = CTAS == 2 ? cluster_ctarank() : 0;  // 0 = leader
  const int cluster_id = blockIdx.x / CTAS;
  const int num_clusters = gridDim.x / CTAS;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_x);
    prefetch_tmap(&tmap_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&bar_full[s], 1);   // the leader's arrive.expect_tx; bytes from every CTA
      mbar_init(&bar_empty[s], 1);  // tcgen05.commit (multicast to both CTAs of a pair)
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bar_tfull[a], 1);                         // tcgen05.commit (multicast to both CTAs of a pair)
      mbar_init(&bar_tempty[a], CTAS * GEMM_EPI_WARPS);    // epilogue warps of every CTA (pair: used on the leader only)
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 2) {
      tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  // pair: barriers of both CTAs initialised before any remote signal; TMEM allocated in both
  if constexpr (CTAS == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();  // prologue above overlaps the previous kernel's tail; no global memory access before this point

  const int tiles_per_img = cg.tiles_x * cg.tiles_y;
  const int rows_tiles = cg.mode ? (M / (cg.H * cg.W)) * tiles_per_img : (M + GEMM_BM - 1) / GEMM_BM;  // 128-row tiles
  const int tiles_m = (rows_tiles + CTAS - 1) / CTAS;                                                   // 128 x CTAS rows
  const int tiles_n = (N + BN - 1) / BN;
  const int total_tiles = tiles_m * tiles_n;
  const int kblocks = cg.mode ? 9 * cg.cblocks : (K + GEMM_BK - 1) / GEMM_BK;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      UnitWalk walk(cluster_id, num_clusters, total_tiles, sk_lo, kblocks);
      int t, k0, k1;
      while (walk.next(t, k0, k1)) {
        int tm2, tn;
        raster_tile(t, tiles_n, num_clusters, tm2, tn);
        const int tm = tm2 * CTAS + static_cast<int>(cta);  // this CTA's 128-row tile
        const int n0 = tn * BN + static_cast<int>(cta) * (BN / CTAS);
        if (cg.mode) {
          // a pair's row tile past the end (odd tile count) reads image index n: fully out of bounds -> zero fill
          const int img = tm / tiles_per_img;
          const int r = tm - img * tiles_per_img;
          const int y0 = (r / cg.tiles_x) * cg.bh, x0 = (r % cg.tiles_x) * cg.bw;
          const uint32_t bytes = CTAS * (static_cast<uint32_t>(cg.bw * cg.bh * 128) + Cfg::B_BYTES);
          for (int tap = 0; tap < 9; ++tap) {
            const int dy = tap / 3 - 1, dx = tap % 3 - 1;
            for (int cb = 0; cb < cg.cblocks; ++cb) {
              mbar_wait(&bar_empty[stage], phase ^ 1);
              if (cta == 0) mbar_arrive_expect_tx(&bar_full[stage], bytes);
              if constexpr (CTAS == 2) {
                tma_load_4d_2sm(sA + stage * Cfg::A_BYTES, &tmap_x, &bar_full[stage], cb * GEMM_BK, x0 + dx, y0 + dy, img);
                tma_load_2d_2sm(sB + stage * Cfg::B_BYTES, &tmap_w, &bar_full[stage], tap * cg.C + cb * GEMM_BK, n0);
              } else {
                tma_load_4d(sA + stage * Cfg::A_BYTES, &tmap_x, &bar_full[stage], cb * GEMM_BK, x0 + dx, y0 + dy, img);
                tma_load_2d(sB + stage * Cfg::B_BYTES, &tmap_w, &bar_full[stage], tap * cg.C + cb * GEMM_BK, n0);
              }
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        } else {
          const int m0 = tm * GEMM_BM;
          for (int kb = k0; kb < k1; ++kb) {
            mbar_wait(&bar_empty[stage], phase ^ 1);
            if (cta == 0) mbar_arrive_expect_tx(&bar_full[stage], CTAS * Cfg::STAGE_BYTES);
            if constexpr (CTAS == 2) {
              tma_load_2d_2sm(sA + stage * Cfg::A_BYTES, &tmap_x, &bar_full[stage], kb * GEMM_BK, m0);
              tma_load_2d_2sm(sB + stage * Cfg::B_BYTES, &tmap_w, &bar_full[stage], kb * GEMM_BK, n0);
            } else {
              tma_load_2d(sA + stage * Cfg::A_BYTES, &tmap_x, &bar_full[stage], kb * GEMM_BK, m0);
              tma_load_2d(sB + stage * Cfg::B_BYTES, &tmap_w, &bar_full[stage], kb * GEMM_BK, n0);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (cta == 0 && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(CTAS * GEMM_BM, BN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      UnitWalk walk(cluster_id, num_clusters, total_tiles, sk_lo, kblocks);
      int t, k0, k1;
      for (int it = 0; walk.next(t, k0, k1); ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        if constexpr (CTAS == 2) mbar_wait_cluster(&bar_tempty[acc], acc_phase ^ 1);
        else mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = k0; kb < k1; ++kb) {
          mbar_wait(&bar_full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sA + stage * Cfg::A_BYTES);
          const uint32_t b_addr = smem_u32(sB + stage * Cfg::B_BYTES);
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            const uint64_t adesc = make_smem_desc_sw128(a_addr + k * 32, 16, 1024);
            const uint64_t bdesc = make_smem_desc_sw128(b_addr + k * 32, 16, 1024);
            const uint32_t accumulate = (kb != k0 || k != 0) ? 1u : 0u;
            if constexpr (CTAS == 2) umma_bf16_ss_2sm(d_tmem, adesc, bdesc, idesc, accumulate);
            else umma_bf16_ss(d_tmem, adesc, bdesc, idesc, accumulate);
          }
          if constexpr (CTAS == 2) umma_commit_2sm(&bar_empty[stage], 0x3);
          else umma_commit(&bar_empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (CTAS == 2) umma_commit_2sm(&bar_tfull[acc], 0x3);
        else umma_commit(&bar_tfull[acc]);
      }
    }
  } else if (warp >= 4) {
    uint8_t* epi_stage = sEpi + (warp - 4) * EPI_STAGE_BYTES;
    const int quarter = warp & 3;       // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;   // which half of the BN columns this warp drains
    const uint32_t leader_tempty0 = CTAS == 2 ? mapa_shared(smem_u32(&bar_tempty[0]), 0) : 0;
    // fused narrow head (pair, BN == 128 only): the epilogue stages are free (no TMA epilogue in this mode): stage 0 .. 3
    // hold the head weights hw[8][128] fp32 (4 KB), stages 4 .. 7 the partial sums of the upper column half,
    // [tile parity][row][8]
    const bool head = CTAS == 2 && BN == 128 && ep.head_out != nullptr;
    float* hw = reinterpret_cast<float*>(sEpi);
    float* hpart = reinterpret_cast<float*>(sEpi + 4 * EPI_STAGE_BYTES);  // [2][128][8] fp32 = 8 KB
    if (head) {
      for (int i = threadIdx.x - 128; i < 8 * BN; i += GEMM_EPI_WARPS * 32) hw[i] = __ldg(ep.head_w + i);
      named_bar_sync(1, GEMM_EPI_WARPS * 32);
    }
    UnitWalk walk(cluster_id, num_clusters, total_tiles, sk_lo, kblocks);
    int t, k0, k1;
    for (int it = 0; walk.next(t, k0, k1); ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      int tm2, tn;
      raster_tile(t, tiles_n, num_clusters, tm2, tn);
      const int tm = tm2 * CTAS + static_cast<int>(cta);
      const int n0 = tn * BN;
      // output row of this thread's accumulator lane: tile row r = quarter*32 + lane
      int m;
      bool row_ok;
      if (cg.mode) {
        const int img = tm / tiles_per_img;
        const int rr = tm - img * tiles_per_img;
        const int r = quarter * 32 + lane;
        const int y = (rr / cg.tiles_x) * cg.bh + r / cg.bw, x = (rr % cg.tiles_x) * cg.bw + r % cg.bw;
        row_ok = (CTAS == 1 || tm < rows_tiles) && r < cg.bw * cg.bh && y < cg.H && x < cg.W;
        m = (img * cg.H + y) * cg.W + x;
      } else {
        m = tm * GEMM_BM + quarter * 32 + lane;
        row_ok = m < M;
      }
      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      float hsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
      for (int c = 0; c < BN / 2; c += 32) {
        const int col0 = n0 + half * (BN / 2) + c;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN + half * (BN / 2) + c;
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr, v);
        tmem_ld_wait();
        if (head) {
          epilogue_head_chunk(ep, v, col0, BN, hw, hsum);
        } else if (epi_mode) {  // warp-uniform: asynchronous bulk tensor store / reduce-add of the 32 x 32 chunk
          // a stream-K unit that does not hold K block 0 contributes gamma * partial product only (no bias)
          if (col0 < N) epilogue_tma_chunk(&tmap_out, epi_mode, ep, v, tm * GEMM_BM + quarter * 32, col0, epi_stage, lane, k0 == 0);
        } else if (row_ok && col0 < N) {
          epilogue_store_chunk(ep, v, m, col0, N);
        }
      }
      tc_fence_before();
      __syncwarp();
      // the accumulator is drained: the next tile's MMAs may start
      if (lane == 0) {
        if constexpr (CTAS == 2) mbar_arrive_remote(leader_tempty0 + acc * 8);
        else mbar_arrive(&bar_tempty[acc]);
      }
      if (head) {
        // the two warps that own the same 32 rows (column halves 0 / 1) meet at a 64-thread named barrier: the upper half
        // hands its 8 partial sums over through shared memory (double-buffered by tile parity), the lower half adds the
        // head bias and writes 8 fp32 per pixel (consecutive rows -> 1 KB contiguous per warp)
        float* mine = hpart + ((it & 1) * 128 + quarter * 32 + lane) * 8;
        if (half == 1) {
          *reinterpret_cast<float4*>(mine) = make_float4(hsum[0], hsum[1], hsum[2], hsum[3]);
          *reinterpret_cast<float4*>(mine + 4) = make_float4(hsum[4], hsum[5], hsum[6], hsum[7]);
        }
        named_bar_sync(2 + quarter, 64);
        if (half == 0 && row_ok) {
          const float4 a = *reinterpret_cast<const float4*>(mine), b = *reinterpret_cast<const float4*>(mine + 4);
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(ep.head_bias)), b1 = __ldg(reinterpret_cast<const float4*>(ep.head_bias) + 1);
          float4* o = reinterpret_cast<float4*>(ep.head_out + static_cast<size_t>(m) * 8);
          o[0] = make_float4(hsum[0] + a.x + b0.x, hsum[1] + a.y + b0.y, hsum[2] + a.z + b0.z, hsum[3] + a.w + b0.w);
          o[1] = make_float4(hsum[4] + b.x + b1.x, hsum[5] + b.y + b1.y, hsum[6] + b.z + b1.z, hsum[7] + b.w + b1.w);
        }
      }
    }
    if (epi_mode && lane == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  // pair: the peer's smem / TMEM stay alive until the leader's last MMA and all remote arrives are done
  if constexpr (CTAS == 2) cluster_sync_all();
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CTAS == 2) tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
    else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// rows_tiles: 128-row tiles of the output (of the pixel boxes for a conv)
template <int CTAS, int BN>
static int launch_gemm(const CUtensorMap& tx, const CUtensorMap& tw, const CUtensorMap& tout, int epi_mode,
                       const ma_gemm_epilogue& ep, int M, int N, int K, int rows_tiles, cudaStream_t stream, const ConvGeom& cg) {
  using Cfg = GemmCfg<CTAS, BN>;
  static bool configured_dev[MA_MAX_DEVICES] = {};
  bool& configured = configured_dev[current_device()];
  if (!configured) {
    MA_CHECK_CUDA(cudaFuncSetAttribute(gemm_bf16_kernel<CTAS, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    configured = true;
  }
  const int tiles = ((rows_tiles + CTAS - 1) / CTAS) * ((N + BN - 1) / BN);
  const int max_clusters = device_sm_count() / CTAS;
  int clusters = tiles < max_clusters ? tiles : max_clusters;
  // stream-K over the last partial wave (CTA pairs): only where a partial product can leave as a reduce-add (epi_mode 2, no
  // activation) and the K range is long enough for a piece to amortise its own epilogue
  int sk_lo = tiles;
  const int kblocks = (K + GEMM_BK - 1) / GEMM_BK;
  if (CTAS == 2 && stream_k_enabled() && epi_mode == 2 && !cg.mode && ep.act == MA_ACT_NONE && kblocks >= GEMM_SK_MIN_KBLOCKS &&
      tiles % max_clusters != 0) {
    const int tail = tiles % max_clusters;
    if ((tail * kblocks + max_clusters - 1) / max_clusters >= GEMM_SK_MIN_PIECE) {
      sk_lo = tiles - tail;
      clusters = max_clusters;
    }
  }
  MA_CHECK_CUDA(launch_kernel(gemm_bf16_kernel<CTAS, BN>, dim3(CTAS * clusters), dim3(GEMM_THREADS), Cfg::SMEM_BYTES, stream,
                              pdl_enabled(), tx, tw, tout, ep, M, N, K, cg, epi_mode, sk_lo));
  return MA_OK;
}

// Block codes accepted as `block_n`: 64 / 128 / 256 = one CTA per 128 x block_n tile; PAIR_CODE + 128 / 256 = a CTA pair
// per 256 x bn tile.
constexpr int PAIR_CODE = 2000;

constexpr double G2_COST_256 = 0.82, G2_COST_128 = 0.56;

static int pick_block_n(int tiles_m, int N) {
  const int sms = device_sm_count();
  int best = 128;
  double best_cost = 1e30;
  const int cands[3] = {256, 128, 64};
  for (int i = 0; i < 3; ++i) {
    const int bn = cands[i];
    const int tiles = tiles_m * ((N + bn - 1) / bn);
    const int waves = (tiles + sms - 1) / sms;
    // measured on B200 (tools/bench_kernels.py): a 128-wide tile runs at ~75% and a 64-wide tile at ~43% of
    // the 256-wide tile's MMA rate (smem operand bandwidth), so per-tile cost is not proportional to BN.
    const double cost = waves * (bn == 256 ? 1.0 : (bn == 128 ? 0.66 : 0.58));
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  // CTA pairs: 256 x bn tiles over sms/2 clusters.  Per-tile cost relative to a 1-CTA 128x256 tile (measured on B200,
  // tools/bench_kernels.py): the pair tile does twice the work at the full tensor rate (operand traffic per SM is 2/3).
  const int pcands[2] = {256, 128};
  for (int i = 0; i < 2; ++i) {
    const int bn = pcands[i];
    const int tiles = ((tiles_m + 1) / 2) * ((N + bn - 1) / bn);
    const int clusters = sms / 2;
    const int waves = (tiles + clusters - 1) / clusters;
    const double cost = waves * (bn == 256 ? G2_COST_256 : G2_COST_128);
    if (cost < best_cost) { best_cost = cost; best = PAIR_CODE + bn; }
  }
  return best;
}

thread_local int g_last_block = 0;

static bool valid_block_code(int bn) {
  return bn == 64 || bn == 128 || bn == 256 || bn == PAIR_CODE + 128 || bn == PAIR_CODE + 256;
}

// The steps both entry points share: take the block code (or choose one), check and record it, encode the weight tensor
// map (w: [N][K] bf16, row stride ldw; box: this CTA's share of the tile's columns) and launch.  tout is unused when
// epi_mode == 0.
static int run_gemm(const char* who, int block_n, const void* w, int64_t ldw, const CUtensorMap& tx, const CUtensorMap& tout,
                    int epi_mode, const ma_gemm_epilogue& ep, int M, int N, int K, int rows_tiles, cudaStream_t s,
                    const ConvGeom& cg) {
  const int code = block_n ? block_n : pick_block_n(rows_tiles, N);
  MA_REQUIRE(valid_block_code(code), "%s: bad block_n %d", who, block_n);
  g_last_block = code;
  const int ctas = code > PAIR_CODE ? 2 : 1;
  CUtensorMap tw;
  uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
  uint64_t strides[1] = {(uint64_t)ldw * 2};
  uint32_t box[2] = {GEMM_BK, (uint32_t)(code % PAIR_CODE / ctas)};
  const int rc = make_tmap_bf16(&tw, w, 2, dims, strides, box);
  if (rc != MA_OK) return rc;
  switch (code) {
    case 64: return launch_gemm<1, 64>(tx, tw, tout, epi_mode, ep, M, N, K, rows_tiles, s, cg);
    case 128: return launch_gemm<1, 128>(tx, tw, tout, epi_mode, ep, M, N, K, rows_tiles, s, cg);
    case 256: return launch_gemm<1, 256>(tx, tw, tout, epi_mode, ep, M, N, K, rows_tiles, s, cg);
    case PAIR_CODE + 128: return launch_gemm<2, 128>(tx, tw, tout, epi_mode, ep, M, N, K, rows_tiles, s, cg);
    default: return launch_gemm<2, 256>(tx, tw, tout, epi_mode, ep, M, N, K, rows_tiles, s, cg);
  }
}

}  // namespace ma

// Every full 32-column chunk of a row takes the vector path (16-byte loads of bias / colscale / residual, 16-byte stores of
// out / out_relu), also when a ragged last chunk follows it: so with N >= 32 every epilogue operand must be 16-byte
// aligned at each row.  With N < 32 the only chunk is the scalar path, which has no alignment needs.
static int check_epilogue(const ma_gemm_epilogue* epi, int N, const char* who) {
  if (N < 32) return MA_OK;
  const int64_t oalign = epi->out_dtype == MA_F32 ? 4 : 8;
  MA_REQUIRE(epi->ldo % oalign == 0 && (reinterpret_cast<uintptr_t>(epi->out) & 15) == 0,
             "%s: output not 16-byte aligned (ldo=%lld)", who, (long long)epi->ldo);
  if (epi->residual) {
    const int64_t ralign = epi->residual_dtype == MA_F32 ? 4 : 8;
    MA_REQUIRE(epi->ldr % ralign == 0 && (reinterpret_cast<uintptr_t>(epi->residual) & 15) == 0,
               "%s: residual not 16-byte aligned (ldr=%lld)", who, (long long)epi->ldr);
  }
  if (epi->out_relu)
    MA_REQUIRE(epi->ldo_relu % 8 == 0 && (reinterpret_cast<uintptr_t>(epi->out_relu) & 15) == 0,
               "%s: out_relu not 16-byte aligned (ldo_relu=%lld)", who, (long long)epi->ldo_relu);
  if (epi->bias) MA_REQUIRE((reinterpret_cast<uintptr_t>(epi->bias) & 15) == 0, "%s: bias not 16-byte aligned", who);
  if (epi->colscale)
    MA_REQUIRE((reinterpret_cast<uintptr_t>(epi->colscale) & 15) == 0, "%s: colscale not 16-byte aligned", who);
  return MA_OK;
}

extern "C" int ma_conv3x3_bf16(const void* x, int n, int H, int W, int C, const void* w, int64_t ldw, int Cout,
                               const ma_gemm_epilogue* epi, int block_n, void* stream) {
  using namespace ma;
  MA_REQUIRE(x && w && epi && (epi->out || epi->head_out), "ma_conv3x3_bf16: null pointer");
  MA_REQUIRE(n > 0 && H > 0 && W > 0 && C > 0 && Cout > 0, "ma_conv3x3_bf16: bad shape");
  const bool head = epi->head_out != nullptr;
  if (head) {  // fused narrow head: the tile values feed 8 dot products instead of being stored
    MA_REQUIRE(Cout == 128 && (block_n == 0 || block_n == PAIR_CODE + 128),
               "ma_conv3x3_bf16: the fused head needs Cout == 128 and the CTA-pair 256x128 tile (block_n 0 / 2128)");
    MA_REQUIRE(epi->head_w && epi->head_bias && (reinterpret_cast<uintptr_t>(epi->head_w) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(epi->head_bias) & 15) == 0 && (reinterpret_cast<uintptr_t>(epi->head_out) & 15) == 0,
               "ma_conv3x3_bf16: fused head weights / bias / output missing or not 16-byte aligned");
    MA_REQUIRE(!epi->residual && !epi->colscale && !epi->out_relu && epi->flags == 0,
               "ma_conv3x3_bf16: the fused head takes bias + activation only");
    block_n = PAIR_CODE + 128;
  }
  MA_REQUIRE(C % 8 == 0 && ldw % 8 == 0 && ldw >= 9 * (int64_t)C, "ma_conv3x3_bf16: C / ldw must be multiples of 8, ldw >= 9C");
  MA_REQUIRE((int64_t)n * H * W < (1ll << 31), "ma_conv3x3_bf16: too many pixels");
  MA_REQUIRE(epi->rows_per_group_in == 0, "ma_conv3x3_bf16: row remapping is not supported");
  int rc = head ? MA_OK : check_epilogue(epi, Cout, "ma_conv3x3_bf16");
  if (rc != MA_OK) return rc;

  // pixel box of one M tile: maximise useful rows / 128 over all bw x bh <= 128 boxes
  ConvGeom cg;
  cg.mode = 1; cg.H = H; cg.W = W; cg.C = C;
  double best = -1.0;
  for (int bw = 1; bw <= 128 && bw <= W; ++bw) {
    int bh = 128 / bw;
    if (bh > H) bh = H;
    const int tx = (W + bw - 1) / bw, ty = (H + bh - 1) / bh;
    const double eff = (double)W * H / ((double)tx * ty * 128.0);
    if (eff > best + 1e-9) { best = eff; cg.bw = bw; cg.bh = bh; cg.tiles_x = tx; cg.tiles_y = ty; }
  }
  cg.cblocks = (C + GEMM_BK - 1) / GEMM_BK;

  CUtensorMap tx;
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)n};
  uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
  uint32_t box[4] = {GEMM_BK, (uint32_t)cg.bw, (uint32_t)cg.bh, 1};
  rc = make_tmap_bf16(&tx, x, 4, dims, strides, box);
  if (rc != MA_OK) return rc;
  return run_gemm("ma_conv3x3_bf16", block_n, w, ldw, tx, tx, 0, *epi, n * H * W, Cout, 9 * C, n * cg.tiles_x * cg.tiles_y,
                  static_cast<cudaStream_t>(stream), cg);
}

extern "C" int ma_last_gemm_block(void) { return ma::g_last_block; }

extern "C" int ma_gemm_bf16(const void* x, int64_t ldx, const void* w, int64_t ldw, int M, int N, int K,
                            const ma_gemm_epilogue* epi, int block_n, void* stream) {
  using namespace ma;
  MA_REQUIRE(x && w && epi && epi->out, "ma_gemm_bf16: null pointer");
  MA_REQUIRE(epi->head_out == nullptr, "ma_gemm_bf16: the fused narrow head is implemented for ma_conv3x3_bf16 only");
  MA_REQUIRE(M > 0 && N > 0 && K > 0, "ma_gemm_bf16: bad shape M=%d N=%d K=%d", M, N, K);
  MA_REQUIRE(K % 8 == 0 && ldx % 8 == 0 && ldw % 8 == 0, "ma_gemm_bf16: K/ldx/ldw must be multiples of 8 (K=%d ldx=%lld ldw=%lld)",
             K, (long long)ldx, (long long)ldw);
  MA_REQUIRE(ldx >= K && ldw >= K, "ma_gemm_bf16: leading dimension smaller than K");
  int rc = check_epilogue(epi, N, "ma_gemm_bf16");
  if (rc != MA_OK) return rc;

  CUtensorMap tx;
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
    uint64_t strides[1] = {(uint64_t)ldx * 2};
    uint32_t box[2] = {GEMM_BK, GEMM_BM};
    rc = make_tmap_bf16(&tx, x, 2, dims, strides, box);
    if (rc != MA_OK) return rc;
  }
  // TMA epilogue (bulk tensor store / reduce-add) whenever the output rows are the GEMM rows
  const int epi_mode = tma_epilogue_mode(*epi, N);
  CUtensorMap tout = tx;
  if (epi_mode) {
    const bool f32 = epi->out_dtype == MA_F32;
    uint64_t dims[2] = {(uint64_t)N, (uint64_t)M};
    uint64_t strides[1] = {(uint64_t)epi->ldo * (f32 ? 4 : 2)};
    uint32_t box[2] = {32, 32};
    rc = make_tmap(&tout, epi->out, f32 ? MA_F32 : MA_BF16, 2, dims, strides, box, f32 ? 128 : 64);
    if (rc != MA_OK) return rc;
  }
  return run_gemm("ma_gemm_bf16", block_n, w, ldw, tx, tout, epi_mode, *epi, M, N, K, (M + GEMM_BM - 1) / GEMM_BM,
                  static_cast<cudaStream_t>(stream), ConvGeom{});
}
