// Flash-style attention forward for sm_100a (head_dim 64, bf16 in/out, fp32 softmax + accumulate).
//
// Three forward kernels share one pipeline: a TMA producer warp streams Q once and K / V tiles through an mbarrier ring, an
// MMA issuer warp computes S = Q.K^T (tcgen05.mma, K-major A / B) into tensor memory and accumulates O += P.V in tensor
// memory (A = P from tensor memory, B = V MN-major), and a softmax warpgroup -- one query row per thread -- reads S into
// registers, exponentiates it against a lazily updated integer reference maximum and writes P (bf16 pairs) to tensor memory.
//   v2  two 128-row query tiles per CTA sharing every K / V tile, one CTA per SM, 128-key steps, the exponential phases of
//       the two softmax warpgroups alternating (ping-pong): long sequences, key segments, carried state, kv split;
//   v3  one query tile per CTA, three CTAs per SM, 64-key steps: up to 4096 keys when v5 does not apply;
//   v5  persistent CTAs with two independent query-tile streams in ping-pong: plain attention over many short sequences.
// attention_merge_kernel joins partial softmax states (kv split, view-sharded global attention).  ma_attention_fwd_ex picks
// the kernel from the call's shape (the measurements behind each threshold are given there).
//
// Sequences are contiguous row ranges of a token-major matrix ([tokens][heads*64] slices of the fused
// qkv GEMM output, so no head permute/copy is ever materialised).  Keys past kv_len are masked to -inf
// (TMA zero-fills rows beyond the tensor; rows that belong to the next sequence are masked the same way).
#include "host_common.h"
#include "ptx.cuh"

namespace ma {

constexpr int ATT_BM = 128;
constexpr int ATT_BN = 128;
constexpr int ATT_D = 64;
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KB: a Q tile or a 128-row K / V stage

struct AttnParams {
  __nv_bfloat16* out;
  int64_t ldo;
  int q_len;
  int64_t q_seq_stride, kv_seq_stride;  // rows between consecutive sequences
  int q_col0, k_col0, v_col0, o_col0;   // column of head 0 in the respective matrices
  float scale_log2;                     // softmax scale * log2(e)
  // The keys of a sequence are the concatenation of n_segs row ranges [seg_row0[s], seg_row0[s] + seg_len[s]) (relative
  // to the sequence's first kv row): one range for ordinary attention, one per source rank for the view-sharded
  // global attention whose K/V were all-gathered into per-rank slots of a padded buffer.
  int n_segs, n_kv_tiles;
  int seg_row0[MA_ATTN_MAX_SEGMENTS];
  int seg_len[MA_ATTN_MAX_SEGMENTS];
  // Online-softmax state carried between launches (fp32): o = normalised output so far, m = reference maximum in raw
  // score units with the running sum folded in (m' = m + log2(l) / scale_log2), i.e. the state (o, m', l = 1).
  float* state_o;
  int64_t ld_state_o;
  float* state_m;  // [q_rows][num_heads]
  int num_heads, num_seqs;
  int flags;  // MA_ATTN_STATE_IN / MA_ATTN_STATE_OUT
  // kv_split > 1: the kv tile range is cut into kv_split equal parts, each handled by its own CTA, which writes its
  // partial softmax state to state_o + part * split_stride_o / state_m + part * split_stride_m (ma_attention_merge joins
  // them).  Doubles / triples the CTA count when (query blocks x heads) fills the last wave of SMs badly.
  // v2 alternates the exponential phases of its two query tiles whenever it has two; the host always sets 1.  Read at run
  // time on purpose: with the condition known at compile time ptxas schedules v2's exponential phase differently and the
  // kernel measured ~1.3 % slower on the global-attention shapes (B200, same-box A/B).
  int pingpong;
  int kv_split, split_from;  // CTAs of slots >= split_from are split (tail-only splitting); 0 = every slot
  int64_t split_stride_o, split_stride_m;
};

// Cursor over the BN-row kv tiles of all segments, in segment order.
template <int BN>
struct KvCursor {
  int seg = 0, jj = 0;
  __device__ __forceinline__ int row0(const AttnParams& p) const { return p.seg_row0[seg] + jj * BN; }
  __device__ __forceinline__ int valid(const AttnParams& p) const { return p.seg_len[seg] - jj * BN; }
  __device__ __forceinline__ void next(const AttnParams& p) {
    if ((jj + 1) * BN < p.seg_len[seg]) ++jj;
    else { ++seg; jj = 0; }
  }
  __device__ __forceinline__ void skip(const AttnParams& p, int n) {
    for (int i = 0; i < n; ++i) next(p);
  }
};

// ================================================================================================================
// Softmax-row steps shared by the kernels.  A softmax thread owns one query row; mref is the row's reference maximum in
// log2 units (score * scale * log2 e), kept INTEGER valued.  Any reference works (it cancels in O / l), so the true running
// maximum is only tracked to within the lazy-rescale slack.
// ================================================================================================================
constexpr float A2_RESCALE_LOG2 = 8.0f;

// Exponentials of one 32-column chunk of a score row (16 register pairs) -> 16 packed bf16x2 probabilities + row-sum
// contribution, p = 2^(s * sl2 - mref) on the MUFU; all arithmetic that can be is issued as packed fp32x2 (half the issue
// slots).
__device__ __forceinline__ void a2_exp_chunk(const uint32_t (&v)[32], uint32_t* dst, uint64_t sl2_2, uint64_t nm2,
                                             uint64_t (&acc)[4]) {
  // Written stage by stage over all pairs of the chunk (not pair by pair): every stage is a run of independent
  // instructions.  (ptxas re-schedules the result freely -- the SASS consumes each pair of exponentials two MUFU
  // instructions after issuing them whatever the source order, volatile asm included.)
  constexpr int AHEAD = 1;
  uint64_t s2[16];
  float ea[16], eb[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) s2[i] = ffma2(pack2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), sl2_2, nm2);
  auto evaluate = [&](int i) {
    unpack2(s2[i], ea[i], eb[i]);
    ea[i] = fast_exp2(ea[i]);
    eb[i] = fast_exp2(eb[i]);
  };
#pragma unroll
  for (int i = 0; i < AHEAD; ++i) evaluate(i);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if (i + AHEAD < 16) evaluate(i + AHEAD);
    acc[i & 3] = fadd2(acc[i & 3], pack2(ea[i], eb[i]));
    dst[i] = pack_bf16x2(ea[i], eb[i]);
  }
}

// MUFU-only exponentials of a whole 128-score row with the consumption of the results software-pipelined one 32-score chunk
// behind their issue.  ptxas' own order puts the sum / pack of pair i two MUFU instructions behind pair i (16 clk of MUFU time,
// less than the MUFU latency), so a warp alone drives the pipe at ~2/3 of its rate (ncu: a single warp's exponential phase takes
// 1.5x the MUFU time).  Here chunk c+1's exponentials are issued BEFORE chunk c's results are summed, packed and stored, with a
// warp-level fence between the groups so that the order survives instruction scheduling.
template <typename StoreFn, typename HandoverFn>
__device__ __forceinline__ void a2_exp_row_pipelined(uint32_t (&v0)[32], uint32_t (&v1)[32], uint32_t (&v2)[32], uint32_t (&v3)[32],
                                                     float sl2, float mref, uint64_t (&acc)[4], StoreFn&& store,
                                                     HandoverFn&& handover) {
  auto issue = [&](uint32_t (&v)[32]) {   // in place: scores -> probabilities (fp32)
    const uint64_t sl2_2 = pack2(sl2, sl2), nm2 = pack2(-mref, -mref);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float xa, xb;
      unpack2(ffma2(pack2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), sl2_2, nm2), xa, xb);
      v[2 * i] = __float_as_uint(fast_exp2(xa));
      v[2 * i + 1] = __float_as_uint(fast_exp2(xb));
    }
  };
  auto consume = [&](const uint32_t (&v)[32], int chunk) {
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float ea = __uint_as_float(v[2 * i]), eb = __uint_as_float(v[2 * i + 1]);
      acc[i & 3] = fadd2(acc[i & 3], pack2(ea, eb));
      pk[i] = pack_bf16x2(ea, eb);
    }
    store(chunk, pk);
  };
  issue(v0);
  __syncwarp();
  issue(v1);
  consume(v0, 0);
  __syncwarp();
  issue(v2);
  consume(v1, 1);
  __syncwarp();
  issue(v3);
  handover(v3[31]);  // every exponential of the row has been issued: the MUFU pipe can go to the other warpgroup (ping-pong;
                     // handing over one chunk earlier measured 750 / 836 instead of 756 / 850 TFLOP/s)
  consume(v2, 2);
  __syncwarp();
  consume(v3, 3);
}

// Carried state (normalised O, m' in raw score units, l = 1) -> the row's O columns in tensor memory, re-expressed against an
// integer reference maximum (set in mref); returns l.  Rows past the sequence load zeros.
__device__ __forceinline__ float load_state_row(const AttnParams& p, int64_t q_grow, int head, bool q_ok, uint32_t tmem_o,
                                                float& mref) {
  const float sl2 = p.scale_log2;
  const float m_in = q_ok ? p.state_m[q_grow * p.num_heads + head] : 0.f;
  mref = rintf(m_in * sl2);
  const float c_in = q_ok ? fast_exp2(fmaf(m_in, sl2, -mref)) : 0.f;  // in [2^-0.5, 2^0.5]
  const float* so = p.state_o + q_grow * p.ld_state_o + head * ATT_D;
#pragma unroll 1
  for (int c = 0; c < ATT_D; c += 8) {
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = 0u;
    if (q_ok) {
      const float4 x = *reinterpret_cast<const float4*>(so + c), y = *reinterpret_cast<const float4*>(so + c + 4);
      o[0] = __float_as_uint(x.x * c_in); o[1] = __float_as_uint(x.y * c_in); o[2] = __float_as_uint(x.z * c_in);
      o[3] = __float_as_uint(x.w * c_in); o[4] = __float_as_uint(y.x * c_in); o[5] = __float_as_uint(y.y * c_in);
      o[6] = __float_as_uint(y.z * c_in); o[7] = __float_as_uint(y.w * c_in);
    }
    tmem_st_32x32b_x8(tmem_o + c, o);
  }
  tmem_st_wait();
  tc_fence_before();
  return c_in;
}

// The 128 scores of the row (S in tensor memory, four 32-column loads) -> v0..v3, and their maximum.  Columns at or past
// kv_valid are set to -inf (ex2(-inf) = 0 exactly).  The maximum is reduced chunk by chunk UNDER the tensor-memory loads
// of the following chunks (a warp reads tensor memory at ~45 B/clk: the four 4 KB loads take ~360 clk whatever the order),
// and S is released (s_empty) as soon as it is in registers, so the tensor core may overwrite it with the next Q.K^T.
__device__ __forceinline__ float read_scores_max(uint32_t tmem_s, int kv_valid, uint64_t* s_empty, int lane, uint32_t (&v0)[32],
                                                 uint32_t (&v1)[32], uint32_t (&v2)[32], uint32_t (&v3)[32]) {
  float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  auto chunk_max = [&](uint32_t (&v)[32], int c0, float& m) {
    if (kv_valid < c0 + 32) {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (c0 + i >= kv_valid) v[i] = __float_as_uint(-INFINITY);
    }
    float a = -INFINITY, b = -INFINITY;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      a = fmaxf(a, __uint_as_float(v[i]));
      b = fmaxf(b, __uint_as_float(v[16 + i]));
    }
    m = fmaxf(a, b);
  };
  tmem_ld_32x32b_x32(tmem_s, v0);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tmem_s + 32, v1);
  chunk_max(v0, 0, mx4[0]);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tmem_s + 64, v2);
  chunk_max(v1, 32, mx4[1]);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tmem_s + 96, v3);
  chunk_max(v2, 64, mx4[2]);
  tmem_ld_wait();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(s_empty);
  chunk_max(v3, 96, mx4[3]);
  return fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
}

// Lazy rescale: mref moves to the tile maximum mt2 (log2 units) on the row's first tile, and afterwards only when mt2 exceeds
// it by more than 2^8; until then probabilities are computed against the stale reference (they stay <= 256, exact in fp32
// and in bf16's range), so the common tile does no correction work at all.  When any row of the warp moves, O (tensor
// memory) and l are scaled by the exact power of two 2^(old - new), after P.V of the previous tile has completed (p_empty
// with parity prev_parity, waited for when has_prev).  Returns whether it waited for that P.V.
__device__ __forceinline__ bool lazy_rescale(float mt2, bool first, bool has_prev, uint64_t* p_empty, uint32_t prev_parity,
                                             uint32_t tmem_o, float& mref, float& l_run) {
  float m_new = mref;
  bool need = false;
  if (first) m_new = rintf(mt2);
  else if (mt2 - mref > A2_RESCALE_LOG2) { need = true; m_new = rintf(mt2); }
  bool waited = false;
  if (__any_sync(0xffffffffu, need)) {
    if (has_prev) { mbar_wait(p_empty, prev_parity); waited = true; }
    tc_fence_after();
    const float alpha = need ? fast_exp2(mref - m_new) : 1.f;
#pragma unroll 1
    for (int c = 0; c < ATT_D; c += 8) {  // rare path
      uint32_t o[8];
      tmem_ld_32x32b_x8(tmem_o + c, o);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
      tmem_st_32x32b_x8(tmem_o + c, o);
    }
    tmem_st_wait();
    tc_fence_before();
    l_run *= alpha;
  }
  mref = m_new;
  return waited;
}

// Row epilogue, once the row's last P.V has completed: O (tensor memory) / l -> the bf16 output row, or, with write_state,
// the fp32 state row of partial `part` and m' = (mref + log2 l) / (scale log2 e).  Rows past the sequence store nothing.
__device__ __forceinline__ void store_row(const AttnParams& p, uint32_t tmem_o, bool q_ok, bool write_state, int part,
                                          int64_t q_grow, int head, float mref, float l_run) {
  const float inv_l = 1.0f / l_run;
  uint32_t o[32];
#pragma unroll 1
  for (int c = 0; c < ATT_D; c += 32) {
    tmem_ld_32x32b_x32(tmem_o + c, o);
    tmem_ld_wait();
    if (q_ok && write_state) {
      float4* so = reinterpret_cast<float4*>(p.state_o + part * p.split_stride_o + q_grow * p.ld_state_o + head * ATT_D + c);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        so[i] = make_float4(__uint_as_float(o[4 * i]) * inv_l, __uint_as_float(o[4 * i + 1]) * inv_l,
                            __uint_as_float(o[4 * i + 2]) * inv_l, __uint_as_float(o[4 * i + 3]) * inv_l);
    } else if (q_ok) {
      __nv_bfloat16* optr = p.out + q_grow * p.ldo + p.o_col0 + head * ATT_D + c;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        reinterpret_cast<uint4*>(optr)[q] =
            make_uint4(pack_bf16x2(__uint_as_float(o[8 * q]) * inv_l, __uint_as_float(o[8 * q + 1]) * inv_l),
                       pack_bf16x2(__uint_as_float(o[8 * q + 2]) * inv_l, __uint_as_float(o[8 * q + 3]) * inv_l),
                       pack_bf16x2(__uint_as_float(o[8 * q + 4]) * inv_l, __uint_as_float(o[8 * q + 5]) * inv_l),
                       pack_bf16x2(__uint_as_float(o[8 * q + 6]) * inv_l, __uint_as_float(o[8 * q + 7]) * inv_l));
    }
  }
  if (q_ok && write_state)
    p.state_m[part * p.split_stride_m + q_grow * p.num_heads + head] = (mref + __log2f(l_run)) * (1.0f / p.scale_log2);
}


// ================================================================================================================
// v2: one CTA per SM works on TWO 128-row query tiles (A, B) that share every K/V tile, with
//   * 8 softmax warps (4 per query tile), one thread per query ROW: the 128 scores of the row are read from TMEM ONCE
//     into registers and S is released immediately (the tensor core starts Q.K^T of the next tile while the
//     exponentials of this one are computed); row maximum and row sum are thread-local, and the two query tiles' softmax
//     warpgroups meet only at a pair of named barriers that make their exponential phases alternate (ping-pong);
//   * the output accumulator O kept in TMEM (PV accumulates in place) with LAZY rescaling (lazy_rescale);
//   * P written by the softmax warps straight into TENSOR MEMORY (tcgen05.st, two bf16 per 32-bit column) and consumed
//     by the P.V MMA as a TMEM A operand: shared memory carries only Q, K and V.  With P staged in shared memory the
//     kernel was bound by shared-memory bandwidth (Q.K^T reads 8 KB and P.V 6 KB per MMA, plus 32 KB of P writes per
//     tile -- about as many cycles as the exponentials themselves on a 128 B/clk port);
//   * a 4-deep K and V ring shared by both query tiles (half the L2 -> smem traffic per query row).
// Handles key segments, carried state (in and out) and the kv split.
// ================================================================================================================
constexpr int A2_THREADS = 11 * 32;  // warp 0 TMA, warp 1 (/10) MMA issuer of tile A (/B), warps 2..9 softmax
constexpr int A2_KV_STAGES = 4;
constexpr int A2_SMEM_BYTES = (2 + 2 * A2_KV_STAGES) * ATT_TILE_BYTES + 512;
constexpr int A2_TMEM_COLS = 512;  // S tiles [0, 256), O tiles [256, 384), P tiles [384, 512)
constexpr int A2_O_COL0 = 256, A2_P_COL0 = 384;
constexpr int A2_BMQ = 2 * ATT_BM;  // query rows per CTA

__global__ void __launch_bounds__(A2_THREADS, 1)
attention_fwd_v2_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                        const __grid_constant__ CUtensorMap tmap_v, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                                     // [2] tiles
  uint8_t* sK = sQ + 2 * ATT_TILE_BYTES;                  // [stages]
  uint8_t* sV = sK + A2_KV_STAGES * ATT_TILE_BYTES;       // [stages]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + A2_KV_STAGES * ATT_TILE_BYTES);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = k_full + A2_KV_STAGES;
  uint64_t* v_full = k_empty + A2_KV_STAGES;
  uint64_t* v_empty = v_full + A2_KV_STAGES;
  uint64_t* s_full = v_empty + A2_KV_STAGES;  // [2]
  uint64_t* s_empty = s_full + 2;             // [2]
  uint64_t* p_full = s_empty + 2;             // [2]
  uint64_t* p_empty = p_full + 2;             // [2]  (= "PV of the tile has completed")
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_empty + 2);

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = lane_id();
  // 1-D grid over (query block, head, sequence).  All FULL 256-row query blocks come first, the ragged last block of
  // every (head, sequence) -- cheaper, often a single 128-row tile -- is scheduled at the end where it fills the tail
  // wave instead of occupying an SM slot for a full block's duration in the middle (1370-token views: 5 full + 1 ragged).
  const int n_full = p.q_len / A2_BMQ;
  const int hs_count = p.num_heads * p.num_seqs;
  // slots [0, split_from) run as one CTA each; every later slot -- the ones that would form the badly filled last wave
  // of SMs -- is cut into kv_split CTAs that each take a share of the key range and leave a partial softmax state
  int bid = blockIdx.x, part = 0, nparts = 1;
  if (static_cast<int>(blockIdx.x) >= p.split_from && p.kv_split > 1) {
    const int r = blockIdx.x - p.split_from;
    bid = p.split_from + r / p.kv_split;
    part = r % p.kv_split;
    nparts = p.kv_split;
  }
  int qb, hs;
  if (bid < n_full * hs_count) {
    qb = bid % n_full;
    hs = bid / n_full;
  } else {
    qb = n_full;
    hs = bid - n_full * hs_count;
  }
  const int q0 = qb * A2_BMQ;
  const int head = hs % p.num_heads;
  const int seq = hs / p.num_heads;
  const int kv_tile0 = static_cast<int>((static_cast<int64_t>(part) * p.n_kv_tiles) / nparts);
  const int n_kv_tiles = static_cast<int>((static_cast<int64_t>(part + 1) * p.n_kv_tiles) / nparts) - kv_tile0;
  const bool write_state = (p.flags & MA_ATTN_STATE_OUT) != 0 || nparts > 1;
  const int n_qt = q0 + ATT_BM < p.q_len ? 2 : 1;  // query tile B is skipped when it lies past the sequence
  const bool state_in = (p.flags & MA_ATTN_STATE_IN) != 0;

  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("[ma] attention v2: dynamic smem base not 1024-byte aligned\n");
    __trap();
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < A2_KV_STAGES; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], n_qt);  // one tcgen05.commit per query-tile stream
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], n_qt);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&s_empty[t], 4);
      mbar_init(&p_full[t], 4);
      mbar_init(&p_empty[t], 1);
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    if (lane == 0) {
      prefetch_tmap(&tmap_q);
      prefetch_tmap(&tmap_k);
      prefetch_tmap(&tmap_v);
    }
    __syncwarp();
    tmem_alloc(tmem_slot, A2_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();  // prologue above overlaps the previous kernel's tail; no global memory access before this point

  if (warp == 0) {
    if (lane == 0) {
      const int q_row = static_cast<int>(seq * p.q_seq_stride) + q0;
      const int kv_row0 = static_cast<int>(seq * p.kv_seq_stride);
      mbar_arrive_expect_tx(q_full, 2 * ATT_TILE_BYTES);
      tma_load_2d(sQ, &tmap_q, q_full, p.q_col0 + head * ATT_D, q_row);
      tma_load_2d(sQ + ATT_TILE_BYTES, &tmap_q, q_full, p.q_col0 + head * ATT_D, q_row + ATT_BM);
      KvCursor<ATT_BN> cur;
      cur.skip(p, kv_tile0);
      for (int j = 0; j < n_kv_tiles; ++j, cur.next(p)) {
        const int st = j % A2_KV_STAGES;
        const uint32_t ph = (j / A2_KV_STAGES) & 1;
        const int row = kv_row0 + cur.row0(p);
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[st], ATT_TILE_BYTES);
        tma_load_2d(sK + st * ATT_TILE_BYTES, &tmap_k, &k_full[st], p.k_col0 + head * ATT_D, row);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&v_full[st], ATT_TILE_BYTES);
        tma_load_2d(sV + st * ATT_TILE_BYTES, &tmap_v, &v_full[st], p.v_col0 + head * ATT_D, row);
      }
    }
  } else if (warp == 1 || warp == 10) {
    // One MMA issuer per query tile: the two softmax streams only meet at the K / V ring (a stage is released when
    // BOTH issuers have committed it), so a slow row block in one tile never delays the other tile's Q.K^T.
    const int t = warp == 1 ? 0 : 1;
    if (lane == 0 && t < n_qt) {
      constexpr uint32_t idesc_s = make_idesc_bf16(ATT_BM, ATT_BN, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(ATT_BM, ATT_D, 0, 1);  // B (= V) is MN-major
      const uint32_t q_addr = smem_u32(sQ + t * ATT_TILE_BYTES);
      const uint32_t tmem_s = tmem_base + t * ATT_BN;
      const uint32_t tmem_o = tmem_base + A2_O_COL0 + t * ATT_D;
      const uint32_t p_tmem = tmem_base + A2_P_COL0 + t * 64;  // 128 kv x bf16 = 64 columns, 8 columns per K = 16 step
      auto issue_qk = [&](int j) {
        const int st = j % A2_KV_STAGES;
        const uint32_t ph = (j / A2_KV_STAGES) & 1;
        mbar_wait(&k_full[st], ph);
        mbar_wait(&s_empty[t], (j & 1) ^ 1);  // the softmax warps hold S of tile j-1 in registers
        tc_fence_after();
        const uint32_t k_addr = smem_u32(sK + st * ATT_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k)
          umma_bf16_ss(tmem_s, make_smem_desc_sw128(q_addr + k * 32, 16, 1024), make_smem_desc_sw128(k_addr + k * 32, 16, 1024),
                       idesc_s, k != 0 ? 1u : 0u);
        umma_commit(&s_full[t]);
        umma_commit(&k_empty[st]);
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      for (int j = 0; j < n_kv_tiles; ++j) {
        if (j + 1 < n_kv_tiles) issue_qk(j + 1);
        const int st = j % A2_KV_STAGES;
        const uint32_t ph = (j / A2_KV_STAGES) & 1;
        mbar_wait(&v_full[st], ph);
        mbar_wait(&p_full[t], j & 1);
        tc_fence_after();
        const uint32_t v_addr = smem_u32(sV + st * ATT_TILE_BYTES);
        const uint32_t acc0 = (j > 0 || state_in) ? 1u : 0u;
#pragma unroll
        for (int k = 0; k < ATT_BN / 16; ++k)
          umma_bf16_ts(tmem_o, p_tmem + k * 8, make_smem_desc_sw128(v_addr + k * 2048, 1024, 1024), idesc_pv, k != 0 ? 1u : acc0);
        umma_commit(&p_empty[t]);
        umma_commit(&v_empty[st]);
      }
    }
  } else {
    // ---- softmax warps: (query tile t, TMEM lane quarter); thread = query row -------------------------------
    const int t = (warp - 2) >> 2;
    const int quarter = warp & 3;
    if (t < n_qt) {
      const int row = quarter * 32 + lane;
      const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
      const uint32_t tmem_s = tmem_base + lane_base + t * ATT_BN;
      const uint32_t tmem_o = tmem_base + lane_base + A2_O_COL0 + t * ATT_D;
      const uint32_t tmem_p = tmem_base + lane_base + A2_P_COL0 + t * 64;
      const int q_idx = q0 + t * ATT_BM + row;
      const bool q_ok = q_idx < p.q_len;
      const int64_t q_grow = static_cast<int64_t>(seq) * p.q_seq_stride + q_idx;
      const float sl2 = p.scale_log2;

      float mref = 0.f, l_run = 0.f;
      if (state_in) l_run = load_state_row(p, q_grow, head, q_ok, tmem_o, mref);
      // Ping-pong: left free-running, the two softmax warps of a scheduler settle IN PHASE -- both read
      // S and reduce maxima together, then share the MUFU pipe at half rate each: period n + 2e per tile pair (n ~ 1150 clk
      // outside the exponential phase, e = 1024 clk of MUFU work; ncu: MUFU 71 % = 2e / (n + 2e)).  Two named barriers force
      // the exponential phases of the two warpgroups to ALTERNATE, so one owns the pipe at full rate while the other does its
      // tensor-memory reads, maximum and stores: period n + e.  (p.pingpong is always 1; see AttnParams.)
      const bool pingpong = n_qt == 2 && p.pingpong != 0;

      KvCursor<ATT_BN> cur;
      cur.skip(p, kv_tile0);
      for (int j = 0; j < n_kv_tiles; ++j, cur.next(p)) {
        const int kv_valid = cur.valid(p);
        mbar_wait(&s_full[t], j & 1);
        tc_fence_after();
        uint32_t v0[32], v1[32], v2[32], v3[32];  // the 128 scores of this thread's row
        const float m_tile = read_scores_max(tmem_s, kv_valid, &s_empty[t], lane, v0, v1, v2, v3);

        // lazy rescale (the steps of lazy_rescale, written out: called as a function here, ptxas schedules the
        // exponential phase below differently and the kernel measured ~1 % slower)
        const float mt2 = m_tile * sl2;
        float m_new = mref;
        bool need = false;
        if (j == 0 && !state_in) m_new = rintf(mt2);
        else if (mt2 - mref > A2_RESCALE_LOG2) { need = true; m_new = rintf(mt2); }
        bool waited = false;
        if (__any_sync(0xffffffffu, need)) {
          if (j > 0) { mbar_wait(&p_empty[t], (j - 1) & 1); waited = true; }  // PV of tile j-1 has completed
          tc_fence_after();
          const float alpha = need ? fast_exp2(mref - m_new) : 1.f;  // an exact power of two
#pragma unroll 1
          for (int c = 0; c < ATT_D; c += 8) {  // rare path
            uint32_t o[8];
            tmem_ld_32x32b_x8(tmem_o + c, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x32b_x8(tmem_o + c, o);
          }
          tmem_st_wait();
          tc_fence_before();
          l_run *= alpha;
        }
        mref = m_new;

        // exponentials -> bf16 pairs (two per 32-bit P column), stored to tensor memory chunk by chunk (16 columns = 32
        // scores at a time, so the packed probabilities never occupy more than 16 registers).  P.V of tile j-1 still reads
        // the single P buffer: it was issued a whole tile ago, so this wait is normally already satisfied.  Measured
        // placements of this wait (TFLOP/s, 8- / 24-view global shape): here, before the exponential phase 756 / 850; at the
        // first P store inside the phase 665 / 751; after the phase with all four stores deferred 592 / 668.
        if (!waited && j > 0) mbar_wait(&p_empty[t], (j - 1) & 1);
        tc_fence_after();
        uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
        float mref_turn = mref;
        // wait for the turn; the barrier carries the reference maximum so that no exponential can be scheduled above it
        if (pingpong && (t == 1 || j > 0)) asm volatile("bar.sync %1, 256;" : "+f"(mref_turn) : "r"(1 + t) : "memory");
        a2_exp_row_pipelined(v0, v1, v2, v3, sl2, mref_turn, acc,
                             [&](int chunk, const uint32_t (&pk)[16]) { tmem_st_32x32b_x16(tmem_p + 16 * chunk, pk); },
                             [&](uint32_t& last) {
                               if (pingpong && (t == 0 || j + 1 < n_kv_tiles))
                                 asm volatile("bar.arrive %1, 256;" : "+r"(last) : "r"(2 - t) : "memory");
                             });
        {
          float a0, a1, a2, a3;
          unpack2(fadd2(acc[0], acc[1]), a0, a1);
          unpack2(fadd2(acc[2], acc[3]), a2, a3);
          l_run += (a0 + a1) + (a2 + a3);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[t]);
      }

      mbar_wait(&p_empty[t], (n_kv_tiles - 1) & 1);
      tc_fence_after();
      store_row(p, tmem_o, q_ok, write_state, part, q_grow, head, mref, l_run);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, A2_TMEM_COLS);
  }
}


// ================================================================================================================
// v5: persistent CTAs, two INDEPENDENT attention streams per CTA with ping-pong (many short sequences: encoder / frame
// attention, 1370 keys = 11 steps per 128-row query tile).
//   * a work item is one 128-row query tile of one (sequence, head); stream t of CTA c takes the items r * 2G + 2c + t
//     (G = grid size = number of SMs), so 1408 items fill 296 streams in 4.76 -> 5 rounds (v3, three CTAs per SM:
//     3.17 -> 4 waves of 444 resident CTAs);
//   * each stream has its own Q tile, its own 3-stage K / V ring, its own TMA producer warp, MMA issuer warp and softmax
//     warpgroup, its own S / O / P tensor-memory columns (v2's column map) -- two one-tile pipelines inside one CTA.  What
//     the CTA buys is v2's ping-pong: the two softmax warps of a scheduler alternate their exponential phases through a pair of named
//     barriers instead of falling into step (MUFU 82 % instead of 63 - 71 % busy);
//   * every barrier phase runs on across items (global step counters), the producer loads the next item's Q as soon as the
//     last Q.K^T of the current one is issued, and the MMA issuer issues the next item's first Q.K^T right after the current
//     item's last P.V: an item's epilogue (O out of tensor memory, normalise, store) and the next item's ramp run under the
//     OTHER stream's exponential phase.
//   * both streams execute the same number of ping-pong turns (equal steps per item; a stream without an item in the last
//     round only passes the turn), so every bar.sync has its bar.arrive.
// No key segments, carried state or kv split here (ma_attention_fwd_ex routes those to v3 / v2).
// ================================================================================================================
constexpr int A5_THREADS = 12 * 32;  // warp 0 / 11: TMA producer of stream 0 / 1; warp 1 / 10: MMA issuer; warps 2-5 / 6-9: softmax
constexpr int A5_KV_STAGES = 3;
constexpr int A5_SMEM_BYTES = (2 + 2 * 2 * A5_KV_STAGES) * ATT_TILE_BYTES + 1024;
constexpr int A5_BARS_PER_STREAM = 6 + 4 * A5_KV_STAGES;

__global__ void __launch_bounds__(A5_THREADS, 1)
attention_fwd_v5_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                        const __grid_constant__ CUtensorMap tmap_v, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                                              // [2] tiles
  uint8_t* sKV = sQ + 2 * ATT_TILE_BYTES;                          // per stream: K[stages], V[stages]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + 2 * 2 * A5_KV_STAGES * ATT_TILE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * A5_BARS_PER_STREAM);

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = lane_id();
  const int n_qt = (p.q_len + ATT_BM - 1) / ATT_BM;
  const int n_items = n_qt * p.num_heads * p.num_seqs;
  const int S = p.n_kv_tiles;                                      // steps per item (the same for every item)
  const int G = gridDim.x;
  const int c = blockIdx.x;
  // rounds this CTA takes part in = rounds in which its stream 0 has an item
  const int n_rounds = n_items > 2 * c ? (n_items - 2 * c + 2 * G - 1) / (2 * G) : 0;
  const int g_total = n_rounds * S;                                // ping-pong turns per stream

  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("[ma] attention v5: dynamic smem base not 1024-byte aligned\n");
    __trap();
  }
  if (warp == 1 && lane == 0) {
    for (int t = 0; t < 2; ++t) {
      uint64_t* b = bars + t * A5_BARS_PER_STREAM;
      mbar_init(b + 0, 1);   // q_full
      mbar_init(b + 1, 1);   // q_empty (tcgen05.commit after the item's last Q.K^T)
      mbar_init(b + 2, 1);   // s_full
      mbar_init(b + 3, 4);   // s_empty
      mbar_init(b + 4, 4);   // p_full
      mbar_init(b + 5, 1);   // p_empty (= P.V of the step has completed)
      for (int i = 0; i < 4 * A5_KV_STAGES; ++i) mbar_init(b + 6 + i, 1);  // k_full, k_empty, v_full, v_empty [stages]
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    if (lane == 0) {
      prefetch_tmap(&tmap_q);
      prefetch_tmap(&tmap_k);
      prefetch_tmap(&tmap_v);
    }
    __syncwarp();
    tmem_alloc(tmem_slot, A2_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();  // no global memory access before this point

  // role -> stream
  const int t = (warp == 0 || warp == 1 || (warp >= 2 && warp <= 5)) ? 0 : 1;
  uint64_t* b = bars + t * A5_BARS_PER_STREAM;
  uint64_t* q_full = b + 0;
  uint64_t* q_empty = b + 1;
  uint64_t* s_full = b + 2;
  uint64_t* s_empty = b + 3;
  uint64_t* p_full = b + 4;
  uint64_t* p_empty = b + 5;
  uint64_t* k_full = b + 6;
  uint64_t* k_empty = k_full + A5_KV_STAGES;
  uint64_t* v_full = k_empty + A5_KV_STAGES;
  uint64_t* v_empty = v_full + A5_KV_STAGES;
  uint8_t* sQt = sQ + t * ATT_TILE_BYTES;
  uint8_t* sK = sKV + t * 2 * A5_KV_STAGES * ATT_TILE_BYTES;
  uint8_t* sV = sK + A5_KV_STAGES * ATT_TILE_BYTES;
  auto item_of = [&](int r) { return r * 2 * G + 2 * c + t; };
  auto decode = [&](int item, int& qb, int& head, int& seq) {
    const int hs = item / n_qt;
    qb = item - hs * n_qt;
    head = hs % p.num_heads;
    seq = hs / p.num_heads;
  };

  if (warp == 0 || warp == 11) {
    // ---- TMA producer of stream t ------------------------------------------------------------------------------
    if (lane == 0) {
      int gs = 0;  // global step counter = K / V ring position
      for (int r = 0; r < n_rounds; ++r) {
        const int item = item_of(r);
        if (item >= n_items) break;
        int qb, head, seq;
        decode(item, qb, head, seq);
        const int q_row = static_cast<int>(seq * p.q_seq_stride) + qb * ATT_BM;
        const int kv_row0 = static_cast<int>(seq * p.kv_seq_stride);
        if (r > 0) mbar_wait(q_empty, (r - 1) & 1);  // the previous item's last Q.K^T has read the Q tile
        mbar_arrive_expect_tx(q_full, ATT_TILE_BYTES);
        tma_load_2d(sQt, &tmap_q, q_full, p.q_col0 + head * ATT_D, q_row);
        for (int j = 0; j < S; ++j, ++gs) {
          const int st = gs % A5_KV_STAGES;
          const uint32_t ph = (gs / A5_KV_STAGES) & 1;
          const int row = kv_row0 + j * ATT_BN;
          mbar_wait(&k_empty[st], ph ^ 1);
          mbar_arrive_expect_tx(&k_full[st], ATT_TILE_BYTES);
          tma_load_2d(sK + st * ATT_TILE_BYTES, &tmap_k, &k_full[st], p.k_col0 + head * ATT_D, row);
          mbar_wait(&v_empty[st], ph ^ 1);
          mbar_arrive_expect_tx(&v_full[st], ATT_TILE_BYTES);
          tma_load_2d(sV + st * ATT_TILE_BYTES, &tmap_v, &v_full[st], p.v_col0 + head * ATT_D, row);
        }
      }
    }
  } else if (warp == 1 || warp == 10) {
    // ---- MMA issuer of stream t -------------------------------------------------------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(ATT_BM, ATT_BN, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(ATT_BM, ATT_D, 0, 1);  // B (= V) is MN-major
      const uint32_t q_addr = smem_u32(sQt);
      const uint32_t tmem_s = tmem_base + t * ATT_BN;
      const uint32_t tmem_o = tmem_base + A2_O_COL0 + t * ATT_D;
      const uint32_t p_tmem = tmem_base + A2_P_COL0 + t * 64;
      auto issue_qk = [&](int gs, bool last_of_item) {
        const int st = gs % A5_KV_STAGES;
        const uint32_t ph = (gs / A5_KV_STAGES) & 1;
        mbar_wait(&k_full[st], ph);
        mbar_wait(s_empty, (gs & 1) ^ 1);  // the softmax warps hold S of the previous step in registers
        tc_fence_after();
        const uint32_t k_addr = smem_u32(sK + st * ATT_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k)
          umma_bf16_ss(tmem_s, make_smem_desc_sw128(q_addr + k * 32, 16, 1024), make_smem_desc_sw128(k_addr + k * 32, 16, 1024),
                       idesc_s, k != 0 ? 1u : 0u);
        umma_commit(s_full);
        umma_commit(&k_empty[st]);
        if (last_of_item) umma_commit(q_empty);  // the Q tile may be overwritten once these MMAs have completed
      };
      int gs0 = 0;
      bool first_qk_issued = false;
      for (int r = 0; r < n_rounds; ++r) {
        if (item_of(r) >= n_items) break;
        if (!first_qk_issued) {
          mbar_wait(q_full, r & 1);
          issue_qk(gs0, S == 1);
        }
        for (int j = 0; j < S; ++j) {
          const int gs = gs0 + j;
          if (j + 1 < S) issue_qk(gs + 1, j + 2 == S);
          const int st = gs % A5_KV_STAGES;
          const uint32_t ph = (gs / A5_KV_STAGES) & 1;
          mbar_wait(&v_full[st], ph);
          mbar_wait(p_full, gs & 1);
          tc_fence_after();
          const uint32_t v_addr = smem_u32(sV + st * ATT_TILE_BYTES);
#pragma unroll
          for (int k = 0; k < ATT_BN / 16; ++k)
            umma_bf16_ts(tmem_o, p_tmem + k * 8, make_smem_desc_sw128(v_addr + k * 2048, 1024, 1024), idesc_pv,
                         (k != 0 || j > 0) ? 1u : 0u);
          umma_commit(p_empty);
          umma_commit(&v_empty[st]);
        }
        gs0 += S;
        // the next item's first Q.K^T, so that its scores are ready when the softmax warps leave this item's epilogue
        first_qk_issued = false;
        if (r + 1 < n_rounds && item_of(r + 1) < n_items) {
          mbar_wait(q_full, (r + 1) & 1);
          issue_qk(gs0, S == 1);
          first_qk_issued = true;
        }
      }
    }
  } else {
    // ---- softmax warps of stream t: TMEM lane quarter = warp & 3; thread = query row ----------------------------
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t tmem_s = tmem_base + lane_base + t * ATT_BN;
    const uint32_t tmem_o = tmem_base + lane_base + A2_O_COL0 + t * ATT_D;
    const uint32_t tmem_p = tmem_base + lane_base + A2_P_COL0 + t * 64;
    const float sl2 = p.scale_log2;
    const int kv_len = p.seg_len[0];
    int gs0 = 0;
    for (int r = 0; r < n_rounds; ++r) {
      const int item = item_of(r);
      if (item >= n_items) {
        // no item for this stream in the CTA's last round: pass the turns so that the other stream's barriers pair up
        for (int j = 0; j < S; ++j) {
          const int gs = gs0 + j;
          asm volatile("bar.sync %0, 256;" ::"r"(1 + t) : "memory");          // t == 1 here: always waits
          if (gs + 1 < g_total) asm volatile("bar.arrive %0, 256;" ::"r"(2 - t) : "memory");
        }
        gs0 += S;
        continue;
      }
      int qb, head, seq;
      decode(item, qb, head, seq);
      const int q_idx = qb * ATT_BM + row;
      const bool q_ok = q_idx < p.q_len;
      const int64_t q_grow = static_cast<int64_t>(seq) * p.q_seq_stride + q_idx;
      float mref = 0.f, l_run = 0.f;
      for (int j = 0; j < S; ++j) {
        const int gs = gs0 + j;
        const int kv_valid = kv_len - j * ATT_BN;
        mbar_wait(s_full, gs & 1);
        tc_fence_after();
        uint32_t v0[32], v1[32], v2[32], v3[32];  // the 128 scores of this thread's row
        const float m_tile = read_scores_max(tmem_s, kv_valid, s_empty, lane, v0, v1, v2, v3);
        // no row moves on an item's first step, so the previous step's P.V exists whenever the rescale waits for it
        const bool waited = lazy_rescale(m_tile * sl2, j == 0, true, p_empty, (gs - 1) & 1, tmem_o, mref, l_run);

        // P.V of the previous step (of this item, or the last one of the previous item -- whose completion the epilogue has
        // already waited for) still reads the single P buffer
        if (!waited && j > 0) mbar_wait(p_empty, (gs - 1) & 1);
        tc_fence_after();
        uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
        float mref_turn = mref;
        // wait for the turn; the barrier carries the reference maximum so that no exponential can be scheduled above it
        if (t == 1 || gs > 0) asm volatile("bar.sync %1, 256;" : "+f"(mref_turn) : "r"(1 + t) : "memory");
        a2_exp_row_pipelined(v0, v1, v2, v3, sl2, mref_turn, acc,
                             [&](int chunk, const uint32_t (&pk)[16]) { tmem_st_32x32b_x16(tmem_p + 16 * chunk, pk); },
                             [&](uint32_t& last) {
                               if (t == 0 || gs + 1 < g_total)
                                 asm volatile("bar.arrive %1, 256;" : "+r"(last) : "r"(2 - t) : "memory");
                             });
        {
          float a0, a1, a2, a3;
          unpack2(fadd2(acc[0], acc[1]), a0, a1);
          unpack2(fadd2(acc[2], acc[3]), a2, a3);
          l_run += (a0 + a1) + (a2 + a3);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
      }
      gs0 += S;

      // ---- finish the item: normalise, store (runs under the other stream's exponential phase) ----
      mbar_wait(p_empty, (gs0 - 1) & 1);
      tc_fence_after();
      store_row(p, tmem_o, q_ok, false, 0, q_grow, head, mref, l_run);
      tc_fence_before();   // the tensor-memory reads of O are ordered before the p_full arrive that lets the next P.V overwrite it
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, A2_TMEM_COLS);
  }
}


// ================================================================================================================
// v3: three CTAs per SM.
//   * one 128-row query tile per CTA, and key / value steps of 64 rows: a softmax thread holds 64 scores
//     (112 registers instead of 168) and a CTA needs 64 (S) + 64 (O) + 32 (P) = 160 tensor-memory columns, taken as TWO
//     allocations (128 + 32; a single allocation must be a power of two), so THREE CTAs fit an SM (480 of 512 columns,
//     3 x 64 KB shared memory, 3 x 192 x 112 registers).  Every scheduler then holds three softmax warps from three
//     independent CTAs.  The v2 layout (two per scheduler) leaves the MUFU pipe -- the bound at head_dim 64: 128 x 128
//     exponentials = 1024 clk per tile against 512 clk of MMA -- 29 % idle, because two warps cannot cover each other's
//     tensor-memory reads, maxima and barrier round trips (profiles/r2_attn_v2_poly0_ncu.csv: MUFU 71 %, tensor 35 %);
//   * the intra-CTA pipeline of v2 is kept: S is released as soon as it is in registers, so Q K_{j+1}^T runs under the
//     exponentials of step j; P has its own columns; O accumulates in tensor memory with lazy rescaling.  (A first form
//     without that pipeline -- P written in place over S, 128 columns, the chain S_j -> softmax -> P_j V_j -> S_{j+1}
//     strictly serial per CTA -- measured 494 TFLOP/s on the 8-view global shape against 766 for v2: three CTAs do not
//     hide ~2000 clk of barrier / MMA latency per step.)
//   * exponentials 32 scores at a time (a2_exp_chunk): packed fp32x2 arithmetic, integer reference maximum.
// Same interface / masking / segment / carried-state semantics as v2; the kv split is v2's alone.
// ================================================================================================================
constexpr int A3_BN = 64;
constexpr int A3_STAGES = 3;
constexpr int A3_KV_BYTES = A3_BN * ATT_D * 2;  // 8 KB per K or V stage
constexpr int A3_SMEM_BYTES = ATT_TILE_BYTES + 2 * A3_STAGES * A3_KV_BYTES + 256;
constexpr int A3_THREADS = 6 * 32;  // warp 0: TMA producer, warp 1: MMA issuer, warps 2..5: softmax
constexpr int A3_TMEM_COLS = 128;   // first allocation: S [0, 64), O [64, 128)
constexpr int A3_TMEM_P_COLS = 32;  // second allocation: P (64 probabilities as bf16 pairs)

// Registers: a scheduler (SM sub-partition) owns 16 K registers and the warps of the resident CTAs are spread over the four
// schedulers: 3 CTAs x 6 warps = 18 warps -> one scheduler holds 5 of them -> at most 16384 / (5 x 32) = 102 registers per
// thread, i.e. 96.  (At 104-112 registers only TWO CTAs were resident: launch__occupancy_limit_registers = 2.)
__global__ void __maxnreg__(96)
attention_fwd_v3_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                        const __grid_constant__ CUtensorMap tmap_v, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + ATT_TILE_BYTES;
  uint8_t* sV = sK + A3_STAGES * A3_KV_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + A3_STAGES * A3_KV_BYTES);
  uint64_t* q_full = bars;
  uint64_t* k_full = bars + 1;
  uint64_t* k_empty = k_full + A3_STAGES;
  uint64_t* v_full = k_empty + A3_STAGES;
  uint64_t* v_empty = v_full + A3_STAGES;
  uint64_t* s_full = v_empty + A3_STAGES;
  uint64_t* s_empty = s_full + 1;
  uint64_t* p_full = s_empty + 1;
  uint64_t* p_empty = p_full + 1;  // "P_j V_j has completed"
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_empty + 1);  // [2]

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = lane_id();
  // full 128-row query tiles of every (head, sequence) first, the ragged last tiles at the end (they fill the tail wave)
  const int n_full = p.q_len / ATT_BM;
  const int hs_count = p.num_heads * p.num_seqs;
  const int bid = blockIdx.x;
  int qb, hs;
  if (bid < n_full * hs_count) {
    qb = bid % n_full;
    hs = bid / n_full;
  } else {
    qb = n_full;
    hs = bid - n_full * hs_count;
  }
  const int q0 = qb * ATT_BM;
  const int head = hs % p.num_heads;
  const int seq = hs / p.num_heads;
  int n_kv_tiles = 0;
  for (int sgm = 0; sgm < p.n_segs; ++sgm) n_kv_tiles += (p.seg_len[sgm] + A3_BN - 1) / A3_BN;
  const bool write_state = (p.flags & MA_ATTN_STATE_OUT) != 0;
  const bool state_in = (p.flags & MA_ATTN_STATE_IN) != 0;

  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("[ma] attention v3: dynamic smem base not 1024-byte aligned\n");
    __trap();
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int st = 0; st < A3_STAGES; ++st) {
      mbar_init(&k_full[st], 1);
      mbar_init(&k_empty[st], 1);
      mbar_init(&v_full[st], 1);
      mbar_init(&v_empty[st], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(s_empty, 4);
    mbar_init(p_full, 4);
    mbar_init(p_empty, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    if (lane == 0) {
      prefetch_tmap(&tmap_q);
      prefetch_tmap(&tmap_k);
      prefetch_tmap(&tmap_v);
    }
    __syncwarp();
    // the 128-column block first: three of them tile [0, 384) and the 32-column blocks land behind them, so a CTA that
    // starts while two others are resident always finds its 128 aligned columns free
    tmem_alloc(tmem_slot, A3_TMEM_COLS);
    tmem_alloc(tmem_slot + 1, A3_TMEM_P_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot[0];
  const uint32_t tmem_pbase = tmem_slot[1];
  pdl_sync();  // no global memory access before this point

  if (warp == 0) {
    if (lane == 0) {
      const int q_row = static_cast<int>(seq * p.q_seq_stride) + q0;
      const int kv_row0 = static_cast<int>(seq * p.kv_seq_stride);
      mbar_arrive_expect_tx(q_full, ATT_TILE_BYTES);
      tma_load_2d(sQ, &tmap_q, q_full, p.q_col0 + head * ATT_D, q_row);
      KvCursor<A3_BN> cur;
      for (int j = 0; j < n_kv_tiles; ++j, cur.next(p)) {
        const int st = j % A3_STAGES;
        const uint32_t ph = (j / A3_STAGES) & 1;
        const int row = kv_row0 + cur.row0(p);
        mbar_wait(&k_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&k_full[st], A3_KV_BYTES);
        tma_load_2d(sK + st * A3_KV_BYTES, &tmap_k, &k_full[st], p.k_col0 + head * ATT_D, row);
        mbar_wait(&v_empty[st], ph ^ 1);
        mbar_arrive_expect_tx(&v_full[st], A3_KV_BYTES);
        tma_load_2d(sV + st * A3_KV_BYTES, &tmap_v, &v_full[st], p.v_col0 + head * ATT_D, row);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(ATT_BM, A3_BN, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(ATT_BM, ATT_D, 0, 1);  // B (= V) is MN-major
      const uint32_t q_addr = smem_u32(sQ);
      const uint32_t tmem_s = tmem_base;
      const uint32_t tmem_o = tmem_base + 64;
      auto issue_qk = [&](int j) {
        const int st = j % A3_STAGES;
        mbar_wait(&k_full[st], (j / A3_STAGES) & 1);
        mbar_wait(s_empty, (j & 1) ^ 1);  // the softmax warps hold S of step j-1 in registers
        tc_fence_after();
        const uint32_t k_addr = smem_u32(sK + st * A3_KV_BYTES);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k)
          umma_bf16_ss(tmem_s, make_smem_desc_sw128(q_addr + k * 32, 16, 1024), make_smem_desc_sw128(k_addr + k * 32, 16, 1024),
                       idesc_s, k != 0 ? 1u : 0u);
        umma_commit(s_full);
        umma_commit(&k_empty[st]);
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      for (int j = 0; j < n_kv_tiles; ++j) {
        if (j + 1 < n_kv_tiles) issue_qk(j + 1);
        const int st = j % A3_STAGES;
        mbar_wait(&v_full[st], (j / A3_STAGES) & 1);
        mbar_wait(p_full, j & 1);
        tc_fence_after();
        const uint32_t v_addr = smem_u32(sV + st * A3_KV_BYTES);
        const uint32_t acc0 = (j > 0 || state_in) ? 1u : 0u;
#pragma unroll
        for (int k = 0; k < A3_BN / 16; ++k)
          umma_bf16_ts(tmem_o, tmem_pbase + k * 8, make_smem_desc_sw128(v_addr + k * 2048, 1024, 1024), idesc_pv, k != 0 ? 1u : acc0);
        umma_commit(p_empty);
        umma_commit(&v_empty[st]);
      }
    }
  } else if (warp >= 2) {
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t tmem_s = tmem_base + lane_base;
    const uint32_t tmem_o = tmem_base + lane_base + 64;
    const uint32_t tmem_p = tmem_pbase + lane_base;
    const int q_idx = q0 + row;
    const bool q_ok = q_idx < p.q_len;
    const int64_t q_grow = static_cast<int64_t>(seq) * p.q_seq_stride + q_idx;
    const float sl2 = p.scale_log2;
    float mref = 0.f, l_run = 0.f;
    if (state_in) l_run = load_state_row(p, q_grow, head, q_ok, tmem_o, mref);
    const uint64_t sl2_2 = pack2(sl2, sl2);

    KvCursor<A3_BN> cur;
    for (int j = 0; j < n_kv_tiles; ++j, cur.next(p)) {
      const int kv_valid = cur.valid(p);
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      tmem_ld_32x32b_x32(tmem_s, v0);
      tmem_ld_32x32b_x32(tmem_s + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty);  // S is in registers: the tensor core may overwrite it
      if (kv_valid < A3_BN) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          if (i >= kv_valid) v0[i] = __float_as_uint(-INFINITY);
          if (32 + i >= kv_valid) v1[i] = __float_as_uint(-INFINITY);
        }
      }
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        mx4[0] = fmaxf(mx4[0], __uint_as_float(v0[i]));
        mx4[1] = fmaxf(mx4[1], __uint_as_float(v0[16 + i]));
        mx4[2] = fmaxf(mx4[2], __uint_as_float(v1[i]));
        mx4[3] = fmaxf(mx4[3], __uint_as_float(v1[16 + i]));
      }
      const float mt2 = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])) * sl2;
      const bool waited = lazy_rescale(mt2, j == 0 && !state_in, j > 0, p_empty, (j - 1) & 1, tmem_o, mref, l_run);

      uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
      const uint64_t nm2 = pack2(-mref, -mref);
      uint32_t pk[16];
      // the single P buffer is still read by P_{j-1} V_{j-1}: wait for it only once the first 32 exponentials are done
      a2_exp_chunk(v0, pk, sl2_2, nm2, acc);
      if (!waited && j > 0) mbar_wait(p_empty, (j - 1) & 1);
      tc_fence_after();
      tmem_st_32x32b_x16(tmem_p, pk);
      a2_exp_chunk(v1, pk, sl2_2, nm2, acc);
      tmem_st_32x32b_x16(tmem_p + 16, pk);
      {
        float a0, a1, a2, a3;
        unpack2(fadd2(acc[0], acc[1]), a0, a1);
        unpack2(fadd2(acc[2], acc[3]), a2, a3);
        l_run += (a0 + a1) + (a2 + a3);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }

    mbar_wait(p_empty, (n_kv_tiles - 1) & 1);
    tc_fence_after();
    store_row(p, tmem_o, q_ok, write_state, 0, q_grow, head, mref, l_run);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_pbase, A3_TMEM_P_COLS);
    tmem_dealloc(tmem_base, A3_TMEM_COLS);
  }
}


// ----------------------------------------------------------------------------------------------------------------
// Join of partial softmax states (kv_split > 1, or local + remote key ranges of the view-sharded global attention):
//   out[row, h, :] = sum_p w_p o_p / sum_p w_p,   w_p = 2^((m'_p - max_p m'_p) * scale * log2 e)
// where o_p is the normalised partial output and m'_p its shifted maximum.  One warp per (row, head); 256 B per partial.
// state_m must be pre-filled with -inf: partial slots nobody wrote are skipped, rows without any partial are left alone.
// ----------------------------------------------------------------------------------------------------------------
__global__ void attention_merge_kernel(const float* __restrict__ state_o, int64_t ld_o, int64_t stride_o,
                                       const float* __restrict__ state_m, int64_t stride_m, int n_part, int64_t rows,
                                       int num_heads, float scale_log2, __nv_bfloat16* __restrict__ out, int64_t ldo,
                                       int first_slot) {
  const int64_t wid = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  int64_t row;
  int h;
  if (first_slot < 0) {  // every (row, head)
    if (wid >= rows * num_heads) return;
    row = wid / num_heads;
    h = static_cast<int>(wid - row * num_heads);
  } else {  // only the rows of the (query block, head) slots >= first_slot (slot order of attention_fwd_v2_kernel, 1 sequence)
    const int n_full = static_cast<int>(rows / (2 * ATT_BM));
    const int n_slots = static_cast<int>((rows + 2 * ATT_BM - 1) / (2 * ATT_BM)) * num_heads;
    const int64_t slot = first_slot + wid / (2 * ATT_BM);
    if (slot >= n_slots) return;
    int qb;
    if (slot < static_cast<int64_t>(n_full) * num_heads) { qb = static_cast<int>(slot % n_full); h = static_cast<int>(slot / n_full); }
    else { qb = n_full; h = static_cast<int>(slot - static_cast<int64_t>(n_full) * num_heads); }
    row = static_cast<int64_t>(qb) * 2 * ATT_BM + wid % (2 * ATT_BM);
    if (row >= rows) return;
  }
  float mx = -INFINITY;
  for (int pidx = 0; pidx < n_part; ++pidx) mx = fmaxf(mx, state_m[pidx * stride_m + row * num_heads + h]);
  if (mx == -INFINITY) return;  // no partial was written for this (row, head): its CTA stored the final output itself
  float ax = 0.f, ay = 0.f, wsum = 0.f;
  for (int pidx = 0; pidx < n_part; ++pidx) {
    const float mp = state_m[pidx * stride_m + row * num_heads + h];
    if (mp == -INFINITY) continue;  // unused partial slot (state_m is pre-filled with -inf)
    const float w = fast_exp2((mp - mx) * scale_log2);
    const float2 o = *reinterpret_cast<const float2*>(state_o + pidx * stride_o + row * ld_o + h * ATT_D + 2 * lane);
    ax = fmaf(w, o.x, ax);
    ay = fmaf(w, o.y, ay);
    wsum += w;
  }
  const float inv = 1.0f / wsum;
  *reinterpret_cast<uint32_t*>(out + row * ldo + h * ATT_D + 2 * lane) = pack_bf16x2(ax * inv, ay * inv);
}

}  // namespace ma

extern "C" int ma_attention_fwd(const void* q, int64_t ldq, int64_t q_rows, int q_col0, const void* k, int64_t ldk,
                                int64_t kv_rows, int k_col0, const void* v, int64_t ldv, int v_col0, void* out,
                                int64_t ldo, int o_col0, int num_seqs, int num_heads, int q_len, int kv_len,
                                int64_t q_seq_stride, int64_t kv_seq_stride, float softmax_scale, void* stream) {
  return ma_attention_fwd_ex(q, ldq, q_rows, q_col0, k, ldk, kv_rows, k_col0, v, ldv, v_col0, out, ldo, o_col0, num_seqs,
                             num_heads, q_len, kv_len, q_seq_stride, kv_seq_stride, softmax_scale, nullptr, stream);
}

extern "C" int ma_attention_fwd_ex(const void* q, int64_t ldq, int64_t q_rows, int q_col0, const void* k, int64_t ldk,
                                   int64_t kv_rows, int k_col0, const void* v, int64_t ldv, int v_col0, void* out,
                                   int64_t ldo, int o_col0, int num_seqs, int num_heads, int q_len, int kv_len,
                                   int64_t q_seq_stride, int64_t kv_seq_stride, float softmax_scale,
                                   const ma_attn_ext* ext, void* stream) {
  using namespace ma;
  MA_REQUIRE(q && k && v, "ma_attention_fwd: null pointer");
  const int flags = ext ? ext->flags : 0;
  MA_REQUIRE(out || (flags & MA_ATTN_STATE_OUT), "ma_attention_fwd: null output");
  MA_REQUIRE(num_seqs > 0 && num_heads > 0 && q_len > 0 && kv_len > 0, "ma_attention_fwd: bad sizes");
  AttnParams p;
  p.n_segs = 1;
  p.seg_row0[0] = 0;
  p.seg_len[0] = kv_len;
  if (ext && ext->n_segments > 0) {
    MA_REQUIRE(ext->n_segments <= MA_ATTN_MAX_SEGMENTS, "ma_attention_fwd: more than %d kv segments", MA_ATTN_MAX_SEGMENTS);
    int64_t total = 0;
    for (int s = 0; s < ext->n_segments; ++s) {
      MA_REQUIRE(ext->seg_len[s] > 0 && ext->seg_row0[s] >= 0, "ma_attention_fwd: kv segment %d is empty / negative", s);
      p.seg_row0[s] = ext->seg_row0[s];
      p.seg_len[s] = ext->seg_len[s];
      total += ext->seg_len[s];
    }
    MA_REQUIRE(total == kv_len, "ma_attention_fwd: kv segments sum to %lld, kv_len is %d", (long long)total, kv_len);
    p.n_segs = ext->n_segments;
  }
  p.n_kv_tiles = 0;
  int kv_extent = 0;
  for (int s = 0; s < p.n_segs; ++s) {
    p.n_kv_tiles += (p.seg_len[s] + ATT_BN - 1) / ATT_BN;
    kv_extent = p.seg_row0[s] + p.seg_len[s] > kv_extent ? p.seg_row0[s] + p.seg_len[s] : kv_extent;
  }
  p.state_o = nullptr; p.state_m = nullptr; p.ld_state_o = 0;
  if (flags & (MA_ATTN_STATE_IN | MA_ATTN_STATE_OUT)) {
    MA_REQUIRE(ext->state_o && ext->state_m && ext->ld_state_o % 4 == 0 && ext->ld_state_o >= (int64_t)num_heads * ATT_D &&
                   (reinterpret_cast<uintptr_t>(ext->state_o) & 15) == 0,
               "ma_attention_fwd: softmax state buffers missing / misaligned");
    p.state_o = ext->state_o; p.state_m = ext->state_m; p.ld_state_o = ext->ld_state_o;
  }
  p.num_heads = num_heads;
  p.num_seqs = num_seqs;
  p.flags = flags;
  p.kv_split = 1;
  p.pingpong = 1;
  p.split_from = 0;
  p.split_stride_o = 0;
  p.split_stride_m = 0;
  const int n_slots_host = ((q_len + 2 * ATT_BM - 1) / (2 * ATT_BM)) * num_heads * num_seqs;
  int grid_ctas = n_slots_host;
  if (ext && ext->kv_split > 1) {
    MA_REQUIRE(!(flags & MA_ATTN_STATE_IN), "ma_attention_fwd: kv_split cannot resume from a state");
    MA_REQUIRE(ext->state_o && ext->state_m, "ma_attention_fwd: kv_split needs the partial-state buffers");
    MA_REQUIRE(ext->kv_split_from >= 0 && ext->kv_split_from <= n_slots_host, "ma_attention_fwd: kv_split_from out of range");
    p.state_o = ext->state_o; p.state_m = ext->state_m; p.ld_state_o = ext->ld_state_o;
    p.split_from = ext->kv_split_from;
    grid_ctas = p.split_from + (n_slots_host - p.split_from) * ext->kv_split;
    MA_REQUIRE(ext->kv_split <= p.n_kv_tiles, "ma_attention_fwd: kv_split %d exceeds the %d kv tiles", ext->kv_split, p.n_kv_tiles);
    MA_REQUIRE(ext->split_stride_o % 4 == 0, "ma_attention_fwd: split_stride_o must be a multiple of 4 floats");
    p.kv_split = ext->kv_split;
    p.split_stride_o = ext->split_stride_o;
    p.split_stride_m = ext->split_stride_m;
  }
  MA_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0 && q_col0 % 8 == 0 && k_col0 % 8 == 0 &&
                 v_col0 % 8 == 0 && o_col0 % 8 == 0,
             "ma_attention_fwd: strides / column offsets must be multiples of 8 elements");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "ma_attention_fwd: out not 16-byte aligned");
  MA_REQUIRE((int64_t)(num_seqs - 1) * q_seq_stride + q_len <= q_rows && (int64_t)(num_seqs - 1) * kv_seq_stride + kv_extent <= kv_rows,
             "ma_attention_fwd: sequences exceed the q / kv row counts");
  MA_REQUIRE(q_col0 + num_heads * ATT_D <= ldq && k_col0 + num_heads * ATT_D <= ldk && v_col0 + num_heads * ATT_D <= ldv &&
                 o_col0 + num_heads * ATT_D <= ldo,
             "ma_attention_fwd: head columns exceed the row stride");

  CUtensorMap tq, tk, tv;
  const uint32_t box[2] = {ATT_D, ATT_BM};
  {
    uint64_t dims[2] = {(uint64_t)ldq, (uint64_t)q_rows};
    uint64_t str[1] = {(uint64_t)ldq * 2};
    int rc = make_tmap_bf16(&tq, q, 2, dims, str, box);
    if (rc != MA_OK) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)ldk, (uint64_t)kv_rows};
    uint64_t str[1] = {(uint64_t)ldk * 2};
    int rc = make_tmap_bf16(&tk, k, 2, dims, str, box);
    if (rc != MA_OK) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)ldv, (uint64_t)kv_rows};
    uint64_t str[1] = {(uint64_t)ldv * 2};
    int rc = make_tmap_bf16(&tv, v, 2, dims, str, box);
    if (rc != MA_OK) return rc;
  }
  p.out = static_cast<__nv_bfloat16*>(out);
  p.ldo = ldo;
  p.q_len = q_len;
  p.q_seq_stride = q_seq_stride;
  p.kv_seq_stride = kv_seq_stride;
  p.q_col0 = q_col0;
  p.k_col0 = k_col0;
  p.v_col0 = v_col0;
  p.o_col0 = o_col0;
  p.scale_log2 = softmax_scale * 1.4426950408889634f;
  // Kernel choice (same-box A/B on a B200, tools/bench_kernels.py, TFLOP/s):
  //  * v5 for plain attention over many short sequences, once the (128-row query tile x head x sequence) items fill the
  //    2 x SMs streams for at least three rounds.  Against v3: 8 x 16 x 1370 (encoder, 1408 items) 637 vs 572, 8 x 12 x 1369
  //    (frame, 1056 items) 592 vs 539, 24 x 16 x 1370 698 vs 655; 3 x 12 x 1369 (396 items, 1.3 rounds) 411 vs 468.
  //  * v3 for other calls with up to 4096 keys and no kv split.  Against one query tile per CTA in the v2 layout:
  //    1370-key sequences (encoder, frame attention) 586 / 552 vs 572 / 535 at 8 views, 658 / 634 vs 622 / 604 at 24 views;
  //    one long sequence (global attention) 740 vs 766 at 8 views, 786 vs 799 at 24.
  //  * v2 otherwise (long sequences, kv split): K / V shared by 256 query rows and ping-pong, MUFU 82 % busy instead of
  //    71 %: 881 vs 795 for one tile per CTA at 16 views, 850 vs 799 at 24; at 8 views 756 vs 766 as a plain launch (516
  //    CTAs = 3.5 waves of 148), 860 with the last partial wave split over the key range (Engine._pick_tail_split).
  using KernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, AttnParams);
  const int sms = device_sm_count();
  const int n_items = ((q_len + ATT_BM - 1) / ATT_BM) * num_heads * num_seqs;
  const bool short_keys = kv_len <= 4096 && p.kv_split == 1;
  int kernel;  // index into `configured` below
  KernelFn fn;
  int threads, smem_bytes, ctas;
  if (short_keys && p.n_segs == 1 && p.seg_row0[0] == 0 && !(flags & (MA_ATTN_STATE_IN | MA_ATTN_STATE_OUT)) &&
      n_items >= 6 * sms) {
    kernel = 0;
    fn = attention_fwd_v5_kernel;
    threads = A5_THREADS;
    smem_bytes = A5_SMEM_BYTES;
    ctas = sms < (n_items + 1) / 2 ? sms : (n_items + 1) / 2;
  } else if (short_keys) {
    kernel = 1;
    fn = attention_fwd_v3_kernel;
    threads = A3_THREADS;
    smem_bytes = A3_SMEM_BYTES;
    ctas = n_items;
    // key / value boxes of 64 rows
    const uint32_t box64[2] = {ATT_D, A3_BN};
    uint64_t dims[2] = {(uint64_t)ldk, (uint64_t)kv_rows};
    uint64_t str[1] = {(uint64_t)ldk * 2};
    int rc = make_tmap_bf16(&tk, k, 2, dims, str, box64);
    if (rc != MA_OK) return rc;
    dims[0] = (uint64_t)ldv;
    str[0] = (uint64_t)ldv * 2;
    rc = make_tmap_bf16(&tv, v, 2, dims, str, box64);
    if (rc != MA_OK) return rc;
  } else {
    kernel = 2;
    fn = attention_fwd_v2_kernel;
    threads = A2_THREADS;
    smem_bytes = A2_SMEM_BYTES;
    ctas = grid_ctas;
  }
  static bool configured[3][MA_MAX_DEVICES] = {};  // the large-shared-memory opt-in is per kernel and device
  const int dev = current_device();
  if (!configured[kernel][dev]) {
    MA_CHECK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    if (kernel != 0)  // v2 / v3; v5's shared memory leaves no other carveout
      MA_CHECK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured[kernel][dev] = true;
  }
  MA_CHECK_CUDA(launch_kernel(fn, dim3(ctas), dim3(threads), smem_bytes, static_cast<cudaStream_t>(stream), pdl_enabled(),
                              tq, tk, tv, p));
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}

extern "C" int ma_attention_merge(const float* state_o, int64_t ld_state_o, int64_t split_stride_o, const float* state_m,
                                  int64_t split_stride_m, int n_partials, int64_t rows, int num_heads, float softmax_scale,
                                  void* out, int64_t ldo, int first_slot, void* stream) {
  using namespace ma;
  MA_REQUIRE(state_o && state_m && out && n_partials >= 1 && rows > 0 && num_heads > 0, "ma_attention_merge: bad arguments");
  MA_REQUIRE(ld_state_o % 2 == 0 && split_stride_o % 2 == 0 && ldo % 2 == 0, "ma_attention_merge: strides must be even");
  int64_t warps = rows * num_heads;
  if (first_slot >= 0) {
    const int64_t n_slots = ((rows + 2 * ATT_BM - 1) / (2 * ATT_BM)) * num_heads;
    MA_REQUIRE(first_slot <= n_slots, "ma_attention_merge: first_slot out of range");
    warps = (n_slots - first_slot) * 2 * ATT_BM;
    if (warps == 0) return MA_OK;
  }
  const int64_t blocks = (warps * 32 + 255) / 256;
  attention_merge_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      state_o, ld_state_o, split_stride_o, state_m, split_stride_m, n_partials, rows, num_heads,
      softmax_scale * 1.4426950408889634f, static_cast<__nv_bfloat16*>(out), ldo, first_slot);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
