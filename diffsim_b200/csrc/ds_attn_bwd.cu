// K5 -- backward of the attention (SDPA) and of the directional Aligned Attention Score (tensor-core bound).
//
// Deterministic FlashAttention-2 split: no float atomics, every gradient element is owned by one thread of one CTA and
// is ADDED INTO the caller's fp32 buffer, so a repeated call (and any sequence of calls) is bitwise reproducible.
//
//   dQ kernel    one CTA per (b, h, 128-row q tile), looping over 128-row kv tiles twice:
//                  pass 1  S = Q K^T (SS)                          -> per-row log-sum-exp (online max / sum)
//                  pass 2  S = Q K^T, dP = dO V^T (SS)              -> P = exp2(S scale log2e - LSE2),
//                          dS = P (dP - delta) written as 16-bit IN PLACE over S (TMEM)
//                          dQ += dS K (TS: A = dS from TMEM, B = K as the MN-major operand, like K1's P V)
//                delta = rowsum(dO o O) is taken from global memory in the prologue; LSE and delta go to the workspace.
//   dK/dV kernel one CTA per (b, h, 128-row kv tile), looping over q blocks of BQ rows:
//                  S^T = K Q^T, dP^T = V dO^T (SS)                  -> P^T, dS^T = P^T (dP^T - delta), 16-bit in place
//                  dV += P^T dO, dK += dS^T Q (TS)
//                BQ = 128 while 2 x 128 + 2 x D_PAD TMEM columns fit in 512; at D = 160 (576 columns) BQ = 64 (448).
//
// Operand forms are exactly K1's (ds_attn.cu): 128B / 64B-swizzled TMA tiles of D_PAD columns, K-major for the SS
// products and MN-major for the B operand of the TS products.  One thread issues TMA and MMA; the four warps of the CTA
// own the 128 TMEM lanes (one row each) for the elementwise work.  The phases of an iteration are serialised (load,
// MMA, softmax-gradient, MMA); overlapping them is future work.
//
// All products carry 16-bit operands and fp32 accumulators.  The gradients are linear in dO, so a common scalar factor
// of dO (the similarity gradient g / (|X| |Y|) or 2 g / E, read from device memory) and the softmax scale are applied to
// the fp32 accumulators only: the 16-bit dO operand stays O(1) even where the true dO would underflow fp16.
//
// Algorithmic work per attention backward: 10 B H Sq Skv D flops (QK^T recompute, dP, dV, dK, dQ); this implementation
// issues 12 (the LSE pass recomputes QK^T once more).
#include <algorithm>

#include "ds_attn_common.cuh"

namespace ds {
namespace bwd {

constexpr int kThreads = 128;   // four warps = the four TMEM lane quadrants
constexpr int kTile = 128;      // q rows of a dQ stream, kv rows of a dK/dV stream, kv rows per dQ step

template <int D>
struct Cfg : AttnTile<D> {   // K1's operand tiles
  using Tile = AttnTile<D>;
  static constexpr int BQ = (2 * 128 + 2 * Tile::D_PAD <= 512) ? 128 : 64;   // q rows per dK/dV step
  static constexpr int TILE_BYTES = Tile::NSUB * kTile * Tile::SUB_BYTES;      // 128-row tile
  static constexpr int QB_BYTES = Tile::NSUB * BQ * Tile::SUB_BYTES;           // BQ-row tile
  static constexpr int DQ_SMEM = 4 * TILE_BYTES + 1024;                        // Q, dO, K, V + barriers
  static constexpr int DKV_SMEM = 2 * TILE_BYTES + 2 * QB_BYTES + 2 * BQ * 4 + 1024;
  static_assert(256 + Tile::D_PAD <= 512, "dQ TMEM budget");
  static_assert(2 * BQ + 2 * Tile::D_PAD <= 512, "dK/dV TMEM budget");
  static_assert(DQ_SMEM <= 232448 && DKV_SMEM <= 232448, "shared memory");
  static_assert((kTile * Tile::SUB_BYTES) % 1024 == 0 && (BQ * Tile::SUB_BYTES) % 1024 == 0,
                "swizzle atoms need 1024-byte tiles");
};

struct Params {
  int B, H, Sq, Skv, n_qt, n_kt;
  float scale, scale_log2;
  const void* o;      // forward output (16-bit), for delta
  int64_t o_sb, o_sh, o_ss;
  const void* dout;   // (scaled-down) output gradient (16-bit)
  int64_t do_sb, do_sh, do_ss;
  float* lse;         // [B H][n_qt 128] log2-domain log-sum-exp (written by the dQ kernel)
  float* delta;       // [B H][n_qt 128]
  const float* coef;  // optional device scalar multiplying every gradient
  float* dq;
  int64_t dq_sb, dq_sh, dq_ss;
  float* dk;
  int64_t dk_sb, dk_sh, dk_ss;
  float* dv;
  int64_t dv_sb, dv_sh, dv_ss;
};

// rows x D_PAD tile of a (B, H, S, D) tensor, as K1 loads it: NSUB swizzled sub-tiles of SUBW columns
template <int D>
__device__ __forceinline__ void load_tile(uint8_t* dst, const CUtensorMap* m, uint64_t* bar, int rows, int row0, int h,
                                          int b) {
  using C = Cfg<D>;
#pragma unroll
  for (int s = 0; s < C::NSUB; ++s) tma_load_5d(dst + s * rows * C::SUB_BYTES, m, bar, s * C::SUBW, row0, h, b, 0);
}

// D[tmem] (+)= A B^T over the head dim, both operands K-major tiles (K1's Q K^T form).  a_rows / b_rows: rows of the
// smem tiles (the sub-tile pitch).
template <int D>
__device__ __forceinline__ void mma_ss_kmajor(uint32_t d_tmem, const uint8_t* a, int a_rows, const uint8_t* b, int b_rows,
                                              uint32_t idesc) {
  using C = Cfg<D>;
  constexpr uint32_t SBO = 8 * C::SUB_BYTES;
  const uint64_t a0 = umma_smem_desc(smem_u32(a), 16, SBO, C::LAYOUT);
  const uint64_t b0 = umma_smem_desc(smem_u32(b), 16, SBO, C::LAYOUT);
#pragma unroll
  for (int kc = 0; kc < C::D_PAD / 16; ++kc) {
    const int sub = kc / C::CPS, off = (kc % C::CPS) * 32;
    umma_f16_ss(d_tmem, a0 + (uint64_t)((sub * a_rows * C::SUB_BYTES + off) >> 4),
                b0 + (uint64_t)((sub * b_rows * C::SUB_BYTES + off) >> 4), idesc, kc > 0 ? 1u : 0u);
  }
}

// D[tmem] (+)= A[tmem] B over k_rows rows of B, A packed 16-bit in TMEM as K1's P (32-column groups, the first 16
// columns of each holding 32 values), B an MN-major tile of k_rows rows (K1's P V form)
template <int D>
__device__ __forceinline__ void mma_ts_mnmajor(uint32_t d_tmem, uint32_t a_tmem, const uint8_t* b, int k_rows,
                                               uint32_t idesc, bool accumulate) {
  using C = Cfg<D>;
  const uint64_t b0 = umma_smem_desc(smem_u32(b), k_rows * C::SUB_BYTES, 8 * C::SUB_BYTES, C::LAYOUT);
#pragma unroll 1
  for (int ks = 0; ks < k_rows / 16; ++ks)
    umma_f16_ts(d_tmem, a_tmem + (ks >> 1) * 32 + (ks & 1) * 8, b0 + (uint64_t)((ks * 16 * C::SUB_BYTES) >> 4), idesc,
                (accumulate || ks > 0) ? 1u : 0u);
}

__device__ __forceinline__ void sync_all_tc() {
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
}

template <bool kBf16>
__device__ __forceinline__ float row_dot(const void* x, const void* y, int n) {
  const uint4* a = static_cast<const uint4*>(x);
  const uint4* b = static_cast<const uint4*>(y);
  float acc = 0.f;
  for (int i = 0; i < n / 8; ++i) {
    const uint4 va = a[i], vb = b[i];
    const uint32_t ua[4] = {va.x, va.y, va.z, va.w}, ub[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = unpack2<kBf16>(ua[j]), fb = unpack2<kBf16>(ub[j]);
      acc = fmaf(fa.x, fb.x, acc);
      acc = fmaf(fa.y, fb.y, acc);
    }
  }
  return acc;
}

// fp32 accumulator columns [col, col + D) of this thread's TMEM lane, times f, added into out[0 .. D)
template <int D>
__device__ __forceinline__ void add_row_out(uint32_t taddr, float f, float* out, bool ok) {
  using C = Cfg<D>;
#pragma unroll 1
  for (int c = 0; c < C::D_PAD / 16; ++c) {
    uint32_t v[16];
    tmem_ld_x16(taddr + c * 16, v);
    tmem_wait_ld();
    if (ok) {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (c * 16 + j < D) out[c * 16 + j] += __uint_as_float(v[j]) * f;
    }
  }
}

template <int D, bool kBf16>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                   const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do, const Params p) {
  using C = Cfg<D>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sDO = sQ + C::TILE_BYTES;
  uint8_t* sK = sDO + C::TILE_BYTES;
  uint8_t* sV = sK + C::TILE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + C::TILE_BYTES);
  uint64_t* q_bar = bars;
  uint64_t* kv_bar = bars + 1;
  uint64_t* mma_bar = bars + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5;
  const int bh = blockIdx.x / p.n_qt, qt = blockIdx.x - bh * p.n_qt;
  const int b = bh / p.H, h = bh - b * p.H;
  const int grow = qt * kTile + tid;
  const bool row_ok = grow < p.Sq;

  if (tid == 0) {
    mbar_init(q_bar, 1);
    mbar_init(kv_bar, 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    tma_prefetch_desc(&map_do);
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  sync_all_tc();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_t = tmem + ((uint32_t)(warp * 32) << 16);
  constexpr uint32_t kS = 0, kDP = 128, kDQ = 256;
  const uint32_t fmt = kBf16 ? 1u : 0u;
  const uint32_t idesc_s = umma_idesc_f16(fmt, kTile, kTile, 0, 0);
  const uint32_t idesc_dq = umma_idesc_f16(fmt, kTile, C::D_PAD, 0, 1);

  if (tid == 0) {
    mbar_arrive_expect_tx(q_bar, 2 * C::TILE_BYTES);
    load_tile<D>(sQ, &map_q, q_bar, kTile, qt * kTile, h, b);
    load_tile<D>(sDO, &map_do, q_bar, kTile, qt * kTile, h, b);
  }
  __syncwarp();
  // delta = rowsum(dO o O) in fp32 (while the tiles land)
  float delta = 0.f;
  if (row_ok) {
    const uint8_t* o = static_cast<const uint8_t*>(p.o) + 2 * (b * p.o_sb + h * p.o_sh + grow * p.o_ss);
    const uint8_t* g = static_cast<const uint8_t*>(p.dout) + 2 * (b * p.do_sb + h * p.do_sh + grow * p.do_ss);
    delta = row_dot<kBf16>(o, g, D);
  }
  const float sl2 = p.scale_log2;
  uint32_t kv_ph = 0, mma_ph = 0;
  mbar_wait(q_bar, 0);

  // ---- pass 1: log-sum-exp of every row (log2 domain)
  float m = -INFINITY, l = 0.f;
  for (int kt = 0; kt < p.n_kt; ++kt) {
    if (tid == 0) {
      mbar_arrive_expect_tx(kv_bar, C::TILE_BYTES);
      load_tile<D>(sK, &map_k, kv_bar, kTile, kt * kTile, h, b);
    }
    __syncwarp();
    mbar_wait(kv_bar, kv_ph);
    kv_ph ^= 1;
    if (tid == 0) {
      tc_fence_after_sync();
      mma_ss_kmajor<D>(tmem + kS, sQ, kTile, sK, kTile, idesc_s);
      umma_commit(mma_bar);
    }
    __syncwarp();
    mbar_wait(mma_bar, mma_ph);
    mma_ph ^= 1;
    tc_fence_after_sync();
    const int nv = p.Skv - kt * kTile;   // valid kv columns of this tile (>= 1)
#pragma unroll 1
    for (int c = 0; c < kTile / 32; ++c) {
      uint32_t v[32];
      tmem_ld_x32(lane_t + kS + c * 32, v);
      tmem_wait_ld();
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (c * 32 + j >= nv) v[j] = 0xff800000u;
        mx = fmaxf(mx, __uint_as_float(v[j]));
      }
      if (mx == -INFINITY) continue;
      const float mn = fmaxf(m, mx);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) s += fast_exp2((__uint_as_float(v[j]) - mn) * sl2);
      l = l * fast_exp2((m - mn) * sl2) + s;
      m = mn;
    }
    sync_all_tc();   // S read out before the next tile's MMA overwrites it
  }
  const float lse2 = m * sl2 + __log2f(l);
  {
    const size_t i = (size_t)bh * (p.n_qt * kTile) + grow;
    p.lse[i] = lse2;
    p.delta[i] = delta;
  }

  // ---- pass 2: dQ
  for (int kt = 0; kt < p.n_kt; ++kt) {
    if (tid == 0) {
      mbar_arrive_expect_tx(kv_bar, 2 * C::TILE_BYTES);
      load_tile<D>(sK, &map_k, kv_bar, kTile, kt * kTile, h, b);
      load_tile<D>(sV, &map_v, kv_bar, kTile, kt * kTile, h, b);
    }
    __syncwarp();
    mbar_wait(kv_bar, kv_ph);
    kv_ph ^= 1;
    if (tid == 0) {
      tc_fence_after_sync();
      mma_ss_kmajor<D>(tmem + kS, sQ, kTile, sK, kTile, idesc_s);    // S = Q K^T
      mma_ss_kmajor<D>(tmem + kDP, sDO, kTile, sV, kTile, idesc_s);  // dP = dO V^T
      umma_commit(mma_bar);
    }
    __syncwarp();
    mbar_wait(mma_bar, mma_ph);
    mma_ph ^= 1;
    tc_fence_after_sync();
    const int nv = p.Skv - kt * kTile;
#pragma unroll 1
    for (int c = 0; c < kTile / 32; ++c) {
      uint32_t s[32], dp[32], pk[16];
      tmem_ld_x32(lane_t + kS + c * 32, s);
      tmem_ld_x32(lane_t + kDP + c * 32, dp);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        float ds[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float pr = (c * 32 + j + e < nv) ? fast_exp2(fmaf(__uint_as_float(s[j + e]), sl2, -lse2)) : 0.f;
          ds[e] = pr * (__uint_as_float(dp[j + e]) - delta);
        }
        pk[j >> 1] = pack2<kBf16>(ds[0], ds[1]);
      }
      tmem_st_x16(lane_t + kS + c * 32, pk);   // dS over the first 16 of the 32 S columns just read
    }
    tmem_wait_st();
    sync_all_tc();
    if (tid == 0) {
      mma_ts_mnmajor<D>(tmem + kDQ, tmem + kS, sK, kTile, idesc_dq, kt > 0);   // dQ += dS K
      umma_commit(mma_bar);
    }
    __syncwarp();
    mbar_wait(mma_bar, mma_ph);   // K / V buffers and the S columns are free again
    mma_ph ^= 1;
    tc_fence_after_sync();
  }

  const float f = p.scale * (p.coef ? *p.coef : 1.0f);
  add_row_out<D>(lane_t + kDQ, f, p.dq + b * p.dq_sb + h * p.dq_sh + (int64_t)grow * p.dq_ss, row_ok);
  sync_all_tc();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int D, bool kBf16>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do, const Params p) {
  using C = Cfg<D>;
  constexpr int BQ = C::BQ;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sK = smem;
  uint8_t* sV = sK + C::TILE_BYTES;
  uint8_t* sQ = sV + C::TILE_BYTES;
  uint8_t* sDO = sQ + C::QB_BYTES;
  float* sLse = reinterpret_cast<float*>(sDO + C::QB_BYTES);
  float* sDelta = sLse + BQ;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDelta + BQ);
  uint64_t* kv_bar = bars;
  uint64_t* q_bar = bars + 1;
  uint64_t* mma_bar = bars + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5;
  const int bh = blockIdx.x / p.n_kt, kt = blockIdx.x - bh * p.n_kt;
  const int b = bh / p.H, h = bh - b * p.H;
  const int krow = kt * kTile + tid;
  const bool row_ok = krow < p.Skv;

  if (tid == 0) {
    mbar_init(kv_bar, 1);
    mbar_init(q_bar, 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
    tma_prefetch_desc(&map_do);
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  sync_all_tc();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_t = tmem + ((uint32_t)(warp * 32) << 16);
  constexpr uint32_t kST = 0, kDPT = BQ, kDV = 2 * BQ, kDK = 2 * BQ + C::D_PAD;
  const uint32_t fmt = kBf16 ? 1u : 0u;
  const uint32_t idesc_s = umma_idesc_f16(fmt, kTile, BQ, 0, 0);
  const uint32_t idesc_o = umma_idesc_f16(fmt, kTile, C::D_PAD, 0, 1);

  if (tid == 0) {
    mbar_arrive_expect_tx(kv_bar, 2 * C::TILE_BYTES);
    load_tile<D>(sK, &map_k, kv_bar, kTile, kt * kTile, h, b);
    load_tile<D>(sV, &map_v, kv_bar, kTile, kt * kTile, h, b);
  }
  __syncwarp();
  const float sl2 = p.scale_log2;
  const int n_qb = (p.Sq + BQ - 1) / BQ;
  const float* lse_bh = p.lse + (size_t)bh * (p.n_qt * kTile);
  const float* delta_bh = p.delta + (size_t)bh * (p.n_qt * kTile);
  uint32_t q_ph = 0, mma_ph = 0;
  mbar_wait(kv_bar, 0);
  for (int qb = 0; qb < n_qb; ++qb) {
    if (tid == 0) {
      mbar_arrive_expect_tx(q_bar, 2 * C::QB_BYTES);
      load_tile<D>(sQ, &map_q, q_bar, BQ, qb * BQ, h, b);
      load_tile<D>(sDO, &map_do, q_bar, BQ, qb * BQ, h, b);
    }
    __syncwarp();
    if (tid < BQ) {
      sLse[tid] = lse_bh[qb * BQ + tid];
      sDelta[tid] = delta_bh[qb * BQ + tid];
    }
    mbar_wait(q_bar, q_ph);
    q_ph ^= 1;
    if (tid == 0) {
      tc_fence_after_sync();
      mma_ss_kmajor<D>(tmem + kST, sK, kTile, sQ, BQ, idesc_s);    // S^T = K Q^T
      mma_ss_kmajor<D>(tmem + kDPT, sV, kTile, sDO, BQ, idesc_s);  // dP^T = V dO^T
      umma_commit(mma_bar);
    }
    __syncwarp();
    __syncthreads();   // sLse / sDelta
    mbar_wait(mma_bar, mma_ph);
    mma_ph ^= 1;
    tc_fence_after_sync();
    const int nq = p.Sq - qb * BQ;   // valid q columns of this block
#pragma unroll 1
    for (int c = 0; c < BQ / 32; ++c) {
      uint32_t s[32], dp[32], pk[16], dk[16];
      tmem_ld_x32(lane_t + kST + c * 32, s);
      tmem_ld_x32(lane_t + kDPT + c * 32, dp);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        float pr[2], ds[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int q = c * 32 + j + e;
          pr[e] = q < nq ? fast_exp2(fmaf(__uint_as_float(s[j + e]), sl2, -sLse[q])) : 0.f;
          ds[e] = pr[e] * (__uint_as_float(dp[j + e]) - sDelta[q]);
        }
        pk[j >> 1] = pack2<kBf16>(pr[0], pr[1]);
        dk[j >> 1] = pack2<kBf16>(ds[0], ds[1]);
      }
      tmem_st_x16(lane_t + kST + c * 32, pk);    // P^T over S^T
      tmem_st_x16(lane_t + kDPT + c * 32, dk);   // dS^T over dP^T
    }
    tmem_wait_st();
    sync_all_tc();
    if (tid == 0) {
      mma_ts_mnmajor<D>(tmem + kDV, tmem + kST, sDO, BQ, idesc_o, qb > 0);   // dV += P^T dO
      mma_ts_mnmajor<D>(tmem + kDK, tmem + kDPT, sQ, BQ, idesc_o, qb > 0);   // dK += dS^T Q
      umma_commit(mma_bar);
    }
    __syncwarp();
    mbar_wait(mma_bar, mma_ph);   // Q / dO buffers, sLse and the S^T / dP^T columns are free again
    mma_ph ^= 1;
    tc_fence_after_sync();
    __syncthreads();
  }

  const float g = p.coef ? *p.coef : 1.0f;
  add_row_out<D>(lane_t + kDV, g, p.dv + b * p.dv_sb + h * p.dv_sh + (int64_t)krow * p.dv_ss, row_ok);
  add_row_out<D>(lane_t + kDK, g * p.scale, p.dk + b * p.dk_sb + h * p.dk_sh + (int64_t)krow * p.dk_ss, row_ok);
  sync_all_tc();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------
// similarity gradient (ds_aas_dir_bwd)
// ---------------------------------------------------------------------------
constexpr int kRedBlocks = 256, kRedThreads = 256;

// per-block (dot(X,Y), |X|^2, |Y|^2) over n contiguous elements, fixed split (deterministic)
template <bool kBf16>
__global__ void sim_partials_kernel(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2,
                                    float* __restrict__ part) {
  float d = 0.f, xx = 0.f, yy = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
    const float2 a = unpack2<kBf16>(x[i]), c = unpack2<kBf16>(y[i]);
    d = fmaf(a.x, c.x, fmaf(a.y, c.y, d));
    xx = fmaf(a.x, a.x, fmaf(a.y, a.y, xx));
    yy = fmaf(c.x, c.x, fmaf(c.y, c.y, yy));
  }
  __shared__ float red[3][kRedThreads / 32];
  d = warp_sum(d);
  xx = warp_sum(xx);
  yy = warp_sum(yy);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    red[0][w] = d;
    red[1][w] = xx;
    red[2][w] = yy;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    float s = 0.f;
    for (int i = 0; i < kRedThreads / 32; ++i) s += red[threadIdx.x][i];
    part[blockIdx.x * 3 + threadIdx.x] = s;
  }
}

// coef = {gradient factor of X, of Y, k_X, k_Y}: dX = coef[0] (Y - k_X X), dY = coef[1] (X - k_Y Y) for the cosine
// (torch's per-norm max(|.|, 1e-8) clamp: a clamped norm contributes no k term); dX = -dY = coef[0] (X - Y) for MSE
__global__ void sim_coef_kernel(const float* __restrict__ part, int mode, double E, const float* __restrict__ d_dir,
                                float* __restrict__ coef) {
  if (threadIdx.x != 0) return;
  const float g = *d_dir;
  if (mode == DS_SIM_MSE) {
    const float c = (float)(2.0 * (double)g / E);
    coef[0] = c;
    coef[1] = c;
    coef[2] = coef[3] = 0.f;
    return;
  }
  double d = 0, xx = 0, yy = 0;
  for (int i = 0; i < kRedBlocks; ++i) {
    d += part[3 * i];
    xx += part[3 * i + 1];
    yy += part[3 * i + 2];
  }
  const double nx = sqrt(xx), ny = sqrt(yy);
  const double cx = fmax(nx, 1e-8), cy = fmax(ny, 1e-8);
  const double cos = d / (cx * cy);
  coef[0] = (float)((double)g / (cx * cy));
  coef[1] = coef[0];
  coef[2] = nx > 1e-8 ? (float)(cos * cy / cx) : 0.f;
  coef[3] = ny > 1e-8 ? (float)(cos * cx / cy) : 0.f;
}

// the O(1) factors of dX and dY, rounded to the input dtype (the dO operands of the two attention backwards)
template <bool kBf16>
__global__ void sim_factor_kernel(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2, int mode,
                                  const float* __restrict__ coef, uint32_t* __restrict__ fx, uint32_t* __restrict__ fy) {
  const float kx = coef[2], ky = coef[3];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
    const float2 a = unpack2<kBf16>(x[i]), c = unpack2<kBf16>(y[i]);
    if (mode == DS_SIM_MSE) {
      fx[i] = pack2<kBf16>(a.x - c.x, a.y - c.y);
      fy[i] = pack2<kBf16>(c.x - a.x, c.y - a.y);
    } else {
      fx[i] = pack2<kBf16>(c.x - kx * a.x, c.y - kx * a.y);
      fy[i] = pack2<kBf16>(a.x - ky * c.x, a.y - ky * c.y);
    }
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int check_grad(const ds_tensor4& g, const ds_tensor4& like, const char* who, const char* name) {
  if (!g.ptr) return fail(DS_ERR_INVALID, "%s: %s: null pointer", who, name);
  if (g.dtype != DS_F32) return fail(DS_ERR_INVALID, "%s: %s: gradients are float32", who, name);
  for (int i = 0; i < 4; ++i)
    if (g.size[i] != like.size[i]) return fail(DS_ERR_INVALID, "%s: %s: shape must match its input", who, name);
  if (g.stride[3] != 1) return fail(DS_ERR_INVALID, "%s: %s: innermost stride must be 1", who, name);
  if ((uintptr_t)g.ptr & 3) return fail(DS_ERR_INVALID, "%s: %s: base pointer must be 4-byte aligned", who, name);
  for (int i = 0; i < 3; ++i)
    if (g.size[i] > 1 && g.stride[i] <= 0) return fail(DS_ERR_INVALID, "%s: %s: stride[%d] must be positive", who, name, i);
  return DS_OK;
}

// q, k, v: shapes, dtypes and layouts of one attention backward
static int check_attn(const ds_tensor4& q, const ds_tensor4& k, const ds_tensor4& v, const char* who) {
  int rc;
  if ((rc = check_operand(lift(q), who, "q")) != DS_OK || (rc = check_operand(lift(k), who, "k")) != DS_OK ||
      (rc = check_operand(lift(v), who, "v")) != DS_OK)
    return rc;
  if (k.dtype != q.dtype || v.dtype != q.dtype) return fail(DS_ERR_INVALID, "%s: q, k and v must share one dtype", who);
  for (int i : {0, 1, 3})
    if (k.size[i] != q.size[i] || v.size[i] != q.size[i]) return fail(DS_ERR_INVALID, "%s: B, H and D must match across q, k, v", who);
  if (v.size[2] != k.size[2]) return fail(DS_ERR_INVALID, "%s: k and v must have the same length", who);
  if (q.size[2] > INT32_MAX / 2 || k.size[2] > INT32_MAX / 2) return fail(DS_ERR_INVALID, "%s: sequence too long", who);
  return with_head_dim(q.size[3], who, [](auto) { return DS_OK; });
}

static size_t stats_bytes(const ds_tensor4& q) {
  const int64_t n_qt = (q.size[2] + kTile - 1) / kTile;
  return 2 * align_up((size_t)(q.size[0] * q.size[1] * n_qt * kTile) * sizeof(float), 256);
}

struct BwdArgs {
  ds_tensor4 q, k, v, out, dout, dq, dk, dv;
  float scale;
  const float* coef;
  float* lse;
  float* delta;
};

template <int D, bool kBf16>
static int launch_bwd_t(const BwdArgs& a, cudaStream_t st) {
  using C = Cfg<D>;
  CUtensorMap mq, mk, mv, mdo, mqb, mdob;
  int rc;
  const ds_tensor5 q = lift(a.q), dout = lift(a.dout);
  if ((rc = make_map(&mq, q, C::SUBW, kTile)) != DS_OK || (rc = make_map(&mk, lift(a.k), C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mv, lift(a.v), C::SUBW, kTile)) != DS_OK || (rc = make_map(&mdo, dout, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mqb, q, C::SUBW, C::BQ)) != DS_OK || (rc = make_map(&mdob, dout, C::SUBW, C::BQ)) != DS_OK)
    return rc;
  Params p;
  p.B = (int)a.q.size[0];
  p.H = (int)a.q.size[1];
  p.Sq = (int)a.q.size[2];
  p.Skv = (int)a.k.size[2];
  p.n_qt = (p.Sq + kTile - 1) / kTile;
  p.n_kt = (p.Skv + kTile - 1) / kTile;
  p.scale = a.scale > 0.f ? a.scale : 1.0f / sqrtf((float)D);
  p.scale_log2 = p.scale * 1.4426950408889634f;
  p.o = a.out.ptr;
  p.o_sb = a.out.stride[0], p.o_sh = a.out.stride[1], p.o_ss = a.out.stride[2];
  p.dout = a.dout.ptr;
  p.do_sb = a.dout.stride[0], p.do_sh = a.dout.stride[1], p.do_ss = a.dout.stride[2];
  p.lse = a.lse;
  p.delta = a.delta;
  p.coef = a.coef;
  p.dq = static_cast<float*>(a.dq.ptr);
  p.dq_sb = a.dq.stride[0], p.dq_sh = a.dq.stride[1], p.dq_ss = a.dq.stride[2];
  p.dk = static_cast<float*>(a.dk.ptr);
  p.dk_sb = a.dk.stride[0], p.dk_sh = a.dk.stride[1], p.dk_ss = a.dk.stride[2];
  p.dv = static_cast<float*>(a.dv.ptr);
  p.dv_sb = a.dv.stride[0], p.dv_sh = a.dv.stride[1], p.dv_ss = a.dv.stride[2];
  const int64_t bh = (int64_t)p.B * p.H;
  if (bh * p.n_qt >= INT32_MAX || bh * p.n_kt >= INT32_MAX) return fail(DS_ERR_INVALID, "attention backward: too many tiles");
  DS_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dq_kernel<D, kBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::DQ_SMEM));
  DS_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dkv_kernel<D, kBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::DKV_SMEM));
  attn_bwd_dq_kernel<D, kBf16><<<(unsigned)(bh * p.n_qt), kThreads, C::DQ_SMEM, st>>>(mq, mk, mv, mdo, p);
  DS_CUDA_TRY(cudaGetLastError());
  attn_bwd_dkv_kernel<D, kBf16><<<(unsigned)(bh * p.n_kt), kThreads, C::DKV_SMEM, st>>>(mqb, mk, mv, mdob, p);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

static int launch_bwd(const BwdArgs& a, const char* who, cudaStream_t st) {
  return with_head_dim(a.q.size[3], who, [&](auto d) {
    return with_dtype(a.q.dtype, [&](auto bf) { return launch_bwd_t<decltype(d)::value, decltype(bf)::value>(a, st); });
  });
}

static ds_tensor4 contiguous_like(const ds_tensor4& t, void* ptr) {
  ds_tensor4 r = t;
  r.ptr = ptr;
  r.stride[3] = 1;
  r.stride[2] = t.size[3];
  r.stride[1] = t.size[2] * t.size[3];
  r.stride[0] = t.size[1] * t.size[2] * t.size[3];
  return r;
}

}  // namespace bwd
}  // namespace ds

extern "C" {

size_t ds_attn_bwd_workspace_bytes(ds_tensor4 q, ds_tensor4 k) {
  (void)k;
  return ds::bwd::stats_bytes(q) + 256;
}

int ds_attn_bwd(ds_tensor4 q, ds_tensor4 k, ds_tensor4 v, ds_tensor4 out, ds_tensor4 dout, float scale, ds_tensor4 dq,
                ds_tensor4 dk, ds_tensor4 dv, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_attn_bwd";
  int rc;
  if ((rc = check_attn(q, k, v, who)) != DS_OK || (rc = check_like(lift(out), lift(q), who, "out")) != DS_OK ||
      (rc = check_like(lift(dout), lift(q), who, "dout")) != DS_OK || (rc = check_grad(dq, q, who, "dq")) != DS_OK ||
      (rc = check_grad(dk, k, who, "dk")) != DS_OK || (rc = check_grad(dv, v, who, "dv")) != DS_OK)
    return rc;
  Workspace w(ws, ws_bytes);
  const size_t half = stats_bytes(q) / 2;
  float* lse = static_cast<float*>(w.take(half));
  float* delta = static_cast<float*>(w.take(half));
  if (!lse || !delta)
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes, ds_attn_bwd_workspace_bytes(q, k));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  BwdArgs a{q, k, v, out, dout, dq, dk, dv, scale, nullptr, lse, delta};
  return launch_bwd(a, who, static_cast<cudaStream_t>(stream));
}

size_t ds_aas_dir_bwd_workspace_bytes(ds_tensor4 q_i, ds_tensor4 k_j) {
  using namespace ds;
  (void)k_j;
  const size_t e = align_up((size_t)(q_i.size[0] * q_i.size[1] * q_i.size[2] * q_i.size[3]) * 2, 256);
  return 4 * e + bwd::stats_bytes(q_i) + align_up(bwd::kRedBlocks * 3 * sizeof(float), 256) + 256 /*coef*/ +
         1024 /*forward meta*/ + 256;
}

int ds_aas_dir_bwd(ds_tensor4 q_i, ds_tensor4 k_i, ds_tensor4 v_i, ds_tensor4 k_j, ds_tensor4 v_j, float scale, int mode,
                   const float* d_dir, ds_tensor4 dq_i, ds_tensor4 dk_i, ds_tensor4 dv_i, ds_tensor4 dk_j, ds_tensor4 dv_j,
                   void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_aas_dir_bwd";
  int rc;
  if ((rc = check_attn(q_i, k_i, v_i, who)) != DS_OK || (rc = check_attn(q_i, k_j, v_j, who)) != DS_OK) return rc;
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return fail(DS_ERR_INVALID, "%s: bad mode %d", who, mode);
  if (!d_dir) return fail(DS_ERR_INVALID, "%s: d_dir: null pointer", who);
  if ((rc = check_grad(dq_i, q_i, who, "dq_i")) != DS_OK || (rc = check_grad(dk_i, k_i, who, "dk_i")) != DS_OK ||
      (rc = check_grad(dv_i, v_i, who, "dv_i")) != DS_OK || (rc = check_grad(dk_j, k_j, who, "dk_j")) != DS_OK ||
      (rc = check_grad(dv_j, v_j, who, "dv_j")) != DS_OK)
    return rc;
  const int64_t n = q_i.size[0] * q_i.size[1] * q_i.size[2] * q_i.size[3];
  Workspace w(ws, ws_bytes);
  void* x = w.take((size_t)n * 2);
  void* y = w.take((size_t)n * 2);
  void* fx = w.take((size_t)n * 2);
  void* fy = w.take((size_t)n * 2);
  const size_t half = stats_bytes(q_i) / 2;
  float* lse = static_cast<float*>(w.take(half));
  float* delta = static_cast<float*>(w.take(half));
  float* part = static_cast<float*>(w.take(kRedBlocks * 3 * sizeof(float)));
  float* coef = static_cast<float*>(w.take(4 * sizeof(float)));
  void* meta = w.take(1024);
  if (!x || !y || !fx || !fy || !lse || !delta || !part || !coef || !meta)
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_aas_dir_bwd_workspace_bytes(q_i, k_j));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // X = Attn(Q_i, K_j, V_j), Y = Attn(Q_i, K_i, V_i), rounded to the input dtype as in the forward score
  const ds_tensor4 X = contiguous_like(q_i, x), Y = contiguous_like(q_i, y);
  if ((rc = ds_attn_fwd(q_i, k_j, v_j, scale, X, meta, 1024, stream)) != DS_OK) return rc;
  if ((rc = ds_attn_fwd(q_i, k_i, v_i, scale, Y, meta, 1024, stream)) != DS_OK) return rc;
  const bool bf = q_i.dtype == DS_BF16;
  const int64_t n2 = n / 2;   // D is even
  const uint32_t* xu = static_cast<const uint32_t*>(x);
  const uint32_t* yu = static_cast<const uint32_t*>(y);
  if (bf) sim_partials_kernel<true><<<kRedBlocks, kRedThreads, 0, st>>>(xu, yu, n2, part);
  else sim_partials_kernel<false><<<kRedBlocks, kRedThreads, 0, st>>>(xu, yu, n2, part);
  DS_CUDA_TRY(cudaGetLastError());
  sim_coef_kernel<<<1, 32, 0, st>>>(part, mode, (double)n, d_dir, coef);
  DS_CUDA_TRY(cudaGetLastError());
  const unsigned fb = (unsigned)std::min<int64_t>((n2 + 255) / 256, 4 * (int64_t)sm_count());
  if (bf) sim_factor_kernel<true><<<fb, 256, 0, st>>>(xu, yu, n2, mode, coef, (uint32_t*)fx, (uint32_t*)fy);
  else sim_factor_kernel<false><<<fb, 256, 0, st>>>(xu, yu, n2, mode, coef, (uint32_t*)fx, (uint32_t*)fy);
  DS_CUDA_TRY(cudaGetLastError());
  // cross term first, then the self term: dq_i receives its two contributions in this fixed order
  BwdArgs cross{q_i, k_j, v_j, X, contiguous_like(q_i, fx), dq_i, dk_j, dv_j, scale, coef + 0, lse, delta};
  if ((rc = launch_bwd(cross, who, st)) != DS_OK) return rc;
  BwdArgs self{q_i, k_i, v_i, Y, contiguous_like(q_i, fy), dq_i, dk_i, dv_i, scale, coef + 1, lse, delta};
  return launch_bwd(self, who, st);
}

}  // extern "C"
