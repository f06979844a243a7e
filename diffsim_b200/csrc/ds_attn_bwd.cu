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
// Each kernel exists in two forms that run the same per-term body (dq_term, dkv_term) and the same prologue: the single
// kernels run it once, for ds_attn_bwd and ds_aas_dir_bwd; the list kernels run it once per term of a device-built
// contribution list, for ds_aas_groups_bwd and ds_aas_matrix_bwd.  They differ only in where a term's operands, LSE /
// delta rows and coefficient are found, so the list backwards are bitwise a sequence of single ones by construction.
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
#include <type_traits>

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
  static constexpr int DQ_BARS = 4 * TILE_BYTES;                               // after Q, dO, K, V
  static constexpr int DKV_BARS = 2 * TILE_BYTES + 2 * QB_BYTES + 2 * BQ * 4;  // after K, V, Q, dO, LSE, delta
  static constexpr int DQ_SMEM = DQ_BARS + 1024;
  static constexpr int DKV_SMEM = DKV_BARS + 1024;
  static_assert(256 + Tile::D_PAD <= 512, "dQ TMEM budget");
  static_assert(2 * BQ + 2 * Tile::D_PAD <= 512, "dK/dV TMEM budget");
  static_assert(DQ_SMEM <= 232448 && DKV_SMEM <= 232448, "shared memory");
  static_assert((kTile * Tile::SUB_BYTES) % 1024 == 0 && (BQ * Tile::SUB_BYTES) % 1024 == 0,
                "swizzle atoms need 1024-byte tiles");
};

// the shape of one attention backward, common to the single (Params) and list (ListParams) kernels.  Skv / n_kt: kv
// length and tiles of the cross terms (k, v), Skv_self / n_kt_self: of the self terms (k_self, v_self) of a list; the
// single kernels have one kv length and set both alike.
struct Shape {
  int B, H, Sq, Skv, Skv_self, n_qt, n_kt, n_kt_self;
  float scale, scale_log2;
};

struct Params : Shape {
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
                                          int b, int img = 0) {
  using C = Cfg<D>;
#pragma unroll
  for (int s = 0; s < C::NSUB; ++s) tma_load_5d(dst + s * rows * C::SUB_BYTES, m, bar, s * C::SUBW, row0, h, b, img);
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

// the start of every K5 kernel: its three barriers at bars[0 .. 2], the prefetch of its tensor maps, and all 512 TMEM
// columns (one CTA per SM); returns the TMEM base address
template <class... Maps>
__device__ __forceinline__ uint32_t kernel_prologue(uint64_t* bars, const Maps*... maps) {
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  if (threadIdx.x == 0) {
    mbar_init(bars, 1);
    mbar_init(bars + 1, 1);
    mbar_init(bars + 2, 1);
    fence_mbar_init();
    (tma_prefetch_desc(maps), ...);
  }
  if (threadIdx.x < 32) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  sync_all_tc();
  return *tmem_slot;
}

// One term of a dQ kernel, on the 128-row q tile qt of (b, h): the Q and dO tiles (images q_img of mq and do_img of
// mdo), delta = rowsum(dO o O) from this thread's 16-bit rows o_row and do_row, the LSE pass and the dS / dQ pass over
// the skv rows (the term's own kv length) of image kv_img of mk and mv.  LSE and delta go to *lse and *delta_out,
// dQ x scale coef is added into dq_row.  kStats: the statistics only -- LSE and delta are written, there is no dS / dQ
// pass and no drain (dq_row is not read).
// The barrier phases carry over to the next term.
template <int D, bool kBf16, bool kStats = false>
__device__ __forceinline__ void dq_term(uint8_t* smem, uint32_t tmem, const Shape& p, int b, int h, int qt,
                                        const CUtensorMap* mq, int q_img, const CUtensorMap* mdo, int do_img,
                                        const CUtensorMap* mk, const CUtensorMap* mv, int kv_img, int skv,
                                        const void* o_row, const void* do_row, float* lse, float* delta_out, float coef,
                                        float* dq_row, uint32_t& q_ph, uint32_t& kv_ph, uint32_t& mma_ph) {
  using C = Cfg<D>;
  uint8_t* sQ = smem;
  uint8_t* sDO = sQ + C::TILE_BYTES;
  uint8_t* sK = sDO + C::TILE_BYTES;
  uint8_t* sV = sK + C::TILE_BYTES;
  uint64_t* q_bar = reinterpret_cast<uint64_t*>(smem + C::DQ_BARS);
  uint64_t* kv_bar = q_bar + 1;
  uint64_t* mma_bar = q_bar + 2;
  const int tid = threadIdx.x;
  const uint32_t lane_t = tmem + ((uint32_t)((tid >> 5) * 32) << 16);
  const bool row_ok = qt * kTile + tid < p.Sq;
  constexpr uint32_t kS = 0, kDP = 128, kDQ = 256;
  const uint32_t fmt = kBf16 ? 1u : 0u;
  const uint32_t idesc_s = umma_idesc_f16(fmt, kTile, kTile, 0, 0);
  const uint32_t idesc_dq = umma_idesc_f16(fmt, kTile, C::D_PAD, 0, 1);
  const float sl2 = p.scale_log2;
  const int n_kt = (skv + kTile - 1) / kTile;

  if (tid == 0) {
    mbar_arrive_expect_tx(q_bar, 2 * C::TILE_BYTES);
    load_tile<D>(sQ, mq, q_bar, kTile, qt * kTile, h, b, q_img);
    load_tile<D>(sDO, mdo, q_bar, kTile, qt * kTile, h, b, do_img);
  }
  __syncwarp();
  // delta = rowsum(dO o O) in fp32 (while the tiles land)
  float delta = 0.f;
  if (row_ok) delta = row_dot<kBf16>(o_row, do_row, D);
  mbar_wait(q_bar, q_ph);
  q_ph ^= 1;

  // ---- pass 1: log-sum-exp of every row (log2 domain)
  float m = -INFINITY, l = 0.f;
  for (int kt = 0; kt < n_kt; ++kt) {
    if (tid == 0) {
      mbar_arrive_expect_tx(kv_bar, C::TILE_BYTES);
      load_tile<D>(sK, mk, kv_bar, kTile, kt * kTile, h, b, kv_img);
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
    const int nv = skv - kt * kTile;   // valid kv columns of this tile (>= 1)
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
  *lse = lse2;
  *delta_out = delta;
  // kStats: the last tile's sync_all_tc has freed S, Q and dO for the next term
  if constexpr (!kStats) {
    // ---- pass 2: dQ
    for (int kt = 0; kt < n_kt; ++kt) {
      if (tid == 0) {
        mbar_arrive_expect_tx(kv_bar, 2 * C::TILE_BYTES);
        load_tile<D>(sK, mk, kv_bar, kTile, kt * kTile, h, b, kv_img);
        load_tile<D>(sV, mv, kv_bar, kTile, kt * kTile, h, b, kv_img);
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
      const int nv = skv - kt * kTile;
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

    add_row_out<D>(lane_t + kDQ, p.scale * coef, dq_row, row_ok);
    sync_all_tc();   // dQ read out (and Q / dO free) before the next term
  }
}

// One term of a dK/dV kernel, on the 128-row kv tile kt (< the tiles of skv, the term's kv length) of (b, h): the K and
// V tiles (image kv_img of mk and mv), then per block of BQ q rows the Q and dO tiles (images q_img of mq and do_img of
// mdo) with their LSE and delta, read from the term's (b, h) rows lse and delta.  dV x coef is added into dv_row,
// dK x coef scale into dk_row.  The barrier phases carry over to the next term.
template <int D, bool kBf16>
__device__ __forceinline__ void dkv_term(uint8_t* smem, uint32_t tmem, const Shape& p, int b, int h, int kt,
                                         const CUtensorMap* mk, const CUtensorMap* mv, int kv_img, int skv,
                                         const CUtensorMap* mq, int q_img, const CUtensorMap* mdo, int do_img,
                                         const float* lse, const float* delta, float coef, float* dv_row, float* dk_row,
                                         uint32_t& kv_ph, uint32_t& q_ph, uint32_t& mma_ph) {
  using C = Cfg<D>;
  constexpr int BQ = C::BQ;
  uint8_t* sK = smem;
  uint8_t* sV = sK + C::TILE_BYTES;
  uint8_t* sQ = sV + C::TILE_BYTES;
  uint8_t* sDO = sQ + C::QB_BYTES;
  float* sLse = reinterpret_cast<float*>(sDO + C::QB_BYTES);
  float* sDelta = sLse + BQ;
  uint64_t* kv_bar = reinterpret_cast<uint64_t*>(smem + C::DKV_BARS);
  uint64_t* q_bar = kv_bar + 1;
  uint64_t* mma_bar = kv_bar + 2;
  const int tid = threadIdx.x;
  const uint32_t lane_t = tmem + ((uint32_t)((tid >> 5) * 32) << 16);
  const bool row_ok = kt * kTile + tid < skv;
  constexpr uint32_t kST = 0, kDPT = BQ, kDV = 2 * BQ, kDK = 2 * BQ + C::D_PAD;
  const uint32_t fmt = kBf16 ? 1u : 0u;
  const uint32_t idesc_s = umma_idesc_f16(fmt, kTile, BQ, 0, 0);
  const uint32_t idesc_o = umma_idesc_f16(fmt, kTile, C::D_PAD, 0, 1);
  const float sl2 = p.scale_log2;
  const int n_qb = (p.Sq + BQ - 1) / BQ;

  if (tid == 0) {
    mbar_arrive_expect_tx(kv_bar, 2 * C::TILE_BYTES);
    load_tile<D>(sK, mk, kv_bar, kTile, kt * kTile, h, b, kv_img);
    load_tile<D>(sV, mv, kv_bar, kTile, kt * kTile, h, b, kv_img);
  }
  __syncwarp();
  mbar_wait(kv_bar, kv_ph);
  kv_ph ^= 1;
  for (int qb = 0; qb < n_qb; ++qb) {
    if (tid == 0) {
      mbar_arrive_expect_tx(q_bar, 2 * C::QB_BYTES);
      load_tile<D>(sQ, mq, q_bar, BQ, qb * BQ, h, b, q_img);
      load_tile<D>(sDO, mdo, q_bar, BQ, qb * BQ, h, b, do_img);
    }
    __syncwarp();
    if (tid < BQ) {
      sLse[tid] = lse[qb * BQ + tid];
      sDelta[tid] = delta[qb * BQ + tid];
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

  add_row_out<D>(lane_t + kDV, coef, dv_row, row_ok);
  add_row_out<D>(lane_t + kDK, coef * p.scale, dk_row, row_ok);
  sync_all_tc();   // dK / dV read out (and K / V free) before the next term
}

// one CTA per (b, h, 128-row q tile)
template <int D, bool kBf16>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                   const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do, const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t tmem =
      kernel_prologue(reinterpret_cast<uint64_t*>(smem + Cfg<D>::DQ_BARS), &map_q, &map_k, &map_v, &map_do);
  const int bh = blockIdx.x / p.n_qt, qt = blockIdx.x - bh * p.n_qt;
  const int b = bh / p.H, h = bh - b * p.H;
  const int grow = qt * kTile + threadIdx.x;
  const uint8_t* o = static_cast<const uint8_t*>(p.o) + 2 * (b * p.o_sb + h * p.o_sh + grow * p.o_ss);
  const uint8_t* g = static_cast<const uint8_t*>(p.dout) + 2 * (b * p.do_sb + h * p.do_sh + grow * p.do_ss);
  const size_t i = (size_t)bh * (p.n_qt * kTile) + grow;
  uint32_t q_ph = 0, kv_ph = 0, mma_ph = 0;
  dq_term<D, kBf16>(smem, tmem, p, b, h, qt, &map_q, 0, &map_do, 0, &map_k, &map_v, 0, p.Skv, o, g, p.lse + i,
                    p.delta + i, p.coef ? *p.coef : 1.0f, p.dq + b * p.dq_sb + h * p.dq_sh + (int64_t)grow * p.dq_ss,
                    q_ph, kv_ph, mma_ph);
  if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// one CTA per (b, h, 128-row kv tile)
template <int D, bool kBf16>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do, const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t tmem =
      kernel_prologue(reinterpret_cast<uint64_t*>(smem + Cfg<D>::DKV_BARS), &map_q, &map_k, &map_v, &map_do);
  const int bh = blockIdx.x / p.n_kt, kt = blockIdx.x - bh * p.n_kt;
  const int b = bh / p.H, h = bh - b * p.H;
  const int krow = kt * kTile + threadIdx.x;
  const size_t i = (size_t)bh * (p.n_qt * kTile);
  uint32_t kv_ph = 0, q_ph = 0, mma_ph = 0;
  dkv_term<D, kBf16>(smem, tmem, p, b, h, kt, &map_k, &map_v, 0, p.Skv, &map_q, 0, &map_do, 0, p.lse + i, p.delta + i,
                     p.coef ? *p.coef : 1.0f, p.dv + b * p.dv_sb + h * p.dv_sh + (int64_t)krow * p.dv_ss,
                     p.dk + b * p.dk_sb + h * p.dk_sh + (int64_t)krow * p.dk_ss, kv_ph, q_ph, mma_ph);
  if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------
// similarity gradient (ds_aas_dir_bwd)
// ---------------------------------------------------------------------------
constexpr int kRedBlocks = 256, kRedThreads = 256;

// per-block (dot(X,Y), |X|^2, |Y|^2) over n contiguous elements, fixed split (deterministic)
template <bool kBf16>
__device__ __forceinline__ void sim_partials(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2,
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

template <bool kBf16>
__global__ void sim_partials_kernel(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2,
                                    float* __restrict__ part) {
  sim_partials<kBf16>(x, y, n2, part);
}

// coef = {gradient factor of X, of Y, k_X, k_Y}: dX = coef[0] (Y - k_X X), dY = coef[1] (X - k_Y Y) for the cosine
// (torch's per-norm max(|.|, 1e-8) clamp: a clamped norm contributes no k term); dX = -dY = coef[0] (X - Y) for MSE
__device__ __forceinline__ void sim_coef(const float* __restrict__ part, int mode, double E, const float* __restrict__ d_dir,
                                         float* __restrict__ coef) {
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

__global__ void sim_coef_kernel(const float* __restrict__ part, int mode, double E, const float* __restrict__ d_dir,
                                float* __restrict__ coef) {
  if (threadIdx.x != 0) return;
  sim_coef(part, mode, E, d_dir, coef);
}

// the O(1) factors of dX and dY, rounded to the input dtype (the dO operands of the two attention backwards)
template <bool kBf16>
__device__ __forceinline__ void sim_factor(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2, int mode,
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

template <bool kBf16>
__global__ void sim_factor_kernel(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y, int64_t n2, int mode,
                                  const float* __restrict__ coef, uint32_t* __restrict__ fx, uint32_t* __restrict__ fy) {
  sim_factor<kBf16>(x, y, n2, mode, coef, fx, fy);
}

// ---------------------------------------------------------------------------
// grouped similarity gradient (ds_aas_groups_bwd): the backward of a whole ds_aas_groups work list
// ---------------------------------------------------------------------------
// Entry t of group g contributes two TERMS: tau = 2t (cross: Attn(Q_i, K_j, V_j), dO = fx_t) and tau = 2t + 1 (self:
// Attn(Q_i, K_i, V_i), dO = fy_t).  Every gradient row receives its terms in ascending tau -- the order of one
// ds_aas_dir_bwd call per entry -- with the same arithmetic, so the result is bitwise that of the per-entry loop.

// entry -> group (binary search over group_off), and bad[0] = 1 unless group_off is 0 = off[0] <= ... <= off[G] = E
__global__ void entry_group_kernel(const int32_t* __restrict__ group_off, int64_t n_groups, int64_t n_entries,
                                   int32_t* __restrict__ entry_group, int32_t* __restrict__ bad) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n_groups && (group_off[i] > group_off[i + 1] || (i == 0 && group_off[0] != 0) ||
                       (i == n_groups - 1 && group_off[n_groups] != n_entries)))
    atomicExch(bad, 1);
  if (i < n_entries) {
    int64_t lo = 0, hi = n_groups - 1;   // last g with group_off[g] <= i
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (group_off[mid] <= i) lo = mid;
      else hi = mid - 1;
    }
    entry_group[i] = (int32_t)lo;
  }
}

// One contribution-list family: every term goes to one list, keyed by the gradient image it adds into; lists are ordered
// by key and hold their terms in ascending tau.  Family 0: dQ, key = the query image.  Family 1: dK / dV, key = the kv
// image of a cross term and the query image of a self term, offset by n_kbuf when dk_self is not dk (separate buffers).
struct ListFamily {
  int32_t* cnt;        // [n_keys] scratch
  int32_t* n_lists;    // [1]
  int32_t* list_key;   // [<= n_terms]
  int32_t* list_off;   // [<= n_terms + 1]
  int32_t* terms;      // [n_terms]
  int64_t n_keys;
};

struct ListBuild {
  const int32_t* group_q;
  const int32_t* kv_idx;
  const int32_t* entry_group;
  const int32_t* bad;
  int64_t n_terms;
  int n_kbuf;   // dK / dV self-term key offset (0: dk_self is dk)
  ListFamily fam[2];
};

// ds_aas_matrix_bwd: the row-major matrix list (group r = row r, n_cols entries), with ONE self term per row -- the folded
// one, at tau = 2t + 1 of the row's last entry t, so that it follows the row's cross terms.  rows: the row terms are
// wanted (dQ of every term, dK / dV of the folded self terms); cols: the column terms (dK / dV of the cross terms).
// Without rows no self term is live; without cols the dK / dV family holds the self terms only.  The dQ family keeps
// the cross terms either way: without rows it drives the statistics-only dQ kernel.
struct FoldListBuild : ListBuild {
  int n_cols;
  bool rows, cols;
};

template <bool kFold>
using ListBuildT = std::conditional_t<kFold, FoldListBuild, ListBuild>;

template <bool kFold>
__device__ __forceinline__ bool term_live(const ListBuildT<kFold>& b, int family, int64_t tau) {
  if constexpr (kFold) {
    if (tau & 1) return b.rows && ((tau >> 1) + 1) % b.n_cols == 0;
    return family == 0 || b.cols;
  } else {
    return true;
  }
}

__device__ __forceinline__ int term_key(const ListBuild& b, int family, int64_t tau) {
  const int64_t t = tau >> 1;
  const bool self = tau & 1;
  const int qi = b.group_q[b.entry_group[t]];
  if (family == 0) return qi;
  return self ? b.n_kbuf + qi : b.kv_idx[t];
}

// exclusive block scan of two counters over kListThreads threads; returns the block totals
constexpr int kListThreads = 1024;
__device__ __forceinline__ int2 block_scan2(int a, int c, int& ea, int& ec, int2* s_warp) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int ia = a, ic = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int ua = __shfl_up_sync(0xffffffffu, ia, o), uc = __shfl_up_sync(0xffffffffu, ic, o);
    if (lane >= o) {
      ia += ua;
      ic += uc;
    }
  }
  if (lane == 31) s_warp[w] = make_int2(ia, ic);
  __syncthreads();
  if (w == 0) {
    int2 v = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int ua = __shfl_up_sync(0xffffffffu, v.x, o), uc = __shfl_up_sync(0xffffffffu, v.y, o);
      if (lane >= o) {
        v.x += ua;
        v.y += uc;
      }
    }
    s_warp[lane] = v;   // inclusive warp prefixes
  }
  __syncthreads();
  const int2 before = w > 0 ? s_warp[w - 1] : make_int2(0, 0);
  ea = before.x + ia - a;
  ec = before.y + ic - c;
  const int2 tot = s_warp[31];
  __syncthreads();
  return tot;
}

// block f builds family f: a stable counting sort of the live terms by key (deterministic: integer counts only)
template <bool kFold>
__global__ void __launch_bounds__(kListThreads) build_lists_kernel(const ListBuildT<kFold> b) {
  const int f = blockIdx.x;
  const ListFamily& L = b.fam[f];
  __shared__ int2 s_warp[32];
  __shared__ int s_key[kListThreads];
  if (*b.bad) {   // an index is out of range: no lists, no gradient work (the gradients become NaN)
    if (threadIdx.x == 0) *L.n_lists = 0;
    return;
  }
  for (int64_t k = threadIdx.x; k < L.n_keys; k += kListThreads) L.cnt[k] = 0;
  __syncthreads();
  for (int64_t tau = threadIdx.x; tau < b.n_terms; tau += kListThreads)
    if (term_live<kFold>(b, f, tau)) atomicAdd(&L.cnt[term_key(b, f, tau)], 1);
  __syncthreads();
  int n_lists = 0, n_seen = 0;   // running totals over the key chunks
  for (int64_t k0 = 0; k0 < L.n_keys; k0 += kListThreads) {
    const int64_t k = k0 + threadIdx.x;
    const int c = k < L.n_keys ? L.cnt[k] : 0;
    int el, ec;
    const int2 tot = block_scan2(c > 0 ? 1 : 0, c, el, ec, s_warp);
    if (c > 0) {
      L.list_key[n_lists + el] = (int32_t)k;
      L.list_off[n_lists + el] = n_seen + ec;
    }
    if (k < L.n_keys) L.cnt[k] = n_seen + ec;   // first slot of key k's terms
    n_lists += tot.x;
    n_seen += tot.y;
  }
  if (threadIdx.x == 0) {
    *L.n_lists = n_lists;
    L.list_off[n_lists] = n_seen;
  }
  __syncthreads();
  for (int64_t t0 = 0; t0 < b.n_terms; t0 += kListThreads) {
    const int64_t tau = t0 + threadIdx.x;
    const bool live = tau < b.n_terms && term_live<kFold>(b, f, tau);
    const int key = live ? term_key(b, f, tau) : -1;
    s_key[threadIdx.x] = key;
    __syncthreads();
    if (live) {
      int r = 0;   // earlier terms of this chunk with the same key
      for (int j = 0; j < (int)threadIdx.x; ++j) r += s_key[j] == key;
      L.terms[L.cnt[key] + r] = (int32_t)tau;
    }
    __syncthreads();
    if (live) atomicAdd(&L.cnt[key], 1);
    __syncthreads();
  }
}

// per entry: (dot, |X|^2, |Y|^2) partials, coefficients and factors exactly as for one ds_aas_dir_bwd call
template <bool kBf16>
__global__ void sim_partials_list_kernel(const uint32_t* __restrict__ o, int64_t n2, int n_groups, int64_t n_entries,
                                         const int32_t* __restrict__ entry_group, float* __restrict__ part) {
  for (int64_t t = blockIdx.y; t < n_entries; t += gridDim.y) {
    sim_partials<kBf16>(o + (n_groups + t) * n2, o + entry_group[t] * n2, n2, part + t * (kRedBlocks * 3));
    __syncthreads();
  }
}

__global__ void sim_coef_list_kernel(const float* __restrict__ part, int64_t n_entries, int mode, double E,
                                     const float* __restrict__ d_dir, float* __restrict__ coef) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n_entries) sim_coef(part + t * (kRedBlocks * 3), mode, E, d_dir + t, coef + 4 * t);
}

template <bool kBf16>
__global__ void sim_factor_list_kernel(const uint32_t* __restrict__ o, int64_t n2, int n_groups, int64_t n_entries,
                                       const int32_t* __restrict__ entry_group, int mode, const float* __restrict__ coef,
                                       uint32_t* __restrict__ f) {
  for (int64_t t = blockIdx.y; t < n_entries; t += gridDim.y)
    sim_factor<kBf16>(o + (n_groups + t) * n2, o + entry_group[t] * n2, n2, mode, coef + 4 * t, f + 2 * t * n2,
                      f + (2 * t + 1) * n2);
}

// ---------------------------------------------------------------------------
// matrix similarity gradient (ds_aas_matrix_bwd): the grouped backward of the row-major matrix list, with each row's
// self terms folded into one.  The attention backward is linear in dO and so is delta = rowsum(dO o O): the Nc self terms
// of row r (O = Y_r, dO = coef_self_rc fy_rc) are ONE term with dO = F_r = sum_c coef_self_rc fy_rc.
// ---------------------------------------------------------------------------
// the row-major list (group r = row r: entries t = r n_cols + c, kv image c), entry -> row, and d_dir[t] = d_Dm[r, c]
__global__ void matrix_bwd_setup_kernel(int64_t n_rows, int64_t n_cols, const float* __restrict__ d_Dm, int64_t ldd,
                                        int32_t* __restrict__ group_q, int32_t* __restrict__ group_off,
                                        int32_t* __restrict__ kv_idx, int32_t* __restrict__ entry_group,
                                        float* __restrict__ d_dir) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n_rows * n_cols) {
    const int64_t r = i / n_cols, c = i - r * n_cols;
    kv_idx[i] = (int32_t)c;
    entry_group[i] = (int32_t)r;
    d_dir[i] = d_Dm[r * ldd + c];
  }
  if (i <= n_rows) group_off[i] = (int32_t)(i * n_cols);
  if (i < n_rows) group_q[i] = (int32_t)i;
}

// per row r and element pair: fx_t of every entry t = (r, c) as sim_factor rounds it, and the fp32 fold
// F_r = sum over ascending c of coef[4t + 1] fy_t, fy_t unrounded (F32 [r][n2]); row_max[r] (zeroed before): max |F_r|
// as float bits (non-negative floats order as integers, so the integer atomic is order-independent).
// kSum = false: fx_t only, for a call without the row terms (no fold, F32 and row_max are not touched).
template <bool kBf16, bool kSum = true>
__global__ void matrix_fold_kernel(const uint32_t* __restrict__ o, int64_t n2, int n_rows, int n_cols, int mode,
                                   const float* __restrict__ coef, uint32_t* __restrict__ fx, float2* __restrict__ F32,
                                   int32_t* __restrict__ row_max) {
  __shared__ float s_max[kRedThreads / 32];
  for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
    const uint32_t* y = o + (int64_t)r * n2;
    float mx = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
      const float2 c = unpack2<kBf16>(y[i]);
      float fx0 = 0.f, fx1 = 0.f;
      for (int col = 0; col < n_cols; ++col) {
        const int64_t t = (int64_t)r * n_cols + col;
        const float* cf = coef + 4 * t;
        const float2 a = unpack2<kBf16>(o[(n_rows + t) * n2 + i]);
        float fy0, fy1;
        if (mode == DS_SIM_MSE) {
          fx[t * n2 + i] = pack2<kBf16>(a.x - c.x, a.y - c.y);
          fy0 = c.x - a.x;
          fy1 = c.y - a.y;
        } else {
          const float kx = cf[2], ky = cf[3];
          fx[t * n2 + i] = pack2<kBf16>(c.x - kx * a.x, c.y - kx * a.y);
          fy0 = a.x - ky * c.x;
          fy1 = a.y - ky * c.y;
        }
        if constexpr (kSum) {
          fx0 = fmaf(cf[1], fy0, fx0);
          fx1 = fmaf(cf[1], fy1, fx1);
        }
      }
      if constexpr (kSum) {
        F32[(int64_t)r * n2 + i] = make_float2(fx0, fx1);
        mx = fmaxf(mx, fmaxf(fabsf(fx0), fabsf(fx1)));
      }
    }
    if constexpr (kSum) {
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o2));
      if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = mx;
      __syncthreads();
      if (threadIdx.x == 0) {
        for (int w = 1; w < kRedThreads / 32; ++w) mx = fmaxf(mx, s_max[w]);
        atomicMax(row_max + r, __float_as_int(mx));
      }
      __syncthreads();
    }
  }
}

// F_r rounded ONCE to the input dtype after a power-of-two scale 2^-e that puts max |F_r| in [0.5, 1): at SD-1.5 up0 the
// elements of F_r fall below fp16's normal range.  fold_scale[r] = 2^e, the coefficient of the folded self term.
template <bool kBf16>
__global__ void matrix_fold_round_kernel(const float2* __restrict__ F32, int64_t n2, int n_rows,
                                         const int32_t* __restrict__ row_max, uint32_t* __restrict__ F16,
                                         float* __restrict__ fold_scale) {
  for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
    const float m = __int_as_float(row_max[r]);
    int e = 0;
    if (m > 0.f && m <= 3.402823466e38f) {
      frexpf(m, &e);
      e = min(max(e, -126), 127);
    }
    const float inv = ldexpf(1.f, -e);
    if (blockIdx.x == 0 && threadIdx.x == 0) fold_scale[r] = ldexpf(1.f, e);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
      const float2 v = F32[(int64_t)r * n2 + i];
      F16[(int64_t)r * n2 + i] = pack2<kBf16>(v.x * inv, v.y * inv);
    }
  }
}

struct GradT {   // an fp32 (N, B, H, S, D) gradient
  float* ptr;
  int64_t sn, sb, sh, ss;
};

struct ListParams : Shape {
  int n_groups;
  const int32_t* group_q;
  const int32_t* kv_idx;
  const int32_t* entry_group;
  const int32_t* n_lists;    // device count of the family's lists (the grid covers an upper bound)
  const int32_t* list_key;
  const int32_t* list_off;
  const int32_t* terms;
  int n_kbuf;                // dK / dV keys >= n_kbuf address (dk_self, dv_self) at image key - n_kbuf
  const void* o;             // Y_g at slot g, X_t at slot n_groups + t: contiguous (B, H, Sq, D) images
  const void* f;             // fx_t at slot 2t, fy_t at slot 2t + 1 (= tau)
  int64_t img;               // B H Sq D: slot stride of o and f
  float* lse;                // [tau][B H][n_qt 128]
  float* delta;
  const float* coef;         // [t][4]: factor of the cross term at 4t, of the self term at 4t + 1
  GradT dq, dk, dv, dks, dvs;
};

// ds_aas_matrix_bwd (kFold): the self term of row r is the folded one.  Its dO factor and its LSE / delta rows sit at
// slot n_entries + r, a cross term's at slot t (instead of tau); its coefficient is fold_scale[r].
struct FoldListParams : ListParams {
  int64_t n_entries;
  const float* fold_scale;
};

template <bool kFold>
using ListParamsT = std::conditional_t<kFold, FoldListParams, ListParams>;

// term tau = 2t (+ 1 for the self term) of a list: the slot of its dO factor and of its LSE / delta rows, and its
// coefficient
template <bool kFold>
__device__ __forceinline__ float term_coef(const ListParamsT<kFold>& p, int tau, int& slot) {
  const int t = tau >> 1;
  const bool self = tau & 1;
  if constexpr (kFold) {
    slot = self ? (int)p.n_entries + p.entry_group[t] : t;
    return self ? p.fold_scale[p.entry_group[t]] : p.coef[4 * t];
  }
  slot = tau;
  return p.coef[4 * t + (self ? 1 : 0)];
}

// attn_bwd_dq_kernel over a list: one CTA per (query image, b, h, 128-row q tile), one dQ term per list entry, each
// drained (x its coefficient) into the fp32 rows before the next.  kStats: only every term's LSE and delta (dq_term's
// statistics-only form), for a dK/dV list that runs without the dQ gradient.
template <int D, bool kBf16, bool kFold, bool kStats = false>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dq_list_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                        const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_ks,
                        const __grid_constant__ CUtensorMap map_vs, const __grid_constant__ CUtensorMap map_do,
                        const ListParamsT<kFold> p) {
  const int per_list = p.B * p.H * p.n_qt;
  const int li = blockIdx.x / per_list;
  if (li >= *p.n_lists) return;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t tmem = kernel_prologue(reinterpret_cast<uint64_t*>(smem + Cfg<D>::DQ_BARS), &map_q, &map_k, &map_v,
                                        &map_ks, &map_vs, &map_do);
  const int rest = blockIdx.x - li * per_list;
  const int bh = rest / p.n_qt, qt = rest - bh * p.n_qt;
  const int b = bh / p.H, h = bh - b * p.H;
  const int grow = qt * kTile + threadIdx.x;
  const int qi = p.list_key[li];
  const int i0 = p.list_off[li], i1 = p.list_off[li + 1];
  const int64_t row_off = ((int64_t)b * p.H + h) * p.Sq * D + (int64_t)grow * D;   // in a contiguous (B, H, Sq, D) image
  float* dq_row = p.dq.ptr + qi * p.dq.sn + b * p.dq.sb + h * p.dq.sh + (int64_t)grow * p.dq.ss;
  uint32_t q_ph = 0, kv_ph = 0, mma_ph = 0;

  for (int i = i0; i < i1; ++i) {
    const int tau = p.terms[i], t = tau >> 1;
    const bool self = tau & 1;
    const int64_t o_slot = self ? p.entry_group[t] : p.n_groups + t;
    int slot;
    const float coef = term_coef<kFold>(p, tau, slot);
    const size_t k = ((size_t)slot * (p.B * p.H) + bh) * (p.n_qt * kTile) + grow;
    dq_term<D, kBf16, kStats>(smem, tmem, p, b, h, qt, &map_q, qi, &map_do, slot, self ? &map_ks : &map_k,
                      self ? &map_vs : &map_v, self ? qi : p.kv_idx[t], self ? p.Skv_self : p.Skv,
                      static_cast<const uint16_t*>(p.o) + o_slot * p.img + row_off,
                      static_cast<const uint16_t*>(p.f) + slot * p.img + row_off, p.lse + k, p.delta + k, coef, dq_row,
                      q_ph, kv_ph, mma_ph);
  }
  if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// attn_bwd_dkv_kernel over a list: one CTA per (kv image, b, h, 128-row kv tile), one dK/dV term per list entry.  The
// grid gives every list max(n_kt, n_kt_self) tiles per (b, h); the CTAs past the tiles of the list's own kv length (that
// of k_self for a self-term list, of k otherwise) exit at once.  With separate self buffers (n_kbuf > 0) a list holds
// terms of one kind only; with one shared buffer the two lengths are equal.
template <int D, bool kBf16, bool kFold>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dkv_list_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                         const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_ks,
                         const __grid_constant__ CUtensorMap map_vs, const __grid_constant__ CUtensorMap map_do,
                         const ListParamsT<kFold> p) {
  const int n_kt = max(p.n_kt, p.n_kt_self);
  const int per_list = p.B * p.H * n_kt;
  const int li = blockIdx.x / per_list;
  if (li >= *p.n_lists) return;
  const int rest = blockIdx.x - li * per_list;
  const int bh = rest / n_kt, kt = rest - bh * n_kt;
  int img = p.list_key[li];
  const bool self_list = img >= p.n_kbuf && p.n_kbuf > 0;
  if (kt >= (self_list ? p.n_kt_self : p.n_kt)) return;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t tmem = kernel_prologue(reinterpret_cast<uint64_t*>(smem + Cfg<D>::DKV_BARS), &map_q, &map_k, &map_v,
                                        &map_ks, &map_vs, &map_do);
  const int b = bh / p.H, h = bh - b * p.H;
  const int krow = kt * kTile + threadIdx.x;
  GradT gk = p.dk, gv = p.dv;
  if (self_list) {
    img -= p.n_kbuf;
    gk = p.dks;
    gv = p.dvs;
  }
  const int i0 = p.list_off[li], i1 = p.list_off[li + 1];
  float* dv_row = gv.ptr + img * gv.sn + b * gv.sb + h * gv.sh + (int64_t)krow * gv.ss;
  float* dk_row = gk.ptr + img * gk.sn + b * gk.sb + h * gk.sh + (int64_t)krow * gk.ss;
  uint32_t kv_ph = 0, q_ph = 0, mma_ph = 0;

  for (int i = i0; i < i1; ++i) {
    const int tau = p.terms[i], t = tau >> 1;
    const bool self = tau & 1;
    int slot;
    const float coef = term_coef<kFold>(p, tau, slot);
    const size_t k = ((size_t)slot * (p.B * p.H) + bh) * (p.n_qt * kTile);
    dkv_term<D, kBf16>(smem, tmem, p, b, h, kt, self ? &map_ks : &map_k, self ? &map_vs : &map_v, img,
                       self ? p.Skv_self : p.Skv, &map_q,
                       p.group_q[p.entry_group[t]], &map_do, slot, p.lse + k, p.delta + k, coef, dv_row, dk_row, kv_ph,
                       q_ph, mma_ph);
  }
  if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// every element of the five gradients := NaN when bad[0] is set (an image index of the list was out of range)
struct NanFill {
  float* ptr[5];
  int64_t size[5][5];
  int64_t stride[5][5];
};

__global__ void nan_fill_kernel(const NanFill f, const int32_t* __restrict__ bad) {
  if (!*bad) return;
  for (int k = 0; k < 5; ++k) {
    const int64_t* sz = f.size[k];
    const int64_t n = sz[0] * sz[1] * sz[2] * sz[3] * sz[4];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      int64_t r = i, off = 0;
      for (int d = 4; d >= 0; --d) {
        off += (r % sz[d]) * f.stride[k][d];
        r /= sz[d];
      }
      f.ptr[k][off] = __int_as_float(0x7fc00000);
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

// the Shape of the backward of q (., B, H, Sq, D) against k (., B, H, Skv, D) and, for the self terms of a list, k_self
// (., B, H, Skv_self, D)
static void set_shape(Shape* s, const ds_tensor5& q, const ds_tensor5& k, const ds_tensor5& ks, float scale) {
  s->B = (int)q.size[1];
  s->H = (int)q.size[2];
  s->Sq = (int)q.size[3];
  s->Skv = (int)k.size[3];
  s->Skv_self = (int)ks.size[3];
  s->n_qt = (s->Sq + kTile - 1) / kTile;
  s->n_kt = (s->Skv + kTile - 1) / kTile;
  s->n_kt_self = (s->Skv_self + kTile - 1) / kTile;
  s->scale = scale > 0.f ? scale : 1.0f / sqrtf((float)q.size[4]);
  s->scale_log2 = s->scale * 1.4426950408889634f;
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
  const ds_tensor5 q = lift(a.q), k = lift(a.k), dout = lift(a.dout);
  if ((rc = make_map(&mq, q, C::SUBW, kTile)) != DS_OK || (rc = make_map(&mk, k, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mv, lift(a.v), C::SUBW, kTile)) != DS_OK || (rc = make_map(&mdo, dout, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mqb, q, C::SUBW, C::BQ)) != DS_OK || (rc = make_map(&mdob, dout, C::SUBW, C::BQ)) != DS_OK)
    return rc;
  Params p;
  set_shape(&p, q, k, k, a.scale);
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

// ---- grouped similarity gradient: host side

static int check_grad5(const ds_tensor5& g, const ds_tensor5& like, const char* who, const char* name) {
  if (!g.ptr) return fail(DS_ERR_INVALID, "%s: %s: null pointer", who, name);
  if (g.dtype != DS_F32) return fail(DS_ERR_INVALID, "%s: %s: gradients are float32", who, name);
  for (int i = 0; i < 5; ++i)
    if (g.size[i] != like.size[i]) return fail(DS_ERR_INVALID, "%s: %s: shape must match its input", who, name);
  if (g.stride[4] != 1) return fail(DS_ERR_INVALID, "%s: %s: innermost stride must be 1", who, name);
  if ((uintptr_t)g.ptr & 3) return fail(DS_ERR_INVALID, "%s: %s: base pointer must be 4-byte aligned", who, name);
  for (int i = 0; i < 4; ++i)
    if (g.size[i] > 1 && g.stride[i] <= 0) return fail(DS_ERR_INVALID, "%s: %s: stride[%d] must be positive", who, name, i);
  return DS_OK;
}

static bool same_tensor(const ds_tensor5& a, const ds_tensor5& b) {
  if (a.ptr != b.ptr || a.dtype != b.dtype) return false;
  for (int i = 0; i < 5; ++i)
    if (a.size[i] != b.size[i] || (a.size[i] > 1 && a.stride[i] != b.stride[i])) return false;
  return true;
}

// the address ranges of two fp32 tensors with positive strides intersect
static bool extents_meet(const ds_tensor5& a, const ds_tensor5& b) {
  auto end = [](const ds_tensor5& t) {
    int64_t e = 1;
    for (int i = 0; i < 5; ++i) e += (t.size[i] - 1) * t.stride[i];
    return static_cast<const char*>(t.ptr) + 4 * e;
  };
  const char* a0 = static_cast<const char*>(a.ptr);
  const char* b0 = static_cast<const char*>(b.ptr);
  return a0 < end(b) && b0 < end(a);
}

// workspace layout of ds_aas_groups_bwd (the size query runs it on a dummy base); ds_aas_matrix_bwd's extends it
struct GroupsBwdWs {
  void* o;                 // (n_groups + n_entries) attention outputs, 16-bit
  void* f;                 // 2 n_entries dO factors, 16-bit
  float* part;             // [n_entries][kRedBlocks][3]
  float* coef;             // [n_entries][4]
  float* lse;              // [2 n_entries][B H][n_qt 128]
  float* delta;
  int32_t* entry_group;    // [n_entries]
  int32_t* bad;
  ListFamily fam[2];
};

// a contribution-list family of n_keys keys, at most max_lists lists and n_terms terms
static bool take_family(Workspace& w, ListFamily* F, int64_t n_keys, int64_t max_lists, int64_t n_terms) {
  F->n_keys = n_keys;
  F->cnt = static_cast<int32_t*>(w.take((size_t)n_keys * 4));
  F->n_lists = static_cast<int32_t*>(w.take(4));
  F->list_key = static_cast<int32_t*>(w.take((size_t)max_lists * 4));
  F->list_off = static_cast<int32_t*>(w.take((size_t)(max_lists + 1) * 4));
  F->terms = static_cast<int32_t*>(w.take((size_t)n_terms * 4));
  return F->cnt && F->n_lists && F->list_key && F->list_off && F->terms;
}

static bool groups_bwd_layout(Workspace& w, const ds_tensor5& q, const ds_tensor5& k, int64_t G, int64_t E,
                              GroupsBwdWs* L) {
  const int64_t img = q.size[1] * q.size[2] * q.size[3] * q.size[4];
  const int64_t n_qt = (q.size[3] + kTile - 1) / kTile;
  const size_t stats = (size_t)(2 * E) * q.size[1] * q.size[2] * n_qt * kTile * sizeof(float);
  const int64_t nt = 2 * E;
  L->o = w.take((size_t)(G + E) * img * 2);
  L->f = w.take((size_t)nt * img * 2);
  L->part = static_cast<float*>(w.take((size_t)E * kRedBlocks * 3 * sizeof(float)));
  L->coef = static_cast<float*>(w.take((size_t)E * 4 * sizeof(float)));
  L->lse = static_cast<float*>(w.take(stats));
  L->delta = static_cast<float*>(w.take(stats));
  L->entry_group = static_cast<int32_t*>(w.take((size_t)E * 4));
  L->bad = static_cast<int32_t*>(w.take(4));
  const bool ok = L->o && L->f && L->part && L->coef && L->lse && L->delta && L->entry_group && L->bad;
  return ok && take_family(w, &L->fam[0], q.size[0], nt, nt) &&
         take_family(w, &L->fam[1], k.size[0] + q.size[0], nt, nt);
}

static GradT grad_t(const ds_tensor5& g) {
  return GradT{static_cast<float*>(g.ptr), g.stride[0], g.stride[1], g.stride[2], g.stride[3]};
}

// the dQ and dK/dV list kernels of a list backward; kStats: the dQ kernel in its statistics-only form
template <int D, bool kBf16, bool kFold, bool kStats = false>
static int launch_groups_bwd_t(const ds_tensor5& q, const ds_tensor5& ks, const ds_tensor5& vs, const ds_tensor5& k,
                               const ds_tensor5& v, const ds_tensor5& F, ListParamsT<kFold> p, int64_t grid_q,
                               int64_t grid_kv, const ListFamily* fam, cudaStream_t st) {
  using C = Cfg<D>;
  CUtensorMap mq, mk, mv, mks, mvs, mdo, mqb, mdob;
  int rc;
  if ((rc = make_map(&mq, q, C::SUBW, kTile)) != DS_OK || (rc = make_map(&mk, k, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mv, v, C::SUBW, kTile)) != DS_OK || (rc = make_map(&mks, ks, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mvs, vs, C::SUBW, kTile)) != DS_OK || (rc = make_map(&mdo, F, C::SUBW, kTile)) != DS_OK ||
      (rc = make_map(&mqb, q, C::SUBW, C::BQ)) != DS_OK || (rc = make_map(&mdob, F, C::SUBW, C::BQ)) != DS_OK)
    return rc;
  DS_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dq_list_kernel<D, kBf16, kFold, kStats>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   C::DQ_SMEM));
  DS_CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dkv_list_kernel<D, kBf16, kFold>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   C::DKV_SMEM));
  p.n_lists = fam[0].n_lists;
  p.list_key = fam[0].list_key;
  p.list_off = fam[0].list_off;
  p.terms = fam[0].terms;
  attn_bwd_dq_list_kernel<D, kBf16, kFold, kStats><<<(unsigned)grid_q, kThreads, C::DQ_SMEM, st>>>(mq, mk, mv, mks, mvs, mdo,
                                                                                                 p);
  DS_CUDA_TRY(cudaGetLastError());
  p.n_lists = fam[1].n_lists;
  p.list_key = fam[1].list_key;
  p.list_off = fam[1].list_off;
  p.terms = fam[1].terms;
  attn_bwd_dkv_list_kernel<D, kBf16, kFold><<<(unsigned)grid_kv, kThreads, C::DKV_SMEM, st>>>(mqb, mk, mv, mks, mvs, mdob, p);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

// the factors of a list backward as a contiguous (n_slots, B, H, Sq, D) stack of q's dtype at ptr
static ds_tensor5 factor_stack(const ds_tensor5& q, void* ptr, int64_t n_slots) {
  ds_tensor5 F = q;
  F.ptr = ptr;
  F.size[0] = n_slots;
  F.stride[4] = 1;
  F.stride[3] = q.size[4];
  F.stride[2] = q.size[3] * q.size[4];
  F.stride[1] = q.size[2] * F.stride[2];
  F.stride[0] = q.size[1] * F.stride[1];
  return F;
}

// ListParams of a checked list backward: shapes, grids (false: too many tiles) and everything but the pointers
static bool list_params(const ds_tensor5& q, const ds_tensor5& k, const ds_tensor5& ks, float scale, int64_t G,
                        int64_t E, bool aliased, ListParams* p, int64_t* grid_q, int64_t* grid_kv) {
  set_shape(p, q, k, ks, scale);
  p->n_groups = (int)G;
  p->n_kbuf = aliased ? 0 : (int)k.size[0];
  p->img = q.size[1] * q.size[2] * q.size[3] * q.size[4];
  const int64_t bh = (int64_t)p->B * p->H;
  const int64_t nl_q = std::min<int64_t>(q.size[0], G);
  const int64_t nl_kv = aliased ? std::min<int64_t>(k.size[0], G + E) : nl_q + std::min<int64_t>(k.size[0], E);
  *grid_q = nl_q * bh * p->n_qt;
  *grid_kv = nl_kv * bh * std::max(p->n_kt, p->n_kt_self);   // attn_bwd_dkv_list_kernel's grid
  return *grid_q < INT32_MAX && *grid_kv < INT32_MAX;
}

// the pointers of a ListParams: the work list, the workspace and the five gradients
static void set_pointers(ListParams* p, const int32_t* group_q, const int32_t* kv_idx, const GroupsBwdWs& L,
                         const ds_tensor5& dq, const ds_tensor5& dks, const ds_tensor5& dvs, const ds_tensor5& dk,
                         const ds_tensor5& dv) {
  p->group_q = group_q;
  p->kv_idx = kv_idx;
  p->entry_group = L.entry_group;
  p->o = L.o;
  p->f = L.f;
  p->lse = L.lse;
  p->delta = L.delta;
  p->coef = L.coef;
  p->dq = grad_t(dq);
  p->dk = grad_t(dk);
  p->dv = grad_t(dv);
  p->dks = grad_t(dks);
  p->dvs = grad_t(dvs);
}

// the input of build_lists_kernel for the E entries of a list backward (the matrix adds n_cols); aliased: one dk / dv
// buffer, whose self terms share the kv images' keys
static void set_list_build(ListBuild* lb, const int32_t* group_q, const int32_t* kv_idx, int64_t E,
                           const ds_tensor5& q, const ds_tensor5& k, bool aliased, const ListParams& p,
                           const GroupsBwdWs& L) {
  lb->group_q = group_q;
  lb->kv_idx = kv_idx;
  lb->entry_group = L.entry_group;
  lb->bad = L.bad;
  lb->n_terms = 2 * E;
  lb->n_kbuf = p.n_kbuf;
  lb->fam[0] = L.fam[0];
  lb->fam[1] = L.fam[1];
  lb->fam[1].n_keys = aliased ? k.size[0] : k.size[0] + q.size[0];
}

// per entry of a list backward: the (dot, |X|^2, |Y|^2) partials of X_t and Y_{group(t)} and the coefficients from
// d_dir[t], exactly as one ds_aas_dir_bwd call computes them
static int launch_list_coefs(const ds_tensor5& q, const ListParams& p, int64_t E, int mode, const float* d_dir,
                             const GroupsBwdWs& L, cudaStream_t st) {
  const uint32_t* ou = static_cast<const uint32_t*>(L.o);
  const int64_t n2 = p.img / 2;
  const dim3 grid(kRedBlocks, (unsigned)std::min<int64_t>(E, 65535));
  const bool bf = q.dtype == DS_BF16;
  if (bf) sim_partials_list_kernel<true><<<grid, kRedThreads, 0, st>>>(ou, n2, p.n_groups, E, L.entry_group, L.part);
  else sim_partials_list_kernel<false><<<grid, kRedThreads, 0, st>>>(ou, n2, p.n_groups, E, L.entry_group, L.part);
  DS_CUDA_TRY(cudaGetLastError());
  sim_coef_list_kernel<<<(unsigned)((E + 127) / 128), 128, 0, st>>>(L.part, E, mode, (double)p.img, d_dir, L.coef);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
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

namespace ds {
namespace bwd {

__global__ void pairs_ddir_kernel(const float* __restrict__ d_scores, int64_t n, float* __restrict__ d_dir) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) d_dir[2 * i] = d_dir[2 * i + 1] = d_scores[i] * 0.5f;   // score = (dir[2p] + dir[2p + 1]) / 2
}

// entries 4t .. 4t + 3 = ref->left, ref->right, left->ref, right->ref; ab = (dir[4t] + dir[4t + 2]) / 2, ac likewise
__global__ void triplets_ddir_kernel(const float* __restrict__ d_ab, const float* __restrict__ d_ac, int64_t n,
                                     float* __restrict__ d_dir) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    d_dir[4 * i] = d_dir[4 * i + 2] = d_ab[i] * 0.5f;
    d_dir[4 * i + 1] = d_dir[4 * i + 3] = d_ac[i] * 0.5f;
  }
}

// every argument of a grouped backward except the work list itself; *aliased: dk_self is dk and dv_self is dv.
// rows / cols: the gradient families (dq, dk_self, dv_self) / (dk, dv) are given; a missing family is not checked.
static int groups_bwd_check(const ds_tensor5& q, const ds_tensor5& ks, const ds_tensor5& vs, const ds_tensor5& k,
                            const ds_tensor5& v, int mode, const float* d, const ds_tensor5& dq, const ds_tensor5& dks,
                            const ds_tensor5& dvs, const ds_tensor5& dk, const ds_tensor5& dv, const char* who,
                            bool* aliased, bool rows = true, bool cols = true) {
  int rc;
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return fail(DS_ERR_INVALID, "%s: bad mode %d", who, mode);
  if (!d) return fail(DS_ERR_INVALID, "%s: score gradient: null pointer", who);
  if ((rc = check_group_operands(q, ks, vs, k, v, who)) != DS_OK) return rc;
  if (rows && ((rc = check_grad5(dq, q, who, "dq")) != DS_OK || (rc = check_grad5(dks, ks, who, "dk_self")) != DS_OK ||
               (rc = check_grad5(dvs, vs, who, "dv_self")) != DS_OK))
    return rc;
  if (cols && ((rc = check_grad5(dk, k, who, "dk")) != DS_OK || (rc = check_grad5(dv, v, who, "dv")) != DS_OK)) return rc;
  *aliased = false;
  if (!rows || !cols) return DS_OK;
  const bool ak = same_tensor(dks, dk), av = same_tensor(dvs, dv);
  if (ak != av) return fail(DS_ERR_INVALID, "%s: dk_self / dk and dv_self / dv must both be the same tensor or both be separate", who);
  if (!ak && (extents_meet(dks, dk) || extents_meet(dvs, dv)))
    return fail(DS_ERR_INVALID, "%s: dk_self / dk (dv_self / dv) must be the same tensor or not overlap", who);
  *aliased = ak;
  return DS_OK;
}

// the device work of ds_aas_groups_bwd on a checked call whose work list (and d_dir) is on the device
static int groups_bwd_launch(const ds_tensor5& q, const ds_tensor5& ks, const ds_tensor5& vs, const ds_tensor5& k,
                             const ds_tensor5& v, const int32_t* group_q, const int32_t* group_off, int64_t G,
                             const int32_t* kv_idx, int64_t E, float scale, int mode, const float* d_dir,
                             const ds_tensor5& dq, const ds_tensor5& dks, const ds_tensor5& dvs, const ds_tensor5& dk,
                             const ds_tensor5& dv, bool aliased, const GroupsBwdWs& L, const char* who, cudaStream_t st) {
  int rc;
  ListParams p;
  int64_t grid_q, grid_kv;
  if (!list_params(q, k, ks, scale, G, E, aliased, &p, &grid_q, &grid_kv))
    return fail(DS_ERR_INVALID, "%s: too many tiles: split the work list", who);
  set_pointers(&p, group_q, kv_idx, L, dq, dks, dvs, dk, dv);
  const int64_t n2 = p.img / 2;
  const bool bf = q.dtype == DS_BF16;

  DS_CUDA_TRY(cudaMemsetAsync(L.bad, 0, sizeof(int32_t), st));
  if ((rc = launch_validate_groups(group_q, G, kv_idx, E, q.size[0], k.size[0], L.bad, st)) != DS_OK) return rc;
  entry_group_kernel<<<(unsigned)((std::max(G, E) + 255) / 256), 256, 0, st>>>(group_off, G, E, L.entry_group, L.bad);
  DS_CUDA_TRY(cudaGetLastError());
  ListBuild lb;
  set_list_build(&lb, group_q, kv_idx, E, q, k, aliased, p, L);
  build_lists_kernel<false><<<2, kListThreads, 0, st>>>(lb);
  DS_CUDA_TRY(cudaGetLastError());
  // X_t and Y_g, rounded to the input dtype as ds_attn_fwd rounds them
  if ((rc = attn_list_store(q, ks, vs, k, v, group_q, group_off, G, kv_idx, scale, L.o, who, st)) != DS_OK) return rc;
  if ((rc = launch_list_coefs(q, p, E, mode, d_dir, L, st)) != DS_OK) return rc;
  const uint32_t* ou = static_cast<const uint32_t*>(L.o);
  const unsigned ey = (unsigned)std::min<int64_t>(E, 65535);
  const unsigned fb = (unsigned)std::min<int64_t>((n2 + 255) / 256, 4 * (int64_t)sm_count());
  uint32_t* fu = static_cast<uint32_t*>(L.f);
  if (bf) sim_factor_list_kernel<true><<<dim3(fb, ey), 256, 0, st>>>(ou, n2, (int)G, E, L.entry_group, mode, L.coef, fu);
  else sim_factor_list_kernel<false><<<dim3(fb, ey), 256, 0, st>>>(ou, n2, (int)G, E, L.entry_group, mode, L.coef, fu);
  DS_CUDA_TRY(cudaGetLastError());

  const ds_tensor5 F = factor_stack(q, L.f, 2 * E);
  rc = with_head_dim(q.size[4], who, [&](auto d) {
    return with_dtype(q.dtype, [&](auto b) {
      return launch_groups_bwd_t<decltype(d)::value, decltype(b)::value, false>(q, ks, vs, k, v, F, p, grid_q, grid_kv,
                                                                                L.fam, st);
    });
  });
  if (rc != DS_OK) return rc;
  NanFill nf;
  const ds_tensor5* gs[5] = {&dq, &dks, &dvs, &dk, &dv};
  for (int i = 0; i < 5; ++i) {
    nf.ptr[i] = static_cast<float*>(gs[i]->ptr);
    for (int j = 0; j < 5; ++j) {
      nf.size[i][j] = gs[i]->size[j];
      nf.stride[i][j] = gs[i]->stride[j];
    }
  }
  nan_fill_kernel<<<4 * sm_count(), 256, 0, st>>>(nf, L.bad);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

static Workspace size_query() { return Workspace(reinterpret_cast<void*>(4096), SIZE_MAX / 4); }

}  // namespace bwd
}  // namespace ds

extern "C" {

size_t ds_aas_groups_bwd_workspace_bytes(ds_tensor5 q, ds_tensor5 k, int64_t n_groups, int64_t n_entries) {
  using namespace ds::bwd;
  if (n_groups <= 0 || n_entries <= 0) return 256;
  ds::Workspace w = size_query();
  GroupsBwdWs L;
  groups_bwd_layout(w, q, k, n_groups, n_entries, &L);
  return w.off + 256;
}

int ds_aas_groups_bwd(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v,
                      const int32_t* group_q, const int32_t* group_off, int64_t n_groups, const int32_t* kv_idx,
                      int64_t n_entries, float scale, int mode, const float* d_dir, ds_tensor5 dq, ds_tensor5 dk_self,
                      ds_tensor5 dv_self, ds_tensor5 dk, ds_tensor5 dv, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_aas_groups_bwd";
  if (n_groups < 0 || n_entries < 0) return fail(DS_ERR_INVALID, "%s: negative counts", who);
  if (n_groups == 0 || n_entries == 0) return DS_OK;
  if (!group_q || !group_off || !kv_idx) return fail(DS_ERR_INVALID, "%s: work list: null pointer", who);
  if (n_groups > INT32_MAX / 4 || n_entries > INT32_MAX / 4) return fail(DS_ERR_INVALID, "%s: work list too long", who);
  bool aliased;
  int rc = groups_bwd_check(q, k_self, v_self, k, v, mode, d_dir, dq, dk_self, dv_self, dk, dv, who, &aliased);
  if (rc != DS_OK) return rc;
  Workspace w(ws, ws_bytes);
  GroupsBwdWs L;
  if (!groups_bwd_layout(w, q, k, n_groups, n_entries, &L))
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_aas_groups_bwd_workspace_bytes(q, k, n_groups, n_entries));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  return groups_bwd_launch(q, k_self, v_self, k, v, group_q, group_off, n_groups, kv_idx, n_entries, scale, mode, d_dir,
                           dq, dk_self, dv_self, dk, dv, aliased, L, who, static_cast<cudaStream_t>(stream));
}

size_t ds_aas_pairs_bwd_workspace_bytes(ds_tensor5 q, int64_t n_pairs) {
  using namespace ds;
  if (n_pairs <= 0) return 256;
  const size_t lists = 2 * align_up((size_t)(2 * n_pairs) * 4, 256) + align_up((size_t)(2 * n_pairs + 1) * 4, 256) +
                       align_up((size_t)(2 * n_pairs) * 4, 256);   // group_q, kv_idx, group_off, d_dir
  return lists + ds_aas_groups_bwd_workspace_bytes(q, q, 2 * n_pairs, 2 * n_pairs) + 256;
}

int ds_aas_pairs_bwd(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* pair_idx, int64_t n_pairs, float scale,
                     int mode, const float* d_scores, ds_tensor5 dq, ds_tensor5 dk, ds_tensor5 dv, void* ws,
                     size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_aas_pairs_bwd";
  if (n_pairs < 0) return fail(DS_ERR_INVALID, "%s: negative n_pairs", who);
  if (n_pairs == 0) return DS_OK;
  if (!pair_idx) return fail(DS_ERR_INVALID, "%s: pair_idx: null pointer", who);
  if (n_pairs > INT32_MAX / 8) return fail(DS_ERR_INVALID, "%s: too many pairs", who);
  bool aliased;
  int rc = groups_bwd_check(q, k, v, k, v, mode, d_scores, dq, dk, dv, dk, dv, who, &aliased);
  if (rc != DS_OK) return rc;
  const int64_t G = 2 * n_pairs;
  Workspace w(ws, ws_bytes);
  int32_t* gq = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* kv = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* go = static_cast<int32_t*>(w.take((size_t)(G + 1) * 4));
  float* d_dir = static_cast<float*>(w.take((size_t)G * 4));
  GroupsBwdWs L;
  if (!gq || !kv || !go || !d_dir || !groups_bwd_layout(w, q, k, G, G, &L))
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_aas_pairs_bwd_workspace_bytes(q, n_pairs));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = launch_pairs_setup(pair_idx, n_pairs, gq, go, kv, st)) != DS_OK) return rc;
  pairs_ddir_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(d_scores, n_pairs, d_dir);
  DS_CUDA_TRY(cudaGetLastError());
  return groups_bwd_launch(q, k, v, k, v, gq, go, G, kv, G, scale, mode, d_dir, dq, dk, dv, dk, dv, aliased, L, who, st);
}

size_t ds_aas_triplets_bwd_workspace_bytes(ds_tensor5 q, int64_t n_triplets) {
  using namespace ds;
  if (n_triplets <= 0) return 256;
  const size_t lists = align_up((size_t)(3 * n_triplets) * 4, 256) + align_up((size_t)(3 * n_triplets + 1) * 4, 256) +
                       2 * align_up((size_t)(4 * n_triplets) * 4, 256);   // group_q, group_off, kv_idx, d_dir
  return lists + ds_aas_groups_bwd_workspace_bytes(q, q, 3 * n_triplets, 4 * n_triplets) + 256;
}

int ds_aas_triplets_bwd(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* trip_idx, int64_t n_triplets,
                        float scale, int mode, const float* d_ab, const float* d_ac, ds_tensor5 dq, ds_tensor5 dk,
                        ds_tensor5 dv, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_aas_triplets_bwd";
  if (n_triplets < 0) return fail(DS_ERR_INVALID, "%s: negative n_triplets", who);
  if (n_triplets == 0) return DS_OK;
  if (!trip_idx) return fail(DS_ERR_INVALID, "%s: trip_idx: null pointer", who);
  if (!d_ab || !d_ac) return fail(DS_ERR_INVALID, "%s: d_ab / d_ac: null pointer", who);
  if (n_triplets > INT32_MAX / 16) return fail(DS_ERR_INVALID, "%s: too many triplets", who);
  bool aliased;
  int rc = groups_bwd_check(q, k, v, k, v, mode, d_ab, dq, dk, dv, dk, dv, who, &aliased);
  if (rc != DS_OK) return rc;
  const int64_t G = 3 * n_triplets, T = 4 * n_triplets;
  Workspace w(ws, ws_bytes);
  int32_t* gq = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* go = static_cast<int32_t*>(w.take((size_t)(G + 1) * 4));
  int32_t* kv = static_cast<int32_t*>(w.take((size_t)T * 4));
  float* d_dir = static_cast<float*>(w.take((size_t)T * 4));
  GroupsBwdWs L;
  if (!gq || !go || !kv || !d_dir || !groups_bwd_layout(w, q, k, G, T, &L))
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_aas_triplets_bwd_workspace_bytes(q, n_triplets));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = launch_triplets_setup(trip_idx, n_triplets, gq, go, kv, st)) != DS_OK) return rc;
  triplets_ddir_kernel<<<(unsigned)((n_triplets + 255) / 256), 256, 0, st>>>(d_ab, d_ac, n_triplets, d_dir);
  DS_CUDA_TRY(cudaGetLastError());
  return groups_bwd_launch(q, k, v, k, v, gq, go, G, kv, T, scale, mode, d_dir, dq, dk, dv, dk, dv, aliased, L, who, st);
}

}  // extern "C"

namespace ds {
namespace bwd {

// workspace layout of ds_aas_matrix_bwd (the size query runs it on a dummy base).  E = n_rows n_cols entries.
// The buffers of the grouped backward, with n_rows groups: o holds Y_r at slot r and X_t at n_rows + t; f, lse and delta
// have E + n_rows slots, fx_t at slot t and the folded F_r at E + r.
struct MatrixBwdWs : GroupsBwdWs {
  float* fold32;           // [n_rows] fp32 F_r images
  float* fold_scale;       // [n_rows]
  int32_t* row_max;        // [n_rows]
  int32_t* group_q;        // [n_rows]
  int32_t* group_off;      // [n_rows + 1]
  int32_t* kv_idx;         // [E]
  float* d_dir;            // [E]
};

static bool matrix_bwd_layout(Workspace& w, const ds_tensor5& q, const ds_tensor5& k, MatrixBwdWs* L) {
  const int64_t R = q.size[0], Cn = k.size[0], E = R * Cn, nt = E + R;   // nt: live terms, E cross + R folded self
  const int64_t img = q.size[1] * q.size[2] * q.size[3] * q.size[4];
  const int64_t n_qt = (q.size[3] + kTile - 1) / kTile;
  const size_t stats = (size_t)nt * q.size[1] * q.size[2] * n_qt * kTile * sizeof(float);
  L->o = w.take((size_t)(R + E) * img * 2);
  L->f = w.take((size_t)nt * img * 2);
  L->fold32 = static_cast<float*>(w.take((size_t)R * img * sizeof(float)));
  L->part = static_cast<float*>(w.take((size_t)E * kRedBlocks * 3 * sizeof(float)));
  L->coef = static_cast<float*>(w.take((size_t)E * 4 * sizeof(float)));
  L->lse = static_cast<float*>(w.take(stats));
  L->delta = static_cast<float*>(w.take(stats));
  L->fold_scale = static_cast<float*>(w.take((size_t)R * sizeof(float)));
  L->row_max = static_cast<int32_t*>(w.take((size_t)R * 4));
  L->group_q = static_cast<int32_t*>(w.take((size_t)R * 4));
  L->group_off = static_cast<int32_t*>(w.take((size_t)(R + 1) * 4));
  L->kv_idx = static_cast<int32_t*>(w.take((size_t)E * 4));
  L->entry_group = static_cast<int32_t*>(w.take((size_t)E * 4));
  L->d_dir = static_cast<float*>(w.take((size_t)E * sizeof(float)));
  L->bad = static_cast<int32_t*>(w.take(4));
  const bool ok = L->o && L->f && L->fold32 && L->part && L->coef && L->lse && L->delta && L->fold_scale &&
                  L->row_max && L->group_q && L->group_off && L->kv_idx && L->entry_group && L->d_dir && L->bad;
  return ok && take_family(w, &L->fam[0], R, R, nt) && take_family(w, &L->fam[1], Cn + R, Cn + R, nt);
}

}  // namespace bwd
}  // namespace ds

extern "C" {

size_t ds_aas_matrix_bwd_workspace_bytes(ds_tensor5 q, ds_tensor5 k) {
  using namespace ds::bwd;
  if (q.size[0] <= 0 || k.size[0] <= 0) return 256;
  ds::Workspace w = size_query();
  MatrixBwdWs L;
  matrix_bwd_layout(w, q, k, &L);
  return w.off + 256;
}

int ds_aas_matrix_bwd(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v, float scale,
                      int mode, const float* d_Dm, int64_t ldd, ds_tensor5 dq, ds_tensor5 dk_self, ds_tensor5 dv_self,
                      ds_tensor5 dk, ds_tensor5 dv, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  using namespace ds::bwd;
  const char* who = "ds_aas_matrix_bwd";
  const int64_t R = q.size[0], Cn = k.size[0], E = R * Cn;
  if (R <= 0 || Cn <= 0) return fail(DS_ERR_INVALID, "%s: empty image set", who);
  if (ldd < Cn) return fail(DS_ERR_INVALID, "%s: ldd < columns", who);
  // the term index 2t + 1 of the lists is an int32
  if (E > INT32_MAX / 4) return fail(DS_ERR_INVALID, "%s: more than 2^29 entries; split the rows", who);
  // the two gradient families: row terms (dq, dk_self, dv_self) and column terms (dk, dv), each given whole or null
  const bool rows = dq.ptr || dk_self.ptr || dv_self.ptr, cols = dk.ptr || dv.ptr;
  const bool all_rows = dq.ptr && dk_self.ptr && dv_self.ptr, all_cols = dk.ptr && dv.ptr;
  if ((!all_rows || !all_cols) && ((dk_self.ptr && dk_self.ptr == dk.ptr) || (dv_self.ptr && dv_self.ptr == dv.ptr)))
    return fail(DS_ERR_INVALID, "%s: dk_self / dk (dv_self / dv) may be one tensor only when all five gradients are given",
                who);
  if (rows && !all_rows)
    return fail(DS_ERR_INVALID, "%s: dq, dk_self and dv_self must be all given or all null (no row terms)", who);
  if (cols && !all_cols) return fail(DS_ERR_INVALID, "%s: dk and dv must be both given or both null (no column terms)", who);
  if (!rows && !cols) return fail(DS_ERR_INVALID, "%s: all five gradients are null", who);
  bool aliased;
  int rc = groups_bwd_check(q, k_self, v_self, k, v, mode, d_Dm, dq, dk_self, dv_self, dk, dv, who, &aliased, rows, cols);
  if (rc != DS_OK) return rc;
  ListParamsT<true> p;
  int64_t grid_q, grid_kv;
  if (!list_params(q, k, k_self, scale, R, E, aliased, &p, &grid_q, &grid_kv))
    return fail(DS_ERR_INVALID, "%s: too many tiles: split the rows", who);
  if (!rows || !cols)   // one family: the dK/dV lists are those of the columns only, or of the rows' self terms only
    grid_kv = (rows ? R : Cn) * p.B * p.H * std::max(p.n_kt, p.n_kt_self);
  Workspace w(ws, ws_bytes);
  MatrixBwdWs L;
  if (!matrix_bwd_layout(w, q, k, &L))
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_aas_matrix_bwd_workspace_bytes(q, k));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  set_pointers(&p, L.group_q, L.kv_idx, L, dq, dk_self, dv_self, dk, dv);
  p.n_entries = E;
  p.fold_scale = L.fold_scale;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n2 = p.img / 2;
  const bool bf = q.dtype == DS_BF16;

  DS_CUDA_TRY(cudaMemsetAsync(L.bad, 0, sizeof(int32_t), st));
  if (rows) DS_CUDA_TRY(cudaMemsetAsync(L.row_max, 0, (size_t)R * 4, st));
  matrix_bwd_setup_kernel<<<(unsigned)((E + 256) / 256), 256, 0, st>>>(R, Cn, d_Dm, ldd, L.group_q, L.group_off, L.kv_idx,
                                                                      L.entry_group, L.d_dir);
  DS_CUDA_TRY(cudaGetLastError());
  ListBuildT<true> lb;
  set_list_build(&lb, L.group_q, L.kv_idx, E, q, k, aliased, p, L);
  lb.n_cols = (int)Cn;
  lb.rows = rows;
  lb.cols = cols;
  build_lists_kernel<true><<<2, kListThreads, 0, st>>>(lb);
  DS_CUDA_TRY(cudaGetLastError());
  // X_t and Y_r, rounded to the input dtype as ds_attn_fwd rounds them
  if ((rc = attn_list_store(q, k_self, v_self, k, v, L.group_q, L.group_off, R, L.kv_idx, scale, L.o, who, st)) != DS_OK)
    return rc;
  if ((rc = launch_list_coefs(q, p, E, mode, L.d_dir, L, st)) != DS_OK) return rc;
  const uint32_t* ou = static_cast<const uint32_t*>(L.o);
  const unsigned ry = (unsigned)std::min<int64_t>(R, 65535);
  const unsigned fb = (unsigned)std::min<int64_t>((n2 + 255) / 256, 4 * (int64_t)sm_count());
  uint32_t* fu = static_cast<uint32_t*>(L.f);
  float2* f32 = reinterpret_cast<float2*>(L.fold32);
  if (!rows) {   // fx_t only: no self term is folded
    if (bf) matrix_fold_kernel<true, false><<<dim3(fb, ry), kRedThreads, 0, st>>>(ou, n2, (int)R, (int)Cn, mode, L.coef, fu, f32, L.row_max);
    else matrix_fold_kernel<false, false><<<dim3(fb, ry), kRedThreads, 0, st>>>(ou, n2, (int)R, (int)Cn, mode, L.coef, fu, f32, L.row_max);
    DS_CUDA_TRY(cudaGetLastError());
  } else {
    if (bf) matrix_fold_kernel<true><<<dim3(fb, ry), kRedThreads, 0, st>>>(ou, n2, (int)R, (int)Cn, mode, L.coef, fu, f32, L.row_max);
    else matrix_fold_kernel<false><<<dim3(fb, ry), kRedThreads, 0, st>>>(ou, n2, (int)R, (int)Cn, mode, L.coef, fu, f32, L.row_max);
    DS_CUDA_TRY(cudaGetLastError());
    uint32_t* f16 = fu + E * n2;
    if (bf) matrix_fold_round_kernel<true><<<dim3(fb, ry), 256, 0, st>>>(f32, n2, (int)R, L.row_max, f16, L.fold_scale);
    else matrix_fold_round_kernel<false><<<dim3(fb, ry), 256, 0, st>>>(f32, n2, (int)R, L.row_max, f16, L.fold_scale);
    DS_CUDA_TRY(cudaGetLastError());
  }

  const ds_tensor5 F = factor_stack(q, L.f, E + R);
  return with_head_dim(q.size[4], who, [&](auto d) {
    return with_dtype(q.dtype, [&](auto b) {
      constexpr int kD = decltype(d)::value;
      constexpr bool kB = decltype(b)::value;
      // without the row terms the dQ kernel only writes the cross terms' LSE and delta for the dK/dV kernel
      return rows ? launch_groups_bwd_t<kD, kB, true>(q, k_self, v_self, k, v, F, p, grid_q, grid_kv, L.fam, st)
                  : launch_groups_bwd_t<kD, kB, true, true>(q, k_self, v_self, k, v, F, p, grid_q, grid_kv, L.fam, st);
    });
  });
}

}  // extern "C"
