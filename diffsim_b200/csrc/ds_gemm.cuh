// Shared tcgen05 GEMM core:  C[M,N] = A[M,K] . B[N,K]^T   (both operands K-major 16-bit, fp32 accumulation in TMEM).
//
// Used by K3 (N x N similarity matrix: fp32 split-K partials, ds_simmat.cu) and K4 (QKV projection of the hooked
// attention layer: 16-bit outputs scattered into the Q / K / V caches, ds_qkv.cu).  K4's backward products take MN-major
// operands through the kernels at the end of this file (gemm_bwd_kernel / gemm2_bwd_kernel).
//
// Persistent, warp-specialised, one CTA per SM:
//   warp 0      TMA producer   ring of kGemmStages x (A 128x64 + B 256x64) 128B-swizzled tiles
//   warp 1      MMA issuer     tcgen05.mma cta_group::1, M = 128, N = 256, K = 16; also owns the TMEM allocation
//   warps 2-5   epilogue       one TMEM lane quadrant each; TMEM -> registers -> global
// The 512 TMEM columns hold two 128x256 fp32 accumulators, so the epilogue of work unit u overlaps the main loop of
// unit u+1.  A work unit is (output tile, k split); units are dealt round-robin to the CTAs, tiles n-fastest so that
// CTAs running side by side share the A tile in L2.
//
// Shared-memory budget of the 1-CTA shape: per 64-wide k block TMA writes 48 KB and the four MMAs read 48 KB, 96 KB
// per 512 tensor clocks = 188 B/clk against a 128 B/clk port: this shape tops out near 68% of the tensor peak; the
// cta_group::2 256x256 shape (half the B reads per CTA) is what lifts that and is the next step for this core.
#pragma once

#include "ds_host.h"
#include "ds_ptx.cuh"

namespace ds {

constexpr int kGBM = 128, kGBN = 256, kGBK = 64;
constexpr int kGStages = 4;
constexpr int kGABytes = kGBM * kGBK * 2;   // 16 KB
constexpr int kGBBytes = kGBN * kGBK * 2;   // 32 KB
constexpr int kGStageBytes = kGABytes + kGBBytes;
constexpr int kGThreads = 192;
constexpr size_t kGSmemBytes = 1024 + (size_t)kGStages * kGStageBytes + 256 + 4 * 4096;   // + epilogue staging patches

enum : int { GEMM_EPI_F32 = 0, GEMM_EPI_16 = 1 };

struct GemmParams {
  int M, N;                 // output extent
  int tiles_m, tiles_n;
  int kb_total;             // 64-wide k blocks
  int splits, kb_per_split;
  int sym;                  // 1: C is symmetric (B == A): only tiles holding an element with row <= col are computed
  int tiles_used;           // tiles per split (tiles_m * tiles_n, or the upper-triangle count when sym)
  uint32_t idesc;
  uint32_t idesc2;          // CTA-pair kernel: M = 256
  int tma_store;            // CTA-pair kernel, 16-bit outputs: epilogue through TMA stores (GemmOutMaps)
  int use_pair;             // -1 automatic (set by launch_gemm_tn's callers that leave it 0-initialised: see below), 0, 1
  // CTA-pair kernel only: operand given as a k-blocked copy [k block][rows_pad][64] (rows_pad a multiple of 256, value
  // here; 0 = the row-major operand).  A TMA box is then one contiguous run instead of 128 row pieces 2*ld bytes apart.
  int kblk_rows_a, kblk_rows_b;
  // GEMM_EPI_F32: part[split][M][N] fp32
  float* part;
  int64_t part_split_stride;
  // GEMM_EPI_16: column n goes to out[n / cols_per_out] at column n % cols_per_out; bias (may be null) has the
  // input dtype and N entries
  void* out[3];
  int64_t ld_out[3];
  int cols_per_out;
  const void* bias;
};

// tiles of one split, n fastest.  Symmetric mode enumerates, row of tiles by row of tiles, only the tiles that hold an
// element on or above the diagonal: tile (tm, tn) is needed iff tm * kGBM <= tn * kGBN + kGBN - 1, i.e. tn >= tm*kGBM / kGBN.
__host__ __device__ __forceinline__ int gemm_sym_first_tn(int tm, int bm = kGBM) { return (tm * bm) / kGBN; }

__device__ __forceinline__ void gemm_decode_tile(const GemmParams& p, int tile, int& tm, int& tn, int bm = kGBM) {
  if (!p.sym) {
    tm = tile / p.tiles_n;
    tn = tile - tm * p.tiles_n;
    return;
  }
  tm = 0;
  for (;;) {
    const int first = gemm_sym_first_tn(tm, bm);
    const int cnt = p.tiles_n - first;
    if (tile < cnt) {
      tn = first + tile;
      return;
    }
    tile -= cnt;
    ++tm;
  }
}

static int gemm_sym_tile_count(int tiles_m, int tiles_n, int bm = kGBM) {
  int n = 0;
  for (int tm = 0; tm < tiles_m; ++tm) {
    const int cnt = tiles_n - gemm_sym_first_tn(tm, bm);
    if (cnt > 0) n += cnt;
  }
  return n;
}

// 64 accumulator columns of this thread's row: TMEM -> (+ bias) -> 32 packed 16-bit pairs (128 bytes)
template <bool kBf16>
__device__ __forceinline__ void gemm_load_row64(const GemmParams& p, uint32_t t_addr, int col0, uint32_t (&w)[32]) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    uint32_t v[32];
    tmem_ld_x32(t_addr + half * 32, v);
    tmem_wait_ld();
    const int cb = col0 + half * 32;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(v[g * 8 + j]);
      if (p.bias && cb + g * 8 < p.N) {
        const uint4 b4 = __ldg(reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(p.bias) + cb + g * 8));
        const uint32_t bw[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 bf = unpack2<kBf16>(bw[j]);
          f[2 * j] += bf.x;
          f[2 * j + 1] += bf.y;
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) w[half * 16 + g * 4 + j] = pack2<kBf16>(f[2 * j], f[2 * j + 1]);
    }
  }
}

// Epilogue of one warp: its 32 accumulator rows (TMEM lanes) across the kGBN columns of the tile, 128 bytes of a row per
// pass (32 fp32 partials or 64 16-bit outputs).  A thread owns a ROW in TMEM, so storing straight from registers makes every
// warp-wide 16-byte store touch 32 different 128-byte lines (measured: the projection runs at 1166 TFLOP/s with such stores
// and at 1535 with the stores removed).  The 32 x 128 B block is therefore turned through a 4 KB shared-memory patch
// (16-byte units XOR-swizzled by row: conflict-free both ways) and written out with 8 lanes per row: 4 full lines per store.
constexpr int kGEpiStageBytes = 32 * 128;   // per epilogue warp

template <int EPI, bool kBf16>
__device__ __forceinline__ void gemm_epilogue_rows(const GemmParams& p, uint32_t t_addr, int row0, int n0, int split,
                                                   uint8_t* stage, int lane) {
  constexpr int COLS = (EPI == GEMM_EPI_F32) ? 32 : 64;   // columns per 128-byte row segment
  constexpr int UCOLS = COLS / 8;                         // columns per 16-byte unit
  const uint32_t st_base = smem_u32(stage);
#pragma unroll 1
  for (int ps = 0; ps < kGBN / COLS; ++ps) {
    const int col0 = n0 + ps * COLS;
    if (col0 >= p.N) break;                               // warp-uniform
    uint32_t w[32];
    if constexpr (EPI == GEMM_EPI_F32) {
      tmem_ld_x32(t_addr + ps * 32, w);
      tmem_wait_ld();
    } else {
      gemm_load_row64<kBf16>(p, t_addr + ps * 64, col0, w);
    }
    // registers (thread = row) -> staging patch
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const uint32_t a = st_base + (uint32_t)lane * 128u + (uint32_t)((u ^ (lane & 7)) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(w[4 * u]), "r"(w[4 * u + 1]), "r"(w[4 * u + 2]),
                   "r"(w[4 * u + 3])
                   : "memory");
    }
    __syncwarp();
    // staging patch -> global (8 lanes per row)
    const int u = lane & 7;
    const int col = col0 + u * UCOLS;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int r = (lane >> 3) + 4 * j;
      uint4 x;
      const uint32_t a = st_base + (uint32_t)r * 128u + (uint32_t)((u ^ (r & 7)) << 4);
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w) : "r"(a) : "memory");
      const int row = row0 + r;
      if (row >= p.M || col >= p.N) continue;
      if constexpr (EPI == GEMM_EPI_F32) {
        float* dst = p.part + (size_t)split * p.part_split_stride + (size_t)row * p.N + col;
        if ((p.N & 3) == 0 && col + 4 <= p.N) {
          *reinterpret_cast<uint4*>(dst) = x;
        } else {
          const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (col + e < p.N) dst[e] = __uint_as_float(xs[e]);
        }
      } else {
        // 8-column units: N and cols_per_out are multiples of 8 (checked by the host)
        const int t = col / p.cols_per_out, cc = col - t * p.cols_per_out;
        uint16_t* dst = static_cast<uint16_t*>(p.out[t]) + (size_t)row * p.ld_out[t] + cc;
        *reinterpret_cast<uint4*>(dst) = x;
      }
    }
    __syncwarp();
  }
}

template <int EPI, bool kBf16>
__global__ void __launch_bounds__(kGThreads, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kGStages * kGStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kGStages;
  uint64_t* acc_full = bars + 2 * kGStages;        // [2]
  uint64_t* acc_empty = bars + 2 * kGStages + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kGStages + 4);
  uint8_t* epi_stage = reinterpret_cast<uint8_t*>(bars) + 256;   // 4 x 4 KB, 128-byte aligned

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kGStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 4);   // one elected lane per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles = p.tiles_used;
  const int n_units = tiles * p.splits;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int split = u / tiles, tile = u - split * tiles;
        int tm, tn;
        gemm_decode_tile(p, tile, tm, tn);
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* a = smem + (size_t)stage * kGStageBytes;
          mbar_arrive_expect_tx(&full[stage], kGStageBytes);
          tma_load_2d(a, &map_a, &full[stage], kb * kGBK, tm * kGBM);
          tma_load_2d(a + kGABytes, &map_b, &full[stage], kb * kGBK, tn * kGBN);
          if (++stage == kGStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0, n_local = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++n_local) {
        const int split = u / tiles;
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const uint32_t buf = n_local & 1u;
        mbar_wait(&acc_empty[buf], ((n_local >> 1) & 1u) ^ 1u);   // the epilogue has drained this accumulator
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * kGBN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_addr = smem_u32(smem + (size_t)stage * kGStageBytes);
          const uint64_t a_desc = umma_smem_desc(a_addr, 16, 1024, UMMA_SW128);
          const uint64_t b_desc = umma_smem_desc(a_addr + kGABytes, 16, 1024, UMMA_SW128);
#pragma unroll
          for (int k = 0; k < kGBK / 16; ++k) {
            // advance 16 elements (32 bytes) along K inside the swizzle atom: +2 in 16-byte units
            umma_f16_ss(d_tmem, a_desc + 2 * k, b_desc + 2 * k, p.idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (++stage == kGStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // epilogue: warp w may only touch TMEM lanes [32*(w%4), 32*(w%4)+32)
    const int quad = warp & 3;
    uint32_t n_local = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++n_local) {
      const int split = u / tiles, tile = u - split * tiles;
      int tm, tn;
      gemm_decode_tile(p, tile, tm, tn);
      const uint32_t buf = n_local & 1u;
      mbar_wait(&acc_full[buf], (n_local >> 1) & 1u);
      tc_fence_after_sync();
      const int n0 = tn * kGBN;
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * kGBN;
      gemm_epilogue_rows<EPI, kBf16>(p, t_addr, tm * kGBM + quad * 32, n0, split, epi_stage + (warp - 2) * kGEpiStageBytes, lane);
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Tensor maps of the (up to three) 16-bit output tensors, [M rows, cols_per_out] with their own row strides; box = 64
// columns x 32 rows, 128-byte swizzle (the layout the epilogue's staging patch already has).
struct GemmOutMaps {
  CUtensorMap m[3];
};

// Epilogue of one warp through TMA stores: 32 rows x 64 columns per pass go registers -> swizzled 4 KB patch (two per
// warp, alternating) -> one cp.async.bulk.tensor store issued by lane 0.  The copy engine reads the patch and writes
// full lines; rows past M and columns past the tensor are clipped by the hardware.  `pass` counts this warp's passes.
template <bool kBf16>
__device__ __forceinline__ void gemm_epilogue_rows_tma(const GemmParams& p, const GemmOutMaps& om, uint32_t t_addr, int row0,
                                                       int n0, uint8_t* patches, int lane, uint32_t& pass) {
#pragma unroll 1
  for (int ps = 0; ps < kGBN / 64; ++ps, ++pass) {
    const int col0 = n0 + ps * 64;
    if (col0 >= p.N) break;                               // warp-uniform
    uint8_t* patch = patches + (pass & 1u) * kGEpiStageBytes;
    const uint32_t st_base = smem_u32(patch);
    // the store issued two passes ago has finished reading this patch
    if (lane == 0) tma_store_wait_read<1>();
    __syncwarp();
    uint32_t w[32];
    gemm_load_row64<kBf16>(p, t_addr + ps * 64, col0, w);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const uint32_t a = st_base + (uint32_t)lane * 128u + (uint32_t)((u ^ (lane & 7)) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(w[4 * u]), "r"(w[4 * u + 1]), "r"(w[4 * u + 2]),
                   "r"(w[4 * u + 3])
                   : "memory");
    }
    fence_proxy_async_smem();      // generic-proxy writes -> visible to the copy engine
    __syncwarp();
    if (lane == 0) {
      const int t = col0 / p.cols_per_out;                // cols_per_out % 64 == 0: one tensor per pass
      tma_store_2d(&om.m[t], patch, col0 - t * p.cols_per_out, row0);
      tma_store_commit();
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// CTA-pair variant: one cluster of two CTAs per 256 x 256 output tile (tcgen05.mma.cta_group::2, M = 256).
// Each CTA streams its own 128 rows of A and HALF of the B tile (128 of the 256 rows): per 64-wide k block it writes
// 32 KB and its tensor core reads 32 KB of its own shared memory -- 125 B/clk against the 128 B/clk port, where the
// 1-CTA shape needs 188 -- and the ring holds 6 stages instead of 4.  The leader (cluster rank 0) issues the MMAs for
// both; completion is multicast to the barriers of both CTAs; each CTA's epilogue drains its own 128 accumulator rows.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kG2BM = 256;                          // rows per cluster tile (128 per CTA)
constexpr int kG2Stages = 6;
constexpr int kG2BHalfBytes = (kGBN / 2) * kGBK * 2;   // 16 KB: this CTA's half of the B tile
constexpr int kG2StageBytes = kGABytes + kG2BHalfBytes;
constexpr size_t kG2SmemBytes = 1024 + (size_t)kG2Stages * kG2StageBytes + 1024 + 8 * 4096;   // ring | barriers | 2 patches per epilogue warp

template <int EPI, bool kBf16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGThreads, 1)
gemm2_tn_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                const __grid_constant__ GemmOutMaps omaps, const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kG2Stages * kG2StageBytes);
  uint64_t* full = bars;                              // leader's copy counts the bytes of both CTAs
  uint64_t* empty = bars + kG2Stages;                 // each CTA's copy is signalled by the multicast commit
  uint64_t* acc_full = bars + 2 * kG2Stages;          // [2] multicast commit
  uint64_t* acc_empty = bars + 2 * kG2Stages + 2;     // [2] leader's copy: 8 arrivals (4 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kG2Stages + 4);
  uint8_t* epi_stage = reinterpret_cast<uint8_t*>(bars) + 1024;  // 4 warps x 2 x 4 KB, 1024-byte aligned (swizzle atoms)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kG2Stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 8);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before_sync();
  cluster_sync_all();            // barriers of BOTH CTAs are initialised before anyone signals across the pair
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles = p.tiles_used;
  const int n_units = tiles * p.splits;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = cluster_id; u < n_units; u += n_clusters) {
        const int split = u / tiles, tile = u - split * tiles;
        int tm, tn;
        gemm_decode_tile(p, tile, tm, tn, kG2BM);
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* a = smem + (size_t)stage * kG2StageBytes;
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * kG2StageBytes);
          tma_load_2d_2cta(a, &map_a, &full[stage], p.kblk_rows_a ? 0 : kb * kGBK,
                           kb * p.kblk_rows_a + tm * kG2BM + (int)rank * kGBM);
          tma_load_2d_2cta(a + kGABytes, &map_b, &full[stage], p.kblk_rows_b ? 0 : kb * kGBK,
                           kb * p.kblk_rows_b + tn * kGBN + (int)rank * (kGBN / 2));
          if (++stage == kG2Stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && elect_one()) {
      int stage = 0;
      uint32_t phase = 0, n_local = 0;
      for (int u = cluster_id; u < n_units; u += n_clusters, ++n_local) {
        const int split = u / tiles;
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const uint32_t buf = n_local & 1u;
        mbar_wait(&acc_empty[buf], ((n_local >> 1) & 1u) ^ 1u);   // both epilogues have drained this accumulator
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * kGBN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_addr = smem_u32(smem + (size_t)stage * kG2StageBytes);
          const uint64_t a_desc = umma_smem_desc(a_addr, 16, 1024, UMMA_SW128);
          const uint64_t b_desc = umma_smem_desc(a_addr + kGABytes, 16, 1024, UMMA_SW128);
#pragma unroll
          for (int k = 0; k < kGBK / 16; ++k)
            umma_f16_ss_2cta(d_tmem, a_desc + 2 * k, b_desc + 2 * k, p.idesc2, (kb > kb0 || k > 0) ? 1u : 0u);
          umma_commit_2cta(&empty[stage]);
          if (++stage == kG2Stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_2cta(&acc_full[buf]);
      }
    }
  } else {
    const int quad = warp & 3;
    uint32_t n_local = 0, pass = 0;
    uint8_t* my_patches = epi_stage + (warp - 2) * 2 * kGEpiStageBytes;
    for (int u = cluster_id; u < n_units; u += n_clusters, ++n_local) {
      const int split = u / tiles, tile = u - split * tiles;
      int tm, tn;
      gemm_decode_tile(p, tile, tm, tn, kG2BM);
      const uint32_t buf = n_local & 1u;
      mbar_wait(&acc_full[buf], (n_local >> 1) & 1u);
      tc_fence_after_sync();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * kGBN;
      const int row0 = tm * kG2BM + (int)rank * kGBM + quad * 32;
      if constexpr (EPI == GEMM_EPI_16) {
        if (p.tma_store) gemm_epilogue_rows_tma<kBf16>(p, omaps, t_addr, row0, tn * kGBN, my_patches, lane, pass);
        else gemm_epilogue_rows<EPI, kBf16>(p, t_addr, row0, tn * kGBN, split, my_patches, lane);
      } else {
        gemm_epilogue_rows<EPI, kBf16>(p, t_addr, row0, tn * kGBN, split, my_patches, lane);
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&acc_empty[buf]);
    }
    if (lane == 0) tma_store_wait_all();   // outstanding bulk stores complete before the CTA retires
  }
  tc_fence_before_sync();
  cluster_sync_all();            // the peer may still be reading this CTA's B half / signalling its barriers
  if (warp == 1) tmem_dealloc_2cta(tmem_base, 512);
}

// Which kernel serves a problem: the debug override (ds_debug_set_gemm_variant: -1 automatic, 0 1-CTA only, 2 pairs always),
// else the caller's choice (GemmParams::use_pair: 0 / 1), else pairs when the 256 x 256 tiles fill the clusters twice over.
static bool gemm_use_pair(int64_t M, int64_t N, int splits, int use_pair) {
  if (g_gemm_variant == 0) return false;
  if (g_gemm_variant == 2) return true;
  if (use_pair >= 0) return use_pair != 0;
  const int64_t tiles2 = ((M + kG2BM - 1) / kG2BM) * ((N + kGBN - 1) / kGBN);
  return tiles2 * (splits < 1 ? 1 : splits) >= 2 * (sm_count() / 2);
}

// Host side: tensor maps + launch.  a: [M, K] with leading dimension lda (elements), b: [N, K] with ldb.
template <int EPI>
static int launch_gemm_tn(const void* a, int64_t M, int64_t lda, const void* b, int64_t N, int64_t ldb, int64_t K, int dtype,
                          GemmParams p, cudaStream_t st) {
  CUtensorMap map_a, map_b;
  int rc;
  {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)M};
    uint64_t str[1] = {(uint64_t)lda * 2};
    uint32_t box[2] = {(uint32_t)kGBK, (uint32_t)kGBM};
    if (!p.kblk_rows_a && (rc = encode_tensor_map(&map_a, dtype, 2, a, dims, str, box, 128)) != DS_OK) return rc;
    uint64_t dimsb[2] = {(uint64_t)K, (uint64_t)N};
    uint64_t strb[1] = {(uint64_t)ldb * 2};
    uint32_t boxb[2] = {(uint32_t)kGBK, (uint32_t)kGBN};
    if (!p.kblk_rows_b && (rc = encode_tensor_map(&map_b, dtype, 2, b, dimsb, strb, boxb, 128)) != DS_OK) return rc;
  }
  p.M = (int)M;
  p.N = (int)N;
  // CTA pairs (256 x 256 tiles) when there are enough of them to fill the 74 clusters; small problems keep the 1-CTA shape
  const bool pair = gemm_use_pair(M, N, p.splits, p.use_pair);
  if ((p.kblk_rows_a || p.kblk_rows_b) && !pair) return fail(DS_ERR_INVALID, "gemm: k-blocked operands need the CTA-pair kernel");
  if (pair) {
    uint64_t dimsb2[2] = {(uint64_t)K, (uint64_t)N};
    uint64_t strb2[1] = {(uint64_t)ldb * 2};
    uint32_t boxb2[2] = {(uint32_t)kGBK, (uint32_t)(kGBN / 2)};
    if (!p.kblk_rows_b && (rc = encode_tensor_map(&map_b, dtype, 2, b, dimsb2, strb2, boxb2, 128)) != DS_OK) return rc;
    // k-blocked operands: a 2-D view [k blocks * rows_pad][64], row pitch 128 bytes
    const uint64_t kbt = (uint64_t)((K + kGBK - 1) / kGBK);
    if (p.kblk_rows_a) {
      uint64_t d[2] = {(uint64_t)kGBK, kbt * (uint64_t)p.kblk_rows_a};
      uint64_t s1[1] = {(uint64_t)kGBK * 2};
      uint32_t bx[2] = {(uint32_t)kGBK, (uint32_t)kGBM};
      if (kbt * (uint64_t)p.kblk_rows_a > (uint64_t)INT32_MAX) return fail(DS_ERR_INVALID, "gemm: k-blocked operand too large");
      if ((rc = encode_tensor_map(&map_a, dtype, 2, a, d, s1, bx, 128)) != DS_OK) return rc;
    }
    if (p.kblk_rows_b) {
      uint64_t d[2] = {(uint64_t)kGBK, kbt * (uint64_t)p.kblk_rows_b};
      uint64_t s1[1] = {(uint64_t)kGBK * 2};
      uint32_t bx[2] = {(uint32_t)kGBK, (uint32_t)(kGBN / 2)};
      if (kbt * (uint64_t)p.kblk_rows_b > (uint64_t)INT32_MAX) return fail(DS_ERR_INVALID, "gemm: k-blocked operand too large");
      if ((rc = encode_tensor_map(&map_b, dtype, 2, b, d, s1, bx, 128)) != DS_OK) return rc;
    }
    p.tiles_m = (int)((M + kG2BM - 1) / kG2BM);
    p.tiles_n = (int)((N + kGBN - 1) / kGBN);
    p.kb_total = (int)((K + kGBK - 1) / kGBK);
    if (p.splits < 1) p.splits = 1;
    p.kb_per_split = (p.kb_total + p.splits - 1) / p.splits;
    p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
    p.idesc2 = umma_idesc_f16(dtype == DS_BF16 ? 1u : 0u, kG2BM, kGBN, 0, 0);
    if (p.sym && (M != N || a != b || lda != ldb)) return fail(DS_ERR_INVALID, "gemm: symmetric mode needs B == A");
    p.tiles_used = p.sym ? gemm_sym_tile_count(p.tiles_m, p.tiles_n, kG2BM) : p.tiles_m * p.tiles_n;
    const int64_t units2 = (int64_t)p.tiles_used * p.splits;
    if (units2 <= 0) return DS_OK;
    if (units2 > INT32_MAX) return fail(DS_ERR_INVALID, "gemm: too many work units");
    int clusters = sm_count() / 2;
    if (units2 < clusters) clusters = (int)units2;
    GemmOutMaps om;
    memset(&om, 0, sizeof(om));
    p.tma_store = 0;
    if (EPI == GEMM_EPI_16 && p.cols_per_out % 64 == 0) {
      const int n_t = (int)(N / p.cols_per_out);
      p.tma_store = 1;
      for (int t = 0; t < n_t && t < 3; ++t) {
        uint64_t od[2] = {(uint64_t)p.cols_per_out, (uint64_t)M};
        uint64_t os[1] = {(uint64_t)p.ld_out[t] * 2};
        uint32_t ob[2] = {64u, 32u};
        if ((rc = encode_tensor_map(&om.m[t], dtype, 2, p.out[t], od, os, ob, 128)) != DS_OK) return rc;
      }
    }
    if (dtype == DS_BF16) {
      DS_CUDA_TRY(cudaFuncSetAttribute(gemm2_tn_kernel<EPI, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kG2SmemBytes));
      gemm2_tn_kernel<EPI, true><<<2 * clusters, kGThreads, kG2SmemBytes, st>>>(map_a, map_b, om, p);
    } else {
      DS_CUDA_TRY(cudaFuncSetAttribute(gemm2_tn_kernel<EPI, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kG2SmemBytes));
      gemm2_tn_kernel<EPI, false><<<2 * clusters, kGThreads, kG2SmemBytes, st>>>(map_a, map_b, om, p);
    }
    DS_CUDA_TRY(cudaGetLastError());
    return DS_OK;
  }
  p.tiles_m = (int)((M + kGBM - 1) / kGBM);
  p.tiles_n = (int)((N + kGBN - 1) / kGBN);
  p.kb_total = (int)((K + kGBK - 1) / kGBK);
  if (p.splits < 1) p.splits = 1;
  p.kb_per_split = (p.kb_total + p.splits - 1) / p.splits;
  p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.idesc = umma_idesc_f16(dtype == DS_BF16 ? 1u : 0u, kGBM, kGBN, 0, 0);
  if (p.sym && (M != N || a != b || lda != ldb)) return fail(DS_ERR_INVALID, "gemm: symmetric mode needs B == A");
  p.tiles_used = p.sym ? gemm_sym_tile_count(p.tiles_m, p.tiles_n) : p.tiles_m * p.tiles_n;
  const int64_t units = (int64_t)p.tiles_used * p.splits;
  if (units <= 0) return DS_OK;
  if (units > INT32_MAX) return fail(DS_ERR_INVALID, "gemm: too many work units");
  int grid = sm_count();
  if (units < grid) grid = (int)units;
  if (dtype == DS_BF16) {
    DS_CUDA_TRY(cudaFuncSetAttribute(gemm_tn_kernel<EPI, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGSmemBytes));
    gemm_tn_kernel<EPI, true><<<grid, kGThreads, kGSmemBytes, st>>>(map_a, map_b, p);
  } else {
    DS_CUDA_TRY(cudaFuncSetAttribute(gemm_tn_kernel<EPI, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGSmemBytes));
    gemm_tn_kernel<EPI, false><<<grid, kGThreads, kGSmemBytes, st>>>(map_a, map_b, p);
  }
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward products of a projection Y = X W^T whose output columns are split over n_seg tensors of seg_len columns each
// (K4's q / k / v, or one packed tensor).  dY arrives as those separate tensors and is read in place, one tensor map per
// tensor with its own row stride; a k block (dX) or an M tile (dW) never mixes two tensors, so seg_len need only be a
// multiple of 8: the tail of a tensor's last block is zero-filled by TMA.
//
//   GEMM_BWD_DX  dX[rows, C_in]  = sum_t dY_t W_t       A = dY_t  K-major (as stored), B = W_t [seg_len, C_in] MN-major
//                                                       K = n_seg x seg_len, blocked per tensor: kb -> (t, local kb)
//   GEMM_BWD_DW  dW_t[seg_len, C_in] = dY_t^T X         A = dY_t  MN-major,            B = X [rows, C_in]      MN-major
//                                                       M = n_seg x seg_len, tiled per tensor:   tm -> (t, local tm)
//
// An MN-major tile is stored as MN / 64 swizzled sub-tiles of 64 k rows x 128 bytes (one 64 x 64 TMA box each, as K1 loads
// V for P V); its descriptor has LBO = the sub-tile pitch, SBO = 8 rows, and a K step of 16 rows = 2048 bytes.  Both the
// 1-CTA and the CTA-pair kernel are built on one body; the accumulators always leave as fp32 split-K partials
// part[split][M][N] (GEMM_EPI_F32), which a finishing kernel adds in split order and rounds once.
// ---------------------------------------------------------------------------------------------------------------------
enum : int { GEMM_BWD_DX = 0, GEMM_BWD_DW = 1 };

struct GemmBwdMaps {
  CUtensorMap a[3];   // per tensor: dY_t
  CUtensorMap b[3];   // dX: per tensor W_t; dW: X in b[0]
};

constexpr int kGSubBytes = 64 * kGBK * 2;   // 8 KB: one 64 (MN) x 64 (K) sub-tile of an MN-major operand

template <bool kPair>
__device__ __forceinline__ void gemm_bwd_tma(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  if constexpr (kPair) tma_load_2d_2cta(dst, m, bar, c0, c1);
  else tma_load_2d(dst, m, bar, c0, c1);
}

template <int OP, bool kPair>
__device__ __forceinline__ void gemm_bwd_body(const GemmBwdMaps& maps, const GemmParams& p, int seg_len, int seg_blocks) {
  constexpr int STAGES = kPair ? kG2Stages : kGStages;
  constexpr int STAGE_BYTES = kPair ? kG2StageBytes : kGStageBytes;
  constexpr int BM = kPair ? kG2BM : kGBM;           // output rows per work unit (the pair's tile spans both CTAs)
  constexpr int B_SUBS = (kPair ? kGBN / 2 : kGBN) / 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* acc_full = bars + 2 * STAGES;        // [2]
  uint64_t* acc_empty = bars + 2 * STAGES + 2;   // [2]: one elected lane per epilogue warp (of both CTAs of a pair)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint8_t* epi_stage = reinterpret_cast<uint8_t*>(bars) + (kPair ? 1024 : 256);   // 4 x 4 KB, as the forward kernels

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  if (warp == 0 && lane == 0) {
    for (int t = 0; t < 3; ++t) {
      tma_prefetch_desc(&maps.a[t]);
      tma_prefetch_desc(&maps.b[t]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], kPair ? 8 : 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (kPair) {
      tmem_alloc_2cta(tmem_slot, 512);
      tmem_relinquish_2cta();
    } else {
      tmem_alloc(tmem_slot, 512);
      tmem_relinquish();
    }
  }
  tc_fence_before_sync();
  if constexpr (kPair) cluster_sync_all();
  else __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles = p.tiles_used;
  const int n_units = tiles * p.splits;
  const int unit0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int unit_step = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = unit0; u < n_units; u += unit_step) {
        const int split = u / tiles, tile = u - split * tiles;
        int tm, tn;
        gemm_decode_tile(p, tile, tm, tn, BM);
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const int n_base = tn * kGBN + (int)rank * (kGBN / 2);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* a = smem + (size_t)stage * STAGE_BYTES;
          uint8_t* b = a + kGABytes;
          if (leader) mbar_arrive_expect_tx(&full[stage], kPair ? 2 * STAGE_BYTES : STAGE_BYTES);
          if constexpr (OP == GEMM_BWD_DX) {
            const int t = kb / seg_blocks, k0 = (kb - t * seg_blocks) * kGBK;
            gemm_bwd_tma<kPair>(a, &maps.a[t], &full[stage], k0, tm * BM + (int)rank * kGBM);
#pragma unroll
            for (int s = 0; s < B_SUBS; ++s) gemm_bwd_tma<kPair>(b + s * kGSubBytes, &maps.b[t], &full[stage], n_base + s * 64, k0);
          } else {
            const int t = tm / seg_blocks, m0 = (tm - t * seg_blocks) * BM + (int)rank * kGBM;
#pragma unroll
            for (int s = 0; s < kGBM / 64; ++s) gemm_bwd_tma<kPair>(a + s * kGSubBytes, &maps.a[t], &full[stage], m0 + s * 64, kb * kGBK);
#pragma unroll
            for (int s = 0; s < B_SUBS; ++s) gemm_bwd_tma<kPair>(b + s * kGSubBytes, &maps.b[0], &full[stage], n_base + s * 64, kb * kGBK);
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && elect_one()) {
      int stage = 0;
      uint32_t phase = 0, n_local = 0;
      for (int u = unit0; u < n_units; u += unit_step, ++n_local) {
        const int split = u / tiles;
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const uint32_t buf = n_local & 1u;
        mbar_wait(&acc_empty[buf], ((n_local >> 1) & 1u) ^ 1u);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * kGBN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_addr = smem_u32(smem + (size_t)stage * STAGE_BYTES);
          // K-major: +32 bytes per K = 16 step inside the swizzle atom; MN-major: +16 rows of 128 bytes
          const uint64_t a_desc = OP == GEMM_BWD_DX ? umma_smem_desc(a_addr, 16, 1024, UMMA_SW128)
                                                    : umma_smem_desc(a_addr, kGSubBytes, 1024, UMMA_SW128);
          const uint64_t b_desc = umma_smem_desc(a_addr + kGABytes, kGSubBytes, 1024, UMMA_SW128);
          constexpr uint64_t A_STEP = OP == GEMM_BWD_DX ? 2 : 128, B_STEP = 128;
#pragma unroll
          for (int k = 0; k < kGBK / 16; ++k) {
            const uint32_t acc = (kb > kb0 || k > 0) ? 1u : 0u;
            if constexpr (kPair) umma_f16_ss_2cta(d_tmem, a_desc + A_STEP * k, b_desc + B_STEP * k, p.idesc2, acc);
            else umma_f16_ss(d_tmem, a_desc + A_STEP * k, b_desc + B_STEP * k, p.idesc, acc);
          }
          if constexpr (kPair) umma_commit_2cta(&empty[stage]);
          else umma_commit(&empty[stage]);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if constexpr (kPair) umma_commit_2cta(&acc_full[buf]);
        else umma_commit(&acc_full[buf]);
      }
    }
  } else {
    const int quad = warp & 3;
    uint32_t n_local = 0;
    uint8_t* stage_patch = epi_stage + (warp - 2) * kGEpiStageBytes;
    for (int u = unit0; u < n_units; u += unit_step, ++n_local) {
      const int split = u / tiles, tile = u - split * tiles;
      int tm, tn;
      gemm_decode_tile(p, tile, tm, tn, BM);
      const uint32_t buf = n_local & 1u;
      mbar_wait(&acc_full[buf], (n_local >> 1) & 1u);
      tc_fence_after_sync();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * kGBN;
      const int r0 = (int)rank * kGBM + quad * 32;
      if constexpr (OP == GEMM_BWD_DX) {
        gemm_epilogue_rows<GEMM_EPI_F32, false>(p, t_addr, tm * BM + r0, tn * kGBN, split, stage_patch, lane);
      } else {
        // rows of tensor t: partial rows [t * seg_len, (t + 1) * seg_len)
        const int t = tm / seg_blocks;
        GemmParams q = p;
        q.M = seg_len;
        q.part = p.part + (size_t)t * seg_len * p.N;
        gemm_epilogue_rows<GEMM_EPI_F32, false>(q, t_addr, (tm - t * seg_blocks) * BM + r0, tn * kGBN, split, stage_patch, lane);
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if constexpr (kPair) mbar_arrive_leader(&acc_empty[buf]);
        else mbar_arrive(&acc_empty[buf]);
      }
    }
  }
  tc_fence_before_sync();
  if constexpr (kPair) {
    cluster_sync_all();   // the peer may still be reading this CTA's B half / signalling its barriers
    if (warp == 1) tmem_dealloc_2cta(tmem_base, 512);
  } else {
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
  }
}

template <int OP>
__global__ void __launch_bounds__(kGThreads, 1)
gemm_bwd_kernel(const __grid_constant__ GemmBwdMaps maps, const GemmParams p, int seg_len, int seg_blocks) {
  gemm_bwd_body<OP, false>(maps, p, seg_len, seg_blocks);
}

template <int OP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGThreads, 1)
gemm2_bwd_kernel(const __grid_constant__ GemmBwdMaps maps, const GemmParams p, int seg_len, int seg_blocks) {
  gemm_bwd_body<OP, true>(maps, p, seg_len, seg_blocks);
}

// Split-K policy of the backward products: no partial longer than K3's 256 k blocks (the tensor core's truncating fp32
// adds bias longer chains), then the smallest split count whose work units fill the persistent grid's waves to >= 95%
// (each split keeping >= 4 k blocks, at most 16 splits beyond the minimum); the fullest of those if none reaches 95%.
static int gemm_bwd_splits(int64_t tiles, int kb_total, int units_per_wave) {
  constexpr int kMaxKbPerSplit = 256;
  const int min_s = (kb_total + kMaxKbPerSplit - 1) / kMaxKbPerSplit;
  int max_s = min_s + 16;
  if (max_s > kb_total / 4) max_s = kb_total / 4;
  if (max_s < min_s) max_s = min_s;
  int best_s = min_s;
  double best_eff = 0.0;
  for (int s = min_s; s <= max_s; ++s) {
    const int kps = (kb_total + s - 1) / s;
    const int real_s = (kb_total + kps - 1) / kps;
    const int64_t units = tiles * real_s;
    const int64_t waves = (units + units_per_wave - 1) / units_per_wave;
    const double eff = (double)units / (double)(waves * units_per_wave);
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best_s = real_s;
    }
    if (eff >= 0.95) break;
  }
  return best_s;
}

// Geometry of one backward product: M x N output, kb_total k blocks, tile and split counts for the chosen kernel
struct GemmBwdPlan {
  int pair;
  int tiles_m, tiles_n, kb_total, splits, kb_per_split;
  int seg_blocks;   // dX: k blocks per tensor; dW: M tiles per tensor
};

// n_seg tensors of seg_len columns; rows of the projection input; c_in its channels.  pair: -1 automatic, else 0 / 1.
static GemmBwdPlan gemm_bwd_plan(int op, int64_t rows, int64_t c_in, int n_seg, int64_t seg_len, int pair) {
  GemmBwdPlan g;
  const int64_t M = op == GEMM_BWD_DX ? rows : (int64_t)n_seg * seg_len;
  const int64_t seg_kb = (seg_len + kGBK - 1) / kGBK;
  const int64_t kb = op == GEMM_BWD_DX ? n_seg * seg_kb : (rows + kGBK - 1) / kGBK;
  g.pair = pair >= 0 ? pair : gemm_use_pair(M, c_in, 1, -1) ? 1 : 0;
  const int bm = g.pair ? kG2BM : kGBM;
  g.seg_blocks = op == GEMM_BWD_DX ? (int)seg_kb : (int)((seg_len + bm - 1) / bm);
  g.tiles_m = op == GEMM_BWD_DX ? (int)((rows + bm - 1) / bm) : n_seg * g.seg_blocks;
  g.tiles_n = (int)((c_in + kGBN - 1) / kGBN);
  g.kb_total = (int)kb;
  // the split count is planned on the pair kernel's 256 x 256 tiles and clusters whichever kernel runs, so that both give
  // the same partials and hence bitwise the same result
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  const int64_t tiles2 = (op == GEMM_BWD_DX ? (rows + kG2BM - 1) / kG2BM : n_seg * ((seg_len + kG2BM - 1) / kG2BM)) * g.tiles_n;
  g.splits = gemm_bwd_splits(tiles2, g.kb_total, sms / 2);
  g.kb_per_split = (g.kb_total + g.splits - 1) / g.splits;
  g.splits = (g.kb_total + g.kb_per_split - 1) / g.kb_per_split;
  return g;
}

// One backward product into fp32 partials part[split][M][N] (M = rows for dX, n_seg * seg_len for dW; N = c_in).
// dy[t]: [rows, seg_len] with row stride ld_dy[t]; w: [n_seg * seg_len, c_in] (ldw); x: [rows, c_in] (ldx).
template <int OP>
static int launch_gemm_bwd(const GemmBwdPlan& g, const void* const* dy, const int64_t* ld_dy, int n_seg, int64_t seg_len,
                           const void* w, int64_t ldw, const void* x, int64_t ldx, int64_t rows, int64_t c_in, int dtype,
                           float* part, cudaStream_t st) {
  GemmBwdMaps maps;
  memset(&maps, 0, sizeof(maps));
  int rc;
  for (int t = 0; t < n_seg; ++t) {
    uint64_t dims[2] = {(uint64_t)seg_len, (uint64_t)rows};
    uint64_t str[1] = {(uint64_t)ld_dy[t] * 2};
    // dX: K-major boxes of 64 k x 128 rows; dW: MN-major boxes of 64 (MN) x 64 k
    uint32_t box[2] = {(uint32_t)kGBK, OP == GEMM_BWD_DX ? (uint32_t)kGBM : (uint32_t)kGBK};
    if ((rc = encode_tensor_map(&maps.a[t], dtype, 2, dy[t], dims, str, box, 128)) != DS_OK) return rc;
    if (OP == GEMM_BWD_DX) {
      uint64_t dw[2] = {(uint64_t)c_in, (uint64_t)seg_len};
      uint64_t sw[1] = {(uint64_t)ldw * 2};
      uint32_t bw[2] = {64u, (uint32_t)kGBK};
      const void* wt = static_cast<const uint16_t*>(w) + (size_t)t * seg_len * ldw;
      if ((rc = encode_tensor_map(&maps.b[t], dtype, 2, wt, dw, sw, bw, 128)) != DS_OK) return rc;
    }
  }
  if (OP == GEMM_BWD_DW) {
    uint64_t dx[2] = {(uint64_t)c_in, (uint64_t)rows};
    uint64_t sx[1] = {(uint64_t)ldx * 2};
    uint32_t bx[2] = {64u, (uint32_t)kGBK};
    if ((rc = encode_tensor_map(&maps.b[0], dtype, 2, x, dx, sx, bx, 128)) != DS_OK) return rc;
  }
  for (int t = n_seg; t < 3; ++t) {   // unused slots repeat a valid map (prefetched, never loaded)
    maps.a[t] = maps.a[0];
    maps.b[t] = maps.b[0];
  }
  if (OP == GEMM_BWD_DW)
    for (int t = 1; t < 3; ++t) maps.b[t] = maps.b[0];
  GemmParams p = {};
  p.M = (int)(OP == GEMM_BWD_DX ? rows : n_seg * seg_len);
  p.N = (int)c_in;
  p.tiles_m = g.tiles_m;
  p.tiles_n = g.tiles_n;
  p.kb_total = g.kb_total;
  p.splits = g.splits;
  p.kb_per_split = g.kb_per_split;
  p.tiles_used = g.tiles_m * g.tiles_n;
  p.part = part;
  p.part_split_stride = (int64_t)p.M * p.N;
  const uint32_t fmt = dtype == DS_BF16 ? 1u : 0u, a_mn = OP == GEMM_BWD_DX ? 0u : 1u;
  const int64_t units = (int64_t)p.tiles_used * p.splits;
  if (units <= 0) return DS_OK;
  if (units > INT32_MAX) return fail(DS_ERR_INVALID, "gemm: too many work units");
  if (g.pair) {
    p.idesc2 = umma_idesc_f16(fmt, kG2BM, kGBN, a_mn, 1);
    int clusters = sm_count() / 2;
    if (units < clusters) clusters = (int)units;
    DS_CUDA_TRY(cudaFuncSetAttribute(gemm2_bwd_kernel<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kG2SmemBytes));
    gemm2_bwd_kernel<OP><<<2 * clusters, kGThreads, kG2SmemBytes, st>>>(maps, p, (int)seg_len, g.seg_blocks);
  } else {
    p.idesc = umma_idesc_f16(fmt, kGBM, kGBN, a_mn, 1);
    int grid = sm_count();
    if (units < grid) grid = (int)units;
    DS_CUDA_TRY(cudaFuncSetAttribute(gemm_bwd_kernel<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGSmemBytes));
    gemm_bwd_kernel<OP><<<grid, kGThreads, kGSmemBytes, st>>>(maps, p, (int)seg_len, g.seg_blocks);
  }
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

}  // namespace ds
