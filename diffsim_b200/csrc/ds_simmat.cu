// K3 -- N x N similarity matrix of flat feature vectors (tensor-core bound).
//
//   C[r,c] = sim(rows[r,:], cols[c,:])
//
// One tcgen05 GEMM rows x cols^T (the persistent 128x256 core of ds_gemm.cuh: K-major
// 128B-swizzled TMA tiles, double-buffered fp32 accumulators in TMEM), split along L
// so that the work units fill whole waves of the 148 SMs; per-vector statistics (sum, sum of squares, min, max)
// come from one HBM pass; a finishing kernel adds the split partials in a fixed
// order and applies the cosine / min-max-cosine normalisation.
//
// All-pairs form of the flat-cosine metrics: metrics/diffeats.py:202-205,
// metrics/clip_i.py:183, metrics/dino.py:183, metrics/vgg_gram.py:81.
// Algorithmic work: 2 * Nr * Nc * L flops.
#include "ds_gemm.cuh"

#include <float.h>

#include <type_traits>

namespace ds {

// ---------------------------------------------------------------------------
// per-vector statistics: sum, sum of squares, min, max (one HBM pass)
// ---------------------------------------------------------------------------
constexpr int kStatThreads = 256;
constexpr int kStatMaxChunks = 64;

// With `blocked` (may be null) the pass also writes the k-blocked copy the CTA-pair GEMM reads: element (row, e) goes to
// blocked[((e / 64) * rows_pad + row) * 64 + e % 64], the tail of the last k block is zero-filled (rows >= n of a block are
// never written: they only feed output rows the GEMM epilogue drops).  chunk_elems is a multiple of 64.
template <typename T>
__global__ void __launch_bounds__(kStatThreads)
row_stats_kernel(const T* __restrict__ x, int64_t ld, int64_t L, int chunks, int64_t chunk_elems,
                 float* __restrict__ partials /* [n][chunks][4] */, T* __restrict__ blocked, int64_t rows_pad) {
  const int64_t row = blockIdx.x / chunks;
  const int chunk = blockIdx.x % chunks;
  const T* xp = x + row * ld;
  const int64_t e0 = (int64_t)chunk * chunk_elems;
  const int64_t e1 = min(L, e0 + chunk_elems);
  float s = 0.f, ss = 0.f, mn = FLT_MAX, mx = -FLT_MAX;
  const int64_t nvec = (e1 > e0) ? (e1 - e0) / 8 : 0;
  const uint4* xv = reinterpret_cast<const uint4*>(xp + e0);
  auto blk = [&](int64_t e) -> T* { return blocked + (((e >> 6) * rows_pad + row) << 6) + (e & 63); };
  for (int64_t i = threadIdx.x; i < nvec; i += kStatThreads) {
    uint4 u = __ldg(xv + i);
    if (blocked) *reinterpret_cast<uint4*>(blk(e0 + i * 8)) = u;
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 f;
      if constexpr (sizeof(T) == 2 && std::is_same<T, __nv_bfloat16>::value) f = unpack2<true>(w[k]);
      else f = unpack2<false>(w[k]);
      s += f.x + f.y;
      ss = fmaf(f.x, f.x, ss);
      ss = fmaf(f.y, f.y, ss);
      mn = fminf(mn, fminf(f.x, f.y));
      mx = fmaxf(mx, fmaxf(f.x, f.y));
    }
  }
  if (blocked && e1 == L) {   // the chunk that holds the end of the row: zero the rest of the last k block
    const int64_t pad_end = (L + 63) & ~(int64_t)63;
    for (int64_t e = L + threadIdx.x; e < pad_end; e += kStatThreads) *blk(e) = T(0.f);
  }
  for (int64_t e = e0 + nvec * 8 + threadIdx.x; e < e1; e += kStatThreads) {
    if (blocked) *blk(e) = xp[e];
    float f;
    if constexpr (std::is_same<T, __nv_bfloat16>::value) f = __bfloat162float(xp[e]);
    else f = __half2float(xp[e]);
    s += f;
    ss = fmaf(f, f, ss);
    mn = fminf(mn, f);
    mx = fmaxf(mx, f);
  }
  __shared__ float sred[kStatThreads / 32][4];
  s = warp_sum(s);
  ss = warp_sum(ss);
  mn = warp_min(mn);
  mx = warp_max(mx);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sred[warp][0] = s;
    sred[warp][1] = ss;
    sred[warp][2] = mn;
    sred[warp][3] = mx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kStatThreads / 32; ++w) {
      s += sred[w][0];
      ss += sred[w][1];
      mn = fminf(mn, sred[w][2]);
      mx = fmaxf(mx, sred[w][3]);
    }
    float* dst = partials + ((size_t)row * chunks + chunk) * 4;
    dst[0] = s;
    dst[1] = ss;
    dst[2] = mn;
    dst[3] = mx;
  }
}

// stats[n][4] (double): sum, sumsq, min, max -- chunk partials added in chunk order
__global__ void row_stats_finish_kernel(const float* __restrict__ partials, int chunks, int64_t n,
                                        double* __restrict__ stats) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float* p = partials + (size_t)r * chunks * 4;
  double s = 0.0, ss = 0.0;
  float mn = FLT_MAX, mx = -FLT_MAX;
  for (int c = 0; c < chunks; ++c) {
    s += (double)p[c * 4 + 0];
    ss += (double)p[c * 4 + 1];
    mn = fminf(mn, p[c * 4 + 2]);
    mx = fmaxf(mx, p[c * 4 + 3]);
  }
  stats[r * 4 + 0] = s;
  stats[r * 4 + 1] = ss;
  stats[r * 4 + 2] = (double)mn;
  stats[r * 4 + 3] = (double)mx;
}

__global__ void simmat_finish_kernel(const float* __restrict__ part, int splits, int64_t part_split_stride,
                                     int64_t n_rows, int64_t n_cols, const double* __restrict__ rstats,
                                     const double* __restrict__ cstats, double L, int mode, float* __restrict__ C,
                                     int64_t ldc, int sym) {
  const int64_t col_blocks = (n_cols + blockDim.x - 1) / blockDim.x;
  const int64_t r = blockIdx.x / col_blocks;
  const int64_t c = (blockIdx.x % col_blocks) * (int64_t)blockDim.x + threadIdx.x;
  if (c >= n_cols || r >= n_rows) return;
  // symmetric mode: only the tiles on / above the diagonal hold partials.  The thread of (r, c), c >= r, reads them
  // (coalesced along c) and writes both C[r][c] and its mirror image; the threads below the diagonal have nothing to do
  if (sym && c < r) return;
  double acc = 0.0;
  const size_t e = (size_t)r * n_cols + c;
  for (int z = 0; z < splits; ++z) acc += (double)part[(size_t)z * part_split_stride + e];
  const double* rs = rstats + r * 4;
  const double* cs = cstats + c * 4;
  double out;
  if (mode == DS_SIM_COSINE) {
    double nx = fmax(sqrt(rs[1]), 1e-8), ny = fmax(sqrt(cs[1]), 1e-8);
    out = acc / (nx * ny);
  } else {
    double ax = rs[2], cx = rs[3] - rs[2], ay = cs[2], cy = cs[3] - cs[2];
    double dot = (acc - ay * rs[0] - ax * cs[0] + L * ax * ay) / (cx * cy);
    double xx = (rs[1] - 2.0 * ax * rs[0] + L * ax * ax) / (cx * cx);
    double yy = (cs[1] - 2.0 * ay * cs[0] + L * ay * ay) / (cy * cy);
    double nx = fmax(sqrt(fmax(xx, 0.0)), 1e-8), ny = fmax(sqrt(fmax(yy, 0.0)), 1e-8);
    out = dot / (nx * ny);
  }
  C[(size_t)r * ldc + c] = (float)out;
  if (sym && c != r) C[(size_t)c * ldc + r] = (float)out;
}

static int g_simmat_blocked = -1;   // ds_debug_set_simmat_blocked: -1 automatic, 0 never, 1 whenever the pair kernel runs

struct SimmatPlan {
  int tiles_m, tiles_n, kb_total, splits, kb_per_split;
  int pair;   // 1: CTA-pair kernel (256 x 256 tiles, 74 clusters)
  int stat_chunks;
  int64_t stat_chunk_elems;
  int blocked;   // 1: the statistics pass also writes k-blocked operand copies and the GEMM reads those
  int64_t rows_pad, cols_pad, kb64;   // extents of the k-blocked copies
};

static SimmatPlan simmat_plan(int64_t n_rows, int64_t n_cols, int64_t L, bool sym = false) {
  SimmatPlan p;
  // CTA pairs when both extents are at least two 256-wide tiles (else the 128-row tiles waste less)
  p.pair = (g_gemm_variant == 2 || (g_gemm_variant != 0 && n_rows >= 2 * kG2BM && n_cols >= 2 * kGBN)) ? 1 : 0;
  const int bm = p.pair ? kG2BM : kGBM;
  p.tiles_m = (int)((n_rows + bm - 1) / bm);
  p.tiles_n = (int)((n_cols + kGBN - 1) / kGBN);
  p.kb_total = (int)((L + kGBK - 1) / kGBK);
  // split along L: the smallest split count whose work units (tiles x splits) fill whole waves of the persistent grid
  // to >= 95% (at least 8 k blocks per unit, at most 64 splits: the fp32 partials cost HBM traffic)
  const int64_t tiles = sym ? gemm_sym_tile_count(p.tiles_m, p.tiles_n, bm) : (int64_t)p.tiles_m * p.tiles_n;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  if (p.pair) sms /= 2;   // work units are dealt to clusters
  // accuracy: the tensor core adds each K = 16 MMA into the fp32 accumulator with truncation, a bias that grows with the
  // length of the chain (measured on 655 360-long unit-cosine rows: 2.1e-3 at 20 480 MMAs per partial, 5e-4 at 1 100);
  // a partial therefore never covers more than kMaxKbPerSplit k blocks (1024 MMAs); the partials are added in double
  constexpr int kMaxKbPerSplit = 256;
  const int min_s = (p.kb_total + kMaxKbPerSplit - 1) / kMaxKbPerSplit;
  int max_s = p.kb_total / 8;
  if (max_s > 64) max_s = 64;
  if (max_s < min_s + 8) max_s = min_s + 8;
  if (max_s > p.kb_total) max_s = p.kb_total;
  if (max_s < 1) max_s = 1;
  int best_s = min_s;
  double best_eff = 0.0;
  for (int s = min_s; s <= max_s; ++s) {
    const int kps = (p.kb_total + s - 1) / s;
    const int real_s = (p.kb_total + kps - 1) / kps;
    const int64_t units = tiles * real_s;
    const int64_t waves = (units + sms - 1) / sms;
    const double eff = (double)units / (double)(waves * sms);
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best_s = real_s;
    }
    if (eff >= 0.95) break;
  }
  p.kb_per_split = (p.kb_total + best_s - 1) / best_s;
  p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  // k-blocked operand copies: worth their extra HBM pass when an operand is far larger than the L2 -- the row-major TMA
  // boxes (256 row pieces, 2 * ld bytes apart) then miss the L2 on 55% of the requests although the tiles that share a
  // row block run at the same time; measured (profiles/r2_simmat_experiments.txt): 2032 x 655 360 (2.7 GB) 3.9 -> 3.35 ms,
  // 2032 x 163 840 (0.67 GB) 0.68 -> 0.79 ms.  Writing the copy in stages UNDER the GEMM of the previous stage is slower than
  // back to back (3.8 ms: the copy's stream of writes evicts the GEMM's L2 working set)
  p.rows_pad = (n_rows + 255) / 256 * 256;
  p.cols_pad = (n_cols + 255) / 256 * 256;
  p.kb64 = (L + 63) / 64;
  const bool big = (double)(n_rows > n_cols ? n_rows : n_cols) * (double)L * 2.0 >= 1536.0 * 1024 * 1024;
  p.blocked = (p.pair && g_simmat_blocked != 0 && (big || g_simmat_blocked > 0)) ? 1 : 0;
  if (p.kb64 * (p.rows_pad > p.cols_pad ? p.rows_pad : p.cols_pad) > (int64_t)INT32_MAX) p.blocked = 0;
  const int64_t quantum = 8 * kStatThreads;
  int64_t c = (L + 65535) / 65536;
  if (c > kStatMaxChunks) c = kStatMaxChunks;
  if (c < 1) c = 1;
  int64_t ce = (L + c - 1) / c;
  ce = (ce + quantum - 1) / quantum * quantum;
  p.stat_chunk_elems = ce;
  p.stat_chunks = (int)((L + ce - 1) / ce);
  return p;
}

}  // namespace ds

extern "C" {

int ds_debug_set_simmat_blocked(int mode) {
  if (mode >= -1 && mode <= 1) ds::g_simmat_blocked = mode;
  return ds::g_simmat_blocked;
}

size_t ds_simmat_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t L) {
  using namespace ds;
  if (n_rows <= 0 || n_cols <= 0 || L <= 0) return 256;
  SimmatPlan p = simmat_plan(n_rows, n_cols, L);
  if (n_rows == n_cols) {   // the self-similarity call may take the symmetric plan: size for the larger of the two
    SimmatPlan ps = simmat_plan(n_rows, n_cols, L, true);
    if (ps.splits > p.splits) p.splits = ps.splits;
  }
  size_t b = 0;
  b += align_up((size_t)p.splits * n_rows * n_cols * sizeof(float), 256);
  b += align_up((size_t)(n_rows + n_cols) * p.stat_chunks * 4 * sizeof(float), 256);
  b += align_up((size_t)(n_rows + n_cols) * 4 * sizeof(double), 256);
  if (p.blocked) b += align_up((size_t)p.kb64 * (p.rows_pad + p.cols_pad) * 64 * 2, 256) + 256;
  return b + 1024;
}

int ds_simmat(const void* rows, int64_t n_rows, int64_t ld_rows, const void* cols, int64_t n_cols, int64_t ld_cols,
              int64_t L, int dtype, int mode, float* C, int64_t ldc, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_rows < 0 || n_cols < 0 || L <= 0) return fail(DS_ERR_INVALID, "ds_simmat: bad sizes");
  if (n_rows == 0 || n_cols == 0) return DS_OK;
  if (!rows || !cols || !C) return fail(DS_ERR_INVALID, "ds_simmat: null pointer");
  if (dtype != DS_F16 && dtype != DS_BF16) return fail(DS_ERR_UNSUPPORTED, "ds_simmat: dtype must be f16 or bf16");
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MINMAX_COSINE) return fail(DS_ERR_INVALID, "ds_simmat: bad mode %d", mode);
  if (ld_rows < L || ld_cols < L || (ld_rows & 7) || (ld_cols & 7))
    return fail(DS_ERR_INVALID, "ds_simmat: leading dimensions must be >= L and multiples of 8 elements");
  if (((uintptr_t)rows & 15) || ((uintptr_t)cols & 15)) return fail(DS_ERR_INVALID, "ds_simmat: base pointers must be 16-byte aligned");
  if (ldc < n_cols) return fail(DS_ERR_INVALID, "ds_simmat: ldc < n_cols");
  if (n_rows > INT32_MAX || n_cols > INT32_MAX || L > (int64_t)INT32_MAX * 32) return fail(DS_ERR_INVALID, "ds_simmat: sizes too large");
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;

  // self-similarity (the retrieval case): C is symmetric -- compute the upper triangle of tiles only, one statistics pass
  const bool sym = rows == cols && n_rows == n_cols && ld_rows == ld_cols;
  SimmatPlan p = simmat_plan(n_rows, n_cols, L, sym);
  Workspace w(ws, ws_bytes);
  float* part = static_cast<float*>(w.take((size_t)p.splits * n_rows * n_cols * sizeof(float)));
  float* spart = static_cast<float*>(w.take((size_t)(n_rows + n_cols) * p.stat_chunks * 4 * sizeof(float)));
  double* stats = static_cast<double*>(w.take((size_t)(n_rows + n_cols) * 4 * sizeof(double)));
  void* blk_r = nullptr;
  void* blk_c = nullptr;
  if (p.blocked) {
    blk_r = w.take((size_t)p.kb64 * p.rows_pad * 64 * 2);
    blk_c = sym ? blk_r : w.take((size_t)p.kb64 * p.cols_pad * 64 * 2);
  }
  if (!part || !spart || !stats || (p.blocked && (!blk_r || !blk_c)))
    return fail(DS_ERR_WORKSPACE, "ds_simmat: workspace too small (%zu given, need %zu)", ws_bytes,
                ds_simmat_workspace_bytes(n_rows, n_cols, L));
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  // statistics pass (+ the k-blocked copies)
  float* spart_c = spart + (size_t)n_rows * p.stat_chunks * 4;
  double* stats_c = sym ? stats : stats + (size_t)n_rows * 4;
  if (dtype == DS_F16) {
    row_stats_kernel<__half><<<(unsigned)(n_rows * p.stat_chunks), kStatThreads, 0, st>>>(
        static_cast<const __half*>(rows), ld_rows, L, p.stat_chunks, p.stat_chunk_elems, spart, static_cast<__half*>(blk_r),
        p.rows_pad);
    if (!sym)
      row_stats_kernel<__half><<<(unsigned)(n_cols * p.stat_chunks), kStatThreads, 0, st>>>(
          static_cast<const __half*>(cols), ld_cols, L, p.stat_chunks, p.stat_chunk_elems, spart_c, static_cast<__half*>(blk_c),
          p.cols_pad);
  } else {
    row_stats_kernel<__nv_bfloat16><<<(unsigned)(n_rows * p.stat_chunks), kStatThreads, 0, st>>>(
        static_cast<const __nv_bfloat16*>(rows), ld_rows, L, p.stat_chunks, p.stat_chunk_elems, spart,
        static_cast<__nv_bfloat16*>(blk_r), p.rows_pad);
    if (!sym)
      row_stats_kernel<__nv_bfloat16><<<(unsigned)(n_cols * p.stat_chunks), kStatThreads, 0, st>>>(
          static_cast<const __nv_bfloat16*>(cols), ld_cols, L, p.stat_chunks, p.stat_chunk_elems, spart_c,
          static_cast<__nv_bfloat16*>(blk_c), p.cols_pad);
  }
  DS_CUDA_TRY(cudaGetLastError());
  row_stats_finish_kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, st>>>(spart, p.stat_chunks, n_rows, stats);
  if (!sym) row_stats_finish_kernel<<<(unsigned)((n_cols + 127) / 128), 128, 0, st>>>(spart_c, p.stat_chunks, n_cols, stats_c);
  DS_CUDA_TRY(cudaGetLastError());

  // GEMM: fp32 partials part[split][row][col]
  GemmParams gp = {};
  gp.splits = p.splits;
  gp.sym = sym ? 1 : 0;
  gp.use_pair = p.pair;
  gp.part = part;
  gp.part_split_stride = (int64_t)n_rows * n_cols;
  if (p.blocked) {
    gp.kblk_rows_a = (int)p.rows_pad;
    gp.kblk_rows_b = (int)p.cols_pad;
    rc = launch_gemm_tn<GEMM_EPI_F32>(blk_r, n_rows, 64, blk_c, n_cols, 64, L, dtype, gp, st);
  } else {
    rc = launch_gemm_tn<GEMM_EPI_F32>(rows, n_rows, ld_rows, cols, n_cols, ld_cols, L, dtype, gp, st);
  }
  if (rc != DS_OK) return rc;

  const int64_t fblocks = ((n_cols + 255) / 256) * n_rows;
  if (fblocks > 0x7fffffffLL) return fail(DS_ERR_INVALID, "ds_simmat: matrix too large");
  simmat_finish_kernel<<<(unsigned)fblocks, 256, 0, st>>>(part, p.splits, (int64_t)n_rows * n_cols, n_rows, n_cols, stats, stats_c,
                                            (double)L, mode, C, ldc, sym ? 1 : 0);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
