// K2 -- batched similarity reductions (HBM-bound).
//
// One pass over x and y with 128-bit loads, fp32 accumulation, warp-shuffle +
// shared-memory block reduction, and a deterministic "last CTA finishes" second
// stage (fixed summation order, no float atomics).
//
// Replaces F.cosine_similarity / F.mse_loss on flattened tensors
// (diffsim/diffsim.py:182-197) and min_max_normalize + cosine
// (metrics/diffeats.py:136-140,202-205).  Algorithmic bytes per row pair:
// 2 * E * sizeof(dtype) read + 4 written.
#include "ds_host.h"
#include "ds_ptx.cuh"

#include <float.h>

namespace ds {

constexpr int kRedThreads = 256;
constexpr int kRedUnroll = 4;
constexpr int kRedMaxChunks = 64;
constexpr int kRedSlots = 12;  // floats per partial record

template <typename T>
struct Vec16;
template <>
struct Vec16<__half> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void cvt(const uint4& u, float (&f)[8]) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 t = __half22float2(h[i]);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
  static __device__ __forceinline__ float one(const __half* p) { return __half2float(*p); }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void cvt(const uint4& u, float (&f)[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 t = __bfloat1622float2(h[i]);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
  static __device__ __forceinline__ float one(const __nv_bfloat16* p) { return __bfloat162float(*p); }
};
template <>
struct Vec16<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void cvt(const uint4& u, float (&f)[4]) {
    f[0] = __uint_as_float(u.x);
    f[1] = __uint_as_float(u.y);
    f[2] = __uint_as_float(u.z);
    f[3] = __uint_as_float(u.w);
  }
  static __device__ __forceinline__ float one(const float* p) { return *p; }
};

// streaming 128-bit load: read once, do not pollute L1
__device__ __forceinline__ uint4 ld_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// (value, count) of a running minimum or maximum: ties are counted so that the backward can split the gradient of
// t.min() / t.max() evenly among them, as torch does.  Merging is exact, so the count does not depend on the order.
template <bool kMax>
__device__ __forceinline__ void tie_merge(float& v, unsigned& n, float a, unsigned na) {
  if (kMax ? a > v : a < v) {
    v = a;
    n = na;
  } else if (a == v) {
    n += na;
  }
}

template <bool kMax>
__device__ __forceinline__ void warp_tie(float& v, unsigned& n) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const unsigned on = __shfl_xor_sync(0xffffffffu, n, o);
    tie_merge<kMax>(v, n, ov, on);
  }
}

// kTies: also count the elements equal to each min / max (the backward's statistics pass; min-max mode only)
template <int MODE, bool kTies = false>
struct Acc {
  // COSINE: dot, xx, yy.  MSE: sq.  MINMAX: dot, xx, yy, sx, sy, mnx, mxx, mny, mxy
  float dot = 0.f, xx = 0.f, yy = 0.f, sx = 0.f, sy = 0.f, sq = 0.f;
  float mnx = FLT_MAX, mxx = -FLT_MAX, mny = FLT_MAX, mxy = -FLT_MAX;
  unsigned nmnx = 0, nmxx = 0, nmny = 0, nmxy = 0;
  __device__ __forceinline__ void add(float a, float b) {
    if constexpr (MODE == DS_SIM_MSE) {
      float d = a - b;
      sq = fmaf(d, d, sq);
    } else {
      dot = fmaf(a, b, dot);
      xx = fmaf(a, a, xx);
      yy = fmaf(b, b, yy);
      if constexpr (MODE == DS_SIM_MINMAX_COSINE) {
        sx += a;
        sy += b;
        if constexpr (kTies) {
          tie_merge<false>(mnx, nmnx, a, 1u);
          tie_merge<true>(mxx, nmxx, a, 1u);
          tie_merge<false>(mny, nmny, b, 1u);
          tie_merge<true>(mxy, nmxy, b, 1u);
        } else {
          mnx = fminf(mnx, a);
          mxx = fmaxf(mxx, a);
          mny = fminf(mny, b);
          mxy = fmaxf(mxy, b);
        }
      }
    }
  }
};

// Final similarity from the summed statistics (double: the min-max form cancels).
template <int MODE>
__device__ float finish_stats(const float* s, double E) {
  if constexpr (MODE == DS_SIM_MSE) {
    return (float)((double)s[5] / E);
  } else if constexpr (MODE == DS_SIM_COSINE) {
    double nx = fmax(sqrt((double)s[1]), 1e-8), ny = fmax(sqrt((double)s[2]), 1e-8);
    return (float)((double)s[0] / (nx * ny));
  } else {
    // x' = (x - ax)/cx, y' = (y - ay)/cy   (metrics/diffeats.py:136-140)
    double ax = s[6], cx = (double)s[7] - (double)s[6];
    double ay = s[8], cy = (double)s[9] - (double)s[8];
    double dot = ((double)s[0] - ay * (double)s[3] - ax * (double)s[4] + E * ax * ay) / (cx * cy);
    double xx = ((double)s[1] - 2.0 * ax * (double)s[3] + E * ax * ax) / (cx * cx);
    double yy = ((double)s[2] - 2.0 * ay * (double)s[4] + E * ay * ay) / (cy * cy);
    double nx = fmax(sqrt(fmax(xx, 0.0)), 1e-8), ny = fmax(sqrt(fmax(yy, 0.0)), 1e-8);
    return (float)(dot / (nx * ny));
  }
}

// Backward statistics pass (ds_pair_reduce_bwd): pair_reduce_kernel<T, mode | kBwdStats> is the forward's reduction
// (same body and plan, so the statistics, and s, are bitwise the forward's) plus the min / max tie counts; its last CTA
// of a row reads g = out[p] (d_out) and overwrites the row's first partial record with the gradient pass's coefficients.
constexpr int kBwdStats = 8;
constexpr int kRedTieSlots = 16;  // floats per partial record of the statistics pass: Acc's 10, then 4 tie counts

template <int MODE>
__device__ __forceinline__ void bwd_coefficients(const float* s, const unsigned* n, double E, double g, float* rec);

template <typename T, int MODE>
__global__ void __launch_bounds__(kRedThreads)
pair_reduce_kernel(const T* __restrict__ x, const T* __restrict__ y, int64_t E, int64_t xs, int64_t ys,
                   int chunks, int64_t chunk_elems, int vec_ok, float* __restrict__ partials,
                   unsigned int* __restrict__ counters, float* __restrict__ out) {
  constexpr int VN = Vec16<T>::N;
  constexpr int SIM = MODE & ~kBwdStats;
  constexpr bool kBwd = (MODE & kBwdStats) != 0;
  constexpr bool kTies = kBwd && SIM == DS_SIM_MINMAX_COSINE;
  constexpr int kSlots = kBwd ? kRedTieSlots : kRedSlots;
  const int64_t pair = blockIdx.x / chunks;
  const int chunk = blockIdx.x % chunks;
  const T* xp = x + pair * xs;
  const T* yp = y + pair * ys;
  const int64_t e0 = (int64_t)chunk * chunk_elems;
  const int64_t e1 = min(E, e0 + chunk_elems);

  Acc<SIM, kTies> acc;
  // vector body: chunk_elems is a multiple of VN * threads * unroll, so e0 keeps the rows' 16-byte alignment;
  // rows that are not 16-byte aligned (vec_ok == 0) take the element-wise loop below for everything
  const int64_t nvec = (vec_ok && e1 > e0) ? (e1 - e0) / VN : 0;
  const uint4* xv = reinterpret_cast<const uint4*>(xp + e0);
  const uint4* yv = reinterpret_cast<const uint4*>(yp + e0);
  int64_t i = threadIdx.x;
  for (; i + (kRedUnroll - 1) * kRedThreads < nvec; i += kRedUnroll * kRedThreads) {
    uint4 a[kRedUnroll], b[kRedUnroll];
#pragma unroll
    for (int u = 0; u < kRedUnroll; ++u) {
      a[u] = ld_stream(xv + i + u * kRedThreads);
      b[u] = ld_stream(yv + i + u * kRedThreads);
    }
#pragma unroll
    for (int u = 0; u < kRedUnroll; ++u) {
      float fa[VN], fb[VN];
      Vec16<T>::cvt(a[u], fa);
      Vec16<T>::cvt(b[u], fb);
#pragma unroll
      for (int k = 0; k < VN; ++k) acc.add(fa[k], fb[k]);
    }
  }
  for (; i < nvec; i += kRedThreads) {
    float fa[VN], fb[VN];
    Vec16<T>::cvt(ld_stream(xv + i), fa);
    Vec16<T>::cvt(ld_stream(yv + i), fb);
#pragma unroll
    for (int k = 0; k < VN; ++k) acc.add(fa[k], fb[k]);
  }
  // scalar tail (only the last chunk can have one)
  for (int64_t e = e0 + nvec * VN + threadIdx.x; e < e1; e += kRedThreads)
    acc.add(Vec16<T>::one(xp + e), Vec16<T>::one(yp + e));

  // block reduction: shuffle inside the warp, shared memory across warps
  __shared__ float sred[kRedThreads / 32][kSlots];
  __shared__ bool is_last;
  float v[10] = {acc.dot, acc.xx, acc.yy, acc.sx, acc.sy, acc.sq, acc.mnx, acc.mxx, acc.mny, acc.mxy};
  unsigned n[4] = {acc.nmnx, acc.nmxx, acc.nmny, acc.nmxy};
#pragma unroll
  for (int k = 0; k < 6; ++k) v[k] = warp_sum(v[k]);
  if constexpr (kTies) {
    warp_tie<false>(v[6], n[0]);
    warp_tie<true>(v[7], n[1]);
    warp_tie<false>(v[8], n[2]);
    warp_tie<true>(v[9], n[3]);
  } else if constexpr (SIM == DS_SIM_MINMAX_COSINE) {
    v[6] = warp_min(v[6]);
    v[7] = warp_max(v[7]);
    v[8] = warp_min(v[8]);
    v[9] = warp_max(v[9]);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 10; ++k) sred[warp][k] = v[k];
    if constexpr (kTies) {
#pragma unroll
      for (int k = 0; k < 4; ++k) sred[warp][10 + k] = __uint_as_float(n[k]);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float r[10];
    unsigned cnt[4];
#pragma unroll
    for (int k = 0; k < 10; ++k) r[k] = sred[0][k];
    if constexpr (kTies) {
#pragma unroll
      for (int k = 0; k < 4; ++k) cnt[k] = __float_as_uint(sred[0][10 + k]);
    }
    for (int w = 1; w < kRedThreads / 32; ++w) {
#pragma unroll
      for (int k = 0; k < 6; ++k) r[k] += sred[w][k];
      if constexpr (kTies) {
        tie_merge<false>(r[6], cnt[0], sred[w][6], __float_as_uint(sred[w][10]));
        tie_merge<true>(r[7], cnt[1], sred[w][7], __float_as_uint(sred[w][11]));
        tie_merge<false>(r[8], cnt[2], sred[w][8], __float_as_uint(sred[w][12]));
        tie_merge<true>(r[9], cnt[3], sred[w][9], __float_as_uint(sred[w][13]));
      } else {
        r[6] = fminf(r[6], sred[w][6]);
        r[7] = fmaxf(r[7], sred[w][7]);
        r[8] = fminf(r[8], sred[w][8]);
        r[9] = fmaxf(r[9], sred[w][9]);
      }
    }
    float* dst = partials + ((size_t)pair * chunks + chunk) * kSlots;
#pragma unroll
    for (int k = 0; k < 10; ++k) dst[k] = r[k];
    if constexpr (kTies) {
#pragma unroll
      for (int k = 0; k < 4; ++k) dst[10 + k] = __uint_as_float(cnt[k]);
    }
    __threadfence();
    unsigned int prev = atomicAdd(&counters[pair], 1u);
    is_last = (prev == (unsigned int)(chunks - 1));
  }
  __syncthreads();
  if (!is_last) return;
  // last CTA of this pair: sum the chunk partials in chunk order (deterministic)
  if (threadIdx.x == 0) {
    __threadfence();
    const volatile float* src = partials + (size_t)pair * chunks * kSlots;
    float r[10];
    unsigned cnt[4];
#pragma unroll
    for (int k = 0; k < 10; ++k) r[k] = src[k];
    if constexpr (kTies) {
#pragma unroll
      for (int k = 0; k < 4; ++k) cnt[k] = __float_as_uint(src[10 + k]);
    }
    for (int c = 1; c < chunks; ++c) {
      const volatile float* s = src + (size_t)c * kSlots;
#pragma unroll
      for (int k = 0; k < 6; ++k) r[k] += s[k];
      if constexpr (kTies) {
        tie_merge<false>(r[6], cnt[0], s[6], __float_as_uint(s[10]));
        tie_merge<true>(r[7], cnt[1], s[7], __float_as_uint(s[11]));
        tie_merge<false>(r[8], cnt[2], s[8], __float_as_uint(s[12]));
        tie_merge<true>(r[9], cnt[3], s[9], __float_as_uint(s[13]));
      } else {
        r[6] = fminf(r[6], s[6]);
        r[7] = fmaxf(r[7], s[7]);
        r[8] = fminf(r[8], s[8]);
        r[9] = fmaxf(r[9], s[9]);
      }
    }
    if constexpr (kBwd)
      bwd_coefficients<SIM>(r, cnt, (double)E, (double)out[pair], partials + (size_t)pair * chunks * kSlots);
    else
      out[pair] = finish_stats<MODE>(r, (double)E);
    counters[pair] = 0;  // leave the workspace reusable
  }
}

// ---- backward ----------------------------------------------------------------------------------------------------
//
// Per row, with g = d_out[p], the gradient pass writes
//   dx = ax (x - ox) + b (y - oy) + [x == mnx] tmnx + [x == mxx] tmxx
//   dy = ay (y - oy) + b (x - ox) + [y == mny] tmny + [y == mxy] tmxy
// from a record that the statistics pass leaves in the row's first partial slot (mse needs none:
// dx = 2 g (x - y) / E = -dy).
//   cosine: b = g / (nx ny), ax = -g s / (nx |x|) (0 when |x| = 0), ay likewise, n = max(|.|, 1e-8); o and the tie
//           terms are 0 and not stored
//   minmax: the cosine rule on x^ = (x - mnx) / cx, y^ = (y - mny) / cy (cx = mxx - mnx), with G = dcos/dx^ and
//           S_m = sum G (x^ - 1) / cx, S_M = -sum G x^ / cx split evenly among the elements equal to the min / max
//           (tmnx = g S_m / n_mnx, tmxx = g S_M / n_mxx); both sums follow from the row statistics.  A constant row
//           (cx or cy = 0) has a NaN score and gets NaN gradients, as in torch.
enum { kAx, kAy, kB, kOx, kOy, kMnx, kTmnx, kMxx, kTmxx, kMny, kTmny, kMxy, kTmxy };

// The row record in double (as finish_stats): s the row's statistics, n its tie counts, g = dL/d out[p].
template <int MODE>
__device__ __forceinline__ void bwd_coefficients(const float* s, const unsigned* n, double E, double g, float* rec) {
  if constexpr (MODE == DS_SIM_COSINE) {
    const double ex = sqrt((double)s[1]), ey = sqrt((double)s[2]);
    const double nx = fmax(ex, 1e-8), ny = fmax(ey, 1e-8);
    const double sim = (double)s[0] / (nx * ny);
    rec[kAx] = ex > 0.0 ? (float)(-g * sim / (nx * ex)) : 0.f;
    rec[kAy] = ey > 0.0 ? (float)(-g * sim / (ny * ey)) : 0.f;
    rec[kB] = (float)(g / (nx * ny));
  } else {
    const double mx = s[6], cx = (double)s[7] - (double)s[6];
    const double my = s[8], cy = (double)s[9] - (double)s[8];
    // sums over the normalised rows (as finish_stats)
    const double dot = ((double)s[0] - my * (double)s[3] - mx * (double)s[4] + E * mx * my) / (cx * cy);
    const double xx = fmax(((double)s[1] - 2.0 * mx * (double)s[3] + E * mx * mx) / (cx * cx), 0.0);
    const double yy = fmax(((double)s[2] - 2.0 * my * (double)s[4] + E * my * my) / (cy * cy), 0.0);
    const double sxh = ((double)s[3] - E * mx) / cx, syh = ((double)s[4] - E * my) / cy;
    const double ex = sqrt(xx), ey = sqrt(yy);
    const double nx = fmax(ex, 1e-8), ny = fmax(ey, 1e-8);
    const double sim = dot / (nx * ny);
    // G_x = axy y^ - axx x^,  G_y = axy x^ - ayy y^
    const double axy = 1.0 / (nx * ny);
    const double axx = ex > 0.0 ? sim / (nx * ex) : 0.0, ayy = ey > 0.0 ? sim / (ny * ey) : 0.0;
    const double gxx = axy * dot - axx * xx, gyy = axy * dot - ayy * yy;  // sum G_x x^, sum G_y y^
    const double gx = axy * syh - axx * sxh, gy = axy * sxh - ayy * syh;  // sum G_x, sum G_y
    const bool constant = cx == 0.0 || cy == 0.0;
    rec[kAx] = constant ? __int_as_float(0x7fc00000) : (float)(-g * axx / (cx * cx));
    rec[kAy] = constant ? __int_as_float(0x7fc00000) : (float)(-g * ayy / (cy * cy));
    rec[kB] = constant ? __int_as_float(0x7fc00000) : (float)(g * axy / (cx * cy));
    rec[kOx] = s[6];
    rec[kOy] = s[8];
    rec[kMnx] = s[6];
    rec[kMxx] = s[7];
    rec[kMny] = s[8];
    rec[kMxy] = s[9];
    rec[kTmnx] = (float)(g * (gxx - gx) / cx / (double)n[0]);
    rec[kTmxx] = (float)(-g * gxx / cx / (double)n[1]);
    rec[kTmny] = (float)(g * (gyy - gy) / cy / (double)n[2]);
    rec[kTmxy] = (float)(-g * gyy / cy / (double)n[3]);
  }
}

template <int MODE>
struct RowGrad {
  float ax, ay, b, ox, oy, mnx, tmnx, mxx, tmxx, mny, tmny, mxy, tmxy;
  __device__ __forceinline__ RowGrad(const float* __restrict__ r, const float* __restrict__ d_out, int64_t pair,
                                     int64_t E) {
    if constexpr (MODE == DS_SIM_MSE) {
      ax = ay = (float)(2.0 * (double)d_out[pair] / (double)E);
      b = -ax;
    } else {
      ax = r[kAx], ay = r[kAy], b = r[kB];
      if constexpr (MODE == DS_SIM_MINMAX_COSINE) {
        ox = r[kOx], oy = r[kOy];
        mnx = r[kMnx], tmnx = r[kTmnx], mxx = r[kMxx], tmxx = r[kTmxx];
        mny = r[kMny], tmny = r[kTmny], mxy = r[kMxy], tmxy = r[kTmxy];
      }
    }
  }
  __device__ __forceinline__ float dx(float a, float c) const {
    if constexpr (MODE == DS_SIM_MSE) return ax * (a - c);
    if constexpr (MODE == DS_SIM_COSINE) return fmaf(ax, a, b * c);
    float t = (a == mnx ? tmnx : 0.f) + (a == mxx ? tmxx : 0.f);
    return fmaf(ax, a - ox, fmaf(b, c - oy, t));
  }
  __device__ __forceinline__ float dy(float a, float c) const {
    if constexpr (MODE == DS_SIM_MSE) return b * (a - c);
    if constexpr (MODE == DS_SIM_COSINE) return fmaf(ay, c, b * a);
    float t = (c == mny ? tmny : 0.f) + (c == mxy ? tmxy : 0.f);
    return fmaf(ay, c - oy, fmaf(b, a - ox, t));
  }
};

template <int N>
__device__ __forceinline__ void st_stream(float* p, const float (&v)[N]) {
#pragma unroll
  for (int k = 0; k < N; k += 4) __stcs(reinterpret_cast<float4*>(p + k), make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]));
}

// Gradient pass: one elementwise sweep over x and y (the forward's loads and CTA plan), fp32 dx and dy written (either
// may be null).  vec_ok also requires 16-byte aligned output rows.
template <typename T, int MODE>
__global__ void __launch_bounds__(kRedThreads)
pair_reduce_grad_kernel(const T* __restrict__ x, const T* __restrict__ y, int64_t E, int64_t xs, int64_t ys, int chunks,
                        int64_t chunk_elems, int vec_ok, const float* __restrict__ partials,
                        const float* __restrict__ d_out, float* __restrict__ dx, int64_t dxs, float* __restrict__ dy,
                        int64_t dys) {
  constexpr int VN = Vec16<T>::N;
  const int64_t pair = blockIdx.x / chunks;
  const int chunk = blockIdx.x % chunks;
  const T* xp = x + pair * xs;
  const T* yp = y + pair * ys;
  float* dxp = dx ? dx + pair * dxs : nullptr;
  float* dyp = dy ? dy + pair * dys : nullptr;
  const int64_t e0 = (int64_t)chunk * chunk_elems;
  const int64_t e1 = min(E, e0 + chunk_elems);
  const RowGrad<MODE> rg(MODE == DS_SIM_MSE ? nullptr : partials + (size_t)pair * chunks * kRedTieSlots, d_out, pair, E);

  const int64_t nvec = (vec_ok && e1 > e0) ? (e1 - e0) / VN : 0;
  const uint4* xv = reinterpret_cast<const uint4*>(xp + e0);
  const uint4* yv = reinterpret_cast<const uint4*>(yp + e0);
  auto emit = [&](int64_t i, const uint4& ua, const uint4& ub) {
    float fa[VN], fb[VN], o[VN];
    Vec16<T>::cvt(ua, fa);
    Vec16<T>::cvt(ub, fb);
    if (dxp) {
#pragma unroll
      for (int k = 0; k < VN; ++k) o[k] = rg.dx(fa[k], fb[k]);
      st_stream(dxp + e0 + i * VN, o);
    }
    if (dyp) {
#pragma unroll
      for (int k = 0; k < VN; ++k) o[k] = rg.dy(fa[k], fb[k]);
      st_stream(dyp + e0 + i * VN, o);
    }
  };
  int64_t i = threadIdx.x;
  for (; i + (kRedUnroll - 1) * kRedThreads < nvec; i += kRedUnroll * kRedThreads) {
    uint4 a[kRedUnroll], b[kRedUnroll];
#pragma unroll
    for (int u = 0; u < kRedUnroll; ++u) {
      a[u] = ld_stream(xv + i + u * kRedThreads);
      b[u] = ld_stream(yv + i + u * kRedThreads);
    }
#pragma unroll
    for (int u = 0; u < kRedUnroll; ++u) emit(i + u * kRedThreads, a[u], b[u]);
  }
  for (; i < nvec; i += kRedThreads) emit(i, ld_stream(xv + i), ld_stream(yv + i));
  for (int64_t e = e0 + nvec * VN + threadIdx.x; e < e1; e += kRedThreads) {
    const float a = Vec16<T>::one(xp + e), c = Vec16<T>::one(yp + e);
    if (dxp) dxp[e] = rg.dx(a, c);
    if (dyp) dyp[e] = rg.dy(a, c);
  }
}

static void reduce_plan(int64_t n_pairs, int64_t E, int vn, int* chunks, int64_t* chunk_elems) {
  const int64_t quantum = (int64_t)vn * kRedThreads * kRedUnroll;  // elements one CTA sweep covers
  int64_t max_chunks = (E + quantum - 1) / quantum;
  if (max_chunks < 1) max_chunks = 1;
  int64_t want = (2 * 148 + n_pairs - 1) / n_pairs;        // at least two CTAs per SM overall
  int64_t by_size = (E + 131071) / 131072;                 // at most 128 Ki elements per CTA
  int64_t c = want > by_size ? want : by_size;
  if (c > max_chunks) c = max_chunks;
  if (c > kRedMaxChunks) c = kRedMaxChunks;
  if (c < 1) c = 1;
  int64_t ce = (E + c - 1) / c;
  ce = (ce + quantum - 1) / quantum * quantum;
  c = (E + ce - 1) / ce;
  if (c < 1) c = 1;
  *chunks = (int)c;
  *chunk_elems = ce;
}

template <typename T>
static int launch_reduce(const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t xs, int64_t ys,
                         int mode, float* out, float* partials, unsigned int* counters, int chunks,
                         int64_t chunk_elems, int vec_ok, cudaStream_t st) {
  const T* xp = static_cast<const T*>(x);
  const T* yp = static_cast<const T*>(y);
  int64_t blocks = n_pairs * chunks;
  if (blocks > 0x7fffffffLL) return fail(DS_ERR_INVALID, "ds_pair_reduce: too many pairs");
  dim3 grid((unsigned)blocks), block(kRedThreads);
  switch (mode) {
    case DS_SIM_COSINE:
      pair_reduce_kernel<T, DS_SIM_COSINE><<<grid, block, 0, st>>>(xp, yp, E, xs, ys, chunks, chunk_elems, vec_ok, partials,
                                                                   counters, out);
      break;
    case DS_SIM_MSE:
      pair_reduce_kernel<T, DS_SIM_MSE><<<grid, block, 0, st>>>(xp, yp, E, xs, ys, chunks, chunk_elems, vec_ok, partials,
                                                                counters, out);
      break;
    case DS_SIM_MINMAX_COSINE:
      pair_reduce_kernel<T, DS_SIM_MINMAX_COSINE><<<grid, block, 0, st>>>(xp, yp, E, xs, ys, chunks, chunk_elems,
                                                                          vec_ok, partials, counters, out);
      break;
    default:
      return fail(DS_ERR_INVALID, "ds_pair_reduce: bad mode %d", mode);
  }
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

template <typename T, int MODE>
static void launch_reduce_bwd(const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t xs, int64_t ys,
                              const float* d_out, float* dx, int64_t dxs, float* dy, int64_t dys, float* partials,
                              unsigned int* counters, int chunks, int64_t chunk_elems, int vec_ok, cudaStream_t st) {
  const T* xp = static_cast<const T*>(x);
  const T* yp = static_cast<const T*>(y);
  dim3 grid((unsigned)(n_pairs * chunks)), block(kRedThreads);
  if constexpr (MODE != DS_SIM_MSE)  // the statistics pass only reads d_out
    pair_reduce_kernel<T, MODE | kBwdStats><<<grid, block, 0, st>>>(xp, yp, E, xs, ys, chunks, chunk_elems, vec_ok,
                                                                    partials, counters, const_cast<float*>(d_out));
  pair_reduce_grad_kernel<T, MODE><<<grid, block, 0, st>>>(xp, yp, E, xs, ys, chunks, chunk_elems, vec_ok, partials,
                                                           d_out, dx, dxs, dy, dys);
}

template <typename T>
static void launch_reduce_bwd_mode(int mode, const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t xs,
                                   int64_t ys, const float* d_out, float* dx, int64_t dxs, float* dy, int64_t dys,
                                   float* partials, unsigned int* counters, int chunks, int64_t chunk_elems,
                                   int vec_ok, cudaStream_t st) {
  if (mode == DS_SIM_COSINE)
    launch_reduce_bwd<T, DS_SIM_COSINE>(x, y, n_pairs, E, xs, ys, d_out, dx, dxs, dy, dys, partials, counters, chunks,
                                        chunk_elems, vec_ok, st);
  else if (mode == DS_SIM_MSE)
    launch_reduce_bwd<T, DS_SIM_MSE>(x, y, n_pairs, E, xs, ys, d_out, dx, dxs, dy, dys, partials, counters, chunks,
                                     chunk_elems, vec_ok, st);
  else
    launch_reduce_bwd<T, DS_SIM_MINMAX_COSINE>(x, y, n_pairs, E, xs, ys, d_out, dx, dxs, dy, dys, partials, counters,
                                               chunks, chunk_elems, vec_ok, st);
}

}  // namespace ds

extern "C" {

size_t ds_pair_reduce_workspace_bytes(int64_t n_pairs, int64_t E) {
  if (n_pairs <= 0 || E <= 0) return 256;
  // sized for the widest split so that the plan never needs more
  size_t part = (size_t)n_pairs * ds::kRedMaxChunks * ds::kRedSlots * sizeof(float);
  size_t cnt = (size_t)n_pairs * sizeof(unsigned int);
  return ds::align_up(part, 256) + ds::align_up(cnt, 256) + 256;
}

int ds_pair_reduce(const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t x_stride, int64_t y_stride,
                   int dtype, int mode, float* out, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_pairs < 0 || E <= 0) return fail(DS_ERR_INVALID, "ds_pair_reduce: n_pairs %lld E %lld", (long long)n_pairs, (long long)E);
  if (n_pairs == 0) return DS_OK;
  if (!x || !y || !out) return fail(DS_ERR_INVALID, "ds_pair_reduce: null pointer");
  if (dtype != DS_F16 && dtype != DS_BF16 && dtype != DS_F32) return fail(DS_ERR_INVALID, "ds_pair_reduce: bad dtype %d", dtype);
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE && mode != DS_SIM_MINMAX_COSINE)
    return fail(DS_ERR_INVALID, "ds_pair_reduce: bad mode %d", mode);
  const size_t es = elem_size(dtype);
  if (((uintptr_t)x % es) || ((uintptr_t)y % es)) return fail(DS_ERR_INVALID, "ds_pair_reduce: x and y must be element-aligned");
  if (x_stride < E || y_stride < E) return fail(DS_ERR_INVALID, "ds_pair_reduce: row stride smaller than E");
  // 128-bit loads need every row to start on a 16-byte boundary; otherwise the kernel reads element-wise
  const int vec_ok = !(((uintptr_t)x & 15) || ((uintptr_t)y & 15) ||
                       (n_pairs > 1 && ((((size_t)x_stride * es) & 15) || (((size_t)y_stride * es) & 15))));
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;

  int chunks;
  int64_t chunk_elems;
  reduce_plan(n_pairs, E, dtype == DS_F32 ? 4 : 8, &chunks, &chunk_elems);
  Workspace w(ws, ws_bytes);
  float* partials = static_cast<float*>(w.take((size_t)n_pairs * chunks * kRedSlots * sizeof(float)));
  unsigned int* counters = static_cast<unsigned int*>(w.take((size_t)n_pairs * sizeof(unsigned int)));
  if (!partials || !counters)
    return fail(DS_ERR_WORKSPACE, "ds_pair_reduce: workspace too small (%zu bytes given, need %zu)", ws_bytes,
                ds_pair_reduce_workspace_bytes(n_pairs, E));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DS_CUDA_TRY(cudaMemsetAsync(counters, 0, (size_t)n_pairs * sizeof(unsigned int), st));
  if (dtype == DS_F16)
    return launch_reduce<__half>(x, y, n_pairs, E, x_stride, y_stride, mode, out, partials, counters, chunks, chunk_elems, vec_ok, st);
  if (dtype == DS_BF16)
    return launch_reduce<__nv_bfloat16>(x, y, n_pairs, E, x_stride, y_stride, mode, out, partials, counters, chunks, chunk_elems, vec_ok, st);
  return launch_reduce<float>(x, y, n_pairs, E, x_stride, y_stride, mode, out, partials, counters, chunks, chunk_elems, vec_ok, st);
}

size_t ds_pair_reduce_bwd_workspace_bytes(int64_t n_pairs, int64_t E) {
  if (n_pairs <= 0 || E <= 0) return 256;
  // sized for the widest split so that the plan never needs more
  size_t part = (size_t)n_pairs * ds::kRedMaxChunks * ds::kRedTieSlots * sizeof(float);
  size_t cnt = (size_t)n_pairs * sizeof(unsigned int);
  return ds::align_up(part, 256) + ds::align_up(cnt, 256) + 256;
}

int ds_pair_reduce_bwd(const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t x_stride, int64_t y_stride,
                       int dtype, int mode, const float* d_out, float* dx, int64_t dx_stride, float* dy,
                       int64_t dy_stride, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_pairs < 0 || E <= 0)
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: n_pairs %lld E %lld", (long long)n_pairs, (long long)E);
  if (!x || !y || !d_out) return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: null x, y or d_out");
  if (dtype != DS_F16 && dtype != DS_BF16 && dtype != DS_F32)
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: bad dtype %d", dtype);
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE && mode != DS_SIM_MINMAX_COSINE)
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: bad mode %d", mode);
  const size_t es = elem_size(dtype);
  if (((uintptr_t)x % es) || ((uintptr_t)y % es))
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: x and y must be element-aligned");
  if (((uintptr_t)d_out % 4) || ((uintptr_t)dx % 4) || ((uintptr_t)dy % 4))
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: d_out, dx and dy must be 4-byte aligned");
  if (x_stride < E || y_stride < E) return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: row stride smaller than E");
  if ((dx && dx_stride < E) || (dy && dy_stride < E))
    return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: gradient row stride smaller than E");
  if (n_pairs == 0 || (!dx && !dy)) return DS_OK;
  int chunks;
  int64_t chunk_elems;
  reduce_plan(n_pairs, E, dtype == DS_F32 ? 4 : 8, &chunks, &chunk_elems);
  if (n_pairs * chunks > 0x7fffffffLL) return fail(DS_ERR_INVALID, "ds_pair_reduce_bwd: too many pairs");
  // 128-bit loads and stores need every row of the inputs and of the wanted gradients on a 16-byte boundary
  auto rows16 = [&](const void* p, int64_t stride, size_t bytes) {
    return !p || !(((uintptr_t)p & 15) || (n_pairs > 1 && (((size_t)stride * bytes) & 15)));
  };
  const int vec_ok = rows16(x, x_stride, es) && rows16(y, y_stride, es) && rows16(dx, dx_stride, 4) &&
                     rows16(dy, dy_stride, 4);
  float* partials = nullptr;
  unsigned int* counters = nullptr;
  if (mode != DS_SIM_MSE) {
    Workspace w(ws, ws_bytes);
    partials = static_cast<float*>(w.take((size_t)n_pairs * chunks * kRedTieSlots * sizeof(float)));
    counters = static_cast<unsigned int*>(w.take((size_t)n_pairs * sizeof(unsigned int)));
    if (!partials || !counters)
      return fail(DS_ERR_WORKSPACE, "ds_pair_reduce_bwd: workspace too small (%zu bytes given, need %zu)", ws_bytes,
                  ds_pair_reduce_bwd_workspace_bytes(n_pairs, E));
  }
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (counters) DS_CUDA_TRY(cudaMemsetAsync(counters, 0, (size_t)n_pairs * sizeof(unsigned int), st));
  if (dtype == DS_F16)
    launch_reduce_bwd_mode<__half>(mode, x, y, n_pairs, E, x_stride, y_stride, d_out, dx, dx_stride, dy, dy_stride,
                                   partials, counters, chunks, chunk_elems, vec_ok, st);
  else if (dtype == DS_BF16)
    launch_reduce_bwd_mode<__nv_bfloat16>(mode, x, y, n_pairs, E, x_stride, y_stride, d_out, dx, dx_stride, dy,
                                          dy_stride, partials, counters, chunks, chunk_elems, vec_ok, st);
  else
    launch_reduce_bwd_mode<float>(mode, x, y, n_pairs, E, x_stride, y_stride, d_out, dx, dx_stride, dy, dy_stride,
                                  partials, counters, chunks, chunk_elems, vec_ok, st);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
