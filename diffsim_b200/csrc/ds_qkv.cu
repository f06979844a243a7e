// K4 -- QKV projection of the hooked self-attention layer (tensor-core bound).
//
//   [q | k | v][r, :] = hidden[r, :] . W^T (+ bias)          W = [W_q; W_k; W_v]  (nn.Linear layout: [out, in])
//
// The capture step of the reference: attn.to_q / to_k / to_v on the hook's input (diffsim/hacked_attn.py:61-69;
// the head split of :74-77 is a view and costs nothing here: the outputs ARE the (B,S,H*D) memory the attention
// kernel reads through (B,H,S,D) strides) and DiT's fused module.qkv(x) (diffsim/diffsim_dit.py:21-23, packed
// (B,N,3*H*D) output).  With it the drop-in boundary moves from Q/K/V to the hook INPUT: a third of the bytes.
// One pass of the persistent tcgen05 GEMM core (ds_gemm.cuh), fp32 accumulation, bias added in fp32, rounded once
// to the input dtype (as a cuBLAS-backed nn.Linear does).  Algorithmic work: 2 * rows * C_in * n_out flops.
#include "ds_gemm.cuh"

#include <algorithm>
#include <type_traits>

extern "C" {

int ds_qkv_project(const void* hidden, int64_t n_rows, int64_t ld_hidden, int64_t c_in, const void* weight,
                   int64_t ld_weight, const void* bias, int64_t n_out, int64_t cols_per_out, void* const* out,
                   const int64_t* ld_out, int dtype, void* stream) {
  using namespace ds;
  if (n_rows < 0 || c_in <= 0 || n_out <= 0 || cols_per_out <= 0) return fail(DS_ERR_INVALID, "ds_qkv_project: bad sizes");
  if (n_rows == 0) return DS_OK;
  if (!hidden || !weight || !out || !ld_out) return fail(DS_ERR_INVALID, "ds_qkv_project: null pointer");
  if (dtype != DS_F16 && dtype != DS_BF16) return fail(DS_ERR_UNSUPPORTED, "ds_qkv_project: dtype must be f16 or bf16");
  if (n_out % cols_per_out) return fail(DS_ERR_INVALID, "ds_qkv_project: n_out must be a multiple of cols_per_out");
  const int64_t n_t = n_out / cols_per_out;
  if (n_t < 1 || n_t > 3) return fail(DS_ERR_INVALID, "ds_qkv_project: 1 to 3 output tensors (got %lld)", (long long)n_t);
  if ((cols_per_out & 7) || (c_in & 7) || (ld_hidden & 7) || (ld_weight & 7) || ld_hidden < c_in || ld_weight < c_in)
    return fail(DS_ERR_INVALID, "ds_qkv_project: channel counts and leading dimensions must be multiples of 8 elements");
  if (((uintptr_t)hidden & 15) || ((uintptr_t)weight & 15) || (bias && ((uintptr_t)bias & 15)))
    return fail(DS_ERR_INVALID, "ds_qkv_project: pointers must be 16-byte aligned");
  if (n_rows > INT32_MAX || n_out > INT32_MAX) return fail(DS_ERR_INVALID, "ds_qkv_project: sizes too large");
  GemmParams gp = {};
  for (int64_t t = 0; t < n_t; ++t) {
    if (!out[t] || ((uintptr_t)out[t] & 15) || (ld_out[t] & 7) || ld_out[t] < cols_per_out)
      return fail(DS_ERR_INVALID, "ds_qkv_project: output %lld needs a 16-byte aligned pointer and ld >= cols_per_out, multiple of 8",
                  (long long)t);
    gp.out[t] = out[t];
    gp.ld_out[t] = ld_out[t];
  }
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  gp.splits = 1;
  gp.use_pair = -1;
  gp.cols_per_out = (int)cols_per_out;
  gp.bias = bias;
  return launch_gemm_tn<GEMM_EPI_16>(hidden, n_rows, ld_hidden, weight, n_out, ld_weight, c_in, dtype, gp,
                                     static_cast<cudaStream_t>(stream));
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Backward of the projection (what an fp16 / bf16 nn.Linear backward returns, deterministic):
//   dhidden = dY W        dweight = dY^T hidden        dbias = column sums of dY
// dY is the gradient of the (up to three) outputs, read in place.  The two products run on the GEMM core's backward
// operand layouts (launch_gemm_bwd, ds_gemm.cuh) into fp32 split-K partials; a finishing kernel adds them in split order
// and rounds once to the input dtype.  dbias: per-chunk column sums of 256 rows, added in chunk order.  No atomics.
// ---------------------------------------------------------------------------------------------------------------------
namespace ds {

constexpr int kBwdFinThreads = 256;
constexpr int kBiasChunkRows = 256;

// out[r, c] = round(sum over s, in order, of part[s][r][c]): eight columns per thread (N is a multiple of 8)
template <bool kBf16>
__global__ void __launch_bounds__(kBwdFinThreads)
gemm_bwd_finish_kernel(const float* __restrict__ part, int splits, int64_t split_stride, int64_t M, int64_t N,
                       uint16_t* __restrict__ out, int64_t ld) {
  const int64_t units = N >> 3;
  const int64_t i = blockIdx.x * (int64_t)kBwdFinThreads + threadIdx.x;
  if (i >= M * units) return;
  const int64_t r = i / units, c = (i - r * units) * 8;
  const float* src = part + r * N + c;
  float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src + 4));
  for (int s = 1; s < splits; ++s) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(src + s * split_stride));
    const float4 y = __ldg(reinterpret_cast<const float4*>(src + s * split_stride + 4));
    a.x += x.x, a.y += x.y, a.z += x.z, a.w += x.w;
    b.x += y.x, b.y += y.y, b.z += y.z, b.w += y.w;
  }
  *reinterpret_cast<uint4*>(out + r * ld + c) =
      make_uint4(pack2<kBf16>(a.x, a.y), pack2<kBf16>(a.z, a.w), pack2<kBf16>(b.x, b.y), pack2<kBf16>(b.z, b.w));
}

struct BiasSrc {
  const uint16_t* dy[3];
  int64_t ld[3];
};

// part[chunk][t * seg_len + c] = sum of dy[t][r][c] over the chunk's rows.  A block: 64 columns of one tensor x one chunk;
// 8 threads per row read 16 bytes each, 32 rows at a time; the 32 row sums are then added in row order.
template <bool kBf16>
__global__ void __launch_bounds__(256)
bias_partial_kernel(const BiasSrc src, int64_t rows, int seg_len, int groups_per_seg, int64_t n_out, float* __restrict__ part) {
  __shared__ float red[32][65];
  const int t = blockIdx.x / groups_per_seg;
  const int c0 = (blockIdx.x - t * groups_per_seg) * 64;
  const int cu = threadIdx.x & 7, rl = threadIdx.x >> 3;
  const int col = c0 + cu * 8;
  const int64_t r0 = (int64_t)blockIdx.y * kBiasChunkRows, r1 = min(rows, r0 + kBiasChunkRows);
  // selected, not indexed: a run-time index into the parameter struct would copy it to local memory
  const uint16_t* dy = t == 0 ? src.dy[0] : t == 1 ? src.dy[1] : src.dy[2];
  const int64_t ld = t == 0 ? src.ld[0] : t == 1 ? src.ld[1] : src.ld[2];
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col < seg_len) {
    for (int64_t r = r0 + rl; r < r1; r += 32) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(dy + r * ld + col));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack2<kBf16>(w[j]);
        acc[2 * j] += f.x;
        acc[2 * j + 1] += f.y;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[rl][cu * 8 + j] = acc[j];
  __syncthreads();
  if (threadIdx.x < 64 && c0 + (int)threadIdx.x < seg_len) {
    float s = 0.f;
    for (int i = 0; i < 32; ++i) s += red[i][threadIdx.x];
    part[(int64_t)blockIdx.y * n_out + (int64_t)t * seg_len + c0 + threadIdx.x] = s;
  }
}

template <bool kBf16>
__global__ void bias_finish_kernel(const float* __restrict__ part, int chunks, int64_t n_out, uint16_t* __restrict__ dbias) {
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n >= n_out) return;
  float s = 0.f;
  for (int c = 0; c < chunks; ++c) s += part[(int64_t)c * n_out + n];
  const uint32_t h = pack2<kBf16>(s, 0.f);
  dbias[n] = (uint16_t)(h & 0xFFFFu);
}

static size_t qkv_bwd_gemm_part_bytes(int64_t n_rows, int64_t c_in, int64_t n_out, int64_t cols_per_out) {
  const int n_seg = (int)(n_out / cols_per_out);
  size_t b = 0;
  for (int pair = 0; pair < 2; ++pair) {   // either kernel may serve (ds_debug_set_gemm_variant)
    const GemmBwdPlan gx = gemm_bwd_plan(GEMM_BWD_DX, n_rows, c_in, n_seg, cols_per_out, pair);
    const GemmBwdPlan gw = gemm_bwd_plan(GEMM_BWD_DW, n_rows, c_in, n_seg, cols_per_out, pair);
    b = std::max(b, (size_t)gx.splits * n_rows * c_in * sizeof(float));
    b = std::max(b, (size_t)gw.splits * n_out * c_in * sizeof(float));
  }
  return b;
}

}  // namespace ds

extern "C" {

size_t ds_qkv_project_bwd_workspace_bytes(int64_t n_rows, int64_t c_in, int64_t n_out, int64_t cols_per_out) {
  using namespace ds;
  if (n_rows <= 0 || c_in <= 0 || n_out <= 0 || cols_per_out <= 0 || n_out % cols_per_out || n_out / cols_per_out > 3)
    return 256;
  const int64_t chunks = (n_rows + kBiasChunkRows - 1) / kBiasChunkRows;
  return align_up((size_t)chunks * n_out * sizeof(float), 256) + align_up(qkv_bwd_gemm_part_bytes(n_rows, c_in, n_out, cols_per_out), 256) +
         1024;
}

int ds_qkv_project_bwd(const void* hidden, int64_t n_rows, int64_t ld_hidden, int64_t c_in, const void* weight,
                       int64_t ld_weight, int64_t n_out, int64_t cols_per_out, const void* const* dy, const int64_t* ld_dy,
                       void* dhidden, int64_t ld_dhidden, void* dweight, int64_t ld_dweight, void* dbias, int dtype, void* ws,
                       size_t ws_bytes, void* stream) {
  using namespace ds;
  const char* who = "ds_qkv_project_bwd";
  if (n_rows <= 0 || c_in <= 0 || n_out <= 0 || cols_per_out <= 0) return fail(DS_ERR_INVALID, "%s: bad sizes", who);
  if (!dy || !ld_dy) return fail(DS_ERR_INVALID, "%s: null pointer (dy)", who);
  if (dhidden && !weight) return fail(DS_ERR_INVALID, "%s: null pointer (weight, needed for dhidden)", who);
  if (dweight && !hidden) return fail(DS_ERR_INVALID, "%s: null pointer (hidden, needed for dweight)", who);
  if (dtype != DS_F16 && dtype != DS_BF16) return fail(DS_ERR_UNSUPPORTED, "%s: dtype must be f16 or bf16", who);
  if (n_out % cols_per_out) return fail(DS_ERR_INVALID, "%s: n_out must be a multiple of cols_per_out", who);
  const int64_t n_t = n_out / cols_per_out;
  if (n_t < 1 || n_t > 3) return fail(DS_ERR_INVALID, "%s: 1 to 3 gradient tensors (got %lld)", who, (long long)n_t);
  if ((cols_per_out & 7) || (c_in & 7))
    return fail(DS_ERR_INVALID, "%s: channel counts and leading dimensions must be multiples of 8 elements", who);
  if ((hidden && ((ld_hidden & 7) || ld_hidden < c_in)) || (weight && ((ld_weight & 7) || ld_weight < c_in)) ||
      (dhidden && ((ld_dhidden & 7) || ld_dhidden < c_in)) || (dweight && ((ld_dweight & 7) || ld_dweight < c_in)))
    return fail(DS_ERR_INVALID, "%s: channel counts and leading dimensions must be multiples of 8 elements", who);
  if (((uintptr_t)hidden & 15) || ((uintptr_t)weight & 15) || ((uintptr_t)dhidden & 15) || ((uintptr_t)dweight & 15) ||
      ((uintptr_t)dbias & 15))
    return fail(DS_ERR_INVALID, "%s: pointers must be 16-byte aligned", who);
  if (n_rows > INT32_MAX || n_out > INT32_MAX) return fail(DS_ERR_INVALID, "%s: sizes too large", who);
  BiasSrc bs = {};
  for (int64_t t = 0; t < n_t; ++t) {
    if (!dy[t] || ((uintptr_t)dy[t] & 15) || (ld_dy[t] & 7) || ld_dy[t] < cols_per_out)
      return fail(DS_ERR_INVALID, "%s: dy %lld needs a 16-byte aligned pointer and ld >= cols_per_out, multiple of 8", who,
                  (long long)t);
    bs.dy[t] = static_cast<const uint16_t*>(dy[t]);
    bs.ld[t] = ld_dy[t];
  }
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  if (!dhidden && !dweight && !dbias) return DS_OK;

  const int64_t chunks = (n_rows + kBiasChunkRows - 1) / kBiasChunkRows;
  Workspace w(ws, ws_bytes);
  float* bpart = static_cast<float*>(w.take((size_t)chunks * n_out * sizeof(float)));
  float* gpart = static_cast<float*>(w.take(qkv_bwd_gemm_part_bytes(n_rows, c_in, n_out, cols_per_out)));
  if (!bpart || !gpart)
    return fail(DS_ERR_WORKSPACE, "%s: workspace too small (%zu given, need %zu)", who, ws_bytes,
                ds_qkv_project_bwd_workspace_bytes(n_rows, c_in, n_out, cols_per_out));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n_seg = (int)n_t;
  auto run = [&](auto bf16) -> int {
    constexpr bool kBf16 = decltype(bf16)::value;
    if (dbias) {
      const int groups = (int)((cols_per_out + 63) / 64);
      if (chunks > 65535) return fail(DS_ERR_INVALID, "%s: too many rows for the bias reduction", who);
      bias_partial_kernel<kBf16><<<dim3((unsigned)(n_seg * groups), (unsigned)chunks), 256, 0, st>>>(
          bs, n_rows, (int)cols_per_out, groups, n_out, bpart);
      bias_finish_kernel<kBf16><<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(bpart, (int)chunks, n_out,
                                                                                 static_cast<uint16_t*>(dbias));
      DS_CUDA_TRY(cudaGetLastError());
    }
    auto finish = [&](const GemmBwdPlan& g, int64_t M, void* out, int64_t ld) -> int {
      const int64_t threads = M * (c_in / 8);
      gemm_bwd_finish_kernel<kBf16><<<(unsigned)((threads + kBwdFinThreads - 1) / kBwdFinThreads), kBwdFinThreads, 0, st>>>(
          gpart, g.splits, M * c_in, M, c_in, static_cast<uint16_t*>(out), ld);
      DS_CUDA_TRY(cudaGetLastError());
      return DS_OK;
    };
    if (dhidden) {
      const GemmBwdPlan g = gemm_bwd_plan(GEMM_BWD_DX, n_rows, c_in, n_seg, cols_per_out, -1);
      int r = launch_gemm_bwd<GEMM_BWD_DX>(g, dy, ld_dy, n_seg, cols_per_out, weight, ld_weight, nullptr, 0, n_rows, c_in,
                                           dtype, gpart, st);
      if (r == DS_OK) r = finish(g, n_rows, dhidden, ld_dhidden);
      if (r != DS_OK) return r;
    }
    if (dweight) {
      const GemmBwdPlan g = gemm_bwd_plan(GEMM_BWD_DW, n_rows, c_in, n_seg, cols_per_out, -1);
      int r = launch_gemm_bwd<GEMM_BWD_DW>(g, dy, ld_dy, n_seg, cols_per_out, nullptr, 0, hidden, ld_hidden, n_rows, c_in,
                                           dtype, gpart, st);
      if (r == DS_OK) r = finish(g, n_out, dweight, ld_dweight);
      if (r != DS_OK) return r;
    }
    return DS_OK;
  };
  return dtype == DS_BF16 ? run(std::true_type{}) : run(std::false_type{});
}

}  // extern "C"
