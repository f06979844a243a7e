// Error plumbing, device queries, tensor-map encoding and the small entry points.
#include "ds_host.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <mutex>

namespace ds {

int g_gemm_variant = -1;


static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  // clear the sticky-less error state so that the next call reports its own error
  (void)cudaGetLastError();
  return DS_ERR_CUDA;
}

namespace {
struct DevInfo {
  bool valid = false;
  int sms = 0;
  int major = 0;
};
DevInfo g_dev[64];
std::mutex g_mu;

const DevInfo* dev_info() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
    (void)cudaGetLastError();
    return nullptr;
  }
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_dev[dev].valid) {
    int sms = 0, major = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
      (void)cudaGetLastError();
      return nullptr;
    }
    g_dev[dev].sms = sms;
    g_dev[dev].major = major;
    g_dev[dev].valid = true;
  }
  return &g_dev[dev];
}
}  // namespace

int sm_count() {
  const DevInfo* d = dev_info();
  return d ? d->sms : 0;
}

bool device_is_sm100() {
  const DevInfo* d = dev_info();
  return d && d->major == 10;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
    else (void)cudaGetLastError();
  });
  return fn;
}

int encode_tensor_map(CUtensorMap* out, int dtype, int rank, const void* base, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes, int l2_promotion_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(DS_ERR_CUDA, "cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
  CUtensorMapDataType dt = dtype == DS_F16    ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                           : dtype == DS_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                              : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  CUtensorMapSwizzle sw = swizzle_bytes == 128  ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                          : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                : CU_TENSOR_MAP_SWIZZLE_NONE;
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5];
  cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = fn(out, dt, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  l2_promotion_bytes >= 256   ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                  : l2_promotion_bytes >= 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                  : l2_promotion_bytes >= 64  ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                              : CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    return fail(DS_ERR_INVALID,
                "cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims [%llu,%llu,%llu,%llu,%llu] box "
                "[%u,%u,%u,%u,%u] stride1 %llu swizzle %d base %p",
                (int)r, rank, (unsigned long long)gdim[0], (unsigned long long)(rank > 1 ? gdim[1] : 0),
                (unsigned long long)(rank > 2 ? gdim[2] : 0), (unsigned long long)(rank > 3 ? gdim[3] : 0),
                (unsigned long long)(rank > 4 ? gdim[4] : 0), bx[0], rank > 1 ? bx[1] : 0, rank > 2 ? bx[2] : 0,
                rank > 3 ? bx[3] : 0, rank > 4 ? bx[4] : 0, (unsigned long long)(rank > 1 ? gstr[0] : 0),
                swizzle_bytes, base);
  }
  return DS_OK;
}

// ---------------------------------------------------------------------------
// in-stream timing of the attention kernel
// ---------------------------------------------------------------------------
namespace {
constexpr int kProfRing = 256;
struct Prof {
  bool on = false;
  bool created = false;
  cudaEvent_t ev[kProfRing][2];
  int n = 0;
  bool open = false;
} g_prof;
std::mutex g_prof_mu;
}  // namespace

void profile_begin(cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof.on || g_prof.n >= kProfRing) return;
  if (!g_prof.created) {
    for (int i = 0; i < kProfRing; ++i) {
      if (cudaEventCreate(&g_prof.ev[i][0]) != cudaSuccess || cudaEventCreate(&g_prof.ev[i][1]) != cudaSuccess) {
        (void)cudaGetLastError();
        g_prof.on = false;
        return;
      }
    }
    g_prof.created = true;
  }
  cudaEventRecord(g_prof.ev[g_prof.n][0], st);
  g_prof.open = true;
}

void profile_end(cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof.on || !g_prof.open) return;
  cudaEventRecord(g_prof.ev[g_prof.n][1], st);
  g_prof.n++;
  g_prof.open = false;
}

// ---------------------------------------------------------------------------
// 2AFC decision kernel (cute_main.py:196-205)
// ---------------------------------------------------------------------------
__global__ void twoafc_kernel(const float* __restrict__ ab, const float* __restrict__ ac, int64_t n, int mode,
                              int32_t* __restrict__ counts, uint8_t* __restrict__ flags) {
  int c1 = 0, c2 = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float a = ab[i], b = ac[i];
    bool ok, ok2;
    if (mode == DS_SIM_MSE) {
      ok = a < b;
      ok2 = a * 2.0f < b;
    } else {
      ok = a > b;
      ok2 = a > 2.0f * b;
    }
    if (flags) flags[i] = ok ? 1 : 0;
    c1 += ok ? 1 : 0;
    c2 += ok2 ? 1 : 0;
  }
  for (int o = 16; o > 0; o >>= 1) {
    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
    c2 += __shfl_xor_sync(0xffffffffu, c2, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (c1) atomicAdd(&counts[0], c1);
    if (c2) atomicAdd(&counts[1], c2);
  }
}

}  // namespace ds

extern "C" {

int ds_abi_version(void) { return DS_ABI_VERSION; }

const char* ds_last_error(void) { return ds::g_err; }

int ds_device_ok(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    (void)cudaGetLastError();
    return ds::fail(DS_ERR_CUDA, "no CUDA device available (%s)", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
  }
  if (!ds::device_is_sm100())
    return ds::fail(DS_ERR_UNSUPPORTED, "current device is not compute capability 10.x (B200, sm_100a)");
  return DS_OK;
}

int ds_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(ds::g_prof_mu);
  ds::g_prof.on = on != 0;
  ds::g_prof.n = 0;
  ds::g_prof.open = false;
  return DS_OK;
}

int ds_profile_collect(float* total_ms, int* launches) {
  if (!total_ms || !launches) return ds::fail(DS_ERR_INVALID, "ds_profile_collect: null pointer");
  std::lock_guard<std::mutex> lk(ds::g_prof_mu);
  float tot = 0.f;
  for (int i = 0; i < ds::g_prof.n; ++i) {
    float ms = 0.f;
    DS_CUDA_TRY(cudaEventSynchronize(ds::g_prof.ev[i][1]));
    DS_CUDA_TRY(cudaEventElapsedTime(&ms, ds::g_prof.ev[i][0], ds::g_prof.ev[i][1]));
    tot += ms;
  }
  *total_ms = tot;
  *launches = ds::g_prof.n;
  ds::g_prof.n = 0;
  return DS_OK;
}

int ds_debug_set_gemm_variant(int variant) {
  if (variant == -1 || variant == 0 || variant == 2) ds::g_gemm_variant = variant;
  return ds::g_gemm_variant;
}

int ds_twoafc(const float* ab, const float* ac, int64_t n, int mode, int32_t* counts, uint8_t* flags,
              void* stream) {
  if (!counts || n < 0 || (n > 0 && (!ab || !ac))) return ds::fail(DS_ERR_INVALID, "ds_twoafc: null pointer or negative n");
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return ds::fail(DS_ERR_INVALID, "ds_twoafc: bad mode %d", mode);
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DS_CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
  if (n == 0) return DS_OK;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 1184) blocks = 1184;
  ds::twoafc_kernel<<<blocks, 256, 0, st>>>(ab, ac, n, mode, counts, flags);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
