// Host-side helpers shared by the C-ABI translation units.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/diffsim_b200.h"

namespace ds {

// thread-local error message behind ds_last_error()
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DS_CUDA_TRY(expr)                                      \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) return ::ds::cuda_fail(_e, #expr);  \
  } while (0)

// Device properties of the current device (cached per device).
int sm_count();
bool device_is_sm100();

inline size_t elem_size(int dtype) { return dtype == DS_F32 ? 4 : 2; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// cuTensorMapEncodeTiled through cudaGetDriverEntryPoint (libcuda is not a
// link-time dependency, so the library loads on a machine without a driver).
// dims / box: fastest dimension first.  strides_bytes: rank-1 entries (dim 1..).
// swizzle_bytes: 0, 32, 64 or 128.  Out-of-bounds elements are filled with zero.  l2_promotion_bytes: 0, 64, 128 or 256 --
// the granularity at which the L2 fetches a missing box row from DRAM (256 suits rows that are read whole; rows that are
// thin slices of a wider memory row -- one head of (B, S, H*D) -- would drag their neighbours' bytes in with it).
int encode_tensor_map(CUtensorMap* out, int dtype, int rank, const void* base, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes, int l2_promotion_bytes = 256);

// in-stream kernel timing (ds_profile_enable / ds_profile_collect)
void profile_begin(cudaStream_t st);
void profile_end(cudaStream_t st);

extern int g_gemm_variant;   // ds_debug_set_gemm_variant: -1 automatic, 0 1-CTA GEMM kernel only, 2 CTA-pair kernel always

// simple bump allocator over the caller's workspace
struct Workspace {
  char* base;
  size_t size;
  size_t off;
  Workspace(void* p, size_t n) : base(static_cast<char*>(p)), size(n), off(0) {}
  void* take(size_t bytes, size_t align = 256) {
    size_t o = align_up(off, align);
    if (base == nullptr || o + bytes > size) return nullptr;
    off = o + bytes;
    return base + o;
  }
};

}  // namespace ds
