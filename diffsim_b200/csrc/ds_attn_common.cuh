// Host layer shared by the attention forward (K1, ds_attn.cu) and backward (K5, ds_attn_bwd.cu): the shared-memory tile
// geometry of a head dim, validation of the 16-bit (n, b, h, s, d) operands, their TMA maps, and the dispatch over the
// head dims and dtypes the kernels are built for.
#pragma once

#include <type_traits>

#include "ds_host.h"
#include "ds_ptx.cuh"

namespace ds {

// A tile of D-element operand rows as TMA writes it and tcgen05.mma reads it: NSUB swizzled sub-tiles of SUBW columns.
template <int D>
struct AttnTile {
  static constexpr int D_PAD = (D + 15) / 16 * 16;
  static constexpr int SUBW = (D % 64 == 0) ? 64 : 32;           // elements per swizzle row
  static constexpr int SUB_BYTES = SUBW * 2;                      // 128 or 64: TMA box row == swizzle span
  static constexpr int NSUB = (D_PAD + SUBW - 1) / SUBW;
  static constexpr uint32_t LAYOUT = (SUBW == 64) ? UMMA_SW128 : UMMA_SW64;
  static constexpr int CPS = SUBW / 16;                           // 16-element K chunks per sub-tile
};

// the head dims K1 and K5 are instantiated for
#define DS_ATTN_HEAD_DIMS 40, 64, 72, 80, 128, 160
#define DS_ATTN_STR_(...) #__VA_ARGS__
#define DS_ATTN_STR(...) DS_ATTN_STR_(__VA_ARGS__)

template <int... Ds, typename F>
int dispatch_head_dim(int64_t d, const char* who, F&& f) {
  int rc = DS_OK;
  if (((d == Ds && ((rc = f(std::integral_constant<int, Ds>{})), true)) || ...)) return rc;
  return fail(DS_ERR_UNSUPPORTED, "%s: head dim %lld is not built (supported: " DS_ATTN_STR(DS_ATTN_HEAD_DIMS) ")", who,
              (long long)d);
}

// f(std::integral_constant<int, D>{}) for the built head dim D == d; DS_ERR_UNSUPPORTED for any other d
template <typename F>
int with_head_dim(int64_t d, const char* who, F&& f) {
  return dispatch_head_dim<DS_ATTN_HEAD_DIMS>(d, who, f);
}

// f(std::true_type{}) for bf16 operands, f(std::false_type{}) for f16 ones
template <typename F>
int with_dtype(int dtype, F&& f) {
  return dtype == DS_BF16 ? f(std::true_type{}) : f(std::false_type{});
}

// a 16-bit operand that TMA can read: unit innermost stride, 16-byte aligned base, and 16-byte strides on every dimension
// with more than one element (a size-1 dimension may carry any stride)
inline int check_operand(const ds_tensor5& t, const char* who, const char* name) {
  if (!t.ptr) return fail(DS_ERR_INVALID, "%s: %s: null pointer", who, name);
  if (t.dtype != DS_F16 && t.dtype != DS_BF16) return fail(DS_ERR_UNSUPPORTED, "%s: %s: dtype must be f16 or bf16", who, name);
  for (int i = 0; i < 5; ++i)
    if (t.size[i] <= 0) return fail(DS_ERR_INVALID, "%s: %s: size[%d] = %lld", who, name, i, (long long)t.size[i]);
  if (t.stride[4] != 1)
    return fail(DS_ERR_INVALID, "%s: %s: innermost stride must be 1 (got %lld)", who, name, (long long)t.stride[4]);
  if ((uintptr_t)t.ptr & 15) return fail(DS_ERR_INVALID, "%s: %s: base pointer must be 16-byte aligned", who, name);
  for (int i = 0; i < 4; ++i)
    if (t.size[i] > 1 && (t.stride[i] <= 0 || (t.stride[i] & 7)))
      return fail(DS_ERR_INVALID, "%s: %s: stride[%d] = %lld must be a positive multiple of 8 elements (16 bytes)", who,
                  name, i, (long long)t.stride[i]);
  return DS_OK;
}

// an operand with q's dtype and shape (an attention output or its gradient)
inline int check_like(const ds_tensor5& t, const ds_tensor5& q, const char* who, const char* name) {
  const int rc = check_operand(t, who, name);
  if (rc != DS_OK) return rc;
  if (t.dtype != q.dtype) return fail(DS_ERR_INVALID, "%s: %s must have q's dtype", who, name);
  for (int i = 0; i < 5; ++i)
    if (t.size[i] != q.size[i]) return fail(DS_ERR_INVALID, "%s: %s must have q's shape", who, name);
  return DS_OK;
}

// a (b, h, s, d) tensor as the one-image operand (1, b, h, s, d)
inline ds_tensor5 lift(const ds_tensor4& t) {
  ds_tensor5 r;
  r.ptr = t.ptr;
  r.dtype = t.dtype;
  r.size[0] = 1;
  r.stride[0] = 8;
  for (int i = 0; i < 4; ++i) {
    r.size[i + 1] = t.size[i];
    r.stride[i + 1] = t.stride[i];
  }
  return r;
}

// L2 fetch granularity of the Q / K / V boxes.  A box row is one head's D elements (80-320 bytes) out of a (B, S, H*D)
// memory row whose other heads are needed much later (streams are head-major): with 256-byte promotion every miss dragged
// the neighbouring heads' bytes in from DRAM -- 17.1 MB per triplet against 11.8 MB algorithmic at D = 160, 2.9x at DiT's
// 144-byte rows.  64 bytes: +3% sustained, +5% DiT (profiles/r2bc_attn_l2_promotion_ab.txt).
constexpr int kAttnL2PromotionBytes = 64;

// TMA map of a validated operand: boxes of rows x subw elements, each box row one swizzle span of subw * 2 bytes
inline int make_map(CUtensorMap* m, const ds_tensor5& t, int subw, int rows) {
  // TMA dims, fastest first: (d, s, h, b, n)
  uint64_t dims[5] = {(uint64_t)t.size[4], (uint64_t)t.size[3], (uint64_t)t.size[2], (uint64_t)t.size[1],
                      (uint64_t)t.size[0]};
  // a size-1 dimension may carry any stride; give it a harmless 16-byte one
  auto st = [&](int i) -> uint64_t { return (uint64_t)(t.size[i] > 1 ? t.stride[i] : 8) * 2; };
  uint64_t strides[4] = {st(3), st(2), st(1), st(0)};
  uint32_t box[5] = {(uint32_t)subw, (uint32_t)rows, 1, 1, 1};
  return encode_tensor_map(m, t.dtype, 5, t.ptr, dims, strides, box, subw * 2, kAttnL2PromotionBytes);
}

// Grouped work lists (ds_attn.cu), for the AAS backward (ds_attn_bwd.cu):
// the argument checks of ds_aas_groups' five operands (no device work)
int check_group_operands(const ds_tensor5& q, const ds_tensor5& k_self, const ds_tensor5& v_self, const ds_tensor5& k,
                         const ds_tensor5& v, const char* who);
// bad[0] = 1 when an image index of the list is out of range (bad[0] must be zeroed first)
int launch_validate_groups(const int32_t* group_q, int64_t n_groups, const int32_t* kv_idx, int64_t n_entries,
                           int64_t nq_images, int64_t nk_images, int32_t* bad, cudaStream_t st);
// the work lists of ds_aas_pairs / ds_aas_triplets (pairs_setup_kernel, triplets_setup_kernel)
int launch_pairs_setup(const int32_t* pair_idx, int64_t n_pairs, int32_t* group_q, int32_t* group_off, int32_t* kv_idx,
                       cudaStream_t st);
int launch_triplets_setup(const int32_t* trip_idx, int64_t n_triplets, int32_t* group_q, int32_t* group_off,
                          int32_t* kv_idx, cudaStream_t st);
// one K1 launch storing Y_g = Attn(Q_i, K_i, V_i) at slot g and X_t = Attn(Q_i, K_j, V_j) at slot n_groups + t of `out`, a
// contiguous (n_groups + n_entries, B, H, Sq, D) stack of q's dtype, rounded exactly as ds_attn_fwd rounds its output
int attn_list_store(const ds_tensor5& q, const ds_tensor5& k_self, const ds_tensor5& v_self, const ds_tensor5& k,
                    const ds_tensor5& v, const int32_t* group_q, const int32_t* group_off, int64_t n_groups,
                    const int32_t* kv_idx, float scale, void* out, const char* who, cudaStream_t st);

}  // namespace ds
