/*
 * diffsim_b200 -- C ABI of the B200-native DiffSim scoring hot path.
 *
 * This is the drop-in boundary for the Aligned Attention Score (AAS) path of
 * showlab/DiffSim.  Every entry point names the reference lines it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions
 *   - return value: DS_OK (0) on success, a negative DS_ERR_* otherwise.  Nothing
 *     is thrown across the ABI.  ds_last_error() returns a thread-local message
 *     describing the last failure on the calling thread.
 *   - ownership: the caller owns every buffer.  The library allocates no device
 *     memory; scratch space is sized with ds_*_workspace_bytes() and passed in.
 *   - pointers are DEVICE pointers unless the name ends in _host.
 *   - all work is enqueued on the caller's stream (a cudaStream_t passed as
 *     void*); there are no hidden synchronisations.
 *   - there is NO CPU fallback: without a CUDA device of compute capability 10.x
 *     every compute entry point fails with DS_ERR_CUDA / DS_ERR_UNSUPPORTED.
 *   - tensors are described by sizes and ELEMENT strides, so the reference's
 *     non-contiguous (B,H,S,D) views over (B,S,H*D) memory
 *     (diffsim/hacked_attn.py:74-77) and DiT's packed qkv
 *     (diffsim/diffsim_dit.py:22-23) are consumed in place, without copies.
 */
#ifndef DIFFSIM_B200_H_
#define DIFFSIM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DS_ABI_VERSION 1

/* error codes */
#define DS_OK               0
#define DS_ERR_INVALID     -1   /* bad argument (shape, stride, alignment, null) */
#define DS_ERR_UNSUPPORTED -2   /* valid request this build has no kernel for     */
#define DS_ERR_CUDA        -3   /* CUDA runtime / driver error, or no sm_100 GPU   */
#define DS_ERR_WORKSPACE   -4   /* workspace missing or too small                  */

/* element types */
#define DS_F16  0
#define DS_BF16 1
#define DS_F32  2

/* similarity modes (diffsim/diffsim.py:182-195, metrics/diffeats.py:136-140,202-205,
 * metrics/clip_i.py:92-96, metrics/dino.py:87-91) */
#define DS_SIM_COSINE        0  /* sum(x*y) / (max(|x|,1e-8) * max(|y|,1e-8))   */
#define DS_SIM_MSE           1  /* mean((x-y)^2)                                 */
#define DS_SIM_MINMAX_COSINE 2  /* cosine of the min-max normalised vectors      */

/* (B,H,S,D) tensor of one image; stride[3] must be 1. */
typedef struct ds_tensor4 {
  void*   ptr;
  int64_t size[4];
  int64_t stride[4];   /* in elements */
  int32_t dtype;       /* DS_F16 | DS_BF16 */
} ds_tensor4;

/* (N,B,H,S,D) stack of N images (a Q, K or V cache); stride[4] must be 1. */
typedef struct ds_tensor5 {
  void*   ptr;
  int64_t size[5];
  int64_t stride[5];   /* in elements */
  int32_t dtype;       /* DS_F16 | DS_BF16 */
} ds_tensor5;

/* ---- housekeeping ------------------------------------------------------- */

int         ds_abi_version(void);
const char* ds_last_error(void);
/* Device check: DS_OK iff the current device is compute capability 10.x. */
int         ds_device_ok(void);

/*
 * Optional in-stream timing of the dominant kernel (the fused attention): when enabled, every
 * attention launch is bracketed by cudaEventRecord on the caller's stream (up to 256 launches are
 * kept).  ds_profile_collect waits for the recorded launches, returns their summed device time and
 * count, and resets the ring.  Used by bench.py for the roofline figure; off by default.
 */
int ds_profile_enable(int on);
int ds_profile_collect(float* total_ms, int* launches);

/*
 * Debug only: device buffer of 8 x cap + 1 64-bit words.  A library built with -DDS_TRACE fills the first
 * 8 x cap words with (tag << 48 | SM clock) events of CTA 0 of the attention kernel; every build stores the SM
 * clocks CTA 0 spent in the last attention launch in word [8 x cap].  Returns 1 if tracing is compiled in, else 0.
 */
int ds_debug_set_trace(void* dev_buf, int cap);
/* Debug / A-B only: GEMM kernel behind ds_qkv_project and ds_simmat: -1 automatic (default), 0 the 1-CTA 128x256 kernel
 * only, 2 the CTA-pair (cta_group::2, 256x256) kernel always.  Adding 16 to 0 / 2 (or passing -17 for automatic) selects
 * the epilogue without TMA stores. */
int ds_debug_set_gemm_variant(int variant);
/* Debug / A-B only: longest k range (in 64-element blocks, >= 8) one fp32 partial of ds_simmat may cover (default 256).
 * Shorter ranges mean more partials (HBM traffic) but a smaller L2 working set and a shorter truncating accumulation
 * chain.  Returns the value in force. */
int ds_debug_set_simmat_max_kb(int kb);
/* Debug / A-B only: K1's K/V multicast over CTA pairs (clusters of two CTAs on the q tiles 2j, 2j + 1 of one (group, b, h),
 * every K/V tile read from L2 once for both): -1 automatic (default: ds_aas_matrix only, where it measures +2-3%), 0 off,
 * 1 on in every call whose q tile count is even.  Returns the value in force. */
int ds_debug_set_attn_mc(int mode);
/* Debug / A-B only: granularity (0, 64, 128 or 256 bytes) at which the L2 fetches a missing row piece of K1's Q / K / V TMA
 * boxes from DRAM.  Returns the value in force. */
int ds_debug_set_attn_l2_promotion(int bytes);
/* Debug / experiments only: cap K1's persistent grid at `ctas` CTAs (0 = default, one CTA per SM) -- how the clocks per item
 * depend on how loaded the chip is.  Returns the value in force. */
int ds_debug_set_attn_grid(int ctas);
/* Debug / A-B only: whether ds_simmat's statistics pass also writes k-blocked operand copies for the CTA-pair GEMM:
 * -1 automatic (default: when the operands exceed 512 MB), 0 never, 1 whenever the pair kernel runs.  Returns the value
 * in force. */
int ds_debug_set_simmat_blocked(int mode);

/* ---- K1: attention ------------------------------------------------------ */

/*
 * out = softmax(q k^T * scale) v   per (b,h); non-causal, no mask, no dropout.
 * Replaces F.scaled_dot_product_attention(q,k,v,dropout_p=0.0,is_causal=False)
 * at diffsim/hacked_attn.py:81-83 and diffsim/diffsim.py:177-180.
 * q:(B,H,Sq,D) k,v:(B,H,Skv,D) out:(B,H,Sq,D); scale <= 0 selects 1/sqrt(D).
 * out has the dtype of q (as torch's SDPA does).
 */
int ds_attn_fwd(ds_tensor4 q, ds_tensor4 k, ds_tensor4 v, float scale,
                ds_tensor4 out, void* ws, size_t ws_bytes, void* stream);
size_t ds_attn_fwd_workspace_bytes(ds_tensor4 q, ds_tensor4 k);

/*
 * Grouped Aligned Attention Score -- the fused replacement for the tail of
 * DiffSim.diffsim (diffsim/diffsim.py:177-197; copies diffsim_xl.py:135-155,
 * diffsim_dit.py:130-142).
 *
 * Images live in Q/K/V caches of N images.  Group g has one query image
 * group_q[g] and the kv images kv_idx[group_off[g] .. group_off[g+1]).  For
 * every entry t of group g the library computes the DIRECTIONAL similarity
 *     dir[t] = sim( Attn(Q_i, K_j, V_j), Attn(Q_i, K_i, V_i) ),
 *     i = group_q[g], j = kv_idx[t]
 * where the self attention Attn(Q_i,K_i,V_i) is evaluated once per group and
 * never leaves the chip.  Attention outputs are rounded to the input dtype
 * before the reduction, as the reference's SDPA outputs are; the reduction
 * accumulates in fp32 in a fixed order (deterministic, independent of how the
 * work is split over SMs or GPUs).
 *
 * (q, k_self, v_self) are indexed by group_q; (k, v) are indexed by kv_idx.
 * For ordinary pair scoring pass k_self = k and v_self = v.
 * mode: DS_SIM_COSINE | DS_SIM_MSE.   dir: float[n_entries].
 */
int ds_aas_groups(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self,
                  ds_tensor5 k, ds_tensor5 v,
                  const int32_t* group_q, const int32_t* group_off, int64_t n_groups,
                  const int32_t* kv_idx, int64_t n_entries,
                  float scale, int mode, float* dir,
                  void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_groups_workspace_bytes(ds_tensor5 q, int64_t n_groups, int64_t n_entries);

/*
 * score[p] = ( dir(a->b) + dir(b->a) ) / 2   for pair_idx[p] = (a,b):
 * exactly the value DiffSim.diffsim returns (diffsim/diffsim.py:197) for the
 * images a and b of the cache.  pair_idx: int32[P][2] on the device.
 */
int ds_aas_pairs(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v,
                 const int32_t* pair_idx, int64_t n_pairs,
                 float scale, int mode, float* scores,
                 void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_pairs_workspace_bytes(ds_tensor5 q, int64_t n_pairs);

/*
 * 2AFC triplets as the benchmark drivers score them (cute_main.py:111-132,196-205;
 * night_main.py:157-163): for trip_idx[t] = (ref, left, right)
 *     ab[t] = DiffSim.diffsim(ref, left),  ac[t] = DiffSim.diffsim(ref, right)
 * plus the decision counts of ds_twoafc.  The reference image's queries and self
 * attention are shared by both pairs (7 attentions per triplet instead of the
 * reference's 8; the reference recomputes image A, cute_main.py:111-132).
 * flags_out (optional): uint8[n] per-triplet "correct".  counts: int32[2].
 * opts: DS_OPT_ROUND_SCORES rounds every directional similarity and the pair
 * score to the input dtype before comparing, emulating the dtype of the
 * reference's score tensors (diffsim/diffsim.py:187-197 return fp16/bf16).
 */
#define DS_OPT_ROUND_SCORES 1
int ds_aas_triplets(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v,
                    const int32_t* trip_idx, int64_t n_triplets,
                    float scale, int mode, int opts,
                    float* ab, float* ac, int32_t* counts, uint8_t* flags_out,
                    void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_triplets_workspace_bytes(ds_tensor5 q, int64_t n_triplets);

/*
 * Directional score matrix for retrieval (SURVEY 8 a9; the reference only
 * ships the consumer of its output, retrieval_vis.py:57-68):
 *     Dm[r*ldd + c] = dir(row image r -> column image c)
 * rows: (q, k_self, v_self) of Nr images; columns: (k, v) of Nc images.
 * The symmetric score is S = (Dm + Dm^T)/2 over a square index set.
 * Row-block sharding over GPUs calls this with the local rows and all columns.
 */
int ds_aas_matrix(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self,
                  ds_tensor5 k, ds_tensor5 v,
                  float scale, int mode, float* Dm, int64_t ldd,
                  void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_matrix_workspace_bytes(ds_tensor5 q, ds_tensor5 k);

/* ---- K5: gradients ------------------------------------------------------ */

/*
 * Backward of ds_attn_fwd (of F.scaled_dot_product_attention without mask or
 * dropout): given out = ds_attn_fwd(q, k, v, scale) and dout = dL/dout,
 *     dq += dL/dq,  dk += dL/dk,  dv += dL/dv.
 * q, k, v, out, dout: 16-bit tensors as in ds_attn_fwd (any strides with a unit
 * innermost one).  dq, dk, dv: FLOAT32 tensors of q's / k's / v's shape that the
 * call ADDS INTO (so several calls accumulate in fp32 in a fixed order).  No
 * float atomics: the result is bitwise reproducible.  Head dims 40, 64, 72,
 * 80, 128, 160.
 */
int ds_attn_bwd(ds_tensor4 q, ds_tensor4 k, ds_tensor4 v, ds_tensor4 out, ds_tensor4 dout, float scale,
                ds_tensor4 dq, ds_tensor4 dk, ds_tensor4 dv, void* ws, size_t ws_bytes, void* stream);
size_t ds_attn_bwd_workspace_bytes(ds_tensor4 q, ds_tensor4 k);

/*
 * Backward of the directional similarity of ds_aas_groups,
 *     dir = sim( Attn(q_i, k_j, v_j), Attn(q_i, k_i, v_i) )   (mode DS_SIM_COSINE | DS_SIM_MSE),
 * with both attention outputs rounded to the input dtype as in the forward and
 * the rounding passed straight through.  d_dir: ONE float on the device (dL/ddir;
 * read there, no host synchronisation).  The five FLOAT32 gradients are added
 * into; they may alias (dk_i = dk_j when image i is image j).  dq_i receives
 * the cross term before the self term.
 */
int ds_aas_dir_bwd(ds_tensor4 q_i, ds_tensor4 k_i, ds_tensor4 v_i, ds_tensor4 k_j, ds_tensor4 v_j,
                   float scale, int mode, const float* d_dir,
                   ds_tensor4 dq_i, ds_tensor4 dk_i, ds_tensor4 dv_i, ds_tensor4 dk_j, ds_tensor4 dv_j,
                   void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_dir_bwd_workspace_bytes(ds_tensor4 q_i, ds_tensor4 k_j);

/* ---- K2: similarity reductions ----------------------------------------- */

/*
 * out[p] = sim(x[p,:], y[p,:]) over E elements, for n_pairs rows.
 * Replaces F.cosine_similarity(x.reshape(-1).unsqueeze(0), y.reshape(-1).unsqueeze(0))
 * (diffsim/diffsim.py:187-188, metrics/clip_i.py:156-157,183, metrics/dino.py:158-159,183,
 * metrics/vgg_gram.py:81), F.mse_loss (diffsim/diffsim.py:194-195) and
 * min_max_normalize + cosine (metrics/diffeats.py:136-140,202-205).
 * x_stride / y_stride: elements between consecutive rows (>= E, multiple of
 * 16 bytes); dtype DS_F16 | DS_BF16 | DS_F32; out: float[n_pairs].
 */
int ds_pair_reduce(const void* x, const void* y, int64_t n_pairs, int64_t E,
                   int64_t x_stride, int64_t y_stride, int dtype, int mode,
                   float* out, void* ws, size_t ws_bytes, void* stream);
size_t ds_pair_reduce_workspace_bytes(int64_t n_pairs, int64_t E);

/* ---- K3: N x N similarity matrix of feature vectors --------------------- */

/*
 * C[r*ldc + c] = sim(rows[r,:], cols[c,:])   (DS_SIM_COSINE | DS_SIM_MINMAX_COSINE)
 * rows: [Nr, L], cols: [Nc, L] 16-bit features (leading dimensions ld_rows,
 * ld_cols in elements, multiples of 8).  One tensor-core GEMM rows x cols^T
 * with fp32 accumulation; the per-vector statistics are a single HBM pass.
 * All-pairs form of the flat-cosine metrics (metrics/diffeats.py:202-205,
 * metrics/clip_i.py:183, metrics/dino.py:183, metrics/vgg_gram.py:81).
 */
int ds_simmat(const void* rows, int64_t n_rows, int64_t ld_rows,
              const void* cols, int64_t n_cols, int64_t ld_cols,
              int64_t L, int dtype, int mode, float* C, int64_t ldc,
              void* ws, size_t ws_bytes, void* stream);
size_t ds_simmat_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t L);

/* ---- K4: QKV projection of the hooked layer ------------------------------ */

/*
 * [out_0 | out_1 | out_2][r, :] = hidden[r, :] . weight^T (+ bias),  r < n_rows
 * The capture step of the reference, on the hook's input: attn.to_q / to_k / to_v
 * (diffsim/hacked_attn.py:61-69; the head split of :74-77 is a view of the output rows)
 * and DiT's fused module.qkv(x) (diffsim/diffsim_dit.py:21-23).
 * hidden: [n_rows, c_in] (n_rows = images * B * S), weight: [n_out, c_in] in nn.Linear
 * layout -- for separate to_q/to_k/to_v modules the three weights stacked along dim 0 --,
 * bias: [n_out] or null, all of `dtype` (DS_F16 | DS_BF16).  Output column n goes to
 * out[n / cols_per_out] at column n % cols_per_out, row stride ld_out[.] elements:
 * SD: n_out = 3C, cols_per_out = C, three (rows, C) tensors = the Q / K / V caches;
 * DiT: cols_per_out = n_out = 3C, one packed (rows, 3C) tensor.
 * fp32 accumulation, bias added in fp32, one rounding to `dtype`.  No workspace.
 */
int ds_qkv_project(const void* hidden, int64_t n_rows, int64_t ld_hidden, int64_t c_in,
                   const void* weight, int64_t ld_weight, const void* bias,
                   int64_t n_out, int64_t cols_per_out,
                   void* const* out, const int64_t* ld_out, int dtype, void* stream);

/* ---- decisions ---------------------------------------------------------- */

/*
 * 2AFC decision of the benchmark drivers (cute_main.py:196-205,
 * night_main.py:157-163): for triplet t with scores ab[t], ac[t]
 *   cosine: correct = ab > ac, correct2x = ab > 2*ac
 *   mse   : correct = ab < ac, correct2x = 2*ab < ac
 * counts: int32[2] = {sum correct, sum correct2x}; flags (optional, may be
 * null): uint8[n] per-triplet "correct".  One launch, no host sync.
 */
int ds_twoafc(const float* ab, const float* ac, int64_t n, int mode,
              int32_t* counts, uint8_t* flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFSIM_B200_H_ */
