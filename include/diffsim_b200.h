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
/*
 * Test hooks: each forces one side of an automatic kernel choice, so that tests can compare both sides bitwise.  -1
 * restores the automatic choice (the default); any other value not listed is ignored.  Each returns the value in force.
 */
/* GEMM kernel behind ds_qkv_project, both products of ds_qkv_project_bwd and ds_simmat: 0 the 1-CTA 128x256 kernel only,
 * 2 the CTA-pair (cta_group::2, 256x256) kernel always. */
int ds_debug_set_gemm_variant(int variant);
/* K1's K/V multicast over CTA pairs (clusters of two CTAs on the q tiles 2j, 2j + 1 of one (group, b, h), every K/V tile
 * read from L2 once for both; automatic: ds_aas_matrix only, where it measures +2-3%): 0 off, 1 on in every call whose
 * q tile count is even. */
int ds_debug_set_attn_mc(int mode);
/* Whether ds_simmat's statistics pass also writes k-blocked operand copies for the CTA-pair GEMM (automatic: when an
 * operand reaches 1.5 GB): 0 never, 1 whenever the pair kernel runs. */
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
 * Lengths: (k_self, v_self) share one kv length S_self and (k, v) one kv
 * length S_cross; both are independent of q's S_q (for AAS S_self is S_q, the
 * query image's own token count, and S_cross that of the other images: two
 * captures at different resolutions score against each other).  B, H, D and
 * the dtype match across all five.  k_self / v_self (k / v) of different
 * lengths are DS_ERR_INVALID.
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
 * The kv lengths of rows and columns may differ, as in ds_aas_groups.
 * The symmetric score is S = (Dm + Dm^T)/2 over a square index set; between
 * two image sets A and B it is (Dm(A->B) + Dm(B->A)^T)/2.
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
 * the cross term before the self term.  k_i / v_i and k_j / v_j may have
 * different kv lengths (each pair one length), independent of q_i's.
 */
int ds_aas_dir_bwd(ds_tensor4 q_i, ds_tensor4 k_i, ds_tensor4 v_i, ds_tensor4 k_j, ds_tensor4 v_j,
                   float scale, int mode, const float* d_dir,
                   ds_tensor4 dq_i, ds_tensor4 dk_i, ds_tensor4 dv_i, ds_tensor4 dk_j, ds_tensor4 dv_j,
                   void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_dir_bwd_workspace_bytes(ds_tensor4 q_i, ds_tensor4 k_j);

/*
 * Backward of ds_aas_groups (the directional similarities dir[t] of a whole work list) for d_dir = dL/ddir, float[n_entries]
 * on the device.  Same arguments as ds_aas_groups; the five FLOAT32 (N,B,H,S,D) gradients (of q, k_self, v_self, k, v;
 * any strides with a unit innermost one) are ADDED INTO.  dk_self / dk, and dv_self / dv, are either the same tensor
 * (same pointer, sizes and strides: the pairs / triplets case, where k_self is k) or have disjoint address ranges.
 * The kv lengths follow ds_aas_groups: S_self for (k_self, v_self), S_cross for (k, v); every term walks its own length
 * (shared gradient buffers imply S_self = S_cross).
 *
 * Bitwise contract: the buffers end up exactly as after one ds_aas_dir_bwd call per entry, t = 0 .. n_entries - 1 in order,
 * on the slices (q, k_self, v_self)[group_q[g(t)]], (k, v)[kv_idx[t]], d_dir + t and the matching gradient slices: every
 * gradient row receives its terms in that order (entry, then cross term before self term) with the same arithmetic.
 * One K1 launch recomputes every X_t and Y_g; one dQ launch (a CTA per query image, b, h and 128-row q tile) and one dK/dV
 * launch (per kv image, b, h, 128-row kv tile) walk contribution lists built on the device.  No float atomics, no host
 * synchronisation.  An out-of-range image index fills every gradient buffer of the call with NaN.  Workspace: about
 * (3 n_entries + n_groups) x B H S D x 2 bytes.
 */
int ds_aas_groups_bwd(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v,
                      const int32_t* group_q, const int32_t* group_off, int64_t n_groups,
                      const int32_t* kv_idx, int64_t n_entries, float scale, int mode,
                      const float* d_dir,
                      ds_tensor5 dq, ds_tensor5 dk_self, ds_tensor5 dv_self, ds_tensor5 dk, ds_tensor5 dv,
                      void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_groups_bwd_workspace_bytes(ds_tensor5 q, ds_tensor5 k, int64_t n_groups, int64_t n_entries);

/*
 * Backward of ds_aas_pairs for d_scores = dL/dscore (float[n_pairs] on the device): ds_aas_groups_bwd on the pairs'
 * work list with d_dir[2p] = d_dir[2p+1] = d_scores[p] / 2.  dq, dk, dv: FLOAT32 gradients of q, k, v, added into.
 */
int ds_aas_pairs_bwd(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* pair_idx, int64_t n_pairs,
                     float scale, int mode, const float* d_scores,
                     ds_tensor5 dq, ds_tensor5 dk, ds_tensor5 dv, void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_pairs_bwd_workspace_bytes(ds_tensor5 q, int64_t n_pairs);

/*
 * Backward of the scores ab, ac of ds_aas_triplets (without DS_OPT_ROUND_SCORES; with it, the rounding passes straight
 * through) for d_ab, d_ac (float[n_triplets] each, on the device): entries 4t .. 4t+3 of the triplets' work list are
 * ref->left, ref->right, left->ref, right->ref, so d_dir = (d_ab, d_ac, d_ab, d_ac)[t] / 2.
 */
int ds_aas_triplets_bwd(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* trip_idx, int64_t n_triplets,
                        float scale, int mode, const float* d_ab, const float* d_ac,
                        ds_tensor5 dq, ds_tensor5 dk, ds_tensor5 dv, void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_triplets_bwd_workspace_bytes(ds_tensor5 q, int64_t n_triplets);

/*
 * Backward of ds_aas_matrix for d_Dm[r*ldd + c] = dL/dDm[r, c] (float, Nr rows of Nc values, on the device; read there,
 * no host synchronisation).  Same operands as ds_aas_matrix; the five FLOAT32 (N,B,H,S,D) gradients (of q, k_self,
 * v_self, k, v; any strides with a unit innermost one) are ADDED INTO, with the aliasing rule of ds_aas_groups_bwd:
 * dk_self / dk (dv_self / dv) are the same tensor or have disjoint address ranges.  The rows' and the columns' kv
 * lengths may differ, as in ds_aas_matrix.
 *
 * It is the grouped backward of the row-major matrix list (group r = row r, entries (r, c) for c = 0 .. Nc-1), except
 * that the Nc self terms of row r -- Attn(q_r, k_self_r, v_self_r) with dO = coef_self_rc fy_rc -- are FOLDED into one
 * attention backward with dO = F_r = sum_c coef_self_rc fy_rc (fp32, ascending c, fy unrounded), rounded once to the input
 * dtype after a per-row power-of-two scale: Nr Nc + Nr attention backwards instead of 2 Nr Nc.
 * Term order of every gradient row: ascending row r, the cross terms of row r in ascending column, then the folded self
 * term of row r.  So dk and dv, when they are not dk_self and dv_self, are bitwise those of ds_aas_groups_bwd on the
 * row-major list.  No float atomics: repeated calls are bitwise equal.  At most 2^29 entries (the lists' term index is an
 * int32).  Workspace: per entry about 2 x B H S D x 2 bytes (X, fx) plus 3 KB of partials; per row about B H S D x 8
 * bytes (Y, F_r in 16 and 32 bits); LSE and delta for every entry and row.
 *
 * Gradient families: the ROW terms (dq of every term; dk_self, dv_self of the folded self terms) and the COLUMN terms
 * (dk, dv of the cross terms).  A family whose pointers are all null is not computed: (dq, dk_self, dv_self) all null, or
 * (dk, dv) both null, not both.  A partly null family is DS_ERR_INVALID, and so is dk_self / dk (dv_self / dv) as one
 * tensor unless all five are given.  Only the work of the given family runs: without the column terms the dK/dV kernel
 * runs the folded self terms only; without the row terms nothing is folded, and the dQ kernel writes only the cross
 * terms' LSE and delta.  Every per-term quantity depends only on its entry (r, c) and its row r, so each family alone is
 * bitwise what the full call gives it with separate self buffers.  The rows [r0, r1) against all columns and all rows
 * against the columns [c0, c1) thus give bitwise the full call's gradients of those images.  The workspace query is
 * that of the full call (an upper bound).
 */
int ds_aas_matrix_bwd(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v,
                      float scale, int mode, const float* d_Dm, int64_t ldd,
                      ds_tensor5 dq, ds_tensor5 dk_self, ds_tensor5 dv_self, ds_tensor5 dk, ds_tensor5 dv,
                      void* ws, size_t ws_bytes, void* stream);
size_t ds_aas_matrix_bwd_workspace_bytes(ds_tensor5 q, ds_tensor5 k);

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

/*
 * Backward of ds_pair_reduce: for row p with g = d_out[p] (float[n_pairs] on the device, no host sync), the gradients
 * of out[p] that float64 torch autograd gives on the same inputs:
 *   cosine  s = x.y / (nx ny), n = max(|.|, 1e-8):  dx = g (y / (nx ny) - s x / (nx |x|)), the second term 0 when
 *           |x| = 0 (torch clamps the norm without a gradient); dy symmetric.
 *   mse     dx = 2 g (x - y) / E,  dy = -dx.
 *   minmax  x^ = (x - m) / (M - m) with the row's min m and max M, G = dcos/dx^ by the cosine rule:
 *           dx = g (G / (M - m) + [x = m] S_m / n_m + [x = M] S_M / n_M),
 *           S_m = sum G (x^ - 1) / (M - m), S_M = -sum G x^ / (M - m), n_m / n_M the numbers of elements equal to m / M
 *           (t.min() / t.max() split the gradient evenly among ties); dy symmetric.  A constant row (M = m) has a NaN
 *           score and gets NaN gradients in that row only.
 * x, y, n_pairs, E, strides, dtype and mode as for ds_pair_reduce.  dx, dy: float[n_pairs, E] with row strides
 * dx_stride, dy_stride (>= E) elements, written (not added into); either may be null (not computed), and both null is
 * DS_OK and does nothing.  Launches: a counter memset, a statistics pass (the forward's reduction plus min / max tie
 * counts) and one elementwise gradient pass; mse runs the gradient pass only.  No float atomics: repeated calls are
 * bitwise equal.
 */
size_t ds_pair_reduce_bwd_workspace_bytes(int64_t n_pairs, int64_t E);
int ds_pair_reduce_bwd(const void* x, const void* y, int64_t n_pairs, int64_t E, int64_t x_stride, int64_t y_stride,
                       int dtype, int mode, const float* d_out,
                       float* dx, int64_t dx_stride, float* dy, int64_t dy_stride,
                       void* ws, size_t ws_bytes, void* stream);

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

/*
 * Backward of ds_qkv_project for the gradient dy of its outputs (the same hidden / weight / n_out / cols_per_out):
 *   dhidden = dY . weight  [n_rows, c_in]    dweight = dY^T . hidden  [n_out, c_in]    dbias = sum over rows of dY  [n_out]
 * where dY[r, n] = dy[n / cols_per_out][r, n % cols_per_out]: n_out / cols_per_out tensors of n_rows x cols_per_out,
 * row stride ld_dy[.] elements, read in place.  Each of dhidden (row stride ld_dhidden), dweight (ld_dweight) and dbias
 * may be null: not wanted, not computed; hidden may be null when dweight is, weight when dhidden is.  Outputs are of
 * `dtype`, written (not added into): fp32 accumulation, split-K partials added in a fixed order, one rounding --
 * bitwise reproducible, no atomics.  Launches: 2 per wanted output (product or column sums, then its finish).
 */
size_t ds_qkv_project_bwd_workspace_bytes(int64_t n_rows, int64_t c_in, int64_t n_out, int64_t cols_per_out);
int ds_qkv_project_bwd(const void* hidden, int64_t n_rows, int64_t ld_hidden, int64_t c_in,
                       const void* weight, int64_t ld_weight, int64_t n_out, int64_t cols_per_out,
                       const void* const* dy, const int64_t* ld_dy,
                       void* dhidden, int64_t ld_dhidden, void* dweight, int64_t ld_dweight, void* dbias,
                       int dtype, void* ws, size_t ws_bytes, void* stream);

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
