// K1 -- fused cross-image attention + similarity epilogue (tensor-core bound).
//
// One persistent, warp-specialised CTA per SM:
//
//   warp 0        TMA producer   Q tile (per stream) and a ring of 128-row K / V stages
//   warp 1        MMA issuer     tcgen05.mma: S = Q K^T (fp32, TMEM), O (+)= P V (fp32, TMEM; P read from TMEM);
//                                also allocates / frees TMEM
//   warps 10-25   softmax        512 threads; thread = (q row, 32 of the 128 kv columns of an S half);
//                                S (TMEM) -> exp2 -> P (16-bit, written IN PLACE over S: the A operand of PV)
//   warps 2-9     epilogue       256 threads; thread = (q row, half of the head dim); O (TMEM) -> 1/l ->
//                                  self item : O_self rounded to the input dtype, kept on chip (TMEM), |O_self|^2
//                                  cross item: dot(O_cross,O_self), |O_cross|^2 or sum (O_cross-O_self)^2
//                                  store mode: write O to global (the SDPA replacement)
//
// (O is single-buffered in TMEM -- 2 x 160 columns do not fit next to S -- so the time the epilogue needs to drain
// it sits on the critical path of the next item's first PV: hence eight epilogue warps, two per scheduler.)
//
// Work decomposition.  A "stream" is (group, b, h, 128-row q tile): the Q tile stays resident while the kv
// images of the group ("items") stream through; the first item of a group is the query image's own K/V (the
// self attention of diffsim/diffsim.py:179-180), whose output never leaves the SM.  An item is cut into kv
// GROUPS of 256 rows, a group into two HALVES (A, B) of 128 rows = one ring stage = one N=128 MMA slice with
// its own 128 TMEM columns.
//
// Why this shape: the kernel is bound by shared-memory bandwidth (128 B/clk/SM), not by the tensor pipe, as
// soon as operands are re-read from shared memory: an SS-mode MMA with N=64 reads 6 KB per 32 tensor-clocks.
// So S is produced by N=128 MMAs (Q is re-read only twice per item), P never touches shared memory (the
// softmax warps overwrite S in TMEM with 16-bit P and the PV MMA takes its A operand from TMEM), and O_self
// lives in TMEM as well.  Shared memory then carries only TMA writes + one read of K and V + two reads of Q.
//
// Softmax.  Online over 128-column halves with a LAZY running maximum: the first half of an item fixes the
// reference maximum m of every row; a later half only moves a row's m (and rescales its O and running sum) when the
// half's maximum exceeds m by more than tau = 14 (fp16) or 30 (bf16) in log2 units -- otherwise p = exp2(s - m) is
// simply allowed to grow up to 2^14 (fp16) or 2^30 (bf16), which 16-bit P and fp32 sums hold without loss.  The
// result is the exact softmax either way (any common offset cancels in O / l).  The rare rescale is done by the
// first-quarter softmax warps themselves before they release P, so the common path has no extra barrier and half A
// never waits for half B.
//
// Pipeline.  The MMA warp issues, in this fixed order, PV_A(u), QK_A(u+1), PV_B(u), QK_B(u+1): tcgen05 ops of
// one thread execute in issue order, so QK_A(u+1) may overwrite the columns PV_A(u) reads P from without any
// barrier; while the tensor core works on half A the softmax warps turn half B into P.  The TMA producer feeds
// the ring in the same order.
//
// Replaces diffsim/diffsim.py:177-197 (diffsim_xl.py:135-155, diffsim_dit.py:130-142).
// Algorithmic work per directional attention: 4*B*H*Sq*Skv*D flops.
#include "ds_attn_common.cuh"

namespace ds {

// LIST: the store form of a grouped work list (the recompute of the AAS backward): every item's O is written, rounded as in
// STORE, to output slot g (the self item of group g) or n_groups + t (entry t) of a contiguous (slot, B, H, Sq, D) stack
enum : int { ATTN_MODE_COS = 0, ATTN_MODE_MSE = 1, ATTN_MODE_STORE = 2, ATTN_MODE_LIST = 3 };

constexpr int kAttnThreads = 832;   // 26 warps: producer, MMA, 8 epilogue, 16 softmax
constexpr int kWarpProducer = 0;
constexpr int kWarpMma = 1;
constexpr int kWarpSoftmax0 = 10;
constexpr int kBlockQ = 128;     // q rows per tile == TMEM lanes
constexpr int kHalfKV = 128;     // kv rows per S half == per ring stage
constexpr int kGroupKV = 256;    // kv rows per softmax group (two halves)
constexpr int kTmemCols = 512;
constexpr int kTmemS = 0;        // S_A: columns [0,128), S_B: [128,256); P of the thread's 32 kv columns
                                 // overwrites the first 16 of its own 32 S columns
constexpr int kTmemO = 256;      // O: [256, 256 + D_PAD)
constexpr int kTmemOs = 416;     // O_self, packed 16-bit: [416, 416 + D_PAD/2)
constexpr int kTmemL = 496;      // softmax denominators l = P . 1 (a 16-column MMA against a constant ones tile): [496,512)

template <int D>
struct AttnCfg : AttnTile<D> {
  using Tile = AttnTile<D>;
  // Every POLY_STRIDE-th pair of exponentials is evaluated with a degree-3 polynomial on the FMA pipe instead of MUFU
  // (0: none).  With head dims <= 80 an item carries at most half the tensor work of D = 160 but the same 32 768
  // exponentials, and long-kv streams of such items are MUFU-bound: measured +13% on SDXL (2,20,1024,64) / (2,10,4096,64),
  // +6% on SD-1.5 up1 / up2, neutral on DiT-XL/2, and -4% at D = 160 (profiles/r1z_poly_shapes.txt).
  static constexpr int POLY_STRIDE = D <= 80 ? 3 : 0;
  static constexpr int Q_SUB_BYTES = kBlockQ * Tile::SUB_BYTES;
  static constexpr int Q_BYTES = Tile::NSUB * Q_SUB_BYTES;
  static constexpr int KV_SUB_BYTES = kHalfKV * Tile::SUB_BYTES;
  static constexpr int STAGE_BYTES = Tile::NSUB * KV_SUB_BYTES;
  static constexpr int MISC_BYTES = 2048 /*ones tile*/ + 4096 /*max exchange*/ + 128 /*epilogue reduce*/ + 512 /*barriers*/;
  static constexpr int kMaxSmem = 232448;
  static constexpr int STAGES_RAW = (kMaxSmem - Q_BYTES - MISC_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 12 ? 12 : STAGES_RAW;
  static constexpr int SMEM_BYTES = Q_BYTES + STAGES * STAGE_BYTES + MISC_BYTES;
  static_assert(STAGES >= 4, "not enough shared memory for the K/V ring");
  static_assert(kTmemO + Tile::D_PAD <= kTmemOs && kTmemOs + Tile::D_PAD / 2 <= kTmemL, "TMEM budget");
  static_assert(Q_BYTES % 1024 == 0 && STAGE_BYTES % 1024 == 0, "swizzle atoms need 1024-byte aligned tiles");
};

struct AttnParams {
  // group description (device pointers)
  const int32_t* group_q;    // [n_groups] query image of each group
  const int32_t* group_off;  // [n_groups + 1] entry range of each group
  const int32_t* kv_idx;     // [n_entries] kv image of each entry
  int n_groups;
  int self_first;            // 1: every group starts with the query image's own K/V (AAS)
  int B, H, Sq, Skv;         // Skv: kv length of the cross items (k, v)
  int Skv_self;              // kv length of the self item (k_self, v_self); independent of Sq and of Skv
  // kv groups of a cross item / of the self item, and the valid rows of the two halves of their last group (set by the
  // host: the walkers select them per item and divide nothing)
  int n_grp, rowsA_last, rowsB_last;
  int n_grp_self, rowsA_last_self, rowsB_last_self;
  int n_qt;                  // q tiles per (b,h)
  float scale_log2;          // softmax scale * log2(e)
  // AAS output: part[entry][bh * n_qt + qt] = (dot, |Oc|^2, |Os|^2, sum (Oc-Os)^2)
  float4* part;
  // store-mode output: element strides of (b, h, s); the innermost stride is 1
  void* out;
  int64_t out_sb, out_sh, out_ss;
  // debug timeline (ds_debug_set_trace; compiled in only with -DDS_TRACE): [8 slots][cap] of (tag << 48 | clock)
  unsigned long long* trace;
  int trace_cap;
  // 1: the kernel runs as clusters of two CTAs that work on the two q tiles (2j, 2j + 1) of the same (group, b, h) -- the
  // same K/V sequence -- and load every K/V tile ONCE for both (TMA multicast, alternating which CTA issues a load)
  int mc;
  unsigned long long* cycles;   // optional: CTA 0 stores its elapsed SM clocks here (ds_debug_set_trace(buf, cap): buf[8*cap])
};

#ifdef DS_TRACE
#define DS_TRACE_DECL(slot) int _tr_n = 0; const int _tr_slot = (slot); const bool _tr_on = p.trace && blockIdx.x == 0;
#define DS_TRACE_EV(tag)                                                                                   \
  do {                                                                                                     \
    if (_tr_on && _tr_n < p.trace_cap)                                                                     \
      p.trace[(size_t)_tr_slot * p.trace_cap + _tr_n++] = ((unsigned long long)(tag) << 48) | (clock64() & 0xFFFFFFFFFFFFull); \
  } while (0)
#else
#define DS_TRACE_DECL(slot)
#define DS_TRACE_EV(tag)
#endif

// One kv group of one item of one stream, as every warp role enumerates them (identically).
struct GroupInfo {
  int b, h, qt, bh, qi, g;  // stream
  int img, entry;           // item: kv image, index into kv_idx / part (cross items)
  int kv0, rowsA, rowsB;    // group: first kv row, valid rows of the two halves
  bool self, first_of_stream, last_of_stream, first_of_item, last_of_item;
};

template <typename F>
__device__ __forceinline__ void for_each_group(const AttnParams& p, F&& f) {
  const uint32_t BH = (uint32_t)(p.B * p.H);
  const uint32_t n_streams = (uint32_t)p.n_groups * BH * (uint32_t)p.n_qt;   // < 2^31, checked by the host
  // stream -> (bh, group, q tile): q tile fastest so that neighbouring CTAs share K/V in L2.  32-bit arithmetic only:
  // this decode sits between two items on every role's critical path.
  for (uint32_t st = blockIdx.x; st < n_streams; st += gridDim.x) {
    GroupInfo G;
    const uint32_t r = st / (uint32_t)p.n_qt;
    G.qt = (int)(st - r * (uint32_t)p.n_qt);
    G.bh = (int)(r / (uint32_t)p.n_groups);
    const int g = (int)(r - (uint32_t)G.bh * (uint32_t)p.n_groups);
    G.g = g;
    G.b = G.bh / p.H;
    G.h = G.bh - G.b * p.H;
    // the work list lives in global memory and every role walks it between barriers the compiler cannot move loads
    // across: pull the entries of the NEXT stream / item into L1 now so that the dependent loads below hit
    if (st + gridDim.x < n_streams) {
      const uint32_t r_n = (st + gridDim.x) / (uint32_t)p.n_qt;
      const uint32_t g_n = r_n % (uint32_t)p.n_groups;
      prefetch_l1(p.group_q + g_n);
      prefetch_l1(p.group_off + g_n);
    }
    G.qi = p.group_q[g];
    const int t0 = p.group_off[g], t1 = p.group_off[g + 1];
    const int n_items = (t1 - t0) + p.self_first;
    for (int it = 0; it < n_items; ++it) {
      G.self = p.self_first && it == 0;
      G.entry = t0 + it - p.self_first;
      if (it + 1 < n_items) prefetch_l1(p.kv_idx + G.entry + 1);
      G.img = G.self ? G.qi : p.kv_idx[G.entry];
      const int skv = G.self ? p.Skv_self : p.Skv;   // each item is cut by its own kv length
      const int n_grp = G.self ? p.n_grp_self : p.n_grp;
      for (int gg = 0; gg < n_grp; ++gg) {
        G.kv0 = gg * kGroupKV;
        const int rem = skv - G.kv0;
        G.rowsA = min(rem, kHalfKV);
        G.rowsB = max(0, min(rem - kHalfKV, kHalfKV));
        G.first_of_item = gg == 0;
        G.last_of_item = gg == n_grp - 1;
        G.first_of_stream = it == 0 && gg == 0;
        G.last_of_stream = it == n_items - 1 && gg == n_grp - 1;
        f(G);
      }
    }
  }
}

// Light-weight enumeration for the roles that only need the SHAPE of the work (MMA issuer, softmax warps): per kv group the
// valid rows of its two halves and the first / last flags.  No divisions per stream -- (q tile, group) advance incrementally
// -- and one pair of (L1-prefetched) loads per stream for the group's item count.
struct LiteGroup {
  int rowsA, rowsB;
  bool first_of_stream, last_of_stream, first_of_item, last_of_item;
};

template <typename F>
__device__ __forceinline__ void for_each_group_lite(const AttnParams& p, F&& f) {
  const uint32_t nq = (uint32_t)p.n_qt, ng = (uint32_t)p.n_groups;
  const uint32_t n_streams = ng * (uint32_t)(p.B * p.H) * nq;   // < 2^31, checked by the host
  // stream st = (bh * n_groups + g) * n_qt + qt
  uint32_t qt = blockIdx.x % nq, g = (blockIdx.x / nq) % ng;
  const uint32_t d_qt = gridDim.x % nq, d_g = (gridDim.x / nq) % ng;
  for (uint32_t st = blockIdx.x; st < n_streams; st += gridDim.x) {
    const int n_items = p.group_off[g + 1] - p.group_off[g] + p.self_first;
    qt += d_qt;
    uint32_t carry = 0;
    if (qt >= nq) {
      qt -= nq;
      carry = 1;
    }
    g += d_g + carry;
    if (g >= ng) g -= ng;
    prefetch_l1(p.group_off + g);
    LiteGroup G;
    for (int it = 0; it < n_items; ++it) {
      // each item by its own kv length: the self item is item 0 of a self_first stream
      const bool self = it < p.self_first;
      const int n_grp = self ? p.n_grp_self : p.n_grp;
      const int rowsA_last = self ? p.rowsA_last_self : p.rowsA_last, rowsB_last = self ? p.rowsB_last_self : p.rowsB_last;
      for (int gg = 0; gg < n_grp; ++gg) {
        const bool last = gg == n_grp - 1;
        G.rowsA = last ? rowsA_last : kHalfKV;
        G.rowsB = last ? rowsB_last : kHalfKV;
        G.first_of_item = gg == 0;
        G.last_of_item = last;
        G.first_of_stream = it == 0 && gg == 0;
        G.last_of_stream = it == n_items - 1 && last;
        f(G);
      }
    }
  }
}

template <int D, bool kBf16, int MODE>
__global__ void __launch_bounds__(kAttnThreads, 1)
aas_attn_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_ks,
                const __grid_constant__ CUtensorMap map_vs, const __grid_constant__ CUtensorMap map_k,
                const __grid_constant__ CUtensorMap map_v, const AttnParams p) {
  using C = AttnCfg<D>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sRing = sQ + C::Q_BYTES;
  uint8_t* sOnes = sRing + C::STAGES * C::STAGE_BYTES;   // [16 rows][64] K-major tile: row 0 = 1.0, rows 1..15 = 0
  float* sMax = reinterpret_cast<float*>(sOnes + 2048);  // [2 parity][4 col quarter][128]
  float* sRed = sMax + 1024;                                                   // [2 parity][4 warps][4]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRed + 32);
  uint64_t* q_full = bars + 0;
  uint64_t* q_empty = bars + 1;
  uint64_t* s_full = bars + 2;      // [2] S half written by the tensor core
  uint64_t* p_full = bars + 4;      // [2] P half written (over S) by the softmax warps
  uint64_t* o_full = bars + 10;     // all PV of an item done: O complete (one phase per item)
  uint64_t* pv_half = bars + 12;    // PV of one half done (one phase per half; only the rare rescale path waits on it)
  uint64_t* o_empty = bars + 11;    // O read out by the epilogue warps
  uint64_t* kv_full = bars + 16;
  uint64_t* kv_empty = bars + 16 + C::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16 + 2 * C::STAGES);
  static_assert((16 + 2 * C::STAGES) * 8 + 16 <= 512, "barrier area");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long clk_start = clock64();

  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) {
    printf("diffsim_b200: dynamic shared memory is not 1024-byte aligned\n");
    __trap();
  }
  if (warp == kWarpProducer && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_ks);
    tma_prefetch_desc(&map_vs);
    tma_prefetch_desc(&map_k);
    tma_prefetch_desc(&map_v);
  }
  if (warp == kWarpMma && lane == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int h = 0; h < 2; ++h) {
      mbar_init(&s_full[h], 1);
      mbar_init(&p_full[h], 512);
    }
    mbar_init(o_full, 1);
    mbar_init(pv_half, 1);
    mbar_init(o_empty, 256);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], p.mc ? 2 : 1);   // multicast: a slot is free once BOTH CTAs' MMAs have read it
    }
    fence_mbar_init();
  }
  if (warp == kWarpMma) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  // constant B operand of the row-sum MMA: l[r] = sum_k P[r,k] * 1.  Row 0 of a 128B-swizzled K-major tile is not
  // permuted (its swizzle XOR is 0) and the other rows are all zero, so the fill is layout-trivial.
  if (threadIdx.x < 512) {
    const uint32_t one2 = kBf16 ? 0x3F803F80u : 0x3C003C00u;
    reinterpret_cast<uint32_t*>(sOnes)[threadIdx.x] = threadIdx.x < 32 ? one2 : 0u;
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  if (p.mc) cluster_sync_all();   // the peer's barriers are initialised before anything is multicast at them
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kWarpProducer) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0, sc = 0;
      // one ring stage = up to 128 kv rows (rows past the tensor end are zero-filled by TMA)
      DS_TRACE_DECL(0)
      const uint32_t mc_rank = p.mc ? cluster_ctarank() : 0u;
      uint32_t n_loads = 0;
      auto load_half = [&](const CUtensorMap* m, int img, int bb, int hh, int row0) {
        DS_TRACE_EV(1);
        mbar_wait(&kv_empty[stage], phase ^ 1);
        DS_TRACE_EV(2);
        uint8_t* dst = sRing + (size_t)stage * C::STAGE_BYTES;
        mbar_arrive_expect_tx(&kv_full[stage], C::STAGE_BYTES);
        if (p.mc) {
          // both CTAs walk the same K/V sequence: sub-tile s of load n is fetched by CTA (n + s) % 2 for both
#pragma unroll
          for (int s = 0; s < C::NSUB; ++s)
            if (((n_loads + s) & 1u) == mc_rank)
              tma_load_5d_mc(dst + s * C::KV_SUB_BYTES, m, &kv_full[stage], s * C::SUBW, row0, hh, bb, img, (uint16_t)3);
          ++n_loads;
        } else {
#pragma unroll
          for (int s = 0; s < C::NSUB; ++s)
            tma_load_5d(dst + s * C::KV_SUB_BYTES, m, &kv_full[stage], s * C::SUBW, row0, hh, bb, img);
        }
        if (++stage == C::STAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      GroupInfo prev = {};
      bool have_prev = false;
      for_each_group(p, [&](const GroupInfo& G) {
        // the order the MMA warp consumes the ring in: V_A(u-1), K_A(u), V_B(u-1), K_B(u).  V_A(u-1) goes first, BEFORE
        // the wait for the Q buffer: at a stream boundary that wait lasts until the old stream's last QK has completed,
        // and PV_A(u-1) must not queue behind it.
        if (have_prev) load_half(prev.self ? &map_vs : &map_v, prev.img, prev.b, prev.h, prev.kv0);
        if (G.first_of_stream) {
          DS_TRACE_EV(3);
          mbar_wait(q_empty, (sc & 1) ^ 1);
          mbar_arrive_expect_tx(q_full, C::Q_BYTES);
#pragma unroll
          for (int s = 0; s < C::NSUB; ++s)
            tma_load_5d(sQ + s * C::Q_SUB_BYTES, &map_q, q_full, s * C::SUBW, G.qt * kBlockQ, G.h, G.b, G.qi);
          ++sc;
          DS_TRACE_EV(4);
        }
        load_half(G.self ? &map_ks : &map_k, G.img, G.b, G.h, G.kv0);
        if (have_prev && prev.rowsB) load_half(prev.self ? &map_vs : &map_v, prev.img, prev.b, prev.h, prev.kv0 + kHalfKV);
        if (G.rowsB) load_half(G.self ? &map_ks : &map_k, G.img, G.b, G.h, G.kv0 + kHalfKV);
        prev = G;
        have_prev = true;
      });
      if (have_prev) {
        load_half(prev.self ? &map_vs : &map_v, prev.img, prev.b, prev.h, prev.kv0);
        if (prev.rowsB) load_half(prev.self ? &map_vs : &map_v, prev.img, prev.b, prev.h, prev.kv0 + kHalfKV);
      }
    }
  } else if (warp == kWarpMma) {
    // ------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      const uint32_t fmt = kBf16 ? 1u : 0u;
      const uint32_t idesc_pv = umma_idesc_f16(fmt, kBlockQ, C::D_PAD, 0, 1);
      const uint32_t idesc_l = umma_idesc_f16(fmt, kBlockQ, 16, 0, 0);
      const uint64_t ones_desc = umma_smem_desc(smem_u32(sOnes), 16, 1024, UMMA_SW128);
      constexpr uint32_t SBO = 8 * C::SUB_BYTES;  // eight swizzle rows
      // descriptors of the buffer bases; tiles are addressed by adding (byte offset >> 4) to the low word
      const uint64_t q_desc0 = umma_smem_desc(smem_u32(sQ), 16, SBO, C::LAYOUT);
      const uint64_t k_desc0 = umma_smem_desc(smem_u32(sRing), 16, SBO, C::LAYOUT);
      const uint64_t v_desc0 = umma_smem_desc(smem_u32(sRing), C::KV_SUB_BYTES, SBO, C::LAYOUT);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t pv_cntA = 0, pv_cntB = 0, sc = 0, items_pv = 0;
      auto advance = [&]() {
        if (++stage == C::STAGES) {
          stage = 0;
          phase ^= 1;
        }
      };
      // S_h = Q K_h^T: N = the half's kv rows rounded up to 16.  Overwrites the columns PV_h of the previous group
      // read P from: safe without a barrier because both are issued by this thread, in this order.
      DS_TRACE_DECL(1)
      auto issue_qk = [&](const LiteGroup& G, int h) {
        const int rows = h ? G.rowsB : G.rowsA;
        DS_TRACE_EV(10 + h);
        const uint32_t idesc_qk = umma_idesc_f16(fmt, kBlockQ, (uint32_t)((rows + 15) & ~15), 0, 0);
        if (h == 0 && G.first_of_stream) {
          DS_TRACE_EV(17);
          mbar_wait(q_full, sc & 1);
          ++sc;
          DS_TRACE_EV(18);
        }
        if (!mbar_test_wait(&kv_full[stage], phase)) mbar_wait(&kv_full[stage], phase);
        DS_TRACE_EV(12 + h);
        tc_fence_after_sync();
        const uint64_t k_desc = k_desc0 + (uint64_t)((stage * C::STAGE_BYTES) >> 4);
        const uint32_t d_tmem = tmem_base + kTmemS + h * kHalfKV;
#pragma unroll
        for (int kc = 0; kc < C::D_PAD / 16; ++kc) {
          const int sub = kc / C::CPS, off = (kc % C::CPS) * 32;
          umma_f16_ss(d_tmem, q_desc0 + (uint64_t)((sub * C::Q_SUB_BYTES + off) >> 4),
                      k_desc + (uint64_t)((sub * C::KV_SUB_BYTES + off) >> 4), idesc_qk, kc > 0 ? 1u : 0u);
        }
        if (p.mc) umma_commit_mc(&kv_empty[stage], (uint16_t)3);
        else umma_commit(&kv_empty[stage]);
        advance();
        umma_commit(&s_full[h]);
        DS_TRACE_EV(14 + h);
        if (G.last_of_stream && (h == 1 || G.rowsB == 0)) umma_commit(q_empty);
      };
      // O (+)= P_h V_h with P_h read from TMEM (written by the softmax warps over S_h)
      auto issue_pv = [&](const LiteGroup& G, int h) {
        const int rows = h ? G.rowsB : G.rowsA;
        DS_TRACE_EV(20 + h);
        {
          // the tensor queue hides only ~175 clk of this thread's time between two bursts (tools/ubench/ubench_k1_mma.cu), and
          // a wait costs 100+ clk even on a completed barrier: probe all barriers of the burst at once (the probes' latencies
          // overlap), then wait properly only on those that were not complete (-80 clk per item)
          const uint32_t par_p = (h ? pv_cntB : pv_cntA) & 1;
          const bool need_o = h == 0 && G.first_of_item;
          const bool ok_p = mbar_test_wait(&p_full[h], par_p);
          const bool ok_k = mbar_test_wait(&kv_full[stage], phase);
          const bool ok_o = need_o ? mbar_test_wait(o_empty, (items_pv & 1) ^ 1) : true;
          if (!ok_p) mbar_wait(&p_full[h], par_p);
          DS_TRACE_EV(22 + h);
          if (!ok_o) mbar_wait(o_empty, (items_pv & 1) ^ 1);
          if (!ok_k) mbar_wait(&kv_full[stage], phase);
        }
        DS_TRACE_EV(24 + h);
        tc_fence_after_sync();
        const uint64_t v_desc = v_desc0 + (uint64_t)((stage * C::STAGE_BYTES) >> 4);
        const int ksteps = (rows + 15) >> 4;
        auto pv_step = [&](int ks) {
          // A = P[:, 16 ks .. 16 ks + 15]: 8 packed TMEM columns inside the 32-column quarter the kv columns belong to
          const uint32_t a_tmem = tmem_base + kTmemS + h * kHalfKV + (ks >> 1) * 32 + (ks & 1) * 8;
          const uint32_t acc = (G.first_of_item && h == 0 && ks == 0) ? 0u : 1u;
          umma_f16_ts(tmem_base + kTmemO, a_tmem, v_desc + (uint64_t)((ks * 16 * C::SUB_BYTES) >> 4), idesc_pv, acc);
          umma_f16_ts(tmem_base + kTmemL, a_tmem, ones_desc, idesc_l, acc);   // l += P . 1
        };
        // full halves (the common case) with compile-time operand offsets: the rolled loop spends ~25 dependent
        // uniform-datapath instructions per step, about as long as the tensor core needs for the step itself
        if (ksteps == kHalfKV / 16) {
#pragma unroll
          for (int ks = 0; ks < kHalfKV / 16; ++ks) pv_step(ks);
        } else {
#pragma unroll 1
          for (int ks = 0; ks < ksteps; ++ks) pv_step(ks);
        }
        if (p.mc) umma_commit_mc(&kv_empty[stage], (uint16_t)3);
        else umma_commit(&kv_empty[stage]);
        advance();
        if (h) ++pv_cntB; else ++pv_cntA;
        umma_commit(pv_half);
        DS_TRACE_EV(26 + h);
        if (G.last_of_item && (h == 1 || G.rowsB == 0)) {
          umma_commit(o_full);
          ++items_pv;
        }
      };
      LiteGroup prev = {};
      bool have_prev = false;
      for_each_group_lite(p, [&](const LiteGroup& G) {
        if (have_prev) issue_pv(prev, 0);
        issue_qk(G, 0);
        if (have_prev && prev.rowsB) issue_pv(prev, 1);
        if (G.rowsB) issue_qk(G, 1);
        prev = G;
        have_prev = true;
      });
      if (have_prev) {
        issue_pv(prev, 0);
        if (prev.rowsB) issue_pv(prev, 1);
      }
    }
  } else if (warp >= kWarpSoftmax0) {
    // ------------------------------------------------------------------ softmax
    const int qtr = (warp - kWarpSoftmax0) >> 2;            // which 32 columns of each S half
    const int quad = warp & 3;                   // TMEM lane quadrant this warp may touch
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const uint32_t s_col = tmem_base + lane_addr + kTmemS + qtr * 32;   // + h * 128; P goes to the first 16 of the 32
    const uint32_t o_col = tmem_base + lane_addr + kTmemO;
    const float sl2 = p.scale_log2;
    uint32_t cntA = 0, cntB = 0, w = 0;   // halves A / B seen, half-steps
    float m_run = 0.f;
#ifdef DS_TRACE
    int _tr_n = 0;
    const int _tr_slot = warp == kWarpSoftmax0 ? 2 : 3;
    const bool _tr_on = p.trace && blockIdx.x == 0 && lane == 0 && (warp == kWarpSoftmax0 || warp == 25);
#endif

    for_each_group_lite(p, [&](const LiteGroup& G) {
      const int n_half = G.rowsB ? 2 : 1;
#pragma unroll 1
      for (int h = 0; h < n_half; ++h, ++w) {
        const int nv = max(0, min((h ? G.rowsB : G.rowsA) - qtr * 32, 32));   // valid columns of this thread's 32
        const bool first = G.first_of_item && h == 0;
        DS_TRACE_EV(30 + h);
        mbar_wait(&s_full[h], (h ? cntB : cntA) & 1);
        DS_TRACE_EV(32 + h);
        tc_fence_after_sync();
        uint32_t v[32];
        tmem_ld_x32(s_col + h * kHalfKV, v);   // also when nv == 0: stale columns, never used
        tmem_wait_ld();
        DS_TRACE_EV(48 + h);
        // ragged tail (rare): columns past the kv length hold stale data, possibly NaN -- overwrite them with -inf once,
        // so that the common path below carries no per-column selects (-inf is neutral for the maximum and
        // exp2(-inf * scale - m) = 0; the host guarantees scale > 0)
        if (nv < 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j >= nv) v[j] = 0xff800000u;
        }
        // ---- row maximum of this half (4 threads per row exchange through shared memory)
        float m;
        {
          float a0 = -INFINITY, a1 = -INFINITY, a2 = -INFINITY, a3 = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            a0 = fmaxf(a0, fmaxf(__uint_as_float(v[j]), __uint_as_float(v[j + 1])));
            a1 = fmaxf(a1, fmaxf(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])));
            a2 = fmaxf(a2, fmaxf(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5])));
            a3 = fmaxf(a3, fmaxf(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7])));
          }
          m = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
        }
        m *= sl2;
        float* mx = sMax + (w & 1) * 512;
        mx[qtr * 128 + row] = m;
        DS_TRACE_EV(34 + h);
        named_bar_sync(1 + quad, 128);   // the four warps of this TMEM quadrant (= of this scheduler) hold the row
        DS_TRACE_EV(36 + h);
        const float Mh = fmaxf(fmaxf(mx[row], mx[128 + row]), fmaxf(mx[256 + row], mx[384 + row]));
        // Lazy running maximum: the first half of the item fixes the row's reference m_run; a later half keeps it and
        // simply lets p = exp2(s - m_run) grow -- up to 2^14 for fp16 P, 2^30 for bf16 -- which 16-bit P and the fp32
        // accumulators hold without loss (the offset cancels in O / l).  Only beyond that does the reference move, which
        // rescales O and l (rare; the four threads of the row decide identically).
        constexpr float kTau = kBf16 ? 30.0f : 14.0f;
        float alpha = 1.0f;
        if (first) {
          m_run = Mh;
        } else if (Mh > m_run + kTau) {
          alpha = fast_exp2(m_run - Mh);
          m_run = Mh;
        }
        if (qtr == 0 && !first) {
          // the first-quarter thread of a row rescales O and l before P is released
          if (__any_sync(0xffffffffu, alpha != 1.0f)) {
            mbar_wait(pv_half, (w - 1) & 1);   // the previous half's PV has landed in O (phases <= w-2 are known complete)
            tc_fence_after_sync();
#pragma unroll 1
            for (int c = 0; c < C::D_PAD / 16; ++c) {
              uint32_t o[16];
              tmem_ld_x16(o_col + c * 16, o);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * alpha);
              tmem_st_x16(o_col + c * 16, o);
            }
            const uint32_t l_addr = tmem_base + lane_addr + kTmemL;
            const float lv = __uint_as_float(tmem_ld_x1(l_addr));
            tmem_wait_ld();
            tmem_st_x1(l_addr, __float_as_uint(lv * alpha));
          }
        }
        // ---- p = exp2(s * scale - m), written as packed 16-bit pairs over the first half of the columns just read (the A
        //      operand of the PV product); the row sum is taken by the tensor core (ones column)
        if (nv > 0) {
          uint32_t pk[16];
          const uint64_t sl2_2 = f2_pack(sl2, sl2), nm_2 = f2_pack(-m_run, -m_run);
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float x0, x1, e0, e1;
            f2_unpack(f2_fma(f2_pack_u(v[j], v[j + 1]), sl2_2, nm_2), x0, x1);
            // the MUFU pipe (16 ex2 / clk / SM) is what bounds this phase: every kPolyStride-th pair is evaluated on the
            // FMA pipe instead
            constexpr int kPolyStride = C::POLY_STRIDE;
            if (kPolyStride > 0 && ((j >> 1) % (kPolyStride > 0 ? kPolyStride : 1)) == 0) {
              exp2_poly_f2(x0, x1, e0, e1);
            } else {
              e0 = fast_exp2(x0);
              e1 = fast_exp2(x1);
            }
            pk[j >> 1] = pack2<kBf16>(e0, e1);
          }
          tmem_st_x16(s_col + h * kHalfKV, pk);
        }
        DS_TRACE_EV(44 + h);
        tmem_wait_st();
        DS_TRACE_EV(46 + h);
        tc_fence_before_sync();
        mbar_arrive(&p_full[h]);
        DS_TRACE_EV(38 + h);
        if (h) ++cntB; else ++cntA;
      }
    });
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2-9)
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const int dh = (warp - 2) >> 2;                       // which half of the 16-column chunks of O
    constexpr int NC_ALL = C::D_PAD / 16;
    constexpr int NC0 = (NC_ALL + 1) / 2;                 // chunks of the first half (the second gets the rest)
    const int c_base = dh ? NC0 : 0;
    const uint32_t o_col = tmem_base + lane_addr + kTmemO + c_base * 16;
    const uint32_t os_col = tmem_base + lane_addr + kTmemOs + c_base * 8;
    const int tiles = p.B * p.H * p.n_qt;
    uint32_t n = 0;   // items seen
#ifdef DS_TRACE
    int _tr_n = 0;
    const int _tr_slot = 4;
    const bool _tr_on = p.trace && blockIdx.x == 0 && lane == 0 && warp == 2;
#endif
    float ns_tile = 0.f;  // |O_self|^2 of the current stream (meaningful on the reducing thread)
    for_each_group(p, [&](const GroupInfo& G) {
      if (!G.last_of_item) return;
      const uint32_t par = n & 1;
      // one phase per item; the tensor core cannot complete the next item before this warp has released O
      mbar_wait(o_full, par);
      DS_TRACE_EV(40);

      const bool row_ok = G.qt * kBlockQ + row < p.Sq;
      tc_fence_after_sync();
      float inv_l;
      {
        const uint32_t lv = tmem_ld_x1(tmem_base + lane_addr + kTmemL);
        tmem_wait_ld();
        inv_l = 1.0f / __uint_as_float(lv);
      }
      // cosine: (acc0+acc1) = dot (cross) or |Os|^2 (self), (acc2+acc3) = |Oc|^2; mse: (acc0+acc1) = sum of squared differences
      uint64_t acc01 = 0ull, acc23 = 0ull;   // packed fp32 pairs, (+0.f, +0.f)
      uint8_t* out_row = nullptr;
      if constexpr (MODE == ATTN_MODE_STORE)
        out_row = static_cast<uint8_t*>(p.out) + 2 * ((int64_t)G.b * p.out_sb + (int64_t)G.h * p.out_sh +
                                                     (int64_t)(G.qt * kBlockQ + row) * p.out_ss + c_base * 16);
      if constexpr (MODE == ATTN_MODE_LIST) {
        const int64_t slot = G.self ? G.g : p.n_groups + G.entry;   // contiguous slots: slot stride B * out_sb
        out_row = static_cast<uint8_t*>(p.out) + 2 * ((slot * p.B + G.b) * p.out_sb + (int64_t)G.h * p.out_sh +
                                                     (int64_t)(G.qt * kBlockQ + row) * p.out_ss + c_base * 16);
      }
      const bool cross = (MODE < ATTN_MODE_STORE) && !G.self;
      constexpr int NC = NC0;                 // trip count of the unrolled loop; the second half may own one chunk less
      const int nc_mine = dh ? NC_ALL - NC0 : NC0;
      // software pipeline over the 16-column chunks of O: the TMEM loads of chunk c+1 are in flight while chunk c is
      // consumed; O is released to the tensor core as soon as its last chunk has landed in registers
      uint32_t v[2][16], os[2][8];
      tmem_ld_x16(o_col, v[0]);
      if (cross) tmem_ld_x8(os_col, os[0]);
      tmem_wait_ld();
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const int cur = c & 1;
        if (c >= nc_mine) break;
        if (c + 1 < nc_mine) {
          tmem_ld_x16(o_col + (c + 1) * 16, v[cur ^ 1]);
          if (cross) tmem_ld_x8(os_col + (c + 1) * 8, os[cur ^ 1]);
        } else {
          tc_fence_before_sync();
          mbar_arrive(o_empty);
        }
        if constexpr (MODE >= ATTN_MODE_STORE) {
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            pk[j] = pack2<kBf16>(__uint_as_float(v[cur][2 * j]) * inv_l, __uint_as_float(v[cur][2 * j + 1]) * inv_l);
          if (row_ok) {
#pragma unroll
            for (int hlf = 0; hlf < 2; ++hlf) {
              if ((c_base + c) * 16 + hlf * 8 < D) {
                uint4 w4 = make_uint4(pk[4 * hlf], pk[4 * hlf + 1], pk[4 * hlf + 2], pk[4 * hlf + 3]);
                *reinterpret_cast<uint4*>(out_row + (c * 16 + hlf * 8) * 2) = w4;
              }
            }
          }
        } else if (!cross) {
          // O_self is rounded to the input dtype (as the reference's SDPA output is) and kept in TMEM
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            pk[j] = pack2<kBf16>(__uint_as_float(v[cur][2 * j]) * inv_l, __uint_as_float(v[cur][2 * j + 1]) * inv_l);
          tmem_st_x8(os_col + c * 8, pk);
          if constexpr (MODE == ATTN_MODE_COS) {
            // |O_self|^2 from the unrounded values, normalised once per row below (differs from the norm of the
            // rounded vector by O(eps^2))
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              const uint64_t o2 = f2_pack_u(v[cur][j], v[cur][j + 1]);
              acc01 = f2_fma(o2, o2, acc01);
            }
          }
        } else if constexpr (MODE == ATTN_MODE_COS) {
          // unnormalised: dot = inv_l * sum o s, |Oc|^2 = inv_l^2 * sum o^2 (applied once per row below)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 sv = unpack2<kBf16>(os[cur][j]);
            const uint64_t o2 = f2_pack_u(v[cur][2 * j], v[cur][2 * j + 1]);
            acc01 = f2_fma(o2, f2_pack(sv.x, sv.y), acc01);
            acc23 = f2_fma(o2, o2, acc23);
          }
        } else {
          // MSE: the cross output is rounded to the input dtype like O_self (and like the reference's SDPA outputs), so
          // that an image scored against itself gives exactly 0
          const uint64_t inv_l2 = f2_pack(inv_l, inv_l);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 sv = unpack2<kBf16>(os[cur][j]);
            float x0, x1;
            f2_unpack(f2_mul(f2_pack_u(v[cur][2 * j], v[cur][2 * j + 1]), inv_l2), x0, x1);
            const float2 ov = unpack2<kBf16>(pack2<kBf16>(x0, x1));
            const uint64_t d2 = f2_add(f2_pack(ov.x, ov.y), f2_pack(-sv.x, -sv.y));
            acc01 = f2_fma(d2, d2, acc01);
          }
        }
        if (c + 1 < nc_mine) tmem_wait_ld();
      }
      if constexpr (MODE < ATTN_MODE_STORE) {
        if (G.self) tmem_wait_st();
        float r0, r1;   // cross: (dot, |Oc|^2) or (sq, 0); self: (|Os|^2, 0)
        if (G.self) {
          r0 = f2_hsum(acc01) * inv_l * inv_l;
          r1 = 0.f;
        } else if constexpr (MODE == ATTN_MODE_COS) {
          r0 = f2_hsum(acc01) * inv_l;
          r1 = f2_hsum(acc23) * inv_l * inv_l;
        } else {
          r0 = f2_hsum(acc01);
          r1 = 0.f;
        }
        if (!row_ok) r0 = r1 = 0.f;
        // fixed-order reduction over the 128 rows: shuffle tree, then warps 0..3 in order
        r0 = warp_sum(r0);
        r1 = warp_sum(r1);
        float* red = sRed + par * 16;   // [8 warps][2]
        if (lane == 0) {
          red[(dh * 4 + quad) * 2 + 0] = r0;
          red[(dh * 4 + quad) * 2 + 1] = r1;
        }
        named_bar_sync(5, 256);
        if (warp == 2 && lane == 0) {
          const float t0 = ((red[0] + red[2]) + (red[4] + red[6])) + ((red[8] + red[10]) + (red[12] + red[14]));
          const float t1 = ((red[1] + red[3]) + (red[5] + red[7])) + ((red[9] + red[11]) + (red[13] + red[15]));
          if (G.self) {
            ns_tile = t0;
          } else if constexpr (MODE == ATTN_MODE_COS) {
            p.part[(size_t)G.entry * tiles + G.bh * p.n_qt + G.qt] = make_float4(t0, t1, ns_tile, 0.f);
          } else {
            p.part[(size_t)G.entry * tiles + G.bh * p.n_qt + G.qt] = make_float4(0.f, 0.f, 0.f, t0);
          }
        }
      }
      DS_TRACE_EV(41);
      ++n;
    });
  }
  tc_fence_before_sync();
  __syncthreads();
  if (p.mc) cluster_sync_all();   // the peer may still multicast into this CTA's ring / arrive on its barriers
  if (warp == kWarpMma) tmem_dealloc(tmem_base, kTmemCols);
  if (p.cycles && blockIdx.x == 0 && threadIdx.x == 0) *p.cycles = (unsigned long long)(clock64() - clk_start);
}


// Image indices of a work list against the image counts of the tensors they address.  An out-of-range index would become
// a TMA coordinate outside the tensor -- TMA zero-fills such loads, so the kernel would return a finite but WRONG score.
// bad[0] is set instead and aas_finish_kernel turns every score of the call into NaN (loud, no host sync).
__global__ void validate_groups_kernel(const int32_t* __restrict__ group_q, int64_t n_groups, const int32_t* __restrict__ kv_idx,
                                       int64_t n_entries, int64_t nq_images, int64_t nk_images, int32_t* __restrict__ bad) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  bool b = false;
  if (i < n_groups) b |= group_q[i] < 0 || group_q[i] >= nq_images;
  if (i < n_entries) b |= kv_idx[i] < 0 || kv_idx[i] >= nk_images;
  if (b) atomicExch(bad, 1);
}

// dir[t] from the per-tile partials, tiles added in index order (deterministic)
__global__ void aas_finish_kernel(const float4* __restrict__ part, int64_t n_entries, int tiles, double E, int mode,
                                  float* __restrict__ dir, int64_t ncols, int64_t ldd, int64_t nrows, int64_t chunk_cols,
                                  const int32_t* __restrict__ bad) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n_entries) return;
  const float4* pp = part + (size_t)t * tiles;
  float d = 0.f, nc = 0.f, ns = 0.f, sq = 0.f;
  for (int i = 0; i < tiles; ++i) {
    float4 v = pp[i];
    d += v.x;
    nc += v.y;
    ns += v.z;
    sq += v.w;
  }
  float r;
  if (mode == DS_SIM_MSE) r = (float)((double)sq / E);
  else {
    double nx = fmax(sqrt((double)nc), 1e-8), ny = fmax(sqrt((double)ns), 1e-8);
    r = (float)((double)d / (nx * ny));
  }
  if (bad && *bad) r = __int_as_float(0x7fc00000);   // an image index of the work list was out of range
  if (ncols > 0) {
    // matrix layout, entries in column-chunk-major order (matrix_setup_kernel): chunk ch holds, row after row, the
    // w(ch) = min(chunk_cols, ncols - ch * chunk_cols) columns starting at ch * chunk_cols
    const int64_t full = nrows * chunk_cols;                 // entries of a full chunk
    const int64_t ch = t / full;
    const int64_t w = min(chunk_cols, ncols - ch * chunk_cols);
    const int64_t rem = t - ch * full;
    const int64_t row = rem / w, col = ch * chunk_cols + rem % w;
    dir[row * ldd + col] = r;
  } else {
    dir[t] = r;
  }
}

__global__ void single_meta_kernel(int32_t* __restrict__ meta) {
  // group_q[0] = 0, group_off = {0, 1}, kv_idx[0] = 0
  if (threadIdx.x < 4) meta[threadIdx.x] = (threadIdx.x == 2) ? 1 : 0;
}

__global__ void pairs_setup_kernel(const int32_t* __restrict__ pair_idx, int64_t n_pairs, int32_t* __restrict__ group_q,
                                   int32_t* __restrict__ group_off, int32_t* __restrict__ kv_idx) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < 2 * n_pairs) {
    int64_t pr = i >> 1;
    int s = (int)(i & 1);
    group_q[i] = pair_idx[2 * pr + s];
    kv_idx[i] = pair_idx[2 * pr + (s ^ 1)];
    group_off[i] = (int32_t)i;
  }
  if (i == 2 * n_pairs) group_off[i] = (int32_t)i;
}

__global__ void pairs_finish_kernel(const float* __restrict__ dir, int64_t n_pairs, float* __restrict__ scores) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n_pairs) scores[i] = (dir[2 * i] + dir[2 * i + 1]) * 0.5f;
}

// triplet t = (ref, left, right): groups ref:[left,right], left:[ref], right:[ref]
__global__ void triplets_setup_kernel(const int32_t* __restrict__ trip, int64_t n, int32_t* __restrict__ group_q,
                                      int32_t* __restrict__ group_off, int32_t* __restrict__ kv_idx) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    const int32_t r = trip[3 * i], l = trip[3 * i + 1], rt = trip[3 * i + 2];
    group_q[3 * i] = r;
    group_q[3 * i + 1] = l;
    group_q[3 * i + 2] = rt;
    group_off[3 * i] = (int32_t)(4 * i);
    group_off[3 * i + 1] = (int32_t)(4 * i + 2);
    group_off[3 * i + 2] = (int32_t)(4 * i + 3);
    kv_idx[4 * i] = l;       // ref  -> left
    kv_idx[4 * i + 1] = rt;  // ref  -> right
    kv_idx[4 * i + 2] = r;   // left -> ref
    kv_idx[4 * i + 3] = r;   // right-> ref
  }
  if (i == n) group_off[3 * n] = (int32_t)(4 * n);
}

template <bool kBf16>
__device__ __forceinline__ float round_like_input(float x) {
  if constexpr (kBf16) return __bfloat162float(__float2bfloat16_rn(x));
  else return __half2float(__float2half_rn(x));
}

// (a_on_b + b_on_a) / 2 and the drivers' strict comparisons (cute_main.py:196-205)
template <bool kBf16>
__global__ void triplets_finish_kernel(const float* __restrict__ dir, int64_t n, int mode, int round_scores,
                                       float* __restrict__ ab, float* __restrict__ ac, int32_t* __restrict__ counts,
                                       uint8_t* __restrict__ flags) {
  int c1 = 0, c2 = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float d0 = dir[4 * i], d1 = dir[4 * i + 1], d2 = dir[4 * i + 2], d3 = dir[4 * i + 3];
    float sab, sac;
    if (round_scores) {
      sab = round_like_input<kBf16>(round_like_input<kBf16>(d0) + round_like_input<kBf16>(d2)) * 0.5f;
      sac = round_like_input<kBf16>(round_like_input<kBf16>(d1) + round_like_input<kBf16>(d3)) * 0.5f;
      sab = round_like_input<kBf16>(sab);
      sac = round_like_input<kBf16>(sac);
    } else {
      sab = (d0 + d2) * 0.5f;
      sac = (d1 + d3) * 0.5f;
    }
    ab[i] = sab;
    ac[i] = sac;
    bool ok, ok2;
    if (mode == DS_SIM_MSE) {
      ok = sab < sac;
      ok2 = sab * 2.0f < sac;
    } else {
      ok = sab > sac;
      ok2 = sab > 2.0f * sac;
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

// Work list of the N x N matrix.  Groups (and their entries) are laid out COLUMN-CHUNK-MAJOR: group g = ch * n_rows + row
// scores row image `row` against the columns of chunk ch.  The CTAs of a wave then work on ~74 different rows of the SAME
// chunk, whose K / V slices of the current (b, h) -- chunk_cols x 2 x S x D x 2 bytes, sized by matrix_plan to a third of
// the L2 -- stay resident while every row streams over them (row-major order made all CTAs stream all N columns: a 333 MB
// working set per (b, h) at the Sref shape, kept out of DRAM only by the CTAs happening to run in lock-step).
__global__ void matrix_setup_kernel(int64_t n_rows, int64_t n_cols, int chunks, int64_t chunk_cols,
                                    int32_t* __restrict__ group_q, int32_t* __restrict__ group_off,
                                    int32_t* __restrict__ kv_idx) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t n_groups = n_rows * chunks;
  const int64_t full = n_rows * chunk_cols;
  if (i < n_rows * n_cols) {
    const int64_t ch = i / full;
    const int64_t w = min(chunk_cols, n_cols - ch * chunk_cols);
    kv_idx[i] = (int32_t)(ch * chunk_cols + (i - ch * full) % w);
  }
  if (i < n_groups) {
    const int64_t ch = i / n_rows, r = i % n_rows;
    const int64_t w = min(chunk_cols, n_cols - ch * chunk_cols);
    group_q[i] = (int32_t)r;
    group_off[i] = (int32_t)(ch * full + r * w);
  }
  if (i == n_groups) group_off[i] = (int32_t)(n_rows * n_cols);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
// ds_debug_set_attn_mc: -1 automatic (the N x N matrix only: +2-3% there, -1% sustained and +16% DRAM reads on pair / triplet
// lists, profiles/r2_attn_experiments.txt section 8), 0 off, 1 on wherever the q tile count is even
static int g_attn_mc = -1;
static unsigned long long* g_trace_ptr = nullptr;
static int g_trace_cap = 0;

struct AttnLaunch {
  ds_tensor5 q, ks, vs, k, v;
  AttnParams p;
  int mode;   // ATTN_MODE_*
  int prefer_mc = 0;   // the caller's work list has many kv images per query image: share K/V loads over CTA pairs
};

template <int D, bool kBf16, int MODE>
static int launch_attn_one(const AttnLaunch& a, int grid, const CUtensorMap& mq, const CUtensorMap& mks,
                           const CUtensorMap& mvs, const CUtensorMap& mk, const CUtensorMap& mv, cudaStream_t st) {
  using C = AttnCfg<D>;
  DS_CUDA_TRY(cudaFuncSetAttribute(aas_attn_kernel<D, kBf16, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   C::SMEM_BYTES));
  if (!a.p.mc) {
    aas_attn_kernel<D, kBf16, MODE><<<grid, kAttnThreads, C::SMEM_BYTES, st>>>(mq, mks, mvs, mk, mv, a.p);
    return DS_OK;
  }
  // clusters of two CTAs (the q tiles 2j, 2j + 1 of a stream pair share every K/V load).  The schedule is static, so the
  // grid must not exceed what is co-resident: a GPC with an odd SM count cannot pair its last SM.
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3((unsigned)(grid & ~1));
  cfg.blockDim = dim3(kAttnThreads);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  static int max_clusters[64] = {};
  int dev = 0;
  DS_CUDA_TRY(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64) {
    if (max_clusters[dev] == 0) {
      int n = 0;
      cudaLaunchConfig_t q = cfg;
      q.gridDim = dim3((unsigned)(sm_count() & ~1));
      DS_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, aas_attn_kernel<D, kBf16, MODE>, &q));
      max_clusters[dev] = n > 0 ? n : -1;
    }
    if (max_clusters[dev] > 0 && (int)cfg.gridDim.x > 2 * max_clusters[dev]) cfg.gridDim.x = 2 * max_clusters[dev];
  }
  DS_CUDA_TRY(cudaLaunchKernelEx(&cfg, aas_attn_kernel<D, kBf16, MODE>, mq, mks, mvs, mk, mv, a.p));
  return DS_OK;
}

template <int D, bool kBf16>
static int launch_attn_mode(const AttnLaunch& a, int grid, const CUtensorMap& mq, const CUtensorMap& mks,
                            const CUtensorMap& mvs, const CUtensorMap& mk, const CUtensorMap& mv, cudaStream_t st) {
  switch (a.mode) {
    case ATTN_MODE_COS: return launch_attn_one<D, kBf16, ATTN_MODE_COS>(a, grid, mq, mks, mvs, mk, mv, st);
    case ATTN_MODE_MSE: return launch_attn_one<D, kBf16, ATTN_MODE_MSE>(a, grid, mq, mks, mvs, mk, mv, st);
    case ATTN_MODE_LIST: return launch_attn_one<D, kBf16, ATTN_MODE_LIST>(a, grid, mq, mks, mvs, mk, mv, st);
    default: return launch_attn_one<D, kBf16, ATTN_MODE_STORE>(a, grid, mq, mks, mvs, mk, mv, st);
  }
}

template <int D>
static int launch_attn_d(AttnLaunch a, cudaStream_t st) {
  using C = AttnCfg<D>;
  CUtensorMap mq, mks, mvs, mk, mv;
  int rc;
  if ((rc = make_map(&mq, a.q, C::SUBW, kBlockQ)) != DS_OK) return rc;
  if ((rc = make_map(&mks, a.ks, C::SUBW, kHalfKV)) != DS_OK) return rc;
  if ((rc = make_map(&mvs, a.vs, C::SUBW, kHalfKV)) != DS_OK) return rc;
  if ((rc = make_map(&mk, a.k, C::SUBW, kHalfKV)) != DS_OK) return rc;
  if ((rc = make_map(&mv, a.v, C::SUBW, kHalfKV)) != DS_OK) return rc;
  const int64_t n_streams = (int64_t)a.p.n_groups * a.p.B * a.p.H * a.p.n_qt;
  if (n_streams >= (int64_t)1 << 31) return fail(DS_ERR_INVALID, "too many (group, head, q-tile) streams in one call: split the work list");
  a.p.trace = g_trace_ptr;
  a.p.trace_cap = g_trace_cap;
  a.p.cycles = g_trace_ptr ? g_trace_ptr + (size_t)8 * g_trace_cap : nullptr;
  int grid = sm_count();
  if (n_streams < grid) grid = (int)n_streams;
  if (grid <= 0) return DS_OK;
  // K/V multicast over CTA pairs needs the two q tiles of a pair to exist (q tile is the fastest stream index, so CTAs
  // 2c and 2c + 1 hold q tiles 2j and 2j + 1 of the same (group, b, h) when n_qt and the grid are even)
  const bool want_mc = g_attn_mc == 1 || (g_attn_mc < 0 && a.prefer_mc);
  a.p.mc = (want_mc && a.p.n_qt % 2 == 0 && grid >= 2) ? 1 : 0;
  profile_begin(st);
  rc = with_dtype(a.q.dtype, [&](auto bf) {
    return launch_attn_mode<D, decltype(bf)::value>(a, grid, mq, mks, mvs, mk, mv, st);
  });
  if (rc != DS_OK) return rc;
  profile_end(st);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

static int launch_attn(const AttnLaunch& a, const char* who, cudaStream_t st) {
  return with_head_dim(a.q.size[4], who, [&](auto d) { return launch_attn_d<decltype(d)::value>(a, st); });
}

// kv groups of an item of skv rows and the valid rows of the two halves of its last group
static void kv_split(int skv, int* n_grp, int* rowsA_last, int* rowsB_last) {
  *n_grp = (skv + kGroupKV - 1) / kGroupKV;
  const int rem = skv - (*n_grp - 1) * kGroupKV;
  *rowsA_last = rem < kHalfKV ? rem : kHalfKV;
  *rowsB_last = rem <= kHalfKV ? 0 : rem - kHalfKV;   // rem <= kGroupKV
}

// common validation of a (q, k_self, v_self, k, v) set, before any device work; fills the shape part of AttnParams
static int prepare(AttnLaunch& a, float scale, const char* who) {
  const ds_tensor5* all[5] = {&a.q, &a.ks, &a.vs, &a.k, &a.v};
  const char* const names[5] = {"q", "k_self", "v_self", "k", "v"};
  int rc;
  for (int i = 0; i < 5; ++i) {
    if ((rc = check_operand(*all[i], who, names[i])) != DS_OK) return rc;
    if (all[i]->size[0] > INT32_MAX || all[i]->size[3] > INT32_MAX)
      return fail(DS_ERR_INVALID, "%s: %s: too large", who, names[i]);
  }
  for (int i = 1; i < 5; ++i) {
    if (all[i]->dtype != a.q.dtype) return fail(DS_ERR_INVALID, "%s: all tensors must share one dtype", who);
    if (all[i]->size[1] != a.q.size[1] || all[i]->size[2] != a.q.size[2] || all[i]->size[4] != a.q.size[4])
      return fail(DS_ERR_INVALID, "%s: B, H and D must match across q, k, v", who);
  }
  // (k_self, v_self) share one kv length and (k, v) another; the two are independent of each other and of q's length
  if (a.vs.size[3] != a.ks.size[3]) return fail(DS_ERR_INVALID, "%s: k_self and v_self must share the kv length", who);
  if (a.v.size[3] != a.k.size[3]) return fail(DS_ERR_INVALID, "%s: k and v must share the kv length", who);
  if (a.ks.size[0] != a.q.size[0] || a.vs.size[0] != a.q.size[0])
    return fail(DS_ERR_INVALID, "%s: k_self / v_self must hold the same images as q", who);
  if (a.k.size[0] != a.v.size[0]) return fail(DS_ERR_INVALID, "%s: k and v must hold the same images", who);
  const int64_t Skv = a.k.size[3], Skv_self = a.ks.size[3];
  if (Skv > INT32_MAX / 2 || Skv_self > INT32_MAX / 2) return fail(DS_ERR_INVALID, "%s: kv length too large", who);
  const int64_t D = a.q.size[4];
  if ((rc = with_head_dim(D, who, [](auto) { return DS_OK; })) != DS_OK) return rc;
  a.p.B = (int)a.q.size[1];
  a.p.H = (int)a.q.size[2];
  a.p.Sq = (int)a.q.size[3];
  a.p.Skv = (int)Skv;
  a.p.Skv_self = (int)Skv_self;
  kv_split(a.p.Skv, &a.p.n_grp, &a.p.rowsA_last, &a.p.rowsB_last);
  kv_split(a.p.Skv_self, &a.p.n_grp_self, &a.p.rowsA_last_self, &a.p.rowsB_last_self);
  a.p.n_qt = (int)((a.q.size[3] + kBlockQ - 1) / kBlockQ);
  const float sc = scale > 0.f ? scale : 1.0f / sqrtf((float)D);
  a.p.scale_log2 = sc * 1.4426950408889634f;
  return DS_OK;
}

int check_group_operands(const ds_tensor5& q, const ds_tensor5& k_self, const ds_tensor5& v_self, const ds_tensor5& k,
                         const ds_tensor5& v, const char* who) {
  AttnLaunch a;
  a.q = q;
  a.ks = k_self;
  a.vs = v_self;
  a.k = k;
  a.v = v;
  return prepare(a, 0.f, who);
}

int launch_validate_groups(const int32_t* group_q, int64_t n_groups, const int32_t* kv_idx, int64_t n_entries,
                           int64_t nq_images, int64_t nk_images, int32_t* bad, cudaStream_t st) {
  const int64_t nv = n_groups > n_entries ? n_groups : n_entries;
  validate_groups_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(group_q, n_groups, kv_idx, n_entries, nq_images,
                                                                       nk_images, bad);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

int launch_pairs_setup(const int32_t* pair_idx, int64_t n_pairs, int32_t* group_q, int32_t* group_off, int32_t* kv_idx,
                       cudaStream_t st) {
  pairs_setup_kernel<<<(unsigned)((2 * n_pairs + 1 + 255) / 256), 256, 0, st>>>(pair_idx, n_pairs, group_q, group_off, kv_idx);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

int launch_triplets_setup(const int32_t* trip_idx, int64_t n_triplets, int32_t* group_q, int32_t* group_off,
                          int32_t* kv_idx, cudaStream_t st) {
  triplets_setup_kernel<<<(unsigned)((n_triplets + 1 + 255) / 256), 256, 0, st>>>(trip_idx, n_triplets, group_q, group_off,
                                                                                kv_idx);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

int attn_list_store(const ds_tensor5& q, const ds_tensor5& k_self, const ds_tensor5& v_self, const ds_tensor5& k,
                    const ds_tensor5& v, const int32_t* group_q, const int32_t* group_off, int64_t n_groups,
                    const int32_t* kv_idx, float scale, void* out, const char* who, cudaStream_t st) {
  AttnLaunch a;
  a.q = q;
  a.ks = k_self;
  a.vs = v_self;
  a.k = k;
  a.v = v;
  int rc = prepare(a, scale, who);
  if (rc != DS_OK) return rc;
  a.p.group_q = group_q;
  a.p.group_off = group_off;
  a.p.kv_idx = kv_idx;
  a.p.n_groups = (int)n_groups;
  a.p.self_first = 1;
  a.mode = ATTN_MODE_LIST;
  a.p.part = nullptr;
  a.p.out = out;
  a.p.out_ss = q.size[4];
  a.p.out_sh = q.size[3] * q.size[4];
  a.p.out_sb = q.size[2] * a.p.out_sh;
  return launch_attn(a, who, st);
}

}  // namespace ds

extern "C" {

int ds_debug_set_trace(void* dev_buf, int cap) {
  ds::g_trace_ptr = static_cast<unsigned long long*>(dev_buf);
  ds::g_trace_cap = cap;
#ifdef DS_TRACE
  return 1;
#else
  return 0;
#endif
}

int ds_debug_set_attn_mc(int mode) {
  if (mode >= -1 && mode <= 1) ds::g_attn_mc = mode;
  return ds::g_attn_mc;
}

size_t ds_attn_fwd_workspace_bytes(ds_tensor4 q, ds_tensor4 k) {
  (void)k;
  return 1024;
}

int ds_attn_fwd(ds_tensor4 q, ds_tensor4 k, ds_tensor4 v, float scale, ds_tensor4 out, void* ws, size_t ws_bytes,
                void* stream) {
  using namespace ds;
  const char* who = "ds_attn_fwd";
  AttnLaunch a;
  a.q = lift(q);
  a.k = lift(k);
  a.v = lift(v);
  a.ks = a.k;
  a.vs = a.v;
  // k_self / v_self are unused in store mode, but must pass validation: give them q's image count
  int rc;
  if ((rc = prepare(a, scale, who)) != DS_OK || (rc = check_like(lift(out), a.q, who, "out")) != DS_OK) return rc;
  Workspace w(ws, ws_bytes);
  int32_t* meta = static_cast<int32_t*>(w.take(4 * sizeof(int32_t)));
  if (!meta) return fail(DS_ERR_WORKSPACE, "ds_attn_fwd: workspace too small (need %zu bytes)", (size_t)1024);
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // one group: query image 0, one entry: kv image 0
  single_meta_kernel<<<1, 32, 0, st>>>(meta);
  DS_CUDA_TRY(cudaGetLastError());
  a.p.group_q = meta;
  a.p.group_off = meta + 1;
  a.p.kv_idx = meta + 3;
  a.p.n_groups = 1;
  a.p.self_first = 0;
  a.mode = ATTN_MODE_STORE;
  a.p.part = nullptr;
  a.p.out = out.ptr;
  a.p.out_sb = out.stride[0];
  a.p.out_sh = out.stride[1];
  a.p.out_ss = out.stride[2];
  return launch_attn(a, who, st);
}

size_t ds_aas_groups_workspace_bytes(ds_tensor5 q, int64_t n_groups, int64_t n_entries) {
  (void)n_groups;
  if (n_entries <= 0) return 256;
  const int64_t tiles = q.size[1] * q.size[2] * ((q.size[3] + ds::kBlockQ - 1) / ds::kBlockQ);
  return ds::align_up((size_t)n_entries * tiles * sizeof(float4), 256) + 512;
}

int ds_aas_groups(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v,
                  const int32_t* group_q, const int32_t* group_off, int64_t n_groups, const int32_t* kv_idx,
                  int64_t n_entries, float scale, int mode, float* dir, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_groups < 0 || n_entries < 0) return fail(DS_ERR_INVALID, "ds_aas_groups: negative counts");
  if (n_groups == 0 || n_entries == 0) return DS_OK;
  if (!group_q || !group_off || !kv_idx || !dir) return fail(DS_ERR_INVALID, "ds_aas_groups: null pointer");
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return fail(DS_ERR_INVALID, "ds_aas_groups: bad mode %d", mode);
  if (n_groups > INT32_MAX || n_entries > INT32_MAX) return fail(DS_ERR_INVALID, "ds_aas_groups: too many groups");
  AttnLaunch a;
  a.q = q;
  a.ks = k_self;
  a.vs = v_self;
  a.k = k;
  a.v = v;
  int rc = prepare(a, scale, "ds_aas_groups");
  if (rc != DS_OK) return rc;
  const int tiles = a.p.B * a.p.H * a.p.n_qt;
  Workspace w(ws, ws_bytes);
  float4* part = static_cast<float4*>(w.take((size_t)n_entries * tiles * sizeof(float4)));
  int32_t* bad = static_cast<int32_t*>(w.take(sizeof(int32_t)));
  if (!part || !bad)
    return fail(DS_ERR_WORKSPACE, "ds_aas_groups: workspace too small (%zu given, need %zu)", ws_bytes,
                ds_aas_groups_workspace_bytes(q, n_groups, n_entries));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DS_CUDA_TRY(cudaMemsetAsync(bad, 0, sizeof(int32_t), st));
  {
    const int64_t nv = n_groups > n_entries ? n_groups : n_entries;
    validate_groups_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(group_q, n_groups, kv_idx, n_entries, q.size[0],
                                                                         k.size[0], bad);
    DS_CUDA_TRY(cudaGetLastError());
  }
  a.p.group_q = group_q;
  a.p.group_off = group_off;
  a.p.kv_idx = kv_idx;
  a.p.n_groups = (int)n_groups;
  a.p.self_first = 1;
  a.mode = (mode == DS_SIM_MSE) ? ATTN_MODE_MSE : ATTN_MODE_COS;
  a.p.part = part;
  a.p.out = nullptr;
  a.p.out_sb = a.p.out_sh = a.p.out_ss = 0;
  rc = launch_attn(a, "ds_aas_groups", st);
  if (rc != DS_OK) return rc;
  const double E = (double)a.p.B * a.p.H * a.p.Sq * (double)q.size[4];
  aas_finish_kernel<<<(unsigned)((n_entries + 127) / 128), 128, 0, st>>>(part, n_entries, tiles, E, mode, dir, 0, 0, 0, 0, bad);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

size_t ds_aas_pairs_workspace_bytes(ds_tensor5 q, int64_t n_pairs) {
  if (n_pairs <= 0) return 256;
  size_t b = ds_aas_groups_workspace_bytes(q, 2 * n_pairs, 2 * n_pairs);
  b += ds::align_up((size_t)(2 * n_pairs) * 4, 256) * 2;      // group_q, kv_idx
  b += ds::align_up((size_t)(2 * n_pairs + 1) * 4, 256);      // group_off
  b += ds::align_up((size_t)(2 * n_pairs) * 4, 256);          // directional scores
  return b + 256;
}

int ds_aas_pairs(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* pair_idx, int64_t n_pairs, float scale,
                 int mode, float* scores, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_pairs < 0) return fail(DS_ERR_INVALID, "ds_aas_pairs: negative n_pairs");
  if (n_pairs == 0) return DS_OK;
  if (!pair_idx || !scores) return fail(DS_ERR_INVALID, "ds_aas_pairs: null pointer");
  if (2 * n_pairs + 1 > INT32_MAX) return fail(DS_ERR_INVALID, "ds_aas_pairs: too many pairs");
  Workspace w(ws, ws_bytes);
  const int64_t G = 2 * n_pairs;
  int32_t* gq = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* kv = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* go = static_cast<int32_t*>(w.take((size_t)(G + 1) * 4));
  float* dir = static_cast<float*>(w.take((size_t)G * 4));
  if (!gq || !kv || !go || !dir)
    return fail(DS_ERR_WORKSPACE, "ds_aas_pairs: workspace too small (%zu given, need %zu)", ws_bytes,
                ds_aas_pairs_workspace_bytes(q, n_pairs));
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  pairs_setup_kernel<<<(unsigned)((G + 1 + 255) / 256), 256, 0, st>>>(pair_idx, n_pairs, gq, go, kv);
  DS_CUDA_TRY(cudaGetLastError());
  void* rest = w.take(0);
  rc = ds_aas_groups(q, k, v, k, v, gq, go, G, kv, G, scale, mode, dir, rest, ws_bytes - w.off, stream);
  if (rc != DS_OK) return rc;
  pairs_finish_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(dir, n_pairs, scores);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

size_t ds_aas_triplets_workspace_bytes(ds_tensor5 q, int64_t n_triplets) {
  if (n_triplets <= 0) return 256;
  size_t b = ds_aas_groups_workspace_bytes(q, 3 * n_triplets, 4 * n_triplets);
  b += ds::align_up((size_t)(3 * n_triplets) * 4, 256);      // group_q
  b += ds::align_up((size_t)(3 * n_triplets + 1) * 4, 256);  // group_off
  b += ds::align_up((size_t)(4 * n_triplets) * 4, 256) * 2;  // kv_idx, directional scores
  return b + 256;
}

int ds_aas_triplets(ds_tensor5 q, ds_tensor5 k, ds_tensor5 v, const int32_t* trip_idx, int64_t n_triplets, float scale,
                    int mode, int opts, float* ab, float* ac, int32_t* counts, uint8_t* flags_out, void* ws,
                    size_t ws_bytes, void* stream) {
  using namespace ds;
  if (n_triplets < 0) return fail(DS_ERR_INVALID, "ds_aas_triplets: negative n_triplets");
  if (!counts) return fail(DS_ERR_INVALID, "ds_aas_triplets: null counts");
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return fail(DS_ERR_INVALID, "ds_aas_triplets: bad mode %d", mode);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ds_device_ok();
  if (rc != DS_OK) return rc;
  DS_CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
  if (n_triplets == 0) return DS_OK;
  if (!trip_idx || !ab || !ac) return fail(DS_ERR_INVALID, "ds_aas_triplets: null pointer");
  if (4 * n_triplets + 1 > INT32_MAX) return fail(DS_ERR_INVALID, "ds_aas_triplets: too many triplets");
  Workspace w(ws, ws_bytes);
  const int64_t G = 3 * n_triplets, T = 4 * n_triplets;
  int32_t* gq = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* go = static_cast<int32_t*>(w.take((size_t)(G + 1) * 4));
  int32_t* kv = static_cast<int32_t*>(w.take((size_t)T * 4));
  float* dir = static_cast<float*>(w.take((size_t)T * 4));
  if (!gq || !go || !kv || !dir)
    return fail(DS_ERR_WORKSPACE, "ds_aas_triplets: workspace too small (%zu given, need %zu)", ws_bytes,
                ds_aas_triplets_workspace_bytes(q, n_triplets));
  triplets_setup_kernel<<<(unsigned)((n_triplets + 1 + 255) / 256), 256, 0, st>>>(trip_idx, n_triplets, gq, go, kv);
  DS_CUDA_TRY(cudaGetLastError());
  void* rest = w.take(0);
  rc = ds_aas_groups(q, k, v, k, v, gq, go, G, kv, T, scale, mode, dir, rest, ws_bytes - w.off, stream);
  if (rc != DS_OK) return rc;
  int blocks = (int)((n_triplets + 255) / 256);
  if (blocks > 1184) blocks = 1184;
  const int rs = (opts & DS_OPT_ROUND_SCORES) ? 1 : 0;
  if (q.dtype == DS_BF16)
    triplets_finish_kernel<true><<<blocks, 256, 0, st>>>(dir, n_triplets, mode, rs, ab, ac, counts, flags_out);
  else
    triplets_finish_kernel<false><<<blocks, 256, 0, st>>>(dir, n_triplets, mode, rs, ab, ac, counts, flags_out);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

static void matrix_plan(const ds_tensor5& q, const ds_tensor5& k, int64_t n_rows, int64_t n_cols, int* chunks, int64_t* chunk_cols) {
  const int64_t per_row = q.size[1] * q.size[2] * ((q.size[3] + ds::kBlockQ - 1) / ds::kBlockQ);
  // (1) L2 blocking: the K and V slices of one (b, h) of a chunk's columns should fill about a third of the 126 MB L2
  //     (sized from the column K / V, whose kv length may differ from the rows' k_self / v_self)
  const int64_t slice_bytes = 2 * k.size[3] * k.size[4] * 2;
  int64_t cc = (40ll << 20) / (slice_bytes > 0 ? slice_bytes : 1);
  if (cc > n_cols) cc = n_cols;
  // (2) enough streams to fill the machine: >= 4 per SM
  const int64_t want = (4 * 148 + n_rows * per_row - 1) / (n_rows * per_row);
  if (want > 1) {
    const int64_t c2 = (n_cols + want - 1) / want;
    if (c2 < cc) cc = c2;
  }
  // (3) the query image's self attention is recomputed once per chunk: keep that <= 1/8 of the work
  if (cc < 8) cc = n_cols < 8 ? n_cols : 8;
  *chunk_cols = cc;
  *chunks = (int)((n_cols + cc - 1) / cc);
}

size_t ds_aas_matrix_workspace_bytes(ds_tensor5 q, ds_tensor5 k) {
  const int64_t nr = q.size[0], nc = k.size[0];
  if (nr <= 0 || nc <= 0) return 256;
  int chunks;
  int64_t cc;
  matrix_plan(q, k, nr, nc, &chunks, &cc);
  size_t b = ds_aas_groups_workspace_bytes(q, nr * chunks, nr * nc);
  b += ds::align_up((size_t)(nr * chunks) * 4, 256);
  b += ds::align_up((size_t)(nr * chunks + 1) * 4, 256);
  b += ds::align_up((size_t)(nr * nc) * 4, 256);
  return b + 256;
}

int ds_aas_matrix(ds_tensor5 q, ds_tensor5 k_self, ds_tensor5 v_self, ds_tensor5 k, ds_tensor5 v, float scale, int mode,
                  float* Dm, int64_t ldd, void* ws, size_t ws_bytes, void* stream) {
  using namespace ds;
  const int64_t nr = q.size[0], nc = k.size[0];
  if (nr <= 0 || nc <= 0) return fail(DS_ERR_INVALID, "ds_aas_matrix: empty image set");
  if (!Dm || ldd < nc) return fail(DS_ERR_INVALID, "ds_aas_matrix: null output or ldd < columns");
  if (mode != DS_SIM_COSINE && mode != DS_SIM_MSE) return fail(DS_ERR_INVALID, "ds_aas_matrix: bad mode %d", mode);
  if (nr * nc > INT32_MAX) return fail(DS_ERR_INVALID, "ds_aas_matrix: more than 2^31 entries; split the rows");
  int chunks;
  int64_t cc;
  matrix_plan(q, k, nr, nc, &chunks, &cc);
  const int64_t G = nr * chunks, T = nr * nc;
  AttnLaunch a;
  a.q = q;
  a.ks = k_self;
  a.vs = v_self;
  a.k = k;
  a.v = v;
  int rc = prepare(a, scale, "ds_aas_matrix");
  if (rc != DS_OK) return rc;
  const int tiles = a.p.B * a.p.H * a.p.n_qt;
  Workspace w(ws, ws_bytes);
  int32_t* gq = static_cast<int32_t*>(w.take((size_t)G * 4));
  int32_t* go = static_cast<int32_t*>(w.take((size_t)(G + 1) * 4));
  int32_t* kv = static_cast<int32_t*>(w.take((size_t)T * 4));
  float4* part = static_cast<float4*>(w.take((size_t)T * tiles * sizeof(float4)));
  if (!gq || !go || !kv || !part)
    return fail(DS_ERR_WORKSPACE, "ds_aas_matrix: workspace too small (%zu given, need %zu)", ws_bytes,
                ds_aas_matrix_workspace_bytes(q, k));
  if ((rc = ds_device_ok()) != DS_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t setup_n = (T > G + 1 ? T : G + 1);
  matrix_setup_kernel<<<(unsigned)((setup_n + 255) / 256), 256, 0, st>>>(nr, nc, chunks, cc, gq, go, kv);
  DS_CUDA_TRY(cudaGetLastError());
  a.p.group_q = gq;
  a.p.group_off = go;
  a.p.kv_idx = kv;
  a.p.n_groups = (int)G;
  a.p.self_first = 1;
  a.mode = (mode == DS_SIM_MSE) ? ATTN_MODE_MSE : ATTN_MODE_COS;
  a.prefer_mc = 1;
  a.p.part = part;
  a.p.out = nullptr;
  a.p.out_sb = a.p.out_sh = a.p.out_ss = 0;
  rc = launch_attn(a, "ds_aas_matrix", st);
  if (rc != DS_OK) return rc;
  const double E = (double)a.p.B * a.p.H * a.p.Sq * (double)q.size[4];
  aas_finish_kernel<<<(unsigned)((T + 127) / 128), 128, 0, st>>>(part, T, tiles, E, mode, Dm, nc, ldd, nr, cc, nullptr);
  DS_CUDA_TRY(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
