// LongNet dilated attention on the 5th-generation tensor cores (sm_100a): TMA-staged Q/K/V tiles, tcgen05 MMAs with
// TMEM accumulators, online softmax in fp32.
//
// One CTA = one (branch, segment, head, 128-slot query tile); it streams the 128-slot key/value tiles of the same
// (branch, segment, head).  The dilated gather of the reference (dilated_attention.py:22-37, 82-111) is the TMA box
// itself: the qkv buffer [n_alloc, 3*768] is described per branch as a 3-D tensor (column, residue o, slot j) with
// position = j * r + o, so a box of (64 columns, 1, 128 slots) IS the sparse tile of one head -- no sparse copy exists.
// Rows >= n_tokens are zero in memory and rows >= n_alloc are zero-filled by TMA: these are the reference's zero
// keys (score 0, value 0, counted in the softmax denominator).  Slots past the segment's own m = ceil(g / r) belong to
// the next segment and are masked to -inf.
//
// head_dim = 48: the box is 64 columns wide (one 128-byte swizzle atom per row), the MMAs only consume K = 48 (three
// k-steps of 16) for S = Q K^T and N = 48 for O = P V, so no tensor-core work is spent on the padding columns.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM owner), warps 2-5 = softmax (one query
// row per thread = one TMEM lane).  P is written back to TMEM as packed bf16 (tcgen05.st) and is the A operand of the
// P V MMA straight from TMEM (no shared-memory round trip); O accumulates in TMEM over the whole key loop with a lazily
// raised row maximum (see the kernel comment).
#include <cuda.h>

#include <type_traits>

#include "mt_common.cuh"
#include "sm100_ptx.cuh"

namespace mt {
using namespace sm100;

// experiment-only phase tracing (compile with -DMT_DEBUG_TRACE): block 0 prints clock64 stamps of its first iterations
#ifdef MT_DEBUG_TRACE
#ifndef MT_TRACE_BLOCK
#define MT_TRACE_BLOCK 0
#endif
#define MT_TRACE_DECL long long tr_[96]; int trn_ = 0; const bool tron_ = (blockIdx.x == MT_TRACE_BLOCK);
#define MT_TRACE(tag) do { if (tron_ && trn_ < 94) { tr_[trn_++] = (long long)(tag); tr_[trn_++] = clock64(); } } while (0)
#define MT_TRACE_DUMP(who) do { if (tron_) for (int q_ = 0; q_ + 1 < trn_; q_ += 2) printf("%s %lld %lld\n", who, tr_[q_], tr_[q_ + 1] & 0xffffffffll); } while (0)
#ifndef MT_TRACE_ITEM
#define MT_TRACE_ITEM 5
#endif
// persistent kernels: stamps only while the CTA works on items MT_TRACE_ITEM .. MT_TRACE_ITEM + 1 (one hand-over)
#define MT_TRACEW(n, tag) do { if (tron_ && (n) >= MT_TRACE_ITEM && (n) <= MT_TRACE_ITEM + 1 && trn_ < 94) { tr_[trn_++] = (long long)(tag); tr_[trn_++] = clock64(); } } while (0)
#else
#define MT_TRACE_DECL
#define MT_TRACE(tag)
#define MT_TRACE_DUMP(who)
#define MT_TRACEW(n, tag)
#endif

// experiment-only CTA timeline (compile with -DMT_DEBUG_TIMELINE): every CTA records (SM id, loop length, clock64 at entry
// and exit) so that tools/attn_timeline.py can separate the time inside CTAs from the gaps between them on each SM
#ifdef MT_DEBUG_TIMELINE
__device__ long long mt_timeline[32768 * 4];
#define MT_TL_BEGIN const long long tl_t0_ = clock64();
#define MT_TL_END(n)                                                        \
  if (threadIdx.x == 0 && blockIdx.x < 32768) {                             \
    unsigned sm_;                                                           \
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_));                        \
    long long* e_ = mt_timeline + 4 * blockIdx.x;                           \
    e_[0] = sm_; e_[1] = (n); e_[2] = tl_t0_; e_[3] = clock64();            \
  }
// persistent kernels: one record per ITEM (loop length, clock at the first score tile, clock after the last one)
__device__ long long mt_item_timeline[65536 * 4];
__device__ int mt_item_count;
#define MT_TL_ITEM(n, t_first, t_last)                                      \
  do {                                                                      \
    const int k_ = atomicAdd(&mt_item_count, 1);                            \
    if (k_ < 65536) {                                                       \
      long long* e_ = mt_item_timeline + 4 * k_;                            \
      e_[0] = blockIdx.x; e_[1] = (n); e_[2] = (t_first); e_[3] = (t_last); \
    }                                                                       \
  } while (0)
#else
#define MT_TL_BEGIN
#define MT_TL_END(n)
#endif

#ifndef MT_FWD_POLY
#define MT_FWD_POLY 0                     // exponentials per 8 computed on the FMA pipes in the forward (ex2_poly)
#endif
static constexpr int DH = 48;            // head dim
static constexpr int BT = 128;           // slots per tile (queries and keys)
static constexpr int TILE_BYTES = BT * 128;  // [128 rows][128 B]: 64 bf16 columns per row, SWIZZLE_128B
static constexpr int KV_STAGES = 2;
static constexpr int FWD_THREADS = 192;
static constexpr uint32_t TMEM_COLS = 256;  // S: [0,128)  P (bf16 pairs): [128,192)  O tile: [192,256)

struct TensorMaps {
  CUtensorMap m[MT_MAX_BRANCHES];
};

struct Sm100Params {
  DilatedGeom geo;
  int item_prefix[MT_MAX_BRANCHES + 1];  // first CTA of each launch-order branch
  int order[MT_MAX_BRANCHES];            // launch order -> branch (longest key loops first)
  int tiles[MT_MAX_BRANCHES];            // 128-slot tiles per (segment, head), indexed by branch
  float scale_log2;                      // head_dim^-0.5 * log2(e)
  float scale;
};

// smem carve-up (dynamic, base must be 1024-byte aligned)
struct FwdSmem {
  static constexpr int Q = 0;
  static constexpr int K = Q + TILE_BYTES;
  static constexpr int V = K + KV_STAGES * TILE_BYTES;
  static constexpr int BAR = V + KV_STAGES * TILE_BYTES;
  // barriers (8 B each): q_full, kv_full[2], kv_empty[2], s_full, s_free, p_full, o_full[2]; then the TMEM pointer
  static constexpr int NBAR = 10;
  static constexpr int TMEM_PTR = BAR + NBAR * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
};

// ---------------------------------------------------------------------------------------------------------------------
// forward: O accumulated in TMEM with a lazily raised row maximum (no per-tile fold / rescale in registers), the whole
// 128-column score row loaded once, 3-input maxima.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FWD_THREADS, 2)
dilated_fwd_sm100_kernel(const __grid_constant__ TensorMaps maps, const Sm100Params P, __nv_bfloat16* __restrict__ o_br,
                         float* __restrict__ lse_br) {
  MT_TL_BEGIN
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  // roles by warp id: the scheduler favours high warp ids, so the latency-critical single-thread roles sit last
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_TMA = 4, W_MMA = 5;
  if ((sbase & 1023u) != 0) {  // SWIZZLE_128B tiles need 1024-byte alignment; never expected, but fail loudly
    __trap();
  }
  // ---- which tile -------------------------------------------------------------------------------------------------
  int oi = 0;
  while (oi + 1 < P.geo.nb && (int)blockIdx.x >= P.item_prefix[oi + 1]) ++oi;
  const int b = P.order[oi];
  const BranchGeom bg = P.geo.b[b];
  int local = blockIdx.x - P.item_prefix[oi];
  const int qt = local % P.tiles[b];
  local /= P.tiles[b];
  const int h = local % P.geo.H;
  const int s = local / P.geo.H;
  const int H = P.geo.H, N = P.geo.N, E = H * DH;
  const int off = (h * bg.r) / H;                    // residue of the positions this head owns
  const int jseg = (s * bg.g) / bg.r;                // first slot of the segment in the branch's j axis
  const int q0 = qt * BT;
  // Zero padding (positions >= N in the last segment, dilated_attention.py:82-111) in whole tiles is never computed:
  // a query tile without a real position writes nothing, and key tiles without a real position are all zero keys
  // (score 0, value 0), whose only effect -- n_zero_tail * exp(0 - max) in the softmax denominator -- is added in
  // closed form in the epilogue.  At 32k tiles 30 % of the padded tile pairs of the reference disappear this way.
  const int seg_lo = s * bg.g + off;
  const int c_real = min(N, (s + 1) * bg.g) > seg_lo ? (min(N, (s + 1) * bg.g) - seg_lo + bg.r - 1) / bg.r : 0;
  if (q0 >= c_real) return;
  const int n_kv = min(P.tiles[b], (c_real + BT - 1) / BT);
  const int n_zero_tail = max(0, bg.m - n_kv * BT);

  const uint32_t bar_q_full = sbase + FwdSmem::BAR + 0;
  const uint32_t bar_kv_full = sbase + FwdSmem::BAR + 8;    // [2]
  const uint32_t bar_kv_empty = sbase + FwdSmem::BAR + 24;  // [2]
  const uint32_t bar_s_full = sbase + FwdSmem::BAR + 40;
  const uint32_t bar_s_free = sbase + FwdSmem::BAR + 48;
  const uint32_t bar_p_full = sbase + FwdSmem::BAR + 56;
  const uint32_t bar_o_full = sbase + FwdSmem::BAR + 64;    // [2]
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + FwdSmem::TMEM_PTR);

  if (threadIdx.x == 0) {
    mbar_init(bar_q_full, 1);
    for (int i = 0; i < KV_STAGES; ++i) {
      mbar_init(bar_kv_full + 8 * i, 1);
      mbar_init(bar_kv_empty + 8 * i, 1);
      mbar_init(bar_o_full + 8 * i, 1);
    }
    mbar_init(bar_s_full, 1);
    mbar_init(bar_s_free, 128);
    mbar_init(bar_p_full, 128);
    fence_barrier_init();
    tma_prefetch_desc(&maps.m[b]);
  }
  if (warp == W_MMA) {
    tmem_alloc(smem_u32((const void*)tmem_slot), TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_s = tmem;
  const uint32_t tmem_p = tmem + 128;  // P as the A operand of P V: lane = query row, column k/2 holds keys (k, k+1)
  const uint32_t tmem_o = tmem + 192;

  if (warp == W_TMA) {
    // ===== TMA producer ===============================================================================================
    if (lane == 0) {
      const void* map = &maps.m[b];
      mbar_expect_tx(bar_q_full, TILE_BYTES);
      tma_load_3d(sbase + FwdSmem::Q, map, bar_q_full, h * DH, off, jseg + q0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1, use = j >> 1;
        mbar_wait(bar_kv_empty + 8 * st, (use & 1) ^ 1);
        mbar_expect_tx(bar_kv_full + 8 * st, 2 * TILE_BYTES);
        tma_load_3d(sbase + FwdSmem::K + st * TILE_BYTES, map, bar_kv_full + 8 * st, E + h * DH, off, jseg + j * BT);
        tma_load_3d(sbase + FwdSmem::V + st * TILE_BYTES, map, bar_kv_full + 8 * st, 2 * E + h * DH, off, jseg + j * BT);
      }
    }
  } else if (warp == W_MMA) {
    // ===== MMA issuer =================================================================================================
    constexpr uint32_t IDESC_QK = umma_idesc_bf16(BT, BT, 0, 0);
    constexpr uint32_t IDESC_PV = umma_idesc_bf16(BT, DH, 0, 1);
    // descriptors are built once; inside the loops an MMA costs one UTCHMMA (+ a constant descriptor advance)
    const uint64_t q_desc = umma_smem_desc(sbase + FwdSmem::Q, 16, 1024);
    const uint64_t k_desc0 = umma_smem_desc(sbase + FwdSmem::K, 16, 1024);
    const uint64_t k_desc1 = umma_smem_desc(sbase + FwdSmem::K + TILE_BYTES, 16, 1024);
    const uint64_t v_desc0 = umma_smem_desc(sbase + FwdSmem::V, TILE_BYTES, 1024);
    const uint64_t v_desc1 = umma_smem_desc(sbase + FwdSmem::V + TILE_BYTES, TILE_BYTES, 1024);
    auto issue_qk = [&](int j) {  // S = Q K_j^T : three k-steps of 16 inside the 128-byte swizzle atom
      if (elect_one()) {
        const uint64_t kd = (j & 1) ? k_desc1 : k_desc0;
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          umma_ss(tmem_s, umma_desc_adv(q_desc, k * 32), umma_desc_adv(kd, k * 32), IDESC_QK, k > 0);
        umma_commit(bar_s_full);
      }
      __syncwarp();
    };
    MT_TRACE_DECL
    mbar_wait(bar_q_full, 0);
    mbar_wait(bar_kv_full, 0);
    tc_fence_after();
    MT_TRACE(0);
    issue_qk(0);
    for (int j = 0; j < n_kv; ++j) {
      if (j + 1 < n_kv) {
        mbar_wait(bar_kv_full + 8 * ((j + 1) & 1), ((j + 1) >> 1) & 1);
        MT_TRACE(100 + j);
        mbar_wait(bar_s_free, j & 1);  // the softmax threads have read S_j out of TMEM
        tc_fence_after();
        MT_TRACE(200 + j);
        issue_qk(j + 1);
      }
      mbar_wait(bar_p_full, j & 1);    // P_j is in TMEM (and the O tile of P_{j-1} V_{j-1} has been folded)
      tc_fence_after();
      MT_TRACE(300 + j);
      if (elect_one()) {
        // O_tile = P_j V_j : A = P straight from TMEM (16 keys = 8 packed columns per k-step), B = V in place as an
        // MN-major operand (keys are the rows of the tile: 16 rows = 2048 B per k-step)
        const uint64_t vd = (j & 1) ? v_desc1 : v_desc0;
#pragma unroll
        for (int k = 0; k < BT / 16; ++k)
          umma_ts(tmem_o, tmem_p + k * 8, umma_desc_adv(vd, k * 2048), IDESC_PV, (j > 0) || (k > 0));
        umma_commit(bar_kv_empty + 8 * (j & 1));
        umma_commit(bar_o_full);
      }
      __syncwarp();
    }
    if (lane == 0) { MT_TRACE_DUMP("mma"); }
  } else {
    // ===== softmax: one query row per thread; O accumulates in TMEM over the whole key loop =========================
    // The row maximum used for the exponentials is only raised when the new maximum exceeds it by more than 8 in the
    // log2 domain (P <= 2^8 stays exact enough in bf16, l is fp32): the O accumulator then never needs the per-tile
    // rescale, and in the rare tile where a row does move, its warp rescales its 32 rows of O in TMEM in place.
    const int lane_grp = warp & 3;                    // TMEM lanes this warp may touch: [32*lane_grp, +32)
    constexpr int half = 0;
    constexpr int NC = BT;                            // score columns per thread
    constexpr int OC = DH;                            // output columns per thread
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    float m_used = -INFINITY, l_run = 0.f;
    const float scale_log2 = P.scale_log2;
    MT_TRACE_DECL
    auto tile = [&](int j, auto mask_tag) {
      constexpr bool MASK = decltype(mask_tag)::value;
      const int kvalid = bg.m - j * BT;  // key slots of this tile that belong to the segment (>= 1)
      MT_TRACE(1000 + j);
      mbar_wait(bar_s_full, j & 1);
      tc_fence_after();
      MT_TRACE(1100 + j);
      float sv[NC];
      tmem_ld64(tmem_s + t_lane + half * NC, sv);
      tmem_ld64(tmem_s + t_lane + 64, sv + 64);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bar_s_free);          // S_j is in registers: the MMA warp may overwrite it with S_{j+1}
      if (MASK) {
#pragma unroll
        for (int i = 0; i < NC; ++i) sv[i] = (half * NC + i < kvalid) ? sv[i] : -INFINITY;
      }
      float mx = fmax3(sv[0], sv[1], sv[2]);
#pragma unroll
      for (int i = 3; i + 1 < NC; i += 2) mx = fmax3(mx, sv[i], sv[i + 1]);
      mx = fmaxf(mx, sv[NC - 1]);
      MT_TRACE(1200 + j);
      bool waited = false;
      if (j == 0) {
        m_used = mx;
      } else {
        const bool need = (mx - m_used) * scale_log2 > 8.f;
        if (__any_sync(0xffffffffu, need)) {
          mbar_wait(bar_o_full, (j - 1) & 1);   // P V of tile j-1 has completed: O may be touched
          tc_fence_after();
          waited = true;
          const float alpha = need ? ex2((m_used - mx) * scale_log2) : 1.f;
          float t[8];
#pragma unroll
          for (int c = 0; c < OC / 8; ++c) {
            tmem_ld8(tmem_o + t_lane + half * OC + c * 8, t);
            tmem_ld_wait();
            uint32_t u[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = __float_as_uint(t[i] * alpha);
            tmem_st8(tmem_o + t_lane + half * OC + c * 8, u);
          }
          if (need) {
            l_run *= alpha;
            m_used = mx;
          }
        }
      }
      const float mb = m_used * scale_log2;
      if (j > 0 && !waited) {             // P_j overwrites P_{j-1}: its P V must have read it
        mbar_wait(bar_o_full, (j - 1) & 1);
        tc_fence_after();
      }
      MT_TRACE(1300 + j);
      float rs = 0.f;
#pragma unroll
      for (int c = 0; c < NC / 32; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          // MT_FWD_POLY of every 8 exponentials run as an FMA-pipe polynomial (full tiles only: masked slots need
          // ex2(-inf) = 0 exactly)
          const float x0 = fmaf(sv[c * 32 + i], scale_log2, -mb);
          const float x1 = fmaf(sv[c * 32 + i + 1], scale_log2, -mb);
#ifndef MT_EXP_NO_MUFU  // experiment builds only: the loop without the exponentials (wrong results)
          const float p0 = (!MASK && (i & 7) < MT_FWD_POLY) ? ex2_poly(x0) : ex2(x0);
          const float p1 = (!MASK && ((i + 1) & 7) < MT_FWD_POLY) ? ex2_poly(x1) : ex2(x1);
#else
          const float p0 = x0 * 0.01f, p1 = x1 * 0.01f;
#endif
          rs += p0 + p1;
          pk[i >> 1] = pack_bf16(p0, p1);
        }
#ifndef MT_EXP_NO_PST   // experiment builds only: time the loop without the P stores (wrong results)
        tmem_st16(tmem_p + t_lane + half * (NC / 2) + c * 16, pk);  // 32 keys = 16 packed columns
#else
        if (pk[0] == 0x12345678u && pk[15] == 0x9abcdef0u) l_run += 1.f;
#endif
      }
      l_run += rs;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar_p_full);
      MT_TRACE(1400 + j);
    };
    for (int j = 0; j < n_kv; ++j) {
      if (bg.m - j * BT >= BT) tile(j, std::false_type{});
      else tile(j, std::true_type{});
    }
    mbar_wait(bar_o_full, (n_kv - 1) & 1);
    tc_fence_after();
    if (warp == 0 && lane == 0) { MT_TRACE_DUMP("smx"); }
    // ---- epilogue: normalise and write the compact per-branch output ---------------------------------------------
    const int slot = q0 + row;
    const int pos = s * bg.g + off + slot * bg.r;
    const int seg_end = min(N, (s + 1) * bg.g);
    float o_acc[OC];
#pragma unroll
    for (int c = 0; c < OC / 8; ++c) {
      float t[8];
      tmem_ld8(tmem_o + t_lane + half * OC + c * 8, t);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 8; ++i) o_acc[c * 8 + i] = t[i];
    }
    if (n_zero_tail > 0) {   // the zero keys of the tiles that were skipped
      const float m_fin = fmaxf(m_used, 0.f);
      const float alpha = ex2((m_used - m_fin) * scale_log2);
      l_run = l_run * alpha + (float)n_zero_tail * ex2(-m_fin * scale_log2);
#pragma unroll
      for (int i = 0; i < OC; ++i) o_acc[i] *= alpha;
      m_used = m_fin;
    }
    if (slot < bg.m && pos < seg_end) {
      const float inv = 1.f / l_run;
      const int slot_h = h - off * bg.hpb;
      __nv_bfloat16* dst = o_br + bg.o_off + ((int64_t)pos * bg.hpb + slot_h) * DH + half * OC;
#pragma unroll
      for (int c = 0; c < OC / 8; ++c) {
        uint4 u;
        u.x = pack_bf16(o_acc[c * 8 + 0] * inv, o_acc[c * 8 + 1] * inv);
        u.y = pack_bf16(o_acc[c * 8 + 2] * inv, o_acc[c * 8 + 3] * inv);
        u.z = pack_bf16(o_acc[c * 8 + 4] * inv, o_acc[c * 8 + 5] * inv);
        u.w = pack_bf16(o_acc[c * 8 + 6] * inv, o_acc[c * 8 + 7] * inv);
        *reinterpret_cast<uint4*>(dst + c * 8) = u;
      }
      if (half == 0) lse_br[bg.lse_off + (int64_t)pos * bg.hpb + slot_h] = m_used * P.scale + logf(l_run);
    }
  }
  // ---- teardown ------------------------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, TMEM_COLS);
  MT_TL_END(n_kv)
}

// ---------------------------------------------------------------------------------------------------------------------
// forward with 48-key score tiles (impl 3): the same pipeline as dilated_fwd_sm100_kernel with S 48 + P 24 + O 48 = 120
// TMEM columns (a 128-column allocation) and 40 KB of shared memory per CTA, so FOUR CTAs are resident per SM instead of
// two: sixteen softmax warps (four per scheduler) keep the MUFU pipe fed where two per scheduler leave it idle 23 % of
// the time (DESIGN.md 4.1).  The Q K^T MMAs are N = 48 (bound by the A read: 3 x 46 cycles per tile), P V is three
// k-steps; per 128 x 128 score block that is ~560 tensor cycles against the 1 024-cycle MUFU floor.
// ---------------------------------------------------------------------------------------------------------------------
#ifndef MT_K48_KT
#define MT_K48_KT 48
#endif
static constexpr int KT = MT_K48_KT;          // key slots per score tile: 48 (or 32 in experiment builds)
static constexpr int KT_BYTES = KT * 128;     // [48 key slots][128 B], SWIZZLE_128B: six 1 KB atoms
static constexpr uint32_t TMEM48_COLS = 128;  // S: [0,48)  P (bf16 pairs): [48,72)  O: [80,128)
#ifndef MT_K48_STAGES
#define MT_K48_STAGES 3
#endif
#ifndef MT_K48_POLY
#define MT_K48_POLY 0                        // exponentials per 8 computed on the FMA pipes (ex2_poly)
#endif
#ifndef MT_K48_PACKED
#define MT_K48_PACKED 1
#endif
static constexpr int KS = MT_K48_STAGES;     // K / V ring stages
struct Fwd48Smem {
  static constexpr int Q = 0;
  static constexpr int K = Q + TILE_BYTES;
  static constexpr int V = K + KS * KT_BYTES;
  static constexpr int BAR = V + KS * KT_BYTES;
  // barriers (8 B each): q_full, s_full, s_free, p_full, o_full[2], kv_full[KS], kv_empty[KS]; then the TMEM pointer
  static constexpr int NBAR = 6 + 2 * KS;
  static constexpr int TMEM_PTR = BAR + NBAR * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
};

__global__ void __launch_bounds__(FWD_THREADS, 4)
dilated_fwd_sm100_k48_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ TensorMaps kv_maps,
                             const Sm100Params P, __nv_bfloat16* __restrict__ o_br,
                         float* __restrict__ lse_br) {
  MT_TL_BEGIN
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  // roles by warp id: the scheduler favours high warp ids, so the latency-critical single-thread roles sit last
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_TMA = 4, W_MMA = 5;
  if ((sbase & 1023u) != 0) {  // SWIZZLE_128B tiles need 1024-byte alignment; never expected, but fail loudly
    __trap();
  }
  // ---- which tile -------------------------------------------------------------------------------------------------
  int oi = 0;
  while (oi + 1 < P.geo.nb && (int)blockIdx.x >= P.item_prefix[oi + 1]) ++oi;
  const int b = P.order[oi];
  const BranchGeom bg = P.geo.b[b];
  int local = blockIdx.x - P.item_prefix[oi];
  const int qt = local % P.tiles[b];
  local /= P.tiles[b];
  const int h = local % P.geo.H;
  const int s = local / P.geo.H;
  const int H = P.geo.H, N = P.geo.N, E = H * DH;
  const int off = (h * bg.r) / H;                    // residue of the positions this head owns
  const int jseg = (s * bg.g) / bg.r;                // first slot of the segment in the branch's j axis
  const int q0 = qt * BT;
  // Zero padding (positions >= N in the last segment, dilated_attention.py:82-111) in whole tiles is never computed:
  // a query tile without a real position writes nothing, and key tiles without a real position are all zero keys
  // (score 0, value 0), whose only effect -- n_zero_tail * exp(0 - max) in the softmax denominator -- is added in
  // closed form in the epilogue.  At 32k tiles 30 % of the padded tile pairs of the reference disappear this way.
  const int seg_lo = s * bg.g + off;
  const int c_real = min(N, (s + 1) * bg.g) > seg_lo ? (min(N, (s + 1) * bg.g) - seg_lo + bg.r - 1) / bg.r : 0;
  if (q0 >= c_real) return;
  const int n_kv = min((bg.m + KT - 1) / KT, (c_real + KT - 1) / KT);
  const int n_zero_tail = max(0, bg.m - n_kv * KT);

  const uint32_t bar_q_full = sbase + Fwd48Smem::BAR + 0;
  const uint32_t bar_s_full = sbase + Fwd48Smem::BAR + 8;
  const uint32_t bar_s_free = sbase + Fwd48Smem::BAR + 16;
  const uint32_t bar_p_full = sbase + Fwd48Smem::BAR + 24;
  const uint32_t bar_o_full = sbase + Fwd48Smem::BAR + 32;    // [2]
  const uint32_t bar_kv_full = sbase + Fwd48Smem::BAR + 48;   // [KS]
  const uint32_t bar_kv_empty = bar_kv_full + 8 * KS;         // [KS]
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Fwd48Smem::TMEM_PTR);

  if (threadIdx.x == 0) {
    mbar_init(bar_q_full, 1);
    for (int i = 0; i < KS; ++i) {
      mbar_init(bar_kv_full + 8 * i, 1);
      mbar_init(bar_kv_empty + 8 * i, 1);
    }
    mbar_init(bar_o_full, 1);
    mbar_init(bar_o_full + 8, 1);
    mbar_init(bar_s_full, 1);
    mbar_init(bar_s_free, 128);
    mbar_init(bar_p_full, 128);
    fence_barrier_init();
    tma_prefetch_desc(&maps.m[b]);
    tma_prefetch_desc(&kv_maps.m[b]);
  }
  if (warp == W_MMA) {
    tmem_alloc(smem_u32((const void*)tmem_slot), TMEM48_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_s = tmem;
  const uint32_t tmem_p = tmem + KT;   // P as the A operand of P V: lane = query row, column k/2 holds keys (k, k+1)
  const uint32_t tmem_o = tmem + 80;

  if (warp == W_TMA) {
    // ===== TMA producer ===============================================================================================
    if (lane == 0) {
      const void* map = &maps.m[b];
      const void* kmap = &kv_maps.m[b];    // the same view with a 48-slot box
      mbar_expect_tx(bar_q_full, TILE_BYTES);
      tma_load_3d(sbase + Fwd48Smem::Q, map, bar_q_full, h * DH, off, jseg + q0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j % KS, use = j / KS;
        mbar_wait(bar_kv_empty + 8 * st, (use & 1) ^ 1);
        mbar_expect_tx(bar_kv_full + 8 * st, 2 * KT_BYTES);
        tma_load_3d(sbase + Fwd48Smem::K + st * KT_BYTES, kmap, bar_kv_full + 8 * st, E + h * DH, off, jseg + j * KT);
        tma_load_3d(sbase + Fwd48Smem::V + st * KT_BYTES, kmap, bar_kv_full + 8 * st, 2 * E + h * DH, off, jseg + j * KT);
      }
    }
  } else if (warp == W_MMA) {
    // ===== MMA issuer =================================================================================================
    constexpr uint32_t IDESC_QK = umma_idesc_bf16(BT, KT, 0, 0);
    constexpr uint32_t IDESC_PV = umma_idesc_bf16(BT, DH, 0, 1);
    // descriptors are built once; inside the loops an MMA costs one UTCHMMA (+ a constant descriptor advance)
    const uint64_t q_desc = umma_smem_desc(sbase + Fwd48Smem::Q, 16, 1024);
    const uint64_t k_desc0 = umma_smem_desc(sbase + Fwd48Smem::K, 16, 1024);
    const uint64_t v_desc0 = umma_smem_desc(sbase + Fwd48Smem::V, KT_BYTES, 1024);
    auto issue_qk = [&](int j) {  // S = Q K_j^T : three k-steps of 16 inside the 128-byte swizzle atom
      if (elect_one()) {
        const uint64_t kd = umma_desc_adv(k_desc0, (uint32_t)(j % KS) * KT_BYTES);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          umma_ss(tmem_s, umma_desc_adv(q_desc, k * 32), umma_desc_adv(kd, k * 32), IDESC_QK, k > 0);
        umma_commit(bar_s_full);
      }
      __syncwarp();
    };
    MT_TRACE_DECL
    mbar_wait(bar_q_full, 0);
    mbar_wait(bar_kv_full, 0);
    tc_fence_after();
    MT_TRACE(0);
    issue_qk(0);
    for (int j = 0; j < n_kv; ++j) {
      if (j + 1 < n_kv) {
        mbar_wait(bar_kv_full + 8 * ((j + 1) % KS), ((j + 1) / KS) & 1);
        MT_TRACE(100 + j);
        mbar_wait(bar_s_free, j & 1);  // the softmax threads have read S_j out of TMEM
        tc_fence_after();
        MT_TRACE(200 + j);
        issue_qk(j + 1);
      }
      mbar_wait(bar_p_full, j & 1);    // P_j is in TMEM (and the O tile of P_{j-1} V_{j-1} has been folded)
      tc_fence_after();
      MT_TRACE(300 + j);
      if (elect_one()) {
        // O_tile = P_j V_j : A = P straight from TMEM (16 keys = 8 packed columns per k-step), B = V in place as an
        // MN-major operand (keys are the rows of the tile: 16 rows = 2048 B per k-step)
        const uint64_t vd = umma_desc_adv(v_desc0, (uint32_t)(j % KS) * KT_BYTES);
#pragma unroll
        for (int k = 0; k < KT / 16; ++k)
          umma_ts(tmem_o, tmem_p + k * 8, umma_desc_adv(vd, k * 2048), IDESC_PV, (j > 0) || (k > 0));
        umma_commit(bar_kv_empty + 8 * (j % KS));
        umma_commit(bar_o_full);
      }
      __syncwarp();
    }
    if (lane == 0) { MT_TRACE_DUMP("mma"); }
  } else {
    // ===== softmax: one query row per thread; O accumulates in TMEM over the whole key loop =========================
    // The row maximum used for the exponentials is only raised when the new maximum exceeds it by more than 8 in the
    // log2 domain (P <= 2^8 stays exact enough in bf16, l is fp32): the O accumulator then never needs the per-tile
    // rescale, and in the rare tile where a row does move, its warp rescales its 32 rows of O in TMEM in place.
    const int lane_grp = warp & 3;                    // TMEM lanes this warp may touch: [32*lane_grp, +32)
    constexpr int half = 0;
    constexpr int NC = KT;                            // score columns per thread
    constexpr int OC = DH;                            // output columns per thread
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    float m_used = -INFINITY, l_run = 0.f;
    const float scale_log2 = P.scale_log2;
    MT_TRACE_DECL
    auto tile = [&](int j, auto mask_tag) {
      constexpr bool MASK = decltype(mask_tag)::value;
      const int kvalid = bg.m - j * KT;  // key slots of this tile that belong to the segment (>= 1)
      MT_TRACE(1000 + j);
      mbar_wait(bar_s_full, j & 1);
      tc_fence_after();
      MT_TRACE(1100 + j);
      float sv[NC];
      {
        float lo[32], hi[16];
        tmem_ld32(tmem_s + t_lane, lo);
        if constexpr (KT > 32) tmem_ld16(tmem_s + t_lane + 32, hi);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) sv[i] = lo[i];
        if constexpr (KT > 32) {
#pragma unroll
          for (int i = 0; i < 16; ++i) sv[32 + i] = hi[i];
        }
      }
      tc_fence_before();
      mbar_arrive(bar_s_free);          // S_j is in registers: the MMA warp may overwrite it with S_{j+1}
      if (MASK) {
#pragma unroll
        for (int i = 0; i < NC; ++i) sv[i] = (half * NC + i < kvalid) ? sv[i] : -INFINITY;
      }
      float mx = fmax3(sv[0], sv[1], sv[2]);
#pragma unroll
      for (int i = 3; i + 1 < NC; i += 2) mx = fmax3(mx, sv[i], sv[i + 1]);
      mx = fmaxf(mx, sv[NC - 1]);
      MT_TRACE(1200 + j);
      bool waited = false;
      if (j == 0) {
        m_used = mx;
      } else {
        const bool need = (mx - m_used) * scale_log2 > 8.f;
        if (__any_sync(0xffffffffu, need)) {
          mbar_wait(bar_o_full, (j - 1) & 1);   // P V of tile j-1 has completed: O may be touched
          tc_fence_after();
          waited = true;
          const float alpha = need ? ex2((m_used - mx) * scale_log2) : 1.f;
          float t[8];
#pragma unroll
          for (int c = 0; c < OC / 8; ++c) {
            tmem_ld8(tmem_o + t_lane + half * OC + c * 8, t);
            tmem_ld_wait();
            uint32_t u[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = __float_as_uint(t[i] * alpha);
            tmem_st8(tmem_o + t_lane + half * OC + c * 8, u);
          }
          if (need) {
            l_run *= alpha;
            m_used = mx;
          }
        }
      }
      const float mb = m_used * scale_log2;
      if (j > 0 && !waited) {             // P_j overwrites P_{j-1}: its P V must have read it
        mbar_wait(bar_o_full, (j - 1) & 1);
        tc_fence_after();
      }
      MT_TRACE(1300 + j);
      float rs = 0.f;
#if MT_K48_PACKED
      // packed fp32 pairs (FFMA2 / FADD2): the scale-and-shift and the row sum cost one instruction per TWO scores; with
      // four softmax warps per scheduler the kernel is at 65 % issue-active, so instructions are worth saving
      const float2 sc2 = make_float2(scale_log2, scale_log2), nb2 = make_float2(-mb, -mb);
      float2 rs2 = make_float2(0.f, 0.f);
#endif
#pragma unroll
      for (int c = 0; c < NC / 16; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
#if MT_K48_PACKED
          const float2 x = ffma2(make_float2(sv[c * 16 + i], sv[c * 16 + i + 1]), sc2, nb2);
          const float2 pp = make_float2(ex2(x.x), ex2(x.y));
          rs2 = fadd2(rs2, pp);
          pk[i >> 1] = pack_bf16(pp.x, pp.y);
#else
          const float x0 = fmaf(sv[c * 16 + i], scale_log2, -mb);
          const float x1 = fmaf(sv[c * 16 + i + 1], scale_log2, -mb);
          const float p0 = (!MASK && (i & 7) < MT_K48_POLY) ? ex2_poly(x0) : ex2(x0);
          const float p1 = (!MASK && ((i + 1) & 7) < MT_K48_POLY) ? ex2_poly(x1) : ex2(x1);
          rs += p0 + p1;
          pk[i >> 1] = pack_bf16(p0, p1);
#endif
        }
        tmem_st8(tmem_p + t_lane + c * 8, pk);   // 16 keys = 8 packed columns
      }
#if MT_K48_PACKED
      rs = rs2.x + rs2.y;
#endif
      l_run += rs;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar_p_full);
      MT_TRACE(1400 + j);
    };
    for (int j = 0; j < n_kv; ++j) {
      if (bg.m - j * KT >= KT) tile(j, std::false_type{});
      else tile(j, std::true_type{});
    }
    mbar_wait(bar_o_full, (n_kv - 1) & 1);
    tc_fence_after();
    if (warp == 0 && lane == 0) { MT_TRACE_DUMP("smx"); }
    // ---- epilogue: normalise and write the compact per-branch output ---------------------------------------------
    const int slot = q0 + row;
    const int pos = s * bg.g + off + slot * bg.r;
    const int seg_end = min(N, (s + 1) * bg.g);
    float o_acc[OC];
#pragma unroll
    for (int c = 0; c < OC / 8; ++c) {
      float t[8];
      tmem_ld8(tmem_o + t_lane + half * OC + c * 8, t);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 8; ++i) o_acc[c * 8 + i] = t[i];
    }
    if (n_zero_tail > 0) {   // the zero keys of the tiles that were skipped
      const float m_fin = fmaxf(m_used, 0.f);
      const float alpha = ex2((m_used - m_fin) * scale_log2);
      l_run = l_run * alpha + (float)n_zero_tail * ex2(-m_fin * scale_log2);
#pragma unroll
      for (int i = 0; i < OC; ++i) o_acc[i] *= alpha;
      m_used = m_fin;
    }
    if (slot < bg.m && pos < seg_end) {
      const float inv = 1.f / l_run;
      const int slot_h = h - off * bg.hpb;
      __nv_bfloat16* dst = o_br + bg.o_off + ((int64_t)pos * bg.hpb + slot_h) * DH + half * OC;
#pragma unroll
      for (int c = 0; c < OC / 8; ++c) {
        uint4 u;
        u.x = pack_bf16(o_acc[c * 8 + 0] * inv, o_acc[c * 8 + 1] * inv);
        u.y = pack_bf16(o_acc[c * 8 + 2] * inv, o_acc[c * 8 + 3] * inv);
        u.z = pack_bf16(o_acc[c * 8 + 4] * inv, o_acc[c * 8 + 5] * inv);
        u.w = pack_bf16(o_acc[c * 8 + 6] * inv, o_acc[c * 8 + 7] * inv);
        *reinterpret_cast<uint4*>(dst + c * 8) = u;
      }
      if (half == 0) lse_br[bg.lse_off + (int64_t)pos * bg.hpb + slot_h] = m_used * P.scale + logf(l_run);
    }
  }
  // ---- teardown ------------------------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, TMEM48_COLS);
  MT_TL_END(n_kv)
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 3-D view of a row-major [n_alloc, ld] bf16 matrix for dilation r: (column, residue o, slot j) -> row j*r + o
static int encode_branch_map(CUtensorMap* map, const void* base, int64_t ld, int64_t n_alloc, int r, int box_rows = BT) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return MT_E_UNSUPPORTED;
  }
  cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)r, (cuuint64_t)(n_alloc / r)};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)ld * 2 * (cuuint64_t)r};
  cuuint32_t box[3] = {64, 1, (cuuint32_t)box_rows};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for dilation %d, ld %lld, rows %lld", (int)rc, r, (long long)ld,
              (long long)n_alloc);
    return MT_E_BADARG;
  }
  return 0;
}

// fp32 [n_alloc, ld] gradient buffer, same (column, residue, slot) view, for the TMA reduce-add of dQ tiles:
// box = [128 slots][cols] floats; cols = 48 unswizzled (dense staging tile), or 32 / 16 with the 128 B / 64 B swizzle
// (row pitch = swizzle span, so that one-row-per-thread staging stores are bank-conflict free)
static int encode_branch_map_f32(CUtensorMap* map, const void* base, int64_t ld, int64_t n_alloc, int r, int cols = DH) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return MT_E_UNSUPPORTED;
  }
  cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)r, (cuuint64_t)(n_alloc / r)};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)ld * 4 * (cuuint64_t)r};
  cuuint32_t box[3] = {(cuuint32_t)cols, 1, (cuuint32_t)BT};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle swz = cols == 32 ? CU_TENSOR_MAP_SWIZZLE_128B
                                            : (cols == 16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (fp32, %d columns) failed (%d) for dilation %d", cols, (int)rc, r);
    return MT_E_BADARG;
  }
  return 0;
}

static int make_sm100_params(const mt_dilated_geometry* geom, Sm100Params* P) {
  int rc = make_dilated_geom(geom, &P->geo);
  if (rc) return rc;
  if (P->geo.D != DH || P->geo.H != 16) {
    set_error("tcgen05 dilated attention is built for 16 heads x 48 (got %d x %d)", P->geo.H, P->geo.D);
    return MT_E_UNSUPPORTED;
  }
  const int nb = P->geo.nb;
  for (int b = 0; b < nb; ++b) {
    P->tiles[b] = (P->geo.b[b].m + BT - 1) / BT;
    P->order[b] = b;
  }
  for (int i = 0; i < nb; ++i)  // longest key loops first
    for (int j = i + 1; j < nb; ++j)
      if (P->tiles[P->order[j]] > P->tiles[P->order[i]]) {
        int t = P->order[i];
        P->order[i] = P->order[j];
        P->order[j] = t;
      }
  int total = 0;
  for (int i = 0; i < nb; ++i) {
    const int b = P->order[i];
    P->item_prefix[i] = total;
    total += P->geo.b[b].n_seg * P->geo.H * P->tiles[b];
  }
  P->item_prefix[nb] = total;
  P->scale = 1.0f / sqrtf((float)DH);
  P->scale_log2 = P->scale * 1.4426950408889634f;
  return 0;
}

// Work counters of the persistent kernels: a ring of {next item, finished CTAs} pairs in device memory, zero at rest (the
// last CTA of a launch re-arms its pair).  Consecutive launches take consecutive pairs, so launches that overlap on
// different streams (the three task passes of a step) never share one; a pair comes round again 256 launches later.
static int* next_work_counter() {
  static int* ring[64] = {nullptr};          // per device
  static unsigned seq = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (ring[dev] == nullptr) {
    if (cudaMalloc(&ring[dev], 256 * 2 * sizeof(int)) != cudaSuccess) return nullptr;
    if (cudaMemset(ring[dev], 0, 256 * 2 * sizeof(int)) != cudaSuccess) return nullptr;
  }
  return ring[dev] + 2 * (seq++ % 256);
}

int dilated_attn_fwd_sm100(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                           void* o_br, float* lse_br, int impl, cudaStream_t st) {
  Sm100Params P;
  int rc = make_sm100_params(geom, &P);
  if (rc) return rc;
  MT_REQUIRE(n_alloc >= P.geo.N && n_alloc % 128 == 0, "dilated_attn_fwd: n_alloc must be a multiple of 128 >= n_tokens");
  MT_REQUIRE(qkv_ld % 8 == 0 && ((uintptr_t)qkv & 15) == 0, "dilated_attn_fwd: qkv must be 16-byte aligned");
  TensorMaps maps;
  memset(&maps, 0, sizeof(maps));
  for (int b = 0; b < P.geo.nb; ++b) {
    rc = encode_branch_map(&maps.m[b], qkv, qkv_ld, n_alloc, P.geo.b[b].r);
    if (rc) return rc;
  }
  if (impl == 3) {   // 48-key score tiles, four CTAs per SM
    TensorMaps kv_maps;
    memset(&kv_maps, 0, sizeof(kv_maps));
    for (int b = 0; b < P.geo.nb; ++b) {
      rc = encode_branch_map(&kv_maps.m[b], qkv, qkv_ld, n_alloc, P.geo.b[b].r, KT);
      if (rc) return rc;
    }
    static bool attr_set = false;
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(dilated_fwd_sm100_k48_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Fwd48Smem::TOTAL));
      attr_set = true;
    }
    dilated_fwd_sm100_k48_kernel<<<P.item_prefix[P.geo.nb], FWD_THREADS, Fwd48Smem::TOTAL, st>>>(
        maps, kv_maps, P, (__nv_bfloat16*)o_br, lse_br);
    return check_launch("dilated_fwd_sm100_k48_kernel");
  }
  MT_REQUIRE(impl == 1, "dilated_attn_fwd: impl must be 0 (SIMT), 1 (128-key tiles) or 3 (48-key tiles, default); the "
             "persistent forward of round 2 (impl 2) measured 4 %% slower than impl 1 and was removed");
  {
    static bool attr_set = false;   // once per process: the call is not free and never changes
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(dilated_fwd_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdSmem::TOTAL));
      attr_set = true;
    }
  }
  dilated_fwd_sm100_kernel<<<P.item_prefix[P.geo.nb], FWD_THREADS, FwdSmem::TOTAL, st>>>(
      maps, P, (__nv_bfloat16*)o_br, lse_br);
  return check_launch("dilated_fwd_sm100_kernel");
}

// =====================================================================================================================
// backward
// =====================================================================================================================
// =====================================================================================================================
// backward, third version: the per-query statistics ride on the tensor cores
// =====================================================================================================================
// Same transposed formulation as version 2 (keys on the TMEM lanes, K / V resident in TMEM, P^T / dS^T written back to
// TMEM as the A operands of dV / dK).  What changed, each item measured on B200 (tools/ubench, MT_DEBUG_TRACE):
//   * the 64-column (128-byte) tile rows only carry 48 head columns, so columns 48..51 are used as an AUGMENTED
//     contraction: a dedicated warp overwrites them in every Q tile with the 3-way bf16 split of -lse/scale (and a
//     -32768 mask column) and in every dO tile with the split of -delta; K' / V' in TMEM carry ones there.  The MMAs
//     then deliver S^T - lse/scale and dP^T - delta directly (fp32 accumulation of exact 1 x bf16 products): no
//     per-query statistics ring in shared memory, no broadcast loads, no subtraction per element.  Key rows past the
//     segment's m get a one in the mask column (S = -32768 -> P = 0), queries that do not exist get -32768 as their lse.
//   * all 16 compute warps work on the SAME 64-query half tile (16 scores per thread) while the MMAs of the other
//     half run, instead of two groups of 8 warps ping-ponging over 32 scores per thread.
//   * the MMA issue loop is unrolled over stages x halves: every descriptor is a base plus a compile-time constant
//     (the single issuing thread shares its scheduler with busy warps; its instructions are critical-path latency).
//   * dQ, dK and dV leave through swizzled fp32 staging tiles and TMA reduce-adds (cp.reduce.async.bulk.tensor)
//     instead of red.global from registers, which costs one L1 request per row and instruction (~1500 LSU cycles per
//     dQ tile).  fp32 reduce-adds saturate at ~5.3 TB/s chip-wide (tools/ubench/red_rate.cu): ~1300 cycles per dQ tile
//     and SM, so the staging tile is a buffer of its own and nobody but the drain warps ever waits for it.
//   * separate warps for the TMA issue, the statistics columns and the dQ drain; the first loads are issued before
//     the CTA-wide setup barrier.
// scale is applied to dQ and dK when they leave TMEM (dS is kept as P (dP - delta)).
static constexpr int BWD3_THREADS = 32 * 23;   // 16 compute, 4 dQ drain, TMA, statistics, MMA
struct Bwd3Smem {
  static constexpr int NQ = 3;
  static constexpr int K = 0;
  static constexpr int V = K + TILE_BYTES;
  static constexpr int Q = V + TILE_BYTES;                 // [NQ]
  static constexpr int DO = Q + NQ * TILE_BYTES;           // [NQ]
  static constexpr int DS = DO + NQ * TILE_BYTES;          // [2] dS^T tiles: [128 key rows][2 blocks of 64 queries]
  static constexpr int STG = DS + 4 * TILE_BYTES;          // fp32 staging tile of the dQ reduce-add (24 KB)
  static constexpr int BAR = STG + BT * DH * 4;
  // kv_full, kvt_full, st_full[2], pt_full[2], dq_full, dq_free, done, qdo_full[NQ], qdo_empty[NQ], aug_full[NQ]
  static constexpr int NBAR = 9 + 3 * NQ;
  static constexpr int TMEM_PTR = BAR + NBAR * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
  // fp32 staging of a [128][48] gradient tile: columns 0..31 as [128][32] with the 128 B
  // swizzle, columns 32..47 as [128][16] with the 64 B swizzle (row pitch = swizzle span: one-row-per-thread stores are
  // bank-conflict free); each part is the box of one TMA reduce-add
  static constexpr int STG16 = BT * 128;
};
static_assert(Bwd3Smem::TOTAL <= 232448, "shared memory of the backward kernel");

__device__ __forceinline__ void split3_bf16(float a, uint32_t& w0, uint32_t& w1, float fourth) {
  const __nv_bfloat16 hi = __float2bfloat16_rn(a);
  const float r1 = a - __bfloat162float(hi);
  const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(mid);
  w0 = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(mid) << 16);
  w1 = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(r2)) |
       ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(fourth)) << 16);
}

// 16-byte chunk c (4 floats, columns 4c..4c+3 of 48) of row `row` of a staged fp32 gradient tile
__device__ __forceinline__ void stage_chunk(uint8_t* stg, int row, int c, float4 v) {
  uint8_t* dst = c < 8 ? stg + row * 128 + ((c ^ (row & 7)) << 4)
                       : stg + Bwd3Smem::STG16 + row * 64 + (((c - 8) ^ ((row >> 1) & 3)) << 4);
  *reinterpret_cast<float4*>(dst) = v;
}

// WITH_DQ = false (impl 4, the deterministic backward): dK / dV only -- no dQ MMA, no dS^T shared-memory tile (it only
// feeds that MMA) and idle drain warps; dQ comes from dilated_bwd_dq_sm100_kernel.  Every key slot of a branch belongs to
// exactly one key tile, so its dK / dV rows receive one non-zero reduce-add per launch.
template <bool WITH_DQ>
__global__ void __launch_bounds__(BWD3_THREADS, 1)
dilated_bwd_sm100_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ TensorMaps do_maps,
                          const __grid_constant__ TensorMaps dq32_maps, const __grid_constant__ TensorMaps dq16_maps,
                          const Sm100Params P, const float* __restrict__ lse, const float* __restrict__ delta_br) {
  MT_TL_BEGIN
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  // roles by warp id: compute 0-15, dQ drain 16-19, TMA 20, statistics columns 21, MMA 22 (last: the scheduler
  // favours high warp ids and the single-thread issuer must never starve)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_DRAIN = 16, W_TMA = 20, W_AUG = 21, W_MMA = 22;
  if ((sbase & 1023u) != 0) {
    __trap();
  }
  int oi = 0;
  while (oi + 1 < P.geo.nb && (int)blockIdx.x >= P.item_prefix[oi + 1]) ++oi;
  const int b = P.order[oi];
  const BranchGeom bg = P.geo.b[b];
  int local = blockIdx.x - P.item_prefix[oi];
  const int kt = local % P.tiles[b];
  local /= P.tiles[b];
  const int h = local % P.geo.H;
  const int s = local / P.geo.H;
  const int H = P.geo.H, N = P.geo.N, E = H * DH;
  const int off = (h * bg.r) / H;
  const int jseg = (s * bg.g) / bg.r;
  const int k0 = kt * BT;
  const int seg_end = min(N, (s + 1) * bg.g);
  const int slot_h = h - off * bg.hpb;
  // Whole tiles of zero padding (positions >= N in the last segment) are skipped: a zero key tile has K = V = 0, so it
  // adds nothing to dQ and its own dK / dV rows are scratch; a padding query tile has P = 0.
  const int seg_lo = s * bg.g + off;
  const int c_real = seg_end > seg_lo ? (seg_end - seg_lo + bg.r - 1) / bg.r : 0;   // real slots of this (segment, head)
  if (k0 >= c_real) return;
  const int n_q = min(P.tiles[b], (c_real + BT - 1) / BT);

  constexpr int NQ = Bwd3Smem::NQ;
  const uint32_t bar_kv_full = sbase + Bwd3Smem::BAR + 0;
  const uint32_t bar_kvt_full = sbase + Bwd3Smem::BAR + 8;
  const uint32_t bar_st_full = sbase + Bwd3Smem::BAR + 16;     // [2]
  const uint32_t bar_pt_full = sbase + Bwd3Smem::BAR + 32;     // [2]
  const uint32_t bar_dq_full = sbase + Bwd3Smem::BAR + 48;
  const uint32_t bar_dq_free = sbase + Bwd3Smem::BAR + 56;
  const uint32_t bar_done = sbase + Bwd3Smem::BAR + 64;        // every MMA of the CTA has completed
  const uint32_t bar_qdo_full = sbase + Bwd3Smem::BAR + 72;    // [NQ] TMA landed
  const uint32_t bar_qdo_empty = bar_qdo_full + 8 * NQ;        // [NQ]
  const uint32_t bar_aug_full = bar_qdo_empty + 8 * NQ;        // [NQ] statistics columns written into the stage
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Bwd3Smem::TMEM_PTR);
  constexpr int NCOMP = 512;

  if (warp == W_TMA && lane == 0) {
    // barrier setup and the first loads by the producer itself, ahead of the CTA-wide sync: the first tiles are on
    // the critical path of every CTA (one CTA per SM, nothing overlaps its prologue)
    mbar_init(bar_kv_full, 1);
    mbar_init(bar_kvt_full, 256);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_st_full + 8 * i, 1);
      mbar_init(bar_pt_full + 8 * i, NCOMP);
    }
    for (int i = 0; i < NQ; ++i) {
      mbar_init(bar_qdo_full + 8 * i, 1);
      mbar_init(bar_qdo_empty + 8 * i, 1);
      mbar_init(bar_aug_full + 8 * i, 32);
    }
    mbar_init(bar_dq_full, 1);
    mbar_init(bar_dq_free, 128);
    mbar_init(bar_done, 1);
    fence_barrier_init();
    const void* map = &maps.m[b];
    const void* dmap = &do_maps.m[b];
    mbar_expect_tx(bar_kv_full, 2 * TILE_BYTES);
    tma_load_3d(sbase + Bwd3Smem::K, map, bar_kv_full, E + h * DH, off, jseg + k0);
    tma_load_3d(sbase + Bwd3Smem::V, map, bar_kv_full, 2 * E + h * DH, off, jseg + k0);
    for (int i = 0; i < NQ && i < n_q; ++i) {
      mbar_expect_tx(bar_qdo_full + 8 * i, 2 * TILE_BYTES);
      tma_load_3d(sbase + Bwd3Smem::Q + i * TILE_BYTES, map, bar_qdo_full + 8 * i, h * DH, off, jseg + i * BT);
      tma_load_3d(sbase + Bwd3Smem::DO + i * TILE_BYTES, dmap, bar_qdo_full + 8 * i, h * DH, off, jseg + i * BT);
    }
    tma_prefetch_desc(&dq32_maps.m[b]);
    tma_prefetch_desc(&dq16_maps.m[b]);
  }
  if (warp == W_MMA) {
    tmem_alloc(smem_u32((const void*)tmem_slot), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // columns: [0,64) S^T buf0 | [64,128) dP^T buf0 | [128,192) S^T buf1 | [192,256) dP^T buf1 | dV 256 | dK 320 | dQ 384
  //          K' (64 bf16 = 32 columns) 448 | V' 480
  const uint32_t tm_dv = tmem + 256, tm_dk = tmem + 320, tm_dq = tmem + 384, tm_k = tmem + 448, tm_v = tmem + 480;

  if (warp == W_TMA) {
    // ===== TMA producer (tiles >= NQ; the first NQ were issued above) ================================================
    if (lane == 0) {
      const void* map = &maps.m[b];
      const void* dmap = &do_maps.m[b];
      for (int i = NQ; i < n_q; ++i) {
        const int st = i % NQ, use = i / NQ;
        mbar_wait(bar_qdo_empty + 8 * st, (use & 1) ^ 1);
        mbar_expect_tx(bar_qdo_full + 8 * st, 2 * TILE_BYTES);
        tma_load_3d(sbase + Bwd3Smem::Q + st * TILE_BYTES, map, bar_qdo_full + 8 * st, h * DH, off, jseg + i * BT);
        tma_load_3d(sbase + Bwd3Smem::DO + st * TILE_BYTES, dmap, bar_qdo_full + 8 * st, h * DH, off, jseg + i * BT);
      }
    }
  } else if (warp == W_AUG) {
    // ===== statistics columns: lane owns rows lane + 32 j of every Q / dO tile ==========================================
    const float inv_sc = 1.f / P.scale;
    float lr[4], dr[4], ln[4], dn[4];
    // raw per-query statistics of tile i: strided 4-byte loads issued one tile ahead; consumed (and masked) at use
    auto load_raw = [&](int i, float (&l)[4], float (&d)[4]) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int slot = i * BT + lane + 32 * j;
        const int pos = s * bg.g + off + slot * bg.r;
        const bool qok = i < n_q && slot < bg.m && pos < seg_end;
        const int pc = qok ? pos : 0;
        l[j] = lse[(int64_t)pc * H + h];
        d[j] = delta_br[bg.lse_off + (int64_t)pc * bg.hpb + slot_h];
      }
    };
    load_raw(0, lr, dr);
    for (int i = 0; i < n_q; ++i) {
      load_raw(i + 1, ln, dn);
      const int st = i % NQ;
      mbar_wait(bar_qdo_full + 8 * st, (i / NQ) & 1);      // the TMA has written the stage
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int row = lane + 32 * j;
        const int slot = i * BT + row;
        const int pos = s * bg.g + off + slot * bg.r;
        const bool qok = slot < bg.m && pos < seg_end;
        uint32_t w0, w1;
        // columns 48..55 (16-byte chunk 6) of the row: [hi, mid, lo, mask, 0, 0, 0, 0]
        split3_bf16(qok ? -lr[j] * inv_sc : -32768.f, w0, w1, -32768.f);   // -32768 -> P = 0 for rows that do not exist
        *reinterpret_cast<uint4*>(smem + Bwd3Smem::Q + st * TILE_BYTES + row * 128 + ((6 ^ (row & 7)) << 4)) =
            make_uint4(w0, w1, 0u, 0u);
        split3_bf16(qok ? -dr[j] : 0.f, w0, w1, 0.f);
        *reinterpret_cast<uint4*>(smem + Bwd3Smem::DO + st * TILE_BYTES + row * 128 + ((6 ^ (row & 7)) << 4)) =
            make_uint4(w0, w1, 0u, 0u);
      }
      fence_proxy_async_smem();
      mbar_arrive(bar_aug_full + 8 * st);
#pragma unroll
      for (int j = 0; j < 4; ++j) { lr[j] = ln[j]; dr[j] = dn[j]; }
    }
  } else if (warp == W_MMA) {
    // ===== MMA issuer =================================================================================================
    constexpr uint32_t IDESC_ST = umma_idesc_bf16(BT, 64, 0, 0);    // A = K' / V' (TMEM), B = Q' / dO' half tile (K-major)
    constexpr uint32_t IDESC_TS = umma_idesc_bf16(BT, DH, 0, 1);    // A = P^T / dS^T (TMEM), B = dO / Q (MN-major)
    constexpr uint32_t IDESC_DQ = umma_idesc_bf16(BT, DH, 1, 1);    // A = dS^T tile (smem, MN-major), B = K (MN-major)
    const int n_half = 2 * n_q;
    const uint64_t qk_desc = umma_smem_desc(sbase + Bwd3Smem::Q, 16, 1024);          // K-major views (stage 0)
    const uint64_t dk_desc = umma_smem_desc(sbase + Bwd3Smem::DO, 16, 1024);
    const uint64_t qm_desc = umma_smem_desc(sbase + Bwd3Smem::Q, TILE_BYTES, 1024);  // MN-major views (stage 0)
    const uint64_t dm_desc = umma_smem_desc(sbase + Bwd3Smem::DO, TILE_BYTES, 1024);
    const uint64_t k_mn_desc = umma_smem_desc(sbase + Bwd3Smem::K, TILE_BYTES, 1024);
    const uint64_t ds_desc0 = umma_smem_desc(sbase + Bwd3Smem::DS, TILE_BYTES, 1024);
    const uint64_t ds_desc1 = umma_smem_desc(sbase + Bwd3Smem::DS + 2 * TILE_BYTES, TILE_BYTES, 1024);
    auto issue_st = [&](auto U) {  // S'^T and dP'^T of a half tile (stage U / 2, half U & 1) into TMEM buffer U & 1
      constexpr int u = decltype(U)::value;
      if (elect_one()) {
        constexpr uint32_t so = (uint32_t)((u >> 1) * TILE_BYTES + (u & 1) * 64 * 128);
        const uint32_t ts = tmem + (u & 1) * 128, td = ts + 64;
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ts(ts, tm_k + k * 8, umma_desc_adv(qk_desc, so + k * 32), IDESC_ST, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ts(td, tm_v + k * 8, umma_desc_adv(dk_desc, so + k * 32), IDESC_ST, k > 0);
        umma_commit(bar_st_full + 8 * (u & 1));
      }
      __syncwarp();
    };
    MT_TRACE_DECL
    mbar_wait(bar_kvt_full, 0);       // K' and V' are in TMEM
    mbar_wait(bar_qdo_full, 0);
    mbar_wait(bar_aug_full, 0);
    tc_fence_after();
    MT_TRACE(0);
    issue_st(std::integral_constant<int, 0>{});
    issue_st(std::integral_constant<int, 1>{});
    // one half tile: t = trip of the unrolled loop (tile i = NQ * t + U / 2)
    auto half = [&](int g, int t, auto U) {
      constexpr int u = decltype(U)::value;
      constexpr int st = u >> 1, hh = u & 1;
      const int i = g >> 1;
      mbar_wait(bar_pt_full + 8 * hh, i & 1);   // P^T, dS^T of half g are in TMEM (+ dS^T half in smem)
      tc_fence_after();
      MT_TRACE(100 + g);
      if (elect_one()) {
        constexpr uint32_t so = (uint32_t)(st * TILE_BYTES + hh * 64 * 128);
        const uint32_t ts = tmem + hh * 128, td = ts + 64;
        // packed P^T / dS^T: query pair (2c, 2c+1) of 16-query quarter qq sits in column 16*qq + c of its buffer;
        // 64 queries = 4 k-steps of 16 (rows of the dO / Q half tile: 2048 B each)
        umma_ts(tm_dv, ts, umma_desc_adv(dm_desc, so), IDESC_TS, g > 0);
#pragma unroll
        for (int k = 1; k < 4; ++k) umma_ts(tm_dv, ts + k * 16, umma_desc_adv(dm_desc, so + k * 2048), IDESC_TS, 1);
        umma_ts(tm_dk, td, umma_desc_adv(qm_desc, so), IDESC_TS, g > 0);
#pragma unroll
        for (int k = 1; k < 4; ++k) umma_ts(tm_dk, td + k * 16, umma_desc_adv(qm_desc, so + k * 2048), IDESC_TS, 1);
        if (hh == 1) umma_commit(bar_qdo_empty + 8 * st);   // last readers of this Q / dO stage (dQ reads K, dS)
      }
      __syncwarp();
      if (g + 2 < n_half) {          // the buffer is free once the MMAs above have consumed it (the pipe is in order)
        constexpr int st2 = (st + 1) % NQ;                  // stage of tile i + 1
        if (hh == 0) {
          const uint32_t par = (uint32_t)(t + (st2 == 0 ? 1 : 0)) & 1u;   // (i + 1) / NQ
          mbar_wait(bar_qdo_full + 8 * st2, par);
          mbar_wait(bar_aug_full + 8 * st2, par);
        }
        tc_fence_after();
        MT_TRACE(200 + g);
        issue_st(std::integral_constant<int, 2 * st2 + hh>{});
      }
      if (WITH_DQ && hh == 1) {      // both halves of query tile i are done: dQ_i = dS_i K
        if (i > 0) mbar_wait(bar_dq_free, (i - 1) & 1);
        tc_fence_after();
        MT_TRACE(300 + g);
        if (elect_one()) {
          const uint64_t ds = (i & 1) ? ds_desc1 : ds_desc0;
#pragma unroll
          for (int k = 0; k < BT / 16; ++k)   // contraction over the 128 keys = rows of the dS^T tile and of K
            umma_ss(tm_dq, umma_desc_adv(ds, k * 2048), umma_desc_adv(k_mn_desc, k * 2048), IDESC_DQ, k > 0);
          umma_commit(bar_dq_full);
        }
        __syncwarp();
      }
    };
    auto trip = [&](int g0, int t, auto... Us) {
      ((g0 + decltype(Us)::value < n_half ? (half(g0 + decltype(Us)::value, t, Us), 0) : 0), ...);
    };
    static_assert(NQ == 3, "the issue loop is unrolled for three stages");
    for (int g = 0, t = 0; g < n_half; g += 2 * NQ, ++t)
      trip(g, t, std::integral_constant<int, 0>{}, std::integral_constant<int, 1>{}, std::integral_constant<int, 2>{},
           std::integral_constant<int, 3>{}, std::integral_constant<int, 4>{}, std::integral_constant<int, 5>{});
    if (elect_one()) umma_commit(bar_done);
    __syncwarp();
    if (lane == 0) { MT_TRACE_DUMP("mma3"); }
  } else if (warp < W_DRAIN) {
    // ===== compute: 16 warps, thread = (key row, 16 queries of the current 64-query half tile) =======================
    const int lane_grp = warp & 3;               // TMEM lanes of this warp
    const int qq = warp >> 2;                    // 16-query quarter of every half tile; also the dK / dV column group
    const int row = lane_grp * 32 + lane;        // key slot k0 + row
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    const int sw = row & 7;
    const bool key_ok = (k0 + row) < bg.m;       // rows past m belong to the next segment: mask column -> P = dS = 0
    const float scale_log2 = P.scale_log2, sc = P.scale;
    MT_TRACE_DECL
    MT_TRACE(1);

    // ---- K' and V' -> TMEM (A operands of S^T / dP^T for the whole CTA): quarter 0 copies K, quarter 1 copies V.
    // columns 48..50 = 1 (the three statistics columns), column 51 of K' = 1 for masked key rows, the rest 0
    mbar_wait(bar_kv_full, 0);
    MT_TRACE(2);
    if (qq < 2) {
      const uint8_t* src = smem + (qq == 0 ? Bwd3Smem::K : Bwd3Smem::V) + row * 128;
      uint32_t w[32];
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        const uint4 u = *reinterpret_cast<const uint4*>(src + ((c ^ sw) << 4));
        w[4 * c] = u.x; w[4 * c + 1] = u.y; w[4 * c + 2] = u.z; w[4 * c + 3] = u.w;
      }
      w[24] = 0x3f803f80u;
      w[25] = (qq == 0 && !key_ok) ? 0x3f803f80u : 0x00003f80u;
#pragma unroll
      for (int c = 26; c < 32; ++c) w[c] = 0u;
      const uint32_t dst = (qq == 0 ? tm_k : tm_v) + t_lane;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t r8[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) r8[e] = w[8 * c + e];
        tmem_st8(dst + c * 8, r8);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar_kvt_full);
    }

    const int n_half = 2 * n_q;
    MT_TRACE(3);
    for (int g = 0; g < n_half; ++g) {
      const int i = g >> 1, hh = g & 1;
      uint8_t* drow = smem + Bwd3Smem::DS + (i & 1) * 2 * TILE_BYTES + hh * TILE_BYTES + row * 128;
      const uint32_t ts = tmem + hh * 128 + t_lane + qq * 16, td = ts + 64;
      mbar_wait(bar_st_full + 8 * hh, i & 1);
      tc_fence_after();
      float sv[16], dp[16];
      tmem_ld16(ts, sv);
      tmem_ld16(td, dp);
      tmem_ld_wait();
      uint32_t pk[8], dk[8];
#pragma unroll
      for (int c = 0; c < 16; c += 2) {
        const float p0 = ex2(sv[c] * scale_log2);
        const float p1 = ex2(sv[c + 1] * scale_log2);
        pk[c >> 1] = pack_bf16(p0, p1);
        dk[c >> 1] = pack_bf16(p0 * dp[c], p1 * dp[c + 1]);
      }
      // packed results over the first 8 of the 16 columns this thread has just read (nobody else touches them)
      tmem_st8(ts, pk);
      tmem_st8(td, dk);
      // dS^T half tile for dQ = dS K: [key row][64 queries] block hh, 16 queries = 2 swizzled 16-byte chunks
      if constexpr (WITH_DQ) {
        *reinterpret_cast<uint4*>(drow + (((2 * qq) ^ sw) << 4)) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
        *reinterpret_cast<uint4*>(drow + (((2 * qq + 1) ^ sw) << 4)) = make_uint4(dk[4], dk[5], dk[6], dk[7]);
      }
      tmem_st_wait();
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bar_pt_full + 8 * hh);
    }
    MT_TRACE(4);
    mbar_wait(bar_done, 0);
    tc_fence_after();
    MT_TRACE(5);
    // ---- dK / dV of this key tile: TMEM -> fp32 staging (dK in dS^T buffer 0, dV in buffer 1) -> TMA reduce-adds.
    // Rows past the segment's m carry zeros (mask column); zero-key rows (position >= N) land in the scratch rows of dqkv.
    {
      float a[3][4], c2[3][4];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        tmem_ld4(tm_dk + t_lane + qq * 12 + c * 4, a[c]);
        tmem_ld4(tm_dv + t_lane + qq * 12 + c * 4, c2[c]);
      }
      tmem_ld_wait();
      uint8_t* stg_k = smem + Bwd3Smem::DS;
      uint8_t* stg_v = smem + Bwd3Smem::DS + 2 * TILE_BYTES;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        stage_chunk(stg_k, row, qq * 3 + c, make_float4(a[c][0] * sc, a[c][1] * sc, a[c][2] * sc, a[c][3] * sc));
        stage_chunk(stg_v, row, qq * 3 + c, make_float4(c2[c][0], c2[c][1], c2[c][2], c2[c][3]));
      }
      fence_proxy_async_smem();
      named_bar_sync(2, NCOMP);
      if (threadIdx.x == 0) {
        const uint32_t sk = sbase + Bwd3Smem::DS, sv_ = sbase + Bwd3Smem::DS + 2 * TILE_BYTES;
        tma_reduce_add_3d(&dq32_maps.m[b], sk, E + h * DH, off, jseg + k0);
        tma_reduce_add_3d(&dq16_maps.m[b], sk + Bwd3Smem::STG16, E + h * DH + 32, off, jseg + k0);
        tma_reduce_add_3d(&dq32_maps.m[b], sv_, 2 * E + h * DH, off, jseg + k0);
        tma_reduce_add_3d(&dq16_maps.m[b], sv_ + Bwd3Smem::STG16, 2 * E + h * DH + 32, off, jseg + k0);
        bulk_commit_group();
        bulk_wait_group_read<0>();          // the staging must outlive the reads; the adds complete with the kernel
      }
    }
    MT_TRACE(6);
    if (warp == 0 && lane == 0) { MT_TRACE_DUMP("cmp3"); }
  } else if constexpr (WITH_DQ) {
    // ===== dQ drain (4 warps, one query row per thread) ================================================================
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    const float sc = P.scale;
    const bool leader = threadIdx.x == W_DRAIN * 32;
    MT_TRACE_DECL
    for (int i = 0; i < n_q; ++i) {
      // dQ of query tile i: TMEM -> registers -> fp32 staging tile -> one TMA reduce-add per box
      MT_TRACE(2000 + i);
      mbar_wait(bar_dq_full, i & 1);
      tc_fence_after();
      MT_TRACE(2100 + i);
      float v[3][16];
#pragma unroll
      for (int c = 0; c < 3; ++c) tmem_ld16(tm_dq + t_lane + c * 16, v[c]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bar_dq_free);
      if (leader) bulk_wait_group_read<0>();   // the previous reduce-add has read the staging tile
      named_bar_sync(1, 128);
      uint8_t* stg = smem + Bwd3Smem::STG;
#pragma unroll
      for (int c = 0; c < 12; ++c)
        stage_chunk(stg, row, c, make_float4(v[c >> 2][(c & 3) * 4] * sc, v[c >> 2][(c & 3) * 4 + 1] * sc,
                                             v[c >> 2][(c & 3) * 4 + 2] * sc, v[c >> 2][(c & 3) * 4 + 3] * sc));
      fence_proxy_async_smem();
      named_bar_sync(1, 128);
      if (leader) {
        // rows past the segment's m (next segment / padding) carry dS = 0 -> they add zeros; rows >= n_alloc are clipped
        tma_reduce_add_3d(&dq32_maps.m[b], sbase + Bwd3Smem::STG, h * DH, off, jseg + i * BT);
        tma_reduce_add_3d(&dq16_maps.m[b], sbase + Bwd3Smem::STG + Bwd3Smem::STG16, h * DH + 32, off, jseg + i * BT);
        bulk_commit_group();
      }
      MT_TRACE(2200 + i);
    }
    if (leader) bulk_wait_group_read<0>();
    if (leader) { MT_TRACE_DUMP("drn3"); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, 512);
  MT_TL_END(n_q)
}

// =====================================================================================================================
// backward, persistent (impl 2): one CTA per SM stays resident and pulls key tiles from a device counter
// =====================================================================================================================
// Measured on B200 (tools/attn_timeline.py): a one-shot backward CTA lives 2 394 cycles per query tile + 9 300 cycles
// of prologue / epilogue, and the SM idles another 1 400 cycles until the next CTA starts -- with ONE CTA per SM (512
// TMEM columns, 221 KB of shared memory) nothing hides that: 25 % of the launch at 10k tokens, where a CTA streams only
// 8-23 query tiles.  Here the per-item pipeline is the one above, but consecutive items overlap:
//   * K / V of the NEXT item travel through the Q / dO ring as one more entry (K in the Q half, V in the dO half), so
//     they are in shared memory two tiles before the current item ends; the dedicated V buffer is gone (V is only ever
//     read once, for the TMEM copy), K is copied ring -> its fixed buffer once the current item's last dQ MMA is done.
//   * K' / V' of the next item go to TMEM as soon as the compute warps have finished the last half tile of the current
//     item (its S^T / dP^T MMAs have completed by then), while the MMA warp still issues the last dV / dK / dQ MMAs.
//   * dK leaves through the dS^T buffer the last tile used, dV through the dQ staging tile of the drain warps; the next
//     item's first dV / dK MMA only waits until both accumulators have been read into registers.
struct BwdPSmem {
  static constexpr int NQ = 3;
  static constexpr int K = 0;
  static constexpr int RING = K + TILE_BYTES;              // [NQ] x {Q tile, dO tile}
  static constexpr int DS = RING + NQ * 2 * TILE_BYTES;    // [2] dS^T tiles: [128 key rows][2 blocks of 64 queries]
  static constexpr int STG = DS + 4 * TILE_BYTES;          // fp32 staging tile of the dQ / dV reduce-adds (24 KB)
  static constexpr int BAR = STG + BT * DH * 4;
  // sched_full[2], sched_empty[2], ring_full[NQ], ring_empty[NQ], aug_full[NQ], kvt_full, st_full[2], pt_full[2],
  // dq_full, dq_free, done, acc_free
  static constexpr int NBAR = 4 + 3 * NQ + 9;
  static constexpr int QUEUE = (BAR + NBAR * 8 + 15) / 16 * 16;   // 2 x 16 ints: decoded items published by the scheduler
  static constexpr int TMEM_PTR = QUEUE + 128;
  static constexpr int TOTAL = TMEM_PTR + 16;
  static constexpr int STG16 = BT * 128;
};
static_assert(BwdPSmem::TOTAL <= 232448, "shared memory of the persistent backward kernel");

struct BwdItem {   // 12 ints: three 16-byte shared-memory accesses
  int n_q;         // query tiles of the item; <= 0: no more work
  int b, s, h, off, jseg, k0, seg_end, slot_h, pad0, pad1, pad2;
};

__device__ __forceinline__ bool bwd_decode(const Sm100Params& P, int idx, BwdItem& it) {
  int oi = 0;
  while (oi + 1 < P.geo.nb && idx >= P.item_prefix[oi + 1]) ++oi;
  it.b = P.order[oi];
  const BranchGeom& bg = P.geo.b[it.b];
  int local = idx - P.item_prefix[oi];
  const int kt = local % P.tiles[it.b];
  local /= P.tiles[it.b];
  it.h = local % P.geo.H;
  it.s = local / P.geo.H;
  it.off = (it.h * bg.r) / P.geo.H;
  it.jseg = (it.s * bg.g) / bg.r;
  it.k0 = kt * BT;
  it.seg_end = min(P.geo.N, (it.s + 1) * bg.g);
  it.slot_h = it.h - it.off * bg.hpb;
  const int seg_lo = it.s * bg.g + it.off;
  const int c_real = it.seg_end > seg_lo ? (it.seg_end - seg_lo + bg.r - 1) / bg.r : 0;
  it.n_q = min(P.tiles[it.b], (c_real + BT - 1) / BT);
  return it.k0 < c_real;
}

__global__ void __launch_bounds__(BWD3_THREADS, 1)
dilated_bwd_sm100_persistent_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ TensorMaps do_maps,
                                    const __grid_constant__ TensorMaps dq32_maps, const __grid_constant__ TensorMaps dq16_maps,
                                    const Sm100Params P, const float* __restrict__ lse, const float* __restrict__ delta_br,
                                    int* __restrict__ work_counter) {
  MT_TL_BEGIN
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_DRAIN = 16, W_TMA = 20, W_AUG = 21, W_MMA = 22;
  if ((sbase & 1023u) != 0) __trap();
  const int H = P.geo.H, E = H * DH;
  const int total = P.item_prefix[P.geo.nb];
  constexpr int NQ = BwdPSmem::NQ;
  constexpr int NCOMP = 512;

  const uint32_t bar_sched_full = sbase + BwdPSmem::BAR + 0;      // [2]
  const uint32_t bar_sched_empty = sbase + BwdPSmem::BAR + 16;    // [2]
  const uint32_t bar_ring_full = sbase + BwdPSmem::BAR + 32;      // [NQ] TMA landed
  const uint32_t bar_ring_empty = bar_ring_full + 8 * NQ;         // [NQ]
  const uint32_t bar_aug_full = bar_ring_empty + 8 * NQ;          // [NQ] statistics columns written into the entry
  const uint32_t bar_kvt_full = bar_aug_full + 8 * NQ;            // K' / V' of an item are in TMEM
  const uint32_t bar_st_full = bar_kvt_full + 8;                  // [2]
  const uint32_t bar_pt_full = bar_st_full + 16;                  // [2]
  const uint32_t bar_dq_full = bar_pt_full + 16;
  const uint32_t bar_dq_free = bar_dq_full + 8;
  const uint32_t bar_done = bar_dq_free + 8;                      // every MMA of an item has completed
  const uint32_t bar_acc_free = bar_done + 8;                     // dK / dV of an item have been read out of TMEM
  uint8_t* queue = smem + BwdPSmem::QUEUE;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + BwdPSmem::TMEM_PTR);

  if (warp == W_TMA && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_sched_full + 8 * i, 1);
      mbar_init(bar_sched_empty + 8 * i, 22);   // one arrival per consumer warp: 16 compute, 4 drain, statistics, MMA
      mbar_init(bar_st_full + 8 * i, 1);
      mbar_init(bar_pt_full + 8 * i, NCOMP);
    }
    for (int i = 0; i < NQ; ++i) {
      mbar_init(bar_ring_full + 8 * i, 1);
      mbar_init(bar_ring_empty + 8 * i, 1);
      mbar_init(bar_aug_full + 8 * i, 32);
    }
    mbar_init(bar_kvt_full, 256);
    mbar_init(bar_dq_full, 1);
    mbar_init(bar_dq_free, 128);
    mbar_init(bar_done, 1);
    mbar_init(bar_acc_free, NCOMP + 128);
    fence_barrier_init();
    for (int b = 0; b < P.geo.nb; ++b) {
      tma_prefetch_desc(&maps.m[b]);
      tma_prefetch_desc(&do_maps.m[b]);
      tma_prefetch_desc(&dq32_maps.m[b]);
      tma_prefetch_desc(&dq16_maps.m[b]);
    }
  }
  if (warp == W_MMA) {
    tmem_alloc(smem_u32((const void*)tmem_slot), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tm_dv = tmem + 256, tm_dk = tmem + 320, tm_dq = tmem + 384, tm_k = tmem + 448, tm_v = tmem + 480;
  int tl_tiles = 0;   // timeline only

  // item n of this CTA, decoded once by the scheduler thread (the integer divisions of the decode are hundreds of
  // cycles of cold code; the consumers sit on the hand-over critical path): every consumer warp copies the record out
  // of shared memory and releases the queue slot with one arrival.  false = no more work.
  auto read_item = [&](int n, BwdItem& it) -> bool {
    const int slot = n & 1;
    mbar_wait(bar_sched_full + 8 * slot, (n >> 1) & 1);
    const uint4* q = reinterpret_cast<const uint4*>(queue + slot * 64);
    const uint4 a = q[0], b2 = q[1], c = q[2];
    it.n_q = (int)a.x; it.b = (int)a.y; it.s = (int)a.z; it.h = (int)a.w;
    it.off = (int)b2.x; it.jseg = (int)b2.y; it.k0 = (int)b2.z; it.seg_end = (int)b2.w;
    it.slot_h = (int)c.x;
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_sched_empty + 8 * slot);
    return it.n_q > 0;
  };

  if (warp == W_TMA) {
    // ===== scheduler + TMA producer ====================================================================================
    if (lane == 0) {
      int e = 0;                                   // ring entries issued so far
      int next_idx = atomicAdd(work_counter, 1);
      MT_TRACE_DECL
      for (int n = 0;; ++n) {
        BwdItem it;
        int idx = next_idx;
        while (idx < total && !bwd_decode(P, idx, it)) idx = atomicAdd(work_counter, 1);
        const int qs = n & 1;
        mbar_wait(bar_sched_empty + 8 * qs, ((n >> 1) & 1) ^ 1);
        {
          uint4* q = reinterpret_cast<uint4*>(queue + qs * 64);
          q[0] = make_uint4((uint32_t)(idx < total ? it.n_q : 0), (uint32_t)it.b, (uint32_t)it.s, (uint32_t)it.h);
          q[1] = make_uint4((uint32_t)it.off, (uint32_t)it.jseg, (uint32_t)it.k0, (uint32_t)it.seg_end);
          q[2] = make_uint4((uint32_t)it.slot_h, 0u, 0u, 0u);
        }
        mbar_arrive(bar_sched_full + 8 * qs);
        MT_TRACEW(n, 5000);
        if (idx >= total) break;
        const void* map = &maps.m[it.b];
        const void* dmap = &do_maps.m[it.b];
        {  // K / V entry
          const int st = e % NQ;
          mbar_wait(bar_ring_empty + 8 * st, ((e / NQ) & 1) ^ 1);
          mbar_expect_tx(bar_ring_full + 8 * st, 2 * TILE_BYTES);
          const uint32_t dst = sbase + BwdPSmem::RING + st * 2 * TILE_BYTES;
          tma_load_3d(dst, map, bar_ring_full + 8 * st, E + it.h * DH, it.off, it.jseg + it.k0);
          tma_load_3d(dst + TILE_BYTES, map, bar_ring_full + 8 * st, 2 * E + it.h * DH, it.off, it.jseg + it.k0);
          MT_TRACEW(n, 5100);
          ++e;
        }
        for (int i = 0; i < it.n_q; ++i, ++e) {
          // the next item is claimed late -- three tiles before this one ends, enough to hide the atomic's latency --
          // so that near the end of the launch no CTA sits on a claimed item while others have run out of work
          if (i == max(0, it.n_q - 3)) next_idx = atomicAdd(work_counter, 1);
          const int st = e % NQ;
          mbar_wait(bar_ring_empty + 8 * st, ((e / NQ) & 1) ^ 1);
          mbar_expect_tx(bar_ring_full + 8 * st, 2 * TILE_BYTES);
          const uint32_t dst = sbase + BwdPSmem::RING + st * 2 * TILE_BYTES;
          tma_load_3d(dst, map, bar_ring_full + 8 * st, it.h * DH, it.off, it.jseg + i * BT);
          tma_load_3d(dst + TILE_BYTES, dmap, bar_ring_full + 8 * st, it.h * DH, it.off, it.jseg + i * BT);
          if (i < 3 || i >= it.n_q - 2) MT_TRACEW(n, 5200 + i);
        }
      }
      MT_TRACE_DUMP("tma");
    }
  } else if (warp == W_AUG) {
    // ===== statistics columns: lane owns rows lane + 32 j of every Q / dO tile ==========================================
    // The raw per-query statistics (strided 4-byte gathers of lse / delta: thousands of cycles when they miss L2) are
    // always loaded ONE RING ENTRY AHEAD, across item boundaries too: at the last tile of an item the warp already
    // fetches the first tile of the next item, whose record the scheduler has published by then.
    const float inv_sc = 1.f / P.scale;
    int e = 0;
    MT_TRACE_DECL
    auto load_raw = [&](const BwdItem& t, int i, float (&l)[4], float (&d)[4]) {
      const BranchGeom& tb = P.geo.b[t.b];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int slot = i * BT + lane + 32 * j;
        const int pos = t.s * tb.g + t.off + slot * tb.r;
        const bool qok = slot < tb.m && pos < t.seg_end;
        const int pc = qok ? pos : 0;
        l[j] = lse[(int64_t)pc * H + t.h];
        d[j] = delta_br[tb.lse_off + (int64_t)pc * tb.hpb + t.slot_h];
      }
    };
    BwdItem it;
    bool have = read_item(0, it);
    float lr[4], dr[4], ln[4], dn[4];
    if (have) load_raw(it, 0, lr, dr);
    for (int n = 0; have; ++n) {
      const BranchGeom& bg = P.geo.b[it.b];
      MT_TRACEW(n, 4000);
      // the K / V entry carries no statistics, but every use of a ring slot must advance the slot's aug_full phase
      mbar_arrive(bar_aug_full + 8 * (e % NQ));
      ++e;
      BwdItem nxt;
      bool have_next = false;
      for (int i = 0; i < it.n_q; ++i, ++e) {
        if (i + 1 < it.n_q) {
          load_raw(it, i + 1, ln, dn);
        } else {
          have_next = read_item(n + 1, nxt);
          if (have_next) load_raw(nxt, 0, ln, dn);
        }
        const int st = e % NQ;
        mbar_wait(bar_ring_full + 8 * st, (e / NQ) & 1);
        uint8_t* qt = smem + BwdPSmem::RING + st * 2 * TILE_BYTES;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int row = lane + 32 * j;
          const int slot = i * BT + row;
          const int pos = it.s * bg.g + it.off + slot * bg.r;
          const bool qok = slot < bg.m && pos < it.seg_end;
          uint32_t w0, w1;
          split3_bf16(qok ? -lr[j] * inv_sc : -32768.f, w0, w1, -32768.f);
          *reinterpret_cast<uint4*>(qt + row * 128 + ((6 ^ (row & 7)) << 4)) = make_uint4(w0, w1, 0u, 0u);
          split3_bf16(qok ? -dr[j] : 0.f, w0, w1, 0.f);
          *reinterpret_cast<uint4*>(qt + TILE_BYTES + row * 128 + ((6 ^ (row & 7)) << 4)) = make_uint4(w0, w1, 0u, 0u);
        }
        fence_proxy_async_smem();
        mbar_arrive(bar_aug_full + 8 * st);
        if (i < 3 || i >= it.n_q - 2) MT_TRACEW(n, 4100 + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) { lr[j] = ln[j]; dr[j] = dn[j]; }
      }
      it = nxt;
      have = have_next;
    }
    if (lane == 0) { MT_TRACE_DUMP("aug"); }
  } else if (warp == W_MMA) {
    // ===== MMA issuer =================================================================================================
    constexpr uint32_t IDESC_ST = umma_idesc_bf16(BT, 64, 0, 0);    // A = K' / V' (TMEM), B = Q' / dO' half tile (K-major)
    constexpr uint32_t IDESC_TS = umma_idesc_bf16(BT, DH, 0, 1);    // A = P^T / dS^T (TMEM), B = dO / Q (MN-major)
    constexpr uint32_t IDESC_DQ = umma_idesc_bf16(BT, DH, 1, 1);    // A = dS^T tile (smem, MN-major), B = K (MN-major)
    const uint64_t ring_k_desc = umma_smem_desc(sbase + BwdPSmem::RING, 16, 1024);          // K-major view of entry 0
    const uint64_t ring_m_desc = umma_smem_desc(sbase + BwdPSmem::RING, TILE_BYTES, 1024);  // MN-major view of entry 0
    const uint64_t k_mn_desc = umma_smem_desc(sbase + BwdPSmem::K, TILE_BYTES, 1024);
    const uint64_t ds_desc0 = umma_smem_desc(sbase + BwdPSmem::DS, TILE_BYTES, 1024);
    // S'^T and dP'^T of one half tile (ring slot ST, half HH: compile-time, every descriptor is a base plus a constant --
    // the single issuing thread shares its scheduler with five busy warps and its instructions are critical-path
    // latency) into TMEM buffer HH
    auto issue_st = [&](auto ST, auto HH) {
      constexpr int st = decltype(ST)::value, hh = decltype(HH)::value;
      if (elect_one()) {
        constexpr uint32_t so = (uint32_t)(st * 2 * TILE_BYTES + hh * 64 * 128);
        const uint32_t ts = tmem + hh * 128, td = ts + 64;
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_ts(ts, tm_k + k * 8, umma_desc_adv(ring_k_desc, so + k * 32), IDESC_ST, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_ts(td, tm_v + k * 8, umma_desc_adv(ring_k_desc, so + TILE_BYTES + k * 32), IDESC_ST, k > 0);
        umma_commit(bar_st_full + 8 * hh);
      }
      __syncwarp();
    };
    // dQ of global query tile tg = dS[tg & 1] K: nothing here depends on the ring slot
    auto issue_dq = [&](int tg) {
      if (tg > 0) mbar_wait(bar_dq_free, (tg - 1) & 1);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t ds = umma_desc_adv(ds_desc0, (uint32_t)(tg & 1) * 2 * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < BT / 16; ++k)
          umma_ss(tm_dq, umma_desc_adv(ds, k * 2048), umma_desc_adv(k_mn_desc, k * 2048), IDESC_DQ, k > 0);
        umma_commit(bar_dq_full);
      }
      __syncwarp();
    };
    int e = 0, ti = 0;   // ring entries / query tiles consumed so far (all items)
    int n = 0, n_half = 0;
    BwdItem it, nxt;
    bool have_next = false;
    MT_TRACE_DECL
    // S'^T / dP'^T of BOTH halves of the first query tile of item n_item, whose first Q / dO entry is ring entry `ent`:
    // issued by the previous item's tail (ahead of its last dQ MMA), so that the compute warps find the first score
    // tile of the next item ready right after the last one of this item
    auto issue_first = [&](int n_item, int ent) {
      const int st = ent % NQ;
      const uint32_t par = (uint32_t)(ent / NQ) & 1u;
      mbar_wait(bar_kvt_full, n_item & 1);       // K' and V' of that item are in TMEM
      mbar_wait(bar_ring_full + 8 * st, par);
      mbar_wait(bar_aug_full + 8 * st, par);
      tc_fence_after();
      if (st == 0) {
        issue_st(std::integral_constant<int, 0>{}, std::integral_constant<int, 0>{});
        issue_st(std::integral_constant<int, 0>{}, std::integral_constant<int, 1>{});
      } else if (st == 1) {
        issue_st(std::integral_constant<int, 1>{}, std::integral_constant<int, 0>{});
        issue_st(std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{});
      } else {
        issue_st(std::integral_constant<int, 2>{}, std::integral_constant<int, 0>{});
        issue_st(std::integral_constant<int, 2>{}, std::integral_constant<int, 1>{});
      }
    };
    // One item whose first Q / dO entry sits in ring slot S0 (compile time: the three instantiations differ only in
    // constants).  e = entry index of that first Q / dO entry.
    auto run_item = [&](auto S0) {
      constexpr int s0 = decltype(S0)::value;
      const int ediv = e / NQ;              // ring use count of entry e (e % NQ == s0)
      MT_TRACEW(n, 2000);
      // half tile g = 6 * trip + U of the item: tile i = 3 * trip + U / 2 in ring slot (s0 + U / 2) % NQ
      auto half = [&](int g, int trip, auto U) {
        constexpr int u = decltype(U)::value;
        constexpr int u2 = u >> 1, hh = u & 1;
        constexpr int st = (s0 + u2) % NQ;
        const int tg = ti + (g >> 1);                              // global tile index
        mbar_wait(bar_pt_full + 8 * hh, tg & 1);                   // P^T, dS^T of this half are in TMEM (+ dS^T in smem)
        if (g < 4 || g >= n_half - 4) MT_TRACEW(n, 2100 + g);
        if (g == 0 && n > 0) mbar_wait(bar_acc_free, (n - 1) & 1);   // the previous item's dK / dV have been read out
        if (g == 0) MT_TRACEW(n, 2003);
        tc_fence_after();
        if (elect_one()) {
          constexpr uint32_t so = (uint32_t)(st * 2 * TILE_BYTES + hh * 64 * 128);
          const uint32_t ts = tmem + hh * 128, td = ts + 64;
          umma_ts(tm_dv, ts, umma_desc_adv(ring_m_desc, so + TILE_BYTES), IDESC_TS, g > 0);
#pragma unroll
          for (int k = 1; k < 4; ++k)
            umma_ts(tm_dv, ts + k * 16, umma_desc_adv(ring_m_desc, so + TILE_BYTES + k * 2048), IDESC_TS, 1);
          umma_ts(tm_dk, td, umma_desc_adv(ring_m_desc, so), IDESC_TS, g > 0);
#pragma unroll
          for (int k = 1; k < 4; ++k) umma_ts(tm_dk, td + k * 16, umma_desc_adv(ring_m_desc, so + k * 2048), IDESC_TS, 1);
          if (hh == 1) umma_commit(bar_ring_empty + 8 * st);      // last readers of this Q / dO entry
        }
        __syncwarp();
        if (g + 2 < n_half) {          // the S^T / dP^T buffer is free once the MMAs above have consumed it (in order)
          constexpr int st2 = (st + 1) % NQ;
          if (hh == 0) {
            // ring use count of entry e + 3 trip + u2 + 1
            constexpr int carry = (s0 + u2 + 1) / NQ;
            const uint32_t par = (uint32_t)(ediv + trip + carry) & 1u;
            mbar_wait(bar_ring_full + 8 * st2, par);
            mbar_wait(bar_aug_full + 8 * st2, par);
            if (g < 4 || g >= n_half - 4) MT_TRACEW(n, 2200 + g);
          }
          tc_fence_after();
          issue_st(std::integral_constant<int, st2>{}, std::integral_constant<int, hh>{});
        }
        // both halves of this query tile are done: dQ = dS K (the last tile's dQ is issued by the caller, behind the
        // score MMAs of the next item's first tile)
        if (hh == 1 && g != n_half - 1) issue_dq(tg);
      };
      auto trip6 = [&](int g0, int trip, auto... Us) {
        ((g0 + decltype(Us)::value < n_half ? (half(g0 + decltype(Us)::value, trip, Us), 0) : 0), ...);
      };
      for (int g0 = 0, trip = 0; g0 < n_half; g0 += 2 * NQ, ++trip)
        trip6(g0, trip, std::integral_constant<int, 0>{}, std::integral_constant<int, 1>{},
              std::integral_constant<int, 2>{}, std::integral_constant<int, 3>{}, std::integral_constant<int, 4>{},
              std::integral_constant<int, 5>{});
    };
    static_assert(NQ == 3, "the issue loop is unrolled for three ring slots");
    bool have = read_item(0, it);
    if (have) issue_first(0, 1);             // entry 0 = K / V of the first item, entry 1 = its first Q / dO tile
    for (n = 0; have; ++n) {
      n_half = 2 * it.n_q;
      have_next = false;
      ++e;                                  // the K / V entry (consumed by the compute warps)
      switch (e % NQ) {
        case 0: run_item(std::integral_constant<int, 0>{}); break;
        case 1: run_item(std::integral_constant<int, 1>{}); break;
        default: run_item(std::integral_constant<int, 2>{}); break;
      }
      // tail of the item: its last dQ, then the score MMAs of the next item's first tile.  (Measured the other way round
      // -- next item's score MMAs ahead of the last dQ, dK epilogue deferred into the next item's first tile: the
      // hand-over bubble drops from 2 700 to 1 150 cycles, but the first tile of every item grows by 2 800 and the
      // launch gets 3 % slower: whatever runs once per item is slow wherever it sits.)
      issue_dq(ti + it.n_q - 1);
      if (elect_one()) umma_commit(bar_done);
      __syncwarp();
      MT_TRACEW(n, 2900);
      have_next = read_item(n + 1, nxt);
      if (have_next) issue_first(n + 1, e + it.n_q + 1);
      MT_TRACEW(n, 2002);
      e += it.n_q;
      ti += it.n_q;
      it = nxt;
      have = have_next;
    }
    tl_tiles = ti;
    if (lane == 0) { MT_TRACE_DUMP("mma"); }
  } else if (warp < W_DRAIN) {
    // ===== compute: 16 warps, thread = (key row, 16 queries of the current 64-query half tile) =======================
    const int lane_grp = warp & 3;
    const int qq = warp >> 2;
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    const int sw = row & 7;
    const float scale_log2 = P.scale_log2, sc = P.scale;
    const int ctid = threadIdx.x;   // 0..511
    MT_TRACE_DECL
    int trn_item = 0;                // trace builds only: the item the hand-over helpers belong to

    // K' / V' of an item -> TMEM from its ring entry (quarter 0 copies K, quarter 1 copies V); columns 48..50 = 1 (the
    // statistics columns), column 51 of K' = 1 for key rows past the segment's m, the rest 0
    auto kv_to_tmem = [&](int ent, bool key_ok) {
      mbar_wait(bar_ring_full + 8 * (ent % NQ), (ent / NQ) & 1);
      if (qq < 2) {
        const uint8_t* src = smem + BwdPSmem::RING + (ent % NQ) * 2 * TILE_BYTES + (qq == 0 ? 0 : TILE_BYTES) + row * 128;
        uint32_t w[32];
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const uint4 u = *reinterpret_cast<const uint4*>(src + ((c ^ sw) << 4));
          w[4 * c] = u.x; w[4 * c + 1] = u.y; w[4 * c + 2] = u.z; w[4 * c + 3] = u.w;
        }
        w[24] = 0x3f803f80u;
        w[25] = (qq == 0 && !key_ok) ? 0x3f803f80u : 0x00003f80u;
#pragma unroll
        for (int c = 26; c < 32; ++c) w[c] = 0u;
        const uint32_t dst = (qq == 0 ? tm_k : tm_v) + t_lane;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t r8[8];
#pragma unroll
          for (int e2 = 0; e2 < 8; ++e2) r8[e2] = w[8 * c + e2];
          tmem_st8(dst + c * 8, r8);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bar_kvt_full);
      }
    };
    // K of an item: ring entry -> its fixed buffer (B operand of every dQ MMA of the item), then the entry is released.
    // Only legal once the previous item's last dQ MMA has completed (bar_done).
    auto k_to_buffer = [&](int ent) {
      const uint8_t* src = smem + BwdPSmem::RING + (ent % NQ) * 2 * TILE_BYTES;
      uint8_t* dst = smem + BwdPSmem::K;
      const uint4 a = *reinterpret_cast<const uint4*>(src + ctid * 32);
      const uint4 b2 = *reinterpret_cast<const uint4*>(src + ctid * 32 + 16);
      *reinterpret_cast<uint4*>(dst + ctid * 32) = a;
      *reinterpret_cast<uint4*>(dst + ctid * 32 + 16) = b2;
      MT_TRACEW(trn_item, 1210);
      fence_proxy_async_smem();
      MT_TRACEW(trn_item, 1211);
      named_bar_sync(2, NCOMP);
      MT_TRACEW(trn_item, 1212);
      if (ctid == 0) mbar_arrive(bar_ring_empty + 8 * (ent % NQ));
    };

    int e = 0, ti = 0;
    int pending_buf = -1;            // dS^T buffer that still feeds an in-flight dK reduce-add
    // dK of a finished item: wait until all of its MMAs are done, TMEM -> registers (the accumulator is then free for
    // the next item), fp32 staging in the dS^T buffer its last tile used, one TMA reduce-add per box.
    struct Pending { int n, b, col, off, j, ti_last; };
    auto finish_item = [&](const Pending& pd, int kv_entry_next) {
      MT_TRACEW(pd.n, 1201);
      mbar_wait(bar_done, pd.n & 1);       // every MMA of that item has completed
      MT_TRACEW(pd.n, 1202);
      tc_fence_after();
      float a[3][4];
#pragma unroll
      for (int c = 0; c < 3; ++c) tmem_ld4(tm_dk + t_lane + qq * 12 + c * 4, a[c]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bar_acc_free);
      MT_TRACEW(pd.n, 1203);
      if (kv_entry_next >= 0) k_to_buffer(kv_entry_next);   // the K buffer is free: that item's last dQ MMA is done
      MT_TRACEW(pd.n, 1204);
      uint8_t* stg_k = smem + BwdPSmem::DS + (pd.ti_last & 1) * 2 * TILE_BYTES;
#pragma unroll
      for (int c = 0; c < 3; ++c)
        stage_chunk(stg_k, row, qq * 3 + c, make_float4(a[c][0] * sc, a[c][1] * sc, a[c][2] * sc, a[c][3] * sc));
      fence_proxy_async_smem();
      if (ctid == 0) bulk_wait_group_read<0>();   // at most one dK reduce-add in flight (the previous one is long done)
      named_bar_sync(2, NCOMP);
      if (ctid == 0) {
        const uint32_t sk = sbase + BwdPSmem::DS + (pd.ti_last & 1) * 2 * TILE_BYTES;
#ifndef MT_EXP_SKIP_DKV   // experiment builds only (wrong results): the launch without the dK / dV reduce-adds
        tma_reduce_add_3d(&dq32_maps.m[pd.b], sk, pd.col, pd.off, pd.j);
        tma_reduce_add_3d(&dq16_maps.m[pd.b], sk + BwdPSmem::STG16, pd.col + 32, pd.off, pd.j);
#endif
        bulk_commit_group();
      }
      pending_buf = pd.ti_last & 1;
      MT_TRACEW(pd.n, 1205);
    };

    BwdItem it;
    bool have = read_item(0, it);
    if (have) {
      kv_to_tmem(e, (it.k0 + row) < P.geo.b[it.b].m);
      k_to_buffer(e);
    }
    Pending pd;
#ifdef MT_DEBUG_TIMELINE
    long long tl_first = 0;
#endif
    for (int n = 0; have; ++n) {
      trn_item = n;
      ++e;   // past the K / V entry of this item
      const int n_half = 2 * it.n_q;
      auto half_tile = [&](int g) {
        const int i = g >> 1, hh = g & 1;
        const int tg = ti + i;
        if (hh == 0 && pending_buf == (tg & 1)) {   // this tile's dS^T buffer still feeds the last dK reduce-add
          if (ctid == 0) bulk_wait_group_read<0>();
          named_bar_sync(2, NCOMP);
          pending_buf = -1;
        }
        uint8_t* drow = smem + BwdPSmem::DS + (tg & 1) * 2 * TILE_BYTES + hh * TILE_BYTES + row * 128;
        const uint32_t ts = tmem + hh * 128 + t_lane + qq * 16, td = ts + 64;
        mbar_wait(bar_st_full + 8 * hh, tg & 1);
#ifdef MT_DEBUG_TIMELINE
        if (g == 0) tl_first = clock64();
#endif
        if (g < 4 || g >= n_half - 4) MT_TRACEW(n, 1000 + g);
        tc_fence_after();
        float sv[16], dp[16];
        tmem_ld16(ts, sv);
        tmem_ld16(td, dp);
        tmem_ld_wait();
        uint32_t pk[8], dk[8];
#pragma unroll
        for (int c = 0; c < 16; c += 2) {
          const float p0 = ex2(sv[c] * scale_log2);
          const float p1 = ex2(sv[c + 1] * scale_log2);
          pk[c >> 1] = pack_bf16(p0, p1);
          dk[c >> 1] = pack_bf16(p0 * dp[c], p1 * dp[c + 1]);
        }
        tmem_st8(ts, pk);
        tmem_st8(td, dk);
        *reinterpret_cast<uint4*>(drow + (((2 * qq) ^ sw) << 4)) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
        *reinterpret_cast<uint4*>(drow + (((2 * qq + 1) ^ sw) << 4)) = make_uint4(dk[4], dk[5], dk[6], dk[7]);
        tmem_st_wait();
        fence_proxy_async_smem();
        tc_fence_before();
        mbar_arrive(bar_pt_full + 8 * hh);
        if (g < 4 || g >= n_half - 4) MT_TRACEW(n, 1100 + g);
      };
#pragma unroll 1
      for (int g = 0; g < n_half; ++g) half_tile(g);
#ifdef MT_DEBUG_TIMELINE
      if (ctid == 0) MT_TL_ITEM(it.n_q, tl_first, clock64());
#endif
      pd.n = n; pd.b = it.b; pd.col = E + it.h * DH; pd.off = it.off; pd.j = it.jseg + it.k0;
      pd.ti_last = ti + it.n_q - 1;
      ti += it.n_q;
      e += it.n_q;
      // ---- hand-over: the next item's K' / V' go to TMEM while the MMA warp finishes this item ----------------------
      have = read_item(n + 1, it);
      MT_TRACEW(n, 1200);
      // S^T / dP^T of this item's last half have completed (st_full): K' / V' in TMEM are free for the next item
      if (have) kv_to_tmem(e, (it.k0 + row) < P.geo.b[it.b].m);
      finish_item(pd, have ? e : -1);   // this item's dK; the next item's K into the buffer its dQ MMAs read
    }
    if (ctid == 0) bulk_wait_group_read<0>();
    if (ctid == 0) { MT_TRACE_DUMP("cmp"); }
  } else {
    // ===== drain (4 warps, one row per thread): dQ of every query tile, dV of every item ===============================
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    const float sc = P.scale;
    const bool leader = threadIdx.x == W_DRAIN * 32;
    MT_TRACE_DECL
    int trn_item = -1;
    uint8_t* stg = smem + BwdPSmem::STG;
    int ti = 0;
    // one [128][48] fp32 tile: TMEM -> registers -> staging -> one TMA reduce-add per box at column c0 of dqkv
    auto drain_tile = [&](uint32_t tm_src, float mul, int b, int c0, int off, int j0, uint32_t free_bar) {
      float v[3][16];
#pragma unroll
      for (int c = 0; c < 3; ++c) tmem_ld16(tm_src + t_lane + c * 16, v[c]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(free_bar);
      MT_TRACEW(trn_item, 3400);
      if (leader) bulk_wait_group_read<0>();   // the previous reduce-add has read the staging tile
      MT_TRACEW(trn_item, 3401);
      named_bar_sync(1, 128);
#pragma unroll
      for (int c = 0; c < 12; ++c)
        stage_chunk(stg, row, c, make_float4(v[c >> 2][(c & 3) * 4] * mul, v[c >> 2][(c & 3) * 4 + 1] * mul,
                                             v[c >> 2][(c & 3) * 4 + 2] * mul, v[c >> 2][(c & 3) * 4 + 3] * mul));
      fence_proxy_async_smem();
      named_bar_sync(1, 128);
      if (leader) {
#ifdef MT_EXP_SKIP_DKV
        if (mul != 1.f)
#endif
#ifndef MT_EXP_SKIP_DQ    // experiment builds only (wrong results): the launch without any reduce-add of the drain warps
        {
          tma_reduce_add_3d(&dq32_maps.m[b], sbase + BwdPSmem::STG, c0, off, j0);
          tma_reduce_add_3d(&dq16_maps.m[b], sbase + BwdPSmem::STG + BwdPSmem::STG16, c0 + 32, off, j0);
        }
#endif
        bulk_commit_group();
      }
    };
    for (int n = 0;; ++n) {
      BwdItem it;
      if (!read_item(n, it)) break;
      for (int i = 0; i < it.n_q; ++i, ++ti) {
        trn_item = (i >= it.n_q - 2) ? n : -1;
        mbar_wait(bar_dq_full, ti & 1);
        if (i < 2 || i >= it.n_q - 2) MT_TRACEW(n, 3000 + i);
        tc_fence_after();
        drain_tile(tm_dq, sc, it.b, it.h * DH, it.off, it.jseg + i * BT, bar_dq_free);
        if (i < 2 || i >= it.n_q - 2) MT_TRACEW(n, 3100 + i);
      }
      mbar_wait(bar_done, n & 1);
      MT_TRACEW(n, 3200);
      tc_fence_after();
      drain_tile(tm_dv, 1.f, it.b, 2 * E + it.h * DH, it.off, it.jseg + it.k0, bar_acc_free);
      MT_TRACEW(n, 3300);
    }
    if (leader) bulk_wait_group_read<0>();
    if (leader) { MT_TRACE_DUMP("drn"); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, 512);
  if (threadIdx.x == 0) {
    if (atomicAdd(work_counter + 1, 1) == (int)gridDim.x - 1) {
      work_counter[1] = 0;
      __threadfence();
      work_counter[0] = 0;
    }
  }
#ifdef MT_DEBUG_TIMELINE
  if (threadIdx.x == W_MMA * 32) {
    unsigned sm_;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_));
    long long* e_ = mt_timeline + 4 * blockIdx.x;
    e_[0] = sm_; e_[1] = tl_tiles; e_[2] = tl_t0_; e_[3] = clock64();
  }
#endif
}

// =====================================================================================================================
// backward, deterministic (impl 4): dQ query tile by query tile
// =====================================================================================================================
// One CTA = one (branch, segment, head, 128-slot query tile) -- the pipeline of dilated_fwd_sm100_k48_kernel with the dO
// tile and a second score MMA.  Per 48-key tile of the segment:
//   S = Q K^T and dP = dO V^T into TMEM (SS MMAs, N = 48);
//   P = exp2(S scale log2e - lse log2e) with the FINAL merged lse: no running maximum and no rescale;
//   dS = P (dP - delta_b), packed to bf16 pairs in TMEM;
//   dQ += dS K: a TS MMA with K as the MN-major B operand, the way the forward uses P and V.
// A query row is a TMEM lane, so lse and delta are one scalar per thread.  dQ * scale leaves once per tile: the thread of
// a row adds it to that row of dqkv, a plain load-add-store, because no other CTA of the launch touches the element.
// Rows of the tile that are not its queries (slots >= m belong to the next segment, positions >= N are padding) are
// not written at all: their S against this segment's keys is not zero, so they are given P = 0 and skipped.
// TMEM: S [0,48) | dP [48,96) | dS (bf16 pairs) [96,120) | dQ [128,176) -> a 256-column allocation (two CTAs per SM).
// Shared memory: Q + dO tiles (32 KB) and a four-stage ring of 48-key K / V tiles (48 KB): 80 KB, so at most two CTAs
// share an SM, the number the TMEM allocation allows.
static constexpr int DQ_KS = 4;                   // K / V ring stages
static constexpr uint32_t TMEM_DQ_COLS = 256;
struct BwdDqSmem {
  static constexpr int Q = 0;
  static constexpr int DO = Q + TILE_BYTES;
  static constexpr int K = DO + TILE_BYTES;
  static constexpr int V = K + DQ_KS * KT_BYTES;
  static constexpr int BAR = V + DQ_KS * KT_BYTES;
  // barriers (8 B each): qdo_full, s_full, s_free, p_full, dq_full, kv_full[DQ_KS], kv_empty[DQ_KS]; the TMEM pointer
  static constexpr int NBAR = 5 + 2 * DQ_KS;
  static constexpr int TMEM_PTR = BAR + NBAR * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
};
static_assert(KT == 48, "the dQ kernel's TMEM layout is laid out for 48-key tiles");

__global__ void __launch_bounds__(FWD_THREADS, 2)
dilated_bwd_dq_sm100_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ TensorMaps kv_maps,
                            const __grid_constant__ TensorMaps do_maps, const Sm100Params P,
                            const float* __restrict__ lse, const float* __restrict__ delta_br, float* __restrict__ dqkv) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_TMA = 4, W_MMA = 5;
  if ((sbase & 1023u) != 0) {
    __trap();
  }
  int oi = 0;
  while (oi + 1 < P.geo.nb && (int)blockIdx.x >= P.item_prefix[oi + 1]) ++oi;
  const int b = P.order[oi];
  const BranchGeom bg = P.geo.b[b];
  int local = blockIdx.x - P.item_prefix[oi];
  const int qt = local % P.tiles[b];
  local /= P.tiles[b];
  const int h = local % P.geo.H;
  const int s = local / P.geo.H;
  const int H = P.geo.H, N = P.geo.N, E = H * DH;
  const int off = (h * bg.r) / H;
  const int jseg = (s * bg.g) / bg.r;
  const int q0 = qt * BT;
  const int seg_lo = s * bg.g + off;
  const int seg_end = min(N, (s + 1) * bg.g);
  const int c_real = seg_end > seg_lo ? (seg_end - seg_lo + bg.r - 1) / bg.r : 0;
  if (q0 >= c_real) return;                                   // a tile of padding queries only
  const int n_kv = min((bg.m + KT - 1) / KT, (c_real + KT - 1) / KT);   // key tiles of padding only have K = 0

  const uint32_t bar_qdo_full = sbase + BwdDqSmem::BAR + 0;
  const uint32_t bar_s_full = sbase + BwdDqSmem::BAR + 8;
  const uint32_t bar_s_free = sbase + BwdDqSmem::BAR + 16;
  const uint32_t bar_p_full = sbase + BwdDqSmem::BAR + 24;
  const uint32_t bar_dq_full = sbase + BwdDqSmem::BAR + 32;
  const uint32_t bar_kv_full = sbase + BwdDqSmem::BAR + 40;   // [DQ_KS]
  const uint32_t bar_kv_empty = bar_kv_full + 8 * DQ_KS;      // [DQ_KS]
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + BwdDqSmem::TMEM_PTR);

  if (threadIdx.x == 0) {
    mbar_init(bar_qdo_full, 1);
    for (int i = 0; i < DQ_KS; ++i) {
      mbar_init(bar_kv_full + 8 * i, 1);
      mbar_init(bar_kv_empty + 8 * i, 1);
    }
    mbar_init(bar_s_full, 1);
    mbar_init(bar_s_free, 128);
    mbar_init(bar_p_full, 128);
    mbar_init(bar_dq_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&maps.m[b]);
    tma_prefetch_desc(&kv_maps.m[b]);
    tma_prefetch_desc(&do_maps.m[b]);
  }
  if (warp == W_MMA) {
    tmem_alloc(smem_u32((const void*)tmem_slot), TMEM_DQ_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_s = tmem, tmem_dp = tmem + KT, tmem_ds = tmem + 2 * KT, tmem_dq = tmem + 128;

  if (warp == W_TMA) {
    // ===== TMA producer ===============================================================================================
    if (lane == 0) {
      const void* kmap = &kv_maps.m[b];    // the qkv view with a 48-slot box
      mbar_expect_tx(bar_qdo_full, 2 * TILE_BYTES);
      tma_load_3d(sbase + BwdDqSmem::Q, &maps.m[b], bar_qdo_full, h * DH, off, jseg + q0);
      tma_load_3d(sbase + BwdDqSmem::DO, &do_maps.m[b], bar_qdo_full, h * DH, off, jseg + q0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j % DQ_KS, use = j / DQ_KS;
        mbar_wait(bar_kv_empty + 8 * st, (use & 1) ^ 1);
        mbar_expect_tx(bar_kv_full + 8 * st, 2 * KT_BYTES);
        tma_load_3d(sbase + BwdDqSmem::K + st * KT_BYTES, kmap, bar_kv_full + 8 * st, E + h * DH, off, jseg + j * KT);
        tma_load_3d(sbase + BwdDqSmem::V + st * KT_BYTES, kmap, bar_kv_full + 8 * st, 2 * E + h * DH, off, jseg + j * KT);
      }
    }
  } else if (warp == W_MMA) {
    // ===== MMA issuer =================================================================================================
    constexpr uint32_t IDESC_S = umma_idesc_bf16(BT, KT, 0, 0);    // S, dP: A = Q / dO, B = K / V (both K-major)
    constexpr uint32_t IDESC_DQ = umma_idesc_bf16(BT, DH, 0, 1);   // dQ: A = dS (TMEM), B = K (MN-major)
    const uint64_t q_desc = umma_smem_desc(sbase + BwdDqSmem::Q, 16, 1024);
    const uint64_t do_desc = umma_smem_desc(sbase + BwdDqSmem::DO, 16, 1024);
    const uint64_t k_desc0 = umma_smem_desc(sbase + BwdDqSmem::K, 16, 1024);
    const uint64_t v_desc0 = umma_smem_desc(sbase + BwdDqSmem::V, 16, 1024);
    const uint64_t kmn_desc0 = umma_smem_desc(sbase + BwdDqSmem::K, KT_BYTES, 1024);
    auto issue_s = [&](int j) {   // S_j = Q K_j^T and dP_j = dO V_j^T: three k-steps of 16 each
      if (elect_one()) {
        const uint32_t so = (uint32_t)(j % DQ_KS) * KT_BYTES;
        const uint64_t kd = umma_desc_adv(k_desc0, so), vd = umma_desc_adv(v_desc0, so);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          umma_ss(tmem_s, umma_desc_adv(q_desc, k * 32), umma_desc_adv(kd, k * 32), IDESC_S, k > 0);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          umma_ss(tmem_dp, umma_desc_adv(do_desc, k * 32), umma_desc_adv(vd, k * 32), IDESC_S, k > 0);
        umma_commit(bar_s_full);
      }
      __syncwarp();
    };
    mbar_wait(bar_qdo_full, 0);
    mbar_wait(bar_kv_full, 0);
    tc_fence_after();
    issue_s(0);
    for (int j = 0; j < n_kv; ++j) {
      if (j + 1 < n_kv) {
        mbar_wait(bar_kv_full + 8 * ((j + 1) % DQ_KS), ((j + 1) / DQ_KS) & 1);
        mbar_wait(bar_s_free, j & 1);   // S_j and dP_j are in registers
        tc_fence_after();
        issue_s(j + 1);
      }
      mbar_wait(bar_p_full, j & 1);     // dS_j is in TMEM
      tc_fence_after();
      if (elect_one()) {
        const uint64_t kd = umma_desc_adv(kmn_desc0, (uint32_t)(j % DQ_KS) * KT_BYTES);
#pragma unroll
        for (int k = 0; k < KT / 16; ++k)   // 16 keys = 8 packed dS columns = 16 rows of the K tile (2048 B)
          umma_ts(tmem_dq, tmem_ds + k * 8, umma_desc_adv(kd, k * 2048), IDESC_DQ, (j > 0) || (k > 0));
        umma_commit(bar_kv_empty + 8 * (j % DQ_KS));
        umma_commit(bar_dq_full);
      }
      __syncwarp();
    }
  } else {
    // ===== dS: one query row per thread =================================================================================
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    const int slot = q0 + row;
    const int pos = seg_lo + slot * bg.r;
    const bool qok = slot < bg.m && pos < seg_end;     // this tile's own query
    const int slot_h = h - off * bg.hpb;
    const float lb = qok ? lse[(int64_t)pos * H + h] * 1.4426950408889634f : INFINITY;   // +inf: P = 0
    const float dl = qok ? delta_br[bg.lse_off + (int64_t)pos * bg.hpb + slot_h] : 0.f;
    const float scale_log2 = P.scale_log2;
    auto tile = [&](int j, auto mask_tag) {
      constexpr bool MASK = decltype(mask_tag)::value;
      const int kvalid = bg.m - j * KT;  // key slots of this tile that belong to the segment
      mbar_wait(bar_s_full, j & 1);
      tc_fence_after();
      float sv[KT], dp[KT];
      {
        float lo[32], hi[16], dlo[32], dhi[16];
        tmem_ld32(tmem_s + t_lane, lo);
        tmem_ld16(tmem_s + t_lane + 32, hi);
        tmem_ld32(tmem_dp + t_lane, dlo);
        tmem_ld16(tmem_dp + t_lane + 32, dhi);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) { sv[i] = lo[i]; dp[i] = dlo[i]; }
#pragma unroll
        for (int i = 0; i < 16; ++i) { sv[32 + i] = hi[i]; dp[32 + i] = dhi[i]; }
      }
      tc_fence_before();
      mbar_arrive(bar_s_free);           // the MMA warp may overwrite S / dP with tile j + 1
      if (j > 0) {                       // dS_j overwrites dS_{j-1}: its dQ MMA must have read it
        mbar_wait(bar_dq_full, (j - 1) & 1);
        tc_fence_after();
      }
#pragma unroll
      for (int c = 0; c < KT / 16; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          const int k = c * 16 + i;
          float p0 = ex2(fmaf(sv[k], scale_log2, -lb));
          float p1 = ex2(fmaf(sv[k + 1], scale_log2, -lb));
          if (MASK) {
            p0 = k < kvalid ? p0 : 0.f;
            p1 = k + 1 < kvalid ? p1 : 0.f;
          }
          pk[i >> 1] = pack_bf16(p0 * (dp[k] - dl), p1 * (dp[k + 1] - dl));
        }
        tmem_st8(tmem_ds + t_lane + c * 8, pk);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar_p_full);
    };
    for (int j = 0; j < n_kv; ++j) {
      if (bg.m - j * KT >= KT) tile(j, std::false_type{});
      else tile(j, std::true_type{});
    }
    mbar_wait(bar_dq_full, (n_kv - 1) & 1);
    tc_fence_after();
    float lo[32], hi[16];
    tmem_ld32(tmem_dq + t_lane, lo);
    tmem_ld16(tmem_dq + t_lane + 32, hi);
    tmem_ld_wait();
    if (qok) {
      const float sc = P.scale;
      float* dst = dqkv + (int64_t)pos * 3 * E + h * DH;
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        float4 a = *reinterpret_cast<const float4*>(dst + 4 * c);
        const float* v = c < 8 ? lo + 4 * c : hi + 4 * (c - 8);
        // product and sum rounded separately (no FMA contraction): the branch's value is v * sc whatever came before
        a.x = __fadd_rn(a.x, __fmul_rn(v[0], sc));
        a.y = __fadd_rn(a.y, __fmul_rn(v[1], sc));
        a.z = __fadd_rn(a.z, __fmul_rn(v[2], sc));
        a.w = __fadd_rn(a.w, __fmul_rn(v[3], sc));
        *reinterpret_cast<float4*>(dst + 4 * c) = a;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, TMEM_DQ_COLS);
}

// The launch parameters of ONE branch b of P: item i of the launch is item i of branch b.
static Sm100Params branch_only(const Sm100Params& P, int b) {
  Sm100Params Q = P;
  Q.order[0] = b;
  Q.item_prefix[0] = 0;
  for (int i = 1; i <= P.geo.nb; ++i) Q.item_prefix[i] = P.geo.b[b].n_seg * P.geo.H * P.tiles[b];
  return Q;
}

// impl 4.  Why the result is the same in every run:
//   * dqkv is zeroed by the caller (mt_dilated_attn_bwd); then the branches run one after another on the stream, branch
//     b = 0, 1, ..., nb - 1, each as two launches: dQ (dilated_bwd_dq_sm100_kernel) and dK / dV
//     (dilated_bwd_sm100_kernel<false>).  Stream order fixes the order in which the branches are added.
//   * Within one launch every element receives at most ONE non-zero addition: a (position, head) of a branch belongs to
//     exactly one (segment, head, slot), hence to one query tile (dQ: written by the thread of its row) and to one key
//     tile (dK / dV: one TMA reduce-add by the CTA of that tile).
//   * The only other additions are the +0.0 rows a key tile carries past its segment's m (the next segment's keys, masked
//     to P = 0).  Adding +0.0 gives the same bits in either order: x + 0 = x for x != -0, and the sum comes out +0 both
//     ways when it is zero.
// No CTA waits for another: the order comes from the stream, never from counters or spinning.
static int dilated_attn_bwd_deterministic(const Sm100Params& P, const TensorMaps& maps, const TensorMaps& do_maps,
                                          const TensorMaps& dq32_maps, const TensorMaps& dq16_maps, const void* qkv,
                                          int64_t qkv_ld, int64_t n_alloc, const float* lse, const float* delta_br,
                                          float* dqkv, cudaStream_t st) {
  TensorMaps kv_maps;
  memset(&kv_maps, 0, sizeof(kv_maps));
  for (int b = 0; b < P.geo.nb; ++b) {
    const int rc = encode_branch_map(&kv_maps.m[b], qkv, qkv_ld, n_alloc, P.geo.b[b].r, KT);
    if (rc) return rc;
  }
  static bool attr_set = false;   // once per process: the call is not free and never changes
  if (!attr_set) {
    MT_CUDA(cudaFuncSetAttribute(dilated_bwd_dq_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdDqSmem::TOTAL));
    MT_CUDA(cudaFuncSetAttribute(dilated_bwd_sm100_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Bwd3Smem::TOTAL));
    attr_set = true;
  }
  for (int b = 0; b < P.geo.nb; ++b) {
    const Sm100Params Pb = branch_only(P, b);
    const int items = Pb.item_prefix[1];
    if (items == 0) continue;
    dilated_bwd_dq_sm100_kernel<<<items, FWD_THREADS, BwdDqSmem::TOTAL, st>>>(maps, kv_maps, do_maps, Pb, lse, delta_br,
                                                                              dqkv);
    if (int rc = check_launch("dilated_bwd_dq_sm100_kernel")) return rc;
    dilated_bwd_sm100_kernel<false><<<items, BWD3_THREADS, Bwd3Smem::TOTAL, st>>>(maps, do_maps, dq32_maps, dq16_maps, Pb,
                                                                                  lse, delta_br);
    if (int rc = check_launch("dilated_bwd_sm100_kernel<false>")) return rc;
  }
  return 0;
}

int dilated_attn_bwd_sm100(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                           const void* dattn, const float* lse, const float* delta_br, float* dqkv, int impl,
                           cudaStream_t st) {
  Sm100Params P;
  int rc = make_sm100_params(geom, &P);
  if (rc) return rc;
  MT_REQUIRE(n_alloc >= P.geo.N && n_alloc % 128 == 0, "dilated_attn_bwd: n_alloc must be a multiple of 128 >= n_tokens");
  MT_REQUIRE(qkv_ld % 8 == 0 && ((uintptr_t)qkv & 15) == 0 && ((uintptr_t)dattn & 15) == 0 && ((uintptr_t)dqkv & 15) == 0,
             "dilated_attn_bwd: buffers must be 16-byte aligned");
  TensorMaps maps, do_maps, dq32_maps, dq16_maps;
  memset(&maps, 0, sizeof(maps));
  memset(&do_maps, 0, sizeof(do_maps));
  memset(&dq32_maps, 0, sizeof(dq32_maps));
  memset(&dq16_maps, 0, sizeof(dq16_maps));
  const int64_t E = (int64_t)P.geo.H * DH;
  for (int b = 0; b < P.geo.nb; ++b) {
    rc = encode_branch_map(&maps.m[b], qkv, qkv_ld, n_alloc, P.geo.b[b].r);
    if (rc) return rc;
    rc = encode_branch_map(&do_maps.m[b], dattn, E, n_alloc, P.geo.b[b].r);
    if (rc) return rc;
    rc = encode_branch_map_f32(&dq32_maps.m[b], dqkv, 3 * E, n_alloc, P.geo.b[b].r, 32);
    if (rc) return rc;
    rc = encode_branch_map_f32(&dq16_maps.m[b], dqkv, 3 * E, n_alloc, P.geo.b[b].r, 16);
    if (rc) return rc;
  }
  if (impl == 2) {   // persistent CTAs (one per SM) with a device work counter
    int* counter = next_work_counter();
    MT_REQUIRE(counter != nullptr, "dilated_attn_bwd: cannot allocate the work counters");
    const int items = P.item_prefix[P.geo.nb];
    const int grid = items < kNumSMs ? items : kNumSMs;
    {
    static bool attr_set = false;   // once per process: the call is not free and never changes
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(dilated_bwd_sm100_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdPSmem::TOTAL));
      attr_set = true;
    }
  }
    dilated_bwd_sm100_persistent_kernel<<<grid, BWD3_THREADS, BwdPSmem::TOTAL, st>>>(maps, do_maps, dq32_maps, dq16_maps, P,
                                                                                    lse, delta_br, counter);
    return check_launch("dilated_bwd_sm100_persistent_kernel");
  }
  if (impl == 4) return dilated_attn_bwd_deterministic(P, maps, do_maps, dq32_maps, dq16_maps, qkv, qkv_ld, n_alloc, lse,
                                                      delta_br, dqkv, st);
  {
    static bool attr_set = false;   // once per process: the call is not free and never changes
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(dilated_bwd_sm100_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Bwd3Smem::TOTAL));
      attr_set = true;
    }
  }
  dilated_bwd_sm100_kernel<true><<<P.item_prefix[P.geo.nb], BWD3_THREADS, Bwd3Smem::TOTAL, st>>>(
      maps, do_maps, dq32_maps, dq16_maps, P, lse, delta_br);
  return check_launch("dilated_bwd_sm100_kernel");
}

}  // namespace mt

#ifdef MT_DEBUG_TIMELINE
// experiment builds only: copy the CTA timeline to the host ([n][4] long long) and clear it
extern "C" int mt_debug_item_timeline(long long* dst, int n) {
  if (n > 65536) n = 65536;
  cudaDeviceSynchronize();
  int cnt = 0;
  if (cudaMemcpyFromSymbol(&cnt, mt::mt_item_count, sizeof(int)) != cudaSuccess) return -1;
  if (cnt > n) cnt = n;
  if (cudaMemcpyFromSymbol(dst, mt::mt_item_timeline, sizeof(long long) * 4 * (size_t)cnt) != cudaSuccess) return -1;
  int zero = 0;
  cudaMemcpyToSymbol(mt::mt_item_count, &zero, sizeof(int));
  return cnt;
}
extern "C" int mt_debug_timeline(long long* dst, int n) {
  if (n > 32768) n = 32768;
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(dst, mt::mt_timeline, sizeof(long long) * 4 * (size_t)n) != cudaSuccess) return -1;
  void* p = nullptr;
  cudaGetSymbolAddress(&p, mt::mt_timeline);
  cudaMemset(p, 0, sizeof(long long) * 4 * 32768);
  return 0;
}
#endif
