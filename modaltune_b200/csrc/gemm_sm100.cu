// Frozen-linear GEMMs of the LongNet encoder layer on the 5th-generation tensor cores (sm_100a), with the element-wise
// work that follows each projection fused into the epilogue.
//
//     C[M, N] = A[M, K] . W[N, K]^T        A = activations (bf16, row-major), W = nn.Linear weight (bf16, [out, in])
//
// replaces, per encoder layer (torchscale/component/multihead_attention.py:44-54, feedforward_network.py:132-143,
// architecture/encoder.py:137-175): the q/k/v projection (+ bias), out_proj (+ bias + residual add), fc1 (+ bias + GELU
// + the row statistics of ffn_layernorm), fc2 (ffn_layernorm folded in algebraically + bias + residual add), and the
// dX GEMMs of the backward (every encoder weight is frozen: no dW).
//
// One persistent CTA per SM walks the 128 x 256 output tiles (n fastest: the ~12 row blocks in flight and the whole
// weight stay in L2).  Warp roles: warp 0 = TMA producer (A 128 x 64 and W 256 x 64 bf16 boxes, 128-byte swizzle, 4-stage
// ring), warp 1 = tcgen05.mma issuer (M 128, N 256, K 16; fp32 accumulators in TMEM, two 256-column accumulators so that
// the epilogue of tile t overlaps the main loop of tile t + 1), warps 2-9 = epilogue (TMEM lane = output row; warps w and
// w + 4 share 32 rows and take 128 columns each).
//
// LayerNorm folding (fc2): fc2(LN(u)) = rstd * (u W2'^T - mean * c1) + c2 with W2' = W2 diag(gamma), c1 = W2' 1,
// c2 = W2 beta + b2 -- all constants of the frozen layer -- so the normalised [M, 3072] tensor is never written: fc1's
// epilogue emits gelu(h) in bf16 plus per-row (sum, sum of squares), fc2's epilogue applies mean / rstd per row.
#include <cuda.h>

#include <cstring>

#include "mt_common.cuh"
#include "sm100_ptx.cuh"

namespace mt {
using namespace sm100;

namespace gemm {
constexpr int BM = 128, BN = 256, BK = 64;
constexpr int A_BYTES = BM * BK * 2;        // 16 KB
constexpr int THREADS = 32 * 10;            // TMA, MMA, 8 epilogue warps
constexpr int STG_F32 = 32 * 128;           // per epilogue warp: [32 rows][32 floats], 128-byte swizzle
constexpr int STG_BF16 = 32 * 64;           // per epilogue warp: [32 rows][32 bf16], 64-byte swizzle

// PAIR = two CTAs of a cluster execute M = 256 MMAs (cta_group::2): every CTA keeps its own 128 rows of A and HALF of
// the 256 rows of W in shared memory.  Measured on B200: the one-CTA kernel is bound by shared-memory bandwidth (per
// 128 x 256 x 768 tile the tensor core reads 576 KB of operands, TMA writes 576 KB and the epilogue stages 256 KB:
// 11 k cycles of the 128 B / clk pipe against 6.1 k cycles of MMA); the pair halves the W traffic of both kinds.
template <bool PAIR>
struct Cfg {
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;        // W rows held by one CTA
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = PAIR ? 5 : 3;
  static constexpr int SMEM_STG32 = STAGES * STAGE_BYTES;
  static constexpr int SMEM_STG16 = SMEM_STG32 + 8 * STG_F32;
  static constexpr int SMEM_BAR = SMEM_STG16 + 8 * STG_BF16;
  static constexpr int NBAR = 2 * STAGES + 4;              // full[S], empty[S], acc_full[2], acc_empty[2]
  static constexpr int SMEM_TMEM_PTR = SMEM_BAR + NBAR * 8;
  static constexpr int SMEM_TOTAL = SMEM_TMEM_PTR + 16;
};
static_assert(Cfg<false>::SMEM_TOTAL <= 232448 && Cfg<true>::SMEM_TOTAL <= 232448, "shared memory of the GEMM kernels");

struct Params {
  int M, N, K;
  int mode;
  const float* bias;        // [N] or null
  const float* residual;    // [M, N] f32 (modes 0, 4)
  const float* col_c1;      // [N] (mode 4)
  const float* col_c2;      // [N] (mode 4)
  float* stats;             // [M, cols / 128, 2]: (sum, sum of squares) per 128-column slab: written in mode 3, read in mode 4
  const float4* rowv;       // mode 5: [M] (mean, rstd, m1, m2) per row (mt_ffn_bwd_prep)
  float* mean_out;          // mode 4: [M] or null
  float* rstd_out;
  float* out_f32;           // [M, N] or null
  __nv_bfloat16* out_bf16;  // [M, N] or null
  __nv_bfloat16* out_aux;   // mode 3: [M, N] gelu'(h) in bf16 or null
  const __nv_bfloat16* in_u;   // mode 5 without h: [M, N] gelu(h) and gelu'(h) in bf16 as written by mode 3
  const __nv_bfloat16* in_g;
  int64_t ld_res;
  float ln_eps;
  float inv_ln_cols;        // 1 / (number of columns the statistics were summed over)
  int ln_parts;             // mode 4: partial sums per row = ln_cols / 128
};

// gelu(x) = x * Phi(x) with erf from Abramowitz-Stegun 7.1.26 (absolute error 1.5e-7: fp32-level; two MUFU ops)
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t;   // 1 / (1 + p z): the approximate reciprocal is one MUFU op (1 ulp), __frcp_rn is a software routine
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = ex2(-z * z * 1.4426950408889634f);
  const float erf_abs = 1.f - p * t * e;                 // erf(|x| / sqrt 2)
  const float half_x = 0.5f * x;
  return fmaf(copysignf(erf_abs, x), half_x, half_x);     // 0.5 x (1 + erf(x / sqrt 2))
}

// u = gelu(x) and gelu'(x) = Phi(x) + x phi(x) from one erf evaluation (same two MUFU ops as gelu_erf)
__device__ __forceinline__ void gelu_erf_val_grad(float x, float& u, float& du) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = ex2(-z * z * 1.4426950408889634f);    // exp(-x^2 / 2)
  const float erf_abs = 1.f - p * t * e;
  const float cdf = fmaf(copysignf(erf_abs, x), 0.5f, 0.5f);
  u = x * cdf;
  du = fmaf(x * 0.3989422804014327f, e, cdf);
}

template <bool PAIR>
__device__ __forceinline__ void linear_body(const CUtensorMap& map_a, const CUtensorMap& map_b, const CUtensorMap& map_c,
                                            const CUtensorMap& map_c16, const CUtensorMap& map_aux, const Params& P) {
  using C = Cfg<PAIR>;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sbase & 1023u) != 0) __trap();
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;      // 0 = leader of the pair
  const uint32_t bar_full = sbase + C::SMEM_BAR;
  const uint32_t bar_empty = bar_full + 8 * C::STAGES;
  const uint32_t bar_acc_full = bar_empty + 8 * C::STAGES;   // [2]
  const uint32_t bar_acc_empty = bar_acc_full + 16;          // [2] (PAIR: the leader's copy collects both CTAs)
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + C::SMEM_TMEM_PTR);

  constexpr int TILE_M = PAIR ? 2 * BM : BM;                  // rows of one work item (both CTAs of a pair)
  const int m_tiles = (P.M + TILE_M - 1) / TILE_M, n_tiles = P.N / BN, k_blocks = P.K / BK;
  const int tiles = m_tiles * n_tiles;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < C::STAGES; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, PAIR ? 512 : 256);
    }
    fence_barrier_init();
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    if (P.out_f32 != nullptr) tma_prefetch_desc(&map_c);
    if (P.out_bf16 != nullptr) tma_prefetch_desc(&map_c16);
    if (P.out_aux != nullptr) tma_prefetch_desc(&map_aux);
  }
  if (warp == 1) {
    if (PAIR) {
      tmem_alloc_pair(smem_u32((const void*)tmem_slot), 512);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(smem_u32((const void*)tmem_slot), 512);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (both CTAs of a pair: each loads its own rows of A and its half of W) ========================
    if (lane == 0) {
      int it = 0;
      for (int t = worker; t < tiles; t += n_workers) {
        const int m0 = (t / n_tiles) * TILE_M + (int)rank * BM, n0 = (t % n_tiles) * BN + (int)rank * C::B_ROWS;
        for (int kb = 0; kb < k_blocks; ++kb, ++it) {
#ifdef MT_EXP_NO_TMA    // experiment builds only (wrong results): the tensor pipe alone, operands loaded once
          if (it >= C::STAGES) continue;
#endif
          const int st = it % C::STAGES;
          mbar_wait(bar_empty + 8 * st, ((it / C::STAGES) & 1) ^ 1);
          const uint32_t dst = sbase + st * C::STAGE_BYTES;
          if (PAIR) {
            // the leader's barrier collects the bytes of both CTAs; only the leader arms it
            if (rank == 0) mbar_expect_tx(bar_full + 8 * st, 2 * C::STAGE_BYTES);
            tma_load_2d_pair(dst, &map_a, bar_full + 8 * st, kb * BK, m0);
            tma_load_2d_pair(dst + A_BYTES, &map_b, bar_full + 8 * st, kb * BK, n0);
          } else {
            mbar_expect_tx(bar_full + 8 * st, C::STAGE_BYTES);
            tma_load_2d(dst, &map_a, bar_full + 8 * st, kb * BK, m0);
            tma_load_2d(dst + A_BYTES, &map_b, bar_full + 8 * st, kb * BK, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (the leader CTA of a pair) =======================================================================
    if (!PAIR || rank == 0) {
      constexpr uint32_t IDESC = umma_idesc_bf16(TILE_M, BN, 0, 0);
      const uint64_t a_desc0 = umma_smem_desc(sbase, 16, 1024);
      const uint64_t b_desc0 = umma_smem_desc(sbase + A_BYTES, 16, 1024);
      int it = 0, tl = 0;
      for (int t = worker; t < tiles; t += n_workers, ++tl) {
        const int buf = tl & 1;
        mbar_wait(bar_acc_empty + 8 * buf, ((tl >> 1) & 1) ^ 1);   // the epilogue(s) have read this accumulator
        tc_fence_after();
        const uint32_t acc = tmem + buf * BN;
        for (int kb = 0; kb < k_blocks; ++kb, ++it) {
          const int st = it % C::STAGES;
#ifdef MT_EXP_NO_TMA
          if (it < C::STAGES)
#endif
          mbar_wait(bar_full + 8 * st, (it / C::STAGES) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t ad = umma_desc_adv(a_desc0, (uint32_t)st * C::STAGE_BYTES);
            const uint64_t bd = umma_desc_adv(b_desc0, (uint32_t)st * C::STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              if (PAIR) umma_ss_pair(acc, umma_desc_adv(ad, k * 32), umma_desc_adv(bd, k * 32), IDESC, (kb > 0) || (k > 0));
              else umma_ss(acc, umma_desc_adv(ad, k * 32), umma_desc_adv(bd, k * 32), IDESC, (kb > 0) || (k > 0));
            }
            if (PAIR) {
              umma_commit_pair(bar_empty + 8 * st);
              if (kb == k_blocks - 1) umma_commit_pair(bar_acc_full + 8 * buf);
            } else {
              umma_commit(bar_empty + 8 * st);
              if (kb == k_blocks - 1) umma_commit(bar_acc_full + 8 * buf);
            }
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ===== epilogue: 8 warps, thread = (output row, 128 of the 256 tile columns) ======================================
    const int ew = warp - 2;
    const int lane_grp = warp & 3;                 // TMEM lanes this warp may touch: 32 * (warp id % 4)
    const int half = ew >> 2;                      // which 128 columns
    const int row_in_tile = lane_grp * 32 + lane;
    const uint32_t t_lane = (uint32_t)(lane_grp * 32) << 16;
    // Outputs leave through per-warp staging tiles and TMA stores: a thread owns a ROW of the accumulator, so direct
    // stores touch 32 different rows per instruction (measured: 80 k of the epilogue's 90 k cycles with bf16 output);
    // staged, every global write is a full line and asynchronous.
    uint8_t* stg32 = smem + C::SMEM_STG32 + ew * STG_F32;
    uint8_t* stg16 = smem + C::SMEM_STG16 + ew * STG_BF16;
    const uint32_t stg32_u32 = sbase + C::SMEM_STG32 + ew * STG_F32;
    const uint32_t stg16_u32 = sbase + C::SMEM_STG16 + ew * STG_BF16;
    // one 32-column chunk of this warp's 32 rows: fp32 and / or bf16 copy
    auto store_chunk = [&](const float (&o)[32], int col, int row0, bool f32, bool b16, bool aux = false) {
      if (lane == 0) bulk_wait_group_read<0>();       // the previous stores of this warp have read the staging tiles
      __syncwarp();
      if (f32) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<float4*>(stg32 + lane * 128 + ((i ^ (lane & 7)) << 4)) =
              make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
      }
      if (b16) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<uint4*>(stg16 + lane * 64 + ((i ^ ((lane >> 1) & 3)) << 4)) =
              make_uint4(pack_bf16(o[8 * i], o[8 * i + 1]), pack_bf16(o[8 * i + 2], o[8 * i + 3]),
                         pack_bf16(o[8 * i + 4], o[8 * i + 5]), pack_bf16(o[8 * i + 6], o[8 * i + 7]));
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (f32) tma_store_2d(&map_c, stg32_u32, col, row0);
        if (b16) tma_store_2d(aux ? &map_aux : &map_c16, stg16_u32, col, row0);
        bulk_commit_group();
      }
    };
    int tl = 0;
    for (int t = worker; t < tiles; t += n_workers, ++tl) {
      const int buf = tl & 1;
      const int m0 = (t / n_tiles) * TILE_M + (int)rank * BM, n0 = (t % n_tiles) * BN + half * 128;
      const int row = m0 + row_in_tile;
      const bool row_ok = row < P.M;
      mbar_wait(bar_acc_full + 8 * buf, (tl >> 1) & 1);
      tc_fence_after();
#ifdef MT_EXP_NO_EPI    // experiment builds only (wrong results): main loop alone
      tc_fence_before();
      if (PAIR) mbar_arrive_leader(bar_acc_empty + 8 * buf); else mbar_arrive(bar_acc_empty + 8 * buf);
      continue;
#endif
      const uint32_t acc = tmem + buf * BN + half * 128 + t_lane;
      float mean = 0.f, rstd = 1.f;
      if (P.mode == 4 && row_ok) {
        // the partial (sum, sum of squares) of every 128-column slab of the producing GEMM, added in a fixed order:
        // deterministic, and nobody has to zero the buffer
        const float2* part = reinterpret_cast<const float2*>(P.stats) + (int64_t)row * P.ln_parts;
        float2 ss = make_float2(0.f, 0.f);
        for (int i = 0; i < P.ln_parts; ++i) {
          const float2 pi = part[i];
          ss.x += pi.x;
          ss.y += pi.y;
        }
        mean = ss.x * P.inv_ln_cols;
        const float var = fmaxf(ss.y * P.inv_ln_cols - mean * mean, 0.f);
        rstd = rsqrtf(var + P.ln_eps);
        if (P.mean_out != nullptr && n0 == 0) {      // one thread per row publishes the statistics for the backward
          P.mean_out[row] = mean;
          P.rstd_out[row] = rstd;
        }
      }
      float4 rv = make_float4(0.f, 1.f, 0.f, 0.f);
      if (P.mode == 5 && row_ok) rv = P.rowv[row];
      float s1 = 0.f, s2 = 0.f;
      const int row0 = m0 + lane_grp * 32;          // first row of this warp's 32-row slab (rows >= M are clipped by TMA)
#pragma unroll 1
      for (int c = 0; c < 128; c += 32) {
        float v[32];
        tmem_ld32(acc + c, v);
        tmem_ld_wait();
        if (c == 96) {                             // the whole accumulator is in registers: release it to the MMA warp
          tc_fence_before();
          if (PAIR) mbar_arrive_leader(bar_acc_empty + 8 * buf); else mbar_arrive(bar_acc_empty + 8 * buf);
        }
        const int col = n0 + c;
        if (P.mode == 3) {
          // h = acc + bias (kept in fp32 for the backward), u = gelu(h) in bf16 for fc2, row statistics of the ROUNDED u
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b = *reinterpret_cast<const float4*>(P.bias + col + i);
            v[i] += b.x; v[i + 1] += b.y; v[i + 2] += b.z; v[i + 3] += b.w;
          }
          if (P.out_f32 != nullptr) store_chunk(v, col, row0, true, false);
          float gd[32];   // gelu'(h): costs one FMA more than gelu(h) alone (the exponential is shared)
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float u0, u1;
            gelu_erf_val_grad(v[i], u0, gd[i]);
            gelu_erf_val_grad(v[i + 1], u1, gd[i + 1]);
            const __nv_bfloat162 u2 = __floats2bfloat162_rn(u0, u1);
            const float2 f = __bfloat1622float2(u2);
            s1 += f.x + f.y;
            s2 = fmaf(f.x, f.x, fmaf(f.y, f.y, s2));
            v[i] = f.x;
            v[i + 1] = f.y;
          }
          store_chunk(v, col, row0, false, true);
          if (P.out_aux != nullptr) store_chunk(gd, col, row0, false, true, true);
        } else if (P.mode == 5) {
          // backward of GELU + LayerNorm(3072) on the accumulator of the dX GEMM of fc2 (W = (W2 diag gamma)^T, so
          // acc_j = gamma_j dn_j): d_h_j = gelu'(h_j) rstd (acc_j - m1 - uhat_j m2), uhat_j = (gelu(h_j) - mean) rstd,
          // with h = fc1's fp32 output (P.residual) and the row means m1, m2 formed BEFORE the GEMM (mt_ffn_bwd_prep)
          if (row_ok && P.in_u != nullptr) {
            // gelu(h) (the ROUNDED values the forward's statistics were taken over) and gelu'(h) saved by the forward
            const uint4* us = reinterpret_cast<const uint4*>(P.in_u + (int64_t)row * P.N + col);
            const uint4* gs = reinterpret_cast<const uint4*>(P.in_g + (int64_t)row * P.N + col);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint4 uu = us[i], gg = gs[i];
              const __nv_bfloat162* up = reinterpret_cast<const __nv_bfloat162*>(&uu);
              const __nv_bfloat162* gp = reinterpret_cast<const __nv_bfloat162*>(&gg);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 uf = __bfloat1622float2(up[j]), gf = __bfloat1622float2(gp[j]);
                const int e = 8 * i + 2 * j;
                v[e] = gf.x * rv.y * (v[e] - rv.z - (uf.x - rv.x) * rv.y * rv.w);
                v[e + 1] = gf.y * rv.y * (v[e + 1] - rv.z - (uf.y - rv.x) * rv.y * rv.w);
              }
            }
          } else if (row_ok) {
            const float* hs = P.residual + (int64_t)row * P.ld_res + col;
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 h4 = *reinterpret_cast<const float4*>(hs + i);
              const float hv[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float u, du;
                gelu_erf_val_grad(hv[j], u, du);
                const float uh = (u - rv.x) * rv.y;
                v[i + j] = du * rv.y * (v[i + j] - rv.z - uh * rv.w);
              }
            }
          }
          store_chunk(v, col, row0, P.out_f32 != nullptr, P.out_bf16 != nullptr);
        } else {
          if (P.mode == 4) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 c1 = *reinterpret_cast<const float4*>(P.col_c1 + col + i);
              const float4 c2 = *reinterpret_cast<const float4*>(P.col_c2 + col + i);
              v[i] = fmaf(rstd, fmaf(-mean, c1.x, v[i]), c2.x);
              v[i + 1] = fmaf(rstd, fmaf(-mean, c1.y, v[i + 1]), c2.y);
              v[i + 2] = fmaf(rstd, fmaf(-mean, c1.z, v[i + 2]), c2.z);
              v[i + 3] = fmaf(rstd, fmaf(-mean, c1.w, v[i + 3]), c2.w);
            }
          } else if (P.bias != nullptr) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b = *reinterpret_cast<const float4*>(P.bias + col + i);
              v[i] += b.x; v[i + 1] += b.y; v[i + 2] += b.z; v[i + 3] += b.w;
            }
          }
          if (P.residual != nullptr && row_ok) {
            const float* rs = P.residual + (int64_t)row * P.ld_res + col;
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 r = *reinterpret_cast<const float4*>(rs + i);
              v[i] += r.x; v[i + 1] += r.y; v[i + 2] += r.z; v[i + 3] += r.w;
            }
          }
          store_chunk(v, col, row0, P.out_f32 != nullptr, P.out_bf16 != nullptr);
        }
      }
      if (P.mode == 3 && row_ok)   // this thread's 128-column slab of the row: slab index = n0 / 128 of N / 128
        reinterpret_cast<float2*>(P.stats)[(int64_t)row * (P.N / 128) + n0 / 128] = make_float2(s1, s2);
    }
    if (lane == 0) bulk_wait_group_read<0>();
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // PAIR: no CTA may exit while its peer still signals its barriers
  if (warp == 1) {
    if (PAIR) tmem_dealloc_pair(tmem, 512);
    else tmem_dealloc(tmem, 512);
  }
}

__global__ void __launch_bounds__(THREADS, 1)
linear_sm100_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_c16,
                    const __grid_constant__ CUtensorMap map_aux, const Params P) {
  linear_body<false>(map_a, map_b, map_c, map_c16, map_aux, P);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
linear_sm100_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                         const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_c16,
                         const __grid_constant__ CUtensorMap map_aux, const Params P) {
  linear_body<true>(map_a, map_b, map_c, map_c16, map_aux, P);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
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

// row-major [rows, ld] output, box = [32 rows][32 columns]: fp32 = one 128-byte swizzle atom per row, bf16 = 64-byte
static int encode_out(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, bool bf16) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return MT_E_UNSUPPORTED;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (bf16 ? 2 : 4)};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a [%lld, %lld] output", (int)rc, (long long)rows, (long long)cols);
    return MT_E_BADARG;
  }
  return 0;
}

// row-major [rows, ld] bf16 matrix, box = [box_rows][64 columns], 128-byte swizzle, rows past the end read as zero
static int encode_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return MT_E_UNSUPPORTED;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a [%lld, %lld] bf16 matrix", (int)rc, (long long)rows, (long long)cols);
    return MT_E_BADARG;
  }
  return 0;
}
}  // namespace gemm
}  // namespace mt

using namespace mt;

extern "C" int mt_linear_sm100(const void* a, int64_t lda, const void* w, int64_t ldw, int64_t M, int64_t N, int64_t K,
                               const mt_linear_epilogue* ep, void* stream) {
  MT_REQUIRE(a != nullptr && w != nullptr && ep != nullptr, "linear_sm100: NULL argument");
  MT_REQUIRE(M > 0 && N > 0 && K > 0 && N % gemm::BN == 0 && K % gemm::BK == 0,
             "linear_sm100: N must be a multiple of 256 and K a multiple of 64 (got M=%lld N=%lld K=%lld)", (long long)M,
             (long long)N, (long long)K);
  MT_REQUIRE(lda % 8 == 0 && ldw % 8 == 0 && ((uintptr_t)a & 15) == 0 && ((uintptr_t)w & 15) == 0,
             "linear_sm100: operands must be 16-byte aligned with row strides that are multiples of 8 elements");
  MT_REQUIRE(ep->mode == MT_EPI_PLAIN || ep->mode == MT_EPI_GELU_STATS || ep->mode == MT_EPI_LN_RESIDUAL ||
                 ep->mode == MT_EPI_GELU_LN_BWD, "linear_sm100: bad epilogue mode %d", ep->mode);
  MT_REQUIRE(ep->out_f32 != nullptr || ep->out_bf16 != nullptr, "linear_sm100: no output");
  if (ep->mode == MT_EPI_GELU_STATS)
    MT_REQUIRE(ep->bias && ep->out_bf16 && ep->stats, "linear_sm100: GELU epilogue needs bias, the bf16 output and stats");
  MT_REQUIRE(ep->out_aux_bf16 == nullptr || ep->mode == MT_EPI_GELU_STATS, "linear_sm100: out_aux_bf16 belongs to the GELU epilogue");
  if (ep->mode == MT_EPI_LN_RESIDUAL)
    MT_REQUIRE(ep->col_c1 && ep->col_c2 && ep->stats && ep->ln_cols > 0, "linear_sm100: LN-fold epilogue needs c1, c2, stats, ln_cols");
  if (ep->mode == MT_EPI_GELU_LN_BWD)
    MT_REQUIRE((ep->residual || (ep->in_u_bf16 && ep->in_g_bf16)) && ep->stats && ((uintptr_t)ep->stats & 15) == 0 &&
                   ep->bias == nullptr && (((uintptr_t)ep->in_u_bf16 | (uintptr_t)ep->in_g_bf16) & 15) == 0,
               "linear_sm100: GELU-LN backward epilogue needs h (residual) or gelu / gelu' (in_u_bf16, in_g_bf16), "
               "stats = [M, 4] row vector, no bias");
  gemm::Params P;
  P.M = (int)M; P.N = (int)N; P.K = (int)K;
  P.rowv = reinterpret_cast<const float4*>(ep->stats);
  P.mode = ep->mode;
  P.bias = ep->bias; P.residual = ep->residual; P.col_c1 = ep->col_c1; P.col_c2 = ep->col_c2; P.stats = ep->stats;
  P.mean_out = ep->ln_mean_out; P.rstd_out = ep->ln_rstd_out;
  MT_REQUIRE((P.mean_out == nullptr) == (P.rstd_out == nullptr), "linear_sm100: ln_mean_out and ln_rstd_out go together");
  P.out_f32 = ep->out_f32; P.out_bf16 = (__nv_bfloat16*)ep->out_bf16;
  P.out_aux = (__nv_bfloat16*)ep->out_aux_bf16;
  P.in_u = (const __nv_bfloat16*)ep->in_u_bf16; P.in_g = (const __nv_bfloat16*)ep->in_g_bf16;
  const int64_t ld_f32 = ep->ld_out_f32 ? ep->ld_out_f32 : N;
  const int64_t ld_bf16 = ep->ld_out_bf16 ? ep->ld_out_bf16 : N;
  P.ld_res = ep->ld_residual ? ep->ld_residual : N;
  P.ln_eps = ep->ln_eps;
  P.inv_ln_cols = ep->ln_cols > 0 ? 1.0f / (float)ep->ln_cols : 0.f;
  P.ln_parts = ep->ln_cols / 128;
  MT_REQUIRE(ep->mode != MT_EPI_LN_RESIDUAL || ep->ln_cols % 128 == 0, "linear_sm100: ln_cols must be a multiple of 128");
  MT_REQUIRE(ld_f32 % 4 == 0 && ld_bf16 % 8 == 0 && P.ld_res % 4 == 0, "linear_sm100: output row strides must keep 16-byte alignment");
  // impl: 0 = pick (CTA pairs when there is more than one 256-row block), 1 = one CTA per tile, 2 = CTA pairs
  int impl = ep->impl;
  if (impl == 0) impl = M > gemm::BM ? 2 : 1;
  MT_REQUIRE(impl == 1 || impl == 2, "linear_sm100: bad impl %d", ep->impl);
  const bool pair = impl == 2;
  CUtensorMap map_a, map_b, map_c, map_c16, map_aux;
  memset(&map_c, 0, sizeof(map_c));
  memset(&map_c16, 0, sizeof(map_c16));
  memset(&map_aux, 0, sizeof(map_aux));
  int rc = gemm::encode_2d(&map_a, a, M, K, lda, gemm::BM);
  if (rc) return rc;
  rc = gemm::encode_2d(&map_b, w, N, K, ldw, pair ? gemm::BN / 2 : gemm::BN);
  if (rc) return rc;
  if (ep->out_f32 != nullptr) {
    MT_REQUIRE(((uintptr_t)ep->out_f32 & 15) == 0, "linear_sm100: the fp32 output must be 16-byte aligned");
    rc = gemm::encode_out(&map_c, ep->out_f32, M, N, ld_f32, false);
    if (rc) return rc;
  }
  if (ep->out_bf16 != nullptr) {
    MT_REQUIRE(((uintptr_t)ep->out_bf16 & 15) == 0, "linear_sm100: the bf16 output must be 16-byte aligned");
    rc = gemm::encode_out(&map_c16, ep->out_bf16, M, N, ld_bf16, true);
    if (rc) return rc;
  }
  if (ep->out_aux_bf16 != nullptr) {
    MT_REQUIRE(((uintptr_t)ep->out_aux_bf16 & 15) == 0, "linear_sm100: the auxiliary bf16 output must be 16-byte aligned");
    rc = gemm::encode_out(&map_aux, ep->out_aux_bf16, M, N, N, true);
    if (rc) return rc;
  }
  if (pair) {
    const int tiles = (int)((M + 2 * gemm::BM - 1) / (2 * gemm::BM) * (N / gemm::BN));
    const int pairs = tiles < kNumSMs / 2 ? tiles : kNumSMs / 2;
    {
    static bool attr_set = false;   // once per process: the call is not free and never changes
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(gemm::linear_sm100_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm::Cfg<true>::SMEM_TOTAL));
      attr_set = true;
    }
  }
    gemm::linear_sm100_pair_kernel<<<2 * pairs, gemm::THREADS, gemm::Cfg<true>::SMEM_TOTAL, (cudaStream_t)stream>>>(
        map_a, map_b, map_c, map_c16, map_aux, P);
    return check_launch("linear_sm100_pair_kernel");
  }
  const int tiles = (int)((M + gemm::BM - 1) / gemm::BM * (N / gemm::BN));
  const int grid = tiles < kNumSMs ? tiles : kNumSMs;
  {
    static bool attr_set = false;   // once per process: the call is not free and never changes
    if (!attr_set) {
      MT_CUDA(cudaFuncSetAttribute(gemm::linear_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm::Cfg<false>::SMEM_TOTAL));
      attr_set = true;
    }
  }
  gemm::linear_sm100_kernel<<<grid, gemm::THREADS, gemm::Cfg<false>::SMEM_TOTAL, (cudaStream_t)stream>>>(
      map_a, map_b, map_c, map_c16, map_aux, P);
  return check_launch("linear_sm100_kernel");
}
