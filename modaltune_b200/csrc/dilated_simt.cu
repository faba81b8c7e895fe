// LongNet dilated attention, fp32-math SIMT kernels (the fp32 mode of the path, and the on-device cross-check of the
// tcgen05 kernels) + the branch merge fused with inner_attn_ln (fwd and bwd).
//
// Work decomposition: one CTA per (branch, segment, head, 64-slot tile); the dilated gather is index math on the
// tile load (position = s*g + floor(h*r/H) + slot*r), nothing is materialised.  Slots whose position falls outside the
// sequence / segment are the reference's zero-padded tokens: loaded as zero rows, they take part in the softmax
// denominator with score 0 (dilated_attention.py:82-111, see oracle/modaltune_oracle.py:dilated_attention_core).
#include "mt_common.cuh"

namespace mt {

static constexpr int D = 48;       // head dim of LongNet-12L-768d (16 heads)
static constexpr int BM = 64;      // slots per tile
static constexpr int LDQ = D + 1;  // padded smem row (bank-conflict free column reads)
static constexpr int LDP = BM + 1;

struct SimtParams {
  DilatedGeom geo;
  int item_prefix[MT_MAX_BRANCHES + 1];  // first CTA of each branch
  int tiles[MT_MAX_BRANCHES];            // 64-slot tiles per (segment, head)
  int64_t qkv_ld;
};

struct Item {
  int b, h, s, tile;
};

__device__ __forceinline__ Item decode_item(const SimtParams& P, int bid) {
  Item it;
  it.b = 0;
  while (it.b + 1 < P.geo.nb && bid >= P.item_prefix[it.b + 1]) ++it.b;
  int local = bid - P.item_prefix[it.b];
  it.tile = local % P.tiles[it.b];
  local /= P.tiles[it.b];
  it.h = local % P.geo.H;
  it.s = local / P.geo.H;
  return it;
}

// load a [64 x 48] tile of q / k / v / dO rows for slots slot0.. of (branch, segment, head) into padded smem (fp32)
template <typename T>
__device__ __forceinline__ void load_tile(float* dst, const T* __restrict__ base, int64_t ld, int col0, int slot0,
                                          int m, int pos0, int r, int seg_end) {
  // 64 rows x 6 chunks of 8 elements = 384 chunk loads over 256 threads
  for (int idx = threadIdx.x; idx < BM * (D / 8); idx += blockDim.x) {
    const int row = idx / (D / 8), ch = idx % (D / 8);
    const int slot = slot0 + row;
    const int p = pos0 + slot * r;
    float v[8];
    if (slot < m && p < seg_end) {
      load8(base + (int64_t)p * ld + col0 + ch * 8, v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[row * LDQ + ch * 8 + j] = v[j];
  }
}

// blockIdx.y = sequence of a batch: qkv, o_br and lse_br advance by seq_qkv / seq_o / seq_lse elements per sequence
template <typename T>
__global__ void __launch_bounds__(256) dilated_fwd_simt_kernel(const SimtParams P, const T* __restrict__ qkv,
                                                               T* __restrict__ o_br, float* __restrict__ lse_br,
                                                               int64_t seq_qkv, int64_t seq_o, int64_t seq_lse) {
  extern __shared__ float smem[];
  qkv += blockIdx.y * seq_qkv;
  o_br += blockIdx.y * seq_o;
  lse_br += blockIdx.y * seq_lse;
  float* Qs = smem;
  float* Ks = Qs + BM * LDQ;
  float* Vs = Ks + BM * LDQ;
  float* Ps = Vs + BM * LDQ;
  const Item it = decode_item(P, blockIdx.x);
  const BranchGeom bg = P.geo.b[it.b];
  const int H = P.geo.H, N = P.geo.N, E = H * D;
  const int off = (it.h * bg.r) / H;
  const int pos0 = it.s * bg.g + off;
  const int seg_end = min(N, (it.s + 1) * bg.g);
  const int q0 = it.tile * BM;
  const float scale = rsqrtf((float)D);
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;

  load_tile(Qs, qkv, P.qkv_ld, it.h * D, q0, bg.m, pos0, bg.r, seg_end);
  float m_run[4], l_run[4], o[4][3];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_run[i] = -INFINITY;
    l_run[i] = 0.f;
    o[i][0] = o[i][1] = o[i][2] = 0.f;
  }
  for (int k0 = 0; k0 < bg.m; k0 += BM) {
    __syncthreads();  // previous iteration done with Ks/Vs/Ps (and Qs visible on the first one)
    load_tile(Ks, qkv, P.qkv_ld, E + it.h * D, k0, bg.m, pos0, bg.r, seg_end);
    load_tile(Vs, qkv, P.qkv_ld, 2 * E + it.h * D, k0, bg.m, pos0, bg.r, seg_end);
    __syncthreads();
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 8
    for (int d = 0; d < D; ++d) {
      float qv[4], kv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) qv[i] = Qs[(ty * 4 + i) * LDQ + d];
#pragma unroll
      for (int j = 0; j < 4; ++j) kv[j] = Ks[(tx + 16 * j) * LDQ + d];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(qv[i], kv[j], s[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[i][j] = (k0 + tx + 16 * j < bg.m) ? s[i][j] * scale : -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int w = 8; w > 0; w >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, w));
      const float m_new = fmaxf(m_run[i], mx);  // finite: every tile holds at least one slot < m
      const float alpha = expf(m_run[i] - m_new);
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float p = expf(s[i][j] - m_new);
        rs += p;
        Ps[(ty * 4 + i) * LDP + tx + 16 * j] = p;
      }
#pragma unroll
      for (int w = 8; w > 0; w >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, w);
      l_run[i] = l_run[i] * alpha + rs;
      m_run[i] = m_new;
      o[i][0] *= alpha;
      o[i][1] *= alpha;
      o[i][2] *= alpha;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < BM; ++k) {
      const float v0 = Vs[k * LDQ + tx * 3], v1 = Vs[k * LDQ + tx * 3 + 1], v2 = Vs[k * LDQ + tx * 3 + 2];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float p = Ps[(ty * 4 + i) * LDP + k];
        o[i][0] = fmaf(p, v0, o[i][0]);
        o[i][1] = fmaf(p, v1, o[i][1]);
        o[i][2] = fmaf(p, v2, o[i][2]);
      }
    }
  }
  const int slot_h = it.h - off * bg.hpb;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int slot = q0 + ty * 4 + i;
    const int p = pos0 + slot * bg.r;
    if (slot < bg.m && p < seg_end) {
      const float inv = 1.f / l_run[i];
      T* dst = o_br + bg.o_off + ((int64_t)p * bg.hpb + slot_h) * D + tx * 3;
      dst[0] = from_float<T>(o[i][0] * inv);
      dst[1] = from_float<T>(o[i][1] * inv);
      dst[2] = from_float<T>(o[i][2] * inv);
      if (tx == 0) lse_br[bg.lse_off + (int64_t)p * bg.hpb + slot_h] = m_run[i] + logf(l_run[i]);
    }
  }
}

// key-tile-outer backward: the CTA owns 64 key slots (dK, dV in registers), streams the query tiles of its segment,
// dQ goes out through fp32 atomics; dK/dV are added to the dense gradient at the end (several branches share a row).
template <typename T>
__global__ void __launch_bounds__(256) dilated_bwd_simt_kernel(const SimtParams P, const T* __restrict__ qkv,
                                                               const T* __restrict__ dattn,
                                                               const float* __restrict__ lse,
                                                               const float* __restrict__ delta_br,
                                                               float* __restrict__ dqkv) {
  extern __shared__ float smem[];
  float* Ks = smem;
  float* Vs = Ks + BM * LDQ;
  float* Qs = Vs + BM * LDQ;
  float* dOs = Qs + BM * LDQ;
  float* Ps = dOs + BM * LDQ;
  float* dSs = Ps + BM * LDP;
  float* lse_s = dSs + BM * LDP;
  float* del_s = lse_s + BM;
  const Item it = decode_item(P, blockIdx.x);
  const BranchGeom bg = P.geo.b[it.b];
  const int H = P.geo.H, N = P.geo.N, E = H * D;
  const int off = (it.h * bg.r) / H;
  const int pos0 = it.s * bg.g + off;
  const int seg_end = min(N, (it.s + 1) * bg.g);
  const int k0 = it.tile * BM;
  const int slot_h = it.h - off * bg.hpb;
  const float scale = rsqrtf((float)D);
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;

  load_tile(Ks, qkv, P.qkv_ld, E + it.h * D, k0, bg.m, pos0, bg.r, seg_end);
  load_tile(Vs, qkv, P.qkv_ld, 2 * E + it.h * D, k0, bg.m, pos0, bg.r, seg_end);
  float dk[4][3], dv[4][3];
#pragma unroll
  for (int i = 0; i < 4; ++i) dk[i][0] = dk[i][1] = dk[i][2] = dv[i][0] = dv[i][1] = dv[i][2] = 0.f;

  for (int q0 = 0; q0 < bg.m; q0 += BM) {
    __syncthreads();
    load_tile(Qs, qkv, P.qkv_ld, it.h * D, q0, bg.m, pos0, bg.r, seg_end);
    load_tile(dOs, dattn, (int64_t)E, it.h * D, q0, bg.m, pos0, bg.r, seg_end);
    if (threadIdx.x < BM) {
      const int slot = q0 + threadIdx.x;
      const int p = pos0 + slot * bg.r;
      const bool ok = slot < bg.m && p < seg_end;
      lse_s[threadIdx.x] = ok ? lse[(int64_t)p * H + it.h] : INFINITY;  // exp(s - inf) = 0 for padded queries
      del_s[threadIdx.x] = ok ? delta_br[bg.lse_off + (int64_t)p * bg.hpb + slot_h] : 0.f;
    }
    __syncthreads();
    float s[4][4], dp[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = dp[i][j] = 0.f;
#pragma unroll 4
    for (int d = 0; d < D; ++d) {
      float qv[4], gv[4], kv[4], vv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        qv[i] = Qs[(ty * 4 + i) * LDQ + d];
        gv[i] = dOs[(ty * 4 + i) * LDQ + d];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        kv[j] = Ks[(tx + 16 * j) * LDQ + d];
        vv[j] = Vs[(tx + 16 * j) * LDQ + d];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          s[i][j] = fmaf(qv[i], kv[j], s[i][j]);
          dp[i][j] = fmaf(gv[i], vv[j], dp[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float l = lse_s[ty * 4 + i], de = del_s[ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool kok = k0 + tx + 16 * j < bg.m;
        const float p = kok ? expf(s[i][j] * scale - l) : 0.f;
        Ps[(ty * 4 + i) * LDP + tx + 16 * j] = p;
        dSs[(ty * 4 + i) * LDP + tx + 16 * j] = p * (dp[i][j] - de) * scale;
      }
    }
    __syncthreads();
    // dV[k] += P^T dO ; dK[k] += dS^T Q   (thread: key rows ty*4+i, dims tx*3+c)
#pragma unroll 4
    for (int q = 0; q < BM; ++q) {
      const float g0 = dOs[q * LDQ + tx * 3], g1 = dOs[q * LDQ + tx * 3 + 1], g2 = dOs[q * LDQ + tx * 3 + 2];
      const float x0 = Qs[q * LDQ + tx * 3], x1 = Qs[q * LDQ + tx * 3 + 1], x2 = Qs[q * LDQ + tx * 3 + 2];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float p = Ps[q * LDP + ty * 4 + i], ds = dSs[q * LDP + ty * 4 + i];
        dv[i][0] = fmaf(p, g0, dv[i][0]);
        dv[i][1] = fmaf(p, g1, dv[i][1]);
        dv[i][2] = fmaf(p, g2, dv[i][2]);
        dk[i][0] = fmaf(ds, x0, dk[i][0]);
        dk[i][1] = fmaf(ds, x1, dk[i][1]);
        dk[i][2] = fmaf(ds, x2, dk[i][2]);
      }
    }
    // dQ[q] += dS K   (thread: query rows ty*4+i, dims tx*3+c)
    float dq[4][3];
#pragma unroll
    for (int i = 0; i < 4; ++i) dq[i][0] = dq[i][1] = dq[i][2] = 0.f;
#pragma unroll 4
    for (int k = 0; k < BM; ++k) {
      const float k0v = Ks[k * LDQ + tx * 3], k1v = Ks[k * LDQ + tx * 3 + 1], k2v = Ks[k * LDQ + tx * 3 + 2];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float ds = dSs[(ty * 4 + i) * LDP + k];
        dq[i][0] = fmaf(ds, k0v, dq[i][0]);
        dq[i][1] = fmaf(ds, k1v, dq[i][1]);
        dq[i][2] = fmaf(ds, k2v, dq[i][2]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int slot = q0 + ty * 4 + i;
      const int p = pos0 + slot * bg.r;
      if (slot < bg.m && p < seg_end) {
        float* dst = dqkv + (int64_t)p * (3 * E) + it.h * D + tx * 3;
        atomicAdd(dst, dq[i][0]);
        atomicAdd(dst + 1, dq[i][1]);
        atomicAdd(dst + 2, dq[i][2]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int slot = k0 + ty * 4 + i;
    const int p = pos0 + slot * bg.r;
    if (slot < bg.m && p < seg_end) {
      float* dst = dqkv + (int64_t)p * (3 * E) + E + it.h * D + tx * 3;
      atomicAdd(dst, dk[i][0]);
      atomicAdd(dst + 1, dk[i][1]);
      atomicAdd(dst + 2, dk[i][2]);
      atomicAdd(dst + E, dv[i][0]);
      atomicAdd(dst + E + 1, dv[i][1]);
      atomicAdd(dst + E + 2, dv[i][2]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Branch merge + inner_attn_ln.  One warp per position; lane l owns head l/2, half l%2 (24 contiguous channels).
// Ownership of (position, head) by a branch is pure index arithmetic, so every load of a row -- the lse AND the 24
// output channels of all owning branches -- is issued before the first one is consumed (one memory latency per row),
// and the branch outputs stay in registers for the per-branch delta of the backward (o_br is read once).
// NB = compile-time bound on the number of branches (5 for the GigaPath configuration, MT_MAX_BRANCHES otherwise).
// ---------------------------------------------------------------------------------------------------------------------
template <typename T> struct Raw24;
template <> struct Raw24<__nv_bfloat16> {
  uint4 u[3];
  __device__ __forceinline__ void load(const __nv_bfloat16* p) {
    const uint4* s = reinterpret_cast<const uint4*>(p);
    u[0] = s[0]; u[1] = s[1]; u[2] = s[2];
  }
  __device__ __forceinline__ float get(int j) const {
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(u)[j]);
  }
};
template <> struct Raw24<float> {
  float4 u[6];
  __device__ __forceinline__ void load(const float* p) {
    const float4* s = reinterpret_cast<const float4*>(p);
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] = s[i];
  }
  __device__ __forceinline__ float get(int j) const { return reinterpret_cast<const float*>(u)[j]; }
};

template <typename T, int NB>
struct MergedRow {
  Raw24<T> o[NB];     // the 24 channels of every owning branch
  float w[NB];        // merge weight softmax_b(lse_b) (0 where the branch does not own the position)
  int slot[NB];       // compact head slot of the (position, head) in branch b
  bool own[NB];
};

template <typename T, int NB>
__device__ __forceinline__ void merge_row(const DilatedGeom& G, const T* __restrict__ o_br,
                                          const float* __restrict__ lse_br, int p, int lane, float (&acc)[24],
                                          float* lse_out, MergedRow<T, NB>& R) {
  const int h = lane >> 1, half = lane & 1;
  float l[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    l[b] = -INFINITY;
    R.own[b] = false;
    R.slot[b] = 0;
    if (b < G.nb) {
      int sl;
      R.own[b] = branch_owns(G.b[b], G.H, p, h, &sl);
      R.slot[b] = sl;
      if (R.own[b]) {
        l[b] = lse_br[G.b[b].lse_off + (int64_t)p * G.b[b].hpb + sl];
        R.o[b].load(o_br + G.b[b].o_off + ((int64_t)p * G.b[b].hpb + sl) * D + half * 24);
      }
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int b = 0; b < NB; ++b) mx = fmaxf(mx, l[b]);
  float den = 0.f;
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    R.w[b] = R.own[b] ? expf(l[b] - mx) : 0.f;
    den += R.w[b];
  }
  const float inv = den > 0.f ? 1.f / den : 0.f;  // no owning branch (needs a config without r = 1): output 0
#pragma unroll
  for (int j = 0; j < 24; ++j) acc[j] = 0.f;
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    R.w[b] *= inv;
    if (R.own[b]) {
#pragma unroll
      for (int j = 0; j < 24; ++j) acc[j] = fmaf(R.w[b], R.o[b].get(j), acc[j]);
    }
  }
  *lse_out = mx + logf(den);
}

template <typename T, int NB>
__global__ void __launch_bounds__(256, 2) merge_ln_fwd_kernel(const DilatedGeom G, const T* __restrict__ o_br,
                                                           const float* __restrict__ lse_br, T* __restrict__ attn,
                                                           float* __restrict__ lse, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, float eps,
                                                           T* __restrict__ y, float* __restrict__ mean,
                                                           float* __restrict__ rstd) {
  const int lane = threadIdx.x & 31;
  const int E = G.H * D;
  for (int p = blockIdx.x * 8 + (threadIdx.x >> 5); p < G.N; p += gridDim.x * 8) {
    float acc[24], L;
    MergedRow<T, NB> R;
    merge_row<T, NB>(G, o_br, lse_br, p, lane, acc, &L, R);
    if ((lane & 1) == 0) lse[(int64_t)p * G.H + (lane >> 1)] = L;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 24; ++j) s += acc[j];
    const float mu = warp_sum(s) / (float)E;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 24; ++j) q += (acc[j] - mu) * (acc[j] - mu);
    const float rs = rsqrtf(warp_sum(q) / (float)E + eps);
    if (lane == 0) {
      mean[p] = mu;
      rstd[p] = rs;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int col = lane * 24 + c * 8;
      float g[8], b[8], o[8], a[8];
      load8(gamma + col, g);
      load8(beta + col, b);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        a[j] = acc[c * 8 + j];
        o[j] = (a[j] - mu) * rs * g[j] + b[j];
      }
      store8(y + (int64_t)p * E + col, o);
      if (attn != nullptr) store8(attn + (int64_t)p * E + col, a);
    }
  }
}

// dattn = LN'(dy) with attn recomputed from the branch outputs; delta_b[p, h] = dattn[p, h, :] . o_b[p, h, :]
template <typename T, typename TDY, int NB>
__global__ void __launch_bounds__(256, 2) merge_ln_bwd_kernel(const DilatedGeom G, const TDY* __restrict__ dy,
                                                           const T* __restrict__ o_br,
                                                           const float* __restrict__ lse_br,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ mean,
                                                           const float* __restrict__ rstd, T* __restrict__ dattn,
                                                           float* __restrict__ delta_br) {
  const int lane = threadIdx.x & 31;
  const int E = G.H * D;
  const int half = lane & 1;
  for (int p = blockIdx.x * 8 + (threadIdx.x >> 5); p < G.N; p += gridDim.x * 8) {
    // the row of dy and the statistics do not depend on the merge: request them first
    float d[3][8];
#pragma unroll
    for (int c = 0; c < 3; ++c) load8(dy + (int64_t)p * E + lane * 24 + c * 8, d[c]);
    const float mu = mean[p], rs = rstd[p];
    float acc[24], L;
    MergedRow<T, NB> R;
    merge_row<T, NB>(G, o_br, lse_br, p, lane, acc, &L, R);
    float g[24], s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float gm[8];
      load8(gamma + lane * 24 + c * 8, gm);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[c * 8 + j] = (acc[c * 8 + j] - mu) * rs;  // xhat
        g[c * 8 + j] = d[c][j] * gm[j];
        s1 += g[c * 8 + j];
        s2 += g[c * 8 + j] * acc[c * 8 + j];
      }
    }
    const float m1 = warp_sum(s1) / (float)E, m2 = warp_sum(s2) / (float)E;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        g[c * 8 + j] = rs * (g[c * 8 + j] - m1 - acc[c * 8 + j] * m2);
        o[j] = g[c * 8 + j];
      }
      store8(dattn + (int64_t)p * E + lane * 24 + c * 8, o);
    }
    // per-branch delta against the same (rounded) dattn the attention backward will read; o_b is still in registers
#pragma unroll
    for (int j = 0; j < 24; ++j) g[j] = to_float(from_float<T>(g[j]));
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (b < G.nb) {
        float dsum = 0.f;
        if (R.own[b]) {
#pragma unroll
          for (int j = 0; j < 24; ++j) dsum = fmaf(g[j], R.o[b].get(j), dsum);
        }
        dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
        if (R.own[b] && half == 0) delta_br[G.b[b].lse_off + (int64_t)p * G.b[b].hpb + R.slot[b]] = dsum;
      }
    }
  }
}

static int make_simt_params(const mt_dilated_geometry* geom, int64_t qkv_ld, SimtParams* P) {
  int rc = make_dilated_geom(geom, &P->geo);
  if (rc) return rc;
  if (P->geo.D != D || P->geo.H != 16) {
    set_error("dilated attention kernels are built for 16 heads x 48 (got %d x %d)", P->geo.H, P->geo.D);
    return MT_E_UNSUPPORTED;
  }
  P->qkv_ld = qkv_ld;
  int total = 0;
  for (int b = 0; b < P->geo.nb; ++b) {
    P->item_prefix[b] = total;
    P->tiles[b] = (P->geo.b[b].m + BM - 1) / BM;
    total += P->geo.b[b].n_seg * P->geo.H * P->tiles[b];
  }
  P->item_prefix[P->geo.nb] = total;
  return 0;
}

int dilated_attn_fwd_simt(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc, int batch,
                          int dtype, void* o_br, float* lse_br, cudaStream_t st) {
  SimtParams P;
  int rc = make_simt_params(geom, qkv_ld, &P);
  if (rc) return rc;
  MT_REQUIRE(batch >= 1 && batch <= 65535, "dilated_attn_fwd: batch must be in [1, 65535] (got %d)", batch);
  MT_REQUIRE(batch == 1 || n_alloc >= P.geo.N, "dilated_attn_fwd: n_alloc < n_tokens");
  int64_t seq_o = 0, seq_lse = 0;
  for (int b = 0; b < P.geo.nb; ++b) {
    seq_o += (int64_t)P.geo.N * P.geo.b[b].hpb * D;
    seq_lse += (int64_t)P.geo.N * P.geo.b[b].hpb;
  }
  const int64_t seq_qkv = n_alloc * qkv_ld;
  const dim3 grid(P.item_prefix[P.geo.nb], batch);
  const size_t smem = (size_t)(3 * BM * LDQ + BM * LDP) * sizeof(float);
  if (dtype == MT_F32) {
    MT_CUDA(cudaFuncSetAttribute(dilated_fwd_simt_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dilated_fwd_simt_kernel<float><<<grid, 256, smem, st>>>(P, (const float*)qkv, (float*)o_br, lse_br, seq_qkv, seq_o,
                                                            seq_lse);
  } else {
    MT_CUDA(cudaFuncSetAttribute(dilated_fwd_simt_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dilated_fwd_simt_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>(P, (const __nv_bfloat16*)qkv, (__nv_bfloat16*)o_br,
                                                                    lse_br, seq_qkv, seq_o, seq_lse);
  }
  return check_launch("dilated_fwd_simt_kernel");
}

int dilated_attn_bwd_simt(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, const void* dattn,
                          const float* lse, const float* delta_br, int dtype, float* dqkv, cudaStream_t st) {
  SimtParams P;
  int rc = make_simt_params(geom, qkv_ld, &P);
  if (rc) return rc;
  const int total = P.item_prefix[P.geo.nb];
  const size_t smem = (size_t)(4 * BM * LDQ + 2 * BM * LDP + 2 * BM) * sizeof(float);
  if (dtype == MT_F32) {
    MT_CUDA(cudaFuncSetAttribute(dilated_bwd_simt_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dilated_bwd_simt_kernel<float><<<total, 256, smem, st>>>(P, (const float*)qkv, (const float*)dattn, lse, delta_br, dqkv);
  } else {
    MT_CUDA(cudaFuncSetAttribute(dilated_bwd_simt_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dilated_bwd_simt_kernel<__nv_bfloat16><<<total, 256, smem, st>>>(P, (const __nv_bfloat16*)qkv, (const __nv_bfloat16*)dattn, lse, delta_br, dqkv);
  }
  return check_launch("dilated_bwd_simt_kernel");
}

// implemented in dilated_sm100.cu
int dilated_attn_fwd_sm100(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc, int batch,
                           void* o_br, float* lse_br, int impl, cudaStream_t st);
int dilated_attn_bwd_sm100(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                           const void* dattn, const float* lse, const float* delta_br, float* dqkv, int impl,
                           cudaStream_t st);

}  // namespace mt

using namespace mt;

extern "C" int mt_dilated_attn_fwd_batch(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld,
                                         int64_t n_alloc, int batch, int dtype, void* o_br, float* lse_br, int impl,
                                         void* stream) {
  MT_REQUIRE(dtype == MT_F32 || dtype == MT_BF16, "dilated_attn_fwd: bad dtype %d", dtype);
  MT_REQUIRE(qkv_ld % 8 == 0, "dilated_attn_fwd: qkv row stride must be a multiple of 8 elements");
  if (impl == 0)
    return dilated_attn_fwd_simt(geom, qkv, qkv_ld, n_alloc, batch, dtype, o_br, lse_br, (cudaStream_t)stream);
  MT_REQUIRE(dtype == MT_BF16, "dilated_attn_fwd: the tcgen05 path computes in bf16");
  return dilated_attn_fwd_sm100(geom, qkv, qkv_ld, n_alloc, batch, o_br, lse_br, impl, (cudaStream_t)stream);
}

extern "C" int mt_dilated_attn_fwd(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                                   int dtype, void* o_br, float* lse_br, int impl, void* stream) {
  return mt_dilated_attn_fwd_batch(geom, qkv, qkv_ld, n_alloc, 1, dtype, o_br, lse_br, impl, stream);
}

extern "C" int mt_dilated_attn_bwd(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                                   const void* dattn, const float* lse, const float* delta_br, int dtype,
                                   float* dqkv_f32, int impl, void* stream) {
  MT_REQUIRE(dtype == MT_F32 || dtype == MT_BF16, "dilated_attn_bwd: bad dtype %d", dtype);
  MT_REQUIRE(geom != nullptr, "dilated_attn_bwd: geometry is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  MT_REQUIRE(n_alloc >= geom->n_tokens, "dilated_attn_bwd: n_alloc < n_tokens");
  MT_CUDA(cudaMemsetAsync(dqkv_f32, 0, sizeof(float) * (size_t)n_alloc * 3 * geom->n_heads * geom->head_dim, st));
  if (impl == 0) return dilated_attn_bwd_simt(geom, qkv, qkv_ld, dattn, lse, delta_br, dtype, dqkv_f32, st);
  MT_REQUIRE(dtype == MT_BF16, "dilated_attn_bwd: the tcgen05 path computes in bf16");
  return dilated_attn_bwd_sm100(geom, qkv, qkv_ld, n_alloc, dattn, lse, delta_br, dqkv_f32, impl, st);
}

extern "C" int mt_dilated_merge_ln_fwd(const mt_dilated_geometry* geom, const void* o_br, const float* lse_br,
                                       int dtype, void* attn, float* lse, const float* gamma, const float* beta,
                                       float eps, void* y, float* mean, float* rstd, void* stream) {
  DilatedGeom G;
  int rc = make_dilated_geom(geom, &G);
  if (rc) return rc;
  MT_REQUIRE(G.H == 16 && G.D == D, "merge_ln: built for 16 heads x 48");
  cudaStream_t st = (cudaStream_t)stream;
  int grid = (G.N + 7) / 8;
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  using bf = __nv_bfloat16;
#define MT_MERGE_FWD(T, NB) \
  merge_ln_fwd_kernel<T, NB><<<grid, 256, 0, st>>>(G, (const T*)o_br, lse_br, (T*)attn, lse, gamma, beta, eps, (T*)y, mean, rstd)
  if (dtype == MT_F32) {
    if (G.nb <= 5) MT_MERGE_FWD(float, 5); else MT_MERGE_FWD(float, MT_MAX_BRANCHES);
  } else {
    if (G.nb <= 5) MT_MERGE_FWD(bf, 5); else MT_MERGE_FWD(bf, MT_MAX_BRANCHES);
  }
#undef MT_MERGE_FWD
  return check_launch("merge_ln_fwd_kernel");
}

extern "C" int mt_dilated_merge_ln_bwd(const mt_dilated_geometry* geom, const void* dy, int dy_dtype,
                                       const void* o_br, const float* lse_br, const float* gamma, const float* mean,
                                       const float* rstd, int dtype, void* dattn, float* delta_br, void* stream) {
  DilatedGeom G;
  int rc = make_dilated_geom(geom, &G);
  if (rc) return rc;
  MT_REQUIRE(G.H == 16 && G.D == D, "merge_ln: built for 16 heads x 48");
  cudaStream_t st = (cudaStream_t)stream;
  int grid = (G.N + 7) / 8;
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  using bf = __nv_bfloat16;
#define MT_MERGE_BWD(T, TDY, NB)                                                                                   \
  merge_ln_bwd_kernel<T, TDY, NB><<<grid, 256, 0, st>>>(G, (const TDY*)dy, (const T*)o_br, lse_br, gamma, mean, rstd, \
                                                        (T*)dattn, delta_br)
  if (dtype == MT_F32 && dy_dtype == MT_F32) {
    if (G.nb <= 5) MT_MERGE_BWD(float, float, 5); else MT_MERGE_BWD(float, float, MT_MAX_BRANCHES);
  } else if (dtype == MT_BF16 && dy_dtype == MT_BF16) {
    if (G.nb <= 5) MT_MERGE_BWD(bf, bf, 5); else MT_MERGE_BWD(bf, bf, MT_MAX_BRANCHES);
  } else if (dtype == MT_BF16 && dy_dtype == MT_F32) {
    if (G.nb <= 5) MT_MERGE_BWD(bf, float, 5); else MT_MERGE_BWD(bf, float, MT_MAX_BRANCHES);
  } else {
    set_error("merge_ln_bwd: unsupported dtype combination (%d, dy %d)", dtype, dy_dtype);
    return MT_E_UNSUPPORTED;
  }
#undef MT_MERGE_BWD
  return check_launch("merge_ln_bwd_kernel");
}
