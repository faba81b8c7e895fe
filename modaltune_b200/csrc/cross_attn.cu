// Injector / Extractor cross-attention core: softmax(q k^T / sqrt(16)) v with 12 heads x 16 in the 192-d compressed
// space (models/vitadapter/adapter_modules.py:225-229 -> nn.MultiheadAttention).  The reference materialises the
// [12, Lq, Lk] probabilities (and their head average, which it discards); here nothing of that size is ever written.
//
//   Injector  (Lq = tiles ~1e4, Lk = modal tokens ~66): one thread per query, K/V tiles broadcast from shared memory.
//   Extractor (Lq ~66, Lk = tiles ~1e4): split-K over the keys (grid.z), partial (m, l, acc) per split, LSE combine.
// Backward is two kernels, each accumulating in registers along its own loop (plain stores when the loop is not split,
// 16-byte fp32 reduce-adds when it is):
//   dq-kernel (thread per query, loop over keys) and dkv-kernel (thread per key, loop over queries).
#include "mt_common.cuh"

namespace mt {

static constexpr int HD = 16;
static constexpr int XT = 128;  // threads per CTA = rows (queries or keys) per CTA
static constexpr int XC = 64;   // staged rows per chunk

// row strides (elements): q | k and v | o and d_o | dq | dk and dv.  The Extractor hands k / v (and takes dk / dv) as the
// two halves of one [L, 384] projection buffer, so no split / concat copies exist on either side of the kernels.
struct Strides {
  int64_t q, kv, o, dq, dkv;
};

// Two fp32 FMAs in one instruction (FFMA2, new with sm_100): the kernels below are bound by instruction issue (one
// shared-memory operand per four FMAs plus the exponentials), so halving the FMA instruction count is a direct win.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t ra = *reinterpret_cast<uint64_t*>(&a), rb = *reinterpret_cast<uint64_t*>(&b);
  uint64_t rc = *reinterpret_cast<uint64_t*>(&c), rd;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
}
// dot product of a register row (8 float2) with a 16-float shared-memory row, two accumulator chains
__device__ __forceinline__ float dot16(const float2 (&a)[HD / 2], const float* __restrict__ row) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
  float2 d0 = make_float2(0.f, 0.f), d1 = make_float2(0.f, 0.f);
#pragma unroll
  for (int c = 0; c < HD / 4; ++c) {
    const float4 k = r4[c];
    d0 = ffma2(a[2 * c], make_float2(k.x, k.y), d0);
    d1 = ffma2(a[2 * c + 1], make_float2(k.z, k.w), d1);
  }
  return (d0.x + d1.x) + (d0.y + d1.y);
}
// register-register dot product in EXACTLY the order of dot16: delta = dO.o must equal dO.v bit for bit when a query
// has a single key (p = 1, o = v), so that dS is exactly zero there
__device__ __forceinline__ float dot16v(const float (&a)[HD], const float (&b)[HD]) {
  float2 d0 = make_float2(0.f, 0.f), d1 = make_float2(0.f, 0.f);
#pragma unroll
  for (int c = 0; c < HD / 4; ++c) {
    d0 = ffma2(make_float2(a[4 * c], a[4 * c + 1]), make_float2(b[4 * c], b[4 * c + 1]), d0);
    d1 = ffma2(make_float2(a[4 * c + 2], a[4 * c + 3]), make_float2(b[4 * c + 2], b[4 * c + 3]), d1);
  }
  return (d0.x + d1.x) + (d0.y + d1.y);
}
// acc += w * row
__device__ __forceinline__ void axpy16(float2 (&acc)[HD / 2], float w, const float* __restrict__ row) {
  const float4* r4 = reinterpret_cast<const float4*>(row);
  const float2 w2 = make_float2(w, w);
#pragma unroll
  for (int c = 0; c < HD / 4; ++c) {
    const float4 k = r4[c];
    acc[2 * c] = ffma2(w2, make_float2(k.x, k.y), acc[2 * c]);
    acc[2 * c + 1] = ffma2(w2, make_float2(k.z, k.w), acc[2 * c + 1]);
  }
}
// acc += w * r (register row)
__device__ __forceinline__ void axpy16r(float2 (&acc)[HD / 2], float w, const float2 (&r)[HD / 2]) {
  const float2 w2 = make_float2(w, w);
#pragma unroll
  for (int c = 0; c < HD / 2; ++c) acc[c] = ffma2(w2, r[c], acc[c]);
}
__device__ __forceinline__ void to_pairs(const float (&v)[HD], float scale, float2 (&o)[HD / 2]) {
#pragma unroll
  for (int c = 0; c < HD / 2; ++c) o[c] = make_float2(v[2 * c] * scale, v[2 * c + 1] * scale);
}

template <typename T>
__device__ __forceinline__ void load16(const T* p, float (&v)[HD]) {
  float a[8], b[8];
  load8(p, a);
  load8(p + 8, b);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    v[j] = a[j];
    v[8 + j] = b[j];
  }
}

// stage rows [r0, r0+XC) of a [L, heads*HD] matrix (head h) into smem [XC][HD] (fp32); rows >= lim zero-filled
template <typename T>
__device__ __forceinline__ void stage16(float* dst, const T* __restrict__ src, int64_t ld, int h, int64_t r0,
                                        int64_t lim) {
  // XC rows x 2 chunks of 8 = 128 chunk loads = one per thread
  const int row = threadIdx.x >> 1, ch = threadIdx.x & 1;
  float v[8];
  if (r0 + row < lim) {
    load8(src + (r0 + row) * ld + h * HD + ch * 8, v);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) dst[row * HD + ch * 8 + j] = v[j];
}

template <typename T>
__global__ void __launch_bounds__(XT) cross_fwd_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                       const T* __restrict__ v, T* __restrict__ o,
                                                       float* __restrict__ lse, float* __restrict__ ws, int64_t lq,
                                                       int64_t lk, int heads, int64_t keys_per_split, Strides sd) {
  __shared__ float Ks[XC * HD], Vs[XC * HD];
  const int h = blockIdx.y, split = blockIdx.z, nsplit = gridDim.z;
  const int64_t qi = (int64_t)blockIdx.x * XT + threadIdx.x;
  const bool live = qi < lq;
  float qv[HD];
  if (live) load16(q + qi * sd.q + h * HD, qv);
  else
#pragma unroll
    for (int j = 0; j < HD; ++j) qv[j] = 0.f;
  float2 q2[HD / 2], acc2[HD / 2];
  to_pairs(qv, 0.25f, q2);  // 1/sqrt(16)
  float m = -INFINITY, l = 0.f;
#pragma unroll
  for (int j = 0; j < HD / 2; ++j) acc2[j] = make_float2(0.f, 0.f);
  const int64_t kbeg = split * keys_per_split, kend = min(lk, kbeg + keys_per_split);
  for (int64_t k0 = kbeg; k0 < kend; k0 += XC) {
    __syncthreads();
    stage16(Ks, k, sd.kv, h, k0, kend);
    stage16(Vs, v, sd.kv, h, k0, kend);
    __syncthreads();
    const int cnt = (int)min((int64_t)XC, kend - k0);
    for (int j0 = 0; j0 < cnt; j0 += 8) {
      float s[8], mx = m;
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const float d = dot16(q2, Ks + (j0 + jj) * HD);
        s[jj] = (j0 + jj < cnt) ? d : -INFINITY;
        mx = fmaxf(mx, s[jj]);
      }
      const float alpha = expf(m - mx);
      l *= alpha;
#pragma unroll
      for (int e = 0; e < HD / 2; ++e) acc2[e] = make_float2(acc2[e].x * alpha, acc2[e].y * alpha);
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const float p = expf(s[jj] - mx);
        l += p;
        axpy16(acc2, p, Vs + (j0 + jj) * HD);
      }
      m = mx;
    }
  }
  if (!live) return;
  float acc[HD];
#pragma unroll
  for (int e = 0; e < HD / 2; ++e) {
    acc[2 * e] = acc2[e].x;
    acc[2 * e + 1] = acc2[e].y;
  }
  if (nsplit == 1) {
    const float inv = 1.f / l;
    float out[HD];
#pragma unroll
    for (int e = 0; e < HD; ++e) out[e] = acc[e] * inv;
    float a[8], b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      a[j] = out[j];
      b[j] = out[8 + j];
    }
    store8(o + qi * sd.o + h * HD, a);
    store8(o + qi * sd.o + h * HD + 8, b);
    lse[qi * heads + h] = m + logf(l);
  } else {
    float* w = ws + (((int64_t)split * lq + qi) * heads + h) * (HD + 2);
    w[0] = m;
    w[1] = l;
#pragma unroll
    for (int e = 0; e < HD; ++e) w[2 + e] = acc[e];
  }
}

// one WARP per (query, head): the lanes take the splits (a serial loop over up to 128 partials per thread was the
// longest kernel of the Extractor forward), then a warp reduction per output element
template <typename T>
__global__ void __launch_bounds__(128) cross_combine_kernel(const float* __restrict__ ws, T* __restrict__ o,
                                                            float* __restrict__ lse, int64_t lq, int heads,
                                                            int nsplit, int64_t ldo) {
  const int64_t idx = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (idx >= lq * heads) return;
  float m = -INFINITY;
  for (int s = lane; s < nsplit; s += 32) m = fmaxf(m, ws[((int64_t)s * lq * heads + idx) * (HD + 2)]);
  m = warp_max(m);
  float l = 0.f, acc[HD];
#pragma unroll
  for (int e = 0; e < HD; ++e) acc[e] = 0.f;
  for (int s = lane; s < nsplit; s += 32) {
    const float* w = ws + ((int64_t)s * lq * heads + idx) * (HD + 2);
    const float2 ml = *reinterpret_cast<const float2*>(w);
    const float f = (ml.x == -INFINITY) ? 0.f : expf(ml.x - m);
    l = fmaf(f, ml.y, l);
#pragma unroll
    for (int e = 0; e < HD; e += 2) {
      const float2 a = *reinterpret_cast<const float2*>(w + 2 + e);
      acc[e] = fmaf(f, a.x, acc[e]);
      acc[e + 1] = fmaf(f, a.y, acc[e + 1]);
    }
  }
  l = warp_sum(l);
#pragma unroll
  for (int e = 0; e < HD; ++e) acc[e] = warp_sum(acc[e]);
  const float inv = 1.f / l;
  const int64_t qi = idx / heads;
  const int h = (int)(idx % heads);
  if (lane < HD) {
    float val = 0.f;
#pragma unroll
    for (int e = 0; e < HD; ++e) val = (lane == e) ? acc[e] : val;
    o[qi * ldo + h * HD + lane] = from_float<T>(val * inv);
  }
  if (lane == 0) lse[idx] = m + logf(l);
}

// dq[qi] += sum_k exp(s - lse) * (dO.v_k - delta) * k_k / 4
template <typename T>
__global__ void __launch_bounds__(XT) cross_bwd_dq_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                          const T* __restrict__ v, const T* __restrict__ o,
                                                          const T* __restrict__ d_o, const float* __restrict__ lse,
                                                          float* __restrict__ dq, int64_t lq, int64_t lk, int heads,
                                                          int64_t keys_per_split, Strides sd) {
  __shared__ float Ks[XC * HD], Vs[XC * HD];
  const int h = blockIdx.y, split = blockIdx.z;
  const int64_t qi = (int64_t)blockIdx.x * XT + threadIdx.x;
  const bool live = qi < lq;
  float qv[HD], gv[HD], acc[HD], delta = 0.f, L = INFINITY;
#pragma unroll
  for (int j = 0; j < HD; ++j) qv[j] = gv[j] = acc[j] = 0.f;
  if (live) {
    float ov[HD];
    load16(q + qi * sd.q + h * HD, qv);
    load16(d_o + qi * sd.o + h * HD, gv);
    load16(o + qi * sd.o + h * HD, ov);
    delta = dot16v(gv, ov);
    L = lse[qi * heads + h];
  }
  float2 q2[HD / 2], g2[HD / 2], acc2[HD / 2];
  to_pairs(qv, 0.25f, q2);
  to_pairs(gv, 1.f, g2);
#pragma unroll
  for (int j = 0; j < HD / 2; ++j) acc2[j] = make_float2(0.f, 0.f);
  const int64_t kbeg = split * keys_per_split, kend = min(lk, kbeg + keys_per_split);
  for (int64_t k0 = kbeg; k0 < kend; k0 += XC) {
    __syncthreads();
    stage16(Ks, k, sd.kv, h, k0, kend);
    stage16(Vs, v, sd.kv, h, k0, kend);
    __syncthreads();
    const int cnt = (int)min((int64_t)XC, kend - k0);
#pragma unroll 2
    for (int j = 0; j < cnt; ++j) {
      const float s = dot16(q2, Ks + j * HD), dp = dot16(g2, Vs + j * HD);
      const float ds = expf(s - L) * (dp - delta) * 0.25f;
      axpy16(acc2, ds, Ks + j * HD);
    }
  }
#pragma unroll
  for (int e = 0; e < HD / 2; ++e) {
    acc[2 * e] = acc2[e].x;
    acc[2 * e + 1] = acc2[e].y;
  }
  if (live) {
    float* dst = dq + qi * sd.dq + h * HD;
    if (gridDim.z == 1) {   // the only contribution to this row: plain 16-byte stores, no zero fill needed
#pragma unroll
      for (int e = 0; e < HD; e += 4)
        *reinterpret_cast<float4*>(dst + e) = make_float4(acc[e], acc[e + 1], acc[e + 2], acc[e + 3]);
    } else {
#pragma unroll
      for (int e = 0; e < HD; e += 4)
        atomicAdd(reinterpret_cast<float4*>(dst + e), make_float4(acc[e], acc[e + 1], acc[e + 2], acc[e + 3]));
    }
  }
}

// thread per key: dv[k] += sum_q p dO_q ; dk[k] += sum_q p (dO_q.v_k - delta_q) q_q / 4
template <typename T>
__global__ void __launch_bounds__(XT) cross_bwd_dkv_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                           const T* __restrict__ v, const T* __restrict__ o,
                                                           const T* __restrict__ d_o, const float* __restrict__ lse,
                                                           float* __restrict__ dk, float* __restrict__ dv, int64_t lq,
                                                           int64_t lk, int heads, int64_t q_per_split, Strides sd) {
  __shared__ float Qs[XC * HD], Gs[XC * HD], Ls[XC], Ds[XC];
  const int h = blockIdx.y, split = blockIdx.z;
  const int64_t ki = (int64_t)blockIdx.x * XT + threadIdx.x;
  const bool live = ki < lk;
  float kv[HD], vv[HD], dka[HD], dva[HD];
#pragma unroll
  for (int j = 0; j < HD; ++j) kv[j] = vv[j] = dka[j] = dva[j] = 0.f;
  if (live) {
    load16(k + ki * sd.kv + h * HD, kv);
    load16(v + ki * sd.kv + h * HD, vv);
  }
  float2 k2[HD / 2], v2[HD / 2], dk2[HD / 2], dv2[HD / 2];
  to_pairs(kv, 1.f, k2);
  to_pairs(vv, 1.f, v2);
#pragma unroll
  for (int j = 0; j < HD / 2; ++j) dk2[j] = dv2[j] = make_float2(0.f, 0.f);
  const int64_t qbeg = split * q_per_split, qend = min(lq, qbeg + q_per_split);
  for (int64_t q0 = qbeg; q0 < qend; q0 += XC) {
    __syncthreads();
    if (threadIdx.x < XC) {
      const int64_t qi = q0 + threadIdx.x;
      float a[HD], g[HD], ov[HD], de = 0.f;
      if (qi < qend) {
        load16(q + qi * sd.q + h * HD, a);
        load16(d_o + qi * sd.o + h * HD, g);
        load16(o + qi * sd.o + h * HD, ov);
        de = dot16v(g, ov);
        Ls[threadIdx.x] = lse[qi * heads + h];
      } else {
#pragma unroll
        for (int e = 0; e < HD; ++e) a[e] = g[e] = 0.f;
        Ls[threadIdx.x] = INFINITY;
      }
      Ds[threadIdx.x] = de;
#pragma unroll
      for (int e = 0; e < HD; ++e) {
        Qs[threadIdx.x * HD + e] = a[e] * 0.25f;
        Gs[threadIdx.x * HD + e] = g[e];
      }
    }
    __syncthreads();
    const int cnt = (int)min((int64_t)XC, qend - q0);
#pragma unroll 2
    for (int j = 0; j < cnt; ++j) {
      const float s = dot16(k2, Qs + j * HD), dp = dot16(v2, Gs + j * HD);
      const float p = expf(s - Ls[j]);
      const float ds = p * (dp - Ds[j]);
      axpy16(dv2, p, Gs + j * HD);
      axpy16(dk2, ds, Qs + j * HD);  // Qs already carries the 1/4
    }
  }
#pragma unroll
  for (int e = 0; e < HD / 2; ++e) {
    dka[2 * e] = dk2[e].x;
    dka[2 * e + 1] = dk2[e].y;
    dva[2 * e] = dv2[e].x;
    dva[2 * e + 1] = dv2[e].y;
  }
  if (live) {
    float* dstk = dk + ki * sd.dkv + h * HD;
    float* dstv = dv + ki * sd.dkv + h * HD;
    if (gridDim.z == 1) {
#pragma unroll
      for (int e = 0; e < HD; e += 4) {
        *reinterpret_cast<float4*>(dstk + e) = make_float4(dka[e], dka[e + 1], dka[e + 2], dka[e + 3]);
        *reinterpret_cast<float4*>(dstv + e) = make_float4(dva[e], dva[e + 1], dva[e + 2], dva[e + 3]);
      }
    } else {
#pragma unroll
      for (int e = 0; e < HD; e += 4) {
        atomicAdd(reinterpret_cast<float4*>(dstk + e), make_float4(dka[e], dka[e + 1], dka[e + 2], dka[e + 3]));
        atomicAdd(reinterpret_cast<float4*>(dstv + e), make_float4(dva[e], dva[e + 1], dva[e + 2], dva[e + 3]));
      }
    }
  }
}


// =====================================================================================================================
// Tensor-core variant (impl 1, fp32 tensors, TF32 operands / fp32 accumulation): mma.sync.m16n8k8 with the 16-wide head
// as two k-steps.  One warp owns 16 rows of the M side (queries in the forward / dq kernels, keys in the dkv kernel) and
// loops over chunks of up to 72 rows of the other side staged in shared memory as TF32 bit patterns (row stride 20
// words: both fragment access patterns below are bank-conflict free).  Probabilities / dS go straight from the
// accumulator registers into the A operand of the next MMA: the k-index of that MMA is a PERMUTATION of the 8 chunk rows
// (k = t <-> row 2t, k = t + 4 <-> row 2t + 1), which the B-fragment loads apply as well, so no shuffle is needed.
// These are 0.3 % of the step's FLOPs and bound by latency / HBM, not by tensor throughput: mma.sync (no TMEM, no
// 128-row tiles) is the right tool for a 16-wide head.  SIMT kernels above: 35 / 42 / 51 us per launch at 10k tiles.
// =====================================================================================================================
static constexpr int TC = 72;    // rows of the streamed side per chunk (9 MMA n-tiles)
static constexpr int TNT = TC / 8;
static constexpr int TS = 20;    // shared-memory row stride in words
static constexpr float kLog2e = 1.4426950408889634f;
static constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ uint32_t tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
// A fragments (two k-steps) of rows r_lo = row0 + g, r_hi = r_lo + 8 of head h of a [rows, ld] matrix: raw loads (issued
// early, no dependent instruction), converted to scaled TF32 by cvt_a_frag right before the first MMA
__device__ __forceinline__ void load_a_raw(float (&a)[2][4], const float* __restrict__ src, int64_t ld, int h,
                                           int64_t r_lo, int64_t lim, int t) {
  const int64_t r_hi = r_lo + 8;
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int c = h * HD + 8 * s + t;
    a[s][0] = r_lo < lim ? src[r_lo * ld + c] : 0.f;
    a[s][1] = r_hi < lim ? src[r_hi * ld + c] : 0.f;
    a[s][2] = r_lo < lim ? src[r_lo * ld + c + 4] : 0.f;
    a[s][3] = r_hi < lim ? src[r_hi * ld + c + 4] : 0.f;
  }
}
__device__ __forceinline__ void cvt_a_frag(uint32_t (&a)[2][4], const float (&raw)[2][4], float scale) {
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int i = 0; i < 4; ++i) a[s][i] = tf32(raw[s][i] * scale);
}
// stage rows [r0, r0 + TC) (head h) of TWO [rows, ld] fp32 matrices into smem [TC][TS] as TF32; rows >= lim = 0.  All
// loads of a pass are issued before the first conversion (three float4 per matrix and thread in flight): the kernels are
// latency bound, one dependent load -> convert -> store chain per iteration was a third of a CTA's life.
__device__ __forceinline__ void stage2_tf32(uint32_t* dst_a, uint32_t* dst_b, const float* __restrict__ src_a,
                                            const float* __restrict__ src_b, int64_t ld, int h, int64_t r0, int64_t lim) {
  constexpr int U = 3;
  for (int base = threadIdx.x; base < TC * 4; base += U * blockDim.x) {
    float4 va[U], vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int idx = base + u * blockDim.x, row = idx >> 2, c4 = idx & 3;
      va[u] = vb[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (idx < TC * 4 && r0 + row < lim) {
        const int64_t off = (r0 + row) * ld + h * HD + c4 * 4;
        va[u] = *reinterpret_cast<const float4*>(src_a + off);
        vb[u] = *reinterpret_cast<const float4*>(src_b + off);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int idx = base + u * blockDim.x, row = idx >> 2, c4 = idx & 3;
      if (idx < TC * 4) {
        *reinterpret_cast<uint4*>(dst_a + row * TS + c4 * 4) = make_uint4(tf32(va[u].x), tf32(va[u].y), tf32(va[u].z), tf32(va[u].w));
        *reinterpret_cast<uint4*>(dst_b + row * TS + c4 * 4) = make_uint4(tf32(vb[u].x), tf32(vb[u].y), tf32(vb[u].z), tf32(vb[u].w));
      }
    }
  }
}
// S tile j (16 x 8) = A (16 x 16, two k-steps) . B^T with B rows 8j .. 8j+7 staged in `sm`
__device__ __forceinline__ void mma_rows(float (&d)[4], const uint32_t (&a)[2][4], const uint32_t* sm, int j, int g, int t) {
  const uint32_t* r = sm + (8 * j + g) * TS + t;
  mma_tf32(d, a[0], r[0], r[4]);
  mma_tf32(d, a[1], r[8], r[12]);
}
// acc (16 x 16, two n-tiles) += P (16 x 8 chunk rows, accumulator registers) . B with B rows 8j .. 8j+7 staged in `sm`
__device__ __forceinline__ void mma_acc(float (&acc)[2][4], const float (&p)[4], const uint32_t* sm, int j, int g, int t) {
  const uint32_t a[4] = {tf32(p[0]), tf32(p[2]), tf32(p[1]), tf32(p[3])};
  const uint32_t* r0 = sm + (8 * j + 2 * t) * TS + g;
  mma_tf32(acc[0], a, r0[0], r0[TS]);
  mma_tf32(acc[1], a, r0[8], r0[TS + 8]);
}

// forward: warp = 16 queries of head blockIdx.y, keys [split range) in chunks of TC
__global__ void __launch_bounds__(256, 4) cross_fwd_tc_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                           const float* __restrict__ v, float* __restrict__ o,
                                                           float* __restrict__ lse, float* __restrict__ ws, int64_t lq,
                                                           int64_t lk, int heads, int64_t keys_per_split, Strides sd) {
  __shared__ __align__(16) uint32_t Ks[TC * TS], Vs[TC * TS];
  const int h = blockIdx.y, split = blockIdx.z, nsplit = gridDim.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int64_t r_lo = ((int64_t)blockIdx.x * (blockDim.x >> 5) + warp) * 16 + g, r_hi = r_lo + 8;
  uint32_t qa[2][4];
  float qraw[2][4];
  load_a_raw(qraw, q, sd.q, h, r_lo, lq, t);
  float m_lo = -INFINITY, m_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f, acc[2][4] = {};
  const int64_t kbeg = split * keys_per_split, kend = min(lk, kbeg + keys_per_split);
  for (int64_t k0 = kbeg; k0 < kend; k0 += TC) {
    __syncthreads();
    stage2_tf32(Ks, Vs, k, v, sd.kv, h, k0, kend);
    if (k0 == kbeg) cvt_a_frag(qa, qraw, 0.25f * kLog2e);   // scores in the log2 domain
    __syncthreads();
    const int cnt = (int)min((int64_t)TC, kend - k0), nt = (cnt + 7) >> 3;
    // pass 1: row maxima only.  The score MMAs are issued again in pass 2 instead of keeping nine accumulator tiles
    // alive (tensor work is free here; 60 registers less is twice the resident warps, and the kernel is latency bound)
    float mx_lo = m_lo, mx_hi = m_hi;
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      if (j < nt) {
        float s[4] = {};
        mma_rows(s, qa, Ks, j, g, t);
        const bool dead0 = 8 * j + 2 * t >= cnt, dead1 = 8 * j + 2 * t + 1 >= cnt;
        mx_lo = fmaxf(mx_lo, fmaxf(dead0 ? -INFINITY : s[0], dead1 ? -INFINITY : s[1]));
        mx_hi = fmaxf(mx_hi, fmaxf(dead0 ? -INFINITY : s[2], dead1 ? -INFINITY : s[3]));
      }
    }
    mx_lo = quad_max(mx_lo);
    mx_hi = quad_max(mx_hi);
    const float a_lo = ex2(m_lo - mx_lo), a_hi = ex2(m_hi - mx_hi);   // first chunk: ex2(-inf) = 0
    m_lo = mx_lo;
    m_hi = mx_hi;
    l_lo *= a_lo;
    l_hi *= a_hi;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      acc[d][0] *= a_lo;
      acc[d][1] *= a_lo;
      acc[d][2] *= a_hi;
      acc[d][3] *= a_hi;
    }
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      if (j < nt) {
        float s[4] = {};
        mma_rows(s, qa, Ks, j, g, t);
        const bool dead0 = 8 * j + 2 * t >= cnt, dead1 = 8 * j + 2 * t + 1 >= cnt;
        float p[4] = {dead0 ? 0.f : ex2(s[0] - m_lo), dead1 ? 0.f : ex2(s[1] - m_lo),
                      dead0 ? 0.f : ex2(s[2] - m_hi), dead1 ? 0.f : ex2(s[3] - m_hi)};
        l_lo += p[0] + p[1];
        l_hi += p[2] + p[3];
        mma_acc(acc, p, Vs, j, g, t);
      }
    }
  }
  l_lo = quad_sum(l_lo);
  l_hi = quad_sum(l_hi);
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int64_t r = half ? r_hi : r_lo;
    if (r >= lq) continue;
    const float m = half ? m_hi : m_lo, l = half ? l_hi : l_lo;
    if (nsplit == 1) {
      const float inv = 1.f / l;
#pragma unroll
      for (int d = 0; d < 2; ++d)
        *reinterpret_cast<float2*>(o + r * sd.o + h * HD + 8 * d + 2 * t) =
            make_float2(acc[d][2 * half] * inv, acc[d][2 * half + 1] * inv);
      if (t == 0) lse[r * heads + h] = (m + log2f(l)) * kLn2;
    } else {   // partial (m, l, acc) in natural-log units for cross_combine_kernel
      float* w = ws + (((int64_t)split * lq + r) * heads + h) * (HD + 2);
      if (t == 0) *reinterpret_cast<float2*>(w) = make_float2(m * kLn2, l);
#pragma unroll
      for (int d = 0; d < 2; ++d)
        *reinterpret_cast<float2*>(w + 2 + 8 * d + 2 * t) = make_float2(acc[d][2 * half], acc[d][2 * half + 1]);
    }
  }
}

// dq[q] (+)= sum_k P (dO.v_k - delta) k_k / 4 : warp = 16 queries, keys streamed
struct BwdSmem {   // the two roles of cross_bwd_tc_kernel use the same shared memory
  uint32_t a[TC * TS], b[TC * TS];
  float ls[TC], ds[TC];
};
__device__ __forceinline__ void cross_bwd_dq_tc(BwdSmem& sm, int bx, int h, int split, int nsplit,
                                                const float* __restrict__ q, const float* __restrict__ k,
                                                const float* __restrict__ v, const float* __restrict__ o,
                                                const float* __restrict__ d_o, const float* __restrict__ lse,
                                                float* __restrict__ dq, int64_t lq, int64_t lk, int heads,
                                                int64_t keys_per_split, const Strides& sd, float* __restrict__ part) {
  uint32_t* Ks = sm.a;
  uint32_t* Vs = sm.b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int64_t r_lo = ((int64_t)bx * (blockDim.x >> 5) + warp) * 16 + g, r_hi = r_lo + 8;
  uint32_t qa[2][4], ga[2][4];
  float qraw[2][4], graw[2][4], oraw[2][4];
  load_a_raw(qraw, q, sd.q, h, r_lo, lq, t);
  load_a_raw(graw, d_o, sd.o, h, r_lo, lq, t);
  load_a_raw(oraw, o, sd.o, h, r_lo, lq, t);
  float L_lo = r_lo < lq ? lse[r_lo * heads + h] : INFINITY;
  float L_hi = r_hi < lq ? lse[r_hi * heads + h] : INFINITY;
  float de_lo = 0.f, de_hi = 0.f;   // delta = dO . o over the 16 head columns (fp32, unrounded operands)
  float acc[2][4] = {};
  const int64_t kbeg = split * keys_per_split, kend = min(lk, kbeg + keys_per_split);
  for (int64_t k0 = kbeg; k0 < kend; k0 += TC) {
    __syncthreads();
    stage2_tf32(Ks, Vs, k, v, sd.kv, h, k0, kend);
    if (k0 == kbeg) {   // first use of the row operands: everything above was loads only
      cvt_a_frag(qa, qraw, 0.25f * kLog2e);
      cvt_a_frag(ga, graw, 1.f);
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        de_lo = fmaf(graw[s][0], oraw[s][0], fmaf(graw[s][2], oraw[s][2], de_lo));
        de_hi = fmaf(graw[s][1], oraw[s][1], fmaf(graw[s][3], oraw[s][3], de_hi));
      }
      de_lo = quad_sum(de_lo);
      de_hi = quad_sum(de_hi);
      L_lo *= kLog2e;
      L_hi *= kLog2e;
    }
    __syncthreads();
    const int cnt = (int)min((int64_t)TC, kend - k0), nt = (cnt + 7) >> 3;
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      if (j < nt) {
        float s[4] = {}, dp[4] = {};
        mma_rows(s, qa, Ks, j, g, t);
        mma_rows(dp, ga, Vs, j, g, t);
        const bool dead0 = 8 * j + 2 * t >= cnt, dead1 = 8 * j + 2 * t + 1 >= cnt;
        float ds[4];
        ds[0] = dead0 ? 0.f : ex2(s[0] - L_lo) * (dp[0] - de_lo);
        ds[1] = dead1 ? 0.f : ex2(s[1] - L_lo) * (dp[1] - de_lo);
        ds[2] = dead0 ? 0.f : ex2(s[2] - L_hi) * (dp[2] - de_hi);
        ds[3] = dead1 ? 0.f : ex2(s[3] - L_hi) * (dp[3] - de_hi);
        mma_acc(acc, ds, Ks, j, g, t);
      }
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int64_t r = half ? r_hi : r_lo;
    if (r >= lq) continue;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      float2* dst = reinterpret_cast<float2*>(dq + r * sd.dq + h * HD + 8 * d + 2 * t);
      const float2 val = make_float2(acc[d][2 * half] * 0.25f, acc[d][2 * half + 1] * 0.25f);
      if (nsplit == 1) *dst = val;
      else if (part != nullptr)   // deterministic: [split][lq][heads * HD], summed in split order by cross_split_sum_kernel
        *reinterpret_cast<float2*>(part + ((int64_t)split * lq + r) * heads * HD + h * HD + 8 * d + 2 * t) = val;
      else atomicAdd(dst, val);
    }
  }
}

// dv[k] (+)= sum_q P dO_q ; dk[k] (+)= sum_q P (dO_q.v_k - delta_q) q_q / 4 : warp = 16 keys, queries streamed.
// Transposed tiles: S^T = K Q^T with the keys on the MMA rows, the per-query lse / delta per accumulator column.
__device__ __forceinline__ void cross_bwd_dkv_tc(BwdSmem& sm, int bx, int h, int split, int nsplit,
                                                 const float* __restrict__ q, const float* __restrict__ k,
                                                 const float* __restrict__ v, const float* __restrict__ o,
                                                 const float* __restrict__ d_o, const float* __restrict__ lse,
                                                 float* __restrict__ dk, float* __restrict__ dv, int64_t lq,
                                                 int64_t lk, int heads, int64_t q_per_split, const Strides& sd,
                                                 float* __restrict__ part) {
  uint32_t* Qs = sm.a;
  uint32_t* Gs = sm.b;
  float* Ls = sm.ls;
  float* Ds = sm.ds;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int64_t r_lo = ((int64_t)bx * (blockDim.x >> 5) + warp) * 16 + g, r_hi = r_lo + 8;
  uint32_t ka[2][4], va[2][4];
  float kraw[2][4], vraw[2][4];
  load_a_raw(kraw, k, sd.kv, h, r_lo, lk, t);
  load_a_raw(vraw, v, sd.kv, h, r_lo, lk, t);
  float dka[2][4] = {}, dva[2][4] = {};
  const int64_t qbeg = split * q_per_split, qend = min(lq, qbeg + q_per_split);
  for (int64_t q0 = qbeg; q0 < qend; q0 += TC) {
    __syncthreads();
    // stage q (scaled into the log2 domain) and dO as TF32; four consecutive lanes share a row: delta by a quad reduce.
    // All loads of a pass (three rows of q, dO, o and lse per thread) are issued before the first dependent instruction.
    constexpr int U = 3;
    for (int base = threadIdx.x; base < TC * 4; base += U * blockDim.x) {
      float4 a[U], gq[U], ov[U];
      float lv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = base + u * blockDim.x, row = idx >> 2, c4 = idx & 3;
        const int64_t qi = q0 + row;
        a[u] = gq[u] = ov[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        lv[u] = INFINITY;   // dead query: P = 0
        if (idx < TC * 4 && qi < qend) {
          a[u] = *reinterpret_cast<const float4*>(q + qi * sd.q + h * HD + c4 * 4);
          gq[u] = *reinterpret_cast<const float4*>(d_o + qi * sd.o + h * HD + c4 * 4);
          ov[u] = *reinterpret_cast<const float4*>(o + qi * sd.o + h * HD + c4 * 4);
          if (c4 == 0) lv[u] = lse[qi * heads + h] * kLog2e;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = base + u * blockDim.x, row = idx >> 2, c4 = idx & 3;
        if (idx < TC * 4) {   // warp-uniform: TC * 4 and blockDim.x are multiples of 32
          const float c = 0.25f * kLog2e;
          *reinterpret_cast<uint4*>(Qs + row * TS + c4 * 4) =
              make_uint4(tf32(a[u].x * c), tf32(a[u].y * c), tf32(a[u].z * c), tf32(a[u].w * c));
          *reinterpret_cast<uint4*>(Gs + row * TS + c4 * 4) = make_uint4(tf32(gq[u].x), tf32(gq[u].y), tf32(gq[u].z), tf32(gq[u].w));
          const float de = quad_sum(fmaf(gq[u].x, ov[u].x, fmaf(gq[u].y, ov[u].y, fmaf(gq[u].z, ov[u].z, gq[u].w * ov[u].w))));
          if (c4 == 0) {
            Ds[row] = de;
            Ls[row] = lv[u];
          }
        }
      }
    }
    if (q0 == qbeg) {
      cvt_a_frag(ka, kraw, 1.f);
      cvt_a_frag(va, vraw, 1.f);
    }
    __syncthreads();
    const int cnt = (int)min((int64_t)TC, qend - q0), nt = (cnt + 7) >> 3;
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      if (j < nt) {
        float st[4] = {}, dpt[4] = {};
        mma_rows(st, ka, Qs, j, g, t);
        mma_rows(dpt, va, Gs, j, g, t);
        const float2 L = *reinterpret_cast<const float2*>(Ls + 8 * j + 2 * t);
        const float2 D = *reinterpret_cast<const float2*>(Ds + 8 * j + 2 * t);
        float p[4] = {ex2(st[0] - L.x), ex2(st[1] - L.y), ex2(st[2] - L.x), ex2(st[3] - L.y)};
        float ds[4] = {p[0] * (dpt[0] - D.x), p[1] * (dpt[1] - D.y), p[2] * (dpt[2] - D.x), p[3] * (dpt[3] - D.y)};
        mma_acc(dva, p, Gs, j, g, t);
        mma_acc(dka, ds, Qs, j, g, t);   // Qs carries 0.25 log2e: dk = acc * ln2
      }
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int64_t r = half ? r_hi : r_lo;
    if (r >= lk) continue;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      float2* dstk = reinterpret_cast<float2*>(dk + r * sd.dkv + h * HD + 8 * d + 2 * t);
      float2* dstv = reinterpret_cast<float2*>(dv + r * sd.dkv + h * HD + 8 * d + 2 * t);
      const float2 vk = make_float2(dka[d][2 * half] * kLn2, dka[d][2 * half + 1] * kLn2);
      const float2 vv = make_float2(dva[d][2 * half], dva[d][2 * half + 1]);
      if (nsplit == 1) {
        *dstk = vk;
        *dstv = vv;
      } else if (part != nullptr) {   // deterministic: dk then dv partials, each [split][lk][heads * HD]
        const int64_t i = ((int64_t)split * lk + r) * heads * HD + h * HD + 8 * d + 2 * t;
        *reinterpret_cast<float2*>(part + i) = vk;
        *reinterpret_cast<float2*>(part + (int64_t)nsplit * lk * heads * HD + i) = vv;
      } else {
        atomicAdd(dstk, vk);
        atomicAdd(dstv, vv);
      }
    }
  }
}

// ONE launch for the whole backward: CTAs [0, nq) run the dq role, the rest the dk / dv role (the two are independent and
// each is a few microseconds of latency: back to back they cost twice that)
struct BwdGrid {
  int xq, sq, xk, sk;   // x-blocks and loop splits of the dq role / the dkv role
};
__global__ void __launch_bounds__(256, 2) cross_bwd_tc_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                              const float* __restrict__ v, const float* __restrict__ o,
                                                              const float* __restrict__ d_o, const float* __restrict__ lse,
                                                              float* __restrict__ dq, float* __restrict__ dk,
                                                              float* __restrict__ dv, int64_t lq, int64_t lk, int heads,
                                                              int64_t keys_per_split, int64_t q_per_split, Strides sd,
                                                              BwdGrid bg, float* __restrict__ part_q,
                                                              float* __restrict__ part_kv) {
  __shared__ __align__(16) BwdSmem sm;
  int b = blockIdx.x;
  const int nq = bg.xq * heads * bg.sq;
  if (b < nq) {
    const int bx = b % bg.xq, h = (b / bg.xq) % heads, split = b / (bg.xq * heads);
    cross_bwd_dq_tc(sm, bx, h, split, bg.sq, q, k, v, o, d_o, lse, dq, lq, lk, heads, keys_per_split, sd, part_q);
  } else {
    b -= nq;
    const int bx = b % bg.xk, h = (b / bg.xk) % heads, split = b / (bg.xk * heads);
    cross_bwd_dkv_tc(sm, bx, h, split, bg.sk, q, k, v, o, d_o, lse, dk, dv, lq, lk, heads, q_per_split, sd, part_kv);
  }
}

// out[r][c] = sum_s part[s][r][c] over the splits in index order (the deterministic backward's combine, one thread per
// element: no atomics)
__global__ void __launch_bounds__(256) cross_split_sum_kernel(const float* __restrict__ part, int splits, int64_t rows,
                                                              int e, float* __restrict__ out, int64_t ld_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * e) return;
  const int64_t r = i / e, c = i % e;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += part[(int64_t)s * rows * e + i];
  out[r * ld_out + c] = acc;
}

// ---------------------------------------------------------------------------------------------------------------------
// Head-averaged attention probabilities P[i, j] = (1/H) sum_h exp(s_ij^h - lse_ih): nn.MultiheadAttention's
// need_weights=True output, for the forward hooks of the adapter's attention modules.  Both kernels recompute the scores
// from the SAME operands with the SAME arithmetic as the forward of their impl (bitwise the same s) and take the lse that
// forward returned, so a row sums to 1 against the probabilities the forward actually used.  Every output element is
// written once by one thread, heads summed in index order in registers: no atomics, bitwise reproducible.
// ---------------------------------------------------------------------------------------------------------------------
static constexpr int PQ = 16;   // queries per CTA of the SIMT kernel (one thread per key, XT keys per CTA)

// SIMT (impl 0): thread = one key, loops over PQ staged queries per head.  dot16(k, q / 4) forms the products and sums of
// the forward's dot16(q / 4, k) in the same order (fma is commutative), so s is the forward's s bit for bit.
template <typename T>
__global__ void __launch_bounds__(XT) cross_probs_kernel(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k,
                                                         int64_t ldk, const float* __restrict__ lse, float* __restrict__ p,
                                                         int64_t ldp, int64_t lq, int64_t lk, int heads) {
  __shared__ __align__(16) float Qs[PQ * HD];
  __shared__ float Ls[PQ];
  const int64_t kj = (int64_t)blockIdx.x * XT + threadIdx.x, q0 = (int64_t)blockIdx.y * PQ;
  const bool live = kj < lk;
  float acc[PQ];
#pragma unroll
  for (int i = 0; i < PQ; ++i) acc[i] = 0.f;
  for (int h = 0; h < heads; ++h) {
    __syncthreads();
    if (threadIdx.x < PQ) {
      const int64_t qi = q0 + threadIdx.x;
      float a[HD];
      if (qi < lq) load16(q + qi * ldq + h * HD, a);
      else
#pragma unroll
        for (int e = 0; e < HD; ++e) a[e] = 0.f;
#pragma unroll
      for (int e = 0; e < HD; ++e) Qs[threadIdx.x * HD + e] = a[e] * 0.25f;   // 1/sqrt(16), as the forward's to_pairs
      Ls[threadIdx.x] = qi < lq ? lse[qi * heads + h] : 0.f;
    }
    __syncthreads();
    float kv[HD];
    if (live) load16(k + kj * ldk + h * HD, kv);
    else
#pragma unroll
      for (int e = 0; e < HD; ++e) kv[e] = 0.f;
    float2 k2[HD / 2];
    to_pairs(kv, 1.f, k2);
#pragma unroll
    for (int i = 0; i < PQ; ++i) acc[i] += expf(dot16(k2, Qs + i * HD) - Ls[i]);
  }
  if (!live) return;
  const float inv = 1.f / heads;
#pragma unroll
  for (int i = 0; i < PQ; ++i)
    if (q0 + i < lq) p[(q0 + i) * ldp + kj] = acc[i] * inv;
}

// Tensor cores (impl 1, f32 tensors): warp = 16 queries, CTA = those warps x one chunk of TC keys (grid.x), heads looped
// two at a time (stage2_tf32 stages head h into Ka and head h + 1 into Kb).  q is scaled by 0.25 log2e BEFORE the TF32
// rounding and the score MMAs are the forward's mma_rows on the same fragments: P = ex2(s - lse log2e) is the forward's
// probability.  The nine 16 x 8 accumulator tiles of the head sum stay in registers.
__global__ void __launch_bounds__(256) cross_probs_tc_kernel(const float* __restrict__ q, int64_t ldq,
                                                             const float* __restrict__ k, int64_t ldk,
                                                             const float* __restrict__ lse, float* __restrict__ p,
                                                             int64_t ldp, int64_t lq, int64_t lk, int heads) {
  __shared__ __align__(16) uint32_t Ka[TC * TS], Kb[TC * TS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int64_t r_lo = ((int64_t)blockIdx.y * (blockDim.x >> 5) + warp) * 16 + g, r_hi = r_lo + 8;
  const int64_t k0 = (int64_t)blockIdx.x * TC;
  const int cnt = (int)min((int64_t)TC, lk - k0), nt = (cnt + 7) >> 3;
  float acc[TNT][4] = {};
  for (int h0 = 0; h0 < heads; h0 += 2) {
    const int npair = h0 + 1 < heads ? 2 : 1;
    float qraw[2][2][4], L[2][2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {   // row operands of both heads in flight before the staging barrier
      const int h = u < npair ? h0 + u : h0;
      load_a_raw(qraw[u], q, ldq, h, r_lo, lq, t);
      L[u][0] = r_lo < lq ? lse[r_lo * heads + h] : 0.f;
      L[u][1] = r_hi < lq ? lse[r_hi * heads + h] : 0.f;
    }
    __syncthreads();
    stage2_tf32(Ka, Kb, k, k + (npair - 1) * HD, ldk, h0, k0, lk);
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (u >= npair) break;
      uint32_t qa[2][4];
      cvt_a_frag(qa, qraw[u], 0.25f * kLog2e);
      const float l_lo = L[u][0] * kLog2e, l_hi = L[u][1] * kLog2e;
#pragma unroll
      for (int j = 0; j < TNT; ++j) {
        if (j < nt) {
          float s[4] = {};
          mma_rows(s, qa, u ? Kb : Ka, j, g, t);
          acc[j][0] += ex2(s[0] - l_lo);
          acc[j][1] += ex2(s[1] - l_lo);
          acc[j][2] += ex2(s[2] - l_hi);
          acc[j][3] += ex2(s[3] - l_hi);
        }
      }
    }
  }
  const float inv = 1.f / heads;
  const bool vec = (ldp & 1) == 0 && (reinterpret_cast<uintptr_t>(p) & 7) == 0;   // k0 and the column 2t are even
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int64_t r = half ? r_hi : r_lo;
    if (r >= lq) continue;
    float* row = p + r * ldp + k0;
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      const int c = 8 * j + 2 * t;
      const float v0 = acc[j][2 * half] * inv, v1 = acc[j][2 * half + 1] * inv;
      if (vec && c + 1 < cnt) {
        *reinterpret_cast<float2*>(row + c) = make_float2(v0, v1);
      } else {
        if (c < cnt) row[c] = v0;
        if (c + 1 < cnt) row[c + 1] = v1;
      }
    }
  }
}

// rows_parallel rows spread over CTAs of `rows_per_cta`, the other side looped in chunks of `chunk`: how many loop splits?
static int pick_splits(int64_t rows_parallel, int64_t loop_len, int heads, int rows_per_cta, int chunk, bool tc) {
  const int64_t ctas = ((rows_parallel + rows_per_cta - 1) / rows_per_cta) * heads;
  if (ctas >= 2 * kNumSMs) return 1;
  // SIMT: four CTAs per SM, at least two chunks per split.  Tensor-core kernels: a chunk costs a few microseconds of
  // latency (stage, barrier, MMAs) and nothing else, so they want many short CTAs: eight per SM, single-chunk splits
  int64_t want = ((tc ? 8 : 4) * kNumSMs + ctas - 1) / ctas;
  int64_t maxs = tc ? (loop_len + chunk - 1) / chunk : (loop_len + 2 * chunk - 1) / (2 * chunk);
  if (want > maxs) want = maxs;
  if (want > (tc ? 128 : 64)) want = tc ? 128 : 64;
  return (int)(want < 1 ? 1 : want);
}
// warps per CTA of the tensor-core kernels: 16 rows per warp, at most 8 warps, at least enough for a short M side
static int tc_warps(int64_t rows) {
  const int64_t w = (rows + 15) / 16;
  return (int)(w < 4 ? (w < 1 ? 1 : w) : (w <= 8 ? w : 4));
}
struct Plan {
  int splits, warps;      // loop splits (grid.z), warps per CTA (tensor-core kernels)
  int64_t per_split;      // loop rows per split, a multiple of the chunk
  unsigned grid_x;
};
static Plan make_plan(int64_t rows_parallel, int64_t loop_len, int heads, bool tc, int force_warps = 0) {
  Plan p;
  p.warps = tc ? (force_warps ? force_warps : tc_warps(rows_parallel)) : XT / 32;
  const int rows_per_cta = tc ? 16 * p.warps : XT, chunk = tc ? TC : XC;
  p.splits = pick_splits(rows_parallel, loop_len, heads, rows_per_cta, chunk, tc);
  p.per_split = ((loop_len + p.splits - 1) / p.splits + chunk - 1) / chunk * chunk;
  p.splits = (int)((loop_len + p.per_split - 1) / p.per_split);   // no empty trailing splits
  p.grid_x = (unsigned)((rows_parallel + rows_per_cta - 1) / rows_per_cta);
  return p;
}
static bool use_tc(int impl, int dtype) { return impl == 1 && dtype == MT_F32; }

}  // namespace mt

using namespace mt;

extern "C" int64_t mt_cross_attn_workspace_floats(int64_t lq, int64_t lk, int heads, int head_dim, int dtype, int impl) {
  (void)head_dim;
  const Plan p = make_plan(lq, lk, heads, use_tc(impl, dtype));
  return p.splits == 1 ? 0 : (int64_t)p.splits * lq * heads * (HD + 2);
}

extern "C" int mt_cross_attn_fwd(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, int dtype,
                                 void* o, int64_t ldo, float* lse, int64_t lq, int64_t lk, int heads, int head_dim,
                                 float* workspace, int64_t workspace_floats, int impl, void* stream) {
  MT_REQUIRE(head_dim == HD, "cross_attn: head_dim must be 16 (got %d)", head_dim);
  MT_REQUIRE(lq > 0 && lk > 0 && heads > 0 && heads <= 65535, "cross_attn: bad sizes");
  MT_REQUIRE(impl == 0 || impl == 1, "cross_attn: impl must be 0 (SIMT fp32) or 1 (TF32 tensor cores)");
  const int64_t e = (int64_t)heads * HD;
  MT_REQUIRE(ldq >= e && ldkv >= e && ldo >= e && ((ldq | ldkv | ldo) & 7) == 0, "cross_attn: bad row strides");
  cudaStream_t st = (cudaStream_t)stream;
  const bool tc = use_tc(impl, dtype);
  const Plan p = make_plan(lq, lk, heads, tc);
  MT_REQUIRE(p.splits == 1 || (workspace != nullptr && workspace_floats >= (int64_t)p.splits * lq * heads * (HD + 2)),
             "cross_attn: workspace too small");
  const Strides sd{ldq, ldkv, ldo, 0, 0};
  dim3 grid(p.grid_x, (unsigned)heads, (unsigned)p.splits);
  const unsigned cgrid = (unsigned)((lq * heads * 32 + 127) / 128);   // one warp per (query, head)
  if (tc) {
    cross_fwd_tc_kernel<<<grid, 32 * p.warps, 0, st>>>((const float*)q, (const float*)k, (const float*)v, (float*)o, lse,
                                                      workspace, lq, lk, heads, p.per_split, sd);
    if (p.splits > 1) cross_combine_kernel<float><<<cgrid, 128, 0, st>>>(workspace, (float*)o, lse, lq, heads, p.splits, ldo);
  } else if (dtype == MT_F32) {
    cross_fwd_kernel<float><<<grid, XT, 0, st>>>((const float*)q, (const float*)k, (const float*)v, (float*)o, lse,
                                                 workspace, lq, lk, heads, p.per_split, sd);
    if (p.splits > 1) cross_combine_kernel<float><<<cgrid, 128, 0, st>>>(workspace, (float*)o, lse, lq, heads, p.splits, ldo);
  } else if (dtype == MT_BF16) {
    using bf = __nv_bfloat16;
    cross_fwd_kernel<bf><<<grid, XT, 0, st>>>((const bf*)q, (const bf*)k, (const bf*)v, (bf*)o, lse, workspace, lq, lk,
                                              heads, p.per_split, sd);
    if (p.splits > 1) cross_combine_kernel<bf><<<cgrid, 128, 0, st>>>(workspace, (bf*)o, lse, lq, heads, p.splits, ldo);
  } else {
    set_error("cross_attn: bad dtype %d", dtype);
    return MT_E_BADARG;
  }
  return check_launch("cross_fwd_kernel");
}

extern "C" int mt_cross_attn_probs(const void* q, int64_t ldq, const void* k, int64_t ldk, int dtype, const float* lse,
                                   float* p, int64_t ldp, int64_t lq, int64_t lk, int heads, int head_dim, int impl,
                                   void* stream) {
  MT_REQUIRE(head_dim == HD, "cross_attn_probs: head_dim must be 16 (got %d)", head_dim);
  MT_REQUIRE(lq > 0 && lk > 0 && heads > 0, "cross_attn_probs: bad sizes");
  MT_REQUIRE(impl == 0 || impl == 1, "cross_attn_probs: impl must be 0 (SIMT fp32) or 1 (TF32 tensor cores)");
  MT_REQUIRE(dtype == MT_F32 || dtype == MT_BF16, "cross_attn_probs: bad dtype %d", dtype);
  const int64_t e = (int64_t)heads * HD;
  MT_REQUIRE(ldq >= e && ldk >= e && ((ldq | ldk) & 7) == 0 && ldp >= lk, "cross_attn_probs: bad row strides");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_tc(impl, dtype)) {
    const int warps = tc_warps(lq);
    const int64_t gy = (lq + 16 * warps - 1) / (16 * warps), gx = (lk + TC - 1) / TC;
    MT_REQUIRE(gy <= 65535 && gx < (1ll << 31), "cross_attn_probs: too many queries");
    cross_probs_tc_kernel<<<dim3((unsigned)gx, (unsigned)gy), 32 * warps, 0, st>>>((const float*)q, ldq, (const float*)k,
                                                                                 ldk, lse, p, ldp, lq, lk, heads);
    return check_launch("cross_probs_tc_kernel");
  }
  const int64_t gy = (lq + PQ - 1) / PQ, gx = (lk + XT - 1) / XT;
  MT_REQUIRE(gy <= 65535 && gx < (1ll << 31), "cross_attn_probs: too many queries");
  const dim3 grid((unsigned)gx, (unsigned)gy);
  if (dtype == MT_F32)
    cross_probs_kernel<float><<<grid, XT, 0, st>>>((const float*)q, ldq, (const float*)k, ldk, lse, p, ldp, lq, lk, heads);
  else
    cross_probs_kernel<__nv_bfloat16><<<grid, XT, 0, st>>>((const __nv_bfloat16*)q, ldq, (const __nv_bfloat16*)k, ldk, lse,
                                                           p, ldp, lq, lk, heads);
  return check_launch("cross_probs_kernel");
}

// Plans of the two roles of the backward: tensor-core path: both roles of the one backward kernel run with the same CTA size
static void bwd_plans(int64_t lq, int64_t lk, int heads, bool tc, int* fw, Plan* pq, Plan* pk) {
  *fw = tc ? (tc_warps(lq) > tc_warps(lk) ? tc_warps(lq) : tc_warps(lk)) : 0;
  *pq = make_plan(lq, lk, heads, tc, *fw);
  *pk = make_plan(lk, lq, heads, tc, *fw);
}

extern "C" int64_t mt_cross_attn_bwd_workspace_floats(int64_t lq, int64_t lk, int heads, int head_dim, int dtype, int impl) {
  (void)head_dim;
  int fw;
  Plan pq, pk;
  bwd_plans(lq, lk, heads, use_tc(impl, dtype), &fw, &pq, &pk);
  const int64_t e = (int64_t)heads * HD;
  return (pq.splits > 1 ? (int64_t)pq.splits * lq * e : 0) + (pk.splits > 1 ? 2 * (int64_t)pk.splits * lk * e : 0);
}

static int cross_attn_bwd(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* o,
                          const void* d_o, int64_t ldo, const float* lse, int dtype, float* dq_f32, int64_t lddq,
                          float* dk_f32, float* dv_f32, int64_t lddkv, int64_t lq, int64_t lk, int heads, int head_dim,
                          float* workspace, int64_t workspace_floats, bool deterministic, int impl, cudaStream_t st) {
  MT_REQUIRE(head_dim == HD, "cross_attn: head_dim must be 16 (got %d)", head_dim);
  MT_REQUIRE(lq > 0 && lk > 0 && heads > 0 && heads <= 65535, "cross_attn: bad sizes");
  MT_REQUIRE(impl == 0 || impl == 1, "cross_attn: impl must be 0 (SIMT fp32) or 1 (TF32 tensor cores)");
  const int64_t e = (int64_t)heads * HD;
  MT_REQUIRE(ldq >= e && ldkv >= e && ldo >= e && lddq >= e && lddkv >= e && ((ldq | ldkv | ldo | lddq | lddkv) & 7) == 0,
             "cross_attn_bwd: bad row strides");
  const bool tc = use_tc(impl, dtype);
  int fw;
  Plan pq, pk;
  bwd_plans(lq, lk, heads, tc, &fw, &pq, &pk);
  MT_REQUIRE(((reinterpret_cast<uintptr_t>(dq_f32) | reinterpret_cast<uintptr_t>(dk_f32) |
               reinterpret_cast<uintptr_t>(dv_f32)) & 15) == 0, "cross_attn_bwd: gradients must be 16-byte aligned");
  if (deterministic) {
    MT_REQUIRE(tc, "cross_attn_bwd: the deterministic backward is the tensor-core one (impl 1, f32 tensors)");
    MT_REQUIRE(workspace_floats >= mt_cross_attn_bwd_workspace_floats(lq, lk, heads, head_dim, dtype, impl) &&
               (workspace != nullptr || workspace_floats == 0) && ((uintptr_t)workspace & 15) == 0,
               "cross_attn_bwd: workspace too small or not 16-byte aligned");
  }
  // split loops accumulate with vector reduce-adds into zero-filled gradients (deterministic: store partials that a
  // second pass sums in split order); an unsplit loop owns its rows and stores
  float* part_q = deterministic && pq.splits > 1 ? workspace : nullptr;
  float* part_kv = deterministic && pk.splits > 1 ? workspace + (pq.splits > 1 ? (int64_t)pq.splits * lq * e : 0) : nullptr;
  const size_t wbytes = sizeof(float) * (size_t)e;
  if (pq.splits > 1 && part_q == nullptr) MT_CUDA(cudaMemset2DAsync(dq_f32, sizeof(float) * lddq, 0, wbytes, (size_t)lq, st));
  if (pk.splits > 1 && part_kv == nullptr) {
    MT_CUDA(cudaMemset2DAsync(dk_f32, sizeof(float) * lddkv, 0, wbytes, (size_t)lk, st));
    MT_CUDA(cudaMemset2DAsync(dv_f32, sizeof(float) * lddkv, 0, wbytes, (size_t)lk, st));
  }
  const Strides sd{ldq, ldkv, ldo, lddq, lddkv};
  dim3 gq(pq.grid_x, (unsigned)heads, (unsigned)pq.splits);
  dim3 gk(pk.grid_x, (unsigned)heads, (unsigned)pk.splits);
  if (tc) {
    using f = float;
    const BwdGrid bg{(int)pq.grid_x, pq.splits, (int)pk.grid_x, pk.splits};
    const unsigned total = (unsigned)((int64_t)bg.xq * heads * bg.sq + (int64_t)bg.xk * heads * bg.sk);
    cross_bwd_tc_kernel<<<total, 32 * fw, 0, st>>>((const f*)q, (const f*)k, (const f*)v, (const f*)o, (const f*)d_o, lse,
                                                  dq_f32, dk_f32, dv_f32, lq, lk, heads, pq.per_split, pk.per_split, sd, bg,
                                                  part_q, part_kv);
    if (part_q != nullptr || part_kv != nullptr) {
      if (int rc = check_launch("cross_bwd_tc_kernel")) return rc;
      if (part_q != nullptr)
        cross_split_sum_kernel<<<(unsigned)((lq * e + 255) / 256), 256, 0, st>>>(part_q, pq.splits, lq, (int)e, dq_f32, lddq);
      if (part_kv != nullptr) {
        const int64_t n = lk * e;
        cross_split_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(part_kv, pk.splits, lk, (int)e, dk_f32, lddkv);
        cross_split_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(part_kv + (int64_t)pk.splits * n, pk.splits, lk,
                                                                            (int)e, dv_f32, lddkv);
      }
      return check_launch("cross_split_sum_kernel");
    }
  } else if (dtype == MT_F32) {
    using f = float;
    cross_bwd_dq_kernel<f><<<gq, XT, 0, st>>>((const f*)q, (const f*)k, (const f*)v, (const f*)o, (const f*)d_o, lse,
                                              dq_f32, lq, lk, heads, pq.per_split, sd);
    cross_bwd_dkv_kernel<f><<<gk, XT, 0, st>>>((const f*)q, (const f*)k, (const f*)v, (const f*)o, (const f*)d_o, lse,
                                               dk_f32, dv_f32, lq, lk, heads, pk.per_split, sd);
  } else if (dtype == MT_BF16) {
    using f = __nv_bfloat16;
    cross_bwd_dq_kernel<f><<<gq, XT, 0, st>>>((const f*)q, (const f*)k, (const f*)v, (const f*)o, (const f*)d_o, lse,
                                              dq_f32, lq, lk, heads, pq.per_split, sd);
    cross_bwd_dkv_kernel<f><<<gk, XT, 0, st>>>((const f*)q, (const f*)k, (const f*)v, (const f*)o, (const f*)d_o, lse,
                                               dk_f32, dv_f32, lq, lk, heads, pk.per_split, sd);
  } else {
    set_error("cross_attn: bad dtype %d", dtype);
    return MT_E_BADARG;
  }
  return check_launch("cross_bwd kernels");
}

extern "C" int mt_cross_attn_bwd(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* o,
                                 const void* d_o, int64_t ldo, const float* lse, int dtype, float* dq_f32, int64_t lddq,
                                 float* dk_f32, float* dv_f32, int64_t lddkv, int64_t lq, int64_t lk, int heads,
                                 int head_dim, int impl, void* stream) {
  return cross_attn_bwd(q, ldq, k, v, ldkv, o, d_o, ldo, lse, dtype, dq_f32, lddq, dk_f32, dv_f32, lddkv, lq, lk, heads,
                        head_dim, nullptr, 0, false, impl, (cudaStream_t)stream);
}

extern "C" int mt_cross_attn_bwd_ws(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* o,
                                    const void* d_o, int64_t ldo, const float* lse, int dtype, float* dq_f32, int64_t lddq,
                                    float* dk_f32, float* dv_f32, int64_t lddkv, int64_t lq, int64_t lk, int heads,
                                    int head_dim, float* workspace, int64_t workspace_floats, int impl, void* stream) {
  return cross_attn_bwd(q, ldq, k, v, ldkv, o, d_o, ldo, lse, dtype, dq_f32, lddq, dk_f32, dv_f32, lddkv, lq, lk, heads,
                        head_dim, workspace, workspace_floats, true, impl, (cudaStream_t)stream);
}
