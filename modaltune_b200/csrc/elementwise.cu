// HBM-bound fused kernels of the path: embedding assembly (A0), LayerNorm fwd/bwd (A1), GELU+LayerNorm(3072) fwd/bwd
// (A6), gated residual (A7 tail), casts.  All accesses are 128-bit vectorised; one row is owned by COLS/8 threads and
// every thread keeps its 8 elements in registers between the statistics pass and the write (single HBM pass).
#include "mt_common.cuh"

namespace mt {

// ---------------------------------------------------------------------------------------------------------------------
// row reductions: TPR threads per row (32 -> one warp, otherwise TPR / 32 warps through shared memory)
// ---------------------------------------------------------------------------------------------------------------------
template <int TPR>
__device__ __forceinline__ float row_sum(float v, float* red, int row_in_block, int t) {
  v = warp_sum(v);
  if constexpr (TPR == 32) {
    return v;
  } else {
    constexpr int W = TPR / 32;
    __syncthreads();
    if ((t & 31) == 0) red[row_in_block * W + (t >> 5)] = v;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < W; ++i) s += red[row_in_block * W + i];
    return s;
  }
}

// One 8-element chunk per thread: 96 threads per row for 768 columns (4 rows per 384-thread block), 384 threads per row
// for 3072 columns.  With three chunks per thread the backward kernels need ~100-128 registers, which caps them at 512
// resident threads per SM -- too few loads in flight to hide the arithmetic (erf, reductions) behind HBM; with one chunk
// they fit in 56 registers and run three 384-thread blocks per SM (measured: LN backward 768 -25 %, GELU+LN(3072)
// forward -18 %, backward -10 %).
template <int COLS> struct RowCfg {
  static constexpr int NCH = 1;                      // 8-element chunks per thread
  static constexpr int TPR = COLS / (8 * NCH);       // threads per row: 96 (768 columns) or 384 (3072 columns)
  static constexpr int THREADS = 384;
  static constexpr int MINB = 3;                     // resident blocks per SM the register budget is set for
  static constexpr int RPB = THREADS / TPR;          // rows per block iteration
  static_assert(COLS % (8 * NCH) == 0 && TPR % 32 == 0 && THREADS % TPR == 0, "supported widths: 768, 3072");
};

// ---------------------------------------------------------------------------------------------------------------------
// train-mode dropout + DropPath: Philox4x32-10 keyed by the step seed, counter = (8-element chunk, stream id, half)
// ---------------------------------------------------------------------------------------------------------------------
struct DropArgs {
  int on;                  // 0 = eval mode
  uint32_t threshold;      // keep iff random u32 >= threshold (threshold = p * 2^32)
  float inv_keep;          // 1 / (1 - p)
  const int64_t* seed;
  int64_t stream_id;
  const float* path_scale;
};

static int make_drop_args(const mt_dropout* d, DropArgs* out) {
  out->on = 0;
  out->threshold = 0;
  out->inv_keep = 1.f;
  out->seed = nullptr;
  out->stream_id = 0;
  out->path_scale = nullptr;
  if (d == nullptr) return 0;
  if (!(d->p >= 0.f && d->p < 1.f) || d->seed == nullptr) {
    set_error("dropout: p must be in [0, 1) and seed a device pointer");
    return MT_E_BADARG;
  }
  out->on = 1;
  out->threshold = (uint32_t)((double)d->p * 4294967296.0);
  out->inv_keep = 1.f / (1.f - d->p);
  out->seed = d->seed;
  out->stream_id = d->stream_id;
  out->path_scale = d->path_scale;
  return 0;
}

__device__ __forceinline__ uint4 philox4x32_10(uint2 key, uint4 ctr) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// multiplicative factors (0 or inv_keep * path_scale) of the 8 elements of chunk `chunk` (element index = 8 chunk + j)
__device__ __forceinline__ void drop_factors8(const DropArgs& d, int64_t chunk, float (&m)[8]) {
  const uint64_t seed = (uint64_t)__ldg(d.seed);
  const float sc = d.inv_keep * (d.path_scale != nullptr ? __ldg(d.path_scale) : 1.f);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const uint4 r = philox4x32_10(key, make_uint4((uint32_t)chunk, (uint32_t)((uint64_t)chunk >> 32),
                                                  (uint32_t)d.stream_id, (uint32_t)(2 * (d.stream_id >> 32) + half)));
    m[4 * half + 0] = r.x >= d.threshold ? sc : 0.f;
    m[4 * half + 1] = r.y >= d.threshold ? sc : 0.f;
    m[4 * half + 2] = r.z >= d.threshold ? sc : 0.f;
    m[4 * half + 3] = r.w >= d.threshold ? sc : 0.f;
  }
}

// erf(x) = sign(x) (1 - 2^-r(|x|)), r = -log2(erfc) as ONE degree-6 polynomial on [0, 4] (erf = 1 in fp32 beyond):
// |error| <= 3.2e-7 absolute (tests/test_kernel_math.py pins the coefficients), 10 instructions and no divergent
// branches, where erff() evaluates both of its ranges for a warp with mixed arguments (~25 instructions and a select
// per element).  The GELU+LN(3072) kernels are bound by instruction issue, not by HBM: 56 instructions per element.
__device__ __forceinline__ float erf_fast(float x) {
  const float t = fminf(fabsf(x), 4.0f);
  float r = -0x1.29e67ep-13f;
  r = fmaf(r, t, 0x1.e049eep-9f);
  r = fmaf(r, t, -0x1.fa343ep-6f);
  r = fmaf(r, t, 0x1.3295a4p-3f);
  r = fmaf(r, t, 0x1.d619c8p-1f);
  r = fmaf(r, t, 0x1.a0bfb2p+0f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-(r * t)));
  return copysignf(1.f - e, x);
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erf_fast(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
  float cdf = 0.5f * (1.f + erf_fast(x * 0.70710678118654752f));
  float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// y = LN(f(x)) * gamma + beta (+ add[row % add_rows]);  f = identity or GELU
template <int COLS, typename TX, typename TY, typename TA, bool GELU>
__global__ void __launch_bounds__(RowCfg<COLS>::THREADS, RowCfg<COLS>::MINB) ln_fwd_kernel(const TX* __restrict__ x, const float* __restrict__ xbias,
                                                     const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, const TA* __restrict__ add,
                                                     int64_t add_rows, TY* __restrict__ y, float* __restrict__ mean,
                                                     float* __restrict__ rstd, int64_t rows, float eps) {
  using C = RowCfg<COLS>;
  __shared__ float red[C::RPB * (C::TPR / 32) + 1];
  const int t = threadIdx.x % C::TPR, rib = threadIdx.x / C::TPR;
  for (int64_t row0 = (int64_t)blockIdx.x * C::RPB; row0 < rows; row0 += (int64_t)gridDim.x * C::RPB) {
    const int64_t row = row0 + rib;
    const bool live = row < rows;
    float v[C::NCH][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C::NCH; ++i) {
      if (live) {
        load8(x + row * COLS + (i * C::TPR + t) * 8, v[i]);
        if (xbias != nullptr) {  // bias of the producing GEMM, folded in here (the GEMM keeps a plain fp32 output)
          float bv[8];
          load8(xbias + (i * C::TPR + t) * 8, bv);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[i][j] += bv[j];
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i][j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (GELU) v[i][j] = gelu_erf(v[i][j]);
        s += v[i][j];
      }
    }
    const float mu = row_sum<C::TPR>(s, red, rib, t) * (1.f / COLS);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < C::NCH; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float d = v[i][j] - mu;
        q += d * d;
      }
    const float var = row_sum<C::TPR>(q, red, rib, t) * (1.f / COLS);
    const float rs = rsqrtf(var + eps);
    if (live) {
      if (t == 0) {
        if (mean) mean[row] = mu;
        if (rstd) rstd[row] = rs;
      }
#pragma unroll
      for (int i = 0; i < C::NCH; ++i) {
        const int c = (i * C::TPR + t) * 8;
        float g[8], b[8], o[8];
        load8(gamma + c, g);
        load8(beta + c, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mu) * rs * g[j] + b[j];
        if (add != nullptr) {
          float a[8];
          load8(add + (row % add_rows) * COLS + c, a);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] += a[j];
        }
        store8(y + row * COLS + c, o);
      }
    }
  }
}

// dx = [gelu'(x)] * rstd * (g - mean(g) - xhat * mean(g * xhat)) (+ residual), g = dy * gamma, xhat = (f(x) - mean) * rstd
template <int COLS, typename TDY, typename TX, typename TR, typename TDX, bool GELU, bool WGRAD>
__global__ void __launch_bounds__(RowCfg<COLS>::THREADS, RowCfg<COLS>::MINB) ln_bwd_kernel(const TDY* __restrict__ dy, const TX* __restrict__ x,
                                                     const float* __restrict__ xbias,
                                                     const float* __restrict__ gamma, const float* __restrict__ mean,
                                                     const float* __restrict__ rstd, const TR* __restrict__ residual,
                                                     TDX* __restrict__ dx, __nv_bfloat16* __restrict__ dx_lp,
                                                     float* __restrict__ dgamma, float* __restrict__ dbeta, int64_t rows,
                                                     float* __restrict__ part) {
  using C = RowCfg<COLS>;
  __shared__ float red[C::RPB * (C::TPR / 32) + 1];
  const int t = threadIdx.x % C::TPR, rib = threadIdx.x / C::TPR;
  float gam[C::NCH][8];
  float dg_acc[WGRAD ? C::NCH : 1][8], db_acc[WGRAD ? C::NCH : 1][8];
#pragma unroll
  for (int i = 0; i < C::NCH; ++i) {
    load8(gamma + (i * C::TPR + t) * 8, gam[i]);
    if constexpr (WGRAD) {
#pragma unroll
      for (int j = 0; j < 8; ++j) dg_acc[i][j] = db_acc[i][j] = 0.f;
    }
  }
  for (int64_t row0 = (int64_t)blockIdx.x * C::RPB; row0 < rows; row0 += (int64_t)gridDim.x * C::RPB) {
    const int64_t row = row0 + rib;
    const bool live = row < rows;
    float xh[C::NCH][8], g[C::NCH][8], raw[C::NCH][8];  // raw holds x, or gelu'(x) when GELU
    const float mu = live ? mean[row] : 0.f, rs = live ? rstd[row] : 0.f;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < C::NCH; ++i) {
      const int c = (i * C::TPR + t) * 8;
      float d[8];
      if (live) {
        load8(x + row * COLS + c, raw[i]);
        load8(dy + row * COLS + c, d);
        if (xbias != nullptr) {
          float bv[8];
          load8(xbias + c, bv);
#pragma unroll
          for (int j = 0; j < 8; ++j) raw[i][j] += bv[j];
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) raw[i][j] = d[j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float u = raw[i][j];
        if (GELU) {  // value and derivative share the erf: u = x * cdf, gelu' = cdf + x * pdf
          const float xv = raw[i][j];
          const float cdf = 0.5f * (1.f + erf_fast(xv * 0.70710678118654752f));
          u = xv * cdf;
          raw[i][j] = cdf + xv * 0.3989422804014327f * __expf(-0.5f * xv * xv);
        }
        xh[i][j] = (u - mu) * rs;
        g[i][j] = d[j] * gam[i][j];
        s1 += g[i][j];
        s2 += g[i][j] * xh[i][j];
        if constexpr (WGRAD) {
          dg_acc[i][j] += d[j] * xh[i][j];
          db_acc[i][j] += d[j];
        }
      }
    }
    const float m1 = row_sum<C::TPR>(s1, red, rib, t) * (1.f / COLS);
    const float m2 = row_sum<C::TPR>(s2, red, rib, t) * (1.f / COLS);
    if (live) {
#pragma unroll
      for (int i = 0; i < C::NCH; ++i) {
        const int c = (i * C::TPR + t) * 8;
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          o[j] = rs * (g[i][j] - m1 - xh[i][j] * m2);
          if (GELU) o[j] *= raw[i][j];
        }
        if (residual != nullptr) {
          float r[8];
          load8(residual + row * COLS + c, r);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] += r[j];
        }
        store8(dx + row * COLS + c, o);
        if (dx_lp != nullptr) store8(dx_lp + row * COLS + c, o);   // bf16 twin for the GEMM that consumes dx next
      }
    }
  }
  if constexpr (WGRAD) {
    // the RPB row-lanes of the block hold partials for the same columns: combine them in shared memory first, so that
    // every column receives ONE global atomic per block (same-address atomics serialise in L2)
    __shared__ float wsum[2 * COLS];
    if (part != nullptr) {
      // deterministic: the row-lanes add their partials in index order, the block's sums go to part[0 / 1][block][COLS]
      // and colsum_partials_kernel adds the blocks in index order
      for (int r = 0; r < C::RPB; ++r) {
        if (rib == r) {
#pragma unroll
          for (int i = 0; i < C::NCH; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = (i * C::TPR + t) * 8 + j;
              wsum[c] = r == 0 ? dg_acc[i][j] : wsum[c] + dg_acc[i][j];
              wsum[COLS + c] = r == 0 ? db_acc[i][j] : wsum[COLS + c] + db_acc[i][j];
            }
        }
        __syncthreads();
      }
      for (int c = threadIdx.x; c < COLS; c += blockDim.x) {
        part[(int64_t)blockIdx.x * COLS + c] = wsum[c];
        part[(int64_t)(gridDim.x + blockIdx.x) * COLS + c] = wsum[COLS + c];
      }
      return;
    }
    for (int c = threadIdx.x; c < 2 * COLS; c += blockDim.x) wsum[c] = 0.f;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < C::NCH; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = (i * C::TPR + t) * 8 + j;
        atomicAdd(wsum + c, dg_acc[i][j]);
        atomicAdd(wsum + COLS + c, db_acc[i][j]);
      }
    __syncthreads();
    for (int c = threadIdx.x; c < COLS; c += blockDim.x) {
      atomicAdd(dgamma + c, wsum[c]);
      atomicAdd(dbeta + c, wsum[COLS + c]);
    }
  }
}

template <typename TP>
__global__ void __launch_bounds__(256) embed_assemble_kernel(const TP* __restrict__ proj, const float* __restrict__ bias,
                                                             const float* __restrict__ coords,
                                                             const float* __restrict__ table,
                                                             const float* __restrict__ cls, float* __restrict__ x,
                                                             int64_t n_tiles, int embed, int ngrids, float inv_tile) {
  const int chunks = embed / 8;
  const int64_t total = (n_tiles + 1) * chunks;
  const int half = embed / 2;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = idx / chunks;
    const int c = (int)(idx % chunks) * 8;
    float o[8];
    if (row == 0) {
      load8(cls + c, o);  // cls_token + pos_embed[0], and pos_embed[0] == 0
    } else {
      const int64_t i = row - 1;
      float p[8], b[8], e[8];
      load8(proj + i * embed + c, p);
      load8(bias + c, b);
      // pos = floor(c0/256) * G + floor(c1/256) + 1 (slide_encoder.py:198-211), then pos_embed[pos] = [T[j'] | T[i']]
      // with (i', j') = divmod(pos - 1, G): a column index >= G wraps into the next grid row exactly as the reference's
      // flat table does, pos == 0 is the all-zero cls row.  An index outside the table is an error in the reference
      // (device-side index assert); here the kernel traps instead of clamping to a plausible but different embedding.
      const long long pos = (long long)floorf(coords[2 * i] * inv_tile) * ngrids +
                            (long long)floorf(coords[2 * i + 1] * inv_tile) + 1;
      if (pos < 0 || pos > (long long)ngrids * ngrids) __trap();
      if (pos == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) e[j] = 0.f;
      } else {
        const int gi = (int)((pos - 1) / ngrids), gj = (int)((pos - 1) % ngrids);
        if (c < half) load8(table + (int64_t)gj * half + c, e);
        else load8(table + (int64_t)gi * half + (c - half), e);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = p[j] + b[j] + e[j];
    }
    store8(x + row * embed + c, o);
  }
}

template <typename TB>
__global__ void __launch_bounds__(256) gated_residual_kernel(const float* __restrict__ a, const TB* __restrict__ b,
                                                             const float* __restrict__ gate, float* __restrict__ y,
                                                             int64_t rows, int cols) {
  const int chunks = cols / 8;
  const int64_t total = rows * chunks;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % chunks) * 8;
    float av[8], bv[8], gv[8], o[8];
    load8(a + idx * 8, av);
    load8(b + idx * 8, bv);
    if (gate) load8(gate + c, gv);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = av[j] + (gate ? gv[j] : 1.f) * (av[j] + bv[j]);
    store8(y + idx * 8, o);
  }
}

// x_out = x + a (fp32 residual stream), y = LN(x_out) * gamma + beta: the residual add after the attention / FFN branch
// fused with the next block's pre-LN (encoder.py:152-166), one pass over HBM.
template <int COLS, typename TA, typename TY>
__global__ void __launch_bounds__(RowCfg<COLS>::THREADS, RowCfg<COLS>::MINB) add_ln_fwd_kernel(const float* __restrict__ x, const TA* __restrict__ a,
                                                         const float* __restrict__ abias,
                                                         const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, float* __restrict__ x_out,
                                                         TY* __restrict__ y, float* __restrict__ mean,
                                                         float* __restrict__ rstd, int64_t rows, float eps,
                                                         const DropArgs drop) {
  using C = RowCfg<COLS>;
  __shared__ float red[C::RPB * (C::TPR / 32) + 1];
  const int t = threadIdx.x % C::TPR, rib = threadIdx.x / C::TPR;
  for (int64_t row0 = (int64_t)blockIdx.x * C::RPB; row0 < rows; row0 += (int64_t)gridDim.x * C::RPB) {
    const int64_t row = row0 + rib;
    const bool live = row < rows;
    float v[C::NCH][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C::NCH; ++i) {
      if (live) {
        float av[8];
        load8(x + row * COLS + (i * C::TPR + t) * 8, v[i]);
        load8(a + row * COLS + (i * C::TPR + t) * 8, av);
        if (abias != nullptr) {
          float bv[8];
          load8(abias + (i * C::TPR + t) * 8, bv);
#pragma unroll
          for (int j = 0; j < 8; ++j) av[j] += bv[j];
        }
        if (drop.on) {   // train mode: Dropout then DropPath on the branch, before the residual add (encoder.py:149-155)
          float m[8];
          drop_factors8(drop, row * (COLS / 8) + i * C::TPR + t, m);
#pragma unroll
          for (int j = 0; j < 8; ++j) av[j] *= m[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i][j] += av[j];
        store8(x_out + row * COLS + (i * C::TPR + t) * 8, v[i]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i][j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[i][j];
    }
    const float mu = row_sum<C::TPR>(s, red, rib, t) * (1.f / COLS);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < C::NCH; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float d = v[i][j] - mu;
        q += d * d;
      }
    const float var = row_sum<C::TPR>(q, red, rib, t) * (1.f / COLS);
    const float rs = rsqrtf(var + eps);
    if (live) {
      if (t == 0) {
        mean[row] = mu;
        rstd[row] = rs;
      }
#pragma unroll
      for (int i = 0; i < C::NCH; ++i) {
        const int c = (i * C::TPR + t) * 8;
        float g[8], b[8], o[8];
        load8(gamma + c, g);
        load8(beta + c, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mu) * rs * g[j] + b[j];
        store8(y + row * COLS + c, o);
      }
    }
  }
}

// backward of y = a + gate * (a + b):  da = dy * (1 + gate), db = dy * gate, dgate[c] += sum_r dy * (a + b)
// The column sums are reduced over the rows of a block in shared memory and flushed with one 16-byte reduce-add pair
// per column chunk and block: a few hundred blocks adding 8 scalars per thread into the same 24 cache lines spent
// most of the kernel serialised in the L2 atomic units.
template <typename TB>
__global__ void __launch_bounds__(768) gated_residual_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ a,
                                                                 const TB* __restrict__ b,
                                                                 const float* __restrict__ gate, float* __restrict__ da,
                                                                 TB* __restrict__ db, float* __restrict__ dgate,
                                                                 float* __restrict__ dysum, int64_t rows, int cols,
                                                                 float* __restrict__ part) {
  // thread t owns column chunk (t % chunks) for rows (blockIdx.x * rpb + t / chunks) + k * gridDim.x * rpb;
  // blockDim.x == chunks * rpb
  extern __shared__ float gr_red[];
  const int chunks = cols / 8;
  const int rpb = blockDim.x / chunks;
  const int ch = threadIdx.x % chunks, rib = threadIdx.x / chunks;
  float gv[8], acc[8], dsum[8];
  load8(gate + ch * 8, gv);
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = dsum[j] = 0.f;
#pragma unroll 2
  for (int64_t row = (int64_t)blockIdx.x * rpb + rib; row < rows; row += (int64_t)gridDim.x * rpb) {
    const int64_t off = row * cols + ch * 8;
    float d[8], av[8], bv[8], oa[8], ob[8];
    load8(dy + off, d);
    load8(a + off, av);
    load8(b + off, bv);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      oa[j] = d[j] * (1.f + gv[j]);
      ob[j] = d[j] * gv[j];
      acc[j] = fmaf(d[j], av[j] + bv[j], acc[j]);
      dsum[j] += d[j];
    }
    store8(da + off, oa);
    store8(db + off, ob);
  }
  // block-level column sums first (one reduce-add per column and block), for dgate and then, if wanted, for sum_r dy
  for (int pass = 0; pass < (dysum != nullptr ? 2 : 1); ++pass) {
    if (pass == 1) {
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = dsum[j];
    }
    if (rib > 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) gr_red[((rib - 1) * chunks + ch) * 8 + j] = acc[j];
    }
    __syncthreads();
    if (rib == 0) {
      for (int r = 0; r + 1 < rpb; ++r) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += gr_red[(r * chunks + ch) * 8 + j];
      }
      if (part != nullptr) {   // deterministic: part[pass][block][cols], summed in block order by colsum_partials_kernel
        float4* dst = reinterpret_cast<float4*>(part + ((int64_t)pass * gridDim.x + blockIdx.x) * cols + ch * 8);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        continue;
      }
      float4* dst = reinterpret_cast<float4*>((pass == 0 ? dgate : dysum) + ch * 8);
      atomicAdd(dst, make_float4(acc[0], acc[1], acc[2], acc[3]));
      atomicAdd(dst + 1, make_float4(acc[4], acc[5], acc[6], acc[7]));
    }
  }
}

// y = x + a + bias[c]: the residual add after fc2 (encoder.py:169-175) with the GEMM's bias folded in
template <typename TA>
__global__ void __launch_bounds__(256) residual_bias_add_kernel(const float* __restrict__ x, const TA* __restrict__ a,
                                                                const float* __restrict__ bias, float* __restrict__ y,
                                                                int64_t rows, int cols, const DropArgs drop) {
  const int chunks = cols / 8;
  const int64_t total = rows * chunks;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % chunks) * 8;
    float xv[8], av[8], bv[8], o[8];
    load8(x + idx * 8, xv);
    load8(a + idx * 8, av);
    if (bias != nullptr) load8(bias + c, bv);
#pragma unroll
    for (int j = 0; j < 8; ++j) av[j] += (bias != nullptr ? bv[j] : 0.f);
    if (drop.on) {
      float m[8];
      drop_factors8(drop, idx, m);
#pragma unroll
      for (int j = 0; j < 8; ++j) av[j] *= m[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = xv[j] + av[j];
    store8(y + idx * 8, o);
  }
}

// dst = src * keep_mask / (1 - p) * path_scale: the gradient of a dropped residual branch, converted for the dX GEMM
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) dropout_bwd_cast_kernel(const TS* __restrict__ s, TD* __restrict__ d, int64_t n8,
                                                               const DropArgs drop) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n8; idx += (int64_t)gridDim.x * blockDim.x) {
    float v[8], m[8];
    load8(s + idx * 8, v);
    drop_factors8(drop, idx, m);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= m[j];
    store8(d + idx * 8, v);
  }
}

template <typename TS, typename TD>
__global__ void __launch_bounds__(256) cast_kernel(const TS* __restrict__ s, TD* __restrict__ d, int64_t n8, int64_t n) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n8; idx += (int64_t)gridDim.x * blockDim.x) {
    float v[8];
    load8(s + idx * 8, v);
    store8(d + idx * 8, v);
  }
  if (blockIdx.x == 0) {
    for (int64_t i = n8 * 8 + threadIdx.x; i < n; i += blockDim.x) d[i] = from_float<TD>(to_float(s[i]));
  }
}

// Row means of the LayerNorm(3072) backward formed before fc2's dX GEMM (see mt_ffn_bwd_prep in the header): per row
// m1 = dy16 . c1 / C, m2 = dy16 . (y - x1 - c2) / C with dy16 = dy rounded to bf16 (also written: the GEMM's A operand).
__global__ void __launch_bounds__(RowCfg<768>::THREADS, RowCfg<768>::MINB)
ffn_bwd_prep_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ x1,
                    const float* __restrict__ c1, const float* __restrict__ c2, const float* __restrict__ mean,
                    const float* __restrict__ rstd, float4* __restrict__ rowv, __nv_bfloat16* __restrict__ dy16,
                    int64_t rows, float inv_ln_cols) {
  using C = RowCfg<768>;
  __shared__ float red[C::RPB * (C::TPR / 32) + 1];
  const int t = threadIdx.x % C::TPR, rib = threadIdx.x / C::TPR;
  float a1[8], a2[8];
  load8(c1 + t * 8, a1);
  load8(c2 + t * 8, a2);
  for (int64_t row0 = (int64_t)blockIdx.x * C::RPB; row0 < rows; row0 += (int64_t)gridDim.x * C::RPB) {
    const int64_t row = row0 + rib;
    const bool live = row < rows;
    float s1 = 0.f, s2 = 0.f;
    if (live) {
      float d[8], yv[8], xv[8];
      load8(dy + row * 768 + t * 8, d);
      load8(y + row * 768 + t * 8, yv);
      load8(x1 + row * 768 + t * 8, xv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        d[j] = __bfloat162float(__float2bfloat16_rn(d[j]));
        s1 = fmaf(d[j], a1[j], s1);
        s2 = fmaf(d[j], (yv[j] - xv[j]) - a2[j], s2);
      }
      store8(dy16 + row * 768 + t * 8, d);
    }
    const float m1 = row_sum<C::TPR>(s1, red, rib, t) * inv_ln_cols;
    const float m2 = row_sum<C::TPR>(s2, red, rib, t) * inv_ln_cols;
    if (live && t == 0) rowv[row] = make_float4(mean[row], rstd[row], m1, m2);
  }
}

// out[c] = sum_r x[r, c] (bias gradients of the adapter's projections): float4 column quads, RL row lanes per block,
// shared-memory combine, ONE 16-byte reduce-add per column quad and block into the zeroed output
__global__ void __launch_bounds__(1024) colsum_kernel(const float* __restrict__ x, int64_t ld, float* __restrict__ out,
                                                      int64_t rows, int quads, int row_lanes, float4* __restrict__ part) {
  extern __shared__ float4 cs_red[];
  const int qd = threadIdx.x % quads, rl = threadIdx.x / quads;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (rl < row_lanes) {
#pragma unroll 4
    for (int64_t r = (int64_t)blockIdx.x * row_lanes + rl; r < rows; r += (int64_t)gridDim.x * row_lanes) {
      const float4 v = *reinterpret_cast<const float4*>(x + r * ld + qd * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (rl > 0) cs_red[(rl - 1) * quads + qd] = acc;
  }
  __syncthreads();
  if (rl == 0) {
    for (int i = 0; i + 1 < row_lanes; ++i) {
      const float4 v = cs_red[i * quads + qd];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (part != nullptr) part[(int64_t)blockIdx.x * quads + qd] = acc;   // deterministic: summed by colsum_partials_kernel
    else atomicAdd(reinterpret_cast<float4*>(out) + qd, acc);
  }
}

// Second pass of the deterministic column reductions: out0[c] = sum_b part[b][c] over the nblk block partials in index
// order (and out1 from the next nblk rows when it is not NULL).  One thread per column: a fixed order, no atomics.
__global__ void __launch_bounds__(256) colsum_partials_kernel(const float* __restrict__ part, int nblk, int cols,
                                                              float* __restrict__ out0, float* __restrict__ out1) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int which = blockIdx.y;
  if (c >= cols) return;
  const float* p = part + (int64_t)which * nblk * cols + c;
  float acc = 0.f;
  for (int b = 0; b < nblk; ++b) acc += p[(int64_t)b * cols];
  (which == 0 ? out0 : out1)[c] = acc;
}

// LayerNorm(768) backward of the pre-attention LN (+ residual gradient, + bf16 twin) that ALSO prepares the FFN backward of
// the layer BELOW: its output dx is that layer's dy, and this kernel already holds dx and the layer's input x (= the
// output y of the layer below) in registers, so the two row means of mt_ffn_bwd_prep cost one more read (x1 of the layer
// below) instead of a separate pass over three [rows, 768] tensors:  rowv = (mean_f, rstd_f, dx16 . c1 / C,
// dx16 . (x - x1b - c2) / C) with dx16 = dx rounded to bf16 (the twin written here).
__global__ void __launch_bounds__(RowCfg<768>::THREADS, RowCfg<768>::MINB)
ln_bwd_prep_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
                   const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ residual,
                   float* __restrict__ dx, __nv_bfloat16* __restrict__ dx_lp, const float* __restrict__ x1b,
                   const float* __restrict__ c1, const float* __restrict__ c2, const float* __restrict__ mean_f,
                   const float* __restrict__ rstd_f, float4* __restrict__ rowv, int64_t rows, float inv_ln_cols) {
  using C = RowCfg<768>;
  __shared__ float red[C::RPB * (C::TPR / 32) + 1];
  const int t = threadIdx.x % C::TPR, rib = threadIdx.x / C::TPR;
  float gam[8], a1[8], a2[8];
  load8(gamma + t * 8, gam);
  load8(c1 + t * 8, a1);
  load8(c2 + t * 8, a2);
  for (int64_t row0 = (int64_t)blockIdx.x * C::RPB; row0 < rows; row0 += (int64_t)gridDim.x * C::RPB) {
    const int64_t row = row0 + rib;
    const bool live = row < rows;
    float xv[8], xh[8], g[8], xb[8];
    const float mu = live ? mean[row] : 0.f, rs = live ? rstd[row] : 0.f;
    float s1 = 0.f, s2 = 0.f;
    if (live) {
      float d[8];
      load8(x + row * 768 + t * 8, xv);
      load8(dy + row * 768 + t * 8, d);
      load8(x1b + row * 768 + t * 8, xb);     // requested early: consumed after the two reductions below
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        xh[j] = (xv[j] - mu) * rs;
        g[j] = d[j] * gam[j];
        s1 += g[j];
        s2 = fmaf(g[j], xh[j], s2);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) xv[j] = xh[j] = g[j] = xb[j] = 0.f;
    }
    const float m1 = row_sum<C::TPR>(s1, red, rib, t) * (1.f / 768.f);
    const float m2 = row_sum<C::TPR>(s2, red, rib, t) * (1.f / 768.f);
    float p1 = 0.f, p2 = 0.f;
    if (live) {
      float o[8], r[8];
      load8(residual + row * 768 + t * 8, r);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = rs * (g[j] - m1 - xh[j] * m2) + r[j];
        const float o16 = __bfloat162float(__float2bfloat16_rn(o[j]));
        p1 = fmaf(o16, a1[j], p1);
        p2 = fmaf(o16, (xv[j] - xb[j]) - a2[j], p2);
      }
      store8(dx + row * 768 + t * 8, o);
      store8(dx_lp + row * 768 + t * 8, o);
    }
    const float q1 = row_sum<C::TPR>(p1, red, rib, t) * inv_ln_cols;
    const float q2 = row_sum<C::TPR>(p2, red, rib, t) * inv_ln_cols;
    if (live && t == 0) rowv[row] = make_float4(mean_f[row], rstd_f[row], q1, q2);
  }
}

static inline int grid_for(int64_t work_items, int per_block) {
  int64_t blocks = (work_items + per_block - 1) / per_block;
  int64_t cap = (int64_t)kNumSMs * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ---- dispatch helpers ------------------------------------------------------------------------------------------------
template <int COLS, bool GELU, typename TX, typename TY>
static int launch_ln_fwd(const void* x, const float* xbias, const float* gamma, const float* beta, const void* add, int add_dtype,
                         int64_t add_rows, void* y, float* mean, float* rstd, int64_t rows, float eps, cudaStream_t st) {
  using C = RowCfg<COLS>;
  const int grid = grid_for(rows, C::RPB);
  if (add == nullptr || add_dtype == MT_F32)
    ln_fwd_kernel<COLS, TX, TY, float, GELU><<<grid, C::THREADS, 0, st>>>((const TX*)x, xbias, gamma, beta, (const float*)add,
                                                                   add_rows > 0 ? add_rows : 1, (TY*)y, mean, rstd,
                                                                   rows, eps);
  else
    ln_fwd_kernel<COLS, TX, TY, __nv_bfloat16, GELU><<<grid, C::THREADS, 0, st>>>(
        (const TX*)x, xbias, gamma, beta, (const __nv_bfloat16*)add, add_rows > 0 ? add_rows : 1, (TY*)y, mean, rstd, rows, eps);
  return check_launch("ln_fwd_kernel");
}

template <int COLS, bool GELU>
static int dispatch_ln_fwd(const void* x, int xd, const float* xbias, const float* gamma, const float* beta, const void* add, int ad,
                           int64_t add_rows, void* y, int yd, float* mean, float* rstd, int64_t rows, float eps,
                           cudaStream_t st) {
  if (xd == MT_F32 && yd == MT_F32)
    return launch_ln_fwd<COLS, GELU, float, float>(x, xbias, gamma, beta, add, ad, add_rows, y, mean, rstd, rows, eps, st);
  if (xd == MT_F32 && yd == MT_BF16)
    return launch_ln_fwd<COLS, GELU, float, __nv_bfloat16>(x, xbias, gamma, beta, add, ad, add_rows, y, mean, rstd, rows, eps, st);
  if (xd == MT_BF16 && yd == MT_BF16)
    return launch_ln_fwd<COLS, GELU, __nv_bfloat16, __nv_bfloat16>(x, xbias, gamma, beta, add, ad, add_rows, y, mean, rstd, rows, eps, st);
  if (xd == MT_BF16 && yd == MT_F32)
    return launch_ln_fwd<COLS, GELU, __nv_bfloat16, float>(x, xbias, gamma, beta, add, ad, add_rows, y, mean, rstd, rows, eps, st);
  set_error("layernorm: unsupported dtype combination");
  return MT_E_UNSUPPORTED;
}

// The column-reducing kernels (LayerNorm dgamma / dbeta, gated-residual dgate / dysum, colsum) run at most this many
// blocks; their deterministic variants write one partial row per block and output (mt_colreduce_workspace_floats).
static constexpr int kColReduceBlocks = 2 * kNumSMs;

// out0 (and out1) = the block partials of `part` summed in block order
static int sum_partials(const float* part, int nblk, int cols, float* out0, float* out1, cudaStream_t st) {
  const dim3 grid((unsigned)((cols + 255) / 256), out1 != nullptr ? 2u : 1u);
  colsum_partials_kernel<<<grid, 256, 0, st>>>(part, nblk, cols, out0, out1);
  return check_launch("colsum_partials_kernel");
}

template <int COLS, bool GELU, typename TDY, typename TX, typename TDX>
static int launch_ln_bwd(const void* dy, const void* x, const float* xbias, const float* gamma, const float* mean, const float* rstd,
                         const void* residual, int rd, void* dx, void* dx_lp, float* dgamma, float* dbeta, int64_t rows,
                         float* part, cudaStream_t st) {
  using C = RowCfg<COLS>;
  int grid = grid_for(rows, C::RPB);
  if (dgamma != nullptr && grid > kColReduceBlocks) grid = kColReduceBlocks;  // bound the number of atomic flushes
  if (dgamma != nullptr) {
    if constexpr (!GELU) {
      if (residual != nullptr && rd != MT_F32) {
        set_error("layernorm bwd with weight grads: residual must be f32");
        return MT_E_UNSUPPORTED;
      }
      ln_bwd_kernel<COLS, TDY, TX, float, TDX, GELU, true><<<grid, C::THREADS, 0, st>>>(
          (const TDY*)dy, (const TX*)x, xbias, gamma, mean, rstd, (const float*)residual, (TDX*)dx, (__nv_bfloat16*)dx_lp, dgamma, dbeta, rows, part);
      if (part != nullptr) {
        if (int rc = check_launch("ln_bwd_kernel")) return rc;
        return sum_partials(part, grid, COLS, dgamma, dbeta, st);
      }
    }
  } else if (residual == nullptr || rd == MT_F32)
    ln_bwd_kernel<COLS, TDY, TX, float, TDX, GELU, false><<<grid, C::THREADS, 0, st>>>(
        (const TDY*)dy, (const TX*)x, xbias, gamma, mean, rstd, (const float*)residual, (TDX*)dx, (__nv_bfloat16*)dx_lp, dgamma, dbeta, rows, nullptr);
  else
    ln_bwd_kernel<COLS, TDY, TX, __nv_bfloat16, TDX, GELU, false><<<grid, C::THREADS, 0, st>>>(
        (const TDY*)dy, (const TX*)x, xbias, gamma, mean, rstd, (const __nv_bfloat16*)residual, (TDX*)dx, (__nv_bfloat16*)dx_lp, dgamma, dbeta, rows, nullptr);
  return check_launch("ln_bwd_kernel");
}

template <int COLS, bool GELU>
static int dispatch_ln_bwd(const void* dy, int dyd, const void* x, int xd, const float* xbias, const float* gamma, const float* mean,
                           const float* rstd, const void* residual, int rd, void* dx, int dxd, void* dx_lp, float* dgamma,
                           float* dbeta, int64_t rows, cudaStream_t st, float* part = nullptr) {
#define MT_LNB(TDY, TX, TDX) \
  return launch_ln_bwd<COLS, GELU, TDY, TX, TDX>(dy, x, xbias, gamma, mean, rstd, residual, rd, dx, dx_lp, dgamma, dbeta, rows, part, st)
  using bf = __nv_bfloat16;
  if (dyd == MT_F32 && xd == MT_F32 && dxd == MT_F32) MT_LNB(float, float, float);
  if (dyd == MT_BF16 && xd == MT_F32 && dxd == MT_F32) MT_LNB(bf, float, float);
  if (dyd == MT_BF16 && xd == MT_BF16 && dxd == MT_BF16) MT_LNB(bf, bf, bf);
  if (dyd == MT_F32 && xd == MT_BF16 && dxd == MT_BF16) MT_LNB(float, bf, bf);
  if (dyd == MT_BF16 && xd == MT_BF16 && dxd == MT_F32) MT_LNB(bf, bf, float);
  if (dyd == MT_F32 && xd == MT_BF16 && dxd == MT_F32) MT_LNB(float, bf, float);
  if (dyd == MT_BF16 && xd == MT_F32 && dxd == MT_BF16) MT_LNB(bf, float, bf);
  if (dyd == MT_F32 && xd == MT_F32 && dxd == MT_BF16) MT_LNB(float, float, bf);
#undef MT_LNB
  set_error("layernorm bwd: unsupported dtype combination");
  return MT_E_UNSUPPORTED;
}

}  // namespace mt

using namespace mt;

extern "C" int mt_embed_assemble(const void* proj, int proj_dtype, const float* bias, const float* coords,
                                 const float* table, const float* cls, float* x, int64_t n_tiles, int64_t embed,
                                 int64_t ngrids, float tile_size, void* stream) {
  MT_REQUIRE(embed % 16 == 0 && n_tiles >= 0, "embed_assemble: embed must be a multiple of 16");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = grid_for((n_tiles + 1) * (embed / 8), 256);
  if (proj_dtype == MT_F32)
    embed_assemble_kernel<float><<<grid, 256, 0, st>>>((const float*)proj, bias, coords, table, cls, x, n_tiles,
                                                       (int)embed, (int)ngrids, 1.f / tile_size);
  else
    embed_assemble_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)proj, bias, coords, table, cls, x,
                                                               n_tiles, (int)embed, (int)ngrids, 1.f / tile_size);
  return check_launch("embed_assemble_kernel");
}

extern "C" int mt_layernorm_fwd(const void* x, int x_dtype, const float* gamma, const float* beta, const void* add,
                                int add_dtype, int64_t add_rows, void* y, int y_dtype, float* mean, float* rstd,
                                int64_t rows, int64_t cols, float eps, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  if (cols == 768)
    return dispatch_ln_fwd<768, false>(x, x_dtype, nullptr, gamma, beta, add, add_dtype, add_rows, y, y_dtype, mean, rstd, rows, eps, st);
  if (cols == 3072)
    return dispatch_ln_fwd<3072, false>(x, x_dtype, nullptr, gamma, beta, add, add_dtype, add_rows, y, y_dtype, mean, rstd, rows, eps, st);
  set_error("layernorm: width %lld not supported (768, 3072)", (long long)cols);
  return MT_E_UNSUPPORTED;
}

extern "C" int64_t mt_colreduce_workspace_floats(int64_t cols) { return 2 * (int64_t)kColReduceBlocks * cols; }

static int layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma, const float* mean,
                         const float* rstd, const void* residual, int res_dtype, void* dx, int dx_dtype, void* dx_bf16,
                         float* dgamma, float* dbeta, int64_t rows, int64_t cols, float* part, cudaStream_t st) {
  if (rows == 0) return 0;
  MT_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "layernorm bwd: dgamma and dbeta go together");
  if (cols == 768)
    return dispatch_ln_bwd<768, false>(dy, dy_dtype, x, x_dtype, nullptr, gamma, mean, rstd, residual, res_dtype, dx, dx_dtype, dx_bf16, dgamma, dbeta, rows, st, part);
  if (cols == 3072)
    return dispatch_ln_bwd<3072, false>(dy, dy_dtype, x, x_dtype, nullptr, gamma, mean, rstd, residual, res_dtype, dx, dx_dtype, dx_bf16, dgamma, dbeta, rows, st, part);
  set_error("layernorm bwd: width %lld not supported (768, 3072)", (long long)cols);
  return MT_E_UNSUPPORTED;
}

extern "C" int mt_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma,
                                const float* mean, const float* rstd, const void* residual, int res_dtype, void* dx,
                                int dx_dtype, void* dx_bf16, float* dgamma, float* dbeta, int64_t rows, int64_t cols,
                                void* stream) {
  return layernorm_bwd(dy, dy_dtype, x, x_dtype, gamma, mean, rstd, residual, res_dtype, dx, dx_dtype, dx_bf16, dgamma,
                       dbeta, rows, cols, nullptr, (cudaStream_t)stream);
}

extern "C" int mt_layernorm_bwd_ws(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma,
                                   const float* mean, const float* rstd, const void* residual, int res_dtype, void* dx,
                                   int dx_dtype, void* dx_bf16, float* dgamma, float* dbeta, int64_t rows, int64_t cols,
                                   float* workspace, int64_t workspace_floats, void* stream) {
  MT_REQUIRE(dgamma == nullptr || (workspace != nullptr && workspace_floats >= mt_colreduce_workspace_floats(cols)),
             "layernorm bwd: workspace too small");
  return layernorm_bwd(dy, dy_dtype, x, x_dtype, gamma, mean, rstd, residual, res_dtype, dx, dx_dtype, dx_bf16, dgamma,
                       dbeta, rows, cols, dgamma != nullptr ? workspace : nullptr, (cudaStream_t)stream);
}

extern "C" int mt_gelu_ln_fwd(const void* h, int h_dtype, const float* hbias, const float* gamma, const float* beta,
                              void* y, int y_dtype,
                              float* mean, float* rstd, int64_t rows, int64_t cols, float eps, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  if (cols == 3072)
    return dispatch_ln_fwd<3072, true>(h, h_dtype, hbias, gamma, beta, nullptr, 0, 1, y, y_dtype, mean, rstd, rows, eps, st);
  if (cols == 768)
    return dispatch_ln_fwd<768, true>(h, h_dtype, hbias, gamma, beta, nullptr, 0, 1, y, y_dtype, mean, rstd, rows, eps, st);
  set_error("gelu_ln: width %lld not supported (768, 3072)", (long long)cols);
  return MT_E_UNSUPPORTED;
}

extern "C" int mt_gelu_ln_bwd(const void* dy, int dy_dtype, const void* h, int h_dtype, const float* hbias,
                              const float* gamma,
                              const float* mean, const float* rstd, void* dh, int dh_dtype, int64_t rows, int64_t cols,
                              void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  if (cols == 3072)
    return dispatch_ln_bwd<3072, true>(dy, dy_dtype, h, h_dtype, hbias, gamma, mean, rstd, nullptr, 0, dh, dh_dtype, nullptr, nullptr, nullptr, rows, st);
  if (cols == 768)
    return dispatch_ln_bwd<768, true>(dy, dy_dtype, h, h_dtype, hbias, gamma, mean, rstd, nullptr, 0, dh, dh_dtype, nullptr, nullptr, nullptr, rows, st);
  set_error("gelu_ln bwd: width %lld not supported (768, 3072)", (long long)cols);
  return MT_E_UNSUPPORTED;
}

extern "C" int mt_gated_residual(const float* a, const void* b, int b_dtype, const float* gate, float* y, int64_t rows,
                                 int64_t cols, void* stream) {
  MT_REQUIRE(cols % 8 == 0, "gated_residual: cols must be a multiple of 8");
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  const int grid = grid_for(rows * (cols / 8), 256);
  if (b_dtype == MT_F32)
    gated_residual_kernel<float><<<grid, 256, 0, st>>>(a, (const float*)b, gate, y, rows, (int)cols);
  else
    gated_residual_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(a, (const __nv_bfloat16*)b, gate, y, rows, (int)cols);
  return check_launch("gated_residual_kernel");
}

extern "C" int mt_add_layernorm_fwd(const float* x, const void* a, int a_dtype, const float* abias, const float* gamma,
                                    const float* beta,
                                    float* x_out, void* y, int y_dtype, float* mean, float* rstd, int64_t rows,
                                    int64_t cols, float eps, const mt_dropout* drop, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  MT_REQUIRE(cols == 768, "add_layernorm: width %lld not supported (768)", (long long)cols);
  DropArgs D;
  if (int rc = make_drop_args(drop, &D)) return rc;
  using C = RowCfg<768>;
  using bf = __nv_bfloat16;
  const int grid = grid_for(rows, C::RPB);
  if (a_dtype == MT_F32 && y_dtype == MT_F32)
    add_ln_fwd_kernel<768, float, float><<<grid, C::THREADS, 0, st>>>(x, (const float*)a, abias, gamma, beta, x_out, (float*)y, mean, rstd, rows, eps, D);
  else if (a_dtype == MT_BF16 && y_dtype == MT_BF16)
    add_ln_fwd_kernel<768, bf, bf><<<grid, C::THREADS, 0, st>>>(x, (const bf*)a, abias, gamma, beta, x_out, (bf*)y, mean, rstd, rows, eps, D);
  else if (a_dtype == MT_F32 && y_dtype == MT_BF16)
    add_ln_fwd_kernel<768, float, bf><<<grid, C::THREADS, 0, st>>>(x, (const float*)a, abias, gamma, beta, x_out, (bf*)y, mean, rstd, rows, eps, D);
  else
    add_ln_fwd_kernel<768, bf, float><<<grid, C::THREADS, 0, st>>>(x, (const bf*)a, abias, gamma, beta, x_out, (float*)y, mean, rstd, rows, eps, D);
  return check_launch("add_ln_fwd_kernel");
}

static int gated_residual_bwd(const float* dy, const float* a, const void* b, int b_dtype, const float* gate, float* da,
                              void* db, int db_dtype, float* dgate, float* dysum, int64_t rows, int64_t cols, float* part,
                              cudaStream_t st) {
  MT_REQUIRE(cols % 8 == 0 && cols / 8 <= 256, "gated_residual_bwd: cols must be a multiple of 8, at most 2048");
  MT_REQUIRE(b_dtype == db_dtype, "gated_residual_bwd: db must have the dtype of b");
  MT_REQUIRE(gate != nullptr && dgate != nullptr, "gated_residual_bwd: gate and dgate are required");
  if (part == nullptr || rows == 0) {
    MT_CUDA(cudaMemsetAsync(dgate, 0, sizeof(float) * (size_t)cols, st));
    if (dysum != nullptr) MT_CUDA(cudaMemsetAsync(dysum, 0, sizeof(float) * (size_t)cols, st));
  }
  if (rows == 0) return 0;
  const int chunks = (int)(cols / 8);
  const int rpb = 768 / chunks;                  // >= 3 (chunks <= 256)
  const int threads = chunks * rpb;
  int grid = grid_for(rows, rpb);
  if (grid > kNumSMs) grid = kNumSMs;            // one 768-thread block per SM; bounds the number of reduce-add flushes
  static_assert(kNumSMs <= kColReduceBlocks, "partials of the deterministic variant");
  const size_t smem = sizeof(float) * 8 * (size_t)chunks * (rpb - 1);
  MT_REQUIRE(((reinterpret_cast<uintptr_t>(dgate) | reinterpret_cast<uintptr_t>(dysum)) & 15) == 0,
             "gated_residual_bwd: dgate / dysum must be 16-byte aligned");
  if (b_dtype == MT_F32)
    gated_residual_bwd_kernel<float><<<grid, threads, smem, st>>>(dy, a, (const float*)b, gate, da, (float*)db, dgate, dysum, rows, (int)cols, part);
  else
    gated_residual_bwd_kernel<__nv_bfloat16><<<grid, threads, smem, st>>>(dy, a, (const __nv_bfloat16*)b, gate, da, (__nv_bfloat16*)db, dgate, dysum, rows, (int)cols, part);
  if (int rc = check_launch("gated_residual_bwd_kernel")) return rc;
  return part != nullptr ? sum_partials(part, grid, (int)cols, dgate, dysum, st) : 0;
}

extern "C" int mt_gated_residual_bwd(const float* dy, const float* a, const void* b, int b_dtype, const float* gate,
                                     float* da, void* db, int db_dtype, float* dgate, float* dysum, int64_t rows,
                                     int64_t cols, void* stream) {
  return gated_residual_bwd(dy, a, b, b_dtype, gate, da, db, db_dtype, dgate, dysum, rows, cols, nullptr,
                            (cudaStream_t)stream);
}

extern "C" int mt_gated_residual_bwd_ws(const float* dy, const float* a, const void* b, int b_dtype, const float* gate,
                                        float* da, void* db, int db_dtype, float* dgate, float* dysum, int64_t rows,
                                        int64_t cols, float* workspace, int64_t workspace_floats, void* stream) {
  MT_REQUIRE(workspace != nullptr && workspace_floats >= mt_colreduce_workspace_floats(cols),
             "gated_residual_bwd: workspace too small");
  return gated_residual_bwd(dy, a, b, b_dtype, gate, da, db, db_dtype, dgate, dysum, rows, cols, workspace,
                            (cudaStream_t)stream);
}

extern "C" int mt_residual_bias_add(const float* x, const void* a, int a_dtype, const float* bias, float* y,
                                    int64_t rows, int64_t cols, const mt_dropout* drop, void* stream) {
  MT_REQUIRE(cols % 8 == 0, "residual_bias_add: cols must be a multiple of 8");
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return 0;
  DropArgs D;
  if (int rc = make_drop_args(drop, &D)) return rc;
  const int grid = grid_for(rows * (cols / 8), 256);
  if (a_dtype == MT_F32)
    residual_bias_add_kernel<float><<<grid, 256, 0, st>>>(x, (const float*)a, bias, y, rows, (int)cols, D);
  else
    residual_bias_add_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(x, (const __nv_bfloat16*)a, bias, y, rows, (int)cols, D);
  return check_launch("residual_bias_add_kernel");
}

extern "C" int mt_dropout_bwd_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n,
                                   const mt_dropout* drop, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MT_REQUIRE(drop != nullptr, "dropout_bwd_cast: drop must not be NULL (use mt_cast in eval mode)");
  MT_REQUIRE(n % 8 == 0, "dropout_bwd_cast: element count must be a multiple of 8");
  if (n == 0) return 0;
  DropArgs D;
  if (int rc = make_drop_args(drop, &D)) return rc;
  const int64_t n8 = n / 8;
  const int grid = grid_for(n8, 256);
  using bf = __nv_bfloat16;
  if (src_dtype == MT_F32 && dst_dtype == MT_BF16)
    dropout_bwd_cast_kernel<float, bf><<<grid, 256, 0, st>>>((const float*)src, (bf*)dst, n8, D);
  else if (src_dtype == MT_F32 && dst_dtype == MT_F32)
    dropout_bwd_cast_kernel<float, float><<<grid, 256, 0, st>>>((const float*)src, (float*)dst, n8, D);
  else if (src_dtype == MT_BF16 && dst_dtype == MT_BF16)
    dropout_bwd_cast_kernel<bf, bf><<<grid, 256, 0, st>>>((const bf*)src, (bf*)dst, n8, D);
  else
    dropout_bwd_cast_kernel<bf, float><<<grid, 256, 0, st>>>((const bf*)src, (float*)dst, n8, D);
  return check_launch("dropout_bwd_cast_kernel");
}

extern "C" int mt_ffn_bwd_prep(const float* dy, const float* y, const float* x1, const float* c1, const float* c2,
                               const float* mean, const float* rstd, float* rowv, void* dy_bf16, int64_t rows,
                               int64_t cols, int64_t ln_cols, void* stream) {
  MT_REQUIRE(cols == 768 && ln_cols > 0, "ffn_bwd_prep: cols must be 768 (got %lld)", (long long)cols);
  MT_REQUIRE(dy && y && x1 && c1 && c2 && mean && rstd && rowv && dy_bf16, "ffn_bwd_prep: NULL argument");
  MT_REQUIRE(((uintptr_t)rowv & 15) == 0, "ffn_bwd_prep: rowv must be 16-byte aligned");
  if (rows == 0) return 0;
  using C = RowCfg<768>;
  const int grid = grid_for(rows, C::RPB);
  ffn_bwd_prep_kernel<<<grid, C::THREADS, 0, (cudaStream_t)stream>>>(dy, y, x1, c1, c2, mean, rstd, (float4*)rowv,
                                                                     (__nv_bfloat16*)dy_bf16, rows, 1.0f / (float)ln_cols);
  return check_launch("ffn_bwd_prep_kernel");
}

static int colsum(const float* x, int64_t ld, float* out, int64_t rows, int64_t cols, float* part, cudaStream_t st) {
  MT_REQUIRE(x != nullptr && out != nullptr && rows >= 0, "colsum: NULL argument");
  MT_REQUIRE(cols > 0 && cols % 4 == 0 && cols <= 4096 && ld >= cols && ld % 4 == 0, "colsum: cols must be a multiple of 4, at most 4096");
  MT_REQUIRE((((uintptr_t)x | (uintptr_t)out | (uintptr_t)part) & 15) == 0, "colsum: 16-byte alignment");
  if (part == nullptr || rows == 0) MT_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)cols, st));
  if (rows == 0) return 0;
  const int quads = (int)(cols / 4);
  int row_lanes = 1024 / quads;
  if (row_lanes > 8) row_lanes = 8;
  if (row_lanes > rows) row_lanes = (int)rows;
  int64_t grid = (rows + (int64_t)row_lanes * 4 - 1) / ((int64_t)row_lanes * 4);   // >= 4 rows per lane
  if (grid > kColReduceBlocks) grid = kColReduceBlocks;
  if (grid < 1) grid = 1;
  const size_t smem = sizeof(float4) * (size_t)quads * (size_t)(row_lanes > 1 ? row_lanes - 1 : 1);
  colsum_kernel<<<(unsigned)grid, quads * row_lanes, smem, st>>>(x, ld, out, rows, quads, row_lanes, (float4*)part);
  if (int rc = check_launch("colsum_kernel")) return rc;
  return part != nullptr ? sum_partials(part, (int)grid, (int)cols, out, nullptr, st) : 0;
}

extern "C" int mt_colsum(const float* x, int64_t ld, float* out, int64_t rows, int64_t cols, void* stream) {
  return colsum(x, ld, out, rows, cols, nullptr, (cudaStream_t)stream);
}

extern "C" int mt_colsum_ws(const float* x, int64_t ld, float* out, int64_t rows, int64_t cols, float* workspace,
                            int64_t workspace_floats, void* stream) {
  MT_REQUIRE(workspace != nullptr && workspace_floats >= mt_colreduce_workspace_floats(cols), "colsum: workspace too small");
  return colsum(x, ld, out, rows, cols, workspace, (cudaStream_t)stream);
}

extern "C" int mt_layernorm_bwd_ffn_prep(const float* dy, const float* x, const float* gamma, const float* mean,
                                         const float* rstd, const float* residual, float* dx, void* dx_bf16,
                                         const float* x1_below, const float* c1, const float* c2, const float* mean_f,
                                         const float* rstd_f, float* rowv, int64_t rows, int64_t cols, int64_t ln_cols,
                                         void* stream) {
  MT_REQUIRE(cols == 768 && ln_cols > 0, "layernorm_bwd_ffn_prep: cols must be 768 (got %lld)", (long long)cols);
  MT_REQUIRE(dy && x && gamma && mean && rstd && residual && dx && dx_bf16 && x1_below && c1 && c2 && mean_f && rstd_f && rowv,
             "layernorm_bwd_ffn_prep: NULL argument");
  MT_REQUIRE(((uintptr_t)rowv & 15) == 0, "layernorm_bwd_ffn_prep: rowv must be 16-byte aligned");
  if (rows == 0) return 0;
  using C = RowCfg<768>;
  const int grid = grid_for(rows, C::RPB);
  ln_bwd_prep_kernel<<<grid, C::THREADS, 0, (cudaStream_t)stream>>>(dy, x, gamma, mean, rstd, residual, dx,
                                                                    (__nv_bfloat16*)dx_bf16, x1_below, c1, c2, mean_f, rstd_f,
                                                                    (float4*)rowv, rows, 1.0f / (float)ln_cols);
  return check_launch("ln_bwd_prep_kernel");
}

extern "C" int mt_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return 0;
  const int64_t n8 = n / 8;
  const int grid = grid_for(n8 > 0 ? n8 : 1, 256);
  if (src_dtype == MT_F32 && dst_dtype == MT_BF16)
    cast_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>((const float*)src, (__nv_bfloat16*)dst, n8, n);
  else if (src_dtype == MT_BF16 && dst_dtype == MT_F32)
    cast_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>((const __nv_bfloat16*)src, (float*)dst, n8, n);
  else if (src_dtype == MT_F32 && dst_dtype == MT_F32)
    cast_kernel<float, float><<<grid, 256, 0, st>>>((const float*)src, (float*)dst, n8, n);
  else
    cast_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, n8, n);
  return check_launch("cast_kernel");
}
