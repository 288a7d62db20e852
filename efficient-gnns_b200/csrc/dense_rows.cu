// Row-major [n_rows, K] fp32 passes that sit between the aggregations of a student GNN layer
// (arxiv_pyg/gnn.py:46-50: conv -> BatchNorm1d -> ReLU -> dropout) and their backward.
// All are HBM-bound streaming kernels: 128-bit accesses, per-CTA deterministic partial
// reductions (no atomics), grid sized to a multiple of the 148 SMs.
#include "common.cuh"
#include "philox.cuh"

namespace b200gnn {

constexpr int ROWS_THREADS = 256;

// thread -> (vector column cv, row group rg); rows_per_iter row groups cover 256 threads.
struct RowMap {
  int nvec, rows_per_iter, cv, rg;
  bool active;
};
__device__ __forceinline__ RowMap make_row_map(int K) {
  RowMap m;
  m.nvec = K >> 2;
  m.rows_per_iter = ROWS_THREADS / m.nvec;
  m.rg = threadIdx.x / m.nvec;
  m.cv = threadIdx.x - m.rg * m.nvec;
  m.active = m.rg < m.rows_per_iter;
  return m;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4s(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

// Deterministic cross-row-group reduction of two float4 accumulators into partial[slot][2][K].
__device__ __forceinline__ void reduce_store_2xK(const RowMap& m, int K, float4 a, float4 b, float* smem /*2*K*/,
                                                 float* out) {
  for (int i = threadIdx.x; i < 2 * K; i += ROWS_THREADS) smem[i] = 0.f;
  __syncthreads();
  for (int g = 0; g < m.rows_per_iter; ++g) {
    if (m.active && m.rg == g) {
      float* s = smem + 4 * m.cv;
      float* q = smem + K + 4 * m.cv;
      s[0] += a.x; s[1] += a.y; s[2] += a.z; s[3] += a.w;
      q[0] += b.x; q[1] += b.y; q[2] += b.z; q[3] += b.w;
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 2 * K; i += ROWS_THREADS) out[i] = smem[i];
}

// ---------------------------------------------------------------- column statistics
__global__ void __launch_bounds__(ROWS_THREADS) col_stats4_kernel(const float* __restrict__ Y, int64_t n_rows, int K,
                                                                  float* __restrict__ partial, int slots) {
  extern __shared__ float smem[];
  const RowMap m = make_row_map(K);
  const int64_t per = (n_rows + slots - 1) / slots;
  const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(n_rows, r0 + per);
  float4 s = make_float4(0, 0, 0, 0), q = s;
  if (m.active)
    for (int64_t r = r0 + m.rg; r < r1; r += m.rows_per_iter) {
      const float4 y = ld4(Y + (size_t)r * K + 4 * m.cv);
      vstat(s, q, y);
    }
  reduce_store_2xK(m, K, s, q, smem, partial + (size_t)blockIdx.x * 2 * K);
}

// ---------------------------------------------------------------- BatchNorm finalize (training mode)
// partial[slots][2][K] -> mean, invstd, scale=gamma*invstd, shift=beta-mean*scale; running stats updated
// like nn.BatchNorm1d (momentum, unbiased running variance).  fp64 accumulation of the partials.
// Reduce partial[slots][2][K] over slots for 4 columns per CTA (64 slot groups x 4 columns = 256 threads, K/4 CTAs:
// these kernels sit on the step's critical path and are latency-bound, so more, shorter chains), fp64 accumulation,
// fixed order => deterministic.
constexpr int FIN_COLS = 4, FIN_GROUPS = 64;
__device__ __forceinline__ bool finalize_reduce(const float* __restrict__ partial, int slots, int K, bool second,
                                                double& s_out, double& q_out, int& k_out) {
  __shared__ double sh[2][FIN_GROUPS][FIN_COLS];
  const int c = threadIdx.x % FIN_COLS, g = threadIdx.x / FIN_COLS;
  const int k = blockIdx.x * FIN_COLS + c;
  double s = 0.0, q = 0.0;
  if (k < K)
    for (int j = g; j < slots; j += FIN_GROUPS) {
      s += (double)partial[(size_t)j * 2 * K + k];
      if (second) q += (double)partial[(size_t)j * 2 * K + K + k];
    }
  sh[0][g][c] = s; sh[1][g][c] = q;
  __syncthreads();
  if (g == 0 && k < K) {
    s = 0.0; q = 0.0;
    for (int j = 0; j < FIN_GROUPS; ++j) { s += sh[0][j][c]; q += sh[1][j][c]; }
    s_out = s; q_out = q; k_out = k;
    return true;
  }
  return false;
}

__global__ void __launch_bounds__(256) bn_finalize_kernel(const float* __restrict__ partial, int slots, int K,
                                                          int64_t n, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, float eps, float momentum,
                                                          float* running_mean, float* running_var, float* mean_out,
                                                          float* invstd_out, float* scale_out, float* shift_out) {
  double s, q; int k;
  if (finalize_reduce(partial, slots, K, true, s, q, k)) {
    const double mean = s / (double)n;
    double var = q / (double)n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = gamma[k] * invstd;
    mean_out[k] = (float)mean;
    invstd_out[k] = invstd;
    scale_out[k] = sc;
    shift_out[k] = beta[k] - (float)mean * sc;
    if (running_mean) {
      const double unbiased = n > 1 ? var * (double)n / (double)(n - 1) : var;
      running_mean[k] = (1.f - momentum) * running_mean[k] + momentum * (float)mean;
      running_var[k] = (1.f - momentum) * running_var[k] + momentum * (float)unbiased;
    }
  }
}

// ---------------------------------------------------------------- forward: affine + ReLU + dropout
// out = dropout(relu(y*scale + shift)); kept values scaled by 1/(1-p).  The keep decision of element e is a pure
// function of (seed, offset, global element index), so masks are identical under any row sharding:
//   P16 (p * 65536 integral, e.g. the reference's p = 0.5): Philox block b = (global float4 index) / 2 yields eight
//       16-bit uniforms, keep iff u16 >= p * 65536 — exact for such p, and half the generator work per element
//       (the pass is integer-bound on Philox, not HBM-bound, otherwise);
//   else: block b = global float4 index, four 24-bit uniforms, keep iff u >= p.
__device__ __forceinline__ float4 affine_relu4(float4 y, const float* __restrict__ scale, const float* __restrict__ shift,
                                               int cv, int relu) {
  if (scale) {
    const float4 sc = ld4(scale + 4 * cv), sh = ld4(shift + 4 * cv);
    y.x = fmaf(y.x, sc.x, sh.x); y.y = fmaf(y.y, sc.y, sh.y);
    y.z = fmaf(y.z, sc.z, sh.z); y.w = fmaf(y.w, sc.w, sh.w);
  }
  if (relu) { y.x = fmaxf(y.x, 0.f); y.y = fmaxf(y.y, 0.f); y.z = fmaxf(y.z, 0.f); y.w = fmaxf(y.w, 0.f); }
  return y;
}
__device__ __forceinline__ uchar4 keep16(uint32_t a, uint32_t b, uint32_t thr) {
  uchar4 m;
  m.x = (a & 0xffffu) >= thr; m.y = (a >> 16) >= thr; m.z = (b & 0xffffu) >= thr; m.w = (b >> 16) >= thr;
  return m;
}
__device__ __forceinline__ uchar4 keep24(const uint4& r, float p) {
  uchar4 m;
  m.x = u32_to_unit(r.x) >= p; m.y = u32_to_unit(r.y) >= p; m.z = u32_to_unit(r.z) >= p; m.w = u32_to_unit(r.w) >= p;
  return m;
}

template <bool P16>
__global__ void __launch_bounds__(256) affine_relu_dropout_kernel(const float* __restrict__ Y, float* __restrict__ out,
                                                                  int64_t n_vec, int nvec_row,
                                                                  const float* __restrict__ scale,
                                                                  const float* __restrict__ shift, int relu, float p,
                                                                  uint32_t thr16, uint64_t seed, uint64_t offset,
                                                                  const int32_t* __restrict__ step_dev,
                                                                  uint64_t step_mul, uint64_t index_offset) {
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  if (step_dev) offset += (uint64_t)(*step_dev) * step_mul;  // graph-replayable per-step offset
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  if (P16) {
    const uint64_t g0 = index_offset, g1 = index_offset + (uint64_t)n_vec;
    for (uint64_t b = (g0 >> 1) + (uint64_t)tid; b < ((g1 + 1) >> 1); b += (uint64_t)stride) {
      const uint4 r = philox4x32(seed, offset, b);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const uint64_t g = 2 * b + half;
        if (g < g0 || g >= g1) continue;
        const int64_t i = (int64_t)(g - g0);
        float4 y = affine_relu4(ld4s(Y + 4 * i), scale, shift, (int)(i % nvec_row), relu);
        const uchar4 m = keep16(half ? r.z : r.x, half ? r.w : r.y, thr16);
        y.x = m.x ? y.x * inv_keep : 0.f; y.y = m.y ? y.y * inv_keep : 0.f;
        y.z = m.z ? y.z * inv_keep : 0.f; y.w = m.w ? y.w * inv_keep : 0.f;
        st4(out + 4 * i, y);
      }
    }
  } else {
    for (int64_t i = tid; i < n_vec; i += stride) {
      float4 y = affine_relu4(ld4s(Y + 4 * i), scale, shift, (int)(i % nvec_row), relu);
      if (p > 0.f) {
        const uchar4 m = keep24(philox4x32(seed, offset, (uint64_t)i + index_offset), p);
        y.x = m.x ? y.x * inv_keep : 0.f; y.y = m.y ? y.y * inv_keep : 0.f;
        y.z = m.z ? y.z * inv_keep : 0.f; y.w = m.w ? y.w * inv_keep : 0.f;
      }
      st4(out + 4 * i, y);
    }
  }
}

// Same pass on a BLOCK of the activation matrix: local rows r (global node id rowmap[r], or r + row_offset) and the
// local columns [4*cv_off, 4*cv_off + 4*nvec_l) of a matrix that is nvec_g float4 wide globally.  The keep decision of
// an element is the one affine_relu_dropout_kernel takes for the same (node, feature) of the full matrix, so any
// row/column sharding and any node relabelling of the node-parallel engine reproduces the single-GPU mask bit for bit.
// Optional second destination of the block pass: the fused C->R layout exchange (hybrid.py) — row r of this [n_rows, K]
// block belongs to the rank q with off[q] <= r < off[q+1] and is ALSO stored to ptr[q] + (r - off[q]) * ld + col.
struct RowScatter {
  float* ptr[16];
  int32_t off[17];
  int32_t n;
  int64_t ld, col;
};
__device__ __forceinline__ float* scatter_row(const RowScatter& sc, int64_t r) {
  int q = 0;
#pragma unroll 1
  while (q + 1 < sc.n && r >= sc.off[q + 1]) ++q;
  return sc.ptr[q] + (size_t)(r - sc.off[q]) * (size_t)sc.ld + sc.col;
}

template <bool P16>
__global__ void __launch_bounds__(256) affine_relu_dropout_mapped_kernel(
    const float* __restrict__ Y, float* __restrict__ out, int64_t n_rows, int nvec_l, const float* __restrict__ scale,
    const float* __restrict__ shift, int relu, float p, uint32_t thr16, uint64_t seed, uint64_t offset,
    const int32_t* __restrict__ step_dev, uint64_t step_mul, const int32_t* __restrict__ rowmap, uint64_t row_offset,
    uint64_t nvec_g, uint64_t cv_off, int paired, const RowScatter sc) {
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  if (step_dev) offset += (uint64_t)(*step_dev) * step_mul;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  if (P16 && paired) {                       // nvec_l, nvec_g, cv_off all even: one Philox block serves two float4s
    const int half_l = nvec_l >> 1;
    for (int64_t u = tid; u < n_rows * half_l; u += stride) {
      const int64_t r = u / half_l;
      const int cv = (int)(u - r * half_l) * 2;
      const uint64_t gid = rowmap ? (uint64_t)rowmap[r] : (uint64_t)r + row_offset;
      const uint64_t g = gid * nvec_g + cv_off + (uint64_t)cv;
      const uint4 rnd = philox4x32(seed, offset, g >> 1);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int64_t i = r * nvec_l + cv + half;
        float4 y = affine_relu4(ld4s(Y + 4 * i), scale, shift, cv + half, relu);
        const uchar4 m = keep16(half ? rnd.z : rnd.x, half ? rnd.w : rnd.y, thr16);
        y.x = m.x ? y.x * inv_keep : 0.f; y.y = m.y ? y.y * inv_keep : 0.f;
        y.z = m.z ? y.z * inv_keep : 0.f; y.w = m.w ? y.w * inv_keep : 0.f;
        st4(out + 4 * i, y);
        if (sc.n) st4(scatter_row(sc, r) + 4 * (cv + half), y);
      }
    }
    return;
  }
  for (int64_t i = tid; i < n_rows * nvec_l; i += stride) {
    const int64_t r = i / nvec_l;
    const int cv = (int)(i - r * nvec_l);
    float4 y = affine_relu4(ld4s(Y + 4 * i), scale, shift, cv, relu);
    if (p > 0.f) {
      const uint64_t gid = rowmap ? (uint64_t)rowmap[r] : (uint64_t)r + row_offset;
      const uint64_t g = gid * nvec_g + cv_off + (uint64_t)cv;
      uchar4 m;
      if (P16) {
        const uint4 rnd = philox4x32(seed, offset, g >> 1);
        m = keep16((g & 1) ? rnd.z : rnd.x, (g & 1) ? rnd.w : rnd.y, thr16);
      } else {
        m = keep24(philox4x32(seed, offset, g), p);
      }
      y.x = m.x ? y.x * inv_keep : 0.f; y.y = m.y ? y.y * inv_keep : 0.f;
      y.z = m.z ? y.z * inv_keep : 0.f; y.w = m.w ? y.w * inv_keep : 0.f;
    }
    st4(out + 4 * i, y);
    if (sc.n) st4(scatter_row(sc, r) + 4 * cv, y);
  }
}

// The keep-mask the kernel above uses, materialised (tests inject it into the CPU oracle).
__global__ void __launch_bounds__(256) dropout_mask_kernel(uint8_t* __restrict__ mask, int64_t n_vec, float p, int p16,
                                                           uint32_t thr16, uint64_t seed, uint64_t offset) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    uchar4 m;
    if (p16) {
      const uint4 r = philox4x32(seed, offset, (uint64_t)i >> 1);
      m = keep16((i & 1) ? r.z : r.x, (i & 1) ? r.w : r.y, thr16);
    } else {
      m = keep24(philox4x32(seed, offset, (uint64_t)i), p);
    }
    reinterpret_cast<uchar4*>(mask)[i] = m;
  }
}

// p * 65536 integral (and p > 0): the 16-bit decision path is exact
static inline bool dropout_p16(float p, uint32_t& thr16) {
  const double t = (double)p * 65536.0;
  thr16 = (uint32_t)t;
  return p > 0.f && t == (double)thr16;
}

// ---------------------------------------------------------------- backward of BN(train)+ReLU+dropout
// dz = dOut * [Xout > 0] / (1-p)       (Xout>0  <=>  kept by dropout AND relu-active)
// pass 1: partial column sums of dz and dz*xhat, xhat = (Y-mean)*invstd
__global__ void __launch_bounds__(ROWS_THREADS) bn_act_bwd_reduce_kernel(
    const float* __restrict__ dOut, const float* __restrict__ Xout, const float* __restrict__ Y,
    const float* __restrict__ mean, const float* __restrict__ invstd, int64_t n_rows, int K, float inv_keep,
    float* __restrict__ partial, int slots) {
  extern __shared__ float smem[];
  const RowMap m = make_row_map(K);
  const int64_t per = (n_rows + slots - 1) / slots;
  const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(n_rows, r0 + per);
  float4 s = make_float4(0, 0, 0, 0), q = s;
  if (m.active) {
    const float4 mu = ld4(mean + 4 * m.cv), is = ld4(invstd + 4 * m.cv);
    for (int64_t r = r0 + m.rg; r < r1; r += m.rows_per_iter) {
      const size_t o = (size_t)r * K + 4 * m.cv;
      const float4 g = ld4(dOut + o), x = ld4(Xout + o), y = ld4(Y + o);
      const float dx = x.x > 0.f ? g.x * inv_keep : 0.f, dy = x.y > 0.f ? g.y * inv_keep : 0.f;
      const float dz = x.z > 0.f ? g.z * inv_keep : 0.f, dw = x.w > 0.f ? g.w * inv_keep : 0.f;
      s.x += dx; s.y += dy; s.z += dz; s.w += dw;
      q.x = fmaf(dx, (y.x - mu.x) * is.x, q.x); q.y = fmaf(dy, (y.y - mu.y) * is.y, q.y);
      q.z = fmaf(dz, (y.z - mu.z) * is.z, q.z); q.w = fmaf(dw, (y.w - mu.w) * is.w, q.w);
    }
  }
  reduce_store_2xK(m, K, s, q, smem, partial + (size_t)blockIdx.x * 2 * K);
}

// partials -> dgamma, dbeta, and the per-column coefficients of pass 2.
__global__ void __launch_bounds__(256) bn_bwd_finalize_kernel(const float* __restrict__ partial, int slots, int K,
                                                              int64_t n, const float* __restrict__ gamma,
                                                              const float* __restrict__ invstd, float* dgamma,
                                                              float* dbeta, float* coef /*[3][K]*/) {
  double s, q; int k;
  if (finalize_reduce(partial, slots, K, true, s, q, k)) {
    dbeta[k] = (float)s;
    dgamma[k] = (float)q;
    coef[k] = gamma[k] * invstd[k];
    coef[K + k] = (float)(s / (double)n);
    coef[2 * K + k] = (float)(q / (double)n);
  }
}

// pass 2: dY = gamma*invstd * (dz - mean(dz) - xhat*mean(dz*xhat)); optional partial column sums of dY
// (gradient of the conv bias in front of the BatchNorm).  DZ: dOut already holds dz (the fused input-gradient GEMM,
// b200gnn_gemm_tf32x3_bnbwd_f32, stored it) — Xout is not read.
template <bool DZ>
__global__ void __launch_bounds__(ROWS_THREADS) bn_act_bwd_apply_kernel(
    const float* __restrict__ dOut, const float* __restrict__ Xout, const float* __restrict__ Y,
    const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ coef, int64_t n_rows,
    int K, float inv_keep, float* __restrict__ dY, float* __restrict__ colsum_partial, int slots) {
  extern __shared__ float smem[];
  const RowMap m = make_row_map(K);
  const int64_t per = (n_rows + slots - 1) / slots;
  const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(n_rows, r0 + per);
  float4 s = make_float4(0, 0, 0, 0), q = s;
  if (m.active) {
    const float4 mu = ld4(mean + 4 * m.cv), is = ld4(invstd + 4 * m.cv);
    const float4 c1 = ld4(coef + 4 * m.cv), c2 = ld4(coef + K + 4 * m.cv), c3 = ld4(coef + 2 * K + 4 * m.cv);
    for (int64_t r = r0 + m.rg; r < r1; r += m.rows_per_iter) {
      const size_t o = (size_t)r * K + 4 * m.cv;
      float4 g = ld4s(dOut + o);
      const float4 y = ld4s(Y + o);
      if (!DZ) {
        const float4 x = ld4s(Xout + o);
        g.x = x.x > 0.f ? g.x * inv_keep : 0.f; g.y = x.y > 0.f ? g.y * inv_keep : 0.f;
        g.z = x.z > 0.f ? g.z * inv_keep : 0.f; g.w = x.w > 0.f ? g.w * inv_keep : 0.f;
      }
      float4 d;
      d.x = c1.x * (g.x - c2.x - (y.x - mu.x) * is.x * c3.x);
      d.y = c1.y * (g.y - c2.y - (y.y - mu.y) * is.y * c3.y);
      d.z = c1.z * (g.z - c2.z - (y.z - mu.z) * is.z * c3.z);
      d.w = c1.w * (g.w - c2.w - (y.w - mu.w) * is.w * c3.w);
      st4(dY + o, d);
      s.x += d.x; s.y += d.y; s.z += d.z; s.w += d.w;
    }
  }
  if (colsum_partial) reduce_store_2xK(m, K, s, q, smem, colsum_partial + (size_t)blockIdx.x * 2 * K);
}

// Sum partial[slots][2][K] (first plane only) -> out[K]   (bias gradients)
__global__ void __launch_bounds__(256) partial_reduce_kernel(const float* __restrict__ partial, int slots, int K2,
                                                             float* __restrict__ out) {
  __shared__ double sh[FIN_GROUPS][FIN_COLS];
  const int c = threadIdx.x % FIN_COLS, g = threadIdx.x / FIN_COLS;
  const int k = blockIdx.x * FIN_COLS + c;
  double s = 0.0;
  if (k < K2)
    for (int j = g; j < slots; j += FIN_GROUPS) s += (double)partial[(size_t)j * K2 + k];
  sh[g][c] = s;
  __syncthreads();
  if (g == 0 && k < K2) {
    s = 0.0;
    for (int j = 0; j < FIN_GROUPS; ++j) s += sh[j][c];
    out[k] = (float)s;
  }
}

__global__ void __launch_bounds__(256) colsum_finalize_kernel(const float* __restrict__ partial, int slots, int K,
                                                              float* __restrict__ out) {
  double s, q; int k;
  if (finalize_reduce(partial, slots, K, false, s, q, k)) out[k] = (float)s;
}

// ---------------------------------------------------------------- Adam (torch.optim.Adam defaults, no amsgrad/decay)
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, int64_t n, float lr,
                                                   float b1, float b2, float eps, const int32_t* __restrict__ step) {
  const float t = (float)(*step + 1);
  const float bc1 = 1.f - powf(b1, t), bc2 = 1.f - powf(b2, t);
  const float step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= step_size * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
  }
}
__global__ void adam_tick_kernel(int32_t* step) { *step += 1; }

// dY = dOut * [Xout > 0] * inv_keep over n_vec float4s (Xout = dropout(relu(Y)) > 0 <=> ReLU-active and kept)
__global__ void __launch_bounds__(256) relu_dropout_bwd_kernel(const float4* dOut, const float4* __restrict__ Xout,
                                                               int64_t n_vec, float inv_keep, float4* dY) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 d = dOut[i], x = __ldg(Xout + i);
    dY[i] = make_float4(x.x > 0.f ? d.x * inv_keep : 0.f, x.y > 0.f ? d.y * inv_keep : 0.f,
                        x.z > 0.f ? d.z * inv_keep : 0.f, x.w > 0.f ? d.w * inv_keep : 0.f);
  }
}

// The same with an added upstream gradient: dY = (dOut + dExtra) * [Xout > 0] * inv_keep, add then scale.  dExtra is an
// unpadded row-strided [n, K_extra] matrix (scalar loads: its rows need not be 16-byte aligned); columns at or past
// K_extra add 0.
__global__ void __launch_bounds__(256) relu_dropout_bwd_add_kernel(const float4* dOut, const float* __restrict__ dExtra,
                                                                   int64_t ld_extra, int64_t K_extra,
                                                                   const float4* __restrict__ Xout, int64_t n_vec,
                                                                   int64_t K_vec, float inv_keep, float4* dY) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / K_vec, c = (i - row * K_vec) * 4;
    const float* e = dExtra + row * ld_extra;
    const float4 d = dOut[i], x = __ldg(Xout + i);
    const float s0 = d.x + (c + 0 < K_extra ? __ldg(e + c + 0) : 0.f), s1 = d.y + (c + 1 < K_extra ? __ldg(e + c + 1) : 0.f);
    const float s2 = d.z + (c + 2 < K_extra ? __ldg(e + c + 2) : 0.f), s3 = d.w + (c + 3 < K_extra ? __ldg(e + c + 3) : 0.f);
    dY[i] = make_float4(x.x > 0.f ? s0 * inv_keep : 0.f, x.y > 0.f ? s1 * inv_keep : 0.f,
                        x.z > 0.f ? s2 * inv_keep : 0.f, x.w > 0.f ? s3 * inv_keep : 0.f);
  }
}

static inline int grid_for(int64_t n_items, int per_cta, int cap = 148 * 8) {
  int64_t g = (n_items + per_cta - 1) / per_cta;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace b200gnn

using namespace b200gnn;

static bool rows_ok(int64_t n_rows, int64_t K) { return n_rows >= 0 && K > 0 && K % 4 == 0 && K <= 1024; }

extern "C" int64_t b200gnn_rows_slots(int64_t n_rows) {
  // one slot per CTA; ~2 CTAs per SM keeps the partial buffer small and the reduction order fixed
  int64_t s = (n_rows + 255) / 256;
  if (s > 148 * 4) s = 148 * 4;
  return s < 1 ? 1 : s;
}

extern "C" int b200gnn_col_stats_f32(const float* Y, int64_t n_rows, int64_t K, float* partial, int64_t slots,
                                     void* stream) {
  if (!rows_ok(n_rows, K) || !Y || !partial || slots < 1 || !aligned_to(Y, 16)) return B200GNN_ERR_BAD_ARG;
  col_stats4_kernel<<<(int)slots, ROWS_THREADS, 2 * K * sizeof(float), (cudaStream_t)stream>>>(Y, n_rows, (int)K, partial,
                                                                                             (int)slots);
  return check_launch();
}

extern "C" int b200gnn_bn_finalize_f32(const float* partial, int64_t slots, int64_t K, int64_t n_rows,
                                       const float* gamma, const float* beta, float eps, float momentum,
                                       float* running_mean, float* running_var, float* mean_out, float* invstd_out,
                                       float* scale_out, float* shift_out, void* stream) {
  if (!partial || slots < 1 || K <= 0 || n_rows <= 0 || !gamma || !beta || !mean_out || !invstd_out || !scale_out ||
      !shift_out || ((running_mean == nullptr) != (running_var == nullptr)))
    return B200GNN_ERR_BAD_ARG;
  bn_finalize_kernel<<<(int)((K + FIN_COLS - 1) / FIN_COLS), 256, 0, (cudaStream_t)stream>>>(
      partial, (int)slots, (int)K, n_rows, gamma, beta, eps, momentum, running_mean, running_var, mean_out, invstd_out,
      scale_out, shift_out);
  return check_launch();
}

extern "C" int b200gnn_affine_relu_dropout_f32(const float* Y, float* out, int64_t n_rows, int64_t K,
                                               const float* scale, const float* shift, int relu, float p, uint64_t seed,
                                               uint64_t offset, const int32_t* step_dev, uint64_t step_mul,
                                               uint64_t row_offset, void* stream) {
  if (!rows_ok(n_rows, K) || !Y || !out || p < 0.f || p >= 1.f || ((scale == nullptr) != (shift == nullptr)) ||
      !aligned_to(Y, 16) || !aligned_to(out, 16))
    return B200GNN_ERR_BAD_ARG;
  if (n_rows == 0) return B200GNN_OK;
  const int64_t n_vec = n_rows * (K / 4);
  uint32_t thr16 = 0;
  if (dropout_p16(p, thr16))
    affine_relu_dropout_kernel<true><<<grid_for((n_vec + 1) / 2 + 1, 256 * 2), 256, 0, (cudaStream_t)stream>>>(
        Y, out, n_vec, (int)(K / 4), scale, shift, relu, p, thr16, seed, offset, step_dev, step_mul,
        row_offset * (uint64_t)(K / 4));
  else
    affine_relu_dropout_kernel<false><<<grid_for(n_vec, 256 * 4), 256, 0, (cudaStream_t)stream>>>(
        Y, out, n_vec, (int)(K / 4), scale, shift, relu, p, 0u, seed, offset, step_dev, step_mul,
        row_offset * (uint64_t)(K / 4));
  return check_launch();
}

// Block form of the pass above (node-parallel engine): rows are nodes rowmap[r] (or r + row_offset), columns are
// [col_offset, col_offset + K) of a K_global-wide activation matrix; masks equal the single-GPU ones elementwise.
static int mapped_launch(const float* Y, float* out, int64_t n_rows, int64_t K, const float* scale, const float* shift, int relu,
                         float p, uint64_t seed, uint64_t offset, const int32_t* step_dev, uint64_t step_mul, const int32_t* rowmap,
                         uint64_t row_offset, int64_t K_global, int64_t col_offset, const RowScatter& sc, void* stream) {
  if (!rows_ok(n_rows, K) || !Y || !out || p < 0.f || p >= 1.f || ((scale == nullptr) != (shift == nullptr)) ||
      !aligned_to(Y, 16) || !aligned_to(out, 16) || K_global < K || K_global % 4 || col_offset < 0 || col_offset % 4 ||
      col_offset + K > K_global)
    return B200GNN_ERR_BAD_ARG;
  if (n_rows == 0) return B200GNN_OK;
  const int nvec_l = (int)(K / 4);
  const uint64_t nvec_g = (uint64_t)(K_global / 4), cv_off = (uint64_t)(col_offset / 4);
  const int paired = (nvec_l % 2 == 0 && nvec_g % 2 == 0 && cv_off % 2 == 0) ? 1 : 0;
  const int64_t n_vec = n_rows * nvec_l;
  uint32_t thr16 = 0;
  if (dropout_p16(p, thr16))
    affine_relu_dropout_mapped_kernel<true><<<grid_for(paired ? n_vec / 2 : n_vec, 256 * 2), 256, 0, (cudaStream_t)stream>>>(
        Y, out, n_rows, nvec_l, scale, shift, relu, p, thr16, seed, offset, step_dev, step_mul, rowmap, row_offset, nvec_g,
        cv_off, paired, sc);
  else
    affine_relu_dropout_mapped_kernel<false><<<grid_for(n_vec, 256 * 4), 256, 0, (cudaStream_t)stream>>>(
        Y, out, n_rows, nvec_l, scale, shift, relu, p, 0u, seed, offset, step_dev, step_mul, rowmap, row_offset, nvec_g,
        cv_off, 0, sc);
  return check_launch();
}

// Block form of the pass above (node-parallel engine): rows are nodes rowmap[r] (or r + row_offset), columns are
// [col_offset, col_offset + K) of a K_global-wide activation matrix; masks equal the single-GPU ones elementwise.
extern "C" int b200gnn_affine_relu_dropout_mapped_f32(const float* Y, float* out, int64_t n_rows, int64_t K,
                                                      const float* scale, const float* shift, int relu, float p,
                                                      uint64_t seed, uint64_t offset, const int32_t* step_dev,
                                                      uint64_t step_mul, const int32_t* rowmap, uint64_t row_offset,
                                                      int64_t K_global, int64_t col_offset, void* stream) {
  RowScatter sc;
  sc.n = 0; sc.ld = 0; sc.col = 0;
  return mapped_launch(Y, out, n_rows, K, scale, shift, relu, p, seed, offset, step_dev, step_mul, rowmap, row_offset, K_global,
                       col_offset, sc, stream);
}

// ... and with the C->R layout exchange fused: every output row is ALSO stored to the R-layout buffer of the rank that owns
// the node (dst_ptrs[q] + (r - row_off[q]) * ld_dst + col_offset; HOST arrays, peer-mapped pointers).
extern "C" int b200gnn_affine_relu_dropout_scatter_f32(const float* Y, float* out, int64_t n_rows, int64_t K,
                                                       const float* scale, const float* shift, int relu, float p,
                                                       uint64_t seed, uint64_t offset, const int32_t* step_dev,
                                                       uint64_t step_mul, const int32_t* rowmap, uint64_t row_offset,
                                                       int64_t K_global, int64_t col_offset, float* const* dst_ptrs,
                                                       const int32_t* row_off, int32_t world, int64_t ld_dst, void* stream) {
  if (!dst_ptrs || !row_off || world <= 0 || world > 16 || ld_dst < K_global || ld_dst % 4 || row_off[0] != 0 ||
      row_off[world] != n_rows)
    return B200GNN_ERR_BAD_ARG;
  RowScatter sc;
  sc.n = world; sc.ld = ld_dst; sc.col = col_offset;
  for (int q = 0; q < world; ++q) {
    if (!dst_ptrs[q] || !aligned_to(dst_ptrs[q], 16) || row_off[q + 1] < row_off[q]) return B200GNN_ERR_BAD_ARG;
    sc.ptr[q] = dst_ptrs[q]; sc.off[q] = row_off[q];
  }
  sc.off[world] = row_off[world];
  return mapped_launch(Y, out, n_rows, K, scale, shift, relu, p, seed, offset, step_dev, step_mul, rowmap, row_offset, K_global,
                       col_offset, sc, stream);
}

extern "C" int b200gnn_dropout_mask_u8(uint8_t* mask, int64_t n_rows, int64_t K, float p, uint64_t seed,
                                       uint64_t offset, void* stream) {
  if (!rows_ok(n_rows, K) || !mask || p < 0.f || p >= 1.f) return B200GNN_ERR_BAD_ARG;
  if (n_rows == 0) return B200GNN_OK;
  const int64_t n_vec = n_rows * (K / 4);
  uint32_t thr16 = 0;
  const int p16 = dropout_p16(p, thr16) ? 1 : 0;
  dropout_mask_kernel<<<grid_for(n_vec, 256 * 4), 256, 0, (cudaStream_t)stream>>>(mask, n_vec, p, p16, thr16, seed, offset);
  return check_launch();
}

extern "C" int b200gnn_relu_dropout_bwd_f32(const float* dOut, const float* Xout, int64_t n_rows, int64_t K, float p, float* dY,
                                            void* stream) {
  if (!rows_ok(n_rows, K) || !dOut || !Xout || !dY || p < 0.f || p >= 1.f || !aligned_to(dOut, 16) || !aligned_to(Xout, 16) ||
      !aligned_to(dY, 16))
    return B200GNN_ERR_BAD_ARG;
  if (n_rows == 0) return B200GNN_OK;
  const int64_t n_vec = n_rows * (K / 4);
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  relu_dropout_bwd_kernel<<<grid_for(n_vec, 256 * 4), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(dOut), reinterpret_cast<const float4*>(Xout), n_vec, inv_keep, reinterpret_cast<float4*>(dY));
  return check_launch();
}

extern "C" int b200gnn_relu_dropout_bwd_add_f32(const float* dOut, const float* dExtra, int64_t ld_extra, int64_t K_extra,
                                                const float* Xout, int64_t n_rows, int64_t K, float p, float* dY, void* stream) {
  if (!rows_ok(n_rows, K) || p < 0.f || p >= 1.f || K_extra < 0 || K_extra > K || ld_extra < K_extra) return B200GNN_ERR_BAD_ARG;
  if (n_rows == 0) return B200GNN_OK;                  // empty tensors may come with null pointers
  if (!dOut || !Xout || !dY || (K_extra > 0 && !dExtra) || !aligned_to(dOut, 16) || !aligned_to(Xout, 16) || !aligned_to(dY, 16))
    return B200GNN_ERR_BAD_ARG;
  const int64_t n_vec = n_rows * (K / 4);
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  relu_dropout_bwd_add_kernel<<<grid_for(n_vec, 256 * 4), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(dOut), dExtra, ld_extra, K_extra, reinterpret_cast<const float4*>(Xout), n_vec, K / 4,
      inv_keep, reinterpret_cast<float4*>(dY));
  return check_launch();
}

// phase 1: partial[slots][2][K] = per-slot column sums of dz and dz*xhat
extern "C" int b200gnn_bn_act_bwd_reduce_f32(const float* dOut, const float* Xout, const float* Y, const float* mean,
                                             const float* invstd, int64_t n_rows, int64_t K, float p, float* partial,
                                             int64_t slots, void* stream) {
  if (!rows_ok(n_rows, K) || n_rows == 0 || !dOut || !Xout || !Y || !mean || !invstd || !partial || slots < 1 ||
      p < 0.f || p >= 1.f)
    return B200GNN_ERR_BAD_ARG;
  if (ROWS_THREADS / (K / 4) < 1) return B200GNN_ERR_UNSUPPORTED;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  bn_act_bwd_reduce_kernel<<<(int)slots, ROWS_THREADS, 2 * K * sizeof(float), (cudaStream_t)stream>>>(
      dOut, Xout, Y, mean, invstd, n_rows, (int)K, inv_keep, partial, (int)slots);
  return check_launch();
}

// phase 2: sums[sum_slots][2][K] (local partials, or one slot of globally reduced sums) + the normalisation count
// n_norm (global row count) -> dgamma, dbeta, dY (and dbias = column sums of the LOCAL dY rows if requested).
// Xout == NULL: dOut already holds dz = dOut * [Xout > 0] / (1-p) (written by b200gnn_gemm_tf32x3_bnbwd_f32, whose
// partial buffer is then `sums`); dY may alias dOut.
extern "C" int b200gnn_bn_act_bwd_apply_f32(const float* dOut, const float* Xout, const float* Y, const float* mean,
                                            const float* invstd, const float* gamma, const float* sums,
                                            int64_t sum_slots, int64_t n_norm, int64_t n_rows, int64_t K, float p,
                                            float* dY, float* dgamma, float* dbeta, float* dbias, float* partial,
                                            int64_t slots, float* coef, void* stream) {
  if (!rows_ok(n_rows, K) || n_rows == 0 || !dOut || !Y || !mean || !invstd || !gamma || !sums || !dY ||
      !dgamma || !dbeta || !partial || !coef || slots < 1 || sum_slots < 1 || n_norm < 1 || p < 0.f || p >= 1.f)
    return B200GNN_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const size_t smem = 2 * K * sizeof(float);
  int rc;
  bn_bwd_finalize_kernel<<<(int)((K + FIN_COLS - 1) / FIN_COLS), 256, 0, st>>>(sums, (int)sum_slots, (int)K, n_norm, gamma,
                                                                              invstd, dgamma, dbeta, coef);
  if ((rc = check_launch())) return rc;
  if (Xout)
    bn_act_bwd_apply_kernel<false><<<(int)slots, ROWS_THREADS, smem, st>>>(dOut, Xout, Y, mean, invstd, coef, n_rows, (int)K,
                                                                          inv_keep, dY, dbias ? partial : nullptr, (int)slots);
  else
    bn_act_bwd_apply_kernel<true><<<(int)slots, ROWS_THREADS, smem, st>>>(dOut, nullptr, Y, mean, invstd, coef, n_rows, (int)K,
                                                                         inv_keep, dY, dbias ? partial : nullptr, (int)slots);
  if ((rc = check_launch())) return rc;
  if (dbias) {
    colsum_finalize_kernel<<<(int)((K + FIN_COLS - 1) / FIN_COLS), 256, 0, st>>>(partial, (int)slots, (int)K, dbias);
    if ((rc = check_launch())) return rc;
  }
  return B200GNN_OK;
}

extern "C" int b200gnn_bn_act_bwd_f32(const float* dOut, const float* Xout, const float* Y, const float* mean,
                                      const float* invstd, const float* gamma, int64_t n_rows, int64_t K, float p,
                                      float* dY, float* dgamma, float* dbeta, float* dbias, float* partial,
                                      int64_t slots, float* coef, void* stream) {
  int rc = b200gnn_bn_act_bwd_reduce_f32(dOut, Xout, Y, mean, invstd, n_rows, K, p, partial, slots, stream);
  if (rc) return rc;
  return b200gnn_bn_act_bwd_apply_f32(dOut, Xout, Y, mean, invstd, gamma, partial, slots, n_rows, n_rows, K, p, dY,
                                      dgamma, dbeta, dbias, partial, slots, coef, stream);
}

// out[2K] = sum over slots of partial[slot][2K]  (fp64 accumulation; used before a cross-rank all-reduce)
extern "C" int b200gnn_partial_reduce_f32(const float* partial, int64_t slots, int64_t K2, float* out, void* stream) {
  if (!partial || !out || slots < 1 || K2 < 1) return B200GNN_ERR_BAD_ARG;
  partial_reduce_kernel<<<(int)((K2 + FIN_COLS - 1) / FIN_COLS), 256, 0, (cudaStream_t)stream>>>(partial, (int)slots, (int)K2,
                                                                                               out);
  return check_launch();
}

extern "C" int b200gnn_col_sum_f32(const float* Y, int64_t n_rows, int64_t K, float* out, float* partial,
                                   int64_t slots, void* stream) {
  if (!rows_ok(n_rows, K) || !Y || !out || !partial || slots < 1) return B200GNN_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  col_stats4_kernel<<<(int)slots, ROWS_THREADS, 2 * K * sizeof(float), st>>>(Y, n_rows, (int)K, partial, (int)slots);
  if ((rc = check_launch())) return rc;
  colsum_finalize_kernel<<<(int)((K + FIN_COLS - 1) / FIN_COLS), 256, 0, st>>>(partial, (int)slots, (int)K, out);
  return check_launch();
}

extern "C" int b200gnn_adam_step_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                     float lr, float beta1, float beta2, float eps, int32_t* step, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || !step || n < 0) return B200GNN_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (n > 0) {
    adam_kernel<<<grid_for(n, 256), 256, 0, st>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step);
    if ((rc = check_launch())) return rc;
  }
  adam_tick_kernel<<<1, 1, 0, st>>>(step);
  return check_launch();
}
