// Memory-bound kernels of the UNet step: BatchNorm(+ReLU)(+MaxPool) apply and backward, max-pool,
// bilinear x2 upsample, layout gathers and channel-slice copies.  All are HBM-bound: coalesced
// 16-byte accesses over NHWC (8 channels per thread when C % 8 == 0), grid-stride loops sized to
// the SM count, warp-shuffle + shared-memory reductions, fp64 cross-block accumulation.
#include "common.cuh"

namespace ub {

// ------------------------------------------------------------------------------------------
// vector helpers: V = 8 (16-byte path) or V = 1 (any C / alignment)
// ------------------------------------------------------------------------------------------
template <typename T, int V>
__device__ __forceinline__ void ldv(const T* p, float v[V]) {
  if constexpr (V == 8) {
    load8(p, v);
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = Elem<T>::ld(p + i);
  }
}
template <typename T, int V>
__device__ __forceinline__ void stv(T* p, const float v[V]) {
  if constexpr (V == 8) {
    store8(p, v);
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) Elem<T>::st(p + i, v[i]);
  }
}
template <int V>
__device__ __forceinline__ void ldf(const float* p, float v[V]) {
#pragma unroll
  for (int i = 0; i < V; ++i) v[i] = __ldg(p + i);
}

static inline int grid_for(int64_t work, int threads, int per_sm = 8) {
  int64_t b = (work + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * per_sm;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

struct CsGeom {
  int CVB, gy;
  unsigned gx;
};
static CsGeom cs_geom(int CV, int64_t items, int per_thread, int max_cvb = 256) {
  CsGeom g;
  g.CVB = CV < max_cvb ? CV : max_cvb;
  const int lanes = 256 / g.CVB;
  g.gy = (CV + g.CVB - 1) / g.CVB;
  int64_t gx = (items + (int64_t)lanes * per_thread - 1) / ((int64_t)lanes * per_thread);
  int64_t cap = (int64_t)sm_count() * 8 / g.gy;
  if (cap < 1) cap = 1;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  g.gx = (unsigned)gx;
  return g;
}

template <typename T>
static bool vec_ok(int C, std::initializer_list<int64_t> lds, std::initializer_list<const void*> ptrs) {
  if (C % 8) return false;
  for (int64_t l : lds)
    if (l % 8) return false;
  for (const void* p : ptrs)
    if (p && (reinterpret_cast<uintptr_t>(p) % (8 * sizeof(T)))) return false;
  return true;
}

// ------------------------------------------------------------------------------------------
// BN finalize  (forward statistics -> scale/shift, running stats)
// ------------------------------------------------------------------------------------------
__global__ void bn_finalize_kernel(const double* __restrict__ stats, double inv_count, double unbias,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float eps, float momentum, float* running_mean, float* running_var,
                                   float* save_mean, float* save_invstd, float* scale, float* shift, int C,
                                   long long* num_batches_tracked) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;      // nn.BatchNorm2d's step counter, same launch
  if (c >= C) return;
  double mean = stats[c] * inv_count;
  double var = stats[C + c] * inv_count - mean * mean;
  if (var < 0) var = 0;
  float invstd = (float)(1.0 / sqrt(var + (double)eps));
  float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  float sc = g * invstd;
  save_mean[c] = (float)mean;
  save_invstd[c] = invstd;
  scale[c] = sc;
  shift[c] = b - (float)mean * sc;
  if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
  if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)(var * unbias);
}

__global__ void bn_eval_coeffs_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ rm, const float* __restrict__ rv, float eps,
                                      float* scale, float* shift, float* save_mean, float* save_invstd, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float invstd = 1.0f / sqrtf(rv[c] + eps);
  float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  float sc = g * invstd;
  scale[c] = sc;
  shift[c] = b - rm[c] * sc;
  if (save_mean) save_mean[c] = rm[c];
  if (save_invstd) save_invstd[c] = invstd;
}

// ------------------------------------------------------------------------------------------
// BN apply + ReLU (+ 2x2 max-pool)
// ------------------------------------------------------------------------------------------
// Channel-stationary mapping used by the BN kernels: a block of 256 threads = CVB channel vectors x
// LANES pixel lanes (blockIdx.y selects the channel-vector block when C is wide).  Each thread keeps
// its per-channel coefficients in registers and streams over pixels with 4 independent 16-byte loads
// in flight; a warp touches LANES consecutive pixels x CVB vectors = one contiguous run of NHWC.
struct CsThread {
  int cv, lane, lanes;
  bool active;
};
__device__ __forceinline__ CsThread cs_thread(int CV, int CVB) {
  CsThread t;
  t.lanes = blockDim.x / CVB;
  t.lane = threadIdx.x / CVB;
  t.cv = blockIdx.y * CVB + threadIdx.x % CVB;
  t.active = t.cv < CV && t.lane < t.lanes;
  return t;
}

template <typename T, int V>
__global__ void __launch_bounds__(256)
bn_relu_apply_kernel(const T* __restrict__ y, int64_t ld_y, const float* __restrict__ scale,
                     const float* __restrict__ shift, T* __restrict__ z, int64_t ld_z, int64_t npix, int CV,
                     int CVB) {
  const CsThread t = cs_thread(CV, CVB);
  if (!t.active) return;
  const int c = t.cv * V;
  float sc[V], sh[V];
  ldf<V>(scale + c, sc);
  ldf<V>(shift + c, sh);
  const int64_t stride = (int64_t)gridDim.x * t.lanes;
  int64_t p = (int64_t)blockIdx.x * t.lanes + t.lane;
  for (; p + 3 * stride < npix; p += 4 * stride) {
    float v[4][V];
#pragma unroll
    for (int u = 0; u < 4; ++u) ldv<T, V>(y + (p + u * stride) * ld_y + c, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int i = 0; i < V; ++i) v[u][i] = fmaxf(fmaf(v[u][i], sc[i], sh[i]), 0.f);
      stv<T, V>(z + (p + u * stride) * ld_z + c, v[u]);
    }
  }
  for (; p < npix; p += stride) {
    float v[V];
    ldv<T, V>(y + p * ld_y + c, v);
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = fmaxf(fmaf(v[i], sc[i], sh[i]), 0.f);
    stv<T, V>(z + p * ld_z + c, v);
  }
}

__device__ __forceinline__ float pool_max(float m, float v) { return (v > m || v != v) ? v : m; }

// one thread = one 2x2 window (ceil grid, so odd rows/cols still get their z written) x V channels
template <typename T, int V>
__global__ void __launch_bounds__(256)
bn_relu_apply_pool_kernel(const T* __restrict__ y, int64_t ld_y, const float* __restrict__ scale,
                          const float* __restrict__ shift, T* __restrict__ z, int64_t ld_z, T* __restrict__ pooled,
                          int64_t ld_p, int B, int H, int W, int CV, int CVB) {
  const CsThread t = cs_thread(CV, CVB);
  if (!t.active) return;
  const int c = t.cv * V;
  float sc[V], sh[V];
  ldf<V>(scale + c, sc);
  ldf<V>(shift + c, sh);
  const int Hc = (H + 1) >> 1, Wc = (W + 1) >> 1, Hp = H >> 1, Wp = W >> 1;
  const int64_t nwin = (int64_t)B * Hc * Wc;
  const int64_t stride = (int64_t)gridDim.x * t.lanes;
  for (int64_t wdx = (int64_t)blockIdx.x * t.lanes + t.lane; wdx < nwin; wdx += stride) {
    const int j = (int)(wdx % Wc);
    int64_t r = wdx / Wc;
    const int i = (int)(r % Hc);
    const int n = (int)(r / Hc);
    const bool full = (2 * i + 1 < H) && (2 * j + 1 < W);
    float v[4][V], m[V];
    if (full) {
      const int64_t p00 = ((int64_t)n * H + 2 * i) * W + 2 * j;
      ldv<T, V>(y + p00 * ld_y + c, v[0]);
      ldv<T, V>(y + (p00 + 1) * ld_y + c, v[1]);
      ldv<T, V>(y + (p00 + W) * ld_y + c, v[2]);
      ldv<T, V>(y + (p00 + W + 1) * ld_y + c, v[3]);
#pragma unroll
      for (int k = 0; k < V; ++k) m[k] = -INFINITY;
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int k = 0; k < V; ++k) {
          v[q][k] = Elem<T>::round(fmaxf(fmaf(v[q][k], sc[k], sh[k]), 0.f));
          m[k] = pool_max(m[k], v[q][k]);
        }
      stv<T, V>(z + p00 * ld_z + c, v[0]);
      stv<T, V>(z + (p00 + 1) * ld_z + c, v[1]);
      stv<T, V>(z + (p00 + W) * ld_z + c, v[2]);
      stv<T, V>(z + (p00 + W + 1) * ld_z + c, v[3]);
      stv<T, V>(pooled + (((int64_t)n * Hp + i) * Wp + j) * ld_p + c, m);
    } else {
      for (int q = 0; q < 4; ++q) {
        const int h = 2 * i + (q >> 1), w = 2 * j + (q & 1);
        if (h < H && w < W) {
          const int64_t p = ((int64_t)n * H + h) * W + w;
          ldv<T, V>(y + p * ld_y + c, v[0]);
#pragma unroll
          for (int k = 0; k < V; ++k) v[0][k] = fmaxf(fmaf(v[0][k], sc[k], sh[k]), 0.f);
          stv<T, V>(z + p * ld_z + c, v[0]);
        }
      }
    }
  }
}

template <typename T, int V>
__global__ void maxpool2_fwd_kernel(const T* __restrict__ x, int64_t ld_x, T* __restrict__ p, int64_t ld_p, int B,
                                    int H, int W, int CV) {
  const int Hp = H >> 1, Wp = W >> 1;
  const int64_t total = (int64_t)B * Hp * Wp * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(idx % CV);
    int64_t r = idx / CV;
    int j = (int)(r % Wp);
    r /= Wp;
    int i = (int)(r % Hp);
    int n = (int)(r / Hp);
    int c = cv * V;
    float m[V];
#pragma unroll
    for (int k = 0; k < V; ++k) m[k] = -INFINITY;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        float v[V];
        ldv<T, V>(x + (((int64_t)n * H + 2 * i + a) * W + 2 * j + b) * ld_x + c, v);
#pragma unroll
        for (int k = 0; k < V; ++k) m[k] = pool_max(m[k], v[k]);
      }
    stv<T, V>(p + (((int64_t)n * Hp + i) * Wp + j) * ld_p + c, m);
  }
}

// gradient goes to the FIRST max of the window in row-major order (ATen rule: val > max || isnan)
template <typename T, int V, bool ACC>
__global__ void maxpool2_bwd_kernel(const T* __restrict__ x, int64_t ld_x, const T* __restrict__ gp, int64_t ld_gp,
                                    T* __restrict__ gx, int64_t ld_gx, int B, int H, int W, int CV) {
  const int Hc = (H + 1) >> 1, Wc = (W + 1) >> 1, Hp = H >> 1, Wp = W >> 1;
  const int64_t total = (int64_t)B * Hc * Wc * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(idx % CV);
    int64_t r = idx / CV;
    int j = (int)(r % Wc);
    r /= Wc;
    int i = (int)(r % Hc);
    int n = (int)(r / Hc);
    int c = cv * V;
    const bool full = (i < Hp && j < Wp);
    float g[V], m[V];
    int arg[V];
#pragma unroll
    for (int k = 0; k < V; ++k) { m[k] = -INFINITY; arg[k] = 0; g[k] = 0.f; }
    if (full) {
      ldv<T, V>(gp + (((int64_t)n * Hp + i) * Wp + j) * ld_gp + c, g);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float v[V];
        ldv<T, V>(x + (((int64_t)n * H + 2 * i + (q >> 1)) * W + 2 * j + (q & 1)) * ld_x + c, v);
#pragma unroll
        for (int k = 0; k < V; ++k)
          if (v[k] > m[k] || v[k] != v[k]) { m[k] = v[k]; arg[k] = q; }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int h = 2 * i + (q >> 1), w = 2 * j + (q & 1);
      if (h < H && w < W) {
        T* dst = gx + (((int64_t)n * H + h) * W + w) * ld_gx + c;
        float o[V];
        if (ACC) ldv<T, V>(dst, o);
#pragma unroll
        for (int k = 0; k < V; ++k) {
          float t = (full && arg[k] == q) ? g[k] : 0.f;
          o[k] = ACC ? o[k] + t : t;
        }
        stv<T, V>(dst, o);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// BN + ReLU backward
// ------------------------------------------------------------------------------------------
// block = 256 threads = CVB channel-vectors x LANES pixel lanes; blockIdx.y = channel-vector block.
template <typename T, int V>
__global__ void __launch_bounds__(256)
bn_relu_bwd_reduce_kernel(const T* __restrict__ gz, int64_t ld_gz, const T* __restrict__ y, int64_t ld_y,
                          const float* __restrict__ scale, const float* __restrict__ shift,
                          const float* __restrict__ mean, const float* __restrict__ invstd,
                          double* __restrict__ sums, int64_t npix, int C, int CV, int CVB) {
  constexpr int RED = (V == 8) ? 512 : 256;      // 4 KB: small enough to co-reside with a tensor kernel that holds ~200 KB
  __shared__ float red[2][RED];
  const CsThread t = cs_thread(CV, CVB);
  const int cvl = threadIdx.x % CVB;
  float s0[V], s1[V];
#pragma unroll
  for (int k = 0; k < V; ++k) s0[k] = s1[k] = 0.f;
  if (t.active) {
    const int c = t.cv * V;
    float sc[V], sh[V], mu[V], is[V];
    ldf<V>(scale + c, sc);
    ldf<V>(shift + c, sh);
    ldf<V>(mean + c, mu);
    ldf<V>(invstd + c, is);
    const int64_t stride = (int64_t)gridDim.x * t.lanes;
    int64_t p = (int64_t)blockIdx.x * t.lanes + t.lane;
    for (; p + stride < npix; p += 2 * stride) {
      float g[2][V], v[2][V];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        ldv<T, V>(gz + (p + u * stride) * ld_gz + c, g[u]);
        ldv<T, V>(y + (p + u * stride) * ld_y + c, v[u]);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int k = 0; k < V; ++k) {
          float gg = (fmaf(v[u][k], sc[k], sh[k]) > 0.f) ? g[u][k] : 0.f;
          s0[k] += gg;
          s1[k] += gg * ((v[u][k] - mu[k]) * is[k]);
        }
    }
    for (; p < npix; p += stride) {
      float g[V], v[V];
      ldv<T, V>(gz + p * ld_gz + c, g);
      ldv<T, V>(y + p * ld_y + c, v);
#pragma unroll
      for (int k = 0; k < V; ++k) {
        float gg = (fmaf(v[k], sc[k], sh[k]) > 0.f) ? g[k] : 0.f;
        s0[k] += gg;
        s1[k] += gg * ((v[k] - mu[k]) * is[k]);
      }
    }
  }
  // reduce over pixel lanes through shared memory, `chunk` lanes at a time: red[.][lane][cvl*V + k]
  const int lanes = t.lanes, lane = t.lane;
  const int row = CVB * V;
  const int chunk = RED / row;   // >= 1 by construction (row <= RED)
  // (row <= RED = 2 * blockDim: a thread owns at most two columns; it carries their sums over the chunks and
  // issues ONE pair of fp64 atomics per column per block)
  float fa[2] = {0.f, 0.f}, fb[2] = {0.f, 0.f};
  for (int base = 0; base < lanes; base += chunk) {
    __syncthreads();
    if (t.active && lane >= base && lane < base + chunk) {
#pragma unroll
      for (int k = 0; k < V; ++k) {
        red[0][(lane - base) * row + cvl * V + k] = s0[k];
        red[1][(lane - base) * row + cvl * V + k] = s1[k];
      }
    }
    __syncthreads();
    const int nl = lanes - base < chunk ? lanes - base : chunk;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int e = threadIdx.x + u * blockDim.x;
      if (e < row)
        for (int l = 0; l < nl; ++l) { fa[u] += red[0][l * row + e]; fb[u] += red[1][l * row + e]; }
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int e = threadIdx.x + u * blockDim.x;
    const int ch = blockIdx.y * CVB * V + e;
    if (e < row && ch < C) {
      atomicAdd(sums + ch, (double)fa[u]);
      atomicAdd(sums + C + ch, (double)fb[u]);
    }
  }
}

__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sums, double inv_count, int training,
                                       float* dgamma, float* dbeta, float* coef, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double sg = sums[c], sgx = sums[C + c];
  if (dbeta) dbeta[c] = (float)sg;
  if (dgamma) dgamma[c] = (float)sgx;
  coef[c] = training ? (float)(sg * inv_count) : 0.f;
  coef[C + c] = training ? (float)(sgx * inv_count) : 0.f;
}


// Max-pool backward accumulated into the skip gradient (as above, ACC) + the reduction pass of the BatchNorm/ReLU
// backward of the layer that produced x = relu(bn(y)): an encoder stage's output feeds the pool AND the skip
// connection, its gradient is final only after this kernel, and the BatchNorm backward reads it right away -- so the
// sums ride here (one extra read of y instead of a pass over gx and y).  Channel-stationary: a thread owns V channels
// (coefficients and sums in registers) and walks 2x2 windows; block reduction like bn_relu_bwd_reduce_kernel.
template <typename T, int V>
__global__ void __launch_bounds__(256)
maxpool2_bwd_bnreduce_kernel(const T* __restrict__ x, int64_t ld_x, const T* __restrict__ gp, int64_t ld_gp,
                             T* __restrict__ gx, int64_t ld_gx, const T* __restrict__ y, int64_t ld_y,
                             const float* __restrict__ scale, const float* __restrict__ shift,
                             const float* __restrict__ mean, const float* __restrict__ invstd,
                             double* __restrict__ sums, int B, int H, int W, int C, int CV, int CVB) {
  constexpr int RED = (V == 8) ? 512 : 256;
  __shared__ float red[2][RED];
  const CsThread t = cs_thread(CV, CVB);
  const int cvl = threadIdx.x % CVB;
  float s0[V], s1[V];
#pragma unroll
  for (int k = 0; k < V; ++k) s0[k] = s1[k] = 0.f;
  if (t.active) {
    const int c = t.cv * V;
    float sc[V], sh[V], mu[V], is[V];
    ldf<V>(scale + c, sc);
    ldf<V>(shift + c, sh);
    ldf<V>(mean + c, mu);
    ldf<V>(invstd + c, is);
    const int Hc = (H + 1) >> 1, Wc = (W + 1) >> 1, Hp = H >> 1, Wp = W >> 1;
    const int64_t nwin = (int64_t)B * Hc * Wc;
    const int64_t stride = (int64_t)gridDim.x * t.lanes;
    for (int64_t wdx = (int64_t)blockIdx.x * t.lanes + t.lane; wdx < nwin; wdx += stride) {
      const int j = (int)(wdx % Wc);
      int64_t r = wdx / Wc;
      const int i = (int)(r % Hc);
      const int n = (int)(r / Hc);
      const bool full = (i < Hp && j < Wp);
      float g[V], m[V];
      int arg[V];
#pragma unroll
      for (int k = 0; k < V; ++k) { m[k] = -INFINITY; arg[k] = 0; g[k] = 0.f; }
      if (full) {
        ldv<T, V>(gp + (((int64_t)n * Hp + i) * Wp + j) * ld_gp + c, g);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float v[V];
          ldv<T, V>(x + (((int64_t)n * H + 2 * i + (q >> 1)) * W + 2 * j + (q & 1)) * ld_x + c, v);
#pragma unroll
          for (int k = 0; k < V; ++k)
            if (v[k] > m[k] || v[k] != v[k]) { m[k] = v[k]; arg[k] = q; }
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int h = 2 * i + (q >> 1), w = 2 * j + (q & 1);
        if (h < H && w < W) {
          const int64_t pix = ((int64_t)n * H + h) * W + w;
          float o[V], yv[V];
          ldv<T, V>(gx + pix * ld_gx + c, o);
          ldv<T, V>(y + pix * ld_y + c, yv);
#pragma unroll
          for (int k = 0; k < V; ++k) o[k] += (full && arg[k] == q) ? g[k] : 0.f;
          stv<T, V>(gx + pix * ld_gx + c, o);
#pragma unroll
          for (int k = 0; k < V; ++k) {
            const float gg = (fmaf(yv[k], sc[k], sh[k]) > 0.f) ? Elem<T>::round(o[k]) : 0.f;      // the gradient as stored
            s0[k] += gg;
            s1[k] += gg * ((yv[k] - mu[k]) * is[k]);
          }
        }
      }
    }
  }
  const int lanes = t.lanes, lane = t.lane;
  const int row = CVB * V;
  const int chunk = RED / row;
  float fa[2] = {0.f, 0.f}, fb[2] = {0.f, 0.f};
  for (int base = 0; base < lanes; base += chunk) {
    __syncthreads();
    if (t.active && lane >= base && lane < base + chunk) {
#pragma unroll
      for (int k = 0; k < V; ++k) {
        red[0][(lane - base) * row + cvl * V + k] = s0[k];
        red[1][(lane - base) * row + cvl * V + k] = s1[k];
      }
    }
    __syncthreads();
    const int nl = lanes - base < chunk ? lanes - base : chunk;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int e = threadIdx.x + u * blockDim.x;
      if (e < row)
        for (int l = 0; l < nl; ++l) { fa[u] += red[0][l * row + e]; fb[u] += red[1][l * row + e]; }
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int e = threadIdx.x + u * blockDim.x;
    const int ch = blockIdx.y * CVB * V + e;
    if (e < row && ch < C) {
      atomicAdd(sums + ch, (double)fa[u]);
      atomicAdd(sums + C + ch, (double)fb[u]);
    }
  }
}

// gy = sc*g*mask + A*(y - mu) + B0 with A = -sc*c1*invstd, B0 = -sc*c0 (per channel, in registers)
template <typename T, int V>
__global__ void __launch_bounds__(256)
bn_relu_bwd_apply_kernel(const T* __restrict__ gz, int64_t ld_gz, const T* __restrict__ y, int64_t ld_y,
                         const float* __restrict__ scale, const float* __restrict__ shift,
                         const float* __restrict__ mean, const float* __restrict__ invstd,
                         const float* __restrict__ coef, T* __restrict__ gy, int64_t ld_gy, int64_t npix, int C,
                         int CV, int CVB) {
  const CsThread t = cs_thread(CV, CVB);
  if (!t.active) return;
  const int c = t.cv * V;
  float sc[V], sh[V], mu[V], A[V], B0[V];
  {
    float is[V], c0[V], c1[V];
    ldf<V>(scale + c, sc);
    ldf<V>(shift + c, sh);
    ldf<V>(mean + c, mu);
    ldf<V>(invstd + c, is);
    ldf<V>(coef + c, c0);
    ldf<V>(coef + C + c, c1);
#pragma unroll
    for (int k = 0; k < V; ++k) { A[k] = -sc[k] * c1[k] * is[k]; B0[k] = -sc[k] * c0[k]; }
  }
  const int64_t stride = (int64_t)gridDim.x * t.lanes;
  int64_t p = (int64_t)blockIdx.x * t.lanes + t.lane;
  for (; p + stride < npix; p += 2 * stride) {
    float g[2][V], v[2][V];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      ldv<T, V>(gz + (p + u * stride) * ld_gz + c, g[u]);
      ldv<T, V>(y + (p + u * stride) * ld_y + c, v[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
#pragma unroll
      for (int k = 0; k < V; ++k) {
        float gg = (fmaf(v[u][k], sc[k], sh[k]) > 0.f) ? g[u][k] : 0.f;
        g[u][k] = fmaf(sc[k], gg, fmaf(A[k], v[u][k] - mu[k], B0[k]));
      }
      stv<T, V>(gy + (p + u * stride) * ld_gy + c, g[u]);
    }
  }
  for (; p < npix; p += stride) {
    float g[V], v[V];
    ldv<T, V>(gz + p * ld_gz + c, g);
    ldv<T, V>(y + p * ld_y + c, v);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      float gg = (fmaf(v[k], sc[k], sh[k]) > 0.f) ? g[k] : 0.f;
      g[k] = fmaf(sc[k], gg, fmaf(A[k], v[k] - mu[k], B0[k]));
    }
    stv<T, V>(gy + p * ld_gy + c, g);
  }
}

// ------------------------------------------------------------------------------------------
// bilinear x2, align_corners=True
// ------------------------------------------------------------------------------------------
struct Lerp { int i0, i1; float w0, w1; };
__device__ __forceinline__ Lerp lerp_coords(int o, int in_size, float s) {
  float src = s * (float)o;
  int i0 = (int)src;
  if (i0 > in_size - 1) i0 = in_size - 1;
  int i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  float l1 = src - (float)i0;
  return {i0, i1, 1.f - l1, l1};
}

template <typename T, int V>
__global__ void upsample2x_fwd_kernel(const T* __restrict__ x, int64_t ld_x, T* __restrict__ y, int64_t ld_y, int B,
                                      int h, int w, int CV, int Hout, int Wout, int off_y, int off_x, float sy,
                                      float sx) {
  const int H2 = 2 * h, W2 = 2 * w;
  const int64_t total = (int64_t)B * H2 * W2 * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(idx % CV);
    int64_t r = idx / CV;
    int ox = (int)(r % W2);
    r /= W2;
    int oy = (int)(r % H2);
    int n = (int)(r / H2);
    int c = cv * V;
    Lerp ly = lerp_coords(oy, h, sy), lx = lerp_coords(ox, w, sx);
    const T* base = x + (int64_t)n * h * w * ld_x + c;
    float v00[V], v01[V], v10[V], v11[V], o[V];
    ldv<T, V>(base + ((int64_t)ly.i0 * w + lx.i0) * ld_x, v00);
    ldv<T, V>(base + ((int64_t)ly.i0 * w + lx.i1) * ld_x, v01);
    ldv<T, V>(base + ((int64_t)ly.i1 * w + lx.i0) * ld_x, v10);
    ldv<T, V>(base + ((int64_t)ly.i1 * w + lx.i1) * ld_x, v11);
#pragma unroll
    for (int k = 0; k < V; ++k)
      o[k] = ly.w0 * (lx.w0 * v00[k] + lx.w1 * v01[k]) + ly.w1 * (lx.w0 * v10[k] + lx.w1 * v11[k]);
    stv<T, V>(y + (((int64_t)n * Hout + oy + off_y) * Wout + ox + off_x) * ld_y + c, o);
  }
}

// gather form of the transpose: each input pixel sums the (<= ~4 x 4) outputs that interpolate from it
__device__ __forceinline__ int lerp_sources(int i, int in_size, float s, int idx[8], float wt[8]) {
  const int out = 2 * in_size;
  int lo = 0, hi = out - 1;
  if (s > 0.f) {
    lo = (int)floorf((float)(i - 1) / s) - 1;
    hi = (int)ceilf((float)(i + 1) / s) + 1;
    if (lo < 0) lo = 0;
    if (hi > out - 1) hi = out - 1;
  }
  int n = 0;
  for (int o = lo; o <= hi && n < 8; ++o) {
    Lerp l = lerp_coords(o, in_size, s);
    float wsum = (l.i0 == i ? l.w0 : 0.f) + (l.i1 == i ? l.w1 : 0.f);
    if ((l.i0 == i || l.i1 == i) && wsum != 0.f) { idx[n] = o; wt[n] = wsum; ++n; }
  }
  return n;
}

template <typename T, int V>
__global__ void upsample2x_bwd_kernel(const T* __restrict__ gy, int64_t ld_gy, T* __restrict__ gx, int64_t ld_gx,
                                      int B, int h, int w, int CV, int Hout, int Wout, int off_y, int off_x,
                                      float sy, float sx) {
  const int64_t total = (int64_t)B * h * w * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(idx % CV);
    int64_t r = idx / CV;
    int ix = (int)(r % w);
    r /= w;
    int iy = (int)(r % h);
    int n = (int)(r / h);
    int c = cv * V;
    int ys[8], xs[8];
    float wy[8], wx[8];
    int ny = lerp_sources(iy, h, sy, ys, wy), nx = lerp_sources(ix, w, sx, xs, wx);
    float acc[V];
#pragma unroll
    for (int k = 0; k < V; ++k) acc[k] = 0.f;
    for (int a = 0; a < ny; ++a)
      for (int b = 0; b < nx; ++b) {
        float g[V];
        ldv<T, V>(gy + (((int64_t)n * Hout + ys[a] + off_y) * Wout + xs[b] + off_x) * ld_gy + c, g);
        float wgt = wy[a] * wx[b];
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = fmaf(wgt, g[k], acc[k]);
      }
    stv<T, V>(gx + (((int64_t)n * h + iy) * w + ix) * ld_gx + c, acc);
  }
}

// ------------------------------------------------------------------------------------------
// layout plumbing
// ------------------------------------------------------------------------------------------
template <typename S, typename D>
__global__ void gather_nhwc_kernel(const S* __restrict__ src, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                                   D* __restrict__ dst, int64_t ld, int B, int C, int H, int W) {
  const int64_t total = (int64_t)B * H * W * C;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(idx % C);
    int64_t p = idx / C;
    int x = (int)(p % W);
    int64_t r = p / W;
    int y = (int)(r % H);
    int n = (int)(r / H);
    Elem<D>::st(dst + p * ld + c, Elem<S>::ld(src + n * sn + c * sc + y * sh + x * sw));
  }
}

// dense NHWC source and destination (what train.py / predict.py hand over: channels_last fp32, any C): a flat dtype
// conversion, 8 elements per thread -- the generic gather above makes three integer divisions per ELEMENT and moved the
// 3-channel 1024 x 1024 input of configs[4] at 0.14 of the copy rate
template <typename S, typename D>
__global__ void __launch_bounds__(256) convert_flat_kernel(const S* __restrict__ src, D* __restrict__ dst, int64_t total) {
  const int64_t n8 = total >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float v[8];
    ldv<S, 8>(src + i * 8, v);
    stv<D, 8>(dst + i * 8, v);
  }
  if (blockIdx.x == 0 && threadIdx.x < (total & 7)) {
    const int64_t i = (n8 << 3) + threadIdx.x;
    Elem<D>::st(dst + i, Elem<S>::ld(src + i));
  }
}

template <typename S, typename D, int V>
__global__ void copy_channels_kernel(const S* __restrict__ src, int64_t ld_s, D* __restrict__ dst, int64_t ld_d,
                                     int64_t npix, int CV) {
  const int64_t total = npix * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t p = idx / CV;
    int c = (int)(idx - p * CV) * V;
    float v[V];
    ldv<S, V>(src + p * ld_s + c, v);
    stv<D, V>(dst + p * ld_d + c, v);
  }
}

template <typename T, int V>
__global__ void zero_channels_kernel(T* __restrict__ dst, int64_t ld_d, int64_t npix, int CV) {
  const int64_t total = npix * CV;
  float z[V];
#pragma unroll
  for (int k = 0; k < V; ++k) z[k] = 0.f;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t p = idx / CV;
    int c = (int)(idx - p * CV) * V;
    stv<T, V>(dst + p * ld_d + c, z);
  }
}

template <typename T, int V>
__global__ void add_channels_kernel(T* __restrict__ a, int64_t ld_a, const T* __restrict__ b, int64_t ld_b,
                                    int64_t npix, int CV) {
  const int64_t total = npix * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t p = idx / CV;
    int c = (int)(idx - p * CV) * V;
    float x[V], y[V];
    ldv<T, V>(a + p * ld_a + c, x);
    ldv<T, V>(b + p * ld_b + c, y);
#pragma unroll
    for (int k = 0; k < V; ++k) x[k] += y[k];
    stv<T, V>(a + p * ld_a + c, x);
  }
}

// out[c] = sum over pixels; block = 256 threads = CB channels x lanes; fp64 atomics across blocks
template <typename T>
__global__ void channel_sum_kernel(const T* __restrict__ g, int64_t ld, int64_t npix, int C, int CB,
                                   double* __restrict__ acc) {
  __shared__ float red[256];
  const int lanes = blockDim.x / CB;
  const int cl = threadIdx.x % CB, lane = threadIdx.x / CB;
  const int c = blockIdx.y * CB + cl;
  float s = 0.f;
  if (c < C && lane < lanes)
    for (int64_t p = (int64_t)blockIdx.x * lanes + lane; p < npix; p += (int64_t)gridDim.x * lanes)
      s += Elem<T>::ld(g + p * ld + c);
  red[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x < CB && c < C) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[l * CB + threadIdx.x];
    atomicAdd(acc + c, (double)t);
  }
}
// vectorised form: a thread owns 8 consecutive channels (one 16-byte load per pixel), 4 pixels in flight
template <typename T>
__global__ void __launch_bounds__(256) channel_sum_vec_kernel(const T* __restrict__ g, int64_t ld, int64_t npix, int C,
                                                               double* __restrict__ acc) {
  __shared__ float red[256][9];
  const int G = C >> 3, lanes = 256 / G;                  // G divides 256 (checked on the host)
  const int cg = threadIdx.x % G, lane = threadIdx.x / G;
  float s[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * lanes;
  int64_t p = (int64_t)blockIdx.x * lanes + lane;
  for (; p + 3 * stride < npix; p += 4 * stride) {
    float v[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u) load8(g + (p + u * stride) * ld + cg * 8, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] += v[u][i];
  }
  for (; p < npix; p += stride) {
    float v[8];
    load8(g + p * ld + cg * 8, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] += v[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = s[i];
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    const int gq = c >> 3, i = c & 7;
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[l * G + gq][i];
    atomicAdd(acc + c, (double)t);
  }
}
__global__ void double_to_float_kernel(const double* __restrict__ a, float* __restrict__ o, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = (float)a[i];
}

}  // namespace ub

using namespace ub;

// ---- 3xTF32 operand split (fp32 exactness mode on the tensor cores) ------------------------------------------
// x = hi + lo exactly, hi = x rounded to TF32's 10-bit mantissa (round half away from zero on the magnitude bits),
// lo = x - hi (representable: at most 13 significant bits).  A product x*w is then recovered to ~2^-22 relative from
// three kind::tf32 MMAs hi*hi + lo*hi + hi*lo (lo*lo ~ 2^-24 is dropped) accumulated in fp32 -- independent of how
// the tensor core converts its fp32 inputs, because every value fed to it already is a TF32 number or gets rounded
// at 2^-11 of an already 2^-11-small term.  Written as ONE tensor with three channel groups, so that the ordinary
// implicit-GEMM kernels run it as a convolution over 3*C input channels:
//   pattern 0 (left operand: activations / output gradients)  [hi | lo | hi]
//   pattern 1 (right operand: packed weights, per tap)         [hi | hi | lo]
__device__ __forceinline__ float tf32_hi(float x) {
  const uint32_t u = __float_as_uint(x);
  return __uint_as_float((u + 0x1000u) & 0xffffe000u);
}

template <int V>
__global__ void __launch_bounds__(256) split_tf32_kernel(const float* __restrict__ x, int64_t ld_x, float* __restrict__ out,
                                                         int64_t npix, int CV, int pattern) {
  const int64_t total = npix * CV;
  const int C = CV * V;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / CV;
    const int c = (int)(i - p * CV) * V;
    float v[V], hi[V], lo[V];
    if (V == 4) {
      const float4 t = *reinterpret_cast<const float4*>(x + p * ld_x + c);
      v[0] = t.x; v[1 % V] = t.y; v[2 % V] = t.z; v[3 % V] = t.w;
    } else {
      v[0] = x[p * ld_x + c];
    }
#pragma unroll
    for (int k = 0; k < V; ++k) { hi[k] = tf32_hi(v[k]); lo[k] = v[k] - hi[k]; }
    float* o = out + p * 3 * C + c;
    const float* g1 = pattern == 0 ? lo : hi;
    const float* g2 = pattern == 0 ? hi : lo;
    if (V == 4) {
      *reinterpret_cast<float4*>(o) = make_float4(hi[0], hi[1 % V], hi[2 % V], hi[3 % V]);
      *reinterpret_cast<float4*>(o + C) = make_float4(g1[0], g1[1 % V], g1[2 % V], g1[3 % V]);
      *reinterpret_cast<float4*>(o + 2 * C) = make_float4(g2[0], g2[1 % V], g2[2 % V], g2[3 % V]);
    } else {
      o[0] = hi[0]; o[C] = g1[0]; o[2 * C] = g2[0];
    }
  }
}

extern "C" {

int unetb200_bn_finalize_track(const double* stats, int64_t count, const float* gamma, const float* beta, float eps,
                               float momentum, float* running_mean, float* running_var, float* save_mean,
                               float* save_invstd, float* scale, float* shift, int64_t* num_batches_tracked, int C,
                               void* stream) {
  UB_CHECK_ARG(C > 0 && count > 0, "bn_finalize: C=%d count=%lld", C, (long long)count);
  double unbias = count > 1 ? (double)count / (double)(count - 1) : 1.0;
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      stats, 1.0 / (double)count, unbias, gamma, beta, eps, momentum, running_mean, running_var, save_mean,
      save_invstd, scale, shift, C, reinterpret_cast<long long*>(num_batches_tracked));
  UB_LAUNCH_CHECK("bn_finalize");
  return 0;
}

int unetb200_bn_finalize(const double* stats, int64_t count, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, float* save_mean,
                         float* save_invstd, float* scale, float* shift, int C, void* stream) {
  return unetb200_bn_finalize_track(stats, count, gamma, beta, eps, momentum, running_mean, running_var, save_mean,
                                    save_invstd, scale, shift, nullptr, C, stream);
}

int unetb200_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                            const float* running_var, float eps, float* scale, float* shift, float* save_mean,
                            float* save_invstd, int C, void* stream) {
  UB_CHECK_ARG(C > 0, "bn_eval_coeffs: C=%d", C);
  bn_eval_coeffs_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gamma, beta, running_mean, running_var,
                                                                          eps, scale, shift, save_mean,
                                                                          save_invstd, C);
  UB_LAUNCH_CHECK("bn_eval_coeffs");
  return 0;
}

int unetb200_bn_relu_apply(const void* y, int64_t ld_y, const float* scale, const float* shift, void* z,
                           int64_t ld_z, void* pooled, int64_t ld_p, int dtype, int B, int H, int W, int C,
                           void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && ld_y >= C && ld_z >= C, "bn_relu_apply: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t npix = (int64_t)B * H * W;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_y, ld_z, pooled ? ld_p : 0}, {y, z, pooled}), [&](auto V) {
      int CV = C / V;
      if (pooled) {
        CsGeom g_ = cs_geom(CV, (int64_t)B * ((H + 1) / 2) * ((W + 1) / 2), 2);
        bn_relu_apply_pool_kernel<T, V><<<dim3(g_.gx, g_.gy), 256, 0, s>>>(
            (const T*)y, ld_y, scale, shift, (T*)z, ld_z, (T*)pooled, ld_p, B, H, W, CV, g_.CVB);
      } else {
        CsGeom g_ = cs_geom(CV, npix, 8);
        bn_relu_apply_kernel<T, V><<<dim3(g_.gx, g_.gy), 256, 0, s>>>((const T*)y, ld_y, scale, shift, (T*)z,
                                                                     ld_z, npix, CV, g_.CVB);
      }
    });
  });
  UB_LAUNCH_CHECK("bn_relu_apply");
  return 0;
}

int unetb200_maxpool2_fwd(const void* x, int64_t ld_x, void* p, int64_t ld_p, int dtype, int B, int H, int W,
                          int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H >= 2 && W >= 2 && C > 0, "maxpool2_fwd: bad shape %d %d %d %d", B, H, W, C);
  cudaStream_t s = (cudaStream_t)stream;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_x, ld_p}, {x, p}), [&](auto V) {
      int CV = C / V;
      int64_t work = (int64_t)B * (H / 2) * (W / 2) * CV;
      maxpool2_fwd_kernel<T, V><<<grid_for(work, 256, 16), 256, 0, s>>>((const T*)x, ld_x, (T*)p, ld_p, B, H, W, CV);
    });
  });
  UB_LAUNCH_CHECK("maxpool2_fwd");
  return 0;
}

int unetb200_maxpool2_bwd(const void* x, int64_t ld_x, const void* gp, int64_t ld_gp, void* gx, int64_t ld_gx,
                          int accumulate, int dtype, int B, int H, int W, int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H >= 2 && W >= 2 && C > 0, "maxpool2_bwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_x, ld_gp, ld_gx}, {x, gp, gx}), [&](auto V) {
      int CV = C / V;
      int64_t work = (int64_t)B * ((H + 1) / 2) * ((W + 1) / 2) * CV;
      with_bool(accumulate, [&](auto ACC) {
        maxpool2_bwd_kernel<T, V, ACC><<<grid_for(work, 256, 16), 256, 0, s>>>(
            (const T*)x, ld_x, (const T*)gp, ld_gp, (T*)gx, ld_gx, B, H, W, CV);
      });
    });
  });
  UB_LAUNCH_CHECK("maxpool2_bwd");
  return 0;
}

int unetb200_maxpool2_bwd_bnreduce(const void* x, int64_t ld_x, const void* gp, int64_t ld_gp, void* gx, int64_t ld_gx,
                                   const void* y, int64_t ld_y, const float* scale, const float* shift, const float* mean,
                                   const float* invstd, double* sums, int dtype, int B, int H, int W, int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H >= 2 && W >= 2 && C > 0 && x && gp && gx && y && scale && shift && mean && invstd && sums,
               "maxpool2_bwd_bnreduce: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t nwin = (int64_t)B * ((H + 1) / 2) * ((W + 1) / 2);
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_x, ld_gp, ld_gx, ld_y}, {x, gp, gx, y}), [&](auto V) {
      const int CV = (C + V - 1) / V;
      CsGeom g_ = cs_geom(CV, nwin, 2, V == 8 ? 64 : 256);
      maxpool2_bwd_bnreduce_kernel<T, V><<<dim3(g_.gx, g_.gy), 256, 0, s>>>(
          (const T*)x, ld_x, (const T*)gp, ld_gp, (T*)gx, ld_gx, (const T*)y, ld_y, scale, shift, mean, invstd,
          sums, B, H, W, C, CV, g_.CVB);
    });
  });
  UB_LAUNCH_CHECK("maxpool2_bwd_bnreduce");
  return 0;
}

int unetb200_bn_relu_bwd_reduce(const void* gz, int64_t ld_gz, const void* y, int64_t ld_y, const float* scale,
                                const float* shift, const float* mean, const float* invstd, double* sums,
                                int dtype, int B, int H, int W, int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0, "bn_relu_bwd_reduce: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t npix = (int64_t)B * H * W;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_gz, ld_y}, {gz, y}), [&](auto V) {
      int CV = C / V;
      CsGeom g_ = cs_geom(CV, npix, 8, V == 8 ? 64 : 256);   // CVB * V <= the kernel's shared reduction row
      bn_relu_bwd_reduce_kernel<T, V><<<dim3(g_.gx, g_.gy), 256, 0, s>>>(
          (const T*)gz, ld_gz, (const T*)y, ld_y, scale, shift, mean, invstd, sums, npix, C, CV, g_.CVB);
    });
  });
  UB_LAUNCH_CHECK("bn_relu_bwd_reduce");
  return 0;
}

int unetb200_bn_bwd_finalize(const double* sums, int64_t count, int training, float* dgamma, float* dbeta,
                             float* coef, int C, void* stream) {
  UB_CHECK_ARG(C > 0 && count > 0, "bn_bwd_finalize: bad shape");
  bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, 1.0 / (double)count, training,
                                                                            dgamma, dbeta, coef, C);
  UB_LAUNCH_CHECK("bn_bwd_finalize");
  return 0;
}

int unetb200_bn_relu_bwd_apply(const void* gz, int64_t ld_gz, const void* y, int64_t ld_y, const float* scale,
                               const float* shift, const float* mean, const float* invstd, const float* coef,
                               void* gy, int64_t ld_gy, int dtype, int B, int H, int W, int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0, "bn_relu_bwd_apply: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t npix = (int64_t)B * H * W;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_gz, ld_y, ld_gy}, {gz, y, gy}), [&](auto V) {
      int CV = C / V;
      CsGeom g_ = cs_geom(CV, npix, 8);
      bn_relu_bwd_apply_kernel<T, V><<<dim3(g_.gx, g_.gy), 256, 0, s>>>(
          (const T*)gz, ld_gz, (const T*)y, ld_y, scale, shift, mean, invstd, coef, (T*)gy, ld_gy, npix, C, CV,
          g_.CVB);
    });
  });
  UB_LAUNCH_CHECK("bn_relu_bwd_apply");
  return 0;
}

static inline float ac_scale(int in, int out) { return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f; }

int unetb200_upsample2x_fwd(const void* x, int64_t ld_x, void* y, int64_t ld_y, int dtype, int B, int h, int w,
                            int C, int Hout, int Wout, int off_y, int off_x, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && h > 0 && w > 0 && C > 0 && off_y >= 0 && off_x >= 0 && 2 * h + off_y <= Hout &&
                   2 * w + off_x <= Wout,
               "upsample2x_fwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  float sy = ac_scale(h, 2 * h), sx = ac_scale(w, 2 * w);
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_x, ld_y}, {x, y}), [&](auto V) {
      int CV = C / V;
      int64_t work = (int64_t)B * 4 * h * w * CV;
      upsample2x_fwd_kernel<T, V><<<grid_for(work, 256, 16), 256, 0, s>>>(
          (const T*)x, ld_x, (T*)y, ld_y, B, h, w, CV, Hout, Wout, off_y, off_x, sy, sx);
    });
  });
  UB_LAUNCH_CHECK("upsample2x_fwd");
  return 0;
}

int unetb200_upsample2x_bwd(const void* gy, int64_t ld_gy, void* gx, int64_t ld_gx, int dtype, int B, int h,
                            int w, int C, int Hout, int Wout, int off_y, int off_x, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(B > 0 && h > 0 && w > 0 && C > 0 && off_y >= 0 && off_x >= 0 && 2 * h + off_y <= Hout &&
                   2 * w + off_x <= Wout,
               "upsample2x_bwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  float sy = ac_scale(h, 2 * h), sx = ac_scale(w, 2 * w);
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_gy, ld_gx}, {gy, gx}), [&](auto V) {
      int CV = C / V;
      int64_t work = (int64_t)B * h * w * CV;
      upsample2x_bwd_kernel<T, V><<<grid_for(work, 128, 16), 128, 0, s>>>(
          (const T*)gy, ld_gy, (T*)gx, ld_gx, B, h, w, CV, Hout, Wout, off_y, off_x, sy, sx);
    });
  });
  UB_LAUNCH_CHECK("upsample2x_bwd");
  return 0;
}

int unetb200_gather_nhwc(const void* src, int src_dtype, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                         void* dst, int dst_dtype, int64_t ld_dst, int B, int C, int H, int W, void* stream) {
  UB_DTYPE_OK(src_dtype);
  UB_DTYPE_OK(dst_dtype);
  UB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && ld_dst >= C, "gather_nhwc: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t work = (int64_t)B * C * H * W;
  const bool dense = (C == 1 || sc == 1) && sw == C && sh == (int64_t)W * C && sn == (int64_t)H * W * C && ld_dst == C &&
                     (reinterpret_cast<uintptr_t>(src) & 31) == 0 && (reinterpret_cast<uintptr_t>(dst) & 31) == 0;
  if (dense) {
    const int gf = grid_for(work / 8 + 1, 256, 16);
    with_elem(src_dtype, [&](auto src_t) {
      with_elem(dst_dtype, [&](auto dst_t) {
        using S = decltype(src_t);
        using D = decltype(dst_t);
        convert_flat_kernel<S, D><<<gf, 256, 0, s>>>((const S*)src, (D*)dst, work);
      });
    });
    UB_LAUNCH_CHECK("gather_nhwc (flat)");
    return 0;
  }
  int g = grid_for(work, 256, 16);
  with_elem(src_dtype, [&](auto src_t) {
    with_elem(dst_dtype, [&](auto dst_t) {
      using S = decltype(src_t);
      using D = decltype(dst_t);
      gather_nhwc_kernel<S, D><<<g, 256, 0, s>>>((const S*)src, sn, sc, sh, sw, (D*)dst, ld_dst, B, C, H, W);
    });
  });
  UB_LAUNCH_CHECK("gather_nhwc");
  return 0;
}

int unetb200_copy_channels(const void* src, int src_dtype, int64_t ld_src, void* dst, int dst_dtype,
                           int64_t ld_dst, int64_t npix, int C, void* stream) {
  UB_DTYPE_OK(src_dtype);
  UB_DTYPE_OK(dst_dtype);
  UB_CHECK_ARG(npix > 0 && C > 0 && ld_src >= C && ld_dst >= C, "copy_channels: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  with_elem(src_dtype, [&](auto src_t) {
    with_elem(dst_dtype, [&](auto dst_t) {
      using S = decltype(src_t);
      using D = decltype(dst_t);
      with_vec<8>(vec_ok<S>(C, {ld_src}, {src}) && vec_ok<D>(C, {ld_dst}, {dst}), [&](auto V) {
        copy_channels_kernel<S, D, V><<<grid_for(npix * (C / V), 256, 16), 256, 0, s>>>((const S*)src, ld_src,
                                                                                        (D*)dst, ld_dst, npix, C / V);
      });
    });
  });
  UB_LAUNCH_CHECK("copy_channels");
  return 0;
}

int unetb200_zero_channels(void* dst, int dtype, int64_t ld_dst, int64_t npix, int C, void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(npix > 0 && C > 0 && ld_dst >= C, "zero_channels: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_dst}, {dst}), [&](auto V) {
      zero_channels_kernel<T, V><<<grid_for(npix * (C / V), 256, 16), 256, 0, s>>>((T*)dst, ld_dst, npix, C / V);
    });
  });
  UB_LAUNCH_CHECK("zero_channels");
  return 0;
}

int unetb200_add_channels(void* a, int64_t ld_a, const void* b, int64_t ld_b, int dtype, int64_t npix, int C,
                          void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(npix > 0 && C > 0 && ld_a >= C && ld_b >= C, "add_channels: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    with_vec<8>(vec_ok<T>(C, {ld_a, ld_b}, {a, b}), [&](auto V) {
      add_channels_kernel<T, V><<<grid_for(npix * (C / V), 256, 16), 256, 0, s>>>((T*)a, ld_a, (const T*)b, ld_b,
                                                                                  npix, C / V);
    });
  });
  UB_LAUNCH_CHECK("add_channels");
  return 0;
}

int unetb200_channel_sum(const void* g, int dtype, int64_t ld, int64_t npix, int C, double* acc, float* out,
                         void* stream) {
  UB_DTYPE_OK(dtype);
  UB_CHECK_ARG(npix > 0 && C > 0 && ld >= C && acc && out, "channel_sum: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(double) * C, s);
  if (e != cudaSuccess) return cuda_fail(e, "channel_sum memset");
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  if (C % 8 == 0 && C <= 2048 && 256 % (C / 8) == 0 && ld % 8 == 0 && reinterpret_cast<uintptr_t>(g) % (8 * esz) == 0) {
    const int lanes_v = 256 / (C / 8);
    int64_t gx_v = (npix + (int64_t)lanes_v * 32 - 1) / ((int64_t)lanes_v * 32);
    const int64_t cap_v = (int64_t)sm_count() * 4;
    if (gx_v > cap_v) gx_v = cap_v;
    if (gx_v < 1) gx_v = 1;
    with_elem(dtype, [&](auto t) {
      using T = decltype(t);
      channel_sum_vec_kernel<T><<<(unsigned)gx_v, 256, 0, s>>>((const T*)g, ld, npix, C, acc);
    });
    double_to_float_kernel<<<(C + 127) / 128, 128, 0, s>>>(acc, out, C);
    UB_LAUNCH_CHECK("channel_sum_vec");
    return 0;
  }
  const CsGeom g_ = cs_geom(C, npix, 16);
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    channel_sum_kernel<T><<<dim3(g_.gx, g_.gy), 256, 0, s>>>((const T*)g, ld, npix, C, g_.CVB, acc);
  });
  double_to_float_kernel<<<(C + 127) / 128, 128, 0, s>>>(acc, out, C);
  UB_LAUNCH_CHECK("channel_sum");
  return 0;
}

int unetb200_f64_to_f32(const double* src, float* dst, int n, void* stream) {
  UB_CHECK_ARG(src && dst && n > 0, "f64_to_f32: bad args");
  double_to_float_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(src, dst, n);
  UB_LAUNCH_CHECK("f64_to_f32");
  return 0;
}

int unetb200_split_tf32(const float* x, int64_t ld_x, float* out, int64_t npix, int C, int pattern, void* stream) {
  UB_CHECK_ARG(x && out && npix > 0 && C > 0 && ld_x >= C && (pattern == 0 || pattern == 1), "split_tf32: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  with_vec<4>(C % 4 == 0 && ld_x % 4 == 0 && aligned16(x) && aligned16(out), [&](auto V) {
    split_tf32_kernel<V><<<grid_for(npix * (C / V), 256, 16), 256, 0, s>>>(x, ld_x, out, npix, C / V, pattern);
  });
  UB_LAUNCH_CHECK("split_tf32");
  return 0;
}
}
