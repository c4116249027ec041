// Optimizer side of the training step (train.py:80-84,153-159): clip_grad_norm_ + RMSprop(momentum) as two
// multi-tensor kernels instead of PyTorch's ~25 foreach launches over the 64 parameter tensors.
//   1. grad_sqnorm : sum of squares of all gradients -> one double (the squared total norm of clip_grad_norm_)
//   2. rmsprop_step: per element, exactly torch.optim.RMSprop (centered=False):
//        g  = grad * min(1, max_norm / (total_norm + 1e-6))          (clip_grad_norm_, optional)
//        g += weight_decay * w
//        sq = alpha * sq + (1 - alpha) * g * g ;  avg = sqrt(sq) + eps
//        buf = momentum * buf + g / avg ;  w -= lr * buf             (momentum > 0)
//        w -= lr * g / avg                                            (momentum == 0)
// The tensor table travels by value in the kernel parameters (no device-side table to maintain): up to
// kMaxTensors tensors per launch, the host loops over longer lists.  Memory-bound: 4 reads + 3 writes per element.
//
// The *_amp variants serve torch.amp.GradScaler and LR schedulers inside a captured step (train.py:154-159:
// scale(loss).backward(), unscale_, clip_grad_norm_, step, update): the learning rate, GradScaler's inverse scale
// and its found_inf flag are read from device memory, so a replayed graph follows values written between replays.
// A non-zero found_inf makes rmsprop_step_amp store nothing (torch skips optimizer.step()); the per-parameter
// step counters are incremented on the device only when the step is taken.
#include "common.cuh"

namespace ub {

constexpr int kMaxTensors = 48;
constexpr int kChunk = 8192;          // elements per block

struct alignas(16) OptTable {
  float* w[kMaxTensors];
  float* g[kMaxTensors];
  float* sq[kMaxTensors];
  float* mom[kMaxTensors];
  int chunk_start[kMaxTensors + 1];   // prefix sum of chunks per tensor
  long long numel[kMaxTensors];
  int ntensors;
};

struct alignas(16) AmpOptTable {
  OptTable t;
  float* step[kMaxTensors];           // fp32 0-dim step counter of each tensor
};
// kernel parameters (table by value + pointers + scalars) must stay within the 4 KB launch-parameter limit
static_assert(sizeof(AmpOptTable) + 4 * sizeof(void*) + 6 * sizeof(float) <= 4096, "AmpOptTable too large");

__device__ __forceinline__ int find_tensor(const OptTable& t, int chunk) {
  int lo = 0, hi = t.ntensors - 1;
  while (lo < hi) {                   // last tensor with chunk_start <= chunk
    const int mid = (lo + hi + 1) >> 1;
    if (t.chunk_start[mid] <= chunk) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(256) grad_sqnorm_kernel(const __grid_constant__ OptTable t, double* __restrict__ out) {
  const int ti = find_tensor(t, blockIdx.x);
  const long long n = t.numel[ti];
  const long long begin = (long long)(blockIdx.x - t.chunk_start[ti]) * kChunk;
  long long end = begin + kChunk;
  if (end > n) end = n;
  const float* g = t.g[ti];
  float s = 0.f;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const long long nvec = (end - begin) >> 2;
    for (long long v = threadIdx.x; v < nvec; v += 256) {
      const float4 x = *reinterpret_cast<const float4*>(g + begin + 4 * v);
      s += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
    }
    for (long long i = begin + 4 * nvec + threadIdx.x; i < end; i += 256) s += g[i] * g[i];
  } else {
    for (long long i = begin + threadIdx.x; i < end; i += 256) s += g[i] * g[i];
  }
  double d = warp_sum((double)s);
  __shared__ double red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += red[i];
    atomicAdd(out, a);
  }
}

// grad_sqnorm_kernel over g * inv_scale (same per-thread / warp / block order), fused with GradScaler's check:
// any non-finite raw element (isfinite per element, so an overflowing square is not a false positive) sets
// *found_inf = 1 -- one store per block at most, never cleared here.  out / found_inf may each be NULL.
__global__ void __launch_bounds__(256) grad_sqnorm_amp_kernel(const __grid_constant__ OptTable t,
                                                              const float* __restrict__ inv_scale,
                                                              double* __restrict__ out, float* __restrict__ found_inf) {
  const int ti = find_tensor(t, blockIdx.x);
  const long long n = t.numel[ti];
  const long long begin = (long long)(blockIdx.x - t.chunk_start[ti]) * kChunk;
  long long end = begin + kChunk;
  if (end > n) end = n;
  const float* g = t.g[ti];
  const float inv = inv_scale ? *inv_scale : 1.f;
  bool bad = false;
  auto sq = [&](float x) {
    bad |= !isfinite(x);
    x *= inv;
    return x * x;
  };
  float s = 0.f;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const long long nvec = (end - begin) >> 2;
    for (long long v = threadIdx.x; v < nvec; v += 256) {
      const float4 x = *reinterpret_cast<const float4*>(g + begin + 4 * v);
      s += sq(x.x) + sq(x.y) + sq(x.z) + sq(x.w);
    }
    for (long long i = begin + 4 * nvec + threadIdx.x; i < end; i += 256) s += sq(g[i]);
  } else {
    for (long long i = begin + threadIdx.x; i < end; i += 256) s += sq(g[i]);
  }
  double d = warp_sum((double)s);
  __shared__ double red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
  const int any_bad = __syncthreads_or(bad);
  if (threadIdx.x == 0) {
    if (out) {
      double a = 0.0;
#pragma unroll
      for (int i = 0; i < 8; ++i) a += red[i];
      atomicAdd(out, a);
    }
    if (found_inf && any_bad) *found_inf = 1.f;
  }
}

__device__ __forceinline__ float clip_coef(const double* sumsq, float max_norm) {
  if (!sumsq) return 1.f;
  const float total = (float)sqrt(*sumsq);
  // torch.nn.utils.clip_grad_norm_: clamp(max_norm / (total + 1e-6), max=1); a non-finite norm propagates to
  // every gradient as it does in torch (fminf alone would drop a NaN)
  const float c = max_norm / (total + 1e-6f);
  return (c == c) ? fminf(c, 1.f) : c;
}

// The per-element RMSprop update of chunk [begin, end) of tensor ti.  kScaled: g is first multiplied by inv
// (GradScaler's unscale, before the clip coefficient, as unscale_ precedes clip_grad_norm_ in train.py).
template <bool kScaled>
__device__ __forceinline__ void rmsprop_chunk(const OptTable& t, int ti, long long begin, long long end, float inv,
                                              float coef, float lr, float alpha, float eps, float weight_decay,
                                              float momentum, int write_clipped_grad) {
  float* w = t.w[ti];
  float* g = t.g[ti];
  float* sq = t.sq[ti];
  float* mom = t.mom[ti];
  const float one_m_alpha = 1.f - alpha;
  auto update = [&](float gi, float wi, float si, float mi, float& w_out, float& s_out, float& m_out, float& g_out) {
    if (kScaled) gi *= inv;
    gi *= coef;
    g_out = gi;
    if (weight_decay != 0.f) gi = fmaf(weight_decay, wi, gi);
    const float s = fmaf(one_m_alpha * gi, gi, si * alpha);       // square_avg.mul_(alpha).addcmul_(g, g, value=1-alpha)
    s_out = s;
    const float avg = sqrtf(s) + eps;
    if (mom) {
      const float b = fmaf(momentum, mi, gi / avg);               // buf.mul_(momentum).addcdiv_(g, avg)
      m_out = b;
      w_out = fmaf(-lr, b, wi);
    } else {
      m_out = 0.f;
      w_out = fmaf(-lr, gi / avg, wi);
    }
  };
  const bool vec = ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(sq) |
                     reinterpret_cast<uintptr_t>(mom)) & 15) == 0;
  long long i0 = begin;
  if (vec) {
    const long long nvec = (end - begin) >> 2;
    for (long long v = threadIdx.x; v < nvec; v += 256) {
      const long long i = begin + 4 * v;
      const float4 g4 = *reinterpret_cast<const float4*>(g + i), w4 = *reinterpret_cast<const float4*>(w + i),
                   s4 = *reinterpret_cast<const float4*>(sq + i);
      const float4 m4 = mom ? *reinterpret_cast<const float4*>(mom + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 wo, so, mo, go;
      update(g4.x, w4.x, s4.x, m4.x, wo.x, so.x, mo.x, go.x);
      update(g4.y, w4.y, s4.y, m4.y, wo.y, so.y, mo.y, go.y);
      update(g4.z, w4.z, s4.z, m4.z, wo.z, so.z, mo.z, go.z);
      update(g4.w, w4.w, s4.w, m4.w, wo.w, so.w, mo.w, go.w);
      *reinterpret_cast<float4*>(w + i) = wo;
      *reinterpret_cast<float4*>(sq + i) = so;
      if (mom) *reinterpret_cast<float4*>(mom + i) = mo;
      if (write_clipped_grad) *reinterpret_cast<float4*>(g + i) = go;
    }
    i0 = begin + 4 * nvec;
  }
  for (long long i = i0 + threadIdx.x; i < end; i += 256) {
    float wo, so, mo, go;
    update(g[i], w[i], sq[i], mom ? mom[i] : 0.f, wo, so, mo, go);
    w[i] = wo;
    sq[i] = so;
    if (mom) mom[i] = mo;
    if (write_clipped_grad) g[i] = go;
  }
}

__global__ void __launch_bounds__(256) rmsprop_step_kernel(const __grid_constant__ OptTable t, const double* __restrict__ sumsq,
                                                           float max_norm, float lr, float alpha, float eps,
                                                           float weight_decay, float momentum, int write_clipped_grad) {
  const int ti = find_tensor(t, blockIdx.x);
  const long long n = t.numel[ti];
  const long long begin = (long long)(blockIdx.x - t.chunk_start[ti]) * kChunk;
  long long end = begin + kChunk;
  if (end > n) end = n;
  rmsprop_chunk<false>(t, ti, begin, end, 1.f, clip_coef(sumsq, max_norm), lr, alpha, eps, weight_decay, momentum,
                       write_clipped_grad);
}

// rmsprop_step_kernel with lr, GradScaler's inverse scale (nullable: 1) and found_inf (nullable: 0) read from the
// device.  found_inf != 0: the block returns before any store, so w, square_avg, momentum_buffer, grad and step
// stay bit-for-bit unchanged.  Otherwise the first block of each tensor increments its step counter.
__global__ void __launch_bounds__(256) rmsprop_step_amp_kernel(const __grid_constant__ AmpOptTable at,
                                                               const double* __restrict__ sumsq, float max_norm,
                                                               const float* __restrict__ lr,
                                                               const float* __restrict__ inv_scale,
                                                               const float* __restrict__ found_inf, float alpha,
                                                               float eps, float weight_decay, float momentum,
                                                               int write_clipped_grad) {
  if (found_inf && *found_inf != 0.f) return;
  const OptTable& t = at.t;
  const int ti = find_tensor(t, blockIdx.x);
  if (threadIdx.x == 0 && blockIdx.x == t.chunk_start[ti]) *at.step[ti] += 1.f;
  const long long n = t.numel[ti];
  const long long begin = (long long)(blockIdx.x - t.chunk_start[ti]) * kChunk;
  long long end = begin + kChunk;
  if (end > n) end = n;
  rmsprop_chunk<true>(t, ti, begin, end, inv_scale ? *inv_scale : 1.f, clip_coef(sumsq, max_norm), *lr, alpha, eps,
                      weight_decay, momentum, write_clipped_grad);
}

static int build_table(OptTable* T, float* const* w, float* const* g, float* const* sq, float* const* mom,
                       const int64_t* numel, int first, int count) {
  int chunks = 0;
  for (int i = 0; i < count; ++i) {
    T->w[i] = w ? w[first + i] : nullptr;
    T->g[i] = g[first + i];
    T->sq[i] = sq ? sq[first + i] : nullptr;
    T->mom[i] = mom ? mom[first + i] : nullptr;
    T->numel[i] = numel[first + i];
    T->chunk_start[i] = chunks;
    chunks += (int)((numel[first + i] + kChunk - 1) / kChunk);
  }
  T->chunk_start[count] = chunks;
  T->ntensors = count;
  return chunks;
}

}  // namespace ub

using namespace ub;

extern "C" {

int unetb200_grad_sqnorm(float* const* grads, const int64_t* numel, int ntensors, double* out, void* stream) {
  UB_CHECK_ARG(grads && numel && out && ntensors >= 1, "grad_sqnorm: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double), s);
  if (e != cudaSuccess) return cuda_fail(e, "grad_sqnorm memset");
  for (int first = 0; first < ntensors; first += kMaxTensors) {
    const int count = ntensors - first < kMaxTensors ? ntensors - first : kMaxTensors;
    OptTable T;
    for (int i = 0; i < count; ++i) UB_CHECK_ARG(grads[first + i] && numel[first + i] > 0, "grad_sqnorm: tensor %d", first + i);
    const int chunks = build_table(&T, nullptr, grads, nullptr, nullptr, numel, first, count);
    grad_sqnorm_kernel<<<chunks, 256, 0, s>>>(T, out);
  }
  UB_LAUNCH_CHECK("grad_sqnorm");
  return 0;
}

int unetb200_rmsprop_step(float* const* w, float* const* g, float* const* sq, float* const* mom, const int64_t* numel,
                          int ntensors, const double* sumsq, float max_norm, float lr, float alpha, float eps,
                          float weight_decay, float momentum, int write_clipped_grad, void* stream) {
  UB_CHECK_ARG(w && g && sq && numel && ntensors >= 1, "rmsprop_step: bad args");
  UB_CHECK_ARG((momentum != 0.f) == (mom != nullptr), "rmsprop_step: momentum buffers must be given iff momentum != 0");
  cudaStream_t s = (cudaStream_t)stream;
  for (int first = 0; first < ntensors; first += kMaxTensors) {
    const int count = ntensors - first < kMaxTensors ? ntensors - first : kMaxTensors;
    OptTable T;
    for (int i = 0; i < count; ++i)
      UB_CHECK_ARG(w[first + i] && g[first + i] && sq[first + i] && numel[first + i] > 0, "rmsprop_step: tensor %d", first + i);
    const int chunks = build_table(&T, w, g, sq, mom, numel, first, count);
    rmsprop_step_kernel<<<chunks, 256, 0, s>>>(T, sumsq, max_norm, lr, alpha, eps, weight_decay, momentum,
                                               write_clipped_grad);
  }
  UB_LAUNCH_CHECK("rmsprop_step");
  return 0;
}

int unetb200_grad_sqnorm_amp(float* const* grads, const int64_t* numel, int ntensors, const float* inv_scale,
                             double* sumsq, float* found_inf, void* stream) {
  UB_CHECK_ARG(grads && numel && ntensors >= 1 && (sumsq || found_inf), "grad_sqnorm_amp: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  if (sumsq) {
    cudaError_t e = cudaMemsetAsync(sumsq, 0, sizeof(double), s);
    if (e != cudaSuccess) return cuda_fail(e, "grad_sqnorm_amp memset");
  }
  for (int first = 0; first < ntensors; first += kMaxTensors) {
    const int count = ntensors - first < kMaxTensors ? ntensors - first : kMaxTensors;
    OptTable T;
    for (int i = 0; i < count; ++i)
      UB_CHECK_ARG(grads[first + i] && numel[first + i] > 0, "grad_sqnorm_amp: tensor %d", first + i);
    const int chunks = build_table(&T, nullptr, grads, nullptr, nullptr, numel, first, count);
    grad_sqnorm_amp_kernel<<<chunks, 256, 0, s>>>(T, inv_scale, sumsq, found_inf);
  }
  UB_LAUNCH_CHECK("grad_sqnorm_amp");
  return 0;
}

int unetb200_rmsprop_step_amp(float* const* w, float* const* g, float* const* sq, float* const* mom,
                              float* const* step, const int64_t* numel, int ntensors, const double* sumsq,
                              float max_norm, const float* lr, const float* inv_scale, const float* found_inf,
                              float alpha, float eps, float weight_decay, float momentum, int write_clipped_grad,
                              void* stream) {
  UB_CHECK_ARG(w && g && sq && step && numel && lr && ntensors >= 1, "rmsprop_step_amp: bad args");
  UB_CHECK_ARG((momentum != 0.f) == (mom != nullptr), "rmsprop_step_amp: momentum buffers must be given iff momentum != 0");
  cudaStream_t s = (cudaStream_t)stream;
  for (int first = 0; first < ntensors; first += kMaxTensors) {
    const int count = ntensors - first < kMaxTensors ? ntensors - first : kMaxTensors;
    AmpOptTable T;
    for (int i = 0; i < count; ++i) {
      UB_CHECK_ARG(w[first + i] && g[first + i] && sq[first + i] && step[first + i] && numel[first + i] > 0,
                   "rmsprop_step_amp: tensor %d", first + i);
      T.step[i] = step[first + i];
    }
    const int chunks = build_table(&T.t, w, g, sq, mom, numel, first, count);
    rmsprop_step_amp_kernel<<<chunks, 256, 0, s>>>(T, sumsq, max_norm, lr, inv_scale, found_inf, alpha, eps,
                                                   weight_decay, momentum, write_clipped_grad);
  }
  UB_LAUNCH_CHECK("rmsprop_step_amp");
  return 0;
}
}
