// OutConv: nn.Conv2d(C, n_classes, kernel_size=1) with bias (unet_parts.py:100-106), n_classes <= 8.
// N = 2..4 makes this HBM-bound (one read of the last activation), so it stays on the CUDA cores:
// LPP = C/8 lanes cooperate on one pixel (each owns 8 channels = one 16-byte load), partial dot
// products are combined with warp shuffles.  Backward produces gx, and dW/dbias through per-block
// partials + a deterministic second-stage reduce.
#include <cstdlib>

#include "common.cuh"

namespace ub {

constexpr int kMaxK = 8;

// K (= n_classes) is a template parameter so that the class loops carry no predicated-off iterations, and every
// thread keeps UNR pixels' 16-byte loads in flight (the kernel is a pure stream over the last activation).
constexpr int kOutUnr = 4;
template <typename T, int K>
__global__ void __launch_bounds__(256) outconv_fwd_vec_kernel(const T* __restrict__ x, int64_t ld_x, const float* __restrict__ w,
                                                              const float* __restrict__ bias, T* __restrict__ out,
                                                              int64_t npix, int C, int LPP) {
  extern __shared__ float sw[];   // [K][C] rounded to T, then bias[K]
  for (int i = threadIdx.x; i < K * C; i += blockDim.x) sw[i] = Elem<T>::round(w[i]);
  for (int i = threadIdx.x; i < K; i += blockDim.x) sw[K * C + i] = bias ? Elem<T>::round(bias[i]) : 0.f;
  __syncthreads();
  const int sub = threadIdx.x % LPP;
  const int ppb = blockDim.x / LPP;
  const int c0 = sub * 8;
  float wr[K][8];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int i = 0; i < 8; ++i) wr[k][i] = sw[k * C + c0 + i];
  // the trip count is block-uniform so that the shuffles below are executed by full warps
  for (int64_t base = (int64_t)blockIdx.x * ppb * kOutUnr; base < npix; base += (int64_t)gridDim.x * ppb * kOutUnr) {
    float v[kOutUnr][8];
#pragma unroll
    for (int u = 0; u < kOutUnr; ++u) {
      const int64_t p = base + u * ppb + threadIdx.x / LPP;
      if (p < npix) {
        load8(x + p * ld_x + c0, v[u]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[u][i] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < kOutUnr; ++u) {
      const int64_t p = base + u * ppb + threadIdx.x / LPP;
      float acc[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        acc[k] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[k] = fmaf(v[u][i], wr[k][i], acc[k]);
      }
      for (int o = LPP >> 1; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      }
      if (sub == 0 && p < npix) {
#pragma unroll
        for (int k = 0; k < K; ++k) Elem<T>::st(out + p * K + k, acc[k] + sw[K * C + k]);
      }
    }
  }
}

template <typename T>
__global__ void outconv_fwd_scalar_kernel(const T* __restrict__ x, int64_t ld_x, const float* __restrict__ w,
                                          const float* __restrict__ bias, T* __restrict__ out, int64_t npix, int C,
                                          int K) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
    for (int k = 0; k < K; ++k) {
      float a = 0.f;
      for (int c = 0; c < C; ++c) a = fmaf(Elem<T>::ld(x + p * ld_x + c), Elem<T>::round(w[k * C + c]), a);
      Elem<T>::st(out + p * K + k, a + (bias ? Elem<T>::round(bias[k]) : 0.f));
    }
  }
}

// backward, vector path.  partial layout per block: float[K*C] dW, float[K] dbias (, float[2*C] BatchNorm sums).
// BNB: x = relu(bn(yprev)) (the OutConv input is the last DoubleConv's activation, unet_model.py:25,37): the kernel
// holds the rounded gx in registers, so it also makes the reduction pass of that BatchNorm + ReLU backward
// (sum gx*mask, sum gx*mask*xhat per channel; unetb200_bn_relu_bwd_reduce) with one extra read of yprev.
template <typename T, int K, bool BNB>
__global__ void __launch_bounds__(256, (K <= 2 && !BNB) ? 3 : 1) outconv_bwd_vec_kernel(const T* __restrict__ x, int64_t ld_x, const float* __restrict__ w,
                                                              const T* __restrict__ g, T* __restrict__ gx, int64_t ld_gx,
                                                              float* __restrict__ partial, int64_t npix, int C, int LPP,
                                                              const T* __restrict__ yprev, int64_t ld_y,
                                                              const float* __restrict__ bnc) {
  constexpr int UNR = BNB ? 2 : kOutUnr;       // the fused variant carries 48 more registers per thread
  extern __shared__ float sm[];   // [K][C] weights; then reduction scratch [K][C] + [K] (+ [2][C])
  float* sw = sm;
  float* red = sm + K * C;
  const int nred = K * C + K + (BNB ? 2 * C : 0);
  for (int i = threadIdx.x; i < K * C; i += blockDim.x) sw[i] = Elem<T>::round(w[i]);
  for (int i = threadIdx.x; i < nred; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  const int sub = threadIdx.x % LPP;
  const int ppb = blockDim.x / LPP;
  const int c0 = sub * 8;
  float wr[K][8], dw[K][8], db[K];
  float bmu[BNB ? 8 : 1], bis[BNB ? 8 : 1], bsc[BNB ? 8 : 1], bsh[BNB ? 8 : 1], s0[BNB ? 8 : 1], s1[BNB ? 8 : 1];
  if constexpr (BNB) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      bmu[i] = __ldg(bnc + c0 + i); bis[i] = __ldg(bnc + C + c0 + i);
      bsc[i] = __ldg(bnc + 2 * C + c0 + i); bsh[i] = __ldg(bnc + 3 * C + c0 + i);
      s0[i] = s1[i] = 0.f;
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    db[k] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { dw[k][i] = 0.f; wr[k][i] = sw[k * C + c0 + i]; }
  }
  for (int64_t base = (int64_t)blockIdx.x * ppb * UNR; base < npix; base += (int64_t)gridDim.x * ppb * UNR) {
    float v[UNR][8], gk[UNR][K], yv[BNB ? UNR : 1][8];
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int64_t p = base + u * ppb + threadIdx.x / LPP;
      if (p < npix) {
        load8(x + p * ld_x + c0, v[u]);
        if constexpr (BNB) load8(yprev + p * ld_y + c0, yv[u]);
#pragma unroll
        for (int k = 0; k < K; ++k) gk[u][k] = Elem<T>::ld(g + p * K + k);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[u][i] = 0.f;
        if constexpr (BNB) {
#pragma unroll
          for (int i = 0; i < 8; ++i) yv[u][i] = 0.f;
        }
#pragma unroll
        for (int k = 0; k < K; ++k) gk[u][k] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int64_t p = base + u * ppb + threadIdx.x / LPP;
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        db[k] += gk[u][k];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          o[i] = fmaf(gk[u][k], wr[k][i], o[i]);
          dw[k][i] = fmaf(gk[u][k], v[u][i], dw[k][i]);
        }
      }
      if (gx && p < npix) store8(gx + p * ld_gx + c0, o);
      if constexpr (BNB) {
        if (p < npix) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float gg = (fmaf(yv[u][i], bsc[i], bsh[i]) > 0.f) ? Elem<T>::round(o[i]) : 0.f;   // gx as stored
            s0[i] += gg;
            s1[i] += gg * ((yv[u][i] - bmu[i]) * bis[i]);
          }
        }
      }
    }
  }
  // block reduction in a FIXED order (no float atomics: the BatchNorm sums feed the whole rest of the backward pass,
  // where bf16 rounding amplifies last-bit noise; run-to-run reproducibility is part of the contract): the ppb
  // pixel lanes stage their 8-channel partials as [lane][C], then thread c adds column c top to bottom
  float* stage = red + nred;       // ppb * C = 2048 floats
  const int pl = threadIdx.x / LPP;
  auto block_sum = [&](const float (&v)[8], float* out) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) stage[pl * C + c0 + i] = v[i];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float acc = 0.f;
      for (int l = 0; l < ppb; ++l) acc += stage[l * C + c];
      out[c] = acc;
    }
  };
#pragma unroll
  for (int k = 0; k < K; ++k) block_sum(dw[k], red + k * C);
  __syncthreads();
  if (sub == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) stage[pl * K + k] = db[k];
  }
  __syncthreads();
  if (threadIdx.x < K) {
    float acc = 0.f;
    for (int l = 0; l < ppb; ++l) acc += stage[l * K + threadIdx.x];
    red[K * C + threadIdx.x] = acc;
  }
  if constexpr (BNB) {
    block_sum(s0, red + K * C + K);
    block_sum(s1, red + K * C + K + C);
  }
  __syncthreads();
  float* dst = partial + (int64_t)blockIdx.x * nred;
  for (int i = threadIdx.x; i < nred; i += blockDim.x) dst[i] = red[i];
}

template <typename T>
__global__ void outconv_bwd_scalar_kernel(const T* __restrict__ x, int64_t ld_x, const float* __restrict__ w,
                                          const T* __restrict__ g, T* __restrict__ gx, int64_t ld_gx,
                                          float* __restrict__ partial, int64_t npix, int C, int K) {
  // one block per (k, c) pair group is overkill for the generic path: blocks stride over pixels and
  // accumulate dW through shared-memory atomics.
  extern __shared__ float red[];   // [K*C + K]
  for (int i = threadIdx.x; i < K * C + K; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
    for (int c = 0; c < C; ++c) {
      float xv = Elem<T>::ld(x + p * ld_x + c);
      float o = 0.f;
      for (int k = 0; k < K; ++k) {
        float gk = Elem<T>::ld(g + p * K + k);
        o = fmaf(gk, Elem<T>::round(w[k * C + c]), o);
        atomicAdd(&red[k * C + c], gk * xv);
      }
      if (gx) Elem<T>::st(gx + p * ld_gx + c, o);
    }
    for (int k = 0; k < K; ++k) atomicAdd(&red[K * C + k], Elem<T>::ld(g + p * K + k));
  }
  __syncthreads();
  float* dst = partial + (int64_t)blockIdx.x * (K * C + K);
  for (int i = threadIdx.x; i < K * C + K; i += blockDim.x) dst[i] = red[i];
}

// One warp per output element: lane l sums the partials of blocks l, l + 32, ... (independent loads in flight),
// then a shuffle tree in fp64 -- a fixed order, so the result is reproducible.  (The first version walked the
// ~600 block partials serially in one thread per element: one L2 latency per block.)
__global__ void __launch_bounds__(256) outconv_reduce_kernel(const float* __restrict__ partial, int nblocks, int KC, int K,
                                                             int extra, float* dw, float* dbias, double* sums) {
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int n = KC + K + extra;
  if (i >= n) return;
  double s = 0;
  for (int b = lane; b < nblocks; b += 32) s += (double)partial[(int64_t)b * n + i];
  s = warp_sum(s);
  if (lane == 0) {
    if (i < KC) dw[i] = (float)s;
    else if (i < KC + K) { if (dbias) dbias[i - KC] = (float)s; }
    else sums[i - KC - K] += s;
  }
}

static int outconv_blocks(int64_t npix) {
  int64_t b = (npix + 2047) / 2048;
  int64_t cap = (int64_t)sm_count() * 4;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}
static bool outconv_vec(int C, int64_t ld, const void* p, size_t esz) {
  int l = C / 8;
  return C % 8 == 0 && l >= 1 && l <= 32 && (l & (l - 1)) == 0 && ld % 8 == 0 &&
         (reinterpret_cast<uintptr_t>(p) % (8 * esz)) == 0;
}

}  // namespace ub

using namespace ub;

extern "C" {

int unetb200_outconv_fwd(const void* x, int64_t ld_x, const float* w, const float* bias, void* logits, int dtype,
                         int64_t npix, int C, int ncls, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "outconv_fwd: dtype");
  UB_CHECK_ARG(npix > 0 && C > 0 && ncls >= 1 && ncls <= kMaxK && ld_x >= C,
               "outconv_fwd: npix=%lld C=%d n_classes=%d (n_classes <= %d)", (long long)npix, C, ncls, kMaxK);
  cudaStream_t s = (cudaStream_t)stream;
  int blocks = outconv_blocks(npix);
  size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  size_t smem = sizeof(float) * ((size_t)ncls * C + ncls);
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    if (outconv_vec(C, ld_x, x, esz) && smem <= 48 * 1024) {
      with_int<1, 2, 3, 4, 5, 6, 7, 8>(ncls, [&](auto KK) {
        outconv_fwd_vec_kernel<T, KK><<<blocks, 256, smem, s>>>((const T*)x, ld_x, w, bias, (T*)logits, npix, C, C / 8);
      });
    } else {
      outconv_fwd_scalar_kernel<T><<<blocks, 256, 0, s>>>((const T*)x, ld_x, w, bias, (T*)logits, npix, C, ncls);
    }
  });
  UB_LAUNCH_CHECK("outconv_fwd");
  return 0;
}

int64_t unetb200_outconv_bwd_workspace(int64_t npix, int C, int ncls) {
  // floats; >= blocks * (K*C + K + 2*C): the BatchNorm-fused variant appends two per-channel sums per block
  return (int64_t)148 * 4 * 2 * ((int64_t)ncls * C + ncls + 2 * (int64_t)C) + 64 + 0 * npix;
}

static bool outconv_bwd_vec_ok(const void* x, int64_t ld_x, const void* gx, int64_t ld_gx, int dtype, int C, int ncls,
                               bool bnb) {
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  const size_t smem_v = sizeof(float) * (2 * (size_t)ncls * C + ncls + (bnb ? 2 * (size_t)C : 0) + 2048);
  return outconv_vec(C, ld_x, x, esz) && (!gx || outconv_vec(C, ld_gx, gx, esz)) && smem_v <= 48 * 1024;
}

static int outconv_bwd_impl(const void* x, int64_t ld_x, const float* w, const void* glogits, void* gx, int64_t ld_gx,
                            float* dw, float* dbias, float* workspace, int dtype, int64_t npix, int C, int ncls,
                            const void* yprev, int64_t ld_y, const float* bnc, double* sums, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "outconv_bwd: dtype");
  UB_CHECK_ARG(npix > 0 && C > 0 && ncls >= 1 && ncls <= kMaxK && ld_x >= C, "outconv_bwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  int blocks = outconv_blocks(npix);
  if (blocks > 148 * 4 * 2) blocks = 148 * 4 * 2;
  const bool bnb = yprev != nullptr;
  // n_classes <= 2 (the path: 2 classes) is compiled for three resident blocks per SM (80 registers): one full wave
  static const bool wave3 = getenv("UNETB200_OUTCONV_WAVE4") == nullptr;
  if (wave3 && ncls <= 2 && !bnb && blocks > sm_count() * 3) blocks = sm_count() * 3;
  const int KC = ncls * C;
  const int extra = bnb ? 2 * C : 0;
  size_t smem_v = sizeof(float) * (2 * (size_t)KC + ncls + extra + 2048);
  size_t smem_s = sizeof(float) * ((size_t)KC + ncls);
  UB_CHECK_ARG(smem_s <= 48 * 1024, "outconv_bwd: n_classes*C too large (%d)", KC);
  bool vec = outconv_bwd_vec_ok(x, ld_x, gx, ld_gx, dtype, C, ncls, bnb);
  UB_CHECK_ARG(!bnb || vec, "outconv_bwd_bnbwd: shape not covered (query _supported first)");
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    if (vec) {
      with_int<1, 2, 3, 4, 5, 6, 7, 8>(ncls, [&](auto KK) {
        with_bool(bnb, [&](auto BNB) {
          outconv_bwd_vec_kernel<T, KK, BNB><<<blocks, 256, smem_v, s>>>((const T*)x, ld_x, w, (const T*)glogits,
                                                                         (T*)gx, ld_gx, workspace, npix, C, C / 8,
                                                                         (const T*)yprev, ld_y, bnc);
        });
      });
    } else {
      outconv_bwd_scalar_kernel<T><<<blocks, 256, smem_s, s>>>((const T*)x, ld_x, w, (const T*)glogits, (T*)gx, ld_gx,
                                                               workspace, npix, C, ncls);
    }
  });
  outconv_reduce_kernel<<<(KC + ncls + extra + 7) / 8, 256, 0, s>>>(workspace, blocks, KC, ncls, extra, dw, dbias, sums);
  UB_LAUNCH_CHECK("outconv_bwd");
  return 0;
}

int unetb200_outconv_bwd(const void* x, int64_t ld_x, const float* w, const void* glogits, void* gx, int64_t ld_gx,
                         float* dw, float* dbias, float* workspace, int dtype, int64_t npix, int C, int ncls,
                         void* stream) {
  return outconv_bwd_impl(x, ld_x, w, glogits, gx, ld_gx, dw, dbias, workspace, dtype, npix, C, ncls, nullptr, 0, nullptr,
                          nullptr, stream);
}

int unetb200_outconv_bwd_bnbwd_supported(const void* x, int64_t ld_x, const void* gx, int64_t ld_gx, const void* yprev,
                                         int64_t ld_yprev, int dtype, int C, int ncls) {
  static const bool off = getenv("UNETB200_NO_BNBWD_FUSE") != nullptr;
  if (off || !gx || !yprev || ncls < 1 || ncls > kMaxK) return 0;
  if (dtype != UNETB200_F32 && dtype != UNETB200_BF16) return 0;
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  return outconv_bwd_vec_ok(x, ld_x, gx, ld_gx, dtype, C, ncls, true) && outconv_vec(C, ld_yprev, yprev, esz);
}

int unetb200_outconv_bwd_bnbwd(const void* x, int64_t ld_x, const float* w, const void* glogits, void* gx, int64_t ld_gx,
                               float* dw, float* dbias, float* workspace, const void* yprev, int64_t ld_yprev,
                               const float* coefs, double* sums, int dtype, int64_t npix, int C, int ncls, void* stream) {
  UB_CHECK_ARG(gx && yprev && coefs && sums, "outconv_bwd_bnbwd: null pointer");
  UB_CHECK_ARG(unetb200_outconv_bwd_bnbwd_supported(x, ld_x, gx, ld_gx, yprev, ld_yprev, dtype, C, ncls),
               "outconv_bwd_bnbwd: shape not covered (query _supported first and run outconv_bwd + bn_relu_bwd_reduce)");
  return outconv_bwd_impl(x, ld_x, w, glogits, gx, ld_gx, dw, dbias, workspace, dtype, npix, C, ncls, yprev, ld_yprev, coefs,
                          sums, stream);
}
}
