// First-layer convolution: 3x3, C_in = 1..4 (grayscale / RGB input, unet_model.py:15), K = 9*C_in <= 36.
// With so little reduction depth the layer is HBM-bound (it writes / reads the full-resolution 64-channel
// activation once), so it stays on the CUDA cores with a channel-stationary mapping: a thread owns 8
// output channels (one 16-byte NHWC store) and streams over pixels; the 8 threads of a pixel cover
// 128 contiguous bytes.  fprop keeps its 72 weights in registers (C_in = 1) and also produces the
// BatchNorm partial sums; wgrad keeps its 72 accumulators in registers and reads dY exactly once.
#include "gconv.cuh"

namespace ub {

__device__ __forceinline__ void first_decode(const GconvDev& d, int m, int& b, int& i, int& j) {
  j = m % d.Wm;                 // 32-bit: M < 2^31 is checked on the host (64-bit div costs ~100 instr)
  const int r = m / d.Wm;
  i = r % d.Hm;
  b = r / d.Hm;
}

template <typename T, int CIN>
__global__ void __launch_bounds__(256)
first_conv_fprop_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ wp, T* __restrict__ y,
                        float* __restrict__ stats_ws) {
  constexpr int K = 9 * CIN;
  __shared__ float sstat[2][256];
  __shared__ float sw[CIN == 1 ? 1 : K * 256];          // [k][n], only for C_in > 1
  const int G = d.N >> 3, lanes = 256 / G;
  const int g = threadIdx.x % G, lane = threadIdx.x / G;
  const bool active = lane < lanes;
  for (int i = threadIdx.x; i < 2 * 256; i += 256) (&sstat[0][0])[i] = 0.f;
  float wr[CIN == 1 ? K : 1][8];
  if constexpr (CIN == 1) {
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int i = 0; i < 8; ++i) wr[k][i] = Elem<T>::ld(wp + (long long)(g * 8 + i) * K + k);
  } else {
    for (int e = threadIdx.x; e < K * d.N; e += 256) {
      const int n = e / K, k = e - n * K;
      sw[k * d.N + n] = Elem<T>::ld(wp + e);
    }
  }
  __syncthreads();
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  if (active) {
    // source grid == M grid (checked on the host): the source pixel of tap t is simply m + dy*W + dx
    int toff[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) toff[t] = d.tap_dy[t] * d.Win + d.tap_dx[t];
    const int M = (int)d.M, mstride = gridDim.x * lanes;
    for (int m = blockIdx.x * lanes + lane; m < M; m += mstride) {
      int b, pi, pj;
      first_decode(d, m, b, pi, pj);
      // all loads first, branch-free (out-of-range taps read pixel m itself and are zeroed by a select)
      float xv[9][CIN];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const bool ok = (unsigned)(pi + d.tap_dy[t]) < (unsigned)d.Hin && (unsigned)(pj + d.tap_dx[t]) < (unsigned)d.Win;
        const T* src = x + (long long)(ok ? m + toff[t] : m) * d.ld_in;
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          const float v = Elem<T>::ld(src + c);
          xv[t][c] = ok ? v : 0.f;
        }
      }
      float acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          if constexpr (CIN == 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(xv[t][c], wr[t][i], acc[i]);
          } else {
            const float4 w0 = *reinterpret_cast<const float4*>(&sw[(t * CIN + c) * d.N + g * 8]);
            const float4 w1 = *reinterpret_cast<const float4*>(&sw[(t * CIN + c) * d.N + g * 8 + 4]);
            acc[0] = fmaf(xv[t][c], w0.x, acc[0]); acc[1] = fmaf(xv[t][c], w0.y, acc[1]);
            acc[2] = fmaf(xv[t][c], w0.z, acc[2]); acc[3] = fmaf(xv[t][c], w0.w, acc[3]);
            acc[4] = fmaf(xv[t][c], w1.x, acc[4]); acc[5] = fmaf(xv[t][c], w1.y, acc[5]);
            acc[6] = fmaf(xv[t][c], w1.z, acc[6]); acc[7] = fmaf(xv[t][c], w1.w, acc[7]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc[i] = Elem<T>::round(acc[i]);
        s[i] += acc[i];
        q[i] += acc[i] * acc[i];
      }
      store8(y + (long long)m * d.ld_out + g * 8, acc);
    }
  }
  if (stats_ws) {
    if (active) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { atomicAdd(&sstat[0][g * 8 + i], s[i]); atomicAdd(&sstat[1][g * 8 + i], q[i]); }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 2 * d.N; e += 256) {
      const int which = e / d.N, c = e - which * d.N;
      stats_ws[((long long)blockIdx.x * 2 + which) * d.N + c] = sstat[which][c];
    }
  }
}

// C_in = 2..4 (RGB input, BASELINE configs[4]): the kernel above re-reads its 9*C_in weight vectors from shared
// memory for every pixel (54 LDS.128 per 216 FMAs at C_in = 3: shared-memory bandwidth bound, 2.75 ms for the
// 8 x 1024 x 1024 first layer).  Here a thread owns FOUR horizontally adjacent pixels x 8 output channels: one weight
// vector feeds 32 FMAs and the 3 x 6 input window is loaded once for the four pixels.
template <typename T, int CIN>
__global__ void __launch_bounds__(256)
first_conv_fprop_px4_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ wp, T* __restrict__ y,
                            float* __restrict__ stats_ws) {
  constexpr int K = 9 * CIN;
  __shared__ float sstat[2][256];
  __shared__ float sw[K * 256];                          // [(window position, c)][n]
  __shared__ int tmap[9];
  const int G = d.N >> 3, lanes = 256 / G;
  const int g = threadIdx.x % G, lane = threadIdx.x / G;
  const bool active = lane < lanes;
  for (int i = threadIdx.x; i < 2 * 256; i += 256) (&sstat[0][0])[i] = 0.f;
  if (threadIdx.x < 9) tmap[(d.tap_dy[threadIdx.x] + 1) * 3 + d.tap_dx[threadIdx.x] + 1] = threadIdx.x;
  __syncthreads();
  for (int e = threadIdx.x; e < K * d.N; e += 256) {
    const int n = e / K, k = e - n * K;                  // k = (window position, c) -> packed index (tap, c)
    const int pos = k / CIN, c = k - pos * CIN;
    sw[k * d.N + n] = Elem<T>::ld(wp + (long long)n * K + tmap[pos] * CIN + c);
  }
  __syncthreads();
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  if (active) {
    const int Wq = d.Wm >> 2;                            // W % 4 == 0 (checked on the host)
    const int Mq = d.B * d.Hm * Wq, qstride = gridDim.x * lanes;
    for (int mq = blockIdx.x * lanes + lane; mq < Mq; mq += qstride) {
      const int jq = mq % Wq, r = mq / Wq;
      const int pi = r % d.Hm, b = r / d.Hm;
      const int j0 = jq << 2;
      float acc[4][8];
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[p][i] = 0.f;
      // one window row at a time (not unrolled: 6 * C_in live inputs + 32 accumulators stay in registers)
#pragma unroll 1
      for (int a = 0; a < 3; ++a) {
        const int gi = pi - 1 + a;
        const bool rok = (unsigned)gi < (unsigned)d.Hin;
        float xr[6][CIN];
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) {
          const int gj = j0 - 1 + cc;
          const bool ok = rok && (unsigned)gj < (unsigned)d.Win;
          const T* src = x + ((long long)(b * d.Hin + (ok ? gi : pi)) * d.Win + (ok ? gj : j0)) * d.ld_in;
#pragma unroll
          for (int c = 0; c < CIN; ++c) {
            const float v = Elem<T>::ld(src + c);
            xr[cc][c] = ok ? v : 0.f;
          }
        }
        const float* wa = &sw[a * 3 * CIN * d.N + g * 8];
#pragma unroll
        for (int cw = 0; cw < 3; ++cw)
#pragma unroll
          for (int c = 0; c < CIN; ++c) {
            const float* wrow = wa + (cw * CIN + c) * d.N;
            const float4 w0 = *reinterpret_cast<const float4*>(wrow);
            const float4 w1 = *reinterpret_cast<const float4*>(wrow + 4);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              const float xe = xr[p + cw][c];
              acc[p][0] = fmaf(xe, w0.x, acc[p][0]); acc[p][1] = fmaf(xe, w0.y, acc[p][1]);
              acc[p][2] = fmaf(xe, w0.z, acc[p][2]); acc[p][3] = fmaf(xe, w0.w, acc[p][3]);
              acc[p][4] = fmaf(xe, w1.x, acc[p][4]); acc[p][5] = fmaf(xe, w1.y, acc[p][5]);
              acc[p][6] = fmaf(xe, w1.z, acc[p][6]); acc[p][7] = fmaf(xe, w1.w, acc[p][7]);
            }
          }
      }
      T* dst = y + ((long long)(b * d.Hm + pi) * d.Wm + j0) * d.ld_out + g * 8;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          acc[p][i] = Elem<T>::round(acc[p][i]);
          s[i] += acc[p][i];
          q[i] += acc[p][i] * acc[p][i];
        }
        store8(dst + (long long)p * d.ld_out, acc[p]);
      }
    }
  }
  if (stats_ws) {
    if (active) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { atomicAdd(&sstat[0][g * 8 + i], s[i]); atomicAdd(&sstat[1][g * 8 + i], q[i]); }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 2 * d.N; e += 256) {
      const int which = e / d.N, c = e - which * d.N;
      stats_ws[((long long)blockIdx.x * 2 + which) * d.N + c] = sstat[which][c];
    }
  }
}

// dWp[(t)][n] partial per block (C_in == 1): partials[block][9][N]
template <typename T>
__global__ void __launch_bounds__(256)
first_conv_wgrad_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ gy, float* __restrict__ partials) {
  __shared__ float red[8][9 * 128];
  const int G = d.N >> 3, lanes = 256 / G;              // G is a power of two <= 16 (checked on the host)
  const int g = threadIdx.x % G, lane = threadIdx.x / G;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[t][i] = 0.f;
  int toff[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) toff[t] = d.tap_dy[t] * d.Win + d.tap_dx[t];
  const int M = (int)d.M, mstride = gridDim.x * lanes;
  for (int m = blockIdx.x * lanes + lane; m < M; m += mstride) {
    int b, pi, pj;
    first_decode(d, m, b, pi, pj);
    float gv[8], xv[9];
    load8(gy + (long long)m * d.ld_out + g * 8, gv);
#pragma unroll
    for (int t = 0; t < 9; ++t) {            // branch-free: all loads in flight together
      const bool ok = (unsigned)(pi + d.tap_dy[t]) < (unsigned)d.Hin && (unsigned)(pj + d.tap_dx[t]) < (unsigned)d.Win;
      const float v = Elem<T>::ld(x + (long long)(ok ? m + toff[t] : m) * d.ld_in);
      xv[t] = ok ? v : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[t][i] = fmaf(xv[t], gv[i], acc[t][i]);
  }
  // lanes of one warp that share a channel group: xor-shuffle over the lane bits above log2(G)
  const int warp = threadIdx.x >> 5;
  __syncwarp();
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float v = acc[t][i];
      for (int o = G; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      acc[t][i] = v;
    }
  if ((threadIdx.x & 31) < G) {
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int i = 0; i < 8; ++i) red[warp][t * d.N + g * 8 + i] = acc[t][i];
  }
  __syncthreads();
  float* out = partials + (long long)blockIdx.x * 9 * d.N;
  for (int e = threadIdx.x; e < 9 * d.N; e += 256) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][e];
    out[e] = v;
  }
}

// ------------------------------------------------------------------------------------------
// Tiled variants for the layer the path actually has (C_in = 1, 64 output channels): a block owns an
// 8 x 32 pixel tile, stages its 10 x 34 input halo in shared memory once (no per-pixel index division, no
// global-load latency in the inner loop) and walks down the 8 rows with a 3 x 3 register window.
// Thread = (pixel column of the tile, 8-channel group): the 8 threads of a pixel write / read 128 contiguous bytes.
// ------------------------------------------------------------------------------------------
constexpr int kFT_H = 8, kFT_W = 32, kFT_LD = 36;

template <typename T>
__device__ __forceinline__ void first_load_halo(const GconvDev& d, const T* __restrict__ x, float (*halo)[kFT_LD], int b,
                                                int i0, int j0) {
  for (int e = threadIdx.x; e < (kFT_H + 2) * (kFT_W + 2); e += 256) {
    const int r = e / (kFT_W + 2), c = e - r * (kFT_W + 2);
    const int gi = i0 - 1 + r, gj = j0 - 1 + c;
    float v = 0.f;
    if ((unsigned)gi < (unsigned)d.Hin && (unsigned)gj < (unsigned)d.Win)
      v = Elem<T>::ld(x + ((long long)(b * d.Hin + gi) * d.Win + gj) * d.ld_in);
    halo[r][c] = v;
  }
}

template <typename T>
__global__ void __launch_bounds__(256, 2)
first_conv_fprop_tiled_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ wp, T* __restrict__ y,
                              float* __restrict__ stats_ws, int tiles_w, int tiles_h, int ntiles) {
  __shared__ float halo[kFT_H + 2][kFT_LD];
  const int g = threadIdx.x & 7, pl = threadIdx.x >> 3;
  // weights by window position (row a = dy + 1, column c = dx + 1)
  __shared__ int tmap[9];
  if (threadIdx.x < 9) tmap[(d.tap_dy[threadIdx.x] + 1) * 3 + d.tap_dx[threadIdx.x] + 1] = threadIdx.x;
  __syncthreads();
  float wr[3][3][8];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int t = tmap[a * 3 + c];
#pragma unroll
      for (int i = 0; i < 8; ++i) wr[a][c][i] = Elem<T>::ld(wp + (long long)(g * 8 + i) * 9 + t);
    }
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tj = tile % tiles_w;
    const int rest = tile / tiles_w;
    const int ti = rest % tiles_h, b = rest / tiles_h;
    const int i0 = ti * kFT_H, j0 = tj * kFT_W;
    __syncthreads();
    first_load_halo<T>(d, x, halo, b, i0, j0);
    __syncthreads();
    const int j = j0 + pl;
    float win[3][3];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 3; ++c) win[a][c] = halo[a][pl + c];
#pragma unroll
    for (int r = 0; r < kFT_H; ++r) {
#pragma unroll
      for (int c = 0; c < 3; ++c) win[2][c] = halo[r + 2][pl + c];
      float acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] = fmaf(win[a][c], wr[a][c][i], acc[i]);
      const int i = i0 + r;
      if (i < d.Hm && j < d.Wm) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          acc[k] = Elem<T>::round(acc[k]);
          s[k] += acc[k];
          q[k] = fmaf(acc[k], acc[k], q[k]);
        }
        store8(y + ((long long)(b * d.Hm + i) * d.Wm + j) * d.ld_out + g * 8, acc);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) { win[0][c] = win[1][c]; win[1][c] = win[2][c]; }
    }
  }
  if (stats_ws) {
    // deterministic: per-warp partials in shared memory, summed in a fixed order (float atomics would make the
    // BatchNorm statistics -- and through ReLU flips the whole step -- differ from run to run)
    __shared__ float wstat[8][2][64];
    const int warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      // the 4 pixel columns of a warp share a channel group: combine them first (lanes g, g+8, g+16, g+24)
      float a = s[i], c = q[i];
      a += __shfl_xor_sync(0xffffffffu, a, 8); a += __shfl_xor_sync(0xffffffffu, a, 16);
      c += __shfl_xor_sync(0xffffffffu, c, 8); c += __shfl_xor_sync(0xffffffffu, c, 16);
      if ((threadIdx.x & 31) < 8) { wstat[warp][0][g * 8 + i] = a; wstat[warp][1][g * 8 + i] = c; }
    }
    __syncthreads();
    if (threadIdx.x < 128) {
      const int which = threadIdx.x >> 6, c = threadIdx.x & 63;
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += wstat[w][which][c];
      stats_ws[((long long)blockIdx.x * 2 + which) * 64 + c] = v;
    }
  }
}

// dWp[t][n] partial per block: partials[block][9][64]
// Software-pipelined: the halo of the NEXT tile and the dY rows of the next row pair are loaded (into registers)
// before the FMAs of the current ones, so global-load latency hides behind the 72 FMAs per pixel.
template <typename T>
__device__ __forceinline__ float first_halo_elem(const GconvDev& d, const T* __restrict__ x, int b, int i0, int j0, int e) {
  const int r = e / (kFT_W + 2), c = e - r * (kFT_W + 2);
  const int gi = i0 - 1 + r, gj = j0 - 1 + c;
  if (e < (kFT_H + 2) * (kFT_W + 2) && (unsigned)gi < (unsigned)d.Hin && (unsigned)gj < (unsigned)d.Win)
    return Elem<T>::ld(x + ((long long)(b * d.Hin + gi) * d.Win + gj) * d.ld_in);
  return 0.f;
}

template <typename T>
__global__ void __launch_bounds__(256, 2)
first_conv_wgrad_tiled_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ gy, float* __restrict__ partials,
                              int tiles_w, int tiles_h, int ntiles) {
  __shared__ float halo[kFT_H + 2][kFT_LD];
  const int g = threadIdx.x & 7, pl = threadIdx.x >> 3;
  float acc[3][3][8];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[a][c][i] = 0.f;
  auto decode = [&](int tile, int& b, int& i0, int& j0) {
    const int tj = tile % tiles_w;
    const int rest = tile / tiles_w;
    b = rest / tiles_h;
    i0 = (rest % tiles_h) * kFT_H;
    j0 = tj * kFT_W;
  };
  // dY rows travel packed (16 bytes per pixel and channel group for bf16) and are unpacked at use; the four rows of
  // the NEXT half tile are requested before the FMAs of the current half (prefetch distance ~4 x 72 FMAs)
  struct Row { uint4 a, b; };
  auto load_half = [&](int tile, int half, Row* dst) {
    int b, i0, j0;
    decode(tile, b, i0, j0);
    const int j = j0 + pl;
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int i = i0 + half * 4 + rr;
      dst[rr].a = make_uint4(0u, 0u, 0u, 0u);
      dst[rr].b = make_uint4(0u, 0u, 0u, 0u);
      if (tile < ntiles && i < d.Hm && j < d.Wm) {
        const T* src = gy + ((long long)(b * d.Hm + i) * d.Wm + j) * d.ld_out + g * 8;
        dst[rr].a = *reinterpret_cast<const uint4*>(src);
        if constexpr (sizeof(T) == 4) dst[rr].b = *reinterpret_cast<const uint4*>(src + 4);
      }
    }
  };
  auto unpack = [&](const Row& r, float v[8]) {
    if constexpr (sizeof(T) == 4) {
      v[0] = __uint_as_float(r.a.x); v[1] = __uint_as_float(r.a.y); v[2] = __uint_as_float(r.a.z); v[3] = __uint_as_float(r.a.w);
      v[4] = __uint_as_float(r.b.x); v[5] = __uint_as_float(r.b.y); v[6] = __uint_as_float(r.b.z); v[7] = __uint_as_float(r.b.w);
    } else {
      const uint32_t w[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
    }
  };
  int tile = blockIdx.x;
  float h0 = 0.f, h1 = 0.f;                       // this thread's two halo elements of the tile about to be staged
  Row cur[4], nxt[4];
  if (tile < ntiles) {
    int b, i0, j0;
    decode(tile, b, i0, j0);
    h0 = first_halo_elem<T>(d, x, b, i0, j0, threadIdx.x);
    h1 = first_halo_elem<T>(d, x, b, i0, j0, threadIdx.x + 256);
  }
  load_half(tile, 0, cur);
  for (; tile < ntiles; tile += gridDim.x) {
    __syncthreads();                              // everyone is done with the previous halo
    (&halo[0][0])[(threadIdx.x / (kFT_W + 2)) * kFT_LD + threadIdx.x % (kFT_W + 2)] = h0;
    if (threadIdx.x + 256 < (kFT_H + 2) * (kFT_W + 2))
      (&halo[0][0])[((threadIdx.x + 256) / (kFT_W + 2)) * kFT_LD + (threadIdx.x + 256) % (kFT_W + 2)] = h1;
    __syncthreads();
    const int nxt_tile = tile + gridDim.x;
    if (nxt_tile < ntiles) {                      // prefetch the next tile's halo
      int nb, ni0, nj0;
      decode(nxt_tile, nb, ni0, nj0);
      h0 = first_halo_elem<T>(d, x, nb, ni0, nj0, threadIdx.x);
      h1 = first_halo_elem<T>(d, x, nb, ni0, nj0, threadIdx.x + 256);
    }
    float win[3][3];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 3; ++c) win[a][c] = halo[a][pl + c];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      if (half == 0) load_half(tile, 1, nxt); else load_half(nxt_tile, 0, nxt);
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int r = half * 4 + rr;
        float gv[8];
        unpack(cur[rr], gv);
#pragma unroll
        for (int c = 0; c < 3; ++c) win[2][c] = halo[r + 2][pl + c];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
          for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[a][c][k] = fmaf(win[a][c], gv[k], acc[a][c][k]);
#pragma unroll
        for (int c = 0; c < 3; ++c) { win[0][c] = win[1][c]; win[1][c] = win[2][c]; }
      }
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) cur[rr] = nxt[rr];
    }
  }
  __syncthreads();
  // window position (a, c) -> tap index t (a 9-entry table in shared memory), then per-warp partials without atomics
  __shared__ int tmap[9];
  __shared__ float wred[8][9 * 64];
  if (threadIdx.x < 9) tmap[(d.tap_dy[threadIdx.x] + 1) * 3 + d.tap_dx[threadIdx.x] + 1] = threadIdx.x;
  __syncthreads();
  const int warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int t = tmap[a * 3 + c];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float v = acc[a][c][k];
        v += __shfl_xor_sync(0xffffffffu, v, 8);      // the 4 pixel columns of a warp share the channel group
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if ((threadIdx.x & 31) < 8) wred[warp][t * 64 + g * 8 + k] = v;
      }
    }
  __syncthreads();
  float* out = partials + (long long)blockIdx.x * 9 * 64;
  for (int e = threadIdx.x; e < 9 * 64; e += 256) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += wred[w][e];
    out[e] = v;
  }
}

static bool first_tiled_ok(const unetb200_gconv_t* d) {
  static const bool v1 = getenv("UNETB200_FIRST_V1") != nullptr;
  if (v1) return false;
  if (d->Cin != 1 || d->N != 64 || d->ld_out % 8) return false;
  for (int t = 0; t < 9; ++t)
    if (d->tap_dy[t] < -1 || d->tap_dy[t] > 1 || d->tap_dx[t] < -1 || d->tap_dx[t] > 1) return false;
  return (long long)d->B * d->Hin * d->Win < (1LL << 31);
}

// four pixels per thread (C_in = 2..4): needs the plain 3x3 window and W % 4 == 0
static bool first_px4_ok(const unetb200_gconv_t* d) {
  static const bool v1 = getenv("UNETB200_FIRST_V1") != nullptr;
  if (v1) return false;
  if (d->Cin < 2 || d->Cin > 4 || (d->Wm & 3)) return false;
  bool seen[9] = {false};
  for (int t = 0; t < 9; ++t) {
    const int dy = d->tap_dy[t], dx = d->tap_dx[t];
    if (dy < -1 || dy > 1 || dx < -1 || dx > 1 || seen[(dy + 1) * 3 + dx + 1]) return false;
    seen[(dy + 1) * 3 + dx + 1] = true;
  }
  return true;
}

static bool first_common(const unetb200_gconv_t* d) {
  if (d->ntaps != 9 || d->in_scale != 1 || d->out_scale != 1 || d->nquad != 1) return false;
  if (d->in_off_y || d->in_off_x || d->out_off_y || d->out_off_x) return false;
  if (d->Hm != d->Hout || d->Wm != d->Wout || d->Hm != d->Hin || d->Wm != d->Win) return false;
  if (d->N % 8 || d->N > 256 || d->ld_out % 8) return false;
  if ((long long)d->B * d->Hm * d->Wm >= (1LL << 31) - (1 << 20)) return false;
  return true;
}

int first_fprop_supported(const unetb200_gconv_t* d, const void* y) {
  if (!first_common(d) || d->Cin < 1 || d->Cin > 4) return 0;
  const int G = d->N / 8;
  if (256 % G) return 0;
  return aligned16(y) ? 1 : 0;
}

static int first_blocks(long long M, int lanes) {
  long long b = (M + (long long)lanes * 16 - 1) / ((long long)lanes * 16);
  long long cap = (long long)sm_count() * 6;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

long long first_fprop_tiles(const unetb200_gconv_t* d) {
  if (!first_common(d)) return 0;
  return first_blocks((long long)d->B * d->Hm * d->Wm, 256 / (d->N / 8));
}

int first_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, void* y, double* stats,
                float* stats_ws, cudaStream_t s) {
  const int blocks = first_blocks(g.M, 256 / (d->N / 8));
  if (first_tiled_ok(d)) {
    const int tiles_w = (d->Wm + kFT_W - 1) / kFT_W, tiles_h = (d->Hm + kFT_H - 1) / kFT_H;
    const int ntiles = d->B * tiles_w * tiles_h;
    with_elem(d->dtype, [&](auto t) {
      using T = decltype(t);
      first_conv_fprop_tiled_kernel<T><<<blocks, 256, 0, s>>>(g, (const T*)x, (const T*)wp, (T*)y,
                                                              stats ? stats_ws : nullptr, tiles_w, tiles_h, ntiles);
    });
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "first_conv_fprop_tiled");
    if (stats) return launch_stats_reduce(stats_ws, blocks, 2 * d->N, stats, s);
    return 0;
  }
  if (first_px4_ok(d)) {
    with_elem(d->dtype, [&](auto t) {
      with_int<2, 3, 4>(d->Cin, [&](auto CIN) {
        using T = decltype(t);
        first_conv_fprop_px4_kernel<T, CIN><<<blocks, 256, 0, s>>>(g, (const T*)x, (const T*)wp, (T*)y,
                                                                   stats ? stats_ws : nullptr);
      });
    });
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "first_conv_fprop_px4");
    if (stats) return launch_stats_reduce(stats_ws, blocks, 2 * d->N, stats, s);
    return 0;
  }
  with_elem(d->dtype, [&](auto t) {
    with_int<1, 2, 3, 4>(d->Cin, [&](auto CIN) {
      using T = decltype(t);
      first_conv_fprop_kernel<T, CIN><<<blocks, 256, 0, s>>>(g, (const T*)x, (const T*)wp, (T*)y,
                                                             stats ? stats_ws : nullptr);
    });
  });
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "first_conv_fprop");
  if (stats) return launch_stats_reduce(stats_ws, blocks, 2 * d->N, stats, s);
  return 0;
}

int first_wgrad_supported(const unetb200_gconv_t* d, const void* gy) {
  if (!first_common(d) || d->Cin != 1 || d->N > 128) return 0;
  const int G = d->N / 8;
  if (G & (G - 1)) return 0;
  return (!gy || aligned16(gy)) ? 1 : 0;
}

int first_wgrad_splits(const unetb200_gconv_t* d) {
  return first_blocks((long long)d->B * d->Hm * d->Wm, 256 / (d->N / 8));
}

int first_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials,
                int splits, cudaStream_t s) {
  if (first_tiled_ok(d)) {
    const int tiles_w = (d->Wm + kFT_W - 1) / kFT_W, tiles_h = (d->Hm + kFT_H - 1) / kFT_H;
    const int ntiles = d->B * tiles_w * tiles_h;
    with_elem(d->dtype, [&](auto t) {
      using T = decltype(t);
      first_conv_wgrad_tiled_kernel<T><<<splits, 256, 0, s>>>(g, (const T*)x, (const T*)gy, partials, tiles_w, tiles_h,
                                                              ntiles);
    });
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "first_conv_wgrad_tiled");
    return 0;
  }
  with_elem(d->dtype, [&](auto t) {
    using T = decltype(t);
    first_conv_wgrad_kernel<T><<<splits, 256, 0, s>>>(g, (const T*)x, (const T*)gy, partials);
  });
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "first_conv_wgrad");
  return 0;
}

}  // namespace ub
