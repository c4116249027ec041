// CUDA-core (fp32 FMA) implicit-GEMM engine for the generalised convolution of unetb200.h.
// It handles every shape (C_in = 1 or 3 first layer, widths that do not fill a UMMA tile, unaligned
// channel slices) and is the arithmetic of the fp32 "exactness" mode; gconv.cu routes a descriptor here
// when no specialised engine covers it.  Also the split-K reductions and the weight packing.
#include "gconv.cuh"

namespace ub {

constexpr int FBM = 128, FBN = 64, FBK = 16;   // fprop tile
constexpr int WBK = 64, WBN = 64, WBM = 16;    // wgrad tile (K rows x N cols, M step)

__device__ __forceinline__ void decode_m(const GconvDev& d, long long m, int& b, int& i, int& j) {
  j = (int)(m % d.Wm);
  long long r = m / d.Wm;
  i = (int)(r % d.Hm);
  b = (int)(r / d.Hm);
}
// source element offset of (b,i,j) under tap t, or -1 when it falls in the padding
__device__ __forceinline__ long long src_offset(const GconvDev& d, int b, int i, int j, int t) {
  int si = i * d.in_scale + d.tap_dy[t] + d.in_off_y;
  int sj = j * d.in_scale + d.tap_dx[t] + d.in_off_x;
  if (si < 0 || si >= d.Hin || sj < 0 || sj >= d.Win) return -1;
  return (((long long)b * d.Hin + si) * d.Win + sj) * d.ld_in;
}
__device__ __forceinline__ long long dst_offset(const GconvDev& d, int b, int i, int j, int q) {
  int oi = i * d.out_scale + (q >> 1) + d.out_off_y;
  int oj = j * d.out_scale + (q & 1) + d.out_off_x;
  return (((long long)b * d.Hout + oi) * d.Wout + oj) * d.ld_out;
}

template <typename T>
__device__ __forceinline__ void load4(const T* p, float v[4]);
template <>
__device__ __forceinline__ void load4<float>(const float* p, float v[4]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
template <>
__device__ __forceinline__ void load4<__nv_bfloat16>(const __nv_bfloat16* p, float v[4]) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  v[0] = __uint_as_float(r.x << 16); v[1] = __uint_as_float(r.x & 0xffff0000u);
  v[2] = __uint_as_float(r.y << 16); v[3] = __uint_as_float(r.y & 0xffff0000u);
}
__device__ __forceinline__ void store4(float* p, const float v[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void store4(__nv_bfloat16* p, const float v[4]) {
  uint2 r;
  r.x = pack_bf16x2(v[0], v[1]);
  r.y = pack_bf16x2(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = r;
}

// ------------------------------------------------------------------------------------------
// fprop: D[128 x 64] tile per block, 256 threads, 8x4 micro-tile, K chunks of 16
// ------------------------------------------------------------------------------------------
// FBN_ = 64 / 32 / 16 output channels per block (narrow layers: a 64-wide tile wastes 3/4 of its FMAs at N = 16);
// the block keeps 256 threads with an 8 x 4 micro-tile, so FBM_ = 8 * 256 / (FBN_ / 4) = 128 / 256 / 512 pixels.
template <typename T, bool VEC, int FBN_>
__global__ void __launch_bounds__(256)
gconv_fprop_simt_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ wp, const float* __restrict__ bias,
                        T* __restrict__ y, float* __restrict__ stats_ws) {
  constexpr int TX = FBN_ / 4, TY = 256 / TX, FBM_ = TY * 8;
  constexpr int FBM = FBM_, FBN = FBN_;   // (shadow the file-scope defaults inside this kernel)
  __shared__ __align__(16) float As[FBK][FBM + 4];
  __shared__ __align__(16) float Bs[FBK][FBN + 4];
  __shared__ int pb[FBM], pi[FBM], pj[FBM];
  __shared__ float wstat[8][2][FBN];      // per-warp BatchNorm partials (256 threads = 8 warps)
  const int tid = threadIdx.x;
  const long long m0 = (long long)blockIdx.x * FBM;
  const int n0 = blockIdx.y * FBN;
  for (int t = tid; t < FBM; t += 256) {
    long long m = m0 + t;
    int b = -1, i = 0, j = 0;
    if (m < d.M) decode_m(d, m, b, i, j);
    pb[t] = b; pi[t] = i; pj[t] = j;
  }
  __syncthreads();
  const int tx = tid % TX, ty = tid / TX;
  float acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;

  for (int k0 = 0; k0 < d.K; k0 += FBK) {
    if (VEC) {
      for (int it = tid; it < FBM * 2; it += 256) {  // A: item -> pixel it/2, 8 channels
        const int ml = it >> 1, kv = (it & 1) * 8;
        const int k = k0 + kv;
        const int t = k / d.Cin, c = k - t * d.Cin;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
        if (pb[ml] >= 0) {
          long long off = src_offset(d, pb[ml], pi[ml], pj[ml], t);
          if (off >= 0) load8(x + off + c, v);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) As[kv + e][ml] = v[e];
      }
      if (tid < FBN * 4) {  // B: thread -> row n tid/4, 4 consecutive k
        const int nl = tid >> 2, k4 = (tid & 3) * 4;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (n0 + nl < d.N) load4<T>(wp + (long long)(n0 + nl) * d.K + k0 + k4, v);
#pragma unroll
        for (int e = 0; e < 4; ++e) Bs[k4 + e][nl] = v[e];
      }
    } else {
#pragma unroll
      for (int r = 0; r < FBM / 16; ++r) {
        const int e = tid + r * 256;
        const int kl = e & 15, ml = e >> 4;
        const int k = k0 + kl;
        float v = 0.f;
        if (k < d.K && pb[ml] >= 0) {
          const int t = k / d.Cin, c = k - t * d.Cin;
          long long off = src_offset(d, pb[ml], pi[ml], pj[ml], t);
          if (off >= 0) v = Elem<T>::ld(x + off + c);
        }
        As[kl][ml] = v;
      }
      for (int e = tid; e < FBN * 16; e += 256) {
        const int kl = e & 15, nl = e >> 4;
        const int k = k0 + kl;
        float v = 0.f;
        if (k < d.K && n0 + nl < d.N) v = Elem<T>::ld(wp + (long long)(n0 + nl) * d.K + k);
        Bs[kl][nl] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < FBK; ++kk) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[4] = {b0.x, b0.y, b0.z, b0.w};
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
    }
    __syncthreads();
  }

  // epilogue
  const int nb = n0 + tx * 4;
  float bs[4] = {0.f, 0.f, 0.f, 0.f};
  int qq[4], cc[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    int n = nb + c;
    qq[c] = (n < d.N) ? n / d.Cq : 0;
    cc[c] = (n < d.N) ? n - qq[c] * d.Cq : 0;
    if (bias && n < d.N) bs[c] = Elem<T>::round(bias[cc[c]]);
  }
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int ml = ty * 8 + r;
    if (pb[ml] < 0) continue;
    float v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      v[c] = Elem<T>::round(acc[r][c] + bs[c]);
      if (nb + c < d.N) { s1[c] += v[c]; s2[c] += v[c] * v[c]; }
    }
    if (VEC) {
      if (nb < d.N) store4(y + dst_offset(d, pb[ml], pi[ml], pj[ml], qq[0]) + cc[0], v);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (nb + c < d.N) Elem<T>::st(y + dst_offset(d, pb[ml], pi[ml], pj[ml], qq[c]) + cc[c], v[c]);
    }
  }
  if (stats_ws) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      // the ty rows of a warp first (lanes with the same tx), then the 8 warps in a fixed order below (float atomics
      // would make the statistics run-dependent)
      float a = s1[c], b = s2[c];
#pragma unroll
      for (int o = TX; o < 32; o <<= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if ((tid & 31) < TX) { wstat[tid >> 5][0][tx * 4 + c] = a; wstat[tid >> 5][1][tx * 4 + c] = b; }
    }
    __syncthreads();
    // per-tile partials [tile][2][N]: plain stores, reduced by stats_reduce_kernel (no global atomics)
    if (tid < 2 * FBN) {
      const int which = tid / FBN, c = tid % FBN;
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += wstat[w][which][c];
      if (n0 + c < d.N) stats_ws[((long long)blockIdx.x * 2 + which) * d.N + n0 + c] = v;
    }
  }
}

// stats[col] += sum over tiles of ws[tile][col]; ws rows have C2 = 2*C columns laid out like stats
__global__ void stats_reduce_kernel(const float* __restrict__ ws, long long ntiles, int C2, double* __restrict__ stats) {
  __shared__ double red[8][33];
  const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  double acc = 0.0;
  if (col < C2)
    for (long long t = (long long)blockIdx.y * 8 + ry; t < ntiles; t += (long long)gridDim.y * 8)
      acc += (double)ws[t * C2 + col];
  red[ry][lane] = acc;
  __syncthreads();
  if (ry == 0 && col < C2) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][lane];
    atomicAdd(stats + col, s);
  }
}

int launch_stats_reduce(const float* ws, long long ntiles, int C2, double* stats, cudaStream_t s) {
  long long sy = ntiles / 32;
  if (sy < 1) sy = 1;
  if (sy > 256) sy = 256;
  stats_reduce_kernel<<<dim3((unsigned)((C2 + 31) / 32), (unsigned)sy), 256, 0, s>>>(ws, ntiles, C2, stats);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "stats_reduce");
  return 0;
}

// ------------------------------------------------------------------------------------------
// wgrad: dWp[64 k x 64 n] tile per block, reduction over a slice of m, 4x4 micro-tile
// ------------------------------------------------------------------------------------------
// WBN_ = 64 / 32 / 16 columns per block; 256 threads with a 4 x 4 micro-tile, so WBK_ = 4 * 256 / (WBN_ / 4) = 64 / 128 / 256 rows
template <typename T, bool VEC, int WBN_>
__global__ void __launch_bounds__(256)
gconv_wgrad_simt_kernel(GconvDev d, const T* __restrict__ x, const T* __restrict__ gy, float* __restrict__ partials,
                        long long m_per_split) {
  constexpr int TN = WBN_ / 4, TK = 256 / TN, WBK_ = TK * 4;
  constexpr int WBK = WBK_, WBN = WBN_;   // (shadow the file-scope defaults inside this kernel)
  __shared__ __align__(16) float As[WBM][WBK + 4];
  __shared__ __align__(16) float Gs[WBM][WBN + 4];
  const int tid = threadIdx.x;
  const int k0 = blockIdx.x * WBK, n0 = blockIdx.y * WBN;
  const long long mb = (long long)blockIdx.z * m_per_split;
  long long me = mb + m_per_split;
  if (me > d.M) me = d.M;
  const int tk = tid / TN, tn = tid % TN;
  float acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;

  for (long long m0 = mb; m0 < me; m0 += WBM) {
    if (VEC) {
      constexpr int AV = WBK / 4, GV = WBN / 4;          // float4 items per pixel
      for (int it = tid; it < WBM * (AV + GV); it += 256) {
        const int ml = it / (AV + GV), r = it - ml * (AV + GV);
        const long long m = m0 + ml;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (m < me) {
          int b, i, j;
          decode_m(d, m, b, i, j);
          if (r < AV) {
            const int k = k0 + r * 4;
            if (k < d.K) {
              const int t = k / d.Cin, c = k - t * d.Cin;
              long long off = src_offset(d, b, i, j, t);
              if (off >= 0) load4<T>(x + off + c, v);
            }
          } else {
            const int n = n0 + (r - AV) * 4;
            if (n < d.N) {
              const int q = n / d.Cq, co = n - q * d.Cq;
              load4<T>(gy + dst_offset(d, b, i, j, q) + co, v);
            }
          }
        }
        if (r < AV) *reinterpret_cast<float4*>(&As[ml][r * 4]) = make_float4(v[0], v[1], v[2], v[3]);
        else *reinterpret_cast<float4*>(&Gs[ml][(r - AV) * 4]) = make_float4(v[0], v[1], v[2], v[3]);
      }
    } else {
      for (int e = tid; e < WBM * (WBK + WBN); e += 256) {
        const int ml = e / (WBK + WBN), r = e - ml * (WBK + WBN);
        const long long m = m0 + ml;
        float v = 0.f;
        if (m < me) {
          int b, i, j;
          decode_m(d, m, b, i, j);
          if (r < WBK) {
            const int k = k0 + r;
            if (k < d.K) {
              const int t = k / d.Cin, c = k - t * d.Cin;
              long long off = src_offset(d, b, i, j, t);
              if (off >= 0) v = Elem<T>::ld(x + off + c);
            }
          } else {
            const int n = n0 + r - WBK;
            if (n < d.N) {
              const int q = n / d.Cq, co = n - q * d.Cq;
              v = Elem<T>::ld(gy + dst_offset(d, b, i, j, q) + co);
            }
          }
        }
        if (r < WBK) As[ml][r] = v;
        else Gs[ml][r - WBK] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < WBM; ++mm) {
      float4 a4 = *reinterpret_cast<const float4*>(&As[mm][tk * 4]);
      float4 g4 = *reinterpret_cast<const float4*>(&Gs[mm][tn * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], g[c], acc[r][c]);
    }
    __syncthreads();
  }
  float* out = partials + (long long)blockIdx.z * d.K * d.N;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int k = k0 + tk * 4 + r;
    if (k >= d.K) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int n = n0 + tn * 4 + c;
      if (n < d.N) out[(long long)k * d.N + n] = acc[r][c];
    }
  }
}

__global__ void wgrad_reduce_kernel(const float* __restrict__ partials, int splits, int Cin, long long K, int N,
                                    int Cq, float* __restrict__ dst, long long st, long long sc, long long sq,
                                    long long sn, int accumulate) {
  const long long total = K * N;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int p = 0; p < splits; ++p) s += partials[(long long)p * total + idx];
    const long long k = idx / N;
    const int n = (int)(idx - k * N);
    const long long t = k / Cin, c = k - t * Cin;
    const int q = n / Cq, co = n - q * Cq;
    float* o = dst + t * st + c * sc + q * sq + (long long)co * sn;
    *o = accumulate ? *o + s : s;
  }
}

template <typename D>
__global__ void pack_weights_kernel(const float* __restrict__ src, D* __restrict__ dst, long long n0, long long n1,
                                    long long n2, long long s0, long long s1, long long s2, long long off) {
  const long long total = n0 * n1 * n2;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long i2 = idx % n2;
    long long r = idx / n2;
    long long i1 = r % n1, i0 = r / n1;
    Elem<D>::st(dst + idx, src[off + i0 * s0 + i1 * s1 + i2 * s2]);
  }
}

// Split reduction + transpose for the case dst[co * sn + k] (k = t*Cin + c linear in the parameter: a
// channels_last weight gradient): partial rows [k][n] are read coalesced along n, summed over the splits in a
// fixed order (deterministic), transposed through shared memory and written coalesced along k.
template <int SL>
__global__ void __launch_bounds__(32 * SL) wgrad_reduce_t_kernel(const float* __restrict__ partials, int splits, long long K,
                                                                 int N, float* __restrict__ dst, long long sn, int accumulate) {
  // many splits: a block owns an 8 (k) x 32 (n) tile; thread (tx, ty) sums column n0 + tx over the splits
  // ty, ty + SL, ... with its 8 row sums in registers (8 loads in flight), then the SL lanes are combined in
  // a fixed order through shared memory (deterministic)
  __shared__ float red[SL][8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long k0 = (long long)blockIdx.x * 8;
  const int n0 = blockIdx.y * 32;
  const long long total = K * N;
  const int n = n0 + tx;
  float acc[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) acc[r] = 0.f;
  if (n < N) {
    for (int sp = ty; sp < splits; sp += SL) {
      const float* p = partials + (long long)sp * total + k0 * N + n;
      float v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) v[r] = (k0 + r < K) ? p[(long long)r * N] : 0.f;
#pragma unroll
      for (int r = 0; r < 8; ++r) acc[r] += v[r];
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) red[ty][r][tx] = acc[r];
  __syncthreads();
  if (threadIdx.x < 256) {
    const int kl = threadIdx.x & 7, nl = threadIdx.x >> 3;
    float v = 0.f;
#pragma unroll 4
    for (int j = 0; j < SL; ++j) v += red[j][kl][nl];
    const long long k = k0 + kl;
    const int nn = n0 + nl;
    if (k < K && nn < N) {
      float* o = dst + (long long)nn * sn + k;
      *o = accumulate ? *o + v : v;
    }
  }
}

// few splits: threads over the tile (4 rows each), loop over the splits
__global__ void __launch_bounds__(256) wgrad_reduce_t4_kernel(const float* __restrict__ partials, int splits, long long K,
                                                               int N, float* __restrict__ dst, long long sn, int accumulate) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8
  const long long k0 = (long long)blockIdx.x * 32;
  const int n0 = blockIdx.y * 32;
  const long long total = K * N;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  const int n = n0 + tx;
  if (n < N) {
    for (int sp = 0; sp < splits; ++sp) {
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const long long k = k0 + ty + 8 * r;
        v[r] = k < K ? partials[(long long)sp * total + k * N + n] : 0.f;
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) s[r] += v[r];
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) tile[ty + 8 * r][tx] = s[r];
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int nn = n0 + ty + 8 * r;
    const long long k = k0 + tx;
    if (k < K && nn < N) {
      float* o = dst + (long long)nn * sn + k;
      const float v = tile[tx][ty + 8 * r];
      *o = accumulate ? *o + v : v;
    }
  }
}

// dst[i0][i1][i2] = cast(src[off + i0 + i1*s1 + i2*s2]) (source contiguous along i0): 32 x 32 transpose tiles
// of (i0, i2) per i1, reads coalesced along i0, writes coalesced along i2.
template <typename D>
__global__ void __launch_bounds__(256) pack_weights_t_kernel(const float* __restrict__ src, D* __restrict__ dst, int n0,
                                                              int n1, int n2, long long s1, long long s2, long long off) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int a0 = blockIdx.x * 32, c0 = blockIdx.y * 32, i1 = blockIdx.z;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i2 = c0 + ty + 8 * r, i0 = a0 + tx;
    tile[ty + 8 * r][tx] = (i0 < n0 && i2 < n2) ? src[off + i0 + i1 * s1 + (long long)i2 * s2] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i0 = a0 + ty + 8 * r, i2 = c0 + tx;
    if (i0 < n0 && i2 < n2) Elem<D>::st(dst + ((long long)i0 * n1 + i1) * n2 + i2, tile[tx][ty + 8 * r]);
  }
}

// ---- multi-tensor weight packing ------------------------------------------------------------------------------
// Every 3x3 / transposed-conv weight of the network is packed into its GEMM operand(s) by ONE launch per step (the
// job table travels by value in the kernel parameters): job j is dst[i0][i1][i2] = cast(src[off + i0*s0 + i1*s1 +
// i2*s2]), cut into 32 (i0) x 32 (i2) tiles per i1.  A tile is read along whichever of i0 / i2 is contiguous in the
// source and always written along i2 (contiguous in the destination), through shared memory when the two differ.

// Split reduction of MANY layers in one launch (the 22 per-layer launches of a backward pass were launch / ramp bound:
// 0.64 ms for ~0.5 GB): job j reduces partials[s][(t,c)][n] over its splits in a fixed order (deterministic) and
// scatters into the parameter layout exactly like unetb200_wgrad_reduce.  A block owns an 8 (k) x 32 (n) tile of
// one job; its 8 split lanes each sum every 8th split (8 row loads in flight per thread), then the lanes are
// combined in a fixed order through shared memory; the tile is written k-fastest (channels_last conv weight:
// k-linear) or n-fastest (sn == 1), whichever is contiguous in the parameter.
constexpr int kMaxReduceJobs = 32;
struct ReduceJob {
  const float* partials;
  float* dst;
  long long st, sc, sq, sn, K;
  int splits, Cin, N, Cq;
  int tiles_n, block0, accumulate, pad_;      // pad_ = tile mode: 0 = 32 x 32 (few splits), 1 = 8 x 32 x 8 split lanes
};
struct alignas(16) ReduceTable {
  ReduceJob job[kMaxReduceJobs];
  int njobs;
};

__global__ void __launch_bounds__(256) wgrad_reduce_multi_kernel(const __grid_constant__ ReduceTable T) {
  __shared__ float red[8][8][33];
  int lo = 0, hi = T.njobs - 1;
  while (lo < hi) {                   // last job with block0 <= blockIdx.x
    const int mid = (lo + hi + 1) >> 1;
    if (T.job[mid].block0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const ReduceJob& J = T.job[lo];
  const int local = (int)blockIdx.x - J.block0;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long total = J.K * J.N;
  const int n0 = (local % J.tiles_n) * 32;
  const int n = n0 + tx;
  const bool n_fast = J.sn == 1;
  auto store = [&](long long k, int nn, float v) {
    if (k < J.K && nn < J.N) {
      const long long t = k / J.Cin, c = k - t * J.Cin;
      const int q = nn / J.Cq, co = nn - q * J.Cq;
      float* o = J.dst + t * J.st + c * J.sc + q * J.sq + (long long)co * J.sn;
      *o = J.accumulate ? *o + v : v;
    }
  };
  if (J.pad_ == 0) {
    // few splits (the deep layers: large K x N): a 32 (k) x 32 (n) tile per block, every thread sums 4 rows over the
    // splits in order -- all 256 threads load, 12-30 KB per block
    float (*tile)[33] = reinterpret_cast<float (*)[33]>(&red[0][0][0]);
    const long long k0 = (long long)(local / J.tiles_n) * 32;
    float sacc[4] = {0.f, 0.f, 0.f, 0.f};
    if (n < J.N) {
      for (int sp = 0; sp < J.splits; ++sp) {
        float v[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const long long k = k0 + ty + 8 * r;
          v[r] = k < J.K ? J.partials[(long long)sp * total + k * J.N + n] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) sacc[r] += v[r];
      }
    }
    if (n_fast) {
#pragma unroll
      for (int r = 0; r < 4; ++r) store(k0 + ty + 8 * r, n, sacc[r]);
      return;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) tile[ty + 8 * r][tx] = sacc[r];
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) store(k0 + tx, n0 + ty + 8 * r, tile[tx][ty + 8 * r]);
    return;
  }
  // many splits (the shallow layers: small K x N, split over > 100 CTAs): an 8 (k) x 32 (n) tile, 8 split lanes
  const long long k0 = (long long)(local / J.tiles_n) * 8;
  float acc[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) acc[r] = 0.f;
  if (n < J.N) {
    for (int sp = ty; sp < J.splits; sp += 8) {
      const float* p = J.partials + (long long)sp * total + k0 * J.N + n;
      float v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) v[r] = (k0 + r < J.K) ? p[(long long)r * J.N] : 0.f;
#pragma unroll
      for (int r = 0; r < 8; ++r) acc[r] += v[r];
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) red[ty][r][tx] = acc[r];
  __syncthreads();
  const int kl = n_fast ? (threadIdx.x >> 5) : (threadIdx.x & 7);
  const int nl = n_fast ? (threadIdx.x & 31) : (threadIdx.x >> 3);
  float v = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) v += red[j][kl][nl];
  store(k0 + kl, n0 + nl, v);
}

constexpr int kMaxPackJobs = 40;
struct PackJob {
  const float* src;
  void* dst;
  long long s0, s1, s2, off;
  int n0, n1, n2;
  int tiles2;      // ceil(n2 / 32)
  int block0;      // first block of this job
  int pad_;
};
struct alignas(16) PackTable {
  PackJob job[kMaxPackJobs];
  int njobs;
};

template <typename D>
__global__ void __launch_bounds__(256) pack_multi_kernel(const __grid_constant__ PackTable T) {
  __shared__ float tile[32][33];
  int lo = 0, hi = T.njobs - 1;
  while (lo < hi) {                   // last job with block0 <= blockIdx.x
    const int mid = (lo + hi + 1) >> 1;
    if (T.job[mid].block0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const PackJob& J = T.job[lo];
  int b = blockIdx.x - J.block0;
  const int i1 = b % J.n1;
  b /= J.n1;
  const int c0 = (b % J.tiles2) * 32, a0 = (b / J.tiles2) * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* src = J.src + J.off + (long long)i1 * J.s1;
  D* dst = reinterpret_cast<D*>(J.dst);
  if (J.s0 == 1 && J.s2 != 1) {       // source contiguous along i0: transpose the tile
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i2 = c0 + ty + 8 * r, i0 = a0 + tx;
      tile[ty + 8 * r][tx] = (i0 < J.n0 && i2 < J.n2) ? src[i0 + (long long)i2 * J.s2] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i0 = a0 + ty + 8 * r, i2 = c0 + tx;
      if (i0 < J.n0 && i2 < J.n2) Elem<D>::st(dst + ((long long)i0 * J.n1 + i1) * J.n2 + i2, tile[tx][ty + 8 * r]);
    }
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i0 = a0 + ty + 8 * r, i2 = c0 + tx;
      if (i0 < J.n0 && i2 < J.n2)
        Elem<D>::st(dst + ((long long)i0 * J.n1 + i1) * J.n2 + i2, src[(long long)i0 * J.s0 + (long long)i2 * J.s2]);
    }
  }
}

static bool simt_vec_ok(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y) {
  const size_t esz = d->dtype == UNETB200_BF16 ? 2 : 4;
  const int Cq = d->N / d->nquad;
  return d->Cin % 16 == 0 && Cq % 4 == 0 && d->ld_in % 8 == 0 && d->ld_out % 4 == 0 &&
         (reinterpret_cast<uintptr_t>(x) % (8 * esz)) == 0 && (!wp || (reinterpret_cast<uintptr_t>(wp) % 16) == 0) &&
         (reinterpret_cast<uintptr_t>(y) % (4 * esz)) == 0;
}

static int simt_fbn(int N) { return N <= 16 ? 16 : (N <= 32 ? 32 : 64); }
static int simt_fbm(int N) { return 8 * 256 / (simt_fbn(N) / 4); }
static int simt_wbk(int N) { return 4 * 256 / (simt_fbn(N) / 4); }

long long simt_fprop_tiles(const GconvDev& g) { return (g.M + FBM - 1) / FBM; }

int simt_wgrad_splits(const GconvDev& g) {
  const int wbn = simt_fbn(g.N), wbk = simt_wbk(g.N);
  long long tiles = (long long)((g.K + wbk - 1) / wbk) * ((g.N + wbn - 1) / wbn);
  long long want = ((long long)sm_count() * 6 + tiles - 1) / tiles;
  long long max_by_m = (g.M + 255) / 256;
  if (want > max_by_m) want = max_by_m;
  if (want > 1024) want = 1024;
  if (want < 1) want = 1;
  return (int)want;
}

int simt_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, const float* bias, void* y,
               double* stats, float* stats_ws, cudaStream_t s) {
  const int fbn = simt_fbn(g.N), fbm = simt_fbm(g.N);
  dim3 grid((unsigned)((g.M + fbm - 1) / fbm), (unsigned)((g.N + fbn - 1) / fbn));
  const bool vec = simt_vec_ok(d, x, wp, y) && (g.K % 4 == 0);
  with_elem(d->dtype, [&](auto t) {
    with_bool(vec, [&](auto V) {
      with_int<16, 32, 64>(fbn, [&](auto BN) {
        using T = decltype(t);
        gconv_fprop_simt_kernel<T, V, BN><<<grid, 256, 0, s>>>(g, (const T*)x, (const T*)wp, bias, (T*)y, stats_ws);
      });
    });
  });
  UB_LAUNCH_CHECK("gconv_fprop_simt");
  if (stats) return launch_stats_reduce(stats_ws, (g.M + fbm - 1) / fbm, 2 * g.N, stats, s);
  return 0;
}

int simt_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
               cudaStream_t s) {
  long long mper = (g.M + splits - 1) / splits;
  mper = (mper + WBM - 1) / WBM * WBM;
  const int wbn = simt_fbn(g.N), wbk = simt_wbk(g.N);
  dim3 grid((unsigned)((g.K + wbk - 1) / wbk), (unsigned)((g.N + wbn - 1) / wbn), (unsigned)splits);
  const size_t esz = d->dtype == UNETB200_BF16 ? 2 : 4;
  const bool vec = d->Cin % 4 == 0 && g.Cq % 4 == 0 && d->ld_in % 4 == 0 && d->ld_out % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(x) % (4 * esz)) == 0 &&
                   (reinterpret_cast<uintptr_t>(gy) % (4 * esz)) == 0;
  with_elem(d->dtype, [&](auto t) {
    with_bool(vec, [&](auto V) {
      with_int<16, 32, 64>(wbn, [&](auto BN) {
        using T = decltype(t);
        gconv_wgrad_simt_kernel<T, V, BN><<<grid, 256, 0, s>>>(g, (const T*)x, (const T*)gy, partials, mper);
      });
    });
  });
  UB_LAUNCH_CHECK("gconv_wgrad_simt");
  return 0;
}

}  // namespace ub

using namespace ub;

extern "C" {

int unetb200_wgrad_reduce(const float* partials, int splits, int ntaps, int Cin, int N, int Cq, float* dst,
                          int64_t st, int64_t sc, int64_t sq, int64_t sn, int accumulate, void* stream) {
  UB_CHECK_ARG(partials && dst && splits >= 1 && ntaps >= 1 && Cin >= 1 && N >= 1 && Cq >= 1 && N % Cq == 0,
               "wgrad_reduce: bad args");
  long long K = (long long)ntaps * Cin;
  long long total = K * N;
  if (Cq == N && sc == 1 && (ntaps == 1 || st == Cin) && sn != 1) {
    // the parameter is k-linear (channels_last Conv2d weight): coalesced transpose
    dim3 grid((unsigned)((K + 31) / 32), (unsigned)((N + 31) / 32));
    dim3 grid8((unsigned)((K + 7) / 8), (unsigned)((N + 31) / 32));
    if (splits >= 32) wgrad_reduce_t_kernel<32><<<grid8, 1024, 0, (cudaStream_t)stream>>>(partials, splits, K, N, dst, sn, accumulate);
    else if (splits >= 8) wgrad_reduce_t_kernel<8><<<grid8, 256, 0, (cudaStream_t)stream>>>(partials, splits, K, N, dst, sn, accumulate);
    else wgrad_reduce_t4_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(partials, splits, K, N, dst, sn, accumulate);
    UB_LAUNCH_CHECK("wgrad_reduce_t");
    return 0;
  }
  long long blocks = (total + 255) / 256;
  long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  wgrad_reduce_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(partials, splits, Cin, K, N, Cq, dst, st, sc,
                                                                          sq, sn, accumulate);
  UB_LAUNCH_CHECK("wgrad_reduce");
  return 0;
}

int unetb200_wgrad_reduce_multi(const unetb200_reduce_job_t* jobs, int njobs, void* stream) {
  UB_CHECK_ARG(jobs && njobs >= 1, "wgrad_reduce_multi: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  for (int first = 0; first < njobs; first += kMaxReduceJobs) {
    const int count = njobs - first < kMaxReduceJobs ? njobs - first : kMaxReduceJobs;
    ReduceTable T;
    long long blocks = 0;
    for (int i = 0; i < count; ++i) {
      const unetb200_reduce_job_t& j = jobs[first + i];
      UB_CHECK_ARG(j.partials && j.dst && j.splits >= 1 && j.ntaps >= 1 && j.Cin >= 1 && j.N >= 1 && j.Cq >= 1 &&
                       j.N % j.Cq == 0,
                   "wgrad_reduce_multi: job %d", first + i);
      ReduceJob& J = T.job[i];
      J.partials = j.partials; J.dst = j.dst; J.st = j.st; J.sc = j.sc; J.sq = j.sq; J.sn = j.sn;
      J.K = (long long)j.ntaps * j.Cin;
      J.splits = j.splits; J.Cin = j.Cin; J.N = j.N; J.Cq = j.Cq;
      J.tiles_n = (j.N + 31) / 32;
      J.block0 = (int)blocks;
      J.accumulate = j.accumulate;
      J.pad_ = j.splits >= 8 ? 1 : 0;
      blocks += (J.pad_ ? (J.K + 7) / 8 : (J.K + 31) / 32) * J.tiles_n;
      UB_CHECK_ARG(blocks < (1LL << 31), "wgrad_reduce_multi: too many tiles");
    }
    T.njobs = count;
    wgrad_reduce_multi_kernel<<<(unsigned)blocks, 256, 0, s>>>(T);
  }
  UB_LAUNCH_CHECK("wgrad_reduce_multi");
  return 0;
}

int unetb200_pack_weights(const float* src, void* dst, int dst_dtype, int64_t n0, int64_t n1, int64_t n2,
                          int64_t s0, int64_t s1, int64_t s2, int64_t off, void* stream) {
  UB_CHECK_ARG(dst_dtype == UNETB200_F32 || dst_dtype == UNETB200_BF16, "pack_weights: dtype");
  UB_CHECK_ARG(src && dst && n0 > 0 && n1 > 0 && n2 > 0, "pack_weights: bad args");
  long long total = n0 * n1 * n2;
  long long blocks = (total + 255) / 256;
  long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cudaStream_t s = (cudaStream_t)stream;
  if (s0 == 1 && s2 != 1 && n0 >= 32 && n2 >= 32 && n1 <= 65535) {
    // source contiguous along the OUTER destination index (e.g. the dgrad operand of a channels_last weight)
    dim3 grid((unsigned)((n0 + 31) / 32), (unsigned)((n2 + 31) / 32), (unsigned)n1);
    with_elem(dst_dtype, [&](auto t) {
      using D = decltype(t);
      pack_weights_t_kernel<D><<<grid, 256, 0, s>>>(src, (D*)dst, (int)n0, (int)n1, (int)n2, s1, s2, off);
    });
    UB_LAUNCH_CHECK("pack_weights_t");
    return 0;
  }
  with_elem(dst_dtype, [&](auto t) {
    using D = decltype(t);
    pack_weights_kernel<D><<<(unsigned)blocks, 256, 0, s>>>(src, (D*)dst, n0, n1, n2, s0, s1, s2, off);
  });
  UB_LAUNCH_CHECK("pack_weights");
  return 0;
}

int unetb200_pack_weights_multi(const unetb200_pack_job_t* jobs, int njobs, int dst_dtype, void* stream) {
  UB_CHECK_ARG(dst_dtype == UNETB200_F32 || dst_dtype == UNETB200_BF16, "pack_weights_multi: dtype");
  UB_CHECK_ARG(jobs && njobs >= 1, "pack_weights_multi: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  for (int first = 0; first < njobs; first += kMaxPackJobs) {
    const int count = njobs - first < kMaxPackJobs ? njobs - first : kMaxPackJobs;
    PackTable T;
    long long blocks = 0;
    for (int i = 0; i < count; ++i) {
      const unetb200_pack_job_t& j = jobs[first + i];
      UB_CHECK_ARG(j.src && j.dst && j.n0 > 0 && j.n1 > 0 && j.n2 > 0 && j.n0 < (1LL << 31) && j.n1 < (1LL << 31) &&
                       j.n2 < (1LL << 31),
                   "pack_weights_multi: job %d", first + i);
      PackJob& J = T.job[i];
      J.src = j.src; J.dst = j.dst; J.s0 = j.s0; J.s1 = j.s1; J.s2 = j.s2; J.off = j.off;
      J.n0 = (int)j.n0; J.n1 = (int)j.n1; J.n2 = (int)j.n2;
      J.tiles2 = (J.n2 + 31) / 32;
      J.block0 = (int)blocks;
      J.pad_ = 0;
      blocks += (long long)((J.n0 + 31) / 32) * J.tiles2 * J.n1;
      UB_CHECK_ARG(blocks < (1LL << 31), "pack_weights_multi: too many tiles");
    }
    T.njobs = count;
    with_elem(dst_dtype, [&](auto t) { pack_multi_kernel<decltype(t)><<<(unsigned)blocks, 256, 0, s>>>(T); });
  }
  UB_LAUNCH_CHECK("pack_weights_multi");
  return 0;
}
}
