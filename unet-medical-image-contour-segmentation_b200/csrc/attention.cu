// SpatialAttention gate of the reference's UNet_SA (unet_parts.py:39-60,91-92; unet_model.py:140-189):
//   gate = sigmoid(conv7x7([mean_c(x), max_c(x)]))  (2 -> 1 channels, padding 3, no bias),   out = x * gate
// All of it is memory-bound (one or two streams over the skip tensor plus per-pixel maps), so it runs on the CUDA
// cores: LPP = C/8 lanes cooperate on a pixel (16-byte loads, warp shuffles) like the OutConv kernels; the per-pixel
// maps (statistics, gate, their gradients) are fp32.  Rounding points follow the reference under autocast: the
// statistics, the conv output, the gate and the product are each rounded to the storage type.
//
// forward : sa_stats (mean, max over channels) -> sa_gate (7x7 conv + sigmoid on the 2-channel map) -> sa_apply
// backward: sa_bwd_dgate (dgate = sum_c g*x; da = dgate * gate * (1 - gate))
//           sa_bwd_dw    (dw[ch][ky][kx] = sum_p da[p] * stats[p + (ky-3, kx-3)][ch]; per-block partials, fixed order)
//           sa_bwd_dx    (dstats = conv7x7^T(da);  dx = g*gate + dstats_mean / C + [c == argmax_c x] * dstats_max,
//                         first maximum on ties like torch.max)
#include "common.cuh"

namespace ub {

constexpr int kSaK = 7, kSaR = 3, kSaTaps = 2 * kSaK * kSaK;      // 98 weights

__device__ __forceinline__ float sigmoidf_(float a) { return 1.f / (1.f + expf(-a)); }

// one pixel per LPP lanes; lane `sub` owns channels [8*sub, 8*sub + 8)
template <typename T>
__global__ void __launch_bounds__(256) sa_stats_kernel(const T* __restrict__ x, int64_t ld, float* __restrict__ stats,
                                                       int64_t npix, int C, int LPP) {
  const int sub = threadIdx.x % LPP, ppb = blockDim.x / LPP;
  const float inv_c = 1.f / (float)C;
  for (int64_t base = (int64_t)blockIdx.x * ppb; base < npix; base += (int64_t)gridDim.x * ppb) {
    const int64_t p = base + threadIdx.x / LPP;
    float s = 0.f, m = -INFINITY;
    if (p < npix) {
      float v[8];
      load8(x + p * ld + sub * 8, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) { s += v[i]; m = fmaxf(m, v[i]); }
    }
    for (int o = LPP >> 1; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    if (sub == 0 && p < npix) {
      stats[2 * p] = Elem<T>::round(s * inv_c);
      stats[2 * p + 1] = m;                       // a maximum of stored values needs no rounding
    }
  }
}

template <typename T>
__global__ void sa_stats_scalar_kernel(const T* __restrict__ x, int64_t ld, float* __restrict__ stats, int64_t npix,
                                       int C) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f, m = -INFINITY;
    for (int c = 0; c < C; ++c) {
      const float v = Elem<T>::ld(x + p * ld + c);
      s += v;
      m = fmaxf(m, v);
    }
    stats[2 * p] = Elem<T>::round(s / (float)C);
    stats[2 * p + 1] = m;
  }
}

// gate[p] = sigmoid(sum_{ch,ky,kx} w[ch][ky][kx] * stats[p + (ky-3, kx-3)][ch]), zero padding.
// Tiled: a block owns an 8 x 32 pixel tile, the
// (8 + 6) x (32 + 6) x 2 halo of the statistics map sits in shared memory (zeros outside the image add nothing), a
// thread owns one pixel.  (First version: one thread per pixel with 49 bounds-checked 8-byte global loads -- 0.23 ms per
// full-resolution gate where the map is 34 MB; the transposed stencil of the backward pass likewise, 0.42 -> 0.2 ms.)
constexpr int kSgTH = 8, kSgTW = 32;
template <typename T>
__global__ void __launch_bounds__(256) sa_gate_tiled_kernel(const float* __restrict__ stats, const float* __restrict__ w,
                                                            float* __restrict__ gate, int B, int H, int W, int tiles_h,
                                                            int tiles_w) {
  __shared__ float sw[kSaTaps];
  __shared__ float sst[2][kSgTH + 2 * kSaR][kSgTW + 2 * kSaR + 1];
  for (int i = threadIdx.x; i < kSaTaps; i += blockDim.x) sw[i] = Elem<T>::round(w[i]);
  int rest = blockIdx.x;
  const int tj = rest % tiles_w;
  rest /= tiles_w;
  const int ti = rest % tiles_h;
  const int b = rest / tiles_h;
  const int i0 = ti * kSgTH, j0 = tj * kSgTW;
  const float* stb = stats + 2LL * b * H * W;
  constexpr int HH = kSgTH + 2 * kSaR, HW = kSgTW + 2 * kSaR;
  for (int e = threadIdx.x; e < HH * HW; e += blockDim.x) {
    const int i = e / HW, j = e - i * HW;
    const int yy = i0 + i - kSaR, xx = j0 + j - kSaR;
    float2 v = make_float2(0.f, 0.f);
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = *reinterpret_cast<const float2*>(stb + 2 * ((long long)yy * W + xx));
    sst[0][i][j] = v.x;
    sst[1][i][j] = v.y;
  }
  __syncthreads();
  const int ty = threadIdx.x / kSgTW, tx = threadIdx.x % kSgTW;
  const int yy = i0 + ty, xx = j0 + tx;
  if (yy >= H || xx >= W) return;
  float a = 0.f;
#pragma unroll
  for (int ky = 0; ky < kSaK; ++ky)
#pragma unroll
    for (int kx = 0; kx < kSaK; ++kx) {
      a = fmaf(sw[ky * kSaK + kx], sst[0][ty + ky][tx + kx], a);
      a = fmaf(sw[kSaK * kSaK + ky * kSaK + kx], sst[1][ty + ky][tx + kx], a);
    }
  gate[(long long)b * H * W + (long long)yy * W + xx] = Elem<T>::round(sigmoidf_(Elem<T>::round(a)));
}

// (dmean, dmax)[q] = sum_{ky,kx} w[ch][ky][kx] * da[q - (ky-3, kx-3)]: the transposed 7x7 conv of the backward pass as a
// tiled stencil (da halo in shared memory), written as a float2 map that sa_bwd_dx streams.
template <typename T>
__global__ void __launch_bounds__(256) sa_bwd_dstats_kernel(const float* __restrict__ da, const float* __restrict__ w,
                                                            float* __restrict__ dstats, int B, int H, int W, int tiles_h,
                                                            int tiles_w) {
  __shared__ float sw[kSaTaps];
  __shared__ float sda[kSgTH + 2 * kSaR][kSgTW + 2 * kSaR + 1];
  for (int i = threadIdx.x; i < kSaTaps; i += blockDim.x) sw[i] = Elem<T>::round(w[i]);
  int rest = blockIdx.x;
  const int tj = rest % tiles_w;
  rest /= tiles_w;
  const int ti = rest % tiles_h;
  const int b = rest / tiles_h;
  const int i0 = ti * kSgTH, j0 = tj * kSgTW;
  const float* dab = da + (long long)b * H * W;
  constexpr int HH = kSgTH + 2 * kSaR, HW = kSgTW + 2 * kSaR;
  for (int e = threadIdx.x; e < HH * HW; e += blockDim.x) {
    const int i = e / HW, j = e - i * HW;
    const int yy = i0 + i - kSaR, xx = j0 + j - kSaR;
    sda[i][j] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? dab[(long long)yy * W + xx] : 0.f;
  }
  __syncthreads();
  const int ty = threadIdx.x / kSgTW, tx = threadIdx.x % kSgTW;
  const int yy = i0 + ty, xx = j0 + tx;
  if (yy >= H || xx >= W) return;
  float dmean = 0.f, dmax = 0.f;
#pragma unroll
  for (int ky = 0; ky < kSaK; ++ky)
#pragma unroll
    for (int kx = 0; kx < kSaK; ++kx) {
      const float d = sda[ty + 2 * kSaR - ky][tx + 2 * kSaR - kx];
      dmean = fmaf(sw[ky * kSaK + kx], d, dmean);
      dmax = fmaf(sw[kSaK * kSaK + ky * kSaK + kx], d, dmax);
    }
  *reinterpret_cast<float2*>(dstats + 2 * ((long long)b * H * W + (long long)yy * W + xx)) = make_float2(dmean, dmax);
}

// out[p][c] = x[p][c] * gate[p]
template <typename T, int V>
__global__ void __launch_bounds__(256) sa_apply_kernel(const T* __restrict__ x, int64_t ld_x, const float* __restrict__ gate,
                                                       T* __restrict__ out, int64_t ld_o, int64_t npix, int CV) {
  const int64_t total = npix * CV;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = idx / CV;
    const int c = (int)(idx - p * CV) * V;
    const float g = __ldg(gate + p);
    float v[V];
    if constexpr (V == 8) load8(x + p * ld_x + c, v);
    else v[0] = Elem<T>::ld(x + p * ld_x + c);
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] *= g;
    if constexpr (V == 8) store8(out + p * ld_o + c, v);
    else Elem<T>::st(out + p * ld_o + c, v[0]);
  }
}

// da[p] = (sum_c g[p][c] * x[p][c]) * gate * (1 - gate)
template <typename T>
__global__ void __launch_bounds__(256) sa_bwd_dgate_kernel(const T* __restrict__ g, int64_t ld_g, const T* __restrict__ x,
                                                           int64_t ld_x, const float* __restrict__ gate,
                                                           float* __restrict__ da, int64_t npix, int C, int LPP) {
  const int sub = threadIdx.x % LPP, ppb = blockDim.x / LPP;
  for (int64_t base = (int64_t)blockIdx.x * ppb; base < npix; base += (int64_t)gridDim.x * ppb) {
    const int64_t p = base + threadIdx.x / LPP;
    float s = 0.f;
    if (p < npix) {
      if (LPP * 8 == C) {
        float a[8], b[8];
        load8(g + p * ld_g + sub * 8, a);
        load8(x + p * ld_x + sub * 8, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) s = fmaf(a[i], b[i], s);
      } else {                                    // scalar layout: LPP == 1, any C
        for (int c = 0; c < C; ++c) s = fmaf(Elem<T>::ld(g + p * ld_g + c), Elem<T>::ld(x + p * ld_x + c), s);
      }
    }
    for (int o = LPP >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (sub == 0 && p < npix) {
      const float gt = gate[p];
      da[p] = s * gt * (1.f - gt);
    }
  }
}

// partial[block][98]: a block owns a 16 x 32 pixel tile of one image: the da tile and the (16 + 6) x (32 + 6) x 2 halo
// of the statistics map are staged in shared memory, thread t < 98 owns weight t = (ch, ky, kx) and walks the tile in
// a fixed order.  (First version: one thread per weight walking 4096 pixels of global memory with 64-bit index
// arithmetic -- 6.2 ms per UNet_SA step.)
constexpr int kSaTH = 16, kSaTW = 32;
__global__ void __launch_bounds__(128) sa_bwd_dw_kernel(const float* __restrict__ da, const float* __restrict__ stats,
                                                        float* __restrict__ partial, int B, int H, int W, int tiles_h,
                                                        int tiles_w) {
  __shared__ float sda[kSaTH][kSaTW];
  __shared__ float sst[2][kSaTH + 2 * kSaR][kSaTW + 2 * kSaR + 1];
  int rest = blockIdx.x;
  const int tj = rest % tiles_w;
  rest /= tiles_w;
  const int ti = rest % tiles_h;
  const int b = rest / tiles_h;
  const int i0 = ti * kSaTH, j0 = tj * kSaTW;
  const float* dab = da + (long long)b * H * W;
  const float* stb = stats + 2LL * b * H * W;
  for (int e = threadIdx.x; e < kSaTH * kSaTW; e += blockDim.x) {
    const int i = e / kSaTW, j = e - i * kSaTW;
    const int yy = i0 + i, xx = j0 + j;
    sda[i][j] = (yy < H && xx < W) ? dab[(long long)yy * W + xx] : 0.f;
  }
  constexpr int HH = kSaTH + 2 * kSaR, HW = kSaTW + 2 * kSaR;
  for (int e = threadIdx.x; e < HH * HW; e += blockDim.x) {
    const int i = e / HW, j = e - i * HW;
    const int yy = i0 + i - kSaR, xx = j0 + j - kSaR;
    float2 v = make_float2(0.f, 0.f);
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = *reinterpret_cast<const float2*>(stb + 2 * ((long long)yy * W + xx));
    sst[0][i][j] = v.x;
    sst[1][i][j] = v.y;
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= kSaTaps) return;
  const int ch = t / (kSaK * kSaK), ky = (t / kSaK) % kSaK, kx = t % kSaK;
  float acc = 0.f;
#pragma unroll 1
  for (int i = 0; i < kSaTH; ++i)
#pragma unroll 8
    for (int j = 0; j < kSaTW; ++j) acc = fmaf(sda[i][j], sst[ch][i + ky][j + kx], acc);
  partial[(long long)blockIdx.x * kSaTaps + t] = acc;
}

__global__ void sa_bwd_dw_reduce_kernel(const float* __restrict__ partial, int nblocks, float* __restrict__ dw) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (t >= kSaTaps) return;
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += (double)partial[(int64_t)b * kSaTaps + t];
  s = warp_sum(s);
  if (lane == 0) dw[t] = (float)s;
}

// dx[p][c] = g[p][c]*gate[p] + dmean[p]/C + [c == argmax_c x[p][:]] * dmax[p],
// (dmean, dmax)[q] = sum_{ky,kx} w[ch][ky][kx] * da[q - (ky-3, kx-3)]   (transposed 7x7 conv, zero outside)
template <typename T>
__global__ void __launch_bounds__(256) sa_bwd_dx_kernel(const T* __restrict__ g, int64_t ld_g, const T* __restrict__ x,
                                                        int64_t ld_x, const float* __restrict__ gate,
                                                        const float* __restrict__ dstats,
                                                        T* __restrict__ dx, int64_t ld_dx, int B, int H, int W, int C,
                                                        int LPP) {
  const int sub = threadIdx.x % LPP, ppb = blockDim.x / LPP;
  const int64_t npix = (int64_t)B * H * W;
  const float inv_c = 1.f / (float)C;
  for (int64_t base = (int64_t)blockIdx.x * ppb; base < npix; base += (int64_t)gridDim.x * ppb) {
    const int64_t p = base + threadIdx.x / LPP;
    const bool live = p < npix;
    // (dmean, dmax) of the pixel from the map sa_bwd_dstats_kernel made (every lane of the pixel reads the same 8 bytes)
    float dmean = 0.f, dmax = 0.f;
    if (live) {
      const float2 ds = *reinterpret_cast<const float2*>(dstats + 2 * p);
      dmean = ds.x;
      dmax = ds.y;
    }
    if (LPP * 8 == C) {
      float xv[8], gv[8];
      float m = -INFINITY;
      int arg = 0;
      if (live) {
        load8(x + p * ld_x + sub * 8, xv);
        load8(g + p * ld_g + sub * 8, gv);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (xv[k] > m) { m = xv[k]; arg = sub * 8 + k; }
      }
      for (int o = LPP >> 1; o > 0; o >>= 1) {               // first maximum: larger value, then smaller index
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
        const int a2 = __shfl_xor_sync(0xffffffffu, arg, o);
        if (m2 > m || (m2 == m && a2 < arg)) { m = m2; arg = a2; }
      }
      if (live) {
        const float gt = gate[p];
        float o8[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
          o8[k] = fmaf(gv[k], gt, dmean * inv_c) + ((sub * 8 + k == arg) ? dmax : 0.f);
        store8(dx + p * ld_dx + sub * 8, o8);
      }
    } else if (live) {                                        // scalar layout (LPP == 1)
      float m = -INFINITY;
      int arg = 0;
      for (int c = 0; c < C; ++c) {
        const float v = Elem<T>::ld(x + p * ld_x + c);
        if (v > m) { m = v; arg = c; }
      }
      const float gt = gate[p];
      for (int c = 0; c < C; ++c)
        Elem<T>::st(dx + p * ld_dx + c, fmaf(Elem<T>::ld(g + p * ld_g + c), gt, dmean * inv_c) + (c == arg ? dmax : 0.f));
    }
  }
}

static bool sa_vec(int C, std::initializer_list<int64_t> lds, std::initializer_list<const void*> ptrs, size_t esz) {
  const int l = C / 8;
  if (C % 8 || l < 1 || l > 32 || (l & (l - 1))) return false;
  for (int64_t ld : lds)
    if (ld % 8) return false;
  for (const void* p : ptrs)
    if (reinterpret_cast<uintptr_t>(p) % (8 * esz)) return false;
  return true;
}
static int sa_blocks(int64_t work_items, int per_block) {
  int64_t b = (work_items + per_block - 1) / per_block;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace ub

using namespace ub;

extern "C" {

int unetb200_sa_forward(const void* x, int64_t ld_x, const float* w, float* stats, float* gate, void* out, int64_t ld_out,
                        int dtype, int B, int H, int W, int C, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "sa_forward: dtype");
  UB_CHECK_ARG(x && w && stats && gate && out && B > 0 && H > 0 && W > 0 && C > 0 && ld_x >= C && ld_out >= C,
               "sa_forward: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t npix = (int64_t)B * H * W;
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  const bool vec = sa_vec(C, {ld_x, ld_out}, {x, out}, esz);
  const int LPP = vec ? C / 8 : 1;
  const int gth = (H + kSgTH - 1) / kSgTH, gtw = (W + kSgTW - 1) / kSgTW;
  const int64_t gblocks = (int64_t)B * gth * gtw;
  UB_CHECK_ARG(gblocks < (1LL << 31), "sa_forward: too many tiles");
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    if (vec) sa_stats_kernel<T><<<sa_blocks(npix, 256 / LPP), 256, 0, s>>>((const T*)x, ld_x, stats, npix, C, LPP);
    else sa_stats_scalar_kernel<T><<<sa_blocks(npix, 256), 256, 0, s>>>((const T*)x, ld_x, stats, npix, C);
    sa_gate_tiled_kernel<T><<<(unsigned)gblocks, 256, 0, s>>>(stats, w, gate, B, H, W, gth, gtw);
    with_vec<8>(vec, [&](auto V) {
      sa_apply_kernel<T, V><<<sa_blocks(npix * (C / V), 256), 256, 0, s>>>((const T*)x, ld_x, gate, (T*)out, ld_out,
                                                                           npix, C / V);
    });
  });
  UB_LAUNCH_CHECK("sa_forward");
  return 0;
}

int64_t unetb200_sa_backward_workspace(int B, int H, int W) {
  const int64_t npix = (int64_t)B * H * W;
  const int64_t blocks = (int64_t)B * ((H + kSaTH - 1) / kSaTH) * ((W + kSaTW - 1) / kSaTW);
  return 3 * npix + blocks * kSaTaps + 64;       // floats: (dmean, dmax) map + da map + dw partials
}

int unetb200_sa_backward(const void* g, int64_t ld_g, const void* x, int64_t ld_x, const float* w, const float* stats,
                         const float* gate, void* dx, int64_t ld_dx, float* dw, float* workspace, int dtype, int B, int H,
                         int W, int C, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "sa_backward: dtype");
  UB_CHECK_ARG(g && x && w && stats && gate && dx && dw && workspace && B > 0 && H > 0 && W > 0 && C > 0 && ld_g >= C &&
                   ld_x >= C && ld_dx >= C,
               "sa_backward: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t npix = (int64_t)B * H * W;
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  const bool vec = sa_vec(C, {ld_g, ld_x, ld_dx}, {g, x, dx}, esz);
  const int LPP = vec ? C / 8 : 1;
  float* dstats = workspace;                     // float2 per pixel (first: 8-byte aligned for any npix)
  float* da = workspace + 2 * npix;
  float* partial = workspace + 3 * npix;
  const int gth = (H + kSgTH - 1) / kSgTH, gtw = (W + kSgTW - 1) / kSgTW;
  const int64_t gblocks = (int64_t)B * gth * gtw;
  UB_CHECK_ARG(gblocks < (1LL << 31), "sa_backward: too many tiles");
  const int tiles_h = (H + kSaTH - 1) / kSaTH, tiles_w = (W + kSaTW - 1) / kSaTW;
  const int64_t blocks = (int64_t)B * tiles_h * tiles_w;
  UB_CHECK_ARG(blocks < (1LL << 31), "sa_backward: too many tiles");
  with_elem(dtype, [&](auto t) {
    using T = decltype(t);
    sa_bwd_dgate_kernel<T><<<sa_blocks(npix, 256 / LPP), 256, 0, s>>>((const T*)g, ld_g, (const T*)x, ld_x, gate, da,
                                                                      npix, C, LPP);
    sa_bwd_dw_kernel<<<(unsigned)blocks, 128, 0, s>>>(da, stats, partial, B, H, W, tiles_h, tiles_w);
    sa_bwd_dw_reduce_kernel<<<(kSaTaps + 7) / 8, 256, 0, s>>>(partial, (int)blocks, dw);
    sa_bwd_dstats_kernel<T><<<(unsigned)gblocks, 256, 0, s>>>(da, w, dstats, B, H, W, gth, gtw);
    sa_bwd_dx_kernel<T><<<sa_blocks(npix, 256 / LPP), 256, 0, s>>>((const T*)g, ld_g, (const T*)x, ld_x, gate, dstats,
                                                                   (T*)dx, ld_dx, B, H, W, C, LPP);
  });
  UB_LAUNCH_CHECK("sa_backward");
  return 0;
}
}
