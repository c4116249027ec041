// Loss kernels: fused softmax + cross-entropy + dice (train.py:137-142, dice_score.py:5-36), fused
// BCE-with-logits + sigmoid dice (train.py:118-134), generic dice_coeff, and the integer-count boundary loss
// (boundary_loss.py:5-118).
// All memory-bound single-pass reductions: warp shuffles -> shared memory -> fp64 / int64 atomics, or (BCE + dice)
// per-block fp64 partials summed in a fixed order.
#include "common.cuh"

namespace ub {

constexpr int kMaxClasses = 8;

__device__ __forceinline__ double block_sum(double v, double* smem) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) smem[w] = v;
  __syncthreads();
  double r = 0;
  if (w == 0) {
    r = l < (int)(blockDim.x >> 5) ? smem[l] : 0.0;
    r = warp_sum(r);
  }
  return r;  // valid in warp 0
}

// ------------------------------------------------------------------------------------------
// fused softmax / CE / dice
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void ce_dice_fwd_kernel(const T* __restrict__ logits, const int64_t* __restrict__ target, int64_t npix,
                                   int C, double* __restrict__ acc) {
  __shared__ double sm[32];
  float ce = 0.f, inter = 0.f, psum = 0.f, valid = 0.f;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
    float z[kMaxClasses];
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { z[c] = Elem<T>::ld(logits + p * C + c); mx = fmaxf(mx, z[c]); }
    const int64_t t = target[p];
    float den = 0.f, zt = 0.f;                          // zt = z_t - max: the exact log-sum-exp form of the cross entropy
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { if (c == t) zt = z[c] - mx; z[c] = expf(z[c] - mx); den += z[c]; }
    const float inv = 1.f / den;
    float pt = 0.f, ps = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { float pc = z[c] * inv; ps += pc; if (c == t) pt = pc; }
    if (t >= 0 && t < C) {
      ce += logf(den) - zt;                             // (-log(max(p_t, 1e-38)) saturated near 87.5 for huge margins)
      inter += pt;
      valid += 1.f;
    }
    psum += ps;
  }
  double r0 = block_sum((double)ce, sm), r1 = block_sum((double)inter, sm), r2 = block_sum((double)psum, sm),
         r3 = block_sum((double)valid, sm);
  if (threadIdx.x == 0) {
    atomicAdd(acc + 0, r0);
    atomicAdd(acc + 1, r1);
    atomicAdd(acc + 2, r2);
    atomicAdd(acc + 3, r3);
  }
}

__global__ void ce_dice_finalize_kernel(const double* __restrict__ acc, int64_t npix, float eps, float* out,
                                        float* coefs) {
  if (threadIdx.x || blockIdx.x) return;
  double valid = acc[3];
  float ce = (float)(acc[0] / (double)npix);
  float inter = 2.f * (float)acc[1];
  float sets = (float)acc[2] + (float)valid;
  if (sets == 0.f) sets = inter;
  float dice = (inter + eps) / (sets + eps);
  float dl = 1.f - dice;
  if (valid != (double)npix) { ce = NAN; }       // a class index outside [0, C): the reference's one_hot raises
  out[0] = ce + dl;
  out[1] = ce;
  out[2] = dl;
  out[3] = dice;
  coefs[0] = 1.f / (float)npix;
  coefs[1] = 2.f / (sets + eps);
  coefs[2] = (inter + eps) / ((sets + eps) * (sets + eps));
  coefs[3] = 0.f;
}

// d(ce + 1 - dice)/dz_c = (p_c - [c==t])/npix  +  p_c * (h_c - sum_k p_k h_k),  h_k = -(a [k==t] - b)
template <typename T>
__global__ void ce_dice_bwd_kernel(const T* __restrict__ logits, const int64_t* __restrict__ target, int64_t npix,
                                   int C, const float* __restrict__ coefs, const float* __restrict__ gscale,
                                   T* __restrict__ glogits) {
  const float invn = coefs[0], a = coefs[1], b = coefs[2];
  const float gs = gscale ? gscale[0] : 1.f;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
    float z[kMaxClasses];
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { z[c] = Elem<T>::ld(logits + p * C + c); mx = fmaxf(mx, z[c]); }
    float den = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { z[c] = expf(z[c] - mx); den += z[c]; }
    const float inv = 1.f / den;
    const int64_t t = target[p];
    float dot = 0.f;   // sum_k p_k h_k
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) { z[c] *= inv; dot += z[c] * (b - (c == t ? a : 0.f)); }
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c)
      if (c < C) {
        float h = b - (c == t ? a : 0.f);
        float g = (z[c] - (c == t ? 1.f : 0.f)) * invn + z[c] * (h - dot);
        Elem<T>::st(glogits + p * C + c, gs * g);
      }
  }
}

// ------------------------------------------------------------------------------------------
// fused BCE-with-logits / sigmoid / dice of the binary branch (train.py:118-134)
// ------------------------------------------------------------------------------------------
// 8 consecutive target values widened to fp32 (16-byte loads; 8 bytes for uint8)
__device__ __forceinline__ void load8t(const float* p, float v[8]) { load8(p, v); }
__device__ __forceinline__ void load8t(const long long* p, float v[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    longlong2 r = reinterpret_cast<const longlong2*>(p)[i];
    v[2 * i] = (float)r.x;
    v[2 * i + 1] = (float)r.y;
  }
}
__device__ __forceinline__ void load8t(const uint8_t* p, float v[8]) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i] = (float)((r.x >> (8 * i)) & 0xffu);
    v[4 + i] = (float)((r.y >> (8 * i)) & 0xffu);
  }
}

struct BceDiceSums {
  float bce = 0.f, st = 0.f, s = 0.f, t = 0.f;
  // BCE on the unrounded logit (binary_cross_entropy_with_logits is on autocast's fp32 list), dice on the
  // sigmoid rounded to the logits' storage type (F.sigmoid of bf16 logits returns bf16)
  template <typename T>
  __device__ __forceinline__ void add(float x, float tv) {
    bce += fmaxf(x, 0.f) - x * tv + log1pf(expf(-fabsf(x)));
    const float sr = Elem<T>::round(1.f / (1.f + expf(-x)));
    st += sr * tv;
    s += sr;
    t += tv;
  }
};

// vec: the vector path over npix / 8 groups of 8 pixels (every pointer aligned for it); the pixels after the last
// full group -- all of them when !vec -- are a grid-stride scalar loop.  Each block writes its four sums to
// partials[k * gridDim.x + blockIdx.x]: no atomics, so the finalize's fixed-order sum is reproducible.
template <typename T, typename TT>
__global__ void __launch_bounds__(256) bce_dice_fwd_kernel(const T* __restrict__ logits, const TT* __restrict__ target,
                                                           int64_t npix, bool vec, double* __restrict__ partials) {
  __shared__ double sm[32];
  BceDiceSums acc;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  const int64_t nvec = vec ? npix >> 3 : 0;
  for (int64_t v = tid; v < nvec; v += nthr) {
    float x[8], t[8];
    load8(logits + 8 * v, x);
    load8t(target + 8 * v, t);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc.add<T>(x[i], t[i]);
  }
  for (int64_t p = 8 * nvec + tid; p < npix; p += nthr) acc.add<T>(Elem<T>::ld(logits + p), (float)target[p]);
  const double r0 = block_sum((double)acc.bce, sm), r1 = block_sum((double)acc.st, sm),
               r2 = block_sum((double)acc.s, sm), r3 = block_sum((double)acc.t, sm);
  if (threadIdx.x == 0) {
    partials[0 * gridDim.x + blockIdx.x] = r0;
    partials[1 * gridDim.x + blockIdx.x] = r1;
    partials[2 * gridDim.x + blockIdx.x] = r2;
    partials[3 * gridDim.x + blockIdx.x] = r3;
  }
}

// one block: the nblk partials of each sum in a fixed order, then dice_coeff(reduce_batch_first=True) on the
// 3-D input (dice_score.py:12-18: one global ratio, sets == 0 -> inter)
__global__ void bce_dice_finalize_kernel(const double* __restrict__ partials, int nblk, int64_t npix, float eps,
                                         float* __restrict__ out, float* __restrict__ coefs) {
  __shared__ double sm[32];
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  for (int b = threadIdx.x; b < nblk; b += blockDim.x)
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] += partials[k * nblk + b];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = block_sum(v[k], sm);
  if (threadIdx.x) return;
  const float bce = (float)(v[0] / (double)npix);
  const float inter = 2.f * (float)v[1];
  float sets = (float)v[2] + (float)v[3];
  const bool empty = (sets == 0.f);
  if (empty) sets = inter;
  const float dice = (inter + eps) / (sets + eps);
  const float dl = 1.f - dice;
  out[0] = bce + dl;
  out[1] = bce;
  out[2] = dl;
  out[3] = dice;
  coefs[0] = 1.f / (float)npix;
  // d(1 - dice)/ds = -(a t - b); an empty set makes the ratio (inter+eps)/(inter+eps), a constant
  coefs[1] = empty ? 0.f : 2.f / (sets + eps);
  coefs[2] = empty ? 0.f : (inter + eps) / ((sets + eps) * (sets + eps));
  coefs[3] = 0.f;
}

// d(bce + 1 - dice)/dx = (sigma(x) - t)/npix - (a t - b) s (1 - s),  s = sigma(x) rounded to T
template <typename T>
__device__ __forceinline__ float bce_dice_grad(float x, float tv, float invn, float a, float b, float gs) {
  const float sig = 1.f / (1.f + expf(-x));
  const float sr = Elem<T>::round(sig);
  return gs * ((sig - tv) * invn - (a * tv - b) * sr * (1.f - sr));
}

template <typename T, typename TT>
__global__ void __launch_bounds__(256) bce_dice_bwd_kernel(const T* __restrict__ logits, const TT* __restrict__ target,
                                                           int64_t npix, bool vec, const float* __restrict__ coefs,
                                                           const float* __restrict__ gscale, T* __restrict__ glogits) {
  const float invn = coefs[0], a = coefs[1], b = coefs[2];
  const float gs = gscale ? gscale[0] : 1.f;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  const int64_t nvec = vec ? npix >> 3 : 0;
  for (int64_t v = tid; v < nvec; v += nthr) {
    float x[8], t[8];
    load8(logits + 8 * v, x);
    load8t(target + 8 * v, t);
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = bce_dice_grad<T>(x[i], t[i], invn, a, b, gs);
    store8(glogits + 8 * v, x);
  }
  for (int64_t p = 8 * nvec + tid; p < npix; p += nthr)
    Elem<T>::st(glogits + p, bce_dice_grad<T>(Elem<T>::ld(logits + p), (float)target[p], invn, a, b, gs));
}

// ------------------------------------------------------------------------------------------
// generic dice on fp32 [G][L]
// ------------------------------------------------------------------------------------------
__global__ void dice_fwd_kernel(const float* __restrict__ x, const float* __restrict__ t, int64_t L,
                                double* __restrict__ acc) {
  __shared__ double sm[32];
  const int64_t g = blockIdx.y;
  const float* xg = x + g * L;
  const float* tg = t + g * L;
  float a = 0.f, b = 0.f, c = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < L; i += (int64_t)gridDim.x * blockDim.x) {
    float xv = xg[i], tv = tg[i];
    a += xv * tv;
    b += xv;
    c += tv;
  }
  double r0 = block_sum((double)a, sm), r1 = block_sum((double)b, sm), r2 = block_sum((double)c, sm);
  if (threadIdx.x == 0) {
    atomicAdd(acc + 3 * g + 0, r0);
    atomicAdd(acc + 3 * g + 1, r1);
    atomicAdd(acc + 3 * g + 2, r2);
  }
}

__global__ void dice_finalize_kernel(const double* __restrict__ acc, int64_t G, float eps, float* out, float* saved) {
  __shared__ double sm[32];
  double s = 0;
  for (int64_t g = threadIdx.x; g < G; g += blockDim.x) {
    float inter = 2.f * (float)acc[3 * g];
    float sets = (float)acc[3 * g + 1] + (float)acc[3 * g + 2];
    bool empty = (sets == 0.f);
    if (empty) sets = inter;
    float d = (inter + eps) / (sets + eps);
    s += d;
    // d(dice_g)/dx_i = A t_i - B   (zero for an empty group: (i+eps)/(i+eps) is constant)
    saved[2 * g] = empty ? 0.f : 2.f / (sets + eps);
    saved[2 * g + 1] = empty ? 0.f : (inter + eps) / ((sets + eps) * (sets + eps));
  }
  double r = block_sum(s, sm);
  if (threadIdx.x == 0) out[0] = (float)(r / (double)G);
}

__global__ void dice_bwd_kernel(const float* __restrict__ t, int64_t G, int64_t L, const float* __restrict__ saved,
                                const float* __restrict__ gscale, float* __restrict__ gx) {
  const int64_t g = blockIdx.y;
  const float gs = (gscale ? gscale[0] : 1.f) / (float)G;
  const float A = saved[2 * g] * gs, Bc = saved[2 * g + 1] * gs;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < L; i += (int64_t)gridDim.x * blockDim.x)
    gx[g * L + i] = A * t[g * L + i] - Bc;
}

// ------------------------------------------------------------------------------------------
// boundary loss
// ------------------------------------------------------------------------------------------
// work layout: unsigned long long cnt[12] = [variant(raw,sigmoid)][region(inner,edge)][P,T,I];
//              then 4 spare; then uint32 enc_min, enc_max (order-preserving float encodings).
struct BoundaryGeom {
  int B, H, W, ewh, eww, has_edge;
};
__device__ __forceinline__ bool is_edge(const BoundaryGeom& g, int h, int w) {
  return g.has_edge && (h < g.ewh || h >= g.H - g.ewh || w < g.eww || w >= g.W - g.eww);
}
__device__ __forceinline__ uint32_t enc_float(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_float(uint32_t e) {
  uint32_t u = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
  return __uint_as_float(u);
}

template <typename P, typename TT>
struct BoundaryIO {
  const P* pred;
  int64_t sb, sh, sw;
  const TT* tgt;
  int64_t tb, th, tw;
  // bits: 1 = raw > 0.5, 2 = sigmoid > 0.5 (rounded to the pred dtype like torch.sigmoid), 4 = target == 255
  __device__ __forceinline__ int bits(int b, int h, int w, float* val) const {
    float v = Elem<P>::ld(pred + b * sb + h * sh + w * sw);
    if (val) *val = v;
    float s = Elem<P>::round(1.f / (1.f + expf(-v)));
    TT tv = tgt[b * tb + h * th + w * tw];
    return (v > 0.5f ? 1 : 0) | (s > 0.5f ? 2 : 0) | (tv == (TT)255 ? 4 : 0);
  }
};

template <typename P, typename TT>
__global__ void boundary_counts_kernel(BoundaryIO<P, TT> io, BoundaryGeom g, unsigned long long* __restrict__ cnt,
                                       uint32_t* __restrict__ mm) {
  __shared__ unsigned int sc[12];
  __shared__ uint32_t smin, smax;
  if (threadIdx.x < 12) sc[threadIdx.x] = 0;
  if (threadIdx.x == 0) { smin = 0xffffffffu; smax = 0u; }
  __syncthreads();
  unsigned int loc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) loc[i] = 0;
  uint32_t lmin = 0xffffffffu, lmax = 0u;
  const int64_t total = (int64_t)g.B * g.H * g.W;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int w = (int)(idx % g.W);
    int64_t r = idx / g.W;
    int h = (int)(r % g.H);
    int b = (int)(r / g.H);
    float v;
    int self = io.bits(b, h, w, &v);
    uint32_t e = enc_float(v);
    lmin = min(lmin, e);
    lmax = max(lmax, e);
    const bool edge = is_edge(g, h, w);
    // next pixel of the same region in row-major order (boundary_loss.py:68-74 compaction)
    int nh = h, nw = w + 1;
    bool has_n = true;
    if (nw >= g.W) { nw = 0; nh = h + 1; }
    if (nh >= g.H) has_n = false;
    if (has_n && is_edge(g, nh, nw) != edge) {
      if (edge) { nw = g.W - g.eww; }                                    // skip the inner run of row nh
      else { nh = h + 1; nw = g.eww; has_n = (nh < g.H - g.ewh); }       // first inner pixel of the next row
    }
    int ph = h, pw = w - 1;
    bool has_p = true;
    if (pw < 0) { pw = g.W - 1; ph = h - 1; }
    if (ph < 0) has_p = false;
    if (has_p && is_edge(g, ph, pw) != edge) {
      if (edge) { pw = g.eww - 1; }
      else { ph = h - 1; pw = g.W - g.eww - 1; has_p = (ph >= g.ewh); }
    }
    int nb = has_n ? io.bits(b, nh, nw, nullptr) : 0;
    int pb = has_p ? io.bits(b, ph, pw, nullptr) : 0;
    int u = self | nb | pb;          // 3-tap OR over the compacted run (dilation; erosion never fires)
    int tb = (u >> 2) & 1;
    int reg = edge ? 1 : 0;
#pragma unroll
    for (int var = 0; var < 2; ++var) {
      int pbit = (u >> var) & 1;
      int base = (var * 2 + reg) * 3;
      loc[base + 0] += pbit;
      loc[base + 1] += tb;
      loc[base + 2] += pbit & tb;
    }
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    unsigned int v = loc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sc[i], v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lmin = min(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
    lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&smin, lmin); atomicMax(&smax, lmax); }
  __syncthreads();
  if (threadIdx.x < 12 && sc[threadIdx.x]) atomicAdd(cnt + threadIdx.x, (unsigned long long)sc[threadIdx.x]);
  if (threadIdx.x == 0) { atomicMin(mm, smin); atomicMax(mm + 1, smax); }
}

__device__ double region_loss(double n, double p, double t, double i, float smooth) {
  if (n <= 0) return 0.0;                                   // boundary_loss.py:64-65
  // fp32 values of BCEWithLogits(logit(clamp(pb,1e-6,1-1e-6)), tb) for (pb,tb) = 00,01,10,11
  const double c00 = 9.5367431640625e-07, c01 = 13.815510749816895, c10 = 13.802318572998047,
               c11 = 1.0132797569895047e-06;
  float inter = (float)i, uni = (float)p + (float)t - (float)i;
  float iou = (inter + smooth) / (uni + smooth);
  double bce = (c11 * i + c10 * (p - i) + c01 * (t - i) + c00 * (n - p - t + i)) / n;
  return (double)(1.f - iou) + 0.5 * bce;
}

__global__ void boundary_finalize_kernel(const unsigned long long* __restrict__ cnt, const uint32_t* __restrict__ mm,
                                         BoundaryGeom g, float edge_weight, float smooth, float* out) {
  if (threadIdx.x || blockIdx.x) return;
  float mn = dec_float(mm[0]), mx = dec_float(mm[1]);
  int var = (mn < -10.f || mx > 10.f) ? 1 : 0;              // boundary_loss.py:28-29
  double total = (double)g.H * g.W;
  double inner_h = g.has_edge ? (double)max(g.H - 2 * g.ewh, 0) : g.H;
  double inner_w = g.has_edge ? (double)max(g.W - 2 * g.eww, 0) : g.W;
  double n_inner = inner_h * inner_w * g.B, n_edge = total * g.B - n_inner;
  const unsigned long long* c = cnt + var * 6;
  double normal = region_loss(n_inner, (double)c[0], (double)c[1], (double)c[2], smooth);
  double edge = region_loss(n_edge, (double)c[3], (double)c[4], (double)c[5], smooth);
  out[0] = (float)((normal + (double)edge_weight * edge) / (1.0 + (double)edge_weight));
}

}  // namespace ub

using namespace ub;
typedef __nv_bfloat16 bf16;

static inline int loss_grid(int64_t work, int threads) {
  int64_t b = (work + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

extern "C" {

int unetb200_ce_dice_fwd(const void* logits, int dtype, const int64_t* target, int64_t npix, int C, float epsilon,
                         double* acc, float* out, float* coefs, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "ce_dice_fwd: dtype");
  UB_CHECK_ARG(npix > 0 && C >= 1 && C <= kMaxClasses, "ce_dice_fwd: npix=%lld C=%d (C <= %d)", (long long)npix, C,
               kMaxClasses);
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(acc, 0, 4 * sizeof(double), s);
  if (e != cudaSuccess) return cuda_fail(e, "ce_dice_fwd memset");
  int g = loss_grid(npix, 256);
  if (dtype == UNETB200_BF16)
    ce_dice_fwd_kernel<bf16><<<g, 256, 0, s>>>((const bf16*)logits, target, npix, C, acc);
  else
    ce_dice_fwd_kernel<float><<<g, 256, 0, s>>>((const float*)logits, target, npix, C, acc);
  ce_dice_finalize_kernel<<<1, 32, 0, s>>>(acc, npix, epsilon, out, coefs);
  UB_LAUNCH_CHECK("ce_dice_fwd");
  return 0;
}

int unetb200_ce_dice_bwd(const void* logits, int dtype, const int64_t* target, int64_t npix, int C,
                         const float* coefs, const float* gscale, void* glogits, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "ce_dice_bwd: dtype");
  UB_CHECK_ARG(npix > 0 && C >= 1 && C <= kMaxClasses, "ce_dice_bwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  int g = loss_grid(npix, 256);
  if (dtype == UNETB200_BF16)
    ce_dice_bwd_kernel<bf16><<<g, 256, 0, s>>>((const bf16*)logits, target, npix, C, coefs, gscale, (bf16*)glogits);
  else
    ce_dice_bwd_kernel<float><<<g, 256, 0, s>>>((const float*)logits, target, npix, C, coefs, gscale,
                                                (float*)glogits);
  UB_LAUNCH_CHECK("ce_dice_bwd");
  return 0;
}

static inline int bce_dice_grid(int64_t npix) { return loss_grid((npix + 7) / 8, 256); }

static inline bool bce_dice_vec(const void* logits, const void* target, int tgt_dtype, const void* glogits) {
  const uintptr_t talign = tgt_dtype == UNETB200_U8 ? 8 : 16;
  return aligned16(logits) && (reinterpret_cast<uintptr_t>(target) & (talign - 1)) == 0 &&
         (glogits == nullptr || aligned16(glogits));
}

// GO(T, TT) for the (logits, target) storage types given by `dtype`, `tgt_dtype`
#define BCE_DICE_DISPATCH()                                                      \
  do {                                                                           \
    if (dtype == UNETB200_BF16) {                                                \
      if (tgt_dtype == UNETB200_F32) GO(bf16, float);                            \
      else if (tgt_dtype == UNETB200_I64) GO(bf16, long long);                   \
      else GO(bf16, uint8_t);                                                    \
    } else {                                                                     \
      if (tgt_dtype == UNETB200_F32) GO(float, float);                           \
      else if (tgt_dtype == UNETB200_I64) GO(float, long long);                  \
      else GO(float, uint8_t);                                                   \
    }                                                                            \
  } while (0)

int64_t unetb200_bce_dice_work_bytes(int64_t npix) {
  if (npix <= 0) return 0;
  return 4 * (int64_t)bce_dice_grid(npix) * (int64_t)sizeof(double);
}

int unetb200_bce_dice_fwd(const void* logits, int dtype, const void* target, int tgt_dtype, int64_t npix, float epsilon,
                          void* work, float* out, float* coefs, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "bce_dice_fwd: dtype");
  UB_CHECK_ARG(tgt_dtype == UNETB200_F32 || tgt_dtype == UNETB200_I64 || tgt_dtype == UNETB200_U8,
               "bce_dice_fwd: target dtype");
  UB_CHECK_ARG(npix > 0, "bce_dice_fwd: npix=%lld", (long long)npix);
  cudaStream_t s = (cudaStream_t)stream;
  const int g = bce_dice_grid(npix);
  const bool vec = bce_dice_vec(logits, target, tgt_dtype, nullptr);
  double* partials = (double*)work;
#define GO(T, TT) \
  bce_dice_fwd_kernel<T, TT><<<g, 256, 0, s>>>((const T*)logits, (const TT*)target, npix, vec, partials)
  BCE_DICE_DISPATCH();
#undef GO
  bce_dice_finalize_kernel<<<1, 256, 0, s>>>(partials, g, npix, epsilon, out, coefs);
  UB_LAUNCH_CHECK("bce_dice_fwd");
  return 0;
}

int unetb200_bce_dice_bwd(const void* logits, int dtype, const void* target, int tgt_dtype, int64_t npix,
                          const float* coefs, const float* gscale, void* glogits, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "bce_dice_bwd: dtype");
  UB_CHECK_ARG(tgt_dtype == UNETB200_F32 || tgt_dtype == UNETB200_I64 || tgt_dtype == UNETB200_U8,
               "bce_dice_bwd: target dtype");
  UB_CHECK_ARG(npix > 0, "bce_dice_bwd: npix=%lld", (long long)npix);
  cudaStream_t s = (cudaStream_t)stream;
  const int g = bce_dice_grid(npix);
  const bool vec = bce_dice_vec(logits, target, tgt_dtype, glogits);
#define GO(T, TT)                                                                                               \
  bce_dice_bwd_kernel<T, TT><<<g, 256, 0, s>>>((const T*)logits, (const TT*)target, npix, vec, coefs, gscale, \
                                               (T*)glogits)
  BCE_DICE_DISPATCH();
#undef GO
  UB_LAUNCH_CHECK("bce_dice_bwd");
  return 0;
}
#undef BCE_DICE_DISPATCH

int unetb200_dice_fwd(const float* x, const float* t, int64_t G, int64_t L, float epsilon, double* acc, float* out,
                      float* saved, void* stream) {
  UB_CHECK_ARG(G > 0 && G <= 65535 && L > 0, "dice_fwd: G=%lld L=%lld", (long long)G, (long long)L);
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(acc, 0, 3 * G * sizeof(double), s);
  if (e != cudaSuccess) return cuda_fail(e, "dice_fwd memset");
  int64_t gx = (L + 256 * 8 - 1) / (256 * 8);
  int64_t cap = (int64_t)sm_count() * 8 / G;
  if (cap < 1) cap = 1;
  if (gx > cap) gx = cap;
  dice_fwd_kernel<<<dim3((unsigned)gx, (unsigned)G), 256, 0, s>>>(x, t, L, acc);
  dice_finalize_kernel<<<1, 256, 0, s>>>(acc, G, epsilon, out, saved);
  UB_LAUNCH_CHECK("dice_fwd");
  return 0;
}

int unetb200_dice_bwd(const float* x, const float* t, int64_t G, int64_t L, float epsilon, const float* saved,
                      const float* gscale, float* gx, void* stream) {
  (void)x;
  (void)epsilon;
  UB_CHECK_ARG(G > 0 && G <= 65535 && L > 0, "dice_bwd: bad shape");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t gxn = (L + 256 * 4 - 1) / (256 * 4);
  int64_t cap = (int64_t)sm_count() * 8 / G;
  if (cap < 1) cap = 1;
  if (gxn > cap) gxn = cap;
  dice_bwd_kernel<<<dim3((unsigned)gxn, (unsigned)G), 256, 0, s>>>(t, G, L, saved, gscale, gx);
  UB_LAUNCH_CHECK("dice_bwd");
  return 0;
}

int64_t unetb200_boundary_work_bytes(void) { return 16 * 8 + 16; }

int unetb200_boundary_loss(const void* pred, int pred_dtype, int64_t sb, int64_t sh, int64_t sw, const void* target,
                           int tgt_dtype, int64_t tb, int64_t th, int64_t tw, int B, int H, int W, int edge_width,
                           float edge_weight, float smooth, void* work, float* out, void* stream) {
  UB_CHECK_ARG(pred_dtype == UNETB200_F32 || pred_dtype == UNETB200_BF16, "boundary_loss: pred dtype");
  UB_CHECK_ARG(tgt_dtype == UNETB200_F32 || tgt_dtype == UNETB200_I64, "boundary_loss: target dtype");
  UB_CHECK_ARG(B > 0 && H > 0 && W > 0 && edge_width >= 0, "boundary_loss: bad shape / negative edge_width");
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(work, 0, 16 * 8, s);
  if (e != cudaSuccess) return cuda_fail(e, "boundary memset");
  e = cudaMemsetAsync((char*)work + 16 * 8, 0xff, 4, s);        // encoded running minimum starts at +max
  if (e != cudaSuccess) return cuda_fail(e, "boundary init");
  e = cudaMemsetAsync((char*)work + 16 * 8 + 4, 0, 12, s);      // encoded running maximum starts at -max
  if (e != cudaSuccess) return cuda_fail(e, "boundary init");
  BoundaryGeom g;
  g.B = B; g.H = H; g.W = W;
  g.ewh = edge_width < H ? edge_width : H;
  g.eww = edge_width < W ? edge_width : W;
  g.has_edge = edge_width > 0;
  unsigned long long* cnt = (unsigned long long*)work;
  uint32_t* mm = (uint32_t*)((char*)work + 16 * 8);
  int grid = loss_grid((int64_t)B * H * W, 256);
#define GO(P, TT)                                                                         \
  do {                                                                                    \
    BoundaryIO<P, TT> io{(const P*)pred, sb, sh, sw, (const TT*)target, tb, th, tw};      \
    boundary_counts_kernel<P, TT><<<grid, 256, 0, s>>>(io, g, cnt, mm);                   \
  } while (0)
  if (pred_dtype == UNETB200_BF16) {
    if (tgt_dtype == UNETB200_F32) GO(bf16, float); else GO(bf16, long long);
  } else {
    if (tgt_dtype == UNETB200_F32) GO(float, float); else GO(float, long long);
  }
#undef GO
  boundary_finalize_kernel<<<1, 32, 0, s>>>(cnt, mm, g, edge_weight, smooth, out);
  UB_LAUNCH_CHECK("boundary_loss");
  return 0;
}
}
