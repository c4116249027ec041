// The two ends of the step that touch bytes instead of activations (SURVEY.md section 8(f) N1 and N3):
//   * evaluate.py:111-117 / :56-66  -- argmax (or sigmoid threshold) + per-image class counts -> dice_coeff
//   * predict.py:26-27              -- F.interpolate(bilinear, align_corners=False) + argmax
//   * data_loading.py:65-89, 91-98  -- uint8 image -> fp32 (/255 when any value > 1), mask gray level -> class index,
//                                      the 90/180/270 degree rotation augmentation
// All of them are HBM-bound byte/integer passes: one coalesced read, one coalesced write, counts through
// warp shuffles -> shared memory -> one 64-bit atomic per block.  Integer results are exact by construction.
#include "common.cuh"

namespace ub {

// ------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long block_count(unsigned v, unsigned* smem) {
  // sum of a per-thread count over the block; valid in thread 0
  v = __reduce_add_sync(0xffffffffu, v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) smem[w] = v;
  __syncthreads();
  unsigned long long r = 0;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += smem[i];
  return r;
}

template <typename T>
__device__ __forceinline__ float load_target(const T* p);
template <>
__device__ __forceinline__ float load_target<float>(const float* p) { return *p; }
template <>
__device__ __forceinline__ float load_target<long long>(const long long* p) { return (float)*p; }

template <typename O>
__device__ __forceinline__ void store_index(O* p, int v) { *p = (O)v; }

// ------------------------------------------------------------------------------------------
// evaluate tail.  mode 0 (evaluate.py:111-117): pred = (argmax_c logits == cls), true = (target == cls)
//                 mode 1 (evaluate.py:56-66, n_classes == 1): pred = (sigmoid(z) rounded to T) > 0.5,
//                         true = floor(target / 2), which must be 0 or 1 (the reference asserts it)
// counts[b] = {sum pred*true, sum pred, sum true, #invalid targets}
// ------------------------------------------------------------------------------------------
constexpr int kEvalUnroll = 4;   // pixels per thread and iteration: four independent load chains in flight

template <typename T, typename TT, typename O>
__global__ void __launch_bounds__(256) eval_counts_kernel(const T* __restrict__ logits, int64_t sb, int64_t sc,
                                                          int64_t sh, int64_t sw, const TT* __restrict__ target, int C,
                                                          int H, int W, int cls, int mode, O* __restrict__ pred_out,
                                                          unsigned long long* __restrict__ counts) {
  __shared__ unsigned sm[32];
  constexpr int U = kEvalUnroll;
  const int b = blockIdx.y;
  const int64_t HW = (int64_t)H * W;
  const T* lb = logits + b * sb;
  const TT* tb = target ? target + b * HW : nullptr;
  O* ob = pred_out ? pred_out + b * HW : nullptr;
  unsigned ni = 0, np = 0, nt = 0, nbad = 0;
  const bool flat = sh == (int64_t)W * sw;
  // a block covers U consecutive runs of blockDim.x pixels; every run is one coalesced access per warp
  for (int64_t p0 = (int64_t)blockIdx.x * blockDim.x * U + threadIdx.x; p0 < HW;
       p0 += (int64_t)gridDim.x * blockDim.x * U) {
    int64_t p[U];
    const T* px[U];
    float t[U], best[U];
    int label[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      p[u] = p0 + (int64_t)u * blockDim.x;
      const int64_t q = p[u] < HW ? p[u] : HW - 1;      // out-of-range lanes re-read the last pixel, count nothing
      if (flat) {                                       // rows are back to back: no division
        px[u] = lb + q * sw;
      } else {
        const unsigned h = (unsigned)q / (unsigned)W, w = (unsigned)q - h * (unsigned)W;
        px[u] = lb + h * sh + w * sw;
      }
      t[u] = tb ? load_target<TT>(tb + q) : 0.f;
      best[u] = Elem<T>::ld(px[u]);
      label[u] = 0;
    }
    if (mode == 0) {
      for (int c = 1; c < C; ++c) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float v = Elem<T>::ld(px[u] + c * sc);
          // first maximum; NaN counts as the maximum (torch.argmax)
          if (v > best[u] || (v != v && best[u] == best[u])) { best[u] = v; label[u] = c; }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (p[u] >= HW) continue;
      bool pb, tbit = false;
      if (mode == 0) {
        pb = label[u] == cls;
      } else {
        pb = Elem<T>::round(1.f / (1.f + expf(-best[u]))) > 0.5f;
        label[u] = pb ? 1 : 0;
      }
      if (ob) store_index<O>(ob + p[u], label[u]);
      if (tb) {
        if (mode == 0) {
          tbit = t[u] == (float)cls;
        } else {
          const float th = floorf(t[u] * 0.5f);
          tbit = th == 1.f;
          nbad += !(th == 0.f || th == 1.f);
        }
      }
      ni += pb && tbit;
      np += pb;
      nt += tbit;
    }
  }
  unsigned long long r0 = block_count(ni, sm), r1 = block_count(np, sm), r2 = block_count(nt, sm),
                     r3 = block_count(nbad, sm);
  if (threadIdx.x == 0) {
    unsigned long long* c = counts + 4 * b;
    if (r0) atomicAdd(c + 0, r0);
    if (r1) atomicAdd(c + 1, r1);
    if (r2) atomicAdd(c + 2, r2);
    if (r3) atomicAdd(c + 3, r3);
  }
}

// Packed fast path (mode 0): the layout the UNet hands over -- NHWC with ld == C, C in {2,3,4}, H*W a multiple of 4.
// A thread owns 4 consecutive pixels: C 8-byte (bf16) / 16-byte (fp32) logit loads, one 16/32-byte target load, one
// 4/32-byte label store; ~10x fewer instructions per byte than the strided kernel above.
template <int C>
__device__ __forceinline__ void load_px4(const __nv_bfloat16* p, float* v) {
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < C; ++i) {
    const uint2 r = q[i];
    v[4 * i + 0] = __uint_as_float(r.x << 16);
    v[4 * i + 1] = __uint_as_float(r.x & 0xffff0000u);
    v[4 * i + 2] = __uint_as_float(r.y << 16);
    v[4 * i + 3] = __uint_as_float(r.y & 0xffff0000u);
  }
}
template <int C>
__device__ __forceinline__ void load_px4(const float* p, float* v) {
  const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int i = 0; i < C; ++i) {
    const float4 r = q[i];
    v[4 * i + 0] = r.x; v[4 * i + 1] = r.y; v[4 * i + 2] = r.z; v[4 * i + 3] = r.w;
  }
}
__device__ __forceinline__ void load_t4(const float* p, float* t) {
  const float4 r = *reinterpret_cast<const float4*>(p);
  t[0] = r.x; t[1] = r.y; t[2] = r.z; t[3] = r.w;
}
__device__ __forceinline__ void load_t4(const long long* p, float* t) {
  const longlong2 a = reinterpret_cast<const longlong2*>(p)[0], b = reinterpret_cast<const longlong2*>(p)[1];
  t[0] = (float)a.x; t[1] = (float)a.y; t[2] = (float)b.x; t[3] = (float)b.y;
}
__device__ __forceinline__ void store_lab4(long long* p, const int* l) {
  reinterpret_cast<longlong2*>(p)[0] = make_longlong2(l[0], l[1]);
  reinterpret_cast<longlong2*>(p)[1] = make_longlong2(l[2], l[3]);
}
__device__ __forceinline__ void store_lab4(uint8_t* p, const int* l) {
  *reinterpret_cast<uint32_t*>(p) = (uint32_t)l[0] | ((uint32_t)l[1] << 8) | ((uint32_t)l[2] << 16) | ((uint32_t)l[3] << 24);
}

template <typename T, typename TT, typename O, int C>
__global__ void __launch_bounds__(256) eval_counts_packed_kernel(const T* __restrict__ logits,
                                                                 const TT* __restrict__ target, int64_t groups,
                                                                 int cls, O* __restrict__ pred_out,
                                                                 unsigned long long* __restrict__ counts) {
  __shared__ unsigned sm[32];
  const int b = blockIdx.y;
  const T* lb = logits + (int64_t)b * groups * 4 * C;
  const TT* tb = target ? target + (int64_t)b * groups * 4 : nullptr;
  O* ob = pred_out ? pred_out + (int64_t)b * groups * 4 : nullptr;
  unsigned ni = 0, np = 0, nt = 0;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
    float v[4 * C], t[4] = {0.f, 0.f, 0.f, 0.f};
    load_px4<C>(lb + g * 4 * C, v);
    if (tb) load_t4(tb + g * 4, t);
    int lab[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float best = v[i * C];
      int idx = 0;
#pragma unroll
      for (int c = 1; c < C; ++c) {
        const float x = v[i * C + c];
        if (x > best || (x != x && best == best)) { best = x; idx = c; }
      }
      lab[i] = idx;
      const bool pb = idx == cls, tbit = tb && t[i] == (float)cls;
      ni += pb && tbit;
      np += pb;
      nt += tbit;
    }
    if (ob) store_lab4(ob + g * 4, lab);
  }
  if (counts) {
    unsigned long long r0 = block_count(ni, sm), r1 = block_count(np, sm), r2 = block_count(nt, sm);
    if (threadIdx.x == 0) {
      unsigned long long* c = counts + 4 * b;
      if (r0) atomicAdd(c + 0, r0);
      if (r1) atomicAdd(c + 1, r1);
      if (r2) atomicAdd(c + 2, r2);
    }
  }
}

// dice_coeff(pred, true, reduce_batch_first=False) on [B,H,W] 0/1 tensors (dice_score.py:5-25): per image
// inter = 2*I, sets = P + T (fp32 sums of 0/1 values are exact below 2^24), sets == 0 -> inter, mean over B.
__global__ void eval_dice_finalize_kernel(const unsigned long long* __restrict__ counts, int B, float eps,
                                          float* __restrict__ out) {
  if (threadIdx.x || blockIdx.x) return;
  float acc = 0.f;
  unsigned long long bad = 0;
  for (int b = 0; b < B; ++b) {
    const unsigned long long* c = counts + 4 * b;
    const float inter = 2.f * (float)c[0];
    float sets = (float)c[1] + (float)c[2];
    if (sets == 0.f) sets = inter;
    acc += (inter + eps) / (sets + eps);
    bad += c[3];
  }
  out[0] = bad ? NAN : acc / (float)B;
}

// ------------------------------------------------------------------------------------------
// predict tail: upsample_bilinear2d(align_corners=False) of every class plane, rounded to the storage
// type like ATen's output tensor, then first-max argmax.  ATen's source index (UpSample.h,
// area_pixel_compute_source_index): src = scale*(dst+0.5)-0.5 clamped at 0, scale = in/out in fp32.
// ------------------------------------------------------------------------------------------
struct Lerp { int i0, di; float l0, l1; };
__device__ __forceinline__ Lerp lerp_index(int dst, float scale, int in_size) {
  // ATen's order, without FMA contraction so the host restatement reproduces it bit for bit
  float src = __fsub_rn(__fmul_rn(scale, (float)dst + 0.5f), 0.5f);
  if (src < 0.f) src = 0.f;
  Lerp r;
  r.i0 = min((int)src, in_size - 1);
  r.di = r.i0 < in_size - 1 ? 1 : 0;
  r.l1 = src - (float)r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

template <typename T, typename O>
__global__ void resize_argmax_kernel(const T* __restrict__ logits, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                                     int C, int h, int w, int H, int W, float scale_h, float scale_w,
                                     O* __restrict__ out) {
  const int b = blockIdx.y;
  const int64_t HW = (int64_t)H * W;
  const T* lb = logits + b * sb;
  O* ob = out + b * HW;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < HW; p += (int64_t)gridDim.x * blockDim.x) {
    const int oy = (int)((unsigned)p / (unsigned)W), ox = (int)((unsigned)p - (unsigned)oy * (unsigned)W);
    const Lerp ly = lerp_index(oy, scale_h, h), lx = lerp_index(ox, scale_w, w);
    const T* p00 = lb + ly.i0 * sh + lx.i0 * sw;
    const int64_t dy = ly.di * sh, dx = lx.di * sw;
    float best = 0.f;
    int idx = 0;
    for (int c = 0; c < C; ++c) {
      const T* q = p00 + c * sc;
      const float v00 = Elem<T>::ld(q), v01 = Elem<T>::ld(q + dx), v10 = Elem<T>::ld(q + dy),
                  v11 = Elem<T>::ld(q + dy + dx);
      const float top = __fadd_rn(__fmul_rn(lx.l0, v00), __fmul_rn(lx.l1, v01));
      const float bot = __fadd_rn(__fmul_rn(lx.l0, v10), __fmul_rn(lx.l1, v11));
      float v = __fadd_rn(__fmul_rn(ly.l0, top), __fmul_rn(ly.l1, bot));
      v = Elem<T>::round(v);
      if (c == 0 || v > best || (v != v && best == best)) { best = v; idx = c; }
    }
    store_index<O>(ob + p, idx);
  }
}

// ------------------------------------------------------------------------------------------
// input pipeline: tiles of 32x32 output pixels; the matching input tile is read row-major (coalesced along the
// input x axis), staged in shared memory, and written row-major along the output x axis, so a 90/270 degree
// rotation costs no uncoalesced access.  rot = k means numpy.rot90(a, k) == PIL Image.rotate(90 k, expand=True)
// (counter-clockwise); output pixel (i, j) reads input pixel
//   k=0: (i, j)   k=1: (j, W-1-i)   k=2: (H-1-i, W-1-j)   k=3: (H-1-j, i)
// ------------------------------------------------------------------------------------------
constexpr int kTile = 32;
constexpr int kMaxImgC = 4;

__global__ void u8_any_gt1_kernel(const uint8_t* __restrict__ src, int64_t per_image, int* __restrict__ flags) {
  const int b = blockIdx.y;
  const uint8_t* s = src + b * per_image;
  bool any = false;
  const int64_t nvec = (reinterpret_cast<uintptr_t>(s) & 15) == 0 ? per_image / 16 : 0;
  const uint4* v = reinterpret_cast<const uint4*>(s);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 q = v[i];
    // a byte is > 1 iff any of its bits 1..7 is set
    any |= ((q.x | q.y | q.z | q.w) & 0xfefefefeu) != 0;
  }
  for (int64_t i = nvec * 16 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < per_image;
       i += (int64_t)gridDim.x * blockDim.x)
    any |= s[i] > 1;
  if (__syncthreads_or(any) && threadIdx.x == 0) atomicOr(flags + b, 1);
}

struct ImageOp {        // data_loading.py:82-87: float32(v) / 255.0 when the image has a value > 1, else float32(v)
  const int* flags;
  typedef float out_t;
  __device__ __forceinline__ float apply(uint8_t v, int b) const {
    return flags[b] ? __fdiv_rn((float)v, 255.f) : (float)v;
  }
};
struct MaskOp {         // data_loading.py:74-79: 255 -> 2, 128 -> 1, everything else 0; or a caller-supplied table
  const long long* lut;
  typedef long long out_t;
  __device__ __forceinline__ long long apply(uint8_t v, int) const {
    if (lut) return lut[v];
    return v == 255 ? 2 : (v == 128 ? 1 : 0);
  }
};

template <typename Op, int C>
__global__ void __launch_bounds__(256) rot_convert_kernel(const uint8_t* __restrict__ src, int H, int W,
                                                          const int* __restrict__ rot, int Ho, int Wo, Op op,
                                                          typename Op::out_t* __restrict__ dst) {
  constexpr int kRow = kTile * C;                      // bytes per tile row: divisions below are by constants
  __shared__ uint8_t tile[kTile][kRow + 4];
  const int b = blockIdx.z;
  const int k = rot ? (rot[b] & 3) : 0;
  const int i0 = blockIdx.y * kTile, j0 = blockIdx.x * kTile;   // output tile origin (row, column)
  int y0, x0;                                                   // input tile origin
  switch (k) {
    case 0: y0 = i0; x0 = j0; break;
    case 1: y0 = j0; x0 = W - kTile - i0; break;
    case 2: y0 = H - kTile - i0; x0 = W - kTile - j0; break;
    default: y0 = H - kTile - j0; x0 = i0; break;
  }
  const uint8_t* sb = src + (int64_t)b * H * W * C;
  const int wbytes = W * C;
#pragma unroll
  for (int it = 0; it < kTile * kRow / 256; ++it) {
    const int t = it * 256 + threadIdx.x;
    const int ty = t / kRow, tb = t - ty * kRow;
    const int y = y0 + ty, xb = x0 * C + tb;
    uint8_t v = 0;
    if (y >= 0 && y < H && xb >= 0 && xb < wbytes) v = sb[(int64_t)y * wbytes + xb];
    tile[ty][tb] = v;
  }
  __syncthreads();
  typename Op::out_t* db = dst + (int64_t)b * Ho * Wo * C;
  // tile coordinates of output element (ti, tj, c): (ay*ti + by*tj + cy, ax*ti + bx*tj + cx)
  int ay, by, cy, ax, bx, cx;
  switch (k) {
    case 0: ay = 1; by = 0; cy = 0; ax = 0; bx = 1; cx = 0; break;
    case 1: ay = 0; by = 1; cy = 0; ax = -1; bx = 0; cx = kTile - 1; break;
    case 2: ay = -1; by = 0; cy = kTile - 1; ax = 0; bx = -1; cx = kTile - 1; break;
    default: ay = 0; by = -1; cy = kTile - 1; ax = 1; bx = 0; cx = 0; break;
  }
#pragma unroll
  for (int it = 0; it < kTile * kRow / 256; ++it) {
    const int t = it * 256 + threadIdx.x;
    const int ti = t / kRow, r = t - ti * kRow;
    const int tj = r / C, c = r - tj * C;
    const int i = i0 + ti, j = j0 + tj;
    if (i >= Ho || j >= Wo) continue;
    const int ty = ay * ti + by * tj + cy, tx = ax * ti + bx * tj + cx;
    const int y = y0 + ty, x = x0 + tx;
    typename Op::out_t v = 0;
    if (y >= 0 && y < H && x >= 0 && x < W) v = op.apply(tile[ty][tx * C + c], b);
    db[((int64_t)i * Wo + j) * C + c] = v;
  }
}

template <typename Op>
static void launch_rot_convert(const uint8_t* src, int H, int W, int C, const int* rot, int Ho, int Wo, Op op,
                               typename Op::out_t* dst, int B, cudaStream_t s) {
  dim3 grid((Wo + kTile - 1) / kTile, (Ho + kTile - 1) / kTile, B);
  switch (C) {
    case 1: rot_convert_kernel<Op, 1><<<grid, 256, 0, s>>>(src, H, W, rot, Ho, Wo, op, dst); break;
    case 2: rot_convert_kernel<Op, 2><<<grid, 256, 0, s>>>(src, H, W, rot, Ho, Wo, op, dst); break;
    case 3: rot_convert_kernel<Op, 3><<<grid, 256, 0, s>>>(src, H, W, rot, Ho, Wo, op, dst); break;
    default: rot_convert_kernel<Op, 4><<<grid, 256, 0, s>>>(src, H, W, rot, Ho, Wo, op, dst); break;
  }
}

}  // namespace ub

using namespace ub;

static inline int tail_grid(int64_t work_per_image, int B, int threads) {
  int64_t b = (work_per_image + threads - 1) / threads;
  int64_t cap = ((int64_t)sm_count() * 8 + B - 1) / B;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// mode-0 evaluate tail (and the identity-size predict tail) on packed NHWC logits; returns false when the shape does
// not qualify and the strided kernel has to run
static bool launch_eval_packed(const void* logits, int dtype, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                               const void* target, int tgt_dtype, int B, int C, int H, int W, int cls, void* pred_out,
                               bool u8, unsigned long long* cnt, cudaStream_t s) {
  const int64_t HW = (int64_t)H * W;
  if (C < 2 || C > 4 || (HW & 3)) return false;
  if (sc != 1 || sw != C || sh != (int64_t)W * C || (B > 1 && sb != HW * C)) return false;
  if (!aligned16(logits) || (target && !aligned16(target)) || (pred_out && !aligned16(pred_out))) return false;
  const int64_t groups = HW / 4;
  dim3 grid(tail_grid(groups, B, 256), B);
  with_elem(dtype, [&](auto t) {
    with_type<long long, float>(target ? tgt_dtype : UNETB200_F32, [&](auto tt) {
      with_type<uint8_t, long long>(u8 ? UNETB200_U8 : UNETB200_I64, [&](auto o) {
        with_int<2, 3, 4>(C, [&](auto CC) {
          using T = decltype(t);
          using TT = decltype(tt);
          using O = decltype(o);
          eval_counts_packed_kernel<T, TT, O, CC><<<grid, 256, 0, s>>>((const T*)logits, (const TT*)target, groups,
                                                                       cls, (O*)pred_out, cnt);
        });
      });
    });
  });
  return true;
}

extern "C" {

int unetb200_eval_counts(const void* logits, int dtype, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                         const void* target, int tgt_dtype, int B, int C, int H, int W, int cls, int mode,
                         void* pred_out, int pred_dtype, int64_t* counts, float epsilon, float* dice_out,
                         void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "eval_counts: logits dtype");
  UB_CHECK_ARG(target == nullptr || tgt_dtype == UNETB200_F32 || tgt_dtype == UNETB200_I64,
               "eval_counts: target dtype");
  UB_CHECK_ARG(pred_out == nullptr || pred_dtype == UNETB200_I64 || pred_dtype == UNETB200_U8,
               "eval_counts: prediction dtype must be int64 or uint8");
  UB_CHECK_ARG(B > 0 && B <= 65535 && C >= 1 && H > 0 && W > 0, "eval_counts: bad shape B=%d C=%d H=%d W=%d", B, C,
               H, W);
  UB_CHECK_ARG((int64_t)H * W < (1ll << 31), "eval_counts: H*W must be below 2^31");
  UB_CHECK_ARG(mode == 0 || (mode == 1 && C == 1), "eval_counts: mode %d needs C == 1 (got %d)", mode, C);
  UB_CHECK_ARG(counts != nullptr, "eval_counts: counts workspace");
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(counts, 0, (size_t)B * 4 * sizeof(int64_t), s);
  if (e != cudaSuccess) return cuda_fail(e, "eval_counts memset");
  dim3 grid(tail_grid(((int64_t)H * W + kEvalUnroll - 1) / kEvalUnroll, B, 256), B);
  unsigned long long* cnt = (unsigned long long*)counts;
  const bool u8 = pred_out && pred_dtype == UNETB200_U8;
  if (mode == 0 && launch_eval_packed(logits, dtype, sb, sc, sh, sw, target, tgt_dtype, B, C, H, W, cls, pred_out, u8,
                                      cnt, s)) {
    if (dice_out) eval_dice_finalize_kernel<<<1, 32, 0, s>>>(cnt, B, epsilon, dice_out);
    UB_LAUNCH_CHECK("eval_counts");
    return 0;
  }
  with_elem(dtype, [&](auto t) {
    with_type<long long, float>(tgt_dtype, [&](auto tt) {
      with_type<uint8_t, long long>(u8 ? UNETB200_U8 : UNETB200_I64, [&](auto o) {
        using T = decltype(t);
        using TT = decltype(tt);
        using O = decltype(o);
        eval_counts_kernel<T, TT, O><<<grid, 256, 0, s>>>((const T*)logits, sb, sc, sh, sw, (const TT*)target, C, H,
                                                          W, cls, mode, (O*)pred_out, cnt);
      });
    });
  });
  if (dice_out) eval_dice_finalize_kernel<<<1, 32, 0, s>>>(cnt, B, epsilon, dice_out);
  UB_LAUNCH_CHECK("eval_counts");
  return 0;
}

int unetb200_resize_argmax(const void* logits, int dtype, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int B,
                           int C, int h, int w, int H, int W, void* out, int out_dtype, void* stream) {
  UB_CHECK_ARG(dtype == UNETB200_F32 || dtype == UNETB200_BF16, "resize_argmax: logits dtype");
  UB_CHECK_ARG(out_dtype == UNETB200_I64 || out_dtype == UNETB200_U8, "resize_argmax: output dtype");
  UB_CHECK_ARG(B > 0 && B <= 65535 && C >= 1 && h > 0 && w > 0 && H > 0 && W > 0, "resize_argmax: bad shape");
  UB_CHECK_ARG((int64_t)H * W < (1ll << 31), "resize_argmax: H*W must be below 2^31");
  cudaStream_t s = (cudaStream_t)stream;
  // same size: the interpolation is the identity (lambda = 0 exactly), so this is the plain argmax
  if (h == H && w == W && launch_eval_packed(logits, dtype, sb, sc, sh, sw, nullptr, UNETB200_F32, B, C, H, W, 0, out,
                                             out_dtype == UNETB200_U8, nullptr, s)) {
    UB_LAUNCH_CHECK("resize_argmax");
    return 0;
  }
  dim3 grid(tail_grid((int64_t)H * W, B, 256), B);
  const float sch = (float)h / (float)H, scw = (float)w / (float)W;
  with_elem(dtype, [&](auto t) {
    with_type<uint8_t, long long>(out_dtype, [&](auto o) {
      using T = decltype(t);
      using O = decltype(o);
      resize_argmax_kernel<T, O><<<grid, 256, 0, s>>>((const T*)logits, sb, sc, sh, sw, C, h, w, H, W, sch, scw,
                                                      (O*)out);
    });
  });
  UB_LAUNCH_CHECK("resize_argmax");
  return 0;
}

int unetb200_preprocess_image_u8(const uint8_t* src, int B, int H, int W, int C, const int32_t* rot, int transposed,
                                 float* dst, int32_t* flags, void* stream) {
  UB_CHECK_ARG(B > 0 && B <= 65535 && H > 0 && W > 0 && C >= 1 && C <= kMaxImgC,
               "preprocess_image_u8: bad shape B=%d H=%d W=%d C=%d (C <= %d)", B, H, W, C, kMaxImgC);
  UB_CHECK_ARG(src && dst && flags, "preprocess_image_u8: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)B * sizeof(int32_t), s);
  if (e != cudaSuccess) return cuda_fail(e, "preprocess_image_u8 memset");
  const int64_t per_image = (int64_t)H * W * C;
  u8_any_gt1_kernel<<<dim3(tail_grid(per_image / 16 + 1, B, 256), B), 256, 0, s>>>(src, per_image, flags);
  const int Ho = transposed ? W : H, Wo = transposed ? H : W;
  launch_rot_convert<ImageOp>(src, H, W, C, rot, Ho, Wo, ImageOp{flags}, dst, B, s);
  UB_LAUNCH_CHECK("preprocess_image_u8");
  return 0;
}

int unetb200_preprocess_mask_u8(const uint8_t* src, int B, int H, int W, const int32_t* rot, int transposed,
                                const int64_t* lut, int64_t* dst, void* stream) {
  UB_CHECK_ARG(B > 0 && B <= 65535 && H > 0 && W > 0, "preprocess_mask_u8: bad shape B=%d H=%d W=%d", B, H, W);
  UB_CHECK_ARG(src && dst, "preprocess_mask_u8: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  const int Ho = transposed ? W : H, Wo = transposed ? H : W;
  launch_rot_convert<MaskOp>(src, H, W, 1, rot, Ho, Wo, MaskOp{(const long long*)lut}, (long long*)dst, B, s);
  UB_LAUNCH_CHECK("preprocess_mask_u8");
  return 0;
}
}
