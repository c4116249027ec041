// ConvTranspose2d(k=2, s=2) with narrow channel counts (C_in = 32 / 64 -> C_out = 16 / 32) on the tensor cores, TMA
// staged: the decoder up-samplers of the reference's light variants UNet_S / UNet_T / UNet_SA (unet_parts.py:72-74 at
// the widths of unet_model.py:52-189), which the CTA-pair / 64-channel kernels (conv_tc2.cu) do not cover and the
// CUDA-core engine ran at 0.1 of the HBM rate.  Same operand handling as conv_halo.cu (2C-byte pixel rows under the
// 32 / 64 / 128-byte swizzle, descriptors straight onto what TMA wrote):
//   * fprop  out[b, 2i+a, 2j+c, co] = sum_ci x[b,i,j,ci] W[ci,co,a,c] + bias[co]: a GEMM of 128-pixel tiles (2-D TMA box
//     over the flattened pixels) against the resident [4 C_out][C_in] weights; the epilogue scatters the four quadrants;
//   * dgrad  gx[b,i,j,ci] = sum_{a,c,co} g[b,2i+a,2j+c,co] W[ci,co,a,c]: the gradient is viewed as the 5-D tensor
//     {C_out, 2, w, 2, B h} (possible because H = 2h: image rows and batches merge), so each quadrant of a 16 x 8 pixel
//     tile is ONE dense TMA box = one K chunk of the GEMM;
//   * wgrad  dW[ci][(a,c),co] = sum_p x[p][ci] g_ac[p][co]: the four quadrant boxes sit 128 pixels apart in shared
//     memory, so ONE tcgen05.mma per 16 pixels covers all four (MN-major B with its N atoms one box apart, LBO).
#include <cstring>

#include "halo_common.cuh"

namespace ub {

constexpr int kHtThreads = 320;

// ------------------------------------------------------------------------------------------ fprop
struct HaloTParams {
  CUtensorMap x_map;             // 2-D {C1, npix}, box {C1, 128}
  const __nv_bfloat16* wp;       // [(q, co)][ci]
  const float* bias;             // [CUP] or null
  __nv_bfloat16* y;
  long long ld_out, npix;
  int h, w, Hout, Wout, off_y, off_x;
  int ntiles;
  int cup_real;                  // C_out = 8 rides the CUP = 16 instantiation (weight rows 8..15 of a quadrant are zero)
};

template <int C1, int CUP>
struct HaloTCfg {
  static constexpr int P = 2 * C1, NT = 4 * CUP;
  static constexpr uint32_t kStage = 128 * P;
  static constexpr uint32_t kB = NT * P;
  static constexpr int STAGES = 4;
  static constexpr int smem = STAGES * (int)kStage + (int)kB + 64 * 4 + 256 + 1024;
  static constexpr int CTAS = smem <= 110 * 1024 ? 2 : 1;
  static constexpr int kTmemCols = 2 * NT;
};

template <int C1, int CUP>
__global__ void __launch_bounds__(kHtThreads, HaloTCfg<C1, CUP>::CTAS) halo_t_fprop_kernel(const __grid_constant__ HaloTParams p) {
  using Cfg = HaloTCfg<C1, CUP>;
  constexpr int P = Cfg::P, NT = Cfg::NT, STAGES = Cfg::STAGES;
  constexpr uint32_t LAYOUT = halo_layout<P>();
  constexpr int CMASK = P / 16 - 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_ring = smem;
  uint8_t* b_tile = a_ring + STAGES * Cfg::kStage;
  float* sbias = reinterpret_cast<float*>(b_tile + Cfg::kB);
  uint64_t* full = reinterpret_cast<uint64_t*>(sbias + 64);
  uint64_t* empty = full + STAGES;
  uint64_t* t_full = empty + STAGES;
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], 8); }
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  for (int e = threadIdx.x; e < NT * (C1 / 8); e += blockDim.x) {
    const int n = e / (C1 / 8), c = e - n * (C1 / 8);
    const int q = n / CUP, co = n % CUP;
    const uint32_t addr = smem_u32(b_tile) + n * P;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (co < p.cup_real) v = *reinterpret_cast<const uint4*>(p.wp + (size_t)(q * p.cup_real + co) * C1 + c * 8);
    *reinterpret_cast<uint4*>(b_tile + n * P + ((c ^ ((addr >> 7) & CMASK)) << 4)) = v;
  }
  // the bias in the storage dtype, as the other engines add it (conv_tc2.cu, conv_simt.cu) and as autocast's bf16
  // ConvTranspose2d does
  if (threadIdx.x < 64)
    sbias[threadIdx.x] = (p.bias && threadIdx.x < p.cup_real) ? Elem<__nv_bfloat16>::round(p.bias[threadIdx.x]) : 0.f;
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 1;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        mbar_wait(&empty[s], ph);
        mbar_expect_tx(&full[s], Cfg::kStage);
        tma_load_2d(a_ring + s * Cfg::kStage, &p.x_map, &full[s], 0, tile * 128);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(false, false, false, 128, NT);
    const uint32_t a_base = smem_u32(a_ring), b_base = smem_u32(b_tile);
    uint32_t s = 0, ph = 0, acc = 0, pacc = 1;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      mbar_wait(&full[s], ph);
      mbar_wait(&t_empty[acc], pacc);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < C1 / 16; ++kk)
          umma<false>(tmem_base + acc * NT, make_desc(a_base + s * Cfg::kStage + kk * 32, 16, 8 * P, LAYOUT),
                      make_desc(b_base + kk * 32, 16, 8 * P, LAYOUT), idesc, kk ? 1u : 0u);
        umma_commit(&empty[s]);
        umma_commit(&t_full[acc]);
      }
      __syncwarp();
      if (++s == STAGES) { s = 0; ph ^= 1; }
      if (++acc == 2) { acc = 0; pacc ^= 1; }
    }
  } else {
    // epilogue: warp = (output row parity a, lane quarter); a thread owns one input pixel and writes the two output
    // pixels (2i + a, 2j), (2i + a, 2j + 1): columns [a * 2 CUP, +2 CUP) of the accumulator
    const int e = warp - 2, qy = e >> 2, quad = warp & 3;
    uint32_t acc = 0, pacc = 0;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      const long long pix = (long long)tile * 128 + quad * 32 + lane;
      const bool live = pix < p.npix;
      const long long pr = live ? pix : 0;
      const int j = (int)(pr % p.w);
      const long long r2 = pr / p.w;
      const int i = (int)(r2 % p.h), b = (int)(r2 / p.h);
      __nv_bfloat16* dst = p.y + (((long long)b * p.Hout + 2 * i + qy + p.off_y) * p.Wout + 2 * j + p.off_x) * p.ld_out;
      mbar_wait(&t_full[acc], pacc);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * NT + qy * 2 * CUP;
      __syncwarp();
#pragma unroll
      for (int hh = 0; hh < (2 * CUP) / 32; ++hh) {
        uint32_t v[32];
        tmem_ld32(taddr + hh * 32, v);
        if (hh == (2 * CUP) / 32 - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&t_empty[acc])) : "memory");
        }
        if (live) {
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8) {
            const int col = hh * 32 + c8 * 8;           // column within [0, 2 CUP): quadrant qx = col / CUP
            const int qx = col / CUP, co = col % CUP;
            uint4 o;
            o.x = halo_pack(__uint_as_float(v[c8 * 8 + 0]) + sbias[co + 0], __uint_as_float(v[c8 * 8 + 1]) + sbias[co + 1]);
            o.y = halo_pack(__uint_as_float(v[c8 * 8 + 2]) + sbias[co + 2], __uint_as_float(v[c8 * 8 + 3]) + sbias[co + 3]);
            o.z = halo_pack(__uint_as_float(v[c8 * 8 + 4]) + sbias[co + 4], __uint_as_float(v[c8 * 8 + 5]) + sbias[co + 5]);
            o.w = halo_pack(__uint_as_float(v[c8 * 8 + 6]) + sbias[co + 6], __uint_as_float(v[c8 * 8 + 7]) + sbias[co + 7]);
            if (co < p.cup_real) *reinterpret_cast<uint4*>(dst + qx * p.ld_out + co) = o;
          }
        }
      }
      if (++acc == 2) { acc = 0; pacc ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ dgrad
struct HaloTDParams {
  CUtensorMap g_map;             // 5-D {CUP, 2, w, 2, B h}, box {CUP, 1, 16, 1, 8}
  const __nv_bfloat16* wp;       // [ci][(q, co)]
  __nv_bfloat16* gx;             // [B][h][w][ld_out]
  long long ld_out;
  int h, w, tiles_w, tiles_h, ntiles;
  int cup_real, c1_real;         // 16 -> 8: the (CUP, C1) = (16, 32) instantiation, upper halves zero
};

template <int CUP, int C1>
struct HaloTDCfg {
  static constexpr int PG = 2 * CUP;
  static constexpr uint32_t kQ = 128 * PG;
  static constexpr uint32_t kStage = 4 * kQ;
  static constexpr uint32_t kBQ = C1 * PG < 1024 ? 1024u : (uint32_t)(C1 * PG);
  static constexpr int STAGES = 3;
  static constexpr int smem = STAGES * (int)kStage + 4 * (int)kBQ + 256 + 1024;
  static constexpr int CTAS = smem <= 110 * 1024 ? 2 : 1;
  static constexpr int kTmemCols = 2 * C1;
};

template <int CUP, int C1>
__global__ void __launch_bounds__(kHtThreads, HaloTDCfg<CUP, C1>::CTAS) halo_t_dgrad_kernel(const __grid_constant__ HaloTDParams p) {
  using Cfg = HaloTDCfg<CUP, C1>;
  constexpr int PG = Cfg::PG, STAGES = Cfg::STAGES;
  constexpr uint32_t LAYOUT = halo_layout<PG>();
  constexpr int CMASK = PG / 16 - 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_ring = smem;
  uint8_t* b_tile = a_ring + STAGES * Cfg::kStage;      // 4 quadrants x [C1 rows x PG bytes]
  uint64_t* full = reinterpret_cast<uint64_t*>(b_tile + 4 * Cfg::kBQ);
  uint64_t* empty = full + STAGES;
  uint64_t* t_full = empty + STAGES;
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], 8); }
    fence_barrier_init();
    tma_prefetch_desc(&p.g_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  for (int e = threadIdx.x; e < C1 * 4 * (CUP / 8); e += blockDim.x) {
    const int n = e / (4 * (CUP / 8)), r = e - n * (4 * (CUP / 8));
    const int q = r / (CUP / 8), c = r - q * (CUP / 8);
    const uint32_t off = q * Cfg::kBQ + n * PG;
    const uint32_t addr = smem_u32(b_tile) + off;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (n < p.c1_real && c * 8 < p.cup_real)
      v = *reinterpret_cast<const uint4*>(p.wp + (size_t)n * 4 * p.cup_real + q * p.cup_real + c * 8);
    *reinterpret_cast<uint4*>(b_tile + off + ((c ^ ((addr >> 7) & CMASK)) << 4)) = v;
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 1;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img, r = tile - b * tiles_per_img;
        const int ty = r / p.tiles_w, tx = r - ty * p.tiles_w;
        mbar_wait(&empty[s], ph);
        mbar_expect_tx(&full[s], Cfg::kStage);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          tma_load_5d(a_ring + s * Cfg::kStage + q * Cfg::kQ, &p.g_map, &full[s], 0, q & 1, tx * 16, q >> 1, b * p.h + ty * 8);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(false, false, false, 128, C1);
    const uint32_t a_base = smem_u32(a_ring), b_base = smem_u32(b_tile);
    uint32_t s = 0, ph = 0, acc = 0, pacc = 1;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      mbar_wait(&full[s], ph);
      mbar_wait(&t_empty[acc], pacc);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int kk = 0; kk < CUP / 16; ++kk)
            umma<false>(tmem_base + acc * C1, make_desc(a_base + s * Cfg::kStage + q * Cfg::kQ + kk * 32, 16, 8 * PG, LAYOUT),
                        make_desc(b_base + q * Cfg::kBQ + kk * 32, 16, 8 * PG, LAYOUT), idesc, (q | kk) ? 1u : 0u);
        umma_commit(&empty[s]);
        umma_commit(&t_full[acc]);
      }
      __syncwarp();
      if (++s == STAGES) { s = 0; ph ^= 1; }
      if (++acc == 2) { acc = 0; pacc ^= 1; }
    }
  } else {
    // epilogue: warp = (channel half, lane quarter); row m = 16 * y + x of the 16 x 8 pixel tile
    const int e = warp - 2, half = e >> 2, quad = warp & 3;
    constexpr int HC = C1 / 2;
    uint32_t acc = 0, pacc = 0;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      const int b = tile / tiles_per_img, r = tile - b * tiles_per_img;
      const int ty = r / p.tiles_w, tx = r - ty * p.tiles_w;
      const int m = quad * 32 + lane;
      const int y = ty * 8 + (m >> 4), x = tx * 16 + (m & 15);
      const bool live = y < p.h && x < p.w;
      mbar_wait(&t_full[acc], pacc);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * C1 + half * HC;
      __syncwarp();
      uint32_t v[HC];
      if constexpr (HC == 16) halo_tmem_ld16(taddr, v);
      else tmem_ld32(taddr, v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&t_empty[acc])) : "memory");
      if (live) {
        __nv_bfloat16* dst = p.gx + (((long long)b * p.h + y) * p.w + x) * p.ld_out + half * HC;
#pragma unroll
        for (int c8 = 0; c8 < HC / 8; ++c8) {
          if (half * HC + c8 * 8 >= p.c1_real) break;
          uint4 o;
          o.x = halo_pack(__uint_as_float(v[c8 * 8 + 0]), __uint_as_float(v[c8 * 8 + 1]));
          o.y = halo_pack(__uint_as_float(v[c8 * 8 + 2]), __uint_as_float(v[c8 * 8 + 3]));
          o.z = halo_pack(__uint_as_float(v[c8 * 8 + 4]), __uint_as_float(v[c8 * 8 + 5]));
          o.w = halo_pack(__uint_as_float(v[c8 * 8 + 6]), __uint_as_float(v[c8 * 8 + 7]));
          *reinterpret_cast<uint4*>(dst + c8 * 8) = o;
        }
      }
      if (++acc == 2) { acc = 0; pacc ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ wgrad
struct HaloTWParams {
  CUtensorMap x_map;             // 4-D {C1, w, h, B}, box {C1, 16, 8, 1}
  CUtensorMap g_map;             // 5-D {CUP, 2, w, 2, B h}, box {CUP, 1, 16, 1, 8}
  float* partials;               // [grid][C1][4 CUP]
  int h, tiles_w, tiles_h, ntiles;
  int cup_real;                  // C_out = 8: quadrant atoms of 16 channels whose upper half TMA zero-fills
};

template <int C1, int CUP>
struct HaloTWCfg {
  static constexpr int PX = 2 * C1, PG = 2 * CUP;
  static constexpr uint32_t kX = 128 * PX, kQ = 128 * PG;
  static constexpr uint32_t kStage = kX + 4 * kQ;
  static constexpr int kFixed = 256 + 1024;
  static constexpr int S2 = (110 * 1024 - kFixed) / (int)kStage;
  static constexpr int CTAS = S2 >= 2 ? 2 : 1;
  static constexpr int S1 = (220 * 1024 - kFixed) / (int)kStage;
  static constexpr int STAGES = CTAS == 2 ? (S2 > 4 ? 4 : S2) : (S1 > 4 ? 4 : S1);
  static constexpr int smem = STAGES * (int)kStage + kFixed;
  static constexpr int kCols = 4 * CUP;
};

template <int C1, int CUP>
__global__ void __launch_bounds__(192, HaloTWCfg<C1, CUP>::CTAS) halo_t_wgrad_kernel(const __grid_constant__ HaloTWParams p) {
  using Cfg = HaloTWCfg<C1, CUP>;
  constexpr int PX = Cfg::PX, PG = Cfg::PG, STAGES = Cfg::STAGES, NN = 4 * CUP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::kStage);
  uint64_t* empty = full + STAGES;
  uint64_t* t_full = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(t_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.g_map);
  }
  if (warp == 5) tmem_alloc(tmem_slot, Cfg::kCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (warp == 4) {
    if (lane == 0) {
      uint32_t s = 0, ph = 1;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        const int b = tile / tiles_per_img, r = tile - b * tiles_per_img;
        const int ty = r / p.tiles_w, tx = r - ty * p.tiles_w;
        mbar_wait(&empty[s], ph);
        mbar_expect_tx(&full[s], Cfg::kStage);
        uint8_t* st = smem + s * Cfg::kStage;
        tma_load_4d(st, &p.x_map, &full[s], 0, tx * 16, ty * 8, b);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          tma_load_5d(st + Cfg::kX + q * Cfg::kQ, &p.g_map, &full[s], 0, q & 1, tx * 16, q >> 1, b * p.h + ty * 8);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 5) {
    constexpr uint32_t idesc = make_idesc(false, true, true, 128, NN);
    constexpr uint32_t LX = halo_layout<PX>(), LG = halo_layout<PG>();
    uint32_t s = 0, ph = 0;
    int done = 0;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t xs = smem_u32(smem) + s * Cfg::kStage, gs = xs + Cfg::kX;
#pragma unroll
        for (int r = 0; r < 8; ++r)      // one image row of the tile = 16 pixels of K; the M atoms repeat the C1 channels (LBO = 0)
          umma<false>(tmem_base, make_desc(xs + r * 16 * PX, 0, 8 * PX, LX), make_desc(gs + r * 16 * PG, Cfg::kQ, 8 * PG, LG),
                      idesc, (done > 0 || r > 0) ? 1u : 0u);
        umma_commit(&empty[s]);
      }
      __syncwarp();
      ++done;
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    if (elect_one()) umma_commit(t_full);
    __syncwarp();
  } else if (warp * 32 < C1) {
    const int m = threadIdx.x;           // row = input channel (rows >= C1 repeat the atom: not read)
    mbar_wait(t_full, 0);
    tc_fence_after();
    float* out = p.partials + ((long long)blockIdx.x * C1 + m) * 4 * p.cup_real;
#pragma unroll 1
    for (int c0 = 0; c0 < NN; c0 += 16) {
      uint32_t v[16];
      halo_tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + c0, v);
      const int q = c0 / CUP, co0 = c0 % CUP;          // 16 columns never straddle a quadrant (CUP >= 16)
      if (m < C1) {
        float4* dst = reinterpret_cast<float4*>(out + q * p.cup_real + co0);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (co0 + 4 * e < p.cup_real)
            dst[e] = make_float4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]), __uint_as_float(v[4 * e + 2]),
                                 __uint_as_float(v[4 * e + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    __syncwarp();
    tmem_dealloc(tmem_base, Cfg::kCols);
  }
}

// ------------------------------------------------------------------------------------------ host side
static bool halo_t_pair_ok(int c1, int cup) {
  return (c1 == 32 && cup == 16) || (c1 == 64 && cup == 32) || (c1 == 32 && cup == 32) || (c1 == 64 && cup == 16) ||
         (c1 == 16 && cup == 8);           // UNet_T's last up-sampler: padded instantiations, see *_real
}

static bool halo_t_off() {
  static const bool off = getenv("UNETB200_NO_HALO") != nullptr || getenv("UNETB200_NO_HALO_T") != nullptr;
  return off;
}

// the transposed convolution itself: one tap, four output quadrants
static bool halo_t_fprop_shape(const unetb200_gconv_t* d) {
  if (halo_t_off() || d->dtype != UNETB200_BF16) return false;
  if (d->ntaps != 1 || d->tap_dy[0] || d->tap_dx[0] || d->in_scale != 1 || d->in_off_y || d->in_off_x) return false;
  if (d->nquad != 4 || d->out_scale != 2) return false;
  if (d->Hin != d->Hm || d->Win != d->Wm) return false;
  if (!halo_t_pair_ok(d->Cin, d->N / 4)) return false;
  if ((d->ld_in % 8) || (d->ld_out % 8)) return false;
  return (long long)d->B * d->Hm * d->Wm < (1LL << 31) - 256;
}
// its gradient arrives on a grid exactly twice the input's (no padding offsets): the 5-D view needs H = 2h
static bool halo_t_dense(int H, int W, int h, int w, int oy, int ox) { return H == 2 * h && W == 2 * w && oy == 0 && ox == 0; }

int halo_t_fprop_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y) {
  if (!halo_t_fprop_shape(d)) return 0;
  return aligned16(x) && aligned16(wp) && aligned16(y);
}

static bool halo_t_dgrad_shape(const unetb200_gconv_t* d) {
  if (halo_t_off() || d->dtype != UNETB200_BF16) return false;
  if (d->ntaps != 4 || d->in_scale != 2 || d->nquad != 1 || d->out_scale != 1 || d->out_off_y || d->out_off_x) return false;
  for (int t = 0; t < 4; ++t)
    if (d->tap_dy[t] != (t >> 1) || d->tap_dx[t] != (t & 1)) return false;
  if (d->Hout != d->Hm || d->Wout != d->Wm) return false;
  if (!halo_t_dense(d->Hin, d->Win, d->Hm, d->Wm, d->in_off_y, d->in_off_x)) return false;
  if (!halo_t_pair_ok(d->N, d->Cin)) return false;
  if ((d->ld_in % 8) || (d->ld_out % 8)) return false;
  return (long long)d->B * d->Hm * d->Wm < (1LL << 31) - 256;
}

int halo_t_dgrad_supported(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx) {
  if (!halo_t_dgrad_shape(d)) return 0;
  return aligned16(g) && aligned16(wp) && aligned16(gx);
}

int halo_t_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy) {
  static const bool off = getenv("UNETB200_NO_HALO_WGRAD") != nullptr;
  if (off || !halo_t_fprop_shape(d)) return 0;
  if (!halo_t_dense(d->Hout, d->Wout, d->Hm, d->Wm, d->out_off_y, d->out_off_x)) return 0;
  if ((x && !aligned16(x)) || (gy && !aligned16(gy))) return 0;
  return 1;
}

static int encode_quadrants(CUtensorMap* m, const void* g, int cup, int w, int h, int B, long long ld) {
  const long long W = 2LL * w;
  const unsigned long long dims[5] = {(unsigned long long)cup, 2ULL, (unsigned long long)w, 2ULL, (unsigned long long)B * h};
  const unsigned long long st[4] = {(unsigned long long)(ld * 2), (unsigned long long)(2 * ld * 2), (unsigned long long)(W * ld * 2),
                                    (unsigned long long)(2 * W * ld * 2)};
  const unsigned box[5] = {(unsigned)(cup < 16 ? 16 : cup), 1u, 16u, 1u, 8u};      // 8 channels: zero-filled upper half
  return encode_bf16_box(m, g, 5, dims, st, box);
}

template <int C1, int CUP>
static int halo_t_fprop_launch(const HaloTParams& P, cudaStream_t s) {
  using Cfg = HaloTCfg<C1, CUP>;
  static_assert(Cfg::smem <= 227 * 1024, "shared memory budget");
  if (int rc = set_max_dynamic_smem(reinterpret_cast<const void*>(&halo_t_fprop_kernel<C1, CUP>), Cfg::smem, "halo_t_fprop smem attribute"))
    return rc;
  const int slots = Cfg::CTAS * sm_count();
  const int grid = P.ntiles < slots ? P.ntiles : slots;
  halo_t_fprop_kernel<C1, CUP><<<grid, kHtThreads, Cfg::smem, s>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "halo_t_fprop launch");
  return 0;
}

int halo_t_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, const float* bias, void* y, cudaStream_t s) {
  if (!halo_t_fprop_supported(d, x, wp, y)) { set_error("halo_t_fprop: unsupported shape"); return UNETB200_E_INVALID; }
  HaloTParams P;
  memset(&P, 0, sizeof(P));
  const int cup = d->N / 4;
  P.npix = (long long)d->B * d->Hm * d->Wm;
  {
    const unsigned long long dims[2] = {(unsigned long long)d->Cin, (unsigned long long)P.npix};
    const unsigned long long st[1] = {(unsigned long long)(d->ld_in * 2)};
    const unsigned box[2] = {(unsigned)d->Cin, 128u};
    if (int rc = encode_bf16_box(&P.x_map, x, 2, dims, st, box)) return rc;
  }
  P.wp = (const __nv_bfloat16*)wp; P.bias = bias; P.y = (__nv_bfloat16*)y;
  P.ld_out = d->ld_out;
  P.h = d->Hm; P.w = d->Wm; P.Hout = d->Hout; P.Wout = d->Wout; P.off_y = d->out_off_y; P.off_x = d->out_off_x;
  P.ntiles = (int)((P.npix + 127) / 128);
  P.cup_real = cup;
  if (d->Cin == 16) return halo_t_fprop_launch<16, 16>(P, s);
  if (d->Cin == 32 && cup == 16) return halo_t_fprop_launch<32, 16>(P, s);
  if (d->Cin == 32 && cup == 32) return halo_t_fprop_launch<32, 32>(P, s);
  if (d->Cin == 64 && cup == 16) return halo_t_fprop_launch<64, 16>(P, s);
  return halo_t_fprop_launch<64, 32>(P, s);
}

template <int CUP, int C1>
static int halo_t_dgrad_launch(const HaloTDParams& P, cudaStream_t s) {
  using Cfg = HaloTDCfg<CUP, C1>;
  static_assert(Cfg::smem <= 227 * 1024, "shared memory budget");
  if (int rc = set_max_dynamic_smem(reinterpret_cast<const void*>(&halo_t_dgrad_kernel<CUP, C1>), Cfg::smem, "halo_t_dgrad smem attribute"))
    return rc;
  const int slots = Cfg::CTAS * sm_count();
  const int grid = P.ntiles < slots ? P.ntiles : slots;
  halo_t_dgrad_kernel<CUP, C1><<<grid, kHtThreads, Cfg::smem, s>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "halo_t_dgrad launch");
  return 0;
}

int halo_t_dgrad(const unetb200_gconv_t* d, const void* g, const void* wp, void* gx, cudaStream_t s) {
  if (!halo_t_dgrad_supported(d, g, wp, gx)) { set_error("halo_t_dgrad: unsupported shape"); return UNETB200_E_INVALID; }
  HaloTDParams P;
  memset(&P, 0, sizeof(P));
  if (int rc = encode_quadrants(&P.g_map, g, d->Cin, d->Wm, d->Hm, d->B, d->ld_in)) return rc;
  P.wp = (const __nv_bfloat16*)wp; P.gx = (__nv_bfloat16*)gx; P.ld_out = d->ld_out;
  P.h = d->Hm; P.w = d->Wm;
  P.tiles_w = (d->Wm + 15) / 16; P.tiles_h = (d->Hm + 7) / 8;
  P.ntiles = d->B * P.tiles_w * P.tiles_h;
  P.cup_real = d->Cin; P.c1_real = d->N;
  if (d->Cin == 8) return halo_t_dgrad_launch<16, 32>(P, s);
  if (d->Cin == 16 && d->N == 32) return halo_t_dgrad_launch<16, 32>(P, s);
  if (d->Cin == 32 && d->N == 32) return halo_t_dgrad_launch<32, 32>(P, s);
  if (d->Cin == 16 && d->N == 64) return halo_t_dgrad_launch<16, 64>(P, s);
  return halo_t_dgrad_launch<32, 64>(P, s);
}

template <int C1, int CUP>
static int halo_t_w_ctas() { return HaloTWCfg<C1, CUP>::CTAS; }

static int halo_t_wgrad_grid(const unetb200_gconv_t* d, int* tiles_w, int* tiles_h, int* ntiles) {
  *tiles_w = (d->Wm + 15) / 16;
  *tiles_h = (d->Hm + 7) / 8;
  *ntiles = d->B * *tiles_w * *tiles_h;
  const int cup = d->N / 4;
  if (d->Cin == 16) { const int sl = halo_t_w_ctas<16, 16>() * sm_count(); return *ntiles < sl ? *ntiles : sl; }
  const int per = d->Cin == 32 ? (cup == 16 ? halo_t_w_ctas<32, 16>() : halo_t_w_ctas<32, 32>())
                               : (cup == 16 ? halo_t_w_ctas<64, 16>() : halo_t_w_ctas<64, 32>());
  const int slots = per * sm_count();
  return *ntiles < slots ? *ntiles : slots;
}

int halo_t_wgrad_splits(const unetb200_gconv_t* d) {
  int tw, th, nt;
  return halo_t_wgrad_grid(d, &tw, &th, &nt);
}

template <int C1, int CUP>
static int halo_t_wgrad_launch(const HaloTWParams& P, int grid, cudaStream_t s) {
  using Cfg = HaloTWCfg<C1, CUP>;
  static_assert(Cfg::smem <= 227 * 1024 && Cfg::STAGES >= 2, "shared memory budget");
  if (int rc = set_max_dynamic_smem(reinterpret_cast<const void*>(&halo_t_wgrad_kernel<C1, CUP>), Cfg::smem, "halo_t_wgrad smem attribute"))
    return rc;
  halo_t_wgrad_kernel<C1, CUP><<<grid, 192, Cfg::smem, s>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "halo_t_wgrad launch");
  return 0;
}

int halo_t_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s) {
  if (!halo_t_wgrad_supported(d, x, gy)) { set_error("halo_t_wgrad: unsupported shape"); return UNETB200_E_INVALID; }
  HaloTWParams P;
  memset(&P, 0, sizeof(P));
  const int cup = d->N / 4;
  {
    const unsigned long long dims[4] = {(unsigned long long)d->Cin, (unsigned long long)d->Wm, (unsigned long long)d->Hm, (unsigned long long)d->B};
    const unsigned long long st[3] = {(unsigned long long)(d->ld_in * 2), (unsigned long long)((long long)d->Wm * d->ld_in * 2),
                                      (unsigned long long)((long long)d->Hm * d->Wm * d->ld_in * 2)};
    const unsigned box[4] = {(unsigned)d->Cin, 16u, 8u, 1u};
    if (int rc = encode_bf16_box(&P.x_map, x, 4, dims, st, box)) return rc;
  }
  if (int rc = encode_quadrants(&P.g_map, gy, cup, d->Wm, d->Hm, d->B, d->ld_out)) return rc;
  P.partials = partials;
  P.h = d->Hm;
  P.cup_real = cup;
  const int grid = halo_t_wgrad_grid(d, &P.tiles_w, &P.tiles_h, &P.ntiles);
  if (grid != splits) { set_error("halo_t_wgrad: the planned split count is %d, got %d", grid, splits); return UNETB200_E_INVALID; }
  if (d->Cin == 16) return halo_t_wgrad_launch<16, 16>(P, grid, s);
  if (d->Cin == 32 && cup == 16) return halo_t_wgrad_launch<32, 16>(P, grid, s);
  if (d->Cin == 32 && cup == 32) return halo_t_wgrad_launch<32, 32>(P, grid, s);
  if (d->Cin == 64 && cup == 16) return halo_t_wgrad_launch<64, 16>(P, grid, s);
  return halo_t_wgrad_launch<64, 32>(P, grid, s);
}

}  // namespace ub
