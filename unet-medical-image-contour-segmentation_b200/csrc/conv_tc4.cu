// Fourth-generation weight-gradient kernel for the narrow 3x3 layers (C_in, C_out in {64, 128}: the full- and
// half-resolution DoubleConvs of unet_model.py:15-16,23-24, autograd wgrad of unet_parts.py:15,18).
//
//   dW[(dy,dx)][c][n] = sum_p x[p + (dy,dx)][c] * g[p][n]          (K = pixels, both operands MN-major)
//
// What bounded the previous kernels on these layers (tools/umma_probe.cu, profiles/r1_umma_probe_rate*.txt):
// a tcgen05.mma re-reads both operands from shared memory, ~96 B/cycle/SM.  With the 64 output channels of dY as
// the N operand (tc2_wgrad_kernel) an M = 128 MMA costs 77 cycles against a tensor floor of 32 (41 %); as a CTA
// pair 49 (65 %), and the unit counts of these layers (3 or 6) do not fill pairs of 4.
//
// Here the N operand is made wide by shifting dY instead of x along the row:  with q = p + (0, s - 1)
//   dW[(dy, 1 - s)][c][n] = sum_q x[q + (dy, 0)][c] * g[q + (0, s - 1)][n],     s = 0, 1, 2
// so ONE dY halo box {128 B, 8 + 2 px, 8 rows} serves the three column shifts: an MN-major descriptor whose
// 64-channel sub-tiles are LBO = 128 B (one pixel) apart and whose 8-pixel groups are SBO = 10 * 128 B apart
// reads N = 192 = (s, n) straight out of the box (unaligned starts / strides: probe check (c)).  The x box
// {128 B, 8 px, 8 + 2 rows} serves the three row shifts as before; M = 128 = (dy, dy + 1) x 64 channels with
// LBO = 1024 B.  A CTA owns one (64-channel chunk of x, 64-channel group of dY) pair = all nine taps:
//   accumulator 0: rows (dy = -1 | dy = 0), accumulator 1: rows (dy = +1 | unused), 192 columns each.
// Two M = 128, N = 192 MMAs per 16 pixels (~104 cycles each against a floor of 96) produce 192 x 192 useful
// outputs: 75 % of the MMA volume is useful (3 x 3 does not factor into 2 x k) at ~92 % of the tensor rate,
// against 31-41 % before.  Fill per 64-pixel step: 10 KB + 10 KB for 8 MMAs (~24 B/cycle/SM).
#include <cstring>

#include "tc_common.cuh"

namespace ub {

struct alignas(64) Tc4WParams {
  CUtensorMap a_map;         // x view, box {128 B, 8, 10, 1}
  CUtensorMap o_map;         // dY view, box {128 B, 10, 8, 1}
  int tap[3][3];             // [dy + 1][dx + 1] -> tap index of the gconv descriptor
  int Cin, N, K;
  int cchunks;
  int tiles_w, tiles_h;
  int ptiles, ptiles_per_split;
  float* partials;
};

constexpr uint32_t kT4Box = 10240;            // either box: 80 pixels x 128 B
constexpr uint32_t kT4Stage = 2 * kT4Box;
constexpr int kT4AccCols = 192;

template <int STAGES>
__global__ void __launch_bounds__(192, 1) tc4_wgrad_kernel(const __grid_constant__ Tc4WParams p) {
  constexpr int UMMA_K = 16, MMAS = 64 / UMMA_K;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * kT4Stage);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x % p.cchunks;                // 64-channel chunk of x
  const int g = blockIdx.x / p.cchunks;                // 64-channel group of dY
  const int split = blockIdx.z;
  const int pt_begin = split * p.ptiles_per_split;
  int pt_end = pt_begin + p.ptiles_per_split;
  if (pt_end > p.ptiles) pt_end = p.ptiles;
  const int num_k = pt_end - pt_begin;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.a_map);
    tma_prefetch_desc(&p.o_map);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    int pt = pt_begin;
    int tj = pt % p.tiles_w;
    int rest = pt / p.tiles_w;
    int ti = rest % p.tiles_h;
    int b = rest / p.tiles_h;
    uint32_t s = 0, ph = 1;
    for (int kb = 0; kb < num_k; ++kb) {
      mbar_wait(&empty_bar[s], ph);
      if (elect_one()) {
        mbar_expect_tx(&full_bar[s], kT4Stage);
        const int i0 = ti * 8, j0 = tj * 8;
        uint8_t* sa = smem + s * kT4Stage;
        tma_load_4d(sa, &p.a_map, &full_bar[s], c * 64, j0, i0 - 1, b);              // rows i0-1 .. i0+8
        tma_load_4d(sa + kT4Box, &p.o_map, &full_bar[s], g * 64, j0 - 1, i0, b);     // columns j0-1 .. j0+8
      }
      if (++s == STAGES) { s = 0; ph ^= 1; }
      if (++tj == p.tiles_w) { tj = 0; if (++ti == p.tiles_h) { ti = 0; ++b; } }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(false, true, true, 128, kT4AccCols);
    // A: sub-tile h = row shift dy0 + h (1024 B = one 8-pixel box row apart), 8-pixel groups 1024 B apart
    // B: sub-tile s = column shift s - 1 (one pixel = 128 B apart), 8-pixel groups one 10-pixel box row apart
    const uint64_t da_t = make_desc(smem_u32(smem), 1024, 1024, kLayoutSW128);
    const uint64_t db_t = make_desc(smem_u32(smem) + kT4Box, 128, 1280, kLayoutSW128);
    uint32_t s = 0, ph = 0;
    for (int kb = 0; kb < num_k; ++kb) {
      mbar_wait(&full_bar[s], ph);
      tc_fence_after();
      const uint64_t da0 = da_t + s * (kT4Stage >> 4), db0 = db_t + s * (kT4Stage >> 4);
      if (elect_one()) {
#pragma unroll
        for (int a = 0; a < 2; ++a) {
#pragma unroll
          for (int k = 0; k < MMAS; ++k)
            umma<false>(tmem_base + a * kT4AccCols, da0 + ((a * 2048 + k * 2 * 1024) >> 4), db0 + ((k * 2 * 1280) >> 4),
                        idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty_bar[s]);
      }
      __syncwarp();
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;                  // D row = (row shift half, channel row % 64)
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    for (int a = 0; a < 2; ++a) {
      const int dy1 = 2 * a + (row >> 6);              // dy + 1; 3 = the unused half of accumulator 1
      const bool live = dy1 < 3;                       // warp-uniform (a warp holds 32 consecutive rows)
#pragma unroll 1
      for (int sft = 0; sft < 3; ++sft) {
        const int t = live ? p.tap[dy1][2 - sft] : 0;  // column shift s - 1 of dY <-> tap dx = 1 - s
        const long long k = (long long)t * p.Cin + c * 64 + (row & 63);
        float* out = p.partials + (long long)split * p.K * p.N + k * p.N + g * 64;
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + a * kT4AccCols + sft * 64 + ch * 32, v);
          if (live) {
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              float4 o4 = num_k > 0 ? make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]),
                                                  __uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
              *reinterpret_cast<float4*>(out + ch * 32 + e) = o4;
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

struct Tc4WPlan {
  int cchunks, ngroups, tiles_w, tiles_h, ptiles;
  int tap[3][3];
};

static bool tc4_wgrad_plan(const unetb200_gconv_t* d, Tc4WPlan* w) {
  // UNETB200_TC4W=0: off, for A/B runs (=all is read by the route in gconv.cu)
  static const bool off = [] {
    const char* e = getenv("UNETB200_TC4W");
    return e && !strcmp(e, "0");
  }();
  if (off) return false;
  if (d->dtype != UNETB200_BF16) return false;
  if (d->nquad != 1 || d->in_scale != 1 || d->out_scale != 1 || d->ntaps != 9) return false;
  if (d->in_off_y || d->in_off_x) return false;
  if (d->Cin % 64 || d->N % 64) return false;
  if ((d->ld_in * 2) % 16 || (d->ld_out * 2) % 16) return false;
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) {
      int found = -1;
      for (int t = 0; t < 9; ++t)
        if (d->tap_dy[t] == a - 1 && d->tap_dx[t] == b - 1) found = t;
      if (found < 0) return false;
      w->tap[a][b] = found;
    }
  w->cchunks = d->Cin / 64;
  w->ngroups = d->N / 64;
  w->tiles_w = (d->Wm + 7) / 8;
  w->tiles_h = (d->Hm + 7) / 8;
  w->ptiles = d->B * w->tiles_w * w->tiles_h;
  return true;
}

int tc4_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy) {
  Tc4WPlan w;
  if (!tc4_wgrad_plan(d, &w)) return 0;
  if ((x && !aligned16(x)) || (gy && !aligned16(gy))) return 0;
  return 1;
}

int tc4_wgrad_splits(const unetb200_gconv_t* d) {
  Tc4WPlan w;
  if (!tc4_wgrad_plan(d, &w)) return 1;
  const long long tiles = (long long)w.cchunks * w.ngroups;
  const long long max_by_k = (w.ptiles + 15) / 16;      // at least 16 pixel tiles (1024 pixels) per split
  return pick_splits(tiles, sm_count(), max_by_k);      // one CTA per SM: whole waves
}

int tc4_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
              cudaStream_t stream) {
  Tc4WPlan w;
  if (!tc4_wgrad_plan(d, &w)) { set_error("tc4_wgrad: unsupported shape"); return UNETB200_E_INVALID; }
  Tc4WParams P;
  memset(&P, 0, sizeof(P));
  int rc = encode_act_box(&P.a_map, d->dtype, x, d->Cin, d->Win, d->Hin, d->B, d->ld_in, (long long)d->Win * d->ld_in,
                          (long long)d->Hin * d->Win * d->ld_in, 8, 10, true);
  if (rc) return rc;
  const char* obase = (const char*)gy + ((long long)d->out_off_y * d->Wout + d->out_off_x) * d->ld_out * 2LL;
  rc = encode_act_box(&P.o_map, d->dtype, obase, d->N, d->Wm, d->Hm, d->B, d->ld_out, (long long)d->Wout * d->ld_out,
                      (long long)d->Hout * d->Wout * d->ld_out, 10, 8, true);
  if (rc) return rc;
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) P.tap[a][b] = w.tap[a][b];
  P.Cin = d->Cin; P.N = d->N; P.K = g.K;
  P.cchunks = w.cchunks;
  P.tiles_w = w.tiles_w; P.tiles_h = w.tiles_h;
  P.ptiles = w.ptiles;
  P.ptiles_per_split = (w.ptiles + splits - 1) / splits;
  P.partials = partials;
  constexpr int ST = 10;
  constexpr int smem = ST * (int)kT4Stage + 1024 + 256;
  static_assert(smem <= 227 * 1024, "shared memory budget");
  if (int e = set_max_dynamic_smem(reinterpret_cast<const void*>(&tc4_wgrad_kernel<ST>), smem, "tc4_wgrad")) return e;
  dim3 grid((unsigned)(w.cchunks * w.ngroups), 1, (unsigned)splits);
  tc4_wgrad_kernel<ST><<<grid, 192, smem, stream>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "tc4_wgrad launch");
  return 0;
}

}  // namespace ub
