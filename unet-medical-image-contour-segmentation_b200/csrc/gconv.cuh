// Device-side view of unetb200_gconv_t and the engines of the generalised convolution: each engine's shape check,
// split count and launcher.  gconv.cu routes a descriptor to one of them.
#pragma once
#include "common.cuh"

namespace ub {

struct GconvDev {
  int B, Hm, Wm, Cin, ntaps;
  int tap_dy[9], tap_dx[9];
  int in_scale, in_off_y, in_off_x, Hin, Win;
  long long ld_in;
  int N, nquad, Cq, out_scale, out_off_y, out_off_x, Hout, Wout;
  long long ld_out;
  long long M;   // B*Hm*Wm
  int K;         // ntaps*Cin
};

// Split count for a split-K grid of `tiles` work items per split on `slots` one-per-SM execution slots (SMs, or SM
// pairs for cluster kernels): these kernels hold a whole SM each, so the grid runs in waves and a grid of 2.03
// waves costs 3.  Returns the smallest split count (<= smax) whose last wave is (nearly) full, preferring about
// two waves.
inline int pick_splits(long long tiles, int slots, long long smax) {
  if (tiles < 1) tiles = 1;
  if (smax < 1) smax = 1;
  long long lim = (4LL * slots + tiles - 1) / tiles;     // never more than ~4 waves of splits
  if (lim > smax) lim = smax;
  if (lim > 512) lim = 512;
  if (lim < 1) lim = 1;
  double best = -1.0;
  long long pick = 1;
  for (long long s = 1; s <= lim; ++s) {
    const long long ctas = tiles * s;
    const long long waves = (ctas + slots - 1) / slots;
    const double eff = (double)ctas / (double)(waves * slots);
    // prefer fuller waves; among equals, more splits (more of the machine busy) -- eff is maximal at exact multiples
    if (eff > best + 1e-9 || (eff > best - 0.005 && ctas <= 2LL * slots)) { best = eff > best ? eff : best; pick = s; }
  }
  return (int)pick;
}

// CUDA-core implicit GEMM for any shape, the arithmetic of the exact-fp32 mode (conv_simt.cu)
long long simt_fprop_tiles(const GconvDev& g);
int simt_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, const float* bias, void* y,
               double* stats, float* stats_ws, cudaStream_t s);
int simt_wgrad_splits(const GconvDev& g);
int simt_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
               cudaStream_t s);
int launch_stats_reduce(const float* ws, long long ntiles, int C2, double* stats, cudaStream_t s);

// tcgen05 engines, the layout conditions every kernel generation shares (tc_host.cu)
bool tc_common_ok(const unetb200_gconv_t* d);

// persistent tcgen05 engine, second generation (conv_tc2.cu)
int tc2_fprop_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y);
long long tc2_stats_workspace(const unetb200_gconv_t* d);
int tc2_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, const float* bias, void* y,
              double* stats, float* stats_ws, cudaStream_t stream);

int tc2_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int tc2_wgrad_splits(const unetb200_gconv_t* d);
int tc2_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
              cudaStream_t stream);

// CTA-pair tcgen05 engine for the 3x3 convolutions, third generation (conv_tc3.cu)
int tc3_fprop_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const float* bias, const void* y);
long long tc3_stats_workspace(const unetb200_gconv_t* d);
struct Tc3OutConv {            // OutConv fused into the inference epilogue of the last conv (EPI_AFFINE_OUT)
  const float* w;              // [ncls][64]
  const float* b;              // [ncls] or null
  void* logits;                // [B][Hm][Wm][ncls], storage dtype
  int ncls;
};
int tc3_affine_outconv_supported(const unetb200_gconv_t* d, int ncls);
int tc3_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, void* y, double* stats,
              float* stats_ws, cudaStream_t stream, const float* affine = nullptr, const void* yprev = nullptr,
              long long ld_yprev = 0, const float* bnc = nullptr, const Tc3OutConv* oc = nullptr, void* pooled = nullptr,
              long long ld_pool = 0);
int tc3_bnbwd_supported(const unetb200_gconv_t* d);

int tc3_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int tc3_wgrad_splits(const unetb200_gconv_t* d);
int tc3_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
              cudaStream_t stream);

// N-stacked wgrad for the narrow 3x3 layers, fourth generation (conv_tc4.cu)
int tc4_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int tc4_wgrad_splits(const unetb200_gconv_t* d);
int tc4_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials, int splits,
              cudaStream_t stream);

// first layer (C_in <= 4, N = 64, bf16) on the tensor cores: thread-built im2col rows (conv_first_tc.cu)
int first_tc_supported(const unetb200_gconv_t* d, const void* y);
long long first_tc_stats_rows(const unetb200_gconv_t* d);
int first_tc_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, void* y, double* stats, float* stats_ws,
                   const float* affine, cudaStream_t s);

// 3x3 convolutions with narrow channel counts (C_in, C_out <= 64, bf16) on the tensor cores (conv_narrow.cu)
int narrow_tc_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y);
long long narrow_tc_stats_rows(const unetb200_gconv_t* d);
int narrow_tc_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, void* y, double* stats, float* stats_ws,
                    const float* affine, cudaStream_t s);

// TMA-staged tcgen05 kernels for 16 / 32 / 64 channels on either side (conv_halo.cu)
int halo_fprop_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y);
long long halo_stats_rows(const unetb200_gconv_t* d);
int halo_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, void* y, double* stats, float* stats_ws,
               const float* affine, cudaStream_t s, const void* yprev = nullptr, long long ld_yprev = 0,
               const float* bnc = nullptr, void* pooled = nullptr, long long ld_pool = 0);
int halo_bnbwd_supported(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx);
int halo_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int halo_wgrad_splits(const unetb200_gconv_t* d);
int halo_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s);
// first layer of the light variants: C_in = 1 -> 8 / 16 / 32 channels, CUDA cores (conv_first_narrow.cu)
int first_narrow_supported(const unetb200_gconv_t* d, const void* y);
long long first_narrow_rows(const unetb200_gconv_t* d);
int first_narrow_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, void* y, double* stats, float* stats_ws,
                       const float* affine, cudaStream_t s);
int first_narrow_wgrad_splits(const unetb200_gconv_t* d);
int first_narrow_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s);
// exact-fp32 wgrad of the narrow 3x3 layers on the CUDA cores (conv_simt_narrow.cu)
int fprop_narrow_f32_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y);
long long fprop_narrow_f32_rows(const unetb200_gconv_t* d);
int fprop_narrow_f32(const unetb200_gconv_t* d, const void* x, const void* wp, void* y, double* stats, float* stats_ws,
                     cudaStream_t s);
int wgrad_narrow_f32_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int wgrad_narrow_f32_splits(const unetb200_gconv_t* d);
int wgrad_narrow_f32(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s);
// ConvTranspose2d(k=2, s=2) with narrow channel counts (conv_halo_t.cu)
int halo_t_fprop_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* y);
int halo_t_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, const float* bias, void* y, cudaStream_t s);
int halo_t_dgrad_supported(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx);
int halo_t_dgrad(const unetb200_gconv_t* d, const void* g, const void* wp, void* gx, cudaStream_t s);
int halo_t_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int halo_t_wgrad_splits(const unetb200_gconv_t* d);
int halo_t_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s);
int narrow_wgrad_supported(const unetb200_gconv_t* d, const void* x, const void* gy);
int narrow_wgrad_splits(const unetb200_gconv_t* d);
int narrow_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits, cudaStream_t s);

// first-layer (C_in <= 4) CUDA-core kernels (conv_first.cu)
int first_fprop_supported(const unetb200_gconv_t* d, const void* y);
long long first_fprop_tiles(const unetb200_gconv_t* d);
int first_fprop(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* wp, void* y, double* stats,
                float* stats_ws, cudaStream_t s);
int first_wgrad_supported(const unetb200_gconv_t* d, const void* gy);
int first_wgrad_splits(const unetb200_gconv_t* d);
int first_wgrad(const unetb200_gconv_t* d, const GconvDev& g, const void* x, const void* gy, float* partials,
                int splits, cudaStream_t s);

}  // namespace ub
