// C-ABI entry points of the generalised convolution (unetb200_gconv_*) and the one place that decides which engine
// runs a descriptor.  Every operation has one route: an entry point validates the descriptor, asks the route and
// launches the engine it names, and a _supported query is "the route names an engine".  A route only orders the
// engines' own X_supported checks; what a kernel accepts stays with its engine.
#include <cstdlib>
#include <cstring>

#include "gconv.cuh"

namespace ub {
namespace {

// named after their launchers in gconv.cuh (halo_t_*, first_narrow_*, halo_*, narrow_tc_* / narrow_wgrad, ...)
enum class Engine { NONE, HALO_T, HALO_T_DGRAD, FIRST_NARROW, HALO, NARROW_TC, TC2, TC3, TC4, FIRST_TC, FIRST,
                    NARROW_F32, SIMT };
struct Route { Engine engine; int algo; };   // the engine for a descriptor and the algo_used reported for it

}  // namespace

static int gconv_validate(const unetb200_gconv_t* d, GconvDev* o) {
  UB_CHECK_ARG(d != nullptr, "gconv: null descriptor");
  UB_CHECK_ARG(d->dtype == UNETB200_F32 || d->dtype == UNETB200_BF16, "gconv: dtype %d", d->dtype);
  UB_CHECK_ARG(d->B > 0 && d->Hm > 0 && d->Wm > 0 && d->Cin > 0, "gconv: bad M grid / Cin");
  UB_CHECK_ARG(d->ntaps >= 1 && d->ntaps <= 9, "gconv: ntaps %d", d->ntaps);
  UB_CHECK_ARG(d->in_scale == 1 || d->in_scale == 2, "gconv: in_scale %d", d->in_scale);
  UB_CHECK_ARG(d->out_scale == 1 || d->out_scale == 2, "gconv: out_scale %d", d->out_scale);
  UB_CHECK_ARG(d->nquad == 1 || d->nquad == 4, "gconv: nquad %d", d->nquad);
  UB_CHECK_ARG(d->N > 0 && d->N % d->nquad == 0, "gconv: N %d not divisible by nquad %d", d->N, d->nquad);
  UB_CHECK_ARG(d->nquad == 1 || d->out_scale == 2, "gconv: nquad 4 needs out_scale 2");
  UB_CHECK_ARG(d->Hin > 0 && d->Win > 0 && d->Hout > 0 && d->Wout > 0, "gconv: bad grids");
  UB_CHECK_ARG(d->ld_in >= d->Cin && d->ld_out >= d->N / d->nquad, "gconv: pixel stride smaller than channels");
  UB_CHECK_ARG(d->out_off_y >= 0 && d->out_off_x >= 0 &&
                   (d->Hm - 1) * d->out_scale + (d->nquad == 4 ? 1 : 0) + d->out_off_y < d->Hout &&
                   (d->Wm - 1) * d->out_scale + (d->nquad == 4 ? 1 : 0) + d->out_off_x < d->Wout,
               "gconv: output does not fit the destination grid");
  o->B = d->B; o->Hm = d->Hm; o->Wm = d->Wm; o->Cin = d->Cin; o->ntaps = d->ntaps;
  for (int t = 0; t < 9; ++t) { o->tap_dy[t] = d->tap_dy[t]; o->tap_dx[t] = d->tap_dx[t]; }
  o->in_scale = d->in_scale; o->in_off_y = d->in_off_y; o->in_off_x = d->in_off_x;
  o->Hin = d->Hin; o->Win = d->Win; o->ld_in = d->ld_in;
  o->N = d->N; o->nquad = d->nquad; o->Cq = d->N / d->nquad; o->out_scale = d->out_scale;
  o->out_off_y = d->out_off_y; o->out_off_x = d->out_off_x; o->Hout = d->Hout; o->Wout = d->Wout;
  o->ld_out = d->ld_out;
  o->M = (long long)d->B * d->Hm * d->Wm;
  o->K = d->ntaps * d->Cin;
  return 0;
}

// Forward convolution (and every dgrad, which is one).  The specialised engines first, then AUTO / PREFER_TC resolve
// to the tcgen05 engines when one covers the shape (fp32 only under PREFER_TC: it defaults to exact FMA), else to the
// CUDA cores.  An explicit ALGO_TC on a shape no tcgen05 engine covers, and an unknown algo, route to NONE.
static Route route_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, const float* bias, const void* y,
                         bool has_stats) {
  int algo = d->algo;
  const bool tc_allowed = algo != UNETB200_ALGO_SIMT;
  if (tc_allowed && !has_stats && halo_t_fprop_supported(d, x, wp, y)) return {Engine::HALO_T, UNETB200_ALGO_TC};
  if (tc_allowed && !has_stats && !bias && halo_t_dgrad_supported(d, x, wp, y))
    return {Engine::HALO_T_DGRAD, UNETB200_ALGO_TC};
  if (!bias && first_narrow_supported(d, y)) return {Engine::FIRST_NARROW, UNETB200_ALGO_SIMT};
  if (tc_allowed && !bias && halo_fprop_supported(d, x, wp, y)) return {Engine::HALO, UNETB200_ALGO_TC};
  if (tc_allowed && !bias && narrow_tc_supported(d, x, wp, y)) return {Engine::NARROW_TC, UNETB200_ALGO_TC};
  const bool tc = tc_common_ok(d) && (tc3_fprop_supported(d, x, wp, nullptr, y) || tc2_fprop_supported(d, x, wp, y));
  if (algo == UNETB200_ALGO_AUTO || algo == UNETB200_ALGO_PREFER_TC) algo = tc ? UNETB200_ALGO_TC : UNETB200_ALGO_SIMT;
  if (algo == UNETB200_ALGO_TC) {
    if (!tc) return {Engine::NONE, algo};
    return {tc3_fprop_supported(d, x, wp, bias, y) ? Engine::TC3 : Engine::TC2, algo};
  }
  if (algo != UNETB200_ALGO_SIMT) return {Engine::NONE, algo};
  // the first layer reports ALGO_SIMT on either core type
  if (!bias && first_fprop_supported(d, y))
    return {first_tc_supported(d, y) && aligned16(wp) ? Engine::FIRST_TC : Engine::FIRST, algo};
  if (!bias && fprop_narrow_f32_supported(d, x, wp, y)) return {Engine::NARROW_F32, algo};
  return {Engine::SIMT, algo};
}

// conv3x3 -> BatchNorm(eval) -> ReLU with the normalisation folded into the epilogue (inference only)
static Engine route_affine(const unetb200_gconv_t* d, const void* x, const void* wp, const void* z) {
  static const bool off = getenv("UNETB200_NO_BN_FOLD") != nullptr;
  static const bool wide = getenv("UNETB200_TC3_MAXBN") && atoi(getenv("UNETB200_TC3_MAXBN")) >= 256;
  if (off || d->algo == UNETB200_ALGO_SIMT) return Engine::NONE;
  if (first_tc_supported(d, z) && aligned16(wp)) return Engine::FIRST_TC;
  if (first_narrow_supported(d, z)) return Engine::FIRST_NARROW;
  if (halo_fprop_supported(d, x, wp, z)) return Engine::HALO;
  if (narrow_tc_supported(d, x, wp, z)) return Engine::NARROW_TC;
  if (d->dtype == UNETB200_BF16 && d->N % 256 == 0 && wide) return Engine::NONE;   // no affine epilogue at BN = 256
  return tc_common_ok(d) && tc3_fprop_supported(d, x, wp, nullptr, z) ? Engine::TC3 : Engine::NONE;
}

// the same with MaxPool2d(2) of the activation as a second output (Down: unet_parts.py:26-37 under .eval()): the
// TMA-staged narrow kernel and the CTA-pair kernel only -- a warp's 4 x 8 pixel patch of the epilogue holds whole
// 2 x 2 windows
static Engine route_affine_pool(const unetb200_gconv_t* d, const void* x, const void* wp, const void* z,
                                const void* pooled, int64_t ld_pooled) {
  static const bool off = getenv("UNETB200_NO_POOL_FOLD") != nullptr;
  if (off || d->dtype != UNETB200_BF16 || !pooled || (ld_pooled & 1) || (reinterpret_cast<uintptr_t>(pooled) & 3) ||
      d->Hm < 2 || d->Wm < 2)
    return Engine::NONE;
  const Engine e = route_affine(d, x, wp, z);
  return e == Engine::HALO || e == Engine::TC3 ? e : Engine::NONE;
}

// dgrad of a 3x3 convolution + the reduction pass of the BatchNorm/ReLU backward of the layer that produced its input
static Engine route_dgrad_bnbwd(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx) {
  static const bool off = getenv("UNETB200_NO_BNBWD_FUSE") != nullptr;
  if (off || d->algo == UNETB200_ALGO_SIMT) return Engine::NONE;
  if (halo_bnbwd_supported(d, g, wp, gx)) return Engine::HALO;
  return tc_common_ok(d) && tc3_fprop_supported(d, g, wp, nullptr, gx) && tc3_bnbwd_supported(d) ? Engine::TC3
                                                                                                   : Engine::NONE;
}

// Weight gradient, from the shape alone (the plan has no pointers; the launch checks the chosen engine's alignment).
// Among the tcgen05 generations the N-stacked kernel takes the 3x3 layers the CTA-pair kernel does not cover (that one
// needs C_in >= 256 and N % 128 == 0), or every layer it covers with UNETB200_TC4W=all (A/B runs).
static Route route_wgrad(const unetb200_gconv_t* d) {
  static const bool tc4_all = [] {
    const char* e = getenv("UNETB200_TC4W");
    return e && !strcmp(e, "all");
  }();
  int algo = d->algo;
  if (first_narrow_supported(d, nullptr)) return {Engine::FIRST_NARROW, UNETB200_ALGO_SIMT};
  if (algo != UNETB200_ALGO_SIMT) {
    if (halo_wgrad_supported(d, nullptr, nullptr)) return {Engine::HALO, UNETB200_ALGO_TC};
    if (halo_t_wgrad_supported(d, nullptr, nullptr)) return {Engine::HALO_T, UNETB200_ALGO_TC};
    if (narrow_wgrad_supported(d, nullptr, nullptr)) return {Engine::NARROW_TC, UNETB200_ALGO_TC};
  }
  const bool tc4 = tc4_wgrad_supported(d, nullptr, nullptr), tc3 = tc3_wgrad_supported(d, nullptr, nullptr);
  const bool tc = tc_common_ok(d) && d->in_scale == 1 && (tc4 || tc3 || tc2_wgrad_supported(d, nullptr, nullptr));
  if (algo == UNETB200_ALGO_AUTO || algo == UNETB200_ALGO_PREFER_TC) algo = tc ? UNETB200_ALGO_TC : UNETB200_ALGO_SIMT;
  if (algo == UNETB200_ALGO_TC) {
    if (!tc) return {Engine::NONE, algo};
    if (tc4 && (tc4_all || !tc3)) return {Engine::TC4, algo};
    return {tc3 ? Engine::TC3 : Engine::TC2, algo};
  }
  if (first_wgrad_supported(d, nullptr)) return {Engine::FIRST, algo};
  if (wgrad_narrow_f32_supported(d, nullptr, nullptr)) return {Engine::NARROW_F32, algo};
  return {Engine::SIMT, algo};
}

}  // namespace ub

using namespace ub;

extern "C" {

int64_t unetb200_gconv_stats_workspace(const unetb200_gconv_t* d) {
  GconvDev g;
  if (gconv_validate(d, &g)) return -1;
  // no pointers, so no route: the most any engine writes for the shape ([2][N] floats per row)
  const long long rows[] = {simt_fprop_tiles(g), first_fprop_tiles(d), first_tc_stats_rows(d), narrow_tc_stats_rows(d),
                            halo_stats_rows(d),  first_narrow_rows(d), fprop_narrow_f32_rows(d)};
  long long n = tc2_stats_workspace(d);
  const long long n3 = tc3_stats_workspace(d);
  if (n3 > n) n = n3;
  for (long long r : rows)
    if (r * 2 * g.N > n) n = r * 2 * g.N;
  return n;
}

int unetb200_gconv_fprop(const unetb200_gconv_t* d, const void* x, const void* wp, const float* bias, void* y,
                         double* stats, float* stats_ws, int* algo_used, void* stream) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  UB_CHECK_ARG(x && wp && y, "gconv_fprop: null pointer");
  UB_CHECK_ARG(!stats || (stats_ws && d->nquad == 1), "gconv_fprop: stats need a workspace and nquad == 1");
  if (!stats) stats_ws = nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  const Route r = route_fprop(d, x, wp, bias, y, stats != nullptr);
  if (algo_used) *algo_used = r.algo;
  switch (r.engine) {
    case Engine::HALO_T: return halo_t_fprop(d, x, wp, bias, y, s);
    case Engine::HALO_T_DGRAD: return halo_t_dgrad(d, x, wp, y, s);
    case Engine::FIRST_NARROW: return first_narrow_fprop(d, x, wp, y, stats, stats_ws, nullptr, s);
    case Engine::HALO: return halo_fprop(d, x, wp, y, stats, stats_ws, nullptr, s);
    case Engine::NARROW_TC: return narrow_tc_fprop(d, x, wp, y, stats, stats_ws, nullptr, s);
    case Engine::TC3: return tc3_fprop(d, g, x, wp, y, stats, stats_ws, s);
    case Engine::TC2: return tc2_fprop(d, g, x, wp, bias, y, stats, stats_ws, s);
    case Engine::FIRST_TC: return first_tc_fprop(d, x, wp, y, stats, stats_ws, nullptr, s);
    case Engine::FIRST: return first_fprop(d, g, x, wp, y, stats, stats_ws, s);
    case Engine::NARROW_F32: return fprop_narrow_f32(d, x, wp, y, stats, stats_ws, s);
    case Engine::SIMT: return simt_fprop(d, g, x, wp, bias, y, stats, stats_ws, s);
    default: break;
  }
  UB_CHECK_ARG(r.algo != UNETB200_ALGO_TC, "gconv_fprop: tcgen05 path requested but shape/alignment unsupported");
  set_error("gconv_fprop: unknown algo %d", r.algo);
  return UNETB200_E_INVALID;
}

int unetb200_gconv_fprop_affine_relu_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* z) {
  GconvDev g;
  return !gconv_validate(d, &g) && route_affine(d, x, wp, z) != Engine::NONE;
}

int unetb200_gconv_fprop_affine_relu(const unetb200_gconv_t* d, const void* x, const void* wp, const float* scale_shift,
                                     void* z, void* stream) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  UB_CHECK_ARG(x && wp && z && scale_shift, "gconv_fprop_affine_relu: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  switch (route_affine(d, x, wp, z)) {
    case Engine::FIRST_TC: return first_tc_fprop(d, x, wp, z, nullptr, nullptr, scale_shift, s);
    case Engine::FIRST_NARROW: return first_narrow_fprop(d, x, wp, z, nullptr, nullptr, scale_shift, s);
    case Engine::HALO: return halo_fprop(d, x, wp, z, nullptr, nullptr, scale_shift, s);
    case Engine::NARROW_TC: return narrow_tc_fprop(d, x, wp, z, nullptr, nullptr, scale_shift, s);
    case Engine::TC3: return tc3_fprop(d, g, x, wp, z, nullptr, nullptr, s, scale_shift);
    default: break;
  }
  set_error("gconv_fprop_affine_relu: shape not covered by the fused kernel (query _supported first and run "
            "gconv_fprop + bn_relu_apply instead)");
  return UNETB200_E_INVALID;
}

int unetb200_gconv_fprop_affine_relu_pool_supported(const unetb200_gconv_t* d, const void* x, const void* wp, const void* z,
                                                    const void* pooled, int64_t ld_pooled) {
  GconvDev g;
  return !gconv_validate(d, &g) && route_affine_pool(d, x, wp, z, pooled, ld_pooled) != Engine::NONE;
}

int unetb200_gconv_fprop_affine_relu_pool(const unetb200_gconv_t* d, const void* x, const void* wp, const float* scale_shift,
                                          void* z, void* pooled, int64_t ld_pooled, void* stream) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  UB_CHECK_ARG(x && wp && z && scale_shift && pooled, "gconv_fprop_affine_relu_pool: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  switch (route_affine_pool(d, x, wp, z, pooled, ld_pooled)) {
    case Engine::HALO:
      return halo_fprop(d, x, wp, z, nullptr, nullptr, scale_shift, s, nullptr, 0, nullptr, pooled, (long long)ld_pooled);
    case Engine::TC3:
      return tc3_fprop(d, g, x, wp, z, nullptr, nullptr, s, scale_shift, nullptr, 0, nullptr, nullptr, pooled,
                       (long long)ld_pooled);
    default: break;
  }
  set_error("gconv_fprop_affine_relu_pool: shape not covered (query _supported first and run gconv_fprop_affine_relu + "
            "maxpool2_fwd instead)");
  return UNETB200_E_INVALID;
}

int unetb200_gconv_dgrad_bnbwd_supported(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx) {
  GconvDev gd;
  return !gconv_validate(d, &gd) && route_dgrad_bnbwd(d, g, wp, gx) != Engine::NONE;
}

int unetb200_gconv_dgrad_bnbwd(const unetb200_gconv_t* d, const void* g, const void* wp, void* gx, const void* yprev,
                               int64_t ld_yprev, const float* coefs, double* sums, float* ws, void* stream) {
  GconvDev gd;
  int rc = gconv_validate(d, &gd);
  if (rc) return rc;
  UB_CHECK_ARG(g && wp && gx && yprev && coefs && sums && ws, "gconv_dgrad_bnbwd: null pointer");
  UB_CHECK_ARG(ld_yprev >= d->N, "gconv_dgrad_bnbwd: ld_yprev < N");
  cudaStream_t s = (cudaStream_t)stream;
  switch (route_dgrad_bnbwd(d, g, wp, gx)) {
    case Engine::HALO: return halo_fprop(d, g, wp, gx, sums, ws, nullptr, s, yprev, (long long)ld_yprev, coefs);
    case Engine::TC3: return tc3_fprop(d, gd, g, wp, gx, sums, ws, s, nullptr, yprev, (long long)ld_yprev, coefs);
    default: break;
  }
  set_error("gconv_dgrad_bnbwd: shape not covered by the fused kernel (query _supported first and run gconv_fprop + "
            "bn_relu_bwd_reduce instead)");
  return UNETB200_E_INVALID;
}

// last conv of the network in inference: conv3x3 -> BatchNorm(eval) -> ReLU -> OutConv 1x1 + bias in one kernel
int unetb200_gconv_fprop_affine_relu_outconv_supported(const unetb200_gconv_t* d, const void* x, const void* wp,
                                                       int ncls) {
  GconvDev g;
  if (gconv_validate(d, &g)) return 0;
  static const bool off = getenv("UNETB200_NO_BN_FOLD") != nullptr || getenv("UNETB200_NO_OUTCONV_FOLD") != nullptr;
  if (off || d->algo == UNETB200_ALGO_SIMT || !aligned16(x) || !aligned16(wp)) return 0;
  return tc3_affine_outconv_supported(d, ncls);
}

int unetb200_gconv_fprop_affine_relu_outconv(const unetb200_gconv_t* d, const void* x, const void* wp,
                                             const float* scale_shift, const float* oc_w, const float* oc_b,
                                             void* logits, int ncls, void* stream) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  UB_CHECK_ARG(x && wp && scale_shift && oc_w && logits, "gconv_fprop_affine_relu_outconv: null pointer");
  UB_CHECK_ARG(unetb200_gconv_fprop_affine_relu_outconv_supported(d, x, wp, ncls),
               "gconv_fprop_affine_relu_outconv: shape not covered (query _supported first)");
  Tc3OutConv oc = {oc_w, oc_b, logits, ncls};
  return tc3_fprop(d, g, x, wp, logits, nullptr, nullptr, (cudaStream_t)stream, scale_shift, nullptr, 0, nullptr, &oc);
}

int unetb200_gconv_wgrad_plan(const unetb200_gconv_t* d, int* splits, int* algo_used) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  const Route r = route_wgrad(d);
  UB_CHECK_ARG(r.engine != Engine::NONE, "gconv_wgrad: tcgen05 path requested but shape unsupported");
  if (algo_used) *algo_used = r.algo;
  if (!splits) return 0;
  switch (r.engine) {
    case Engine::FIRST_NARROW: *splits = first_narrow_wgrad_splits(d); break;
    case Engine::HALO: *splits = halo_wgrad_splits(d); break;
    case Engine::HALO_T: *splits = halo_t_wgrad_splits(d); break;
    case Engine::NARROW_TC: *splits = narrow_wgrad_splits(d); break;
    case Engine::TC4: *splits = tc4_wgrad_splits(d); break;
    case Engine::TC3: *splits = tc3_wgrad_splits(d); break;
    case Engine::TC2: *splits = tc2_wgrad_splits(d); break;
    case Engine::FIRST: *splits = first_wgrad_splits(d); break;
    case Engine::NARROW_F32: *splits = wgrad_narrow_f32_splits(d); break;
    default: *splits = simt_wgrad_splits(g); break;
  }
  return 0;
}

int unetb200_gconv_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials, int splits,
                         void* stream) {
  GconvDev g;
  int rc = gconv_validate(d, &g);
  if (rc) return rc;
  UB_CHECK_ARG(x && gy && partials && splits >= 1, "gconv_wgrad: null pointer / bad splits");
  cudaStream_t s = (cudaStream_t)stream;
  // the route saw no pointers: each case checks its engine's alignment and never falls through to another engine
  switch (route_wgrad(d).engine) {
    case Engine::FIRST_NARROW:
      UB_CHECK_ARG(first_narrow_supported(d, gy), "gconv_wgrad: the first-layer kernel needs a 16-byte aligned gradient");
      return first_narrow_wgrad(d, x, gy, partials, splits, s);
    case Engine::HALO:
      UB_CHECK_ARG(halo_wgrad_supported(d, x, gy), "gconv_wgrad: the TMA-staged narrow kernel needs 16-byte aligned operands");
      return halo_wgrad(d, x, gy, partials, splits, s);
    case Engine::HALO_T:
      UB_CHECK_ARG(halo_t_wgrad_supported(d, x, gy), "gconv_wgrad: the TMA-staged narrow kernel needs 16-byte aligned operands");
      return halo_t_wgrad(d, x, gy, partials, splits, s);
    case Engine::NARROW_TC:
      UB_CHECK_ARG(narrow_wgrad_supported(d, x, gy), "gconv_wgrad: the narrow tcgen05 kernel needs 16-byte aligned operands");
      return narrow_wgrad(d, x, gy, partials, splits, s);
    case Engine::TC4: if (tc4_wgrad_supported(d, x, gy)) return tc4_wgrad(d, g, x, gy, partials, splits, s); break;
    case Engine::TC3: if (tc3_wgrad_supported(d, x, gy)) return tc3_wgrad(d, g, x, gy, partials, splits, s); break;
    case Engine::TC2: if (tc2_wgrad_supported(d, x, gy)) return tc2_wgrad(d, g, x, gy, partials, splits, s); break;
    case Engine::FIRST:
      UB_CHECK_ARG(first_wgrad_supported(d, gy) && splits == first_wgrad_splits(d),
                   "gconv_wgrad: first-layer kernel needs 16-byte aligned dY and the planned split count");
      return first_wgrad(d, g, x, gy, partials, splits, s);
    case Engine::NARROW_F32:
      UB_CHECK_ARG(wgrad_narrow_f32_supported(d, x, gy), "gconv_wgrad: the narrow fp32 kernel needs 16-byte aligned operands");
      return wgrad_narrow_f32(d, x, gy, partials, splits, s);
    case Engine::SIMT: return simt_wgrad(d, g, x, gy, partials, splits, s);
    default: break;
  }
  set_error("gconv_wgrad: tcgen05 path requested but shape/alignment unsupported");   // an explicit ALGO_TC, or misaligned
  return UNETB200_E_INVALID;
}

}
