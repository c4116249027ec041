/*
 * unetb200.h -- C ABI of the B200-native UNet training hot path (libunetb200.so, sm_100a).
 *
 * The reference (Florescence/UNet-Medical-Image-Contour-Segmentation) has no native layer: its hot
 * path is the set of PyTorch library calls made by unet/unet_parts.py, unet/unet_model.py,
 * utils/dice_score.py and utils/boundary_loss.py.  Each entry point below replaces one of those
 * library calls (cited as reference file:line) on raw device pointers.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated otherwise; nothing is allocated or freed by
 *     the library (the caller owns inputs, outputs, saved tensors and workspaces);
 *   - activations are NHWC with an explicit pixel stride `ld` (in elements, >= C): element
 *     (n,h,w,c) lives at base[((n*H + h)*W + w)*ld + c].  ld > C addresses a channel slice of a
 *     wider buffer (this is how the skip concat of unet_parts.py:95 is fused away);
 *   - `dtype` is UNETB200_F32 or UNETB200_BF16 (storage type of activations / packed weights);
 *     all accumulation is fp32, cross-tile statistics are fp64;
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it and never
 *     synchronises the device;
 *   - return value: 0 on success, negative on error (UNETB200_E_*); unetb200_last_error() returns
 *     a thread-local message.  Entry points are re-entrant (forward is called from the Python main
 *     thread, backward from the autograd engine's device thread).
 */
#ifndef UNETB200_H_
#define UNETB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNETB200_F32 0
#define UNETB200_BF16 1

#define UNETB200_OK 0
#define UNETB200_E_INVALID (-1)   /* bad argument / unsupported shape (Python raises ValueError) */
#define UNETB200_E_CUDA (-2)      /* CUDA runtime / driver error (Python raises RuntimeError)     */
#define UNETB200_E_NOMEM (-3)     /* workspace too small                                           */

#define UNETB200_ALGO_AUTO 0
#define UNETB200_ALGO_SIMT 1      /* CUDA-core implicit GEMM, fp32 FMA (any shape; exactness mode)  */
#define UNETB200_ALGO_TC 2        /* tcgen05 / TMEM / TMA implicit GEMM (bf16, or fp32 read as tf32) */
#define UNETB200_ALGO_PREFER_TC 3 /* TC when the shape fits (also for fp32 -> tf32), SIMT otherwise     */

int unetb200_version(void);
const char* unetb200_last_error(void);
/* host pointers out */
int unetb200_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------------------------
 * Generalised convolution as an implicit GEMM   D[m][n] = sum_{t,c} A[m][(t,c)] * Wp[n][(t,c)]
 *
 *   m  runs over the "M grid" (b, i, j), b < B, i < Hm, j < Wm;
 *   A[m][(t,c)] = x[b, i*in_scale + tap_dy[t] + in_off_y, j*in_scale + tap_dx[t] + in_off_x, c]
 *                 (zero outside [0,Hin) x [0,Win): this is the conv padding);
 *   n = q*Cq + co with q < nquad (1 or 4), Cq = N / nquad; D[m][n] is stored at
 *   y[b, i*out_scale + (q>>1) + out_off_y, j*out_scale + (q&1) + out_off_x, co]  (+ bias[co]).
 *
 * It covers, with different packed weights:
 *   nn.Conv2d 3x3 pad 1 fprop  (unet_parts.py:15,18)      9 taps (kh-1,kw-1), scales 1
 *   its dgrad (autograd of the same)                      9 taps, rot180 / transposed weights
 *   nn.ConvTranspose2d k2 s2 fprop (unet_parts.py:73)     1 tap, nquad 4, out_scale 2, bias
 *   its dgrad                                             4 taps (a,c), in_scale 2
 *   nn.Conv2d 1x1 (unet_parts.py:103)                     1 tap
 * ------------------------------------------------------------------------------------------- */
typedef struct unetb200_gconv {
  int32_t dtype;              /* storage dtype of x, Wp, y (and gy for wgrad)                       */
  int32_t algo;               /* UNETB200_ALGO_*                                                     */
  int32_t B, Hm, Wm;          /* M grid                                                              */
  int32_t Cin;                /* channels per tap                                                    */
  int32_t ntaps;              /* 1..9                                                                */
  int32_t tap_dy[9], tap_dx[9];
  int32_t in_scale;           /* 1 or 2                                                              */
  int32_t in_off_y, in_off_x;
  int32_t Hin, Win;           /* source grid                                                         */
  int64_t ld_in;              /* source pixel stride, elements                                       */
  int32_t N;                  /* GEMM N = nquad * Cq                                                 */
  int32_t nquad;              /* 1 or 4                                                              */
  int32_t out_scale;          /* 1 or 2                                                              */
  int32_t out_off_y, out_off_x;
  int32_t Hout, Wout;         /* destination grid                                                    */
  int64_t ld_out;             /* destination pixel stride, elements                                  */
} unetb200_gconv_t;           /* HOST struct */

/* y = gconv(x, Wp) (+bias).  `stats` (nullable, nquad == 1 only) = double[2*N], accumulated (+=)
 * with the per-channel sum and sum of squares of the values as stored (i.e. after rounding to
 * `dtype`): the BatchNorm batch statistics of unet_parts.py:16,19 fused into the conv epilogue.
 * Each tile writes its partial sums to `stats_ws` (float[unetb200_gconv_stats_workspace(d)], plain
 * stores) and a second small kernel reduces them in fp64 -- no global atomics on the hot path.
 * Returns the algorithm actually used through *algo_used (host, nullable). */
int64_t unetb200_gconv_stats_workspace(const unetb200_gconv_t* d);   /* number of floats */
int unetb200_gconv_fprop(const unetb200_gconv_t* d, const void* x, const void* wp,
                         const float* bias, void* y, double* stats, float* stats_ws, int* algo_used,
                         void* stream);

/* Inference form of conv3x3 -> BatchNorm2d (running statistics) -> ReLU (unet_parts.py:15-20 under
 * .eval(), evaluate.py:30, predict.py:17): z = relu(gconv(x, Wp) * scale[n] + shift[n]) computed in the
 * epilogue of the tcgen05 kernel, so the activation is written once and the separate BatchNorm pass
 * (4 B per element) disappears.  scale_shift = float[2*N] (scale then shift, 16-byte aligned; rows 2-3
 * of unetb200_bn_eval_coeffs' output).  _supported returns 1 when the fused kernel covers the shape
 * (3x3, stride 1, C_in and N multiples of 64, tcgen05 eligible); otherwise run unetb200_gconv_fprop +
 * unetb200_bn_relu_apply. */
int unetb200_gconv_fprop_affine_relu_supported(const unetb200_gconv_t* d, const void* x, const void* wp,
                                               const void* z);
int unetb200_gconv_fprop_affine_relu(const unetb200_gconv_t* d, const void* x, const void* wp,
                                     const float* scale_shift, void* z, void* stream);

/* The same with MaxPool2d(2) of the activation as a second output (Down under .eval(): unet_parts.py:26-37 reads the
 * DoubleConv output the kernel just produced): pooled[b][i][j][n] = max over the 2x2 window of z, floor semantics
 * ([B][Hm/2][Wm/2] pixels, pixel stride ld_pooled elements, bf16).  The separate pooling pass (2.5 B per element)
 * disappears.  _supported: the CTA-pair tcgen05 kernel covers the shape (bf16, C_in and N multiples of 64); otherwise run
 * unetb200_gconv_fprop_affine_relu + unetb200_maxpool2_fwd. */
int unetb200_gconv_fprop_affine_relu_pool_supported(const unetb200_gconv_t* d, const void* x, const void* wp,
                                                    const void* z, const void* pooled, int64_t ld_pooled);
int unetb200_gconv_fprop_affine_relu_pool(const unetb200_gconv_t* d, const void* x, const void* wp,
                                          const float* scale_shift, void* z, void* pooled, int64_t ld_pooled,
                                          void* stream);

/* The last conv of the network in inference, fused with OutConv (unet_model.py:25,37; unet_parts.py:100-106):
 * logits[p][k] = sum_c relu(gconv(x, Wp)[p][c] * scale[c] + shift[c]) * oc_w[k][c] + oc_b[k], the activation rounded
 * to `dtype` before the 1x1 conv like the stand-alone kernels; the 64-channel activation is never written.  The
 * descriptor's destination fields are ignored (logits are packed [B][Hm][Wm][ncls]).  _supported: bf16, N = 64,
 * n_classes <= 8, the CTA-pair kernel covers the shape. */
int unetb200_gconv_fprop_affine_relu_outconv_supported(const unetb200_gconv_t* d, const void* x, const void* wp,
                                                       int ncls);
int unetb200_gconv_fprop_affine_relu_outconv(const unetb200_gconv_t* d, const void* x, const void* wp,
                                             const float* scale_shift, const float* oc_w, const float* oc_b,
                                             void* logits, int ncls, void* stream);

/* Data gradient of conv3x3 (autograd of unet_parts.py:18) fused with the reduction pass of the BatchNorm2d + ReLU
 * backward of the layer below it (unet_parts.py:16-17; inside a DoubleConv the second conv's input IS that layer's
 * activation z = relu(bn(yprev))): gx = gconv(g, Wp_dgrad) is written as by unetb200_gconv_fprop, and the epilogue
 * -- which holds the rounded gx tile anyway -- also reads the matching yprev tile and accumulates
 *   sums[0][c] += sum gx*mask,  sums[1][c] += sum gx*mask*xhat,   mask = (yprev*scale + shift > 0),
 *   xhat = (yprev - mean)*invstd        (exactly unetb200_bn_relu_bwd_reduce on the stored gx; `sums` zeroed by the caller)
 * so that pass (one more read of gx and yprev, 4 B per element) is not run.  coefs = float[4][N]: mean, invstd, scale,
 * shift (unetb200_bn_finalize's outputs, contiguous).  ws = float[unetb200_gconv_stats_workspace(d)].  _supported
 * returns 1 when the fused tcgen05 kernel covers the shape; otherwise run gconv_fprop + bn_relu_bwd_reduce. */
int unetb200_gconv_dgrad_bnbwd_supported(const unetb200_gconv_t* d, const void* g, const void* wp, const void* gx);
int unetb200_gconv_dgrad_bnbwd(const unetb200_gconv_t* d, const void* g, const void* wp, void* gx, const void* yprev,
                               int64_t ld_yprev, const float* coefs, double* sums, float* ws, void* stream);

/* Weight gradient of the same generalised conv:
 *   dWp[(t,c)][n] = sum_m A[m][(t,c)] * G[m][n],  G[m][n] = gy at the destination of (m,n).
 * The reduction over m is split `splits` ways; partial s is written (not accumulated) to
 * partials + s*K*N floats, K = ntaps*Cin.  unetb200_gconv_wgrad_plan returns the split count the
 * chosen algorithm wants (host out-params) so the caller can size `partials`. */
int unetb200_gconv_wgrad_plan(const unetb200_gconv_t* d, int* splits, int* algo_used);
int unetb200_gconv_wgrad(const unetb200_gconv_t* d, const void* x, const void* gy, float* partials,
                         int splits, void* stream);
/* dst[t*st + c*sc + q*sq + co*sn] (=|+=) sum_s partials[s][(t,c)][n], n = q*Cq + co: reduces the
 * splits and scatters into the parameter's own layout (OIHW for Conv2d, IOHW for ConvTranspose2d),
 * deterministic. */
int unetb200_wgrad_reduce(const float* partials, int splits, int ntaps, int Cin, int N, int Cq,
                          float* dst, int64_t st, int64_t sc, int64_t sq, int64_t sn, int accumulate,
                          void* stream);

/* The same for a whole list of layers in ONE launch (a backward pass produces ~22 weight gradients; their split
 * reductions are small and launch bound one by one).  Jobs must not alias: two jobs writing the same dst (an
 * accumulate chain) belong in separate calls. */
typedef struct unetb200_reduce_job {
  const float* partials;
  float* dst;
  int64_t st, sc, sq, sn;
  int32_t splits, ntaps, Cin, N, Cq, accumulate;
} unetb200_reduce_job_t;
int unetb200_wgrad_reduce_multi(const unetb200_reduce_job_t* jobs, int njobs, void* stream);

/* dst[i0][i1][i2] = cast(src[off + i0*s0 + i1*s1 + i2*s2]) (strides may be negative): packs an fp32
 * parameter (OIHW / IOHW) into the K-major [N][(t,c)] operand layout of gconv, any tap order. */
int unetb200_pack_weights(const float* src, void* dst, int dst_dtype, int64_t n0, int64_t n1,
                          int64_t n2, int64_t s0, int64_t s1, int64_t s2, int64_t off, void* stream);
/* The same for a whole list of parameters in ONE launch (the weights of a network change together, at the
 * optimizer step: train.py:159): job j packs src -> dst exactly like unetb200_pack_weights.  All jobs share
 * dst_dtype. */
typedef struct unetb200_pack_job {
  const float* src;
  void* dst;
  int64_t n0, n1, n2;
  int64_t s0, s1, s2, off;
} unetb200_pack_job_t;
int unetb200_pack_weights_multi(const unetb200_pack_job_t* jobs, int njobs, int dst_dtype, void* stream);

/* fp32 exactness mode on the tensor cores ("3xTF32", BASELINE.json configs[2]): x = hi + lo with hi = x rounded
 * to TF32.  out[p][0:C | C:2C | 2C:3C] = [hi | lo | hi] (pattern 0: left operand -- activations, output
 * gradients) or [hi | hi | lo] (pattern 1: right operand -- packed weights, p = (n, tap)), so that the ordinary
 * gconv kernels compute hi*hi + lo*hi + hi*lo as one convolution over 3*C input channels (fp32 accumulation;
 * the result is within ~2^-22 of the fp32 product sum the reference's nn.Conv2d computes on the CPU). */
int unetb200_split_tf32(const float* x, int64_t ld_x, float* out, int64_t npix, int C, int pattern,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * BatchNorm2d + ReLU (+ MaxPool2d) -- unet_parts.py:16-17,19-20,32.  Memory-bound, vectorised.
 * ------------------------------------------------------------------------------------------- */
/* stats = double[2*C] (sum, sumsq) over `count` values per channel.  Writes save_mean,
 * save_invstd (biased variance, eps inside the sqrt), scale = gamma*invstd, shift = beta -
 * mean*scale, and (if non-null) running_mean/var with `momentum` and the unbiased variance. */
int unetb200_bn_finalize(const double* stats, int64_t count, const float* gamma, const float* beta,
                         float eps, float momentum, float* running_mean, float* running_var,
                         float* save_mean, float* save_invstd, float* scale, float* shift, int C,
                         void* stream);
/* The same, and num_batches_tracked[0] += 1 (int64, nullable) from the same launch: nn.BatchNorm2d's step counter
 * without an elementwise kernel of its own. */
int unetb200_bn_finalize_track(const double* stats, int64_t count, const float* gamma, const float* beta,
                               float eps, float momentum, float* running_mean, float* running_var,
                               float* save_mean, float* save_invstd, float* scale, float* shift,
                               int64_t* num_batches_tracked, int C, void* stream);
/* eval mode: scale/shift from the running statistics */
int unetb200_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                            const float* running_var, float eps, float* scale, float* shift,
                            float* save_mean, float* save_invstd, int C, void* stream);
/* z = relu(y*scale + shift); if pooled != NULL also pooled = maxpool2x2(z) (floor mode). */
int unetb200_bn_relu_apply(const void* y, int64_t ld_y, const float* scale, const float* shift,
                           void* z, int64_t ld_z, void* pooled, int64_t ld_p, int dtype, int B,
                           int H, int W, int C, void* stream);
int unetb200_maxpool2_fwd(const void* x, int64_t ld_x, void* p, int64_t ld_p, int dtype, int B,
                          int H, int W, int C, void* stream);
/* gx (=|+=) scatter of gp to the FIRST maximum of each 2x2 window in row-major order (ATen's tie
 * rule); positions outside any window (odd H/W) get 0. */
int unetb200_maxpool2_bwd(const void* x, int64_t ld_x, const void* gp, int64_t ld_gp, void* gx,
                          int64_t ld_gx, int accumulate, int dtype, int B, int H, int W, int C,
                          void* stream);
/* The accumulating form of unetb200_maxpool2_bwd (gx += scatter of gp) fused with the reduction pass of the
 * BatchNorm2d + ReLU backward of the layer that produced x = relu(bn(y)): an encoder stage's output feeds the pool
 * and the skip connection (unet_model.py:28-36), its gradient is final only after this call and the BatchNorm
 * backward reads it next, so  sums[0][c] += sum gx*mask, sums[1][c] += sum gx*mask*xhat  (gx as stored; `sums`
 * zeroed by the caller; see unetb200_bn_relu_bwd_reduce) are made here with one extra read of y. */
int unetb200_maxpool2_bwd_bnreduce(const void* x, int64_t ld_x, const void* gp, int64_t ld_gp, void* gx,
                                   int64_t ld_gx, const void* y, int64_t ld_y, const float* scale,
                                   const float* shift, const float* mean, const float* invstd, double* sums,
                                   int dtype, int B, int H, int W, int C, void* stream);
/* g = gz * (y*scale+shift > 0);  sums[0][c] += sum g,  sums[1][c] += sum g*xhat,
 * xhat = (y-mean)*invstd.  `sums` must be zeroed by the caller. */
int unetb200_bn_relu_bwd_reduce(const void* gz, int64_t ld_gz, const void* y, int64_t ld_y,
                                const float* scale, const float* shift, const float* mean,
                                const float* invstd, double* sums, int dtype, int B, int H, int W,
                                int C, void* stream);
/* dgamma = sums[1], dbeta = sums[0]; coef[0][c] = mean(g), coef[1][c] = mean(g*xhat)
 * (both 0 when `training` == 0: eval-mode BN has no batch-statistics term). */
int unetb200_bn_bwd_finalize(const double* sums, int64_t count, int training, float* dgamma,
                             float* dbeta, float* coef, int C, void* stream);
/* gy = scale * (g - coef0 - xhat*coef1) */
int unetb200_bn_relu_bwd_apply(const void* gz, int64_t ld_gz, const void* y, int64_t ld_y,
                               const float* scale, const float* shift, const float* mean,
                               const float* invstd, const float* coef, void* gy, int64_t ld_gy,
                               int dtype, int B, int H, int W, int C, void* stream);

/* ---------------------------------------------------------------------------------------------
 * nn.SyncBatchNorm: BatchNorm statistics synchronised over the GPUs of one node (2..16 ranks).
 * ------------------------------------------------------------------------------------------- */
/* A peer group is the exception to "the caller owns memory" (like an NCCL communicator): the library
 * allocates each rank's exchange buffer, exports it with CUDA IPC and maps every peer's buffer; the
 * exchange kernels move data between GPUs by stores only.  Setup, per rank, on the group's device:
 *   1. unetb200_bn_peer_group_create -> ipc_handle (UNETB200_IPC_HANDLE_BYTES) and the PCI bus id
 *      (UNETB200_BUS_ID_BYTES, NUL-terminated) of this rank's buffer;
 *   2. the caller gathers every rank's handle and bus id (rank order, concatenated);
 *   3. unetb200_bn_peer_group_open checks cudaDeviceCanAccessPeer for every peer and maps its
 *      buffer; UNETB200_E_INVALID when a peer's GPU is not visible or not reachable by peer access.
 * destroy frees this rank's side; call it only after every rank's last exchange has completed
 * (device synchronise + a barrier of the group).  Exchanges of one group must be stream-ordered
 * (one stream at a time) and every rank must issue them in the same order. */
#define UNETB200_IPC_HANDLE_BYTES 64
#define UNETB200_BUS_ID_BYTES 32
typedef struct unetb200_bn_peer_group_s unetb200_bn_peer_group_t;
int unetb200_bn_peer_group_create(int rank, int world, int max_channels, void* ipc_handle, char* bus_id,
                                  unetb200_bn_peer_group_t** out);
int unetb200_bn_peer_group_open(unetb200_bn_peer_group_t* g, const void* ipc_handles, const char* bus_ids);
int unetb200_bn_peer_group_destroy(unetb200_bn_peer_group_t* g);
/* Host read of the group's timeout word: *missing_rank = -1 while no exchange has timed out, else the
 * rank whose contribution an exchange waited for in vain (30 s, %globaltimer) and *epoch = that
 * exchange's epoch.  A timed-out exchange writes no outputs; the group is then unusable. */
int unetb200_bn_peer_group_status(const unetb200_bn_peer_group_t* g, int64_t* missing_rank, int64_t* epoch);
/* unetb200_bn_finalize_track on the GLOBAL statistics: one single-CTA launch pushes this rank's
 * stats[2*C] and `count` to every rank, waits for all of theirs, sums them in rank order in fp64
 * (bit-identical results on every rank: coefficients, running statistics with the unbiased variance
 * over the global count) and finalizes. */
int unetb200_bn_sync_finalize(unetb200_bn_peer_group_t* g, const double* stats, int64_t count,
                              const float* gamma, const float* beta, float eps, float momentum,
                              float* running_mean, float* running_var, float* save_mean,
                              float* save_invstd, float* scale, float* shift,
                              int64_t* num_batches_tracked, int C, void* stream);
/* unetb200_bn_bwd_finalize (training) with coef = GLOBAL sums / GLOBAL count; dgamma = sums[1] and
 * dbeta = sums[0] stay this rank's own (the data-parallel gradient mean averages them). */
int unetb200_bn_sync_bwd_finalize(unetb200_bn_peer_group_t* g, const double* sums, int64_t count,
                                  float* dgamma, float* dbeta, float* coef, int C, void* stream);

/* ---------------------------------------------------------------------------------------------
 * nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) -- unet_parts.py:70, and the
 * F.pad placement of unet_parts.py:85-88 (output written at (off_y, off_x) of an Hout x Wout grid).
 * ------------------------------------------------------------------------------------------- */
int unetb200_upsample2x_fwd(const void* x, int64_t ld_x, void* y, int64_t ld_y, int dtype, int B,
                            int h, int w, int C, int Hout, int Wout, int off_y, int off_x,
                            void* stream);
int unetb200_upsample2x_bwd(const void* gy, int64_t ld_gy, void* gx, int64_t ld_gx, int dtype,
                            int B, int h, int w, int C, int Hout, int Wout, int off_y, int off_x,
                            void* stream);

/* ---------------------------------------------------------------------------------------------
 * layout / dtype plumbing
 * ------------------------------------------------------------------------------------------- */
/* dst NHWC(ld_dst) <- src with arbitrary element strides (sn, sc, sh, sw), with dtype cast */
int unetb200_gather_nhwc(const void* src, int src_dtype, int64_t sn, int64_t sc, int64_t sh,
                         int64_t sw, void* dst, int dst_dtype, int64_t ld_dst, int B, int C, int H,
                         int W, void* stream);
/* dst[p*ld_dst + c] = cast(src[p*ld_src + c]) for p < npix, c < C (channel-slice copy) */
int unetb200_copy_channels(const void* src, int src_dtype, int64_t ld_src, void* dst, int dst_dtype,
                           int64_t ld_dst, int64_t npix, int C, void* stream);
/* zero a channel slice */
int unetb200_zero_channels(void* dst, int dtype, int64_t ld_dst, int64_t npix, int C, void* stream);
/* out[c] = sum_p g[p*ld + c]   (bias gradient of ConvTranspose2d); acc = double[C] workspace */
int unetb200_channel_sum(const void* g, int dtype, int64_t ld, int64_t npix, int C, double* acc,
                         float* out, void* stream);
/* dst[i] = (float)src[i]: hands per-channel fp64 sums made by a conv epilogue (the `stats` of unetb200_gconv_fprop run
 * as a dgrad: column sums of the gradient it writes) to an fp32 parameter gradient -- the ConvTranspose2d bias
 * gradient then needs no pass of its own over the concat gradient. */
int unetb200_f64_to_f32(const double* src, float* dst, int n, void* stream);
/* a += b on NHWC channel slices (skip-gradient accumulation) */
int unetb200_add_channels(void* a, int64_t ld_a, const void* b, int64_t ld_b, int dtype,
                          int64_t npix, int C, void* stream);

/* ---------------------------------------------------------------------------------------------
 * OutConv: 1x1 conv with bias to n_classes <= 8 channels -- unet_parts.py:103.  Memory-bound.
 * logits are NHWC [npix][ncls] of `dtype`; w, bias, dw, dbias are fp32 in the parameter layout.
 * ------------------------------------------------------------------------------------------- */
int unetb200_outconv_fwd(const void* x, int64_t ld_x, const float* w, const float* bias,
                         void* logits, int dtype, int64_t npix, int C, int ncls, void* stream);
/* gx = glogits . w ; dw, dbias (overwritten).  workspace: float[outconv_bwd_workspace] */
int64_t unetb200_outconv_bwd_workspace(int64_t npix, int C, int ncls);
int unetb200_outconv_bwd(const void* x, int64_t ld_x, const float* w, const void* glogits,
                         void* gx, int64_t ld_gx, float* dw, float* dbias, float* workspace,
                         int dtype, int64_t npix, int C, int ncls, void* stream);
/* The same, fused with the reduction pass of the BatchNorm2d + ReLU backward of the stage below (the OutConv input
 * is x = relu(bn(yprev)) of the last DoubleConv, unet_model.py:25,37): additionally
 *   sums[0][c] += sum gx*mask, sums[1][c] += sum gx*mask*xhat   (gx as stored; see unetb200_gconv_dgrad_bnbwd)
 * with coefs = float[4][C] (mean, invstd, scale, shift) and `sums` = double[2*C] zeroed by the caller.  _supported
 * returns 1 when the vectorised kernel covers the shape (C % 8 == 0, C/8 a power of two <= 32, 16-byte aligned rows). */
int unetb200_outconv_bwd_bnbwd_supported(const void* x, int64_t ld_x, const void* gx, int64_t ld_gx,
                                         const void* yprev, int64_t ld_yprev, int dtype, int C, int ncls);
int unetb200_outconv_bwd_bnbwd(const void* x, int64_t ld_x, const float* w, const void* glogits, void* gx,
                               int64_t ld_gx, float* dw, float* dbias, float* workspace, const void* yprev,
                               int64_t ld_yprev, const float* coefs, double* sums, int dtype, int64_t npix, int C,
                               int ncls, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SpatialAttention gate of UNet_SA -- unet_parts.py:39-60 (module) and :91-92 (x2 = x2 * attention(x2)):
 *   stats[p] = (mean_c x[p][c], max_c x[p][c]);  gate[p] = sigmoid(conv7x7(stats)[p]) (2 -> 1 channels, padding 3,
 *   no bias; w = float[2][7][7]);  out[p][c] = x[p][c] * gate[p].
 * stats = float[npix][2] and gate = float[npix] are outputs of the forward call and inputs of the backward call,
 * which returns dx (gradient of x through all three uses: the product, the mean and the max -- first maximum on
 * ties, like torch.max) and dw = float[98].  Rounding points under `dtype` = bf16 follow the reference under
 * autocast (statistics, conv output, gate and product each stored in bf16).  Memory-bound.
 * ------------------------------------------------------------------------------------------- */
int unetb200_sa_forward(const void* x, int64_t ld_x, const float* w, float* stats, float* gate, void* out,
                        int64_t ld_out, int dtype, int B, int H, int W, int C, void* stream);
int64_t unetb200_sa_backward_workspace(int B, int H, int W);   /* number of floats */
int unetb200_sa_backward(const void* g, int64_t ld_g, const void* x, int64_t ld_x, const float* w,
                         const float* stats, const float* gate, void* dx, int64_t ld_dx, float* dw,
                         float* workspace, int dtype, int B, int H, int W, int C, void* stream);

/* ---------------------------------------------------------------------------------------------
 * losses
 * ------------------------------------------------------------------------------------------- */
/* Fused criterion of train.py:137-142: CrossEntropyLoss(logits, target) +
 * dice_loss(softmax(logits), one_hot(target), multiclass=True) (dice_score.py:5-36: one global
 * ratio).  logits NHWC [npix][C] (`dtype`), target int64[npix].
 *   acc   : double[4] workspace (zeroed by the callee)
 *   out   : float[4] = {ce + dice_loss, ce, dice_loss, dice_coeff}
 *   coefs : float[4] saved for backward                                                        */
int unetb200_ce_dice_fwd(const void* logits, int dtype, const int64_t* target, int64_t npix, int C,
                         float epsilon, double* acc, float* out, float* coefs, void* stream);
/* glogits = gscale[0] * d(ce + dice_loss)/dlogits  (gscale: device float, upstream gradient) */
int unetb200_ce_dice_bwd(const void* logits, int dtype, const int64_t* target, int64_t npix, int C,
                         const float* coefs, const float* gscale, void* glogits, void* stream);

/* Fused criterion of the binary branch, train.py:118-134 (n_classes == 1), without its boundary term:
 * BCEWithLogitsLoss(x, t) + dice_loss(sigmoid(x), t) (dice_score.py:5-25, reduce_batch_first=True on the
 * 3-D input: one global ratio, sets == 0 -> inter).  BCE uses the logit itself (stable form
 * max(x,0) - x t + log1p(exp(-|x|))), the dice term the sigmoid rounded to `dtype` (autocast: bf16 logits
 * give bf16 probabilities).  logits [npix] of `dtype` (UNETB200_F32 / UNETB200_BF16) in the same element
 * order as target [npix] of `tgt_dtype` (UNETB200_F32, UNETB200_I64 or UNETB200_U8), whose VALUE is used
 * (soft targets and un-remapped class index 2 included).  Deterministic: per-block partials in a fixed order.
 *   work  : unetb200_bce_dice_work_bytes(npix) bytes; every slot is written by the call, no zeroing needed
 *   out   : float[4] = {bce + dice_loss, bce, dice_loss, dice_coeff}
 *   coefs : float[4] saved for backward                                                        */
int64_t unetb200_bce_dice_work_bytes(int64_t npix);
int unetb200_bce_dice_fwd(const void* logits, int dtype, const void* target, int tgt_dtype, int64_t npix,
                          float epsilon, void* work, float* out, float* coefs, void* stream);
/* glogits [npix] of `dtype` = gscale[0] * d(bce + dice_loss)/dlogits (train.py:118-134); fp32 arithmetic,
 * rounded once at the store */
int unetb200_bce_dice_bwd(const void* logits, int dtype, const void* target, int tgt_dtype, int64_t npix,
                          const float* coefs, const float* gscale, void* glogits, void* stream);

/* dice_coeff (dice_score.py:5-25) on fp32 contiguous input/target viewed as [G][L]: per group
 * inter = 2*sum(x*t), sets = sum x + sum t, sets==0 -> inter, dice = (inter+eps)/(sets+eps);
 * out[0] = mean over groups.  acc: double[3*G] workspace.  saved: float[2*G] for backward. */
int unetb200_dice_fwd(const float* x, const float* t, int64_t G, int64_t L, float epsilon,
                      double* acc, float* out, float* saved, void* stream);
/* gx = gscale[0] * d(mean dice)/dx */
int unetb200_dice_bwd(const float* x, const float* t, int64_t G, int64_t L, float epsilon,
                      const float* saved, const float* gscale, float* gx, void* stream);

/* boundary_loss (boundary_loss.py:5-118) as one integer-count pass + a scalar finalize; no host
 * synchronisation (the reference's .min()/.max()/.any() syncs disappear).  pred is addressed as
 * pred[b*sb + h*sh + w*sw] (elements of pred_dtype; the caller has already selected channel 1 /
 * squeezed, boundary_loss.py:20-25); target likewise (tgt_dtype: UNETB200_F32, or 2 = int64).
 *   work : int64[16] + float[2] workspace (zeroed by the callee), see boundary.cu
 *   out  : float[1] loss                                                                         */
#define UNETB200_I64 2
int unetb200_boundary_loss(const void* pred, int pred_dtype, int64_t sb, int64_t sh, int64_t sw,
                           const void* target, int tgt_dtype, int64_t tb, int64_t th, int64_t tw,
                           int B, int H, int W, int edge_width, float edge_weight, float smooth,
                           void* work, float* out, void* stream);
int64_t unetb200_boundary_work_bytes(void);

/* ---------------------------------------------------------------------------------------------
 * Optimizer side of the step -- train.py:80-84 (RMSprop with momentum), :157 (clip_grad_norm_), :158.
 * Multi-tensor: `w`, `g`, `sq`, `mom` are HOST arrays of `ntensors` DEVICE pointers (fp32, contiguous storage of
 * `numel[i]` elements each; any dense layout, all four of a tensor in the same element order).
 * ------------------------------------------------------------------------------------------- */
/* *out (device double) = sum_i sum(g_i^2): the squared total 2-norm clip_grad_norm_ computes. */
int unetb200_grad_sqnorm(float* const* grads, const int64_t* numel, int ntensors, double* out, void* stream);
/* torch.optim.RMSprop (centered=False) update of every tensor in one pass.  sumsq != NULL: gradients are first
 * scaled by min(1, max_norm / (sqrt(*sumsq) + 1e-6)) (clip_grad_norm_), and written back when
 * write_clipped_grad != 0.  mom == NULL iff momentum == 0. */
int unetb200_rmsprop_step(float* const* w, float* const* g, float* const* sq, float* const* mom,
                          const int64_t* numel, int ntensors, const double* sumsq, float max_norm, float lr,
                          float alpha, float eps, float weight_decay, float momentum, int write_clipped_grad,
                          void* stream);
/* GradScaler and LR schedules inside a captured step, train.py:154-159 (scale(loss).backward(), unscale_,
 * clip_grad_norm_, step, update).  Every value that changes between replays is read from DEVICE memory.
 * One read pass: *sumsq = sum_i sum((g_i * inv_scale)^2) (the order of unetb200_grad_sqnorm), and
 * *found_inf = 1.0f if any element of any g_i is non-finite (isfinite per element; accumulated into, never
 * cleared, as torch's found_inf).  inv_scale NULL means 1; sumsq NULL skips the norm (check only); found_inf NULL
 * skips the check. */
int unetb200_grad_sqnorm_amp(float* const* grads, const int64_t* numel, int ntensors, const float* inv_scale,
                             double* sumsq, float* found_inf, void* stream);
/* unetb200_rmsprop_step with *lr read on the device, g multiplied by *inv_scale (NULL: 1) before the clip
 * coefficient, whose norm is that of the unscaled gradients.  found_inf != NULL and *found_inf != 0: nothing is
 * stored (w, sq, mom, g and step unchanged, as when GradScaler skips optimizer.step()).  Otherwise each step[i]
 * (fp32 0-dim) is incremented, and write_clipped_grad stores the unscaled, clipped gradient. */
int unetb200_rmsprop_step_amp(float* const* w, float* const* g, float* const* sq, float* const* mom,
                              float* const* step, const int64_t* numel, int ntensors, const double* sumsq,
                              float max_norm, const float* lr, const float* inv_scale, const float* found_inf,
                              float alpha, float eps, float weight_decay, float momentum, int write_clipped_grad,
                              void* stream);

/* ---------------------------------------------------------------------------------------------
 * Callers either side of the step (SURVEY.md section 8(f) N1, N3): evaluate / predict tail and the
 * uint8 input pipeline.  Byte / index work: results are exact.
 * ------------------------------------------------------------------------------------------- */
#define UNETB200_U8 3
/* evaluate.py:111-117 (mode 0: pred = argmax over classes == cls, true = target == cls) and
 * evaluate.py:56-66 (mode 1, C == 1: pred = sigmoid(logit) > 0.5 with the sigmoid rounded to `dtype`,
 * true = floor(target / 2) which must be 0 or 1), followed by dice_coeff(pred, true,
 * reduce_batch_first=False) (dice_score.py:5-25; per image, mean over the batch).
 * logits element (b,c,h,w) lives at logits[b*sb + c*sc + h*sh + w*sw]; target is contiguous [B][H][W]
 * (tgt_dtype UNETB200_F32 or UNETB200_I64) or NULL (prediction only).
 *   pred_out : NULL, or contiguous [B][H][W] of pred_dtype (UNETB200_I64 / UNETB200_U8): the argmax
 *              index (mode 0) or the 0/1 prediction (mode 1)
 *   counts   : int64[B][4] = {sum pred*true, sum pred, sum true, #targets outside {0,1} (mode 1)};
 *              zeroed by the callee
 *   dice_out : NULL, or float[1] = mean dice (NaN when mode 1 saw an invalid target: the reference
 *              raises AssertionError)                                                          */
int unetb200_eval_counts(const void* logits, int dtype, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                         const void* target, int tgt_dtype, int B, int C, int H, int W, int cls, int mode,
                         void* pred_out, int pred_dtype, int64_t* counts, float epsilon, float* dice_out,
                         void* stream);
/* predict.py:26-27: F.interpolate(logits, (H, W), mode='bilinear') (align_corners=False, result rounded
 * to `dtype` like ATen's output tensor) followed by argmax(dim=1) (first maximum).  logits [B][C][h][w]
 * by strides as above; out contiguous [B][H][W] of out_dtype (UNETB200_I64 / UNETB200_U8).      */
int unetb200_resize_argmax(const void* logits, int dtype, int64_t sb, int64_t sc, int64_t sh, int64_t sw, int B,
                           int C, int h, int w, int H, int W, void* out, int out_dtype, void* stream);
/* data_loading.py:65-89 (BasicDataset.preprocess, scale == 1) + :91-98 (rotation augmentation) for a
 * batch of equally sized uint8 images already in device memory.
 *   src   : uint8 [B][H][W][C] (numpy.asarray of the PIL image; C <= 4)
 *   rot   : NULL, or device int32[B]: quarter turns counter-clockwise (PIL Image.rotate(90*k,
 *           expand=True) == numpy.rot90(a, k)); `transposed` != 0 says every k is odd on a non-square
 *           image, i.e. the output is [W][H] (the caller checks the parity on the host)
 *   dst   : float [B][Ho][Wo][C] = channels_last storage of the logical [B, C, Ho, Wo] batch:
 *           float32(v) / 255 when the image holds any value > 1 (data_loading.py:86-87), else float32(v)
 *   flags : device int32[B] workspace (per-image "any value > 1"), zeroed by the callee          */
int unetb200_preprocess_image_u8(const uint8_t* src, int B, int H, int W, int C, const int32_t* rot, int transposed,
                                 float* dst, int32_t* flags, void* stream);
/* mask branch of preprocess (data_loading.py:73-79): gray level -> class index, 255 -> 2, 128 -> 1,
 * anything else 0 (lut == NULL) or lut[v] (device int64[256]); same rotation; dst int64 [B][Ho][Wo]
 * (what .long() makes of it at data_loading.py:132).                                            */
int unetb200_preprocess_mask_u8(const uint8_t* src, int B, int H, int W, const int32_t* rot, int transposed,
                                const int64_t* lut, int64_t* dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNETB200_H_ */
