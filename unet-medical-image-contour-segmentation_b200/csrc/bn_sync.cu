// Synchronised BatchNorm (nn.SyncBatchNorm) across the GPUs of one node: the per-rank fp64 statistics are exchanged by
// kernel stores into every peer's exchange buffer over NVLink (CUDA IPC mappings), so the exchange is an ordinary
// kernel launch and may sit inside a captured CUDA graph -- unlike an NCCL call on this stack (DESIGN.md section 5).
//
// Exchange buffer of a rank (allocated and owned by the library, exported with CUDA IPC, written by the peers):
//   flag[kMaxRanks]  u64   flag[r] = last epoch whose contribution rank r has delivered here
//   inbox[2][W][S]   f64   inbox[slot][r][0 .. 2C] = rank r's sums (2C values) and its element count
//
// Epochs and slots.  Each exchange kernel reads the rank's device-side epoch counter e, advances it to e + 1 and uses
// slot (e + 1) & 1, so graph replays pair up across ranks without any host involvement.  Two slots are enough because
// (1) every exchange is a barrier: no rank leaves exchange e before every rank has entered it, and (2) all exchanges
// of a rank are stream-ordered one after another (the peer group is used from one stream at a time: forward, backward,
// graph capture and replay all enqueue on the rank's current stream).  A peer can therefore be at most one epoch
// ahead, and the slot it writes then is the one this rank finished reading in the exchange before the current one.
#include <cuda_runtime.h>

#include <cstring>
#include <new>

#include "common.cuh"

namespace {

constexpr int kMaxRanks = 16;                     // one NVLink node; multi-node groups are not supported
constexpr int kFlagBytes = kMaxRanks * 8;
constexpr int kThreads = 256;
constexpr unsigned long long kTimeoutNs = 30ull * 1000 * 1000 * 1000;

struct SyncArgs {
  char* buf[kMaxRanks];                           // every rank's exchange buffer as mapped here (own one included)
  unsigned long long* epoch;                      // this rank's epoch counter (device memory, not exported)
  volatile long long* err;                        // mapped pinned host words: missing rank + 1, epoch
  int rank, world, stride;                        // stride: doubles per inbox row (>= 2 C + 1)
};

__device__ __forceinline__ unsigned long long* flag_of(char* buf, int r) {
  return reinterpret_cast<unsigned long long*>(buf) + r;
}
__device__ __forceinline__ double* inbox_of(char* buf, int slot, int r, const SyncArgs& a) {
  return reinterpret_cast<double*>(buf + kFlagBytes) + ((size_t)slot * a.world + r) * a.stride;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Pushes (local[0 .. 2C), count) to every rank, waits for every rank's contribution of the same epoch and returns the
// slot holding them, or -1 after a timeout (the missing rank and the epoch are then in a.err; the kernel returns
// without writing its outputs and the host raises at its next entry: no trap, the context stays usable).
__device__ int exchange(const SyncArgs& a, const double* __restrict__ local, int C, double count) {
  __shared__ int s_missing;
  const unsigned long long e = *a.epoch + 1;
  const int slot = (int)(e & 1);
  const int nv = 2 * C + 1;
  if (threadIdx.x == 0) s_missing = -1;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const double v = i < 2 * C ? local[i] : count;
    for (int p = 0; p < a.world; ++p) inbox_of(a.buf[p], slot, a.rank, a)[i] = v;
  }
  __threadfence_system();                         // this thread's stores, before the flags below (system scope)
  __syncthreads();
  if (threadIdx.x < a.world) st_release_sys(flag_of(a.buf[threadIdx.x], a.rank), e);
  if (threadIdx.x < a.world) {
    const unsigned long long* f = flag_of(a.buf[a.rank], threadIdx.x);
    const unsigned long long t0 = globaltimer();
    unsigned ns = 32;
    while (ld_acquire_sys(f) < e) {
      if (globaltimer() - t0 > kTimeoutNs) {
        s_missing = threadIdx.x;
        break;
      }
      __nanosleep(ns);
      ns = ns < 1024 ? 2 * ns : 1024;
    }
  }
  __syncthreads();                                // the acquires above order every thread's reads below
  if (s_missing >= 0) {
    if (threadIdx.x == 0) {
      a.err[1] = (long long)e;
      __threadfence_system();
      a.err[0] = s_missing + 1;
      __threadfence_system();
    }
    return -1;
  }
  return slot;
}

// global sum of value i over the ranks, in rank order: every rank gets bit-identical results
__device__ __forceinline__ double rank_sum(const SyncArgs& a, int slot, int i) {
  double s = 0.0;
  for (int r = 0; r < a.world; ++r) s += __ldcg(inbox_of(a.buf[a.rank], slot, r, a) + i);
  return s;
}

__global__ void __launch_bounds__(kThreads)
bn_sync_finalize_kernel(SyncArgs a, const double* __restrict__ stats, double count, const float* __restrict__ gamma,
                        const float* __restrict__ beta, float eps, float momentum, float* running_mean,
                        float* running_var, float* save_mean, float* save_invstd, float* scale, float* shift, int C,
                        long long* num_batches_tracked) {
  const int slot = exchange(a, stats, C, count);
  if (slot < 0) return;
  const double n = rank_sum(a, slot, 2 * C);
  const double inv_count = 1.0 / n, unbias = n > 1.0 ? n / (n - 1.0) : 1.0;
  // as bn_finalize_kernel, on the global sums
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double mean = rank_sum(a, slot, c) * inv_count;
    double var = rank_sum(a, slot, C + c) * inv_count - mean * mean;
    if (var < 0) var = 0;
    float invstd = (float)(1.0 / sqrt(var + (double)eps));
    float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    float sc = g * invstd;
    save_mean[c] = (float)mean;
    save_invstd[c] = invstd;
    scale[c] = sc;
    shift[c] = b - (float)mean * sc;
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)(var * unbias);
  }
  if (threadIdx.x == 0) {
    if (num_batches_tracked) *num_batches_tracked += 1;
    *a.epoch += 1;                                // read again only by the next exchange kernel on this stream
  }
}

__global__ void __launch_bounds__(kThreads)
bn_sync_bwd_finalize_kernel(SyncArgs a, const double* __restrict__ sums, double count, float* dgamma, float* dbeta,
                            float* coef, int C) {
  const int slot = exchange(a, sums, C, count);
  if (slot < 0) return;
  const double inv_count = 1.0 / rank_sum(a, slot, 2 * C);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    // dgamma / dbeta stay the LOCAL sums (the gradient all-reduce averages them, as for torch's SyncBatchNorm)
    if (dbeta) dbeta[c] = (float)sums[c];
    if (dgamma) dgamma[c] = (float)sums[C + c];
    coef[c] = (float)(rank_sum(a, slot, c) * inv_count);
    coef[C + c] = (float)(rank_sum(a, slot, C + c) * inv_count);
  }
  if (threadIdx.x == 0) *a.epoch += 1;
}

}  // namespace

struct unetb200_bn_peer_group_s {
  int device = -1, rank = 0, world = 0, max_c = 0, stride = 0;
  char* local = nullptr;                          // own exchange buffer
  char* buf[kMaxRanks] = {};                      // buf[rank] = local, buf[r] = rank r's buffer opened through IPC
  unsigned long long* epoch = nullptr;
  long long* err_host = nullptr;                  // cudaHostAllocMapped: [missing rank + 1, epoch]
  long long* err_dev = nullptr;
};

namespace {

size_t buffer_bytes(const unetb200_bn_peer_group_t* g) {
  return kFlagBytes + sizeof(double) * 2 * (size_t)g->world * g->stride;
}

void release(unetb200_bn_peer_group_t* g) {
  for (int r = 0; r < g->world; ++r)
    if (r != g->rank && g->buf[r]) cudaIpcCloseMemHandle(g->buf[r]);
  if (g->local) cudaFree(g->local);
  if (g->epoch) cudaFree(g->epoch);
  if (g->err_host) cudaFreeHost(g->err_host);
  delete g;
}

struct DeviceGuard {                              // current device = the group's device, restored on exit
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int launch_ready(const unetb200_bn_peer_group_t* g, int C, const char* what) {
  UB_CHECK_ARG(g && g->buf[g->rank] && C > 0 && C <= g->max_c, "%s: C=%d (peer group capacity %d channels)", what, C,
               g ? g->max_c : 0);
  for (int r = 0; r < g->world; ++r) UB_CHECK_ARG(g->buf[r], "%s: peer group not opened", what);
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return ub::cuda_fail(e, "cudaGetDevice");
  UB_CHECK_ARG(dev == g->device, "%s: current device %d, peer group of device %d", what, dev, g->device);
  return 0;
}

SyncArgs args_of(const unetb200_bn_peer_group_t* g) {
  SyncArgs a{};
  for (int r = 0; r < g->world; ++r) a.buf[r] = g->buf[r];
  a.epoch = g->epoch;
  a.err = g->err_dev;
  a.rank = g->rank;
  a.world = g->world;
  a.stride = g->stride;
  return a;
}

}  // namespace

extern "C" {

int unetb200_bn_peer_group_create(int rank, int world, int max_channels, void* ipc_handle, char* bus_id,
                                  unetb200_bn_peer_group_t** out) {
  UB_CHECK_ARG(out && ipc_handle && bus_id && world >= 2 && world <= kMaxRanks && rank >= 0 && rank < world &&
                   max_channels > 0,
               "bn_peer_group_create: rank %d of %d (2..%d ranks), %d channels", rank, world, kMaxRanks, max_channels);
  *out = nullptr;
  auto* g = new (std::nothrow) unetb200_bn_peer_group_t;
  if (!g) {
    ub::set_error("bn_peer_group_create: out of host memory");
    return UNETB200_E_NOMEM;
  }
  g->rank = rank;
  g->world = world;
  g->max_c = max_channels;
  g->stride = (2 * max_channels + 1 + 1) / 2 * 2;  // rows 16-byte aligned
  cudaError_t e = cudaGetDevice(&g->device);
  const char* what = "cudaGetDevice";
  if (e == cudaSuccess) {
    what = "cudaMalloc (exchange buffer)";
    e = cudaMalloc(&g->local, buffer_bytes(g));
  }
  if (e == cudaSuccess) {
    what = "cudaMemset (exchange buffer)";
    e = cudaMemset(g->local, 0, buffer_bytes(g));
  }
  if (e == cudaSuccess) {
    what = "cudaMalloc (epoch)";
    e = cudaMalloc(&g->epoch, sizeof(unsigned long long));
  }
  if (e == cudaSuccess) {
    what = "cudaMemset (epoch)";
    e = cudaMemset(g->epoch, 0, sizeof(unsigned long long));
  }
  if (e == cudaSuccess) {
    what = "cudaHostAlloc (timeout word)";
    e = cudaHostAlloc(&g->err_host, 2 * sizeof(long long), cudaHostAllocMapped);
  }
  if (e == cudaSuccess) {
    g->err_host[0] = g->err_host[1] = 0;
    what = "cudaHostGetDevicePointer";
    e = cudaHostGetDevicePointer(&g->err_dev, g->err_host, 0);
  }
  if (e == cudaSuccess) {
    what = "cudaIpcGetMemHandle";
    e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle), g->local);
  }
  if (e == cudaSuccess) {
    what = "cudaDeviceGetPCIBusId";
    e = cudaDeviceGetPCIBusId(bus_id, UNETB200_BUS_ID_BYTES, g->device);
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();   // the zero fills are complete before any peer can write
  if (e != cudaSuccess) {
    release(g);
    return ub::cuda_fail(e, what);
  }
  g->buf[rank] = g->local;
  *out = g;
  return 0;
}

int unetb200_bn_peer_group_open(unetb200_bn_peer_group_t* g, const void* ipc_handles, const char* bus_ids) {
  UB_CHECK_ARG(g && ipc_handles && bus_ids, "bn_peer_group_open: bad args");
  DeviceGuard guard(g->device);
  for (int r = 0; r < g->world; ++r) {
    if (r == g->rank) continue;
    int dev = -1, can = 0;
    if (cudaDeviceGetByPCIBusId(&dev, bus_ids + (size_t)r * UNETB200_BUS_ID_BYTES) != cudaSuccess) {
      cudaGetLastError();
      ub::set_error("bn_peer_group_open: the GPU of rank %d (%s) is not visible from rank %d (multi-node groups and "
                    "restricted CUDA_VISIBLE_DEVICES are not supported)", r, bus_ids + (size_t)r * UNETB200_BUS_ID_BYTES,
                    g->rank);
      return UNETB200_E_INVALID;
    }
    if (dev != g->device && (cudaDeviceCanAccessPeer(&can, g->device, dev) != cudaSuccess || !can)) {
      cudaGetLastError();
      ub::set_error("bn_peer_group_open: device %d of rank %d cannot access device %d of rank %d by peer access", g->device,
                    g->rank, dev, r);
      return UNETB200_E_INVALID;
    }
  }
  for (int r = 0; r < g->world; ++r) {
    if (r == g->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(ipc_handles) + (size_t)r * sizeof(h), sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; ++q)
        if (q != g->rank && g->buf[q]) {
          cudaIpcCloseMemHandle(g->buf[q]);
          g->buf[q] = nullptr;
        }
      return ub::cuda_fail(e, "bn_peer_group_open: cudaIpcOpenMemHandle");
    }
    g->buf[r] = static_cast<char*>(p);
  }
  return 0;
}

int unetb200_bn_peer_group_destroy(unetb200_bn_peer_group_t* g) {
  if (!g) return 0;
  DeviceGuard guard(g->device);
  release(g);
  return 0;
}

int unetb200_bn_peer_group_status(const unetb200_bn_peer_group_t* g, int64_t* missing_rank, int64_t* epoch) {
  UB_CHECK_ARG(g && missing_rank && epoch, "bn_peer_group_status: bad args");
  const volatile long long* w = g->err_host;
  *missing_rank = w[0] - 1;
  *epoch = w[1];
  return 0;
}

int unetb200_bn_sync_finalize(unetb200_bn_peer_group_t* g, const double* stats, int64_t count, const float* gamma,
                              const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                              float* save_mean, float* save_invstd, float* scale, float* shift,
                              int64_t* num_batches_tracked, int C, void* stream) {
  if (int rc = launch_ready(g, C, "bn_sync_finalize")) return rc;
  UB_CHECK_ARG(stats && save_mean && save_invstd && scale && shift && count > 0, "bn_sync_finalize: bad args");
  bn_sync_finalize_kernel<<<1, kThreads, 0, (cudaStream_t)stream>>>(
      args_of(g), stats, (double)count, gamma, beta, eps, momentum, running_mean, running_var, save_mean, save_invstd,
      scale, shift, C, reinterpret_cast<long long*>(num_batches_tracked));
  UB_LAUNCH_CHECK("bn_sync_finalize");
  return 0;
}

int unetb200_bn_sync_bwd_finalize(unetb200_bn_peer_group_t* g, const double* sums, int64_t count, float* dgamma,
                                  float* dbeta, float* coef, int C, void* stream) {
  if (int rc = launch_ready(g, C, "bn_sync_bwd_finalize")) return rc;
  UB_CHECK_ARG(sums && coef && count > 0, "bn_sync_bwd_finalize: bad args");
  bn_sync_bwd_finalize_kernel<<<1, kThreads, 0, (cudaStream_t)stream>>>(args_of(g), sums, (double)count, dgamma, dbeta,
                                                                        coef, C);
  UB_LAUNCH_CHECK("bn_sync_bwd_finalize");
  return 0;
}

}  // extern "C"
