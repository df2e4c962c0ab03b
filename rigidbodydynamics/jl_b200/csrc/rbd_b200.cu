// librbd_b200.so -- C ABI (include/rbd_b200.h) over the sm_100a kernels.
//
// Kernel design (DESIGN.md has the long version):
//   * one THREAD owns one sample; a block is one or more independent warps; there are no block-level barriers;
//   * the grid is persistent: blocks_per_SM x SM_count blocks loop over groups of NT consecutive samples;
//   * inputs / outputs are rows x batch with the batch index fastest, so lane l of a warp touches element b0 + l of a
//     row: every global access of a warp is one fully-used 128-byte line (fp32) / two lines (fp64);
//   * the per-sample working set that must survive between the three passes lives in shared memory, laid out
//     [row][lane] so a warp's access to a row hits 32 distinct banks;
//   * the flattened mechanism is a __grid_constant__ kernel parameter: it is read through the constant bank with a
//     warp-uniform index, i.e. as uniform-register operands, not as per-thread loads.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <set>
#include <string>
#include <type_traits>

#include "../../../include/rbd_b200.h"
#include "rbd_rnea_crba.cuh"
#include "rbd_kin.cuh"
#include "rbd_dual.cuh"
#include "rbd_integrate.cuh"
#include "rbd_tmem.cuh"
#include "rbd_model.h"

using namespace rbd;

// ------------------------------------------------------------------------------------------------------------------
// handle, errors
// ------------------------------------------------------------------------------------------------------------------
#include "rbd_handle.h"

namespace {

thread_local std::string g_err;
thread_local rbd_launch_info g_launch = {0, 0, 0, 0, 0, 0.f, 0};

int fail(int status, const std::string& msg) { g_err = msg; return status; }
int fail_cuda(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return RBD_ECUDA;
}
#define CUDA_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return fail_cuda(e_, #expr); } while (0)

}  // namespace

namespace rbd {
int get_props(DeviceProps& p) {
  static std::mutex mu;
  static DeviceProps cache[64];
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (dev >= 0 && dev < 64 && cache[dev].ok) { p = cache[dev]; return RBD_OK; }
  DeviceProps q;
  q.dev = dev;
  CUDA_TRY(cudaDeviceGetAttribute(&q.sms, cudaDevAttrMultiProcessorCount, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&q.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&q.smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  {  // scratch for slots / external wrenches comes from the stream-ordered pool: keep freed blocks cached in the pool
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  q.ok = true;
  if (dev >= 0 && dev < 64) cache[dev] = q;
  p = q;
  return RBD_OK;
}

int configure_once(const void* kernel, const DeviceProps& p) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({kernel, p.dev})) return RBD_OK;
  cudaFuncAttributes fa{};
  CUDA_TRY(cudaFuncGetAttributes(&fa, kernel));
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p.max_smem_optin - (int)fa.sharedSizeBytes));
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  done.insert({kernel, p.dev});
  return RBD_OK;
}

// The pair gives the Tensor-Memory CTA room in the register file (65536 per SM) by running fewer shared-memory blocks: small
// models are not limited by shared memory, and persistent shared-memory blocks would keep the CTA off the SM until they drain
// the queue.  It only pays when shared memory (not the register file) limits the single kernel's residency, i.e. when the pair
// puts at least 15 % more warps on the SM, and when the batch has enough groups to keep both kernels' warps busy.
int pair_blocks(int sms, int bps, int regs_smem, int regs_tmem, int tm_warps, int64_t ngroups) {
  const int rs = ((regs_smem + 7) / 8) * 8 * 32, rt = ((regs_tmem + 7) / 8) * 8 * 32 * tm_warps;
  if (rt + rs > 65536) return 0;
  const int with_pair = std::max(1, std::min(bps, (65536 - rt) / rs));
  if ((with_pair + tm_warps) * 100 < bps * 115) return 0;
  if (ngroups < (int64_t)(with_pair + tm_warps / 2) * sms) return 0;
  return with_pair;
}
}  // namespace rbd

namespace {

// ------------------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Pull the NEXT group's input lines into L2 while this group is being computed (one 128-byte line per row and warp).
template <class T>
__device__ __forceinline__ void prefetch_rows(const T* base, int rows, int64_t ld, int64_t b0) {
  if (!base) return;
  for (int r = threadIdx.x & 31; r < rows; r += 32) prefetch_l2(base + (int64_t)r * ld + b0);
}

template <class T> struct AbaArgs {
  const T* q; const T* v; const T* tau; const T* wext;
  T* vd; T* qd;
  T* scratch;            // [6 * nb][scratch_ld] body-frame external wrenches (EXT only), one column per resident thread
  int64_t ld, B;
  unsigned long long* counter;   // work queue shared by the two kernels of launch_duo
  int64_t scratch_ld;            // columns of `scratch` (queue kernels)
  int64_t scratch_off;           // first scratch column of the Tensor-Memory kernel's threads (after the shared-memory kernel's)
  const int* gate;               // non-NULL: run only if *gate != 0 (fallback behind the model-specialised kernels, rbd_spec.cpp)
};

// KINDS: compile-time promise about the 1-DoF kinds present (kAllKinds, or 0 = revolute / sin-cos-revolute only).
template <class T, int NT, bool GENERAL, bool EXT, int KINDS>
__global__ void __launch_bounds__(NT, (sizeof(T) == 4 && !GENERAL && !EXT) ? 20 : 1)
aba_kernel(const __grid_constant__ ModelDev<T> M, const AbaArgs<T> a) {
  if (a.gate && *a.gate == 0) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sh = reinterpret_cast<T*>(smem_raw);
  using ST = Stash<T, NT>;
  const int64_t nthreads = (int64_t)gridDim.x * NT;
  const int64_t tid = (int64_t)blockIdx.x * NT + threadIdx.x;
  const ST st{sh + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t gn = g + gridDim.x;
    if (gn < ngroups) {
      const int64_t bn = gn * NT + (threadIdx.x & ~31);
      prefetch_rows(a.q, M.nq, a.ld, bn);
      prefetch_rows(a.v, M.nv, a.ld, bn);
      prefetch_rows(a.tau, M.nv, a.ld, bn);
      if (EXT) prefetch_rows(a.wext, 6 * M.nb, a.ld, bn);
    }
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;     // inactive lanes recompute the last sample, stores are masked
    AbaIO<T, EXT, KINDS> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.tau = {a.tau ? a.tau + bl : nullptr, a.ld};
    io.wext = {EXT ? a.wext + bl : nullptr, a.ld};
    io.vd = {a.vd + bl, a.ld, active};
    io.qd = {a.qd ? a.qd + bl : nullptr, a.ld, active};
    io.ext = {EXT ? a.scratch + tid : nullptr, nthreads};
    if (EXT) ext_wrench_pass(M, io.q, io.wext, io.ext, st, M.slot_base, kSlotRowsAba);
    aba_sample<T, ST, GENERAL>(M, io, st);
  }
}

// Work-queue variants for running the shared-memory kernel and the Tensor-Memory kernel SIDE BY SIDE on every SM (two
// launches on two streams; groups of 32 samples are claimed from one atomic counter, so the kernels balance themselves).
__device__ __forceinline__ int64_t claim_group(unsigned long long* counter) {
  unsigned long long g = 0;
  if ((threadIdx.x & 31) == 0) g = atomicAdd(counter, 1ull);
  return (int64_t)__shfl_sync(0xffffffffu, g, 0);
}
template <class T, class ST, int KINDS, bool EXT>
__device__ __forceinline__ void aba_queue_loop(const ModelDev<T>& M, const AbaArgs<T>& a, const ST& st, int64_t tid) {
  constexpr int NT = 32;
  const int lane = threadIdx.x & 31;
  unsigned long long* counter = a.counter;
  const int64_t ngroups = (a.B + NT - 1) / NT;
  int64_t g = claim_group(counter);
  while (g < ngroups) {
    const int64_t gn = claim_group(counter);
    if (gn < ngroups) {
      const int64_t bn = gn * NT;
      prefetch_rows(a.q, M.nq, a.ld, bn);
      prefetch_rows(a.v, M.nv, a.ld, bn);
      prefetch_rows(a.tau, M.nv, a.ld, bn);
      if (EXT) prefetch_rows(a.wext, 6 * M.nb, a.ld, bn);
    }
    const int64_t b = g * NT + lane;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    AbaIO<T, EXT, KINDS> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.tau = {a.tau ? a.tau + bl : nullptr, a.ld};
    io.wext = {EXT ? a.wext + bl : nullptr, a.ld};
    io.vd = {a.vd + bl, a.ld, active};
    io.qd = {a.qd ? a.qd + bl : nullptr, a.ld, active};
    io.ext = {EXT ? a.scratch + tid : nullptr, a.scratch_ld};
    if (EXT) ext_wrench_pass(M, io.q, io.wext, io.ext, st, M.slot_base, kSlotRowsAba);
    aba_sample<T, ST, false>(M, io, st);
    g = gn;
  }
}
template <class T, int KINDS, bool EXT>
__global__ void __launch_bounds__(32, sizeof(T) == 4 ? 16 : 1) aba_kernel_smem_q(const __grid_constant__ ModelDev<T> M, const AbaArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  aba_queue_loop<T, Stash<T, 32>, KINDS, EXT>(M, a, Stash<T, 32>{reinterpret_cast<T*>(smem_raw) + threadIdx.x},
                                              (int64_t)blockIdx.x * 32 + threadIdx.x);
}
// CTA of NW = 4 or 8 warps over COLS TMEM columns.  Warp w may only touch TMEM lane quadrant w % 4, so warps 0-3 keep their
// stash in the first COLS / (NW / 4) columns and warps 4-7 (same lanes) in the second half: in fp32 (one column per row,
// <= 256 rows) one CTA fills all 512 columns with the working sets of 8 warps; fp64 needs two columns per row, 4 warps.
// Register budget: the CTA shares the SM with the 8 single-warp blocks of aba_kernel_smem_q, 16 warps x 32 x 128 = 64 K.
template <class T, int COLS, int KINDS, int NW, bool EXT>
__global__ void __launch_bounds__(32 * NW, NW == 8 ? 2 : 1)
aba_kernel_tmem_q(const __grid_constant__ ModelDev<T> M, const AbaArgs<T> a) {
  __shared__ uint32_t tm_slot;
  const uint32_t tm_base = tmem_alloc_cta<COLS>(&tm_slot);
  using ST = typename StashTMFor<T>::type;
  const uint32_t w = threadIdx.x >> 5;
  aba_queue_loop<T, ST, KINDS, EXT>(M, a, ST{tm_base + (((w & 3u) * 32u) << 16) + (w >> 2) * (uint32_t)(COLS / (NW / 4))},
                                    a.scratch_off + (int64_t)blockIdx.x * (32 * NW) + threadIdx.x);
  tmem_free_cta<COLS>(tm_base);
}


// dynamics! on Dual{Float64,6} arrays: thread t of the launch owns (sample t / 6, partial direction t % 6).
struct DualArgs {
  const double* q; const double* v; const double* tau;
  double* vd;
  int64_t ld, B;
};
template <int NT, bool GENERAL>
__global__ void __launch_bounds__(NT) aba_dual_kernel(const __grid_constant__ ModelDev<Dual64> M, const DualArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Dual64* sh = reinterpret_cast<Dual64*>(smem_raw);
  const Stash<Dual64, NT> st{sh + threadIdx.x};
  const int64_t total = a.B * 6;
  const int64_t ngroups = (total + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t t = g * NT + threadIdx.x;
    const bool active = t < total;
    const int64_t tl = active ? t : total - 1;
    const int64_t b = tl / 6;
    const int dir = (int)(tl - b * 6);
    AbaIO<Dual64, false> io;
    io.q = {a.q + b * kDualWidth, a.ld, dir};
    io.v = {a.v + b * kDualWidth, a.ld, dir};
    io.tau = {a.tau ? a.tau + b * kDualWidth : nullptr, a.ld, dir};
    io.wext = {nullptr, a.ld, dir};
    io.vd = {a.vd + b * kDualWidth, a.ld, dir, active};
    io.qd = {nullptr, a.ld, dir, active};
    io.ext = {nullptr, 0};
    aba_sample<Dual64, Stash<Dual64, NT>, GENERAL>(M, io, st);
  }
}

// Same evaluation with the stash split between shared memory (value parts) and Tensor Memory (partial parts): one 4-warp CTA/SM.
__global__ void __launch_bounds__(128) aba_dual_kernel_tm(const __grid_constant__ ModelDev<Dual64> M, const DualArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint32_t tm_slot;
  const uint32_t tm_base = tmem_alloc_cta<512>(&tm_slot);
  const StashDualTM st{reinterpret_cast<double*>(smem_raw) + threadIdx.x, tm_base + ((uint32_t)((threadIdx.x >> 5) * 32) << 16)};
  const int64_t total = a.B * 6;
  const int64_t ngroups = (total + 127) / 128;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t t = g * 128 + threadIdx.x;
    const bool active = t < total;
    const int64_t tl = active ? t : total - 1;
    const int64_t b = tl / 6;
    const int dir = (int)(tl - b * 6);
    AbaIO<Dual64, false> io;
    io.q = {a.q + b * kDualWidth, a.ld, dir};
    io.v = {a.v + b * kDualWidth, a.ld, dir};
    io.tau = {a.tau ? a.tau + b * kDualWidth : nullptr, a.ld, dir};
    io.wext = {nullptr, a.ld, dir};
    io.vd = {a.vd + b * kDualWidth, a.ld, dir, active};
    io.qd = {nullptr, a.ld, dir, active};
    io.ext = {nullptr, 0};
    aba_sample<Dual64, StashDualTM, false>(M, io, st);
  }
  tmem_free_cta<512>(tm_base);
}

template <class T> struct RneaArgs {
  const T* q; const T* v; const T* vd; const T* wext;
  T* tau;
  T* scratch;
  int64_t ld, B;
  unsigned long long* counter;
  int64_t scratch_ld, scratch_off;
  const int* gate;               // see AbaArgs
};

template <class T, int NT, bool EXT>
__global__ void __launch_bounds__(NT, sizeof(T) == 4 ? 32 : 1) rnea_kernel(const __grid_constant__ ModelDev<T> M, const RneaArgs<T> a) {
  if (a.gate && *a.gate == 0) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sh = reinterpret_cast<T*>(smem_raw);
  const Stash<T, NT> st{sh + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t gn = g + gridDim.x;
    if (gn < ngroups) {
      const int64_t bn = gn * NT + (threadIdx.x & ~31);
      prefetch_rows(a.q, M.nq, a.ld, bn);
      prefetch_rows(a.v, M.nv, a.ld, bn);
      prefetch_rows(a.vd, M.nv, a.ld, bn);
      if (EXT) prefetch_rows(a.wext, 6 * M.nb, a.ld, bn);
    }
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    RneaIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.vd = {a.vd ? a.vd + bl : nullptr, a.ld};
    io.wext = {EXT ? a.wext + bl : nullptr, a.ld};
    io.tau = {a.tau + bl, a.ld, active};
    io.ext = {EXT ? a.scratch + (int64_t)blockIdx.x * NT + threadIdx.x : nullptr, (int64_t)gridDim.x * NT};
    rnea_sample<T>(M, io, st);
  }
}

// Work-queue variants of the RNEA kernel (no external wrenches): shared-memory blocks + one Tensor-Memory CTA per SM.
template <class T, class ST, bool EXT>
__device__ __forceinline__ void rnea_queue_loop(const ModelDev<T>& M, const RneaArgs<T>& a, const ST& st, int64_t tid) {
  constexpr int NT = 32;
  const int lane = threadIdx.x & 31;
  unsigned long long* counter = a.counter;
  const int64_t ngroups = (a.B + NT - 1) / NT;
  int64_t g = claim_group(counter);
  while (g < ngroups) {
    const int64_t gn = claim_group(counter);
    if (gn < ngroups) {
      const int64_t bn = gn * NT;
      prefetch_rows(a.q, M.nq, a.ld, bn);
      prefetch_rows(a.v, M.nv, a.ld, bn);
      prefetch_rows(a.vd, M.nv, a.ld, bn);
      if (EXT) prefetch_rows(a.wext, 6 * M.nb, a.ld, bn);
    }
    const int64_t b = g * NT + lane;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    RneaIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.vd = {a.vd ? a.vd + bl : nullptr, a.ld};
    io.wext = {EXT ? a.wext + bl : nullptr, a.ld};
    io.tau = {a.tau + bl, a.ld, active};
    io.ext = {EXT ? a.scratch + tid : nullptr, a.scratch_ld};
    rnea_sample<T>(M, io, st);
    g = gn;
  }
}
template <class T, bool EXT>
__global__ void __launch_bounds__(32, sizeof(T) == 4 ? 16 : 1) rnea_kernel_smem_q(const __grid_constant__ ModelDev<T> M,
                                                                                   const RneaArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  rnea_queue_loop<T, Stash<T, 32>, EXT>(M, a, Stash<T, 32>{reinterpret_cast<T*>(smem_raw) + threadIdx.x},
                                        (int64_t)blockIdx.x * 32 + threadIdx.x);
}
template <class T, int COLS, int NW, bool EXT>
__global__ void __launch_bounds__(32 * NW, NW == 8 ? 2 : 1)
rnea_kernel_tmem_q(const __grid_constant__ ModelDev<T> M, const RneaArgs<T> a) {
  __shared__ uint32_t tm_slot;
  const uint32_t tm_base = tmem_alloc_cta<COLS>(&tm_slot);
  using ST = typename StashTMFor<T>::type;
  const uint32_t w = threadIdx.x >> 5;
  rnea_queue_loop<T, ST, EXT>(M, a, ST{tm_base + (((w & 3u) * 32u) << 16) + (w >> 2) * (uint32_t)(COLS / (NW / 4))},
                              a.scratch_off + (int64_t)blockIdx.x * (32 * NW) + threadIdx.x);
  tmem_free_cta<COLS>(tm_base);
}

template <class T> struct CrbaArgs {
  const T* q;
  T* M;
  int64_t ld, B;
  bool lower;
  const int* gate;       // non-NULL: run only if *gate != 0 (fallback behind the model-specialised kernel, see AbaArgs)
};

template <class T, int NT, int KMAX>
__global__ void __launch_bounds__(NT, sizeof(T) == 4 ? (KMAX == 1 ? 28 : 20) : 1) crba_kernel(const __grid_constant__ ModelDev<T> M, const CrbaArgs<T> a) {
  if (a.gate && *a.gate == 0) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sh = reinterpret_cast<T*>(smem_raw);
  const Stash<T, NT> st{sh + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t gn = g + gridDim.x;
    if (gn < ngroups) prefetch_rows(a.q, M.nq, a.ld, gn * NT + (threadIdx.x & ~31));
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    CrbaIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.M = {a.M + bl, a.ld, active};
    io.lower = a.lower;
    crba_sample<T, Stash<T, NT>, KMAX>(M, io, st);
  }
}

template <class T> struct KinArgs {
  const T* q; const T* v;
  T* tr; T* com; T* ke; T* pe; T* mom; T* mrb; T* A; T* J;
  T* scratch;
  int64_t ld, B;
  const int* gate;       // non-NULL: run only if *gate != 0 (fallback behind the model-specialised kernel, see AbaArgs)
};

template <class T, int NT>
__global__ void __launch_bounds__(NT, sizeof(T) == 4 ? 28 : 12) kin_kernel(const __grid_constant__ ModelDev<T> M, const KinArgs<T> a,
                                                  const __grid_constant__ KinDev<T> K) {
  if (a.gate && *a.gate == 0) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sh = reinterpret_cast<T*>(smem_raw);
  const Stash<T, NT> st{sh + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t gn = g + gridDim.x;
    if (gn < ngroups) {
      const int64_t bn = gn * NT + (threadIdx.x & ~31);
      prefetch_rows(a.q, M.nq, a.ld, bn);
      if (a.v) prefetch_rows(a.v, M.nv, a.ld, bn);
    }
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    KinIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v ? a.v + bl : nullptr, a.ld};
    auto out = [&](T* p) { return ColOut<T>{p ? p + bl : nullptr, a.ld, active}; };
    io.tr = out(a.tr); io.com = out(a.com); io.ke = out(a.ke); io.pe = out(a.pe);
    io.mom = out(a.mom); io.mrb = out(a.mrb); io.A = out(a.A); io.J = out(a.J);
    io.poses = {a.scratch ? a.scratch + (int64_t)blockIdx.x * NT + threadIdx.x : nullptr, (int64_t)gridDim.x * NT};
    kin_sample<T>(M, K, io, st);
  }
}

template <class T> struct BodiesArgs {
  const T* q; const T* v; const T* vd; const T* wext;
  T* acc; T* jw;
  int64_t ld, B;
};
template <class T, int NT>
__global__ void __launch_bounds__(NT, sizeof(T) == 4 ? 16 : 8) bodies_kernel(const __grid_constant__ ModelDev<T> M, const BodiesArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const Stash<T, NT> st{reinterpret_cast<T*>(smem_raw) + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    BodiesIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.vd = {a.vd ? a.vd + bl : nullptr, a.ld};
    io.wext = {a.wext ? a.wext + bl : nullptr, a.ld};
    io.acc = a.acc ? a.acc + bl : nullptr;
    io.jw = a.jw ? a.jw + bl : nullptr;
    io.ld = a.ld;
    io.active = active;
    bodies_sample<T>(M, io, st);
  }
}

// Soft contact (contact_sample, rbd_kin.cuh): one thread per sample, stash = pending poses + twists.
template <class T> struct ContactArgs {
  const T *q, *v;
  T *s, *sd, *wr;
  int64_t ld, B;
};
template <class T, int NT>
__global__ void __launch_bounds__(NT, sizeof(T) == 4 ? 16 : 8)
contact_kernel(const __grid_constant__ ModelDev<T> M, const __grid_constant__ ContactDev<T> C, const ContactArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const Stash<T, NT> st{reinterpret_cast<T*>(smem_raw) + threadIdx.x};
  const int64_t ngroups = (a.B + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.B;
    const int64_t bl = active ? b : a.B - 1;
    ContactIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.s = a.s ? a.s + bl : nullptr;
    io.sd = a.sd ? a.sd + bl : nullptr;
    io.wr = a.wr + bl;
    io.ld = a.ld;
    io.active = active;
    contact_sample<T>(M, C, io, st);
  }
}

template <class K> int configure(K kernel, int nt, size_t smem, const DeviceProps& p, int& blocks_per_sm) {
  if ((int)smem > p.max_smem_optin) return fail(RBD_EUNSUPPORTED, "model working set exceeds shared memory per block");
  if (int rc = configure_once((const void*)kernel, p)) return rc;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, nt, smem));
  if (blocks_per_sm < 1) return fail(RBD_EUNSUPPORTED, "kernel does not fit on an SM");
  return RBD_OK;
}

// Launch `kernel(args...)` persistently: blocks_per_SM x SMs blocks of `nt` threads (fewer for a small batch) loop over the
// groups of `nt` of the `work` items, with `rows` stash rows of T per thread in shared memory.  `scratch_rows` > 0 requests a
// stream-ordered scratch of that many rows per resident thread (external wrenches, momentum-matrix poses): it is stored into
// `*scratch`, a field of one of `args`, before the launch.
template <class T, class Kern, class... Args>
int launch(Kern kernel, int nt, int rows, int64_t work, T** scratch, int scratch_rows, cudaStream_t stream, const Args&... args) {
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  const size_t smem = (size_t)rows * nt * sizeof(T);
  int bps = 0;
  if (int rc = configure(kernel, nt, smem, p, bps)) return rc;
  const int64_t ngroups = (work + nt - 1) / nt;
  const int grid = (int)std::min<int64_t>(ngroups, (int64_t)bps * p.sms);
  if (scratch_rows > 0) CUDA_TRY(cudaMallocAsync((void**)scratch, (size_t)scratch_rows * grid * nt * sizeof(T), stream));
  kernel<<<grid, nt, smem, stream>>>(args...);
  cudaError_t e = cudaGetLastError();
  if (scratch_rows > 0) cudaFreeAsync(*scratch, stream);
  if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
  g_launch.kernels_launched += 1;
  g_launch.grid = grid; g_launch.block = nt; g_launch.smem_bytes = (int)smem; g_launch.blocks_per_sm = bps;
  return RBD_OK;
}

constexpr int kNT = 32;   // threads per block: one warp; warps never synchronise with each other

// Shared-memory kernel on `stream` plus Tensor-Memory kernel (one CTA per SM, stash in TMEM, no shared memory) on the handle's
// side stream, both claiming groups of 32 samples from one atomic counter.  fp32: one stash row = one TMEM column, so the 512
// columns hold the stash of 8 warps (two column halves x four lane quadrants); fp64: two columns per row, 4 warps.  On Atlas
// that is 8 + 8 resident warps/SM in fp32 (16 x 32 x 128 registers = the whole register file) and 4 + 4 in fp64.
// `used` = false (and nothing launched) when pair_blocks declines the pair or RBD_NO_TMEM is set.
template <class T, class KS, class KT, class Args>
int launch_duo(const rbd_model* model, KS ks, KT kt, int tm_warps, const ModelDev<T>& M, Args a, int rows, int scratch_rows,
               cudaStream_t stream, bool& used) {
  used = false;
  const LaunchEnv& ev = launch_env();
  if (ev.no_tmem) return RBD_OK;
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  const int64_t ngroups = (a.B + kNT - 1) / kNT;
  const size_t smem = (size_t)rows * kNT * sizeof(T);
  int bps = 0;
  if (int rc = configure(ks, kNT, smem, p, bps)) return rc;
  if (int rc = configure_once((const void*)kt, p)) return rc;
  cudaFuncAttributes fs{}, ft{};
  CUDA_TRY(cudaFuncGetAttributes(&fs, ks));
  CUDA_TRY(cudaFuncGetAttributes(&ft, kt));
  bps = pair_blocks(p.sms, bps, fs.numRegs, ft.numRegs, tm_warps, ngroups);
  if (bps == 0) return RBD_OK;
  rbd_model* mm = const_cast<rbd_model*>(model);
  PairCtx ctx;      // side stream, fork / join events and a zeroed queue counter, all cached in the handle
  CUDA_TRY(pair_begin(mm, stream, ctx));
  cudaStream_t side = ctx.side;
  cudaEvent_t fork = ctx.fork, join = ctx.join;
  a.counter = ctx.counter;
  void* scratch = nullptr;
  if (scratch_rows > 0) {       // external wrenches in body frames: one column per resident thread of either kernel
    a.scratch_off = (int64_t)bps * p.sms * kNT;
    a.scratch_ld = a.scratch_off + (int64_t)p.sms * 32 * tm_warps;
    CUDA_TRY(cudaMallocAsync(&scratch, (size_t)scratch_rows * a.scratch_ld * sizeof(T), stream));
    a.scratch = (T*)scratch;
  }
  CUDA_TRY(cudaEventRecord(fork, stream));
  CUDA_TRY(cudaStreamWaitEvent(side, fork, 0));
  // (profiling aid: under ncu kernels are serialised and the first one drains the queue; RBD_ONLY=smem|tmem launches
  //  just one of the two so each can be captured doing the whole batch)
  if (!ev.only || ev.only[0] == 's') ks<<<bps * p.sms, kNT, smem, stream>>>(M, a);
  if (!ev.only || ev.only[0] == 't') kt<<<p.sms, 32 * tm_warps, 0, side>>>(M, a);
  cudaError_t e = cudaGetLastError();
  cudaEventRecord(join, side);
  cudaStreamWaitEvent(stream, join, 0);
  if (scratch) cudaFreeAsync(scratch, stream);
  if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
  g_launch.kernels_launched += 2;
  g_launch.grid = bps * p.sms; g_launch.block = kNT; g_launch.smem_bytes = (int)smem; g_launch.blocks_per_sm = bps;
  used = true;
  return RBD_OK;
}

// The model-specialised kernels for `key` (rbd_spec.cpp: straight-line code generated for this mechanism) when they can serve
// the call, else `generic(nullptr)`.  fp32 specialised programs have no slow sin / cos path: if any sample met an angle beyond
// 1e4 rad they raise a flag on the device, and `generic(gate)` enqueued behind them redoes the batch with the library path (it
// exits at once while the flag is down).  Launch info then describes the specialised launch and counts the kernels of both.
template <class Generic>
int spec_or_generic(const rbd_model* model, const SpecKey& key, const SpecLaunchArgs& sa, cudaStream_t stream, Generic generic) {
  bool used = false;
  const int* gate = nullptr;
  if (int rc = spec_try_launch(const_cast<rbd_model*>(model), key, sa, stream, used, g_launch, &gate)) return rc;
  if (!used) return generic(nullptr);
  g_launch.specialised = 1;
  if (!gate) return RBD_OK;
  const rbd_launch_info keep = g_launch;
  const int rc = generic(gate);
  const int n = g_launch.kernels_launched;
  g_launch = keep;
  g_launch.kernels_launched = n;
  return rc;
}

// The generic ABA kernel for this model: multi-DoF joints below the root (GENERAL), prismatic / fixed joints (all 1-DoF kinds)
// or revolute joints only (KINDS = 0).
template <class T>
int launch_generic_aba(const HostModel& hm, AbaArgs<T> a, bool ext, cudaStream_t stream) {
  const ModelDev<T>& M = dev_model<T>(hm);
  auto kernel = hm.general       ? (ext ? aba_kernel<T, kNT, true, true, kAllKinds> : aba_kernel<T, kNT, true, false, kAllKinds>)
                : hm.other_kinds ? (ext ? aba_kernel<T, kNT, false, true, kAllKinds> : aba_kernel<T, kNT, false, false, kAllKinds>)
                                 : (ext ? aba_kernel<T, kNT, false, true, 0> : aba_kernel<T, kNT, false, false, 0>);
  return launch<T>(kernel, kNT, M.nrows, a.B, &a.scratch, ext ? 6 * hm.nb : 0, stream, M, a);
}

template <class T>
int dynamics_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const void* tau,
               const void* wext, void* vd, void* qd, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  AbaArgs<T> a{(const T*)q, (const T*)v, (const T*)tau, (const T*)wext, (T*)vd, (T*)qd, nullptr, ld, B};
  auto generic = [&](const int* gate) {
    a.gate = gate;
    if (!gate && !hm.general && !hm.other_kinds && M.nrows <= 256) {
      // default path for all-revolute trees whose stash fits Tensor Memory (see launch_duo); its kernels take no gate
      constexpr int kTmWarps = sizeof(T) == 4 ? 8 : 4;
      bool used = false;
      const int rc = launch_duo<T>(model, wext ? aba_kernel_smem_q<T, 0, true> : aba_kernel_smem_q<T, 0, false>,
                                   wext ? aba_kernel_tmem_q<T, 512, 0, kTmWarps, true> : aba_kernel_tmem_q<T, 512, 0, kTmWarps, false>,
                                   kTmWarps, M, a, M.nrows, wext ? 6 * hm.nb : 0, stream, used);
      if (rc || used) return rc;
    }
    return launch_generic_aba<T>(hm, a, wext != nullptr, stream);
  };
  if (wext) return generic(nullptr);      // the model-specialised kernels take no external wrenches
  SpecKey key; key.algo = SPEC_ABA; key.f64 = sizeof(T) == 8; key.has_in2 = tau != nullptr; key.has_out1 = qd != nullptr;
  return spec_or_generic(model, key, {q, v, tau, vd, qd, ld, B}, stream, generic);
}

template <class T>
int inverse_dynamics_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const void* vd,
                       const void* wext, void* tau, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  RneaArgs<T> a{(const T*)q, (const T*)v, (const T*)vd, (const T*)wext, (T*)tau, nullptr, ld, B};
  const int rows = rnea_rows(hm);
  const int sr = wext ? 6 * hm.nb : 0;
  auto generic = [&](const int* gate) {
    a.gate = gate;
    if (!gate && rows <= 256) {      // the kernel pair, see dynamics_t
      constexpr int kTmWarps = sizeof(T) == 4 ? 8 : 4;
      bool used = false;
      const int rc = launch_duo<T>(model, wext ? rnea_kernel_smem_q<T, true> : rnea_kernel_smem_q<T, false>,
                                   wext ? rnea_kernel_tmem_q<T, 512, kTmWarps, true> : rnea_kernel_tmem_q<T, 512, kTmWarps, false>,
                                   kTmWarps, M, a, rows, sr, stream, used);
      if (rc || used) return rc;
    }
    return launch<T>(wext ? rnea_kernel<T, kNT, true> : rnea_kernel<T, kNT, false>, kNT, rows, B, &a.scratch, sr, stream, M, a);
  };
  if (wext) return generic(nullptr);
  SpecKey key; key.algo = SPEC_RNEA; key.f64 = sizeof(T) == 8; key.has_in2 = vd != nullptr;
  return spec_or_generic(model, key, {q, v, vd, tau, nullptr, ld, B}, stream, generic);
}

template <class T>
int mass_matrix_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, void* Mout, cudaStream_t stream, bool lower = false) {
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  CrbaArgs<T> a{(const T*)q, (T*)Mout, ld, B, lower, nullptr};
  const int rows = std::max(1, crba_rows(hm));
  bool multi = false;
  for (int i = 0; i < hm.nb; ++i) multi |= kind_nv(M.body[i].kind) > 1;
  auto generic = [&](const int* gate) {
    a.gate = gate;
    return launch<T>(multi ? crba_kernel<T, kNT, 6> : crba_kernel<T, kNT, 1>, kNT, rows, B, nullptr, 0, stream, M, a);
  };
  // model-specialised kernel: the composite-rigid-body algorithm traced on this mechanism (rbd_codegen.cpp)
  SpecKey key; key.algo = SPEC_CRBA; key.f64 = sizeof(T) == 8; key.has_in2 = false; key.lower = lower;
  return spec_or_generic(model, key, {q, nullptr, nullptr, Mout, nullptr, ld, B}, stream, generic);
}

// Kinematics by-products (SURVEY 8(f) rank 2).  One launch; the momentum matrix additionally parks the 12 nb pose rows of
// every resident thread in a stream-ordered scratch between its outward and inward sweeps.
template <class T>
int kinematics_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const int8_t* path_sign,
                 const rbd_kinematics_out& o, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  KinDev<T> K;
  std::memset(&K, 0, sizeof(K));
  for (int p = 0; p < hm.nb; ++p) {
    for (int k = 0; k < 9; ++k) K.At[p][k] = (T)hm.alignT[9 * p + k];
    K.sign[p] = path_sign ? path_sign[hm.order[p]] : 0;
  }
  K.inv_mass = (T)(1.0 / hm.total_mass);
  KinArgs<T> a{(const T*)q, (const T*)v, (T*)o.transforms_to_root, (T*)o.center_of_mass, (T*)o.kinetic_energy,
               (T*)o.gravitational_potential_energy, (T*)o.momentum, (T*)o.momentum_rate_bias, (T*)o.momentum_matrix,
               (T*)o.geometric_jacobian, nullptr, ld, B, nullptr};
  auto generic = [&](const int* gate) {
    a.gate = gate;
    return launch<T>(kin_kernel<T, kNT>, kNT, std::max(1, kin_rows(hm)), B, &a.scratch, o.momentum_matrix ? 12 * hm.nb : 0, stream,
                     M, a, K);
  };
  // model-specialised kernel for this output subset (and this jacobian path)
  SpecKey key;
  key.algo = SPEC_KIN; key.f64 = sizeof(T) == 8; key.has_in2 = v != nullptr;
  void* const outs[8] = {o.transforms_to_root, o.center_of_mass, o.kinetic_energy, o.gravitational_potential_energy, o.momentum,
                         o.momentum_rate_bias, o.momentum_matrix, o.geometric_jacobian};
  SpecLaunchArgs sa{q, v, nullptr, nullptr, nullptr, ld, B};
  for (int k = 0; k < 8; ++k) { if (outs[k]) key.kin_mask |= 1 << k; sa.ko[k] = outs[k]; }
  for (int i = 0; i < hm.nb; ++i) key.kin_sign[i] = K.sign[i];
  return key.kin_mask ? spec_or_generic(model, key, sa, stream, generic) : generic(nullptr);
}

// dynamics! on Dual{Float64,6} arrays (config 4).  The Dual model (constants with zero partials, 25 KB) is built per call
// from the fp64 one; this path is not the hot one.
int dynamics_dual(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const void* tau, void* vd,
                  cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const ModelDev<double>& S = hm.dev64;
  std::unique_ptr<ModelDev<Dual64>> Mp(new ModelDev<Dual64>());
  Mp->nb = S.nb; Mp->nq = S.nq; Mp->nv = S.nv; Mp->nrows = S.nrows; Mp->slot_base = S.slot_base; Mp->nslots = S.nslots;
  for (int k = 0; k < 3; ++k) Mp->g[k] = Dual64(S.g[k]);
  for (int i = 0; i < S.nb; ++i) {
    const BodyDev<double>& s = S.body[i];
    BodyDev<Dual64>& d = Mp->body[i];
    for (int k = 0; k < 9; ++k) d.Rt[k] = Dual64(s.Rt[k]);
    for (int k = 0; k < 3; ++k) { d.pt[k] = Dual64(s.pt[k]); d.h[k] = Dual64(s.h[k]); }
    for (int k = 0; k < 6; ++k) d.J[k] = Dual64(s.J[k]);
    d.m = Dual64(s.m);
    d.qoff = Dual64(s.qoff);
    d.kind = s.kind; d.parent = s.parent; d.qrow = s.qrow; d.vrow = s.vrow; d.row0 = s.row0;
    d.oslot = s.oslot; d.pslot = s.pslot; d.flags = s.flags; d.refidx = s.refidx;
  }
  const DualArgs a{(const double*)q, (const double*)v, (const double*)tau, (double*)vd, ld, B};
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  // split stash (shared memory + Tensor Memory): 4 warps/SM instead of 2 on Atlas; one CTA per SM, it takes all 512 columns
  const size_t smem_tm = (size_t)S.nrows * 128 * sizeof(double);
  if (!hm.general && S.nrows <= 256 && (int)smem_tm <= p.max_smem_optin && B * 6 >= (int64_t)p.sms * 128 && !launch_env().no_tmem) {
    int bps_tm = 0;
    if (int rc = configure(aba_dual_kernel_tm, 128, smem_tm, p, bps_tm)) return rc;
    const int64_t ng = (B * 6 + 127) / 128;
    const int grid_tm = (int)std::min<int64_t>(ng, p.sms);
    aba_dual_kernel_tm<<<grid_tm, 128, smem_tm, stream>>>(*Mp, a);
    CUDA_TRY(cudaGetLastError());
    g_launch.kernels_launched += 1;
    g_launch.grid = grid_tm; g_launch.block = 128; g_launch.smem_bytes = (int)smem_tm; g_launch.blocks_per_sm = 1;
    return RBD_OK;
  }
  // one thread per (sample, partial direction)
  return launch<Dual64>(hm.general ? aba_dual_kernel<kNT, true> : aba_dual_kernel<kNT, false>, kNT, S.nrows, B * 6, nullptr, 0, stream,
                        *Mp, a);
}

// ---- Munthe-Kaas RK4 (rbd_integrate): elementwise stage kernels around the dynamics kernels -----------------------------
// Stage i of a step, one thread per (sample, joint) -- every joint's coordinate map is independent of the others (blockIdx.y =
// body).  The local coordinates of the stage and the stage velocity are functions of the previous stage's rates,
//   phi = dt a_i phid_{i-1} ,  v_s = v0 + dt a_i vd_{i-1} ,
// evaluated on the fly by the two accessors below (nothing but the kernel's real outputs is written):
//   q_s = global(q0, phi) ,  v_s  -> inputs of the dynamics kernels ;  phid_i = d/dt local(q0, q_s, v_s) -> kept for the next stage
// and for the final combination.  The four (phid_i, vd_i) pairs are stored separately; the finishing kernel forms the weighted sums.
template <class T> struct ScaledRow {      // wa * p[row]  (zero when there is no previous stage)
  const T* p; int64_t ld; T wa;
  RBD_HD T operator()(int row) const { return p ? wa * p[(int64_t)row * ld] : T(0); }
};
template <class T> struct OffsetRow {      // base[row] + wa * p[row]
  const T* base; const T* p; int64_t ld; T wa;
  RBD_HD T operator()(int row) const {
    const T b = base[(int64_t)row * ld];
    return p ? b + wa * p[(int64_t)row * ld] : b;
  }
};
template <class T> struct StageArgs {
  const T* q0; const T* v0;               // state at the start of the step
  const T* phid_prev; const T* vd_prev;   // rates of the previous stage (NULL for stage 0)
  T* phid; T* qs; T* vs;                  // outputs
  T wa;                                   // dt * a_i
  int64_t B;
  bool skip_linear;                       // revolute / prismatic joints are done by the vectorised kernel below
};
template <class T>
__global__ void __launch_bounds__(128) integrate_stage_kernel(const __grid_constant__ ModelDev<T> M, const StageArgs<T> a) {
  const BodyDev<T>& bd = M.body[blockIdx.y];
  const int k0 = bd.vrow, k1 = bd.vrow + kind_nv_dev(bd.kind);
  if (k1 == k0) return;                                    // fixed joint: no coordinates
  if (a.skip_linear && (bd.kind == K_REV || bd.kind == K_PRIS)) return;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += (int64_t)gridDim.x * blockDim.x) {
    const Col<T> q0{a.q0 + b, a.B};
    const ScaledRow<T> phi{a.phid_prev ? a.phid_prev + b : nullptr, a.B, a.wa};
    const OffsetRow<T> vs{a.v0 + b, a.vd_prev ? a.vd_prev + b : nullptr, a.B, a.wa};
    for (int k = k0; k < k1; ++k) a.vs[(int64_t)k * a.B + b] = vs(k);
    const ColOut<T> qs{a.qs + b, a.B, true}, phid{a.phid + b, a.B, true};
    joint_stage(bd, q0, phi, vs, qs, phid);
  }
}
// Revolute / prismatic joints (the bulk of a robot): q_s = q0 + wa phid_prev, v_s = v0 + wa vd_prev, phid = v_s -- plain row
// arithmetic, done VEC samples per thread with 16-byte accesses so that enough loads are in flight to approach the HBM rate (the
// per-(sample, joint) kernel above sits at 15 % of it, long_scoreboard 13 warps per issue: profiles/r2_gen_rk4_stage_summary.txt).
template <class T> struct VecOf { using type = float4; static constexpr int N = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int N = 2; };
template <class T> __device__ __forceinline__ void vec_axpy(const typename VecOf<T>::type& a, T w, const typename VecOf<T>::type& x,
                                                            typename VecOf<T>::type& o);
template <> __device__ __forceinline__ void vec_axpy<float>(const float4& a, float w, const float4& x, float4& o) {
  o.x = a.x + w * x.x; o.y = a.y + w * x.y; o.z = a.z + w * x.z; o.w = a.w + w * x.w;
}
template <> __device__ __forceinline__ void vec_axpy<double>(const double2& a, double w, const double2& x, double2& o) {
  o.x = a.x + w * x.x; o.y = a.y + w * x.y;
}
template <class T> __device__ __forceinline__ typename VecOf<T>::type vec_comb4(const typename VecOf<T>::type& base, T dt, const T* w,
                                                                                const typename VecOf<T>::type* x);
template <> __device__ __forceinline__ float4 vec_comb4<float>(const float4& b, float dt, const float* w, const float4* x) {
  float4 o;
  o.x = b.x + dt * (w[0] * x[0].x + w[1] * x[1].x + w[2] * x[2].x + w[3] * x[3].x);
  o.y = b.y + dt * (w[0] * x[0].y + w[1] * x[1].y + w[2] * x[2].y + w[3] * x[3].y);
  o.z = b.z + dt * (w[0] * x[0].z + w[1] * x[1].z + w[2] * x[2].z + w[3] * x[3].z);
  o.w = b.w + dt * (w[0] * x[0].w + w[1] * x[1].w + w[2] * x[2].w + w[3] * x[3].w);
  return o;
}
template <> __device__ __forceinline__ double2 vec_comb4<double>(const double2& b, double dt, const double* w, const double2* x) {
  double2 o;
  o.x = b.x + dt * (w[0] * x[0].x + w[1] * x[1].x + w[2] * x[2].x + w[3] * x[3].x);
  o.y = b.y + dt * (w[0] * x[0].y + w[1] * x[1].y + w[2] * x[2].y + w[3] * x[3].y);
  return o;
}

template <class T>
__global__ void __launch_bounds__(256) integrate_stage_linear_kernel(const __grid_constant__ ModelDev<T> M, const StageArgs<T> a) {
  using V = typename VecOf<T>::type;
  constexpr int N = VecOf<T>::N;
  const BodyDev<T>& bd = M.body[blockIdx.y];
  if (bd.kind != K_REV && bd.kind != K_PRIS) return;
  const int64_t qo = (int64_t)bd.qrow * a.B, vo = (int64_t)bd.vrow * a.B, nvec = a.B / N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    const V q0 = reinterpret_cast<const V*>(a.q0 + qo)[i];
    const V v0 = reinterpret_cast<const V*>(a.v0 + vo)[i];
    V qs = q0, vs = v0;
    if (a.phid_prev) {
      const V pp = reinterpret_cast<const V*>(a.phid_prev + vo)[i];
      const V vp = reinterpret_cast<const V*>(a.vd_prev + vo)[i];
      vec_axpy<T>(q0, a.wa, pp, qs);
      vec_axpy<T>(v0, a.wa, vp, vs);
    }
    reinterpret_cast<V*>(a.qs + qo)[i] = qs;
    reinterpret_cast<V*>(a.vs + vo)[i] = vs;
    reinterpret_cast<V*>(a.phid + vo)[i] = vs;
  }
}
// v = v0 + dt sum_i b_i vd_i ,  q = global(q0, dt sum_i b_i phid_i)        (ode_integrators.jl:283-296)
template <class T> struct SumRow4 {        // [base[row] +] dt * sum_i w_i p_i[row]
  const T* base; const T* p[4]; int64_t ld; T w[4]; T dt;
  RBD_HD T operator()(int row) const {
    const int64_t e = (int64_t)row * ld;
    const T s = dt * (w[0] * p[0][e] + w[1] * p[1][e] + w[2] * p[2][e] + w[3] * p[3][e]);
    return base ? base[e] + s : s;
  }
};
template <class T> struct FinishArgs {
  const T* q0; const T* v0;
  const T* phid[4]; const T* vd[4];
  T* q; T* v;                              // user arrays (leading dimension ld)
  T w[4]; T dt;
  int64_t B, ld;
  bool refresh;                            // also write the new state into (q0, v0) for the next step (each thread owns its joint's rows)
  bool skip_linear;                        // revolute / prismatic joints are done by integrate_finish_linear_kernel
};
// finishing step of the revolute / prismatic rows, vectorised like integrate_stage_linear_kernel
template <class T>
__global__ void __launch_bounds__(256) integrate_finish_linear_kernel(const __grid_constant__ ModelDev<T> M, const FinishArgs<T> a) {
  using V = typename VecOf<T>::type;
  constexpr int N = VecOf<T>::N;
  const BodyDev<T>& bd = M.body[blockIdx.y];
  if (bd.kind != K_REV && bd.kind != K_PRIS) return;
  const int64_t qo = (int64_t)bd.qrow * a.B, vo = (int64_t)bd.vrow * a.B, nvec = a.B / N;
  V* qu = reinterpret_cast<V*>(a.q + (int64_t)bd.qrow * a.ld);
  V* vu = reinterpret_cast<V*>(a.v + (int64_t)bd.vrow * a.ld);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    V ph[4], vd[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { ph[k] = reinterpret_cast<const V*>(a.phid[k] + vo)[i]; vd[k] = reinterpret_cast<const V*>(a.vd[k] + vo)[i]; }
    const V qn = vec_comb4<T>(reinterpret_cast<const V*>(a.q0 + qo)[i], a.dt, a.w, ph);
    const V vn = vec_comb4<T>(reinterpret_cast<const V*>(a.v0 + vo)[i], a.dt, a.w, vd);
    qu[i] = qn; vu[i] = vn;
    if (a.refresh) {
      reinterpret_cast<V*>(const_cast<T*>(a.q0) + qo)[i] = qn;
      reinterpret_cast<V*>(const_cast<T*>(a.v0) + vo)[i] = vn;
    }
  }
}
template <class T>
__global__ void __launch_bounds__(128) integrate_finish_kernel(const __grid_constant__ ModelDev<T> M, const FinishArgs<T> a) {
  const BodyDev<T>& bd = M.body[blockIdx.y];
  const int k0 = bd.vrow, k1 = bd.vrow + kind_nv_dev(bd.kind);
  if (k1 == k0) return;
  if (a.skip_linear && (bd.kind == K_REV || bd.kind == K_PRIS)) return;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += (int64_t)gridDim.x * blockDim.x) {
    const Col<T> q0{a.q0 + b, a.B};
    const SumRow4<T> phi{nullptr, {a.phid[0] + b, a.phid[1] + b, a.phid[2] + b, a.phid[3] + b}, a.B, {a.w[0], a.w[1], a.w[2], a.w[3]}, a.dt};
    const SumRow4<T> vn{a.v0 + b, {a.vd[0] + b, a.vd[1] + b, a.vd[2] + b, a.vd[3] + b}, a.B, {a.w[0], a.w[1], a.w[2], a.w[3]}, a.dt};
    T vnew[6];
    for (int k = k0; k < k1; ++k) { vnew[k - k0] = vn(k); a.v[(int64_t)k * a.ld + b] = vnew[k - k0]; }
    const ColOut<T> q{a.q + b, a.ld, true}, dump{nullptr, a.B, false};
    joint_stage(bd, q0, phi, vn, q, dump);
    if (a.refresh) {                       // after every read of this joint's (q0, v0) rows above
      const int nqj = kind_nq_dev(bd.kind);
      for (int k = 0; k < nqj; ++k) const_cast<T*>(a.q0)[(int64_t)(bd.qrow + k) * a.B + b] = a.q[(int64_t)(bd.qrow + k) * a.ld + b];
      for (int k = k0; k < k1; ++k) const_cast<T*>(a.v0)[(int64_t)k * a.B + b] = vnew[k - k0];
    }
  }
}

template <class T>
int integrate_t(const rbd_model* model, int64_t B, int64_t ld, void* q, void* v, const void* tau, int64_t step_stride,
                int64_t stage_stride, double dt, int nsteps, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  const size_t nq = hm.nq, nv = hm.nv;
  const size_t rows = 2 * nq + 10 * nv + (tau && ld != B ? nv : 0);
  T* ws = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&ws, rows * (size_t)B * sizeof(T), stream));
  struct Guard { void* p; cudaStream_t s; ~Guard() { if (p) cudaFreeAsync(p, s); } } guard{ws, stream};    // freed on every exit path
  T* q0 = ws; T* qs = q0 + nq * B; T* v0 = qs + nq * B; T* vs = v0 + nv * B;
  T* phid[4]; T* vd[4];
  for (int i = 0; i < 4; ++i) { phid[i] = vs + (size_t)(1 + i) * nv * B; vd[i] = vs + (size_t)(5 + i) * nv * B; }
  T* taud = vs + (size_t)9 * nv * B;
  // torques of (step s, stage i): tau + s * step_stride + i * stage_stride (both 0: one array held over the whole call); the
  // dynamics kernels want leading dimension B, so arrays with ld != B are densified per use
  const bool varying = step_stride != 0 || stage_stride != 0;
  auto tau_at = [&](int s_, int i_) -> const T* { return tau ? (const T*)tau + (size_t)s_ * step_stride + (size_t)i_ * stage_stride : nullptr; };
  const T* tau_dense = (const T*)tau;
  if (tau && ld != B && !varying) {
    CUDA_TRY(cudaMemcpy2DAsync(taud, B * sizeof(T), tau, ld * sizeof(T), B * sizeof(T), nv, cudaMemcpyDeviceToDevice, stream));
    tau_dense = taud;
  }
  const int grid = (int)std::min<int64_t>((B + 127) / 128, (int64_t)p.sms * 8);
  // the vectorised kernel needs whole vectors per row (workspace rows are B long and 256-byte aligned)
  const bool vec_ok = B % VecOf<T>::N == 0 && B >= 1024;
  const int grid_lin = (int)std::min<int64_t>((B / VecOf<T>::N + 255) / 256, (int64_t)p.sms * 4);
  // ... and, for the finishing kernel, vector-aligned rows of the caller's arrays too
  const bool vec_user = vec_ok && ld % VecOf<T>::N == 0 && ((uintptr_t)q % sizeof(typename VecOf<T>::type)) == 0 &&
                        ((uintptr_t)v % sizeof(typename VecOf<T>::type)) == 0;
  bool has_other = false;
  for (int i = 0; i < hm.nb; ++i) has_other |= (M.body[i].kind != K_REV && M.body[i].kind != K_PRIS && M.body[i].kind != K_FIXED);
  const double a[4] = {0.0, 0.5, 0.5, 1.0}, bw[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};   // runge_kutta_4, ode_integrators.jl:48-55
  int rc = RBD_OK, launches = 0;
  // (q0, v0): dense copies of the state at the start of the step; the finishing kernel of step s refreshes them for step s + 1
  CUDA_TRY(cudaMemcpy2DAsync(q0, B * sizeof(T), q, ld * sizeof(T), B * sizeof(T), nq, cudaMemcpyDeviceToDevice, stream));
  CUDA_TRY(cudaMemcpy2DAsync(v0, B * sizeof(T), v, ld * sizeof(T), B * sizeof(T), nv, cudaMemcpyDeviceToDevice, stream));
  for (int s = 0; s < nsteps && rc == RBD_OK; ++s) {
    for (int i = 0; i < 4 && rc == RBD_OK; ++i) {
      if (varying) {
        tau_dense = tau_at(s, i);
        if (tau && ld != B) {
          CUDA_TRY(cudaMemcpy2DAsync(taud, B * sizeof(T), tau_dense, ld * sizeof(T), B * sizeof(T), nv, cudaMemcpyDeviceToDevice, stream));
          tau_dense = taud;
        }
      }
      StageArgs<T> sa{q0, v0, i ? phid[i - 1] : nullptr, i ? vd[i - 1] : nullptr, phid[i], qs, vs, (T)(dt * a[i]), B, vec_ok};
      if (vec_ok) {        // revolute / prismatic rows, VEC samples per thread
        integrate_stage_linear_kernel<T><<<dim3(grid_lin, hm.nb), 256, 0, stream>>>(M, sa);
        CUDA_TRY(cudaGetLastError());
        launches += 1;
      }
      if (!vec_ok || has_other) {
        integrate_stage_kernel<T><<<dim3(grid, hm.nb), 128, 0, stream>>>(M, sa);
        CUDA_TRY(cudaGetLastError());
        launches += 1;
      }
      const int before = g_launch.kernels_launched;
      rc = dynamics_t<T>(model, B, B, qs, vs, tau_dense, nullptr, vd[i], nullptr, stream);
      launches += g_launch.kernels_launched - before;
    }
    if (rc != RBD_OK) break;
    FinishArgs<T> fa{q0, v0, {phid[0], phid[1], phid[2], phid[3]}, {vd[0], vd[1], vd[2], vd[3]}, (T*)q, (T*)v,
                     {(T)bw[0], (T)bw[1], (T)bw[2], (T)bw[3]}, (T)dt, B, ld, s + 1 < nsteps, vec_user};
    if (vec_user) {
      integrate_finish_linear_kernel<T><<<dim3(grid_lin, hm.nb), 256, 0, stream>>>(M, fa);
      CUDA_TRY(cudaGetLastError());
      launches += 1;
    }
    if (!vec_user || has_other) {
      integrate_finish_kernel<T><<<dim3(grid, hm.nb), 128, 0, stream>>>(M, fa);
      CUDA_TRY(cudaGetLastError());
      launches += 1;
    }
  }
  g_launch.kernels_launched = launches;
  return rc;
}

// rbd_dynamics_gather.  Fast path: the model-specialised kernels store v̇ straight into every GPU's gathered array (peer-mapped
// memory, posted writes over NVLink) -- the output store IS the gather.  Fallback (no specialised kernel for this model / dtype,
// or -- gated on their flag -- a sample beyond their fast sin / cos range): the generic kernels evaluate into a dense scratch
// and this kernel scatters it to the peers.
template <class T> struct ScatterArgs {
  const T* src; int64_t src_ld;
  T* dst[8]; int64_t dst_ld;
  int ndst, rows;
  int64_t B;
  const int* gate;
};
template <class T> __global__ void __launch_bounds__(256) gather_scatter_kernel(const ScatterArgs<T> a) {
  if (a.gate && *a.gate == 0) return;
  const int64_t total = (int64_t)a.rows * a.B;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = e / a.B, b = e - k * a.B;
    const T x = a.src[k * a.src_ld + b];
#pragma unroll
    for (int p = 0; p < 8; ++p)
      if (p < a.ndst) a.dst[p][k * a.dst_ld + b] = x;
  }
}

template <class T>
int dynamics_gather_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const void* tau, int npeers,
                      void* const* peers, void* mc, int64_t peer_ld, int64_t col0, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  // generic kernels: they use ONE leading dimension for inputs and outputs, so they write into a [nv x ld] scratch which
  // gather_scatter_kernel then copies to the peers
  auto generic = [&](const int* gate) {
    T* scratch = nullptr;
    CUDA_TRY(cudaMallocAsync((void**)&scratch, (size_t)hm.nv * (size_t)ld * sizeof(T), stream));
    int rc;
    if (gate) {        // behind the peer-writing specialised kernel
      AbaArgs<T> a{(const T*)q, (const T*)v, (const T*)tau, nullptr, scratch, nullptr, nullptr, ld, B};
      a.gate = gate;
      rc = launch_generic_aba<T>(hm, a, false, stream);
    } else {
      rc = dynamics_t<T>(model, B, ld, q, v, tau, nullptr, scratch, nullptr, stream);
    }
    if (rc == RBD_OK) {
      ScatterArgs<T> sc{};
      sc.src = scratch; sc.src_ld = ld; sc.dst_ld = peer_ld; sc.ndst = npeers; sc.rows = hm.nv; sc.B = B; sc.gate = gate;
      for (int p = 0; p < npeers; ++p) sc.dst[p] = (T*)peers[p] + col0;
      DeviceProps p;
      if ((rc = get_props(p)) == RBD_OK) {
        gather_scatter_kernel<T><<<p.sms * 8, 256, 0, stream>>>(sc);
        if (cudaGetLastError() != cudaSuccess) rc = fail(RBD_ECUDA, "gather_scatter_kernel launch failed");
        g_launch.kernels_launched += 1;
      }
    }
    cudaFreeAsync(scratch, stream);
    return rc;
  };
  SpecKey key; key.algo = SPEC_ABA; key.f64 = sizeof(T) == 8; key.has_in2 = tau != nullptr; key.peers = true;
  SpecLaunchArgs sa{q, v, tau, nullptr, nullptr, ld, B};
  sa.peers = peers; sa.npeers = npeers; sa.peer_ld = peer_ld; sa.peer_col0 = col0; sa.mc = mc;
  return spec_or_generic(model, key, sa, stream, generic);
}

template <class T>
int bodies_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const void* vd, const void* wext, void* acc,
             void* jw, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  const BodiesArgs<T> a{(const T*)q, (const T*)v, (const T*)vd, (const T*)wext, (T*)acc, (T*)jw, ld, B};
  return launch<T>(bodies_kernel<T, kNT>, kNT, std::max(1, kin_rows(hm)), B, nullptr, 0, stream, dev_model<T>(hm), a);
}

template <class T>
int contact_t(const rbd_model* model, int64_t B, int64_t ld, const void* q, const void* v, const rbd_contact_desc& cd, void* sx,
              void* sd, void* wr, cudaStream_t stream) {
  const HostModel& hm = model->hm;
  ContactDev<T> C;
  build_contact_dev<T>(hm.nb, hm.pos.data(), hm.alignT.data(), cd, C);
  const ContactArgs<T> a{(const T*)q, (const T*)v, (T*)sx, (T*)sd, (T*)wr, ld, B};
  return launch<T>(contact_kernel<T, kNT>, kNT, std::max(1, kin_rows(hm)), B, nullptr, 0, stream, dev_model<T>(hm), C, a);
}

int check_common(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, bool allow_dual = false) {
  if (!model) return fail(RBD_EINVAL, "model handle is NULL");
  if (dtype != RBD_F32 && dtype != RBD_F64 && dtype != RBD_DUAL64X6)
    return fail(RBD_EINVAL, "dtype must be RBD_F32, RBD_F64 or RBD_DUAL64X6");
  if (dtype == RBD_DUAL64X6 && !allow_dual)
    return fail(RBD_EUNSUPPORTED, "RBD_DUAL64X6 is supported by rbd_dynamics only; use the reference's generic path");
  if (B < 0 || ld < B) return fail(RBD_EDIM, "batch size / leading dimension mismatch (need ld >= B >= 0)");
  return RBD_OK;
}

}  // namespace

// hooks for the other translation units of the library (rbd_deriv.cu): per-thread error text, argument checks, launch statistics
namespace rbd {
int api_fail(int status, const std::string& msg) { return fail(status, msg); }
int api_check(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld) { return check_common(model, dtype, B, ld); }
void api_note_launch(int grid, int block, int smem_bytes, int blocks_per_sm) {
  g_launch.kernels_launched += 1;
  g_launch.grid = grid; g_launch.block = block; g_launch.smem_bytes = smem_bytes; g_launch.blocks_per_sm = blocks_per_sm;
}
}  // namespace rbd

// ------------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------------
int32_t rbd_kinematics(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                       const int8_t* path_sign, const rbd_kinematics_out* out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (dtype != RBD_F32 && dtype != RBD_F64) return fail(RBD_EUNSUPPORTED, "rbd_kinematics: fp32 and fp64 only");
  if (!out) return fail(RBD_EINVAL, "rbd_kinematics: out must not be NULL");
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q) return fail(RBD_EINVAL, "rbd_kinematics: q must not be NULL");
  if (!v && (out->kinetic_energy || out->momentum || out->momentum_rate_bias))
    return fail(RBD_EINVAL, "rbd_kinematics: kinetic_energy / momentum / momentum_rate_bias need v");
  if ((out->geometric_jacobian != nullptr) != (path_sign != nullptr))
    return fail(RBD_EINVAL, "rbd_kinematics: path_sign must be given iff geometric_jacobian is requested");
  if (path_sign)
    for (int i = 0; i < model->hm.nb; ++i)
      if (path_sign[i] < -1 || path_sign[i] > 1) return fail(RBD_EINVAL, "rbd_kinematics: path_sign entries must be -1, 0 or +1");
  if (model->hm.total_mass <= 0 && out->center_of_mass) return fail(RBD_EINVAL, "rbd_kinematics: mechanism has no mass");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? kinematics_t<float>(model, B, ld, q, v, path_sign, *out, s)
                          : kinematics_t<double>(model, B, ld, q, v, path_sign, *out, s);
}

// ---- host-pointer variants: chunked H2D -> kernel -> D2H pipeline over three internal streams ----
namespace {
constexpr int64_t kChunk = 1 << 16;

int ensure_staging(rbd_model* m, size_t bytes_per_stream) {
  for (int i = 0; i < 3; ++i)
    if (!m->streams[i]) CUDA_TRY(cudaStreamCreateWithFlags(&m->streams[i], cudaStreamNonBlocking));
  if (!m->ev0) { CUDA_TRY(cudaEventCreate(&m->ev0)); CUDA_TRY(cudaEventCreate(&m->ev1)); }
  if (m->stage_bytes >= bytes_per_stream) return RBD_OK;
  m->stage_bytes = 0;               // a failed reallocation must not leave a stale size behind
  for (int i = 0; i < 3; ++i) {
    if (m->d_stage[i]) { cudaFree(m->d_stage[i]); m->d_stage[i] = nullptr; }
    CUDA_TRY(cudaMalloc(&m->d_stage[i], bytes_per_stream));
  }
  m->stage_bytes = bytes_per_stream;
  return RBD_OK;
}

struct HostArr { const void* in; void* out; int rows; };

// Chunked host pipeline: chunk c uses stream c % 3 and that stream's staging buffer; H2D copies, the kernel and the D2H
// copies of one chunk are stream-ordered, chunks on different streams overlap (copy engines in both directions + SMs).
template <class Launch>
int host_pipeline_impl(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const HostArr* ins, int nin, const HostArr* outs,
                       int nout, Launch launch_chunk);
template <class Launch>
int host_pipeline(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const HostArr* ins, int nin, const HostArr* outs,
                  int nout, Launch launch_chunk) {
  std::lock_guard<std::mutex> lk(model->host_mu);
  const int rc = host_pipeline_impl(model, dtype, B, ld, ins, nin, outs, nout, launch_chunk);
  if (rc != RBD_OK)                 // never return with copies into the caller's host buffers still in flight
    for (int i = 0; i < 3; ++i) if (model->streams[i]) cudaStreamSynchronize(model->streams[i]);
  return rc;
}
template <class Launch>
int host_pipeline_impl(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const HostArr* ins, int nin, const HostArr* outs,
                       int nout, Launch launch_chunk) {
  const size_t es = dtype == RBD_F32 ? 4 : 8;
  int64_t chunk = kChunk;
  if (const char* e = getenv("RBD_HOST_CHUNK")) chunk = std::max<int64_t>(1024, atoll(e));     // tuning knob
  const int64_t C = std::min<int64_t>(chunk, B);
  size_t rows_total = 0;
  for (int i = 0; i < nin; ++i) rows_total += ins[i].in ? ins[i].rows : 0;
  for (int i = 0; i < nout; ++i) rows_total += outs[i].out ? outs[i].rows : 0;
  if (int rc = ensure_staging(model, rows_total * C * es)) return rc;
  int launches = 0, nchunk = 0;
  rbd_launch_info last = g_launch;
  for (int64_t b0 = 0; b0 < B; b0 += C, ++nchunk) {
    const int64_t n = std::min<int64_t>(C, B - b0);
    const int si = nchunk % 3;
    cudaStream_t s = model->streams[si];
    char* cur = (char*)model->d_stage[si];
    const size_t off = (size_t)b0 * es;
    const void* din[8] = {nullptr};
    void* dout[8] = {nullptr};
    for (int i = 0; i < nin; ++i) {
      if (!ins[i].in) continue;
      din[i] = cur;
      CUDA_TRY(cudaMemcpy2DAsync(cur, C * es, (const char*)ins[i].in + off, ld * es, n * es, ins[i].rows, cudaMemcpyHostToDevice, s));
      cur += (size_t)ins[i].rows * C * es;
    }
    for (int i = 0; i < nout; ++i) {
      if (!outs[i].out) continue;
      dout[i] = cur;
      cur += (size_t)outs[i].rows * C * es;
    }
    g_launch.kernels_launched = 0;
    if (int rc = launch_chunk(n, C, din, dout, s)) return rc;
    launches += g_launch.kernels_launched;
    last = g_launch;
    for (int i = 0; i < nout; ++i) {
      if (!outs[i].out) continue;
      CUDA_TRY(cudaMemcpy2DAsync((char*)outs[i].out + off, ld * es, dout[i], C * es, n * es, outs[i].rows, cudaMemcpyDeviceToHost, s));
    }
  }
  for (int i = 0; i < 3; ++i) CUDA_TRY(cudaStreamSynchronize(model->streams[i]));
  g_launch = last;
  g_launch.kernels_launched = launches;
  return RBD_OK;
}
}  // namespace

extern "C" {

int32_t rbd_version(void) { return RBD_B200_VERSION; }
const char* rbd_last_error(void) { return g_err.c_str(); }
const char* rbd_status_string(int32_t s) {
  switch (s) {
    case RBD_OK: return "RBD_OK";
    case RBD_EINVAL: return "RBD_EINVAL";
    case RBD_EDIM: return "RBD_EDIM";
    case RBD_ELOOP: return "RBD_ELOOP";
    case RBD_ESTALE: return "RBD_ESTALE";
    case RBD_ECUDA: return "RBD_ECUDA";
    case RBD_EUNSUPPORTED: return "RBD_EUNSUPPORTED";
    case RBD_ENOMEM: return "RBD_ENOMEM";
  }
  return "RBD_?";
}

int32_t rbd_model_create(const rbd_model_desc* desc, rbd_model** out) {
  if (!out) return fail(RBD_EINVAL, "rbd_model_create: out is NULL");
  *out = nullptr;
  rbd_model* m = new (std::nothrow) rbd_model();
  if (!m) return fail(RBD_ENOMEM, "out of memory");
  std::string err;
  int rc = build_host_model(desc, m->hm, err);
  if (rc != RBD_OK) { delete m; return fail(rc, err); }
  *out = m;
  return RBD_OK;
}

int32_t rbd_model_destroy(rbd_model* m) {
  if (!m) return RBD_OK;
  for (int i = 0; i < 3; ++i) {
    if (m->d_stage[i]) cudaFree(m->d_stage[i]);
    if (m->streams[i]) cudaStreamDestroy(m->streams[i]);
  }
  spec_release(m);
  if (m->side_stream) {
    cudaStreamDestroy(m->side_stream);
    for (int i = 0; i < kEventRing; ++i) { cudaEventDestroy(m->fork_ev[i]); cudaEventDestroy(m->join_ev[i]); }
    cudaFree(m->counters);
  }
  if (m->ev0) cudaEventDestroy(m->ev0);
  if (m->ev1) cudaEventDestroy(m->ev1);
  delete m;
  return RBD_OK;
}

int32_t rbd_model_get_info(const rbd_model* m, rbd_model_info* info) {
  if (!m || !info) return fail(RBD_EINVAL, "rbd_model_get_info: NULL argument");
  std::memset(info, 0, sizeof(*info));
  info->nb = m->hm.nb; info->nq = m->hm.nq; info->nv = m->hm.nv;
  info->stash_rows = m->hm.dev64.nrows;
  info->max_branch_depth = m->hm.nslots;
  info->general_path = m->hm.general ? 1 : 0;
  info->modcount = m->hm.modcount;
  for (int i = 0; i < m->hm.nb; ++i) {
    info->qstart[i] = m->hm.qstart[i];
    info->vstart[i] = m->hm.vstart[i];
    info->eval_order[i] = m->hm.order[i];
  }
  return RBD_OK;
}

int32_t rbd_model_check_modcount(const rbd_model* m, int64_t modcount) {
  if (!m) return fail(RBD_EINVAL, "model handle is NULL");
  if (m->hm.modcount != modcount)
    return fail(RBD_ESTALE, "ModificationCountMismatch: the Mechanism was modified after the model handle was created");
  return RBD_OK;
}

int32_t rbd_get_launch_info(rbd_launch_info* info) {
  if (!info) return fail(RBD_EINVAL, "rbd_get_launch_info: NULL argument");
  *info = g_launch;
  return RBD_OK;
}

int32_t rbd_model_precompile(rbd_model* model, int32_t dtype, int32_t what, int32_t load) {
  if (!model) return fail(RBD_EINVAL, "model handle is NULL");
  if (dtype != RBD_F32 && dtype != RBD_F64) return fail(RBD_EUNSUPPORTED, "rbd_model_precompile: fp32 / fp64 only");
  int rc_all = RBD_OK;
  std::string err;
  auto one = [&](int algo, bool in2, bool out1) {
    SpecKey key; key.algo = algo; key.f64 = dtype == RBD_F64; key.has_in2 = in2; key.has_out1 = out1;
    std::string e;
    const int rc = spec_prepare(model, key, load != 0, e);
    if (rc != RBD_OK) { rc_all = rc; err = e; }
  };
  if (what & RBD_SPEC_DYNAMICS) one(SPEC_ABA, true, false);
  if (what & RBD_SPEC_DYNAMICS_QDOT) one(SPEC_ABA, true, true);
  if (what & RBD_SPEC_DYNAMICS_NOTAU) { one(SPEC_ABA, false, false); one(SPEC_ABA, false, true); }
  if (what & RBD_SPEC_INVERSE_DYNAMICS) one(SPEC_RNEA, true, false);
  if (what & RBD_SPEC_DYNAMICS_BIAS) one(SPEC_RNEA, false, false);
  if (what & (RBD_SPEC_MASS_MATRIX | RBD_SPEC_MASS_MATRIX_LOWER)) {
    for (int lower = 0; lower < 2; ++lower) {
      if (!(what & (lower ? RBD_SPEC_MASS_MATRIX_LOWER : RBD_SPEC_MASS_MATRIX))) continue;
      SpecKey key; key.algo = SPEC_CRBA; key.f64 = dtype == RBD_F64; key.has_in2 = false; key.lower = lower != 0;
      std::string e;
      const int rc = spec_prepare(model, key, load != 0, e);
      if (rc != RBD_OK) { rc_all = rc; err = e; }
    }
  }
  if (what & RBD_SPEC_DYNAMICS_GATHER) {
    SpecKey key; key.algo = SPEC_ABA; key.f64 = dtype == RBD_F64; key.has_in2 = true; key.peers = true;
    std::string e;
    const int rc = spec_prepare(model, key, load != 0, e);
    if (rc != RBD_OK) { rc_all = rc; err = e; }
  }
  return rc_all == RBD_OK ? RBD_OK : fail(rc_all, err);
}

int32_t rbd_dynamics(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                     const void* tau, const void* wext, void* vd_out, void* qd_out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld, true)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !vd_out) return fail(RBD_EINVAL, "rbd_dynamics: q, v and vd_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == RBD_DUAL64X6) {
    if (wext || qd_out) return fail(RBD_EUNSUPPORTED, "RBD_DUAL64X6: external wrenches / q̇ output are not implemented");
    return dynamics_dual(model, B, ld, q, v, tau, vd_out, s);
  }
  return dtype == RBD_F32 ? dynamics_t<float>(model, B, ld, q, v, tau, wext, vd_out, qd_out, s)
                          : dynamics_t<double>(model, B, ld, q, v, tau, wext, vd_out, qd_out, s);
}

int32_t rbd_dynamics_gather(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                            const void* tau, int32_t npeers, void* const* vd_peers, void* vd_multicast, int64_t peer_ld, int64_t col0,
                            void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (npeers < 1 || npeers > 8 || !vd_peers) return fail(RBD_EINVAL, "rbd_dynamics_gather: need 1..8 peer arrays");
  for (int p = 0; p < npeers; ++p) if (!vd_peers[p]) return fail(RBD_EINVAL, "rbd_dynamics_gather: NULL peer array");
  if (col0 < 0 || peer_ld < col0 + B) return fail(RBD_EDIM, "rbd_dynamics_gather: columns [col0, col0 + B) exceed the gathered array");
  if (B == 0) return RBD_OK;
  if (!q || !v) return fail(RBD_EINVAL, "rbd_dynamics_gather: q and v must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? dynamics_gather_t<float>(model, B, ld, q, v, tau, npeers, vd_peers, vd_multicast, peer_ld, col0, s)
                          : dynamics_gather_t<double>(model, B, ld, q, v, tau, npeers, vd_peers, vd_multicast, peer_ld, col0, s);
}

int32_t rbd_integrate_schedule(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, void* q, void* v, const void* tau,
                               int64_t tau_step_stride, int64_t tau_stage_stride, double dt, int32_t nsteps, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  if (nsteps < 0 || !(dt > 0)) return fail(RBD_EINVAL, "rbd_integrate: need dt > 0 and nsteps >= 0");
  if (tau_step_stride < 0 || tau_stage_stride < 0) return fail(RBD_EINVAL, "rbd_integrate: torque strides must be >= 0");
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0 || nsteps == 0) return RBD_OK;
  if (!q || !v) return fail(RBD_EINVAL, "rbd_integrate: q and v must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? integrate_t<float>(model, B, ld, q, v, tau, tau_step_stride, tau_stage_stride, dt, nsteps, s)
                          : integrate_t<double>(model, B, ld, q, v, tau, tau_step_stride, tau_stage_stride, dt, nsteps, s);
}

int32_t rbd_integrate(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, void* q, void* v, const void* tau,
                      double dt, int32_t nsteps, void* stream) {
  return rbd_integrate_schedule(model, dtype, B, ld, q, v, tau, 0, 0, dt, nsteps, stream);
}

int32_t rbd_inverse_dynamics(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q,
                             const void* v, const void* vd, const void* wext, void* tau_out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !vd || !tau_out) return fail(RBD_EINVAL, "rbd_inverse_dynamics: q, v, vd and tau_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? inverse_dynamics_t<float>(model, B, ld, q, v, vd, wext, tau_out, s)
                          : inverse_dynamics_t<double>(model, B, ld, q, v, vd, wext, tau_out, s);
}

int32_t rbd_inverse_dynamics_bodies(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                                    const void* vd, const void* wext, void* accelerations_out, void* jointwrenches_out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0 || (!accelerations_out && !jointwrenches_out)) return RBD_OK;
  if (!q || !v) return fail(RBD_EINVAL, "rbd_inverse_dynamics_bodies: q and v must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? bodies_t<float>(model, B, ld, q, v, vd, wext, accelerations_out, jointwrenches_out, s)
                          : bodies_t<double>(model, B, ld, q, v, vd, wext, accelerations_out, jointwrenches_out, s);
}

int32_t rbd_contact_dynamics(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                             const rbd_contact_desc* contact, void* state, void* state_deriv_out, void* wrenches_out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (!contact) return fail(RBD_EINVAL, "rbd_contact_dynamics: contact must not be NULL");
  if (contact->npoints < 0 || contact->nhalfspaces < 0) return fail(RBD_EINVAL, "rbd_contact_dynamics: negative counts");
  if (contact->npoints > kMaxContactPoints || contact->nhalfspaces > kMaxHalfSpaces)
    return fail(RBD_EUNSUPPORTED, "rbd_contact_dynamics: at most 32 contact points and 4 half-spaces");
  if (contact->npoints && (!contact->body || !contact->location || !contact->normal_model || !contact->friction_model))
    return fail(RBD_EINVAL, "rbd_contact_dynamics: point arrays must not be NULL");
  if (contact->nhalfspaces && !contact->halfspace) return fail(RBD_EINVAL, "rbd_contact_dynamics: halfspace must not be NULL");
  for (int p = 0; p < contact->npoints; ++p) {
    if (contact->body[p] < 0 || contact->body[p] >= model->hm.nb) return fail(RBD_EINVAL, "rbd_contact_dynamics: body index out of range");
    if (!(contact->friction_model[3 * p + 2] > 0)) return fail(RBD_EINVAL, "rbd_contact_dynamics: friction damping b must be > 0");
  }
  for (int h = 0; h < contact->nhalfspaces; ++h) {
    const double* n = contact->halfspace + 6 * h + 3;
    if (!(n[0] * n[0] + n[1] * n[1] + n[2] * n[2] > 0)) return fail(RBD_EINVAL, "rbd_contact_dynamics: zero half-space normal");
  }
  if (B == 0) return RBD_OK;
  if (!q || !v || !wrenches_out) return fail(RBD_EINVAL, "rbd_contact_dynamics: q, v and wrenches_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? contact_t<float>(model, B, ld, q, v, *contact, state, state_deriv_out, wrenches_out, s)
                          : contact_t<double>(model, B, ld, q, v, *contact, state, state_deriv_out, wrenches_out, s);
}

int32_t rbd_dynamics_result(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                            const void* tau, const void* wext, void* vd_out, void* qd_out, void* M_out, void* c_out,
                            void* accelerations_out, void* jointwrenches_out, void* stream) {
  int rc = rbd_dynamics(model, dtype, B, ld, q, v, tau, wext, vd_out, qd_out, stream);
  if (rc != RBD_OK || B == 0) return rc;
  if (dtype == RBD_DUAL64X6 && (M_out || c_out || accelerations_out || jointwrenches_out))
    return fail(RBD_EUNSUPPORTED, "rbd_dynamics_result: by-products are fp32 / fp64 only");
  rbd_launch_info acc = g_launch;
  auto merge = [&]() { acc.kernels_launched += g_launch.kernels_launched; };
  if (c_out) { if ((rc = rbd_dynamics_bias(model, dtype, B, ld, q, v, wext, c_out, stream)) != RBD_OK) return rc; merge(); }
  if (M_out) { if ((rc = rbd_mass_matrix(model, dtype, B, ld, q, M_out, stream)) != RBD_OK) return rc; merge(); }
  if (accelerations_out || jointwrenches_out) {
    if ((rc = rbd_inverse_dynamics_bodies(model, dtype, B, ld, q, v, vd_out, wext, accelerations_out, jointwrenches_out, stream)) != RBD_OK) return rc;
    merge();
  }
  g_launch = acc;
  return RBD_OK;
}

int32_t rbd_dynamics_bias(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q,
                          const void* v, const void* wext, void* c_out, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !c_out) return fail(RBD_EINVAL, "rbd_dynamics_bias: q, v and c_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? inverse_dynamics_t<float>(model, B, ld, q, v, nullptr, wext, c_out, s)
                          : inverse_dynamics_t<double>(model, B, ld, q, v, nullptr, wext, c_out, s);
}

int32_t rbd_mass_matrix_uplo(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, void* M_out,
                             int32_t uplo, void* stream) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (uplo != RBD_UPLO_FULL && uplo != RBD_UPLO_LOWER) return fail(RBD_EINVAL, "rbd_mass_matrix: uplo must be RBD_UPLO_FULL or RBD_UPLO_LOWER");
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !M_out) return fail(RBD_EINVAL, "rbd_mass_matrix: q and M_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  const bool lower = uplo == RBD_UPLO_LOWER;
  return dtype == RBD_F32 ? mass_matrix_t<float>(model, B, ld, q, M_out, s, lower) : mass_matrix_t<double>(model, B, ld, q, M_out, s, lower);
}

int32_t rbd_mass_matrix(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, void* M_out,
                        void* stream) {
  return rbd_mass_matrix_uplo(model, dtype, B, ld, q, M_out, RBD_UPLO_FULL, stream);
}

int32_t rbd_dynamics_host(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                          const void* tau, const void* wext, void* vd_out, void* qd_out) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !vd_out) return fail(RBD_EINVAL, "rbd_dynamics_host: q, v and vd_out must not be NULL");
  const HostModel& hm = model->hm;
  const HostArr ins[4] = {{q, nullptr, hm.nq}, {v, nullptr, hm.nv}, {tau, nullptr, hm.nv}, {wext, nullptr, 6 * hm.nb}};
  const HostArr outs[2] = {{nullptr, vd_out, hm.nv}, {nullptr, qd_out, hm.nq}};
  return host_pipeline(model, dtype, B, ld, ins, 4, outs, 2,
                       [&](int64_t n, int64_t C, const void** di, void** dq, cudaStream_t s) {
                         return dtype == RBD_F32 ? dynamics_t<float>(model, n, C, di[0], di[1], di[2], di[3], dq[0], dq[1], s)
                                                 : dynamics_t<double>(model, n, C, di[0], di[1], di[2], di[3], dq[0], dq[1], s);
                       });
}

int32_t rbd_inverse_dynamics_host(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q,
                                  const void* v, const void* vd, const void* wext, void* tau_out) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !vd || !tau_out) return fail(RBD_EINVAL, "rbd_inverse_dynamics_host: q, v, vd and tau_out must not be NULL");
  const HostModel& hm = model->hm;
  const HostArr ins[4] = {{q, nullptr, hm.nq}, {v, nullptr, hm.nv}, {vd, nullptr, hm.nv}, {wext, nullptr, 6 * hm.nb}};
  const HostArr outs[1] = {{nullptr, tau_out, hm.nv}};
  return host_pipeline(model, dtype, B, ld, ins, 4, outs, 1,
                       [&](int64_t n, int64_t C, const void** di, void** dq, cudaStream_t s) {
                         return dtype == RBD_F32 ? inverse_dynamics_t<float>(model, n, C, di[0], di[1], di[2], di[3], dq[0], s)
                                                 : inverse_dynamics_t<double>(model, n, C, di[0], di[1], di[2], di[3], dq[0], s);
                       });
}

int32_t rbd_dynamics_bias_host(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q,
                               const void* v, const void* wext, void* c_out) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !v || !c_out) return fail(RBD_EINVAL, "rbd_dynamics_bias_host: q, v and c_out must not be NULL");
  const HostModel& hm = model->hm;
  const HostArr ins[3] = {{q, nullptr, hm.nq}, {v, nullptr, hm.nv}, {wext, nullptr, 6 * hm.nb}};
  const HostArr outs[1] = {{nullptr, c_out, hm.nv}};
  return host_pipeline(model, dtype, B, ld, ins, 3, outs, 1,
                       [&](int64_t n, int64_t C, const void** di, void** dq, cudaStream_t s) {
                         return dtype == RBD_F32 ? inverse_dynamics_t<float>(model, n, C, di[0], di[1], nullptr, di[2], dq[0], s)
                                                 : inverse_dynamics_t<double>(model, n, C, di[0], di[1], nullptr, di[2], dq[0], s);
                       });
}

int32_t rbd_mass_matrix_host(rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, void* M_out) {
  if (int rc = check_common(model, dtype, B, ld)) return rc;
  g_launch = {0, 0, 0, 0, 0, 0.f, 0};
  if (B == 0) return RBD_OK;      // empty batch: nothing to read or write, pointers may be NULL
  if (!q || !M_out) return fail(RBD_EINVAL, "rbd_mass_matrix_host: q and M_out must not be NULL");
  const HostModel& hm = model->hm;
  const HostArr ins[1] = {{q, nullptr, hm.nq}};
  const HostArr outs[1] = {{nullptr, M_out, hm.nv * hm.nv}};
  return host_pipeline(model, dtype, B, ld, ins, 1, outs, 1,
                       [&](int64_t n, int64_t C, const void** di, void** dq, cudaStream_t s) {
                         return dtype == RBD_F32 ? mass_matrix_t<float>(model, n, C, di[0], dq[0], s)
                                                 : mass_matrix_t<double>(model, n, C, di[0], dq[0], s);
                       });
}

}  // extern "C"
