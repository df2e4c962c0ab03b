// The opaque model handle of the C ABI (include/rbd_b200.h), shared by rbd_b200.cu (generic kernels, entry points),
// rbd_spec.cpp (model-specialised kernels) and rbd_deriv.cu (derivatives), with the launch plumbing they have in common.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../../include/rbd_b200.h"
#include "rbd_codegen.h"
#include "rbd_model.h"

namespace rbd {

// One model-specialised kernel pair (shared-memory + Tensor-Memory stash), loaded from a cubin.
struct SpecEntry {
  int state = 0;                 // 0 = not tried, 1 = ready, -1 = unavailable (generic kernels are used)
  cudaLibrary_t lib = nullptr;
  cudaKernel_t k_smem = nullptr, k_tmem = nullptr, k_uni = nullptr;   // shared-memory blocks / Tensor-Memory CTA / unified CTA
  int regs_smem = 0, regs_tmem = 0, regs_uni = 0;
  int choice = 0;                // 0 = not tuned yet, 1 = kernel pair, 2 = unified CTA (for batches that fill the SMs)
  int uni_sw = 0;                // warps with a shared-memory stash in the unified CTA (0 = unified kernel unusable)
  int rows = 0;
  std::string why;               // reason for state -1
  int8_t kin_sign[kMaxBodies] = {0};   // SPEC_KIN: the path this entry was generated for
  bool kin_set = false;
};

// The model-specialised solve kernel of rbd_dynamics_derivatives (rbd_deriv.cu), loaded for one precision on one device.
struct DerivSolve {
  int state = 0;                 // 0 = not loaded yet, 1 = ready, -1 = unavailable (the table-driven solve kernel is used)
  cudaLibrary_t lib = nullptr;
  cudaKernel_t kernel = nullptr;
  int warps = 0;                 // warps per CTA
  size_t smem = 0;               // dynamic shared memory per CTA
  int bps = 0;                   // resident CTAs per SM
};

constexpr int kCounterRing = 256;   // work-queue counters, one per call in flight
constexpr int kEventRing = 8;

}  // namespace rbd

struct rbd_model {
  rbd::HostModel hm;
  // staging for the *_host entry points (allocated on first use, owned by the handle)
  std::mutex host_mu;
  void* d_stage[3] = {nullptr, nullptr, nullptr};
  size_t stage_bytes = 0;
  cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // kernel pairs: the Tensor-Memory kernel runs on the side stream next to the shared-memory kernel (per device)
  std::mutex side_mu;
  int side_device = -1;
  cudaStream_t side_stream = nullptr;
  cudaEvent_t fork_ev[rbd::kEventRing] = {}, join_ev[rbd::kEventRing] = {};
  unsigned long long* counters = nullptr;     // [kCounterRing][2] device memory: work-queue counter, "needs generic kernel" flag
  unsigned next_call = 0;
  // model-specialised kernels, keyed by SpecKey bits, and the derivatives' solve kernel, keyed by (fp64, device)
  std::mutex spec_mu;
  std::map<uint64_t, rbd::SpecEntry> spec;
  std::map<std::pair<bool, int>, rbd::DerivSolve> deriv;
};

namespace rbd {

// Resources of one kernel-pair launch: side stream, fork/join events and a zeroed work-queue counter (enqueued on `stream`).
struct PairCtx {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  unsigned long long* counter = nullptr;
  int* flag = nullptr;       // zeroed with the counter; raised by a specialised kernel that met an angle beyond its fast sin / cos
};
// Returns a cudaError_t (cudaSuccess = 0).
cudaError_t pair_begin(rbd_model* m, cudaStream_t stream, PairCtx& ctx);

inline uint64_t spec_key_bits(const SpecKey& k) {
  uint64_t b = (uint64_t)k.algo | (k.f64 ? 8u : 0u) | (k.has_in2 ? 16u : 0u) | (k.has_out1 ? 32u : 0u) | (k.lower ? 64u : 0u) | (k.peers ? 128u : 0u);
  if (k.algo == SPEC_KIN) {      // output subset and jacobian path: 8 mask bits + a 40-bit hash of the path signs (the entry keeps the
    uint64_t h = 1469598103934665603ull;   // signs themselves and is only used when they match, see spec_try_launch)
    for (int i = 0; i < kMaxBodies; ++i) { h ^= (uint8_t)k.kin_sign[i]; h *= 1099511628211ull; }
    b |= ((uint64_t)(k.kin_mask & 0xff) << 8) | ((h >> 24) << 24);
  }
  return b;
}

struct SpecLaunchArgs {
  const void* q; const void* v; const void* in2;
  void* o0; void* o1;
  int64_t ld, B;
  // key.peers: o0 is unused; row k of sample b goes to peers[p][k * peer_ld + peer_col0 + b] for every p < npeers
  void* const* peers = nullptr;
  void* mc = nullptr;            // NVLS multicast mapping of the peers' arrays, or NULL
  int npeers = 0;
  int64_t peer_ld = 0, peer_col0 = 0;
  void* ko[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // SPEC_KIN: the rbd_kinematics_out pointers
};
// Tries the model-specialised kernels for (model, key).  `used` = false (and RBD_OK) when they are unavailable, not yet
// compiled and the batch is below the compile threshold, or the batch is too small: the caller then runs the generic kernels.
// `gate` (fp32 only, else NULL): device flag the specialised kernels raise when a sample needs the library sin / cos; the caller
// must enqueue the generic kernel gated on it right behind.  Errors are reported through api_fail.
int spec_try_launch(rbd_model* m, const SpecKey& key, const SpecLaunchArgs& a, cudaStream_t stream, bool& used,
                    rbd_launch_info& li, const int** gate);
// Compile (or load from the cubin cache) without launching; RBD_OK / RBD_EUNSUPPORTED.
int spec_prepare(rbd_model* m, const SpecKey& key, bool load_on_device, std::string& err);
// Unloads the handle's model-specialised kernels and derivative solve kernels.
void spec_release(rbd_model* m);

// One kernel of a cubin for load_cubin: its name, where its handle goes, the dynamic shared memory it is opted into (0: the
// default) and, when `regs` is not NULL, where its registers per thread go.
struct CubinKernel { const char* name; cudaKernel_t* kernel; size_t smem; int* regs; };
// Loads `cubin`, looks up its kernels and gives each of them the largest shared-memory carve-out.  On failure the error is
// cleared, nothing stays loaded and `lib` is NULL.
cudaError_t load_cubin(const std::vector<char>& cubin, std::initializer_list<CubinKernel> kernels, cudaLibrary_t& lib);

// Launch switches (DESIGN.md §4.7), read once per process.
struct LaunchEnv {
  bool jit = true;                  // RBD_JIT=0: generic kernels only
  int64_t jit_min_batch = 1 << 15;  // below this a missing cubin is not compiled on the fly (generic kernels serve the call)
  int64_t deriv_jit_min_batch = 4096;   // the same for rbd_dynamics_derivatives' solve kernel (RBD_JIT_MIN_BATCH sets both)
  int jit_variant = 0;              // RBD_JIT_VARIANT=1 (pair) / 2 (unified): skip the tuning
  bool jit_verbose = false;         // RBD_JIT_VERBOSE: print why a specialised kernel is unavailable
  bool no_tmem = false;             // RBD_NO_TMEM: single-kernel paths only
  bool no_gate = false;             // RBD_NO_GATE: no generic kernel behind the fp32 specialised ones (profile captures)
  const char* only = nullptr;       // RBD_ONLY=smem|tmem: launch one kernel of a pair (ncu captures: the profiler serialises them)
  LaunchEnv() {
    if (const char* e = getenv("RBD_JIT")) jit = e[0] != '0';
    if (const char* e = getenv("RBD_JIT_MIN_BATCH")) {
      jit_min_batch = atoll(e);
      deriv_jit_min_batch = jit_min_batch > 1 ? jit_min_batch : 1;
    }
    if (const char* e = getenv("RBD_JIT_VARIANT")) jit_variant = atoi(e);
    jit_verbose = getenv("RBD_JIT_VERBOSE") != nullptr;
    no_tmem = getenv("RBD_NO_TMEM") != nullptr;
    no_gate = getenv("RBD_NO_GATE") != nullptr;
    only = getenv("RBD_ONLY");
  }
};
inline const LaunchEnv& launch_env() { static const LaunchEnv e; return e; }

// Properties of the current device, cached per device.  The first query on a device also keeps freed blocks cached in its
// stream-ordered memory pool (scratch for slots / external wrenches comes from there).
struct DeviceProps { int dev = 0; int sms = 0; int max_smem_optin = 0; int smem_per_sm = 0; bool ok = false; };
int get_props(DeviceProps& p);
// Opt a kernel into large dynamic shared memory ONCE per (kernel, device): the attribute is process-global per kernel, so
// setting it to each call's exact size would race between host threads using different model handles.
int configure_once(const void* kernel, const DeviceProps& p);
// Blocks per SM of a single-warp shared-memory kernel running next to one Tensor-Memory CTA of `tm_warps` warps on every SM,
// or 0 when that kernel pair should not be used.  `bps`: the shared-memory kernel's blocks per SM on its own; `regs_*`: the
// two kernels' registers per thread; `ngroups`: groups of 32 samples in the batch.
int pair_blocks(int sms, int bps, int regs_smem, int regs_tmem, int tm_warps, int64_t ngroups);

// rbd_b200.cu's per-thread error text / argument checks / launch statistics, for the library's other translation units
int api_fail(int status, const std::string& msg);
int api_check(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld);
void api_note_launch(int grid, int block, int smem_bytes, int blocks_per_sm);

}  // namespace rbd
