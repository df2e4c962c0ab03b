// rbd_dynamics_derivatives: batched analytic dv̇/dq, dv̇/dv (csrc/rbd_deriv.cuh has the mathematics and the work split).
//
// Four kernels (after the forward dynamics itself) per chunk of the batch, all with the sample index fastest (lane l of a warp = sample b0 + l, so every global
// access of a warp is one fully used line) and warp-uniform control flow (the tree walk depends on the model only):
//   deriv_world_kernel   one thread per sample            root-frame S, Psi_dot, Psi_ddot, Sdp per coordinate; I, G, f per body
//   deriv_accum_kernel   one thread per (sample, 1 of 52) subtree sums of (I, G, f)
//   deriv_pairs_kernel   one thread per (sample, body)    d tau/dq, d tau/dv (into the output arrays) and M (into the scratch)
//   deriv_solve_kernel   one CTA per 32 samples (lane = sample), W warps: M of the 32 samples is staged in shared memory, factored
//                        there as L^T D L (tree sparsity) by the W warps together, then each warp solves its share of the 2 nv
//                        columns in place with its right-hand side in shared memory, [row][lane]
//   (deriv_factor_kernel one thread per sample, on the scratch: only when M does not fit into shared memory)
// Intermediates: a global scratch of DerivDev::rows rows per sample, allocated from the stream-ordered pool per call and
// bounded by RBD_DERIV_SCRATCH_MB (default 2048): larger batches are processed in chunks on the same stream.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../../include/rbd_b200.h"
// rbd_sincos.cuh defines one out-of-line __device__ function with external linkage (its text is also compiled by NVRTC, where
// `static` would be noise); this second translation unit of the library gets its own copy under another name
#define sincos_slow sincos_slow_deriv_tu
#include "rbd_deriv.cuh"
#include "rbd_deriv_jit.h"
#include "rbd_handle.h"
#include "rbd_jit.h"

using namespace rbd;

namespace {

constexpr int kNT = 128;

template <class T> struct DerivArgs {
  const T* q; const T* v; const T* vd;
  T* dq; T* dv;
  T* s;                 // scratch [rows][sld]
  int64_t ld, sld, C;   // C: samples in this chunk (all pointers already offset to the chunk's first sample)
};

template <class T, int NT>
__global__ void __launch_bounds__(NT) deriv_world_kernel(const __grid_constant__ ModelDev<T> M, const __grid_constant__ DerivDev D,
                                                         const DerivArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const Stash<T, NT> st{reinterpret_cast<T*>(smem_raw) + threadIdx.x};
  const int64_t ngroups = (a.C + NT - 1) / NT;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t b = g * NT + threadIdx.x;
    const bool active = b < a.C;
    const int64_t bl = active ? b : a.C - 1;
    DerivIO<T> io;
    io.q = {a.q + bl, a.ld};
    io.v = {a.v + bl, a.ld};
    io.vd = {a.vd + bl, a.ld};
    io.s = a.s + bl;
    io.sld = a.sld;
    io.active = active;
    deriv_world_sample<T>(M, D, io, st);
  }
}

template <class T, int NT>
__global__ void __launch_bounds__(NT) deriv_accum_kernel(const __grid_constant__ ModelDev<T> M, const __grid_constant__ DerivDev D,
                                                         const DerivArgs<T> a) {
  const int64_t b = (int64_t)blockIdx.x * NT + threadIdx.x;
  if (b >= a.C) return;
  deriv_accumulate<T>(M, D, a.s + b, a.sld, blockIdx.y);
}

// grid = (bodies, sample groups), bodies fastest: the CTAs that are resident together work on the SAME samples, so the per-coordinate
// rows a body shares with its relatives are served by L2 instead of being streamed from HBM once per body
template <class T, int NT>
__global__ void __launch_bounds__(NT) deriv_pairs_kernel(const __grid_constant__ DerivDev D, const __grid_constant__ DerivAnc A,
                                                         const DerivArgs<T> a) {
  const int64_t b = (int64_t)blockIdx.y * NT + threadIdx.x;
  if (b >= a.C) return;
  deriv_pairs<T>(D, A, a.s + b, a.sld, a.dq + b, a.dv + b, a.ld, blockIdx.x, true);
}

// only for models whose factor does not fit into shared memory next to the right-hand sides (deriv_solve_kernel<T, false>)
template <class T, int NT>
__global__ void __launch_bounds__(NT) deriv_factor_kernel(const __grid_constant__ DerivDev D, const __grid_constant__ DerivAnc A,
                                                          const DerivArgs<T> a) {
  const int64_t b = (int64_t)blockIdx.x * NT + threadIdx.x;
  if (b >= a.C) return;
  deriv_factor<T>(D, A, a.s + (int64_t)D.h_base * a.sld + b, a.sld);
}

// blockDim = (32, W): lane = sample, warp = column subset.  HS: M of the block's 32 samples is staged in shared memory, factored
// there by all W warps together (row k's updates of its ancestors' rows are independent of each other: warp w takes the
// ancestors at depth w, w + W, ...; two barriers per row) and then re-used by all 2 nv columns.  Otherwise the factor was made
// by deriv_factor_kernel and is read from the scratch.
template <class T, bool HS>
__global__ void deriv_solve_kernel(const __grid_constant__ DerivDev D, const __grid_constant__ DerivAnc A, const DerivArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sm = reinterpret_cast<T*>(smem_raw);
  const int lane = threadIdx.x, w = threadIdx.y, W = blockDim.y;
  const int nv = D.nv, nnz = D.nnz;
  T* Hs = sm + lane;
  T* xs = sm + (HS ? (size_t)nnz * 32 : 0) + (size_t)w * nv * 32 + lane;
  const int64_t ngroups = (a.C + 31) / 32;
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t b = g * 32 + lane;
    const bool active = b < a.C;
    const int64_t bl = active ? b : a.C - 1;
    const T* Hg = a.s + (int64_t)D.h_base * a.sld + bl;
    if (HS) {
      __syncthreads();      // the previous group's columns are done with Hs
      for (int r = w; r < nnz; r += W) Hs[r * 32] = Hg[(int64_t)r * a.sld];
      for (int k = nv - 1; k >= 0; --k) {
        const int rk = D.rowstart[k], dk = D.depth[k];
        __syncthreads();    // row k has received the updates of all its descendants
        const T inv = T(1) / Hs[(rk + dk) * 32];
        for (int di = w; di < dk; di += W) {
          const int ri = D.rowstart[A.anc[rk + di]];
          const T f = Hs[(rk + di) * 32] * inv;
          for (int d = di; d >= 0; --d) Hs[(ri + d) * 32] -= f * Hs[(rk + d) * 32];
        }
        __syncthreads();    // everybody has read row k
        for (int di = w; di < dk; di += W) Hs[(rk + di) * 32] *= inv;
        if (w == 0) Hs[(rk + dk) * 32] = inv;
      }
      __syncthreads();
    }
    for (int c = w; c < 2 * nv; c += W) {
      const int vj = c < nv ? c : c - nv;
      T* col = (c < nv ? a.dq : a.dv) + (int64_t)vj * nv * a.ld + bl;
      if (HS) {
        const T* Hl = Hs;
        deriv_solve_column<T>(D, A, [Hl](int row) { return Hl[row * 32]; }, xs, 32, col, a.ld, vj, active);
      } else {
        const int64_t sld = a.sld;
        deriv_solve_column<T>(D, A, [Hg, sld](int row) { return Hg[(int64_t)row * sld]; }, xs, 32, col, a.ld, vj, active);
      }
    }
  }
}

// ---- model-specialised solve kernel (rbd_deriv_jit.cpp): compiled with NVRTC on the first large call (or ahead of time by
// rbd_model_precompile_derivatives), cubin cached on disk, loaded once per (precision, device) and owned by the handle ----

// cubin for the model's solve kernel (from the cache, or compiled when `compile`); no GPU needed
bool jit_solve_cubin(const DerivDev& D, const DerivAnc& A, bool f64, bool compile, DerivJitPlan& plan, std::vector<char>& cubin,
                     std::string& err) {
  if (D.nnz * 32 * (f64 ? 8 : 4) > 200 * 1024) { err = "factor does not fit into shared memory"; return false; }
  if (!deriv_jit_plan(D, f64, plan)) { err = "too many velocity coordinates for a register-resident solve"; return false; }
  std::string src;
  deriv_jit_source(D, A, f64, plan, src);
  if (const char* dump = std::getenv("RBD_DERIV_DUMP")) {           // inspection: nvcc -cubin -Xptxas -v on the dumped text
    if (FILE* f = fopen((std::string(dump) + (f64 ? "_f64.cu" : "_f32.cu")).c_str(), "w")) { fwrite(src.data(), 1, src.size(), f); fclose(f); }
  }
  unsigned long long h = 1469598103934665603ull;            // FNV-1a of the text: the cache key
  for (unsigned char c : src) { h ^= c; h *= 1099511628211ull; }
  char name[64];
  snprintf(name, sizeof name, "%016llx_deriv_%s", h, f64 ? "f64" : "f32");
  return jit_cubin(name, true, compile, [&](std::string& s, std::string&) { s = std::move(src); return true; }, cubin, err);
}
DerivSolve* jit_solve_get(rbd_model* m, const DerivDev& D, const DerivAnc& A, bool f64, int64_t B, const DeviceProps& p) {
  const LaunchEnv& ev = launch_env();
  std::lock_guard<std::mutex> lk(m->spec_mu);
  DerivSolve& e = m->deriv[{f64, p.dev}];
  if (e.state == 1) return &e;
  if (e.state == -1) return nullptr;
  DerivJitPlan plan;
  std::vector<char> cubin;
  std::string err;
  if (!jit_solve_cubin(D, A, f64, B >= ev.deriv_jit_min_batch, plan, cubin, err)) {
    if (err != "no cached cubin") {
      e.state = -1;
      if (ev.jit_verbose) fprintf(stderr, "rbd_b200: derivative solve kernel not specialised: %s\n", err.c_str());
    }
    return nullptr;
  }
  e.warps = plan.warps;
  e.smem = (size_t)D.nnz * 32 * (f64 ? 8 : 4);
  cudaError_t ce = load_cubin(cubin, {{"rbd_deriv_solve", &e.kernel, e.smem, nullptr}}, e.lib);
  if (ce == cudaSuccess) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e.bps, (const void*)e.kernel, 32 * e.warps, e.smem);
  if (ce != cudaSuccess || e.bps < 1) {
    cudaGetLastError();
    if (ev.jit_verbose) fprintf(stderr, "rbd_b200: derivative solve kernel failed to load: %s\n", cudaGetErrorString(ce));
    if (e.lib) { cudaLibraryUnload(e.lib); e.lib = nullptr; }
    e.state = -1;
    return nullptr;
  }
  e.state = 1;
  return &e;
}

// The last launch's error, else its geometry goes into the launch statistics.
int launched(const char* name, int grid, int block, int smem_bytes, int blocks_per_sm) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return api_fail(RBD_ECUDA, std::string(name) + " launch failed: " + cudaGetErrorString(e));
  api_note_launch(grid, block, smem_bytes, blocks_per_sm);
  return RBD_OK;
}

template <class T>
int derivatives_t(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const T* q, const T* v, const T* tau, T* vd_out, T* dq,
                  T* dv, cudaStream_t stream) {
  // read on every call, unlike the LaunchEnv switches: tests and tools change them while the process runs
  const char* e_jit = std::getenv("RBD_DERIV_JIT");
  const char* e_mb = std::getenv("RBD_DERIV_SCRATCH_MB");
  const char* e_gf = std::getenv("RBD_DERIV_GLOBAL_FACTOR");
  const bool jit = launch_env().jit && !(e_jit && e_jit[0] == '0');
  const int64_t budget_mb = e_mb ? std::max<int64_t>(1, std::atoll(e_mb)) : 2048;
  const bool global_factor = e_gf && e_gf[0] == '1';        // tests: exercise the fallback
  const HostModel& hm = model->hm;
  const ModelDev<T>& M = dev_model<T>(hm);
  DerivDev D;
  DerivAnc A;
  if (!build_deriv_dev(M, D, A))
    return api_fail(RBD_EUNSUPPORTED, "rbd_dynamics_derivatives: more than 128 velocity coordinates or 4096 mass-matrix entries");
  if (D.nv == 0) return RBD_OK;        // nothing to differentiate (only fixed joints): no outputs have any rows
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  // chunk size from the scratch budget
  const int64_t per_sample = (int64_t)D.rows * (int64_t)sizeof(T);
  int64_t C = std::min<int64_t>(B, std::max<int64_t>(kNT, (budget_mb << 20) / per_sample / kNT * kNT));
  const int64_t sld = (C + 31) / 32 * 32;
  T* scratch = nullptr;
  if (cudaMallocAsync((void**)&scratch, (size_t)per_sample * sld, stream) != cudaSuccess) {
    cudaGetLastError();
    return api_fail(RBD_ENOMEM, "rbd_dynamics_derivatives: scratch allocation failed (lower RBD_DERIV_SCRATCH_MB)");
  }
  struct Guard { void* p; cudaStream_t s; ~Guard() { if (p) cudaFreeAsync(p, s); } } guard{scratch, stream};    // freed on every exit path
  // solve kernel geometry: warps per block so that factor + right-hand sides fit, maximising resident warps
  const size_t hbytes = (size_t)D.nnz * 32 * sizeof(T), xbytes = (size_t)D.nv * 32 * sizeof(T);
  int bestW = 0, bestNb = 0;
  bool hs = true;
  for (int nb = 1; nb <= 4; ++nb) {
    const int64_t avail = std::min<int64_t>(p.max_smem_optin, p.smem_per_sm / nb - 1024) - (int64_t)hbytes;
    if (avail < (int64_t)xbytes) continue;
    const int W = (int)std::min<int64_t>(std::min(16, 2 * D.nv), avail / (int64_t)xbytes);
    if (W * nb > bestW * bestNb) { bestW = W; bestNb = nb; }
  }
  if (global_factor) bestW = 0;
  if (bestW == 0) {       // factor too large for shared memory: read it from the scratch
    hs = false;
    bestW = (int)std::min<int64_t>(std::min(8, 2 * D.nv), p.max_smem_optin / (int64_t)xbytes);
    bestNb = 1;
  }
  DerivSolve* js = hs && jit ? jit_solve_get(const_cast<rbd_model*>(model), D, A, sizeof(T) == 8, B, p) : nullptr;
  const size_t solve_smem = (hs ? hbytes : 0) + (size_t)bestW * xbytes;
  const size_t world_smem = (size_t)std::max(1, kin_rows(hm)) * kNT * sizeof(T);
  auto kworld = deriv_world_kernel<T, kNT>;
  auto ksolve_s = deriv_solve_kernel<T, true>;
  auto ksolve_g = deriv_solve_kernel<T, false>;
  if (int rc = configure_once((const void*)kworld, p)) return rc;
  if (int rc = configure_once(hs ? (const void*)ksolve_s : (const void*)ksolve_g, p)) return rc;
  if (world_smem > (size_t)p.max_smem_optin) return api_fail(RBD_EUNSUPPORTED, "rbd_dynamics_derivatives: too many open branch nodes");
  for (int64_t b0 = 0; b0 < B; b0 += C) {
    const int64_t c = std::min<int64_t>(C, B - b0);
    T* vd = vd_out + b0;
    // v̇ itself: the library's own forward dynamics (model-specialised kernels when available)
    if (int rc = rbd_dynamics(model, dtype, c, ld, q + b0, v + b0, tau ? tau + b0 : nullptr, nullptr, vd, nullptr, stream)) return rc;
    DerivArgs<T> a{q + b0, v + b0, vd, dq + b0, dv + b0, scratch, ld, sld, c};
    const int gx = (int)((c + kNT - 1) / kNT);
    kworld<<<std::min(gx, 8 * p.sms), kNT, world_smem, stream>>>(M, D, a);
    if (int rc = launched("deriv_world_kernel", gx, kNT, (int)world_smem, 0)) return rc;
    deriv_accum_kernel<T, kNT><<<dim3(gx, kBodyRows), kNT, 0, stream>>>(M, D, a);
    if (int rc = launched("deriv_accum_kernel", gx * kBodyRows, kNT, 0, 0)) return rc;
    deriv_pairs_kernel<T, kNT><<<dim3(D.nb, gx), kNT, 0, stream>>>(D, A, a);
    if (int rc = launched("deriv_pairs_kernel", gx * D.nb, kNT, 0, 0)) return rc;
    if (!hs) {
      deriv_factor_kernel<T, kNT><<<gx, kNT, 0, stream>>>(D, A, a);
      if (int rc = launched("deriv_factor_kernel", gx, kNT, 0, 0)) return rc;
    }
    if (js) {
      const T* Hg = scratch + (int64_t)D.h_base * sld;
      long long sld_ = sld, ld_ = ld, c_ = c;
      T* dq_ = dq + b0; T* dv_ = dv + b0;
      void* params[] = {(void*)&Hg, (void*)&sld_, (void*)&dq_, (void*)&dv_, (void*)&ld_, (void*)&c_};
      const int sgj = (int)std::min<int64_t>((c + 31) / 32, (int64_t)js->bps * p.sms);
      cudaLaunchKernel((const void*)js->kernel, dim3(sgj), dim3(32 * js->warps), params, js->smem, stream);   // its error is also the last error
      if (int rc = launched("rbd_deriv_solve", sgj, 32 * js->warps, (int)js->smem, js->bps)) return rc;
      continue;
    }
    const int sg = (int)std::min<int64_t>((c + 31) / 32, (int64_t)bestNb * p.sms);
    if (hs) ksolve_s<<<sg, dim3(32, bestW), solve_smem, stream>>>(D, A, a);
    else ksolve_g<<<sg, dim3(32, bestW), solve_smem, stream>>>(D, A, a);
    if (int rc = launched("deriv_solve_kernel", sg, 32 * bestW, (int)solve_smem, bestNb)) return rc;
  }
  return RBD_OK;
}

}  // namespace

extern "C" int32_t rbd_dynamics_derivatives(const rbd_model* model, int32_t dtype, int64_t B, int64_t ld, const void* q, const void* v,
                                            const void* tau, void* vd_out, void* dvd_dq_out, void* dvd_dv_out, void* stream) {
  if (int rc = api_check(model, dtype, B, ld)) return rc;
  if (B == 0) return RBD_OK;
  if (!q || !v || !vd_out || !dvd_dq_out || !dvd_dv_out)
    return api_fail(RBD_EINVAL, "rbd_dynamics_derivatives: q, v, vd_out, dvd_dq_out and dvd_dv_out must not be NULL");
  cudaStream_t s = (cudaStream_t)stream;
  return dtype == RBD_F32 ? derivatives_t<float>(model, dtype, B, ld, (const float*)q, (const float*)v, (const float*)tau, (float*)vd_out,
                                                 (float*)dvd_dq_out, (float*)dvd_dv_out, s)
                          : derivatives_t<double>(model, dtype, B, ld, (const double*)q, (const double*)v, (const double*)tau,
                                                  (double*)vd_out, (double*)dvd_dq_out, (double*)dvd_dv_out, s);
}

// Ahead-of-time compilation of the model's solve kernel into the cubin cache (no GPU needed): the analogue of rbd_model_precompile
// for this entry point.  RBD_EUNSUPPORTED if NVRTC is missing or the model does not qualify (the generic kernel then serves it).
extern "C" int32_t rbd_model_precompile_derivatives(rbd_model* model, int32_t dtype) {
  if (!model) return api_fail(RBD_EINVAL, "model handle is NULL");
  if (dtype != RBD_F32 && dtype != RBD_F64) return api_fail(RBD_EINVAL, "rbd_model_precompile_derivatives: fp32 / fp64 only");
  DerivDev D;
  DerivAnc A;
  if (!build_deriv_dev(model->hm.dev64, D, A)) return api_fail(RBD_EUNSUPPORTED, "model too large for rbd_dynamics_derivatives");
  DerivJitPlan plan;
  std::vector<char> cubin;
  std::string err;
  if (!jit_solve_cubin(D, A, dtype == RBD_F64, true, plan, cubin, err)) return api_fail(RBD_EUNSUPPORTED, err);
  return RBD_OK;
}
