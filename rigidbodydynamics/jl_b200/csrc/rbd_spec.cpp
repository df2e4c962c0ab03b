// Model-specialised kernels: compile (rbd_jit.cpp), load (cudaLibraryLoadData) and launch.  Host-only C++ on the CUDA runtime.
//
// The kernels come as a pair, exactly like the generic ones in rbd_b200.cu: single-warp shared-memory blocks on the caller's
// stream and one Tensor-Memory CTA per SM on the handle's side stream, both claiming groups of 32 samples from one counter.
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "rbd_handle.h"
#include "rbd_jit.h"

namespace rbd {

cudaError_t pair_begin(rbd_model* m, cudaStream_t stream, PairCtx& ctx) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  unsigned slot;
  {
    std::lock_guard<std::mutex> lk(m->side_mu);
    if (m->side_device != dev) {       // first use (or the caller moved to another device): (re)create the per-device resources
      if (m->side_stream) {
        cudaStreamDestroy(m->side_stream);
        for (int i = 0; i < kEventRing; ++i) { cudaEventDestroy(m->fork_ev[i]); cudaEventDestroy(m->join_ev[i]); }
        cudaFree(m->counters);
        m->side_stream = nullptr; m->counters = nullptr;
      }
      if ((e = cudaStreamCreateWithFlags(&m->side_stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
      for (int i = 0; i < kEventRing; ++i) {
        if ((e = cudaEventCreateWithFlags(&m->fork_ev[i], cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&m->join_ev[i], cudaEventDisableTiming)) != cudaSuccess) return e;
      }
      if ((e = cudaMalloc((void**)&m->counters, kCounterRing * 2 * sizeof(unsigned long long))) != cudaSuccess) return e;
      m->side_device = dev;
    }
    slot = m->next_call++;
  }
  ctx.side = m->side_stream;
  ctx.fork = m->fork_ev[slot % kEventRing];
  ctx.join = m->join_ev[slot % kEventRing];
  ctx.counter = m->counters + 2 * (slot % kCounterRing);
  ctx.flag = reinterpret_cast<int*>(ctx.counter + 1);
  return cudaMemsetAsync(ctx.counter, 0, 2 * sizeof(unsigned long long), stream);
}

void spec_release(rbd_model* m) {
  std::lock_guard<std::mutex> lk(m->spec_mu);
  for (auto& kv : m->spec) if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
  m->spec.clear();
  for (auto& kv : m->deriv) if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
  m->deriv.clear();
}

cudaError_t load_cubin(const std::vector<char>& cubin, std::initializer_list<CubinKernel> kernels, cudaLibrary_t& lib) {
  lib = nullptr;
  cudaError_t e = cudaLibraryLoadData(&lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
  for (const CubinKernel& k : kernels) {
    if (e == cudaSuccess) e = cudaLibraryGetKernel(k.kernel, lib, k.name);
    cudaFuncAttributes fa{};
    if (e == cudaSuccess && k.regs) { e = cudaFuncGetAttributes(&fa, (const void*)*k.kernel); *k.regs = fa.numRegs; }
    if (e == cudaSuccess && k.smem > 0) e = cudaFuncSetAttribute((const void*)*k.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute((const void*)*k.kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    if (lib) { cudaLibraryUnload(lib); lib = nullptr; }
  }
  return e;
}

namespace {
// The cubin of (model, key), cached as <content hash>_<algo>_<f32|f64>_<flags>.cubin; the source is generated on a cache miss only.
bool spec_cubin(const HostModel& hm, const SpecKey& k, bool compile_if_missing, std::vector<char>& cubin, std::string& err) {
  char name[96];
  const char* algo = k.algo == SPEC_ABA ? "aba" : (k.algo == SPEC_RNEA ? "rnea" : (k.algo == SPEC_CRBA ? "crba" : "kin"));
  snprintf(name, sizeof name, "%016llx_%s_%s_%d%d%d%s", (unsigned long long)spec_hash(hm, k), algo, k.f64 ? "f64" : "f32",
           (int)k.has_in2, (int)k.has_out1, (int)k.lower, k.peers ? "p" : "");
  return jit_cubin(name, false, compile_if_missing,
                   [&](std::string& src, std::string& e) { return spec_emit_cuda_tu(hm, k, src, nullptr, e); }, cubin, err);
}
}  // namespace

// Straight-line programs far beyond the instruction caches run at the SM's instruction-fetch rate (~1.4 instr/clk on B200)
// instead of its issue rate; measured against the generic (looping, cache-resident) kernels on Atlas: fp32 ABA 12.7 k nodes
// 1.03x, fp32 RNEA 5.8 k nodes 1.46x, 7-DoF arm 2.2 k nodes 2.7x, but fp64 ABA 0.83x (half the resident warps).  fp32 programs
// are therefore always specialised, fp64 programs only below an estimated size.
bool spec_worthwhile(const HostModel& hm, const SpecKey& key) {
  if (!key.f64) return true;
  if (key.algo == SPEC_CRBA) return true;   // small stash (2 rows per body): fp64 keeps its resident warps
  if (key.algo == SPEC_KIN) return true;    // stash = the pending branch nodes only
  const int est = hm.nb * (key.algo == SPEC_ABA ? 410 : 190);
  return est <= 6500;
}

int spec_prepare(rbd_model* m, const SpecKey& key, bool load_on_device, std::string& err) {
  std::lock_guard<std::mutex> lk(m->spec_mu);
  SpecEntry& se = m->spec[spec_key_bits(key)];
  if (se.state == 1) return RBD_OK;
  if (se.state == -1 && load_on_device) { err = se.why; return RBD_EUNSUPPORTED; }
  std::vector<char> cubin;
  if (!spec_cubin(m->hm, key, true, cubin, err)) {
    se.state = -1; se.why = err;
    return RBD_EUNSUPPORTED;
  }
  if (!load_on_device) return RBD_OK;      // precompile only (CPU build step): the cubin is in the cache now
  se.rows = spec_stash_rows(m->hm, key);
  const size_t smem = (size_t)std::max(1, se.rows) * 32 * (key.f64 ? 8 : 4);
  se.uni_sw = spec_uni_smem_warps(m->hm, key);
  const cudaError_t e = load_cubin(cubin, {{"rbd_jit_smem", &se.k_smem, smem, &se.regs_smem},
                                           {"rbd_jit_tmem", &se.k_tmem, 0, &se.regs_tmem},
                                           {"rbd_jit_uni", &se.k_uni, se.uni_sw > 0 ? smem * se.uni_sw : 0, &se.regs_uni}}, se.lib);
  if (e != cudaSuccess) {
    se.state = -1;
    se.why = err = std::string("loading the specialised cubin: ") + cudaGetErrorString(e);
    return RBD_EUNSUPPORTED;
  }
  se.state = 1;
  return RBD_OK;
}

int spec_try_launch(rbd_model* m, const SpecKey& key, const SpecLaunchArgs& a, cudaStream_t stream, bool& used,
                    rbd_launch_info& li, const int** gate) {
  used = false;
  if (gate) *gate = nullptr;
  const LaunchEnv& ev = launch_env();
  if (!ev.jit || !spec_worthwhile(m->hm, key)) return RBD_OK;
  if (a.ld * (key.f64 ? 8 : 4) >= (1ll << 32)) return RBD_OK;   // the generated code forms row offsets as 32 x 32 -> 64-bit products of the byte stride
  const int rows = spec_stash_rows(m->hm, key);
  if (rows > 256) return RBD_OK;                     // one warp's share of Tensor Memory: 256 fp32 rows (128 x 2 columns in fp64)
  DeviceProps p;
  if (int rc = get_props(p)) return rc;
  const size_t es = key.f64 ? 8 : 4;
  const size_t smem = (size_t)std::max(1, rows) * 32 * es;
  if (smem > (size_t)p.max_smem_optin) return RBD_OK;
  SpecEntry* se = nullptr;
  {
    std::lock_guard<std::mutex> lk(m->spec_mu);
    se = &m->spec[spec_key_bits(key)];
  }
  if (key.algo == SPEC_KIN) {        // the 64-bit map key carries only a hash of the jacobian path: use the entry only for ITS path
    std::lock_guard<std::mutex> lk(m->spec_mu);
    if (!se->kin_set) { std::memcpy(se->kin_sign, key.kin_sign, sizeof se->kin_sign); se->kin_set = true; }
    else if (std::memcmp(se->kin_sign, key.kin_sign, sizeof se->kin_sign) != 0) return RBD_OK;
  }
  if (se->state == -1) return RBD_OK;
  if (se->state == 0) {
    if (a.B < ev.jit_min_batch) {          // small call and nothing loaded yet: use a cached cubin if there is one, never compile
      std::vector<char> probe;
      std::string e2;
      if (!spec_cubin(m->hm, key, false, probe, e2)) return RBD_OK;
    }
    std::string e2;
    if (spec_prepare(m, key, true, e2) != RBD_OK) {      // generic kernels take over; the reason is kept in the entry
      if (ev.jit_verbose) fprintf(stderr, "[rbd_b200] specialised kernels unavailable: %s\n", e2.c_str());
      return RBD_OK;
    }
  }
  const int64_t ngroups = (a.B + 31) / 32;
  const int tm_warps = key.f64 ? 4 : 8;
  int bps = 0;
  if (cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, (const void*)se->k_smem, 32, smem))
    return api_fail(RBD_ECUDA, cudaGetErrorString(e));
  if (bps < 1) return RBD_OK;
  // Three ways to fill an SM (rbd_jit_kernels.cuh): shared-memory blocks alone, the kernel pair, the unified CTA.  The two
  // Tensor-Memory variants are used when they put at least 15 % more warps on the SM than shared memory alone and there is work
  // for them; which of the two is decided by timing both once, on the first call large enough to tell (not while capturing).
  const int bps_pair = ev.no_tmem ? 0 : pair_blocks(p.sms, bps, se->regs_smem, se->regs_tmem, tm_warps, ngroups);
  const bool pair_ok = bps_pair > 0;
  const int uni_warps = se->uni_sw > 0 ? se->uni_sw + tm_warps : 0;
  const bool uni_ok = !ev.no_tmem && uni_warps * 100 >= bps * 115 && ((se->regs_uni + 7) / 8) * 8 * 32 * uni_warps <= 65536 &&
                      ngroups >= (int64_t)(uni_warps - tm_warps / 2) * p.sms;
  struct KArgs {
    const void* q; const void* v; const void* in2; void* o0; void* o1; long long ld, B; unsigned long long* counter; int* flag;
    void* peers[8]; long long peer_ld, peer_col0; void* mc; int npeers;
    void* ko[8];
  };
  int launched = 0;
  int* last_flag = nullptr;
  auto run = [&](int variant) -> cudaError_t {        // 0 = shared memory alone, 1 = pair, 2 = unified
    PairCtx ctx;
    cudaError_t e = pair_begin(m, stream, ctx);
    if (e != cudaSuccess) return e;
    KArgs ka = {a.q, a.v, a.in2, a.o0, a.o1, (long long)a.ld, (long long)a.B, ctx.counter, ctx.flag, {}, (long long)a.peer_ld,
                (long long)a.peer_col0, a.mc, a.npeers};
    for (int i = 0; i < a.npeers && i < 8; ++i) ka.peers[i] = a.peers[i];
    for (int i = 0; i < 8; ++i) ka.ko[i] = a.ko[i];
    void* params[] = {&ka};
    if (variant == 2) {
      e = cudaLaunchKernel((const void*)se->k_uni, dim3(p.sms), dim3(32 * uni_warps), params, smem * se->uni_sw, stream);
      ++launched;
      li.grid = p.sms; li.block = 32 * uni_warps; li.blocks_per_sm = 1; li.smem_bytes = (int)(smem * se->uni_sw);
    } else if (variant == 1) {
      e = cudaEventRecord(ctx.fork, stream);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx.side, ctx.fork, 0);
      if (e == cudaSuccess && (!ev.only || ev.only[0] == 's')) { e = cudaLaunchKernel((const void*)se->k_smem, dim3(bps_pair * p.sms), dim3(32), params, smem, stream); ++launched; }
      if (e == cudaSuccess && (!ev.only || ev.only[0] == 't')) { e = cudaLaunchKernel((const void*)se->k_tmem, dim3(p.sms), dim3(32 * tm_warps), params, 0, ctx.side); ++launched; }
      if (e == cudaSuccess) e = cudaEventRecord(ctx.join, ctx.side);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, ctx.join, 0);
      li.grid = bps_pair * p.sms; li.block = 32; li.blocks_per_sm = bps_pair; li.smem_bytes = (int)smem;
    } else {
      const int grid = (int)std::min<int64_t>(ngroups, (int64_t)bps * p.sms);
      e = cudaLaunchKernel((const void*)se->k_smem, dim3(grid), dim3(32), params, smem, stream);
      ++launched;
      li.grid = grid; li.block = 32; li.blocks_per_sm = bps; li.smem_bytes = (int)smem;
    }
    last_flag = ctx.flag;
    return e;
  };
  cudaError_t e = cudaSuccess;
  int variant = 0;
  if (pair_ok && uni_ok) {
    variant = ev.jit_variant ? ev.jit_variant : se->choice;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &cap);
    if (variant == 0 && cap == cudaStreamCaptureStatusNone && a.B >= (int64_t)p.sms * 32 * 64) {
      // tune: each variant once to warm up, then timed; outputs are simply overwritten with the same values
      float best = 0.f;
      cudaEvent_t t0, t1;
      cudaEventCreate(&t0); cudaEventCreate(&t1);
      for (int v = 1; v <= 2 && e == cudaSuccess; ++v) {
        e = run(v);
        if (e == cudaSuccess) e = cudaEventRecord(t0, stream);
        if (e == cudaSuccess) e = run(v);
        if (e == cudaSuccess) e = cudaEventRecord(t1, stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(t1);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, t0, t1);
        if (e == cudaSuccess && (variant == 0 || ms < best)) { best = ms; variant = v; }
      }
      cudaEventDestroy(t0); cudaEventDestroy(t1);
      if (e == cudaSuccess) se->choice = variant;
      launched = 0;
    }
    if (variant == 0) variant = 1;
  } else if (uni_ok) variant = 2;
  else if (pair_ok) variant = 1;
  if (e == cudaSuccess) e = run(variant);
  if (e != cudaSuccess) return api_fail(RBD_ECUDA, std::string("specialised kernel launch: ") + cudaGetErrorString(e));
  li.kernels_launched += launched;
  if (gate && !key.f64 && !ev.no_gate) *gate = last_flag;
  used = true;
  return RBD_OK;
}

}  // namespace rbd
