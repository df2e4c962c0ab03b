// Run-time compilation of the library's generated kernels (rbd_codegen.cpp, rbd_deriv_jit.cpp) with NVRTC, plus an on-disk
// cubin cache.  NVRTC is dlopen'ed on first use (librbd_b200.so has no link-time dependency on it); compilation needs no GPU, so
// `rbd_model_precompile` also runs in the CPU-only build step and the cubins travel with the source tree.
#pragma once
#include <functional>
#include <string>
#include <vector>

namespace rbd {

// Fetches <name>.cubin from the cache directory or, when it is not there and `compile_if_missing`, compiles the text `source`
// writes (called only then) for sm_100a and stores the cubin in the cache.  fmad = false compiles with --fmad=false.  Returns false
// with `err` set when the cubin is not cached and not to be compiled ("no cached cubin"), `source` fails, NVRTC is unavailable or
// compilation fails.
bool jit_cubin(const std::string& name, bool fmad, bool compile_if_missing,
               const std::function<bool(std::string& src, std::string& err)>& source, std::vector<char>& cubin, std::string& err);

// Directory of the cubin cache: $RBD_JIT_CACHE, else <directory of librbd_b200.so>/jit_cache, else ~/.cache/rbd_b200.
std::string jit_cache_dir();

}  // namespace rbd
