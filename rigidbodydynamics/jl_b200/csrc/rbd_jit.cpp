// NVRTC front end + cubin cache for the library's generated kernels (see rbd_jit.h).  Host-only C++.
#include "rbd_jit.h"

#include <dlfcn.h>
#include <nvrtc.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace rbd {
namespace {

// headers of the NVRTC translation units, embedded at build time (Makefile: rbd_jit_embed.inc)
struct EmbeddedHeader { const char* name; const char* text; };
#include "rbd_jit_embed.inc"

struct Nvrtc {
  void* h = nullptr;
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
  const char* (*GetErrorString)(nvrtcResult) = nullptr;
  std::string err;
};

Nvrtc& nvrtc() {
  static Nvrtc n;
  static std::once_flag once;
  std::call_once(once, [] {
    // the toolkit's own NVRTC first (by path): by soname dlopen would hand back whatever libnvrtc.so.12 the process has
    // already loaded (PyTorch bundles an older one)
    const char* names[] = {"/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so", "libnvrtc.so.12", "libnvrtc.so"};
    for (const char* nm : names) {
      n.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
      if (n.h) break;
    }
    if (!n.h) { n.err = "NVRTC (libnvrtc.so.12) not found"; return; }
#define RBD_SYM(f) n.f = (decltype(n.f))dlsym(n.h, "nvrtc" #f); if (!n.f) { n.err = "NVRTC symbol nvrtc" #f " missing"; n.h = nullptr; return; }
    RBD_SYM(CreateProgram) RBD_SYM(DestroyProgram) RBD_SYM(CompileProgram) RBD_SYM(GetCUBINSize) RBD_SYM(GetCUBIN)
    RBD_SYM(GetProgramLogSize) RBD_SYM(GetProgramLog) RBD_SYM(GetErrorString)
#undef RBD_SYM
  });
  return n;
}

bool dir_writable(const std::string& d) {
  mkdir(d.c_str(), 0755);
  return access(d.c_str(), W_OK | X_OK) == 0;
}

bool read_file(const std::string& path, std::vector<char>& out) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  out.resize(n > 0 ? (size_t)n : 0);
  const bool ok = n > 0 && fread(out.data(), 1, (size_t)n, f) == (size_t)n;
  fclose(f);
  return ok;
}

void write_file_atomic(const std::string& path, const char* data, size_t n) {
  char tmp[32];
  snprintf(tmp, sizeof tmp, ".tmp%d", (int)getpid());
  const std::string t = path + tmp;
  FILE* f = fopen(t.c_str(), "wb");
  if (!f) return;
  const bool ok = fwrite(data, 1, n, f) == n;
  fclose(f);
  if (ok) rename(t.c_str(), path.c_str()); else remove(t.c_str());
}

}  // namespace

std::string jit_cache_dir() {
  if (const char* e = getenv("RBD_JIT_CACHE")) { if (dir_writable(e)) return e; }
  Dl_info info;
  if (dladdr((void*)&jit_cache_dir, &info) && info.dli_fname) {
    std::string p(info.dli_fname);
    const size_t s = p.find_last_of('/');
    const std::string d = (s == std::string::npos ? std::string(".") : p.substr(0, s)) + "/jit_cache";
    if (dir_writable(d)) return d;
  }
  if (const char* home = getenv("HOME")) {
    const std::string c = std::string(home) + "/.cache";
    mkdir(c.c_str(), 0755);
    const std::string d = c + "/rbd_b200";
    if (dir_writable(d)) return d;
  }
  return "/tmp";
}

// NVRTC for sm_100a on a complete source text; the embedded headers are offered to every program.
static bool nvrtc_compile(const std::string& src, bool fmad, std::vector<char>& cubin, std::string& err) {
  Nvrtc& n = nvrtc();
  if (!n.h) { err = n.err; return false; }
  const int nh = (int)(sizeof(kEmbeddedHeaders) / sizeof(kEmbeddedHeaders[0]));
  std::vector<const char*> hn, ht;
  for (int i = 0; i < nh; ++i) { hn.push_back(kEmbeddedHeaders[i].name); ht.push_back(kEmbeddedHeaders[i].text); }
  nvrtcProgram prog = nullptr;
  nvrtcResult r = n.CreateProgram(&prog, src.c_str(), "rbd_spec.cu", nh, ht.data(), hn.data());
  if (r != NVRTC_SUCCESS) { err = std::string("nvrtcCreateProgram: ") + n.GetErrorString(r); return false; }
  const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "--fmad=false"};
  r = n.CompileProgram(prog, fmad ? 3 : 4, opts);
  if (r != NVRTC_SUCCESS) {
    size_t ls = 0;
    n.GetProgramLogSize(prog, &ls);
    std::string log(ls, '\0');
    if (ls) n.GetProgramLog(prog, &log[0]);
    if (log.size() > 2000) log.resize(2000);
    err = std::string("nvrtcCompileProgram: ") + n.GetErrorString(r) + "\n" + log;
    n.DestroyProgram(&prog);
    return false;
  }
  size_t sz = 0;
  r = n.GetCUBINSize(prog, &sz);
  if (r == NVRTC_SUCCESS && sz > 0) { cubin.resize(sz); r = n.GetCUBIN(prog, cubin.data()); }
  n.DestroyProgram(&prog);
  if (r != NVRTC_SUCCESS || sz == 0) { err = "nvrtcGetCUBIN failed"; return false; }
  return true;
}

bool jit_cubin(const std::string& name, bool fmad, bool compile_if_missing,
               const std::function<bool(std::string& src, std::string& err)>& source, std::vector<char>& cubin, std::string& err) {
  const std::string path = jit_cache_dir() + "/" + name + ".cubin";
  const bool use_cache = !getenv("RBD_JIT_NO_CACHE");
  if (use_cache && read_file(path, cubin)) return true;
  if (!compile_if_missing) { err = "no cached cubin"; return false; }
  std::string src;
  if (!source(src, err)) return false;
  if (!nvrtc_compile(src, fmad, cubin, err)) return false;
  if (use_cache) write_file_atomic(path, cubin.data(), cubin.size());
  return true;
}

}  // namespace rbd
