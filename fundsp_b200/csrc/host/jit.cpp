// fundsp_b200 NVRTC path: compile the fused voice program of a graph class that is not in the AOT tables.
//
// A class is named by a C++ type expression over the node templates of csrc/dsp/nodes.cuh (graph.h `sig`), so
// "compiling a new graph" is instantiating `fdsp::bank_kernel<SIG, 128, MODE, TB>` from the SAME hand-written device
// headers the AOT instances use (embedded in this library at build time, _build/jit_headers.inc). This is template
// instantiation at run time, not tracing: the kernel body is the code in bank_kernel.cuh / nodes.cuh.
// libnvrtc / libcuda are dlopen'ed on first use so the library loads on machines without them.
#include <cuda.h>
#include <dlfcn.h>
#include <nvrtc.h>

#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "registry.h"
#include "../dsp/rt_args.h"

#include "jit_headers.inc"  // kJitHeaderNames[], kJitHeaderSrc[], kJitHeaderCount

namespace fdsp {
namespace host {

namespace {

struct Api {
  void* nvrtc = nullptr; void* cuda = nullptr; bool ok = false, ok_nvrtc = false; std::string why;
  nvrtcResult (*Version)(int*, int*);
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
  nvrtcResult (*DestroyProgram)(nvrtcProgram*);
  nvrtcResult (*AddNameExpression)(nvrtcProgram, const char*);
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*);
  nvrtcResult (*GetLoweredName)(nvrtcProgram, const char*, const char**);
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*);
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*);
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*);
  CUresult (*ModuleLoadData)(CUmodule*, const void*);
  CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*);
  CUresult (*ModuleGetGlobal)(CUdeviceptr*, size_t*, CUmodule, const char*);
  CUresult (*MemcpyDtoH)(void*, CUdeviceptr, size_t);
  CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int);
  CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void**, void**);
  CUresult (*GetErrorString)(CUresult, const char**);
};

template <class F> bool sym(void* lib, const char* name, F& f) { f = reinterpret_cast<F>(dlsym(lib, name)); return f != nullptr; }

Api& api() {
  static Api a;
  static std::once_flag once;
  std::call_once(once, []() {
    for (const char* n : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"})
      if ((a.nvrtc = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
    for (const char* n : {"libcuda.so.1", "libcuda.so"})
      if ((a.cuda = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
    if (!a.nvrtc) { a.why = "libnvrtc not found (JIT unavailable; only the ahead-of-time graph classes can run)"; return; }
    a.ok_nvrtc = sym(a.nvrtc, "nvrtcCreateProgram", a.CreateProgram) && sym(a.nvrtc, "nvrtcDestroyProgram", a.DestroyProgram) &&
                 sym(a.nvrtc, "nvrtcAddNameExpression", a.AddNameExpression) && sym(a.nvrtc, "nvrtcCompileProgram", a.CompileProgram) &&
                 sym(a.nvrtc, "nvrtcGetLoweredName", a.GetLoweredName) && sym(a.nvrtc, "nvrtcGetCUBINSize", a.GetCUBINSize) &&
                 sym(a.nvrtc, "nvrtcGetCUBIN", a.GetCUBIN) && sym(a.nvrtc, "nvrtcGetProgramLogSize", a.GetProgramLogSize) &&
                 sym(a.nvrtc, "nvrtcGetProgramLog", a.GetProgramLog) && sym(a.nvrtc, "nvrtcVersion", a.Version);
    if (!a.ok_nvrtc) { a.why = "missing NVRTC symbols"; return; }
    if (!a.cuda) { a.why = "libcuda not found"; return; }
    bool ok = sym(a.cuda, "cuModuleLoadData", a.ModuleLoadData) &&
              sym(a.cuda, "cuModuleGetFunction", a.ModuleGetFunction) && sym(a.cuda, "cuModuleGetGlobal_v2", a.ModuleGetGlobal) &&
              sym(a.cuda, "cuMemcpyDtoH_v2", a.MemcpyDtoH) && sym(a.cuda, "cuFuncSetAttribute", a.FuncSetAttribute) &&
              sym(a.cuda, "cuLaunchKernel", a.LaunchKernel) && sym(a.cuda, "cuGetErrorString", a.GetErrorString);
    if (!ok) { a.why = "missing NVRTC / driver symbols"; return; }
    a.ok = true;
  });
  return a;
}

// One NVRTC translation unit = the headers + `typedef <sig> JitG` + (optionally) one kernel instantiation. The layout TU
// (no kernel) is compiled when the program is created; each (mode, TB) kernel variant is compiled on its first launch, so a
// bank pays for the one variant it uses instead of all six.
// ---- on-disk cache of compiled units. Key: FNV-1a of (NVRTC version, options, embedded headers, unit source, kernel expression), so
// an entry can only be hit by the identical compilation. Directory: $FDSP_JIT_CACHE, else jit_cache/ next to this library (it travels
// with the in-tree build; tools/warm_jit_cache.py fills it on a machine without a GPU). FDSP_JIT_CACHE=off disables it.
static const char* kJitOpts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "--fmad=false", "-lineinfo", "-default-device"};
static uint64_t fnv(uint64_t h, const void* p, size_t n) { const unsigned char* b = (const unsigned char*)p; for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 1099511628211ull; } return h; }
static std::string cache_dir() {
  static const std::string dir = [] {
    const char* e = getenv("FDSP_JIT_CACHE");
    if (e && *e) return std::string(strcmp(e, "off") == 0 ? "" : e);
    Dl_info info;
    if (!dladdr((void*)&cache_dir, &info) || !info.dli_fname) return std::string();
    std::string p(info.dli_fname);
    const size_t k = p.rfind('/');
    return (k == std::string::npos ? std::string(".") : p.substr(0, k)) + "/jit_cache";
  }();
  return dir;
}
static uint64_t unit_key(const std::string& src, const char* kernel_expr) {
  static const uint64_t base = [] {
    uint64_t h = 1469598103934665603ull;
    int maj = 0, min = 0;
    if (api().ok_nvrtc) api().Version(&maj, &min);
    h = fnv(h, &maj, sizeof(maj)); h = fnv(h, &min, sizeof(min));
    for (const char* o : kJitOpts) h = fnv(h, o, strlen(o) + 1);
    for (int i = 0; i < kJitHeaderCount; i++) { h = fnv(h, kJitHeaderNames[i], strlen(kJitHeaderNames[i]) + 1); h = fnv(h, kJitHeaderSrc[i], strlen(kJitHeaderSrc[i]) + 1); }
    return h;
  }();
  uint64_t h = fnv(base, src.data(), src.size() + 1);
  if (kernel_expr) h = fnv(h, kernel_expr, strlen(kernel_expr) + 1);
  return h;
}
static std::string cache_path(uint64_t key) { char b[32]; snprintf(b, sizeof(b), "/%016llx.fdspjit", (unsigned long long)key); return cache_dir() + b; }
static bool cache_load(uint64_t key, std::vector<char>& cubin, std::string& lowered) {
  if (cache_dir().empty()) return false;
  FILE* f = fopen(cache_path(key).c_str(), "rb");
  if (!f) return false;
  uint32_t hdr[3] = {0, 0, 0};   // magic, lowered-name bytes, cubin bytes
  bool ok = fread(hdr, 4, 3, f) == 3 && hdr[0] == 0x4a445346u && hdr[1] < (1u << 20) && hdr[2] > 0 && hdr[2] < (1u << 30);
  if (ok) { lowered.resize(hdr[1]); cubin.resize(hdr[2]); ok = (hdr[1] == 0 || fread(&lowered[0], 1, hdr[1], f) == hdr[1]) && fread(cubin.data(), 1, hdr[2], f) == hdr[2]; }
  fclose(f);
  return ok;
}
static void cache_store(uint64_t key, const std::vector<char>& cubin, const std::string& lowered) {
  if (cache_dir().empty() || cubin.empty()) return;
  mkdir(cache_dir().c_str(), 0755);
  const std::string path = cache_path(key), tmp = path + ".tmp" + std::to_string((long)getpid());
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return;
  const uint32_t hdr[3] = {0x4a445346u, (uint32_t)lowered.size(), (uint32_t)cubin.size()};
  const bool ok = fwrite(hdr, 4, 3, f) == 3 && fwrite(lowered.data(), 1, lowered.size(), f) == lowered.size() && fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
  if (fclose(f) != 0 || !ok || rename(tmp.c_str(), path.c_str()) != 0) remove(tmp.c_str());
}
static int g_cache_hits = 0, g_nvrtc_runs = 0;

static bool compile_unit(const std::string& sig, const char* kernel_expr, std::vector<char>& cubin, std::string& lowered, std::string& err, bool use_cache = true) {
  Api& A = api();
  if (!A.ok_nvrtc) { err = A.why; return false; }
  std::string src = "#include \"dsp/bank_kernel_st.cuh\"\n#include \"dsp/bank_kernel_rt.cuh\"\nnamespace fdsp { typedef " + sig + " JitG; }\n";
  if (!kernel_expr)
    src += "extern \"C\" __device__ int fdsp_jit_layout[8] = {fdsp::JitG::IN, fdsp::JitG::OUT, fdsp::JitG::NP, fdsp::JitG::NS, fdsp::JitG::NU, fdsp::WaveKind<fdsp::JitG>::value, "
           "fdsp::StagePlan<fdsp::JitG>::K, fdsp::MidSum<fdsp::StagePlan<fdsp::JitG>::stages>::value};\n";
  const uint64_t key = unit_key(src, kernel_expr);
  if (use_cache && cache_load(key, cubin, lowered)) { g_cache_hits++; return true; }
  g_nvrtc_runs++;
  nvrtcProgram prog;
  if (A.CreateProgram(&prog, src.c_str(), "fdsp_jit.cu", kJitHeaderCount, kJitHeaderSrc, kJitHeaderNames) != NVRTC_SUCCESS) { err = "nvrtcCreateProgram failed"; return false; }
  if (kernel_expr) A.AddNameExpression(prog, kernel_expr);
  if (A.CompileProgram(prog, 5, kJitOpts) != NVRTC_SUCCESS) {
    size_t n = 0; A.GetProgramLogSize(prog, &n);
    std::string log(n, '\0'); if (n) A.GetProgramLog(prog, &log[0]);
    if (log.size() > 1500) log.resize(1500);
    err = "NVRTC compile of `" + sig + "` failed: " + log;
    A.DestroyProgram(&prog);
    return false;
  }
  if (kernel_expr) {
    const char* low = nullptr;
    if (A.GetLoweredName(prog, kernel_expr, &low) != NVRTC_SUCCESS || !low) { err = "JIT kernel name lookup failed"; A.DestroyProgram(&prog); return false; }
    lowered = low;
  }
  size_t cn = 0; A.GetCUBINSize(prog, &cn);
  cubin.resize(cn); A.GetCUBIN(prog, cubin.data());
  A.DestroyProgram(&prog);
  cache_store(key, cubin, lowered);
  return true;
}

// width 0: the plain kernel (128 threads); 32 / 128: the stage-pipelined kernel with that many voices per CTA; -1: the resident process() kernel
static std::string kernel_expr_of(int mode, int tb, int width) {
  if (width < 0) return std::string("fdsp::bank_kernel_rt<fdsp::JitG, 128, ") + (tb ? "true" : "false") + ">";
  const std::string tail = std::to_string(mode) + ", " + (tb ? "true" : "false") + ">";
  return width ? "fdsp::bank_kernel_st<fdsp::JitG, " + std::to_string(width) + ", " + tail : "fdsp::bank_kernel<fdsp::JitG, 128, " + tail;
}

struct JitProgram : Program {
  int device = 0, mid_sum = 0;   // mid_sum: channels crossing the stage boundaries (sizes the hand-off rings)
  mutable std::mutex mu;
  mutable CUmodule mods[4][3][2] = {};
  mutable CUfunction fn[4][3][2] = {};  // [0 plain | 1 staged x32 | 2 staged x128 | 3 resident][mode-1][TB]
  CUfunction variant(int mode, int tb, int width = 0) const {
    std::lock_guard<std::mutex> lock(mu);
    const int wi = width < 0 ? 3 : (width == 0 ? 0 : (width == 32 ? 1 : 2));
    CUfunction& f = fn[wi][mode - 1][tb]; CUmodule& m = mods[wi][mode - 1][tb];
    if (f) return f;
    const Api& A = api();
    const std::string expr = kernel_expr_of(mode, tb, width);
    std::vector<char> cubin; std::string low, err;
    if (!compile_unit(sig, expr.c_str(), cubin, low, err)) { fprintf(stderr, "fundsp_b200 JIT: %s\n", err.c_str()); return nullptr; }
    if (A.ModuleLoadData(&m, cubin.data()) != CUDA_SUCCESS) {   // a damaged cache entry: compile afresh (which rewrites it)
      if (!compile_unit(sig, expr.c_str(), cubin, low, err, false) || A.ModuleLoadData(&m, cubin.data()) != CUDA_SUCCESS) return nullptr;
    }
    if (A.ModuleGetFunction(&f, m, low.c_str()) != CUDA_SUCCESS) { f = nullptr; return nullptr; }
    return f;
  }
  cudaError_t launch_rt(const BankArgs& a, const RtArgs& rt, size_t table_bytes, cudaStream_t st) const override {
    const Api& A = api();
    const LaunchSmem L = launch_smem(OUT, threads, 0, 2, wave_kind >= 0 ? table_bytes : 0);
    const size_t smem = L.smem;
    CUfunction f = variant(2, L.tb, -1);
    if (!f) return cudaErrorInvalidDeviceFunction;
    if (smem > 48 * 1024 && A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem) != CUDA_SUCCESS) return cudaErrorInvalidValue;
    if (launch_carveout() >= 0) A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, launch_carveout());
    BankArgs args = a; RtArgs r = rt;
    void* params[] = {&args, &r};
    const unsigned vpc = a.vpc ? a.vpc : (unsigned)threads, grid = (a.V + vpc - 1) / vpc;
    CUresult rc = A.LaunchKernel(f, grid, 1, 1, (unsigned)threads, 1, 1, (unsigned)smem, (CUstream)st, params, nullptr);
    return rc == CUDA_SUCCESS ? cudaSuccess : cudaErrorLaunchFailure;
  }
  cudaError_t launch_staged(const BankArgs& a, int mode, size_t table_bytes, cudaStream_t st) const override {
    const Api& A = api();
    mode &= 3;
    if (mode == 0 || stages < 2) return cudaErrorInvalidValue;
    const int width = (a.vpc && a.vpc <= 32u) ? 32 : 128;
    const LaunchSmem L = launch_smem(OUT, width, mid_sum, mode, wave_kind >= 0 ? table_bytes : 0);
    const size_t smem = L.smem;
    if (smem > SMEM_BLOCK_MAX) return cudaErrorInvalidValue;
    CUfunction f = variant(mode, L.tb, width);
    if (!f) return cudaErrorInvalidDeviceFunction;
    if (smem > 48 * 1024 && A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem) != CUDA_SUCCESS) return cudaErrorInvalidValue;
    if (launch_carveout() >= 0) A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, launch_carveout());
    BankArgs args = a;
    void* params[] = {&args};
    const unsigned vpc = a.vpc ? a.vpc : (unsigned)width, grid = (a.V + vpc - 1) / vpc;
    CUresult r = A.LaunchKernel(f, grid, 1, 1, (unsigned)(stages * width), 1, 1, (unsigned)smem, (CUstream)st, params, nullptr);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorLaunchFailure;
  }
  cudaError_t launch(const BankArgs& a, int mode, size_t table_bytes, cudaStream_t st) const override {
    const Api& A = api();
    mode &= 3;
    if (mode == 0) return cudaErrorInvalidValue;
    const LaunchSmem L = launch_smem(OUT, threads, 0, mode, wave_kind >= 0 ? table_bytes : 0);
    const size_t smem = L.smem;
    CUfunction f = variant(mode, L.tb);
    if (!f) return cudaErrorInvalidDeviceFunction;
    if (smem > 48 * 1024 && A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem) != CUDA_SUCCESS) return cudaErrorInvalidValue;
    if (launch_carveout() >= 0) A.FuncSetAttribute(f, CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT, launch_carveout());
    BankArgs args = a;
    void* params[] = {&args};
    const unsigned vpc = a.vpc ? a.vpc : (unsigned)threads, grid = (a.V + vpc - 1) / vpc;
    CUresult r = A.LaunchKernel(f, grid, 1, 1, (unsigned)threads, 1, 1, (unsigned)smem, (CUstream)st, params, nullptr);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorLaunchFailure;
  }
};

std::mutex g_mu;
std::map<std::string, std::shared_ptr<const Program>> g_cache;  // key: device:sig
int g_compiled = 0;

}  // namespace

int jit_compiled_count() { return g_compiled; }
void jit_cache_stats(int* hits, int* nvrtc_runs) { if (hits) *hits = g_cache_hits; if (nvrtc_runs) *nvrtc_runs = g_nvrtc_runs; }

// Compile one unit of a graph class into the on-disk cache without touching a GPU (mode 0: the layout unit; 1..3: that kernel variant).
std::string jit_precompile(const std::string& sig, int mode, int tb, int staged_width) {
  if (sig.find("Unsupported") != std::string::npos) return "the graph contains a node with no device lowering";
  if (mode < 0 || mode > 3) return "mode must be 0 (layout) or 1..3";
  if (cache_dir().empty()) return "the JIT cache is disabled (FDSP_JIT_CACHE=off)";
  std::vector<char> cubin; std::string low, err;
  if (staged_width != 0 && staged_width != 32 && staged_width != 128 && staged_width != 255) return "staged width must be 0, 32, 128 or 255 (the resident process() kernel)";
  if (staged_width == 255) staged_width = -1;
  const std::string expr = kernel_expr_of(mode, tb, staged_width);
  if (!compile_unit(sig, mode == 0 ? nullptr : expr.c_str(), cubin, low, err)) return err;
  return "";
}

std::shared_ptr<const Program> jit_program(const std::string& sig, int device, std::string& err) {
  if (sig.find("Unsupported") != std::string::npos) { err = "the graph contains a node with no device lowering"; return nullptr; }
  Api& A = api();
  if (!A.ok) { err = A.why; return nullptr; }
  std::lock_guard<std::mutex> lock(g_mu);
  const std::string key = std::to_string(device) + ":" + sig;
  auto it = g_cache.find(key);
  if (it != g_cache.end()) return it->second;
  cudaSetDevice(device);
  cudaFree(nullptr);  // make sure the primary context exists and is current for the driver API calls below

  std::vector<char> cubin; std::string low;
  if (!compile_unit(sig, nullptr, cubin, low, err)) return nullptr;
  auto p = std::make_shared<JitProgram>();
  p->sig = sig; p->jit = true; p->device = device;
  CUmodule lm = nullptr;
  if (A.ModuleLoadData(&lm, cubin.data()) != CUDA_SUCCESS) {
    if (!compile_unit(sig, nullptr, cubin, low, err, false)) return nullptr;
    if (A.ModuleLoadData(&lm, cubin.data()) != CUDA_SUCCESS) { err = "cuModuleLoadData failed for the JIT layout unit"; return nullptr; }
  }
  CUdeviceptr d = 0; size_t bytes = 0; int lay[8] = {0, 0, 0, 0, 0, -1, 1, 0};
  if (A.ModuleGetGlobal(&d, &bytes, lm, "fdsp_jit_layout") != CUDA_SUCCESS || bytes != sizeof(lay) || A.MemcpyDtoH(lay, d, sizeof(lay)) != CUDA_SUCCESS) {
    err = "JIT layout readback failed"; return nullptr;
  }
  p->IN = lay[0]; p->OUT = lay[1]; p->NP = lay[2]; p->NS = lay[3]; p->NU = lay[4]; p->wave_kind = lay[5]; p->threads = 128; p->stages = lay[6]; p->mid_sum = lay[7]; p->has_rt = true;
  g_compiled++;
  g_cache[key] = p;
  return p;
}

}  // namespace host
}  // namespace fdsp
