// TEST INFRASTRUCTURE — the kernel side of the mock "GPU": replaces csrc/host/registry.cpp, csrc/host/jit.cpp and csrc/inst/*.cu when the
// host runtime is built for the CPU-only test suite (tests/test_mock_bank_cpu.py). Every graph class becomes a small shared object
// compiled with g++ from tests/cpp/mock/emul_module.cpp (the device node library under FDSP_HOST_EMUL) and cached by signature.
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <vector>
#include <cstring>

#include "host/registry.h"
#include "dsp/fdn_args.h"
#include "dsp/mix_order.h"

namespace fdsp {
namespace host {

namespace {
typedef void (*LayoutFn)(int*);
typedef int (*LaunchFn)(const BankArgs*, int);
typedef int (*LaunchExFn)(const BankArgs*, int, const float*, uint64_t);
struct MockProgram : Program {
  LaunchFn fn = nullptr; LaunchExFn fn_ex = nullptr;
  cudaError_t launch(const BankArgs& a, int mode, size_t, cudaStream_t) const override {
    mode &= 3;
    return (mode && fn && fn(&a, mode) == 0) ? cudaSuccess : cudaErrorLaunchFailure;
  }
};
std::mutex g_mu;
std::map<std::string, std::shared_ptr<const Program>> g_cache;
uint64_t fnv(const std::string& s) { uint64_t h = 1469598103934665603ull; for (unsigned char ch : s) { h ^= ch; h *= 1099511628211ull; } return h; }
}  // namespace

std::shared_ptr<const Program> get_program(const std::string& sig, int, std::string& err) {
  std::lock_guard<std::mutex> lock(g_mu);
  auto it = g_cache.find(sig);
  if (it != g_cache.end()) return it->second;
  if (sig.find("Unsupported") != std::string::npos) { err = "the graph contains a node with no device lowering"; return nullptr; }
  const char* root = getenv("FDSP_MOCK_ROOT");   // repository root
  const char* dir = getenv("FDSP_MOCK_CACHE");
  if (!root || !dir) { err = "mock registry: FDSP_MOCK_ROOT / FDSP_MOCK_CACHE not set"; return nullptr; }
  mkdir(dir, 0755);
  char name[64]; snprintf(name, sizeof(name), "/emul_%016llx.so", (unsigned long long)fnv(sig));
  const std::string so = std::string(dir) + name;
  if (access(so.c_str(), R_OK) != 0) {
    const std::string tmp = so + ".tmp" + std::to_string((long)getpid());
    const char* extra = getenv("FDSP_MOCK_CXXFLAGS");   // e.g. -fsanitize=address -g for a sanitizer run of the whole suite
    const std::string cmd = std::string("g++ -std=c++17 -O1 -ffp-contract=off -w -shared -fPIC ") + (extra ? extra : "") + " '-DGRAPH=" + sig + "' -I '" + root + "/fundsp_b200/csrc' '" + root +
                            "/tests/cpp/mock/emul_module.cpp' -o '" + tmp + "' 2> '" + so + ".log' && mv '" + tmp + "' '" + so + "'";
    if (system(cmd.c_str()) != 0) { err = "mock registry: g++ failed for `" + sig + "` (see " + so + ".log)"; return nullptr; }
  }
  void* h = dlopen(so.c_str(), RTLD_NOW | RTLD_LOCAL);
  if (!h) { err = std::string("mock registry: dlopen: ") + dlerror(); return nullptr; }
  LayoutFn lay = (LayoutFn)dlsym(h, "fdsp_emul_layout");
  auto p = std::make_shared<MockProgram>();
  p->fn = (LaunchFn)dlsym(h, "fdsp_emul_launch");
  p->fn_ex = (LaunchExFn)dlsym(h, "fdsp_emul_launch_ex");
  if (!lay || !p->fn || !p->fn_ex) { err = "mock registry: missing symbols"; return nullptr; }
  int L[6]; lay(L);
  p->sig = sig; p->jit = true; p->IN = L[0]; p->OUT = L[1]; p->NP = L[2]; p->NS = L[3]; p->NU = L[4]; p->wave_kind = L[5]; p->threads = 128;
  g_cache[sig] = p;
  return p;
}
const KernelEntry* find_kernel(const std::string&) { return nullptr; }
int registry_size() { return 0; }
const KernelEntry* registry_at(int) { return nullptr; }
const char* registry_key(int) { return ""; }

cudaError_t launch_mix_reduce(const float* partial, uint32_t nparts, uint32_t outs, uint32_t n, float* mix, uint32_t mix_stride, uint32_t mix_offset, int accumulate, cudaStream_t) {
  for (uint32_t c = 0; c < outs; c++)
    for (uint32_t t = 0; t < n; t++) {   // mix_reduce_kernel: CTA-order left fold
      const float s = cta_order_fold(partial + (size_t)c * n + t, (size_t)outs * n, nparts, [](const float* q) { return *q; });
      float* p = mix + (size_t)c * mix_stride + mix_offset + t;
      *p = accumulate ? *p + s : s;
    }
  return cudaSuccess;
}
cudaError_t launch_tree_mix(const float* rows, uint32_t V, uint32_t outs, uint32_t row_stride, uint32_t row_offset, uint32_t n, float* mix, uint32_t mix_stride, uint32_t mix_offset, int pairwise, cudaStream_t, float*) {
  for (uint32_t ch = 0; ch < outs; ch++)
    for (uint32_t t = 0; t < n; t++) {   // tree_mix_kernel: the binary-carry stack of the balanced tree, or the left fold
      const float* p = rows + (size_t)ch * row_stride + row_offset + t;
      const size_t vstep = (size_t)outs * row_stride;
      float x;
      if (pairwise) {
        float st[32];
        for (uint32_t v = 0; v < V; v++) carry_push(st, p[(size_t)v * vstep], v, 0);
        x = carry_finish(st, V);
      } else { x = p[0]; for (uint32_t v = 1; v < V; v++) x += p[(size_t)v * vstep]; }
      mix[(size_t)ch * mix_stride + mix_offset + t] = x;
    }
  return cudaSuccess;
}
// The warp-per-voice FDN kernel (dsp/fdn_kernel.cuh) computes `reverb_stereo` exactly like the generic thread-per-voice program (the GPU
// tests compare the two bit for bit), so the mock runs that generic program on the kernel's argument block: the last words of the
// class are the reverb's words, the rings are its delay lines, the input is each voice's dry stereo rows. This puts the HOST side of the
// two-stage classes (dry buffers, chunk pipeline, deferred reductions, wet gain row) under the CPU suite.
static const char* kRevSig = "Pipe<Pipe<MultiSplit<2,16>,Feedback<1,Multi<30,0,32,Pipe<Delay,Fir<3>>>>>,Binop<2,Multi<31,0,32,Panner<1>>,Constant<2>>>";
cudaError_t launch_fdn(const FdnArgs& f, int warps, cudaStream_t) {
  std::string err;
  auto prog = std::dynamic_pointer_cast<const MockProgram>(get_program(kRevSig, 0, err));
  if (!prog || warps < 1) return cudaErrorLaunchFailure;
  const uint32_t V = f.V, n = f.n, grid = V;   // the kernel writes one partial-mix row pair per voice
  std::vector<float> rev((size_t)V * 2 * n, 0.0f);
  std::vector<uint32_t> rows(V);
  for (uint32_t v = 0; v < V; v++) rows[v] = 2 * v;
  BankArgs a; memset(&a, 0, sizeof(a));
  a.params = f.params + (size_t)f.p0 * V; a.state = f.state + (size_t)f.s0 * V; a.uniform = f.uniform + f.u0;
  a.dline = f.ring; a.wt = nullptr; a.out = rev.data(); a.V = V; a.n = n; a.vpc = 0;
  a.in = f.dry; a.in_stride = f.dry_ch_stride; a.in_offset = f.dry_offset; a.out_stride = n; a.out_offset = 0; a.row_map = rows.data();
  a.sr = 0.0f; a.sd64 = 0.0f; a.sd32 = 0.0f;   // (the reverb's nodes do not read the rate: delay lengths are class-uniform words)
  if (prog->fn_ex(&a, 1, f.dry_voice_stride ? f.dry : nullptr, f.dry_voice_stride) != 0) return cudaErrorLaunchFailure;
  if (f.partial) for (size_t e = 0; e < (size_t)grid * 2 * n; e++) f.partial[e] = 0.0f;
  for (uint32_t v = 0; v < V; v++)
    for (uint32_t ch = 0; ch < 2; ch++)
      for (uint32_t t = 0; t < n; t++) {
        float y = rev[((size_t)2 * v + ch) * n + t];
        if (f.scalar_row >= 0) {   // Bus<MultiPass<2>, Unop<3, Reverb>>: dry + reverb * g
          float g; memcpy(&g, f.params + (size_t)f.scalar_row * V + v, 4);
          const float dry = f.dry[(size_t)v * f.dry_voice_stride + (size_t)ch * f.dry_ch_stride + f.dry_offset + t];
          y = dry + y * g;
        }
        if (f.out) f.out[(size_t)(f.row_map[v] + ch) * f.out_stride + f.out_offset + t] = y;
        if (f.partial) f.partial[((size_t)v * 2 + ch) * n + t] += y;
      }
  return cudaSuccess;
}
size_t tree_mix_scratch_floats(uint32_t, uint32_t, uint32_t) { return 0; }
int fdn_max_warps() { return 8; }
// the tensor-core convolver form is never selected on the mock (bank.cpp tc_conv_wanted); the symbols only have to link
cudaError_t conv_tc_make_maps(float*, float*, uint32_t, uint32_t, float*, float*, uint32_t, ConvTcMaps*) { return cudaErrorInvalidValue; }
cudaError_t launch_conv_tc(const ConvTcMaps&, float*, uint32_t, uint32_t, const uint32_t*, uint32_t, uint32_t, uint32_t, uint32_t, cudaStream_t) { return cudaErrorInvalidValue; }
cudaError_t launch_conv_split(const float*, float*, uint32_t, uint32_t, uint32_t, uint32_t, cudaStream_t) { return cudaErrorInvalidValue; }
cudaError_t launch_conv_history(float*, float*, uint32_t, uint32_t, uint32_t, uint32_t, cudaStream_t) { return cudaErrorInvalidValue; }
cudaError_t launch_conv_toeplitz(const float*, uint32_t, float*, float*, uint32_t, cudaStream_t) { return cudaErrorInvalidValue; }
uint32_t conv_tc_toeplitz_cols(uint32_t) { return 0; }
std::shared_ptr<const Program> jit_program(const std::string& sig, int device, std::string& err) { return get_program(sig, device, err); }
int jit_compiled_count() { return (int)g_cache.size(); }
void jit_cache_stats(int* hits, int* runs) { if (hits) *hits = 0; if (runs) *runs = 0; }
std::string jit_precompile(const std::string&, int, int, int) { return "mock registry: no NVRTC"; }

}  // namespace host
}  // namespace fdsp
