// Launcher template + registry entry macro shared by the ahead-of-time instance files (csrc/inst/*.cu).
#pragma once
#include "../host/registry.h"
#include "bank_kernel.cuh"
#include "bank_kernel_st.cuh"
#include "bank_kernel_rt.cuh"

namespace fdsp {
namespace host {

constexpr int NT = 128;

template <class G, int MODE, bool TB> cudaError_t launch_one(const BankArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(bank_kernel<G, NT, MODE, TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  if (launch_carveout() >= 0) cudaFuncSetAttribute(bank_kernel<G, NT, MODE, TB>, cudaFuncAttributePreferredSharedMemoryCarveout, launch_carveout());
  bank_kernel<G, NT, MODE, TB><<<grid, NT, smem, st>>>(a);
  return cudaGetLastError();
}
template <class G, bool TB> cudaError_t launch_mode(const BankArgs& a, int mode, size_t smem, cudaStream_t st) {
  const unsigned vpc = a.vpc ? a.vpc : (unsigned)NT, grid = (a.V + vpc - 1) / vpc;
  switch (mode & 3) {
    case 1: return launch_one<G, 1, TB>(a, grid, smem, st);
    case 2: return launch_one<G, 2, TB>(a, grid, smem, st);
    case 3: return launch_one<G, 3, TB>(a, grid, smem, st);
    default: return cudaErrorInvalidValue;
  }
}
// stage-pipelined variant (bank_kernel_st.cuh): K * NTV threads per CTA, the stages of StagePlan<G> in different warps
template <class G, int NTV, int MODE, bool TB> cudaError_t launch_st_one(const BankArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  if constexpr (StagePlan<G>::K >= 2) {
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(bank_kernel_st<G, NTV, MODE, TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
    }
    bank_kernel_st<G, NTV, MODE, TB><<<grid, StagePlan<G>::K * NTV, smem, st>>>(a);
    return cudaGetLastError();
  } else {
    return cudaErrorInvalidValue;
  }
}
template <class G, int NTV, bool TB> cudaError_t launch_st_mode(const BankArgs& a, int mode, size_t smem, cudaStream_t st) {
  const unsigned vpc = a.vpc ? a.vpc : (unsigned)NTV, grid = (a.V + vpc - 1) / vpc;
  switch (mode & 3) {
    case 1: return launch_st_one<G, NTV, 1, TB>(a, grid, smem, st);
    case 2: return launch_st_one<G, NTV, 2, TB>(a, grid, smem, st);
    case 3: return launch_st_one<G, NTV, 3, TB>(a, grid, smem, st);
    default: return cudaErrorInvalidValue;
  }
}
// table_bytes > 0 asks for the shared-memory wavetable variant (only taken when G reads a wavetable and it fits, launch_smem)
template <class G> size_t table_bytes_of(size_t table_bytes) { return WaveKind<G>::value >= 0 ? table_bytes : 0; }
// stage width: 32 voices per CTA when the launch asks for at most 32 (a.vpc), else 128
template <class G> cudaError_t launch_st_t(const BankArgs& a, int mode, size_t table_bytes, cudaStream_t st) {
  constexpr bool WT = WaveKind<G>::value >= 0;
  const bool narrow = a.vpc && a.vpc <= 32u;
  const LaunchSmem L = launch_smem(G::OUT, narrow ? 32 : 128, MidSum<typename StagePlan<G>::stages>::value, mode, table_bytes_of<G>(table_bytes));
  if (L.smem > SMEM_BLOCK_MAX) return cudaErrorInvalidValue;
  if (narrow) return L.tb ? launch_st_mode<G, 32, WT>(a, mode, L.smem, st) : launch_st_mode<G, 32, false>(a, mode, L.smem, st);
  return L.tb ? launch_st_mode<G, 128, WT>(a, mode, L.smem, st) : launch_st_mode<G, 128, false>(a, mode, L.smem, st);
}
template <class G> cudaError_t launch_t(const BankArgs& a, int mode, size_t table_bytes, cudaStream_t st) {
  const LaunchSmem L = launch_smem(G::OUT, NT, 0, mode, table_bytes_of<G>(table_bytes));
  return L.tb ? launch_mode<G, (WaveKind<G>::value >= 0)>(a, mode, L.smem, st) : launch_mode<G, false>(a, mode, L.smem, st);
}
// resident process() kernel (bank_kernel_rt.cuh): one launch serves 64-sample blocks on a doorbell until it is told to leave
template <class G, bool TB> cudaError_t launch_rt_one(const BankArgs& a, const RtArgs& rt, size_t smem, cudaStream_t st) {
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(bank_kernel_rt<G, NT, TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const unsigned vpc = a.vpc ? a.vpc : (unsigned)NT, grid = (a.V + vpc - 1) / vpc;
  bank_kernel_rt<G, NT, TB><<<grid, NT, smem, st>>>(a, rt);
  return cudaGetLastError();
}
template <class G> cudaError_t launch_rt_t(const BankArgs& a, const RtArgs& rt, size_t table_bytes, cudaStream_t st) {
  const LaunchSmem L = launch_smem(G::OUT, NT, 0, 2, table_bytes_of<G>(table_bytes));
  return L.tb ? launch_rt_one<G, (WaveKind<G>::value >= 0)>(a, rt, L.smem, st) : launch_rt_one<G, false>(a, rt, L.smem, st);
}
template <class G> int wave_kind_t() { return WaveKind<G>::value; }
inline int threads_t() { return NT; }

template <class G> int stages_t() { return StagePlan<G>::K; }
#define FDSP_REG(...) \
  {#__VA_ARGS__, __VA_ARGS__::IN, __VA_ARGS__::OUT, __VA_ARGS__::NP, __VA_ARGS__::NS, __VA_ARGS__::NU, &launch_t<__VA_ARGS__>, &threads_t, &wave_kind_t<__VA_ARGS__>, 1, nullptr, &launch_rt_t<__VA_ARGS__>}
// the same, plus the stage-pipelined kernels of the graph (bank_kernel_st.cuh; only graphs with a heavy leaf have any)
#define FDSP_REG_ST(...) \
  {#__VA_ARGS__, __VA_ARGS__::IN, __VA_ARGS__::OUT, __VA_ARGS__::NP, __VA_ARGS__::NS, __VA_ARGS__::NU, &launch_t<__VA_ARGS__>, &threads_t, &wave_kind_t<__VA_ARGS__>, \
   StagePlan<__VA_ARGS__>::K, &launch_st_t<__VA_ARGS__>, &launch_rt_t<__VA_ARGS__>}
#define FDSP_INSTANCES(name, ...)                     \
  extern const KernelEntry kInst_##name[] = {__VA_ARGS__}; \
  extern const int kInst_##name##_n = (int)(sizeof(kInst_##name) / sizeof(kInst_##name[0]));

// ---- shorthand for the config graphs (expanded to canonical type expressions by registry.cpp)
typedef Pipe<Constant<1>, Sine> SineHz;
typedef Pipe<Constant<1>, WaveSynth<0, 1>> SawHz;
typedef Pipe<Unop<1, Unop<3, Unop<3, SineHz>>>, Sine> Fm;                       // sine_hz(f)*f*m+f >> sine()
typedef Pipe<Pipe<MultiSplit<2, 16>, Feedback<1, Multi<30, 0, 32, Pipe<Delay, Fir<3>>>>>,
             Binop<2, Multi<31, 0, 32, Panner<1>>, Constant<2>>> ReverbStereo;  // src/prelude.rs:1732-1762
typedef Pipe<Binop<2, Pipe<Stack<SawHz, Constant<2>>, Moog<3>>, AdsrLive>, Panner<1>> SubtractiveDry;
typedef Pipe<SubtractiveDry, Bus<MultiPass<2>, Unop<3, ReverbStereo>>> SubtractiveVoice;  // config 4

}  // namespace host
}  // namespace fdsp
