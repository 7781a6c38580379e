// How one voice walks a block: the form its program takes over an 8-sample group, the block context built from the launch
// arguments, and the order of the group, end_simd and tail-sample steps. bank_kernel and bank_kernel_rt run it on the GPU; the
// CPU suite's host emulation (tests/cpp/device_emul.cpp) and mock device (tests/cpp/mock/emul_module.cpp) run the same code
// compiled for the host (FDSP_HOST_EMUL), so this header holds no inline assembly.
#pragma once
#include "nodes.cuh"

namespace fdsp {

#ifndef FDSP_NO_GROUP
#define FDSP_NO_GROUP 0
#endif
#ifndef FDSP_GROUP_COST
#define FDSP_GROUP_COST 256   // programs whose group form unrolls to at most this many instructions per sample are evaluated 8 samples at a time
#endif

// group: node by node over the 8-sample group (group_step). Otherwise the program steps sample by sample, the 8 steps of a group
// unrolled `unroll` times: big programs (e.g. the 32-line FDN in thread-per-voice form) are not unrolled over the group.
template <class G> struct VoiceForm {
  static constexpr bool group = GroupPlan<G>::ok && GroupPlan<G>::code <= FDSP_GROUP_COST && !FDSP_NO_GROUP;
  static constexpr int unroll = group ? 8 : (Cost<G>::value <= 160 ? 8 : (Cost<G>::value <= 320 ? 4 : (Cost<G>::value <= 640 ? 2 : 1)));
};

// Block context of voice v of a launch, with no tables staged in shared memory yet. UH: run heavy leaves fully unrolled (a stage of
// bank_kernel_st built around one).
template <bool TB, bool UH = false> FDSP_DEV CtxT<TB, UH> voice_ctx(const BankArgs& a, uint32_t v) {
  CtxT<TB, UH> c;
  c.wt = a.wt; c.tsm = 0u; c.tsm_kind = -1; c.dl = a.dline; c.V = a.V; c.v = v; c.sr = a.sr; c.sd64 = a.sd64; c.sd32 = a.sd32;
  c.rp = a.params; c.rs0 = a.state0; c.ru = a.uniform; c.dl_total = a.dl_floats;
  c.i = 0; c.n = 0; c.first = false; c.rem = false;
  return c;
}

// Samples [s0, s1) of a block of nb <= 64 samples: the 8-sample groups that start there, then, when s1 == nb, end_simd and the
// (nb & 7) tail through the tick path (c.rem), as the reference's `process` exposes a block to the nodes. s0 is a multiple of 8.
//   in(k, i, j)       input channel k at sample i + j of the block (j: the sample within a group, 0 in the tail)
//   put(k, i, y)      output channel k at sample i of a group, as soon as it is computed
//   put8(k, g, v)     output channel k of the whole group at g (v[j] is sample g + j), after its put() calls
//   put_tail(k, i, y) output channel k at tail sample i
template <class G, class C, class In, class Put, class Put8, class PutTail>
FDSP_DEV void walk_block(typename G::R& r, C& c, int nb, int s0, int s1, In&& in, Put&& put, Put8&& put8, PutTail&& put_tail) {
  constexpr int IN = G::IN, OUT = G::OUT;
  const int nfull = nb & ~7;
  const int gend = s1 < nfull ? s1 : nfull;
  c.n = nb;
  c.rem = false;
#pragma unroll 1
  for (int g = s0; g < gend; g += 8) {
    float ob[OUT > 0 ? OUT : 1][8];
    if constexpr (VoiceForm<G>::group) {
      Fr8<IN> in8; Fr8<OUT> o8;
#pragma unroll
      for (int k = 0; k < IN; k++) {
#pragma unroll
        for (int j = 0; j < 8; j++) in8.v[k][j] = in(k, g, j);
      }
      c.i = g; c.first = true;
      group_step<G>(r, c, in8, o8);
#pragma unroll
      for (int k = 0; k < OUT; k++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          ob[k][j] = o8.v[k][j];
          put(k, g + j, o8.v[k][j]);
        }
      }
    } else {
#pragma unroll(VoiceForm<G>::unroll)
      for (int j = 0; j < 8; j++) {
        Fr<IN> x; Fr<OUT> y;
#pragma unroll
        for (int k = 0; k < IN; k++) x.v[k] = in(k, g, j);
        c.i = g + j; c.first = (j == 0);
        G::template step<false>(r, c, x, y);
#pragma unroll
        for (int k = 0; k < OUT; k++) {
          ob[k][j] = y.v[k];
          put(k, g + j, y.v[k]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < OUT; k++) put8(k, g, ob[k]);
  }
  if (s1 == nb) {  // end of the block: wrap up the SIMD part, then the (size & 7) tail through the tick path
    G::end_simd(r);
    c.rem = true; c.first = false;
#pragma unroll 1
    for (int i = nfull; i < nb; i++) {
      Fr<IN> x; Fr<OUT> y;
#pragma unroll
      for (int k = 0; k < IN; k++) x.v[k] = in(k, i, 0);
      c.i = i;
      G::template step<false>(r, c, x, y);
#pragma unroll
      for (int k = 0; k < OUT; k++) put_tail(k, i, y.v[k]);
    }
  }
}

}  // namespace fdsp
