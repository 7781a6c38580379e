// TEST INFRASTRUCTURE — host emulation of ONE voice of a fused device program.
//
// Compiles the DEVICE node library (fundsp_b200/csrc/dsp/nodes.cuh) for the CPU (FDSP_HOST_EMUL shims in math.cuh) and walks it
// through a block with the kernels' own walk_block (dsp/voice_block.cuh: 8-sample groups, end_simd, tick-path tail), so that the
// CPU-only test suite can compare the device templates against the oracle bit for bit. It is never linked into the product and is not a fallback:
// the product library has no CPU DSP path. Build: g++ -std=c++17 -O1 -ffp-contract=off -DGRAPH='<type expression>' device_emul.cpp
//
// stdin-free protocol: argv[1] = input blob, argv[2] = output file.
//   blob: u32 np, ns, nu, nin, n ; f64 sr ; u32 P[np], S[ns], U[nu] ; f32 in[nin][n] ;
//         u32 ntables ; per table: u32 kind, n, total ; f32 pitch[n] ; i32 off[n] ; i32 len[n] ; f32 data[total]   (guard-sample layout)
//   out : f32 y[OUT][n]
#define FDSP_HOST_EMUL 1
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../fundsp_b200/csrc/dsp/voice_block.cuh"
#ifdef STAGED
#include "../../fundsp_b200/csrc/dsp/stage_plan.cuh"
#endif

using namespace fdsp;
typedef GRAPH G;

#ifdef STAGED
// -DSTAGED: the stages of StagePlan<G> (dsp/stage_plan.cuh, what bank_kernel_st runs in different warps) evaluated BACK TO BACK per 64-sample
// block through [channel][64] buffers, each stage with its own registers loaded from its own span of the word arrays.
template <int I> struct StageEmul {
  typedef typename StagePlan<G>::stages STG;
  static constexpr int K = StagePlan<G>::K;
  typedef typename ChainAt<(I < K ? I : 0), STG>::type S;
  template <int J> static void skip(Loader& l) { if constexpr (J < I) { typename ChainAt<J, STG>::type::R sk; ChainAt<J, STG>::type::load(sk, l); skip<J + 1>(l); } }
  static void block(typename S::R& r, const BankArgs& a, int nb, const float* in /*[IN][64]*/, float* out /*[OUT][64]*/) {
    // like bank_kernel_st: a stage built around a heavy leaf runs the leaf's 8 steps fully unrolled (and takes its steady-group path)
    CtxT<false, SpineHeavy<S>::value> c = voice_ctx<false, SpineHeavy<S>::value>(a, 0);
    auto put = [&](int k, int i, float y) { out[k * 64 + i] = y; };
    walk_block<S>(r, c, nb, 0, nb, [&](int k, int i, int j) { return in[k * 64 + i + j]; }, put, [](int, int, const float (&)[8]) {}, put);
  }
};
template <int I> struct StageRegs { typename StageEmul<I>::S::R r; StageRegs<I + 1> next; };
template <> struct StageRegs<StagePlan<G>::K> {};
template <int I> static void staged_load(StageRegs<I>& regs, const uint32_t* P, const uint32_t* S, const uint32_t* U, uint32_t& dl) {
  if constexpr (I < StagePlan<G>::K) {
    Loader l{P, S, U, 1u, 0u, 0u, 0u, 0u, 0u};
    StageEmul<I>::template skip<0>(l);
    StageEmul<I>::S::load(regs.r, l);
    dl = l.dl;
    staged_load<I + 1>(regs.next, P, S, U, dl);
  }
}
template <int I> static void staged_block(StageRegs<I>& regs, const BankArgs& args, int nb, float* a, float* b) {
  if constexpr (I < StagePlan<G>::K) {
    StageEmul<I>::block(regs.r, args, nb, a, b);
    staged_block<I + 1>(regs.next, args, nb, b, a);   // ping-pong: the output of stage I is the input of stage I + 1
  }
}
#endif

int main(int argc, char** argv) {
  if (argc < 3) return 2;
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 3;
  uint32_t hdr[5]; double sr;
  if (fread(hdr, 4, 5, f) != 5 || fread(&sr, 8, 1, f) != 1) return 4;
  const uint32_t np = hdr[0], ns = hdr[1], nu = hdr[2], nin = hdr[3], n = hdr[4];
  if ((int)nin != G::IN) { fprintf(stderr, "inputs %u != %d\n", nin, G::IN); return 5; }
  std::vector<uint32_t> P(np + 1), S(ns + 1), U(nu + 1);
  if (fread(P.data(), 4, np, f) != np || fread(S.data(), 4, ns, f) != ns || fread(U.data(), 4, nu, f) != nu) return 6;
  std::vector<float> in((size_t)(nin ? nin : 1) * n), out((size_t)(G::OUT ? G::OUT : 1) * n, 0.0f);
  if (nin && fread(in.data(), 4, (size_t)nin * n, f) != (size_t)nin * n) return 7;
  WaveTableDev wt[6] = {};
  std::vector<std::vector<float>> tdata;
  uint32_t ntab = 0;
  if (fread(&ntab, 4, 1, f) == 1) {
    tdata.reserve(ntab);   // keep the data pointers stable
    for (uint32_t t = 0; t < ntab; t++) {
      uint32_t h3[3];
      if (fread(h3, 4, 3, f) != 3 || h3[0] > 5 || h3[1] > 48) return 10;
      WaveTableDev& w = wt[h3[0]];
      w.n = (int)h3[1]; w.total = (int)h3[2];
      if (fread(w.pitch, 4, h3[1], f) != h3[1] || fread(w.off, 4, h3[1], f) != h3[1] || fread(w.len, 4, h3[1], f) != h3[1]) return 11;
      tdata.emplace_back(h3[2]);
      if (fread(tdata.back().data(), 4, h3[2], f) != h3[2]) return 12;
      w.data = tdata.back().data();
    }
  }
  fclose(f);
  BankArgs args = {};   // one voice: the launch arguments the block context is built from
  args.params = P.data(); args.state = S.data(); args.uniform = U.data(); args.state0 = S.data(); args.wt = wt; args.V = 1;
  args.sr = (float)sr; args.sd64 = (float)(1.0 / sr); args.sd32 = 1.0f / (float)sr;

#ifdef STAGED
  {
    static_assert(StagePlan<G>::K >= 2, "the graph has no stage plan (no heavy leaf on its spine)");
    fprintf(stderr, "stages=%d\n", StagePlan<G>::K);
    StageRegs<0> regs; uint32_t dl = 0;
    staged_load<0>(regs, P.data(), S.data(), U.data(), dl);
    std::vector<float> dline((size_t)dl + 1, 0.0f);
    fprintf(stderr, "dl=%u\n", dl);
    args.dline = dline.data(); args.dl_floats = dl;
    constexpr int CH = 64;   // widest boundary the ping-pong buffers hold
    std::vector<float> bufa(CH * 64), bufb(CH * 64);
    for (uint32_t t0 = 0; t0 < n; t0 += 64) {
      const int nb = (n - t0) < 64u ? (int)(n - t0) : 64;
      for (uint32_t k = 0; k < nin; k++) for (int i = 0; i < nb; i++) bufa[k * 64 + i] = in[(size_t)k * n + t0 + i];
      staged_block<0>(regs, args, nb, bufa.data(), bufb.data());
      const float* res = (StagePlan<G>::K & 1) ? bufb.data() : bufa.data();
      for (int k = 0; k < G::OUT; k++) for (int i = 0; i < nb; i++) out[(size_t)k * n + t0 + i] = res[k * 64 + i];
    }
    FILE* o = fopen(argv[2], "wb");
    if (!o) return 9;
    fwrite(out.data(), 4, (size_t)G::OUT * n, o);
    fclose(o);
    return 0;
  }
#endif
  typename G::R r;
  Loader l{P.data(), S.data(), U.data(), 1u, 0u, 0u, 0u, 0u, 0u};
  G::load(r, l);
  if (l.pi > np || l.si > ns || l.ui > nu) { fprintf(stderr, "word layout mismatch: consumed %u/%u/%u of %u/%u/%u\n", l.pi, l.si, l.ui, np, ns, nu); return 8; }
  std::vector<float> dline((size_t)l.dl + 1, 0.0f);
  fprintf(stderr, "dl=%u\n", l.dl);   // the delay-line floats the device program claims (the host must allocate exactly this)
  args.dline = dline.data(); args.dl_floats = l.dl;
  CtxT<false> c = voice_ctx<false>(args, 0);
  for (uint32_t t0 = 0; t0 < n; t0 += 64) {
    const int nb = (n - t0) < 64u ? (int)(n - t0) : 64;
    auto put = [&](int k, int i, float y) { out[(size_t)k * n + t0 + i] = y; };
    walk_block<G>(r, c, nb, 0, nb, [&](int k, int i, int j) { return in[(size_t)k * n + t0 + i + j]; }, put, [](int, int, const float (&)[8]) {}, put);
  }
  FILE* o = fopen(argv[2], "wb");
  if (!o) return 9;
  fwrite(out.data(), 4, (size_t)G::OUT * n, o);
  fclose(o);
  return 0;
}
