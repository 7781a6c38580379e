// TEST INFRASTRUCTURE — one graph class of the mock "GPU" (tests/cpp/mock/registry_mock.cpp): the DEVICE node library compiled for the
// CPU (FDSP_HOST_EMUL) and walked through the kernels' own walk_block (dsp/voice_block.cuh) for every voice of a launch, reading and
// writing the same argument block (BankArgs) the real kernel gets. The per-CTA mix partials fold each row of a CTA's voice outputs in
// the kernels' association (dsp/mix_order.h), so they equal the GPU's bit for bit.
// Build: g++ -std=c++17 -O1 -ffp-contract=off -shared -fPIC -DGRAPH='<type expression>' -I fundsp_b200/csrc emul_module.cpp
#define FDSP_HOST_EMUL 1
#include <algorithm>
#include <vector>

#include "dsp/mix_order.h"
#include "dsp/voice_block.cuh"

using namespace fdsp;
typedef GRAPH G;

extern "C" void fdsp_emul_layout(int* lay) {
  lay[0] = G::IN; lay[1] = G::OUT; lay[2] = G::NP; lay[3] = G::NS; lay[4] = G::NU; lay[5] = WaveKind<G>::value;
}

// per_voice_in != null: voice v reads its OWN input rows per_voice_in + v * voice_stride (+ k * a.in_stride + a.in_offset + t) instead of the
// shared bank input — how the mock runs the reverb stage of a two-stage class on the dry rows of the voices (registry_mock.cpp launch_fdn)
extern "C" int fdsp_emul_launch_ex(const BankArgs* ap, int mode, const float* per_voice_in, uint64_t voice_stride);
extern "C" int fdsp_emul_launch(const BankArgs* ap, int mode) { return fdsp_emul_launch_ex(ap, mode, nullptr, 0); }
extern "C" int fdsp_emul_launch_ex(const BankArgs* ap, int mode, const float* per_voice_in, uint64_t voice_stride) {
  const BankArgs& a = *ap;
  constexpr int IN = G::IN, OUT = G::OUT, NT = 128;
  const uint32_t vpc = a.vpc ? a.vpc : (uint32_t)NT, grid = (a.V + vpc - 1) / vpc;
  if ((mode & 2) && !a.partial) return 1;
  if ((mode & 1) && !a.out) return 2;
  if (vpc > (uint32_t)NT) return 3;
  std::vector<float> tile((mode & 2) ? (size_t)OUT * a.n * NT : 0);   // one CTA's mix tile: row k * n + t, column = voice within the CTA
  for (uint32_t b = 0; b < grid; b++) {
    std::fill(tile.begin(), tile.end(), 0.0f);   // columns of absent voices stay zero
    for (uint32_t v = b * vpc; v < a.V && v < (b + 1) * vpc; v++) {
      typename G::R r;
      CtxT<false> c = voice_ctx<false>(a, v);
      Loader l{a.params, a.state, a.uniform, a.V, v, 0u, 0u, 0u, 0u};
      G::load(r, l);
      for (uint32_t t0 = 0; t0 < a.n; t0 += 64) {
        const int nb = (a.n - t0) < 64u ? (int)(a.n - t0) : 64;
        const float* irow = (IN > 0) ? (per_voice_in ? per_voice_in + (size_t)v * voice_stride : a.in) + a.in_offset + t0 : nullptr;
        auto put = [&](int k, int i, float y) {
          const uint32_t t = t0 + (uint32_t)i;
          if (mode & 1) a.out[(size_t)(a.row_map[v] + (uint32_t)k) * a.out_stride + a.out_offset + t] = y;
          if (mode & 2) tile[((size_t)k * a.n + t) * NT + (v - b * vpc)] = y;
        };
        walk_block<G>(r, c, nb, 0, nb, [&](int k, int i, int j) { return irow[(size_t)k * a.in_stride + i + j]; }, put, [](int, int, const float (&)[8]) {}, put);
      }
      Saver s{a.state, a.V, v, 0u};
      G::save(r, s);
    }
    if (mode & 2)
      for (size_t e = 0; e < (size_t)OUT * a.n; e++) a.partial[(size_t)b * OUT * a.n + e] = cta_half_row_sum<NT>(&tile[e * NT], 0) + cta_half_row_sum<NT>(&tile[e * NT], 1);
  }
  if ((mode & 2) && a.ticket) {   // the fused finish of short launches (bank_kernel.cuh): CTA-order left fold into the mix
    for (uint32_t ch = 0; ch < (uint32_t)OUT; ch++)
      for (uint32_t t = 0; t < a.n; t++) {
        const float s = cta_order_fold(a.partial + (size_t)ch * a.n + t, (size_t)OUT * a.n, grid, [](const float* p) { return *p; });
        float* p = a.mix + (size_t)ch * a.mix_stride + a.mix_offset + t;
        *p = a.mix_accumulate ? *p + s : s;
      }
  }
  return 0;
}
