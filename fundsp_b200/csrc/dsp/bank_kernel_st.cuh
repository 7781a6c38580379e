// Stage-pipelined form of the voice-bank kernel: a voice's program is cut into K <= 4 STAGES that run in DIFFERENT warps of
// the CTA and hand 16-sample slots over through shared memory (mbarrier full / empty pairs per warp and slot).
//
// Why: a voice is a serial recurrence and a small bank has far fewer voice-warps than the GPU has warp schedulers (config 4:
// 1024 voices = 32 warps on 592 schedulers), so the plain kernel (bank_kernel.cuh) runs at the dependency latency of the WHOLE
// program — oscillator, ladder filter, envelope and pan back to back in one thread (round 1: 258 instructions per sample at
// 0.3 IPC). Only the Moog ladder (src/moog.rs:81-100, tanh in the loop) is a true per-sample recurrence; everything in front
// of it and behind it is time-parallel work that merely has to be READY. Cutting the program at the heavy leaf gives the
// recurrence a warp (and a scheduler) of its own, fed by a producer warp and drained by a consumer warp of the same voices:
//
//     stage 0 (warp 0..NW-1)      stage 1                      stage 2
//     saw table reads, dc(fc,q) -> Moog ladder (lane = voice) -> x ADSR, pan, rows / CTA mix
//
// Arithmetic per node is untouched (same `step` / `step8` code in the same order on the same 8-sample groups), so results
// are bit-identical to bank_kernel: nodes only communicate through their buffers in the reference too (src/audionode.rs:
// 1445-1449 Pipe::process: X into a temp buffer, then Y).
//
// The cut is computed from the TYPE (`StagePlan<G>`): the program is flattened along its Pipe spine, `Binop` / `Stack` whose
// LEFT operand carries the heavy leaf are re-associated with explicit pass-through channels
//     Binop<K, Pipe<A, M>, Y>  ==  Stack<A, MultiPass<Y::IN>>  >>  Stack<M, MultiPass<Y::IN>>  >>  Binop<K, MultiPass<M::OUT>, Y>
// (depth-first order of the leaves — and therefore the parameter / state / uniform word layout — is unchanged), and
// consecutive light segments are merged. A program without a heavy leaf on its spine has K = 1 and is not staged.
#pragma once
#include "bank_kernel.cuh"
#include "stage_plan.cuh"

namespace fdsp {

FDSP_DEV void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
FDSP_DEV void bar_named(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ------------------------------------------------------------------ one stage of one voice
template <class G, int NT, int MODE, bool TB, int I> struct StRun {
  typedef StagePlan<G> SP;
  typedef typename SP::stages STG;
  typedef typename ChainAt<I, STG>::type S;
  static constexpr int K = SP::K, NW = NT / 32;
  static constexpr bool FIRST = I == 0, LAST = I == K - 1;
  static constexpr int IN = S::IN, OUT = S::OUT;
  static constexpr int TS = (MODE & 2) ? mix_tile_samples(G::OUT) : 64;
  static constexpr int HS = st_hand_samples(G::OUT, (MODE & 2) != 0);
  static constexpr bool GROUP = VoiceForm<S>::group;
  // ring of boundary b (between stage b and b + 1), warp w: [slot][MID_b][HS][32]
  static FDSP_DEV float* ring_of(float* hand, int before_mid, uint32_t w, uint32_t lane, int mid) {
    return hand + ((size_t)before_mid * NT + (size_t)w * mid * 32) * ST_NSLOT * HS + lane;
  }

  // loads the words of every earlier stage into a scratch R: advances the parameter / state / uniform / delay-line cursors
  template <int J> static FDSP_DEV void skip_to(Loader& l) {
    if constexpr (J < I) { typename ChainAt<J, STG>::type::R skip; ChainAt<J, STG>::type::load(skip, l); skip_to<J + 1>(l); }
  }

  static FDSP_DEV void run(const BankArgs& a, float* tile, float* hand, uint32_t bar0, CtxT<TB>& c0, uint32_t lt, uint32_t v, bool active) {
    // a stage built around a heavy leaf is one serial chain per lane: its 8 steps of a group are unrolled outright (static register indices, the
    // group's inputs loaded up front) instead of the rotating loop the one-warp-does-everything kernel uses to keep its instruction stream small
    CtxT<TB, SpineHeavy<S>::value> c = voice_ctx<TB, SpineHeavy<S>::value>(a, v);
    c.tsm = c0.tsm; c.tsm_kind = c0.tsm_kind;
    const uint32_t w = lt >> 5, lane = lt & 31u;
    constexpr int MIDI = FIRST ? 1 : IN, MIDO = LAST ? 1 : OUT;
    // barriers: index 1 + ((b * NW + w) * NSLOT + slot) * 2 (+1 = empty)
    auto full_bar = [&](int b, uint32_t slot) { return bar0 + 8u * (1u + (((uint32_t)b * NW + w) * ST_NSLOT + slot) * 2u); };
    auto empty_bar = [&](int b, uint32_t slot) { return full_bar(b, slot) + 8u; };
    float* const rin = FIRST ? nullptr : ring_of(hand, MidBefore<I - (FIRST ? 0 : 1), STG>::value, w, lane, MIDI);
    float* const rout = LAST ? nullptr : ring_of(hand, MidBefore<I, STG>::value, w, lane, MIDO);
    typename S::R r;
    if (active) {
      Loader l{a.params, a.state, a.uniform, a.V, v, 0u, 0u, 0u, 0u};
      skip_to<0>(l);
      S::load(r, l);
    } else if (LAST && (MODE & 2)) {
      for (int e = 0; e < G::OUT * TS; e++) tile[e * (NT + 1) + lt] = 0.0f;   // columns of absent voices stay zero
    }
    const bool vec_ok = ((a.out_stride | a.out_offset) & 3u) == 0u;
    uint32_t it = 0;   // hand-off counter: the same sequence in every stage
#pragma unroll 1
    for (uint32_t t0 = 0; t0 < a.n; t0 += 64) {
      const int nb = (a.n - t0) < 64u ? (int)(a.n - t0) : 64;
      const int nfull = nb & ~7;
      c.n = nb;
      float* orow = (LAST && active && (MODE & 1)) ? a.out + (size_t)__ldg(a.row_map + v) * a.out_stride + a.out_offset + t0 : nullptr;
      const float* irow = (FIRST && IN > 0) ? a.in + a.in_offset + t0 : nullptr;
#pragma unroll 1
      for (int m0 = 0; m0 < nb; m0 += TS) {   // one pass unless the last stage owns a mix tile
        const int m1 = (m0 + TS) < nb ? (m0 + TS) : nb;
#pragma unroll 1
        for (int s0 = m0; s0 < m1; s0 += HS, it++) {
          const uint32_t slot = it % ST_NSLOT, use = it / ST_NSLOT;
          if (!FIRST) mbar_wait(full_bar(I - 1, slot), use & 1u);                          // the stage in front has filled this slot
          if (!LAST && use > 0) mbar_wait(empty_bar(I, slot), (use - 1u) & 1u);            // the stage behind has drained that slot
          const float* hin = FIRST ? nullptr : rin + (size_t)slot * MIDI * HS * 32;
          float* hout = LAST ? nullptr : rout + (size_t)slot * MIDO * HS * 32;
          const int s1 = (s0 + HS) < nb ? (s0 + HS) : nb;
          if (active) {
            const int gend = s1 < nfull ? s1 : nfull;
            c.rem = false;
#pragma unroll 1
            for (int g = s0; g < gend; g += 8) {
              Fr8<IN> in8; Fr8<OUT> o8;
              if constexpr (!GROUP) {
#pragma unroll
                for (int k = 0; k < OUT; k++) {
#pragma unroll
                  for (int j = 0; j < 8; j++) o8.v[k][j] = 0.0f;
                }
              }
#pragma unroll
              for (int k = 0; k < IN; k++) {
#pragma unroll
                for (int j = 0; j < 8; j++) in8.v[k][j] = FIRST ? __ldg(irow + (size_t)k * a.in_stride + g + j) : hin[(k * HS + (g - s0) + j) * 32];
              }
              if constexpr (GROUP) {
                c.i = g; c.first = true;
                group_step<S>(r, c, in8, o8);
              } else {
#pragma unroll 1
                for (int j = 0; j < 8; j++) {
                  Fr<IN> x; Fr<OUT> y;
#pragma unroll
                  for (int k = 0; k < IN; k++) x.v[k] = in8.v[k][0];
                  c.i = g + j; c.first = (j == 0);
                  S::template step<false>(r, c, x, y);
#pragma unroll
                  for (int k = 0; k < IN; k++) {
#pragma unroll
                    for (int q = 0; q < 7; q++) in8.v[k][q] = in8.v[k][q + 1];
                  }
#pragma unroll
                  for (int k = 0; k < OUT; k++) {
#pragma unroll
                    for (int q = 0; q < 7; q++) o8.v[k][q] = o8.v[k][q + 1];
                    o8.v[k][7] = y.v[k];
                  }
                }
              }
#pragma unroll
              for (int k = 0; k < OUT; k++) {
                if constexpr (!LAST) {
#pragma unroll
                  for (int j = 0; j < 8; j++) hout[(k * HS + (g - s0) + j) * 32] = o8.v[k][j];
                } else {
                  if (MODE & 2) {
#pragma unroll
                    for (int j = 0; j < 8; j++) tile[(k * TS + (g - m0) + j) * (NT + 1) + lt] = o8.v[k][j];
                  }
                  if (MODE & 1) {
                    float* p = orow + (size_t)k * a.out_stride + g;
                    if (vec_ok) {
                      *reinterpret_cast<float4*>(p) = make_float4(o8.v[k][0], o8.v[k][1], o8.v[k][2], o8.v[k][3]);
                      *reinterpret_cast<float4*>(p + 4) = make_float4(o8.v[k][4], o8.v[k][5], o8.v[k][6], o8.v[k][7]);
                    } else {
#pragma unroll
                      for (int j = 0; j < 8; j++) p[j] = o8.v[k][j];
                    }
                  }
                }
              }
            }
            if (s1 == nb) {  // end of the block: SIMD wrap-up, then the (size & 7) tail through the tick path
              S::end_simd(r);
              c.rem = true; c.first = false;
#pragma unroll 1
              for (int i = nfull; i < nb; i++) {
                Fr<IN> x; Fr<OUT> y;
#pragma unroll
                for (int k = 0; k < IN; k++) x.v[k] = FIRST ? __ldg(irow + (size_t)k * a.in_stride + i) : hin[(k * HS + (i - s0)) * 32];
                c.i = i;
                S::template step<false>(r, c, x, y);
#pragma unroll
                for (int k = 0; k < OUT; k++) {
                  if constexpr (!LAST) hout[(k * HS + (i - s0)) * 32] = y.v[k];
                  else {
                    if (MODE & 1) orow[(size_t)k * a.out_stride + i] = y.v[k];
                    if (MODE & 2) tile[(k * TS + (i - m0)) * (NT + 1) + lt] = y.v[k];
                  }
                }
              }
            }
          }
          if (!FIRST) mbar_arrive(empty_bar(I - 1, slot));   // 32 arrivals per barrier: each lane releases its own loads / stores
          if (!LAST) mbar_arrive(full_bar(I, slot));
        }
        if (LAST && (MODE & 2)) {
          // CTA partial mix by the last stage alone (named barrier 1): same association as bank_kernel (mix_order.h)
          bar_named(1, NT);
          constexpr int HALF = NT / 2, ROWS = G::OUT * TS;
          const int h = (int)(lt & 1u);
#pragma unroll 1
          for (int eb = (int)(lt >> 5) * 16; eb < ROWS; eb += HALF) {
            const int e = eb + (int)((lt & 31u) >> 1);
            const bool ok = e < ROWS;
            const int k = e / TS, i = e - k * TS;
            const float s = cta_half_row_sum<NT>(tile + (ok ? e : 0) * (NT + 1), h);
            const float other = __shfl_xor_sync(0xffffffffu, s, 1);
            if (ok && h == 0 && m0 + i < m1) a.partial[((size_t)blockIdx.x * G::OUT + k) * a.n + t0 + m0 + i] = s + other;
          }
          bar_named(1, NT);
        }
      }
    }
    if (active) { Saver s{a.state, a.V, v, (uint32_t)NsBefore<I, STG>::value}; S::save(r, s); }
  }
};

template <class G, int NT, int MODE, bool TB, int I> FDSP_DEV void st_dispatch(uint32_t stage, const BankArgs& a, float* tile, float* hand, uint32_t bar0, CtxT<TB>& c,
                                                                             uint32_t lt, uint32_t v, bool active) {
  if constexpr (I < StagePlan<G>::K) {
    if (stage == (uint32_t)I) StRun<G, NT, MODE, TB, I>::run(a, tile, hand, bar0, c, lt, v, active);
    else st_dispatch<G, NT, MODE, TB, I + 1>(stage, a, tile, hand, bar0, c, lt, v, active);
  }
}

// K * NT threads: thread s * NT + t runs stage s of voice (blockIdx.x * vpc + t). NT = 32 (small banks: one voice-warp per SM, every
// stage on its own scheduler) or 128.
template <class G, int NT, int MODE, bool TB>
__global__ void __launch_bounds__(StagePlan<G>::K * NT, 1) bank_kernel_st(const BankArgs a) {
  typedef StagePlan<G> SP;
  constexpr int K = SP::K, NW = NT / 32;
  static_assert(NT % 32 == 0 && NT >= 32 && (NT == 32 || NT % 8 == 0), "stage width");
  extern __shared__ __align__(16) float tile[];                // MODE&2: [OUT][TS][NT+1]; then hand-off rings; then tables
  float* hand = tile + ((MODE & 2) ? mix_tile_floats(G::OUT, NT) : 0);
  constexpr int NBAR = 1 + (K > 1 ? (K - 1) : 1) * NW * ST_NSLOT * 2;
  __shared__ __align__(8) unsigned long long bars[NBAR];
  const uint32_t tid = threadIdx.x;
  const uint32_t stage = tid / NT, lt = tid - stage * NT;
  const uint32_t vpc = a.vpc ? a.vpc : (uint32_t)NT;
  const uint32_t v = blockIdx.x * vpc + lt;
  const bool active = lt < vpc && v < a.V;
  const uint32_t bar0 = smem_addr(&bars[0]);
  if (tid == 0) {
    mbar_init(bar0, 1);
    for (int q = 1; q < NBAR; q++) mbar_init(bar0 + 8u * q, 32);
  }
  __syncthreads();
  CtxT<TB> c = voice_ctx<TB>(a, v);
  if (TB) stage_tables<G>(a, hand + st_hand_floats<G>(NT, (MODE & 2) != 0), bar0, c);
  st_dispatch<G, NT, MODE, TB, 0>(stage, a, tile, hand, bar0, c, lt, v, active);
}

}  // namespace fdsp
