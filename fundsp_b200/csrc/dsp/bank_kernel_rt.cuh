// Resident form of the voice-bank kernel for the `AudioUnit::process` call pattern (reference src/audiounit.rs:45, driven one 64-sample
// block at a time by Wave::render src/wave.rs:452-462 or an audio callback): instead of one launch per block — parameters and state
// reloaded, 161 KB of wavetables restaged, a launch and a stream synchronisation on the critical path (round 1: 31 us per block of the
// 16384-voice headline bank) — ONE launch stays resident with every voice's state in registers and serves blocks on a doorbell:
//
//   host: writes the block's inputs and size into a mapped, pinned control page, then the request's sequence number (the doorbell);
//         spins on `done` in the same page; copies the mix out.
//   GPU : thread 0 of CTA 0 polls the doorbell over PCIe and relays it to a word in device memory that the other CTAs poll; every CTA
//         evaluates the block exactly like bank_kernel (same group structure, tail, CTA mix); the last CTA to finish folds the partial
//         mixes in CTA order into the control page and publishes `done`.
// The kernel leaves by itself when asked (`RT_QUIT`) or after about a second without a request, saving the state words, so any other
// call on the bank simply stops it first (csrc/host/bank.cpp `rt_stop`). All CTAs must be co-resident: the host only uses this form
// for single-class banks whose grid fits the GPU in one wave. Results are bit-identical to process() through the one-launch-per-block path.
#pragma once
#include "bank_kernel.cuh"
#include "rt_args.h"

namespace fdsp {

FDSP_DEV uint32_t rt_ld_sys(const volatile uint32_t* p) { uint32_t v; asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

template <class G, int NT, bool TB>
__global__ void __launch_bounds__(NT, FDSP_MIN_CTAS) bank_kernel_rt(const BankArgs a, const RtArgs rt) {
  extern __shared__ __align__(16) float tile[];  // [OUT][TS][NT+1]; TB: table data after it
  __shared__ uint32_t s_cmd, s_n, s_last;
  __shared__ float s_in[(G::IN > 0 ? G::IN : 1) * 64];   // the block's shared inputs: fetched from the control page once per CTA, not once per voice
  const uint32_t tid = threadIdx.x;
  const uint32_t vpc = a.vpc ? a.vpc : (uint32_t)NT;
  const uint32_t v = blockIdx.x * vpc + tid;
  const bool active = tid < vpc && v < a.V;
  constexpr int IN = G::IN, OUT = G::OUT;
  constexpr int TS = mix_tile_samples(OUT);
  typename G::R r;
  CtxT<TB> c = voice_ctx<TB>(a, v);
  if (TB) {
    __shared__ __align__(8) unsigned long long mbar;
    const uint32_t bar = smem_addr(&mbar);
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    stage_tables<G>(a, tile + mix_tile_floats(OUT, NT), bar, c);
  }
  if (active) {
    Loader l{a.params, a.state, a.uniform, a.V, v, 0u, 0u, 0u, 0u};
    G::load(r, l);
  } else {
    for (int e = 0; e < OUT * TS; e++) tile[e * (NT + 1) + tid] = 0.0f;  // columns of absent voices stay zero
  }
  uint32_t seq = rt.first_seq - 1u;
#pragma unroll 1
  for (;;) {
    // ---- wait for the next request
    if (tid == 0) {
      uint32_t cur = seq, spins = 0;
      if (blockIdx.x == 0) {
        do { cur = rt_ld_sys(&rt.ctl->doorbell); } while (cur == seq && ++spins < RT_POLL_LIMIT_HOST);
        if (cur == seq) cur = RT_QUIT;                                   // idle: leave (the host restarts the kernel with the next block)
        const uint32_t n = cur == RT_QUIT ? 0u : rt_ld_sys(&rt.ctl->size);
        rt.relay[1] = n;
        __threadfence();
        *reinterpret_cast<volatile uint32_t*>(rt.relay) = cur;
        s_n = n;
      } else {
        do { cur = rt_ld_sys(rt.relay); } while (cur == seq && ++spins < RT_POLL_LIMIT_RELAY);
        if (cur == seq) cur = RT_QUIT;
        __threadfence();
        s_n = rt_ld_sys(rt.relay + 1);
      }
      s_cmd = cur;
    }
    __syncthreads();
    const uint32_t cmd = s_cmd;
    const int nb = (int)s_n;
    if (cmd == RT_QUIT) break;
    seq = cmd;
    for (int e = (int)tid; e < IN * 64; e += NT) s_in[e] = (e & 63) < nb ? __ldcv(&rt.ctl->in[e >> 6][e & 63]) : 0.0f;
    __syncthreads();
    // ---- one block, as bank_kernel evaluates it (MODE 2)
#pragma unroll 1
    for (int s0 = 0; s0 < nb; s0 += TS) {
      const int s1 = (s0 + TS) < nb ? (s0 + TS) : nb;
      if (active) {
        auto put = [&](int k, int i, float y) { tile[(k * TS + (i - s0)) * (NT + 1) + tid] = y; };
        walk_block<G>(r, c, nb, s0, s1, [&](int k, int i, int j) { return s_in[k * 64 + i + j]; }, put, [](int, int, const float (&)[8]) {}, put);
      }
      // CTA partial mix: the association of bank_kernel (mix_order.h)
      __syncthreads();
      constexpr int HALF = NT / 2, ROWS = OUT * TS;
      const int h = (int)(tid & 1u);
#pragma unroll 1
      for (int eb = (int)(tid >> 5) * 16; eb < ROWS; eb += HALF) {
        const int e = eb + (int)((tid & 31u) >> 1);
        const bool ok = e < ROWS;
        const int k = e / TS, i = e - k * TS;
        const float s = cta_half_row_sum<NT>(tile + (ok ? e : 0) * (NT + 1), h);
        const float other = __shfl_xor_sync(0xffffffffu, s, 1);
        if (ok && h == 0 && s0 + i < s1) a.partial[((size_t)blockIdx.x * OUT + k) * 64 + s0 + i] = s + other;
      }
      __syncthreads();
    }
    // ---- the last CTA to finish folds the partials in CTA order (= mix_reduce_kernel) into the control page and publishes `done`
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1u) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
      __threadfence();
      // CTA-order left fold of the partials (= mix_reduce_kernel, bit for bit). (A version that staged the partials in shared memory first
      // measured SLOWER — 44.5 vs 23.4 us per block at 148 CTAs: one CTA cannot keep enough loads in flight to win back the extra pass.)
      for (uint32_t e = tid; e < (uint32_t)OUT * (uint32_t)nb; e += NT) {
        const uint32_t ch = e / (uint32_t)nb, t = e - ch * (uint32_t)nb;
        rt.ctl->out[ch][t] = cta_order_fold(a.partial + (size_t)ch * 64 + t, (size_t)OUT * 64, gridDim.x, [](const float* p) { return __ldcg(p); });
      }
      __threadfence_system();
      __syncthreads();
      if (tid == 0) { *a.ticket = 0u; __threadfence(); rt.ctl->done = seq; }
    }
  }
  if (active) {
    Saver s{a.state, a.V, v, 0u};
    G::save(r, s);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0 && atomicAdd(rt.relay + 2, 1u) == gridDim.x - 1u) { rt.relay[2] = 0u; __threadfence_system(); rt.ctl->done = RT_EXITED; }
}

}  // namespace fdsp
