// fundsp_b200 voice-bank kernel: one thread = one voice instance of the graph type G, V voices in
// lockstep. Replaces the reference's per-voice `AudioUnit::process` recursion (src/audiounit.rs:393-395,
// src/audionode.rs:85-105,1445-1449) driven by `Wave::render` (src/wave.rs:441-466).
//
// Launch shape: grid = ceil(V / NT) CTAs of NT threads; each thread keeps G::R (parameters + state) in
// registers for all blocks of the launch and walks time in 64-sample blocks (8 SIMD groups of 8 + tail),
// exactly the block structure the reference's `process` path exposes to the nodes.
// Outputs: MODE bit 0 = per-voice rows out[(v*OUT+c)*stride + off + t] written as coalesced-by-row
// 16-byte stores; MODE bit 1 = per-CTA index-order partial mix (shared-memory transpose + sequential
// column sums), finished by mix_reduce_kernel in CTA order (deterministic).
#pragma once
#include "nodes.cuh"
#include "mix_order.h"
#include "voice_block.cuh"

namespace fdsp {



// ---- TMA (bulk async copy) + mbarrier primitives used to stage wavetables into shared memory
FDSP_DEV uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
FDSP_DEV void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
FDSP_DEV void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
FDSP_DEV void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
FDSP_DEV void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar),
      "r"(parity)
      : "memory");
}

// TB: stage the wavetable data of kind WaveKind<G> in shared memory at `tsm` (one TMA bulk copy per 32 KB slice on the initialised
// mbarrier `bar`), so the per-sample table taps become conflict-light LDS instead of divergent LDG; then point the context at it.
template <class G, class C> FDSP_DEV void stage_tables(const BankArgs& a, float* tsm, uint32_t bar, C& c) {
  constexpr int KIND = WaveKind<G>::value >= 0 ? WaveKind<G>::value : 0;
  const uint32_t bytes = (uint32_t)a.wt[KIND].total * 4u;
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, bytes);
    const char* src = reinterpret_cast<const char*>(a.wt[KIND].data);
    for (uint32_t o = 0; o < bytes; o += 32768u) bulk_g2s(smem_addr(tsm) + o, src + o, (bytes - o) < 32768u ? (bytes - o) : 32768u, bar);
  }
  mbar_wait(bar, 0);
  c.tsm = smem_addr(tsm); c.tsm_kind = KIND;
}

#ifndef FDSP_MIN_CTAS
#define FDSP_MIN_CTAS 1   // one resident CTA per SM is all a bank needs: lets ptxas spend registers on overlapping the 8-sample group
#endif

template <class G, int NT, int MODE, bool TB>
__global__ void __launch_bounds__(NT, FDSP_MIN_CTAS) bank_kernel(const BankArgs a) {
  extern __shared__ __align__(16) float tile[];  // MODE&2: [OUT][TS][NT+1]; TB: table data after it
  const uint32_t tid = threadIdx.x;
  const uint32_t vpc = a.vpc ? a.vpc : (uint32_t)NT;
  const uint32_t v = blockIdx.x * vpc + tid;
  const bool active = tid < vpc && v < a.V;
  constexpr int IN = G::IN, OUT = G::OUT;
  constexpr int TS = (MODE & 2) ? mix_tile_samples(OUT) : 64;

  typename G::R r;
  CtxT<TB> c = voice_ctx<TB>(a, v);
  if (TB) {
    __shared__ __align__(8) unsigned long long mbar;
    const uint32_t bar = smem_addr(&mbar);
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    stage_tables<G>(a, tile + ((MODE & 2) ? mix_tile_floats(OUT, NT) : 0), bar, c);
  }
  if (active) {
    Loader l{a.params, a.state, a.uniform, a.V, v, 0u, 0u, 0u, 0u};
    G::load(r, l);
  } else if (MODE & 2) {
    for (int e = 0; e < OUT * TS; e++) tile[e * (NT + 1) + tid] = 0.0f;  // columns of absent voices stay zero
  }
  const bool vec_ok = ((a.out_stride | a.out_offset) & 3u) == 0u;

#pragma unroll 1
  for (uint32_t t0 = 0; t0 < a.n; t0 += 64) {
    const int nb = (a.n - t0) < 64u ? (int)(a.n - t0) : 64;
    float* orow = (active && (MODE & 1)) ? a.out + (size_t)__ldg(a.row_map + v) * a.out_stride + a.out_offset + t0 : nullptr;
    const float* irow = (IN > 0) ? a.in + a.in_offset + t0 : nullptr;
#pragma unroll 1
    for (int s0 = 0; s0 < nb; s0 += TS) {   // one pass when there is no mix tile (TS = 64)
      const int s1 = (s0 + TS) < nb ? (s0 + TS) : nb;
      if (active) {
        walk_block<G>(
            r, c, nb, s0, s1, [&](int k, int i, int j) { return __ldg(irow + (size_t)k * a.in_stride + i + j); },
            [&](int k, int i, float y) {
              if (MODE & 2) tile[(k * TS + (i - s0)) * (NT + 1) + tid] = y;
            },
            [&](int k, int g, const float (&y)[8]) {
              if (MODE & 1) {
                float* p = orow + (size_t)k * a.out_stride + g;
                if (vec_ok) {
                  *reinterpret_cast<float4*>(p) = make_float4(y[0], y[1], y[2], y[3]);
                  *reinterpret_cast<float4*>(p + 4) = make_float4(y[4], y[5], y[6], y[7]);
                } else {
#pragma unroll
                  for (int j = 0; j < 8; j++) p[j] = y[j];
                }
              }
            },
            [&](int k, int i, float y) {
              if (MODE & 1) orow[(size_t)k * a.out_stride + i] = y;
              if (MODE & 2) tile[(k * TS + (i - s0)) * (NT + 1) + tid] = y;
            });
      }
      if (MODE & 2) {
        // CTA partial mix: two threads per (channel, sample) row, each folding one half of the voice columns (mix_order.h)
        __syncthreads();
        constexpr int HALF = NT / 2, ROWS = OUT * TS;
        const int h = (int)(tid & 1u);
#pragma unroll 1
        for (int eb = (int)(tid >> 5) * 16; eb < ROWS; eb += HALF) {   // warp-uniform trip count (full-mask shuffle below)
          const int e = eb + (int)((tid & 31u) >> 1);
          const bool ok = e < ROWS;
          const int k = e / TS, i = e - k * TS;
          const float s = cta_half_row_sum<NT>(tile + (ok ? e : 0) * (NT + 1), h);
          const float other = __shfl_xor_sync(0xffffffffu, s, 1);
          if (ok && h == 0 && s0 + i < s1) a.partial[((size_t)blockIdx.x * OUT + k) * a.n + t0 + s0 + i] = s + other;
        }
        __syncthreads();
      }
    }
  }
  if (active) {
    Saver s{a.state, a.V, v, 0u};
    G::save(r, s);
  }
  if ((MODE & 2) && a.ticket) {   // fused finish of the mix-down: same CTA-order left fold as mix_reduce_kernel
    __shared__ uint32_t s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1u) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
      __threadfence();
      for (uint32_t e = tid; e < (uint32_t)OUT * a.n; e += NT) {
        const uint32_t ch = e / a.n, t = e - ch * a.n;
        const float s = cta_order_fold(a.partial + (size_t)ch * a.n + t, (size_t)OUT * a.n, gridDim.x, [](const float* p) { return __ldcg(p); });
        float* p = a.mix + (size_t)ch * a.mix_stride + a.mix_offset + t;
        *p = a.mix_accumulate ? *p + s : s;
      }
      if (tid == 0) *a.ticket = 0u;
    }
  }
}

// Finishes the mix-down: mix[c][off + t] (+)= sum over CTAs in CTA order (deterministic).
static __global__ void mix_reduce_kernel(const float* partial, uint32_t nparts, uint32_t outs, uint32_t n, float* mix,
                                  uint32_t mix_stride, uint32_t mix_offset, int accumulate) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= outs * n) return;
  const uint32_t c = e / n, t = e % n;
  const float s = cta_order_fold(partial + (size_t)c * n + t, (size_t)outs * n, nparts, [](const float* p) { return *p; });
  float* p = mix + (size_t)c * mix_stride + mix_offset + t;
  *p = accumulate ? *p + s : s;
}


// Mix-down of per-voice rows in a FIXED association order, for parity with a reference `Net` whose outputs are adder
// trees (src/net.rs:1693-1767 Net::bus adds one Binop<Add,Pass,Pass> vertex per output per call):
//   pairwise = level-wise adjacent pairing with the odd element carried up (the balanced `Net::bus` tree),
//   chain    = left fold in voice order (a left-leaning chain of `&`, or the index-order sum of a Sequencer).
// One thread per (channel, sample); rows are read coalesced along time; the association is a binary-carry stack.
// Level 1 of the balanced tree for big banks: the subtree sum of every COMPLETE block of 2^LB consecutive voices, one thread per (block,
// channel, sample). A complete aligned block is a whole subtree of the level-wise pairing, so its sum does not depend on the rest of the bank;
// tree_mix_kernel then pushes the block sums at level LB of its carry stack (exactly what pushing the block's voices one by one would have left
// there) and goes on with the tail voices. Same association, every bit — with V / 2^LB times the parallelism over the voices.
template <int LB>
static __global__ void tree_mix_block_kernel(const float* __restrict__ rows, uint32_t outs, uint32_t row_stride, uint32_t row_offset, uint32_t n, float* __restrict__ partial) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x, blk = blockIdx.y;
  if (e >= outs * n) return;
  const uint32_t ch = e / n, t = e - ch * n;
  const size_t vstep = (size_t)outs * row_stride;
  const float* p = rows + (size_t)ch * row_stride + row_offset + t + (size_t)blk * ((size_t)1 << LB) * vstep;
  float st[LB + 1];
  for (uint32_t v0 = 0; v0 < (1u << LB); v0 += 8) {
    float b[8];
#pragma unroll
    for (int u = 0; u < 8; u++) b[u] = __ldg(p + (size_t)(v0 + u) * vstep);
#pragma unroll
    for (int u = 0; u < 8; u++) carry_push(st, b[u], v0 + u, 0);
  }
  partial[((size_t)blk * outs + ch) * n + t] = st[LB];
}

static __global__ void tree_mix_kernel(const float* __restrict__ rows, uint32_t V, uint32_t outs, uint32_t row_stride, uint32_t row_offset, uint32_t n,
                                       float* mix, uint32_t mix_stride, uint32_t mix_offset, int pairwise, const float* __restrict__ partial = nullptr,
                                       uint32_t nfull = 0, int lb = 0) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= outs * n) return;
  const uint32_t ch = e / n, t = e - ch * n;
  const float* p = rows + (size_t)ch * row_stride + row_offset + t;
  const size_t vstep = (size_t)outs * row_stride;
  float x;
  if (pairwise) {
    float st[32];
    // complete blocks of 2^lb voices arrive as their subtree sums (tree_mix_block_kernel): pushed at level lb with the block index as the carry pattern
    for (uint32_t bk = 0; bk < nfull; bk++) {
      carry_push(st, __ldg(partial + ((size_t)bk * outs + ch) * n + t), bk, lb);
    }
    for (uint32_t v0 = nfull << lb; v0 < V; v0 += 8) {
      float b[8];
#pragma unroll
      for (int u = 0; u < 8; u++) b[u] = (v0 + u < V) ? __ldg(p + (size_t)(v0 + u) * vstep) : 0.0f;
#pragma unroll
      for (int u = 0; u < 8; u++) {
        if (v0 + u < V) carry_push(st, b[u], v0 + u, 0);
      }
    }
    x = carry_finish(st, V);
  } else {
    x = __ldg(p);
    for (uint32_t v = 1; v < V; v++) x += __ldg(p + (size_t)v * vstep);
  }
  mix[(size_t)ch * mix_stride + mix_offset + t] = x;
}

}  // namespace fdsp
