// Plain-data kernel arguments shared by host (csrc/host) and device (csrc/dsp) code.
#pragma once
#ifndef __CUDACC_RTC__
#include <cstddef>
#include <cstdint>
#endif

namespace fdsp {

// Wavetable set for one waveform (reference src/wavetable.rs:82-123): up to 48 tables, ascending pitch.
struct WaveTableDev {
  int n;
  float pitch[48];
  int off[48];
  int len[48];
  int total;          // floats in `data`
  const float* data;
};

// Depth (samples) of the CTA mix tile [OUT][TS][NT+1]: the tile is reduced and recycled every TS samples, so wide
// voices keep a ~33 KB tile and the 164 KB wavetable set still fits beside it in shared memory.
#ifdef __CUDACC__
#define FDSP_HDC __host__ __device__
#else
#define FDSP_HDC
#endif
FDSP_HDC constexpr int mix_tile_samples(int outs) { return outs <= 1 ? 64 : (outs == 2 ? 32 : (outs <= 4 ? 16 : 8)); }
FDSP_HDC constexpr size_t mix_tile_floats(int outs, int nt) { return (size_t)outs * (size_t)mix_tile_samples(outs) * (size_t)(nt + 1); }

// Hand-off rings of the stage-pipelined kernel (bank_kernel_st.cuh): per channel crossing a stage boundary and voice slot of the CTA,
// ST_NSLOT slots of HS samples.
constexpr int ST_NSLOT = 2;
FDSP_HDC constexpr int st_hand_samples(int outs, bool mix) { return mix && mix_tile_samples(outs) < 16 ? mix_tile_samples(outs) : 16; }
FDSP_HDC constexpr size_t st_ring_floats(int outs, int mid_sum, int nt, bool mix) { return (size_t)ST_NSLOT * mid_sum * st_hand_samples(outs, mix) * nt; }

// Dynamic shared memory of a bank launch of nt voices per CTA: the mix tile (mode bit 1), the hand-off rings when the launch is
// stage-pipelined (mid_sum channels cross its stage boundaries; 0 otherwise), then the wavetables (table_bytes; 0 when the class reads
// none), which are staged (tb) only when all of it fits in the shared memory a block may have.
constexpr size_t SMEM_BLOCK_MAX = 227 * 1024;
struct LaunchSmem { bool tb; size_t smem; };
FDSP_HDC inline LaunchSmem launch_smem(int outs, int nt, int mid_sum, int mode, size_t table_bytes) {
  const bool mix = (mode & 2) != 0;
  const size_t base = (mix ? sizeof(float) * mix_tile_floats(outs, nt) : 0) + sizeof(float) * st_ring_floats(outs, mid_sum, nt, mix);
  const bool tb = table_bytes > 0 && base + table_bytes <= SMEM_BLOCK_MAX;
  return {tb, base + (tb ? table_bytes : 0)};
}

// CTA shape of a class of V voices with NT threads per CTA: enough CTAs to cover the voices, rounded up to whole waves of the
// 148 SMs once every CTA can still have a full warp, and the voices spread evenly over them (a bank is bound by per-SM
// pipes and per-warp latency, so idle SMs are the first thing to use up).
inline uint32_t bank_grid(uint32_t V, uint32_t nt, uint32_t* vpc) {
  uint32_t grid = (V + nt - 1) / nt;
  if (V >= 148u * 32u) grid = (grid + 147u) / 148u * 148u;
  if (grid == 0) grid = 1;
  *vpc = (V + grid - 1) / grid;
  return (V + *vpc - 1) / *vpc;
}

struct BankArgs {
  const uint32_t* params;   // [NP][V]
  uint32_t* state;          // [NS][V]
  const uint32_t* uniform;  // [NU]
  float* dline;             // [sum(len)][V]
  const WaveTableDev* wt;   // [6]
  const float* in;          // shared bank input [IN][in_stride] or null
  float* out;               // per-voice output rows or null
  float* partial;           // [grid][OUT][n] per-CTA mix partials or null
  uint32_t V, n;
  uint32_t vpc;             // voices per CTA (<= threads per CTA): CTA b runs voices [b*vpc, min(V, (b+1)*vpc)); 0 means NT
  uint32_t in_stride, in_offset;
  uint32_t out_stride, out_offset;  // row stride / first sample (multiples of 4 for the vector path)
  const uint32_t* row_map;          // class-local voice -> first output row (voice-major rows) inside `out`
  float sr, sd64, sd32;
  // fused mix-down for short launches (process()-sized): when `ticket` is set, the last CTA to finish folds the per-CTA
  // partials in CTA order into mix[c*mix_stride + mix_offset + t] itself (no mix_reduce_kernel launch)
  uint32_t* ticket;
  float* mix;
  uint32_t mix_stride, mix_offset;
  int mix_accumulate;
  // reset image of the class's state words [NS][V] and delay-line floats per voice: what Event<X> of a looping sequencer needs to reset its unit
  // on the device (null / 0 when the class has no such voices)
  const uint32_t* state0;
  uint32_t dl_floats;
};

}  // namespace fdsp
