// bf16 implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05.mma, accumulators in
// TMEM), operands staged by TMA, fused bias + activation epilogue.  See conv_tc.cuh for the layout.
//
// Replaces Conv2dBlock.forward (reference models/inpaint_networks.py:494-503) in bf16 mode for every
// conv block of the generator, including the fused channel concat (multi-source K blocks), the fused
// nearest x2 upsample (the producer's epilogue writes the 2x2 replicated pixels) and the dual output
// heads (conv17+conv18 / allconv17+allconv18: clamp and sigmoid from one accumulator tile).
//
// Kernel structure (one persistent CTA per SM, 192 threads):
//   warp 0   : TMA producer  - weights once (cp.async.bulk), then per tile one box per (source, ky) band
//   warp 1   : TMEM allocator + single-thread tcgen05.mma issuer; M=128 positions x N=Cout_pad x K=16
//   warps 2-5: epilogue       - tcgen05.ld (one TMEM lane quadrant each) -> bias/act -> bf16 -> global
// Pipelines: smem band ring (full/empty mbarriers, tcgen05.commit frees a slot) and a 2-deep TMEM
// accumulator ring so the epilogue of tile i overlaps the MMAs of tile i+1.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "hv_common.cuh"
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace hv {

// exp(x) for x <= 0 as one MUFU: ex2.approx.ftz without __expf's sub-normal range handling (6 more instructions per element in
// every epilogue warp; the result is rounded to bf16 anyway and exp(x) -> 0 below -87 is exactly what ELU needs)
__device__ __forceinline__ float exp_neg_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}

template <int ACT>
__device__ __forceinline__ float act_fast(float x, int act_rt) {
  if (ACT == HV_ACT_ELU) return x > 0.f ? x : exp_neg_fast(x) - 1.f;
  if (ACT == HV_ACT_RELU) return fmaxf(x, 0.f);
  switch (act_rt) {
    case HV_ACT_ELU: return x > 0.f ? x : __expf(x) - 1.f;
    case HV_ACT_RELU: return fmaxf(x, 0.f);
    case HV_ACT_SIGMOID: return 1.f / (1.f + __expf(-x));
    case HV_ACT_LRELU02: return x > 0.f ? x : 0.2f * x;
    case HV_ACT_CLAMP1: return fminf(fmaxf(x, -1.f), 1.f);
    default: return x;
  }
}

// optional per-CTA event trace (debug / profiling aid, see tools/trace_conv.py): CTA 0 appends (tag, clock) pairs
__device__ __forceinline__ void trace_ev(long long* tr, int& n, int tag) {   // tr is null except on CTA 0 of a traced launch
  if (tr && n < 2000) { tr[2 * n] = tag; tr[2 * n + 1] = clock64(); ++n; }
}


// All MMAs of one segment, fully unrolled for the common (rows, taps, k-steps) shapes: every descriptor is
// `uniform base + small uniform offset`, so ptxas emits back-to-back UTCHMMA fed from uniform registers.
template <int N_PAD, int NROWS, int NTAPS, int KSTEPS>
__device__ __forceinline__ void issue_segment(bool leader, uint32_t d_tmem, uint32_t a_base, uint32_t b_base, uint32_t a_step,
                                              uint32_t b_step, uint32_t b_row_step, uint32_t idesc, uint32_t first_acc) {
  constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
  constexpr uint32_t a_lbo = (uint32_t)NROWS * TC_TILE_M;
  if (leader) {
#pragma unroll
    for (int r = 0; r < NROWS; ++r)
#pragma unroll
      for (int i = 0; i < NTAPS; ++i)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const uint32_t a_lo = a_base + (uint32_t)r * TC_TILE_M + (uint32_t)i * a_step + (uint32_t)ks * 2u * a_lbo;
          const uint32_t b_lo = b_base + (uint32_t)r * b_row_step + (uint32_t)i * b_step + (uint32_t)ks * 2u * N_PAD;
          umma_bf16(d_tmem, ((uint64_t)desc_hi << 32) | a_lo, ((uint64_t)desc_hi << 32) | b_lo, idesc,
                    (r | i | ks) == 0 ? first_acc : 1u);
        }
  }
}

// Stride-2 3x3 conv on a space-to-depth source, all 9 taps from ONE shared-memory image [chunk][sub-plane 4][row 2][128][8]:
// input pixel (2y+ky-1, 2x+kx-1) lives in sub-plane ((ky+1)&1, (kx+1)&1) at (y+dy, x+dx), dy/dx = -1 for ky/kx = 0; row r = dy+1,
// and the band starts one position early so that dx = -1 is offset 0.
template <int N_PAD, int KSTEPS>
__device__ __forceinline__ void issue_s2d(bool leader, uint32_t d_tmem, uint32_t a_base, uint32_t b_base, uint32_t slab, uint32_t idesc) {
  constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
  constexpr uint32_t a_lbo = 8u * TC_TILE_M;  // 4 sub-planes x 2 rows per chunk
  if (leader) {
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const uint32_t sub = (uint32_t)(((ky + 1) & 1) * 2 + ((kx + 1) & 1)), r = ky == 0 ? 0u : 1u, off = kx == 0 ? 0u : 1u;
          const uint32_t a_lo = a_base + (sub * 2u + r) * TC_TILE_M + off + (uint32_t)ks * 2u * a_lbo;
          const uint32_t b_lo = b_base + (uint32_t)(ky * 3 + kx) * slab + (uint32_t)ks * 2u * N_PAD;
          umma_bf16(d_tmem, ((uint64_t)desc_hi << 32) | a_lo, ((uint64_t)desc_hi << 32) | b_lo, idesc, (ky | kx | ks) == 0 ? 0u : 1u);
        }
  }
}

// 3x3 stride-1 conv on an x-phase (xp = 4) source: accumulator row = position (y, x/4), columns = 4 output phases x cp channels.
// Output pixel x = 4q + j, tap kx reads input x + kx - 1 = 4q + d with d = j + kx - 1 in [-1, 4]: six "views" v = d + 1 of the
// shared-memory image [chunk][phase][row][128]: phase = d mod 4, position shift = floor(d / 4) (+1: the band starts one early).
// The weights of view v hold w[.][.][ky][kx = v - j] in the columns of phase j and zeros elsewhere.
template <int N_PAD, int NROWS, int KSTEPS>
__device__ __forceinline__ void issue_xp4(bool leader, uint32_t d_tmem, uint32_t a_base, uint32_t b_base, uint32_t slab, uint32_t idesc,
                                          uint32_t first_acc) {
  constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
  constexpr uint32_t a_lbo = 4u * NROWS * TC_TILE_M;
  if (leader) {
#pragma unroll
    for (int r = 0; r < NROWS; ++r)
#pragma unroll
      for (int v = 0; v < 6; ++v)
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const uint32_t phase = (uint32_t)((v + 3) & 3), shift = v == 0 ? 0u : (v == 5 ? 2u : 1u);
          const uint32_t a_lo = a_base + (phase * NROWS + (uint32_t)r) * TC_TILE_M + shift + (uint32_t)ks * 2u * a_lbo;
          const uint32_t b_lo = b_base + (uint32_t)(r * 6 + v) * slab + (uint32_t)ks * 2u * N_PAD;
          umma_bf16(d_tmem, ((uint64_t)desc_hi << 32) | a_lo, ((uint64_t)desc_hi << 32) | b_lo, idesc, (r | v | ks) == 0 ? first_acc : 1u);
        }
  }
}

// generic (slow) fallback for shapes without an unrolled instance
template <int N_PAD>
__device__ __forceinline__ void issue_segment_generic(bool leader, uint32_t d_tmem, uint32_t a_base, uint32_t b_base, uint32_t a_step,
                                                      uint32_t b_step, uint32_t b_row_step, uint32_t idesc, uint32_t first_acc,
                                                      int nrows, int ntaps, int ksteps) {
  constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
  const uint32_t a_lbo = (uint32_t)nrows * TC_TILE_M;
  uint32_t accumulate = first_acc;
  for (int r = 0; r < nrows; ++r)
    for (int i = 0; i < ntaps; ++i)
      for (int ks = 0; ks < ksteps; ++ks) {
        const uint32_t a_lo = a_base + (uint32_t)r * TC_TILE_M + (uint32_t)i * a_step + (uint32_t)ks * 2u * a_lbo;
        const uint32_t b_lo = b_base + (uint32_t)r * b_row_step + (uint32_t)i * b_step + (uint32_t)ks * 2u * N_PAD;
        if (leader) umma_bf16(d_tmem, ((uint64_t)desc_hi << 32) | a_lo, ((uint64_t)desc_hi << 32) | b_lo, idesc, accumulate);
        accumulate = 1;
      }
}

constexpr int TC_TMEM_COLS = 256;
constexpr int TC_BAR_BYTES = 1024;  // mbarriers + TMEM slot (512 B) + bias vector (512 B)
// 16 epilogue warps, 16 accumulator columns each: N_PAD/16*4 warps cover one tile (4 TMEM lane quadrants x column groups), so
// 16/that many tiles are in the epilogue concurrently (4 / 2 / 1 for N_PAD = 16 / 32 / 64); group g owns tiles j % groups == g
__host__ __device__ constexpr int tc_epi_warps(int) { return 16; }
__host__ __device__ constexpr int tc_warps_per_tile(int n_pad) { return n_pad >= 64 ? 16 : n_pad / 16 * 4; }
__host__ __device__ constexpr int tc_threads(int n_pad) { return 64 + 32 * tc_epi_warps(n_pad); }
__host__ __device__ constexpr int tc_acc_stages(int n_pad) { return TC_TMEM_COLS / n_pad > 8 ? 8 : TC_TMEM_COLS / n_pad; }
// thin layers (N_PAD <= 32) are bound by the single-lane issue / handshake latencies, not by the tensor pipe: two CTAs per SM
// (2 x 256 TMEM columns, <= 56 registers per thread) interleave their MMA streams
__host__ __device__ constexpr int tc_ctas_per_sm(int n_pad) { return n_pad <= 32 ? 2 : 1; }

// ------------------------------------------------------------------------------------------- kernel
// warps 0..15: epilogue, warp 16: TMA producer, warp 17: TMEM allocator + MMA issuer.  The single-lane roles sit on the
// HIGHEST warp ids on purpose: the SM's warp arbiter favours high warp ids, and an issuer starved by busy epilogue warps
// stalls the tensor pipe.
// FIXED = 0: the issuer picks its unrolled MMA sequence at run time (any layer geometry).  FIXED != 0: the sequence is a compile-time
// constant, which removes the shape switch and every other unrolled sequence from the instruction stream: measured on B200, the
// 64->64 trunk layers run 9 % faster (12.7 -> 11.6 us per launch) for the smaller instruction footprint alone.
//   FIXED = kind << 12 | rows << 8 | taps << 4 | k-steps;  kind 1: plain segments of one shape, 2: space-to-depth (k-steps),
//   3: x-phase (rows, k-steps), 4: two sources, segment 0 = (3 rows, 3 taps, k-steps), segment 1 = kx-packed plane (3, 1, 1)
__host__ __device__ constexpr int tc_shape_code(int kind, int rows, int taps, int ksteps) { return kind << 12 | rows << 8 | taps << 4 | ksteps; }
// DIAG: the diagnostics (per-role clock trace, launch timeline stamps) are compiled in only for the
// instances that the host picks while a diagnostic is active: in the production instances they cost 2.4 % of the forward (the
// single-thread loops pay for every extra instruction).
template <int N_PAD, int ACT, int FIXED = 0, bool DIAG = true>
__global__ void __launch_bounds__(tc_threads(N_PAD), tc_ctas_per_sm(N_PAD)) conv_tc_kernel(const __grid_constant__ TcParams p) {
  constexpr int ACC_STAGES = tc_acc_stages(N_PAD);       // accumulator tiles in flight
  constexpr int EPI_WARPS = tc_epi_warps(N_PAD);
  constexpr int WPT = tc_warps_per_tile(N_PAD), GROUPS = EPI_WARPS / WPT;
  constexpr int NCOL = N_PAD > 64 ? N_PAD / 4 : 16;      // accumulator columns per epilogue warp (16 warps = 4 lane quadrants x 4 slices)
  constexpr int W_PRODUCER = EPI_WARPS, W_MMA = EPI_WARPS + 1;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // output mode / layouts: compile-time constants in the specialised instances (bits 16.. of FIXED: 1 chunked, 2 chunked + x2
  // upsample, 3 heads, 4 space-to-depth, 5 chunked into an x-phase buffer, 6 upsample into an x-phase buffer), else kernel parameters
  constexpr int FO = (FIXED >> 16) & 15;
  // PAIR (bit 20): a round of the producer / issuer / barrier protocol covers TWO consecutive tiles (two bands per slot, two
  // accumulators per stage): the thin layers are bound by the latency of the single-thread handshake chain per round, not by MMAs
  constexpr bool PAIR = ((FIXED >> 20) & 1) != 0;
  constexpr int TPR = PAIR ? 2 : 1;                      // tiles per round
  constexpr int RSTAGES = ACC_STAGES / TPR;              // accumulator barrier stages
  const int k_in_xp = FIXED != 0 ? ((FIXED >> 12 & 15) == 3 ? 4 : 1) : p.in_xp;
  const int k_out_mode = FO == 0 ? p.out_mode : (FO == 1 || FO == 5) ? (int)TC_OUT_CHUNKED : (FO == 2 || FO == 6) ? (int)TC_OUT_CHUNKED_UP2
                                              : FO == 3 ? (int)TC_OUT_HEADS : (int)TC_OUT_CHUNKED_S2D;
  const int k_out_xp = FO == 0 ? p.out_xp : (FO == 5 || FO == 6) ? 4 : FO == 3 ? k_in_xp : 1;
  const uint32_t w_region = (p.w_bytes + 127u) & ~127u;
  uint8_t* s_slots = smem + w_region;
  // 1 KB pad after the band ring: the last chunk of a shifted tap view reads past its band
  const uint32_t slot_stride = p.slot_bytes * TPR;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_slots + (size_t)p.nslots * slot_stride + 1024);
  const uint32_t bar_full = smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8u * p.nslots;
  const uint32_t bar_w = bar_empty + 8u * p.nslots;
  const uint32_t bar_tfull = bar_w + 8u;
  const uint32_t bar_tempty = bar_tfull + 8u * ACC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.nslots + 1 + 2 * ACC_STAGES);
  float* s_bias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);

  if (DIAG && p.trace && threadIdx.x == 0 && blockIdx.x < 400) {   // CTA entry: wall clock (ns) and SM clock
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[12000 + 4 * blockIdx.x] = (long long)gt;
    p.trace[12000 + 4 * blockIdx.x + 2] = clock64();
  }
  if (DIAG && p.timeline && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    atomicMin(reinterpret_cast<unsigned long long*>(p.timeline), gt);
  }
  if (warp == W_PRODUCER && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.maps[0]) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.maps[1]) : "memory");
  }
  if (warp == W_MMA) {
    if (lane == 0) {
      for (int i = 0; i < p.nslots; ++i) { mbar_init(bar_full + 8u * i, 1); mbar_init(bar_empty + 8u * i, 1); }
      mbar_init(bar_w, 1);
      for (int i = 0; i < ACC_STAGES; ++i) { mbar_init(bar_tfull + 8u * i, 1); mbar_init(bar_tempty + 8u * i, 32 * WPT * TPR); }
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TC_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x < N_PAD) s_bias[threadIdx.x] = __ldg(p.bias + threadIdx.x);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // PDL: let the next kernel of the stream start its own prologue as soon as SM resources free up ...
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == W_PRODUCER) {
    // ===================================================================== TMA producer (warp-uniform, one lane issues)
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(bar_w, p.w_bytes);
      bulk_load(smem_u32(smem), p.w_packed, p.w_bytes, bar_w);
    }
    // ... and do not read the previous kernel's output (the activation bands) before it has completed and flushed
    asm volatile("griddepcontrol.wait;" ::: "memory");
    int slot = 0, ntr = 0;
    uint32_t phase = 0;
    long long* tr = (DIAG && p.trace && blockIdx.x == 0) ? p.trace : nullptr;
    const unsigned long long tiles_magic = p.tiles_magic;
    const int tiles_per_image = p.tiles_per_image, tile_adv = p.tile_adv, q_first = p.q_first, total_tiles = p.total_tiles;
    const uint32_t slots_base = smem_u32(s_slots);
    const int nseg = p.nseg, nslots = p.nslots;
    const bool map5d = p.map5d != 0;
    const uint32_t slot_bytes = p.slot_bytes;
    int rel2 = p.segs[0].rel_start2, c1 = p.segs[0].c1;   // single-segment layers keep the load recipe in registers
    uint32_t tx = p.segs[0].tx_bytes;
    bool map1 = false;
    const int rounds = (total_tiles + TPR - 1) / TPR;
    for (int round = blockIdx.x; round < rounds; round += gridDim.x) {
      const int tile = round * TPR;
      const int img = (int)(((unsigned long long)tile * tiles_magic) >> 40);
      const int c_tile = 2 * ((tile - img * tiles_per_image) * tile_adv + q_first);  // tensor-map inner unit = 8 B
      // second tile of a pair (the last round of an odd tile count repeats its first tile: same values stored twice)
      const int tile_b = min(tile + 1, total_tiles - 1);
      const int img_b = (int)(((unsigned long long)tile_b * tiles_magic) >> 40);
      const int c_tile_b = 2 * ((tile_b - img_b * tiles_per_image) * tile_adv + q_first);
      for (int s = 0; s < nseg; ++s) {
        if (nseg > 1) {
          rel2 = p.segs[s].rel_start2; c1 = p.segs[s].c1; tx = p.segs[s].tx_bytes; map1 = p.segs[s].map != 0;
        }
        mbar_wait(bar_empty + 8u * slot, phase ^ 1u);
        if (leader) {
          const uint32_t fb = bar_full + 8u * slot, dst = slots_base + (uint32_t)slot * slot_stride;
          mbar_expect_tx(fb, tx * TPR);
          // one operation per band: the box spans all chunks of the segment
          if (map5d) tma_load_5d(dst, &p.maps[0], fb, c_tile + rel2, c1, 0, 0, img);   // {positions, rows, 4 sub-planes / phases, chunks, image}
          else tma_load_4d(dst, map1 ? &p.maps[1] : &p.maps[0], fb, c_tile + rel2, c1, 0, img);
          if (PAIR) {
            if (map5d) tma_load_5d(dst + slot_bytes, &p.maps[0], fb, c_tile_b + rel2, c1, 0, 0, img_b);
            else tma_load_4d(dst + slot_bytes, map1 ? &p.maps[1] : &p.maps[0], fb, c_tile_b + rel2, c1, 0, img_b);
          }
          trace_ev(tr, ntr, 1);
        }
        if (++slot == nslots) { slot = 0; phase ^= 1u; }
      }
    }
  } else if (warp == W_MMA) {
    // ===================================================================== MMA issuer (warp-uniform, one lane issues)
    const bool leader = elect_one();
    // instruction descriptor: D=f32, A=B=bf16, both K-major, N = N_PAD, M = 128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N_PAD >> 3) << 17) | ((128u >> 4) << 24);
    // smem descriptor = hi word (SBO = 128 B, version 1) : lo word (start >> 4 | LBO >> 4 << 16); offsets add into lo.
    // A: K chunks of a segment are nrows * 128 positions apart; B: [chunk][N_PAD][8] -> N_PAD * 16 B apart
    constexpr uint32_t b_lo_const = (uint32_t)N_PAD << 16;
    mbar_wait(bar_w, 0);
    tc_fence_after();
    const uint32_t b_lo_base = b_lo_const + (smem_u32(smem) >> 4);
    const uint32_t a_lo_base = smem_u32(s_slots) >> 4;
    const uint32_t slot_units = p.slot_bytes >> 4;
    int slot = 0, acc = 0, ntr = 0;
    long long* tr = (DIAG && p.trace && blockIdx.x == 0) ? p.trace + 4000 : nullptr;
    uint32_t phase = 0, acc_phase = 0;
    // peek-ahead: the next barrier is probed BEFORE the current batch of MMAs is issued, so the probe latency
    // hides under the queued MMAs (the tensor pipe accepts only a few MMAs ahead of execution)
    bool ready_full = mbar_peek(bar_full, 0), ready_acc = mbar_peek(bar_tempty, 1);
    const int nseg = p.nseg, nslots = p.nslots, total_tiles = p.total_tiles;
    constexpr int FK = (FIXED >> 12) & 15, FR = (FIXED >> 8) & 15, FT = (FIXED >> 4) & 15, FS = FIXED & 15;
    const bool s2d = FIXED == 0 && p.s2d_in != 0, xp_in = FIXED == 0 && p.in_xp > 1;
    TcSeg sg = p.segs[0];
    const int rounds = (total_tiles + TPR - 1) / TPR;
    const uint32_t stride_units = slot_units * TPR;
    for (int round = blockIdx.x; round < rounds; round += gridDim.x) {
      mbar_wait_peeked(ready_acc, bar_tempty + 8u * acc, acc_phase ^ 1u);
      tc_fence_after();
      if (leader) trace_ev(tr, ntr, 11);
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * TPR * N_PAD);
      const uint32_t cur_tfull = bar_tfull + 8u * acc;
      if (++acc == RSTAGES) { acc = 0; acc_phase ^= 1u; }
      uint32_t accumulate = 0;
      for (int s = 0; s < nseg; ++s) {
        if (nseg > 1) sg = p.segs[s];  // single-segment layers keep the descriptor recipe in registers
        const int nrows = sg.nrows, ntaps = sg.ntaps, ksteps = sg.nchunks >> 1;
        const uint32_t a_lbo = (uint32_t)nrows * TC_TILE_M;  // 16 B units: K chunks of the segment image are nrows bands apart
        const uint32_t a_step = sg.a_step, b_step = sg.b_step, b_row_step = sg.b_row_step;
        mbar_wait_peeked(ready_full, bar_full + 8u * slot, phase);
        tc_fence_after();
        if (leader) trace_ev(tr, ntr, 12);
        const uint32_t cur_slot = (uint32_t)slot, cur_empty = bar_empty + 8u * slot;
        if (++slot == nslots) { slot = 0; phase ^= 1u; }
        ready_full = mbar_peek(bar_full + 8u * slot, phase);
        const uint32_t a_slot = a_lo_base + cur_slot * stride_units;
        const uint32_t a_row = a_slot + (a_lbo << 16) + sg.a0;
        const uint32_t b_row = b_lo_base + sg.b0;
        if (s == nseg - 1) ready_acc = mbar_peek(bar_tempty + 8u * acc, acc_phase ^ 1u);
        if (FIXED != 0) {
#pragma unroll
          for (int u = 0; u < TPR; ++u) {   // the tiles of the round: band u of the slot -> accumulator u of the stage
            const uint32_t dt = d_tmem + (uint32_t)(u * N_PAD), au = (uint32_t)u * slot_units;
            if (FK == 1) {
              issue_segment<N_PAD, FR ? FR : 1, FT ? FT : 1, FS ? FS : 1>(leader, dt, a_row + au, b_row, a_step, b_step, b_row_step, idesc, accumulate);
            } else if (FK == 2) {
              issue_s2d<N_PAD, FS ? FS : 1>(leader, dt, a_slot + au + ((8u * TC_TILE_M) << 16), b_row, b_step, idesc);
            } else if (FK == 3) {
              issue_xp4<N_PAD, FR ? FR : 1, FS ? FS : 1>(leader, dt, a_slot + au + ((4u * (uint32_t)(FR ? FR : 1) * TC_TILE_M) << 16), b_row, b_step, idesc,
                                                       accumulate);
            } else {
              if (s == 0) issue_segment<N_PAD, 3, 3, FS ? FS : 1>(leader, dt, a_row + au, b_row, a_step, b_step, b_row_step, idesc, accumulate);
              else issue_segment<N_PAD, 3, 1, 1>(leader, dt, a_row + au, b_row, a_step, b_step, b_row_step, idesc, accumulate);
            }
          }
          accumulate = 1;
          if (leader) { umma_commit(cur_empty); trace_ev(tr, ntr, 13); }
          continue;
        }
        if (s2d) {
          const uint32_t a_s2d = a_slot + ((8u * TC_TILE_M) << 16);
          if (ksteps == 1) issue_s2d<N_PAD, 1>(leader, d_tmem, a_s2d, b_row, b_step, idesc);
          else if (ksteps == 2) issue_s2d<N_PAD, 2>(leader, d_tmem, a_s2d, b_row, b_step, idesc);
          else issue_s2d<N_PAD, 4>(leader, d_tmem, a_s2d, b_row, b_step, idesc);
          accumulate = 1;
          if (leader) { umma_commit(cur_empty); trace_ev(tr, ntr, 13); }
          continue;
        }
        if (xp_in) {
          const uint32_t a_xp = a_slot + ((4u * (uint32_t)nrows * TC_TILE_M) << 16);
          const int shape_xp = (nrows << 4) | ksteps;
          switch (shape_xp) {
            case (3 << 4) | 1: issue_xp4<N_PAD, 3, 1>(leader, d_tmem, a_xp, b_row, b_step, idesc, accumulate); break;
            case (3 << 4) | 2: issue_xp4<N_PAD, 3, 2>(leader, d_tmem, a_xp, b_row, b_step, idesc, accumulate); break;
            case (1 << 4) | 1: issue_xp4<N_PAD, 1, 1>(leader, d_tmem, a_xp, b_row, b_step, idesc, accumulate); break;
            default: issue_xp4<N_PAD, 1, 2>(leader, d_tmem, a_xp, b_row, b_step, idesc, accumulate); break;
          }
          accumulate = 1;
          if (leader) { umma_commit(cur_empty); trace_ev(tr, ntr, 13); }
          continue;
        }
        const int shape = (nrows << 8) | (ntaps << 4) | ksteps;
#define HV_SEG(R, T, K)                                                                                                   \
  case ((R) << 8) | ((T) << 4) | (K):                                                                                     \
    issue_segment<N_PAD, R, T, K>(leader, d_tmem, a_row, b_row, a_step, b_step, b_row_step, idesc, accumulate);           \
    break;
        switch (shape) {
          HV_SEG(3, 3, 1) HV_SEG(3, 3, 2) HV_SEG(3, 3, 4) HV_SEG(5, 5, 1) HV_SEG(5, 5, 2)
          HV_SEG(1, 3, 1) HV_SEG(1, 3, 2) HV_SEG(1, 3, 4) HV_SEG(1, 2, 1) HV_SEG(1, 2, 2) HV_SEG(1, 1, 1) HV_SEG(1, 1, 2)
          HV_SEG(5, 1, 1) HV_SEG(5, 1, 2) HV_SEG(1, 5, 1) HV_SEG(3, 1, 1) HV_SEG(1, 1, 4)
          default:
            issue_segment_generic<N_PAD>(leader, d_tmem, a_row, b_row, a_step, b_step, b_row_step, idesc, accumulate, nrows, ntaps, ksteps);
        }
#undef HV_SEG
        accumulate = 1;
        if (leader) { umma_commit(cur_empty); trace_ev(tr, ntr, 13); }  // slot is free once these MMAs have read it
      }
      if (leader) umma_commit(cur_tfull);  // accumulator tile complete -> epilogue
    }
    __syncwarp();
  } else {
    // ===================================================================== epilogue (warps 0 .. 15)
    // group g owns the CTA's tiles j = g, g + GROUPS, ...; inside a group a warp reads TMEM lane quadrant warp % 4 and one
    // 16-column slice.  With GROUPS tiles in flight the per-tile latency (tcgen05.ld -> math -> stores) is off the critical path.
    const int quad = warp & 3;               // TMEM lane quadrant this warp may access
    const int group = warp / WPT;
    const int col0 = ((warp % WPT) >> 2) * NCOL;
    int ntr = 0;
    long long* tr = (DIAG && p.trace && blockIdx.x == 0 && warp == 0 && lane == 0) ? p.trace + 8000 : nullptr;
    const unsigned long long tiles_magic = p.tiles_magic;
    const int m = quad * 32 + lane;
    const int total_tiles = p.total_tiles, rounds = (total_tiles + TPR - 1) / TPR;
    // the CTA's tiles in processing order: q = TPR * (round index of this CTA) + (tile of the round); group g owns q % GROUPS == g
    for (int q_lin = group; ; q_lin += GROUPS) {
      const int j = q_lin / TPR, u = q_lin - j * TPR;
      const int round = blockIdx.x + j * (int)gridDim.x;
      if (round >= rounds) break;
      const int tile = min(round * TPR + u, total_tiles - 1);
      const int acc = j % RSTAGES;
      const uint32_t acc_phase = (uint32_t)(j / RSTAGES) & 1u;
      const int img = (int)(((unsigned long long)tile * tiles_magic) >> 40);
      const int q = (tile - img * p.tiles_per_image) * p.tile_adv + m + p.q_first;
      const int qrow = (int)(((unsigned long long)q * p.pitch_magic) >> 40);
      const int yy = qrow - p.in_border;
      const int xx = q - qrow * p.in_pitch - p.in_border;
      // rows >= tile_adv read past the band (their taps shift beyond position 127): garbage, skipped
      const bool valid = m < p.tile_adv && yy >= 0 && yy < p.h_out && xx >= 0 && xx < p.w_out;
      trace_ev(tr, ntr, 20);
      mbar_wait(bar_tfull + 8u * acc, acc_phase);
      tc_fence_after();
      trace_ev(tr, ntr, 21);
      const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)((acc * TPR + u) * N_PAD);

      // position of output pixel (y, x) inside one chunk plane of the output buffer (plain / space-to-depth / x-phase)
      auto out_pos = [&](int y, int x) -> size_t {
        if (k_out_mode == TC_OUT_CHUNKED_S2D)
          return (size_t)((y & 1) * 2 + (x & 1)) * p.out_sub_plane + (size_t)((y >> 1) + p.out_border) * p.out_pitch + (x >> 1) + p.out_border;
        if (k_out_xp > 1)
          return (size_t)(x & (k_out_xp - 1)) * p.out_sub_plane + (size_t)(y + p.out_border) * p.out_pitch + x / k_out_xp + p.out_border;
        return (size_t)(y + p.out_border) * p.out_pitch + x + p.out_border;
      };
      auto aux_store = [&](const TcAux& a, int y, int x, float val) {   // one bf16 channel of an (x-phase or plain) chunked buffer
        const size_t pos = k_out_xp > 1 ? (size_t)(x & (k_out_xp - 1)) * a.sub_plane + (size_t)(y + a.border) * a.pitch + x / k_out_xp + a.border
                                        : (size_t)(y + a.border) * a.pitch + x + a.border;
        a.ptr[(((size_t)img * a.chunks + a.chunk) * a.plane + pos) * 8 + a.channel] = __float2bfloat16(val);
      };

      if (k_out_mode == TC_OUT_HEADS) {
        float v[NCOL];
        if (col0 == 0) { tmem_ld<NCOL>(t_addr, v); tmem_ld_wait(); }
        tc_fence_before();
        mbar_arrive(bar_tempty + 8u * acc);
        if (!valid || col0 != 0) continue;
        const int npix = k_in_xp > 1 ? k_in_xp : 1;   // x-phase source: columns j * cp + {0, 1} = heads of pixel 4 xx + j
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) {
          if (jx >= npix) break;
          const int x = k_in_xp > 1 ? xx * k_in_xp + jx : xx;
          const float a0 = fminf(fmaxf(v[jx * 4] + s_bias[jx * 4], -1.f), 1.f);
          const float a1 = 1.f / (1.f + __expf(-(v[jx * 4 + 1] + s_bias[jx * 4 + 1])));
          const size_t pix = ((size_t)img * p.h_out + yy) * p.w_img + x;
          p.head0[pix] = a0;
          p.head1[pix] = a1;
          if (p.aux0.ptr) aux_store(p.aux0, yy, x, a0);
          if (p.aux1.ptr) aux_store(p.aux1, yy, x, a1);
        }
        continue;
      }
      float v[NCOL];
      tmem_ld<NCOL>(t_addr + col0, v);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bar_tempty + 8u * acc);  // this warp's slice is in registers: release its share of the TMEM stage
      if (!valid) continue;
      __nv_bfloat16* out_img = p.out + ((size_t)img * p.out_chunks_total + p.out_chunk_off) * p.out_plane * 8;
#pragma unroll
      for (int jj = 0; jj < NCOL / 8; ++jj) {
        const int col = col0 + jj * 8;
        // plain source: column = channel.  x-phase source: column = phase * cp + channel of output pixel in_xp * xx + phase.
        // sub-pixel upsample (p.ups): the source is the LOW-resolution map of a nearest-x2-upsampled input; column = parity * cp +
        // channel of output pixel (2 yy + parity / 2, 2 xx + parity % 2)
        const int ph = (k_in_xp > 1 || p.ups) ? col / p.cp : 0;
        const int c = ((k_in_xp > 1 || p.ups) ? col - ph * p.cp : col) >> 3;
        if (c >= p.out_nchunks) continue;
        const int x = p.ups ? 2 * xx + (ph & 1) : (k_in_xp > 1 ? xx * k_in_xp + ph : xx);
        const int yo = p.ups ? 2 * yy + (ph >> 1) : yy;
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float f0 = act_fast<ACT>(v[jj * 8 + 2 * e] + s_bias[col + 2 * e], p.act);
          const float f1 = act_fast<ACT>(v[jj * 8 + 2 * e + 1] + s_bias[col + 2 * e + 1], p.act);
          __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
          pk[e] = *reinterpret_cast<uint32_t*>(&h);
        }
        const uint4 val = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        __nv_bfloat16* plane = out_img + (size_t)c * p.out_plane * 8;
        if (k_out_mode == TC_OUT_CHUNKED_UP2) {  // nearest x2 upsample fused into the store (inpaint_networks.py:97,:105,:219,:222)
          *reinterpret_cast<uint4*>(plane + out_pos(2 * yy, 2 * x) * 8) = val;
          *reinterpret_cast<uint4*>(plane + out_pos(2 * yy, 2 * x + 1) * 8) = val;
          *reinterpret_cast<uint4*>(plane + out_pos(2 * yy + 1, 2 * x) * 8) = val;
          *reinterpret_cast<uint4*>(plane + out_pos(2 * yy + 1, 2 * x + 1) * 8) = val;
        } else {
          *reinterpret_cast<uint4*>(plane + out_pos(yo, x) * 8) = val;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (DIAG && p.trace && threadIdx.x == 0 && blockIdx.x < 400) {   // CTA exit
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[12000 + 4 * blockIdx.x + 1] = (long long)gt;
    p.trace[12000 + 4 * blockIdx.x + 3] = clock64();
  }
  if (DIAG && p.timeline && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    atomicMax(reinterpret_cast<unsigned long long*>(p.timeline) + 1, gt);
  }
  if (warp == W_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- host: tensor maps
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

// Tensor map over one chunked buffer.  The inner dimension is the contiguous run of positions of one
// chunk, described in 8-byte units (two per position) so that one 128-position band is a single
// 2 KB box row (box rows of 16 B make TMA ~20x slower and fetch half-empty sectors).
//   stride-1 sources : dims {positions*2, k rows, chunks, n}, dim 1 steps `dil` image rows, so ONE box of `box_rows`
//                      rows brings the bands of `box_rows` kernel rows (the dims overlap in memory; TMA does not mind)
//   s2d sources      : dims {sub-plane positions*2, 4 sub-planes, chunks, n}, box_rows = 1
static int make_map(CUtensorMap* map, const TcBuf& b, int k, int dil, int box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable (driver entry point lookup failed)"); return HV_ERR_CUDA; }
  const cuuint64_t plane_b = (cuuint64_t)b.plane() * 16, sub_b = (cuuint64_t)b.sub_plane() * 16;
  CUresult r = CUDA_SUCCESS;
  const CUtensorMapDataType types[2] = {CU_TENSOR_MAP_DATA_TYPE_UINT64, CU_TENSOR_MAP_DATA_TYPE_FLOAT64};
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (!b.s2d && b.xp == 1) {
      cuuint64_t dims[4] = {(cuuint64_t)b.sub_plane() * 2, (cuuint64_t)k, (cuuint64_t)b.chunks, (cuuint64_t)b.n};
      cuuint64_t strides[3] = {(cuuint64_t)dil * b.pitch() * 16, plane_b, plane_b * b.image_chunks()};
      cuuint32_t box[4] = {2 * TC_TILE_M, (cuuint32_t)box_rows, (cuuint32_t)b.chunks, 1};
      cuuint32_t es[4] = {1, 1, 1, 1};
      r = enc(map, types[attempt], 4, b.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else if (b.xp > 1) {
      // x-phase source: {positions*2, k rows, xp phases, chunks, n}; one box = `box_rows` kernel rows of all phases
      cuuint64_t dims[5] = {(cuuint64_t)b.sub_plane() * 2, (cuuint64_t)k, (cuuint64_t)b.xp, (cuuint64_t)b.chunks, (cuuint64_t)b.n};
      cuuint64_t strides[4] = {(cuuint64_t)dil * b.pitch() * 16, sub_b, plane_b, plane_b * b.image_chunks()};
      cuuint32_t box[5] = {2 * TC_TILE_M, (cuuint32_t)box_rows, (cuuint32_t)b.xp, (cuuint32_t)b.chunks, 1};
      cuuint32_t es[5] = {1, 1, 1, 1, 1};
      r = enc(map, types[attempt], 5, b.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
      // space-to-depth source: {positions*2, 2 rows (dy = -1, 0), 4 parity sub-planes, chunks, n}: one box = everything a tile needs
      cuuint64_t dims[5] = {(cuuint64_t)b.sub_plane() * 2, 2, 4, (cuuint64_t)b.chunks, (cuuint64_t)b.n};
      cuuint64_t strides[4] = {(cuuint64_t)b.pitch() * 16, sub_b, plane_b, plane_b * b.image_chunks()};
      cuuint32_t box[5] = {2 * TC_TILE_M, 2, 4, (cuuint32_t)b.chunks, 1};
      cuuint32_t es[5] = {1, 1, 1, 1, 1};
      r = enc(map, types[attempt], 5, b.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r == CUDA_SUCCESS) return HV_OK;
  }
  set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return HV_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------- host: setup
static int max_chunks_of(const TcSource* srcs, int nsrc) {
  int m = 0;
  for (int i = 0; i < nsrc; ++i) m = max(m, srcs[i].buf.chunks);
  return m;
}

static int tc_issue_code(const TcConv& c);

int tc_conv_setup(TcConv& c, const TcSource* srcs, int nsrc, int k, int stride, int dil, int cout_real, int n_images, bool allow_pair, bool ups) {
  HV_CHECK_ARG(nsrc >= 1 && nsrc <= 2, "tc_conv: 1 or 2 sources supported");
  HV_CHECK_ARG((k == 3 || k == 5) && (stride == 1 || (stride == 2 && k == 3 && dil == 1)), "tc_conv: unsupported k/stride");
  memset(&c.p, 0, sizeof(c.p));
  c.k = k; c.stride = stride; c.dil = dil; c.nsrc = nsrc; c.cout_real = cout_real;
  for (int i = 0; i < nsrc; ++i) c.src[i] = srcs[i];
  HV_CHECK_ARG(cout_real >= 1 && cout_real <= 64, "tc_conv: cout must be in 1..64");
  const TcBuf& b0 = srcs[0].buf;
  const int xp = b0.xp;
  int cp = 0;   // accumulator columns per output pixel of an x-phase layer
  if (xp > 1) {
    HV_CHECK_ARG(xp == 4 && nsrc == 1 && stride == 1 && k == 3 && dil == 1 && !srcs[0].kxpack && cout_real <= 16 && (b0.w % 4) == 0,
                 "tc_conv: x-phase sources feed single-source 3x3 stride-1 convs with <= 16 filters");
    cp = cout_real <= 4 ? 4 : (cout_real <= 8 ? 8 : 16);
    c.n_pad = 4 * cp;
  } else if (ups) {
    HV_CHECK_ARG(stride == 1 && k == 3 && dil == 1 && !srcs[0].kxpack && cout_real <= 32 && (nsrc == 1 || srcs[1].nbhd4) && srcs[0].buf.xp == 1,
                 "tc_conv: the sub-pixel upsample mode serves 3x3 stride-1 convs with <= 32 filters (second source: a 4x4-neighbourhood plane)");
    cp = cout_real <= 8 ? 8 : (cout_real <= 16 ? 16 : 32);
    c.n_pad = 4 * cp;
  } else {
    c.n_pad = cout_real <= 16 ? 16 : (cout_real <= 32 ? 32 : 64);
  }
  const int half = (k - 1) / 2;
  int max_chunks = 0, total_chunks = 0;
  for (int i = 0; i < nsrc; ++i) {
    const TcBuf& b = srcs[i].buf;
    HV_CHECK_ARG(b.ptr && (b.chunks % 2) == 0, "tc_conv: source %d needs an even number of channel chunks", i);
    HV_CHECK_ARG(b.h == b0.h && b.w == b0.w && b.border == b0.border && b.n == b0.n && b.s2d == b0.s2d && b.xp == b0.xp,
                 "tc_conv: concat sources must share geometry");
    HV_CHECK_ARG(b.s2d == (stride == 2), "tc_conv: a stride-2 conv reads a space-to-depth buffer (and only it does)");
    HV_CHECK_ARG(b.border >= (stride == 2 ? 1 : half * dil), "tc_conv: source border %d smaller than the conv padding", b.border);
    HV_CHECK_ARG(srcs[i].real_channels * (srcs[i].kxpack ? k : 1) <= b.chunks * 8, "tc_conv: real_channels > buffer channels");
    HV_CHECK_ARG(!srcs[i].kxpack || stride == 1, "tc_conv: kx-packed sources feed stride-1 convs only");
    max_chunks = max(max_chunks, b.chunks);
    total_chunks += b.chunks;
  }
  HV_CHECK_ARG(b0.n == n_images, "tc_conv: batch mismatch");
  HV_CHECK_ARG(stride == 1 || nsrc == 1, "tc_conv: stride-2 layers take a single source");
  TcParams& p = c.p;
  const int pitch = b0.pitch();
  HV_CHECK_ARG((long long)b0.plane() < (1ll << 20), "tc_conv: plane too large for the fast row division");
  p.s2d_in = stride == 2;
  p.in_xp = xp; p.cp = cp; p.map5d = (stride == 2 || xp > 1) ? 1 : 0;
  p.ups = ups ? 1 : 0;
  p.w_img = b0.w;
  p.in_pitch = pitch; p.in_border = b0.border;
  p.pitch_magic = ((1ull << 40) + (unsigned long long)pitch - 1) / (unsigned long long)pitch;
  p.h_out = b0.sub_h(); p.w_out = b0.sub_w();
  p.q_first = b0.border * pitch + b0.border;
  p.w_bytes = 0;
  for (int i = 0; i < nsrc; ++i) p.w_bytes += (uint32_t)((xp > 1 ? k * (xp + 2) : (srcs[i].kxpack ? k : k * k)) * srcs[i].buf.chunks * c.n_pad * 16);
  size_t budget = 227 * 1024 - 2048;
  const size_t fixed = ((p.w_bytes + 127u) & ~127u) + 1024 /* over-read pad */ + TC_BAR_BYTES;
  c.ctas_per_sm = 1;
  // Tile pairs (see PAIR in the kernel) for a thin, long layer that cannot run as two co-resident CTAs (its three band slots do not
  // fit in half the shared memory): at least ~6 rounds per SM and two pair slots beside the weights.  Measured per layer on B200:
  // pairs help exactly there (merged fine conv1|pmconv1: 45.0 -> 40.5 us); where two CTAs per SM are possible they are the better
  // latency hiding (pairs: conv3 +4 us, heads +8 us), and the x-phase layers lose too (conv16 +3 us).
  bool want_pair = false;
  {
    const long long est_tiles = ((long long)b0.sub_h() * pitch / (TC_TILE_M - 2) + 1) * n_images;
    const size_t half = (227 * 1024) / 2 - 2048, band = (size_t)TC_TILE_M * max_chunks_of(srcs, nsrc) * 16u * (stride == 2 ? 8 : k * xp);
    const bool two_ctas = tc_ctas_per_sm(c.n_pad) == 2 && fixed + 3 * band <= half;
    want_pair = allow_pair && c.n_pad <= 32 && xp == 1 && !two_ctas && est_tiles >= 12ll * 148 && fixed + 2 * 2 * band <= budget;
  }
  if (!want_pair)
  {  // two co-resident CTAs when the layer is thin and three tile slots still fit in half the shared memory (measured: with
     // only two slots per CTA the merged fine conv1|pmconv1 layer got 30 % slower)
    const size_t half = (227 * 1024) / 2 - 2048, band = (size_t)TC_TILE_M * max_chunks_of(srcs, nsrc) * 16u * (stride == 2 ? 8 : k * xp);
    if (tc_ctas_per_sm(c.n_pad) == 2 && fixed + 3 * band <= half) { c.ctas_per_sm = 2; budget = half; }
  }
  // all k kernel rows of a source in one TMA load when at least 3 such slots fit beside the weights
  const size_t band_bytes = (size_t)TC_TILE_M * max_chunks * 16u;
  const bool multirow = stride == 1 && fixed + 3 * (size_t)k * xp * band_bytes <= budget;
  const int box_rows = multirow ? k : 1;
  p.slot_bytes = (uint32_t)(band_bytes * (stride == 2 ? 8 : box_rows * xp));
  HV_CHECK_ARG(fixed + 2 * (size_t)p.slot_bytes <= budget, "tc_conv: weights (%u B) + 2 band slots do not fit in shared memory", p.w_bytes);
  int seg = 0, max_shift = 0;
  uint32_t woff16 = 0;
  for (int s = 0; s < nsrc; ++s) {
    const int nch = srcs[s].buf.chunks;
    const uint32_t slab = (uint32_t)nch * c.n_pad;  // one tap's weights, 16 B units
    if (xp > 1) {
      // x-phase source: image [chunk][4 phases][rows][128]; the six views of a row are enumerated by issue_xp4
      max_shift = 2;
      for (int ky = 0; ky < (multirow ? 1 : k); ++ky) {
        HV_CHECK_ARG(seg < TC_MAX_SEGS, "tc_conv: too many segments");
        TcSeg& sg = p.segs[seg++];
        sg.map = s; sg.nchunks = nch; sg.nrows = box_rows; sg.ntaps = xp + 2;
        sg.c1 = ky;
        sg.rel_start2 = 2 * (-pitch - 1);
        sg.a0 = 0; sg.a_step = 0;
        sg.b0 = woff16 + (uint32_t)(ky * (xp + 2)) * slab; sg.b_step = slab; sg.b_row_step = (uint32_t)(xp + 2) * slab;
      }
    } else if (stride == 1) {
      const bool kxp = srcs[s].kxpack;
      if (!kxp) max_shift = max(max_shift, (k - 1) * dil);
      for (int ky = 0; ky < (multirow ? 1 : k); ++ky) {
        HV_CHECK_ARG(seg < TC_MAX_SEGS, "tc_conv: too many segments");
        TcSeg& sg = p.segs[seg++];
        sg.map = s; sg.nchunks = nch; sg.nrows = box_rows; sg.ntaps = kxp ? 1 : k;
        sg.c1 = ky;  // kernel row selected through the row dimension of the tensor map
        sg.rel_start2 = 2 * (-half * dil * pitch - (kxp ? 0 : half * dil));
        sg.a0 = 0; sg.a_step = kxp ? 0u : (uint32_t)dil;
        if (kxp) { sg.b0 = woff16 + (uint32_t)ky * slab; sg.b_step = 0; sg.b_row_step = slab; }
        else { sg.b0 = woff16 + (uint32_t)(ky * k) * slab; sg.b_step = slab; sg.b_row_step = (uint32_t)k * slab; }
      }
    } else {
      // one segment = one 5-D box [chunk][4 sub-planes][2 rows][128 positions]; taps are enumerated by issue_s2d
      max_shift = 1;
      HV_CHECK_ARG(seg < TC_MAX_SEGS, "tc_conv: too many segments");
      TcSeg& sg = p.segs[seg++];
      sg.map = s; sg.c1 = 0; sg.nchunks = nch; sg.nrows = 8; sg.ntaps = 9;
      sg.rel_start2 = 2 * (-pitch - 1);
      sg.a0 = 0; sg.a_step = 0; sg.b0 = woff16; sg.b_step = slab; sg.b_row_step = 0;
    }
    woff16 += (uint32_t)(xp > 1 ? k * (xp + 2) : (srcs[s].kxpack ? k : k * k)) * slab;
  }
  p.nseg = seg;
  for (int i = 0; i < seg; ++i) p.segs[i].tx_bytes = (uint32_t)TC_TILE_M * p.segs[i].nchunks * 16u * p.segs[i].nrows * (xp > 1 ? xp : 1);
  p.tile_adv = TC_TILE_M - max_shift;
  const int span = p.h_out * pitch;  // positions from output (0,0) to the end of the last row (incl. side borders)
  p.tiles_per_image = (span + p.tile_adv - 1) / p.tile_adv;
  p.tiles_magic = ((1ull << 40) + (unsigned long long)p.tiles_per_image - 1) / (unsigned long long)p.tiles_per_image;
  p.total_tiles = p.tiles_per_image * n_images;
  p.pair = (want_pair && tc_issue_code(c) != 0) ? 1 : 0;
  const size_t slot_stride = (size_t)p.slot_bytes * (p.pair ? 2 : 1);
  int nslots = (int)((budget - fixed) / slot_stride);
  nslots = min(nslots, max(2 * seg, 4));
  nslots = min(nslots, 12);
  p.nslots = nslots;
  c.smem = fixed + (size_t)nslots * slot_stride;
  for (int s = 0; s < nsrc; ++s) {
    int rc = make_map(&p.maps[s], srcs[s].buf, k, dil, box_rows);
    if (rc) return rc;
  }
  if (nsrc == 1) p.maps[1] = p.maps[0];
  if (c.arena) {
    const size_t wb = ((size_t)p.w_bytes + 255) & ~(size_t)255;
    HV_CHECK_ARG(wb + c.n_pad * sizeof(float) <= TcConv::kArenaBytes, "tc_conv: packed weights (%zu bytes) exceed the caller's arena", wb);
    c.w_packed = c.arena;
    c.bias_pad = reinterpret_cast<float*>(static_cast<char*>(c.arena) + wb);
  } else {
    HV_CUDA(cudaMalloc(&c.w_packed, p.w_bytes));
    HV_CUDA(cudaMalloc(&c.bias_pad, c.n_pad * sizeof(float)));
  }
  p.w_packed = c.w_packed;
  p.bias = c.bias_pad;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  tc_conv_set_batch(c, n_images);
  if (getenv("HV_TC_DUMP")) {
    fprintf(stderr, "tc_conv: n_pad %d k %d stride %d dil %d cout %d ctas/sm %d slots %d nseg %d s2d %d xp %d tiles %d :", c.n_pad, k, stride, dil,
            cout_real, c.ctas_per_sm, p.nslots, p.nseg, p.s2d_in, p.in_xp, p.total_tiles);
    for (int i = 0; i < p.nseg; ++i) fprintf(stderr, " (rows %d taps %d chunks %d)", p.segs[i].nrows, p.segs[i].ntaps, p.segs[i].nchunks);
    fprintf(stderr, "\n");
  }
  return HV_OK;
}

static int sm_count() {   // of the current device; one process drives one GPU (one rank per GPU), so the first answer is cached
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

void tc_conv_set_batch(TcConv& c, int n_images) {
  c.p.total_tiles = c.p.tiles_per_image * n_images;
  const int sms = sm_count();
  const int rounds = c.p.pair ? (c.p.total_tiles + 1) / 2 : c.p.total_tiles;
  c.grid = min(rounds, sms * c.ctas_per_sm);
}

void tc_conv_set_output_chunked(TcConv& c, const TcBuf& out, int chunk_off, int nchunks, bool up2, int act) {
  TcParams& p = c.p;
  p.out_mode = up2 ? TC_OUT_CHUNKED_UP2 : (out.s2d ? TC_OUT_CHUNKED_S2D : TC_OUT_CHUNKED);
  p.out_xp = out.xp;
  p.out = out.ptr; p.out_pitch = out.pitch(); p.out_border = out.border; p.out_plane = out.plane();
  p.out_sub_plane = out.sub_plane();
  p.out_chunks_total = out.image_chunks(); p.out_chunk_off = chunk_off; p.out_nchunks = nchunks;
  p.act = act;
}

void tc_conv_set_output_heads(TcConv& c, float* head0, float* head1, const TcAux* aux0, const TcAux* aux1) {
  TcParams& p = c.p;
  p.out_mode = TC_OUT_HEADS;
  p.out_xp = c.src[0].buf.xp;   // the aux channels go into buffers of the source's layout
  p.head0 = head0; p.head1 = head1;
  memset(&p.aux0, 0, sizeof(TcAux)); memset(&p.aux1, 0, sizeof(TcAux));
  if (aux0) p.aux0 = *aux0;
  if (aux1) p.aux1 = *aux1;
}

void tc_conv_free(TcConv& c) {
  cudaFree(c.w_packed); cudaFree(c.bias_pad);
  c.w_packed = nullptr; c.bias_pad = nullptr;
}

// ------------------------------------------------------------------------------------------- weight packing
// dst[(tap entry e = (source, ky, kx))][chunk][n_pad][8] bf16; padded channels / filters are zero.
// kx-packed sources have one entry per kernel row: channel ch of the entry = (kx = ch / real, c = ch % real).
struct PackSrc { int ch_off, real, chunks, kxpack, xp, cp; int use_map; short map[32]; int ups, nbhd4; };
__global__ void pack_weights_kernel(const float* __restrict__ wa, const float* __restrict__ ba, int cout_a,
                                    const float* __restrict__ wb, const float* __restrict__ bb, int cout_b, int cin_total,
                                    int k, int n_pad, PackSrc s0, PackSrc s1, int nsrc, __nv_bfloat16* __restrict__ dst,
                                    float* __restrict__ bias_pad, int total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) {
    const int co = (s0.xp > 1 || s0.ups) ? i % s0.cp : i;
    float b = 0.f;
    if (co < cout_a) b = ba ? ba[co] : 0.f;
    else if (co < cout_a + cout_b) b = bb ? bb[co - cout_a] : 0.f;
    bias_pad[i] = b;
  }
  if (i >= total) return;
  const int kk = k * k;
  int rem = i;
  const int c8 = rem & 7; rem >>= 3;
  const int n = rem % n_pad; rem /= n_pad;
  // rem = linear (entry, chunk) index with per-source entry / chunk counts
  const int per0 = (s0.xp > 1 ? k * (s0.xp + 2) : (s0.kxpack ? k : kk)) * s0.chunks;
  PackSrc s = s0;
  if (rem >= per0) { rem -= per0; s = s1; }
  const int chunk = rem % s.chunks, entry = rem / s.chunks;
  const int ch = chunk * 8 + c8;
  int c = ch, tap = entry, co = n;
  bool real = ch < s.real;
  if (s.kxpack && s.use_map) { const int mcode = ch < 32 ? s.map[ch] : -1; real = mcode >= 0; c = mcode & 63; tap = entry * k + (mcode >> 6); }
  else if (s.kxpack) { const int kx = ch / s.real; c = ch - kx * s.real; tap = entry * k + kx; real = kx < k; }
  if (s.xp > 1) {   // entry = ky * (xp + 2) + view; column n = phase * cp + filter; view v carries tap kx = v - phase
    const int ky = entry / (s.xp + 2), view = entry - ky * (s.xp + 2), ph = n / s.cp;
    co = n - ph * s.cp;
    const int kx = view - ph;
    tap = ky * k + kx;
    real = real && kx >= 0 && kx < k;
  }
  float v = 0.f;
  if (s0.ups) {
    // sub-pixel upsample conv: column n = parity (py, px) * cp + filter.  Plain source: entry = low-res tap (dy + 1) * 3 + (dx + 1),
    // weight = sum of the original taps (ky, kx) whose upsampled input pixel falls on that low-res pixel: floor((py + ky - 1) / 2) == dy.
    // 4x4-neighbourhood source: one entry per kernel row of the (3-row) band, only the centre row carries weights: channel
    // (ry, rx) of the centre position feeds tap (ky, kx) = (ry - py, rx - px) of parity (py, px).
    const int pp = n / s0.cp, py = pp >> 1, px = pp & 1;
    co = n - pp * s0.cp;
    if (co < cout_a) {
      if (s.nbhd4) {
        const int ky = (ch >> 2) - py, kx = (ch & 3) - px;
        if (entry == 1 && ch < 16 && ky >= 0 && ky < 3 && kx >= 0 && kx < 3) v = wa[((size_t)co * cin_total + s.ch_off) * kk + ky * 3 + kx];
      } else if (ch < s.real) {
        const int dy = entry / 3 - 1, dx = entry % 3 - 1;
        for (int ky = 0; ky < 3; ++ky)
          for (int kx = 0; kx < 3; ++kx)
            if (((py + ky - 1) >> 1) == dy && ((px + kx - 1) >> 1) == dx) v += wa[((size_t)co * cin_total + s.ch_off + ch) * kk + ky * 3 + kx];
      }
    }
    dst[i] = __float2bfloat16(v);
    return;
  }
  if (real) {
    const int cin = s.ch_off + c;
    if (co < cout_a) v = wa[((size_t)co * cin_total + cin) * kk + tap];
    else if (co < cout_a + cout_b) v = wb[((size_t)(co - cout_a) * cin_total + cin) * kk + tap];
  }
  dst[i] = __float2bfloat16(v);
}

int tc_conv_pack_weights(TcConv& c, const float* wa, const float* ba, int cout_a, const float* wb, const float* bb,
                         int cout_b, cudaStream_t st) {
  HV_CHECK_ARG(cout_a + cout_b == c.cout_real, "tc_conv_pack_weights: filter count mismatch");
  PackSrc s0, s1;
  memset(&s0, 0, sizeof(s0)); memset(&s1, 0, sizeof(s1));
  s0.real = c.src[0].real_channels; s0.chunks = c.src[0].buf.chunks; s0.kxpack = c.src[0].kxpack ? 1 : 0; s0.xp = c.p.in_xp; s0.cp = c.p.cp;
  s1.chunks = 1; s1.xp = 1;
  s0.ups = c.p.ups;
  if (c.p.ups) HV_CHECK_ARG(cout_b == 0, "tc_conv_pack_weights: the sub-pixel upsample mode takes one filter bank");
  if (c.src[0].chan_map) {
    HV_CHECK_ARG(c.src[0].kxpack && c.src[0].buf.chunks * 8 <= 32, "tc_conv_pack_weights: a channel map needs a kx-packed source of <= 32 channels");
    s0.use_map = 1;
    for (int i = 0; i < 32; ++i) s0.map[i] = i < c.src[0].buf.chunks * 8 ? c.src[0].chan_map[i] : (short)-1;
  }
  int cin_total = c.src[0].real_channels;
  if (c.nsrc == 2) {
    s1.ch_off = c.src[0].real_channels; s1.real = c.src[1].real_channels; s1.chunks = c.src[1].buf.chunks; s1.kxpack = c.src[1].kxpack ? 1 : 0;
    s1.nbhd4 = c.src[1].nbhd4 ? 1 : 0;
    cin_total += c.src[1].real_channels;
  }
  const int total = (int)(c.p.w_bytes / 2);
  pack_weights_kernel<<<(max(total, c.n_pad) + 255) / 256, 256, 0, st>>>(wa, ba, cout_a, wb, bb, cout_b, cin_total, c.k, c.n_pad, s0,
                                                                          s1, c.nsrc, (__nv_bfloat16*)c.w_packed, c.bias_pad, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

static long long* g_trace = nullptr;
void tc_set_trace(long long* dev_buf) { g_trace = dev_buf; }
static long long* g_timeline = nullptr;
static int g_timeline_count = 0;
void tc_set_timeline(long long* dev_buf) { g_timeline = dev_buf; g_timeline_count = 0; }
long long* tc_timeline_next() { return g_timeline ? g_timeline + 4 * (g_timeline_count++) : nullptr; }

template <int N_PAD, int ACT, int FIXED = 0, bool DIAG = true>
static int tc_launch_na(const TcConv& c, cudaStream_t st) {
  static bool configured = false;  // per instantiation; the attribute is sticky for the process
  if (!configured) {
    HV_CUDA(cudaFuncSetAttribute(conv_tc_kernel<N_PAD, ACT, FIXED, DIAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    configured = true;
  }
  // programmatic dependent launch: the kernel may start while its predecessor in the stream drains; it prefetches its
  // weights / sets up barriers and TMEM, then griddepcontrol.wait's before touching the predecessor's output
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(c.grid);
  cfg.blockDim = dim3(tc_threads(N_PAD));
  cfg.dynamicSmemBytes = c.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TcParams q = c.p;
  q.trace = g_trace;
  q.timeline = g_timeline ? g_timeline + 4 * (g_timeline_count++) : nullptr;
  HV_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<N_PAD, ACT, FIXED, DIAG>, q));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// compile-time issue shape of a layer, or 0 when its segments do not fit one of the specialised families
static int tc_issue_code(const TcConv& c);
static int tc_fixed_code(const TcConv& c) {
  if (c.force_generic) return 0;
  const int issue = tc_issue_code(c);
  if (!issue) return 0;
  const TcParams& p = c.p;
  int out = 0;
  if (p.out_mode == TC_OUT_HEADS) out = 3;
  else if (p.out_mode == TC_OUT_CHUNKED_S2D) out = 4;
  else if (p.out_mode == TC_OUT_CHUNKED) out = p.out_xp > 1 ? 5 : 1;
  else out = p.out_xp > 1 ? 6 : 2;
  return (p.pair ? 1 << 20 : 0) | out << 16 | issue;
}
static int tc_issue_code(const TcConv& c) {
  const TcParams& p = c.p;
  const TcSeg& s0 = p.segs[0];
  const int ks = s0.nchunks >> 1;
  if (p.s2d_in) return p.nseg == 1 ? tc_shape_code(2, 0, 0, ks) : 0;
  if (p.in_xp > 1) {
    for (int i = 1; i < p.nseg; ++i)
      if (p.segs[i].nrows != s0.nrows || p.segs[i].nchunks != s0.nchunks) return 0;
    return tc_shape_code(3, s0.nrows, 0, ks);
  }
  if (p.nseg == 2 && s0.nrows == 3 && s0.ntaps == 3 && p.segs[1].nrows == 3 && p.segs[1].ntaps == 1 && p.segs[1].nchunks == 2)
    return tc_shape_code(4, 0, 0, ks);
  for (int i = 1; i < p.nseg; ++i)
    if (p.segs[i].nrows != s0.nrows || p.segs[i].ntaps != s0.ntaps || p.segs[i].nchunks != s0.nchunks) return 0;
  return tc_shape_code(1, s0.nrows, s0.ntaps, ks);
}

// the specialised instances: (N_PAD, activation, output mode << 16 | issue shape) of every layer of the generator plan (HV_TC_DUMP=1
// prints this list from a live plan); anything else runs the FIXED = 0 instance
#define HV_TC_FIXED_LIST(X) \
  X(64, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 4)) \
  X(64, HV_ACT_ELU, 5 << 16 | tc_shape_code(3, 1, 0, 2)) \
  X(64, HV_ACT_ELU, 2 << 16 | tc_shape_code(1, 3, 3, 4)) \
  X(64, HV_ACT_ELU, 1 << 16 | tc_shape_code(2, 0, 0, 2)) \
  X(32, HV_ACT_ELU, 5 << 16 | tc_shape_code(3, 3, 0, 1)) \
  X(32, HV_ACT_ELU, 4 << 16 | tc_shape_code(1, 3, 3, 1)) \
  X(32, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 4)) \
  X(16, HV_ACT_ELU, 1 << 16 | tc_shape_code(2, 0, 0, 1)) \
  X(16, -1, 3 << 16 | tc_shape_code(3, 3, 0, 1)) \
  X(64, HV_ACT_ELU, 1 << 16 | tc_shape_code(4, 0, 0, 4)) \
  X(64, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(64, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 1, 3, 4)) \
  X(64, HV_ACT_RELU, 1 << 16 | tc_shape_code(1, 3, 3, 4)) \
  X(32, HV_ACT_ELU, 6 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(32, HV_ACT_ELU, 5 << 16 | tc_shape_code(4, 0, 0, 2)) \
  X(32, HV_ACT_ELU, 4 << 16 | tc_shape_code(1, 5, 1, 2)) \
  X(32, HV_ACT_ELU, 4 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(32, HV_ACT_ELU, 2 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(32, HV_ACT_ELU, 1 << 16 | tc_shape_code(2, 0, 0, 2)) \
  X(32, HV_ACT_ELU, 1 << 16 | tc_shape_code(2, 0, 0, 1)) \
  X(16, HV_ACT_ELU, 4 << 16 | tc_shape_code(1, 5, 1, 1)) \
  X(32, HV_ACT_ELU, 1 << 20 | 4 << 16 | tc_shape_code(1, 5, 1, 2)) \
  X(64, HV_ACT_ELU, 5 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(128, HV_ACT_ELU, 5 << 16 | tc_shape_code(4, 0, 0, 2)) \
  X(128, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 1, 3, 4)) \
  X(32, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(64, -1, 1 << 16 | tc_shape_code(1, 3, 3, 4))   /* 64 -> 64 3x3 without a compiled-in activation: the data gradient of the trunk layers */ \
  /* the stand-alone op inside the training step (forward of the thin layers, data gradients: HV_TC_DUMP=1 python tools/bench_train.py): \
     the generic instance costs 2 - 4x a specialised one */ \
  X(16, -1, 1 << 16 | tc_shape_code(1, 3, 3, 1)) \
  X(16, -1, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(16, -1, 1 << 16 | tc_shape_code(1, 5, 5, 1)) \
  X(32, -1, 1 << 16 | tc_shape_code(1, 3, 3, 1)) \
  X(32, -1, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(32, -1, 1 << 16 | tc_shape_code(1, 3, 3, 4)) \
  X(64, -1, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(16, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 5, 5, 1)) \
  X(16, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 1)) \
  X(16, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 2)) \
  X(32, HV_ACT_ELU, 1 << 16 | tc_shape_code(1, 3, 3, 1))

template <int N_PAD>
static int tc_launch_n(const TcConv& c, cudaStream_t st) {
  // activation as a compile-time constant where an instance exists (ELU everywhere, ReLU for pmconv6), else -1 = run-time switch
  int act = -1;
  if (c.p.out_mode != TC_OUT_HEADS && c.p.act == HV_ACT_ELU) act = HV_ACT_ELU;
  const int fixed = tc_fixed_code(c);
  if (c.p.out_mode != TC_OUT_HEADS && c.p.act == HV_ACT_RELU && N_PAD == 64 && fixed == (1 << 16 | tc_shape_code(1, 3, 3, 4))) act = HV_ACT_RELU;
  static const bool dump = getenv("HV_TC_DUMP") != nullptr;
  if (dump) fprintf(stderr, "tc_launch: X(%d, %s, %d << 20 | %d << 16 | tc_shape_code(%d, %d, %d, %d))\n", N_PAD, act == HV_ACT_ELU ? "HV_ACT_ELU" : (act == HV_ACT_RELU ? "HV_ACT_RELU" : "-1"),
                                    fixed >> 20 & 1, fixed >> 16 & 15, (fixed >> 12) & 15, (fixed >> 8) & 15, (fixed >> 4) & 15, fixed & 15);
  if (c.p.pair && !(fixed >> 20 & 1)) { set_error("tc_conv: a paired layer needs a specialised kernel instance"); return HV_ERR_UNSUPPORTED; }
  // a diagnostic is active (trace / timeline hook set): the instances that carry the hooks
  const bool diag = g_trace != nullptr || g_timeline != nullptr;
#define HV_TC_TRY(NP, A, F)                                                                                      \
  if (N_PAD == (NP) && act == (A) && fixed == (F))                                                              \
    return diag ? tc_launch_na<NP, A, (N_PAD == (NP) ? (F) : 0), true>(c, st)                                   \
                : tc_launch_na<NP, A, (N_PAD == (NP) ? (F) : 0), (N_PAD == (NP) ? false : true)>(c, st);
  HV_TC_FIXED_LIST(HV_TC_TRY)
#undef HV_TC_TRY
  if (c.p.pair) { set_error("tc_conv: no specialised kernel instance for paired layer code 0x%x (n_pad %d)", fixed, N_PAD); return HV_ERR_UNSUPPORTED; }
  if (act == HV_ACT_ELU) return tc_launch_na<N_PAD, HV_ACT_ELU>(c, st);
  return tc_launch_na<N_PAD, -1>(c, st);
}

int tc_conv_launch(const TcConv& c, cudaStream_t st) {
  switch (c.n_pad) {
    case 16: return tc_launch_n<16>(c, st);
    case 32: return tc_launch_n<32>(c, st);
    case 64: return tc_launch_n<64>(c, st);
    case 128: return tc_launch_n<128>(c, st);
    default: set_error("tc_conv: bad n_pad %d", c.n_pad); return HV_ERR_INVALID;
  }
}

// ------------------------------------------------------------------------------------------- layout converters
__global__ void pack_nchw_kernel(const float* __restrict__ src, int src_channels, int mode, TcBuf dst, int ch0) {
  const int n = blockIdx.z, c = blockIdx.y, h = dst.h, w = dst.w;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int y = i / w, x = i - y * w;
  float v;
  if (mode == HV_SRC_SCALAR) v = src[n];
  else if (mode == HV_SRC_SUB2) v = src[(((size_t)n * src_channels + c) * (2 * h) + 2 * y) * (2 * w) + 2 * x];
  else if (mode == HV_SRC_UP2) v = src[(((size_t)n * src_channels + c) * (h / 2) + y / 2) * (w / 2) + x / 2];
  else v = src[(((size_t)n * src_channels + c) * h + y) * w + x];
  const int ch = ch0 + c;
  dst.ptr[dst.chunk_base(n, ch >> 3) + dst.pos(y, x) * 8 + (ch & 7)] = __float2bfloat16(v);
}

// whole chunks: one thread = one pixel of one 8-channel chunk - eight plane reads (each coalesced across the warp), ONE 16-byte store
// (the scalar kernel above writes 2 bytes per thread at a 16-byte stride: an eighth of every sector per warp instruction)
__global__ void __launch_bounds__(256) pack_nchw_chunks_kernel(const float* __restrict__ src, int src_channels, int mode, TcBuf dst, int chunk0) {
  const int n = blockIdx.z, cc = blockIdx.y, h = dst.h, w = dst.w;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int y = i / w, x = i - y * w;
  int sh = h, sw = w, sy = y, sx = x;
  if (mode == HV_SRC_SUB2) { sh = 2 * h; sw = 2 * w; sy = 2 * y; sx = 2 * x; }
  else if (mode == HV_SRC_UP2) { sh = h / 2; sw = w / 2; sy = y / 2; sx = x / 2; }
  const float* p = src + (((size_t)n * src_channels + cc * 8) * sh + sy) * sw + sx;
  const size_t plane = (size_t)sh * sw;
  __align__(16) __nv_bfloat16 v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = __float2bfloat16(__ldg(p + j * plane));
  *reinterpret_cast<uint4*>(dst.ptr + dst.chunk_base(n, chunk0 + cc) + dst.pos(y, x) * 8) = *reinterpret_cast<const uint4*>(v);
}

int tc_pack_nchw(const float* src, int src_channels, int mode, const TcBuf& dst, int ch0, cudaStream_t st) {
  HV_CHECK_ARG(src && dst.ptr && ch0 + src_channels <= dst.chunks * 8, "tc_pack_nchw: bad argument");
  if ((ch0 & 7) == 0 && (src_channels & 7) == 0 && mode != HV_SRC_SCALAR) {
    pack_nchw_chunks_kernel<<<dim3((dst.h * dst.w + 255) / 256, src_channels / 8, dst.n), 256, 0, st>>>(src, src_channels, mode, dst, ch0 >> 3);
    HV_LAUNCH_CHECK();
    return HV_OK;
  }
  dim3 grid((dst.h * dst.w + 255) / 256, src_channels, dst.n);
  pack_nchw_kernel<<<grid, 256, 0, st>>>(src, src_channels, mode, dst, ch0);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// kx-packed input planes: one thread = one position; all K * NSRC channels are built with compile-time indices
struct PackKxArgs { const float* ptr[4]; int mode[4]; int dil; };
template <int NSRC, int K>
__global__ void __launch_bounds__(256) pack_kx_kernel(PackKxArgs a, TcBuf dst) {
  pdl_prologue();
  constexpr int NCH = (K * NSRC + 15) / 16 * 2;  // chunks written (even)
  const int n = blockIdx.y, h = dst.h, w = dst.w;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int y = i / w, x = i - y * w;
  __align__(16) __nv_bfloat16 o[NCH * 8];
#pragma unroll
  for (int j = 0; j < NCH * 8; ++j) o[j] = __float2bfloat16(0.f);
  // the kernel is issue-bound (ncu: 78 - 86 % of the issue slots): the source mode is decided once per source, not per tap, and
  // positions whose K taps all lie inside the row skip the per-tap bounds checks
  const int reach = (K / 2) * a.dil;
  const bool interior = x >= reach && x + reach < w;
#pragma unroll
  for (int c = 0; c < NSRC; ++c) {
    const float* src = a.ptr[c];
    const int mode = a.mode[c];
    if (mode == HV_SRC_SCALAR) {
      const __nv_bfloat16 sv = __float2bfloat16(src[n]);
#pragma unroll
      for (int kx = 0; kx < K; ++kx) {
        const int xs = x + (kx - K / 2) * a.dil;
        o[kx * NSRC + c] = (interior || (xs >= 0 && xs < w)) ? sv : __float2bfloat16(0.f);
      }
    } else if (mode == HV_SRC_SUB2) {
      const float* row = src + ((size_t)n * (2 * h) + 2 * y) * (2 * w);
#pragma unroll
      for (int kx = 0; kx < K; ++kx) {
        const int xs = x + (kx - K / 2) * a.dil;
        o[kx * NSRC + c] = __float2bfloat16((interior || (xs >= 0 && xs < w)) ? row[2 * xs] : 0.f);
      }
    } else {
      const float* row = src + ((size_t)n * h + y) * w + x;
      if (interior) {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) o[kx * NSRC + c] = __float2bfloat16(row[(kx - K / 2) * a.dil]);
      } else {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
          const int d = (kx - K / 2) * a.dil, xs = x + d;
          o[kx * NSRC + c] = __float2bfloat16((xs >= 0 && xs < w) ? row[d] : 0.f);
        }
      }
    }
  }
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch)
    *reinterpret_cast<uint4*>(dst.ptr + dst.chunk_base(n, ch) + dst.pos(y, x) * 8) = *reinterpret_cast<const uint4*>(o + ch * 8);
}

int tc_pack_kx(const TcPlaneSrc* srcs, int nsrc, int k, int dil, const TcBuf& dst, cudaStream_t st) {
  HV_CHECK_ARG(srcs && nsrc >= 1 && nsrc <= 4 && dst.ptr && !dst.s2d && k * nsrc <= dst.chunks * 8, "tc_pack_kx: bad argument");
  PackKxArgs a;
  a.dil = dil;
  for (int i = 0; i < 4; ++i) { a.ptr[i] = i < nsrc ? srcs[i].ptr : nullptr; a.mode[i] = i < nsrc ? srcs[i].mode : 0; }
  dim3 grid((dst.h * dst.w + 255) / 256, dst.n);
  const int need = (k * nsrc + 15) / 16 * 2;
  HV_CHECK_ARG(need == dst.chunks, "tc_pack_kx: destination has %d chunks, the packed channels need %d", dst.chunks, need);
  if (nsrc == 1 && k == 3) HV_CUDA(launch_pdl(pack_kx_kernel<1, 3>, grid, dim3(256), 0, st, a, dst));
  else if (nsrc == 1 && k == 5) HV_CUDA(launch_pdl(pack_kx_kernel<1, 5>, grid, dim3(256), 0, st, a, dst));
  else if (nsrc == 3 && k == 5) HV_CUDA(launch_pdl(pack_kx_kernel<3, 5>, grid, dim3(256), 0, st, a, dst));
  else if (nsrc == 4 && k == 5) HV_CUDA(launch_pdl(pack_kx_kernel<4, 5>, grid, dim3(256), 0, st, a, dst));
  else { set_error("tc_pack_kx: no instance for %d sources, k=%d", nsrc, k); return HV_ERR_UNSUPPORTED; }
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// sub = 2 reads every second pixel of every second row: the native-resolution result of a layer whose output is stored
// nearest-x2-upsampled (the producer's epilogue writes the 2 x 2 replicas)
// 4x4 neighbourhood of a high-resolution plane at low resolution (TcSource::nbhd4): one thread = one low-res position, 32-byte store
__global__ void __launch_bounds__(256) pack_nbhd4_kernel(const float* __restrict__ src, TcBuf dst) {
  pdl_prologue();
  const int n = blockIdx.y, h = dst.h, w = dst.w;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int m = i / w, q = i - m * w;
  const float* plane = src + (size_t)n * (2 * h) * (2 * w);
  __align__(16) __nv_bfloat16 o[16];
#pragma unroll
  for (int ry = 0; ry < 4; ++ry) {
    const int y = 2 * m - 1 + ry;
#pragma unroll
    for (int rx = 0; rx < 4; ++rx) {
      const int x = 2 * q - 1 + rx;
      o[ry * 4 + rx] = __float2bfloat16((y >= 0 && y < 2 * h && x >= 0 && x < 2 * w) ? plane[(size_t)y * (2 * w) + x] : 0.f);
    }
  }
#pragma unroll
  for (int ch = 0; ch < 2; ++ch)
    *reinterpret_cast<uint4*>(dst.ptr + dst.chunk_base(n, ch) + dst.pos(m, q) * 8) = *reinterpret_cast<const uint4*>(o + ch * 8);
}

int tc_pack_nbhd4(const float* src, const TcBuf& dst, cudaStream_t st) {
  HV_CHECK_ARG(src && dst.ptr && dst.chunks == 2 && !dst.s2d && dst.xp == 1, "tc_pack_nbhd4: bad argument");
  HV_CUDA(launch_pdl(pack_nbhd4_kernel, dim3((dst.h * dst.w + 255) / 256, dst.n), dim3(256), 0, st, src, dst));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

__global__ void unpack_nchw_kernel(TcBuf src, int ch0, int channels, float* __restrict__ dst, int sub, int c_begin) {
  const int n = blockIdx.z, c = c_begin + blockIdx.y, h = src.h / sub, w = src.w / sub;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int y = i / w, x = i - y * w, ch = ch0 + c;
  dst[((size_t)n * channels + c) * h * w + i] =
      __bfloat162float(src.ptr[src.chunk_base(n, ch >> 3) + src.pos(y * sub, x * sub) * 8 + (ch & 7)]);
}

// whole chunks: one 16-byte load per thread, eight plane stores (each coalesced across the warp)
__global__ void __launch_bounds__(256) unpack_nchw_chunks_kernel(TcBuf src, int chunk0, int channels, float* __restrict__ dst, int sub) {
  const int n = blockIdx.z, cc = blockIdx.y, h = src.h / sub, w = src.w / sub;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int y = i / w, x = i - y * w;
  const uint4 raw = *reinterpret_cast<const uint4*>(src.ptr + src.chunk_base(n, chunk0 + cc) + src.pos(y * sub, x * sub) * 8);
  const __nv_bfloat16* v = reinterpret_cast<const __nv_bfloat16*>(&raw);
  float* out = dst + ((size_t)n * channels + cc * 8) * h * w + i;
#pragma unroll
  for (int j = 0; j < 8; ++j) out[(size_t)j * h * w] = __bfloat162float(v[j]);
}

int tc_unpack_nchw(const TcBuf& src, int ch0, int channels, float* dst, cudaStream_t st, int sub) {
  HV_CHECK_ARG(src.ptr && dst && ch0 + channels <= src.chunks * 8 && (sub == 1 || sub == 2), "tc_unpack_nchw: bad argument");
  const unsigned px_blocks = (unsigned)((src.h / sub * (src.w / sub) + 255) / 256);
  int done = 0;
  if ((ch0 & 7) == 0 && channels >= 8) {       // whole chunks with 16-byte loads, the remainder channel by channel
    unpack_nchw_chunks_kernel<<<dim3(px_blocks, channels / 8, src.n), 256, 0, st>>>(src, ch0 >> 3, channels, dst, sub);
    HV_LAUNCH_CHECK();
    done = channels & ~7;
  }
  if (done < channels) {
    unpack_nchw_kernel<<<dim3(px_blocks, channels - done, src.n), 256, 0, st>>>(src, ch0, channels, dst, sub, done);
    HV_LAUNCH_CHECK();
  }
  return HV_OK;
}

// SHRM height head on a chunked buffer: sigmoid(fc(mean_HW(x)))  (inpaint_networks.py:90-93,:211-214)
// grid (chunks, n): every CTA reduces one 8-channel chunk plane to its share of the dot product; the last CTA of a
// sample (self-resetting ticket counter) adds the shares in a fixed order and applies bias + sigmoid.
__global__ void __launch_bounds__(256) tc_gap_fc_kernel(TcBuf x, const float* __restrict__ fw, const float* __restrict__ fb,
                                                        float* __restrict__ out, float* __restrict__ partial,
                                                        unsigned int* __restrict__ ticket) {
  const int c = blockIdx.x, n = blockIdx.y;
  const int h = x.h, w = x.w;
  __shared__ float red[32];
  __shared__ bool last;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const __nv_bfloat16* pl = x.ptr + x.chunk_base(n, c);
  for (int i = threadIdx.x; i < h * w; i += blockDim.x) {
    const int y = i / w, xx = i - y * w;
    const uint4 raw = *reinterpret_cast<const uint4*>(pl + x.pos(y, xx) * 8);
    const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(hp[j]); acc[2 * j] += f.x; acc[2 * j + 1] += f.y; }
  }
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) dot += acc[j] * fw[c * 8 + j];
  dot = block_sum(dot, red) / (float)(h * w);
  if (threadIdx.x == 0) {
    partial[n * x.chunks + c] = dot;
    __threadfence();
    last = atomicAdd(&ticket[n], 1u) == (unsigned)x.chunks - 1;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    float t = 0.f;
    for (int i = 0; i < x.chunks; ++i) t += __ldcg(&partial[n * x.chunks + i]);
    out[n] = 1.f / (1.f + expf(-(t + fb[0])));
    ticket[n] = 0;
  }
}

// scratch: (max_batch * chunks) floats + max_batch zero-initialised uints
int tc_gap_fc_sigmoid(const TcBuf& x, const float* fw, const float* fb, float* out, float* partial, unsigned int* ticket,
                      cudaStream_t st) {
  HV_CHECK_ARG(x.ptr && fw && fb && out && partial && ticket && !x.s2d, "tc_gap_fc_sigmoid: bad argument");
  tc_gap_fc_kernel<<<dim3(x.chunks, x.n), 256, 0, st>>>(x, fw, fb, out, partial, ticket);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

}  // namespace hv
