// Fused input stem of a generator stage at 256 x 256: the kx-packed 5x5 input conv (ELU) followed by the stride-2 3x3 conv(s) that read
// it, in ONE persistent launch.  Coarse stage: conv1 (3 -> 16) -> conv2_downsample (16 -> 32) (models/inpaint_networks.py:41-42); fine
// stage: the merged conv1 | pmconv1 (4 -> 16 + 16) -> conv2_downsample (channels 0-15) and pmconv2_downsample (channels 16-31) (:126-127,
// :143-144).  The 256 x 256 intermediate lives only in shared memory: per stage it saves one launch ramp and the write + re-read of a
// 33.5 MB (coarse) / 67 MB (fine) bf16 map, and in the fine stage pmconv2 no longer waits on the side stream for a cross-stream event.
//
// Work unit = (image, strip of R stride-2 output rows y0 .. y0+R-1).  The strip needs the 5x5 conv rows 2 y0 - 1 .. 2 y0 + 2R - 1 (the
// first one is recomputed by the strip above; row -1 is the stride-2 conv's zero padding) and the input rows 2 y0 - 3 .. 2 y0 + 2R + 1.
//   5x5 conv     : accumulator tile = half an image row (x = 128 h .. 128 h + 127), two tiles per row; tap row ky reads the input row
//                  slot's positions 128 h .. 128 h + 127 (the input is kx-packed, so one K-step set per kernel row, as in conv_tc)
//   stride-2 conv: accumulator tile = one output row (x2 = 0 .. 127); the intermediate row is stored per chunk as [O' 129][E 128]:
//                  E[j] = pixel 2 j, O'[0] = 0 (the left padding), O'[j + 1] = pixel 2 j + 1.  Tap (ky, kx) of output x2 reads pixel
//                  2 x2 + kx - 1 of row 2 y2 + ky - 1: O'[x2] / E[x2] / O'[x2 + 1], i.e. a shifted descriptor start (0 / 129 / 1)
//                  inside the ring slot of that row.
// Shared memory, fine: weights 10 KB + 2 x 4.5 KB, 11 input row slots x 12 KB (chunks 0-2) + a 4 KB zero chunk, 4 intermediate row
// slots x 16 KB, barriers / bias 1 KB = 220 KB; coarse: weights 11.5 KB, 16 input slots x 8 KB, 6 intermediate slots x 8 KB = 188 KB.
// One CTA per SM.
//
// Roles: warp 24 TMA producer (input rows; weights once), warp 25 MMA issuer of the 5x5 conv, warp 26 MMA issuer of the stride-2
// conv(s), warps 0-15 epilogue of the 5x5 conv (two groups of 8 warps, alternate rows, 4 warps per half row: TMEM -> bias + ELU ->
// bf16 -> intermediate slot, fence.proxy.async, arrive), warps 16-23 epilogue of the stride-2 conv(s) (two groups, alternate rows:
// -> global, conv_tc's layout).  The 5x5 conv's epilogue is the heaviest role (2 x 256 x N1 values per output row): with 8 warps
// (64 values per thread) it bound the launch (fine stem 51 us on B200), hence 16.
// Every accumulator sees exactly the MMA sequence of the per-layer instance ((kernel row, K-step) for the 5x5 conv, issue_s2d's (ky, kx)
// for the stride-2 conv) with the same operand bytes, and the epilogue arithmetic of conv_tc_kernel, so the fused stem equals the
// per-layer launches bit for bit.
#include <string.h>
#include "hv_common.cuh"
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace hv {

namespace {

constexpr int kW = 256, kW2 = 128;        // image width at the input / at the stride-2 output
constexpr int kMidPos = 129 + 128;        // positions per chunk of an intermediate row: O' then E

template <bool FINE>
struct StemCfg {
  static constexpr int KIN = FINE ? 4 : 2;             // input chunks (kx-packed channels / 8)
  // chunks brought by TMA: chunk 3 of the fine input carries no channel (kFineInputMap) and is zero in memory; its K-step reads a zero
  // block of shared memory instead (same operand bytes), which makes room for a deeper input ring
  static constexpr int KLOAD = FINE ? 3 : 2;
  // ring depths: the 5x5 conv of a row holds 5 input rows until its MMAs complete, the rest is prefetch that hides the TMA latency
  static constexpr int kInSlots = FINE ? 11 : 16, kMidSlots = FINE ? 4 : 6;
  static constexpr int N1 = FINE ? 32 : 16;            // 5x5 conv filters (= intermediate channels)
  static constexpr int KMID = N1 / 8;                  // intermediate chunks
  static constexpr int N2 = FINE ? 16 : 32;            // filters of one stride-2 layer
  static constexpr int NL2 = FINE ? 2 : 1;             // stride-2 layers (each reads 2 intermediate chunks)
  static constexpr uint32_t W1 = 5u * KIN * N1 * 16u;  // packed weights of the per-layer instances
  static constexpr uint32_t W2 = 9u * 2u * N2 * 16u;
  static constexpr uint32_t kInSlot = (uint32_t)KLOAD * kW * 16u;
  static constexpr uint32_t kMidSlot = (uint32_t)KMID * kMidPos * 16u;
  static constexpr uint32_t kOffIn = (W1 + NL2 * W2 + 1023u) & ~1023u;
  static constexpr uint32_t kOffZero = kOffIn + kInSlots * kInSlot;          // fine: one zero chunk of a row (4 KB)
  static constexpr uint32_t kOffMid = kOffZero + (FINE ? kW * 16u : 0u);
  static constexpr uint32_t kOffBar = (kOffMid + kMidSlots * kMidSlot + 127u) & ~127u;
  static constexpr uint32_t kSmem = kOffBar + 1024u;
  static constexpr int kTmemCols = FINE ? 256 : 128;   // 2 stages x 2 tiles x N1 (5x5 conv) + 2 stages x 32 (stride-2)
  static_assert(kSmem <= 227u * 1024u, "stem kernel shared memory");
  static_assert(8 * (2 * kInSlots + 2 * kMidSlots + 9) <= 512, "stem kernel barriers");
  static_assert(4 * N1 + 64 <= kTmemCols, "stem kernel TMEM columns");
};
constexpr int kThreads = 27 * 32;   // 16 + 8 epilogue warps, producer, two MMA issuers

__device__ __forceinline__ float elu_fast(float x) {   // == act_fast<HV_ACT_ELU> of conv_tc.cu
  if (x > 0.f) return x;
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y - 1.f;
}

__device__ __forceinline__ uint32_t pack_elu(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(elu_fast(a), elu_fast(b));
  return *reinterpret_cast<uint32_t*>(&h);
}

}  // namespace

template <bool FINE>
__global__ void __launch_bounds__(kThreads, 1) stem_tc_kernel(const __grid_constant__ TcStemParams p) {
  using C = StemCfg<FINE>;
  constexpr int KIN = C::KIN, N1 = C::N1, KMID = C::KMID, N2 = C::N2, NL2 = C::NL2;
  constexpr int kInSlots = C::kInSlots, kMidSlots = C::kMidSlots;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_PRODUCER = 24, W_MMA1 = 25, W_MMA2 = 26;
  const uint32_t s_base = smem_u32(smem);
  const uint32_t bars = s_base + C::kOffBar;
  const uint32_t bar_in_full = bars, bar_in_empty = bar_in_full + 8 * kInSlots;
  const uint32_t bar_mid_ready = bar_in_empty + 8 * kInSlots, bar_mid_free = bar_mid_ready + 8 * kMidSlots;
  const uint32_t bar_a1full = bar_mid_free + 8 * kMidSlots, bar_a1empty = bar_a1full + 16;
  const uint32_t bar_a2full = bar_a1full + 32, bar_a2empty = bar_a1full + 48;
  const uint32_t bar_w = bar_a1full + 64;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + C::kOffBar + 960);
  float* s_bias = reinterpret_cast<float*>(smem + C::kOffBar + 512);   // [0, N1): 5x5 conv, [64, 96): stride-2 conv(s)

  if (p.timeline && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    atomicMin(reinterpret_cast<unsigned long long*>(p.timeline), gt);
  }
  if (warp == W_PRODUCER && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&p.map_in) : "memory");
  if (warp == W_MMA1) {
    if (lane == 0) {
      for (int i = 0; i < kInSlots; ++i) { mbar_init(bar_in_full + 8u * i, 1); mbar_init(bar_in_empty + 8u * i, 1); }
      for (int i = 0; i < kMidSlots; ++i) { mbar_init(bar_mid_ready + 8u * i, 256); mbar_init(bar_mid_free + 8u * i, 1); }
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_a1full + 8u * i, 1); mbar_init(bar_a1empty + 8u * i, 256);
        mbar_init(bar_a2full + 8u * i, 1); mbar_init(bar_a2empty + 8u * i, 128);
      }
      mbar_init(bar_w, 1);
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(C::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x < N1) s_bias[threadIdx.x] = __ldg(p.bias1 + threadIdx.x);
  else if (threadIdx.x >= 64 && threadIdx.x < 96) {
    const int c = threadIdx.x - 64;
    s_bias[threadIdx.x] = NL2 == 2 && c >= N2 ? __ldg(p.bias3 + c - N2) : __ldg(p.bias2 + c);
  }
  // O'[0] of every chunk of every intermediate slot: the stride-2 conv's left zero padding, never written by the epilogue
  if (threadIdx.x >= 128 && threadIdx.x < 128 + kMidSlots * KMID) {
    const int i = threadIdx.x - 128;
    *reinterpret_cast<uint4*>(smem + C::kOffMid + (i / KMID) * C::kMidSlot + (i % KMID) * kMidPos * 16) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  if (FINE && threadIdx.x >= 256 && threadIdx.x < 256 + kW) {
    *reinterpret_cast<uint4*>(smem + C::kOffZero + (threadIdx.x - 256) * 16) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int R = p.rows_per_unit, strips = p.strips, units = p.units;

  if (warp == W_PRODUCER) {
    // ===================================================================== TMA producer: input rows 2 y0 - 3 .. 2 y0 + 2 ru + 1
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(bar_w, C::W1 + NL2 * C::W2);
      bulk_load(s_base, p.w1, C::W1, bar_w);
      bulk_load(s_base + C::W1, p.w2, C::W2, bar_w);
      if (NL2 == 2) bulk_load(s_base + C::W1 + C::W2, p.w3, C::W2, bar_w);
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");   // the input rows are written by earlier kernels of the stream
    uint32_t seq = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int img = u / strips, y0 = (u - img * strips) * R, ru = min(R, kW2 - y0);
      for (int t = 0; t < 2 * ru + 5; ++t, ++seq) {
        const uint32_t slot = seq % kInSlots, par = (seq / kInSlots) & 1u;
        mbar_wait(bar_in_empty + 8u * slot, par ^ 1u);
        if (leader) {
          const uint32_t fb = bar_in_full + 8u * slot;
          mbar_expect_tx(fb, C::kInSlot);   // chunks 0 .. KLOAD - 1
          // plane row of image row 2 y0 - 3 + t (border 2); row -1 is outside the map: zero-filled by the TMA unit
          tma_load_5d(s_base + C::kOffIn + slot * C::kInSlot, &p.map_in, fb, 0, 0, 2 * y0 - 1 + t, 0, img);
        }
      }
    }
  } else if (warp == W_MMA1) {
    // ===================================================================== MMA issuer, 5x5 conv: intermediate row i of the strip
    // (image row 2 y0 - 1 + i) reads input rows i .. i + 4 of the strip
    const bool leader = elect_one();
    constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N1 >> 3) << 17) | ((128u >> 4) << 24);
    constexpr uint32_t lbo = (uint32_t)kW;                 // input chunks are 256 positions apart (16 B units)
    constexpr uint32_t slab = (uint32_t)KIN * N1;          // one kernel row's weights (16 B units)
    mbar_wait(bar_w, 0);
    tc_fence_after();
    const uint32_t b_lo = ((uint32_t)N1 << 16) + (s_base >> 4);
    uint32_t in_base = 0, waited = 0, cnt = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int img = u / strips, y0 = (u - img * strips) * R, ru = min(R, kW2 - y0);
      for (int i = 0; i <= 2 * ru; ++i, ++cnt) {
        while (waited < in_base + (uint32_t)(i + 5)) {
          mbar_wait(bar_in_full + 8u * (waited % kInSlots), (waited / kInSlots) & 1u);
          ++waited;
        }
        const uint32_t acc = cnt & 1u;
        mbar_wait(bar_a1empty + 8u * acc, ((cnt >> 1) & 1u) ^ 1u);
        tc_fence_after();
        uint32_t a_lo[5][KIN / 2];   // per (kernel row, K-step): chunks 2 ks, 2 ks + 1 (fine, ks = 1: chunk 2 and the zero block)
#pragma unroll
        for (int ky = 0; ky < 5; ++ky) {
          const uint32_t slot_lo = ((s_base + C::kOffIn) >> 4) + ((in_base + (uint32_t)(i + ky)) % kInSlots) * (C::kInSlot >> 4);
          a_lo[ky][0] = (lbo << 16) + slot_lo;
          if (KIN == 4) a_lo[ky][KIN / 2 - 1] = ((((s_base + C::kOffZero) >> 4) - slot_lo - 2u * lbo) << 16) + slot_lo + 2u * lbo;
        }
        if (leader) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int ky = 0; ky < 5; ++ky)
#pragma unroll
              for (int ks = 0; ks < KIN / 2; ++ks)
                umma_bf16(tmem_base + acc * 2u * N1 + (uint32_t)(h * N1),
                          ((uint64_t)desc_hi << 32) | (a_lo[ky][ks] + (uint32_t)h * 128u),
                          ((uint64_t)desc_hi << 32) | (b_lo + (uint32_t)ky * slab + (uint32_t)ks * 2u * N1), idesc, (ky | ks) == 0 ? 0u : 1u);
          umma_commit(bar_a1full + 8u * acc);
          umma_commit(bar_in_empty + 8u * ((in_base + (uint32_t)i) % kInSlots));   // input row i: last reader done
          if (i == 2 * ru)
            for (int r = 1; r <= 4; ++r) umma_commit(bar_in_empty + 8u * ((in_base + (uint32_t)(i + r)) % kInSlots));
        }
        __syncwarp();
      }
      in_base += (uint32_t)(2 * ru + 5);
    }
  } else if (warp == W_MMA2) {
    // ===================================================================== MMA issuer, stride-2 conv(s): output row k of the strip
    // reads intermediate rows 2k .. 2k + 2 of the strip
    const bool leader = elect_one();
    constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N2 >> 3) << 17) | ((128u >> 4) << 24);
    constexpr uint32_t lbo = (uint32_t)kMidPos;            // intermediate chunks (16 B units)
    constexpr uint32_t slab = 2u * N2;                     // one tap's weights (16 B units)
    mbar_wait(bar_w, 0);
    tc_fence_after();
    const uint32_t b_lo = ((uint32_t)N2 << 16) + ((s_base + C::W1) >> 4);
    const uint32_t a_mid = (lbo << 16) + ((s_base + C::kOffMid) >> 4);
    uint32_t mid_base = 0, waited = 0, cnt = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int img = u / strips, y0 = (u - img * strips) * R, ru = min(R, kW2 - y0);
      for (int k = 0; k < ru; ++k, ++cnt) {
        while (waited < mid_base + (uint32_t)(2 * k + 3)) {
          mbar_wait(bar_mid_ready + 8u * (waited % kMidSlots), (waited / kMidSlots) & 1u);
          ++waited;
        }
        const uint32_t acc = cnt & 1u;
        mbar_wait(bar_a2empty + 8u * acc, ((cnt >> 1) & 1u) ^ 1u);
        tc_fence_after();
        uint32_t a_lo[3];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) a_lo[ky] = a_mid + ((mid_base + (uint32_t)(2 * k + ky)) % kMidSlots) * (C::kMidSlot >> 4);
        if (leader) {
#pragma unroll
          for (int l = 0; l < NL2; ++l)      // layer l reads intermediate chunks 2l, 2l + 1 and its own weights
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
              for (int kx = 0; kx < 3; ++kx) {
                const uint32_t off = kx == 0 ? 0u : (kx == 1 ? 129u : 1u);
                umma_bf16(tmem_base + 4u * N1 + acc * 32u + (uint32_t)(l * N2),
                          ((uint64_t)desc_hi << 32) | (a_lo[ky] + off + (uint32_t)l * 2u * lbo),
                          ((uint64_t)desc_hi << 32) | (b_lo + (uint32_t)l * (C::W2 >> 4) + (uint32_t)(ky * 3 + kx) * slab), idesc,
                          (ky | kx) == 0 ? 0u : 1u);
              }
          umma_commit(bar_a2full + 8u * acc);
          umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)(2 * k)) % kMidSlots));       // rows 2k, 2k + 1: last reader done
          umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)(2 * k + 1)) % kMidSlots));
          if (k == ru - 1) umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)(2 * k + 2)) % kMidSlots));
        }
        __syncwarp();
      }
      mid_base += (uint32_t)(2 * ru + 1);
    }
  } else {
    // ===================================================================== epilogue
    const int quad = warp & 3, m = quad * 32 + lane;
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    uint32_t cnt = 0;   // intermediate rows (warps 0-15) or output rows (warps 16-23) of this CTA so far
    if (warp < 16) {
      // warps 0-15: group (warp >> 3) takes every other row, warp quad (warp >> 2) & 1 its half h; pixel x = 128 h + m has the parity
      // of m: position in the O' / E halves of each chunk
      const uint32_t group = (uint32_t)(warp >> 3), h = (uint32_t)((warp >> 2) & 1);
      const int pos = ((m & 1) ? (m + 1) >> 1 : 129 + (m >> 1)) + 64 * (int)h;
      for (int u = blockIdx.x; u < units; u += gridDim.x) {
        const int img = u / strips, y0 = (u - img * strips) * R, ru = min(R, kW2 - y0);
        (void)img;
        for (int i = 0; i <= 2 * ru; ++i, ++cnt) {
          if ((cnt & 1u) != group) continue;
          mbar_wait(bar_a1full + 8u * group, (cnt >> 1) & 1u);
          tc_fence_after();
          float v[N1];
          tmem_ld<N1>(tmem_base + lane_off + group * 2u * N1 + h * N1, v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(bar_a1empty + 8u * group);
          const bool inside = 2 * y0 - 1 + i >= 0;   // row -1 is the stride-2 conv's zero padding
          uint4 val[KMID];
#pragma unroll
          for (int c = 0; c < KMID; ++c) {
            uint32_t pk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int col = c * 8 + 2 * e;
              pk[e] = inside ? pack_elu(v[col] + s_bias[col], v[col + 1] + s_bias[col + 1]) : 0u;
            }
            val[c] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
          const uint32_t slot = cnt % kMidSlots;
          mbar_wait(bar_mid_free + 8u * slot, ((cnt / kMidSlots) & 1u) ^ 1u);
          uint8_t* base = smem + C::kOffMid + slot * C::kMidSlot + pos * 16;
#pragma unroll
          for (int c = 0; c < KMID; ++c) *reinterpret_cast<uint4*>(base + c * kMidPos * 16) = val[c];
          fence_proxy_async();
          mbar_arrive(bar_mid_ready + 8u * slot);
        }
      }
    } else {
      const uint32_t group = (uint32_t)((warp >> 2) & 1);   // warps 16-19 / 20-23: every other output row
      for (int u = blockIdx.x; u < units; u += gridDim.x) {
        const int img = u / strips, y0 = (u - img * strips) * R, ru = min(R, kW2 - y0);
        for (int k = 0; k < ru; ++k, ++cnt) {
          if ((cnt & 1u) != group) continue;
          mbar_wait(bar_a2full + 8u * group, (cnt >> 1) & 1u);
          tc_fence_after();
          float v[32];
          tmem_ld<32>(tmem_base + lane_off + 4u * N1 + group * 32u, v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(bar_a2empty + 8u * group);
          const size_t pos = (size_t)(y0 + k + p.out_border) * p.out_pitch + m + p.out_border;
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {   // column chunk cc: chunk cc % (N2 / 8) of stride-2 layer cc / (N2 / 8)
            const int l = cc / (N2 / 8), c = cc % (N2 / 8);
            uint32_t pk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int col = cc * 8 + 2 * e;
              pk[e] = pack_elu(v[col] + s_bias[64 + col], v[col + 1] + s_bias[64 + col + 1]);
            }
            __nv_bfloat16* out = l ? p.out3 : p.out2;
            const int chunks = l ? p.out3_chunks : p.out2_chunks;
            *reinterpret_cast<uint4*>(out + (((size_t)img * chunks + c) * p.out_plane + pos) * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.timeline && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    atomicMax(reinterpret_cast<unsigned long long*>(p.timeline) + 1, gt);
  }
  if (warp == W_MMA1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- host
typedef CUresult (*PFN_encodeTiledStem)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 5-D map over a plain chunked buffer whose rows are 256 pixels: {position in a half row (8-byte units), half, plane row, chunk, image},
// origin at pixel x = 0 of plane row 0.  One box = one whole image row of box_chunks chunks, [chunk][256 positions][16 B] in shared memory;
// rows outside the zero-bordered plane are filled with zeros by the TMA unit.
static int make_stem_map(CUtensorMap* map, const TcBuf& b, int box_chunks) {
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled is unavailable (driver entry point lookup failed)");
    return HV_ERR_CUDA;
  }
  PFN_encodeTiledStem enc = reinterpret_cast<PFN_encodeTiledStem>(ptr);
  const cuuint64_t plane_b = (cuuint64_t)b.plane() * 16;
  cuuint64_t dims[5] = {(cuuint64_t)kW, 2, (cuuint64_t)b.rows(), (cuuint64_t)b.chunks, (cuuint64_t)b.n};
  cuuint64_t strides[4] = {(cuuint64_t)kW / 2 * 16, (cuuint64_t)b.pitch() * 16, plane_b, plane_b * b.image_chunks()};
  cuuint32_t box[5] = {(cuuint32_t)kW, 2, 1, (cuuint32_t)box_chunks, 1};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, b.ptr + (size_t)b.border * 8, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("stem: cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return HV_ERR_CUDA; }
  return HV_OK;
}

int tc_stem_setup(TcStem& s, const TcConv& conv1, const TcConv& down, const TcConv* down2, int n_images) {
  const TcBuf& in = conv1.src[0].buf;
  const bool fine = down2 != nullptr;
  const int kin = fine ? 4 : 2, n1 = fine ? 32 : 16, n2 = fine ? 16 : 32;
  HV_CHECK_ARG(conv1.nsrc == 1 && conv1.k == 5 && conv1.stride == 1 && conv1.dil == 1 && conv1.src[0].kxpack && conv1.n_pad == n1 &&
                   in.chunks == kin && !in.s2d && in.xp == 1 && in.h == kW && in.w == kW && in.border == 2,
               "tc_stem: the first layer must be a kx-packed 5x5 conv over 256 x 256 (%d chunks in, %d filters)", kin, n1);
  HV_CHECK_ARG(conv1.p.out_mode == TC_OUT_CHUNKED_S2D && conv1.p.act == HV_ACT_ELU && conv1.p.out_nchunks == n1 / 8,
               "tc_stem: the first layer must be an ELU conv writing a space-to-depth buffer");
  const TcConv* downs[2] = {&down, down2};
  for (int l = 0; l < (fine ? 2 : 1); ++l) {
    const TcConv& d = *downs[l];
    const TcBuf& b = d.src[0].buf;
    HV_CHECK_ARG(d.nsrc == 1 && d.stride == 2 && d.k == 3 && d.n_pad == n2 && b.s2d && b.chunks == 2 && b.h == kW && b.w == kW &&
                     b.ptr == conv1.p.out + (size_t)2 * l * conv1.p.out_plane * 8,
                 "tc_stem: stride-2 layer %d must read chunks %d-%d of the first layer's output", l, 2 * l, 2 * l + 1);
    HV_CHECK_ARG(d.p.out_mode == TC_OUT_CHUNKED && d.p.out_xp == 1 && d.p.act == HV_ACT_ELU && d.p.out_chunk_off == 0 &&
                     d.p.out_nchunks == n2 / 8 && d.p.out_pitch == kW2 + 1 && d.p.out_border == 1 && d.p.out_plane == down.p.out_plane,
                 "tc_stem: stride-2 layer %d must be an ELU conv writing a plain 128 x 128 chunked buffer", l);
  }
  HV_CHECK_ARG(conv1.p.w_bytes == 5u * kin * n1 * 16u && down.p.w_bytes == 9u * 2u * n2 * 16u && (!fine || down2->p.w_bytes == down.p.w_bytes),
               "tc_stem: unexpected packed weight sizes");
  s.p = TcStemParams();
  s.fine = fine;
  int rc = make_stem_map(&s.p.map_in, in, fine ? StemCfg<true>::KLOAD : StemCfg<false>::KLOAD);
  if (rc) return rc;
  s.p.w1 = conv1.w_packed; s.p.w2 = down.w_packed; s.p.w3 = fine ? down2->w_packed : nullptr;
  s.p.bias1 = conv1.bias_pad; s.p.bias2 = down.bias_pad; s.p.bias3 = fine ? down2->bias_pad : nullptr;
  s.p.out2 = down.p.out; s.p.out2_chunks = down.p.out_chunks_total;
  s.p.out3 = fine ? down2->p.out : nullptr; s.p.out3_chunks = fine ? down2->p.out_chunks_total : 0;
  s.p.out_pitch = down.p.out_pitch; s.p.out_border = down.p.out_border; s.p.out_plane = down.p.out_plane;
  tc_stem_set_batch(s, n_images);
  return HV_OK;
}

void tc_stem_set_batch(TcStem& s, int n_images) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  // one wave: (images) x (strips) units on the SMs; each strip recomputes one 5x5 conv row of the strip above it
  const int want_strips = max(1, min(kW2, sms / n_images));
  const int rows = (kW2 + want_strips - 1) / want_strips;
  s.p.n = n_images;
  s.p.rows_per_unit = rows;
  s.p.strips = (kW2 + rows - 1) / rows;
  s.p.units = n_images * s.p.strips;
  s.grid = min(s.p.units, sms);
}

template <bool FINE>
static int stem_launch(const TcStem& s, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    HV_CUDA(cudaFuncSetAttribute(stem_tc_kernel<FINE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)StemCfg<FINE>::kSmem));
    configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(s.grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = StemCfg<FINE>::kSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TcStemParams q = s.p;
  q.timeline = tc_timeline_next();
  HV_CUDA(cudaLaunchKernelEx(&cfg, stem_tc_kernel<FINE>, q));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

int tc_stem_launch(const TcStem& s, cudaStream_t st) { return s.fine ? stem_launch<true>(s, st) : stem_launch<false>(s, st); }

}  // namespace hv
