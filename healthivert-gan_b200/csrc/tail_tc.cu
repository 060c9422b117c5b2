// Fused thin tail of a generator stage at 256 x 256: a 16 -> 8 3x3 conv (ELU) followed by the dual 3x3 output heads (clamp / sigmoid)
// in ONE persistent launch.  Coarse stage: conv16 -> conv17 | conv18 (models/inpaint_networks.py:112-116); fine stage: allconv16 ->
// allconv17 | allconv18 (:225-231, the heads also read x_stage1 as a ninth input channel).  The 8-channel intermediate lives only in
// shared memory: per stage it saves one launch ramp, the 8.6 MB bf16 write of the intermediate and its three band re-reads from L2.
//
// Work unit = (image pair, strip of R output rows).  An accumulator tile is M = 128 rows = two "streams" x 64 positions: stream s is
// image 2 * pair + s, position q holds the 4 x-phase pixels 4q .. 4q + 3 (N = 4 phases x channels, as in conv_tc's x-phase instances),
// so one tile is one image row of two images.  The two images share every row coordinate, so the TMA box of a row carries both
// (tensor-map dims {position, image, row, chunk, phase}) and rows outside the image are zero-filled by the TMA unit.
//
// Shared-memory row image ("slot"): six views of the 4 x-phase planes, view v = the operand of the x-phase tap view v of conv_tc's
// issue_xp4: phase (v + 3) & 3 at position q - 1 / q / q / q / q / q + 1.  Views 0 and 5 are the two shifted copies; with them every
// MMA reads 128 CONTIGUOUS rows (stream 0 then stream 1), no zero gap column is needed between the streams.
//   input slot   [view 6][chunk 2][stream 2][64 pos] x 16 B = 24 KB   (K chunks 2 KB apart)
//   middle slot  [chunk 2][view 6][stream 2][64 pos] x 16 B = 24 KB   (chunk 0: the conv output, written by the epilogue;
//                                                                       chunk 1: the heads' second input chunk, brought by TMA)
// Budget (227 KB): weights 18 KB (conv, N 32 x 18 views x 2 chunks) + 9 KB (heads, N 16) + 4 input slots 96 KB + 4 middle slots 96 KB
// + barriers / bias 1 KB + head-1 rows for the kx packing 4 KB = 224 KB.  One CTA per SM.
//
// Row pipeline of a unit (rows relative to the strip start y0, Ru = rows of this strip):
//   producers: one warp for input rows -2 .. Ru+1 (one TMA box for views 1-4, two for the shifted views), one warp for the heads'
//              second chunk of middle rows -1 .. Ru (so that input rows never wait for the heads to free a middle slot)
//   MMA      : one issuer warp per layer: the conv of middle row j (reads input rows j-1 .. j+1), the heads of output row k (reads
//              middle rows k-1 .. k+1, as soon as their epilogue and TMA are done); each layer has two TMEM accumulators
//   epilogue : warps 0-7 (two groups, alternate rows): TMEM -> bias + ELU -> bf16 -> middle slot (zero outside the image),
//              fence.proxy.async, arrive; warps 8-15 (two groups): TMEM -> clamp / sigmoid -> fp32 heads (+ bf16 aux copy, and in
//              the coarse stage head 1 kx-packed for the fine network's 5x5 input conv, which replaces a packing launch)
// Every accumulator sees exactly the MMA sequence of the per-layer instance (tap rows, then the six views, K = 16 each) and the
// epilogue arithmetic of conv_tc_kernel, so the fused stage equals the two per-layer launches bit for bit.
#include <string.h>
#include "hv_common.cuh"
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace hv {

namespace {

constexpr int kMidN = 32, kHeadN = 16;                // accumulator columns: 4 phases x 8 channels / 4 phases x (2 heads + 2 pad)
constexpr uint32_t kWMid = 3u * 6u * 2u * kMidN * 16u;    // 18432 B
constexpr uint32_t kWHead = 3u * 6u * 2u * kHeadN * 16u;  // 9216 B
constexpr uint32_t kSlot = 6u * 2u * 2u * 64u * 16u;      // 24576 B
constexpr int kSlots = 4;
constexpr uint32_t kOffIn = kWMid + kWHead;               // 27648
constexpr uint32_t kOffMid = kOffIn + kSlots * kSlot;
constexpr uint32_t kOffBar = kOffMid + kSlots * kSlot;
constexpr uint32_t kOffKx = kOffBar + 1024;               // heads epilogue: one fp32 row of head 1 per (group, stream) + 4 zeros each side
constexpr int kKxRow = 264;
constexpr uint32_t kSmem = kOffKx + 2u * 2u * kKxRow * 4u;
static_assert(kSmem <= 227u * 1024u, "tail kernel shared memory");
constexpr uint32_t kInTx = kSlot;                 // views 0-5 of both chunks
constexpr uint32_t kAuxTx = kSlot / 2;            // views 0-5 of chunk 1
constexpr int kThreads = 20 * 32;                 // 16 epilogue warps, input producer, conv / heads MMA issuers, heads' chunk producer
constexpr int kTmemCols = 128;                    // 2 x 32 (conv) + 2 x 16 (heads)

__device__ __forceinline__ float elu_fast(float x) {   // == act_fast<HV_ACT_ELU> of conv_tc.cu
  if (x > 0.f) return x;
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y - 1.f;
}

// 18 MMAs of one 3x3 x-phase layer in issue_xp4's order (tap row, view); a_lo[ky] = descriptor lo word of view 0 of the row
template <int N>
__device__ __forceinline__ void issue_rows(bool leader, uint32_t d_tmem, const uint32_t (&a_lo)[3], uint32_t a_view, uint32_t b_lo) {
  constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
  constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
  constexpr uint32_t slab = 2u * N;   // one view's weights, 16 B units
  if (leader) {
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int v = 0; v < 6; ++v)
        umma_bf16(d_tmem, ((uint64_t)desc_hi << 32) | (a_lo[ky] + (uint32_t)v * a_view),
                  ((uint64_t)desc_hi << 32) | (b_lo + (uint32_t)(ky * 6 + v) * slab), idesc, (ky | v) == 0 ? 0u : 1u);
  }
}

}  // namespace

__global__ void __launch_bounds__(kThreads, 1) tail_tc_kernel(const __grid_constant__ TcTailParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int W_PRODUCER = 16, W_MMA = 17, W_HEADS = 18, W_AUX = 19;
  const uint32_t s_base = smem_u32(smem);
  const uint32_t bars = s_base + kOffBar;
  // barriers (8 B each)
  const uint32_t bar_in_full = bars, bar_in_empty = bars + 8 * kSlots;
  const uint32_t bar_mid_ready = bars + 16 * kSlots, bar_mid_free = bars + 24 * kSlots;
  const uint32_t bar_mfull = bars + 32 * kSlots, bar_mempty = bar_mfull + 16, bar_hfull = bar_mfull + 32, bar_hempty = bar_mfull + 48;
  const uint32_t bar_w = bar_mfull + 64;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 256);
  float* s_bias = reinterpret_cast<float*>(smem + kOffBar + 512);   // [0, 32): conv, [32, 48): heads

  if (p.timeline && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    atomicMin(reinterpret_cast<unsigned long long*>(p.timeline), gt);
  }
  if ((warp == W_PRODUCER || warp == W_AUX) && lane == 0) {
    for (int i = 0; i < 4; ++i) asm volatile("prefetch.tensormap [%0];" ::"l"(&p.maps[i]) : "memory");
  }
  if (warp == W_MMA) {
    if (lane == 0) {
      for (int i = 0; i < kSlots; ++i) {
        mbar_init(bar_in_full + 8u * i, 1);
        mbar_init(bar_in_empty + 8u * i, 1);
        mbar_init(bar_mid_ready + 8u * i, 128 + 1);   // epilogue threads + the producer's expect_tx of the heads' second chunk
        mbar_init(bar_mid_free + 8u * i, 1);
      }
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_mfull + 8u * i, 1); mbar_init(bar_mempty + 8u * i, 128);
        mbar_init(bar_hfull + 8u * i, 1); mbar_init(bar_hempty + 8u * i, 128);
      }
      mbar_init(bar_w, 1);
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x < kMidN) s_bias[threadIdx.x] = __ldg(p.bias_mid + threadIdx.x);
  else if (threadIdx.x < kMidN + kHeadN) s_bias[threadIdx.x] = __ldg(p.bias_head + threadIdx.x - kMidN);
  // the zero ends of the two shifted views of the conv output (view 0 at q = 0, view 5 at q = 63): the epilogue never writes them
  if (threadIdx.x < kSlots * 2 * 2) {
    const int slot = threadIdx.x >> 2, s = (threadIdx.x >> 1) & 1, e = threadIdx.x & 1;
    *reinterpret_cast<uint4*>(smem + kOffMid + slot * kSlot + (e ? 5 * 2048 + s * 1024 + 63 * 16 : s * 1024)) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + 2 * 2 * 8) {   // the zero ends of the head-1 rows (kx-packed copy, see below)
    const int r = (threadIdx.x - 64) >> 3, e = (threadIdx.x - 64) & 7;
    reinterpret_cast<float*>(smem + kOffKx)[r * kKxRow + (e < 4 ? e : kKxRow - 8 + e)] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int R = p.rows_per_unit, strips = p.strips, units = p.units, h = p.h;

  if (warp == W_PRODUCER || warp == W_AUX) {
    // ===================================================================== TMA producers: input rows (W_PRODUCER) and the heads' second
    // chunk of the middle rows (W_AUX).  Two warps, so that an input row never waits behind a middle slot that the heads still read.
    const bool leader = elect_one();
    const bool in_role = warp == W_PRODUCER;
    if (leader && in_role) {
      mbar_expect_tx(bar_w, kWMid + kWHead);
      bulk_load(s_base, p.w_mid, kWMid, bar_w);
      bulk_load(s_base + kWMid, p.w_head, kWHead, bar_w);
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");   // the input rows are the previous kernel's output
    uint32_t in_seq = 0, mid_seq = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int pair = u / strips, y0 = (u - pair * strips) * R, ru = min(R, h - y0), img = 2 * pair;
      for (int i = -2; i <= ru + 1; ++i) {
        if (in_role) {
          const uint32_t slot = in_seq % kSlots, par = (in_seq / kSlots) & 1u;
          mbar_wait(bar_in_empty + 8u * slot, par ^ 1u);
          if (leader) {
            const uint32_t fb = bar_in_full + 8u * slot, dst = s_base + kOffIn + slot * kSlot;
            const int row = y0 + i + 1;   // row coordinate of the zero-bordered plane
            mbar_expect_tx(fb, kInTx);
            tma_load_5d(dst + 4096u, &p.maps[0], fb, 2, img, row, 0, 0);        // views 1-4: phases 0-3 at q
            tma_load_5d(dst, &p.maps[1], fb, 0, img, row, 0, 3);                // view 0: phase 3 at q - 1
            tma_load_5d(dst + 5u * 4096u, &p.maps[1], fb, 4, img, row, 0, 0);   // view 5: phase 0 at q + 1
          }
          ++in_seq;
        }
        const int j = i - 1;   // middle row whose conv becomes computable with this input row
        if (!in_role && j >= -1) {
          const uint32_t slot = mid_seq % kSlots, par = (mid_seq / kSlots) & 1u;
          mbar_wait(bar_mid_free + 8u * slot, par ^ 1u);
          if (leader) {
            const uint32_t fb = bar_mid_ready + 8u * slot, dst = s_base + kOffMid + slot * kSlot + 12288u;   // chunk 1
            const int row = y0 + j + 1;
            mbar_expect_tx(fb, kAuxTx);
            tma_load_5d(dst + 2048u, &p.maps[2], fb, 2, img, row, 1, 0);
            tma_load_5d(dst, &p.maps[3], fb, 0, img, row, 1, 3);
            tma_load_5d(dst + 5u * 2048u, &p.maps[3], fb, 4, img, row, 1, 0);
          }
          ++mid_seq;
        }
      }
    }
  } else if (warp == W_MMA || warp == W_HEADS) {
    // ===================================================================== MMA issuers: the conv and the heads have one warp each, so
    // that their MMA streams interleave on the tensor pipe (a single issuer is bound by ~60 cycles per warp-uniform MMA issue); they
    // are coupled only through the middle-slot barriers
    const bool leader = elect_one();
    const bool conv_role = warp == W_MMA;
    mbar_wait(bar_w, 0);
    tc_fence_after();
    const uint32_t b_mid = ((uint32_t)kMidN << 16) + (s_base >> 4);
    const uint32_t b_head = ((uint32_t)kHeadN << 16) + ((s_base + kWMid) >> 4);
    // A: conv reads input slots (views 4 KB apart, K chunks 2 KB apart), heads read middle slots (views 2 KB, chunks 12 KB apart)
    const uint32_t a_in = ((2048u >> 4) << 16) + ((s_base + kOffIn) >> 4);
    const uint32_t a_mid = ((12288u >> 4) << 16) + ((s_base + kOffMid) >> 4);
    uint32_t in_base = 0, mid_base = 0, waited = 0, cnt = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int pair = u / strips, y0 = (u - pair * strips) * R, ru = min(R, h - y0);
      if (conv_role) {
        for (int j = -1; j <= ru; ++j, ++cnt) {
          // conv of middle row j: input rows j-1 .. j+1 = sequence numbers in_base + j + 1 .. + 3
          while (waited < in_base + (uint32_t)(j + 4)) {
            mbar_wait(bar_in_full + 8u * (waited % kSlots), (waited / kSlots) & 1u);
            ++waited;
          }
          const uint32_t acc = cnt & 1u;
          mbar_wait(bar_mempty + 8u * acc, ((cnt >> 1) & 1u) ^ 1u);
          tc_fence_after();
          uint32_t a_lo[3];
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) a_lo[ky] = a_in + ((in_base + (uint32_t)(j + 1 + ky)) % kSlots) * (kSlot >> 4);
          issue_rows<kMidN>(leader, tmem_base + acc * kMidN, a_lo, 4096u >> 4, b_mid);
          if (leader) {
            umma_commit(bar_mfull + 8u * acc);
            umma_commit(bar_in_empty + 8u * ((in_base + (uint32_t)(j + 1)) % kSlots));     // input row j-1: last reader done
            if (j == ru) {
              umma_commit(bar_in_empty + 8u * ((in_base + (uint32_t)(j + 2)) % kSlots));
              umma_commit(bar_in_empty + 8u * ((in_base + (uint32_t)(j + 3)) % kSlots));
            }
          }
          __syncwarp();
        }
      } else {
        for (int k = 0; k < ru; ++k, ++cnt) {
          // heads of output row k: middle rows k-1 .. k+1 = sequence numbers mid_base + k .. + 2
          while (waited < mid_base + (uint32_t)(k + 3)) {
            mbar_wait(bar_mid_ready + 8u * (waited % kSlots), (waited / kSlots) & 1u);
            ++waited;
          }
          const uint32_t acc = cnt & 1u;
          mbar_wait(bar_hempty + 8u * acc, ((cnt >> 1) & 1u) ^ 1u);
          tc_fence_after();
          uint32_t a_lo[3];
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) a_lo[ky] = a_mid + ((mid_base + (uint32_t)(k + ky)) % kSlots) * (kSlot >> 4);
          issue_rows<kHeadN>(leader, tmem_base + 2 * kMidN + acc * kHeadN, a_lo, 2048u >> 4, b_head);
          if (leader) {
            umma_commit(bar_hfull + 8u * acc);
            umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)k) % kSlots));          // middle row k-1: last reader done
            if (k == ru - 1) {
              umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)(k + 1)) % kSlots));
              umma_commit(bar_mid_free + 8u * ((mid_base + (uint32_t)(k + 2)) % kSlots));
            }
          }
          __syncwarp();
        }
      }
      in_base += (uint32_t)(ru + 4);
      mid_base += (uint32_t)(ru + 2);
    }
  } else {
    // ===================================================================== epilogue
    const int quad = warp & 3, m = quad * 32 + lane, s = m >> 6, q = m & 63;
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    const bool mid_role = warp < 8;
    const uint32_t group = (uint32_t)((warp >> 2) & 1);
    uint32_t cnt = 0;   // middle rows (conv role) or output rows (heads role) of this CTA so far
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int pair = u / strips, y0 = (u - pair * strips) * R, ru = min(R, h - y0);
      const int img = 2 * pair + s;
      if (mid_role) {
        for (int j = -1; j <= ru; ++j, ++cnt) {
          if ((cnt & 1u) != group) continue;
          mbar_wait(bar_mfull + 8u * group, (cnt >> 1) & 1u);
          tc_fence_after();
          float v[kMidN];
          tmem_ld<32>(tmem_base + lane_off + group * kMidN, v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(bar_mempty + 8u * group);
          const int y = y0 + j;
          const bool inside = y >= 0 && y < h;   // rows outside the image are the next conv's zero padding
          uint4 val[4];
#pragma unroll
          for (int ph = 0; ph < 4; ++ph) {
            uint32_t pk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int col = ph * 8 + 2 * e;
              __nv_bfloat162 hv2 = __floats2bfloat162_rn(elu_fast(v[col] + s_bias[col]), elu_fast(v[col + 1] + s_bias[col + 1]));
              pk[e] = inside ? *reinterpret_cast<uint32_t*>(&hv2) : 0u;
            }
            val[ph] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
          const uint32_t slot = cnt % kSlots;
          mbar_wait(bar_mid_free + 8u * slot, ((cnt / kSlots) & 1u) ^ 1u);
          uint8_t* base = smem + kOffMid + slot * kSlot + s * 1024 + q * 16;   // chunk 0, view 0, (stream, q)
#pragma unroll
          for (int ph = 0; ph < 4; ++ph) *reinterpret_cast<uint4*>(base + (ph + 1) * 2048) = val[ph];
          if (q < 63) *reinterpret_cast<uint4*>(base + 16) = val[3];               // view 0 at q + 1 = phase 3 at q
          if (q > 0) *reinterpret_cast<uint4*>(base + 5 * 2048 - 16) = val[0];     // view 5 at q - 1 = phase 0 at q
          fence_proxy_async();
          mbar_arrive(bar_mid_ready + 8u * slot);
        }
      } else {
        for (int k = 0; k < ru; ++k, ++cnt) {
          if ((cnt & 1u) != group) continue;
          mbar_wait(bar_hfull + 8u * group, (cnt >> 1) & 1u);
          tc_fence_after();
          float v[kHeadN];
          tmem_ld<16>(tmem_base + lane_off + 2 * kMidN + group * kHeadN, v);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(bar_hempty + 8u * group);
          const bool live = img < p.n;   // the second image of the last pair of an odd batch does not exist
          const int y = y0 + k;
          float seg[4];
#pragma unroll
          for (int jx = 0; jx < 4; ++jx) {   // columns jx * 4 + {0, 1} = the two heads of pixel 4 q + jx
            const int x = 4 * q + jx;
            const float a0 = fminf(fmaxf(v[jx * 4] + s_bias[kMidN + jx * 4], -1.f), 1.f);
            const float a1 = 1.f / (1.f + __expf(-(v[jx * 4 + 1] + s_bias[kMidN + jx * 4 + 1])));
            seg[jx] = a1;
            if (!live) continue;
            const size_t pix = ((size_t)img * h + y) * p.w_img + x;
            p.head0[pix] = a0;
            p.head1[pix] = a1;
            if (p.aux0.ptr) {
              const TcAux& a = p.aux0;
              const size_t pos = (size_t)jx * a.sub_plane + (size_t)(y + a.border) * a.pitch + q + a.border;
              a.ptr[(((size_t)img * a.chunks + a.chunk) * a.plane + pos) * 8 + a.channel] = __float2bfloat16(a0);
            }
          }
          if (p.kx.ptr) {
            // head 1 kx-packed for the next stage's 5x5 input conv (what tc_pack_kx(k = 5, dil = 1) writes into channels 0-7 of chunk
            // kx_chunk): channel kx of pixel x = bf16(head1(x + kx - 2)), zero outside the row and in channels 5-7.  The row goes through
            // shared memory (the neighbours x - 2 .. x + 5 belong to other threads), then every thread stores 4 whole 16-byte positions.
            float* row = reinterpret_cast<float*>(smem + kOffKx) + (group * 2 + s) * kKxRow;
            *reinterpret_cast<float4*>(row + 4 + 4 * q) = make_float4(seg[0], seg[1], seg[2], seg[3]);
            asm volatile("bar.sync %0, 128;" ::"r"(1 + (int)group) : "memory");
            if (live) {
              __nv_bfloat16* dst = p.kx.ptr + p.kx.chunk_base(img, p.kx_chunk) + p.kx.pos(y, 4 * q) * 8;
#pragma unroll
              for (int jx = 0; jx < 4; ++jx) {
                const float* r = row + 2 + 4 * q + jx;   // r[kx] = head1(4 q + jx + kx - 2)
                __nv_bfloat162 c01 = __floats2bfloat162_rn(r[0], r[1]), c23 = __floats2bfloat162_rn(r[2], r[3]);
                __nv_bfloat162 c4 = __floats2bfloat162_rn(r[4], 0.f);
                *reinterpret_cast<uint4*>(dst + jx * 8) = make_uint4(*reinterpret_cast<uint32_t*>(&c01), *reinterpret_cast<uint32_t*>(&c23),
                                                                     *reinterpret_cast<uint32_t*>(&c4), 0u);
              }
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + (int)group) : "memory");   // the row buffer is reused by this group's next row
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
  if (warp == W_MMA) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- host
typedef CUresult (*PFN_encodeTiledTail)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 5-D map over an x-phase buffer: {position in the row (8-byte units), image, row, chunk, phase}.  Positions past the row and rows
// past the zero-bordered plane are out of bounds: the TMA unit fills them with zeros (the conv padding).
static int make_tail_map(CUtensorMap* map, const TcBuf& b, int box_chunks, int box_phases) {
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled is unavailable (driver entry point lookup failed)");
    return HV_ERR_CUDA;
  }
  PFN_encodeTiledTail enc = reinterpret_cast<PFN_encodeTiledTail>(ptr);
  const cuuint64_t sub_b = (cuuint64_t)b.sub_plane() * 16, plane_b = (cuuint64_t)b.plane() * 16;
  cuuint64_t dims[5] = {(cuuint64_t)b.pitch() * 2, (cuuint64_t)b.n, (cuuint64_t)b.rows(), (cuuint64_t)b.image_chunks(), 4};
  cuuint64_t strides[4] = {plane_b * b.image_chunks(), (cuuint64_t)b.pitch() * 16, plane_b, sub_b};
  cuuint32_t box[5] = {128, 2, 1, (cuuint32_t)box_chunks, (cuuint32_t)box_phases};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, b.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("tail: cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return HV_ERR_CUDA; }
  return HV_OK;
}

int tc_tail_setup(TcTail& t, const TcConv& mid, const TcConv& heads, int n_images) {
  const TcBuf& in = mid.src[0].buf;
  const TcBuf& hb = heads.src[0].buf;
  HV_CHECK_ARG(mid.nsrc == 1 && mid.k == 3 && mid.dil == 1 && mid.p.in_xp == 4 && mid.n_pad == kMidN && in.chunks == 2 && in.sub_w() == 64,
               "tc_tail: the first layer must be a 16 -> 8 x-phase 3x3 conv over 256-pixel rows");
  HV_CHECK_ARG(mid.p.out_mode == TC_OUT_CHUNKED && mid.p.act == HV_ACT_ELU, "tc_tail: the first layer must be a chunked ELU conv");
  HV_CHECK_ARG(heads.nsrc == 1 && heads.k == 3 && heads.p.in_xp == 4 && heads.n_pad == kHeadN && heads.p.out_mode == TC_OUT_HEADS &&
                   hb.chunks == 2 && hb.h == in.h && hb.w == in.w && hb.border == 1 && in.border == 1,
               "tc_tail: the second layer must be the dual heads over a 2-chunk x-phase buffer of the same geometry");
  HV_CHECK_ARG(mid.p.w_bytes == kWMid && heads.p.w_bytes == kWHead, "tc_tail: unexpected packed weight sizes");
  t.p = TcTailParams();
  int rc = make_tail_map(&t.p.maps[0], in, 2, 4);
  if (!rc) rc = make_tail_map(&t.p.maps[1], in, 2, 1);
  if (!rc) rc = make_tail_map(&t.p.maps[2], hb, 1, 4);
  if (!rc) rc = make_tail_map(&t.p.maps[3], hb, 1, 1);
  if (rc) return rc;
  t.p.w_mid = mid.w_packed; t.p.w_head = heads.w_packed;
  t.p.bias_mid = mid.bias_pad; t.p.bias_head = heads.bias_pad;
  t.p.h = in.h; t.p.w_img = in.w;
  t.p.aux0 = heads.p.aux0;
  tc_tail_set_batch(t, n_images);
  return HV_OK;
}

void tc_tail_set_batch(TcTail& t, int n_images) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  // one wave: (image pairs) x (strips) units on the SMs; each strip recomputes one conv row above and below it
  const int pairs = (n_images + 1) / 2, h = t.p.h;
  const int want_strips = max(1, min(h, sms / pairs));
  const int rows = (h + want_strips - 1) / want_strips;
  t.p.n = n_images;
  t.p.rows_per_unit = rows;
  t.p.strips = (h + rows - 1) / rows;
  t.p.units = pairs * t.p.strips;
  t.grid = min(t.p.units, sms);
}

void tc_tail_set_outputs(TcTail& t, float* head0, float* head1) { t.p.head0 = head0; t.p.head1 = head1; }

int tc_tail_set_kxpack(TcTail& t, const TcBuf* dst, int chunk) {
  if (!dst) { t.p.kx = TcBuf(); return HV_OK; }
  HV_CHECK_ARG(dst->ptr && dst->xp == 1 && !dst->s2d && dst->h == t.p.h && dst->w == t.p.w_img && chunk >= 0 && chunk < dst->image_chunks(),
               "tc_tail_set_kxpack: destination must be a plain chunked buffer of the heads' extent");
  t.p.kx = *dst;
  t.p.kx_chunk = chunk;
  return HV_OK;
}

int tc_tail_launch(const TcTail& t, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    HV_CUDA(cudaFuncSetAttribute(tail_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(t.grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TcTailParams q = t.p;
  q.timeline = tc_timeline_next();
  HV_CUDA(cudaLaunchKernelEx(&cfg, tail_tc_kernel, q));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

}  // namespace hv
