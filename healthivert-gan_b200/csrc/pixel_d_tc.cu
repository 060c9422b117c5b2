// Fused PixelDiscriminator (reference models/networks.py:604-753, netD='pixel'): three 1x1 convolutions at full resolution,
// 1 -> 64 + LeakyReLU, 64 -> 128 + norm + LeakyReLU, 128 -> 1, forward and backward, with the 64- and 128-channel maps kept on chip.
// Every pixel is independent, so pixels are flattened per sample into tiles of M = 128 rows (a tile never spans two samples; the last
// tile of a sample is ragged) and persistent CTAs take contiguous tile ranges.
//
// Precision (the tensor-core training mode's convention): the 64 -> 128 products run on tcgen05 with bf16 operands and fp32
// accumulation; the 1 -> 64 and 128 -> 1 layers, the norm, the LeakyReLUs and every reduction stay fp32 (the final cross-CTA sums in
// fp64).  Rounded to bf16: h1 and W2 in the forward, dh2, W2 and h1 in the backward.
//
// One CTA = 128 threads, thread m owns tile row (pixel) m and TMEM lane m.  Per tile:
//   h1 = lrelu(w1 x + b1) in registers -> bf16 -> shared memory (canonical K-major layout) -> 4 MMAs (K = 64) -> h2 [128 x 128] in TMEM
// The passes recompute h2 with the same MMA sequence, so every pass sees the same bits:
//   kStats   (batch / instance norm): per-channel sum and sum of squares of h2 (+ b2) - K, shifted by K = the CTA's first pixel of the
//              sample, so that a channel whose mean is large against its spread keeps its variance; the partials (count, K, sums) are
//              merged in fp64 with the pairwise (Chan et al.) update
//   kApply   : norm, LeakyReLU, w3 . a + b3 -> fp32 logit
//   kBwdSums : sum g a (dw3), sum g (db3), sum dz (dbeta), sum dz xhat (dgamma); dz = d(pre-LeakyReLU)
//   kBwdGrad : dh2 (bf16) -> dh1 = dh2 W2 (M = 128 pixels, N = 64, K = 128) and dW2 += dh2^T h1 (M = 128 channels, N = 64, K = the
//              tile's pixels, accumulated in TMEM over the CTA's tiles); dpre1 = dh1 lrelu'(pre1), dx = w1 . dpre1, dw1, db1, db2
// Per-channel sums over a tile's pixels: a transposing butterfly inside each warp (31 shuffles reduce 32 channels over 32 lanes, lane l
// ends with channel l), per-thread running sums across tiles, a fixed-order combine of the four warps and per-CTA partials in the
// workspace; small kernels then add the partials in a fixed order.  No float atomics: the same inputs give the same bits.
#include "hv_common.cuh"
#include "tc_ptx.cuh"

namespace hv {

namespace {

constexpr int kC1 = 64, kC2 = 128, kTile = 128, kThreads = 128;
constexpr int kNQ = 4;                 // per-channel quantities of the kStats / kBwdSums partials
constexpr int kTmemCols = 256;         // h2 [0, 128), dh1 [128, 192), dW2 [192, 256)
enum { kStats = 0, kApply = 1, kBwdSums = 2, kBwdGrad = 3 };
enum { kNormNone = 0, kNormBatch = 1, kNormInstance = 2 };

// shared memory (bytes).  Canonical no-swizzle K-major operands: element (row r, k) at (k / 8) * rows * 16 + r * 16 + (k % 8) * 2.
constexpr uint32_t kOffW2 = 0;                         // B of h2 = h1 W2^T:   rows c2 (128), K c1 (64)     16 KB
constexpr uint32_t kOffW2T = kOffW2 + 16384;           // B of dh1 = dh2 W2:   rows c1 (64),  K c2 (128)    16 KB
constexpr uint32_t kOffH1 = kOffW2T + 16384;           // A of h2:             rows pixel,    K c1          16 KB
constexpr uint32_t kOffH1T = kOffH1 + 16384;           // B of dW2:            rows c1,       K pixel       16 KB
constexpr uint32_t kOffDH2 = kOffH1T + 16384;          // A of dh1:            rows pixel,    K c2          32 KB
constexpr uint32_t kOffDH2T = kOffDH2 + 32768;         // A of dW2:            rows c2,       K pixel       32 KB
constexpr uint32_t kOffRed = kOffDH2T + 32768;         // [4 warps][kNQ][128] fp32                          8 KB
constexpr uint32_t kOffPar = kOffRed + 4 * kNQ * 128 * 4;   // parameters, fp32
// parameter block (floats): w1 b1 [64] each, w3 b2 gamma beta mean invstd s1 s2 shift [128] each
constexpr int kPW1 = 0, kPB1 = 64, kPW3 = 128, kPB2 = 256, kPG = 384, kPBeta = 512, kPMean = 640, kPInv = 768, kPS1 = 896, kPS2 = 1024,
              kPShift = 1152;
constexpr int kParFloats = 1280;
constexpr uint32_t kOffBar = kOffPar + kParFloats * 4;
constexpr uint32_t kSmem = kOffBar + 64;
static_assert(kSmem <= 227u * 1024u, "pixel discriminator shared memory");

constexpr uint32_t kIdescN128 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
constexpr uint32_t kIdescN64 = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

struct PixelDParams {
  const float *x, *w1, *b1, *w2, *b2, *gamma, *beta, *w3, *b3;
  const float *mean, *invstd;   // kApply / kBwd*: [C2] (batch) or [n * C2] (instance)
  const float *sums;            // kBwdGrad: [n][2][C2] sum dz, sum dz xhat (per sample; batch uses their totals)
  const float* dy;              // logit gradient
  float* y;                     // kApply: logits
  float* dx;                    // kBwdGrad: input gradient (may be null)
  float* part;                  // kStats: [grid][n][{sum, sum of squares, shift, count bits}][C2]; kBwdSums: [grid][n][kNQ][C2];
                                // kBwdGrad: [grid][2][C2]
  float* part_w2;               // kBwdGrad: [grid][C2][C1] (null: no parameter gradients)
  int n, hw, tiles_per_sample, tiles, norm;
  float slope;
  long long count;              // pixels per statistic: n * hw (batch) or hw (instance)
};

__device__ __forceinline__ float lrelu(float v, float s) { return v > 0.f ? v : s * v; }

// 32 channel values per lane -> lane l returns the sum over the warp's 32 lanes of channel l (v is consumed)
__device__ __forceinline__ float xreduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool up = (lane & w) != 0;
#pragma unroll
    for (int k = 0; k < w; ++k) {
      const float send = up ? v[k] : v[k + w];
      const float keep = up ? v[k + w] : v[k];
      v[k] = keep + __shfl_xor_sync(0xffffffffu, send, w);
    }
  }
  return v[0];
}

__device__ __forceinline__ void sts16(uint8_t* base, uint32_t off, const float (&v)[8]) {
  __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
  *reinterpret_cast<uint4*>(base + off) = make_uint4(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1),
                                                     *reinterpret_cast<uint32_t*>(&p2), *reinterpret_cast<uint32_t*>(&p3));
}

// K-major descriptor of an operand with `rows` rows (LBO = rows * 16 B between 8-element K chunks, SBO = 128 B between 8-row groups)
__device__ __forceinline__ uint64_t kdesc(uint32_t saddr, uint32_t rows) { return umma_desc(saddr, rows * 16u, 128u); }

}  // namespace

template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) pixel_d_kernel(const PixelDParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t s_base = smem_u32(smem);
  const uint32_t bar = s_base + kOffBar;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 16);
  float* par = reinterpret_cast<float*>(smem + kOffPar);
  float* red = reinterpret_cast<float*>(smem + kOffRed);
  const int norm = p.norm;
  const bool want_pg = MODE == kBwdGrad && p.part_w2 != nullptr;

  if (warp == 0) {
    if (lane == 0) {
      mbar_init(bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // W2 [c2][c1] fp32 -> bf16 in both operand layouts
  for (int i = tid; i < kC2 * kC1; i += kThreads) {
    const int c2 = i / kC1, c1 = i - c2 * kC1;
    const __nv_bfloat16 v = __float2bfloat16(__ldg(p.w2 + i));
    *reinterpret_cast<__nv_bfloat16*>(smem + kOffW2 + (c1 >> 3) * (kC2 * 16) + c2 * 16 + (c1 & 7) * 2) = v;
    *reinterpret_cast<__nv_bfloat16*>(smem + kOffW2T + (c2 >> 3) * (kC1 * 16) + c1 * 16 + (c2 & 7) * 2) = v;
  }
  if (tid < kC1) {
    par[kPW1 + tid] = __ldg(p.w1 + tid);
    par[kPB1 + tid] = __ldg(p.b1 + tid);
  }
  par[kPW3 + tid] = __ldg(p.w3 + tid);
  par[kPB2 + tid] = p.b2 ? __ldg(p.b2 + tid) : 0.f;
  par[kPG + tid] = norm == kNormBatch ? __ldg(p.gamma + tid) : 1.f;
  par[kPBeta + tid] = norm == kNormBatch ? __ldg(p.beta + tid) : 0.f;
  const float b3 = p.b3 ? __ldg(p.b3) : 0.f;
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_off = (uint32_t)(warp * 32) << 16;

  const int G = gridDim.x, b = blockIdx.x;
  const int t0 = (int)((long long)b * p.tiles / G), t1 = (int)((long long)(b + 1) * p.tiles / G);
  const int n_first = t0 / p.tiles_per_sample, n_last = (t1 - 1) / p.tiles_per_sample;
  if (MODE == kStats || MODE == kBwdSums) {   // partials of the samples this CTA never sees are zero
    for (int n = 0; n < p.n; ++n)
      if (n < n_first || n > n_last)
        for (int q = 0; q < kNQ; ++q) p.part[(((size_t)b * p.n + n) * kNQ + q) * kC2 + tid] = 0.f;
  }

  float acc[kNQ][4];
#pragma unroll
  for (int q = 0; q < kNQ; ++q)
#pragma unroll
    for (int g = 0; g < 4; ++g) acc[q][g] = 0.f;
  float acc_g = 0.f;   // kBwdSums: sum of the logit gradient
  uint32_t phase = 0;
  int cur_n = -1;
  bool need_shift = false;   // kStats: the sample's shift is taken from its first tile
  int cnt_pix = 0;           // kStats: pixels of the current sample seen by this CTA

  // per-sample partials of kStats / kBwdSums: warps in a fixed order
  auto flush = [&](int n) {
#pragma unroll
    for (int q = 0; q < kNQ; ++q)
#pragma unroll
      for (int g = 0; g < 4; ++g) { red[(warp * kNQ + q) * kC2 + g * 32 + lane] = acc[q][g]; acc[q][g] = 0.f; }
    if (MODE == kBwdSums) {
      const float s = warp_sum(acc_g);
      acc_g = 0.f;
      if (lane == 0) red[(warp * kNQ + 3) * kC2] = s;   // quantity 3, channel 0: sum of g
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kNQ; ++q) {
      float s = red[q * kC2 + tid];
#pragma unroll
      for (int w = 1; w < 4; ++w) s += red[(w * kNQ + q) * kC2 + tid];
      if (MODE == kStats && q == 2) s = par[kPShift + tid];
      if (MODE == kStats && q == 3) s = __int_as_float(cnt_pix);
      p.part[(((size_t)b * p.n + n) * kNQ + q) * kC2 + tid] = s;
    }
    cnt_pix = 0;
    __syncthreads();
  };

  auto issue_and_wait = [&](int which, bool first) {
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        if (which == 0) {   // h2 = h1 W2^T: M 128 pixels, N 128, K 64
#pragma unroll
          for (int k = 0; k < kC1 / 16; ++k)
            umma_bf16(tmem, kdesc(s_base + kOffH1 + k * 2 * 2048, 128), kdesc(s_base + kOffW2 + k * 2 * 2048, 128), kIdescN128, k > 0);
        } else {            // dh1 = dh2 W2: M 128 pixels, N 64, K 128;  dW2 += dh2^T h1: M 128 channels, N 64, K 128 pixels
#pragma unroll
          for (int k = 0; k < kC2 / 16; ++k)
            umma_bf16(tmem + 128, kdesc(s_base + kOffDH2 + k * 2 * 2048, 128), kdesc(s_base + kOffW2T + k * 2 * 1024, 64), kIdescN64, k > 0);
          if (which == 2) {
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
              umma_bf16(tmem + 192, kdesc(s_base + kOffDH2T + k * 2 * 2048, 128), kdesc(s_base + kOffH1T + k * 2 * 1024, 64), kIdescN64,
                        (first && k == 0) ? 0u : 1u);
          }
        }
        umma_commit(bar);
      }
      __syncwarp();
    }
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after();
  };

  for (int t = t0; t < t1; ++t) {
    const int n = t / p.tiles_per_sample;
    const int pix0 = (t - n * p.tiles_per_sample) * kTile;
    const int m = tid;
    const bool valid = pix0 + m < p.hw;
    const size_t gp = (size_t)n * p.hw + pix0 + m;
    if (n != cur_n) {
      if ((MODE == kStats || MODE == kBwdSums) && cur_n >= 0) flush(cur_n);
      cur_n = n;
      need_shift = true;
      if (MODE != kStats && norm != kNormNone) {
        const int si = norm == kNormInstance ? n * kC2 + tid : tid;
        par[kPMean + tid] = __ldg(p.mean + si);
        par[kPInv + tid] = __ldg(p.invstd + si);
        if (MODE == kBwdGrad) {
          if (norm == kNormInstance) {
            par[kPS1 + tid] = __ldg(p.sums + (size_t)n * 2 * kC2 + tid);
            par[kPS2 + tid] = __ldg(p.sums + ((size_t)n * 2 + 1) * kC2 + tid);
          } else {
            float s1 = 0.f, s2 = 0.f;
            for (int i = 0; i < p.n; ++i) {
              s1 += __ldg(p.sums + (size_t)i * 2 * kC2 + tid);
              s2 += __ldg(p.sums + ((size_t)i * 2 + 1) * kC2 + tid);
            }
            par[kPS1 + tid] = s1;
            par[kPS2 + tid] = s2;
          }
        }
      }
    }
    // ---- layer 1 in registers; h1 -> bf16 operand rows (and the transposed copy for dW2)
    const float xv = valid ? __ldg(p.x + gp) : 0.f;
#pragma unroll
    for (int c8 = 0; c8 < kC1 / 8; ++c8) {
      float h[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) h[e] = valid ? lrelu(fmaf(par[kPW1 + c8 * 8 + e], xv, par[kPB1 + c8 * 8 + e]), p.slope) : 0.f;
      sts16(smem + kOffH1, c8 * 2048 + m * 16, h);
      if (want_pg) {
#pragma unroll
        for (int e = 0; e < 8; ++e)
          *reinterpret_cast<__nv_bfloat16*>(smem + kOffH1T + (m >> 3) * (kC1 * 16) + (c8 * 8 + e) * 16 + (m & 7) * 2) = __float2bfloat16(h[e]);
      }
    }
    fence_proxy_async();
    __syncthreads();
    issue_and_wait(0, false);
    if (MODE == kStats) {
      cnt_pix += min(kTile, p.hw - pix0);
      if (need_shift) {   // row 0 (always a pixel of the sample) gives the shift
        if (warp == 0) {
#pragma unroll
          for (int g32 = 0; g32 < 4; ++g32) {
            float v[32];
            tmem_ld<32>(tmem + g32 * 32, v);
            tmem_ld_wait();
            if (lane == 0)
#pragma unroll
              for (int j = 0; j < 32; ++j) par[kPShift + g32 * 32 + j] = v[j] + par[kPB2 + g32 * 32 + j];
          }
        }
        __syncthreads();
        need_shift = false;
      }
    }

    // ---- h2 epilogue, 32 channels at a time
    const float g = (MODE >= kBwdSums && valid) ? __ldg(p.dy + gp) : 0.f;
    float logit = b3;
#pragma unroll
    for (int g32 = 0; g32 < 4; ++g32) {
      float v[32];
      tmem_ld<32>(tmem + lane_off + g32 * 32, v);
      tmem_ld_wait();
      const int c0 = g32 * 32;
      if constexpr (MODE == kStats) {
        float sq[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          v[j] = valid ? v[j] + par[kPB2 + c0 + j] - par[kPShift + c0 + j] : 0.f;
          sq[j] = v[j] * v[j];
        }
        acc[0][g32] += xreduce32(v, lane);
        acc[1][g32] += xreduce32(sq, lane);
      } else {
      float xh[32], dz[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int c = c0 + j;
        const float pre = v[j] + par[kPB2 + c];
        float z;
        if (norm == kNormNone) { xh[j] = 0.f; z = pre; }
        else {
          xh[j] = (pre - par[kPMean + c]) * par[kPInv + c];
          z = fmaf(par[kPG + c], xh[j], par[kPBeta + c]);
        }
        const float a = lrelu(z, p.slope);
        if (MODE == kApply) logit = fmaf(par[kPW3 + c], a, logit);
        v[j] = g * a;                                                    // dw3 term
        dz[j] = g * par[kPW3 + c] * (z > 0.f ? 1.f : p.slope);          // d loss / d z
      }
      if constexpr (MODE == kBwdSums) {
        acc[0][g32] += xreduce32(v, lane);
        if (norm != kNormNone) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = dz[j] * xh[j];
          acc[2][g32] += xreduce32(v, lane);
          acc[1][g32] += xreduce32(dz, lane);
        }
      } else if constexpr (MODE == kBwdGrad) {
      // kBwdGrad: dh2, rounded to bf16 into both operand layouts (zero rows for pixels past the sample)
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int c = c0 + j;
        float d;
        if (norm == kNormNone) d = dz[j];
        else {
          const float gam = par[kPG + c], inv_m = 1.f / (float)p.count;
          d = par[kPInv + c] * (gam * dz[j] - gam * par[kPS1 + c] * inv_m - xh[j] * gam * par[kPS2 + c] * inv_m);
        }
        v[j] = valid ? d : 0.f;
      }
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float h[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) h[e] = v[c8 * 8 + e];
        sts16(smem + kOffDH2, (g32 * 4 + c8) * 2048 + m * 16, h);
      }
      if (want_pg)
#pragma unroll
        for (int j = 0; j < 32; ++j)
          *reinterpret_cast<__nv_bfloat16*>(smem + kOffDH2T + (m >> 3) * (kC2 * 16) + (c0 + j) * 16 + (m & 7) * 2) = __float2bfloat16(v[j]);
      if (want_pg && p.b2) acc[1][g32] += xreduce32(v, lane);   // db2 (instance norm: zero up to rounding)
      }
      }
    }
    if (MODE == kApply && valid) p.y[gp] = logit;
    if (MODE == kBwdSums) acc_g += g;
    if (MODE == kBwdGrad) {
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      issue_and_wait(want_pg ? 2 : 1, t == t0);
      // dh1 -> dpre1 -> dx, dw1, db1
      float dxv = 0.f;
#pragma unroll
      for (int g32 = 0; g32 < 2; ++g32) {
        float v[32], d1[32];
        tmem_ld<32>(tmem + lane_off + 128 + g32 * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int c = g32 * 32 + j;
          const float pre1 = fmaf(par[kPW1 + c], xv, par[kPB1 + c]);
          d1[j] = valid ? v[j] * (pre1 > 0.f ? 1.f : p.slope) : 0.f;
          dxv = fmaf(d1[j], par[kPW1 + c], dxv);
          v[j] = d1[j] * xv;
        }
        if (want_pg) {
          acc[0][g32] += xreduce32(v, lane);          // dw1: channels 0-63
          acc[0][2 + g32] += xreduce32(d1, lane);     // db1: channels 64-127 of the partial row
        }
      }
      if (p.dx && valid) p.dx[gp] = dxv;
    }
    tc_fence_before();
    __syncthreads();   // the next tile overwrites the operand tiles and the TMEM accumulators
  }
  if ((MODE == kStats || MODE == kBwdSums) && cur_n >= 0) flush(cur_n);
  if (want_pg) {
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int g = 0; g < 4; ++g) red[(warp * kNQ + q) * kC2 + g * 32 + lane] = acc[q][g];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      float s = red[q * kC2 + tid];
#pragma unroll
      for (int w = 1; w < 4; ++w) s += red[(w * kNQ + q) * kC2 + tid];
      p.part[((size_t)b * 2 + q) * kC2 + tid] = s;
    }
    tc_fence_after();
    float* dst = p.part_w2 + ((size_t)b * kC2 + tid) * kC1;   // TMEM lane = channel c2
#pragma unroll 1
    for (int c = 0; c < kC1; c += 16) {
      float v[16];
      tmem_ld<16>(tmem + lane_off + 192 + c, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(dst + c + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------- fixed-order reductions of the partials
// norm statistics: block = one sample (instance) or the batch (batch norm), thread = channel
__global__ void __launch_bounds__(kC2) pixel_d_stats_kernel(const float* __restrict__ part, int grid, int n, long long count, int norm,
                                                            float eps, float momentum, float* mean, float* invstd, float* running_mean,
                                                            float* running_var) {
  const int c = threadIdx.x, s = blockIdx.x;
  double cnt = 0.0, mu = 0.0, m2 = 0.0;   // pairwise merge of the (count, mean, M2) of each CTA's sample, in a fixed order
  for (int b = 0; b < grid; ++b)
    for (int i = (norm == kNormInstance ? s : 0); i < (norm == kNormInstance ? s + 1 : n); ++i) {
      const float* r = part + ((size_t)b * n + i) * kNQ * kC2;
      const double cb = (double)__float_as_int(r[3 * kC2 + c]);
      if (cb == 0.0) continue;
      const double sb = r[c], qb = r[kC2 + c];
      const double mb = (double)r[2 * kC2 + c] + sb / cb, m2b = fmax(qb - sb * sb / cb, 0.0);
      const double tot = cnt + cb, delta = mb - mu;
      mu += delta * cb / tot;
      m2 += m2b + delta * delta * cnt * cb / tot;
      cnt = tot;
    }
  const double var = m2 / (double)count;
  const int o = norm == kNormInstance ? s * kC2 + c : c;
  mean[o] = (float)mu;
  invstd[o] = (float)(1.0 / sqrt(var + (double)eps));
  if (norm == kNormBatch && running_mean) {
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mu;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)(var * (double)count / (double)(count - 1));
  }
}

// backward sums: block s < n: per-sample sum dz / sum dz xhat -> sums[s]; block n: parameter gradients dw3, db3, dgamma, dbeta
__global__ void __launch_bounds__(kC2) pixel_d_bwd_sums_kernel(const float* __restrict__ part, int grid, int n, float* sums, float* dw3,
                                                               float* db3, float* dgamma, float* dbeta) {
  const int c = threadIdx.x, s = blockIdx.x;
  if (s < n) {
    double a = 0.0, q = 0.0;
    for (int b = 0; b < grid; ++b) {
      a += part[(((size_t)b * n + s) * kNQ + 1) * kC2 + c];
      q += part[(((size_t)b * n + s) * kNQ + 2) * kC2 + c];
    }
    sums[(size_t)s * 2 * kC2 + c] = (float)a;
    sums[((size_t)s * 2 + 1) * kC2 + c] = (float)q;
    return;
  }
  double w = 0.0, g = 0.0, d1 = 0.0, d2 = 0.0;
  for (int b = 0; b < grid; ++b)
    for (int i = 0; i < n; ++i) {
      const float* r = part + ((size_t)b * n + i) * kNQ * kC2;
      w += r[c]; d1 += r[kC2 + c]; d2 += r[2 * kC2 + c];
      if (c == 0) g += r[3 * kC2];
    }
  if (dw3) dw3[c] = (float)w;
  if (db3 && c == 0) *db3 = (float)g;
  if (dgamma) dgamma[c] = (float)d2;
  if (dbeta) dbeta[c] = (float)d1;
}

// parameter gradients of the second backward pass: blocks 0-63 dW2 (128 entries each), block 64 dw1 / db1, block 65 db2
__global__ void __launch_bounds__(kC2) pixel_d_bwd_params_kernel(const float* __restrict__ part, const float* __restrict__ part_w2,
                                                                 int grid, float* dw1, float* db1, float* dw2, float* db2) {
  const int t = threadIdx.x, blk = blockIdx.x;
  double s = 0.0;
  if (blk < kC2 * kC1 / kC2) {
    const int i = blk * kC2 + t;   // dW2 element (c2, c1), row-major [c2][c1]
    for (int b = 0; b < grid; ++b) s += part_w2[(size_t)b * kC2 * kC1 + i];
    dw2[i] = (float)s;
    return;
  }
  const int q = blk - kC2 * kC1 / kC2;
  for (int b = 0; b < grid; ++b) s += part[((size_t)b * 2 + q) * kC2 + t];
  if (q == 0) {
    if (t < kC1) dw1[t] = (float)s;
    else db1[t - kC1] = (float)s;
  } else if (db2) {
    db2[t] = (float)s;
  }
}

// ------------------------------------------------------------------------------------------- host
namespace {

int sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

struct Layout {
  int tps, tiles, grid;
  size_t part, sums, part_w2, total;   // byte offsets / size
};

Layout layout(int n, int h, int w) {
  Layout L;
  const long long hw = (long long)h * w;
  L.tps = (int)((hw + kTile - 1) / kTile);
  L.tiles = n * L.tps;
  L.grid = L.tiles < sm_count() ? L.tiles : sm_count();
  L.part = 0;
  L.sums = L.part + (size_t)L.grid * n * kNQ * kC2 * 4;
  L.part_w2 = L.sums + (size_t)n * 2 * kC2 * 4;
  L.total = L.part_w2 + (size_t)L.grid * kC2 * kC1 * 4;
  return L;
}

template <int MODE>
int launch(const PixelDParams& p, int grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    HV_CUDA(cudaFuncSetAttribute(pixel_d_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    configured = true;
  }
  pixel_d_kernel<MODE><<<grid, kThreads, kSmem, st>>>(p);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

int check_common(int n, int cin, int ndf, int h, int w, int norm) {
  HV_CHECK_ARG(cin == 1, "pixel_d: input_nc=%d not built (the fused kernels take input_nc = 1)", cin);
  HV_CHECK_ARG(ndf == kC1, "pixel_d: ndf=%d not built (the fused kernels take ndf = 64)", ndf);
  HV_CHECK_ARG(norm >= kNormNone && norm <= kNormInstance, "pixel_d: norm %d unsupported (0 none, 1 batch, 2 instance)", norm);
  HV_CHECK_ARG(n > 0 && h > 0 && w > 0 && (long long)n * h * w < (1ll << 31), "pixel_d: bad extent n=%d h=%d w=%d", n, h, w);
  HV_CHECK_ARG(norm != kNormBatch || (long long)n * h * w > 1, "pixel_d: batch norm needs more than one value per channel");
  return HV_OK;
}

}  // namespace

}  // namespace hv

using namespace hv;

extern "C" size_t hv_pixel_d_workspace_bytes(int n, int h, int w) {
  if (n <= 0 || h <= 0 || w <= 0) return 0;
  return layout(n, h, w).total;
}

extern "C" int hv_pixel_d_fwd_bf16(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* gamma,
                                   const float* beta, const float* w3, const float* b3, float* running_mean, float* running_var,
                                   float* y, float* save_mean, float* save_invstd, int n, int cin, int ndf, int h, int w, int norm,
                                   float momentum, float eps, float slope, void* workspace, hv_stream_t stream) {
  int rc = check_common(n, cin, ndf, h, w, norm);
  if (rc) return rc;
  HV_CHECK_ARG(x && w1 && b1 && w2 && w3 && y && workspace, "pixel_d_fwd: null argument");
  HV_CHECK_ARG(norm == kNormNone || (save_mean && save_invstd), "pixel_d_fwd: the norm needs save_mean / save_invstd");
  HV_CHECK_ARG(norm != kNormBatch || (gamma && beta), "pixel_d_fwd: batch norm needs gamma / beta");
  HV_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr), "pixel_d_fwd: running_mean and running_var go together");
  const Layout L = layout(n, h, w);
  cudaStream_t st = as_stream(stream);
  PixelDParams p = {};
  p.x = x; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.gamma = gamma; p.beta = beta; p.w3 = w3; p.b3 = b3;
  p.mean = save_mean; p.invstd = save_invstd; p.y = y;
  p.n = n; p.hw = h * w; p.tiles_per_sample = L.tps; p.tiles = L.tiles; p.norm = norm; p.slope = slope;
  p.count = norm == kNormInstance ? (long long)h * w : (long long)n * h * w;
  p.part = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + L.part);
  if (norm != kNormNone) {
    if ((rc = launch<kStats>(p, L.grid, st))) return rc;
    pixel_d_stats_kernel<<<norm == kNormInstance ? n : 1, kC2, 0, st>>>(p.part, L.grid, n, p.count, norm, eps, momentum, save_mean,
                                                                       save_invstd, running_mean, running_var);
    HV_LAUNCH_CHECK();
  }
  return launch<kApply>(p, L.grid, st);
}

extern "C" int hv_pixel_d_bwd_bf16(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* gamma,
                                   const float* beta, const float* w3, const float* b3, const float* save_mean, const float* save_invstd,
                                   const float* dy, float* dx, float* dw1, float* db1, float* dw2, float* db2, float* dgamma, float* dbeta,
                                   float* dw3, float* db3, int n, int cin, int ndf, int h, int w, int norm, float slope, void* workspace,
                                   hv_stream_t stream) {
  int rc = check_common(n, cin, ndf, h, w, norm);
  if (rc) return rc;
  HV_CHECK_ARG(x && w1 && b1 && w2 && w3 && dy && workspace, "pixel_d_bwd: null argument");
  HV_CHECK_ARG(norm == kNormNone || (save_mean && save_invstd), "pixel_d_bwd: the norm needs save_mean / save_invstd");
  HV_CHECK_ARG(norm != kNormBatch || (gamma && beta), "pixel_d_bwd: batch norm needs gamma / beta");
  const bool pg = dw1 != nullptr;
  HV_CHECK_ARG(!pg || (db1 && dw2 && dw3), "pixel_d_bwd: parameter gradients need dw1, db1, dw2 and dw3");
  HV_CHECK_ARG(pg || dx, "pixel_d_bwd: nothing to compute (dx and the parameter gradients are NULL)");
  const Layout L = layout(n, h, w);
  cudaStream_t st = as_stream(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  PixelDParams p = {};
  p.x = x; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.gamma = gamma; p.beta = beta; p.w3 = w3; p.b3 = b3;
  p.mean = save_mean; p.invstd = save_invstd; p.dy = dy; p.dx = dx;
  p.n = n; p.hw = h * w; p.tiles_per_sample = L.tps; p.tiles = L.tiles; p.norm = norm; p.slope = slope;
  p.count = norm == kNormInstance ? (long long)h * w : (long long)n * h * w;
  p.sums = reinterpret_cast<float*>(ws + L.sums);
  // pass 1: the sums the norm's backward needs and the logit layer's parameter gradients
  if (norm != kNormNone || pg) {
    p.part = reinterpret_cast<float*>(ws + L.part);
    if ((rc = launch<kBwdSums>(p, L.grid, st))) return rc;
    pixel_d_bwd_sums_kernel<<<n + 1, kC2, 0, st>>>(p.part, L.grid, n, reinterpret_cast<float*>(ws + L.sums), pg ? dw3 : nullptr,
                                                  pg ? db3 : nullptr, pg && norm == kNormBatch ? dgamma : nullptr,
                                                  pg && norm == kNormBatch ? dbeta : nullptr);
    HV_LAUNCH_CHECK();
  }
  // pass 2: dh2 on the tensor cores -> dx, dW2, dw1, db1, db2
  p.part = reinterpret_cast<float*>(ws + L.part);
  p.part_w2 = pg ? reinterpret_cast<float*>(ws + L.part_w2) : nullptr;
  if ((rc = launch<kBwdGrad>(p, L.grid, st))) return rc;
  if (pg) {
    pixel_d_bwd_params_kernel<<<kC1 + 2, kC2, 0, st>>>(p.part, p.part_w2, L.grid, dw1, db1, dw2, b2 ? db2 : nullptr);
    HV_LAUNCH_CHECK();
  }
  return HV_OK;
}
