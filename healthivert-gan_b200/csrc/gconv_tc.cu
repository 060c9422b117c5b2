// Data and weight gradients of the generator's convolutions on the tensor cores (bf16 operands, fp32 accumulate): the backward of
// Conv2dBlock (reference models/inpaint_networks.py:494-503 under torch.autograd, models/pix2pix_model.py:354) for ANY layer of the
// generator - k = 3 / 5, stride 1 / 2, dilation 1 .. 16, fused source gather (channel concat, nearest x2 / x0.5, scalar planes) - as
// batched "NT" GEMMs on the tcgen05 kernel of gemm_tc.cu over explicit im2col operands (same scheme as dconv_tc.cu):
//
//   wgrad   dWt[b,s][r][co] = sum_p colT[b,s][r][p] * dy[b,s][co][p]      r = ci*k*k + tap;  M = rows (padded to 128), N = Cout (padded to
//                                                                        32 / 64 / 128), K = a split of the output pixels;  dW = sum_{b,s}
//   dgrad   dcolT[b][r][p]  = sum_co Wt[r][co] * dyT[b][p][co]             M = rows, N = pixels, K = Cout (padded to 64);  dx = col2im(dcolT)
//
// dx is the gradient over the VIRTUAL concatenated input [n, cin, hin, win] of the forward descriptor, exactly like hv_conv2d_dgrad;
// the host routes channel ranges back to their source tensors.  fp32 SIMT kernels (train_ops.cu) remain the parity path.
#include <cuda_bf16.h>
#include "hv_common.cuh"
#include "kernels.h"

namespace hv {

int gemm_tc_nt(const __nv_bfloat16* A, const __nv_bfloat16* B, void* C, const float* colscale, int M, int N, int K, int batch,
               long long strideA, long long strideB, int out_bf16, cudaStream_t st);
int gemm_tc_taps(const __nv_bfloat16* DY, const __nv_bfloat16* X, float* part, int n, int cout, int cin, int plane, const int* tap_off,
                 const int* tap_rep, int nrep, int ntaps, int tpm, int co8, int bn, int nkc, int kb0, int kblocks, cudaStream_t st);

struct GcGeom {
  hv_conv_src src[4];
  int nsrc;
  int n, cin, cout, hin, win, hout, wout, k, kk, stride, pad, dil;
  int R, Rp;        // im2col rows cin * k * k, padded to a multiple of 128
  int P, Pp;        // output pixels per image, padded to a multiple of 256
  int Np;           // Cout padded to 32 / 64 / a multiple of 128 (wgrad GEMM N)
  int Kc;           // Cout padded to a multiple of 64 (dgrad GEMM K)
  int nsplit, Pc;   // wgrad: the pixels of an image are split into nsplit chunks of Pc (multiple of 64) pixels
};

static int gc_geom(GcGeom& g, const hv_conv_desc* d) {
  HV_CHECK_ARG(d && d->nsrc >= 1 && d->nsrc <= 4 && d->cout >= 1 && d->cout <= 512, "gconv_tc: bad descriptor");
  int csum = 0;
  for (int i = 0; i < 4; ++i) {
    g.src[i] = d->src[i < d->nsrc ? i : 0];
    if (i < d->nsrc) csum += d->src[i].channels;
  }
  HV_CHECK_ARG(csum == d->cin, "gconv_tc: sources have %d channels, cin=%d", csum, d->cin);
  g.nsrc = d->nsrc; g.n = d->n; g.cin = d->cin; g.cout = d->cout; g.hin = d->hin; g.win = d->win;
  g.k = d->k; g.kk = d->k * d->k; g.stride = d->stride; g.pad = d->pad; g.dil = d->dil;
  const int eff = (d->k - 1) * d->dil + 1;
  g.hout = (d->hin + 2 * d->pad - eff) / d->stride + 1; g.wout = (d->win + 2 * d->pad - eff) / d->stride + 1;
  HV_CHECK_ARG(g.hout >= 1 && g.wout >= 1, "gconv_tc: empty output");
  g.R = d->cin * g.kk; g.Rp = (g.R + 127) & ~127;
  g.P = g.hout * g.wout; g.Pp = (g.P + 255) & ~255;
  g.Np = d->cout <= 32 ? 32 : (d->cout <= 64 ? 64 : ((d->cout + 127) & ~127));
  g.Kc = (d->cout + 63) & ~63;
  // wgrad split over the pixels: enough (image, chunk) batches to fill the GPU with Rp / 128 row tiles each; chunks of >= 1024 pixels
  g.Pc = g.Pp;
  g.nsplit = 1;
  while (g.Pc > 1024 && (g.Pc % 128) == 0 && (long long)g.n * g.nsplit * (g.Rp / 128) < 296) { g.Pc >>= 1; g.nsplit <<= 1; }
  return HV_OK;
}

// colT[b][s][r][pc]: row r = ci * kk + tap of image b, pixel s * Pc + pc.  One thread = (b, ci, 8 consecutive pixels): the source of
// the channel is resolved once, every tap gathers 8 values and writes ONE 16-byte store (the kernel is pure data movement: 9 - 25x
// the bytes of the input; 2-byte stores per thread ran at a tenth of the HBM rate).
struct GcSrc { const float* base; int mode, sh, sw; };   // plane of (image, channel) in its own tensor
__device__ __forceinline__ GcSrc gc_resolve(const GcGeom& g, int n, int ch) {
  int s = 0;
  while (s < g.nsrc - 1 && ch >= g.src[s].channels) { ch -= g.src[s].channels; ++s; }
  GcSrc r;
  r.mode = g.src[s].mode;
  r.sh = g.hin; r.sw = g.win;
  if (r.mode == HV_SRC_UP2) { r.sh >>= 1; r.sw >>= 1; }
  else if (r.mode == HV_SRC_SUB2) { r.sh <<= 1; r.sw <<= 1; }
  r.base = r.mode == HV_SRC_SCALAR ? g.src[s].ptr + n : g.src[s].ptr + ((size_t)n * g.src[s].channels + ch) * r.sh * r.sw;
  return r;
}
__device__ __forceinline__ float gc_fetch(const GcGeom& g, const GcSrc& r, int gy, int gx) {
  if (gy < 0 || gy >= g.hin || gx < 0 || gx >= g.win) return 0.f;
  if (r.mode == HV_SRC_SCALAR) return __ldg(r.base);
  if (r.mode == HV_SRC_UP2) { gy >>= 1; gx >>= 1; }
  else if (r.mode == HV_SRC_SUB2) { gy <<= 1; gx <<= 1; }
  return __ldg(r.base + (size_t)gy * r.sw + gx);
}

__global__ void __launch_bounds__(256) gc_im2col_kernel(GcGeom g, __nv_bfloat16* __restrict__ colT) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P8 = g.Pp >> 3;
  if (i >= (long long)g.n * g.cin * P8) return;
  const int p0 = (int)(i % P8) * 8, ci = (int)((i / P8) % g.cin), b = (int)(i / ((long long)P8 * g.cin));
  const GcSrc src = gc_resolve(g, b, ci);
  const int s = p0 / g.Pc, pc = p0 - s * g.Pc;            // Pc is a multiple of 64: the 8 pixels stay in one chunk
  __nv_bfloat16* dst = colT + (((size_t)b * g.nsplit + s) * g.Rp + (size_t)ci * g.kk) * g.Pc + pc;
  int oy[8], ox[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { const int p = p0 + j; oy[j] = p / g.wout; ox[j] = p - oy[j] * g.wout; }
  for (int ky = 0; ky < g.k; ++ky)
    for (int kx = 0; kx < g.k; ++kx) {
      __align__(16) __nv_bfloat16 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j)
        v[j] = __float2bfloat16(p0 + j < g.P ? gc_fetch(g, src, oy[j] * g.stride + ky * g.dil - g.pad, ox[j] * g.stride + kx * g.dil - g.pad) : 0.f);
      *reinterpret_cast<uint4*>(dst + (size_t)(ky * g.k + kx) * g.Pc) = *reinterpret_cast<const uint4*>(v);
    }
}

// dy fp32 [b][cout][P] -> dyb bf16 [b][s][Np][Pc] (wgrad B operand).  Only the rows of real filters are written: rows >= cout feed
// output columns >= cout of the GEMM, which nobody reads (a padding ROW or COLUMN of an operand may hold anything; only padding along
// K - pixels >= P here - must be zero, and is).  One thread = 8 consecutive pixels.
__global__ void __launch_bounds__(256) gc_cast_dy_kernel(const float* __restrict__ dy, __nv_bfloat16* __restrict__ dyb, GcGeom g) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P8 = g.Pp >> 3;
  if (i >= (long long)g.n * g.cout * P8) return;
  const int p0 = (int)(i % P8) * 8, co = (int)((i / P8) % g.cout), b = (int)(i / ((long long)P8 * g.cout));
  const int s = p0 / g.Pc, pc = p0 - s * g.Pc;
  const float* src = dy + ((size_t)b * g.cout + co) * g.P;
  __align__(16) __nv_bfloat16 v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = __float2bfloat16(p0 + j < g.P ? src[p0 + j] : 0.f);
  *reinterpret_cast<uint4*>(dyb + (((size_t)b * g.nsplit + s) * g.Np + co) * g.Pc + pc) = *reinterpret_cast<const uint4*>(v);
}

// dw[co][r] = sum over the (b, s) blocks of part[blk][r][co]   (part: fp32 [blocks][Rp][Np])
__global__ void __launch_bounds__(256) gc_reduce_dw_kernel(const float* __restrict__ part, float* __restrict__ dw, int blocks, int R, int Rp, int cout, int Np) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * cout) return;
  const int co = i % cout, r = i / cout;     // co fastest: coalesced reads of part
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += part[((size_t)b * Rp + r) * Np + co];
  dw[(size_t)co * R + r] = s;
}

// Wt bf16 [Rp][Kc]: Wt[ci * kk + t][co] = w[co][ci][t], zero padding
__global__ void __launch_bounds__(256) gc_wt_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wt, int cout, int R, int Rp, int Kc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Rp * Kc) return;
  const int co = i % Kc, r = i / Kc;
  wt[i] = __float2bfloat16((co < cout && r < R) ? w[(size_t)co * R + r] : 0.f);
}

// dy fp32 [b][cout][P] -> dyT bf16 [b][Pp][Kc] through 32 x 32 shared-memory tiles; grid (Pp / 32, Kc / 32, b)
__global__ void __launch_bounds__(256) gc_dyT_kernel(const float* __restrict__ dy, __nv_bfloat16* __restrict__ dyT, int cout, int Kc, int P, int Pp) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int p = p0 + tx, co = c0 + r;
    tile[r][tx] = (p < P && co < cout) ? dy[((size_t)b * cout + co) * P + p] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) dyT[((size_t)b * Pp + p0 + r) * Kc + c0 + tx] = __float2bfloat16(tile[tx][r]);
}

// dx[b][ci][y][x] = sum over the taps whose output pixel exists: dcolT[b][ci * kk + t][oy * wout + ox], oy = (y + pad - ky * dil) / stride.
// One thread = 4 consecutive x of one input row (one 16-byte store; the row / tap arithmetic is shared by the four).
__global__ void __launch_bounds__(256) gc_col2im_kernel(const __nv_bfloat16* __restrict__ dcolT, float* __restrict__ dx, GcGeom g) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int W4 = (g.win + 3) >> 2;
  if (i >= (long long)g.n * g.cin * g.hin * W4) return;
  const int x0 = (int)(i % W4) * 4, y = (int)((i / W4) % g.hin);
  const long long bc = i / ((long long)W4 * g.hin);
  const int ci = (int)(bc % g.cin), b = (int)(bc / g.cin);
  const __nv_bfloat16* src = dcolT + ((size_t)b * g.Rp + (size_t)ci * g.kk) * g.Pp;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int ky = 0; ky < g.k; ++ky) {
    const int ty = y + g.pad - ky * g.dil;
    if (ty < 0 || (g.stride == 2 && (ty & 1))) continue;
    const int oy = g.stride == 2 ? ty >> 1 : ty;
    if (oy >= g.hout) continue;
    const __nv_bfloat16* row = src + (size_t)oy * g.wout;
    for (int kx = 0; kx < g.k; ++kx) {
      const __nv_bfloat16* tap = row + (size_t)(ky * g.k + kx) * g.Pp;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int tx = x0 + j + g.pad - kx * g.dil;
        if (tx < 0 || (g.stride == 2 && (tx & 1))) continue;
        const int ox = g.stride == 2 ? tx >> 1 : tx;
        if (ox < g.wout) acc[j] += __bfloat162float(tap[ox]);
      }
    }
  }
  float* out = dx + ((size_t)bc * g.hin + y) * g.win + x0;
  if ((g.win & 3) == 0) *reinterpret_cast<float4*>(out) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  else
    for (int j = 0; j < 4 && x0 + j < g.win; ++j) out[j] = acc[j];
}

// wf[ci][co][kk - 1 - t] = w[co][ci][t]: the data gradient of a stride-1 'same' convolution is the convolution of dy with these
__global__ void __launch_bounds__(256) gc_flip_w_kernel(const float* __restrict__ w, float* __restrict__ wf, int cout, int cin, int kk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * cin * kk) return;
  const int t = i % kk, ci = (i / kk) % cin, co = i / (kk * cin);
  wf[((size_t)ci * cout + co) * kk + (kk - 1 - t)] = w[i];
}

// ---- single-filter layers over many input channels (the PatchGAN logit conv 512 -> 1, networks.py:598): their gradients are reductions,
// not GEMMs - through the GEMM path the data gradient alone builds an [8192 rows x 1024 pixels] operand per image for 0.2 GFLOP of work.
// dx[n][ci][y][x] = sum over the taps whose output pixel exists of w[ci][ky][kx] * dy[n][oy][ox]; one thread = one input element
// K / S = 0: run-time kernel size / stride (the generic instance).  The kernels are instruction-bound (16 taps x address arithmetic per
// element), so the PatchGAN shape (4 x 4, stride 1) gets compile-time loops: 157 us -> measured below in profiles/.
template <int KT, int ST>
__global__ void __launch_bounds__(256) sf_dgrad_kernel(const float* __restrict__ w, const float* __restrict__ dy, float* __restrict__ dx, GcGeom g) {
  // grid (pixel blocks, cin, n): 32-bit index arithmetic only
  const int i = blockIdx.x * blockDim.x + threadIdx.x, ci = blockIdx.y, b = blockIdx.z;
  if (i >= g.hin * g.win) return;
  const int k = KT ? KT : g.k, stride = ST ? ST : g.stride;
  const int y = i / g.win, x = i - y * g.win;
  const float* wp = w + ci * g.kk;
  const float* dyp = dy + (size_t)b * g.P;
  float acc = 0.f;
#pragma unroll
  for (int ky = 0; ky < (KT ? KT : 5); ++ky) {
    if (ky >= k) break;
    const int ty = y + g.pad - ky * g.dil;
    if (ty < 0 || (stride == 2 && (ty & 1))) continue;
    const int oy = stride == 2 ? ty >> 1 : ty;
    if (oy >= g.hout) continue;
    const float* row = dyp + oy * g.wout;
#pragma unroll
    for (int kx = 0; kx < (KT ? KT : 5); ++kx) {
      if (kx >= k) break;
      const int tx = x + g.pad - kx * g.dil;
      if (tx < 0 || (stride == 2 && (tx & 1))) continue;
      const int ox = stride == 2 ? tx >> 1 : tx;
      if (ox < g.wout) acc = fmaf(__ldg(wp + ky * k + kx), __ldg(row + ox), acc);
    }
  }
  dx[((size_t)b * g.cin + ci) * g.hin * g.win + i] = acc;
}

// part[split][ci][tap] = sum over the split's share of the (image, output pixel) pairs of dy * x(tap); grid (splits, cin); the taps of a
// thread live in registers (k <= 5), block sums through shared memory; a second kernel adds the splits in a fixed order.  A split is a
// run of whole images plus a pixel range, walked with 32-bit arithmetic.  PLAIN: one directly stored source, stride 1 (no gather logic).
template <int KT, bool PLAIN>
__global__ void __launch_bounds__(256) sf_wgrad_kernel(const float* __restrict__ dy, float* __restrict__ part, GcGeom g, int splits) {
  __shared__ float red[8][25];
  const int ci = blockIdx.y, split = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = KT ? KT : g.k;
  const int total = g.n * g.P, per = (total + splits - 1) / splits;
  const int lo = split * per, hi = min(total, lo + per);
  float acc[25];
#pragma unroll
  for (int t = 0; t < 25; ++t) acc[t] = 0.f;
  for (int e = lo + threadIdx.x; e < hi; e += blockDim.x) {
    const int b = e / g.P, p = e - b * g.P;
    const int oy = p / g.wout, ox = p - oy * g.wout;
    const float gval = __ldg(dy + e);
    const int y0 = oy * g.stride - g.pad, x0 = ox * g.stride - g.pad;
    if (PLAIN) {
      const float* plane = g.src[0].ptr + ((size_t)b * g.cin + ci) * g.hin * g.win;
#pragma unroll
      for (int ky = 0; ky < (KT ? KT : 5); ++ky) {
        if (ky >= k) break;
        const int gy = y0 + ky * g.dil;
        const bool row_ok = gy >= 0 && gy < g.hin;
        const float* row = plane + gy * g.win;
#pragma unroll
        for (int kx = 0; kx < (KT ? KT : 5); ++kx) {
          if (kx >= k) break;
          const int gx = x0 + kx * g.dil;
          const float v = (row_ok && gx >= 0 && gx < g.win) ? __ldg(row + gx) : 0.f;
          acc[ky * 5 + kx] = fmaf(gval, v, acc[ky * 5 + kx]);
        }
      }
    } else {
      const GcSrc src = gc_resolve(g, b, ci);
#pragma unroll
      for (int ky = 0; ky < 5; ++ky) {
        if (ky >= k) break;
#pragma unroll
        for (int kx = 0; kx < 5; ++kx) {
          if (kx >= k) break;
          acc[ky * 5 + kx] = fmaf(gval, gc_fetch(g, src, y0 + ky * g.dil, x0 + kx * g.dil), acc[ky * 5 + kx]);
        }
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 25; ++t) {
    float v = acc[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][t] = v;
  }
  __syncthreads();
  if (threadIdx.x < g.kk) {
    const int ky = threadIdx.x / k, kx = threadIdx.x - ky * k;
    float v = 0.f;
#pragma unroll
    for (int wq = 0; wq < 8; ++wq) v += red[wq][ky * 5 + kx];
    part[((size_t)split * g.cin + ci) * g.kk + threadIdx.x] = v;
  }
}
__global__ void __launch_bounds__(256) sf_wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ dw, int splits, int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float v = 0.f;
  for (int s = 0; s < splits; ++s) v += part[(size_t)s * count + i];
  dw[i] = v;
}

static bool sf_eligible(const hv_conv_desc* d) {
  return d->cout == 1 && d->cin >= 64 && d->k <= 5 && d->n <= 65535 && (long long)d->n * d->hin * d->win < (1ll << 30);
}
static int sf_splits(const GcGeom& g) {
  int s = (592 + g.cin - 1) / g.cin;
  const long long total = (long long)g.n * g.P;
  if (s > total / 1024) s = (int)(total / 1024);
  return s < 1 ? 1 : s;
}

static inline unsigned gc_blocks(long long n) { return (unsigned)((n + 255) / 256); }
static inline size_t gc_al(size_t b) { return (b + 255) & ~(size_t)255; }

// ---- weight gradient of the stride-1 'same' convolutions without an im2col operand (gemm_tc_taps) -----------------------------------
// Both operands are bf16 PLANES: the (virtual, concatenated) input X[b][ci] and the output gradient DY[b][co] on the same zero-bordered
// grid - `pad` zero rows above and below, ONE zero gap of bl = roundup(pad, 8) columns between consecutive rows (it is the right border
// of one row and the left border of the next), pixel (y, x) at position (y + pad) * pitch + bl + x.  A filter tap is then a constant
// shift of the position, and dW[co][ci][tap] = sum_k DY[co][k - off(tap)] * X[ci][k] is a GEMM whose A operand is read through shifted
// TMA boxes: 1x the input bytes instead of the k*k x of an im2col operand.  The innermost TMA coordinate must be 16-byte aligned, so
// the part of a shift below 8 positions (the horizontal tap offset (kx - c) * dil mod 8; pitch is a multiple of 8) is taken out of
// pre-shifted REPLICAS of the DY planes: replica j holds DY moved right by r_j positions, one replica per distinct r_j (k of them, or
// one when dil is a multiple of 8).
struct GpGeom {
  int bl, pitch, rows, plane;     // plane: positions per (image, channel), a multiple of 8
  int co8, tpm, ntg, bn;          // filter rows per tap (cout rounded up to 8), taps per 128-row tile, tap groups, GEMM N (cin padded)
  int kb0, kblocks, nkc;          // first 64-position block holding a real pixel, blocks per K chunk, K chunks per image
  int tap_off[25];                // aligned part of the tap shift (multiple of 8 positions)
  int tap_rep[25];                // replica of the DY planes that carries the rest of it
  int nrep, rep_shift[5];         // replica j = DY moved right by rep_shift[j] (0 .. 7) positions
};

static bool gp_eligible(const hv_conv_desc* d) {
  return (d->win & 7) == 0 && d->stride == 1 && (d->k == 3 || d->k == 5) && d->pad == (d->k - 1) / 2 * d->dil && d->cout <= 128 && d->cin <= 256;
}

static void gp_geom(GpGeom& q, const GcGeom& g) {
  q.bl = (g.pad + 7) & ~7;
  q.pitch = g.win + q.bl;
  q.rows = g.hin + 2 * g.pad;
  q.plane = (q.rows * q.pitch + q.bl + 7) & ~7;
  q.co8 = (g.cout + 7) & ~7;
  q.tpm = 128 / q.co8 < g.kk ? 128 / q.co8 : g.kk;
  q.ntg = (g.kk + q.tpm - 1) / q.tpm;
  q.bn = g.cin <= 32 ? 32 : (g.cin <= 64 ? 64 : (g.cin <= 128 ? 128 : 256));
  const int first = g.pad * q.pitch + q.bl, last = (g.pad + g.hin - 1) * q.pitch + q.bl + g.win;   // real pixels of X: [first, last)
  q.kb0 = first / 64;
  const int kb_total = (last + 63) / 64 - q.kb0;
  int nkc = 296 / (g.n * q.ntg);          // <= two full rounds of tiles on 148 SMs
  if (nkc > kb_total / 8) nkc = kb_total / 8;
  if (nkc < 1) nkc = 1;
  q.kblocks = (kb_total + nkc - 1) / nkc;
  q.nkc = (kb_total + q.kblocks - 1) / q.kblocks;
  const int c = g.k / 2;
  q.nrep = 0;
  for (int kx = 0; kx < g.k; ++kx) {
    const int sx = (kx - c) * g.dil, r = ((sx % 8) + 8) % 8;   // DY[k - off] = replica[k - (off - r)], off - r a multiple of 8
    int j = 0;
    while (j < q.nrep && q.rep_shift[j] != r) ++j;
    if (j == q.nrep) q.rep_shift[q.nrep++] = r;
    for (int ky = 0; ky < g.k; ++ky) {
      q.tap_off[ky * g.k + kx] = (ky - c) * g.dil * q.pitch + sx - r;
      q.tap_rep[ky * g.k + kx] = j;
    }
  }
}

// X planes: one thread = 8 consecutive positions of one (image, channel) plane (one 16-byte store); borders and the tail are zeros
__global__ void __launch_bounds__(256) gp_planes_x_kernel(GcGeom g, GpGeom q, __nv_bfloat16* __restrict__ X) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P8 = q.plane >> 3;
  if (i >= (long long)g.n * g.cin * P8) return;
  const int pos0 = (int)(i % P8) * 8, ci = (int)((i / P8) % g.cin), b = (int)(i / ((long long)P8 * g.cin));
  const GcSrc src = gc_resolve(g, b, ci);
  int row = pos0 / q.pitch, col = pos0 - row * q.pitch;
  __align__(16) __nv_bfloat16 v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    v[j] = __float2bfloat16(gc_fetch(g, src, row - g.pad, col - q.bl));   // 0 outside the image
    if (++col == q.pitch) { col = 0; ++row; }
  }
  *reinterpret_cast<uint4*>(X + ((size_t)b * g.cin + ci) * q.plane + pos0) = *reinterpret_cast<const uint4*>(v);
}

// DY planes [b][replica][cout][plane] from the fp32 pre-activation gradient [b][cout][hin * win] (stride 1: output extent == input
// extent); replica j holds the plane moved right by rep_shift[j] positions.  One thread = 8 positions of one (image, filter) plane.
__global__ void __launch_bounds__(256) gp_planes_dy_kernel(const float* __restrict__ dy, GcGeom g, GpGeom q, __nv_bfloat16* __restrict__ DY) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P8 = q.plane >> 3;
  if (i >= (long long)g.n * g.cout * P8) return;
  const int pos0 = (int)(i % P8) * 8;
  const long long bc = i / P8;
  const int co = (int)(bc % g.cout), b = (int)(bc / g.cout);
  const float* src = dy + (size_t)bc * g.hin * g.win;
  // positions pos0 - 7 .. pos0 + 7 cover every replica's 8 values
  float w[15];
  int row = (pos0 - 7 + q.pitch) / q.pitch - 1, col = pos0 - 7 - row * q.pitch;   // floor division for pos0 - 7 >= -7
#pragma unroll
  for (int j = 0; j < 15; ++j) {
    const int y = row - g.pad, x = col - q.bl;
    w[j] = (y >= 0 && y < g.hin && x >= 0 && x < g.win) ? __ldg(src + (size_t)y * g.win + x) : 0.f;
    if (++col == q.pitch) { col = 0; ++row; }
  }
  for (int r = 0; r < q.nrep; ++r) {
    const int sh = q.rep_shift[r];
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float t = 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u) t = (sh == u) ? w[7 + j - u] : t;     // replica[pos] = plane[pos - sh]
      v[j] = __float2bfloat16(t);
    }
    *reinterpret_cast<uint4*>(DY + (((size_t)b * q.nrep + r) * g.cout + co) * q.plane + pos0) = *reinterpret_cast<const uint4*>(v);
  }
}

// dw[co][ci][t] = sum over the (image, K chunk) blocks of part[(blk * ntg + t / tpm)][(t % tpm) * co8 + co][ci].  32 outputs per CTA (ci
// fastest: coalesced reads), the blocks split over 8 warps and added in a fixed order (a single thread per output walked up to ~300
// strided partials serially: 29 us per call for a few KB of output).
__global__ void __launch_bounds__(256) gp_reduce_dw_kernel(const float* __restrict__ part, float* __restrict__ dw, int blocks, int cout, int cin, int kk,
                                                           int tpm, int ntg, int co8, int bn) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  const bool live = i < cout * cin * kk;
  int ci = 0, co = 0, t = 0;
  float s = 0.f;
  if (live) {
    ci = i % cin; co = (i / cin) % cout; t = i / (cin * cout);
    const float* src = part + ((size_t)(t / tpm) * 128 + (size_t)(t % tpm) * co8 + co) * bn + ci;
    const size_t step = (size_t)ntg * 128 * bn;
    for (int b = slice; b < blocks; b += 8) s += src[(size_t)b * step];
  }
  red[slice][lane] = s;
  __syncthreads();
  if (slice == 0 && live) {
    float r = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) r += red[k][lane];
    dw[((size_t)co * cin + ci) * kk + t] = r;
  }
}

size_t gconv_wgrad_workspace_bytes(const hv_conv_desc* d) {
  GcGeom g;
  if (gc_geom(g, d)) return 0;
  if (sf_eligible(d)) return gc_al((size_t)sf_splits(g) * g.cin * g.kk * 4);
  if (gp_eligible(d)) {
    GpGeom q;
    gp_geom(q, g);
    return gc_al((size_t)g.n * g.cin * q.plane * 2) + gc_al((size_t)g.n * q.nrep * g.cout * q.plane * 2) + gc_al((size_t)g.n * q.nkc * q.ntg * 128 * q.bn * 4);
  }
  const size_t blocks = (size_t)g.n * g.nsplit;
  return gc_al(blocks * g.Rp * g.Pc * 2) + gc_al(blocks * g.Np * g.Pc * 2) + gc_al(blocks * g.Rp * g.Np * 4);
}
size_t gconv_dgrad_workspace_bytes(const hv_conv_desc* d) {
  GcGeom g;
  if (gc_geom(g, d)) return 0;
  const size_t gemm_path = gc_al((size_t)g.Rp * g.Kc * 2) + gc_al((size_t)g.n * g.Pp * g.Kc * 2) + gc_al((size_t)g.n * g.Rp * g.Pp * 2);
  const size_t flipped = gc_al((size_t)g.cout * g.R * 4);
  return gemm_path > flipped ? gemm_path : flipped;
}

int conv2d_wgrad_bf16(const hv_conv_desc* d, const float* dy, float* dw, float* db, void* workspace, cudaStream_t st) {
  HV_CHECK_ARG(d && dy && dw && workspace, "conv2d_wgrad_bf16: null argument");
  GcGeom g;
  int rc = gc_geom(g, d);
  if (rc) return rc;
  char* base = (char*)workspace;
  if (sf_eligible(d)) {
    const int splits = sf_splits(g);
    float* part = reinterpret_cast<float*>(base);
    const bool plain = g.nsrc == 1 && g.src[0].mode == HV_SRC_DIRECT;
    if (plain && g.k == 4) sf_wgrad_kernel<4, true><<<dim3(splits, g.cin), 256, 0, st>>>(dy, part, g, splits);
    else if (plain) sf_wgrad_kernel<0, true><<<dim3(splits, g.cin), 256, 0, st>>>(dy, part, g, splits);
    else sf_wgrad_kernel<0, false><<<dim3(splits, g.cin), 256, 0, st>>>(dy, part, g, splits);
    HV_LAUNCH_CHECK();
    sf_wgrad_reduce_kernel<<<gc_blocks((long long)g.cin * g.kk), 256, 0, st>>>(part, dw, splits, g.cin * g.kk);
    HV_LAUNCH_CHECK();
    if (db) return channel_sum(dy, db, g.n, g.cout, g.P, st);
    return HV_OK;
  }
  if (gp_eligible(d)) {
    GpGeom q;
    gp_geom(q, g);
    __nv_bfloat16* X = (__nv_bfloat16*)base;
    __nv_bfloat16* DY = (__nv_bfloat16*)(base + gc_al((size_t)g.n * g.cin * q.plane * 2));
    float* part = (float*)((char*)DY + gc_al((size_t)g.n * q.nrep * g.cout * q.plane * 2));
    gp_planes_x_kernel<<<gc_blocks((long long)g.n * g.cin * (q.plane >> 3)), 256, 0, st>>>(g, q, X);
    HV_LAUNCH_CHECK();
    gp_planes_dy_kernel<<<gc_blocks((long long)g.n * g.cout * (q.plane >> 3)), 256, 0, st>>>(dy, g, q, DY);
    HV_LAUNCH_CHECK();
    rc = gemm_tc_taps(DY, X, part, g.n, g.cout, g.cin, q.plane, q.tap_off, q.tap_rep, q.nrep, g.kk, q.tpm, q.co8, q.bn, q.nkc, q.kb0, q.kblocks, st);
    if (rc) return rc;
    gp_reduce_dw_kernel<<<(unsigned)((g.cout * g.cin * g.kk + 31) / 32), 256, 0, st>>>(part, dw, g.n * q.nkc, g.cout, g.cin, g.kk, q.tpm, q.ntg, q.co8, q.bn);
    HV_LAUNCH_CHECK();
    if (db) return channel_sum(dy, db, g.n, g.cout, g.P, st);
    return HV_OK;
  }
  const int blocks = g.n * g.nsplit;
  __nv_bfloat16* colT = (__nv_bfloat16*)base;
  __nv_bfloat16* dyb = (__nv_bfloat16*)(base + gc_al((size_t)blocks * g.Rp * g.Pc * 2));
  float* part = (float*)((char*)dyb + gc_al((size_t)blocks * g.Np * g.Pc * 2));
  // rows R .. Rp of colT (padding of the GEMM's M) stay unwritten: they only produce output rows that gc_reduce_dw_kernel never reads
  gc_im2col_kernel<<<gc_blocks((long long)g.n * g.cin * (g.Pp >> 3)), 256, 0, st>>>(g, colT);
  HV_LAUNCH_CHECK();
  gc_cast_dy_kernel<<<gc_blocks((long long)g.n * g.cout * (g.Pp >> 3)), 256, 0, st>>>(dy, dyb, g);
  HV_LAUNCH_CHECK();
  rc = gemm_tc_nt(colT, dyb, part, nullptr, g.Rp, g.Np, g.Pc, blocks, (long long)g.Rp * g.Pc, (long long)g.Np * g.Pc, 0, st);
  if (rc) return rc;
  gc_reduce_dw_kernel<<<gc_blocks((long long)g.R * g.cout), 256, 0, st>>>(part, dw, blocks, g.R, g.Rp, g.cout, g.Np);
  HV_LAUNCH_CHECK();
  if (db) return channel_sum(dy, db, g.n, g.cout, g.P, st);   // bias gradient: fp32, deterministic (train_ops.cu)
  return HV_OK;
}

int conv2d_dgrad_bf16(const hv_conv_desc* d, const float* w, const float* dy, float* dx, void* workspace, cudaStream_t st) {
  HV_CHECK_ARG(d && w && dy && dx && workspace, "conv2d_dgrad_bf16: null argument");
  GcGeom g;
  int rc = gc_geom(g, d);
  if (rc) return rc;
  char* base = (char*)workspace;
  if (sf_eligible(d)) {
    const dim3 grid(gc_blocks((long long)g.hin * g.win), g.cin, g.n);
    if (g.k == 4 && g.stride == 1) sf_dgrad_kernel<4, 1><<<grid, 256, 0, st>>>(w, dy, dx, g);
    else sf_dgrad_kernel<0, 0><<<grid, 256, 0, st>>>(w, dy, dx, g);
    HV_LAUNCH_CHECK();
    return HV_OK;
  }
  if (d->stride == 1 && (d->k == 3 || d->k == 5) && d->pad == (d->k - 1) / 2 * d->dil && d->cin <= 64) {
    // stride-1 'same' convolution (41 of the generator's 47 layers): dx = conv(dy, flipped / transposed filters) on the implicit-GEMM
    // tcgen05 kernel of the forward - no dyT / dcolT operands, no col2im pass.  fp32 accumulation over all taps, ONE rounding to bf16.
    float* wf = reinterpret_cast<float*>(base);
    gc_flip_w_kernel<<<gc_blocks((long long)g.cout * g.cin * g.kk), 256, 0, st>>>(w, wf, g.cout, g.cin, g.kk);
    HV_LAUNCH_CHECK();
    hv_conv_desc t = *d;
    t.cin = d->cout; t.cout = d->cin; t.act = HV_ACT_NONE; t.nsrc = 1;
    t.src[0].ptr = dy; t.src[0].channels = d->cout; t.src[0].mode = HV_SRC_DIRECT;
    return conv2d_bf16(&t, wf, nullptr, dx, nullptr, 0, st);
  }
  __nv_bfloat16* wt = (__nv_bfloat16*)base;
  __nv_bfloat16* dyT = (__nv_bfloat16*)(base + gc_al((size_t)g.Rp * g.Kc * 2));
  __nv_bfloat16* dcolT = (__nv_bfloat16*)((char*)dyT + gc_al((size_t)g.n * g.Pp * g.Kc * 2));
  gc_wt_kernel<<<gc_blocks((long long)g.Rp * g.Kc), 256, 0, st>>>(w, wt, g.cout, g.R, g.Rp, g.Kc);
  HV_LAUNCH_CHECK();
  gc_dyT_kernel<<<dim3(g.Pp / 32, g.Kc / 32, g.n), 256, 0, st>>>(dy, dyT, g.cout, g.Kc, g.P, g.Pp);
  HV_LAUNCH_CHECK();
  rc = gemm_tc_nt(wt, dyT, dcolT, nullptr, g.Rp, g.Pp, g.Kc, g.n, 0, (long long)g.Pp * g.Kc, 1, st);
  if (rc) return rc;
  gc_col2im_kernel<<<gc_blocks((long long)g.n * g.cin * g.hin * ((g.win + 3) >> 2)), 256, 0, st>>>(dcolT, dx, g);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

}  // namespace hv

extern "C" {
size_t hv_conv2d_wgrad_bf16_workspace_bytes(const hv_conv_desc* d) { return hv::gconv_wgrad_workspace_bytes(d); }
size_t hv_conv2d_dgrad_bf16_workspace_bytes(const hv_conv_desc* d) { return hv::gconv_dgrad_workspace_bytes(d); }
int hv_conv2d_wgrad_bf16(const hv_conv_desc* d, const float* dy, float* dw, float* db, void* workspace, hv_stream_t s) {
  return hv::conv2d_wgrad_bf16(d, dy, dw, db, workspace, hv::as_stream(s));
}
int hv_conv2d_dgrad_bf16(const hv_conv_desc* d, const float* w, const float* dy, float* dx, void* workspace, hv_stream_t s) {
  return hv::conv2d_dgrad_bf16(d, w, dy, dx, workspace, hv::as_stream(s));
}
}
