// Backward / training-step kernels of the path (fp32, parity first): convolution data and weight gradients with the
// fused source gather of conv_fp32.cu, activation / upsample / stitch adjoints, spectral-norm backward, the SHRM height
// head backward, BatchNorm(train)+LeakyReLU of the PatchGAN discriminator, the scalar losses of backward_G / backward_D
// (reference models/pix2pix_model.py:267-354, models/networks.py:212-278,:555-602) and a fused Adam step (:127-130).
#include "hv_common.cuh"
#include "kernels.h"

namespace hv {

// ------------------------------------------------------------------ weight flip for the data gradient
// wt[ci][co][k-1-ky][k-1-kx] = w[co][ci][ky][kx]
__global__ void flip_weights_kernel(const float* __restrict__ w, float* __restrict__ wt, int cout, int cin, int k) {
  const int kk = k * k;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * cin * kk) return;
  const int t = i % kk, ci = (i / kk) % cin, co = i / (kk * cin);
  wt[((size_t)ci * cout + co) * kk + (kk - 1 - t)] = w[i];
}

// Sub-pixel weights for the data gradient of a 4x4 stride-2 pad-1 conv: output parity class (py, px) only meets the flipped taps
// a = py + 2 t, b = px + 2 s (the other taps fall on the inserted zeros), i.e. a 2x2 conv over dy itself:
//   ws[(py, px)][ci][co][t][s] = w[co][ci][3 - py - 2 t][3 - px - 2 s]
__global__ void subpixel_weights_kernel(const float* __restrict__ w, float* __restrict__ ws, int cout, int cin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * cin * 16) return;
  const int s = i & 1, t = (i >> 1) & 1, rest = i >> 2;
  const int co = rest % cout, ci = (rest / cout) % cin, cls = rest / (cout * cin), py = cls >> 1, px = cls & 1;
  ws[i] = w[((size_t)co * cin + ci) * 16 + (3 - py - 2 * t) * 4 + (3 - px - 2 * s)];
}

// dx over the VIRTUAL input extent [n, cin, hin, win] of the forward conv described by d (sources concatenated; the caller
// routes channel ranges back to their tensors, see upsample2_bwd for HV_SRC_UP2 sources).  workspace: cin*cout*k*k floats.
int conv2d_dgrad_fp32(const hv_conv_desc* d, const float* w, const float* dy, float* dx, float* workspace, cudaStream_t st) {
  HV_CHECK_ARG(d && w && dy && dx && workspace, "conv2d_dgrad: null argument");
  HV_CHECK_ARG(d->stride == 1 || (d->stride == 2 && d->dil == 1 && (d->hin % 2) == 0 && (d->win % 2) == 0),
               "conv2d_dgrad: stride-2 needs dilation 1 and an even input extent");
  const int eff = (d->k - 1) * d->dil + 1;
  const int hout = (d->hin + 2 * d->pad - eff) / d->stride + 1, wout = (d->win + 2 * d->pad - eff) / d->stride + 1;
  HV_CHECK_ARG(d->stride == 1 || (2 * hout == d->hin && 2 * wout == d->win), "conv2d_dgrad: stride-2 conv must halve the extent");
  const int total = d->cout * d->cin * d->k * d->k;
  if (d->stride == 2 && d->k == 4 && d->pad == 1) {
    // four 2x2 convs over dy, one per output parity class, instead of a 4x4 conv over the zero-inserted dy: a quarter of the
    // multiply-adds, the same non-zero terms in the same order (bit-identical results)
    subpixel_weights_kernel<<<(total + 255) / 256, 256, 0, st>>>(w, workspace, d->cout, d->cin);
    HV_LAUNCH_CHECK();
    hv_conv_desc b;
    b = *d;
    b.cin = d->cout; b.cout = d->cin; b.k = 2; b.stride = 1; b.dil = 1; b.act = HV_ACT_NONE;
    b.nsrc = 1; b.src[0].ptr = dy; b.src[0].channels = d->cout; b.src[0].mode = HV_SRC_DIRECT;
    b.hin = hout; b.win = wout;
    for (int cls = 0; cls < 4; ++cls) {
      const int py = cls >> 1, px = cls & 1;
      b.pad = 1 - py;
      const ConvSubpixel sub{1 - py, 1 - px, 2, py, px, d->hin, d->win};
      int rc = conv2d_fwd_fp32_sub(&b, workspace + (size_t)cls * d->cout * d->cin * 4, nullptr, dx, nullptr, d->hin / 2, d->win / 2, &sub, st);
      if (rc) return rc;
    }
    return HV_OK;
  }
  flip_weights_kernel<<<(total + 255) / 256, 256, 0, st>>>(w, workspace, d->cout, d->cin, d->k);
  HV_LAUNCH_CHECK();
  hv_conv_desc b;
  b = *d;
  b.cin = d->cout; b.cout = d->cin;
  b.nsrc = 1; b.src[0].ptr = dy; b.src[0].channels = d->cout;
  b.act = HV_ACT_NONE;
  b.stride = 1;
  b.pad = (d->k - 1) * d->dil - d->pad;
  HV_CHECK_ARG(b.pad >= 0, "conv2d_dgrad: padding larger than the kernel reach is not supported");
  if (d->stride == 1) { b.src[0].mode = HV_SRC_DIRECT; b.hin = hout; b.win = wout; }
  else { b.src[0].mode = HV_SRC_ZEROINS2; b.hin = 2 * hout; b.win = 2 * wout; }
  return conv2d_fwd_fp32_ex(&b, workspace, nullptr, dx, nullptr, d->hin, d->win, st);
}

// ------------------------------------------------------------------ weight gradient
// dw[co][ci][ky][kx] = sum_{n,oy,ox} dy[n][co][oy][ox] * X(n, ci, oy*s + ky*d - p, ox*s + kx*d - p), X = fused source gather.
// GEMM view: M = co, N = (ci, tap), K = positions.  CTA tile 64 x 64, 32 positions per step, split over K with atomics.
struct WgradArgs {
  hv_conv_src src[4];
  int nsrc;
  const float* dy;
  float* dw;
  int N, Cin, Cout, Hin, Win, Hout, Wout, k, stride, pad, dil;
  int pos_per_split;
};

__device__ __forceinline__ float wg_load(const WgradArgs& p, int n, int ch, int gy, int gx) {
  if (gy < 0 || gy >= p.Hin || gx < 0 || gx >= p.Win) return 0.f;
  int s = 0;
  while (s < p.nsrc - 1 && ch >= p.src[s].channels) { ch -= p.src[s].channels; ++s; }
  const float* sp = p.src[s].ptr;
  const int mode = p.src[s].mode, sch = p.src[s].channels;
  if (mode == HV_SRC_SCALAR) return sp[n];
  int sh = p.Hin, sw = p.Win;
  if (mode == HV_SRC_UP2) { sh >>= 1; sw >>= 1; gy >>= 1; gx >>= 1; }
  else if (mode == HV_SRC_SUB2) { sh <<= 1; sw <<= 1; gy <<= 1; gx <<= 1; }
  return __ldg(sp + (((size_t)n * sch + ch) * sh + gy) * sw + gx);
}

__global__ void __launch_bounds__(256) conv_wgrad_kernel(const WgradArgs p) {
  // tiles of 32 positions: [pos][co] and [pos][col]; rows of 68 floats keep every 4-float group 16-byte aligned (LDS.128)
  __shared__ __align__(16) float s_a[32][68];
  __shared__ __align__(16) float s_b[32][68];
  const int kk = p.k * p.k, ncols = p.Cin * kk;
  const int col0 = blockIdx.x * 64, co0 = blockIdx.y * 64;
  const int hw = p.Hout * p.Wout;
  const long long P = (long long)p.N * hw;
  const long long p_begin = (long long)blockIdx.z * p.pos_per_split;
  const long long p_end = min(P, p_begin + p.pos_per_split);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // Every thread stages position pp = tid % 32 of the tile for rows / columns (tid / 32) + 8 e, e = 0 .. 7: the (ci, ky, kx) of its
  // eight im2col columns never change, and its position advances by 32 per tile, so (n, oy, ox) are carried incrementally -
  // no integer division in the loop (the gather used to cost more than the FMAs).
  const int pp = tid & 31, lane_row = tid >> 5;
  int cci[8], cky[8], ckx[8];
  bool cok[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = col0 + lane_row + 8 * e;
    cok[e] = c < ncols;
    const int ci = cok[e] ? c / kk : 0, t = cok[e] ? c - ci * kk : 0;
    cci[e] = ci; cky[e] = (t / p.k) * p.dil - p.pad; ckx[e] = (t % p.k) * p.dil - p.pad;
  }
  long long pos = p_begin + pp;
  int n = (int)(pos / hw), r = (int)(pos - (long long)n * hw);
  int oy = r / p.Wout, ox = r - oy * p.Wout;

  // software pipeline: the global loads of tile t + 1 are issued before the FMAs of tile t (registers ra / rb carry them over)
  float ra[8], rb[8];
  auto fetch = [&]() {
    const bool live = pos < p_end;
#pragma unroll
    for (int e = 0; e < 8; ++e) {   // dy tile: 64 co x 32 positions (positions contiguous inside a (n, co) plane)
      const int co = lane_row + 8 * e;
      ra[e] = (live && co0 + co < p.Cout) ? __ldg(p.dy + ((size_t)n * p.Cout + co0 + co) * hw + r) : 0.f;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e)     // im2col tile: 64 (ci, tap) x 32 positions
      rb[e] = (live && cok[e]) ? wg_load(p, n, cci[e], oy * p.stride + cky[e], ox * p.stride + ckx[e]) : 0.f;
  };
  fetch();
  for (long long p0 = p_begin; p0 < p_end; p0 += 32) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { s_a[pp][lane_row + 8 * e] = ra[e]; s_b[pp][lane_row + 8 * e] = rb[e]; }
    __syncthreads();
    // next tile: the same lane, 32 positions further
    pos += 32; r += 32; ox += 32;
    while (r >= hw) { r -= hw; ++n; }
    if (ox >= p.Wout) { const int rows = ox / p.Wout; ox -= rows * p.Wout; oy += rows; }   // rare: once per output row
    while (oy >= p.Hout) oy -= p.Hout;
    if (p0 + 32 < p_end) fetch();
#pragma unroll 8
    for (int q = 0; q < 32; ++q) {
      const float4 a4 = *reinterpret_cast<const float4*>(&s_a[q][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&s_b[q][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty * 4 + i;
    if (co >= p.Cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = col0 + tx * 4 + j;
      if (c < ncols) atomicAdd(p.dw + (size_t)co * ncols + c, acc[i][j]);
    }
  }
}

// per-channel sum over (n, hw): db[c] = sum dy[n][c][:]  (bias gradient, BatchNorm sums).  Two deterministic passes: block
// (split, channel) sums one slice of the channel's n * hw elements, then one thread per channel adds the slices in a fixed order
// (a single block per channel left a 1-filter head layer reading 4 MB through one CTA: 578 us per call, 10 % of a training step).
constexpr int kSumSlice = 8192;   // elements per block
__global__ void __launch_bounds__(256) channel_sum_partial_kernel(const float* __restrict__ x, float* __restrict__ partial, int n, int c, int hw) {
  __shared__ float red[32];
  const int ch = blockIdx.y, split = blockIdx.x;
  const long long total = (long long)n * hw, lo = (long long)split * kSumSlice, hi = min(total, lo + kSumSlice);
  float s = 0.f;
  long long e = lo + threadIdx.x;
  long long i = e / hw;
  int j = (int)(e - i * hw);
  for (; e < hi; e += blockDim.x) {
    s += x[((size_t)i * c + ch) * hw + j];
    j += blockDim.x;
    while (j >= hw) { j -= hw; ++i; }
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) partial[(size_t)split * c + ch] = s;
}
__global__ void channel_sum_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int splits, int c) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(size_t)k * c + ch];
  out[ch] = s;
}
static int channel_sum_launch(const float* x, float* out, int n, int c, int hw, cudaStream_t st) {
  const long long total = (long long)n * hw;
  const int splits = (int)((total + kSumSlice - 1) / kSumSlice);
  // scratch for the slice sums: one grow-only buffer per (device, stream) (stream order keeps successive calls from overlapping).
  // cudaMallocAsync per call cost more than the kernels (step 340 -> 448 ms).
  const size_t need = (size_t)splits * c;
  float* partial = static_cast<float*>(stream_scratch(st, sizeof(float) * need + 256)) ;
  HV_CHECK_ARG(partial, "channel_sum: scratch allocation failed");
  partial += 64;   // the first 256 bytes of the stream's scratch belong to the scalar reductions (edge loss)
  channel_sum_partial_kernel<<<dim3(splits, c), 256, 0, st>>>(x, partial, n, c, hw);
  HV_LAUNCH_CHECK();
  channel_sum_final_kernel<<<(c + 127) / 128, 128, 0, st>>>(partial, out, splits, c);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

int channel_sum(const float* x, float* out, int n, int c, int hw, cudaStream_t st) { return channel_sum_launch(x, out, n, c, hw, st); }

int conv2d_wgrad_fp32(const hv_conv_desc* d, const float* dy, float* dw, float* db, cudaStream_t st) {
  HV_CHECK_ARG(d && dy && dw, "conv2d_wgrad: null argument");
  HV_CHECK_ARG(d->nsrc >= 1 && d->nsrc <= 4, "conv2d_wgrad: nsrc out of range");
  WgradArgs a;
  int csum = 0;
  for (int i = 0; i < 4; ++i) {
    a.src[i] = d->src[i < d->nsrc ? i : 0];
    if (i < d->nsrc) csum += d->src[i].channels;
  }
  HV_CHECK_ARG(csum == d->cin, "conv2d_wgrad: sources have %d channels, cin=%d", csum, d->cin);
  a.nsrc = d->nsrc; a.dy = dy; a.dw = dw;
  a.N = d->n; a.Cin = d->cin; a.Cout = d->cout; a.Hin = d->hin; a.Win = d->win;
  a.k = d->k; a.stride = d->stride; a.pad = d->pad; a.dil = d->dil;
  const int eff = (d->k - 1) * d->dil + 1;
  a.Hout = (d->hin + 2 * d->pad - eff) / d->stride + 1;
  a.Wout = (d->win + 2 * d->pad - eff) / d->stride + 1;
  const int ncols = d->cin * d->k * d->k;
  const long long P = (long long)d->n * a.Hout * a.Wout;
  const int tiles = ((ncols + 63) / 64) * ((d->cout + 63) / 64);
  int splits = (int)max(1ll, min((long long)(148 * 8 / max(tiles, 1)), (P + 1023) / 1024));
  long long per = (P + splits - 1) / splits;
  per = (per + 31) / 32 * 32;
  splits = (int)((P + per - 1) / per);
  a.pos_per_split = (int)per;
  HV_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)d->cout * ncols, st));
  dim3 grid((ncols + 63) / 64, (d->cout + 63) / 64, splits);
  conv_wgrad_kernel<<<grid, 256, 0, st>>>(a);
  HV_LAUNCH_CHECK();
  if (db) {
    int rc = channel_sum_launch(dy, db, d->n, d->cout, a.Hout * a.Wout, st);
    if (rc) return rc;
  }
  return HV_OK;
}

// ------------------------------------------------------------------ elementwise adjoints
// dx = dy * act'(.) expressed through the activation OUTPUT (ELU: out > 0 ? 1 : out + 1; clamp: inside (-1, 1))
__global__ void act_bwd_kernel(const float* __restrict__ out, const float* __restrict__ dy, float* __restrict__ dx, int act, size_t count) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) {
    const float o = out[i], g = dy[i];
    float d;
    switch (act) {
      case HV_ACT_ELU: d = o > 0.f ? 1.f : o + 1.f; break;
      case HV_ACT_RELU: d = o > 0.f ? 1.f : 0.f; break;
      case HV_ACT_SIGMOID: d = o * (1.f - o); break;
      case HV_ACT_LRELU02: d = o > 0.f ? 1.f : 0.2f; break;
      case HV_ACT_CLAMP1: d = (o > -1.f && o < 1.f) ? 1.f : 0.f; break;
      default: d = 1.f;
    }
    dx[i] = g * d;
  }
}

static int ew_blocks(size_t count) {
  size_t b = (count + 255) / 256;
  return (int)(b > 148 * 16 ? 148 * 16 : (b ? b : 1));
}

int act_bwd(const float* out, const float* dy, float* dx, int act, size_t count, cudaStream_t st) {
  HV_CHECK_ARG(out && dy && dx, "act_bwd: null argument");
  act_bwd_kernel<<<ew_blocks(count), 256, 0, st>>>(out, dy, dx, act, count);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// dx = dy * act'(out) AND db[c] = sum over (n, hw) of dx, in ONE pass over the tensors (the bias gradient of a conv block is the channel
// sum of its pre-activation gradient: computing it separately re-reads dx: ~1 ms per training step over 47 layers).  Same two-pass,
// deterministic slice scheme as channel_sum.
__device__ __forceinline__ float act_deriv(float o, int act) {
  switch (act) {
    case HV_ACT_ELU: return o > 0.f ? 1.f : o + 1.f;
    case HV_ACT_RELU: return o > 0.f ? 1.f : 0.f;
    case HV_ACT_SIGMOID: return o * (1.f - o);
    case HV_ACT_LRELU02: return o > 0.f ? 1.f : 0.2f;
    case HV_ACT_CLAMP1: return (o > -1.f && o < 1.f) ? 1.f : 0.f;
    default: return 1.f;
  }
}
__global__ void __launch_bounds__(256) act_bwd_bias_kernel(const float* __restrict__ out, const float* __restrict__ dy, float* __restrict__ dx,
                                                           float* __restrict__ partial, int act, int n, int c, int hw) {
  __shared__ float red[32];
  const int ch = blockIdx.y, split = blockIdx.x;
  const long long total = (long long)n * hw, lo = (long long)split * kSumSlice, hi = min(total, lo + kSumSlice);
  float s = 0.f;
  long long e = lo + threadIdx.x;
  long long i = e / hw;
  int j = (int)(e - i * hw);
  for (; e < hi; e += blockDim.x) {
    const size_t at = ((size_t)i * c + ch) * hw + j;
    const float v = dy[at] * act_deriv(out[at], act);
    dx[at] = v;
    s += v;
    j += blockDim.x;
    while (j >= hw) { j -= hw; ++i; }
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) partial[(size_t)split * c + ch] = s;
}

int act_bwd_bias(const float* out, const float* dy, float* dx, float* db, int act, int n, int c, int hw, cudaStream_t st) {
  HV_CHECK_ARG(out && dy && dx && db && n > 0 && c > 0 && c <= 65535 && hw > 0, "act_bwd_bias: bad argument");
  const long long total = (long long)n * hw;
  const int splits = (int)((total + kSumSlice - 1) / kSumSlice);
  float* partial = static_cast<float*>(stream_scratch(st, sizeof(float) * (size_t)splits * c + 256));
  HV_CHECK_ARG(partial, "act_bwd_bias: scratch allocation failed");
  partial += 64;
  act_bwd_bias_kernel<<<dim3(splits, c), 256, 0, st>>>(out, dy, dx, partial, act, n, c, hw);
  HV_LAUNCH_CHECK();
  channel_sum_final_kernel<<<(c + 127) / 128, 128, 0, st>>>(partial, db, splits, c);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// adjoint of the nearest x2 upsample: dx[n][c][y][x] = sum of the 2x2 block of dy (dy has channel stride `dy_cstride`
// planes per image so that a channel range of a concatenated gradient can be read in place)
__global__ void upsample2_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int c, int h, int w, int dy_channels,
                                     int dy_ch0, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int x = i % w, y = (i / w) % h, ch = (i / ((size_t)w * h)) % c, n = i / ((size_t)w * h * c);
    const float* p = dy + (((size_t)n * dy_channels + dy_ch0 + ch) * (2 * h) + 2 * y) * (2 * w) + 2 * x;
    dx[i] = (p[0] + p[1]) + (p[2 * w] + p[2 * w + 1]);
  }
}

int upsample2_bwd(const float* dy, float* dx, int n, int c, int h, int w, int dy_channels, int dy_ch0, cudaStream_t st) {
  HV_CHECK_ARG(dy && dx && n > 0 && c > 0 && dy_ch0 >= 0 && dy_ch0 + c <= dy_channels, "upsample2_bwd: bad argument");
  const size_t total = (size_t)n * c * h * w;
  upsample2_bwd_kernel<<<ew_blocks(total), 256, 0, st>>>(dy, dx, c, h, w, dy_channels, dy_ch0, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// adjoint of the height-adaptive stitch w.r.t. the generated image: rows [xu, xb) pass, the rest is real data
__global__ void stitch_bwd_kernel(const float* __restrict__ dout, const int32_t* __restrict__ rows, float* __restrict__ dgen, int h, int w, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int y = (i / w) % h, n = i / ((size_t)w * h);
    const int xu = rows[n * 4 + 2], xb = rows[n * 4 + 3];
    dgen[i] = (y >= xu && y < xb) ? dout[i] : 0.f;
  }
}

int stitch_bwd(const float* dout, const int32_t* rows, float* dgen, int n, int h, int w, cudaStream_t st) {
  HV_CHECK_ARG(dout && rows && dgen, "stitch_bwd: null argument");
  const size_t total = (size_t)n * h * w;
  stitch_bwd_kernel<<<ew_blocks(total), 256, 0, st>>>(dout, rows, dgen, h, w, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// y = a * x + b * y  (gradient accumulation / scaling), x may be null (y *= b)
__global__ void axpby_kernel(float a, const float* __restrict__ x, float b, float* __restrict__ y, size_t count) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) y[i] = (x ? a * x[i] : 0.f) + b * y[i];
}

int axpby(float a, const float* x, float b, float* y, size_t count, cudaStream_t st) {
  HV_CHECK_ARG(y, "axpby: null argument");
  axpby_kernel<<<ew_blocks(count), 256, 0, st>>>(a, x, b, y, count);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// y = a * x + c
__global__ void affine_kernel(float a, const float* __restrict__ x, float c, float* __restrict__ y, size_t count) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) y[i] = a * x[i] + c;
}

int affine(float a, const float* x, float c, float* y, size_t count, cudaStream_t st) {
  HV_CHECK_ARG(x && y, "affine: null argument");
  affine_kernel<<<ew_blocks(count), 256, 0, st>>>(a, x, c, y, count);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// loss_h = mean_i(40 |m p1_i - h_i| / h_i + 40 |m p2_i - h_i| / h_i)  (pix2pix_model.py:191-192,:350); one small CTA
__global__ void __launch_bounds__(256) height_loss_kernel(const float* __restrict__ p1, const float* __restrict__ p2, const float* __restrict__ h,
                                                          float maxh, int n, float* __restrict__ loss, float* __restrict__ dp1,
                                                          float* __restrict__ dp2) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float hi = h[i], a = maxh * p1[i] - hi, b = maxh * p2[i] - hi;
    acc += 40.f * (fabsf(a) + fabsf(b)) / hi;
    const float g = 40.f * maxh / (hi * (float)n);
    if (dp1) dp1[i] = a > 0.f ? g : (a < 0.f ? -g : 0.f);
    if (dp2) dp2[i] = b > 0.f ? g : (b < 0.f ? -g : 0.f);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) loss[0] = acc / (float)n;
}

int height_loss(const float* p1, const float* p2, const float* h, float maxh, int n, float* loss, float* dp1, float* dp2, cudaStream_t st) {
  HV_CHECK_ARG(p1 && p2 && h && loss && n > 0, "height_loss: bad argument");
  height_loss_kernel<<<1, 256, 0, st>>>(p1, p2, h, maxh, n, loss, dp1, dp2);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// out = x * mask * [col in [c0, c1)]   (fake_B_local / real_B_local, pix2pix_model.py:254-260; also its own adjoint)
__global__ void masked_center_kernel(const float* __restrict__ x, const float* __restrict__ mask, float* __restrict__ out, int w, int c0, int c1, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int col = i % w;
    out[i] = (col >= c0 && col < c1) ? x[i] * mask[i] : 0.f;
  }
}

int masked_center(const float* x, const float* mask, float* out, int w, int c0, int c1, size_t total, cudaStream_t st) {
  HV_CHECK_ARG(x && mask && out, "masked_center: null argument");
  masked_center_kernel<<<ew_blocks(total), 256, 0, st>>>(x, mask, out, w, c0, c1, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ spectral-norm backward (spectral_norm.py:92-114)
// W_eff = W / sigma, sigma = u^T W v with u, v constants:  dW = (dW_eff - <dW_eff, W_eff> u v^T) / sigma
__global__ void __launch_bounds__(512) sn_bwd_kernel(const float* __restrict__ dweff, const float* __restrict__ weff,
                                                     const float* __restrict__ u, const float* __restrict__ v,
                                                     const float* __restrict__ sigma, float* __restrict__ dw, int cout, int kdim) {
  __shared__ float red[32];
  const int total = cout * kdim;
  float dot = 0.f;
  for (int i = threadIdx.x; i < total; i += blockDim.x) dot = fmaf(dweff[i], weff[i], dot);
  dot = block_sum(dot, red);
  const float inv = 1.f / sigma[0];
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    const int r = i / kdim, c = i - r * kdim;
    dw[i] = (dweff[i] - dot * u[r] * v[c]) * inv;
  }
}

int sn_bwd(const float* dweff, const float* weff, const float* u, const float* v, const float* sigma, float* dw, int cout, int kdim, cudaStream_t st) {
  HV_CHECK_ARG(dweff && weff && u && v && sigma && dw, "sn_bwd: null argument");
  sn_bwd_kernel<<<1, 512, 0, st>>>(dweff, weff, u, v, sigma, dw, cout, kdim);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// all layers of a net in one launch (one CTA per layer): rows of seven 64-bit words {dweff, weff, u, v, sigma, dw, cout | kdim << 32}
struct SnBwdJob { const float* dweff; const float* weff; const float* u; const float* v; const float* sigma; float* dw; int cout, kdim; };
__global__ void __launch_bounds__(512) sn_bwd_multi_kernel(const SnBwdJob* __restrict__ jobs) {
  const SnBwdJob j = jobs[blockIdx.x];
  __shared__ float red[32];
  const int total = j.cout * j.kdim;
  float dot = 0.f;
  for (int i = threadIdx.x; i < total; i += blockDim.x) dot = fmaf(j.dweff[i], j.weff[i], dot);
  dot = block_sum(dot, red);
  const float inv = 1.f / j.sigma[0];
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    const int r = i / j.kdim, c = i - r * j.kdim;
    j.dw[i] = (j.dweff[i] - dot * j.u[r] * j.v[c]) * inv;
  }
}

int sn_bwd_multi(const void* d_jobs, int njobs, cudaStream_t st) {
  HV_CHECK_ARG(d_jobs && njobs > 0, "sn_bwd_multi: bad argument");
  sn_bwd_multi_kernel<<<njobs, 512, 0, st>>>(static_cast<const SnBwdJob*>(d_jobs));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ SHRM height head backward (:90-93,:211-214)
// s = sigmoid(fc(mean_HW(x))): dx[n][c][:] = ds[n] s(1-s) w[c] / HW ; dw[c] = sum_n ds s(1-s) mean[n][c] ; db = sum_n ds s(1-s)
__global__ void __launch_bounds__(256) gap_fc_bwd_dx_kernel(const float* __restrict__ s, const float* __restrict__ ds,
                                                            const float* __restrict__ fw, float* __restrict__ dx, int c, int hw, int accumulate) {
  const int n = blockIdx.y, ch = blockIdx.x;
  const float g = ds[n] * s[n] * (1.f - s[n]) * fw[ch] / (float)hw;
  float* p = dx + ((size_t)n * c + ch) * hw;
  for (int i = threadIdx.x; i < hw; i += blockDim.x) p[i] = accumulate ? p[i] + g : g;
}

__global__ void __launch_bounds__(256) gap_fc_bwd_w_kernel(const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ ds,
                                                           float* __restrict__ dfw, float* __restrict__ dfb, int n, int c, int hw) {
  __shared__ float red[32];
  const int ch = blockIdx.x;
  float acc = 0.f;
  for (int i = 0; i < n; ++i) {
    const float g = ds[i] * s[i] * (1.f - s[i]);
    const float* p = x + ((size_t)i * c + ch) * hw;
    float m = 0.f;
    for (int j = threadIdx.x; j < hw; j += blockDim.x) m += p[j];
    acc += g * m;
  }
  acc = block_sum(acc, red) / (float)hw;
  if (threadIdx.x == 0) {
    dfw[ch] = acc;
    if (ch == 0) {
      float b = 0.f;
      for (int i = 0; i < n; ++i) b += ds[i] * s[i] * (1.f - s[i]);
      dfb[0] = b;
    }
  }
}

int gap_fc_sigmoid_bwd(const float* x, const float* s, const float* ds, const float* fw, float* dx, int accumulate, float* dfw,
                       float* dfb, int n, int c, int hw, cudaStream_t st) {
  HV_CHECK_ARG(x && s && ds && fw && dx && dfw && dfb, "gap_fc_sigmoid_bwd: null argument");
  gap_fc_bwd_dx_kernel<<<dim3(c, n), 256, 0, st>>>(s, ds, fw, dx, c, hw, accumulate);
  HV_LAUNCH_CHECK();
  gap_fc_bwd_w_kernel<<<c, 256, 0, st>>>(x, s, ds, dfw, dfb, n, c, hw);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ BatchNorm2d (train) + LeakyReLU (networks.py:583-597)
// stats[c] = (mean, invstd) of the batch; running stats: momentum update with the unbiased variance (torch semantics)
// One CTA per channel (two passes: mean, then centred squares - torch's numerics); 16-byte loads with four independent accumulators
// per thread keep enough bytes in flight for a channel's n * hw * 4 B (the scalar version ran at 0.06 of the HBM peak).
__device__ __forceinline__ bool bn_vec_ok(const float* x, int hw) { return (hw & 3) == 0 && (reinterpret_cast<size_t>(x) & 15) == 0; }

__global__ void __launch_bounds__(512) bn_stats_kernel(const float* __restrict__ x, float* __restrict__ save_mean, float* __restrict__ save_invstd,
                                                       float* __restrict__ running_mean, float* __restrict__ running_var, int n, int c,
                                                       int hw, float momentum, float eps) {
  __shared__ float red[32];
  const int ch = blockIdx.x;
  const float cnt = (float)n * hw;
  const bool vec = bn_vec_ok(x, hw);
  float s = 0.f;
  for (int i = 0; i < n && !vec; ++i) {
    const float* p = x + ((size_t)i * c + ch) * hw;
    for (int j = threadIdx.x; j < hw; j += blockDim.x) s += p[j];
  }
  if (vec) {
    // one CTA per channel: four independent 16-byte loads in flight per thread (a single load per iteration left the CTA latency-bound:
    // 25 us for a 33 MB tensor)
    const int hw4 = hw >> 2, total4 = n * hw4;
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    for (int e0 = threadIdx.x; e0 < total4; e0 += 4 * blockDim.x) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * blockDim.x;
        const int i = e / hw4, j = e - i * hw4;
        v[u] = e < total4 ? __ldg(reinterpret_cast<const float4*>(x + ((size_t)i * c + ch) * hw) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] += (v[u].x + v[u].y) + (v[u].z + v[u].w);
    }
    s = (a[0] + a[1]) + (a[2] + a[3]);
  }
  const float mean = block_sum(s, red) / cnt;
  float q = 0.f;
  for (int i = 0; i < n && !vec; ++i) {
    const float* p = x + ((size_t)i * c + ch) * hw;
    for (int j = threadIdx.x; j < hw; j += blockDim.x) { const float d = p[j] - mean; q = fmaf(d, d, q); }
  }
  if (vec) {
    const int hw4 = hw >> 2, total4 = n * hw4;
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    for (int e0 = threadIdx.x; e0 < total4; e0 += 4 * blockDim.x) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * blockDim.x;
        const int i = e / hw4, j = e - i * hw4;
        v[u] = e < total4 ? __ldg(reinterpret_cast<const float4*>(x + ((size_t)i * c + ch) * hw) + j) : make_float4(mean, mean, mean, mean);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float d0 = v[u].x - mean, d1 = v[u].y - mean, d2 = v[u].z - mean, d3 = v[u].w - mean;
        a[u] += fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3);
      }
    }
    q = (a[0] + a[1]) + (a[2] + a[3]);
  }
  const float var = block_sum(q, red) / cnt;
  if (threadIdx.x == 0) {
    save_mean[ch] = mean;
    save_invstd[ch] = rsqrtf(var + eps);
    if (running_mean) {
      running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * mean;
      running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * var * cnt / fmaxf(cnt - 1.f, 1.f);
    }
  }
}

__global__ void bn_lrelu_apply_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ mean, const float* __restrict__ invstd, float* __restrict__ y, int c,
                                      int hw, float slope, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int ch = (i / hw) % c;
    const float v = (x[i] - mean[ch]) * invstd[ch] * gamma[ch] + beta[ch];
    y[i] = v > 0.f ? v : slope * v;
  }
}

int bn_lrelu_fwd(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var, float* y,
                 float* save_mean, float* save_invstd, int n, int c, int hw, float momentum, float eps, float slope, cudaStream_t st) {
  HV_CHECK_ARG(x && gamma && beta && y && save_mean && save_invstd, "bn_lrelu_fwd: null argument");
  bn_stats_kernel<<<c, 512, 0, st>>>(x, save_mean, save_invstd, running_mean, running_var, n, c, hw, momentum, eps);
  HV_LAUNCH_CHECK();
  const size_t total = (size_t)n * c * hw;
  bn_lrelu_apply_kernel<<<ew_blocks(total), 256, 0, st>>>(x, gamma, beta, save_mean, save_invstd, y, c, hw, slope, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// backward: g = dy * lrelu'(y);  dbeta = sum g;  dgamma = sum g * xhat;  dx = gamma*invstd*(g - dbeta/M - xhat*dgamma/M)
__global__ void __launch_bounds__(512) bn_bwd_reduce_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ dy,
                                                            const float* __restrict__ mean, const float* __restrict__ invstd,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta, int n, int c, int hw, float slope) {
  __shared__ float red[32];
  const int ch = blockIdx.x;
  const float m = mean[ch], is = invstd[ch];
  float sg = 0.f, sgx = 0.f;
  const bool vec = bn_vec_ok(x, hw) && bn_vec_ok(y, hw) && bn_vec_ok(dy, hw);
  for (int i = 0; i < n; ++i) {
    const size_t base = ((size_t)i * c + ch) * hw;
    if (vec) {
      const float4 *x4 = reinterpret_cast<const float4*>(x + base), *y4 = reinterpret_cast<const float4*>(y + base),
                   *d4 = reinterpret_cast<const float4*>(dy + base);
      for (int j = threadIdx.x; j < hw / 4; j += blockDim.x) {
        const float4 xv = __ldg(x4 + j), yv = __ldg(y4 + j), dv = __ldg(d4 + j);
        const float g0 = dv.x * (yv.x > 0.f ? 1.f : slope), g1 = dv.y * (yv.y > 0.f ? 1.f : slope), g2 = dv.z * (yv.z > 0.f ? 1.f : slope),
                    g3 = dv.w * (yv.w > 0.f ? 1.f : slope);
        sg += (g0 + g1) + (g2 + g3);
        sgx = fmaf(g0, (xv.x - m) * is, sgx); sgx = fmaf(g1, (xv.y - m) * is, sgx);
        sgx = fmaf(g2, (xv.z - m) * is, sgx); sgx = fmaf(g3, (xv.w - m) * is, sgx);
      }
    } else {
      for (int j = threadIdx.x; j < hw; j += blockDim.x) {
        const float g = dy[base + j] * (y[base + j] > 0.f ? 1.f : slope);
        sg += g;
        sgx = fmaf(g, (x[base + j] - m) * is, sgx);
      }
    }
  }
  sg = block_sum(sg, red);
  sgx = block_sum(sgx, red);
  if (threadIdx.x == 0) { dbeta[ch] = sg; dgamma[ch] = sgx; }
}

__global__ void bn_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ dy,
                                    const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ invstd,
                                    const float* __restrict__ dgamma, const float* __restrict__ dbeta, float* __restrict__ dx, int c, int hw,
                                    float inv_count, float slope, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int ch = (i / hw) % c;
    const float g = dy[i] * (y[i] > 0.f ? 1.f : slope);
    const float xhat = (x[i] - mean[ch]) * invstd[ch];
    dx[i] = gamma[ch] * invstd[ch] * (g - dbeta[ch] * inv_count - xhat * dgamma[ch] * inv_count);
  }
}

int bn_lrelu_bwd(const float* x, const float* y, const float* dy, const float* gamma, const float* save_mean, const float* save_invstd,
                 float* dx, float* dgamma, float* dbeta, int n, int c, int hw, float slope, cudaStream_t st) {
  HV_CHECK_ARG(x && y && dy && gamma && save_mean && save_invstd && dx && dgamma && dbeta, "bn_lrelu_bwd: null argument");
  bn_bwd_reduce_kernel<<<c, 512, 0, st>>>(x, y, dy, save_mean, save_invstd, dgamma, dbeta, n, c, hw, slope);
  HV_LAUNCH_CHECK();
  const size_t total = (size_t)n * c * hw;
  bn_bwd_apply_kernel<<<ew_blocks(total), 256, 0, st>>>(x, y, dy, gamma, save_mean, save_invstd, dgamma, dbeta, dx, c, hw,
                                                        1.f / ((float)n * hw), slope, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ scalar losses (two-stage deterministic reductions)
// kind: 0 sum|a-b|  1 BCE-with-logits vs constant target t (a = logits, b unused)  2 count_nonzero(a)
//       3 sum a  4 sum a*b  5 sum (a-t)^2 (b unused)
__global__ void __launch_bounds__(256) reduce_partial_kernel(const float* __restrict__ a, const float* __restrict__ b, float t, int kind,
                                                             size_t count, float* __restrict__ partial) {
  __shared__ float red[32];
  float s = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const float x = a[i];
    switch (kind) {
      case 0: s += fabsf(x - b[i]); break;
      case 1: s += fmaxf(x, 0.f) - x * t + log1pf(expf(-fabsf(x))); break;
      case 2: s += x != 0.f ? 1.f : 0.f; break;
      case 3: s += x; break;
      case 4: s += x * b[i]; break;
      case 5: { const float d = x - t; s += d * d; } break;
    }
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(256) reduce_final_kernel(const float* __restrict__ partial, int nparts, float scale, float* __restrict__ out) {
  __shared__ float red[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) s += partial[i];
  s = block_sum(s, red);
  if (threadIdx.x == 0) out[0] = s * scale;
}

// out[0] = scale * reduce(kind);  scratch: 1024 floats
int reduce_scalar(const float* a, const float* b, float t, int kind, size_t count, float scale, float* out, float* scratch, cudaStream_t st) {
  HV_CHECK_ARG(kind >= 0 && kind <= 5, "reduce_scalar: kind %d is not one of 0..5", kind);
  HV_CHECK_ARG(a && out && scratch && ((kind != 0 && kind != 4) || b), "reduce_scalar: null argument");
  int blocks = (int)((count + 255) / 256);
  if (blocks > 1024) blocks = 1024;
  if (blocks < 1) blocks = 1;
  reduce_partial_kernel<<<blocks, 256, 0, st>>>(a, b, t, kind, count, scratch);
  HV_LAUNCH_CHECK();
  reduce_final_kernel<<<1, 256, 0, st>>>(scratch, blocks, scale, out);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// gradients of the elementwise losses, gg = g * S:  kind 0: da = gg * sign(a - b);  1: da = gg * (sigmoid(a) - t);
// 2: da = gg * 2 (a - t);  3: da = gg (a is not read).  S = 1, scale[0] or 1 / scale[0]: `scale` is an
// optional DEVICE scalar multiplier, e.g. 256*256 / count_nonzero(mask); accumulate adds into da
__global__ void loss_grad_kernel(const float* __restrict__ a, const float* __restrict__ b, float t, int kind, float g, const float* __restrict__ scale,
                                 int scale_is_reciprocal, float* __restrict__ da, int accumulate, size_t count) {
  float gg = g;
  if (scale) gg *= scale_is_reciprocal ? 1.f / scale[0] : scale[0];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) {
    float d;
    switch (kind) {
      case 0: { const float df = a[i] - b[i]; d = df > 0.f ? gg : (df < 0.f ? -gg : 0.f); } break;
      case 1: d = gg * (1.f / (1.f + expf(-a[i])) - t); break;
      case 2: d = gg * (2.f * (a[i] - t)); break;
      default: d = gg; break;   // 3 (loss_grad checks the range)
    }
    da[i] = accumulate ? da[i] + d : d;
  }
}

int loss_grad(const float* a, const float* b, float t, int kind, float g, const float* scale, int scale_is_reciprocal, float* da,
              int accumulate, size_t count, cudaStream_t st) {
  HV_CHECK_ARG(kind >= 0 && kind <= 3, "loss_grad: kind %d is not one of 0..3", kind);
  HV_CHECK_ARG(a && da && (kind != 0 || b), "loss_grad: null argument");
  loss_grad_kernel<<<ew_blocks(count), 256, 0, st>>>(a, b, t, kind, g, scale, scale_is_reciprocal, da, accumulate, count);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// Dice (pix2pix_model.py:13-39, activation 'none'): per sample (2 sum(g p) + eps) / (sum p + sum g + eps); out = mean over samples.
// sums[n][3] = (tp, sum p, sum g) are kept for the backward: d dice_n / d p = (2 g D - (2 tp + eps)) / D^2, D = sum p + sum g + eps
__global__ void __launch_bounds__(512) dice_fwd_kernel(const float* __restrict__ pred, const float* __restrict__ gt, float* __restrict__ sums,
                                                       int per, float eps, float* __restrict__ dice_n) {
  __shared__ float red[32];
  const int n = blockIdx.x;
  const float* p = pred + (size_t)n * per;
  const float* g = gt + (size_t)n * per;
  float tp = 0.f, sp = 0.f, sg = 0.f;
  for (int i = threadIdx.x; i < per; i += blockDim.x) { tp = fmaf(g[i], p[i], tp); sp += p[i]; sg += g[i]; }
  tp = block_sum(tp, red); sp = block_sum(sp, red); sg = block_sum(sg, red);
  if (threadIdx.x == 0) {
    sums[n * 3 + 0] = tp; sums[n * 3 + 1] = sp; sums[n * 3 + 2] = sg;
    dice_n[n] = (2.f * tp + eps) / (sp + sg + eps);
  }
}

__global__ void dice_bwd_kernel(const float* __restrict__ gt, const float* __restrict__ sums, float g_out, float eps, float* __restrict__ dpred,
                                int per, int accumulate, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int n = i / per;
    const float tp = sums[n * 3], D = sums[n * 3 + 1] + sums[n * 3 + 2] + eps;
    const float d = g_out * (2.f * gt[i] * D - (2.f * tp + eps)) / (D * D);
    dpred[i] = accumulate ? dpred[i] + d : d;
  }
}

int dice_fwd(const float* pred, const float* gt, float* sums, float* dice_n, int n, int per, float eps, cudaStream_t st) {
  HV_CHECK_ARG(pred && gt && sums && dice_n, "dice_fwd: null argument");
  dice_fwd_kernel<<<n, 512, 0, st>>>(pred, gt, sums, per, eps, dice_n);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// g_out = d loss / d dice_n (the same for every sample: -weight / N)
int dice_bwd(const float* gt, const float* sums, float g_out, float eps, float* dpred, int n, int per, int accumulate, cudaStream_t st) {
  HV_CHECK_ARG(gt && sums && dpred, "dice_bwd: null argument");
  const size_t total = (size_t)n * per;
  dice_bwd_kernel<<<ew_blocks(total), 256, 0, st>>>(gt, sums, g_out, eps, dpred, per, accumulate, total);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ fused Adam (torch.optim.Adam, no weight decay / amsgrad)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t count,
                            float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

int adam_step(float* p, const float* g, float* m, float* v, size_t count, float lr, float b1, float b2, float eps, int step, cudaStream_t st) {
  HV_CHECK_ARG(p && g && m && v && step >= 1, "adam_step: bad argument");
  const float bc1 = 1.f - powf(b1, (float)step), bc2 = 1.f - powf(b2, (float)step);
  adam_kernel<<<ew_blocks(count), 256, 0, st>>>(p, g, m, v, count, lr, b1, b2, eps, bc1, sqrtf(bc2));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

// ------------------------------------------------------------------ multi-tensor variants: ONE launch per optimiser / gradient bucket
// table rows (device, int64): {p, g, m, v, count, first_chunk} for Adam; {ptr, -, -, -, count, first_chunk} + flat offset = first_chunk *
// MT_CHUNK for the gradient bucket (every tensor starts on a chunk boundary of the flat buffer).  A CTA owns one MT_CHUNK-element chunk
// and finds its tensor by bisection over first_chunk.
constexpr int MT_CHUNK = 4096;
struct MtRow { long long p, g, m, v, count, first_chunk; };

__device__ __forceinline__ int mt_find(const MtRow* __restrict__ rows, int n, long long chunk) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (rows[mid].first_chunk <= chunk) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(256) adam_multi_kernel(const MtRow* __restrict__ rows, int n, float lr, float b1, float b2, float eps, float bc1,
                                                         float bc2_sqrt) {
  const MtRow r = rows[mt_find(rows, n, blockIdx.x)];
  float* p = reinterpret_cast<float*>(r.p);
  const float* g = reinterpret_cast<const float*>(r.g);
  float* m = reinterpret_cast<float*>(r.m);
  float* v = reinterpret_cast<float*>(r.v);
  const long long base = ((long long)blockIdx.x - r.first_chunk) * MT_CHUNK;
  for (int k = threadIdx.x; k < MT_CHUNK; k += 256) {
    const long long i = base + k;
    if (i >= r.count) break;
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// to_flat != 0: flat[first_chunk * MT_CHUNK + i] = t[i];  else: t[i] = scale * flat[...]
__global__ void __launch_bounds__(256) bucket_copy_kernel(const MtRow* __restrict__ rows, int n, float* __restrict__ flat, float scale, int to_flat) {
  const MtRow r = rows[mt_find(rows, n, blockIdx.x)];
  float* t = reinterpret_cast<float*>(r.p);
  const long long base = ((long long)blockIdx.x - r.first_chunk) * MT_CHUNK;
  float* f = flat + (long long)blockIdx.x * MT_CHUNK;
  for (int k = threadIdx.x; k < MT_CHUNK; k += 256) {
    const long long i = base + k;
    if (i >= r.count) { if (to_flat) f[k] = 0.f; continue; }
    if (to_flat) f[k] = t[i]; else t[i] = scale * f[k];
  }
}

int adam_step_multi(const void* table, int n, long long chunks, float lr, float b1, float b2, float eps, int step, cudaStream_t st) {
  HV_CHECK_ARG(table && n >= 1 && chunks >= 1 && chunks < (1ll << 31) && step >= 1, "adam_step_multi: bad argument");
  const float bc1 = 1.f - powf(b1, (float)step), bc2 = 1.f - powf(b2, (float)step);
  adam_multi_kernel<<<(unsigned)chunks, 256, 0, st>>>(static_cast<const MtRow*>(table), n, lr, b1, b2, eps, bc1, sqrtf(bc2));
  HV_LAUNCH_CHECK();
  return HV_OK;
}

int bucket_copy(const void* table, int n, long long chunks, float* flat, float scale, int to_flat, cudaStream_t st) {
  HV_CHECK_ARG(table && flat && n >= 1 && chunks >= 1 && chunks < (1ll << 31), "bucket_copy: bad argument");
  bucket_copy_kernel<<<(unsigned)chunks, 256, 0, st>>>(static_cast<const MtRow*>(table), n, flat, scale, to_flat);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

}  // namespace hv

// =============================================================================== C ABI
using namespace hv;
extern "C" {

int hv_conv2d_dgrad(const hv_conv_desc* d, const float* w, const float* dy, float* dx, float* workspace, hv_stream_t s) {
  return conv2d_dgrad_fp32(d, w, dy, dx, workspace, as_stream(s));
}
int hv_conv2d_wgrad(const hv_conv_desc* d, const float* dy, float* dw, float* db, hv_stream_t s) {
  return conv2d_wgrad_fp32(d, dy, dw, db, as_stream(s));
}
int hv_act_bwd(const float* out, const float* dy, float* dx, int act, size_t count, hv_stream_t s) { return act_bwd(out, dy, dx, act, count, as_stream(s)); }
int hv_upsample2_bwd(const float* dy, float* dx, int n, int c, int h, int w, int dy_channels, int dy_ch0, hv_stream_t s) {
  return upsample2_bwd(dy, dx, n, c, h, w, dy_channels, dy_ch0, as_stream(s));
}
int hv_stitch_bwd(const float* dout, const int32_t* rows, float* dgen, int n, int h, int w, hv_stream_t s) { return stitch_bwd(dout, rows, dgen, n, h, w, as_stream(s)); }
int hv_axpby(float a, const float* x, float b, float* y, size_t count, hv_stream_t s) { return axpby(a, x, b, y, count, as_stream(s)); }
int hv_affine(float a, const float* x, float c, float* y, size_t count, hv_stream_t s) { return affine(a, x, c, y, count, as_stream(s)); }
int hv_height_loss(const float* p1, const float* p2, const float* h, float maxh, int n, float* loss, float* dp1, float* dp2, hv_stream_t s) {
  return height_loss(p1, p2, h, maxh, n, loss, dp1, dp2, as_stream(s));
}
int hv_masked_center(const float* x, const float* mask, float* out, int w, int c0, int c1, size_t total, hv_stream_t s) {
  return masked_center(x, mask, out, w, c0, c1, total, as_stream(s));
}
int hv_sn_bwd(const float* dweff, const float* weff, const float* u, const float* v, const float* sigma, float* dw, int cout, int kdim, hv_stream_t s) {
  return sn_bwd(dweff, weff, u, v, sigma, dw, cout, kdim, as_stream(s));
}
int hv_act_bwd_bias(const float* out, const float* dy, float* dx, float* db, int act, int n, int c, int hw, hv_stream_t s) {
  return act_bwd_bias(out, dy, dx, db, act, n, c, hw, as_stream(s));
}
int hv_sn_bwd_multi(const void* d_jobs, int njobs, hv_stream_t s) { return sn_bwd_multi(d_jobs, njobs, as_stream(s)); }
int hv_sn_prepare_multi(const void* d_jobs, int njobs, int training, hv_stream_t s) {
  HV_CHECK_ARG(d_jobs && njobs > 0, "sn_prepare_multi: bad argument");
  static_assert(sizeof(SnJob) == 48, "hv_sn_prepare_multi documents rows of six 64-bit words");
  return sn_prepare_batched(static_cast<const SnJob*>(d_jobs), njobs, training, as_stream(s));
}
int hv_gap_fc_sigmoid_bwd(const float* x, const float* sg, const float* ds, const float* fw, float* dx, int accumulate, float* dfw, float* dfb,
                          int n, int c, int hw, hv_stream_t s) {
  return gap_fc_sigmoid_bwd(x, sg, ds, fw, dx, accumulate, dfw, dfb, n, c, hw, as_stream(s));
}
int hv_bn_lrelu_fwd(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var, float* y, float* save_mean,
                    float* save_invstd, int n, int c, int hw, float momentum, float eps, float slope, hv_stream_t s) {
  return bn_lrelu_fwd(x, gamma, beta, running_mean, running_var, y, save_mean, save_invstd, n, c, hw, momentum, eps, slope, as_stream(s));
}
int hv_bn_lrelu_bwd(const float* x, const float* y, const float* dy, const float* gamma, const float* save_mean, const float* save_invstd, float* dx,
                    float* dgamma, float* dbeta, int n, int c, int hw, float slope, hv_stream_t s) {
  return bn_lrelu_bwd(x, y, dy, gamma, save_mean, save_invstd, dx, dgamma, dbeta, n, c, hw, slope, as_stream(s));
}
int hv_reduce_scalar(const float* a, const float* b, float t, int kind, size_t count, float scale, float* out, float* scratch, hv_stream_t s) {
  return reduce_scalar(a, b, t, kind, count, scale, out, scratch, as_stream(s));
}
int hv_loss_grad(const float* a, const float* b, float t, int kind, float g, const float* scale, int scale_is_reciprocal, float* da, int accumulate,
                 size_t count, hv_stream_t s) {
  return loss_grad(a, b, t, kind, g, scale, scale_is_reciprocal, da, accumulate, count, as_stream(s));
}
int hv_dice_fwd(const float* pred, const float* gt, float* sums, float* dice_n, int n, int per, float eps, hv_stream_t s) {
  return dice_fwd(pred, gt, sums, dice_n, n, per, eps, as_stream(s));
}
int hv_dice_bwd(const float* gt, const float* sums, float g_out, float eps, float* dpred, int n, int per, int accumulate, hv_stream_t s) {
  return dice_bwd(gt, sums, g_out, eps, dpred, n, per, accumulate, as_stream(s));
}
int hv_adam_step(float* p, const float* g, float* m, float* v, size_t count, float lr, float b1, float b2, float eps, int step, hv_stream_t s) {
  return adam_step(p, g, m, v, count, lr, b1, b2, eps, step, as_stream(s));
}
int hv_multi_tensor_chunk(void) { return MT_CHUNK; }
int hv_adam_step_multi(const void* table, int n, long long chunks, float lr, float b1, float b2, float eps, int step, hv_stream_t s) {
  return adam_step_multi(table, n, chunks, lr, b1, b2, eps, step, as_stream(s));
}
int hv_bucket_copy(const void* table, int n, long long chunks, float* flat, float scale, int to_flat, hv_stream_t s) {
  return bucket_copy(table, n, chunks, flat, scale, to_flat, as_stream(s));
}

}  // extern "C"
