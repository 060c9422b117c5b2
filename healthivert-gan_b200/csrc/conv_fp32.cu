// fp32 SIMT direct convolution (parity mode) with fused input gather
// (channel concat, nearest x2 upsample, x0.5 subsample, per-sample scalar plane) and fused
// bias + activation epilogue.  NCHW fp32 in and out, exactly the reference's tensors.
//
// Replaces Conv2dBlock.forward (reference models/inpaint_networks.py:494-503) plus the
// torch.cat / F.interpolate feeding it, and the nn.Conv2d(+LeakyReLU) layers of
// NLayerDiscriminator (models/networks.py:575-598).
//
// Tiling: CTA = 256 threads = 8 warps arranged WCO (output-channel groups) x WPX (pixel
// groups).  One warp owns a 2-row x 64-col output tile (lane -> column, so shared-memory
// reads and global stores are conflict-free / coalesced) for CPT output channels per
// thread: 4 pixels x CPT channels accumulators in registers.  Input channels are staged
// through shared memory CI at a time together with the matching weight slab.
#include "hv_common.cuh"
#include "kernels.h"

namespace hv {

struct ConvArgs {
  hv_conv_src src[4];
  int nsrc;
  const float* w;
  const float* bias;
  float* y;
  float* y2;
  int N, Cin, Cout, Hin, Win, Hout, Wout, pad, dil, act;
  int nrows, rowstep, compact, twin, pitch;
  // sub-pixel outputs (data gradient of stride-2 convs): column padding of its own, output written at (oy * os + ooy, ox * os + oox)
  // of a yH x yW plane.  Plain convs: pad_x = pad, os = 1, offsets 0, yH x yW = Hout x Wout.
  int pad_x, os, ooy, oox, yH, yW;
};

constexpr int CONV_CI = 8;

// CONV_TW = 64: a warp owns 2 rows x 64 columns; CONV_TW = 32: 4 rows x 32 columns (same 4 pixels per lane, same accumulation order,
// so results are bit-identical): the PatchGAN layers are 30 .. 34 pixels wide and left half of every 64-wide tile empty
template <int K, int S, int CPT, int WCO, int WPX, int CONV_TW = 64>
__global__ void __launch_bounds__(256) conv_fp32_kernel(const ConvArgs p) {
  constexpr int RPW = CONV_TW == 64 ? 2 : 4;   // output rows per warp
  constexpr int TH = RPW * WPX;
  constexpr int TH_IN = (TH - 1) * S + 1;
  constexpr int COB = CPT * WCO;
  constexpr int KK = K * K;
  extern __shared__ __align__(16) float smem[];
  float* s_in = smem;                                  // [CI][nrows][pitch]
  float* s_w = smem + CONV_CI * p.nrows * p.pitch;     // [CI][KK][COB]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int warp_co = warp % WCO, warp_px = warp / WCO;
  const int tiles_x = (p.Wout + CONV_TW - 1) / CONV_TW;
  const int ox0 = (blockIdx.x % tiles_x) * CONV_TW;
  const int oy0 = (blockIdx.x / tiles_x) * TH;
  const int co0 = blockIdx.y * COB;
  const int n = blockIdx.z;
  const int gy0 = oy0 * S - p.pad, gx0 = ox0 * S - p.pad_x;

  float acc[4][CPT];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int q = 0; q < CPT; ++q) acc[j][q] = 0.f;

  for (int ci0 = 0; ci0 < p.Cin; ci0 += CONV_CI) {
    const int cn = min(CONV_CI, p.Cin - ci0);
    // ---- stage the input halo tile
    for (int c = 0; c < cn; ++c) {
      int ch = ci0 + c, s = 0;
      while (s < p.nsrc - 1 && ch >= p.src[s].channels) { ch -= p.src[s].channels; ++s; }
      const float* sp = p.src[s].ptr;
      const int mode = p.src[s].mode, sch = p.src[s].channels;
      float* dst = s_in + c * p.nrows * p.pitch;
      const int total = p.nrows * p.twin;
      if (mode == HV_SRC_SCALAR) {
        const float val = sp[n];
        for (int i = tid; i < total; i += 256) {
          int r = i / p.twin, x = i - r * p.twin;
          int gy = gy0 + (p.compact ? (r / TH_IN) * p.dil + (r % TH_IN) : r), gx = gx0 + x;
          bool ok = gy >= 0 && gy < p.Hin && gx >= 0 && gx < p.Win;
          dst[r * p.pitch + x] = ok ? val : 0.f;
        }
      } else {
        int sh, sw;
        if (mode == HV_SRC_UP2 || mode == HV_SRC_ZEROINS2) { sh = p.Hin >> 1; sw = p.Win >> 1; }
        else if (mode == HV_SRC_SUB2) { sh = p.Hin << 1; sw = p.Win << 1; }
        else { sh = p.Hin; sw = p.Win; }
        const float* base = sp + ((size_t)n * sch + ch) * sh * sw;
        for (int i = tid; i < total; i += 256) {
          int r = i / p.twin, x = i - r * p.twin;
          int gy = gy0 + (p.compact ? (r / TH_IN) * p.dil + (r % TH_IN) : r), gx = gx0 + x;
          float v = 0.f;
          if (gy >= 0 && gy < p.Hin && gx >= 0 && gx < p.Win) {
            int yy = gy, xx = gx;
            bool hit = true;
            if (mode == HV_SRC_UP2) { yy >>= 1; xx >>= 1; }
            else if (mode == HV_SRC_SUB2) { yy <<= 1; xx <<= 1; }
            else if (mode == HV_SRC_ZEROINS2) { hit = ((yy | xx) & 1) == 0; yy >>= 1; xx >>= 1; }
            if (hit) v = __ldg(base + (size_t)yy * sw + xx);
          }
          dst[r * p.pitch + x] = v;
        }
      }
    }
    // ---- stage the weight slab  s_w[c][t][co]
    for (int i = tid; i < cn * KK * COB; i += 256) {
      int co = i % COB, t = (i / COB) % KK, c = i / (COB * KK);
      float v = 0.f;
      if (co0 + co < p.Cout) v = __ldg(p.w + ((size_t)(co0 + co) * p.Cin + ci0 + c) * KK + t);
      s_w[i] = v;
    }
    __syncthreads();
    // ---- accumulate
    for (int c = 0; c < cn; ++c) {
      const float* in_c = s_in + c * p.nrows * p.pitch;
      const float* w_c = s_w + c * KK * COB + warp_co * CPT;
#pragma unroll
      for (int ky = 0; ky < K; ++ky) {
        const float* row0 = in_c + (ky * p.rowstep + (warp_px * RPW) * S) * p.pitch + lane * S;
        const float* row1 = row0 + S * p.pitch;
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
          float wv[CPT];
          if (CPT % 4 == 0) {   // the CPT weights of a tap are contiguous and 16-byte aligned: LDS.128 broadcasts
#pragma unroll
            for (int q = 0; q < CPT; q += 4) {
              const float4 w4 = *reinterpret_cast<const float4*>(w_c + (ky * K + kx) * COB + q);
              wv[q] = w4.x; wv[q + 1] = w4.y; wv[q + 2] = w4.z; wv[q + 3] = w4.w;
            }
          } else {
#pragma unroll
            for (int q = 0; q < CPT; ++q) wv[q] = w_c[(ky * K + kx) * COB + q];
          }
          const int xo = kx * p.dil;
          float v0, v1, v2, v3;
          if (CONV_TW == 64) { v0 = row0[xo]; v1 = row0[xo + 32 * S]; v2 = row1[xo]; v3 = row1[xo + 32 * S]; }
          else { v0 = row0[xo]; v1 = row1[xo]; v2 = row1[xo + S * p.pitch]; v3 = row1[xo + 2 * S * p.pitch]; }
#pragma unroll
          for (int q = 0; q < CPT; ++q) {
            acc[0][q] = fmaf(v0, wv[q], acc[0][q]);
            acc[1][q] = fmaf(v1, wv[q], acc[1][q]);
            acc[2][q] = fmaf(v2, wv[q], acc[2][q]);
            acc[3][q] = fmaf(v3, wv[q], acc[3][q]);
          }
        }
      }
    }
    __syncthreads();
  }
  // ---- epilogue: bias + activation, coalesced stores
#pragma unroll
  for (int q = 0; q < CPT; ++q) {
    const int co = co0 + warp_co * CPT + q;
    if (co >= p.Cout) continue;
    const float b = p.bias ? __ldg(p.bias + co) : 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int oy = oy0 + warp_px * RPW + (CONV_TW == 64 ? (j >> 1) : j), ox = ox0 + lane + (CONV_TW == 64 ? 32 * (j & 1) : 0);
      if (oy >= p.Hout || ox >= p.Wout) continue;
      float v = acc[j][q] + b;
      if (p.act == HV_ACT_HEADS) {
        if (co == 0) p.y[((size_t)n * p.Hout + oy) * p.Wout + ox] = act_apply(v, HV_ACT_CLAMP1);
        else p.y2[((size_t)n * p.Hout + oy) * p.Wout + ox] = act_apply(v, HV_ACT_SIGMOID);
      } else {
        p.y[(((size_t)n * p.Cout + co) * p.yH + oy * p.os + p.ooy) * p.yW + ox * p.os + p.oox] = act_apply(v, p.act);
      }
    }
  }
}

// Single-filter convolution over many input channels (the PatchGAN logit layer: 512 -> 1, 4x4): a reduction, not a tile problem.
// One CTA per output row: lanes = consecutive output columns (input rows are read as coalesced 128-byte segments, every element is
// reused by the K horizontal taps out of L1), the 8 warps split the input channels, weights are warp-uniform loads; the partial sums
// meet in shared memory.  (One warp per output pixel with lanes over channels read one sector per element: 298 us for 31 MB.)
template <int K>
__global__ void __launch_bounds__(256) conv_single_filter_kernel(const ConvArgs p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = blockIdx.x / p.Hout, oy = blockIdx.x - n * p.Hout;
  const float* x = p.src[0].ptr + (size_t)n * p.Cin * p.Hin * p.Win;
  __shared__ float red[8][33];
  for (int ox0 = 0; ox0 < p.Wout; ox0 += 32) {
    const int ox = ox0 + lane;
    float acc = 0.f;
    if (ox < p.Wout) {
      for (int ci = warp; ci < p.Cin; ci += 8) {
        const float* xc = x + (size_t)ci * p.Hin * p.Win;
        const float* wc = p.w + (size_t)ci * K * K;
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
          const int gy = oy - p.pad + ky * p.dil;
          if (gy < 0 || gy >= p.Hin) continue;
#pragma unroll
          for (int kx = 0; kx < K; ++kx) {
            const int gx = ox - p.pad_x + kx * p.dil;
            if (gx >= 0 && gx < p.Win) acc = fmaf(__ldg(xc + (size_t)gy * p.Win + gx), __ldg(wc + ky * K + kx), acc);
          }
        }
      }
    }
    red[warp][lane] = acc;
    __syncthreads();
    if (warp == 0 && ox < p.Wout) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[i][lane];
      p.y[((size_t)n * p.Hout + oy) * p.Wout + ox] = act_apply(t + (p.bias ? __ldg(p.bias) : 0.f), p.act);
    }
    __syncthreads();
  }
}

// One input channel, many filters (the PatchGAN input conv 1 -> 64, 4x4 stride 2, networks.py:575): the output is 16x the input and
// the kernel is a write stream.  One thread = one output pixel: its K x K input patch in registers, the filters from shared memory,
// one coalesced store per filter plane (the tiled kernel above ran this layer at 0.7 TB/s: 91 us, this one 35 us).
template <int K, int S>
__global__ void __launch_bounds__(256) conv_cin1_kernel(const ConvArgs p) {
  extern __shared__ float s_w[];      // [Cout][K*K] then [Cout] biases
  for (int i = threadIdx.x; i < p.Cout * K * K; i += blockDim.x) s_w[i] = __ldg(p.w + i);
  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) s_w[p.Cout * K * K + i] = p.bias ? __ldg(p.bias + i) : 0.f;
  __syncthreads();
  const int n = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.Hout * p.Wout) return;
  const int oy = i / p.Wout, ox = i - oy * p.Wout;
  const float* x = p.src[0].ptr + (size_t)n * p.Hin * p.Win;
  float v[K * K];
#pragma unroll
  for (int ky = 0; ky < K; ++ky) {
    const int gy = oy * S - p.pad + ky * p.dil;
#pragma unroll
    for (int kx = 0; kx < K; ++kx) {
      const int gx = ox * S - p.pad_x + kx * p.dil;
      v[ky * K + kx] = (gy >= 0 && gy < p.Hin && gx >= 0 && gx < p.Win) ? __ldg(x + (size_t)gy * p.Win + gx) : 0.f;
    }
  }
  float* y = p.y + (size_t)n * p.Cout * p.Hout * p.Wout + i;
  for (int co = 0; co < p.Cout; ++co) {
    const float* w = s_w + co * K * K;
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < K * K; ++t) acc = fmaf(v[t], w[t], acc);
    y[(size_t)co * p.Hout * p.Wout] = act_apply(acc + s_w[p.Cout * K * K + co], p.act);
  }
}

template <int K, int S, int CPT, int WCO, int WPX, int CONV_TW = 64>
static int launch_cfg(ConvArgs& a, cudaStream_t st) {
  constexpr int TH = (CONV_TW == 64 ? 2 : 4) * WPX, TH_IN = (TH - 1) * S + 1, COB = CPT * WCO;
  const int contiguous_rows = TH_IN + (K - 1) * a.dil, compact_rows = K * TH_IN;
  a.compact = contiguous_rows > compact_rows;
  a.nrows = a.compact ? compact_rows : contiguous_rows;
  a.rowstep = a.compact ? TH_IN : a.dil;
  a.twin = (CONV_TW - 1) * S + (K - 1) * a.dil + 1;
  a.pitch = a.twin | 1;
  size_t smem = sizeof(float) * ((size_t)CONV_CI * a.nrows * a.pitch + (size_t)CONV_CI * K * K * COB);
  if (smem > 220 * 1024) {
    set_error("conv2d_fwd: tile needs %zu bytes of shared memory (k=%d dil=%d)", smem, K, a.dil);
    return HV_ERR_UNSUPPORTED;
  }
  auto kern = conv_fp32_kernel<K, S, CPT, WCO, WPX, CONV_TW>;
  if (smem > 48 * 1024) HV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(((a.Wout + CONV_TW - 1) / CONV_TW) * ((a.Hout + TH - 1) / TH), (a.Cout + COB - 1) / COB, a.N);
  kern<<<grid, 256, smem, st>>>(a);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

template <int K, int S>
static int launch_ks(ConvArgs& a, cudaStream_t st) {
  if (a.Cout == 1 && S == 1 && a.Cin >= 64 && a.nsrc == 1 && a.src[0].mode == HV_SRC_DIRECT && a.act != HV_ACT_HEADS && a.os == 1) {
    conv_single_filter_kernel<K><<<(unsigned)(a.N * a.Hout), 256, 0, st>>>(a);
    HV_LAUNCH_CHECK();
    return HV_OK;
  }
  if (a.Cin == 1 && a.Cout >= 16 && a.Cout <= 256 && a.nsrc == 1 && a.src[0].mode == HV_SRC_DIRECT && a.act != HV_ACT_HEADS && a.os == 1) {
    conv_cin1_kernel<K, S><<<dim3((unsigned)((a.Hout * a.Wout + 255) / 256), a.N), 256, (a.Cout * K * K + a.Cout) * sizeof(float), st>>>(a);
    HV_LAUNCH_CHECK();
    return HV_OK;
  }
  if (a.Cout <= 2) return launch_cfg<K, S, 2, 1, 8>(a, st);
  if (a.Cout <= 8) return launch_cfg<K, S, 8, 1, 8>(a, st);
  if (a.Cout <= 16) return launch_cfg<K, S, 8, 2, 4>(a, st);
  if (a.Cout <= 32) return launch_cfg<K, S, 8, 4, 2>(a, st);
  if ((K == 4 || K == 2) && a.Wout <= 40) return launch_cfg<K, S, 8, 8, 1, 32>(a, st);   // PatchGAN layers: 30 .. 34 pixels wide
  return launch_cfg<K, S, 8, 8, 1>(a, st);
}

int conv2d_fwd_fp32(const hv_conv_desc* d, const float* w, const float* bias, float* y, float* y2,
                    cudaStream_t st) {
  return conv2d_fwd_fp32_ex(d, w, bias, y, y2, 0, 0, st);
}

int conv2d_fwd_fp32_ex(const hv_conv_desc* d, const float* w, const float* bias, float* y, float* y2, int hout, int wout,
                       cudaStream_t st) {
  return conv2d_fwd_fp32_sub(d, w, bias, y, y2, hout, wout, nullptr, st);
}

// hout/wout > 0 override the output extent (reads beyond the virtual input are zero): used by the data gradient; sub != null:
// sub-pixel output (separate row / column padding, strided output positions)
int conv2d_fwd_fp32_sub(const hv_conv_desc* d, const float* w, const float* bias, float* y, float* y2, int hout, int wout,
                        const ConvSubpixel* sub, cudaStream_t st) {
  HV_CHECK_ARG(d && w && y, "conv2d_fwd: null argument");
  HV_CHECK_ARG(d->nsrc >= 1 && d->nsrc <= 4, "conv2d_fwd: nsrc=%d out of range", d->nsrc);
  int csum = 0;
  for (int i = 0; i < d->nsrc; ++i) {
    HV_CHECK_ARG(d->src[i].ptr && d->src[i].channels > 0, "conv2d_fwd: bad source %d", i);
    HV_CHECK_ARG(d->src[i].mode >= 0 && d->src[i].mode <= 4, "conv2d_fwd: bad source mode %d", d->src[i].mode);
    HV_CHECK_ARG(d->src[i].mode != HV_SRC_SCALAR || d->src[i].channels == 1, "conv2d_fwd: scalar source must have 1 channel");
    HV_CHECK_ARG(d->src[i].mode != HV_SRC_UP2 || ((d->hin | d->win) & 1) == 0, "conv2d_fwd: up2 source needs even extent");
    csum += d->src[i].channels;
  }
  HV_CHECK_ARG(csum == d->cin, "conv2d_fwd: sources have %d channels, cin=%d", csum, d->cin);
  HV_CHECK_ARG(d->n > 0 && d->n <= 65535 && d->cout > 0 && d->hin > 0 && d->win > 0, "conv2d_fwd: bad extent");
  HV_CHECK_ARG(d->stride == 1 || d->stride == 2, "conv2d_fwd: stride %d unsupported", d->stride);
  HV_CHECK_ARG(d->dil >= 1 && d->pad >= 0, "conv2d_fwd: bad pad/dilation");
  HV_CHECK_ARG(d->act != HV_ACT_HEADS || (d->cout == 2 && y2), "conv2d_fwd: HEADS needs cout=2 and y2");
  ConvArgs a;
  for (int i = 0; i < 4; ++i) a.src[i] = d->src[i < d->nsrc ? i : 0];
  a.nsrc = d->nsrc; a.w = w; a.bias = bias; a.y = y; a.y2 = y2;
  a.N = d->n; a.Cin = d->cin; a.Cout = d->cout; a.Hin = d->hin; a.Win = d->win;
  const int eff = (d->k - 1) * d->dil + 1;
  a.Hout = (d->hin + 2 * d->pad - eff) / d->stride + 1;
  a.Wout = (d->win + 2 * d->pad - eff) / d->stride + 1;
  if (hout > 0) a.Hout = hout;
  if (wout > 0) a.Wout = wout;
  HV_CHECK_ARG(a.Hout > 0 && a.Wout > 0, "conv2d_fwd: empty output");
  a.pad = d->pad; a.dil = d->dil; a.act = d->act;
  a.pad_x = d->pad; a.os = 1; a.ooy = a.oox = 0; a.yH = a.Hout; a.yW = a.Wout;
  if (sub) {
    HV_CHECK_ARG(d->act != HV_ACT_HEADS && sub->os >= 1, "conv2d_fwd: bad sub-pixel output description");
    a.pad = sub->pad_y; a.pad_x = sub->pad_x; a.os = sub->os; a.ooy = sub->ooy; a.oox = sub->oox; a.yH = sub->yH; a.yW = sub->yW;
  }
  const int key = d->k * 10 + d->stride;
  switch (key) {
    case 11: return launch_ks<1, 1>(a, st);   // PixelDiscriminator (models/networks.py:604-753) and its data gradients
    case 21: return launch_ks<2, 1>(a, st);
    case 31: return launch_ks<3, 1>(a, st);
    case 32: return launch_ks<3, 2>(a, st);
    case 51: return launch_ks<5, 1>(a, st);
    case 41: return launch_ks<4, 1>(a, st);
    case 42: return launch_ks<4, 2>(a, st);
    default:
      set_error("conv2d_fwd: kernel %d stride %d not built", d->k, d->stride);
      return HV_ERR_UNSUPPORTED;
  }
}

}  // namespace hv
