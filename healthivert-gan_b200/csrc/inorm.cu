// InstanceNorm2d(affine=False) + LeakyReLU of the PatchGAN discriminator built with norm='instance' (reference
// models/networks.py:555-602 with get_norm_layer('instance')), and the elementwise activation forward that follows the
// tensor-core convolutions of the norm-free discriminator (norm='none').
//
// One CTA owns one (sample, channel) plane.  Planes of up to kInPlaneMax elements (64 x 64: every plane of the 256 x 256
// discriminator) live in registers between the statistics and the output, so the forward reads x once and writes y once (8 B per
// element) and the backward reads x and dy once and writes dx once (12 B per element); BatchNorm re-reads x for its apply pass.
// Larger planes take a streaming variant inside the same kernels (single-pass Welford statistics, then the apply pass: two reads).
#include "hv_common.cuh"

namespace hv {

constexpr int kInPer = 16;                       // plane elements a thread keeps in registers
constexpr int kInMaxThreads = 256;
constexpr int kInPlaneMax = kInMaxThreads * kInPer;
constexpr int kInStreamThreads = 256;

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : slope * v; }

// element k of this thread's register tile: 16-byte mode holds float4 number t + (k / 4) * T, scalar mode element t + k * T
template <bool kVec>
__device__ __forceinline__ int in_elem(int k) {
  return kVec ? 4 * (threadIdx.x + (k >> 2) * blockDim.x) + (k & 3) : threadIdx.x + k * blockDim.x;
}

template <bool kVec>
__device__ __forceinline__ void in_load(const float* __restrict__ p, float (&v)[kInPer], int hw, float add) {
  if (kVec) {
#pragma unroll
    for (int j = 0; j < kInPer / 4; ++j) {
      const int q = threadIdx.x + j * blockDim.x;
      const float4 f = q < (hw >> 2) ? __ldg(reinterpret_cast<const float4*>(p) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[4 * j] = f.x + add; v[4 * j + 1] = f.y + add; v[4 * j + 2] = f.z + add; v[4 * j + 3] = f.w + add;
    }
  } else {
#pragma unroll
    for (int k = 0; k < kInPer; ++k) {
      const int e = in_elem<false>(k);
      v[k] = e < hw ? __ldg(p + e) + add : 0.f;
    }
  }
}

template <bool kVec>
__device__ __forceinline__ void in_store(float* __restrict__ p, const float (&v)[kInPer], int hw) {
  if (kVec) {
#pragma unroll
    for (int j = 0; j < kInPer / 4; ++j) {
      const int q = threadIdx.x + j * blockDim.x;
      if (q < (hw >> 2)) reinterpret_cast<float4*>(p)[q] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < kInPer; ++k) {
      const int e = in_elem<false>(k);
      if (e < hw) p[e] = v[k];
    }
  }
}

// Chan's merge of two (count, mean, M2) partial statistics
__device__ __forceinline__ void welford_merge(float& n, float& m, float& m2, float nb, float mb, float m2b) {
  const float nn = n + nb;
  if (nb == 0.f) return;
  const float d = mb - m, f = nb / nn;
  m += d * f;
  m2 += m2b + d * d * n * f;
  n = nn;
}

// y = lrelu((x + bias[c] - mean) * invstd) per plane; save_mean / save_invstd [n * c] feed the backward
template <bool kVec>
__global__ void __launch_bounds__(kInMaxThreads) in_lrelu_fwd_kernel(const float* __restrict__ x, const float* __restrict__ bias,
                                                                     float* __restrict__ y, float* __restrict__ save_mean,
                                                                     float* __restrict__ save_invstd, int c, int hw, float eps, float slope) {
  __shared__ float red[3][32];
  const int plane = blockIdx.x;
  const size_t base = (size_t)plane * hw;
  const float b = bias ? __ldg(bias + plane % c) : 0.f;
  float mean, invstd;
  if (hw <= kInPlaneMax) {
    float v[kInPer];
    in_load<kVec>(x + base, v, hw, b);
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kInPer; ++k) s += in_elem<kVec>(k) < hw ? v[k] : 0.f;
    mean = block_sum(s, red[0]) / (float)hw;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kInPer; ++k) {
      const float d = in_elem<kVec>(k) < hw ? v[k] - mean : 0.f;
      q = fmaf(d, d, q);
    }
    invstd = rsqrtf(block_sum(q, red[1]) / (float)hw + eps);
#pragma unroll
    for (int k = 0; k < kInPer; ++k) v[k] = lrelu((v[k] - mean) * invstd, slope);
    in_store<kVec>(y + base, v, hw);
  } else {
    float n = 0.f, m = 0.f, m2 = 0.f;
    for (int e = threadIdx.x; e < hw; e += blockDim.x) {
      const float v = __ldg(x + base + e) + b;
      n += 1.f;
      const float d = v - m;
      m += d / n;
      m2 = fmaf(d, v - m, m2);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
      welford_merge(n, m, m2, __shfl_xor_sync(0xffffffffu, n, o), __shfl_xor_sync(0xffffffffu, m, o), __shfl_xor_sync(0xffffffffu, m2, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (lane == 0) { red[0][warp] = n; red[1][warp] = m; red[2][warp] = m2; }
    __syncthreads();
    n = m = m2 = 0.f;
    for (int w = 0; w < nw; ++w) welford_merge(n, m, m2, red[0][w], red[1][w], red[2][w]);   // same order in every thread
    mean = m;
    invstd = rsqrtf(m2 / (float)hw + eps);
    for (int e = threadIdx.x; e < hw; e += blockDim.x) y[base + e] = lrelu((__ldg(x + base + e) + b - mean) * invstd, slope);
  }
  if (threadIdx.x == 0) { save_mean[plane] = mean; save_invstd[plane] = invstd; }
}

// g = dy * lrelu'(xhat);  dx = invstd * (g - mean(g) - xhat * mean(g * xhat));  plane_db[plane] = sum of the plane's dx (optional)
template <bool kVec>
__global__ void __launch_bounds__(kInMaxThreads) in_lrelu_bwd_kernel(const float* __restrict__ x, const float* __restrict__ bias,
                                                                     const float* __restrict__ dy, const float* __restrict__ save_mean,
                                                                     const float* __restrict__ save_invstd, float* __restrict__ dx,
                                                                     float* __restrict__ plane_db, int c, int hw, float slope) {
  __shared__ float red[3][32];
  const int plane = blockIdx.x;
  const size_t base = (size_t)plane * hw;
  const float b = bias ? __ldg(bias + plane % c) : 0.f;
  const float mean = save_mean[plane], invstd = save_invstd[plane], inv_hw = 1.f / (float)hw;
  float sdx = 0.f;
  if (hw <= kInPlaneMax) {
    float xh[kInPer], g[kInPer];
    in_load<kVec>(x + base, xh, hw, b);
    in_load<kVec>(dy + base, g, hw, 0.f);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int k = 0; k < kInPer; ++k) {
      xh[k] = (xh[k] - mean) * invstd;
      g[k] *= xh[k] > 0.f ? 1.f : slope;        // padding lanes hold dy = 0
      sg += g[k];
      sgx = fmaf(g[k], xh[k], sgx);
    }
    const float mg = block_sum(sg, red[0]) * inv_hw, mgx = block_sum(sgx, red[1]) * inv_hw;
#pragma unroll
    for (int k = 0; k < kInPer; ++k) {
      g[k] = invstd * (g[k] - mg - xh[k] * mgx);
      sdx += in_elem<kVec>(k) < hw ? g[k] : 0.f;
    }
    in_store<kVec>(dx + base, g, hw);
  } else {
    float sg = 0.f, sgx = 0.f;
    for (int e = threadIdx.x; e < hw; e += blockDim.x) {
      const float xh = (__ldg(x + base + e) + b - mean) * invstd;
      const float g = __ldg(dy + base + e) * (xh > 0.f ? 1.f : slope);
      sg += g;
      sgx = fmaf(g, xh, sgx);
    }
    const float mg = block_sum(sg, red[0]) * inv_hw, mgx = block_sum(sgx, red[1]) * inv_hw;
    for (int e = threadIdx.x; e < hw; e += blockDim.x) {
      const float xh = (__ldg(x + base + e) + b - mean) * invstd;
      const float g = __ldg(dy + base + e) * (xh > 0.f ? 1.f : slope);
      const float d = invstd * (g - mg - xh * mgx);
      dx[base + e] = d;
      sdx += d;
    }
  }
  if (plane_db) {
    sdx = block_sum(sdx, red[2]);
    if (threadIdx.x == 0) plane_db[plane] = sdx;
  }
}

// db[ch] = sum over n of the plane sums, in sample order (deterministic)
__global__ void in_db_final_kernel(const float* __restrict__ plane_db, float* __restrict__ db, int n, int c) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  float s = 0.f;
  for (int i = 0; i < n; ++i) s += plane_db[(size_t)i * c + ch];
  db[ch] = s;
}

__global__ void act_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int act, size_t count) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) y[i] = act_apply(x[i], act);
}

static bool aligned16(const void* p) { return (reinterpret_cast<size_t>(p) & 15) == 0; }

static int in_threads(int hw) {
  if (hw > kInPlaneMax) return kInStreamThreads;
  const int t = (hw + kInPer - 1) / kInPer;
  return (t + 31) / 32 * 32;
}

int in_lrelu_fwd(const float* x, const float* bias, float* y, float* save_mean, float* save_invstd, int n, int c, int hw, float eps,
                 float slope, cudaStream_t st) {
  HV_CHECK_ARG(x && y && save_mean && save_invstd, "in_lrelu_fwd: null argument");
  HV_CHECK_ARG(n > 0 && c > 0 && hw > 0 && (long long)n * c <= 0x7fffffffll && eps >= 0.f, "in_lrelu_fwd: bad shape n=%d c=%d hw=%d", n, c, hw);
  const bool vec = (hw & 3) == 0 && aligned16(x) && aligned16(y);
  if (vec) in_lrelu_fwd_kernel<true><<<n * c, in_threads(hw), 0, st>>>(x, bias, y, save_mean, save_invstd, c, hw, eps, slope);
  else in_lrelu_fwd_kernel<false><<<n * c, in_threads(hw), 0, st>>>(x, bias, y, save_mean, save_invstd, c, hw, eps, slope);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

int in_lrelu_bwd(const float* x, const float* bias, const float* dy, const float* save_mean, const float* save_invstd, float* dx, float* dbias,
                 int n, int c, int hw, float slope, cudaStream_t st) {
  HV_CHECK_ARG(x && dy && save_mean && save_invstd && dx, "in_lrelu_bwd: null argument");
  HV_CHECK_ARG(n > 0 && c > 0 && hw > 0 && (long long)n * c <= 0x7fffffffll, "in_lrelu_bwd: bad shape n=%d c=%d hw=%d", n, c, hw);
  float* plane_db = nullptr;
  if (dbias) {
    // one partial per plane; the first 256 bytes of the stream's scratch belong to the scalar reductions
    plane_db = static_cast<float*>(stream_scratch(st, sizeof(float) * (size_t)n * c + 256));
    HV_CHECK_ARG(plane_db, "in_lrelu_bwd: scratch allocation failed");
    plane_db += 64;
  }
  const bool vec = (hw & 3) == 0 && aligned16(x) && aligned16(dy) && aligned16(dx);
  if (vec) in_lrelu_bwd_kernel<true><<<n * c, in_threads(hw), 0, st>>>(x, bias, dy, save_mean, save_invstd, dx, plane_db, c, hw, slope);
  else in_lrelu_bwd_kernel<false><<<n * c, in_threads(hw), 0, st>>>(x, bias, dy, save_mean, save_invstd, dx, plane_db, c, hw, slope);
  HV_LAUNCH_CHECK();
  if (dbias) {
    in_db_final_kernel<<<(c + 127) / 128, 128, 0, st>>>(plane_db, dbias, n, c);
    HV_LAUNCH_CHECK();
  }
  return HV_OK;
}

int act_fwd(const float* x, float* y, int act, size_t count, cudaStream_t st) {
  HV_CHECK_ARG(x && y && count > 0, "act_fwd: bad argument");
  HV_CHECK_ARG(act >= HV_ACT_NONE && act <= HV_ACT_CLAMP1, "act_fwd: unsupported activation %d", act);
  const size_t blocks = (count + 255) / 256;
  act_fwd_kernel<<<(int)(blocks > 148 * 16 ? 148 * 16 : blocks), 256, 0, st>>>(x, y, act, count);
  HV_LAUNCH_CHECK();
  return HV_OK;
}

}  // namespace hv

// =============================================================================== C ABI
using namespace hv;
extern "C" {

int hv_in_lrelu_fwd(const float* x, const float* bias, float* y, float* save_mean, float* save_invstd, int n, int c, int hw, float eps,
                    float slope, hv_stream_t s) {
  return in_lrelu_fwd(x, bias, y, save_mean, save_invstd, n, c, hw, eps, slope, as_stream(s));
}
int hv_in_lrelu_bwd(const float* x, const float* bias, const float* dy, const float* save_mean, const float* save_invstd, float* dx,
                    float* dbias, int n, int c, int hw, float slope, hv_stream_t s) {
  return in_lrelu_bwd(x, bias, dy, save_mean, save_invstd, dx, dbias, n, c, hw, slope, as_stream(s));
}
int hv_act_fwd(const float* x, float* y, int act, size_t count, hv_stream_t s) { return act_fwd(x, y, act, count, as_stream(s)); }

}  // extern "C"
