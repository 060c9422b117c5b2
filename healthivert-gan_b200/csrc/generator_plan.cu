// Native executor for the two-stage generator forward.
//
// Replaces Generator.forward = CoarseGenerator.forward + FineGenerator.forward
// (reference models/inpaint_networks.py:28-32, :68-117, :169-232) in eval()/no_grad mode.
// The plan owns: effective (spectrally normalised) weights, one activation buffer per conv
// block (also the parity taps), the attention workspace, and a second stream + events so the
// two independent branches of the fine network (dilated-conv branch, attention branch) run
// concurrently.
#include <string.h>
#include <vector>
#include "hv_common.cuh"
#include "kernels.h"
#include "conv_tc.cuh"

namespace hv {

struct LayerSpec {
  const char* name;
  int cin, cout, k, stride, pad, dil, act, hout;  // hout = output height = width
};

// models/inpaint_networks.py:41-63 (coarse, 0..19) and :126-165 (fine, 20..46); state_dict order
static const LayerSpec kLayers[] = {
    {"coarse_generator.conv1", 3, 16, 5, 1, 2, 1, HV_ACT_ELU, 256},
    {"coarse_generator.conv2_downsample", 16, 32, 3, 2, 1, 1, HV_ACT_ELU, 128},
    {"coarse_generator.conv3", 32, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"coarse_generator.conv4_downsample", 32, 64, 3, 2, 1, 1, HV_ACT_ELU, 64},
    {"coarse_generator.conv5", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"coarse_generator.conv6", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"coarse_generator.conv7_atrous", 64, 64, 3, 1, 2, 2, HV_ACT_ELU, 64},
    {"coarse_generator.conv8_atrous", 64, 64, 3, 1, 4, 4, HV_ACT_ELU, 64},
    {"coarse_generator.conv9_atrous", 64, 64, 3, 1, 8, 8, HV_ACT_ELU, 64},
    {"coarse_generator.conv10_atrous", 64, 64, 3, 1, 16, 16, HV_ACT_ELU, 64},
    {"coarse_generator.conv11", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"coarse_generator.conv12", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"coarse_generator.conv20", 65, 64, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"coarse_generator.conv13", 64, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"coarse_generator.conv14", 32, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"coarse_generator.conv19", 33, 32, 3, 1, 1, 1, HV_ACT_ELU, 256},
    {"coarse_generator.conv15", 32, 16, 3, 1, 1, 1, HV_ACT_ELU, 256},
    {"coarse_generator.conv16", 16, 8, 3, 1, 1, 1, HV_ACT_ELU, 256},
    {"coarse_generator.conv17", 8, 1, 3, 1, 1, 1, HV_ACT_NONE, 256},
    {"coarse_generator.conv18", 8, 1, 3, 1, 1, 1, HV_ACT_SIGMOID, 256},
    {"fine_generator.conv1", 4, 16, 5, 1, 2, 1, HV_ACT_ELU, 256},
    {"fine_generator.conv2_downsample", 16, 16, 3, 2, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.conv3", 16, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.conv4_downsample", 32, 32, 3, 2, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.conv5", 32, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.conv6", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.conv7_atrous", 64, 64, 3, 1, 2, 2, HV_ACT_ELU, 64},
    {"fine_generator.conv8_atrous", 64, 64, 3, 1, 4, 4, HV_ACT_ELU, 64},
    {"fine_generator.conv9_atrous", 64, 64, 3, 1, 8, 8, HV_ACT_ELU, 64},
    {"fine_generator.conv10_atrous", 64, 64, 3, 1, 16, 16, HV_ACT_ELU, 64},
    {"fine_generator.pmconv1", 4, 16, 5, 1, 2, 1, HV_ACT_ELU, 256},
    {"fine_generator.pmconv2_downsample", 16, 16, 3, 2, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.pmconv3", 16, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.pmconv4_downsample", 32, 64, 3, 2, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.pmconv5", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.pmconv6", 64, 64, 3, 1, 1, 1, HV_ACT_RELU, 64},
    {"fine_generator.pmconv9", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.pmconv10", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.allconv11", 128, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.allconv19", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.allconv12", 64, 64, 3, 1, 1, 1, HV_ACT_ELU, 64},
    {"fine_generator.allconv13", 64, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.allconv14", 32, 32, 3, 1, 1, 1, HV_ACT_ELU, 128},
    {"fine_generator.allconv15", 32, 16, 3, 1, 1, 1, HV_ACT_ELU, 256},
    {"fine_generator.allconv16", 16, 8, 3, 1, 1, 1, HV_ACT_ELU, 256},
    {"fine_generator.allconv17", 9, 1, 3, 1, 1, 1, HV_ACT_NONE, 256},
    {"fine_generator.allconv18", 9, 1, 3, 1, 1, 1, HV_ACT_SIGMOID, 256},
};
constexpr int kNumLayers = sizeof(kLayers) / sizeof(kLayers[0]);
static_assert(kNumLayers == 47, "the generator has 47 conv blocks");
constexpr int kTapAttention = 47;

enum {
  C1 = 0, C2, C3, C4, C5, C6, C7, C8, C9, C10, C11, C12, C20, C13, C14, C19, C15, C16, C17, C18,
  F1, F2, F3, F4, F5, F6, F7, F8, F9, F10, PM1, PM2, PM3, PM4, PM5, PM6, PM9, PM10, A11, A19, A12,
  A13, A14, A15, A16, A17, A18
};

}  // namespace hv

using namespace hv;

namespace hv { struct TcPlan; }

struct hv_generator {
  int max_batch = 0, precision = 0;
  bool prepared = false;
  int last_n = 0;
  const float* w_orig[kNumLayers] = {};
  float* u[kNumLayers] = {};
  float* v[kNumLayers] = {};
  const float* bias_src[kNumLayers] = {};
  const float* fc_w[2] = {};
  const float* fc_b[2] = {};
  // owned device memory
  float* w_eff[kNumLayers] = {};   // fp32 [cout][cin][k][k]; the two heads of a stage are contiguous
  float* bias[kNumLayers] = {};    // owned copies (heads contiguous)
  float* act[kNumLayers] = {};     // fp32 NCHW activation per layer (heads: not materialised)
  float* ca_out = nullptr;
  void* ca_ws = nullptr;
  float* sigma = nullptr;
  SnJob* d_jobs = nullptr;
  float* blob_w = nullptr;
  float* blob_b = nullptr;
  const float* last_heads[4] = {};  // x_stage1, coarse_seg, x_stage2, fine_seg of the last forward
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // bf16 plan: light kernels whose results are needed late (CAM packing, height heads, attention flow) run on `aux`,
  // co-resident with the one-CTA-per-SM conv kernels of the main stream
  cudaStream_t aux = nullptr;
  cudaEvent_t ev_aux[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  struct hv::TcPlan* tc = nullptr;  // bf16 tensor-core plan (precision == HV_PREC_BF16)
};

namespace hv {

static size_t act_elems(int idx, int n) {
  const LayerSpec& L = kLayers[idx];
  return (size_t)n * L.cout * L.hout * L.hout;
}

static int run_conv(hv_generator* g, int idx, int n, int hin, std::initializer_list<hv_conv_src> srcs, float* y,
                    float* y2, int act_override, int cout_override, cudaStream_t st) {
  const LayerSpec& L = kLayers[idx];
  hv_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.n = n; d.cin = L.cin; d.cout = cout_override > 0 ? cout_override : L.cout;
  d.hin = hin; d.win = hin; d.k = L.k; d.stride = L.stride; d.pad = L.pad; d.dil = L.dil;
  d.act = act_override >= 0 ? act_override : L.act;
  d.nsrc = 0;
  for (const hv_conv_src& s : srcs) d.src[d.nsrc++] = s;
  return conv2d_fwd_fp32(&d, g->w_eff[idx], g->bias[idx], y, y2, st);
}

static hv_conv_src S(const float* p, int ch, int mode = HV_SRC_DIRECT) {
  hv_conv_src s; s.ptr = p; s.channels = ch; s.mode = mode; return s;
}

#define RC(expr) do { int _rc = (expr); if (_rc) return _rc; } while (0)

static int forward_fp32(hv_generator* g, const float* x, const float* mask, const float* cam, const float* ratio,
                        int n, float* coarse_seg, float* fine_seg, float* x_stage1, float* x_stage2, float* flow,
                        float* pred1_h, float* pred2_h, int32_t* offsets, int per_sample_mask, cudaStream_t st) {
  float** a = g->act;
  // ---- coarse network (models/inpaint_networks.py:68-117)
  RC(run_conv(g, C1, n, 256, {S(x, 1), S(ratio, 1, HV_SRC_SCALAR), S(mask, 1)}, a[C1], nullptr, -1, 0, st));
  RC(run_conv(g, C2, n, 256, {S(a[C1], 16)}, a[C2], nullptr, -1, 0, st));
  RC(run_conv(g, C3, n, 128, {S(a[C2], 32)}, a[C3], nullptr, -1, 0, st));
  RC(run_conv(g, C4, n, 128, {S(a[C3], 32)}, a[C4], nullptr, -1, 0, st));
  int prev = C4;
  for (int l : {C5, C6, C7, C8, C9, C10}) { RC(run_conv(g, l, n, 64, {S(a[prev], 64)}, a[l], nullptr, -1, 0, st)); prev = l; }
  RC(gap_fc_sigmoid(a[C10], g->fc_w[0], g->fc_b[0], pred1_h, n, 64, 64 * 64, st));
  RC(run_conv(g, C11, n, 64, {S(a[C10], 64)}, a[C11], nullptr, -1, 0, st));
  RC(run_conv(g, C12, n, 64, {S(a[C11], 64)}, a[C12], nullptr, -1, 0, st));
  RC(run_conv(g, C20, n, 128, {S(a[C12], 64, HV_SRC_UP2), S(cam, 1, HV_SRC_SUB2)}, a[C20], nullptr, -1, 0, st));
  RC(run_conv(g, C13, n, 128, {S(a[C20], 64)}, a[C13], nullptr, -1, 0, st));
  RC(run_conv(g, C14, n, 128, {S(a[C13], 32)}, a[C14], nullptr, -1, 0, st));
  RC(run_conv(g, C19, n, 256, {S(a[C14], 32, HV_SRC_UP2), S(cam, 1)}, a[C19], nullptr, -1, 0, st));
  RC(run_conv(g, C15, n, 256, {S(a[C19], 32)}, a[C15], nullptr, -1, 0, st));
  RC(run_conv(g, C16, n, 256, {S(a[C15], 16)}, a[C16], nullptr, -1, 0, st));
  // conv17 (none, clamp) + conv18 (sigmoid) read the same 8-channel input: one dual-head pass
  RC(run_conv(g, C17, n, 256, {S(a[C16], 8)}, x_stage1, coarse_seg, HV_ACT_HEADS, 2, st));

  // ---- fine network (:169-232): fork the attention branch onto the side stream
  HV_CUDA(cudaEventRecord(g->ev_fork, st));
  HV_CUDA(cudaStreamWaitEvent(g->side, g->ev_fork, 0));
  cudaStream_t sa = g->side;
  // attention branch
  RC(run_conv(g, PM1, n, 256, {S(x, 1), S(coarse_seg, 1), S(mask, 1), S(ratio, 1, HV_SRC_SCALAR)}, a[PM1], nullptr, -1, 0, sa));
  RC(run_conv(g, PM2, n, 256, {S(a[PM1], 16)}, a[PM2], nullptr, -1, 0, sa));
  RC(run_conv(g, PM3, n, 128, {S(a[PM2], 16)}, a[PM3], nullptr, -1, 0, sa));
  RC(run_conv(g, PM4, n, 128, {S(a[PM3], 32)}, a[PM4], nullptr, -1, 0, sa));
  RC(run_conv(g, PM5, n, 64, {S(a[PM4], 64)}, a[PM5], nullptr, -1, 0, sa));
  RC(run_conv(g, PM6, n, 64, {S(a[PM5], 64)}, a[PM6], nullptr, -1, 0, sa));
  RC(ctx_attn_fwd_fp32(a[PM6], mask, g->ca_out, offsets, flow, n, 64, 64, 64, 10.f, 1, per_sample_mask, g->ca_ws, sa));
  RC(run_conv(g, PM9, n, 64, {S(g->ca_out, 64)}, a[PM9], nullptr, -1, 0, sa));
  RC(run_conv(g, PM10, n, 64, {S(a[PM9], 64)}, a[PM10], nullptr, -1, 0, sa));
  HV_CUDA(cudaEventRecord(g->ev_join, sa));
  // dilated-conv branch
  RC(run_conv(g, F1, n, 256, {S(x, 1), S(coarse_seg, 1), S(mask, 1), S(ratio, 1, HV_SRC_SCALAR)}, a[F1], nullptr, -1, 0, st));
  RC(run_conv(g, F2, n, 256, {S(a[F1], 16)}, a[F2], nullptr, -1, 0, st));
  RC(run_conv(g, F3, n, 128, {S(a[F2], 16)}, a[F3], nullptr, -1, 0, st));
  RC(run_conv(g, F4, n, 128, {S(a[F3], 32)}, a[F4], nullptr, -1, 0, st));
  RC(run_conv(g, F5, n, 64, {S(a[F4], 32)}, a[F5], nullptr, -1, 0, st));
  prev = F5;
  for (int l : {F6, F7, F8, F9, F10}) { RC(run_conv(g, l, n, 64, {S(a[prev], 64)}, a[l], nullptr, -1, 0, st)); prev = l; }
  // merge
  HV_CUDA(cudaStreamWaitEvent(st, g->ev_join, 0));
  RC(run_conv(g, A11, n, 64, {S(a[F10], 64), S(a[PM10], 64)}, a[A11], nullptr, -1, 0, st));
  RC(gap_fc_sigmoid(a[A11], g->fc_w[1], g->fc_b[1], pred2_h, n, 64, 64 * 64, st));
  RC(run_conv(g, A12, n, 64, {S(a[A11], 64)}, a[A12], nullptr, -1, 0, st));
  RC(run_conv(g, A19, n, 64, {S(a[A12], 64)}, a[A19], nullptr, -1, 0, st));
  RC(run_conv(g, A13, n, 128, {S(a[A19], 64, HV_SRC_UP2)}, a[A13], nullptr, -1, 0, st));
  RC(run_conv(g, A14, n, 128, {S(a[A13], 32)}, a[A14], nullptr, -1, 0, st));
  RC(run_conv(g, A15, n, 256, {S(a[A14], 32, HV_SRC_UP2)}, a[A15], nullptr, -1, 0, st));
  RC(run_conv(g, A16, n, 256, {S(a[A15], 16)}, a[A16], nullptr, -1, 0, st));
  RC(run_conv(g, A17, n, 256, {S(a[A16], 8), S(x_stage1, 1)}, x_stage2, fine_seg, HV_ACT_HEADS, 2, st));
  g->last_heads[0] = x_stage1; g->last_heads[1] = coarse_seg; g->last_heads[2] = x_stage2; g->last_heads[3] = fine_seg;
  g->last_n = n;
  return HV_OK;
}

}  // namespace hv

// =============================================================================== bf16 tensor-core plan
namespace hv {

// chunked bf16 activation buffers of the plan (channels, extent, zero border = padding of the consumer)
enum BufId {
  B_IN_C, B_C1, B_C2, B_C3, B_C4, B_C5, B_C6, B_C7, B_C8, B_C9, B_C10, B_C11, B_C12U, B_CAM128, B_C20, B_C13, B_C14,
  B_CAM4, B_C19, B_C15, B_C16,
  B_IN_F, B_F1, B_F2, B_F3, B_F4, B_F5, B_F6, B_F7, B_F8, B_F9, B_F10,
  B_P1, B_P2, B_P3, B_P4, B_P5, B_P6, B_CA, B_P9, B_P10,
  B_A11, B_A12, B_A19, B_A13, B_A14, B_A15, B_A16CAT, B_COUNT
};
struct BufSpec { int channels, extent, border; };
static const BufSpec kBufs[B_COUNT] = {
    // B_IN_C (kx-packed 5 x [x, ratio, mask]), C1 .. C12U, CAM128 (kx-packed 3 x CAM), C20, C13, C14 (LOW-res input of conv19, which runs
    // in the sub-pixel upsample mode), CAM4 (4x4 CAM neighbourhoods at 128 x 128), C19, C15, C16
    {16, 256, 2}, {16, 256, 1}, {32, 128, 1}, {32, 128, 1}, {64, 64, 1}, {64, 64, 1}, {64, 64, 2}, {64, 64, 4},
    {64, 64, 8}, {64, 64, 16}, {64, 64, 1}, {64, 64, 1}, {64, 128, 1}, {16, 128, 1}, {64, 128, 1}, {32, 128, 1},
    {32, 128, 1}, {16, 128, 1}, {32, 256, 1}, {16, 256, 1}, {16, 256, 1},
    // B_IN_F (kx-packed 5 x [x, coarse_seg, mask, ratio]), B_F1 = conv1 | pmconv1 (merged layer, 16 + 16 channels), F2 ..
    {32, 256, 2}, {32, 256, 1}, {16, 128, 1}, {32, 128, 1}, {32, 64, 1}, {64, 64, 1}, {64, 64, 2}, {64, 64, 4},
    {64, 64, 8}, {64, 64, 16}, {64, 64, 1},
    // B_P1 is a chunk view of B_F1 (no storage of its own)
    {0, 256, 1}, {16, 128, 1}, {32, 128, 1}, {64, 64, 1}, {64, 64, 1}, {64, 64, 1}, {64, 64, 1}, {64, 64, 1}, {64, 64, 1},
    {64, 64, 1}, {64, 64, 1}, {64, 64, 1}, {32, 128, 1}, {32, 128, 1}, {16, 256, 1}, {16, 256, 1},   // A11, A12, A19 (low-res input of allconv13), A13, A14 (low-res input of allconv15), A15, A16CAT
};

// layer -> (sources, output).  real = channels of the source that carry weights.
struct TcLayerSpec { int layer; int src0, real0, src1, real1; int out; bool up2; int out_chunks; bool kx0, kx1; bool ups; };
static const TcLayerSpec kTcLayers[] = {
    {C1, B_IN_C, 3, -1, 0, B_C1, false, 2, true, false},  {C2, B_C1, 16, -1, 0, B_C2, false, 4},
    {C3, B_C2, 32, -1, 0, B_C3, false, 4},      {C4, B_C3, 32, -1, 0, B_C4, false, 8},
    {C5, B_C4, 64, -1, 0, B_C5, false, 8},      {C6, B_C5, 64, -1, 0, B_C6, false, 8},
    {C7, B_C6, 64, -1, 0, B_C7, false, 8},      {C8, B_C7, 64, -1, 0, B_C8, false, 8},
    {C9, B_C8, 64, -1, 0, B_C9, false, 8},      {C10, B_C9, 64, -1, 0, B_C10, false, 8},
    {C11, B_C10, 64, -1, 0, B_C11, false, 8},   {C12, B_C11, 64, -1, 0, B_C12U, true, 8},
    {C20, B_C12U, 64, B_CAM128, 1, B_C20, false, 8, false, true}, {C13, B_C20, 64, -1, 0, B_C13, false, 4},
    // conv19 / allconv15 read a nearest-x2-upsampled map (:105, :222): sub-pixel upsample mode on the LOW-res producer output
    {C14, B_C13, 32, -1, 0, B_C14, false, 4},   {C19, B_C14, 32, B_CAM4, 1, B_C19, false, 4, false, true, true},
    {C15, B_C19, 32, -1, 0, B_C15, false, 2},   {C16, B_C15, 16, -1, 0, B_C16, false, 2},
    {C17, B_C16, 8, -1, 0, -1, false, 0},       // heads conv17 + conv18
    // fine conv1 and pmconv1 read the same input: ONE conv with 16 + 16 filters writes B_F1 (chunks 0-1 | 2-3 = B_P1)
    {F1, B_IN_F, 4, -1, 0, B_F1, false, 4, true, false},  {F2, B_F1, 16, -1, 0, B_F2, false, 2},
    {F3, B_F2, 16, -1, 0, B_F3, false, 4},      {F4, B_F3, 32, -1, 0, B_F4, false, 4},
    {F5, B_F4, 32, -1, 0, B_F5, false, 8},      {F6, B_F5, 64, -1, 0, B_F6, false, 8},
    {F7, B_F6, 64, -1, 0, B_F7, false, 8},      {F8, B_F7, 64, -1, 0, B_F8, false, 8},
    {F9, B_F8, 64, -1, 0, B_F9, false, 8},      {F10, B_F9, 64, -1, 0, B_F10, false, 8},
    {PM2, B_P1, 16, -1, 0, B_P2, false, 2},
    {PM3, B_P2, 16, -1, 0, B_P3, false, 4},     {PM4, B_P3, 32, -1, 0, B_P4, false, 8},
    {PM5, B_P4, 64, -1, 0, B_P5, false, 8},     {PM6, B_P5, 64, -1, 0, B_P6, false, 8},
    {PM9, B_CA, 64, -1, 0, B_P9, false, 8},     {PM10, B_P9, 64, -1, 0, B_P10, false, 8},
    {A11, B_F10, 64, B_P10, 64, B_A11, false, 8}, {A12, B_A11, 64, -1, 0, B_A12, false, 8},
    {A19, B_A12, 64, -1, 0, B_A19, false, 8},   {A13, B_A19, 64, -1, 0, B_A13, false, 4, false, false, true},   // allconv13 after x2 (:219): sub-pixel mode
    {A14, B_A13, 32, -1, 0, B_A14, false, 4},   {A15, B_A14, 32, -1, 0, B_A15, false, 2, false, false, true},
    {A16, B_A15, 16, -1, 0, B_A16CAT, false, 1}, // writes chunk 0 only; chunk 1 holds x_stage1
    {A17, B_A16CAT, 9, -1, 0, -1, false, 0},    // heads allconv17 + allconv18
};
constexpr int kNumTcLayers = sizeof(kTcLayers) / sizeof(kTcLayers[0]);

// Channel layout of the fine network's kx-packed input buffer B_IN_F (32 channels): chunks 0-1 hold the three planes known when the
// forward starts - x (input channel 0), mask (2), ratio (3) of xnow = [xin, coarse_seg, mask, ratio] (:179) - as channel kx * 3 + j,
// chunks 2-3 hold the coarse mask (input channel 1) as channel 16 + kx.  Only the second pair is packed after the coarse heads.
static const short kFineInputMap[32] = {
    0 * 64 + 0, 0 * 64 + 2, 0 * 64 + 3, 1 * 64 + 0, 1 * 64 + 2, 1 * 64 + 3, 2 * 64 + 0, 2 * 64 + 2, 2 * 64 + 3, 3 * 64 + 0, 3 * 64 + 2, 3 * 64 + 3,
    4 * 64 + 0, 4 * 64 + 2, 4 * 64 + 3, -1,
    0 * 64 + 1, 1 * 64 + 1, 2 * 64 + 1, 3 * 64 + 1, 4 * 64 + 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1};

struct TcPlan {
  TcBuf buf[B_COUNT];
  TcConv conv[kNumLayers];   // indexed by layer id (heads: C17 / A17 entries only)
  bool has[kNumLayers] = {};
  int out_buf[kNumLayers];
  bool out_up2[kNumLayers] = {};
  void* ca_ws = nullptr;     // workspace of the tensor-core attention
  float* gap_partial = nullptr;      // [2][max_batch * 8] shares of the two height heads
  unsigned int* gap_ticket = nullptr;  // [2][max_batch]
  __nv_bfloat16* blob = nullptr;
  // the 16 -> 8 conv + dual heads of each stage as ONE launch (tail_tc.cu): conv16 -> conv17 | conv18, allconv16 -> allconv17 | allconv18
  TcTail tail[2];
  bool tail_fused_last = false;        // the last forward ran the fused tails: B_C16 / chunk 0 of B_A16CAT were not written
};

// HV_NO_TAIL_FUSE=1: the per-layer launches for the thin tails (A/B runs, parity tests); read once per process.
static bool tail_fuse_enabled() {
  static const bool on = !(getenv("HV_NO_TAIL_FUSE") && atoi(getenv("HV_NO_TAIL_FUSE")) != 0);
  return on;
}

static TcAux make_aux(const TcBuf& b, int channel) {
  TcAux a;
  a.ptr = b.ptr; a.chunks = b.chunks; a.chunk = channel >> 3; a.channel = channel & 7;
  a.pitch = b.pitch(); a.border = b.border; a.plane = b.plane(); a.sub_plane = b.sub_plane();
  return a;
}

static void tc_plan_destroy(hv_generator* g) {
  if (!g->tc) return;
  for (int i = 0; i < kNumLayers; ++i) if (g->tc->has[i]) tc_conv_free(g->tc->conv[i]);
  cudaFree(g->tc->blob); cudaFree(g->tc->ca_ws); cudaFree(g->tc->gap_partial); cudaFree(g->tc->gap_ticket);
  delete g->tc;
  g->tc = nullptr;
}

static int tc_plan_create(hv_generator* g) {
  TcPlan* t = new TcPlan();
  g->tc = t;
  const int n = g->max_batch;
  size_t total = 0;
  for (int i = 0; i < B_COUNT; ++i) {
    TcBuf& b = t->buf[i];
    b.n = n; b.chunks = kBufs[i].channels / 8; b.h = b.w = kBufs[i].extent; b.border = kBufs[i].border;
    // buffers consumed by a stride-2 conv are stored space-to-depth
    b.s2d = (i == B_C1 || i == B_C3 || i == B_F1 || i == B_F3 || i == B_P1 || i == B_P3);
    // inputs of the thin 256x256 tail layers (<= 16 filters: conv15/16/17+18, allconv15/16/17+18) are stored in 4 x-phases
    b.xp = (i == B_C19 || i == B_C15 || i == B_C16 || i == B_A15 || i == B_A16CAT) ? 4 : 1;
    total += (b.bytes() + 255) & ~(size_t)255;
  }
  total += TcBuf::kSlackBytes;
  HV_CUDA(cudaMalloc((void**)&t->blob, total));
  HV_CUDA(cudaMemset(t->blob, 0, total));  // zero borders and padding channels, once
  size_t off = 0;
  for (int i = 0; i < B_COUNT; ++i) {
    t->buf[i].ptr = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(t->blob) + off);
    off += (t->buf[i].bytes() + 255) & ~(size_t)255;
  }
  t->buf[B_P1] = t->buf[B_F1].chunk_view(2, 2);   // pmconv1's half of the merged conv1 | pmconv1 output
  HV_CUDA(cudaMalloc(&t->ca_ws, ctx_attn_tc_workspace_bytes(n)));
  HV_CUDA(cudaMalloc((void**)&t->gap_partial, sizeof(float) * 2 * n * 8));
  HV_CUDA(cudaMalloc((void**)&t->gap_ticket, sizeof(unsigned int) * 2 * n));
  HV_CUDA(cudaMemset(t->gap_ticket, 0, sizeof(unsigned int) * 2 * n));
  for (int i = 0; i < kNumLayers; ++i) t->out_buf[i] = -1;
  t->out_buf[PM1] = B_P1;
  for (int i = 0; i < kNumTcLayers; ++i) {
    const TcLayerSpec& s = kTcLayers[i];
    const LayerSpec& L = kLayers[s.layer];
    TcSource srcs[2];
    srcs[0].buf = s.layer == F2 ? t->buf[B_F1].chunk_view(0, 2) : t->buf[s.src0];
    srcs[0].real_channels = s.real0; srcs[0].kxpack = s.kx0;
    if (s.layer == F1) srcs[0].chan_map = kFineInputMap;
    int nsrc = 1;
    if (s.src1 >= 0) { srcs[1].buf = t->buf[s.src1]; srcs[1].real_channels = s.real1; srcs[1].kxpack = s.kx1; srcs[1].nbhd4 = s.ups; nsrc = 2; }
    const bool heads = s.out < 0;
    TcConv& c = t->conv[s.layer];
    const int cout = heads ? 2 : (s.layer == F1 ? kLayers[F1].cout + kLayers[PM1].cout : L.cout);
    int rc = tc_conv_setup(c, srcs, nsrc, L.k, L.stride, L.dil, cout, n, /*allow_pair=*/true, s.ups);
    if (rc) return rc;
    t->has[s.layer] = true;
    if (heads) {
      TcAux a0 = make_aux(t->buf[B_A16CAT], 8);   // x_stage1 joins allconv16's output for the final heads (:225)
      tc_conv_set_output_heads(c, nullptr, nullptr, s.layer == C17 ? &a0 : nullptr, nullptr);
    } else {
      tc_conv_set_output_chunked(c, t->buf[s.out], 0, s.out_chunks, s.up2, L.act);
      t->out_buf[s.layer] = s.out; t->out_up2[s.layer] = s.up2;
    }
  }
  if (tail_fuse_enabled()) {
    int rc = tc_tail_setup(t->tail[0], t->conv[C16], t->conv[C17], n);
    if (!rc) rc = tc_tail_setup(t->tail[1], t->conv[A16], t->conv[A17], n);
    // the coarse heads also write the kx-packed coarse mask of the fine network's input (chunk 2 of B_IN_F, see kFineInputMap): the
    // packing launch between the coarse tail and fine conv1 drops out of the critical path
    if (!rc) rc = tc_tail_set_kxpack(t->tail[0], &t->buf[B_IN_F], 2);
    if (rc) return rc;
  }
  return HV_OK;
}

// batch-size dependent fields (the plan is sized for max_batch; a smaller batch runs fewer tiles)
static void tc_set_batch(TcConv& c, int n) { tc_conv_set_batch(c, n); }

static int tc_plan_pack_weights(hv_generator* g, cudaStream_t st) {
  TcPlan* t = g->tc;
  for (int i = 0; i < kNumTcLayers; ++i) {
    const int l = kTcLayers[i].layer;
    int rc;
    if (kTcLayers[i].out < 0)  // heads: conv17|conv18 and allconv17|allconv18 are adjacent layer ids
      rc = tc_conv_pack_weights(t->conv[l], g->w_eff[l], g->bias[l], 1, g->w_eff[l + 1], g->bias[l + 1], 1, st);
    else if (l == F1)
      rc = tc_conv_pack_weights(t->conv[l], g->w_eff[F1], g->bias[F1], kLayers[F1].cout, g->w_eff[PM1], g->bias[PM1], kLayers[PM1].cout, st);
    else
      rc = tc_conv_pack_weights(t->conv[l], g->w_eff[l], g->bias[l], kLayers[l].cout, nullptr, nullptr, 0, st);
    if (rc) return rc;
  }
  return HV_OK;
}

static int forward_bf16(hv_generator* g, const float* x, const float* mask, const float* cam, const float* ratio, int n,
                        float* coarse_seg, float* fine_seg, float* x_stage1, float* x_stage2, float* flow, float* pred1_h,
                        float* pred2_h, int32_t* offsets, int per_sample_mask, cudaStream_t st) {
  TcPlan* t = g->tc;
  auto view = [&](int id) { TcBuf b = t->buf[id]; b.n = n; return b; };
  auto run = [&](int layer, cudaStream_t s) -> int {
    TcConv& c = t->conv[layer];
    tc_set_batch(c, n);
    return tc_conv_launch(c, s);
  };
  static const bool use_aux = getenv("HV_NO_AUX_STREAM") == nullptr;
  cudaStream_t ax = use_aux ? g->aux : st;
  auto fork_aux = [&](int ev) -> int {   // aux continues after everything enqueued on st so far
    if (!use_aux) return HV_OK;
    HV_CUDA(cudaEventRecord(g->ev_aux[ev], st));
    HV_CUDA(cudaStreamWaitEvent(ax, g->ev_aux[ev], 0));
    return HV_OK;
  };
  auto join_aux = [&](int ev) -> int {   // st continues after everything enqueued on aux so far
    if (!use_aux) return HV_OK;
    HV_CUDA(cudaEventRecord(g->ev_aux[ev], ax));
    HV_CUDA(cudaStreamWaitEvent(st, g->ev_aux[ev], 0));
    return HV_OK;
  };
  // ---- pack the fp32 NCHW inputs into kx-packed chunked bf16 buffers (torch.cat of :77 / :179, F.interpolate of :98)
  {
    RC(fork_aux(0));
    const TcPlaneSrc in_c[3] = {{x, HV_SRC_DIRECT}, {ratio, HV_SRC_SCALAR}, {mask, HV_SRC_DIRECT}};
    RC(tc_pack_kx(in_c, 3, 5, 1, view(B_IN_C), st));
    const TcPlaneSrc cam128[1] = {{cam, HV_SRC_SUB2}};
    RC(tc_pack_kx(cam128, 1, 3, 1, view(B_CAM128), ax));   // first needed by conv20 / conv19
    RC(tc_pack_nbhd4(cam, view(B_CAM4), ax));              // the full-resolution CAM plane for conv19's sub-pixel form
    // the fine network's input planes that do not depend on the coarse network (chunks 0-1 of B_IN_F, see kFineInputMap)
    const TcPlaneSrc in_f0[3] = {{x, HV_SRC_DIRECT}, {mask, HV_SRC_DIRECT}, {ratio, HV_SRC_SCALAR}};
    RC(tc_pack_kx(in_f0, 3, 5, 1, view(B_IN_F).chunk_view(0, 2), ax));
    if (use_aux) HV_CUDA(cudaEventRecord(g->ev_aux[1], ax));
  }
  // ---- coarse network
  for (int l : {C1, C2, C3, C4, C5, C6, C7, C8, C9, C10, C11, C12}) RC(run(l, st));
  RC(fork_aux(2));   // the height head reads conv10_atrous (:90-93); nothing of the trunk overwrites it
  RC(tc_gap_fc_sigmoid(view(B_C10), g->fc_w[0], g->fc_b[0], pred1_h, t->gap_partial, t->gap_ticket, ax));
  if (use_aux) HV_CUDA(cudaStreamWaitEvent(st, g->ev_aux[1], 0));
  const bool fuse_tail = tail_fuse_enabled();
  // the heads of a stage and the conv before them: one fused launch (tail_tc.cu), or conv16 + the dual-head instance
  auto tail = [&](int which, int conv, int heads, float* head0, float* head1) -> int {
    if (fuse_tail) {
      tc_tail_set_batch(t->tail[which], n);
      tc_tail_set_outputs(t->tail[which], head0, head1);
      return tc_tail_launch(t->tail[which], st);
    }
    RC(run(conv, st));
    t->conv[heads].p.head0 = head0; t->conv[heads].p.head1 = head1;
    return run(heads, st);
  };
  for (int l : {C20, C13, C14, C19, C15}) RC(run(l, st));
  RC(tail(0, C16, C17, x_stage1, coarse_seg));
  // ---- fine network: xnow = [xin, coarse_seg, mask, ratio]; conv1 | pmconv1 as one 32-filter conv, then the
  // attention branch forks onto the side stream
  if (!fuse_tail) {   // the fused coarse tail writes chunk 2 itself (chunk 3 is zero padding, never written)
    const TcPlaneSrc in_f1[1] = {{coarse_seg, HV_SRC_DIRECT}};   // chunks 2-3: the only part packed on the critical path
    RC(tc_pack_kx(in_f1, 1, 5, 1, view(B_IN_F).chunk_view(2, 2), st));
  }
  RC(run(F1, st));
  HV_CUDA(cudaEventRecord(g->ev_fork, st));
  HV_CUDA(cudaStreamWaitEvent(g->side, g->ev_fork, 0));
  cudaStream_t sa = g->side;
  for (int l : {PM2, PM3, PM4, PM5, PM6}) RC(run(l, sa));
  RC(ctx_attn_fwd_tc(view(B_P6), mask, view(B_CA), offsets, flow, 10.f, 1, per_sample_mask, t->ca_ws, sa, use_aux ? ax : nullptr,
                     use_aux ? &g->ev_aux[6] : nullptr));
  for (int l : {PM9, PM10}) RC(run(l, sa));
  HV_CUDA(cudaEventRecord(g->ev_join, sa));
  for (int l : {F2, F3, F4, F5, F6, F7, F8, F9, F10}) RC(run(l, st));
  HV_CUDA(cudaStreamWaitEvent(st, g->ev_join, 0));
  RC(run(A11, st));
  RC(fork_aux(4));
  RC(tc_gap_fc_sigmoid(view(B_A11), g->fc_w[1], g->fc_b[1], pred2_h, t->gap_partial + g->max_batch * 8, t->gap_ticket + g->max_batch, ax));
  for (int l : {A12, A19, A13, A14, A15}) RC(run(l, st));
  RC(tail(1, A16, A17, x_stage2, fine_seg));
  t->tail_fused_last = fuse_tail;
  RC(join_aux(5));
  g->last_heads[0] = x_stage1; g->last_heads[1] = coarse_seg; g->last_heads[2] = x_stage2; g->last_heads[3] = fine_seg;
  g->last_n = n;
  return HV_OK;
}

}  // namespace hv

// =============================================================================== C ABI
extern "C" {

int hv_generator_num_layers(void) { return kNumLayers; }

int hv_generator_layer_info(int idx, char* name_out, int* cin, int* cout, int* k, int* stride, int* pad, int* dil,
                            int* act) {
  HV_CHECK_ARG(idx >= 0 && idx < kNumLayers, "layer_info: index %d out of range", idx);
  const LayerSpec& L = kLayers[idx];
  if (name_out) { strncpy(name_out, L.name, 63); name_out[63] = 0; }
  if (cin) *cin = L.cin;
  if (cout) *cout = L.cout;
  if (k) *k = L.k;
  if (stride) *stride = L.stride;
  if (pad) *pad = L.pad;
  if (dil) *dil = L.dil;
  if (act) *act = L.act;
  return HV_OK;
}

int hv_generator_destroy(hv_generator* g) {
  if (!g) return HV_OK;
  tc_plan_destroy(g);
  for (int i = 0; i < kNumLayers; ++i) cudaFree(g->act[i]);
  cudaFree(g->ca_out); cudaFree(g->ca_ws); cudaFree(g->sigma); cudaFree(g->d_jobs);
  cudaFree(g->blob_w); cudaFree(g->blob_b);
  if (g->side) cudaStreamDestroy(g->side);
  if (g->ev_fork) cudaEventDestroy(g->ev_fork);
  if (g->ev_join) cudaEventDestroy(g->ev_join);
  if (g->aux) cudaStreamDestroy(g->aux);
  for (cudaEvent_t e : g->ev_aux) if (e) cudaEventDestroy(e);
  delete g;
  return HV_OK;
}

int hv_generator_create(hv_generator** out, int max_batch, int precision) {
  HV_CHECK_ARG(out, "generator_create: null out pointer");
  HV_CHECK_ARG(max_batch >= 1 && max_batch <= 4096, "generator_create: max_batch %d out of range", max_batch);
  HV_CHECK_ARG(precision == HV_PREC_FP32 || precision == HV_PREC_BF16, "generator_create: bad precision %d", precision);
  int ndev = 0;
  HV_CUDA(cudaGetDeviceCount(&ndev));
  hv_generator* g = new hv_generator();
  g->max_batch = max_batch; g->precision = precision;
  size_t wtot = 0, btot = 0;
  for (int i = 0; i < kNumLayers; ++i) { wtot += (size_t)kLayers[i].cout * kLayers[i].cin * kLayers[i].k * kLayers[i].k; btot += kLayers[i].cout; }
#define GEN_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { hv::set_error("%s failed: %s", #expr, cudaGetErrorString(_e)); hv_generator_destroy(g); return HV_ERR_CUDA; } } while (0)
  GEN_TRY(cudaMalloc(&g->blob_w, wtot * sizeof(float)));
  GEN_TRY(cudaMalloc(&g->blob_b, btot * sizeof(float)));
  GEN_TRY(cudaMalloc(&g->sigma, kNumLayers * sizeof(float)));
  GEN_TRY(cudaMalloc(&g->d_jobs, kNumLayers * sizeof(SnJob)));
  size_t wo = 0, bo = 0;
  for (int i = 0; i < kNumLayers; ++i) {  // state_dict order keeps conv17/conv18 (allconv17/18) adjacent
    g->w_eff[i] = g->blob_w + wo; g->bias[i] = g->blob_b + bo;
    wo += (size_t)kLayers[i].cout * kLayers[i].cin * kLayers[i].k * kLayers[i].k; bo += kLayers[i].cout;
    if (i == C17 || i == C18 || i == A17 || i == A18) continue;  // heads write straight to the outputs
    if (precision == HV_PREC_BF16) continue;                     // bf16 plan keeps chunked bf16 activations
    GEN_TRY(cudaMalloc(&g->act[i], act_elems(i, max_batch) * sizeof(float)));
  }
  if (precision == HV_PREC_FP32) {
    GEN_TRY(cudaMalloc(&g->ca_out, (size_t)max_batch * 64 * 64 * 64 * sizeof(float)));
    GEN_TRY(cudaMalloc(&g->ca_ws, ctx_attn_workspace_bytes(max_batch, 64, 64, 64)));
  }
  GEN_TRY(cudaStreamCreateWithFlags(&g->side, cudaStreamNonBlocking));
  GEN_TRY(cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming));
  GEN_TRY(cudaEventCreateWithFlags(&g->ev_join, cudaEventDisableTiming));
  GEN_TRY(cudaStreamCreateWithFlags(&g->aux, cudaStreamNonBlocking));
  for (cudaEvent_t& e : g->ev_aux) GEN_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
#undef GEN_TRY
  if (precision == HV_PREC_BF16) {
    int rc = tc_plan_create(g);
    if (rc) { hv_generator_destroy(g); return rc; }
  }
  *out = g;
  return HV_OK;
}

int hv_generator_set_layer(hv_generator* g, int idx, const float* w_orig, float* u, float* v, const float* bias) {
  HV_CHECK_ARG(g && idx >= 0 && idx < kNumLayers, "generator_set_layer: bad handle or index %d", idx);
  HV_CHECK_ARG(w_orig && u && v && bias, "generator_set_layer: null parameter pointer for layer %d", idx);
  g->w_orig[idx] = w_orig; g->u[idx] = u; g->v[idx] = v; g->bias_src[idx] = bias;
  g->prepared = false;
  return HV_OK;
}

int hv_generator_set_fc(hv_generator* g, int which, const float* w, const float* b) {
  HV_CHECK_ARG(g && (which == 0 || which == 1) && w && b, "generator_set_fc: bad argument");
  g->fc_w[which] = w; g->fc_b[which] = b;
  return HV_OK;
}

int hv_generator_prepare(hv_generator* g, int training, hv_stream_t stream) {
  HV_CHECK_ARG(g, "generator_prepare: null handle");
  cudaStream_t st = as_stream(stream);
  std::vector<SnJob> jobs(kNumLayers);
  for (int i = 0; i < kNumLayers; ++i) {
    if (!g->w_orig[i]) { set_error("generator_prepare: layer %d (%s) has no parameters", i, kLayers[i].name); return HV_ERR_STATE; }
    jobs[i].w = g->w_orig[i]; jobs[i].u = g->u[i]; jobs[i].v = g->v[i];
    jobs[i].cout = kLayers[i].cout; jobs[i].kdim = kLayers[i].cin * kLayers[i].k * kLayers[i].k;
    jobs[i].w_eff = g->w_eff[i]; jobs[i].sigma = g->sigma + i;
    HV_CUDA(cudaMemcpyAsync(g->bias[i], g->bias_src[i], kLayers[i].cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (!g->fc_w[0] || !g->fc_w[1]) { set_error("generator_prepare: fc_height parameters missing"); return HV_ERR_STATE; }
  // pageable host -> device copy is synchronous w.r.t. the host buffer, so `jobs` may go out of scope
  HV_CUDA(cudaMemcpyAsync(g->d_jobs, jobs.data(), sizeof(SnJob) * kNumLayers, cudaMemcpyHostToDevice, st));
  int rc = sn_prepare_batched(g->d_jobs, kNumLayers, training, st);
  if (rc) return rc;
  if (g->tc) {
    rc = tc_plan_pack_weights(g, st);
    if (rc) return rc;
  }
  g->prepared = true;
  return HV_OK;
}

int hv_generator_forward(hv_generator* g, const float* x, const float* mask, const float* cam, const float* ratio,
                         int n, float* coarse_seg, float* fine_seg, float* x_stage1, float* x_stage2, float* flow,
                         float* pred1_h, float* pred2_h, int32_t* offsets, int per_sample_mask, hv_stream_t stream) {
  HV_CHECK_ARG(g, "generator_forward: null handle");
  if (!g->prepared) { set_error("generator_forward: call hv_generator_prepare first"); return HV_ERR_STATE; }
  HV_CHECK_ARG(n >= 1 && n <= g->max_batch, "generator_forward: batch %d outside 1..%d", n, g->max_batch);
  HV_CHECK_ARG(x && mask && cam && ratio && coarse_seg && fine_seg && x_stage1 && x_stage2 && pred1_h && pred2_h,
               "generator_forward: null tensor pointer");
  if (g->tc)
    return forward_bf16(g, x, mask, cam, ratio, n, coarse_seg, fine_seg, x_stage1, x_stage2, flow, pred1_h, pred2_h,
                        offsets, per_sample_mask, as_stream(stream));
  return forward_fp32(g, x, mask, cam, ratio, n, coarse_seg, fine_seg, x_stage1, x_stage2, flow, pred1_h, pred2_h,
                      offsets, per_sample_mask, as_stream(stream));
}

int hv_generator_run_layer(hv_generator* g, int idx, int n, hv_stream_t stream) {
  HV_CHECK_ARG(g && g->tc, "generator_run_layer: needs a bf16 plan");
  if (!g->prepared) { set_error("generator_run_layer: call hv_generator_prepare first"); return HV_ERR_STATE; }
  HV_CHECK_ARG(idx >= 0 && idx < kNumLayers && g->tc->has[idx] && g->tc->out_buf[idx] >= 0,
               "generator_run_layer: layer %d is not a stand-alone tensor-core conv", idx);
  HV_CHECK_ARG(n >= 1 && n <= g->max_batch, "generator_run_layer: batch %d outside 1..%d", n, g->max_batch);
  tc_set_batch(g->tc->conv[idx], n);
  return tc_conv_launch(g->tc->conv[idx], as_stream(stream));
}

int hv_generator_run_chain(hv_generator* g, int first, int count, int n, hv_stream_t stream) {
  HV_CHECK_ARG(g && g->tc, "generator_run_chain: needs a bf16 plan");
  if (!g->prepared) { set_error("generator_run_chain: call hv_generator_prepare first"); return HV_ERR_STATE; }
  HV_CHECK_ARG(n >= 1 && n <= g->max_batch && count >= 1 && first >= 0 && first + count <= kNumLayers, "generator_run_chain: bad range");
  for (int idx = first; idx < first + count; ++idx)
    HV_CHECK_ARG(g->tc->has[idx] && g->tc->out_buf[idx] >= 0, "generator_run_chain: layer %d is not a stand-alone tensor-core conv", idx);
  for (int idx = first; idx < first + count; ++idx) {
    tc_set_batch(g->tc->conv[idx], n);
    int rc = tc_conv_launch(g->tc->conv[idx], as_stream(stream));
    if (rc) return rc;
  }
  return HV_OK;
}

long long hv_generator_read_tap(hv_generator* g, int idx, float* out, hv_stream_t stream) {
  HV_CHECK_ARG(g && out, "generator_read_tap: null argument");
  HV_CHECK_ARG(g->last_n > 0, "generator_read_tap: no forward has run");
  const float* src = nullptr;
  size_t count = 0;
  if (idx == kTapAttention && g->tc) {
    TcBuf v = g->tc->buf[B_CA];
    v.n = g->last_n;
    int rc = tc_unpack_nchw(v, 0, 64, out, as_stream(stream));
    if (rc) return rc;
    return (long long)g->last_n * 64 * 64 * 64;
  }
  if (idx == kTapAttention) { src = g->ca_out; count = (size_t)g->last_n * 64 * 64 * 64; }
  else {
    HV_CHECK_ARG(idx >= 0 && idx < kNumLayers, "generator_read_tap: index %d out of range", idx);
    count = act_elems(idx, g->last_n);
    if (idx == C17) src = g->last_heads[0];
    else if (idx == C18) src = g->last_heads[1];
    else if (idx == A17) src = g->last_heads[2];
    else if (idx == A18) src = g->last_heads[3];
    else if (g->tc) {
      const int b = g->tc->out_buf[idx];
      HV_CHECK_ARG(b >= 0, "generator_read_tap: layer %d has no tap in bf16 mode", idx);
      TcBuf v = g->tc->buf[b];
      v.n = g->last_n;
      if (g->tc->tail_fused_last && (idx == C16 || idx == A16)) {
        // the fused tail kept this layer's output in shared memory: recompute it with the per-layer instance from its input
        // (B_C15 / B_A15), which the forward leaves intact
        tc_set_batch(g->tc->conv[idx], g->last_n);
        int rc = tc_conv_launch(g->tc->conv[idx], as_stream(stream));
        if (rc) return rc;
      }
      const int ch = idx == A16 ? 8 : kLayers[idx].cout;
      // layers whose output is stored nearest-x2-upsampled (conv12, conv14, allconv19, allconv14): read the native grid back
      int rc = tc_unpack_nchw(v, 0, ch, out, as_stream(stream), g->tc->out_up2[idx] ? 2 : 1);
      if (rc) return rc;
      return (long long)count;
    }
    else src = g->act[idx];
  }
  HV_CUDA(cudaMemcpyAsync(out, src, count * sizeof(float), cudaMemcpyDeviceToDevice, as_stream(stream)));
  return (long long)count;
}

}  // extern "C"
