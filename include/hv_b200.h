/*
 * hv_b200.h — C ABI of the B200-native two-stage pseudo-healthy synthesis path.
 *
 * The reference (zhibaishouheilab/HealthiVert-GAN) has no FFI of its own: the path sits
 * behind Python nn.Module classes (SURVEY.md §8b).  This header is the boundary a
 * maintainer binds (ctypes stub in INTEGRATION.md); every entry point names the
 * reference interface it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; all tensor pointers are DEVICE pointers unless a
 *     parameter is documented as host memory;
 *   - every call is stream-ordered on `stream` (a cudaStream_t passed as void*), never
 *     synchronises, and returns 0 on success or a negative hv_status; the message of
 *     the last failure on the calling thread is returned by hv_last_error();
 *   - image tensors are NCHW fp32, contiguous, exactly like the reference's tensors;
 *   - no CPU fallback exists: without a CUDA device every compute call fails.
 */
#ifndef HV_B200_H
#define HV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* hv_stream_t;

enum hv_status {
  HV_OK = 0,
  HV_ERR_INVALID = -1,      /* bad argument / unsupported shape  (reference: assert / assert 0) */
  HV_ERR_CUDA = -2,         /* CUDA runtime error                                         */
  HV_ERR_UNSUPPORTED = -3,  /* valid request, not built for this configuration            */
  HV_ERR_STATE = -4         /* call order violation (e.g. forward before prepare)         */
};

enum hv_act { HV_ACT_NONE = 0, HV_ACT_ELU = 1, HV_ACT_RELU = 2, HV_ACT_SIGMOID = 3,
              HV_ACT_LRELU02 = 4, HV_ACT_CLAMP1 = 5 /* identity then clamp[-1,1] */,
              HV_ACT_HEADS = 6 /* Cout==2: ch0 clamp[-1,1] -> y, ch1 sigmoid -> y2 */ };

enum hv_src_mode { HV_SRC_DIRECT = 0, /* [N,ch,H,W]                                       */
                   HV_SRC_UP2 = 1,    /* [N,ch,H/2,W/2] read through nearest x2 upsample  */
                   HV_SRC_SUB2 = 2,   /* [N,ch,2H,2W]  read through nearest x0.5 (::2)    */
                   HV_SRC_SCALAR = 3  /* [N] one value per sample broadcast to a plane    */ };

enum hv_precision { HV_PREC_FP32 = 0, /* SIMT FFMA, parity mode (max-abs <= 1e-3)         */
                    HV_PREC_BF16 = 1  /* bf16 operands on tcgen05, fp32 accumulate        */ };

const char* hv_last_error(void);
int hv_version(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
uint64_t hv_launch_count(void);

/* ---- A1: Conv2dBlock = spectral_norm(Conv2d)+bias+act ---------------------------------
 * replaces torch.nn.utils.spectral_norm's forward pre-hook (torch/nn/utils/
 * spectral_norm.py:92-114) as installed by models/inpaint_networks.py:491-492.
 * training!=0: v <- normalize(W^T u), u <- normalize(W v) in place (eps 1e-12), then
 * sigma = u^T W v; w_eff = w_orig / sigma (fp32, same [cout, kdim] layout).           */
int hv_sn_prepare(const float* w_orig, float* u, float* v, int cout, int kdim, int training,
                  float* w_eff, float* sigma_out, hv_stream_t stream);

typedef struct hv_conv_src { const float* ptr; int channels; int mode; } hv_conv_src;

typedef struct hv_conv_desc {
  int n, cin, cout;          /* cin = sum of src[i].channels                              */
  int hin, win;              /* virtual input extent (after the per-source up/sub-sample) */
  int k, stride, pad, dil;
  int act;                   /* hv_act                                                    */
  int nsrc;                  /* 1..4 sources concatenated along channels (torch.cat)      */
  hv_conv_src src[4];
} hv_conv_desc;

/* replaces Conv2dBlock.forward (models/inpaint_networks.py:494-503) and the
 * torch.cat / F.interpolate that feed it (:77,:97-99,:105-106,:179,:207,:219,:222,:225);
 * also nn.Conv2d(+LeakyReLU) of NLayerDiscriminator (models/networks.py:575-598).
 * w: [cout,cin,k,k] fp32 effective weights; bias may be NULL; y2 only for HV_ACT_HEADS.  */
int hv_conv2d_fwd(const hv_conv_desc* d, const float* w, const float* bias, float* y, float* y2,
                  hv_stream_t stream);

/* bf16 tensor-core variant of hv_conv2d_fwd (tcgen05.mma, fp32 accumulate in TMEM): same
 * descriptor and fp32 NCHW tensors; inputs and weights are rounded to bf16, the output is rounded to
 * bf16 (heads: fp32).  k in {3,5}, 'same' padding, stride 1 or (k=3) 2, cout <= 64.
 * flags bit 0: additionally apply the nearest x2 upsample of the NEXT layer to the stored result
 * (y is [n,cout,2*hout,2*wout]); bit 1: run the generic kernel instance even where a geometry-
 * specialised one exists (both must agree: tests/test_gpu_conv_bf16.py).                       */
int hv_conv2d_bf16(const hv_conv_desc* d, const float* w, const float* bias, float* y, float* y2,
                   int flags, hv_stream_t stream);

/* replaces global_pool + fc_height + sigmoid (models/inpaint_networks.py:90-93,:211-214) */
int hv_gap_fc_sigmoid(const float* x, const float* fc_w, const float* fc_b, float* out,
                      int n, int c, int hw, hv_stream_t stream);

/* ---- A3: ContextualAttention.forward(f, f, mask) -------------------------------------
 * replaces models/inpaint_networks.py:247-410 for ksize=3, stride=1, rate=2, fuse_k=3.
 * f: [n,c,h,w]; mask: [n,1,4h,4w]; y: [n,c,h,w]; offsets (may be NULL): [n,2,h/2,w/2]
 * int32 (argmax row/col minus own position); flow (may be NULL): [n,3,4h,4w] fp32
 * colour-wheel image in [0,1].  per_sample_mask == 0 reproduces the reference, which
 * reads the mask of sample 0 for the whole batch (:314); != 0 uses each sample's own.
 * workspace: hv_ctx_attn_workspace_bytes(n,c,h,w) bytes of device memory.               */
size_t hv_ctx_attn_workspace_bytes(int n, int c, int h, int w);
int hv_ctx_attn_fwd(const float* f, const float* mask, float* y, int32_t* offsets, float* flow,
                    int n, int c, int h, int w, float softmax_scale, int fuse,
                    int per_sample_mask, void* workspace, hv_stream_t stream);

/* bf16 tensor-core variant (tcgen05 similarity and paste contractions, fused fuse+softmax): same arguments, c = h = w = 64;
 * the workspace is taken from the stream-ordered allocator.                                                   */
int hv_ctx_attn_fwd_bf16(const float* f, const float* mask, float* y, int32_t* offsets, float* flow,
                         int n, int c, int h, int w, float softmax_scale, int fuse,
                         int per_sample_mask, hv_stream_t stream);

/* ---- A4: threshold + height-adaptive stitch -------------------------------------------
 * replaces models/pix2pix_model.py:201-252 and eval_3d_sagittal_twostage.py:103-118.
 * For sample i: pred = ceil(pred_h[i]*maxheight); hgt = max(pred, height[i]);
 * d = hgt-height[i]; xu = x1[i]-d/2; xb = xu+hgt;  out rows [xu,xb) <- gen,
 * rows [0,xu) <- real[d/2 : x1), rows [xb,H) <- real[x2 : x2+H-xb).  No host sync.
 * rows_out (may be NULL): [n,4] int32 = (hgt, d, xu, xb).                              */
int hv_stitch(const float* gen, const float* real, const float* pred_h, const int32_t* x1,
              const int32_t* x2, const int32_t* height, int maxheight, float* out,
              int32_t* rows_out, int n, int h, int w, hv_stream_t stream);
/* out = p > 0.5 ? 1 : 0 (pix2pix_model.py:201-202, eval:105) scaled by `value`; u8 and f32 */
int hv_threshold(const float* p, float* out_f32, uint8_t* out_u8, float value, size_t count,
                 hv_stream_t stream);

/* ---- A5: Sobel + edge loss ------------------------------------------------------------
 * replaces Sobel.forward (models/edge_operator.py:41-48).                               */
int hv_sobel(const float* img, float* edges, int n, int h, int w, hv_stream_t stream);
/* 800*mse(sobel(fake), sobel(real)) as an integer XOR count on {0,1} masks
 * (pix2pix_model.py:109,:263-264,:349; SURVEY F3). xor_count: device uint64; loss: device f32 */
int hv_edge_xor_loss(const float* fake_mask, const float* real_mask, unsigned long long* xor_count,
                     float* loss, int n, int h, int w, hv_stream_t stream);

/* ---- A10: per-column vertebral heights ------------------------------------------------
 * replaces the integer part of calculate_heights (evaluation/RHLV_quantification.py:41-73;
 * coronal twin slices axis 1).  vol_fake / vol_label: u8 {0,1} volumes [d0,d1,d2]
 * C-contiguous; slices are taken along `axis` (2 = sagittal, 1 = coronal) for
 * z in [z0,z1).  Per slice s=z-z0 writes counts[s][8][ncols] int32 in the order
 * all/pre/mid/post fake, all/pre/mid/post label, and meta[s][8] int32 =
 * (valid, t1, t2, center_fake, center_label, ymin, ymax, 0).                            */
int hv_column_heights(const uint8_t* vol_fake, const uint8_t* vol_label, int d0, int d1, int d2,
                      int axis, int z0, int z1, int32_t* counts, int32_t* meta, hv_stream_t stream);

/* ---- A2: the two-stage generator as one native plan -----------------------------------
 * replaces Generator.forward (models/inpaint_networks.py:28-32) in eval()/no_grad mode:
 * CoarseGenerator.forward (:68-117) + FineGenerator.forward (:169-232).                 */
typedef struct hv_generator hv_generator;

int hv_generator_num_layers(void); /* 47 conv blocks, reference state_dict order */
/* name_out: >= 64 bytes, "coarse_generator.conv1" ... ; geometry of the layer */
int hv_generator_layer_info(int idx, char* name_out, int* cin, int* cout, int* k, int* stride,
                            int* pad, int* dil, int* act);
int hv_generator_create(hv_generator** out, int max_batch, int precision);
int hv_generator_destroy(hv_generator* g);
/* device pointers to the reference parameters of layer idx; copied/packed by prepare()  */
int hv_generator_set_layer(hv_generator* g, int idx, const float* w_orig, float* u, float* v,
                           const float* bias);
/* which: 0 = coarse_generator.fc_height, 1 = fine_generator.fc_height; w [64], b [1]     */
int hv_generator_set_fc(hv_generator* g, int which, const float* w, const float* b);
/* sigma, W/sigma and operand packing for all layers; training!=0 runs one power iteration */
int hv_generator_prepare(hv_generator* g, int training, hv_stream_t stream);
/* x, mask, cam: [n,1,256,256]; ratio: [n]; outputs [n,1,256,256] x4, flow [n,3,256,256]
 * (NULL to skip), pred1_h/pred2_h [n]; offsets (NULL to skip) [n,2,32,32] int32.
 * per_sample_mask != 0 uses every sample's own mask in the attention (faithful for the
 * batch-1 eval driver); 0 reproduces the reference's sample-0 quirk.                     */
int hv_generator_forward(hv_generator* g, const float* x, const float* mask, const float* cam,
                         const float* ratio, int n, float* coarse_seg, float* fine_seg,
                         float* x_stage1, float* x_stage2, float* flow, float* pred1_h,
                         float* pred2_h, int32_t* offsets, int per_sample_mask,
                         hv_stream_t stream);
/* measurement hook (bf16 plan): launch the tensor-core conv kernel of layer idx alone on the
 * activations of the last forward (bench.py times the dominant kernel with it)            */
int hv_generator_run_layer(hv_generator* g, int idx, int n, hv_stream_t stream);
/* the same for `count` consecutive layers first .. first+count-1 of the state_dict order, each reading its predecessor's output
 * exactly as in the forward (one host call: bench.py's roofline leg times the chain of 64->64 trunk layers with it)        */
int hv_generator_run_chain(hv_generator* g, int first, int count, int n, hv_stream_t stream);
/* debug/parity tap: copy the fp32 NCHW activation of layer idx (or idx==47: attention
 * output) of the LAST forward into out; returns element count or negative status        */
long long hv_generator_read_tap(hv_generator* g, int idx, float* out, hv_stream_t stream);

/* ---- uint8 HOST interface of the generator: what run_model hands over and keeps ----------
 * replaces, for host buffers, the per-slice tensor plumbing around `model(ct, mask, 1-CAM, ratio)` in
 * eval_3d_sagittal_twostage.py: inputs :84-98 (uint8 CT / CAM planes -> ToTensor -> Normalize(0.5, 0.5); the
 * mask is a row range painted 255, :73-75), outputs :103-121 (seg > 0.5, (x_stage2 + 1) * 127.5 truncated by the
 * next astype(uint8), pred_h).  A pipeline owns `depth` slots of pinned HOST memory and their device mirrors;
 * submit() = 1 H2D copy + ONE CUDA-graph launch of the whole two-stage forward + 1 D2H copy on three streams,
 * so that consecutive slots overlap.  The generator must be prepared and outlive the pipeline; its weights
 * may be re-prepared between submits (the graph reads the plan's buffers, not the parameters).
 * per_sample_mask: see hv_generator_forward; use_graph = 0 launches the kernels directly (A/B, debugging). */
typedef struct hv_pipeline hv_pipeline;
int hv_pipeline_create(hv_pipeline** out, hv_generator* g, int batch, int depth, int per_sample_mask, int use_graph);
int hv_pipeline_destroy(hv_pipeline* p);
/* HOST pointers into slot `slot` (any may be NULL): inputs ct_in / cam_in [batch][256][256] u8, rows_in [batch][2]
 * int32 = mask rows [r0, r1) (eval: (min_x, max_x + 1)), ratio_in [batch] fp32; outputs ct_out = trunc((x_stage2+1)*127.5),
 * fine_mask_out / coarse_mask_out in {0,1} [batch][256][256] u8, heights_out [2][batch] fp32 = pred1_h then pred2_h.  */
int hv_pipeline_slot(hv_pipeline* p, int slot, uint8_t** ct_in, uint8_t** cam_in, int32_t** rows_in, float** ratio_in,
                     uint8_t** ct_out, uint8_t** fine_mask_out, uint8_t** coarse_mask_out, float** heights_out);
/* bytes copied per submit: which = 0 host->device, 1 device->host */
size_t hv_pipeline_bytes(hv_pipeline* p, int which);
/* the pipeline's streams (cudaStream_t): 0 input copies, 1 compute, 2 output copies (for event timing by the caller) */
void* hv_pipeline_stream(hv_pipeline* p, int which);
/* enqueue the first n entries of the slot (fill the inputs first); returns at once.  HV_ERR_STATE while in flight. */
int hv_pipeline_submit(hv_pipeline* p, int slot, int n);
/* block the calling host thread until the slot's outputs have landed in its pinned output block */
int hv_pipeline_wait(hv_pipeline* p, int slot);


/* ======================================================================================
 * Training step (SURVEY.md §8 rows A1/A3 backward, A6, A7, A8), fp32.
 * The host side (healthivert_gan_b200.pix2pix_model) keeps the reference's sequencing
 * (models/pix2pix_model.py:356-382) and calls these in the order autograd would.
 * ==================================================================================== */

/* data gradient of hv_conv2d_fwd: dx over the VIRTUAL concatenated input [n,cin,hin,win] of
 * the forward descriptor d (autograd of F.conv2d w.r.t. input, models/inpaint_networks.py:487-489,
 * models/networks.py:575-598).  dy is the gradient w.r.t. the pre-activation output.
 * workspace: cin*cout*k*k floats.                                                        */
int hv_conv2d_dgrad(const hv_conv_desc* d, const float* w, const float* dy, float* dx,
                    float* workspace, hv_stream_t stream);
/* weight / bias gradient (autograd of F.conv2d w.r.t. weight, bias): the sources of d are
 * the forward inputs; dw [cout,cin,k,k] is overwritten, db [cout] may be NULL.            */
int hv_conv2d_wgrad(const hv_conv_desc* d, const float* dy, float* dw, float* db, hv_stream_t stream);
/* dx = dy * act'(.) through the activation OUTPUT (nn.ELU / ReLU / Sigmoid / LeakyReLU(0.2) /
 * clamp(-1,1) backward, inpaint_networks.py:460-472,:115,:230)                            */
int hv_act_bwd(const float* out, const float* dy, float* dx, int act, size_t count, hv_stream_t stream);
/* hv_act_bwd plus the bias gradient of the conv block in the same pass: dx = dy * act'(out) over [n, c, hw] and
 * db[c] = sum over (n, hw) of dx (deterministic two-pass slice sums).                                           */
int hv_act_bwd_bias(const float* out, const float* dy, float* dx, float* db, int act, int n, int c, int hw, hv_stream_t stream);
/* adjoint of F.interpolate(scale_factor=2, mode='nearest') (:97,:105,:219,:222): channels
 * [dy_ch0, dy_ch0+c) of dy [n,dy_channels,2h,2w] -> dx [n,c,h,w]                          */
int hv_upsample2_bwd(const float* dy, float* dx, int n, int c, int h, int w, int dy_channels,
                     int dy_ch0, hv_stream_t stream);
/* adjoint of hv_stitch w.r.t. gen; rows = rows_out of the forward (pix2pix_model.py:206-252) */
int hv_stitch_bwd(const float* dout, const int32_t* rows, float* dgen, int n, int h, int w, hv_stream_t stream);
/* y = a*x + b*y (x may be NULL) : gradient accumulation */
int hv_axpby(float a, const float* x, float b, float* y, size_t count, hv_stream_t stream);
/* y = a*x + c  (e.g. 1 - CAM, pix2pix_model.py:184) */
int hv_affine(float a, const float* x, float c, float* y, size_t count, hv_stream_t stream);
/* loss_h = mean(40|m p1-h|/h + 40|m p2-h|/h) (pix2pix_model.py:191-192,:350) and its gradients w.r.t. the sigmoid
 * outputs p1, p2 [n] (dp1 / dp2 may be NULL); h: heights as float [n]                      */
int hv_height_loss(const float* p1, const float* p2, const float* h, float maxheight, int n, float* loss,
                   float* dp1, float* dp2, hv_stream_t stream);
/* out = x * mask * [c0 <= column < c1]  (fake_B_local / real_B_local, pix2pix_model.py:254-260; self-adjoint) */
int hv_masked_center(const float* x, const float* mask, float* out, int w, int c0, int c1, size_t total, hv_stream_t stream);
/* backward of the spectral-norm reparametrisation (torch/nn/utils/spectral_norm.py:92-114):
 * dw_orig = (dw_eff - <dw_eff, w_eff> u v^T) / sigma                                      */
int hv_sn_bwd(const float* dw_eff, const float* w_eff, const float* u, const float* v, const float* sigma,
              float* dw_orig, int cout, int kdim, hv_stream_t stream);
/* Every spectral-norm layer of a net in ONE launch (one CTA per layer; the per-layer calls are latency-bound at ~25 us each).
 * d_jobs: DEVICE array of njobs rows of 64-bit words.
 *   hv_sn_prepare_multi rows: {w_orig, u, v, cout | kdim << 32, w_eff, sigma}            (same semantics as hv_sn_prepare)
 *   hv_sn_bwd_multi rows:     {dw_eff, w_eff, u, v, sigma, dw, cout | kdim << 32}        (same semantics as hv_sn_bwd)      */
int hv_sn_prepare_multi(const void* d_jobs, int njobs, int training, hv_stream_t stream);
int hv_sn_bwd_multi(const void* d_jobs, int njobs, hv_stream_t stream);
/* backward of hv_gap_fc_sigmoid: s = forward output [n], ds = its gradient; dx [n,c,hw]
 * (accumulate != 0 adds), dfc_w [c], dfc_b [1]                                            */
int hv_gap_fc_sigmoid_bwd(const float* x, const float* s, const float* ds, const float* fc_w, float* dx, int accumulate,
                          float* dfc_w, float* dfc_b, int n, int c, int hw, hv_stream_t stream);
/* backward of hv_ctx_attn_fwd w.r.t. f (fuse != 0 only).  fwd_workspace = the forward's
 * workspace, untouched since; bwd_workspace: hv_ctx_attn_bwd_workspace_bytes bytes.        */
size_t hv_ctx_attn_bwd_workspace_bytes(int n, int c, int h, int w);
int hv_ctx_attn_bwd(const float* dy, float* df, int n, int c, int h, int w, float softmax_scale, int fuse,
                    void* fwd_workspace, void* bwd_workspace, hv_stream_t stream);
/* hv_ctx_attn_fwd / hv_ctx_attn_bwd with their six dense contractions (2 forward, 4 backward) on tcgen05: the operands are rounded to
 * bf16 (cast / transposed into internal scratch), accumulation and every tensor of the interface and of the workspaces stay fp32.
 * Same arguments and workspaces; the tensor-core training mode (opt.precision = 'bf16') calls these.  Needs c * 9 % 64 == 0.          */
int hv_ctx_attn_fwd_tc(const float* f, const float* mask, float* y, int32_t* offsets, float* flow,
                       int n, int c, int h, int w, float softmax_scale, int fuse, int per_sample_mask,
                       void* workspace, hv_stream_t stream);
int hv_ctx_attn_bwd_tc(const float* dy, float* df, int n, int c, int h, int w, float softmax_scale, int fuse,
                       void* fwd_workspace, void* bwd_workspace, hv_stream_t stream);

/* ---- A7: BatchNorm2d(train) + LeakyReLU(0.2) of NLayerDiscriminator (models/networks.py:583-597).
 * running_mean / running_var may be NULL; save_mean / save_invstd [c] feed the backward.   */
int hv_bn_lrelu_fwd(const float* x, const float* gamma, const float* beta, float* running_mean, float* running_var,
                    float* y, float* save_mean, float* save_invstd, int n, int c, int hw, float momentum, float eps,
                    float slope, hv_stream_t stream);
int hv_bn_lrelu_bwd(const float* x, const float* y, const float* dy, const float* gamma, const float* save_mean,
                    const float* save_invstd, float* dx, float* dgamma, float* dbeta, int n, int c, int hw,
                    float slope, hv_stream_t stream);
/* ---- A7 with norm='instance': InstanceNorm2d(affine=False) + LeakyReLU(slope) per (sample, channel) plane of x [n,c,hw]
 * (models/networks.py:555-602 with get_norm_layer('instance')): y = lrelu((x + bias[c] - mean) / sqrt(var + eps)), biased variance
 * over hw, instance statistics in train and eval alike.  bias [c] (the preceding convolution's, added on load) may be NULL.
 * save_mean / save_invstd [n*c] feed the backward.  8 bytes per element when hw <= 4096 (the plane stays on chip).
 * bwd: dx from x, dy and the saved statistics (12 bytes per element when hw <= 4096); dbias [c] = sum over (n, hw) of dx (the
 * gradient of the bias added on load; may be NULL; zero up to rounding).  Larger planes stream x (and dy) twice.                  */
int hv_in_lrelu_fwd(const float* x, const float* bias, float* y, float* save_mean, float* save_invstd, int n, int c, int hw,
                    float eps, float slope, hv_stream_t stream);
int hv_in_lrelu_bwd(const float* x, const float* bias, const float* dy, const float* save_mean, const float* save_invstd,
                    float* dx, float* dbias, int n, int c, int hw, float slope, hv_stream_t stream);
/* y = act(x) elementwise (act: HV_ACT_NONE .. HV_ACT_CLAMP1; y may equal x): the LeakyReLU after a tensor-core convolution of the
 * norm-free PatchGAN (norm='none'); its backward is hv_act_bwd.                                                                   */
int hv_act_fwd(const float* x, float* y, int act, size_t count, hv_stream_t stream);

/* ---- A6: scalar losses.  out[0] = scale * reduce; kind 0: sum|a-b| (nn.L1Loss), 1: BCE-with-logits
 * against the constant target t (GANLoss vanilla, models/networks.py:237,:270-272), 2: count_nonzero(a)
 * (pix2pix_model.py:336), 3: sum a (GANLoss wgangp with scale -+1/count), 4: sum a*b, 5: sum (a-t)^2
 * against the constant t (GANLoss lsgan).  scratch: 1024 floats.  Deterministic.  A kind outside 0..5
 * returns HV_ERR_INVALID.                                                                    */
int hv_reduce_scalar(const float* a, const float* b, float t, int kind, size_t count, float scale, float* out,
                     float* scratch, hv_stream_t stream);
/* gradients: kind 0: da = g * S * sign(a-b); kind 1: da = g * S * (sigmoid(a) - t); kind 2: da = g * S * 2(a - t)
 * (lsgan); kind 3: da = g * S (wgangp: the sign goes into g; a is not read).  S = 1, *scale or 1 / *scale
 * (device scalar, e.g. count_nonzero(mask)); accumulate != 0 adds into da.  A kind outside 0..3 returns
 * HV_ERR_INVALID.                                                                            */
int hv_loss_grad(const float* a, const float* b, float t, int kind, float g, const float* scale,
                 int scale_is_reciprocal, float* da, int accumulate, size_t count, hv_stream_t stream);
/* diceCoeff(activation='none') (pix2pix_model.py:13-39): dice_n [n], sums [n,3] kept for the backward;
 * g_out = d loss / d dice_n                                                                 */
int hv_dice_fwd(const float* pred, const float* gt, float* sums, float* dice_n, int n, int per, float eps, hv_stream_t stream);
int hv_dice_bwd(const float* gt, const float* sums, float g_out, float eps, float* dpred, int n, int per,
                int accumulate, hv_stream_t stream);

/* bf16 tensor-core variants of hv_conv2d_wgrad / hv_conv2d_dgrad (same descriptor, same fp32 NCHW tensors, same meaning of dx / dw / db):
 * operands rounded to bf16, fp32 accumulation, im2col + batched tcgen05 GEMMs (csrc/gconv_tc.cu).  workspace: the matching
 * *_workspace_bytes(d) bytes of device memory.  The training mode that uses them: Pix2PixModel(opt.precision = 'bf16').          */
size_t hv_conv2d_wgrad_bf16_workspace_bytes(const hv_conv_desc* d);
size_t hv_conv2d_dgrad_bf16_workspace_bytes(const hv_conv_desc* d);
int hv_conv2d_wgrad_bf16(const hv_conv_desc* d, const float* dy, float* dw, float* db, void* workspace, hv_stream_t stream);
int hv_conv2d_dgrad_bf16(const hv_conv_desc* d, const float* w, const float* dy, float* dx, void* workspace, hv_stream_t stream);

/* ---- A4 + A5 fused: the whole tail of Pix2PixModel.forward (models/pix2pix_model.py:201-264) and the edge loss (:109, :349) in one
 * pass over the planes: threshold of both segmentation heads, height-adaptive stitch of both CT heads (rows_* as hv_stitch), masked
 * centre crops (columns [c0, c1)), Sobel of real_B_mask and of the thresholded fine mask, XOR count and 800 * MSE of the two edge
 * maps.  All planes [n,1,h,w] fp32; every output is bit-identical to hv_threshold / hv_stitch / hv_masked_center / hv_sobel /
 * hv_edge_xor_loss on the same inputs.                                                                                          */
int hv_post_forward(const float* fine_seg, const float* coarse_seg, const float* x_stage2, const float* x_stage1, const float* real_B,
                    const float* real_B_mask, const float* mask, const float* pred2_h, const float* pred1_h, const int32_t* x1,
                    const int32_t* x2, const int32_t* height, int maxheight, int c0, int c1, float* fake_B_mask_raw,
                    float* coarse_seg_binary, float* fake_B, float* fake_B_coarse, float* fake_B_local, float* real_B_local,
                    float* real_edges, float* fake_edges, int32_t* rows_fine, int32_t* rows_coarse, unsigned long long* xor_count,
                    float* edge_loss, int n, int h, int w, hv_stream_t stream);

/* ---- A7 on the tensor cores: the BatchNorm-followed PatchGAN convolutions (nn.Conv2d(k=4, padding=1, stride 1|2, bias=False),
 * models/networks.py:583-597) with bf16 operands and fp32 accumulation: batched tcgen05 GEMMs over explicit im2col operands.
 * Cin % 8 == 0, Cout % 128 == 0.  x [n,cin,h,w], w [cout,cin,4,4], y / dy [n,cout,ho,wo] fp32.  workspace:
 * hv_dconv_workspace_bytes(...) bytes (0 = unsupported geometry).  bwd: dx and / or dw may be NULL; x may be NULL when dw is.   */
size_t hv_dconv_workspace_bytes(int n, int cin, int cout, int h, int w, int stride);
int hv_dconv_fwd_bf16(const float* x, const float* w, float* y, int n, int cin, int cout, int h, int wd, int stride,
                      void* workspace, hv_stream_t stream);
int hv_dconv_bwd_bf16(const float* x, const float* w, const float* dy, float* dx, float* dw, int n, int cin, int cout, int h,
                      int wd, int stride, void* workspace, hv_stream_t stream);

/* ---- PixelDiscriminator (netD='pixel', models/networks.py:604-753) fused on the tensor cores, ndf = 64 and input_nc = 1: conv1x1 1->64
 * + LeakyReLU, conv1x1 64->128 + norm + LeakyReLU, conv1x1 128->1, with the 64- and 128-channel maps kept on chip.  The 64->128 product
 * runs on tcgen05 with bf16 operands (h1, W2; dh2, W2, h1 in the backward) and fp32 accumulation; everything else is fp32.
 * norm: 0 none, 1 batch (train-mode statistics; running_mean / running_var, both or neither, updated with momentum and the unbiased
 * variance), 2 instance (affine-free).  x / y / dy / dx [n,1,h,w]; w1 [64], b1 [64], w2 [128,64], w3 [128] fp32; b2 [128] and b3 [1]
 * may be NULL (no bias); gamma / beta [128] for batch norm.  save_mean / save_invstd: [128] (batch) or [n*128] (instance) written by
 * the forward, read by the backward.  bwd: dx may be NULL; dw1 == NULL skips every parameter gradient, otherwise db1, dw2, dw3 are
 * required and db2 / db3 / dgamma / dbeta are written where non-NULL.  workspace: hv_pixel_d_workspace_bytes(n, h, w) bytes (0 = bad
 * extent).  No float atomics: repeated calls give the same bits.  Other ndf / input_nc: HV_ERR_INVALID before any launch.         */
size_t hv_pixel_d_workspace_bytes(int n, int h, int w);
int hv_pixel_d_fwd_bf16(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* gamma,
                        const float* beta, const float* w3, const float* b3, float* running_mean, float* running_var, float* y,
                        float* save_mean, float* save_invstd, int n, int cin, int ndf, int h, int w, int norm, float momentum,
                        float eps, float slope, void* workspace, hv_stream_t stream);
int hv_pixel_d_bwd_bf16(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* gamma,
                        const float* beta, const float* w3, const float* b3, const float* save_mean, const float* save_invstd,
                        const float* dy, float* dx, float* dw1, float* db1, float* dw2, float* db2, float* dgamma, float* dbeta,
                        float* dw3, float* db3, int n, int cin, int ndf, int h, int w, int norm, float slope, void* workspace,
                        hv_stream_t stream);

/* ---- A8: torch.optim.Adam step (pix2pix_model.py:127-130), fused, in place */
int hv_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t count, float lr,
                 float beta1, float beta2, float eps, int step, hv_stream_t stream);
/* multi-tensor variants: ONE launch for all parameters of an optimiser / all gradients of a net.
 * table: DEVICE array of n rows of six int64 {param, grad, exp_avg, exp_avg_sq, count, first_chunk}; tensor r owns the chunks
 * [first_chunk_r, first_chunk_r + ceil(count_r / hv_multi_tensor_chunk())) of `chunks` chunks in total, rows sorted by first_chunk. */
int hv_multi_tensor_chunk(void);
int hv_adam_step_multi(const void* table, int n, long long chunks, float lr, float beta1, float beta2, float eps, int step,
                       hv_stream_t stream);
/* gradient bucket of the data-parallel step (4 all-reduces per step: D_1, D_2, D_3, G; SURVEY 8e): to_flat != 0 gathers the
 * tensors (row field `param`) into flat[chunks * chunk] (tensor r at first_chunk_r * chunk, padding zeroed); to_flat == 0
 * scatters scale * flat back.  The collective on `flat` in between is torch.distributed / NCCL.                               */
int hv_bucket_copy(const void* table, int n, long long chunks, float* flat, float scale, int to_flat, hv_stream_t stream);

/* ======================================================================================
 * A9 / N1: device-side slice preparation and post-processing of the iterative eval loop
 * (run_model, eval_3d_sagittal_twostage.py:46-133), batched over the slices of a stage.
 * Volumes are held as uint8 SLICE-MAJOR planes [S][h][w] (numpy astype(uint8) semantics).
 * ==================================================================================== */
/* out[s][r][c] = (uint8) trunc(vol * scale): vol float64 [d0][d1][d2]; axis 2: slices vol[:,:,s]
 * (sagittal, eval:201), axis 1: vol[:,s,:] (coronal, RHLV_quantification_coronal.py:51-54)  */
int hv_vol_to_u8(const double* vol, uint8_t* out, int d0, int d1, int d2, int axis, double scale, hv_stream_t stream);
/* counts[s][j] = #pixels of slice s equal to id_j (np.sum(label[:,:,z]==id) > 200 tests, eval:204,:213; z range :186-197) */
int hv_slice_id_counts(const uint8_t* label, int nslices, int hw, int id0, int id1, int id2, int32_t* counts, hv_stream_t stream);
/* per batch entry b (slice slice_idx[b], vertebra vert_ids[b]): label==id, 8-connected components < 50 px removed
 * (eval:16-30), bounds / window (:51-72) -> meta[b][8] = (valid, x1, x2, height, min_x, max_x, pixels, 0); then the
 * generator inputs ct / mask / cam1m (= 1 - CAM) / ori_ct [nb,1,h,w] fp32 (:73-98) and x1 / x2 / height [nb].
 * lab_scratch: 2*nb*h*w int32; keep_scratch: nb*h*w bytes.                                  */
int hv_slice_prepare(const uint8_t* label_planes, const uint8_t* ct_planes, const uint8_t* cam_planes,
                     const int32_t* slice_idx, const int32_t* vert_ids, int nb, int h, int w, int maxheight,
                     int32_t* lab_scratch, uint8_t* keep_scratch, int32_t* meta, float* ct, float* mask, float* cam1m,
                     float* ori, int32_t* x1, int32_t* x2, int32_t* height, hv_stream_t stream);
/* after the forward and hv_stitch(x_stage2, ori, pred2_h, ...): (x+1)*127.5 -> ct_out (fp32 slice of the output volume,
 * may be NULL) and its uint8 truncation ct_u8_next; thresholded seg * id stitched into the label map (eval:119-130) ->
 * label_out (fp32, may be NULL) / label_next (uint8; must not alias label_in)               */
int hv_slice_finish(const float* fake_ct, const float* fine_seg, const int32_t* rows, const int32_t* meta,
                    const int32_t* slice_idx, const int32_t* vert_ids, const uint8_t* label_in, int nb, int h, int w,
                    float* ct_out, float* label_out, uint8_t* ct_u8_next, uint8_t* label_next, hv_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * Spine straightening resampler (SURVEY 8f N4): straighten/straighten/curve.py:54-101 (Interpolator.get_grid +
 * interpolate_along = scipy.ndimage.map_coordinates(array, grid, order, cval), mode 'constant') as one gather kernel.
 * vol: float64 [d0][d1][d2] (C order); knots: float64 [npts][3]; basis: float64 [npts][3][3] (basis[n][i][j] = component i of
 * local basis vector j, vector 0 = tangent); out: float64 [npts][s1][s0], out[n][a][b] = sample at
 * knots[n] + basis[n][:,1] * (b - s0/2) + basis[n][:,2] * (a - s1/2); order 0 = nearest (label maps), 1 = trilinear (CT);
 * samples with a coordinate outside [0, extent-1] get cval.                                                            */
int hv_resample_curve(const double* vol, int d0, int d1, int d2, const double* knots, const double* basis, int npts, int s0,
                      int s1, int order, double cval, double* out, hv_stream_t stream);

/* ======================================================================================
 * Debug / measurement hooks.  NOT part of the drop-in surface: no reference interface stands behind them; they only
 * make the library's own kernels observable (tools/trace_conv.py, tools/timeline_forward.py).
 * dev_buf = NULL switches a hook off.
 * ==================================================================================== */
/* CTA 0 of every subsequent conv_tc launch appends (tag, clock64) stamps per role: dev_buf = 12000 + 4 * 400 int64 */
int hv_debug_conv_trace(void* dev_buf);
/* conv_tc launch i (host launch order) records {first CTA entry, last CTA exit} globaltimer ns at dev_buf[4 i], [4 i + 1] */
int hv_debug_conv_timeline(void* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* HV_B200_H */
