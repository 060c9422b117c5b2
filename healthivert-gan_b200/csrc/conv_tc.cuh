// bf16 tensor-core convolution path (tcgen05 + TMEM + TMA): shared declarations.
//
// Activation layout ("chunked"): [n][chunk = channel/8][plane position][8 channels] bf16, where a
// plane is the zero-bordered image flattened row-major: position = (y + border) * pitch + (x + border),
// pitch = w + 2*border.  With this layout
//   * a run of consecutive positions of one chunk is contiguous (16 B per position), so TMA brings a
//     [chunks][positions][8] box straight into the canonical no-swizzle K-major UMMA operand layout;
//   * a conv tap is a constant shift of the flattened position, so every tap of a band reads the SAME
//     shared-memory tile through a shifted start address (no per-tap reload from L2);
//   * the epilogue stores 32 consecutive positions x 16 B = 512 contiguous bytes per warp instruction.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace hv {

// s2d ("space to depth"): the buffer feeds a stride-2 conv; it is stored as 4 sub-planes selected by
// (y&1, x&1), each a zero-bordered (h/2) x (w/2) image, so that every stride-2 tap is a constant shift
// inside one sub-plane (the producer's epilogue scatters its pixels accordingly).
struct TcBuf {
  __nv_bfloat16* ptr = nullptr;
  int n = 0, chunks = 0, h = 0, w = 0, border = 0;
  bool s2d = false;
  // xp ("x phases", 1 or 4): the buffer feeds a THIN conv (<= 16 output channels); it is stored as xp sub-planes selected by
  // x % xp, each a zero-bordered h x (w/xp) image.  The consumer then computes xp horizontally adjacent output pixels per
  // accumulator row (N = xp * Cout columns), i.e. 4x fewer, 4x wider MMAs than one pixel per row.
  int xp = 1;
  int img_chunks = 0;  // chunks per image in memory when this is a view of a chunk range of a wider buffer (0: == chunks)
  __host__ __device__ int image_chunks() const { return img_chunks ? img_chunks : chunks; }
  // element offset of chunk plane c of image i
  __host__ __device__ size_t chunk_base(int i, int c) const { return ((size_t)i * image_chunks() + c) * (size_t)plane() * 8; }
  // view of chunks [c0, c0 + count)
  TcBuf chunk_view(int c0, int count) const {
    TcBuf v = *this;
    v.img_chunks = image_chunks();
    v.ptr = ptr + (size_t)c0 * plane() * 8;
    v.chunks = count;
    return v;
  }
  __host__ __device__ int sub_h() const { return s2d ? h / 2 : h; }
  __host__ __device__ int sub_w() const { return s2d ? w / 2 : w / xp; }
  // ONE zero gap of `border` columns between consecutive rows: it is the right border of row y and the left border of row y + 1 (a tap is
  // a shift of the flattened position, so x + dx >= w lands in the next row's gap).  The tiles of a layer cover rows x pitch positions:
  // w + border instead of w + 2 border is 17 % fewer tiles at dilation 16, 1.5 % at dilation 1 (64 x 64 maps).
  __host__ __device__ int pitch() const { return sub_w() + border; }
  __host__ __device__ int rows() const { return sub_h() + 2 * border; }
  __host__ __device__ int sub_plane() const { return (pitch() * rows() + 7) & ~7; }
  __host__ __device__ int plane() const { return s2d ? 4 * sub_plane() : xp * sub_plane(); }
  __host__ __device__ size_t pos(int y, int x) const {
    if (xp > 1) return (size_t)(x % xp) * sub_plane() + (size_t)(y + border) * pitch() + x / xp + border;
    if (!s2d) return (size_t)(y + border) * pitch() + x + border;
    return (size_t)((y & 1) * 2 + (x & 1)) * sub_plane() + (size_t)((y >> 1) + border) * pitch() + (x >> 1) + border;
  }
  size_t elems() const { return (size_t)n * image_chunks() * plane() * 8; }
  size_t bytes() const { return elems() * sizeof(__nv_bfloat16); }
  // multi-row TMA boxes of the last tiles of the last image read (and discard) up to 4 rows past the plane
  static constexpr size_t kSlackBytes = 256 * 1024;
};

constexpr int TC_MAX_SEGS = 12;
constexpr int TC_TILE_M = 128;

// One TMA load of the producer = one "segment": `nrows` bands of 128 consecutive positions (one per kernel row ky,
// `row pitch * dilation` positions apart, fetched by a single 4-D box) x all channel chunks of one source.
// Shared-memory image of a segment: [chunk][row][128 positions][8 ch].  Every tap (row r, i-th kx of the segment) of the
// segment is a shifted view of that image; offsets are affine, so the MMA issuer needs no per-tap table:
//   A start (16 B units) = r * 128 + a0 + i * a_step          B start = b0 + r * b_row_step + i * b_step
struct TcSeg {
  int map;            // which tensor map (source)
  int rel_start2;     // 2 * (start of row 0's band relative to the tile origin): tensor-map inner unit = 8 B
  int c1;             // second box coordinate: sub-plane (s2d sources) or 0
  int nchunks;        // channel chunks of this source
  int nrows;          // kernel rows brought by this load
  int ntaps;          // taps per row
  uint32_t a0, a_step, b0, b_step, b_row_step;
  uint32_t tx_bytes;  // bytes this load brings
};

enum TcOutMode { TC_OUT_CHUNKED = 0, TC_OUT_CHUNKED_UP2 = 1, TC_OUT_HEADS = 2, TC_OUT_CHUNKED_S2D = 3 };

struct TcAux {  // optional bf16 side output of a head: one channel of a chunked buffer
  __nv_bfloat16* ptr;
  int chunks, chunk, channel, pitch, border, plane, sub_plane;
};

struct TcParams {
  CUtensorMap maps[2];
  TcSeg segs[TC_MAX_SEGS];
  int nseg;
  const void* w_packed;
  uint32_t w_bytes;
  const float* bias;  // [n_pad]
  int s2d_in;     // sources are space-to-depth buffers (stride-2 conv)
  int in_xp;      // sources are x-phase buffers: every accumulator row holds in_xp adjacent output pixels (N = in_xp * cp)
  int cp;         // accumulator columns per output pixel when in_xp > 1
  int out_xp;     // the output buffer is an x-phase buffer (aux outputs of the heads too)
  int ups;        // sub-pixel upsample conv: sources are LOW-res maps, accumulator columns = 4 output parities x cp channels
  int map5d;      // tensor maps are 5-D (s2d / x-phase sources)
  int pair;       // two consecutive tiles per producer / issuer / barrier round (thin layers: halves the single-thread handshakes)
  int tile_adv;   // valid output positions per 128-row MMA tile (128 - widest tap shift)
  int tiles_per_image, total_tiles;
  int in_pitch, in_border, q_first;
  unsigned long long pitch_magic;  // ceil(2^40 / in_pitch): q / in_pitch == (q * magic) >> 40 for q < 2^20
  unsigned long long tiles_magic;  // ceil(2^40 / tiles_per_image), same trick for tile -> image
  int h_out, w_out;   // extent of the accumulator-row grid (w_out = image width / in_xp)
  int w_img;          // image width in pixels
  int act;
  int out_mode;
  __nv_bfloat16* out;
  int out_pitch, out_border, out_plane, out_sub_plane, out_chunks_total, out_chunk_off, out_nchunks;
  float* head0;
  float* head1;
  TcAux aux0, aux1;
  uint32_t slot_bytes;
  int nslots;
  long long* trace;  // debug event trace (device buffer of 12000 int64) or null
  long long* timeline;  // debug: {min CTA entry, max CTA exit} globaltimer ns of this launch, or null
};

struct TcSource {
  TcBuf buf;
  int real_channels;  // channels of this source that carry weights (<= buf.chunks*8)
  // kx-packed source: channel kx*real_channels + c of the buffer holds input channel c shifted by (kx - k/2)*dil pixels
  // along x, so the conv needs one tap (and one MMA K-step set) per kernel ROW instead of per tap.  Pays off for
  // sources with few channels (network inputs, the CAM plane): k*real_channels must fit the buffer.
  bool kxpack = false;
  // optional explicit channel layout of a kx-packed buffer: packed channel ch holds input channel (chan_map[ch] & 63) shifted by
  // tap kx = chan_map[ch] >> 6, or nothing (-1).  Null = the default layout ch = kx * real_channels + c.  (The fine network's input
  // keeps the planes known at the start of the forward and the coarse mask in separate chunks, so that only the latter is packed
  // on the critical path.)
  const short* chan_map = nullptr;   // [buf.chunks * 8], host memory, must outlive tc_conv_pack_weights
  // second source of a sub-pixel upsample conv (see tc_conv_setup `ups`): a HIGH-resolution single-channel plane packed at low
  // resolution, channel ry * 4 + rx of position (m, n) = plane(2m - 1 + ry, 2n - 1 + rx) (tc_pack_nbhd4): all 3x3 taps of the four
  // output parities of (m, n) read this one position, so the source costs one K = 16 MMA step per tile
  bool nbhd4 = false;
};

struct TcConv {
  TcParams p;
  int n_pad = 0;
  int grid = 0;
  int ctas_per_sm = 1;
  size_t smem = 0;
  void* w_packed = nullptr;   // owned
  float* bias_pad = nullptr;  // owned
  int k = 0, stride = 1, dil = 1;
  int nsrc = 0;
  TcSource src[2];
  int cout_real = 0;
  bool force_generic = false;   // run the FIXED = 0 kernel instance even when a specialised one matches (parity tests)
  // caller-provided memory for the packed weights + bias (>= kArenaBytes, 256-byte aligned); null: tc_conv_setup allocates (cudaMalloc,
  // which synchronises the device - fine at plan creation, not inside a training step)
  void* arena = nullptr;
  static constexpr size_t kArenaBytes = 4u << 20;
};

// geometry + tensor maps + tables; allocates the packed-weight / bias buffers
// allow_pair: the caller has a tile-pair kernel instance for this layer (the generator plan does for its layers; a stand-alone
// conv of arbitrary geometry does not and runs the generic instance)
// ups: the conv reads a nearest-x2-upsampled map (models/inpaint_networks.py:105, :222: F.interpolate(scale_factor=2) before conv19 /
// allconv15).  Instead of materialising the upsampled map, srcs[0] is the LOW-resolution map: output pixel (2m + py, 2n + px) only
// sees the 2 x 2 low-res pixels around (m, n), so the conv becomes 3 x 3 low-res taps with per-parity SUMMED weights and
// N = 4 parities x cp accumulator columns: 4x fewer tiles, band loads and MMAs of 4x the width.  cout <= 32.
int tc_conv_setup(TcConv& c, const TcSource* srcs, int nsrc, int k, int stride, int dil, int cout_real,
                  int n_images, bool allow_pair = false, bool ups = false);
// batch of the next launches (<= the n_images of the setup): tile count and grid
void tc_conv_set_batch(TcConv& c, int n_images);
// w_eff_a: [cout_a][cin_total][k][k] fp32 effective weights (cin_total = sum real_channels);
// w_eff_b (heads only): second filter bank stacked after the first along cout
int tc_conv_pack_weights(TcConv& c, const float* w_eff_a, const float* bias_a, int cout_a, const float* w_eff_b,
                         const float* bias_b, int cout_b, cudaStream_t st);
void tc_conv_set_output_chunked(TcConv& c, const TcBuf& out, int chunk_off, int nchunks, bool up2, int act);
void tc_conv_set_output_heads(TcConv& c, float* head0, float* head1, const TcAux* aux0, const TcAux* aux1);
int tc_conv_launch(const TcConv& c, cudaStream_t st);
void tc_set_trace(long long* dev_buf);  // debug: CTA 0 of every subsequent launch records its event timeline
void tc_conv_free(TcConv& c);

// fused thin tail of a generator stage (tail_tc.cu): a 16 -> 8 x-phase 3x3 ELU conv and the dual heads that read its output (plus
// chunk 1 of the heads' own source buffer) in one persistent launch; the 8-channel intermediate stays in shared memory
struct TcTailParams {
  CUtensorMap maps[4];   // conv input: views 1-4, shifted views; heads' second chunk: views 1-4, shifted views
  const void* w_mid;     // packed weights / padded bias of the two per-layer instances (TcConv::w_packed, bias_pad)
  const void* w_head;
  const float* bias_mid;
  const float* bias_head;
  int n, h, w_img;
  int rows_per_unit, strips, units;   // work unit = (image pair, strip of rows_per_unit output rows)
  float* head0;
  float* head1;
  TcAux aux0;            // bf16 copy of head 0 (coarse stage: x_stage1 for the fine heads), or ptr == null
  TcBuf kx;              // head 1 kx-packed (5 taps, channels 0-4 of chunk kx_chunk; coarse stage: the fine conv1 input), or ptr == null
  int kx_chunk;
  long long* timeline;
};
struct TcTail {
  TcTailParams p;
  int grid = 0;
};
// mid: the 16 -> 8 conv (x-phase source, chunked output), heads: the dual-head instance reading mid's output buffer; the weights are
// read from the instances' packed buffers at launch time
int tc_tail_setup(TcTail& t, const TcConv& mid, const TcConv& heads, int n_images);
void tc_tail_set_batch(TcTail& t, int n_images);
void tc_tail_set_outputs(TcTail& t, float* head0, float* head1);
// also write head 1 as tc_pack_kx(k = 5, dil = 1) would into chunk `chunk` of dst (null: off)
int tc_tail_set_kxpack(TcTail& t, const TcBuf* dst, int chunk);
int tc_tail_launch(const TcTail& t, cudaStream_t st);
// next slot of the timeline hook (or null), shared with conv_tc.cu
long long* tc_timeline_next();

// fp32 NCHW <-> chunked bf16 converters (channel c of the source lands in chunk c/8, lane c%8)
int tc_pack_nchw(const float* src, int src_channels, int mode /*hv_src_mode*/, const TcBuf& dst, int dst_channel0,
                 cudaStream_t st);
// kx-packed variant for up to 4 single-channel sources (planes [n,1,h,w] / [n,1,2h,2w] (SUB2) / scalars [n]):
// dst channel kx*nsrc + c at (y, x) = source c at (y, x + (kx - k/2)*dil), zero outside the image
struct TcPlaneSrc { const float* ptr; int mode; };
int tc_pack_kx(const TcPlaneSrc* srcs, int nsrc, int k, int dil, const TcBuf& dst, cudaStream_t st);
// dst (16 channels, extent h/2 x w/2): channel ry * 4 + rx of (m, n) = src[n][2m - 1 + ry][2n - 1 + rx] (zero outside), src fp32 [n,1,h,w]
int tc_pack_nbhd4(const float* src, const TcBuf& dst, cudaStream_t st);
int tc_unpack_nchw(const TcBuf& src, int channel0, int channels, float* dst, cudaStream_t st, int sub = 1);
int tc_gap_fc_sigmoid(const TcBuf& x, const float* fc_w, const float* fc_b, float* out, float* partial /*[n*chunks]*/,
                      unsigned int* ticket /*[n], zero-initialised, left zero*/, cudaStream_t st);

// contextual attention on tensor cores (ctx_attn_tc.cu): f and y are 64-channel 64x64 chunked buffers
void tc_set_timeline(long long* dev_buf);   // debug: launch i records {first CTA entry, last CTA exit} at dev_buf[4 i], [4 i + 1]
size_t ctx_attn_tc_workspace_bytes(int n);
int ctx_attn_fwd_tc(const TcBuf& f, const float* mask, const TcBuf& y, int32_t* offsets, float* flow, float scale, int fuse,
                    int per_sample_mask, void* workspace, cudaStream_t st, cudaStream_t st_aux = nullptr, cudaEvent_t* evs = nullptr);

}  // namespace hv
