/*
 * wmd.h - C ABI of libwmd.so: the B200 (sm_100a) wavelet-monodepth decoder hot path.
 *
 * The reference (nianticlabs/wavelet-monodepth) has no native/FFI layer: its
 * boundary for this path is a Python nn.Module / function API built on ATen ops
 * and the un-vendored pytorch_wavelets package.  Every entry point below names
 * the reference interface it replaces (paths relative to the reference tree).
 * The Python mirror of that API lives in wavelet_monodepth_b200/ and reaches
 * these symbols through ctypes with tensor.data_ptr() (INTEGRATION.md).
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is DEVICE memory unless the
 *    name says host; all tensors are contiguous fp32 / int32 / uint8;
 *  - the caller owns every buffer; nothing is allocated, freed or retained;
 *  - every call is asynchronous on `stream` (a cudaStream_t), re-entrant, and
 *    never synchronises the device; data-dependent counts stay on the device;
 *  - return value: WMD_OK (0) or a negative wmd_status; never throws / exits.
 *
 * Sparse feature layout ("rows"): active pixels of all samples are enumerated
 * in (n, y, x) row-major order - the reference's order (KITTI/layers.py:377-378,
 * 387) extended over the batch - and a feature tensor is a row-major matrix
 * [rows][ld] (pixel-major, channels contiguous), not the reference's
 * channel-major (C, M) vector (layers.py:358).  wmd_nchw_to_rows_f32 /
 * wmd_rows_to_nchw_f32 (with N=1, HW=M) convert at the functional-API boundary.
 */
#ifndef WMD_H
#define WMD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WMD_VERSION 100 /* major*100 + minor */

typedef void* wmd_stream_t; /* cudaStream_t */

typedef enum wmd_status {
  WMD_OK = 0,
  WMD_ERR_ARG = -1,         /* null pointer / bad enum */
  WMD_ERR_SHAPE = -2,       /* unsupported size (odd extent, misaligned leading dim ...) */
  WMD_ERR_CUDA = -3,        /* a CUDA call failed; see wmd_last_cuda_error() */
  WMD_ERR_WORKSPACE = -4,   /* workspace too small */
  WMD_ERR_UNSUPPORTED = -5
} wmd_status;

enum { WMD_PAD_ZERO = 0, WMD_PAD_REFLECT = 1, WMD_PAD_REPLICATE = 2 };
enum { WMD_ACT_NONE = 0, WMD_ACT_ELU = 1, WMD_ACT_LRELU = 2, WMD_ACT_SIGMOID = 3 };

int wmd_version(void);
const char* wmd_status_string(int status);
/* last cudaError_t recorded by a failing call on this host thread (0 if none) */
int wmd_last_cuda_error(void);
/* number of kernels this library has launched on this host thread since load (bench.py's gpu_launches) */
long long wmd_launch_count(void);

/* ---------------------------------------------------------------- Haar transforms
 * Replaces pytorch_wavelets.DWTInverse.forward((yl,[yh])) for wave='haar', one level
 * (call sites KITTI/networks/decoders/depth_decoder.py:164,372,416;
 * NYUv2/networks/decoders/densedepth_decoder.py:129,137,145,309,357,404) and the
 * reference's closed form my_iwt_once (depth_decoder.py:225-239).
 *   ll (N,C,H,W), hf (N,C,3,H,W) [LH,HL,HH] -> out (N,C,2H,2W)
 *   out[2i+a,2j+b] = 1/2 (ll + (-1)^a lh + (-1)^b hl + (-1)^(a+b) hh), evaluated in
 *   the dependency's separable order (two 1/sqrt2 passes) so results are bit-equal to it.
 * Fused consumer (optional, disp may be NULL):
 *   disp  (N,C,2H,2W) = out * disp_scale, clamped to [0,1] if clamp01   (depth_decoder.py:166)
 */
int wmd_idwt_haar_f32(const float* ll, const float* hf, float* out, float* disp, float disp_scale, int clamp01,
                      int N, int C, int H, int W, wmd_stream_t stream);

/* Fused IDWT + disparity epilogue + bilinear resize: full (N,C,full_h,full_w) = bilinear(disp) with
 * disp = [clamp01](idwt(ll,hf) * disp_scale), PyTorch F.interpolate(mode="bilinear") index arithmetic for either
 * align_corners setting.  Replaces the consumers of ("disp", s): KITTI/trainer.py:338-339 (align_corners=False),
 * NYUv2/utils.py:223-227, NYUv2/train.py:305-306 (align_corners=True).  The intermediate disp plane is not read
 * back from HBM.  Supports upsampling (and downsampling up to ~1.3x). */
int wmd_idwt_bilinear_f32(const float* ll, const float* hf, float* full, float disp_scale, int clamp01, int full_h,
                          int full_w, int align_corners, int N, int C, int H, int W, wmd_stream_t stream);

/* Replaces one level of pytorch_wavelets.DWTForward.forward (NYUv2/train.py:258,289); also the
 * adjoint used for the IDWT's backward (KITTI/trainer.py:208-212 trains through inverse_wt).
 *   x (N,C,H,W), H and W even -> ll (N,C,H/2,W/2), hf (N,C,3,H/2,W/2) */
int wmd_dwt_haar_f32(const float* x, float* ll, float* hf, int N, int C, int H, int W, wmd_stream_t stream);

/* ---------------------------------------------------------------- threshold + masks
 * thresh[n] = (max(x_n) - min(x_n)) * ratio over per_sample contiguous floats of sample n.
 * Replaces `thresh = (yl.max() - yl.min()) * thresh_ratio` (depth_decoder.py:308;
 * densedepth_decoder.py:316,363), per sample instead of the reference's batch-1.
 * minmax (2N floats: min,max) is optional.  N <= 16384.  ws: wmd_range_ws_bytes() bytes whose first
 * 64 KiB (per-sample ticket counters) must be zero before the FIRST use only: the kernel leaves them
 * zeroed, for any later N, so one scratch buffer can be shared by all calls on a stream. */
size_t wmd_range_ws_bytes(int N, long long per_sample);
int wmd_range_thresh_f32(const float* x, int N, long long per_sample, float ratio, float* thresh, float* minmax,
                         void* ws, size_t ws_bytes, wmd_stream_t stream);

/* The six per-level pixel sets (depth_decoder.py:305-319, densedepth_decoder.py:316-322):
 *   S0 = max_band |yh| > thresh[n]  (strict; thresh == NULL -> all ones, the reference's level-4 case :305-306)
 *   S1 = dilate3(S0)  S2 = dilate5(S0)                  low resolution  (N,H,W)
 *   S5 = up2(S0)  S4 = dilate3(S5)  S3 = dilate5(S5)    high resolution (N,2H,2W)
 * yh is (N,3,H,W).  Any output pointer may be NULL.  Masks are 0/1 bytes. */
int wmd_level_masks(const float* yh, const float* thresh, uint8_t* s0, uint8_t* s1, uint8_t* s2, uint8_t* s3,
                    uint8_t* s4, uint8_t* s5, int N, int H, int W, wmd_stream_t stream);

/* Replaces mask2idxmap + mask2yx (KITTI/layers.py:371-389) for a whole batch, without the
 * reference's host sync (layers.py:385):
 *   idxmap  (N,H,W) int32 : running row index over the batch, -1 where inactive   [nullable]
 *   pixels  (<= N*H*W) int32 : linear pixel index (n*H + y)*W + x of each active pixel [nullable]
 *   offsets (N+1) int32 : offsets[n] = rows before sample n, offsets[N] = total rows */
size_t wmd_compact_ws_bytes(int N, int H, int W);
int wmd_compact_mask(const uint8_t* mask, int32_t* idxmap, int32_t* pixels, int32_t* offsets, int N, int H, int W,
                     void* ws, size_t ws_bytes, wmd_stream_t stream);

/* out[p] = gate[p] ? (idxmap ? idxmap[p] : p) : -1   for p < count.
 * The fused form of sparse_select (layers.py:337-362): re-indexing onto a subset is a map rewrite. */
int wmd_gate_map(const uint8_t* gate, const int32_t* idxmap, int32_t* out, long long count, wmd_stream_t stream);

/* ---------------------------------------------------------------- layout helpers
 * (N,C,HW) <-> (N,HW,ld) batched transposes (ld >= C; pad columns are zero-filled on the way in).
 * Used for NCHW encoder features -> pixel-major rows, and for the reference's channel-major
 * wire format (layers.py:358) at the functional API. */
int wmd_nchw_to_rows_f32(const float* src, float* dst, int N, int C, long long HW, int ld, wmd_stream_t stream);
int wmd_rows_to_nchw_f32(const float* src, float* dst, int N, int C, long long HW, int ld, wmd_stream_t stream);
/* Same move, but only for the pixels marked in gate (N, HW) bytes: rows of unmarked pixels are left untouched and
 * their source is not read (whole 32-pixel groups without a mark cost no traffic).  The sparse levels read a skip map
 * only under the level's upsample mask (sparse_upsample: skip[mask], KITTI/layers.py:500; the conv's gate argument
 * below), so the decoder passes that mask here and the transpose scales with the mask density. */
int wmd_nchw_to_rows_gated_f32(const float* src, float* dst, const uint8_t* gate, int N, int C, long long HW, int ld,
                               wmd_stream_t stream);
/* rows at an active-pixel list <-> dense NCHW (x[mask] selection, depth_decoder.py:347; make_result, layers.py:365-368) */
int wmd_gather_rows_nchw_f32(const float* src_nchw, float* rows, int ld, int C, const int32_t* pixels,
                             const int32_t* count, int max_rows, int N, int H, int W, wmd_stream_t stream);
int wmd_scatter_rows_nchw_f32(const float* rows, int ld, int C, const int32_t* pixels, const int32_t* count,
                              int max_rows, float* dst_nchw, int N, int H, int W, wmd_stream_t stream);
/* conv weight (Cout,Cin,kh,kw) -> packed [kh*kw][Cin][ldw] (ldw >= Cout, multiple of 4, pad zero) */
int wmd_pack_conv_weight_f32(const float* w, float* packed, int Cout, int Cin, int taps, int ldw, wmd_stream_t stream);

/* ---------------------------------------------------------------- fused 1x1 head stages
 * z = Wz . lrelu(W1 . x + b1): the 1x1 stages of a level's + / - coefficient heads (Conv1x1 + LeakyReLU(0.1),
 * depth_decoder.py:111-120) chained with the per-row tap products of their 3x3 stages (the 9 x 6 values
 * wmd_head_gather_f32 sums per pixel).  x rows (M, c), W1 (n1, c), Wz (nz <= 56, n1); z rows (M, ldz >= 56), columns
 * nz..55 are written as zeros.  The intermediate (M, n1) never reaches memory.  Supported (c, n1): (32, 64), (64, 128);
 * other shapes return WMD_ERR_UNSUPPORTED (the caller then runs the two stages as wmd_conv_rows launches). */
int wmd_head_mlp_supported(int c, int n1);
size_t wmd_head_mlp_weight_floats(int c, int n1);
int wmd_pack_head_mlp_f32(const float* w1, const float* wz, const float* b1, int c, int n1, int nz, float* packed,
                          wmd_stream_t stream);
int wmd_head_mlp_f32(const float* x, int ldx, int c, const float* packed, int n1, float slope, const int32_t* count,
                     int max_rows, float* z, int ldz, wmd_stream_t stream);

/* ---------------------------------------------------------------- gather-GEMM convolution
 * Replaces sparse_conv3x3 / sparse_conv1x1 / sparse_upsample / sparse_select (KITTI/layers.py:337-508,
 * NYUv2/networks/layers.py:82-223) and, with pixels == NULL, the dense Conv3x3/ConvBlock/Conv1x1 layers
 * (KITTI/layers.py:120-173) of the decoder.  For each output row m (pixel p = pixels[m], or m itself):
 *   y[m, :] = act( bias + sum_{tap, c} in(p + tap)[c] * w[tap][c][:] )
 * where in(q) is the channel concatenation of
 *   source 0: x0[ row0(q), 0:c0 ]  with row0(q) = map0[n, qy>>shift0, qx>>shift0]  (map0 NULL: that pixel's
 *             linear index; taps==1 && map0==NULL: row m itself), zero if row0 < 0        [sparse_select/upsample]
 *   source 1: x1[ (n*H+qy)*W+qx, 0:c1 ]  (dense pixel-major skip map at output resolution)  [skip concat, :500]
 * and in(q) = 0 entirely if gate != NULL and gate[q] == 0, or q is out of the image under WMD_PAD_ZERO.
 * q is mapped into the image by pad_mode exactly as padding the index map does (layers.py:444).
 */
typedef struct wmd_conv_desc {
  int32_t N, H, W;          /* output grid */
  const float* x0;          /* source 0 rows [*][ld0] */
  int32_t c0, ld0;
  const int32_t* map0;      /* (N, H>>shift0, W>>shift0) or NULL */
  int32_t shift0;           /* 0 or 1 */
  const float* x1;          /* source 1 rows [N*H*W][ld1] or NULL */
  int32_t c1, ld1;
  const uint8_t* gate;      /* (N,H,W) or NULL */
  const float* w;           /* packed [taps][c0+c1][ldw] */
  const float* bias;        /* [cout] or NULL */
  int32_t cout, ldw, taps;  /* taps: 1 or 9 */
  int32_t pad_mode;         /* WMD_PAD_* */
  const int32_t* pixels;    /* active output list or NULL (= every pixel) */
  const int32_t* count;     /* device row count (with pixels) */
  int32_t max_rows;         /* capacity of y / upper bound of *count */
  float* y;                 /* rows [max_rows][ldy] */
  int32_t ldy;
  int32_t act;              /* WMD_ACT_* */
  float act_param;          /* LeakyReLU slope */
  const int32_t* map1;      /* (N,H,W): row of pixel q in x1, -1 = none; NULL = x1 is dense (row q).  With a map, x1 holds
                               only the rows of the listed pixels (sparse_upsample's skip[mask], KITTI/layers.py:500, kept
                               compact: wmd_gather_rows_list_f32) */
  int32_t precision;        /* tensor-core engine only.  0 = WMD_PREC_TF32X3: operands split into tf32 hi + lo.  1 = WMD_PREC_F16X3:
                               operands split into two fp16 pieces of x * 2^k (same 22 mantissa bits; k from amax0 / amax1, so
                               nothing overflows) - half the MMA instructions and twice their rate; needs amax0 (and amax1 when
                               c1 > 0) and weights packed by wmd_pack_conv_weight_tc16_f32 */
  const float* amax0;       /* device scalars: max |x0|, max |x1| over the rows the launch can read (upper bounds are fine) */
  const float* amax1;
  float* amax_out;          /* device scalar, or NULL: atomically raised to max |y| of the rows written (zero it before the
                               first producer; both precisions) */
  int32_t rows0;            /* rows allocated in x0, 0 = unknown.  Only used by the tensor-core engine's 1x1 form (taps == 1,
                               map0 == NULL: output row m reads x0 row m) without a gate: with rows0 > 0 it loads source 0 in
                               whole 256-row tiles by TMA (reads past rows0 are zero-filled) instead of gathering row by row */
} wmd_conv_desc;

int wmd_conv_rows_f32(const wmd_conv_desc* d, wmd_stream_t stream);

/* Tensor-core engine for the same contract: tcgen05.mma.kind::tf32 with a 3xTF32 split (hi*hi + lo*hi + hi*lo,
 * fp32 accumulation in TMEM), so results stay fp32-faithful: max|y - ref| / max|ref| <= 8e-6 against an fp64 reference
 * at any K (4e-6 in the f16x3 form; the SIMT kernel: 1.2e-6), measured on B200 by tests/test_gpu_conv_reference.py.  d->w must
 * point to weights packed by wmd_pack_conv_weight_tc_f32 for the same (cout, c0, c1, taps); d->ldw is ignored.
 *   wmd_conv_tc_tile_n(cout)                 N-tile of the kernel for this cout (128 / 64 / 32; the CTA tile is 256 rows x N)
 *   wmd_conv_tc_weight_floats(...)           size of the packed weight buffer, in floats
 *   wmd_pack_conv_weight_tc_f32(w, packed..) (Cout, c0+c1, kh, kw) -> per (n-tile, 32-channel chunk) fp32
 *                                            shared-memory images [tf32 hi | tf32 lo] of N x 32, K-major, 128-byte swizzled
 * Accumulation runs in epochs of K = 1024 inside TMEM and is drained into fp32 registers with round-to-nearest
 * adds, because the tensor core's own fp32 accumulation rounds toward zero (bias ~6.5e-9 * K relative). */
enum { WMD_PREC_TF32X3 = 0, WMD_PREC_F16X3 = 1 };
int wmd_conv_tc_tile_n(int cout);
/* Weights for precision = WMD_PREC_F16X3: 128-byte header (float 0: 1 / s_w) + per (n-tile, 32-channel chunk) one N x 128 B
 * image whose rows hold [fp16(w s_w): 32 channels | fp16(w s_w - that): 32 channels], s_w = the power of two that puts
 * max |w| into (2^13, 2^14] (computed on the device, no host sync).  `packed` needs wmd_conv_tc16_weight_bytes() bytes. */
size_t wmd_conv_tc16_weight_bytes(int cout, int c0, int c1, int taps);
int wmd_pack_conv_weight_tc16_f32(const float* w, void* packed, int Cout, int c0, int c1, int taps, wmd_stream_t stream);
/* max |x| of `count` floats, atomically raised into *amax (device scalar, zero it first): for sources that no libwmd
 * kernel produced (channels_last feature maps used in place).  The layout moves below take an optional `amax` too. */
int wmd_amax_f32(const float* x, long long count, float* amax, wmd_stream_t stream);
int wmd_nchw_to_rows_amax_f32(const float* src, float* dst, int N, int C, long long HW, int ld, float* amax, wmd_stream_t stream);
/* gated move: the maximum covers the 32-pixel groups that hold a marked pixel (a superset of the rows written) */
int wmd_nchw_to_rows_gated_amax_f32(const float* src, float* dst, const uint8_t* gate, int N, int C, long long HW, int ld,
                                    float* amax, wmd_stream_t stream);
int wmd_gather_rows_list_amax_f32(const float* src_nchw, float* rows, int ld, int C, const int32_t* pixels,
                                  const int32_t* count, int max_rows, int N, int H, int W, float* amax, wmd_stream_t stream);
size_t wmd_conv_tc_weight_floats(int cout, int c0, int c1, int taps);
int wmd_pack_conv_weight_tc_f32(const float* w, float* packed, int Cout, int c0, int c1, int taps, wmd_stream_t stream);
int wmd_conv_rows_tc_f32(const wmd_conv_desc* d, wmd_stream_t stream);
/* Same, with the reduction split `splits` ways across CTAs (split-K): layers with few output tiles then fill all
 * SMs.  Partial sums go to `ws` (wmd_conv_tc_splitk_ws_bytes) and are summed in a fixed order, biased and
 * activated by a second small kernel, so results stay deterministic.  splits = 1 is wmd_conv_rows_tc_f32.
 * splits = 0 selects BALANCED scheduling (data-parallel + stream-K): full rounds of tiles run whole; the (tile,
 * 32-channel chunk) units of the remainder tiles are dealt to the CTAs in equal contiguous ranges computed on the
 * device from the actual row count, so sparse layers whose tile count is data dependent still finish on all SMs
 * together; only remainder tiles cut by a range boundary (<= 8 segments) go through the workspace: the LAST segment of
 * a tile to arrive (per-tile arrival counter) sums all of them in slab order - bias first - inside the same kernel, so
 * there is no second pass and the bits do not depend on the arrival order.  Its workspace size does not depend on the
 * layer (4 KiB of counters + SMs x 8 x 256 x 128 floats).  The first 4 KiB of `ws` (any splits) must be ZERO before the
 * first launch that uses the buffer; every launch leaves them zero. */
size_t wmd_conv_tc_splitk_ws_bytes(int max_rows, int ldy, int splits);
/* 3x3 layers gather the A operand once per (channel chunk, dy) and feed the three dx taps from that one shared-memory
 * stage through a per-tile slot table (sparse_conv3x3's nine shifted selections, KITTI/layers.py:445-453, read almost the
 * same rows).  On by default; wmd_conv_tc_set_shared_taps(0) restores one gather per tap (A/B measurements, tests:
 * both forms produce identical bits).  on < 0 only queries.  Returns the previous setting.  Process-wide. */
int wmd_conv_tc_set_shared_taps(int on);
/* The tcgen05 engine runs one persistent CTA per SM, and such a CTA holds the SM's whole register file: no other kernel -
 * an NCCL collective of the previous step in particular - can run beside it.  wmd_conv_tc_set_reserved_sms(n) makes the
 * persistent grid n CTAs smaller so that n SMs stay free (multi-GPU serving: the all-gather of step k then really runs
 * under the convolutions of step k + 1).  0 by default; n < 0 only queries.  Returns the previous setting.  Process-wide;
 * set it before capturing CUDA graphs. */
int wmd_conv_tc_set_reserved_sms(int n);
int wmd_conv_rows_tc_splitk_f32(const wmd_conv_desc* d, int splits, void* ws, size_t ws_bytes, wmd_stream_t stream);

/* ---------------------------------------------------------------- coefficient heads (few output channels)
 * The 3x3 stage of the wavelet heads (depth_decoder.py:104-120,126-136,242-290; NYU wave convs
 * densedepth_decoder.py:104-115) on pixel-major rows `t`, scattered to a dense NCHW tensor:
 *   a = conv3x3(t[:, off_a:off_a+c]; wa, ba)   b = conv3x3(t[:, off_b:off_b+c]; wb, bb)   (off_b < 0: single head)
 *   out[n, :, y, x] = scale * (act(a) - act(b))     or   scale * act(a)
 * out must be zero-filled by the caller when pixels != NULL (the reference's make_result, layers.py:473-478).
 */
typedef struct wmd_head_desc {
  int32_t N, H, W;
  const float* t;
  int32_t ld, c, off_a, off_b;
  const int32_t* map;       /* (N,H,W) row of each pixel, -1 inactive; NULL = linear pixel index */
  const float* wa; const float* ba;   /* packed [9][c][cout], bias [cout] */
  const float* wb; const float* bb;
  int32_t cout;             /* 1..4 */
  int32_t pad_mode, act;
  float scale;
  const int32_t* pixels; const int32_t* count; int32_t max_rows;
  float* out;               /* (N,cout,H,W) */
} wmd_head_desc;

int wmd_head_conv3x3_f32(const wmd_head_desc* d, wmd_stream_t stream);

/* Factored form of the same stage (what the decoders use for the +/- heads): the per-tap products
 * z[row, tap*groups + g] = t[row, :] . w_g[:, tap] are computed once per active input row by wmd_conv_rows_*_f32
 * (taps = 1, cout = 9*groups); this entry point gathers and sums the nine taps per output pixel,
 *   s_g = bias[g] + sum_tap z[map(p + tap), tap*groups + g],
 * and scatters  out[n, j, y, x] = scale * (act(s_j) - act(s_{cout+j}))  (dual, groups = 2*cout)  or  scale * act(s_j)
 * (groups = cout) into the dense NCHW tensor (zero-filled by the caller when pixels != NULL).  groups in {1,2,3,4,6,8}. */
int wmd_head_gather_f32(const float* z, int ldz, int groups, const int32_t* map, const float* bias, float scale, int act,
                        int dual, int pad_mode, const int32_t* pixels, const int32_t* count, int max_rows, float* out,
                        int cout, int N, int H, int W, wmd_stream_t stream);

/* ---------------------------------------------------------------- fused tail of a decoder level
 * One kernel for:  factored 3x3 stage of the +/- coefficient heads (get_coefficients / get_sparse_coefficients,
 * depth_decoder.py:126-136,242-290: yh = 2^(i-1) (sigmoid(.) - sigmoid(.)), zero outside the wavelet mask)
 *                  -> pytorch_wavelets.DWTInverse (depth_decoder.py:164,372,416)
 *                  -> disp = clamp(yl / 2^(i-1), 0, 1) (depth_decoder.py:166)
 *                  -> the consumer's epilogue of ("disp", 0): disp_to_depth (KITTI/layers.py:16-25) or depth / 100
 *                     + clamp (NYUv2/utils.py:219,229)
 *                  -> thresh = (max - min)(yl) * ratio of the NEXT level's masks (depth_decoder.py:308), per sample.
 * z: rows of tap products from wmd_head_mlp_f32 / the tap-product GEMM, 54 floats [tap][+LH,+HL,+HH,-LH,-HL,-HH] from
 * z[0] (pass z + col0 for a column offset), row of pixel q = map[q] (map == NULL: q), pixels with mask == 0 (mask != NULL)
 * get zero coefficients.  yh (N,3,H,W) is written once (an output of the decoder) and not read back; out / disp are
 * (N,1,2H,2W).  ll / mask rows of a tile are staged by TMA bulk copies when W % 16 == 0.  Results are bit-identical to
 * wmd_head_gather_f32 + wmd_idwt_haar_f32 + wmd_range_thresh_f32.  thresh == NULL skips the range reduction (then ws may
 * be NULL); otherwise ws needs wmd_head_idwt_ws_bytes() bytes whose first 64 KiB are zero before the first use (the kernel
 * leaves them zeroed, like wmd_range_thresh_f32). */
enum { WMD_EPI_NONE = 0, WMD_EPI_DISP_TO_DEPTH = 1, WMD_EPI_DIV_CLAMP = 2 };
typedef struct wmd_head_idwt_desc {
  int32_t N, H, W;           /* coefficient grid of the level */
  const float* z;            /* tap-product rows [*][ldz] */
  int32_t ldz;
  const int32_t* map;        /* (N,H,W) row of a pixel in z, -1 = none; NULL = linear index */
  const uint8_t* mask;       /* (N,H,W) wavelet mask (S5) or NULL = every pixel */
  const float* bias;         /* [6]: + head's 3 biases then - head's, or NULL */
  float scale;               /* 2^(i-1) */
  int32_t pad_mode;          /* WMD_PAD_* of the heads' 3x3 stage */
  const float* ll;           /* (N,1,H,W) */
  float* yh;                 /* (N,3,H,W) */
  float* out;                /* (N,1,2H,2W) reconstruction */
  float* disp;               /* (N,1,2H,2W) = [clamp01](out * disp_scale), or NULL */
  float disp_scale;
  int32_t clamp01;
  int32_t epi_mode;          /* WMD_EPI_*: DISP_TO_DEPTH: epi_out0 = epi_a + epi_b * disp, epi_out1 = 1 / epi_out0 (nullable);
                                DIV_CLAMP: epi_out0 = out / epi_a, clamped to [epi_lo, epi_hi] if epi_b != 0 */
  float epi_a, epi_b, epi_lo, epi_hi;
  float* epi_out0;
  float* epi_out1;
  float* thresh;             /* (N) (max - min)(out_n) * thresh_ratio, or NULL */
  float thresh_ratio;
} wmd_head_idwt_desc;
/* The plain IDWT with the same consumer epilogue (NYU decoders: the last level's reconstruction IS ("disp", 0)). */
int wmd_idwt_haar_epi_f32(const float* ll, const float* hf, float* out, float* disp, float disp_scale, int clamp01,
                          int epi_mode, float epi_a, float epi_b, float epi_lo, float epi_hi, float* epi_out0,
                          float* epi_out1, int N, int C, int H, int W, wmd_stream_t stream);
/* rows[m][0..C) = src[n, :, y, x] for the m-th pixel of a list (pixels[m] = (n*H + y)*W + x, m < *count), columns C..ld-1
 * zero: the layout move of a skip map restricted to EXACTLY the active pixels (the reference's skip[mask],
 * KITTI/layers.py:500) - 128 list entries x 32 channels per tile, coalesced on both sides for clustered lists.  `src` may
 * be pinned HOST memory (read in place over PCIe: only the listed pixels cross the bus).  ld % 4 == 0. */
int wmd_gather_rows_list_f32(const float* src_nchw, float* rows, int ld, int C, const int32_t* pixels, const int32_t* count,
                             int max_rows, int N, int H, int W, wmd_stream_t stream);
size_t wmd_head_idwt_ws_bytes(int N, int H, int W);
int wmd_head_idwt_f32(const wmd_head_idwt_desc* d, void* ws, size_t ws_bytes, wmd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* WMD_H */
