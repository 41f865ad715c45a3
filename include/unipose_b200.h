/*
 * unipose_b200.h — C-ABI of the B200-native (sm_100a) UniPose hot path.
 *
 * The reference (bmartacho/UniPose) is pure PyTorch and has no FFI of its own; every entry
 * point below replaces the ATen/cuDNN operator that a reference `nn.Module.forward()` call
 * dispatches to.  The citation beside each function names the reference call site
 * (file:line under /root/reference) whose arithmetic the function implements.
 *
 * Conventions
 *   - plain pointers + sizes; no torch types.  All pointers are DEVICE pointers unless named h_*.
 *   - every function returns 0 on success or a negative UpStatus; `up_last_error()` returns a
 *     thread-local human readable message.  Nothing throws across the ABI.
 *   - all launches are asynchronous on the `stream` argument (a cudaStream_t passed as void*);
 *     the library never synchronises and never allocates persistent device memory.
 *   - activations are NHWC, 16-bit (bf16 or fp16).  In UP_SPLIT mode a tensor is TWO bf16
 *     planes (hi, lo = bf16(x - hi)) `plane_stride` elements apart; GEMMs then run the three
 *     bf16 products hi*hi + lo*hi + hi*lo with fp32 accumulation (fp32-grade results on the
 *     bf16 tensor cores).  The user-facing tensors (input image, heat-maps, ConvLSTM states)
 *     are fp32 NCHW exactly as in the reference.
 */
#ifndef UNIPOSE_B200_H_
#define UNIPOSE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UP_VERSION 100

typedef enum UpStatus {
  UP_OK = 0,
  UP_ERR_INVALID = -1,   /* bad shape / alignment / flag combination */
  UP_ERR_CUDA = -2,      /* CUDA runtime or driver call failed */
  UP_ERR_UNSUPPORTED = -3
} UpStatus;

typedef enum UpDtype {
  UP_BF16 = 0,  /* bf16 storage, one tensor-core pass */
  UP_FP16 = 1,  /* fp16 storage, one tensor-core pass */
  UP_SPLIT = 2  /* bf16 hi+lo planes, three tensor-core passes: fp32-grade ("parity") mode */
} UpDtype;

enum {
  UP_FLAG_RELU = 1,          /* y = max(y, 0) after scale/shift(/residual) */
  UP_FLAG_RESIDUAL = 2,      /* the residual tile (same NHWC geometry as y) is accumulated INSIDE the tensor-core
                                pipeline (identity MMA into the fp32 accumulator): y = act(scale*(conv + res) + shift).
                                Callers fold a BatchNorm scale into the weights and pass scale = 1. */
  UP_FLAG_OUT_NCHW_F32 = 4,  /* write fp32 NCHW [n, cout_valid, ho, wo] instead of 16-bit NHWC */
  UP_FLAG_PROJ = 16,         /* projection shortcut of a stage's first bottleneck (resnet.py:36-37: out += downsample(x))
                                inside the same GEMM: `residual` points to a SECOND input x2 [n, ho*proj_stride,
                                wo*proj_stride, r_cstride] (view r_coff .. r_coff + proj_cin) whose 1x1 projection of
                                stride proj_stride extends K.  1x1 stride-1 main filter, 16-bit NHWC output, not with
                                UP_FLAG_RESIDUAL / UP_SPLIT.  Packed filter: [1 + proj_cin / cin][cout][cin] - the
                                projection's filter follows the main one as proj_cin / cin slices of cin columns. */
  UP_FLAG_STATS = 8          /* RESERVED: per-channel sum / sum-of-squares of the stored output fused into the
                                epilogue.  Not implemented in this build - up_conv2d_fwd rejects it with an error;
                                train-mode BatchNorm statistics come from up_bn_stats. */
};

const char* up_last_error(void);
int up_version(void);
/* Number of SMs / compute capability of the current device (for tests and the bench). */
int up_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (TMA-staged, im2col-free), fused
 * per-channel scale/shift (+residual) (+ReLU) epilogue.
 *
 * Replaces every nn.Conv2d (+ eval-mode BatchNorm2d + ReLU + residual add) of the hot path:
 *   Bottleneck.forward            model/modules/backbone/resnet.py:22-42
 *   ResNet.forward stem           model/modules/backbone/resnet.py:114-116 (as a 4x4 conv on the
 *                                 2x2 space-to-depth image, see up_pack_input_s2d)
 *   _AtrousModule.forward         model/modules/wasp.py:16-20
 *   wasp.forward conv1/conv2      model/modules/wasp.py:72-88
 *   Decoder.forward               model/modules/decoder.py:39-41,52
 *   video "middle CNN" conv1..5   model/uniposeLSTM.py:120-124
 *
 * Geometry: y[n,ho,wo,co] = sum_{kh,kw,ci} w[co,kh,kw,ci] * x[n, ho*stride + kh*dil - pad_h,
 *                                                            wo*stride + kw*dil - pad_w, ci]
 * (cross-correlation, zero padding; the bottom/right padding is implied by ho/wo).
 * stride is 1 or 2 (2 needs even h, w).  Channel counts are the PADDED ones: cin % 16 == 0
 * (and % 64 == 0 when cin > 64 ... see up_conv2d_check), cout % 32 == 0.
 *
 * Weights are pre-packed by up_pack_conv_weight: 16-bit [plane][kh*kw][cout][cin].
 * scale/shift are fp32 [cout] (eval BatchNorm folded, or scale=1 / shift=bias).
 * ------------------------------------------------------------------------------------------ */
typedef struct UpConvDesc {
  int32_t n, h, w;       /* input batch / height / width */
  int32_t ho, wo;        /* output height / width */
  int32_t cin, cout;     /* padded channel counts seen by the GEMM */
  int32_t kh, kw;
  int32_t stride, dil;
  int32_t pad_h, pad_w;  /* top / left zero padding */
  int32_t x_cstride, x_coff;   /* channels per pixel of the x buffer, first channel of the view */
  int32_t x_groups;            /* K-split concat: cin = x_groups * (cin / x_groups); group g of the
                                  channels lives x_group_nstride images further along n */
  int32_t x_group_nstride;
  int32_t y_cstride, y_coff;
  int32_t r_cstride, r_coff;   /* residual view (UP_FLAG_RESIDUAL) */
  int32_t dtype;               /* UpDtype */
  int32_t flags;               /* UP_FLAG_* */
  int32_t cout_valid;          /* UP_FLAG_OUT_NCHW_F32: number of real output channels written */
  int32_t out_c_total;         /* UP_FLAG_OUT_NCHW_F32: channels of the fp32 NCHW destination (0 -> cout_valid);
                                  lets the head write the first cout_valid channels of a wider tensor */
  int32_t x_cextent;           /* 0, or > x_cstride: OVERLAPPING channel windows - the K-chunk of a "pixel" spans
                                  x_cextent consecutive elements (several neighbouring pixels) while pixels stay
                                  x_cstride elements apart (stride 1, x_groups 1).  The 2x2 space-to-depth stem uses
                                  x_cstride 16 / x_cextent 64: one K-chunk = 4 horizontal taps x 16 channels. */
  int32_t x_wpitch;            /* 0, or the row pitch of x in pixels when rows are padded (>= w) */
  int64_t x_plane_stride;      /* UP_SPLIT: elements between hi and lo planes */
  int64_t y_plane_stride;
  int64_t r_plane_stride;
  int64_t w_plane_stride;
  int32_t proj_cin;            /* UP_FLAG_PROJ: channels of the second input that are projected (multiple of cin) */
  int32_t proj_stride;         /* UP_FLAG_PROJ: 1 or 2 */
} UpConvDesc;

int up_conv2d_fwd(const UpConvDesc* desc, const void* x, const void* w_packed, const float* scale,
                  const float* shift, const void* residual, void* y, float* stats, void* stream);

/* ------------------------------------------------------------------------------------------
 * The whole WASP block as ONE persistent kernel (eval mode, fp16 / bf16): wasp.forward, model/modules/wasp.py:66-90
 * (waspVideo.py:67-91 with shift_gap = 0).  aspp1 -> aspp2 -> aspp3 -> aspp4 cascade with per-image dependencies (no
 * grid barrier), conv1 accumulated stage by stage from the on-chip tiles, pooling branch folded into a per-image bias.
 * Filters are the packed / folded ones the layer-wise plan uses (BatchNorm scales folded in, conv2 o conv2 folded into
 * conv1); `gap_t` and `conv1_pool_t` are TRANSPOSED packings (UpPackJob.transpose = 1).
 *   x [n,h,w,cin] dense NHWC 16-bit;  s_stack [4n,h,w,256]: receives x1..x4 (stage s at images [s*n, (s+1)*n));
 *   out [n,h,w,256];  workspace: up_wasp_chain_workspace_bytes() bytes, 256-byte aligned, ZEROED ONCE by the caller
 *   (the kernel re-arms its counters itself).  up_wasp_chain_supported() == 0 when the shape can take this path
 *   (otherwise callers run the layer-wise convolutions).
 * ------------------------------------------------------------------------------------------ */
typedef struct UpWaspChainDesc {
  int32_t n, h, w, cin;
  int32_t dil[3];        /* dilation (= padding) of aspp2 / aspp3 / aspp4 */
  int32_t dtype;         /* UP_FP16 or UP_BF16 */
  int32_t conv1_cin;     /* K of the packed conv1' filter: 5 groups of 256 */
} UpWaspChainDesc;

typedef struct UpWaspChainWeights {
  const void* aspp[4];        /* packed [taps][256][cin_s] */
  const float* shift[4];      /* [256] BatchNorm shifts */
  const void* conv1;          /* packed [1][256][conv1_cin] */
  const float* shift1;        /* bn1 shift [256] */
  const void* gap_t;          /* pooling-branch 1x1, transposed packing [1][cin][256] */
  const float* shift_gap;     /* [256] */
  const void* conv1_pool_t;   /* conv1' group 5 (pooling branch), transposed packing [1][256][256] */
} UpWaspChainWeights;

int up_wasp_chain_supported(const UpWaspChainDesc* desc);
int64_t up_wasp_chain_workspace_bytes(const UpWaspChainDesc* desc);
int up_wasp_chain_fwd(const UpWaspChainDesc* desc, const UpWaspChainWeights* weights, const void* x, void* s_stack,
                      void* out, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * A run of identical stride-1 bottlenecks without downsample path (layer3 blocks 1..22 of the dilated ResNet-101,
 * Bottleneck.forward model/modules/backbone/resnet.py:22-42) as ONE persistent kernel (eval mode, fp16 / bf16,
 * planes = 256): per-image halo dependencies through release/acquire counters, conv3 -> next conv1 accumulated on
 * chip, residual added inside the tensor-core pipe.
 *   xa: [n,h,w,1024] input X_0 (overwritten: ping buffer), xb: [n,h,w,1024] pong buffer; block b reads X_b from
 *   (b even ? xa : xb) and writes X_{b+1} to the other one -> the result is in (nblocks even ? xa : xb).
 *   t1: [2n,h,w,256] scratch (conv1 outputs, double buffered).  Filters packed CONTIGUOUSLY over the blocks:
 *   w1 [nblocks][256][1024], w2 [nblocks][9][256][256], w3 [nblocks][1024][256] (BatchNorm scales folded in),
 *   shifts fp32 [nblocks][256] / [nblocks][256] / [nblocks][1024].  workspace: zeroed once by the caller.
 * ------------------------------------------------------------------------------------------ */
typedef struct UpBneckChainDesc {
  int32_t n, h, w;
  int32_t planes;      /* 256 */
  int32_t nblocks;
  int32_t dil;         /* dilation (= padding) of the 3x3 convs */
  int32_t dtype;       /* UP_FP16 or UP_BF16 */
} UpBneckChainDesc;

typedef struct UpBneckChainWeights {
  const void* w1;
  const void* w2;
  const void* w3;
  const float* shift1;
  const float* shift2;
  const float* shift3;
} UpBneckChainWeights;

int up_bneck_chain_supported(const UpBneckChainDesc* desc);
int64_t up_bneck_chain_workspace_bytes(const UpBneckChainDesc* desc);
int up_bneck_chain_fwd(const UpBneckChainDesc* desc, const UpBneckChainWeights* weights, void* xa, void* xb, void* t1,
                       void* workspace, int64_t workspace_bytes, void* stream);
int up_debug_bneck_timing(unsigned long long* h_out);

/* ------------------------------------------------------------------------------------------
 * Second half of a bottleneck as one launch (eval mode, fp16 / bf16, planes 64 or 128, stride 1):
 *   y = ReLU( bn3(conv3( ReLU(bn2(conv2_3x3(t1))) )) + residual )        Bottleneck.forward, resnet.py:28-41
 * The 3x3 output stays in shared memory (it is the A operand of the 1x1 expansion); the residual enters the
 * accumulator as identity MMAs.  t1 [n,h,w,planes], residual and y [n,h,w,4*planes], all dense NHWC 16-bit;
 * w2 packed [9][planes][planes], w3 packed [1][4*planes][planes] (BatchNorm scales folded in), shifts fp32.
 * ------------------------------------------------------------------------------------------ */
typedef struct UpBneckTailDesc {
  int32_t n, h, w;
  int32_t planes;      /* 64 or 128 */
  int32_t dil;         /* dilation (= padding) of the 3x3 conv */
  int32_t dtype;       /* UP_FP16 or UP_BF16 */
  int32_t proj_cin;    /* 0: identity shortcut (`residual` = the block input, 4*planes channels);
                          > 0 (multiple of 64): projection shortcut of a stage's first block (resnet.py:36-37,
                          `downsample` = 1x1 conv + BN, stride 1): `residual` = the block input x [n,h,w,proj_cin],
                          wd packed [1][4*planes][proj_cin] (BN scale folded in), shiftd fp32 [4*planes] -
                          Wd x is accumulated into the output accumulator, the shortcut tensor is never written */
  int32_t next_planes; /* 0, or (planes 64 only) 64 / 128: ALSO compute the following bottleneck's conv1 + bn1 + ReLU
                          (resnet.py:25-27: 1x1, 4*planes -> next_planes, stride 1) from the output tile while it is on
                          chip: t1n [n,h,w,next_planes] = ReLU(w1n . y + shift1n), w1n packed [1][next_planes][4*planes]
                          (BN scale folded in).  The following block then starts at its 3x3 conv. */
} UpBneckTailDesc;
int up_bneck_tail_supported(const UpBneckTailDesc* desc);
int up_bneck_tail_fwd(const UpBneckTailDesc* desc, const void* t1, const void* w2, const float* shift2, const void* w3,
                      const float* shift3, const void* residual, const void* wd, const float* shiftd, void* y,
                      const void* w1n, const float* shift1n, void* t1n, void* stream);

/* Debug aid (UP_DEBUG_TIMING=1): per-CTA phase timestamps (ns) of the last up_wasp_chain_fwd launch, 160 CTAs x 32 slots. */
int up_debug_chain_timing(unsigned long long* h_out);
/* Debug aid (UP_DEBUG_TIMING=1 in the environment): per-CTA phase timestamps (ns) of the last up_conv2d_fwd launch,
 * 160 CTAs x 16 slots, copied to host memory (synchronising). */
int up_debug_conv_timing(unsigned long long* h_out);

/* Pack OIHW fp32 weights [cout_real][cin_real][kh][kw] -> 16-bit [plane][kh*kw][cout][cin]
 * (zero padded).  dtype UP_SPLIT writes two bf16 planes `w_plane_stride` elements apart. */
int up_pack_conv_weight(const float* w_oihw, void* w_packed, int cout_real, int cin_real, int kh, int kw,
                        int cout, int cin, int dtype, int64_t w_plane_stride, void* stream);

/* Fold eval-mode BatchNorm2d into per-channel scale/shift (torch semantics, eps inside sqrt):
 *   scale = gamma / sqrt(var + eps), shift = beta - mean * scale;  channels >= c_real get 0/0.
 * nn.BatchNorm2d call sites: resnet.py:26,30,34 wasp.py:18,86 decoder.py:40 */
int up_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
               float* scale, float* shift, int c_real, int c, void* stream);

/* Table-driven weight preparation: one launch for every filter / every epilogue constant of a plan (the per-layer
 * up_pack_conv_weight + up_bn_fold calls above remain for single layers).  Job tables live in DEVICE memory.
 *
 * UpPackJob: OIHW fp32 `w` [cout_real][cin_total][kh][kw] -> 16-bit `out` [plane][kh*kw][rows][cols], zero padded.
 *   transpose = 0 (forward layout): rows = padded cout, cols = padded cin; element (tap, co, ci) = w[co][ci_off+ci][tap]
 *   transpose = 1 (dgrad layout, what loss.backward() needs for the input gradient): rows = padded input channels of
 *     the slice [ci_off, ci_off+cin_slice), cols = padded cout; element (tap, ci, co) = w[co][ci_off+ci][taps-1-tap]
 *   row_scale (optional): every output channel co is multiplied by row_scale[co % scale_period] (folded eval BatchNorm).
 *   tile_start: exclusive prefix sum of up_pack_job_tiles() over the table (filled by the caller).
 * UpEpilogueJob: the fp32 [cout] scale / shift vectors of the conv epilogue from an eval-mode BatchNorm2d
 *   (torch semantics, resnet.py:26-34) or a conv bias; fold_into_weights = 1 writes gamma/sqrt(var+eps) to fold_scale
 *   [c_bn] (to be used as UpPackJob.row_scale) and leaves scale = 1. */
typedef struct UpPackJob {
  const float* w;
  void* out;
  const float* row_scale;
  int64_t plane_stride;   /* UP_SPLIT: elements between the hi and lo planes of `out` */
  int64_t tile_start;
  int32_t kh, kw;
  int32_t rows, cols;
  int32_t cout_real;
  int32_t cin_total, ci_off, cin_slice;
  int32_t scale_period;
  int32_t dtype;          /* UpDtype */
  int32_t transpose;
  int32_t reserved;
} UpPackJob;

typedef struct UpEpilogueJob {
  const float* gamma;     /* BatchNorm weight / bias / running_mean / running_var [c_bn]; unused when c_bn == 0 */
  const float* beta;
  const float* mean;
  const float* var;
  const float* bias;      /* conv bias [bias_len] when c_bn == 0 (may be NULL) */
  float* fold_scale;      /* [c_bn] or NULL */
  float* scale;           /* [cout] */
  float* shift;           /* [cout] */
  float eps;
  int32_t c_bn, bias_len;
  int32_t cout_real, cout;   /* channels >= cout_real get scale = shift = 0; the BN / bias vectors repeat with period
                                c_bn / bias_len (the stem's four-pixels-per-super-pixel output) */
  int32_t fold_into_weights;
  int32_t reserved[2];
} UpEpilogueJob;

int64_t up_pack_job_tiles(const UpPackJob* h_job);   /* HOST pointer: thread blocks this job needs */
int up_pack_conv_weights(const UpPackJob* d_jobs, int njobs, int64_t total_tiles, void* stream);
int up_epilogue_consts(const UpEpilogueJob* d_jobs, int njobs, int max_channels, void* stream);

/* ------------------------------------------------------------------------------------------
 * Bandwidth kernels (NHWC 16-bit unless noted)
 * ------------------------------------------------------------------------------------------ */
/* fp32 NCHW image [n,3,h,w] -> 2x2 space-to-depth NHWC [n,h/2,w/2,16] (12 real channels, order
 * (ph,pw,c)), so that the 7x7/s2 stem (resnet.py:61,114) becomes a 4x4/s1 tensor-core conv.  Rows of y may
 * be padded: pixel (yq, xq) is written at row pitch y_wpitch (0 -> w/2) and column xq + y_wpad_left; the
 * padding pixels are left untouched (the caller zero-fills them once). */
int up_pack_input_s2d(const float* x_nchw, void* y, int n, int h, int w, int dtype, int64_t y_plane_stride,
                      int y_wpitch, int y_wpad_left, void* stream);
/* uint8 HWC images [n,h,w,3] (what cv2.imread / a video decoder delivers) -> (x - mean) / std -> the same space-to-depth
 * tensor as up_pack_input_s2d: utils/mpii_data.py:184-185 (Mytransforms.to_tensor + normalize with mean 128, std 256)
 * fused with the stem's input packing; a quarter of the host->device bytes of the fp32 NCHW path, identical bits. */
int up_pack_input_u8_s2d(const uint8_t* x_nhwc, void* y, int n, int h, int w, int dtype, int64_t y_plane_stride,
                         int y_wpitch, int y_wpad_left, float mean, float std_, void* stream);
/* Ragged batch of decoded uint8 HWC images (3 channels, any sizes) -> the network input, in one launch:
 * cv2.resize(img, (out_w, out_h)) (utils/mpii_data.py:159-162, utils/lsp_lspet_data.py:211, penn_action_data.py),
 * bit for bit OpenCV's 8-bit INTER_LINEAR path (11-bit fixed-point weights, the SIMD vertical rounding
 * ((r0 >> 4) * b0 >> 16) + ((r1 >> 4) * b1 >> 16), (v + 2) >> 2; a source of exactly twice the target size takes
 * cv2's 2x2 INTER_AREA average), then, where UpImageJob.flip is set, the mirror of Mytransforms.hflip
 * (utils/Mytransforms.py:501-505: output column x takes resized column out_w - 1 - x).
 *   jobs:      HOST copy of the table (validated, and sizes the launch); jobs_dev: the same n entries in device memory,
 *              which the kernel reads.  Each `src` must stay valid until the launch has run on `stream`.
 *   out_format UP_BF16 / UP_FP16 / UP_SPLIT: the normalised (x - mean) / std space-to-depth tensor of
 *              up_pack_input_u8_s2d, same layout (y_plane_stride, y_wpitch, y_wpad_left) and same bits;
 *              UP_RESIZE_OUT_U8: uint8 HWC [n, out_h, out_w, 3] (the resized images);
 *              UP_RESIZE_OUT_F32: fp32 NCHW [n, 3, out_h, out_w], (x - mean) / std (Mytransforms.normalize).
 *   out_h, out_w: multiples of 16 (the stem's requirement). */
enum { UP_RESIZE_OUT_U8 = 8, UP_RESIZE_OUT_F32 = 9 };
typedef struct UpImageJob {
  const uint8_t* src;     /* row 0, column 0, channel 0 of the image, device memory */
  int32_t h, w;           /* source size in pixels, both > 0 */
  int32_t pitch;          /* bytes from one row to the next, >= 3 * w */
  int32_t flip;           /* 1: mirror the resized image horizontally */
} UpImageJob;
int up_resize_pack_u8(const UpImageJob* jobs, const UpImageJob* jobs_dev, int n, int out_h, int out_w, int out_format,
                      void* y, int64_t y_plane_stride, int y_wpitch, int y_wpad_left, float mean, float std_,
                      void* stream);
/* Ground-truth heat-maps on the device (utils/mpii_data.py:62-65,165-181; same code in lsp_lspet_data / bbc_data):
 * kpts fp32 [n,k,2] (x, y in input-image pixels) -> heat fp32 NCHW [n, k + background, h, w]: channel j+background
 * = exp(-((x - cx)^2 + (y - cy)^2) / 2 / sigma / sigma) in float64 with cx = int(kx) / stride (truncate_mode 1) or
 * cx = int(kx / stride) (truncate_mode 2: the centre map, mpii_data.py:178), clipped (> 1 -> 1, < 0.0099 -> 0), stored
 * as fp32; background != 0 adds channel 0 = 1 - max over the joints. */
int up_gaussian_labels(const float* kpts, float* heat, int n, int k, int h, int w, float stride, float sigma,
                       int background, int truncate_mode, void* stream);
/* Generic fp32 NCHW [n,c_real,h,w] -> NHWC 16-bit view (channels >= c_real zero-filled up to c). */
int up_nchw_f32_to_nhwc(const float* x, void* y, int n, int c_real, int h, int w, int c, int y_cstride,
                        int y_coff, int dtype, int64_t y_plane_stride, void* stream);
/* NHWC 16-bit view -> fp32 NCHW [n,c_real,h,w]. */
int up_nhwc_to_nchw_f32(const void* x, float* y, int n, int c_real, int h, int w, int x_cstride, int x_coff,
                        int dtype, int64_t x_plane_stride, void* stream);

/* nn.MaxPool2d(kernel_size=3, stride=2, padding=1): resnet.py:64,117  decoder.py:33,47 */
int up_maxpool3x3s2(const void* x, void* y, int n, int h, int w, int c, int x_cstride, int x_coff,
                    int y_cstride, int y_coff, int dtype, int64_t x_plane_stride, int64_t y_plane_stride,
                    void* stream);
/* F.interpolate(mode='bilinear', align_corners=True): wasp.py:83 decoder.py:49 unipose.py:32 */
int up_upsample_bilinear_ac(const void* x, void* y, int n, int h, int w, int ho, int wo, int c, int x_cstride,
                            int x_coff, int y_cstride, int y_coff, int dtype, int64_t x_plane_stride,
                            int64_t y_plane_stride, void* stream);
/* nn.AdaptiveAvgPool2d((1,1)): wasp.py:51.  x NHWC view -> 16-bit [n,1,1,c] view. */
int up_global_avgpool(const void* x, void* y, int n, int h, int w, int c, int x_cstride, int x_coff,
                      int y_cstride, int y_coff, int dtype, int64_t x_plane_stride, int64_t y_plane_stride,
                      void* stream);
/* Sum over h*w (adjoint of up_broadcast_hw): x NHWC view -> 16-bit [n,1,1,c] view. */
int up_global_sumpool(const void* x, void* y, int n, int h, int w, int c, int x_cstride, int x_coff,
                      int y_cstride, int y_coff, int dtype, int64_t x_plane_stride, int64_t y_plane_stride,
                      void* stream);
/* Broadcast a [n,1,1,c] tensor over ho x wo (bilinear from 1x1 with align_corners, wasp.py:83). */
int up_broadcast_hw(const void* x, void* y, int n, int ho, int wo, int c, int x_cstride, int x_coff,
                    int y_cstride, int y_coff, int dtype, int64_t x_plane_stride, int64_t y_plane_stride,
                    void* stream);
/* fp32 NCHW F.interpolate(bilinear, align_corners=True) for the stride != 8 output path
 * (model/unipose.py:31-32). */
int up_upsample_bilinear_ac_nchw_f32(const float* x, float* y, int n, int c, int h, int w, int ho, int wo,
                                     void* stream);

/* ------------------------------------------------------------------------------------------
 * Video variant (model/uniposeLSTM.py)
 * ------------------------------------------------------------------------------------------ */
/* nn.AvgPool2d(kernel_size=9, stride=8, padding=1), count_include_pad: uniposeLSTM.py:91,114.
 * fp32 [n,c,h,w] -> channels [y_c_off, y_c_off+c) of an fp32 [n,y_c_total,ho,wo] tensor
 * (y_c_total <= 0 means y_c_total = c), i.e. the pooled centre map lands directly in the
 * torch.cat((x, centermap)) buffer of uniposeLSTM.py:116. */
int up_avgpool9s8p1_f32(const float* x, float* y, int n, int c, int h, int w, int ho, int wo, int y_c_total,
                        int y_c_off, void* stream);
/* LSTM_0.forward (uniposeLSTM.py:16-24): x fp32 NCHW [b,cin,h,w];  w3 [3][c][cin][3][3] and b3 [3][c]
 * hold conv_{g,i,o}_lstm in that order;  outputs cell, hide fp32 NCHW [b,c,h,w]  (c <= 16). */
int up_convlstm_cell0_fwd(const float* x, const float* w3, const float* b3, float* cell, float* hide, int b,
                          int cin, int c, int h, int w, float* gates, void* stream);
/* LSTM.forward (uniposeLSTM.py:40-64): gates g,i,o,f each conv_x(x)+conv_h(h_prev) with both biases.
 * wx/bx: [4][c][cin][3][3] / [4][c] in gate order g,i,o,f;  wh/bh: [4][c][c][3][3] / [4][c]. */
int up_convlstm_cell_fwd(const float* x, const float* h_prev, const float* c_prev, const float* wx,
                         const float* bx, const float* wh, const float* bh, float* cell, float* hide, int b,
                         int cin, int c, int h, int w, float* gates, void* stream);
/* Both forwards: `gates` (optional, training) receives the ACTIVATED gates fp32 [b, G, c, h, w] in the order g, i, o
 * (G = 3, LSTM_0) / g, i, o, f (G = 4, LSTM) for the backward pass.
 *
 * Backward of either cell (loss.backward() through uniposeLSTM.py:16-24 / :40-64 - the video model trains through all
 * 5 frames with ONE backward, uniposeLSTM.py:116-132): from dcell / dhide (either may be NULL = zero) to
 *   dx [b,cin,h,w], dwx / dbx ([G,c,cin,3,3] / [G,c], the stacked layouts of the forwards), and for LSTM (wh != NULL)
 *   dh_prev, dc_prev [b,c,h,w], dwh / dbh.  (The reference adds the x- and h-conv biases, so dbh == dbx.)
 * dpre: scratch fp32 [b, G, c, h, w].  All reductions are fixed-order (deterministic). */
int up_convlstm_cell_bwd(const float* x, const float* h_prev, const float* c_prev, const float* gates, const float* cell,
                         const float* dcell, const float* dhide, const float* wx, const float* wh, float* dx,
                         float* dh_prev, float* dc_prev, float* dwx, float* dbx, float* dwh, float* dbh, float* dpre,
                         int b, int cin, int c, int h, int w, void* stream);

/* ------------------------------------------------------------------------------------------
 * Evaluation (utils/evaluate.py)
 * ------------------------------------------------------------------------------------------ */
/* get_max_preds (utils/evaluate.py:32-54): per (n, joint) first-occurrence argmax over h*w (numpy
 * semantics incl. NaN).  heat fp32 [n,k,h,w] -> idx int32 [n,k] (flat index), preds fp32 [n,k,2]
 * (x, y; zeroed where max <= 0), maxvals fp32 [n,k]. */
int up_argmax2d(const float* heat, int32_t* idx, float* preds, float* maxvals, int n, int k, int h, int w,
                void* stream);
/* calc_dists (utils/evaluate.py:5-19): dists float64 [k,n] (the reference's dtype); -1 where the
 * target has x<=1 or y<=1. */
int up_calc_dists(const float* preds, const float* target, double* dists, int n, int k, double norm_x,
                  double norm_y, void* stream);
/* dist_acc (utils/evaluate.py:22-29) for every joint at once: acc float64 [k] (-1 if no valid sample). */
int up_dist_acc(const double* dists, double* acc, int n, int k, double threshold, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training glue (unipose.py:113-124)
 * ------------------------------------------------------------------------------------------ */
/* nn.MSELoss() (mean), unipose.py:70,117: loss[0] = mean((pred-target)^2);
 * grad (optional) = gscale * 2*(pred-target)/count.  scratch: one device double. */
int up_mse_fwd_bwd(const float* pred, const float* target, float* loss, float* grad, double* scratch,
                   int64_t count, float gscale, void* stream);
/* ---- backward of the convolutions (what loss.backward() runs for every nn.Conv2d, unipose.py:123) ----
 * dgrad is up_conv2d_fwd itself on the incoming gradient with the filter transposed + flipped
 * (pack w[ci][co][kh'][kw'] = w[co][ci][KH-1-kh'][KW-1-kw'], pad' = dil*(k-1) - pad; for stride 2 first
 * up_zero_insert2x the gradient).  wgrad is its own tcgen05 kernel (both operands MN-major):
 *   dw[co][ci][kh][kw] (+)= sum_{n,ho,wo} dz[n,ho,wo,co] * x[n, ho*stride + kh*dil - pad_h, wo*stride + kw*dil - pad_w, ci]
 * `desc` is the FORWARD descriptor of the layer (x geometry / view, cin, cout, filter, stride, dil, pad, dtype,
 * x_groups); dz must be a dense NHWC [n,ho,wo,cout] tensor whose hi/lo plane stride is desc->y_plane_stride.
 * scratch: fp32 workspace of at least up_conv2d_wgrad_scratch_bytes(desc). */
int64_t up_conv2d_wgrad_scratch_bytes(const UpConvDesc* desc);
int up_conv2d_wgrad(const UpConvDesc* desc, const void* x, const void* dz, float* dw_oihw, int cout_real,
                    int cin_real, float* scratch, int64_t scratch_bytes, int accumulate, void* stream);

/* NHWC 16-bit channel-slice view used by the training kernels below. */
typedef struct UpView {
  void* ptr;            /* base of the buffer (plane 0, channel 0 of pixel 0) */
  int32_t cstride;      /* channels per pixel of the buffer */
  int32_t coff;         /* first channel of the view */
  int64_t plane_stride; /* UP_SPLIT: elements between hi and lo planes */
} UpView;

/* Train-mode nn.BatchNorm2d forward (resnet.py:26-34, wasp.py:18,86, decoder.py:40 in .train()):
 *   up_bn_stats     per-channel sum / sum of squares of the conv output z over npix pixels -> sums[2*c] (double)
 *   up_bn_finalize  batch mean / biased var -> scale, shift, save_mean, save_invstd; running stats updated with
 *                   momentum and the unbiased variance (torch semantics); running_* may be NULL
 *   up_scale_shift_act  y = [relu](z*scale + shift (+ residual)) (* mask)   (mask = pre-scaled dropout mask) */
/* Every BatchNorm reduction works in a caller-owned buffer of up_bn_work_doubles(c) doubles:
 *   [0, 2c) the two per-channel sums | [2c, 4c) coefficient scratch of the backward | partial rows (one per block). */
int64_t up_bn_work_doubles(int c);
int up_bn_stats(const UpView* z, int64_t npix, int c, int dtype, double* work, void* stream);
int up_bn_finalize(const double* sums, int64_t count, const float* gamma, const float* beta, float* running_mean,
                   float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                   float* save_invstd, int c_real, int c, void* stream);
/* up_bn_stats + up_bn_finalize over the same npix pixels in two launches instead of three (the partial rows are
 * reduced and turned into the epilogue constants by one kernel); bit-identical to the two calls. */
int up_bn_stats_finalize(const UpView* z, int64_t npix, int c, int dtype, double* work, const float* gamma,
                         const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                         float* scale, float* shift, float* save_mean, float* save_invstd, int c_real, void* stream);
/* Frozen (eval-mode) BatchNorm inside a training step - the reference's freeze_bn=True / model.freeze_bn()
 * (model/unipose.py:24-25,40-43): scale/shift from the RUNNING statistics, plus save_mean = running_mean and
 * save_invstd = 1/sqrt(running_var + eps) for the backward (up_bn_bwd with flags | 2). */
int up_bn_eval_prepare(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                       float eps, float* scale, float* shift, float* save_mean, float* save_invstd, int c_real, int c,
                       void* stream);
int up_scale_shift_act(const UpView* z, const UpView* y, const UpView* residual, const UpView* mask,
                       const float* scale, const float* shift, int64_t npix, int c, int relu, int dtype,
                       void* stream);
/* BatchNorm (+ReLU) backward (autograd of nn.BatchNorm2d + nn.ReLU, reference call site unipose.py:123), three
 * launches: reduce sum(dy'), sum(dy'*xhat) with dy' = dy*(y>0) into one partial row per block; rows -> work[0 .. 2*c)
 * -> per-channel coefficients (+ dgamma / dbeta, optional, both or neither); then
 *   dz = gamma*invstd*(dy' - sum_dy/M - xhat*sum_dy_xhat/M), optional dres = dy'.
 * `work` holds up_bn_work_doubles(c) doubles (see up_bn_stats); c/8 must be a power of two <= 256.
 * `flags` is a bit mask: 1 = gate by the forward output (y > 0); 2 = frozen BatchNorm, whose statistics are
 * constants: dz = gamma*invstd*dy' (dgamma / dbeta are still the two sums). */
int up_bn_bwd(const UpView* dy, const UpView* y, const UpView* z, const UpView* dz, const UpView* dres,
              const float* save_mean, const float* save_invstd, const float* gamma, double* work, int64_t npix,
              int c_real, int c, int flags, int dtype, float* dgamma, float* dbeta, void* stream);
/* out (+)= a            (mode_op 0)
 * out (+)= a * m        (mode_op 1, dropout mask)
 * out (+)= a * (m > 0)  (mode_op 2, ReLU gate with the forward output m) */
int up_ew_mul(const UpView* a, const UpView* m, const UpView* out, int64_t npix, int c, int mode_op, int accumulate,
              int dtype, void* stream);
/* adjoints of the bandwidth kernels */
/* idx_scratch: optional n*ho*wo*c bytes (8-byte aligned) -> two-pass form (arg-max map, then gather); NULL -> one
 * pass that re-scans every window (slower). */
int up_maxpool3x3s2_bwd(const UpView* x, const UpView* dy, const UpView* dx, int n, int h, int w, int c,
                        int accumulate, int dtype, void* idx_scratch, void* stream);
int up_upsample_bilinear_ac_bwd(const UpView* dy, const UpView* dx, int n, int h, int w, int ho, int wo, int c,
                                int accumulate, int dtype, void* stream);
/* dx[n,h,w,:] (+)= g[n,:] * mult  (adjoint of the global average pool with mult = 1/(h*w)) */
int up_add_broadcast(const UpView* g, const UpView* dx, int n, int hw, int c, float mult, int accumulate, int dtype,
                     void* stream);
/* y[n,2i,2j,:] = x[n,i,j,:], zeros elsewhere */
int up_zero_insert2x(const UpView* x, const UpView* y, int n, int h, int w, int c, int dtype, void* stream);

/* torch.optim.Adam step (no weight decay, no amsgrad) over a flat fp32 buffer. */
int up_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t count, float lr,
                 float beta1, float beta2, float eps, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNIPOSE_B200_H_ */
