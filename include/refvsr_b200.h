/*
 * refvsr_b200 — C ABI of the B200 (sm_100a) kernels behind RefVSR's per-frame forward hot path.
 *
 * The reference (codeslake/RefVSR) is pure Python: it has no FFI of its own.  Its boundary for this
 * path is the nn.Module contract `SRNet.forward(x, ref, is_first_frame, is_log, is_train)`
 * (models/SRNet.py:57-61) and, below it, a sequence of ATen calls.  This header declares one entry
 * point per *fused group* of those ATen calls; each comment cites the reference lines the entry
 * point replaces.  The Python host (refvsr_b200/lib.py) binds them with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless stated otherwise; `stream` is a cudaStream_t passed as
 *     void* (NULL = legacy default stream); every call is asynchronous on that stream;
 *   - activations are NHWC ("pixel rows"): element (y, x, c) at  (y*W + x)*C + c;
 *   - dtype codes: RV_F32 = 0, RV_F16 = 1, RV_BF16 = 2;
 *   - return value: 0 on success, otherwise a negative RV_E_* code; rv_last_error() returns a
 *     human-readable message for the calling thread (the Python binding raises RuntimeError /
 *     ValueError from it, matching the reference's "Python exceptions only" error convention,
 *     mmedit/models/common/flow_warp.py:27-29, models/archs/SPyNet.py:32-34).
 */
#ifndef REFVSR_B200_H_
#define REFVSR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RV_F32 0
#define RV_F16 1
#define RV_BF16 2

#define RV_OK 0
#define RV_E_INVALID (-1) /* bad argument (shape / dtype / alignment)            */
#define RV_E_CUDA (-2)    /* CUDA runtime / driver error, see rv_last_error()   */
#define RV_E_UNSUPPORTED (-3)

/* activation codes used by rv_conv2d epilogues */
#define RV_ACT_NONE 0
#define RV_ACT_RELU 1     /* SPyNet ConvModule, ResidualBlockNoBN (sr_backbone_utils.py:85-97)      */
#define RV_ACT_LRELU01 2  /* LeakyReLU(0.1): RefVSR.py:94,115-116,343                               */
#define RV_ACT_LRELU02 3  /* LeakyReLU(0.2): BasicBlock / ResBlock (RefVSR_/common.py:25-39,96-109) */
#define RV_ACT_CLAMP3 4   /* clamp(-3, 3): affine map of AlignedConv2d (alignment.py:56)            */

#define RV_CONV_IMPL_SIMT 0 /* fp32-accumulate CUDA-core implicit GEMM (any geometry, any dtype)    */
#define RV_CONV_IMPL_TC 1   /* tcgen05/TMEM implicit GEMM fed by TMA (f16/bf16, stride 1)           */

const char* rv_last_error(void);
int rv_version(void);
/* number of kernels launched by this library since load (bench.py's `gpu_launches`) */
uint64_t rv_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * rv_conv2d — fused convolution.  Replaces every nn.Conv2d on the path *together with* the
 * elementwise ops around it:
 *   torch.cat of the two inputs          (RefVSR.py:128,138,139,110,225,266; SPyNet.py:96-102)
 *   bias + ReLU / LeakyReLU              (SPyNet.py:152-191; RefVSR_/common.py:25-39,96-109)
 *   alpha-gating and residual adds       (RefVSR.py:131,143,112; common.py:38,80-81;
 *                                          sr_backbone_utils.py:96-97; SPyNet.py:95)
 *   F.pixel_shuffle                      (mmedit/models/common/upsample.py:48-51)
 *
 *   acc[n]  = bias[n] + sum_{ky,kx,c} W[n][c][ky][kx] * in[(y*stride+ky-pad, x*stride+kx-pad), c]
 *             with in = concat(src0, src1) along channels, zero padding outside the image
 *   v       = act_pre(acc);  if (gate) v *= gate[pix][n];  if (res) v += res[pix][n];
 *   v       = act_post(v);
 *   out     = pixel_shuffle ? out[(2y+a, 2x+b)][n/4] (n = 4c+2a+b) : out[pix][n]
 * ------------------------------------------------------------------------------------------------ */
typedef struct rv_conv_desc {
  const void* src0;   /* [H][W][c0]                                                       */
  const void* src1;   /* [H][W][c1] or NULL                                               */
  int32_t c0, c1;     /* allocated channels of src0/src1 (TC: multiples of 8)             */
  int32_t in_dtype;   /* dtype of src0/src1/gate                                          */
  int32_t H, W;       /* input spatial size                                               */
  const void* wpack;  /* packed weights, layout produced by refvsr_b200/packing.py        */
  const float* bias;  /* [cout] fp32                                                      */
  int32_t cout;       /* real output channels                                             */
  int32_t kh, kw, stride, pad;
  int32_t act_pre, act_post;
  const void* gate;   /* [Ho][Wo][gate_cs] (in_dtype) or NULL                             */
  int32_t gate_cs;
  const void* res;    /* [Ho][Wo][res_cs] (res_dtype) or NULL                             */
  int32_t res_cs, res_dtype;
  void* out;          /* [Ho][Wo][out_cs]   (or [2Ho][2Wo][out_cs] when pixel_shuffle)    */
  int32_t out_cs, out_dtype;
  int32_t pixel_shuffle; /* 0 | 1 (factor 2)                                              */
  int32_t impl;          /* RV_CONV_IMPL_*                                                */
  int32_t nb;            /* TC: output channels per CTA column block (packing.py decides) */
  int32_t k_real;        /* SIMT: rows of wpack = kh*kw*(c0+c1)                           */
  int32_t layout;        /* TC: 0 = [nblk][kx][chunk][ky][NB][64] (one TMA box per kx),    */
                         /*     1 = [nblk][chunk][ky][kx][NB][64] (one box per tile+chunk; */
                         /*         3x3 convs with the all-16-bit epilogue run kx-folded,  */
                         /*         N = 3*NB per MMA),                                     */
                         /*     2 = 32B-swizzled 16-channel quads,                         */
                         /*     3 = weight image of 1, kx-folding disabled (test / A-B)    */
} rv_conv_desc;

int rv_conv2d(const rv_conv_desc* d, void* stream);
/* Upper bound of the persistent grid of the following rv_conv2d (tensor-core) launches made by this process; 0 restores one CTA
 * per SM.  Returns the previous value.  The engine's own scheduling knob, no counterpart in the reference: the forward-branch
 * step of a window (RefVSR.py:248-277) is independent of its backward branch (RefVSR.py:211-238), so network.py enqueues the two on
 * different streams with half the SMs each - two capped launches overlap each other's prologue / first-box latency / last-tile tail,
 * which a single dependent chain of launches exposes once per layer (profiles/r02_trunk_knockout.md). */
int rv_set_conv_cta_cap(int cap);

/* Host-only: the launch plan rv_conv2d's tensor-core path would use on a device with `max_smem_optin` bytes of opt-in shared memory
 * per block and `num_sms` SMs -> out8 = {mode, smem slots, stages per barrier group, stages per tile, MMA-issuing warps, TMEM
 * accumulators, nb, dynamic smem bytes}.  No CUDA call is made (pointers in `d` are only tested for null / alignment).  Lets the
 * ring invariants (every issuing warp owns its slots and accumulators) be checked without a GPU. */
int rv_conv2d_tc_plan(const rv_conv_desc* d, int max_smem_optin, int num_sms, int32_t* out8);

/* ------------------------------------------------------------------------------------------------
 * rv_resblock - fused residual block  out = act_post( x + conv2( act_mid( conv1(x) ) ) ), 3x3 / stride 1 / pad 1,
 * C -> C -> C channels (C <= 64), f16/bf16 NHWC.  One launch instead of two rv_conv2d calls for
 * ResidualBlockNoBN (mmedit/models/common/sr_backbone_utils.py:85-97, act_mid = ReLU) and ResBlock
 * (models/archs/RefVSR_/common.py:33-39, act_mid = LeakyReLU(0.2); act_post = LeakyReLU(0.2) inside
 * AlignedConv2d, alignment.py:19-21).  w1 / w2: packing.pack_tc(..., layout=1) images ([9 taps][nb][64]).
 * ------------------------------------------------------------------------------------------------ */
typedef struct rv_resblock_desc {
  const void* src;   /* [H][W][c] */
  int32_t c;         /* allocated channels of src (multiple of 8, <= 64) */
  int32_t dtype;     /* RV_F16 | RV_BF16 (input, intermediate and output) */
  int32_t H, W;
  const void* w1;
  const float* b1;   /* [cout] */
  const void* w2;
  const float* b2;
  int32_t cout, nb, act_mid, act_post;
  void* out;         /* [H][W][out_cs] */
  int32_t out_cs;
} rv_resblock_desc;

int rv_resblock(const rv_resblock_desc* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * rv_conv_chain - a CHAIN of 3x3 C->C convolutions (+ bias, activation, residual, activation) over a small set of NHWC
 * f16/bf16 buffers of identical geometry, executed by ONE persistent tcgen05 launch with per-tile dependencies between
 * layers and a TMA-store epilogue (refvsr_b200/csrc/conv_chain.cu).  Replaces, launch for launch,
 *   make_layer(ResidualBlockNoBN, num_blocks)  (mmedit/models/common/sr_backbone_utils.py:26-39,85-97; RefVSR.py:346-349)
 *   ResList: N x ResBlock + conv_tail + skip    (RefVSR_/common.py:25-39,64-82; RefVSR.py:48-60,233-234)
 * Layer l computes  buf[dst] = act_post( act_pre( conv3x3(buf[src]) + bias ) + buf[res] )   (res < 0: no residual), zero
 * padding 1.  dst must differ from src.  wpack = the layout-1 tensor-core weight image of rv_conv2d ([9 taps][nb][64]
 * 16-bit, SWIZZLE_128B byte image), bias = nb floats (zero beyond cout).  All buffers: (H, W, C), C % 8 == 0, C <= 48.
 * `flags` is device scratch of >= ceil(H/16) * ceil(W/8) int32 (zeroed by the call, on `stream`).
 * Results are bit-identical to the same layers issued one by one through rv_conv2d.
 * ------------------------------------------------------------------------------------------------ */
#define RV_CHAIN_MAX_LAYERS 64
#define RV_CHAIN_MAX_BUFFERS 6
typedef struct {
  const void* wpack;
  const float* bias;
  int32_t src, res, dst;
  int32_t act_pre, act_post; /* RV_ACT_NONE / RELU / LRELU01 / LRELU02 */
} rv_chain_layer;
typedef struct {
  void* buf[RV_CHAIN_MAX_BUFFERS];
  int32_t nbuf;
  int32_t H, W, C, dtype; /* C = allocated channels (row pitch) of every buffer */
  int32_t nb;             /* rows of the weight image (16 / 32 / 48), >= C */
  const rv_chain_layer* layers; /* HOST array */
  int32_t nlayers;
  int32_t* flags;
  int32_t max_ctas; /* 0: one persistent CTA per SM.  > 0: cap (leave SMs free for kernels of OTHER streams that must stay
                       co-resident, e.g. NCCL point-to-point kernels: the chain's CTAs spin on each other's flags and all
                       of them have to be resident) */
} rv_conv_chain_desc;
int rv_conv_chain(const rv_conv_chain_desc* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * rv_dcn3x3 - modulated deformable 3x3 convolution (DCNv2), the ModulatedDCNPack of the RefVSR_IR refill extractor
 * (models/archs/edvr_net.py:15-58: conv_offset -> chunk / cat / sigmoid -> mmcv modulated_deform_conv2d with stride 1,
 * pad 1, dilation 1, groups 1, 8 deform groups), minus conv_offset itself, which is an ordinary rv_conv2d:
 *   om (H, W, om_cs) fp32, om_cs >= 216: conv_offset's RAW output.  For deform group g (input channels 8g..8g+7) and
 *      tap k = 3*ky + kx:  dy = om[18g + 2k], dx = om[18g + 2k + 1], m = sigmoid(om[144 + 9g + k]);
 *   x  (H, W, 64) `dtype`, 16-byte aligned;
 *   s  = bilinear(x[.., c], y - 1 + ky + dy, x - 1 + kx + dx): 0 when the sample lies at or beyond one pixel outside the
 *        map (h <= -1, h >= H, w <= -1, w >= W), corners outside the map contribute 0 (mmcv dmcn_im2col_bilinear);
 *   out[(y, x)][n] = act(bias[n] + sum_{k, c} W[n][c][ky][kx] * m * s),  n < cout <= 64, out (H, W, out_cs) `dtype`.
 * impl RV_CONV_IMPL_TC: tcgen05 implicit GEMM, f16 / bf16, wpack = packing.pack_tc(W, [(64, 64)], dtype, nb, layout=1);
 * impl RV_CONV_IMPL_SIMT: CUDA cores, any dtype, wpack = packing.pack_simt(W, [(64, 64)]) fp32 (nb ignored).
 * ------------------------------------------------------------------------------------------------ */
int rv_dcn3x3(const void* x, const float* om, int om_cs, int H, int W, int dtype, const void* wpack, const float* bias,
              int cout, int nb, int act, int impl, void* out, int out_cs, void* stream);

/* space-to-depth by 2: out[(Y,X)][(ry*2+rx)*C + c] = src[(2Y+ry, 2X+rx)][c].  Turns the two stride-2
 * convolutions of the path (ref_encoder2.0.0, RefVSR.py:45; aa2.align.p_conv.0, alignment.py:21) into
 * stride-1 3x3 convolutions over 4C channels (weights re-indexed by packing.s2d_weights), so they run on
 * the tcgen05 kernel.  H, W even; C*elemsize a multiple of 16. */
int rv_space_to_depth2(const void* src, int H, int W, int C, int dtype, void* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Image / map preparation
 * ------------------------------------------------------------------------------------------------ */
/* NCHW fp32 image (3,H,W) -> NHWC `out` with `out_c` channels (>=3, rest zero).
 * mat12 != NULL: out_c = mat[c][0..2]·rgb + mat[c][3]  (MeanShift 1x1 conv, common.py:84-94,
 *                attention.py:62-63).  pool2: 2x2 mean after the affine map (attention.py:51,75). */
int rv_prep_image(const float* src_nchw, int H, int W, const float* mat12_host, int pool2,
                  void* out, int out_c, int out_dtype, void* stream);

/* SPyNet input resize: bilinear (align_corners=False) to (Ho,Wo) then (x-mean)/std
 * (SPyNet.py:117-126, 62-63). src NCHW fp32 (3,H,W) -> out HWC fp32 (Ho,Wo,3) */
int rv_spynet_resize_norm(const float* src_nchw, int H, int W, float* out, int Ho, int Wo,
                          void* stream);
/* 2x2 mean pool, HWC fp32 with C channels (SPyNet.py:66-78) */
int rv_avgpool2(const float* src, int H, int W, int C, float* out, void* stream);
/* 2x2 / stride 2 max pool of an NHWC map (torchvision vgg19.features[4] inside FeatureMatching with vgg_range = 7,
 * i.e. the flag_HD_in "8K" configs, attention.py:31-40).  src (H,W,C) -> out (H/2,W/2,C), same dtype. */
int rv_maxpool2(const void* src, int H, int W, int C, int dtype, void* out, void* stream);
/* Resize of `n` planar fp32 maps (n,H,W) -> (n,Ho,Wo) with the source coordinate scale `inv_scale` = 1 / scale_factor:
 *   mode 0: bicubic, A = -0.75, align_corners=False, clamped taps (F.interpolate(mode='bicubic')): the x4 upsample
 *           of the relevance map (attention.py:96-98) and lr_down = bicubic x0.5 of the LR frame (RefVSR.py:125);
 *   mode 1: nearest, src = floor(dst * inv_scale) (F.interpolate(scale_factor=0.5, mode='nearest'), attention.py:65-67).
 * clamp01: clamp the result to [0,1] (both bicubic call sites do). */
int rv_resize_planes(const float* src, int n, int H, int W, float inv_scale, int Ho, int Wo, int mode, int clamp01,
                     float* out, void* stream);
/* One pyramid level's network input (SPyNet.py:84-102):
 *   flow_up = level0 ? 0 : 2 * bilinear_x2_align_corners(flow_prev)      -> flow_up (H,W,2) fp32
 *   out8    = [ref(3), flow_warp(supp, flow_up, border, align_corners=True)(3), flow_up(2)]
 * flow_prev is (H/2, W/2, 2) fp32 or NULL. */
int rv_spynet_level_input(const float* ref, const float* supp, const float* flow_prev, int H, int W,
                          void* out8, int out_dtype, float* flow_up, void* stream);
/* final flow resize back to (h,w) + per-axis rescale (SPyNet.py:129-137) */
int rv_flow_resize(const float* flow, int H, int W, float* out, int h, int w, void* stream);

/* ------------------------------------------------------------------------------------------------
 * rv_warp — models/utils.py:34-43 (`warp`: grid_sample bilinear / zeros / align_corners=False with
 * the reference's linspace grid) fused with the x2 flow upsample of RefVSR.py:220,254,259.
 *   src (Hi,Wi,C) `dtype`; flow (hf,wf,2) fp32 in LR pixels;
 *   flow_up2 == 0: output grid = flow grid (hf,wf);
 *   flow_up2 == 1: output grid = (2hf,2wf), flow' = 2*bilinear_align_corners_true(flow).
 * ------------------------------------------------------------------------------------------------ */
int rv_warp(const void* src, int Hi, int Wi, int C, int dtype, const float* flow, int hf, int wf,
            int flow_up2, void* out, void* stream);
/* The three warps of one propagation step fused into ONE launch (RefVSR.py:216-220 backward branch, :256-260 steady forward
 * step): out_feat = warp(feat, flow), out_conf = warp(conf, flow), out_featUP = warp(featUP, interpolate(flow, x2, bilinear,
 * align_corners=True) * 2).  feat (h,w,C), featUP (2h,2w,C) f16/bf16, conf (h,w) fp32, flow (h,w,2) fp32.  The flow is read
 * once; same arithmetic as three rv_warp calls (feat / conf bit-identical, featUP to the last bit of the storage type).  (Not for the first-window quirk RefVSR.py:252-254, whose 2x warp
 * reads the OUTPUT of the LR warp.) */
int rv_warp3(const void* feat, const void* featUP, const float* conf, const float* flow, int h, int w, int C, int dtype,
             void* out_feat, void* out_featUP, float* out_conf, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Matching (models/archs/RefVSR_/attention.py:69-91)
 * ------------------------------------------------------------------------------------------------ */
/* 3x3 reflection-padded patches of a 16-channel feature map, L2-normalised (eps 1e-12), written
 * K-major as fp16 rows for the GEMM:   mode 0: [hi]                 (kpad >= 144)
 *                                      mode 1: [hi | lo | hi]       (A side, kpad >= 432)
 *                                      mode 2: [hi | hi | lo]       (B side)
 * values are pre-scaled by 2^6 so the fp16 `lo` part stays normal; rv_match_argmax undoes it.
 * (RefVSR_/utils.py:10-57 same_padding + Unfold; attention.py:83-85 F.normalize) */
int rv_patch_pack(const void* feat, int H, int W, int C, int dtype, int mode, void* out_f16,
                  int kpad, void* stream);
/* conf[l] = max_r <A[l], B[r]>,  idx[l] = argmax_r (lowest r wins ties)  (attention.py:91).
 * A (P,kpad) fp16, B (R,kpad) fp16, outputs conf (P) fp32, idx (P) int32.
 * impl: 0 = CUDA-core fp32 reference kernel, 1 = tcgen05 (TMA-fed, TMEM accumulators). */
int rv_match_argmax(const void* A, int P, const void* B, int R, int kpad, float out_scale,
                    float* conf, int32_t* idx, int impl, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Reference alignment (attention.py:131-159, alignment.py:39-100)
 * ------------------------------------------------------------------------------------------------ */
/* AlignedAttention gather: out[(ks*i+a, ks*j+b)] = value[(ks*ry+a, ks*rx+b)],
 * (ry,rx) = divmod(idx[i*wq+j], Wv/ks).  value (Hv,Wv,C); out (ks*hq, ks*wq, C). ks=1 -> aa1. */
int rv_gather_blocks(const void* value, int Hv, int Wv, int C, int dtype, const int32_t* idx, int hq,
                     int wq, int ks, void* out, void* stream);
/* AlignedConv2d sampling (alignment.py:45-100,102-178): x (ks*h, ks*w, C), affine (h,w,3) fp32
 * already = clamp(p_conv(..)+1, -3, 3); reflection pad 1; output (ks*h, ks*w, C). */
int rv_aligned_sample(const void* x, int h, int w, int ks, int C, int dtype, const float* affine,
                      void* out, void* stream);
/* bicubic x2 of an image, A=-0.75, align_corners=False, NO clamp (alignment.py:41):
 * src NCHW fp32 (3,H,W) -> out NHWC (2H,2W,out_c) */
int rv_bicubic_up2_image(const float* src_nchw, int H, int W, void* out, int out_c, int out_dtype,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Confidence maps (RefVSR.py:105-106,110,129,140-142,147)
 * ------------------------------------------------------------------------------------------------ */
/* out[(y,x)] = [A(y,x), B(y,x), 0...] (out_c channels); up2: A,B are first bicubic-x2 upsampled and
 * clamped to [0,1].  a,b planar fp32 (h,w). */
int rv_conf_pair(const float* a, const float* b, int h, int w, int up2, void* out, int out_c,
                 int out_dtype, void* stream);
int rv_conf_max(const float* a, const float* b, float* out, int n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Guard of the sliding-window reuse (no reference counterpart: the reference silently ASSUMES that consecutive calls slide
 * the window by one frame when it reuses forward_*_prev, RefVSR.py:256-260; this implementation also reuses per-frame
 * products, so it checks).  Compares n <= 16 (a[i], b[i], nbytes[i]) DEVICE buffer pairs; the pointer / size arrays
 * themselves are HOST arrays.  *flag (device int32, zeroed by the caller) becomes non-zero iff any pair differs.
 * ------------------------------------------------------------------------------------------------ */
int rv_frames_differ(const void* const* a, const void* const* b, const uint64_t* nbytes, int n, int32_t* flag,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * Reconstruction tail (RefVSR.py:118,288,297): out = conv_last_out + clamp(bicubic_x4(lr),0,1),
 * optionally clamped to [0,1]; written NCHW fp32 (3, 4h, 4w).  x (4h,4w,xc) is conv_last's output.
 * ------------------------------------------------------------------------------------------------ */
int rv_reconstruct(const void* x, int xc, int x_dtype, const float* lr_nchw, int h, int w, int scale,
                   int clamp01, float* out_nchw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* REFVSR_B200_H_ */
