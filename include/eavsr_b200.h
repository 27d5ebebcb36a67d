/*
 * eavsr_b200 -- C ABI of the B200-native (sm_100a) inter-frame alignment kernels for EAVSR, and of the
 * reconstruction tail that turns the network's HR features into 8-bit RGB frames.
 *
 * The reference (HITRainer/EAVSR) has no C ABI: its hot path is reached through Python
 * symbols.  Each entry point below replaces the native code that sits under one of those
 * symbols; the Python mirror of the reference interface lives in eavsr_b200/ops.py and
 * binds these functions with ctypes (see INTEGRATION.md for the reference-side stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - feature tensors are described by 4 element strides in (n, c, h, w) order, so NCHW and
 *     channels_last (NHWC) buffers are both accepted without copies;  the vectorised /
 *     tensor-core fast paths need stride_c == 1 (NHWC), 16-byte aligned rows;
 *   - flow / offset / mask are always fp32 (sampling coordinates are never rounded to bf16);
 *   - `stream` is a cudaStream_t (NULL = legacy default stream);  calls are asynchronous,
 *     re-entrant, keep no global mutable state besides an atomic launch counter, and are
 *     CUDA-graph capturable;
 *   - return value: EAVSR_OK or an error code; eavsr_last_error() gives the message of
 *     the calling thread's last failure;
 *   - inputs are borrowed and never written; outputs/workspaces are caller-allocated.
 */
#ifndef EAVSR_B200_H_
#define EAVSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EAVSR_OK 0
#define EAVSR_ERR_INVALID 1     /* bad argument (shape, alignment, enum)            */
#define EAVSR_ERR_CUDA 2        /* CUDA runtime error (message has the cuda string) */
#define EAVSR_ERR_UNSUPPORTED 3 /* valid request that this build does not implement */

#define EAVSR_F32 0
#define EAVSR_BF16 1

#define EAVSR_FLOW_N2HW 0 /* models/networks.py:699  flow_warp(x, flow[n,2,h,w])      */
#define EAVSR_FLOW_NHW2 1 /* models/eavsrp_model.py:587 flow_warp(x, flow[n,h,w,2])   */

#define EAVSR_PAD_ZEROS 0
#define EAVSR_PAD_BORDER 1

#define EAVSR_DCN_FORCE_GENERIC 1u /* flags bit: skip the tcgen05 path (validation only) */
#define EAVSR_DCN_FORCE_V1 2u      /* flags bit: first-generation tcgen05 kernel (A/B timing only) */
#define EAVSR_DCN_FORCE_WS 4u      /* flags bit: second-generation (warp-specialised, L1 gather) kernel */
#define EAVSR_DCN_BLEND_FP32 8u    /* flags bit: window kernel with fp32 blend instead of bf16x2 HFMA2 */
#define EAVSR_DCN_FORCE_WIN1 128u  /* flags bit: third-generation window kernel (cp.async-staged offsets) instead of
                                      the fourth (TMA-staged offsets; deform_groups = 8, w % 4 == 0) -- A/B timing */
#define EAVSR_DCN_FORCE_WIN2 256u  /* flags bit: fourth-generation window kernel (A tile in shared memory) instead of
                                      the fifth (A tile in tensor memory, dcn_fwd_win3.cuh); A/B timing and tests */
#define EAVSR_DCN_BWD_GENERIC_DATA 32u   /* flags bit (backward): d(x), d(offset), d(mask) on the generic kernel */
#define EAVSR_DCN_BWD_GENERIC_WEIGHT 64u /* flags bit (backward): d(weight) on the generic kernel */
#define EAVSR_DCN_WS_PACKED 16u    /* flags bit: `workspace` still holds the packed image of this same `weight`
                                      written by an earlier eavsr_dcn_forward call (constant inference
                                      weights): skip the re-pack launch */

/* ---- library ------------------------------------------------------------------------ */
int eavsr_version(void);
const char* eavsr_last_error(void);
/* number of CUDA kernels launched by this library in this process (all threads). */
uint64_t eavsr_launch_count(void);

/* ---- flow_warp -------------------------------------------------------------------------
 * Replaces F.grid_sample(bilinear, align_corners=True) under
 *   models/networks.py:699-739 (flow_layout N2HW) and
 *   models/eavsrp_model.py:587-626 / models/eavsrpx2_model.py:588-627 (flow_layout NHW2),
 * including the meshgrid/normalise prologue those functions run on the host per call.
 * out[n,c,y,x] = bilinear(x[n,c], y + flow_y, x + flow_x); flow channel 0 is x.
 * padding: zeros (each out-of-image corner contributes 0) or border (clamp coordinate). */
int eavsr_flow_warp_forward(const void* x, const int64_t x_strides[4], const float* flow, int flow_layout,
                            void* out, const int64_t out_strides[4], int n, int c, int h, int w, int dtype,
                            int padding_mode, void* stream);

/* Two feature maps warped with the same flow in one launch (SURVEY.md section 8 row f2: `nbr` and
 * `feat_prop` in MultiAdSTN.forward, models/networks.py:621-623).  Dense NHWC bf16, c = 64 only; anything
 * else returns EAVSR_ERR_UNSUPPORTED and the caller issues two eavsr_flow_warp_forward calls. */
int eavsr_flow_warp2_forward(const void* x1, const int64_t x1_strides[4], const void* x2,
                             const int64_t x2_strides[4], const float* flow, int flow_layout, void* out1,
                             const int64_t out1_strides[4], void* out2, const int64_t out2_strides[4], int n, int c,
                             int h, int w, int dtype, int padding_mode, void* stream);

/* Warp with a PYRAMID flow (SURVEY.md section 8 row f2): flow(y, x) = sum_i scale_i * resize(flow_i)(y, x), resize =
 * bilinear with align_corners=True to (h, w) -- the F.interpolate(offset, s) * s / ... + ... chains of
 * MultiAdSTN.forward (models/networks.py:600-615, :619) evaluated inside the warp's coordinate phase instead of
 * being materialised by F.interpolate + elementwise launches.  terms[i].flow: (n, 2, terms[i].h, terms[i].w) fp32
 * contiguous; terms[i].scaled_out (optional, (n,2,h,w) fp32) receives scale_i * resize(flow_i); flow_out (optional,
 * (n,2,h,w) fp32) the sum.  x2 / out2 (optional): a second map warped with the same flow (models/networks.py:
 * 621-623).  Dense NHWC 64-channel bf16 / fp32 maps, zeros padding (x2: bf16); anything else returns
 * EAVSR_ERR_UNSUPPORTED and the caller composes the reference's operations. */
typedef struct EavsrFlowTerm {
  const float* flow;
  float* scaled_out;
  int h, w;
  float scale;
} EavsrFlowTerm;
int eavsr_flow_warp_pyramid_forward(const void* x, const int64_t x_strides[4], const void* x2,
                                    const int64_t x2_strides[4], const EavsrFlowTerm* terms, int nterms, void* out,
                                    const int64_t out_strides[4], void* out2, const int64_t out2_strides[4],
                                    float* flow_out, int n, int c, int h, int w, int dtype, int padding_mode,
                                    void* stream);

/* SPyNet level input (SURVEY.md section 8 row f4; SPyNet.compute_flow, models/eavsrp_model.py:468-486):
 * out (n,8,h,w) = cat[ref, flow_warp(supp, up, 'border'), up] with up = 2 * resize_x2(flow_prev) (bilinear,
 * align_corners=True; flow_prev (n,2,prev_h,prev_w) or NULL = zero flow at the coarsest level).  NCHW fp32. */
int eavsr_spynet_level_input_forward(const float* ref, const float* supp, const float* flow_prev, float* out, int n,
                                     int h, int w, int prev_h, int prev_w, void* stream);

/* Gradients of eavsr_flow_warp_forward.  gx32 is an fp32 accumulation buffer with strides gx_strides that
 * the call zero-fills and scatter-adds into (for dtype F32 it is the final gradient);
 * gflow (fp32, same layout as flow) may be NULL when the flow needs no gradient.
 * gx32 may be NULL when x needs no gradient. */
int eavsr_flow_warp_backward(const void* gout, const int64_t gout_strides[4], const void* x,
                             const int64_t x_strides[4], const float* flow, int flow_layout, float* gx32,
                             const int64_t gx_strides[4], float* gflow, int n, int c, int h, int w, int dtype,
                             int padding_mode, void* stream);

/* ---- backwarp ---------------------------------------------------------------------------
 * Replaces BaseModel.backwarp + the masking of get_backwarp (models/base_model.py:321-354) and
 * PWCNET.Decoder.backwarp (models/pwc_net.py:184-207): F.grid_sample(cat[x, ones], cached_grid +
 * flow / ((size-1)/2), bilinear, zeros, align_corners=False), mask = warped_ones > 0.999, out = warp * mask.
 * The sample point is (y + flow_y * H/(H-1), x + flow_x * W/(W-1)).  flow: (n,2,h,w) fp32 contiguous,
 * channel 0 = x.  out: (n,c,h,w) `dtype` by strides; mask: (n,1,h,w) contiguous `dtype` (values 0 / 1) or
 * NULL.  h, w must be > 1 (the reference divides by (size-1)/2). */
int eavsr_backwarp_forward(const void* x, const int64_t x_strides[4], const float* flow, void* out,
                           const int64_t out_strides[4], void* mask, int n, int c, int h, int w, int dtype,
                           void* stream);
/* Gradients of out wrt x (fp32 accumulation buffer gx32, zero-filled by the call) and wrt flow (fp32
 * (n,2,h,w)); either may be NULL.  The mask is piecewise constant and carries no gradient. */
int eavsr_backwarp_backward(const void* gout, const int64_t gout_strides[4], const void* x,
                            const int64_t x_strides[4], const float* flow, float* gx32,
                            const int64_t gx_strides[4], float* gflow, int n, int c, int h, int w, int dtype,
                            void* stream);

/* ---- modulated deformable convolution (DCNv2) --------------------------------------------
 * Replaces mmcv.ops.modulated_deform_conv2d as called at models/networks.py:627-630
 * (ext_module.modulated_deform_conv_forward / _backward of mmcv-full 1.x).
 *   offset: (n, dg*2*kh*kw, ho, wo) fp32 contiguous, channel (g*K+k)*2 = dy, +1 = dx
 *   mask:   (n, dg*kh*kw,   ho, wo) fp32 contiguous
 *   weight: (cout, cin/groups, kh, kw) contiguous, dtype = `dtype`;  bias: (cout) or NULL
 *   x / out: `dtype`, described by strides.
 * Fast path (tcgen05 implicit GEMM): cin=cout=64, 3x3, stride 1, pad 1, dilation 1, groups 1,
 * dg in {1,2,4,8,16}, NHWC x/out.  It needs `workspace` of eavsr_dcn_forward_workspace() bytes
 * (packed weights).  Everything else runs the generic kernel (no workspace). */
size_t eavsr_dcn_forward_workspace(int cin, int cout, int kh, int kw, int groups, int deform_groups,
                                   int dtype);
/* 1 if the arguments select the tcgen05 path, 0 for the generic kernel. */
int eavsr_dcn_forward_uses_tensor_cores(const int64_t x_strides[4], const int64_t out_strides[4], int cin,
                                        int cout, int kh, int kw, int sh, int sw, int ph, int pw, int dh,
                                        int dw, int groups, int deform_groups, unsigned flags);
int eavsr_dcn_forward(const void* x, const int64_t x_strides[4], const float* offset, const float* mask,
                      const void* weight, const void* bias, void* out, const int64_t out_strides[4], int n,
                      int cin, int h, int w, int cout, int kh, int kw, int sh, int sw, int ph, int pw, int dh,
                      int dw, int groups, int deform_groups, int dtype, void* workspace,
                      size_t workspace_bytes, unsigned flags, void* stream);

/* DCNv2 with the offset generation fused in (SURVEY.md section 8 row f1).  Replaces the tail of
 * AdaptBlockOffset.forward -- the T*R - R + t expansion, the sigmoid and the 144 + 72 channel fp32
 * offset / mask tensors, models/networks.py:302-315 -- together with the modulated_deform_conv2d call at
 * :627-630.  affine: (n, h, w, 15*dg) dense NHWC bf16, per pixel [4*dg transform | 2*dg translation |
 * 9*dg mask logits] = the raw output of the transform / translation / mask convolutions;
 * affine_bias: their 15*dg biases (bf16) or NULL.  For group g and tap k = 3i + j:
 *   offset_y = T[g][0]*(i-1) + T[g][1]*(j-1) - (i-1) + t[g][0]
 *   offset_x = T[g][2]*(i-1) + T[g][3]*(j-1) - (j-1) + t[g][1],   mask = sigmoid(logit[g*9+k]).
 * Only the tensor-core configuration is implemented (64 -> 64, 3x3, stride/pad/dilation 1, groups 1,
 * dg = 8 -- the model's configuration --, bf16 NHWC x / out): anything else returns EAVSR_ERR_UNSUPPORTED and the caller
 * composes eavsr_affine_offsets_forward + eavsr_dcn_forward.  workspace as for eavsr_dcn_forward.
 * `out` may be a 64-channel slice of a wider NHWC buffer (out_strides[3] = its channel count, a multiple
 * of 8): the aligned feature is then written straight into the concatenated input of the next convolution
 * (torch.cat([cond1, cur, cond2]) in EAVSRP.propagate, models/eavsrp_model.py:271-324). */
int eavsr_dcn_affine_forward(const void* x, const int64_t x_strides[4], const void* affine, const void* affine_bias,
                             const void* weight, const void* bias, void* out, const int64_t out_strides[4], int n,
                             int h, int w, int deform_groups, int dtype, void* workspace, size_t workspace_bytes,
                             unsigned flags, void* stream);

/* Gradients wrt x, offset, mask, weight, bias (any output pointer may be NULL = not needed).
 * gx32: fp32 accumulation buffer (zero-filled by the call) with strides gx_strides;
 * goffset/gmask: fp32, layouts of offset/mask;  gweight32: fp32 (cout,cin/groups,kh,kw),
 * gbias32: fp32 (cout) -- both zero-filled by the call.
 * bf16 NHWC 64->64 3x3 (stride/pad/dilation 1, deform_groups 1/2/4/8/16) runs on the tcgen05 kernels
 * (csrc/dcn_bwd_tc.cu) when `workspace` holds eavsr_dcn_backward_workspace() bytes (16-byte aligned);
 * with workspace == NULL, or any other configuration, the generic kernels run.  This replaces the
 * autograd of mmcv's ModulatedDeformConv2dFunction.backward under models/networks.py:627-630. */
size_t eavsr_dcn_backward_workspace(int cin, int cout, int kh, int kw, int groups, int deform_groups, int dtype);
int eavsr_dcn_backward(const void* gout, const int64_t gout_strides[4], const void* x,
                       const int64_t x_strides[4], const float* offset, const float* mask, const void* weight,
                       float* gx32, const int64_t gx_strides[4], float* goffset, float* gmask,
                       float* gweight32, float* gbias32, int n, int cin, int h, int w, int cout, int kh, int kw,
                       int sh, int sw, int ph, int pw, int dh, int dw, int groups, int deform_groups,
                       int dtype, void* workspace, size_t workspace_bytes, unsigned flags, void* stream);

/* ---- PWC-Net cost volume -----------------------------------------------------------------
 * Replaces kernel_Correlation_rearrange + kernel_Correlation_updateOutput
 * (pwc/correlation/correlation.py:8-103, launched :293-322) and the two backward kernels
 * (:105-233, launched :343-373).  first/second: (n,c,h,w) NCHW contiguous (the reference
 * asserts contiguity, :286-287); out: (n,81,h,w) NCHW contiguous, same dtype.
 * out[n,(dy+4)*9+(dx+4),y,x] = 1/c * sum_ch first[n,ch,y,x]*second[n,ch,y+dy,x+dx]. */
int eavsr_correlation_forward(const void* first, const void* second, void* out, int n, int c, int h, int w,
                              int dtype, void* stream);
/* Same with flags.  EAVSR_CORR_TF32 (opt-in): fp32 maps larger than 16x16 with w % 4 == 0 run as a banded GEMM on
 * tcgen05 (kind::tf32, operands MN-major straight from NCHW through TMA).  tf32 truncates the inputs to 10 mantissa
 * bits: max-abs error 0.8e-3 .. 2.5e-3 on unit-variance features (the fp32 bound of BASELINE.json is 1e-3), which is
 * why the exact fp32 SIMT kernels stay the default. */
#define EAVSR_CORR_TF32 2u
int eavsr_correlation_forward_ex(const void* first, const void* second, void* out, int n, int c, int h, int w,
                                 int dtype, unsigned flags, void* stream);
/* gfirst/gsecond: (n,c,h,w) same dtype, either may be NULL. */
int eavsr_correlation_backward(const void* first, const void* second, const void* gout, void* gfirst,
                               void* gsecond, int n, int c, int h, int w, int dtype, void* stream);

/* ---- fused producers / consumers around the hot path (inference) -----------------------------
 * The offset/mask generator that feeds the DCN (SURVEY.md section 8 row a3) and the channel
 * attention of the residual backbone (row f3), as single passes instead of PyTorch glue.
 *
 * adapt_mix: concat2(concat(cat[a, b])) of AdaptBlockOffset / AdaptBlock2_3x3
 *   (models/networks.py:289-290,299 and :327-328,334): depthwise 3x3 on the 128 concatenated
 *   channels + LeakyReLU, then grouped 3x3 (groups=64, 2 -> 1) + LeakyReLU.
 *   a, b, out: (n,64,h,w) dense NHWC;  w1 (128,1,3,3), b1 (128), w2 (64,2,3,3), b2 (64); all `dtype`. */
int eavsr_adapt_mix_forward(const void* a, const void* b, const void* w1, const void* b1, const void* w2,
                            const void* b2, void* out, int n, int c, int h, int w, float negative_slope,
                            int dtype, void* stream);
/* affine_offsets: offset = T*R - R + t per deformable group and mask = sigmoid(logits)
 *   (models/networks.py:302-313).  transform (n,4D,h,w), translation (n,2D,h,w), mask_logits (n,9D,h,w)
 *   are `dtype` with arbitrary strides; offset (n,18D,h,w) / mask (n,9D,h,w) are fp32 NCHW contiguous,
 *   the layout eavsr_dcn_forward consumes.  mask (and mask_logits) may be NULL.  The optional *_bias
 *   vectors are added to the inputs first, so the three producing convolutions can run bias-free. */
int eavsr_affine_offsets_forward(const void* transform, const int64_t transform_strides[4],
                                 const void* translation, const int64_t translation_strides[4],
                                 const void* mask_logits, const int64_t mask_strides[4],
                                 const void* transform_bias /* (4D) or NULL */,
                                 const void* translation_bias /* (2D) or NULL */,
                                 const void* mask_bias /* (9D) or NULL */, float* offset, float* mask, int n,
                                 int deform_groups, int h, int w, int dtype, void* stream);
/* ca_residual: out = res * sigmoid(W2 relu(W1 mean_hw(res) + b1) + b2) + skip  (CALayer + residual of
 *   RCABlock, models/networks.py:449-465).  res, skip, out: (n,64,h,w) dense NHWC; w1 (4,64), w2 (64,4);
 *   sums_workspace: n*64 floats. */
int eavsr_ca_residual_forward(const void* res, const void* skip, const void* w1, const void* b1, const void* w2,
                              const void* b2, const void* res_bias /* bias of the conv that produced res, or NULL */,
                              void* out, float* sums_workspace, int n, int c, int h, int w, int reduction, int dtype,
                              void* stream);
/* bias_act: x = LeakyReLU_slope(x + bias[c]) in place on a dense NHWC tensor of `pixels` x c elements
 *   (slope 1 = plain bias add, 0 = ReLU): the bias/activation epilogue of the cuDNN convolutions around
 *   the hot path in one vectorised pass.  c must be a multiple of 16 bytes / sizeof(dtype). */
int eavsr_bias_act_forward(void* x, const void* bias, int c, long long pixels, float negative_slope, int dtype,
                           void* stream);

/* grouped_conv3x3: the grouped 3x3 convolutions of AdaptBlockOffset / AdaptBlock2_3x3 (`concat`: depthwise over
 *   2*ch channels, `concat2`: 2 inputs per output channel; models/networks.py:289-290, 327-328), stride 1, pad 1,
 *   differentiable: forward, d(input) and d(weight) + d(bias) -- the training step's replacement for cuDNN's grouped
 *   kernels.  x (n,cin,h,w), out / gout (n,cout,h,w) dense NHWC in `dtype`; weight (cout, cin/cout, 3, 3) and bias
 *   (cout) in `dtype`; groups = cout, cin/cout in {1, 2}, channel counts multiples of 8.  backward: gx may be NULL;
 *   gweight (cout, cin/cout, 3, 3) and gbias (cout) are fp32, must be ZERO on entry and go together (or both NULL). */
int eavsr_grouped_conv3x3_forward(const void* x, const void* weight, const void* bias, void* out, int n, int cin,
                                  int cout, int h, int w, int dtype, void* stream);
int eavsr_grouped_conv3x3_backward(const void* gout, const void* x, const void* weight, void* gx, float* gweight,
                                   float* gbias, int n, int cin, int cout, int h, int w, int dtype, void* stream);

/* channel_sum: sums(n, 64) [fp32, zero-filled by the call] = sum over the hw pixels of x (n, 64, h, w) dense NHWC:
 *   the bias gradient of the 64-output convolutions (`grad.sum((0, 2, 3))` = its sum over n) and the global average
 *   pooling of CALayer (models/networks.py:431-447) in the training step. */
int eavsr_channel_sum_forward(const void* x, float* sums, int n, int c, long long hw, int dtype, void* stream);

/* channel_dot: sums(n, 64) [fp32, zero-filled by the call] = sum over the hw pixels of a * b: the gradient of the
 *   channel-attention scale in RCABlock's `res * scale + x` (models/networks.py:449-465) in the training step. */
int eavsr_channel_dot_forward(const void* a, const void* b, float* sums, int n, int c, long long hw, int dtype,
                              void* stream);

/* nhwc_cat: torch.cat(dim=1) of `nsrc` (<= 8) dense NHWC tensors of `pixels` = n*h*w pixels into the channel slice
 *   [out_channel_offset, +sum(src_channels)) of a dense NHWC buffer with out_channels channels -- the inputs of the
 *   fusion / backbone / reconstruction convolutions, models/eavsrp_model.py:271-324 (torch.cat([cond1, cur, cond2])),
 *   :315 (torch.cat([cur, *others, prop])), :350-364.  All channel counts and the offset multiples of 16 bytes. */
int eavsr_nhwc_cat_forward(const void* const* srcs, const int* src_channels, int nsrc, void* out, int out_channels,
                           int out_channel_offset, long long pixels, int dtype, void* stream);

/* bias_act_shuffle: PixelShuffle(2) with the producing convolution's bias and LeakyReLU folded in
 *   (the upsample1/upsample2 stages of EAVSRP.upsample, models/eavsrp_model.py:350-364):
 *   out[n, c, 2h+i, 2w+j] = LeakyReLU_slope(x[n, 4c+2i+j, h, w] + bias[4c+2i+j]);
 *   x: (n, 4*c_out, h, w), out: (n, c_out, 2h, 2w), both dense NHWC; bias may be NULL. */
int eavsr_bias_act_shuffle_forward(const void* x, const void* bias, void* out, int n, int c_out, int h, int w,
                                   float negative_slope, int dtype, void* stream);
/* Second half of ca_residual with channel sums produced elsewhere (eavsr_conv3x3_forward). */
int eavsr_ca_scale_forward(const void* res, const void* skip, const float* sums, const void* w1, const void* b1,
                           const void* w2, const void* b2, const void* res_bias, void* out, int n, int c, int h,
                           int w, int reduction, int dtype, void* stream);

/* ---- 3x3 convolution 64 -> 64 on tcgen05 (SURVEY.md section 8 row f3: the RCAB backbone convs,
 * models/networks.py:449-482) -------------------------------------------------------------------
 * x, out: (n,64,h,w) dense NHWC bf16, stride 1, pad 1.  out = LeakyReLU_slope(conv(x) + bias)
 * (slope 1 = none, 0 = ReLU).  If channel_sums != NULL it receives sum over (h,w) of `out` per
 * (n, channel) in fp32 -- the global average pool of CALayer for free.  The call zero-fills it unless
 * EAVSR_CONV_SUMS_PREZEROED is set in `flags` (the caller zeroes one buffer for a whole residual group).
 * Weights are packed once with eavsr_conv3x3_pack_weight into eavsr_conv3x3_packed_weight_bytes()
 * bytes (16-byte aligned). */
size_t eavsr_conv3x3_packed_weight_bytes(void);
int eavsr_conv3x3_pack_weight(const void* weight /* (64,64,3,3) */, void* packed, int cin, int cout, int dtype,
                              void* stream);
#define EAVSR_CONV_SUMS_PREZEROED 1u
int eavsr_conv3x3_forward(const void* x, const void* packed_weight, const void* bias, void* out,
                          float* channel_sums, int n, int cin, int cout, int h, int w, float negative_slope,
                          int dtype, unsigned flags, void* stream);

/* The same convolution with the tail of the previous RCABlock folded into its input
 * (models/networks.py:449-465): the producer warps build y = res * sigmoid(W2 relu(W1 mean(res) + b1) + b2)
 * + skip while staging the halo tile (res_sums = per-(n, channel) sums of res from the call that produced
 * it, reduction 16), the convolution runs on y, and y itself is written to y_out (the next block's
 * skip).  One launch and ~17 MB of HBM traffic less than eavsr_ca_scale_forward + eavsr_conv3x3_forward
 * per block.  n <= 8; everything dense NHWC bf16. */
int eavsr_conv3x3_ca_forward(const void* skip, const void* res, const float* res_sums, const void* w1,
                             const void* b1, const void* w2, const void* b2, void* y_out,
                             const void* packed_weight, const void* bias, void* out, float* channel_sums, int n,
                             int h, int w, float negative_slope, int dtype, unsigned flags, void* stream);

/* A whole chain of such convolutions -- the 61 of one RCAGroup (models/networks.py:467-482) -- in ONE cooperative
 * launch: layer i + 1 reads what layer i wrote (grid-wide barrier between layers), the launch gap, TMEM allocation
 * and cold weight load that a launch per convolution pays are paid once, and the next layer's weights stream in
 * while a CTA waits at the barrier.  Each layer is eavsr_conv3x3_forward (res == NULL) or eavsr_conv3x3_ca_forward
 * (res != NULL, `x` is the skip tensor).  channel_sums buffers must be ZERO on entry (as with
 * EAVSR_CONV_SUMS_PREZEROED).  Buffers may be recycled between layers (activations are read through L2 only).
 * sync_workspace: 4 bytes of device memory (the call zero-fills it).  nlayers <= 64, n <= 8 when any layer is fused. */
typedef struct EavsrConvLayer {
  const void* x;              /* input, or the skip tensor of the fused mode */
  const void* packed_weight;  /* eavsr_conv3x3_pack_weight image */
  const void* bias;           /* (64) bf16 or NULL */
  void* out;
  float* channel_sums;        /* (n, 64) fp32, zeroed, or NULL */
  const void* res;            /* fused channel-attention input, or NULL */
  const float* res_sums;
  const void* w1;
  const void* b1;
  const void* w2;
  const void* b2;
  void* y_out;
  float negative_slope;
} EavsrConvLayer;
int eavsr_conv3x3_chain_forward(const EavsrConvLayer* layers, int nlayers, int n, int h, int w, int dtype,
                                void* sync_workspace, void* stream);

/* ---- reconstruction tail to 8-bit frames on tcgen05 (EAVSRP.upsample, models/eavsrp_model.py:350-364, followed by
 * the visuals of models/base_model.py:146-150) ------------------------------------------------------------------
 * For y < out_h, x < out_w and c < 3:
 *   out[n, y, x, c] = rint(clamp(255 * (bias[c] + sum_{ci, ky, kx} W[c, ci, ky, kx] * x[n, ci, y+ky-1, x+kx-1]
 *                                        + up_s(lr)[n, c, y, x]), 0, 255))
 * i.e. conv_last(x) + F.interpolate(lr, scale_factor=s, mode='bilinear', align_corners=False), then
 * torch.clamp(sr * 255, 0, 255).round() as uint8.
 *   x:    (n, 64, h, w) bf16, dense channels_last (x_strides = {h*w*64, 1, w*64, 64}), 16-byte aligned; zero
 *         padding at the borders as nn.Conv2d(64, 3, 3, 1, 1).  Rows and columns beyond the crop are still read.
 *   W, bias: conv_last's (3, 64, 3, 3) weight, packed once with eavsr_sr_tail_pack_weight into
 *         eavsr_sr_tail_packed_weight_bytes() bytes (16-byte aligned), and its (3) bf16 bias or NULL.
 *   lr:   (n, 3, h/s, w/s) fp32 by element strides lr_strides (n, c, h, w) -- e.g. one frame of a padded clip.
 *         up_s is ATen's upsample_bilinear2d: source max((dst + 0.5) / s - 0.5, 0), upper neighbour clamped.
 *   out:  uint8 by element strides out_strides in (n, y, x, c) order -- e.g. frame i of an (n, t, Ho, Wo, 3) clip.
 * Products are bf16 x bf16 with fp32 accumulation; the sum, bias and bilinear base are added in fp32 (the residual
 * is never rounded to bf16), and rint rounds half to even as torch.round does.  scale = s is 2 or 4; h and w are
 * multiples of s; 0 < out_h <= h, 0 < out_w <= w (the crop of a replicate-padded clip).  Anything else returns
 * EAVSR_ERR_INVALID; dtype other than EAVSR_BF16 returns EAVSR_ERR_UNSUPPORTED. */
size_t eavsr_sr_tail_packed_weight_bytes(void);
int eavsr_sr_tail_pack_weight(const void* weight /* (3,64,3,3) */, void* packed, int cin, int cout, int dtype,
                              void* stream);
int eavsr_sr_tail_u8_forward(const void* x, const int64_t x_strides[4], const void* packed_weight, const void* bias,
                             const float* lr, const int64_t lr_strides[4], void* out, const int64_t out_strides[4],
                             int n, int c, int h, int w, int scale, int out_h, int out_w, int dtype, void* stream);

/* ---- the same tail to 8-bit limited-range Y'CbCr 4:2:0 planes ---------------------------------------------------
 * With v = clamp(bias + conv_last(x) + up_s(lr), 0, 1) per pixel (the residual in fp32, as above), writes
 *   Y[n, y, x]           = rint(16 + 219 * Yc(v[n, :, y, x]))                           for y < out_h, x < out_w
 *   U[n, y/2, x/2]       = rint(128 + 112 / (1 - kb) * (m_b - Yc(m))),  V likewise with m_r and kr,
 * where Yc(p) = kr p_r + kg p_g + kb p_b, kg = 1 - kr - kb, and m is the mean of v over the 2x2 block of even y, x
 * (centre-sited chroma).  The fp32 order of operations is that of rgb_to_yuv420 in eavsr_b200/yuv.py.  kr, kb are
 * the matrix (BT.709: 0.2126, 0.0722; BT.601: 0.299, 0.114).
 *   x, W, bias, lr: as eavsr_sr_tail_u8_forward, with the same packed weight.
 *   out_y, out_u, out_v: uint8 planes by element strides of the plane viewed as (n, 1, H, W) (the second stride is
 *         not read); out_u and out_v are (out_h/2, out_w/2).  Arbitrary strides write I420 planes or NV12 (u = uv[...,
 *         0::2], v = uv[..., 1::2]).
 * out_h and out_w must be even; everything eavsr_sr_tail_u8_forward rejects, and a bad matrix, returns
 * EAVSR_ERR_INVALID; dtype other than EAVSR_BF16 returns EAVSR_ERR_UNSUPPORTED. */
int eavsr_sr_tail_yuv420_forward(const void* x, const int64_t x_strides[4], const void* packed_weight, const void* bias,
                                 const float* lr, const int64_t lr_strides[4], void* out_y, const int64_t y_strides[4],
                                 void* out_u, const int64_t u_strides[4], void* out_v, const int64_t v_strides[4],
                                 int n, int c, int h, int w, int scale, int out_h, int out_w, float kr, float kb,
                                 int dtype, void* stream);

/* ---- the same tail to 16-bit RGB frames (10-, 12- or 16-bit codes) ----------------------------------------------
 * With M = 2^bits - 1, for y < out_h, x < out_w and c < 3:
 *   out[n, y, x, c] = rint(clamp(M * (bias[c] + conv_last(x)[n, c, y, x] + up_s(lr)[n, c, y, x]), 0, M))
 * i.e. eavsr_sr_tail_u8_forward with M in place of 255, the code in the low bits of a uint16 sample.
 *   x, W, bias, lr: as eavsr_sr_tail_u8_forward, with the same packed weight.
 *   out:  uint16, 2-byte aligned, by element strides out_strides in (n, y, x, c) order.
 * bits must be 10, 12 or 16; that, a misaligned out, and everything eavsr_sr_tail_u8_forward rejects return
 * EAVSR_ERR_INVALID; dtype other than EAVSR_BF16 returns EAVSR_ERR_UNSUPPORTED. */
int eavsr_sr_tail_u16_forward(const void* x, const int64_t x_strides[4], const void* packed_weight, const void* bias,
                              const float* lr, const int64_t lr_strides[4], void* out, const int64_t out_strides[4],
                              int n, int c, int h, int w, int scale, int out_h, int out_w, int bits, int dtype,
                              void* stream);

/* ---- the same tail to limited-range Y'CbCr 4:2:0 planes of 10, 12 or 16 bits ------------------------------------
 * eavsr_sr_tail_yuv420_forward at bits b with k = 2^(b - 8), each code stored times 2^shift in a uint16 sample:
 *   Y[n, y, x]     = rint(16k + 219k * Yc(v[n, :, y, x]))                         for y < out_h, x < out_w
 *   U[n, y/2, x/2] = rint(128k + 112k / (1 - kb) * (m_b - Yc(m))),  V likewise with m_r and kr,
 * in the fp32 order of rgb_to_yuv420(..., bits=b, shift=shift) in eavsr_b200/yuv.py (112k / (1 - kb) is computed as
 * k * (112 / (1 - kb)), the same fp32 value).  shift = 0 keeps the codes in the low bits (yuv420p10le), shift =
 * 16 - b puts them in the high bits (P010, P012).  kr, kb as for eavsr_sr_tail_yuv420_forward; BT.2020 is 0.2627,
 * 0.0593.
 *   x, W, bias, lr: as eavsr_sr_tail_u8_forward, with the same packed weight.
 *   out_y, out_u, out_v: uint16 planes, each 2-byte aligned, by element strides of the plane viewed as (n, 1, H, W)
 *         (the second stride is not read); out_u and out_v are (out_h/2, out_w/2).  Arbitrary strides write planar
 *         yuv420p10le or P010 (u = uv[..., 0::2], v = uv[..., 1::2] of a uint16 view with a row pitch).
 * bits not in {10, 12, 16}, shift not in {0, 16 - bits}, a misaligned plane, an odd out_h or out_w, a bad matrix and
 * everything eavsr_sr_tail_u8_forward rejects return EAVSR_ERR_INVALID; dtype other than EAVSR_BF16 returns
 * EAVSR_ERR_UNSUPPORTED. */
int eavsr_sr_tail_yuv420_u16_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                     const void* bias, const float* lr, const int64_t lr_strides[4], void* out_y,
                                     const int64_t y_strides[4], void* out_u, const int64_t u_strides[4], void* out_v,
                                     const int64_t v_strides[4], int n, int c, int h, int w, int scale, int out_h,
                                     int out_w, float kr, float kb, int bits, int shift, int dtype, void* stream);

/* ---- the same tail's 8-bit frame measured against a ground-truth frame (the error sum of PSNR) --------------------
 * With q[n, y, x, c] the code eavsr_sr_tail_u8_forward writes (the same expression, bit for bit), adds
 *   sse[n * sse_stride] += sum_{y < out_h, x < out_w, c < 3} (q[n, y, x, c] - gt[n, y, x, c])^2
 * exactly, in 64-bit integers, and, when out is not NULL, also stores q into out as eavsr_sr_tail_u8_forward does.
 * sse is added to, not overwritten: the caller zeroes it (e.g. once per clip, then passes frame i's column of an
 * (n, t) int64 tensor with sse_stride = t).  Each image's sum is exact and independent of the order of the additions,
 * so two calls on the same operands give the same bits.
 *   x, W, bias, lr: as eavsr_sr_tail_u8_forward, with the same packed weight.
 *   gt:   uint8 by element strides gt_strides in (n, y, x, c) order, (n, out_h, out_w, 3).
 *   out, out_strides: as eavsr_sr_tail_u8_forward, or both NULL for no store.
 *   sse:  n unsigned 64-bit integers (an int64 tensor holds the same bits: a sum stays below 2^63 for any frame
 *         under 4.7e13 pixels), 8-byte aligned, by element stride sse_stride.
 * A null x, gt, sse or stride array (out_strides only when out is set), a misaligned sse and everything
 * eavsr_sr_tail_u8_forward rejects return EAVSR_ERR_INVALID; dtype other than EAVSR_BF16 returns
 * EAVSR_ERR_UNSUPPORTED. */
int eavsr_sr_tail_u8_sse_forward(const void* x, const int64_t x_strides[4], const void* packed_weight, const void* bias,
                                 const float* lr, const int64_t lr_strides[4], const void* gt,
                                 const int64_t gt_strides[4], void* out, const int64_t out_strides[4],
                                 unsigned long long* sse, long long sse_stride, int n, int c, int h, int w, int scale,
                                 int out_h, int out_w, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EAVSR_B200_H_ */
