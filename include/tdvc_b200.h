/* tdvc_b200 — C-ABI of the B200-native (sm_100a) kernels behind TDVC's P-frame coding forward pass.
 *
 * Drop-in boundary (SURVEY.md 8b):
 *   b2  tdvc_dcn_v2_forward      replaces the reference's only native op,
 *                                `_ext.dcn_v2_forward` (reference main/utils/dcnv2/src/vision.cpp:5,
 *                                src/dcn_v2.h:9-46, src/cuda/dcn_v2_cuda.cu:20-95).
 *   b3  every other entry point  is one fused stage of `VideoCompressor.forward`
 *                                (reference main/model/pnet.py:26-83); each comment cites the
 *                                reference lines it replaces.
 * Conventions: plain pointers and sizes, no torch types. All pointers are DEVICE pointers unless a name
 * ends in `_host`. No allocation, no host synchronisation, no global mutable state inside: the caller
 * owns every buffer (workspace sizes are spelled out per call) and passes the CUDA stream (a
 * `cudaStream_t` cast to void*), so calls are re-entrant and thread-safe (nn.DataParallel replicas).
 * Return value: 0 on success, a negative TDVC_E* code otherwise; tdvc_last_error() gives the text.
 * Activations are fp32, channels-last (NHWC): element (n,y,x,c) at ((n*H + y)*W + x)*ld + c, where `ld`
 * (floats per pixel) may exceed the channel count (views into wider tensors).
 */
#ifndef TDVC_B200_H
#define TDVC_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define TDVC_OK 0
#define TDVC_EINVAL (-1)   /* bad argument (shape / alignment / unsupported configuration) */
#define TDVC_ECUDA (-2)    /* CUDA launch error */

#define TDVC_ACT_NONE 0
#define TDVC_ACT_RELU 1
#define TDVC_ACT_LRELU 2   /* slope in `slope` */
#define TDVC_ACT_CLAMP01 3
#define TDVC_POST_NONE 0
#define TDVC_POST_GDN 1    /* v = mul * rsqrt(v)   (compressai GDN,  SURVEY App. A) */
#define TDVC_POST_IGDN 2   /* v = mul * sqrt(v)    (compressai IGDN) */

int tdvc_version(void);
const char* tdvc_last_error(void);

/* ---- generic 2-D convolution, implicit GEMM over NHWC (every nn.Conv2d / Conv3d(1,3,3) /
 * 1x1 / MaskedConv2d / GDN channel mix of the hot path; reference pnet.py passim, utils.py:43-56,
 * flownet.py:187-227; compressai layers per SURVEY App. A).
 * Input = channel concatenation of up to 4 sources (replaces torch.cat/stack, pnet.py:148,156,181,257,259,288).
 * v = bias + sum w*x ; post (GDN/IGDN with `mul`) ; act ; + res1 ; + res2 ; store (optionally pixel-shuffled x2).
 * weight layout: [kh*kw][cin_pad][cout_pad] fp32, zero padded; for shuffle==2 the output-channel order is
 * permuted on the host to co' = (dy*2+dx)*(cout/4) + c (nn.PixelShuffle folded into the store).
 * Constraints: src_c[i] % 4 == 0, src_ld[i] % 4 == 0, 16-byte aligned sources, cin_pad % 8 == 0,
 * cout_pad % 16 == 0.  `impl`: 0 = auto, 1 = SIMT fp32 FFMA kernel, 3 = SIMT fp32 kernel for <= 4 output channels
 * (single source, 3x3 / 7x7, stride 1; csrc/conv_small.cu; auto picks it for those shapes), 2 = tcgen05 tensor-core kernel
 * (fp16 split: x = hi + lo, w = hi + lo, (w_hi + w_lo)*(x_hi + x_lo), fp32 accumulate in TMEM; needs weight_f16).                                             */
typedef struct {
  const float* src[4];
  int32_t src_c[4];
  int32_t src_ld[4];
  int32_t n_src;
  int32_t N, H, W;          /* input size */
  int32_t Ho, Wo;           /* output size (before pixel shuffle) */
  const float* weight;
  const float* bias;        /* [cout_pad] or NULL */
  int32_t cin, cin_pad, cout, cout_pad;
  int32_t kh, kw, stride, pad;
  int32_t in_square;        /* 1: x -> x*x on load (GDN) */
  int32_t act;
  float slope;
  int32_t post;
  const float* mul; int32_t mul_ld;
  const float* res1; int32_t res1_ld;
  const float* res2; int32_t res2_ld;
  float* out; int32_t out_ld;
  int32_t shuffle;          /* 0 or 2 */
  int32_t impl;
  const void* weight_f16;  /* tcgen05 path: fp16 (hi | lo*2^12) weight blocks built by tdvc_conv2d_pack_f16, or NULL */
  float* chan_sum;          /* optional, tcgen05 path: partial channel sums of the stored output, [rows][N][cout] floats with
                               rows = tdvc_conv2d_chan_sum_rows(p) (the caller zeroes the buffer): the squeeze-excitation mean of
                               reference inflate.py:189-207 comes out of the producing layer's epilogue, tdvc_se_apply(nblk = rows)
                               finishes it.  Deterministic (one owner per cell, fixed walk order).  NULL: not computed */
  int32_t w_shift;          /* tcgen05 split scheme (tdvc_conv2d_f16_is_split): the fp16 weight blocks hold w * 2^w_shift, chosen by
                               the caller so that max|w| * 2^w_shift lies in [2^13, 2^14]; same value at pack time and at launch */
  int32_t order;            /* tcgen05 path: 1 = walk the output tiles in descending order.  Alternating the direction between
                               consecutive layers lets a layer start on the tiles its producer wrote last (still in the 126 MB L2) */
  int32_t out_planar;       /* 1: store NCHW planes, out[((n*cout + c)*Ho + y)*Wo + x] (no shuffle / residual / post);
                               the DCN offset/mask head writes the reference's planar offset & mask tensors this way */
  float* out_absmax;        /* optional device scalar: *out_absmax = max(*out_absmax, max |v| over every value stored) (atomic
                               max on the float bits; the caller zeroes it).  Feeds `in_absmax` of the GDN that squares this output */
  const float* in_absmax;   /* tcgen05 path with in_square: device scalar >= max |x| of the input.  x*x is pre-scaled by the exact
                               power of two that keeps max x*x below 2^15 (fp16 operands saturate at 65504) and the scale is undone
                               in the epilogue; NULL or a value <= 181 leaves the arithmetic unchanged.  The SIMT path ignores it */
  int32_t products;         /* tcgen05 path: 0 = fp32-class scheme (fp16 hi+lo split of both operands, 4 or 3 MMA products per
                               MAC); 1 = one product, fp16(w) * fp16(x) with fp32 accumulation - the arithmetic of the reference
                               under autocast (`enabled_amp`); weight_f16 must have been packed with the same value */
} TdvcConvParams;
int tdvc_conv2d(const TdvcConvParams* p, void* stream);
/* tcgen05 path: size of / builder for the fp16 (hi, lo) weight blocks of a convolution, from its fp32 packed
 * `weight` ([kh*kw][cin_pad][cout_pad]).  Only geometry fields (kh, kw, stride, pad, cin, cin_pad, cout, cout_pad,
 * post, in_square) and `weight` are read.  bytes == 0: the shape has no tensor-core path (SIMT kernel is used). */
size_t tdvc_conv2d_f16_bytes(const TdvcConvParams* p);
int tdvc_conv2d_pack_f16(const TdvcConvParams* p, void* out, void* stream);
/* 1 when the fp16 weight blocks of the shape are pre-scaled by 2^w_shift (3-product split scheme with 128-channel tiles, and
 * every one-product layer; the caller must then set p->w_shift as described above), else 0 */
int tdvc_conv2d_f16_is_split(const TdvcConvParams* p);
/* which kernel tdvc_conv2d runs for *p, as fp16 MMA products issued per algorithmic MAC: 0 = an exact fp32 SIMT kernel,
 * 4 = hi/lo rows, 3 = split scheme, 1 = one product; -1 = invalid parameters (bench.py's `products_per_mac`) */
int tdvc_conv2d_products(const TdvcConvParams* p);
/* rows of the `chan_sum` buffer tdvc_conv2d would fill for *p; 0 = this launch cannot produce channel sums */
int tdvc_conv2d_chan_sum_rows(const TdvcConvParams* p);

/* ---- DCNv2 forward, the reference's `_ext.dcn_v2_forward` (dcn_v2.h:9-46): contiguous NCHW fp32,
 * offset (N, 2*dg*kh*kw, H, W) ordered [g][tap][dy,dx], mask (N, dg*kh*kw, H, W), weight (O, C, kh, kw),
 * bias (O; NULL is accepted and means no bias - the reference's op always passes one, dcn_v2.h:12).  The configuration TDVC uses (3x3, stride 1,
 * pad 1, dilation 1, 8 channels per deformable group) runs on the fused channels-last kernel through `workspace`; every
 * other geometry (any kernel size / stride / padding / dilation / group width) is answered by a generic NCHW kernel that
 * needs no workspace.  Inconsistent shapes return TDVC_EINVAL (the reference raises through AT_ASSERTM,
 * dcn_v2_cuda.cu:38-62).  workspace: at least tdvc_dcn_v2_workspace_bytes(N,C,O,H,W,dg) bytes.  No im2col `columns`
 * tensor is materialised (reference dcn_v2_cuda.cu:68, 4.5 GB at 1920x1024).                            */
size_t tdvc_dcn_v2_workspace_bytes(int N, int C, int O, int H, int W, int dg);
int tdvc_dcn_v2_forward(const float* input, const float* weight, const float* bias, const float* offset,
                        const float* mask, float* output, int N, int C, int O, int H, int W,
                        int kh, int kw, int sh, int sw, int ph, int pw, int dh, int dw, int dg,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- DCNv2 backward, the reference's `_ext.dcn_v2_backward` (dcn_v2.h:48-92, dcn_v2_cuda.cu:97-216,
 * dcn_v2_im2col_cuda.cu:197-327): same tensor conventions as the forward, any geometry; grad_output (N, O, Ho, Wo).
 * Writes grad_input (N,C,H,W), grad_offset / grad_mask (shapes of offset / mask), grad_weight (O,C,kh,kw), grad_bias (O).
 * Deterministic (the reference's col2im uses float atomicAdd): grad_input is accumulated as 64-bit fixed point in `workspace`
 * (>= tdvc_dcn_v2_backward_workspace_bytes(N,C,O,H,W,Ho,Wo,kh*kw) bytes, 16-byte aligned: fixed-point grad_input, the im2col rows and the partial sums of the weight gradient), everything else has one owner per element.
 * `bias` is not needed (its gradient is the plain sum of grad_output).                                                      */
size_t tdvc_dcn_v2_backward_workspace_bytes(int N, int C, int O, int H, int W, int Ho, int Wo, int K);
int tdvc_dcn_v2_backward(const float* input, const float* weight, const float* offset, const float* mask,
                         const float* grad_output, float* grad_input, float* grad_offset, float* grad_mask,
                         float* grad_weight, float* grad_bias, int N, int C, int O, int H, int W, int kh, int kw,
                         int sh, int sw, int ph, int pw, int dh, int dw, int dg, void* workspace, size_t workspace_bytes,
                         void* stream);

/* Fused channels-last form used inside the P-frame graph (reference dcn_v2_amp.py:219-234 + :67-69 +
 * pnet.py:180): offsets / mask read straight from the 27*dg-channel conv_offset_mask output, sigmoid,
 * bilinear gather, 9*C -> O contraction, bias, optional fp16 rounding (`round_fp16`, the reference's
 * `.half()`), optional LeakyReLU evaluated on the fp16 value.  weight_packed: [C*9][O_pad] fp32 with
 * row j = c*9 + tap (O_pad = O rounded up to 64).                                                      */
typedef struct {
  const float* input; int32_t in_ld;      /* (N,H,W,C) */
  const float* offset; int32_t off_ld;    /* channel g*18 + 2*tap (+1)  */
  const float* mask; int32_t mask_ld;     /* channel g*9 + tap */
  int32_t mask_is_logit;                  /* 1: apply sigmoid */
  const float* weight_packed; const float* bias;
  float* out; int32_t out_ld;
  int32_t N, H, W, C, O, O_pad, dg;
  int32_t round_fp16;
  int32_t act; float slope;
  int32_t impl;                           /* 0 = auto, 1 = SIMT fp32 contraction, 2 = tcgen05 (fp16 hi/lo split) */
  const void* weight_f16;                 /* tcgen05 path: tdvc_dcn_pack_f16 output, or NULL */
  /* tcgen05 path (csrc/dcn_tc.cu) reads gather-friendly layouts instead of `input` / channels-last offsets:   */
  const float* input_gp;                  /* "group planar" input [(n*dg + g)][H][W][8] (tdvc_nhwc_to_group_planar) */
  int32_t params_planar;                  /* 1: offset / mask are NCHW planes as in the reference (dcn_v2.h:9-46):
                                             offset plane g*18 + 2*tap (+1), mask plane g*9 + tap, H*W floats each;
                                             off_ld / mask_ld then count the PLANES per image of the tensor they live in */
} TdvcDcnParams;
int tdvc_dcn_nhwc(const TdvcDcnParams* p, void* stream);
/* tcgen05 DCN: fp16 (hi | lo*2^12) weight blocks from weight_packed ([C*9][O_pad] fp32); O <= 64, 8 channels per group */
size_t tdvc_dcn_f16_bytes(int dg);
int tdvc_dcn_pack_f16(const float* weight_packed, int O, int O_pad, int dg, void* out, void* stream);
/* NHWC (src_ld floats per pixel, C % 8 == 0) -> [(n*C/8 + g)][H][W][8]: one 32-byte sector per (pixel, group) */
int tdvc_nhwc_to_group_planar(const float* src, int src_ld, float* dst, int N, int H, int W, int C, void* stream);

/* ---- frame plumbing ----
 * zero_bytes: cudaMemsetAsync(p, 0, n) on the stream (per-frame accumulators).
 * slices_hash: 128-bit content hash of n_slices slabs of slice_words 32-bit words each (slab i starts at base + i*stride_words):
 *   out[2*i], out[2*i+1] = two independent order-free sums of mixed (word, position) pairs.  VideoCompressor.forward keys its
 *   per-GOP caches on it (features of the I-frame, reference pnet.py:213-217, and of the previous reconstructions, :277-283,
 *   are recomputed by the reference for every P-frame although their inputs repeat).
 * bpp_finish: bpp[c] = (acc[2c] + acc[2c+1]) * scale for the two coders (reference pnet.py:38-43, 62-67).                    */
int tdvc_zero_bytes(void* p, size_t n, void* stream);
int tdvc_slices_hash(const void* base, int64_t slice_words, int64_t stride_words, int n_slices, uint64_t* out, void* stream);
int tdvc_bpp_finish(const double* acc4, float* bpp2, double scale, void* stream);

/* ---- layout ---- */
int tdvc_nchw_to_nhwc(const float* src, float* dst, int N, int C, int H, int W, int dst_ld, void* stream); /* pads c>=C with 0 */
int tdvc_nhwc_to_nchw(const float* src, int src_ld, float* dst, int N, int C, int H, int W, void* stream);

/* ---- SPyNet pieces (reference flownet.py:82-140) ----
 * avgpool2x2: F.avg_pool2d(2,2) (:102-114).
 * spynet_prep: flow_up = 2 * bilinear_x2(flow_prev, align_corners=True) (:124-128) [zeros if flow_prev NULL];
 *   warped = grid_sample(supp, border, align_corners=True) with the reference's normalise round trip (:8-48);
 *   out8 = [ref(3), warped(3), flow_up(2)] (:131-138).  Images are NHWC with ld 4 (3 channels + 0 pad). */
int tdvc_avgpool2x2(const float* src, float* dst, int N, int H, int W, int C, void* stream);
int tdvc_spynet_prep(const float* ref4, const float* supp4, const float* flow_prev, float* out8,
                     int N, int h, int w, void* stream);
/* Backward of spynet_prep with respect to the coarse flow (the images are network inputs): grad_out8 (N,h,w,8) ->
 * grad_flow_prev (N,h/2,w/2,2).  The warp's derivative follows grid_sample's border rule (a clamped coordinate has zero
 * derivative, corners outside the image contribute zero); the x2 upsample's adjoint is a gather (deterministic).
 * grad_fine_ws: N*h*w*2 floats of scratch (d loss / d upsampled flow).                                             */
int tdvc_spynet_prep_backward(const float* supp4, const float* flow_prev, const float* grad_out8, float* grad_fine_ws,
                              float* grad_flow_prev, int N, int h, int w, void* stream);
/* nn.Upsample(x2, bilinear, align_corners=False) on NHWC (reference pnet.py:117,159) */
int tdvc_upsample2x(const float* src, float* dst, int N, int H, int W, int C, void* stream);
/* offset + flow.repeat(1, C/2, 1, 1)  (reference pnet.py:163) */
int tdvc_add_flow_tiled(const float* offset, const float* flow2, float* out, int N, int H, int W, int C, void* stream);

/* ---- element-wise ---- */
int tdvc_axpby(const float* a, const float* b, float* out, int64_t n, float alpha, float beta, void* stream);
/* out[t] = lrelu(x[t] + tmp) for t < T (Bottleneck3D temporal broadcast add, reference pnet.py:313-314) */
int tdvc_bcast_add_lrelu(const float* x, const float* tmp, float* out, int T, int64_t n_per_t, float slope, void* stream);
/* the same for T <= 4 frames that do not lie next to each other: out[t] = lrelu(x[t] + tmp), `x` / `out` are HOST arrays of T
 * device pointers (n floats each); tmp is read once for all of them */
int tdvc_bcast_add_lrelu_multi(const float* const* x, const float* tmp, float* const* out, int T, int64_t n, float slope,
                               void* stream);
int tdvc_round_half_even(const float* x, float* out, int64_t n, void* stream);

/* ---- squeeze-excitation (reference inflate.py:159-208): two launches.
 * se_partial_sums: partial[b][n][c] = sum over a slab of pixels (deterministic two-stage mean).
 * se_apply: s = sigmoid(W2 relu(W1 mean + b1) + b2) computed once per image (a one-block kernel that overwrites
 * partial[n*C + c] with the gate), then out = act(x*s) (+ res) streamed by a second kernel.
 * w1: [Cr][C], w2: [C][Cr] (the 1x1 conv weights as stored). nblk <= 1024.
 * Optional second output in the same pass: out2 = sub_from - out (the residual `input_feat - prediction` of reference
 * pnet.py:55 when `out` is the prediction); both NULL otherwise.                                      */
int tdvc_se_partial_sums(const float* x, int ld, int N, int64_t HW, int C, float* partial, int nblk, void* stream);
int tdvc_se_apply(const float* x, int ld, float* partial, int nblk, const float* w1, const float* b1,
                  const float* w2, const float* b2, int N, int64_t HW, int C, int Cr, int act, float slope,
                  const float* res, int res_ld, float* out, int out_ld, const float* sub_from, int sub_ld,
                  float* out2, int out2_ld, void* stream);

/* ---- entropy models -> bits (compressai EntropyBottleneck / GaussianConditional forward in eval mode,
 * SURVEY App. A; reductions of reference pnet.py:38-43,62-67).  `acc` is a device double: += sum ln(p).
 * eb_bits: z NHWC (ld=C); per-channel MLP params already softplus'ed / tanh'ed on the host side:
 *   mats: [C][33] = M0(3x1) M1(3x3) M2(3x3) M3(3x3) M4(1x3); biases: [C][13]; factors: [C][12]; medians [C].
 *   writes z_hat = round(z - med) + med.
 * gc_bits: y NHWC (ld=C), params NHWC with scales at channel c and means at channel C + c (ld = params_ld).   */
int tdvc_eb_bits(const float* z, float* z_hat, const float* mats, const float* biases, const float* factors,
                 const float* medians, int64_t npix, int C, double* acc, void* stream);
int tdvc_gc_bits(const float* y, const float* params, int params_ld, int64_t npix, int C, double* acc, void* stream);
/* Training-mode forms (`self.training`, reference pnet.py:26-83 with compressai's quantize(.., "noise")): the quantisers add
 * uniform noise instead of rounding.  eb_bits_noise: z_tilde = z + noise, likelihood at z_tilde.  gc_bits_noise: likelihood of
 * y + noise under (scales, means).  `noise` has the layout of the latent it is added to.
 * eb_aux_loss: EntropyBottleneck.loss() = sum |logits_cumulative(quantiles) - target| (quantiles [C][3], target3 [3]) -> *out.
 * uniform_noise: out[i] ~ U[-0.5, 0.5) from Philox4x32-10 keyed by `seed`, sub-stream `stream_id`, counter i / 4.          */
int tdvc_eb_bits_noise(const float* z, const float* noise, float* z_tilde, const float* mats, const float* biases,
                       const float* factors, int64_t npix, int C, double* acc, void* stream);
int tdvc_gc_bits_noise(const float* y, const float* noise, const float* params, int params_ld, int64_t npix, int C,
                       double* acc, void* stream);
int tdvc_eb_aux_loss(const float* mats, const float* biases, const float* factors, const float* quantiles,
                     const float* target3, int C, float* out, void* stream);
/* d eb_aux_loss / d quantiles ([C][3]) times *grad_out (device scalar): the gradient `aux_loss.backward()` needs to step the
 * aux optimiser on `.quantiles` (reference tools/train.py:101-113,147-159; matrices / biases / factors are detached there). */
int tdvc_eb_aux_loss_grad(const float* mats, const float* biases, const float* factors, const float* quantiles,
                          const float* target3, const float* grad_out, int C, float* grad_quantiles, void* stream);
int tdvc_uniform_noise(float* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream);
/* the same draws with the seed read from device memory at run time: inside a captured CUDA graph the caller advances *seed_dev
 * with a captured operation, so that every replay of a training step quantises with fresh noise */
int tdvc_uniform_noise_dev(float* out, int64_t n, const uint64_t* seed_dev, uint64_t stream_id, void* stream);
/* Backward of the two noise-mode reductions (the reference takes them from autograd through compressai, tools/train.py:132-145).
 * S = sum ln max(p, 1e-9); grad_sum = d loss / d S (device scalar); compressai's LowerBound gradient rule (pass where the input
 * is above the bound or the gradient is negative) for the likelihood bound and the 0.11 scale bound.
 * gc_bits_backward: grad_y (ld = C), grad_params (ld = params_ld: d / d scale at channel c, d / d mean at C + c).
 * eb_bits_backward: grad_z (ld = C) and the gradients with respect to the TRANSFORMED parameters the kernels read (mats =
 *   softplus(matrix) [C][33], biases [C][13], factors = tanh(factor) [C][12]); deterministic (one CTA per channel).          */
int tdvc_gc_bits_backward(const float* y, const float* noise, const float* params, int params_ld, const float* grad_sum,
                          float* grad_y, float* grad_params, int64_t npix, int C, void* stream);
int tdvc_eb_bits_backward(const float* z_tilde, const float* mats, const float* biases, const float* factors, const float* grad_sum,
                          float* grad_z, float* grad_mats, float* grad_biases, float* grad_factors, int64_t npix, int C,
                          void* stream);

/* ---- backward pieces of the convolutions (SURVEY 8f row 1; the reference's training step takes them from cuDNN through
 * autograd, tools/train.py:125-159).  dgrad is tdvc_conv2d itself on the transposed, flipped weight (pad' = k - 1 - pad),
 * after zero_insert for a strided layer; see tdvc_b200/ops.py `conv2d`.
 * act_backward: grad_pre = grad_y * f'(y) from the layer's OUTPUT y (TDVC_ACT_*; NONE copies).
 * zero_insert: out (N,H,W,C) <- g (N,Ho,Wo,C): out[n][oy*stride][ox*stride] = g[n][oy][ox], zero elsewhere (C % 4 == 0).
 * conv2d_wgrad: grad_w[cout][cin][k][k] (nn.Conv2d.weight layout) = sum_p x[p*stride + tap - pad][ci] * grad_y[p][co] and
 *   grad_b[co] = sum_p grad_y[p][co] (NULL: skipped); x (N,H,W,cin) / grad_y (N,Ho,Wo,cout) NHWC with leading dimensions;
 *   `products` = 3: fp32-class (warp-level TF32 MMAs over staged 32-pixel chunks, (hi, lo) operand pairs, three products),
 *   1: one TF32 product (what cuDNN runs by default for fp32 training convolutions; the reference's shipped cfg/train.yaml
 *   trains under AMP, i.e. with fp16 products) - on tcgen05 for stride-1 "same"-padded 1x1 / 3x3 / 7x7 layers at least 16
 *   pixels wide (csrc/wgrad_tc.cu; operands truncated to TF32 by the tensor core), on the warp-level kernel otherwise;
 *   deterministic (fixed-order two-stage sum) in every case.
 *   workspace: tdvc_conv2d_wgrad_workspace_bytes(N,Ho,Wo,cin,cout,k). */
int tdvc_act_backward(const float* y, const float* grad_y, float* grad_pre, int64_t n, int act, float slope, void* stream);
int tdvc_zero_insert(const float* g, int g_ld, float* out, int out_ld, int N, int H, int W, int Ho, int Wo, int C, int stride,
                     void* stream);
size_t tdvc_conv2d_wgrad_workspace_bytes(int N, int Ho, int Wo, int cin, int cout, int k);
int tdvc_conv2d_wgrad(const float* x, int x_ld, const float* grad_y, int g_ld, int N, int H, int W, int cin, int cout, int k,
                      int stride, int pad, int in_square, int products, float* grad_w, float* grad_b_or_null, void* workspace,
                      size_t workspace_bytes, void* stream);
/* conv2d_pack_weight: nn.Conv2d.weight (O, I, k, k) -> the implicit-GEMM layout tdvc_conv2d reads, out[k*k][cin_pad][cout_pad]
 *   fp32, zero padded, in ONE launch (the training step re-packs every weight after every optimiser step).  transposed = 0:
 *   out[tap][ci][co] = w[co][ci][tap] (cin_pad >= I, cout_pad >= O), bias (O) copied to bias_out[cout_pad] when given;
 *   transposed = 1: the dgrad operator, w flipped spatially with input and output channels swapped:
 *   out[tap][ci][co] = w[ci][co][k*k - 1 - tap] (cin_pad >= O, cout_pad >= I). */
int tdvc_conv2d_pack_weight(const float* w, int O, int I, int k, int transposed, float* out, int cin_pad, int cout_pad,
                            const float* bias_or_null, float* bias_out_or_null, void* stream);
/* GDN / IGDN backward (compressai GDN: out = x * norm^(-1/2), inverse: x * norm^(1/2), norm = beta + gamma . x^2), element-wise
 * parts on flat fp32 arrays (n % 4 == 0): pre -> dx_direct = g * norm^(-+1/2), dnorm = d loss / d norm; the 1x1 convolution's
 * dgrad (tdvc_conv2d on gamma^T) turns dnorm into d(x^2) and tdvc_conv2d_wgrad(in_square = 1) into d gamma / d beta;
 * post -> dx = dx_direct + 2 x d(x^2).  (`in_square` of conv2d_wgrad: x is squared on load.)                             */
int tdvc_gdn_backward_pre(const float* x, const float* norm, const float* grad_out, float* dx_direct, float* dnorm, int64_t n,
                          int inverse, void* stream);
int tdvc_gdn_backward_post(const float* dx_direct, const float* x, const float* dxsq, float* dx, int64_t n, void* stream);
/* Per-(image, channel) pieces of the squeeze-excitation layer in training (reference inflate.py:159-208), dense NHWC rows
 * (C % 4 == 0): chan_affine: out[n][p][c] = a[n][p][c] * s[n][c] + t[n][c] (a NULL: out = s broadcast; t may be NULL) - the
 * gated product, its grad_input, and the backward of the spatial mean; chan_dot: out[n][c] = scale * sum_p a * b (b NULL:
 * plain sums) - the mean and the gate's gradient, two fixed-order stages (deterministic).                                   */
int tdvc_chan_affine(const float* a_or_null, const float* s, const float* t_or_null, float* out, int N, int64_t HW, int C,
                     void* stream);
size_t tdvc_chan_dot_workspace_bytes(int N, int64_t HW, int C);
int tdvc_chan_dot(const float* a, const float* b_or_null, float* out, int N, int64_t HW, int C, float scale, void* workspace,
                  size_t workspace_bytes, void* stream);

/* ---- real entropy coding (`is_compress=True`: reference pnet.py:45-49,69-73 -> compressai `update(force=True)` and
 * `compress()`; compressai is not in the reference tree, SURVEY App. A / DESIGN.md section 7) ----
 * Tables (`update`): pmf_to_quantized_cdf (HOST pointers, host code as in compressai): n probabilities (the last one the
 *   tail mass) -> n + 1 cumulative 16-bit counts; empty bins steal from the smallest bin above 1.
 * Symbols (`compress`):
 *   eb_symbols: z NHWC -> symbols round(z - median) and table indexes (= channel) in NCHW order.
 *   TdvcArChain: the autoregressive chain of compressai's y coding, which ar_code and ar_decode must compute identically.
 *     All pointers are DEVICE pointers.  `params`: the hyper-decoder output, NHWC rows of params_ld >= 2C floats.  Weights
 *     in the fp32 layout of tdvc_conv2d ([tap][cin_pad][cout_pad]): w_ctx the masked 5x5 context model (C -> 2C), w1 / w2
 *     / w3 the entropy-parameter 1x1 layers (4C -> c1 -> c2 -> 2C, LeakyReLU 0.01 between; w1 rows: hyper-decoder output
 *     first, context second).  `scale_table`: the n_scales scales of the Gaussian tables.  Outputs, all NHWC ((h, w, c):
 *     the order compressai codes them in): symbols round(y - mean), table indexes of max(scale, 0.11) and y_hat =
 *     symbol + mean.
 *   ar_code: the autoregressive pass over y of compressai `_compress_ar` as wavefronts inside one launch, one thread-block
 *     cluster per image.  `cluster` = CTAs per image (8; 16 = non-portable size; 0 = 16 where that launches, else 8).
 *     `cluster_used_host` (optional, HOST pointer) receives the size launched: the summation order, and so what a decoder
 *     must reproduce, depends on it.  `workspace`: tdvc_ar_code_workspace_bytes(N, c1_pad, c2_pad) bytes.
 * Coder (HOST pointers, host code: compressai's `ans` extension runs on the CPU too): 64-bit rANS, 16-bit precision, one CDF
 *   row per table index, out-of-range symbols escape through the last bin + a 4-bit bypass code.  encode returns the stream
 *   length in bytes (< 0: error code); decode is its inverse given the same indexes and raises on a truncated or corrupt
 *   stream, an escape whose value does not fit in int32 included.                                                           */
typedef struct TdvcArChain {
  const float* params;   int32_t params_ld;
  const float* w_ctx;    const float* b_ctx;
  const float* w1;       const float* b1;   int32_t c1, c1_pad;
  const float* w2;       const float* b2;   int32_t c2, c2_pad;
  const float* w3;       const float* b3;
  const float* scale_table;  int32_t n_scales;
  float* y_hat;          /* [N][H][W][C] */
  int32_t* symbols;      /* [N][H][W][C] */
  int32_t* indexes;      /* [N][H][W][C] */
  int32_t N, H, W, C;
} TdvcArChain;
typedef struct TdvcArParams {
  TdvcArChain chain;
  const float* y;        int32_t y_ld;
  int32_t cluster;
  int32_t* cluster_used_host;
} TdvcArParams;
/* ar_decode: the inverse of ar_code (compressai `_decompress_ar`), one thread-block cluster per image walking the latent in
 *   raster order: per position the context model over the already decoded y_hat, the three entropy-parameter layers, then
 *   the 128 symbols of the position from the rANS stream (on the device, compressai's bypass escape included), y_hat =
 *   symbol + mean.  The predictions are bit-identical to ar_code's for the same chain only if ar_code ran with `cluster`
 *   CTAs per image (its K splits, and so its fp32 summation order, depend on it): pass the encoder's cluster size (8 or 16;
 *   a container records it).  All pointers are DEVICE pointers.  `words` / `word_offsets`: the N y strings as 32-bit
 *   little-endian words, string n = words[word_offsets[n] .. word_offsets[n + 1]).  `cdfs` [n_tables][cdf_stride],
 *   `cdf_lengths`, `cdf_offsets`: the Gaussian tables of the rANS coder; cdf_total = sum of cdf_lengths.  Outputs those of
 *   the chain plus `status` [N]: -1 when image n decoded, -2 when the CDF tables are not valid rows (lengths outside
 *   [2, cdf_stride] or not summing to cdf_total; nothing is decoded), else the index (h * W + w) * C + c of the first
 *   symbol that could not be decoded (truncated or corrupt stream; nothing after it is written).  A malformed stream never
 *   faults the kernel: the caller reads `status` after the stream synchronises.                                            */
typedef struct TdvcArDecodeParams {
  TdvcArChain chain;
  const uint32_t* words;  const int64_t* word_offsets;
  const int32_t* cdfs;   int32_t cdf_stride;
  const int32_t* cdf_lengths;  const int32_t* cdf_offsets;
  int32_t n_tables, cdf_total;
  int64_t* status;       /* [N] */
  int32_t cluster;
} TdvcArDecodeParams;
int tdvc_pmf_to_quantized_cdf(const float* pmf, int n, int precision, int32_t* cdf);
int tdvc_eb_symbols(const float* z, int ld, const float* medians, int N, int HW, int C, int32_t* symbols, int32_t* indexes,
                    void* stream);
size_t tdvc_ar_code_workspace_bytes(int N, int c1_pad, int c2_pad);
int tdvc_ar_code(const TdvcArParams* p, void* workspace, size_t workspace_bytes, void* stream);
int tdvc_ar_decode(const TdvcArDecodeParams* p, void* stream);
int64_t tdvc_rans_encode_with_indexes(const int32_t* symbols, const int32_t* indexes, int64_t n, const int32_t* cdfs,
                                      int cdf_stride, const int32_t* cdf_lengths, const int32_t* offsets, int n_tables,
                                      uint8_t* out, int64_t capacity);
int tdvc_rans_decode_with_indexes(const uint8_t* data, int64_t nbytes, const int32_t* indexes, int64_t n, const int32_t* cdfs,
                                  int cdf_stride, const int32_t* cdf_lengths, const int32_t* offsets, int n_tables,
                                  int32_t* symbols);

/* ---- reference-based in-loop filter pieces (reference pnet.py:213-257) ----
 * avgpool_scale: nn.AvgPool2d(scale) -> (N, H/scale, W/scale, C)                         (:219-226)
 * ff_descriptors: unfold(3, pad 3, stride 3) + F.normalize -> desc (N, P, C*9), feature c*9 + ky*3 + kx;
 *   PH = (ph + 3)/3 + 1 ... as F.unfold computes; transpose irrelevant                   (:230-236)
 * ff_match: ind[n][q] = first argmax_r <q, r>                                             (:235-238)
 * ff_gather: block placement of f_ref by ind (unfold/gather/fold, :247-254), cor = cosine similarity over
 *   channels (:255), writes a = f_in*cor, b = gathered*cor (the two halves of cat(...)*cor, :257);
 *   optional debug outputs gathered / cor may be NULL.                                                  */
int tdvc_avgpool_scale(const float* x, int ld, float* out, int N, int H, int W, int C, int scale, void* stream);
int tdvc_ff_descriptors(const float* pooled, float* desc, int N, int ph, int pw, int C, void* stream);
int tdvc_ff_match(const float* desc_q, const float* desc_r, int32_t* ind, float* sim_or_null, int N, int P, int D, void* stream);
int tdvc_ff_gather(const float* f_in, const float* f_ref, const int32_t* ind, float* out_a, float* out_b,
                   float* gathered_or_null, float* cor_or_null, int N, int H, int W, int C, int scale, void* stream);

/* ---- on-device metrics for the GOP driver (reference tools/predict.py:86-90): acc[0] += sum (a-b)^2 */
int tdvc_sq_err_sum(const float* a, const float* b, int64_t n, double* acc, void* stream);

/* ---- MS-SSIM (reference main/model/ms_ssim_torch.py:21-87,138-200; tools/predict.py:93-96) ----
 * ssim_level: one scale of `_ssim` on contiguous NCHW planes: separable 11-tap Gaussian (`win11_host`: the 11 window
 *   weights, HOST pointer, copied into the launch), SSIM and contrast-structure maps over the (H-10)x(W-10) valid region;
 *   acc[2*n] += sum of the SSIM map, acc[2*n+1] += sum of the cs map of image n (fp64, caller zeroes them and divides by
 *   C*(H-10)*(W-10)).
 * avgpool2_pad: F.avg_pool2d(x, 2, padding=(H%2, W%2)), the downsampling between scales (:188-190). */
int tdvc_ssim_level(const float* x, const float* y, int N, int C, int H, int W, const float* win11_host, float C1, float C2,
                    double* acc, void* stream);
int tdvc_avgpool2_pad(const float* src, float* dst, int planes, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif
