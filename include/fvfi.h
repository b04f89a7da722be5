/*
 * fvfi.h -- C-ABI of libfvfi.so: the B200-native (sm_100a) frame-synthesis hot path of
 * stefan01/Fusion-Method-for-Video-Frame-Interpolation.
 *
 * Drop-in boundary (SURVEY.md 8(b)).  Every entry point replaces one call the reference
 * makes today from Python into CuPy/NVRTC kernels, torch elementwise chains or the absent
 * third-party `steerable` package.  The citation on each function is the reference
 * interface it replaces (paths relative to the reference root).
 *
 * Conventions (same as the reference's CuPy launches, src/adacof/cupy_module/adacof.py:337-354):
 *   - all tensor pointers are DEVICE pointers to contiguous fp32 NCHW storage that the
 *     CALLER allocated (torch's caching allocator stays in charge); the library never
 *     allocates user-visible tensors.  `*_host` variants take HOST pointers and do the
 *     host<->device copies themselves (used for the end-to-end measurement).
 *   - `stream` is a cudaStream_t / CUstream passed as void* (torch.cuda.current_stream().cuda_stream);
 *     nothing synchronises the host except the `*_host` variants.
 *   - return 0 on success; non-zero = error, text in fvfi_last_error() (thread-local).
 *     The Python mirror raises (AssertionError / RuntimeError) like the reference does.
 *   - re-entrant; no global mutable state except immutable plans.
 */
#ifndef FVFI_H
#define FVFI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    FVFI_OK = 0,
    FVFI_EINVAL = 1, /* bad shape / argument (the reference's Python asserts, adacof.py:326-332) */
    FVFI_ECUDA = 2,  /* CUDA runtime error */
    FVFI_ENOMEM = 3
};

/* operand split of fvfi_conv2d_* */
enum { FVFI_CONV_TF32X3 = 0, FVFI_CONV_F16X3 = 1 };

/* gradInput modes of fvfi_adacof_backward */
enum {
    FVFI_GIN_NONE = 0,  /* gin pointer ignored */
    FVFI_GIN_ZEROS = 1, /* reference semantics: gradInput = zeros (adacof.py:382,445) */
    FVFI_GIN_TRUE = 2   /* extension: true adjoint.  Default adacof_grad_input_tile: every CTA accumulates its 64x16 output pixels in a
                           shared-memory image of the reachable frame region, one global red.add per touched sample; large F*dilation or
                           FVFI_GIN_SCATTER=warp: adacof_grad_input_scatter groups the lanes of a warp by target address
                           (__match_any_sync) and issues one red.add per distinct address */
};

int fvfi_version(void);
const char* fvfi_last_error(void);
/* Device properties the library was built for / sees: returns SM count of the current device, or -1. */
int fvfi_device_sm_count(void);
/* Number of CUDA kernels this library has launched in the calling process (evidence for bench.py's gpu_launches). */
unsigned long long fvfi_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * AdaCoF warp.  Replaces FunctionAdaCoF.forward + kernel_AdaCoF_updateOutput
 * (src/adacof/cupy_module/adacof.py:313-361, :6-65).
 *   input  [B,C,Hin,Win]   weight/off_i/off_j [B,F*F,H,W]   output [B,C,H,W]
 *   requires Hin == H + (F-1)*dilation, Win == W + (F-1)*dilation  (adacof.py:326-327)
 * algo: 0 = auto, 1 = direct (global gathers), 2 = tiled (smem-staged frame tile, register-prefetched coefficients),
 *       3 = TMA (persistent CTAs, coefficient planes streamed by cp.async.bulk.tensor; F = 5, dilation 1, W % 4 == 0)
 */
int fvfi_adacof_forward(const float* input, const float* weight, const float* off_i, const float* off_j,
                        float* output, int B, int C, int Hin, int Win, int H, int W, int F, int dilation,
                        int algo, void* stream);

/* Replaces FunctionAdaCoF.backward + kernel_AdaCoF_updateGradWeight/-Alpha/-Beta
 * (adacof.py:364-445, :67-258) with ONE fused kernel.  C must be 3 (the reference hard-codes
 * three channels, adacof.py:86,150,215; algo as in fvfi_adacof_forward).  gw/goi/goj [B,F*F,H,W] are fully overwritten
 * (no pre-zeroing needed).  gin [B,C,Hin,Win] per gin_mode. */
int fvfi_adacof_backward(const float* gout, const float* input, const float* weight, const float* off_i,
                         const float* off_j, float* gin, float* gw, float* goi, float* goj, int B, int C,
                         int Hin, int Win, int H, int W, int F, int dilation, int gin_mode, int algo,
                         void* stream);

/* Occlusion blend + flow-variance uncertainty mask of AdaCoFNet.forward
 * (src/fusion_net/fusion_adacofnet.py:198-213), one pass over the six coefficient maps.
 *   t1,t2,frame [B,C,H,W]  occ,mask [B,1,H,W]  w*,a*,b* [B,FF,H,W]; frame/mask may be NULL. */
int fvfi_adacofnet_tail(const float* t1, const float* t2, const float* occ, const float* w1, const float* a1,
                        const float* b1, const float* w2, const float* a2, const float* b2, float* frame,
                        float* mask, int B, int C, int H, int W, int FF, void* stream);

/* Both warps of AdaCoFNet.forward + blend + uncertainty mask in ONE kernel
 * (fusion_adacofnet.py:195-213): each coefficient map is read from HBM once.
 *   in1,in2 [B,3,Hin,Win] (replicate-padded frames)  t1,t2,frame [B,3,H,W]  occ,mask [B,1,H,W] */
int fvfi_adacofnet_warp_blend(const float* in1, const float* in2, const float* w1, const float* a1,
                              const float* b1, const float* w2, const float* a2, const float* b2,
                              const float* occ, float* t1, float* t2, float* frame, float* mask, int B,
                              int Hin, int Win, int H, int W, int F, int dilation, void* stream);

/* Same synthesis for frames that were reflect-padded at the bottom to a multiple of 32 rows (fusion_adacofnet.py:179-188, 214-226: the
 * reference crops the result back): frame [B,3,out_rows,W] and mask [B,1,out_rows,W] (mask may be NULL) receive only the first out_rows
 * rows, so the crop copies never happen; no warped frames are returned.  Needs the TMA-streamed kernel (F = 5, dilation 1, W % 4 == 0,
 * 16-byte aligned coefficient maps), FVFI_EINVAL otherwise. */
int fvfi_adacofnet_warp_blend_rows(const float* in1, const float* in2, const float* w1, const float* a1, const float* b1,
                                   const float* w2, const float* a2, const float* b2, const float* occ, float* frame, float* mask,
                                   int out_rows, int B, int Hin, int Win, int H, int W, int F, int dilation, void* stream);

/* FusionNet's last step (src/fusion_net/fusion_net.py:67-77): out = clamp(base + tanh(x), 0, 1). */
int fvfi_fusion_blend(const float* base, const float* x_pre_tanh, float* out, size_t n, void* stream);
/* The same blend for 8-bit output: base / x_pre_tanh [B,3,H,W] planar -> out [B,H,W,3] uint8 interleaved (rgb24),
 * out = rint(clamp(base + tanh(x), 0, 1) * 255) with ties to even.  The fp32 frame is never written. */
int fvfi_fusion_blend_rgb8(const float* base, const float* x_pre_tanh, uint8_t* out, int B, int H, int W, void* stream);

/* ---------------------------------------------------------------------------------------
 * Per-pixel stages the reference runs on the host CPU (SURVEY.md 8(f) f1/f2), device-resident here.
 * rgb/lab [B,3,H,W] planar.  Replaces rgb2lab / lab2rgb (src/train/transform.py:6-49: skimage.color,
 * then L/100 and (a,b+128)/255). */
int fvfi_rgb2lab(const float* rgb, float* lab, int B, int H, int W, void* stream);
int fvfi_lab2rgb(const float* lab, float* rgb, int B, int H, int W, void* stream);
/* Decoder frames rgb8 [T,H,W,3] uint8 interleaved (ffmpeg -pix_fmt rgb24) -> rgb [T,3,H,W] planar fp32 (the correctly rounded
 * k / 255) and lab [T,3,H,W] planar scaled Lab, in one pass; lab is bit-identical to fvfi_rgb2lab of rgb. */
int fvfi_rgb8_to_rgb_lab(const uint8_t* rgb8, float* rgb, float* lab, int T, int H, int W, void* stream);
/* scipy.ndimage.gaussian_filter(x, sigma) on N maps [N,H,W] (truncate 4, mode 'reflect';
 * src/fusion_net/interpolate_twoframe.py:212-213).  tmp: scratch of the same size. */
int fvfi_gaussian_filter(const float* in, float* out, float* tmp, int N, int H, int W, float sigma, void* stream);
/* scipy.ndimage.median_filter(x, size=size) on N maps (rank size*size/2, mode 'reflect';
 * interpolate_twoframe.py:221-222).  Exact. */
int fvfi_median_filter(const float* in, float* out, int N, int H, int W, int size, void* stream);

/* ---------------------------------------------------------------------------------------
 * Convolution on the tcgen05 tensor cores (split-operand error-compensated, fp32 in/out), NHWC activations.
 * precision: FVFI_CONV_F16X3 (default of the Python mirror: three kind::f16 products of fp16 hi/lo halves, 22 mantissa
 * bits, twice the TF32 rate) or FVFI_CONV_TF32X3 (three kind::tf32 products, no range limit).  Packed weights are
 * specific to the precision they were packed for.
 * Replaces torch.nn.Conv2d -> cuDNN for the stride-1 "same" convolutions of PhaseNetBlock
 * (src/phase_net/phase_net.py:190-199), KernelEstimation (src/fusion_net/fusion_adacofnet.py:19-83) and
 * FusionNet (src/fusion_net/fusion_net.py:24-36).
 *   weight_oihw [Cout,Cin,KH,KW] -> packed (fvfi_conv2d_packed_weight_floats floats), once per weight update.
 *   x: NHWC, x_pixel_stride floats between pixels (>= Cin); y likewise.  Cout <= 256 per call.
 *   KH == KW in {1,3,5}; pad_mode 0 = zeros, 1 = reflect (torch 'reflect'); activation 0 none, 1 ReLU, 2 ELU,
 *   3 tanh, 4 sigmoid, 5 softmax over the Cout channels; bias [Cout] or NULL.
 *   out_nchw: 0 = NHWC; 1 = planar [B,Cout,H,W] (the layout the AdaCoF warp streams its coefficient maps in);
 *   2 = NHWC with round16(Cout) channels written per pixel, the padding zero-filled (so that a consumer with a channel
 *   count that is not a multiple of 4 can still use 16-byte loads: x_pixel_stride >= roundup4(Cin) enables them). */
size_t fvfi_conv2d_packed_weight_floats(int Cout, int Cin, int KH, int KW, int precision);
int fvfi_conv2d_pack_weights(const float* weight_oihw, float* packed, int Cout, int Cin, int KH, int KW, int precision,
                             void* stream);
int fvfi_conv2d_nhwc(const float* x, int x_pixel_stride, const float* packed_weight, const float* bias, float* y,
                     int y_pixel_stride, int B, int H, int W, int Cin, int Cout, int KH, int KW, int pad_mode,
                     int activation, int out_nchw, int precision, void* stream);
/* Same with a skip connection fused into the epilogue:  y = act(conv(x) + bias) + residual,  residual [B,H,W,>=Cout] NHWC with
 * residual_pixel_stride floats per pixel (KernelEstimation's decoder, src/fusion_net/fusion_adacofnet.py:128-138: d5 + c5, ...);
 * residual == NULL is fvfi_conv2d_nhwc.  Not with the softmax activation. */
int fvfi_conv2d_nhwc_residual(const float* x, int x_pixel_stride, const float* packed_weight, const float* bias,
                              const float* residual, int residual_pixel_stride, float* y, int y_pixel_stride, int B, int H,
                              int W, int Cin, int Cout, int KH, int KW, int pad_mode, int activation, int out_nchw,
                              int precision, void* stream);
/* torch.nn.Upsample(mode='bilinear') -> Conv2d as ONE kernel (KernelEstimation's Upsample blocks and the tails of its heads,
 * src/fusion_net/fusion_adacofnet.py:29-36,41-48: `Upsample(scale_factor=2, mode='bilinear', align_corners=True)` followed by a
 * 3x3 convolution):  y = act(conv(resize(x, [H,W])) + bias) + residual.  x is the SOURCE [B,Hs,Ws,>=Cin] NHWC; the loaders of the
 * convolution evaluate the bilinear resampling (ATen's upsample_bilinear2d arithmetic, the same as fvfi_resize_bilinear_nhwc)
 * while they stage the operand, so the [B,H,W,Cin] intermediate never exists in HBM.  x must be 32-byte aligned (FVFI_CONV_TF32X3: 16)
 * with x_pixel_stride a multiple of 8 (4) that covers Cin rounded up to it; channels between Cin and that bound must be finite.
 * Hs == Ws == 0 is fvfi_conv2d_nhwc_residual.
 * Two-source form (x_direct != NULL):  conv(cat(resize(x[:, :cin_upsampled]), x_direct), ...) without the concatenated tensor --
 * PhaseNet's level input `cat(values, interpolate(previous features), interpolate(previous prediction))` (src/phase_net/phase_net.py:
 * 138-148): the first cin_upsampled input channels (a multiple of 32; FVFI_CONV_TF32X3: 16) are the resampled x, the remaining
 * Cin - cin_upsampled come from x_direct [B,H,W,x_direct_pixel_stride] at the convolution's own resolution. */
int fvfi_conv2d_nhwc_upsampled(const float* x, int x_pixel_stride, int Hs, int Ws, int align_corners, const float* x_direct,
                               int x_direct_pixel_stride, int cin_upsampled, const float* packed_weight, const float* bias, const float* residual, int residual_pixel_stride,
                               float* y, int y_pixel_stride, int B, int H, int W, int Cin, int Cout, int KH, int KW, int pad_mode,
                               int activation, int out_nchw, int precision, void* stream);
/* FVFI_CONV_F16X3 scales activations by 2^4 before the fp16 split; |x| > 4094 would leave fp16's range.  Returns 1
 * (and clears the flag) if any convolution since the last call saw such a value, 0 if not, -1 on error.
 * Synchronises the device. */
int fvfi_conv2d_overflow_count(void);

/* ---------------------------------------------------------------------------------------
 * Backward of the same convolutions, for the FusionNet training step (src/fusion_net/trainer.py:246-259; the reference takes
 * these gradients from torch.nn.Conv2d's cuDNN autograd for the layers of src/fusion_net/fusion_net.py:24-36).
 * With y = act(conv(pad(x), w) + b) and g = dL/dy * act'(y):
 *   fvfi_conv2d_grad_act: g written into the interior of a zero canvas g_canvas [B, H+2*border, W+2*border, C] (contiguous NHWC;
 *     border = 0: plain g) from gy and the SAVED OUTPUT y (activation 0 none -- y may be NULL --, 1 ReLU, 2 ELU, 3 tanh, 4 sigmoid),
 *     and, if gbias != NULL, the bias gradient gbias[C] = sum over pixels of g (fixed summation order).  workspace:
 *     fvfi_conv2d_grad_act_workspace_floats floats (only needed with gbias).
 *   data gradient: dL/d(pad x) = fvfi_conv2d_nhwc(g_canvas with border K/2, weights [Cin,Cout,K,K] = w[o,c,K-1-ky,K-1-kx], zero
 *     padding, FVFI_CONV_TF32X3 -- gradients have no bounded range) on [B, H+2*(K/2), W+2*(K/2)]; for pad_mode zeros the interior
 *     of that result is dL/dx, for reflect padding fvfi_reflect_pad_backward_nhwc folds the mirrored border back
 *     (the adjoint of torch's 'reflect' padding; gx [B,H,W,C], H, W > P).
 *   fvfi_conv2d_wgrad_nhwc: gw_oihw [Cout,Cin,K,K] = sum_{b,y,x} g[b,y,x,o] * pad(x)[b,y+ky,x+kx,c].  g may live inside a canvas:
 *     pixel (b,y,x) at ((b * g_image_pixels + y * g_row_pixels + x) * g_pixel_stride.  Split over pixel ranges into partial sums
 *     (workspace: fvfi_conv2d_wgrad_workspace_floats floats) that are added in a fixed order: bit-reproducible. */
size_t fvfi_conv2d_grad_act_workspace_floats(int B, int H, int W, int C, int border);
int fvfi_conv2d_grad_act(const float* gy, int gy_pixel_stride, const float* y, int y_pixel_stride, float* g_canvas, int B, int H,
                         int W, int C, int border, int activation, float* gbias, float* workspace, void* stream);
int fvfi_reflect_pad_backward_nhwc(const float* gxp, int gxp_pixel_stride, float* gx, int gx_pixel_stride, int B, int H, int W, int C,
                                   int P, void* stream);
size_t fvfi_conv2d_wgrad_workspace_floats(int B, int H, int W, int Cin, int Cout, int K);
int fvfi_conv2d_wgrad_nhwc(const float* x, int x_pixel_stride, const float* g, int g_pixel_stride, long long g_row_pixels,
                           long long g_image_pixels, float* gw_oihw, int B, int H, int W, int Cin, int Cout, int K, int pad_mode,
                           float* workspace, void* stream);

/* The other differentiable steps of FusionNet's training forward (src/fusion_net/fusion_net.py:52-77; the reference differentiates
 * nn.MaxPool2d, nn.Upsample and tanh / clamp through torch autograd):
 *   fvfi_max_pool2_backward_nhwc: gx [B,Hi,Wi,C] from gy [B,Hi/2,Wi/2,C] and the forward input x; the gradient of a window goes to its
 *     first maximum in scan order (ATen's rule); an odd last row / column gets zero.
 *   fvfi_resize_bilinear_backward_nhwc: adjoint of fvfi_resize_bilinear_nhwc_fused (upsampling by at most 3 per axis): gx [B,Hi,Wi,C]
 *     from gy [B,Ho,Wo,C]; relu_input: the forward resampled max(x, 0), so gx is zero where x <= 0 (x = the forward input).  The
 *     addend of the fused forward receives gy unchanged.
 *   fvfi_fusion_blend_backward: out = clamp(base + tanh(x), 0, 1) -> gx = gout * [0 < out < 1] * (1 - tanh(x)^2), gbase (or NULL) =
 *     gout * [0 < out < 1]; n elements. */
int fvfi_max_pool2_backward_nhwc(const float* x, int x_pixel_stride, const float* gy, int gy_pixel_stride, float* gx, int gx_pixel_stride,
                                 int B, int Hi, int Wi, int C, void* stream);
/* nn.AvgPool2d(2, 2) backward (KernelEstimation's encoder, src/fusion_net/fusion_adacofnet.py:62-70, under autograd): every pixel of a
 * window receives gy / 4. */
int fvfi_avg_pool2_backward_nhwc(const float* gy, int gy_pixel_stride, float* gx, int gx_pixel_stride, int B, int Hi, int Wi, int C,
                                 void* stream);
int fvfi_resize_bilinear_backward_nhwc(const float* gy, int gy_pixel_stride, const float* x, int x_pixel_stride, float* gx,
                                       int gx_pixel_stride, int B, int Hi, int Wi, int Ho, int Wo, int C, int align_corners,
                                       int relu_input, void* stream);
int fvfi_fusion_blend_backward(const float* base, const float* x, const float* gout, float* gx, float* gbase, size_t n, void* stream);

/* Direct (CUDA-core, fp32 FFMA) 1x1 convolution for Cout <= 8 -- the layers that are a pure stream of the activation:
 * PhaseNet's per-level prediction Conv2d(64, 8, 1) + tanh (src/phase_net/phase_net.py:197-200) and FusionNet's last
 * Conv2d(32, 3, 1) (src/fusion_net/fusion_net.py:36).  x [npix, x_pixel_stride] NHWC pixels (32-byte aligned, Cin a multiple
 * of 8, <= 128), weight [Cout, Cin] (the OIHW tensor of a 1x1 convolution), bias [Cout] or NULL, y [npix, y_pixel_stride].
 * activation: 0 none, 1 ReLU, 2 ELU, 3 tanh, 4 sigmoid. */
int fvfi_conv1x1_nhwc(const float* x, int x_pixel_stride, const float* weight, const float* bias, float* y,
                      int y_pixel_stride, size_t npix, int Cin, int Cout, int activation, void* stream);

/* Tail of KernelEstimation's occlusion head, Upsample(x2, bilinear, align_corners=True) -> Conv2d(C, 1, 3, padding 1) ->
 * Sigmoid (src/fusion_net/fusion_adacofnet.py:50-59, 103-104), with the channel contraction done first at half resolution:
 * z [B,Hi,Wi,z_pixel_stride] (or, with z_pixel_stride == 0, planar [B,9,Hi,Wi]) holds the nine tap maps z_t = sum_c w[0,c,t] x_c (t = ky*3 + kx; a 1x1
 * convolution C -> 9 of the half-resolution feature), and  y[b,i,j] = act(bias[0] + sum_t [p_t inside] bilinear(z_t)(p_t)),
 * p_t = (i + ky - 1, j + kx - 1), y [B, 2*Hi, 2*Wi].  Same real-number result as the reference's order of operations. */
int fvfi_upsample2_tapsum(const float* z, int z_pixel_stride, const float* bias, float* y, int B, int Hi, int Wi,
                          int activation, void* stream);

/* Input preparation of AdaCoFNet.forward in one pass (src/fusion_net/fusion_adacofnet.py:176-196, src/adacof/utility.py:86-87):
 * frames [B,3,H,W] -> x_nhwc8 [B,Hp,Wp,8] = (frame0 - mean | frame2 - mean | 0 0) of the frames reflect-padded at the bottom /
 * right to Hp x Wp (multiples of 32), KernelEstimation's NHWC input; padded0 / padded2 [B,3,Hp+2k,Wp+2k] = ReplicationPad2d(k)
 * of the reflect-padded frames, what the warp samples.  mean3_host: three floats on the HOST (the channel means). */
int fvfi_adacofnet_prep(const float* frame0, const float* frame2, float* x_nhwc8, float* padded0, float* padded2, int B,
                        int H, int W, int Hp, int Wp, int kpad, const float* mean3_host, void* stream);

/* PhaseNet glue, fused (src/train/utils.py:47-127 separate_vals / get_concat_layers_inf, src/phase_net/phase_net.py:42-78
 * normalize_vals, :141 concat, :155-156 amplitude blend, :80-105 reverse_normalize).
 * phase / amp: one level of fvfi_pyr_decompose of [frame-1 planes | frame-2 planes]: [2*P*nb, H, W], channel = plane*nb + band.
 * fvfi_phasenet_assemble writes, for planes [p0, p0+pc), the 4*nb value channels of the NHWC concat
 *   y[p - p0][h][w][0 .. 4nb) = [phase_1 / pi | phase_2 / pi | amp_1 / den[p] | amp_2 / den[p]]   (den [P]: per-plane max + eps).
 * fvfi_phasenet_outputs takes the block's prediction pred [pc,H,W,>=2nb] (NHWC, tanh outputs) and writes
 *   phase_out[(p*nb + b)] = pred[b] * pi,  amp_out[(p*nb + b)] = beta * amp_2 + (1 - beta) * amp_1,  beta = (pred[nb + b] + 1) / 2
 * into [P*nb, H, W] tensors (the un-normalised values Pyramid.inv_filter consumes).  nb must be 4. */
int fvfi_phasenet_assemble(const float* phase, const float* amp, const float* den, float* y, int y_pixel_stride, int P,
                           int p0, int pc, int nb, int H, int W, void* stream);
int fvfi_phasenet_outputs(const float* pred, int pred_pixel_stride, const float* amp, float* phase_out, float* amp_out,
                          int P, int p0, int pc, int nb, int H, int W, void* stream);
/* The same two steps for any plane layout: phase / amp hold N planes and frame 2 of pair-plane p is plane p + q (the two entry
 * points above are q = P, N = 2P).  A clip of T' consecutive frames decomposed once is q = 3, P = N - 3: pair t reads frames t and
 * t + 1.  FVFI_EINVAL if p0 + pc - 1 + q >= N. */
int fvfi_phasenet_assemble_offset(const float* phase, const float* amp, const float* den, float* y, int y_pixel_stride, int N, int P,
                                  int q, int p0, int pc, int nb, int H, int W, void* stream);
int fvfi_phasenet_outputs_offset(const float* pred, int pred_pixel_stride, const float* amp, float* phase_out, float* amp_out, int N,
                                 int P, int q, int p0, int pc, int nb, int H, int W, void* stream);

/* Bilinear resize of NHWC tensors (torch.nn.Upsample / F.interpolate 'bilinear' semantics, both align_corners
 * modes; src/fusion_net/fusion_adacofnet.py:31, src/fusion_net/fusion_net.py:41, src/phase_net/phase_net.py:138-139).
 * x [B,Hi,Wi,C] with x_pixel_stride floats per pixel -> y [B,Ho,Wo,C] (may be a channel slice: y_pixel_stride). */
int fvfi_resize_bilinear_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi,
                              int Ho, int Wo, int C, int align_corners, void* stream);
/* The decoder step of FusionNet in one pass (src/fusion_net/fusion_net.py:60-62: x = Upsample(ReLU(x)); x = x + skip):
 * y = resize(relu_input ? max(x, 0) : x) + addend (addend [B,Ho,Wo,C] NHWC with its own pixel stride, or NULL). */
int fvfi_resize_bilinear_nhwc_fused(const float* x, int x_pixel_stride, const float* addend, int addend_pixel_stride, float* y,
                                    int y_pixel_stride, int B, int Hi, int Wi, int Ho, int Wo, int C, int align_corners,
                                    int relu_input, void* stream);

/* nn.AvgPool2d(kernel_size=2, stride=2) on NHWC tensors (KernelEstimation's encoder, src/fusion_net/fusion_adacofnet.py:62-70,
 * 111-123): x [B,Hi,Wi,C] -> y [B,Hi/2,Wi/2,C]. */
int fvfi_avg_pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C,
                        void* stream);
/* nn.MaxPool2d(2, stride=2) on NHWC tensors (FusionNet's encoder, src/fusion_net/fusion_net.py:39,56-60), same layout contract. */
int fvfi_max_pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C,
                        void* stream);

/* Planar [B,C,H,W] -> channels [0,C) of an NHWC buffer whose pixels are y_pixel_stride floats apart (pass y + offset for a
 * channel slice): PhaseNet's concat of phase / amplitude planes with NHWC features (src/phase_net/phase_net.py:141). */
int fvfi_nchw_to_nhwc_slice(const float* x, float* y, int y_pixel_stride, int B, int C, int H, int W, void* stream);

/* torch.cat(sources, dim=1) of planar tensors [B,channels[s],H,W] written as ONE NHWC tensor y [B,H,W,y_pixel_stride] (FusionNet's
 * input, src/fusion_net/fusion_net.py:47: cat([base, adacof, phase, other, maps], 1), which the tensor-core convolution wants NHWC): the
 * concatenated planar tensor and its transposing copy never exist.  sources / channels: HOST arrays of nsources device pointers / channel
 * counts (at most 32 channels in total); channels between the total and its multiple of 4 are written as zeros; y_pixel_stride a multiple
 * of 4 that covers them, y 16-byte aligned. */
int fvfi_planar_concat_nhwc(const float* const* sources, const int* channels, int nsources, float* y, int y_pixel_stride, int B, int H,
                            int W, void* stream);

/* Host-buffer variants for end-to-end timing: pointers are HOST memory (pinned preferred);
 * the call does H2D, the kernel(s), D2H and synchronises. */
int fvfi_adacof_forward_host(const float* input, const float* weight, const float* off_i, const float* off_j,
                             float* output, int B, int C, int Hin, int Win, int H, int W, int F, int dilation);
int fvfi_adacof_backward_host(const float* gout, const float* input, const float* weight, const float* off_i,
                              const float* off_j, float* gw, float* goi, float* goj, int B, int C, int Hin,
                              int Win, int H, int W, int F, int dilation);

/* ---------------------------------------------------------------------------------------
 * Complex steerable pyramid.  Replaces steerable.SCFpyr_PyTorch.build / .reconstruct (third
 * party, absent; call sites src/train/pyramid.py:28-33,37,44) fused with
 * Pyramid.coeff_to_values / values_to_coeff (src/train/pyramid.py:48-112).
 * A plan owns the immutable device tables (level sizes, FFT factorizations, twiddles).
 */
typedef struct fvfi_pyr_plan fvfi_pyr_plan;

int fvfi_pyr_plan_create(int H, int W, int height, int nbands, double scale_factor, fvfi_pyr_plan** out);
void fvfi_pyr_plan_destroy(fvfi_pyr_plan* plan);
int fvfi_pyr_num_levels(const fvfi_pyr_plan* plan); /* height - 2 */
/* level 0..L-1 = band levels (finest first); level L = low-pass residual */
int fvfi_pyr_level_shape(const fvfi_pyr_plan* plan, int level, int* h, int* w);
/* Level-size rule shared with the oracle: n_next = ceil((n - 0.5) / s)  (SURVEY.md F2, Appendix A.4). */
int fvfi_pyr_next_size(int n, double scale_factor);
size_t fvfi_pyr_workspace_bytes(const fvfi_pyr_plan* plan, int N);

/* Decompose N planes.  img [N,H,W] -> high [N,1,H,W], phase[l]/amp[l] [N*nb,1,h_l,w_l] (channel
 * = plane*nb + band, src/train/pyramid.py:64-66), low [N,1,h_L,w_L].  amp_max (optional,
 * [L,N] per-level per-plane max amplitude over the nb bands) feeds PhaseNet.normalize_vals
 * (src/phase_net/phase_net.py:42-78).  high may be NULL (skipped). */
int fvfi_pyr_decompose(const fvfi_pyr_plan* plan, const float* img, int N, float* high, float* const* phase,
                       float* const* amp, float* low, float* amp_max, void* workspace, void* stream);

/* Reconstruct N planes from (high, phase, amp, low).  phase[l]/amp[l] may be NULL for a level
 * that contributes nothing (the reference passes the int 0, src/phase_net/phase_net.py:91-93;
 * get_last/first_value_levels zero-fill, src/train/utils.py:242-320); high/low may be NULL (zeros). */
int fvfi_pyr_reconstruct(const fvfi_pyr_plan* plan, const float* high, const float* const* phase,
                         const float* const* amp, const float* low, int N, float* img, void* workspace,
                         void* stream);

/* Backward of fvfi_pyr_reconstruct for PhaseNet training (src/train/trainer.py:139-147 back-propagates the L1 image loss through
 * Pyramid.inv_filter): grad_img [N,H,W] -> gradients w.r.t. high [N,1,H,W], phase[l] / amp[l] [N*nb,1,h_l,w_l] and low.  A level
 * whose grad_phase[l] / grad_amp[l] is NULL is skipped; grad_high / grad_low may be NULL.  phase / amp are the forward's inputs. */
int fvfi_pyr_reconstruct_backward(const fvfi_pyr_plan* plan, const float* grad_img, int N, const float* const* phase,
                                  const float* const* amp, float* grad_high, float* const* grad_phase,
                                  float* const* grad_amp, float* grad_low, void* workspace, void* stream);

/* out[N,H,W] = inv_filter(get_last_value_levels(filter(img), 1)) -- the high residual plus the finest band level of img, put back
 * together (src/train/utils.py:242-280 with use_levels = 1; the h_freq maps of src/fusion_net/interpolate_twoframe.py:205-209).
 * Decomposition and reconstruction are linear and nothing touches the coefficients in between, so this is ONE multiplication of
 * the image spectrum by a real transfer function tabulated in the plan: 2 two-dimensional FFTs instead of 10. */
int fvfi_pyr_highband_filter(const fvfi_pyr_plan* plan, const float* img, int N, float* out, void* workspace, void* stream);

/* Complex coefficient interface (the SCFpyr_PyTorch.build/reconstruct layout, band tensors
 * [N,h_l,w_l,2], src/train/pyramid.py:58): bands[l*nb + b]. */
int fvfi_pyr_build_complex(const fvfi_pyr_plan* plan, const float* img, int N, float* high,
                           float* const* bands, float* low, void* workspace, void* stream);
int fvfi_pyr_reconstruct_complex(const fvfi_pyr_plan* plan, const float* high, const float* const* bands,
                                 const float* low, int N, float* img, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FVFI_H */
