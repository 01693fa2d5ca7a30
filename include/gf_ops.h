/*
 * gf_ops.h -- C ABI of the memory-bound companions of the attention hot path (SURVEY.md row f3).
 *
 * B200-native equivalents of the reference's two native CUDA ops -- dnnlib/tflib/ops/fused_bias_act.cu and
 * dnnlib/tflib/ops/upfirdn_2d.cu (expected upstream locations; NOT in the reference checkout,
 * /root/reference/.SUBMODULES.json:2) -- restricted to the uses the generator makes of them, plus the
 * activation-scaling form of StyleGAN2's weight (de)modulation.  Channels-last fp32, raw device pointers,
 * enqueue-only on `stream` (a cudaStream_t passed as void*), same error convention as gf_attn.h.
 */
#ifndef GF_OPS_H_
#define GF_OPS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* y[b,t,c] = x[b,t,c] * s[b*s_ld + c].   Style modulation of a conv input / demodulation of a conv output
 * (modulated_conv2d_layer in the reference, activation-scaling form).  y may alias x.  C % 4 == 0; s_ld (row stride
 * of s in floats) % 4 == 0 so that rows of a column slice of a wider [B, sum C] style matrix can be passed directly. */
int gf_chan_scale_nhwc(const float* x, const float* s, int s_ld, float* y, int B, int HW, int C, void* stream);

/* upfirdn_2d, use (a): the FIR blur that follows a stride-2 transposed convolution.
 * x [B, Hout+1, Wout+1, C] -> y [B, Hout, Wout, C]; separable filter [1,3,3,1]/8 per axis, total gain `gain`
 * (4 after an upsampling conv), zero padding 1 on every side; optional per-(b,c) scale (demodulation). C % 4 == 0. */
int gf_blur_up_nhwc(const float* x, float* y, const float* scale, int B, int Hout, int Wout, int C, float gain, void* stream);

/* Use (a) again, with the transposed convolution's output T [B, Hout+1, Wout+1, C] given as its four polyphase components
 * pab[b, i, j, c] = T[b, 2i+a, 2j+b', c] (p00 [B,H+1,W+1,C], p01 [B,H+1,W,C], p10 [B,H,W+1,C], p11 [B,H,W,C]; H = Hout/2,
 * W = Wout/2): the stride-2 transposed 3x3 convolution equals four stride-1 convolutions of the low-resolution input
 * (2x2, 2x1, 1x2 and 1x1 taps), which cuDNN runs 1.3-1.7x faster than its strided dgrad; they are never interleaved. */
int gf_blur_up_phases_nhwc(const float* p00, const float* p01, const float* p10, const float* p11, float* y, const float* scale,
                           int B, int Hout, int Wout, int C, float gain, void* stream);

/* upfirdn_2d, general stride-1 form with the [1,3,3,1]^2/64 filter and symmetric zero padding `pad` in 0..3:
 * x [B,Hin,Win,C] -> y [B,Hin+2*pad-3,Win+2*pad-3,C] times `gain`.  pad 1 = use (a); pad 2 = its adjoint (the backward pass:
 * the filter is symmetric, so d/dx of a pad-p blur is a pad-(3-p) blur of the incoming gradient) and the blur in front of the
 * discriminator's stride-2 3x3 convolutions; pad 1 also serves the discriminator's 1x1 skip path.  C % 4 == 0. */
int gf_fir4_nhwc(const float* x, float* y, int B, int Hin, int Win, int C, int pad, float gain, void* stream);

/* upfirdn_2d, use (b): 2x upsampling of an NCHW image (skip connection of the tRGB outputs):
 * zero-insert, pad (2,1,2,1), FIR [1,3,3,1]^2/64 * 4.  y [B,C,2H,2W] = up(x [B,C,H,W]) (+ add, nullable, same shape as y). */
int gf_upsample2x_nchw(const float* x, const float* add, float* y, int B, int C, int H, int W, void* stream);

/* fused_bias_act (+ the noise input of the synthesis layer):
 *   y = act(x + noise[b*noise_bstride + t] * (*strength) + bias[c]) * gain
 * act: 0 linear, 1 leaky-ReLU(0.2).  noise / strength / bias nullable.  y may alias x.  C % 4 == 0. */
int gf_bias_act_nhwc(const float* x, float* y, const float* bias, const float* noise, const float* strength,
                     long long noise_bstride, int B, int HW, int C, int act, float gain, void* stream);

/* StyleGAN2 demodulation coefficients of the activation-scaling form:
 *   d[b,o] = rsqrt( sum_i styles[b*s_ld + i]^2 * wsq[o,i] + eps ),  wsq[o,i] = sum_{kh,kw} w_eff[o,i,kh,kw]^2 */
int gf_demod_coef(const float* styles, int s_ld, const float* wsq, float* d, int B, int O, int I, float eps, void* stream);

/* The same for every convolution layer of a network in ONE launch (the layers' style vectors all come from one latent, so their
 * demodulation coefficients can be computed up front): n <= GF_DEMOD_MAX_JOBS jobs, common batch B. */
#define GF_DEMOD_MAX_JOBS 32
typedef struct gf_demod_job {
  const float* styles;   /* [B][s_ld], I used */
  const float* wsq;      /* [O][I] */
  float* d;              /* [B][O] out */
  int32_t s_ld, O, I, pad_;
} gf_demod_job;
int gf_demod_coef_batch(const gf_demod_job* jobs, int n, int B, float eps, void* stream);

/* tRGB (SURVEY row f4): 1x1 modulated convolution WITHOUT demodulation from channels-last activations to a planar image,
 *   y[b,o,t] = sum_c x[b,t,c] * w[o*C + c] * styles[b*s_ld + c] * wscale + bias[o],   o < 3
 * (modulated_conv2d_layer(..., demodulate=False, kernel=1) + bias of the reference's torgb); x is read once.
 * C % 4 == 0, C <= 512; s_ld % 4 == 0; bias nullable. */
int gf_torgb_nhwc(const float* x, const float* w, const float* styles, int s_ld, const float* bias, float wscale, float* y,
                  int B, int HW, int C, void* stream);

/* gf_torgb_nhwc with a second output from the same read of x: xs_out[b,t,c] = x[b,t,c] * s2[b*s2_ld + c] -- the style modulation
 * of the NEXT block's first convolution (replaces a gf_chan_scale_nhwc pass over the same tensor).  s2 / xs_out both NULL or both
 * given. */
int gf_torgb_scale_nhwc(const float* x, const float* w, const float* styles, int s_ld, const float* bias, float wscale, float* y,
                        const float* s2, int s2_ld, float* xs_out, int B, int HW, int C, void* stream);

/* G_mapping (SURVEY row f4) as one kernel: z [B, k+1, D] -> out [B, k+1, D].  Every latent is pixel-normalised
 * (x * rsqrt(mean x^2 + 1e-8)), then runs through L fully connected layers with leaky-ReLU(0.2) -- path 0 (shared by the k local
 * components) or path 1 (the last, global latent) -- and, when w_avg [2, D] is given, the truncation lerp
 * out = w_avg[path] + psi * (y - w_avg[path]).  w [2, L, D(in), D(out)] and b [2, L, D] are the EFFECTIVE weights (equalised-LR
 * scale lr_mul/sqrt(D), bias scale lr_mul and the activation gain sqrt(2) folded in: lrelu(g x) = g lrelu(x)).
 * Replaces the reference's G_mapping dense_layer chain.  D <= 128 and 2*L*D*D floats must fit shared memory. */
int gf_mapping_fwd(const float* z, const float* w, const float* b, const float* w_avg, float psi, float* out,
                   int B, int k, int D, int L, void* stream);

/* Row f1, first kernel: the 3x3 stride-1 convolution of the synthesis layers (zero padding 1) as a tcgen05 implicit GEMM in TF32,
 * channels-last: y[b,h,w,o] = sum_{dy,dx,i} x[b,h+dy-1,w+dx-1,i] * wt[dy*3+dx][o][i].  This is the convolution inside the reference's
 * modulated_conv2d_layer in its activation-scaling form (x already carries the style, demodulation is applied by the consumer).
 * wt comes from gf_conv3x3_pack_weights (w [Cout,Cin,3,3] * scale -> [9][Cout][Cin], rounded to TF32).
 * H % 8 == 0, W % 16 == 0, Cin % 32 == 0, Cout % 64 == 0; 16-byte aligned pointers. */
int gf_conv3x3_pack_weights(const float* w, float* wt, int Cout, int Cin, float scale, void* stream);
int gf_conv3x3_nhwc_tf32(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout, void* stream);

/* gf_conv3x3_nhwc_tf32 on a chosen kernel instantiation: version 1 (one activation box per tap) or 2 (one box per filter column),
 * bn = output channels per tile (64 / 128 / 256), mt = 8 x 16 patches stacked per tile (1 or 2); the accumulator count follows
 * (one set for bn 256, mt 2, else two).  (0, 0, 0) = the shape dispatch of gf_conv3x3_nhwc_tf32, GF_CONV_* overrides included.
 * Any other triple must be one of the twelve, with Cout % bn == 0 and H % (8 mt) == 0, else GF_ERR_UNSUPPORTED before any device
 * work.  All instantiations of one version sum in the same order, so they give bit-identical results. */
int gf_conv3x3_nhwc_tf32_ex(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout,
                            int version, int bn, int mt, void* stream);
/* (version, bn, mt) of the kernel the last gf_conv3x3_nhwc_tf32[_ex] call on this host thread launched; zeros if that call failed. */
int gf_conv3x3_last_variant(int* version, int* bn, int* mt);

#ifdef __cplusplus
}
#endif
#endif /* GF_OPS_H_ */
