/*
 * sae_b200.h — C ABI of the B200-native Swapping-Autoencoder conv hot path.
 *
 * Every entry point takes raw DEVICE pointers to fp32 data, explicit sizes and a
 * cudaStream_t (passed as void*); nothing is allocated inside, nothing depends on
 * torch.  Return value: 0 on success, a negative SAE_E_* code otherwise;
 * sae_last_error() returns a thread-local human-readable message for the last
 * failure.  All entry points are re-entrant (no global mutable state apart from a
 * per-device attribute cache guarded by std::call_once).
 *
 * Activation layout: NHWC ("[major, H, W, minor]" in the reference's own native
 * signature, reference/models/networks/stylegan2_op/upfirdn2d.cpp:12-23, called
 * here with major = batch, minor = channels instead of major = B*C, minor = 1).
 * Weight layout for the conv entry points: [Cout, R, S, Cin] ("KRSC").
 *
 * Each declaration cites the reference interface it replaces (paths relative to
 * the reference checkout, taesungp/swapping-autoencoder-pytorch @ 6baa180).
 */
#ifndef SAE_B200_H_
#define SAE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAE_OK              0
#define SAE_E_INVALID      -1   /* bad argument (shape / alignment / unsupported combination) */
#define SAE_E_CUDA         -2   /* a CUDA runtime / driver call or the launch itself failed */
#define SAE_E_UNSUPPORTED  -3   /* valid request this build has no kernel for                */

/* ABI version of this header; bumped on any signature change. */
#define SAE_ABI_VERSION 14
int         sae_abi_version(void);
const char* sae_last_error(void);
/* number of kernels launched by this library in the calling process since load
 * (monotonic, relaxed atomic) — bench.py reports the delta as "gpu_launches". */
int64_t     sae_launch_count(void);
/* 1 when the tcgen05/TMA conv path is usable on the current device (sm_100 + driver entry points) */
int         sae_tcgen05_available(void);

/* ------------------------------------------------------------------------------------------
 * upfirdn2d — zero-insert upsample, pad / crop, 2-D FIR (true convolution: taps read flipped),
 * decimate.  Replaces  upfirdn2d_op.upfirdn2d(input[major,H,W,minor], kernel[kh,kw], up_x, up_y,
 * down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1)
 *   (models/networks/stylegan2_op/upfirdn2d.cpp:12-23, upfirdn2d_kernel.cu:140-271).
 * out is [major, out_h, out_w, minor] with out_h = (in_h*up_y + pad_y0 + pad_y1 - kh)/down_y + 1
 * (upfirdn2d.py:108-109).  Unlike the reference there is no mode table: every
 * (up, down, kh, kw <= 32) combination is handled by the same kernel.  Negative pads crop.
 * 64-bit indexing throughout (the reference overflows int32 at >= 2^31 elements).
 * round_tf32 (here and below): when non-zero the result is rounded to the nearest TF32 value before it is stored
 * (still an fp32 array).  The tensor-core convolutions read operands at TF32 precision by IGNORING the low 13
 * mantissa bits; rounding-to-nearest in the producer makes that truncation exact and unbiased.
 * ------------------------------------------------------------------------------------------ */
int sae_upfirdn2d(const float* input, const float* kernel, float* out,
                  int64_t major, int in_h, int in_w, int minor,
                  int kernel_h, int kernel_w,
                  int up_x, int up_y, int down_x, int down_y,
                  int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                  int round_tf32, void* stream);

/* Fast path of the above for the FIRs the networks actually use: kernel = outer(taps_y, taps_x) with at most 4 taps
 * (e.g. make_kernel([1,3,3,1]) of stylegan2_layers.py:27-35), (up, down) in {(1,1), (1,2), (2,1)}: taps are HOST arrays,
 * unflipped.  Returns SAE_E_UNSUPPORTED when the restrictions (minor % 4, alignment, 32-bit work-item count) do not hold. */
int sae_upfirdn2d_separable(const float* input, const float* taps_y, const float* taps_x, float* out,
                            int64_t major, int in_h, int in_w, int minor, int kernel_h, int kernel_w,
                            int up, int down, int pad_x0, int pad_x1, int pad_y0, int pad_y1, int round_tf32, void* stream);

/* ------------------------------------------------------------------------------------------
 * fused_bias_act — out = act(x + b[(i / step_b) % size_b]) * scale.
 * Replaces  fused.fused_bias_act(input, bias, refer, act, grad, alpha, scale)
 *   (models/networks/stylegan2_op/fused_bias_act.cpp:11-20, fused_bias_act_kernel.cu:19-99).
 * act: 1 = linear, 3 = leaky-relu(alpha);  grad: 0 = forward, 1 = first-derivative form (masked
 * by sign of ref = saved OUTPUT), 2 = second derivative (zero).  bias == NULL / ref == NULL mean
 * "empty tensor" exactly as numel()==0 does in the reference.
 * noise/noise_weight (extension, NULL to disable): adds noise_weight[0] * noise[i / noise_div]
 * before the activation — NoiseInjection (stylegan2_layers.py:328-351) folded into the same pass.
 * ------------------------------------------------------------------------------------------ */
int sae_fused_bias_act(const float* x, const float* bias, const float* ref, float* out,
                       int64_t size_x, int64_t step_b, int size_b,
                       int act, int grad, float alpha, float scale,
                       const float* noise, const float* noise_weight, int64_t noise_div,
                       int round_tf32, void* stream);

/* Backward of the above in one pass: grad_in = grad_out * (out > 0 ? 1 : alpha) * scale and,
 * fused, grad_bias[c] += sum over everything but the bias dim (the reference runs a separate
 * .sum() kernel, fused_act.py:32-41).  grad_bias must be zero-initialised by the caller (or hold
 * a value to accumulate into).  Optional: noise != NULL accumulates d/d(noise_weight) =
 * sum(grad_in * noise) into grad_noise_weight[0].  Layout restriction: step_b == 1 (channels
 * innermost, i.e. NHWC or [B, C]).  act_mask != NULL (size_b % 32 == 0): the branch is read from the bit mask a
 * forward kernel wrote (sae_conv_epilogue.act_mask, sae_fir_bias_act) and `out` is not touched (may be NULL). */
int sae_bias_act_backward(const float* grad_out, const float* out, float* grad_in, float* grad_bias,
                          int64_t size_x, int size_b, float alpha, float scale,
                          const float* noise, int64_t noise_div, float* grad_noise_weight,
                          int round_tf32, const uint32_t* act_mask, void* stream);

/* sae_upfirdn2d_separable (up = down = 1) followed by sae_bias_act_backward, in ONE pass:
 *   grad_in = FIR(grad) * (act_out > 0 ? 1 : alpha) * scale,   grad_bias[c] += sum over pixels of grad_in
 * — the adjoint of the Blur that follows a ConvLayer's FusedLeakyReLU inside ResBlock (stylegan2_layers.py:672-693):
 * reference upfirdn2d.py:24-60 (UpFirDn2dBackward) + fused_act.py:23-41 (FusedLeakyReLUFunctionBackward) back to back;
 * the blurred gradient never travels through HBM.  grad: [major, in_h, in_w, minor]; act_out / grad_in:
 * [major, out_h, out_w, minor] with out = in + pad0 + pad1 - k + 1.  taps are HOST arrays, unflipped, 3 or 4 of them.
 * grad_bias (may be NULL) is accumulated into.  act_mask (may be NULL): the activation bit mask of act_out (see
 * sae_conv_epilogue.act_mask), read instead of act_out, which may then be NULL.  Returns SAE_E_UNSUPPORTED outside the
 * TMA-tiled configuration (minor % 32 == 0, outputs >= 8 x 8): issue the two separate calls then. */
int sae_fir_act_backward(const float* grad, const float* taps_y, const float* taps_x, const float* act_out,
                         float* grad_in, float* grad_bias, int64_t major, int in_h, int in_w, int minor,
                         int kernel_h, int kernel_w, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                         float alpha, float scale, int round_tf32, const uint32_t* act_mask, void* stream);

/* sae_upfirdn2d_separable (up = down = 1) followed by NoiseInjection + bias + leaky-ReLU, in ONE pass:
 *   out = lrelu(FIR(x) + noise_weight * noise[pixel] + bias[c], alpha) * scale
 * — the Blur behind the generator's transposed modulated convolution and the StyledConv tail after it
 * (stylegan2_layers.py:306-309 self.blur(out), then :398-405 noise -> FusedLeakyReLU; fused_act.py:89-96):
 * the blurred activation never travels through HBM.  x: [major, in_h, in_w, minor]; out: [major, out_h, out_w, minor];
 * noise: one value per OUTPUT pixel ([major, out_h, out_w]) or NULL; bias: [minor] or NULL.  taps are HOST arrays,
 * unflipped.  act_mask (may be NULL): receives the activation bit mask of out, [major * out_h * out_w * minor / 32] words.
 * Returns SAE_E_UNSUPPORTED outside the TMA-tiled configuration (minor % 32 == 0, outputs >= 8 x 8). */
int sae_fir_bias_act(const float* x, const float* taps_y, const float* taps_x, const float* bias, const float* noise,
                     const float* noise_weight, float* out, int64_t major, int in_h, int in_w, int minor,
                     int kernel_h, int kernel_w, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                     float alpha, float scale, int round_tf32, uint32_t* act_mask, void* stream);

/* ------------------------------------------------------------------------------------------
 * modulate — x_s[n,h,w,c] = x[n,h,w,c] * s[n,c]: the "input * style" step of
 * ModulatedConv2d.forward with new_demodulation (stylegan2_layers.py:278-284).
 * backward: dx = dy * s;  ds[n,c] = sum_hw dy * x  (ds must be zero-initialised).
 * round_tf32 != 0 rounds the result to TF32 (round-to-nearest) so the tensor-core conv that
 * consumes it sees exactly-representable operands.
 * ------------------------------------------------------------------------------------------ */
int sae_modulate(const float* x, const float* s, float* out,
                 int n, int64_t hw, int c, int round_tf32, void* stream);
int sae_modulate_backward(const float* dy, const float* x, const float* s, float* dx, float* ds,
                          int n, int64_t hw, int c, int round_tf32, void* stream);

/* ------------------------------------------------------------------------------------------
 * modulate_spatial — the "input * style" step for a spatially varying style (a texture code map
 * [N, C, h, w], stylegan2_layers.py:269-276 and generator.py:62-67), without the code map ever
 * reaching the layer's resolution.  The modulation affine commutes with bilinear interpolation
 * (its weights sum to 1), so the caller evaluates it at the map's own resolution: s_lo [ns, hs, ws, c]
 * NHWC, ns == 1 (broadcast over the batch) or ns == n.  Per pixel of x [n, h, w, c]:
 *   v = bilerp(s_lo)(h, w)     F.interpolate(..., size=(h, w), mode='bilinear', align_corners=False):
 *                              scale = hs / h, src = max(scale (y + 0.5) - 0.5, 0), i0 = floor(src),
 *                              i1 = i0 + (i0 < hs - 1), lambda = src - i0 (likewise along w)
 *   u = demodulate ? v * rsqrt(mean_c v^2 + 1e-8) : v
 *   out = x * u                (rounded to TF32 when round_tf32 != 0)
 * One read of x and one write of out; any c >= 1 (float4 path when c % 4 == 0 and the pointers are
 * 16-byte aligned), any ratio between (hs, ws) and (h, w).
 * backward: dx = dy * u (rounded like the forward) and ds_lo = the adjoint of the interpolation
 * applied to dv, where g = dy * x and dv = r (g - v r^2 mean_c(g v)), r = rsqrt(mean_c v^2 + 1e-8)
 * (demodulate) or dv = g; with ns == 1 the adjoint also sums over the batch.  ds_lo is overwritten.
 * No atomics: a per-pixel pass, then a gather over the columns and one over the rows (and batch) that
 * each low-resolution cell's stencil touches, in a fixed order — identical inputs give identical bits.
 * workspace: caller-owned device buffer of 4 * ceil(n * h * ws * c / 4) + 2 * n * h * w floats,
 * 16-byte aligned.
 * ------------------------------------------------------------------------------------------ */
int sae_modulate_spatial(const float* x, const float* s_lo, float* out, int n, int h, int w, int c, int ns, int hs, int ws,
                         int demodulate, int round_tf32, void* stream);
int sae_modulate_spatial_backward(const float* dy, const float* x, const float* s_lo, float* dx, float* ds_lo, float* workspace,
                                  int n, int h, int w, int c, int ns, int hs, int ws, int demodulate, int round_tf32, void* stream);

/* out = (a + b) * scale — the residual merge "(out + skip) / sqrt(2)" of ResBlock (stylegan2_layers.py:691) and of the
 * generator blocks (generator.py:36,53) in one pass; b == NULL gives out = a * scale (its backward).
 * sae_round_tf32: out = rna_tf32(x) (used on the small filter tensors before a tensor-core conv). */
int sae_add_scale(const float* a, const float* b, float* out, int64_t n, float scale, int round_tf32, void* stream);
int sae_round_tf32(const float* x, float* out, int64_t n, void* stream);

/* out[n,2h,2w,c] = (bilinear_x2(skip[n,h,w,c]) + res) * scale — the generator's skip branch
 * F.interpolate(skip, scale_factor=2, mode='bilinear', align_corners=False) followed by (skip + res) / sqrt(2)
 * (models/networks/generator.py:51-53) in one pass; sae_upsample2x_backward is the adjoint of the interpolation
 * times scale (gradient w.r.t. skip; the gradient w.r.t. res is sae_add_scale(dy, NULL, scale)). c % 4 == 0. */
int sae_upsample2x_add_scale(const float* skip, const float* res, float* out, int n, int h, int w, int c, float scale,
                             int round_tf32, void* stream);
int sae_upsample2x_backward(const float* dy, float* dskip, int n, int h, int w, int c, float scale, int round_tf32,
                            void* stream);

/* Filter preparation: parameter layout [K,C,R,S] -> out_krsc [K,R,S,C] (and out_crsk [C,R,S,K] when non-NULL), times
 * `scale` (the equalised-lr factor of EqualConv2d / EqualLinear / ModulatedConv2d, stylegan2_layers.py:122,164,246),
 * rounded to TF32 when round_tf32 — one pass instead of mul + permute + copy + round.  sae_filter_unprep is its adjoint
 * (d_w[k,c,r,s] = scale * d_krsc[k,r,s,c]) for the weight gradient. */
int sae_filter_prep(const float* w, float* out_krsc, float* out_crsk, int k, int c, int r, int s, float scale,
                    int round_tf32, void* stream);
int sae_filter_unprep(const float* d_krsc, float* d_w, int k, int c, int r, int s, float scale, void* stream);

/* nn.ReflectionPad2d((pad_l, pad_r, pad_t, pad_b)) on NHWC data and its adjoint (the encoder's ReflectionPad2d,
 * stylegan2_layers.py:104,642); c % 4 == 0. */
int sae_reflect_pad(const float* x, float* out, int n, int h, int w, int c, int pad_l, int pad_r, int pad_t, int pad_b,
                    void* stream);
int sae_reflect_pad_backward(const float* dy, float* dx, int n, int h, int w, int c, int pad_l, int pad_r, int pad_t,
                             int pad_b, void* stream);

/* Zero-pad the channel dimension while converting to the kernels' NHWC layout: out[n, p, 0:c_out] = (x[n, 0:c_in, p], 0...)
 * for the `pixels` positions of each image; x is addressed with element strides (stride_n, stride_c, stride_p), so the
 * reference's NCHW image batches (stride_c = H*W, stride_p = 1) and channels-last tensors (stride_c = 1, stride_p = c_in)
 * are both read in place.  Feeds the 3-channel inputs of FromRGB (ConvLayer(3, ch, 1), stylegan2_layers.py:716,
 * encoder.py:38) and of the patch discriminator's first conv (patch_discriminator.py:111) to the tensor-core conv
 * kernels, whose TMA rows are 32 channels; c_out % 4 == 0, c_in <= c_out. */
int sae_pad_channels(const float* x, float* out, int64_t n, int64_t pixels, int c_in, int c_out,
                     int64_t stride_n, int64_t stride_c, int64_t stride_p, int round_tf32, void* stream);

/* ------------------------------------------------------------------------------------------
 * conv2d — dense implicit-GEMM convolution family on NHWC fp32 activations, TF32 tensor cores,
 * fp32 accumulate.  Replaces the F.conv2d / F.conv_transpose2d call sites of
 * EqualConv2d.forward (stylegan2_layers.py:136-142), EqualLinear.forward (:174-186, H=W=1) and
 * ModulatedConv2d.forward (:299-323; the groups=batch grouped conv there uses identical weights
 * for every sample — SURVEY.md §0.1 — so it is one dense conv on the style-scaled input).
 *
 * Geometry (one struct for the three directions of the same convolution):
 *   y[n,p,q,o] = sum_{r,s,c} x[n, p*stride - pad_t + r, q*stride - pad_l + s, c] * w[o,r,s,c]
 *   x: [N, H, W, C]   w: [K, R, S, C]   y: [N, P, Q, K]
 * fprop computes y from (x, w); dgrad computes x-gradient from (dy, w) — and is also the forward
 * of the stride-2 transposed convolution in the generator's upsampling path (:306);
 * wgrad computes w-gradient from (dy, x).
 * ------------------------------------------------------------------------------------------ */
typedef struct sae_conv_geom {
    int32_t N, H, W, C;      /* input  activation  [N,H,W,C]              */
    int32_t K, R, S;         /* filter             [K,R,S,C]              */
    int32_t P, Q;            /* output activation  [N,P,Q,K]              */
    int32_t stride;          /* same in y and x                           */
    int32_t pad_t, pad_l;    /* top / left zero padding (bottom/right implied by P,Q) */
} sae_conv_geom;

/* Optional fused epilogue for fprop / dgrad (all pointers may be NULL):
 *   v = acc
 *   v += bias[col]                                   (EqualConv2d bias, stylegan2_layers.py:139)
 *   v += noise_weight[0] * noise[pixel]              (NoiseInjection, :351)
 *   if act == 3: v = (v > 0 ? v : alpha * v) * gain  (FusedLeakyReLU, fused_act.py:89-96)
 *   else       : v = v * gain
 *   if residual: v = (v + residual[pixel, col]) * res_scale   (ResBlock (out+skip)/sqrt2, :691)
 *   if round_tf32: v = rna_tf32(v)
 */
typedef struct sae_conv_epilogue {
    const float* bias;
    const float* noise;
    const float* noise_weight;
    const float* residual;
    float   alpha;
    float   gain;
    float   res_scale;
    int32_t act;           /* 1 = linear, 3 = leaky relu */
    int32_t round_tf32;
    uint32_t* act_mask;    /* optional (tcgen05 kernels only, K % 32 == 0; NULL elsewhere): bit (i & 31) of word i >> 5 is set
                              when element i of y (NHWC order) went through the positive branch of the activation.  The backward
                              passes take it instead of the 4-byte-per-element output (sae_bias_act_backward, sae_fir_act_backward):
                              12 -> 8.1 bytes per element on kernels that run at the HBM roofline. */
} sae_conv_epilogue;

/* impl: 0 = auto (tcgen05/TMA kernel when the shape qualifies, otherwise the generic
 * mma.sync kernel), 1 = force generic, 2 = force tcgen05 (SAE_E_UNSUPPORTED if not eligible). */
int sae_conv2d_fprop(const float* x, const float* w, float* y, const sae_conv_geom* g,
                     const sae_conv_epilogue* epi, int impl, void* stream);
/* wt is the filter pre-transposed to [C, R, S, K] (host side does the tiny permute). */
int sae_conv2d_dgrad(const float* dy, const float* wt, float* dx, const sae_conv_geom* g,
                     const sae_conv_epilogue* epi, int impl, void* stream);
/* dw [K,R,S,C] is ACCUMULATED into (split-K reduction with fp32 atomics): zero it first. */
int sae_conv2d_wgrad(const float* dy, const float* x, float* dw, const sae_conv_geom* g,
                     int impl, void* stream);

/* Which kernel `impl = 0` would pick for this geometry: 1 generic, 2 tcgen05. dir: 0 fprop, 1 dgrad, 2 wgrad */
int sae_conv2d_query_impl(const sae_conv_geom* g, int dir);

/* ------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange helpers (SURVEY.md §8(e)): pack the active parameter group's
 * gradients into one flat fp32 bucket for a single NCCL all-reduce, then unpack scaled by 1/world.
 * Replaces nn.DataParallel's ReduceAddCoalesced onto GPU 0 (models/__init__.py:80).
 * ptrs: device array of n pointers; sizes / offsets: device arrays of n int64 (elements).
 * ------------------------------------------------------------------------------------------ */
int sae_bucket_pack(const float* const* ptrs, const int64_t* offsets, const int64_t* sizes, int n,
                    float* bucket, int64_t total, void* stream);
int sae_bucket_unpack(float* const* ptrs, const int64_t* offsets, const int64_t* sizes, int n,
                      const float* bucket, int64_t total, float scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Style-modulated convolution WITHOUT a modulated copy of the activation (SURVEY.md §8 a5).
 * Reference ModulatedConv2d.forward (stylegan2_layers.py:266-325) scales the input by the style ("input * style", :284) and
 * runs a grouped convolution over `batch` copies of the filter (:286, :321); a first B200 design scaled the input in a
 * separate pass.  Here the style goes into the FILTER the tensor-core kernel reads: image n is convolved with
 *   Wn[k,r,s,c] = W[k,r,s,c] * s[n,c]           (sae_filter_modulate: [N,K,R,S,C] and, for the data gradient, [N,C,R,S,K])
 * selected per pixel tile inside the implicit-GEMM kernel (sae_conv2d_fprop_per_sample / sae_conv2d_dgrad_per_sample; same
 * epilogue as sae_conv2d_fprop).  The weight gradient takes x UNSCALED and drains its accumulators once per image:
 *   dW[k,r,s,c] += s[n,c] * Gn[k,r,s,c],   ds[n,c] += sum_{k,r,s} W[k,r,s,c] * Gn[k,r,s,c],   Gn = sum_pixels dy (x) x
 * (sae_conv2d_wgrad_modulated; dw and ds zero-initialised by the caller).  Pays when N * |W| << |x| (the 128- and 256-channel
 * 3x3 layers at 256^2 / 128^2).  sae_conv2d_query_modulated: 1 when all three kernels take the geometry (stride 1, map a
 * multiple of 16 x 8 tiles with an even tile count per image, Q % 32 == 0, channels % 32 == 0), 0 otherwise — the caller
 * then scales the input (sae_modulate).
 * ------------------------------------------------------------------------------------------ */
int sae_filter_modulate(const float* w_krsc, const float* s, float* out_nkrsc, float* out_ncrsk, int n, int k, int c, int r,
                        int s_, int round_tf32, void* stream);
int sae_conv2d_query_modulated(const sae_conv_geom* g);
int sae_conv2d_fprop_per_sample(const float* x, const float* w_nkrsc, float* y, const sae_conv_geom* g,
                                const sae_conv_epilogue* epi, void* stream);
int sae_conv2d_dgrad_per_sample(const float* dy, const float* w_ncrsk, float* dx, const sae_conv_geom* g,
                                const sae_conv_epilogue* epi, void* stream);
int sae_conv2d_wgrad_modulated(const float* dy, const float* x, const float* s, const float* w_krsc, float* dw, float* ds,
                               const sae_conv_geom* g, void* stream);

/* ------------------------------------------------------------------------------------------
 * Multi-tensor Adam (SURVEY.md §8 f2).  Replaces the two torch.optim.Adam instances of
 * optimizers/swapping_autoencoder_optimizer.py:34-42 with one launch per parameter group.
 * torch.optim.Adam semantics (amsgrad off, no weight decay):  for every tensor t with g_ptrs[t] != NULL
 *   steps[t] += 1;  m += (1 - beta1)(g - m);  v = beta2 v + (1 - beta2) g^2;
 *   p -= lr / (1 - beta1^steps[t]) * m / (sqrt(v) / sqrt(1 - beta2^steps[t]) + eps),        g = grad_scale * *g_ptrs[t]
 * a NULL gradient pointer skips the tensor and leaves its step count alone (a parameter whose .grad is None).
 * p_ptrs / g_ptrs: device arrays of n pointers; offsets / sizes: device arrays of n int64 (elements) locating each
 * tensor's moments inside the flat exp_avg / exp_avg_sq buffers; steps: device array of n floats.
 * g_ptrs may point into the flat all-reduce bucket (sae_bucket_pack) with grad_scale = 1 / world: the gradient
 * average is then never written back to the per-parameter gradient tensors.
 * ------------------------------------------------------------------------------------------ */
int sae_adam_step(float* const* p_ptrs, const float* const* g_ptrs, const int64_t* offsets, const int64_t* sizes, int n,
                  float* exp_avg, float* exp_avg_sq, float* steps, float lr, float beta1, float beta2, float eps,
                  float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Random-crop resampler of the patch discriminator (SURVEY.md §8 f1).  Replaces
 *   apply_random_crop: affine sampling grid + F.grid_sample(bilinear, zeros padding, align_corners=False)
 *   (util/util.py:323-343, called from models/swapping_autoencoder_model.py:100-103)
 * and the channel pad / layout copy in front of the first Dpatch convolution (patch_discriminator.py:146-158).
 * x: source images, logical [B, C, H, W] addressed through element strides (any layout), C <= 4.
 * Crop q (Q = B * num_crops of them, q / num_crops = source image) samples
 *   gx = (lin_j * flip[q]) * scale[q][0] + offset[q][0],  gy = lin_i * scale[q][1] + offset[q][1],  lin = linspace(-1, 1, S)
 * out: NHWC [Q, S, S, CP] with channels C..CP-1 written as zeros (CP % 4 == 0), optionally TF32-rounded.
 * sae_crop_gather_backward: the adjoint in gather form (no atomics, deterministic): dx [B, C, H, W] contiguous is
 * OVERWRITTEN with the sum over each image's crops; dy is addressed through element strides (n, c, h, w).
 * ------------------------------------------------------------------------------------------ */
int sae_crop_gather(const float* x, const float* flip, const float* scale, const float* offset, float* out,
                    int Q, int num_crops, int C, int H, int W, int S, int CP,
                    int64_t xs_n, int64_t xs_c, int64_t xs_h, int64_t xs_w, int round_tf32, void* stream);
int sae_crop_gather_backward(const float* dy, const float* flip, const float* scale, const float* offset, float* dx,
                             int Q, int num_crops, int C, int H, int W, int S,
                             int64_t ds_n, int64_t ds_c, int64_t ds_h, int64_t ds_w, void* stream);

/* ------------------------------------------------------------------------------------------
 * ToRGB — the generator's final 1x1 style-modulated convolution without demodulation, as a bandwidth kernel.
 * Replaces ToRGB.forward -> ModulatedConv2d(in_channel, 3, 1, demodulate=False) + bias
 *   (models/networks/stylegan2_layers.py:408-427, :266-325: input * style, grouped F.conv2d, + bias).
 * forward:  y[n,p,o] = bias[o] + sum_c x[n,p,c] * (wscale * s[n,c] * w[o,c]),  o < 3;  y is NHWC with 4 channels (4th = 0).
 *   x [N,H,W,C] NHWC, s [N,C], w [3,C], bias [3] or NULL; C % 4 == 0, C <= 1024.  x is read once; nothing else is large.
 * backward (one pass over x): dx[n,p,c] = sum_o dy[n,p,o] * wscale * s[n,c] * w[o,c]   (NHWC, optional)
 *                             gw[n,o,c] += sum_p dy[n,p,o] * x[n,p,c]                   ([N,3,C], zero-initialised, optional)
 *   dy is addressed through element strides (n, c, h, w).  The caller forms d s = wscale * sum_o gw * w and
 *   d w = wscale * sum_n gw * s from the [N,3,C] values.
 * ------------------------------------------------------------------------------------------ */
int sae_torgb_forward(const float* x, const float* s, const float* w, const float* bias, float* y,
                      int N, int H, int W, int C, float wscale, int round_tf32, void* stream);
int sae_torgb_backward(const float* dy, const float* x, const float* s, const float* w, float* dx, float* gw,
                       int N, int H, int W, int C, float wscale,
                       int64_t ds_n, int64_t ds_c, int64_t ds_h, int64_t ds_w, int round_tf32, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* SAE_B200_H_ */
