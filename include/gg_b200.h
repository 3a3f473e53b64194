/*
 * gg_b200.h -- C ABI of libgg_b200.so: the sm_100a kernels behind GANgealing's op-level hot path.
 *
 * Every entry point replaces one native binding (or one cluster of ATen launches) of the reference
 * wpeebles/gangealing; the reference location is cited on each declaration (paths relative to the
 * reference checkout).  Conventions, identical for all entry points:
 *
 *   - plain pointers and sizes only, no torch types; all pointers are DEVICE pointers unless the
 *     parameter name ends in `_host`;
 *   - the caller owns every buffer (inputs, outputs, workspaces); the library allocates nothing,
 *     keeps no mutable global state and never synchronises the device;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - return value: 0 = ok, negative = error (GG_ERR_*); gg_last_error() returns a thread-local
 *     human-readable message for the last failing call on this thread.  Never calls exit();
 *   - re-entrant: safe to call concurrently from the Python main thread and PyTorch's autograd thread;
 *   - tensors are dense ("contiguous") in the layout stated per function; element type is selected
 *     by a gg_dtype code; accumulation is always fp32.
 *   - staged (bulk-TMA) kernels may READ, never write, up to 15 bytes before/after an input buffer so
 *     that transfers are 16-byte aligned; those bytes never influence results.  (Any CUDA allocation
 *     is at least 256-byte granular, so the enclosing 16-byte window is always mapped.)
 */
#ifndef GG_B200_H_
#define GG_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GG_API __attribute__((visibility("default")))

/* element types */
enum { GG_F32 = 0, GG_F16 = 1, GG_BF16 = 2, GG_F64 = 3 };

/* error codes */
enum {
  GG_OK = 0,
  GG_ERR_BAD_ARG = -1,      /* null pointer, negative size, inconsistent shape            */
  GG_ERR_UNSUPPORTED = -2,  /* dtype / mode not implemented by this entry point           */
  GG_ERR_CUDA = -3          /* a CUDA runtime call failed; message holds cudaGetErrorString */
};

/* padding modes of the samplers (torch.nn.functional.grid_sample's padding_mode) */
enum { GG_PAD_ZEROS = 0, GG_PAD_BORDER = 1, GG_PAD_REFLECTION = 2 };

GG_API int gg_version(void);                 /* ABI version, bumped on any signature change */
GG_API const char* gg_last_error(void);      /* thread-local, never NULL */
GG_API int gg_sm_count(void);                /* multiProcessorCount of the current device (cached) */

/* ------------------------------------------------------------------------------------------------
 * fused_bias_act -- replaces `fused.fused_bias_act(input, bias, refer, act, grad, alpha, scale)`
 *   reference: models/stylegan2/op/fused_bias_act.cpp:11-21, fused_bias_act_kernel.cu:18-99
 *   x'   = x + bias[(i / step_b) % size_b]            (bias == NULL: no bias)
 *   act=1: y = x'                       (grad 0/1), 0 (grad 2)
 *   act=3: y = x'   > 0 ? x' : alpha*x' (grad 0)
 *          y = ref  > 0 ? x' : alpha*x' (grad 1; ref = saved forward OUTPUT), 0 (grad 2)
 *   out = y * scale
 *   x/out/ref: `size_x` elements of `dtype`; bias: `size_b` elements of `dtype`.
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_fused_bias_act(void* out, const void* x, const void* bias, const void* ref, int dtype,
                             int act, int grad, float alpha, float scale, int64_t size_x,
                             int64_t step_b, int64_t size_b, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_noise_bias_act -- NoiseInjection + FusedLeakyReLU of a StyledConv in one pass
 *   reference: models/stylegan2/networks.py:291-298 (noise) + :344-350 + op/fused_act.py:52-58
 *   out[n,c,p] = lrelu(row_scale[n*C+c]*x[n,c,p] + noise_weight[0]*noise[n,p] + bias[c], alpha) * scale
 *   x/out: (N, C, HW) `dtype`;  noise: (N, HW) `dtype` or NULL;  noise_weight: 1 fp32 (device) or
 *   NULL (=1);  bias: C fp32 or NULL;  row_scale: N*C fp32 or NULL (=1; the demodulation coefficients when
 *   the convolution ran with shared weights on modulated activations).
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_noise_bias_act(void* out, const void* x, const void* noise, const float* noise_weight,
                             const float* bias, const float* row_scale, int dtype, float alpha, float scale,
                             int64_t N, int64_t C, int64_t HW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_channel_scale -- per-(sample, channel) scaling of an activation, the modulation of
 *   reference models/stylegan2/networks.py:236,243 applied to the convolution's INPUT instead of its weights:
 *   conv(scale*W*s[b,i], x) == conv(scale*W, x*s[b,i])  -> weight-shared (dense, tensor-core friendly) convolutions.
 *   out[r,p] = x[r,p] * s[r]        rows r = n*C + c, p < HW
 *   row_dot[r] = sum_p x[r,p]*y[r,p]   (optional; with y = upstream gradient this is d/ds; fp32, deterministic;
 *   needs gg_channel_scale_workspace(rows, HW) bytes)
 * ---------------------------------------------------------------------------------------------- */
GG_API int64_t gg_channel_scale_workspace(int64_t rows, int64_t HW);
GG_API int gg_channel_scale(void* out, float* row_dot, void* workspace, const void* x, const void* y,
                            const float* s, int dtype, int64_t rows, int64_t HW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_bias_act_backward -- FusedLeakyReLUFunctionBackward in one pass
 *   reference: models/stylegan2/op/fused_act.py:20-38 (kernel call act=3,grad=1 + grad_input.sum(dims))
 *   gx[n,c,p] = (out[n,c,p] > 0 ? g : alpha*g) * scale
 *   grad_bias[c] = sum_{n,p} gx[n,c,p]      (fp32; skipped when grad_bias == NULL)
 *   Deterministic two-stage reduction; `workspace` must hold gg_bias_act_backward_workspace() bytes
 *   (may be NULL when grad_bias is NULL).
 * ---------------------------------------------------------------------------------------------- */
GG_API int64_t gg_bias_act_backward_workspace(int64_t N, int64_t C, int64_t HW);
GG_API int gg_bias_act_backward(void* gx, float* grad_bias, void* workspace, const void* g,
                                const void* out, int dtype, float alpha, float scale, int64_t N,
                                int64_t C, int64_t HW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_upfirdn2d -- replaces `upfirdn2d_op.upfirdn2d(input, kernel, up_x, up_y, down_x, down_y,
 *                                                  pad_x0, pad_x1, pad_y0, pad_y1)`
 *   reference: models/stylegan2/op/upfirdn2d.cpp:12-23, upfirdn2d_kernel.cu:209-369
 *   (semantics: upfirdn2d.py:159-200 -- zero-insert upsample, pad/crop, TRUE convolution with
 *    `kernel`, decimate).  in: (major, in_h, in_w) dense; out: (major, out_h, out_w) with
 *    out_h = (in_h*up_y + pad_y0 + pad_y1 - kernel_h) / down_y + 1 (same for w); the reference's
 *    trailing `minor` dimension is always 1 in GANgealing and is not modelled.
 *   kernel: kernel_h*kernel_w fp32 taps (device), NOT flipped (the library flips, as the reference).
 *   Dispatch: up=down=1 and kernel <= 4x4 -> bulk-TMA staged band kernel; otherwise generic gather.
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_upfirdn2d(void* out, const void* in, const float* kernel, int dtype, int64_t major,
                        int in_h, int in_w, int kernel_h, int kernel_w, int up_x, int up_y,
                        int down_x, int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_blur_noise_bias_act -- the fused StyledConv(upsample) tail: Blur -> NoiseInjection ->
 *   FusedLeakyReLU in ONE pass over the activation (the "fused upfirdn2d+bias-act path").
 *   reference: models/stylegan2/networks.py:266 (blur) + :346-348 (noise, activate);
 *              op/upfirdn2d_kernel.cu:107-207 + op/fused_bias_act_kernel.cu:18-49
 *   t = upfirdn2d(in, kernel, up=1, down=1, pad)               (kernel <= 4x4)
 *   out[n,c,y,x] = lrelu(row_scale[n*C+c]*t + noise_weight[0]*noise[n,y,x] + bias[c], alpha) * scale
 *   in: (N*C, in_h, in_w) dtype; out: (N*C, out_h, out_w); noise: (N, out_h, out_w) dtype or NULL;
 *   noise_weight: 1 fp32 or NULL(=1); bias: C fp32 or NULL; row_scale: N*C fp32 or NULL (=1; lets a
 *   caller fold the per-sample demodulation of a weight-shared conv into the tail);
 *   act: 1 linear, 3 leaky-relu.
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_blur_noise_bias_act(void* out, const void* in, const float* kernel, const void* noise,
                                  const float* noise_weight, const float* bias,
                                  const float* row_scale, int dtype, int64_t N, int64_t C, int in_h,
                                  int in_w, int kernel_h, int kernel_w, int pad_x0, int pad_x1,
                                  int pad_y0, int pad_y1, int act, float alpha, float scale,
                                  void* stream);

/* ------------------------------------------------------------------------------------------------
 * Antialiased (mip-mapped) bilinear grid sampling -- replaces MipmapWarp / Warp
 *   reference: models/spatial_transformers/antialiased_sampling.py:9-16 (Warp), :35-238 (MipmapWarp)
 *   and the ATen kernels behind F.grid_sample(align_corners=False) / F.interpolate / F.conv2d they call.
 *
 *   Pyramid: level i (1..extra_levels) = i applications of [ReflectionPad2d(1) -> depthwise
 *   [1,3,3,1]^2/64 stride-2 conv] (:111-117) to the source, after the reference's reflect padding to the
 *   next power of two when the width is not one (:130-137).  Stored fp32, level-major, at native
 *   resolution: gg_mipmap_pyramid_elems() floats (returns -1 if the size cannot host that many levels,
 *   exactly when the reference's stack construction would fail).
 *
 *   forward : out[n,c,y,x] = lerp(S_floor(l), S_ceil(l), l mod 1),  S_i = bilinear sample of level i
 *             upsampled x2^i (align_corners=False) at grid[n,y,x]; l = clamp(log2(max 4-neighbour
 *             distance of the (size-1)-scaled coordinates, each >= 1), 0, max_level) clamped >= min_level
 *             (:62-97, :181-210).  extra_levels == 0: plain bilinear grid_sample (Warp).
 *             levels_out (N,Ho,Wo) fp32 receives l (NULL to skip).
 *   backward: gradients w.r.t. the source (through every pyramid level; grad_src/grad_pyramid are fp32,
 *             ZERO-INITIALISED by the caller and accumulated with atomics; finish with
 *             gg_mipmap_build_backward) and w.r.t. the grid (sampling position AND level-of-detail terms,
 *             like autograd through the reference; grad_grid fp32, zero-initialised by the caller).
 *   src/out/grad_out: `dtype`; grid: fp32 (N, Ho, Wo, 2), normalised to [-1, 1].
 * ---------------------------------------------------------------------------------------------- */
GG_API int64_t gg_mipmap_pyramid_elems(int64_t planes, int hs, int ws, int extra_levels);
GG_API int gg_mipmap_build(float* pyramid, const void* src, int dtype, int64_t planes, int hs, int ws,
                           int extra_levels, void* stream);
GG_API int gg_mipmap_build_backward(float* grad_src, float* grad_pyramid, int64_t planes, int hs, int ws,
                                    int extra_levels, void* stream);
GG_API int gg_mipmap_warp_forward(void* out, float* levels_out, const void* src, const float* pyramid,
                                  const float* grid, int dtype, int64_t N, int C, int hs, int ws, int ho,
                                  int wo, int extra_levels, float max_level, float min_level,
                                  int padding_mode, void* stream);
/* grad_grid is written in full; with extra_levels > 0 it needs a workspace of gg_mipmap_warp_backward_workspace
 * bytes (the level-of-detail gradient owed to a neighbour pixel, summed in a fixed order: reproducible bits). */
GG_API int64_t gg_mipmap_warp_backward_workspace(int64_t N, int ho, int wo);
GG_API int gg_mipmap_warp_backward(float* grad_src, float* grad_pyramid, float* grad_grid, void* workspace,
                                   const void* grad_out, const void* src, const float* pyramid,
                                   const float* grid, int dtype, int64_t N, int C, int hs, int ws, int ho,
                                   int wo, int extra_levels, float max_level, float min_level,
                                   int padding_mode, void* stream);
/* The sampler's INTEGER work, exported for exact parity tests (no reference counterpart: ATen's grid_sampler_2d and
 * antialiased_sampling.py:228-229 compute these integers internally).  indices: int32 (N, Ho, Wo, 4), 16-byte aligned =
 * (x0, y0, l0, l1): north-west bilinear corner after the padding-mode transform, floor / ceil of the level of detail --
 * evaluated by the same device functions as gg_mipmap_warp_forward / gg_stn_sample_forward. */
GG_API int gg_warp_sample_indices(int32_t* indices, const float* grid, int64_t N, int hs, int ws, int ho, int wo,
                                  float max_level, float min_level, int padding_mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Flow composition of the flow STN head -- replaces upsample_flow + identity add + apply_affine + alpha lerp
 *   reference: models/spatial_transformers/warping_heads.py:180-193 (RAFT convex upsampling: softmax over the
 *   9 mask logits x F.unfold(S*flow, 3x3, padding=1)), :239-244, :268-277 (apply_affine: [gx, gy, 1] @ M^T)
 *   low_flow (N, H, W, 2); mask (N, 9*S*S, H, W); identity_flow (S*H, S*W, 2) = F.affine_grid(identity);
 *   base_warp (N, 2, 3) or NULL; alpha (N) or NULL.  All fp32.
 *   forward : delta_flow (N, S*H, S*W, 2) and, if `flow` != NULL, flow = lerp(identity, affine(identity + delta), alpha)
 *   backward: grad_mask, grad_low_flow and grad_base_warp (each may be NULL) are written in full; the latter two need a
 *             workspace of gg_flow_compose_backward_workspace bytes (per-pixel terms summed in a fixed order:
 *             reproducible bits); grad_delta / grad_flow are the incoming gradients (either may be NULL).
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_flow_compose_forward(float* delta_flow, float* flow, const float* low_flow, const float* mask,
                                   const float* identity_flow, const float* base_warp, const float* alpha,
                                   int64_t N, int H, int W, int S, void* stream);
GG_API int64_t gg_flow_compose_backward_workspace(int64_t N, int H, int W, int S);
GG_API int gg_flow_compose_backward(float* grad_mask, float* grad_low_flow, float* grad_base_warp, void* workspace,
                                    const float* grad_delta, const float* grad_flow, const float* low_flow,
                                    const float* mask, const float* identity_flow, const float* base_warp,
                                    const float* alpha, int64_t N, int H, int W, int S, void* stream);

/* ------------------------------------------------------------------------------------------------
 * gg_splat2d_forward -- replaces `_splat.splat_forward_cuda(input, coordinates, values, sigma, soft_normalize)`
 *   reference: utils/splat2d_cuda/src/splat_gpu.c:12-42 (host: zeros/clone/clamp/divide) and
 *              splat_gpu_impl.cu:41-96 / splat_gpu_impl.cuh:11-22 (kernel `SplatForward`, extern-C `SplatForwardGpu`)
 *   For every point (x, y) inside the image (0 <= x < W, 0 <= y < H) and every pixel of its footprint
 *   [floor(y-2s), ceil(y+2s)] x [floor(x-2s), ceil(x+2s)] clipped to the image:
 *       a = exp(-((px-x)^2 + (py-y)^2) / (2 s^2));  A[py,px] += a;  S[c,py,px] += a * value[c]
 *   out = (input + S) / ((soft_normalize ? max(A, 1) : A) + 1e-8)
 *   input/out (N, C, H, W); coordinates (N, P, 2) as (x, y); values (N, P, C); sigma (N).  fp32 only, forward
 *   only (as the reference).  `workspace`: gg_splat2d_workspace() bytes (interleaved accumulators; the
 *   library zeroes it).
 * ---------------------------------------------------------------------------------------------- */
GG_API int64_t gg_splat2d_workspace(int64_t N, int C, int H, int W);
GG_API int gg_splat2d_forward(float* out, void* workspace, const float* input, const float* coordinates,
                              const float* values, const float* sigma, int64_t N, int64_t P, int C, int H,
                              int W, int soft_normalize, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The STN's sampling in ONE pass (north_star: "antialiased bilinear grid_sample fused with flow-compose in one pass").
 * The sampling grid is generated per output pixel from the head's raw outputs instead of being read from memory:
 *   mode 1  SimilarityHead (reference warping_heads.py:120-136): grid = F.affine_grid(theta (N, 2, 3), align_corners=False)
 *   mode 2  FlowHead (warping_heads.py:180-193 upsample_flow, :239-244, :268-277 apply_affine): low (N, lh, lw, 2),
 *           mask (N, 9*s*s, lh, lw), identity (s*lh, s*lw, 2), optional base warp `theta` (N, 2, 3) and alpha (N);
 *           ho == s*lh, wo == s*lw
 * then the level-of-detail selection + trilinear sample of gg_mipmap_warp_forward (antialiased_sampling.py:35-238) on
 * `src` (N, C, hs, ws) and its `pyramid` (gg_mipmap_build; extra_levels == 0: plain bilinear sampling).
 * Outputs: out (N, C, ho, wo); grid_out (N, ho, wo, 2) and delta_out (mode 2: the residual flow of the TV regulariser,
 * reference models/losses/loss.py:4-12) are written as by-products (NULL: skipped); levels_out (N, ho, wo) or NULL.
 * The backward pass is gg_mipmap_warp_backward on grid_out (+ gg_flow_compose_backward for mode 2).
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_stn_sample_forward(void* out, float* grid_out, float* delta_out, float* levels_out, const void* src,
                                 const float* pyramid, const float* theta, const float* low, const float* mask,
                                 const float* identity, const float* alpha, int mode, int dtype, int64_t N, int C,
                                 int hs, int ws, int ho, int wo, int lh, int lw, int s, int extra_levels,
                                 float max_level, float min_level, int padding_mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Modulated-convolution weight path -- replaces the tensor-op chain of ModulatedConv2d.forward
 *   reference: models/stylegan2/networks.py:233-253 (modulate, demodulate), :255-262 (layout for the up-conv)
 *   weight (O, I, kk) fp32 [kk = k*k]; style (B, I) fp32 (output of the modulation EqualLinear).
 *   gg_modconv_wsq      wsq[o,i] = sum_kk weight[o,i,kk]^2
 *   gg_modconv_demod    demod[b,o] = rsqrt(scale^2 * sum_i wsq[o,i]*style[b,i]^2 + eps)   (B <= 256)
 *                       tcgen05.mma kind::tf32 with a hi/lo operand split (fp32-grade accuracy), TMEM accumulator
 *   gg_modconv_modulate out = scale * weight * style[b,i] * demod[b,o]   (demod == NULL: no demodulation)
 *                       transposed == 0: out (B, O, I, kk), `weight` given as (O, I, kk)
 *                       transposed != 0: out (B, I, O, kk), `weight` given PRE-TRANSPOSED as (I, O, kk)
 *                       (I*kk, resp. O*kk, must be a multiple of 4)
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_modconv_wsq(float* wsq, const float* weight, int O, int I, int kk, void* stream);
GG_API int gg_modconv_demod(float* demod, const float* wsq, const float* style, float scale, float eps, int B,
                            int O, int I, void* stream);
/* all layers of a generator in ONE launch: tables (host arrays of `layers` entries) of per-layer demod (B, O[l]) outputs,
 * wsq (O[l], I[l]), style (B, I[l]), scale, O, I; every layer shares the batch size B <= 256; layers <= 32. */
GG_API int gg_modconv_demod_batched(int layers, float* const* demod, const float* const* wsq, const float* const* style,
                                    const float* scale, const int* O, const int* I, float eps, int B, void* stream);
GG_API int gg_modconv_modulate(float* out, const float* weight, const float* style, const float* demod,
                               float scale, int B, int O, int I, int kk, int transposed, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Channels-last (N, H, W, C) variants of the StyledConv tail family.  Same math and reference citations as
 * gg_noise_bias_act / gg_bias_act_backward / gg_channel_scale / gg_blur_noise_bias_act; they exist so the generator's
 * activations can stay NHWC between cuDNN's (NHWC-native) tensor-core convolutions.
 *   dtype: GG_F32 or GG_BF16 = the STORAGE type of the activations (arithmetic is fp32; BASELINE config 3 runs bf16
 *     activations -- the reference has no bf16 at all: models/stylegan2/op/upfirdn2d_kernel.cu:311 dispatches
 *     float/double/half only).  An activation moves 16 bytes at a time: C % 4 == 0 (fp32) / C % 8 == 0 (bf16).
 *     noise, bias, row scales, reductions are always fp32.
 *   gg_blur_nhwc: upfirdn2d(up = down = 1, filter <= 4x4) on (N, H, W, C), C % 32 == 0 (fp32) / C % 64 == 0 (bf16), input
 *     rows streamed with 4-D TMA tensor-map loads whose out-of-bounds zero fill is the padding; `separable` != 0 asserts a
 *     rank-1 filter (two 4-tap passes; the caller tests this once per filter).  mode:
 *       0  out = B(in)                                                          (Blur, networks.py:70-86)
 *       1  o = lrelu(row_scale[n,c]*B(in) + noise_weight*noise[n,y,x] + bias[c], alpha)*scale   (networks.py:266,291-298,346-348)
 *          out = o (may be NULL) and/or out2 = o*scale2[n,c] (may be NULL): out2 is the NEXT modulated convolution's
 *          input with its style modulation applied (networks.py:236,243), written by the pass that produces o
 *       2  adjoint epilogue (backward of mode 1's blur): t = B(in); out = t*row_scale[n,c]; row_dot[n,c] = sum_yx t*mul[n,y,x,c]
 *          (mul: same shape as out; NULL row_dot: no reduction) -- `workspace` of gg_blur_nhwc_workspace() bytes
 *   workspaces: gg_nhwc_rowwise_workspace(N, C, HW) bytes for the optional reductions (row_dot (N, C); grad_bias (C)).
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_noise_bias_act_nhwc(void* out, const void* x, const float* noise, const float* noise_weight,
                                  const float* bias, const float* row_scale, int dtype, float alpha, float scale,
                                  int64_t N, int C, int64_t HW, void* stream);
GG_API int64_t gg_nhwc_rowwise_workspace(int64_t N, int C, int64_t HW);
GG_API int gg_channel_scale_nhwc(void* out, float* row_dot, void* workspace, const void* x, const void* y,
                                 const float* s, int dtype, int64_t N, int C, int64_t HW, void* stream);
GG_API int gg_bias_act_backward_nhwc(void* gx, float* grad_bias, void* workspace, const void* g,
                                     const void* out_saved, int dtype, float alpha, float scale, int64_t N, int C,
                                     int64_t HW, void* stream);
GG_API int64_t gg_blur_nhwc_workspace(int dtype, int64_t N, int C, int in_h, int in_w, int kernel_h, int kernel_w,
                                      int pad_x0, int pad_x1, int pad_y0, int pad_y1);
GG_API int gg_blur_nhwc(void* out, void* out2, const void* in, const float* kernel, const float* noise,
                        const float* noise_weight, const float* bias, const float* row_scale, const float* scale2,
                        const void* mul, float* row_dot, void* workspace, int dtype, int64_t N, int C, int in_h,
                        int in_w, int kernel_h, int kernel_w, int separable, int pad_x0, int pad_x1, int pad_y0,
                        int pad_y1, int mode, int act, float alpha, float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * StyledConv / ToRGB tails fused across layer boundaries (csrc/styled.cu), channels-last, dtype as above.
 * reference: models/stylegan2/networks.py:291-298 (NoiseInjection), :346-348 (StyledConv.forward), :236,243 (the style
 * modulation of the NEXT ModulatedConv2d, applied to its input here because conv(scale*W*s, x) == conv(scale*W, x*s)),
 * :389-405 (ToRGB: 1x1 modulated convolution without demodulation + bias + up-sampled skip).
 *   gg_styled_tail_nhwc:  o = act(demod[n,c]*raw + noise_weight*noise[n,p] + bias[c])*scale       raw: (N, HW, C)
 *        out = o                         (NULL: not written -- only a later backward pass needs it)
 *        xs  = o*s_next[n,c]             (NULL: not written)
 *        rgb[n,o3,p] = sum_c wm[n,o3,c]*o + rgb_bias[o3] + skip[n,o3,p]    (NULL: not computed; planar (N, 3, HW) fp32)
 *      C % 32 == 0 (fp32) / C % 64 == 0 (bf16).  One read of raw.
 *   gg_styled_tail_backward_nhwc: one pass over (g_xs, out[, raw]) ->
 *        g_o = g_xs*s_next + sum_o3 wm[n,o3,c]*g_rgb[n,o3,p];  g_t = act'(out)*scale*g_o;  g_raw = g_t*demod[n,c]
 *        d_s_next[n,c] = sum_p g_xs*out;  d_demod[n,c] = sum_p g_t*raw;  d_wm[n,o3,c] = sum_p g_rgb[n,o3,p]*out
 *      (each NULL: skipped; g_xs or g_rgb may be NULL; demod NULL: g_raw = g_t -- the blur layers apply demod in
 *      gg_blur_nhwc mode 2).  `workspace`: gg_styled_tail_backward_workspace() bytes.  Deterministic reductions.
 *      reduce_pitch: floats between consecutive samples of the sum outputs -- C (each a dense (N, C) / (N, 3, C) tensor) or
 *      R*C when they are the row slices [d_s_next | d_demod | d_wm x3] (requested ones only, in that order) of ONE (N, R, C)
 *      block, which is then finished by a single launch.
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_styled_tail_nhwc(void* out, void* xs, float* rgb, const void* raw, const float* noise,
                               const float* noise_weight, const float* bias, const float* demod, const float* s_next,
                               const float* wm, const float* rgb_bias, const float* skip, int dtype, int act,
                               float alpha, float scale, int64_t N, int C, int64_t HW, void* stream);
GG_API int64_t gg_styled_tail_backward_workspace(int dtype, int64_t N, int C, int64_t HW);
GG_API int gg_styled_tail_backward_nhwc(void* g_raw, float* d_s_next, float* d_demod, float* d_wm, void* workspace,
                                        const void* g_xs, const float* g_rgb, const void* out_saved, const void* raw,
                                        const float* s_next, const float* demod, const float* wm, int dtype,
                                        float alpha, float scale, int64_t N, int C, int64_t HW, int64_t reduce_pitch,
                                        void* stream);

/* to-RGB on channels-last activations (reference models/stylegan2/networks.py:389-405 `ToRGB.forward`: a 1x1 modulated
 * convolution without demodulation + bias + the up-sampled skip image; the reference builds B filter banks and runs a
 * grouped convolution).  One pass over the activation:
 *   out[n,o,p] = sum_i wm[n,o,i] * x[n,p,i] + bias[o] + skip[n,o,p]      x: (N, HW, C) NHWC; wm: (N, 3, C) fp32
 *   out, skip (optional), g: planar (N, 3, HW).  C % 32 == 0, C <= 1024.
 * backward: gx[n,p,i] = sum_o wm[n,o,i] g[n,o,p]  (NULL: skipped);  gwm[n,o,i] = sum_p g[n,o,p] x[n,p,i]  (NULL: skipped;
 * otherwise `workspace` of gg_to_rgb_nhwc_workspace(N, C, HW) bytes, deterministic two-stage reduction). */
GG_API int64_t gg_to_rgb_nhwc_workspace(int64_t N, int C, int64_t HW);
GG_API int gg_to_rgb_nhwc_forward(float* out, const float* x, const float* wm, const float* bias, const float* skip,
                                  int64_t N, int C, int64_t HW, void* stream);
GG_API int gg_to_rgb_nhwc_backward(float* gx, float* gwm, void* workspace, const float* g, const float* x,
                                   const float* wm, int64_t N, int C, int64_t HW, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Perceptual-loss front end (SURVEY.md 8(f) rank 2) on channels-last feature maps.
 * reference: models/losses/lpips.py:26-28 normalize_tensor, :193-195 squared difference, :197-205 per-channel `lins`
 * weights or plain channel sum, :226 spatial_average.
 *   out[n] = 1/HW * sum_p sum_c w[c] * (f0[n,p,c]/(|f0[n,p,:]|+eps) - f1[n,p,c]/(|f1[n,p,:]|+eps))^2
 * f0, f1 (and g0, g1): (N, HW, C) NHWC stored as `dtype` = GG_F32 or GG_BF16 (fp32 arithmetic, fp32 out / grad_out);
 * weight: (C) fp32 or NULL (= 1); C a power of two < 128, or a multiple of 128 up to 1024.
 * forward needs gg_feature_distance_workspace(N, C, HW) bytes (deterministic two-stage reduction).
 * backward: g0 / g1 (either may be NULL) = grad_out[n] * d out[n] / d f0 / d f1, one pass over both maps. */
GG_API int64_t gg_feature_distance_workspace(int64_t N, int C, int64_t HW);
GG_API int gg_feature_distance_forward(float* out, void* workspace, const void* f0, const void* f1,
                                       const float* weight, int dtype, int64_t N, int C, int64_t HW, float eps,
                                       void* stream);
GG_API int gg_feature_distance_backward(void* g0, void* g1, const float* grad_out, const void* f0, const void* f1,
                                        const float* weight, int dtype, int64_t N, int C, int64_t HW, float eps,
                                        void* stream);

/* VGG16 slice boundary of the perceptual loss: Conv2d -> ReLU -> [tap] -> MaxPool2d(2, 2) -> Conv2d
 * (reference models/losses/lpips_backbones.py:106-121 = torchvision vgg16().features 2-4, 7-9, 14-16, 21-23; ATen
 * threshold / max_pool2d_with_indices and their backwards).  One pass each on channels-last maps:
 *   forward : y = relu(raw + bias[c]) (N, H, W, C) and pooled = max over 2x2 windows, stride 2 (N, H/2, W/2, C)
 *   backward: grad_raw = [y > 0] * (grad_y + [pixel is the FIRST maximum of its window, row-major] * grad_pooled);
 *             grad_y / grad_pooled may be NULL (= 0).  No index map: the arg-max is recomputed from y with ATen's rule.
 * raw / y / pooled / grads: `dtype` = GG_F32 or GG_BF16; bias: (C) fp32 or NULL; C % (16 / sizeof(dtype)) == 0; H, W even. */
GG_API int gg_bias_relu_pool_nhwc_forward(void* y, void* pooled, const void* raw, const float* bias, int dtype, int64_t N,
                                          int C, int H, int W, void* stream);
GG_API int gg_bias_relu_pool_nhwc_backward(void* grad_raw, const void* grad_y, const void* grad_pooled, const void* y,
                                           int dtype, int64_t N, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------
 * BilinearDownsample (SURVEY.md 8(f) rank 1): reference models/spatial_transformers/antialiased_sampling.py:241-256 --
 * ReflectionPad2d(stride/2) + depthwise 1x2s conv, stride (1,s) + depthwise 2sx1 conv, stride (s,1).  One gather:
 *   out[m,oy,ox] = sum_i sum_j taps_v[c][i] taps_h[c][j] in[m, R(oy*s+i-p), R(ox*s+j-p)],  p = s/2, R = reflection
 * in: (N, C, in_h, in_w) fp32 NCHW; taps_h / taps_v: (C, 2*stride) (the module's `kernel_horz` / `kernel_vert` buffers);
 * out: (N, C, (in_h+2p-2s)/s+1, (in_w+2p-2s)/s+1).  backward = the exact adjoint, gather form (deterministic). */
GG_API int gg_tent_downsample_forward(float* out, const float* in, const float* taps_h, const float* taps_v, int64_t N,
                                      int C, int in_h, int in_w, int stride, void* stream);
GG_API int gg_tent_downsample_backward(float* grad_in, const float* grad_out, const float* taps_h, const float* taps_v,
                                       int64_t N, int C, int in_h, int in_w, int stride, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Point-transfer path (SURVEY.md 8(f) rank 4), csrc/points.cu + csrc/splat.cu.
 *   gg_nn_argmin: reference spatial_transformer.py:655-668 (`congeal_points` of a flow STN): index[n, p] = argmin over the
 *     HW entries of grid (N, HW, 2) of |p|^2 + |g|^2 - 2 g.p (the reference's expanded form and rounding; first minimum
 *     wins) for points (N, P, 2).  No (N, H, W, P) distance tensor; `workspace` of gg_nn_argmin_workspace(N, P) bytes.
 *   gg_splat2d_lookup_forward: reference spatial_transformer.py:141-157 (`uncongeal_points`: F.grid_sample of the sampling
 *     grid at the query points, 'border', align_corners=False; `unnormalize` :621-623) fused into gg_splat2d_forward's point
 *     load: query (N, P, 2) normalised congealed-frame coordinates, grid (N, grid_h, grid_w, 2); pixel coordinate =
 *     ((g / unnorm_k) / 2 + 0.5) * unnorm_m with unnorm_k = (res-1)/res, unnorm_m = out_res - 1; points_out (N, P, 2) or NULL
 *     receives the looked-up coordinates.  C <= 3.
 * ---------------------------------------------------------------------------------------------- */
GG_API int64_t gg_nn_argmin_workspace(int64_t N, int64_t P);
GG_API int gg_nn_argmin(int64_t* index, void* workspace, const float* grid, const float* points, int64_t N, int64_t P, int HW,
                        void* stream);
GG_API int gg_splat2d_lookup_forward(float* out, float* points_out, void* workspace, const float* input, const float* grid,
                                     const float* query, const float* values, const float* sigma, int64_t N, int64_t P,
                                     int C, int H, int W, int grid_h, int grid_w, float unnorm_k, float unnorm_m,
                                     int soft_normalize, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training-loop bookkeeping (SURVEY.md 8(f) rank 3), csrc/optim.cu.
 *   gg_adam_ema_step: reference train.py:126-134 -- torch.optim.Adam.step() for every parameter of both optimisers and the
 *     EMA `accumulate(t_ema, t_module)` (models/__init__.py:19-24) -- as one multi-tensor pass.
 *     table: DEVICE array of rows {float* p; const float* g; float* m; float* v; float* ema (may be NULL); int64 numel;
 *     const float* lr (device scalar)}; block_tensor / block_chunk: DEVICE int arrays of `blocks` entries mapping a CTA to
 *     (table row, chunk of `chunk` elements); state: DEVICE float[3] = {step, 1 - b1^step, sqrt(1 - b2^step)} -- the call
 *     increments step first (torch's default Adam arithmetic: m, v, step_size = lr/bc1, denom = sqrt(v)/sqrt(bc2) + eps).
 *   gg_tv_loss_forward/backward: reference models/losses/loss.py:4-12 total_variation_loss(delta_flow (N, H, W, 2)),
 *     reduce_batch=True: out[0] = mean huber|d/dy| + mean huber|d/dx|; backward is gather-form (deterministic).
 * ---------------------------------------------------------------------------------------------- */
GG_API int gg_adam_ema_step(const void* table, const int* block_tensor, const int* block_chunk, int blocks, int chunk,
                            float* state, double beta1, double beta2, double eps, double ema_decay, void* stream);
GG_API int64_t gg_tv_loss_workspace(int64_t N, int H, int W);
GG_API int gg_tv_loss_forward(float* out, void* workspace, const float* flow, int64_t N, int H, int W, void* stream);
GG_API int gg_tv_loss_backward(float* grad_flow, const float* grad_out, const float* flow, int64_t N, int H, int W,
                               void* stream);

/* Equalised-learning-rate weights of a whole network in one launch: reference networks.py:121-127 (EqualConv2d) and :146-149
 * (EqualLinear) multiply `self.weight * self.scale` inside every forward (and autograd multiplies again in every backward).
 *   for each table row t:  dst_t[i] = (dst dtype) (src_t[i] * scale_t),  i < numel_t
 * table: device array of rows {const void* src; void* dst; int64 numel; float scale; int32 dtypes = src_dtype | dst_dtype << 8}
 * (32 bytes; dtypes GG_F32 / GG_BF16); CTA b handles elements [block_chunk[b]*chunk, +chunk) of tensor block_tensor[b]
 * (chunk a multiple of 4).  Forward: fp32 master weights -> scaled weights in the convolution's dtype; backward: gradients of
 * the scaled weights -> fp32 gradients of the master weights. */
GG_API int gg_scale_cast_multi(const void* table, const int* block_tensor, const int* block_chunk, int blocks, int chunk,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GG_B200_H_ */
