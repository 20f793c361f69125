/*
 * pww_b200.h -- C ABI of the B200-native Paint-with-Words attention path (libpww_b200.so).
 *
 * The reference (cloneofsimo/paint-with-words-sd) has no FFI: its boundary is the Python callable
 * `inj_forward(self, hidden_states, context=None, mask=None)` that it monkey-patches over
 * diffusers' `CrossAttention.__call__` (paint_with_words/paint_with_words.py:60-125, 193-195).
 * These entry points replace the region of that function BETWEEN the q/k/v projections and the
 * output projection (paint_with_words.py:83-118); the Python shim
 * `paint_with_words_sd_b200.attention.inj_forward` keeps the reference calling convention and calls
 * them through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions: plain pointers and sizes, no torch types.  Every pointer is a DEVICE pointer owned by
 * the caller.  Calls enqueue work on `stream` (a cudaStream_t passed as void*) and return without
 * synchronising; they allocate nothing and are CUDA-graph capturable.  Return value: PWW_OK (0) or a
 * negative pww_status_t; nothing throws.  Unsupported (D, T) combinations return
 * PWW_ERR_UNSUPPORTED -- there is no fallback path inside or outside the library.
 *
 * Tensor layouts (fp16 = IEEE binary16):
 *   q, out : [B, N, H*D] fp16, element (b,n,h,d) at  b*q_batch_stride + n*q_row_stride + h*D + d
 *   k, v   : [B, T, H*D] fp16, element (b,t,h,d) at  b*k_batch_stride + t*k_row_stride + h*D + d
 *            (strides in ELEMENTS; the head slice of a row is contiguous -- no head permute/copy,
 *             unlike paint_with_words.py:83-85,118)
 *   wmap   : [Bw, N, T] fp32 dense weight maps, the reference's CROSS_ATTENTION_WEIGHT_{N} tensors
 *            (paint_with_words.py:255-268, 370-377) stacked along dim 0
 *   wmap_index : [B] int32, image b uses wmap[wmap_index[b]]; -1 = no bias for that image (the
 *            reference's uncond dict / tensor context, paint_with_words.py:107-110, 379-386, 493)
 */
#ifndef PWW_B200_H_
#define PWW_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  PWW_OK = 0,
  PWW_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, misaligned pointer/stride        */
  PWW_ERR_UNSUPPORTED = -2,  /* (D, T, H) outside the compiled kernel family                        */
  PWW_ERR_CUDA = -3,         /* a CUDA runtime/driver call failed; see pww_last_cuda_error()        */
  PWW_ERR_WORKSPACE = -4     /* workspace_bytes smaller than pww_xattn_workspace_bytes()            */
} pww_status_t;

#define PWW_STAT_MAX 0 /* qk.max()                       (paint_with_words.py:405) */
#define PWW_STAT_STD 1 /* qk.std(), unbiased (Bessel)    (README.md:129-152)       */

/* Library version: major*10000 + minor*100 + patch. */
int pww_version(void);

/* Static string for a status code. */
const char* pww_status_str(int status);

/* cudaGetErrorString of the last CUDA failure seen by this library on the calling thread ("" if none). */
const char* pww_last_cuda_error(void);

/* 1 if the running device is compute capability 10.x (the only target), 0 otherwise, <0 on error. */
int pww_device_supported(void);

/* Bytes of scratch `pww_xattn_stats_f16` needs for this problem size.  The scratch must be zero-filled
 * ONCE after allocation (cudaMemset); calls leave it zeroed again (self-cleaning arrival counters). */
size_t pww_xattn_workspace_bytes(int B, int H, int N, int T, int D);

/*
 * Per-image statistic of the UNSCALED score tensor S[b] = Q_h K_h^T over all heads, pixels and tokens
 * (one scalar per image per call -- what `qk.max()` / `qk.std()` evaluate to inside the reference's
 * weight_function, paint_with_words.py:87,106,402-405).  S is rounded to fp16 before the reduction, as
 * the reference's autocast matmul does; the result is rounded to fp16 and stored as float.
 * Images with wmap_index[b] < 0 are skipped (stats[b] = 0).  wmap_index may be NULL (= all images).
 */
int pww_xattn_stats_f16(const void* q, const void* k,
                        int B, int H, int N, int T, int D,
                        int64_t q_batch_stride, int64_t q_row_stride,
                        int64_t k_batch_stride, int64_t k_row_stride,
                        int stat, const int32_t* wmap_index,
                        float* stats /* [B] out */,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * Fused cross-attention with the Paint-with-Words bias (paint_with_words.py:87-118):
 *   P[b,h,n,:] = softmax_t( scale * ( S[b,h,n,t] + g_sigma[0] * stats[b] * wmap[wmap_index[b]][n,t] ) )
 *   out[b,n,h,:] = sum_t P[b,h,n,t] * V[b,t,h,:]
 * `g_sigma` is a 1-element device array holding G(sigma) = coef*ln(1+sigma^p) for this step (a device
 * scalar so a captured CUDA graph can be replayed with a new sigma).  wmap/wmap_index/stats/g_sigma may
 * all be NULL: plain cross-attention (tensor context, paint_with_words.py:67-69,107-108).
 * Requires T <= 80 (Stable Diffusion's 77-token context).
 */
int pww_xattn_fwd_f16(const void* q, const void* k, const void* v, void* out,
                      int B, int H, int N, int T, int D,
                      int64_t q_batch_stride, int64_t q_row_stride,
                      int64_t k_batch_stride, int64_t k_row_stride,
                      int64_t o_batch_stride, int64_t o_row_stride,
                      const float* wmap, int64_t wmap_batch_stride, const int32_t* wmap_index,
                      const float* stats, const float* g_sigma, float scale, void* stream);

/*
 * ONE-LAUNCH Paint-with-Words cross-attention: statistic + bias + softmax + P.V (paint_with_words.py:87-118 with the
 * weight function of paint_with_words.py:402-405 inlined).  Replaces the pww_xattn_stats_f16 + pww_xattn_fwd_f16 pair:
 * the per-image statistic is reduced inside the kernel (cooperative launch, deterministic fixed-order reduction of
 * per-CTA partials) and the bias enters as two extra k-steps of the Q K^T tensor-core chain.
 *
 * The weight map is passed in PACKED form (SURVEY 8f-4).  The reference's dense [N, T] fp32 map
 * (paint_with_words.py:255-272) has one distinct non-zero column per painted region, so it is a column dictionary
 *     W[n, t] = Mu[n, cidx[t]]       Mu [N, R] fp32, R <= 10 distinct columns; cidx[t] = -1 for an all-zero column
 *   mpack : [Bw, N, 32] fp16, row n = [ hi(Mu[n,0..9]) | lo(Mu[n,0..9]) | hi(Mu[n,0..9]) | 0 0 ] with
 *           hi(x) = fp16(x), lo(x) = fp16(x - hi(x));  64 bytes per pixel instead of 308
 *           (element (w,n,c) at w*mpack_batch_stride + n*32 + c; 16-byte aligned)
 *   cidx  : [Bw, 80] int8, dictionary column of token t (0..9) or -1 (also for t >= T)
 * `paint_with_words_sd_b200.conditioning.pack_weight_map` builds both, bit-exactly reversible to the dense map.
 * Maps with more than 10 distinct columns use the two-launch dense path above.
 *
 *   stats [B] out : the per-image statistic (fp16-rounded, as float; 0 for images without a map); may be NULL
 *   workspace     : pww_xattn_fused_workspace_bytes() bytes, zero-filled ONCE after allocation (self-cleaning)
 * mpack == NULL (or every wmap_index[b] < 0): plain cross-attention, workspace may be NULL.
 * Requires T <= 80, B <= 32 per launch (larger batches are split internally), 16-byte aligned `out` strides.
 */
size_t pww_xattn_fused_workspace_bytes(void);
int pww_xattn_fused_f16(const void* q, const void* k, const void* v, void* out,
                        int B, int H, int N, int T, int D,
                        int64_t q_batch_stride, int64_t q_row_stride,
                        int64_t k_batch_stride, int64_t k_row_stride,
                        int64_t o_batch_stride, int64_t o_row_stride,
                        const void* mpack, int64_t mpack_batch_stride, int Bw, const int8_t* cidx,
                        const int32_t* wmap_index, int stat, const float* g_sigma, float scale,
                        float* stats, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Self-attention through the same patched function (context=None, paint_with_words.py:71-72):
 *   out = softmax(scale * Q_h K_h^T) V_h  with keys/values [B, N, H*D]; no bias; online softmax.
 */
int pww_attn_fwd_f16(const void* q, const void* k, const void* v, void* out,
                     int B, int H, int N, int D,
                     int64_t qkv_batch_stride, int64_t qkv_row_stride,
                     int64_t o_batch_stride, int64_t o_row_stride,
                     float scale, void* stream);

/*
 * Fused memory-bound ops of the UNet that calls the attention path (the reference gets them from diffusers/ATen as
 * separate eager launches): channels-last fp16 activations, deterministic reductions.
 *
 * GroupNorm over [B, HW, C] (channels last) with G groups:  y = act((x + add[b,c] - mean) * rstd * gamma + beta),
 * `add` ([B, C] with row stride `add_batch_stride`, may be NULL) is the ResNet block's time-embedding term (added before normalisation), act = SiLU when
 * `silu` != 0.  Needs C % 8 == 0, C % G == 0, G <= 64 and pww_groupnorm_workspace_bytes() of scratch that was
 * zero-filled once after allocation (self-cleaning arrival counters, like the attention statistics workspace).
 */
size_t pww_groupnorm_workspace_bytes(int B, int HW, int G);
int pww_groupnorm_nhwc_f16(const void* x, const void* add, int64_t add_batch_stride /* elements */,
                           const void* gamma, const void* beta, void* y,
                           int B, int HW, int C, int G, float eps, int silu,
                           void* workspace, size_t workspace_bytes, void* stream);

/* GEGLU: out[m, i] = in[m, i] * gelu(in[m, I + i]) for in [M, 2*I], out [M, I] (exact erf GELU); I % 8 == 0. */
int pww_geglu_f16(const void* in, void* out, int64_t M, int I, void* stream);

/* Residual add + LayerNorm over the last dim of [M, C]:  s = x + res (res may be NULL);  sum_out = s (may be NULL);
 * y = LayerNorm(s) * gamma + beta.  The transformer block's "x = attn(...) + x; h = norm(x)" pair in one pass.
 * C % 8 == 0, C <= 2048. */
int pww_add_layernorm_f16(const void* x, const void* res, const void* gamma, const void* beta, void* sum_out, void* y,
                          int64_t M, int C, float eps, void* stream);

/*
 * Sampler step of the Euler, Euler-ancestral and DPM-Solver++(2M) schedulers (paint_with_words_sd_b200/scheduler.py),
 * around the UNet forward of one denoising step of m images.  Each of them updates the latents as
 *     eps = eps_u + g * (eps_c - eps_u),  x0 = x - sigma * eps,
 *     x'  = a * x + b * eps + c * x0 + d * x0_prev + s * xi,  x0_prev <- x0
 * with per-step scalars read from a DEVICE coefficient row `coef` of 12 fp32 (so a CUDA graph replays each step with
 * new values after a copy into the row):
 *     coef[0] sigma   coef[1] c_in = 1/sqrt(sigma^2+1)   coef[2] UNet timestep   coef[3..7] a, b, c, d, s
 *     coef[8] G(sigma) (read by the attention path)   coef[9] absolute step index (for the noise)   coef[10..11] unused
 * Latent-shaped fp32 tensors are NCHW contiguous.
 */

/* UNet input of a step: out [2m, C+Ce, H, W] fp16 CHANNELS-LAST (element (n,c,y,x) at ((n*H + y)*W + x)*(C+Ce) + c),
 * rows n and n+m both = cat(c_in * latents[n], extra[n]) rounded to fp16.  latents [m, C, H, W] fp32; extra
 * [m, Ce, H, W] fp32 (e.g. the inpaint mask and masked-image latents), NULL iff Ce == 0.  C + Ce <= 16. */
int pww_sampler_prepare_f16(const float* latents, const float* extra, const float* coef, void* out,
                            int m, int C, int Ce, int H, int W, void* stream);

/* CFG combine + sampler update.  eps: the UNet output [2m, C, H, W] fp16 (cond rows 0..m-1, uncond rows m..2m-1) at
 * the given element strides (any layout, e.g. channels-last).  latents and x0_prev [m, C, H, W] fp32 are updated in
 * place.  seeds [m]: the noise seed of each image; xi is pww_randn_f32(seed, step) of that image (drawn only when
 * coef[7] != 0). */
int pww_sampler_step_f32(const void* eps, int64_t eps_n_stride, int64_t eps_c_stride, int64_t eps_h_stride,
                         int64_t eps_w_stride, float* latents, float* x0_prev, const float* coef,
                         const uint64_t* seeds, float guidance_scale, int m, int C, int H, int W, void* stream);

/* n standard normals: Philox4x32-10 keyed by `seed`, counter (element / 4, step), Box-Muller.  out[e] is the noise
 * pww_sampler_step_f32 adds to element e (NCHW index within the image) of an image with this seed at this step; it
 * depends on nothing else (not on batch position, batch size or device). */
int pww_randn_f32(float* out, int64_t n, uint64_t seed, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PWW_B200_H_ */
