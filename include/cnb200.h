/*
 * cnb200.h - C ABI of the B200-native ControlNet denoising hot path (libcnb200.so).
 *
 * The reference (henriChevreux/ControlNet-PyTorch) has no FFI / plugin boundary: every FLOP of the path is an
 * ATen library call issued from Python nn.Modules (SURVEY.md section 2.1).  This header therefore declares one
 * entry point per ATen call site class of the path; each comment names the reference lines it replaces.  The
 * Python drop-in modules in controlnet-pytorch_b200/{models,scheduler}/ bind these with ctypes
 * (controlnet-pytorch_b200/runtime.py) and pass raw device pointers + the current CUDA stream.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; activations are fp32, channels-last
 *     ("NHWC": [B, H, W, ld] with a channel offset/leading dimension so concatenations are free);
 *   - every function returns 0 on success or a negative CNB_ERR_* code; cnb_last_error() gives the text;
 *   - functions only enqueue work on `stream` (a cudaStream_t); they never synchronise and never allocate,
 *     so a whole denoising step can be captured into a CUDA graph;
 *   - there is no CPU fallback anywhere: without a CUDA device every compute entry point fails with CNB_ERR_CUDA.
 */
#ifndef CNB200_H
#define CNB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CNB_OK 0
#define CNB_ERR_BAD_ARG (-1)
#define CNB_ERR_CUDA (-2)
#define CNB_ERR_UNSUPPORTED (-3)
#define CNB_ERR_TIMEOUT (-4)

#define CNB_MAX_TAPS 16

/* compute modes of the GEMM-class entry points */
#define CNB_MODE_F32 0   /* CUDA-core FFMA, exact fp32 ("fp32 mode", 1e-4 gate)                      */
#define CNB_MODE_F16 1   /* tensor-core mode: tcgen05.mma kind::f16 on fp16 operands (fp16 activation stream), kind::tf32
                          * where a tensor is still fp32; fp32 accumulate in TMEM, fp32 statistics ("f16 mode", 1e-2 gate).
                          * There is no bf16 mode: bf16 operands miss the 1e-2 gate on the MNIST widths (SURVEY App. D). */

typedef void* cnb_stream_t; /* cudaStream_t */

int cnb_abi_version(void);
/* sizeof(cnb_conv_params) as compiled into the library (bindings assert their mirror struct against it). */
int cnb_sizeof_conv_params(void);
const char* cnb_last_error(void);
/* Number of kernels this library has launched since load / last reset (bench.py's gpu_launches). */
long long cnb_launch_count(void);
void cnb_reset_launch_count(void);
/* 1 if the current device is sm_100 class and the tcgen05 path may be used. */
int cnb_has_tcgen05(void);

/*
 * Implicit-GEMM convolution / linear layer with fused epilogue.
 *   out[b, oy*oy_mul+oy_add, ox*ox_mul+ox_add, out_coff+n] =
 *        act( sum_{tap,c} W[n][tap][c] * in[b, oy*stride+dy[tap], ox*stride+dx[tap], in_coff+c]   (0 outside)
 *             [+ sum_c W[n][ntaps][c] * in2[b, oy, ox, in2_coff+c]]
 *             + bias[n] + temb[(temb_per_sample ? b : 0)*temb_ld + n] + residual[b, oy', ox', res_coff+n] )
 * Replaces nn.Conv2d 3x3/1x1/4x4s2/3x3s2 (models/unet_base.py:49,67,84,88,131,149,166,220,238,259,320,339;
 * models/blocks.py:54,73,112,...; models/controlnet.py:70-106; models/controlnet_ldm.py:48-96), one output-parity
 * phase of nn.ConvTranspose2d 4x4 s2 p1 (unet_base.py:263, blocks.py:461), nn.Linear inside nn.MultiheadAttention
 * (in_proj / out_proj, unet_base.py:79,107), the "+ t_emb_layers(t_emb)[:, :, None, None]" add (unet_base.py:98),
 * the "+ residual_input_conv(resnet_input)" add (:100), the "+ out_attn" add (:109) and the zero-conv injections
 * (controlnet.py:184,207,216-218).
 */
typedef struct cnb_conv_params {
  const void* in;         /* [B, H, W, ldi] fp32 (in_dtype 0) or fp16 (in_dtype 1) */
  const float* weight;    /* [Cout][ntaps][Cin] fp32 (cnb_pack_* output)      */
  const void* weight_lp;  /* fp16 copy of `weight`, required when in_dtype==1 */
  const float* bias;      /* [Cout] or NULL                                   */
  const float* temb;      /* [(B|1), temb_ld] or NULL                         */
  const void* residual;   /* [B, OHf, OWf, ldr] fp32 (res_dtype 0) or fp16 (res_dtype 1), or NULL */
  void* out;              /* [B, OHf, OWf, ldo] fp32 (out_dtype 0) or fp16 (out_dtype 1) */
  int32_t B, H, W, Cin, ldi, in_coff;
  int32_t OH, OW;         /* output grid that is iterated                     */
  int32_t OHf, OWf;       /* full spatial size of `out` / `residual`          */
  int32_t oy_mul, oy_add, ox_mul, ox_add;
  int32_t Cout, ldo, out_coff;
  int32_t ldr, res_coff;
  int32_t stride;
  int32_t ntaps;
  int8_t dy[CNB_MAX_TAPS];
  int8_t dx[CNB_MAX_TAPS];
  int32_t temb_ld, temb_per_sample;
  int32_t act;            /* 0 = none, 1 = SiLU on the result                 */
  int32_t mode;           /* CNB_MODE_*                                       */
  int32_t in_dtype;       /* 0 = fp32 activations, 1 = fp16 activations (tensor-core modes only) */
  int32_t out_dtype;      /* 0 = fp32 `out`, 1 = fp16 `out` (ldo / out_coff stay in elements; tensor-core modes only) */
  int32_t res_dtype;      /* 0 = fp32 `residual`, 1 = fp16 `residual` (ldr / res_coff in elements)                   */
  /* Optional second input, contracted with one extra (0,0) tap: [B, OH, OW, ldi2] of `in`'s dtype; the packed weight
   * rows are then [ntaps*Cin | Cin2] long.  This is how "+ residual_input_conv(resnet_input)" (unet_base.py:100) is
   * folded into the second 3x3 convolution of a resnet block as extra K.  NULL when unused; tcgen05 path only. */
  const void* in2;
  int32_t Cin2, ldi2, in2_coff;
} cnb_conv_params;

int cnb_conv2d(const cnb_conv_params* p, cnb_stream_t stream);

/* The kernel route cnb_conv2d takes for `p` on the current device, without launching anything: route[] receives
 * CNB_ROUTE_LEN values indexed by CNB_ROUTE_* (fields that do not apply to the path are 0).  Returns the error
 * cnb_conv2d would return before its launch.  cnb_conv2d makes the same decision in the same code, so tests can name
 * the variant a call site reaches and check that a replay of it reaches the same one. */
#define CNB_ROUTE_LEN 16
#define CNB_PATH_F32 0     /* CUDA-core fp32 implicit GEMM (conv_f32.cu)          */
#define CNB_PATH_SMALL 1   /* direct kernels for Cin <= 4 or Cout <= 4 (conv_small.cu) */
#define CNB_PATH_TMA 2     /* TMA-fed tcgen05 kernel (conv_tma.cu)                */
#define CNB_ROUTE_PATH 0         /* CNB_PATH_*                                                   */
#define CNB_ROUTE_RB 1           /* TMA: bytes of K per smem row (swizzle span 32 / 64 / 128)    */
#define CNB_ROUTE_BN 2           /* TMA: N tile after N-split narrowing                           */
#define CNB_ROUTE_EPI 3          /* TMA: epilogue variant 0..6 (conv_tma_impl.cuh)                */
#define CNB_ROUTE_HALO 4         /* TMA: 1 = halo mode (3x3 bands loaded once per channel chunk)  */
#define CNB_ROUTE_BRES 5         /* TMA: 1 = weights resident in shared memory                    */
#define CNB_ROUTE_CTAS_PER_SM 6  /* TMA: 1 or 2                                                   */
#define CNB_ROUTE_EPI_ALT 7      /* TMA: 1 = the epilogue warp groups alternate tiles             */
#define CNB_ROUTE_EPI_NBUF 8     /* TMA, EPI 6: staging buffers per epilogue warp (2 or 3)        */
#define CNB_ROUTE_GRID 9         /* TMA: CTAs launched (tile = blockIdx.x + k * grid)             */
#define CNB_ROUTE_NTILES 10      /* TMA: tiles_m * tiles_n                                        */
#define CNB_ROUTE_TILES_N 11     /* TMA: N tiles per M tile (tile = m_tile * tiles_n + n_tile)    */
#define CNB_ROUTE_HALO_R 12      /* TMA, halo: image rows per band                                */
#define CNB_ROUTE_TILES_Y 13     /* TMA, halo: bands per sample (sample = tile / tiles_y)         */
int cnb_conv2d_route(const cnb_conv_params* p, int32_t* route);

/* OIHW -> [O][KH*KW][I] (tap = ky*KW+kx).  round_tf32 != 0 rounds to nearest tf32 (for CNB_MODE_F16). */
int cnb_pack_conv_weight(const float* w_oihw, float* dst, int O, int I, int KH, int KW, int round_tf32,
                         cnb_stream_t stream);
/* ConvTranspose2d weight (I, O, 4, 4), stride 2, pad 1 -> [4 phases (py*2+px)][O][4 taps (a*2+b)][I]
 * with the taps of SURVEY.md Appendix F: T(0) = {(ky=1,dy=0),(ky=3,dy=-1)}, T(1) = {(ky=0,dy=+1),(ky=2,dy=0)}. */
int cnb_pack_convT_weight(const float* w_iohw, float* dst, int I, int O, int round_tf32, cnb_stream_t stream);
/* fp32 -> fp16 (round to nearest even) */
int cnb_cast_f16(const float* src, void* dst, long long n, cnb_stream_t stream);

/*
 * GroupNorm (+ optional SiLU) over channels-last activations: x, y are [B, HW, C] contiguous; x is fp32, or fp16
 * when in_f16 != 0 (the fp16 activation stream of the tensor-core modes); y is fp32, or fp16 when out_f16 != 0 (the
 * operand type of the kind::f16 tensor-core convolution that consumes it).  Statistics are always fp32.
 * Replaces nn.GroupNorm(G, C) [+ nn.SiLU] (unet_base.py:47-48,65-66,74,104-105,338 + :372; eps = 1e-5,
 * biased variance, per-channel affine).
 */
int cnb_groupnorm(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
                  float eps, int silu, int in_f16, int out_f16, cnb_stream_t stream);
/* Large samples (fp16 slab of HW * C * 2 bytes beyond one CTA's shared memory: the VAE decoder's 64x64 / 128x128
 * levels, vae.py:102-114 through blocks.py:347-374) are normalised by a split-statistics + apply kernel pair that
 * needs a scratch buffer: cnb_groupnorm_workspace_bytes returns its size (0: cnb_groupnorm's one-CTA-per-sample
 * kernels are the right ones), cnb_groupnorm_ws takes it (workspace == NULL behaves like cnb_groupnorm). */
size_t cnb_groupnorm_workspace_bytes(int B, int HW, int C, int G, int in_f16);
int cnb_groupnorm_ws(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
                     float eps, int silu, int in_f16, int out_f16, void* workspace, size_t ws_bytes, cnb_stream_t stream);

/*
 * Self-attention core on packed projections: qkv is [B, L, 3E] (q | k | v, heads split along E), out is [B, L, E].
 * out = concat_h softmax(Q_h K_h^T / sqrt(E/heads)) V_h.   Replaces the core of nn.MultiheadAttention
 * (unet_base.py:107; no mask, no dropout, attention weights discarded).
 */
int cnb_attention(const float* qkv, float* out, int B, int L, int E, int heads, int mode, cnb_stream_t stream);
/* Same contraction on fp16 operands: qkv [B, L, 3E] fp16 (as the in_proj convolution emits it with out_dtype 1),
 * out [B, L, E] fp16 (the A operand of the out_proj convolution); fp32 softmax statistics and accumulators.
 * Dispatches to cnb_attention_tmem for every head dim that kernel instantiates (CNB_ATTN_TMEM=0: never), else to
 * cnb_attention_mma. */
int cnb_attention_f16(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream);
/* The tcgen05 / TMEM flash-attention kernel (csrc/attention_tmem.cu; head dim 4, 8, 16, 24, 32, 48 or 64):
 * S = Q K^T as tcgen05.mma tiles fed by TMA, S / P / O resident in tensor memory (P is the A operand of the second MMA
 * straight from TMEM), thread-per-row online softmax with lazy rescale, denominator accumulated by the tensor core. */
int cnb_attention_tmem(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream);
/* The register-resident mma.sync (m16n8k16) flash-attention kernel (csrc/attention_f16.cu): head dims the TMEM kernel
 * does not instantiate (96, 128, 192: CelebHQ-latent students) and the comparison arm of the kernel tests. */
int cnb_attention_mma(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream);

/* y[r, n] = post( sum_k pre(x[r, k]) * w[n, k] + b[n] ), pre/post = SiLU if the flag is set.  x is [R, K]
 * contiguous, y has leading dimension ldy.   Replaces Unet.t_proj (unet_base.py:313-317), the per-block
 * t_emb_layers SiLU->Linear (unet_base.py:55-61) and the students' t_proj (consistency_...py:35-38). */
int cnb_linear_small(const float* x, const float* w, const float* b, float* y, int R, int K, int N, int ldy,
                     int silu_in, int silu_out, cnb_stream_t stream);

/* out[i, :] = [sin(t_i / factor) | cos(t_i / factor)], factor is the fp32 table 10000^(j/(D/2)), j < D/2
 * (get_time_embedding, unet_base.py:5-28). */
int cnb_time_embedding(const int64_t* t, const float* factor, float* out, int n, int D, cnb_stream_t stream);

/*
 * LinearNoiseScheduler.sample_prev_timestep (scheduler/linear_noise_scheduler.py:49-77), evaluated in the
 * reference's fp32 operation order (no FMA contraction).  coef (device, 6 floats):
 *   [0] sqrt_one_minus_alpha_cum_prod[t]  [1] sqrt(alpha_cum_prod[t])  [2] betas[t]  [3] sqrt(alphas[t])
 *   [4] sigma_t  [5] 1.0 if t > 0 (noise is added) else 0.0
 * z may be NULL: the noise is then Philox4x32-10 + Box-Muller keyed by (seed, step, elem_offset + i), i.e. by the
 * GLOBAL element index, so results do not depend on how the batch is sharded over GPUs.  x0 may be NULL.
 * If step_dev != NULL the Philox step is read from the device (step_dev[0]) so a captured CUDA graph of one
 * denoising step can be replayed for every timestep.
 */
int cnb_sched_step(const float* xt, const float* eps, const float* z, float* xt_prev, float* x0, long long n,
                   const float* coef, uint64_t seed, uint64_t step, const int32_t* step_dev, uint64_t elem_offset,
                   cnb_stream_t stream);
/*
 * One DDIM update (scheduler/ddim_scheduler.py; no counterpart in the reference).  For step k of the timesteps
 * tau_0 > ... > tau_{S-1}, with a_t = alpha_cum_prod[tau_k] and a_p = alpha_cum_prod[tau_{k+1}] (1.0 at the last step),
 * coef (device, 6 floats) holds
 *   [0] sqrt_one_minus_alpha_cum_prod[tau_k]  [1] sqrt_alpha_cum_prod[tau_k]  [2] sqrt(a_p)
 *   [3] sqrt(max(1 - a_p - sigma^2, 0))  [4] sigma  [5] 1.0 if sigma > 0 (noise is added) else 0.0
 * where sigma = eta * sqrt((1 - a_p) / (1 - a_t)) * sqrt(1 - a_t / a_p).  Per element, fp32, no FMA contraction:
 *   x0 = (xt - c0 * eps) / c1   (the operations of cnb_sched_step's x0, so that x0 is bit-identical to it)
 *   x_prev = c2 * (clip_sample ? clamp(x0, -1, 1) : x0) + c3 * eps  (+ c4 * z when c5 != 0)
 * and the x0 output is clamp(x0, -1, 1).  z, x0, seed, step, step_dev and elem_offset behave as in cnb_sched_step:
 * z == NULL draws the same Philox stream, keyed by (seed, step, elem_offset + i); x0 may be NULL; xt_prev may alias xt.
 */
int cnb_ddim_step(const float* xt, const float* eps, const float* z, float* xt_prev, float* x0, long long n,
                  const float* coef, int clip_sample, uint64_t seed, uint64_t step, const int32_t* step_dev,
                  uint64_t elem_offset, cnb_stream_t stream);
/*
 * One DPM-Solver++ multistep update (scheduler/dpm_solver_scheduler.py; no counterpart in the reference).  Step k of
 * the timesteps tau_0 > ... > tau_{S-1} goes from s = tau_k to t = tau_{k+1} (to alpha_cum_prod = 1 after the last
 * step), with alpha = sqrt(alpha_cum_prod), sigma = sqrt(1 - alpha_cum_prod), lambda = log(alpha / sigma),
 * h_k = lambda_t - lambda_s, r_k = h_{k-1} / h_k and e^{-h} = (sigma_t alpha_s) / (alpha_t sigma_s).  coef (device,
 * 6 floats) holds
 *   [0] sqrt_one_minus_alpha_cum_prod[tau_k]  [1] sqrt_alpha_cum_prod[tau_k]  [2] A  [3] B0  [4] B1  [5] C
 * where, with F = alpha_t (1 - e^{-h}) for variant "ode" and F = alpha_t (1 - e^{-2h}) for "sde",
 *   A = sigma_t / sigma_s ("ode") or (sigma_t / sigma_s) e^{-h} ("sde");  C = 0 ("ode") or sigma_t sqrt(1 - e^{-2h})
 *   first order (the first step, the last step, order 1):  B0 = F, B1 = 0
 *   second order (2M, midpoint):  B0 = F (1 + 1 / (2 r_k)),  B1 = -F / (2 r_k).
 * Per element, fp32, no FMA contraction:
 *   v = (xt - c0 * eps) / c1   (the operations of cnb_sched_step's x0, so that x0 is bit-identical to it)
 *   D = clip_sample ? clamp(v, -1, 1) : v
 *   x_prev = A * xt + B0 * D  (+ B1 * hist when B1 != 0)  (+ C * z when C != 0);  hist = D
 * and the x0 output is clamp(v, -1, 1).  hist (n floats, not overlapping xt, xt_prev or x0) carries the data
 * prediction D from one step to the next; it is read only when B1 != 0, so the first step may pass an uninitialised
 * buffer.  z, x0, seed, step, step_dev and elem_offset behave as in cnb_sched_step: z == NULL draws the same Philox
 * stream; x0 may be NULL; xt_prev may alias xt.
 */
int cnb_dpm_solver_step(const float* xt, const float* eps, const float* z, float* hist, float* xt_prev, float* x0,
                        long long n, const float* coef, int clip_sample, uint64_t seed, uint64_t step,
                        const int32_t* step_dev, uint64_t elem_offset, cnb_stream_t stream);
/*
 * Image-to-image start (sampler.DDPMSampler.img2img; the forward diffusion of LinearNoiseScheduler.add_noise).  Per
 * element, fp32, no FMA contraction, in add_noise's operation order (mul, mul, add):
 *   out = sqrt_acp * x_ref + sqrt_one_minus * z
 * so with the base scheduler's fp32 sqrt_alpha_cum_prod[t] / sqrt_one_minus_alpha_cum_prod[t] the result is
 * add_noise(x_ref, z, t) bit for bit.  z == NULL draws the Philox stream of cnb_sched_step keyed by
 * (seed, step, elem_offset + i).  out may alias x_ref (and must not overlap it otherwise).  16-byte aligned pointers.
 */
int cnb_add_noise(const float* x_ref, const float* z, float* out, long long n, float sqrt_acp, float sqrt_one_minus,
                  uint64_t seed, uint64_t step, uint64_t elem_offset, cnb_stream_t stream);
/*
 * Inpainting blend (sampler.DDPMSampler.img2img with a mask), in place on x (NCHW fp32, n = B * C * HW elements).
 * k = step_dev ? step_dev[0] : step selects row k of levels, a device fp32 [n_steps, 2] table, as (a, s).  Per element,
 * fp32, separate IEEE operations:
 *   known = a * x_ref + s * z                      (cnb_add_noise's operation order)
 *   x     = m == 1 ? x : (m == 0 ? known : (m * x) + ((1 - m) * known))
 * so m == 1 leaves x unchanged bit for bit and m == 0 writes known exactly.  m is mask[b, c, p] with mask shaped
 * [B, mask_c, HW] and mask_c == C, or mask[b, 0, p] with mask_c == 1 (broadcast over the channels).  1 means
 * "generate", 0 means "keep the reference".  z == NULL draws the Philox stream keyed by (seed, noise_step,
 * elem_offset + i).  x must not overlap x_ref or mask; 16-byte aligned pointers.
 */
int cnb_inpaint_blend(float* x, const float* x_ref, const float* mask, const float* z, long long n, int C,
                      long long HW, int mask_c, const float* levels, long long step, const int32_t* step_dev,
                      uint64_t seed, uint64_t noise_step, uint64_t elem_offset, cnb_stream_t stream);
/* out[p, oy, ox] = max over in[p, oy*f + dy, ox*f + dx], 0 <= dy, dx < f, for B planes of H x W (H and W divisible by
 * f): an image-space inpainting mask on the latent grid, a latent cell touching any repainted pixel repainted. */
int cnb_mask_max_pool(const float* in, float* out, int B, int H, int W, int f, cnb_stream_t stream);
/* Fill out[i] with the same N(0,1) stream as cnb_sched_step (used for x_T and by tests). */
int cnb_philox_normal(float* out, long long n, uint64_t seed, uint64_t step, uint64_t elem_offset,
                      cnb_stream_t stream);
/* Start of a replayed denoising step: k = step_idx[0]; t_out[0] = t_seq[k] (int64, what the model's
 * time-embedding reads); coef_out[0..6) = coef_table[t_seq[k]][0..6) (what cnb_sched_step reads). */
int cnb_sampler_prologue(const int32_t* step_idx, const int64_t* t_seq, int64_t* t_out, const float* coef_table,
                         float* coef_out, cnb_stream_t stream);
/* idx[0] += delta (device-side step counter of a replayed graph) */
int cnb_bump_index(int32_t* idx, int delta, cnb_stream_t stream);

/* EDM pre-conditioning of the consistency student (consistency_controlnet_distilled.py:45-74,91-98):
 * coef is [4][B]: c_in, c_skip, c_out, (float) clamp(trunc(1000 * 0.25 * ln(max(sigma,1e-8))), 0, 999);
 * flag[0] = 1 if all(sigma <= sigma_min) (the early-return test at :81). */
int cnb_edm_coeffs(const float* sigma, int B, float sigma_data, float sigma_min, float* coef, int64_t* t_index,
                   int32_t* flag, cnb_stream_t stream);
/* out[b, i] = a[b] * x[b, i] (+ c[b] * y[b, i] if y != NULL); per-sample scalars (consistency :92, :132). */
int cnb_scale_rows(const float* a, const float* x, const float* c, const float* y, float* out, int B,
                   long long per_sample, cnb_stream_t stream);
/* The same two expressions fused with the layout change around the student body (:92 -> conv_in, conv_out -> :132):
 * dst (NHWC fp32) = a[b] * src (NCHW fp32);   dst (NCHW fp32) = c_skip[b] * x (NCHW fp32) + c_out[b] * f, f the
 * channels-last body output (fp32 or fp16, leading dimension ldi, channel offset in_coff).  Bit-identical to
 * cnb_scale_rows composed with cnb_nchw_to_nhwc / cnb_nhwc_to_nchw. */
int cnb_scale_nchw_to_nhwc(const float* a, const float* src, float* dst, int B, int C, int HW, cnb_stream_t stream);
int cnb_edm_combine_to_nchw(const float* c_skip, const float* x, const float* c_out, const void* f, int ldi, int in_coff,
                            float* dst, int B, int C, int HW, int f_f16, cnb_stream_t stream);
/* Teacher-side x0 from a noise prediction with per-sample timesteps (distribution_matching_controlnet.py:191-216,
 * consistency_controlnet_distilled.py:201-228): out = clamp((xt - sqrt_one_minus[t_b] * eps) / sqrt_alpha[t_b], -1, 1);
 * t holds t_count in {1, B} int64 indices < num_timesteps into the two scheduler tables (device fp32). */
int cnb_x0_from_eps(const float* xt, const float* eps, const float* sqrt_one_minus, const float* sqrt_alpha,
                    const int64_t* t, int t_count, int num_timesteps, float* out, int B, long long per_sample,
                    cnb_stream_t stream);

/* layout plumbing between the reference's NCHW tensors and the channels-last workspace */
int cnb_nchw_to_nhwc(const float* src, float* dst, int B, int C, int HW, int ldo, int out_coff, cnb_stream_t stream);
/* src is fp32 (src_f16 == 0) or fp16; dst is always the fp32 NCHW tensor of the public API */
int cnb_nhwc_to_nchw(const void* src, int ldi, int in_coff, float* dst, int B, int C, int HW, int src_f16,
                     cnb_stream_t stream);
/* Hint guidance (classifier-free guidance with the hint as the condition): h_c and h_u are the channels-last outputs
 * of the ControlNet and of the frozen U-Net, both fp32 (src_f16 == 0) or both fp16, with leading dimensions ldc / ldu
 * >= C (each pointer addresses channel 0 of its view).  Per element, in fp32, separate IEEE operations:
 *   dst[b, c, p] = eu + w * (ec - eu)
 * so the result equals that fp32 expression on the two cnb_nhwc_to_nchw results bit for bit (w == 0 gives eu).  dst is
 * contiguous fp32 NCHW and must not overlap either input; pointers aligned to their element size. */
int cnb_guidance_combine(const void* h_c, int ldc, const void* h_u, int ldu, float* dst, int B, int C, int HW, float w,
                         int src_f16, cnb_stream_t stream);
/* elt =bytes per element (4 or 2); offsets and leading dimensions in elements */
int cnb_copy_channels(const void* src, int lds, int s_coff, void* dst, int ldd, int d_coff, long long npix,
                      int C, int elt, cnb_stream_t stream);

/* Reads (and clears) the device-side hang-guard flag set by tcgen05 kernels; synchronises the device. */
int cnb_tc_error_flag(void);

#ifdef __cplusplus
}
#endif
#endif /* CNB200_H */
