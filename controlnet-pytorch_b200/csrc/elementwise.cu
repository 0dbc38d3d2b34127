// Small / memory-bound kernels of the path: time embedding, t-embedding MLP rows, scheduler step (bit-exact fp32
// restatement of scheduler/linear_noise_scheduler.py:58-77 with optional fused Philox noise), DDIM and DPM-Solver++
// steps, EDM scalings, NCHW <-> channels-last plumbing and one-time weight packers.
#include <cuda_fp16.h>

#include "common.cuh"

namespace cnb {

// ------------------------------------------------------------------------------------------------
// get_time_embedding (models/unet_base.py:20-27): t (int64) -> fp32, IEEE divide by the factor table, sin | cos
// ------------------------------------------------------------------------------------------------
__global__ void time_embedding_kernel(const int64_t* __restrict__ t, const float* __restrict__ factor,
                                      float* __restrict__ out, int n, int D) {
  const int half = D >> 1;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * half) return;
  int r = i / half, j = i - r * half;
  float arg = __fdiv_rn((float)t[r], factor[j]);
  out[(size_t)r * D + j] = sinf(arg);
  out[(size_t)r * D + half + j] = cosf(arg);
}

// ------------------------------------------------------------------------------------------------
// y[r, n] = post(sum_k pre(x[r,k]) w[n,k] + b[n]); one warp per output element (R is 1 or B, K <= 512)
// ------------------------------------------------------------------------------------------------
__global__ void linear_small_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                    const float* __restrict__ b, float* __restrict__ y, int R, int K, int N,
                                    int ldy, int silu_in, int silu_out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= R * N) return;
  const int r = warp / N, n = warp - r * N;
  const float* xr = x + (size_t)r * K;
  const float* wr = w + (size_t)n * K;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) {
    float xv = xr[k];
    if (silu_in) xv = xv / (1.0f + expf(-xv));
    acc = fmaf(xv, wr[k], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (b) acc += b[n];
    if (silu_out) acc = acc / (1.0f + expf(-acc));
    y[(size_t)r * ldy + n] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller, keyed by the global element index
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}

__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t step, uint64_t quad) {
  uint32_t c[4] = {(uint32_t)quad, (uint32_t)(quad >> 32), (uint32_t)step, (uint32_t)(step >> 32)};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float S = 2.3283064365386963e-10f;  // 2^-32
  float u0 = ((float)c[0] + 0.5f) * S, u1 = ((float)c[1] + 0.5f) * S;
  float u2 = ((float)c[2] + 0.5f) * S, u3 = ((float)c[3] + 0.5f) * S;
  u0 = fminf(fmaxf(u0, 1.0e-10f), 1.0f);
  u2 = fminf(fmaxf(u2, 1.0e-10f), 1.0f);
  float r0 = sqrtf(-2.0f * logf(u0)), r1 = sqrtf(-2.0f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.0f * u1, &s0, &c0);
  sincospif(2.0f * u3, &s1, &c1);
  return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}

__device__ __forceinline__ float philox_pick(float4 v, int k) {
  return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w));
}

// One Philox4x32-10 block yields the four normals of global elements 4q .. 4q+3; a thread owns one such block and
// stores it with one float4 when the output is 16-byte aligned with the global element grid (same element -> value
// mapping as the fused draw inside update_kernel).
__global__ void philox_normal_kernel(float* __restrict__ out, long long n, uint64_t seed, uint64_t step,
                                     uint64_t elem_offset) {
  const uint64_t g0 = elem_offset & ~3ull;                       // first Philox block that overlaps the output
  const long long nblk = (long long)(((elem_offset + (uint64_t)n + 3ull) >> 2) - (g0 >> 2));
  const long long stride = (long long)gridDim.x * blockDim.x;
  const bool vec = (elem_offset & 3ull) == 0 && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nblk; q += stride) {
    const float4 v = philox_normal4(seed, step, (g0 >> 2) + (uint64_t)q);
    const long long i0 = (long long)(g0 + 4ull * (uint64_t)q) - (long long)elem_offset;   // output index of lane 0
    if (vec && i0 + 4 <= n) {
      reinterpret_cast<float4*>(out)[i0 >> 2] = v;
    } else {
      const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (i0 + k >= 0 && i0 + k < n) out[i0 + k] = e[k];
    }
  }
}

// The noise of the fused scheduler updates: z[4i .. 4i+3] (or z[i]) when the caller supplies it, otherwise the Philox
// normals of global elements elem_offset + 4i .. (or elem_offset + i), whatever the alignment of elem_offset.
__device__ __forceinline__ float4 step_noise4(const float* __restrict__ z, long long i, uint64_t seed, uint64_t step,
                                              uint64_t elem_offset, bool aligned4) {
  if (z) return reinterpret_cast<const float4*>(z)[i];
  if (aligned4) return philox_normal4(seed, step, (elem_offset >> 2) + (uint64_t)i);
  const uint64_t g = elem_offset + 4ull * (uint64_t)i;
  float4 zz;
  zz.x = philox_pick(philox_normal4(seed, step, (g + 0) >> 2), (int)((g + 0) & 3));
  zz.y = philox_pick(philox_normal4(seed, step, (g + 1) >> 2), (int)((g + 1) & 3));
  zz.z = philox_pick(philox_normal4(seed, step, (g + 2) >> 2), (int)((g + 2) & 3));
  zz.w = philox_pick(philox_normal4(seed, step, (g + 3) >> 2), (int)((g + 3) & 3));
  return zz;
}

__device__ __forceinline__ float step_noise1(const float* __restrict__ z, long long i, uint64_t seed, uint64_t step,
                                             uint64_t elem_offset) {
  if (z) return z[i];
  const uint64_t g = elem_offset + (uint64_t)i;
  return philox_pick(philox_normal4(seed, step, g >> 2), (int)(g & 3));
}

// ------------------------------------------------------------------------------------------------
// The fused scheduler updates: one grid-stride kernel, one rule per scheduler.  Every rule evaluates its scheduler's
// fp32 operation order with separate IEEE ops (the *_rn intrinsics are never contracted into an FMA) and starts from
// the same data prediction, so x0 is bit-identical across the three.  A rule maps one element's (xt, eps, z, hist) to
// (x_prev, its new hist value, x0); kHist marks the rule that carries a history buffer, which the kernel reads only
// when the rule's `second` is set and writes every step.
// ------------------------------------------------------------------------------------------------
// v = (xt - c0 * eps) / c1 with c0 = sqrt(1 - alpha_cum_prod[t]), c1 = sqrt(alpha_cum_prod[t]): x0 before its clamp
__device__ __forceinline__ float data_prediction(float xt, float e, float c0, float c1) {
  return __fdiv_rn(__fsub_rn(xt, __fmul_rn(c0, e)), c1);
}

__device__ __forceinline__ float clamp1(float v) { return fminf(fmaxf(v, -1.0f), 1.0f); }

// DDPM (scheduler/linear_noise_scheduler.py, the reference's sample_prev_timestep):
// x_prev = (xt - beta * eps / s1) / sqrt(alpha) (+ sigma * z)
struct DdpmRule {
  static constexpr bool kHist = false;
  float s1, sq_acp, beta, sq_alpha, sigma;
  bool noisy;
  __device__ DdpmRule(const float* c, int)
      : s1(c[0]), sq_acp(c[1]), beta(c[2]), sq_alpha(c[3]), sigma(c[4]), noisy(c[5] != 0.0f) {}
  __device__ void operator()(float xt, float e, float zv, float, float& prev, float&, float& x0) const {
    x0 = clamp1(data_prediction(xt, e, s1, sq_acp));
    const float mean = __fdiv_rn(__fsub_rn(xt, __fdiv_rn(__fmul_rn(beta, e), s1)), sq_alpha);
    prev = noisy ? __fadd_rn(mean, __fmul_rn(sigma, zv)) : mean;
  }
};

// DDIM (scheduler/ddim_scheduler.py): x_prev = c2 * x0' + c3 * eps (+ c4 * z), x0' = clamp(v) with clip_sample, else v
struct DdimRule {
  static constexpr bool kHist = false;
  float c0, c1, c2, c3, c4;
  bool noisy, clip;
  __device__ DdimRule(const float* c, int clip_sample)
      : c0(c[0]), c1(c[1]), c2(c[2]), c3(c[3]), c4(c[4]), noisy(c[5] != 0.0f), clip(clip_sample != 0) {}
  __device__ void operator()(float xt, float e, float zv, float, float& prev, float&, float& x0) const {
    const float v = data_prediction(xt, e, c0, c1);
    x0 = clamp1(v);
    const float p = __fadd_rn(__fmul_rn(c2, clip ? x0 : v), __fmul_rn(c3, e));
    prev = noisy ? __fadd_rn(p, __fmul_rn(c4, zv)) : p;
  }
};

// DPM-Solver++ multistep (scheduler/dpm_solver_scheduler.py): D = clamp(v) with clip_sample, else v;
// x_prev = A * xt + B0 * D (+ B1 * hist) (+ C * z), hist = D.  hist is read only when B1 != 0, so a first-order row
// never touches the previous step's (possibly uninitialised) buffer.
struct DpmSolverRule {
  static constexpr bool kHist = true;
  float c0, c1, A, B0, B1, C;
  bool second, noisy, clip;
  __device__ DpmSolverRule(const float* c, int clip_sample)
      : c0(c[0]), c1(c[1]), A(c[2]), B0(c[3]), B1(c[4]), C(c[5]), second(c[4] != 0.0f), noisy(c[5] != 0.0f),
        clip(clip_sample != 0) {}
  __device__ void operator()(float xt, float e, float zv, float hv, float& prev, float& d, float& x0) const {
    const float v = data_prediction(xt, e, c0, c1);
    x0 = clamp1(v);
    d = clip ? x0 : v;
    float p = __fadd_rn(__fmul_rn(A, xt), __fmul_rn(B0, d));
    if (second) p = __fadd_rn(p, __fmul_rn(B1, hv));
    prev = noisy ? __fadd_rn(p, __fmul_rn(C, zv)) : p;
  }
};

template <class Rule>
__global__ void update_kernel(const float* __restrict__ xt, const float* __restrict__ eps, const float* __restrict__ z,
                              float* __restrict__ hist, float* __restrict__ prev, float* __restrict__ x0, long long n,
                              const float* __restrict__ coef, int clip_sample, uint64_t seed, uint64_t step,
                              const int32_t* __restrict__ step_dev, uint64_t elem_offset) {
  if (step_dev) step = (uint64_t)step_dev[0];
  const Rule rule(coef, clip_sample);
  const long long n4 = n >> 2;
  const bool aligned4 = ((elem_offset & 3) == 0);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 a = reinterpret_cast<const float4*>(xt)[i];
    float4 e = reinterpret_cast<const float4*>(eps)[i];
    const float4 zz =
        rule.noisy ? step_noise4(z, i, seed, step, elem_offset, aligned4) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
    if constexpr (Rule::kHist)
      if (rule.second) h = reinterpret_cast<const float4*>(hist)[i];
    float4 p, d, o;
    rule(a.x, e.x, zz.x, h.x, p.x, d.x, o.x);
    rule(a.y, e.y, zz.y, h.y, p.y, d.y, o.y);
    rule(a.z, e.z, zz.z, h.z, p.z, d.z, o.z);
    rule(a.w, e.w, zz.w, h.w, p.w, d.w, o.w);
    reinterpret_cast<float4*>(prev)[i] = p;
    if constexpr (Rule::kHist) reinterpret_cast<float4*>(hist)[i] = d;
    if (x0) reinterpret_cast<float4*>(x0)[i] = o;
  }
  // tail (n % 4 elements)
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    long long i = (n4 << 2) + threadIdx.x;
    const float zv = rule.noisy ? step_noise1(z, i, seed, step, elem_offset) : 0.f;
    float hv = 0.f;
    if constexpr (Rule::kHist)
      if (rule.second) hv = hist[i];
    float p, d, o;
    rule(xt[i], eps[i], zv, hv, p, d, o);
    prev[i] = p;
    if constexpr (Rule::kHist) hist[i] = d;
    if (x0) x0[i] = o;
  }
}

// ------------------------------------------------------------------------------------------------
// image-to-image start and inpainting (sampler.DDPMSampler.img2img): out = a * x_ref + s * z with the operation order
// of LinearNoiseScheduler.add_noise (mul, mul, add), and the per-step blend that puts the known region back,
// out = m == 1 ? x : (m == 0 ? known : m * x + (1 - m) * known); separate IEEE ops.  out may alias x_ref, so neither
// is __restrict__.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float noised(float xr, float zv, float a, float s) {
  return __fadd_rn(__fmul_rn(a, xr), __fmul_rn(s, zv));
}

__global__ void add_noise_kernel(const float* x_ref, const float* __restrict__ z, float* out, long long n, float a,
                                 float s, uint64_t seed, uint64_t step, uint64_t elem_offset) {
  const long long n4 = n >> 2;
  const bool aligned4 = ((elem_offset & 3) == 0);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 xr = reinterpret_cast<const float4*>(x_ref)[i];
    const float4 zz = step_noise4(z, i, seed, step, elem_offset, aligned4);
    reinterpret_cast<float4*>(out)[i] =
        make_float4(noised(xr.x, zz.x, a, s), noised(xr.y, zz.y, a, s), noised(xr.z, zz.z, a, s),
                    noised(xr.w, zz.w, a, s));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    long long i = (n4 << 2) + threadIdx.x;
    out[i] = noised(x_ref[i], step_noise1(z, i, seed, step, elem_offset), a, s);
  }
}

__device__ __forceinline__ float blend_one(float xv, float xr, float zv, float m, float a, float s) {
  if (m == 1.0f) return xv;
  const float known = noised(xr, zv, a, s);
  if (m == 0.0f) return known;
  return __fadd_rn(__fmul_rn(m, xv), __fmul_rn(__fsub_rn(1.0f, m), known));
}

// mask element of NCHW element e: [B, mask_c, H, W] with mask_c == C, or mask_c == 1 broadcast over the channels
__device__ __forceinline__ long long mask_index(long long e, int C, long long HW, int mask_c) {
  if (mask_c != 1) return e;
  const long long row = e / HW;          // b * C + c
  return (row / C) * HW + (e - row * HW);
}

__global__ void inpaint_blend_kernel(float* __restrict__ x, const float* __restrict__ x_ref,
                                     const float* __restrict__ mask, const float* __restrict__ z, long long n, int C,
                                     long long HW, int mask_c, const float* __restrict__ levels, long long step,
                                     const int32_t* __restrict__ step_dev, uint64_t seed, uint64_t noise_step,
                                     uint64_t elem_offset) {
  const long long k = step_dev ? (long long)step_dev[0] : step;
  const float a = levels[2 * k], s = levels[2 * k + 1];
  const long long n4 = n >> 2;
  const bool aligned4 = ((elem_offset & 3) == 0);
  // four consecutive elements share one mask row (and a 16-byte aligned mask float4) unless a broadcast mask row
  // length is not a multiple of 4
  const bool mvec = mask_c != 1 || (HW & 3) == 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const long long e = i << 2;
    float4 m;
    if (mvec) {
      m = reinterpret_cast<const float4*>(mask)[mask_index(e, C, HW, mask_c) >> 2];
    } else {
      m = make_float4(mask[mask_index(e, C, HW, 1)], mask[mask_index(e + 1, C, HW, 1)],
                      mask[mask_index(e + 2, C, HW, 1)], mask[mask_index(e + 3, C, HW, 1)]);
    }
    float4 xv = reinterpret_cast<const float4*>(x)[i];
    if (m.x == 1.0f && m.y == 1.0f && m.z == 1.0f && m.w == 1.0f) continue;   // all generated: x stays as it is
    const float4 xr = reinterpret_cast<const float4*>(x_ref)[i];
    const float4 zz = step_noise4(z, i, seed, noise_step, elem_offset, aligned4);
    xv.x = blend_one(xv.x, xr.x, zz.x, m.x, a, s);
    xv.y = blend_one(xv.y, xr.y, zz.y, m.y, a, s);
    xv.z = blend_one(xv.z, xr.z, zz.z, m.z, a, s);
    xv.w = blend_one(xv.w, xr.w, zz.w, m.w, a, s);
    reinterpret_cast<float4*>(x)[i] = xv;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    long long i = (n4 << 2) + threadIdx.x;
    const float m = mask[mask_index(i, C, HW, mask_c)];
    x[i] = blend_one(x[i], x_ref[i], m == 1.0f ? 0.f : step_noise1(z, i, seed, noise_step, elem_offset), m, a, s);
  }
}

// out[p, oy, ox] = max of in[p, oy*f .. oy*f+f-1, ox*f .. ox*f+f-1] over the planes p of a [P, H, W] tensor
__global__ void mask_max_pool_kernel(const float* __restrict__ in, float* __restrict__ out, long long total, int H,
                                     int W, int f) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int OW = W / f, OH = H / f;
  const int ox = (int)(i % OW);
  const long long r = i / OW;
  const int oy = (int)(r % OH);
  const long long p = r / OH;
  const float* src = in + (p * H + (long long)oy * f) * W + (long long)ox * f;
  float v = src[0];
  for (int dy = 0; dy < f; ++dy)
    for (int dx = 0; dx < f; ++dx) v = fmaxf(v, src[(long long)dy * W + dx]);
  out[i] = v;
}

__global__ void bump_index_kernel(int32_t* idx, int delta) { idx[0] += delta; }

__global__ void sampler_prologue_kernel(const int32_t* __restrict__ step_idx, const int64_t* __restrict__ t_seq,
                                        int64_t* __restrict__ t_out, const float* __restrict__ coef_table,
                                        float* __restrict__ coef_out) {
  const int64_t t = t_seq[step_idx[0]];
  if (threadIdx.x == 0) t_out[0] = t;
  if (threadIdx.x < 6) coef_out[threadIdx.x] = coef_table[t * 6 + threadIdx.x];
}

// ------------------------------------------------------------------------------------------------
// EDM pre-conditioning (consistency_controlnet_distilled.py:45-74, :95-98), per-sample scalars
// ------------------------------------------------------------------------------------------------
__global__ void edm_coeffs_kernel(const float* __restrict__ sigma, int B, float sigma_data, float sigma_min,
                                  float* __restrict__ coef, int64_t* __restrict__ t_index, int32_t* flag) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) {
    int all_small = 1;
    for (int i = 0; i < B; ++i) all_small &= (sigma[i] <= sigma_min) ? 1 : 0;
    flag[0] = all_small;
  }
  if (b >= B) return;
  const float s = sigma[b];
  const float sd2 = __fmul_rn(sigma_data, sigma_data);
  const float den = __fadd_rn(__fmul_rn(s, s), sd2);
  coef[0 * B + b] = __fdiv_rn(1.0f, __fsqrt_rn(den));                         // c_in
  coef[1 * B + b] = __fdiv_rn(sd2, den);                                      // c_skip
  coef[2 * B + b] = __fdiv_rn(__fmul_rn(s, sigma_data), __fsqrt_rn(den));     // c_out
  float cn = __fmul_rn(0.25f, logf(fmaxf(s, 1e-8f)));                         // c_noise
  long long idx = (long long)__fmul_rn(cn, 1000.0f);                          // .long() truncates toward zero
  idx = idx < 0 ? 0 : (idx > 999 ? 999 : idx);
  coef[3 * B + b] = (float)idx;
  t_index[b] = idx;
}

__global__ void scale_rows_kernel(const float* __restrict__ a, const float* __restrict__ x,
                                  const float* __restrict__ c, const float* __restrict__ y,
                                  float* __restrict__ out, long long per_sample, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int b = (int)(i / per_sample);
  float v = __fmul_rn(a[b], x[i]);
  if (y) v = __fadd_rn(v, __fmul_rn(c[b], y[i]));
  out[i] = v;
}

// x0 = clamp((x_t - s1[t_b] * eps) / s2[t_b], -1, 1) with per-sample timesteps: the teacher-side conversion of a noise
// prediction (distribution_matching_controlnet.py:204-214, consistency_controlnet_distilled.py:219-227).  Same operation
// order as the reference (mul, sub, div, clamp), no FMA contraction: bit-identical to the fp32 ATen expression.
__global__ void x0_from_eps_kernel(const float* __restrict__ xt, const float* __restrict__ eps,
                                   const float* __restrict__ sqrt_one_minus, const float* __restrict__ sqrt_alpha,
                                   const long long* __restrict__ t, int t_count, int num_timesteps,
                                   float* __restrict__ out, long long per_sample, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int b = (int)(i / per_sample);
  long long tb = t[t_count == 1 ? 0 : b];
  // torch indexing semantics of `table[t]`: negative indices wrap once, anything else out of range is an error - the
  // reference raises IndexError on the host; a device kernel cannot, so the sample is poisoned with NaN instead of
  // reading outside the tables
  if (tb < 0) tb += num_timesteps;
  if (tb < 0 || tb >= num_timesteps) {
    out[i] = __int_as_float(0x7fc00000);
    return;
  }
  out[i] = clamp1(data_prediction(xt[i], eps[i], sqrt_one_minus[tb], sqrt_alpha[tb]));
}

// ------------------------------------------------------------------------------------------------
// layout plumbing
// ------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW,
                                    int ldo, int out_coff, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // index over (b, p, c): c fastest
  if (i >= total) return;
  int c = (int)(i % C);
  long long bp = i / C;
  int pix = (int)(bp % HW);
  long long b = bp / HW;
  dst[bp * ldo + out_coff + c] = src[(b * C + c) * HW + pix];
}

template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ src, int ldi, int in_coff, float* __restrict__ dst,
                                    int C, int HW, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // index over (b, c, p): p fastest
  if (i >= total) return;
  int pix = (int)(i % HW);
  long long bc = i / HW;
  int c = (int)(bc % C);
  long long b = bc / C;
  dst[i] = (float)src[(b * HW + pix) * ldi + in_coff + c];
}

// EDM pre-conditioning fused with the layout change (consistency_controlnet_distilled.py:92 and :132): the scaled input
// c_in[b] * x goes straight to the channels-last workspace, and the student's output c_skip[b] * x + c_out[b] * F is
// formed while F leaves it.  Same fp32 operations in the same order as the separate launches (mul; mul, mul, add - no
// FMA contraction), so the results are bit-identical to scale_rows + the plain layout kernels.
__global__ void scale_nchw_to_nhwc_kernel(const float* __restrict__ a, const float* __restrict__ src,
                                          float* __restrict__ dst, int C, int HW, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // index over (b, p, c): c fastest
  if (i >= total) return;
  int c = (int)(i % C);
  long long bp = i / C;
  int pix = (int)(bp % HW);
  long long b = bp / HW;
  dst[i] = __fmul_rn(a[b], src[(b * C + c) * HW + pix]);
}

template <typename T>
__global__ void edm_combine_to_nchw_kernel(const float* __restrict__ cskip, const float* __restrict__ x,
                                           const float* __restrict__ cout, const T* __restrict__ f, int ldi, int in_coff,
                                           float* __restrict__ dst, int C, int HW, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // index over (b, c, p): p fastest
  if (i >= total) return;
  int pix = (int)(i % HW);
  long long bc = i / HW;
  int c = (int)(bc % C);
  long long b = bc / C;
  const float fv = (float)f[(b * HW + pix) * ldi + in_coff + c];
  dst[i] = __fadd_rn(__fmul_rn(cskip[b], x[i]), __fmul_rn(cout[b], fv));
}

// Hint guidance (models/_controlnet_common.controlnet_forward with guidance=w): the two conv_out outputs leave the
// channels-last workspace (fp32 or fp16, leading dimensions ldc / ldu) as eps = eu + w * (ec - eu) in NCHW fp32.  Sub,
// mul, add as separate IEEE operations (no FMA contraction): bit-identical to that fp32 expression evaluated on the
// two cnb_nhwc_to_nchw results.
template <typename T>
__global__ void guidance_combine_kernel(const T* __restrict__ hc, int ldc, const T* __restrict__ hu, int ldu,
                                        float* __restrict__ dst, int C, int HW, float w, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // index over (b, c, p): p fastest
  if (i >= total) return;
  int pix = (int)(i % HW);
  long long bc = i / HW;
  int c = (int)(bc % C);
  long long q = (bc / C) * HW + pix;
  const float ec = (float)hc[q * ldc + c];
  const float eu = (float)hu[q * ldu + c];
  dst[i] = __fadd_rn(eu, __fmul_rn(w, __fsub_rn(ec, eu)));
}

template <typename T>
__global__ void copy_channels_kernel(const T* __restrict__ src, int lds, int s_coff, T* __restrict__ dst,
                                     int ldd, int d_coff, int C, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % C);
  long long pix = i / C;
  dst[pix * ldd + d_coff + c] = src[pix * lds + s_coff + c];
}

// ------------------------------------------------------------------------------------------------
// one-time weight packers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float round_tf32(float v) {
  uint32_t u = __float_as_uint(v);
  if ((u & 0x7f800000u) == 0x7f800000u) return v;
  u += 0x00000fffu + ((u >> 13) & 1u);   // round to nearest even on the 13 dropped bits
  u &= 0xffffe000u;
  return __uint_as_float(u);
}

__global__ void pack_conv_weight_kernel(const float* __restrict__ w, float* __restrict__ dst, int O, int I, int KH,
                                        int KW, int rtf32, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // dst index: [o][tap][c]
  if (i >= total) return;
  int c = (int)(i % I);
  long long ot = i / I;
  int tap = (int)(ot % (KH * KW));
  int o = (int)(ot / (KH * KW));
  float v = w[((long long)o * I + c) * (KH * KW) + tap];
  dst[i] = rtf32 ? round_tf32(v) : v;
}

__global__ void pack_convT_weight_kernel(const float* __restrict__ w, float* __restrict__ dst, int I, int O,
                                         int rtf32, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // dst index: [phase][o][tap][c]
  if (i >= total) return;
  int c = (int)(i % I);
  long long r = i / I;
  int tap = (int)(r % 4); r /= 4;
  int o = (int)(r % O);
  int phase = (int)(r / O);
  int py = phase >> 1, px = phase & 1, ta = tap >> 1, tb = tap & 1;
  // T(0) = {ky=1, ky=3}; T(1) = {ky=0, ky=2}
  int ky = py == 0 ? (ta == 0 ? 1 : 3) : (ta == 0 ? 0 : 2);
  int kx = px == 0 ? (tb == 0 ? 1 : 3) : (tb == 0 ? 0 : 2);
  float v = w[(((long long)c * O + o) * 4 + ky) * 4 + kx];
  dst[i] = rtf32 ? round_tf32(v) : v;
}

__global__ void cast_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2half_rn(src[i]);
}

}  // namespace cnb

// ================================================================================================
// C ABI
// ================================================================================================
using namespace cnb;

static inline unsigned blocks_for(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

extern "C" int cnb_time_embedding(const int64_t* t, const float* factor, float* out, int n, int D, cnb_stream_t s) {
  CNB_REQUIRE(D % 2 == 0 && n > 0, "time embedding dimension must be divisible by 2 (D=%d, n=%d)", D, n);
  time_embedding_kernel<<<blocks_for((long long)n * (D / 2), 128), 128, 0, (cudaStream_t)s>>>(t, factor, out, n, D);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_linear_small(const float* x, const float* w, const float* b, float* y, int R, int K, int N,
                                int ldy, int silu_in, int silu_out, cnb_stream_t s) {
  CNB_REQUIRE(R > 0 && K > 0 && N > 0 && ldy >= N, "linear_small: bad dims R=%d K=%d N=%d ldy=%d", R, K, N, ldy);
  long long threads = (long long)R * N * 32;
  linear_small_kernel<<<blocks_for(threads, 256), 256, 0, (cudaStream_t)s>>>(x, w, b, y, R, K, N, ldy, silu_in,
                                                                            silu_out);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

static bool cnb_overlaps(const float* a, const float* b, long long n) {
  return a && b && a < b + n && b < a + n;
}

static unsigned elementwise4_blocks(long long n) {
  long long blocks = ((n >> 2) + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 16) blocks = 148 * 16;
  return (unsigned)blocks;
}

// The checks every scheduler update takes (hist is null for the rules without a history buffer), then one launch.
template <class Rule>
static int launch_update(const char* name, const float* xt, const float* eps, const float* z, float* hist,
                         float* xt_prev, float* x0, long long n, const float* coef, int clip_sample, uint64_t seed,
                         uint64_t step, const int32_t* step_dev, uint64_t elem_offset, cnb_stream_t s) {
  CNB_REQUIRE(n > 0 && xt && eps && xt_prev && coef && (hist || !Rule::kHist), "%s: null pointer or n=%lld", name, n);
  CNB_REQUIRE(!cnb_overlaps(hist, xt, n) && !cnb_overlaps(hist, xt_prev, n) && !cnb_overlaps(hist, x0, n),
              "%s: hist must not overlap xt, xt_prev or x0", name);
  CNB_REQUIRE((((uintptr_t)xt | (uintptr_t)eps | (uintptr_t)xt_prev | (uintptr_t)z | (uintptr_t)x0 |
                (uintptr_t)hist) & 15) == 0,
              "%s: pointers must be 16-byte aligned", name);
  update_kernel<Rule><<<elementwise4_blocks(n), 256, 0, (cudaStream_t)s>>>(xt, eps, z, hist, xt_prev, x0, n, coef,
                                                                           clip_sample, seed, step, step_dev,
                                                                           elem_offset);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_sched_step(const float* xt, const float* eps, const float* z, float* xt_prev, float* x0,
                              long long n, const float* coef, uint64_t seed, uint64_t step, const int32_t* step_dev,
                              uint64_t elem_offset, cnb_stream_t s) {
  return launch_update<DdpmRule>("sched_step", xt, eps, z, nullptr, xt_prev, x0, n, coef, 0, seed, step, step_dev,
                                 elem_offset, s);
}

extern "C" int cnb_ddim_step(const float* xt, const float* eps, const float* z, float* xt_prev, float* x0, long long n,
                             const float* coef, int clip_sample, uint64_t seed, uint64_t step, const int32_t* step_dev,
                             uint64_t elem_offset, cnb_stream_t s) {
  return launch_update<DdimRule>("ddim_step", xt, eps, z, nullptr, xt_prev, x0, n, coef, clip_sample, seed, step,
                                 step_dev, elem_offset, s);
}

extern "C" int cnb_dpm_solver_step(const float* xt, const float* eps, const float* z, float* hist, float* xt_prev,
                                   float* x0, long long n, const float* coef, int clip_sample, uint64_t seed,
                                   uint64_t step, const int32_t* step_dev, uint64_t elem_offset, cnb_stream_t s) {
  return launch_update<DpmSolverRule>("dpm_solver_step", xt, eps, z, hist, xt_prev, x0, n, coef, clip_sample, seed,
                                      step, step_dev, elem_offset, s);
}

extern "C" int cnb_add_noise(const float* x_ref, const float* z, float* out, long long n, float sqrt_acp,
                             float sqrt_one_minus, uint64_t seed, uint64_t step, uint64_t elem_offset,
                             cnb_stream_t s) {
  CNB_REQUIRE(n > 0 && x_ref && out, "add_noise: null pointer or n=%lld", n);
  CNB_REQUIRE((((uintptr_t)x_ref | (uintptr_t)z | (uintptr_t)out) & 15) == 0,
              "add_noise: pointers must be 16-byte aligned");
  CNB_REQUIRE(x_ref == out || !cnb_overlaps(x_ref, out, n), "add_noise: out must be x_ref or not overlap it");
  add_noise_kernel<<<elementwise4_blocks(n), 256, 0, (cudaStream_t)s>>>(x_ref, z, out, n, sqrt_acp, sqrt_one_minus,
                                                                      seed, step, elem_offset);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_inpaint_blend(float* x, const float* x_ref, const float* mask, const float* z, long long n, int C,
                                 long long HW, int mask_c, const float* levels, long long step,
                                 const int32_t* step_dev, uint64_t seed, uint64_t noise_step, uint64_t elem_offset,
                                 cnb_stream_t s) {
  CNB_REQUIRE(n > 0 && x && x_ref && mask && levels, "inpaint_blend: null pointer or n=%lld", n);
  CNB_REQUIRE(C > 0 && HW > 0 && n % ((long long)C * HW) == 0 && (mask_c == 1 || mask_c == C) &&
                  (step_dev || step >= 0),
              "inpaint_blend: bad dims n=%lld C=%d HW=%lld mask_c=%d step=%lld", n, C, HW, mask_c, step);
  const long long n_mask = n / C * mask_c;
  CNB_REQUIRE(!cnb_overlaps(x, x_ref, n) && !(mask < x + n && x < mask + n_mask),
              "inpaint_blend: x must not overlap x_ref or mask");
  CNB_REQUIRE((((uintptr_t)x | (uintptr_t)x_ref | (uintptr_t)mask | (uintptr_t)z) & 15) == 0,
              "inpaint_blend: pointers must be 16-byte aligned");
  inpaint_blend_kernel<<<elementwise4_blocks(n), 256, 0, (cudaStream_t)s>>>(
      x, x_ref, mask, z, n, C, HW, mask_c, levels, step, step_dev, seed, noise_step, elem_offset);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_mask_max_pool(const float* in, float* out, int B, int H, int W, int f, cnb_stream_t s) {
  CNB_REQUIRE(in && out && B > 0 && f > 0 && H > 0 && W > 0 && H % f == 0 && W % f == 0,
              "mask_max_pool: bad args B=%d H=%d W=%d f=%d", B, H, W, f);
  const long long total = (long long)B * (H / f) * (W / f);
  CNB_REQUIRE(!cnb_overlaps(in, out, (long long)B * H * W), "mask_max_pool: out must not overlap in");
  mask_max_pool_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(in, out, total, H, W, f);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_philox_normal(float* out, long long n, uint64_t seed, uint64_t step, uint64_t elem_offset,
                                 cnb_stream_t s) {
  CNB_REQUIRE(n > 0 && out, "philox_normal: bad args");
  {
    long long blocks = (n / 4 + 256) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    philox_normal_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(out, n, seed, step, elem_offset);
  }
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_sampler_prologue(const int32_t* step_idx, const int64_t* t_seq, int64_t* t_out,
                                    const float* coef_table, float* coef_out, cnb_stream_t s) {
  CNB_REQUIRE(step_idx && t_seq && t_out && coef_table && coef_out, "sampler_prologue: null pointer");
  sampler_prologue_kernel<<<1, 32, 0, (cudaStream_t)s>>>(step_idx, t_seq, t_out, coef_table, coef_out);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_bump_index(int32_t* idx, int delta, cnb_stream_t s) {
  bump_index_kernel<<<1, 1, 0, (cudaStream_t)s>>>(idx, delta);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_edm_coeffs(const float* sigma, int B, float sigma_data, float sigma_min, float* coef,
                              int64_t* t_index, int32_t* flag, cnb_stream_t s) {
  CNB_REQUIRE(B > 0, "edm_coeffs: B=%d", B);
  edm_coeffs_kernel<<<blocks_for(B, 128), 128, 0, (cudaStream_t)s>>>(sigma, B, sigma_data, sigma_min, coef, t_index,
                                                                    flag);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_scale_rows(const float* a, const float* x, const float* c, const float* y, float* out, int B,
                              long long per_sample, cnb_stream_t s) {
  long long total = (long long)B * per_sample;
  CNB_REQUIRE(total > 0 && (y == nullptr || c != nullptr), "scale_rows: bad args");
  scale_rows_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(a, x, c, y, out, per_sample, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_x0_from_eps(const float* xt, const float* eps, const float* sqrt_one_minus, const float* sqrt_alpha,
                               const int64_t* t, int t_count, int num_timesteps, float* out, int B, long long per_sample,
                               cnb_stream_t s) {
  long long total = (long long)B * per_sample;
  CNB_REQUIRE(xt && eps && sqrt_one_minus && sqrt_alpha && t && out && total > 0 && (t_count == 1 || t_count == B) &&
                  num_timesteps > 0, "x0_from_eps: bad args");
  x0_from_eps_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
      xt, eps, sqrt_one_minus, sqrt_alpha, reinterpret_cast<const long long*>(t), t_count, num_timesteps, out, per_sample,
      total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_nchw_to_nhwc(const float* src, float* dst, int B, int C, int HW, int ldo, int out_coff,
                                cnb_stream_t s) {
  long long total = (long long)B * C * HW;
  CNB_REQUIRE(total > 0 && ldo >= out_coff + C, "nchw_to_nhwc: bad dims");
  nchw_to_nhwc_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(src, dst, C, HW, ldo, out_coff, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_scale_nchw_to_nhwc(const float* a, const float* src, float* dst, int B, int C, int HW,
                                      cnb_stream_t s) {
  long long total = (long long)B * C * HW;
  CNB_REQUIRE(a && src && dst && total > 0, "scale_nchw_to_nhwc: bad args");
  scale_nchw_to_nhwc_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(a, src, dst, C, HW, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_edm_combine_to_nchw(const float* c_skip, const float* x, const float* c_out, const void* f, int ldi,
                                       int in_coff, float* dst, int B, int C, int HW, int f_f16, cnb_stream_t s) {
  long long total = (long long)B * C * HW;
  CNB_REQUIRE(c_skip && x && c_out && f && dst && total > 0 && ldi >= in_coff + C, "edm_combine_to_nchw: bad args");
  if (f_f16)
    edm_combine_to_nchw_kernel<__half><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        c_skip, x, c_out, reinterpret_cast<const __half*>(f), ldi, in_coff, dst, C, HW, total);
  else
    edm_combine_to_nchw_kernel<float><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        c_skip, x, c_out, reinterpret_cast<const float*>(f), ldi, in_coff, dst, C, HW, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_guidance_combine(const void* h_c, int ldc, const void* h_u, int ldu, float* dst, int B, int C,
                                    int HW, float w, int src_f16, cnb_stream_t s) {
  const long long total = (long long)B * C * HW;
  CNB_REQUIRE(h_c && h_u && dst && B > 0 && C > 0 && HW > 0 && ldc >= C && ldu >= C,
              "guidance_combine: bad args B=%d C=%d HW=%d ldc=%d ldu=%d", B, C, HW, ldc, ldu);
  const size_t elt = src_f16 ? 2 : 4;
  CNB_REQUIRE((((uintptr_t)h_c | (uintptr_t)h_u) & (elt - 1)) == 0 && ((uintptr_t)dst & 3) == 0,
              "guidance_combine: pointers must be aligned to their element size");
  // byte ranges: the last element an input is read at is ((B * HW - 1) * ld + C - 1)
  const char* o0 = reinterpret_cast<const char*>(dst);
  const char* o1 = o0 + total * 4;
  const char* c0 = reinterpret_cast<const char*>(h_c);
  const char* c1 = c0 + ((long long)B * HW - 1) * ldc * elt + C * elt;
  const char* u0 = reinterpret_cast<const char*>(h_u);
  const char* u1 = u0 + ((long long)B * HW - 1) * ldu * elt + C * elt;
  CNB_REQUIRE(!(o0 < c1 && c0 < o1) && !(o0 < u1 && u0 < o1), "guidance_combine: out must not overlap h_c or h_u");
  if (src_f16)
    guidance_combine_kernel<__half><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const __half*>(h_c), ldc, reinterpret_cast<const __half*>(h_u), ldu, dst, C, HW, w, total);
  else
    guidance_combine_kernel<float><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const float*>(h_c), ldc, reinterpret_cast<const float*>(h_u), ldu, dst, C, HW, w, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_nhwc_to_nchw(const void* src, int ldi, int in_coff, float* dst, int B, int C, int HW, int src_f16,
                                cnb_stream_t s) {
  long long total = (long long)B * C * HW;
  CNB_REQUIRE(total > 0 && ldi >= in_coff + C, "nhwc_to_nchw: bad dims");
  if (src_f16)
    nhwc_to_nchw_kernel<__half><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const __half*>(src), ldi, in_coff, dst, C, HW, total);
  else
    nhwc_to_nchw_kernel<float><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const float*>(src), ldi, in_coff, dst, C, HW, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_copy_channels(const void* src, int lds, int s_coff, void* dst, int ldd, int d_coff,
                                 long long npix, int C, int elt, cnb_stream_t s) {
  long long total = npix * C;
  CNB_REQUIRE(total > 0 && (elt == 4 || elt == 2), "copy_channels: bad dims");
  if (elt == 2 && C % 2 == 0 && lds % 2 == 0 && s_coff % 2 == 0 && ldd % 2 == 0 && d_coff % 2 == 0) {
    total /= 2;      // move fp16 pairs as 32-bit words
    copy_channels_kernel<uint32_t><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const uint32_t*>(src), lds / 2, s_coff / 2, reinterpret_cast<uint32_t*>(dst), ldd / 2,
        d_coff / 2, C / 2, total);
  } else if (elt == 2) {
    copy_channels_kernel<uint16_t><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const uint16_t*>(src), lds, s_coff, reinterpret_cast<uint16_t*>(dst), ldd, d_coff, C, total);
  } else {
    copy_channels_kernel<float><<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        reinterpret_cast<const float*>(src), lds, s_coff, reinterpret_cast<float*>(dst), ldd, d_coff, C, total);
  }
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_pack_conv_weight(const float* w, float* dst, int O, int I, int KH, int KW, int round_tf32,
                                    cnb_stream_t s) {
  long long total = (long long)O * I * KH * KW;
  CNB_REQUIRE(total > 0 && KH * KW <= CNB_MAX_TAPS, "pack_conv_weight: bad dims");
  pack_conv_weight_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(w, dst, O, I, KH, KW, round_tf32,
                                                                              total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_pack_convT_weight(const float* w, float* dst, int I, int O, int round_tf32, cnb_stream_t s) {
  long long total = (long long)I * O * 16;
  CNB_REQUIRE(total > 0, "pack_convT_weight: bad dims");
  pack_convT_weight_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)s>>>(w, dst, I, O, round_tf32, total);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

extern "C" int cnb_cast_f16(const float* src, void* dst, long long n, cnb_stream_t s) {
  CNB_REQUIRE(n > 0, "cast_f16: n=%lld", n);
  cast_f16_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)s>>>(src, (__half*)dst, n);
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}
