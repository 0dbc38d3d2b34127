// GroupNorm (+SiLU) over channels-last fp32 activations [B, HW, C]  (memory-bound: judged by HBM GB/s).
// One CTA per sample: the [HW, C] slab is contiguous, so every global access is a fully coalesced float4.
// Statistics are two-pass (mean, then centred sum of squares) to match ATen's numerics; the second and third
// sweeps of the slab are L1/L2 hits (a slab is at most a few hundred KB), so DRAM sees one read + one write.
// Per-thread column ownership (thread <-> fixed 4 channels) makes the reduction a deterministic tree:
// registers -> smem [rows][C] -> per-channel -> per-group.
#include <cuda_fp16.h>

#include "common.cuh"

namespace cnb {

// SiLU for fp16 outputs: x * sigmoid(x) = h + h * tanh(h) with h = x / 2 -- ONE MUFU op (tanh.approx, ~2^-11 relative,
// the rounding of the fp16 result) instead of ex2 + rcp.  At B = 1024 the 64-channel 28x28 tensor alone carries 51 M
// activations: two MUFU ops each would cost 23 us of XU time, as much as the kernel's DRAM time.
__device__ __forceinline__ float silu_tanh(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
template <bool HALF>
__device__ __forceinline__ float silu_out(float x) { return HALF ? silu_tanh(x) : silu_f(x); }

template <bool HALF> struct OutVec;
template <> struct OutVec<false> {
  using type = float4;
  static __device__ __forceinline__ float4 pack(float4 v) { return v; }
};
template <> struct OutVec<true> {
  using type = uint2;   // 4 x fp16
  static __device__ __forceinline__ uint2 pack(float4 v) {
    __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
    return make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
  }
};

// input vector of 4 channels: float4 (fp32 stream) or 4 x fp16 (fp16 activation stream), widened to fp32
template <bool HIN> struct InVec;
template <> struct InVec<false> {
  using type = float4;
  static __device__ __forceinline__ float4 load(const float4* p) { return *p; }
  static __device__ __forceinline__ float4 load_cs(const float4* p) { return __ldcs(p); }
};
template <> struct InVec<true> {
  using type = uint2;
  static __device__ __forceinline__ float4 widen(uint2 raw) {
    const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
    const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
  }
  static __device__ __forceinline__ float4 load(const uint2* p) { return widen(*p); }
  static __device__ __forceinline__ float4 load_cs(const uint2* p) { return widen(__ldcs(p)); }
};

// STAGE: the fp16 slab of the sample is first brought into shared memory by ONE bulk copy (cp.async.bulk + mbarrier, no
// per-thread load instructions, the whole slab in flight at once) and the three sweeps read smem; with two CTAs per SM
// the copy of one sample overlaps the arithmetic of the other, so the kernel runs at DRAM speed instead of at the
// latency of three dependent sweeps.
template <bool SILU, bool HALF, bool HIN, bool STAGE>
__global__ void __launch_bounds__(1024)
groupnorm_nhwc_kernel(const void* __restrict__ x, void* __restrict__ y, const float* __restrict__ gamma,
                      const float* __restrict__ beta, int HW, int C, int G, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int C4 = C >> 2;
  const int NT = blockDim.x;
  const int R = NT / C4;            // pixel rows swept per iteration
  float* part = sm;                 // [R][C]
  float* chan = part + R * C;       // [C]
  float* g_mean = chan + C;         // [G]
  float* g_rstd = g_mean + G;       // [G]

  const int tid = threadIdx.x;
  const int col = tid % C4;
  const int r0 = tid / C4;
  const int cg = C / G;
  using IV = InVec<HIN>;
  struct XS {   // xs[i] reads the i-th 4-channel vector of this sample as fp32
    const typename IV::type* p;
    __device__ __forceinline__ float4 operator[](size_t i) const { return IV::load(p + i); }
  };
  const typename IV::type* src = reinterpret_cast<const typename IV::type*>(x) + (size_t)blockIdx.x * HW * C4;
  if (STAGE) {
    __shared__ __align__(8) uint64_t bar;
    typename IV::type* slab = reinterpret_cast<typename IV::type*>(
        reinterpret_cast<char*>(sm) + (((size_t)(R * C + C + 2 * G) * sizeof(float) + 127) / 128) * 128);
    const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
    const uint32_t bytes = (uint32_t)((size_t)HW * C4 * sizeof(typename IV::type));
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(slab)), "l"(src), "r"(bytes), "r"(bar_a)
                   : "memory");
    }
    __syncthreads();                                       // barrier object initialised before anyone polls it
    uint32_t done = 0;
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done) : "r"(bar_a) : "memory");
    }
    src = slab;
  }
  const XS xs{src};
  using OV = OutVec<HALF>;
  typename OV::type* ys = reinterpret_cast<typename OV::type*>(y) + (size_t)blockIdx.x * HW * C4;
  const float inv_n = 1.0f / (float)(cg * HW);

  // ---- pass 1: per-channel sums -> group means
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  int pidx = r0;
  for (; pidx + 3 * R < HW; pidx += 4 * R) {
    float4 v0 = xs[(size_t)pidx * C4 + col];
    float4 v1 = xs[(size_t)(pidx + R) * C4 + col];
    float4 v2 = xs[(size_t)(pidx + 2 * R) * C4 + col];
    float4 v3 = xs[(size_t)(pidx + 3 * R) * C4 + col];
    s.x += (v0.x + v1.x) + (v2.x + v3.x);
    s.y += (v0.y + v1.y) + (v2.y + v3.y);
    s.z += (v0.z + v1.z) + (v2.z + v3.z);
    s.w += (v0.w + v1.w) + (v2.w + v3.w);
  }
  for (; pidx < HW; pidx += R) {
    float4 v = xs[(size_t)pidx * C4 + col];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  reinterpret_cast<float4*>(part + r0 * C)[col] = s;
  __syncthreads();
  for (int c = tid; c < C; c += NT) {
    float t = 0.f;
    for (int r = 0; r < R; ++r) t += part[r * C + c];
    chan[c] = t;
  }
  __syncthreads();
  for (int g = tid; g < G; g += NT) {
    float t = 0.f;
    for (int c = 0; c < cg; ++c) t += chan[g * cg + c];
    g_mean[g] = t * inv_n;
  }
  __syncthreads();

  // ---- pass 2: centred second moment -> rstd
  const int c0 = col * 4;
  const float m0 = g_mean[(c0 + 0) / cg], m1 = g_mean[(c0 + 1) / cg];
  const float m2 = g_mean[(c0 + 2) / cg], m3 = g_mean[(c0 + 3) / cg];
  s = make_float4(0.f, 0.f, 0.f, 0.f);
  pidx = r0;
  for (; pidx + 3 * R < HW; pidx += 4 * R) {
    float4 v0 = xs[(size_t)pidx * C4 + col];
    float4 v1 = xs[(size_t)(pidx + R) * C4 + col];
    float4 v2 = xs[(size_t)(pidx + 2 * R) * C4 + col];
    float4 v3 = xs[(size_t)(pidx + 3 * R) * C4 + col];
    float d;
    d = v0.x - m0; s.x = fmaf(d, d, s.x); d = v1.x - m0; s.x = fmaf(d, d, s.x);
    d = v2.x - m0; s.x = fmaf(d, d, s.x); d = v3.x - m0; s.x = fmaf(d, d, s.x);
    d = v0.y - m1; s.y = fmaf(d, d, s.y); d = v1.y - m1; s.y = fmaf(d, d, s.y);
    d = v2.y - m1; s.y = fmaf(d, d, s.y); d = v3.y - m1; s.y = fmaf(d, d, s.y);
    d = v0.z - m2; s.z = fmaf(d, d, s.z); d = v1.z - m2; s.z = fmaf(d, d, s.z);
    d = v2.z - m2; s.z = fmaf(d, d, s.z); d = v3.z - m2; s.z = fmaf(d, d, s.z);
    d = v0.w - m3; s.w = fmaf(d, d, s.w); d = v1.w - m3; s.w = fmaf(d, d, s.w);
    d = v2.w - m3; s.w = fmaf(d, d, s.w); d = v3.w - m3; s.w = fmaf(d, d, s.w);
  }
  for (; pidx < HW; pidx += R) {
    float4 v = xs[(size_t)pidx * C4 + col];
    float d;
    d = v.x - m0; s.x = fmaf(d, d, s.x);
    d = v.y - m1; s.y = fmaf(d, d, s.y);
    d = v.z - m2; s.z = fmaf(d, d, s.z);
    d = v.w - m3; s.w = fmaf(d, d, s.w);
  }
  reinterpret_cast<float4*>(part + r0 * C)[col] = s;
  __syncthreads();
  for (int c = tid; c < C; c += NT) {
    float t = 0.f;
    for (int r = 0; r < R; ++r) t += part[r * C + c];
    chan[c] = t;
  }
  __syncthreads();
  for (int g = tid; g < G; g += NT) {
    float t = 0.f;
    for (int c = 0; c < cg; ++c) t += chan[g * cg + c];
    g_rstd[g] = rsqrtf(t * inv_n + eps);
  }
  __syncthreads();

  // ---- pass 3: normalise, affine, (SiLU), store
  const float4 ga = reinterpret_cast<const float4*>(gamma)[col];
  const float4 be = reinterpret_cast<const float4*>(beta)[col];
  const float a0 = g_rstd[(c0 + 0) / cg] * ga.x, a1 = g_rstd[(c0 + 1) / cg] * ga.y;
  const float a2 = g_rstd[(c0 + 2) / cg] * ga.z, a3 = g_rstd[(c0 + 3) / cg] * ga.w;
  const float b0 = be.x - m0 * a0, b1 = be.y - m1 * a1, b2 = be.z - m2 * a2, b3 = be.w - m3 * a3;
  auto apply = [&](float4 v) {
    float4 o;
    o.x = fmaf(v.x, a0, b0); o.y = fmaf(v.y, a1, b1); o.z = fmaf(v.z, a2, b2); o.w = fmaf(v.w, a3, b3);
    if (SILU) { o.x = silu_out<HALF>(o.x); o.y = silu_out<HALF>(o.y); o.z = silu_out<HALF>(o.z); o.w = silu_out<HALF>(o.w); }
    return o;
  };
  pidx = r0;
  for (; pidx + 3 * R < HW; pidx += 4 * R) {
    float4 v0 = xs[(size_t)pidx * C4 + col];
    float4 v1 = xs[(size_t)(pidx + R) * C4 + col];
    float4 v2 = xs[(size_t)(pidx + 2 * R) * C4 + col];
    float4 v3 = xs[(size_t)(pidx + 3 * R) * C4 + col];
    ys[(size_t)pidx * C4 + col] = OV::pack(apply(v0));
    ys[(size_t)(pidx + R) * C4 + col] = OV::pack(apply(v1));
    ys[(size_t)(pidx + 2 * R) * C4 + col] = OV::pack(apply(v2));
    ys[(size_t)(pidx + 3 * R) * C4 + col] = OV::pack(apply(v3));
  }
  for (; pidx < HW; pidx += R) ys[(size_t)pidx * C4 + col] = OV::pack(apply(xs[(size_t)pidx * C4 + col]));
}

// ---------------------------------------------------------------------------------------------------------
// Register-resident variant: one CTA per sample (grid (1, B)).  The CTA loads the [HW, C] slab ONCE into registers (up
// to KMAX float4 per thread, all loads in flight together), statistics are reduced thread -> smem -> CTA, and the
// normalised values are stored from the same registers: exactly one global read and one global write per element, no
// L2 re-read.  Same two-pass numerics (mean, then centred second moment) as the kernel above.
// ---------------------------------------------------------------------------------------------------------
template <int KMAX, bool SILU, bool HALF, bool HIN>
__global__ void __launch_bounds__(256)
groupnorm_reg_kernel(const void* __restrict__ x, void* __restrict__ y, const float* __restrict__ gamma,
                     const float* __restrict__ beta, int HW, int C, int G, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];
  const int C4 = C >> 2;
  const int NT = blockDim.x;
  const int R = NT / C4;            // pixel rows covered per sweep
  float* part = sm;                 // [R][C]
  float* chan = part + R * C;       // [C]
  float* g_mean = chan + C;         // [G]
  float* g_rstd = g_mean + G;       // [G]

  const int tid = threadIdx.x;
  const int col = tid % C4;
  const int r0 = tid / C4;
  const int cg = C / G;
  const size_t slab = (size_t)blockIdx.y * HW * C4;
  using IV = InVec<HIN>;
  const typename IV::type* xs = reinterpret_cast<const typename IV::type*>(x) + slab;
  using OV = OutVec<HALF>;
  typename OV::type* ys = reinterpret_cast<typename OV::type*>(y) + slab;
  const float inv_n = 1.0f / (float)(cg * HW);

  float4 v[KMAX];
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const int row = r0 + k * R;
    v[k] = row < HW ? IV::load_cs(xs + (size_t)row * C4 + col) : make_float4(0.f, 0.f, 0.f, 0.f);
  }

  // ---- pass 1: sums -> group means
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int k = 0; k < KMAX; ++k) { s.x += v[k].x; s.y += v[k].y; s.z += v[k].z; s.w += v[k].w; }
  reinterpret_cast<float4*>(part + r0 * C)[col] = s;
  __syncthreads();
  for (int c = tid; c < C; c += NT) {
    float t = 0.f;
    for (int r = 0; r < R; ++r) t += part[r * C + c];
    chan[c] = t;
  }
  __syncthreads();
  for (int g = tid; g < G; g += NT) {
    float t = 0.f;
    for (int c = 0; c < cg; ++c) t += chan[g * cg + c];
    g_mean[g] = t * inv_n;
  }
  __syncthreads();

  // ---- pass 2: centred second moment -> rstd
  const int c0 = col * 4;
  const float m0 = g_mean[(c0 + 0) / cg], m1 = g_mean[(c0 + 1) / cg];
  const float m2 = g_mean[(c0 + 2) / cg], m3 = g_mean[(c0 + 3) / cg];
  s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    if (r0 + k * R < HW) {
      float d;
      d = v[k].x - m0; s.x = fmaf(d, d, s.x);
      d = v[k].y - m1; s.y = fmaf(d, d, s.y);
      d = v[k].z - m2; s.z = fmaf(d, d, s.z);
      d = v[k].w - m3; s.w = fmaf(d, d, s.w);
    }
  }
  reinterpret_cast<float4*>(part + r0 * C)[col] = s;
  __syncthreads();
  for (int c = tid; c < C; c += NT) {
    float t = 0.f;
    for (int r = 0; r < R; ++r) t += part[r * C + c];
    chan[c] = t;
  }
  __syncthreads();
  for (int g = tid; g < G; g += NT) {
    float t = 0.f;
    for (int c = 0; c < cg; ++c) t += chan[g * cg + c];
    g_rstd[g] = rsqrtf(t * inv_n + eps);
  }
  __syncthreads();

  // ---- normalise, affine, (SiLU), store from registers
  const float4 ga = reinterpret_cast<const float4*>(gamma)[col];
  const float4 be = reinterpret_cast<const float4*>(beta)[col];
  const float a0 = g_rstd[(c0 + 0) / cg] * ga.x, a1 = g_rstd[(c0 + 1) / cg] * ga.y;
  const float a2 = g_rstd[(c0 + 2) / cg] * ga.z, a3 = g_rstd[(c0 + 3) / cg] * ga.w;
  const float b0 = be.x - m0 * a0, b1 = be.y - m1 * a1, b2 = be.z - m2 * a2, b3 = be.w - m3 * a3;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const int row = r0 + k * R;
    if (row < HW) {
      float4 o;
      o.x = fmaf(v[k].x, a0, b0); o.y = fmaf(v[k].y, a1, b1); o.z = fmaf(v[k].z, a2, b2); o.w = fmaf(v[k].w, a3, b3);
      if (SILU) { o.x = silu_out<HALF>(o.x); o.y = silu_out<HALF>(o.y); o.z = silu_out<HALF>(o.z); o.w = silu_out<HALF>(o.w); }
      ys[(size_t)row * C4 + col] = OV::pack(o);
    }
  }
}

template <int KMAX, bool SILU, bool HALF, bool HIN>
static cudaError_t launch_reg_one(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C,
                                  int G, float eps, int NT, cudaStream_t st) {
  const size_t smem = ((size_t)(NT / (C / 4)) * C + C + 2 * G) * sizeof(float);
  return launch_pdl((long long)B * HW * C, groupnorm_reg_kernel<KMAX, SILU, HALF, HIN>, dim3(1, B), dim3(NT), smem, st,
                    x, y, gamma, beta, HW, C, G, eps);
}

template <int KMAX>
static int launch_reg(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
                      float eps, int silu, int in_f16, int out_f16, int NT, cudaStream_t st) {
  const int sel = (silu ? 4 : 0) | (out_f16 ? 2 : 0) | (in_f16 ? 1 : 0);
  switch (sel) {
    case 0: CNB_CUDA((launch_reg_one<KMAX, false, false, false>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 1: CNB_CUDA((launch_reg_one<KMAX, false, false, true>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 2: CNB_CUDA((launch_reg_one<KMAX, false, true, false>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 3: CNB_CUDA((launch_reg_one<KMAX, false, true, true>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 4: CNB_CUDA((launch_reg_one<KMAX, true, false, false>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 5: CNB_CUDA((launch_reg_one<KMAX, true, false, true>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    case 6: CNB_CUDA((launch_reg_one<KMAX, true, true, false>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
    default: CNB_CUDA((launch_reg_one<KMAX, true, true, true>(x, y, gamma, beta, B, HW, C, G, eps, NT, st))); break;
  }
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Warp-per-group variant for small groups (<= 32 lanes x 13 vectors, >= 16 channels per group): one warp owns one
// (sample, group), keeps it in registers, reduces with shuffles only -- no shared memory, no block barrier, so the
// 7x7 / 14x14 levels (45 of the 87 GroupNorms of an MNIST step) stop being bound by barrier latency.
// ---------------------------------------------------------------------------------------------------------
template <int KMAX, bool SILU, bool HALF, bool HIN>
__global__ void __launch_bounds__(256)
groupnorm_warp_kernel(const void* __restrict__ x, void* __restrict__ y, const float* __restrict__ gamma,
                      const float* __restrict__ beta, int BG, int HW, int C, int G, float eps) {
  pdl_trigger();
  pdl_wait();
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (wid >= BG) return;
  const int lane = threadIdx.x & 31;
  const int b = wid / G, g = wid - b * G;
  const int C4 = C >> 2;
  const int LPP = (C / G) >> 2;          // lanes per pixel (4-channel vectors per group)
  const int PPI = 32 / LPP;              // pixels per iteration
  const int lc = lane % LPP, lp = lane / LPP;
  using IV = InVec<HIN>;
  using OV = OutVec<HALF>;
  const size_t base = (size_t)b * HW * C4 + (size_t)g * LPP + lc;
  const typename IV::type* xs = reinterpret_cast<const typename IV::type*>(x) + base;
  typename OV::type* ys = reinterpret_cast<typename OV::type*>(y) + base;

  float4 v[KMAX];
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const int p = lp + k * PPI;
    v[k] = p < HW ? IV::load_cs(xs + (size_t)p * C4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  const float inv_n = 1.0f / (float)((C / G) * HW);
  const float mean = warp_sum(s) * inv_n;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    if (lp + k * PPI < HW) {
      float d;
      d = v[k].x - mean; q = fmaf(d, d, q);
      d = v[k].y - mean; q = fmaf(d, d, q);
      d = v[k].z - mean; q = fmaf(d, d, q);
      d = v[k].w - mean; q = fmaf(d, d, q);
    }
  }
  const float rstd = rsqrtf(warp_sum(q) * inv_n + eps);
  const float4 ga = reinterpret_cast<const float4*>(gamma)[g * LPP + lc];
  const float4 be = reinterpret_cast<const float4*>(beta)[g * LPP + lc];
  const float a0 = rstd * ga.x, a1 = rstd * ga.y, a2 = rstd * ga.z, a3 = rstd * ga.w;
  const float b0 = be.x - mean * a0, b1 = be.y - mean * a1, b2 = be.z - mean * a2, b3 = be.w - mean * a3;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const int p = lp + k * PPI;
    if (p < HW) {
      float4 o;
      o.x = fmaf(v[k].x, a0, b0); o.y = fmaf(v[k].y, a1, b1); o.z = fmaf(v[k].z, a2, b2); o.w = fmaf(v[k].w, a3, b3);
      if (SILU) { o.x = silu_out<HALF>(o.x); o.y = silu_out<HALF>(o.y); o.z = silu_out<HALF>(o.z); o.w = silu_out<HALF>(o.w); }
      ys[(size_t)p * C4] = OV::pack(o);
    }
  }
}

template <int KMAX, bool SILU, bool HALF, bool HIN>
static void launch_warp_one(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
                            float eps, cudaStream_t st) {
  const int BG = B * G;
  launch_pdl((long long)B * HW * C, groupnorm_warp_kernel<KMAX, SILU, HALF, HIN>, dim3(ceil_div(BG, 8)), dim3(256), 0, st, x, y, gamma, beta, BG,
             HW, C, G, eps);
}

template <int KMAX>
static void launch_warp(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
                        float eps, int silu, int in_f16, int out_f16, cudaStream_t st) {
  const int sel = (silu ? 4 : 0) | (out_f16 ? 2 : 0) | (in_f16 ? 1 : 0);
  switch (sel) {
    case 0: launch_warp_one<KMAX, false, false, false>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 1: launch_warp_one<KMAX, false, false, true>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 2: launch_warp_one<KMAX, false, true, false>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 3: launch_warp_one<KMAX, false, true, true>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 4: launch_warp_one<KMAX, true, false, false>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 5: launch_warp_one<KMAX, true, false, true>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    case 6: launch_warp_one<KMAX, true, true, false>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
    default: launch_warp_one<KMAX, true, true, true>(x, y, gamma, beta, B, HW, C, G, eps, st); break;
  }
}

template <bool SILU, bool HALF, bool HIN>
static void launch_sweep(const void* x, void* y, const float* gamma, const float* beta, int B, int NT, size_t smem,
                         int HW, int C, int G, float eps, cudaStream_t st) {
  const size_t slab = (size_t)HW * C * 2;                  // fp16 slab
  const size_t staged = (smem + 127) / 128 * 128 + slab;
  if (HIN && slab % 16 == 0 && slab < (1u << 20) && staged <= 110 * 1024) {
    static DeviceOnce attr_once;
    if (attr_once.first()) {
      cudaFuncSetAttribute(groupnorm_nhwc_kernel<SILU, HALF, HIN, HIN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           110 * 1024);
    }
    launch_pdl((long long)B * HW * C, groupnorm_nhwc_kernel<SILU, HALF, HIN, HIN>, dim3(B), dim3(NT), staged, st, x, y, gamma, beta, HW, C, G,
               eps);
  } else {
    launch_pdl((long long)B * HW * C, groupnorm_nhwc_kernel<SILU, HALF, HIN, false>, dim3(B), dim3(NT), smem, st, x, y, gamma, beta, HW, C, G,
               eps);
  }
}

int groupnorm(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
              float eps, int silu, int in_f16, int out_f16, cudaStream_t st) {
  CNB_REQUIRE(C % 4 == 0 && C % G == 0 && C / 4 <= 1024, "groupnorm: C=%d G=%d unsupported", C, G);
  // Warp-per-group kernel: groups of 16 / 32 / 64 / 128 channels whose pixels fit 13 vectors per lane
  {
    const int cgq = (C / G) / 4;
    if ((C / G) % 4 == 0 && (cgq == 4 || cgq == 8 || cgq == 16 || cgq == 32)) {
      const int k = ceil_div(HW, 32 / cgq);
      if (k <= 13) {      // (25 vectors per lane was tried for 128 ch @ 14x14: register pressure makes it lose to the staged kernel)
        if (k <= 7) launch_warp<7>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, st);
        else launch_warp<13>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, st);
        CNB_LAUNCH_CHECK();
        return CNB_OK;
      }
    }
  }
  // Register-resident kernel when one CTA holds a whole sample (<= 256 threads x 16 float4): measured 1.2-1.6x faster
  // than the three-sweep kernel on the 7x7 / 16-channel slabs.  (Splitting a sample over a thread-block cluster was
  // measured too: it loses to the three-sweep kernel on the large slabs - cluster barriers + co-scheduling.)
  if (C / 4 <= 256 && B <= 65535) {
    const int C4r = C / 4;
    const int NTr = (256 / C4r) * C4r;
    const int k = ceil_div(HW, NTr / C4r);
    if (k <= 4) return launch_reg<4>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, NTr, st);
    if (k <= 8) return launch_reg<8>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, NTr, st);
    if (k <= 13) return launch_reg<13>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, NTr, st);
    if (k <= 16) return launch_reg<16>(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, NTr, st);
  }
  const int C4 = C / 4;
  int R = 512 / C4;
  if (R < 1) R = 1;
  if (R > HW) R = HW;
  const int NT = R * C4;
  size_t smem = ((size_t)R * C + C + 2 * G) * sizeof(float);
  CNB_REQUIRE(smem <= 48 * 1024, "groupnorm: smem %zu too large", smem);
  const int sel = (silu ? 4 : 0) | (out_f16 ? 2 : 0) | (in_f16 ? 1 : 0);
  switch (sel) {
    case 0: launch_sweep<false, false, false>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 1: launch_sweep<false, false, true>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 2: launch_sweep<false, true, false>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 3: launch_sweep<false, true, true>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 4: launch_sweep<true, false, false>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 5: launch_sweep<true, false, true>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    case 6: launch_sweep<true, true, false>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
    default: launch_sweep<true, true, true>(x, y, gamma, beta, B, NT, smem, HW, C, G, eps, st); break;
  }
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

}  // namespace cnb
