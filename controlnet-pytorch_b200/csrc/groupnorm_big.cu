// GroupNorm (+SiLU) for samples whose [HW, C] fp16 slab does not fit one CTA's shared memory (VAE decoder: 128x128x256 =
// 8 MB per sample; CelebHQ-latent students: 32x32x256 = 512 KB).  The one-CTA-per-sample kernels of groupnorm.cu then
// sweep the slab three times from L2 / HBM with B CTAs on 148 SMs; here a sample is split over S row ranges:
//
//   stats kernel   grid (S, B): each CTA streams its rows ONCE with 16-byte loads (default caching: the apply kernel's
//                  re-read hits L2 when B * slab fits; the apply kernel reads evict-first) (thread <-> 8 fixed channels) and
//                  accumulates shifted sums  sum(x - p), sum((x - p)^2)  per channel, p = the channel's value in the
//                  block's first row (no cancellation: |mean - p| ~ sigma); per-channel (n, mean, M2) are merged per
//                  group with Chan's parallel-variance formula, blocks are merged in double and written as three
//                  doubles per (sample, range, group)
//   finalize       one thread per (sample, group) merges the sample's block partials in block order (Chan, double)
//   apply kernel   grid (S, B): folds mean / rstd / gamma / beta into one FMA per element, applies SiLU (tanh form for
//                  fp16 outputs) and stores 16 bytes
//
// Algorithmic bytes: 2 B read + 2 B written per element; the second read of a range follows its first within a few
// hundred microseconds and is an L2 hit whenever B * slab stays under the 126 MB L2, else DRAM sees 2 reads + 1 write.
#include <cuda_fp16.h>

#include "common.cuh"

namespace cnb {

namespace gnb {

constexpr int NT = 256;

__device__ __forceinline__ void widen8(const uint4& raw, float* v) {
  const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ float silu_tanh(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// (n_a, mean_a, M2_a) <- merge with (n_b, mean_b, M2_b)
template <typename T>
__device__ __forceinline__ void chan_merge(T& n, T& mean, T& m2, T nb, T mb, T m2b) {
  if (nb == T(0)) return;
  const T nt = n + nb, d = mb - mean;
  mean += d * (nb / nt);
  m2 += m2b + d * d * (n * nb / nt);
  n = nt;
}

// Statistics are computed on FIXED blocks of BLK_SWEEPS * R rows (fp32, deterministic per block) and merged in double,
// so the result does not depend on how many row ranges S a sample is split into (S follows the batch size): GroupNorm
// stays batch / shard invariant like the one-CTA-per-sample kernels.
constexpr int BLK_SWEEPS = 32;

__global__ void __launch_bounds__(NT)
stats_kernel(const __half* __restrict__ x, double* __restrict__ partial, int HW, int C, int G, int rows_per_cta) {
  extern __shared__ float sm[];
  const int C8 = C >> 3;
  const int R = NT / C8;                       // pixel rows per sweep
  float* part = sm;                            // [R][C][2]  shifted sum, shifted sum of squares
  float* cstat = part + (size_t)R * C * 2;     // [C][2]     per-channel mean, M2
  const int tid = threadIdx.x, col = tid % C8, r0 = tid / C8;
  const int S = gridDim.x, s = blockIdx.x, b = blockIdx.y;
  const int cta_row0 = s * rows_per_cta;
  const int cta_rows = max(0, min(rows_per_cta, HW - cta_row0));
  const int BLK = BLK_SWEEPS * R;              // rows_per_cta is a multiple of BLK (host)
  const int cg = C / G;
  const int nblk_total = (HW + BLK - 1) / BLK;  // blocks per sample (global block index = row0 / BLK)
  for (int blk0 = 0; blk0 < cta_rows; blk0 += BLK) {
    const int row0 = cta_row0 + blk0;
    const int nrows = min(BLK, cta_rows - blk0);
    const uint4* xs = reinterpret_cast<const uint4*>(x) + ((size_t)b * HW + row0) * C8;
    float piv[8], sum[8], sq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { piv[i] = 0.f; sum[i] = 0.f; sq[i] = 0.f; }
    if (r0 < R) {
      widen8(__ldg(xs + col), piv);
      int row = r0;
      // four rows (64 bytes per thread) in flight per iteration: ~60 KB per SM, what HBM latency x bandwidth needs
      for (; row + 3 * R < nrows; row += 4 * R) {
        uint4 raw[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) raw[u] = __ldg(xs + (size_t)(row + u * R) * C8 + col);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float v[8];
          widen8(raw[u], v);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float d = v[i] - piv[i];
            sum[i] += d;
            sq[i] = fmaf(d, d, sq[i]);
          }
        }
      }
      for (; row < nrows; row += R) {
        float v[8];
        widen8(__ldg(xs + (size_t)row * C8 + col), v);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float d = v[i] - piv[i];
          sum[i] += d;
          sq[i] = fmaf(d, d, sq[i]);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        part[((size_t)r0 * C + col * 8 + i) * 2] = sum[i];
        part[((size_t)r0 * C + col * 8 + i) * 2 + 1] = sq[i];
      }
    }
    __syncthreads();
    for (int c = tid; c < C; c += NT) {
      const float p = __half2float(x[((size_t)b * HW + row0) * C + c]);
      float s1 = 0.f, s2 = 0.f;
      for (int r = 0; r < R; ++r) {
        s1 += part[((size_t)r * C + c) * 2];
        s2 += part[((size_t)r * C + c) * 2 + 1];
      }
      const float dm = s1 / (float)nrows;
      cstat[2 * c] = p + dm;
      cstat[2 * c + 1] = fmaxf(s2 - s1 * dm, 0.f);
    }
    __syncthreads();
    // one (n, mean, M2) triple per (sample, BLOCK, group): the apply kernel merges a sample's blocks in block order, so
    // the statistics are bit-identical however the blocks were distributed over CTAs
    for (int g = tid; g < G; g += NT) {
      float n = 0.f, mean = 0.f, m2 = 0.f;
      for (int c = 0; c < cg; ++c) chan_merge(n, mean, m2, (float)nrows, cstat[2 * (g * cg + c)], cstat[2 * (g * cg + c) + 1]);
      double* o = partial + (((size_t)b * nblk_total + row0 / BLK) * G + g) * 3;
      o[0] = (double)n; o[1] = (double)mean; o[2] = (double)m2;
    }
    // (the next block's writes to part / cstat are ordered behind these reads by its own two barriers)
  }
}

// One thread per (sample, group): merge the sample's block partials in block order (double, Chan) -> mean, rstd.
__global__ void finalize_kernel(const double* __restrict__ partial, float2* __restrict__ stats, int BG, int G,
                                int nblk_total, float eps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= BG) return;
  const int b = i / G, g = i - b * G;
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int q = 0; q < nblk_total; ++q) {                 // fixed block order: independent of the CTA split
    const double* p = partial + (((size_t)b * nblk_total + q) * G + g) * 3;
    chan_merge(n, mean, m2, p[0], p[1], p[2]);
  }
  stats[i] = make_float2((float)mean, rsqrtf((float)(m2 / n) + eps));
}

template <bool SILU, bool HALF>
__global__ void __launch_bounds__(NT)
apply_kernel(const __half* __restrict__ x, void* __restrict__ y, const float2* __restrict__ stats,
             const float* __restrict__ gamma, const float* __restrict__ beta, int HW, int C, int G, float eps,
             int rows_per_cta) {
  extern __shared__ float sm[];
  float* g_mean = sm;            // [G]
  float* g_rstd = sm + G;        // [G]
  const int C8 = C >> 3;
  const int R = NT / C8;
  const int tid = threadIdx.x, col = tid % C8, r0 = tid / C8;
  const int s = blockIdx.x, b = blockIdx.y;
  for (int g = tid; g < G; g += NT) {
    const float2 st = __ldg(stats + (size_t)b * G + g);
    g_mean[g] = st.x;
    g_rstd[g] = st.y;
  }
  __syncthreads();
  if (r0 >= R) return;
  const int cg = C / G;
  float sc[8], sh[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = col * 8 + i, g = c / cg;
    sc[i] = __ldg(gamma + c) * g_rstd[g];
    sh[i] = fmaf(-g_mean[g], sc[i], __ldg(beta + c));
  }
  const int row0 = s * rows_per_cta;
  const int nrows = max(0, min(rows_per_cta, HW - row0));
  const uint4* xs = reinterpret_cast<const uint4*>(x) + ((size_t)b * HW + row0) * C8;
  auto emit = [&](const uint4& raw, int row) {
    float v[8];
    widen8(raw, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i] = fmaf(v[i], sc[i], sh[i]);
      if (SILU) v[i] = HALF ? silu_tanh(v[i]) : silu_f(v[i]);
    }
    const size_t o = ((size_t)b * HW + row0 + row) * C8 + col;
    if (HALF) {
      uint4 out;
      __half2* h = reinterpret_cast<__half2*>(&out);
#pragma unroll
      for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      reinterpret_cast<uint4*>(y)[o] = out;
    } else {
      float4* yo = reinterpret_cast<float4*>(y) + 2 * o;
      yo[0] = make_float4(v[0], v[1], v[2], v[3]);
      yo[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
  };
  int row = r0;
  for (; row + 3 * R < nrows; row += 4 * R) {                // four 16-byte loads in flight per thread
    uint4 raw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) raw[u] = __ldcs(xs + (size_t)(row + u * R) * C8 + col);
#pragma unroll
    for (int u = 0; u < 4; ++u) emit(raw[u], row + u * R);
  }
  for (; row < nrows; row += R) emit(__ldcs(xs + (size_t)row * C8 + col), row);
}

// row ranges per sample: enough CTAs to fill the GPU ~8 deep; a range is a whole number of statistics blocks
static void plan(int B, int HW, int C, int* S_out, int* rows_out) {
  const int R = NT / (C / 8);
  const int BLK = BLK_SWEEPS * R;
  const int nblk = ceil_div(HW, BLK);
  int S = ceil_div(148 * 8, B);
  if (S > nblk) S = nblk;
  if (S < 1) S = 1;
  const int rows = ceil_div(nblk, S) * BLK;
  *S_out = ceil_div(HW, rows);
  *rows_out = rows;
}

}  // namespace gnb

bool groupnorm_big_eligible(int B, int HW, int C, int G, int in_f16) {
  if (!in_f16 || C % 8 || C % G || C / 8 > gnb::NT || B > 65535) return false;
  return (long long)HW * C * 2 > 110 * 1024;              // beyond the staged one-CTA-per-sample kernel
}

size_t groupnorm_big_workspace(int B, int HW, int C, int G) {
  int S, rows;
  gnb::plan(B, HW, C, &S, &rows);
  (void)S;
  const int R = gnb::NT / (C / 8);
  const int nblk = ceil_div(HW, gnb::BLK_SWEEPS * R);
  return (size_t)B * nblk * G * 3 * sizeof(double) + (size_t)B * G * sizeof(float2);
}

int groupnorm_big(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G, float eps,
                  int silu, int out_f16, void* workspace, size_t ws_bytes, cudaStream_t st) {
  using namespace gnb;
  int S, rows;
  plan(B, HW, C, &S, &rows);
  const int R = NT / (C / 8);
  const int nblk = ceil_div(HW, BLK_SWEEPS * R);
  const size_t partial_bytes = (size_t)B * nblk * G * 3 * sizeof(double);
  CNB_REQUIRE(workspace && ws_bytes >= partial_bytes + (size_t)B * G * sizeof(float2), "groupnorm: workspace too small");
  const size_t smem_stats = ((size_t)R * C * 2 + 2 * C) * sizeof(float);
  CNB_REQUIRE(smem_stats <= 48 * 1024, "groupnorm_big: smem %zu too large", smem_stats);
  double* partial = reinterpret_cast<double*>(workspace);
  stats_kernel<<<dim3(S, B), NT, smem_stats, st>>>(reinterpret_cast<const __half*>(x), partial, HW, C, G, rows);
  CNB_LAUNCH_CHECK();
  float2* stats = reinterpret_cast<float2*>(reinterpret_cast<char*>(workspace) + partial_bytes);
  finalize_kernel<<<ceil_div(B * G, 128), 128, 0, st>>>(partial, stats, B * G, G, nblk, eps);
  CNB_LAUNCH_CHECK();
  const size_t smem_apply = 2 * G * sizeof(float);
  const __half* xh = reinterpret_cast<const __half*>(x);
  const dim3 grid(S, B);
  if (silu) {
    if (out_f16) apply_kernel<true, true><<<grid, NT, smem_apply, st>>>(xh, y, stats, gamma, beta, HW, C, G, eps, rows);
    else apply_kernel<true, false><<<grid, NT, smem_apply, st>>>(xh, y, stats, gamma, beta, HW, C, G, eps, rows);
  } else {
    if (out_f16) apply_kernel<false, true><<<grid, NT, smem_apply, st>>>(xh, y, stats, gamma, beta, HW, C, G, eps, rows);
    else apply_kernel<false, false><<<grid, NT, smem_apply, st>>>(xh, y, stats, gamma, beta, HW, C, G, eps, rows);
  }
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

}  // namespace cnb
