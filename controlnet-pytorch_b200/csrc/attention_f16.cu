// Flash attention on fp16 operands (the tensor-core modes' attention core):  qkv [B, L, 3E] fp16 -> out [B, L, E] fp16.
//
// Roofline note.  Head dims on this path are 4..64 (128/192 only in the widest students) and L <= 1024, so per score
// the kernel does 4*d tensor FLOPs but one ex2 (MUFU, 16/clk/SM) and ~4 FP32/ALU ops: at d = 16 the tensor pipe would
// be <10 % busy even at the MUFU limit of 148 SM x 16 x 1.9 GHz = 4.5 T scores/s.  The kernel is therefore built
// to keep the MUFU pipe fed, not the tensor pipe: register-resident S/P (FA2 formulation), no TMEM round trip.
//   * CTA = (batch, head) x BQ queries, one warp per 16 query rows; K/V tiles of BK keys are double-buffered in
//     shared memory with cp.async (8- or 16-byte chunks; padded rows -> conflict-free ldmatrix), 3-stage ring with
//     one block barrier per tile;
//   * S = Q K^T and O += P V use mma.sync.m16n8k16 f16 with fp32 accumulate; K fragments come from ldmatrix.x4,
//     V fragments from ldmatrix.x4.trans; the S accumulator fragment is re-packed in registers (cvt.rn.f16x2) as
//     the A operand of the second MMA;
//   * online softmax in the exp2 domain: p = ex2(fma(s, scale*log2e, -m*scale*log2e)), row max / sum reduced across
//     the 4 lanes of a quad with shuffles, running (m, l) per row, O rescaled per tile.
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"

namespace cnb {
namespace af16 {

__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
template <int BYTES>
__device__ __forceinline__ void cp_async(uint32_t dst, const void* src, uint32_t src_bytes) {
  if (BYTES == 16)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// D: head dim (even; padded to a multiple of 16 for Q K^T); BK: keys per tile (multiple of 16); NW: warps per CTA
// (BQ = 16 * NW).
// The softmax denominator is accumulated by the tensor core as one more output column tile whose B fragment is the
// constant half2(1, 1): l = P . 1 in fp32, consistent with the fp16 P that multiplies V.
// Minimum resident CTAs per SM: 7 for the narrow 4-warp kernels; 3 for the 8-warp kernels, i.e. <= 85 registers
// (d = 24: 122 -> 80, L = 1024 launch 2.15 -> 1.97 ms); the 64-register build (VAR bit 1) asks for 8 / 4.
template <int D, int BK, int NW, int VAR>
__global__ void __launch_bounds__(NW * 32, (NW == 4 && D <= 16) ? ((VAR & 2) ? 8 : 7) : (NW == 8 ? ((VAR & 2) ? 4 : 3) : 0))
attention_f16_kernel(const __half* __restrict__ qkv, __half* __restrict__ out, int L, int E, float scale_log2) {
  constexpr int d = D;
  constexpr int DP = (D + 15) / 16 * 16;         // K extent of Q K^T
  constexpr int NV = (D + 7) / 8;                // 8-wide output column tiles
  constexpr int CH = (D * 2) % 16 == 0 ? 16 : 8; // cp.async chunk bytes
  constexpr int STRIDE = DP + 8;                 // halfs per smem row (16-byte pad: conflict-free ldmatrix)
  constexpr int TILE = BK * STRIDE;              // halfs per K (or V) tile
  constexpr int NT = BK / 8;                     // S column tiles
  constexpr int KS = DP / 16;                    // k-steps of Q K^T
  constexpr int THREADS = NW * 32;
  // VAR: bit 0 = 64-key tiles processed as two 32-key halves, bit 1 = 64-register build (8 CTAs of 4 warps per SM),
  //      bit 2 = two tiles per block barrier from a ring of TWO groups (the next group is requested right after the
  //      barrier that frees the other one; a group's compute time covers the L2 latency)
  constexpr bool HALVES = (VAR & 1) != 0;
  constexpr bool RING2 = (VAR & 4) != 0;
  constexpr int SUB = RING2 ? 2 : 1;                     // key tiles per block barrier
  constexpr int NSLOT = (RING2 ? 2 : 3) * SUB;           // smem ring: two / three groups of SUB tiles
  static_assert(BK % 16 == 0, "BK must be a multiple of 16");
  extern __shared__ __align__(16) __half smem[];   // [3 * SUB slots][K | V][BK][STRIDE]
  pdl_trigger();
  pdl_wait();

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, q4 = lane & 3;
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = blockIdx.x * (16 * NW) + warp * 16;
  const size_t row3 = (size_t)3 * E;
  const __half* base = qkv + (size_t)b * L * row3 + (size_t)h * d;
  const uint32_t smem_u = (uint32_t)__cvta_generic_to_shared(smem);

  // zero the pad columns once (cp.async only ever writes the d real columns)
  if (d < DP) {
    for (int i = tid; i < NSLOT * 2 * TILE / 2; i += THREADS) reinterpret_cast<uint32_t*>(smem)[i] = 0u;
    __syncthreads();
  }

  // ---- Q fragments, kept in registers for the whole kernel
  uint32_t qf[KS][4];
  {
    const int r0 = q0 + g, r1 = q0 + g + 8;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const int c0 = ks * 16 + 2 * q4, c1 = c0 + 8;
      uint32_t v00 = 0, v10 = 0, v01 = 0, v11 = 0;      // d is even, so a half2 is all-valid or all-pad
      if (r0 < L) {
        if (c0 < d) v00 = *reinterpret_cast<const uint32_t*>(base + (size_t)r0 * row3 + c0);
        if (c1 < d) v01 = *reinterpret_cast<const uint32_t*>(base + (size_t)r0 * row3 + c1);
      }
      if (r1 < L) {
        if (c0 < d) v10 = *reinterpret_cast<const uint32_t*>(base + (size_t)r1 * row3 + c0);
        if (c1 < d) v11 = *reinterpret_cast<const uint32_t*>(base + (size_t)r1 * row3 + c1);
      }
      qf[ks][0] = v00; qf[ks][1] = v10; qf[ks][2] = v01; qf[ks][3] = v11;
    }
  }

  float o[NV][4];
#pragma unroll
  for (int i = 0; i < NV; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float lsum[4] = {0.f, 0.f, 0.f, 0.f};          // [0] = denominator of row g, [2] = of row g + 8
  float m0 = -INFINITY, m1 = -INFINITY;
  float ms0 = 0.f, ms1 = 0.f;                    // m * scale_log2 of the current reference maxima
  const float lazy = 8.0f / scale_log2;          // 2^8 headroom, in raw score units

  const int ntiles = (L + BK - 1) / BK;
  constexpr int CPR = D * 2 / CH;                // chunks per row
  constexpr int NCHUNK = BK * CPR;               // chunks per K (or V) tile
  constexpr int SLOTS = (NCHUNK + THREADS - 1) / THREADS;
  const char* kbase_g = reinterpret_cast<const char*>(base + E);   // K columns of key 0
  // Tiles are loaded strictly in order.  RUN_PTR: the per-thread source pointers and key indices are running values (one
  // 64-bit add per slot and tile) instead of being recomputed from t -- the address arithmetic was ~15 % of a tile's
  // instructions; measured it pays only where registers are not tight (d = 16, 4 warps: 926 -> 903 us; the other
  // instantiations lose 1-6 % to the extra live registers and keep the recomputation).
  constexpr bool RUN_PTR = (D <= 16 && NW == 4);
  const char* ld_src[SLOTS];
  uint32_t ld_dst[SLOTS];
  int ld_key[SLOTS];
  if (RUN_PTR) {
#pragma unroll
    for (int i = 0; i < SLOTS; ++i) {
      const int u = tid + i * THREADS;
      const int j = u / CPR, c = u % CPR;
      ld_src[i] = kbase_g + (size_t)j * row3 * 2 + c * CH;
      ld_dst[i] = smem_u + (uint32_t)(j * STRIDE) * 2u + (uint32_t)(c * CH);
      ld_key[i] = j;
    }
  }
  const size_t tile_bytes = (size_t)BK * row3 * 2;
  int ld_slot = 0, ld_t = 0;                     // ring slot / index of the next tile to load
  auto load_tile = [&]() {
    const uint32_t slot_off = (uint32_t)(ld_slot * 2 * TILE) * 2u;
#pragma unroll
    for (int i = 0; i < SLOTS; ++i) {
      if (NCHUNK % THREADS == 0 || tid + i * THREADS < NCHUNK) {
        if (RUN_PTR) {
          const bool ok = ld_key[i] < L;
          const char* kp = ok ? ld_src[i] : kbase_g;
          const uint32_t dst = ld_dst[i] + slot_off;
          cp_async<CH>(dst, kp, ok ? CH : 0u);
          cp_async<CH>(dst + (uint32_t)TILE * 2u, kp + (size_t)E * 2, ok ? CH : 0u);
        } else {
          const int u = tid + i * THREADS;
          const int j = u / CPR, c = u % CPR;
          const bool ok = ld_t * BK + j < L;
          const char* kp = kbase_g + ((size_t)(ok ? ld_t * BK + j : 0) * row3) * 2 + c * CH;
          const uint32_t dst = smem_u + slot_off + (uint32_t)(j * STRIDE) * 2u + (uint32_t)(c * CH);
          cp_async<CH>(dst, kp, ok ? CH : 0u);
          cp_async<CH>(dst + (uint32_t)TILE * 2u, kp + (size_t)E * 2, ok ? CH : 0u);
        }
      }
      if (RUN_PTR) {
        ld_src[i] += tile_bytes;
        ld_key[i] += BK;
      }
    }
    ++ld_t;
    if (++ld_slot == NSLOT) ld_slot = 0;
  };
  auto load_group = [&](int grp) {               // SUB consecutive tiles, one commit group
#pragma unroll
    for (int hh = 0; hh < SUB; ++hh)
      if (grp * SUB + hh < ntiles) load_tile();
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  // per-lane ldmatrix row/column selectors
  const int lr = lane & 7, lm = lane >> 3;       // row within an 8x8 matrix, matrix index 0..3
  // K (non-trans): m0 = keys 0-7 / d 0-7, m1 = keys 0-7 / d 8-15, m2 = keys 8-15 / d 0-7, m3 = keys 8-15 / d 8-15
  const uint32_t k_lane_off = (uint32_t)(((lm >> 1) * 8 + lr) * STRIDE + (lm & 1) * 8) * 2u;
  // V (trans):     m0 = keys 0-7 / d 0-7, m1 = keys 8-15 / d 0-7, m2 = keys 0-7 / d 8-15, m3 = keys 8-15 / d 8-15
  const uint32_t v_lane_off = (uint32_t)(((lm & 1) * 8 + lr) * STRIDE + (lm >> 1) * 8) * 2u;
  constexpr uint32_t ONES = 0x3C003C00u;         // half2(1, 1)

  // one key tile; MASK = the (only) tile that may contain keys >= L; NG = 16-key groups of the tile that hold any
  // valid key (the ragged last tile skips its fully padded groups: 784 = 12 x 64 + 16 keys costs 12.25 tiles, not 13)
  int cur_slot = 0;                              // ring slot of the tile being consumed (advanced by the main loop)
  auto tile_body = [&](int t, auto mask_tag, auto ng_tag, auto g0_tag) {
    constexpr bool MASK = decltype(mask_tag)::value;
    constexpr int NG = decltype(ng_tag)::value;
    constexpr int G0 = decltype(g0_tag)::value;    // first 16-key group of the tile this call covers
    constexpr int NTA = NG * 2;                    // active S column tiles
    const uint32_t sK = smem_u + (uint32_t)(cur_slot * 2 * TILE) * 2u + (uint32_t)(G0 * 16 * STRIDE) * 2u;
    const uint32_t sV = sK + (uint32_t)TILE * 2u;

    // ---- S = Q K^T  (16 x BK per warp)
    float s[NTA][4];
#pragma unroll
    for (int nt = 0; nt < NTA; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
    for (int np = 0; np < NG; ++np) {
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t r0, r1, r2, r3;
        ldsm_x4(sK + k_lane_off + (uint32_t)(np * 16 * STRIDE + ks * 16) * 2u, r0, r1, r2, r3);
        mma_f16(s[2 * np], qf[ks], r0, r1);
        mma_f16(s[2 * np + 1], qf[ks], r2, r3);
      }
    }
    if (MASK) {
      const int kbase = t * BK + G0 * 16;
#pragma unroll
      for (int nt = 0; nt < NTA; ++nt) {
        const int key = kbase + nt * 8 + 2 * q4;
        if (key >= L) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
        if (key + 1 >= L) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
      }
    }
    // ---- online softmax (rows g and g + 8)
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < NTA; ++nt) {
      mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
    }
    // Lazy reference maximum: it only moves when a score exceeds it by more than 2^LAZY (P <= 2^LAZY is harmless in
    // fp16, the sums are fp32).  The test is per lane on its own 2 x 2 NTA scores -- no quad shuffles on the common path;
    // only when some lane of the warp trips it are the row maxima reduced across the quad and the correction
    // (2 MUFU + the O / l rescale) applied, which after the first tiles is rare.
    if (__any_sync(0xffffffffu, mx0 > m0 + lazy || mx1 > m1 + lazy)) {
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);   // finite: every tile has >= 1 valid key
      const float cr0 = ex2((m0 - mn0) * scale_log2), cr1 = ex2((m1 - mn1) * scale_log2);
      m0 = mn0; m1 = mn1;
      ms0 = mn0 * scale_log2; ms1 = mn1 * scale_log2;
      lsum[0] *= cr0; lsum[1] *= cr0; lsum[2] *= cr1; lsum[3] *= cr1;
#pragma unroll
      for (int i = 0; i < NV; ++i) { o[i][0] *= cr0; o[i][1] *= cr0; o[i][2] *= cr1; o[i][3] *= cr1; }
    }
    // ---- P = exp2(.) packed to fp16 = A fragments of the second MMA;  O += P V,  l += P 1
#pragma unroll
    for (int kk = 0; kk < NG; ++kk) {
      uint32_t pa[4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float* sv = s[2 * kk + j];
        const float x0 = fmaf(sv[0], scale_log2, -ms0), x1 = fmaf(sv[1], scale_log2, -ms0);
        const float x2 = fmaf(sv[2], scale_log2, -ms1), x3 = fmaf(sv[3], scale_log2, -ms1);
        pa[2 * j] = pack_h2(ex2(x0), ex2(x1));
        pa[2 * j + 1] = pack_h2(ex2(x2), ex2(x3));
      }
      mma_f16(lsum, pa, ONES, ONES);
      const uint32_t vrow = sV + (uint32_t)(kk * 16 * STRIDE) * 2u;
#pragma unroll
      for (int vp = 0; vp < NV / 2; ++vp) {
        uint32_t r0, r1, r2, r3;
        ldsm_x4_t(vrow + v_lane_off + (uint32_t)(vp * 16) * 2u, r0, r1, r2, r3);
        mma_f16(o[2 * vp], pa, r0, r1);
        mma_f16(o[2 * vp + 1], pa, r2, r3);
      }
      if (NV & 1) {
        uint32_t r0, r1;
        // x2: lanes 0-15 supply the addresses (keys 0-7, keys 8-15 of the last 8-wide column tile)
        ldsm_x2_t(vrow + (uint32_t)((((lane >> 3) & 1) * 8 + lr) * STRIDE + (NV - 1) * 8) * 2u, r0, r1);
        mma_f16(o[NV - 1], pa, r0, r1);
      }
    }
  };

  // Ring of three GROUPS of SUB tiles, ONE block barrier per group: the barrier that publishes group g also proves every
  // warp has finished group g-1, whose slots are exactly the ones group g+2 is loaded into right after it.
  const bool active = q0 < L;
  const int ngroups = (ntiles + SUB - 1) / SUB;
  load_group(0);
  if (!RING2 && ngroups > 1) load_group(1);
  const bool ragged = (L % BK) != 0;
  for (int grp = 0; grp < ngroups; ++grp) {
    if (!RING2 && grp + 1 < ngroups) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (RING2) { if (grp + 1 < ngroups) load_group(grp + 1); }
    else if (grp + 2 < ngroups) load_group(grp + 2);
    if (active) {                                  // warps whose 16 query rows are all padding only help with the loads
#pragma unroll
      for (int hh = 0; hh < SUB; ++hh) {
        const int t = grp * SUB + hh;
        if (t >= ntiles) break;
        using G0_ = std::integral_constant<int, 0>;
        if constexpr (HALVES && BK == 64) {
          // the tile in two 32-key halves (S of a half = 16 registers instead of 32): at 7 CTAs per SM (72 registers) the
          // compiler otherwise re-derives every lane-dependent address from %tid inside the tile loop - ~40 % of the
          // instructions of a tile were that bookkeeping (ncu: 7.4 issued instructions per exponential)
          using G2_ = std::integral_constant<int, 2>;
          using N1_ = std::integral_constant<int, 1>;
          using N2_ = std::integral_constant<int, 2>;
          if (ragged && t == ntiles - 1) {
            const int groups = (L - t * BK + 15) / 16;
            if (groups == 1) tile_body(t, std::true_type{}, N1_{}, G0_{});
            else if (groups == 2) tile_body(t, std::true_type{}, N2_{}, G0_{});
            else {
              tile_body(t, std::false_type{}, N2_{}, G0_{});
              if (groups == 3) tile_body(t, std::true_type{}, N1_{}, G2_{});
              else tile_body(t, std::true_type{}, N2_{}, G2_{});
            }
          } else {
            tile_body(t, std::false_type{}, N2_{}, G0_{});
            tile_body(t, std::false_type{}, N2_{}, G2_{});
          }
        } else
        if (ragged && t == ntiles - 1) {
          const int groups = (L - t * BK + 15) / 16;
          if (groups == 1) tile_body(t, std::true_type{}, std::integral_constant<int, 1>{}, G0_{});
          if constexpr (BK >= 32) { if (groups == 2) tile_body(t, std::true_type{}, std::integral_constant<int, 2>{}, G0_{}); }
          if constexpr (BK >= 48) { if (groups == 3) tile_body(t, std::true_type{}, std::integral_constant<int, 3>{}, G0_{}); }
          if constexpr (BK >= 64) { if (groups == 4) tile_body(t, std::true_type{}, std::integral_constant<int, 4>{}, G0_{}); }
        } else {
          tile_body(t, std::false_type{}, std::integral_constant<int, BK / 16>{}, G0_{});
        }
        if (++cur_slot == NSLOT) cur_slot = 0;
      }
    }
  }

  // ---- normalise and store
  const float i0 = 1.0f / lsum[0], i1 = 1.0f / lsum[2];
  const int r0 = q0 + g, r1 = q0 + g + 8;
  __half* ob = out + (size_t)b * L * E + (size_t)h * d;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 8 + 2 * q4;
    if (c < d) {   // d is even, so c + 1 < d as well
      if (r0 < L) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * E + c) = pack_h2(o[i][0] * i0, o[i][1] * i0);
      if (r1 < L) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * E + c) = pack_h2(o[i][2] * i1, o[i][3] * i1);
    }
  }
}

template <int D, int BK, int NW, int VAR>
static int launch2(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  constexpr int DP = (D + 15) / 16 * 16;
  constexpr size_t SMEM = (size_t)((VAR & 4) ? 4 : 3) * 2 * BK * (DP + 8) * sizeof(__half);
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    CNB_CUDA(cudaFuncSetAttribute(attention_f16_kernel<D, BK, NW, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)SMEM));
  }
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)D);
  dim3 grid(ceil_div(L, 16 * NW), heads, B);
  CNB_CUDA(launch_pdl((long long)B * L * E, attention_f16_kernel<D, BK, NW, VAR>, grid, dim3(NW * 32), SMEM, st,
                      reinterpret_cast<const __half*>(qkv), reinterpret_cast<__half*>(out), L, E, scale_log2));
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

template <int D, int BK, int NW>
static int launch(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  // measured (profiles/r02_attention_table.md): halves pay everywhere at head dims <= 16; with them the kernel also fits
  // 64 registers = 8 CTAs (4 warps) / 4 CTAs (8 warps) per SM, which wins or ties except at d = 16 with 4 warps (spills)
  constexpr bool NARROW = BK == 64 && D <= 16;
  // halves, + the 64-register build where it does not spill, + two tiles per barrier for the 8-warp CTAs (measured:
  // L = 1024 d = 16 1362 -> 1311 us, L = 196 d = 16 88 -> 82 us; the 4-warp CTAs lose: L = 784 d = 16 854 -> 877 us)
  constexpr int HV = NARROW ? (((D == 16 && NW == 4) ? 1 : 3) | (NW == 8 ? 4 : 0)) : 0;
  return launch2<D, BK, NW, HV>(qkv, out, B, L, E, heads, st);
}

static inline long long padded(int L, int bq, int bk) {
  return (long long)ceil_div(L, bq) * bq * ((long long)ceil_div(L, bk) * bk);
}

// Tile choice: 64-key tiles (32 for the widest heads); 4 or 8 warps (64 / 128 queries) per CTA, whichever pads the
// sequence less (784 tokens: 13 x 64 = 832 beats 7 x 128 = 896); warp counts stay multiples of 4 so the four
// schedulers of an SM carry equal load.
template <int D, int BK>
static int launch_l(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  if (L <= 16) return launch<D, 16, 1>(qkv, out, B, L, E, heads, st);
  if (L <= 32) return launch<D, 32, 2>(qkv, out, B, L, E, heads, st);
  if (D > 64 || padded(L, 64, BK) < padded(L, 128, BK))
    return launch<D, BK, 4>(qkv, out, B, L, E, heads, st);
  return launch<D, BK, 8>(qkv, out, B, L, E, heads, st);
}

}  // namespace af16

bool attention_f16_supported(int E, int heads) {
  if (heads <= 0 || E % heads || E % 8) return false;
  const int d = E / heads;
  return d == 4 || d == 8 || d == 16 || d == 24 || d == 32 || d == 48 || d == 64 || d == 96 || d == 128 || d == 192;
}

int attention_f16(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  CNB_REQUIRE(B <= 65535 && heads <= 65535, "attention: grid too large (B=%d)", B);
  CNB_REQUIRE((((uintptr_t)qkv | (uintptr_t)out) & 15) == 0, "attention: qkv / out must be 16-byte aligned");
  const int d = E / heads;
  switch (d) {
    case 4: return af16::launch_l<4, 64>(qkv, out, B, L, E, heads, st);
    case 8: return af16::launch_l<8, 64>(qkv, out, B, L, E, heads, st);
    case 16: return af16::launch_l<16, 64>(qkv, out, B, L, E, heads, st);
    case 24: return af16::launch_l<24, 64>(qkv, out, B, L, E, heads, st);
    case 32: return af16::launch_l<32, 32>(qkv, out, B, L, E, heads, st);   // measured: 154 -> 137 us at L = 196, E = 128
    case 48: return af16::launch_l<48, 64>(qkv, out, B, L, E, heads, st);
    case 64: return af16::launch_l<64, 64>(qkv, out, B, L, E, heads, st);
    case 96: return af16::launch_l<96, 32>(qkv, out, B, L, E, heads, st);
    case 128: return af16::launch_l<128, 32>(qkv, out, B, L, E, heads, st);
    case 192: return af16::launch_l<192, 32>(qkv, out, B, L, E, heads, st);
    default:
      set_error("attention_f16: head dim %d not instantiated", d);
      return CNB_ERR_UNSUPPORTED;
  }
}

}  // namespace cnb
