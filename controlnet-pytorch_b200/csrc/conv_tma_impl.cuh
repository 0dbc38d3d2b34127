// TMA-fed, persistent, warp-specialised tcgen05 implicit-GEMM convolution (the wide-channel path of cnb_conv2d).
//
//   GEMM view     M = B*OH*OW output pixels (tile 128 = one UMMA M), N = Cout (tile BN in {16..256}, one CTA usually
//                 owns the full Cout), K = ntaps*Cin walked as (tap, channel chunk) with a chunk = one 128-byte
//                 SWIZZLE_128B row: 64 fp16 (kind::f16) or 32 fp32 (kind::tf32) channels.
//   A operand     cp.async.bulk.tensor.4d ... im2col: ONE instruction gathers the 128 pixels x chunk channels of a tap
//                 straight from the channels-last activation tensor [B, H, W, ldi] into the canonical K-major
//                 SWIZZLE_128B tile (zero fill outside the image and past the last pixel); the tap is the
//                 instruction's {offset_w, offset_h}, the conv stride is the tensor map's traversal stride.
//   B operand     cp.async.bulk.tensor.2d tile {chunk, BN} of the packed weights [Cout][ntaps*Cin].
//   roles         warp 0 = TMA producer (one elected lane), warp 1 = tcgen05.mma issuer (one elected lane, fp32
//                 accumulators in TMEM, double buffered: 2 x BN columns), warps 2..5 = epilogue (TMEM -> registers ->
//                 per-warp smem slab -> coalesced channels-last stores with + bias + time-embedding row + residual
//                 (+SiLU), fp32 or fp16 out).  S-stage smem ring with full/empty mbarriers; tmem_full/tmem_empty
//                 mbarriers hand accumulators between the MMA warp and the epilogue, so the epilogue of tile i overlaps
//                 the main loop of tile i+1.
//   schedule      persistent: grid = min(#tiles, #SMs), tile = blockIdx.x + k*gridDim.x, n-tile fastest.
//
// Every mbarrier wait is bounded (tc_common.cuh): a broken pipeline raises the hang-guard flag and drains.
#include <cuda.h>   // CUtensorMap + enums only; the encoders are resolved at run time (no link against libcuda)
#include <cuda_fp16.h>
#pragma once
#include <stdlib.h>
#include <string.h>

#include "tc_common.cuh"

namespace cnb {
namespace tma {

using namespace tc;

constexpr int BM = 128;
constexpr int EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;   // warp 0: TMA, warp 1: MMA, warps 2..9: epilogue
constexpr int SMEM_BUDGET = 227 * 1024;

struct alignas(64) TmaArgs {
  CUtensorMap map_a;
  CUtensorMap map_a2;   // optional second input (one (0,0) tap appended to K); used when kchunks2 > 0
  CUtensorMap map_b;
  CUtensorMap map_out;  // EPI 6: fp16 output rows [M][Cout] (pitch ldo), box {SLAB, 32}, swizzle = row bytes
  CUtensorMap map_res;  // EPI 6: fp16 residual rows, same box
  const float* bias;
  const float* temb;
  const void* residual;
  void* out;
  int M, OHW, OW;
  int OHf, OWf, oy_mul, oy_add, ox_mul, ox_add;
  int Cout, ldo, out_coff, ldr, res_coff, temb_ld, temb_per_sample, act, out_f16, res_f16;
  int Cin, ntaps, kchunks, kchunks2;
  int stride, lower_w, lower_h;
  int tiles_m, tiles_n;
  // shared-memory plan (runtime: the resident-weights variant trades ring depth for a [nkb][BN x RB] weight area)
  // halo mode (3x3, stride 1, pad 1): a stage holds (R+2) x (W+2) input pixels of one channel chunk, loaded ONCE by a
  // tiled TMA (zero fill outside the image), and the 9 taps are 9 MMAs whose A descriptors start dy*(W+2)+dx rows
  // further into the same tile.  GEMM rows are padded-flat positions y*(W+2)+x of R image rows; x >= W is discarded.
  int halo, Wp, R, tiles_y, H, W, halo_stage_bytes;
  int bres;         // 1 = the whole packed weight tile stays resident in smem, the ring carries A stages only
  int s_run;        // ring depth actually used (<= Cfg::S)
  int ring_off, stage_bytes, epi_off, bar_off;
  int epi_alt;      // 1 = the two epilogue warp groups alternate TILES (short-K layers), 0 = they split a tile's columns
  int tma_epi;      // 1 = host built map_out (/ map_res): the dense fp16 epilogue may run through TMA (EPI 6)
  int epi_nbuf;     // EPI 6: staging buffers per epilogue warp (2 or 3)
  uint32_t tap_off[CNB_MAX_TAPS];   // offset_w | offset_h << 16
};

__device__ __forceinline__ void tma_load_im2col_4d(uint32_t dst, const void* map, uint64_t* bar, int c, int w, int h,
                                                   int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n),
        "h"(off_w), "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void tma_load_tiled_4d(uint32_t dst, const void* map, uint64_t* bar, int c, int w, int h,
                                                  int n) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n)
      : "memory");
}
__device__ __forceinline__ float4 ld_half4(const __half* p) {
  const uint2 raw = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
  const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}

__device__ __forceinline__ void tma_store_2d(const void* map, uint32_t src, int x, int y) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

constexpr int pow2_at_least(int v, int p = 32) { return p >= v ? p : pow2_at_least(v, p * 2); }

// RB = bytes of K per smem row = the swizzle span: 128 (SWIZZLE_128B), 64 (SWIZZLE_64B) or 32 (SWIZZLE_32B); a stage holds
// RB / sizeof(element) channels of one tap, so layers with 16 or 32 input channels still run one tap per stage.
template <int BN, int RB>
struct Cfg {
  static constexpr int A_STAGE_BYTES = BM * RB;
  static constexpr int SLAB = (BN % 64 == 0) ? 32 : 16;   // epilogue column slab; BN / SLAB is even where it can be
  static constexpr int SLAB_STRIDE = SLAB + 4;            // floats
  static constexpr int EPI_BYTES = EPI_WARPS * 32 * SLAB_STRIDE * 4;
  static constexpr int B_STAGE_BYTES = BN * RB;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int BAR_BYTES = 512;                   // ring / accumulator barriers + 3 per epilogue warp (EPI 6)
  // EPI 6 (dense fp16 out through TMA): per epilogue warp NB staging buffers of 32 rows x SLAB fp16 (swizzled rows of
  // SLAB * 2 bytes) + the bias (+ time-embedding row) of the slabs the warp owns; NB = 2 fits EPI_BYTES for every BN
  static constexpr int E6_BUF = 32 * SLAB * 2;
  static constexpr int E6_BIAS = (((BN / SLAB + 1) / 2) * SLAB * 4 + 511) / 512 * 512;
  __host__ __device__ static constexpr int e6_warp_bytes(int nb) { return nb * E6_BUF + E6_BIAS; }
  static constexpr int S_RAW = (SMEM_BUDGET - 1024 - EPI_BYTES - BAR_BYTES) / STAGE_BYTES;
  static constexpr int S = S_RAW > 8 ? 8 : S_RAW;
  static constexpr int EPI_OFFSET = S * STAGE_BYTES;
  static constexpr int BAR_OFFSET = EPI_OFFSET + EPI_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + BAR_BYTES + 1024;   // + alignment slack
  static constexpr int ACC_STRIDE = pow2_at_least(BN);
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  static_assert(S >= 2, "pipeline needs at least two stages");
  static_assert(EPI_WARPS * (2 * E6_BUF + E6_BIAS) <= EPI_BYTES, "EPI 6 staging (two buffers) must fit the epilogue area");
  static_assert(TMEM_COLS <= 512, "accumulators exceed TMEM");
  static_assert(A_STAGE_BYTES % (8 * RB) == 0 && B_STAGE_BYTES % (8 * RB) == 0,
                "operand tiles must keep swizzle-atom alignment (8 rows x RB bytes)");
};

// EPI selects the epilogue: 0 = dense fp32 out, 1 = dense fp32 out + fp32 residual, 2 = dense fp16 out,
// 4 = dense fp16 out + fp16 residual (the fp16 activation stream), 5 = halo tiles with fp16 out (+ fp16 residual),
// 6 = dense fp16 out (+ fp16 residual) staged per warp and moved by TMA (the default for the fp16 stream), 3 = generic.
template <int BN, bool HALF, int EPI, int RB>
__global__ void __launch_bounds__(NUM_THREADS, (BN <= 128 && EPI != 3) ? 2 : 1)   // two CTAs per SM: <= 102 registers
conv_tma_kernel(const __grid_constant__ TmaArgs a) {
  using C = Cfg<BN, RB>;
  constexpr int S = C::S;
  constexpr int KC = RB / (HALF ? 2 : 4);            // channels per stage
  constexpr int A_STAGE_BYTES = C::A_STAGE_BYTES;
  constexpr uint32_t IDESC = make_idesc(BM, BN, HALF);
  constexpr int SLAB = C::SLAB;
  constexpr int SSTR = C::SLAB_STRIDE;

  pdl_trigger();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  const uint32_t smem_base = raw_addr + pad;

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + a.bar_off);       // [S]
  uint64_t* empty_bar = full_bar + S;                                       // [S]
  uint64_t* tfull_bar = empty_bar + S;                                      // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;                                     // [2] accumulator drained
  uint64_t* bres_bar = tempty_bar + 2;                                      // [1] resident weights landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_bar + 1);
  const int s_run = a.s_run;
  const uint32_t ring_base = smem_base + (uint32_t)a.ring_off;
  const uint32_t stage_bytes = (uint32_t)a.stage_bytes;
  const bool bres = a.bres != 0;
  volatile int* abort_flag = reinterpret_cast<volatile int*>(tmem_slot + 1);
  uint64_t* e6_bar = reinterpret_cast<uint64_t*>(smem + a.bar_off + 192);   // [EPI_WARPS][3] residual landed (EPI 6)

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int nkb = a.ntaps * a.kchunks + a.kchunks2;
  const int ntiles = a.tiles_m * a.tiles_n;

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], a.epi_alt ? EPI_WARPS / 2 : EPI_WARPS);
    }
    mbar_init(bres_bar, 1);
    if (EPI == 6)
      for (int i = 0; i < EPI_WARPS * 3; ++i) mbar_init(&e6_bar[i], 1);
    *abort_flag = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  if (warp == 0 && lane == 0) {                  // descriptor fetches overlap the previous kernel's tail (before pdl_wait)
    prefetch_tensormap(&a.map_a);
    prefetch_tensormap(&a.map_b);
    if (a.kchunks2 > 0) prefetch_tensormap(&a.map_a2);
  }
  if (EPI == 6 && warp == 2 && lane == 0) {
    prefetch_tensormap(&a.map_out);
    if (a.residual) prefetch_tensormap(&a.map_res);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();      // everything above overlapped the previous kernel's tail; no global memory touched yet

  if (warp == 0) {
    // ============================ TMA producer ============================
    if (lane == 0) {
      if (bres) {
        // resident weights: every k-block's {chunk, BN} tile once per CTA (tiles_n == 1)
        mbar_expect_tx(bres_bar, (uint32_t)(nkb * C::B_STAGE_BYTES));
        int kb = 0;
        for (int tap = 0; tap < a.ntaps; ++tap)
          for (int kc = 0; kc < a.kchunks; ++kc, ++kb)
            tma_load_2d(smem_base + (uint32_t)(kb * C::B_STAGE_BYTES), &a.map_b, bres_bar, tap * a.Cin + kc * KC, 0);
        for (int kc = 0; kc < a.kchunks2; ++kc, ++kb)
          tma_load_2d(smem_base + (uint32_t)(kb * C::B_STAGE_BYTES), &a.map_b, bres_bar, a.ntaps * a.Cin + kc * KC, 0);
      }
      uint32_t tx = bres ? (uint32_t)A_STAGE_BYTES : (uint32_t)C::STAGE_BYTES;
      int s = 0, round = 0;
      bool ok = true;
      auto stage_begin = [&]() -> uint32_t {      // waits for the slot, arms its barrier, returns its smem address
        if (round > 0) ok = mbar_wait(&empty_bar[s], (uint32_t)((round - 1) & 1), abort_flag);
        if (ok) mbar_expect_tx(&full_bar[s], tx);
        return ring_base + (uint32_t)s * stage_bytes;
      };
      auto stage_end = [&]() {
        if (++s == s_run) { s = 0; ++round; }
      };
      if (a.halo) {
        for (int tile = blockIdx.x; tile < ntiles && ok; tile += gridDim.x) {
          const int b = tile / a.tiles_y;
          const int y0 = (tile - b * a.tiles_y) * a.R;
          tx = (uint32_t)((a.R + 2) * a.Wp * RB);
          for (int kc = 0; kc < a.kchunks && ok; ++kc) {
            const uint32_t sa = stage_begin();
            if (!ok) break;
            tma_load_tiled_4d(sa, &a.map_a, &full_bar[s], kc * KC, -1, y0 - 1, b);
            stage_end();
          }
          tx = (uint32_t)(a.R * a.Wp * RB);
          for (int kc = 0; kc < a.kchunks2 && ok; ++kc) {
            const uint32_t sa = stage_begin();
            if (!ok) break;
            tma_load_tiled_4d(sa, &a.map_a2, &full_bar[s], kc * KC, 0, y0, b);
            stage_end();
          }
        }
      } else
      for (int tile = blockIdx.x; tile < ntiles && ok; tile += gridDim.x) {
        const int mt = tile / a.tiles_n, nt = tile - mt * a.tiles_n;
        const int m0 = mt * BM;
        const int b = m0 / a.OHW;
        const int rem = m0 - b * a.OHW;
        const int oy = rem / a.OW;
        const int ox = rem - oy * a.OW;
        const int w0 = ox * a.stride + a.lower_w, h0 = oy * a.stride + a.lower_h;
        // K is walked chunk-major (channel chunk outer, tap inner) -- the same order as the halo mode, so the fp32
        // accumulation sequence of every output element, and with it the result, does not depend on which of the two
        // plans the batch size selects (batch / shard invariance, tests/test_models_gpu.py)
        for (int kc = 0; kc < a.kchunks && ok; ++kc) {
          for (int tap = 0; tap < a.ntaps; ++tap) {
            const uint32_t off = a.tap_off[tap];
            const uint32_t sa = stage_begin();
            if (!ok) break;
            tma_load_im2col_4d(sa, &a.map_a, &full_bar[s], kc * KC, w0, h0, b, (uint16_t)(off & 0xffffu),
                               (uint16_t)(off >> 16));
            if (!bres) tma_load_2d(sa + A_STAGE_BYTES, &a.map_b, &full_bar[s], tap * a.Cin + kc * KC, nt * BN);
            stage_end();
          }
        }
        // second input: one (0,0) tap over the output grid, weight columns after the ntaps*Cin of the main input
        for (int kc = 0; kc < a.kchunks2 && ok; ++kc) {
          const uint32_t sa = stage_begin();
          if (!ok) break;
          tma_load_im2col_4d(sa, &a.map_a2, &full_bar[s], kc * KC, ox, oy, b, (uint16_t)0, (uint16_t)0);
          if (!bres) tma_load_2d(sa + A_STAGE_BYTES, &a.map_b, &full_bar[s], a.ntaps * a.Cin + kc * KC, nt * BN);
          stage_end();
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ============================
    int s = 0, round = 0, tcount = 0;
    bool ok = true;
    if (bres) ok = mbar_wait(bres_bar, 0u, abort_flag);
    for (int tile = blockIdx.x; tile < ntiles && ok; tile += gridDim.x, ++tcount) {
      const int acc = tcount & 1;
      if (tcount >= 2) ok = mbar_wait(&tempty_bar[acc], (uint32_t)(((tcount >> 1) - 1) & 1), abort_flag);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * C::ACC_STRIDE);
      if (a.halo) {
        // One thread issues 9 taps x RB/32 MMAs per stage, so the descriptor arithmetic is kept to 64-bit adds: the
        // tap's row shift and the weight block's offset are both expressed in the descriptor's 16-byte address units.
        const int nstage = a.kchunks + a.kchunks2;
        const uint64_t b_first = make_desc_kmajor<RB>(smem_base);
        const uint64_t b_blk = (uint64_t)(C::B_STAGE_BYTES >> 4);
        const uint64_t b_tap = b_blk * (uint64_t)a.kchunks;          // consecutive taps of one channel chunk
        const uint64_t a_row = (uint64_t)(a.Wp * RB) >> 4;           // one padded image row
        for (int st = 0; st < nstage && ok; ++st) {
          ok = mbar_wait(&full_bar[s], (uint32_t)(round & 1), abort_flag);
          tc_fence_after();
          if (lane == 0 && ok) {
            const uint64_t abase = make_desc_kmajor<RB>(ring_base + (uint32_t)s * stage_bytes);
            if (st < a.kchunks) {
              const uint64_t bbase = b_first + b_blk * (uint64_t)st;
#pragma unroll
              for (int tap = 0; tap < 9; ++tap) {
                const uint64_t adesc = abase + a_row * (uint64_t)(tap / 3) + (uint64_t)((tap % 3) * (RB >> 4));
                const uint64_t bdesc = bbase + b_tap * (uint64_t)tap;
#pragma unroll
                for (int k = 0; k < RB / 32; ++k)
                  umma<HALF>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, (st | tap | k) ? 1u : 0u);
              }
            } else {
              const uint64_t bdesc = b_first + b_tap * 9ull + b_blk * (uint64_t)(st - a.kchunks);
#pragma unroll
              for (int k = 0; k < RB / 32; ++k)
                umma<HALF>(d_tmem, abase + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, 1u);
            }
            umma_commit(&empty_bar[s]);
            if (st == nstage - 1) umma_commit(&tfull_bar[acc]);
          }
          __syncwarp();
          if (++s == s_run) { s = 0; ++round; }
        }
      } else
      for (int kb = 0, tap = 0, kc = 0; kb < nkb && ok; ++kb) {
        ok = mbar_wait(&full_bar[s], (uint32_t)(round & 1), abort_flag);
        tc_fence_after();
        // stages arrive chunk-major (kc outer, tap inner); the resident weight blocks are stored tap-major
        const int bidx = kb < a.ntaps * a.kchunks ? tap * a.kchunks + kc : kb;
        if (++tap == a.ntaps) { tap = 0; ++kc; }
        if (lane == 0 && ok) {
          const uint32_t a_addr = ring_base + (uint32_t)s * stage_bytes;
          const uint64_t adesc = make_desc_kmajor<RB>(a_addr);
          const uint64_t bdesc = make_desc_kmajor<RB>(bres ? smem_base + (uint32_t)(bidx * C::B_STAGE_BYTES)
                                                           : a_addr + A_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < RB / 32; ++k)
            umma<HALF>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, (kb | k) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
          if (kb == nkb - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++s == s_run) { s = 0; ++round; }
      }
    }
    tc_fence_before();
  } else {
    // ============================ epilogue (warps 2..9) ============================
    // Two warps share each TMEM lane quarter (q = warp % 4).  Long-K layers: they split the accumulator's column slabs by
    // parity.  Short-K layers (epi_alt): a tile's MMAs take a few hundred cycles while its epilogue is a ~2-3 k cycle
    // latency chain (barrier wake-up, tcgen05.ld, smem transpose, residual loads, stores), so the two warp groups take
    // alternate TILES (= alternate TMEM accumulators) and two epilogues are in flight at once.
    // With one warp per scheduler the epilogue is instruction-latency bound, so the dense variants (EPI 0..2) keep
    // the per-row work to LDS.128 (+LDG.128 residual) + 4 FADD + STG and fully unroll it.
    const int ew = warp - 2;
    const int q = warp & 3;
    const int par = ew >> 2;
    if constexpr (EPI == 6) {
      // ---- dense fp16 output (+ fp16 residual) through TMA.  A lane owns one accumulator row (tcgen05.ld 32x32b), so a
      // slab of SLAB columns is SLAB * 2 contiguous bytes per lane: it goes bias-added and packed into a per-warp staging
      // buffer (rows swizzled like the tensor map: 16-byte stores of eight lanes hit eight different bank groups) and
      // leaves as ONE cp.async.bulk.tensor store of the 32 x SLAB box; the residual box arrives the same way, one slab
      // ahead, into the buffer it is then added to in place.  No transposing round trip through shared memory, no
      // per-row address arithmetic, no global-load latency inside the per-slab chain; the M tail is the tensor map's.
      constexpr int NSLAB = BN / SLAB;
      constexpr int ROWB = SLAB * 2;
      constexpr int BUF = C::E6_BUF;
      constexpr int CH = ROWB / 16;                            // 16-byte chunks per staged row
      const int nb = a.epi_nbuf;
      const uint32_t wb_off = (uint32_t)a.epi_off + (uint32_t)ew * (uint32_t)C::e6_warp_bytes(nb);
      uint8_t* wbase = smem + wb_off;
      const uint32_t wbase_u = smem_base + wb_off;
      float* bias_s = reinterpret_cast<float*>(wbase + nb * BUF);
      uint64_t* rbar = e6_bar + ew * 3;
      const bool has_res = a.residual != nullptr;
      const float* bias = a.bias;
      const float* temb_row = (a.temb && !a.temb_per_sample) ? a.temb : nullptr;
      const bool has_bias = bias != nullptr || temb_row != nullptr;
      const int M = a.M, tiles_n = a.tiles_n;
      const int si0 = par, sstep = 2;                          // the two warps of a lane quarter split the slabs by parity
      const bool has_items = si0 < NSLAB;
      const int sw = SLAB == 32 ? ((lane >> 1) & 3) : ((lane >> 2) & 1);   // SWIZZLE_64B / _32B pattern of this lane's row
      auto issue_res = [&](int tile_, int si_, int buf_) {     // lane 0: residual box of one (tile, slab) -> buffer buf_
        const int mt_ = tile_ / tiles_n, nt_ = tile_ - mt_ * tiles_n;
        const int m_ = mt_ * BM + q * 32;
        if (m_ < M) {
          mbar_expect_tx(&rbar[buf_], (uint32_t)BUF);
          tma_load_2d(wbase_u + (uint32_t)(buf_ * BUF), &a.map_res, &rbar[buf_], nt_ * BN + si_ * SLAB, m_);
        }
      };
      int cb = 0;                                              // staging buffer of the current slab
      uint32_t rphase = 0;                                     // bit b: parity of the next completion of rbar[b]
      int last_nt = -1, tcount = 0;
      int tile = blockIdx.x;
      if (has_res && has_items && tile < ntiles && lane == 0) issue_res(tile, si0, 0);
      bool ok = true;
      for (; tile < ntiles && ok; tile += gridDim.x, ++tcount) {
        const int mt = tile / tiles_n, nt = tile - mt * tiles_n;
        const int m_w = mt * BM + q * 32;
        const int n0 = nt * BN;
        if (has_items && has_bias && nt != last_nt) {          // bias (+ time-embedding row) of this warp's slabs
          __syncwarp();
          int k = 0;
          for (int si = si0; si < NSLAB; si += sstep, ++k) {
            if (lane < SLAB) {
              const int n = n0 + si * SLAB + lane;
              float v = bias ? __ldg(bias + n) : 0.f;
              if (temb_row) v += __ldg(temb_row + n);
              bias_s[k * SLAB + lane] = v;
            }
          }
          last_nt = nt;
          __syncwarp();
        }
        const int acc = tcount & 1;
        if (!mbar_wait(&tfull_bar[acc], (uint32_t)((tcount >> 1) & 1), abort_flag)) break;
        tc_fence_after();
        const uint32_t t_addr = tmem_base + (uint32_t)(acc * C::ACC_STRIDE) + ((uint32_t)(q * 32) << 16);
        if (!has_items) {                                      // single-slab tiles: the odd warps have nothing to read
          tc_fence_before();
          if (lane == 0) mbar_arrive(&tempty_bar[acc]);
          continue;
        }
        const bool rows_valid = m_w < M;                       // warp-uniform: the whole 32-row box is past the M tail
        int k = 0;
#pragma unroll 1
        for (int si = si0; si < NSLAB; si += sstep, ++k) {
          uint32_t r[SLAB];
#pragma unroll
          for (int j = 0; j < SLAB / 16; ++j) tmem_ld16_nowait(t_addr + (uint32_t)(si * SLAB + 16 * j), r + 16 * j);
          if (lane == 0) {
            if (has_res) {
              // the slab after this one (possibly of the next tile): its buffer was last read by the store nb slabs back
              int ntile = tile, nsi = si + sstep;
              if (nsi >= NSLAB) { ntile = tile + gridDim.x; nsi = si0; }
              if (ntile < ntiles) {
                if (nb == 2) bulk_wait_read<0>(); else bulk_wait_read<1>();
                issue_res(ntile, nsi, cb + 1 == nb ? 0 : cb + 1);
              }
            } else {
              if (nb == 2) bulk_wait_read<1>(); else bulk_wait_read<2>();   // the store that last read buffer cb
            }
          }
          tmem_ld_wait();
          if (si + sstep >= NSLAB) {                           // this warp's last slab: hand its share of the accumulator back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
          }
          if (rows_valid) {
            if (has_res) {
              ok = mbar_wait(&rbar[cb], (rphase >> cb) & 1u, abort_flag);
              rphase ^= 1u << cb;
              if (!ok) break;
            } else {
              __syncwarp();                                    // lane 0 has seen buffer cb released
            }
            uint8_t* row = wbase + cb * BUF + lane * ROWB;
            const float4* b4 = reinterpret_cast<const float4*>(bias_s + k * SLAB);
#pragma unroll
            for (int j = 0; j < CH; ++j) {
              uint4* cell = reinterpret_cast<uint4*>(row + ((j ^ sw) << 4));
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[8 * j + e]);
              if (has_bias) {
                const float4 b0 = b4[2 * j], b1 = b4[2 * j + 1];
                v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
                v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
              }
              if (has_res) {
                const uint4 rr = *cell;
                const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&rw[e]));
                  v[2 * e] += f.x; v[2 * e + 1] += f.y;
                }
              }
              uint32_t o[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const __half2 h = h2_sat(v[2 * e], v[2 * e + 1]);
                o[e] = *reinterpret_cast<const uint32_t*>(&h);
              }
              *cell = make_uint4(o[0], o[1], o[2], o[3]);
            }
            fence_proxy_async();
          }
          __syncwarp();
          if (lane == 0) {
            if (rows_valid) tma_store_2d(&a.map_out, wbase_u + (uint32_t)(cb * BUF), n0 + si * SLAB, m_w);
            bulk_commit();                                     // an empty group for skipped boxes keeps the group count in step
          }
          cb = cb + 1 == nb ? 0 : cb + 1;
        }
      }
      if (lane == 0) bulk_wait_all();                          // the staging buffers must outlive the stores' reads
      tc_fence_before();
    } else {
    float* slab = reinterpret_cast<float*>(smem + a.epi_off) + (size_t)ew * 32 * SSTR;
    constexpr int NSLAB = BN / SLAB;
    constexpr int LPR = SLAB / 4;                             // lanes per row in the coalesced pass
    constexpr int RPI = 32 / LPR;                             // rows per iteration
    const int sub_r = lane / LPR, sub_c = (lane % LPR) * 4;
    const int M = a.M, ldo = a.ldo, ldr = a.ldr, tiles_n = a.tiles_n;
    const float* bias = a.bias;
    const float* temb_row = (a.temb && !a.temb_per_sample) ? a.temb : nullptr;
    int tcount = 0;
    const bool alt = a.epi_alt != 0;
    const int si0 = alt ? 0 : par, sstep = alt ? 1 : 2;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      if (alt && (tcount & 1) != par) continue;               // the other warp group owns this accumulator
      const int mt = tile / tiles_n, nt = tile - mt * tiles_n;
      const int m_w = mt * BM + q * 32;                       // first GEMM row of this warp
      const int n0 = nt * BN;
      long long pix = -1;
      int b = 0;
      int pixi = -1;                                          // EPI 5: 32-bit output pixel index of this lane's row
      if (EPI == 5) {
        const int r = q * 32 + lane;
        const int bb = tile / a.tiles_y;
        const int yy = r / a.Wp, xx = r - yy * a.Wp;
        const int y = (tile - bb * a.tiles_y) * a.R + yy;
        if (yy < a.R && xx < a.W && y < a.H) pixi = (bb * a.H + y) * a.W + xx;
      }
      if (EPI == 3 && a.halo) {
        const int r = q * 32 + lane;                          // padded-flat position inside the tile
        b = tile / a.tiles_y;
        const int yy = r / a.Wp, xx = r - yy * a.Wp;
        const int y = (tile - b * a.tiles_y) * a.R + yy;
        if (yy < a.R && xx < a.W && y < a.H) pix = ((long long)b * a.H + y) * a.W + xx;
      } else if (EPI == 3) {
        const int m = m_w + lane;
        if (m < M) {
          b = m / a.OHW;
          const int rem = m - b * a.OHW;
          const int oy = rem / a.OW;
          const int ox = rem - oy * a.OW;
          pix = ((long long)b * a.OHf + (oy * a.oy_mul + a.oy_add)) * a.OWf + (ox * a.ox_mul + a.ox_add);
        }
      }
      // Halo tiles: the residual rows of this warp's first slab are fetched BEFORE the accumulator is waited for, so
      // their ~1 us global latency overlaps the tile's MMAs instead of being exposed once per tile (3x3 64->64 @28 +
      // residual: 220 -> 141 us).
      float4 rv[32 / RPI];
      auto load_residual = [&](int si) {
        const int n = n0 + si * SLAB + sub_c;
        if (EPI == 5) {
          const __half* resh = reinterpret_cast<const __half*>(a.residual);
          if (resh) {
#pragma unroll
            for (int i = 0; i < 32 / RPI; ++i) {
              const int rp = __shfl_sync(0xffffffffu, pixi, i * RPI + sub_r);
              rv[i] = rp >= 0 ? ld_half4(resh + (size_t)rp * ldr + a.res_coff + n) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
        } else if (EPI == 1 || EPI == 4) {
          const int rows_left = M - m_w - sub_r;
#pragma unroll
          for (int i = 0; i < 32 / RPI; ++i) {
            if (i * RPI < rows_left) {
              const size_t off = (size_t)(m_w + sub_r + i * RPI) * ldr + a.res_coff + n;
              rv[i] = EPI == 1 ? __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(a.residual) + off))
                               : ld_half4(reinterpret_cast<const __half*>(a.residual) + off);
            }
          }
        }
      };
      const int si_first = alt ? 0 : par;
      if (EPI == 5 && si_first < NSLAB) load_residual(si_first);
      const int acc = tcount & 1;
      if (!mbar_wait(&tfull_bar[acc], (uint32_t)((tcount >> 1) & 1), abort_flag)) break;
      tc_fence_after();
      const uint32_t t_addr = tmem_base + (uint32_t)(acc * C::ACC_STRIDE) + ((uint32_t)(q * 32) << 16);
      if (!alt && par >= NSLAB) {                             // single-slab tiles: the odd warps have nothing to read
        tc_fence_before();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      }
#pragma unroll 1
      for (int si = si0; si < NSLAB; si += sstep) {
        const int c0 = si * SLAB;
        uint32_t r[SLAB];
#pragma unroll
        for (int j = 0; j < SLAB / 16; ++j) tmem_ld16_nowait(t_addr + (uint32_t)(c0 + 16 * j), r + 16 * j);
        if (EPI == 5 && si != si_first) load_residual(si);   // later slabs of halo tiles: overlaps tcgen05.ld + transpose
        tmem_ld_wait();
        if (si + sstep >= NSLAB) {        // this warp's last slab: hand its share of the TMEM buffer back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        }
        float4* d = reinterpret_cast<float4*>(slab + (size_t)lane * SSTR);
#pragma unroll
        for (int j = 0; j < SLAB / 4; ++j)
          d[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                             __uint_as_float(r[4 * j + 3]));
        __syncwarp();
        const int n = n0 + c0 + sub_c;                        // < Cout: BN divides Cout
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (bias) bv = __ldg(reinterpret_cast<const float4*>(bias + n));
        if (temb_row) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(temb_row + n));
          bv.x += t.x; bv.y += t.y; bv.z += t.z; bv.w += t.w;
        }
        if (EPI == 5) {
          // ---- halo tiles, fp16 activation stream: row -> pixel through one shuffle, fp16 out (+ fp16 residual)
          const __half* resh = reinterpret_cast<const __half*>(a.residual);
          __half* outh = reinterpret_cast<__half*>(a.out);
#pragma unroll
          for (int i = 0; i < 32 / RPI; ++i) {
            const int rp = __shfl_sync(0xffffffffu, pixi, i * RPI + sub_r);
            if (rp >= 0) {
              float4 o = *reinterpret_cast<const float4*>(slab + (size_t)(i * RPI + sub_r) * SSTR + sub_c);
              o.x += bv.x; o.y += bv.y; o.z += bv.z; o.w += bv.w;
              if (resh) { o.x += rv[i].x; o.y += rv[i].y; o.z += rv[i].z; o.w += rv[i].w; }
              const __half2 lo = h2_sat(o.x, o.y), hi = h2_sat(o.z, o.w);
              *reinterpret_cast<uint2*>(outh + (size_t)rp * ldo + a.out_coff + n) =
                  make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
            }
          }
        } else if (EPI != 3) {
          // ---- dense output: GEMM row m is output pixel m
          const int rows_left = M - m_w - sub_r;              // row rr + sub_r is valid iff rr < rows_left
          const float* sp = slab + (size_t)sub_r * SSTR + sub_c;
          const size_t o_off = (size_t)(m_w + sub_r) * ldo + a.out_coff + n;
          // dense tiles fetch the residual here, right before it is consumed: issuing it before the accumulator wait or
          // before tcgen05.wait::ld measured SLOWER on the BN = 256 layers (1x1 256->256 @7: 34 -> 39-42 us)
          if (EPI == 1 || EPI == 4) load_residual(si);
#pragma unroll
          for (int i = 0; i < 32 / RPI; ++i) {
            if (i * RPI < rows_left) {
              float4 o = *reinterpret_cast<const float4*>(sp + i * RPI * SSTR);
              o.x += bv.x; o.y += bv.y; o.z += bv.z; o.w += bv.w;
              if (EPI == 1 || EPI == 4) { o.x += rv[i].x; o.y += rv[i].y; o.z += rv[i].z; o.w += rv[i].w; }
              if (EPI == 2 || EPI == 4) {
                const __half2 lo = h2_sat(o.x, o.y), hi = h2_sat(o.z, o.w);
                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(a.out) + o_off + (size_t)i * RPI * ldo) =
                    make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
              } else {
                *reinterpret_cast<float4*>(reinterpret_cast<float*>(a.out) + o_off + (size_t)i * RPI * ldo) = o;
              }
            }
          }
        } else {
          // ---- generic output mapping (ConvTranspose phases, per-sample time embedding, SiLU, fp16 + residual)
#pragma unroll 2
          for (int rr = 0; rr < 32; rr += RPI) {
            const int row = rr + sub_r;
            const long long rp = __shfl_sync(0xffffffffu, pix, row);
            const int rb = __shfl_sync(0xffffffffu, b, row);
            if (rp >= 0) {
              float4 o = *reinterpret_cast<const float4*>(slab + (size_t)row * SSTR + sub_c);
              o.x += bv.x; o.y += bv.y; o.z += bv.z; o.w += bv.w;
              if (a.temb && a.temb_per_sample) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(a.temb + (size_t)rb * a.temb_ld + n));
                o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w;
              }
              if (a.residual) {
                const float4 t = a.res_f16
                    ? ld_half4(reinterpret_cast<const __half*>(a.residual) + rp * ldr + a.res_coff + n)
                    : __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(a.residual) + rp * ldr +
                                                            a.res_coff + n));
                o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w;
              }
              if (a.act == 1) { o.x = silu_f(o.x); o.y = silu_f(o.y); o.z = silu_f(o.z); o.w = silu_f(o.w); }
              if (a.out_f16) {
                const __half2 lo = h2_sat(o.x, o.y), hi = h2_sat(o.z, o.w);
                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(a.out) + rp * ldo + a.out_coff + n) =
                    make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
              } else {
                *reinterpret_cast<float4*>(reinterpret_cast<float*>(a.out) + rp * ldo + a.out_coff + n) = o;
              }
            }
          }
        }
        __syncwarp();
      }
    }
    tc_fence_before();
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

template <int BN, bool HALF, int EPI, int RB>
static int launch_epi(const TmaArgs& a_in, int num_sms, cudaStream_t st, int32_t* route) {
  using C = Cfg<BN, RB>;
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    CNB_CUDA(cudaFuncSetAttribute(conv_tma_kernel<BN, HALF, EPI, RB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  SMEM_BUDGET));
  }
  TmaArgs a = a_in;
  const int ntiles = a.tiles_m * a.tiles_n;
  const int nkb = a.ntaps * a.kchunks + a.kchunks2;
  const int b_res_bytes = (nkb * C::B_STAGE_BYTES + 1023) / 1024 * 1024;   // ring starts on a 1 KB boundary
  // smem plan for a given per-CTA budget; returns the ring depth (0: does not fit)
  auto plan = [&](int budget, int ctas, TmaArgs& o) -> int {
    const int room = budget - 1024 - C::EPI_BYTES - C::BAR_BYTES - b_res_bytes;
    int s_res = room > 0 ? room / C::A_STAGE_BYTES : 0;
    if (s_res > C::S) s_res = C::S;
    if (o.halo) {
      int s_h = room > 0 ? room / o.halo_stage_bytes : 0;
      if (s_h > C::S) s_h = C::S;
      o.bres = 1;
      o.s_run = s_h;
      o.ring_off = b_res_bytes;
      o.stage_bytes = o.halo_stage_bytes;
      o.epi_off = o.ring_off + s_h * o.halo_stage_bytes;
      return s_h;
    }
    // Resident weights pay off when a CTA runs several tiles against the same [nkb][BN x RB] weight block and that block
    // leaves room for a >= 4-deep A ring: L2 -> smem traffic per tile drops from A + B to A.
    if (o.tiles_n == 1 && ntiles >= 3 * ctas && s_res >= 4) {
      o.bres = 1;
      o.s_run = s_res;
      o.ring_off = b_res_bytes;
      o.stage_bytes = C::A_STAGE_BYTES;
      o.epi_off = o.ring_off + s_res * C::A_STAGE_BYTES;
      return s_res;
    }
    int s_ring = (budget - 1024 - C::EPI_BYTES - C::BAR_BYTES) / C::STAGE_BYTES;
    if (s_ring > C::S) s_ring = C::S;
    o.bres = 0;
    o.s_run = s_ring;
    o.ring_off = 0;
    o.stage_bytes = C::STAGE_BYTES;
    o.epi_off = s_ring * C::STAGE_BYTES;
    return s_ring;
  };
  // Two CTAs per SM (half the shared memory each, TMEM 2 x <= 256 columns): two independent load -> MMA -> epilogue
  // pipelines share an SM, which hides the per-tile latency chains of the short-K layers and lets the next kernel's
  // prologue overlap this kernel's tail.  Needs BN <= 128 (TMEM), a specialised epilogue (<= 102 registers) and a ring
  // of depth >= 2 in 112 KB.
  int grid = ntiles < num_sms ? ntiles : num_sms;
  bool two = false;
  if (BN <= 128 && EPI != 3 && ntiles >= 2 * num_sms) {
    TmaArgs t = a_in;
    if (plan(112 * 1024, 2 * num_sms, t) >= 2) {
      a = t;
      two = true;
      grid = ntiles < 2 * num_sms ? ntiles : 2 * num_sms;
    }
  }
  if (!two) {
    const int depth = plan(SMEM_BUDGET, grid, a);
    if (depth < 2) {
      set_error("conv_tma: smem plan does not fit shared memory (host-side check out of sync)");
      return CNB_ERR_UNSUPPORTED;
    }
  }
  size_t smem_bytes;
  a.bar_off = a.epi_off + C::EPI_BYTES;
  if (EPI == 6) {
    // a third staging buffer per epilogue warp where shared memory is left over: the residual box of slab i+1 can then
    // be requested while the store of slab i-1 is still reading its buffer
    const int budget = two ? 112 * 1024 : SMEM_BUDGET;
    const int e6_3 = EPI_WARPS * C::e6_warp_bytes(3);
    const bool fits3 = a.epi_off + e6_3 + C::BAR_BYTES + 1024 <= budget;
    a.epi_nbuf = fits3 ? 3 : 2;
    if (a.epi_nbuf == 3 && e6_3 > C::EPI_BYTES) a.bar_off = a.epi_off + e6_3;
  }
  {
    // alternate-tile epilogue when a tile's tensor work (~BN * K / 32 cycles) is shorter than its epilogue
    const long long ktot = (long long)nkb * (RB / (HALF ? 2 : 4));   // nkb counts every (tap, chunk) block
    // measured (B = 1024): halo 3x3 16->16 @28 54 -> 44 us, 64->64 @28 97 -> 91, 32->64 @28 89 -> 83; dense 1x1 layers
    // with several column slabs lose (256->768 @7 40 -> 44 us), so only the halo layers switch
    a.epi_alt = (a.halo && (long long)BN * ktot < 131072) ? 1 : 0;
    if (EPI == 6) a.epi_alt = 0;
  }
  smem_bytes = (size_t)a.bar_off + C::BAR_BYTES + 1024;
  if (route) {        // cnb_conv2d_route: everything above is the launch's own decision
    route[CNB_ROUTE_EPI] = EPI;
    route[CNB_ROUTE_BRES] = a.bres;
    route[CNB_ROUTE_CTAS_PER_SM] = two ? 2 : 1;
    route[CNB_ROUTE_EPI_ALT] = a.epi_alt;
    route[CNB_ROUTE_EPI_NBUF] = EPI == 6 ? a.epi_nbuf : 0;
    route[CNB_ROUTE_GRID] = grid;
    route[CNB_ROUTE_NTILES] = ntiles;
    return CNB_OK;
  }
  CNB_CUDA(launch_pdl((long long)ntiles * 128 * BN, conv_tma_kernel<BN, HALF, EPI, RB>, dim3(grid), dim3(NUM_THREADS), smem_bytes, st, a));
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

template <int BN, bool HALF, int RB>
static int launch(const TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route) {
  const bool dense = !a.halo && a.oy_mul == 1 && a.ox_mul == 1 && a.oy_add == 0 && a.ox_add == 0 &&
                     a.OHf * a.OWf == a.OHW;
  const bool simple = dense && a.act == 0 && !(a.temb && a.temb_per_sample);
  if (a.halo && a.act == 0 && !(a.temb && a.temb_per_sample) && a.out_f16 && (!a.residual || a.res_f16))
    return launch_epi<BN, HALF, 5, RB>(a, num_sms, st, route);
  if (simple && !a.out_f16 && !a.residual) return launch_epi<BN, HALF, 0, RB>(a, num_sms, st, route);
  if (simple && !a.out_f16 && a.residual && !a.res_f16) return launch_epi<BN, HALF, 1, RB>(a, num_sms, st, route);
  if constexpr (HALF) {
    if (simple && a.out_f16 && a.tma_epi && (!a.residual || a.res_f16)) return launch_epi<BN, HALF, 6, RB>(a, num_sms, st, route);
  }
  if (simple && a.out_f16 && !a.residual) return launch_epi<BN, HALF, 2, RB>(a, num_sms, st, route);
  if (simple && a.out_f16 && a.residual && a.res_f16) return launch_epi<BN, HALF, 4, RB>(a, num_sms, st, route);
  return launch_epi<BN, HALF, 3, RB>(a, num_sms, st, route);
}

template <bool HALF, int RB>
static int dispatch_bn(int bn, const TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route) {
  switch (bn) {
    case 256: return launch<256, HALF, RB>(a, num_sms, st, route);
    case 192: return launch<192, HALF, RB>(a, num_sms, st, route);
    case 128: return launch<128, HALF, RB>(a, num_sms, st, route);
    case 96: return launch<96, HALF, RB>(a, num_sms, st, route);
    case 64: return launch<64, HALF, RB>(a, num_sms, st, route);
    case 48: return launch<48, HALF, RB>(a, num_sms, st, route);
    case 32: return launch<32, HALF, RB>(a, num_sms, st, route);
    case 16: return launch<16, HALF, RB>(a, num_sms, st, route);
  }
  set_error("conv_tma: no tile for Cout");
  return CNB_ERR_UNSUPPORTED;
}

template <bool HALF>
static int dispatch_rb(int rb, int bn, const TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route) {
  switch (rb) {
    case 128: return dispatch_bn<HALF, 128>(bn, a, num_sms, st, route);
    case 64: return dispatch_bn<HALF, 64>(bn, a, num_sms, st, route);
    case 32: return dispatch_bn<HALF, 32>(bn, a, num_sms, st, route);
  }
  set_error("conv_tma: row bytes %d", rb);
  return CNB_ERR_UNSUPPORTED;
}

}  // namespace tma
}  // namespace cnb
