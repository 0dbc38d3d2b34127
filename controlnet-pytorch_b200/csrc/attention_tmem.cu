// Flash attention on the 5th-generation tensor core with S, P AND O resident in tensor memory
// (fp16 q|k|v [B, L, 3E] -> fp16 out [B, L, E]; replaces the core of nn.MultiheadAttention, unet_base.py:107).
//
// Why this shape of kernel.  At the head dims of this model (4 .. 64) a score costs 4 d tensor FLOPs but one exponential,
// so the roofline is the MUFU pipe (16 ex2 / clk / SM), not the tensor pipe.  Measured on the way here (ncu captures
// under profiles/r02_attn_*): ONE softmax warp per SM sub-partition and CTA cannot keep that pipe busy - an in-order
// warp alternates between its MUFU burst and everything else (scale, row maximum, pack, TMEM traffic, barrier round),
// and with two such warps per sub-partition the pipe sat at 45 - 52 %.  The kernel therefore runs FOUR softmax warps per
// sub-partition with the registers and tensor memory of two CTAs per SM:
//
//   CTA = (sample b, head h, TWO 128-row query tiles A and B sharing every K / V tile)            2 CTAs per SM, 12 warps:
//     warp 0      TMA producer: both Q tiles once, K tiles (3-stage ring), raw V tiles (2 stages)       (one thread)
//     warp 1      MMA issuer: O_g += P_g [V_j | 1] with P_g read straight from tensor memory ("TS" MMA), then
//                 S_g = Q_g K_{j+1}^T into the same columns, for g = A, B                               (one thread)
//     warp 2      V transposer: [BK keys][DL] (TMA, no swizzle) -> V^T atoms [NV rows][64 keys], K-major SWIZZLE_128B;
//                 row D of V^T is all ones, so column D of O is the softmax denominator, accumulated by the tensor core
//     warp 3      idle
//     warps 4-7   softmax of tile A, warps 8-11 softmax of tile B; thread = one query row = one TMEM lane
//   A softmax thread reads its row of S_g with tcgen05.ld (no ldmatrix, no HMMA, no shuffles: the row maximum is
//   thread-local), writes P_g back as packed fp16 pairs OVER the S columns it came from (tcgen05.st), and arrives on
//   p_full[g]; the O issuer consumes P_g from there - no shared-memory round trip, no proxy fence.  S_g is single
//   buffered: while tile A waits for  PV_A(j) -> Q_A K_{j+1}^T  (MMA issue ~250 cycles each, 300 - 450 until a commit is
//   visible, ~150 to wake a parked waiter: ~2000 cycles) the MUFU pipe belongs to tile B and to the other CTA - the
//   two-tile ping-pong of FlashAttention-4, with the exchange driven by mbarriers only.
//   Lazy rescale: a row's reference maximum only moves when a 32-score chunk exceeds it by more than 2^8 (P <= 256 is
//   harmless in fp16, sums are fp32); only then the warp scales its 32 rows of O_g and the part of P_g it already wrote,
//   in TMEM (PV_g(j-1) is complete whenever S_g(j) exists, so no extra wait).  After the first tile this is rare.
//   Head dims that are not a TMA / UMMA granule: DL >= D channels are loaded (D = 4 / 8: the aligned group of 16 that
//   contains the head; D = 24 / 48: 32 / 64 channels from the head's first) and the softmax threads zero the foreign
//   channels of their Q row in shared memory before the first MMA, so Q_masked K^T = Q_h K_h^T exactly.
//   TMEM (256 columns per CTA): S_A [0, BK) | S_B [BK, 2 BK) | O_A, O_B (NV = round16(D + 1) columns each).
//   Every mbarrier wait is bounded (tc_common.cuh) and latches the device error flag instead of hanging.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include "tc_common.cuh"

namespace cnb {
namespace atm {

using namespace tc;

constexpr int BQ = 128;            // query rows per tile (UMMA M); a CTA owns two tiles
constexpr int NUM_THREADS = 384;
constexpr int KS = 3;              // K ring stages
constexpr float LAZY = 8.0f;       // log2 headroom before a row's reference maximum moves

struct alignas(64) Args {
  CUtensorMap map_q;               // [B*L, 3E] fp16, box {DL, 128}, swizzle = row bytes
  CUtensorMap map_k;               // box {DL, BK}, swizzle = row bytes
  CUtensorMap map_v;               // box {DL, BK}, no swizzle (read by the transposer warp)
  __half* out;
  int L, E;
  float scale_log2;
  int safe;                        // 1: wait for PV_g(j)'s commit before Q_g K_{j+1}^T overwrites its P (cross-check)
};

template <int DL, int D, int BK>
struct Cfg {
  static_assert(DL == 16 || DL == 32 || DL == 64, "loaded channels per row = one swizzle span");
  static_assert(D <= DL && BK % 16 == 0 && BK >= 32 && BK <= 112, "tile");
  static constexpr int RB = DL * 2;                          // bytes per Q / K / raw-V row
  static constexpr int NV = (D + 1 + 15) / 16 * 16;          // PV MMA N: D value columns, the ones column, zero pad
  static constexpr int NA = (BK + 63) / 64;                  // 64-key V^T atoms per tile
  static constexpr int Q_TILE = BQ * RB;
  static constexpr int K_TILE = BK * RB;
  static constexpr int VT_ATOM = NV * 128;
  static constexpr int VT_TILE = NA * VT_ATOM;
  static constexpr int OFF_Q = 0;                            // two Q tiles
  static constexpr int OFF_K = (OFF_Q + 2 * Q_TILE + 1023) / 1024 * 1024;
  static constexpr int OFF_VR = (OFF_K + KS * K_TILE + 1023) / 1024 * 1024;
  static constexpr int OFF_VT = (OFF_VR + 2 * K_TILE + 1023) / 1024 * 1024;
  static constexpr int OFF_BAR = OFF_VT + 2 * VT_TILE;
  static constexpr int TOTAL = OFF_BAR + 256 + 1024;         // + alignment slack
  static constexpr int TMEM_COLS = 256;
  static constexpr int O_COL = 2 * BK;                       // O_g at O_COL + g * NV
  static_assert(O_COL + 2 * NV <= TMEM_COLS, "TMEM budget: S_A, S_B, O_A, O_B in 256 columns");
  static constexpr bool MASK_Q = D != DL;
};

// ---- PTX wrappers local to this kernel ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]   (A = P, packed fp16 pairs, lane = row)
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float y;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(y) : "f"(a), "f"(b), "f"(c));
  return y;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// One chunk of W (16 or 32) scores of this thread's row: raw scores r[] -> packed P (W / 2 registers).
//   c = scale * log2 e, mc = m * c.  `vk` = number of valid keys in the chunk (MASK only).
template <int W, bool MASK>
__device__ __forceinline__ void exp_pack(const uint32_t* r, float c, float mc, int vk, uint32_t* pk) {
#pragma unroll
  for (int i = 0; i < W; i += 2) {
    float x0 = fmaf(__uint_as_float(r[i]), c, -mc), x1 = fmaf(__uint_as_float(r[i + 1]), c, -mc);
    float e0 = ex2f(x0);
    float e1 = ex2f(x1);
    if (MASK) {
      if (i >= vk) e0 = 0.f;
      if (i + 1 >= vk) e1 = 0.f;
    }
    pk[i >> 1] = pack2(e0, e1);
  }
}

template <int W, bool MASK>
__device__ __forceinline__ float chunk_max(const uint32_t* r, int vk) {
  if (!MASK) {
    float t0 = fmax3(__uint_as_float(r[0]), __uint_as_float(r[1]), __uint_as_float(r[2]));
    float t1 = fmax3(__uint_as_float(r[3]), __uint_as_float(r[4]), __uint_as_float(r[5]));
#pragma unroll
    for (int i = 6; i + 3 < W; i += 4) {
      t0 = fmax3(t0, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
      t1 = fmax3(t1, __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
    }
    // W = 16: indices 6..13 consumed by the loop (i = 6, 10), 14, 15 left; W = 32: i = 6 .. 26, then 30, 31 left
    return fmax3(t0, t1, fmaxf(__uint_as_float(r[W - 2]), __uint_as_float(r[W - 1])));
  }
  float t = -INFINITY;
#pragma unroll
  for (int i = 0; i < W; ++i)
    if (i < vk) t = fmaxf(t, __uint_as_float(r[i]));
  return t;
}

// Rare path: a chunk exceeded the row's reference maximum by more than the headroom.  Moves the reference of the lanes
// that need it, scales this warp's rows of O (first == false: the PV MMA of the previous tile is complete, because the S
// tile being processed was only issued after it) and the `nwritten` 16-column P granules of the current tile that were
// written against the old reference.  Warp-uniform control flow (tcgen05.ld / st are .sync.aligned).
template <int NV>
__device__ __forceinline__ void rescale_rows(float& m, float tm, float lazy, float c, bool first, uint32_t t_o, uint32_t t_s,
                                             int nwritten, uint64_t* o_bar, uint32_t o_par, volatile int* abort_flag) {
  const float m_new = tm > m + lazy ? tm : m;
  const float f = ex2f((m - m_new) * c);                    // 1 for the lanes that keep their reference
  m = m_new;
  if (!first) {
    if (o_bar != nullptr) {                                 // geometry B2: PV of the previous tile may still be in flight
      mbar_wait_parked(o_bar, o_par, abort_flag);
      tc_fence_after();
    }
#pragma unroll
    for (int cb = 0; cb < NV; cb += 16) {
      uint32_t o[16];
      tmem_ld16_nowait(t_o + cb, o);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * f);
      tmem_st16(t_o + cb, o);
    }
  }
  const __half2 f2 = __float2half2_rn(f);
  for (int pc = 0; pc < nwritten; ++pc) {
    uint32_t o[16];
    tmem_ld16_nowait(t_s + (uint32_t)(pc * 16), o);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      __half2 hv = *reinterpret_cast<__half2*>(&o[i]);
      hv = __hmul2(hv, f2);
      o[i] = *reinterpret_cast<uint32_t*>(&hv);
    }
    tmem_st16(t_s + (uint32_t)(pc * 16), o);
  }
  tmem_st_wait();
}

// Softmax of one S tile for this thread's row.  LAST = false: every key valid, no masks (the steady state); LAST = true:
// `vk_tile` valid keys, whole chunks beyond them are skipped (the PV MMA skips the same 16-key blocks).
template <int BK, int NV, bool LAST>
__device__ __forceinline__ void softmax_tile(float& m, bool first_tile, int vk_tile, float c, float lazy, uint32_t t_s,
                                             uint32_t t_o, uint64_t* o_bar = nullptr, uint32_t o_par = 0,
                                             volatile int* abort_flag = nullptr) {
  constexpr int NCH = (BK + 31) / 32;
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
    const int col = ch * 32;
    const bool w16 = (BK - col) < 32;                        // tail chunk of 16 columns (BK = 112, 80, 48): compile time
    if (LAST && col >= vk_tile) break;
    uint32_t r[32];
    if (w16) tmem_ld16_nowait(t_s + (uint32_t)col, r);
    else tmem_ld32(t_s + (uint32_t)col, r);
    tmem_ld_wait();
    const int vk = LAST ? vk_tile - col : 32;                // valid scores of this chunk (>= 1)
    const bool full = !LAST || (w16 ? vk >= 16 : vk >= 32);
    float tm;
    if (full) tm = w16 ? chunk_max<16, false>(r, 16) : chunk_max<32, false>(r, 32);
    else tm = w16 ? chunk_max<16, true>(r, vk) : chunk_max<32, true>(r, vk);
    if (first_tile && ch == 0) {
      m = tm;
    } else if (__any_sync(0xffffffffu, tm > m + lazy)) {
      rescale_rows<NV>(m, tm, lazy, c, first_tile, t_o, t_s, ch, o_bar, o_par, abort_flag);
    }
    const float mc = m * c;
    uint32_t pk[16];
    if (w16) {
      if (full) exp_pack<16, false>(r, c, mc, 16, pk);
      else exp_pack<16, true>(r, c, mc, vk, pk);
      tmem_st8(t_s + (uint32_t)(ch * 16), pk);
    } else {
      if (full) exp_pack<32, false>(r, c, mc, 32, pk);
      else exp_pack<32, true>(r, c, mc, vk, pk);
      tmem_st16(t_s + (uint32_t)(ch * 16), pk);
    }
  }
}

template <int DL, int D, int BK>
__global__ void __launch_bounds__(NUM_THREADS, 2)
attention_tmem_kernel(const __grid_constant__ Args a) {
  using C = Cfg<DL, D, BK>;
  constexpr int RB = C::RB, NV = C::NV;
  constexpr uint32_t IDESC_S = make_idesc(BQ, BK, true);
  constexpr uint32_t IDESC_PV = make_idesc(BQ, NV, true);

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  const uint32_t sbase = raw_addr + pad;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
  uint64_t* q_full = bars + 0;              // both Q tiles landed
  uint64_t* q_ready = bars + 1;             // Q rows masked by the softmax warps (MASK_Q only)
  uint64_t* k_full = bars + 2;              // [KS]
  uint64_t* k_empty = k_full + KS;          // [KS]
  uint64_t* v_full = k_empty + KS;          // [2] raw V landed (TMA)
  uint64_t* v_empty = v_full + 2;           // [2] raw V consumed by the transposer
  uint64_t* vt_full = v_empty + 2;          // [2] V^T written
  uint64_t* s_full = vt_full + 2;           // [2: tile A / B] S_g written by the MMA
  uint64_t* p_full = s_full + 2;            // [2] P_g written over S_g by the active softmax warps of tile g
  uint64_t* s_free = p_full + 2;            // [2] PV_g finished: S_g may be overwritten, O_g is up to date
  uint64_t* pv_done = s_free + 2;           // [2: V^T stage] both PV MMAs of the tile finished: V^T stage free
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 2);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(tmem_slot + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = a.L;
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = blockIdx.x * 2 * BQ;                       // first query row of tile A
  const int NT = (L + BK - 1) / BK;                         // key tiles
  const int row0 = b * L;                                   // first row of this sample in the [B*L, 3E] matrix
  // softmax warps with at least one real query row, per tile (tile B may be empty)
  const int nact0 = min(4, (L - q0 + 31) >> 5);
  const int nact1 = max(0, min(4, (L - q0 - BQ + 31) >> 5));
  // channel group of this head: xg = first loaded channel, c0 = offset of the head inside the loaded group
  const int xg = (DL % D == 0) ? (h * D / DL) * DL : h * D;
  const int c0 = h * D - xg;
  const int vlast = L - (NT - 1) * BK;                      // valid keys of the last tile (1 .. BK)

  if (tid == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_ready, (uint32_t)(nact0 + nact1));
    for (int i = 0; i < KS; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&vt_full[i], 1);
      mbar_init(&pv_done[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], (uint32_t)max(1, i == 0 ? nact0 : nact1));
      mbar_init(&s_free[i], 1);
    }
    *abort_flag = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  // rows D .. NV-1 of every V^T atom are constant: the ones row, then zeros (uniform rows: swizzle-free)
  if (warp == 2) {
    constexpr int ROWS = NV - D;
    for (int i = lane; i < 2 * C::NA * ROWS * 8; i += 32) {   // (atom of either stage, row, 16-byte chunk)
      const int chunk = i & 7, row = (i >> 3) % ROWS, atom = (i >> 3) / ROWS;
      const uint32_t v = row == 0 ? 0x3C003C00u : 0u;          // half2(1, 1)
      *reinterpret_cast<uint4*>(smem + C::OFF_VT + atom * C::VT_ATOM + (D + row) * 128 + chunk * 16) = make_uint4(v, v, v, v);
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                               // every global access of this kernel comes after this point
  pdl_trigger();

  if (warp == 0) {
    // ======================= TMA producer (one thread) =======================
    if (lane == 0) {
      mbar_expect_tx(q_full, (uint32_t)(2 * C::Q_TILE));
      tma_load_2d(sbase + C::OFF_Q, &a.map_q, q_full, xg, row0 + q0);
      tma_load_2d(sbase + C::OFF_Q + C::Q_TILE, &a.map_q, q_full, xg, row0 + q0 + BQ);
      const int xk = a.E + xg, xv = 2 * a.E + xg;
      int st = 0;
      uint32_t ph = 1;                                       // parity of the k_empty phase that frees stage st (first lap: free)
      for (int j = 0; j < NT; ++j) {
        if (j >= KS && !mbar_wait_parked(&k_empty[st], ph, abort_flag)) break;
        mbar_expect_tx(&k_full[st], (uint32_t)C::K_TILE);
        tma_load_2d(sbase + C::OFF_K + st * C::K_TILE, &a.map_k, &k_full[st], xk, row0 + j * BK);
        if (++st == KS) { st = 0; ph ^= 1; }
        const int vs = j & 1;
        if (j >= 2 && !mbar_wait_parked(&v_empty[vs], (uint32_t)(((j >> 1) - 1) & 1), abort_flag)) break;
        mbar_expect_tx(&v_full[vs], (uint32_t)C::K_TILE);
        tma_load_2d(sbase + C::OFF_VR + vs * C::K_TILE, &a.map_v, &v_full[vs], xv, row0 + j * BK);
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer (one thread): S_g = Q_g K_j^T and O_g += P_g [V_j | 1] =======================
    // One thread issues, per tile g and key tile j, PV_g(j) immediately followed by Q_g K_{j+1}^T, which overwrites the
    // P_g(j) that PV_g(j) reads.  The tensor pipe executes the MMAs of one thread in issue order, so the pair needs no
    // barrier in between (a.safe = 1 waits for PV's commit first: the debugging cross-check of that ordering); the commit
    // after the second MMA tells the softmax warps that S_g(j+1) is there AND that O_g holds every tile up to j.
    if (lane == 0 && mbar_wait_parked(C::MASK_Q ? q_ready : q_full, 0u, abort_flag)) {
      tc_fence_after();
      const uint64_t qdesc0 = make_desc_kmajor<RB>(sbase + C::OFF_Q);
      const uint64_t kdesc0 = make_desc_kmajor<RB>(sbase + C::OFF_K);
      const uint64_t vdesc0 = make_desc_kmajor<128>(sbase + C::OFF_VT);
      auto issue_qk = [&](int g, int j) {                    // S_g = Q_g K_j^T (K tile j sits in ring stage j % KS)
        const uint64_t kdesc = kdesc0 + (uint64_t)(((j % KS) * C::K_TILE) >> 4);
        const uint64_t qdesc = qdesc0 + (uint64_t)((g * C::Q_TILE) >> 4);
#pragma unroll
        for (int k = 0; k < DL / 16; ++k)
          umma<true>(tmem_base + (uint32_t)(g * BK), qdesc + (uint64_t)(2 * k), kdesc + (uint64_t)(2 * k), IDESC_S, k ? 1u : 0u);
        umma_commit(&s_full[g]);
      };
      auto issue_pv = [&](int g, int j) {                    // O_g += P_g [V_j | 1] (V^T of tile j sits in stage j & 1)
        const int nkb = j + 1 < NT ? BK / 16 : (vlast + 15) >> 4;      // 16-key blocks with at least one valid key
        const uint64_t vdesc_t = vdesc0 + (uint64_t)(((j & 1) * C::VT_TILE) >> 4);
        const uint32_t p_col = tmem_base + (uint32_t)(g * BK);
        const uint32_t o_col = tmem_base + (uint32_t)(C::O_COL + g * NV);
#pragma unroll
        for (int kb = 0; kb < BK / 16; ++kb) {
          if (kb < nkb)
            umma_ts(o_col, p_col + (uint32_t)(kb * 8),
                    vdesc_t + (uint64_t)(((kb >> 2) * C::VT_ATOM + (kb & 3) * 32) >> 4), IDESC_PV, (j | kb) ? 1u : 0u);
        }
      };
      // (Running tile B one key tile behind tile A, so that one tile exponentiates while the other waits for its MMAs,
      // was measured and is slower: L = 784, d = 16: 1147 vs 1093 us - gpu_jobs/r2_11.)
      bool ok = mbar_wait_parked(&k_full[0], 0u, abort_flag);
      const bool has_b = nact1 > 0;
      if (ok) {
        tc_fence_after();
        issue_qk(0, 0);
        if (has_b) issue_qk(1, 0);
        umma_commit(&k_empty[0]);
      }
      for (int j = 0; ok && j < NT; ++j) {
        const int st = j & 1;
        if (!mbar_wait_parked(&vt_full[st], (uint32_t)((j >> 1) & 1), abort_flag)) break;
        const bool more = j + 1 < NT;
        if (more && !mbar_wait_parked(&k_full[(j + 1) % KS], (uint32_t)(((j + 1) / KS) & 1), abort_flag)) break;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (g == 1 && !has_b) continue;                    // tile B is empty: the CTA runs tile A only
          if (!mbar_wait_parked(&p_full[g], (uint32_t)(j & 1), abort_flag)) { ok = false; break; }
          tc_fence_after();
          issue_pv(g, j);
          if (more) {
            if (a.safe) {
              umma_commit(&s_free[g]);
              if (!mbar_wait_parked(&s_free[g], (uint32_t)(j & 1), abort_flag)) { ok = false; break; }
              tc_fence_after();
            }
            issue_qk(g, j + 1);
          } else {
            umma_commit(&s_free[g]);                          // last tile: O_g is final (the softmax epilogue waits on this)
          }
        }
        umma_commit(&pv_done[st]);
        if (more) umma_commit(&k_empty[(j + 1) % KS]);
      }
    }
    __syncwarp();
    tc_fence_before();
  } else if (warp == 2) {
    // ======================= V transposer: lane = key pair of each 64-key atom =======================
    const int chunk = lane >> 2, within = (lane & 3) * 4;   // 16-byte chunk of the V^T row, byte offset inside it
    for (int j = 0; j < NT; ++j) {
      const int vs = j & 1, st = j & 1;
      if (!mbar_wait_parked(&v_full[vs], (uint32_t)((j >> 1) & 1), abort_flag)) break;
      if (j >= 2 && !mbar_wait_parked(&pv_done[st], (uint32_t)(((j >> 1) - 1) & 1), abort_flag)) break;
#pragma unroll
      for (int atom = 0; atom < C::NA; ++atom) {
        const int key = atom * 64 + 2 * lane;
        if (key < BK) {                                      // BK is even and a multiple of 16: key + 1 < BK too
          const uint8_t* src = smem + C::OFF_VR + vs * C::K_TILE + key * RB + c0 * 2;
          uint8_t* vt = smem + C::OFF_VT + st * C::VT_TILE + atom * C::VT_ATOM + within;
          if constexpr (D % 8 == 0) {
#pragma unroll
            for (int v = 0; v < D / 8; ++v) {
              const uint4 x0 = *reinterpret_cast<const uint4*>(src + v * 16);            // key
              const uint4 x1 = *reinterpret_cast<const uint4*>(src + RB + v * 16);       // key + 1
              const uint32_t w0[4] = {x0.x, x0.y, x0.z, x0.w}, w1[4] = {x1.x, x1.y, x1.z, x1.w};
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int dd = v * 8 + e;                      // V^T row
                const uint32_t val = (e & 1) ? __byte_perm(w0[e >> 1], w1[e >> 1], 0x7632) : __byte_perm(w0[e >> 1], w1[e >> 1], 0x5410);
                *reinterpret_cast<uint32_t*>(vt + dd * 128 + ((chunk ^ (dd & 7)) << 4)) = val;
              }
            }
          } else {                                             // D = 4: 8 bytes per key
            const uint2 x0 = *reinterpret_cast<const uint2*>(src);
            const uint2 x1 = *reinterpret_cast<const uint2*>(src + RB);
            const uint32_t w0[2] = {x0.x, x0.y}, w1[2] = {x1.x, x1.y};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const uint32_t val = (e & 1) ? __byte_perm(w0[e >> 1], w1[e >> 1], 0x7632) : __byte_perm(w0[e >> 1], w1[e >> 1], 0x5410);
              *reinterpret_cast<uint32_t*>(vt + e * 128 + ((chunk ^ (e & 7)) << 4)) = val;
            }
          }
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&vt_full[st]);
        mbar_arrive(&v_empty[vs]);
      }
    }
  } else if (warp >= 4 && ((warp - 4) & 3) < (((warp - 4) >> 2) == 0 ? nact0 : nact1)) {
    // ======================= softmax: thread = query row of tile g =======================
    const int g = (warp - 4) >> 2, q = (warp - 4) & 3;
    const int row = q * 32 + lane;                          // TMEM lane = row of the tile
    const int grow = q0 + g * BQ + row;                     // row of the sequence
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t t_s = t_lane + (uint32_t)(g * BK);
    const uint32_t t_o = t_lane + (uint32_t)(C::O_COL + g * NV);
    const float c = a.scale_log2;
    const float lazy = LAZY / c;                            // headroom in raw score units
    bool dead = false;

    if constexpr (C::MASK_Q) {
      // zero the channels of this Q row that belong to other heads: Q_masked K^T = Q_h K_h^T
      if (mbar_wait_parked(q_full, 0u, abort_flag)) {
        constexpr int NC = RB / 16;                          // 16-byte chunks per row
        const int sw = (row >> (RB == 32 ? 2 : (RB == 64 ? 1 : 0))) & (NC - 1);
        uint8_t* qrow = smem + C::OFF_Q + g * C::Q_TILE + row * RB;
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          uint4* ptr = reinterpret_cast<uint4*>(qrow + ((j ^ sw) << 4));
          uint4 v = *ptr;
          uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int ch = j * 8 + 2 * e;                    // channels ch, ch + 1 (c0 and D are even)
            if (ch < c0 || ch >= c0 + D) w[e] = 0u;
          }
          *ptr = make_uint4(w[0], w[1], w[2], w[3]);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(q_ready);
      } else {
        dead = true;
      }
    }

    float m = 0.f;                                          // reference maximum (raw score units), set by the first chunk
    for (int j = 0; !dead && j < NT; ++j) {
      if (!mbar_wait_parked(&s_full[g], (uint32_t)(j & 1), abort_flag)) { dead = true; break; }
      tc_fence_after();
      if (j < NT - 1) softmax_tile<BK, NV, false>(m, j == 0, BK, c, lazy, t_s, t_o);
      else softmax_tile<BK, NV, true>(m, j == 0, vlast, c, lazy, t_s, t_o);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[g]);
    }

    // ---- epilogue: out = O[:, :D] / O[:, D]
    if (!dead && mbar_wait_parked(&s_free[g], a.safe ? (uint32_t)((NT - 1) & 1) : 0u, abort_flag)) {
      tc_fence_after();
      uint32_t od[16];
      tmem_ld16_nowait(t_o + (D / 16) * 16, od);             // the 16-column block that holds column D = sum of P
      tmem_ld_wait();
      const float inv = 1.0f / __uint_as_float(od[D % 16]);
      __half* op = a.out + ((size_t)(row0 + grow) * a.E + h * D);
#pragma unroll
      for (int cb = 0; cb < D; cb += 16) {
        uint32_t o[16];
        tmem_ld16_nowait(t_o + cb, o);
        tmem_ld_wait();
        if (grow < L) {
          if constexpr (D % 8 == 0) {
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              if (cb + 8 * v < D) {
                uint4 w;
                w.x = pack2(__uint_as_float(o[8 * v + 0]) * inv, __uint_as_float(o[8 * v + 1]) * inv);
                w.y = pack2(__uint_as_float(o[8 * v + 2]) * inv, __uint_as_float(o[8 * v + 3]) * inv);
                w.z = pack2(__uint_as_float(o[8 * v + 4]) * inv, __uint_as_float(o[8 * v + 5]) * inv);
                w.w = pack2(__uint_as_float(o[8 * v + 6]) * inv, __uint_as_float(o[8 * v + 7]) * inv);
                *reinterpret_cast<uint4*>(op + cb + 8 * v) = w;
              }
            }
          } else {
            uint2 w;
            w.x = pack2(__uint_as_float(o[0]) * inv, __uint_as_float(o[1]) * inv);
            w.y = pack2(__uint_as_float(o[2]) * inv, __uint_as_float(o[3]) * inv);
            *reinterpret_cast<uint2*>(op) = w;
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

template <int DL, int D, int BK>
static int launch(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  using C = Cfg<DL, D, BK>;
  if (!g_encode) {
    cudaDriverEntryPointQueryResult q;
    void* f = nullptr;
    CNB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
    if (!f || q != cudaDriverEntryPointSuccess) {
      set_error("attention_tmem: cuTensorMapEncodeTiled unavailable");
      return CNB_ERR_UNSUPPORTED;
    }
    g_encode = reinterpret_cast<EncodeTiledFn>(f);
  }
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    CNB_CUDA(cudaFuncSetAttribute(attention_tmem_kernel<DL, D, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::TOTAL));
  }
  Args a;
  memset(&a, 0, sizeof(a));
  const cuuint64_t dims[2] = {(cuuint64_t)3 * E, (cuuint64_t)B * L};
  const cuuint64_t strides[1] = {(cuuint64_t)3 * E * 2};
  const cuuint32_t box_q[2] = {(cuuint32_t)DL, (cuuint32_t)BQ};
  const cuuint32_t box_k[2] = {(cuuint32_t)DL, (cuuint32_t)BK};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle swz = DL == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : (DL == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B);
  CUresult r = g_encode(&a.map_q, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(qkv), dims, strides, box_q, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS)
    r = g_encode(&a.map_k, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(qkv), dims, strides, box_k, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS)
    r = g_encode(&a.map_v, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(qkv), dims, strides, box_k, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("attention_tmem: cuTensorMapEncodeTiled failed (%d): B=%d L=%d E=%d", (int)r, B, L, E);
    return CNB_ERR_CUDA;
  }
  a.out = reinterpret_cast<__half*>(out);
  a.L = L;
  a.E = E;
  a.scale_log2 = 1.4426950408889634f / sqrtf((float)D);
  static int safe = -1;
  if (safe < 0) {
    const char* e = getenv("CNB_ATTN_SAFE");
    safe = e ? atoi(e) : 0;
  }
  a.safe = safe;
  dim3 grid(ceil_div(L, 2 * BQ), heads, B);
  CNB_CUDA(launch_pdl((long long)B * L * E, attention_tmem_kernel<DL, D, BK>, grid, dim3(NUM_THREADS),
                      (size_t)C::TOTAL, st, a));
  CNB_LAUNCH_CHECK();
  return CNB_OK;
}

// Key-tile size: S_A, S_B (BK columns each) and O_A, O_B (NV each) share the CTA's 256 TMEM columns, and two CTAs (Q
// tiles, K ring, raw V, V^T stages) share one SM's shared memory.  The largest tile that fits, shrunk when a smaller
// one pads the sequence less (784 = 7 x 112 = 8.2 x 96; 1024 = 10.7 x 96 = 12.8 x 80 = 16 x 64).
template <int DL, int D>
static int launch_bk(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  constexpr int NV = (D + 1 + 15) / 16 * 16;
  constexpr int BKMAX = DL == 64 ? 48 : ((256 - 2 * NV) / 2) / 16 * 16;   // 112 (NV 16), 96 (NV 32), 80 (NV 48); 48 for 64-channel rows
  auto padded = [&](int bk) { return ceil_div(L, bk) * bk; };
  int bk = BKMAX;
  const int cands[4] = {96, 80, 64, 48};                    // a smaller tile only if it saves more than 6 % of the padded keys
  for (int i = 0; i < 4; ++i)
    if (cands[i] < bk && padded(cands[i]) * 100 < padded(bk) * 94) bk = cands[i];
  if constexpr (BKMAX >= 112) if (bk >= 112) return launch<DL, D, 112>(qkv, out, B, L, E, heads, st);
  if constexpr (BKMAX >= 96) if (bk >= 96) return launch<DL, D, 96>(qkv, out, B, L, E, heads, st);
  if constexpr (BKMAX >= 80) if (bk >= 80) return launch<DL, D, 80>(qkv, out, B, L, E, heads, st);
  if constexpr (BKMAX >= 64) if (bk >= 64) return launch<DL, D, 64>(qkv, out, B, L, E, heads, st);
  return launch<DL, D, 48>(qkv, out, B, L, E, heads, st);
}

}  // namespace atm

int attention_tmem_error_flag() { return tc_read_clear_error(); }

// Default routing of cnb_attention_f16, from the measured table (profiles/r02_attention_table.md, B200, batch 1024 / 256):
// this kernel wins where the head dim is >= 24 and the sequence >= 128 tokens (CIFAR 32x32 d = 32: 1.54 vs 2.12 ms, 16x16
// d = 64: 0.19 vs 0.49 ms; CelebHQ-latent 32x32 d = 24: 1.50 vs 1.95 ms, 16x16 d = 32: 0.139 vs 0.167 ms; MNIST 14x14
// d = 32: 0.131 vs 0.135 ms); at head dims <= 16 the register-resident mma.sync kernel is still ahead (28x28 d = 16:
// 0.90 vs 1.09 ms) and sequences of <= 64 tokens are one tile of either kernel (latency only).
// runtime.attention_kernel_name mirrors this rule.
bool attention_tmem_default(int L, int d) { return L >= 128 && d >= 24; }

bool attention_tmem_supported(const void* qkv, const void* out, int B, int L, int E, int heads) {
  if (heads <= 0 || E % heads) return false;
  const int d = E / heads;
  if (d != 4 && d != 8 && d != 16 && d != 24 && d != 32 && d != 48 && d != 64) return false;
  if (L < 1 || B > 65535 || heads > 65535) return false;
  if ((3 * E * 2) % 16 || (((uintptr_t)qkv | (uintptr_t)out) & 15)) return false;
  return true;
}

int attention_tmem(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st) {
  switch (E / heads) {
    case 4: return atm::launch_bk<16, 4>(qkv, out, B, L, E, heads, st);
    case 8: return atm::launch_bk<16, 8>(qkv, out, B, L, E, heads, st);
    case 16: return atm::launch_bk<16, 16>(qkv, out, B, L, E, heads, st);
    case 24: return atm::launch_bk<32, 24>(qkv, out, B, L, E, heads, st);
    case 32: return atm::launch_bk<32, 32>(qkv, out, B, L, E, heads, st);
    case 48: return atm::launch_bk<64, 48>(qkv, out, B, L, E, heads, st);
    case 64: return atm::launch_bk<64, 64>(qkv, out, B, L, E, heads, st);
    default:
      set_error("attention_tmem: head dim %d not instantiated", E / heads);
      return CNB_ERR_UNSUPPORTED;
  }
}

}  // namespace cnb
