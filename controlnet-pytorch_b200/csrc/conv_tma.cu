// Host side of the TMA-fed tcgen05 convolution: tensor-map construction (im2col map for the activations, tiled map for
// the packed weights), tile / swizzle-span choice and launch.  The kernel lives in conv_tma_impl.cuh and is
// instantiated in conv_tma_f16.cu / conv_tma_tf32.cu.
#include "conv_tma_impl.cuh"

namespace cnb {
namespace tma {

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeIm2colFn g_encode_im2col = nullptr;
static EncodeTiledFn g_encode_tiled = nullptr;
static int g_num_sms = 0;
static int g_driver_version = 0;

static int resolve_driver() {
  if (g_encode_im2col && g_encode_tiled) return CNB_OK;
  cudaDriverEntryPointQueryResult q1, q2;
  void *f1 = nullptr, *f2 = nullptr;
  CNB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &f1, cudaEnableDefault, &q1));
  CNB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f2, cudaEnableDefault, &q2));
  if (!f1 || !f2 || q1 != cudaDriverEntryPointSuccess || q2 != cudaDriverEntryPointSuccess) {
    set_error("conv_tma: the driver does not export cuTensorMapEncodeIm2col / cuTensorMapEncodeTiled");
    return CNB_ERR_UNSUPPORTED;
  }
  int dev = 0;
  CNB_CUDA(cudaGetDevice(&dev));
  CNB_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  CNB_CUDA(cudaDriverGetVersion(&g_driver_version));
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(f1);
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(f2);
  return CNB_OK;
}

}  // namespace tma

int conv_tma_launch_f16(int rb, int bn, const tma::TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route);
int conv_tma_launch_tf32(int rb, int bn, const tma::TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route);
int conv_tma_error_flag_f16();
int conv_tma_error_flag_tf32();

int conv_tma_error_flag() {
  const int a = conv_tma_error_flag_f16(), b = conv_tma_error_flag_tf32();
  return (a < 0 || b < 0) ? -1 : (a | b);
}

static int pick_bn(int cout) {
  static const int cand[] = {256, 192, 128, 96, 64, 48, 32, 16};
  for (int bn : cand)
    if (cout % bn == 0) return bn;
  return 0;
}

// widest swizzle span whose channel chunk divides Cin; channel counts that are whole 16-byte units but not a multiple of
// the narrowest chunk (fp16: Cin % 16 == 8) take 32-byte chunks with a partial last one - TMA zero-fills the channels
// past Cin, so whatever weight columns the chunk covers there multiply zeros
static int pick_rb(int cin, int elt) {
  for (int rb = 128; rb >= 32; rb >>= 1)
    if (cin % (rb / elt) == 0) return rb;
  return (cin * elt) % 16 == 0 ? 32 : 0;
}

bool conv2d_tma_supported(const cnb_conv_params* p) {
  if (p->mode == CNB_MODE_F32) return false;
  const bool half = p->in_dtype == 1;
  const int elt = half ? 2 : 4;
  if (half && !p->weight_lp) return false;
  if (pick_rb(p->Cin, elt) == 0) return false;
  if (p->in2) {
    if (p->stride != 1 || p->H != p->OH || p->W != p->OW) return false;      // second input lives on the output grid
    if (p->Cin2 % (16 / elt)) return false;      // rows of the second input must be whole 16-byte chunks
    if ((p->ldi2 * elt) % 16 || (p->in2_coff * elt) % 16 || ((uintptr_t)p->in2 & 15)) return false;
  }
  if ((p->ldi * elt) % 16 || (p->in_coff * elt) % 16) return false;
  if (pick_bn(p->Cout) == 0) return false;
  const int oelt = p->out_dtype == 1 ? 2 : 4;
  if (p->ldo % 4 || p->out_coff % 4 || ((size_t)p->out_coff * oelt) % 8) return false;
  if (p->residual && (p->ldr % 4 || p->res_coff % 4)) return false;
  if (p->temb && (p->temb_ld % 4)) return false;
  if (((uintptr_t)p->in | (uintptr_t)p->weight | (uintptr_t)p->weight_lp | (uintptr_t)p->out | (uintptr_t)p->bias |
       (uintptr_t)p->temb | (uintptr_t)p->residual) & 15)
    return false;
  // tap window must be expressible as im2col offsets from a lower corner
  int dxmin = 127, dymin = 127, dxmax = -128, dymax = -128;
  for (int t = 0; t < p->ntaps; ++t) {
    dxmin = p->dx[t] < dxmin ? p->dx[t] : dxmin;
    dymin = p->dy[t] < dymin ? p->dy[t] : dymin;
    dxmax = p->dx[t] > dxmax ? p->dx[t] : dxmax;
    dymax = p->dy[t] > dymax ? p->dy[t] : dymax;
  }
  if (dxmax - dxmin > 255 || dymax - dymin > 255) return false;
  const int uw = dxmin + (p->OW - 1) * p->stride + 1 - p->W, uh = dymin + (p->OH - 1) * p->stride + 1 - p->H;
  if (uw < -128 || uw > 127 || uh < -128 || uh > 127 || p->stride < 1 || p->stride > 8) return false;
  return true;
}

// route != nullptr: fill in the route (cnb_conv2d_route) instead of launching
int conv2d_tma(const cnb_conv_params* p, cudaStream_t st, int32_t* route) {
  using namespace tma;
  int rc = resolve_driver();
  if (rc != CNB_OK) return rc;
  const bool half = p->in_dtype == 1;
  const int elt = half ? 2 : 4;
  // the second input reuses the main input's chunk width; a last partial chunk is zero-filled by TMA (channels and
  // weight columns past the end are out of bounds)
  const int rb = pick_rb(p->Cin, elt), kc = rb / elt;
  const CUtensorMapSwizzle swz = rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                           : (rb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  TmaArgs a;
  memset(&a, 0, sizeof(a));
  int dxmin = 127, dymin = 127;
  for (int t = 0; t < p->ntaps; ++t) {
    dxmin = p->dx[t] < dxmin ? p->dx[t] : dxmin;
    dymin = p->dy[t] < dymin ? p->dy[t] : dymin;
  }
  for (int t = 0; t < p->ntaps; ++t)
    a.tap_off[t] = (uint32_t)(p->dx[t] - dxmin) | ((uint32_t)(p->dy[t] - dymin) << 16);
  const int lower[2] = {dxmin, dymin};
  const int upper[2] = {dxmin + (p->OW - 1) * p->stride + 1 - p->W, dymin + (p->OH - 1) * p->stride + 1 - p->H};

  // ---- halo mode: 3x3 / stride 1 / pad 1 with resident weights; the input tile is loaded once per channel chunk
  const int bn_h = pick_bn(p->Cout);
  bool halo = false;
  int Wp = p->W + 2, R = 0, halo_stage = 0;
  {
    bool std3 = p->ntaps == 9 && p->stride == 1 && p->OH == p->H && p->OW == p->W && p->oy_mul == 1 && p->ox_mul == 1 &&
                p->oy_add == 0 && p->ox_add == 0 && p->OHf == p->OH && p->OWf == p->OW && p->Cout == bn_h;
    for (int t = 0; t < 9 && std3; ++t) std3 = p->dy[t] == t / 3 - 1 && p->dx[t] == t % 3 - 1;
    if (std3 && Wp <= 64 && p->W >= 12) {
      R = BM / Wp;
      const int tiles_y = ceil_div(p->H, R);
      const double useful = (double)p->H * p->W / ((double)tiles_y * BM);
      const int nkb_all = 9 * ceil_div(p->Cin, kc) + (p->in2 ? ceil_div(p->Cin2, kc) : 0);
      const int b_res = (nkb_all * bn_h * rb + 1023) / 1024 * 1024;
      halo_stage = ((BM + 2 * Wp + 2) * rb + 1023) / 1024 * 1024;
      const int room = SMEM_BUDGET - 1024 - 36864 - 512 - b_res;
      halo = useful >= 0.7 && room >= 3 * halo_stage && (long long)p->B * tiles_y >= 2 * g_num_sms;
    }
  }
  if (halo) {
    const cuuint64_t dims[4] = {(cuuint64_t)p->Cin, (cuuint64_t)p->W, (cuuint64_t)p->H, (cuuint64_t)p->B};
    const cuuint64_t strides[3] = {(cuuint64_t)p->ldi * elt, (cuuint64_t)p->W * p->ldi * elt,
                                   (cuuint64_t)p->H * p->W * p->ldi * elt};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const cuuint32_t box[4] = {(cuuint32_t)kc, (cuuint32_t)Wp, (cuuint32_t)(R + 2), 1};
    void* base = const_cast<char*>(reinterpret_cast<const char*>(p->in) + (size_t)p->in_coff * elt);
    CUresult r = g_encode_tiled(&a.map_a, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base,
                                dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled(halo input) failed (%d): Cin=%d W=%d H=%d B=%d box=(%d,%d,%d)", (int)r, p->Cin,
                p->W, p->H, p->B, kc, Wp, R + 2);
      return CNB_ERR_CUDA;
    }
    if (p->in2) {
      const cuuint64_t dims2[4] = {(cuuint64_t)p->Cin2, (cuuint64_t)p->W, (cuuint64_t)p->H, (cuuint64_t)p->B};
      const cuuint64_t strides2[3] = {(cuuint64_t)p->ldi2 * elt, (cuuint64_t)p->W * p->ldi2 * elt,
                                      (cuuint64_t)p->H * p->W * p->ldi2 * elt};
      const cuuint32_t box2[4] = {(cuuint32_t)kc, (cuuint32_t)Wp, (cuuint32_t)R, 1};
      void* base2 = const_cast<char*>(reinterpret_cast<const char*>(p->in2) + (size_t)p->in2_coff * elt);
      r = g_encode_tiled(&a.map_a2, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base2,
                         dims2, strides2, box2, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(halo second input) failed (%d)", (int)r);
        return CNB_ERR_CUDA;
      }
      a.kchunks2 = ceil_div(p->Cin2, kc);
    }
    a.halo = 1; a.Wp = Wp; a.R = R; a.tiles_y = ceil_div(p->H, R); a.H = p->H; a.W = p->W;
    a.halo_stage_bytes = halo_stage;
  }
  // ---- activations: [B, H, W, ldi] viewed as (C, W, H, N), im2col box = 128 pixels x kc channels
  if (!halo) {
    const cuuint64_t dims[4] = {(cuuint64_t)p->Cin, (cuuint64_t)p->W, (cuuint64_t)p->H, (cuuint64_t)p->B};
    const cuuint64_t strides[3] = {(cuuint64_t)p->ldi * elt, (cuuint64_t)p->W * p->ldi * elt,
                                   (cuuint64_t)p->H * p->W * p->ldi * elt};
    const cuuint32_t estr[4] = {1, (cuuint32_t)p->stride, (cuuint32_t)p->stride, 1};
    void* base = const_cast<char*>(reinterpret_cast<const char*>(p->in) + (size_t)p->in_coff * elt);
    CUresult r = g_encode_im2col(&a.map_a, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                                 base, dims, strides, lower, upper, (cuuint32_t)kc, (cuuint32_t)BM, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeIm2col failed (%d): Cin=%d W=%d H=%d B=%d ldi=%d stride=%d lower=(%d,%d) upper=(%d,%d)",
                (int)r, p->Cin, p->W, p->H, p->B, p->ldi, p->stride, lower[0], lower[1], upper[0], upper[1]);
      return CNB_ERR_CUDA;
    }
    // same small-tensor descriptor fix-up CUTLASS applies (cute/atom/copy_traits_sm90_im2col.hpp) on drivers <= 13.1
    const size_t bytes = (size_t)p->B * p->H * p->W * p->ldi * elt;
    if (g_driver_version <= 13010 && bytes < 131072) reinterpret_cast<uint64_t*>(&a.map_a)[1] &= ~(1llu << 21);
  }
  // ---- optional second input: [B, OH, OW, ldi2], a single (0,0) tap on the output grid
  if (p->in2 && !halo) {
    const int zero2[2] = {0, 0};
    const cuuint64_t dims[4] = {(cuuint64_t)p->Cin2, (cuuint64_t)p->OW, (cuuint64_t)p->OH, (cuuint64_t)p->B};
    const cuuint64_t strides[3] = {(cuuint64_t)p->ldi2 * elt, (cuuint64_t)p->OW * p->ldi2 * elt,
                                   (cuuint64_t)p->OH * p->OW * p->ldi2 * elt};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    void* base = const_cast<char*>(reinterpret_cast<const char*>(p->in2) + (size_t)p->in2_coff * elt);
    CUresult r = g_encode_im2col(&a.map_a2, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                                 base, dims, strides, zero2, zero2, (cuuint32_t)kc, (cuuint32_t)BM, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeIm2col(second input) failed (%d): Cin2=%d OW=%d OH=%d B=%d ldi2=%d", (int)r, p->Cin2,
                p->OW, p->OH, p->B, p->ldi2);
      return CNB_ERR_CUDA;
    }
    const size_t bytes2 = (size_t)p->B * p->OH * p->OW * p->ldi2 * elt;
    if (g_driver_version <= 13010 && bytes2 < 131072) reinterpret_cast<uint64_t*>(&a.map_a2)[1] &= ~(1llu << 21);
    a.kchunks2 = ceil_div(p->Cin2, kc);
  }
  // ---- packed weights [Cout][K] -> tile {kc, BN}
  int bn = pick_bn(p->Cout);
  if (!halo) {
    // Few tiles (small per-GPU batch, the strong-scaling regime): each CTA of an im2col layer streams the WHOLE weight matrix
    // and its own A tile through one SM's L2 port (~64 B/clk: measured 24 us for 3x3 256+256->256 @7x7 at batch 128, 49
    // CTAs on 49 SMs, 2 MB each, against 10 us of tensor time).  Narrower N tiles spread the weights over more SMs - the K
    // order, hence the result, does not change.  Enter when the layer has fewer CTAs than SMs / ENTER, narrow until it has
    // at least SMs / STOP (ENTER = STOP = 2, measured: profiles/r02_conv_nsplit.md).
    constexpr int NS_ENTER = 2, NS_STOP = 2;
    const int tiles_m = ceil_div((long long)p->B * p->OH * p->OW, BM);
    if (tiles_m * (p->Cout / bn) * NS_ENTER <= g_num_sms) {
      static const int cand[] = {128, 96, 64, 48, 32};
      for (int c : cand) {
        if (c >= bn || p->Cout % c) continue;
        bn = c;
        if (tiles_m * (p->Cout / bn) * NS_STOP >= g_num_sms) break;
      }
    }
  }
  {
    const int K = p->ntaps * p->Cin + (p->in2 ? p->Cin2 : 0);
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)p->Cout};
    const cuuint64_t strides[1] = {(cuuint64_t)K * elt};
    const cuuint32_t box[2] = {(cuuint32_t)kc, (cuuint32_t)bn};
    const cuuint32_t estr[2] = {1, 1};
    void* base = const_cast<void*>(half ? p->weight_lp : reinterpret_cast<const void*>(p->weight));
    CUresult r = g_encode_tiled(&a.map_b, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                                base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled(weights) failed (%d): K=%d Cout=%d", (int)r, K, p->Cout);
      return CNB_ERR_CUDA;
    }
  }
  // ---- dense fp16 output (+ fp16 residual): the epilogue stores / fetches 32-row x SLAB-column boxes by TMA (EPI 6)
  {
    const bool dense = !halo && p->oy_mul == 1 && p->ox_mul == 1 && p->oy_add == 0 && p->ox_add == 0 &&
                       p->OHf * p->OWf == p->OH * p->OW;
    const bool simple = dense && p->act == 0 && !(p->temb && p->temb_per_sample);
    const bool res_ok = !p->residual || (p->res_dtype == 1 && p->ldr % 8 == 0 && p->res_coff % 8 == 0);
    if (half && simple && p->out_dtype == 1 && p->ldo % 8 == 0 && p->out_coff % 8 == 0 && res_ok) {
      const int slab = bn % 64 == 0 ? 32 : 16;
      const CUtensorMapSwizzle sw_o = slab == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
      const cuuint64_t dims[2] = {(cuuint64_t)p->Cout, (cuuint64_t)p->B * p->OH * p->OW};
      const cuuint32_t box[2] = {(cuuint32_t)slab, 32u};
      const cuuint32_t estr[2] = {1, 1};
      const cuuint64_t so[1] = {(cuuint64_t)p->ldo * 2};
      void* ob = reinterpret_cast<char*>(p->out) + (size_t)p->out_coff * 2;
      CUresult r = g_encode_tiled(&a.map_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ob, dims, so, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw_o, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r == CUDA_SUCCESS && p->residual) {
        const cuuint64_t sr[1] = {(cuuint64_t)p->ldr * 2};
        void* rb_ = const_cast<char*>(reinterpret_cast<const char*>(p->residual) + (size_t)p->res_coff * 2);
        r = g_encode_tiled(&a.map_res, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, rb_, dims, sr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, sw_o, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      }
      a.tma_epi = r == CUDA_SUCCESS ? 1 : 0;                 // on failure the register / shared-memory epilogue runs
    }
  }
  a.bias = p->bias; a.temb = p->temb; a.residual = p->residual; a.out = p->out;
  a.M = p->B * p->OH * p->OW; a.OHW = p->OH * p->OW; a.OW = p->OW;
  a.OHf = p->OHf; a.OWf = p->OWf;
  a.oy_mul = p->oy_mul; a.oy_add = p->oy_add; a.ox_mul = p->ox_mul; a.ox_add = p->ox_add;
  a.Cout = p->Cout; a.ldo = p->ldo; a.out_coff = p->out_coff; a.ldr = p->ldr; a.res_coff = p->res_coff;
  a.temb_ld = p->temb_ld; a.temb_per_sample = p->temb_per_sample; a.act = p->act; a.out_f16 = p->out_dtype == 1; a.res_f16 = p->res_dtype == 1;
  a.Cin = p->Cin; a.ntaps = p->ntaps; a.kchunks = ceil_div(p->Cin, kc);
  a.stride = p->stride; a.lower_w = dxmin; a.lower_h = dymin;
  a.tiles_m = halo ? p->B * a.tiles_y : ceil_div(a.M, BM); a.tiles_n = p->Cout / bn;
  if (route) {
    route[CNB_ROUTE_PATH] = CNB_PATH_TMA;
    route[CNB_ROUTE_RB] = rb;
    route[CNB_ROUTE_BN] = bn;
    route[CNB_ROUTE_HALO] = halo ? 1 : 0;
    route[CNB_ROUTE_TILES_N] = a.tiles_n;
    route[CNB_ROUTE_HALO_R] = halo ? a.R : 0;
    route[CNB_ROUTE_TILES_Y] = halo ? a.tiles_y : 0;
  }
  return half ? conv_tma_launch_f16(rb, bn, a, g_num_sms, st, route)
              : conv_tma_launch_tf32(rb, bn, a, g_num_sms, st, route);
}

}  // namespace cnb
