// C-ABI glue: error text, launch counter, argument validation and mode dispatch.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>

#include "common.cuh"

namespace cnb {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

bool pdl_enabled(long long work) {
  static int mode = -1;
  static long long limit = 4ll << 20;
  if (mode < 0) {
    const char* e = getenv("CNB_PDL");
    const char* w = getenv("CNB_PDL_WORK");
    if (w) limit = atoll(w);
    mode = e ? atoi(e) : 2;      // 0 = never, 1 = always, 2 = auto (short launches only; see common.cuh)
  }
  return mode == 1 || (mode == 2 && work <= limit);
}

int conv2d_f32(const cnb_conv_params* p, cudaStream_t st);
int conv2d_small(const cnb_conv_params* p, cudaStream_t st);
bool conv2d_small_supported(const cnb_conv_params* p);
int conv2d_tma(const cnb_conv_params* p, cudaStream_t st, int32_t* route);
bool conv2d_tma_supported(const cnb_conv_params* p);
bool groupnorm_big_eligible(int B, int HW, int C, int G, int in_f16);
size_t groupnorm_big_workspace(int B, int HW, int C, int G);
int groupnorm_big(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G, float eps,
                  int silu, int out_f16, void* workspace, size_t ws_bytes, cudaStream_t st);
int groupnorm(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C, int G,
              float eps, int silu, int in_f16, int out_f16, cudaStream_t st);
int attention_f32(const float* qkv, float* out, int B, int L, int E, int heads, cudaStream_t st);
int attention_f16(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st);
bool attention_f16_supported(int E, int heads);
int attention_tmem(const void* qkv, void* out, int B, int L, int E, int heads, cudaStream_t st);
bool attention_tmem_supported(const void* qkv, const void* out, int B, int L, int E, int heads);
bool attention_tmem_default(int L, int d);

static int g_has_tc = -1;
static int query_tc() {
  if (g_has_tc >= 0) return g_has_tc;
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;   // not cached: a device may appear later
  }
  g_has_tc = (prop.major == 10) ? 1 : 0;
  return g_has_tc;
}

}  // namespace cnb

using namespace cnb;

extern "C" int cnb_abi_version(void) { return 1; }
extern "C" int cnb_sizeof_conv_params(void) { return (int)sizeof(cnb_conv_params); }
extern "C" const char* cnb_last_error(void) { return g_err; }
extern "C" long long cnb_launch_count(void) { return g_launches.load(); }
extern "C" void cnb_reset_launch_count(void) { g_launches.store(0); }
extern "C" int cnb_has_tcgen05(void) { return query_tc(); }

// One decision for cnb_conv2d and cnb_conv2d_route: with `route` set, every branch fills it in and returns where it
// would launch.
static int conv2d_dispatch(const cnb_conv_params* p, cudaStream_t st, int32_t* route) {
  CNB_REQUIRE(p != nullptr, "conv2d: null params");
  CNB_REQUIRE(p->in && p->weight && p->out, "conv2d: null tensor pointer");
  CNB_REQUIRE(p->B > 0 && p->H > 0 && p->W > 0 && p->Cin > 0 && p->Cout > 0 && p->OH > 0 && p->OW > 0,
              "conv2d: non-positive dimension");
  CNB_REQUIRE(p->ntaps >= 1 && p->ntaps <= CNB_MAX_TAPS, "conv2d: ntaps=%d", p->ntaps);
  CNB_REQUIRE(p->ldi >= p->in_coff + p->Cin && p->ldo >= p->out_coff + p->Cout, "conv2d: leading dimension too small");
  CNB_REQUIRE(!p->residual || p->ldr >= p->res_coff + p->Cout, "conv2d: residual leading dimension too small");
  CNB_REQUIRE(!p->temb || p->temb_ld >= p->Cout, "conv2d: temb leading dimension too small");
  CNB_REQUIRE((long long)p->B * p->OH * p->OW < (1ll << 31), "conv2d: M overflows int32");
  CNB_REQUIRE((p->OH - 1) * p->oy_mul + p->oy_add < p->OHf && (p->OW - 1) * p->ox_mul + p->ox_add < p->OWf,
              "conv2d: output mapping exceeds the output tensor");
  CNB_REQUIRE(p->in_dtype == 0 || p->in_dtype == 1, "conv2d: in_dtype=%d", p->in_dtype);
  CNB_REQUIRE(p->out_dtype == 0 || p->out_dtype == 1, "conv2d: out_dtype=%d", p->out_dtype);
  CNB_REQUIRE(p->res_dtype == 0 || p->res_dtype == 1, "conv2d: res_dtype=%d", p->res_dtype);
  if (p->in2) {
    CNB_REQUIRE(p->Cin2 > 0 && p->ldi2 >= p->in2_coff + p->Cin2, "conv2d: bad second input");
    CNB_REQUIRE(p->mode != CNB_MODE_F32 && conv2d_tma_supported(p),
                "conv2d: a second input (K-concatenated 1x1 tap) needs the TMA tensor-core path");
    return conv2d_tma(p, st, route);
  }
  // tiny-channel ends of the U-Net (Cin <= 4 or Cout <= 4): direct exact-fp32 kernels in every mode
  if ((p->Cin <= 4 || p->Cout <= 4) && conv2d_small_supported(p)) {
    if (route) {
      route[CNB_ROUTE_PATH] = CNB_PATH_SMALL;
      return CNB_OK;
    }
    return conv2d_small(p, st);
  }
  if (p->mode == CNB_MODE_F16) {
    if (conv2d_tma_supported(p)) return conv2d_tma(p, st, route);     // TMA-im2col fed persistent tcgen05 kernel
  } else if (p->mode != CNB_MODE_F32) {
    set_error("conv2d: unknown mode %d", p->mode);
    return CNB_ERR_BAD_ARG;
  }
  // fp32 mode, and tiny-channel layers (Cin % 4 != 0 or Cout < 16) which are HBM-bound CUDA-core work
  CNB_REQUIRE(p->out_dtype == 0 && p->res_dtype == 0, "conv2d: fp16 output / residual needs a tensor-core eligible layer");
  CNB_REQUIRE(p->in_dtype == 0, "conv2d: fp16 activations need a tensor-core eligible layer (Cin %% 8 == 0, Cout %% 16 == 0)");
  if (route) {
    route[CNB_ROUTE_PATH] = CNB_PATH_F32;
    return CNB_OK;
  }
  return conv2d_f32(p, st);
}

extern "C" int cnb_conv2d(const cnb_conv_params* p, cnb_stream_t stream) {
  return conv2d_dispatch(p, (cudaStream_t)stream, nullptr);
}

extern "C" int cnb_conv2d_route(const cnb_conv_params* p, int32_t* route) {
  CNB_REQUIRE(route != nullptr, "conv2d_route: null route");
  memset(route, 0, CNB_ROUTE_LEN * sizeof(int32_t));
  return conv2d_dispatch(p, nullptr, route);
}

extern "C" size_t cnb_groupnorm_workspace_bytes(int B, int HW, int C, int G, int in_f16) {
  if (B <= 0 || HW <= 0 || C <= 0 || G <= 0 || !groupnorm_big_eligible(B, HW, C, G, in_f16)) return 0;
  return groupnorm_big_workspace(B, HW, C, G);
}

extern "C" int cnb_groupnorm_ws(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C,
                                int G, float eps, int silu, int in_f16, int out_f16, void* workspace, size_t ws_bytes,
                                cnb_stream_t stream) {
  CNB_REQUIRE(x && y && gamma && beta && B > 0 && HW > 0 && C > 0 && G > 0, "groupnorm: bad args");
  if (workspace && groupnorm_big_eligible(B, HW, C, G, in_f16))
    return groupnorm_big(x, y, gamma, beta, B, HW, C, G, eps, silu, out_f16, workspace, ws_bytes, (cudaStream_t)stream);
  return groupnorm(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, (cudaStream_t)stream);
}

extern "C" int cnb_groupnorm(const void* x, void* y, const float* gamma, const float* beta, int B, int HW, int C,
                             int G, float eps, int silu, int in_f16, int out_f16, cnb_stream_t stream) {
  CNB_REQUIRE(x && y && gamma && beta && B > 0 && HW > 0 && C > 0 && G > 0, "groupnorm: bad args");
  return groupnorm(x, y, gamma, beta, B, HW, C, G, eps, silu, in_f16, out_f16, (cudaStream_t)stream);
}

extern "C" int cnb_attention(const float* qkv, float* out, int B, int L, int E, int heads, int mode,
                             cnb_stream_t stream) {
  CNB_REQUIRE(qkv && out && B > 0 && L > 0 && E > 0, "attention: bad args");
  (void)mode;   // fp32 q|k|v always take the exact fp32 core (the tensor-core modes keep q|k|v in fp16: cnb_attention_f16)
  return attention_f32(qkv, out, B, L, E, heads, (cudaStream_t)stream);
}

extern "C" int cnb_attention_f16(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream) {
  CNB_REQUIRE(qkv && out && B > 0 && L > 0 && E > 0, "attention_f16: bad args");
  if (!attention_f16_supported(E, heads)) {
    set_error("attention_f16: E=%d heads=%d (head dim %d) is not instantiated", E, heads, heads > 0 ? E / heads : 0);
    return CNB_ERR_UNSUPPORTED;
  }
  // the tcgen05 / TMEM kernel (S, P and O in tensor memory, csrc/attention_tmem.cu) where it measured faster (head dim
  // >= 24, >= 128 tokens: the CIFAR and CelebHQ-latent levels), the register-resident mma.sync kernel elsewhere
  if (heads > 0 && attention_tmem_default(L, E / heads) && attention_tmem_supported(qkv, out, B, L, E, heads))
    return attention_tmem(qkv, out, B, L, E, heads, (cudaStream_t)stream);
  return attention_f16(qkv, out, B, L, E, heads, (cudaStream_t)stream);
}

extern "C" int cnb_attention_tmem(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream) {
  CNB_REQUIRE(qkv && out && B > 0 && L > 0 && E > 0, "attention_tmem: bad args");
  if (!attention_tmem_supported(qkv, out, B, L, E, heads)) {
    set_error("attention_tmem: needs head dim in {4, 8, 16, 24, 32, 48, 64} and 16-byte aligned fp16 rows (E=%d heads=%d L=%d)",
              E, heads, L);
    return CNB_ERR_UNSUPPORTED;
  }
  return attention_tmem(qkv, out, B, L, E, heads, (cudaStream_t)stream);
}

extern "C" int cnb_attention_mma(const void* qkv, void* out, int B, int L, int E, int heads, cnb_stream_t stream) {
  CNB_REQUIRE(qkv && out && B > 0 && L > 0 && E > 0, "attention_mma: bad args");
  if (!attention_f16_supported(E, heads)) {
    set_error("attention_mma: E=%d heads=%d (head dim %d) is not instantiated", E, heads, heads > 0 ? E / heads : 0);
    return CNB_ERR_UNSUPPORTED;
  }
  return attention_f16(qkv, out, B, L, E, heads, (cudaStream_t)stream);
}

// Reads (and clears) the hang-guard latch of every translation unit that issues tcgen05 / TMA work (csrc/tc_common.cuh).
namespace cnb {
int conv_tma_error_flag();        // conv_tma.cu
int attention_tmem_error_flag();  // attention_tmem.cu
}
extern "C" int cnb_tc_error_flag(void) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cnb::set_error("device error: %s", cudaGetErrorString(e));
    return CNB_ERR_CUDA;
  }
  const int h = cnb::conv_tma_error_flag() | cnb::attention_tmem_error_flag();
  if (h < 0) {
    cnb::set_error("cudaMemcpyFromSymbol failed while reading the tcgen05 hang-guard flag");
    return CNB_ERR_CUDA;
  }
  return h;
}
