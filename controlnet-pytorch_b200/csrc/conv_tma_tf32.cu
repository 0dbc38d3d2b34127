// kind::tf32 instantiations of conv_tma_kernel (fp32 activations x tf32-rounded fp32 weights).
#include "conv_tma_impl.cuh"

namespace cnb {
int conv_tma_launch_tf32(int rb, int bn, const tma::TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route) {
  return tma::dispatch_rb<false>(rb, bn, a, num_sms, st, route);
}
int conv_tma_error_flag_tf32() { return tc_read_clear_error(); }
}  // namespace cnb
