// kind::f16 instantiations of conv_tma_kernel (fp16 activations x fp16 weights).  Split from conv_tma_tf32.cu only so the
// two halves of the template matrix compile in parallel.
#include "conv_tma_impl.cuh"

namespace cnb {
int conv_tma_launch_f16(int rb, int bn, const tma::TmaArgs& a, int num_sms, cudaStream_t st, int32_t* route) {
  return tma::dispatch_rb<true>(rb, bn, a, num_sms, st, route);
}
int conv_tma_error_flag_f16() { return tc_read_clear_error(); }
}  // namespace cnb
