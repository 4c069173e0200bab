// Translation unit of the tcgen05 weight-gradient kernel (see wgrad_tc.cuh).
#define LEWIN_TU_LITE 1      // no GELU tables / non-template kernels in this unit (they live in lewin_abi.cu)
#include "wgrad_tc_api.h"
#include "wgrad_tc.cuh"

namespace lewin {
bool wgrad_tc_supported(const WgradArgs<__nv_bfloat16>& g) { return wg3::supported(g); }
cudaError_t wgrad_tc_launch(const WgradArgs<__nv_bfloat16>& g, int num_sms, bool det, cudaStream_t stream) {
    return det ? wg3::launch<true>(g, num_sms, stream) : wg3::launch<false>(g, num_sms, stream);
}
}  // namespace lewin
