// Translation unit of the fp32 tcgen05 token GEMM (see gemm_t32.cuh).
#define LEWIN_TU_LITE 1      // no GELU tables / non-template kernels in this unit (they live in lewin_abi.cu)
#include "gemm_t32_api.h"
#include "gemm_t32.cuh"

namespace lewin {

bool gemm_t32_supported(const GemmArgs<float>& g, int epi) {
    if (epi == EPI_BIAS) return t32::supported<EPI_BIAS>(g);
    if (epi == EPI_BIAS_GELU) return t32::supported<EPI_BIAS_GELU>(g);
    if (epi == EPI_BIAS_RESID) return t32::supported<EPI_BIAS_RESID>(g);
    return false;
}

cudaError_t gemm_t32_launch(const GemmArgs<float>& g, int epi, int sms, cudaStream_t stream) {
    if (epi == EPI_BIAS) return t32::launch<EPI_BIAS>(g, sms, stream);
    if (epi == EPI_BIAS_GELU) return t32::launch<EPI_BIAS_GELU>(g, sms, stream);
    if (epi == EPI_BIAS_RESID) return t32::launch<EPI_BIAS_RESID>(g, sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace lewin

#ifdef LEWIN_T32_PROF_BUILD
// diagnostic build only (nvcc -DLEWIN_T32_PROF_BUILD): copy the LEWIN_T32_PROF counters to `out` (8 launch slots x 16 values) and optionally clear them; returns 0 if profiling is off
extern "C" int lewin_debug_t32_prof(unsigned long long* out, int reset) {
    unsigned long long* p = lewin::t32::prof_buffer();
    if (!p) return 0;
    cudaDeviceSynchronize();
    cudaMemcpy(out, p, 128 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    if (reset) { cudaMemset(p, 0, 128 * sizeof(unsigned long long)); lewin::t32::prof_launches() = 0; }
    return 1;
}
#endif
