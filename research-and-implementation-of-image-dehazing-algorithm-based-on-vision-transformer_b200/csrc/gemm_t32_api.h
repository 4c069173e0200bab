// Entry of the fp32 tcgen05 (3xTF32) token GEMM (gemm_t32.cuh), compiled as its own translation unit (lewin_gemm_t32.cu).
#pragma once
#include "gemm_fused.cuh"

namespace lewin {
// true if the forward GEMM described by `g` with epilogue `epi` (EPI_BIAS / EPI_BIAS_GELU / EPI_BIAS_RESID) can run on it
bool gemm_t32_supported(const GemmArgs<float>& g, int epi);
// launches it on `stream` (persistent grid sized from the current device's SM count)
cudaError_t gemm_t32_launch(const GemmArgs<float>& g, int epi, int num_sms, cudaStream_t stream);
}  // namespace lewin
