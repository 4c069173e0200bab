// Entry of the tcgen05 weight-gradient kernel (wgrad_tc.cuh), compiled as its own translation unit (lewin_wgrad_tc.cu).
#pragma once
#include <cuda_bf16.h>
#include "wgrad_args.cuh"

namespace lewin {
// true if dW[N,K] += dY^T X with these arguments can run on the tensor-memory kernel: plain bf16 operands (no gather / LN /
// DropPath / gelu' prologue), N % 128 == 0, K % 128 == 0
bool wgrad_tc_supported(const WgradArgs<__nv_bfloat16>& g);
// det: stores per-split partials into the slabs g.dW / g.db (det_wgrad_rows_per_split) instead of accumulating
cudaError_t wgrad_tc_launch(const WgradArgs<__nv_bfloat16>& g, int num_sms, bool det, cudaStream_t stream);
}  // namespace lewin
