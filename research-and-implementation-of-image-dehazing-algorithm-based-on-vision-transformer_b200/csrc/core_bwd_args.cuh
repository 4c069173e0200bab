// Arguments of the ProbSparse core backward kernels (backward.cuh: generic; probsparse_core_bwd_v2.cuh: bf16 fast path).
#pragma once
#include "common.cuh"

namespace lewin {

template <typename T>
struct CoreBwdArgs {
    const T* qkv;            // [B_*64, 3C]
    const T* dctx;           // [B_*64, C]
    T* dqkv;                 // [B_*64, 3C]
    const uint8_t* top;      // [B_, nH, 25]
    const float* rpb_table; const float* rpb_dense;
    float* d_rpb_table;      // [225, nH] accumulated (null => skipped)
    float* d_rpb_dense;      // [nH, 64, 64] accumulated: gradient w.r.t. the gathered bias (null => skipped)
    const float* mask; int nW_mask;
    int B_, nH, C, use_rpb;
    int shift, H, W, nWw, nWin;
    const float* tmask; int Bm;   // input mask per token [Bm, H, W] or null (CoreFwdArgs::tmask)
};

}  // namespace lewin
