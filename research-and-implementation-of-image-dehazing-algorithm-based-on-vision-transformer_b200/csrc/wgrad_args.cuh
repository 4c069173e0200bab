// Arguments of the weight-gradient kernels (backward.cuh: generic wgrad_kernel; wgrad_bf16.cuh: bf16 fast path).
#pragma once
#include "common.cuh"

namespace lewin {

template <typename T>
struct WgradArgs {
    const T* dY; long long lddy;      // [rows, lddy]; columns [0, N) used
    const T* X;  long long ldx;       // [rows, ldx];  columns [0, K) used
    float* dW;                        // [N, K] fp32, accumulated with atomics (deterministic kernels: slab [splits][N, K], stored)
    float* db;                        // [N] or null (deterministic kernels: slab [splits][N])
    long long M;
    int N, K;
    int mapDY, mapX;                  // operand rows are tokens addressed through `map` (row m is window-ordered)
    WinMap map;
    const float* dy_row_scale;        // [B] or null (DropPath factor on dY rows)
    int tokens_per_image;
    const float* mean; const float* rstd; const float* ln_w; const float* ln_b;   // LN prologue on X (null mean => none)
    const T* dy_aux;                  // null, or pre-activation: dY is multiplied by gelu'(aux) (same indexing as dY)
    long long rows_per_split;         // multiple of 32
};

// Deterministic weight gradients: every kernel family splits the token axis the same way, as a function of the shape alone
// (never of the SM count), so the partial slabs [splits][N, K] and the workspace that holds them are known on the host.
// About one 128 x 256 tile of dW per SM of a full B200 (148 SMs), at least four 64-token stages per split, at most 256 splits.
inline long long det_wgrad_rows_per_split(long long M, int N, int K) {
    const long long nk = static_cast<long long>(N) * K;
    long long want = (148ll * 32768 + nk - 1) / nk;
    const long long max_splits = (M + 255) / 256;
    if (want > max_splits) want = max_splits;
    if (want > 256) want = 256;
    if (want < 1) want = 1;
    long long rps = (M + want - 1) / want;
    return (rps + 63) / 64 * 64;
}
inline long long det_wgrad_splits(long long M, int N, int K) {
    const long long rps = det_wgrad_rows_per_split(M, N, K);
    return (M + rps - 1) / rps;
}


}  // namespace lewin
