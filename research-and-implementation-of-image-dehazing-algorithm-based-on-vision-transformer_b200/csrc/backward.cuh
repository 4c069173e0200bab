// Backward of the LeWin hot path (the reference has no backward code: these kernels restate what
// torch.autograd derives from My_model_1.py:785-875 and ProbSparse/attn.py:287-461; gradient paths in
// SURVEY.md section 3.4, oracle restatement in oracle/lewin_oracle.py::lewin_block_bwd).
//
//   wgrad_kernel          dW[n,k] += sum_m dY[m,n] * X[m,k],  db[n] += sum_m dY[m,n]   (tokens are the K dim)
//   ln_bwd_kernel         LayerNorm backward + residual-path add + d(gamma), d(beta)
//   dwconv_bwd_kernel     depthwise 3x3 backward (data + weight + bias) with both GELU derivatives fused
//   probsparse_core_bwd   dq, dk, dv and d(rpb table) of the ProbSparse core for the saved top-u selection
//   transpose_kernel      W -> W^T staging for the data-gradient GEMMs (gemm_fused_kernel)
#pragma once
#include "../../include/lewin_b200.h"
#include "common.cuh"
#include "dwconv.cuh"
#include "gemm_fused.cuh"
#include "gemm_tc.cuh"
#include "probsparse_core.cuh"
#include "wgrad_args.cuh"
#include "wgrad_bf16.cuh"
#include "wgrad_tc_api.h"
#include "core_bwd_args.cuh"
#include "probsparse_core_bwd_v2.cuh"

namespace lewin {

inline size_t bw_align(size_t v) { return (v + 255) / 256 * 256; }

// ------------------------------------------------------------------------------ transpose
__global__ void transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int R, int Cc) {
    __shared__ float tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int r = by + i, c = bx + threadIdx.x;
        tile[i][threadIdx.x] = (r < R && c < Cc) ? src[static_cast<long long>(r) * Cc + c] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int c = bx + i, r = by + threadIdx.x;
        if (r < R && c < Cc) dst[static_cast<long long>(c) * R + r] = tile[threadIdx.x][i];
    }
}
inline cudaError_t launch_transpose(const float* src, float* dst, int R, int Cc, cudaStream_t st) {
    dim3 grid((Cc + 31) / 32, (R + 31) / 32), block(32, 8);
    transpose_kernel<<<grid, block, 0, st>>>(src, dst, R, Cc);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------ weight gradient (WgradArgs: wgrad_args.cuh)
constexpr int WG_BM = 32;             // tokens per stage
constexpr int WG_THREADS = 256;

template <typename T, int TILE>       // TILE = 64 or 32: dW tile is TILE x TILE
__global__ void __launch_bounds__(WG_THREADS) wgrad_kernel(const WgradArgs<T> g) {
    constexpr int PASSES = Act<T>::kPasses;
    constexpr int LD = TILE + 8;                  // (8t + g) % 32 distinct -> conflict-free transposed fragment loads
    constexpr int WN = TILE / 2;                  // warp tile rows (n): 2 warps along n
    constexpr int WK = TILE / 4;                  // warp tile cols (k): 4 warps along k
    constexpr int MT = WN / 16, NT = WK / 8;
    __shared__ __align__(16) float dYs[WG_BM * LD];
    __shared__ __align__(16) float Xs[WG_BM * LD];
    __shared__ long long offD[WG_BM], offX[WG_BM];
    __shared__ float s_mu[WG_BM], s_rs[WG_BM], s_sc[WG_BM];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int wn = warp & 1, wk = warp >> 1;
    const int n0 = blockIdx.x * TILE, k0 = blockIdx.y * TILE;
    const long long m_begin = static_cast<long long>(blockIdx.z) * g.rows_per_split;
    long long m_end = m_begin + g.rows_per_split;
    if (m_end > g.M) m_end = g.M;
    const bool has_ln = g.mean != nullptr;

    float acc[MT][NT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;
    float bsum = 0.f;

    for (long long mb = m_begin; mb < m_end; mb += WG_BM) {
        __syncthreads();
        if (tid < WG_BM) {
            long long m = mb + tid;
            long long od = -1, ox = -1;
            float mu = 0.f, rs = 1.f, sc = 1.f;
            if (m < m_end) {
                long long tok = (g.mapDY || g.mapX) ? g.map.token(m) : m;
                long long rd = g.mapDY ? tok : m, rx = g.mapX ? tok : m;
                od = rd * g.lddy; ox = rx * g.ldx;
                if (has_ln) { mu = g.mean[rx]; rs = g.rstd[rx]; }
                if (g.dy_row_scale) sc = g.dy_row_scale[rd / g.tokens_per_image];
            }
            offD[tid] = od; offX[tid] = ox; s_mu[tid] = mu; s_rs[tid] = rs; s_sc[tid] = sc;
        }
        __syncthreads();
        // stage 32 x TILE of dY and X (float4 chunks)
        constexpr int CH = WG_BM * TILE / 4;
        for (int c = tid; c < 2 * CH; c += WG_THREADS) {
            const bool isx = c >= CH;
            const int cc = isx ? c - CH : c;
            const int r = cc / (TILE / 4), q4 = (cc % (TILE / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!isx) {
                const long long o = offD[r];
                if (o >= 0) {
                    v = ld4(g.dY + o + n0 + q4);
                    if (g.dy_aux) {
                        const float4 p = ld4(g.dy_aux + o + n0 + q4);
                        v.x *= gelu_erf_grad(p.x); v.y *= gelu_erf_grad(p.y);
                        v.z *= gelu_erf_grad(p.z); v.w *= gelu_erf_grad(p.w);
                    }
                    const float sc = s_sc[r];
                    v.x *= sc; v.y *= sc; v.z *= sc; v.w *= sc;
                }
                *reinterpret_cast<float4*>(dYs + r * LD + q4) = v;
            } else {
                const long long o = offX[r];
                if (o >= 0) {
                    v = ld4(g.X + o + k0 + q4);
                    if (has_ln) {
                        const float mu = s_mu[r], rs = s_rs[r];
                        const float4 w = *reinterpret_cast<const float4*>(g.ln_w + k0 + q4);
                        const float4 b = *reinterpret_cast<const float4*>(g.ln_b + k0 + q4);
                        v.x = (v.x - mu) * rs * w.x + b.x; v.y = (v.y - mu) * rs * w.y + b.y;
                        v.z = (v.z - mu) * rs * w.z + b.z; v.w = (v.w - mu) * rs * w.w + b.w;
                        if (Act<T>::kIsBf16) {
                            v.x = Act<T>::round(v.x); v.y = Act<T>::round(v.y);
                            v.z = Act<T>::round(v.z); v.w = Act<T>::round(v.w);
                        }
                    }
                }
                *reinterpret_cast<float4*>(Xs + r * LD + q4) = v;
            }
        }
        __syncthreads();
        if (g.db && blockIdx.y == 0 && tid < TILE) {
#pragma unroll 8
            for (int r = 0; r < WG_BM; ++r) bsum += dYs[r * LD + tid];
        }
#pragma unroll
        for (int ks = 0; ks < WG_BM / 8; ++ks) {
            float af[MT][4], bf[NT][2];
#pragma unroll
            for (int i = 0; i < MT; ++i) {      // A[n][m] = dYs[m][n]
                const float* p = dYs + (ks * 8 + tq) * LD + wn * WN + i * 16 + gq;
                af[i][0] = p[0]; af[i][1] = p[8]; af[i][2] = p[4 * LD]; af[i][3] = p[4 * LD + 8];
            }
#pragma unroll
            for (int j = 0; j < NT; ++j) {      // B[m][k] = Xs[m][k]
                const float* p = Xs + (ks * 8 + tq) * LD + wk * WK + j * 8 + gq;
                bf[j][0] = p[0]; bf[j][1] = p[4 * LD];
            }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < NT; ++j) mma_x<PASSES>(acc[i][j], af[i], bf[j]);
        }
    }
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int n = n0 + wn * WN + i * 16 + gq + half * 8;
                const int k = k0 + wk * WK + j * 8 + 2 * tq;
                atomicAdd(g.dW + static_cast<long long>(n) * g.K + k, acc[i][j][half * 2]);
                atomicAdd(g.dW + static_cast<long long>(n) * g.K + k + 1, acc[i][j][half * 2 + 1]);
            }
    if (g.db && blockIdx.y == 0 && tid < TILE) atomicAdd(g.db + n0 + tid, bsum);
}

template <typename T>
cudaError_t launch_wgrad(WgradArgs<T> g, int num_sms, cudaStream_t st) {
    if constexpr (Act<T>::kIsBf16) {
        if (wgrad_tc_supported(g)) return wgrad_tc_launch(g, num_sms, st);   // plain operands, C >= 128: tcgen05 (wgrad_tc.cuh)
        if (wg2::supported(g)) return wg2::launch(g, num_sms, st);      // pipelined bf16 path (wgrad_bf16.cuh)
    }
    const int tile = (g.N % 64 == 0 && g.K % 64 == 0) ? 64 : 32;
    const long long tiles = static_cast<long long>(g.N / tile) * (g.K / tile);
    long long want = (static_cast<long long>(num_sms) * 4 + tiles - 1) / tiles;
    long long max_splits = (g.M + WG_BM - 1) / WG_BM;
    if (want > max_splits) want = max_splits;
    if (want < 1) want = 1;
    long long rps = (g.M + want - 1) / want;
    rps = (rps + WG_BM - 1) / WG_BM * WG_BM;
    const unsigned splits = static_cast<unsigned>((g.M + rps - 1) / rps);
    g.rows_per_split = rps;
    dim3 grid(g.N / tile, g.K / tile, splits);
    if (tile == 64) wgrad_kernel<T, 64><<<grid, WG_THREADS, 0, st>>>(g);
    else wgrad_kernel<T, 32><<<grid, WG_THREADS, 0, st>>>(g);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------ LayerNorm backward
// dx[row] = dres[row] + LNbwd(dz[row]; x[row], gamma);  dgamma += sum dz * xhat;  dbeta += sum dz.
// G lanes per row with 16-byte loads (a warp streams 32/G rows at once), grid-stride over rows, per-lane register
// partials for dgamma / dbeta reduced through shuffles + shared memory, one global atomic per column per block.
template <typename T, int G, int MAXV>
__global__ void __launch_bounds__(256, MAXV == 1 ? 3 : 1) ln_bwd_kernel(const T* __restrict__ dz, const T* __restrict__ x,
                                                     const T* __restrict__ dres, T* __restrict__ dx,
                                                     const float* __restrict__ gamma, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, long long rows, int C) {
    constexpr int EPL = 16 / sizeof(T);
    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31, sub = lane / G, gl = lane % G;
    const long long warp_global = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long nwarps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    float gacc[MAXV][EPL], bacc[MAXV][EPL], gm[MAXV][EPL];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int k = (gl + i * G) * EPL;
#pragma unroll
        for (int j = 0; j < EPL; ++j) { gacc[i][j] = 0.f; bacc[i][j] = 0.f; gm[i][j] = (k < C) ? gamma[k + j] : 0.f; }
    }
    auto unpack = [&](const uint4 u, float (&f)[EPL]) {
        if (sizeof(T) == 4) {
            f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w);
        } else {
            f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
            f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
            f[EPL - 4] = __uint_as_float(u.z << 16); f[EPL - 3] = __uint_as_float(u.z & 0xFFFF0000u);
            f[EPL - 2] = __uint_as_float(u.w << 16); f[EPL - 1] = __uint_as_float(u.w & 0xFFFF0000u);
        }
    };
    // software pipeline: the raw 16-byte pieces of the NEXT row group (x, dz, dres) are requested before this one is reduced,
    // so a warp always has a row group in flight under its three shuffle reductions (the loop was one exposed memory latency
    // per iteration: ncu long-scoreboard 4.7 at 34 % occupancy).  Zero bits = 0.0f in both dtypes.
    uint4 nx[MAXV], nd[MAXV], nr[MAXV];
    auto request = [&](long long row0) {
        const long long row = row0 + sub;
        const bool live = row0 < rows && row < rows;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int k = (gl + i * G) * EPL;
            const uint4 z = make_uint4(0u, 0u, 0u, 0u);
            nx[i] = z; nd[i] = z; nr[i] = z;
            if (live && k < C) {
                nx[i] = *reinterpret_cast<const uint4*>(x + row * C + k);
                nd[i] = *reinterpret_cast<const uint4*>(dz + row * C + k);
                if (dres) nr[i] = *reinterpret_cast<const uint4*>(dres + row * C + k);
            }
        }
    };
    request(warp_global * RPW);
    for (long long row0 = warp_global * RPW; row0 < rows; row0 += nwarps * RPW) {
        const long long row = row0 + sub;
        const bool live = row < rows;
        float xv[MAXV][EPL], dv[MAXV][EPL], rv[MAXV][EPL];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            unpack(nx[i], xv[i]); unpack(nd[i], dv[i]); unpack(nr[i], rv[i]);
#pragma unroll
            for (int j = 0; j < EPL; ++j) s += xv[i][j];
        }
        request(row0 + nwarps * RPW);
        const float mu = group_sum<G>(s) / C;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int k = (gl + i * G) * EPL;
            if (k < C) {
#pragma unroll
                for (int j = 0; j < EPL; ++j) { xv[i][j] -= mu; q += xv[i][j] * xv[i][j]; }
            }
        }
        const float rs = rsqrtf(group_sum<G>(q) / C + 1e-5f);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int k = (gl + i * G) * EPL;
            if (live && k < C) {
#pragma unroll
                for (int j = 0; j < EPL; ++j) {
                    xv[i][j] *= rs;                                   // xhat
                    gacc[i][j] += dv[i][j] * xv[i][j];
                    bacc[i][j] += dv[i][j];
                    dv[i][j] *= gm[i][j];                             // dxhat
                    s1 += dv[i][j];
                    s2 += dv[i][j] * xv[i][j];
                }
            }
        }
        s1 = group_sum<G>(s1) / C;
        s2 = group_sum<G>(s2) / C;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int k = (gl + i * G) * EPL;
            if (live && k < C) {
                float r[EPL];
#pragma unroll
                for (int j = 0; j < EPL; ++j) r[j] = rv[i][j] + rs * (dv[i][j] - s1 - xv[i][j] * s2);
#pragma unroll
                for (int j = 0; j < EPL; j += 4) st4(dx + row * C + k + j, make_float4(r[j], r[j + 1], r[j + 2], r[j + 3]));
            }
        }
    }
    // combine the row sub-groups of the warp, then the block, then one atomic per column
    __shared__ float sg[1024], sb[1024];
    for (int i = threadIdx.x; i < C; i += blockDim.x) { sg[i] = 0.f; sb[i] = 0.f; }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int k = (gl + i * G) * EPL;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            float gv = gacc[i][j], bv = bacc[i][j];
#pragma unroll
            for (int o = G; o < 32; o <<= 1) { gv += __shfl_xor_sync(0xffffffffu, gv, o); bv += __shfl_xor_sync(0xffffffffu, bv, o); }
            if (sub == 0 && k < C) { atomicAdd(&sg[k + j], gv); atomicAdd(&sb[k + j], bv); }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        atomicAdd(dgamma + i, sg[i]);
        atomicAdd(dbeta + i, sb[i]);
    }
}

template <typename T>
cudaError_t launch_ln_bwd(const T* dz, const T* x, const T* dres, T* dx, const float* gamma, float* dgamma,
                          float* dbeta, long long rows, int C, int num_sms, cudaStream_t st) {
    constexpr int EPL = 16 / sizeof(T);
    const int chunks = C / EPL;
    auto go = [&](auto gtag, auto vtag) -> cudaError_t {
        constexpr int G = decltype(gtag)::value, MAXV = decltype(vtag)::value;
        long long blocks = (rows + 8 * (32 / G) - 1) / (8 * (32 / G));
        const long long cap = static_cast<long long>(num_sms) * 8;
        if (blocks > cap) blocks = cap;
        ln_bwd_kernel<T, G, MAXV><<<static_cast<unsigned>(blocks), 256, 0, st>>>(dz, x, dres, dx, gamma, dgamma, dbeta, rows, C);
        return cudaGetLastError();
    };
    using std::integral_constant;
    if (C > 1024 || chunks > 128) return cudaErrorInvalidValue;
    if (chunks <= 4) return go(integral_constant<int, 4>{}, integral_constant<int, 1>{});
    if (chunks <= 8) return go(integral_constant<int, 8>{}, integral_constant<int, 1>{});
    if (chunks <= 16) return go(integral_constant<int, 16>{}, integral_constant<int, 1>{});
    if (chunks <= 32) return go(integral_constant<int, 32>{}, integral_constant<int, 1>{});
    if (chunks <= 64) return go(integral_constant<int, 32>{}, integral_constant<int, 2>{});
    return go(integral_constant<int, 32>{}, integral_constant<int, 4>{});
}

// ------------------------------------------------------------------------------ depthwise conv backward
// Inputs: g2 = d(h2) (gradient after the second GELU), a2 (pre-GELU conv output), h1 (conv input), a1 (pre-GELU
// linear1 output).  Outputs: da1 = (conv^T(da2)) * gelu'(a1) with da2 = g2 * gelu'(a2);  dWdw, dbdw accumulated.
// Block = 32 channel-groups (128 channels) x 8 pixel lanes; persistent over (b, slab, strip) work items so that the
// weight-gradient partials stay in registers and are flushed once per block.
template <typename T>
__global__ void __launch_bounds__(256) dwconv_bwd_kernel(const T* __restrict__ g2, const T* __restrict__ a2,
                                                         const T* __restrict__ h1, const T* __restrict__ a1,
                                                         T* __restrict__ da1, const float* __restrict__ w,
                                                         float* __restrict__ dw, float* __restrict__ dbias,
                                                         int B, int H, int W, int Ch) {
    const int cgl = threadIdx.x & 31;          // channel group within the slab
    const int pl = threadIdx.x >> 5;           // pixel lane 0..7
    constexpr int STRIP = 16;                  // rows per work item
    const int slabs = (Ch + 127) / 128;
    const int xgroups = (W + 7) / 8;
    const int strips = (H + STRIP - 1) / STRIP;
    const long long per_slab = static_cast<long long>(B) * xgroups * strips;
    const long long items = per_slab * slabs;       // slab-major: a CTA's item sequence is monotone in the slab index
    __shared__ float red[8][32][41];

    float wacc[4][9], bacc[4];
    int cur_slab = -1;
    float wk[4][9];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        bacc[i] = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) { wacc[i][t] = 0.f; wk[i][t] = 0.f; }
    }
    auto flush = [&](int slab) {
        // reduce the 8 pixel lanes, then one atomic per (channel, tap)
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int t = 0; t < 9; ++t) red[pl][cgl][i * 9 + t] = wacc[i][t];
            red[pl][cgl][36 + i] = bacc[i];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < 32 * 40; e += 256) {
            const int cg = e / 40, j = e % 40;
            float s = 0.f;
#pragma unroll
            for (int p = 0; p < 8; ++p) s += red[p][cg][j];
            const int c = slab * 128 + cg * 4 + (j < 36 ? j / 9 : j - 36);
            if (c < Ch) {
                if (j < 36) atomicAdd(dw + c * 9 + (j % 9), s);
                else atomicAdd(dbias + c, s);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            bacc[i] = 0.f;
#pragma unroll
            for (int t = 0; t < 9; ++t) wacc[i][t] = 0.f;
        }
    };

    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int slab = static_cast<int>(item / per_slab);
        long long rest = item - slab * per_slab;
        const int xg = static_cast<int>(rest % xgroups);
        rest /= xgroups;
        const int strip = static_cast<int>(rest % strips);
        const int b = static_cast<int>(rest / strips);
        const int ys = strip * STRIP, ye = min(ys + STRIP, H);
        if (slab != cur_slab) {
            if (cur_slab >= 0) flush(cur_slab);
            cur_slab = slab;
            const int c = slab * 128 + cgl * 4;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int t = 0; t < 9; ++t) wk[i][t] = (c + i < Ch) ? __ldg(w + (c + i) * 9 + t) : 0.f;
        }
        const int c = slab * 128 + cgl * 4;
        const int xx = xg * 8 + pl;
        if (c >= Ch || xx >= W) continue;
        const long long base = static_cast<long long>(b) * H * W * Ch + c;
        auto ld_da2 = [&](int y, int xq) -> float4 {       // da2 = g2 * gelu'(a2), zero outside the map
            if (y < 0 || y >= H || xq < 0 || xq >= W) return make_float4(0.f, 0.f, 0.f, 0.f);
            const long long o = base + (static_cast<long long>(y) * W + xq) * Ch;
            float4 gv = ld4(g2 + o);
            const float4 p = ld4(a2 + o);
            gv.x *= gelu_erf_grad(p.x); gv.y *= gelu_erf_grad(p.y); gv.z *= gelu_erf_grad(p.z); gv.w *= gelu_erf_grad(p.w);
            return gv;
        };
        auto ld_h1 = [&](int y, int xq) -> float4 {
            if (y < 0 || y >= H || xq < 0 || xq >= W) return make_float4(0.f, 0.f, 0.f, 0.f);
            return ld4(h1 + base + (static_cast<long long>(y) * W + xq) * Ch);
        };
        float4 dwin[3][3];      // da2 at rows y-1..y+1, cols x-1..x+1
#pragma unroll
        for (int j = 0; j < 3; ++j) { dwin[0][j] = ld_da2(ys - 1, xx - 1 + j); dwin[1][j] = ld_da2(ys, xx - 1 + j); }
        for (int y = ys; y < ye; ++y) {
#pragma unroll
            for (int j = 0; j < 3; ++j) dwin[2][j] = ld_da2(y + 1, xx - 1 + j);
            // data gradient: dh1[y,x] = sum_{ky,kx} da2[y-ky+1, x-kx+1] * w[ky,kx]
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float4 v = dwin[2 - ky][2 - kx];
                    acc.x = fmaf(v.x, wk[0][ky * 3 + kx], acc.x);
                    acc.y = fmaf(v.y, wk[1][ky * 3 + kx], acc.y);
                    acc.z = fmaf(v.z, wk[2][ky * 3 + kx], acc.z);
                    acc.w = fmaf(v.w, wk[3][ky * 3 + kx], acc.w);
                }
            const long long o = base + (static_cast<long long>(y) * W + xx) * Ch;
            const float4 p1 = ld4(a1 + o);
            acc.x *= gelu_erf_grad(p1.x); acc.y *= gelu_erf_grad(p1.y);
            acc.z *= gelu_erf_grad(p1.z); acc.w *= gelu_erf_grad(p1.w);
            st4(da1 + o, acc);
            // weight gradient: dw[ky,kx] += da2[y,x] * h1[y+ky-1, x+kx-1]
            const float4 d = dwin[1][1];
            bacc[0] += d.x; bacc[1] += d.y; bacc[2] += d.z; bacc[3] += d.w;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float4 hv = ld_h1(y + ky - 1, xx + kx - 1);
                    wacc[0][ky * 3 + kx] = fmaf(d.x, hv.x, wacc[0][ky * 3 + kx]);
                    wacc[1][ky * 3 + kx] = fmaf(d.y, hv.y, wacc[1][ky * 3 + kx]);
                    wacc[2][ky * 3 + kx] = fmaf(d.z, hv.z, wacc[2][ky * 3 + kx]);
                    wacc[3][ky * 3 + kx] = fmaf(d.w, hv.w, wacc[3][ky * 3 + kx]);
                }
#pragma unroll
            for (int j = 0; j < 3; ++j) { dwin[0][j] = dwin[1][j]; dwin[1][j] = dwin[2][j]; }
        }
    }
    if (cur_slab >= 0) flush(cur_slab);
}

template <typename T>
cudaError_t launch_dwconv_bwd(const T* g2, const T* a2, const T* h1, const T* a1, T* da1, const float* w, float* dw,
                              float* dbias, int B, int H, int W, int Ch, int num_sms, cudaStream_t st) {
    const long long items = static_cast<long long>(B) * ((Ch + 127) / 128) * ((W + 7) / 8) * ((H + 15) / 16);
    long long grid = static_cast<long long>(num_sms) * 8;
    if (grid > items) grid = items;
    dwconv_bwd_kernel<T><<<static_cast<unsigned>(grid), 256, 0, st>>>(g2, a2, h1, a1, da1, w, dw, dbias, B, H, W, Ch);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------ ProbSparse core backward
// head_dim D in {32, 64, 128} (see CoreLd in probsparse_core.cuh)
template <int D>
struct CoreBwdSmem {
    float q[kTok * CoreLd<D>::QK];
    float k[kTok * CoreLd<D>::QK];
    float v[kTok * CoreLd<D>::QK];
    float dc[kTok * CoreLd<D>::QK];       // dctx tile
    float p1[32 * P_LD];
    float p2[32 * P_LD];
    float ds[32 * P_LD];          // dP2, then dS (scaled)
    float tbl[232];
    float tacc[16 * 225];         // d(rpb table) partials per head
    float dmean[D];
    float dpart[4 * D];
    int tok_of[32];
    int slot_of[kTok];
    int region[kTok];
};

template <typename T, int D>
__global__ void __launch_bounds__(CORE_THREADS) probsparse_core_bwd_kernel(const CoreBwdArgs<T> a) {
    constexpr int PASSES = Act<T>::kPasses;
    constexpr int QK_LD = CoreLd<D>::QK;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CoreBwdSmem<D>& s = *reinterpret_cast<CoreBwdSmem<D>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int C3 = 3 * a.C;
    const float scale = rsqrtf(static_cast<float>(D));
    const bool want_tab = a.d_rpb_table != nullptr && a.use_rpb;
    const bool want_dense = a.d_rpb_dense != nullptr && a.use_rpb;
    for (int i = tid; i < 16 * 225; i += CORE_THREADS) s.tacc[i] = 0.f;

    const int items = a.B_ * a.nH;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int wg = item / a.nH;
        const int h = item - wg * a.nH;
        __syncthreads();
        {   // stage q, k, v, dctx
            const T* base = a.qkv + static_cast<long long>(wg) * kTok * C3 + h * D;
            const T* dbase = a.dctx + static_cast<long long>(wg) * kTok * a.C + h * D;
            constexpr int CPR = D / 4;
            for (int c = tid; c < 4 * kTok * CPR; c += CORE_THREADS) {
                const int which = c / (kTok * CPR);
                const int rem = c - which * kTok * CPR;
                const int r = rem / CPR, d4 = (rem % CPR) * 4;
                float4 v;
                if (which < 3) v = ld4(base + static_cast<long long>(r) * C3 + which * a.C + d4);
                else v = ld4(dbase + static_cast<long long>(r) * a.C + d4);
                float* dst = (which == 0 ? s.q : which == 1 ? s.k : which == 2 ? s.v : s.dc) + r * QK_LD + d4;
                *reinterpret_cast<float4*>(dst) = v;
            }
            if (a.use_rpb && a.rpb_table)
                for (int i = tid; i < 225; i += CORE_THREADS) s.tbl[i] = a.rpb_table[i * a.nH + h];
            if (tid < kTok) s.slot_of[tid] = -1;
            if (a.shift > 0 && tid < kTok) {
                int w = wg % a.nWin;
                int wy = w / a.nWw, wx = w - wy * a.nWw;
                int y = wy * 8 + (tid >> 3), x = wx * 8 + (tid & 7);
                int rb = y < a.H - 8 ? 0 : (y < a.H - a.shift ? 1 : 2);
                int cb = x < a.W - 8 ? 0 : (x < a.W - a.shift ? 1 : 2);
                s.region[tid] = rb * 3 + cb;
            }
        }
        __syncthreads();
        if (tid < 32) {
            const int t = tid < kTopU ? a.top[static_cast<long long>(item) * kTopU + tid] : -1;
            s.tok_of[tid] = t;
            if (t >= 0) s.slot_of[t] = tid;
        }
        __syncthreads();

        // ---- S_sel = Q[top] K^T * scale   (32 x 64 x D): warp -> m-tile (warp&1), n-tiles 4*(warp>>1)..+3
        const int mt = warp & 1, nb4 = (warp >> 1) * 4;
        {
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
            const int t0 = s.tok_of[mt * 16 + gq], t1 = s.tok_of[mt * 16 + gq + 8];
            const float* q0 = s.q + (t0 < 0 ? 0 : t0) * QK_LD;
            const float* q1 = s.q + (t1 < 0 ? 0 : t1) * QK_LD;
#pragma unroll
            for (int ks = 0; ks < D / 8; ++ks) {
                float af[4] = {q0[ks * 8 + tq], q1[ks * 8 + tq], q0[ks * 8 + tq + 4], q1[ks * 8 + tq + 4]};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float* pb = s.k + ((nb4 + j) * 8 + gq) * QK_LD + ks * 8 + tq;
                    float bf[2] = {pb[0], pb[4]};
                    mma_x<PASSES>(acc[j], af, bf);
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float2 v2;
                    v2.x = Act<T>::round(Act<T>::round(acc[j][half * 2]) * scale);
                    v2.y = Act<T>::round(Act<T>::round(acc[j][half * 2 + 1]) * scale);
                    *reinterpret_cast<float2*>(s.p1 + (mt * 16 + gq + half * 8) * P_LD + (nb4 + j) * 8 + 2 * tq) = v2;
                }
        }
        // sum of dctx over the NON-selected rows / 64 (gradient of the mean(V) fill, attn.py:168-172)
        for (int e = tid; e < 4 * D; e += CORE_THREADS) {
            const int d = e % D, part = e / D;
            float sum = 0.f;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int row = part * 16 + r;
                if (s.slot_of[row] < 0) sum += s.dc[row * QK_LD + d];
            }
            s.dpart[part * D + d] = sum;
        }
        __syncthreads();
        for (int d = tid; d < D; d += CORE_THREADS)
            s.dmean[d] = (s.dpart[d] + s.dpart[D + d] + s.dpart[2 * D + d] + s.dpart[3 * D + d]) * (1.0f / kTok);

        // ---- recompute P1, P2 (attn.py:195-264)
        for (int slot = warp; slot < 32; slot += 4) {
            float* r1 = s.p1 + slot * P_LD;
            float* r2 = s.p2 + slot * P_LD;
            if (slot >= kTopU) { r1[lane] = 0.f; r1[lane + 32] = 0.f; r2[lane] = 0.f; r2[lane + 32] = 0.f; continue; }
            const int r = s.tok_of[slot];
            float x0 = r1[lane], x1 = r1[lane + 32];
            float mx = group_max<32>(fmaxf(x0, x1));
            float e0 = expf(x0 - mx), e1 = expf(x1 - mx);
            float inv = 1.0f / group_sum<32>(e0 + e1);
            float p0 = e0 * inv, p1v = e1 * inv;
            r1[lane] = p0; r1[lane + 32] = p1v;
            if (a.use_rpb) {
                if (a.rpb_table) {
                    const int ry = r >> 3, rx = r & 7;
                    p0 += s.tbl[(ry - (lane >> 3) + 7) * 15 + (rx - (lane & 7) + 7)];
                    p1v += s.tbl[(ry - ((lane + 32) >> 3) + 7) * 15 + (rx - (lane & 7) + 7)];
                } else {
                    const float* brow = a.rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok;
                    p0 += brow[lane]; p1v += brow[lane + 32];
                }
            }
            if (a.mask) {
                const float* mrow = a.mask + (static_cast<long long>(wg % a.nW_mask) * kTok + r) * kTok;
                p0 += mrow[lane]; p1v += mrow[lane + 32];
            }
            if (a.shift > 0) {
                const int rr = s.region[r];
                p0 += (s.region[lane] != rr) ? -100.0f : 0.f;
                p1v += (s.region[lane + 32] != rr) ? -100.0f : 0.f;
            }
            mx = group_max<32>(fmaxf(p0, p1v));
            e0 = expf(p0 - mx); e1 = expf(p1v - mx);
            inv = 1.0f / group_sum<32>(e0 + e1);
            r2[lane] = Act<T>::round(e0 * inv);
            r2[lane + 32] = Act<T>::round(e1 * inv);
        }
        __syncthreads();

        // ---- dP2 = dctx[top] V^T  (32 x 64 x D)
        {
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
            const int t0 = s.tok_of[mt * 16 + gq], t1 = s.tok_of[mt * 16 + gq + 8];
            const float* d0 = s.dc + (t0 < 0 ? 0 : t0) * QK_LD;
            const float* d1 = s.dc + (t1 < 0 ? 0 : t1) * QK_LD;
            const float z0 = t0 < 0 ? 0.f : 1.f, z1 = t1 < 0 ? 0.f : 1.f;
#pragma unroll
            for (int ks = 0; ks < D / 8; ++ks) {
                float af[4] = {d0[ks * 8 + tq] * z0, d1[ks * 8 + tq] * z1, d0[ks * 8 + tq + 4] * z0, d1[ks * 8 + tq + 4] * z1};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float* pb = s.v + ((nb4 + j) * 8 + gq) * QK_LD + ks * 8 + tq;
                    float bf[2] = {pb[0], pb[4]};
                    mma_x<PASSES>(acc[j], af, bf);
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<float2*>(s.ds + (mt * 16 + gq + half * 8) * P_LD + (nb4 + j) * 8 + 2 * tq) =
                        make_float2(acc[j][half * 2], acc[j][half * 2 + 1]);
        }
        __syncthreads();

        // ---- softmax backward twice: dA = P2 * (dP2 - <dP2,P2>); d(bias) += dA; dS = P1 * (dA - <dA,P1>) * scale
        for (int slot = warp; slot < 32; slot += 4) {
            float* rd = s.ds + slot * P_LD;
            if (slot >= kTopU) { rd[lane] = 0.f; rd[lane + 32] = 0.f; continue; }
            const int r = s.tok_of[slot];
            const float* r1 = s.p1 + slot * P_LD;
            const float* r2 = s.p2 + slot * P_LD;
            const float g0 = rd[lane], g1 = rd[lane + 32];
            const float q0 = r2[lane], q1 = r2[lane + 32];
            float dot = group_sum<32>(g0 * q0 + g1 * q1);
            const float da0 = q0 * (g0 - dot), da1 = q1 * (g1 - dot);
            if (want_tab && a.rpb_table) {
                const int ry = r >> 3, rx = r & 7;
                atomicAdd(&s.tacc[h * 225 + (ry - (lane >> 3) + 7) * 15 + (rx - (lane & 7) + 7)], da0);
                atomicAdd(&s.tacc[h * 225 + (ry - ((lane + 32) >> 3) + 7) * 15 + (rx - (lane & 7) + 7)], da1);
            }
            if (want_dense) {       // gradient w.r.t. the gathered bias [nH, 64, 64] (AttentionLayer.forward's argument, attn.py:385)
                float* drow = a.d_rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok;
                atomicAdd(drow + lane, da0);
                atomicAdd(drow + lane + 32, da1);
            }
            const float p0 = r1[lane], p1v = r1[lane + 32];
            dot = group_sum<32>(da0 * p0 + da1 * p1v);
            rd[lane] = p0 * (da0 - dot) * scale;
            rd[lane + 32] = p1v * (da1 - dot) * scale;
        }
        __syncthreads();

        T* obase = a.dqkv + static_cast<long long>(wg) * kTok * C3 + h * D;
        // ---- dq[top] = dS K  (32 x D x 64): warp -> m-tile (warp&1), D/16 n-tiles ; other rows zero
        {
            constexpr int NT = D / 16;
            const int nb2 = (warp >> 1) * NT;
            float o[NT][4];
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) o[j][c] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                const float* pa = s.ds + (mt * 16 + gq) * P_LD + ks * 8 + tq;
                float af[4] = {pa[0], pa[8 * P_LD], pa[4], pa[8 * P_LD + 4]};
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    const float* pb = s.k + (ks * 8 + tq) * QK_LD + (nb2 + j) * 8 + gq;
                    float bf[2] = {pb[0], pb[4 * QK_LD]};
                    mma_x<PASSES>(o[j], af, bf);
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = s.tok_of[mt * 16 + gq + half * 8];
                if (r >= 0) {
#pragma unroll
                    for (int j = 0; j < NT; ++j)
                        st2(obase + static_cast<long long>(r) * C3 + (nb2 + j) * 8 + 2 * tq, o[j][half * 2], o[j][half * 2 + 1]);
                }
            }
            for (int c = tid; c < kTok * (D / 4); c += CORE_THREADS) {
                const int r = c / (D / 4), d4 = (c % (D / 4)) * 4;
                if (s.slot_of[r] < 0) st4(obase + static_cast<long long>(r) * C3 + d4, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        }
        // ---- dK = dS^T Q[top] ; dV = P2^T dctx[top] + dmean   (64 x D x 32slots): warp -> m-tile `warp`, 4 n-tiles per pass
#pragma unroll 1
        for (int n0 = 0; n0 < D / 8; n0 += 4) {
            float ok[4][4], ov[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) { ok[j][c] = 0.f; ov[j][c] = 0.f; }
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                // A[m = token][k = slot] = ds[slot][token]  /  p2[slot][token]
                const float* pa = s.ds + (ks * 8 + tq) * P_LD + warp * 16 + gq;
                const float* pp = s.p2 + (ks * 8 + tq) * P_LD + warp * 16 + gq;
                float ak[4] = {pa[0], pa[8], pa[4 * P_LD], pa[4 * P_LD + 8]};
                float av[4] = {pp[0], pp[8], pp[4 * P_LD], pp[4 * P_LD + 8]};
                const int s0 = s.tok_of[ks * 8 + tq], s1 = s.tok_of[ks * 8 + tq + 4];
                const float* qa = s.q + (s0 < 0 ? 0 : s0) * QK_LD;
                const float* qb = s.q + (s1 < 0 ? 0 : s1) * QK_LD;
                const float* da = s.dc + (s0 < 0 ? 0 : s0) * QK_LD;
                const float* db = s.dc + (s1 < 0 ? 0 : s1) * QK_LD;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float bq[2] = {qa[(n0 + j) * 8 + gq], qb[(n0 + j) * 8 + gq]};
                    float bd[2] = {da[(n0 + j) * 8 + gq], db[(n0 + j) * 8 + gq]};
                    mma_x<PASSES>(ok[j], ak, bq);
                    mma_x<PASSES>(ov[j], av, bd);
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = warp * 16 + gq + half * 8;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int d = (n0 + j) * 8 + 2 * tq;
                    st2(obase + static_cast<long long>(r) * C3 + a.C + d, ok[j][half * 2], ok[j][half * 2 + 1]);
                    st2(obase + static_cast<long long>(r) * C3 + 2 * a.C + d, ov[j][half * 2] + s.dmean[d],
                        ov[j][half * 2 + 1] + s.dmean[d + 1]);
                }
            }
        }
    }
    __syncthreads();
    if (want_tab && a.rpb_table) {
        for (int i = tid; i < a.nH * 225; i += CORE_THREADS) {
            const int h = i / 225, rel = i - h * 225;
            const float v = s.tacc[i];
            if (v != 0.f) atomicAdd(a.d_rpb_table + rel * a.nH + h, v);
        }
    }
}

template <typename T, int D>
cudaError_t launch_core_bwd_d(const CoreBwdArgs<T>& a, int num_sms, cudaStream_t stream) {
    auto k = probsparse_core_bwd_kernel<T, D>;
    const size_t smem = sizeof(CoreBwdSmem<D>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    long long items = static_cast<long long>(a.B_) * a.nH;
    const int resident = static_cast<int>((227 * 1024) / (smem + 1024));
    long long cap = static_cast<long long>(num_sms) * (resident < 1 ? 1 : resident > 2 ? 2 : resident) * 2;
    unsigned grid = static_cast<unsigned>(items < cap ? items : cap);
    k<<<grid, CORE_THREADS, smem, stream>>>(a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_core_bwd(const CoreBwdArgs<T>& a, int num_sms, cudaStream_t stream) {
    const int D = a.C / a.nH;
    if (D == 32) {
        if constexpr (Act<T>::kIsBf16) return pcb2::launch(a, num_sms, stream);       // register-resident bf16 path
        else return launch_core_bwd_d<T, 32>(a, num_sms, stream);
    }
    if (D == 64) return launch_core_bwd_d<T, 64>(a, num_sms, stream);
    if (D == 128) return launch_core_bwd_d<T, 128>(a, num_sms, stream);
    return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------ host orchestration
#define BCK(expr)                                           \
    do {                                                    \
        cudaError_t _e = (expr);                            \
        if (_e != cudaSuccess) return static_cast<int>(_e); \
    } while (0)

inline int bw_device(int* sms) {
    int dev = 0, cc = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return LEWIN_E_ARCH;
    cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&cc, cudaDevAttrComputeCapabilityMajor, dev);
    return cc == 10 ? 0 : LEWIN_E_ARCH;
}

inline size_t attn_bwd_ws(const LewinAttnBwdArgs* a, int dtype) {
    const LewinAttnFwdArgs& f = a->fwd;
    const size_t tokens = static_cast<size_t>(f.B) * f.H * f.W;
    const size_t es = dtype == LEWIN_DTYPE_BF16 ? 2 : 4;
    const size_t C = f.C;
    return 2 * bw_align(tokens * 4) + bw_align(tokens * C * es) + bw_align(tokens * 3 * C * es) +
           bw_align(tokens * C * es) + bw_align(C * C * 4) + bw_align(3 * C * C * 4) +
           (dtype == LEWIN_DTYPE_BF16 ? bw_align(3 * C * C * 2) + bw_align(C * C * 2) + bw_align(tokens * C * 2) : 0);
           // bf16: images of W_qkv^T / W_out^T and the scaled, window-ordered dy rows for the streamed-W GEMMs
}

// Data-gradient GEMM dX = dY . W (W^T staged as the [N, K] operand).  bf16 at the C >= 256 levels: the forward's
// warp-specialised streamed-W tcgen05 kernel (TMA operands, 3x the first-generation kernel's rate) whenever the operand
// needs no row gather / row scale; `wT_bf16` is workspace for the bf16 image of the transposed weight.
// out[m, :] = bf16(scale[row / tokens_per_image] * in[row, :]),  row = window-order source token of m (mapped) or m:
// the DropPath scale and the roll + window_partition gather of a data-gradient GEMM's A operand as a pre-pass, so that the
// GEMM itself can stream plain rows by TMA (same rounding point as the in-GEMM prologue of gemm_tc.cuh).
__global__ void __launch_bounds__(256) scale_gather_rows_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                                const float* __restrict__ scale, long long rows, int C, int lda,
                                                                int mapped, WinMap map, int tokens_per_image) {
    const int cpr = C / 8;                                  // 16-byte chunks per row
    const long long total = rows * cpr;
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * 256) {
        const long long m = i / cpr;
        const int ch = static_cast<int>(i - m * cpr);
        const long long row = mapped ? static_cast<long long>(map.token32(static_cast<uint32_t>(m))) : m;
        uint4 v = *reinterpret_cast<const uint4*>(in + row * lda + ch * 8);
        if (scale) {
            const float sc = scale[row / tokens_per_image];
            __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 t2 = __bfloat1622float2(h[j]);
                h[j] = __floats2bfloat162_rn(t2.x * sc, t2.y * sc);
            }
        }
        *reinterpret_cast<uint4*>(out + m * C + ch * 8) = v;
    }
}

// window-ordered / DropPath-scaled copy of [M, K] bf16 rows (one pass), so that a TMA-fed kernel can stream plain rows
inline cudaError_t launch_scale_gather_rows(const __nv_bfloat16* A, __nv_bfloat16* out, const float* row_scale, long long M, int K,
                                            long long lda, int mapA, const WinMap& map, int tokens_per_image, int sms, cudaStream_t st) {
    const long long chunks = M * (K / 8);
    long long grid = (chunks + 255) / 256;
    if (grid > static_cast<long long>(sms) * 16) grid = static_cast<long long>(sms) * 16;
    scale_gather_rows_kernel<<<static_cast<unsigned>(grid), 256, 0, st>>>(A, out, row_scale, M, K, lda, mapA, map, tokens_per_image);
    return cudaGetLastError();
}

template <typename T>
inline cudaError_t launch_dgrad_gemm(const GemmArgs<T>& g, __nv_bfloat16* wT_bf16, int sms, cudaStream_t st,
                                     __nv_bfloat16* a_scratch = nullptr, bool* scratch_filled = nullptr) {
    if constexpr (Act<T>::kIsBf16) {
        constexpr int min_dim = 128;
        GemmArgs<T> h = g;
        const bool prepass = (g.mapA || g.a_row_scale) && a_scratch && !g.mean && g.K % 8 == 0 && g.M < (1ll << 31);
        if (prepass) { h.A = a_scratch; h.lda = g.K; h.mapA = 0; h.a_row_scale = nullptr; }
        const bool big = wT_bf16 && g.K >= min_dim && g.N >= min_dim && ws::wss_supported(h);   // streamed-W tcgen05 kernel
        const bool small = !big && ws::plain_supported(h);                                      // resident-W warp-specialised kernel
        if (big || small) {
            if (prepass) {
                cudaError_t e = launch_scale_gather_rows(g.A, a_scratch, g.a_row_scale, g.M, g.K, g.lda, g.mapA, g.map,
                                                         g.tokens_per_image, sms, st);
                if (e != cudaSuccess) return e;
                if (scratch_filled) *scratch_filled = true;   // [M, K] rows with the gather / DropPath scale applied
            }
            if (small) return ws::launch_plain(h, sms, st);
            cudaError_t e = launch_convert_w(g.Wt, wT_bf16, static_cast<long long>(g.N) * g.K, st);
            if (e != cudaSuccess) return e;
            return ws::wss_launch<EPI_BIAS>(h, wT_bf16, sms, st);
        }
    }
    return launch_gemm_any<T, EPI_BIAS>(g, st);
}

template <typename T>
int attn_bwd(const LewinAttnBwdArgs* a, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (!a || !a->dy || !a->dx) return LEWIN_E_NULL;
    const LewinAttnFwdArgs& f = a->fwd;
    if (!f.x || !f.w_qkv || !f.w_out || !f.qkv || !f.ctx || !f.top) return LEWIN_E_NULL;
    if (!a->d_w_qkv || !a->d_b_qkv || !a->d_w_out || !a->d_b_out) return LEWIN_E_NULL;
    if (!f.windowed && (!f.ln_w || !f.ln_b || !a->d_ln_w || !a->d_ln_b)) return LEWIN_E_NULL;
    if (f.H % 8 || f.W % 8 || f.C % 32 || !head_dim_ok(f.C, f.nH) || f.C > 512 || f.nH > 16) return LEWIN_E_SHAPE;
    int sms = 0;
    if (int rc = bw_device(&sms)) return rc;
    const int dtype = Act<T>::kIsBf16 ? LEWIN_DTYPE_BF16 : LEWIN_DTYPE_F32;
    if (!ws || ws_bytes < attn_bwd_ws(a, dtype)) return LEWIN_E_WORKSPACE;

    const long long tokens = static_cast<long long>(f.B) * f.H * f.W;
    const int C = f.C, nWin = (f.H / 8) * (f.W / 8), B_ = f.B * nWin;
    const int tpi = f.H * f.W;
    unsigned char* p = static_cast<unsigned char*>(ws);
    float* mean = reinterpret_cast<float*>(p); p += bw_align(tokens * 4);
    float* rstd = reinterpret_cast<float*>(p); p += bw_align(tokens * 4);
    T* dctx = reinterpret_cast<T*>(p); p += bw_align(tokens * C * sizeof(T));
    T* dqkv = reinterpret_cast<T*>(p); p += bw_align(tokens * 3 * C * sizeof(T));
    T* dxh = reinterpret_cast<T*>(p); p += bw_align(tokens * C * sizeof(T));
    float* woT = reinterpret_cast<float*>(p); p += bw_align(static_cast<size_t>(C) * C * 4);
    float* wqkvT = reinterpret_cast<float*>(p); p += bw_align(static_cast<size_t>(3) * C * C * 4);
    __nv_bfloat16* wqkvT_b = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p) : nullptr;
    p += bw_align(static_cast<size_t>(3) * C * C * 2);
    __nv_bfloat16* woT_b = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p) : nullptr;
    p += bw_align(static_cast<size_t>(C) * C * 2);
    __nv_bfloat16* dy_s = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p) : nullptr;

    const T* x = static_cast<const T*>(f.x);
    const T* dy = static_cast<const T*>(a->dy);
    WinMap map{f.H, f.W, f.W / 8, nWin, f.shift, f.shift};
    const int mapped = f.windowed ? 0 : 1;

    // W_out [C(out), C(in)] -> as the [N = in, K = out] operand of dctx = do . W_out
    BCK(launch_transpose(f.w_out, woT, C, C, st));
    BCK(launch_transpose(f.w_qkv, wqkvT, 3 * C, C, st));

    bool dy_s_filled = false;
    {   // dctx = (s_b * gather(dy)) . W_out
        GemmArgs<T> g{};
        g.A = dy; g.lda = C; g.Wt = woT; g.bias = nullptr;
        g.Y = dctx; g.ldy = C; g.M = tokens; g.N = C; g.K = C;
        g.mapA = mapped; g.mapY = 0; g.map = map; g.tokens_per_image = tpi;
        g.a_row_scale = f.windowed ? nullptr : f.drop_scale;
        BCK(launch_dgrad_gemm<T>(g, woT_b, sms, st, dy_s, &dy_s_filled));
    }
    {   // dW_out += do^T ctx ; db_out += colsum(do)
        WgradArgs<T> w{};
        w.dY = dy; w.lddy = C; w.X = static_cast<const T*>(f.ctx); w.ldx = C;
        w.dW = a->d_w_out; w.db = a->d_b_out; w.M = tokens; w.N = C; w.K = C;
        w.mapDY = mapped; w.mapX = 0; w.map = map; w.tokens_per_image = tpi;
        w.dy_row_scale = f.windowed ? nullptr : f.drop_scale;
        if constexpr (Act<T>::kIsBf16) {
            // plain operand for the tcgen05 kernel: the window-ordered, DropPath-scaled rows (left behind by the data-gradient
            // GEMM at C >= 128, made here otherwise)
            WgradArgs<T> v = w;
            v.dY = dy_s; v.mapDY = 0; v.dy_row_scale = nullptr;
            if ((w.mapDY || w.dy_row_scale) && wgrad_tc_supported(v)) {
                if (!dy_s_filled) BCK(launch_scale_gather_rows(dy, dy_s, w.dy_row_scale, tokens, C, C, mapped, map, tpi, sms, st));
                w = v;
            }
        }
        BCK(launch_wgrad<T>(w, sms, st));
    }
    {   // core backward -> dq | dk | dv
        CoreBwdArgs<T> c{};
        c.qkv = static_cast<const T*>(f.qkv); c.dctx = dctx; c.dqkv = dqkv; c.top = f.top;
        c.rpb_table = f.rpb_table; c.rpb_dense = f.rpb_table ? nullptr : f.rpb_dense;
        c.d_rpb_table = a->d_rpb_table;
        c.d_rpb_dense = a->d_rpb_dense;
        c.mask = f.mask; c.nW_mask = f.mask ? f.nW_mask : 1;
        c.B_ = B_; c.nH = f.nH; c.C = C; c.use_rpb = f.use_rpb;
        c.shift = (f.analytic_shift_mask && !f.windowed) ? f.shift : 0;
        c.H = f.H; c.W = f.W; c.nWw = f.W / 8; c.nWin = nWin;
        BCK(launch_core_bwd<T>(c, sms, st));
    }
    {   // dW_qkv += dqkv^T LN1(x)[window order] ; db_qkv += colsum(dqkv)
        WgradArgs<T> w{};
        w.dY = dqkv; w.lddy = 3 * C; w.X = x; w.ldx = C;
        w.dW = a->d_w_qkv; w.db = a->d_b_qkv; w.M = tokens; w.N = 3 * C; w.K = C;
        w.mapDY = 0; w.mapX = mapped; w.map = map; w.tokens_per_image = tpi;
        if (!f.windowed) { w.mean = mean; w.rstd = rstd; w.ln_w = f.ln_w; w.ln_b = f.ln_b; }
        if constexpr (Act<T>::kIsBf16) {
            // LN1 + roll + window_partition in one C-sized pass (into dxh, which is free until the next GEMM writes
            // it), so the weight gradient streams plain rows into the tcgen05 kernel
            WgradArgs<T> v = w;
            v.X = dxh; v.mapX = 0; v.mean = nullptr; v.rstd = nullptr; v.ln_w = nullptr; v.ln_b = nullptr;
            if (!f.windowed && wgrad_tc_supported(v)) {
                BCK(launch_ln_apply(x, dxh, f.ln_w, f.ln_b, tokens, C, 1, map, st));
                w = v;
            }
        }
        if (w.mean) BCK(launch_ln_stats<T>(x, tokens, C, mean, rstd, st));      // only the register-prologue kernels need them
        BCK(launch_wgrad<T>(w, sms, st));
    }
    {   // d(LN1 out) = dqkv . W_qkv, scattered back to token order (window_reverse + un-roll)
        GemmArgs<T> g{};
        g.A = dqkv; g.lda = 3 * C; g.Wt = wqkvT; g.bias = nullptr;
        g.Y = f.windowed ? static_cast<T*>(a->dx) : dxh; g.ldy = C; g.M = tokens; g.N = C; g.K = 3 * C;
        g.mapA = 0; g.mapY = mapped; g.map = map; g.tokens_per_image = tpi;
        BCK(launch_dgrad_gemm<T>(g, wqkvT_b, sms, st));
    }
    if (!f.windowed)   // dx = dy + LN1_bwd(dxh)
        BCK(launch_ln_bwd<T>(dxh, x, dy, static_cast<T*>(a->dx), f.ln_w, a->d_ln_w, a->d_ln_b, tokens, C, sms, st));
    return 0;
}

inline size_t leff_bwd_ws(const LewinLeffBwdArgs* a, int dtype) {
    const LewinLeffFwdArgs& f = a->fwd;
    const size_t tokens = static_cast<size_t>(f.B) * f.H * f.W;
    const size_t es = dtype == LEWIN_DTYPE_BF16 ? 2 : 4;
    const size_t C = f.C, Ch = f.hidden;
    return 2 * bw_align(tokens * 4) + 3 * bw_align(tokens * Ch * es) + bw_align(tokens * C * es) + 2 * bw_align(C * Ch * 4) +
           (dtype == LEWIN_DTYPE_BF16 ? 2 * bw_align(C * Ch * 2) + bw_align(tokens * C * 2) : 0);
           // bf16: images of W2^T, W1^T and the DropPath-scaled dout rows
}

template <typename T>
int leff_bwd(const LewinLeffBwdArgs* a, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (!a || !a->dout || !a->dy) return LEWIN_E_NULL;
    const LewinLeffFwdArgs& f = a->fwd;
    if (!f.y || !f.w1 || !f.w_dw || !f.w2 || !f.h1 || !f.h2 || !f.a1 || !f.a2) return LEWIN_E_NULL;
    if (!a->d_w1 || !a->d_b1 || !a->d_w_dw || !a->d_b_dw || !a->d_w2 || !a->d_b2) return LEWIN_E_NULL;
    if (f.fused && (!f.ln_w || !f.ln_b || !a->d_ln_w || !a->d_ln_b)) return LEWIN_E_NULL;
    if (f.C % 32 || f.hidden % 32 || f.C > 512) return LEWIN_E_SHAPE;
    int sms = 0;
    if (int rc = bw_device(&sms)) return rc;
    const int dtype = Act<T>::kIsBf16 ? LEWIN_DTYPE_BF16 : LEWIN_DTYPE_F32;
    if (!ws || ws_bytes < leff_bwd_ws(a, dtype)) return LEWIN_E_WORKSPACE;

    const long long tokens = static_cast<long long>(f.B) * f.H * f.W;
    const int C = f.C, Ch = f.hidden, tpi = f.H * f.W;
    unsigned char* p = static_cast<unsigned char*>(ws);
    float* mean = reinterpret_cast<float*>(p); p += bw_align(tokens * 4);
    float* rstd = reinterpret_cast<float*>(p); p += bw_align(tokens * 4);
    T* dh2 = reinterpret_cast<T*>(p); p += bw_align(tokens * Ch * sizeof(T));
    T* da1 = reinterpret_cast<T*>(p); p += bw_align(tokens * Ch * sizeof(T));
    T* da2 = reinterpret_cast<T*>(p); p += bw_align(tokens * Ch * sizeof(T));
    T* dz = reinterpret_cast<T*>(p); p += bw_align(tokens * C * sizeof(T));
    float* w2T = reinterpret_cast<float*>(p); p += bw_align(static_cast<size_t>(C) * Ch * 4);
    float* w1T = reinterpret_cast<float*>(p); p += bw_align(static_cast<size_t>(C) * Ch * 4);
    __nv_bfloat16* w2T_b = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p) : nullptr;
    __nv_bfloat16* w1T_b = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p + bw_align(static_cast<size_t>(C) * Ch * 2)) : nullptr;
    __nv_bfloat16* dout_s = Act<T>::kIsBf16 ? reinterpret_cast<__nv_bfloat16*>(p + 2 * bw_align(static_cast<size_t>(C) * Ch * 2)) : nullptr;

    const T* y = static_cast<const T*>(f.y);
    const T* dout = static_cast<const T*>(a->dout);
    const float* dscale = f.fused ? f.drop_scale : nullptr;

    BCK(launch_transpose(f.w2, w2T, C, Ch, st));      // [C, Ch] -> [Ch, C]  (N = Ch, K = C)
    BCK(launch_transpose(f.w1, w1T, Ch, C, st));      // [Ch, C] -> [C, Ch]  (N = C, K = Ch)

    bool dout_s_filled = false;
    {   // dh2 = (s*dout) . W2
        GemmArgs<T> g{};
        g.A = dout; g.lda = C; g.Wt = w2T; g.bias = nullptr;
        g.Y = dh2; g.ldy = Ch; g.M = tokens; g.N = Ch; g.K = C;
        g.tokens_per_image = tpi; g.a_row_scale = dscale;
        BCK(launch_dgrad_gemm<T>(g, w2T_b, sms, st, dout_s, &dout_s_filled));
    }
    {   // dW2 += (s*dout)^T h2 ; db2 += colsum(s*dout)
        WgradArgs<T> w{};
        w.dY = dout; w.lddy = C; w.X = static_cast<const T*>(f.h2); w.ldx = Ch;
        w.dW = a->d_w2; w.db = a->d_b2; w.M = tokens; w.N = C; w.K = Ch;
        w.tokens_per_image = tpi; w.dy_row_scale = dscale;
        if constexpr (Act<T>::kIsBf16) {
            WgradArgs<T> v = w;                  // DropPath-scaled rows: left by the GEMM above at C >= 128, made here otherwise
            v.dY = dout_s; v.dy_row_scale = nullptr;
            if (w.dy_row_scale && wgrad_tc_supported(v)) {
                WinMap nomap{};
                if (!dout_s_filled) BCK(launch_scale_gather_rows(dout, dout_s, dscale, tokens, C, C, 0, nomap, tpi, sms, st));
                w = v;
            }
        }
        BCK(launch_wgrad<T>(w, sms, st));
    }
    // depthwise conv backward: da1 = conv^T(dh2 * gelu'(a2)) * gelu'(a1); dWdw, dbdw
    {
        if (Act<T>::kIsBf16) BCK(launch_gelu_tab_init(st));
        cudaError_t derr = cudaSuccess;
        if (launch_dwconv_bwd_tiled<T>(dh2, static_cast<const T*>(f.a2), static_cast<const T*>(f.h1), static_cast<const T*>(f.a1),
                                       da1, da2, f.w_dw, a->d_w_dw, a->d_b_dw, f.B, f.H, f.W, Ch, sms, st, &derr)) {
            BCK(derr);
        } else {
            BCK(launch_dwconv_bwd<T>(dh2, static_cast<const T*>(f.a2), static_cast<const T*>(f.h1), static_cast<const T*>(f.a1),
                                     da1, f.w_dw, a->d_w_dw, a->d_b_dw, f.B, f.H, f.W, Ch, sms, st));
        }
    }
    {   // dW1 += da1^T LN2(y) ; db1 += colsum(da1)
        WgradArgs<T> w{};
        w.dY = da1; w.lddy = Ch; w.X = y; w.ldx = C;
        w.dW = a->d_w1; w.db = a->d_b1; w.M = tokens; w.N = Ch; w.K = C;
        w.tokens_per_image = tpi;
        if (f.fused) { w.mean = mean; w.rstd = rstd; w.ln_w = f.ln_w; w.ln_b = f.ln_b; }
        if constexpr (Act<T>::kIsBf16) {
            // LN2(y) in one C-sized pass (into dz, free until the next GEMM writes it) -> plain operand for the tcgen05 kernel
            WgradArgs<T> v = w;
            v.X = dz; v.mean = nullptr; v.rstd = nullptr; v.ln_w = nullptr; v.ln_b = nullptr;
            if (f.fused && wgrad_tc_supported(v)) {
                WinMap nomap{};
                BCK(launch_ln_apply(y, dz, f.ln_w, f.ln_b, tokens, C, 0, nomap, st));
                w = v;
            }
        }
        if (w.mean) BCK(launch_ln_stats<T>(y, tokens, C, mean, rstd, st));      // only the register-prologue kernels need them
        BCK(launch_wgrad<T>(w, sms, st));
    }
    {   // dz = da1 . W1
        GemmArgs<T> g{};
        g.A = da1; g.lda = Ch; g.Wt = w1T; g.bias = nullptr;
        g.Y = f.fused ? dz : static_cast<T*>(a->dy); g.ldy = C; g.M = tokens; g.N = C; g.K = Ch;
        g.tokens_per_image = tpi;
        BCK(launch_dgrad_gemm<T>(g, w1T_b, sms, st));
    }
    if (f.fused)   // dy = dout + LN2_bwd(dz)
        BCK(launch_ln_bwd<T>(dz, y, dout, static_cast<T*>(a->dy), f.ln_w, a->d_ln_w, a->d_ln_b, tokens, C, sms, st));
    return 0;
}

}  // namespace lewin
