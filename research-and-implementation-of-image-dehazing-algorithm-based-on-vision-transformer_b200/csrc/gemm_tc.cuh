// tcgen05 (5th-gen tensor core) token GEMM for bf16 activations:  Y = epi( pro(A)[M,K] * W[N,K]^T + bias )
//
// Same contract, prologues and epilogues as gemm_fused_kernel (gemm_fused.cuh), Blackwell-native datapath:
//   * A (tokens) and W (weights) tiles are staged in shared memory in the canonical K-major
//     SWIZZLE_128B / SWIZZLE_64B UMMA layout by the CTA's threads (the LayerNorm + shift/window gather
//     prologue and the fp32->bf16 weight cast happen on the way in, so no TMA descriptor is needed);
//   * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) per 16-wide k-step,
//     accumulating fp32 in TMEM; tcgen05.commit arrives on an mbarrier per smem stage (2-stage ring);
//   * the epilogue reads the accumulator with tcgen05.ld.32x32b (one TMEM lane == one token row per thread),
//     applies bias / exact GELU / DropPath scale + residual and writes bf16 rows (window_reverse + un-shift
//     folded into the row address).
// CTA = 128 threads, one 128 x BN output tile; smem <= 98 KB and TMEM <= 256 columns so two CTAs share an
// SM and overlap each other's load / MMA / epilogue phases.
#pragma once
#include "common.cuh"
#include "tc_helpers.cuh"
#include "gemm_t32_api.h"
#include "gemm_fused.cuh"

#include <cstdlib>

namespace lewin {


constexpr int TC_BM = 128;

constexpr int TC_THREADS_MAX = 256;

// Epilogue shared by the tcgen05 GEMM kernels: thread == TMEM lane == tile row; the two warpgroups (if present) split the
// 32-column chunks.  bias -> {store | bf16 table GELU | DropPath scale + residual} -> 16-byte bf16 row stores.
template <int BN, int EPI, int NWG>
__device__ __forceinline__ void tc_epilogue(const GemmArgs<__nv_bfloat16>& g, uint32_t tmem_d, const long long* offY,
                                            const float* s_bias, const uint16_t* gtab, int n0,
                                            const float* s_rowscale = nullptr) {
    using T = __nv_bfloat16;
    const int tid = threadIdx.x, warp = tid >> 5;
    {
        const int r = (warp & 3) * 32 + (tid & 31);
        const int half = warp >> 2;
        const long long oy = offY[r];
        float sc = 1.f;
        if (EPI == EPI_BIAS_RESID && g.drop_scale && oy >= 0) sc = g.drop_scale[(oy / g.ldy) / g.tokens_per_image];
        const uint32_t lane_addr = tmem_d + (static_cast<uint32_t>((warp & 3) * 32) << 16);
#pragma unroll 1
        for (int c0 = half * 32; c0 < BN; c0 += 32 * NWG) {
            float v[32];
            tc::tmem_ld32(lane_addr + c0, v);
            if (oy < 0) continue;
            if (s_rowscale) {                      // (s * a) . W == s * (a . W): per-row DropPath factor of the A operand
                const float rsc = s_rowscale[r];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] *= rsc;
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += s_bias[c0 + j];
            T* yrow = g.Y + oy + n0 + c0;
            if (EPI == EPI_BIAS_GELU && !g.Y2) {       // inference: bf16 bits in -> table -> bf16 bits out
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    uint32_t q[4];
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        const uint32_t in2 = tc::pack_bf16(v[j + 2 * h], v[j + 2 * h + 1]);
                        q[h] = gelu_bits(gtab, in2 & 0xFFFFu) | (gelu_bits(gtab, in2 >> 16) << 16);
                    }
                    *reinterpret_cast<uint4*>(yrow + j) = make_uint4(q[0], q[1], q[2], q[3]);
                }
                continue;
            } else if (EPI == EPI_BIAS_GELU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = Act<T>::round(v[j]);
                if (g.Y2) {
                    T* prow = g.Y2 + oy + n0 + c0;
#pragma unroll
                    for (int j = 0; j < 32; j += 8)
                        *reinterpret_cast<uint4*>(prow + j) = make_uint4(tc::pack_bf16(v[j], v[j + 1]), tc::pack_bf16(v[j + 2], v[j + 3]),
                                                                         tc::pack_bf16(v[j + 4], v[j + 5]), tc::pack_bf16(v[j + 6], v[j + 7]));
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = gelu_tab(gtab, v[j]);
            } else if (EPI == EPI_BIAS_RESID) {
                const T* rrow = g.R + oy + n0 + c0;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const uint4 rv = *reinterpret_cast<const uint4*>(rrow + j);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float2 t2 = __bfloat1622float2(h[q]);
                        v[j + 2 * q] = t2.x + sc * Act<T>::round(v[j + 2 * q]);
                        v[j + 2 * q + 1] = t2.y + sc * Act<T>::round(v[j + 2 * q + 1]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 32; j += 8)
                *reinterpret_cast<uint4*>(yrow + j) = make_uint4(tc::pack_bf16(v[j], v[j + 1]), tc::pack_bf16(v[j + 2], v[j + 3]),
                                                                 tc::pack_bf16(v[j + 4], v[j + 5]), tc::pack_bf16(v[j + 6], v[j + 7]));
        }
    }
}

template <int BN, int KC, int STAGES, int EPI>
constexpr size_t tc_smem_bytes() {
    return 1024 /*align slack*/ + STAGES * (TC_BM * KC * 2) + STAGES * (BN * KC * 2) + TC_BM * (2 * 8 + 3 * 4) + BN * 4 + 64 +
           (EPI == EPI_BIAS_GELU ? kGeluTabSize * 2 : 0);
}

template <int BN, int KC, int EPI, int TC_THREADS, int STAGES>
__global__ void __launch_bounds__(TC_THREADS, (TC_THREADS == 128 ? (STAGES == 1 ? 4 : 2) : 2)) gemm_tc_kernel(const GemmArgs<__nv_bfloat16> g) {
    using T = __nv_bfloat16;
    constexpr int NWG = TC_THREADS / 128;             // epilogue warpgroups (each warp reads its own 32 TMEM lanes)
    constexpr int CPR = KC / 8;                       // 16-byte chunks per tile row
    constexpr int A_STAGE = TC_BM * KC * 2;
    constexpr int W_STAGE = BN * KC * 2;
    constexpr int TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(TC_BM >> 4) << 24);

    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* As = base;                         // [STAGES][A_STAGE]
    unsigned char* Ws = As + STAGES * A_STAGE;        // [STAGES][W_STAGE]
    long long* offA = reinterpret_cast<long long*>(Ws + STAGES * W_STAGE);
    long long* offY = offA + TC_BM;
    float* s_mean = reinterpret_cast<float*>(offY + TC_BM);
    float* s_rstd = s_mean + TC_BM;
    float* s_ascale = s_rstd + TC_BM;
    float* s_bias = s_ascale + TC_BM;                 // [BN]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(s_bias + BN);   // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 2);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(mbar + 4);          // EPI_BIAS_GELU only
    if (EPI == EPI_BIAS_GELU) gelu_tab_to_smem(gtab, threadIdx.x, TC_THREADS);

    const int tid = threadIdx.x, warp = tid >> 5;
    const long long m0 = static_cast<long long>(blockIdx.x) * TC_BM;
    const int n0 = blockIdx.y * BN;
    const bool has_ln = g.mean != nullptr;

    // ---- one-time setup
    if (tid < TC_BM) {
        const int r = tid;
        const long long m = m0 + r;
        long long oa = -1, oy = -1;
        float mu = 0.f, rs = 1.f, asc = 1.f;
        if (m < g.M) {
            const long long tok = (g.mapA || g.mapY) ? g.map.token(m) : m;
            const long long ra = g.mapA ? tok : m, ry = g.mapY ? tok : m;
            oa = ra * g.lda; oy = ry * g.ldy;
            if (has_ln) { mu = g.mean[ra]; rs = g.rstd[ra]; }
            if (g.a_row_scale) asc = g.a_row_scale[ra / g.tokens_per_image];
        }
        offA[r] = oa; offY[r] = oy; s_mean[r] = mu; s_rstd[r] = rs; s_ascale[r] = asc;
    }
    for (int i = tid; i < BN; i += TC_THREADS) s_bias[i] = g.bias ? Act<T>::round(g.bias[n0 + i]) : 0.f;
    if (tid == 0) {
        tc::mbar_init(&mbar[0], 1);
        tc::mbar_init(&mbar[1], 1);
        tc::fence_barrier_init();
    }
    if (warp == 0) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    // ---- staging helpers (global -> registers -> swizzled smem)
    constexpr int A_CH = TC_BM * CPR / TC_THREADS;    // chunks per thread per stage (4 for KC=64, 2 for KC=32)
    constexpr int W_TOTAL = BN * CPR;
    constexpr int W_CH = (W_TOTAL + TC_THREADS - 1) / TC_THREADS;
    uint4 areg[A_CH];
    uint4 wreg[W_CH];
    auto load_a = [&](int kc) {
#pragma unroll
        for (int i = 0; i < A_CH; ++i) {
            const int c = tid + i * TC_THREADS;
            const int r = c / CPR, ch = c % CPR;
            const long long o = offA[r];
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (o >= 0) {
                const int k = kc * KC + ch * 8;
                v = *reinterpret_cast<const uint4*>(g.A + o + k);
                if (has_ln || g.a_row_scale) {
                    float f[8];
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { float2 t2 = __bfloat1622float2(h[j]); f[2 * j] = t2.x; f[2 * j + 1] = t2.y; }
                    if (g.a_row_scale) {
                        const float asc = s_ascale[r];
#pragma unroll
                        for (int j = 0; j < 8; ++j) f[j] *= asc;
                    }
                    if (has_ln) {
                        const float mu = s_mean[r], rs = s_rstd[r];
                        const float4 w0 = *reinterpret_cast<const float4*>(g.ln_w + k);
                        const float4 w1 = *reinterpret_cast<const float4*>(g.ln_w + k + 4);
                        const float4 b0 = *reinterpret_cast<const float4*>(g.ln_b + k);
                        const float4 b1 = *reinterpret_cast<const float4*>(g.ln_b + k + 4);
                        f[0] = (f[0] - mu) * rs * w0.x + b0.x; f[1] = (f[1] - mu) * rs * w0.y + b0.y;
                        f[2] = (f[2] - mu) * rs * w0.z + b0.z; f[3] = (f[3] - mu) * rs * w0.w + b0.w;
                        f[4] = (f[4] - mu) * rs * w1.x + b1.x; f[5] = (f[5] - mu) * rs * w1.y + b1.y;
                        f[6] = (f[6] - mu) * rs * w1.z + b1.z; f[7] = (f[7] - mu) * rs * w1.w + b1.w;
                    }
                    v.x = tc::pack_bf16(f[0], f[1]); v.y = tc::pack_bf16(f[2], f[3]);
                    v.z = tc::pack_bf16(f[4], f[5]); v.w = tc::pack_bf16(f[6], f[7]);
                }
            }
            areg[i] = v;
        }
    };
    auto load_w = [&](int kc) {
#pragma unroll
        for (int i = 0; i < W_CH; ++i) {
            const int c = tid + i * TC_THREADS;
            if (W_TOTAL % TC_THREADS != 0 && c >= W_TOTAL) break;
            const int r = c / CPR, ch = c % CPR;
            const float* src = g.Wt + static_cast<long long>(n0 + r) * g.K + kc * KC + ch * 8;
            const float4 a = *reinterpret_cast<const float4*>(src);
            const float4 b = *reinterpret_cast<const float4*>(src + 4);
            wreg[i] = make_uint4(tc::pack_bf16(a.x, a.y), tc::pack_bf16(a.z, a.w), tc::pack_bf16(b.x, b.y), tc::pack_bf16(b.z, b.w));
        }
    };
    auto store_stage = [&](int s) {
#pragma unroll
        for (int i = 0; i < A_CH; ++i) {
            const int c = tid + i * TC_THREADS;
            *reinterpret_cast<uint4*>(As + s * A_STAGE + tc::swz_off<KC>(c / CPR, c % CPR)) = areg[i];
        }
#pragma unroll
        for (int i = 0; i < W_CH; ++i) {
            const int c = tid + i * TC_THREADS;
            if (W_TOTAL % TC_THREADS != 0 && c >= W_TOTAL) break;
            *reinterpret_cast<uint4*>(Ws + s * W_STAGE + tc::swz_off<KC>(c / CPR, c % CPR)) = wreg[i];
        }
    };
    auto issue = [&](int kc, int s) {      // one elected thread
        const uint64_t da = tc::make_desc<KC>(tc::smem_u32(As + s * A_STAGE));
        const uint64_t db = tc::make_desc<KC>(tc::smem_u32(Ws + s * W_STAGE));
#pragma unroll
        for (int k16 = 0; k16 < KC / 16; ++k16)
            tc::mma_bf16(tmem_d, da + 2 * k16, db + 2 * k16, IDESC, (kc > 0 || k16 > 0) ? 1u : 0u);
        tc::mma_commit(&mbar[s]);
    };

    const int nk = g.K / KC;
    for (int kc = 0; kc < nk; ++kc) {
        const int s = kc % STAGES;
        load_a(kc);
        load_w(kc);
        if (kc >= STAGES) tc::mbar_wait(&mbar[s], ((kc / STAGES) - 1) & 1);   // MMAs that read stage s have retired
        store_stage(s);
        tc::fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            issue(kc, s);
        }
    }
    tc::mbar_wait(&mbar[(nk - 1) % STAGES], ((nk - 1) / STAGES) & 1);   // the last commit covers every MMA issued
    tc::tc_fence_after();

    // ---- epilogue: thread == TMEM lane == tile row
    tc_epilogue<BN, EPI, NWG>(g, tmem_d, offY, s_bias, gtab, n0);
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

// ------------------------------------------------------------------------------------------------------------------
// Persistent variant for K <= 2*KC (the HBM-heavy levels): the weight tile W[BN x K] is converted once and stays
// resident in shared memory, the CTA walks row tiles (stride gridDim.x) and the global loads of the NEXT tile's A rows
// (with their LayerNorm / gather prologue) are issued before the current tile's accumulator is drained, so DRAM
// latency is hidden behind the TMEM epilogue instead of being exposed once per tile.
template <int BN, int KC, int NKC, int EPI>
constexpr size_t tcp_smem_bytes() {
    return 1024 + NKC * (TC_BM * KC * 2) + NKC * (BN * KC * 2) + 2 * TC_BM * (2 * 8 + 3 * 4) + BN * 4 + 64 +
           (EPI == EPI_BIAS_GELU ? kGeluTabSize * 2 : 0);
}

template <int BN, int KC, int NKC, int EPI>
__global__ void __launch_bounds__(256, 2) gemm_tcp_kernel(const GemmArgs<__nv_bfloat16> g, int row_tiles) {
    using T = __nv_bfloat16;
    constexpr int THREADS = 256;
    constexpr int CPR = KC / 8;
    constexpr int A_CHUNK = TC_BM * KC * 2;
    constexpr int W_CHUNK = BN * KC * 2;
    constexpr int TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(TC_BM >> 4) << 24);
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* As = base;                          // [NKC][A_CHUNK]
    unsigned char* Ws = As + NKC * A_CHUNK;            // [NKC][W_CHUNK] resident
    long long* offA = reinterpret_cast<long long*>(Ws + NKC * W_CHUNK);     // [2][128] double-buffered row info
    long long* offY = offA + 2 * TC_BM;
    float* s_mean = reinterpret_cast<float*>(offY + 2 * TC_BM);
    float* s_rstd = s_mean + 2 * TC_BM;
    float* s_ascale = s_rstd + 2 * TC_BM;
    float* s_bias = s_ascale + 2 * TC_BM;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(s_bias + BN);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 2);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(mbar + 4);
    if (EPI == EPI_BIAS_GELU) gelu_tab_to_smem(gtab, threadIdx.x, THREADS);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int n0 = blockIdx.y * BN;
    const bool has_ln = g.mean != nullptr;

    auto rowinfo = [&](long long tile, int buf) {
        if (tid < TC_BM) {
            const long long m = tile * TC_BM + tid;
            long long oa = -1, oy = -1;
            float mu = 0.f, rs = 1.f, asc = 1.f;
            if (m < g.M) {
                const long long tok = (g.mapA || g.mapY) ? g.map.token(m) : m;
                const long long ra = g.mapA ? tok : m, ry = g.mapY ? tok : m;
                oa = ra * g.lda; oy = ry * g.ldy;
                if (has_ln) { mu = g.mean[ra]; rs = g.rstd[ra]; }
                if (g.a_row_scale) asc = g.a_row_scale[ra / g.tokens_per_image];
            }
            const int o = buf * TC_BM + tid;
            offA[o] = oa; offY[o] = oy; s_mean[o] = mu; s_rstd[o] = rs; s_ascale[o] = asc;
        }
    };
    constexpr int A_CH = TC_BM * CPR / THREADS;
    uint4 areg[NKC][A_CH];
    // raw 16-byte loads only: nothing consumes the registers until store_a, so the loads stay in flight across the
    // mbarrier wait and the whole TMEM epilogue of the previous tile
    auto load_a = [&](int buf) {
#pragma unroll
        for (int kc = 0; kc < NKC; ++kc)
#pragma unroll
            for (int i = 0; i < A_CH; ++i) {
                const int c = tid + i * THREADS;
                const int r = c / CPR, ch = c % CPR;
                const long long o = offA[buf * TC_BM + r];
                areg[kc][i] = o >= 0 ? *reinterpret_cast<const uint4*>(g.A + o + kc * KC + ch * 8) : make_uint4(0u, 0u, 0u, 0u);
            }
    };
    // LayerNorm / row-scale prologue applied on the way into the swizzled smem tile
    auto store_a = [&](int buf) {
#pragma unroll
        for (int kc = 0; kc < NKC; ++kc)
#pragma unroll
            for (int i = 0; i < A_CH; ++i) {
                const int c = tid + i * THREADS;
                const int r = c / CPR, ch = c % CPR;
                uint4 v = areg[kc][i];
                if ((has_ln || g.a_row_scale) && offA[buf * TC_BM + r] >= 0) {
                    const int k = kc * KC + ch * 8;
                    float f[8];
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { float2 t2 = __bfloat1622float2(h[j]); f[2 * j] = t2.x; f[2 * j + 1] = t2.y; }
                    if (g.a_row_scale) {
                        const float asc = s_ascale[buf * TC_BM + r];
#pragma unroll
                        for (int j = 0; j < 8; ++j) f[j] *= asc;
                    }
                    if (has_ln) {
                        const float mu = s_mean[buf * TC_BM + r], rs = s_rstd[buf * TC_BM + r];
                        const float4 w0 = *reinterpret_cast<const float4*>(g.ln_w + k);
                        const float4 w1 = *reinterpret_cast<const float4*>(g.ln_w + k + 4);
                        const float4 b0 = *reinterpret_cast<const float4*>(g.ln_b + k);
                        const float4 b1 = *reinterpret_cast<const float4*>(g.ln_b + k + 4);
                        f[0] = (f[0] - mu) * rs * w0.x + b0.x; f[1] = (f[1] - mu) * rs * w0.y + b0.y;
                        f[2] = (f[2] - mu) * rs * w0.z + b0.z; f[3] = (f[3] - mu) * rs * w0.w + b0.w;
                        f[4] = (f[4] - mu) * rs * w1.x + b1.x; f[5] = (f[5] - mu) * rs * w1.y + b1.y;
                        f[6] = (f[6] - mu) * rs * w1.z + b1.z; f[7] = (f[7] - mu) * rs * w1.w + b1.w;
                    }
                    v.x = tc::pack_bf16(f[0], f[1]); v.y = tc::pack_bf16(f[2], f[3]);
                    v.z = tc::pack_bf16(f[4], f[5]); v.w = tc::pack_bf16(f[6], f[7]);
                }
                *reinterpret_cast<uint4*>(As + kc * A_CHUNK + tc::swz_off<KC>(r, ch)) = v;
            }
    };
    auto issue = [&]() {
#pragma unroll
        for (int kc = 0; kc < NKC; ++kc) {
            const uint64_t da = tc::make_desc<KC>(tc::smem_u32(As + kc * A_CHUNK));
            const uint64_t db = tc::make_desc<KC>(tc::smem_u32(Ws + kc * W_CHUNK));
#pragma unroll
            for (int k16 = 0; k16 < KC / 16; ++k16)
                tc::mma_bf16(*tmem_slot, da + 2 * k16, db + 2 * k16, IDESC, (kc > 0 || k16 > 0) ? 1u : 0u);
        }
        tc::mma_commit(&mbar[0]);
    };

    // ---- one-time setup: bias, barrier, TMEM, resident weight tile
    for (int i = tid; i < BN; i += THREADS) s_bias[i] = g.bias ? Act<T>::round(g.bias[n0 + i]) : 0.f;
    if (tid == 0) { tc::mbar_init(&mbar[0], 1); tc::fence_barrier_init(); }
    if (warp == 0) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    for (int c = tid; c < NKC * BN * CPR; c += THREADS) {
        const int kc = c / (BN * CPR), rem = c - kc * (BN * CPR);
        const int r = rem / CPR, ch = rem % CPR;
        const float* src = g.Wt + static_cast<long long>(n0 + r) * g.K + kc * KC + ch * 8;
        const float4 a4 = *reinterpret_cast<const float4*>(src);
        const float4 b4 = *reinterpret_cast<const float4*>(src + 4);
        *reinterpret_cast<uint4*>(Ws + kc * W_CHUNK + tc::swz_off<KC>(r, ch)) =
            make_uint4(tc::pack_bf16(a4.x, a4.y), tc::pack_bf16(a4.z, a4.w), tc::pack_bf16(b4.x, b4.y), tc::pack_bf16(b4.z, b4.w));
    }
    long long tile = blockIdx.x;
    int buf = 0;
    rowinfo(tile, 0);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    load_a(0);
    store_a(0);
    tc::fence_proxy_async();
    __syncthreads();
    if (tid == 0) { tc::tc_fence_after(); issue(); }
    uint32_t phase = 0;
    while (true) {
        const long long next = tile + gridDim.x;
        const bool has_next = next < row_tiles;
        if (has_next) rowinfo(next, buf ^ 1);
        __syncthreads();
        if (has_next) load_a(buf ^ 1);                 // DRAM loads of the next tile fly during the wait + epilogue
        tc::mbar_wait(&mbar[0], phase);
        phase ^= 1;
        tc::tc_fence_after();
        tc_epilogue<BN, EPI, 2>(g, tmem_d, offY + buf * TC_BM, s_bias, gtab, n0);
        tc::tc_fence_before();
        __syncthreads();                               // accumulator drained, A tile free (its MMAs completed)
        if (!has_next) break;
        store_a(buf ^ 1);
        tc::fence_proxy_async();
        __syncthreads();
        if (tid == 0) { tc::tc_fence_after(); issue(); }
        tile = next;
        buf ^= 1;
    }
    if (warp == 0) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

template <int BN, int KC, int NKC, int EPI>
cudaError_t launch_gemm_tcp(const GemmArgs<__nv_bfloat16>& g, int num_sms, cudaStream_t stream) {
    constexpr size_t smem = tcp_smem_bytes<BN, KC, NKC, EPI>();
    auto k = gemm_tcp_kernel<BN, KC, NKC, EPI>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int row_tiles = static_cast<int>((g.M + TC_BM - 1) / TC_BM);
    const int col_tiles = g.N / BN;
    int gx = (2 * num_sms + col_tiles - 1) / col_tiles;
    if (gx > row_tiles) gx = row_tiles;
    k<<<dim3(gx, col_tiles), 256, smem, stream>>>(g, row_tiles);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------------
// Asynchronous multi-stage variant for the tensor-bound levels (K > 128): both operands are plain bf16 in global
// memory (weights pre-converted once per call by convert_w_kernel, LayerNorm applied by ln_apply_kernel), so every
// 16-byte chunk goes global -> swizzled shared memory with cp.async (no register staging, no conversion in the main
// loop) through a STAGES-deep ring; tcgen05.commit on a per-stage mbarrier releases a stage back to the loaders.
__global__ void convert_w_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ o, long long n) {
    const long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        const float4 v = *reinterpret_cast<const float4*>(w + i);
        *reinterpret_cast<uint2*>(o + i) = make_uint2(tc::pack_bf16(v.x, v.y), tc::pack_bf16(v.z, v.w));
    } else {
        for (long long j = i; j < n; ++j) o[j] = __float2bfloat16_rn(w[j]);
    }
}
inline cudaError_t launch_convert_w(const float* w, __nv_bfloat16* o, long long n, cudaStream_t st) {
    convert_w_kernel<<<static_cast<unsigned>((n / 4 + 255) / 256 + 1), 256, 0, st>>>(w, o, n);
    return cudaGetLastError();
}

// xhat[m] = bf16( LN(x[token(m)]) ) for window-ordered row m (or m itself), C = NI * 256 (the C >= 256 levels): a warp
// normalises R rows at a time - all R x NI 16-byte loads are issued before the first reduction, so a warp keeps R x NI x 512
// bytes in flight instead of 512 (the one-row-per-warp version ran at 2.7 TB/s of the 6.5 the copy roofline allows).
template <int NI, int R>
__global__ void __launch_bounds__(256) ln_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       long long rows, int mapped, WinMap map) {
    constexpr int C = NI * 256;
    const int lane = threadIdx.x & 31;
    const long long m0 = (static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R;
    if (m0 >= rows) return;
    uint4 u[R][NI];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long m = m0 + r < rows ? m0 + r : rows - 1;
        const long long tok = mapped ? map.token(m) : m;
        const __nv_bfloat16* src = x + tok * C;
#pragma unroll
        for (int i = 0; i < NI; ++i) u[r][i] = *reinterpret_cast<const uint4*>(src + (lane + i * 32) * 8);
    }
    float4 g0[NI], g1[NI], b0[NI], b1[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        const int k = (lane + i * 32) * 8;
        g0[i] = *reinterpret_cast<const float4*>(gamma + k); g1[i] = *reinterpret_cast<const float4*>(gamma + k + 4);
        b0[i] = *reinterpret_cast<const float4*>(beta + k); b1[i] = *reinterpret_cast<const float4*>(beta + k + 4);
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        float f[NI][8];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const uint4 v = u[r][i];
            f[i][0] = __uint_as_float(v.x << 16); f[i][1] = __uint_as_float(v.x & 0xFFFF0000u);
            f[i][2] = __uint_as_float(v.y << 16); f[i][3] = __uint_as_float(v.y & 0xFFFF0000u);
            f[i][4] = __uint_as_float(v.z << 16); f[i][5] = __uint_as_float(v.z & 0xFFFF0000u);
            f[i][6] = __uint_as_float(v.w << 16); f[i][7] = __uint_as_float(v.w & 0xFFFF0000u);
#pragma unroll
            for (int j = 0; j < 8; ++j) s += f[i][j];
        }
        const float mu = group_sum<32>(s) / C;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < NI; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) { f[i][j] -= mu; q += f[i][j] * f[i][j]; }
        const float rs = rsqrtf(group_sum<32>(q) / C + 1e-5f);
        if (m0 + r < rows) {
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int k = (lane + i * 32) * 8;
                *reinterpret_cast<uint4*>(out + (m0 + r) * C + k) = make_uint4(
                    tc::pack_bf16(f[i][0] * rs * g0[i].x + b0[i].x, f[i][1] * rs * g0[i].y + b0[i].y),
                    tc::pack_bf16(f[i][2] * rs * g0[i].z + b0[i].z, f[i][3] * rs * g0[i].w + b0[i].w),
                    tc::pack_bf16(f[i][4] * rs * g1[i].x + b1[i].x, f[i][5] * rs * g1[i].y + b1[i].y),
                    tc::pack_bf16(f[i][6] * rs * g1[i].z + b1[i].z, f[i][7] * rs * g1[i].w + b1[i].w));
            }
        }
    }
}
// C in {32, 64, 128}: G = C / 8 lanes per row (one 16-byte load each), 32 / G rows per warp and pass, two passes in flight
template <int G>
__global__ void __launch_bounds__(256) ln_apply_small_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             long long rows, int mapped, WinMap map) {
    constexpr int C = G * 8, RPW = 32 / G;
    const int lane = threadIdx.x & 31, sub = lane / G, gl = lane % G;
    const long long warp_global = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long nwarps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    const float4 g0 = *reinterpret_cast<const float4*>(gamma + gl * 8), g1 = *reinterpret_cast<const float4*>(gamma + gl * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(beta + gl * 8), b1 = *reinterpret_cast<const float4*>(beta + gl * 8 + 4);
    auto fetch = [&](long long m) -> uint4 {
        if (m >= rows) return make_uint4(0u, 0u, 0u, 0u);
        const long long tok = mapped ? static_cast<long long>(map.token32(static_cast<uint32_t>(m))) : m;
        return *reinterpret_cast<const uint4*>(x + tok * C + gl * 8);
    };
    long long m = warp_global * RPW + sub;
    uint4 nxt = fetch(m);
    for (; m - sub < rows; m += nwarps * RPW) {
        const uint4 u = nxt;
        nxt = fetch(m + nwarps * RPW);
        float f[8];
        f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
        f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
        f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xFFFF0000u);
        f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xFFFF0000u);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += f[j];
        const float mu = group_sum<G>(s) / C;
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) { f[j] -= mu; q += f[j] * f[j]; }
        const float rs = rsqrtf(group_sum<G>(q) / C + 1e-5f);
        if (m < rows)
            *reinterpret_cast<uint4*>(out + m * C + gl * 8) = make_uint4(
                tc::pack_bf16(f[0] * rs * g0.x + b0.x, f[1] * rs * g0.y + b0.y), tc::pack_bf16(f[2] * rs * g0.z + b0.z, f[3] * rs * g0.w + b0.w),
                tc::pack_bf16(f[4] * rs * g1.x + b1.x, f[5] * rs * g1.y + b1.y), tc::pack_bf16(f[6] * rs * g1.z + b1.z, f[7] * rs * g1.w + b1.w));
    }
}
// general C <= 1024 (any multiple of 8): one warp per row
__global__ void __launch_bounds__(256) ln_apply_any_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           long long rows, int C, int mapped, WinMap map) {
    const int lane = threadIdx.x & 31;
    const long long m = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= rows) return;
    const long long tok = mapped ? map.token(m) : m;
    const __nv_bfloat16* src = x + tok * C;
    float f[4][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = (lane + i * 32) * 8;
        uint4 u = make_uint4(0u, 0u, 0u, 0u);
        if (k < C) u = *reinterpret_cast<const uint4*>(src + k);
        f[i][0] = __uint_as_float(u.x << 16); f[i][1] = __uint_as_float(u.x & 0xFFFF0000u);
        f[i][2] = __uint_as_float(u.y << 16); f[i][3] = __uint_as_float(u.y & 0xFFFF0000u);
        f[i][4] = __uint_as_float(u.z << 16); f[i][5] = __uint_as_float(u.z & 0xFFFF0000u);
        f[i][6] = __uint_as_float(u.w << 16); f[i][7] = __uint_as_float(u.w & 0xFFFF0000u);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += f[i][j];
    }
    const float mu = group_sum<32>(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = (lane + i * 32) * 8;
        if (k < C) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { f[i][j] -= mu; q += f[i][j] * f[i][j]; }
        }
    }
    const float rs = rsqrtf(group_sum<32>(q) / C + 1e-5f);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = (lane + i * 32) * 8;
        if (k < C) {
            const float4 g0 = *reinterpret_cast<const float4*>(gamma + k), g1 = *reinterpret_cast<const float4*>(gamma + k + 4);
            const float4 b0 = *reinterpret_cast<const float4*>(beta + k), b1 = *reinterpret_cast<const float4*>(beta + k + 4);
            *reinterpret_cast<uint4*>(out + m * C + k) = make_uint4(
                tc::pack_bf16(f[i][0] * rs * g0.x + b0.x, f[i][1] * rs * g0.y + b0.y),
                tc::pack_bf16(f[i][2] * rs * g0.z + b0.z, f[i][3] * rs * g0.w + b0.w),
                tc::pack_bf16(f[i][4] * rs * g1.x + b1.x, f[i][5] * rs * g1.y + b1.y),
                tc::pack_bf16(f[i][6] * rs * g1.z + b1.z, f[i][7] * rs * g1.w + b1.w));
        }
    }
}
inline cudaError_t launch_ln_apply(const __nv_bfloat16* x, __nv_bfloat16* out, const float* gamma, const float* beta,
                                   long long rows, int C, int mapped, const WinMap& map, cudaStream_t st) {
    if (C == 256) {
        ln_apply_kernel<1, 4><<<static_cast<unsigned>((rows + 31) / 32), 256, 0, st>>>(x, out, gamma, beta, rows, mapped, map);
    } else if (C == 512) {
        ln_apply_kernel<2, 4><<<static_cast<unsigned>((rows + 31) / 32), 256, 0, st>>>(x, out, gamma, beta, rows, mapped, map);
    } else if ((C == 32 || C == 64 || C == 128) && rows < (1ll << 31)) {
        long long blocks = (rows + 8 * (256 / C) - 1) / (8 * (256 / C));
        if (blocks > 148 * 16) blocks = 148 * 16;
        const unsigned gb = static_cast<unsigned>(blocks);
        if (C == 32) ln_apply_small_kernel<4><<<gb, 256, 0, st>>>(x, out, gamma, beta, rows, mapped, map);
        else if (C == 64) ln_apply_small_kernel<8><<<gb, 256, 0, st>>>(x, out, gamma, beta, rows, mapped, map);
        else ln_apply_small_kernel<16><<<gb, 256, 0, st>>>(x, out, gamma, beta, rows, mapped, map);
    } else {
        ln_apply_any_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, st>>>(x, out, gamma, beta, rows, C, mapped, map);
    }
    return cudaGetLastError();
}


template <int BN, int STAGES, int EPI>
constexpr size_t tca_smem_bytes() {
    return 1024 + STAGES * (TC_BM * 64 * 2 + BN * 64 * 2) + TC_BM * (2 * 8 + 4) + BN * 4 + 64 + 8 * STAGES +
           (EPI == EPI_BIAS_GELU ? kGeluTabSize * 2 : 0);
}

template <int BN, int STAGES, int EPI>
__global__ void __launch_bounds__(256, (STAGES <= 2 ? 2 : 1)) gemm_tca_kernel(const GemmArgs<__nv_bfloat16> g,
                                                                             const __nv_bfloat16* __restrict__ Wb) {
    using T = __nv_bfloat16;
    constexpr int KC = 64, CPR = 8, THREADS = 256;
    constexpr int A_STAGE = TC_BM * KC * 2, W_STAGE = BN * KC * 2;
    constexpr int TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(TC_BM >> 4) << 24);
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* As = base;
    unsigned char* Ws = As + STAGES * A_STAGE;
    long long* offA = reinterpret_cast<long long*>(Ws + STAGES * W_STAGE);
    long long* offY = offA + TC_BM;
    float* s_rowscale = reinterpret_cast<float*>(offY + TC_BM);
    float* s_bias = s_rowscale + TC_BM;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(s_bias + BN);          // [STAGES]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + STAGES);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(mbar + STAGES + 2);
    if (EPI == EPI_BIAS_GELU) gelu_tab_to_smem(gtab, threadIdx.x, THREADS);

    const int tid = threadIdx.x, warp = tid >> 5;
    const long long m0 = static_cast<long long>(blockIdx.x) * TC_BM;
    const int n0 = blockIdx.y * BN;

    if (tid < TC_BM) {
        const long long m = m0 + tid;
        long long oa = -1, oy = -1;
        float rsc = 1.f;
        if (m < g.M) {
            const long long tok = (g.mapA || g.mapY) ? g.map.token(m) : m;
            const long long ra = g.mapA ? tok : m, ry = g.mapY ? tok : m;
            oa = ra * g.lda; oy = ry * g.ldy;
            if (g.a_row_scale) rsc = g.a_row_scale[ra / g.tokens_per_image];
        }
        offA[tid] = oa; offY[tid] = oy; s_rowscale[tid] = rsc;
    }
    for (int i = tid; i < BN; i += THREADS) s_bias[i] = g.bias ? Act<T>::round(g.bias[n0 + i]) : 0.f;
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < STAGES; ++i) tc::mbar_init(&mbar[i], 1);
        tc::fence_barrier_init();
    }
    if (warp == 0) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    const uint32_t As_u = tc::smem_u32(As), Ws_u = tc::smem_u32(Ws);
    auto load_stage = [&](int kc, int st) {
#pragma unroll
        for (int i = 0; i < TC_BM * CPR / THREADS; ++i) {
            const int c = tid + i * THREADS, r = c >> 3, ch = c & 7;
            const long long o = offA[r];
            cp_async16_z(As_u + st * A_STAGE + tc::swz_off<64>(r, ch), g.A + (o >= 0 ? o : 0) + kc * KC + ch * 8, o >= 0);
        }
#pragma unroll
        for (int i = 0; i < BN * CPR / THREADS; ++i) {
            const int c = tid + i * THREADS, r = c >> 3, ch = c & 7;
            cp_async16_z(Ws_u + st * W_STAGE + tc::swz_off<64>(r, ch), Wb + static_cast<long long>(n0 + r) * g.K + kc * KC + ch * 8, true);
        }
    };
    const int nk = g.K / KC;
#pragma unroll
    for (int p = 0; p < STAGES - 1; ++p) {
        if (p < nk) load_stage(p, p);
        cp_async_commit();
    }
    for (int kc = 0; kc < nk; ++kc) {
        const int st = kc % STAGES;
        const int pre = kc + STAGES - 1;                       // chunk to prefetch into the stage MMA(kc-1) is freeing
        if (pre < nk) {
            const int ps = pre % STAGES;
            if (kc >= 1) tc::mbar_wait(&mbar[ps], ((kc - 1) / STAGES) & 1);
            load_stage(pre, ps);
        }
        cp_async_commit();
        cp_async_wait<STAGES - 1>();                           // chunk kc has landed (this thread's copies)
        tc::fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            const uint64_t da = tc::make_desc<64>(As_u + st * A_STAGE);
            const uint64_t db = tc::make_desc<64>(Ws_u + st * W_STAGE);
#pragma unroll
            for (int k16 = 0; k16 < 4; ++k16) tc::mma_bf16(tmem_d, da + 2 * k16, db + 2 * k16, IDESC, (kc > 0 || k16 > 0) ? 1u : 0u);
            tc::mma_commit(&mbar[st]);
        }
    }
    tc::mbar_wait(&mbar[(nk - 1) % STAGES], ((nk - 1) / STAGES) & 1);
    tc::tc_fence_after();
    tc_epilogue<BN, EPI, 2>(g, tmem_d, offY, s_bias, gtab, n0, s_rowscale);
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

template <int BN, int STAGES, int EPI>
cudaError_t launch_gemm_tca_st(const GemmArgs<__nv_bfloat16>& g, const __nv_bfloat16* Wb, cudaStream_t stream) {
    constexpr size_t smem = tca_smem_bytes<BN, STAGES, EPI>();
    auto k = gemm_tca_kernel<BN, STAGES, EPI>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    dim3 grid(static_cast<unsigned>((g.M + TC_BM - 1) / TC_BM), g.N / BN);
    k<<<grid, 256, smem, stream>>>(g, Wb);
    return cudaGetLastError();
}

// plain-bf16-operand GEMM (K % 64 == 0, no LayerNorm prologue): Wb = bf16 copy of g.Wt; two cp.async stages
template <int EPI>
cudaError_t launch_gemm_tca(const GemmArgs<__nv_bfloat16>& g, const __nv_bfloat16* Wb, cudaStream_t stream) {
    if (g.N % 256 == 0) return launch_gemm_tca_st<256, 2, EPI>(g, Wb, stream);
    if (g.N % 192 == 0) return launch_gemm_tca_st<192, 2, EPI>(g, Wb, stream);
    if (g.N % 128 == 0) return launch_gemm_tca_st<128, 2, EPI>(g, Wb, stream);
    return launch_gemm_tca_st<64, 2, EPI>(g, Wb, stream);
}

template <int BN, int KC, int EPI, int STAGES>
cudaError_t launch_gemm_tc_stages(const GemmArgs<__nv_bfloat16>& g, cudaStream_t stream) {
    constexpr size_t smem = tc_smem_bytes<BN, KC, STAGES, EPI>();
    // narrow tiles: 128-thread CTAs, up to 4 per SM (TMEM 4 x 128 columns) -> more independent load / MMA / epilogue
    // phases in flight; a single k-chunk (K == KC) needs no second smem stage
    constexpr int THREADS = BN <= 128 ? 128 : 256;
    auto k = gemm_tc_kernel<BN, KC, EPI, THREADS, STAGES>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    dim3 grid(static_cast<unsigned>((g.M + TC_BM - 1) / TC_BM), g.N / BN);
    k<<<grid, THREADS, smem, stream>>>(g);
    return cudaGetLastError();
}

inline int tc_num_sms() {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}

template <int BN, int KC, int EPI>
cudaError_t launch_gemm_tc_inst(const GemmArgs<__nv_bfloat16>& g, cudaStream_t stream) {
    if (g.M >= 4 * TC_BM) {
        if (g.K == KC) return launch_gemm_tcp<BN, KC, 1, EPI>(g, tc_num_sms(), stream);
        if (g.K == 2 * KC) return launch_gemm_tcp<BN, KC, 2, EPI>(g, tc_num_sms(), stream);
    }
    if (g.K == KC) return launch_gemm_tc_stages<BN, KC, EPI, 1>(g, stream);
    return launch_gemm_tc_stages<BN, KC, EPI, 2>(g, stream);
}

template <int KC, int EPI>
cudaError_t launch_gemm_tc_kc(const GemmArgs<__nv_bfloat16>& g, cudaStream_t stream) {
    const int N = g.N;
    // wide (192/256-column, 256-thread) tiles measured faster than 128-column / 128-thread tiles on every shape
    if (N % 256 == 0) return launch_gemm_tc_inst<256, KC, EPI>(g, stream);
    if (N % 192 == 0) return launch_gemm_tc_inst<192, KC, EPI>(g, stream);
    if (N % 128 == 0) return launch_gemm_tc_inst<128, KC, EPI>(g, stream);
    if (N % 96 == 0) return launch_gemm_tc_inst<96, KC, EPI>(g, stream);
    if (N % 64 == 0) return launch_gemm_tc_inst<64, KC, EPI>(g, stream);
    return launch_gemm_tc_inst<32, KC, EPI>(g, stream);
}

// bf16 GEMM dispatch: tcgen05 path (N % 32 == 0, K % 32 == 0 always hold for LeWin shapes)
template <int EPI>
cudaError_t launch_gemm_tc(const GemmArgs<__nv_bfloat16>& g, cudaStream_t stream) {
    if (g.K % 64 == 0) return launch_gemm_tc_kc<64, EPI>(g, stream);
    return launch_gemm_tc_kc<32, EPI>(g, stream);
}

// Dispatch used by the ABI: bf16 activations -> tcgen05 kernel; fp32 activations -> 3xTF32 on tcgen05 (gemm_t32.cuh) for
// the forward shapes, the 3xTF32 mma.sync kernel otherwise
template <typename T, int EPI>
cudaError_t launch_gemm_any(const GemmArgs<T>& g, cudaStream_t stream) {
    if constexpr (Act<T>::kIsBf16) {
        return launch_gemm_tc<EPI>(g, stream);
    } else {
        if (gemm_t32_supported(g, EPI)) return gemm_t32_launch(g, EPI, stream);
        return launch_gemm<EPI>(g, stream);
    }
}

}  // namespace lewin
