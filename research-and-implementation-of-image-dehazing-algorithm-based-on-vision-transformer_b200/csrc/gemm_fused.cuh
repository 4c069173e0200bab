// Token GEMM with fused prologue / epilogue:  Y = epi( pro(A)[M,K] * W[N,K]^T + bias )
//
// Serves the four linears of a LeWin block (reference: ProbSparse/attn.py:420-422 q/k/v projections,
// attn.py:456 out projection, My_model_1.py:508 LeFF linear1, :529 LeFF linear2) with what surrounds
// them in the reference folded in:
//   prologue : LayerNorm (My_model_1.py:839/873) from precomputed row stats, cyclic shift +
//              window_partition (My_model_1.py:846-852) as row addressing;
//   epilogue : bias, exact GELU (My_model_1.py:487), DropPath scale + residual (My_model_1.py:872-873),
//              window_reverse + un-shift (My_model_1.py:861-866) as row addressing.
// Tensor cores: mma.sync m16n8k8 TF32, 3-pass error-compensated (fp32-grade accuracy).  fp32 activations only: the bf16
// GEMMs run on tcgen05 (gemm_tc.cuh, gemm_ws.cuh).
#pragma once
#include "common.cuh"

#include <type_traits>

namespace lewin {

enum : int { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RESID = 2, EPI_MUL_GELUGRAD = 3 };

template <typename T>
struct GemmArgs {
    const T* A;           // [rowsA, lda]
    long long lda;
    const float* Wt;      // [N, K] row-major (PyTorch Linear.weight)
    const float* bias;    // [N] or null
    T* Y;                 // [rowsY, ldy]
    T* Y2;                // optional pre-activation copy (EPI_BIAS_GELU), may be null
    long long ldy;
    long long M;
    int N, K;
    // LayerNorm prologue (null mean => plain A)
    const float* mean;    // [M] indexed by A row (token), null => no LN
    const float* rstd;
    const float* ln_w;    // [K]
    const float* ln_b;
    // row addressing
    int mapA, mapY;       // 1: row m is in window order and maps to a token through `map`
    WinMap map;
    // residual epilogue
    const T* R;           // residual rows, indexed like Y with row stride ldr (gemm_ws.cuh kernels; 0 = ldy)
    long long ldr;
    const float* drop_scale;   // [B] or null (EPI_BIAS_RESID: scales the GEMM result per sample)
    int tokens_per_image;
    // backward helpers
    const float* a_row_scale;  // [B] or null: A row (token) is multiplied by a_row_scale[token / tokens_per_image]
    const T* aux;              // EPI_MUL_GELUGRAD: pre-activation, indexed like Y; result = acc * gelu'(aux)
    // pixel-shuffle output addressing of the 2x2 / stride-2 transposed convolution (gemm_ws.cuh only): row m = (b, i, j) of an
    // up_H x up_W map, column block q = col / up_C = 2*di + dj  ->  output token (b, 2i + di, 2j + dj), channel col % up_C
    int up2, up_H, up_W, up_C;
};

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 32;
constexpr int GEMM_LDS = GEMM_BK + 4;   // padded smem row stride (floats): conflict-free fragment loads
constexpr int GEMM_THREADS = 256;

template <int BN>
constexpr size_t gemm_smem_bytes() {
    return sizeof(float) * (2 * GEMM_BM * GEMM_LDS + 2 * BN * GEMM_LDS) + sizeof(long long) * 2 * GEMM_BM +
           sizeof(float) * 4 * GEMM_BM;
}

// T is always float; it stays a template parameter so that the kernel keeps the symbol name the profiles record
template <typename T, int BN, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_fused_kernel(const GemmArgs<T> g) {
    static_assert(std::is_same<T, float>::value, "gemm_fused_kernel serves fp32 activations only");
    constexpr int PASSES = Act<T>::kPasses;
    constexpr int NT = BN / 16;    // n8-tiles per warp (warp covers BN/2 columns)
    constexpr int MT = 2;          // m16-tiles per warp (warp covers 32 rows)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* As = reinterpret_cast<float*>(smem_raw);                       // [2][BM][LDS]
    float* Ws = As + 2 * GEMM_BM * GEMM_LDS;                              // [2][BN][LDS]
    long long* offA = reinterpret_cast<long long*>(Ws + 2 * BN * GEMM_LDS);  // [BM] element offsets, -1 = out of range
    long long* offY = offA + GEMM_BM;
    float* s_mean = reinterpret_cast<float*>(offY + GEMM_BM);
    float* s_rstd = s_mean + GEMM_BM;
    float* s_scale = s_rstd + GEMM_BM;
    float* s_ascale = s_scale + GEMM_BM;

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int warp_m = warp & 3, warp_n = warp >> 2;
    const long long m0 = static_cast<long long>(blockIdx.x) * GEMM_BM;
    const int n0 = blockIdx.y * BN;
    const bool has_ln = g.mean != nullptr;

    for (int r = tid; r < GEMM_BM; r += GEMM_THREADS) {
        long long m = m0 + r;
        long long oa = -1, oy = -1;
        float mu = 0.f, rs = 1.f, sc = 1.f, asc = 1.f;
        if (m < g.M) {
            long long tok = (g.mapA || g.mapY) ? g.map.token(m) : m;
            long long ra = g.mapA ? tok : m;
            long long ry = g.mapY ? tok : m;
            oa = ra * g.lda;
            oy = ry * g.ldy;
            if (has_ln) { mu = g.mean[ra]; rs = g.rstd[ra]; }
            if (EPI == EPI_BIAS_RESID && g.drop_scale) sc = g.drop_scale[ry / g.tokens_per_image];
            if (g.a_row_scale) asc = g.a_row_scale[ra / g.tokens_per_image];
        }
        offA[r] = oa; offY[r] = oy; s_mean[r] = mu; s_rstd[r] = rs; s_scale[r] = sc; s_ascale[r] = asc;
    }
    __syncthreads();

    float acc[MT][NT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;

    const int nk = g.K / GEMM_BK;
    // A staging: 128 rows x 8 float4-chunks = 1024 chunks, 4 per thread
    float4 areg[4];
    auto load_a = [&](int kc) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int c = tid + i * GEMM_THREADS;
            int r = c >> 3, kq = (c & 7) * 4;
            long long o = offA[r];
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (o >= 0) {
                int k = kc * GEMM_BK + kq;
                v = ld4(g.A + o + k);
                if (g.a_row_scale) {
                    const float asc = s_ascale[r];
                    v.x *= asc; v.y *= asc; v.z *= asc; v.w *= asc;
                }
                if (has_ln) {
                    float mu = s_mean[r], rs = s_rstd[r];
                    float4 w = *reinterpret_cast<const float4*>(g.ln_w + k);
                    float4 b = *reinterpret_cast<const float4*>(g.ln_b + k);
                    v.x = (v.x - mu) * rs * w.x + b.x;
                    v.y = (v.y - mu) * rs * w.y + b.y;
                    v.z = (v.z - mu) * rs * w.z + b.z;
                    v.w = (v.w - mu) * rs * w.w + b.w;
                }
            }
            areg[i] = v;
        }
    };
    auto store_a = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int c = tid + i * GEMM_THREADS;
            int r = c >> 3, kq = (c & 7) * 4;
            *reinterpret_cast<float4*>(As + (buf * GEMM_BM + r) * GEMM_LDS + kq) = areg[i];
        }
    };
    auto load_w = [&](int kc, int buf) {
        constexpr int CH = BN * 8;   // 16-byte chunks per stage
        for (int c = tid; c < CH; c += GEMM_THREADS) {
            int r = c >> 3, kq = (c & 7) * 4;
            cp_async16(Ws + (buf * BN + r) * GEMM_LDS + kq,
                       g.Wt + static_cast<long long>(n0 + r) * g.K + kc * GEMM_BK + kq);
        }
        cp_async_commit();
    };

    load_w(0, 0);
    load_a(0);
    store_a(0);
    cp_async_wait<0>();
    __syncthreads();

    for (int kc = 0; kc < nk; ++kc) {
        const int buf = kc & 1;
        const bool more = (kc + 1) < nk;
        if (more) {
            load_w(kc + 1, buf ^ 1);
            load_a(kc + 1);
        }
        const float* Ab = As + (buf * GEMM_BM + warp_m * 32) * GEMM_LDS;
        const float* Wb = Ws + (buf * BN + warp_n * (BN / 2)) * GEMM_LDS;
#pragma unroll
        for (int ks = 0; ks < GEMM_BK / 8; ++ks) {
            float af[MT][4], bf[NT][2];
#pragma unroll
            for (int i = 0; i < MT; ++i) {
                const float* p = Ab + (i * 16 + gq) * GEMM_LDS + ks * 8 + tq;
                af[i][0] = p[0];
                af[i][1] = p[8 * GEMM_LDS];
                af[i][2] = p[4];
                af[i][3] = p[8 * GEMM_LDS + 4];
            }
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const float* p = Wb + (j * 8 + gq) * GEMM_LDS + ks * 8 + tq;
                bf[j][0] = p[0];
                bf[j][1] = p[4];
            }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < NT; ++j) mma_x<PASSES>(acc[i][j], af[i], bf[j]);
        }
        if (more) {
            store_a(buf ^ 1);
            cp_async_wait<0>();
        }
        __syncthreads();
    }

    // ------------------------------------------------------------------ epilogue
#pragma unroll
    for (int i = 0; i < MT; ++i) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = warp_m * 32 + i * 16 + gq + half * 8;
            const long long oy = offY[r];
            if (oy < 0) continue;
            const float sc = s_scale[r];
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const int col = n0 + warp_n * (BN / 2) + j * 8 + 2 * tq;
                float v0 = acc[i][j][half * 2 + 0];
                float v1 = acc[i][j][half * 2 + 1];
                if (g.bias) { v0 += g.bias[col]; v1 += g.bias[col + 1]; }
                if (EPI == EPI_MUL_GELUGRAD) {
                    const float2 pre = ld2(g.aux + oy + col);
                    v0 *= gelu_erf_grad(pre.x);
                    v1 *= gelu_erf_grad(pre.y);
                } else if (EPI == EPI_BIAS_GELU) {
                    if (g.Y2) st2(g.Y2 + oy + col, v0, v1);
                    v0 = gelu_erf(v0);
                    v1 = gelu_erf(v1);
                } else if (EPI == EPI_BIAS_RESID) {
                    float2 rr = ld2(g.R + oy + col);
                    v0 = rr.x + sc * v0;
                    v1 = rr.y + sc * v1;
                }
                st2(g.Y + oy + col, v0, v1);
            }
        }
    }
}

// Per-token LayerNorm statistics (mean, 1/sqrt(var+eps)), biased variance, eps = 1e-5
// (nn.LayerNorm, My_model_1.py:769/776).  G lanes per row (G = min(32, row bytes / 16)), 16-byte loads, so a warp
// streams 512 contiguous bytes per load whatever C is; two-pass statistics from registers.  HBM-bound: C*sizeof(T)
// bytes per token.
template <typename T, int G, int MAXV = 4>          // MAXV loads per lane: C <= G * EPL * MAXV
__global__ void __launch_bounds__(256) ln_stats_kernel(const T* __restrict__ x, long long rows, int C,
                                                       float* __restrict__ mean, float* __restrict__ rstd) {
    constexpr int EPL = 16 / sizeof(T);            // elements per 16-byte load
    constexpr int RPW = 32 / G;                    // rows per warp
    const int lane = threadIdx.x & 31;
    const int sub = lane / G, gl = lane % G;
    const long long warp_global = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long row = warp_global * RPW + sub;
    const bool live = row < rows;
    float v[MAXV][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int k = (gl + i * G) * EPL;
        const bool ok = live && k < C;
        if (sizeof(T) == 4) {
            float4 t = ok ? *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + row * C + k) : make_float4(0.f, 0.f, 0.f, 0.f);
            v[i][0] = t.x; v[i][1] = t.y; v[i][2] = t.z; v[i][3] = t.w;
            v[i][4] = v[i][5] = v[i][6] = v[i][7] = 0.f;
        } else {
            uint4 t = ok ? *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(x) + row * C + k) : make_uint4(0u, 0u, 0u, 0u);
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
            for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(h[j]); v[i][2 * j] = f.x; v[i][2 * j + 1] = f.y; }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[i][j];
    }
    s = group_sum<G>(s);
    const float mu = s / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int k = (gl + i * G) * EPL;
        if (k < C) {
#pragma unroll
            for (int j = 0; j < EPL; ++j) { const float d = v[i][j] - mu; q += d * d; }
        }
    }
    q = group_sum<G>(q);
    if (live && gl == 0) {
        mean[row] = mu;
        rstd[row] = rsqrtf(q / C + 1e-5f);
    }
}

template <int EPI>
cudaError_t launch_gemm(const GemmArgs<float>& g, cudaStream_t stream) {
    dim3 block(GEMM_THREADS);
    const unsigned gm = static_cast<unsigned>((g.M + GEMM_BM - 1) / GEMM_BM);
    if (g.N % 64 == 0) {
        constexpr size_t smem = gemm_smem_bytes<64>();
        auto k = gemm_fused_kernel<float, 64, EPI>;
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
        k<<<dim3(gm, g.N / 64), block, smem, stream>>>(g);
    } else {
        constexpr size_t smem = gemm_smem_bytes<32>();
        auto k = gemm_fused_kernel<float, 32, EPI>;
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
        k<<<dim3(gm, g.N / 32), block, smem, stream>>>(g);
    }
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_ln_stats(const T* x, long long rows, int C, float* mean, float* rstd, cudaStream_t stream) {
    constexpr int EPL = 16 / sizeof(T);
    const int chunks = C / EPL;                 // 16-byte chunks per row (C % 32 == 0 => >= 4)
    const int wpb = 8;
    auto go = [&](auto gtag) -> cudaError_t {
        constexpr int G = decltype(gtag)::value;
        const long long rows_per_block = static_cast<long long>(wpb) * (32 / G);
        const unsigned grid = static_cast<unsigned>((rows + rows_per_block - 1) / rows_per_block);
        ln_stats_kernel<T, G><<<grid, wpb * 32, 0, stream>>>(x, rows, C, mean, rstd);
        return cudaGetLastError();
    };
    if (chunks > 256) return cudaErrorInvalidValue;      // C <= 32 lanes * 8 loads * EPL
    if (chunks > 128) {                                   // fp32 rows of 516 ... 1024 channels (embed_dim 64: C = 1024 at the bottleneck)
        const unsigned grid = static_cast<unsigned>((rows + wpb - 1) / wpb);
        ln_stats_kernel<T, 32, 8><<<grid, wpb * 32, 0, stream>>>(x, rows, C, mean, rstd);
        return cudaGetLastError();
    }
    if (chunks <= 4) return go(std::integral_constant<int, 4>{});
    if (chunks <= 8) return go(std::integral_constant<int, 8>{});
    if (chunks <= 16) return go(std::integral_constant<int, 16>{});
    return go(std::integral_constant<int, 32>{});
}

}  // namespace lewin
