// Weight gradient of the LeWin linears for bf16 activations:  dW[N,K] += dY[M,N]^T * X[M,K],  db[N] += colsum(dY)
// (autograd of attn.py:420-422 / :456 and My_model_1.py:508 / :529; same contract as wgrad_kernel in backward.cuh).
//
// It is a reduction over the token axis M with a tiny output, i.e. HBM-bound: read every dY and X row once.  The generic
// kernel staged 32 tokens at a time through fp32 shared memory with three block barriers per stage and exposed every
// load; here:
//   * a CTA owns a [NT x KT] slice of dW (128 x 64 or 64 x 64) for one contiguous range of tokens, accumulators in
//     registers, one atomicAdd per element at the end;
//   * tokens advance in 64-row stages; the next stage's 16-byte global loads (with the LN / DropPath / window-order
//     prologues applied in registers, bf16 rounding points as the forward) are in flight while the current stage runs
//     its MMAs, two shared-memory buffers, ONE barrier per stage;
//   * both operands are token-major in memory, i.e. "transposed" for this product: ldmatrix.trans delivers the
//     mma.sync.m16n8k16 bf16 fragments straight from the [token][channel] tiles;
//   * the bias gradient is one extra MMA per m-tile against a constant all-ones B fragment.
#pragma once
#include "wgrad_args.cuh"
#include "probsparse_core_bf16.cuh"

namespace lewin {
namespace wg2 {

constexpr int THREADS = 256;
constexpr int TOK = 64;                               // tokens per stage

template <int NT, int KT>
struct Smem {
    static constexpr int LDN = NT + 8, LDK = KT + 8;  // +16 B: conflict-free ldmatrix rows
    __nv_bfloat16 dy[2][TOK * LDN];
    __nv_bfloat16 x[2][TOK * LDK];
    long long offD[2][TOK], offX[2][TOK];
    float mu[2][TOK], rs[2][TOK], sc[2][TOK];
};

__device__ __forceinline__ void ldsm_x2_t(uint32_t (&r)[2], const void* p) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}

// WARPS_N warps along n (dW rows), 8 / WARPS_N along k: 4 x 2 for the 128- and 64-row tiles, 2 x 4 for the 32-row tiles of C = 32
// DET: the per-element partials are stored into split blockIdx.z's slab of [splits][N, K] / [splits][N] instead of added
template <int NT, int KT, int WARPS_N, bool DET = false>
__global__ void __launch_bounds__(THREADS) wgrad_bf16_kernel(const WgradArgs<__nv_bfloat16> g) {
    using S = Smem<NT, KT>;
    constexpr int LDN = S::LDN, LDK = S::LDK;
    constexpr int WARPS_K = 8 / WARPS_N;
    constexpr int WN = NT / WARPS_N, WK = KT / WARPS_K;
    static_assert(WN % 16 == 0 && WK % 8 == 0, "warp tile");
    constexpr int MT = WN / 16, NTL = WK / 8;         // m16 tiles, n8 tiles per warp
    constexpr int DTOT = TOK * NT / 8, XTOT = TOK * KT / 8;       // 16-byte chunks per stage
    constexpr int DCH = (DTOT + THREADS - 1) / THREADS, XCH = (XTOT + THREADS - 1) / THREADS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S& s = *reinterpret_cast<S*>(smem_raw);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int wn = warp % WARPS_N, wk = warp / WARPS_N;
    const int n0 = blockIdx.x * NT, k0 = blockIdx.y * KT;
    const long long m_begin = static_cast<long long>(blockIdx.z) * g.rows_per_split;
    long long m_end = m_begin + g.rows_per_split;
    if (m_end > g.M) m_end = g.M;
    const int stages = static_cast<int>((m_end - m_begin + TOK - 1) / TOK);
    const bool has_ln = g.mean != nullptr;
    const bool want_db = g.db != nullptr && blockIdx.y == 0 && wk == 0;

    float acc[MT][NTL][4];
    float accb[MT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i) {
#pragma unroll
        for (int j = 0; j < NTL; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[i][j][c] = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) accb[i][c] = 0.f;
    }

    auto rowinfo = [&](int st, int b) {               // threads 0..63: addressing + per-row prologue scalars of stage st
        if (tid < TOK) {
            const long long m = m_begin + static_cast<long long>(st) * TOK + tid;
            long long od = -1, ox = -1;
            float mu = 0.f, rs = 1.f, sc = 1.f;
            if (st < stages && m < m_end) {
                const long long tok = (g.mapDY || g.mapX) ? static_cast<long long>(g.map.token32(static_cast<uint32_t>(m))) : m;
                const long long rd = g.mapDY ? tok : m, rx = g.mapX ? tok : m;
                od = rd * g.lddy; ox = rx * g.ldx;
                if (has_ln) { mu = g.mean[rx]; rs = g.rstd[rx]; }
                if (g.dy_row_scale) sc = g.dy_row_scale[rd / g.tokens_per_image];
            }
            s.offD[b][tid] = od; s.offX[b][tid] = ox; s.mu[b][tid] = mu; s.rs[b][tid] = rs; s.sc[b][tid] = sc;
        }
    };
    uint4 dreg[DCH], xreg[XCH];
    auto load = [&](int b) {                          // raw 16-byte loads of one stage (nothing consumes them until store)
#pragma unroll
        for (int i = 0; i < DCH; ++i) {
            const int c = tid + i * THREADS, r = c / (NT / 8), ch = c % (NT / 8);
            const long long o = (DTOT % THREADS == 0 || c < DTOT) ? s.offD[b][r] : -1;
            dreg[i] = o >= 0 ? *reinterpret_cast<const uint4*>(g.dY + o + n0 + ch * 8) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int i = 0; i < XCH; ++i) {
            const int c = tid + i * THREADS, r = c / (KT / 8), ch = c % (KT / 8);
            const long long o = (XTOT % THREADS == 0 || c < XTOT) ? s.offX[b][r] : -1;
            xreg[i] = o >= 0 ? *reinterpret_cast<const uint4*>(g.X + o + k0 + ch * 8) : make_uint4(0u, 0u, 0u, 0u);
        }
    };
    auto unpack = [](const uint4& u, float (&f)[8]) {
        f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
        f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
        f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xFFFF0000u);
        f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xFFFF0000u);
    };
    auto store = [&](int b) {                         // prologues in registers, bf16 tiles to shared memory
#pragma unroll
        for (int i = 0; i < DCH; ++i) {
            const int c = tid + i * THREADS, r = c / (NT / 8), ch = c % (NT / 8);
            if (DTOT % THREADS != 0 && c >= DTOT) break;
            uint4 v = dreg[i];
            if (g.dy_row_scale && s.offD[b][r] >= 0) {
                float f[8];
                unpack(v, f);
                const float sc = s.sc[b][r];
                v = make_uint4(pc::pack2(f[0] * sc, f[1] * sc), pc::pack2(f[2] * sc, f[3] * sc), pc::pack2(f[4] * sc, f[5] * sc),
                               pc::pack2(f[6] * sc, f[7] * sc));
            }
            *reinterpret_cast<uint4*>(s.dy[b] + r * LDN + ch * 8) = v;
        }
#pragma unroll
        for (int i = 0; i < XCH; ++i) {
            const int c = tid + i * THREADS, r = c / (KT / 8), ch = c % (KT / 8);
            if (XTOT % THREADS != 0 && c >= XTOT) break;
            uint4 v = xreg[i];
            if (has_ln && s.offX[b][r] >= 0) {
                float f[8];
                unpack(v, f);
                const float mu = s.mu[b][r], rs = s.rs[b][r];
                const float4 w0 = *reinterpret_cast<const float4*>(g.ln_w + k0 + ch * 8), w1 = *reinterpret_cast<const float4*>(g.ln_w + k0 + ch * 8 + 4);
                const float4 b0 = *reinterpret_cast<const float4*>(g.ln_b + k0 + ch * 8), b1 = *reinterpret_cast<const float4*>(g.ln_b + k0 + ch * 8 + 4);
                v = make_uint4(pc::pack2((f[0] - mu) * rs * w0.x + b0.x, (f[1] - mu) * rs * w0.y + b0.y),
                               pc::pack2((f[2] - mu) * rs * w0.z + b0.z, (f[3] - mu) * rs * w0.w + b0.w),
                               pc::pack2((f[4] - mu) * rs * w1.x + b1.x, (f[5] - mu) * rs * w1.y + b1.y),
                               pc::pack2((f[6] - mu) * rs * w1.z + b1.z, (f[7] - mu) * rs * w1.w + b1.w));
            }
            *reinterpret_cast<uint4*>(s.x[b] + r * LDK + ch * 8) = v;
        }
    };

    rowinfo(0, 0);
    rowinfo(1, 1);
    __syncthreads();
    load(0);
    for (int st = 0; st < stages; ++st) {
        const int b = st & 1;
        store(b);
        __syncthreads();            // tile b visible; row info of stage st+1 visible; everyone is done with tile b^1
        if (st + 1 < stages) load(b ^ 1);
        rowinfo(st + 2, b);         // buffer b's row info was last read by store(b) above (before the barrier)
        const __nv_bfloat16* dys = s.dy[b];
        const __nv_bfloat16* xs = s.x[b];
#pragma unroll
        for (int ks = 0; ks < TOK / 16; ++ks) {
            uint32_t bf[(NTL + 1) / 2][4];
            if constexpr (NTL == 1) {
                uint32_t b2[2];
                ldsm_x2_t(b2, xs + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LDK + wk * WK);
                bf[0][0] = b2[0]; bf[0][1] = b2[1]; bf[0][2] = 0u; bf[0][3] = 0u;
            } else {
#pragma unroll
                for (int jp = 0; jp < NTL / 2; ++jp)
                    pc::ldsm_x4_t(bf[jp], xs + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LDK + wk * WK + jp * 16 + (lane >> 4) * 8);
            }
#pragma unroll
            for (int i = 0; i < MT; ++i) {
                uint32_t af[4];     // A[n][tok] = dY[tok][n], transposed on load
                pc::ldsm_x4_t(af, dys + (ks * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * LDN + wn * WN + i * 16 + ((lane >> 3) & 1) * 8);
                if constexpr (NTL == 1) {
                    pc::mma16816(acc[i][0], af, bf[0][0], bf[0][1]);
                } else {
#pragma unroll
                    for (int jp = 0; jp < NTL / 2; ++jp) {
                        pc::mma16816(acc[i][2 * jp], af, bf[jp][0], bf[jp][1]);
                        pc::mma16816(acc[i][2 * jp + 1], af, bf[jp][2], bf[jp][3]);
                    }
                }
                if (want_db) pc::mma16816(accb[i], af, 0x3F803F80u, 0x3F803F80u);      // x 1.0: column sums of dY
            }
        }
    }
    if constexpr (DET) {
        float* dW = g.dW + static_cast<long long>(blockIdx.z) * g.N * g.K;
        float* db = g.db + static_cast<long long>(blockIdx.z) * g.N;      // (read only when want_db)
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int n = n0 + wn * WN + i * 16 + gq + half * 8;
#pragma unroll
                for (int j = 0; j < NTL; ++j) {
                    const int k = k0 + wk * WK + j * 8 + 2 * tq;
                    *reinterpret_cast<float2*>(dW + static_cast<long long>(n) * g.K + k) = make_float2(acc[i][j][half * 2], acc[i][j][half * 2 + 1]);
                }
                if (want_db && tq == 0) db[n] = accb[i][half * 2];
            }
        return;
    }
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int n = n0 + wn * WN + i * 16 + gq + half * 8;
#pragma unroll
            for (int j = 0; j < NTL; ++j) {
                const int k = k0 + wk * WK + j * 8 + 2 * tq;
                atomicAdd(g.dW + static_cast<long long>(n) * g.K + k, acc[i][j][half * 2]);
                atomicAdd(g.dW + static_cast<long long>(n) * g.K + k + 1, acc[i][j][half * 2 + 1]);
            }
            if (want_db && tq == 0) atomicAdd(g.db + n, accb[i][half * 2]);
        }
}

inline bool supported(const WgradArgs<__nv_bfloat16>& g) {
    return !g.dy_aux && g.N % 32 == 0 && g.K % 32 == 0 && g.M < (1ll << 31);
}

template <int NT, int KT, int WARPS_N, bool DET>
cudaError_t launch_t(WgradArgs<__nv_bfloat16> g, int num_sms, cudaStream_t st) {
    const long long tiles = static_cast<long long>(g.N / NT) * (g.K / KT);
    long long want = (static_cast<long long>(num_sms) * 3 + tiles - 1) / tiles;
    const long long max_splits = (g.M + TOK - 1) / TOK;
    if (want > max_splits) want = max_splits;
    if (want < 1) want = 1;
    long long rps = (g.M + want - 1) / want;
    rps = (rps + TOK - 1) / TOK * TOK;
    if (DET) rps = det_wgrad_rows_per_split(g.M, g.N, g.K);
    const unsigned splits = static_cast<unsigned>((g.M + rps - 1) / rps);
    g.rows_per_split = rps;
    auto k = wgrad_bf16_kernel<NT, KT, WARPS_N, DET>;
    const size_t smem = sizeof(Smem<NT, KT>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    k<<<dim3(g.N / NT, g.K / KT, splits), THREADS, smem, st>>>(g);
    return cudaGetLastError();
}

template <bool DET>
cudaError_t launch(const WgradArgs<__nv_bfloat16>& g, int num_sms, cudaStream_t st) {
    if (g.K % 64 == 0) {
        if (g.N % 128 == 0) return launch_t<128, 64, 4, DET>(g, num_sms, st);
        if (g.N % 64 == 0) return launch_t<64, 64, 4, DET>(g, num_sms, st);
        return launch_t<32, 64, 2, DET>(g, num_sms, st);
    }
    if (g.N % 128 == 0) return launch_t<128, 32, 4, DET>(g, num_sms, st);
    return launch_t<32, 32, 2, DET>(g, num_sms, st);
}

}  // namespace wg2
}  // namespace lewin
