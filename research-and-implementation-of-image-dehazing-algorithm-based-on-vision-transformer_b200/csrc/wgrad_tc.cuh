// Weight gradient of the LeWin linears on tcgen05 (bf16, C >= 128 levels):
//
//   dW[N, K] += dY[M, N]^T . X[M, K]        db[N] += colsum(dY)        (autograd of attn.py:420-422 / :456, My_model_1.py:508 / :529)
//
// The contraction runs over the TOKEN axis, and both operands are token-major in memory, i.e. "transposed" for this product.
// mma.sync needed ldmatrix.trans and reached 131 TFLOP/s at C = 512 (wgrad_bf16.cuh, the top item of the training step);
// tcgen05.mma reads MN-major operands directly: a TMA box of [64 tokens x 64 features] in SWIZZLE_128B is exactly the
// canonical MN-major atom ((8,n),(8,k)):((1,LBO),(8,SBO)) with SBO = 1024 B between 8-token groups and LBO = 8 KB between
// 64-feature blocks, so no transposition happens anywhere:
//   * CTA = one [128 x BK] tile of dW (128 dY features x BK <= 256 X features) for one contiguous range of tokens; feature
//     counts that are not multiples of 128 / 64 (C = 32, 64 levels) ride on the TMA unit's zero fill of out-of-range columns;
//   * one TMA thread streams 64-token stages (2 boxes of dY, BK / 64 boxes of X) through an S-deep ring;
//   * one MMA thread issues 4 x tcgen05.mma kind::f16 (a_major = b_major = MN, K = 16 tokens each) per stage into the TMEM
//     accumulator, plus 4 N = 16 MMAs against a constant all-ones tile whose result column is colsum(dY) (the bias gradient);
//   * after the last stage 4 warps read the accumulator (thread == dW row), transpose 32 x 32 pieces through shared memory and
//     add them to dW with coalesced red.global.add.f32 (splits over the token axis accumulate in place).  DET: the same
//     coalesced rows are stored into split blockIdx.z's slab of [splits][N, K] (det_wgrad_rows_per_split), summed later in
//     split order.
// Operands with a prologue (LayerNorm, roll + window gather, DropPath scale) are materialised by their callers first
// (ln_apply_kernel / scale_gather_rows_kernel, one C-sized pass each - small next to the hidden-sized operands).
#pragma once
#include "wgrad_args.cuh"
#include "tc_helpers.cuh"
#include "tma.cuh"

namespace lewin {
namespace wg3 {

constexpr int TOK = 64;                       // tokens per stage
constexpr int NT = 128;                       // dW rows per CTA (dY features)
constexpr int THREADS = 6 * 32;               // 4 epilogue warps, MMA warp, TMA warp
constexpr int MMA_WARP = 4, TMA_WARP = 5;
constexpr int BLK = TOK * 128;                // bytes of one [64 tokens x 64 features] block
constexpr int STG_LD = 33;                    // transpose tile row stride (floats)
constexpr int SMEM_MAX = 227 * 1024;

// MN-major SWIZZLE_128B descriptor: LBO = 8 KB (next 64-feature block), SBO = 1 KB (next 8-token group)
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr) {
    return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF) | (static_cast<uint64_t>(BLK >> 4) << 16) |
           (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

constexpr size_t fixed_smem() { return 1024 + BLK /*ones*/ + 4 * 32 * STG_LD * 4 + (2 * 8 + 1) * 8 + 16; }

template <int BK, bool DET = false>
__global__ void __launch_bounds__(THREADS, 1) wgrad_tc_kernel(const WgradArgs<__nv_bfloat16> g, const __grid_constant__ CUtensorMap dymap,
                                                             const __grid_constant__ CUtensorMap xmap, int S) {
    constexpr int NB = (BK + 63) / 64;            // 64-feature blocks of X per stage
    constexpr int STAGE = 2 * BLK + NB * BLK;
    constexpr int TMEM_COLS = BK + 16 <= 64 ? 64 : BK + 16 <= 128 ? 128 : BK + 16 <= 256 ? 256 : 512;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | (static_cast<uint32_t>(BK >> 3) << 17) |
                               (static_cast<uint32_t>(NT >> 4) << 24);
    constexpr uint32_t IDESC_DB = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | (static_cast<uint32_t>(16 >> 3) << 17) |
                                  (static_cast<uint32_t>(NT >> 4) << 24);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* ring = base;                                         // [S][dY 2 blocks | X BK/64 blocks]
    unsigned char* ones = ring + static_cast<size_t>(S) * STAGE;        // [64 tokens x 64] of bf16 1.0
    float* stg = reinterpret_cast<float*>(ones + BLK);                  // [4 warps][32][STG_LD]
    uint64_t* full = reinterpret_cast<uint64_t*>(stg + 4 * 32 * STG_LD);
    uint64_t* empty = full + 8;
    uint64_t* done = empty + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.x * NT, k0 = blockIdx.y * BK;
    const long long m_begin = static_cast<long long>(blockIdx.z) * g.rows_per_split;
    long long m_end = m_begin + g.rows_per_split;
    if (m_end > g.M) m_end = g.M;
    const int stages = static_cast<int>((m_end - m_begin + TOK - 1) / TOK);
    const bool want_db = g.db != nullptr && blockIdx.y == 0;

    for (int i = tid; i < BLK / 16; i += THREADS) reinterpret_cast<uint4*>(ones)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    if (tid == 0) {
        for (int i = 0; i < S; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        tc::mbar_init(done, 1);
        tc::fence_barrier_init();
        tma::prefetch_map(&dymap);
        tma::prefetch_map(&xmap);
    }
    if (warp == MMA_WARP) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::fence_proxy_async();                         // the ones tile: generic-proxy writes -> async proxy
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    if (warp == TMA_WARP) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int st = 0; st < stages; ++st) {
                const int m = static_cast<int>(m_begin) + st * TOK;
                tc::mbar_wait(&empty[s], ph ^ 1u);
                tma::mbar_expect_tx(&full[s], STAGE);
                unsigned char* dst = ring + static_cast<size_t>(s) * STAGE;
                tma::load_2d(dst, &dymap, &full[s], n0, m);
                tma::load_2d(dst + BLK, &dymap, &full[s], n0 + 64, m);
#pragma unroll
                for (int j = 0; j < NB; ++j) tma::load_2d(dst + (2 + j) * BLK, &xmap, &full[s], k0 + 64 * j, m);
                if (++s == S) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0) {
            const uint32_t ring_u = tc::smem_u32(ring);
            const uint64_t d_ones = make_desc_mn(tc::smem_u32(ones));
            int s = 0;
            uint32_t ph = 0;
            for (int st = 0; st < stages; ++st) {
                tc::mbar_wait(&full[s], ph);
                tc::tc_fence_after();
                const uint64_t da = make_desc_mn(ring_u + s * STAGE);
                const uint64_t db = make_desc_mn(ring_u + s * STAGE + 2 * BLK);
#pragma unroll
                for (int k16 = 0; k16 < TOK / 16; ++k16) {               // 16 tokens = two 8-token groups = 2 KB further on
                    const uint32_t acc = (st > 0 || k16 > 0) ? 1u : 0u;
                    tc::mma_bf16(tmem_d, da + 128 * k16, db + 128 * k16, IDESC, acc);
                    if (want_db) tc::mma_bf16(tmem_d + BK, da + 128 * k16, d_ones + 128 * k16, IDESC_DB, acc);
                }
                tc::mma_commit(&empty[s]);
                if (++s == S) { s = 0; ph ^= 1u; }
            }
            tc::mma_commit(done);
        }
    } else {
        // ============================================================ epilogue: thread == TMEM lane == dW row
        float* my = stg + warp * 32 * STG_LD;
        tc::mbar_wait(done, 0);
        tc::tc_fence_after();
        if (stages > 0) {
            const uint32_t t_addr = tmem_d + (static_cast<uint32_t>(warp * 32) << 16);
            const int row0 = n0 + warp * 32;          // this warp's first dW row; rows >= N exist only as zero-filled operand rows
            float* dW = DET ? g.dW + static_cast<long long>(blockIdx.z) * g.N * g.K : g.dW;
            float* dst = dW + static_cast<long long>(row0) * g.K + k0;
            const int nrows = g.N - row0 < 32 ? g.N - row0 : 32;
#pragma unroll 1
            for (int c = 0; c < BK / 32; ++c) {
                float v[32];
                tc::tmem_ld32(t_addr + c * 32, v);    // (warp-collective: also executed by warps whose rows are all >= N)
#pragma unroll
                for (int j = 0; j < 32; ++j) my[lane * STG_LD + j] = v[j];
                __syncwarp();
                if constexpr (DET) {
                    for (int r = 0; r < nrows; ++r) dst[static_cast<long long>(r) * g.K + c * 32 + lane] = my[r * STG_LD + lane];
                } else {
                    for (int r = 0; r < nrows; ++r) atomicAdd(dst + static_cast<long long>(r) * g.K + c * 32 + lane, my[r * STG_LD + lane]);
                }
                __syncwarp();
            }
            if (want_db) {
                float v[32];
                tc::tmem_ld32(t_addr + BK, v);       // 16 identical columns (+ 16 unused): colsum(dY) of this row's feature
                if constexpr (DET) {
                    if (lane < nrows) g.db[static_cast<long long>(blockIdx.z) * g.N + row0 + lane] = v[0];
                } else {
                    if (lane < nrows) atomicAdd(g.db + row0 + lane, v[0]);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

inline bool supported(const WgradArgs<__nv_bfloat16>& g) {
    if (g.mapDY || g.mapX || g.dy_row_scale || g.mean || g.dy_aux) return false;
    if (g.N % 32 || g.K % 32 || (g.K > 256 && g.K % 256) || g.M < 1024 || g.M >= (1ll << 31)) return false;
    if (!(g.K % 256 == 0 || g.K == 32 || g.K == 64 || g.K == 96 || g.K == 128 || g.K == 192)) return false;
    if ((g.lddy % 8) || (g.ldx % 8)) return false;
    if ((reinterpret_cast<uintptr_t>(g.dY) & 15) || (reinterpret_cast<uintptr_t>(g.X) & 15)) return false;
    return tma::encode_fn() != nullptr;
}

template <int BK, bool DET>
cudaError_t launch_bk(WgradArgs<__nv_bfloat16> g, int num_sms, cudaStream_t stream) {
    constexpr int STAGE = 2 * BLK + ((BK + 63) / 64) * BLK;
    constexpr size_t fixed = fixed_smem();
    int S = static_cast<int>((SMEM_MAX - fixed) / STAGE);
    if (S > 8) S = 8;
    const size_t smem = fixed + static_cast<size_t>(S) * STAGE;
    CUtensorMap dymap{}, xmap{};
    if (!tma::make_2d_bf16_sw128(&dymap, g.dY, g.M, g.N, g.lddy, TOK) || !tma::make_2d_bf16_sw128(&xmap, g.X, g.M, g.K, g.ldx, TOK))
        return cudaErrorNotSupported;
    auto k = wgrad_tc_kernel<BK, DET>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int n_tiles = (g.N + NT - 1) / NT;
    const long long tiles = static_cast<long long>(n_tiles) * (g.K / BK);
    long long want = (num_sms + tiles - 1) / tiles;                  // about one CTA per SM
    const long long max_splits = (g.M + 4 * TOK - 1) / (4 * TOK);    // at least four stages per CTA
    if (want > max_splits) want = max_splits;
    if (want < 1) want = 1;
    long long rps = (g.M + want - 1) / want;
    rps = (rps + TOK - 1) / TOK * TOK;
    if (DET) rps = det_wgrad_rows_per_split(g.M, g.N, g.K);
    const unsigned splits = static_cast<unsigned>((g.M + rps - 1) / rps);
    g.rows_per_split = rps;
    k<<<dim3(n_tiles, g.K / BK, splits), THREADS, smem, stream>>>(g, dymap, xmap, S);
    return cudaGetLastError();
}

template <bool DET>
cudaError_t launch(const WgradArgs<__nv_bfloat16>& g, int num_sms, cudaStream_t stream) {
    if (g.K % 256 == 0) return launch_bk<256, DET>(g, num_sms, stream);
    if (g.K == 128) return launch_bk<128, DET>(g, num_sms, stream);
    if (g.K == 64) return launch_bk<64, DET>(g, num_sms, stream);
    if (g.K == 32) return launch_bk<32, DET>(g, num_sms, stream);
    if (g.K == 96) return launch_bk<96, DET>(g, num_sms, stream);
    if (g.K == 192) return launch_bk<192, DET>(g, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace wg3
}  // namespace lewin
