// Warp-specialised persistent tcgen05 token GEMM for the HBM-bound LeWin levels (C <= 128, bf16):
//
//   Y = epi( LN?(A)[M,K] * W[N,K]^T + bias )
//
// Same contract as gemm_fused_kernel / gemm_tc_kernel (q|k|v projections attn.py:420-422, out projection :456,
// LeFF linear1 My_model_1.py:508, linear2 :529, with LN / roll / window_partition / window_reverse / DropPath /
// residual folded in), restructured so that the three things that bound it run concurrently inside ONE resident
// CTA per SM instead of taking turns:
//
//   * 8 producer warps  : global -> registers (a register ring keeps >= 8 x 16 B per thread in flight across stage
//                         boundaries) -> LayerNorm computed on the fly from the row itself (no ln_stats pre-pass,
//                         no second read of x) -> bf16 -> swizzled UMMA tile in an S-stage shared-memory ring;
//   * 1 MMA thread      : tcgen05.mma kind::f16 M=128 x N=BN, accumulating into one of TWO TMEM accumulator stages;
//                         tcgen05.commit releases the smem stage to the producers and hands the accumulator over;
//   * 8 epilogue warps  : tcgen05.ld (thread == row) -> bias / exact table GELU / DropPath * residual -> per-warp
//                         staging tile -> row-cooperative, fully coalesced 16-byte global stores (window_reverse +
//                         un-shift as the row address); residual rows are prefetched into the staging tile with
//                         cp.async before the accumulator is awaited.
//
// The weight tile W[BN x K] (bf16-rounded, autocast semantics) stays resident in shared memory for the whole kernel;
// every hand-over is an mbarrier, there is no __syncthreads in the steady state.
#pragma once
#include "gemm_tc.cuh"
#include "tma.cuh"

namespace lewin {
namespace ws {

// warp roles: [0, NEW) epilogue (warp % 4 == TMEM lane group, warp / 4 == column group), NEW: MMA issuer,
// (NEW, NEW + NPW]: producers.  NEW + NPW == 16 (17 warps); the split is a template parameter because the balance differs:
// 8 + 8 for the plain epilogues, 12 + 4 where the epilogue carries the GELU.
constexpr int WARPS = 17;
constexpr int THREADS = WARPS * 32;
constexpr int STG_ROW = 80;                   // staging row: 32 bf16 columns (64 B) + 16 B pad (conflict-free 16 B accesses)
constexpr int STG_BUF = 32 * STG_ROW;
constexpr int SMEM_MAX = 227 * 1024;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
    f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
    f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xFFFF0000u);
    f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xFFFF0000u);
}


// packed fp32x2 arithmetic (one issue slot for two lanes of work; same IEEE rounding as the scalar instructions)
__device__ __forceinline__ float2 add2(const float2 a, const float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 mul2(const float2 a, const float2 b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fma2(const float2 a, const float2 b, const float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)),
          "l"(*reinterpret_cast<const unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}

// fixed shared memory besides the weight tile and the A ring
template <int BN, int EPI, int NEW>
constexpr size_t fixed_smem() {
    return 1024 /*align*/ + NEW * 2 * STG_BUF + BN * 4 + (2 * 8 + 8) * 8 + 16 + (EPI == EPI_BIAS_GELU ? kGelu2TabSize * 2 : 0);
}

// residual rows of one warp's 32 rows x 32 columns of tile `tile` -> staging buffer (cp.async, coalesced 64-byte row pieces)
template <int NCG>
__device__ __forceinline__ void resid_prefetch(const GemmArgs<__nv_bfloat16>& g, uint32_t tile, int col0, unsigned char* sbuf, int lg, int lane) {
    const uint32_t m = tile * TC_BM + lg * 32 + lane;
    long long oy = -1;
    if (m < g.M) oy = static_cast<long long>(g.mapY ? g.map.token32(m) : m) * (g.ldr ? g.ldr : g.ldy);
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
        const long long o = __shfl_sync(0xffffffffu, oy, rl);
        if (o >= 0) cp_async16(sbuf + rl * STG_ROW + cc * 16, g.R + o + col0 + cc * 8);
    }
}

// One warp's share of one output tile: wait for the accumulator, tcgen05.ld 32-column chunks (thread == TMEM lane == tile
// row), bias / GELU / residual, stage, row-cooperative coalesced stores.  Shared by the resident-W and streamed-W kernels.
template <int BN, int EPI, int NCG, int NBUF = 2, bool ALLOW_XT = true>
__device__ __forceinline__ void epilogue_tile(const GemmArgs<__nv_bfloat16>& g, uint32_t tmem_d, int acc, uint32_t aph, uint32_t tile,
                                              int n0, const float* s_bias, const uint16_t* gtab, unsigned char* my_stg,
                                              uint64_t* tfull, uint64_t* tempty, int lg, int half, int lane,
                                              long long tile_next = -1, int parity = 0, const CUtensorMap* ymap = nullptr) {
    using T = __nv_bfloat16;
    constexpr int ACC = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr int NCH = BN / 32;
    // One chunk per warp (BN <= 32 * NCG): the residual rows of the NEXT tile are prefetched into the other staging buffer
    // while this tile is processed -- at C <= 64 a tile is so small that waiting for this tile's own residual (one DRAM
    // latency per tile and warp) was the critical path.  The caller issues the first tile's prefetch (resid_prefetch).
    constexpr bool XT = ALLOW_XT && (EPI == EPI_BIAS_RESID) && (NCH <= NCG) && NBUF == 2;   // (the streamed-W kernel walks tiles column-fastest and does not use the cross-tile prefetch)
    static_assert(NBUF == 2 || EPI != EPI_BIAS_RESID, "the residual prefetch uses two staging buffers");
        if (EPI != EPI_BIAS_RESID && ymap != nullptr) {      // staging buffers restart at 0 every tile: drain my outstanding box stores
            if (lane == 0) tma::store_wait_read<0>();
            __syncwarp();
        }
        const uint32_t m = tile * TC_BM + lg * 32 + lane;
        long long oy = -1, orr = -1;                  // element offsets of my output row and my residual row
        float sc = 1.f;
        uint32_t up_t00 = 0;                          // up2: output token of (di, dj) = (0, 0)
        if (m < g.M) {
            const uint32_t ry = g.mapY ? g.map.token32(m) : m;
            oy = static_cast<long long>(ry) * g.ldy;
            orr = static_cast<long long>(ry) * (g.ldr ? g.ldr : g.ldy);
            if (EPI == EPI_BIAS_RESID && g.drop_scale) sc = g.drop_scale[ry / static_cast<uint32_t>(g.tokens_per_image)];
            if (g.up2) {
                const uint32_t hw = static_cast<uint32_t>(g.up_H) * g.up_W;
                const uint32_t b = m / hw, rem = m - b * hw, i = rem / static_cast<uint32_t>(g.up_W), j = rem - i * g.up_W;
                up_t00 = (b * 2u * g.up_H + 2u * i) * 2u * g.up_W + 2u * j;
            }
        }
        const long long oy_plain = oy;
        if constexpr (XT) {
            if (tile_next >= 0 && half < NCH) resid_prefetch<NCG>(g, static_cast<uint32_t>(tile_next), n0 + half * 32, my_stg + (parity ^ 1) * STG_BUF, lg, lane);
            cp_async_commit();
        } else if (EPI == EPI_BIAS_RESID) {     // residual rows of my first two chunks -> staging (async, coalesced)
            int q = 0;
            for (int c = half; c < NCH && q < 2; c += NCG, ++q) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const long long o = __shfl_sync(0xffffffffu, orr, rl);
                    if (o >= 0) cp_async16(my_stg + q * STG_BUF + rl * STG_ROW + cc * 16, g.R + o + n0 + c * 32 + cc * 8);
                }
            }
            cp_async_commit();
        }
        tc::mbar_wait(&tfull[acc], aph);
        tc::tc_fence_after();
        if constexpr (XT) { cp_async_wait<1>(); __syncwarp(); }      // this tile's residual landed (the next tile's may still fly)
        else if (EPI == EPI_BIAS_RESID) { cp_async_wait<0>(); __syncwarp(); }
        const uint32_t t_addr = tmem_d + (static_cast<uint32_t>(lg * 32) << 16) + static_cast<uint32_t>(acc * ACC);
        int q = 0;
        for (int c = half; c < NCH; c += NCG, ++q) {
            float v[32];
            tc::tmem_ld32(t_addr + c * 32, v);
            if (c + NCG >= NCH) {               // last chunk of this warp is in registers: hand the accumulator back
                tc::tc_fence_before();
                mbar_arrive(&tempty[acc]);
            }
            unsigned char* sb = my_stg + (XT ? parity : (NBUF == 2 ? (q & 1) : 0)) * STG_BUF;
            if (g.up2 && oy_plain >= 0) {             // pixel shuffle: this chunk's column block selects the output pixel
                const int col = n0 + c * 32, qb = col / g.up_C, cb = col - qb * g.up_C;
                oy = static_cast<long long>(up_t00 + (qb >> 1) * 2u * g.up_W + (qb & 1)) * g.ldy + cb - col;
            }
            unsigned char* srow = sb + lane * STG_ROW;
            const float2* bs2 = reinterpret_cast<const float2*>(s_bias + c * 32);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float2 t2 = add2(make_float2(v[2 * j], v[2 * j + 1]), bs2[j]);
                v[2 * j] = t2.x; v[2 * j + 1] = t2.y;
            }
            if (EPI == EPI_BIAS_RESID) {
                if (q >= 2) {                   // (not reached for BN <= 128) late residual chunk: synchronous, coalesced
                    __syncwarp();
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                        const long long o = __shfl_sync(0xffffffffu, orr, rl);
                        if (o >= 0)
                            *reinterpret_cast<uint4*>(sb + rl * STG_ROW + cc * 16) =
                                *reinterpret_cast<const uint4*>(g.R + o + n0 + c * 32 + cc * 8);
                    }
                    __syncwarp();
                }
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const uint4 rv = *reinterpret_cast<const uint4*>(srow + j * 2);
                    float rf[8];
                    unpack8(rv, rf);
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[j + e] = rf[e] + sc * Act<T>::round(v[j + e]);
                }
            }
            if (EPI == EPI_BIAS_GELU && g.Y2) {          // training: pre-activation copy first
#pragma unroll
                for (int j = 0; j < 32; j += 8)
                    *reinterpret_cast<uint4*>(srow + j * 2) = make_uint4(tc::pack_bf16(v[j], v[j + 1]), tc::pack_bf16(v[j + 2], v[j + 3]),
                                                                          tc::pack_bf16(v[j + 4], v[j + 5]), tc::pack_bf16(v[j + 6], v[j + 7]));
                __syncwarp();
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const uint4 val = *reinterpret_cast<const uint4*>(sb + rl * STG_ROW + cc * 16);
                    const long long o = __shfl_sync(0xffffffffu, oy, rl);
                    if (o >= 0) *reinterpret_cast<uint4*>(g.Y2 + o + n0 + c * 32 + cc * 8) = val;
                }
                __syncwarp();
            }
            {
                uint32_t pk[16];
#pragma unroll
                for (int h = 0; h < 16; ++h) pk[h] = tc::pack_bf16(v[2 * h], v[2 * h + 1]);
                if (EPI == EPI_BIAS_GELU) {        // branch-free table GELU, one deferred range test per thread and chunk
                    uint32_t oor = 0, ge[16];
#pragma unroll
                    for (int h = 0; h < 16; ++h) ge[h] = gelu_pair_fast(gtab, pk[h], oor);
                    if (__builtin_expect(gelu_pair_oor(oor), 0)) {
#pragma unroll
                        for (int h = 0; h < 16; ++h) ge[h] = gelu_pair_exact(gtab, pk[h]);
                    }
#pragma unroll
                    for (int h = 0; h < 16; ++h) pk[h] = ge[h];
                }
                if (EPI != EPI_BIAS_RESID && ymap != nullptr) {
                    // TMA store: dense 64-byte rows, 16-byte chunks XOR-swizzled (SWIZZLE_64B) -> conflict-free row writes;
                    // one elected lane hands the 32 x 32 box to the TMA unit, nobody reads the tile back
                    if (lane == 0) tma::store_wait_read<NBUF - 1>();       // the box stored from this buffer NBUF chunks ago is drained
                    __syncwarp();
                    unsigned char* drow = sb + lane * 64;
                    const int sw = (lane >> 1) & 3;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4*>(drow + ((j ^ sw) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    tma::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma::store_2d(ymap, sb, n0 + c * 32, static_cast<int>(tile * TC_BM) + lg * 32);
                        tma::store_commit();
                    }
                    continue;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<uint4*>(srow + j * 16) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            }
            __syncwarp();
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {             // 8 rows x 64 contiguous bytes per warp instruction
                const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                const uint4 val = *reinterpret_cast<const uint4*>(sb + rl * STG_ROW + cc * 16);
                const long long o = __shfl_sync(0xffffffffu, oy, rl);
                if (o >= 0) *reinterpret_cast<uint4*>(g.Y + o + n0 + c * 32 + cc * 8) = val;
            }
            __syncwarp();                                // staging buffer reusable
        }
        if (half >= NCH) {                               // this warp owns no chunk (BN == 32): still hand back
            tc::tc_fence_before();
            mbar_arrive(&tempty[acc]);
        }
}

// BN: tile columns; KC: k-chunk (64 -> SWIZZLE_128B, 32 -> SWIZZLE_64B); CPS: k-chunks per ring stage (LN needs the
// whole row in one stage: CPS * KC == K); LN: LayerNorm prologue over the K channels of the A row.
template <int BN, int KC, int CPS, int EPI, bool LN, int NEW>
__global__ void __launch_bounds__(THREADS, 1) gemm_ws_kernel(const GemmArgs<__nv_bfloat16> g, int row_tiles, int nkc, int S,
                                                             const __grid_constant__ CUtensorMap ymap, int use_ymap) {
    using T = __nv_bfloat16;
    constexpr int NPW = WARPS - 1 - NEW;               // producer warps
    constexpr int MMA_WARP = NEW;
    constexpr int NCG = NEW / 4;                       // epilogue column groups
    static_assert(NEW % 4 == 0 && (NPW == 4 || NPW == 8), "warp split");
    constexpr int CPR = KC / 8;                        // 16-byte chunks per tile row per k-chunk
    constexpr int A_CHUNK = TC_BM * KC * 2;
    constexpr int W_CHUNK = BN * KC * 2;
    constexpr int STAGE = CPS * A_CHUNK;
    constexpr int ACC = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;   // TMEM columns per accumulator stage
    constexpr int NACC = ACC <= 128 ? 4 : 2;           // accumulator stages: narrow tiles are handshake-latency bound, give the MMA more run-ahead
    constexpr int TMEM_COLS = NACC * ACC;
    constexpr int NCH = BN / 32;                       // 32-column epilogue chunks
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(TC_BM >> 4) << 24);
    static_assert(BN % 32 == 0 && BN <= 256, "tile width");

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // align inside the shared window with pointer arithmetic only (an integer round-trip would turn every later
    // access into a generic LD/ST instead of LDS/STS)
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Ws = base;                                       // [nkc][W_CHUNK] resident
    unsigned char* As = Ws + static_cast<size_t>(nkc) * W_CHUNK;    // [S][STAGE]
    unsigned char* stg = As + static_cast<size_t>(S) * STAGE;       // [NEW][2][STG_BUF]
    float* s_bias = reinterpret_cast<float*>(stg + NEW * 2 * STG_BUF);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_bias + BN);      // [8]
    uint64_t* empty = full + 8;                                     // [8]
    uint64_t* tfull = empty + 8;                                    // [NACC]
    uint64_t* tempty = tfull + 4;                                   // [NACC]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 4);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(tmem_slot + 4);    // EPI_BIAS_GELU only

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.y * BN;
    const int SPT = nkc / CPS;                                      // ring stages per row tile
    const int my_tiles = (row_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

    // ---------------------------------------------------------------- one-time setup (all threads)
    for (int c = tid; c < nkc * BN * CPR; c += THREADS) {
        const int kc = c / (BN * CPR), rem = c - kc * (BN * CPR);
        const int r = rem / CPR, ch = rem % CPR;
        const float* src = g.Wt + static_cast<long long>(n0 + r) * g.K + kc * KC + ch * 8;
        const float4 a4 = *reinterpret_cast<const float4*>(src);
        const float4 b4 = *reinterpret_cast<const float4*>(src + 4);
        *reinterpret_cast<uint4*>(Ws + static_cast<size_t>(kc) * W_CHUNK + tc::swz_off<KC>(r, ch)) =
            make_uint4(tc::pack_bf16(a4.x, a4.y), tc::pack_bf16(a4.z, a4.w), tc::pack_bf16(b4.x, b4.y), tc::pack_bf16(b4.z, b4.w));
    }
    for (int i = tid; i < BN; i += THREADS) s_bias[i] = g.bias ? Act<T>::round(g.bias[n0 + i]) : 0.f;
    if (EPI == EPI_BIAS_GELU) gelu_tab2_to_smem(gtab, tid, THREADS);
    if (tid == 0) {
        for (int i = 0; i < S; ++i) { tc::mbar_init(&full[i], NPW * 32); tc::mbar_init(&empty[i], 1); }
        for (int i = 0; i < NACC; ++i) { tc::mbar_init(&tfull[i], 1); tc::mbar_init(&tempty[i], NEW * 32); }
        tc::fence_barrier_init();
    }
    if (warp == MMA_WARP) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::fence_proxy_async();                         // resident W tile: generic-proxy writes -> async proxy (tensor core)
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    if (warp > MMA_WARP) {
        // ============================================================ producers
        constexpr int G = CPS * CPR;                   // lanes per row (one 16-byte chunk each)
        constexpr int RPW = 32 / G;                    // rows per warp pass
        constexpr int RPP = NPW * RPW;                 // rows per pass over all producer warps
        constexpr int U = TC_BM / RPP;                 // rows (== 16-byte loads) per thread per stage
        constexpr int UB = U > 4 ? 4 : U;              // rows per register batch
        constexpr int NB = U / UB;                     // batches per stage
        const int pw = warp - (MMA_WARP + 1);
        const int gl = lane % G, sub = lane / G;
        const int kcl = gl / CPR, ch = gl % CPR;
        // running positions (no divisions in the steady state): loader and writer each walk batch -> stage -> tile
        int l_b = 0, l_st = 0;
        uint32_t l_tile = blockIdx.x;
        uint32_t wb[2] = {0u, 0u}, wy[2] = {0u, 0u}, wx[2] = {0u, 0u};
        // global address of this thread's 16-byte chunk of batch row p (nullptr: row beyond M); advance() steps to the next batch
        auto src_of = [&](int p) -> const __nv_bfloat16* {
            const uint32_t r = (l_b * UB + p) * RPP + pw * RPW + sub;
            const uint32_t m = l_tile * TC_BM + r;
            if (m >= g.M) return nullptr;
            const uint32_t hi = r >> 6;
            const uint32_t ra = g.mapA ? g.map.pixel(hi ? wb[1] : wb[0], hi ? wy[1] : wy[0], hi ? wx[1] : wx[0], r & 63u) : m;
            return g.A + static_cast<long long>(ra) * g.lda + (l_st * CPS + kcl) * KC + ch * 8;
        };
        auto decode_tile = [&]() {                     // a 128-row tile is two consecutive windows: decode the first, step once
            if (g.mapA && l_b == 0 && l_st == 0) {
                const uint32_t wg = l_tile * 2u;
                wb[0] = wg / static_cast<uint32_t>(g.map.nWin);
                const uint32_t w = wg - wb[0] * static_cast<uint32_t>(g.map.nWin);
                wy[0] = w / static_cast<uint32_t>(g.map.nWw);
                wx[0] = w - wy[0] * static_cast<uint32_t>(g.map.nWw);
                wb[1] = wb[0]; wy[1] = wy[0]; wx[1] = wx[0] + 1u;
                if (wx[1] == static_cast<uint32_t>(g.map.nWw)) {
                    wx[1] = 0u; wy[1] += 1u;
                    if (wy[1] * static_cast<uint32_t>(g.map.nWw) == static_cast<uint32_t>(g.map.nWin)) { wy[1] = 0u; wb[1] += 1u; }
                }
            }
        };
        auto advance = [&]() { if (++l_b == NB) { l_b = 0; if (++l_st == SPT) { l_st = 0; l_tile += gridDim.x; } } };
        const int total = my_tiles * SPT * NB;         // batches this CTA produces

        if constexpr (LN) {
            // ---- LayerNorm prologue: global -> register ring -> LN (row statistics by shuffles over the G lanes of the row)
            //      -> bf16 -> swizzled stage.  The UB rows of a batch are processed side by side (independent dependency
            //      chains interleave); element-wise steps are packed fp32x2.  Summation order == ln_stats_kernel's.
            constexpr int D = (UB * 2 >= 8) ? 2 : 8 / UB;   // ring depth in batches: >= 8 loads in flight per thread
            float2 gam[4], bet[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                gam[j] = make_float2(g.ln_w[gl * 8 + 2 * j], g.ln_w[gl * 8 + 2 * j + 1]);
                bet[j] = make_float2(g.ln_b[gl * 8 + 2 * j], g.ln_b[gl * 8 + 2 * j + 1]);
            }
            uint4 buf[D][UB];
            auto load = [&](uint4 (&dst)[UB], int jb) {
                if (jb >= total) return;
                decode_tile();
#pragma unroll
                for (int p = 0; p < UB; ++p) {
                    const __nv_bfloat16* src = src_of(p);
                    dst[p] = src ? *reinterpret_cast<const uint4*>(src) : make_uint4(0u, 0u, 0u, 0u);
                }
                advance();
            };
            int p_b = 0, p_s = 0;
            uint32_t p_ph = 0;
            auto process = [&](const uint4 (&src)[UB]) {
                if (p_b == 0) tc::mbar_wait(&empty[p_s], p_ph ^ 1u);     // the MMAs that read this stage last time have retired
                unsigned char* dstA = As + static_cast<size_t>(p_s) * STAGE + kcl * A_CHUNK;
                constexpr int PB = UB < 2 ? UB : 2;    // rows processed side by side (register budget: 96 per thread)
#pragma unroll
                for (int p0 = 0; p0 < UB; p0 += PB) {
                    float2 f[PB][4];
                    float sum[PB], sq[PB];
#pragma unroll
                    for (int p = 0; p < PB; ++p) {
                        const uint32_t w4[4] = {src[p0 + p].x, src[p0 + p].y, src[p0 + p].z, src[p0 + p].w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) f[p][q] = make_float2(__uint_as_float(w4[q] << 16), __uint_as_float(w4[q] & 0xFFFF0000u));
                        sum[p] = 0.f;
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int p = 0; p < PB; ++p) { sum[p] += f[p][q].x; sum[p] += f[p][q].y; }
#pragma unroll
                    for (int o = G / 2; o > 0; o >>= 1)
#pragma unroll
                        for (int p = 0; p < PB; ++p) sum[p] += __shfl_xor_sync(0xffffffffu, sum[p], o);
#pragma unroll
                    for (int p = 0; p < PB; ++p) {
                        const float nmu = -(sum[p] * (1.0f / (G * 8)));
                        const float2 nm2 = make_float2(nmu, nmu);
#pragma unroll
                        for (int q = 0; q < 4; ++q) f[p][q] = add2(f[p][q], nm2);
                        sq[p] = 0.f;
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int p = 0; p < PB; ++p) { sq[p] = fmaf(f[p][q].x, f[p][q].x, sq[p]); sq[p] = fmaf(f[p][q].y, f[p][q].y, sq[p]); }
#pragma unroll
                    for (int o = G / 2; o > 0; o >>= 1)
#pragma unroll
                        for (int p = 0; p < PB; ++p) sq[p] += __shfl_xor_sync(0xffffffffu, sq[p], o);
#pragma unroll
                    for (int p = 0; p < PB; ++p) {
                        const int r = (p_b * UB + p0 + p) * RPP + pw * RPW + sub;
                        const float rs = rsqrtf(sq[p] * (1.0f / (G * 8)) + 1e-5f);
                        const float2 rs2 = make_float2(rs, rs);
                        uint32_t o4[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float2 y2 = fma2(mul2(f[p][q], rs2), gam[q], bet[q]);
                            o4[q] = tc::pack_bf16(y2.x, y2.y);
                        }
                        *reinterpret_cast<uint4*>(dstA + tc::swz_off<KC>(r, ch)) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
                    }
                }
                if (++p_b == NB) {
                    tc::fence_proxy_async();           // my generic-proxy smem writes -> visible to the tensor core
                    mbar_arrive(&full[p_s]);
                    p_b = 0;
                    if (++p_s == S) { p_s = 0; p_ph ^= 1u; }
                }
            };
#pragma unroll
            for (int d = 0; d < D - 1; ++d) load(buf[d], d);
            for (int j0 = 0; j0 < total; j0 += D) {
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const int jb = j0 + d;
                    if (jb < total) {
                        load(buf[(d + D - 1) % D], jb + D - 1);
                        process(buf[d]);
                    }
                }
            }
        } else {
            // ---- plain bf16 operand: 16-byte cp.async straight into the swizzled stage, DD stages in flight per thread
            //      (no register staging: the in-flight depth is bounded by shared memory, not registers)
            static_assert(NB == 1, "plain operands: one batch per stage");
            const int DD = S - 1 < 4 ? S - 1 : 4;      // stages issued ahead (S >= 2)
            const uint32_t As_u = tc::smem_u32(As);
            int i_s = 0;                               // issue-side ring position
            uint32_t i_ph = 0;
            auto issue = [&](int j) {
                if (j < total) {
                    tc::mbar_wait(&empty[i_s], i_ph ^ 1u);
                    decode_tile();
#pragma unroll
                    for (int p = 0; p < UB; ++p) {
                        const int r = p * RPP + pw * RPW + sub;
                        const __nv_bfloat16* src = src_of(p);
                        cp_async16_z(As_u + i_s * STAGE + kcl * A_CHUNK + tc::swz_off<KC>(r, ch), src ? src : g.A, src != nullptr);
                    }
                    advance();
                    if (++i_s == S) { i_s = 0; i_ph ^= 1u; }
                }
                cp_async_commit();
            };
            for (int d = 0; d < DD; ++d) issue(d);
            int c_s = 0;
            for (int j = 0; j < total; ++j) {
                issue(j + DD);
                // groups complete in order: allow DD newer groups to stay in flight
                if (DD == 4) cp_async_wait<4>(); else if (DD == 3) cp_async_wait<3>(); else if (DD == 2) cp_async_wait<2>(); else cp_async_wait<1>();
                tc::fence_proxy_async();
                mbar_arrive(&full[c_s]);
                if (++c_s == S) c_s = 0;
            }
        }
    } else if (warp == MMA_WARP) {
        // ============================================================ MMA issuer (one thread)
        if (lane == 0) {
            const uint32_t As_u = tc::smem_u32(As), Ws_u = tc::smem_u32(Ws);
            int s = 0;
            uint32_t ph = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const int acc = it % NACC;
                const uint32_t aph = static_cast<uint32_t>(it / NACC) & 1u;
                tc::mbar_wait(&tempty[acc], aph ^ 1u);             // epilogue drained this accumulator
                tc::tc_fence_after();
                const uint32_t d_addr = tmem_d + static_cast<uint32_t>(acc * ACC);
                for (int st = 0; st < SPT; ++st) {
                    tc::mbar_wait(&full[s], ph);
                    tc::tc_fence_after();
#pragma unroll
                    for (int c = 0; c < CPS; ++c) {
                        const uint64_t da = tc::make_desc<KC>(As_u + s * STAGE + c * A_CHUNK);
                        const uint64_t db = tc::make_desc<KC>(Ws_u + (st * CPS + c) * W_CHUNK);
#pragma unroll
                        for (int k16 = 0; k16 < KC / 16; ++k16)
                            tc::mma_bf16(d_addr, da + 2 * k16, db + 2 * k16, IDESC, (st > 0 || c > 0 || k16 > 0) ? 1u : 0u);
                    }
                    tc::mma_commit(&empty[s]);                     // stage free once these MMAs have read it
                    if (++s == S) { s = 0; ph ^= 1u; }
                }
                tc::mma_commit(&tfull[acc]);                       // accumulator complete
            }
        }
    } else {
        // ============================================================ epilogue: thread == TMEM lane == tile row
        const int lg = warp & 3, half = warp >> 2;     // TMEM lane group, column group
        unsigned char* my_stg = stg + warp * 2 * STG_BUF;
        constexpr bool XT = (EPI == EPI_BIAS_RESID) && (BN / 32 <= NCG);
        if (XT && my_tiles > 0) {
            if (half < BN / 32) resid_prefetch<NCG>(g, blockIdx.x, n0 + half * 32, my_stg, lg, lane);
            cp_async_commit();
        }
        for (int it = 0; it < my_tiles; ++it) {
            const long long tnext = (XT && it + 1 < my_tiles) ? static_cast<long long>(blockIdx.x) + static_cast<long long>(it + 1) * gridDim.x : -1;
            epilogue_tile<BN, EPI, NCG>(g, tmem_d, it % NACC, static_cast<uint32_t>(it / NACC) & 1u, blockIdx.x + static_cast<uint32_t>(it) * gridDim.x,
                                        n0, s_bias, gtab, my_stg, tfull, tempty, lg, half, lane, tnext, it & 1, use_ymap ? &ymap : nullptr);
        }
        if (use_ymap && lane == 0) tma::store_wait_read<0>();      // my box stores have read their staging tiles
    }

    // ---------------------------------------------------------------- teardown
    tc::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

template <int BN, int KC, int CPS, int EPI, bool LN>
cudaError_t launch_inst(const GemmArgs<__nv_bfloat16>& g, int num_sms, cudaStream_t stream) {
    constexpr int A_CHUNK = TC_BM * KC * 2, W_CHUNK = BN * KC * 2, STAGE = CPS * A_CHUNK;
    const int nkc = g.K / KC;
    constexpr int NEW = 8;   // (12 + 4 measured slower for the GELU epilogue: the 4 producer warps become the bottleneck)
    const size_t fixed = fixed_smem<BN, EPI, NEW>() + static_cast<size_t>(nkc) * W_CHUNK;
    if (fixed + 2 * STAGE > SMEM_MAX) return cudaErrorInvalidConfiguration;
    int S = static_cast<int>((SMEM_MAX - fixed) / STAGE);
    if (S > 8) S = 8;
    const size_t smem = fixed + static_cast<size_t>(S) * STAGE;
    auto k = gemm_ws_kernel<BN, KC, CPS, EPI, LN, NEW>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int row_tiles = static_cast<int>((g.M + TC_BM - 1) / TC_BM);
    const int col_tiles = g.N / BN;
    int gx = num_sms / col_tiles;
    if (gx < 1) gx = 1;
    if (gx > row_tiles) gx = row_tiles;
    CUtensorMap ymap{};
    const int use_ymap = (EPI != EPI_BIAS_RESID && !g.mapY && !g.up2 && (g.ldy % 8) == 0 &&
                          tma::make_2d_bf16_store32(&ymap, g.Y, g.M, g.N, g.ldy)) ? 1 : 0;
    k<<<dim3(gx, col_tiles), THREADS, smem, stream>>>(g, row_tiles, nkc, S, ymap, use_ymap);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------------
// Streamed-W variant for the tensor-bound levels (C >= 256): the weight matrix no longer fits next to the A ring, so a
// ring stage carries one k-chunk of BOTH operands (A[128 x 64] + W[BN x 64], plain bf16 in global memory: weights
// pre-converted by convert_w_kernel, LayerNorm pre-applied by ln_apply_kernel).  Same three roles and the same
// epilogue as above; tiles are walked column-fastest so that the CTAs working on one row band share its A rows in L2.
template <int EPI> struct WssCfg {
    static constexpr int NEW = (EPI == EPI_BIAS_RESID) ? 8 : 16;     // epilogue warps (the residual prefetch needs 2 staging buffers)
    static constexpr int NBUF = (EPI == EPI_BIAS_RESID) ? 2 : 1;
    static constexpr int THREADS = (NEW + 2) * 32;                   // + MMA warp + TMA warp
};

template <int BN, int EPI>
constexpr size_t wss_fixed_smem(int N) {
    return 1024 + WssCfg<EPI>::NEW * WssCfg<EPI>::NBUF * STG_BUF + static_cast<size_t>(N) * 4 + (2 * 8 + 4) * 8 + 16 +
           (EPI == EPI_BIAS_GELU ? kGelu2TabSize * 2 : 0);
}

// Both operands arrive by TMA (one elected thread, 2 boxes per stage, SWIZZLE_128B = the UMMA layout, zero fill for the
// M tail), so no warp spends issue slots on loads: 16 epilogue warps (4 column groups) for the bias / GELU epilogues.
template <int BN, int EPI>
__global__ void __launch_bounds__(WssCfg<EPI>::THREADS, 1) gemm_wss_kernel(const GemmArgs<__nv_bfloat16> g, const __grid_constant__ CUtensorMap amap,
                                                                         const __grid_constant__ CUtensorMap wmap,
                                                                         int row_tiles, int col_tiles, int nkc, int S,
                                                                         const __grid_constant__ CUtensorMap ymap, int use_ymap) {
    using T = __nv_bfloat16;
    constexpr int NEW = WssCfg<EPI>::NEW, NBUF = WssCfg<EPI>::NBUF, THREADS_ = WssCfg<EPI>::THREADS;
    constexpr int MMA_WARP = NEW, TMA_WARP = NEW + 1, NCG = NEW / 4;
    constexpr int KC = 64;
    constexpr int A_CHUNK = TC_BM * KC * 2, W_CHUNK = BN * KC * 2, STAGE = A_CHUNK + W_CHUNK;
    constexpr int ACC = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    constexpr int TMEM_COLS = 2 * ACC;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(TC_BM >> 4) << 24);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* ring = base;                                     // [S][A_CHUNK | W_CHUNK]
    unsigned char* stg = ring + static_cast<size_t>(S) * STAGE;     // [NEW][NBUF][STG_BUF]
    float* s_bias = reinterpret_cast<float*>(stg + NEW * NBUF * STG_BUF);       // [N] (all column tiles)
    uint64_t* full = reinterpret_cast<uint64_t*>(s_bias + g.N);
    uint64_t* empty = full + 8;
    uint64_t* tfull = empty + 8;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(tmem_slot + 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int total_tiles = row_tiles * col_tiles;
    const int my_tiles = (total_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

    for (int i = tid; i < g.N; i += THREADS_) s_bias[i] = g.bias ? Act<T>::round(g.bias[i]) : 0.f;
    if (EPI == EPI_BIAS_GELU) gelu_tab2_to_smem(gtab, tid, THREADS_);
    if (tid == 0) {
        for (int i = 0; i < S; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&tfull[i], 1); tc::mbar_init(&tempty[i], NEW * 32); }
        tc::fence_barrier_init();
        tma::prefetch_map(&amap);
        tma::prefetch_map(&wmap);
    }
    if (warp == MMA_WARP) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;

    if (warp == TMA_WARP) {
        // ============================================================ producer: one thread, two TMA boxes per stage
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const int t = blockIdx.x + it * static_cast<int>(gridDim.x);
                const int rt = t / col_tiles, ct = t - rt * col_tiles;
                for (int kc = 0; kc < nkc; ++kc) {
                    tc::mbar_wait(&empty[s], ph ^ 1u);
                    tma::mbar_expect_tx(&full[s], STAGE);
                    tma::load_2d(ring + s * STAGE, &amap, &full[s], kc * KC, rt * TC_BM);
                    tma::load_2d(ring + s * STAGE + A_CHUNK, &wmap, &full[s], kc * KC, ct * BN);
                    if (++s == S) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0) {
            const uint32_t ring_u = tc::smem_u32(ring);
            int s = 0;
            uint32_t ph = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const int acc = it & 1;
                const uint32_t aph = static_cast<uint32_t>(it >> 1) & 1u;
                tc::mbar_wait(&tempty[acc], aph ^ 1u);
                tc::tc_fence_after();
                const uint32_t d_addr = tmem_d + static_cast<uint32_t>(acc * ACC);
                for (int kc = 0; kc < nkc; ++kc) {
                    tc::mbar_wait(&full[s], ph);
                    tc::tc_fence_after();
                    const uint64_t da = tc::make_desc<64>(ring_u + s * STAGE);
                    const uint64_t db = tc::make_desc<64>(ring_u + s * STAGE + A_CHUNK);
#pragma unroll
                    for (int k16 = 0; k16 < 4; ++k16) tc::mma_bf16(d_addr, da + 2 * k16, db + 2 * k16, IDESC, (kc > 0 || k16 > 0) ? 1u : 0u);
                    tc::mma_commit(&empty[s]);
                    if (++s == S) { s = 0; ph ^= 1u; }
                }
                tc::mma_commit(&tfull[acc]);
            }
        }
    } else {
        const int lg = warp & 3, half = warp >> 2;
        unsigned char* my_stg = stg + warp * NBUF * STG_BUF;
        for (int it = 0; it < my_tiles; ++it) {
            const int t = blockIdx.x + it * static_cast<int>(gridDim.x);
            const int rt = t / col_tiles, ct = t - rt * col_tiles;
            epilogue_tile<BN, EPI, NCG, NBUF, false>(g, tmem_d, it & 1, static_cast<uint32_t>(it >> 1) & 1u, static_cast<uint32_t>(rt), ct * BN,
                                              s_bias + ct * BN, gtab, my_stg, tfull, tempty, lg, half, lane, -1, 0, use_ymap ? &ymap : nullptr);
        }
        if (use_ymap && lane == 0) tma::store_wait_read<0>();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

template <int BN, int EPI>
cudaError_t wss_launch_bn(const GemmArgs<__nv_bfloat16>& g, const __nv_bfloat16* Wb, int num_sms, cudaStream_t stream) {
    constexpr int STAGE = TC_BM * 64 * 2 + BN * 64 * 2;
    const size_t fixed = wss_fixed_smem<BN, EPI>(g.N);
    if (fixed + 2 * STAGE > SMEM_MAX) return cudaErrorInvalidConfiguration;
    int S = static_cast<int>((SMEM_MAX - fixed) / STAGE);
    if (S > 8) S = 8;
    const size_t smem = fixed + static_cast<size_t>(S) * STAGE;
    CUtensorMap amap{}, wmap{};
    if (!tma::make_2d_bf16_sw128(&amap, g.A, g.M, g.K, g.lda, TC_BM) || !tma::make_2d_bf16_sw128(&wmap, Wb, g.N, g.K, g.K, BN))
        return cudaErrorNotSupported;
    auto k = gemm_wss_kernel<BN, EPI>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int row_tiles = static_cast<int>((g.M + TC_BM - 1) / TC_BM);
    const int col_tiles = g.N / BN;
    int grid = num_sms;
    if (grid > row_tiles * col_tiles) grid = row_tiles * col_tiles;
    CUtensorMap ymap{};
    const int use_ymap = (EPI != EPI_BIAS_RESID && !g.mapY && !g.up2 && (g.ldy % 8) == 0 &&
                          tma::make_2d_bf16_store32(&ymap, g.Y, g.M, g.N, g.ldy)) ? 1 : 0;
    k<<<grid, WssCfg<EPI>::THREADS, smem, stream>>>(g, amap, wmap, row_tiles, col_tiles, g.K / 64, S, ymap, use_ymap);
    return cudaGetLastError();
}

// plain bf16 operands, K % 64 == 0, N % 128 == 0, no A-row gather / scale (callers fall back to gemm_tca otherwise)
inline bool wss_supported(const GemmArgs<__nv_bfloat16>& g) {
    return !g.mapA && !g.a_row_scale && !g.aux && !g.mean && g.K % 64 == 0 && g.N % 128 == 0 && g.N <= 4096 &&
           (g.M >= 4 * TC_BM || g.up2) && (g.lda % 8) == 0 && tma::encode_fn() != nullptr;
}
// Tile width by occupancy: the widest BN whose tile count still fills the SMs.  At the deep levels of a small tile shard
// (8-GPU config 3: 1408 tokens at the bottleneck = 11 row tiles) BN = 256 left 22-66 CTAs for 148 SMs; narrower tiles give
// every SM a CTA (the A rows they share come from L2).
template <int EPI>
cudaError_t wss_launch(const GemmArgs<__nv_bfloat16>& g, const __nv_bfloat16* Wb, int num_sms, cudaStream_t stream) {
    const long long row_tiles = (g.M + TC_BM - 1) / TC_BM;
    if (g.N % 256 == 0 && row_tiles * (g.N / 256) >= num_sms) return wss_launch_bn<256, EPI>(g, Wb, num_sms, stream);
    if (row_tiles * (g.N / 128) >= num_sms || g.up2) return wss_launch_bn<128, EPI>(g, Wb, num_sms, stream);
    return wss_launch_bn<64, EPI>(g, Wb, num_sms, stream);
}


// Shapes served (everything the C <= 128 levels of the fused block path need); anything else -> caller's fallback.
//   LN + EPI_BIAS       (q|k|v)   : K = C in {32, 64, 128}, N = 3C
//   LN + EPI_BIAS_GELU  (linear1) : K = C in {32, 64, 128}, N = 4C
//   EPI_BIAS_RESID      (out, linear2): N = C in {32, 64, 128}, K in {C, 4C}
template <int EPI>
inline bool supported(const GemmArgs<__nv_bfloat16>& g, bool ln) {
    if (g.a_row_scale || g.aux) return false;
    if (g.M < 4 * TC_BM) return false;
    if (ln) {
        if (!(g.K == 32 || g.K == 64 || g.K == 128)) return false;
        if (EPI == EPI_BIAS) return g.N == 3 * g.K && !g.Y2;
        if (EPI == EPI_BIAS_GELU) return g.N == 4 * g.K;
        return false;
    }
    if (EPI != EPI_BIAS_RESID || !g.R) return false;
    if (!(g.N == 32 || g.N == 64 || g.N == 128)) return false;
    return g.K == g.N || g.K == 4 * g.N;
}

template <int EPI>
cudaError_t launch(const GemmArgs<__nv_bfloat16>& g, bool ln, int num_sms, cudaStream_t stream) {
    if constexpr (EPI == EPI_BIAS) {
        if (g.K == 32) return launch_inst<96, 32, 1, EPI_BIAS, true>(g, num_sms, stream);
        if (g.K == 64) return launch_inst<192, 64, 1, EPI_BIAS, true>(g, num_sms, stream);
        return launch_inst<192, 64, 2, EPI_BIAS, true>(g, num_sms, stream);
    } else if constexpr (EPI == EPI_BIAS_GELU) {
        if (g.K == 32) return launch_inst<128, 32, 1, EPI_BIAS_GELU, true>(g, num_sms, stream);
        if (g.K == 64) return launch_inst<256, 64, 1, EPI_BIAS_GELU, true>(g, num_sms, stream);
        return launch_inst<256, 64, 2, EPI_BIAS_GELU, true>(g, num_sms, stream);
    } else {
        if (g.N == 32 && g.K == 32) return launch_inst<32, 32, 1, EPI_BIAS_RESID, false>(g, num_sms, stream);
        if (g.N == 32) return launch_inst<32, 64, 1, EPI_BIAS_RESID, false>(g, num_sms, stream);
        if (g.N == 64) return launch_inst<64, 64, 1, EPI_BIAS_RESID, false>(g, num_sms, stream);
        return launch_inst<128, 64, 1, EPI_BIAS_RESID, false>(g, num_sms, stream);
    }
}

// Plain bf16 operand, no LayerNorm, bias-only epilogue (optionally scattered through window_reverse + un-roll): the
// data-gradient GEMMs dX = dY . W of the C <= 64 levels (N in {32, 64} or the 4C-wide dh2), weights resident in shared memory.
inline bool plain_supported(const GemmArgs<__nv_bfloat16>& g) {
    if (g.mapA || g.a_row_scale || g.aux || g.mean || g.up2 || g.Y2 || g.R) return false;
    if (g.M < 4 * TC_BM || (g.lda % 8) || (g.ldy % 8)) return false;
    if (g.N == 32) return g.K % 32 == 0 && g.K <= 256;
    if (g.N == 64) return g.K % 64 == 0 && g.K <= 512;
    if (g.N == 128) return g.K == 32;
    if (g.N == 256) return g.K == 64;
    return false;
}
inline cudaError_t launch_plain(const GemmArgs<__nv_bfloat16>& g, int num_sms, cudaStream_t stream) {
    if (g.N == 32) return launch_inst<32, 32, 1, EPI_BIAS, false>(g, num_sms, stream);
    if (g.N == 64) return launch_inst<64, 64, 1, EPI_BIAS, false>(g, num_sms, stream);
    if (g.N == 128) return launch_inst<128, 32, 1, EPI_BIAS, false>(g, num_sms, stream);
    return launch_inst<256, 64, 1, EPI_BIAS, false>(g, num_sms, stream);
}

}  // namespace ws
}  // namespace lewin
