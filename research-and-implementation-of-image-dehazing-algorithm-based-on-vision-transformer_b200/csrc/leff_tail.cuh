// The tail of LeFF as ONE kernel (bf16 inference, C in {32, 64}: the HBM-bound levels):
//
//   out = y + s_b * ( GELU( dwconv3x3( h1 ) + b_dw ) . W2^T + b2 )
//
// Reference: LeFF.forward My_model_1.py:512-531 (depthwise conv + GELU on the [B, 4C, H, W] map, linear2) and the residual /
// DropPath of LeWinTransformerBlock.forward :873.  The three-kernel pipeline writes h2 = GELU(dwconv(h1)) to HBM and reads it
// back in linear2 (8 * 4C bytes per token of the 38 C the LeFF half moves); here the depthwise kernel's output tile goes
// straight into the swizzled A operand of a tcgen05.mma and h2 never exists in global memory.
//
// One persistent CTA per SM.  Work unit = (8 x 16-pixel tile, 64-channel slab of the hidden dimension):
//
//   control thread (one per team): TMA box load of the (8+2) x (16+2) x 64 halo of h1 (zero fill == the conv's zero padding)
//        two units ahead; tcgen05.mma [128 x 64] x [64 x C] per unit into the tile's TMEM accumulator; commits;
//   2 teams x 8 conv warps: the arithmetic of dws::dwconv_stream_kernel (same tap order, same packed FFMA2, same table GELU:
//        bit-identical h2 values) with thread = (channel pair, pixel-column pair), rolling 3 x 4 register window;
//        results -> swizzled UMMA A tile (128 tokens x 64 channels);
//   4 epilogue warps: tcgen05.ld -> + b2 -> DropPath scale -> + residual (rows prefetched one tile ahead by cp.async)
//        -> staging -> row-cooperative coalesced 16-byte stores.
//
// The k-slabs of a tile are accumulated in slab order and every rounding point equals the three-kernel path's
// (dws::dwconv_stream_kernel + ws::gemm_ws_kernel<EPI_BIAS_RESID>), so the two are bit-identical (tests/test_gpu_leff_tail.py).
#pragma once
#include "tc_helpers.cuh"
#include "tma.cuh"

namespace lewin {
namespace lt {

constexpr int TY = 8, TX = 16, SLAB = 64;
constexpr int HY = TY + 2, HX = TX + 2;
constexpr int HALO_BYTES = HY * HX * SLAB * 2;          // 23040 (a multiple of 128)
constexpr int A_BYTES = 128 * SLAB * 2;                 // 16384
constexpr int TEAMS = 2, TEAM_THREADS = 256;
constexpr int EPI_WARPS = 4;
constexpr int CONV_WARP0 = EPI_WARPS;                   // warps [4, 20): conv teams
constexpr int CTRL_WARP0 = CONV_WARP0 + TEAMS * 8;      // warps 20, 21: control threads (lane 0)
constexpr int WARPS = CTRL_WARP0 + TEAMS;
constexpr int THREADS = WARPS * 32;                     // 704
constexpr int STG_ROW = 80;                             // staging row: 32 bf16 columns (64 B) + 16 B pad
constexpr int STG_BUF = 32 * STG_ROW;

struct Args {
    const __nv_bfloat16* h1;     // [B, H, W, 4C]  GELU(linear1)
    const __nv_bfloat16* resid;  // [B, H, W, C]   y (residual)
    __nv_bfloat16* out;          // [B, H, W, C]
    const float* w_dw;           // [4C, 9]
    const float* b_dw;           // [4C]
    const float* w2;             // [C, 4C]
    const float* b2;             // [C]
    const float* drop_scale;     // [B] or null
    const uint16_t* gelu_tab2;   // device address of the 8192-entry table (common.cuh)
    int B, H, W;
    int ld_out;                  // elements between consecutive output tokens (>= C; the right half of a concat buffer)
    int tiles_x, tiles_y, tiles;
};

template <int C>
struct Cfg {
    static constexpr int CH = 4 * C, NS = CH / SLAB, NCH = C / 32;
    static constexpr int W2_SLAB = C * SLAB * 2;
    static constexpr int W2_BYTES = NS * W2_SLAB;
    static constexpr int STG_BYTES = EPI_WARPS * 2 * NCH * STG_BUF;
    static constexpr int CW_BYTES = CH * 10 * 4;
    static constexpr int SMEM = 1024 + W2_BYTES + TEAMS * A_BYTES + TEAMS * 2 * HALO_BYTES + STG_BYTES + kGelu2TabSize * 2 +
                                CW_BYTES + C * 4 + 32 * 8 + 16;
    static constexpr int TMEM_COLS = 4 * C < 32 ? 32 : 4 * C;        // 2 teams x 2 accumulators x C columns
    static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS <= 512, "TMEM allocation is a power of two <= 512");
    static_assert(SMEM <= 227 * 1024, "shared memory");
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ffma2(float2& d, const float2 a, const float2 b) {
    unsigned long long dd = *reinterpret_cast<unsigned long long*>(&d);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(dd)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    d = *reinterpret_cast<float2*>(&dd);
}
__device__ __forceinline__ float2 add2(const float2 a, const float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}

template <int C>
__global__ void __launch_bounds__(THREADS, 1) leff_tail_kernel(const Args a, const __grid_constant__ CUtensorMap hmap) {
    using Cf = Cfg<C>;
    constexpr int NS = Cf::NS, NCH = Cf::NCH;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(C >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* W2s = base;                                       // [NS][C x 64] bf16, K-major SWIZZLE_128B (UMMA B operand)
    unsigned char* As = W2s + Cf::W2_BYTES;                          // [TEAMS][128 x 64] bf16, SWIZZLE_128B (UMMA A operand)
    unsigned char* halo = As + TEAMS * A_BYTES;                      // [TEAMS][2][HY][HX][64] bf16
    unsigned char* stg = halo + TEAMS * 2 * HALO_BYTES;              // [EPI_WARPS][2 sets][NCH][STG_BUF]
    uint16_t* gtab = reinterpret_cast<uint16_t*>(stg + Cf::STG_BYTES);
    float* cw = reinterpret_cast<float*>(gtab + kGelu2TabSize);      // [NS][10][64]: 9 taps + bias, bf16-rounded
    float* s_b2 = cw + Cf::CH * 10;                                  // [C]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_b2 + C);
    uint64_t* halo_full = bars;                                      // [TEAMS][2]
    uint64_t* a_full = bars + 4;                                     // [TEAMS]
    uint64_t* a_empty = bars + 6;                                    // [TEAMS]
    uint64_t* acc_full = bars + 8;                                   // [TEAMS][2]
    uint64_t* acc_empty = bars + 12;                                 // [TEAMS][2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = static_cast<int>(gridDim.x);
    // tiles of team t: (blockIdx.x * 2 + t) + k * 2G
    auto count_of = [&](int t) {
        const int first = static_cast<int>(blockIdx.x) * TEAMS + t;
        return first < a.tiles ? (a.tiles - first + TEAMS * G - 1) / (TEAMS * G) : 0;
    };
    auto decode = [&](int tile, int& b, int& ty, int& tx) {
        tx = tile % a.tiles_x;
        const int r = tile / a.tiles_x;
        ty = r % a.tiles_y;
        b = r / a.tiles_y;
    };

    // ---------------------------------------------------------------- one-time setup (all threads)
    for (int c = tid; c < NS * C * 8; c += THREADS) {                // W2 [C, 4C] fp32 -> bf16 swizzled slabs
        const int s = c / (C * 8), rem = c - s * (C * 8);
        const int r = rem >> 3, ch = rem & 7;
        const float* src = a.w2 + static_cast<long long>(r) * Cf::CH + s * SLAB + ch * 8;
        const float4 a4 = *reinterpret_cast<const float4*>(src);
        const float4 b4 = *reinterpret_cast<const float4*>(src + 4);
        *reinterpret_cast<uint4*>(W2s + s * Cf::W2_SLAB + tc::swz_off<64>(r, ch)) =
            make_uint4(tc::pack_bf16(a4.x, a4.y), tc::pack_bf16(a4.z, a4.w), tc::pack_bf16(b4.x, b4.y), tc::pack_bf16(b4.z, b4.w));
    }
    for (int i = tid; i < Cf::CH * 10; i += THREADS) {               // cw[(s * 10 + k) * 64 + c]
        const int c = i & 63, k = (i >> 6) % 10, s = i / 640;
        const int ch = s * SLAB + c;
        cw[i] = Act<__nv_bfloat16>::round(k < 9 ? a.w_dw[ch * 9 + k] : a.b_dw[ch]);
    }
    for (int i = tid; i < C; i += THREADS) s_b2[i] = Act<__nv_bfloat16>::round(a.b2[i]);
    for (int i = tid; i < kGelu2TabSize / 8; i += THREADS)
        reinterpret_cast<uint4*>(gtab)[i] = reinterpret_cast<const uint4*>(a.gelu_tab2)[i];
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) tc::mbar_init(&halo_full[i], 1);
        for (int t = 0; t < TEAMS; ++t) { tc::mbar_init(&a_full[t], TEAM_THREADS); tc::mbar_init(&a_empty[t], 1); }
        for (int i = 0; i < 4; ++i) { tc::mbar_init(&acc_full[i], 1); tc::mbar_init(&acc_empty[i], EPI_WARPS * 32); }
        tc::fence_barrier_init();
        tma::prefetch_map(&hmap);
    }
    if (warp == 0) tc::tmem_alloc<Cf::TMEM_COLS>(tmem_slot);
    tc::fence_proxy_async();                                         // resident W2: generic-proxy writes -> tensor core
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem0 = *tmem_slot;

    if (warp >= CTRL_WARP0) {
        // ============================================================ control thread of team t: TMA loads + MMA issue
        if (lane == 0) {
            const int t = warp - CTRL_WARP0;
            const int cnt = count_of(t), units = cnt * NS;
            const int first = static_cast<int>(blockIdx.x) * TEAMS + t;
            unsigned char* my_halo = halo + t * 2 * HALO_BYTES;
            auto fetch = [&](int n) {                                // halo of unit n -> buffer n & 1
                const int k = n / NS, s = n - k * NS;
                int b, ty, tx;
                decode(first + k * TEAMS * G, b, ty, tx);
                uint64_t* bar = &halo_full[t * 2 + (n & 1)];
                tma::mbar_expect_tx(bar, HALO_BYTES);
                tma::load_4d(my_halo + (n & 1) * HALO_BYTES, &hmap, bar, s * SLAB, tx * TX - 1, ty * TY - 1, b);
            };
            if (units > 0) fetch(0);
            if (units > 1) fetch(1);
            const uint32_t a_u = tc::smem_u32(As + t * A_BYTES), w_u = tc::smem_u32(W2s);
            int n = 0;
            for (int k = 0; k < cnt; ++k) {
                const int acc = k & 1;
                tc::mbar_wait(&acc_empty[t * 2 + acc], (static_cast<uint32_t>(k >> 1) & 1u) ^ 1u);   // epilogue drained this accumulator
                tc::tc_fence_after();
                const uint32_t d_addr = tmem0 + static_cast<uint32_t>((t * 2 + acc) * C);
                for (int s = 0; s < NS; ++s, ++n) {
                    tc::mbar_wait(&a_full[t], static_cast<uint32_t>(n) & 1u);      // conv of unit n done: A tile written, halo buffer read
                    tc::tc_fence_after();
                    const uint64_t da = tc::make_desc<64>(a_u), db = tc::make_desc<64>(w_u + s * Cf::W2_SLAB);
#pragma unroll
                    for (int k16 = 0; k16 < 4; ++k16) tc::mma_bf16(d_addr, da + 2 * k16, db + 2 * k16, IDESC, (s > 0 || k16 > 0) ? 1u : 0u);
                    tc::mma_commit(&a_empty[t]);                                   // A tile reusable once these MMAs have read it
                    if (n + 2 < units) fetch(n + 2);
                }
                tc::mma_commit(&acc_full[t * 2 + acc]);
            }
        }
    } else if (warp >= CONV_WARP0) {
        // ============================================================ conv teams
        const int t = (warp - CONV_WARP0) >> 3;
        const int tt = tid - (CONV_WARP0 + t * 8) * 32;              // thread in the team
        const int cp = tt & 31, pxp = tt >> 5;                       // channel pair, pixel-column pair (columns 2 pxp, 2 pxp + 1)
        const int units = count_of(t) * NS;
        const unsigned char* my_halo = halo + t * 2 * HALO_BYTES;
        unsigned char* my_A = As + t * A_BYTES;
        // A-tile byte offset of my channel pair inside a row: 16-byte chunk cp >> 2 (XOR-swizzled by the row), 4 bytes at (cp & 3) * 4
        for (int n = 0; n < units; ++n) {
            const int s = n % NS;
            float2 wk[9], bz;
            {
                const float* cws = cw + s * 640 + cp * 2;
#pragma unroll
                for (int k = 0; k < 9; ++k) wk[k] = *reinterpret_cast<const float2*>(cws + k * 64);
                bz = *reinterpret_cast<const float2*>(cws + 9 * 64);
            }
            tc::mbar_wait(&halo_full[t * 2 + (n & 1)], static_cast<uint32_t>(n >> 1) & 1u);
            const unsigned char* tile = my_halo + (n & 1) * HALO_BYTES + cp * 4;
            auto ldrow = [&](float2 (&dst)[4], int hy) {             // 4 halo columns x my channel pair of halo row hy
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t u = *reinterpret_cast<const uint32_t*>(tile + ((hy * HX + 2 * pxp + j) * SLAB) * 2);
                    dst[j] = make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
                }
            };
            float2 win[3][4];
            ldrow(win[0], 0);
            ldrow(win[1], 1);
#pragma unroll
            for (int y = 0; y < TY; ++y) {
                ldrow(win[(y + 2) % 3], y + 2);
                float2 acc0 = bz, acc1 = bz;
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        ffma2(acc0, win[(y + ky) % 3][kx], wk[ky * 3 + kx]);
                        ffma2(acc1, win[(y + ky) % 3][kx + 1], wk[ky * 3 + kx]);
                    }
                const uint32_t in0 = tc::pack_bf16(acc0.x, acc0.y), in1 = tc::pack_bf16(acc1.x, acc1.y);
                uint32_t oor = 0;
                uint32_t q0 = gelu_pair_fast(gtab, in0, oor), q1 = gelu_pair_fast(gtab, in1, oor);
                if (__builtin_expect(gelu_pair_oor(oor), 0)) { q0 = gelu_pair_exact(gtab, in0); q1 = gelu_pair_exact(gtab, in1); }
                if (y == 0) tc::mbar_wait(&a_empty[t], (static_cast<uint32_t>(n) & 1u) ^ 1u);     // the MMAs of unit n - 1 have read the A tile
                const int r0 = y * TX + 2 * pxp;
                *reinterpret_cast<uint32_t*>(my_A + tc::swz_off<64>(r0, cp >> 2) + (cp & 3) * 4) = q0;
                *reinterpret_cast<uint32_t*>(my_A + tc::swz_off<64>(r0 + 1, cp >> 2) + (cp & 3) * 4) = q1;
            }
            tc::fence_proxy_async();                                 // my A-tile writes -> visible to the tensor core
            mbar_arrive(&a_full[t]);
        }
    } else {
        // ============================================================ epilogue warps: thread == TMEM lane == tile row
        const int lg = warp;                                         // warp % 4 == TMEM lane group
        const int cnt0 = count_of(0), cnt1 = count_of(1), total = cnt0 + cnt1;
        unsigned char* my_stg = stg + warp * 2 * NCH * STG_BUF;
        const int r = lg * 32 + lane, py = r >> 4, px = r & 15;
        auto row_off = [&](int j, float* sc) -> long long {          // token index of my row of item j (or -1), DropPath scale
            const int t = j & 1, k = j >> 1;
            int b, ty, tx;
            decode(static_cast<int>(blockIdx.x) * TEAMS + t + k * TEAMS * G, b, ty, tx);
            const int gy = ty * TY + py;
            if (sc) *sc = a.drop_scale ? a.drop_scale[b] : 1.f;
            if (gy >= a.H) return -1;
            return (static_cast<long long>(b) * a.H + gy) * a.W + tx * TX + px;
        };
        auto prefetch = [&](int j) {                                 // residual rows of item j -> staging set j & 1
            const long long oy = row_off(j, nullptr);
            unsigned char* set = my_stg + (j & 1) * NCH * STG_BUF;
#pragma unroll
            for (int c = 0; c < NCH; ++c)
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const long long o = __shfl_sync(0xffffffffu, oy, rl);
                    if (o >= 0) cp_async16(set + c * STG_BUF + rl * STG_ROW + cc * 16, a.resid + o * C + c * 32 + cc * 8);
                }
        };
        if (total > 0) prefetch(0);
        cp_async_commit();
        for (int j = 0; j < total; ++j) {
            if (j + 1 < total) prefetch(j + 1);
            cp_async_commit();
            const int t = j & 1, k = j >> 1, acc = k & 1;
            float sc;
            const long long oy = row_off(j, &sc);
            tc::mbar_wait(&acc_full[t * 2 + acc], static_cast<uint32_t>(k >> 1) & 1u);
            tc::tc_fence_after();
            cp_async_wait<1>();                                      // this item's residual landed (the next one's may still fly)
            __syncwarp();
            const uint32_t t_addr = tmem0 + (static_cast<uint32_t>(lg * 32) << 16) + static_cast<uint32_t>((t * 2 + acc) * C);
            unsigned char* set = my_stg + (j & 1) * NCH * STG_BUF;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                float v[32];
                tc::tmem_ld32(t_addr + c * 32, v);
                if (c == NCH - 1) {                                  // accumulator is in registers: hand it back
                    tc::tc_fence_before();
                    mbar_arrive(&acc_empty[t * 2 + acc]);
                }
                const float2* bs2 = reinterpret_cast<const float2*>(s_b2 + c * 32);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float2 t2 = add2(make_float2(v[2 * i], v[2 * i + 1]), bs2[i]);
                    v[2 * i] = t2.x; v[2 * i + 1] = t2.y;
                }
                unsigned char* sb = set + c * STG_BUF;
                unsigned char* srow = sb + lane * STG_ROW;
#pragma unroll
                for (int i = 0; i < 32; i += 8) {
                    const uint4 rv = *reinterpret_cast<const uint4*>(srow + i * 2);
                    const uint32_t w4[4] = {rv.x, rv.y, rv.z, rv.w};
                    uint32_t o4[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float x0 = __uint_as_float(w4[e] << 16) + sc * Act<__nv_bfloat16>::round(v[i + 2 * e]);
                        const float x1 = __uint_as_float(w4[e] & 0xFFFF0000u) + sc * Act<__nv_bfloat16>::round(v[i + 2 * e + 1]);
                        o4[e] = tc::pack_bf16(x0, x1);
                    }
                    *reinterpret_cast<uint4*>(srow + i * 2) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
                }
                __syncwarp();
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {                     // 8 rows x 64 contiguous bytes per warp instruction
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const uint4 val = *reinterpret_cast<const uint4*>(sb + rl * STG_ROW + cc * 16);
                    const long long o = __shfl_sync(0xffffffffu, oy, rl);
                    if (o >= 0) *reinterpret_cast<uint4*>(a.out + o * a.ld_out + c * 32 + cc * 8) = val;
                }
            }
            __syncwarp();                                            // staging set reusable (prefetch of item j + 2)
        }
        cp_async_wait<0>();
    }

    // ---------------------------------------------------------------- teardown
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<Cf::TMEM_COLS>(tmem0);
}

inline bool supported(int C, int hidden, int B, int H, int W) {
    return (C == 32 || C == 64) && hidden == 4 * C && W % TX == 0 && H >= 1 &&
           static_cast<long long>(B) * H * W >= 4 * 128 && tma::encode_fn() != nullptr;
}

template <int C>
inline cudaError_t launch_c(Args a, int num_sms, cudaStream_t stream) {
    a.tiles_x = a.W / TX;
    a.tiles_y = (a.H + TY - 1) / TY;
    a.tiles = a.B * a.tiles_x * a.tiles_y;
    CUtensorMap map{};
    if (!tma::make_nhwc_bf16(&map, a.h1, a.B, a.H, a.W, 4 * C, HY, HX, SLAB)) return cudaErrorNotSupported;
    auto k = leff_tail_kernel<C>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<C>::SMEM);
    if (e != cudaSuccess) return e;
    int grid = (a.tiles + TEAMS - 1) / TEAMS;
    if (grid > num_sms) grid = num_sms;
    k<<<grid, THREADS, Cfg<C>::SMEM, stream>>>(a, map);
    return cudaGetLastError();
}

inline cudaError_t launch(int C, const Args& a, int num_sms, cudaStream_t stream) {
    if (C == 32) return launch_c<32>(a, num_sms, stream);
    if (C == 64) return launch_c<64>(a, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace lt
}  // namespace lewin
