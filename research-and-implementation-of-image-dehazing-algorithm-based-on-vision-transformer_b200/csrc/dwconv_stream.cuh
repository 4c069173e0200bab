// Persistent, double-buffered depthwise 3x3 + bias + exact GELU for bf16 channel-last maps (My_model_1.py:489-491, :517).
//
// The element-wise work, not HBM, bounded the earlier kernels (dwconv.cuh): ~0.66 SM-cycles per hidden element.  This
// variant is built around the instruction count per element:
//   * persistent CTAs (2 per SM) walk 16x16-pixel x 64-channel tiles, slab-major so the 36 weights + 4 biases a thread
//     needs stay in registers until the channel slab changes; the 16 KB GELU table is staged once per CTA;
//   * the (16+2)x(16+2) halo tile of the NEXT tile is fetched with 16-byte cp.async (zero-filled outside the map ==
//     the conv's zero padding) while the current one is computed (two shared-memory buffers);
//   * thread = (4-channel group, pixel column): it walks the 16 rows with a rolling 3x3 register window, so every input
//     value is loaded from shared memory and unpacked once per thread-row (3 LDS.64 + 12 unpacks per 4 outputs) and the
//     36 MACs are 18 packed FFMA2;
//   * GELU is the branch-free pair lookup (common.cuh) with one deferred range test per 4 outputs;
//   * a warp stores 2 pixels x 128 contiguous bytes per instruction.
// Algorithmic HBM traffic: read Ch + write Ch per pixel (the halo re-reads hit L2).
#pragma once
#include <type_traits>
#include "common.cuh"
#include "tma.cuh"

namespace lewin {
namespace dws {

constexpr int TY = 16, TX = 16, SLAB = 64;
constexpr int HY = TY + 2, HX = TX + 2;
constexpr int TILE_BYTES = HY * HX * SLAB * 2;            // 41472
constexpr int THREADS = 256;
constexpr size_t SMEM = 128 /*align*/ + 2 * TILE_BYTES + kGelu2TabSize * 2 + 64 /*mbarriers*/;

__device__ __forceinline__ void ffma2(float2& d, const float2 a, const float2 b) {
    unsigned long long dd = *reinterpret_cast<unsigned long long*>(&d);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(dd)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    d = *reinterpret_cast<float2*>(&dd);
}
__device__ __forceinline__ void cp16z(uint32_t smem_addr, const void* gmem, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr), "l"(gmem), "r"(sz));
}

struct Args {
    const __nv_bfloat16* x;      // [B, H, W, Ch]
    __nv_bfloat16* out;          // [B, H, W, Ch]
    __nv_bfloat16* preact;       // optional pre-GELU copy (training), may be null
    const __nv_bfloat16* aux;    // BWD mode: a1 (pre-GELU linear1 output), da1 = conv^T(da2) * gelu'(a1)
    const float* w;              // [Ch, 9]
    const float* bias;           // [Ch]
    int B, H, W, Ch;
    int tiles_x, tiles_y, spatial_tiles, total_tiles;
};

// USE_TMA: the halo tile is ONE cp.async.bulk.tensor box per tile (issued by thread 0, zero-filled outside the map by
// the TMA unit, completion on an mbarrier) instead of 2592 per-thread 16-byte cp.async with their index arithmetic.
// BWD: the same pipeline computes the data gradient of the depthwise conv: x = da2, taps flipped, no bias, and the
// epilogue multiplies by gelu'(a1) instead of applying GELU (da1 = conv^T(da2) * gelu'(a1), autograd of :508-517).
template <bool USE_TMA, bool BWD = false>
__global__ void __launch_bounds__(THREADS, 2) dwconv_stream_kernel(const Args a, const __grid_constant__ CUtensorMap xmap) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((128u - (tma::smem_u32(smem_raw) & 127u)) & 127u);
    uint16_t* gtab = reinterpret_cast<uint16_t*>(smem + 2 * TILE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * TILE_BYTES + kGelu2TabSize * 2);
    const uint32_t smem_u = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
    const int tid = threadIdx.x;
    const int cq = tid & 15, px = tid >> 4;                // 4-channel group, pixel column

    auto decode = [&](int t, int& slab, int& b, int& ty, int& tx) {
        slab = t / a.spatial_tiles;
        int r = t - slab * a.spatial_tiles;
        tx = r % a.tiles_x; r /= a.tiles_x;
        ty = r % a.tiles_y;
        b = r / a.tiles_y;
    };
    auto fetch = [&](int t, int bufi) {
        int slab, b, ty, tx;
        decode(t, slab, b, ty, tx);
        if constexpr (USE_TMA) {
            if (tid == 0) {
                tma::mbar_expect_tx(&bars[bufi], TILE_BYTES);
                tma::load_4d(smem + bufi * TILE_BYTES, &xmap, &bars[bufi], slab * SLAB, tx * TX - 1, ty * TY - 1, b);
            }
            return;
        }
        const int y0 = ty * TY - 1, x0 = tx * TX - 1;
        const __nv_bfloat16* src0 = a.x + static_cast<long long>(b) * a.H * a.W * a.Ch + slab * SLAB;
        const uint32_t dst0 = smem_u + bufi * TILE_BYTES;
        for (int i = tid; i < HY * HX * 8; i += THREADS) {
            const int ch = i & 7, p = i >> 3;
            const int hy = p / HX, hx = p - hy * HX;
            const int yy = y0 + hy, xx = x0 + hx;
            const bool ok = yy >= 0 && yy < a.H && xx >= 0 && xx < a.W;
            cp16z(dst0 + i * 16, src0 + (static_cast<long long>(ok ? yy : 0) * a.W + (ok ? xx : 0)) * a.Ch + ch * 8, ok);
        }
    };

    if constexpr (USE_TMA) {
        if (tid == 0) {
            tma::prefetch_map(&xmap);
            tma::mbar_init(&bars[0], 1);
            tma::mbar_init(&bars[1], 1);
            tma::fence_barrier_init();
        }
        __syncthreads();
    }
    int t = blockIdx.x;
    if (t < a.total_tiles) fetch(t, 0);
    cp_async_commit();
    if constexpr (BWD) gelu_grad_tab2_to_smem(gtab, tid, THREADS); else gelu_tab2_to_smem(gtab, tid, THREADS);
    uint32_t bphase[2] = {0u, 0u};

    float2 wk[9][2];                                       // taps x channel pairs (autocast: bf16-rounded weights)
    float2 bz[2];
    int cur_slab = -1;
    bool cur_slab_first = true;
    int bufi = 0;
    for (; t < a.total_tiles; t += gridDim.x, bufi ^= 1) {
        const int tn = t + gridDim.x;
        if (tn < a.total_tiles) fetch(tn, bufi ^ 1);
        cp_async_commit();
        int slab, b, ty, tx;
        decode(t, slab, b, ty, tx);
        if (slab != cur_slab) {
            cur_slab = slab;
            const int c = slab * SLAB + cq * 4;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                wk[k][0] = make_float2(Act<__nv_bfloat16>::round(__ldg(a.w + (c + 0) * 9 + k)), Act<__nv_bfloat16>::round(__ldg(a.w + (c + 1) * 9 + k)));
                wk[k][1] = make_float2(Act<__nv_bfloat16>::round(__ldg(a.w + (c + 2) * 9 + k)), Act<__nv_bfloat16>::round(__ldg(a.w + (c + 3) * 9 + k)));
            }
            if constexpr (BWD) {
                bz[0] = make_float2(0.f, 0.f); bz[1] = bz[0];
            } else {
                const float4 b4 = *reinterpret_cast<const float4*>(a.bias + c);
                bz[0] = make_float2(Act<__nv_bfloat16>::round(b4.x), Act<__nv_bfloat16>::round(b4.y));
                bz[1] = make_float2(Act<__nv_bfloat16>::round(b4.z), Act<__nv_bfloat16>::round(b4.w));
            }
        }
        if constexpr (USE_TMA) {
            tma::mbar_wait(&bars[bufi], bphase[bufi]);         // this tile's box has landed (async proxy -> visible after the wait)
            bphase[bufi] ^= 1u;
            if (cur_slab_first) { __syncthreads(); cur_slab_first = false; }   // GELU table staged by all threads
        } else {
            cp_async_wait<1>();                            // this tile's halo has landed (the next one may still fly)
            __syncthreads();
        }

        const unsigned char* tile = smem + bufi * TILE_BYTES + cq * 8;
        auto ldrow = [&](float2 (&dst)[3][2], int hy) {    // 3 columns x 4 channels of halo row hy
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const uint2 u = *reinterpret_cast<const uint2*>(tile + ((hy * HX + px + j) * SLAB) * 2);
                dst[j][0] = make_float2(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u));
                dst[j][1] = make_float2(__uint_as_float(u.y << 16), __uint_as_float(u.y & 0xFFFF0000u));
            }
        };
        float2 win[3][3][2];                               // [row][col][channel pair]
        ldrow(win[0], 0);
        ldrow(win[1], 1);
        const long long obase = ((static_cast<long long>(b) * a.H + ty * TY) * a.W + tx * TX + px) * a.Ch + slab * SLAB + cq * 4;
        const long long rstride = static_cast<long long>(a.W) * a.Ch;
        __nv_bfloat16* op = a.out + obase;
        __nv_bfloat16* pp = a.preact ? a.preact + obase : nullptr;
        const __nv_bfloat16* ap = BWD ? a.aux + obase : nullptr;
        const int rows_here = (tx * TX + px < a.W) ? a.H - ty * TY : 0;   // < TY in the last tile row of a map whose height is not a
                                                           // multiple of 16; 0 for the columns beyond a map narrower than the tile (W = 8)
        // BWD: this thread's pre-activations a1 of all TY rows are requested up front (the loop's early exit keeps the compiler
        // from hoisting them, and a dependent global load per row was the critical path of the backward pass)
        uint2 pav[BWD ? TY : 1];
        if constexpr (BWD) {
#pragma unroll
            for (int y = 0; y < TY; ++y)
                pav[y] = y < rows_here ? __ldg(reinterpret_cast<const uint2*>(ap + y * rstride)) : make_uint2(0u, 0u);
        }
#pragma unroll
        for (int y = 0; y < TY; ++y) {
            if (y >= rows_here) break;                     // (the rows below the map were zero-filled: nothing to compute or store)
            ldrow(win[(y + 2) % 3], y + 2);
            float2 acc0 = bz[0], acc1 = bz[1];
            if constexpr (BWD) {
                // dh1[y,x] = sum_{ky,kx} da2[y - ky + 1, x - kx + 1] * w[ky,kx]  (same summation order as dwconv_bwd_data_kernel)
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        ffma2(acc0, win[(y + 2 - ky) % 3][2 - kx][0], wk[ky * 3 + kx][0]);
                        ffma2(acc1, win[(y + 2 - ky) % 3][2 - kx][1], wk[ky * 3 + kx][1]);
                    }
                const uint2 pa = pav[y];
                uint32_t oor = 0;
                uint32_t g0 = gelu_pair_fast(gtab, pa.x, oor), g1 = gelu_pair_fast(gtab, pa.y, oor);     // gtab holds gelu' here
                if (__builtin_expect(gelu_pair_oor(oor), 0)) { g0 = gelu_grad_pair_exact(gtab, pa.x); g1 = gelu_grad_pair_exact(gtab, pa.y); }
                __nv_bfloat162 h0 = __floats2bfloat162_rn(acc0.x * __uint_as_float(g0 << 16), acc0.y * __uint_as_float(g0 & 0xFFFF0000u));
                __nv_bfloat162 h1 = __floats2bfloat162_rn(acc1.x * __uint_as_float(g1 << 16), acc1.y * __uint_as_float(g1 & 0xFFFF0000u));
                *reinterpret_cast<uint2*>(op) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
                op += rstride;
            } else {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        ffma2(acc0, win[(y + ky) % 3][kx][0], wk[ky * 3 + kx][0]);
                        ffma2(acc1, win[(y + ky) % 3][kx][1], wk[ky * 3 + kx][1]);
                    }
                __nv_bfloat162 h0 = __floats2bfloat162_rn(acc0.x, acc0.y), h1 = __floats2bfloat162_rn(acc1.x, acc1.y);
                const uint32_t in0 = *reinterpret_cast<uint32_t*>(&h0), in1 = *reinterpret_cast<uint32_t*>(&h1);
                uint32_t oor = 0;
                uint32_t q0 = gelu_pair_fast(gtab, in0, oor), q1 = gelu_pair_fast(gtab, in1, oor);
                if (__builtin_expect(gelu_pair_oor(oor), 0)) { q0 = gelu_pair_exact(gtab, in0); q1 = gelu_pair_exact(gtab, in1); }
                if (pp) { *reinterpret_cast<uint2*>(pp) = make_uint2(in0, in1); pp += rstride; }
                *reinterpret_cast<uint2*>(op) = make_uint2(q0, q1);
                op += rstride;
            }
        }
        __syncthreads();                                   // every thread is done with this buffer before it is refilled
    }
}


// A tensor-core variant of this kernel (9 taps as mma.m16n8k8 with diag(w) B fragments) was built and measured in round 1:
// 0.43 instead of 0.66 warp-instructions per output, identical results, but 1.5x SLOWER (LSU data pipe 71 %: the fragment
// layout costs 16 wavefronts per STG.64 and the GELU table lookups are unchanged) - profiles/r1_h_ncu_dwconv_mma_negative_result.txt.
// The code was removed in round 2; the conclusion stands: this kernel is bound by the GELU lookups' LSU traffic, not the MACs.

inline bool supported(int H, int W, int Ch) {
    return H >= 1 && W >= TX && W % 8 == 0 && Ch % SLAB == 0;   // any height; widths that are not a multiple of the tile are cut at the edge (an 8-wide map would waste half of every tile: first-generation kernel)
}

template <bool BWD>
inline cudaError_t launch_mode(const __nv_bfloat16* x, __nv_bfloat16* out, __nv_bfloat16* preact, const __nv_bfloat16* aux, const float* w,
                               const float* bias, int B, int H, int W, int Ch, int num_sms, cudaStream_t stream) {
    Args a{};
    a.x = x; a.out = out; a.preact = preact; a.aux = aux; a.w = w; a.bias = bias;
    a.B = B; a.H = H; a.W = W; a.Ch = Ch;
    a.tiles_x = (W + TX - 1) / TX; a.tiles_y = (H + TY - 1) / TY;
    a.spatial_tiles = B * a.tiles_x * a.tiles_y;
    a.total_tiles = a.spatial_tiles * (Ch / SLAB);
    int grid = 2 * num_sms;
    if (grid > a.total_tiles) grid = a.total_tiles;
    CUtensorMap map{};
    if (tma::make_nhwc_bf16(&map, x, B, H, W, Ch, HY, HX, SLAB)) {
        cudaError_t e = cudaFuncSetAttribute(dwconv_stream_kernel<true, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SMEM));
        if (e != cudaSuccess) return e;
        dwconv_stream_kernel<true, BWD><<<grid, THREADS, SMEM, stream>>>(a, map);
    } else {
        cudaError_t e = cudaFuncSetAttribute(dwconv_stream_kernel<false, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SMEM));
        if (e != cudaSuccess) return e;
        dwconv_stream_kernel<false, BWD><<<grid, THREADS, SMEM, stream>>>(a, map);
    }
    return cudaGetLastError();
}

inline cudaError_t launch(const __nv_bfloat16* x, __nv_bfloat16* out, __nv_bfloat16* preact, const float* w, const float* bias,
                          int B, int H, int W, int Ch, int num_sms, cudaStream_t stream) {
    return launch_mode<false>(x, out, preact, nullptr, w, bias, B, H, W, Ch, num_sms, stream);
}

// ---- backward, data path:  da2 = g2 * gelu'(a2) (element-wise, also the weight-gradient kernel's input), then
//      da1 = conv^T(da2) * gelu'(a1) on the streaming kernel above
__global__ void __launch_bounds__(256) dgelu_mul_kernel(const __nv_bfloat16* __restrict__ g2, const __nv_bfloat16* __restrict__ a2,
                                                        __nv_bfloat16* __restrict__ da2, long long n8) {
    __shared__ __align__(16) uint16_t gtab[kGelu2TabSize];
    gelu_grad_tab2_to_smem(gtab, threadIdx.x, 256);
    __syncthreads();
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<long long>(gridDim.x) * 256) {
        const uint4 g = reinterpret_cast<const uint4*>(g2)[i];
        const uint4 p = reinterpret_cast<const uint4*>(a2)[i];
        const uint32_t gw[4] = {g.x, g.y, g.z, g.w}, pw[4] = {p.x, p.y, p.z, p.w};
        uint32_t o[4], oor = 0, d[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) d[j] = gelu_pair_fast(gtab, pw[j], oor);
        if (__builtin_expect(gelu_pair_oor(oor), 0)) {
#pragma unroll
            for (int j = 0; j < 4; ++j) d[j] = gelu_grad_pair_exact(gtab, pw[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(gw[j] << 16) * __uint_as_float(d[j] << 16),
                                                     __uint_as_float(gw[j] & 0xFFFF0000u) * __uint_as_float(d[j] & 0xFFFF0000u));
            o[j] = *reinterpret_cast<uint32_t*>(&h);
        }
        reinterpret_cast<uint4*>(da2)[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

inline cudaError_t launch_bwd_data(const __nv_bfloat16* g2, const __nv_bfloat16* a2, const __nv_bfloat16* a1, __nv_bfloat16* da1,
                                   __nv_bfloat16* da2, const float* w, int B, int H, int W, int Ch, int num_sms, cudaStream_t stream) {
    const long long n8 = static_cast<long long>(B) * H * W * Ch / 8;
    long long grid = static_cast<long long>(num_sms) * 8;
    if (grid > (n8 + 255) / 256) grid = (n8 + 255) / 256;
    dgelu_mul_kernel<<<static_cast<unsigned>(grid), 256, 0, stream>>>(g2, a2, da2, n8);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_mode<true>(da2, da1, nullptr, a1, w, nullptr, B, H, W, Ch, num_sms, stream);
}

}  // namespace dws
}  // namespace lewin
