// LeFF depthwise 3x3 convolution + bias + exact GELU on channel-last maps.
//
// Reference: nn.Conv2d(hidden, hidden, groups=hidden, kernel_size=3, stride=1, padding=1) + nn.GELU,
// My_model_1.py:489-491, applied at :517 over the WHOLE H x W map (zero padding at the image border;
// it crosses window borders).  The reference round-trips [B,L,4C] -> NCHW -> conv -> NHWC
// (My_model_1.py:514,520); here the map stays token-major [B,H,W,Ch] and each thread owns 4
// channels of a vertical strip of pixels with a rolling 3x3 register window (3 new 128-bit loads
// per output instead of 9).  HBM-bound: algorithmic traffic = read Ch + write Ch per pixel.
#pragma once
#include "common.cuh"
#include "dwconv_stream.cuh"

namespace lewin {

constexpr int DW_TY = 8;   // pixels per thread along y

template <typename T>
__global__ void __launch_bounds__(256) dwconv3x3_gelu_kernel(const T* __restrict__ x, T* __restrict__ out,
                                                             T* __restrict__ preact,
                                                             const float* __restrict__ w, const float* __restrict__ bias,
                                                             int B, int H, int W, int Ch) {
    const int cgs = Ch >> 2;
    const int strips = (H + DW_TY - 1) / DW_TY;
    const long long total = static_cast<long long>(B) * strips * W * cgs;
    const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (gid >= total) return;
    const int cg = static_cast<int>(gid % cgs);
    long long rest = gid / cgs;
    const int xx = static_cast<int>(rest % W);
    rest /= W;
    const int strip = static_cast<int>(rest % strips);
    const int b = static_cast<int>(rest / strips);
    const int c = cg * 4;
    const int y0 = strip * DW_TY;

    float wk[4][9];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int t = 0; t < 9; ++t) wk[i][t] = Act<T>::round(__ldg(w + (c + i) * 9 + t));   // autocast: conv weight/bias cast to bf16
    float4 bz = *reinterpret_cast<const float4*>(bias + c);
    bz.x = Act<T>::round(bz.x); bz.y = Act<T>::round(bz.y); bz.z = Act<T>::round(bz.z); bz.w = Act<T>::round(bz.w);

    const T* xb = x + static_cast<long long>(b) * H * W * Ch + c;
    auto ldpix = [&](int y, int xq) -> float4 {
        if (y < 0 || y >= H || xq < 0 || xq >= W) return make_float4(0.f, 0.f, 0.f, 0.f);
        return ld4(xb + (static_cast<long long>(y) * W + xq) * Ch);
    };
    float4 win[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        win[0][j] = ldpix(y0 - 1, xx - 1 + j);
        win[1][j] = ldpix(y0, xx - 1 + j);
    }
#pragma unroll
    for (int dy = 0; dy < DW_TY; ++dy) {
        const int y = y0 + dy;
        if (y >= H) break;
#pragma unroll
        for (int j = 0; j < 3; ++j) win[2][j] = ldpix(y + 1, xx - 1 + j);
        float4 acc = bz;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const float4 v = win[ky][kx];
                acc.x = fmaf(v.x, wk[0][ky * 3 + kx], acc.x);
                acc.y = fmaf(v.y, wk[1][ky * 3 + kx], acc.y);
                acc.z = fmaf(v.z, wk[2][ky * 3 + kx], acc.z);
                acc.w = fmaf(v.w, wk[3][ky * 3 + kx], acc.w);
            }
        if (Act<T>::kIsBf16) {
            acc.x = Act<T>::round(acc.x); acc.y = Act<T>::round(acc.y);
            acc.z = Act<T>::round(acc.z); acc.w = Act<T>::round(acc.w);
        }
        const long long o = (static_cast<long long>(b) * H * W + static_cast<long long>(y) * W + xx) * Ch + c;
        if (preact) st4(preact + o, acc);
        if (Act<T>::kIsBf16)
            st4(out + o, make_float4(gelu_tab(g_gelu_tab, acc.x), gelu_tab(g_gelu_tab, acc.y), gelu_tab(g_gelu_tab, acc.z),
                                     gelu_tab(g_gelu_tab, acc.w)));
        else
            st4(out + o, make_float4(gelu_erf(acc.x), gelu_erf(acc.y), gelu_erf(acc.z), gelu_erf(acc.w)));
#pragma unroll
        for (int j = 0; j < 3; ++j) { win[0][j] = win[1][j]; win[1][j] = win[2][j]; }
    }
}

template <typename T>
cudaError_t launch_dwconv_gelu(const T* x, T* out, T* preact, const float* w, const float* bias,
                               int B, int H, int W, int Ch, cudaStream_t stream) {
    const int strips = (H + DW_TY - 1) / DW_TY;
    const long long total = static_cast<long long>(B) * strips * W * (Ch >> 2);
    const unsigned grid = static_cast<unsigned>((total + 255) / 256);
    dwconv3x3_gelu_kernel<T><<<grid, 256, 0, stream>>>(x, out, preact, w, bias, B, H, W, Ch);
    return cudaGetLastError();
}

}  // namespace lewin

// ------------------------------------------------------------------------------------------------------------------
// Shared-memory tiled variant (used when the map is at least 8x8): a CTA stages a (8+2) x (TX+2) pixel halo tile of
// one 8-chunk channel slab (64 bf16 / 32 fp32 channels) with 16-byte cp.async (zero-filled outside the map == the
// conv's zero padding), then every thread produces 4 (TX=16) or 2 (TX=8) pixels of one 16-byte channel chunk from
// shared memory.  Global traffic is one coalesced read (+ halo from L2) and one coalesced write per element; the
// bf16 GELU is the exact 16-bit table.
namespace lewin {

__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, bool valid) {
    const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz));
}

template <typename T, int TX>
__global__ void __launch_bounds__(256) dwconv3x3_gelu_tiled_kernel(const T* __restrict__ x, T* __restrict__ out,
                                                                   T* __restrict__ preact, const float* __restrict__ w,
                                                                   const float* __restrict__ bias, int B, int H, int W, int Ch) {
    constexpr int EPC = 16 / sizeof(T);            // channels per 16-byte chunk
    constexpr int SLAB = 8 * EPC;                  // channels per CTA
    constexpr int TY = 8;
    constexpr int HX = TX + 2, HY = TY + 2;
    constexpr int PPT = TY * TX / 32;              // pixels per thread (4 or 2)
    __shared__ __align__(16) unsigned char tile[HY * HX * 8 * 16];
    __shared__ __align__(16) float ws[9 * SLAB];
    __shared__ float bs[SLAB];
    __shared__ __align__(16) uint16_t gtab[Act<T>::kIsBf16 ? kGeluTabSize : 8];

    const int tid = threadIdx.x;
    const int slabs = Ch / SLAB, tiles_x = W / TX, tiles_y = H / TY;
    int t = blockIdx.x;
    const int slab = t % slabs; t /= slabs;
    const int tx = t % tiles_x; t /= tiles_x;
    const int ty = t % tiles_y;
    const int b = t / tiles_y;
    const int c0 = slab * SLAB;
    const int y0 = ty * TY - 1, x0 = tx * TX - 1;

    for (int i = tid; i < HY * HX * 8; i += 256) {
        const int ch = i & 7, p = i >> 3;
        const int hy = p / HX, hx = p - hy * HX;
        const int yy = y0 + hy, xx = x0 + hx;
        const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
        const T* src = x + ((static_cast<long long>(b) * H + (ok ? yy : 0)) * W + (ok ? xx : 0)) * Ch + c0 + ch * EPC;
        cp_async16_zfill(tile + i * 16, src, ok);
    }
    cp_async_commit();
    for (int i = tid; i < 9 * SLAB; i += 256) {
        const int tap = i / SLAB, c = i - tap * SLAB;
        ws[i] = Act<T>::round(w[static_cast<long long>(c0 + c) * 9 + tap]);
    }
    if (tid < SLAB) bs[tid] = Act<T>::round(bias[c0 + tid]);
    if (Act<T>::kIsBf16) gelu_tab_to_smem(gtab, tid, 256);
    cp_async_wait<0>();
    __syncthreads();

    const int ch = tid & 7, lane = tid >> 3;                 // 32 pixel lanes
    const int px = lane % TX, py0 = (lane / TX) * PPT;       // column, first row of this thread's strip
    float acc[PPT][EPC];
#pragma unroll
    for (int p = 0; p < PPT; ++p)
#pragma unroll
        for (int j = 0; j < EPC; ++j) acc[p][j] = bs[ch * EPC + j];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            float wv[EPC];
#pragma unroll
            for (int j = 0; j < EPC; j += 4) {
                const float4 t4 = *reinterpret_cast<const float4*>(ws + (ky * 3 + kx) * SLAB + ch * EPC + j);
                wv[j] = t4.x; wv[j + 1] = t4.y; wv[j + 2] = t4.z; wv[j + 3] = t4.w;
            }
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const unsigned char* src = tile + (((py0 + p + ky) * HX + px + kx) * 8 + ch) * 16;
                float f[EPC];
                if (sizeof(T) == 2) {
                    const uint4 u = *reinterpret_cast<const uint4*>(src);
                    f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
                    f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
                    if (EPC == 8) {
                        f[EPC - 4] = __uint_as_float(u.z << 16); f[EPC - 3] = __uint_as_float(u.z & 0xFFFF0000u);
                        f[EPC - 2] = __uint_as_float(u.w << 16); f[EPC - 1] = __uint_as_float(u.w & 0xFFFF0000u);
                    }
                } else {
                    const float4 u = *reinterpret_cast<const float4*>(src);
                    f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
                }
#pragma unroll
                for (int j = 0; j < EPC; ++j) acc[p][j] = fmaf(f[j], wv[j], acc[p][j]);
            }
        }
#pragma unroll
    for (int p = 0; p < PPT; ++p) {
        const int yy = ty * TY + py0 + p, xx = tx * TX + px;
        const long long o = ((static_cast<long long>(b) * H + yy) * W + xx) * Ch + c0 + ch * EPC;
        if (sizeof(T) == 2) {
            uint32_t in[4], q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                __nv_bfloat162 h2 = __floats2bfloat162_rn(acc[p][2 * j], acc[p][2 * j + 1]);
                in[j] = *reinterpret_cast<uint32_t*>(&h2);
                q[j] = gelu_bits(gtab, in[j] & 0xFFFFu) | (gelu_bits(gtab, in[j] >> 16) << 16);
            }
            if (preact) *reinterpret_cast<uint4*>(preact + o) = make_uint4(in[0], in[1], in[2], in[3]);
            *reinterpret_cast<uint4*>(out + o) = make_uint4(q[0], q[1], q[2], q[3]);
        } else {
            if (preact) st4(preact + o, make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]));
            st4(out + o, make_float4(gelu_erf(acc[p][0]), gelu_erf(acc[p][1]), gelu_erf(acc[p][2]), gelu_erf(acc[p][3])));
        }
    }
}

template <typename T>
cudaError_t launch_dwconv_gelu_auto(const T* x, T* out, T* preact, const float* w, const float* bias,
                                    int B, int H, int W, int Ch, cudaStream_t stream) {
    constexpr int SLAB = 8 * (16 / sizeof(T));
    if (H % 8 == 0 && W % 8 == 0 && Ch % SLAB == 0) {
        if (W % 16 == 0) {
            const unsigned grid = static_cast<unsigned>(B) * (H / 8) * (W / 16) * (Ch / SLAB);
            dwconv3x3_gelu_tiled_kernel<T, 16><<<grid, 256, 0, stream>>>(x, out, preact, w, bias, B, H, W, Ch);
        } else {
            const unsigned grid = static_cast<unsigned>(B) * (H / 8) * (W / 8) * (Ch / SLAB);
            dwconv3x3_gelu_tiled_kernel<T, 8><<<grid, 256, 0, stream>>>(x, out, preact, w, bias, B, H, W, Ch);
        }
        return cudaGetLastError();
    }
    return launch_dwconv_gelu<T>(x, out, preact, w, bias, B, H, W, Ch, stream);
}


// ------------------------------------------------------------------------------------------------------------------
// Backward of dwconv3x3 + GELU, shared-memory tiled, split in two kernels:
//   dwconv_bwd_data_kernel : da2 = g2 * gelu'(a2) computed ONCE per element into the halo tile (and written to a
//                            global scratch for the weight kernel), dh1 = conv^T(da2, w), da1 = dh1 * gelu'(a1)
//   dwconv_bwd_wgrad_kernel: dW[c,t] += sum_p da2[p,c] * h1[p+t,c], db[c] += sum_p da2[p,c]; persistent per channel
//                            slab, register accumulators, one shuffle + shared-memory reduction per CTA.
template <typename T>
__device__ __forceinline__ void dw_unpack(const unsigned char* src, float (&f)[16 / sizeof(T)]) {
    if (sizeof(T) == 2) {
        const uint4 u = *reinterpret_cast<const uint4*>(src);
        f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xFFFF0000u);
        f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xFFFF0000u);
        constexpr int E = 16 / sizeof(T);
        f[E - 4] = __uint_as_float(u.z << 16); f[E - 3] = __uint_as_float(u.z & 0xFFFF0000u);
        f[E - 2] = __uint_as_float(u.w << 16); f[E - 1] = __uint_as_float(u.w & 0xFFFF0000u);
    } else {
        const float4 u = *reinterpret_cast<const float4*>(src);
        f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
    }
}
template <typename T>
__device__ __forceinline__ void dw_pack_store(void* dst, const float (&f)[16 / sizeof(T)]) {
    if (sizeof(T) == 2) {
        constexpr int E = 16 / sizeof(T);
        __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
        __nv_bfloat162 c = __floats2bfloat162_rn(f[E - 4], f[E - 3]), e = __floats2bfloat162_rn(f[E - 2], f[E - 1]);
        *reinterpret_cast<uint4*>(dst) = make_uint4(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b),
                                                    *reinterpret_cast<uint32_t*>(&c), *reinterpret_cast<uint32_t*>(&e));
    } else {
        *reinterpret_cast<float4*>(dst) = make_float4(f[0], f[1], f[2], f[3]);
    }
}
// gelu'(x) for the EPC values of a 16-byte chunk of pre-activations
template <typename T>
__device__ __forceinline__ void dw_gelu_grad(const unsigned char* src, const uint16_t* gtab, float (&g)[16 / sizeof(T)]) {
    constexpr int E = 16 / sizeof(T);
    if (sizeof(T) == 2) {
        const uint4 u = *reinterpret_cast<const uint4*>(src);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            g[(2 * j) % E] = gelu_grad_bits(gtab, w[j] & 0xFFFFu);
            g[(2 * j + 1) % E] = gelu_grad_bits(gtab, w[j] >> 16);
        }
    } else {
        const float4 u = *reinterpret_cast<const float4*>(src);
        g[0] = gelu_erf_grad(u.x); g[1] = gelu_erf_grad(u.y); g[2] = gelu_erf_grad(u.z); g[3] = gelu_erf_grad(u.w);
    }
}

template <typename T, int TX>
__global__ void __launch_bounds__(256) dwconv_bwd_data_kernel(const T* __restrict__ g2, const T* __restrict__ a2,
                                                              const T* __restrict__ a1, T* __restrict__ da1,
                                                              T* __restrict__ da2_out, const float* __restrict__ w,
                                                              int B, int H, int W, int Ch) {
    constexpr int EPC = 16 / sizeof(T), SLAB = 8 * EPC, TY = 8, HX = TX + 2, HY = TY + 2, PPT = TY * TX / 32;
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    unsigned char* gt = dyn_smem;                                      // g2 halo tile, then da2
    unsigned char* at = gt + HY * HX * 8 * 16;                         // a2 halo tile
    float* ws = reinterpret_cast<float*>(at + HY * HX * 8 * 16);       // [9][SLAB]
    uint16_t* gtab = reinterpret_cast<uint16_t*>(ws + 9 * SLAB);       // gelu' table (bf16 path)
    if (Act<T>::kIsBf16)
        for (int i = threadIdx.x; i < kGeluTabSize / 8; i += 256)
            reinterpret_cast<uint4*>(gtab)[i] = reinterpret_cast<const uint4*>(g_gelu_grad_tab)[i];
    const int tid = threadIdx.x;
    const int slabs = Ch / SLAB, tiles_x = W / TX, tiles_y = H / TY;
    int t = blockIdx.x;
    const int slab = t % slabs; t /= slabs;
    const int tx = t % tiles_x; t /= tiles_x;
    const int ty = t % tiles_y;
    const int b = t / tiles_y;
    const int c0 = slab * SLAB, y0 = ty * TY - 1, x0 = tx * TX - 1;
    for (int i = tid; i < HY * HX * 8; i += 256) {
        const int ch = i & 7, p = i >> 3, hy = p / HX, hx = p - hy * HX;
        const int yy = y0 + hy, xx = x0 + hx;
        const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
        const long long o = ((static_cast<long long>(b) * H + (ok ? yy : 0)) * W + (ok ? xx : 0)) * Ch + c0 + ch * EPC;
        cp_async16_zfill(gt + i * 16, g2 + o, ok);
        cp_async16_zfill(at + i * 16, a2 + o, ok);
    }
    cp_async_commit();
    for (int i = tid; i < 9 * SLAB; i += 256) {
        const int tap = i / SLAB, c = i - tap * SLAB;
        ws[i] = Act<T>::round(w[static_cast<long long>(c0 + c) * 9 + tap]);
    }
    cp_async_wait<0>();
    __syncthreads();
    // da2 = g2 * gelu'(a2), once per halo element
    for (int i = tid; i < HY * HX * 8; i += 256) {
        float gv[EPC], gg[EPC];
        dw_unpack<T>(gt + i * 16, gv);
        dw_gelu_grad<T>(at + i * 16, gtab, gg);
#pragma unroll
        for (int j = 0; j < EPC; ++j) gv[j] *= gg[j];
        dw_pack_store<T>(gt + i * 16, gv);
        const int ch = i & 7, p = i >> 3, hy = p / HX, hx = p - hy * HX;
        if (hy >= 1 && hy <= TY && hx >= 1 && hx <= TX) {
            const long long o = ((static_cast<long long>(b) * H + (y0 + hy)) * W + (x0 + hx)) * Ch + c0 + ch * EPC;
            *reinterpret_cast<uint4*>(da2_out + o) = *reinterpret_cast<const uint4*>(gt + i * 16);
        }
    }
    __syncthreads();
    const int ch = tid & 7, lane = tid >> 3;
    const int px = lane % TX, py0 = (lane / TX) * PPT;
    float acc[PPT][EPC];
#pragma unroll
    for (int p = 0; p < PPT; ++p)
#pragma unroll
        for (int j = 0; j < EPC; ++j) acc[p][j] = 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            float wv[EPC];
#pragma unroll
            for (int j = 0; j < EPC; j += 4) {
                const float4 t4 = *reinterpret_cast<const float4*>(ws + (ky * 3 + kx) * SLAB + ch * EPC + j);
                wv[j] = t4.x; wv[j + 1] = t4.y; wv[j + 2] = t4.z; wv[j + 3] = t4.w;
            }
#pragma unroll
            for (int p = 0; p < PPT; ++p) {       // dh1[y,x] = sum da2[y - ky + 1, x - kx + 1] * w[ky,kx]
                float f[EPC];
                dw_unpack<T>(gt + (((py0 + p + 2 - ky) * HX + px + 2 - kx) * 8 + ch) * 16, f);
#pragma unroll
                for (int j = 0; j < EPC; ++j) acc[p][j] = fmaf(f[j], wv[j], acc[p][j]);
            }
        }
#pragma unroll
    for (int p = 0; p < PPT; ++p) {
        const int yy = ty * TY + py0 + p, xx = tx * TX + px;
        const long long o = ((static_cast<long long>(b) * H + yy) * W + xx) * Ch + c0 + ch * EPC;
        float gg[EPC];
        dw_gelu_grad<T>(reinterpret_cast<const unsigned char*>(a1 + o), gtab, gg);
#pragma unroll
        for (int j = 0; j < EPC; ++j) acc[p][j] *= gg[j];
        dw_pack_store<T>(da1 + o, acc[p]);
    }
}

__device__ __forceinline__ float2 dw_add2(const float2 a, const float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}

// USE_TMA (bf16): each tile is TWO cp.async.bulk.tensor boxes issued by thread 0 (h1 halo box, zero-filled outside the map by
// the TMA unit = the convolution's padding; da2 interior box) completing on one mbarrier per buffer, instead of ~10 per-thread
// 16-byte cp.async with their index arithmetic (ncu: those loops were 40 % of the kernel's instructions; the box layout
// [row][column][64 channels] is exactly the layout the accumulation loop reads).
// DET: each CTA stores its sums into slab blockIdx.x of [gridDim.x][Ch, 9] / [gridDim.x][Ch] instead of adding them
template <typename T, int TX, bool USE_TMA = false, bool DET = false>
__global__ void __launch_bounds__(256, 2) dwconv_bwd_wgrad_kernel(const T* __restrict__ da2, const T* __restrict__ h1,
                                                                  float* __restrict__ dw, float* __restrict__ dbias,
                                                                  int B, int H, int W, int Ch,
                                                                  const __grid_constant__ CUtensorMap hmap,
                                                                  const __grid_constant__ CUtensorMap dmap) {
    constexpr int EPC = 16 / sizeof(T), SLAB = 8 * EPC, TY = 8, HX = TX + 2, HY = TY + 2, PPT = TY * TX / 32;
    // two buffers of (h1 halo tile, da2 interior tile): the next tile arrives (cp.async / TMA) while this one is accumulated
    constexpr int HT_BYTES = HY * HX * 8 * 16, DT_BYTES = TY * TX * 8 * 16;
    extern __shared__ __align__(128) unsigned char wg_smem_raw[];
    unsigned char* const wg_smem = USE_TMA ? wg_smem_raw + ((128u - (tma::smem_u32(wg_smem_raw) & 127u)) & 127u) : wg_smem_raw;
    unsigned char* const ht0 = wg_smem;
    unsigned char* const dt0 = wg_smem + 2 * HT_BYTES;
    uint64_t* const bars = reinterpret_cast<uint64_t*>(wg_smem + 2 * HT_BYTES + 2 * DT_BYTES);     // USE_TMA: one per buffer
    const int tid = threadIdx.x, ch = tid & 7, lane = tid >> 3;
    const int px = lane % TX, py0 = (lane / TX) * PPT;
    const int slab = blockIdx.y, c0 = slab * SLAB;
    const int tiles_x = W / TX, tiles_y = H / TY;
    const int ntiles = B * tiles_y * tiles_x;
    // accumulators as fp32 pairs: the 9 taps + the bias sum cost one fma.rn.f32x2 / add.rn.f32x2 per two channels
    // (same IEEE results as the scalar instructions, half the issue slots)
    constexpr int EP2 = EPC / 2;
    float2 wacc[9][EP2], bacc[EP2];
#pragma unroll
    for (int j = 0; j < EP2; ++j) {
        bacc[j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 9; ++t) wacc[t][j] = make_float2(0.f, 0.f);
    }
    auto issue = [&](int tile, int buf) {
        int t = tile;
        const int tx = t % tiles_x; t /= tiles_x;
        const int ty = t % tiles_y;
        const int b = t / tiles_y;
        const int y0 = ty * TY - 1, x0 = tx * TX - 1;
        unsigned char* hb = ht0 + buf * HT_BYTES;
        unsigned char* db = dt0 + buf * DT_BYTES;
        if constexpr (USE_TMA) {
            if (tid == 0) {
                tma::mbar_expect_tx(&bars[buf], HT_BYTES + DT_BYTES);
                tma::load_4d(hb, &hmap, &bars[buf], c0, x0, y0, b);
                tma::load_4d(db, &dmap, &bars[buf], c0, tx * TX, ty * TY, b);
            }
        } else {
            for (int i = tid; i < HY * HX * 8; i += 256) {
                const int c = i & 7, p = i >> 3, hy = p / HX, hx = p - hy * HX;
                const int yy = y0 + hy, xx = x0 + hx;
                const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
                const long long o = ((static_cast<long long>(b) * H + (ok ? yy : 0)) * W + (ok ? xx : 0)) * Ch + c0 + c * EPC;
                cp_async16_zfill(hb + i * 16, h1 + o, ok);
            }
            for (int i = tid; i < TY * TX * 8; i += 256) {
                const int c = i & 7, p = i >> 3, iy = p / TX, ix = p - iy * TX;
                const long long o = ((static_cast<long long>(b) * H + ty * TY + iy) * W + tx * TX + ix) * Ch + c0 + c * EPC;
                cp_async16(db + i * 16, da2 + o);
            }
            cp_async_commit();
        }
    };
    int buf = 0;
    uint32_t bphase[2] = {0u, 0u};
    if constexpr (USE_TMA) {
        if (tid == 0) {
            tma::prefetch_map(&hmap);
            tma::prefetch_map(&dmap);
            tma::mbar_init(&bars[0], 1);
            tma::mbar_init(&bars[1], 1);
            tma::fence_barrier_init();
        }
        __syncthreads();
    }
    if (static_cast<int>(blockIdx.x) < ntiles) issue(blockIdx.x, 0);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, buf ^= 1) {
        if constexpr (USE_TMA) {
            tma::mbar_wait(&bars[buf], bphase[buf]);      // both boxes of this tile have landed (visible after the wait)
            bphase[buf] ^= 1u;
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();               // this tile has landed; everyone is done with the other buffer
        if (tile + static_cast<int>(gridDim.x) < ntiles) issue(tile + gridDim.x, buf ^ 1);
        const unsigned char* ht = ht0 + buf * HT_BYTES;
        const unsigned char* dt = dt0 + buf * DT_BYTES;
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            float dv[EPC];
            dw_unpack<T>(dt + (((py0 + p) * TX + px) * 8 + ch) * 16, dv);
            float2 dv2[EP2];
#pragma unroll
            for (int j = 0; j < EP2; ++j) {
                dv2[j] = make_float2(dv[2 * j], dv[2 * j + 1]);
                bacc[j] = dw_add2(bacc[j], dv2[j]);
            }
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {   // dw[ky,kx] += da2[y,x] * h1[y + ky - 1, x + kx - 1]
                    float hv[EPC];
                    dw_unpack<T>(ht + (((py0 + p + ky) * HX + px + kx) * 8 + ch) * 16, hv);
#pragma unroll
                    for (int j = 0; j < EP2; ++j) dws::ffma2(wacc[ky * 3 + kx][j], dv2[j], make_float2(hv[2 * j], hv[2 * j + 1]));
                }
        }
    }
    // lanes tid, tid^8, tid^16, tid^24 of a warp share the channel chunk: shuffle-reduce, then across the 8 warps
    __syncthreads();
    float* red = reinterpret_cast<float*>(ht0);          // [8 warps][8 chunks][10 * EPC]
#pragma unroll
    for (int t = 0; t < 10; ++t)
#pragma unroll
        for (int j = 0; j < EPC; ++j) {
            const float2 v2 = t < 9 ? wacc[t][j >> 1] : bacc[j >> 1];
            float v = (j & 1) ? v2.y : v2.x;
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if ((tid & 31) < 8) red[(((tid >> 5) * 8 + ch) * 10 + t) * EPC + j] = v;
        }
    __syncthreads();
    for (int e = tid; e < 8 * 10 * EPC; e += 256) {
        const int c = e / (10 * EPC), rem = e - c * 10 * EPC, t = rem / EPC, j = rem - t * EPC;
        float sum = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) sum += red[((wv * 8 + c) * 10 + t) * EPC + j];
        const int cc = c0 + c * EPC + j;
        if constexpr (DET) {
            if (t < 9) dw[(static_cast<long long>(blockIdx.x) * Ch + cc) * 9 + t] = sum;
            else dbias[static_cast<long long>(blockIdx.x) * Ch + cc] = sum;
        } else {
            if (t < 9) atomicAdd(dw + static_cast<long long>(cc) * 9 + t, sum);
            else atomicAdd(dbias + cc, sum);
        }
    }
}

// the tiled kernels serve this shape (otherwise the register-window kernel dwconv_bwd_kernel runs)
inline bool dwconv_bwd_tiled_ok(int H, int W, int Ch, int elem_bytes) { return !(H % 8 || W % 8 || Ch % (8 * (16 / elem_bytes))); }
// CTAs along x of the tiled weight-gradient kernel (= its slabs in deterministic mode, with sms = 148)
inline int dwconv_bwd_wgrad_gx(int B, int H, int W, int Ch, int elem_bytes, int sms) {
    const int slabs = Ch / (8 * (16 / elem_bytes));
    const int ntiles = B * (H / 8) * (W / (W % 16 == 0 ? 16 : 8));
    int gx = (2 * sms + slabs - 1) / slabs;
    return gx > ntiles ? ntiles : gx;
}

// returns false if the shape is not covered (caller falls back to the register-window kernel).  DET: dw / dbias are the slabs
// [gx][Ch, 9] / [gx][Ch] of dwconv_bwd_wgrad_gx(.., 148), every element stored once
template <typename T, bool DET = false>
bool launch_dwconv_bwd_tiled(const T* g2, const T* a2, const T* h1, const T* a1, T* da1, T* da2_scratch, const float* w,
                             float* dw, float* dbias, int B, int H, int W, int Ch, int num_sms, cudaStream_t st,
                             cudaError_t* err) {
    constexpr int SLAB = 8 * (16 / sizeof(T));
    if (!dwconv_bwd_tiled_ok(H, W, Ch, sizeof(T))) return false;
    const int slabs = Ch / SLAB;
    const int gx = dwconv_bwd_wgrad_gx(B, H, W, Ch, sizeof(T), DET ? 148 : num_sms);
    if (W % 16 == 0) {
        if constexpr (Act<T>::kIsBf16) {      // element-wise dGELU + streaming TMA kernel (dwconv_stream.cuh; dws::supported holds here)
            *err = dws::launch_bwd_data(g2, a2, a1, da1, da2_scratch, w, B, H, W, Ch, num_sms, st);
            if (*err != cudaSuccess) return true;
        } else {
            const unsigned grid = static_cast<unsigned>(B) * (H / 8) * (W / 16) * slabs;
            constexpr int smem16 = 2 * 10 * 18 * 128 + 9 * SLAB * 4 + kGeluTabSize * 2;
            cudaFuncSetAttribute(dwconv_bwd_data_kernel<T, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem16);
            dwconv_bwd_data_kernel<T, 16><<<grid, 256, smem16, st>>>(g2, a2, a1, da1, da2_scratch, w, B, H, W, Ch);
        }
        constexpr int wg_smem16 = 2 * (10 * (16 + 2) * 128 + 8 * 16 * 128);
        CUtensorMap hmap{}, dmap{};
        bool tma_done = false;
        if constexpr (Act<T>::kIsBf16) {
            if (tma::make_nhwc_bf16(&hmap, h1, B, H, W, Ch, 10, 18, SLAB) &&
                tma::make_nhwc_bf16(&dmap, da2_scratch, B, H, W, Ch, 8, 16, SLAB)) {
                constexpr int smem_tma = wg_smem16 + 128 /*alignment*/ + 16 /*mbarriers*/;
                cudaFuncSetAttribute(dwconv_bwd_wgrad_kernel<T, 16, true, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tma);
                dwconv_bwd_wgrad_kernel<T, 16, true, DET><<<dim3(gx, slabs), 256, smem_tma, st>>>(da2_scratch, h1, dw, dbias, B, H, W, Ch,
                                                                                               hmap, dmap);
                tma_done = true;
            }
        }
        if (!tma_done) {
            cudaFuncSetAttribute(dwconv_bwd_wgrad_kernel<T, 16, false, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_smem16);
            dwconv_bwd_wgrad_kernel<T, 16, false, DET><<<dim3(gx, slabs), 256, wg_smem16, st>>>(da2_scratch, h1, dw, dbias, B, H, W, Ch,
                                                                                              hmap, dmap);
        }
    } else {
        const unsigned grid = static_cast<unsigned>(B) * (H / 8) * (W / 8) * slabs;
        constexpr int smem8 = 2 * 10 * 10 * 128 + 9 * SLAB * 4 + kGeluTabSize * 2;
        cudaFuncSetAttribute(dwconv_bwd_data_kernel<T, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem8);
        dwconv_bwd_data_kernel<T, 8><<<grid, 256, smem8, st>>>(g2, a2, a1, da1, da2_scratch, w, B, H, W, Ch);
        constexpr int wg_smem8 = 2 * (10 * (8 + 2) * 128 + 8 * 8 * 128);
        cudaFuncSetAttribute(dwconv_bwd_wgrad_kernel<T, 8, false, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_smem8);
        CUtensorMap unused{};
        dwconv_bwd_wgrad_kernel<T, 8, false, DET><<<dim3(gx, slabs), 256, wg_smem8, st>>>(da2_scratch, h1, dw, dbias, B, H, W, Ch, unused, unused);
    }
    *err = cudaGetLastError();
    return true;
}

}  // namespace lewin
