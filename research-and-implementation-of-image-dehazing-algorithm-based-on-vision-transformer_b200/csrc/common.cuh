// Shared device helpers for the sm_100a LeWin kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <atomic>
#include <mutex>

namespace lewin {

constexpr int kWin = 8;
constexpr int kTok = 64;
constexpr int kTopU = 25;
constexpr int kSampleK = 25;
constexpr int kHeadDim = 32;      // head_dim of the embed_dim = 32 model (the register-resident bf16 kernels are specialised for it)
// head_dim = C / nH as ProbSparse/attn.py:370-372 derives it; {32, 64, 128} are built (BASELINE config 5: embed_dim 32-128)
inline bool head_dim_ok(int C, int nH) {
    if (nH <= 0 || C % nH) return false;
    const int d = C / nH;
    return d == 32 || d == 64 || d == 128;
}

// ---------------------------------------------------------------- activation dtype traits
template <typename T> struct Act;
template <> struct Act<float> {
    static constexpr int kPasses = 3;           // 3xTF32 error-compensated MMA
    static constexpr bool kIsBf16 = false;
    __device__ static __forceinline__ float ld(const float* p) { return *p; }
    __device__ static __forceinline__ void st(float* p, float v) { *p = v; }
    __device__ static __forceinline__ float round(float v) { return v; }
};
template <> struct Act<__nv_bfloat16> {
    static constexpr int kPasses = 1;           // bf16 values are exact in TF32
    static constexpr bool kIsBf16 = true;
    __device__ static __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
    __device__ static __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
    __device__ static __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

// 4 consecutive activations <-> float4 (16-byte load for fp32, 8-byte for bf16)
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
    uint2 u = *reinterpret_cast<const uint2*>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&a);
    u.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ void st2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
__device__ __forceinline__ void st2(__nv_bfloat16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}
__device__ __forceinline__ float2 ld2(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ float2 ld2(const __nv_bfloat16* p) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}

// ---------------------------------------------------------------- TF32 tensor-core MMA
__device__ __forceinline__ uint32_t f2tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

// D(16x8) += A(16x8, row) * B(8x8, col), tf32 inputs, fp32 accumulate.
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// Split an fp32 value into tf32 hi + tf32 lo (x ~= hi + lo to ~2^-22 relative).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = f2tf32(x);
    lo = f2tf32(x - __uint_as_float(hi));
}

// Error-compensated product: PASSES == 3 -> a_hi*b_hi + a_hi*b_lo + a_lo*b_hi (small terms first);
// PASSES == 1 -> a_hi*b_hi only (exact when the operands are bf16-valued).
template <int PASSES>
__device__ __forceinline__ void mma_x(float (&d)[4], const float (&a)[4], const float (&b)[2]) {
    uint32_t ah[4], bh[2];
    if (PASSES == 3) {
        uint32_t al[4], bl[2];
#pragma unroll
        for (int i = 0; i < 4; ++i) split_tf32(a[i], ah[i], al[i]);
#pragma unroll
        for (int i = 0; i < 2; ++i) split_tf32(b[i], bh[i], bl[i]);
        mma_tf32(d, al, bh);
        mma_tf32(d, ah, bl);
        mma_tf32(d, ah, bh);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) ah[i] = f2tf32(a[i]);
#pragma unroll
        for (int i = 0; i < 2; ++i) bh[i] = f2tf32(b[i]);
        mma_tf32(d, ah, bh);
    }
}

// ---------------------------------------------------------------- cp.async
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// ---------------------------------------------------------------- math
__device__ __forceinline__ float gelu_erf(float x) {      // nn.GELU() exact form (My_model_1.py:487-491)
    return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
    return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.39894228040143267794f * __expf(-0.5f * x * x);
}

// GELU for bf16 outputs: erf by Abramowitz-Stegun 7.1.26 (|err| <= 1.5e-7, far below a bf16 ulp) with one
// MUFU.RCP and one MUFU.EX2 instead of the ~45-instruction erff; the fp32 path keeps erff.
__device__ __forceinline__ float gelu_fast(float x) {
    const float z = fabsf(x) * 0.70710678118654752440f;
    const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    const float e = 1.0f - p * t * __expf(-z * z);      // erf(|x|/sqrt2)
    return 0.5f * x + 0.5f * fabsf(x) * e;
}

// exp(x - mx) for the softmaxes of the bf16 core kernels: one FFMA + one MUFU.EX2 (ftz).  __expf() costs 3 FMUL + FSETP +
// MUFU because the non-ftz ex2 rescales around denormal results, which are below a bf16 ulp of any probability here.
__device__ __forceinline__ float exp_sub(float x, float mxl2 /* mx * log2(e) */) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaf(x, 1.4426950408889634f, -mxl2)));
    return r;
}

// ---------------------------------------------------------------- exact bf16 GELU by table
// In the bf16 path GELU always acts on a value that was just rounded to bf16 (the linear / conv output), and its
// result is rounded to bf16 again, so it is a 16-bit -> 16-bit function.  Outside 2^-12 <= |x| < 16 the result is
// 0.5*x (correction below a quarter ulp), x, or -0; inside, 16 exponents x 128 mantissas x 2 signs = 4096 entries
// (8 KB) hold bf16(gelu_erf(x)) exactly as torch computes it (fp32 erf, one rounding).  A lookup costs ~8 ALU
// instructions + one shared-memory load instead of ~45 (erff) — the element-wise GELUs, not the GEMMs, are the
// instruction bottleneck of LeFF on B200.
constexpr int kGeluTabSize = 4096;
constexpr int kGelu2TabSize = 8192;                    // wide table (below)
constexpr uint32_t kGelu2Base = 99u << 7;              // bf16 bits of 2^-28
#ifndef LEWIN_TU_LITE      // the GELU tables and their (non-template) kernels belong to ONE translation unit: lewin_abi.cu
__device__ uint16_t g_gelu_tab[kGeluTabSize];
__device__ uint16_t g_gelu_grad_tab[kGeluTabSize];     // bf16(gelu'(x)) on the same index space (backward, bf16 path)

// Wide table for the branch-free pair lookup below: 32 binades (2^-28 <= |x| < 16) x 128 mantissas x 2 signs =
// 8192 entries (16 KB), index = (|x| bits - 0x3180) | sign << 12.  With 2^-28 as the lower edge an out-of-table
// element is a once-per-billions event for activations, so the range check is deferred to one test per thread and
// chunk (OR of the biased magnitudes) and the exact slow path (gelu_bits) is practically never taken.
__device__ uint16_t g_gelu_tab2[kGelu2TabSize];
__device__ uint16_t g_gelu_grad_tab2[kGelu2TabSize];   // bf16(gelu'(x)) on the same index space (backward)

__global__ void gelu_tab_init_kernel() {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kGelu2TabSize) {
        const uint32_t sign2 = (i >> 12) & 1, em = kGelu2Base + (i & 4095);
        const float x2 = __uint_as_float((sign2 << 31) | (em << 16));
        g_gelu_tab2[i] = __bfloat16_as_ushort(__float2bfloat16_rn(gelu_erf(x2)));
        g_gelu_grad_tab2[i] = __bfloat16_as_ushort(__float2bfloat16_rn(gelu_erf_grad(x2)));
    }
    if (i >= kGeluTabSize) return;
    const uint32_t sign = (i >> 11) & 1, e = 115 + ((i >> 7) & 15), m = i & 127;
    const float x = __uint_as_float((sign << 31) | (e << 23) | (m << 16));
    g_gelu_tab[i] = __bfloat16_as_ushort(__float2bfloat16_rn(gelu_erf(x)));
    g_gelu_grad_tab[i] = __bfloat16_as_ushort(__float2bfloat16_rn(gelu_erf_grad(x)));
}
// The tables are constants of the library: they are filled ONCE per device (round 1 relaunched the fill in front of every
// LeFF call: 18 launches per forward).  state 0 = never launched, 1 = launched, completion event pending, 2 = complete.
// A caller whose stream is being captured into a CUDA graph before the tables are complete gets the (idempotent) fill
// captured into its graph instead; other streams are ordered behind the first fill by its event.
struct GeluTabInit { std::atomic<int> state{0}; cudaEvent_t ev{nullptr}; std::mutex mu; };
inline GeluTabInit& gelu_tab_state(int dev) { static GeluTabInit st[64]; return st[dev & 63]; }
inline cudaError_t launch_gelu_tab_init(cudaStream_t st) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    GeluTabInit& g = gelu_tab_state(dev);
    if (g.state.load(std::memory_order_acquire) == 2) return cudaSuccess;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    e = cudaStreamIsCapturing(st, &cs);
    if (e != cudaSuccess) return e;
    if (cs != cudaStreamCaptureStatusNone) {              // inside a capture: keep the graph self-contained
        gelu_tab_init_kernel<<<kGelu2TabSize / 256, 256, 0, st>>>();
        return cudaGetLastError();
    }
    std::lock_guard<std::mutex> lk(g.mu);
    const int s = g.state.load(std::memory_order_acquire);
    if (s == 2) return cudaSuccess;
    if (s == 1) {
        if (cudaEventQuery(g.ev) == cudaSuccess) { g.state.store(2, std::memory_order_release); return cudaSuccess; }
        (void)cudaGetLastError();                         // cudaErrorNotReady is not sticky, clear it
        return cudaStreamWaitEvent(st, g.ev, 0);
    }
    gelu_tab_init_kernel<<<kGelu2TabSize / 256, 256, 0, st>>>();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = cudaEventCreateWithFlags(&g.ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return e;
    e = cudaEventRecord(g.ev, st);
    if (e != cudaSuccess) return e;
    g.state.store(1, std::memory_order_release);
    return cudaSuccess;
}
__device__ __forceinline__ void gelu_tab_to_smem(uint16_t* dst, int tid, int nthreads) {
    for (int i = tid; i < kGeluTabSize / 8; i += nthreads)
        reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(g_gelu_tab)[i];
}
#endif  // LEWIN_TU_LITE
// bf16 bits of GELU(x) for x given as bf16 bits.  Fast path (2^-12 <= |x| < 16): 5 integer ops + one 16-bit load;
// the out-of-range cases are rare (|x| < 2.4e-4 or >= 16) and take a divergent slow path.
__device__ __forceinline__ uint32_t gelu_bits(const uint16_t* __restrict__ tab, uint32_t u) {
    const uint32_t r = (u & 0x7FFFu) - 0x3980u;                    // |x| bits relative to 2^-12 (exponent 115)
    if (__builtin_expect(r < 2048u, 1)) return tab[r + ((u >> 15) << 11)];
    if (static_cast<int32_t>(r) < 0)                               // tiny: 0.5 * x (last binades flush to signed zero)
        return ((u & 0x7F80u) > 0x0080u) ? (u - 0x80u) : (u & 0x8000u);
    return (u & 0x8000u) ? 0x8000u : u;                            // huge: x, or -0 for negative x
}
#ifndef LEWIN_TU_LITE
__device__ __forceinline__ void gelu_tab2_to_smem(uint16_t* dst, int tid, int nthreads) {
    for (int i = tid; i < kGelu2TabSize / 8; i += nthreads)
        reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(g_gelu_tab2)[i];
}
#endif
// Packed pair: bf16x2 bits in -> bf16x2 bits of GELU out, ~7 ALU instructions + one 16-bit shared load per element and
// no branch.  `oor` accumulates the biased magnitudes: (oor >> 12) != 0 afterwards means some element handled by this
// thread was outside the table and the caller must redo its elements with gelu_pair_exact.
__device__ __forceinline__ uint32_t gelu_pair_fast(const uint16_t* __restrict__ tab2, uint32_t in2, uint32_t& oor) {
    // both halves at once: biased magnitudes (a borrow out of the low half only happens when that half is out of range,
    // and then the whole pair is redone exactly), sign bits moved to bit 12 of each half
    const uint32_t t = (in2 & 0x7FFF7FFFu) - (kGelu2Base | (kGelu2Base << 16));
    oor |= t;
    const uint32_t idx2 = (t & 0x0FFF0FFFu) | ((in2 >> 3) & 0x10001000u);
    const uint32_t lo = tab2[idx2 & 0xFFFFu], hi = tab2[idx2 >> 16];
    return lo | (hi << 16);
}
// true if any element accumulated into `oor` by gelu_pair_fast was outside the table
__device__ __forceinline__ bool gelu_pair_oor(uint32_t oor) { return (oor & 0xF000F000u) != 0u; }
#ifndef LEWIN_TU_LITE
__device__ __forceinline__ void gelu_grad_tab2_to_smem(uint16_t* dst, int tid, int nthreads) {
    for (int i = tid; i < kGelu2TabSize / 8; i += nthreads)
        reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(g_gelu_grad_tab2)[i];
}
#endif
// gelu'(x) of a packed bf16 pair as packed bf16 bits; outside the table: 0.5 (tiny), 1 or 0 (huge, by sign)
static __device__ __noinline__ uint32_t gelu_grad_pair_exact(const uint16_t* __restrict__ tab2g, uint32_t in2) {
    uint32_t out = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t u = (in2 >> (16 * h)) & 0xFFFFu;
        const uint32_t r = (u & 0x7FFFu) - kGelu2Base;
        uint32_t v;
        if (r < 4096u) v = tab2g[r | ((u >> 3) & 0x1000u)];
        else if (static_cast<int32_t>(r) < 0) v = 0x3F00u;
        else v = (u & 0x8000u) ? 0u : 0x3F80u;
        out |= v << (16 * h);
    }
    return out;
}
// exact for every bf16 input (table inside 2^-28 <= |x| < 16, closed forms outside: 0.5 x, x or -0)
static __device__ __noinline__ uint32_t gelu_pair_exact(const uint16_t* __restrict__ tab2, uint32_t in2) {
    uint32_t out = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t u = (in2 >> (16 * h)) & 0xFFFFu;
        const uint32_t r = (u & 0x7FFFu) - kGelu2Base;
        uint32_t v;
        if (r < 4096u) v = tab2[r | ((u >> 3) & 0x1000u)];
        else if (static_cast<int32_t>(r) < 0) v = ((u & 0x7F80u) > 0x0080u) ? (u - 0x80u) : (u & 0x8000u);
        else v = (u & 0x8000u) ? 0x8000u : u;
        out |= v << (16 * h);
    }
    return out;
}

// gelu'(x) for x given as bf16 bits (table value is bf16-rounded; outside the table: 0.5, 1 or 0)
__device__ __forceinline__ float gelu_grad_bits(const uint16_t* __restrict__ tab, uint32_t u) {
    const uint32_t r = (u & 0x7FFFu) - 0x3980u;
    if (__builtin_expect(r < 2048u, 1)) return __uint_as_float(static_cast<uint32_t>(tab[r + ((u >> 15) << 11)]) << 16);
    if (static_cast<int32_t>(r) < 0) return 0.5f;
    return (u & 0x8000u) ? 0.0f : 1.0f;
}

// GELU of a float that is rounded to bf16 first; returns the bf16-valued result as float
__device__ __forceinline__ float gelu_tab(const uint16_t* __restrict__ tab, float x) {
    const uint32_t u = __bfloat16_as_ushort(__float2bfloat16_rn(x));
    return __uint_as_float(gelu_bits(tab, u) << 16);
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {     // reduce over aligned groups of G lanes
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---------------------------------------------------------------- window addressing
// Row m of the window-ordered token matrix -> token offset in the [B, H, W] map, with the cyclic
// shift of My_model_1.py:846 and window_partition of :550-574 folded in:
//   window (b, wy, wx), token (ty, tx)  ->  pixel ((8*wy + ty + s) mod H, (8*wx + tx + s) mod W)
struct WinMap {
    int H, W, nWw, nWin, shift;   // nWin = windows per image; shift: cyclic shift of the columns
    int shift_y;                  // cyclic shift of the rows (== shift for a whole image; 0 for a row band whose rows the caller
                                  // has already laid out in shifted-frame order, see LewinAttnFwdArgs::band_mode)
    __device__ __forceinline__ long long token(long long m) const {
        int n = static_cast<int>(m & 63);
        long long wg = m >> 6;
        int b = static_cast<int>(wg / nWin);
        int w = static_cast<int>(wg - static_cast<long long>(b) * nWin);
        int wy = w / nWw, wx = w - wy * nWw;
        int y = wy * 8 + (n >> 3) + shift_y;
        int x = wx * 8 + (n & 7) + shift;
        if (y >= H) y -= H;
        if (x >= W) x -= W;
        return (static_cast<long long>(b) * H + y) * W + x;
    }
    // 32-bit variant (token counts are far below 2^31): two 32-bit divisions instead of two 64-bit ones
    __device__ __forceinline__ uint32_t token32(uint32_t m) const {
        const uint32_t n = m & 63u, wg = m >> 6;
        const uint32_t b = wg / static_cast<uint32_t>(nWin), w = wg - b * static_cast<uint32_t>(nWin);
        const uint32_t wy = w / static_cast<uint32_t>(nWw), wx = w - wy * static_cast<uint32_t>(nWw);
        return pixel(b, wy, wx, n);
    }
    // token of window (b, wy, wx), in-window index n
    __device__ __forceinline__ uint32_t pixel(uint32_t b, uint32_t wy, uint32_t wx, uint32_t n) const {
        int y = static_cast<int>(wy * 8 + (n >> 3)) + shift_y;
        int x = static_cast<int>(wx * 8 + (n & 7u)) + shift;
        if (y >= H) y -= H;
        if (x >= W) x -= W;
        return (b * static_cast<uint32_t>(H) + static_cast<uint32_t>(y)) * static_cast<uint32_t>(W) + static_cast<uint32_t>(x);
    }
};

// ---------------------------------------------------------------- input mask per token (LewinAttnFwdArgs::token_mask)
// Value of token n of global window wg (batch-major) in the [Bm, H, W] level mask: image b takes mask b mod Bm, and the window
// is partitioned in the UNSHIFTED frame (My_model_1.py:791-798 partitions the mask, not the rolled tokens).
__device__ __forceinline__ float window_token_mask(const float* __restrict__ tm, int Bm, int H, int W, int nWw, int nWin, int wg, int n) {
    const int b = wg / nWin, w = wg - b * nWin;
    const int wy = w / nWw, wx = w - wy * nWw;
    return tm[(static_cast<long long>(b % Bm) * H + wy * 8 + (n >> 3)) * W + wx * 8 + (n & 7)];
}
// Input-mask term of query token i and key token j: -100 where the fp32 product m_i * m_j is non-zero (NaN and inf included,
// products that underflow to zero excluded), exactly as the reference's masked_fill(mask != 0, -100) on that product
__device__ __forceinline__ float token_mask_term(float mi, float mj) { return __fmul_rn(mi, mj) != 0.f ? -100.0f : 0.f; }

}  // namespace lewin
