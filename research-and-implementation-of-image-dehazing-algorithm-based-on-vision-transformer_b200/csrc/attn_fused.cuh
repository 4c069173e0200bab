// The attention half of a LeWin block as ONE kernel (bf16, head_dim 32, C in {32, 64}: the HBM-bound levels):
//
//   y = x + s_b * unroll(unwindow( out_proj( ProbAttention( q|k|v_proj( window(roll( LN1(x) )) ) ) ) ))
//
// Reference: LeWinTransformerBlock.forward My_model_1.py:803-872 -> WindowAttention.forward :400-415 -> AttentionLayer.forward
// ProbSparse/attn.py:385-461 -> ProbAttention.forward attn.py:287-342.  The three-kernel pipeline (gemm_ws q|k|v, core v3,
// gemm_ws out) moves 22 C bytes per token through HBM (x, q|k|v written and re-read, ctx written and re-read, x again, y);
// here x is read once and y written once (4 C bytes): q|k|v live in TMEM / shared memory, ctx in shared memory.
//
// One persistent CTA per SM, two independent 8-warp groups that ping-pong over 128-token tiles (= 2 windows) and share the
// resident weights; a group runs its tile as a sequence of phases separated by named barriers (no warp specialisation: the
// ProbSparse core is instruction-issue bound, so every warp of the group takes part in it, and the other group fills the
// issue slots while this one waits on a load, an MMA or a barrier):
//
//   raw x rows (cp.async, gathered through roll + window_partition, prefetched one tile ahead)
//   -> LayerNorm in registers (same lane partition and summation order as gemm_ws's producers) -> swizzled UMMA A tile
//   -> tcgen05.mma  [128 x C] x [C x 3C]  -> TMEM  -> + bias -> bf16 q | k | v tiles (XOR-swizzled 64-byte rows)
//   -> ProbSparse core on mma.sync fragments, 4 warps per (window, head) item: the arithmetic of probsparse_core_v3.cuh
//      (S = Q K^T, sparsity measure from the sample multiplicities, rank-count top-25, softmax -> +rpb -> +shift mask ->
//      softmax, P.V, mean(V) fill), context rows written straight into the swizzled A tile of the second GEMM
//   -> tcgen05.mma  [128 x C] x [C x C]  -> TMEM  -> + bias, DropPath scale, + residual (x rows re-read through L2)
//   -> per-warp staging -> row-cooperative coalesced stores through window_reverse + un-roll.
//
// Every rounding point equals the three-kernel path's, so the two are bit-identical (tests/test_gpu_fused_attn.py).
#pragma once
#include "tc_helpers.cuh"
#include "probsparse_core_bf16.cuh"

namespace lewin {
namespace af {

constexpr int GROUPS = 2;
constexpr int GTHREADS = 256;                 // threads per group (8 warps)
constexpr int THREADS = GROUPS * GTHREADS;
constexpr int TM = 128;                       // tile rows: two windows
constexpr int STG_ROW = 80;                   // staging row: 32 bf16 columns (64 B) + 16 B pad
constexpr int STG_BUF = 32 * STG_ROW;

struct Args {
    const __nv_bfloat16* x;
    __nv_bfloat16* y;
    const float* ln_w; const float* ln_b;
    const float* w_qkv; const float* b_qkv;   // [3C, C], [3C]
    const float* w_out; const float* b_out;   // [C, C], [C]
    const float* rpb_table;                   // [225, nH] or null
    const float* drop_scale;                  // [B] or null
    const int32_t* index_sample;              // [64, 25]
    uint8_t* top;                             // [B_, nH, 25] or null
    int use_rpb, shift;                       // shift > 0: analytic shift mask (My_model_1.py:803-836)
    int mask_y0, mask_Hg;                     // mask row regions at shifted-frame row mask_y0 + local row of an image mask_Hg tall
    long long M;                              // tokens
    int windows;                              // B * nWin
    int tiles;                                // ceil(windows / 2)
    int tokens_per_image;
    WinMap map;
};

struct SetScratch {                           // per 4-warp set (one (window, head) item at a time)
    alignas(16) float M[kTok];
    int slot_of[kTok];
    int tok_of[32];
    alignas(8) int region[kTok];
    int mixed;
    int pad[3];
    alignas(16) __nv_bfloat16 vmean[kHeadDim];
};

template <int C>
struct Cfg {
    static constexpr int NH = C / kHeadDim;
    static constexpr int KC = C >= 64 ? 64 : 32;            // k-chunk: SWIZZLE_128B / SWIZZLE_64B
    static constexpr int NKC = C / KC;
    static constexpr int G = C / 8;                         // 16-byte chunks (= LN lanes) per row
    static constexpr int RPP = GTHREADS / G;                // rows per pass of the group's 256 threads
    static constexpr int NP = TM / RPP;                     // passes (chunks per thread) per tile
    static constexpr int A_CHUNK = TM * KC * 2;
    static constexpr int A_BYTES = TM * C * 2;
    static constexpr int QKV_BYTES = 3 * TM * C * 2;
    static constexpr int WQ_CHUNK = 3 * C * KC * 2;
    static constexpr int WO_CHUNK = C * KC * 2;
    static constexpr int WQ_BYTES = 3 * C * C * 2;
    static constexpr int WO_BYTES = (C * C * 2 + 1023) / 1024 * 1024;
    static constexpr int GROUP_BYTES = 2 * A_BYTES + QKV_BYTES;      // raw | A (ctx) | q k v (staging)
    static constexpr int MISC_BYTES = (3 * C + C + 2 * C + NH * 232) * 4 + 4 * static_cast<int>(sizeof(SetScratch)) + 64;
    static constexpr int SMEM = 1024 + WQ_BYTES + WO_BYTES + GROUPS * GROUP_BYTES + MISC_BYTES;
    static constexpr int TMEM_G = 4 * C;                    // TMEM columns per group: q|k|v accumulator + out accumulator
    static constexpr int TMEM_COLS = GROUPS * TMEM_G < 32 ? 32 : GROUPS * TMEM_G;
    static_assert(NKC == 1, "C <= 64: one k-chunk");
    static_assert(QKV_BYTES >= 8 * STG_BUF, "epilogue staging aliases the q|k|v tiles");
    static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS <= 512, "TMEM allocation is a power of two <= 512");
};

// packed fp32x2 arithmetic (same IEEE rounding as the scalar instructions; identical to gemm_ws.cuh's)
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

__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// 16-byte chunk `ch` of row `row` of a [rows x 32] bf16 core tile (64-byte rows, chunk index XOR-swizzled by the row pair:
// 8 consecutive rows of one chunk column hit 8 different bank groups -> conflict-free ldmatrix and row-per-lane stores)
__device__ __forceinline__ uint32_t core_off(int row, int ch) { return static_cast<uint32_t>(row * 64 + ((ch ^ ((row >> 1) & 3)) << 4)); }

template <int C>
__global__ void __launch_bounds__(THREADS, 1) attn_fused_kernel(const Args a) {
    using Cf = Cfg<C>;
    constexpr int NH = Cf::NH, KC = Cf::KC, G = Cf::G, RPP = Cf::RPP, NP = Cf::NP;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Wq = base;                                    // [3C x C] bf16, K-major swizzled (UMMA B operand)
    unsigned char* Wo = Wq + Cf::WQ_BYTES;                       // [C x C]
    unsigned char* gmem0 = Wo + Cf::WO_BYTES;
    unsigned char* misc = gmem0 + GROUPS * Cf::GROUP_BYTES;
    float* s_bqkv = reinterpret_cast<float*>(misc);              // [3C] bf16-rounded
    float* s_bo = s_bqkv + 3 * C;                                // [C]
    float* s_gam = s_bo + C;                                     // [C]
    float* s_bet = s_gam + C;                                    // [C]
    float* s_tbl = s_bet + C;                                    // [NH][232]
    SetScratch* sets = reinterpret_cast<SetScratch*>(s_tbl + NH * 232);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sets + 4);      // [GROUPS][2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 4);

    const int tid = threadIdx.x, lane = tid & 31;
    const int g = tid >> 8, gt = tid & 255, gw = gt >> 5;        // group, thread / warp in the group
    const int set = gw >> 2, sw = gw & 3;                        // 4-warp set in the group, warp in the set
    const int gq = lane >> 2, tq = lane & 3;
    unsigned char* raw = gmem0 + g * Cf::GROUP_BYTES;            // [128][C] bf16 raw x rows, chunk i at i * 16
    unsigned char* At = raw + Cf::A_BYTES;                       // swizzled UMMA A tile: LN(x), later ctx
    unsigned char* qkv = At + Cf::A_BYTES;                       // [3][NH][128][64 B] core tiles; later epilogue staging
    SetScratch& s = sets[g * 2 + set];

    // ---------------------------------------------------------------- one-time setup (all 512 threads)
    for (int c = tid; c < 4 * C * G; c += THREADS) {             // W_qkv rows 0..3C-1, then W_out rows
        const int r = c / G, ch = c % G;
        const float* src = (r < 3 * C ? a.w_qkv + static_cast<long long>(r) * C : a.w_out + static_cast<long long>(r - 3 * C) * C) + ch * 8;
        const float4 a4 = *reinterpret_cast<const float4*>(src);
        const float4 b4 = *reinterpret_cast<const float4*>(src + 4);
        unsigned char* dst = r < 3 * C ? Wq + tc::swz_off<KC>(r, ch) : Wo + tc::swz_off<KC>(r - 3 * C, ch);
        *reinterpret_cast<uint4*>(dst) = make_uint4(tc::pack_bf16(a4.x, a4.y), tc::pack_bf16(a4.z, a4.w), tc::pack_bf16(b4.x, b4.y), tc::pack_bf16(b4.z, b4.w));
    }
    for (int i = tid; i < 3 * C; i += THREADS) s_bqkv[i] = Act<__nv_bfloat16>::round(a.b_qkv[i]);
    for (int i = tid; i < C; i += THREADS) {
        s_bo[i] = Act<__nv_bfloat16>::round(a.b_out[i]);
        s_gam[i] = a.ln_w[i];
        s_bet[i] = a.ln_b[i];
    }
    if (a.use_rpb && a.rpb_table)
        for (int i = tid; i < NH * 225; i += THREADS) { const int h = i / 225, e = i - h * 225; s_tbl[h * 232 + e] = a.rpb_table[e * NH + h]; }
    if (tid < 4 * 32) sets[tid >> 5].tok_of[tid & 31] = -1;      // slots 25..31 stay -1 for the whole kernel
    // sample multiplicities of my fragment positions (rows sw*16 + gq (+8), columns j*8 + 2tq (+1)): registers
    __half2 cntp[2][8];
    uint32_t sampled = 0;
    {
        uint8_t* cnt = gmem0 + Cf::A_BYTES * 2;                  // group 0's q|k|v region, free during setup
        build_cnt_smem(cnt, a.index_sample, tid, THREADS);
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int r = sw * 16 + gq + half * 8, c = j * 8 + 2 * tq;
                const uint32_t c2 = *reinterpret_cast<const uint16_t*>(cnt + r * kTok + c);
                const int c0 = c2 & 0xFF, c1 = c2 >> 8;
                cntp[half][j] = __halves2half2(__int2half_rn(c0), __int2half_rn(c1));
                if (c0) sampled |= 1u << (half * 16 + j * 2);
                if (c1) sampled |= 1u << (half * 16 + j * 2 + 1);
            }
    }
    if (tid == 0) {
        for (int i = 0; i < 2 * GROUPS; ++i) tc::mbar_init(&mbar[i], 1);
        tc::fence_barrier_init();
    }
    if (tid < 32) tc::tmem_alloc<Cf::TMEM_COLS>(tmem_slot);
    tc::fence_proxy_async();                                     // resident weights: generic-proxy writes -> tensor core
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_g = *tmem_slot + static_cast<uint32_t>(g * Cf::TMEM_G);

    // ---------------------------------------------------------------- per-thread constants
    const int gl = gt % G, r0 = gt / G;                          // my 16-byte chunk column and first row (rows r0 + k * RPP)
    float2 gam[4], bet[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        gam[j] = make_float2(s_gam[gl * 8 + 2 * j], s_gam[gl * 8 + 2 * j + 1]);
        bet[j] = make_float2(s_bet[gl * 8 + 2 * j], s_bet[gl * 8 + 2 * j + 1]);
    }
    const uint32_t raw_u = tc::smem_u32(raw);
    const float scale = rsqrtf(static_cast<float>(kHeadDim));
    constexpr uint32_t IDESC1 = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>((3 * C) >> 3) << 17) | (static_cast<uint32_t>(TM >> 4) << 24);
    constexpr uint32_t IDESC2 = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(C >> 3) << 17) | (static_cast<uint32_t>(TM >> 4) << 24);

    // windows (b, wy, wx) of the two halves of tile t
    struct Win2 { uint32_t b[2], wy[2], wx[2]; };
    auto decode = [&](int t) {
        Win2 w;
        const uint32_t wg = static_cast<uint32_t>(t) * 2u;
        w.b[0] = wg / static_cast<uint32_t>(a.map.nWin);
        const uint32_t ww = wg - w.b[0] * static_cast<uint32_t>(a.map.nWin);
        w.wy[0] = ww / static_cast<uint32_t>(a.map.nWw);
        w.wx[0] = ww - w.wy[0] * static_cast<uint32_t>(a.map.nWw);
        w.b[1] = w.b[0]; w.wy[1] = w.wy[0]; w.wx[1] = w.wx[0] + 1u;
        if (w.wx[1] == static_cast<uint32_t>(a.map.nWw)) {
            w.wx[1] = 0u; w.wy[1] += 1u;
            if (w.wy[1] * static_cast<uint32_t>(a.map.nWw) == static_cast<uint32_t>(a.map.nWin)) { w.wy[1] = 0u; w.b[1] += 1u; }
        }
        return w;
    };
    // raw x rows of tile t -> shared memory: thread (r0, gl) copies chunk gl of rows r0 + k * RPP (and is their only reader)
    auto load_raw = [&](int t) {
        const Win2 w = decode(t);
#pragma unroll
        for (int k = 0; k < NP; ++k) {
            const int r = r0 + k * RPP, hi = r >> 6;
            const bool ok = t * 2 + hi < a.windows;
            const uint32_t tok = ok ? a.map.pixel(w.b[hi], w.wy[hi], w.wx[hi], static_cast<uint32_t>(r & 63)) : 0u;
            cp_async16_z(raw_u + static_cast<uint32_t>(gt + k * GTHREADS) * 16u, a.x + static_cast<long long>(tok) * C + gl * 8, ok);
        }
    };

    const int gstride = GROUPS * static_cast<int>(gridDim.x);
    int tile = static_cast<int>(blockIdx.x) * GROUPS + g;
    uint32_t ph = 0;
    if (tile < a.tiles) load_raw(tile);
    cp_async_commit();

    for (; tile < a.tiles; tile += gstride) {
        // ============================================================ LayerNorm: my raw chunks -> swizzled A tile
        cp_async_wait<0>();
        {
            float2 f[NP][4];
            float sum[NP], sq[NP];
#pragma unroll
            for (int k = 0; k < NP; ++k) {
                const uint4 u = *reinterpret_cast<const uint4*>(raw + (gt + k * GTHREADS) * 16);
                const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) f[k][q] = make_float2(__uint_as_float(w4[q] << 16), __uint_as_float(w4[q] & 0xFFFF0000u));
                sum[k] = 0.f;
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int k = 0; k < NP; ++k) { sum[k] += f[k][q].x; sum[k] += f[k][q].y; }
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1)
#pragma unroll
                for (int k = 0; k < NP; ++k) sum[k] += __shfl_xor_sync(0xffffffffu, sum[k], o);
#pragma unroll
            for (int k = 0; k < NP; ++k) {
                const float nmu = -(sum[k] * (1.0f / C));
                const float2 nm2 = make_float2(nmu, nmu);
#pragma unroll
                for (int q = 0; q < 4; ++q) f[k][q] = add2(f[k][q], nm2);
                sq[k] = 0.f;
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int k = 0; k < NP; ++k) { sq[k] = fmaf(f[k][q].x, f[k][q].x, sq[k]); sq[k] = fmaf(f[k][q].y, f[k][q].y, sq[k]); }
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1)
#pragma unroll
                for (int k = 0; k < NP; ++k) sq[k] += __shfl_xor_sync(0xffffffffu, sq[k], o);
#pragma unroll
            for (int k = 0; k < NP; ++k) {
                const float rs = rsqrtf(sq[k] * (1.0f / C) + 1e-5f);
                const float2 rs2 = make_float2(rs, rs);
                uint32_t o4[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float2 y2 = fma2(mul2(f[k][q], rs2), gam[q], bet[q]);
                    o4[q] = tc::pack_bf16(y2.x, y2.y);
                }
                *reinterpret_cast<uint4*>(At + tc::swz_off<KC>(r0 + k * RPP, gl)) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
            }
        }
        tc::fence_proxy_async();                                   // my A-tile writes -> visible to the tensor core
        bar_sync(1 + g, GTHREADS);                                 // [G1] A tile complete; the previous tile is fully retired
        if (tile + gstride < a.tiles) load_raw(tile + gstride);    // the raw buffer was consumed above: prefetch the next tile
        cp_async_commit();
        if (gt == 0) {                                             // q | k | v = LN(x) . W_qkv^T  -> TMEM columns [0, 3C)
            tc::tc_fence_after();
            const uint64_t da = tc::make_desc<KC>(tc::smem_u32(At)), db = tc::make_desc<KC>(tc::smem_u32(Wq));
#pragma unroll
            for (int k16 = 0; k16 < KC / 16; ++k16) tc::mma_bf16(tmem_g, da + 2 * k16, db + 2 * k16, IDESC1, k16 > 0 ? 1u : 0u);
            tc::mma_commit(&mbar[g * 2]);
        }
        tc::mbar_wait(&mbar[g * 2], ph);
        tc::tc_fence_after();
        // ============================================================ accumulator -> + bias -> bf16 q | k | v core tiles
        {
            const int r = (gw & 3) * 32 + lane;                    // thread == TMEM lane == tile row
            const uint32_t t_addr = tmem_g + (static_cast<uint32_t>((gw & 3) * 32) << 16);
            const int swz = (r >> 1) & 3;
#pragma unroll 1
            for (int c = gw >> 2; c < 3 * NH; c += 2) {            // 32-column chunk == one (q|k|v, head) tile
                float v[32];
                tc::tmem_ld32(t_addr + c * 32, v);
                const float2* bs2 = reinterpret_cast<const float2*>(s_bqkv + c * 32);
                uint32_t pk[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 t2 = add2(make_float2(v[2 * j], v[2 * j + 1]), bs2[j]);
                    pk[j] = tc::pack_bf16(t2.x, t2.y);
                }
                unsigned char* dst = qkv + (c * TM + r) * 64;       // c == which * NH + head
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<uint4*>(dst + ((j ^ swz) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            }
        }
        tc::tc_fence_before();
        bar_sync(1 + g, GTHREADS);                                 // [G2] q | k | v tiles complete

        // ============================================================ ProbSparse core: items (window half, head), 4 warps each
#pragma unroll 1
        for (int item = set; item < 2 * NH; item += 2) {
            const int wl = item / NH, h = item - wl * NH;
            const int wg = tile * 2 + wl;                          // global window index (batch-major)
            if (wg >= a.windows) break;                            // odd window count: the tile's second half is empty
            const unsigned char* sq = qkv + ((0 * NH + h) * TM + wl * 64) * 64;
            const unsigned char* sk = qkv + ((1 * NH + h) * TM + wl * 64) * 64;
            const unsigned char* sv = qkv + ((2 * NH + h) * TM + wl * 64) * 64;
            // ---- phase 1: S = Q K^T for rows 16*sw..+15, sparsity measure M (attn.py:71-117)
            {
                float acc[8][4];
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    uint32_t af[4];
                    pc::ldsm_x4(af, sq + core_off(sw * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)));
#pragma unroll
                    for (int jp = 0; jp < 4; ++jp) {
                        uint32_t bf[4];
                        pc::ldsm_x4(bf, sk + core_off(jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8, ks * 2 + ((lane >> 3) & 1)));
                        pc::mma16816(acc[2 * jp], af, bf[0], bf[1]);
                        pc::mma16816(acc[2 * jp + 1], af, bf[2], bf[3]);
                    }
                }
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float mx = -INFINITY, sm = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t pk = pc::pack2(acc[j][half * 2], acc[j][half * 2 + 1]);      // S~ is a bf16 matmul output (A.4)
                        const float s0 = __uint_as_float(pk << 16), s1 = __uint_as_float(pk & 0xFFFF0000u);
                        const float2 cn = __half22float2(cntp[half][j]);
                        const float m0 = (sampled >> (half * 16 + j * 2)) & 1u ? s0 : -INFINITY;
                        const float m1 = (sampled >> (half * 16 + j * 2 + 1)) & 1u ? s1 : -INFINITY;
                        mx = fmaxf(mx, fmaxf(m0, m1));
                        sm = fmaf(cn.x, s0, sm);
                        sm = fmaf(cn.y, s1, sm);
                    }
                    mx = group_max<4>(mx);
                    sm = group_sum<4>(sm);
                    if (tq == 0) s.M[sw * 16 + gq + half * 8] = mx - sm * (1.0f / kTok);
                }
            }
            bar_sync(3 + 2 * g + set, 128);                        // [S1] M complete; the previous item of this set is retired
            // ---- phase 2: top-u by rank counting (ties -> lower index), 2 lanes per row
            {
                const int r = sw * 16 + (lane & 15), hf = lane >> 4;
                const float mine = s.M[r];
                int rank = 0;
#pragma unroll
                for (int m4 = 0; m4 < 8; ++m4) {
                    const float4 o = *reinterpret_cast<const float4*>(s.M + hf * 32 + m4 * 4);
                    const int m = hf * 32 + m4 * 4;
                    rank += (o.x > mine) || (o.x == mine && m < r);
                    rank += (o.y > mine) || (o.y == mine && m + 1 < r);
                    rank += (o.z > mine) || (o.z == mine && m + 2 < r);
                    rank += (o.w > mine) || (o.w == mine && m + 3 < r);
                }
                rank += __shfl_xor_sync(0xffffffffu, rank, 16);
                if (hf == 0) {
                    const int slot = rank < kTopU ? rank : -1;
                    s.slot_of[r] = slot;
                    if (slot >= 0) {
                        s.tok_of[slot] = r;
                        if (a.top) a.top[(static_cast<long long>(wg) * NH + h) * kTopU + slot] = static_cast<uint8_t>(r);
                    }
                }
                if (a.shift > 0 && sw == 0) {                      // shift-mask regions of this window (read in phase 3 only)
                    const int w = wg % a.map.nWin, wy = w / a.map.nWw, wx = w - wy * a.map.nWw;
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int t = lane + 32 * i;
                        const int yy = a.mask_y0 + wy * 8 + (t >> 3), xx = wx * 8 + (t & 7);
                        const int rb = yy < a.mask_Hg - 8 ? 0 : (yy < a.mask_Hg - a.shift ? 1 : 2);
                        const int cb = xx < a.map.W - 8 ? 0 : (xx < a.map.W - a.shift ? 1 : 2);
                        s.region[t] = rb * 3 + cb;
                    }
                    if (lane == 0) s.mixed = (a.mask_y0 + wy * 8 + 8 > a.mask_Hg - 8) || (wx * 8 + 8 > a.map.W - 8);
                }
            }
            bar_sync(3 + 2 * g + set, 128);                        // [S2] slots assigned
            // ---- phase 3: slots 8*sw..+7 = rows 0..7 of this warp's m16 tile (rows 8..15 are dummies)
            {
                const int my_tok = s.tok_of[sw * 8 + gq];
                float acc[8][2];
                {
                    float full[8][4];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) full[j][c] = 0.f;
                    int arow = s.tok_of[sw * 8 + (lane & 7)];
                    if (arow < 0) arow = 0;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        uint32_t af[4];
                        pc::ldsm_x4(af, sq + core_off(arow, ks * 2 + (lane >> 4)));
#pragma unroll
                        for (int jp = 0; jp < 4; ++jp) {
                            uint32_t bf[4];
                            pc::ldsm_x4(bf, sk + core_off(jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8, ks * 2 + ((lane >> 3) & 1)));
                            pc::mma16816(full[2 * jp], af, bf[0], bf[1]);
                            pc::mma16816(full[2 * jp + 1], af, bf[2], bf[3]);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {                   // bf16(S) * scale -> bf16 (attn.py:150, 327-329)
                        const uint32_t pk = pc::pack2(full[j][0], full[j][1]);
                        const uint32_t p2 = pc::pack2(__uint_as_float(pk << 16) * scale, __uint_as_float(pk & 0xFFFF0000u) * scale);
                        acc[j][0] = __uint_as_float(p2 << 16);
                        acc[j][1] = __uint_as_float(p2 & 0xFFFF0000u);
                    }
                }
                float mx = acc[0][0];
#pragma unroll
                for (int j = 0; j < 8; ++j) mx = fmaxf(mx, fmaxf(acc[j][0], acc[j][1]));
                mx = group_max<4>(mx);
                float mxl = mx * 1.4426950408889634f;
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc[j][0] = exp_sub(acc[j][0], mxl); acc[j][1] = exp_sub(acc[j][1], mxl);
                    sum += acc[j][0]; sum += acc[j][1];
                }
                float inv = __fdividef(1.0f, group_sum<4>(sum));
#pragma unroll
                for (int j = 0; j < 8; ++j) { acc[j][0] *= inv; acc[j][1] *= inv; }
                const int r = my_tok < 0 ? 0 : my_tok;
                if (a.use_rpb && a.rpb_table) {                     // + bias on the PROBABILITIES (attn.py:195-264)
                    const int ry = r >> 3, rx = r & 7;
                    const float* tb = s_tbl + h * 232 + (ry + 7) * 15 + (rx - 2 * tq + 7);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { acc[j][0] += tb[-j * 15]; acc[j][1] += tb[-j * 15 - 1]; }
                }
                if (a.shift > 0 && s.mixed) {
                    const int rr = s.region[r];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int2 rc = *reinterpret_cast<const int2*>(s.region + j * 8 + 2 * tq);
                        acc[j][0] += (rc.x != rr) ? -100.0f : 0.f;
                        acc[j][1] += (rc.y != rr) ? -100.0f : 0.f;
                    }
                }
                mx = acc[0][0];
#pragma unroll
                for (int j = 0; j < 8; ++j) mx = fmaxf(mx, fmaxf(acc[j][0], acc[j][1]));
                mx = group_max<4>(mx);
                mxl = mx * 1.4426950408889634f;
                sum = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc[j][0] = exp_sub(acc[j][0], mxl); acc[j][1] = exp_sub(acc[j][1], mxl);
                    sum += acc[j][0]; sum += acc[j][1];
                }
                inv = __fdividef(1.0f, group_sum<4>(sum));
                uint32_t pfrag[8];
                const bool mean_row = (sw == 3 && gq == 7);        // slot 31 is never live: its row computes mean(V)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    pfrag[j] = pc::pack2(acc[j][0] * inv, acc[j][1] * inv);
                    if (my_tok < 0) pfrag[j] = mean_row ? 0x3C803C80u : 0u;      // bf16 1/64 | zero row
                }
                float o[4][4];
#pragma unroll
                for (int n = 0; n < 4; ++n)
#pragma unroll
                    for (int c = 0; c < 4; ++c) o[n][c] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint32_t af[4] = {pfrag[2 * ks], 0u, pfrag[2 * ks + 1], 0u};
#pragma unroll
                    for (int nb = 0; nb < 2; ++nb) {
                        uint32_t bf[4];
                        pc::ldsm_x4_t(bf, sv + core_off(ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, nb * 2 + (lane >> 4)));
                        pc::mma16816(o[2 * nb], af, bf[0], bf[1]);
                        pc::mma16816(o[2 * nb + 1], af, bf[2], bf[3]);
                    }
                }
                // context rows -> swizzled A tile of the out projection (row = tile row, columns h*32 .. h*32+31)
                if (my_tok >= 0) {
#pragma unroll
                    for (int n = 0; n < 4; ++n)
                        *reinterpret_cast<uint32_t*>(At + tc::swz_off<KC>(wl * 64 + my_tok, h * 4 + n) + tq * 4) = pc::pack2(o[n][0], o[n][1]);
                }
                if (mean_row) {
#pragma unroll
                    for (int n = 0; n < 4; ++n)
                        *reinterpret_cast<uint32_t*>(s.vmean + n * 8 + 2 * tq) = pc::pack2(o[n][0], o[n][1]);
                }
                if (sw == 3) {                                      // lazy queries: mean(V) (attn.py:168-172)
                    __syncwarp();
                    const uint4 vm = *reinterpret_cast<const uint4*>(s.vmean + (lane & 3) * 8);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int rr = (lane >> 2) + i * 8;
                        if (s.slot_of[rr] < 0) *reinterpret_cast<uint4*>(At + tc::swz_off<KC>(wl * 64 + rr, h * 4 + (lane & 3))) = vm;
                    }
                }
            }
        }
        tc::fence_proxy_async();                                   // my ctx writes -> visible to the tensor core
        bar_sync(1 + g, GTHREADS);                                 // [G3] ctx tile complete; q | k | v tiles are dead -> staging

        // ============================================================ out projection + DropPath scale + residual + store
        {
            const int r = (gw & 3) * 32 + lane;
            const int hi = r >> 6;
            const Win2 w = decode(tile);
            const bool ok = tile * 2 + hi < a.windows;
            const uint32_t tok = ok ? a.map.pixel(w.b[hi], w.wy[hi], w.wx[hi], static_cast<uint32_t>(r & 63)) : 0u;
            const long long oy = ok ? static_cast<long long>(tok) * C : -1;
            const float sc = (ok && a.drop_scale) ? a.drop_scale[tok / static_cast<uint32_t>(a.tokens_per_image)] : 1.f;
            unsigned char* my_stg = qkv + gw * STG_BUF;
            const int c = gw >> 2;                                  // this warp's 32-column chunk (C / 32 <= 2 chunks)
            const bool active = c < C / 32;
            if (active) {                                           // residual rows (x through L2) -> staging, coalesced 64-byte pieces
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const long long o = __shfl_sync(0xffffffffu, oy, rl);
                    if (o >= 0) cp_async16(my_stg + rl * STG_ROW + cc * 16, a.x + o + c * 32 + cc * 8);
                }
            }
            cp_async_commit();
            if (gt == 0) {                                          // out = ctx . W_out^T -> TMEM columns [3C, 4C)
                tc::tc_fence_after();
                const uint64_t da = tc::make_desc<KC>(tc::smem_u32(At)), db = tc::make_desc<KC>(tc::smem_u32(Wo));
#pragma unroll
                for (int k16 = 0; k16 < KC / 16; ++k16) tc::mma_bf16(tmem_g + 3 * C, da + 2 * k16, db + 2 * k16, IDESC2, k16 > 0 ? 1u : 0u);
                tc::mma_commit(&mbar[g * 2 + 1]);
            }
            tc::mbar_wait(&mbar[g * 2 + 1], ph);
            tc::tc_fence_after();
            // NOTE: the wait above also keeps the next tile's raw prefetch (an older cp.async group) behind us, harmless
            cp_async_wait<0>();
            __syncwarp();
            if (active) {
                float v[32];
                tc::tmem_ld32(tmem_g + (static_cast<uint32_t>((gw & 3) * 32) << 16) + 3 * C + c * 32, v);
                const float2* bs2 = reinterpret_cast<const float2*>(s_bo + c * 32);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 t2 = add2(make_float2(v[2 * j], v[2 * j + 1]), bs2[j]);
                    v[2 * j] = t2.x; v[2 * j + 1] = t2.y;
                }
                unsigned char* srow = my_stg + lane * STG_ROW;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const uint4 rv = *reinterpret_cast<const uint4*>(srow + j * 2);
                    const uint32_t w4[4] = {rv.x, rv.y, rv.z, rv.w};
                    uint32_t o4[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float x0 = __uint_as_float(w4[e] << 16) + sc * Act<__nv_bfloat16>::round(v[j + 2 * e]);
                        const float x1 = __uint_as_float(w4[e] & 0xFFFF0000u) + sc * Act<__nv_bfloat16>::round(v[j + 2 * e + 1]);
                        o4[e] = tc::pack_bf16(x0, x1);
                    }
                    *reinterpret_cast<uint4*>(srow + j * 2) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
                }
                __syncwarp();
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {                    // 8 rows x 64 contiguous bytes per warp instruction
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    const uint4 val = *reinterpret_cast<const uint4*>(my_stg + rl * STG_ROW + cc * 16);
                    const long long o = __shfl_sync(0xffffffffu, oy, rl);
                    if (o >= 0) *reinterpret_cast<uint4*>(a.y + o + c * 32 + cc * 8) = val;
                }
            }
            tc::tc_fence_before();
        }
        ph ^= 1u;
    }
    cp_async_wait<0>();
    tc::tc_fence_before();
    __syncthreads();
    if (tid < 32) tc::tmem_dealloc<Cf::TMEM_COLS>(*tmem_slot);
}

inline bool supported(int C, int nH, long long tokens) {
    return (C == 32 || C == 64) && C == nH * kHeadDim && tokens >= 4 * TM && tokens < (1ll << 31);
}

template <int C>
inline cudaError_t launch_c(const Args& a, int num_sms, cudaStream_t stream) {
    auto k = attn_fused_kernel<C>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<C>::SMEM);
    if (e != cudaSuccess) return e;
    int grid = (a.tiles + GROUPS - 1) / GROUPS;
    if (grid > num_sms) grid = num_sms;
    k<<<grid, THREADS, Cfg<C>::SMEM, stream>>>(a);
    return cudaGetLastError();
}

inline cudaError_t launch(int C, const Args& a, int num_sms, cudaStream_t stream) {
    if (C == 32) return launch_c<32>(a, num_sms, stream);
    if (C == 64) return launch_c<64>(a, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace af
}  // namespace lewin
