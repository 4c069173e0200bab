// ProbSparse window-attention core, backward, bf16 (autograd of ProbSparse/attn.py:287-342 for the selected top-u rows and
// the mean(V) fill) — register-resident restatement of probsparse_core_bwd_kernel in the style of probsparse_core_v3:
//   * q | k | v | dctx of the next (window, head) item prefetched by cp.async (two buffers), bf16 tiles, ldmatrix fragments;
//   * warp w owns slots 8w..8w+7 (rows 0..7 of an m16 tile): S_sel = Q_sel K^T and dP2 = dctx_sel V^T are recomputed on
//     the tensor cores, softmax -> +rpb -> +mask -> softmax and BOTH softmax backward passes run on the accumulator
//     fragments (quad-shuffle row reductions), dS feeds dq = dS K directly as an A fragment;
//   * dS and P2 (bf16) are exchanged through a 9 KB shared tile for the transposed products dk = dS^T Q_sel,
//     dv = P2^T dctx_sel + dmean (each warp 16 keys), Q_sel / dctx_sel rows gathered by ldmatrix row addresses;
//   * dmean (gradient of the mean(V) fill) is one MMA of a 0 / (1/64) row-selector against the dctx tile;
//   * the selected-token list is read per warp and distributed by shuffles: 2 block barriers per item (was 8).
// Rounding points: S, P2, dS, dP2 operands are bf16 (autocast semantics); accumulation fp32; d(rpb table) fp32 atomics.
#pragma once
#include "core_bwd_args.cuh"
#include "probsparse_core_bf16.cuh"

namespace lewin {
namespace pcb2 {

constexpr int THREADS = 128;
constexpr int LD = 40;                       // bf16 row stride of the 64 x 32 operand tiles
constexpr int TILE = kTok * LD;
constexpr int PLD = 72;                      // bf16 row stride of the [32 slots][64 keys] exchange tiles

struct Smem {
    alignas(16) __nv_bfloat16 in[2][4 * TILE];          // q | k | v | dctx, double buffered
    alignas(16) __nv_bfloat16 dss[32 * PLD];            // dS   [slot][key]
    alignas(16) __nv_bfloat16 p2s[32 * PLD];            // P2   [slot][key]
    alignas(16) __nv_bfloat16 ostage[4][2][16 * kHeadDim];   // per-warp output staging (dq / dk, dv)
    float tbl[232];
    float dmean[kHeadDim];
    alignas(8) int region[kTok];
    int mixed;
    float tacc[16 * 225];                               // d(rpb table) partials per head
    alignas(16) float tm[kTok];                         // input mask of the window's tokens (a.tmask)
    int tm_live[2];                                     // per staging warp: some token has a non-zero input-mask value
};

// DET (deterministic mode): dynamic shared memory also holds DetDa, the fp32 dA rows of the item's slots; after [B3] each
// relative-position entry of the table sums them in slot order (no shared atomics), the table partials are stored into slab
// blockIdx.x of [gridDim.x][225, nH], and d(rpb dense) is added with plain stores into slab blockIdx.x of [gridDim.x][nH, 64, 64]
// (zeroed by the caller).  Two CTAs per SM.
constexpr int DA_LD = 68;
struct DetDa { float da[32 * DA_LD]; };

// TMASK: the call has an input mask per token (a.tmask); a template parameter, as in probsparse_core_v3_kernel
template <bool TMASK, bool DET = false>
__global__ void __launch_bounds__(THREADS, 3) core_bwd_v2_kernel(const CoreBwdArgs<__nv_bfloat16> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    float* const dab = reinterpret_cast<DetDa*>(smem_raw + sizeof(Smem))->da;      // DET only
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int C3 = 3 * a.C;
    const float scale = rsqrtf(static_cast<float>(kHeadDim));
    const int items = a.B_ * a.nH;
    const bool want_tab = a.d_rpb_table != nullptr && a.use_rpb && a.rpb_table != nullptr;
    const bool want_dense = a.d_rpb_dense != nullptr && a.use_rpb;
    for (int i = tid; i < 16 * 225; i += THREADS) s.tacc[i] = 0.f;

    auto prefetch = [&](int item, int buf) {
        const int wg = item / a.nH, h = item - wg * a.nH;
        const __nv_bfloat16* base = a.qkv + static_cast<long long>(wg) * kTok * C3 + h * kHeadDim;
        const __nv_bfloat16* dbase = a.dctx + static_cast<long long>(wg) * kTok * a.C + h * kHeadDim;
        __nv_bfloat16* dst = s.in[buf];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = tid + i * THREADS;
            const int which = c >> 8, r = (c >> 2) & 63, ch = c & 3;
            const __nv_bfloat16* src = which < 3 ? base + static_cast<long long>(r) * C3 + which * a.C + ch * 8
                                                 : dbase + static_cast<long long>(r) * a.C + ch * 8;
            cp_async16(dst + which * TILE + r * LD + ch * 8, src);
        }
    };

    int item = blockIdx.x, buf = 0;
    if (item < items) prefetch(item, 0);
    cp_async_commit();
    for (; item < items; item += gridDim.x, buf ^= 1) {
        const int wg = item / a.nH, h = item - wg * a.nH;
        // selected tokens of this item: every warp keeps its own copy (lane s holds slot s) -> no shared table, no barrier
        const int my_sel = lane < kTopU ? static_cast<int>(a.top[static_cast<long long>(item) * kTopU + lane]) : -1;
        cp_async_wait<0>();
        __syncthreads();                                                        // [B1] tiles landed; previous item retired
        if (item + static_cast<int>(gridDim.x) < items) prefetch(item + gridDim.x, buf ^ 1);
        cp_async_commit();
        const __nv_bfloat16* sq = s.in[buf];
        const __nv_bfloat16* sk = sq + TILE;
        const __nv_bfloat16* sv = sk + TILE;
        const __nv_bfloat16* sdc = sv + TILE;
        if (a.use_rpb && a.rpb_table)
            for (int i = tid; i < 225; i += THREADS) s.tbl[i] = a.rpb_table[i * a.nH + h];
        if (a.shift > 0 && tid < kTok) {
            const int w = wg % a.nWin, wy = w / a.nWw, wx = w - wy * a.nWw;
            const int y = wy * 8 + (tid >> 3), x = wx * 8 + (tid & 7);
            const int rb = y < a.H - 8 ? 0 : (y < a.H - a.shift ? 1 : 2);
            const int cb = x < a.W - 8 ? 0 : (x < a.W - a.shift ? 1 : 2);
            s.region[tid] = rb * 3 + cb;
            if (tid == 0) s.mixed = (wy * 8 + 8 > a.H - 8) || (wx * 8 + 8 > a.W - 8);
        }
        if (TMASK && tid < kTok) {
            const float m = window_token_mask(a.tmask, a.Bm, a.H, a.W, a.nWw, a.nWin, wg, tid);
            s.tm[tid] = m;
            const bool live = __any_sync(0xffffffffu, m != 0.f);
            if (lane == 0) s.tm_live[warp] = live;
        }
        // membership mask of the selected tokens (uniform in the warp)
        unsigned long long selmask = my_sel >= 0 ? (1ull << my_sel) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) selmask |= __shfl_xor_sync(0xffffffffu, selmask, o);
        const bool need_tbl_sync = (a.use_rpb && a.rpb_table) || a.shift > 0 || TMASK;
        if (need_tbl_sync) __syncthreads();                                     // [B2] bias table / region of this item visible

        const int my_tok = __shfl_sync(0xffffffffu, my_sel, (warp * 8 + gq) & 31);          // token of my fragment row (-1: dummy)
        __nv_bfloat16* obase = a.dqkv + static_cast<long long>(wg) * kTok * C3 + h * kHeadDim;
        // ================= phase A: slots 8*warp..+7 as rows 0..7 of the warp's m16 tile
        {
            float x[8][2], gr[8][2];
            {
                float S[8][4], G[8][4];
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) { S[j][c] = 0.f; G[j][c] = 0.f; }
                int arow = __shfl_sync(0xffffffffu, my_sel, (warp * 8 + (lane & 7)) & 31);
                if (arow < 0) arow = 0;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    uint32_t aq[4], ad[4];
                    pc::ldsm_x4(aq, sq + arow * LD + ks * 16 + (lane >> 4) * 8);
                    pc::ldsm_x4(ad, sdc + arow * LD + ks * 16 + (lane >> 4) * 8);
#pragma unroll
                    for (int jp = 0; jp < 4; ++jp) {
                        uint32_t bk[4], bv[4];
                        const int off = (jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * LD + ks * 16 + ((lane >> 3) & 1) * 8;
                        pc::ldsm_x4(bk, sk + off);
                        pc::ldsm_x4(bv, sv + off);
                        pc::mma16816(S[2 * jp], aq, bk[0], bk[1]);
                        pc::mma16816(S[2 * jp + 1], aq, bk[2], bk[3]);
                        pc::mma16816(G[2 * jp], ad, bv[0], bv[1]);          // dP2 = dctx_sel V^T
                        pc::mma16816(G[2 * jp + 1], ad, bv[2], bv[3]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t pk = pc::pack2(S[j][0], S[j][1]);
                    const uint32_t p2 = pc::pack2(__uint_as_float(pk << 16) * scale, __uint_as_float(pk & 0xFFFF0000u) * scale);
                    x[j][0] = __uint_as_float(p2 << 16); x[j][1] = __uint_as_float(p2 & 0xFFFF0000u);
                    gr[j][0] = G[j][0]; gr[j][1] = G[j][1];
                }
            }
            // forward recompute: P1 = softmax(S), P2 = bf16(softmax(P1 + rpb + mask))
            float p1[8][2];
            float mxl;
            float mx = x[0][0];
#pragma unroll
            for (int j = 0; j < 8; ++j) mx = fmaxf(mx, fmaxf(x[j][0], x[j][1]));
            mx = group_max<4>(mx);
            mxl = mx * 1.4426950408889634f;
            float sum = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                p1[j][0] = exp_sub(x[j][0], mxl); p1[j][1] = exp_sub(x[j][1], mxl);
                sum += p1[j][0]; sum += p1[j][1];
            }
            float inv = __fdividef(1.0f, group_sum<4>(sum));
#pragma unroll
            for (int j = 0; j < 8; ++j) { p1[j][0] *= inv; p1[j][1] *= inv; x[j][0] = p1[j][0]; x[j][1] = p1[j][1]; }
            const int r = my_tok < 0 ? 0 : my_tok;
            const int ry = r >> 3, rx = r & 7;
            if (a.use_rpb) {
                if (a.rpb_table) {
                    const float* tb = s.tbl + (ry + 7) * 15 + (rx - 2 * tq + 7);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { x[j][0] += tb[-j * 15]; x[j][1] += tb[-j * 15 - 1]; }
                } else {
                    const float* bd = a.rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                    for (int j = 0; j < 8; ++j) { const float2 b2 = *reinterpret_cast<const float2*>(bd + j * 8); x[j][0] += b2.x; x[j][1] += b2.y; }
                }
            }
            if (a.mask) {
                const float* mk = a.mask + (static_cast<long long>(wg % a.nW_mask) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                for (int j = 0; j < 8; ++j) { const float2 m2 = *reinterpret_cast<const float2*>(mk + j * 8); x[j][0] += m2.x; x[j][1] += m2.y; }
            }
            if (TMASK && (s.tm_live[0] | s.tm_live[1])) {                  // input + shift mask, one add (as the forward)
                const float mr = s.tm[r];
                const bool sh = a.shift > 0 && s.mixed;
                const int rr = s.region[r];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float2 mc = *reinterpret_cast<const float2*>(s.tm + j * 8 + 2 * tq);
                    float m0 = token_mask_term(mr, mc.x), m1 = token_mask_term(mr, mc.y);
                    if (sh) {
                        const int2 rc = *reinterpret_cast<const int2*>(s.region + j * 8 + 2 * tq);
                        m0 += (rc.x != rr) ? -100.0f : 0.f;
                        m1 += (rc.y != rr) ? -100.0f : 0.f;
                    }
                    x[j][0] += m0;
                    x[j][1] += m1;
                }
            } else if (a.shift > 0 && s.mixed) {
                const int rr = s.region[r];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int2 rc = *reinterpret_cast<const int2*>(s.region + j * 8 + 2 * tq);
                    x[j][0] += (rc.x != rr) ? -100.0f : 0.f;
                    x[j][1] += (rc.y != rr) ? -100.0f : 0.f;
                }
            }
            mx = x[0][0];
#pragma unroll
            for (int j = 0; j < 8; ++j) mx = fmaxf(mx, fmaxf(x[j][0], x[j][1]));
            mx = group_max<4>(mx);
            mxl = mx * 1.4426950408889634f;
            sum = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                x[j][0] = exp_sub(x[j][0], mxl); x[j][1] = exp_sub(x[j][1], mxl);
                sum += x[j][0]; sum += x[j][1];
            }
            inv = __fdividef(1.0f, group_sum<4>(sum));
            uint32_t pfrag[8], dsfrag[8];
            float dot = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {                                        // x := P2 (bf16-rounded)
                pfrag[j] = pc::pack2(x[j][0] * inv, x[j][1] * inv);
                x[j][0] = __uint_as_float(pfrag[j] << 16); x[j][1] = __uint_as_float(pfrag[j] & 0xFFFF0000u);
                dot = fmaf(gr[j][0], x[j][0], dot); dot = fmaf(gr[j][1], x[j][1], dot);
            }
            dot = group_sum<4>(dot);
            // softmax backward twice: dA = P2 (dP2 - <dP2,P2>); d(table) += dA; dS = P1 (dA - <dA,P1>) scale
            float dot2 = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                gr[j][0] = x[j][0] * (gr[j][0] - dot); gr[j][1] = x[j][1] * (gr[j][1] - dot);      // gr := dA
                dot2 = fmaf(gr[j][0], p1[j][0], dot2); dot2 = fmaf(gr[j][1], p1[j][1], dot2);
            }
            dot2 = group_sum<4>(dot2);
            if constexpr (DET) {
                if (want_tab && my_tok >= 0) {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float2*>(dab + (warp * 8 + gq) * DA_LD + j * 8 + 2 * tq) = make_float2(gr[j][0], gr[j][1]);
                }
                if (want_dense && my_tok >= 0) {
                    float* dd = a.d_rpb_dense + static_cast<long long>(blockIdx.x) * a.nH * kTok * kTok +
                                (static_cast<long long>(h) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                    for (int j = 0; j < 8; ++j) { dd[j * 8] += gr[j][0]; dd[j * 8 + 1] += gr[j][1]; }
                }
            } else {
                if (want_tab && my_tok >= 0) {
                    float* tb = s.tacc + h * 225 + (ry + 7) * 15 + (rx - 2 * tq + 7);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { atomicAdd(tb - j * 15, gr[j][0]); atomicAdd(tb - j * 15 - 1, gr[j][1]); }
                }
                if (want_dense && my_tok >= 0) {     // gradient w.r.t. the gathered bias [nH, 64, 64] (AttentionLayer.forward's argument)
                    float* dd = a.d_rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                    for (int j = 0; j < 8; ++j) { atomicAdd(dd + j * 8, gr[j][0]); atomicAdd(dd + j * 8 + 1, gr[j][1]); }
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                dsfrag[j] = pc::pack2(p1[j][0] * (gr[j][0] - dot2) * scale, p1[j][1] * (gr[j][1] - dot2) * scale);
                if (my_tok < 0) { dsfrag[j] = 0u; pfrag[j] = 0u; }
                *reinterpret_cast<uint32_t*>(s.dss + (warp * 8 + gq) * PLD + j * 8 + 2 * tq) = dsfrag[j];
                *reinterpret_cast<uint32_t*>(s.p2s + (warp * 8 + gq) * PLD + j * 8 + 2 * tq) = pfrag[j];
            }
            // dq[sel] = dS K  (16 x 32 x 64 per warp; rows 8..15 zero)
            float o[4][4];
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
                for (int c = 0; c < 4; ++c) o[n][c] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const uint32_t af[4] = {dsfrag[2 * ks], 0u, dsfrag[2 * ks + 1], 0u};
#pragma unroll
                for (int nb = 0; nb < 2; ++nb) {
                    uint32_t bf[4];
                    pc::ldsm_x4_t(bf, sk + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + nb * 16 + (lane >> 4) * 8);
                    pc::mma16816(o[2 * nb], af, bf[0], bf[1]);
                    pc::mma16816(o[2 * nb + 1], af, bf[2], bf[3]);
                }
            }
            __nv_bfloat16* st = s.ostage[warp][0];
#pragma unroll
            for (int n = 0; n < 4; ++n)
                *reinterpret_cast<uint32_t*>(st + gq * kHeadDim + n * 8 + 2 * tq) = pc::pack2(o[n][0], o[n][1]);
            __syncwarp();
            {
                const int row = lane >> 2, part = lane & 3;
                const int tok = __shfl_sync(0xffffffffu, my_sel, (warp * 8 + row) & 31);
                if (tok >= 0)
                    *reinterpret_cast<uint4*>(obase + static_cast<long long>(tok) * C3 + part * 8) =
                        *reinterpret_cast<const uint4*>(st + row * kHeadDim + part * 8);
            }
            // dq of the lazy queries is zero
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int c = tid + i * THREADS, rr = c >> 2, part = c & 3;
                if (!((selmask >> rr) & 1ull)) *reinterpret_cast<uint4*>(obase + static_cast<long long>(rr) * C3 + part * 8) = make_uint4(0u, 0u, 0u, 0u);
            }
            // dmean = (1/64) sum over the lazy rows of dctx: row-selector MMA against the dctx tile (warp 3 has one live slot)
            if (warp == 3) {
                float om[4][4];
#pragma unroll
                for (int n = 0; n < 4; ++n)
#pragma unroll
                    for (int c = 0; c < 4; ++c) om[n][c] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    uint32_t af[4] = {0u, 0u, 0u, 0u};
                    if (gq == 0) {
                        const int r0 = ks * 16 + 2 * tq;
                        af[0] = (((selmask >> r0) & 1ull) ? 0u : 0x3C80u) | (((selmask >> (r0 + 1)) & 1ull) ? 0u : 0x3C800000u);
                        af[2] = (((selmask >> (r0 + 8)) & 1ull) ? 0u : 0x3C80u) | (((selmask >> (r0 + 9)) & 1ull) ? 0u : 0x3C800000u);
                    }
#pragma unroll
                    for (int nb = 0; nb < 2; ++nb) {
                        uint32_t bf[4];
                        pc::ldsm_x4_t(bf, sdc + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + nb * 16 + (lane >> 4) * 8);
                        pc::mma16816(om[2 * nb], af, bf[0], bf[1]);
                        pc::mma16816(om[2 * nb + 1], af, bf[2], bf[3]);
                    }
                }
                if (gq == 0) {
#pragma unroll
                    for (int n = 0; n < 4; ++n) { s.dmean[n * 8 + 2 * tq] = om[n][0]; s.dmean[n * 8 + 2 * tq + 1] = om[n][1]; }
                }
            }
        }
        __syncthreads();                                                        // [B3] dS / P2 / dmean exchanged
        if constexpr (DET) {
            if (want_tab) {     // table entry e = (dy + 7) * 15 + (dx + 7) takes, per slot in order, the key at (ry - dy, rx - dx)
                for (int e0 = 0; e0 < 225; e0 += THREADS) {
                    const int e = e0 + tid, ey = e / 15 - 7, ex = e % 15 - 7;
                    float sum = 0.f;
                    for (int sl = 0; sl < kTopU; ++sl) {
                        const int t = __shfl_sync(0xffffffffu, my_sel, sl);
                        const int ly = (t >> 3) - ey, lx = (t & 7) - ex;
                        if (e < 225 && ly >= 0 && ly < 8 && lx >= 0 && lx < 8) sum += dab[sl * DA_LD + ly * 8 + lx];
                    }
                    if (e < 225) s.tacc[h * 225 + e] += sum;
                }
            }
        }

        // ================= phase B: keys 16*warp..+15:  dk = dS^T Q_sel,  dv = P2^T dctx_sel + dmean   (K = 32 slots)
        {
            float okk[4][4], ovv[4][4];
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
                for (int c = 0; c < 4; ++c) { okk[n][c] = 0.f; ovv[n][c] = 0.f; }
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                uint32_t ak[4], av[4];     // A[m = key][k = slot] = tile[slot][key], transposed on load
                const int aoff = (ks * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * PLD + warp * 16 + ((lane >> 3) & 1) * 8;
                pc::ldsm_x4_t(ak, s.dss + aoff);
                pc::ldsm_x4_t(av, s.p2s + aoff);
                int brow = __shfl_sync(0xffffffffu, my_sel, (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) & 31);
                if (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8 >= kTopU || brow < 0) brow = 0;      // dummy slots carry zero dS / P2
#pragma unroll
                for (int nb = 0; nb < 2; ++nb) {
                    uint32_t bq[4], bd[4];  // B[k = slot][n = d] = Q_sel / dctx_sel rows gathered by address
                    pc::ldsm_x4_t(bq, sq + brow * LD + nb * 16 + (lane >> 4) * 8);
                    pc::ldsm_x4_t(bd, sdc + brow * LD + nb * 16 + (lane >> 4) * 8);
                    pc::mma16816(okk[2 * nb], ak, bq[0], bq[1]);
                    pc::mma16816(okk[2 * nb + 1], ak, bq[2], bq[3]);
                    pc::mma16816(ovv[2 * nb], av, bd[0], bd[1]);
                    pc::mma16816(ovv[2 * nb + 1], av, bd[2], bd[3]);
                }
            }
            __nv_bfloat16* stk = s.ostage[warp][0];
            __nv_bfloat16* stv = s.ostage[warp][1];
            __syncwarp();                                                        // phase A's reads of ostage[warp][0] are done
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                const int d = n * 8 + 2 * tq;
                const float m0 = s.dmean[d], m1 = s.dmean[d + 1];
                *reinterpret_cast<uint32_t*>(stk + gq * kHeadDim + d) = pc::pack2(okk[n][0], okk[n][1]);
                *reinterpret_cast<uint32_t*>(stk + (gq + 8) * kHeadDim + d) = pc::pack2(okk[n][2], okk[n][3]);
                *reinterpret_cast<uint32_t*>(stv + gq * kHeadDim + d) = pc::pack2(ovv[n][0] + m0, ovv[n][1] + m1);
                *reinterpret_cast<uint32_t*>(stv + (gq + 8) * kHeadDim + d) = pc::pack2(ovv[n][2] + m0, ovv[n][3] + m1);
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int c = lane + 32 * i, row = c >> 2, part = c & 3;
                __nv_bfloat16* orow = obase + static_cast<long long>(warp * 16 + row) * C3 + part * 8;
                *reinterpret_cast<uint4*>(orow + a.C) = *reinterpret_cast<const uint4*>(stk + row * kHeadDim + part * 8);
                *reinterpret_cast<uint4*>(orow + 2 * a.C) = *reinterpret_cast<const uint4*>(stv + row * kHeadDim + part * 8);
            }
        }
    }
    cp_async_wait<0>();
    __syncthreads();
    if (want_tab) {
        for (int i = tid; i < a.nH * 225; i += THREADS) {
            const int hh = i / 225, rel = i - hh * 225;
            const float v = s.tacc[i];
            if constexpr (DET) a.d_rpb_table[static_cast<long long>(blockIdx.x) * a.nH * 225 + rel * a.nH + hh] = v;
            else if (v != 0.f) atomicAdd(a.d_rpb_table + rel * a.nH + hh, v);
        }
    }
}

// CTAs of a launch (in deterministic mode with sms = 148: the slabs of the bias gradients)
inline long long grid(long long items, int sms, bool det) {
    const long long cap = static_cast<long long>(sms) * (det ? 2 : 3);
    return items < cap ? items : cap;
}

inline cudaError_t launch(const CoreBwdArgs<__nv_bfloat16>& a, int num_sms, bool det, cudaStream_t stream) {
    auto k = det ? (a.tmask ? core_bwd_v2_kernel<true, true> : core_bwd_v2_kernel<false, true>)
                 : (a.tmask ? core_bwd_v2_kernel<true> : core_bwd_v2_kernel<false>);
    const size_t smem = sizeof(Smem) + (det ? sizeof(DetDa) : 0);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const long long items = static_cast<long long>(a.B_) * a.nH;
    k<<<static_cast<unsigned>(grid(items, det ? 148 : num_sms, det)), THREADS, smem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace pcb2
}  // namespace lewin
