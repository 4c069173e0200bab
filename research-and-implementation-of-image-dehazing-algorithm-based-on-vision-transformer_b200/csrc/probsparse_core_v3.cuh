// ProbSparse window-attention core, forward, bf16 — register-resident restatement (ProbSparse/attn.py:287-342).
//
// Same algorithm, rounding points and selection rule as probsparse_core_fwd_kernel (probsparse_core.cuh); restructured around the measured
// bound of that kernel (instruction issue + 7 block barriers per (window, head) item, ~7500 warp-instructions per item):
//   * q | k | v of the NEXT item are prefetched with cp.async into a second shared-memory buffer while the current one is
//     processed (the item's DRAM latency is never exposed);
//   * the sample multiplicities of a thread's MMA-fragment positions never change, so they live in registers (16 packed
//     half2 + one 32-bit "sampled" mask) instead of a 16 KB shared table re-read for every item;
//   * the 25 selected rows are re-gathered straight from Q by ldmatrix row addresses (8 slots per warp), S_sel = Q_sel K^T
//     is recomputed on the tensor cores (bit-identical to the first pass) and scale -> softmax -> +rpb -> +mask -> softmax
//     -> P.V all happen on the accumulator fragments: no score / probability tile in shared memory, row reductions are
//     two quad shuffles, P2 feeds the P.V MMA directly as its A fragment;
//   * mean(V) for the lazy queries comes out of the same P.V MMA (a spare tile row holds the constant 1/64);
//   * 3 block barriers per item instead of 7.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "probsparse_core_bf16.cuh"

namespace lewin {
namespace pc3 {

constexpr int THREADS = 128;
constexpr int CTAS = 5;                                 // resident CTAs per SM the register budget is compiled for (96 registers;
                                                        // 6 CTAs at 80 registers measured 1.6 % slower: the kernel is issue-bound)
constexpr int LD = 40;                                  // bf16 row stride of the q/k/v tiles (80 B: conflict-free ldmatrix)
constexpr int TILE = kTok * LD;                         // elements per q / k / v tile

struct Smem {
    alignas(16) __nv_bfloat16 qkv[2][3 * TILE];                     // double-buffered q | k | v
    alignas(16) float M[kTok];
    float tbl[232];
    int slot_of[kTok];
    int tok_of[32];
    alignas(8) int region[kTok];
    int mixed;                                          // window crosses a shift-mask region border
    alignas(16) __nv_bfloat16 vmean[kHeadDim];
    alignas(16) __nv_bfloat16 ostage[4][8 * kHeadDim];              // per-warp staging of the 8 selected context rows
};

__global__ void __launch_bounds__(THREADS, CTAS) probsparse_core_v3_kernel(const CoreFwdArgs<__nv_bfloat16> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int C3 = 3 * a.C;
    const float scale = rsqrtf(static_cast<float>(kHeadDim));
    const int items = a.B_ * a.nH;

    // ---- per-thread constants: multiplicities of my fragment positions (rows warp*16 + gq (+8), columns j*8 + 2tq (+1)).
    //      The multiplicity matrix cnt[n][m] = #{t : idx[n, t] == m} (attn.py:88-104) is built by the CTA itself in the second
    //      q|k|v buffer (free until the first in-loop prefetch): no pre-pass kernel, no global table.
    __half2 cntp[2][8];
    uint32_t sampled = 0;
    {
        uint8_t* cnt = reinterpret_cast<uint8_t*>(s.qkv[1]);
        build_cnt_smem(cnt, a.index_sample, tid, THREADS);
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int r = warp * 16 + gq + half * 8, c = j * 8 + 2 * tq;
                const uint32_t c2 = *reinterpret_cast<const uint16_t*>(cnt + r * kTok + c);
                const int c0 = c2 & 0xFF, c1 = c2 >> 8;
                cntp[half][j] = __halves2half2(__int2half_rn(c0), __int2half_rn(c1));
                if (c0) sampled |= 1u << (half * 16 + j * 2);
                if (c1) sampled |= 1u << (half * 16 + j * 2 + 1);
            }
        __syncthreads();                                  // everyone has read the table before the buffer is reused
    }
    if (tid < 32) s.tok_of[tid] = -1;                   // slots 25..31 stay -1 for the whole kernel
    // the grid is a multiple of nH whenever it is smaller than the item count, so a CTA keeps one head: its bias table
    // is staged once
    const bool fixed_head = (gridDim.x % a.nH) == 0;
    if (a.use_rpb && a.rpb_table && fixed_head)
        for (int i = tid; i < 225; i += THREADS) s.tbl[i] = a.rpb_table[i * a.nH + static_cast<int>(blockIdx.x) % a.nH];

    auto prefetch = [&](int item, int buf) {
        const int wg = item / a.nH, h = item - wg * a.nH;
        const __nv_bfloat16* base = a.qkv + static_cast<long long>(wg) * kTok * C3 + h * kHeadDim;
        __nv_bfloat16* dst = s.qkv[buf];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int c = tid + i * THREADS;
            const int which = c >> 8, r = (c >> 2) & 63, ch = c & 3;
            cp_async16(dst + which * TILE + r * LD + ch * 8, base + static_cast<long long>(r) * C3 + which * a.C + ch * 8);
        }
    };

    int item = blockIdx.x, buf = 0;
    if (item < items) prefetch(item, 0);
    cp_async_commit();
    for (; item < items; item += gridDim.x, buf ^= 1) {
        const int wg = item / a.nH, h = item - wg * a.nH;
        cp_async_wait<0>();
        __syncthreads();                                                        // [B1] this item's q|k|v landed; previous item fully retired
        if (item + static_cast<int>(gridDim.x) < items) prefetch(item + gridDim.x, buf ^ 1);
        cp_async_commit();
        const __nv_bfloat16* sq = s.qkv[buf];
        const __nv_bfloat16* sk = sq + TILE;
        const __nv_bfloat16* sv = sk + TILE;
        // per-item tables (visible to their readers after B2 / B3)
        if (a.use_rpb && a.rpb_table && !fixed_head)
            for (int i = tid; i < 225; i += THREADS) s.tbl[i] = a.rpb_table[i * a.nH + h];
        if (a.shift > 0) {
            if (tid < kTok) {
                const int w = wg % a.nWin, wy = w / a.nWw, wx = w - wy * a.nWw;
                const int y = a.y0 + wy * 8 + (tid >> 3), x = wx * 8 + (tid & 7);
                const int rb = y < a.Hg - 8 ? 0 : (y < a.Hg - a.shift ? 1 : 2);
                const int cb = x < a.W - 8 ? 0 : (x < a.W - a.shift ? 1 : 2);
                s.region[tid] = rb * 3 + cb;
                if (tid == 0) {                                                  // only the last window row / column is mixed
                    const int w0 = wg % a.nWin, wy0 = w0 / a.nWw, wx0 = w0 - wy0 * a.nWw;
                    s.mixed = (a.y0 + wy0 * 8 + 8 > a.Hg - 8) || (wx0 * 8 + 8 > a.W - 8);
                }
            }
        }

        // ================= phase 1: S = Q K^T for rows 16*warp..+15, sparsity measure M (attn.py:71-117)
        {
            float acc[8][4];
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                uint32_t af[4];
                pc::ldsm_x4(af, sq + (warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + ks * 16 + (lane >> 4) * 8);
#pragma unroll
                for (int jp = 0; jp < 4; ++jp) {
                    uint32_t bf[4];
                    pc::ldsm_x4(bf, sk + (jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * LD + ks * 16 + ((lane >> 3) & 1) * 8);
                    pc::mma16816(acc[2 * jp], af, bf[0], bf[1]);
                    pc::mma16816(acc[2 * jp + 1], af, bf[2], bf[3]);
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float mx = -INFINITY, sm = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    // S~ is a bf16 matmul output under autocast: round once (A.4)
                    const uint32_t pk = pc::pack2(acc[j][half * 2], acc[j][half * 2 + 1]);
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
                if (tq == 0) s.M[warp * 16 + gq + half * 8] = mx - sm * (1.0f / kTok);
            }
        }
        __syncthreads();                                                        // [B2] M complete

        // ================= phase 2: top-u by rank counting (ties -> lower index), 16 rows per warp, 2 lanes per row
        {
            const int r = warp * 16 + (lane & 15), hf = lane >> 4;
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
                    if (a.top) a.top[static_cast<long long>(item) * kTopU + slot] = static_cast<uint8_t>(r);
                }
            }
        }
        __syncthreads();                                                        // [B3] slots assigned

        // ================= phase 3: slots 8*warp..+7 = rows 0..7 of this warp's m16 tile (rows 8..15 are dummies)
        {
            const int my_tok = s.tok_of[warp * 8 + gq];                          // token of the row this thread's fragments hold (-1: dummy)
            float acc[8][2];                                                      // row gq only
            {
                float full[8][4];
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) full[j][c] = 0.f;
                int arow = s.tok_of[warp * 8 + (lane & 7)];
                if (arow < 0) arow = 0;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    uint32_t af[4];
                    pc::ldsm_x4(af, sq + arow * LD + ks * 16 + (lane >> 4) * 8);
#pragma unroll
                    for (int jp = 0; jp < 4; ++jp) {
                        uint32_t bf[4];
                        pc::ldsm_x4(bf, sk + (jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * LD + ks * 16 + ((lane >> 3) & 1) * 8);
                        pc::mma16816(full[2 * jp], af, bf[0], bf[1]);
                        pc::mma16816(full[2 * jp + 1], af, bf[2], bf[3]);
                    }
                }
                // bf16(S) * scale -> bf16 (attn.py:150, 327-329)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t pk = pc::pack2(full[j][0], full[j][1]);
                    const uint32_t p2 = pc::pack2(__uint_as_float(pk << 16) * scale, __uint_as_float(pk & 0xFFFF0000u) * scale);
                    acc[j][0] = __uint_as_float(p2 << 16);
                    acc[j][1] = __uint_as_float(p2 & 0xFFFF0000u);
                }
            }
            // softmax 1
            float mxl;
            float mx = acc[0][0];
#pragma unroll
            for (int j = 0; j < 8; ++j) mx = fmaxf(mx, fmaxf(acc[j][0], acc[j][1]));
            mx = group_max<4>(mx);
            mxl = mx * 1.4426950408889634f;
            float sum = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                acc[j][0] = exp_sub(acc[j][0], mxl); acc[j][1] = exp_sub(acc[j][1], mxl);
                sum += acc[j][0]; sum += acc[j][1];
            }
            float inv = __fdividef(1.0f, group_sum<4>(sum));
#pragma unroll
            for (int j = 0; j < 8; ++j) { acc[j][0] *= inv; acc[j][1] *= inv; }
            // + relative position bias, + masks (added to PROBABILITIES: attn.py:195-264), live rows only
            const int r = my_tok < 0 ? 0 : my_tok;
            if (a.use_rpb) {
                if (a.rpb_table) {
                    const int ry = r >> 3, rx = r & 7;
                    const float* tb = s.tbl + (ry + 7) * 15 + (rx - 2 * tq + 7);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { acc[j][0] += tb[-j * 15]; acc[j][1] += tb[-j * 15 - 1]; }
                } else {
                    const float* bd = a.rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                    for (int j = 0; j < 8; ++j) { const float2 b2 = *reinterpret_cast<const float2*>(bd + j * 8); acc[j][0] += b2.x; acc[j][1] += b2.y; }
                }
            }
            if (a.mask) {
                const float* mk = a.mask + (static_cast<long long>(wg % a.nW_mask) * kTok + r) * kTok + 2 * tq;
#pragma unroll
                for (int j = 0; j < 8; ++j) { const float2 m2 = *reinterpret_cast<const float2*>(mk + j * 8); acc[j][0] += m2.x; acc[j][1] += m2.y; }
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
            // softmax 2 -> P2 (bf16), kept as the A fragments of the P.V MMA
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
            const bool mean_row = (warp == 3 && gq == 7);                        // slot 31 is never live: its row computes mean(V)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                pfrag[j] = pc::pack2(acc[j][0] * inv, acc[j][1] * inv);
                if (my_tok < 0) pfrag[j] = mean_row ? 0x3C803C80u : 0u;          // bf16 1/64 | zero row
            }
            // ctx rows = P2 . V  (16 x 32 x 64 per warp; rows 8..15 are zero)
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
                    pc::ldsm_x4_t(bf, sv + (ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LD + nb * 16 + (lane >> 4) * 8);
                    pc::mma16816(o[2 * nb], af, bf[0], bf[1]);
                    pc::mma16816(o[2 * nb + 1], af, bf[2], bf[3]);
                }
            }
            // selected rows: stage the warp's 8 x 32 tile, then one 16-byte store per lane (attn.py:271 scatter)
            __nv_bfloat16* cbase = a.ctx + static_cast<long long>(wg) * kTok * a.C + h * kHeadDim;
            __nv_bfloat16* st = s.ostage[warp];
#pragma unroll
            for (int n = 0; n < 4; ++n)
                *reinterpret_cast<uint32_t*>(st + gq * kHeadDim + n * 8 + 2 * tq) = pc::pack2(o[n][0], o[n][1]);
            if (mean_row) {
#pragma unroll
                for (int n = 0; n < 4; ++n)
                    *reinterpret_cast<uint32_t*>(s.vmean + n * 8 + 2 * tq) = pc::pack2(o[n][0], o[n][1]);
            }
            __syncwarp();
            {
                const int row = lane >> 2, part = lane & 3;
                const int tok = s.tok_of[warp * 8 + row];
                if (tok >= 0)
                    *reinterpret_cast<uint4*>(cbase + static_cast<long long>(tok) * a.C + part * 8) =
                        *reinterpret_cast<const uint4*>(st + row * kHeadDim + part * 8);
            }
            // lazy queries: mean(V) (attn.py:168-172), written by the warp that produced it
            if (warp == 3) {
                const uint4 vm = *reinterpret_cast<const uint4*>(s.vmean + (lane & 3) * 8);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int rr = (lane >> 2) + i * 8;
                    if (s.slot_of[rr] < 0)
                        *reinterpret_cast<uint4*>(cbase + static_cast<long long>(rr) * a.C + (lane & 3) * 8) = vm;
                }
            }
        }
    }
    cp_async_wait<0>();
}

inline cudaError_t launch(const CoreFwdArgs<__nv_bfloat16>& a, int num_sms, cudaStream_t stream) {
    auto k = probsparse_core_v3_kernel;
    const size_t smem = sizeof(Smem);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const long long items = static_cast<long long>(a.B_) * a.nH;
    long long cap = static_cast<long long>(num_sms) * CTAS;
    cap -= cap % a.nH;                                   // one head per CTA (see fixed_head)
    if (cap < a.nH) cap = a.nH;
    k<<<static_cast<unsigned>(items < cap ? items : cap), THREADS, smem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace pc3

// head_dim = C / nH in {32, 64, 128}; bf16 at head_dim 32 runs the register-resident kernel above
template <typename T>
cudaError_t launch_core_fwd(const CoreFwdArgs<T>& a, int num_sms, cudaStream_t stream) {
    const int D = a.C / a.nH;
    if (D == 32) {
        if constexpr (Act<T>::kIsBf16) return pc3::launch(a, num_sms, stream);
        else return launch_core_fwd_d<T, 32>(a, num_sms, stream);
    }
    if (D == 64) return launch_core_fwd_d<T, 64>(a, num_sms, stream);
    if (D == 128) return launch_core_fwd_d<T, 128>(a, num_sms, stream);
    return cudaErrorInvalidValue;
}
}  // namespace lewin
