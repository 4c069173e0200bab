// ProbSparse window-attention core, forward: one CTA (4 warps) per (window, head).
//
// Reference: ProbAttention.forward, ProbSparse/attn.py:287-342
//   _prob_QK           attn.py:71-152   sampled scores, sparsity measure M, top-u, Q^K^T
//   _get_initial_context attn.py:154-176 mean(V) fill
//   _update_context    attn.py:178-281  softmax -> +rpb -> +mask -> softmax (double softmax!) -> P.V scatter
//
// B200 restatement: the full 64x64 score tile S = Q.K^T is produced on tensor cores (cheaper than
// gathering 25 keys per query, and the top-u rows of S are re-used); the reference's materialised
// K_sample[B_,nH,64,25,D] gather (attn.py:104) becomes a multiplicity matrix cnt[n][m] = #{t :
// idx[n,t] == m}, so  M_n = max_{cnt>0} S[n,m] - (sum_m cnt[n,m] S[n,m]) / 64  (attn.py:117) is a
// quad-shuffle reduction over the MMA accumulators.  Top-u is rank-by-counting (ties -> lower
// index).  Only the 25 selected rows go through the two softmaxes and P.V.
#pragma once
#include "common.cuh"

namespace lewin {

template <typename T>
struct CoreFwdArgs {
    const T* qkv;            // [B_*64, 3C]  q | k | v
    T* ctx;                  // [B_*64, C]
    uint8_t* top;            // [B_, nH, 25] or null
    const float* rpb_table;  // [225, nH] (or null)
    const float* rpb_dense;  // [nH, 64, 64] (or null)
    const int32_t* index_sample;   // [64, 25] key-sample indices (attn.py:91); the multiplicity matrix is built per CTA
    const float* mask;       // dense [nW_mask, 64, 64] or null
    int nW_mask;
    int B_, nH, C;
    int use_rpb;
    // analytic shift mask (My_model_1.py:803-836): row regions are evaluated at shifted-frame row y0 + (row in this map) of an
    // image Hg rows tall (y0 = 0, Hg = H unless the map is a row band of a taller image)
    int shift, H, W, nWw, nWin;
    int y0, Hg;
    // input mask per token [Bm, H, W] (LewinAttnFwdArgs::token_mask) or null; its term and the shift mask's are one add
    const float* tmask;
    int Bm;
};

constexpr int CORE_THREADS = 128;
constexpr int P_LD = 68;    // selected-row score / probability stride
// head_dim D in {32, 64, 128} (d_keys = d_model // n_heads, attn.py:370-372; = embed_dim in this model, My_model_1.py:962):
// q/k row stride D + 4 floats and v row stride D + 8 keep the fragment loads conflict-free for every D (== 4 / 8 mod 32)
template <int D> struct CoreLd { static constexpr int QK = D + 4, V = D + 8; };

template <int D>
struct CoreSmem {
    float q[kTok * CoreLd<D>::QK];
    float k[kTok * CoreLd<D>::QK];
    float v[kTok * CoreLd<D>::V];
    float p[32 * P_LD];           // rows = selection slots (25 used, 7 zero)
    float M[kTok];
    float vmean[D];
    float vpart[4 * D];
    float tbl[232];
    alignas(16) uint8_t cnt[kTok * kTok];
    int slot_of[kTok];            // token -> slot (or -1)
    int tok_of[32];               // slot -> token
    int region[kTok];
    float tm[kTok];               // input mask of the window's tokens (a.tmask)
};

// cnt[n][m] = #{t : idx[n, t] == m} (the reference's K_sample gather, attn.py:88-104, as a multiplicity matrix), built in
// shared memory by the CTA itself: 4 KB, 1600 byte-lane atomics, once per persistent CTA (no pre-pass kernel)
__device__ __forceinline__ void build_cnt_smem(uint8_t* cnt, const int32_t* __restrict__ idx, int tid, int nthreads) {
    uint32_t* c32 = reinterpret_cast<uint32_t*>(cnt);
    for (int i = tid; i < kTok * kTok / 4; i += nthreads) c32[i] = 0u;
    __syncthreads();
    for (int i = tid; i < kTok * kSampleK; i += nthreads) {
        const int n = i / kSampleK, m = idx[i] & 63;
        atomicAdd(&c32[(n * kTok + m) >> 2], 1u << (8 * (m & 3)));      // <= 25 per byte: no carry into the neighbour
    }
    __syncthreads();
}

template <typename T, int D>
__global__ void __launch_bounds__(CORE_THREADS) probsparse_core_fwd_kernel(const CoreFwdArgs<T> a) {
    constexpr int PASSES = Act<T>::kPasses;
    constexpr int QK_LD = CoreLd<D>::QK, V_LD = CoreLd<D>::V;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CoreSmem<D>& s = *reinterpret_cast<CoreSmem<D>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int C3 = 3 * a.C;
    const float scale = rsqrtf(static_cast<float>(D));   // attn.py:327

    // launch-invariant: sample multiplicities
    build_cnt_smem(s.cnt, a.index_sample, tid, CORE_THREADS);

    const int items = a.B_ * a.nH;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int wg = item / a.nH;          // global window index (batch-major)
        const int h = item - wg * a.nH;
        __syncthreads();                     // previous item fully consumed

        // ---- stage q, k, v (64 x D each) as fp32
        {
            const T* base = a.qkv + static_cast<long long>(wg) * kTok * C3 + h * D;
            constexpr int CPR = D / 4;       // float4 chunks per row
            for (int c = tid; c < 3 * kTok * CPR; c += CORE_THREADS) {
                int which = c / (kTok * CPR);
                int rem = c - which * kTok * CPR;
                int r = rem / CPR, d4 = (rem % CPR) * 4;
                float4 v = ld4(base + static_cast<long long>(r) * C3 + which * a.C + d4);
                float* dst = which == 0 ? s.q + r * QK_LD + d4 : which == 1 ? s.k + r * QK_LD + d4 : s.v + r * V_LD + d4;
                *reinterpret_cast<float4*>(dst) = v;
            }
            if (a.use_rpb && a.rpb_table)
                for (int i = tid; i < 225; i += CORE_THREADS) s.tbl[i] = a.rpb_table[i * a.nH + h];
            if (a.shift > 0 && tid < kTok) {
                // region id of each token in the shifted frame (My_model_1.py:809-820)
                int w = wg % a.nWin;
                int wy = w / a.nWw, wx = w - wy * a.nWw;
                int y = a.y0 + wy * 8 + (tid >> 3), x = wx * 8 + (tid & 7);
                int rb = y < a.Hg - 8 ? 0 : (y < a.Hg - a.shift ? 1 : 2);
                int cb = x < a.W - 8 ? 0 : (x < a.W - a.shift ? 1 : 2);
                s.region[tid] = rb * 3 + cb;
            }
            if (a.tmask && tid < kTok) s.tm[tid] = window_token_mask(a.tmask, a.Bm, a.H, a.W, a.nWw, a.nWin, wg, tid);
        }
        __syncthreads();

        // ---- S = Q K^T : warp owns query rows [16*warp, 16*warp+16), all 64 keys
        float acc[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[j][c] = 0.f;
#pragma unroll
        for (int ks = 0; ks < D / 8; ++ks) {
            float af[4];
            const float* pa = s.q + (warp * 16 + gq) * QK_LD + ks * 8 + tq;
            af[0] = pa[0]; af[1] = pa[8 * QK_LD]; af[2] = pa[4]; af[3] = pa[8 * QK_LD + 4];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float bf[2];
                const float* pb = s.k + (j * 8 + gq) * QK_LD + ks * 8 + tq;
                bf[0] = pb[0]; bf[1] = pb[4];
                mma_x<PASSES>(acc[j], af, bf);
            }
        }

        // ---- sparsity measure (attn.py:117) on unscaled scores; bf16 mode rounds S~ first (A.4)
        {
            float mx[2] = {-INFINITY, -INFINITY}, sm[2] = {0.f, 0.f};
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = warp * 16 + gq + half * 8;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = j * 8 + 2 * tq;
                    const uint16_t c2 = *reinterpret_cast<const uint16_t*>(s.cnt + r * kTok + col);
                    const int c0 = c2 & 0xff, c1 = c2 >> 8;
                    const float s0 = Act<T>::round(acc[j][half * 2 + 0]);
                    const float s1 = Act<T>::round(acc[j][half * 2 + 1]);
                    if (c0) { mx[half] = fmaxf(mx[half], s0); sm[half] += c0 * s0; }
                    if (c1) { mx[half] = fmaxf(mx[half], s1); sm[half] += c1 * s1; }
                }
                mx[half] = group_max<4>(mx[half]);
                sm[half] = group_sum<4>(sm[half]);
                if (tq == 0) s.M[r] = mx[half] - sm[half] * (1.0f / kTok);
            }
        }
        __syncthreads();

        // ---- top-u by rank counting (attn.py:122); ties -> lower index first
        if (tid < kTok) {
            const float mine = s.M[tid];
            int rank = 0;
#pragma unroll 8
            for (int m = 0; m < kTok; ++m) {
                const float o = s.M[m];
                rank += (o > mine) || (o == mine && m < tid);
            }
            const int slot = rank < kTopU ? rank : -1;
            s.slot_of[tid] = slot;
            if (slot >= 0) {
                s.tok_of[slot] = tid;
                if (a.top) a.top[static_cast<long long>(item) * kTopU + slot] = static_cast<uint8_t>(tid);
            }
        } else if (tid < kTok + 7) {
            s.tok_of[kTopU + tid - kTok] = -1;
        }
        __syncthreads();

        // ---- selected rows: scaled scores -> smem (attn.py:150, 327-329)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = warp * 16 + gq + half * 8;
            const int slot = s.slot_of[r];
            if (slot >= 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float2 v;
                    v.x = Act<T>::round(Act<T>::round(acc[j][half * 2 + 0]) * scale);
                    v.y = Act<T>::round(Act<T>::round(acc[j][half * 2 + 1]) * scale);
                    *reinterpret_cast<float2*>(s.p + slot * P_LD + j * 8 + 2 * tq) = v;
                }
            }
        }
        // column means of V (attn.py:168): 4 row quarters x D columns, then combined
        for (int e = tid; e < 4 * D; e += CORE_THREADS) {
            const int d = e % D, part = e / D;
            float sum = 0.f;
#pragma unroll
            for (int r = 0; r < 16; ++r) sum += s.v[(part * 16 + r) * V_LD + d];
            s.vpart[part * D + d] = sum;
        }
        __syncthreads();
        for (int d = tid; d < D; d += CORE_THREADS)
            s.vmean[d] = Act<T>::round((s.vpart[d] + s.vpart[D + d] + s.vpart[2 * D + d] + s.vpart[3 * D + d]) * (1.0f / kTok));

        // ---- softmax -> +rpb -> +mask -> softmax on the selected rows (attn.py:195-264)
        for (int slot = warp; slot < 32; slot += 4) {
            float* prow = s.p + slot * P_LD;
            if (slot >= kTopU) { prow[lane] = 0.f; prow[lane + 32] = 0.f; continue; }
            const int r = s.tok_of[slot];
            float x0 = prow[lane], x1 = prow[lane + 32];
            float mx = group_max<32>(fmaxf(x0, x1));
            float e0 = expf(x0 - mx), e1 = expf(x1 - mx);
            float inv = 1.0f / group_sum<32>(e0 + e1);
            float p0 = e0 * inv, p1 = e1 * inv;                  // P1 (first softmax)
            if (a.use_rpb) {                                     // My_model_1.py:366-381 index, attn.py:229
                if (a.rpb_table) {
                    const int ry = r >> 3, rx = r & 7;
                    const int c0 = lane, c1 = lane + 32;
                    p0 += s.tbl[(ry - (c0 >> 3) + 7) * 15 + (rx - (c0 & 7) + 7)];
                    p1 += s.tbl[(ry - (c1 >> 3) + 7) * 15 + (rx - (c1 & 7) + 7)];
                } else {
                    const float* brow = a.rpb_dense + (static_cast<long long>(h) * kTok + r) * kTok;
                    p0 += brow[lane];
                    p1 += brow[lane + 32];
                }
            }
            if (a.mask) {                                        // attn.py:250: window index within the image
                const float* mrow = a.mask + (static_cast<long long>(wg % a.nW_mask) * kTok + r) * kTok;
                p0 += mrow[lane];
                p1 += mrow[lane + 32];
            }
            if (a.tmask) {                                       // input + shift mask, one add (== the dense sum)
                const float mr = s.tm[r];
                float m0 = token_mask_term(mr, s.tm[lane]), m1 = token_mask_term(mr, s.tm[lane + 32]);
                if (a.shift > 0) {
                    const int rr = s.region[r];
                    m0 += (s.region[lane] != rr) ? -100.0f : 0.f;
                    m1 += (s.region[lane + 32] != rr) ? -100.0f : 0.f;
                }
                p0 += m0;
                p1 += m1;
            } else if (a.shift > 0) {
                const int rr = s.region[r];
                p0 += (s.region[lane] != rr) ? -100.0f : 0.f;
                p1 += (s.region[lane + 32] != rr) ? -100.0f : 0.f;
            }
            mx = group_max<32>(fmaxf(p0, p1));
            e0 = expf(p0 - mx); e1 = expf(p1 - mx);
            inv = 1.0f / group_sum<32>(e0 + e1);
            prow[lane] = Act<T>::round(e0 * inv);                // P2 (second softmax)
            prow[lane + 32] = Act<T>::round(e1 * inv);
        }
        __syncthreads();

        // ---- ctx_sel[32 x D] = P2[32 x 64] . V[64 x D]  (attn.py:272): warp -> (m-tile, D/16 n-tiles)
        {
            constexpr int NT = D / 16;
            const int mt = warp & 1, nb = (warp >> 1) * NT;
            float o[NT][4];
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) o[j][c] = 0.f;
#pragma unroll
            for (int ks = 0; ks < kTok / 8; ++ks) {
                float af[4];
                const float* pa = s.p + (mt * 16 + gq) * P_LD + ks * 8 + tq;
                af[0] = pa[0]; af[1] = pa[8 * P_LD]; af[2] = pa[4]; af[3] = pa[8 * P_LD + 4];
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    float bf[2];
                    const float* pb = s.v + (ks * 8 + tq) * V_LD + (nb + j) * 8 + gq;
                    bf[0] = pb[0]; bf[1] = pb[4 * V_LD];
                    mma_x<PASSES>(o[j], af, bf);
                }
            }
            T* cbase = a.ctx + static_cast<long long>(wg) * kTok * a.C + h * D;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int slot = mt * 16 + gq + half * 8;
                const int r = s.tok_of[slot];
                if (r >= 0) {
#pragma unroll
                    for (int j = 0; j < NT; ++j)
                        st2(cbase + static_cast<long long>(r) * a.C + (nb + j) * 8 + 2 * tq, o[j][half * 2], o[j][half * 2 + 1]);
                }
            }
            // lazy queries: mean(V) (attn.py:172)
            for (int c = tid; c < kTok * (D / 4); c += CORE_THREADS) {
                const int r = c / (D / 4), d4 = (c % (D / 4)) * 4;
                if (s.slot_of[r] < 0)
                    st4(cbase + static_cast<long long>(r) * a.C + d4, *reinterpret_cast<const float4*>(s.vmean + d4));
            }
        }
    }
}

template <typename T, int D>
cudaError_t launch_core_fwd_d(const CoreFwdArgs<T>& a, int num_sms, cudaStream_t stream) {
    auto k = probsparse_core_fwd_kernel<T, D>;
    const size_t smem = sizeof(CoreSmem<D>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    long long items = static_cast<long long>(a.B_) * a.nH;
    const int resident = static_cast<int>((227 * 1024) / (smem + 1024));      // CTAs per SM by shared memory
    long long cap = static_cast<long long>(num_sms) * (resident < 1 ? 1 : resident > 4 ? 4 : resident) * 4;   // ~4 waves before looping
    unsigned grid = static_cast<unsigned>(items < cap ? items : cap);
    k<<<grid, CORE_THREADS, smem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace lewin
