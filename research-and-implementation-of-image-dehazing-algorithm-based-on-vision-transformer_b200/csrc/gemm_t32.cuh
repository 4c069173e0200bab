// fp32 token GEMM on tcgen05 (kind::tf32) with 3xTF32 error compensation -- the reference's own inference precision
// (test_long_GPU.py:91 runs the model in fp32, no autocast) on the 5th-generation tensor cores:
//
//   Y = epi( LN?(A)[M,K] * W[N,K]^T + bias ),       A, W, Y fp32
//
// Same contract as gemm_fused_kernel<float> (q|k|v projections attn.py:420-422, out projection :456, LeFF linear1
// My_model_1.py:508, linear2 :529; LN from precomputed row statistics, roll + window_partition / window_reverse as row
// addressing, bias, erf GELU, DropPath * residual), which it replaces for the forward pass.  An fp32 operand x is split
// into hi = tf32(x) and lo = x - hi; a product is accumulated as a_lo*b_hi + a_hi*b_lo + a_hi*b_hi (the a_lo*b_lo term is
// below 2^-22 relative), so the result is fp32-grade -- the top-u selection downstream of q|k|v is precision-critical
// (SURVEY finding 9) -- at three tensor-core passes instead of one.
//
// One persistent CTA per SM, every hand-over an mbarrier:
//   * 16 producer warps: fp32 k-chunks (32 floats = one 128-byte swizzle row) of A (gathered through roll +
//                        window_partition) and of W go global -> registers (DA k-chunks of A and two of W in flight per
//                        thread) -> LayerNorm (A only) -> hi / lo split -> the stage's four swizzled tiles; the only
//                        wait on the tensor core is for the stage it consumed S k-chunks ago.  The per-tile row table
//                        (gathered token index, LayerNorm mean / rstd) is loaded one tile ahead;
//   * 1 MMA thread     : per k-chunk 4 k8-steps x 3 tcgen05.mma kind::tf32 (M = 128, N = BN) into one of two TMEM
//                        accumulator stages; tcgen05.commit frees the stage / publishes the accumulator;
//   * 4 or 8 epilogue warps: tcgen05.ld (thread == row) -> bias -> erf GELU | DropPath * residual -> per-warp staging
//                        tile -> row-cooperative coalesced 16-byte stores through window_reverse + un-roll; the residual
//                        rows of the next tile are prefetched into shared memory by cp.async (BN <= 128).
// Tiles are walked column-fastest so the CTAs that work on one row band share its A rows in L2.
// What bounds it (cycle counters per role, scripts/t32_prof.py; ncu profiles/r2_*t32*): the K = C GEMMs with wide outputs
// (linear1, out) by the epilogue warps, the others by the producers' memory latency; the tensor pipe is 20-35 % busy.
#pragma once
#include "gemm_fused.cuh"
#include "tc_helpers.cuh"

namespace lewin {
namespace t32 {

constexpr int BM = 128;
constexpr int KC = 32;                        // floats per k-chunk: 128-byte rows (SWIZZLE_128B)
constexpr int A_TILE = BM * 128;              // bytes of one [128 x 32] fp32 tile
constexpr int STG_ROW = 80;                   // staging row: 16 fp32 columns (64 B) + 16 B pad (conflict-free 16-byte accesses)
constexpr int STG_BUF = 32 * STG_ROW;
constexpr int NTAB = 8;                       // per-tile row tables in flight (the A loads run up to DA tiles ahead of the convert)
constexpr int SMEM_MAX = 227 * 1024;

#ifdef LEWIN_T32_PROF_BUILD
// Diagnostic build (-DLEWIN_T32_PROF_BUILD, run with LEWIN_T32_PROF=1): per-role cycle counters, launch i since the last
// reset counts into slot i % 8:  [0] producer total  [1] producer table barrier  [2] producer wait-for-free-stage
// [3] stages  [4] MMA thread total  [5] MMA wait-for-accumulator  [6] MMA wait-for-stage  [7] tiles  [8] CTA total
// [9] epilogue warp 0 wait-for-accumulator  [10] CTAs
#define T32P(x) x
inline unsigned long long* prof_buffer() {
    static unsigned long long* buf = [] {
        const char* e = getenv("LEWIN_T32_PROF");
        unsigned long long* p = nullptr;
        if (e && e[0] == '1' && cudaMalloc(&p, 128 * sizeof(unsigned long long)) == cudaSuccess) cudaMemset(p, 0, 128 * sizeof(unsigned long long));
        return p;
    }();
    return buf;
}
inline int& prof_launches() { static int n = 0; return n; }
inline unsigned long long* prof_slot() {
    unsigned long long* b = prof_buffer();
    return b ? b + 16 * (prof_launches()++ % 8) : nullptr;
}
#else
#define T32P(x)
inline unsigned long long* prof_buffer() { return nullptr; }
inline int& prof_launches() { static int n = 0; return n; }
inline unsigned long long* prof_slot() { return nullptr; }
#endif

__device__ __forceinline__ void mma_tf32_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(tc::smem_u32(bar)) : "memory");
}
template <int PT> __device__ __forceinline__ void producer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(PT) : "memory"); }
// 32 lanes x 16 columns of fp32: thread i of the warp gets lane (lane_base + i), columns [col, col + 16)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// byte offset of 16-byte piece `c` (0..7) of row `r` in a SWIZZLE_128B tile of 128-byte rows
__device__ __forceinline__ uint32_t swz(int r, int c) { return (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4); }

// hi = x rounded to tf32 (nearest, ties away: the same value cvt.rna.tf32.f32 gives for finite x, in two integer
// instructions -- the cvt expands to four with its NaN / Inf select); lo = x - hi is exact in fp32 and is handed to the
// tensor core as it is: kind::tf32 reads the upper 19 bits of the 32-bit container, and lo's 12 significant bits lose at
// most 2^-22 of x to that truncation.
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
    hi.x = tf32_hi(v.x); hi.y = tf32_hi(v.y); hi.z = tf32_hi(v.z); hi.w = tf32_hi(v.w);
    lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}

template <int BN>
constexpr size_t stage_bytes() { return 2 * A_TILE + 2 * static_cast<size_t>(BN) * 128; }
// per-warp residual tile in shared memory: 32 rows x (BN + 4) floats (the pad keeps rows 16-byte aligned and staggers banks)
template <int BN, int EPI>
__host__ __device__ constexpr bool resid_in_smem() { return EPI == EPI_BIAS_RESID && BN <= 128; }
template <int BN, int EPI>
__host__ __device__ constexpr size_t resid_bytes() { return resid_in_smem<BN, EPI>() ? 32 * (BN + 4) * 4 : 0; }
template <int BN, int EPI, int NEW>
constexpr size_t fixed_smem() {
    return 1024 /*align*/ + NEW * (STG_BUF + resid_bytes<BN, EPI>()) + NTAB * BM * 12 + (2 * 8 + 4) * 8 + 16;
}

// BN: tile columns; NEW / NPW: epilogue / producer warps; DA: k-chunks of A in flight per producer thread
template <int BN, int EPI, int NEW, int NPW, int DA>
__global__ void __launch_bounds__((NEW + 1 + NPW) * 32, 1) gemm_t32_kernel(const GemmArgs<float> g, int row_tiles, int col_tiles, int nkc, int S,
                                                                          unsigned long long* prof) {
    constexpr int MMA_WARP = NEW;
    constexpr int PTHREADS = NPW * 32;
    constexpr int RPP = PTHREADS / 8;              // rows per producer pass (8 lanes x 16 B = one 128-byte row piece)
    constexpr int AP = BM / RPP;                   // producer passes over the A rows
    constexpr int WP = (BN + RPP - 1) / RPP;       // ... over the W rows (the last pass may be partial: BN = 96, RPP = 64)
    constexpr int NCG = NEW / 4;                   // epilogue column groups
    constexpr int W_TILE = BN * 128;
    constexpr int STAGE = 2 * A_TILE + 2 * W_TILE;
    constexpr int ACC = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;     // TMEM columns per accumulator stage
    constexpr int TMEM_COLS = 2 * ACC;
    constexpr int NCH = BN / 32;                   // 32-column epilogue chunks
    constexpr bool RS = resid_in_smem<BN, EPI>();
    constexpr int RROW = (BN + 4) * 4;             // bytes per residual row in shared memory
    constexpr int RBUF = static_cast<int>(resid_bytes<BN, EPI>());
    constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                               (static_cast<uint32_t>(BM >> 4) << 24);            // D = f32, A = B = tf32, K-major
    static_assert(BN % 32 == 0 && BN <= 256, "tile width");
    static_assert(NEW % 4 == 0 && BM % RPP == 0 && DA % 2 == 0 && DA + 3 <= NTAB, "warp split / ring depth");
    (void)prof;

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* ring = base;                                         // [S][A_hi | A_lo | W_hi | W_lo]
    unsigned char* stg = ring + static_cast<size_t>(S) * STAGE;         // [NEW][STG_BUF + RBUF]
    uint32_t* t_tok = reinterpret_cast<uint32_t*>(stg + NEW * (STG_BUF + RBUF)); // [NTAB][BM] A row (token) index, 0xFFFFFFFF = beyond M
    float* t_mu = reinterpret_cast<float*>(t_tok + NTAB * BM);          // [NTAB][BM]
    float* t_rs = t_mu + NTAB * BM;                                     // [NTAB][BM]
    uint64_t* full = reinterpret_cast<uint64_t*>(t_rs + NTAB * BM);     // [8]
    uint64_t* empty = full + 8;                                         // [8]
    uint64_t* tfull = empty + 8;                                        // [2]
    uint64_t* tempty = tfull + 2;                                       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int total_tiles = row_tiles * col_tiles;
    const int my_tiles = (total_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
    const bool has_ln = g.mean != nullptr;

    if (tid == 0) {
        for (int i = 0; i < S; ++i) { tc::mbar_init(&full[i], NPW); tc::mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&tfull[i], 1); tc::mbar_init(&tempty[i], NEW * 32); }
        tc::fence_barrier_init();
    }
    if (warp == MMA_WARP) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;
    T32P(const long long cta_t0 = clock64();)

    if (warp > MMA_WARP) {
        // ============================================================ producers
        const int pt = tid - (MMA_WARP + 1) * 32;
        const int row_l = pt >> 3, ch = pt & 7;        // 8 lanes x 16 B = one 128-byte row piece; RPP rows per pass
        const uint32_t sw0 = swz(row_l, ch);           // pass p adds p * RPP * 128 bytes, the XOR term depends on row_l & 7 only
        const int total = my_tiles * nkc;
        T32P(long long p_bar = 0; long long p_empty = 0; const long long p_t0 = clock64();)
        // register rings: A rows come from HBM at the bandwidth-bound levels, so DA k-chunks of A are kept in flight per
        // thread; the W rows (L2 / L1 resident) run two k-chunks ahead
        float4 abuf[DA][AP], wbuf[2][WP];
        // row table of a tile, fetched one tile ahead of its first use (threads pt < BM own one row each): the LayerNorm
        // statistics are a dependent global load, and every producer waits on the table at the tile boundary
        uint32_t n_tok = 0xFFFFFFFFu;
        float n_mu = 0.f, n_rs = 1.f;
        auto fetch_row = [&](int it) {                 // it: this CTA's tile counter
            n_tok = 0xFFFFFFFFu; n_mu = 0.f; n_rs = 1.f;
            if (pt < BM && it < my_tiles) {
                const int t = static_cast<int>(blockIdx.x) + it * static_cast<int>(gridDim.x);
                const uint32_t m = static_cast<uint32_t>(t / col_tiles) * BM + pt;
                if (m < g.M) {
                    n_tok = g.mapA ? g.map.token32(m) : m;
                    if (has_ln) { n_mu = __ldg(g.mean + n_tok); n_rs = __ldg(g.rstd + n_tok); }
                }
            }
        };
        fetch_row(0);
        int l_it = 0, l_kc = 0;                        // A-load stream position
        auto load_a = [&](float4 (&a)[AP], int j) {
            if (j >= total) return;
            const int tb = (l_it & (NTAB - 1)) * BM;
            if (l_kc == 0) {
                if (pt < BM) { t_tok[tb + pt] = n_tok; t_mu[tb + pt] = n_mu; t_rs[tb + pt] = n_rs; }
                fetch_row(l_it + 1);
                T32P(const long long tb0 = clock64();)
                producer_bar<PTHREADS>();
                T32P(p_bar += clock64() - tb0;)
            }
            const int k0 = l_kc * KC + ch * 4;
#pragma unroll
            for (int p = 0; p < AP; ++p) {
                const uint32_t tok = t_tok[tb + p * RPP + row_l];
                a[p] = tok != 0xFFFFFFFFu ? __ldg(reinterpret_cast<const float4*>(g.A + static_cast<long long>(tok) * g.lda + k0))
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (++l_kc == nkc) { l_kc = 0; ++l_it; }
        };
        int w_it = 0, w_kc = 0;                        // W-load stream position
        auto load_w = [&](float4 (&w)[WP], int j) {
            if (j >= total) return;
            const int t = static_cast<int>(blockIdx.x) + w_it * static_cast<int>(gridDim.x);
            const int ct = t % col_tiles;
            const float* wsrc = g.Wt + static_cast<long long>(ct * BN + row_l) * g.K + w_kc * KC + ch * 4;
#pragma unroll
            for (int p = 0; p < WP; ++p)
                if (BN % RPP == 0 || p * RPP + row_l < BN) w[p] = __ldg(reinterpret_cast<const float4*>(wsrc + static_cast<long long>(p) * RPP * g.K));
            if (++w_kc == nkc) { w_kc = 0; ++w_it; }
        };
        int c_it = 0, c_kc = 0, c_s = 0;
        uint32_t c_ph = 0;
        auto convert = [&](const float4 (&a)[AP], const float4 (&w)[WP]) {
            T32P(const long long te0 = clock64();)
            tc::mbar_wait(&empty[c_s], c_ph ^ 1u);     // the MMAs that read this stage S k-chunks ago have retired
            T32P(p_empty += clock64() - te0;)
            unsigned char* st = ring + static_cast<size_t>(c_s) * STAGE + sw0;
            const int tb = (c_it & (NTAB - 1)) * BM;
            float4 gam = make_float4(1.f, 1.f, 1.f, 1.f), bet = make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_ln) {
                gam = __ldg(reinterpret_cast<const float4*>(g.ln_w + c_kc * KC + ch * 4));
                bet = __ldg(reinterpret_cast<const float4*>(g.ln_b + c_kc * KC + ch * 4));
            }
            float mu[AP], rs[AP];                      // read before the first store (the compiler cannot move a shared load above one)
#pragma unroll
            for (int p = 0; p < AP; ++p) { mu[p] = t_mu[tb + p * RPP + row_l]; rs[p] = t_rs[tb + p * RPP + row_l]; }
#pragma unroll
            for (int p = 0; p < AP; ++p) {
                float4 v = a[p];
                if (has_ln) {
                    v.x = (v.x - mu[p]) * rs[p] * gam.x + bet.x;
                    v.y = (v.y - mu[p]) * rs[p] * gam.y + bet.y;
                    v.z = (v.z - mu[p]) * rs[p] * gam.z + bet.z;
                    v.w = (v.w - mu[p]) * rs[p] * gam.w + bet.w;
                }
                float4 hi, lo;
                split4(v, hi, lo);
                *reinterpret_cast<float4*>(st + p * (RPP * 128)) = hi;
                *reinterpret_cast<float4*>(st + p * (RPP * 128) + A_TILE) = lo;
            }
#pragma unroll
            for (int p = 0; p < WP; ++p) {
                if (BN % RPP == 0 || p * RPP + row_l < BN) {
                    float4 hi, lo;
                    split4(w[p], hi, lo);
                    *reinterpret_cast<float4*>(st + 2 * A_TILE + p * (RPP * 128)) = hi;
                    *reinterpret_cast<float4*>(st + 2 * A_TILE + p * (RPP * 128) + W_TILE) = lo;
                }
            }
            tc::fence_proxy_async();                   // my generic-proxy smem writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[c_s]);
            if (++c_kc == nkc) { c_kc = 0; ++c_it; }
            if (++c_s == S) { c_s = 0; c_ph ^= 1u; }
        };
#pragma unroll
        for (int u = 0; u < DA; ++u) load_a(abuf[u], u);
        load_w(wbuf[0], 0);
        load_w(wbuf[1], 1);
        for (int j0 = 0; j0 < total; j0 += DA) {
#pragma unroll
            for (int u = 0; u < DA; ++u) {
                const int j = j0 + u;
                if (j < total) {
                    convert(abuf[u], wbuf[u & 1]);
                    load_a(abuf[u], j + DA);
                    load_w(wbuf[u & 1], j + 2);
                }
            }
        }
#ifdef LEWIN_T32_PROF_BUILD
        if (prof && pt == 0) {
            atomicAdd(prof + 0, static_cast<unsigned long long>(clock64() - p_t0));
            atomicAdd(prof + 1, static_cast<unsigned long long>(p_bar));
            atomicAdd(prof + 2, static_cast<unsigned long long>(p_empty));
            atomicAdd(prof + 3, static_cast<unsigned long long>(total));
        }
#endif
    } else if (warp == MMA_WARP) {
        // ============================================================ MMA issuer (one thread)
        if (lane == 0) {
            const uint32_t ring_u = tc::smem_u32(ring);
            int s = 0;
            uint32_t ph = 0;
            T32P(long long m_tempty = 0; long long m_full = 0; const long long m_t0 = clock64();)
            for (int it = 0; it < my_tiles; ++it) {
                const int acc = it & 1;
                const uint32_t aph = static_cast<uint32_t>(it >> 1) & 1u;
                T32P(const long long tm0 = clock64();)
                tc::mbar_wait(&tempty[acc], aph ^ 1u);             // epilogue drained this accumulator
                T32P(m_tempty += clock64() - tm0;)
                tc::tc_fence_after();
                const uint32_t d_addr = tmem_d + static_cast<uint32_t>(acc * ACC);
                for (int kc = 0; kc < nkc; ++kc) {
                    T32P(const long long tf0 = clock64();)
                    tc::mbar_wait(&full[s], ph);
                    T32P(m_full += clock64() - tf0;)
                    tc::tc_fence_after();
                    const uint32_t st_u = ring_u + static_cast<uint32_t>(s) * STAGE;
                    const uint64_t a_hi = tc::make_desc<64>(st_u), a_lo = tc::make_desc<64>(st_u + A_TILE);
                    const uint64_t w_hi = tc::make_desc<64>(st_u + 2 * A_TILE), w_lo = tc::make_desc<64>(st_u + 2 * A_TILE + W_TILE);
#pragma unroll
                    for (int k8 = 0; k8 < KC / 8; ++k8) {          // small terms first
                        mma_tf32_ss(d_addr, a_lo + 2 * k8, w_hi + 2 * k8, IDESC, (kc > 0 || k8 > 0) ? 1u : 0u);
                        mma_tf32_ss(d_addr, a_hi + 2 * k8, w_lo + 2 * k8, IDESC, 1u);
                        mma_tf32_ss(d_addr, a_hi + 2 * k8, w_hi + 2 * k8, IDESC, 1u);
                    }
                    tc::mma_commit(&empty[s]);                     // stage free once these MMAs have read it
                    if (++s == S) { s = 0; ph ^= 1u; }
                }
                tc::mma_commit(&tfull[acc]);                       // accumulator complete
            }
#ifdef LEWIN_T32_PROF_BUILD
            if (prof) {
                atomicAdd(prof + 4, static_cast<unsigned long long>(clock64() - m_t0));
                atomicAdd(prof + 5, static_cast<unsigned long long>(m_tempty));
                atomicAdd(prof + 6, static_cast<unsigned long long>(m_full));
                atomicAdd(prof + 7, static_cast<unsigned long long>(my_tiles));
            }
#endif
        }
    } else {
        // ============================================================ epilogue: thread == TMEM lane == tile row
        const int lg = warp & 3, half = warp >> 2;     // TMEM lane group, column group
        unsigned char* sb = stg + warp * (STG_BUF + RBUF);
        unsigned char* srow = sb + lane * STG_ROW;
        unsigned char* rbuf = sb + STG_BUF;            // [32][BN + 4] residual rows of this warp's 32 tile rows (RS)
        (void)rbuf;
        T32P(long long e_tfull = 0;)
        // output / residual row offsets and DropPath scale of this thread's row of the current tile
        long long oy = -1, orr = -1;
        float sc = 1.f;
        int n0 = 0;
        auto row_info = [&](int it) {
            oy = -1; orr = -1; sc = 1.f;
            if (it >= my_tiles) return;
            const int t = static_cast<int>(blockIdx.x) + it * static_cast<int>(gridDim.x);
            const int rt = t / col_tiles;
            n0 = (t - rt * col_tiles) * BN;
            const uint32_t m = static_cast<uint32_t>(rt) * BM + lg * 32 + lane;
            if (m < g.M) {
                const uint32_t ry = g.mapY ? g.map.token32(m) : m;
                oy = static_cast<long long>(ry) * g.ldy;
                orr = static_cast<long long>(ry) * (g.ldr ? g.ldr : g.ldy);
                if (EPI == EPI_BIAS_RESID && g.drop_scale) sc = g.drop_scale[ry / static_cast<uint32_t>(g.tokens_per_image)];
            }
        };
        // residual rows of the current tile, this warp's column chunks -> rbuf (cp.async; a row's pieces by consecutive lanes)
        auto resid_prefetch = [&]() {
            if constexpr (RS) {
                for (int c = half; c < NCH; c += NCG) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {      // 32 rows x 8 pieces of 16 B
                        const int i = lane + 32 * k, rl = i >> 3, cc = i & 7;
                        const long long o = __shfl_sync(0xffffffffu, orr, rl);
                        if (o >= 0) cp_async16(rbuf + rl * RROW + (c * 32 + cc * 4) * 4, g.R + o + n0 + c * 32 + cc * 4);
                    }
                }
                cp_async_commit();
            }
        };
        row_info(0);
        resid_prefetch();
        for (int it = 0; it < my_tiles; ++it) {
            const int acc = it & 1;
            const uint32_t aph = static_cast<uint32_t>(it >> 1) & 1u;
            // row-cooperative pass over a staged [32 rows x 16 columns] piece: 4 lanes x 16 B per row, 8 rows per instruction
            auto flush16 = [&](float* dst, int colt /* column within the tile */, bool resid) {
                __syncwarp();
                float4 val[4], rv[4];
                long long o[4];
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2, cc = i & 3;
                    o[jj] = __shfl_sync(0xffffffffu, oy, rl);
                    if (resid) {
                        if constexpr (RS) {
                            rv[jj] = *reinterpret_cast<const float4*>(rbuf + rl * RROW + (colt + cc * 4) * 4);
                        } else {
                            const long long orl = __shfl_sync(0xffffffffu, orr, rl);
                            rv[jj] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (o[jj] >= 0) rv[jj] = *reinterpret_cast<const float4*>(g.R + orl + n0 + colt + cc * 4);
                        }
                    }
                    val[jj] = *reinterpret_cast<const float4*>(sb + rl * STG_ROW + cc * 16);
                }
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int i = lane + 32 * jj, rl = i >> 2;
                    if (resid) {
                        const float s = __shfl_sync(0xffffffffu, sc, rl);
                        val[jj].x = rv[jj].x + s * val[jj].x; val[jj].y = rv[jj].y + s * val[jj].y;
                        val[jj].z = rv[jj].z + s * val[jj].z; val[jj].w = rv[jj].w + s * val[jj].w;
                    }
                    if (o[jj] >= 0) *reinterpret_cast<float4*>(dst + o[jj] + n0 + colt + (i & 3) * 4) = val[jj];
                }
                __syncwarp();
            };
            T32P(const long long tw0 = clock64();)
            tc::mbar_wait(&tfull[acc], aph);
            T32P(e_tfull += clock64() - tw0;)
            tc::tc_fence_after();
            if constexpr (RS) { cp_async_wait<0>(); __syncwarp(); }       // this tile's residual rows have landed
            const uint32_t t_addr = tmem_d + (static_cast<uint32_t>(lg * 32) << 16) + static_cast<uint32_t>(acc * ACC);
            for (int c = half; c < NCH; c += NCG) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    float v[16];
                    tmem_ld16(t_addr + c * 32 + hh * 16, v);
                    if (c + NCG >= NCH && hh == 1) {   // last piece of this warp is in registers: hand the accumulator back
                        tc::tc_fence_before();
                        mbar_arrive(&tempty[acc]);
                    }
                    const int colt = c * 32 + hh * 16;
                    if (g.bias) {
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {
                            const float4 b4 = __ldg(reinterpret_cast<const float4*>(g.bias + n0 + colt + j));
                            v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                        }
                    }
                    if (EPI == EPI_BIAS_GELU && g.Y2) {    // training: pre-activation copy
#pragma unroll
                        for (int j = 0; j < 16; j += 4)
                            *reinterpret_cast<float4*>(srow + j * 4) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                        flush16(g.Y2, colt, false);
                    }
                    if (EPI == EPI_BIAS_GELU) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = gelu_fast(v[j]);   // erf by A&S 7.1.26: |err| <= 1.5e-7, i.e. at fp32 rounding level
                    }
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                        *reinterpret_cast<float4*>(srow + j * 4) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                    flush16(g.Y, colt, EPI == EPI_BIAS_RESID);
                }
            }
            if (half >= NCH) {                         // this warp owns no chunk (BN == 32 with two column groups): still hand back
                tc::tc_fence_before();
                mbar_arrive(&tempty[acc]);
            }
            row_info(it + 1);                          // next tile: row offsets, and its residual rows while the MMAs run
            if (it + 1 < my_tiles) resid_prefetch();
        }
#ifdef LEWIN_T32_PROF_BUILD
        if (prof && tid == 0) atomicAdd(prof + 9, static_cast<unsigned long long>(e_tfull));
#endif
    }

#ifdef LEWIN_T32_PROF_BUILD
    if (prof && tid == 0) {
        atomicAdd(prof + 8, static_cast<unsigned long long>(clock64() - cta_t0));
        atomicAdd(prof + 10, 1ull);
    }
#endif
    // ---------------------------------------------------------------- teardown
    tc::tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tc::tmem_dealloc<TMEM_COLS>(tmem_d);
}

template <int BN, int EPI>
cudaError_t launch_bn(const GemmArgs<float>& g, int num_sms, cudaStream_t stream) {
    // linear1 (K = C, N = 4C, GELU) is bound by its epilogue: 8 epilogue warps, shallow A ring (25 warps -> 72 registers);
    // the others by the producers: 4 epilogue warps, deeper A ring where the registers allow (21 warps -> 80 registers)
    constexpr int NEW = EPI == EPI_BIAS_GELU ? 8 : 4, NPW = 16;
    constexpr int DA = (EPI != EPI_BIAS_GELU && BN <= 64) ? 4 : 2;
    constexpr size_t STAGE = stage_bytes<BN>();
    constexpr size_t fixed = fixed_smem<BN, EPI, NEW>();
    static_assert(fixed + 2 * STAGE <= SMEM_MAX, "two stages must fit");
    int S = static_cast<int>((SMEM_MAX - fixed) / STAGE);
    if (S > 8) S = 8;
    const size_t smem = fixed + static_cast<size_t>(S) * STAGE;
    auto k = gemm_t32_kernel<BN, EPI, NEW, NPW, DA>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    const int row_tiles = static_cast<int>((g.M + BM - 1) / BM);
    const int col_tiles = g.N / BN;
    int grid = num_sms;
    if (grid > row_tiles * col_tiles) grid = row_tiles * col_tiles;
    k<<<grid, (NEW + 1 + NPW) * 32, smem, stream>>>(g, row_tiles, col_tiles, g.K / KC, S, prof_slot());
    return cudaGetLastError();
}

// forward-pass shapes of the LeWin block: K, N multiples of 32, 16-byte aligned rows, no backward-only prologues
template <int EPI>
inline bool supported(const GemmArgs<float>& g) {
    if (g.a_row_scale || g.aux || g.up2) return false;
    if (EPI != EPI_BIAS && EPI != EPI_BIAS_GELU && EPI != EPI_BIAS_RESID) return false;
    if (EPI == EPI_BIAS_RESID && !g.R) return false;
    if (g.K % 32 || g.N % 32 || g.M <= 0 || g.M >= (1ll << 31)) return false;
    if ((g.lda % 4) || (g.ldy % 4) || (g.ldr % 4)) return false;
    if (g.mean && (!g.rstd || !g.ln_w || !g.ln_b)) return false;
    return true;
}

template <int EPI>
cudaError_t launch(const GemmArgs<float>& g, int num_sms, cudaStream_t stream) {
    // tensor-bound shapes (long K): 256-wide tiles halve the A traffic per FLOP; two 96 KB stages
    if (g.N % 256 == 0 && g.K >= 128 && (g.M + BM - 1) / BM * (g.N / 256) >= num_sms) return launch_bn<256, EPI>(g, num_sms, stream);
    if (g.N % 128 == 0) return launch_bn<128, EPI>(g, num_sms, stream);
    if (g.N % 96 == 0) return launch_bn<96, EPI>(g, num_sms, stream);
    if (g.N % 64 == 0) return launch_bn<64, EPI>(g, num_sms, stream);
    return launch_bn<32, EPI>(g, num_sms, stream);
}

}  // namespace t32
}  // namespace lewin
