// C-ABI of the sm_100a LeWin hot path (see include/lewin_b200.h for the contract).
#include "../../include/lewin_b200.h"

#include "common.cuh"
#include "dwconv.cuh"
#include "dwconv_stream.cuh"
#include "gemm_fused.cuh"
#include "gemm_tc.cuh"
#include "gemm_ws.cuh"
#include "probsparse_core.cuh"
#include "probsparse_core_v3.cuh"
#include "backward.cuh"
#include "attn_fused_api.h"
#include "leff_tail_api.h"

#include <atomic>

using namespace lewin;

namespace {

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct DeviceInfo { int sms; int cc_major; };

inline int device_info(DeviceInfo* d) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return static_cast<int>(e);
    e = cudaDeviceGetAttribute(&d->sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return static_cast<int>(e);
    e = cudaDeviceGetAttribute(&d->cc_major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return static_cast<int>(e);
    return d->cc_major == 10 ? 0 : LEWIN_E_ARCH;
}

std::atomic<long long> g_launches{0};   // diagnostic only (lewin_launch_count)

constexpr int kAsyncMinC = 128;   // channels above which the bf16 GEMMs take the streamed-W kernels on pre-converted weights

// Which kernels a forward call will run (shared by the launch code and the kernel-mask queries).
inline bool ws_level(int C, long long tokens) {     // warp-specialised persistent GEMM (gemm_ws.cuh) serves this level
    return (C == 32 || C == 64 || C == 128) && tokens >= 4 * TC_BM;
}
struct AttnPlan { bool fused, async_gemm, ws_gemm, ln_stats; };
inline AttnPlan plan_attn(const LewinAttnFwdArgs* a, bool bf) {
    AttnPlan p{};
    const long long tokens = static_cast<long long>(a->B) * a->H * a->W;
    p.fused = bf && attn_fused_supported(a);            // the whole half as one kernel (attn_fused.cuh): inference, C <= 64
    if (p.fused) return p;
    p.ws_gemm = bf && !a->windowed && ws_level(a->C, tokens);
    p.async_gemm = bf && !p.ws_gemm && a->C > kAsyncMinC && a->C % 64 == 0;
    p.ln_stats = !a->windowed && !p.async_gemm && !p.ws_gemm;
    return p;
}

// Optional per-kernel timing with caller-owned events (LewinAttnFwdArgs::timing).
struct KTimer {
    lewin_event_t* ev;
    cudaStream_t st;
    void begin(int k) const { if (ev) cudaEventRecord(reinterpret_cast<cudaEvent_t>(ev[2 * k]), st); }
    void end(int k) const {
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (ev) cudaEventRecord(reinterpret_cast<cudaEvent_t>(ev[2 * k + 1]), st);
    }
};

#define CK(expr)                                         \
    do {                                                 \
        cudaError_t _e = (expr);                         \
        if (_e != cudaSuccess) return static_cast<int>(_e); \
    } while (0)

// One linear of a forward call on the kernel its plan chose.  ws_gemm: the warp-specialised GEMM with resident weights,
// which computes the LayerNorm statistics itself when the linear has a LayerNorm prologue (g.mean set).  Wb: the streamed-W
// GEMM on that pre-converted bf16 weight (gemm_tca where wss_supported rules the shape out).  Otherwise the generic dispatch.
template <int EPI, typename T>
cudaError_t launch_linear(GemmArgs<T> g, bool ws_gemm, const __nv_bfloat16* Wb, int sms, cudaStream_t st) {
    if constexpr (Act<T>::kIsBf16) {
        if (ws_gemm) {
            const bool ln = g.mean != nullptr;
            g.mean = nullptr; g.rstd = nullptr;
            return ws::launch<EPI>(g, ln, sms, st);
        }
        if (Wb) return ws::wss_supported(g) ? ws::wss_launch<EPI>(g, Wb, sms, st) : launch_gemm_tca<EPI>(g, Wb, st);
    }
    return launch_gemm_any<T, EPI>(g, st);
}

// ------------------------------------------------------------------ attention forward
int check_attn(const LewinAttnFwdArgs* a) {
    if (!a) return LEWIN_E_NULL;
    if (!a->x || !a->y || !a->w_qkv || !a->b_qkv || !a->w_out || !a->b_out || !a->index_sample || !a->qkv || !a->ctx)
        return LEWIN_E_NULL;
    if (!a->windowed && (!a->ln_w || !a->ln_b)) return LEWIN_E_NULL;
    if (a->use_rpb && !a->rpb_table && !a->rpb_dense) return LEWIN_E_NULL;
    if (a->B <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->nH <= 0) return LEWIN_E_SHAPE;
    if (a->H % 8 || a->W % 8 || a->C % 32 || !head_dim_ok(a->C, a->nH)) return LEWIN_E_SHAPE;
    if (a->C > 1024) return LEWIN_E_SHAPE;        // the LayerNorm pre-passes handle rows of up to 1024 channels (embed_dim 64's bottleneck)
    if (a->shift < 0 || a->shift >= 8) return LEWIN_E_SHAPE;
    if (a->shift > 0 && ((a->H <= 8 && !a->band_mode) || a->W <= 8)) return LEWIN_E_SHAPE;   // My_model_1.py:764-766 forces shift 0
    if (a->band_mode && (a->windowed || a->save_for_backward || a->band_y0 < 0 || a->band_Hg < a->H || a->band_y0 % 8 || a->band_Hg % 8))
        return LEWIN_E_SHAPE;
    if (a->windowed && (a->shift != 0 || a->analytic_shift_mask)) return LEWIN_E_SHAPE;
    if (a->mask && a->nW_mask <= 0) return LEWIN_E_SHAPE;
    if (a->mask && ((a->B * (a->H / 8) * (a->W / 8)) % a->nW_mask)) return LEWIN_E_SHAPE;
    const void* ps[] = {a->x, a->y, a->ln_w, a->ln_b, a->w_qkv, a->b_qkv, a->w_out, a->b_out, a->qkv, a->ctx, a->mask,
                        a->w_qkv_bf16, a->w_out_bf16};
    for (const void* p : ps)
        if (p && !aligned16(p)) return LEWIN_E_ALIGN;
    return 0;
}

size_t attn_fwd_ws(const LewinAttnFwdArgs* a) {
    const size_t tokens = static_cast<size_t>(a->B) * a->H * a->W;
    // + bf16 staging for the async tcgen05 GEMMs (C > 128): LN-applied window-ordered x, bf16 copies of W_qkv / W_out
    const size_t C = a->C;
    return 2 * align_up(tokens * sizeof(float), 256) +
           (C >= 64 ? align_up(tokens * C * 2, 256) + align_up(4 * C * C * 2, 256) : 0);
}

template <typename T>
int attn_fwd(const LewinAttnFwdArgs* a, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (int rc = check_attn(a)) return rc;
    DeviceInfo di;
    if (int rc = device_info(&di)) return rc;
    if (!ws || ws_bytes < attn_fwd_ws(a)) return LEWIN_E_WORKSPACE;
    if (!aligned16(ws)) return LEWIN_E_ALIGN;

    const long long tokens = static_cast<long long>(a->B) * a->H * a->W;
    const int nWin = (a->H / 8) * (a->W / 8);
    const int B_ = a->B * nWin;
    const int C = a->C;
    unsigned char* wsp = static_cast<unsigned char*>(ws);
    float* mean = reinterpret_cast<float*>(wsp);
    float* rstd = reinterpret_cast<float*>(wsp + align_up(tokens * sizeof(float), 256));
    unsigned char* ws_gemm = wsp + 2 * align_up(tokens * sizeof(float), 256);      // bf16 staging of the streamed-W GEMMs

    WinMap map{a->H, a->W, a->W / 8, nWin, a->shift, a->band_mode ? 0 : a->shift};
    const T* x = static_cast<const T*>(a->x);

    const KTimer kt{a->timing, stream};
    const AttnPlan plan = plan_attn(a, Act<T>::kIsBf16);
    if (plan.fused) {                                   // LN1 -> q|k|v MMA -> ProbSparse core -> out MMA -> residual, one launch
        kt.begin(LEWIN_ATTN_K_FUSED);
        if (int rc = attn_fused_launch(a, di.sms, stream)) return rc;
        kt.end(LEWIN_ATTN_K_FUSED);
        return 0;
    }
    if (plan.ln_stats) {
        kt.begin(LEWIN_ATTN_K_LNSTATS);
        CK(launch_ln_stats<T>(x, tokens, C, mean, rstd, stream));
        kt.end(LEWIN_ATTN_K_LNSTATS);
    }
    __nv_bfloat16* xhat = nullptr; __nv_bfloat16* wqkv_b = nullptr; __nv_bfloat16* wout_b = nullptr;
    if constexpr (Act<T>::kIsBf16) {
        if (plan.async_gemm) {
            unsigned char* q = ws_gemm;
            xhat = reinterpret_cast<__nv_bfloat16*>(q); q += align_up(static_cast<size_t>(tokens) * C * 2, 256);
            wqkv_b = reinterpret_cast<__nv_bfloat16*>(q);
            wout_b = wqkv_b + static_cast<size_t>(3) * C * C;
            if (a->w_qkv_bf16 && a->w_out_bf16) {        // caller-converted constants (inference): no per-call conversion
                wqkv_b = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(a->w_qkv_bf16));
                wout_b = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(a->w_out_bf16));
            } else {
                CK(launch_convert_w(a->w_qkv, wqkv_b, static_cast<long long>(3) * C * C, stream));
                CK(launch_convert_w(a->w_out, wout_b, static_cast<long long>(C) * C, stream));
            }
        }
    }
    {   // q | k | v projections (attn.py:420-422) with LN1 + roll + window_partition as the A prologue
        GemmArgs<T> g{};
        g.A = x; g.lda = C;
        g.Wt = a->w_qkv; g.bias = a->b_qkv;
        g.Y = static_cast<T*>(a->qkv); g.Y2 = nullptr; g.ldy = 3 * C;
        g.M = tokens; g.N = 3 * C; g.K = C;
        if (!a->windowed) { g.mean = mean; g.rstd = rstd; g.ln_w = a->ln_w; g.ln_b = a->ln_b; }
        g.mapA = a->windowed ? 0 : 1; g.mapY = 0; g.map = map;
        g.tokens_per_image = a->H * a->W;
        kt.begin(LEWIN_ATTN_K_QKV);
        if constexpr (Act<T>::kIsBf16) {
            if (plan.async_gemm && !a->windowed) {      // LN1 + roll + partition in one pre-pass; the GEMM then streams plain bf16 rows
                CK(launch_ln_apply(static_cast<const __nv_bfloat16*>(a->x), xhat, a->ln_w, a->ln_b, tokens, C, 1, map, stream));
                g.A = xhat; g.mapA = 0; g.mean = nullptr; g.rstd = nullptr;
            }
        }
        CK(launch_linear<EPI_BIAS>(g, plan.ws_gemm, wqkv_b, di.sms, stream));
        kt.end(LEWIN_ATTN_K_QKV);
    }
    {   // ProbSparse core (attn.py:287-342)
        CoreFwdArgs<T> c{};
        c.qkv = static_cast<const T*>(a->qkv);
        c.ctx = static_cast<T*>(a->ctx);
        c.top = a->top;
        c.rpb_table = a->rpb_table;
        c.rpb_dense = a->rpb_table ? nullptr : a->rpb_dense;
        c.index_sample = a->index_sample;
        c.mask = a->mask; c.nW_mask = a->mask ? a->nW_mask : 1;
        c.B_ = B_; c.nH = a->nH; c.C = C;
        c.use_rpb = a->use_rpb;
        c.shift = (a->analytic_shift_mask && !a->windowed) ? a->shift : 0;
        c.H = a->H; c.W = a->W; c.nWw = a->W / 8; c.nWin = nWin;
        c.y0 = a->band_mode ? a->band_y0 : 0; c.Hg = a->band_mode ? a->band_Hg : a->H;
        kt.begin(LEWIN_ATTN_K_CORE);
        CK(launch_core_fwd<T>(c, di.sms, stream));
        kt.end(LEWIN_ATTN_K_CORE);
    }
    {   // out projection (attn.py:456) + window_reverse + un-roll + DropPath scale + residual
        GemmArgs<T> g{};
        g.A = static_cast<const T*>(a->ctx); g.lda = C;
        g.Wt = a->w_out; g.bias = a->b_out;
        g.Y = static_cast<T*>(a->y); g.ldy = C;
        g.M = tokens; g.N = C; g.K = C;
        g.mapA = 0; g.mapY = a->windowed ? 0 : 1; g.map = map;
        g.tokens_per_image = a->H * a->W;
        kt.begin(LEWIN_ATTN_K_OUT);
        if (a->windowed) {
            CK(launch_linear<EPI_BIAS>(g, plan.ws_gemm, wout_b, di.sms, stream));
        } else {
            g.R = x; g.drop_scale = a->drop_scale;
            CK(launch_linear<EPI_BIAS_RESID>(g, plan.ws_gemm, wout_b, di.sms, stream));
        }
        kt.end(LEWIN_ATTN_K_OUT);
    }
    return 0;
}

inline int core_head_dim(const LewinCoreFwdArgs* a) { return a->head_dim > 0 ? a->head_dim : kHeadDim; }

int check_core(const LewinCoreFwdArgs* a) {
    if (!a || !a->qkv || !a->ctx) return LEWIN_E_NULL;
    if (a->use_rpb && !a->rpb_table && !a->rpb_dense) return LEWIN_E_NULL;
    const int D = core_head_dim(a);
    if (a->B_ <= 0 || a->nH <= 0 || !(D == 32 || D == 64 || D == 128)) return LEWIN_E_SHAPE;
    if (a->mask && (a->nW_mask <= 0 || a->B_ % a->nW_mask)) return LEWIN_E_SHAPE;
    if (!aligned16(a->qkv) || !aligned16(a->ctx) || (a->mask && !aligned16(a->mask))) return LEWIN_E_ALIGN;
    return 0;
}

template <typename T>
int core_only_fwd(const LewinCoreFwdArgs* a, void*, size_t, cudaStream_t stream) {
    if (int rc = check_core(a)) return rc;
    if (!a->index_sample) return LEWIN_E_NULL;
    DeviceInfo di;
    if (int rc = device_info(&di)) return rc;
    const int D = core_head_dim(a);
    CoreFwdArgs<T> c{};
    c.qkv = static_cast<const T*>(a->qkv);
    c.ctx = static_cast<T*>(a->ctx);
    c.top = a->top;
    c.rpb_table = a->rpb_table;
    c.rpb_dense = a->rpb_table ? nullptr : a->rpb_dense;
    c.index_sample = a->index_sample;
    c.mask = a->mask; c.nW_mask = a->mask ? a->nW_mask : 1;
    c.B_ = a->B_; c.nH = a->nH; c.C = a->nH * D;
    c.use_rpb = a->use_rpb;
    c.shift = 0; c.H = 8; c.W = 8; c.nWw = 1; c.nWin = 1; c.y0 = 0; c.Hg = 8;
    CK(launch_core_fwd<T>(c, di.sms, stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// autograd of ProbAttention.forward for the saved selection: dq | dk | dv, d(bias)
template <typename T>
int core_only_bwd(const LewinCoreBwdArgs* a, void*, size_t, cudaStream_t stream) {
    if (!a) return LEWIN_E_NULL;
    const LewinCoreFwdArgs* f = &a->fwd;
    if (int rc = check_core(f)) return rc;
    if (!f->top || !a->dctx || !a->dqkv) return LEWIN_E_NULL;
    if (f->nH > 16) return LEWIN_E_SHAPE;
    if (!aligned16(a->dctx) || !aligned16(a->dqkv)) return LEWIN_E_ALIGN;
    int sms = 0;
    if (int rc = bw_device(&sms)) return rc;
    const int D = core_head_dim(f);
    CoreBwdArgs<T> c{};
    c.qkv = static_cast<const T*>(f->qkv); c.dctx = static_cast<const T*>(a->dctx); c.dqkv = static_cast<T*>(a->dqkv);
    c.top = f->top;
    c.rpb_table = f->rpb_table; c.rpb_dense = f->rpb_table ? nullptr : f->rpb_dense;
    c.d_rpb_table = a->d_rpb_table; c.d_rpb_dense = f->rpb_table ? nullptr : a->d_rpb_dense;
    c.mask = f->mask; c.nW_mask = f->mask ? f->nW_mask : 1;
    c.B_ = f->B_; c.nH = f->nH; c.C = f->nH * D; c.use_rpb = f->use_rpb;
    c.shift = 0; c.H = 8; c.W = 8; c.nWw = 1; c.nWin = 1;
    CK(launch_core_bwd<T>(c, sms, stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// ------------------------------------------------------------------ LeFF forward
int check_leff(const LewinLeffFwdArgs* a) {
    if (!a) return LEWIN_E_NULL;
    if (!a->y || !a->out || !a->w1 || !a->b1 || !a->w_dw || !a->b_dw || !a->w2 || !a->b2 || !a->h1 || !a->h2)
        return LEWIN_E_NULL;
    if (a->fused && (!a->ln_w || !a->ln_b)) return LEWIN_E_NULL;
    if (a->save_for_backward && (!a->a1 || !a->a2)) return LEWIN_E_NULL;
    if (a->B <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->hidden <= 0) return LEWIN_E_SHAPE;
    if (a->C % 32 || a->hidden % 32) return LEWIN_E_SHAPE;
    if (a->C > 1024) return LEWIN_E_SHAPE;        // as in check_attn
    if (a->ld_out != 0 && (a->ld_out < a->C || a->ld_out % 8)) return LEWIN_E_SHAPE;
    const void* ps[] = {a->y, a->out, a->ln_w, a->ln_b, a->w1, a->b1, a->w_dw, a->b_dw, a->w2, a->b2, a->h1, a->h2, a->a1, a->a2,
                        a->w1_bf16, a->w2_bf16};
    for (const void* p : ps)
        if (p && !aligned16(p)) return LEWIN_E_ALIGN;
    return 0;
}

size_t leff_fwd_ws(const LewinLeffFwdArgs* a) {
    const size_t tokens = static_cast<size_t>(a->B) * a->H * a->W;
    const size_t C = a->C, Ch = a->hidden;
    return 2 * align_up(tokens * sizeof(float), 256) +
           (C >= 64 ? align_up(tokens * C * 2, 256) + align_up(2 * C * Ch * 2, 256) : 0);
}

// bf16 LeFF: three kernels (linear1 + GELU, depthwise 3x3 + GELU, linear2 + residual); h1 / h2 round-trip HBM once each.
// (A single on-chip kernel was built and measured 2-3x slower in round 1 - halo recompute of linear1 and per-tile staging
// cost more instructions than the 8 bytes per hidden element of HBM traffic they save - and has been removed.)
struct LeffPlan { bool ws_gemm, async_gemm, ln_stats, tail; };
inline LeffPlan plan_leff(const LewinLeffFwdArgs* a, bool bf) {
    LeffPlan p{};
    const long long tokens = static_cast<long long>(a->B) * a->H * a->W;
    p.ws_gemm = bf && a->fused && a->hidden == 4 * a->C && ws_level(a->C, tokens);
    p.async_gemm = bf && !p.ws_gemm && a->C > kAsyncMinC && a->C % 64 == 0 && a->hidden % 64 == 0;
    p.ln_stats = a->fused && !p.async_gemm && !p.ws_gemm;
    p.tail = bf && p.ws_gemm && leff_tail_supported(a);      // dwconv + GELU + linear2 + residual in one kernel (leff_tail.cuh)
    return p;
}

// `out` with a row stride > C: the fused tail and the warp-specialised / streamed-W linear2 epilogues address the output and
// the residual rows separately; the first-generation kernels do not
inline bool leff_ld_out_ok(const LewinLeffFwdArgs* a, const LeffPlan& p) {
    if (a->ld_out == 0 || a->ld_out == a->C) return true;
    if (!a->fused || a->save_for_backward) return false;
    if (p.tail || p.ws_gemm) return true;
    if (!p.async_gemm) return false;
    GemmArgs<__nv_bfloat16> g{};                 // the linear2 GEMM as leff_fwd builds it
    g.lda = a->hidden; g.M = static_cast<long long>(a->B) * a->H * a->W; g.N = a->C; g.K = a->hidden;
    return ws::wss_supported(g);
}

template <typename T>
int leff_fwd(const LewinLeffFwdArgs* a, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (int rc = check_leff(a)) return rc;
    DeviceInfo di;
    if (int rc = device_info(&di)) return rc;
    if (!ws || ws_bytes < leff_fwd_ws(a)) return LEWIN_E_WORKSPACE;
    if (!aligned16(ws)) return LEWIN_E_ALIGN;
    const long long tokens = static_cast<long long>(a->B) * a->H * a->W;
    const int C = a->C, Ch = a->hidden;
    unsigned char* wsp = static_cast<unsigned char*>(ws);
    float* mean = reinterpret_cast<float*>(wsp);
    float* rstd = reinterpret_cast<float*>(wsp + align_up(tokens * sizeof(float), 256));
    const T* y = static_cast<const T*>(a->y);
    const bool save = a->save_for_backward != 0;

    const KTimer kt{a->timing, stream};
    const LeffPlan plan = plan_leff(a, Act<T>::kIsBf16);
    if (!leff_ld_out_ok(a, plan)) return LEWIN_E_SHAPE;
    const long long ldo = a->ld_out > 0 ? a->ld_out : a->C;
    if constexpr (Act<T>::kIsBf16) CK(launch_gelu_tab_init(stream));     // idempotent 8 KB table (common.cuh)
    __nv_bfloat16* xhat = nullptr; __nv_bfloat16* w1b = nullptr; __nv_bfloat16* w2b = nullptr;
    if constexpr (Act<T>::kIsBf16) {
        if (plan.async_gemm) {
            unsigned char* q = wsp + 2 * align_up(tokens * sizeof(float), 256);
            xhat = reinterpret_cast<__nv_bfloat16*>(q); q += align_up(static_cast<size_t>(tokens) * C * 2, 256);
            w1b = reinterpret_cast<__nv_bfloat16*>(q);
            w2b = w1b + static_cast<size_t>(C) * Ch;
            if (a->w1_bf16 && a->w2_bf16) {
                w1b = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(a->w1_bf16));
                w2b = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(a->w2_bf16));
            } else {
                CK(launch_convert_w(a->w1, w1b, static_cast<long long>(C) * Ch, stream));
                CK(launch_convert_w(a->w2, w2b, static_cast<long long>(C) * Ch, stream));
            }
        }
    }
    if (plan.ln_stats) {
        kt.begin(LEWIN_LEFF_K_LNSTATS);
        CK(launch_ln_stats<T>(y, tokens, C, mean, rstd, stream));
        kt.end(LEWIN_LEFF_K_LNSTATS);
    }
    {   // linear1 + GELU (My_model_1.py:508) with LN2 as the A prologue
        GemmArgs<T> g{};
        g.A = y; g.lda = C;
        g.Wt = a->w1; g.bias = a->b1;
        g.Y = static_cast<T*>(a->h1); g.Y2 = save ? static_cast<T*>(a->a1) : nullptr; g.ldy = Ch;
        g.M = tokens; g.N = Ch; g.K = C;
        if (a->fused) { g.mean = mean; g.rstd = rstd; g.ln_w = a->ln_w; g.ln_b = a->ln_b; }
        g.tokens_per_image = a->H * a->W;
        kt.begin(LEWIN_LEFF_K_FC1);
        if constexpr (Act<T>::kIsBf16) {
            if (plan.async_gemm && a->fused) {          // LN2 in one pre-pass; the GEMM then streams plain bf16 rows
                WinMap nomap{a->H, a->W, a->W / 8, (a->H / 8) * (a->W / 8), 0, 0};
                CK(launch_ln_apply(static_cast<const __nv_bfloat16*>(a->y), xhat, a->ln_w, a->ln_b, tokens, C, 0, nomap, stream));
                g.A = xhat; g.mean = nullptr; g.rstd = nullptr;
            }
        }
        CK(launch_linear<EPI_BIAS_GELU>(g, plan.ws_gemm, w1b, di.sms, stream));
        kt.end(LEWIN_LEFF_K_FC1);
    }
    if (plan.tail) {
        const uint16_t* tab2 = nullptr;
        if constexpr (Act<T>::kIsBf16) CK(cudaGetSymbolAddress(reinterpret_cast<void**>(const_cast<uint16_t**>(&tab2)), g_gelu_tab2));
        kt.begin(LEWIN_LEFF_K_TAIL);
        if (int rc = leff_tail_launch(a, tab2, di.sms, stream)) return rc;
        kt.end(LEWIN_LEFF_K_TAIL);
        return 0;
    }
    kt.begin(LEWIN_LEFF_K_DWCONV);
    if (Act<T>::kIsBf16 && dws::supported(a->H, a->W, Ch))      // persistent double-buffered kernel (dwconv_stream.cuh)
        CK(dws::launch(static_cast<const __nv_bfloat16*>(a->h1), static_cast<__nv_bfloat16*>(a->h2),
                       save ? static_cast<__nv_bfloat16*>(a->a2) : nullptr, a->w_dw, a->b_dw, a->B, a->H, a->W, Ch, di.sms, stream));
    else
        CK(launch_dwconv_gelu_auto<T>(static_cast<const T*>(a->h1), static_cast<T*>(a->h2), save ? static_cast<T*>(a->a2) : nullptr,
                                      a->w_dw, a->b_dw, a->B, a->H, a->W, Ch, stream));
    kt.end(LEWIN_LEFF_K_DWCONV);
    {   // linear2 (My_model_1.py:529) + DropPath scale + residual (My_model_1.py:873)
        GemmArgs<T> g{};
        g.A = static_cast<const T*>(a->h2); g.lda = Ch;
        g.Wt = a->w2; g.bias = a->b2;
        g.Y = static_cast<T*>(a->out); g.ldy = ldo; g.ldr = C;
        g.M = tokens; g.N = C; g.K = Ch;
        g.tokens_per_image = a->H * a->W;
        kt.begin(LEWIN_LEFF_K_FC2);
        if (a->fused) {
            g.R = y; g.drop_scale = a->drop_scale;
            CK(launch_linear<EPI_BIAS_RESID>(g, plan.ws_gemm, w2b, di.sms, stream));
        } else {
            CK(launch_linear<EPI_BIAS>(g, plan.ws_gemm, w2b, di.sms, stream));
        }
        kt.end(LEWIN_LEFF_K_FC2);
    }
    return 0;
}

// ------------------------------------------------------------------ Upsample (SURVEY 8(f) rank 2)
// Wb[(2*di + dj) * Cout + co][ci] = bf16(w[ci][co][di][dj]);  bias4[q * Cout + co] = bias[co]
__global__ void upsample_prep_kernel(const float* __restrict__ w, const float* __restrict__ bias, __nv_bfloat16* __restrict__ wb,
                                     float* __restrict__ bias4, int Cin, int Cout) {
    const int n = blockIdx.x;                       // output column (q, co)
    const int q = n / Cout, co = n - q * Cout;
    for (int ci = threadIdx.x; ci < Cin; ci += blockDim.x)
        wb[static_cast<long long>(n) * Cin + ci] = __float2bfloat16_rn(w[(static_cast<long long>(ci) * Cout + co) * 4 + q]);
    if (threadIdx.x == 0) bias4[n] = bias[co];
}

size_t upsample_ws(const LewinUpsampleFwdArgs* a) {
    return align_up(static_cast<size_t>(4) * a->Cout * a->Cin * 2, 256) + align_up(static_cast<size_t>(4) * a->Cout * 4, 256);
}

int upsample_fwd_bf16(const LewinUpsampleFwdArgs* a, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (!a || !a->x || !a->weight || !a->bias || !a->out) return LEWIN_E_NULL;
    if (a->B <= 0 || a->H <= 0 || a->W <= 0 || a->Cin % 64 || a->Cout % 32 || a->Cout <= 0 || a->ld_out < a->Cout || a->ld_out % 8)
        return LEWIN_E_SHAPE;
    if (!aligned16(a->x) || !aligned16(a->out)) return LEWIN_E_ALIGN;
    DeviceInfo di;
    if (int rc = device_info(&di)) return rc;
    if (!ws || ws_bytes < upsample_ws(a)) return LEWIN_E_WORKSPACE;
    if (!aligned16(ws)) return LEWIN_E_ALIGN;
    __nv_bfloat16* wb = static_cast<__nv_bfloat16*>(ws);
    float* bias4 = reinterpret_cast<float*>(static_cast<unsigned char*>(ws) + align_up(static_cast<size_t>(4) * a->Cout * a->Cin * 2, 256));
    upsample_prep_kernel<<<4 * a->Cout, 128, 0, stream>>>(a->weight, a->bias, wb, bias4, a->Cin, a->Cout);
    CK(cudaGetLastError());
    GemmArgs<__nv_bfloat16> g{};
    g.A = static_cast<const __nv_bfloat16*>(a->x); g.lda = a->Cin;
    g.Wt = nullptr; g.bias = bias4;
    g.Y = static_cast<__nv_bfloat16*>(a->out); g.ldy = a->ld_out;
    g.M = static_cast<long long>(a->B) * a->H * a->W; g.N = 4 * a->Cout; g.K = a->Cin;
    g.tokens_per_image = a->H * a->W;
    g.up2 = 1; g.up_H = a->H; g.up_W = a->W; g.up_C = a->Cout;
    if (!ws::wss_supported(g)) return LEWIN_E_SHAPE;       // M >= 512, Cin % 64, 4*Cout % 128 (no fallback kernel for this op)
    CK((ws::wss_launch<EPI_BIAS>(g, wb, di.sms, stream)));
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return 0;
}

// ------------------------------------------------------------------ InputProj (SURVEY 8(f) rank 2)
// thread == pixel, COUT accumulators; weights (bf16-rounded) broadcast from shared memory; one 2 x COUT-byte row store
template <int COUT>
__global__ void __launch_bounds__(128) input_proj_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                                         __nv_bfloat16* __restrict__ out, int B, int H, int W, int Cin, float slope) {
    __shared__ __align__(16) float ws[4 * 9 * COUT];
    __shared__ float bs[COUT];
    for (int i = threadIdx.x; i < Cin * 9 * COUT; i += 128) {     // ws[(ci * 9 + tap) * COUT + co]
        const int co = i % COUT, t = i / COUT;
        ws[i] = Act<__nv_bfloat16>::round(w[co * Cin * 9 + t]);
    }
    for (int i = threadIdx.x; i < COUT; i += 128) bs[i] = Act<__nv_bfloat16>::round(bias[i]);
    __syncthreads();
    const long long p = static_cast<long long>(blockIdx.x) * 128 + threadIdx.x;
    const long long total = static_cast<long long>(B) * H * W;
    if (p >= total) return;
    const int xx = static_cast<int>(p % W);
    const int yy = static_cast<int>((p / W) % H);
    const long long b = p / (static_cast<long long>(W) * H);
    float acc[COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) acc[c] = 0.f;
    for (int ci = 0; ci < Cin; ++ci) {
        const float* plane = x + (b * Cin + ci) * static_cast<long long>(H) * W;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int y2 = yy + ky - 1, x2 = xx + kx - 1;
                float v = 0.f;
                if (y2 >= 0 && y2 < H && x2 >= 0 && x2 < W) v = Act<__nv_bfloat16>::round(plane[static_cast<long long>(y2) * W + x2]);
                const float4* wr = reinterpret_cast<const float4*>(ws + (ci * 9 + ky * 3 + kx) * COUT);
#pragma unroll
                for (int c4 = 0; c4 < COUT / 4; ++c4) {
                    const float4 w4 = wr[c4];
                    acc[4 * c4] = fmaf(v, w4.x, acc[4 * c4]); acc[4 * c4 + 1] = fmaf(v, w4.y, acc[4 * c4 + 1]);
                    acc[4 * c4 + 2] = fmaf(v, w4.z, acc[4 * c4 + 2]); acc[4 * c4 + 3] = fmaf(v, w4.w, acc[4 * c4 + 3]);
                }
            }
    }
    uint4* orow = reinterpret_cast<uint4*>(out + p * COUT);
#pragma unroll
    for (int c8 = 0; c8 < COUT / 8; ++c8) {
        uint32_t pk[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            float v2[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = c8 * 8 + 2 * h + e;
                float t = Act<__nv_bfloat16>::round(Act<__nv_bfloat16>::round(acc[c]) + bs[c]);      // conv -> bf16, + bias -> bf16
                v2[e] = t >= 0.f ? t : t * slope;                                                      // LeakyReLU -> bf16 (by the pack)
            }
            __nv_bfloat162 hh = __floats2bfloat162_rn(v2[0], v2[1]);
            pk[h] = *reinterpret_cast<uint32_t*>(&hh);
        }
        orow[c8] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

int input_proj_fwd_bf16(const LewinInputProjArgs* a, cudaStream_t stream) {
    if (!a || !a->x || !a->weight || !a->bias || !a->out) return LEWIN_E_NULL;
    if (a->B <= 0 || a->H <= 0 || a->W <= 0 || a->Cin <= 0 || a->Cin > 4 || (a->Cout != 32 && a->Cout != 64)) return LEWIN_E_SHAPE;
    if (!aligned16(a->out)) return LEWIN_E_ALIGN;
    DeviceInfo di;
    if (int rc = device_info(&di)) return rc;
    const long long total = static_cast<long long>(a->B) * a->H * a->W;
    const unsigned grid = static_cast<unsigned>((total + 127) / 128);
    __nv_bfloat16* out = static_cast<__nv_bfloat16*>(a->out);
    if (a->Cout == 32) input_proj_kernel<32><<<grid, 128, 0, stream>>>(a->x, a->weight, a->bias, out, a->B, a->H, a->W, a->Cin, a->negative_slope);
    else input_proj_kernel<64><<<grid, 128, 0, stream>>>(a->x, a->weight, a->bias, out, a->B, a->H, a->W, a->Cin, a->negative_slope);
    CK(cudaGetLastError());
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

}  // namespace

extern "C" {

int lewin_attn_fwd_f32(const LewinAttnFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return attn_fwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_attn_fwd_bf16(const LewinAttnFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return attn_fwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_probsparse_core_fwd_f32(const LewinCoreFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return core_only_fwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_probsparse_core_fwd_bf16(const LewinCoreFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return core_only_fwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
size_t lewin_probsparse_core_fwd_workspace_bytes(const LewinCoreFwdArgs*, int) { return 0; }
int lewin_probsparse_core_bwd_f32(const LewinCoreBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return core_only_bwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_probsparse_core_bwd_bf16(const LewinCoreBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return core_only_bwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
size_t lewin_probsparse_core_bwd_workspace_bytes(const LewinCoreBwdArgs*, int) { return 0; }
int lewin_attn_fwd_kernel_mask(const LewinAttnFwdArgs* a, int dtype) {
    if (!a) return 0;
    const AttnPlan p = plan_attn(a, dtype == LEWIN_DTYPE_BF16);
    if (p.fused) return 1 << LEWIN_ATTN_K_FUSED;
    return (p.ln_stats ? 1 : 0) | 0x1C;
}
int lewin_leff_fwd_kernel_mask(const LewinLeffFwdArgs* a, int dtype) {
    if (!a) return 0;
    if (check_leff(a) != 0) return 0;
    const LeffPlan p = plan_leff(a, dtype == LEWIN_DTYPE_BF16);
    if (p.tail) return (1 << LEWIN_LEFF_K_FC1) | (1 << LEWIN_LEFF_K_TAIL);
    return (p.ln_stats ? 1 : 0) | 0xE;
}
int lewin_leff_fwd_supports_ld_out(const LewinLeffFwdArgs* a, int dtype) {
    if (!a || check_leff(a) != 0) return 0;
    LewinLeffFwdArgs b = *a;
    if (b.ld_out == 0 || b.ld_out == b.C) b.ld_out = b.C + 8;      // ask about a strided output
    return leff_ld_out_ok(&b, plan_leff(&b, dtype == LEWIN_DTYPE_BF16)) ? 1 : 0;
}
int lewin_leff_fwd_f32(const LewinLeffFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return leff_fwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_leff_fwd_bf16(const LewinLeffFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return leff_fwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}

int lewin_attn_bwd_f32(const LewinAttnBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return lewin::attn_bwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_attn_bwd_bf16(const LewinAttnBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return lewin::attn_bwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_leff_bwd_f32(const LewinLeffBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return lewin::leff_bwd<float>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
int lewin_leff_bwd_bf16(const LewinLeffBwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return lewin::leff_bwd<__nv_bfloat16>(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}

size_t lewin_attn_fwd_workspace_bytes(const LewinAttnFwdArgs* a, int) { return a ? attn_fwd_ws(a) : 0; }
size_t lewin_leff_fwd_workspace_bytes(const LewinLeffFwdArgs* a, int) { return a ? leff_fwd_ws(a) : 0; }
size_t lewin_attn_bwd_workspace_bytes(const LewinAttnBwdArgs* a, int dtype) { return a ? lewin::attn_bwd_ws(a, dtype) : 0; }
size_t lewin_leff_bwd_workspace_bytes(const LewinLeffBwdArgs* a, int dtype) { return a ? lewin::leff_bwd_ws(a, dtype) : 0; }

int lewin_upsample_fwd_bf16(const LewinUpsampleFwdArgs* a, void* ws, size_t n, lewin_stream_t s) {
    return upsample_fwd_bf16(a, ws, n, reinterpret_cast<cudaStream_t>(s));
}
size_t lewin_upsample_fwd_workspace_bytes(const LewinUpsampleFwdArgs* a, int) { return a ? upsample_ws(a) : 0; }

int lewin_input_proj_fwd_bf16(const LewinInputProjArgs* a, lewin_stream_t s) {
    return input_proj_fwd_bf16(a, reinterpret_cast<cudaStream_t>(s));
}

int lewin_abi_version(void) { return LEWIN_ABI_VERSION; }
long long lewin_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* lewin_build_info(void) {
#define LEWIN_STR2(x) #x
#define LEWIN_STR(x) LEWIN_STR2(x)
    return "lewin_b200 sm_100a; nvcc " LEWIN_STR(__CUDACC_VER_MAJOR__) "." LEWIN_STR(__CUDACC_VER_MINOR__)
           "; f32: mma.sync 3xTF32; bf16: tcgen05.mma kind::f16 + TMEM";
}

const char* lewin_error_string(int code) {
    switch (code) {
        case 0: return "ok";
        case LEWIN_E_NULL: return "required pointer is NULL";
        case LEWIN_E_SHAPE: return "unsupported shape (need H,W % 8 == 0, C % 32 == 0, C <= 1024, head_dim = C / nH in {32, 64, 128}, shift in {0..7})";
        case LEWIN_E_ALIGN: return "pointer not 16-byte aligned";
        case LEWIN_E_WORKSPACE: return "workspace missing or too small";
        case LEWIN_E_DTYPE: return "unknown dtype";
        case LEWIN_E_ARCH: return "device is not compute capability 10.x (sm_100a only, no fallback)";
        default: return code > 0 ? "CUDA runtime error (cudaError_t)" : "unknown error";
    }
}

}  // extern "C"
