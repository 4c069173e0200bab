// Translation unit of the implicit-GEMM projection convolutions (see conv_igemm.cuh): Downsample and OutputProj, bf16 inference.
#define LEWIN_TU_LITE 1
#include "abi_host.h"
#include "conv_igemm.cuh"

using namespace lewin;

namespace {

inline cudaError_t prep(const float* w, __nv_bfloat16* wb, int n_real, int N, int C, int taps, cudaStream_t st) {
    const long long total = static_cast<long long>(taps) * N * C;
    long long grid = (total + 255) / 256;
    if (grid > 2048) grid = 2048;
    cv::conv_prep_kernel<<<static_cast<unsigned>(grid), 256, 0, st>>>(w, wb, n_real, N, C, taps);
    return cudaGetLastError();
}

// bf16 images of the weights: [16 taps][2 Cin][Cin] (downsample), [9 taps][Cout][Cin] (conv3x3 unless the caller gives w_bf16)
__nv_bfloat16* downsample_layout(const LewinDownsampleArgs* a, WsLayout& L) {
    return L.take<__nv_bfloat16>(static_cast<size_t>(16) * 2 * a->Cin * a->Cin * 2);
}
__nv_bfloat16* conv3x3_layout(const LewinConv3x3Args* a, WsLayout& L) {
    return a->w_bf16 ? nullptr : L.take<__nv_bfloat16>(static_cast<size_t>(9) * a->Cout * a->Cin * 2);
}

}  // namespace

extern "C" {

size_t lewin_downsample_fwd_workspace_bytes(const LewinDownsampleArgs* a, int) { return a ? layout_bytes(downsample_layout, a) : 0; }

int lewin_downsample_fwd_bf16(const LewinDownsampleArgs* a, void* ws, size_t ws_bytes, lewin_stream_t s) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(s);
    if (!a || !a->x || !a->weight || !a->bias || !a->out) return LEWIN_E_NULL;
    const int Cin = a->Cin, N = 2 * Cin;
    const int ldx = a->ld_x > 0 ? a->ld_x : Cin, ldo = a->ld_out > 0 ? a->ld_out : N;
    if (a->B <= 0 || a->H < 4 || a->W < 4 || a->H % 2 || a->W % 2 || Cin % 32 || Cin > 512 || (Cin > 32 && Cin % 64) || (a->W / 2) % 8 ||
        ldx < Cin || ldx % 8 || ldo < N || ldo % 8)
        return LEWIN_E_SHAPE;
    if (!aligned16(a->x) || !aligned16(a->out)) return LEWIN_E_ALIGN;
    WsLayout L;
    __nv_bfloat16* wb = nullptr;
    int sms = 0;
    if (int rc = enter(ws, ws_bytes, downsample_layout, a, L, wb, sms)) return rc;

    const int pad = a->pad_h ? 1 : 0;
    cv::Args k{};
    k.B = a->B; k.Hout = pad ? a->H / 2 : a->H / 2 - 1; k.Wout = a->W / 2;
    k.N = N; k.n_real = N; k.px_shift = 3;
    const int BN = N < 256 ? N : 256;
    k.tiles_x = k.Wout / 8; k.tiles_y = (k.Hout + 15) / 16; k.col_tiles = N / BN;
    k.tiles = a->B * k.tiles_x * k.tiles_y * k.col_tiles;
    const int KCH = Cin == 32 ? 32 : 64;
    k.ntaps = 16; k.nkc = Cin / KCH;
    for (int ky = 0; ky < 4; ++ky)
        for (int kx = 0; kx < 4; ++kx) {
            cv::Tap& t = k.taps[ky * 4 + kx];
            const int hx = kx - 1;                      // input column 2 j + hx
            t.dj = hx < 0 ? -1 : hx >> 1; t.dc = (hx & 1) * ldx;
            const int hy = ky - pad;
            t.di = hy < 0 ? -1 : hy >> 1; t.dq = hy & 1;
        }
    k.bias = a->bias;
    k.out_tok = static_cast<__nv_bfloat16*>(a->out); k.ld_out = ldo;
    const unsigned long long dims[5] = {static_cast<unsigned long long>(ldx + Cin), static_cast<unsigned long long>(a->W / 2), 2ull,
                                        static_cast<unsigned long long>(a->H / 2), static_cast<unsigned long long>(a->B)};
    const unsigned long long ld2 = static_cast<unsigned long long>(ldx) * 2;
    const unsigned long long st[4] = {2 * ld2, static_cast<unsigned long long>(a->W) * ld2, 2ull * a->W * ld2,
                                      static_cast<unsigned long long>(a->H) * a->W * ld2};
    CUtensorMap amap{}, wmap{};
    if (!cv::make_5d(&amap, a->x, dims, st, KCH, 8, 16, KCH == 64) || !cv::make_w2d(&wmap, wb, 16ll * N, Cin, BN, KCH)) return LEWIN_E_SHAPE;
    CK(prep(a->weight, wb, N, N, Cin, 16, stream));
    if (KCH == 32) { CK((cv::launch_inst<32, 64>(k, amap, wmap, sms, stream))); }
    else if (BN == 128) { CK((cv::launch_inst<64, 128>(k, amap, wmap, sms, stream))); }
    else { CK((cv::launch_inst<64, 256>(k, amap, wmap, sms, stream))); }
    return 0;
}

size_t lewin_conv3x3_fwd_workspace_bytes(const LewinConv3x3Args* a, int) { return a ? layout_bytes(conv3x3_layout, a) : 0; }

int lewin_conv3x3_fwd_bf16(const LewinConv3x3Args* a, void* ws, size_t ws_bytes, lewin_stream_t s) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(s);
    if (!a || !a->x || (!a->weight && !a->w_bf16) || !a->out) return LEWIN_E_NULL;
    const int Cin = a->Cin, N = a->Cout;
    const int ldx = a->ld_x > 0 ? a->ld_x : Cin, ldo = a->ld_out > 0 ? a->ld_out : N;
    if (a->B <= 0 || a->H < 1 || a->W < 8 || a->W % 8 || Cin % 64 || Cin > 512 || N % 64 || N > 512 || ldx < Cin || ldx % 8 || ldo < N || ldo % 8)
        return LEWIN_E_SHAPE;
    if (!aligned16(a->x) || !aligned16(a->out) || (a->w_bf16 && !aligned16(a->w_bf16))) return LEWIN_E_ALIGN;
    WsLayout L;
    __nv_bfloat16* w_img = nullptr;                   // the per-call image of `weight`, or null
    int sms = 0;
    if (int rc = enter(ws, ws_bytes, conv3x3_layout, a, L, w_img, sms)) return rc;
    const __nv_bfloat16* wb = w_img ? w_img : static_cast<const __nv_bfloat16*>(a->w_bf16);
    cv::Args k{};
    k.B = a->B; k.Hout = a->H; k.Wout = a->W;
    k.N = N; k.n_real = N;
    k.px_shift = (a->W % 16 == 0) ? 4 : 3;                       // 8 x 16 or 16 x 8 output pixels per tile
    const int PX = 1 << k.px_shift, PY = 128 >> k.px_shift;
    const int BN = N < 256 ? N : 256;
    k.tiles_x = a->W / PX; k.tiles_y = (a->H + PY - 1) / PY; k.col_tiles = N / BN;
    k.tiles = a->B * k.tiles_x * k.tiles_y * k.col_tiles;
    k.ntaps = 9; k.nkc = Cin / 64;
    for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
            cv::Tap& t = k.taps[ky * 3 + kx];
            t.dj = kx - 1; t.dc = 0; t.di = ky - 1; t.dq = 0;   // zero fill outside the map == padding 1
        }
    k.bias = a->bias; k.relu = a->relu ? 1 : 0;
    k.out_tok = static_cast<__nv_bfloat16*>(a->out); k.ld_out = ldo;
    const unsigned long long ld2 = static_cast<unsigned long long>(ldx) * 2;
    const unsigned long long dims[5] = {static_cast<unsigned long long>(Cin), static_cast<unsigned long long>(a->W), 1ull,
                                        static_cast<unsigned long long>(a->H), static_cast<unsigned long long>(a->B)};
    const unsigned long long st[4] = {ld2, static_cast<unsigned long long>(a->W) * ld2, static_cast<unsigned long long>(a->W) * ld2,
                                      static_cast<unsigned long long>(a->H) * a->W * ld2};
    CUtensorMap amap{}, wmap{};
    if (!cv::make_5d(&amap, a->x, dims, st, 64, PX, PY, true) || !cv::make_w2d(&wmap, wb, 9ll * N, Cin, BN, 64)) return LEWIN_E_SHAPE;
    if (w_img) CK(prep(a->weight, w_img, N, N, Cin, 9, stream));
    if (BN == 64) { CK((cv::launch_inst<64, 64>(k, amap, wmap, sms, stream))); }
    else if (BN == 128) { CK((cv::launch_inst<64, 128>(k, amap, wmap, sms, stream))); }
    else { CK((cv::launch_inst<64, 256>(k, amap, wmap, sms, stream))); }
    return 0;
}

size_t lewin_output_proj_fwd_workspace_bytes(const LewinOutputProjArgs*, int) { return 0; }

int lewin_output_proj_fwd_bf16(const LewinOutputProjArgs* a, void*, size_t, lewin_stream_t s) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(s);
    if (!a || !a->x || !a->weight || !a->bias || !a->out) return LEWIN_E_NULL;
    const int Cin = a->Cin;
    const int ldx = a->ld_x > 0 ? a->ld_x : Cin;
    if (a->B <= 0 || a->H < 3 || a->W < 1 || Cin % 64 || Cin > 256 || a->Cout < 1 || a->Cout > 8 || ldx < Cin || ldx % 8)
        return LEWIN_E_SHAPE;
    if (!aligned16(a->x)) return LEWIN_E_ALIGN;
    int sms = 0;
    if (int rc = device_sms(&sms)) return rc;
    cv::op::Args k{};
    k.B = a->B; k.H = a->H; k.W = a->W; k.Cin = Cin; k.Cout = a->Cout;
    k.pad = a->pad_h ? 1 : 0;
    k.Hout = k.pad ? a->H : a->H - 2;
    k.weight = a->weight; k.bias = a->bias; k.resid = a->residual; k.out = a->out;
    CK(cv::op::launch(k, a->x, ldx, sms, stream));
    return 0;
}

}  // extern "C"
