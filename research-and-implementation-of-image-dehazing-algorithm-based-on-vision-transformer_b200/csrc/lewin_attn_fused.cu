// Translation unit of the fused attention-half kernel (see attn_fused.cuh).
#define LEWIN_TU_LITE 1      // no GELU tables / non-template kernels in this unit (they live in lewin_abi.cu)
#include "attn_fused_api.h"
#include "attn_fused.cuh"

namespace lewin {

bool attn_fused_supported(const LewinAttnFwdArgs* a) {
    const long long tokens = static_cast<long long>(a->B) * a->H * a->W;
    return !a->windowed && !a->save_for_backward && !a->mask && !(a->use_rpb && !a->rpb_table) &&
           (a->shift == 0 || a->analytic_shift_mask) && af::supported(a->C, a->nH, tokens);
}

int attn_fused_launch(const LewinAttnFwdArgs* a, int num_sms, cudaStream_t stream) {
    af::Args k{};
    k.x = static_cast<const __nv_bfloat16*>(a->x);
    k.y = static_cast<__nv_bfloat16*>(a->y);
    k.ln_w = a->ln_w; k.ln_b = a->ln_b;
    k.w_qkv = a->w_qkv; k.b_qkv = a->b_qkv; k.w_out = a->w_out; k.b_out = a->b_out;
    k.rpb_table = a->rpb_table; k.drop_scale = a->drop_scale;
    k.index_sample = a->index_sample; k.top = a->top;
    k.use_rpb = a->use_rpb; k.shift = a->shift;
    const int nWin = (a->H / 8) * (a->W / 8);
    k.M = static_cast<long long>(a->B) * a->H * a->W;
    k.windows = a->B * nWin;
    k.tiles = (k.windows + 1) / 2;
    k.tokens_per_image = a->H * a->W;
    k.map = WinMap{a->H, a->W, a->W / 8, nWin, a->shift, a->band_mode ? 0 : a->shift};
    k.mask_y0 = a->band_mode ? a->band_y0 : 0;
    k.mask_Hg = a->band_mode ? a->band_Hg : a->H;
    k.tmask = a->token_mask; k.Bm = a->token_mask ? a->Bm : 1;
    return static_cast<int>(af::launch(a->C, k, num_sms, stream));
}

}  // namespace lewin
