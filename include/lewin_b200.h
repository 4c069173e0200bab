/*
 * lewin_b200.h — C ABI of the B200 (sm_100a) LeWin hot path.
 *
 * The reference (xin-fight/...Vision-Transformer, Uformer_ProbSparse/) is pure PyTorch; the
 * "FFI" a maintainer binds is ctypes from Python (see INTEGRATION.md).  Every entry point
 * replaces a reference nn.Module forward (or its autograd backward), cited per function
 * as file:line relative to /root/reference/Uformer_ProbSparse/.
 *
 * Contract (all functions):
 *   - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller
 *     (inputs, outputs, saved tensors and the workspace) — the library never allocates,
 *     frees or retains pointers;
 *   - work is enqueued on `stream` of the caller's current device and never synchronises;
 *   - re-entrant, no global mutable state (safe under nn.DataParallel threads and under
 *     one-process-per-GPU torch.distributed);
 *   - return 0 on success; negative = argument/shape/alignment violation detected before
 *     any launch (LEWIN_E_*); positive = cudaError_t of a failed launch.  No C++ exception
 *     crosses the boundary;
 *   - there is no CPU fallback and no other architecture: the library contains sm_100a
 *     code only.
 *
 * dtype: `_f32` entry points take fp32 activations (the reference's inference precision,
 * test_long_GPU.py:91) and compute every contraction with error-compensated 3xTF32 tensor
 * core MMAs (fp32-grade accuracy, needed for exact top-u parity).  `_bf16` entry points
 * take bf16 activations (the reference under torch.autocast(bfloat16); My_train.py:224 uses
 * fp16 autocast) with fp32 accumulation and the reference's rounding points
 * (SURVEY.md A.4).  Parameters are always fp32 (the state_dict dtype).
 */
#ifndef LEWIN_B200_H
#define LEWIN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* lewin_stream_t; /* == cudaStream_t */
typedef struct CUevent_st*  lewin_event_t;  /* == cudaEvent_t  */

#define LEWIN_ABI_VERSION 7

/* error codes (negative) */
#define LEWIN_E_NULL      (-1)  /* a required pointer is NULL */
#define LEWIN_E_SHAPE     (-2)  /* unsupported dims (C % 32, C > 1024, head_dim = C / nH not in {32, 64, 128}, H/W % 8, ...) */
#define LEWIN_E_ALIGN     (-3)  /* a pointer is not 16-byte aligned */
#define LEWIN_E_WORKSPACE (-4)  /* workspace too small */
#define LEWIN_E_DTYPE     (-5)  /* unknown dtype tag */
#define LEWIN_E_ARCH      (-6)  /* current device is not compute capability 10.x */

#define LEWIN_DTYPE_F32  0
#define LEWIN_DTYPE_BF16 1

#define LEWIN_WIN      8     /* window side, My_model_1.py:752 */
#define LEWIN_NTOK     64    /* tokens per window */
#define LEWIN_TOPU     25    /* u = U_part = 5*ceil(ln 64), ProbSparse/attn.py:310-315 */
#define LEWIN_RPB_ROWS 225   /* (2*8-1)^2, My_model_1.py:362 */

/* ------------------------------------------------------------------------------------------
 * Attention half of LeWinTransformerBlock.forward (My_model_1.py:803-872):
 *   y = x + drop_scale[b] * unroll(unwindow( WindowAttention( window(roll( LN1(x) )) ) ))
 * with WindowAttention.forward (My_model_1.py:400-415) -> AttentionLayer.forward
 * (ProbSparse/attn.py:385-461) -> ProbAttention.forward (attn.py:287-342).
 *
 * Two addressing modes:
 *   windowed == 0 (fused block half): x, y are [B, H, W, C] token-major; LN1, the cyclic shift,
 *       window_partition / window_reverse (My_model_1.py:550-601) and the residual add are folded
 *       into the load / store addressing.
 *   windowed == 1 (strict drop-in at WindowAttention.forward): x, y are [B_, 64, C] windows
 *       (B_ = B * (H/8) * (W/8), batch-major); no LN, no roll, no residual.
 * Masks are added to the post-softmax probabilities exactly as attn.py:236-261, in one fp32 add
 * after the relative-position bias:
 *   - `mask` (nullable) is a dense fp32 [nW_mask, 64, 64], window w takes slice (w mod nW_mask);
 *   - if `analytic_shift_mask` != 0 and shift > 0, the shift mask of My_model_1.py:803-836 is
 *     evaluated from window coordinates instead of being materialised (combinable with `mask`);
 *   - `token_mask` (nullable, fused block half only) is the input mask of My_model_1.py:791-798
 *     as one fp32 value per token: the caller's F.interpolate(mask, size=(H, W)) as [Bm, H, W],
 *     image b using mask (b mod Bm).  For query token i and key token j of a window the term is
 *     -100 where the fp32 product m_i * m_j != 0, else 0, and is combined with the analytic
 *     shift mask before the single add, so the result equals the dense [B*nW, 64, 64] mask the
 *     reference builds.  Window (wy, wx) reads m[wy*8 + r/8, wx*8 + r%8] for its row r: the
 *     unshifted frame, as the reference partitions the mask (not the pixel a rolled token came
 *     from).  Not combinable with `mask`, `windowed` or `band_mode` (LEWIN_E_SHAPE); B % Bm == 0.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t B, H, W, C, nH;        /* head_dim = C / nH (d_keys = d_model // n_heads, attn.py:370-372) in {32, 64, 128};
                                      32 (embed_dim 32, My_model_1.py:962) takes the register-resident bf16 kernels */
    int32_t shift;                 /* 0 or 4 (My_model_1.py:927) */
    int32_t windowed;              /* addressing mode, see above */
    int32_t use_rpb;               /* options.is_relative_position_bias (options.py:5, attn.py:227) */
    int32_t analytic_shift_mask;   /* evaluate the shift mask from coordinates */
    int32_t nW_mask;               /* windows in `mask` (0 if mask == NULL) */
    int32_t save_for_backward;     /* 1: qkv / ctx / top are kept valid for lewin_attn_bwd_* */
    int32_t reserved;

    const void*  x;                /* activations, dtype per entry point */
    void*        y;
    const float* ln_w;             /* norm1.weight [C]   (ignored when windowed) */
    const float* ln_b;             /* norm1.bias   [C] */
    const float* w_qkv;            /* [3C, C]: rows = query|key|value_projection.weight (attn.py:377-379) */
    const float* b_qkv;            /* [3C] */
    const float* w_out;            /* out_projection.weight [C, C] (attn.py:381) */
    const float* b_out;            /* [C] */
    const float* rpb_table;        /* relative_position_bias_table [225, nH] (My_model_1.py:362), or NULL if rpb_dense */
    const float* rpb_dense;        /* gathered bias [nH, 64, 64] as AttentionLayer.forward receives it (attn.py:385), or NULL */
    const int32_t* index_sample;   /* [64, 25] key-sample indices drawn by the caller exactly as attn.py:91 */
    const float* mask;             /* dense [nW_mask, 64, 64] or NULL */
    const float* drop_scale;       /* [B] per-sample DropPath factor (0 or 1/keep) or NULL (My_model_1.py:872) */

    /* caller-owned intermediates (also the saved tensors for backward).  A call that lewin_attn_fwd_kernel_mask reports as
     * the single fused kernel (bit LEWIN_ATTN_K_FUSED) keeps q|k|v and ctx on chip: the two buffers must still be non-NULL
     * and 16-byte aligned but are not touched (16 bytes each suffice). */
    void*    qkv;                  /* [B_*64, 3C] activations dtype */
    void*    ctx;                  /* [B_*64, C]  activations dtype */
    uint8_t* top;                  /* [B_, nH, 25] selected query indices (M_top, attn.py:122), by descending M */

    /* optional per-kernel timing: caller-owned events, 2 per kernel (begin, end) recorded on `stream`
     * around each launch, in the order LEWIN_ATTN_K_*; NULL = off */
    lewin_event_t* timing;

    /* optional (bf16 calls, C >= 256): the caller's own bf16 images of w_qkv [3C, C] and w_out [C, C] (round-to-nearest
     * of the fp32 weights).  When both are given the library skips its per-call weight conversion kernels (inference:
     * the weights are constants, the caller converts once); NULL = convert into the workspace on every call. */
    const void* w_qkv_bf16;
    const void* w_out_bf16;

    /* Row-band mode (canvas-mode sharding, test_long_GPU.py:85-92 split over GPUs by rows; fused block half, forward only):
     * x / y are a band of H rows of an image band_Hg rows tall, laid out by the caller in SHIFTED-FRAME row order (for a
     * shifted block: the band's own rows from `shift` on, followed by the first `shift` rows of the next band - the rows
     * torch.roll would bring in).  The cyclic shift then applies to the columns only, and the analytic shift mask
     * (My_model_1.py:803-836) takes its row regions at shifted-frame row band_y0 + (row in the band).  band_mode = 0: whole image. */
    int32_t band_mode, band_y0, band_Hg, reserved2;

    /* Input mask per token (see the mask paragraph above): [Bm, H, W] fp32, 16-byte aligned, or NULL.  Saved for and read
     * again by lewin_attn_bwd_*. */
    const float* token_mask;
    int32_t Bm, reserved3;
} LewinAttnFwdArgs;

#define LEWIN_ATTN_K_LNSTATS 0
#define LEWIN_ATTN_K_FUSED   1   /* the whole half as ONE kernel (bf16 inference, C <= 64): replaces slots 0 and 2-4.  (Slot 1 was the
                                    sample-multiplicity pre-pass until ABI 2; that table is now built inside the core kernels.) */
#define LEWIN_ATTN_K_QKV     2
#define LEWIN_ATTN_K_CORE    3
#define LEWIN_ATTN_K_OUT     4
#define LEWIN_ATTN_NKERNELS  5

int lewin_attn_fwd_f32 (const LewinAttnFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_attn_fwd_bf16(const LewinAttnFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);

/* Backward of the attention half (autograd of the same reference lines; gradient paths in
 * SURVEY.md section 3.4).  Gradients of parameters are ACCUMULATED (+=) into fp32 buffers the
 * caller zero-initialises, dx is written.  Shapes as the forward's (C % 32 == 0, C <= 1024,
 * head_dim = C / nH in {32, 64, 128}) with nH <= 16; anything else returns LEWIN_E_SHAPE.
 *
 * `deterministic` (all three backward structs): 0 = parameter gradients are summed with fp32 atomics, whose order varies from
 * run to run.  1 = every parameter gradient of the call is a fixed-order sum: each reduction unit stores its partial into its
 * own slot of a workspace slab, and one reduction launch at the end of the call sums the slots in order and adds the result
 * ONCE into the caller's buffer (still accumulated).  The slot counts depend on the shape alone, so the bits are the same on
 * any sm_100 device.  The data gradients (dx / dy / dqkv) are the same in both modes.  The *_workspace_bytes queries read the
 * flag (the slabs are included with 1).  torch.use_deterministic_algorithms(True) sets it from the Python layer. */
typedef struct {
    LewinAttnFwdArgs fwd;          /* same tensors as the forward call (x, params, qkv, ctx, top, ...) */
    const void* dy;                /* same shape/dtype as y */
    void*       dx;                /* same shape/dtype as x */
    float* d_ln_w;  float* d_ln_b; /* [C]  (ignored when windowed) */
    float* d_w_qkv; float* d_b_qkv;/* [3C, C], [3C] */
    float* d_w_out; float* d_b_out;/* [C, C], [C] */
    float* d_rpb_table;            /* [225, nH] (when fwd.rpb_table is given) */
    float* d_rpb_dense;            /* [nH, 64, 64] gradient w.r.t. the gathered bias (when fwd.rpb_dense is given: the
                                      relative_position_bias argument of AttentionLayer.forward, attn.py:385), or NULL */
    int32_t deterministic;         /* 1: fixed-order parameter-gradient sums (see above) */
    int32_t reserved;
} LewinAttnBwdArgs;

int lewin_attn_bwd_f32 (const LewinAttnBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_attn_bwd_bf16(const LewinAttnBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * ProbAttention.forward alone (ProbSparse/attn.py:287-342) on already-projected q | k | v:
 * qkv is [B_*64, 3C] (columns q | k | v, head h at [h*D, h*D+D) of each third, D = head_dim,
 * C = nH * D), ctx is [B_*64, C] == the reference's returned context [B_, 64, nH, D].
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t B_, nH, use_rpb, nW_mask;
    int32_t head_dim;              /* D in {32, 64, 128}; 0 = 32 */
    int32_t reserved;
    const void*  qkv;
    void*        ctx;
    const float* rpb_table;        /* [225, nH] or NULL */
    const float* rpb_dense;        /* [nH, 64, 64] or NULL */
    const int32_t* index_sample;   /* [64, 25] */
    const float* mask;             /* [nW_mask, 64, 64] or NULL */
    uint8_t*     top;              /* [B_, nH, 25] or NULL */
} LewinCoreFwdArgs;

int lewin_probsparse_core_fwd_f32 (const LewinCoreFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_probsparse_core_fwd_bf16(const LewinCoreFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_probsparse_core_fwd_workspace_bytes(const LewinCoreFwdArgs* a, int dtype);

/* Backward of ProbAttention.forward (what autograd derives from attn.py:287-342, SURVEY.md section 3.4) for the
 * selection saved by the forward (`fwd.top`, required): dqkv [B_*64, 3C] is WRITTEN (dq is zero on the lazy rows),
 * the bias gradients are ACCUMULATED into fp32 buffers the caller zero-initialises (either may be NULL).  The workspace is
 * empty unless `deterministic` is 1. */
typedef struct {
    LewinCoreFwdArgs fwd;          /* same qkv / rpb / mask / top as the forward call (index_sample, ctx unused) */
    const void* dctx;              /* [B_*64, C] gradient of the returned context */
    void*       dqkv;              /* [B_*64, 3C] */
    float*      d_rpb_table;       /* [225, nH], used when fwd.rpb_table is given */
    float*      d_rpb_dense;       /* [nH, 64, 64], used when fwd.rpb_dense is given */
    int32_t     deterministic;     /* 1: fixed-order bias-gradient sums (see LewinAttnBwdArgs) */
    int32_t     reserved;
} LewinCoreBwdArgs;

int lewin_probsparse_core_bwd_f32 (const LewinCoreBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_probsparse_core_bwd_bf16(const LewinCoreBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_probsparse_core_bwd_workspace_bytes(const LewinCoreBwdArgs* a, int dtype);

/* ------------------------------------------------------------------------------------------
 * LeFF half of the block (My_model_1.py:873 with LeFF.forward :496-534):
 *   out = y + drop_scale[b] * Linear2( GELU( dwconv3x3( GELU( Linear1( LN2(y) ) ) ) ) )
 * fused == 1: y, out are [B, H, W, C] and LN2 + residual are applied (block half);
 * fused == 0: strict drop-in at LeFF.forward: out = LeFF(y), no LN, no residual.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t B, H, W, C, hidden;    /* hidden = 4C (mlp_ratio 4, My_model_1.py:777) */
    int32_t fused;
    int32_t save_for_backward;     /* 1: pre-activations a1, a2 are written as well */
    int32_t ld_out;                /* elements between consecutive tokens of `out` (0 = C).  > C: `out` is a column block of a
                                    * wider buffer, e.g. the right half of the decoder's torch.cat([up, skip]) buffer
                                    * (My_model_1.py:1189-1204), so the skip copy disappears; bf16 inference calls for which
                                    * lewin_leff_fwd_supports_ld_out() returns 1 */

    const void*  y;
    void*        out;
    const float* ln_w;  const float* ln_b;   /* norm2 [C] (ignored when !fused) */
    const float* w1;    const float* b1;     /* mlp.linear1.0 [hidden, C], [hidden] */
    const float* w_dw;  const float* b_dw;   /* mlp.dwconv.0 [hidden, 1, 3, 3], [hidden] */
    const float* w2;    const float* b2;     /* mlp.linear2.0 [C, hidden], [C] */
    const float* drop_scale;                 /* [B] or NULL */

    void* h1;                      /* [B*H*W, hidden] GELU(linear1), activations dtype */
    void* h2;                      /* [B*H*W, hidden] GELU(dwconv).  A call that lewin_leff_fwd_kernel_mask reports with bit
                                    * LEWIN_LEFF_K_TAIL keeps h2 on chip: the pointer must still be non-NULL and 16-byte
                                    * aligned but may be a small placeholder */
    void* a1;                      /* pre-GELU linear1 output (only if save_for_backward) */
    void* a2;                      /* pre-GELU dwconv output  (only if save_for_backward) */

    lewin_event_t* timing;         /* optional, 2 events per kernel in the order LEWIN_LEFF_K_*; NULL = off */

    /* optional (bf16 calls, C >= 256): caller's bf16 images of w1 [hidden, C] and w2 [C, hidden]; see LewinAttnFwdArgs */
    const void* w1_bf16;
    const void* w2_bf16;
} LewinLeffFwdArgs;

#define LEWIN_LEFF_K_LNSTATS 0
#define LEWIN_LEFF_K_FC1     1
#define LEWIN_LEFF_K_DWCONV  2
#define LEWIN_LEFF_K_FC2     3
#define LEWIN_LEFF_K_TAIL    4   /* depthwise conv + GELU + linear2 + residual as ONE kernel (bf16 inference, C <= 64): replaces
                                  * slots 2 and 3 (csrc/leff_tail.cuh: the conv tile is the tcgen05.mma A operand, h2 stays on chip) */
#define LEWIN_LEFF_NKERNELS  5

/* Bit k set <=> the forward call will record timing slot k (LEWIN_ATTN_K_* / LEWIN_LEFF_K_*) for these arguments. */
int lewin_attn_fwd_kernel_mask(const LewinAttnFwdArgs* a, int dtype);
int lewin_leff_fwd_kernel_mask(const LewinLeffFwdArgs* a, int dtype);
/* 1 if the forward call for these arguments can write `out` with a row stride ld_out > C */
int lewin_leff_fwd_supports_ld_out(const LewinLeffFwdArgs* a, int dtype);

int lewin_leff_fwd_f32 (const LewinLeffFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_leff_fwd_bf16(const LewinLeffFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);

/* Backward of the LeFF half: parameter gradients ACCUMULATED into zero-initialised fp32 buffers (with `deterministic` = 1 as
 * fixed-order sums, see LewinAttnBwdArgs), dy written.
 * C % 32 == 0, hidden % 32 == 0, C <= 1024 (as the forward); anything else returns LEWIN_E_SHAPE. */
typedef struct {
    LewinLeffFwdArgs fwd;
    const void* dout;              /* gradient of `out` */
    void*       dy;                /* gradient of `y` */
    float* d_ln_w; float* d_ln_b;
    float* d_w1;   float* d_b1;
    float* d_w_dw; float* d_b_dw;
    float* d_w2;   float* d_b2;
    int32_t deterministic;         /* 1: fixed-order parameter-gradient sums (see LewinAttnBwdArgs) */
    int32_t reserved;
} LewinLeffBwdArgs;

int lewin_leff_bwd_f32 (const LewinLeffBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
int lewin_leff_bwd_bf16(const LewinLeffBwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);

/* Workspace sizes (bytes) for the calls above; dtype = LEWIN_DTYPE_*.  0 is a valid answer. */
size_t lewin_attn_fwd_workspace_bytes(const LewinAttnFwdArgs* a, int dtype);
size_t lewin_attn_bwd_workspace_bytes(const LewinAttnBwdArgs* a, int dtype);
size_t lewin_leff_fwd_workspace_bytes(const LewinLeffFwdArgs* a, int dtype);
size_t lewin_leff_bwd_workspace_bytes(const LewinLeffBwdArgs* a, int dtype);

/* Library / build identification. */
/* ------------------------------------------------------------------------------------------
 * SURVEY section 8(f) rank 2 (first step beyond the block): Upsample.forward, My_model_1.py:633-648 —
 * nn.ConvTranspose2d(in, out, kernel_size=2, stride=2) on the token map.  Kernel 2 / stride 2 never
 * overlaps, so it is a token GEMM  [B*H*W, Cin] x [Cin, 4*Cout]  whose output row (b, i, j) / column
 * block (di, dj) lands at pixel (2i+di, 2j+dj): the pixel shuffle is the epilogue's row address, the
 * bias is fused, and `out` may be the left half of the [.., 2*Cout] buffer that torch.cat([up, skip])
 * would build (My_model_1.py:1189-1204; ld_out = row stride of `out` in elements).  bf16 inference.
 */
typedef struct LewinUpsampleFwdArgs {
    int32_t B, H, W;               /* input map */
    int32_t Cin, Cout;
    int32_t ld_out;                /* elements between consecutive output tokens (>= Cout) */
    int32_t reserved0, reserved1;
    const void*  x;                /* [B, H, W, Cin] bf16 */
    const float* weight;           /* [Cin, Cout, 2, 2] (ConvTranspose2d.weight) */
    const float* bias;             /* [Cout] */
    void*        out;              /* [B, 2H, 2W, ld_out] bf16; columns [0, Cout) are written */
} LewinUpsampleFwdArgs;
int    lewin_upsample_fwd_bf16(const LewinUpsampleFwdArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_upsample_fwd_workspace_bytes(const LewinUpsampleFwdArgs* a, int dtype);

/* InputProj.forward, My_model_1.py:659-682: Conv2d(3 -> Cout, 3x3, pad 1) + LeakyReLU, NCHW fp32 image in, token-major
 * bf16 [B, H*W, Cout] out, with the autocast rounding points (conv -> bf16, + bias -> bf16, LeakyReLU -> bf16) in ONE pass
 * (the stock path is a cuDNN convolution + a bias-add pass + an activation pass over the 32-channel map). */
typedef struct LewinInputProjArgs {
    int32_t B, H, W, Cin, Cout;    /* Cin <= 4, Cout in {32, 64} */
    float   negative_slope;        /* nn.LeakyReLU default 0.01 */
    int32_t reserved0, reserved1;
    const float* x;                /* [B, Cin, H, W] fp32 */
    const float* weight;           /* [Cout, Cin, 3, 3] */
    const float* bias;             /* [Cout] */
    void*        out;              /* [B, H*W, Cout] bf16 */
} LewinInputProjArgs;
int lewin_input_proj_fwd_bf16(const LewinInputProjArgs* a, lewin_stream_t stream);

/* Downsample.forward, My_model_1.py:606-630: Conv2d(Cin, 2*Cin, kernel 4, stride 2, padding 1) on the token map, tokens out.
 * Implicit GEMM on tcgen05 (csrc/conv_igemm.cuh): one TMA box per (tap, 64-channel chunk), bias fused with torch's two
 * roundings (conv -> bf16, + bias -> bf16).  The input may be the right half of a torch.cat([up, skip]) buffer (ld_x >
 * Cin).  pad_h = 0: no padding in the row direction - the caller supplies the halo rows (canvas row bands), and the output
 * has H/2 - 1 rows.  bf16 inference.  (SURVEY 8(f) rank 2.) */
typedef struct LewinDownsampleArgs {
    int32_t B, H, W, Cin;          /* input map; H, W even, (W/2) % 8 == 0, Cin in {32, 64, 128, ..., 512} */
    int32_t ld_x;                  /* elements between consecutive input tokens (0 = Cin) */
    int32_t ld_out;                /* elements between consecutive output tokens (0 = 2*Cin) */
    int32_t pad_h;                 /* 1: padding 1 above / below (the reference); 0: rows already carry their halo */
    int32_t reserved;
    const void*  x;                /* [B, H, W, ld_x] bf16, channels [0, Cin) of each token */
    const float* weight;           /* [2*Cin, Cin, 4, 4] */
    const float* bias;             /* [2*Cin] */
    void*        out;              /* [B, Hout, W/2, ld_out] bf16, Hout = H/2 (pad_h) or H/2 - 1 */
} LewinDownsampleArgs;
int    lewin_downsample_fwd_bf16(const LewinDownsampleArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_downsample_fwd_workspace_bytes(const LewinDownsampleArgs* a, int dtype);

/* OutputProj.forward, My_model_1.py:696-733 (+ the `x + y` of Uformer.forward :1207): Conv2d(Cin, Cout <= 8, kernel 3,
 * padding 1) from the token map to an fp32 NCHW image, bias fused (conv -> bf16, + bias -> bf16), optional residual image
 * added in fp32.  One TMA halo tile per 16 x 16 pixels, the 9 taps gathered from it by ldmatrix into mma.sync (n8 tile):
 * the map is read once.  pad_h = 0: the caller supplies the halo rows, H - 2 rows out. */
typedef struct LewinOutputProjArgs {
    int32_t B, H, W, Cin, Cout;    /* Cin % 64 == 0, Cin <= 256, Cout <= 8 */
    int32_t ld_x;                  /* elements between consecutive input tokens (0 = Cin) */
    int32_t pad_h;
    int32_t reserved;
    const void*  x;                /* [B, H, W, ld_x] bf16 */
    const float* weight;           /* [Cout, Cin, 3, 3] */
    const float* bias;             /* [Cout] */
    const float* residual;         /* [B, Cout, Hout, W] fp32 or NULL */
    float*       out;              /* [B, Cout, Hout, W] fp32, Hout = H (pad_h) or H - 2 */
} LewinOutputProjArgs;
int    lewin_output_proj_fwd_bf16(const LewinOutputProjArgs* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_output_proj_fwd_workspace_bytes(const LewinOutputProjArgs* a, int dtype);

/* Conv2d(Cin, Cout, kernel 3, stride 1, padding 1) + bias (+ ReLU) on channel-last bf16 maps: the conv / ReLU pairs of the frozen
 * VGG19 feature extractor behind the reference's contrastive loss (My_CR.py:56-84 Vgg19.forward, :86-123 ContrastLoss.forward;
 * SURVEY 8(f) rank 1), and - with the kernel flipped and its channel axes swapped by the caller - their data gradients (the VGG
 * weights are frozen, so no weight gradient exists).  Implicit GEMM on tcgen05: one TMA box per (tap, 64-channel chunk), zero fill
 * outside the map = the padding, TMEM accumulator, bias / ReLU in the epilogue.  w_bf16: optional caller-owned image
 * [9][Cout][Cin] bf16 (tap = ky * 3 + kx) of the constant weights; otherwise `weight` is converted into the workspace per call. */
typedef struct LewinConv3x3Args {
    int32_t B, H, W, Cin, Cout;    /* W % 8 == 0; Cin, Cout multiples of 64, <= 512 */
    int32_t ld_x;                  /* elements between consecutive input pixels (0 = Cin) */
    int32_t ld_out;                /* elements between consecutive output pixels (0 = Cout) */
    int32_t relu;                  /* 1: ReLU after the bias */
    const void*  x;                /* [B, H, W, ld_x] bf16 (== an NCHW tensor in channels_last memory format) */
    const float* weight;           /* [Cout, Cin, 3, 3] fp32, or NULL if w_bf16 is given */
    const void*  w_bf16;           /* [9, Cout, Cin] bf16 or NULL */
    const float* bias;             /* [Cout] or NULL */
    void*        out;              /* [B, H, W, ld_out] bf16 */
} LewinConv3x3Args;
int    lewin_conv3x3_fwd_bf16(const LewinConv3x3Args* a, void* workspace, size_t workspace_bytes, lewin_stream_t stream);
size_t lewin_conv3x3_fwd_workspace_bytes(const LewinConv3x3Args* a, int dtype);

int         lewin_abi_version(void);     /* == LEWIN_ABI_VERSION */
long long   lewin_launch_count(void);    /* kernels launched by this library in this process (diagnostic counter) */
const char* lewin_build_info(void);      /* "sm_100a nvcc <ver> ..." */
const char* lewin_error_string(int code);/* text for a negative LEWIN_E_* code */

#ifdef __cplusplus
}
#endif
#endif /* LEWIN_B200_H */
