"""CPU: the backward entries refuse what the forward entries refuse.  One table of edits to a valid LewinAttnFwdArgs /
LewinLeffFwdArgs, each with the code both directions must return; the backward's own rules; and a misaligned workspace.

Every call passes no workspace (or a misaligned one) and fake device addresses, so a call that passed its checks would stop
at LEWIN_E_WORKSPACE / LEWIN_E_ALIGN: none of them can reach a launch."""
import os

import pytest
import torch

NULL, SHAPE, ALIGN, WORKSPACE = -1, -2, -3, -4
P, Q = 0x1000, 0x1004          # a 16-byte aligned and a 4-byte aligned fake address


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    if not os.path.isfile(g.LIB):
        g.build()
    from lewin_b200 import _lib
    return _lib.load()


def _set(**kw):
    return lambda f: [setattr(f, k, v) for k, v in kw.items()]


def _attn_fwd(C=64, nH=2, hw=16, shift=4):
    from lewin_b200 import _lib
    f = _lib.LewinAttnFwdArgs()
    f.B, f.H, f.W, f.C, f.nH, f.shift, f.use_rpb, f.analytic_shift_mask = 2, hw, hw, C, nH, shift, 1, 1
    for n in ("x", "y", "ln_w", "ln_b", "w_qkv", "b_qkv", "w_out", "b_out", "rpb_table", "index_sample", "qkv", "ctx", "top"):
        setattr(f, n, P)
    return f


def _attn_bwd(**kw):
    from lewin_b200 import _lib
    a = _lib.LewinAttnBwdArgs()
    a.fwd = _attn_fwd(**kw)
    a.fwd.save_for_backward, a.fwd.y = 1, None          # as ops._attn_backward passes it
    for n in ("dy", "dx", "d_ln_w", "d_ln_b", "d_w_qkv", "d_b_qkv", "d_w_out", "d_b_out", "d_rpb_table"):
        setattr(a, n, P)
    return a


def _leff_fwd(C=64):
    from lewin_b200 import _lib
    f = _lib.LewinLeffFwdArgs()
    f.B, f.H, f.W, f.C, f.hidden, f.fused, f.save_for_backward = 2, 16, 16, C, 4 * C, 1, 1
    for n in ("y", "out", "ln_w", "ln_b", "w1", "b1", "w_dw", "b_dw", "w2", "b2", "h1", "h2", "a1", "a2"):
        setattr(f, n, P)
    return f


def _leff_bwd(**kw):
    from lewin_b200 import _lib
    a = _lib.LewinLeffBwdArgs()
    a.fwd = _leff_fwd(**kw)
    a.fwd.out = None                                    # as ops._leff_backward passes it
    for n in ("dout", "dy", "d_ln_w", "d_ln_b", "d_w1", "d_b1", "d_w_dw", "d_b_dw", "d_w2", "d_b2"):
        setattr(a, n, P)
    return a


# (edit of the forward struct, code of the forward and the backward)
ATTN_SHARED = {
    "valid": (_set(), WORKSPACE),
    "shift_9": (_set(shift=9), SHAPE),
    "shift_without_room": (_set(H=8, W=8, B=8), SHAPE),
    "B_0": (_set(B=0), SHAPE),
    "H_not_multiple_of_8": (_set(H=20), SHAPE),
    "W_not_multiple_of_8": (_set(W=12), SHAPE),
    "C_not_multiple_of_32": (_set(C=48), SHAPE),
    "C_above_1024": (_set(C=1056, nH=33), SHAPE),
    "head_dim_96": (_set(C=96, nH=1), SHAPE),
    "nH_0": (_set(nH=0), SHAPE),
    "x_misaligned": (_set(x=Q), ALIGN),
    "qkv_misaligned": (_set(qkv=Q), ALIGN),
    "ctx_misaligned": (_set(ctx=Q), ALIGN),
    "w_qkv_misaligned": (_set(w_qkv=Q), ALIGN),
    "w_out_bf16_misaligned": (_set(w_out_bf16=Q), ALIGN),
    "mask_without_nW_mask": (_set(mask=P, nW_mask=0), SHAPE),
    "mask_nW_not_dividing": (_set(mask=P, nW_mask=3), SHAPE),
    "mask_misaligned": (_set(mask=Q, nW_mask=8), ALIGN),
    "windowed_with_shift": (_set(windowed=1, analytic_shift_mask=0), SHAPE),
    "band_row_not_multiple_of_8": (_set(band_mode=1, band_y0=4, band_Hg=32), SHAPE),
    "token_mask_Bm_not_dividing": (_set(token_mask=P, Bm=3), SHAPE),
    "token_mask_with_dense_mask": (_set(token_mask=P, Bm=1, mask=P, nW_mask=8), SHAPE),
    "token_mask_misaligned": (_set(token_mask=Q, Bm=1), ALIGN),
    "x_null": (_set(x=None), NULL),
    "w_qkv_null": (_set(w_qkv=None), NULL),
    "qkv_null": (_set(qkv=None), NULL),
    "ln_w_null": (_set(ln_w=None), NULL),
}

LEFF_SHARED = {
    "valid": (_set(), WORKSPACE),
    "B_0": (_set(B=0), SHAPE),
    "H_0": (_set(H=0), SHAPE),
    "C_not_multiple_of_32": (_set(C=48), SHAPE),
    "C_above_1024": (_set(C=1056, hidden=4224), SHAPE),
    "hidden_not_multiple_of_32": (_set(hidden=100), SHAPE),
    "ld_out_below_C": (_set(ld_out=32), SHAPE),
    "ld_out_not_multiple_of_8": (_set(ld_out=68), SHAPE),
    "y_misaligned": (_set(y=Q), ALIGN),
    "w1_misaligned": (_set(w1=Q), ALIGN),
    "h1_misaligned": (_set(h1=Q), ALIGN),
    "a2_misaligned": (_set(a2=Q), ALIGN),
    "w2_bf16_misaligned": (_set(w2_bf16=Q), ALIGN),
    "y_null": (_set(y=None), NULL),
    "w2_null": (_set(w2=None), NULL),
    "ln_b_null": (_set(ln_b=None), NULL),
}


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("row", sorted(ATTN_SHARED))
def test_attention_backward_returns_the_forwards_code(lib, dtype, row):
    edit, code = ATTN_SHARED[row]
    f, b = _attn_fwd(), _attn_bwd()
    edit(f)
    edit(b.fwd)
    assert getattr(lib, f"lewin_attn_fwd_{dtype}")(f, None, 0, None) == code
    assert getattr(lib, f"lewin_attn_bwd_{dtype}")(b, None, 0, None) == code


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("row", sorted(LEFF_SHARED))
def test_leff_backward_returns_the_forwards_code(lib, dtype, row):
    edit, code = LEFF_SHARED[row]
    f, b = _leff_fwd(), _leff_bwd()
    edit(f)
    edit(b.fwd)
    assert getattr(lib, f"lewin_leff_fwd_{dtype}")(f, None, 0, None) == code
    assert getattr(lib, f"lewin_leff_bwd_{dtype}")(b, None, 0, None) == code


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_backward_rules_of_its_own(lib, dtype):
    """Beyond the forward's rules: at most 16 heads, and dy / dx / dout and every gradient pointer given present and aligned.
    The forward needs neither y nor out from the backward (ops passes NULL)."""
    attn = getattr(lib, f"lewin_attn_bwd_{dtype}")
    leff = getattr(lib, f"lewin_leff_bwd_{dtype}")
    assert getattr(lib, f"lewin_attn_fwd_{dtype}")(_attn_fwd(C=1024, nH=32), None, 0, None) == WORKSPACE
    assert attn(_attn_bwd(C=1024, nH=32), None, 0, None) == SHAPE
    b = _attn_bwd()
    b.fwd.index_sample = None                                       # read by the forward only
    assert attn(b, None, 0, None) == WORKSPACE
    for n, v, code in (("dy", Q, ALIGN), ("dx", Q, ALIGN), ("d_w_qkv", Q, ALIGN), ("d_rpb_table", Q, ALIGN),
                       ("d_rpb_dense", Q, ALIGN), ("dx", None, NULL), ("d_b_out", None, NULL)):
        b = _attn_bwd()
        setattr(b, n, v)
        assert attn(b, None, 0, None) == code, n
    for n, v, code in (("dout", Q, ALIGN), ("dy", Q, ALIGN), ("d_w_dw", Q, ALIGN), ("d_ln_b", Q, ALIGN),
                       ("dout", None, NULL), ("d_w1", None, NULL)):
        b = _leff_bwd()
        setattr(b, n, v)
        assert leff(b, None, 0, None) == code, n


@pytest.mark.skipif(torch.cuda.is_available(), reason="a non-NULL fake workspace must not be able to reach a launch")
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("deterministic", [0, 1])
def test_misaligned_workspace_is_refused(lib, dtype, deterministic):
    """A workspace large enough but not 16-byte aligned is LEWIN_E_ALIGN before the device query, in both modes."""
    big = 1 << 40
    a, l = _attn_bwd(), _leff_bwd()
    a.deterministic = l.deterministic = deterministic
    assert getattr(lib, f"lewin_attn_bwd_{dtype}")(a, Q, big, None) == ALIGN
    assert getattr(lib, f"lewin_leff_bwd_{dtype}")(l, Q, big, None) == ALIGN
    assert getattr(lib, f"lewin_attn_fwd_{dtype}")(_attn_fwd(), Q, big, None) == ALIGN
    assert getattr(lib, f"lewin_leff_fwd_{dtype}")(_leff_fwd(), Q, big, None) == ALIGN


@pytest.mark.skipif(torch.cuda.is_available(), reason="a non-NULL fake workspace must not be able to reach a launch")
def test_misaligned_workspace_of_the_convolutions(lib):
    from lewin_b200 import _lib
    big = 1 << 40
    up = _lib.LewinUpsampleFwdArgs(B=1, H=16, W=16, Cin=64, Cout=32, ld_out=32, x=P, weight=P, bias=P, out=P)
    assert lib.lewin_upsample_fwd_bf16(up, Q, big, None) == ALIGN
    assert lib.lewin_upsample_fwd_bf16(up, None, 0, None) == WORKSPACE
    down = _lib.LewinDownsampleArgs(B=1, H=16, W=16, Cin=32, pad_h=1, x=P, weight=P, bias=P, out=P)
    assert lib.lewin_downsample_fwd_bf16(down, Q, big, None) == ALIGN
    assert lib.lewin_downsample_fwd_bf16(down, None, 0, None) == WORKSPACE
    conv = _lib.LewinConv3x3Args(B=1, H=8, W=8, Cin=64, Cout=64, x=P, weight=P, bias=P, out=P)
    assert lib.lewin_conv3x3_fwd_bf16(conv, Q, big, None) == ALIGN
    assert lib.lewin_conv3x3_fwd_bf16(conv, None, 0, None) == WORKSPACE
