"""The two block halves as ``torch.library`` custom ops (SURVEY 8(b), "Python glue": opaque ops for torch.compile / export).

``torch.ops.lewin_b200.attn_fwd`` / ``attn_bwd`` and ``leff_fwd`` / ``leff_bwd`` wrap the same C-ABI calls as the
autograd.Functions of ops.py (``ops._attn_forward`` ... are shared), with shape-only fake implementations and a registered
autograd formula, so a traced graph carries ONE node per block half instead of breaking at the ctypes call.
``ops.lewin_attn`` / ``ops.lewin_leff`` route here while ``torch.compiler.is_compiling()``; eager calls keep the direct
autograd.Function path (no dispatcher overhead in the CUDA-graph-captured loops).  CUDA only, like everything else: the ops are
registered for ``device_types="cuda"`` and there is no CPU implementation to fall back to.

Custom-op schemas cannot return optional tensors, so an absent gradient / saved tensor crosses the op boundary as an empty
tensor and is turned back into ``None`` by the wrappers below.
"""
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import ops

_NS = "lewin_b200"


def _req(t, like):
    """None -> empty tensor (custom-op schemas have no optional returns)."""
    return t if t is not None else like.new_empty((0,))


# ----------------------------------------------------------------------------------------------------- attention half
@torch.library.custom_op(f"{_NS}::attn_fwd", mutates_args=(), device_types="cuda")
def attn_fwd(x: Tensor, ln_w: Optional[Tensor], ln_b: Optional[Tensor], w_qkv: Tensor, b_qkv: Tensor, w_out: Tensor,
             b_out: Tensor, rpb_table: Optional[Tensor], rpb_dense: Optional[Tensor], index_sample: Tensor,
             mask: Optional[Tensor], drop_scale: Optional[Tensor], B: int, H: int, W: int, num_heads: int, shift: int,
             windowed: bool, use_rpb: bool, analytic_shift_mask: bool, save: bool, token_mask: Optional[Tensor] = None
             ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (y, top u8 [B_, nH, 25], qkv [tokens, 3C], ctx [tokens, C]); qkv / ctx are empty unless ``save``."""
    geom = (B, H, W, num_heads, shift, windowed, use_rpb, analytic_shift_mask, save)
    y, top, saved = ops._attn_forward(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask,
                                      drop_scale, geom, token_mask)
    if not save:
        return y, top, x.new_empty((0,)), x.new_empty((0,))
    return y, top, saved.qkv, (saved.ctx if saved.ctx is not saved.qkv else saved.ctx.clone())      # op outputs must not alias


@attn_fwd.register_fake
def _(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, B, H, W, num_heads,
      shift, windowed, use_rpb, analytic_shift_mask, save, token_mask=None):
    C = x.shape[-1]
    tokens = B * H * W
    y = torch.empty_like(x, memory_format=torch.contiguous_format)
    top = x.new_empty((tokens // 64, num_heads, 25), dtype=torch.uint8)
    if not save:
        return y, top, x.new_empty((0,)), x.new_empty((0,))
    return y, top, x.new_empty((tokens, 3 * C)), x.new_empty((tokens, C))


@torch.library.custom_op(f"{_NS}::attn_bwd", mutates_args=(), device_types="cuda")
def attn_bwd(dy: Tensor, x: Tensor, ln_w: Optional[Tensor], ln_b: Optional[Tensor], w_qkv: Tensor, b_qkv: Tensor,
             w_out: Tensor, b_out: Tensor, rpb_table: Optional[Tensor], rpb_dense: Optional[Tensor], index_sample: Tensor,
             mask: Optional[Tensor], drop_scale: Optional[Tensor], qkv: Tensor, ctx: Tensor, top: Tensor, B: int, H: int,
             W: int, num_heads: int, shift: int, windowed: bool, use_rpb: bool, analytic_shift_mask: bool,
             token_mask: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (dx, d_ln_w, d_ln_b, d_w_qkv, d_b_qkv, d_w_out, d_b_out, d_rpb); d_rpb has the shape of whichever bias was given."""
    geom = (B, H, W, num_heads, shift, windowed, use_rpb, analytic_shift_mask, True)
    f = ops._f32c
    saved = ops.AttnSaved(x.contiguous(), f(ln_w), f(ln_b), f(w_qkv), f(b_qkv), f(w_out), f(b_out), f(rpb_table), f(rpb_dense),
                          ops.prepare_index_sample(index_sample, x.device), f(mask), f(drop_scale), qkv, ctx, top,
                          ops._token_mask(token_mask, B, H, W, x.device))
    dx, d_ln_w, d_ln_b, d_wq, d_bq, d_wo, d_bo, d_tab, d_dense = ops._attn_backward(saved, geom, dy, separate_grads=True)
    d_rpb = d_tab if d_tab is not None else d_dense
    z = dx.new_empty((0,), dtype=torch.float32)
    return dx, _req(d_ln_w, z), _req(d_ln_b, z), d_wq, d_bq, d_wo, d_bo, _req(d_rpb, z)


@attn_bwd.register_fake
def _(dy, x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, qkv, ctx, top,
      B, H, W, num_heads, shift, windowed, use_rpb, analytic_shift_mask, token_mask=None):
    def g(t):
        return x.new_empty((0,) if t is None else tuple(t.shape), dtype=torch.float32)
    return (torch.empty_like(x, memory_format=torch.contiguous_format), g(ln_w), g(ln_b), g(w_qkv), g(b_qkv), g(w_out),
            g(b_out), g(rpb_table if rpb_table is not None else rpb_dense))


def _attn_setup(ctx, inputs, output):
    (x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, *rest) = inputs
    geom, token_mask = rest[:9], (rest[9] if len(rest) > 9 else None)
    if not geom[-1]:
        ctx.geom = None              # an inference call reached autograd: refused in the backward, with the reason
        return
    _y, top, qkv, cbuf = output
    ctx.geom = tuple(geom[:-1])
    ctx.have = (ln_w is not None, rpb_table is not None, rpb_dense is not None)
    ctx.save_for_backward(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale,
                          qkv, cbuf, top, token_mask)


def _attn_backward(ctx, dy, _dtop, _dqkv, _dctx):
    if ctx.geom is None:
        raise RuntimeError("lewin_b200::attn_fwd was called with save=False but its output needs a gradient")
    (x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, qkv, cbuf,
     top, token_mask) = ctx.saved_tensors
    dx, d_ln_w, d_ln_b, d_wq, d_bq, d_wo, d_bo, d_rpb = torch.ops.lewin_b200.attn_bwd(
        dy, x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, qkv, cbuf, top,
        *ctx.geom, token_mask)
    has_ln, has_tab, has_dense = ctx.have
    return (dx, d_ln_w if has_ln else None, d_ln_b if has_ln else None, d_wq, d_bq, d_wo, d_bo,
            d_rpb if has_tab else None, d_rpb if (has_dense and not has_tab) else None,
            None, None, None) + (None,) * 10


torch.library.register_autograd(f"{_NS}::attn_fwd", _attn_backward, setup_context=_attn_setup)


# ---------------------------------------------------------------------------------------------------------- LeFF half
@torch.library.custom_op(f"{_NS}::leff_fwd", mutates_args=(), device_types="cuda")
def leff_fwd(y: Tensor, ln_w: Optional[Tensor], ln_b: Optional[Tensor], w1: Tensor, b1: Tensor, w_dw: Tensor, b_dw: Tensor,
             w2: Tensor, b2: Tensor, drop_scale: Optional[Tensor], B: int, H: int, W: int, fused: bool, save: bool
             ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (out, h1, h2, a1, a2): the hidden activations and pre-activations [tokens, 4C] the backward reads (empty unless
    ``save``)."""
    out, saved = ops._leff_forward(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, (B, H, W, fused, save))
    if saved is None:
        return (out,) + tuple(y.new_empty((0,)) for _ in range(4))
    return out, saved.h1, (saved.h2 if saved.h2 is not saved.h1 else saved.h2.clone()), saved.a1, saved.a2      # no aliasing


@leff_fwd.register_fake
def _(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, B, H, W, fused, save):
    out = torch.empty_like(y, memory_format=torch.contiguous_format)
    shape = (B * H * W, w1.shape[0]) if save else (0,)
    return (out,) + tuple(y.new_empty(shape) for _ in range(4))


@torch.library.custom_op(f"{_NS}::leff_bwd", mutates_args=(), device_types="cuda")
def leff_bwd(dout: Tensor, y: Tensor, ln_w: Optional[Tensor], ln_b: Optional[Tensor], w1: Tensor, b1: Tensor, w_dw: Tensor,
             b_dw: Tensor, w2: Tensor, b2: Tensor, drop_scale: Optional[Tensor], h1: Tensor, h2: Tensor, a1: Tensor,
             a2: Tensor, B: int, H: int, W: int, fused: bool
             ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (dy, d_ln_w, d_ln_b, d_w1, d_b1, d_w_dw, d_b_dw, d_w2, d_b2)."""
    f = ops._f32c
    saved = ops.LeffSaved(y.contiguous(), f(ln_w), f(ln_b), f(w1), f(b1), f(w_dw), f(b_dw), f(w2), f(b2), f(drop_scale), h1, h2,
                          a1, a2)
    dy, d_ln_w, d_ln_b, *rest = ops._leff_backward(saved, (B, H, W, fused, True), dout, separate_grads=True)
    z = dy.new_empty((0,), dtype=torch.float32)
    return (dy, _req(d_ln_w, z), _req(d_ln_b, z)) + tuple(rest)


@leff_bwd.register_fake
def _(dout, y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, h1, h2, a1, a2, B, H, W, fused):
    def g(t):
        return y.new_empty((0,) if t is None else tuple(t.shape), dtype=torch.float32)
    return (torch.empty_like(y, memory_format=torch.contiguous_format), g(ln_w), g(ln_b), g(w1), g(b1), g(w_dw), g(b_dw),
            g(w2), g(b2))


def _leff_setup(ctx, inputs, output):
    (y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, B, H, W, fused, save) = inputs
    if not save:
        ctx.geom = None
        return
    _out, h1, h2, a1, a2 = output
    ctx.geom = (B, H, W, fused)
    ctx.has_ln = ln_w is not None
    ctx.save_for_backward(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, h1, h2, a1, a2)


def _leff_backward(ctx, dout, _dh1, _dh2, _da1, _da2):
    if ctx.geom is None:
        raise RuntimeError("lewin_b200::leff_fwd was called with save=False but its output needs a gradient")
    (y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, h1, h2, a1, a2) = ctx.saved_tensors
    dy, d_ln_w, d_ln_b, d_w1, d_b1, d_wdw, d_bdw, d_w2, d_b2 = torch.ops.lewin_b200.leff_bwd(
        dout, y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, h1, h2, a1, a2, *ctx.geom)
    return (dy, d_ln_w if ctx.has_ln else None, d_ln_b if ctx.has_ln else None, d_w1, d_b1, d_wdw, d_bdw, d_w2, d_b2,
            None) + (None,) * 5


torch.library.register_autograd(f"{_NS}::leff_fwd", _leff_backward, setup_context=_leff_setup)


# --------------------------------------------------------------------------------- what ops.lewin_attn / lewin_leff call
def lewin_attn(x, *, B, H, W, num_heads, shift, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample,
               mask, drop_scale, windowed, use_rpb, analytic_shift_mask, need, token_mask=None):
    index_sample = ops.prepare_index_sample(index_sample, x.device)
    y, top, _qkv, _ctx = torch.ops.lewin_b200.attn_fwd(
        x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, int(B), int(H), int(W),
        int(num_heads), int(shift), bool(windowed), bool(use_rpb), bool(analytic_shift_mask), bool(need), token_mask)
    return y, top


def lewin_leff(y, *, B, H, W, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, fused, need):
    return torch.ops.lewin_b200.leff_fwd(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, int(B), int(H), int(W),
                                         bool(fused), bool(need))[0]
