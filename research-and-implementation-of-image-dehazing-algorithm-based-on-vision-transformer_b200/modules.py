"""nn.Module surface of the reference hot path, backed by the sm_100a ops.

Same class names, constructor arguments, forward signatures and state_dict layout as the reference
(SURVEY.md section 8b, Appendix B) so checkpoints load strictly and callers run unchanged:

  ProbAttention, AttentionLayer        ProbSparse/attn.py:43-342, 345-461
  WindowAttention                      My_model_1.py:336-415
  LeFF                                 My_model_1.py:477-534
  LeWinTransformerBlock                My_model_1.py:738-875
  LinearProjection (dead parameters)   My_model_1.py:264-300 — kept only for state_dict parity

All arithmetic of the block runs in the CUDA library; these classes hold parameters, draw
``index_sample`` from the CPU RNG exactly as attn.py:91 does, and call the ops.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from . import ops
from . import options as _options


def to_2tuple(x):
    return x if isinstance(x, tuple) else (x, x)


class DropPath(nn.Module):
    """Stochastic depth per sample (timm.models.layers.DropPath as used at My_model_1.py:775).

    ``sample_scale`` consumes the device RNG exactly like timm (``new_empty(B,1,..).bernoulli_``)."""

    def __init__(self, drop_prob=0.0):
        super().__init__()
        self.drop_prob = float(drop_prob)

    def sample_scale(self, x):
        """Per-sample factor [B] (0 or 1/keep), or None when inactive."""
        if self.drop_prob == 0.0 or not self.training:
            return None
        keep = 1.0 - self.drop_prob
        shape = (x.shape[0],) + (1,) * (x.ndim - 1)
        m = x.new_empty(shape).bernoulli_(keep)
        if keep > 0.0:
            m.div_(keep)
        return m.reshape(-1).float()

    def forward(self, x):
        s = self.sample_scale(x)
        return x if s is None else x * s.to(x.dtype).view((-1,) + (1,) * (x.ndim - 1))

    def extra_repr(self):
        return f"drop_prob={self.drop_prob}"


def draw_index_sample(L_K=64, L_Q=64, factor=5):
    """``torch.randint(L_K, (L_Q, sample_k))`` on the CPU global generator — the exact call of attn.py:91
    (same shape, same generator), so the RNG stream stays in lock-step with the reference."""
    sample_k = min(factor * int(np.ceil(np.log(L_K))), L_K)
    return torch.randint(L_K, (L_Q, sample_k))


def _use_rpb():
    """options.is_relative_position_bias, read at call time like attn.py:227 (the reference's own
    ``options`` module wins when it is importable, e.g. under patch())."""
    import sys
    ref = sys.modules.get("options")
    if ref is not None and hasattr(ref, "is_relative_position_bias"):
        return bool(ref.is_relative_position_bias)
    return bool(_options.is_relative_position_bias)


_FP16_NOTE = [False]


def _act_dtype(x):
    """bf16 under torch.autocast(cuda, bfloat16) (SURVEY A.4), else the input dtype.

    Under the reference's own fp16 autocast (My_train.py:224: ``torch.cuda.amp.autocast()`` + NativeScaler) the LeWin ops also
    compute in bf16 - the library has no fp16 kernels - and hand bf16 activations to the surrounding autocast ops, which
    cast them as they cast any other input.  bf16 has fp32's exponent range, so the scaler's loss scaling is unnecessary for
    these ops but harmless; the training script runs unchanged (tests/test_gpu_bf16.py::test_fp16_autocast_runs_on_bf16_kernels)."""
    if torch.is_autocast_enabled():
        adt = torch.get_autocast_dtype("cuda")
        if adt == torch.bfloat16:
            return torch.bfloat16
        if adt == torch.float16:
            if not _FP16_NOTE[0]:
                _FP16_NOTE[0] = True
                import warnings
                warnings.warn("lewin_b200: fp16 autocast requested; the LeWin ops compute in bf16 (no fp16 kernels)", stacklevel=3)
            return torch.bfloat16
    if x.dtype == torch.float16:
        return torch.bfloat16
    return x.dtype


# ------------------------------------------------------------------------------ ProbSparse
class ProbAttention(nn.Module):
    """ProbSparse/attn.py:43-342.  Holds no parameters.  ``forward`` takes already-projected
    q, k, v [B_, 64, nH, D] and returns (context [B_, 64, nH, D], None); differentiable in q, k, v and the bias."""

    def __init__(self, mask_flag=False, factor=5, scale=None, attention_dropout=0.1, output_attention=False):
        super().__init__()
        if mask_flag or output_attention or scale is not None or factor != 5:
            raise NotImplementedError("lewin_b200 implements the configuration hard-coded at attn.py:374 "
                                      "(mask_flag=False, factor=5, scale=None, output_attention=False)")
        self.factor = factor
        self.scale = scale
        self.mask_flag = mask_flag
        self.output_attention = output_attention
        self.dropout = nn.Dropout(attention_dropout)   # constructed but never applied (attn.py:68)
        self.softmax = nn.Softmax(dim=-1)

    def forward(self, queries, keys, values, relative_position_bias, SW_mask, attn_mask=None, index_sample=None):
        B_, L, H, D = queries.shape
        C = H * D
        if index_sample is None:
            index_sample = draw_index_sample(L, L, self.factor)
        if L != 64 or keys.shape[1] != 64:
            raise NotImplementedError("lewin_b200 ProbAttention supports 8x8 windows (L_Q = L_K = 64)")
        if D not in (32, 64, 128):
            raise NotImplementedError(f"lewin_b200 ProbAttention: head_dim {D} not built (32, 64, 128 are)")
        dt = _act_dtype(queries)
        qkv = torch.cat([queries.reshape(B_, L, C), keys.reshape(B_, L, C), values.reshape(B_, L, C)], -1).to(dt)
        out = ops.probsparse_core(qkv, num_heads=H, rpb_dense=relative_position_bias, mask=SW_mask,
                                  index_sample=index_sample, use_rpb=_use_rpb())
        return out.view(B_, L, H, D), None


class AttentionLayer(nn.Module):
    """ProbSparse/attn.py:345-461: q/k/v/out linears around ProbAttention (self-attention only)."""

    def __init__(self, d_model, n_heads, d_keys=None, d_values=None, mix=False):
        super().__init__()
        d_keys = d_keys or (d_model // n_heads)
        d_values = d_values or (d_model // n_heads)
        if mix:
            raise NotImplementedError("mix=True is not used by the reference (My_model_1.py:357)")
        self.inner_attention = ProbAttention(mask_flag=False, factor=5, scale=None, attention_dropout=0.1,
                                             output_attention=False)
        self.query_projection = nn.Linear(d_model, d_keys * n_heads)
        self.key_projection = nn.Linear(d_model, d_keys * n_heads)
        self.value_projection = nn.Linear(d_model, d_values * n_heads)
        self.out_projection = nn.Linear(d_values * n_heads, d_model)
        self.n_heads = n_heads
        self.mix = mix
        self._cat_cache = None

    def qkv_weights(self):
        """[3C, C] / [3C] concatenation of the three projections; cached while no grad is needed."""
        ps = (self.query_projection.weight, self.key_projection.weight, self.value_projection.weight,
              self.query_projection.bias, self.key_projection.bias, self.value_projection.bias)
        if torch.is_grad_enabled() and any(p.requires_grad for p in ps):
            return torch.cat(ps[:3], 0), torch.cat(ps[3:], 0)
        key = tuple((p.data_ptr(), p._version, p.device) for p in ps)
        if self._cat_cache is None or self._cat_cache[0] != key:
            with torch.no_grad():
                self._cat_cache = (key, torch.cat(ps[:3], 0).float().contiguous(), torch.cat(ps[3:], 0).float().contiguous())
        return self._cat_cache[1], self._cat_cache[2]

    def forward(self, queries, keys, values, relative_position_bias, SW_mask, attn_mask=None, index_sample=None):
        if not (queries is keys and keys is values):
            raise NotImplementedError("lewin_b200 AttentionLayer is self-attention only (the reference calls "
                                      "ProbSpare(x, x, x, ...), My_model_1.py:413)")
        x = queries
        B_, L, C = x.shape
        if index_sample is None:
            index_sample = draw_index_sample(L, L)
        w_qkv, b_qkv = self.qkv_weights()
        dt = _act_dtype(x)
        out = ops.lewin_attn(
            x.to(dt), B=B_, H=8, W=8, num_heads=self.n_heads, shift=0, ln_w=None, ln_b=None,
            w_qkv=w_qkv, b_qkv=b_qkv, w_out=self.out_projection.weight, b_out=self.out_projection.bias,
            rpb_table=None, rpb_dense=relative_position_bias, index_sample=index_sample, mask=SW_mask,
            windowed=True, use_rpb=_use_rpb(), analytic_shift_mask=False)
        return out, None


class LinearProjection(nn.Module):
    """My_model_1.py:264-300.  DEAD in the reference forward (SURVEY finding 6) — constructed only so the
    state_dict carries attn.qkv.to_q / attn.qkv.to_kv exactly like the reference."""

    def __init__(self, dim, heads=8, dim_head=64, dropout=0., bias=True):
        super().__init__()
        inner_dim = dim_head * heads
        self.heads = heads
        self.to_q = nn.Linear(dim, inner_dim, bias=bias)
        self.to_kv = nn.Linear(dim, inner_dim * 2, bias=bias)
        self.dim = dim
        self.inner_dim = inner_dim


class WindowAttention(nn.Module):
    """My_model_1.py:336-415."""

    def __init__(self, dim, win_size, num_heads, token_projection='linear', qkv_bias=True, qk_scale=None,
                 attn_drop=0., proj_drop=0., se_layer=False):
        super().__init__()
        if token_projection != 'linear' or se_layer:
            raise NotImplementedError("lewin_b200 implements token_projection='linear', se_layer=False "
                                      "(utils/model_utils.py:94 defaults)")
        self.dim = dim
        self.win_size = to_2tuple(win_size)
        self.num_heads = num_heads
        head_dim = dim // num_heads
        if dim % num_heads or head_dim not in (32, 64, 128):
            raise NotImplementedError(f"lewin_b200: head_dim = dim // num_heads = {dim}/{num_heads} is not built; 32, 64 and "
                                      "128 are (head_dim = embed_dim, My_model_1.py:962; the reference's embed_dim=16 "
                                      "variant, utils/model_utils.py:97, is not)")
        self.scale = qk_scale or head_dim ** -0.5
        self.ProbSpare = AttentionLayer(self.dim, self.num_heads)
        self.relative_position_bias_table = nn.Parameter(
            torch.zeros((2 * self.win_size[0] - 1) * (2 * self.win_size[1] - 1), num_heads))
        ws = self.win_size[0]
        ty, tx = torch.meshgrid(torch.arange(ws), torch.arange(self.win_size[1]), indexing="ij")
        ty, tx = ty.reshape(-1), tx.reshape(-1)
        rel = (ty[:, None] - ty[None, :] + ws - 1) * (2 * self.win_size[1] - 1) + (tx[:, None] - tx[None, :] + self.win_size[1] - 1)
        self.register_buffer("relative_position_index", rel.long())
        self.qkv = LinearProjection(dim, num_heads, dim // num_heads, bias=qkv_bias)   # dead, state_dict only
        self.token_projection = token_projection
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)                                                # dead, state_dict only
        self.se_layer = nn.Identity()
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)

    def forward(self, x, attn_kv=None, mask=None, index_sample=None):
        """x [B_, 64, C] pre-partitioned windows; mask [nW, 64, 64] or None -> [B_, 64, C]."""
        B_, N, C = x.shape
        if N != 64:
            raise NotImplementedError("lewin_b200 supports 8x8 windows (N=64)")
        if index_sample is None:
            index_sample = draw_index_sample(N, N)
        w_qkv, b_qkv = self.ProbSpare.qkv_weights()
        dt = _act_dtype(x)
        return ops.lewin_attn(
            x.to(dt), B=B_, H=8, W=8, num_heads=self.num_heads, shift=0, ln_w=None, ln_b=None,
            w_qkv=w_qkv, b_qkv=b_qkv, w_out=self.ProbSpare.out_projection.weight,
            b_out=self.ProbSpare.out_projection.bias, rpb_table=self.relative_position_bias_table,
            index_sample=index_sample, mask=mask, windowed=True, use_rpb=_use_rpb(), analytic_shift_mask=False)

    def extra_repr(self) -> str:
        return f'dim={self.dim}, win_size={self.win_size}, num_heads={self.num_heads}'


# ------------------------------------------------------------------------------------ LeFF
class LeFF(nn.Module):
    """My_model_1.py:477-534."""

    def __init__(self, dim=32, hidden_dim=128, act_layer=nn.GELU, drop=0.):
        super().__init__()
        if act_layer is not nn.GELU:
            raise NotImplementedError("lewin_b200 LeFF implements the exact (erf) GELU of the reference")
        self.linear1 = nn.Sequential(nn.Linear(dim, hidden_dim), act_layer())
        self.dwconv = nn.Sequential(
            nn.Conv2d(hidden_dim, hidden_dim, groups=hidden_dim, kernel_size=3, stride=1, padding=1), act_layer())
        self.linear2 = nn.Sequential(nn.Linear(hidden_dim, dim))
        self.dim = dim
        self.hidden_dim = hidden_dim

    def forward(self, x):
        bs, hw, c = x.shape
        hh = int(math.sqrt(hw))
        dt = _act_dtype(x)
        return ops.lewin_leff(
            x.to(dt), B=bs, H=hh, W=hh, ln_w=None, ln_b=None,
            w1=self.linear1[0].weight, b1=self.linear1[0].bias, w_dw=self.dwconv[0].weight, b_dw=self.dwconv[0].bias,
            w2=self.linear2[0].weight, b2=self.linear2[0].bias, fused=False)


# ------------------------------------------------------------------------------ LeWin block
def lewin_block_forward(blk, x, mask=None, index_sample=None, out=None):
    """LeWinTransformerBlock.forward (My_model_1.py:785-875) on the sm_100a ops.

    ``blk`` is any module with the reference attribute layout (norm1, attn.ProbSpare.*, attn.
    relative_position_bias_table, norm2, mlp.{linear1,dwconv,linear2}, shift_size, win_size, drop_path) —
    this package's LeWinTransformerBlock or the reference's own class after ``patch()``."""
    B, L, C = x.shape
    H = W = int(math.sqrt(L))
    if blk.win_size != 8:
        raise NotImplementedError("lewin_b200 supports win_size 8")
    ps = blk.attn.ProbSpare
    if index_sample is None:
        index_sample = draw_index_sample(64, 64)            # same point in the RNG stream as attn.py:91
    dt = _act_dtype(x)
    x = x.to(dt)
    token_mask = None
    if mask is not None:                                    # input-mask path (test_in_any_resolution.py:106)
        # My_model_1.py:791-792: the nearest-resized level mask, one value per token; the window partition and the pairwise
        # product (:793-798) are evaluated inside the attention kernels, together with the analytic shift mask
        token_mask = torch.nn.functional.interpolate(mask, size=(H, W))[:, 0]
    dp = blk.drop_path
    s0 = dp.sample_scale(x) if isinstance(dp, DropPath) else _foreign_droppath_scale(dp, x)
    if hasattr(ps, "qkv_weights"):
        w_qkv, b_qkv = ps.qkv_weights()
    else:
        w_qkv, b_qkv = _cat_qkv(ps)
    y = ops.lewin_attn(
        x, B=B, H=H, W=W, num_heads=blk.num_heads, shift=blk.shift_size,
        ln_w=blk.norm1.weight, ln_b=blk.norm1.bias, w_qkv=w_qkv, b_qkv=b_qkv,
        w_out=ps.out_projection.weight, b_out=ps.out_projection.bias,
        rpb_table=blk.attn.relative_position_bias_table, index_sample=index_sample, token_mask=token_mask,
        drop_scale=s0, windowed=False, use_rpb=_use_rpb(), analytic_shift_mask=True)
    s1 = dp.sample_scale(y) if isinstance(dp, DropPath) else _foreign_droppath_scale(dp, y)
    mlp = blk.mlp
    return ops.lewin_leff(
        y, B=B, H=H, W=W, ln_w=blk.norm2.weight, ln_b=blk.norm2.bias,
        w1=mlp.linear1[0].weight, b1=mlp.linear1[0].bias, w_dw=mlp.dwconv[0].weight, b_dw=mlp.dwconv[0].bias,
        w2=mlp.linear2[0].weight, b2=mlp.linear2[0].bias, drop_scale=s1, fused=True, out=out)


def _cat_qkv(ps):
    w = torch.cat([ps.query_projection.weight, ps.key_projection.weight, ps.value_projection.weight], 0)
    b = torch.cat([ps.query_projection.bias, ps.key_projection.bias, ps.value_projection.bias], 0)
    return w, b


def _foreign_droppath_scale(dp, x):
    """DropPath of another library (timm) under patch(): reproduce its Bernoulli draw."""
    p = float(getattr(dp, "drop_prob", 0.0) or 0.0)
    if p == 0.0 or not dp.training:
        return None
    keep = 1.0 - p
    m = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
    if keep > 0.0 and getattr(dp, "scale_by_keep", True):
        m.div_(keep)
    return m.reshape(-1).float()


class LeWinTransformerBlock(nn.Module):
    """My_model_1.py:738-875."""

    def __init__(self, dim, input_resolution, num_heads, win_size=8, shift_size=0, mlp_ratio=4., qkv_bias=True,
                 qk_scale=None, drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm,
                 token_projection='linear', token_mlp='leff', se_layer=False):
        super().__init__()
        if token_mlp != 'leff':
            raise NotImplementedError("lewin_b200 implements token_mlp='leff'")
        if norm_layer is not nn.LayerNorm:
            raise NotImplementedError("lewin_b200 implements norm_layer=nn.LayerNorm")
        self.dim = dim
        self.input_resolution = input_resolution
        self.num_heads = num_heads
        self.win_size = win_size
        self.shift_size = shift_size
        self.mlp_ratio = mlp_ratio
        self.token_mlp = token_mlp
        if min(self.input_resolution) <= self.win_size:      # My_model_1.py:764-766
            self.shift_size = 0
            self.win_size = min(self.input_resolution)
        assert 0 <= self.shift_size < self.win_size, "shift_size must in 0-win_size"
        self.norm1 = norm_layer(dim)
        self.attn = WindowAttention(dim, win_size=to_2tuple(self.win_size), num_heads=num_heads, qkv_bias=qkv_bias,
                                    qk_scale=qk_scale, attn_drop=attn_drop, proj_drop=drop,
                                    token_projection=token_projection, se_layer=se_layer)
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = LeFF(dim, int(dim * mlp_ratio), act_layer=act_layer, drop=drop)

    def extra_repr(self) -> str:
        return (f"dim={self.dim}, input_resolution={self.input_resolution}, num_heads={self.num_heads}, "
                f"win_size={self.win_size}, shift_size={self.shift_size}, mlp_ratio={self.mlp_ratio}")

    def forward(self, x, mask=None, index_sample=None, out=None):
        """out: optional destination view for the block's result (see ops.lewin_leff); the returned tensor is `out` when the
        call could use it."""
        return lewin_block_forward(self, x, mask, index_sample, out=out)
