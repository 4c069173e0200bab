"""Differentiable whole-model forward of oracle/torch_port.py with forced per-block top-u selections (test helper).

torch_port.uformer_forward runs under torch.no_grad and chooses every block's selection itself.  The gradient test of the
embed_dim 64 model needs the same op sequence with autograd on, in fp64, and with the device's selections (the form
ops.TopRecorder records) forced, so that near-tie queries chosen differently in fp32 / bf16 do not count as gradient error.
This module restates the port's op sequence with those two changes and reuses its helpers; tests/test_wide_backward_cpu.py
pins it to torch_port.uformer_forward bit for bit.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle.torch_port import STAGES, _partition, _rel_index, _reverse, _shift_mask


def prob_attention(q, k, v, rpb, mask, idx, top=None):     # torch_port.prob_attention; top [B, H, u] forced -> (ctx, top)
    B, L, H, D = q.shape
    q, k, v = q.transpose(2, 1), k.transpose(2, 1), v.transpose(2, 1)
    u = 25
    if top is None:
        k_exp = k.unsqueeze(-3).expand(B, H, L, L, D)
        k_sample = k_exp[:, :, torch.arange(L).unsqueeze(1), idx, :]
        qk_s = torch.matmul(q.unsqueeze(-2), k_sample.transpose(-2, -1)).squeeze(-2)
        M = qk_s.max(-1)[0] - torch.div(qk_s.sum(-1), L)
        top = M.topk(u, sorted=False)[1]
    bi, hi = torch.arange(B)[:, None, None], torch.arange(H)[None, :, None]
    s = torch.matmul(q[bi, hi, top, :], k.transpose(-2, -1)) * (1.0 / math.sqrt(D))
    ctx = v.mean(dim=-2).unsqueeze(-2).expand(B, H, L, D).clone()
    a = torch.softmax(s, dim=-1)
    a = a + rpb.unsqueeze(0).repeat(B, 1, 1, 1)[bi, hi, top, :]
    if mask is not None:
        nW = mask.shape[0]
        mm = mask.unsqueeze(1).unsqueeze(0).repeat(B // nW, 1, H, 1, 1)
        ti = top.unsqueeze(1).view(B // nW, nW, H, u)
        a = a.view(B // nW, nW, H, u, L) + mm[torch.arange(B // nW)[:, None, None, None],
                                               torch.arange(nW)[None, :, None, None],
                                               torch.arange(H)[None, None, :, None], ti, :]
        a = a.view(-1, H, u, L)
    a = torch.softmax(a, dim=-1)
    ctx[bi, hi, top, :] = torch.matmul(a, v)
    return ctx.transpose(2, 1).contiguous(), top


def lewin_block(x, p, shift, idx, top=None):               # torch_port.lewin_block -> (out, top)
    B, L, C = x.shape
    H = W = int(math.sqrt(L))
    nH = p["attn.relative_position_bias_table"].shape[1]
    mask = _shift_mask(H, W, 8, shift) if shift > 0 else None
    xn = F.layer_norm(x, (C,), p["norm1.weight"], p["norm1.bias"]).view(B, H, W, C)
    if shift > 0:
        xn = torch.roll(xn, shifts=(-shift, -shift), dims=(1, 2))
    xw = _partition(xn).view(-1, 64, C)
    rpb = p["attn.relative_position_bias_table"][_rel_index().view(-1)].view(64, 64, -1).permute(2, 0, 1).contiguous()
    pre = "attn.ProbSpare."
    x2 = xw.reshape(-1, C)
    q = F.linear(x2, p[pre + "query_projection.weight"], p[pre + "query_projection.bias"]).view(-1, 64, nH, C // nH)
    k = F.linear(x2, p[pre + "key_projection.weight"], p[pre + "key_projection.bias"]).view(-1, 64, nH, C // nH)
    v = F.linear(x2, p[pre + "value_projection.weight"], p[pre + "value_projection.bias"]).view(-1, 64, nH, C // nH)
    ctx, top = prob_attention(q, k, v, rpb, mask, idx, top)
    aw = F.linear(ctx.view(-1, C), p[pre + "out_projection.weight"], p[pre + "out_projection.bias"]).view(-1, 8, 8, C)
    sx = _reverse(aw, 8, H, W)
    if shift > 0:
        sx = torch.roll(sx, shifts=(shift, shift), dims=(1, 2))
    y = x + sx.view(B, L, C)
    z = F.layer_norm(y, (C,), p["norm2.weight"], p["norm2.bias"])
    h = F.gelu(F.linear(z.reshape(-1, C), p["mlp.linear1.0.weight"], p["mlp.linear1.0.bias"])).view(B, L, -1)
    h = h.view(B, H, W, -1).permute(0, 3, 1, 2)
    h = F.gelu(F.conv2d(h, p["mlp.dwconv.0.weight"], p["mlp.dwconv.0.bias"], padding=1, groups=h.shape[1]))
    h = h.permute(0, 2, 3, 1).reshape(B * L, -1)
    return y + F.linear(h, p["mlp.linear2.0.weight"], p["mlp.linear2.0.bias"]).view(B, L, C), top


def uformer_forward_tops(x, sd, idx, tops=None, record=None, depths=(2,) * 9, img_size=128, win=8):
    """torch_port.uformer_forward with autograd on (any float dtype).  tops: one selection per LeWin block in call order
    ([B_, nH, 25] integer tensors, e.g. ops.TopRecorder.tops) forced instead of the block's own top-u; record: a list that
    receives each block's selection."""
    it = iter(range(sum(depths)))

    def tok2img(t):
        B, L, C = t.shape
        H = int(math.sqrt(L))
        return t.transpose(1, 2).contiguous().view(B, C, H, H)

    def img2tok(t):
        return t.flatten(2).transpose(1, 2).contiguous()

    def stage(name, tok, res_div):
        for i in range(depths[STAGES.index(name)]):
            shift = 0 if (i % 2 == 0 or img_size // res_div <= win) else win // 2
            pre = f"{name}.blocks.{i}."
            p = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
            b = next(it)
            tok, top = lewin_block(tok, p, shift, idx[b], None if tops is None else tops[b].long())
            if record is not None:
                record.append(top)
        return tok

    y = F.leaky_relu(F.conv2d(x, sd["input_proj.proj.0.weight"], sd["input_proj.proj.0.bias"], padding=1), 0.01)
    tok = img2tok(y)
    skips = []
    for lvl in range(4):
        tok = stage(f"encoderlayer_{lvl}", tok, 2 ** lvl)
        skips.append(tok)
        tok = img2tok(F.conv2d(tok2img(tok), sd[f"dowsample_{lvl}.conv.0.weight"], sd[f"dowsample_{lvl}.conv.0.bias"],
                               stride=2, padding=1))
    tok = stage("conv", tok, 16)
    for lvl in range(4):
        up = F.conv_transpose2d(tok2img(tok), sd[f"upsample_{lvl}.deconv.0.weight"], sd[f"upsample_{lvl}.deconv.0.bias"],
                                stride=2)
        tok = torch.cat([img2tok(up), skips[3 - lvl]], -1)
        tok = stage(f"decoderlayer_{lvl}", tok, 2 ** (3 - lvl))
    y = F.conv2d(tok2img(tok), sd["output_proj.proj.0.weight"], sd["output_proj.proj.0.bias"], padding=1)
    return x + y
