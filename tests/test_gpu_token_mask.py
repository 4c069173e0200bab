"""The input mask evaluated per token inside the attention kernels (LewinAttnFwdArgs::token_mask) against the dense
[B*nW, 64, 64] mask the reference builds (My_model_1.py:791-836, restated in tests/token_mask_ref.py and pinned to the numpy
oracle by tests/test_token_mask_cpu.py).  The kernels form the same fp32 values (0, -100, -200) and add them once at the same
point, so the two paths must agree BIT FOR BIT: outputs, selections and the data gradient.  Parameter gradients accumulate
with atomics in an unfixed order, so they are held to the run-to-run spread of the dense path against itself."""
import numpy as np
import pytest
import torch

from oracle import lewin_oracle as O
from tests.token_mask_ref import dense_from_token_mask, level_mask
from tests.util import load_fixture

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HW = 24                          # the inmask golden's level size (its mask is 48 x 48)


def _masks(Bm, rng):
    """Named input masks [Bm, 1, 48, 48]: the golden's, a centred rectangle and its complement, random binary, and
    non-binary values (0.5, negatives, 1e-30 whose pairwise products underflow to zero, one NaN)."""
    gold = torch.from_numpy(load_fixture("block_c64_h2_s4_inmask")["input_mask"]).float()
    rect = torch.zeros(1, 1, 48, 48)
    rect[..., 10:38, 6:42] = 1.0
    rnd = torch.from_numpy((rng.random((1, 1, 48, 48)) < 0.5).astype(np.float32))
    odd = torch.from_numpy(rng.choice(np.array([0.0, 0.5, -1.0, 1e-30, 1.0, -2.5], np.float32), size=(1, 1, 48, 48)))
    odd[..., 5, 7] = float("nan")
    out = {"golden": gold, "rect": rect, "rect_complement": 1.0 - rect, "random": rnd, "nonbinary": odd}
    # Bm = 2: the second image gets a different mask
    second = {"golden": 1.0 - gold, "rect": 1.0 - rect, "rect_complement": rect, "random": 1.0 - rnd, "nonbinary": odd.flip(-1)}
    return {k: (v if Bm == 1 else torch.cat([v, second[k]], 0)) for k, v in out.items()}


def _block(C, nH, shift, seed):
    import lewin_b200 as L
    rng = np.random.default_rng(seed)
    blk = L.LeWinTransformerBlock(dim=C, input_resolution=(128, 128), num_heads=nH, win_size=8, shift_size=shift)
    sd = blk.state_dict()
    for k, v in O.random_block_params(C, nH, rng).items():
        sd[k].copy_(torch.from_numpy(v))
    return blk.to(DEV), rng


def _attn_kw(blk, B, idx):
    w_qkv, b_qkv = blk.attn.ProbSpare.qkv_weights()
    return dict(B=B, H=HW, W=HW, num_heads=blk.num_heads, shift=blk.shift_size, ln_w=blk.norm1.weight, ln_b=blk.norm1.bias,
                w_qkv=w_qkv, b_qkv=b_qkv, w_out=blk.attn.ProbSpare.out_projection.weight,
                b_out=blk.attn.ProbSpare.out_projection.bias, rpb_table=blk.attn.relative_position_bias_table, index_sample=idx,
                return_top=True)


def _both(kw, mask, shift):
    """(token-mask kwargs, dense-mask kwargs) for an input mask [Bm, 1, h, w]."""
    tm = level_mask(mask.to(DEV), HW, HW)
    return dict(token_mask=tm, analytic_shift_mask=True), dict(mask=dense_from_token_mask(tm, shift), analytic_shift_mask=False)


CASES = [(32, 1), (64, 2), (64, 1), (128, 1)]         # head_dim 32 (C = 32, 64), 64 and 128


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shift", [0, 4])
@pytest.mark.parametrize("C,nH", CASES)
@pytest.mark.parametrize("Bm", [1, 2])
def test_token_mask_forward_equals_the_dense_mask(dtype, shift, C, nH, Bm):
    import lewin_b200 as L
    blk, rng = _block(C, nH, shift, seed=C + nH + shift + Bm)
    B = 2
    x = torch.from_numpy(rng.standard_normal((B, HW * HW, C)).astype(np.float32)).to(DEV, dtype)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    kw = _attn_kw(blk, B, idx)
    with torch.no_grad():
        for name, mask in _masks(Bm, rng).items():
            tok, dense = _both(kw, mask, shift)
            y_t, top_t = L.ops.lewin_attn(x, **kw, **tok)
            y_d, top_d = L.ops.lewin_attn(x, **kw, **dense)
            torch.cuda.synchronize()
            assert torch.equal(top_t, top_d), name
            assert torch.equal(y_t, y_d), (name, float((y_t.float() - y_d.float()).abs().max()))


def _grads(L, x, kw, extra, dy):
    xr = x.detach().clone().requires_grad_(True)
    params = [kw[k] for k in ("ln_w", "ln_b", "w_out", "b_out", "rpb_table")]
    for p in params:
        p.grad = None
    w_qkv = kw["w_qkv"].detach().clone().requires_grad_(True)
    y, top = L.ops.lewin_attn(xr, **{**kw, "w_qkv": w_qkv}, **extra)
    y.backward(dy)
    torch.cuda.synchronize()
    return y.detach(), top, xr.grad, [p.grad.clone() for p in params] + [w_qkv.grad]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shift", [0, 4])
@pytest.mark.parametrize("C,nH", CASES)
@pytest.mark.parametrize("Bm", [1, 2])
def test_token_mask_backward_equals_the_dense_mask(dtype, shift, C, nH, Bm):
    import lewin_b200 as L
    blk, rng = _block(C, nH, shift, seed=7 * C + nH + shift + Bm)
    B = 2
    x = torch.from_numpy(rng.standard_normal((B, HW * HW, C)).astype(np.float32)).to(DEV, dtype)
    dy = torch.from_numpy(rng.standard_normal((B, HW * HW, C)).astype(np.float32)).to(DEV, dtype)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    kw = _attn_kw(blk, B, idx)
    for name, mask in _masks(Bm, rng).items():
        tok, dense = _both(kw, mask, shift)
        y_t, top_t, dx_t, g_t = _grads(L, x, kw, tok, dy)
        y_d, top_d, dx_d, g_d = _grads(L, x, kw, dense, dy)
        _, _, dx_d2, g_d2 = _grads(L, x, kw, dense, dy)
        assert torch.equal(top_t, top_d) and torch.equal(y_t, y_d), name
        assert torch.equal(dx_t, dx_d) and torch.equal(dx_d2, dx_d), name
        for a, b, b2 in zip(g_t, g_d, g_d2):
            spread = float((b2 - b).abs().max())
            scale = float(b.abs().max())
            assert float((a - b).abs().max()) <= 2 * spread + 1e-6 * scale, (name, float((a - b).abs().max()), spread)


@pytest.mark.parametrize("C,nH", [(32, 1), (64, 2)])
@pytest.mark.parametrize("shift", [0, 4])
@pytest.mark.parametrize("Bm", [1, 2])
def test_masked_bf16_inference_runs_the_fused_kernel(C, nH, shift, Bm):
    """A masked bf16 inference call is the single fused kernel (one launch) and equals, bit for bit, the masked three-kernel
    path that a gradient-saving call takes."""
    import lewin_b200 as L
    from lewin_b200 import _lib
    lib = _lib.load()
    blk, rng = _block(C, nH, shift, seed=11 * C + shift + Bm)
    B = 2
    x = torch.from_numpy(rng.standard_normal((B, HW * HW, C)).astype(np.float32)).to(DEV, torch.bfloat16)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    kw = _attn_kw(blk, B, idx)
    for name, mask in _masks(Bm, rng).items():
        tok, _ = _both(kw, mask, shift)
        n0 = lib.lewin_launch_count()
        with torch.no_grad():
            y_f, top_f = L.ops.lewin_attn(x, **kw, **tok)
        n_fused = lib.lewin_launch_count() - n0
        n0 = lib.lewin_launch_count()
        y_u, top_u = L.ops.lewin_attn(x.detach().clone().requires_grad_(True), **kw, **tok)
        n_unfused = lib.lewin_launch_count() - n0
        torch.cuda.synchronize()
        assert (n_fused, n_unfused) == (1, 3), name
        assert torch.equal(top_f, top_u), name
        assert torch.equal(y_f, y_u.detach()), (name, float((y_f.float() - y_u.float()).abs().max()))


def _dense_attn(monkeypatch, L):
    """Every block's attention call gets the dense mask built from its token mask, as before the kernels evaluated it."""
    orig = L.ops.lewin_attn

    def dense_attn(x, **kw):
        tm = kw.pop("token_mask", None)
        if tm is not None:
            kw["mask"] = dense_from_token_mask(tm, kw["shift"])
            kw["analytic_shift_mask"] = False
        return orig(x, **kw)
    monkeypatch.setattr(L.ops, "lewin_attn", dense_attn)


def _canvas_mask(B, S, hw_list):
    m = torch.zeros(B, 1, S, S)
    for b, (h, w) in enumerate(hw_list[:B]):
        y0, x0 = (S - h) // 2, (S - w) // 2
        m[b, :, y0:y0 + h, x0:x0 + w] = 1.0
    return m


@pytest.mark.parametrize("embed_dim,S,B,dtype", [(32, 384, 1, torch.float32), (32, 384, 2, torch.float32),
                                                 (32, 384, 1, torch.bfloat16), (32, 384, 2, torch.bfloat16),
                                                 (64, 256, 1, torch.bfloat16)])
def test_whole_model_with_an_input_mask_equals_the_dense_mask(monkeypatch, embed_dim, S, B, dtype):
    """Uformer.forward(x, mask) on a canvas with a centred rectangle mask (B = 2: a mask per image) equals, bit for bit, the
    same model whose blocks are given the dense mask."""
    import lewin_b200 as L
    torch.manual_seed(embed_dim + S + B)
    model = L.Uformer(img_size=128, embed_dim=embed_dim, win_size=8, token_projection="linear", token_mlp="leff").to(DEV).eval()
    idx = model.draw_index_samples()
    x = torch.rand(B, 3, S, S, device=DEV)
    mask = _canvas_mask(B, S, [(200, 300), (300, 200)] if S == 384 else [(100, 150)]).to(DEV)
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        with torch.no_grad(), torch.autocast("cuda", torch.bfloat16, enabled=dtype == torch.bfloat16):
            y_t = model(x, mask, index_samples=idx).float()
            with monkeypatch.context() as mp:
                _dense_attn(mp, L)
                y_d = model(x, mask, index_samples=idx).float()
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.deterministic = det
    assert torch.isfinite(y_t).all()
    assert torch.equal(y_t, y_d), float((y_t - y_d).abs().max())
