"""GPU: the LeWin backward under torch.use_deterministic_algorithms(True).  Every parameter gradient is then a fixed-order sum
(per-unit partial slabs, one reduction launch per backward call), so repeated runs give the same bits; the data gradients
are the same as in the default (atomic) mode, the parameter gradients differ from it only by the order of the additions."""
import os

import numpy as np
import pytest
import torch

from oracle import lewin_oracle as O
from tests import test_gpu_block_backward as block_bwd
from tests.util import force_drop_scales

# torch's own cuBLAS calls (whole-model tests) refuse deterministic mode without a fixed workspace configuration
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

pytestmark = pytest.mark.gpu


@pytest.fixture
def deterministic():
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


def _block(C, nH, shift, drop, seed, mlp_ratio=4):
    import lewin_b200 as L
    rng = np.random.default_rng(seed)
    blk = L.LeWinTransformerBlock(dim=C, input_resolution=(128, 128), num_heads=nH, win_size=8, shift_size=shift,
                                  drop_path=0.25 if drop else 0., mlp_ratio=mlp_ratio)
    sd = blk.state_dict()
    if mlp_ratio == 4:
        for k, v in O.random_block_params(C, nH, rng, std=0.1).items():
            sd[k].copy_(torch.from_numpy(v))
    else:                                          # the oracle's parameter set is for mlp_ratio 4: seeded normal draws here
        for k, v in sd.items():
            if v.is_floating_point():
                v.copy_(torch.from_numpy(0.1 * rng.standard_normal(tuple(v.shape)).astype(np.float32)))
    return blk.to("cuda:0").eval(), rng


def _fwd_bwd(blk, x, dout, idx, mask=None, drop_scale=None):
    """forward + backward of one block from fresh gradient buffers -> (out, dx, {name: grad})"""
    blk.zero_grad(set_to_none=True)
    if drop_scale is not None:
        blk.train(True)
        force_drop_scales(blk, drop_scale, x.device)
    xs = x.detach().clone().requires_grad_(True)
    out = blk(xs, mask, idx)
    out.backward(dout)
    torch.cuda.synchronize()
    return out.detach(), xs.grad.detach(), {k: v.grad.detach().clone() for k, v in blk.named_parameters() if v.grad is not None}


def _inputs(blk, rng, C, hw, B, dtype, drop, masked):
    dev = torch.device("cuda:0")
    x = torch.from_numpy(rng.standard_normal((B, hw * hw, C)).astype(np.float32)).to(dev, dtype)
    dout = torch.from_numpy(rng.standard_normal((B, hw * hw, C)).astype(np.float32)).to(dev, dtype)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    drop_scale = None
    if drop:
        drop_scale = (rng.random((2, B)) < 0.75).astype(np.float32) / 0.75
        drop_scale[:, 0] = 1.0 / 0.75
    mask = None
    if masked:
        m = np.ones((B, 1, hw, hw), np.float32)
        m[:, :, hw // 4: 3 * hw // 4, : hw // 2] = 0.0
        mask = torch.from_numpy(m).to(dev)
    return x, dout, idx, drop_scale, mask


# (C, nH, hw, B, shift, drop, masked, mlp_ratio): every parameter-gradient reduction of the backward in both dtypes
#   C = 32 / 64 below 1024 tokens: the pipelined bf16 weight gradients (wg2); hw = 32: >= 1024 tokens, tcgen05 (wg3);
#   fp32: the generic weight-gradient kernel; C = 1024 fp32: the wide LayerNorm backward; 16 x 64 / 8 x 128 heads: the generic
#   core backward at head_dim 64 / 128 (head_dim 32 bf16: core_bwd_v2); the tiled depthwise weight gradient (W % 16 and W % 8);
#   mlp_ratio 3 at C = 32: hidden 96 is not a multiple of the bf16 tiled kernel's 64-channel slab, so bf16 runs the
#   register-window depthwise backward (dwconv_bwd_kernel: cleared slabs; fp32 at H % 8 != 0 in test_leff_dropin_off_grid)
CASES = [
    (32, 1, 8, 2, 0, False, False, 4), (32, 1, 32, 1, 4, False, False, 4), (64, 2, 24, 2, 4, False, False, 4),
    (64, 2, 32, 2, 4, True, False, 4), (128, 4, 16, 2, 4, False, True, 4), (128, 4, 32, 1, 0, False, False, 4),
    (256, 8, 16, 2, 4, True, False, 4), (512, 16, 8, 3, 0, False, False, 4), (1024, 16, 16, 1, 4, False, False, 4),
    (1024, 8, 8, 2, 0, False, False, 4), (64, 2, 16, 2, 4, False, True, 4),
    (32, 1, 16, 2, 4, False, False, 3), (32, 1, 40, 1, 4, True, False, 3),
]


def _grad_keys(blk):
    return sorted(k for k, _ in blk.named_parameters() if k in O.GRAD_KEYS)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C,nH,hw,B,shift,drop,masked,ratio", CASES)
def test_block_backward_is_reproducible(deterministic, dtype, C, nH, hw, B, shift, drop, masked, ratio):
    blk, rng = _block(C, nH, shift, drop, 4000 + C + hw, ratio)
    x, dout, idx, ds, mask = _inputs(blk, rng, C, hw, B, dtype, drop, masked)
    runs = [_fwd_bwd(blk, x, dout, idx, mask, ds) for _ in range(3)]
    assert sorted(runs[0][2]) == sorted(O.GRAD_KEYS) == _grad_keys(blk)
    for out, dx, g in runs[1:]:
        assert torch.equal(out, runs[0][0])
        assert torch.equal(dx, runs[0][1])
        for k in O.GRAD_KEYS:
            assert torch.equal(g[k], runs[0][2][k]), k


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C,nH,hw,B,shift,drop,masked,ratio", CASES)
def test_only_the_sum_order_changes(dtype, C, nH, hw, B, shift, drop, masked, ratio):
    """Default mode against deterministic mode: dx equal, parameter gradients within 1e-5 (fp32) / 1e-3 (bf16) relative L2."""
    blk, rng = _block(C, nH, shift, drop, 4000 + C + hw, ratio)
    x, dout, idx, ds, mask = _inputs(blk, rng, C, hw, B, dtype, drop, masked)
    assert not torch.are_deterministic_algorithms_enabled()
    out0, dx0, g0 = _fwd_bwd(blk, x, dout, idx, mask, ds)
    torch.use_deterministic_algorithms(True)
    try:
        out1, dx1, g1 = _fwd_bwd(blk, x, dout, idx, mask, ds)
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(out0, out1)
    assert torch.equal(dx0, dx1)
    tol = 1e-5 if dtype == torch.float32 else 1e-3
    for k in O.GRAD_KEYS:
        if k.endswith("key_projection.bias"):      # analytically zero: rounding noise only, compared on its weight's scale
            assert (g1[k] - g0[k]).abs().max() <= tol * g0[k.replace(".bias", ".weight")].abs().max() + 1e-30, k
            continue
        assert _rel_l2(g1[k], g0[k]) < tol, (k, _rel_l2(g1[k], g0[k]))


@pytest.mark.parametrize("C,nH,hw,B,shift", [(32, 1, 24, 2, 4), (256, 8, 16, 2, 4), (1024, 8, 8, 2, 0)])
def test_deterministic_block_backward_matches_oracle_f32(deterministic, C, nH, hw, B, shift):
    block_bwd.test_block_backward_matches_oracle_f32(C, nH, hw, B, shift)


@pytest.mark.parametrize("C,nH,hw,B,shift,drop", [(32, 1, 32, 1, 4, False), (128, 4, 32, 1, 4, False),
                                                  (256, 8, 16, 5, 4, True), (512, 16, 32, 1, 0, False)])
def test_deterministic_block_backward_bf16_close_to_oracle(deterministic, C, nH, hw, B, shift, drop):
    block_bwd.test_block_backward_bf16_close_to_oracle(C, nH, hw, B, shift, drop)


def _leff_grads(mlp, z, dz):
    mlp.zero_grad(set_to_none=True)
    zt = z.clone().requires_grad_(True)
    mlp(zt).backward(dz)
    torch.cuda.synchronize()
    return [zt.grad.clone()] + [p.grad.clone() for p in mlp.parameters()]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C,ratio,hw", [(32, 4, 12), (32, 3, 12), (64, 4, 20)])
def test_leff_dropin_off_grid(dtype, C, ratio, hw):
    """LeFF.forward on a map whose side is not a multiple of 8: the depthwise backward runs the register-window kernel
    (dwconv_bwd_kernel) in both dtypes.  Reproducible in deterministic mode; the input gradient equals the default mode's and
    the parameter gradients agree within 1e-5 (fp32) / 1e-3 (bf16) relative L2."""
    blk, rng = _block(C, 1, 0, False, 500 + C + hw, ratio)
    dev = torch.device("cuda:0")
    z = torch.from_numpy(rng.standard_normal((2, hw * hw, C)).astype(np.float32)).to(dev, dtype)
    dz = torch.from_numpy(rng.standard_normal((2, hw * hw, C)).astype(np.float32)).to(dev, dtype)
    g0 = _leff_grads(blk.mlp, z, dz)
    torch.use_deterministic_algorithms(True)
    try:
        g1, g2 = _leff_grads(blk.mlp, z, dz), _leff_grads(blk.mlp, z, dz)
    finally:
        torch.use_deterministic_algorithms(False)
    assert len(g1) == 7
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))
    assert torch.equal(g0[0], g1[0])
    tol = 1e-5 if dtype == torch.float32 else 1e-3
    for a, b in zip(g1[1:], g0[1:]):
        assert _rel_l2(a, b) < tol, _rel_l2(a, b)


def test_strict_dropin_dense_bias_is_reproducible(deterministic):
    """WindowAttention.forward with the gathered [nH, 64, 64] bias (d_rpb_dense slabs) and LeFF.forward (fused = 0)."""
    blk, rng = _block(64, 2, 4, False, 77)
    dev = torch.device("cuda:0")
    xw = torch.from_numpy(rng.standard_normal((24, 64, 64)).astype(np.float32)).to(dev)
    dyw = torch.from_numpy(rng.standard_normal((24, 64, 64)).astype(np.float32)).to(dev)
    mask = torch.from_numpy(np.where(rng.random((3, 64, 64)) < 0.2, -100.0, 0.0).astype(np.float32)).to(dev)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    z = torch.from_numpy(rng.standard_normal((2, 256, 64)).astype(np.float32)).to(dev)

    def run():
        blk.zero_grad(set_to_none=True)
        xt = xw.clone().requires_grad_(True)
        blk.attn(xt, mask=mask, index_sample=idx).backward(dyw)
        zt = z.clone().requires_grad_(True)
        blk.mlp(zt).backward(z)
        torch.cuda.synchronize()
        return [xt.grad.clone(), zt.grad.clone()] + [p.grad.clone() for p in blk.parameters() if p.grad is not None]

    a, b = run(), run()
    assert len(a) > 2
    assert all(torch.equal(u, v) for u, v in zip(a, b))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("nH,D,dense", [(2, 32, False), (2, 32, True), (4, 64, False), (2, 128, True)])
def test_core_backward_alone(dtype, nH, D, dense):
    """lewin_probsparse_core_bwd_*: reproducible in deterministic mode, dqkv equal to the default mode's, bias gradient close."""
    import lewin_b200.ops as ops
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(9 + D)
    B_, C = 48, nH * D
    qkv = torch.from_numpy(rng.standard_normal((B_, 64, 3 * C)).astype(np.float32)).to(dev, dtype)
    dctx = torch.from_numpy(rng.standard_normal((B_, 64, C)).astype(np.float32)).to(dev, dtype)
    idx = torch.from_numpy(rng.integers(0, 64, size=(64, 25)).astype(np.int64))
    bias = torch.from_numpy(0.1 * rng.standard_normal((nH, 64, 64) if dense else (225, nH)).astype(np.float32)).to(dev)

    def run():
        q = qkv.clone().requires_grad_(True)
        b = bias.clone().requires_grad_(True)
        kw = {"rpb_dense": b} if dense else {"rpb_table": b}
        ops.probsparse_core(q, num_heads=nH, index_sample=idx, **kw).backward(dctx)
        torch.cuda.synchronize()
        return q.grad.clone(), b.grad.clone()

    dq0, db0 = run()
    torch.use_deterministic_algorithms(True)
    try:
        dq1, db1 = run()
        dq2, db2 = run()
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(dq1, dq2) and torch.equal(db1, db2)
    assert torch.equal(dq0, dq1)
    assert _rel_l2(db1, db0) < 1e-5


def _uformer_grads(autocast):
    import lewin_b200 as L
    torch.manual_seed(0)
    model = L.Uformer(img_size=128, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff").to("cuda:0").train()
    gen = torch.Generator().manual_seed(1)
    x = torch.rand((2, 3, 128, 128), generator=gen).to("cuda:0").requires_grad_(True)
    idx = model.draw_index_samples()
    with torch.autocast("cuda", torch.bfloat16, enabled=autocast):
        y = model(x, index_samples=idx)
    y.float().square().mean().backward()
    torch.cuda.synchronize()
    return [x.grad.clone()] + [p.grad.clone() for p in model.parameters() if p.grad is not None]


@pytest.mark.parametrize("autocast", [False, True], ids=["f32", "bf16-autocast"])
def test_whole_model_gradients_are_reproducible(deterministic, autocast):
    a, b = _uformer_grads(autocast), _uformer_grads(autocast)
    assert len(a) == len(b) > 100
    for i, (u, v) in enumerate(zip(a, b)):
        assert torch.equal(u, v), i


def _train_step(graph):
    import lewin_b200 as L
    torch.manual_seed(0)
    model = L.Uformer(img_size=128, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff").to("cuda:0")
    torch.manual_seed(1)
    return L.training.TrainStep(model, batch_shape=(2, 3, 128, 128), contrast=False, graph=graph), model


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "eager"])
def test_train_step_is_reproducible(deterministic, graph):
    """Two TrainSteps built from the same seeds: after four steps on the same batches the losses and every parameter are
    equal.  (A graph TrainStep and an eager one are not compared with each other: the capture's warm-up steps update the
    parameters.)"""
    gen = torch.Generator().manual_seed(3)
    batches = [(torch.rand((2, 3, 128, 128), generator=gen), torch.rand((2, 3, 128, 128), generator=gen)) for _ in range(4)]
    out = []
    for _ in range(2):
        ts, model = _train_step(graph)
        losses = [ts.step(x.cuda(), y.cuda()).clone() for x, y in batches]
        torch.cuda.synchronize()
        assert ts.launch_mode.startswith("cuda-graph") == graph
        out.append((losses, [p.detach().clone() for p in model.parameters()]))
    (l0, p0), (l1, p1) = out
    assert all(torch.equal(a, b) for a, b in zip(l0, l1))
    assert all(torch.equal(a, b) for a, b in zip(p0, p1))


def test_train_step_refuses_a_changed_flag():
    ts, _ = _train_step(True)
    x = torch.rand((2, 3, 128, 128), device="cuda:0")
    ts.step(x, x)
    assert ts.launch_mode.startswith("cuda-graph")
    torch.use_deterministic_algorithms(True)
    try:
        with pytest.raises(RuntimeError, match="new TrainStep"):
            ts.step(x, x)
    finally:
        torch.use_deterministic_algorithms(False)


def test_default_mode_forward_is_reproducible():
    """With the flag off the forward is already deterministic (only the backward needed work)."""
    blk, rng = _block(128, 4, 4, False, 5)
    x, _, idx, _, _ = _inputs(blk, rng, 128, 32, 2, torch.bfloat16, False, False)
    with torch.no_grad():
        a, b = blk(x, None, idx), blk(x, None, idx)
    assert torch.equal(a, b)
    blk32, rng = _block(32, 1, 0, False, 6)
    x, _, idx, _, _ = _inputs(blk32, rng, 32, 32, 2, torch.float32, False, False)
    with torch.no_grad():
        assert torch.equal(blk32(x, None, idx), blk32(x, None, idx))
