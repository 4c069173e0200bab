"""GPU: training at C = 1024, the bottleneck of the embed_dim 64 Uformer (`conv` and `decoderlayer_0`: 16 heads of 64).  Block
backward in fp32 and bf16 at the two C = 1024 head layouts (16 x 64, 8 x 128) with the gates of tests/test_gpu_block_backward.py;
the whole embed_dim 64 model's gradients against the fp64 torch port with the device's selections forced; TrainStep."""
import math
import os

import numpy as np
import pytest
import torch

from tests import test_gpu_block_backward as block_bwd

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("C,nH,hw,B,shift", [(1024, 16, 16, 1, 4), (1024, 8, 8, 2, 0)])
def test_wide_block_backward_matches_oracle_f32(C, nH, hw, B, shift):
    """dx and all 19 parameter gradients within 1e-3 of scale of the fp64 oracle (GPU selection forced); the fp32 LayerNorm
    backward of rows wider than 512 channels runs ln_bwd_wide_kernel."""
    block_bwd.test_block_backward_matches_oracle_f32(C, nH, hw, B, shift)


@pytest.mark.parametrize("C,nH,hw,B,shift,drop", [
    (1024, 16, 32, 1, 4, False),     # 1024 tokens: tcgen05 weight gradients (N = 3072 / 4096 / 1024, K = 1024 / 4096)
    (1024, 8, 16, 2, 0, False),      # 512 tokens: the pipelined bf16 weight-gradient fallback, 8 heads of 128
    (1024, 16, 16, 2, 4, True),      # DropPath scales on (scale_gather_rows pre-pass below 1024 tokens)
    (1024, 8, 32, 1, 4, True)])      # DropPath scales on with the tcgen05 weight gradients
def test_wide_block_backward_bf16_close_to_oracle(C, nH, hw, B, shift, drop):
    """Gates of test_block_backward_bf16_close_to_oracle: cosine > 0.995 and max error < 6e-2 of the reference's max for dx
    and every gradient, the analytically zero key bias within 6e-2 of its weight's gradient."""
    block_bwd.test_block_backward_bf16_close_to_oracle(C, nH, hw, B, shift, drop)


def _model64(golden_dir):
    import lewin_b200 as L
    from oracle import param_fill
    z = np.load(os.path.join(golden_dir, "uformer64_b1.npz"))
    model = L.Uformer(img_size=128, embed_dim=64, win_size=8, token_projection="linear", token_mlp="leff")
    param_fill.fill_module(model, int(z["seed"]))
    return model, z


def _device_grads(model, z, dout, autocast):
    """Gradients of <model(x), dout> on cuda:0 (eval mode, cuDNN TF32 off) and the selection of every LeWin block."""
    import lewin_b200 as L
    dev = torch.device("cuda:0")
    model = model.to(dev).eval()
    model.zero_grad(set_to_none=True)
    x = torch.from_numpy(z["x"]).to(dev).requires_grad_(True)
    idx = torch.from_numpy(z["idx"].astype(np.int64))
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with L.ops.TopRecorder() as rec, torch.autocast("cuda", torch.bfloat16, enabled=autocast):
            y = model(x, index_samples=idx)
        y.backward(torch.from_numpy(dout).to(dev, y.dtype))
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    grads = {n: p.grad.detach().double().cpu() for n, p in model.named_parameters() if p.grad is not None}
    grads["input"] = x.grad.detach().double().cpu()
    return grads, [t.cpu() for t in rec.tops]


def _port_grads(model, z, dout, tops):
    """The same gradients from the torch port's op sequence (tests/port_forced.py) in fp64 with the device's selections forced."""
    from tests import port_forced
    sd = {k: v.detach().cpu().double().requires_grad_() if v.is_floating_point() else v.detach().cpu()
          for k, v in model.state_dict().items()}
    x = torch.from_numpy(z["x"]).double().requires_grad_(True)
    out = port_forced.uformer_forward_tops(x, sd, torch.from_numpy(z["idx"].astype(np.int64)), tops=tops)
    out.backward(torch.from_numpy(dout).double())
    grads = {n: sd[n].grad for n, _ in model.named_parameters() if sd[n].grad is not None}
    grads["input"] = x.grad
    return grads


def _rel_l2(a, b):
    return float((a - b).norm() / b.norm())


def _cos(a, b):
    a, b = a.ravel(), b.ravel()
    return float(a @ b / (a.norm() * b.norm() + 1e-300))


def test_embed_dim_64_model_gradients_match_fp64_port(golden_dir):
    """Whole embed_dim 64 model (C = 64 ... 1024) on the uformer64_b1 input, weights and 18 key-sample draws, gradients of a fixed
    random cotangent.  fp32: every live parameter and the input within 1e-3 relative L2 of the fp64 port; the dead parameters
    get no gradient on either side; the key biases, analytically zero (the bias shifts every score of a row equally), stay
    below 1e-3 of their weight's gradient.  bf16 autocast: cosine >= 0.99 for every gradient of norm >= 1e-3 of the largest."""
    model, z = _model64(golden_dir)
    dout = np.random.default_rng(64).standard_normal(z["x"].shape).astype(np.float32)

    got, tops = _device_grads(model, z, dout, autocast=False)
    assert len(tops) == 18
    ref = _port_grads(model, z, dout, tops)
    assert sorted(got) == sorted(ref)                     # the same dead parameters on both sides
    worst = ("", 0.0)
    for n, r in ref.items():
        if n.endswith("key_projection.bias"):
            assert got[n].norm() < 1e-3 * got[n.replace(".bias", ".weight")].norm(), n
            continue
        e = _rel_l2(got[n], r)
        worst = max(worst, (n, e), key=lambda t: t[1])
        assert e <= 1e-3, (n, e)
    print(f"uformer64 fp32 gradients: worst relative L2 {worst[1]:.2e} ({worst[0]})")

    gotb, topsb = _device_grads(model, z, dout, autocast=True)
    refb = _port_grads(model, z, dout, topsb)
    assert sorted(gotb) == sorted(refb)
    big = max(float(r.norm()) for r in refb.values())
    worst = ("", 1.0)
    for n, r in refb.items():
        if float(r.norm()) < 1e-3 * big:
            continue
        c = _cos(gotb[n], r)
        worst = min(worst, (n, c), key=lambda t: t[1])
        assert c >= 0.99, (n, c)
    print(f"uformer64 bf16 gradients: worst cosine {worst[1]:.5f} ({worst[0]})")


def test_train_step_embed_dim_64_graph_and_eager_learn():
    """TrainStep on Uformer(embed_dim=64), CUDA-graph replay and eager: six steps on a fixed batch give finite, falling losses,
    and the dead parameters stay without gradient."""
    import copy
    import lewin_b200 as L
    from lewin_b200 import training, parallel
    dev = torch.device("cuda:0")
    torch.manual_seed(3)
    model = L.Uformer(img_size=128, embed_dim=64, win_size=8, token_projection="linear", token_mlp="leff").to(dev).train()
    model2 = copy.deepcopy(model)
    x = torch.rand(2, 3, 128, 128, device=dev)
    y = (x * 0.8 + 0.1)
    for name, mdl, graph in (("graph", model, True), ("eager", model2, False)):
        torch.manual_seed(11)
        ts = training.TrainStep(mdl, (2, 3, 128, 128), contrast=False, graph=graph, device=dev)
        seq = []
        for _ in range(6):
            ts.step(x, y)
            seq.append(ts.loss())
        print(f"embed_dim 64 TrainStep ({name}, {ts.launch_mode}): losses {seq}")
        assert ("cuda-graph" in ts.launch_mode) == graph
        assert all(math.isfinite(v) for v in seq) and seq[-1] < seq[0], seq
    dead = set(parallel.dead_parameter_names(model))
    assert len(dead) == 18 * 6
    for n, p in model.named_parameters():
        assert (p.grad is None) == (n in dead) or not p.requires_grad, n
