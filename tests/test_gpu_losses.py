"""The contrastive loss's frozen VGG19 on this library's implicit-GEMM convolution (SURVEY 8(f) rank 1; My_CR.py:56-123):
lewin_conv3x3_fwd_bf16 (conv 3x3 / padding 1 + bias + ReLU on channel-last bf16 maps, tcgen05) forward and as the data gradient,
against torch's convolution on the same bf16-rounded operands, and ContrastLoss end to end against the cuDNN path."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("B,Cin,Cout,H,W", [(2, 64, 64, 32, 32), (1, 128, 256, 16, 16), (2, 512, 512, 8, 8), (1, 256, 512, 20, 24),
                                           (3, 64, 128, 128, 128)])
def test_conv3x3_relu_forward_and_data_gradient(B, Cin, Cout, H, W):
    from lewin_b200 import ops
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + Cin + Cout + H)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) * (2.0 / (9 * Cin)) ** 0.5).to(DEV)
    b = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    x = torch.randn(B, Cin, H, W, generator=g).to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    dy = torch.randn(B, Cout, H, W, generator=g).to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    assert ops.conv3x3_supported(x, Cin, Cout)
    fwd, bwd = ops.conv3x3_weight_images(w)
    xr = x.clone().requires_grad_(True)
    y = ops.conv3x3_relu(xr, fwd, bwd, b)
    assert y.dtype == torch.bfloat16 and y.is_contiguous(memory_format=torch.channels_last)
    y.backward(dy)
    # reference: fp32 convolution of the same bf16-rounded operands
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        xf = x.float().requires_grad_(True)
        yf = F.relu(F.conv2d(xf, w.to(torch.bfloat16).float(), b, padding=1))
        # the data gradient passes through the ReLU mask of the kernel's own output (elements at 0 +- a rounding may differ)
        (yf * 0).sum().backward()
        xf.grad = None
        mask = (y > 0).float()
        F.conv2d(xf, w.to(torch.bfloat16).float(), b, padding=1).backward(dy.float() * mask)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    scale = float(yf.abs().max())
    err = float((y.float() - yf).abs().max())
    assert err < 1.2e-2 * scale, (err, scale)                 # one bf16 ulp of the output scale
    gs = float(xf.grad.abs().max())
    gerr = float((xr.grad.float() - xf.grad).abs().max())
    cos = float(F.cosine_similarity(xr.grad.float().flatten(), xf.grad.flatten(), dim=0))
    assert gerr < 2e-2 * gs and cos > 0.9995, (gerr, gs, cos)


def test_contrast_loss_on_own_kernels_matches_the_cudnn_path(monkeypatch):
    from torch.profiler import profile, ProfilerActivity
    from lewin_b200.losses import ContrastLoss
    torch.manual_seed(0)
    crit = ContrastLoss(pretrained=False, device=torch.device(DEV))
    B = 4
    a0 = torch.rand(B, 3, 128, 128, device=DEV)
    p, n = torch.rand(B, 3, 128, 128, device=DEV), torch.rand(B, 3, 128, 128, device=DEV)

    def run():
        a = a0.clone().requires_grad_(True)
        with torch.autocast("cuda", torch.bfloat16):
            loss, ap, an = crit(a, p, n)
        loss.backward()
        return float(loss), float(ap), float(an), a.grad.clone()

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        l1, ap1, an1, g1 = run()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    n_own = sum("conv_igemm_kernel" in k for k in names)
    # features[0:30] hold 13 convolutions; all but the 3-channel conv1_1: 12 layers x (a pass + p|n pass) forward, 12 data gradients
    assert n_own == 12 * 2 + 12, n_own
    monkeypatch.setattr(crit.vgg, "_own_kernels", lambda X: False)      # the cuDNN path
    l2, ap2, an2, g2 = run()
    assert abs(l1 - l2) < 2e-2 * abs(l2) and abs(ap1 - ap2) < 2e-2 * abs(ap2) and abs(an1 - an2) < 2e-2 * abs(an2), (l1, l2)
    # the gradient of an L1 loss through 13 bf16 layers is noisy in either implementation (sign(fa - fp) flips wherever two
    # features agree to a bf16 ulp): judge both against the fp32 evaluation of the same loss
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        a = a0.clone().requires_grad_(True)
        loss, _, _ = crit(a, p, n)
        loss.backward()
        g_ref, l_ref = a.grad.clone(), float(loss)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    cos_own = float(F.cosine_similarity(g1.flatten(), g_ref.flatten(), dim=0))
    cos_cudnn = float(F.cosine_similarity(g2.flatten(), g_ref.flatten(), dim=0))
    print(f"loss fp32 {l_ref:.5f}, own {l1:.5f}, cuDNN bf16 {l2:.5f}; gradient cosine vs fp32: own {cos_own:.4f}, cuDNN bf16 {cos_cudnn:.4f}")
    assert abs(l1 - l_ref) < 2e-2 * abs(l_ref)
    assert cos_own > 0.85 and cos_own > cos_cudnn - 0.03, (cos_own, cos_cudnn)     # measured 0.897 for both bf16 paths
