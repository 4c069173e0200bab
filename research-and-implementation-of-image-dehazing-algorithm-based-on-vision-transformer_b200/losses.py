"""Training losses of the reference step (SURVEY section 8(f) rank 1): CharbonnierLoss (losses.py:41-52) and the VGG19
contrastive regulariser ContrastLoss (My_CR.py:56-123, called at My_train.py:236).

Same constructor arguments, forward signatures and return values as the reference classes, so `criterion[0]`,
`criterion[1]` of My_train.py:144-147 can be swapped for these.  The arithmetic is the reference's:

    loss = sum_i w_i * L1(vgg_i(a), vgg_i(p)) / (L1(vgg_i(a), vgg_i(n)) + 1e-7),  w = (1/32, 1/16, 1/8, 1/4, 1)

over the five feature maps relu1_1, relu2_1, relu3_1, relu4_1, relu5_1 of a frozen VGG19 (`features[0:30]` cut at the same
five indices as My_CR.py:62-76).  What changes is how the three VGG passes are run on a B200:
  * the positive and the negative image are constants of the step (the reference builds their autograd graphs and then
    `.detach()`es the results, My_CR.py:112,115): they run under `no_grad`, as ONE batched pass of 2B images;
  * the network is kept channels-last, so under autocast every convolution is a bf16 NHWC implicit GEMM on the tensor
    cores without layout transposes;
  * all shapes are static, so the loss is CUDA-graph capturable together with the model's step (scripts/train_step.py).
On the GPU under bf16 autocast 12 of the 13 convolutions of `features[0:30]` (+ their ReLUs) run on this library's implicit-GEMM tcgen05 kernel
(`lewin_conv3x3_fwd_bf16`), forward and data gradient (the VGG weights are frozen: no weight gradient); the 3-channel conv1_1
and the max-pools stay on torch.  Elsewhere (CPU, fp32, trainable VGG) the stock modules run.
"""
from __future__ import annotations

import torch
import torch.nn as nn

VGG_CUTS = (2, 7, 12, 21, 30)          # My_CR.py:68-77: slices [0,2) [2,7) [7,12) [12,21) [21,30)


class CharbonnierLoss(nn.Module):
    """mean(sqrt((x - y)^2 + eps^2)) (losses.py:41-52)."""

    def __init__(self, eps=1e-3):
        super().__init__()
        self.eps = eps

    def forward(self, x, y):
        diff = x - y
        return torch.mean(torch.sqrt(diff * diff + self.eps * self.eps))


class Vgg19(nn.Module):
    """The five feature slices of torchvision's VGG19 (My_CR.py:56-92).  `pretrained=True` is the reference's behaviour
    and needs the torchvision weight file in the local cache (no network here); `pretrained=False` builds the same
    architecture with torchvision's seeded random init (synthetic throughput runs and the parity fixtures)."""

    def __init__(self, requires_grad=False, pretrained=True):
        super().__init__()
        from torchvision import models
        feats = models.vgg19(weights=models.VGG19_Weights.IMAGENET1K_V1 if pretrained else None).features
        lo = 0
        for i, hi in enumerate(VGG_CUTS, 1):
            seq = nn.Sequential()
            for k in range(lo, hi):
                seq.add_module(str(k), feats[k])       # same child names as the reference => same state_dict keys
            setattr(self, f"slice{i}", seq)
            lo = hi
        if not requires_grad:
            for p in self.parameters():
                p.requires_grad = False

    def forward(self, X):
        if self._own_kernels(X):
            return self._forward_own(X)
        h1 = self.slice1(X)
        h2 = self.slice2(h1)
        h3 = self.slice3(h2)
        h4 = self.slice4(h3)
        h5 = self.slice5(h4)
        return [h1, h2, h3, h4, h5]

    # ---- B200 path: every conv + ReLU pair with Cin >= 64 (12 of the 13) as one implicit-GEMM tcgen05 kernel, forward and data
    #      gradient (ops.conv3x3_relu -> lewin_conv3x3_fwd_bf16); conv1_1 (3 input channels) and the max-pools stay on torch
    def _own_kernels(self, X):
        if not X.is_cuda:
            return False
        if any(p.requires_grad for p in self.parameters()):
            return False                                  # the kernel path has no weight gradient (the reference freezes VGG too)
        return torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16 and X.shape[-1] % 128 == 0

    def _images(self, conv):
        from . import ops
        cache = self.__dict__.setdefault("_w_images", {})
        key = id(conv)
        ent = cache.get(key)
        if ent is None or ent[0] != conv.weight._version or ent[1].device != conv.weight.device:
            fwd, bwd = ops.conv3x3_weight_images(conv.weight)
            ent = (conv.weight._version, fwd, bwd)
            cache[key] = ent
        return ent[1], ent[2]

    def _forward_own(self, X):
        from . import ops
        outs = []
        h = X
        for sl in (self.slice1, self.slice2, self.slice3, self.slice4, self.slice5):
            mods = list(sl.children())
            i = 0
            while i < len(mods):
                m = mods[i]
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                if isinstance(m, nn.Conv2d) and isinstance(nxt, nn.ReLU) and m.kernel_size == (3, 3) and m.padding == (1, 1) and \
                        m.stride == (1, 1) and h.dtype == torch.bfloat16 and ops.conv3x3_supported(h, m.in_channels, m.out_channels):
                    fwd, bwd = self._images(m)
                    h = ops.conv3x3_relu(h, fwd, bwd, m.bias)
                    i += 2
                    continue
                h = m(h)
                if isinstance(m, nn.ReLU) or isinstance(m, nn.MaxPool2d) or isinstance(m, nn.Conv2d):
                    if h.dim() == 4 and not h.is_contiguous(memory_format=torch.channels_last):
                        h = h.contiguous(memory_format=torch.channels_last)
                i += 1
            outs.append(h)
        return outs


class ContrastLoss(nn.Module):
    """ContrastLoss(ablation) -> forward(a, p, n) = (loss, all_ap, all_an)  (My_CR.py:95-123).

    a: restored (carries the gradient), p: clear target, n: hazy input."""

    def __init__(self, ablation=False, pretrained=True, device=None):
        super().__init__()
        self.vgg = Vgg19(pretrained=pretrained)
        if device is not None:
            self.vgg = self.vgg.to(device)
        self.vgg = self.vgg.to(memory_format=torch.channels_last).eval()
        self.weights = [1.0 / 32, 1.0 / 16, 1.0 / 8, 1.0 / 4, 1.0]
        self.ab = ablation

    def forward(self, a, p, n):
        B = a.shape[0]
        a_vgg = self.vgg(a.contiguous(memory_format=torch.channels_last))
        with torch.no_grad():
            const = p if self.ab else torch.cat([p, n], 0)
            pn_vgg = self.vgg(const.contiguous(memory_format=torch.channels_last))
        loss = 0
        all_ap, all_an = 0, 0
        for i in range(len(a_vgg)):
            fa = a_vgg[i]
            d_ap = torch.nn.functional.l1_loss(fa, pn_vgg[i][:B])
            all_ap = all_ap + d_ap
            if not self.ab:
                d_an = torch.nn.functional.l1_loss(fa, pn_vgg[i][B:])
                all_an = all_an + d_an
                contrastive = d_ap / (d_an + 1e-7)
            else:
                contrastive = d_ap
            loss = loss + self.weights[i] * contrastive
        return loss, all_ap, all_an
