"""The training iteration of My_train.py:212-310 as product API (SURVEY 8(f) rank 4: training-loop host overheads).

What the reference does per iteration, and what changes here (same arithmetic, same RNG consumption of the hot path):

  My_train.py:221   ``utils.MixUp_AUG().aug(target, input_)`` builds a new Beta(1.2, 1.2) distribution object and samples on the
                    CPU every step            -> `MixUp`: one persistent device-side sampler, no host round trip
  My_train.py:224   fp16 autocast + NativeScaler -> bf16 autocast (BASELINE config 2), no loss scaling needed
  My_train.py:227   DataParallel replicate + scatter per step -> one process per GPU, DDP (parallel.wrap_ddp)
  My_train.py:249   backward + optimizer.step as ~1500 separate launches -> forward + backward + AdamW captured ONCE as a CUDA
                    graph and replayed (single GPU); the 18 key-sample draws of attn.py:91 are still made on the CPU generator
                    every step and copied into the graph's static buffer
  My_train.py:250   ``loss.item()`` (device->host sync) every step -> the loss stays on the device; `TrainStep.loss()` syncs on demand
  My_train.py:258-310  validation 4x per epoch with per-image skimage PSNR / SSIM on the CPU -> `validate`: PSNR and SSIM
                    (Gaussian 11x11, sigma 1.5, the skimage/Wang et al. definition in its `gaussian_weights` form) on the device,
                    one sync at the end

`TrainStep` holds the model, optimizer and criteria; `step(input_, target)` is one iteration.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import parallel
from .losses import CharbonnierLoss, ContrastLoss


class MixUp:
    """utils/dataset_utils.py:41-63 (`MixUp_AUG.aug`): a random permutation of the batch blended in with per-sample weights
    lam ~ Beta(1.2, 1.2).  Device-side: the permutation and the Beta samples are drawn on the tensors' device by one
    persistent sampler (the reference constructs the distribution and samples on the host every iteration)."""

    def __init__(self, alpha=1.2, device=None):
        self.alpha = float(alpha)
        self._dist = None
        self._device = device

    def _sampler(self, device):
        if self._dist is None or self._device != device:
            a = torch.tensor([self.alpha], device=device)
            self._dist = torch.distributions.beta.Beta(a, a)
            self._device = device
        return self._dist

    def aug(self, rgb_gt, rgb_noisy):
        bs = rgb_gt.size(0)
        idx = torch.randperm(bs, device=rgb_gt.device)
        lam = self._sampler(rgb_gt.device).rsample((bs, 1)).view(-1, 1, 1, 1).to(rgb_gt.dtype)
        return lam * rgb_gt + (1 - lam) * rgb_gt[idx], lam * rgb_noisy + (1 - lam) * rgb_noisy[idx]


def batch_psnr(restored, target):
    """Per-image PSNR on [0, 1] images (skimage.metrics.peak_signal_noise_ratio with data_range 1, My_train.py:283): [B]."""
    mse = ((restored.float() - target.float()) ** 2).flatten(1).mean(1)
    return 10.0 * torch.log10(1.0 / mse.clamp_min(1e-20))


def _gauss_window(device, dtype, size=11, sigma=1.5):
    x = torch.arange(size, device=device, dtype=dtype) - (size - 1) / 2
    g = torch.exp(-(x * x) / (2 * sigma * sigma))
    g = g / g.sum()
    return (g[:, None] * g[None, :])


def batch_ssim(restored, target, data_range=1.0):
    """Per-image mean SSIM over channels with a Gaussian 11x11, sigma 1.5 window and K = (0.01, 0.03) (Wang et al. 2004; the
    structure of utils/image_utils.py:75-125): [B].  Computed on the device."""
    x, y = restored.float(), target.float()
    C = x.shape[1]
    w = _gauss_window(x.device, x.dtype).expand(C, 1, 11, 11).contiguous()
    mu_x, mu_y = F.conv2d(x, w, groups=C), F.conv2d(y, w, groups=C)
    sxx = F.conv2d(x * x, w, groups=C) - mu_x * mu_x
    syy = F.conv2d(y * y, w, groups=C) - mu_y * mu_y
    sxy = F.conv2d(x * y, w, groups=C) - mu_x * mu_y
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    s = ((2 * mu_x * mu_y + c1) * (2 * sxy + c2)) / ((mu_x * mu_x + mu_y * mu_y + c1) * (sxx + syy + c2))
    return s.flatten(1).mean(1)


@torch.no_grad()
def validate(model, batches, autocast_dtype=torch.bfloat16):
    """My_train.py:258-310 without the per-image host round trips: ``batches`` yields (target, input_) device tensors; returns
    (mean PSNR, mean SSIM, images) with ONE device->host sync."""
    was_training = model.training
    model.eval()
    psnr_sum = ssim_sum = None
    n = 0
    for target, input_ in batches:
        with torch.autocast("cuda", autocast_dtype, enabled=autocast_dtype is not None and input_.is_cuda):
            restored = model(input_)
        restored = torch.clamp(restored.float(), 0, 1)
        p, s = batch_psnr(restored, target).sum(), batch_ssim(restored, target).sum()
        psnr_sum = p if psnr_sum is None else psnr_sum + p
        ssim_sum = s if ssim_sum is None else ssim_sum + s
        n += restored.shape[0]
    model.train(was_training)
    if n == 0:
        return float("nan"), float("nan"), 0
    both = torch.stack([psnr_sum, ssim_sum]).cpu() / n
    return float(both[0]), float(both[1]), n


class TrainStep:
    """One training iteration of My_train.py:212-250 on the sm_100a LeWin ops.

        ts = TrainStep(model, batch_shape=(32, 3, 128, 128))        # AdamW(2e-4, wd 0.02), Charbonnier + VGG19 contrastive
        for target, input_ in loader:   ts.step(input_, target, epoch)
        print(ts.loss())                                            # one sync, when the caller wants the number

    graph=True (single GPU): forward + backward + optimizer are captured once and replayed; inputs are copied into static
    buffers and the 18 key-sample draws (attn.py:91, CPU generator) are refreshed before every replay.  Under an initialised
    torch.distributed process group the model is wrapped in DDP over NCCL (dead parameters frozen, parallel.wrap_ddp) and the
    step runs eagerly (DDP's bucketed all-reduce overlaps the backward)."""

    def __init__(self, model, batch_shape, lr=2e-4, weight_decay=0.02, autocast_dtype=torch.bfloat16, contrast=True,
                 contrast_loss=None, w_charbonnier=1.0, w_contrast=1.0, mixup_after_epoch=5, graph=True, device=None):
        import torch.distributed as dist
        self.model = model
        self.dev = device or next(model.parameters()).device
        self.autocast_dtype = autocast_dtype
        self.w_char, self.w_cr = float(w_charbonnier), float(w_contrast)
        self.mixup_after_epoch = mixup_after_epoch
        self.mixup = MixUp(device=self.dev)
        parallel.freeze_dead_parameters(model)
        self.distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self.net = parallel.wrap_ddp(model, self.dev) if self.distributed else model
        self.crit_char = CharbonnierLoss(eps=1e-3)
        self.crit_cr = None
        if contrast and self.w_cr > 0:
            self.crit_cr = contrast_loss if contrast_loss is not None else ContrastLoss(ablation=False, pretrained=False, device=self.dev)
        self.use_graph = bool(graph) and not self.distributed and self.dev.type == "cuda"
        params = [p for p in model.parameters() if p.requires_grad]
        # fused multi-tensor AdamW on the GPU (the foreach form costs 44 launches / 0.9 ms of a 19 ms step)
        self.opt = torch.optim.AdamW(params, lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay,
                                     capturable=self.use_graph, fused=self.dev.type == "cuda")
        self.x = torch.zeros(batch_shape, device=self.dev)           # static step inputs (graph replay reads these)
        self.y = torch.zeros(batch_shape, device=self.dev)
        self.idx = model.draw_index_samples().to(self.dev, dtype=torch.int32)
        self._loss = torch.zeros((), device=self.dev)
        self._graph = None
        self._graph_deterministic = None
        self.steps = 0

    # ---------------------------------------------------------------- pieces
    def _loss_fn(self):
        with torch.autocast("cuda", self.autocast_dtype, enabled=self.autocast_dtype is not None and self.dev.type == "cuda"):
            restored = torch.clamp(self.net(self.x, index_samples=self.idx), 0, 1)      # My_train.py:227-230
            loss = self.w_char * self.crit_char(restored.float(), self.y)               # :234
            if self.crit_cr is not None:
                loss = loss + self.w_cr * self.crit_cr(restored, self.y, self.x)[0]     # :236
        return loss

    def _eager(self):
        self.opt.zero_grad(set_to_none=True)
        loss = self._loss_fn()
        loss.backward()
        self.opt.step()
        return loss

    def _capture(self):
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for _ in range(3):                       # warm-up: lazy initialisations, cuDNN autotuning, optimizer state
                self._eager()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=True)
        with torch.cuda.graph(g):
            loss = self._loss_fn()
            loss.backward()
            self.opt.step()
            self._loss.copy_(loss.detach())
        self._graph = g
        self._graph_deterministic = torch.are_deterministic_algorithms_enabled()

    # ---------------------------------------------------------------- public
    def step(self, input_, target, epoch=0):
        """One iteration on device (or pinned-host) tensors ``input_`` (hazy) and ``target`` (clean), [B, 3, H, W] in [0, 1].

        A captured graph keeps the backward kernels of the torch.use_deterministic_algorithms setting it was captured under;
        if the setting has changed since, this raises instead of replaying them."""
        if self._graph is not None and torch.are_deterministic_algorithms_enabled() != self._graph_deterministic:
            raise RuntimeError(
                "TrainStep: torch.use_deterministic_algorithms changed since this step's CUDA graph was captured "
                f"(captured with {self._graph_deterministic}); a captured graph cannot switch its backward kernels. "
                "Build a new TrainStep after changing the setting.")
        input_ = input_.to(self.dev, non_blocking=True)
        target = target.to(self.dev, non_blocking=True)
        if self.mixup_after_epoch is not None and epoch > self.mixup_after_epoch:       # My_train.py:220-221
            target, input_ = self.mixup.aug(target, input_)
        self.x.copy_(input_, non_blocking=True)
        self.y.copy_(target, non_blocking=True)
        self.idx.copy_(self.model.draw_index_samples(), non_blocking=True)             # fresh CPU-generator draws, attn.py:91
        if self.use_graph:
            if self._graph is None:
                try:
                    self._capture()
                except Exception:                    # capture is an optimisation: fall back to the eager step
                    self.use_graph = False
                    self._graph = None
            if self._graph is not None:
                self._graph.replay()
                self.steps += 1
                return self._loss
        self._loss = self._eager().detach()
        self.steps += 1
        return self._loss

    def loss(self):
        """The last step's loss as a Python float (this is the device->host sync the reference pays every step)."""
        return float(self._loss.item())

    @property
    def launch_mode(self):
        return "cuda-graph (forward + backward + optimizer)" if self._graph is not None else ("ddp eager" if self.distributed else "eager")
