"""Import the UNMODIFIED reference model (read-only, /root/reference) in the build container.

TEST INFRASTRUCTURE ONLY (see oracle/lewin_oracle.py header).  The reference source is not part
of this repository, so the package, the tests and the benchmark never import this module; only
``oracle/make_golden.py`` uses it, and the tests read the fixtures it wrote.

The reference needs ``timm.models.layers.{DropPath,to_2tuple,trunc_normal_}``
(My_model_1.py:10); timm is not installed, so an in-memory shim provides the three
symbols (SURVEY.md Appendix D).
"""
from __future__ import annotations

import os
import sys
import types

import torch
import torch.nn as nn

REF_ROOT = os.environ.get("REF_DIR", "/root/reference")
REF_PKG = os.path.join(REF_ROOT, "Uformer_ProbSparse")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_PKG, "My_model_1.py"))


class _DropPath(nn.Module):
    """timm.models.layers.DropPath: per-sample Bernoulli keep, scaled by 1/keep, identity in eval."""

    def __init__(self, drop_prob=0.0):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        shape = (x.shape[0],) + (1,) * (x.ndim - 1)
        mask = x.new_empty(shape).bernoulli_(keep)
        if keep > 0.0:
            mask.div_(keep)
        return x * mask


def _install_timm_shim():
    if "timm" in sys.modules:
        return
    timm = types.ModuleType("timm")
    models = types.ModuleType("timm.models")
    layers = types.ModuleType("timm.models.layers")
    layers.DropPath = _DropPath
    layers.to_2tuple = lambda x: x if isinstance(x, tuple) else (x, x)
    layers.trunc_normal_ = torch.nn.init.trunc_normal_
    timm.models = models
    models.layers = layers
    sys.modules["timm"] = timm
    sys.modules["timm.models"] = models
    sys.modules["timm.models.layers"] = layers


def import_reference():
    """Returns the reference's ``My_model_1`` module (and makes ``ProbSparse.attn``/``options`` importable)."""
    if not available():
        raise RuntimeError(f"reference tree not found under {REF_ROOT}")
    _install_timm_shim()
    sys.dont_write_bytecode = True          # the reference mount is read-only
    if REF_PKG not in sys.path:
        sys.path.insert(0, REF_PKG)
    import My_model_1  # noqa: E402
    return My_model_1


def block_params_numpy(block: nn.Module):
    """state_dict of one reference LeWinTransformerBlock -> {name: ndarray} (live + dead keys)."""
    return {k: v.detach().cpu().numpy() for k, v in block.state_dict().items()}
