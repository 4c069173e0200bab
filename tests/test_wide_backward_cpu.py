"""CPU: the backward entry points take rows of up to 1024 channels (embed_dim 64's bottleneck) and refuse wider ones, and the
differentiable whole-model port with forced selections (tests/port_forced.py, the reference side of the GPU gradient test) is
the pinned forward of oracle/torch_port.py."""
import os

import numpy as np
import pytest
import torch

LEWIN_E_SHAPE, LEWIN_E_WORKSPACE, LEWIN_E_ARCH = -2, -4, -6


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    if not os.path.isfile(g.LIB):
        g.build()
    from lewin_b200 import _lib
    return _lib.load()


def _attn_args(C, nH):
    from lewin_b200 import _lib
    a = _lib.LewinAttnBwdArgs()
    f = a.fwd
    f.B, f.H, f.W, f.C, f.nH, f.use_rpb = 1, 16, 16, C, nH, 1
    for n in ("x", "y", "ln_w", "ln_b", "w_qkv", "b_qkv", "w_out", "b_out", "rpb_table", "index_sample", "qkv", "ctx", "top"):
        setattr(f, n, 0x1000)
    for n in ("dy", "dx", "d_ln_w", "d_ln_b", "d_w_qkv", "d_b_qkv", "d_w_out", "d_b_out", "d_rpb_table"):
        setattr(a, n, 0x1000)
    return a


def _leff_args(C):
    from lewin_b200 import _lib
    a = _lib.LewinLeffBwdArgs()
    f = a.fwd
    f.B, f.H, f.W, f.C, f.hidden, f.fused, f.save_for_backward = 1, 16, 16, C, 4 * C, 1, 1
    for n in ("y", "out", "ln_w", "ln_b", "w1", "b1", "w_dw", "b_dw", "w2", "b2", "h1", "h2", "a1", "a2"):
        setattr(f, n, 0x1000)
    for n in ("dout", "dy", "d_ln_w", "d_ln_b", "d_w1", "d_b1", "d_w_dw", "d_b_dw", "d_w2", "d_b2"):
        setattr(a, n, 0x1000)
    return a


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_backward_abi_accepts_rows_of_up_to_1024_channels(lib, dtype):
    """C = 1024 (16 heads of 64, 8 heads of 128) passes the shape checks of both backward entries, like the forward's; the
    call then stops at the device lookup (no GPU) or the missing workspace.  C = 1056 is still refused."""
    attn = getattr(lib, f"lewin_attn_bwd_{dtype}")
    leff = getattr(lib, f"lewin_leff_bwd_{dtype}")
    for nH in (16, 8):
        rc = attn(_attn_args(1024, nH), None, 0, None)
        assert rc in (LEWIN_E_ARCH, LEWIN_E_WORKSPACE), (nH, rc)
    assert leff(_leff_args(1024), None, 0, None) in (LEWIN_E_ARCH, LEWIN_E_WORKSPACE)
    assert attn(_attn_args(1056, 33), None, 0, None) == LEWIN_E_SHAPE      # head_dim 32, C > 1024
    assert attn(_attn_args(1024, 32), None, 0, None) == LEWIN_E_SHAPE      # more than 16 heads
    assert leff(_leff_args(1056), None, 0, None) == LEWIN_E_SHAPE


def test_forced_selection_port_reproduces_uformer_forward(golden_dir):
    """tests.port_forced.uformer_forward_tops, with its own selections and forced with them, is torch_port.uformer_forward
    bit for bit on the embed_dim 64 recording's input, weights and key-sample draws."""
    import lewin_b200 as L
    from oracle import param_fill, torch_port
    from tests import port_forced
    z = np.load(os.path.join(golden_dir, "uformer64_b1.npz"))
    model = L.Uformer(img_size=128, embed_dim=64, win_size=8, token_projection="linear", token_mlp="leff")
    param_fill.fill_module(model, int(z["seed"]))
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    x = torch.from_numpy(z["x"])
    idx = torch.from_numpy(z["idx"].astype(np.int64))
    ref = torch_port.uformer_forward(x, sd, idx)
    rec = []
    with torch.no_grad():
        own = port_forced.uformer_forward_tops(x, sd, idx, record=rec)
        assert len(rec) == 18
        tops = [t.to(torch.uint8) for t in rec]               # the form ops.TopRecorder records
        out = port_forced.uformer_forward_tops(x, sd, idx, tops=tops)
    assert torch.equal(own, ref)
    assert torch.equal(out, ref)
