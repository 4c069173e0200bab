"""CPU: the input mask per token (LewinAttnFwdArgs::token_mask) - the ABI's refusals, the masked forward's kernel plan, tracing
of a masked block, and the frame rule the kernels implement (token map -> dense window mask) against the numpy oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import lewin_oracle as O
from tests.token_mask_ref import dense_from_token_mask, level_mask

LEWIN_E_SHAPE, LEWIN_E_ALIGN, LEWIN_E_WORKSPACE, LEWIN_E_ARCH = -2, -3, -4, -6
LEWIN_ATTN_K_FUSED = 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    if not os.path.isfile(g.LIB):
        g.build()
    from lewin_b200 import _lib
    return _lib.load()


def _fwd_args(C=32, nH=1, B=2, hw=32, shift=4):
    from lewin_b200 import _lib
    f = _lib.LewinAttnFwdArgs()
    f.B, f.H, f.W, f.C, f.nH, f.shift, f.use_rpb, f.analytic_shift_mask = B, hw, hw, C, nH, shift, 1, 1
    for n in ("x", "y", "ln_w", "ln_b", "w_qkv", "b_qkv", "w_out", "b_out", "rpb_table", "index_sample", "qkv", "ctx", "top"):
        setattr(f, n, 0x1000)
    f.token_mask, f.Bm = 0x2000, 1
    return f


def _bwd_args(**kw):
    from lewin_b200 import _lib
    a = _lib.LewinAttnBwdArgs()
    a.fwd = _fwd_args(**kw)
    a.fwd.save_for_backward = 1
    for n in ("dy", "dx", "d_ln_w", "d_ln_b", "d_w_qkv", "d_b_qkv", "d_w_out", "d_b_out", "d_rpb_table"):
        setattr(a, n, 0x1000)
    return a


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_token_mask_abi_refusals(lib, dtype):
    """token_mask with `windowed`, `band_mode` or the dense `mask`, or with Bm not dividing B, is LEWIN_E_SHAPE; a misaligned
    pointer is LEWIN_E_ALIGN.  A valid call passes the checks and stops at the device lookup (no GPU: LEWIN_E_ARCH or the CUDA
    runtime's error) or the missing workspace."""
    fwd = getattr(lib, f"lewin_attn_fwd_{dtype}")
    bwd = getattr(lib, f"lewin_attn_bwd_{dtype}")
    passes = lambda rc: rc > 0 or rc in (LEWIN_E_ARCH, LEWIN_E_WORKSPACE)

    def both(edit):
        f = _fwd_args()
        edit(f)
        b = _bwd_args()
        edit(b.fwd)
        return fwd(f, None, 0, None), bwd(b, None, 0, None)

    assert all(passes(rc) for rc in both(lambda f: None))
    assert all(passes(rc) for rc in both(lambda f: setattr(f, "Bm", 2)))
    fw = lambda f: (setattr(f, "windowed", 1), setattr(f, "shift", 0), setattr(f, "analytic_shift_mask", 0),
                    setattr(f, "ln_w", None), setattr(f, "ln_b", None))
    assert both(fw) == (LEWIN_E_SHAPE, LEWIN_E_SHAPE)
    assert both(lambda f: (setattr(f, "mask", 0x3000), setattr(f, "nW_mask", 16))) == (LEWIN_E_SHAPE, LEWIN_E_SHAPE)
    assert both(lambda f: setattr(f, "Bm", 3)) == (LEWIN_E_SHAPE, LEWIN_E_SHAPE)
    assert both(lambda f: setattr(f, "Bm", 0)) == (LEWIN_E_SHAPE, LEWIN_E_SHAPE)
    assert both(lambda f: setattr(f, "token_mask", 0x2004)) == (LEWIN_E_ALIGN, LEWIN_E_ALIGN)
    band = _fwd_args()
    band.band_mode, band.band_y0, band.band_Hg = 1, 0, 64
    assert fwd(band, None, 0, None) == LEWIN_E_SHAPE
    band.token_mask = None
    assert passes(fwd(band, None, 0, None))


@pytest.mark.parametrize("C,shift", [(32, 0), (32, 4), (64, 0), (64, 4)])
def test_masked_bf16_inference_plans_the_fused_kernel(lib, C, shift):
    """A masked bf16 inference call at C <= 64 runs as the single fused kernel, like an unmasked one; fp32, a gradient-saving
    call and the dense mask keep the three-kernel pipeline."""
    f = _fwd_args(C=C, nH=C // 32, shift=shift)
    assert lib.lewin_attn_fwd_kernel_mask(f, 1) == 1 << LEWIN_ATTN_K_FUSED
    assert lib.lewin_attn_fwd_kernel_mask(f, 0) & (1 << LEWIN_ATTN_K_FUSED) == 0
    f.save_for_backward = 1
    assert lib.lewin_attn_fwd_kernel_mask(f, 1) & (1 << LEWIN_ATTN_K_FUSED) == 0
    f.save_for_backward, f.token_mask, f.Bm, f.mask, f.nW_mask = 0, None, 0, 0x3000, 16
    assert lib.lewin_attn_fwd_kernel_mask(f, 1) & (1 << LEWIN_ATTN_K_FUSED) == 0


@pytest.mark.parametrize("shift", [0, 4])
def test_compile_ops_trace_a_masked_block(shift):
    """torch.compile of a LeWinTransformerBlock called with an input mask, on meta tensors: the token mask rides through
    torch.ops.lewin_b200.attn_fwd / attn_bwd as their optional trailing argument (fake implementations included), the graph
    has no break and one node per half, and every live parameter receives a gradient."""
    import torch._dynamo
    from torch._dynamo.utils import counters
    import lewin_b200 as L
    blk = L.LeWinTransformerBlock(dim=64, input_resolution=(16, 16), num_heads=2, win_size=8, shift_size=shift).to("meta")
    idx = torch.randint(64, (64, 25))
    x = torch.empty(2, 256, 64, device="meta", requires_grad=True)
    mask = torch.empty(2, 1, 37, 41, device="meta")
    graphs = []

    def backend(gm, example_inputs):
        graphs.append([str(n.target) for n in gm.graph.nodes if n.op == "call_function"])
        return gm.forward

    torch._dynamo.reset()
    counters.clear()
    out = torch.compile(blk, backend=backend)(x, mask, idx)
    assert len(graphs) == 1 and not dict(counters["graph_break"]), (graphs, dict(counters["graph_break"]))
    assert sum("lewin_b200.attn_fwd" in t for t in graphs[0]) == 1 and sum("lewin_b200.leff_fwd" in t for t in graphs[0]) == 1
    assert any("interpolate" in t or "upsample" in t for t in graphs[0]), graphs[0]
    out.backward(torch.empty_like(out))
    assert x.grad is not None and sum(p.grad is not None for p in blk.parameters()) == 19
    torch._dynamo.reset()


@pytest.mark.parametrize("hw,img,shift", [(24, (37, 53), 0), (24, (37, 53), 4), (40, (17, 91), 4), (16, (16, 16), 4)])
def test_token_map_restatement_equals_the_oracle_masks(hw, img, shift):
    """The frame rule of the kernels: window (wy, wx) row r takes m[8 wy + r / 8, 8 wx + r % 8] of the nearest-resized mask (the
    unshifted frame), the pair term is -100 where m_i * m_j != 0, and the shift mask is added: the torch restatement equals
    lewin_oracle.input_attn_mask + shift_attn_mask on odd source sizes, for both shifts."""
    rng = np.random.default_rng(hw + shift + img[0])
    src = (rng.random((1, 1) + img) < 0.5).astype(np.float32)
    src[0, 0, rng.random(img) < 0.1] = 0.5
    got = dense_from_token_mask(level_mask(torch.from_numpy(src), hw, hw), shift).numpy()
    ref = O.input_attn_mask(src, hw, hw, 8)
    if shift > 0:
        ref = ref + O.shift_attn_mask(hw, hw, 8, shift)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref)
