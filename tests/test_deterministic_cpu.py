"""CPU: the deterministic-mode ABI (version 7) - the `deterministic` fields, the workspace arithmetic of the partial slabs (host
arithmetic, no device involved), the Python layer mapping torch.use_deterministic_algorithms onto the field, and tracing."""
import contextlib
import os
import types

import pytest
import torch

from tests import test_gpu_deterministic as gpu_det


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    if not os.path.isfile(g.LIB):
        g.build()
    from lewin_b200 import _lib
    return _lib.load()


@pytest.fixture
def deterministic():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def test_abi_version_and_field_offsets(lib):
    from lewin_b200 import _lib
    assert lib.lewin_abi_version() == 7 == _lib.ABI_VERSION
    for cls, last in ((_lib.LewinAttnBwdArgs, "d_rpb_dense"), (_lib.LewinLeffBwdArgs, "d_b2"), (_lib.LewinCoreBwdArgs, "d_rpb_dense")):
        assert cls.deterministic.offset == getattr(cls, last).offset + 8, cls       # right after the last gradient pointer
        assert cls.deterministic.size == 4


def _attn(B, hw, C, nH, shift=4, windowed=0, dense=False):
    from lewin_b200 import _lib
    f = _lib.LewinAttnFwdArgs(B=B, H=hw, W=hw, C=C, nH=nH, shift=shift, windowed=windowed, use_rpb=1, analytic_shift_mask=1,
                              save_for_backward=1)
    if dense:
        f.rpb_dense = 0x1000
    else:
        f.rpb_table = 0x1000
    return _lib.LewinAttnBwdArgs(fwd=f, d_ln_w=0x1000, d_ln_b=0x1000, d_w_qkv=0x1000, d_b_qkv=0x1000, d_w_out=0x1000,
                                 d_b_out=0x1000, d_rpb_table=0 if dense else 0x1000, d_rpb_dense=0x1000 if dense else 0)


def _leff(B, hw, C, fused=1):
    from lewin_b200 import _lib
    f = _lib.LewinLeffFwdArgs(B=B, H=hw, W=hw, C=C, hidden=4 * C, fused=fused, save_for_backward=1)
    return _lib.LewinLeffBwdArgs(fwd=f, d_ln_w=0x1000, d_ln_b=0x1000, d_w1=0x1000, d_b1=0x1000, d_w_dw=0x1000, d_b_dw=0x1000,
                                 d_w2=0x1000, d_b2=0x1000)


def _core(B_, nH, D, dense=False):
    from lewin_b200 import _lib
    f = _lib.LewinCoreFwdArgs(B_=B_, nH=nH, use_rpb=1, head_dim=D)
    if dense:
        f.rpb_dense = 0x1000
    else:
        f.rpb_table = 0x1000
    return _lib.LewinCoreBwdArgs(fwd=f, d_rpb_table=0 if dense else 0x1000, d_rpb_dense=0x1000 if dense else 0)


def _grad_floats(C, hidden, nH, windowed=False, dense=False):
    return (4 * C * C + 4 * C + (0 if windowed else 2 * C) + (nH * 4096 if dense else 225 * nH), 2 * C * hidden + 11 * hidden + C + 2 * C)


# the batch-32 training shapes of bench.py's block microbenchmark (nine levels) for embed_dim 32 and 64, and the GPU file's
TRAIN_SHAPES = [(32, hw, k * C, k * C // 32) for C, hw in ((32, 128), (64, 64), (128, 32), (256, 16), (512, 8),
                                                          (512, 16), (256, 32), (128, 64), (64, 128)) for k in (1, 2)]
GPU_SHAPES = [(B, hw, C, nH) for C, nH, hw, B, *_ in gpu_det.CASES] + [(2, 24, 32, 1), (5, 16, 256, 8), (1, 32, 512, 16)]


@pytest.mark.parametrize("dtype", [0, 1], ids=["f32", "bf16"])
@pytest.mark.parametrize("B,hw,C,nH", TRAIN_SHAPES + GPU_SHAPES)
def test_workspace_grows_by_the_slabs(lib, dtype, B, hw, C, nH):
    """deterministic = 1 asks for more workspace than 0 (at least one slab of every parameter gradient), without a device."""
    a = _attn(B, hw, C, nH)
    base = lib.lewin_attn_bwd_workspace_bytes(a, dtype)
    a.deterministic = 1
    det = lib.lewin_attn_bwd_workspace_bytes(a, dtype)
    attn_floats, leff_floats = _grad_floats(C, 4 * C, nH)
    assert det >= base + 4 * attn_floats
    l = _leff(B, hw, C)
    base = lib.lewin_leff_bwd_workspace_bytes(l, dtype)
    l.deterministic = 1
    assert lib.lewin_leff_bwd_workspace_bytes(l, dtype) >= base + 4 * leff_floats
    c = _core(B * (hw // 8) ** 2, nH, C // nH)
    assert lib.lewin_probsparse_core_bwd_workspace_bytes(c, dtype) == 0
    c.deterministic = 1
    assert lib.lewin_probsparse_core_bwd_workspace_bytes(c, dtype) >= 4 * 225 * nH


def _align(n):
    return (n + 255) // 256 * 256


@pytest.mark.parametrize("dtype,hw,hidden", [(0, 12, 96), (1, 12, 96), (1, 16, 96), (0, 12, 128)])
def test_workspace_of_the_register_window_depthwise_backward(lib, dtype, hw, hidden):
    """LeFF shapes the tiled depthwise kernels do not serve (H % 8 != 0, or bf16 with hidden % 64 != 0) run dwconv_bwd_kernel,
    whose slab count is its grid for 148 SMs: min(148 * 8, B * ceil(hidden / 128) * ceil(W / 8) * ceil(H / 16)).  The slabs of
    the call, slot by slot: linear2 (2 token splits of 288 / 512 tokens), the depthwise weight and bias, linear1, LayerNorm."""
    from lewin_b200 import _lib
    B, C = 2, 32
    f = _lib.LewinLeffFwdArgs(B=B, H=hw, W=hw, C=C, hidden=hidden, fused=1, save_for_backward=1)
    l = _lib.LewinLeffBwdArgs(fwd=f)
    base = lib.lewin_leff_bwd_workspace_bytes(l, dtype)
    l.deterministic = 1
    tokens = B * hw * hw
    splits = 2                                                   # ceil(tokens / 256) caps the weight-gradient splits
    dw_slots = B * -(-hidden // 128) * -(-hw // 8) * -(-hw // 16)
    lanes = {0: 8, 1: 4}[dtype]                                  # ln_bwd_kernel lanes per row at C = 32
    ln_slots = -(-tokens // (8 * (32 // lanes)))
    slabs = [splits * C * hidden, splits * C, dw_slots * hidden * 9, dw_slots * hidden, splits * hidden * C, splits * hidden,
             ln_slots * C, ln_slots * C]
    assert lib.lewin_leff_bwd_workspace_bytes(l, dtype) - base == sum(_align(4 * n) for n in slabs)


@pytest.mark.parametrize("dtype", [0, 1], ids=["f32", "bf16"])
def test_workspace_of_the_dense_bias_and_drop_in_surfaces(lib, dtype):
    a = _attn(1, 16, 64, 2, shift=0, windowed=1, dense=True)
    base = lib.lewin_attn_bwd_workspace_bytes(a, dtype)
    a.deterministic = 1
    assert lib.lewin_attn_bwd_workspace_bytes(a, dtype) >= base + 4 * _grad_floats(64, 256, 2, windowed=True, dense=True)[0]
    c = _core(48, 2, 128, dense=True)
    c.deterministic = 1
    assert lib.lewin_probsparse_core_bwd_workspace_bytes(c, dtype) >= 4 * 2 * 4096
    l = _leff(2, 16, 64, fused=0)
    l.deterministic = 1
    assert lib.lewin_leff_bwd_workspace_bytes(l, dtype) > 0


def test_largest_training_workspace_is_bounded(lib):
    """The slabs at the batch-32 training shapes stay far below the activations a training step already holds."""
    worst = 0
    for B, hw, C, nH in TRAIN_SHAPES:
        for dt in (0, 1):
            a, l = _attn(B, hw, C, nH), _leff(B, hw, C)
            b0 = lib.lewin_attn_bwd_workspace_bytes(a, dt) + lib.lewin_leff_bwd_workspace_bytes(l, dt)
            a.deterministic = l.deterministic = 1
            worst = max(worst, lib.lewin_attn_bwd_workspace_bytes(a, dt) + lib.lewin_leff_bwd_workspace_bytes(l, dt) - b0)
    assert worst < 256 << 20, worst


class _Recorder:
    """Stand-in for the loaded library: records the argument structs of the backward calls, launches nothing."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if name.endswith("_workspace_bytes"):
            return lambda a, dt: 0
        if "_bwd_" in name:
            def call(a, ws, n, stream):
                self.calls.append((name, a.deterministic))
                return 0
            return call
        raise AttributeError(name)


@pytest.fixture
def recorder(monkeypatch):
    import lewin_b200.ops as ops
    from lewin_b200 import _lib
    rec = _Recorder()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(ops, "_stream", lambda: None)
    monkeypatch.setattr(ops, "_dtype_tag", lambda x: "f32")
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    return rec


def _run_backwards():
    import lewin_b200.ops as ops
    C, nH, B, hw = 32, 1, 1, 8
    T = B * hw * hw
    t = lambda *s: torch.zeros(*s)
    attn_saved = (t(T, C), t(C), t(C), t(3 * C, C), t(3 * C), t(C, C), t(C), t(225, nH), None, t(64, 25).int(), None, None,
                  t(T, 3 * C), t(T, C), torch.zeros(T // 64, nH, 25, dtype=torch.uint8), None)
    ops._attn_backward(attn_saved, (B, hw, hw, nH, 0, False, True, True, None), t(T, C))
    leff_saved = (t(T, C), t(C), t(C), t(4 * C, C), t(4 * C), t(4 * C, 1, 3, 3), t(4 * C), t(C, 4 * C), t(C), None,
                  t(T, 4 * C), t(T, 4 * C), t(T, 4 * C), t(T, 4 * C))
    ops._leff_backward(leff_saved, (B, hw, hw, True, None), t(T, C))
    ctx = types.SimpleNamespace(saved_tensors=(t(1, 64, 3 * C), t(225, nH), None, None, torch.zeros(1, nH, 25, dtype=torch.uint8)),
                                geom=(nH, True), dt="f32")
    ops._CoreFn.backward(ctx, t(1, 64, C), None)


def test_python_backward_passes_the_flag(recorder):
    _run_backwards()
    assert [d for _, d in recorder.calls] == [0, 0, 0]
    recorder.calls.clear()
    torch.use_deterministic_algorithms(True, warn_only=True)        # warn_only too: the library has the deterministic kernels
    try:
        _run_backwards()
    finally:
        torch.use_deterministic_algorithms(False)
    assert [n for n, _ in recorder.calls] == ["lewin_attn_bwd_f32", "lewin_leff_bwd_f32", "lewin_probsparse_core_bwd_f32"]
    assert [d for _, d in recorder.calls] == [1, 1, 1]


def test_compiled_block_traces_on_meta_under_the_flag(deterministic):
    """The torch.library ops need no new argument (the implementation reads the flag when it runs): a compiled block still
    traces on meta tensors, forward and backward."""
    import torch._dynamo
    import lewin_b200 as L
    blk = L.LeWinTransformerBlock(dim=64, input_resolution=(16, 16), num_heads=2, win_size=8, shift_size=4).to("meta")
    x = torch.empty(2, 256, 64, device="meta", requires_grad=True)
    torch._dynamo.reset()
    out = torch.compile(blk, backend="eager")(x, None, torch.randint(64, (64, 25)))
    out.backward(torch.empty_like(out))
    assert x.grad is not None and sum(p.grad is not None for p in blk.parameters()) == 19
    torch._dynamo.reset()
