"""CPU: the C-ABI library loads and exports every symbol include/lewin_b200.h declares, the ctypes
structs match the C layout, and the host-side mirror keeps the reference's module surface."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "lewin_b200.h")


@pytest.fixture(scope="module")
def lib_path():
    import __graft_entry__ as g
    if not os.path.isfile(g.LIB):
        g.build()
    return g.LIB


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lewin_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    names = _declared_functions()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/lewin_b200.h but not exported"
    from lewin_b200 import _lib
    assert sorted(_lib.EXPORTS) == names
    lib.lewin_abi_version.restype = ctypes.c_int
    assert lib.lewin_abi_version() == _lib.ABI_VERSION
    lib.lewin_build_info.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.lewin_build_info()


def test_ctypes_structs_match_c_layout(tmp_path):
    from lewin_b200 import _lib
    structs = ["LewinAttnFwdArgs", "LewinAttnBwdArgs", "LewinCoreFwdArgs", "LewinCoreBwdArgs", "LewinLeffFwdArgs", "LewinLeffBwdArgs",
               "LewinUpsampleFwdArgs", "LewinInputProjArgs"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
    for s in structs:
        cls = getattr(_lib, s)
        lines.append(f'printf("{s} %zu\\n", sizeof({s}));')
        for f, _t in cls._fields_:
            lines.append(f'printf("{s}.{f} %zu\\n", offsetof({s}, {f}));')
    lines.append("return 0;}")
    c = tmp_path / "layout.c"
    c.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(c)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip().split("\n"))
    for s in structs:
        cls = getattr(_lib, s)
        assert int(out[s]) == ctypes.sizeof(cls), s
        for f, _t in cls._fields_:
            assert int(out[f"{s}.{f}"]) == getattr(cls, f).offset, (s, f)


def test_argument_validation_without_gpu(lib_path):
    """Argument checks run before any CUDA call: NULL / shape / alignment errors are reported on a CPU box."""
    from lewin_b200 import _lib
    lib = _lib.load()
    a = _lib.LewinAttnFwdArgs(B=1, H=16, W=16, C=32, nH=1)
    assert lib.lewin_attn_fwd_f32(a, None, 0, None) == -1          # LEWIN_E_NULL
    for f in ("x", "y", "ln_w", "ln_b", "w_qkv", "b_qkv", "w_out", "b_out", "rpb_table", "index_sample", "qkv", "ctx"):
        setattr(a, f, 0x1000)
    a.use_rpb = 1
    a.C = 48
    assert lib.lewin_attn_fwd_f32(a, None, 0, None) == -2          # LEWIN_E_SHAPE
    a.C = 32
    a.x = 0x1004
    assert lib.lewin_attn_fwd_f32(a, None, 0, None) == -3          # LEWIN_E_ALIGN
    assert b"aligned" in lib.lewin_error_string(-3)
    l = _lib.LewinLeffFwdArgs(B=1, H=8, W=8, C=32, hidden=128)
    assert lib.lewin_leff_fwd_bf16(l, None, 0, None) == -1
    assert lib.lewin_attn_fwd_workspace_bytes(a, 0) >= 2 * 256 * 4
    a.nH = 3                                                       # head_dim = C / nH must be 32, 64 or 128
    a.x = 0x1000
    assert lib.lewin_attn_fwd_f32(a, None, 0, None) == -2
    c = _lib.LewinCoreBwdArgs()
    assert lib.lewin_probsparse_core_bwd_f32(c, None, 0, None) == -1      # LEWIN_E_NULL


def test_ops_refuse_cpu_tensors():
    import lewin_b200 as L
    blk = L.LeWinTransformerBlock(dim=32, input_resolution=(128, 128), num_heads=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        blk(torch.zeros(1, 64, 32))


def test_missing_library_fails_loudly(monkeypatch):
    from lewin_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/liblewin_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_state_dict_layout_matches_reference(golden_dir):
    import lewin_b200 as L
    model = L.Uformer(img_size=128, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff")
    mine = {k: f"{tuple(v.shape)} {str(v.dtype).replace('torch.', '')}" for k, v in model.state_dict().items()}
    ref = dict(l.split(" ", 1) for l in open(os.path.join(golden_dir, "uformer32_state_dict_keys.txt")).read().strip().split("\n"))
    assert mine == ref
    assert sum(p.numel() for p in model.parameters()) == 26222685
    blk = model.encoderlayer_0.blocks[1]
    assert blk.shift_size == 4 and model.conv.blocks[1].shift_size == 0    # bottleneck: shift forced to 0
    assert len(blk.state_dict()) == 26


def test_rng_stream_lockstep(golden_dir):
    """index_sample is drawn with the reference's call (attn.py:91): same seed -> the recorded draws."""
    import lewin_b200 as L
    z = np.load(os.path.join(golden_dir, "uformer32_b2.npz"))
    torch.manual_seed(int(z["seed"]) + 2)
    model = L.Uformer.__new__(L.Uformer)
    model.depths = [2] * 9
    got = L.Uformer.draw_index_samples(model).numpy()
    assert np.array_equal(got, z["idx"].astype(np.int64))


def test_relative_position_index_buffer_matches_reference_formula():
    import lewin_b200 as L
    from oracle import lewin_oracle as O
    wa = L.WindowAttention(32, (8, 8), 1)
    assert np.array_equal(wa.relative_position_index.numpy(), O.relative_position_index(8))


def test_fullres_pad_tile_roundtrip():
    from lewin_b200 import fullres as F
    img = torch.rand(1, 3, 1200, 1600)
    canvas = F.wrap_pad(img)
    assert canvas.shape == (1, 3, 1664, 1664)
    assert torch.equal(canvas[:, :, :1200, 1600:], img[:, :, :, :64])           # test_long_GPU.py:88
    assert torch.equal(canvas[:, :, 1200:, :], canvas[:, :, :464, :])            # test_long_GPU.py:89
    tiles = F.to_tiles(canvas)
    assert tiles.shape == (169, 3, 128, 128)
    assert torch.equal(tiles[14], canvas[0, :, 128:256, 128:256])
    assert torch.equal(F.from_tiles(tiles, 1664), canvas)
    cover = []
    for r in range(8):
        s, e = F.shard_range(169, r, 8)
        cover += list(range(s, e))
        assert e - s in (21, 22)
    assert cover == list(range(169))


def test_patch_reference_model_structure(golden_dir):
    """patch() / unpatch() on a block with the reference's class names and module layout: the foreign stand-in of
    tests/test_gpu_patch.py, whose state_dict must equal the reference's recorded layout of a shifted embed_dim 32 block."""
    import lewin_b200 as L
    from tests.test_gpu_patch import LeWinTransformerBlock
    pre = "encoderlayer_0.blocks.1."
    lines = open(os.path.join(golden_dir, "uformer32_state_dict_keys.txt")).read().strip().split("\n")
    ref = {k[len(pre):]: v for k, v in (l.split(" ", 1) for l in lines) if k.startswith(pre)}
    torch.manual_seed(0)
    blk = LeWinTransformerBlock(32, 1, 4).eval()
    assert {k: f"{tuple(v.shape)} {str(v.dtype).replace('torch.', '')}" for k, v in blk.state_dict().items()} == ref
    x = torch.randn(1, 256, 32)
    torch.manual_seed(1)
    with torch.no_grad():
        before = blk(x)
    keys = list(blk.state_dict().keys())
    L.patch(blk)
    assert list(blk.state_dict().keys()) == keys
    assert blk.forward.__func__.__name__ == "_block_forward"
    assert blk.attn.forward.__func__.__name__ == "_window_attention_forward"
    assert blk.mlp.forward.__func__.__name__ == "_leff_forward"
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        blk(torch.zeros(1, 256, 32))
    L.unpatch(blk)
    torch.manual_seed(1)
    with torch.no_grad():
        out = blk(x)                            # the block's own forward restored, runs on CPU
    assert out.shape == (1, 256, 32) and torch.equal(out, before)


def test_rows_needed_cover_each_ranks_tiles():
    """fullres.rows_needed: uploading only those image rows (NaN elsewhere) leaves every tile of the rank's shard identical
    to the tiles cut from the full image - for every world size of BASELINE config 3 and an odd image size."""
    import torch
    from lewin_b200 import fullres
    for (H, W) in ((1200, 1600), (300, 500), (250, 130)):
        g = torch.Generator().manual_seed(H)
        img = torch.rand(1, 3, H, W, generator=g)
        full_tiles = fullres.to_tiles(fullres.wrap_pad(img, ps=128), 128)
        T = full_tiles.shape[0]
        for world in (1, 2, 4, 8):
            covered = 0
            for rank in range(world):
                rows = fullres.rows_needed(H, W, rank, world)
                part = torch.full_like(img, float("nan"))
                for r0, r1 in rows:
                    assert 0 <= r0 < r1 <= H
                    part[:, :, r0:r1] = img[:, :, r0:r1]
                    covered += r1 - r0
                s, e = fullres.shard_range(T, rank, world)
                tiles = fullres.to_tiles(fullres.wrap_pad(part, ps=128), 128)[s:e]
                assert torch.equal(tiles, full_tiles[s:e]), (H, W, world, rank)
            if world == 1:
                assert covered == H


def test_bf16_weight_image_cache_follows_in_place_updates():
    """ops._bf16_image (the caller-converted weights of ABI v2): the image is reused while the parameter is untouched and
    rebuilt after any in-place update (optimizer step, load_state_dict), and never shared between distinct tensors."""
    import torch
    from lewin_b200 import ops
    w = torch.nn.Parameter(torch.randn(8, 8))
    a = ops._bf16_image(w)
    assert a.dtype == torch.bfloat16 and torch.equal(a, w.detach().to(torch.bfloat16))
    assert ops._bf16_image(w) is a                       # cached
    with torch.no_grad():
        w.add_(1.0)                                      # what an optimizer step / load_state_dict does: _version bump
    b = ops._bf16_image(w)
    assert b is not a and torch.equal(b, w.detach().to(torch.bfloat16))
    w2 = torch.nn.Parameter(w.detach().clone())
    assert ops._bf16_image(w2) is not b
    # one entry per LIVE tensor: the stale version of `w` was replaced, dead tensors drop out, pinned images are handed back
    n = len(ops.weight_images)
    with ops.weight_images.pin() as held:
        for _ in range(5):
            with torch.no_grad():
                w.mul_(0.5)
            c = ops._bf16_image(w)
        t = torch.randn(4, 4)
        ops._bf16_image(t)
    assert len(ops.weight_images) == n + 1 and any(h is c for h in held) and len(held) == 6
    del t
    import gc
    gc.collect()
    assert len(ops.weight_images) == n


def test_uformer_constructor_rejects_unbuilt_configurations_with_a_message():
    """ADVICE r1: Uformer() with the reference's default token_mlp='ffn' and the embed_dim=16 variant (model_utils.py:97)
    must fail at construction with an actionable message, not at the first forward."""
    import lewin_b200 as L
    with pytest.raises(NotImplementedError, match="token_mlp='leff'"):
        L.Uformer()
    with pytest.raises(NotImplementedError, match="embed_dim 16"):
        L.Uformer(embed_dim=16, token_mlp="leff")
    with pytest.raises(NotImplementedError, match="head_dim"):
        L.WindowAttention(48, 8, 3)
    L.WindowAttention(128, 8, 1)        # head_dim 128 (BASELINE config 5) constructs


@pytest.mark.parametrize("H,W,world", [(200, 300, 1), (200, 300, 3), (250, 130, 2), (1200, 1600, 8)])
def test_tile_glue_indices_equal_the_slicing_functions(H, W, world):
    """fullres.tile_glue_indices (one index gather per side) == wrap_pad + to_tiles / from_tiles + crop (test_long_GPU.py:85-93
    geometry), for every rank of a sharded run, including the all-gather layout with one padded slot per short rank."""
    from lewin_b200 import fullres
    ps, C = 128, 3
    torch.manual_seed(H + W + world)
    img = torch.rand(1, C, H, W)
    L = fullres.canvas_size(H, W, ps)
    tiles = fullres.to_tiles(fullres.wrap_pad(img, ps=ps), ps)
    T = tiles.shape[0]
    per = (T + world - 1) // world
    gathered = torch.full((world * per, C, ps, ps), float("nan"))
    fake_out = tiles * 2.0 + 1.0                                   # stands in for the model: any per-tile function
    for r in range(world):
        in_idx, out_idx, per_r, s, e = fullres.tile_glue_indices(H, W, C, ps, r, world, img.device)
        assert per_r == per and (s, e) == fullres.shard_range(T, r, world)
        mine = img.reshape(-1).index_select(0, in_idx).view(e - s, C, ps, ps)
        assert torch.equal(mine, tiles[s:e])
        gathered[r * per:r * per + (e - s)] = fake_out[s:e]
    for r in range(world):
        _, out_idx, _, _, _ = fullres.tile_glue_indices(H, W, C, ps, r, world, img.device)
        got = gathered.reshape(-1).index_select(0, out_idx).view(1, C, H, W)
        assert torch.equal(got, fullres.from_tiles(fake_out, L, ps)[:, :, :H, :W])


def test_uformer_constructor_states_what_is_built():
    """Whole models exist for embed_dim 32 and 64 (head_dim = embed_dim, My_model_1.py:962; the widest level has 16 x embed_dim
    channels and the kernels take rows of up to 1024); anything else is refused at construction with the reason, instead of
    failing inside a forward (ADVICE r1: embed_dim 16 used to fail at the first launch with LEWIN_E_SHAPE)."""
    import lewin_b200 as L
    for ed in (32, 64):
        m = L.Uformer(img_size=128, embed_dim=ed, win_size=8, token_projection="linear", token_mlp="leff")
        assert m.embed_dim == ed
    for ed in (16, 128):
        with pytest.raises(NotImplementedError, match="embed_dim"):
            L.Uformer(img_size=128, embed_dim=ed, win_size=8, token_projection="linear", token_mlp="leff")
    with pytest.raises(NotImplementedError, match="token_mlp"):
        L.Uformer(img_size=128, embed_dim=32)                      # the reference signature's default token_mlp='ffn'
