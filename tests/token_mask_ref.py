"""Torch restatement of the reference's dense input + shift mask (My_model_1.py:791-836), the form the attention kernels
received before they evaluated the input mask per token: the reference side of tests/test_gpu_token_mask.py, pinned to the
numpy oracle by tests/test_token_mask_cpu.py."""
import torch
import torch.nn.functional as F


def level_mask(mask, H, W):
    """The token mask lewin_block_forward passes for an input mask [Bm, 1, h, w]: nearest-resized to the level, [Bm, H, W]."""
    return F.interpolate(mask, size=(H, W))[:, 0]


def dense_from_token_mask(tm, shift, win=8):
    """[Bm, H, W] level mask -> dense fp32 [Bm * nW, 64, 64] mask: the input term (-100 where m_i * m_j != 0, windows
    partitioned in the unshifted frame), plus the shift mask of a shifted block, summed in fp32."""
    Bm, H, W = tm.shape
    mw = tm.reshape(Bm, H // win, win, W // win, win).permute(0, 1, 3, 2, 4).reshape(-1, win * win)
    am = mw.unsqueeze(2) * mw.unsqueeze(1)
    dense = am.masked_fill(am != 0, -100.0).masked_fill(am == 0, 0.0).float()
    if shift > 0:
        img = torch.zeros((1, H, W, 1), device=tm.device)
        sl = (slice(0, -win), slice(-win, -shift), slice(-shift, None))
        cnt = 0
        for h in sl:
            for w in sl:
                img[:, h, w, :] = cnt
                cnt += 1
        sw = img.view(1, H // win, win, W // win, win, 1).permute(0, 1, 3, 2, 4, 5).reshape(-1, win * win)
        d = sw.unsqueeze(1) - sw.unsqueeze(2)
        dense = dense + d.masked_fill(d != 0, -100.0).masked_fill(d == 0, 0.0).float().repeat(Bm, 1, 1)
    return dense
