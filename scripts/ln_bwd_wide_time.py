"""Kernel time of ln_bwd_wide_kernel (fp32 LayerNorm backward, rows of 516 ... 1024 channels) at the bottleneck shapes of a
batch-32 embed_dim 64 training step, against its HBM floor: per row it reads x, dz and dres and writes dx, 16 KB at C = 1024.
Shapes: `conv` (8 x 8 map) and `decoderlayer_0` (16 x 16 map, shift 4), C = 1024, 16 heads of 64, batch 32.  One LeWin block
forward + backward (fp32) under torch.profiler with CUDA activities; each block backward launches the kernel twice (LN1, LN2).
Prints one JSON line with the card's name and power limit read in the same run.
Usage (GPU box):  python scripts/ln_bwd_wide_time.py [--iters 20] [--hbm-gbs 7700]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--hbm-gbs", type=float, default=7700.0, help="HBM bandwidth of the floor (data-sheet B200: 7.7 TB/s)")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import lewin_b200 as L
    dev = torch.device("cuda:0")
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True).stdout.strip()
    C, nH, B = 1024, 16, 32
    rows_out = []
    for name, hw, shift in (("conv", 8, 0), ("decoderlayer_0", 16, 4)):
        torch.manual_seed(0)
        blk = L.LeWinTransformerBlock(dim=C, input_resolution=(hw, hw), num_heads=nH, win_size=8, shift_size=shift).to(dev).eval()
        x = torch.randn(B, hw * hw, C, device=dev)
        dy = torch.randn_like(x)
        idx = torch.randint(64, (64, 25))

        def step():
            xr = x.detach().requires_grad_(True)
            blk.zero_grad(set_to_none=True)
            blk(xr, None, idx).backward(dy)

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.iters):
                step()
            torch.cuda.synchronize()
        ts = [ev.device_time for ev in prof.events()
              if ev.device_type == torch.autograd.DeviceType.CUDA and "ln_bwd_wide_kernel" in ev.name]
        rows = B * hw * hw
        floor_us = rows * 4 * C * 4 / (args.hbm_gbs * 1e9) * 1e6
        us = sum(ts) / len(ts) if ts else float("nan")
        rows_out.append(dict(level=name, rows=rows, C=C, launches=len(ts), kernel_us=us, hbm_floor_us=floor_us,
                             share_of_floor=floor_us / us if ts else None, achieved_gbs=rows * 16 * C / (us * 1e3) if ts else None))
    print(json.dumps(dict(kernel="ln_bwd_wide_kernel (fp32)", gpu=torch.cuda.get_device_name(0), power_limit_and_max_sm_clock=power,
                          hbm_gbs_floor=args.hbm_gbs, iters=args.iters, rows=rows_out)), flush=True)


if __name__ == "__main__":
    main()
