"""Cost of an input mask on a whole-image canvas forward (the masked inference path of test_in_any_resolution.py).

Uformer(embed_dim=32), batch 1, a 1664 x 1664 canvas (the size a 1200 x 1600 image pads to), in fp32 and under bf16 autocast:
  (a) the unmasked forward;
  (b) the masked forward: the input mask evaluated per token inside the attention kernels (model(x, mask));
  (c) the dense-mask forward the library ran before: every block given the [B*nW, 64, 64] input + shift mask built with torch
      ops (as modules.input_attn_mask / dense_shift_mask did) and the analytic shift mask switched off.
The mask is ones over a centred 1200 x 1600 rectangle, or its complement.  Each configuration is warmed up, then timed with CUDA
events in interleaved rounds (median reported); peak memory is measured in a separate call of each.  Also checks that (b) and (c)
return the same image bit for bit.

    python scripts/masked_canvas_time.py --out profiles/r3_b_masked_canvas.txt
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def dense_from_token_mask(tm, shift, win=8):
    """[Bm, H, W] level mask -> dense fp32 [Bm * nW, 64, 64] input + shift mask (tests/token_mask_ref.py)."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1664)
    ap.add_argument("--rect", type=int, nargs=2, default=(1200, 1600))
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("masked_canvas_time.py measures on the GPU; no CUDA device found")
    import lewin_b200 as L

    dev = torch.device("cuda:0")
    S = args.size
    torch.manual_seed(0)
    model = L.Uformer(img_size=128, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff").to(dev).eval()
    idx = model.draw_index_samples()
    x = torch.rand(1, 3, S, S, device=dev)
    rect = torch.zeros(1, 1, S, S, device=dev)
    h, w = args.rect
    rect[..., (S - h) // 2:(S - h) // 2 + h, (S - w) // 2:(S - w) // 2 + w] = 1.0
    masks = {"rect": rect, "complement": 1.0 - rect}

    orig = L.ops.lewin_attn

    def dense_attn(xx, **kw):
        tm = kw.pop("token_mask", None)
        if tm is not None:
            kw["mask"] = dense_from_token_mask(tm, kw["shift"])
            kw["analytic_shift_mask"] = False
        return orig(xx, **kw)

    def run(dt, mask, dense):
        L.ops.lewin_attn = dense_attn if dense else orig
        try:
            with torch.no_grad(), torch.autocast("cuda", torch.bfloat16, enabled=dt == "bf16"):
                return model(x, mask, index_samples=idx)
        finally:
            L.ops.lewin_attn = orig

    cfgs = [("a unmasked", None, False)]
    for mn, m in masks.items():
        cfgs += [(f"b token mask ({mn})", m, False), (f"c dense mask ({mn})", m, True)]

    props = torch.cuda.get_device_properties(dev)
    try:
        plim = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        plim = "unknown"
    lines = [f"# scripts/masked_canvas_time.py --size {S} --rect {h} {w} --warmup {args.warmup} --reps {args.reps}",
             f"# device: {props.name}, power limit {plim}; torch {torch.__version__}",
             "# Uformer(embed_dim=32), batch 1, whole-canvas forward; median of interleaved CUDA-event timings; peak = "
             "torch.cuda.max_memory_allocated over one call (model weights and input included)", ""]
    for dt in ("f32", "bf16"):
        outs = {}
        for name, m, dense in cfgs:
            for _ in range(args.warmup):
                run(dt, m, dense)
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            outs[name] = run(dt, m, dense).float()
            torch.cuda.synchronize()
            outs[name + "/peak"] = torch.cuda.max_memory_allocated(dev)
        times = {name: [] for name, _, _ in cfgs}
        for _ in range(args.reps):
            for name, m, dense in cfgs:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(dt, m, dense)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1))
        base = statistics.median(times["a unmasked"])
        lines.append(f"[{dt}]{'':22s} median ms   min ms   vs (a)   peak MiB")
        for name, _, _ in cfgs:
            med = statistics.median(times[name])
            lines.append(f"  {name:26s} {med:9.2f} {min(times[name]):8.2f} {med / base:8.3f} {outs[name + '/peak'] / 2**20:10.0f}")
        for mn in masks:
            same = torch.equal(outs[f"b token mask ({mn})"], outs[f"c dense mask ({mn})"])
            lines.append(f"  (b) == (c) bit for bit, {mn}: {same}")
        lines.append("")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
