"""BASELINE config 5: LeWin ProbSparse-attention + LeFF op microbench.

Sweep: window 8 (N = 64 tokens, u = U = 25), heads 1..16 at head_dim 32 (C = 32 * heads, what the reference's
Uformer_ProbSparse produces at embed_dim 32) over 64..1024 windows, plus head_dim = embed_dim 64 and 128 (My_model_1.py:962
makes head_dim = embed_dim; C = heads * head_dim up to 1024, the bottleneck of the embed_dim 64 model: 16 heads of 64, and
8 heads of 128) over 64 / 256 / 1024 windows; shift 0 / 4, bf16 and f32; forward and
forward+backward microseconds per block (attention half + LeFF half through the C ABI, `ops.lewin_attn` / `ops.lewin_leff`),
CUDA events over `--iters` calls after 3 warm-up calls, x ~ N(0, 1) seed 0, weights N(0, C^-1/2), index_sample from
torch.manual_seed(0); torch.randint(64, (64, 25)).  Also prints the fraction of the block's roofline time (SURVEY 8d: fully
fused ideal = max(algorithmic FLOPs / sustained bf16 TFLOP/s, 4 C s bytes per token / HBM GB/s)).
Usage (GPU box):  python scripts/op_microbench.py [--iters 20] [--channels 1024] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--head-dim-32-only", action="store_true", help="skip the head_dim 64 / 128 rows")
    ap.add_argument("--channels", type=int, nargs="*", help="only the rows of these widths C")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "op_microbench.json"))
    args = ap.parse_args()
    import torch
    from lewin_b200 import ops
    dev = torch.device("cuda:0")
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pk = {}
    hbm = float(pk.get("hbm_gbs", 6650.0))
    tf = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0)))
    rows = []
    for dtype in ("bf16", "f32"):
        tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
        sweep = [(32, h, (64, 128, 256, 512, 1024)) for h in (1, 2, 4, 8, 16)]
        if not args.head_dim_32_only:
            sweep += [(hd, h, (64, 256, 1024)) for hd in (64, 128) for h in (1, 2, 4, 8, 16) if hd * h <= 1024]
        if args.channels:
            sweep = [t for t in sweep if t[0] * t[1] in args.channels]
        for head_dim, heads, window_counts in sweep:
            C = head_dim * heads
            for windows in window_counts:
                # windows * 64 tokens as one H x W map (H = W or H = 2 W), B = 1
                W = 8
                while W * W * 4 <= windows * 64:
                    W *= 2
                H = windows * 64 // W                       # 64 -> 64x64, 128 -> 128x64, 256 -> 128x128, ...
                for shift in (0, 4):
                    g = torch.Generator().manual_seed(0)
                    r = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).to(dev)
                    x = r(1, H * W, C).to(tdt).requires_grad_(True)
                    p = dict(ln_w=1 + r(C, sc=0.1), ln_b=r(C, sc=0.1), w_qkv=r(3 * C, C, sc=C ** -0.5), b_qkv=r(3 * C, sc=0.1),
                             w_out=r(C, C, sc=C ** -0.5), b_out=r(C, sc=0.1), rpb_table=r(225, heads, sc=0.2))
                    q = dict(ln_w=1 + r(C, sc=0.1), ln_b=r(C, sc=0.1), w1=r(4 * C, C, sc=C ** -0.5), b1=r(4 * C, sc=0.1),
                             w_dw=r(4 * C, 1, 3, 3, sc=0.3), b_dw=r(4 * C, sc=0.1), w2=r(C, 4 * C, sc=(4 * C) ** -0.5), b2=r(C, sc=0.1))
                    for d in (p, q):
                        for v in d.values():
                            v.requires_grad_(True)
                    torch.manual_seed(0)
                    idx = torch.randint(64, (64, 25)).to(dev, dtype=torch.int32)
                    dout = r(1, H * W, C).to(tdt)

                    def fwd():
                        with torch.no_grad():
                            y = ops.lewin_attn(x, B=1, H=H, W=W, num_heads=heads, shift=shift, index_sample=idx, **p)
                            return ops.lewin_leff(y, B=1, H=H, W=W, **q)

                    def fwd_bwd():
                        y = ops.lewin_attn(x, B=1, H=H, W=W, num_heads=heads, shift=shift, index_sample=idx, **p)
                        ops.lewin_leff(y, B=1, H=H, W=W, **q).backward(dout)

                    def timeit(fn):
                        for _ in range(3):
                            fn()
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(args.iters):
                            fn()
                        e1.record()
                        torch.cuda.synchronize()
                        return e0.elapsed_time(e1) / args.iters * 1e3

                    try:
                        f_eager, fb_eager = timeit(fwd), timeit(fwd_bwd)
                    except (RuntimeError, NotImplementedError) as e:      # a shape the library rejects: report it, keep sweeping
                        print(f"{dtype} heads={heads} head_dim={head_dim} C={C} windows={windows} shift={shift}: not run ({e})", flush=True)
                        rows.append(dict(dtype=dtype, heads=heads, head_dim=head_dim, C=C, windows=windows, shift=shift, error=str(e)[:200]))
                        continue
                    # device time without the host's launch gaps (~110 us of Python / ctypes per block at the small sizes):
                    # the same call sequences replayed as CUDA graphs, as bench.py's block microbench and the training step do
                    launch = "cuda-graph replay"
                    try:
                        side = torch.cuda.Stream(device=dev)
                        side.wait_stream(torch.cuda.current_stream(dev))
                        with torch.cuda.stream(side):
                            fwd(); fwd_bwd()
                        torch.cuda.current_stream(dev).wait_stream(side)
                        torch.cuda.synchronize()
                        for t in [x] + list(p.values()) + list(q.values()):
                            t.grad = None
                        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g1):
                            y_static = fwd()
                        with torch.cuda.graph(g2):
                            fwd_bwd()
                        f_us, fb_us = timeit(g1.replay), timeit(g2.replay)
                        del g1, g2, y_static
                    except Exception as e:
                        f_us, fb_us, launch = f_eager, fb_eager, "eager (graph capture failed: %s)" % repr(e)[:80]
                    tokens = windows * 64
                    s = 2 if dtype == "bf16" else 4
                    flops = tokens * (24 * C * C + 222 * C)
                    ideal_us = max(flops / (tf * 1e12), tokens * 4 * C * s / (hbm * 1e9)) * 1e6
                    rows.append(dict(dtype=dtype, heads=heads, head_dim=head_dim, C=C, windows=windows, H=H, W=W, shift=shift, fwd_us=f_us,
                                     fwd_bwd_us=fb_us, fwd_us_eager=f_eager, fwd_bwd_us_eager=fb_eager, launch=launch, fwd_tflops=flops / f_us / 1e6, ideal_fwd_us=ideal_us))
                    print(f"{dtype} heads={heads:2d} head_dim={head_dim:3d} C={C:4d} windows={windows:4d} ({H}x{W}) shift={shift}: fwd {f_us:8.1f} us  "
                          f"fwd+bwd {fb_us:8.1f} us (eager {f_eager:7.1f} / {fb_eager:7.1f})  {flops / f_us / 1e6:7.1f} TFLOP/s fwd  "
                          f"(fused-ideal {ideal_us:6.1f} us)", flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(dict(config="BASELINE config 5", launch="CUDA-graph replay of the C-ABI call sequence (eager python launch numbers alongside)",
                   iters=args.iters, rows=rows), open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
