"""Cost of the deterministic backward (torch.use_deterministic_algorithms(True)) on one GPU, the two modes alternated in one
process: block forward + backward microseconds per level at the batch-32 training shapes of bench.py's block microbenchmark
(CUDA-graph replays), the TrainStep time of embed_dim 32 at batch 32 (bf16 autocast, contrast=False, graph replay), and the
largest deterministic-mode workspace over those shapes.  Prints one JSON object (card name and power limit included).

Usage:  python scripts/deterministic_cost.py [--rounds 3] [--iters 20] [--steps 20]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

LEVELS = [("enc0", 32, 128), ("enc1", 64, 64), ("enc2", 128, 32), ("enc3", 256, 16), ("bottleneck", 512, 8),
          ("dec0", 512, 16), ("dec1", 256, 32), ("dec2", 128, 64), ("dec3", 64, 128)]


def _time(fn, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _block_graphs(dev, batch):
    """one captured forward + backward per level and mode: {(level, det): graph}"""
    import torch
    import lewin_b200 as L
    graphs, keep = {}, []
    for name, C, hw in LEVELS:
        torch.manual_seed(0)
        blk = L.LeWinTransformerBlock(dim=C, input_resolution=(hw, hw), num_heads=C // 32, win_size=8,
                                      shift_size=4 if hw > 8 else 0).to(dev)
        x = torch.randn(batch, hw * hw, C, device=dev, dtype=torch.bfloat16).requires_grad_(True)
        dy = torch.randn_like(x)
        idx = torch.randint(64, (64, 25)).to(dev, dtype=torch.int32)
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    x.grad = None
                    blk.zero_grad(set_to_none=True)
                    blk(x, None, idx).backward(dy)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            x.grad = None
            blk.zero_grad(set_to_none=True)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                blk(x, None, idx).backward(dy)
            graphs[(name, det)] = g
        keep.append((blk, x, dy, idx))
    torch.use_deterministic_algorithms(False)
    return graphs, keep


def _train_steps(dev, batch):
    import torch
    import lewin_b200 as L
    steps = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        torch.manual_seed(1234)
        model = L.Uformer(img_size=128, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff").to(dev).train()
        ts = L.training.TrainStep(model, (batch, 3, 128, 128), autocast_dtype=torch.bfloat16, contrast=False, graph=True, device=dev)
        g = torch.Generator().manual_seed(1234)
        x = torch.rand(batch, 3, 128, 128, generator=g).to(dev)
        y = torch.rand(batch, 3, 128, 128, generator=g).to(dev)
        for _ in range(3):
            ts.step(x, y)
        assert ts.launch_mode.startswith("cuda-graph"), ts.launch_mode
        steps[det] = (ts, x, y)
    torch.use_deterministic_algorithms(False)
    return steps


def _largest_workspace(batch):
    from lewin_b200 import _lib
    lib = _lib.load()
    worst = 0
    for _, C, hw in LEVELS:
        f = _lib.LewinAttnFwdArgs(B=batch, H=hw, W=hw, C=C, nH=C // 32, shift=4, use_rpb=1, analytic_shift_mask=1, rpb_table=1)
        a = _lib.LewinAttnBwdArgs(fwd=f, d_rpb_table=1)
        lf = _lib.LewinLeffFwdArgs(B=batch, H=hw, W=hw, C=C, hidden=4 * C, fused=1)
        le = _lib.LewinLeffBwdArgs(fwd=lf)
        for dt in (0, 1):
            a.deterministic = le.deterministic = 0
            base = [lib.lewin_attn_bwd_workspace_bytes(a, dt), lib.lewin_leff_bwd_workspace_bytes(le, dt)]
            a.deterministic = le.deterministic = 1
            worst = max(worst, lib.lewin_attn_bwd_workspace_bytes(a, dt) - base[0], lib.lewin_leff_bwd_workspace_bytes(le, dt) - base[1])
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_cost.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    graphs, _keep = _block_graphs(dev, args.batch)
    block = {(n, d): [] for n, _, _ in LEVELS for d in (False, True)}
    for _ in range(args.rounds):
        for name, _, _ in LEVELS:
            for det in (False, True):
                block[(name, det)].append(_time(graphs[(name, det)].replay, args.iters) * 1e3)
    del graphs
    steps = _train_steps(dev, args.batch)
    step_ms = {False: [], True: []}
    for _ in range(args.rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            ts, x, y = steps[det]
            step_ms[det].append(_time(lambda: ts.step(x, y), args.steps))
    torch.use_deterministic_algorithms(False)
    med = lambda v: sorted(v)[len(v) // 2]
    levels = [{"level": n, "C": C, "map": hw, "fwd_bwd_us_default": round(med(block[(n, False)]), 1),
               "fwd_bwd_us_deterministic": round(med(block[(n, True)]), 1),
               "ratio": round(med(block[(n, True)]) / med(block[(n, False)]), 3)} for n, C, hw in LEVELS]
    out = {"card": card, "batch": args.batch, "rounds": args.rounds, "block_fwd_bwd_graph_replay": levels,
           "block_mean_us_default": round(sum(l["fwd_bwd_us_default"] for l in levels) / len(levels), 1),
           "block_mean_us_deterministic": round(sum(l["fwd_bwd_us_deterministic"] for l in levels) / len(levels), 1),
           "train_step_ms_default": [round(v, 3) for v in step_ms[False]],
           "train_step_ms_deterministic": [round(v, 3) for v in step_ms[True]],
           "largest_det_workspace_extra_bytes": _largest_workspace(args.batch)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
