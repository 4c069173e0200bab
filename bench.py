#!/usr/bin/env python
"""Benchmark of the B200 LeWin hot path on BASELINE.json's headline metric:

    full-res 1600x1200 dehaze images/sec at N B200s  (config 3: 1200x1600 image wrap-padded to 1664^2,
    cut into 169 tiles of 128x128, tiles sharded over the ranks, final all_gather of the outputs)

    python bench.py --gpus N --steps K --warmup W [--dtype f32|bf16] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one full image.  `value` is measured with the image already resident in HBM, `e2e` through
the public API from pinned HOST memory (H2D + D2H inside the timed region).  `roofline` is for the
dominant kernel type of the step, timed with CUDA events through the ABI's per-kernel timing hook;
`cpu_baseline` / `--impl reference` time the reference's CPU op sequence (oracle/torch_port.py) on the
host cores on a bounded sample of tiles.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG_H, IMG_W, PS = 1200, 1600, 128
N_TILES = 169
METRIC = "full-res 1600x1200 dehaze images/sec"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# --------------------------------------------------------------------------------- reference arm
def cpu_reference_images_per_s(sample_tiles, steps, warmup, seed=1234):
    """oracle/torch_port.py (reference op sequence, torch CPU eager, all host threads) on `sample_tiles` of the
    169 tiles per step; images/s = (sample/169) / step time."""
    import torch
    import lewin_b200 as L
    from oracle import torch_port
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(seed)
    model = L.Uformer(img_size=PS, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff")
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    tiles = torch.rand(sample_tiles, 3, PS, PS)
    idx = model.draw_index_samples()
    for _ in range(warmup):
        torch_port.uformer_forward(tiles, sd, idx)
    t0 = time.perf_counter()
    for _ in range(steps):
        torch_port.uformer_forward(tiles, sd, idx)
    dt = (time.perf_counter() - t0) / steps
    return (sample_tiles / N_TILES) / dt, dt, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = 8
    v, dt, cores = cpu_reference_images_per_s(sample, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config3: 1200x1600 -> 1664^2 canvas, 169 tiles of 128^2, Uformer_ProbSparse embed_dim=32 "
                               "(random init); CPU step = %d-tile sample scaled to 169" % sample},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} of 169 tiles per step, oracle/torch_port.py (reference ATen op sequence, torch CPU eager)"},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------- our arm
def kernel_work(op, name, info):
    """Algorithmic FLOPs and minimum HBM bytes of one launch (DESIGN.md section 5; SURVEY 8d)."""
    t, C = info["tokens"], info["C"]
    s = 4 if info["dtype"] == "f32" else 2
    if name == "gemm_qkv":
        return 2.0 * t * C * 3 * C, t * C * s + t * 3 * C * s + 3 * C * C * 4
    if name == "gemm_out":
        return 2.0 * t * C * C, 3 * t * C * s + C * C * 4
    if name == "gemm_fc1_gelu":
        return 2.0 * t * C * 4 * C, t * C * s + t * 4 * C * s + 4 * C * C * 4
    if name == "gemm_fc2":
        return 2.0 * t * 4 * C * C, t * 4 * C * s + 2 * t * C * s + 4 * C * C * 4
    if name == "probsparse_core":
        return 150.0 * t * C, 4 * t * C * s
    if name == "dwconv_gelu":
        return 72.0 * t * C, 8 * t * C * s
    if name == "attn_fused":      # LN1 -> q|k|v -> ProbSparse core -> out projection -> residual in one kernel: x read, y written
        return 8.0 * t * C * C + 150.0 * t * C, 2 * t * C * s + 4 * C * C * 4
    if name == "leff_tail":       # dwconv + GELU -> linear2 -> residual in one kernel: h1 read, y read, out written (h2 stays on chip)
        return 72.0 * t * C + 2.0 * t * 4 * C * C, t * 4 * C * s + 2 * t * C * s + 4 * C * C * 4 + 40 * C * 4
    if name == "ln_stats":
        return 0.0, t * C * s
    return 0.0, 0.0


LEVELS = [("enc0", 32, 128), ("enc1", 64, 64), ("enc2", 128, 32), ("enc3", 256, 16), ("bottleneck", 512, 8),
          ("dec0", 512, 16), ("dec1", 256, 32), ("dec2", 128, 64), ("dec3", 64, 128)]


def block_microbench(dev, dtype, batch=32, iters=5):
    """Second half of BASELINE's metric: LeWin block forward and forward+backward microseconds per block, at the
    training shapes of config 2 (batch 32 x 128^2 patches), one block per level, shift 4 (0 at the bottleneck)."""
    import torch
    import lewin_b200 as L
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    out = []
    for name, C, hw in LEVELS:
        torch.manual_seed(0)
        blk = L.LeWinTransformerBlock(dim=C, input_resolution=(hw, hw), num_heads=C // 32, win_size=8,
                                      shift_size=4 if hw > 8 else 0).to(dev)
        x = torch.randn(batch, hw * hw, C, device=dev, dtype=tdt)
        idx = torch.randint(64, (64, 25))
        dy = torch.randn_like(x)

        def fwd():
            with torch.no_grad():
                return blk(x, None, idx)

        def fwd_bwd():
            xr = x.detach().requires_grad_(True)
            blk.zero_grad(set_to_none=True)
            blk(xr, None, idx).backward(dy)

        idx_dev = idx.to(dev, dtype=torch.int32)
        xg = x.detach().clone().requires_grad_(True)

        def fwd_bwd_static():           # static buffers: capturable (the key-sample indices are refreshed outside the graph)
            xg.grad = None
            blk.zero_grad(set_to_none=True)
            blk(xg, None, idx_dev).backward(dy)

        def timeit(fn):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters * 1e3

        res = {"fwd_us_eager": timeit(fwd), "fwd_bwd_us_eager": timeit(fwd_bwd)}
        # device time without host launch gaps: the same call sequences replayed as CUDA graphs (as the training step does)
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    with torch.no_grad():
                        blk(x, None, idx_dev)
                    fwd_bwd_static()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                with torch.no_grad():
                    y_static = blk(x, None, idx_dev)
            xg.grad = None
            blk.zero_grad(set_to_none=True)
            with torch.cuda.graph(g2):
                blk(xg, None, idx_dev).backward(dy)
            res["fwd_us"] = timeit(g1.replay)
            res["fwd_bwd_us"] = timeit(g2.replay)
            res["launch"] = "cuda-graph replay (eager numbers alongside)"
            del g1, g2, y_static
        except Exception as e:
            res["fwd_us"], res["fwd_bwd_us"] = res["fwd_us_eager"], res["fwd_bwd_us_eager"]
            res["launch"] = "eager (graph capture failed: %s)" % repr(e)[:100]
        out.append(dict(level=name, C=C, map=hw, windows=batch * (hw // 8) ** 2, **res))
        del blk, x, dy
    return dict(batch=batch, dtype=dtype, per_level=out,
                mean_fwd_us=sum(o["fwd_us"] for o in out) / len(out),
                mean_fwd_bwd_us=sum(o["fwd_bwd_us"] for o in out) / len(out),
                mean_fwd_us_eager=sum(o["fwd_us_eager"] for o in out) / len(out),
                mean_fwd_bwd_us_eager=sum(o["fwd_bwd_us_eager"] for o in out) / len(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="bf16", choices=["f32", "bf16"],
                    help="compute dtype of the headline number (bf16 = BASELINE's compute dtype; f32 = the reference's "
                         "inference precision, always reported as well under 'fp32')")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--e2e-lanes", type=int, default=0,
                    help="lanes of the end-to-end (host to host) pipeline; 0 = the same as --lanes")
    ap.add_argument("--lanes", type=int, default=2,
                    help="images in flight per rank in the serving pipeline (fullres.TiledPipeline lanes: one CUDA graph and one "
                         "stream each; 1 = one forward at a time)")
    ap.add_argument("--no-train-step", action="store_true", help="skip the config 2 / 4 training-step measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the restored image of the last timed step to DIR/restored.npy (float32, 1 x 3 x 1200 x 1600); "
                         "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import lewin_b200 as L
    from lewin_b200 import fullres, ops, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peaks = load_peaks()

    torch.manual_seed(1234)
    model = L.Uformer(img_size=PS, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff").to(dev).eval()
    g = torch.Generator().manual_seed(4321)
    img_host = torch.rand(1, 3, IMG_H, IMG_W, generator=g).pin_memory()
    out_host = torch.empty(1, 3, IMG_H, IMG_W).pin_memory()
    img_dev = img_host.to(dev)
    idx = model.draw_index_samples()            # 18 draws of attn.py:91 (identical on every rank: same seed)
    if world > 1:                               # checked once, so the per-image broadcast of the draws can be skipped
        w = torch.arange(1, idx.numel() + 1, dtype=torch.float64)
        c = (idx.double().flatten() * w).sum().to(dev)
        lo, hi = c.clone(), c.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert float(lo) == float(hi), "index_samples differ between ranks"

    cur_dtype = [args.dtype]
    graphs = {}

    def graphed_for(dt):
        """CUDA graph of this rank's tile-batch forward (static shape), captured once per precision."""
        if args.no_graph or ops.KernelTimer.active is not None:
            return None
        if dt not in graphs:
            s0, e0 = fullres.shard_range(N_TILES, rank, world)
            ex = torch.zeros(e0 - s0, 3, PS, PS, device=dev)
            graphs[dt] = fullres.GraphedForward(model, ex, idx, torch.bfloat16 if dt == "bf16" else None)
        return graphs[dt]

    lane_graphs = {}

    def graphed_lanes(dt):
        """`--lanes` graphs of the same forward (own static buffers each): TiledPipeline keeps that many images in flight."""
        g0 = graphed_for(dt)
        if g0 is None or args.lanes <= 1:
            return g0
        if dt not in lane_graphs:
            lane_graphs[dt] = [g0] + [fullres.GraphedForward(model, torch.zeros_like(g0.x), idx, torch.bfloat16 if dt == "bf16" else None)
                                      for _ in range(args.lanes - 1)]
        return lane_graphs[dt]

    def forward(img):
        g = graphed_for(cur_dtype[0])
        if g is None and cur_dtype[0] == "bf16":
            with torch.autocast("cuda", torch.bfloat16):
                return fullres.dehaze_tiled(model, img, ps=PS, index_samples=idx, broadcast_index_samples=False)
        return fullres.dehaze_tiled(model, img, ps=PS, index_samples=idx, graphed=g, broadcast_index_samples=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # N > 1: the rank's tile forward of image i+1 overlaps the all_gather + stitch of image i (fullres.TiledPipeline; same
    # kernels per image, bit-identical output - checked below before anything is timed); N == 1 has no collective to hide
    tpipes = {}
    last_out = [None]

    def step_resident():
        dt = cur_dtype[0]
        if (world > 1 or args.lanes > 1) and not args.no_graph and ops.KernelTimer.active is None:
            if dt not in tpipes:
                tpipes[dt] = fullres.TiledPipeline(model, graphed_lanes(dt), (1, 3, IMG_H, IMG_W), dev, ps=PS,
                                                   dtype=torch.bfloat16 if dt == "bf16" else torch.float32)
            last_out[0] = tpipes[dt].submit(img_dev, idx)[0]
        else:
            last_out[0] = forward(img_dev)
        return last_out[0]

    def finish_resident():
        for tp in tpipes.values():
            tp.flush()

    def step_e2e_serial():                      # copies and compute on one stream
        x = img_host.to(dev, non_blocking=True)
        out_host.copy_(forward(x).float(), non_blocking=True)

    # the public streaming call: every step copies its image in from pinned host memory and its result back out, on side
    # streams that overlap the neighbouring steps' compute (fullres.StreamingDehazer)
    # At N > 1 a rank uploads only the image rows its tile shard reads (fullres.rows_needed) and rank 0 alone delivers the
    # gathered result to the host; `e2e.serial_value` keeps the naive form (every rank moves the whole image both ways).
    rows = fullres.rows_needed(IMG_H, IMG_W, rank, world) if world > 1 else None
    e2e_pipes = {}
    e2e_lanes = args.e2e_lanes if args.e2e_lanes > 0 else args.lanes

    def e2e_fn(x):
        """The device stage of the streaming call: staged (fullres.TiledPipeline: gather + stitch on a side stream, the fp32
        conversion on the download stream) when the forward is graph-replayed, the plain serial call otherwise."""
        dt = cur_dtype[0]
        if args.no_graph or ops.KernelTimer.active is not None:
            return forward(x).float()
        if dt not in e2e_pipes:
            e2e_pipes[dt] = fullres.TiledPipeline(model, graphed_lanes(dt) if e2e_lanes > 1 else graphed_for(dt),
                                                  (1, 3, IMG_H, IMG_W), dev, ps=PS)
        return e2e_pipes[dt].submit(x, idx)

    # (a host ring as deep as the lanes' 4-slot device ring was measured: no change on one GPU - 60.0 images/s end to end - and
    # SLOWER on two, 81 against 105 images/s, so the host ring keeps its two slots)
    pipe = fullres.StreamingDehazer(e2e_fn, (1, 3, IMG_H, IMG_W), dev, rows=rows, download=(rank == 0))

    def step_e2e():
        pipe.submit(img_host, out_host)

    for _ in range(args.warmup):
        step_resident()
    step_e2e()
    step_e2e_serial()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.lewin_launch_count()
    if tpipes:                         # the pipelined form must reproduce the serial call bit for bit, on every lane
        want = forward(img_dev).clone()
        for _ in range(max(2, args.lanes)):
            tp = tpipes[cur_dtype[0]]
            k = tp.i % tp.depth
            tp.out[k].zero_()              # the slot still holds an earlier (identical) result: make the check mean something
            torch.cuda.synchronize()
            a = step_resident(); finish_resident(); torch.cuda.synchronize()
            assert torch.equal(a, want), "TiledPipeline differs from dehaze_tiled"
    ms_total = timed(step_resident, args.steps, finish=finish_resident)
    # copied now: a pipeline slot is reused by the later passes
    restored = last_out[0].float().cpu().numpy() if args.dump_outputs and rank == 0 else None
    launches = lib.lewin_launch_count() - n0
    if args.dtype in graphs:          # graph replay: the captured library launches run once per replay
        launches += graphs[args.dtype].launches_per_replay * args.steps
    ms_e2e = timed(step_e2e, args.steps, finish=pipe.flush)
    ms_e2e_serial = timed(step_e2e_serial, args.steps)
    ms_one = timed(lambda: forward(img_dev), args.steps)          # the serial call: one image at a time on one stream
    # second pass with per-kernel events (roofline of the dominant kernel type)
    with ops.KernelTimer() as kt:
        timed(step_resident, args.steps)
    # the other precision, same workload (fp32 = the reference's own inference precision, test_long_GPU.py:91)
    other = "f32" if args.dtype == "bf16" else "bf16"
    cur_dtype[0] = other
    for _ in range(2):
        step_resident()
    ms_other = timed(step_resident, args.steps, finish=finish_resident)
    ms_other_e2e = timed(step_e2e, args.steps, finish=pipe.flush)
    cur_dtype[0] = args.dtype
    clocks = sampler.stop() if rank == 0 else None

    agg = {}
    if os.environ.get("LEWIN_BREAKDOWN") and rank == 0:
        per = {}
        for op, name, info, ms in kt.summary():
            key = (name, info["C"], info["tokens"])
            per[key] = per.get(key, 0.0) + ms / args.steps
        for (name, C, tok), ms in sorted(per.items(), key=lambda kv: (kv[0][0], kv[0][1], kv[0][2])):
            fl, by = kernel_work("", name, dict(tokens=tok, C=C, dtype=args.dtype))
            print(f"[breakdown] {name:16s} C={C:4d} tokens={tok:8d} ms/step={ms:8.3f}  (2 blocks)  "
                  f"{fl*2/ms/1e9:8.1f} TFLOP/s  {by*2/ms/1e6:8.1f} GB/s", file=sys.stderr)
    for op, name, info, ms in kt.summary():
        fl, by = kernel_work(op, name, info)
        a = agg.setdefault(name, dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
        a["ms"] += ms; a["flops"] += fl; a["bytes"] += by; a["launches"] += 1
    # BASELINE configs 2 / 4: one training step (batch 32 per GPU, bf16, Charbonnier, AdamW; DDP + NCCL all-reduce at N > 1)
    train = None
    if not args.no_train_step:
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("train_step", os.path.join(ROOT, "scripts", "train_step.py"))
            ts = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(ts)
            torch.cuda.empty_cache()
            train, _ = ts.run(batch=32, steps=5, warmup=3, dtype="bf16", contrast=True)      # config 2 as BASELINE states it
            torch.cuda.empty_cache()
            t2, _ = ts.run(batch=32, steps=5, warmup=3, dtype="bf16", contrast=False)       # the LeWin path alone
            train["without_contrast"] = {k: t2[k] for k in ("step_ms", "patches_per_s", "loss", "loss_terms", "launch")}
        except Exception as e:      # the headline line must survive a failure of the secondary measurement
            train = {"error": repr(e)[:300]}
    lt = torch.tensor([float(launches)], device=dev)
    if world > 1:
        dist.all_reduce(lt)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    kernels = []
    for name, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        sec = a["ms"] / 1e3
        t_tensor = a["flops"] / (peaks["tf_sustained"] * 1e12)
        t_hbm = a["bytes"] / (peaks["hbm"] * 1e9)
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        ach = a["flops"] / sec / 1e12 if bound == "tensor" else a["bytes"] / sec / 1e9
        peak = peaks["tf_sustained"] if bound == "tensor" else peaks["hbm"]
        kernels.append(dict(kernel=name, ms_per_step=a["ms"] / args.steps, launches_per_step=a["launches"] // args.steps,
                            bound=bound, achieved=ach, peak=peak, unit="TFLOP/s" if bound == "tensor" else "GB/s",
                            frac=ach / peak))
    dom = kernels[0]
    traffic = None
    traffic_note = None
    tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.isfile(tpath):
        try:
            tj = json.load(open(tpath))
            ent = tj.get("kernels", {}).get(dom["kernel"])
            if ent and tj.get("dtype") == args.dtype:
                traffic = ent.get("dram_bytes_per_launch")
                traffic_note = (f"ncu DRAM bytes of ONE launch ({tj.get('shape')}; {ent.get('ncu_kernel')}; capture: {ent.get('capture')}); "
                                f"algorithmic bytes of that launch = {ent.get('algorithmic_bytes_per_launch')}; {tj.get('source')}")
        except Exception:
            pass
    roofline = dict(bound=dom["bound"], achieved=dom["achieved"], peak=dom["peak"], unit=dom["unit"], frac=dom["frac"],
                    traffic=traffic, traffic_note=traffic_note, kernel=dom["kernel"], peak_source=peaks["source"],
                    note="aggregate over the launches of this kernel type in one step (all 18 blocks), CUDA events via ABI timing hook")

    # secondary measurements must not cost the headline line
    try:
        blocks = block_microbench(dev, args.dtype) if world == 1 else None
    except Exception as e:
        blocks = {"error": repr(e)[:300]}
    # the reference's own full-image computation (test_long_GPU.py:74-93): ONE forward over the 1664^2 wrap-padded canvas
    # (43 264 windows at level 0) - "canvas mode", SURVEY 8(d) config 3; a different computation from tiled mode (finding 7)
    canvas = None
    if world == 1:
        try:
            def canvas_step(dt):
                if dt == "bf16":
                    with torch.autocast("cuda", torch.bfloat16):
                        return fullres.dehaze_canvas(model, img_dev, ps=PS, index_samples=idx)
                return fullres.dehaze_canvas(model, img_dev, ps=PS, index_samples=idx)
            canvas = {}
            for dt, n in (("bf16", 5), ("f32", 2)):
                for _ in range(2):
                    canvas_step(dt)
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    canvas_step(dt)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / n
                canvas[dt] = {"images_per_s": 1e3 / ms, "ms_per_image": ms, "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
            canvas["note"] = ("fullres.dehaze_canvas: wrap-pad to 1664^2, one Uformer forward over the whole canvas, crop, clamp "
                              "(test_long_GPU.py:85-93), image resident in HBM, eager launches")
            torch.cuda.empty_cache()
        except Exception as e:
            canvas = {"error": repr(e)[:300]}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            sample = 24
            v, dt, cores = cpu_reference_images_per_s(sample, 1, 1)
            cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                   "sample": f"{sample} of 169 tiles once (+1 warm-up), oracle/torch_port.py (reference ATen op sequence, torch CPU eager, fp32)"}
        except Exception as e:
            cpu = {"error": repr(e)[:300]}

    ms_step = ms_total / args.steps
    up_rows = sum(r1 - r0 for rk in range(world) for r0, r1 in fullres.rows_needed(IMG_H, IMG_W, rk, world))
    bi = up_rows * IMG_W * 3 * 4 + world * idx.numel() * 4      # all ranks: their image rows + the 18 key-sample draws
    bo = out_host.numel() * 4                                   # rank 0: the restored image
    line = {
        "metric": METRIC, "value": 1e3 / ms_step, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": "config3: synthetic 1200x1600 image wrap-padded to 1664^2, 169 tiles of 128^2 sharded over "
                               f"{world} rank(s), Uformer_ProbSparse embed_dim=32 random init, tiled mode, final all_gather",
                   "tiles_per_rank_max": -(-N_TILES // world), "l2": "working set (>=354 MB per level-0 tensor) exceeds the 126 MB L2",
                   "convs": ("all ten projections run on this library's kernels (InputProj, 4 x Downsample as implicit GEMM on tcgen05, 4 x Upsample as "
                             "token GEMM with pixel-shuffle epilogue, OutputProj with the x + y residual fused); the encoder outputs are written straight "
                             "into the decoder's concat buffers" if args.dtype == "bf16" else
                             "fp32: the projections are stock cuDNN (outside the LeWin block)"),
                   "leff": "C <= 64 levels: linear1 + GELU kernel, then ONE kernel for depthwise conv + GELU -> tcgen05.mma linear2 -> residual (h2 stays on chip); C >= 128: three kernels",
                   "attention": "C <= 64 levels: ONE fused kernel per block (LN1 -> q|k|v tcgen05.mma -> TMEM -> ProbSparse core -> out tcgen05.mma -> residual); C >= 128: three kernels",
                   "launch": "python launches" if args.no_graph else "CUDA graph replay of the per-rank tile-batch forward",
                   "pipeline": ((f"fullres.TiledPipeline, {args.lanes} lane(s): image i runs on lane i mod {args.lanes} (own CUDA graph, own stream), so "
                                 f"{args.lanes} forwards are in flight and one image's under-filled deep-level kernels share the SMs with the other's; "
                                 "the all_gather + stitch of an image run on a side stream under the following forwards; every one of the K timed "
                                 "steps is a whole image, started and finished inside the timed region; every lane's output is asserted "
                                 "bit-identical to the serial call before timing") if ((world > 1 or args.lanes > 1) and not args.no_graph) else
                                "serial: gather indices -> forward -> stitch on one stream"),
                   "images_in_flight": args.lanes if ((world > 1 or args.lanes > 1) and not args.no_graph) else 1,
                   "one_in_flight": {"value": 1e3 / (ms_one / args.steps), "ms_per_step": ms_one / args.steps,
                                     "note": "fullres.dehaze_tiled, one image at a time on one stream (= the latency of an image)"},
                   "lewin_compute": "3xTF32 (fp32-grade): the four linears on tcgen05.mma kind::tf32 (hi/lo split in the producer warps, TMEM), mma.sync ProbSparse core" if args.dtype == "f32" else
                                    "bf16 operands, fp32 accumulate: warp-specialised tcgen05 GEMMs (TMEM, TMA at C >= 256), mma.sync ProbSparse core, TMA-fed depthwise conv"},
        "e2e": {"value": 1e3 / (ms_e2e / args.steps), "unit": "images/s", "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo, "images_in_flight": e2e_lanes,
                "mode": "fullres.StreamingDehazer over fullres.TiledPipeline: pinned host image -> H2D -> tile gather / forward -> (side stream) all_gather / stitch / crop -> D2H every step; the "
                        "copies run on side streams and overlap the neighbouring steps' compute (double-buffered); at N > 1 each rank uploads "
                        "only the image rows its tiles read and rank 0 downloads the gathered result (bytes = sum over ranks)",
                "serial_value": 1e3 / (ms_e2e_serial / args.steps)},
        "gpu_launches": int(lt.item()),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        ("fp32" if other == "f32" else "bf16"): {
            "value": 1e3 / (ms_other / args.steps), "unit": "images/s", "ms_per_step": ms_other / args.steps,
            "e2e": 1e3 / (ms_other_e2e / args.steps),
            "note": "same workload at the other precision (f32 = 3xTF32 error-compensated kernels, strict parity path)"},
        "lewin_block_us": blocks,
        "canvas_mode": canvas,
        "train_step": train,
        "kernels": kernels,
    }
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "restored.npy"), restored)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
