"""BASELINE configs 2 / 4: one Uformer_ProbSparse training step (batch 32 x 3 x 128 x 128 per GPU, bf16 autocast,
restored = clamp(model(input), 0, 1), loss = Charbonnier(eps 1e-3) + ContrastLoss(VGG19, random init: no weight file
offline), AdamW 2e-4 / wd 0.02; My_train.py:221-250) on the sm_100a LeWin ops; under torchrun the model is wrapped with
parallel.wrap_ddp (NCCL gradient all-reduce).  `contrast=False` drops the VGG term (the LeWin path alone).
Prints one JSON line (rank 0).
Usage:  python scripts/train_step.py [batch] [--embed-dim 32|64]   (embed_dim 64: C = 64 ... 1024, 16 heads of 64 at the bottleneck)"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(batch=32, steps=10, warmup=3, dtype="bf16", graph=True, contrast=True, embed_dim=32):
    import torch
    import torch.distributed as dist
    import lewin_b200 as L
    from lewin_b200 import training
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1234)
    model = L.Uformer(img_size=128, embed_dim=embed_dim, win_size=8, token_projection="linear", token_mlp="leff").to(dev).train()
    crit = None
    if contrast:
        from lewin_b200.losses import ContrastLoss
        torch.manual_seed(0)
        crit = ContrastLoss(ablation=False, pretrained=False, device=dev)     # frozen VGG19, seed 0 (SURVEY 8c / 8d config 2)
    ts = training.TrainStep(model, (batch, 3, 128, 128), autocast_dtype=torch.bfloat16 if dtype == "bf16" else None,
                            contrast=contrast, contrast_loss=crit, graph=graph, device=dev)
    g = torch.Generator().manual_seed(1234 + rank)
    x = torch.rand(batch, 3, 128, 128, generator=g).to(dev)
    y = torch.rand(batch, 3, 128, 128, generator=g).to(dev)
    for _ in range(max(warmup, 1)):
        ts.step(x, y)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ts.step(x, y)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    res = dict(step_ms=float(ms.item()), patches_per_s=batch * world / (float(ms.item()) / 1e3), batch_per_gpu=batch, n_gpus=world,
               embed_dim=embed_dim, dtype=dtype, loss=ts.loss(),
               loss_terms="Charbonnier + ContrastLoss (VGG19 random init, p / n passes batched under no_grad, channels-last bf16)"
               if contrast else "Charbonnier only",
               optimizer="AdamW(2e-4, wd 0.02)", parallelism="ddp" if world > 1 else "single", launch=ts.launch_mode,
               api="lewin_b200.training.TrainStep")
    return res, rank


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("batch", type=int, nargs="?", default=32)
    ap.add_argument("--embed-dim", type=int, default=32, choices=(32, 64))
    args = ap.parse_args()
    r, rank = run(batch=args.batch, embed_dim=args.embed_dim)
    if rank == 0:
        print(json.dumps(r), flush=True)
