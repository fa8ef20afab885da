"""torchrun harness (launched by tests/test_eval_gpu.py on 2 and 4 GPUs): Trainer.evaluate over W ranks -- uniform
strips, halo rows exchanged between neighbouring strips, (views,3,3) sums all-reduced -- equals a one-rank evaluation
of the same scene on every rank's own GPU.  Cases: 400x400 views, 1060-row views (the last tile row holds 4 rows), and
distributed_dataset_storage=True (only rank 0 holds the ground truth).  Prints "[mgpu-eval] PASS" on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "grendel-gs_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from gs_b200 import pipeline, synthetic as syn  # noqa: E402


def case(rank, world, dev, W, H, n, views, bs, distributed):
    scene = syn.make_scene(n, W, H, seed=3)
    train_cams = syn.make_batch_cameras(W, H, 2)
    tgts = [torch.from_numpy(syn.make_gt_image(W, H, seed=k)).pin_memory() for k in range(2)]
    cams = [syn.make_camera(W, H, yaw_deg=2.5 * k - 4.0, uid=50 + k) for k in range(views)]
    gts = [torch.from_numpy(syn.make_gt_image(W, H, seed=70 + k)) for k in range(views)]
    multi = pipeline.Trainer(scene, train_cams, tgts if not distributed or rank == 0 else None, dev, rank, world,
                             distributed_dataset_storage=distributed)
    single = pipeline.Trainer(scene, train_cams, tgts, dev, 0, 1)
    worst = 0.0
    for protocol in ("report", "saved"):
        got = multi.evaluate(cams, gts if not distributed or rank == 0 else None, batch_size=bs, protocol=protocol)
        ref = single.evaluate(cams, gts, batch_size=bs, protocol=protocol)
        for g, r in zip(got["per_view"], ref["per_view"]):
            worst = max(worst, abs(g["l1"] / r["l1"] - 1), abs(g["ssim"] - r["ssim"]), abs(g["psnr"] - r["psnr"]) / 10)
    return worst


def main():
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda", torch.cuda.current_device())
    ok = True
    for name, args in (("400x400 uniform", (400, 400, 50_000, 6, 4, False)),
                       ("1060 rows (4-row last tile row)", (608, 1060, 80_000, 5, 4, False)),
                       ("distributed dataset storage", (400, 400, 50_000, 6, 4, True))):
        worst = case(rank, world, dev, *args)
        t = torch.tensor([worst], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        worst = float(t.item())
        if rank == 0:
            print(f"[mgpu-eval] W={world} {name}: worst relative difference to one rank {worst:.2e}", flush=True)
        ok = ok and worst <= 1e-6
    if rank == 0:
        print("[mgpu-eval] PASS" if ok else "[mgpu-eval] FAIL", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
