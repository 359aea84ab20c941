#!/usr/bin/env python
"""Batched superquadric refinement by gradient descent -- the loop of torch/visu.py:120-186 without the GUI, run for
thousands of SQs at once (SURVEY 8f-4).

    python harness/optimize.py [--pairs 4096] [--steps 200] [--render 32] [--loss explicit|implicit|voxels|voxels-fused]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 harness/optimize.py

Per step and per SQ, exactly the reference's update (visu.py:176-186): params[:8] -= lr * grad[:8];
q -= lr * grad[8:]; q <- q / |q|, with lr = 0.001 and the loss ExplicitLoss(render_size=32) (visu.py:71).  The reference
optimises ONE pair (batch 1); here every pair must see the gradient of ITS OWN loss, so the batch-mean loss the classes
return is scaled back by the batch size.  Pairs are sharded over the ranks; no collective during the descent.
--loss voxels fits to voxel data instead of ground-truth parameters: the target is the binarised occupancy
(occupancy(true) > 0.5) on ExplicitLoss(R)'s grid, the criterion 100 mean((soft_occupancy(pred) - voxels)^2) (VoxelLoss).
--loss voxels-fused is the same objective through ExplicitLoss.voxel_loss: the target is that grid as bool (read as bytes),
loss and gradient are one fused walk, and no occupancy grid is held in memory.
Prints one JSON line on rank 0: steps/s, loss evaluations (grid points) per second, IoU(128) before / after.
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LR = 0.001                                                  # visu.py:120


def descend(crit, true, pred, steps, lr=LR, record=None):
    """`steps` updates of visu.py:176-186 for every row of `pred` (modified in place); returns the last batch-mean loss.
    `crit(true, pred)` is any of the loss classes (or anything with their call signature); true = targets of that loss."""
    B = pred.shape[0]
    loss = None
    for _ in range(steps):
        p = pred.detach().requires_grad_(True)
        loss = crit(true, p)
        loss.backward()
        with torch.no_grad():
            g = p.grad * B                                  # d (own loss) / d (own params)
            pred[:, :8] -= lr * g[:, :8]
            q = pred[:, 8:] - lr * g[:, 8:]
            pred[:, 8:] = q / q.norm(dim=1, keepdim=True)   # helpers.normalize (visu.py:179)
        if record is not None:
            record.append(loss.detach())
    return loss


class VoxelLoss:
    """100 mean((occupancy(pred) - voxels)^2) over the batch and the grid, with the call signature of the loss classes:
    crit(voxels, pred).  `occupancy` maps (B, 12) parameters to a differentiable (B, n, n, n) occupancy grid --
    ExplicitLoss.soft_occupancy, or the oracle's ExplicitLoss.occupancy; `voxels` is the target grid on the same points."""

    def __init__(self, occupancy):
        self.occupancy = occupancy

    def __call__(self, voxels, pred):
        return 100.0 * ((self.occupancy(pred) - voxels) ** 2).mean()


def voxelize(explicit_loss, params):
    """Binarised occupancy (occupancy > 0.5, i.e. F < 1) of `params` on `explicit_loss`'s grid, fp32 (B, n, n, n)."""
    with torch.no_grad():
        return (explicit_loss.occupancy(params) > 0.5).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--render", type=int, default=32)
    ap.add_argument("--loss", default="explicit", choices=["explicit", "implicit", "voxels", "voxels-fused"])
    args = ap.parse_args()
    import sq_recovery_b200 as S
    from sq_recovery_b200 import distributed as D
    from sq_recovery_b200 import inputs as O          # seeded randsq / randquat workloads
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    b0, b1 = D.shard_range(args.pairs, rank, world)
    true = O.random_params(args.pairs, 0)[b0:b1].to(dev)
    pred = O.perturbed_params(O.random_params(args.pairs, 0), 3, sigma=0.05)[b0:b1].to(dev)     # start near, like a CNN guess
    R = args.render
    if args.loss == "explicit":
        crit, target, pts = S.ExplicitLoss(R, dev), true, (b1 - b0) * (R + 1) ** 3
    elif args.loss == "voxels":
        grid = S.ExplicitLoss(R, dev)
        crit, target, pts = VoxelLoss(grid.soft_occupancy), voxelize(grid, true), (b1 - b0) * grid._n ** 3
    elif args.loss == "voxels-fused":
        grid = S.ExplicitLoss(R, dev)
        crit, target, pts = grid.voxel_loss, voxelize(grid, true).bool(), (b1 - b0) * grid._n ** 3
    else:
        crit = S.ImplicitLoss(R, dev, 1.5, 260)
        target = S.ImplicitLoss(256, dev, 1.5, 260).depth_projection(true).unsqueeze(1).contiguous()
        pts = (b1 - b0) * R ** 3
    iou = S.IoUAccuracy(128, dev)
    i0, u0 = iou.counts(true, pred)
    descend(crit, target, pred.clone(), 3)                  # warm-up on a copy
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rec = []
    e0.record()
    descend(crit, target, pred, args.steps, record=rec)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    i1, u1 = iou.counts(true, pred)
    stats = torch.stack([i0.sum(), u0.sum(), i1.sum(), u1.sum()]).double()
    losses = torch.stack(rec).double()
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats)
        dist.all_reduce(losses); losses /= world
    if rank == 0:
        s = ms.item() * 1e-3
        print(json.dumps({
            "harness": "optimize", "n_gpus": world, "pairs": args.pairs, "loss": args.loss, "render_size": R,
            "steps": args.steps, "steps_per_s": args.steps / s, "ms_per_step": s / args.steps * 1e3,
            "gpoints_per_s": world * pts * args.steps / s / 1e9,
            "loss_first": losses[0].item(), "loss_last": losses[-1].item(),
            "iou128_before": (stats[0] / stats[1]).item(), "iou128_after": (stats[2] / stats[3]).item(),
            "finite": bool(torch.isfinite(pred).all().item())}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
