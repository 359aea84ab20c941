"""Cost of the fused voxel loss (ExplicitLoss.voxel_loss) next to the fused loss on true parameters and the soft path.

    python tools/voxel_loss_bench.py [--steps 100] [--warmup 10] [--out FILE]

Two shapes: BASELINE config 2's explicit workload (B = 256, R = 64, n = 65: 281 MB per fp32 grid, above the 126 MB of L2)
and config 1's (B = 32, R = 32); then voxel_loss alone with bool voxels at 4096 x 129^3 (R = 128: 8.8 GB of voxels, 35 GB
per fp32 grid).  Predictions perturbed from seeded true parameters, the target the binarised occupancy of the true ones;
4 input sets rotated (2 at the large shape).  Every step is a CUDA graph per input set, replayed back to back; CUDA events
over `steps` replays after `warmup`.  Reports, per step:
  fused        crit(true, p).backward()                                    (the fused ExplicitLoss, one walk)
  soft_mse     100 mean((crit.soft_occupancy(p) - voxels)^2).backward()    (field + torch MSE + VJP)
  voxel_f32    crit.voxel_loss(voxels, p).backward(), fp32 voxels          (one walk)
  voxel_bool   the same with bool voxels (read as bytes)
the column kernel of each (sq_profile_events, eager), the voxel bytes the fused voxel loss reads (every voxel once) over its
column kernel time, and the peak torch.cuda.max_memory_allocated of one eager step above what the inputs hold.  Prints one
JSON document; the card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import sq_recovery_b200 as S                      # noqa: E402
from sq_recovery_b200 import inputs as I          # noqa: E402
from occupancy_vjp_bench import card, column_kernel_us, time_graphs     # noqa: E402

SHAPES = (("config2", 256, 64), ("config1", 32, 32))
LARGE = ("large", 4096, 128)
HBM_TBS = 7.7


def steps_of(crit, sets):
    """name -> function(k) running one step on input set k through the public API."""
    def fused(k):
        true, pred, _ = sets[k]
        crit(true, pred.detach().requires_grad_(True)).backward()

    def soft_mse(k):
        _, pred, vox = sets[k]
        p = pred.detach().requires_grad_(True)
        (100.0 * ((crit.soft_occupancy(p) - vox["f32"]) ** 2).mean()).backward()

    def voxel(kind):
        def run(k):
            _, pred, vox = sets[k]
            crit.voxel_loss(vox[kind], pred.detach().requires_grad_(True)).backward()
        return run

    return {"fused": fused, "soft_mse": soft_mse, "voxel_f32": voxel("f32"), "voxel_bool": voxel("bool")}


def peak_mb(fn, dev):
    """Peak allocation of one eager step above what was allocated before it, MB."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    fn(0)
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated(dev) - base) / 1e6


def voxelize(crit, true, chunk=256):
    """Binarised occupancy of `true`, bool, built in chunks (the fp32 grid of a large batch is not held at once)."""
    with torch.no_grad():
        return torch.cat([crit.occupancy(true[i:i + chunk]) > 0.5 for i in range(0, true.shape[0], chunk)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("voxel_loss_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "steps": args.steps, "warmup": args.warmup,
           "timing": "CUDA events over graph replays (one graph per input set), microseconds per step; column kernels: "
                     "eager, sq_profile_events; peak_MB: torch.cuda.max_memory_allocated of one eager step above the inputs"}
    for name, B, R in SHAPES:
        crit = S.ExplicitLoss(R, dev)
        n = crit._n
        sets = []
        for k in range(4):
            true = I.random_params(B, 100 + k).to(dev)
            pred = I.perturbed_params(I.random_params(B, 100 + k), 200 + k).to(dev)
            b = voxelize(crit, true)
            sets.append((true, pred, {"bool": b, "f32": b.float()}))
        fns = steps_of(crit, sets)
        r = {"B": B, "R": R, "n": n, "grid_MB_fp32": B * n ** 3 * 4 / 1e6}
        r["step_us"] = {k: time_graphs(f, B, n, dev, args.steps, args.warmup) for k, f in fns.items()}
        r["column_kernel_us"] = {k: column_kernel_us(fns[k]) for k in ("fused", "voxel_f32", "voxel_bool")}
        r["peak_MB"] = {k: peak_mb(f, dev) for k, f in fns.items()}
        r["voxel_read"] = {}
        for kind, size in (("f32", 4), ("bool", 1)):
            nbytes = B * n ** 3 * size
            t = r["column_kernel_us"][f"voxel_{kind}"] * 1e-6
            r["voxel_read"][kind] = {"bytes": nbytes, "TBs": nbytes / t / 1e12, "share_of_7.7TBs": nbytes / t / 1e12 / HBM_TBS}
        res[name] = r
        del sets, fns
        torch.cuda.empty_cache()
    name, B, R = LARGE
    crit = S.ExplicitLoss(R, dev)
    n = crit._n
    sets = []
    for k in range(2):
        true = I.random_params(B, 300 + k).to(dev)
        pred = I.perturbed_params(I.random_params(B, 300 + k), 400 + k).to(dev)
        sets.append((true, pred, {"bool": voxelize(crit, true)}))
    run = steps_of(crit, sets)["voxel_bool"]
    steps = max(2, args.steps // 10)
    r = {"B": B, "R": R, "n": n, "voxels_GB_bool": B * n ** 3 / 1e9, "grid_GB_fp32": B * n ** 3 * 4 / 1e9,
         "steps": steps, "input_sets": 2}
    r["step_us"] = {"voxel_bool": time_graphs(lambda k: run(k % 2), B, n, dev, steps, 2)}
    r["column_kernel_us"] = {"voxel_bool": column_kernel_us(lambda k: run(k % 2), n=6)}
    r["peak_MB"] = {"voxel_bool": peak_mb(run, dev)}
    t = r["column_kernel_us"]["voxel_bool"] * 1e-6
    r["voxel_read"] = {"bool": {"bytes": B * n ** 3, "TBs": B * n ** 3 / t / 1e12}}
    res[name] = r
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
