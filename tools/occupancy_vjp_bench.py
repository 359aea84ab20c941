"""Cost of a custom voxel loss through ExplicitLoss.soft_occupancy (forward field + CUDA VJP) next to the fused loss step.

    python tools/occupancy_vjp_bench.py [--steps 100] [--warmup 10] [--out FILE]

Two shapes: BASELINE config 2's explicit workload (B = 256, R = 64, n = 65: 281 MB per field tensor, above the 126 MB of
L2) and config 1's (B = 32, R = 32).  Predictions perturbed from seeded true parameters, 4 input sets rotated.  Every step
is a CUDA graph per input set, replayed back to back; CUDA events over `steps` replays after `warmup`.  Reports, per step:
  fused        crit(true, p).backward()                                    (the fused ExplicitLoss, one walk)
  soft_mse     100 mean((crit.soft_occupancy(p) - voxels)^2).backward()    (field + torch MSE + VJP)
  vjp          sq_occupancy_vjp alone (plan + column + finalize), and its column kernel (sq_profile_events, eager)
  field        the forward field alone (crit.occupancy)
and the upstream bytes the VJP's walk reads over its column kernel time, against 7.7 TB/s: at least the voxels above the
cut (o (1 - o) >= 2^-36, counted on the field), at most the whole field.  Prints one JSON document; the card's name and
power limit are read in the same run (nvidia-smi --query-gpu, read-only).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import sq_recovery_b200 as S                      # noqa: E402
from sq_recovery_b200 import _lib, functional as Fn, inputs as I     # noqa: E402

SHAPES = (("config2", 256, 64), ("config1", 32, 32))
HBM_TBS = 7.7
CUT = 2.0 ** -36


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                         # noqa: BLE001
        return f"unknown ({e})"


def steps_of(crit, sets, B, dev):
    """name -> function(k) running one step on input set k (public API, and the C entry point for the VJP alone)."""
    n = crit._n
    go = [torch.randn(B, n, n, n, device=dev, generator=torch.Generator(dev).manual_seed(k)) * (200.0 / n ** 3)
          for k in range(4)]
    outs = [torch.empty(B, 12, device=dev) for _ in range(4)]

    def fused(k):
        true, pred, _ = sets[k]
        p = pred.detach().requires_grad_(True)
        crit(true, p).backward()

    def soft_mse(k):
        _, pred, vox = sets[k]
        p = pred.detach().requires_grad_(True)
        (100.0 * ((crit.soft_occupancy(p) - vox) ** 2).mean()).backward()

    def vjp(k):
        pred = sets[k][1]
        sc = Fn._get_scratch(dev, B, n)
        rc = _lib.lib().sq_occupancy_vjp(ctypes.c_void_p(pred.data_ptr()), _lib.SQ_F32, B, n, crit._step, crit._z0, 5.0,
                                         ctypes.c_void_p(go[k].data_ptr()), ctypes.c_void_p(outs[k].data_ptr()),
                                         ctypes.c_void_p(sc.data_ptr()), sc.numel(), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "sq_occupancy_vjp")

    def field(k):
        crit.occupancy(sets[k][1])

    return {"fused": fused, "soft_mse": soft_mse, "vjp": vjp, "field": field}


def time_graphs(fn, B, n, dev, steps, warmup):
    side = torch.cuda.Stream(dev)
    Fn.prepare_stream(dev, B, n, side)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for k in range(4):
            fn(k); fn(k)
    torch.cuda.synchronize()
    graphs = []
    for k in range(4):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fn(k)
        graphs.append(g)
    for i in range(warmup):
        graphs[i % 4].replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for i in range(steps):
        graphs[i % 4].replay()
    b.record()
    torch.cuda.synchronize()
    del graphs
    return a.elapsed_time(b) * 1e3 / steps


def column_kernel_us(fn, n=12):
    ms = []
    for i in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); b.record()
        torch.cuda.synchronize()
        _lib.lib().sq_profile_events(a.cuda_event, b.cuda_event)
        fn(i % 4)
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.mean(ms[2:])) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("occupancy_vjp_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "steps": args.steps, "warmup": args.warmup, "input_sets": 4,
           "timing": "CUDA events over graph replays (one graph per input set), microseconds per step"}
    for name, B, R in SHAPES:
        crit = S.ExplicitLoss(R, dev)
        n = crit._n
        sets = []
        for k in range(4):
            true = I.random_params(B, 100 + k).to(dev)
            pred = I.perturbed_params(I.random_params(B, 100 + k), 200 + k).to(dev)
            sets.append((true, pred, (crit.occupancy(true) > 0.5).float()))
        fns = steps_of(crit, sets, B, dev)
        r = {"B": B, "R": R, "n": n, "field_MB": B * n ** 3 * 4 / 1e6}
        r.update({k: time_graphs(f, B, n, dev, args.steps, args.warmup) for k, f in fns.items()})
        r["vjp_column_kernel"] = column_kernel_us(fns["vjp"])
        r["fused_column_kernel"] = column_kernel_us(fns["fused"])
        with torch.no_grad():
            above = 0.0
            for _, pred, _ in sets:
                o = crit.occupancy(pred)
                above += float(((o * (1 - o)) >= CUT).sum().item())
            above /= len(sets)
        r["voxels_above_cut_fraction"] = above / (B * n ** 3)
        lo, hi = above * 4, B * n ** 3 * 4.0
        t = r["vjp_column_kernel"] * 1e-6
        r["upstream_read"] = {"bytes_at_least": lo, "bytes_at_most": hi, "TBs_at_least": lo / t / 1e12,
                              "TBs_at_most": hi / t / 1e12, "share_of_7.7TBs_at_most": hi / t / 1e12 / HBM_TBS}
        res[name] = r
        del sets, fns
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
