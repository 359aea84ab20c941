"""Cost of a custom image loss through ImplicitLoss.render (forward render + CUDA VJP) next to the fused MAE step.

    python tools/render_vjp_bench.py [--steps 200] [--warmup 20] [--out FILE]

BASELINE config 2 (B = 256, R = 64, tau = 1.5, k = 260, 256 x 256 synthetic depth maps = soft renders of the true
parameters, predictions perturbed from them), 4 input batches rotated so the inputs exceed L2, like bench.py.  Every step
is a CUDA graph per input set, replayed back to back; CUDA events over `steps` replays after `warmup`.  Reports, per step:
  fused       crit(img, p).backward()                        (the fused loss, one walk)
  render_mae  crit.render(p), torch MAE, .backward()         (render + VJP: two walks)
  render_mse  crit.render(p), torch MSE, .backward()
  vjp         sq_depth_projection_vjp alone (plan + column + finalize), and its column kernel (sq_profile_events, eager)
on the headline workload and on `dense` (a ~ U(0.5, 1)), plus the counting build's point counts (queued, refined,
on-the-spot backward blocks) of one VJP call next to one fused call.  Prints one JSON document; the card's name and power
limit are read in the same run (nvidia-smi --query-gpu, read-only).
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
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import sq_recovery_b200 as S                      # noqa: E402
from sq_recovery_b200 import _lib, counting, functional as Fn, inputs as I     # noqa: E402

B, R, H, TAU, SHARP = 256, 64, 256, 1.5, 260.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                         # noqa: BLE001
        return f"unknown ({e})"


class Sets:
    def __init__(self, size_range, dev):
        render = S.ImplicitLoss(H, dev, TAU, SHARP)
        self.sets = []
        for k in range(4):
            true = I.random_params(B, k, size_range=size_range)
            pred = I.perturbed_params(true, 7 + k).to(dev)
            img = render.depth_projection(true.to(dev)).unsqueeze(1).contiguous()
            tgt = F.interpolate(img, size=(R, R), mode="nearest")[:, 0].contiguous()
            self.sets.append((img, tgt, pred))


def steps_of(crit, sets, dev):
    """name -> function(k) running one step on input set k (public API)."""
    go = [torch.randn(B, R, R, device=dev, generator=torch.Generator(dev).manual_seed(k)) / (R * R * B) for k in range(4)]
    scratch = {}

    def fused(k):
        img, _, pred = sets[k]
        p = pred.detach().requires_grad_(True)
        crit(img, p).backward()

    def render_mae(k):
        _, tgt, pred = sets[k]
        p = pred.detach().requires_grad_(True)
        (crit.render(p) - tgt).abs().mean().backward()

    def render_mse(k):
        _, tgt, pred = sets[k]
        p = pred.detach().requires_grad_(True)
        ((crit.render(p) - tgt) ** 2).mean().backward()

    def vjp(k):
        pred = sets[k][2]
        out = scratch.setdefault(("g", k), torch.empty(B, 12, device=dev))
        sc = Fn._get_scratch(dev, B, R)
        rc = _lib.lib().sq_depth_projection_vjp(ctypes.c_void_p(pred.data_ptr()), _lib.SQ_F32, B, R, 1.0 / (R - 1), 1e-4, TAU,
                                                SHARP, ctypes.c_void_p(go[k].data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                ctypes.c_void_p(sc.data_ptr()), sc.numel(), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "sq_depth_projection_vjp")

    return {"fused": fused, "render_mae": render_mae, "render_mse": render_mse, "vjp": vjp}, go


def time_graphs(fn, dev, steps, warmup):
    side = torch.cuda.Stream(dev)
    Fn.prepare_stream(dev, B, R, side)
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


def vjp_counts(pred, go, dev):
    h = counting.lib()
    nb = h.sq_scratch_bytes(B, R)
    scratch = torch.zeros(nb, dtype=torch.uint8, device=dev)
    h.sq_scratch_init(ctypes.c_void_p(scratch.data_ptr()), nb, torch.cuda.current_stream(dev).cuda_stream)
    grad = torch.empty(B, 12, device=dev)
    cnt = (ctypes.c_ulonglong * 8)()
    torch.cuda.synchronize()
    _lib.check(h.sq_debug_counters(cnt, 1), "sq_debug_counters")
    rc = h.sq_depth_projection_vjp(ctypes.c_void_p(pred.data_ptr()), _lib.SQ_F32, B, R, 1.0 / (R - 1), 1e-4, TAU, SHARP,
                                   ctypes.c_void_p(go.data_ptr()), ctypes.c_void_p(grad.data_ptr()),
                                   ctypes.c_void_p(scratch.data_ptr()), nb, torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "sq_depth_projection_vjp (counting build)")
    torch.cuda.synchronize()
    _lib.check(h.sq_debug_counters(cnt, 1), "sq_debug_counters")
    return dict(zip(counting.NAMES, (int(v) for v in cnt)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("render_vjp_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    crit = S.ImplicitLoss(R, dev, TAU, SHARP)
    res = {"card": card(), "config": {"B": B, "R": R, "image": H, "tau": TAU, "k": SHARP, "input_sets": 4,
                                      "steps": args.steps, "warmup": args.warmup},
           "timing": "CUDA events over graph replays (one graph per input set), microseconds per step"}
    for name, size_range in (("headline", I.SIZE_RANGE), ("dense", I.DENSE_SIZE_RANGE)):
        sets = Sets(size_range, dev).sets
        fns, go = steps_of(crit, sets, dev)
        r = {k: time_graphs(f, dev, args.steps, args.warmup) for k, f in fns.items()}
        r["vjp_column_kernel"] = column_kernel_us(fns["vjp"])
        r["fused_column_kernel"] = column_kernel_us(fns["fused"])
        keys = ("queued_points", "refined_points", "spot_backward_blocks", "plane_steps")
        cv = [vjp_counts(p, g, dev) for (_, _, p), g in zip(sets, go)]
        cf = [counting.implicit_counts(img, p, R, TAU, SHARP)["counters"] for img, _, p in sets]
        r["counts_per_call"] = {"vjp": {k: float(np.mean([c[k] for c in cv])) for k in keys},
                                "fused": {k: float(np.mean([c[k] for c in cf])) for k in keys}}
        res[name] = r
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
