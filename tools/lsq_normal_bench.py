"""Cost of LeastSquares' normal equations (normal_equations / normal_equations_points) next to the loss + gradient they extend
and to the only other way to get J^T J, and the Levenberg-Marquardt fit they make possible against plain descent.

    python tools/lsq_normal_bench.py [--steps 100] [--warmup 10] [--oracle FILE] [--out FILE]

Shape: B = 256, R = 64 on 256^2 depth images (renders of seeded random SQs; predictions perturbed from them, sigma 0.05);
4 input sets rotated.  Every step is a CUDA graph per input set, replayed back to back; CUDA events over `steps` replays after
`warmup`.  Reports, microseconds per call:
  image_loss_grad      LeastSquares(R)(img, p).backward()                   (sq_least_squares, loss + gradient)
  image_normal         LeastSquares(R).normal_equations(img, p)             (sq_least_squares_normal)
  points_energy_grad   energy_function's LsqEnergyFn(p, packed).sum().backward()  (sq_least_squares_points, the image's points)
  points_normal        normal_equations_points' call on the same packed lists     (sq_least_squares_points_normal)
  oracle_jacobian      the fp64 oracle's J^T J for the 256 samples on the same GPU: measured by the test tool
                       tests/tools/oracle_jacobian_timing.py (the product's tools do not run the oracle) and merged from
                       its JSON line with --oracle
Then the fits of harness/optimize.py --loss lsq (4096 pairs, R = 32): --method gd (200 steps, its default) and --method lm
(20 iterations), each one JSON line from its own process.  Prints one JSON document; the card's name and power limit are
read in the same run (nvidia-smi --query-gpu, read-only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import sq_recovery_b200 as S                      # noqa: E402
from sq_recovery_b200 import functional as Fn     # noqa: E402
from sq_recovery_b200 import inputs as I          # noqa: E402
from occupancy_vjp_bench import card, time_graphs     # noqa: E402

B, R, IMG = 256, 64, 256


def points(img, R):
    """The (3, m_i) point lists LeastSquares(R) builds from (B, 1, H, W) depth images (classes.py:359-369)."""
    t = F.interpolate(img, size=(R, R), mode="nearest")
    out = []
    for i in range(img.shape[0]):
        rc = torch.where(t[i][0] > 0)
        x, y = rc[0].float() / R, rc[1].float() / R
        out.append(torch.stack([y, 1 - x, t[i][0][rc]]))
    return out


def fit(method, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "harness", "optimize.py"), "--loss", "lsq", "--method", method,
                          "--steps", str(steps)], capture_output=True, text=True, check=True, cwd=ROOT)
    return json.loads(out.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--oracle", default=None, help="JSON line of tests/tools/oracle_jacobian_timing.py")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lsq_normal_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "steps": args.steps, "warmup": args.warmup, "input_sets": 4, "B": B, "R": R, "image": IMG,
           "timing": "CUDA events over graph replays (one graph per input set), microseconds per call; oracle: host clock "
                     "around synchronised eager work (tests/tools/oracle_jacobian_timing.py)"}
    ls = S.LeastSquares(R, dev)
    render = S.ImplicitLoss(IMG, dev, 1.5, 260)
    sets = []
    for k in range(4):
        true = I.random_params(B, 500 + k).to(dev)
        pred = I.perturbed_params(I.random_params(B, 500 + k), 600 + k, sigma=0.05).to(dev)
        img = render.depth_projection(true).unsqueeze(1).contiguous()
        pts = points(img, R)
        sets.append((img, pred, Fn.pack_points(pts, dev)))    # packed once: the timed calls copy nothing to the device
    res["points_per_sample_mean"] = sets[0][2][1][-1].item() / B

    def image_loss_grad(k):
        img, pred, _ = sets[k]
        ls(img, pred.detach().requires_grad_(True)).backward()

    def image_normal(k):
        img, pred, _ = sets[k]
        ls.normal_equations(img, pred)

    def points_energy_grad(k):
        _, pred, packed = sets[k]
        Fn.LsqEnergyFn.apply(pred.detach().requires_grad_(True), *packed).sum().backward()

    def points_normal(k):
        _, pred, packed = sets[k]
        Fn.lsq_points_normal_packed(pred, *packed)

    fns = {"image_loss_grad": image_loss_grad, "image_normal": image_normal, "points_energy_grad": points_energy_grad,
           "points_normal": points_normal}
    res["call_us"] = {k: time_graphs(f, B, R, dev, args.steps, args.warmup) for k, f in fns.items()}
    c = res["call_us"]
    res["ratios"] = {"image_normal_over_loss_grad": c["image_normal"] / c["image_loss_grad"],
                     "points_normal_over_energy_grad": c["points_normal"] / c["points_energy_grad"]}
    if args.oracle:
        with open(args.oracle) as f:
            c["oracle_jacobian"] = json.loads(f.read().strip().splitlines()[-1])["oracle_jacobian_us"]
        res["ratios"]["oracle_over_image_normal"] = c["oracle_jacobian"] / c["image_normal"]
    res["fit"] = {"gd": fit("gd", 200), "lm": fit("lm", 20)}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
