"""Cost of the depth-render Jacobian (ImplicitLoss.render_jacobian / render_normal_equations) next to the render and its
VJP, and the Levenberg-Marquardt fit it makes possible against plain descent and the LeastSquares fit.

    python tools/render_jacobian_bench.py [--steps 100] [--warmup 10] [--out FILE]

Shape: BASELINE config 2 (B = 256, R = 64, tau = 1.5, k = 260, 256 x 256 depth maps), on the headline workload and on `dense`
(the input sets of tools/render_vjp_bench.py).  Every step is a CUDA graph per input set, replayed back to back; CUDA events
over `steps` replays after `warmup`.  Reports, microseconds per call:
  depth_projection   crit.depth_projection(p)                          (sq_implicit_loss, forward-only render)
  vjp                the render's VJP alone                             (sq_depth_projection_vjp)
  render_jacobian    crit.render_jacobian(p)                            (sq_depth_projection_jacobian)
  normal_equations   crit.render_normal_equations(img, p)               (the above + one batched fp64 matmul in torch)
  fused              crit(img, p).backward()                            (sq_implicit_loss, loss + gradient)
and the column kernel of the Jacobian call alone (sq_profile_events).  Then harness/optimize.py on 4096 pairs at R = 32:
--loss implicit --method lm (20 iterations), --loss implicit (gd, 200 steps), --loss lsq --method lm (20 iterations), each
one JSON line from its own process.  Prints one JSON document; the card's name and power limit are read in the same run
(nvidia-smi --query-gpu, read-only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import sq_recovery_b200 as S                      # noqa: E402
from sq_recovery_b200 import inputs as I          # noqa: E402
from render_vjp_bench import B, R, SHARP, TAU, Sets, card, column_kernel_us, steps_of, time_graphs     # noqa: E402


def fit(loss, method, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "harness", "optimize.py"), "--loss", loss, "--method", method,
                          "--steps", str(steps)], capture_output=True, text=True, check=True, cwd=ROOT)
    return json.loads(out.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("render_jacobian_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "config": {"B": B, "R": R, "image": 256, "tau": TAU, "k": SHARP, "input_sets": 4,
                                      "steps": args.steps, "warmup": args.warmup},
           "timing": "CUDA events over graph replays (one graph per input set), microseconds per call",
           "jac_bytes": B * R * R * 48}
    crit = S.ImplicitLoss(R, dev, TAU, SHARP)
    for name, size_range in (("headline", I.SIZE_RANGE), ("dense", I.DENSE_SIZE_RANGE)):
        sets = Sets(size_range, dev).sets
        base, _ = steps_of(crit, sets, dev)

        def depth_projection(k):
            crit.depth_projection(sets[k][2])

        def render_jacobian(k):
            crit.render_jacobian(sets[k][2])

        def normal_equations(k):
            crit.render_normal_equations(sets[k][0], sets[k][2])

        fns = {"depth_projection": depth_projection, "vjp": base["vjp"], "render_jacobian": render_jacobian,
               "normal_equations": normal_equations, "fused": base["fused"]}
        res[name] = {"call_us": {k: time_graphs(f, dev, args.steps, args.warmup) for k, f in fns.items()},
                     "jacobian_column_kernel_us": column_kernel_us(render_jacobian)}
        c = res[name]["call_us"]
        res[name]["ratios"] = {"render_jacobian_over_vjp": c["render_jacobian"] / c["vjp"],
                               "render_jacobian_over_depth_projection": c["render_jacobian"] / c["depth_projection"]}
    res["fit"] = {"implicit_lm": fit("implicit", "lm", 20), "implicit_gd": fit("implicit", "gd", 200),
                  "lsq_lm": fit("lsq", "lm", 20)}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
