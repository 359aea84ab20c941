"""The only other way to get LeastSquares' J^T J: the fp64 oracle's Jacobian by forward-mode autograd through
oracle.sq_oracle.inside_outside_single (12 passes per sample), on the SAME GPU, for tools/lsq_normal_bench.py's workload
(B = 256, R = 64, 256^2 depth renders, the same seeds).  Host clock around synchronised eager work.  Prints one JSON line;
tools/lsq_normal_bench.py --oracle FILE merges it."""
import json
import os
import sys
import time

import torch
import torch.autograd.forward_ad as fwAD

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import sq_oracle as O       # noqa: E402
import sq_recovery_b200 as S            # noqa: E402

dev = torch.device("cuda:0")
B, R = 256, 64


def jtj(p, P):
    def res(q):
        c = O.preprocess_sq(q)
        return torch.sqrt(c[0] * c[1] * c[2]) * (O.inside_outside_single(q, P, True, True) - 1.0)

    eye = torch.eye(12, dtype=torch.float64, device=p.device)
    cols = []
    with fwAD.dual_level():
        for k in range(12):
            cols.append(fwAD.unpack_dual(res(fwAD.make_dual(p, eye[k]))).tangent)
    J = torch.stack(cols, dim=1)
    return J.T @ J


true = O.random_params(B, 500).to(dev)
pred = O.perturbed_params(O.random_params(B, 500), 600, sigma=0.05).to(dev).double()
img = S.ImplicitLoss(256, dev, 1.5, 260).depth_projection(true).unsqueeze(1).contiguous()
pts = [p.to(dev).double() for p in O.LeastSquares(R).points(img.cpu())]
jtj(pred[0], pts[0])
torch.cuda.synchronize()
t0 = time.perf_counter()
for b in range(B):
    jtj(pred[b], pts[b])
torch.cuda.synchronize()
print(json.dumps({"oracle_jacobian_us": (time.perf_counter() - t0) * 1e6, "B": B, "R": R,
                  "what": "fp64 oracle J (forward-mode autograd, 12 passes per sample) and J^T J, 256 samples, eager"}))
