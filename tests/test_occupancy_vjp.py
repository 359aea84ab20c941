"""Differentiable occupancy grid: ExplicitLoss.soft_occupancy and its vector-Jacobian product (sq_occupancy_vjp).

The VJP is held per sample against the fp64 reference VJP (autograd through the oracle's ExplicitLoss.occupancy), fed the
same fp32-rounded upstream g.  Entry j of grad_params[b] must be within
    1e-4 |ref| + 5e-9 n^3 max|g_b| + 1e-6 sum_vox |g_b d occ / d theta_j|.
The second term is the loss path's 1e-6 when g is ExplicitLoss's own upstream 200 (o_p - o_t) / n^3 at B = 1.  The third
is the fp32 floor of a sum over the grid: an entry that cancels over the whole field -- the translation and rotation
entries of the soft volume (constant g), 1e-5 of the size entries -- cannot be resolved better than a few fp32 roundings
of the sum of the magnitudes of its terms.  Autograd through the reference itself in fp32 misses the first two terms alone
by 3-5x there.  Each case reports the worst entry in units of the first two
terms and of all three.

CPU tests: the host build of the VJP (tests/emu/emu_occ_vjp.cpp) against the oracle.  GPU tests (-m gpu): the CUDA path
against the oracle, the fused loss, the voxel-fitting harness, and the workspace / graph contracts.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import sq_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu_occ_vjp_lib as EV     # noqa: E402

RANDOM = ("random_s4_b8_r8.npz", "random_s1_b6_r16.npz", "random_s2_b4_r32.npz", "random_s3_b2_r64.npz")
K = 5.0


def cases():
    """(label, pred, true, R) of the comparison with the oracle."""
    out = []
    for fname in RANDOM:
        g = load_golden(fname)
        for tag in ("far", "near"):
            out.append((f"{fname}:{tag}", g[f"pred_{tag}"], g["true"], int(g["R"])))
    g = load_golden("edge.npz")                              # clamp boundaries; R = 24: n = R + 2
    out.append(("edge", g["pred"], g["true"], int(g["R"])))
    out.append(("edge pred24", g["pred24"], g["true24"], 24))
    g = load_golden("edge_zero_planes.npz")                  # the planes of exact zeros (fix-up)
    out.append(("zero planes", g["pred"], g["true"], int(g["R"])))
    return out


def grid(R):
    return len(O.explicit_axis(R)), 1.0 / R, 1e-4       # n, step, z0


class Reference:
    """The oracle's occupancy of `pred` (fp64, with autograd history) and what the tolerance needs of it."""

    def __init__(self, pred, R):
        self.R = R
        self.crit = O.ExplicitLoss(R, "cpu")
        self.p = torch.tensor(np.asarray(pred, dtype=np.float64), requires_grad=True)
        self.occ = self.crit.occupancy(self.p)
        self.o = self.occ.detach().numpy()
        self._jac = None

    def vjp(self, go):
        ref, = torch.autograd.grad(self.occ, self.p, torch.tensor(go, dtype=torch.float64), retain_graph=True)
        return ref.numpy()

    def jac(self):
        """d occ / d theta_j for every voxel (12 forward-mode passes), (12, B, n, n, n)."""
        if self._jac is None:
            p = self.p.detach()
            cols = []
            for j in range(12):
                t = torch.zeros_like(p)
                t[:, j] = 1.0
                cols.append(torch.func.jvp(self.crit.occupancy, (p,), (t,))[1].numpy())
            self._jac = np.stack(cols)
        return self._jac

    def condition(self, go):
        """sum_vox |g d occ / d theta_j| per sample and entry, (B, 12)."""
        g = np.abs(np.asarray(go, dtype=np.float64))
        return np.stack([(g * np.abs(J)).reshape(g.shape[0], -1).sum(axis=1) for J in self.jac()], axis=1)


def vjp_errors(grad, ref, go, cond):
    """Worst entry of |grad - ref| in units of (rtol + atol) and of the whole per-sample tolerance (<= 1 passes)."""
    B, n = go.shape[0], go.shape[-1]
    atol = 5e-9 * n ** 3 * np.abs(np.asarray(go, dtype=np.float64)).reshape(B, -1).max(axis=1)[:, None]
    d = np.abs(np.asarray(grad, dtype=np.float64) - ref)
    base = atol + 1e-4 * np.abs(ref)
    e_base, e_all = d / base, d / (base + 1e-6 * cond)
    for e in (e_base, e_all):
        e[(base == 0) & (d == 0)] = 0.0
    return float(e_base.max()), float(e_all.max())


def upstreams(o, o_true, seed):
    """The upstreams, fp32, (B, n, n, n): Gaussian; ExplicitLoss-shaped 200 (o_p - o_t) / n^3; 90 % zeros; one voxel on
    the object; constant (the soft volume); +1 on the shell o (1 - o) in [2^-34, 2^-20] (one sign beyond the loss path's
    cut: what a cut drops there adds up)."""
    rng = np.random.RandomState(seed)
    B, n = o.shape[0], o.shape[-1]
    single = np.zeros(o.shape)
    for b in range(B):
        on = np.argwhere(o[b] > 0.5)
        i = tuple(on[rng.randint(len(on))]) if len(on) else (n // 2, n // 2, n // 2)
        single[(b,) + i] = rng.choice((-1.0, 1.0)) * rng.uniform(0.5, 2.0)
    w = o * (1.0 - o)
    out = {"gauss": rng.randn(*o.shape), "loss": 200.0 * (o - o_true) / n ** 3,
           "sparse": rng.randn(*o.shape) * (rng.uniform(size=o.shape) < 0.1), "single": single,
           "constant": np.ones(o.shape), "shell": ((w >= 2.0 ** -34) & (w <= 2.0 ** -20)).astype(np.float64)}
    return {k: v.astype(np.float32) for k, v in out.items()}


def case_upstreams(pred, true, R):
    ref = Reference(pred, R)
    o_true = O.ExplicitLoss(R, "cpu").occupancy(torch.tensor(np.asarray(true, dtype=np.float64))).numpy()
    return ref, upstreams(ref.o, o_true, R)


def rounded(pred, dtype):
    return np.asarray(pred, dtype=np.float32 if dtype == "fp32" else np.float64).astype(np.float64)


# ------------------------------------------------------------------ CPU: host build of the kernel core
@pytest.mark.parametrize("dtype", ["fp32", "fp64"])
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_emulated_vjp_matches_oracle(case, dtype):
    label, pred, true, R = case
    n, step, z0 = grid(R)
    # the reference is fed the parameters the kernel sees (fp32: the rounded ones; the edge goldens sit on clamp boundaries)
    p_in = rounded(pred, dtype)
    ref, gos = case_upstreams(p_in, true, R)
    worst = []
    for name, go in gos.items():
        gr = EV.occupancy_vjp(p_in, go, n, step, z0, K)
        e_base, e_all = vjp_errors(gr, ref.vjp(go), go, ref.condition(go))
        worst.append(f"{name} {e_base:.3g}/{e_all:.3g}")
        assert e_all <= 1.0, (label, dtype, name, e_base, e_all)
    print(f"\n[occupancy vjp, host] {label} {dtype}: " + ", ".join(worst))


def test_emulated_cut_is_below_the_tolerance():
    """The shell upstream sits entirely below the loss path's cut (2^-24); the VJP's cut (2^-36) keeps all of it, and
    cutting at 2^-28 would lose more than the whole tolerance there: the test can tell the cut."""
    g = load_golden("random_s1_b6_r16.npz")
    R = int(g["R"])
    n, step, z0 = grid(R)
    ref, gos = case_upstreams(g["pred_near"], g["true"], R)
    go = gos["shell"]
    want, cond = ref.vjp(go), ref.condition(go)
    assert vjp_errors(EV.occupancy_vjp(g["pred_near"], go, n, step, z0, K), want, go, cond)[1] <= 0.01
    assert vjp_errors(EV.occupancy_vjp(g["pred_near"], go, n, step, z0, K, bits=28.0), want, go, cond)[1] > 1.0


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def S():
    import sq_recovery_b200 as pkg
    return pkg


def cuda_vjp(crit, pred, go, dev, dtype=torch.float32, split=False, transposed=False):
    """d <soft_occupancy(p), go> / d p through the public path; `split`: p is a non-leaf torch.cat of head-like pieces;
    `transposed`: the upstream arrives as a non-contiguous view."""
    base = torch.as_tensor(np.asarray(pred)).to(dev, dtype)
    if split:
        pieces = [t.clone().requires_grad_(True) for t in torch.split(base, (3, 2, 3, 4), dim=1)]
        p = torch.cat(pieces, dim=1)
    else:
        pieces = [base.clone().requires_grad_(True)]
        p = pieces[0]
    occ = crit.soft_occupancy(p)
    g = torch.as_tensor(go).to(dev)
    if transposed:
        g = g.transpose(1, 3).contiguous().transpose(1, 3)
        assert not g.is_contiguous()
    occ.backward(g)
    grad = torch.cat([q.grad for q in pieces], dim=1)
    assert grad.dtype == dtype
    return grad.double().cpu().numpy()


@pytest.mark.gpu
def test_soft_occupancy_is_the_forward_only_field(dev, S):
    B, R = 6, 32
    pred = O.random_params(B, 11).to(dev)
    crit = S.ExplicitLoss(R, dev)
    p = pred.clone().requires_grad_(True)
    occ = crit.soft_occupancy(p)
    assert occ.requires_grad and occ.shape == (B, R + 1, R + 1, R + 1) and occ.dtype == torch.float32
    assert torch.equal(occ.detach(), crit.occupancy(pred))
    with torch.no_grad():
        assert not crit.soft_occupancy(p).requires_grad
    assert not crit.soft_occupancy(pred).requires_grad
    assert torch.equal(crit.soft_occupancy(pred), crit.occupancy(pred))
    with pytest.raises(RuntimeError, match="soft_occupancy"):
        crit.occupancy(p)


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_cuda_vjp_matches_oracle(case, dev, S):
    label, pred, true, R = case
    crit = S.ExplicitLoss(R, dev)
    for dtype in (torch.float32, torch.float64):
        p_in = rounded(pred, "fp32" if dtype == torch.float32 else "fp64")
        ref, gos = case_upstreams(p_in, true, R)
        worst = []
        for i, (name, go) in enumerate(gos.items()):
            gr = cuda_vjp(crit, p_in, go, dev, dtype, split=(i % 2 == 0), transposed=(i % 2 == 1))
            e_base, e_all = vjp_errors(gr, ref.vjp(go), go, ref.condition(go))
            worst.append(f"{name} {e_base:.3g}/{e_all:.3g}")
            assert e_all <= 1.0, (label, dtype, name, e_base, e_all)
        print(f"\n[occupancy vjp, cuda] {label} {dtype}: " + ", ".join(worst))


@pytest.mark.gpu
def test_soft_occupancy_mse_equals_the_fused_loss(dev, S):
    B, R = 16, 32
    true, pred = O.random_params(B, 31), O.perturbed_params(O.random_params(B, 31), 32)
    crit = S.ExplicitLoss(R, dev)
    p = pred.double().clone().requires_grad_(True)
    ref = O.ExplicitLoss(R, "cpu")(true.double(), p)
    ref.backward()
    p1 = pred.to(dev).clone().requires_grad_(True)
    l1 = 100.0 * ((crit.soft_occupancy(p1) - crit.occupancy(true.to(dev))) ** 2).mean()
    l1.backward()
    p2 = pred.to(dev).clone().requires_grad_(True)
    l2 = crit(true.to(dev), p2)
    l2.backward()
    assert abs(l1.item() - l2.item()) <= 1e-5 * abs(l2.item())
    for g in (p1.grad, p2.grad):
        err = np.abs(g.double().cpu().numpy() - p.grad.numpy()) / (1e-6 + 1e-4 * np.abs(p.grad.numpy()))
        assert err.max() <= 1.0, err.max()


@pytest.mark.gpu
def test_vjp_exact_zeros(dev, S):
    B, R = 8, 64
    pred = O.random_params(B, 41)
    pred[:, 0:3] = 0.06                                       # small objects near the centre
    pred[:, 5:8] = 0.5
    crit = S.ExplicitLoss(R, dev)
    n = R + 1
    zero = torch.zeros(B, n, n, n)
    assert (cuda_vjp(crit, pred, zero, dev) == 0).all()
    corner = torch.zeros(B, n, n, n)
    corner[:, :8, :8, :8] = torch.randn(B, 8, 8, 8)           # upstream only on voxels far outside the culled ranges
    assert (cuda_vjp(crit, pred, corner, dev) == 0).all()


@pytest.mark.gpu
def test_vjp_workspace_contract_and_determinism(dev, S):
    B, R = 12, 32
    true, pred = O.random_params(B, 51).to(dev), O.perturbed_params(O.random_params(B, 51), 52).to(dev)
    crit = S.ExplicitLoss(R, dev)
    go = torch.randn(B, R + 1, R + 1, R + 1, device=dev)

    def vjp():
        p = pred.clone().requires_grad_(True)
        crit.soft_occupancy(p).backward(go)
        return p.grad

    def fused():
        p = pred.clone().requires_grad_(True)
        l = crit(true, p)
        l.backward()
        return l.detach().clone(), p.grad

    alone_v, alone_f = vjp(), fused()
    # forward, fused loss, VJP backward, fused loss: the VJP reads nothing the forward left in the workspace
    p = pred.clone().requires_grad_(True)
    occ = crit.soft_occupancy(p)
    f1 = fused()
    occ.backward(go)
    f2 = fused()
    assert torch.equal(p.grad, alone_v)
    for l, g in (f1, f2):
        assert torch.equal(l, alone_f[0]) and torch.equal(g, alone_f[1])
    assert torch.equal(vjp(), alone_v)                        # bit-identical run to run


@pytest.mark.gpu
def test_vjp_cuda_graph(dev, S):
    B, R = 16, 32
    pred = O.random_params(B, 61).to(dev)
    crit = S.ExplicitLoss(R, dev)
    vox = (crit.occupancy(O.random_params(B, 62).to(dev)) > 0.5).float()
    p0 = pred.clone().requires_grad_(True)
    ((crit.soft_occupancy(p0) - vox) ** 2).mean().backward()
    from sq_recovery_b200 import functional as Fn
    s = torch.cuda.Stream(dev)
    Fn.prepare_stream(dev, B, R + 1, s)
    s.wait_stream(torch.cuda.current_stream(dev))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    p = pred.clone().requires_grad_(True)
    with torch.cuda.graph(g, stream=s):
        ((crit.soft_occupancy(p) - vox) ** 2).mean().backward()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(p.grad, p0.grad)


@pytest.mark.gpu
def test_vjp_large_batch(dev, S):
    """B = 1024: the plan kernel's 128-thread block path; a subset of samples against the oracle."""
    B, R = 1024, 16
    n = R + 1
    pred = O.random_params(B, 71)
    go = np.random.RandomState(72).randn(B, n, n, n).astype(np.float32)
    gr = cuda_vjp(S.ExplicitLoss(R, dev), pred, go, dev)
    idx = np.arange(0, B, 97)
    ref = Reference(pred.numpy()[idx].astype(np.float64), R)
    assert vjp_errors(gr[idx], ref.vjp(go[idx]), go[idx], ref.condition(go[idx]))[1] <= 1.0


@pytest.mark.gpu
def test_voxel_descent_follows_the_oracle(dev, S):
    """harness/optimize.py --loss voxels: a few descent steps on a voxel target through soft_occupancy land where the
    same steps through the fp64 oracle's autograd land, and the loss goes down."""
    from harness import optimize
    B, R, steps = 5, 32, 6
    true = O.random_params(B, 41)
    start = O.perturbed_params(O.random_params(B, 41), 4, sigma=0.05)
    crit = S.ExplicitLoss(R, dev)
    vox = optimize.voxelize(crit, true.to(dev))
    ref = start.clone().double()
    optimize.descend(optimize.VoxelLoss(O.ExplicitLoss(R, "cpu").occupancy), vox.cpu().double(), ref, steps)
    got = start.clone().to(dev)
    rec = []
    optimize.descend(optimize.VoxelLoss(crit.soft_occupancy), vox, got, steps, record=rec)
    assert rec[-1].item() < rec[0].item()
    np.testing.assert_allclose(got.cpu().double().numpy(), ref.numpy(), rtol=0, atol=2e-6)


@pytest.mark.gpu
def test_vjp_against_the_live_reference(dev, S):
    from oracle import ref_import
    if not (ref_import.available() or ref_import.staged()):
        pytest.skip("reference not staged under oracle/_ref (python -m oracle.build_ref in the dev container)")
    rc, _ = ref_import.load()
    R, B = 16, 6
    n = R + 1
    pred = O.random_params(B, 81)
    go = np.random.RandomState(82).randn(B, n, n, n).astype(np.float32)
    p = pred.double().clone().requires_grad_(True)
    occ = rc.ExplicitLoss(R, torch.device("cpu")).occupancy(p)
    want, = torch.autograd.grad(occ, p, torch.tensor(go, dtype=torch.float64))
    gr = cuda_vjp(S.ExplicitLoss(R, dev), pred, go, dev)
    cond = Reference(pred.numpy().astype(np.float64), R).condition(go)
    assert vjp_errors(gr, want.numpy(), go, cond)[1] <= 1.0
