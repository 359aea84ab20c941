"""Fused voxel loss: ExplicitLoss.voxel_loss and its C entry point sq_voxel_loss.

Per sample, against the fp64 reference l_b = mult mean_vox (v_b - o_b)^2 through the oracle's ExplicitLoss.occupancy (with
autograd history), fed the fp32 voxel values and the parameters the kernel sees:
  loss:      |l_b - ref_b| <= 1e-6 ref_b + 1e-10 mult
  gradient:  the occupancy VJP's contract (tests/test_occupancy_vjp.py) applied to the loss's own upstream
             g_b = 2 mult (o_b - v_b) / n^3:  1e-4 |ref| + 5e-9 n^3 max|g_b| + 1e-6 sum_vox |g_b d o / d theta_j|.
Each case reports its worst loss and gradient entries in units of the tolerance.

CPU tests: the host build (tests/emu/emu_voxel.cpp) against the oracle, and the cut.  GPU tests (-m gpu): the CUDA path
against the oracle, the byte / float / layout equalities, the soft and fused paths, errors, and the workspace, graph and
large-batch contracts.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import sq_oracle as O
from test_occupancy_vjp import Reference, cases, grid, rounded, vjp_errors

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu_voxel_lib as EX     # noqa: E402

K, MULT = 5.0, 100.0
RANDOM = ("random_s4_b8_r8.npz", "random_s1_b6_r16.npz", "random_s2_b4_r32.npz", "random_s3_b2_r64.npz")


def targets(o, o_true, seed):
    """The voxel targets, fp32 (B, n, n, n): binarised and soft occupancy of the true SQ; binarised occupancy of pred itself
    (near convergence: the loss is small against sum v^2); uniform noise (nonzero far outside the walk); zeros; ones; a
    block disjoint from the object; 1 on the shell o (1 - o) in [2^-34, 2^-20] (one sign below the loss path's cut)."""
    rng = np.random.RandomState(seed)
    n = o.shape[-1]
    w = o * (1.0 - o)
    block = np.zeros(o.shape)
    m = max(n // 3, 1)
    block[:, :m, :m, :m] = 1.0
    block[o >= 2.0 ** -40] = 0.0
    out = {"bin true": o_true > 0.5, "soft true": o_true, "bin pred": o > 0.5, "noise": rng.uniform(size=o.shape),
           "zeros": np.zeros(o.shape), "ones": np.ones(o.shape), "block": block,
           "shell": (w >= 2.0 ** -34) & (w <= 2.0 ** -20)}
    return {k: np.asarray(v, dtype=np.float32) for k, v in out.items()}


def case_targets(pred, true, R):
    ref = Reference(pred, R)
    o_true = O.ExplicitLoss(R, "cpu").occupancy(torch.tensor(np.asarray(true, dtype=np.float64))).numpy()
    return ref, targets(ref.o, o_true, R)


def reference(ref, vox):
    """Per-sample loss (B,), its gradient (B, 12), the upstream g_b and the condition term of the tolerance."""
    n3 = vox.shape[-1] ** 3
    v = vox.astype(np.float64)
    loss = MULT * ((v - ref.o) ** 2).reshape(len(v), -1).sum(axis=1) / n3
    g = 2.0 * MULT * (ref.o - v) / n3
    return loss, ref.vjp(g), g, ref.condition(g)


def loss_error(loss, want):
    """Worst |loss - want| in units of 1e-6 want + 1e-10 mult."""
    return float((np.abs(np.asarray(loss) - want) / (1e-6 * want + 1e-10 * MULT)).max())


def check(label, ref, vox, loss, grad):
    want, gwant, g, cond = reference(ref, vox)
    e_loss = loss_error(loss, want)
    e_grad = vjp_errors(grad, gwant, g, cond)[1]
    assert e_loss <= 1.0 and e_grad <= 1.0, (label, e_loss, e_grad)
    return f"{e_loss:.3g}/{e_grad:.3g}"


# ------------------------------------------------------------------ CPU: host build of the kernel core
@pytest.mark.parametrize("dtype", ["fp32", "fp64"])
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_emulated_voxel_loss_matches_oracle(case, dtype):
    label, pred, true, R = case
    n, step, z0 = grid(R)
    p_in = rounded(pred, dtype)
    ref, vox = case_targets(p_in, true, R)
    worst = []
    for name, v in vox.items():
        loss, gr = EX.voxel_loss(p_in, v, n, step, z0, K, MULT)
        worst.append(f"{name} " + check((label, dtype, name), ref, v, loss, gr))
    print(f"\n[voxel loss, host] {label} {dtype} (loss/grad): " + ", ".join(worst))


@pytest.mark.parametrize("fname", RANDOM[:3])
def test_emulated_cut(fname):
    """The shell target lies entirely below the loss path's cut (2^-24), with one sign.  What a cut drops is measured against
    a walk cut at 2^-64 (nothing of the shell dropped), in units of the gradient tolerance: at 2^-36 it is below 1e-3; at
    2^-28 it is 0.006-0.01 and at 2^-24 more than rtol + atol alone, so the test can tell the cut.  (Unlike the occupancy
    VJP's shell upstream, the loss's own upstream always carries the object's term 2 mult o / n^3 where v = 0, whose size
    sets the tolerance: a 2^-28 cut would still pass the contract here; DESIGN.md 3.)"""
    g = load_golden(fname)
    R = int(g["R"])
    n, step, z0 = grid(R)
    ref, vox = case_targets(g["pred_near"], g["true"], R)
    v = vox["shell"]
    want, gwant, up, cond = reference(ref, v)
    loss, gr = EX.voxel_loss(g["pred_near"], v, n, step, z0, K, MULT)
    assert loss_error(loss, want) <= 1.0 and vjp_errors(gr, gwant, up, cond)[1] <= 1.0
    _, full = EX.voxel_loss(g["pred_near"], v, n, step, z0, K, MULT, bits=64.0)
    dropped = {bits: vjp_errors(EX.voxel_loss(g["pred_near"], v, n, step, z0, K, MULT, bits=bits)[1], full, up, cond)
               for bits in (24.0, 28.0, 36.0)}
    assert dropped[36.0][1] <= 1e-3 < 3e-3 < dropped[28.0][1]
    assert dropped[24.0][0] > 1.0


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


def c_voxel_loss(crit, vox, p, per_sample=True, grad=True, dtype_tag=None):
    """sq_voxel_loss called directly: (return code, batch-mean loss, per-sample losses, gradient of the batch mean)."""
    from sq_recovery_b200 import _lib
    from sq_recovery_b200 import functional as Fn
    dev = p.device
    B, n = p.shape[0], crit._n
    pc, tag = Fn._params(p)
    v, vtag, scale = Fn._voxels(vox, B, n, None)
    loss = torch.empty((), dtype=torch.float64, device=dev)
    per = torch.empty(B, dtype=torch.float64, device=dev) if per_sample else None
    gr = torch.empty_like(pc) if grad else None
    scratch = Fn._get_scratch(dev, B, n)
    rc = _lib.lib().sq_voxel_loss(Fn._ptr(v), vtag if dtype_tag is None else dtype_tag, scale, Fn._ptr(pc), tag, B, n,
                                  crit._step, crit._z0, K, MULT, Fn._ptr(loss), Fn._ptr(per), Fn._ptr(gr),
                                  Fn._ptr(scratch), scratch.numel(), Fn._stream(dev))
    torch.cuda.synchronize()
    return rc, loss, per, gr


def public_voxel_loss(crit, vox, pred, dev, dtype):
    """crit.voxel_loss with a non-leaf pred (torch.cat of head-like pieces): (loss, gradient of the batch mean)."""
    base = torch.as_tensor(np.asarray(pred)).to(dev, dtype)
    pieces = [t.clone().requires_grad_(True) for t in torch.split(base, (3, 2, 3, 4), dim=1)]
    p = torch.cat(pieces, dim=1)
    loss = crit.voxel_loss(vox, p)
    loss.backward()
    grad = torch.cat([q.grad for q in pieces], dim=1)
    assert grad.dtype == dtype and loss.dtype == torch.float64 and loss.dim() == 0
    return loss.detach(), grad


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_cuda_voxel_loss_matches_oracle(case, dev, S):
    label, pred, true, R = case
    crit = S.ExplicitLoss(R, dev)
    for dtype in (torch.float32, torch.float64):
        p_in = rounded(pred, "fp32" if dtype == torch.float32 else "fp64")
        ref, vox = case_targets(p_in, true, R)
        worst = []
        for name, v in vox.items():
            vt = torch.as_tensor(v).to(dev)
            loss, grad = public_voxel_loss(crit, vt, p_in, dev, dtype)
            rc, l_c, per, g_c = c_voxel_loss(crit, vt, torch.as_tensor(p_in).to(dev, dtype))
            assert rc == 0
            assert torch.equal(loss, l_c) and torch.equal(grad, g_c)          # the public path is this call
            B = len(p_in)
            worst.append(f"{name} " + check((label, dtype, name), ref, v, per.cpu().numpy(),
                                            grad.double().cpu().numpy() * B))
        print(f"\n[voxel loss, cuda] {label} {dtype} (loss/grad): " + ", ".join(worst))


@pytest.mark.gpu
def test_voxel_dtypes_and_layouts_are_bit_identical(dev, S):
    B, R = 8, 32
    n = R + 1
    crit = S.ExplicitLoss(R, dev)
    pred = O.perturbed_params(O.random_params(B, 21), 22, sigma=0.05).to(dev)
    b = crit.occupancy(O.random_params(B, 21).to(dev)) > 0.5
    u8 = torch.randint(0, 256, (B, n, n, n), dtype=torch.uint8, generator=torch.Generator().manual_seed(23)).to(dev)

    def run(v, **kw):
        p = pred.clone().requires_grad_(True)
        loss = crit.voxel_loss(v, p, **kw)
        loss.backward()
        return loss.detach(), p.grad

    def same(a, c):
        assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])

    same(run(b), run(b.float()))
    same(run(u8), run(u8.float() * np.float32(1 / 255)))
    same(run(u8, voxel_scale=0.5), run(u8.float() * 0.5))
    same(run(b.double()), run(b.float()))
    v = torch.rand(B, n, n, n, device=dev)
    vt = v.transpose(1, 3).contiguous().transpose(1, 3)
    assert not vt.is_contiguous()
    same(run(vt), run(v))
    bt = b.transpose(1, 2).contiguous().transpose(1, 2)
    same(run(bt), run(b))


@pytest.mark.gpu
def test_voxel_loss_equals_the_soft_path(dev, S):
    """100 ((soft_occupancy(p) - v)^2).mean() backward: the same loss to 1e-6 and a gradient within the contract."""
    B, R = 16, 32
    crit = S.ExplicitLoss(R, dev)
    true, pred = O.random_params(B, 31), O.perturbed_params(O.random_params(B, 31), 32)
    vox = (crit.occupancy(true.to(dev)) > 0.5).float()
    p1 = pred.to(dev).clone().requires_grad_(True)
    l1 = 100.0 * ((crit.soft_occupancy(p1) - vox) ** 2).mean()
    l1.backward()
    p2 = pred.to(dev).clone().requires_grad_(True)
    l2 = crit.voxel_loss(vox.bool(), p2)
    l2.backward()
    assert abs(l1.item() - l2.item()) <= 1e-6 * abs(l1.item())
    ref = Reference(pred.numpy().astype(np.float32).astype(np.float64), R)
    _, gwant, g, cond = reference(ref, vox.cpu().numpy())
    for gr in (p1.grad, p2.grad):
        assert vjp_errors(gr.double().cpu().numpy() * B, gwant, g, cond)[1] <= 1.0


@pytest.mark.gpu
def test_soft_target_equals_the_fused_loss(dev, S):
    """Voxels = the soft occupancy of `true`: the objective of ExplicitLoss(true, p) (as in
    test_soft_occupancy_mse_equals_the_fused_loss)."""
    B, R = 16, 32
    true, pred = O.random_params(B, 31), O.perturbed_params(O.random_params(B, 31), 32)
    crit = S.ExplicitLoss(R, dev)
    p = pred.double().clone().requires_grad_(True)
    ref = O.ExplicitLoss(R, "cpu")(true.double(), p)
    ref.backward()
    p1 = pred.to(dev).clone().requires_grad_(True)
    l1 = crit.voxel_loss(crit.occupancy(true.to(dev)), p1)
    l1.backward()
    p2 = pred.to(dev).clone().requires_grad_(True)
    l2 = crit(true.to(dev), p2)
    l2.backward()
    assert abs(l1.item() - l2.item()) <= 1e-5 * abs(l2.item())
    for g in (p1.grad, p2.grad):
        err = np.abs(g.double().cpu().numpy() - p.grad.numpy()) / (1e-6 + 1e-4 * np.abs(p.grad.numpy()))
        assert err.max() <= 1.0, err.max()


@pytest.mark.gpu
def test_loss_does_not_depend_on_grad_mode(dev, S):
    B, R = 12, 32
    crit = S.ExplicitLoss(R, dev)
    pred = O.random_params(B, 35).to(dev)
    for vox in (crit.occupancy(O.random_params(B, 36).to(dev)) > 0.5, torch.rand(B, R + 1, R + 1, R + 1, device=dev)):
        p = pred.clone().requires_grad_(True)
        with_grad = crit.voxel_loss(vox, p)
        with_grad.backward()
        with torch.no_grad():
            no_grad = crit.voxel_loss(vox, p)
        plain = crit.voxel_loss(vox, pred)
        assert not no_grad.requires_grad and not plain.requires_grad
        assert torch.equal(no_grad, with_grad.detach()) and torch.equal(plain, with_grad.detach())


@pytest.mark.gpu
def test_voxel_loss_errors(dev, S):
    B, R = 4, 16
    n = R + 1
    crit = S.ExplicitLoss(R, dev)
    pred = O.random_params(B, 37).to(dev).requires_grad_(True)
    vox = torch.zeros(B, n, n, n, device=dev)
    with pytest.raises(RuntimeError, match="soft_occupancy"):
        crit.voxel_loss(vox.clone().requires_grad_(True), pred)
    with torch.no_grad():
        crit.voxel_loss(vox.clone().requires_grad_(True), pred)          # nothing to differentiate: accepted
    for bad in (torch.zeros(B, n, n, n + 1, device=dev), torch.zeros(B, n + 1, n + 1, n + 1, device=dev),
                torch.zeros(B + 1, n, n, n, device=dev), torch.zeros(B, n, n, device=dev)):
        with pytest.raises(ValueError):
            crit.voxel_loss(bad, pred)
    for v in (vox, vox.bool(), vox.double()):
        with pytest.raises(ValueError, match="voxel_scale"):
            crit.voxel_loss(v, pred, voxel_scale=0.5)
    cudaErrorInvalidValue = 1
    p = pred.detach()
    assert c_voxel_loss(crit, vox, p, dtype_tag=1)[0] == cudaErrorInvalidValue       # SQ_F64 voxels: not a voxel type
    assert c_voxel_loss(crit, vox, p, dtype_tag=7)[0] == cudaErrorInvalidValue
    from sq_recovery_b200 import _lib
    from sq_recovery_b200 import functional as Fn
    scratch = Fn._get_scratch(dev, B, n)
    L = _lib.lib()
    for vp, pp in ((None, Fn._ptr(p)), (Fn._ptr(vox), None)):
        rc = L.sq_voxel_loss(vp, _lib.SQ_F32, 1.0, pp, _lib.SQ_F32, B, n, crit._step, crit._z0, K, MULT, None, None, None,
                             Fn._ptr(scratch), scratch.numel(), Fn._stream(dev))
        assert rc == cudaErrorInvalidValue
    assert c_voxel_loss(crit, vox, p)[0] == 0                            # the workspace is still good


@pytest.mark.gpu
def test_voxel_loss_workspace_contract_and_determinism(dev, S):
    B, R = 12, 32
    true, pred = O.random_params(B, 51).to(dev), O.perturbed_params(O.random_params(B, 51), 52).to(dev)
    crit = S.ExplicitLoss(R, dev)
    render = S.ImplicitLoss(R, dev, 1.5, 260)
    vox = (crit.occupancy(true) > 0.5)
    go = torch.randn(B, R + 1, R + 1, R + 1, device=dev)

    def vl():
        p = pred.clone().requires_grad_(True)
        loss = crit.voxel_loss(vox, p)
        loss.backward()
        return loss.detach().clone(), p.grad

    alone = vl()
    # soft_occupancy forward, voxel loss, render, fused loss, VJP backward, voxel loss: nothing is read across calls
    p = pred.clone().requires_grad_(True)
    occ = crit.soft_occupancy(p)
    r1 = vl()
    pr = pred.clone().requires_grad_(True)
    render.render(pr).sum().backward()
    crit(true, pred.clone().requires_grad_(True)).backward()
    occ.backward(go)
    r2 = vl()
    for r in (r1, r2, vl()):                                              # the last one: run to run
        assert torch.equal(r[0], alone[0]) and torch.equal(r[1], alone[1])


@pytest.mark.gpu
def test_voxel_loss_cuda_graph(dev, S):
    B, R = 16, 32
    pred = O.random_params(B, 61).to(dev)
    crit = S.ExplicitLoss(R, dev)
    vox = crit.occupancy(O.random_params(B, 62).to(dev)) > 0.5
    p0 = pred.clone().requires_grad_(True)
    l0 = crit.voxel_loss(vox, p0)
    l0.backward()
    from sq_recovery_b200 import functional as Fn
    s = torch.cuda.Stream(dev)
    Fn.prepare_stream(dev, B, R + 1, s)
    s.wait_stream(torch.cuda.current_stream(dev))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    p = pred.clone().requires_grad_(True)
    with torch.cuda.graph(g, stream=s):
        loss = crit.voxel_loss(vox, p)
        loss.backward()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(loss, l0) and torch.equal(p.grad, p0.grad)


@pytest.mark.gpu
def test_voxel_loss_large_batch(dev, S):
    """B = 1024: the plan kernel's 128-thread block path; a subset of samples against the oracle."""
    B, R = 1024, 16
    n = R + 1
    crit = S.ExplicitLoss(R, dev)
    pred = O.random_params(B, 71)
    vox = np.random.RandomState(72).uniform(size=(B, n, n, n)).astype(np.float32)
    vox[: B // 2] = vox[: B // 2] > 0.5
    p = pred.to(dev)
    rc, _, per, gr = c_voxel_loss(crit, torch.as_tensor(vox).to(dev), p)
    assert rc == 0
    idx = np.arange(0, B, 97)
    ref = Reference(pred.numpy()[idx].astype(np.float32).astype(np.float64), R)
    check("B = 1024", ref, vox[idx], per.cpu().numpy()[idx], gr.double().cpu().numpy()[idx] * B)


@pytest.mark.gpu
def test_voxel_descent_follows_the_soft_path(dev, S):
    """harness/optimize.py --loss voxels-fused: a few descent steps through voxel_loss land where the same steps through
    soft_occupancy land, and the loss goes down."""
    from harness import optimize
    B, R, steps = 5, 32, 6
    true = O.random_params(B, 41)
    start = O.perturbed_params(O.random_params(B, 41), 4, sigma=0.05)
    crit = S.ExplicitLoss(R, dev)
    vox = optimize.voxelize(crit, true.to(dev))
    soft = start.clone().to(dev)
    optimize.descend(optimize.VoxelLoss(crit.soft_occupancy), vox, soft, steps)
    fused = start.clone().to(dev)
    rec = []
    optimize.descend(crit.voxel_loss, vox.bool(), fused, steps, record=rec)
    assert rec[-1].item() < rec[0].item()
    np.testing.assert_allclose(fused.cpu().double().numpy(), soft.cpu().double().numpy(), rtol=0, atol=2e-6)
