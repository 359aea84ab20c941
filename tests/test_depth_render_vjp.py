"""Differentiable depth render: ImplicitLoss.render and its vector-Jacobian product (sq_depth_projection_vjp).

The VJP is held per sample: every entry of grad_pred[b] within rtol 1e-4 and atol 1e-6 n^2 max|grad_depth[b]| of the fp64
reference VJP (autograd through the oracle's depth_projection), fed the same fp32-rounded upstream.  For the MAE upstream
+-1/n^2 of a single sample this is the loss path's contract at batch 1.

CPU tests: the host build of the kernel core's VJP mode (tests/emu/emu_vjp.cpp) against the oracle, and bit-equality with the loss path where every
scaling is exact.  GPU tests (-m gpu): the CUDA path against the oracle, the fused loss, and the workspace / graph contracts.
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from oracle import sq_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu_lib as E          # noqa: E402
import emu_vjp_lib as EV     # noqa: E402

RANDOM = ("random_s4_b8_r8.npz", "random_s1_b6_r16.npz", "random_s2_b4_r32.npz", "random_s3_b2_r64.npz")
TAU_K = ((1.5, 260.0), (1.0, 100.0))


def vjp_error(grad, ref, go):
    """Worst entry of |grad - ref| in units of the per-sample tolerance (<= 1 passes)."""
    B, n = go.shape[0], go.shape[-1]
    atol = 1e-6 * n * n * np.abs(np.asarray(go, dtype=np.float64)).reshape(B, -1).max(axis=1)[:, None]
    err = np.abs(np.asarray(grad, dtype=np.float64) - ref) / (atol + 1e-4 * np.abs(ref))
    err[np.broadcast_to(atol == 0, err.shape) & (grad == ref)] = 0.0
    return float(err.max())


def upstreams(depth, target, seed):
    """The upstreams of the issue, fp32, (B, n, n): Gaussian; MSE-shaped 2 (d - t) / (n^2 B); 90 % zeros; one pixel."""
    rng = np.random.RandomState(seed)
    B, n = depth.shape[0], depth.shape[-1]
    gauss = rng.randn(B, n, n)
    sparse = rng.randn(B, n, n) * (rng.uniform(size=(B, n, n)) < 0.1)
    single = np.zeros((B, n, n))
    for b in range(B):        # a pixel on the object, so that the VJP is not trivially 0
        on = np.argwhere(depth[b] > 1e-3)
        r, c = on[rng.randint(len(on))] if len(on) else (n // 2, n // 2)
        single[b, r, c] = rng.choice((-1.0, 1.0)) * rng.uniform(0.5, 2.0)
    out = {"gauss": gauss, "mse": 2.0 * (depth - target) / (n * n * B), "sparse": sparse, "single": single}
    return {k: v.astype(np.float32) for k, v in out.items()}


def oracle_vjps(pred, R, tau, k, gos):
    """{name: fp64 VJP} through autograd on the oracle's render, one graph for all upstreams."""
    p = torch.tensor(np.asarray(pred, dtype=np.float64), requires_grad=True)
    d = O.ImplicitLoss(R, "cpu", tau, k).depth_projection(p)
    out = {}
    for i, (name, go) in enumerate(gos.items()):
        out[name], = torch.autograd.grad(d, p, torch.tensor(go, dtype=torch.float64), retain_graph=i + 1 < len(gos))
        out[name] = out[name].numpy()
    return d.detach().numpy(), out


def resized(img, R):
    return F.interpolate(torch.tensor(img).float(), size=(R, R), mode="nearest")[:, 0].numpy()


def cpu_cases():
    """(label, pred, target (B,R,R), R, tau, k) of the emulator-vs-oracle comparison."""
    cases = []
    for fname in RANDOM:
        g = load_golden(fname)
        R = int(g["R"])
        tgt = resized(g["img"], R)
        for tag in ("far", "near"):
            for tau, k in TAU_K:
                cases.append((f"{fname}:{tag}:{tau}/{k}", g[f"pred_{tag}"], tgt, R, tau, k))
    g = load_golden("random_s2_b4_r32.npz")                  # a soft sigmoid on a fine grid, reduced batch
    cases.append(("soft k=20 R=96", g["pred_near"][:2], resized(g["img"][:2], 96), 96, 1.0, 20.0))
    g = load_golden("edge.npz")                              # clamped parameters
    cases.append(("edge", g["pred"], resized(g["img"], int(g["R"])), int(g["R"]), 1.5, 260.0))
    g = load_golden("edge_zero_planes.npz")
    R = int(g["R"])
    cases.append(("zero planes", g["pred"], resized(g["img"], R), R, 1.5, 260.0))
    cases.append(("zero planes soft", g["pred"], resized(g["img"], R), R, 1.0, 20.0))
    g = load_golden("edge_grazing.npz")
    cases.append(("grazing", g["pred"], resized(g["img"], int(g["R"])), int(g["R"]), float(g["tau"]), float(g["k"])))
    return cases


# ------------------------------------------------------------------ CPU: host build of the kernel core
@pytest.mark.parametrize("case", cpu_cases(), ids=lambda c: c[0])
def test_emulated_vjp_matches_oracle(case):
    label, pred, tgt, R, tau, k = case
    depth = E.implicit(pred, None, R, 1 / (R - 1), 1e-4, tau, k, want_grad=False, want_depth=True)[2]
    gos = upstreams(depth.astype(np.float64), tgt, R)
    _, refs = oracle_vjps(pred, R, tau, k, gos)
    for name, go in gos.items():
        gr = EV.depth_vjp(pred, go, R, 1 / (R - 1), 1e-4, tau, k)
        assert vjp_error(gr, refs[name], go) <= 1.0, (label, name, vjp_error(gr, refs[name], go))


@pytest.mark.parametrize("fname", ["random_s1_b6_r16.npz", "random_s2_b4_r32.npz", "random_s3_b2_r64.npz"])
def test_emulated_vjp_of_the_mae_is_the_loss_gradient(fname):
    """B = 1, n a power of two, upstream sign(d - t) / n^2 from the emulator's own depth: 1/n^2, the finalize scales
    k tau / n vs k tau / n^3 and the weight cut (batch 1 in both) make every scaling exact, so the VJP is the fused loss
    path's gradient bit for bit."""
    g = load_golden(fname)
    R = int(g["R"])
    tgt = resized(g["img"], R)
    for tag in ("far", "near"):
        for tau, k in TAU_K:
            for b in range(len(g[f"pred_{tag}"])):
                pred, t = g[f"pred_{tag}"][b:b + 1], tgt[b:b + 1]
                _, want, depth = E.implicit(pred, t, R, 1 / (R - 1), 1e-4, tau, k, want_depth=True)
                go = (np.sign(depth - t) / (R * R)).astype(np.float32)
                got = EV.depth_vjp(pred, go, R, 1 / (R - 1), 1e-4, tau, k)
                assert np.array_equal(got, want), (tag, tau, k, b, np.abs(got - want).max())


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
    """d <render(p), go> / d p through the public path; `split`: p is a non-leaf torch.cat of head-like pieces;
    `transposed`: the upstream arrives as a non-contiguous (transposed) view."""
    base = torch.as_tensor(np.asarray(pred)).to(dev, dtype)
    if split:
        pieces = [t.clone().requires_grad_(True) for t in torch.split(base, (3, 2, 3, 4), dim=1)]
        p = torch.cat(pieces, dim=1)
    else:
        pieces = [base.clone().requires_grad_(True)]
        p = pieces[0]
    d = crit.render(p)
    g = torch.as_tensor(go).to(dev)
    if transposed:
        g = g.transpose(1, 2).contiguous().transpose(1, 2)
        assert not g.is_contiguous()
    d.backward(g)
    grad = torch.cat([q.grad for q in pieces], dim=1)
    assert grad.dtype == dtype
    return grad.double().cpu().numpy()


@pytest.mark.gpu
def test_render_is_the_forward_only_render(dev, S):
    B, R = 6, 32
    pred = O.random_params(B, 11).to(dev)
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    p = pred.clone().requires_grad_(True)
    d = crit.render(p)
    assert d.requires_grad and d.shape == (B, R, R) and d.dtype == torch.float32
    assert torch.equal(d.detach(), crit.depth_projection(pred))
    with torch.no_grad():
        assert not crit.render(p).requires_grad
    assert not crit.render(pred).requires_grad
    with pytest.raises(RuntimeError, match="forward-only"):
        crit.depth_projection(p)


@pytest.mark.gpu
@pytest.mark.parametrize("case", cpu_cases(), ids=lambda c: c[0])
def test_cuda_vjp_matches_oracle(case, dev, S):
    label, pred, tgt, R, tau, k = case
    depth, _ = oracle_vjps(pred, R, tau, k, {})
    gos = upstreams(depth, tgt, R)
    crit = S.ImplicitLoss(R, dev, tau, k)
    for dtype in (torch.float32, torch.float64):
        # the reference is fed the parameters the kernel sees (the edge goldens sit on clamp boundaries in fp64)
        p_in = np.asarray(pred, dtype=np.float32 if dtype == torch.float32 else np.float64).astype(np.float64)
        _, refs = oracle_vjps(p_in, R, tau, k, gos)
        for i, (name, go) in enumerate(gos.items()):
            gr = cuda_vjp(crit, p_in, go, dev, dtype, split=(i % 2 == 0), transposed=(i % 2 == 1))
            err = vjp_error(gr, refs[name], go)
            assert err <= 1.0, (label, name, dtype, err)


@pytest.mark.gpu
def test_render_mae_equals_the_fused_loss(dev, S):
    B, R = 16, 32
    true, pred = O.random_params(B, 31), O.perturbed_params(O.random_params(B, 31), 32)
    img = S.ImplicitLoss(2 * R, dev, 1.5, 260).depth_projection(true.to(dev)).unsqueeze(1).contiguous()
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    oc = O.ImplicitLoss(R, "cpu", 1.5, 260)
    p = pred.double().clone().requires_grad_(True)
    ref = oc(img.cpu(), p)
    ref.backward()
    keep = np.asarray(unambiguous(oc, img.cpu(), pred))
    assert keep.sum() >= B // 2
    t = F.interpolate(img, size=(R, R), mode="nearest")
    p1 = pred.to(dev).clone().requires_grad_(True)
    l1 = (crit.render(p1) - t[:, 0]).abs().mean()
    l1.backward()
    p2 = pred.to(dev).clone().requires_grad_(True)
    l2 = crit(img, p2)
    l2.backward()
    assert abs(l1.item() - l2.item()) <= 1e-5 * abs(l2.item())
    for g in (p1.grad, p2.grad):
        err = np.abs(g.double().cpu().numpy() - p.grad.numpy()) / (1e-6 + 1e-4 * np.abs(p.grad.numpy()))
        assert err[keep].max() <= 1.0


def unambiguous(oracle_crit, img, pred):
    with torch.no_grad():
        d = oracle_crit.depth_projection(torch.as_tensor(pred))
        t = oracle_crit.resize(torch.as_tensor(img))[:, 0].double()
    tie = ((d - t).abs() < 1e-6) & (d > 1e-5)
    return ~tie.flatten(1).any(dim=1).numpy()


@pytest.mark.gpu
def test_vjp_exact_zeros(dev, S):
    B, R = 8, 64
    pred = O.random_params(B, 41)
    pred[:, 0:3] = 0.06                                       # small objects near the centre
    pred[:, 5:8] = 0.5
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    d = crit.depth_projection(pred.to(dev))
    assert (d[:, :8, :8] == 0).all()
    zero = torch.zeros(B, R, R)
    assert (cuda_vjp(crit, pred, zero, dev) == 0).all()
    corner = torch.zeros(B, R, R)
    corner[:, :8, :8] = torch.randn(B, 8, 8)                  # upstream only on columns far outside the culled ranges
    assert (cuda_vjp(crit, pred, corner, dev) == 0).all()


@pytest.mark.gpu
def test_vjp_workspace_contract_and_determinism(dev, S):
    B, R = 12, 32
    true, pred = O.random_params(B, 51).to(dev), O.perturbed_params(O.random_params(B, 51), 52).to(dev)
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    img = crit.depth_projection(true).unsqueeze(1).contiguous()
    go = torch.randn(B, R, R, device=dev)

    def vjp():
        p = pred.clone().requires_grad_(True)
        crit.render(p).backward(go)
        return p.grad

    def fused():
        p = pred.clone().requires_grad_(True)
        l = crit(img, p)
        l.backward()
        return l.detach().clone(), p.grad

    alone_v, alone_f = vjp(), fused()
    # render, fused loss, VJP backward, fused loss: the VJP reads nothing the forward left in the workspace
    p = pred.clone().requires_grad_(True)
    d = crit.render(p)
    f1 = fused()
    d.backward(go)
    f2 = fused()
    assert torch.equal(p.grad, alone_v)
    for l, g in (f1, f2):
        assert torch.equal(l, alone_f[0]) and torch.equal(g, alone_f[1])
    assert torch.equal(vjp(), alone_v)                        # bit-identical run to run


@pytest.mark.gpu
def test_vjp_cuda_graph(dev, S):
    B, R = 16, 32
    pred = O.random_params(B, 61).to(dev)
    tgt = S.ImplicitLoss(R, dev, 1.5, 260).depth_projection(O.random_params(B, 62).to(dev))
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    p0 = pred.clone().requires_grad_(True)
    ((crit.render(p0) - tgt) ** 2).mean().backward()
    from sq_recovery_b200 import functional as Fn
    s = torch.cuda.Stream(dev)
    Fn.prepare_stream(dev, B, R, s)
    s.wait_stream(torch.cuda.current_stream(dev))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    p = pred.clone().requires_grad_(True)
    with torch.cuda.graph(g, stream=s):
        ((crit.render(p) - tgt) ** 2).mean().backward()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(p.grad, p0.grad)


@pytest.mark.gpu
def test_vjp_large_batch(dev, S):
    """B = 1024: the plan kernel's 128-thread block path; a subset of samples against the oracle."""
    B, R, tau, k = 1024, 32, 1.5, 260.0
    pred = O.random_params(B, 71)
    go = np.random.RandomState(72).randn(B, R, R).astype(np.float32)
    crit = S.ImplicitLoss(R, dev, tau, k)
    gr = cuda_vjp(crit, pred, go, dev)
    idx = np.arange(0, B, 97)
    _, refs = oracle_vjps(pred.numpy()[idx], R, tau, k, {"g": go[idx]})
    assert vjp_error(gr[idx], refs["g"], go[idx]) <= 1.0


@pytest.mark.gpu
def test_vjp_against_the_live_reference(dev, S):
    from oracle import ref_import
    if not (ref_import.available() or ref_import.staged()):
        pytest.skip("reference not staged under oracle/_ref (python -m oracle.build_ref in the dev container)")
    rc, _ = ref_import.load()
    R, B = 16, 6
    pred = O.random_params(B, 81)
    go = np.random.RandomState(82).randn(B, R, R).astype(np.float32)
    p = pred.double().clone().requires_grad_(True)
    d = rc.ImplicitLoss(R, torch.device("cpu"), 1.5, 260).depth_projection(p)
    ref, = torch.autograd.grad(d, p, torch.tensor(go, dtype=torch.float64))
    gr = cuda_vjp(S.ImplicitLoss(R, dev, 1.5, 260), pred, go, dev)
    assert vjp_error(gr, ref.numpy(), go) <= 1.0
