"""Depth-render Jacobian: ImplicitLoss.render_jacobian / render_normal_equations and their C entry point
sq_depth_projection_jacobian.

The reference is the fp64 oracle's Jacobian, by forward-mode autograd (12 tangents) through its depth_projection, on the
parameters the kernel sees (fp32 parameters rounded first).  Row (b, r, c) is the VJP of a unit one-hot upstream on that
pixel, so the per-pixel contract is the render VJP's for that upstream:
  J:      |J - J_ref| <= 1e-4 |J_ref| + 1e-6 n^2                      (entry by entry)
  J^T J:  |H - H_ref|_jk <= sum_pix (t_j |J_ref,k| + |J_ref,j| t_k + t_j t_k),  t = 1e-6 n^2 + 1e-4 |J_ref|
Each case prints its worst entries in units of the tolerance.

CPU tests: the host build (tests/emu/emu_jac.cpp: the group loop of the render VJP's host build with weight 1 and
per-column sums).  GPU tests (-m gpu): the CUDA path through the classes and the C ABI, its agreement with render's VJP
and depth_projection, the normal equations, errors, workspace, determinism, graph capture, large batches and grids, and
the Levenberg-Marquardt fit of harness/optimize.py.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.autograd.forward_ad as fwAD
import torch.nn.functional as F

from conftest import ROOT, load_golden
from harness import optimize
from oracle import sq_oracle as O
from test_depth_render_vjp import cpu_cases, oracle_vjps, resized, upstreams, vjp_error

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu_lib as E          # noqa: E402
import emu_jac_lib as EJ     # noqa: E402
import emu_vjp_lib as EV     # noqa: E402

EINVAL = 1                   # cudaErrorInvalidValue
CASES = cpu_cases()          # the render VJP's cases, the soft k = 20 R = 96 one among them


def oracle_jacobian(pred, R, tau, k):
    """(depth (B, R, R), J (B, R, R, 12)) fp64 through the oracle's depth_projection, one forward-mode pass per parameter."""
    p = torch.tensor(np.asarray(pred, dtype=np.float64))
    crit = O.ImplicitLoss(R, "cpu", tau, k)
    cols = []
    with torch.no_grad():
        for j in range(12):
            tan = torch.zeros_like(p)
            tan[:, j] = 1.0
            with fwAD.dual_level():
                d = crit.depth_projection(fwAD.make_dual(p, tan))
                primal, tangent = fwAD.unpack_dual(d)
                cols.append(tangent)
    return primal.numpy(), torch.stack(cols, -1).numpy()


def jac_error(J, ref):
    n = J.shape[1]
    return float((np.abs(np.asarray(J, np.float64) - ref) / (1e-6 * n * n + 1e-4 * np.abs(ref))).max())


def jtj_error(J, ref):
    B, n = J.shape[0], J.shape[1]
    J, ref = np.asarray(J, np.float64).reshape(B, -1, 12), ref.reshape(B, -1, 12)
    t = 1e-6 * n * n + 1e-4 * np.abs(ref)
    a = np.abs(ref)
    tol = np.einsum("bpj,bpk->bjk", t, a) + np.einsum("bpj,bpk->bjk", a, t) + np.einsum("bpj,bpk->bjk", t, t)
    H, Hr = np.einsum("bpj,bpk->bjk", J, J), np.einsum("bpj,bpk->bjk", ref, ref)
    return float((np.abs(H - Hr) / tol).max())


def check(label, J, ref):
    ej, eh = jac_error(J, ref), jtj_error(J, ref)
    print(f"\n[{label}] worst J entry {ej:.3f}, worst J^T J entry {eh:.3f} of the tolerance")
    assert ej <= 1.0 and eh <= 1.0, (label, ej, eh)


def onehot_pixels(J, rng, count=3):
    """Per sample `count` pixels: rows that are not zero where there are any, and one row that is."""
    out = []
    for b in range(J.shape[0]):
        nz = np.argwhere(np.abs(J[b]).sum(-1) > 0)
        z = np.argwhere(np.abs(J[b]).sum(-1) == 0)
        pick = [tuple(nz[rng.randint(len(nz))]) for _ in range(count - 1)] if len(nz) else []
        if len(z):
            pick.append(tuple(z[rng.randint(len(z))]))
        out.append(pick)
    return out


def small_objects(B=6, seed=41):
    """Small SQs near the centre, with a1 and t_y clamped out (a1 > 1 is clamped to 1, t_y < 0 to 0)."""
    pred = O.random_params(B, seed)
    pred[:, 0] = 1.3
    pred[:, 1:3] = 0.06
    pred[:, 5:8] = 0.5
    pred[:, 6] = -0.2
    return pred.numpy()


def assert_exact_zeros(J, depth):
    assert (depth[:, :8, :8] == 0).all() and (J[:, :8, :8] == 0).all()      # columns far outside every culled range
    assert (J[..., 0] == 0).all() and (J[..., 6] == 0).all()                # clamped-out parameters
    assert (np.abs(J).sum(-1) > 0).any()


def normal_from(J, depth, t):
    r = (np.asarray(depth, np.float64) - t).reshape(len(J), -1)
    J = np.asarray(J, np.float64).reshape(len(J), -1, 12)
    return (r * r).sum(1), 2.0 * np.einsum("bpj,bp->bj", J, r), np.einsum("bpj,bpk->bjk", J, J)


def lm_start():
    """Train-like perturbed starts (sigma 0.02) of random SQs; the target is their 64^2 render resized to 32^2."""
    true = O.random_params(6, 11, torch.float64)
    with torch.no_grad():
        img = O.ImplicitLoss(64, "cpu", 1.5, 260).depth_projection(true).float().unsqueeze(1)
    return O.perturbed_params(true, 5, sigma=0.02), img, resized(img.numpy(), 32).astype(np.float64)


def lm_run(normal, target, p0, iters=10):
    p = p0.clone()
    rec = []
    Ef = optimize.levenberg_marquardt(normal, target, p, iters, record=rec)
    return Ef.cpu().numpy(), [ok.cpu().numpy() for _, ok in rec]


def oracle_normal(t):
    def normal(_, params):
        depth, J = oracle_jacobian(params.numpy(), t.shape[-1], 1.5, 260.0)
        e, g, h = normal_from(J, depth, t)
        return torch.tensor(e), torch.tensor(g, dtype=params.dtype), torch.tensor(h)
    return normal


# ------------------------------------------------------------------ CPU: host build
@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_emulated_jacobian_matches_oracle(case):
    label, pred, _, R, tau, k = case
    J = EJ.depth_jacobian(pred, R, 1 / (R - 1), 1e-4, tau, k)
    check(label, J, oracle_jacobian(pred, R, tau, k)[1])


@pytest.mark.parametrize("case", [c for c in CASES if "100.0" not in c[0]], ids=lambda c: c[0])
def test_emulated_onehot_vjp_is_the_row(case):
    """The VJP host build's result for a one-hot upstream on pixel (b, r, c) is the Jacobian host build's row (b, r, c),
    bit for bit: the two loops form the same sums in the same order."""
    label, pred, _, R, tau, k = case
    J = EJ.depth_jacobian(pred, R, 1 / (R - 1), 1e-4, tau, k)
    picks = onehot_pixels(J, np.random.RandomState(R))
    for i in range(max(len(p) for p in picks)):
        u = np.zeros((len(J), R, R), np.float32)
        for b, pix in enumerate(picks):
            if i < len(pix):
                u[b][pix[i]] = 1.0
        g = EV.depth_vjp(pred, u, R, 1 / (R - 1), 1e-4, tau, k).astype(np.float32)
        for b, pix in enumerate(picks):
            if i < len(pix):
                assert np.array_equal(g[b], J[b][pix[i]]), (label, b, pix[i], g[b], J[b][pix[i]])


def test_emulated_exact_zeros():
    pred, R = small_objects(), 64
    J = EJ.depth_jacobian(pred, R, 1 / (R - 1), 1e-4, 1.5, 260.0)
    depth = E.implicit(pred, None, R, 1 / (R - 1), 1e-4, 1.5, 260.0, want_grad=False, want_depth=True)[2]
    assert_exact_zeros(J, depth)


def test_emulated_lm_decisions():
    """LM on the oracle's normal equations for 10 iterations; at every state it visits, the host build's energies make the
    same accept / reject decision and its first step is the oracle's.  (Two separate trajectories are not compared: once
    the damping has fallen to ~1e-11 the steps are Gauss-Newton steps on a near-singular J^T J, which amplify the 1e-6
    differences between the two Jacobians -- measured: energies 1.5 % apart after 9 iterations, a first flip at the 10th.)"""
    p0, _, t = lm_start()
    oracle, seen = oracle_normal(t), []

    def host(params):
        p = params.numpy()
        J = EJ.depth_jacobian(p, 32, 1 / 31, 1e-4, 1.5, 260.0)
        depth = E.implicit(p, None, 32, 1 / 31, 1e-4, 1.5, 260.0, want_grad=False, want_depth=True)[2]
        return normal_from(J, depth, t)

    def both(_, params):
        out = oracle(None, params)
        seen.append((host(params), out))
        return out
    _, oks = lm_run(both, None, p0)
    def first_step(g, h):          # levenberg_marquardt's first solve (lam0, delta)
        A = h + optimize.LM_LAMBDA0 * (np.einsum("bjj->bj", h)[:, :, None] * np.eye(12) + optimize.LM_DELTA * np.eye(12))
        return np.linalg.solve(A, -0.5 * g[..., None])[..., 0]
    (_, g0, h0), (_, gr, hr) = seen[0]
    dh, do = first_step(g0, h0), first_step(gr.numpy(), hr.numpy())
    assert (np.abs(dh - do) <= 1e-3 * np.abs(do).max(axis=1, keepdims=True)).all()
    cur_h, cur_o = seen[0][0][0], seen[0][1][0].numpy()
    for i, ok in enumerate(oks):
        Eh, Eo = seen[i + 1][0][0], seen[i + 1][1][0].numpy()
        assert np.array_equal(Eh < cur_h, ok) and np.array_equal(Eo < cur_o, ok), (i, Eh, cur_h, Eo, cur_o)
        assert (np.abs(Eh - Eo) <= 1e-5 * Eo).all(), (i, Eh, Eo)
        cur_h, cur_o = np.where(ok, Eh, cur_h), np.where(ok, Eo, cur_o)
    print(f"\n[LM] accepted per iteration: {[int(a.sum()) for a in oks]}; energies {cur_o}")


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


def to_np(t):
    return t.detach().double().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_cuda_jacobian_matches_oracle(case, dev, S):
    label, pred, _, R, tau, k = case
    crit = S.ImplicitLoss(R, dev, tau, k)
    for dtype in (torch.float32, torch.float64):
        p_in = np.asarray(pred, dtype=np.float32 if dtype == torch.float32 else np.float64).astype(np.float64)
        base = torch.tensor(p_in, device=dev, dtype=dtype)
        if dtype == torch.float64:          # a non-leaf pred that requires grad: read detached
            pieces = [t.clone().requires_grad_(True) for t in torch.split(base, (3, 2, 3, 4), dim=1)]
            base = torch.cat(pieces, dim=1)
        depth, J = crit.render_jacobian(base)
        assert depth.shape == (len(p_in), R, R) and J.shape == (len(p_in), R, R, 12)
        assert depth.dtype == J.dtype == torch.float32 and not depth.requires_grad and not J.requires_grad
        check(f"{label} {dtype}", to_np(J), oracle_jacobian(p_in, R, tau, k)[1])
        assert torch.equal(depth, crit.depth_projection(base.detach())), (label, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if "r8" in c[0] or "r32" in c[0] or c[0] in ("edge", "grazing")],
                         ids=lambda c: c[0])
def test_cuda_jacobian_sums_to_the_vjp(case, dev, S):
    """sum_pix u J against render's VJP for the render tests' upstreams: both within the VJP contract of the oracle."""
    label, pred, tgt, R, tau, k = case
    depth, _ = oracle_vjps(pred, R, tau, k, {})
    gos = {name: go for name, go in upstreams(depth, tgt, R).items() if name != "single"}
    _, refs = oracle_vjps(pred, R, tau, k, gos)
    crit = S.ImplicitLoss(R, dev, tau, k)
    p = torch.tensor(np.asarray(pred, np.float64), device=dev)
    J = to_np(crit.render_jacobian(p)[1])
    for name, go in gos.items():
        pr = p.clone().requires_grad_(True)
        crit.render(pr).backward(torch.tensor(go, device=dev))
        for got in (np.einsum("brc,brcj->bj", go.astype(np.float64), J), to_np(pr.grad)):
            assert vjp_error(got, refs[name], go) <= 1.0, (label, name, vjp_error(got, refs[name], go))


@pytest.mark.gpu
def test_cuda_exact_zeros(dev, S):
    crit = S.ImplicitLoss(64, dev, 1.5, 260)
    depth, J = crit.render_jacobian(torch.tensor(small_objects(), device=dev))
    assert_exact_zeros(to_np(J), to_np(depth))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_cuda_render_normal_equations(dtype, dev, S):
    """E, g and H against an fp64 recomputation from the returned (depth, jac) and the target resized as the loss does."""
    B, R = 8, 32
    true, pred = O.random_params(B, 21).to(dev), O.perturbed_params(O.random_params(B, 21), 2, 0.05).to(dev, dtype)
    img = S.ImplicitLoss(100, dev, 1.5, 260).depth_projection(true).unsqueeze(1)
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    depth, J = crit.render_jacobian(pred)
    t = F.interpolate(img, size=(R, R), mode="nearest")[:, 0].double()
    r = (depth.double() - t).reshape(B, -1)
    Jd = J.double().reshape(B, -1, 12)
    w = torch.rand(B, R, R, device=dev) * (torch.rand(B, R, R, device=dev) > 0.2)
    for weight in (None, w):
        wd = torch.ones_like(r) if weight is None else weight.double().reshape(B, -1)
        E, g, H = crit.render_normal_equations(img, pred, weight)
        assert E.dtype == H.dtype == torch.float64 and g.dtype == dtype
        assert E.shape == (B,) and g.shape == (B, 12) and H.shape == (B, 12, 12)
        assert torch.allclose(E, (wd * r * r).sum(1), rtol=1e-12, atol=0)
        assert torch.allclose(g.double(), 2 * torch.einsum("bpj,bp->bj", Jd, wd * r), rtol=1e-6 if dtype == torch.float32 else 1e-12,
                              atol=1e-30)
        assert torch.allclose(H, torch.einsum("bpj,bpk->bjk", Jd * wd[..., None], Jd), rtol=1e-12, atol=1e-300)
        assert torch.equal(H, H.transpose(1, 2))


@pytest.mark.gpu
def test_cuda_errors(dev, S):
    from sq_recovery_b200 import _lib, functional as Fn
    L = _lib.lib()
    crit = S.ImplicitLoss(16, dev, 1.5, 260)
    p = O.random_params(2, 1).to(dev)
    img = torch.rand(2, 1, 20, 20, device=dev)
    for bad in (lambda: crit.render_jacobian(p[:, :11]),
                lambda: crit.render_normal_equations(img[:1], p),                          # batch
                lambda: crit.render_normal_equations(img[:, 0], p),                        # shape
                lambda: crit.render_normal_equations(img, p[:, :11]),
                lambda: crit.render_normal_equations(img, p, torch.ones(2, 15, 16, device=dev)),
                lambda: crit.render_normal_equations(img, p, torch.ones(2, 16, 16))):      # weight device
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(RuntimeError, match="CUDA"):
        crit.render_jacobian(p.cpu())
    pc, tag = Fn._params(p)
    B, n = 2, 16
    need = L.sq_scratch_bytes(B, n)
    scratch = torch.zeros(need, dtype=torch.uint8, device=dev)
    Fn._lib.check(L.sq_scratch_init(Fn._ptr(scratch), need, torch.cuda.current_stream(dev).cuda_stream), "init")
    depth = torch.empty(B, n, n, device=dev)
    jac = torch.empty(B, n, n, 12, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream

    def call(pred_=pc, jac_=jac, nbytes=need, dtype=tag, depth_=depth):
        P = lambda t: Fn._ptr(t) if t is not None else None       # noqa: E731
        return L.sq_depth_projection_jacobian(P(pred_), dtype, B, n, 1 / (n - 1), 1e-4, 1.5, 260.0, P(depth_), P(jac_),
                                              P(scratch), nbytes, st)
    assert call() == 0
    torch.cuda.synchronize()
    first = (depth.clone(), jac.clone())
    for kw in ({"pred_": None}, {"jac_": None}, {"nbytes": need - 1}, {"dtype": 7}):
        assert call(**kw) == EINVAL, kw
    torch.cuda.synchronize()
    assert torch.equal(depth, first[0]) and torch.equal(jac, first[1])    # a refused call writes nothing
    jac2 = torch.empty_like(jac)
    assert call(depth_=None, jac_=jac2) == 0                     # depth_out may be NULL
    assert call() == 0
    torch.cuda.synchronize()
    assert torch.equal(depth, first[0]) and torch.equal(jac, first[1]) and torch.equal(jac2, first[1])


@pytest.mark.gpu
def test_cuda_workspace_interleaving_and_determinism(dev, S):
    """The Jacobian call shares the per-stream workspace with every other call: interleaved with the fused loss, render and
    its VJP, voxel_loss and LeastSquares.normal_equations, every call returns the bits it returns alone; two calls are
    bit-identical."""
    B, R = 8, 32
    true, pred = O.random_params(B, 23).to(dev), O.perturbed_params(O.random_params(B, 23), 2, 0.05).to(dev)
    img = S.ImplicitLoss(128, dev, 1.5, 260).depth_projection(true).unsqueeze(1)
    im, ex, ls = S.ImplicitLoss(R, dev, 1.5, 260), S.ExplicitLoss(R, dev), S.LeastSquares(R, dev)
    vox = ex.occupancy(true) > 0.5
    go = torch.randn(B, R, R, device=dev)

    def others():
        pr = pred.clone().requires_grad_(True)
        l = im(img, pr)
        l.backward()
        pv = pred.clone().requires_grad_(True)
        im.render(pv).backward(go)
        return (l.detach(), pr.grad, pv.grad, ex.voxel_loss(vox, pred)) + ls.normal_equations(img, pred)

    j0, n0, o0 = im.render_jacobian(pred), im.render_normal_equations(img, pred), others()
    j1 = im.render_jacobian(pred)
    o1 = others()
    n1 = im.render_normal_equations(img, pred)
    j2 = im.render_jacobian(pred)
    for a, b in zip(j0 + j0 + n0 + o0, j1 + j2 + n1 + o1):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_cuda_graph_capture(dev, S):
    B, R = 16, 32
    true, pred = O.random_params(B, 31).to(dev), O.perturbed_params(O.random_params(B, 31), 4, 0.05).to(dev)
    img = S.ImplicitLoss(128, dev, 1.5, 260).depth_projection(true).unsqueeze(1)
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    ref_j, ref_n = crit.render_jacobian(pred), crit.render_normal_equations(img, pred)
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):                               # eager first on the capture stream: creates its workspace
        crit.render_jacobian(pred); crit.render_normal_equations(img, pred)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out_j = crit.render_jacobian(pred)
        out_n = crit.render_normal_equations(img, pred)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    for a, b in zip(ref_j + ref_n, out_j + out_n):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_cuda_large_batch(dev, S):
    """B = 1024: the plan kernel's 128-thread block path; a subset of samples against the oracle."""
    B, R, tau, k = 1024, 32, 1.5, 260.0
    pred = O.random_params(B, 71)
    depth, J = S.ImplicitLoss(R, dev, tau, k).render_jacobian(pred.to(dev))
    idx = np.arange(0, B, 97)
    check("B=1024", to_np(J)[idx], oracle_jacobian(pred.numpy()[idx], R, tau, k)[1])


@pytest.mark.gpu
def test_cuda_large_grid(dev, S):
    """R = 256 at B = 2: sum_pix u J against render's VJP (both are held to the oracle elsewhere), depth against the
    render, exact zeros on columns outside every object."""
    B, R = 2, 256
    pred = torch.tensor(small_objects(B, 43), device=dev)
    pred[:, 1:3] = 0.3
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    depth, J = crit.render_jacobian(pred)
    assert torch.equal(depth, crit.depth_projection(pred))
    go = torch.randn(B, R, R, device=dev)
    p = pred.clone().requires_grad_(True)
    crit.render(p).backward(go)
    got = torch.einsum("brc,brcj->bj", go.double(), J.double())
    tol = 1e-6 * R * R * go.abs().amax(dim=(1, 2))[:, None] + 1e-4 * p.grad.abs()
    assert ((got - p.grad).abs() <= tol).all(), ((got - p.grad).abs() / tol).max().item()
    assert (J[:, :8, :8] == 0).all() and (J[..., 0] == 0).all() and (J[..., 6] == 0).all()


@pytest.mark.gpu
def test_cuda_lm_fit(dev, S):
    """harness/optimize.py --loss implicit --method lm: every sample's energy never increases, and the result is finite."""
    B, R = 64, 32
    true = O.random_params(B, 0).to(dev)
    pred = O.perturbed_params(O.random_params(B, 0), 3, sigma=0.05).to(dev)
    img = S.ImplicitLoss(256, dev, 1.5, 260).depth_projection(true).unsqueeze(1).contiguous()
    crit = S.ImplicitLoss(R, dev, 1.5, 260)
    E0 = crit.render_normal_equations(img, pred)[0]
    rec = []
    optimize.levenberg_marquardt(crit.render_normal_equations, img, pred, 20, record=rec)
    prev = E0
    for E, _ in rec:
        assert (E <= prev).all()
        prev = E
    assert torch.isfinite(pred).all() and torch.isfinite(prev).all() and (prev < E0).any()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "harness", "optimize.py"), "--pairs", "256", "--steps", "10",
                          "--loss", "implicit", "--method", "lm"], capture_output=True, text=True, check=True, cwd=ROOT)
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["method"] == "lm" and res["loss"] == "implicit" and res["finite"] and res["loss_last"] <= res["loss_first"]
