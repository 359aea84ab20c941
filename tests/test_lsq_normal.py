"""Gauss-Newton normal equations of LeastSquares: LeastSquares.normal_equations / normal_equations_points and their C entry
points sq_least_squares_normal / sq_least_squares_points_normal.

Per sample, against the fp64 oracle: residuals r_i = sqrt(a1 a2 a3) (F(x_i) - 1) through oracle.sq_oracle.inside_outside_single
with the reference's clamps and zero fix-up, and their Jacobian J by forward-mode autograd (one pass per parameter), on the
parameters the kernel sees (fp32 parameters rounded first) and the fp32 points.  Points whose F >= 1e18 add no row to J^T J
(the gradient's rule):
  jtj:     |got - ref| <= 1e-3 |ref| + 1e-4 sqrt(ref_jj ref_kk)
  grad:    the LeastSquares gradient tolerance of energy_function: 1e-3 max_j |ref_j| + 2e-3 |ref| + 1e-5 per sample
  energy:  2e-4 |ref| + 1e-7
Each case prints its worst entries in units of the tolerance (energy / grad / jtj).

CPU tests: the host build (tests/emu/emu_lsq_normal.cpp) on the points of the images.  GPU tests (-m gpu): both variants
through the classes and the C ABI, equality with the existing calls, errors, workspace, determinism, graph capture and the
Levenberg-Marquardt fit of harness/optimize.py.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.autograd.forward_ad as fwAD

from conftest import ROOT, load_golden, random_golden_files
from oracle import sq_oracle as O
from harness import optimize

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu_lib as EM               # noqa: E402
import emu_lsq_normal_lib as EN    # noqa: E402

F_CUT = 1e18
EINVAL = 1                         # cudaErrorInvalidValue


# ------------------------------------------------------------------ cases and the reference
def cases():
    """(label, pred (B, 12), depth images (B, 1, H, W) fp32, R): the random goldens at R 8..64 (far and near predictions),
    the fixture images with their own and with rolled labels, the clamped edge golden and the zero-plane golden."""
    out = []
    for f in random_golden_files():
        g = load_golden(f)
        for tag in ("far", "near"):
            out.append((f"{f[:-4]} {tag}", g[f"pred_{tag}"], g["img"].astype(np.float32), int(g["R"])))
    g = load_golden("fixtures.npz")
    imgs = g["imgs_u8"].astype(np.float32) / 255.0
    out.append(("fixtures own", g["labels"], imgs, 64))
    out.append(("fixtures rolled", np.roll(g["labels"], 1, 0), imgs, 64))
    for f in ("edge.npz", "edge_zero_planes.npz"):
        g = load_golden(f)
        out.append((f[:-4], g["pred"], g["img"].astype(np.float32), int(g["R"])))
    return out


def rounded(p, dtype):
    p = np.asarray(p, dtype=np.float64)
    return p.astype(np.float32).astype(np.float64) if dtype == "fp32" else p


def image_points(img, R):
    """The (3, m_i) fp32 point lists LeastSquares builds from the depth images (classes.py:359-369)."""
    return [p.numpy() for p in O.LeastSquares(R).points(torch.as_tensor(img))]


def oracle_sample(p, pts):
    """fp64 energy, gradient 2 J^T r and J^T J (rows with F >= 1e18 left out) of one sample."""
    p = torch.as_tensor(p, dtype=torch.float64)
    P = torch.as_tensor(np.asarray(pts, dtype=np.float32)).double().reshape(3, -1)
    if P.shape[1] == 0:
        return 0.0, np.zeros(12), np.zeros((12, 12))

    def res(q):
        c = O.preprocess_sq(q)
        return torch.sqrt(c[0] * c[1] * c[2]) * (O.inside_outside_single(q, P, True, True) - 1.0)

    cols = []
    eye = torch.eye(12, dtype=torch.float64)
    with fwAD.dual_level():
        for k in range(12):
            r, t = fwAD.unpack_dual(res(fwAD.make_dual(p, eye[k])))
            cols.append(t)
        r = r.detach()
    J = torch.stack(cols, dim=1)
    with torch.no_grad():
        F = O.inside_outside_single(p, P, True, True)
    Jk = J[F < F_CUT]
    return float((r * r).sum()), (2.0 * J.T @ r).numpy(), (Jk.T @ Jk).numpy()


def oracle_normal(params, batch_points):
    out = [oracle_sample(p, pts) for p, pts in zip(np.asarray(params, dtype=np.float64), batch_points)]
    return np.array([o[0] for o in out]), np.stack([o[1] for o in out]), np.stack([o[2] for o in out])


def errors(got, ref):
    """Worst energy, gradient and J^T J entries in units of their tolerances."""
    (e, g, h), (re, rg, rh) = [tuple(np.asarray(x, dtype=np.float64) for x in t) for t in (got, ref)]
    e_e = np.abs(e - re) / (2e-4 * np.abs(re) + 1e-7)
    e_g = np.abs(g - rg) / (1e-3 * np.abs(rg).max(axis=1, keepdims=True) + 2e-3 * np.abs(rg) + 1e-5)
    d = np.sqrt(np.abs(np.diagonal(rh, axis1=1, axis2=2)))
    tol = 1e-3 * np.abs(rh) + 1e-4 * d[:, :, None] * d[:, None, :]
    diff = np.abs(h - rh)
    e_h = np.where(tol > 0, diff / np.where(tol > 0, tol, 1.0), np.where(diff > 0, np.inf, 0.0))
    return tuple(float(x.max()) if x.size else 0.0 for x in (e_e, e_g, e_h))


def check(label, got, ref):
    err = errors(got, ref)
    assert max(err) <= 1.0, (label, err)
    return "/".join(f"{x:.3g}" for x in err)


def check_structure(jtj, clamped=()):
    """Exactly symmetric; smallest eigenvalue >= -1e-6 of the largest; the rows and columns of clamped-out parameters
    exactly zero."""
    jtj = np.asarray(jtj, dtype=np.float64)
    assert np.array_equal(jtj, jtj.transpose(0, 2, 1))
    for b, h in enumerate(jtj):
        w = np.linalg.eigvalsh(h)
        assert w[0] >= -1e-6 * max(w[-1], 0.0), (b, w[0], w[-1])
        for j in clamped:
            assert not h[j].any() and not h[:, j].any(), (b, j)


def clamped_params(seed=7, B=4):
    """Random SQs with one parameter per sample outside its clamp box (a1 > 1, e1 < 0.1, t3 < 0, a3 < 0.05): that
    parameter's mask is 0."""
    p = O.random_params(B, seed, torch.float64).numpy()
    p[:, 5:8] = 0.5
    bad = [(0, 1.3), (3, 0.05), (7, -0.2), (2, 0.01)]
    for b in range(B):
        j, v = bad[b % len(bad)]
        p[b, j] = v
    return p, [bad[b % len(bad)][0] for b in range(B)]


def cloud_points(params, m, seed):
    """m points near the surface of each SQ of `params` (depth-image-like, within the unit cube), (3, m) fp32."""
    rng = np.random.RandomState(seed)
    out = []
    for p in np.asarray(params, dtype=np.float64):
        u = rng.normal(size=(3, m))
        u /= np.linalg.norm(u, axis=0, keepdims=True)
        M = O.mat_from_quaternion(torch.tensor(p[8:12])).numpy()
        x = (M @ (u * np.clip(p[0:3], 0.05, 1.0)[:, None] * rng.uniform(0.8, 1.2, size=(1, m)))) + p[5:8, None]
        out.append(np.clip(x, 0.0, 1.0).astype(np.float32))
    return out


def far_points(pts):
    """Each list with four points appended whose F >= max s_i^2 > 1e18.  Lists of a multiple of four points stay so: every
    other point keeps its thread, and the far ones take a thread of their own (the J^T J sums are then comparable bit for
    bit)."""
    assert all(x.shape[1] % 4 == 0 for x in pts)
    return [np.concatenate([x, np.full((3, 4), 1e10, np.float32)], axis=1) for x in pts]


def ragged_lists(seed=3):
    """Ragged point lists: two image lists, one of a single point, an empty one, and lists that are not multiples of 4."""
    g = load_golden("random_s1_b6_r16.npz")
    pts = image_points(g["img"].astype(np.float32), int(g["R"]))
    pts[1] = pts[1][:, :1]
    pts[2] = pts[2][:, :0]
    pts[3] = pts[3][:, :4 * (pts[3].shape[1] // 4) - 1]
    return g["pred_near"], pts


def lm_run(normal, target, p0, iters=10):
    p = p0.clone() if isinstance(p0, torch.Tensor) else torch.tensor(np.asarray(p0, dtype=np.float64))
    rec = []
    E = optimize.levenberg_marquardt(normal, target, p, iters, record=rec)
    return E.cpu().numpy(), [ok.cpu().numpy() for _, ok in rec], p.cpu().numpy()


def oracle_provider(batch_points):
    def normal(_, params):
        e, g, h = oracle_normal(params.cpu().numpy(), batch_points)
        return torch.tensor(e), torch.tensor(g, dtype=params.dtype), torch.tensor(h)
    return normal


def lm_start():
    """Train-like perturbed starts (sigma 0.02) and depth-image points of random SQs, R = 32.  From starts further out
    (sigma 0.05) both fits still make the same decisions, but after 10 iterations their energies differ by up to 7e-4: steps
    along poorly conditioned directions amplify the small differences between the two J^T J (DESIGN.md 2)."""
    true = O.random_params(6, 11, torch.float64)
    with torch.no_grad():
        img = O.ImplicitLoss(64, "cpu", 1.5, 260).depth_projection(true).float().unsqueeze(1)
    p0 = O.perturbed_params(true, 5, sigma=0.02).numpy()
    return p0, img, image_points(img.numpy(), 32)


def assert_same_trajectory(got, ref):
    (Eg, okg, _), (Er, okr, _) = got, ref
    assert all(np.array_equal(a, b) for a, b in zip(okg, okr)), (okg, okr)
    assert (np.abs(Eg - Er) <= 1e-4 * np.abs(Er)).all(), (Eg, Er)
    print(f"\n[LM] accepted per iteration: {[int(a.sum()) for a in okg]}; energies {Er}")


# ------------------------------------------------------------------ CPU: host build
@pytest.mark.parametrize("dtype", ["fp32", "fp64"])
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_emulated_matches_oracle(case, dtype):
    label, pred, img, R = case
    p = rounded(pred, dtype)
    pts = image_points(img, R)
    got = EN.normal_equations(p, pts)
    print(f"\n[normal equations, host] {label} {dtype} (energy/grad/jtj): {check((label, dtype), got, oracle_normal(p, pts))}")
    check_structure(got[2])


def test_emulated_lists():
    pred, pts = ragged_lists()
    got = EN.normal_equations(pred, pts)
    check("ragged", got, oracle_normal(pred, pts))
    assert got[0][2] == 0.0 and not got[1][2].any() and not got[2][2].any()      # the empty list: all zeros
    one = EN.normal_equations(pred[:1], pts[:1])                                    # B = 1
    assert all(np.array_equal(a[:1], b) for a, b in zip(got, one))
    p8, l8 = np.resize(pred, (8, 12)), (pts * 2)[:8]                                 # B = 1024: eight samples, 128 times
    ref8 = oracle_normal(p8, l8)
    check("B=1024", EN.normal_equations(np.tile(p8, (128, 1)), l8 * 128),
          tuple(np.tile(x, (128,) + (1,) * (x.ndim - 1)) for x in ref8))


def test_emulated_equals_existing():
    """Energy bit for bit, gradient to fp64 rounding, against the host build of the existing point-list loss (B = 1)."""
    g = load_golden("random_s2_b4_r32.npz")
    pts = image_points(g["img"].astype(np.float32), 32)
    e, gr, _ = EN.normal_equations(g["pred_far"], pts)
    for b, x in enumerate(pts):
        xyz = np.ascontiguousarray(x.T)
        loss, grad = EM.lsq(g["pred_far"][b:b + 1], xyz, np.array([0, xyz.shape[0]]))
        assert e[b] == loss
        np.testing.assert_allclose(gr[b], grad[0], rtol=1e-12, atol=1e-12 * np.abs(grad[0]).max())


def test_emulated_structure():
    p, bad = clamped_params()
    pts = cloud_points(p, 300, 1)
    got = EN.normal_equations(p, pts)
    check("clamped", got, oracle_normal(p, pts))
    for b, j in enumerate(bad):
        check_structure(got[2][b:b + 1], clamped=(j,))
        assert got[1][b, j] == 0.0
    assert np.array_equal(got[2], EN.normal_equations(p, far_points(pts))[2])


def test_emulated_lm_trajectory():
    """LM driven by the host build and by the oracle's fp64 normal equations, from the same start: the same accept / reject
    decisions over 10 iterations, final energies within 1e-4."""
    p0, _, pts = lm_start()

    def host(_, params):
        e, g, h = EN.normal_equations(params.numpy(), pts)
        return torch.tensor(e), torch.tensor(g, dtype=params.dtype), torch.tensor(h)
    assert_same_trajectory(lm_run(host, None, p0), lm_run(oracle_provider(pts), None, p0))


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
    return tuple(x.double().cpu().numpy() for x in t)


def torch_params(p, dtype, dev):
    return torch.tensor(np.asarray(p), dtype=torch.float32 if dtype == "fp32" else torch.float64, device=dev)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "fp64"])
@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_cuda_matches_oracle(case, dtype, dev, S):
    label, pred, img, R = case
    p = rounded(pred, dtype)
    pts = image_points(img, R)
    ref = oracle_normal(p, pts)
    ls = S.LeastSquares(R, dev)
    pt = torch_params(pred, dtype, dev)
    out_img = ls.normal_equations(torch.tensor(img, device=dev), pt)
    out_pts = ls.normal_equations_points([torch.tensor(x, device=dev) for x in pts], pt)
    for out in (out_img, out_pts):
        e, g, h = out
        assert e.dtype == torch.float64 and h.dtype == torch.float64 and g.dtype == pt.dtype
        assert e.shape == (len(p),) and g.shape == (len(p), 12) and h.shape == (len(p), 12, 12)
        assert not (e.requires_grad or g.requires_grad or h.requires_grad)
        check_structure(h.cpu().numpy())
    print(f"\n[normal equations, CUDA] {label} {dtype} (energy/grad/jtj) image {check(label, to_np(out_img), ref)}, "
          f"points {check(label, to_np(out_pts), ref)}")


@pytest.mark.gpu
def test_cuda_lists(dev, S):
    pred, pts = ragged_lists()
    ls = S.LeastSquares(16, dev)
    pt = torch.tensor(pred, device=dev)
    got = to_np(ls.normal_equations_points([torch.tensor(x, device=dev) for x in pts], pt))
    check("ragged", got, oracle_normal(pred, pts))
    assert got[0][2] == 0.0 and not got[1][2].any() and not got[2][2].any()
    one = to_np(ls.normal_equations_points([torch.tensor(pts[0], device=dev)], pt[:1]))
    check("B=1", one, oracle_normal(pred[:1], pts[:1]))
    p8, l8 = np.resize(pred, (8, 12)), (pts * 2)[:8]
    ref8 = oracle_normal(p8, l8)
    big = to_np(ls.normal_equations_points([torch.tensor(x, device=dev) for x in l8 * 128],
                                           torch.tensor(np.tile(p8, (128, 1)), device=dev)))
    check("B=1024", big, tuple(np.tile(x, (128,) + (1,) * (x.ndim - 1)) for x in ref8))
    with torch.enable_grad():                                   # parameters that require grad are read detached
        pg = pt.clone().requires_grad_(True)
        out = ls.normal_equations_points([torch.tensor(x, device=dev) for x in pts], pg)
    assert all(x.grad_fn is None for x in out)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "fp64"])
def test_cuda_equals_existing(dtype, dev, S):
    """Points: energy and gradient bit for bit those of sq_least_squares_points.  Image: energies bit for bit those of
    sq_least_squares' per_sample."""
    from sq_recovery_b200 import _lib, functional as Fn
    L = _lib.lib()
    g = load_golden("fixtures.npz")
    imgs = torch.tensor(g["imgs_u8"].astype(np.float32) / 255.0, device=dev)
    pt = torch_params(g["labels"], dtype, dev)
    ls = S.LeastSquares(64, dev)
    pts = [torch.tensor(x, device=dev) for x in image_points(imgs.cpu().numpy(), 64)]
    e, gr, _ = ls.normal_equations_points(pts, pt)
    p, tag = Fn._params(pt)
    B = p.shape[0]
    packed, offsets, mp = Fn.pack_points(pts, dev)
    per, grad = torch.empty(B, dtype=torch.float64, device=dev), torch.empty_like(p)
    scratch = torch.zeros(L.sq_points_scratch_bytes(B, mp), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.sq_least_squares_points(Fn._ptr(p), tag, B, Fn._ptr(packed), packed.shape[1], Fn._ptr(offsets), mp, None,
                                         Fn._ptr(per), Fn._ptr(grad), Fn._ptr(scratch), scratch.numel(), st), "points")
    assert torch.equal(e, per) and torch.equal(gr, grad)
    ei, _, _ = ls.normal_equations(imgs.unsqueeze(1) if imgs.dim() == 3 else imgs, pt)
    row_off, col_off = Fn.nearest_offsets(256, 256, 64, dev)
    img = Fn._image(imgs)
    per_i, loss = torch.empty(B, dtype=torch.float64, device=dev), torch.empty((), dtype=torch.float64, device=dev)
    scratch = torch.zeros(L.sq_scratch_bytes(B, 64), dtype=torch.uint8, device=dev)
    _lib.check(L.sq_least_squares(Fn._ptr(p), tag, B, 64, Fn._ptr(img), 256 * 256, Fn._ptr(row_off), Fn._ptr(col_off),
                                  Fn._ptr(loss), Fn._ptr(per_i), None, Fn._ptr(scratch), scratch.numel(), st), "image")
    assert torch.equal(ei, per_i)
    # and the public energy_function agrees (it returns the energies in the parameters' dtype)
    assert torch.equal(ls.energy_function(pts, pt), e.to(pt.dtype))


@pytest.mark.gpu
def test_cuda_structure(dev, S):
    p, bad = clamped_params()
    pts = cloud_points(p, 300, 1)
    ls = S.LeastSquares(16, dev)
    got = to_np(ls.normal_equations_points([torch.tensor(x, device=dev) for x in pts], torch.tensor(p, device=dev)))
    check("clamped", got, oracle_normal(p, pts))
    for b, j in enumerate(bad):
        check_structure(got[2][b:b + 1], clamped=(j,))
        assert got[1][b, j] == 0.0
    with_far = ls.normal_equations_points([torch.tensor(x, device=dev) for x in far_points(pts)],
                                          torch.tensor(p, device=dev))[2]
    assert np.array_equal(got[2], with_far.cpu().numpy())


@pytest.mark.gpu
def test_cuda_lm_trajectory(dev, S):
    p0, img, pts = lm_start()
    ls = S.LeastSquares(32, dev)
    got = lm_run(ls.normal_equations, img.to(dev), torch.tensor(p0, device=dev))
    assert_same_trajectory(got, lm_run(oracle_provider(pts), None, p0))


@pytest.mark.gpu
def test_cuda_errors(dev, S):
    from sq_recovery_b200 import _lib, functional as Fn
    L = _lib.lib()
    ls = S.LeastSquares(16, dev)
    p = O.random_params(2, 1).to(dev)
    img = torch.rand(2, 1, 16, 16, device=dev)
    with pytest.raises(ValueError):
        ls.normal_equations(img[:1], p)                           # batch
    with pytest.raises(ValueError):
        ls.normal_equations(img[:, 0], p)                         # shape
    with pytest.raises(ValueError):
        ls.normal_equations(img, p[:, :11])
    with pytest.raises(ValueError):
        ls.normal_equations_points([torch.rand(3, 5, device=dev)], p)
    with pytest.raises(ValueError):
        ls.normal_equations_points([torch.rand(4, 5, device=dev)] * 2, p)
    with pytest.raises(RuntimeError, match="CUDA"):
        ls.normal_equations(img.cpu(), p.cpu())
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            ls.normal_equations(img.to("cuda:1"), p)
    # the C ABI: NULL outputs, scratch too small, bad dtype -> cudaErrorInvalidValue
    pc, tag = Fn._params(p)
    B = 2
    packed, offsets, mp = Fn.pack_points([torch.rand(3, 7, device=dev)] * 2, dev)
    per, grad = torch.empty(B, dtype=torch.float64, device=dev), torch.empty_like(pc)
    jtj = torch.empty(B, 12, 12, dtype=torch.float64, device=dev)
    need = L.sq_normal_scratch_bytes(B, mp)
    assert need > 0 and L.sq_normal_scratch_bytes(0, mp) == 0 and L.sq_normal_scratch_bytes(B, -1) == 0
    scratch = torch.zeros(need, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    P = Fn._ptr

    def pts_call(per_=per, grad_=grad, jtj_=jtj, nbytes=need, dtype=tag):
        return L.sq_least_squares_points_normal(P(pc), dtype, B, P(packed), packed.shape[1], P(offsets), mp, P(per_) if per_ is not None else None,
                                                P(grad_) if grad_ is not None else None, P(jtj_) if jtj_ is not None else None,
                                                P(scratch), nbytes, st)
    assert pts_call() == 0
    torch.cuda.synchronize()
    first = (per.clone(), grad.clone(), jtj.clone())
    for kw in ({"per_": None}, {"grad_": None}, {"jtj_": None}, {"nbytes": need - 1}, {"dtype": 7}):
        assert pts_call(**kw) == EINVAL, kw
    row_off, col_off = Fn.nearest_offsets(16, 16, 16, dev)
    imgc = Fn._image(img)
    need_i = L.sq_normal_scratch_bytes(B, 16 * 16)
    scr_i = torch.zeros(need_i, dtype=torch.uint8, device=dev)

    def img_call(per_=per, grad_=grad, jtj_=jtj, nbytes=need_i, R=16):
        return L.sq_least_squares_normal(P(pc), tag, B, R, P(imgc), 256, P(row_off), P(col_off),
                                         P(per_) if per_ is not None else None, P(grad_) if grad_ is not None else None,
                                         P(jtj_) if jtj_ is not None else None, P(scr_i), nbytes, st)
    assert img_call() == 0
    for kw in ({"per_": None}, {"grad_": None}, {"jtj_": None}, {"nbytes": need_i - 1}, {"R": 0}):
        assert img_call(**kw) == EINVAL, kw
    # the calls that failed left nothing behind: the next one gives the first one's bits
    assert pts_call() == 0
    torch.cuda.synchronize()
    assert torch.equal(per, first[0]) and torch.equal(grad, first[1]) and torch.equal(jtj, first[2])


@pytest.mark.gpu
def test_cuda_workspace_interleaving_and_determinism(dev, S):
    """The normal equations share the per-stream workspace with every other call: interleaved with the loss calls, render
    and voxel_loss, every call returns the bits it returns alone; two calls are bit-identical."""
    B, R = 8, 32
    true, pred = O.random_params(B, 21).to(dev), O.perturbed_params(O.random_params(B, 21), 2, 0.05).to(dev)
    img = S.ImplicitLoss(128, dev, 1.5, 260).depth_projection(true).unsqueeze(1)
    ls, ex, im = S.LeastSquares(R, dev), S.ExplicitLoss(R, dev), S.ImplicitLoss(R, dev, 1.5, 260)
    pts = [torch.tensor(x, device=dev) for x in image_points(img.cpu().numpy(), R)]
    vox = ex.occupancy(true) > 0.5

    def others():
        return (ls(img, pred), ex(true, pred), im(img, pred), im.render(pred), ex.voxel_loss(vox, pred), ls.energy_function(pts, pred))

    n0, q0, o0 = ls.normal_equations(img, pred), ls.normal_equations_points(pts, pred), others()
    n1 = ls.normal_equations(img, pred)
    o1 = others()
    q1 = ls.normal_equations_points(pts, pred)
    n2 = ls.normal_equations(img, pred)
    for a, b in zip(n0 + q0 + n0, n1 + q1 + n2):
        assert torch.equal(a, b)
    for a, b in zip(o0, o1):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_cuda_graph_capture(dev, S):
    from sq_recovery_b200 import functional as Fn
    B, R = 16, 32
    true, pred = O.random_params(B, 31).to(dev), O.perturbed_params(O.random_params(B, 31), 4, 0.05).to(dev)
    img = S.ImplicitLoss(128, dev, 1.5, 260).depth_projection(true).unsqueeze(1)
    ls = S.LeastSquares(R, dev)
    pts = [torch.tensor(x, device=dev) for x in image_points(img.cpu().numpy(), R)]
    ref_i, ref_p = ls.normal_equations(img, pred), ls.normal_equations_points(pts, pred)
    packed = Fn.pack_points(pts, dev)                        # the lists cross to the device before the capture
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):                               # eager first on the capture stream: creates its workspace
        ls.normal_equations(img, pred); Fn.lsq_points_normal_packed(pred, *packed)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out_i = ls.normal_equations(img, pred)
        out_p = Fn.lsq_points_normal_packed(pred, *packed)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(ref_i + ref_p, out_i + out_p):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_cuda_lm_fit(dev, S):
    """harness/optimize.py --loss lsq --method lm: every sample's energy never increases, and the result is finite."""
    B, R = 64, 32
    true = O.random_params(B, 0).to(dev)
    pred = O.perturbed_params(O.random_params(B, 0), 3, sigma=0.05).to(dev)
    img = S.ImplicitLoss(256, dev, 1.5, 260).depth_projection(true).unsqueeze(1).contiguous()
    ls = S.LeastSquares(R, dev)
    E0 = ls.normal_equations(img, pred)[0]
    rec = []
    optimize.levenberg_marquardt(ls.normal_equations, img, pred, 20, record=rec)
    prev = E0
    for E, _ in rec:
        assert (E <= prev).all()
        prev = E
    assert torch.isfinite(pred).all() and torch.isfinite(prev).all() and (prev < E0).any()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "harness", "optimize.py"), "--pairs", "256", "--steps", "10",
                          "--loss", "lsq", "--method", "lm"], capture_output=True, text=True, check=True, cwd=ROOT)
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["method"] == "lm" and res["loss"] == "lsq" and res["finite"] and res["loss_last"] <= res["loss_first"]
