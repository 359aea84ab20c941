"""Drop-in replacements for the loss classes of the reference's ``torch/classes.py``.

Same class names, constructor signatures, public attributes, call signatures and autograd behaviour
(SURVEY 8b); the per-sample Python loop of ~1.5 k fp64 tensor ops is replaced by one fused CUDA kernel per call
(csrc/sqloss.cu through include/sqloss.h).  Swap in with

    from sq_recovery_b200.classes import ExplicitLoss, ImplicitLoss, IoUAccuracy, LeastSquares

There is no CPU path: ``device`` must be a CUDA device.
"""
from __future__ import annotations

import numpy as np
import torch

from . import functional as Fn

_ZERO_FIX = 1e-4        # torch/classes.py:126, :221


def _cuda_device(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"sq_recovery_b200 runs on CUDA devices only (got device={device!r}); "
                           "there is no CPU fallback")
    return dev


def _preprocess_sq(p: torch.Tensor) -> torch.Tensor:
    """Clamp a to [0.05, 1], e to [0.1, 1], t to [0, 1]; q untouched (torch/classes.py:129-136)."""
    a, e, t, q = torch.split(p, (3, 2, 3, 4), dim=-1)
    return torch.cat([a.clamp(0.05, 1), e.clamp(0.1, 1), t.clamp(0, 1), q], dim=-1)


def _no_history(p: torch.Tensor, what: str, instead: str = "") -> None:
    """The grid-returning conveniences are forward-only here (the reference returns fp64 grids WITH autograd history,
    torch/classes.py:138-189, 232-282, 394-426).  Differentiating through them would silently yield no gradient, so a
    tensor that asks for one is refused instead."""
    if torch.is_grad_enabled() and isinstance(p, torch.Tensor) and p.requires_grad:
        raise RuntimeError(
            f"sq_recovery_b200: {what}() is forward-only (fp32 grid, no autograd history); it was given a tensor that "
            "requires grad.  Call it under torch.no_grad() / on p.detach(), or differentiate through the loss call "
            f"(loss(true, pred).backward()), which is fused.{instead}")


class _GridLoss:
    """Shared bookkeeping: the reference stores these attributes on every loss object."""

    def _setup(self, render_size, device, reduce, axis, fix_zero):
        self.render_size = render_size
        self.render_type = np.float64
        self.eps = 1e-8
        self.reduce = reduce
        self.device = _cuda_device(device)
        self._axis = axis                       # the reference's 1-D coordinate table, fp64
        self._n = int(len(axis))
        self._step = float(axis[1] - axis[0]) if len(axis) > 1 else 1.0
        self._z0 = _ZERO_FIX if fix_zero else 0.0
        self._xyz = None
        Fn._lib.lib()                           # fail at construction time if libsqloss.so is missing

    @property
    def xyz(self) -> torch.Tensor:
        """(3, n, n, n) fp64 meshgrid like the reference's attribute; built on first access (the kernels
        generate grid points from indices and never read it)."""
        if self._xyz is None:
            r = torch.tensor(self._axis)
            grid = torch.stack(torch.meshgrid([r, r, r], indexing="ij")).to(self.device)
            if self._z0:
                grid[grid == 0] += self._z0
            self._xyz = grid
        return self._xyz

    preprocess_sq = staticmethod(_preprocess_sq)


class ExplicitLoss(_GridLoss):
    """MSE x 100 between the occupancy grids of true and predicted parameters (torch/classes.py:109-201)."""

    def __init__(self, render_size, device, reduce=True):
        step = 1 / render_size
        axis = np.arange(0, 1 + step, step).astype(np.float64)          # classes.py:122-123 (n = R+1, R+2 for R=24,96)
        self._setup(render_size, device, reduce, axis, fix_zero=True)
        self._step = step

    def occupancy(self, p):
        """(B, n, n, n) sigmoid(5 (1 - F)) (classes.py:138-189), fp32, no autograd."""
        _no_history(p, "occupancy", "  For an occupancy grid to differentiate through (any loss on voxels), use "
                    "soft_occupancy(p).")
        return Fn.field(p, self._n, self._step, self._z0, 1, 5.0)

    def soft_occupancy(self, p):
        """(B, n, n, n) fp32 occupancy sigmoid(5 (1 - F)), differentiable w.r.t. ``p`` (the reference's occupancy with
        autograd history, classes.py:138-189): the same bits as ``occupancy``; its backward is one CUDA vector-Jacobian
        product, so any loss on the grid (MSE or BCE against voxels, masks, per-voxel weights, a soft-volume term, sums
        of these) can be trained through it.  When ground-truth parameters exist, ``self(true, pred)`` is cheaper: it is
        fused into one walk and never holds a grid in memory.  Under torch.no_grad(), or for a ``p`` that does not
        require grad, a plain tensor."""
        args = (self._n, self._step, self._z0, 5.0)
        if torch.is_grad_enabled() and isinstance(p, torch.Tensor) and p.requires_grad:
            return Fn.OccupancyFn.apply(p, *args)
        return Fn.field(p, self._n, self._step, self._z0, 1, 5.0)

    def __call__(self, true, pred):
        return Fn.ExplicitLossFn.apply(true, pred, self._n, self._step, self._z0, 5.0, 100.0, torch.is_grad_enabled())

    def voxel_loss(self, voxels, pred, voxel_scale=None):
        """0-dim fp64 loss 100 mean((occupancy(pred) - v)^2), averaged over the batch like ``self(true, pred)``, against
        voxel data instead of true parameters: the reference's objective with the target occupancy replaced by voxels.
        ``voxels`` is (B, n, n, n) on this loss's grid, index order [x][y][z], on ``pred``'s device: float32 (float64 is
        rounded to it), bool, or uint8 read as v = voxel_scale * byte (default 1/255).  Forward and backward are one CUDA
        walk; no occupancy grid is held in memory, and 8-bit voxels are read as bytes.  The gradient reaches ``pred``
        only: for a loss that must differentiate the voxels too, use soft_occupancy(pred)."""
        if torch.is_grad_enabled() and isinstance(voxels, torch.Tensor) and voxels.requires_grad:
            raise RuntimeError(
                "sq_recovery_b200: voxel_loss() gives a gradient for pred only, and it was given voxels that require grad. "
                "Pass voxels.detach(), or build the loss from soft_occupancy(pred), which differentiates any loss on the grid.")
        return Fn.VoxelLossFn.apply(voxels, pred, self._n, self._step, self._z0, 5.0, 100.0, voxel_scale,
                                    torch.is_grad_enabled())


class ImplicitLoss(_GridLoss):
    """MAE between the input depth image and a soft depth render of the predicted SQ (torch/classes.py:203-295)."""

    def __init__(self, render_size, device, tau=1, sigmoid_sharpness=100, reduce=True):
        axis = np.linspace(0, 1, render_size).astype(np.float64)        # classes.py:218
        self._setup(render_size, device, reduce, axis, fix_zero=True)
        self.tau = tau
        self.sigmoid_sharpness = sigmoid_sharpness

    def depth_projection(self, p):
        """(B, R, R) depth render in image orientation (classes.py:232-282), fp32, no autograd."""
        _no_history(p, "depth_projection", "  For a depth render to differentiate through (any image-space loss), "
                    "use render(p).")
        return Fn.depth_projection(p, self._n, self._step, self._z0, float(self.tau), float(self.sigmoid_sharpness))

    def render(self, p):
        """(B, R, R) fp32 depth render in image orientation, differentiable w.r.t. ``p`` (the reference's depth_projection
        with autograd history, classes.py:232-282): the same bits as ``depth_projection``; its backward is one CUDA
        vector-Jacobian product, so any image-space loss (L2, Huber, masks, weights, sums of terms) can be trained through
        it.  For the plain MAE against a target image, ``self(true, pred)`` is cheaper: it is fused into one walk.
        Under torch.no_grad(), or for a ``p`` that does not require grad, a plain tensor."""
        args = (self._n, self._step, self._z0, float(self.tau), float(self.sigmoid_sharpness))
        if torch.is_grad_enabled() and isinstance(p, torch.Tensor) and p.requires_grad:
            return Fn.DepthProjectionFn.apply(p, *args)
        return Fn.depth_projection(p, *args)

    def __call__(self, true, pred):
        return Fn.ImplicitLossFn.apply(true, pred, self._n, self._step, self._z0, float(self.tau),
                                       float(self.sigmoid_sharpness), False, torch.is_grad_enabled())

    def from_heads(self, true, raw_heads):
        """The same loss taken straight from the RAW outputs of the four linear heads, (B, 12) =
        [size(3) | shape(2) | position(3) | rotation(4)]: the sigmoids, the quaternion normalisation
        (torch/models.py:28,52,75,98), the torch.cat of torch/train.py:89 and all their backward kernels run inside
        the loss kernels.  Not in the reference (SURVEY 8f-3); equals ``self(true, heads(raw_heads))``."""
        return Fn.ImplicitLossFn.apply(true, raw_heads, self._n, self._step, self._z0, float(self.tau),
                                       float(self.sigmoid_sharpness), True, torch.is_grad_enabled())


class LeastSquares(_GridLoss):
    """Solina-Bajcsy energy on the points back-projected from the depth image (torch/classes.py:297-371)."""

    def __init__(self, render_size, device, reduce=True):
        self._setup(render_size, device, reduce, np.array([0.0, 1.0]), fix_zero=False)

    @property
    def xyz(self):
        raise AttributeError("LeastSquares has no grid (torch/classes.py:303-308)")

    def energy_function(self, batch_points, params):
        """Per-sample energies (B,) of explicit point lists (classes.py:318-356): ``batch_points[i]`` is a (3, m_i) tensor
        of (x, y, z) rows, ``params`` (B, 12).  The lists are packed into one compacted structure-of-arrays buffer and
        read with float4 loads by ``sq_least_squares_points``; gradient reaches ``params``."""
        return Fn.lsq_energy(batch_points, params)

    def __call__(self, true, pred):
        return Fn.LeastSquaresFn.apply(true, pred, int(self.render_size), torch.is_grad_enabled())


class IoUAccuracy(_GridLoss):
    """IoU of the binarised (F <= 1) grids of true and predicted parameters (torch/classes.py:374-447)."""

    def __init__(self, render_size, device, reduce=True, full=False):
        axis = np.linspace(0, 1, render_size).astype(np.float64)        # classes.py:389
        self._setup(render_size, device, reduce, axis, fix_zero=False)
        self.full = full

    def ins_outs(self, p):
        """(B, R, R, R) inside-outside values F (classes.py:394-426), fp32, no autograd."""
        _no_history(p, "ins_outs")
        return Fn.field(p, self._n, self._step, 0.0, 0)

    def counts(self, true, pred):
        """Per-sample (intersection, union) voxel counts, int64."""
        return Fn.iou_counts(true, pred, self._n, self._step, 0.0)

    def __call__(self, true, pred):
        inter, union = self.counts(true, pred)
        if not self.reduce:
            return inter.double() / union.double()                      # classes.py:441-445
        return torch.sum(inter) / torch.sum(union)                      # classes.py:437-439 (batch-wide ratio)
