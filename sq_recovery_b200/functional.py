"""torch.autograd.Function wrappers over the C ABI (include/sqloss.h).

Each Function runs the fused forward+backward kernel once in ``forward`` and keeps d loss / d params for
``backward`` (SURVEY 8b); under ``torch.no_grad()`` or when no input needs a gradient the forward-only kernel
runs.  Everything is launched on torch's current stream; nothing here synchronises the host.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

from . import _lib

_scratch: Dict[Tuple[int, int], torch.Tensor] = {}
_retired: list = []          # outgrown workspaces, kept alive (see _get_scratch)
_offsets: Dict[Tuple[int, int, int, int], Tuple[torch.Tensor, torch.Tensor]] = {}


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"sq_recovery_b200: {what} must live on a CUDA device (got {t.device}); "
                           "there is no CPU path in this package")


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_need: Dict[Tuple[int, int], int] = {}


class _on_device:
    """torch.cuda.device(dev) only when dev is not already current (the context manager costs ~5 us per call)."""

    def __init__(self, device: torch.device):
        idx = device.index
        self._ctx = None if idx is None or idx == torch.cuda.current_device() else torch.cuda.device(device)

    def __enter__(self):
        if self._ctx is not None:
            self._ctx.__enter__()

    def __exit__(self, *exc):
        if self._ctx is not None:
            self._ctx.__exit__(*exc)


def _get_scratch(device: torch.device, batch: int, n: int, need: Optional[int] = None) -> torch.Tensor:
    """Per (device, stream) workspace, grown on demand and reused (stream-ordered, so reuse is safe)."""
    if need is None:
        need = _need.get((batch, n))
        if need is None:
            need = _need[(batch, n)] = _lib.lib().sq_scratch_bytes(batch, n)
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream(device))
    buf = _scratch.get(key)
    if buf is None or buf.numel() < need:
        if torch.cuda.is_current_stream_capturing():
            # Allocated here, the buffer would come from the graph's private pool and its one-time zeroing would be a node
            # of THIS graph only: another graph captured on the same stream and replayed first would start the kernels on
            # uninitialised queue counters.  So the workspace of a capture stream must exist before the capture starts.
            raise RuntimeError(
                "sq_recovery_b200: no workspace for this stream yet (or it is too small for this batch / grid size) and "
                "the stream is being captured into a CUDA graph.  Run the same call once eagerly on the capture stream "
                "first -- `s = torch.cuda.Stream(); with torch.cuda.stream(s): loss_fn(true, pred)` -- and capture with "
                "`torch.cuda.graph(g, stream=s)`, or call sq_recovery_b200.functional.prepare_stream(device, batch, n, s).")
        if buf is not None:
            _retired.append(buf)             # a CUDA graph captured earlier may still hold pointers into the smaller buffer
        buf = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=device)
        with torch.cuda.device(device):      # zero the control block once; every call leaves it zero (include/sqloss.h)
            _lib.check(_lib.lib().sq_scratch_init(ctypes.c_void_p(buf.data_ptr()), buf.numel(), _stream(device)),
                       "sq_scratch_init")
        _scratch[key] = buf
    return buf


def prepare_stream(device, batch: int, n: int, stream: "torch.cuda.Stream") -> None:
    """Create (and zero the control block of) the workspace `stream` will use for calls with up to this batch and grid
    size.  Needed only before capturing a CUDA graph on a stream that has not run the call eagerly (INTEGRATION.md 5)."""
    device = torch.device(device)
    with torch.cuda.stream(stream):
        _get_scratch(device, batch, n)


def _params(p: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Contiguous fp32 or fp64 copy of a (B,12) parameter tensor and its dtype tag."""
    if p.dim() != 2 or p.shape[1] != 12:
        raise ValueError(f"expected parameters of shape (B, 12), got {tuple(p.shape)}")
    if p.dtype == torch.float64:
        return p.detach().contiguous(), _lib.SQ_F64
    return p.detach().float().contiguous(), _lib.SQ_F32


def nearest_offsets(height: int, width: int, size: int, device: torch.device):
    """Element offsets of the rows / columns F.interpolate(mode='nearest') samples (torch/classes.py:286, :359).

    Derived from F.interpolate itself so the index rule is PyTorch's by construction.
    """
    key = (height, width, size, device.index if device.index is not None else -1)
    hit = _offsets.get(key)
    if hit is None:
        rows = F.interpolate(torch.arange(height, dtype=torch.float32).view(1, 1, height, 1), size=(size, 1), mode="nearest")
        cols = F.interpolate(torch.arange(width, dtype=torch.float32).view(1, 1, 1, width), size=(1, size), mode="nearest")
        row_off = (rows.view(-1).to(torch.int32) * width).to(device)
        col_off = cols.view(-1).to(torch.int32).to(device)
        hit = (row_off, col_off)
        _offsets[key] = hit
    return hit


def _image(true: torch.Tensor) -> torch.Tensor:
    if true.dim() != 4 or true.shape[1] != 1:
        raise ValueError(f"expected depth images of shape (B, 1, H, W), got {tuple(true.shape)}")
    return true.detach().float().contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class ImplicitLossFn(torch.autograd.Function):
    """ImplicitLoss.__call__ (torch/classes.py:284-295) -> 0-dim fp64 loss; gradient reaches ``pred`` only."""

    @staticmethod
    def forward(ctx, true, pred, n, step, z0, tau, sharpness, heads=False, grad_mode=True):
        # heads=True: `pred` holds the RAW outputs of the four network heads; sigmoid / quaternion normalisation, the
        # torch.cat and their Jacobians run inside the kernels (sq_implicit_loss_heads, SURVEY 8f-3)
        _require_cuda(pred, "pred"); _require_cuda(true, "true")
        dev = pred.device
        img = _image(true)
        p, tag = _params(pred)
        B = p.shape[0]
        if img.shape[0] != B:
            raise ValueError("true and pred disagree on the batch size")
        row_off, col_off = nearest_offsets(img.shape[2], img.shape[3], n, dev)
        # needs_input_grad follows pred.requires_grad whatever the grad mode: under torch.no_grad() (validation,
        # train.py:135) the forward-only kernel runs
        want_grad = grad_mode and ctx.needs_input_grad[1]
        loss = torch.empty((), dtype=torch.float64, device=dev)
        grad = torch.empty_like(p) if want_grad else None
        scratch = _get_scratch(dev, B, n)
        entry = _lib.lib().sq_implicit_loss_heads if heads else _lib.lib().sq_implicit_loss
        with _on_device(dev):
            rc = entry(
                _ptr(p), tag, B, n, step, z0, _ptr(img), img.shape[2] * img.shape[3], _ptr(row_off), _ptr(col_off),
                tau, sharpness, _ptr(loss), None, _ptr(grad), None, _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_implicit_loss_heads" if heads else "sq_implicit_loss")
        ctx.grad = grad
        ctx.pred_dtype = pred.dtype
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        g = None
        if ctx.grad is not None:
            g = (ctx.grad * go).to(ctx.pred_dtype)      # 0-dim fp64 `go` does not promote the result: one kernel
        return None, g, None, None, None, None, None, None, None


class ExplicitLossFn(torch.autograd.Function):
    """ExplicitLoss.__call__ (torch/classes.py:191-201).  The loss is symmetric in (true, pred), so a gradient for
    ``true`` (no reference caller asks for one) is the same kernel with the roles swapped."""

    @staticmethod
    def forward(ctx, true, pred, n, step, z0, sharpness, mult, grad_mode=True):
        _require_cuda(pred, "pred"); _require_cuda(true, "true")
        dev = pred.device
        if true.dtype == torch.float64 or pred.dtype == torch.float64:
            true_c, pred_c = true.double(), pred.double()
        else:
            true_c, pred_c = true, pred
        t, tag = _params(true_c)
        p, _ = _params(pred_c)
        B = p.shape[0]
        if t.shape[0] != B:
            raise ValueError("true and pred disagree on the batch size")
        loss = torch.empty((), dtype=torch.float64, device=dev)
        scratch = _get_scratch(dev, B, n)
        L = _lib.lib()

        def run(a, b, grad):
            with _on_device(dev):
                rc = L.sq_explicit_loss(_ptr(a), _ptr(b), tag, B, n, step, z0, sharpness, mult, _ptr(loss), None,
                                        _ptr(grad), _ptr(scratch), scratch.numel(), _stream(dev))
            _lib.check(rc, "sq_explicit_loss")

        ctx.grad_true = ctx.grad_pred = None
        if grad_mode and ctx.needs_input_grad[0]:
            ctx.grad_true = torch.empty_like(t)
            run(p, t, ctx.grad_true)
        ctx.grad_pred = torch.empty_like(p) if (grad_mode and ctx.needs_input_grad[1]) else None
        run(t, p, ctx.grad_pred)
        ctx.dtypes = (true.dtype, pred.dtype)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        gt = gp = None
        if ctx.grad_true is not None:
            gt = (ctx.grad_true * go).to(ctx.dtypes[0])
        if ctx.grad_pred is not None:
            gp = (ctx.grad_pred * go).to(ctx.dtypes[1])
        return gt, gp, None, None, None, None, None, None


class LeastSquaresFn(torch.autograd.Function):
    """LeastSquares.__call__ (torch/classes.py:358-371) -> 0-dim loss in fp32 like the reference (``:319``)."""

    @staticmethod
    def forward(ctx, true, pred, render_size, grad_mode=True):
        _require_cuda(pred, "pred"); _require_cuda(true, "true")
        dev = pred.device
        img = _image(true)
        p, tag = _params(pred)
        B = p.shape[0]
        if img.shape[0] != B:
            raise ValueError("true and pred disagree on the batch size")
        row_off, col_off = nearest_offsets(img.shape[2], img.shape[3], render_size, dev)
        want_grad = grad_mode and ctx.needs_input_grad[1]
        loss = torch.empty((), dtype=torch.float64, device=dev)
        grad = torch.empty_like(p) if want_grad else None
        scratch = _get_scratch(dev, B, render_size)
        with _on_device(dev):
            rc = _lib.lib().sq_least_squares(
                _ptr(p), tag, B, render_size, _ptr(img), img.shape[2] * img.shape[3], _ptr(row_off), _ptr(col_off),
                _ptr(loss), None, _ptr(grad), _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_least_squares")
        ctx.grad = grad
        ctx.pred_dtype = pred.dtype
        return loss.to(pred.dtype if pred.dtype.is_floating_point else torch.float32)

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        g = None
        if ctx.grad is not None:
            g = (ctx.grad * go).to(ctx.pred_dtype)
        return None, g, None, None


class LsqEnergyFn(torch.autograd.Function):
    """LeastSquares.energy_function (torch/classes.py:318-356) on a packed point list -> (B,) energies."""

    @staticmethod
    def forward(ctx, params, packed, offsets, max_points, grad_mode=True):
        _require_cuda(params, "params")
        dev = params.device
        p, tag = _params(params)
        B = p.shape[0]
        want_grad = grad_mode and ctx.needs_input_grad[0]
        per = torch.empty(B, dtype=torch.float64, device=dev)
        grad = torch.empty_like(p) if want_grad else None
        L = _lib.lib()
        scratch = _get_scratch(dev, B, 0, need=L.sq_points_scratch_bytes(B, max_points))
        with _on_device(dev):
            rc = L.sq_least_squares_points(_ptr(p), tag, B, _ptr(packed), packed.shape[1], _ptr(offsets), max_points, None,
                                           _ptr(per), _ptr(grad), _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_least_squares_points")
        ctx.grad = grad
        ctx.pred_dtype = params.dtype
        return per.to(params.dtype if params.dtype.is_floating_point else torch.float32)

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        g = None
        if ctx.grad is not None:
            g = (ctx.grad * go.reshape(-1, 1).to(ctx.grad.dtype)).to(ctx.pred_dtype)
        return g, None, None, None, None


def pack_points(batch_points, device):
    """List of (3, m_i) tensors -> ((3, stride) fp32 structure-of-arrays buffer, int64 offsets [B+1] on the device, max m_i).
    The sizes are host metadata (tensor shapes): no device synchronisation."""
    counts = []
    for pts in batch_points:
        if pts.dim() != 2 or pts.shape[0] != 3:
            raise ValueError(f"expected point lists of shape (3, m), got {tuple(pts.shape)}")
        counts.append(int(pts.shape[1]))
    total = sum(counts)
    stride = max(4, (total + 3) // 4 * 4)
    packed = torch.zeros((3, stride), dtype=torch.float32, device=device)
    if total:
        packed[:, :total].copy_(torch.cat([pts.detach().to(device=device, dtype=torch.float32) for pts in batch_points], dim=1))
    offsets = torch.tensor(np.concatenate(([0], np.cumsum(counts))), dtype=torch.int64).to(device)
    return packed, offsets, max(counts) if counts else 0


def lsq_energy(batch_points, params: torch.Tensor) -> torch.Tensor:
    if len(batch_points) != params.shape[0]:
        raise ValueError("one point list per parameter row is required")
    _require_cuda(params, "params")
    packed, offsets, max_points = pack_points(batch_points, params.device)
    return LsqEnergyFn.apply(params, packed, offsets, max_points, torch.is_grad_enabled())


def iou_counts(true: torch.Tensor, pred: torch.Tensor, n: int, step: float, z0: float = 0.0):
    """(intersection[B], union[B]) int64 voxel counts of F<=1 (torch/classes.py:433-438).  Forward only."""
    _require_cuda(pred, "pred"); _require_cuda(true, "true")
    dev = pred.device
    if true.dtype == torch.float64 or pred.dtype == torch.float64:
        true, pred = true.double(), pred.double()
    t, tag = _params(true)
    p, _ = _params(pred)
    B = p.shape[0]
    if t.shape[0] != B:
        raise ValueError("true and pred disagree on the batch size")
    out = torch.empty((2, B), dtype=torch.int64, device=dev)
    scratch = _get_scratch(dev, B, n)
    with _on_device(dev):
        rc = _lib.lib().sq_iou_counts(_ptr(t), _ptr(p), tag, B, n, step, z0, _ptr(out[0]), _ptr(out[1]),
                                      _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "sq_iou_counts")
    return out[0], out[1]


def depth_projection(pred: torch.Tensor, n: int, step: float, z0: float, tau: float, sharpness: float) -> torch.Tensor:
    """ImplicitLoss.depth_projection (torch/classes.py:232-282): (B, n, n) fp32 render, image orientation."""
    _require_cuda(pred, "pred")
    p, tag = _params(pred)
    return _render(p, tag, n, step, z0, tau, sharpness)


def _render(p: torch.Tensor, tag: int, n: int, step: float, z0: float, tau: float, sharpness: float) -> torch.Tensor:
    dev = p.device
    B = p.shape[0]
    out = torch.empty((B, n, n), dtype=torch.float32, device=dev)
    scratch = _get_scratch(dev, B, n)
    with _on_device(dev):
        rc = _lib.lib().sq_implicit_loss(_ptr(p), tag, B, n, step, z0, None, 0, None, None, tau, sharpness, None, None,
                                         None, _ptr(out), _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "sq_implicit_loss(depth)")
    return out


class DepthProjectionFn(torch.autograd.Function):
    """Differentiable ImplicitLoss.depth_projection: the forward is the forward-only render (same bits as
    ``depth_projection``); the backward is the vector-Jacobian product kernel (sq_depth_projection_vjp), which walks the
    grid again with the upstream pixels as column weights.  Any image-space loss on the render can be trained through it;
    for the MAE against a target image the fused ImplicitLossFn is cheaper (one walk instead of two)."""

    @staticmethod
    def forward(ctx, pred, n, step, z0, tau, sharpness):
        _require_cuda(pred, "pred")
        p, tag = _params(pred)
        ctx.p, ctx.tag, ctx.pred_dtype = p, tag, pred.dtype
        ctx.args = (n, step, z0, tau, sharpness)
        return _render(p, tag, n, step, z0, tau, sharpness)

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        p, (n, step, z0, tau, sharpness) = ctx.p, ctx.args
        dev = p.device
        B = p.shape[0]
        g = go.float().contiguous()
        grad = torch.empty_like(p)
        scratch = _get_scratch(dev, B, n)
        with _on_device(dev):
            rc = _lib.lib().sq_depth_projection_vjp(_ptr(p), ctx.tag, B, n, step, z0, tau, sharpness, _ptr(g), _ptr(grad),
                                                    _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_depth_projection_vjp")
        return grad.to(ctx.pred_dtype), None, None, None, None, None


def field(params: torch.Tensor, n: int, step: float, z0: float, mode: int, sharpness: float = 0.0) -> torch.Tensor:
    """Full (B, n, n, n) fp32 grid: mode 0 = F (ins_outs), mode 1 = occupancy sigmoid(sharpness (1 - F))."""
    _require_cuda(params, "params")
    dev = params.device
    p, tag = _params(params)
    B = p.shape[0]
    out = torch.empty((B, n, n, n), dtype=torch.float32, device=dev)
    scratch = _get_scratch(dev, B, n)
    with _on_device(dev):
        rc = _lib.lib().sq_field(_ptr(p), tag, B, n, step, z0, mode, sharpness, _ptr(out), _ptr(scratch),
                                 scratch.numel(), _stream(dev))
    _lib.check(rc, "sq_field")
    return out


class OccupancyFn(torch.autograd.Function):
    """Differentiable ExplicitLoss.occupancy: the forward is the forward-only field (mode 1, same bits as ``field``); the
    backward is the vector-Jacobian product kernel (sq_occupancy_vjp), which walks the grid again with the upstream voxels
    as point weights.  Any loss on the occupancy grid can be trained through it; for the MSE against the occupancy of
    known parameters the fused ExplicitLossFn is cheaper (no grid in memory, one walk)."""

    @staticmethod
    def forward(ctx, params, n, step, z0, sharpness):
        _require_cuda(params, "params")
        p, tag = _params(params)
        ctx.p, ctx.tag, ctx.params_dtype = p, tag, params.dtype
        ctx.args = (n, step, z0, sharpness)
        return field(p, n, step, z0, 1, sharpness)

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        p, (n, step, z0, sharpness) = ctx.p, ctx.args
        dev = p.device
        B = p.shape[0]
        g = go.float().contiguous()
        grad = torch.empty_like(p)
        scratch = _get_scratch(dev, B, n)
        with _on_device(dev):
            rc = _lib.lib().sq_occupancy_vjp(_ptr(p), ctx.tag, B, n, step, z0, sharpness, _ptr(g), _ptr(grad),
                                             _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_occupancy_vjp")
        return grad.to(ctx.params_dtype), None, None, None, None


def _voxels(voxels: torch.Tensor, B: int, n: int, voxel_scale: Optional[float]) -> Tuple[torch.Tensor, int, float]:
    """Contiguous voxel grid, its dtype tag and scale: float32 as is, float64 as float32, bool as bytes with scale 1,
    uint8 with scale 1/255 (the convention of 8-bit depth images) unless `voxel_scale` says otherwise."""
    if voxels.shape != (B, n, n, n):
        raise ValueError(f"expected voxels of shape {(B, n, n, n)} (B, n, n, n) on this loss's grid, got {tuple(voxels.shape)}")
    if voxel_scale is not None and voxels.dtype != torch.uint8:
        raise ValueError(f"voxel_scale applies to uint8 voxels only (got {voxels.dtype})")
    if voxels.dtype == torch.uint8:
        return voxels.contiguous(), _lib.SQ_U8, float(voxel_scale) if voxel_scale is not None else 1.0 / 255.0
    if voxels.dtype == torch.bool:
        return voxels.contiguous().view(torch.uint8), _lib.SQ_U8, 1.0
    return voxels.float().contiguous(), _lib.SQ_F32, 1.0


class VoxelLossFn(torch.autograd.Function):
    """ExplicitLoss.voxel_loss: mult * mean((occupancy(pred) - voxels)^2) per sample, averaged over the batch, forward and
    backward in one walk (sq_voxel_loss); no occupancy grid is held in memory.  The gradient reaches ``pred`` only."""

    @staticmethod
    def forward(ctx, voxels, pred, n, step, z0, sharpness, mult, voxel_scale=None, grad_mode=True):
        _require_cuda(pred, "pred"); _require_cuda(voxels, "voxels")
        dev = pred.device
        if voxels.device != dev:
            raise ValueError(f"voxels ({voxels.device}) must be on pred's device ({dev})")
        p, tag = _params(pred)
        B = p.shape[0]
        v, vtag, scale = _voxels(voxels, B, n, voxel_scale)
        loss = torch.empty((), dtype=torch.float64, device=dev)
        grad = torch.empty_like(p) if (grad_mode and ctx.needs_input_grad[1]) else None
        scratch = _get_scratch(dev, B, n)
        with _on_device(dev):
            rc = _lib.lib().sq_voxel_loss(_ptr(v), vtag, scale, _ptr(p), tag, B, n, step, z0, sharpness, mult, _ptr(loss),
                                          None, _ptr(grad), _ptr(scratch), scratch.numel(), _stream(dev))
        _lib.check(rc, "sq_voxel_loss")
        ctx.grad = grad
        ctx.pred_dtype = pred.dtype
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, go):
        g = None
        if ctx.grad is not None:
            g = (ctx.grad * go).to(ctx.pred_dtype)
        return None, g, None, None, None, None, None, None, None


class HostContext:
    """sq_ctx wrapper: the host-buffer entry points of the C ABI (what a non-torch caller binds)."""

    def __init__(self, device: int = 0):
        self._h = ctypes.c_void_p()
        self._pending = {}
        _lib.check(_lib.lib().sq_ctx_create(device, ctypes.byref(self._h)), "sq_ctx_create")

    def close(self):
        if self._h:
            _lib.lib().sq_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _np(a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        return a, a.__array_interface__["data"][0]            # the address as an int (ctypes' data_as costs microseconds per call)

    def implicit_loss(self, pred, images, render_size, tau, sharpness, want_grad=True):
        pred, p_pred = self._np(pred, np.float32)
        images, p_img = self._np(images, np.float32)
        B = pred.shape[0]
        H, W = images.shape[-2], images.shape[-1]
        loss = ctypes.c_double()
        grad = np.empty((B, 12), dtype=np.float32) if want_grad else None
        rc = _lib.lib().sq_implicit_loss_host(self._h, p_pred, B, render_size, p_img, H, W, tau, sharpness,
                                              ctypes.cast(ctypes.byref(loss), ctypes.c_void_p),
                                              grad.ctypes.data_as(ctypes.c_void_p) if want_grad else None)
        _lib.check(rc, "sq_implicit_loss_host")
        return loss.value, grad

    def submit_implicit(self, slot, pred, images, render_size, tau, sharpness, want_grad=True, image_scale=None):
        """First half of a pipelined ImplicitLoss call on slot 0..3 (sq_implicit_loss_host_submit).  `images` is a
        float32 or uint8 numpy array (B, [1,] H, W) -- uint8 images are divided by 255 on the device unless image_scale
        says otherwise; of pinned images (e.g. a pinned torch tensor's .numpy()) only the sampled rows cross PCIe.  Both
        arrays are kept alive, and must stay unchanged, until result(slot)."""
        pred, p_pred = self._np(pred, np.float32)
        if images.dtype == np.uint8:
            images, tag, scale = np.ascontiguousarray(images), _lib.SQ_U8, 1.0 / 255.0
        else:
            images, tag, scale = np.ascontiguousarray(images, dtype=np.float32), _lib.SQ_F32, 1.0
        if image_scale is not None:
            scale = float(image_scale)
        B = pred.shape[0]
        H, W = images.shape[-2], images.shape[-1]
        rc = _lib.lib().sq_implicit_loss_host_submit(self._h, slot, p_pred, B, render_size, images.__array_interface__["data"][0],
                                                     tag, H, W, scale, tau, sharpness, 1 if want_grad else 0)
        _lib.check(rc, "sq_implicit_loss_host_submit")
        self._pending[slot] = (pred, images, B, want_grad)

    def result(self, slot):
        """Second half: blocks until the slot's call is done; returns (loss, grad or None)."""
        pred, images, B, want_grad = self._pending.pop(slot)
        loss = ctypes.c_double()
        grad = np.empty((B, 12), dtype=np.float32) if want_grad else None
        rc = _lib.lib().sq_implicit_loss_host_wait(self._h, slot, ctypes.addressof(loss),
                                                   grad.__array_interface__["data"][0] if want_grad else None)
        _lib.check(rc, "sq_implicit_loss_host_wait")
        return loss.value, grad

    def explicit_loss(self, true, pred, render_size, want_grad=True):
        true, p_true = self._np(true, np.float32)
        pred, p_pred = self._np(pred, np.float32)
        B = pred.shape[0]
        loss = ctypes.c_double()
        grad = np.empty((B, 12), dtype=np.float32) if want_grad else None
        rc = _lib.lib().sq_explicit_loss_host(self._h, p_true, p_pred, B, render_size,
                                              ctypes.cast(ctypes.byref(loss), ctypes.c_void_p),
                                              grad.ctypes.data_as(ctypes.c_void_p) if want_grad else None)
        _lib.check(rc, "sq_explicit_loss_host")
        return loss.value, grad

    def iou_counts(self, true, pred, render_size):
        true, p_true = self._np(true, np.float32)
        pred, p_pred = self._np(pred, np.float32)
        B = pred.shape[0]
        inter, uni = np.empty(B, dtype=np.int64), np.empty(B, dtype=np.int64)
        rc = _lib.lib().sq_iou_counts_host(self._h, p_true, p_pred, B, render_size,
                                           inter.ctypes.data_as(ctypes.c_void_p), uni.ctypes.data_as(ctypes.c_void_p))
        _lib.check(rc, "sq_iou_counts_host")
        return inter, uni
