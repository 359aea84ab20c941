"""ctypes loader for the host build of sq_core.cuh (tests/emu/emu.cpp) -- TEST TOOL ONLY."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
_lib = None


def lib():
    global _lib
    if _lib is None:
        flags = os.environ.get("SQ_EMU_FLAGS", "").split()            # experiments: -DSQ_KREFINE=32.0f ...
        src = os.path.join(HERE, "emu.cpp")
        csrc = os.path.join(ROOT, "sq_recovery_b200", "csrc")
        # the temporary directory is shared with other checkouts: the cached build is named after what it was built from
        h = hashlib.sha256(" ".join(flags).encode())
        for path in (src, os.path.join(csrc, "sq_core.cuh"), os.path.join(csrc, "sq_tables.inc")):
            h.update(open(path, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libsqemu_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            try:
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", *flags, "-I", csrc,
                                       "-x", "c++", src, "-o", tmp])
                os.replace(tmp, out)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        _lib = ctypes.CDLL(out)
    return _lib


def _f32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _ptr(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t)) if a is not None else None


def implicit(pred, target, n, step, z0, tau, k, want_grad=True, want_depth=False):
    pred, B = _f64(pred), len(pred)
    target = _f32(target) if target is not None else None
    loss = ctypes.c_double()
    grad = np.zeros((B, 12)) if want_grad else None
    depth = np.zeros((B, n, n), dtype=np.float32) if want_depth else None
    lib().emu_implicit(_ptr(pred, ctypes.c_double), B, n, ctypes.c_double(step), ctypes.c_double(z0),
                       _ptr(target, ctypes.c_float), ctypes.c_float(tau), ctypes.c_float(k), ctypes.byref(loss),
                       _ptr(grad, ctypes.c_double), _ptr(depth, ctypes.c_float))
    return loss.value, grad, depth


def explicit(true, pred, n, step, z0, k=5.0, mult=100.0, want_grad=True):
    true, pred, B = _f64(true), _f64(pred), len(pred)
    loss = ctypes.c_double()
    grad = np.zeros((B, 12)) if want_grad else None
    lib().emu_explicit(_ptr(true, ctypes.c_double), _ptr(pred, ctypes.c_double), B, n, ctypes.c_double(step),
                       ctypes.c_double(z0), ctypes.c_float(k), ctypes.c_float(mult), ctypes.byref(loss),
                       _ptr(grad, ctypes.c_double))
    return loss.value, grad


def iou(true, pred, n, step):
    true, pred, B = _f64(true), _f64(pred), len(pred)
    inter, uni = np.zeros(B, dtype=np.int64), np.zeros(B, dtype=np.int64)
    lib().emu_iou(_ptr(true, ctypes.c_double), _ptr(pred, ctypes.c_double), B, n, ctypes.c_double(step),
                  _ptr(inter, ctypes.c_longlong), _ptr(uni, ctypes.c_longlong))
    return inter, uni


def lsq(pred, points, offsets, want_grad=True):
    pred, B = _f64(pred), len(pred)
    points = _f32(points)
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    loss = ctypes.c_double()
    grad = np.zeros((B, 12)) if want_grad else None
    lib().emu_lsq(_ptr(pred, ctypes.c_double), B, _ptr(points, ctypes.c_float), _ptr(offsets, ctypes.c_int),
                  ctypes.byref(loss), _ptr(grad, ctypes.c_double))
    return loss.value, grad


def check_culling(params, n, step, z0, clamp, bound, f_min):
    """(violations, proven-empty patches, patches): see emu_check_culling in emu.cpp."""
    params, B = _f64(params), len(params)
    pe, pt = ctypes.c_longlong(), ctypes.c_longlong()
    fn = lib().emu_check_culling
    fn.restype = ctypes.c_longlong
    bad = fn(_ptr(params, ctypes.c_double), B, n, ctypes.c_double(step), ctypes.c_double(z0), int(clamp),
             ctypes.c_float(bound), ctypes.c_double(f_min), ctypes.byref(pe), ctypes.byref(pt))
    return int(bad), int(pe.value), int(pt.value)


def check_walk_estimate(params, n, step, z0, bound, die):
    """(violations, groups whose estimate the early exit shortened, live groups): see emu_check_walk_estimate in emu.cpp."""
    params, B = _f64(params), len(params)
    cut, live = ctypes.c_longlong(), ctypes.c_longlong()
    fn = lib().emu_check_walk_estimate
    fn.restype = ctypes.c_longlong
    bad = fn(_ptr(params, ctypes.c_double), B, n, ctypes.c_double(step), ctypes.c_double(z0), ctypes.c_float(bound),
             ctypes.c_float(die), ctypes.byref(cut), ctypes.byref(live))
    return int(bad), int(cut.value), int(live.value)
