"""ctypes loader for the host build of the fused voxel loss (tests/emu/emu_voxel.cpp) -- TEST TOOL ONLY."""
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
        src = os.path.join(HERE, "emu_voxel.cpp")
        csrc = os.path.join(ROOT, "sq_recovery_b200", "csrc")
        # the temporary directory is shared with other checkouts: the cached build is named after what it was built from
        h = hashlib.sha256()
        for path in (src, os.path.join(csrc, "sq_core.cuh"), os.path.join(csrc, "sq_tables.inc")):
            h.update(open(path, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libsqemu_voxel_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            try:
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", csrc, "-x", "c++", src, "-o", tmp])
                os.replace(tmp, out)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        _lib = ctypes.CDLL(out)
        _lib.emu_voxel_set_bits.argtypes = [ctypes.c_float]
    return _lib


def voxel_loss(params, voxels, n, step, z0, k=5.0, mult=100.0, bits=0.0):
    """Per-sample loss mult * mean_vox (v - o)^2, (B,), and its gradient d loss[b] / d params[b], (B, 12); voxels (B, n, n, n)
    fp32, index order [x][y][z].  `bits` > 0 cuts at that many bits instead of the product's choice (measuring the cut)."""
    params = np.ascontiguousarray(np.asarray(params, dtype=np.float64))
    voxels = np.ascontiguousarray(np.asarray(voxels, dtype=np.float32))
    B = len(params)
    assert voxels.shape == (B, n, n, n)
    loss, grad = np.zeros(B), np.zeros((B, 12))
    dp = ctypes.POINTER(ctypes.c_double)
    L = lib()
    L.emu_voxel_set_bits(float(bits))
    try:
        L.emu_voxel_loss(params.ctypes.data_as(dp), B, n, ctypes.c_double(step), ctypes.c_double(z0),
                         voxels.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), ctypes.c_float(k), ctypes.c_float(mult),
                         loss.ctypes.data_as(dp), grad.ctypes.data_as(dp))
    finally:
        L.emu_voxel_set_bits(0.0)
    return loss, grad
