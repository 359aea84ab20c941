"""ctypes loader for the host build of the LeastSquares normal equations (tests/emu/emu_lsq_normal.cpp) -- TEST TOOL ONLY."""
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
        src = os.path.join(HERE, "emu_lsq_normal.cpp")
        csrc = os.path.join(ROOT, "sq_recovery_b200", "csrc")
        # the temporary directory is shared with other checkouts: the cached build is named after what it was built from
        h = hashlib.sha256()
        for path in (src, os.path.join(csrc, "sq_core.cuh"), os.path.join(csrc, "sq_tables.inc")):
            h.update(open(path, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libsqemu_lsq_normal_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            try:
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", csrc, "-x", "c++", src, "-o", tmp])
                os.replace(tmp, out)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        _lib = ctypes.CDLL(out)
    return _lib


def normal_equations(params, batch_points):
    """Per-sample energy (B,), gradient (B, 12) and J^T J (B, 12, 12) of the (3, m_i) point lists, all fp64."""
    params = np.ascontiguousarray(np.asarray(params, dtype=np.float64))
    B = len(params)
    assert len(batch_points) == B
    pts = [np.asarray(p, dtype=np.float32).reshape(3, -1) for p in batch_points]
    packed = np.ascontiguousarray(np.concatenate([p.T for p in pts], axis=0) if B else np.zeros((0, 3), np.float32))
    offsets = np.ascontiguousarray(np.concatenate(([0], np.cumsum([p.shape[1] for p in pts]))).astype(np.int64))
    energy, grad, jtj = np.zeros(B), np.zeros((B, 12)), np.zeros((B, 12, 12))
    dp = ctypes.POINTER(ctypes.c_double)
    lib().emu_lsq_normal(params.ctypes.data_as(dp), B, packed.ctypes.data_as(ctypes.POINTER(ctypes.c_float)),
                         offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), energy.ctypes.data_as(dp),
                         grad.ctypes.data_as(dp), jtj.ctypes.data_as(dp))
    return energy, grad, jtj
