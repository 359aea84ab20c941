"""ctypes loader for the host build of the render's Jacobian (tests/emu/emu_jac.cpp) -- TEST TOOL ONLY."""
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
        src = os.path.join(HERE, "emu_jac.cpp")
        csrc = os.path.join(ROOT, "sq_recovery_b200", "csrc")
        # the temporary directory is shared with other checkouts: the cached build is named after what it was built from
        h = hashlib.sha256()
        for path in (src, os.path.join(csrc, "sq_core.cuh"), os.path.join(csrc, "sq_tables.inc")):
            h.update(open(path, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libsqemu_jac_{os.getuid()}_{h.hexdigest()[:16]}.so")
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


def depth_jacobian(pred, n, step, z0, tau, k):
    """(B, n, n, 12) fp32 d depth[b, row, col] / d pred[b], image orientation."""
    pred = np.ascontiguousarray(np.asarray(pred, dtype=np.float64))
    B = len(pred)
    jac = np.zeros((B, n, n, 12), dtype=np.float32)
    lib().emu_depth_jacobian(pred.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), B, n, ctypes.c_double(step),
                             ctypes.c_double(z0), ctypes.c_float(tau), ctypes.c_float(k),
                             jac.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
    return jac
