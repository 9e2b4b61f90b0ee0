"""TEST INFRASTRUCTURE ONLY -- ctypes/numpy binding of tests/grad_oracle.c: the row-gather and
Chamfer gradients as sequential C loops, the bitwise targets of the deterministic backwards next to
oracle/cpu.py's gather_grad / group_grad / three_interpolate_grad.

The library is compiled with gcc (the oracle's flags) into a per-user temporary directory, keyed by
the source's hash, so that running the tests writes nothing into the repository tree.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "grad_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"mocopci_grad_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, f"libgrad_oracle_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11",
                                   "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = ctypes.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def index_rows_grad(grad_out, idx, N):
    """grad_out [B,...,C] float32, idx [B,...] (any integer dtype) -> grad_points [B,N,C]."""
    grad_out = np.ascontiguousarray(grad_out, dtype=np.float32)
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    B, C = grad_out.shape[0], grad_out.shape[-1]
    T = idx.size // B if B else 0
    g = np.zeros((B, N, C), np.float32)
    lib().orc_index_rows_grad(B, N, ctypes.c_longlong(T), C, _p(grad_out), _p(idx), _p(g))
    return g


def chamfer_backward(x, y, ix, iy, grad_loss=1.0):
    """x [B,N,3], y [B,M,3], nearest-neighbour indices ix [B,N], iy [B,M] -> (gx [B,N,3], gy [B,M,3])."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32)
    ix = np.ascontiguousarray(ix, dtype=np.int32)
    iy = np.ascontiguousarray(iy, dtype=np.int32)
    B, N, _ = x.shape
    M = y.shape[1]
    gx = np.empty((B, N, 3), np.float32)
    gy = np.empty((B, M, 3), np.float32)
    lib().orc_chamfer_backward(B, N, M, _p(x), _p(y), _p(ix), _p(iy), ctypes.c_float(grad_loss), _p(gx), _p(gy))
    return gx, gy
