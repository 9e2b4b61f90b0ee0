"""TEST INFRASTRUCTURE ONLY -- ctypes/numpy binding of tests/p3d_oracle.c: pytorch3d-form ball query
and farthest point sampling as sequential C loops, the bitwise targets of b200pci_ball_query_p3d and
b200pci_fps_p3d.

The library is compiled with gcc (the oracle's flags) into a per-user temporary directory, keyed by
the source's hash, so that running the tests writes nothing into the repository tree.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "p3d_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"mocopci_p3d_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, f"libp3d_oracle_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = ctypes.CDLL(so)
        _lib.orc_ball_query_p3d.argtypes = [ctypes.c_int] * 4 + [ctypes.c_float] + [ctypes.c_void_p] * 6
        _lib.orc_fps_p3d.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 6
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _lengths(lengths, B, P):
    if lengths is None:
        return np.full(B, P, np.int64)
    return np.ascontiguousarray(np.asarray(lengths), dtype=np.int64)


def ball_query(p1, p2, K, radius, lengths1=None, lengths2=None):
    """p1 [B,P1,3], p2 [B,P2,3] (any layout numpy converts) -> (idx int64 [B,P1,K], dists [B,P1,K])."""
    p1 = np.ascontiguousarray(p1, dtype=np.float32)
    p2 = np.ascontiguousarray(p2, dtype=np.float32)
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    l1, l2 = _lengths(lengths1, B, P1), _lengths(lengths2, B, P2)
    idx = np.empty((B, P1, K), np.int64)
    dists = np.empty((B, P1, K), np.float32)
    lib().orc_ball_query_p3d(B, P1, P2, K, radius, _p(p1), _p(p2), _p(l1), _p(l2), _p(idx), _p(dists))
    return idx, dists


def fps(points, K, lengths=None, start=None):
    """points [B,P,3]; K an int or (B,) ints; start (B,) or None (0) -> idx int64 [B, max K]."""
    pts = np.ascontiguousarray(points, dtype=np.float32)
    B, P, _ = pts.shape
    Ks = np.full(B, K, np.int64) if np.isscalar(K) else np.ascontiguousarray(np.asarray(K), dtype=np.int64)
    M = int(Ks.max()) if B else 0
    ln = _lengths(lengths, B, P)
    st = np.zeros(B, np.int64) if start is None else np.ascontiguousarray(np.asarray(start), dtype=np.int64)
    idx = np.empty((B, M), np.int64)
    mind = np.empty(max(P, 1), np.float32)
    lib().orc_fps_p3d(B, P, M, _p(pts), _p(ln), _p(Ks), _p(st), _p(idx), _p(mind))
    return idx
