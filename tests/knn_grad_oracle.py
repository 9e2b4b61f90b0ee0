"""TEST INFRASTRUCTURE ONLY -- ctypes/numpy binding of tests/knn_grad_oracle.c: the K-NN distance
gradient as a sequential C loop, the bitwise target of b200pci_knn_backward_det (and of the atomic
entry point's grad_q).

The library is compiled with gcc (the oracle's flags) into a per-user temporary directory, keyed by
the source's hash, so that running the tests writes nothing into the repository tree.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "knn_grad_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"mocopci_grad_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, f"libknn_grad_oracle_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11",
                                   "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = ctypes.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def knn_backward(q, r, idx, grad_dist):
    """q [B,S,3], r [B,N,3], idx [B,S,K] (any integer dtype), grad_dist [B,S,K] -> (gq [B,S,3], gr [B,N,3])."""
    q = np.ascontiguousarray(q, dtype=np.float32)
    r = np.ascontiguousarray(r, dtype=np.float32)
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    grad_dist = np.ascontiguousarray(grad_dist, dtype=np.float32)
    B, S, K = idx.shape
    N = r.shape[1]
    gq = np.empty((B, S, 3), np.float32)
    gr = np.empty((B, N, 3), np.float32)
    lib().orc_knn_backward(B, S, N, K, _p(q), _p(r), _p(idx), _p(grad_dist), _p(gq), _p(gr))
    return gq, gr
