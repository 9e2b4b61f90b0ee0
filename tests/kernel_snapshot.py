"""TEST INFRASTRUCTURE ONLY: a stored snapshot of kernel outputs on the GPU parity tests' seeded
inputs (tests/golden/kernel_snapshot.npz, written by tests/golden/make_kernel_snapshot.py).

The tests used to compare these outputs, bit for bit, with the reference's own CUDA kernels
compiled from a MoCoPCI checkout (tests/refgpu.py), which the repository does not carry. The
snapshot was recorded on a B200 from this project's kernels at the change that added it; its
``source`` entry says so. A mismatch therefore means "differs from that recorded output", not
"proven to differ from the reference". Where the C oracle covers an operator, the tests keep an
independent check against it next to the snapshot.

An entry is stored whole when it is small. A larger one is stored as the SHA-256 of its bytes,
which still pins every element bit for bit, plus a fixed sample of elements for the message when
it differs. Comparisons with a tolerance use entries stored whole.
"""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kernel_snapshot.npz")
FULL_BYTES = 64 * 1024
SAMPLE = 512


def _np(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a)


def _digest(a):
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)


def record(store, key, a, full=False):
    """Add array ``a`` under ``key`` to the dict ``store`` (file entries ``key/...``)."""
    a = _np(a)
    store[key + "/shape"] = np.asarray(a.shape, np.int64)
    if full or a.nbytes <= FULL_BYTES:
        store[key + "/full"] = a
        return
    flat = a.reshape(-1)
    pos = np.sort(np.random.default_rng(len(flat)).choice(len(flat), min(SAMPLE, len(flat)), replace=False))
    store[key + "/sha256"] = _digest(a)
    store[key + "/pos"] = pos
    store[key + "/sample"] = flat[pos]


_cache = None


def _load():
    global _cache
    if _cache is None:
        with np.load(PATH) as z:
            _cache = {k: z[k] for k in z.files}
    return _cache


def get(key):
    """The stored array (entries stored whole only)."""
    return _load()[key + "/full"]


def check(key, a, rtol=None, atol=0.0):
    """Assert that ``a`` equals the snapshot entry ``key``: bit for bit, or within rtol / atol."""
    g = _load()
    assert key + "/shape" in g, f"no snapshot entry {key!r}"
    a = _np(a)
    assert tuple(a.shape) == tuple(g[key + "/shape"]), f"{key}: shape {a.shape} != {tuple(g[key + '/shape'])}"
    if key + "/full" in g:
        want = g[key + "/full"]
        assert a.dtype == want.dtype, f"{key}: dtype {a.dtype} != {want.dtype}"
        if rtol is None:
            bad = int((a.reshape(-1).view(np.uint8).reshape(a.size, -1) !=
                       want.reshape(-1).view(np.uint8).reshape(want.size, -1)).any(-1).sum()) if a.size else 0
            assert bad == 0, f"{key}: {bad} of {a.size} elements differ from the kernel snapshot"
        else:
            np.testing.assert_allclose(a, want, rtol=rtol, atol=atol, err_msg=f"{key} vs the kernel snapshot")
        return
    assert rtol is None, f"{key}: a tolerance needs an entry stored whole"
    if not np.array_equal(_digest(a), g[key + "/sha256"]):
        flat = a.reshape(-1)
        pos, want = g[key + "/pos"], g[key + "/sample"]
        bad = int((flat[pos].view(np.uint8).reshape(len(pos), -1) !=
                   want.view(np.uint8).reshape(len(pos), -1)).any(-1).sum())
        raise AssertionError(f"{key}: differs from the kernel snapshot ({bad} of {len(pos)} sampled elements)")
