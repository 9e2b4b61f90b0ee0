"""ctypes binding of ``libb200pci.so`` (the C ABI declared in ``include/b200pci.h``).

There is no CPU or PyTorch fallback: if the CUDA library is missing or fails to load, importing
this module raises, and every op raises ``RuntimeError`` on a non-zero return code (the
reference's launchers ``exit(-1)`` instead, e.g. pointnet2/src/sampling_gpu.cu:39-43).
"""
import ctypes
import os

import torch  # noqa: F401  (loads libcudart.so.12 into the process before our library)

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200PCI_LIB: developer hook to load an experimental build of the same library
LIB_PATH = os.environ.get("B200PCI_LIB") or os.path.join(_HERE, "libb200pci.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build the sm_100a kernels first with "
        "`python -m mocopci_b200.build` (or __graft_entry__.build()). "
        "mocopci_b200 has no CPU fallback.")

lib = ctypes.CDLL(LIB_PATH)

_c = ctypes
_P, _I, _F, _L, _Z = _c.c_void_p, _c.c_int, _c.c_float, _c.c_int64, _c.c_size_t

# name -> (restype, argtypes); mirrors include/b200pci.h one to one
PROTOTYPES = {
    "b200pci_version": (_I, []),
    "b200pci_last_error": (_c.c_char_p, []),
    "b200pci_knn_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "b200pci_knn": (_I, [_I, _I, _I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _P, _P, _Z, _P]),
    "b200pci_knn_cosine_workspace_bytes": (_Z, [_I, _I, _I, _I, _I]),
    "b200pci_knn_cosine": (_I, [_I, _I, _I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _P, _P, _Z, _P]),
    "b200pci_knn_host": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "b200pci_host_release": (_I, []),
    "b200pci_furthest_point_sampling": (_I, [_I, _I, _I, _P, _P, _P, _P]),
    "b200pci_index_points_rows": (_I, [_I, _I, _c.c_longlong, _I, _P, _L, _L, _L, _P, _I, _P, _P]),
    "b200pci_index_points_rows_grad": (_I, [_I, _I, _c.c_longlong, _I, _P, _P, _I, _P, _P]),
    "b200pci_group_concat": (_I, [_I, _I, _I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I,
                                  _P, _P, _P]),
    "b200pci_gather_points": (_I, [_I, _I, _I, _I, _P, _P, _P, _P]),
    "b200pci_gather_points_grad": (_I, [_I, _I, _I, _I, _P, _P, _P, _P]),
    "b200pci_ball_query_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "b200pci_ball_query": (_I, [_I, _I, _I, _F, _I, _P, _P, _P, _P, _Z, _P]),
    "b200pci_group_points": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "b200pci_group_points_grad": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "b200pci_query_group": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P]),
    "b200pci_three_nn_workspace_bytes": (_Z, [_I, _I, _I]),
    "b200pci_three_nn": (_I, [_I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "b200pci_three_nn_weights": (_I, [_I, _I, _I, _P, _P, _F, _P, _P, _P, _P, _Z, _P]),
    "b200pci_three_interpolate": (_I, [_I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "b200pci_three_interpolate_grad": (_I, [_I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "b200pci_chamfer_workspace_bytes": (_Z, [_I, _I, _I]),
    "b200pci_chamfer_forward": (_I, [_I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L,
                                     _P, _P, _P, _P, _P, _P, _Z, _P]),
    "b200pci_chamfer_backward": (_I, [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "b200pci_chamfer_backward_det_workspace_bytes": (_Z, [_I, _I, _I]),
    "b200pci_chamfer_backward_det": (_I, [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "b200pci_scatter_workspace_bytes": (_Z, [_I, _I, _c.c_longlong]),
    "b200pci_gather_points_grad_det": (_I, [_I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "b200pci_group_points_grad_det": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "b200pci_three_interpolate_grad_det": (_I, [_I, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "b200pci_index_points_rows_grad_det": (_I, [_I, _I, _c.c_longlong, _I, _P, _P, _I, _P, _P, _Z, _P]),
    "b200pci_knn_backward": (_I, [_I, _I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _P, _P, _P, _P]),
    "b200pci_knn_backward_det": (_I, [_I, _I, _I, _I, _P, _L, _L, _L, _P, _L, _L, _L, _P, _I, _P, _P, _P,
                                      _P, _Z, _P]),
    "b200pci_ball_query_p3d": (_I, [_I, _I, _I, _I, _F, _P, _L, _L, _L, _P, _L, _L, _L, _P, _P, _P, _P, _P, _P]),
    "b200pci_fps_p3d": (_I, [_I, _I, _I, _P, _L, _L, _L, _P, _P, _P, _P, _P, _P]),
    "b200pci_emd_workspace_bytes": (_Z, [_I, _I, _I]),
    "b200pci_emd_approxmatch": (_I, [_I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "b200pci_emd_matchcost": (_I, [_I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "b200pci_emd_matchcost_grad": (_I, [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "b200pci_emd_cost": (_I, [_I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "b200pci_probe_fp32": (_I, [_I, _I, _P, _P, _P]),
    "b200pci_debug_set": (_I, [_I, _c.c_double]),
    "b200pci_debug_get": (_c.c_double, [_I]),
}

for _name, (_res, _args) in PROTOTYPES.items():
    _fn = getattr(lib, _name)  # AttributeError here == the library is stale: rebuild
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc, what=""):
    if rc != 0:
        msg = lib.b200pci_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"b200pci {what} failed ({rc}): {msg}")


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def stream_ptr():
    """cudaStream_t of torch's current stream on the current device. The model makes ~600 calls
    into the library per forward and is host-bound, so this avoids building a ``torch.cuda.Stream``
    object per call (3.2 us -> 0.2 us) where torch exposes the raw handle."""
    if _raw_stream is not None and _raw_device is not None:
        return _raw_stream(_raw_device())
    return torch.cuda.current_stream().cuda_stream


def workspace(nbytes, device):
    """Scratch from torch's caching allocator (stream-ordered on the current stream)."""
    return torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=device)


def require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError("mocopci_b200 ops need CUDA tensors (there is no CPU fallback)")


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_GUARD = _NoGuard()


def on_device(t):
    """Device guard for the tensor's GPU (the reference has none: the current device must equal
    the tensors' device there); free when that device is already current -- the model makes ~500
    calls per forward, so the host-side cost of a call matters. Raises for CPU tensors."""
    require_cuda(t)
    dev = t.device
    if dev.index is None or dev.index == (_raw_device() if _raw_device is not None else torch.cuda.current_device()):
        return _NO_GUARD
    return torch.cuda.device(dev)
