"""Drop-in for the reference's pybind module ``emd_cuda`` (models/EMD/cuda/emd.cpp:23-27).

Callee allocates the outputs, like ``at::zeros`` in emd_kernel.cu:188-189,275,392-393. Shape errors
raise ``RuntimeError`` (the reference's CHECK_EQ / TORCH_CHECK). Only float32 is implemented (the
reference also dispatches float64, which MoCoPCI never uses). Launches on the CURRENT stream; the
reference uses the legacy default stream (emd_kernel.cu:192), a latent ordering hazard.
"""
import torch

from . import _lib

_L = _lib.lib


def _check_pair(xyz1, xyz2):
    _lib.require_cuda(xyz1, xyz2)
    if xyz1.dim() != 3 or xyz2.dim() != 3 or xyz1.size(2) != 3 or xyz2.size(2) != 3:
        raise RuntimeError("xyz1 / xyz2 must be (B, N, 3)")
    if xyz2.size(0) != xyz1.size(0):
        raise RuntimeError("CHECK_EQ failed: xyz2.size(0) == b")
    if xyz2.device != xyz1.device:
        raise RuntimeError("xyz1 and xyz2 must be on the same device")
    for t, n in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        if not t.is_contiguous():
            raise RuntimeError(f"{n} must be contiguous")
        if t.dtype != torch.float32:
            raise RuntimeError(f"{n} must be float32")
    return xyz1.size(0), xyz1.size(1), xyz2.size(1)


def _check_match(match, b, n, m, xyz1):
    """The kernels read B*N2*N1 floats of ``match`` in row-major (B, N2, N1) order on xyz1's device."""
    if (tuple(match.shape) != (b, m, n) or not match.is_contiguous() or match.dtype != torch.float32
            or match.device != xyz1.device):
        raise RuntimeError("match must be a contiguous float32 (B, N2, N1) tensor on xyz1's device")


def approxmatch_forward(xyz1, xyz2):
    """ApproxMatchForward, emd_kernel.cu:175-197 -> match (B, N2, N1)."""
    b, n, m = _check_pair(xyz1, xyz2)
    with _lib.on_device(xyz1):
        match = torch.empty((b, m, n), dtype=torch.float32, device=xyz1.device)
        ws = _lib.workspace(_L.b200pci_emd_workspace_bytes(b, n, m), xyz1.device)
        _lib.check(_L.b200pci_emd_approxmatch(b, n, m, xyz1.data_ptr(), xyz2.data_ptr(),
                                              match.data_ptr(), ws.data_ptr(), ws.numel(),
                                              _lib.stream_ptr()), "emd_approxmatch")
    return match


def matchcost_forward(xyz1, xyz2, match):
    """MatchCostForward, emd_kernel.cu:261-283 -> cost (B)."""
    b, n, m = _check_pair(xyz1, xyz2)
    _check_match(match, b, n, m, xyz1)
    with _lib.on_device(xyz1):
        cost = torch.empty((b,), dtype=torch.float32, device=xyz1.device)
        ws = _lib.workspace(_L.b200pci_emd_workspace_bytes(b, n, m), xyz1.device)
        _lib.check(_L.b200pci_emd_matchcost(b, n, m, xyz1.data_ptr(), xyz2.data_ptr(),
                                            match.data_ptr(), cost.data_ptr(), ws.data_ptr(),
                                            ws.numel(), _lib.stream_ptr()), "emd_matchcost")
    return cost


def emd_cost(xyz1, xyz2):
    """Forward-only ``matchcost_forward(xyz1, xyz2, approxmatch_forward(xyz1, xyz2))`` that never
    stores the (B, N2, N1) match matrix (b200pci_emd_cost); not part of the reference's module,
    used by :func:`mocopci_b200.ops.earth_mover_distance` when no gradient is needed."""
    b, n, m = _check_pair(xyz1, xyz2)
    with _lib.on_device(xyz1):
        cost = torch.empty((b,), dtype=torch.float32, device=xyz1.device)
        ws = _lib.workspace(_L.b200pci_emd_workspace_bytes(b, n, m), xyz1.device)
        _lib.check(_L.b200pci_emd_cost(b, n, m, xyz1.data_ptr(), xyz2.data_ptr(), cost.data_ptr(),
                                       ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "emd_cost")
    return cost


def matchcost_backward(grad_cost, xyz1, xyz2, match):
    """MatchCostBackward, emd_kernel.cu:377-402 -> [grad1 (B,N1,3), grad2 (B,N2,3)]."""
    b, n, m = _check_pair(xyz1, xyz2)
    _check_match(match, b, n, m, xyz1)
    if grad_cost.numel() != b or grad_cost.device != xyz1.device:
        raise RuntimeError("grad_cost must have B elements on xyz1's device")
    grad_cost = grad_cost.contiguous().float()
    with _lib.on_device(xyz1):
        g1 = torch.empty((b, n, 3), dtype=torch.float32, device=xyz1.device)
        g2 = torch.empty((b, m, 3), dtype=torch.float32, device=xyz1.device)
        _lib.check(_L.b200pci_emd_matchcost_grad(b, n, m, grad_cost.data_ptr(), xyz1.data_ptr(),
                                                 xyz2.data_ptr(), match.data_ptr(), g1.data_ptr(),
                                                 g2.data_ptr(), _lib.stream_ptr()),
                   "emd_matchcost_grad")
    return [g1, g2]
