"""Chamfer distance and pytorch3d shims.

The reference gets both from pytorch3d 0.7.5 (environment.yaml:90), which is neither vendored nor
installed here: ``models/utils.py:36-45`` calls ``pytorch3d.loss.chamfer_distance(pc1, pc2)`` with
defaults, ``models/pointconv_util.py:910`` calls ``pytorch3d.ops.knn_points(xyz2, xyz1, K=16)``.
These functions keep those call signatures (for the arguments MoCoPCI uses) on top of the fused
B200 neighbour kernel, in the arithmetic of pytorch3d's CUDA kernel (``dist += diff * diff`` over
x, y, z as nvcc contracts it: fma(dz,dz,fma(dy,dy,dx*dx)) -- DIST_DIRECT_XYZ). PARITY UNPINNED
against pytorch3d itself, which cannot be obtained here (DESIGN.md section 4).
"""
from collections import namedtuple

import torch
from torch.autograd import Function

from . import _lib
from .pointconv_util import DIST_DIRECT_XYZ, _knn

_L = _lib.lib


class _ChamferFunction(Function):
    @staticmethod
    def forward(ctx, x, y):
        _lib.require_cuda(x, y)
        B, N, _ = x.shape
        M = y.shape[1]
        dev = x.device
        with torch.cuda.device(dev):
            dist_x = torch.empty((B, N), dtype=torch.float32, device=dev)
            dist_y = torch.empty((B, M), dtype=torch.float32, device=dev)
            idx_x = torch.empty((B, N), dtype=torch.int32, device=dev)
            idx_y = torch.empty((B, M), dtype=torch.int32, device=dev)
            loss = torch.empty((1,), dtype=torch.float32, device=dev)
            ws = _lib.workspace(_L.b200pci_chamfer_workspace_bytes(B, N, M), dev)
            xs, ys = x.stride(), y.stride()
            _lib.check(_L.b200pci_chamfer_forward(
                B, N, M, x.data_ptr(), xs[0], xs[1], xs[2], y.data_ptr(), ys[0], ys[1], ys[2],
                dist_x.data_ptr(), idx_x.data_ptr(), dist_y.data_ptr(), idx_y.data_ptr(),
                loss.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "chamfer_forward")
        ctx.save_for_backward(x, y, idx_x, idx_y)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_loss):
        x, y, idx_x, idx_y = ctx.saved_tensors
        B, N, _ = x.shape
        M = y.shape[1]
        xc, yc = x.contiguous(), y.contiguous()
        with torch.cuda.device(x.device):
            gx = torch.empty((B, N, 3), dtype=torch.float32, device=x.device)
            gy = torch.empty((B, M, 3), dtype=torch.float32, device=x.device)
            g = grad_loss.reshape(1).contiguous().float()
            if torch.are_deterministic_algorithms_enabled():  # fixed summation order (b200pci.h, _det)
                ws = _lib.workspace(_L.b200pci_chamfer_backward_det_workspace_bytes(B, N, M), x.device)
                _lib.check(_L.b200pci_chamfer_backward_det(
                    B, N, M, xc.data_ptr(), yc.data_ptr(), idx_x.data_ptr(), idx_y.data_ptr(),
                    g.data_ptr(), gx.data_ptr(), gy.data_ptr(), ws.data_ptr(), ws.numel(),
                    _lib.stream_ptr()), "chamfer_backward_det")
            else:
                _lib.check(_L.b200pci_chamfer_backward(
                    B, N, M, xc.data_ptr(), yc.data_ptr(), idx_x.data_ptr(), idx_y.data_ptr(),
                    g.data_ptr(), gx.data_ptr(), gy.data_ptr(), _lib.stream_ptr()), "chamfer_backward")
        return gx, gy


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None,
                     weights=None, batch_reduction="mean", point_reduction="mean", norm=2,
                     **kwargs):
    """``pytorch3d.loss.chamfer_distance`` for the arguments MoCoPCI uses (all defaults):
    x (B, N, 3), y (B, M, 3) -> (loss, None),
    loss = mean_b( mean_i min_j |x_i-y_j|^2 + mean_j min_i |x_i-y_j|^2 )."""
    if (x_lengths is not None or y_lengths is not None or x_normals is not None
            or y_normals is not None or weights is not None or batch_reduction != "mean"
            or point_reduction != "mean" or norm != 2 or kwargs):
        raise NotImplementedError("mocopci_b200.chamfer_distance implements the default arguments only")
    if x.dtype != torch.float32 or y.dtype != torch.float32:
        raise RuntimeError("chamfer_distance: float32 inputs required")
    return _ChamferFunction.apply(x, y), None


def chamfer_loss(pc1, pc2):
    """models/utils.py:36-45. pc1, pc2: [B, 3, N]."""
    return chamfer_distance(pc1.permute(0, 2, 1), pc2.permute(0, 2, 1))[0]


_KNN = namedtuple("KNN", "dists idx knn")


def knn_points(p1, p2, lengths1=None, lengths2=None, norm=2, K=1, version=-1, return_nn=False,
               return_sorted=True):
    """``pytorch3d.ops.knn_points`` (models/pointconv_util.py:910): for each point of p1 the K
    nearest points of p2 -> KNN(dists (B,P1,K) squared, idx int64 (B,P1,K), knn or None)."""
    if lengths1 is not None or lengths2 is not None or norm != 2:
        raise NotImplementedError("mocopci_b200.knn_points: lengths / norm != 2 not implemented")
    idx, dists = _knn(K, p2, p1, DIST_DIRECT_XYZ, True)
    nn = None
    if return_nn:
        B, P1, _ = p1.shape
        nn = torch.gather(p2.unsqueeze(1).expand(B, P1, p2.shape[1], 3), 2,
                          idx.unsqueeze(-1).expand(B, P1, K, 3))
    return _KNN(dists=dists, idx=idx, knn=nn)


def knn_gather(x, idx, lengths=None):
    """``pytorch3d.ops.knn_gather`` (imported by models/layers.py:18): x (B, M, U), idx (B, P, K)
    -> (B, P, K, U) with out[b,p,k] = x[b, idx[b,p,k]]."""
    if lengths is not None:
        raise NotImplementedError("mocopci_b200.knn_gather: lengths not implemented")
    from .pointconv_util import index_points_group
    if x.is_cuda and x.dtype == torch.float32:
        return index_points_group(x, idx)
    B, P, K = idx.shape
    return torch.gather(x.unsqueeze(1).expand(B, P, x.shape[1], x.shape[2]), 2,
                        idx.unsqueeze(-1).expand(B, P, K, x.shape[2]))
