"""Chamfer distance and pytorch3d shims.

The reference gets both from pytorch3d 0.7.5 (environment.yaml:90), which is neither vendored nor
installed here: ``models/utils.py:36-45`` calls ``pytorch3d.loss.chamfer_distance(pc1, pc2)`` with
defaults, ``models/pointconv_util.py:910`` calls ``pytorch3d.ops.knn_points(xyz2, xyz1, K=16)``.
These functions keep those call signatures (for the arguments MoCoPCI uses) on top of the fused
B200 neighbour kernel, in the arithmetic of pytorch3d's CUDA kernel (``dist += diff * diff`` over
x, y, z as nvcc contracts it: fma(dz,dz,fma(dy,dy,dx*dx)) -- DIST_DIRECT_XYZ). PARITY UNPINNED
against pytorch3d itself, which cannot be obtained here (DESIGN.md section 4).

Both are differentiable like pytorch3d's: ``knn_points(...).dists`` backpropagates into both clouds
through b200pci_knn_backward (b200pci_knn_backward_det under torch.use_deterministic_algorithms),
``knn`` (return_nn) through the row-gather backward. ``chamfer_distance`` with default arguments runs
the fused Chamfer kernels; its other reduction options, per-cloud weights and the one-way form are
composed in torch from two differentiable ``knn_points(K=1)`` calls, as pytorch3d 0.7.5 does. Ragged
batches (lengths), normals and the L1 norm are not implemented here; pytorch3d's ``ball_query`` and
``sample_farthest_points``, which do take per-cloud lengths, are in p3d_ops.py.
"""
from collections import namedtuple

import torch
from torch.autograd import Function

from . import _lib
from .pointconv_util import DIST_DIRECT_XYZ, _knn, _needs_grad, index_points_group

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


def _chamfer_one_way(x, y, weights, batch_reduction, point_reduction):
    """One direction of chamfer_distance: the squared distance of each point of x to its nearest
    point of y, weighted and reduced as pytorch3d 0.7.5's _chamfer_distance_single_direction."""
    B, P = x.shape[0], x.shape[1]
    if weights is not None and not bool(weights.sum() != 0):
        # all weights zero (they are >= 0): zeros of the result's shape, still in the graph
        zero = x.sum((1, 2)) * weights * 0.0
        if point_reduction is None:
            return zero[:, None].expand(B, P)
        return zero.sum() if batch_reduction is not None else zero
    cham = knn_points(x, y, K=1).dists[..., 0]
    if weights is not None:
        cham = cham * weights.view(B, 1)
    if point_reduction == "max":
        cham = cham.max(1).values
    elif point_reduction is not None:
        cham = cham.sum(1)
        if point_reduction == "mean":
            cham = cham / max(P, 1)
    if point_reduction is not None and batch_reduction is not None:
        cham = cham.sum()
        if batch_reduction == "mean":
            cham = cham / (weights.sum() if weights is not None else max(B, 1))
    return cham


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None,
                     weights=None, batch_reduction="mean", point_reduction="mean", norm=2,
                     single_directional=False, abs_cosine=True, **kwargs):
    """``pytorch3d.loss.chamfer_distance``: x (B, N, 3), y (B, M, 3), squared L2.

    Default arguments (what MoCoPCI passes) run the fused Chamfer kernels and return (loss, None),
    loss = mean_b( mean_i min_j |x_i-y_j|^2 + mean_j min_i |x_i-y_j|^2 ).

    Every other combination is composed in torch from two differentiable ``knn_points(K=1)`` calls,
    following pytorch3d 0.7.5. Per direction (x to y; y to x the same with the clouds exchanged):
      cham_x = knn_points(x, y, K=1).dists[..., 0], then ``* weights.view(B, 1)`` if weights are given;
      point_reduction "max": .max(1).values, "sum": .sum(1), "mean": .sum(1) / N, None: per point;
      batch_reduction (only when point_reduction is not None) "sum": .sum(), "mean":
      .sum() / (weights.sum() if weights is not None else max(B, 1)), None: per cloud.
    Result: single_directional -> (cham_x, None); else with "max" (torch.maximum(cham_x, cham_y), None);
    with another point reduction (cham_x + cham_y, None); with point_reduction None
    ((cham_x, cham_y), (None, None)). If every weight is zero, each direction is zeros of its
    result's shape that stay connected to the graph (pytorch3d multiplies by 0.0).

    ValueError: an unknown reduction, point_reduction None with a batch_reduction, weights not
    shaped (B,) or negative. NotImplementedError: x_lengths / y_lengths (ragged batches), normals,
    norm != 2. abs_cosine is accepted and has no effect without normals."""
    if kwargs:
        raise NotImplementedError(f"mocopci_b200.chamfer_distance: unsupported arguments {sorted(kwargs)}")
    if x_lengths is not None or y_lengths is not None:
        raise NotImplementedError("mocopci_b200.chamfer_distance: x_lengths / y_lengths (ragged batches) "
                                  "not implemented")
    if x_normals is not None or y_normals is not None:
        raise NotImplementedError("mocopci_b200.chamfer_distance: normals not implemented")
    if norm != 2:
        raise NotImplementedError("mocopci_b200.chamfer_distance: only norm=2 is implemented")
    if batch_reduction is not None and batch_reduction not in ("mean", "sum"):
        raise ValueError('batch_reduction must be one of ["mean", "sum"] or None')
    if point_reduction is not None and point_reduction not in ("mean", "sum", "max"):
        raise ValueError('point_reduction must be one of ["mean", "sum", "max"] or None')
    if point_reduction is None and batch_reduction is not None:
        raise ValueError("batch_reduction must be None if point_reduction is None")
    if x.dtype != torch.float32 or y.dtype != torch.float32:
        raise RuntimeError("chamfer_distance: float32 inputs required")
    if weights is None and batch_reduction == "mean" and point_reduction == "mean" and not single_directional:
        return _ChamferFunction.apply(x, y), None
    if weights is not None:
        if weights.dim() != 1 or weights.shape[0] != x.shape[0]:
            raise ValueError("weights must be of shape (B,)")
        if not bool((weights >= 0).all()):
            raise ValueError("weights cannot be negative")
    cham_x = _chamfer_one_way(x, y, weights, batch_reduction, point_reduction)
    if single_directional:
        return cham_x, None
    cham_y = _chamfer_one_way(y, x, weights, batch_reduction, point_reduction)
    if point_reduction == "max":
        return torch.maximum(cham_x, cham_y), None
    if point_reduction is not None:
        return cham_x + cham_y, None
    return (cham_x, cham_y), (None, None)


def chamfer_loss(pc1, pc2):
    """models/utils.py:36-45. pc1, pc2: [B, 3, N]."""
    return chamfer_distance(pc1.permute(0, 2, 1), pc2.permute(0, 2, 1))[0]


_KNN = namedtuple("KNN", "dists idx knn")


class _KnnDists(Function):
    """knn_points' search (queries p1, refs p2, DIST_DIRECT_XYZ) with a backward for dists into
    both clouds: b200pci_knn_backward, or b200pci_knn_backward_det (fixed summation order) under
    torch.use_deterministic_algorithms. p1 / p2 may be strided views, and the same tensor."""

    @staticmethod
    def forward(ctx, p1, p2, K):
        idx, dists = _knn(K, p2, p1, DIST_DIRECT_XYZ, True)
        ctx.save_for_backward(p1, p2, idx)
        ctx.mark_non_differentiable(idx)
        return dists, idx

    @staticmethod
    def backward(ctx, grad_dists, _grad_idx):
        p1, p2, idx = ctx.saved_tensors
        B, S, _ = p1.shape
        N, K = p2.shape[1], idx.shape[2]
        g = grad_dists.contiguous()
        dev = p1.device
        with _lib.on_device(p1):
            gq = torch.empty((B, S, 3), dtype=torch.float32, device=dev)
            gr = torch.empty((B, N, 3), dtype=torch.float32, device=dev)
            qs, rs = p1.stride(), p2.stride()
            args = (B, S, N, K, p1.data_ptr(), qs[0], qs[1], qs[2], p2.data_ptr(), rs[0], rs[1], rs[2],
                    idx.data_ptr(), 1, g.data_ptr(), gq.data_ptr(), gr.data_ptr())
            if torch.are_deterministic_algorithms_enabled():  # fixed summation order (b200pci.h, _det)
                ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(B, N, S * K), dev)
                _lib.check(_L.b200pci_knn_backward_det(*args, ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
                           "knn_backward_det")
            else:
                _lib.check(_L.b200pci_knn_backward(*args, _lib.stream_ptr()), "knn_backward")
        return (gq if ctx.needs_input_grad[0] else None, gr if ctx.needs_input_grad[1] else None, None)


def knn_points(p1, p2, lengths1=None, lengths2=None, norm=2, K=1, version=-1, return_nn=False,
               return_sorted=True):
    """``pytorch3d.ops.knn_points`` (models/pointconv_util.py:910): for each point of p1 the K
    nearest points of p2 -> KNN(dists (B,P1,K) squared, idx int64 (B,P1,K), knn (B,P1,K,3) or None).

    dists is differentiable in p1 and p2 when grad is enabled and either requires grad (an
    autograd node only then: the model's forward is host-bound); knn = p2[idx] through the fused
    row gather, whose backward scatters into p2 without a P1 x P2 buffer."""
    if lengths1 is not None or lengths2 is not None or norm != 2:
        raise NotImplementedError("mocopci_b200.knn_points: lengths / norm != 2 not implemented")
    if _needs_grad(p1, p2):
        dists, idx = _KnnDists.apply(p1, p2, K)
    else:
        idx, dists = _knn(K, p2, p1, DIST_DIRECT_XYZ, True)
    nn = index_points_group(p2, idx) if return_nn else None
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
