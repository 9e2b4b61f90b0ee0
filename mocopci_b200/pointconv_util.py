"""Host-side mirror of the hot-path helpers of the reference's ``models/pointconv_util.py``
(second live copy in ``models/m_models/mocopci.py:1130-1266``): same names, argument order and
return types, bound to the fused B200 kernels.

``knn_point`` never materialises the [B,S,N] distance matrix the reference builds
(pointconv_util.py:85-87, 1 GiB per cloud at 16384 points): distances are evaluated with the
reference's exact FP32 rounding sequence inside the selection kernel and only the k indices
leave the chip.
"""
import os

import torch

from . import _lib

_L = _lib.lib

DIST_EXPANDED = 0    # torch square_distance (pointconv_util.py:67-88)
DIST_DIRECT = 1      # pointnet2 kernels: fma(dz,dz,fma(dx,dx,dy*dy))
DIST_DIRECT_XYZ = 2  # pytorch3d CUDA knn: fma(dz,dz,fma(dy,dy,dx*dx))
DIST_SQDIFF = 3      # torch.sum((a - b) ** 2, -1) (pointT_layer2.py:20): no fused multiply-add
# torch.sum over the 3 coordinates adds (a+b)+c on the CPU and (a+c)+b on CUDA (tools/gpu_probe.py):
# the two torch-defined forms exist in both orders. "cuda" is what the reference computes for the
# CUDA tensors these functions take (bit-identical neighbour distances for a model moved over from
# the reference's GPU path); "cpu" is BASELINE's CPU torch path and the committed golden vectors.
DIST_SQDIFF_CUDA = 4
DIST_EXPANDED_CUDA = 5
_EXPANDED = {"cuda": DIST_EXPANDED_CUDA, "cpu": DIST_EXPANDED}
_SQDIFF = {"cuda": DIST_SQDIFF_CUDA, "cpu": DIST_SQDIFF}


def _knn(k, xyz, new_xyz, mode, want_dist, int64=True):
    """xyz: refs [B,N,3] (any strides), new_xyz: queries [B,S,3] (any strides)."""
    _lib.require_cuda(xyz, new_xyz)
    if xyz.dtype != torch.float32 or new_xyz.dtype != torch.float32:
        raise RuntimeError("knn: float32 inputs required")
    if xyz.dim() != 3 or new_xyz.dim() != 3 or xyz.size(2) != 3 or new_xyz.size(2) != 3:
        raise RuntimeError("knn: inputs must be [B, N, 3] / [B, S, 3]")
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    if new_xyz.shape[0] != B:
        raise RuntimeError("knn: batch sizes differ")
    dev = xyz.device
    with _lib.on_device(xyz):
        idx = torch.empty((B, S, k), dtype=torch.int64 if int64 else torch.int32, device=dev)
        dist = torch.empty((B, S, k), dtype=torch.float32, device=dev) if want_dist else None
        ws = _lib.workspace(_L.b200pci_knn_workspace_bytes(B, S, N, k), dev)
        qs, rs = new_xyz.stride(), xyz.stride()
        _lib.check(_L.b200pci_knn(
            B, S, N, k, mode,
            new_xyz.data_ptr(), qs[0], qs[1], qs[2],
            xyz.data_ptr(), rs[0], rs[1], rs[2],
            idx.data_ptr(), 1 if int64 else 0, dist.data_ptr() if want_dist else None,
            ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "knn")
    return idx, dist


def knn_point(nsample, xyz, new_xyz, arith="cuda"):
    """pointconv_util.py:129-140 (copy mocopci.py:1158-1169).

    xyz: all points [B, N, C=3]; new_xyz: query points [B, S, 3] -> int64 [B, S, nsample].
    The reference returns ``torch.topk(..., sorted=False)`` order (unspecified); here the
    neighbours come out sorted by (distance, index), the lowest index winning ties.
    ``arith``: "cuda" (default) = the rounding sequence of the reference's square_distance as CUDA
    torch executes it, "cpu" = as CPU torch executes it (see DIST_EXPANDED_CUDA above).
    """
    return _knn(nsample, xyz, new_xyz, _EXPANDED[arith], False)[0]


def knn_point_sqdiff(nsample, xyz, new_xyz, arith="cuda"):
    """``square_distance(new_xyz, xyz).argsort()[:, :, :nsample]`` of models/pointT_layer2.py:20,62-63
    (the broadcast-difference distance, every product and sum rounded) without the N x N matrix and
    the full sort: int64 [B, S, nsample], ascending by (distance, index). ``argsort`` is not stable,
    so among EQUAL distances the reference's order is unspecified; here the lowest index is first."""
    return _knn(nsample, xyz, new_xyz, _SQDIFF[arith], False)[0]


def cosine_supported(nsample, xyz, new_xyz):
    """Whether the fused feature-space kernel covers this call (else the reference's torch path runs):
    float32 CUDA [B,N,C] / [B,S,C], C a multiple of 16, nsample <= 32, nsample <= N <= 4096."""
    if xyz.dim() != 3 or new_xyz.dim() != 3 or xyz.size(0) != new_xyz.size(0) or xyz.size(2) != new_xyz.size(2):
        return False
    B, N, C = xyz.shape
    return _L.b200pci_knn_cosine_workspace_bytes(B, new_xyz.size(1), N, C, nsample) > 0


def _knn_cosine(nsample, xyz, new_xyz, want_dist):
    _lib.require_cuda(xyz, new_xyz)
    if xyz.dtype != torch.float32 or new_xyz.dtype != torch.float32:
        raise RuntimeError("knn_point_cosine: float32 inputs required")
    B, N, C = xyz.shape
    S = new_xyz.shape[1]
    dev = xyz.device
    with _lib.on_device(xyz):
        nbytes = _L.b200pci_knn_cosine_workspace_bytes(B, S, N, C, nsample)
        if nbytes == 0:
            raise RuntimeError("knn_point_cosine: shape not covered by the fused kernel "
                               "(C % 16 == 0, nsample <= 32, nsample <= N <= 4096)")
        idx = torch.empty((B, S, nsample), dtype=torch.int64, device=dev)
        dist = torch.empty((B, S, nsample), dtype=torch.float32, device=dev) if want_dist else None
        ws = _lib.workspace(nbytes, dev)
        qs, rs = new_xyz.stride(), xyz.stride()
        _lib.check(_L.b200pci_knn_cosine(
            B, S, N, C, nsample, new_xyz.data_ptr(), qs[0], qs[1], qs[2], xyz.data_ptr(), rs[0], rs[1], rs[2],
            idx.data_ptr(), 1, dist.data_ptr() if want_dist else None, ws.data_ptr(), ws.numel(),
            _lib.stream_ptr()), "knn_cosine")
    return idx, dist


def knn_point_cosine(nsample, xyz, new_xyz):
    """pointconv_util.py:142-153: the nsample refs (xyz [B,N,C]) with the smallest cosine distance
    1 - <q/|q|, r/|r|> to each query (new_xyz [B,S,C]) -> int64 [B,S,nsample], sorted by
    (distance, index). One normalise+split pass and one tensor-core kernel instead of the reference's
    normalise / bmm / rsub / topk chain over a materialised [B,S,N] matrix."""
    return _knn_cosine(nsample, xyz, new_xyz, False)[0]


def knn_point_cosine_with_dist(nsample, xyz, new_xyz):
    return _knn_cosine(nsample, xyz, new_xyz, True)


def knn_point_with_dist(nsample, xyz, new_xyz, arith="cuda"):
    """knn_point plus the selected values of ``square_distance(new_xyz, xyz)`` (bit-identical
    to the reference's matrix entries, pointconv_util.py:85-87)."""
    return _knn(nsample, xyz, new_xyz, _EXPANDED[arith], True)


_TRANSPOSE_TABLES = os.environ.get("B200PCI_TRANSPOSE_TABLES", "1") != "0"  # developer switch


def _row_major(points, gathered_rows):
    """A gather of whole rows wants the row (all channels of a point) contiguous: from the
    channel-major [B,C,N] tensors the model keeps (passed as permuted views) every gathered float
    would be its own 32-byte sector. When many more rows are gathered than the table holds, the
    table is transposed once (a [B,N,C] copy of N*C floats) and the gather reads 16-byte pieces."""
    if (_TRANSPOSE_TABLES and points.stride(2) != 1 and points.size(2) > 1
            and gathered_rows >= 2 * points.size(1)):
        return points.contiguous()
    return points


def _index_rows(points, idx):
    """out[b,t,:] = points[b, idx[b,t], :] (b200pci_index_points_rows) -> (out, contiguous idx)."""
    _lib.require_cuda(points, idx)
    if points.dtype != torch.float32 or points.dim() != 3:
        raise RuntimeError("index_points: points must be float32 [B, N, C]")
    if idx.dtype not in (torch.int64, torch.int32) or idx.size(0) != points.size(0):
        raise RuntimeError("index_points: idx must be int64/int32 [B, ...]")
    B, N, C = points.shape
    idx_c = idx.contiguous()
    T = idx_c.numel() // B if B > 0 else 0
    out = torch.empty(tuple(idx.shape) + (C,), dtype=torch.float32, device=points.device)
    points = _row_major(points, T)
    ps = points.stride()
    with _lib.on_device(points):
        _lib.check(_L.b200pci_index_points_rows(
            B, N, T, C, points.data_ptr(), ps[0], ps[1], ps[2], idx_c.data_ptr(),
            1 if idx_c.dtype == torch.int64 else 0, out.data_ptr(), _lib.stream_ptr()),
            "index_points_rows")
    return out, idx_c


class _IndexRows(torch.autograd.Function):
    """out[b,t,:] = points[b, idx[b,t], :] (b200pci_index_points_rows); idx [B, ...] int64/int32."""

    @staticmethod
    def forward(ctx, points, idx):
        out, idx_c = _index_rows(points, idx)
        ctx.save_for_backward(idx_c)
        ctx.pshape = tuple(points.shape)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (idx_c,) = ctx.saved_tensors
        B, N, C = ctx.pshape
        g = grad_out.contiguous()
        grad_points = torch.zeros((B, N, C), dtype=torch.float32, device=g.device)
        T = idx_c[0].numel() if B > 0 else 0
        is64 = 1 if idx_c.dtype == torch.int64 else 0
        with _lib.on_device(g):
            if torch.are_deterministic_algorithms_enabled():  # fixed summation order (b200pci.h, _det)
                ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(B, N, T), g.device)
                _lib.check(_L.b200pci_index_points_rows_grad_det(
                    B, N, T, C, g.data_ptr(), idx_c.data_ptr(), is64, grad_points.data_ptr(),
                    ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "index_points_rows_grad_det")
            else:
                _lib.check(_L.b200pci_index_points_rows_grad(
                    B, N, T, C, g.data_ptr(), idx_c.data_ptr(), is64, grad_points.data_ptr(),
                    _lib.stream_ptr()), "index_points_rows_grad")
        return grad_points, None


def index_points_gather(points, fps_idx):
    """pointconv_util.py:168-179. points [B, N, C], idx [B, S] -> [B, S, C] contiguous.

    One fused kernel on the [B,N,C] layout (the reference transposes to [B,C,N], runs
    gather_operation and transposes back)."""
    if torch.is_grad_enabled() and points.requires_grad:
        return _IndexRows.apply(points, fps_idx)
    return _index_rows(points, fps_idx)[0]


def index_points_group(points, knn_idx):
    """pointconv_util.py:181-192. points [B, N, C], idx [B, S, K] -> [B, S, K, C].

    The reference returns a permuted view of a [B,C,S,K] tensor after a transpose copy and an
    int64 -> int32 cast of the indices; here one kernel reads the (possibly permuted) points view
    and the int64 indices directly and writes the contiguous [B,S,K,C] result every consumer in
    models/m_models/mocopci.py concatenates / reduces along the last axis."""
    if torch.is_grad_enabled() and points.requires_grad:
        return _IndexRows.apply(points, knn_idx)
    return _index_rows(points, knn_idx)[0]  # no autograd node on the inference path


def _needs_grad(*ts):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _group_concat(xyz, centre, points, idx):
    """[xyz[idx] - centre | points[idx]] and xyz[idx] - centre in one kernel (b200pci_group_concat)."""
    B, N, _ = xyz.shape
    S, K = idx.shape[1], idx.shape[2]
    D = 0 if points is None else points.shape[2]
    dev = xyz.device
    idx_c = idx.contiguous()
    if D:
        points = _row_major(points, S * K)
    norm = torch.empty((B, S, K, 3), dtype=torch.float32, device=dev)
    out = torch.empty((B, S, K, 3 + D), dtype=torch.float32, device=dev) if D else None
    xs, cs = xyz.stride(), centre.stride()
    ps = points.stride() if D else (0, 0, 0)
    with _lib.on_device(xyz):
        _lib.check(_L.b200pci_group_concat(
            B, N, S, K, D, xyz.data_ptr(), xs[0], xs[1], xs[2], centre.data_ptr(), cs[0], cs[1], cs[2],
            points.data_ptr() if D else None, ps[0], ps[1], ps[2], idx_c.data_ptr(),
            1 if idx_c.dtype == torch.int64 else 0, out.data_ptr() if D else None, norm.data_ptr(),
            _lib.stream_ptr()), "group_concat")
    return (out if D else norm), norm


def group_query(nsample, s_xyz, xyz, s_points):
    """pointconv_util.py:217-241: the nsample nearest support points (s_xyz [B,N,3], features s_points
    [B,N,D] or None) of every query (xyz [B,S,3]) -> (new_points [B,S,nsample,3+D], grouped_xyz_norm
    [B,S,nsample,3]). Neighbour search + ONE gather/subtract/concatenate kernel when no gradient is
    required; with autograd the same values through the differentiable row gathers."""
    idx = knn_point(nsample, s_xyz, xyz)
    if not _needs_grad(s_xyz, xyz, s_points) and (s_points is None or s_points.dtype == torch.float32):
        return _group_concat(s_xyz, xyz, s_points, idx)
    rel = index_points_group(s_xyz, idx) - xyz.unsqueeze(2)
    if s_points is None:
        return rel, rel
    return torch.cat([rel, index_points_group(s_points, idx)], dim=-1), rel


def group(nsample, xyz, points):
    """pointconv_util.py:194-215: ``group_query`` of a cloud with itself."""
    return group_query(nsample, xyz, xyz, points)
