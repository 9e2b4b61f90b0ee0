"""Functional API of the PointNet++ / EMD operators on the B200 kernels.

The reference exposes these operators through ``pointnet2/pointnet2_utils.py`` and
``models/EMD/emd.py`` (autograd classes around the pybind modules); those two files run UNCHANGED
on :mod:`mocopci_b200.pointnet2_cuda` / :mod:`mocopci_b200.emd_cuda` after
``mocopci_b200.install()``, and that is the drop-in path the parity tests drive. This module is the
package's own entry for code that does not carry a MoCoPCI checkout: the same operator names and
argument meaning (so call sites read the same), a single table-driven autograd node instead of one
class per operator, outputs allocated on the input's device, no contiguity asserts (inputs are
made contiguous), plus the fused variants the reference does not have (``three_nn_weights``,
``emd_cost``).
"""
import torch

from . import _lib, emd_cuda, pointnet2_cuda as _k

_L = _lib.lib


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# kind -> (forward launcher, backward launcher, output shape, size arguments of both launchers)
def _gather_sizes(feat_shape, idx):
    B, C, N = feat_shape
    return (B, C, N, idx.size(1))


def _group_sizes(feat_shape, idx):
    B, C, N = feat_shape
    return (B, C, N, idx.size(1), idx.size(2))


_SPECS = {
    # sampling_gpu.cu:8-83
    "gather": (_k.gather_points_wrapper, _k.gather_points_grad_wrapper, _gather_sizes,
               lambda sz: (sz[0], sz[1], sz[3])),
    # group_points_gpu.cu:8-86
    "group": (_k.group_points_wrapper, _k.group_points_grad_wrapper, _group_sizes,
              lambda sz: (sz[0], sz[1], sz[3], sz[4])),
}


class _IndexedCopy(torch.autograd.Function):
    """out = features[..., idx] for the [B, C, N] layout; the gradient is the matching scatter-add
    (atomics, like the reference's kernels; in a fixed order under torch's deterministic flag)."""

    @staticmethod
    def forward(ctx, kind, features, idx):
        fwd, _bwd, sizes, out_shape = _SPECS[kind]
        features, idx = _c(features), _c(idx)
        sz = sizes(features.shape, idx)
        out = features.new_empty(out_shape(sz))
        fwd(*sz, features, idx, out)
        ctx.kind, ctx.sz = kind, sz
        ctx.save_for_backward(idx)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (idx,) = ctx.saved_tensors
        B, C, N = ctx.sz[:3]
        grad = grad_out.new_zeros((B, C, N))
        _SPECS[ctx.kind][1](*ctx.sz, _c(grad_out), idx, grad)
        return None, grad, None


class _Interpolate(torch.autograd.Function):
    """interpolate_gpu.cu:77-161: out[b,c,i] = sum_j weight[b,i,j] * features[b,c,idx[b,i,j]]."""

    @staticmethod
    def forward(ctx, features, idx, weight):
        features, idx, weight = _c(features), _c(idx), _c(weight)
        B, C, m = features.shape
        n = idx.size(1)
        out = features.new_empty((B, C, n))
        _k.three_interpolate_wrapper(B, C, m, n, features, idx, weight, out)
        ctx.m = m
        ctx.save_for_backward(idx, weight)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        idx, weight = ctx.saved_tensors
        B, C, n = grad_out.shape
        grad = grad_out.new_zeros((B, C, ctx.m))
        _k.three_interpolate_grad_wrapper(B, C, n, ctx.m, _c(grad_out), idx, weight, grad)
        return grad, None, None


def furthest_point_sample(xyz, npoint):
    """pointnet2_utils.py:10-36. xyz (B, N, 3) -> int32 (B, npoint); idx[:, 0] == 0, ties broken
    exactly like the reference kernel's shared-memory tree (sampling_gpu.cu:86-209)."""
    xyz = _c(xyz)
    B, N, _ = xyz.shape
    idx = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
    scratch = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
    _k.furthest_point_sampling_wrapper(B, N, npoint, xyz, scratch, idx)
    return idx


def gather_operation(features, idx):
    """pointnet2_utils.py:39-73. features (B, C, N), idx int32 (B, M) -> (B, C, M)."""
    return _IndexedCopy.apply("gather", features, idx)


def grouping_operation(features, idx):
    """pointnet2_utils.py:156-197. features (B, C, N), idx int32 (B, P, S) -> (B, C, P, S)."""
    return _IndexedCopy.apply("group", features, idx)


def three_nn(unknown, known):
    """pointnet2_utils.py:76-105. -> (distance (B, n, 3) = sqrt of the squared distance the kernel
    returns, idx int32 (B, n, 3)), ascending, lowest index first among equals."""
    unknown, known = _c(unknown), _c(known)
    B, n, _ = unknown.shape
    d2 = torch.empty((B, n, 3), dtype=torch.float32, device=unknown.device)
    idx = torch.empty((B, n, 3), dtype=torch.int32, device=unknown.device)
    _k.three_nn_wrapper(B, n, known.size(1), unknown, known, d2, idx)
    return torch.sqrt(d2), idx


def three_nn_weights(unknown, known, eps=1e-8):
    """three_nn plus the caller-side inverse-distance weights of pointnet2_modules.py:139-144
    (``1/(d+eps)`` normalised over the three neighbours) in one kernel epilogue.
    -> (weight (B, n, 3), idx int32 (B, n, 3), distance (B, n, 3))."""
    unknown, known = _c(unknown), _c(known)
    B, n, _ = unknown.shape
    m = known.size(1)
    dev = unknown.device
    dist = torch.empty((B, n, 3), dtype=torch.float32, device=dev)
    weight = torch.empty((B, n, 3), dtype=torch.float32, device=dev)
    idx = torch.empty((B, n, 3), dtype=torch.int32, device=dev)
    with _lib.on_device(unknown):
        ws = _lib.workspace(_L.b200pci_three_nn_workspace_bytes(B, n, m), dev)
        _lib.check(_L.b200pci_three_nn_weights(
            B, n, m, unknown.data_ptr(), known.data_ptr(), float(eps), dist.data_ptr(),
            weight.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
            "three_nn_weights")
    return weight, idx, dist


def three_interpolate(features, idx, weight):
    """pointnet2_utils.py:108-153. features (B, C, m), idx (B, n, 3), weight (B, n, 3) -> (B, C, n)."""
    return _Interpolate.apply(features, idx, weight)


def ball_query(radius, nsample, xyz, new_xyz):
    """pointnet2_utils.py:200-228. xyz (B, N, 3), new_xyz (B, M, 3) -> int32 (B, M, nsample): the
    first nsample refs (ascending index) within the radius, padded with the first hit; all zero
    when there is none."""
    xyz, new_xyz = _c(xyz), _c(new_xyz)
    B, N, _ = xyz.shape
    M = new_xyz.size(1)
    idx = torch.zeros((B, M, nsample), dtype=torch.int32, device=xyz.device)
    _k.ball_query_wrapper(B, N, M, radius, nsample, new_xyz, xyz, idx)
    return idx


def query_and_group(radius, nsample, xyz, new_xyz, features=None, use_xyz=True):
    """``QueryAndGroup(radius, nsample, use_xyz)(xyz, new_xyz, features)``,
    pointnet2_utils.py:231-264 -> (B, 3 + C, M, nsample) (or (B, C, ...) / (B, 3, ...))."""
    idx = ball_query(radius, nsample, xyz, new_xyz)
    if features is None and not use_xyz:
        raise ValueError("query_and_group: nothing to group (features is None and use_xyz=False)")
    needs_grad = torch.is_grad_enabled() and (xyz.requires_grad or new_xyz.requires_grad
                                              or (features is not None and features.requires_grad))
    if not needs_grad and (features is None or features.dtype == torch.float32):
        # one pass into the concatenated tensor (b200pci_query_group): no transposed copy of the
        # cloud, no separate subtraction, no torch.cat
        _lib.require_cuda(xyz, new_xyz)
        B, N, _ = xyz.shape
        M = new_xyz.shape[1]
        C = 0 if features is None else features.shape[1]
        xyz_c, new_c = _c(xyz), _c(new_xyz)
        feat_c = _c(features) if features is not None else None
        out = torch.empty((B, (3 if use_xyz else 0) + C, M, nsample), dtype=torch.float32, device=xyz.device)
        with _lib.on_device(xyz):
            _lib.check(_L.b200pci_query_group(
                B, N, M, nsample, C, xyz_c.data_ptr(), new_c.data_ptr(),
                feat_c.data_ptr() if feat_c is not None else None, idx.data_ptr(), out.data_ptr(),
                1 if use_xyz else 0, _lib.stream_ptr()), "query_group")
        return out
    rel = grouping_operation(xyz.transpose(1, 2), idx) - new_xyz.transpose(1, 2).unsqueeze(-1)
    if features is None:
        return rel
    grouped = grouping_operation(features, idx)
    return torch.cat([rel, grouped], dim=1) if use_xyz else grouped


class _EmdCost(torch.autograd.Function):
    """models/EMD/emd.py:5-22: cost = matchcost(approxmatch(xyz1, xyz2)); the forward-only case
    (no input requires grad) uses the fused ``emd_cost`` and never stores the match matrix."""

    @staticmethod
    def forward(ctx, xyz1, xyz2):
        xyz1, xyz2 = _c(xyz1), _c(xyz2)
        if not (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
            return emd_cuda.emd_cost(xyz1, xyz2)
        match = emd_cuda.approxmatch_forward(xyz1, xyz2)
        ctx.save_for_backward(xyz1, xyz2, match)
        return emd_cuda.matchcost_forward(xyz1, xyz2, match)

    @staticmethod
    def backward(ctx, grad_cost):
        xyz1, xyz2, match = ctx.saved_tensors
        g1, g2 = emd_cuda.matchcost_backward(_c(grad_cost), xyz1, xyz2, match)
        return g1, g2


def earth_mover_distance(xyz1, xyz2, transpose=True):
    """models/EMD/emd.py:25-46. (B, 3, n) inputs when ``transpose`` else (B, n, 3) -> cost (B)."""
    xyz1 = xyz1[None] if xyz1.dim() == 2 else xyz1
    xyz2 = xyz2[None] if xyz2.dim() == 2 else xyz2
    if transpose:
        xyz1, xyz2 = xyz1.transpose(1, 2), xyz2.transpose(1, 2)
    return _EmdCost.apply(xyz1, xyz2)


def emd_metric(pc1, pc2):
    """The eval metric ``EMD`` of models/utils.py:223-235: pc1, pc2 (B, 3, M) -> mean(cost) / M."""
    return earth_mover_distance(pc1, pc2, transpose=True).mean() / pc1.shape[2]
