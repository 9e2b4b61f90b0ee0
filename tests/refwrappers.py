"""TEST INFRASTRUCTURE ONLY: an ABI-shaped restatement of the reference's autograd wrappers around
``pointnet2_cuda`` and ``emd_cuda`` (pointnet2/pointnet2_utils.py, models/EMD/emd.py, the ``EMD``
metric of models/utils.py), for the ``reference_wrappers`` variant of the GPU parity tests when no
MoCoPCI checkout is available to import the reference's own files from. It is not those files:
it calls the two modules the way they do (positional sizes, caller-allocated outputs, contiguous
inputs, zero-filled gradient buffers), so that variant exercises the pybind-compatible surface
rather than the package's own ops. Import only after ``mocopci_b200.install()`` has registered
the modules.
"""
import torch
from torch import nn
from torch.autograd import Function

import emd_cuda
import pointnet2_cuda as pointnet2


def _empty(shape, dtype, like):
    return torch.empty(shape, dtype=dtype, device=like.device)


class FurthestPointSampling(Function):
    @staticmethod
    def forward(ctx, xyz, npoint):
        assert xyz.is_contiguous()
        B, N, _ = xyz.size()
        output = _empty((B, npoint), torch.int32, xyz)
        temp = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
        pointnet2.furthest_point_sampling_wrapper(B, N, npoint, xyz, temp, output)
        return output

    @staticmethod
    def backward(ctx, a=None):
        return None, None


furthest_point_sample = FurthestPointSampling.apply


class GatherOperation(Function):
    @staticmethod
    def forward(ctx, features, idx):
        assert features.is_contiguous() and idx.is_contiguous()
        B, npoint = idx.size()
        _, C, N = features.size()
        output = _empty((B, C, npoint), torch.float32, features)
        pointnet2.gather_points_wrapper(B, C, N, npoint, features, idx, output)
        ctx.for_backwards = (idx, C, N)
        return output

    @staticmethod
    def backward(ctx, grad_out):
        idx, C, N = ctx.for_backwards
        B, npoint = idx.size()
        grad_features = torch.zeros((B, C, N), dtype=torch.float32, device=grad_out.device)
        pointnet2.gather_points_grad_wrapper(B, C, N, npoint, grad_out.contiguous(), idx, grad_features)
        return grad_features, None


gather_operation = GatherOperation.apply


class ThreeNN(Function):
    @staticmethod
    def forward(ctx, unknown, known):
        assert unknown.is_contiguous() and known.is_contiguous()
        B, N, _ = unknown.size()
        m = known.size(1)
        dist2 = _empty((B, N, 3), torch.float32, unknown)
        idx = _empty((B, N, 3), torch.int32, unknown)
        pointnet2.three_nn_wrapper(B, N, m, unknown, known, dist2, idx)
        return torch.sqrt(dist2), idx

    @staticmethod
    def backward(ctx, a=None, b=None):
        return None, None


three_nn = ThreeNN.apply


class ThreeInterpolate(Function):
    @staticmethod
    def forward(ctx, features, idx, weight):
        assert features.is_contiguous() and idx.is_contiguous() and weight.is_contiguous()
        B, c, m = features.size()
        n = idx.size(1)
        ctx.three_interpolate_for_backward = (idx, weight, m)
        output = _empty((B, c, n), torch.float32, features)
        pointnet2.three_interpolate_wrapper(B, c, m, n, features, idx, weight, output)
        return output

    @staticmethod
    def backward(ctx, grad_out):
        idx, weight, m = ctx.three_interpolate_for_backward
        B, c, n = grad_out.size()
        grad_features = torch.zeros((B, c, m), dtype=torch.float32, device=grad_out.device)
        pointnet2.three_interpolate_grad_wrapper(B, c, n, m, grad_out.contiguous(), idx, weight, grad_features)
        return grad_features, None, None


three_interpolate = ThreeInterpolate.apply


class GroupingOperation(Function):
    @staticmethod
    def forward(ctx, features, idx):
        assert features.is_contiguous() and idx.is_contiguous()
        B, nfeatures, nsample = idx.size()
        _, C, N = features.size()
        output = _empty((B, C, nfeatures, nsample), torch.float32, features)
        pointnet2.group_points_wrapper(B, C, N, nfeatures, nsample, features, idx, output)
        ctx.for_backwards = (idx, N)
        return output

    @staticmethod
    def backward(ctx, grad_out):
        idx, N = ctx.for_backwards
        B, C, npoint, nsample = grad_out.size()
        grad_features = torch.zeros((B, C, N), dtype=torch.float32, device=grad_out.device)
        pointnet2.group_points_grad_wrapper(B, C, N, npoint, nsample, grad_out.contiguous(), idx, grad_features)
        return grad_features, None


grouping_operation = GroupingOperation.apply


class BallQuery(Function):
    @staticmethod
    def forward(ctx, radius, nsample, xyz, new_xyz):
        assert new_xyz.is_contiguous() and xyz.is_contiguous()
        B, N, _ = xyz.size()
        npoint = new_xyz.size(1)
        idx = torch.zeros((B, npoint, nsample), dtype=torch.int32, device=xyz.device)
        pointnet2.ball_query_wrapper(B, N, npoint, radius, nsample, new_xyz, xyz, idx)
        return idx

    @staticmethod
    def backward(ctx, a=None):
        return None, None, None, None


ball_query = BallQuery.apply


class QueryAndGroup(nn.Module):
    def __init__(self, radius, nsample, use_xyz=True):
        super().__init__()
        self.radius, self.nsample, self.use_xyz = radius, nsample, use_xyz

    def forward(self, xyz, new_xyz, features=None):
        idx = ball_query(self.radius, self.nsample, xyz, new_xyz)
        xyz_trans = xyz.transpose(1, 2).contiguous()
        grouped_xyz = grouping_operation(xyz_trans, idx)
        grouped_xyz -= new_xyz.transpose(1, 2).unsqueeze(-1)
        if features is None:
            assert self.use_xyz, "Cannot have not features and not use xyz as a feature!"
            return grouped_xyz
        grouped_features = grouping_operation(features, idx)
        if self.use_xyz:
            return torch.cat([grouped_xyz, grouped_features], dim=1)
        return grouped_features


class EarthMoverDistanceFunction(Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2):
        xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()
        assert xyz1.is_cuda and xyz2.is_cuda, "Only support cuda currently."
        match = emd_cuda.approxmatch_forward(xyz1, xyz2)
        cost = emd_cuda.matchcost_forward(xyz1, xyz2, match)
        ctx.save_for_backward(xyz1, xyz2, match)
        return cost

    @staticmethod
    def backward(ctx, grad_cost):
        xyz1, xyz2, match = ctx.saved_tensors
        grad_xyz1, grad_xyz2 = emd_cuda.matchcost_backward(grad_cost.contiguous(), xyz1, xyz2, match)
        return grad_xyz1, grad_xyz2


def earth_mover_distance(xyz1, xyz2, transpose=True):
    if xyz1.dim() == 2:
        xyz1 = xyz1.unsqueeze(0)
    if xyz2.dim() == 2:
        xyz2 = xyz2.unsqueeze(0)
    if transpose:
        xyz1, xyz2 = xyz1.transpose(1, 2), xyz2.transpose(1, 2)
    return EarthMoverDistanceFunction.apply(xyz1, xyz2)


def EMD(pc1, pc2):
    """pc1, pc2 (B, 3, M) -> mean cost per point."""
    pc1, pc2 = pc1.permute(0, 2, 1).contiguous(), pc2.permute(0, 2, 1).contiguous()
    return earth_mover_distance(pc1, pc2, transpose=False).mean() / pc1.shape[1]
