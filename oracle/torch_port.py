"""TEST INFRASTRUCTURE ONLY -- torch restatement of the reference's pure-torch CPU KNN/Chamfer path
and of the distance helpers the GPU parity tests run on CUDA tensors.

This is what ``bench.py --impl reference`` and the ``cpu_baseline`` leg time on the GPU box's
host cores (the reference's Python cannot travel there): the same torch ops, in the same order,
as models/pointconv_util.py:67-88 (square_distance) and :129-140 (knn_point), plus Chamfer via
square_distance + min (the semantics of pytorch3d.loss.chamfer_distance used at
models/utils.py:44; pytorch3d itself is not installed).
"""
import torch


def square_distance(src, dst):
    # models/pointconv_util.py:83-88
    B, N, _ = src.shape
    _, M, _ = dst.shape
    dist = -2 * torch.matmul(src, dst.permute(0, 2, 1))
    dist += torch.sum(src ** 2, -1).view(B, N, 1)
    dist += torch.sum(dst ** 2, -1).view(B, 1, M)
    return dist


def knn_point(nsample, xyz, new_xyz):
    # models/pointconv_util.py:138-140
    sqrdists = square_distance(new_xyz, xyz)
    _, group_idx = torch.topk(sqrdists, nsample, dim=-1, largest=False, sorted=False)
    return group_idx


def chamfer(pc1, pc2):
    # models/utils.py:36-45 with pytorch3d defaults: [B,3,N] inputs
    x = pc1.permute(0, 2, 1)
    y = pc2.permute(0, 2, 1)
    d = square_distance(x, y)
    return (d.min(dim=2)[0].mean(dim=1) + d.min(dim=1)[0].mean(dim=1)).mean()


def square_distance_sqdiff(src, dst):
    # models/pointT_layer2.py:20: sum of squared coordinate differences; CUDA torch adds
    # (dx^2 + dz^2) + dy^2, CPU torch (dx^2 + dy^2) + dz^2
    return torch.sum((src[:, :, None] - dst[:, None]) ** 2, dim=-1)


def cosine_distance(src, dst):
    # models/pointconv_util.py:111-127: 1 - <q/|q|, r/|r|> for q in src [B,S,C], r in dst [B,N,C].
    # Restated from the definition, not op for op: compare with a tolerance
    src = src / torch.norm(src, dim=-1, keepdim=True)
    dst = dst / torch.norm(dst, dim=-1, keepdim=True)
    return 1 - torch.matmul(src, dst.permute(0, 2, 1))
