"""TEST INFRASTRUCTURE ONLY: float64 restatements of the approximate Earth-Mover distance
(models/EMD/cuda/emd_kernel.cu) in plain torch, on CPU or CUDA tensors.

* ``approxmatch64`` follows ApproxMatch (emd_kernel.cu:29-162) line by line: the integer-division
  multipliers, ten temperature levels, three sweeps per level, the ``1e-9`` guards and the
  ``fminf`` / ``fmaxf`` clamps. Only the arithmetic differs: float64 and an exact ``exp``.
* ``cost64`` is ``matchcost64(approxmatch64(...))`` without storing ``match``: the cost is linear in
  ``match``, so each level's increment is weighted with the squared distance and summed as it is
  made. It works on blocks of ``xyz2`` rows, which makes 16384 x 16384 feasible.
* ``matchcost64`` and ``matchcost_grad64`` are the closed forms of MatchCost and its gradient on a
  given ``match`` (emd_kernel.cu:204-247, 290-359).

Inputs are (B, n, 3) / (B, m, 3) clouds of any float dtype; ``match`` is (B, m, n). Results are
float64 on the inputs' device. No tolerances here: the tests that use this module own them.
"""
import torch


def multipliers(n, m):
    """emd_kernel.cu:33-38: the larger cloud's points carry mass 1, the smaller one's the integer
    quotient (so n = 300, m = 1000 gives 3, not 10/3)."""
    return (1.0, float(n // m)) if n >= m else (float(m // n), 1.0)


def levels():
    """emd_kernel.cu:51-54: -4^7, -4^6, ..., -4^-1, then 0."""
    return [-(4.0 ** j) for j in range(7, -2, -1)] + [0.0]


def _sqdist(p2, p1):
    """(rows of p2, points of p1) squared distances, float64."""
    return ((p2[:, None, :] - p1[None, :, :]) ** 2).sum(-1)


def _blocks(m, block):
    return [(l0, min(m, l0 + block)) for l0 in range(0, m, block)]


def _approxmatch_pair(p1, p2, block, match=None):
    """One pair. Fills ``match`` (m, n) when given; returns the cost sum over k, l of d * match."""
    n, m = p1.shape[0], p2.shape[0]
    multiL, multiR = multipliers(n, m)
    remainL = torch.full((n,), multiL, dtype=torch.float64, device=p1.device)
    remainR = torch.full((m,), multiR, dtype=torch.float64, device=p1.device)
    ratioR = torch.empty_like(remainR)
    cost = torch.zeros((), dtype=torch.float64, device=p1.device)
    for level in levels():
        # sweep 1 (:54-87): ratioL[k] = remainL[k] / (1e-9 + sum_l exp(level d) remainR[l])
        suml = torch.full((n,), 1e-9, dtype=torch.float64, device=p1.device)
        for l0, l1 in _blocks(m, block):
            suml += (torch.exp(level * _sqdist(p2[l0:l1], p1)) * remainR[l0:l1, None]).sum(0)
        ratioL = remainL / suml
        # sweep 2 (:89-123), per xyz2 point l
        for l0, l1 in _blocks(m, block):
            rr = remainR[l0:l1]
            sumr = (torch.exp(level * _sqdist(p2[l0:l1], p1)) * ratioL[None, :]).sum(1) * rr
            consumption = torch.clamp(rr / (sumr + 1e-9), max=1.0)
            ratioR[l0:l1] = consumption * rr
            remainR[l0:l1] = torch.clamp(rr - sumr, min=0.0)
        # sweep 3 (:125-158): match[l][k] += w, remainL[k] -= sum_l w
        used = torch.zeros((n,), dtype=torch.float64, device=p1.device)
        for l0, l1 in _blocks(m, block):
            d = _sqdist(p2[l0:l1], p1)
            w = torch.exp(level * d) * ratioL[None, :] * ratioR[l0:l1, None]
            if match is not None:
                match[l0:l1] += w
            cost += (w * d).sum()
            used += w.sum(0)
        remainL = torch.clamp(remainL - used, min=0.0)
    return cost


def _pairs(xyz1, xyz2):
    p1, p2 = xyz1.detach().double(), xyz2.detach().double()
    assert p1.dim() == 3 and p2.dim() == 3 and p1.shape[0] == p2.shape[0]
    return p1, p2


def approxmatch64(xyz1, xyz2, block=4096):
    """match (B, m, n), float64."""
    p1, p2 = _pairs(xyz1, xyz2)
    B, n, m = p1.shape[0], p1.shape[1], p2.shape[1]
    match = torch.zeros((B, m, n), dtype=torch.float64, device=p1.device)
    if n and m:
        for b in range(B):
            _approxmatch_pair(p1[b], p2[b], block, match[b])
    return match


def cost64(xyz1, xyz2, block=1024):
    """matchcost64(xyz1, xyz2, approxmatch64(xyz1, xyz2)) -> (B,), without a (m, n) matrix."""
    p1, p2 = _pairs(xyz1, xyz2)
    B, n, m = p1.shape[0], p1.shape[1], p2.shape[1]
    out = torch.zeros((B,), dtype=torch.float64, device=p1.device)
    if n and m:
        for b in range(B):
            out[b] = _approxmatch_pair(p1[b], p2[b], block)
    return out


def matchcost64(xyz1, xyz2, match, block=1024):
    """sum over k, l of |xyz2[l] - xyz1[k]|^2 match[l, k] -> (B,)."""
    p1, p2 = _pairs(xyz1, xyz2)
    out = torch.zeros((p1.shape[0],), dtype=torch.float64, device=p1.device)
    for b in range(p1.shape[0]):
        for l0, l1 in _blocks(p2.shape[1], block):
            out[b] += (_sqdist(p2[b, l0:l1], p1[b]) * match[b, l0:l1].double()).sum()
    return out


def matchcost_grad64(grad_cost, xyz1, xyz2, match):
    """Gradients of grad_cost[b] * matchcost with ``match`` held fixed:
    grad1[k] = g sum_l 2 match[l, k] (xyz1[k] - xyz2[l]),
    grad2[l] = g sum_k 2 match[l, k] (xyz2[l] - xyz1[k])."""
    p1, p2 = _pairs(xyz1, xyz2)
    mt = match.double()
    g = grad_cost.double().reshape(-1, 1, 1)
    grad1 = 2 * g * (mt.sum(1)[..., None] * p1 - mt.transpose(1, 2) @ p2)
    grad2 = 2 * g * (mt.sum(2)[..., None] * p2 - mt @ p1)
    return grad1, grad2
