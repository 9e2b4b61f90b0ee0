"""Regenerate tests/golden/kernel_snapshot.npz (read by tests/kernel_snapshot.py): kernel outputs on
the GPU parity tests' seeded inputs. Needs a CUDA device:

    python tests/golden/make_kernel_snapshot.py OUTDIR

The outputs come from the reference's own kernels (tests/refgpu.py) when oracle/_ref has been built
from a MoCoPCI checkout (make -C oracle ref), otherwise from this project's kernels. The file's
``source`` entry records which.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from mocopci_b200 import emd_cuda, ops, pointconv_util as pcu, pointnet2_cuda as p2c, synth  # noqa: E402
from tests import kernel_snapshot as snap, refgpu  # noqa: E402


def kernels():
    """(source name, module with refgpu's functions)."""
    if refgpu.available():
        return "reference kernels (oracle/_ref)", refgpu

    class Own:
        @staticmethod
        def fps(xyz, npoint):
            B, N, _ = xyz.shape
            idx = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
            temp = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
            p2c.furthest_point_sampling_wrapper(B, N, npoint, xyz, temp, idx)
            return idx, temp

        gather = staticmethod(ops.gather_operation)
        group = staticmethod(ops.grouping_operation)
        ball_query = staticmethod(ops.ball_query)

        @staticmethod
        def three_nn(unknown, known):
            B, n, _ = unknown.shape
            d2 = torch.empty((B, n, 3), device=unknown.device)
            idx = torch.empty((B, n, 3), dtype=torch.int32, device=unknown.device)
            p2c.three_nn_wrapper(B, n, known.shape[1], unknown, known, d2, idx)
            return d2, idx

        three_interpolate = staticmethod(ops.three_interpolate)
        emd_approxmatch = staticmethod(emd_cuda.approxmatch_forward)
        emd_matchcost = staticmethod(emd_cuda.matchcost_forward)
        emd_matchcost_grad = staticmethod(emd_cuda.matchcost_backward)
    return "this project's kernels", Own


def kernel_entries(st, ref):
    a, _ = synth.frame_pair(1, 4096)
    known, unknown = a[:1024][None].cuda().contiguous(), a[None].cuda().contiguous()
    d2, idx = ref.three_nn(unknown, known)
    snap.record(st, "three_nn/d2", d2)
    snap.record(st, "three_nn/idx", idx)

    for B, C, m, n in [(2, 128, 64, 256), (1, 5, 33, 1000), (2, 19, 1024, 4096), (1, 128, 4096, 16384),
                       (2, 64, 1000, 5000)]:
        g = torch.Generator().manual_seed(C)
        feat = torch.randn(B, C, m, generator=g)
        idx = torch.randint(0, m, (B, n, 3), generator=g, dtype=torch.int32)
        w = torch.rand(B, n, 3, generator=g)
        w = w / w.sum(-1, keepdim=True)
        snap.record(st, f"three_interpolate/{B}-{C}-{m}-{n}",
                    ref.three_interpolate(feat.cuda(), idx.cuda(), w.cuda()))

    for B, C, N, M in [(2, 3, 1000, 256), (1, 64, 4096, 1023), (3, 17, 50, 7)]:
        g = torch.Generator().manual_seed(N)
        feat = torch.randn(B, C, N, generator=g)
        idx = torch.randint(0, N, (B, M), generator=g, dtype=torch.int32)
        snap.record(st, f"gather/{B}-{C}-{N}-{M}", ref.gather(feat.cuda(), idx.cuda()))

    for B, C, N, np_, ns in [(2, 3, 1000, 128, 32), (1, 35, 2048, 300, 16), (2, 7, 64, 33, 3),
                             (1, 128, 4096, 1024, 32)]:
        g = torch.Generator().manual_seed(np_)
        feat = torch.randn(B, C, N, generator=g)
        idx = torch.randint(0, N, (B, np_, ns), generator=g, dtype=torch.int32)
        snap.record(st, f"group/{B}-{C}-{N}-{np_}-{ns}", ref.group(feat.cuda(), idx.cuda()))

    for N, M in ((1200, 200), (512, 128), (3000, 256)):
        xyz = synth.tie_stress_cloud(N, 2, N, grid=3).cuda()
        snap.record(st, f"fps_ties/{N}-{M}", ref.fps(xyz, M)[0])

    a, _ = synth.frame_pairs(0, 2)
    ridx, rtemp = ref.fps(a.cuda(), 4096)
    snap.record(st, "fps_full/idx", ridx)
    snap.record(st, "fps_full/temp", rtemp)

    for r, ns, shift in [(3.0, 128, 0.0), (1.5, 128, 0.0), (0.4, 96, 500.0), (6.0, 200, 0.0)]:
        a, _ = synth.frame_pairs(6, 1, 16384)
        a = (a + shift).contiguous()
        new = a[:, ::40].contiguous()
        snap.record(st, f"ball_query_split/{r}-{ns}-{shift}", ref.ball_query(r, ns, a.cuda(), new.cuda()))

    a, _ = synth.frame_pairs(2, 2, 8192)
    a = a.cuda()
    centres = pcu.index_points_gather(a, ops.furthest_point_sample(a, 1024))
    snap.record(st, "ball_query_lidar", ref.ball_query(0.5, 32, a, centres))

    a, _ = synth.frame_pairs(4, 1, 4096)
    a = a.cuda()
    feats = torch.randn(1, 16, 4096, generator=torch.Generator().manual_seed(4)).cuda()
    centres = pcu.index_points_gather(a, ops.furthest_point_sample(a, 256))
    idx = ref.ball_query(2.0, 16, a, centres)
    gx = ref.group(a.transpose(1, 2).contiguous(), idx) - centres.transpose(1, 2).unsqueeze(-1)
    snap.record(st, "query_and_group", torch.cat([gx, ref.group(feats, idx)], 1))

    for B, n, m in [(2, 256, 256), (1, 1000, 500), (2, 300, 1200), (1, 2048, 2048)]:
        x1 = (synth.uniform_cloud(n, B, n) * 0.5).cuda()
        x2 = (synth.uniform_cloud(m + 3, B, m) * 0.5).cuda()
        match = ref.emd_approxmatch(x1, x2)
        gc = (torch.rand(B, generator=torch.Generator().manual_seed(n + m)) + 0.5).cuda()
        g1, g2 = ref.emd_matchcost_grad(gc, x1, x2, match)
        key = f"emd/{B}-{n}-{m}"
        snap.record(st, key + "/match", match)
        snap.record(st, key + "/cost", ref.emd_matchcost(x1, x2, match), full=True)
        snap.record(st, key + "/grad1", g1)
        snap.record(st, key + "/grad2", g2, full=True)

    for B, n, m in [(2, 256, 256), (1, 1000, 500), (2, 300, 1200), (1, 4096, 4096)]:
        x1 = (synth.uniform_cloud(n + 1, B, n) * 0.5).cuda()
        x2 = (synth.uniform_cloud(m + 4, B, m) * 0.5).cuda()
        snap.record(st, f"emd_cost/{B}-{n}-{m}",
                    ref.emd_matchcost(x1, x2, ref.emd_approxmatch(x1, x2)), full=True)

    a, b = synth.frame_pair(0, 4096)
    x1, x2 = a.cuda()[None].contiguous(), b.cuda()[None].contiguous()
    snap.record(st, "emd_metric", (ref.emd_matchcost(x1, x2, ref.emd_approxmatch(x1, x2)).mean() / 4096)[None],
                full=True)


def main(out):
    os.makedirs(out, exist_ok=True)
    src, ref = kernels()
    st = {}
    kernel_entries(st, ref)
    torch.cuda.synchronize()
    st["source"] = np.asarray(src)
    path = os.path.join(out, "kernel_snapshot.npz")
    np.savez_compressed(path, **st)
    print(path, os.path.getsize(path), "bytes, from", src)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__)))
