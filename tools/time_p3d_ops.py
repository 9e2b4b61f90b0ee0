"""pytorch3d-form ball_query and sample_farthest_points (mocopci_b200.p3d_ops) against a torch
restatement and the pointnet2-form kernels, at bench.py's config-2 shape (8 frames of 16384 points,
4096 centres, r = 0.5, K = 32 and 500):
python tools/time_p3d_ops.py [--reps 20] [--out profiles/r5_p3d_ops_times.json]

The torch restatement of ball_query works on chunks of queries: d2 = ((p1 - p2) ** 2).sum(-1),
mask d2 < r^2, sort the masked ref indices and keep the first K ("cdist + mask + sort"; torch's
sum order, so its last bits may differ from the kernels'). The torch FPS is the sequential loop of
one minimum and one argmax per pick. The pointnet2-form rows are ops.ball_query /
ops.furthest_point_sample (int32, empty slots filled with the first hit, the reference's tie order). Each time is the median of --reps CUDA-event timings after warm-up, the
variants alternating, with the L2 (126 MB) overwritten before every timed call. The card's name and
power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mocopci_b200 import ops as p2u, p3d_ops, pointconv_util as pcu, synth  # noqa: E402

flush = None


def timed(fn):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def torch_ball_query(p1, p2, K, radius, chunk=512):
    """First K refs with d2 < r^2 in index order: masked index sort per chunk of queries."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    r2 = torch.tensor(radius, dtype=torch.float32) ** 2
    idx = torch.empty((B, P1, K), dtype=torch.int64, device=p1.device)
    dists = torch.empty((B, P1, K), dtype=torch.float32, device=p1.device)
    ar = torch.arange(P2, device=p1.device)
    for s in range(0, P1, chunk):
        d = p1[:, s:s + chunk, None, :] - p2[:, None, :, :]
        d2 = (d * d).sum(-1)
        hit = d2 < r2.to(p1.device)
        key = torch.where(hit, ar, P2)
        first = key.sort(-1).values[..., :K]
        ok = first < P2
        idx[:, s:s + chunk] = torch.where(ok, first, -1)
        dists[:, s:s + chunk] = torch.where(ok, torch.gather(d2, 2, first.clamp(max=P2 - 1)), 0.0)
    return idx, dists


def torch_fps(points, K):
    """Sequential farthest point sampling in torch (one argmax per pick, lowest index on ties)."""
    B, P, _ = points.shape
    idx = torch.zeros((B, K), dtype=torch.int64, device=points.device)
    mind = torch.full((B, P), float("inf"), device=points.device)
    bi = torch.arange(B, device=points.device)
    last = torch.zeros(B, dtype=torch.int64, device=points.device)
    for t in range(1, K):
        d = points - points[bi, last][:, None]
        mind = torch.minimum(mind, (d * d).sum(-1))
        last = mind.argmax(-1)
        idx[:, t] = last
    return idx


def median_ms(fns, reps):
    for _ in range(2):
        for fn in fns:
            fn()
    times = [[] for _ in fns]
    for _ in range(reps):
        for t, fn in zip(times, fns):
            t.append(timed(fn))
    return [round(statistics.median(t) * 1e3, 1) for t in times]


def main():
    global flush
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join("profiles", "r5_p3d_ops_times.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_p3d_ops.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    a = synth.frame_pairs(0, 8)[0].cuda()
    centres = pcu.index_points_gather(a, p2u.furthest_point_sample(a, 4096))
    rows = []
    with torch.no_grad():
        for K in (32, 500):
            fns = [lambda: p3d_ops.ball_query(centres, a, K=K, radius=0.5, return_nn=False),
                   lambda: p3d_ops.ball_query(centres, a, K=K, radius=0.5),
                   lambda: p2u.ball_query(0.5, K, a, centres),
                   lambda: torch_ball_query(centres, a, K, 0.5)]
            t = median_ms(fns, args.reps)
            rows.append({"op": f"ball_query r=0.5 K={K}, 8 x 4096 centres x 16384 points",
                         "p3d_us": t[0], "p3d_return_nn_us": t[1], "pointnet2_form_us": t[2],
                         "torch_restatement_us": t[3]})
            print(json.dumps(rows[-1]), flush=True)
        fns = [lambda: p3d_ops.sample_farthest_points(a, K=4096),
               lambda: p2u.furthest_point_sample(a, 4096),
               lambda: torch_fps(a, 4096)]
        t = median_ms(fns, max(3, args.reps // 4))
        rows.append({"op": "sample_farthest_points 8 x 16384 -> 4096", "p3d_us": t[0], "pointnet2_form_us": t[1],
                     "torch_restatement_us": t[2]})
        print(json.dumps(rows[-1]), flush=True)
    res = {"gpu": gpu, "torch": torch.__version__, "reps": args.reps,
           "method": "median of CUDA-event timings, variants alternating, L2 overwritten before each call "
                     "(the FPS rows use reps // 4, at least 3)",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("gpu:", gpu)


if __name__ == "__main__":
    main()
