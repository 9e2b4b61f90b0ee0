"""Backward of the K-NN distances: the atomic entry point, the deterministic (_det) one and the torch
restatement ((p1[:, :, None] - p2[idx]) ** 2).sum(-1) under autograd, on the same clouds and indices:
python tools/time_knn_grad.py [--reps 30] [--out profiles/r4_knn_grad_times.json]

The two entry points are called directly (as tools/time_grad.py does: under
torch.use_deterministic_algorithms torch would also fill every torch.empty with NaN); their outputs
are overwritten, so no pre-zeroing is timed. The torch restatement is timed as
torch.autograd.grad of its retained graph with the flag off (its gather backward adds with atomics).
The three alternate in one process; each time is the median of --reps CUDA-event timings after
warm-up, with the L2 (126 MB) overwritten before every timed call. A separate profiled pass splits
the _det time into the inverse-index build (scatter_* kernels) and the two reductions. The card's
name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mocopci_b200 import _lib, pointconv_util as pcu, synth  # noqa: E402

L = _lib.lib
flush = None
SHAPES = [("K=16, 8 x 16384^2", 8, 16), ("K=1, 8 x 16384^2 (one Chamfer direction)", 8, 1),
          ("K=16, 1 x 2048^2", 1, 16)]


def timed(fn):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def split(det, reps=5):
    """Device time of the det call's kernels: (inverse-index build us, reductions us) per call."""
    from torch.profiler import ProfilerActivity, profile
    det()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            det()
        torch.cuda.synchronize()
    build = red = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "scatter_" in e.key or e.key.startswith("Memset"):
            build += t
        elif "_det_kernel" in e.key:
            red += t
    return build / reps, red / reps


def case(B, K):
    n = 16384 if B == 8 else 2048
    a, b = synth.frame_pairs(0, B, n)
    p1, p2 = a.cuda(), b.cuda()
    idx, _ = pcu._knn(K, p2, p1, pcu.DIST_DIRECT_XYZ, True)
    g = torch.randn(idx.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(K))
    gq, gr = torch.empty((B, n, 3), device="cuda"), torch.empty((B, n, 3), device="cuda")
    ws = _lib.workspace(L.b200pci_scatter_workspace_bytes(B, n, n * K), p1.device)
    st = _lib.stream_ptr()
    args = (B, n, n, K, p1.data_ptr(), n * 3, 3, 1, p2.data_ptr(), n * 3, 3, 1, idx.data_ptr(), 1, g.data_ptr(),
            gq.data_ptr(), gr.data_ptr())
    atomic = lambda: _lib.check(L.b200pci_knn_backward(*args, st), "knn_backward")  # noqa: E731
    det = lambda: _lib.check(L.b200pci_knn_backward_det(*args, ws.data_ptr(), ws.numel(), st),  # noqa: E731
                             "knn_backward_det")
    x, y = p1.clone().requires_grad_(True), p2.clone().requires_grad_(True)
    bi = torch.arange(B, device="cuda")[:, None, None]
    d = ((x[:, :, None] - y[bi, idx]) ** 2).sum(-1)
    restated = lambda: torch.autograd.grad(d, (x, y), g, retain_graph=True)  # noqa: E731
    return atomic, det, restated, (gq, gr, ws, g, idx, d)


def main():
    global flush
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join("profiles", "r4_knn_grad_times.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_knn_grad.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rows = []
    for name, B, K in SHAPES:
        fns = case(B, K)[:3]
        for _ in range(3):
            for fn in fns:
                fn()
        times = [[], [], []]
        for _ in range(args.reps):  # alternating
            for t, fn in zip(times, fns):
                t.append(timed(fn))
        ta, td, tt = (statistics.median(t) * 1e3 for t in times)
        build, red = split(fns[1])
        rows.append({"case": name, "atomic_us": round(ta, 1), "det_us": round(td, 1), "torch_autograd_us": round(tt, 1),
                     "det_over_atomic": round(td / ta, 2), "det_index_build_us": round(build, 1),
                     "det_reductions_us": round(red, 1)})
        print(json.dumps(rows[-1]), flush=True)
    res = {"gpu": gpu, "torch": torch.__version__, "reps": args.reps,
           "method": "median of CUDA-event timings, atomic / det / torch restatement alternating, L2 overwritten "
                     "before each call; index build / reductions from torch.profiler kernel times of 5 det calls",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("gpu:", gpu)


if __name__ == "__main__":
    main()
