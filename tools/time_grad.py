"""Atomic vs deterministic (fixed-order) backward of every scatter-add gradient, at the shapes the
tests check them at: python tools/time_grad.py [--reps 30] [--out profiles/r3_grad_det_times.json]

Calls the C entry points directly: under torch.use_deterministic_algorithms(True) torch also fills
every torch.empty with NaN, which would blur a comparison of the kernels. The two paths alternate in
one process; each time is the median of --reps CUDA-event timings after warm-up, with the L2 (126 MB)
overwritten before every timed call. The pre-zeroing of the output (torch.zeros in the autograd
functions) is inside both timings; Chamfer's backward overwrites its output and needs none. A
separate profiled pass splits the deterministic time into the inverse-index build (scatter_*
kernels) and the reduction. The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mocopci_b200 import _lib, ops, pointconv_util as pcu, synth  # noqa: E402

L = _lib.lib
flush = None


def timed(fn):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def compare(atomic, det, reps):
    for _ in range(3):
        atomic()
        det()
    ta, td = [], []
    for _ in range(reps):  # alternating
        ta.append(timed(atomic))
        td.append(timed(det))
    return statistics.median(ta) * 1e3, statistics.median(td) * 1e3


def split(det, reps=5):
    """Device time of the det call's kernels: (inverse-index build us, reduction us) per call."""
    from torch.profiler import ProfilerActivity, profile
    det()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            det()
        torch.cuda.synchronize()
    build = red = 0.0
    for e in prof.key_averages():
        name = e.key
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "scatter_" in name or name.startswith("Memset"):
            build += t
        elif "_det_kernel" in name:
            red += t
    return build / reps, red / reps


def cases():
    a, b = synth.frame_pairs(0, 8)
    a, b = a.cuda(), b.cuda()
    fidx = ops.furthest_point_sample(a, 4096)
    centres = pcu.index_points_gather(a, fidx)
    bq = ops.ball_query(0.5, 32, a, centres)
    st = _lib.stream_ptr()
    g = torch.Generator("cuda").manual_seed(0)

    def gg(name, C, idx, group):
        T = idx[0].numel()
        gout = torch.randn((8, C) + tuple(idx.shape[1:]), device="cuda", generator=g)
        gp = torch.zeros((8, C, 16384), device="cuda")
        ws = _lib.workspace(L.b200pci_scatter_workspace_bytes(8, 16384, T), a.device)
        if group:
            P, S = idx.shape[1], idx.shape[2]
            atomic = lambda: (gp.zero_(), L.b200pci_group_points_grad(8, C, 16384, P, S, gout.data_ptr(), idx.data_ptr(), gp.data_ptr(), st))  # noqa: E731,E501
            det = lambda: (gp.zero_(), L.b200pci_group_points_grad_det(8, C, 16384, P, S, gout.data_ptr(), idx.data_ptr(), gp.data_ptr(), ws.data_ptr(), ws.numel(), st))  # noqa: E731,E501
        else:
            P = idx.shape[1]
            atomic = lambda: (gp.zero_(), L.b200pci_gather_points_grad(8, C, 16384, P, gout.data_ptr(), idx.data_ptr(), gp.data_ptr(), st))  # noqa: E731,E501
            det = lambda: (gp.zero_(), L.b200pci_gather_points_grad_det(8, C, 16384, P, gout.data_ptr(), idx.data_ptr(), gp.data_ptr(), ws.data_ptr(), ws.numel(), st))  # noqa: E731,E501
        return name, atomic, det, (gout, gp, ws)

    yield gg("group_points_grad_C128 (config 2, B=8, 4096x32 -> 16384)", 128, bq, True)
    yield gg("group_points_grad_C3 (config 2)", 3, bq, True)
    yield gg("gather_points_grad_C128 (4096 FPS centres -> 16384, B=8)", 128, fidx, False)
    yield gg("group_points_grad_C128, idx all one value", 128, torch.full_like(bq, 4321), True)
    for n, m in ((16384, 4096), (4096, 1024), (1024, 256), (256, 64)):
        w, i3, _ = ops.three_nn_weights(a[:, :n].contiguous(), a[:, :m].contiguous())
        gout = torch.randn((8, 128, n), device="cuda", generator=g)
        gp = torch.zeros((8, 128, m), device="cuda")
        ws = _lib.workspace(L.b200pci_scatter_workspace_bytes(8, m, 3 * n), a.device)
        yield (f"three_interpolate_grad_C128 {m}->{n} (B=8)",
               lambda gout=gout, gp=gp, i3=i3, w=w, n=n, m=m: (gp.zero_(), L.b200pci_three_interpolate_grad(8, 128, n, m, gout.data_ptr(), i3.data_ptr(), w.data_ptr(), gp.data_ptr(), st)),  # noqa: E501
               lambda gout=gout, gp=gp, i3=i3, w=w, n=n, m=m, ws=ws: (gp.zero_(), L.b200pci_three_interpolate_grad_det(8, 128, n, m, gout.data_ptr(), i3.data_ptr(), w.data_ptr(), gp.data_ptr(), ws.data_ptr(), ws.numel(), st)),  # noqa: E501
               (gout, gp, ws, w, i3))
    kidx = pcu.knn_point(16, a, b)
    gout = torch.randn((8, 16384, 16, 64), device="cuda", generator=g)
    gp = torch.zeros((8, 16384, 64), device="cuda")
    T = 16384 * 16
    ws = _lib.workspace(L.b200pci_scatter_workspace_bytes(8, 16384, T), a.device)
    yield ("index_points_rows_grad_C64_k16 (int64, B=8)",
           lambda: (gp.zero_(), L.b200pci_index_points_rows_grad(8, 16384, T, 64, gout.data_ptr(), kidx.data_ptr(), 1, gp.data_ptr(), st)),  # noqa: E501
           lambda: (gp.zero_(), L.b200pci_index_points_rows_grad_det(8, 16384, T, 64, gout.data_ptr(), kidx.data_ptr(), 1, gp.data_ptr(), ws.data_ptr(), ws.numel(), st)),  # noqa: E501
           (gout, gp, ws, kidx))
    # chamfer_B8: indices from the forward
    ix = torch.empty((8, 16384), dtype=torch.int32, device="cuda")
    iy = torch.empty_like(ix)
    dx, dy = torch.empty((8, 16384), device="cuda"), torch.empty((8, 16384), device="cuda")
    loss = torch.empty((1,), device="cuda")
    fws = _lib.workspace(L.b200pci_chamfer_workspace_bytes(8, 16384, 16384), a.device)
    _lib.check(L.b200pci_chamfer_forward(8, 16384, 16384, a.data_ptr(), 16384 * 3, 3, 1, b.data_ptr(), 16384 * 3, 3, 1,
                                         dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(), loss.data_ptr(),
                                         fws.data_ptr(), fws.numel(), st), "chamfer_forward")
    gl = torch.ones(1, device="cuda")
    gx, gy = torch.empty((8, 16384, 3), device="cuda"), torch.empty((8, 16384, 3), device="cuda")
    cws = _lib.workspace(L.b200pci_chamfer_backward_det_workspace_bytes(8, 16384, 16384), a.device)
    yield ("chamfer_backward_B8 (16384 x 16384)",
           lambda: L.b200pci_chamfer_backward(8, 16384, 16384, a.data_ptr(), b.data_ptr(), ix.data_ptr(), iy.data_ptr(), gl.data_ptr(), gx.data_ptr(), gy.data_ptr(), st),  # noqa: E501
           lambda: L.b200pci_chamfer_backward_det(8, 16384, 16384, a.data_ptr(), b.data_ptr(), ix.data_ptr(), iy.data_ptr(), gl.data_ptr(), gx.data_ptr(), gy.data_ptr(), cws.data_ptr(), cws.numel(), st),  # noqa: E501
           (gx, gy, cws))


def main():
    global flush
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join("profiles", "r3_grad_det_times.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_grad.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rows = []
    for name, atomic, det, _keep in cases():
        for fn in (atomic, det):
            rc = fn()
            rc = rc[-1] if isinstance(rc, tuple) else rc
            _lib.check(rc, name)
        ta, td = compare(atomic, det, args.reps)
        build, red = split(det)
        rows.append({"case": name, "atomic_us": round(ta, 1), "det_us": round(td, 1),
                     "det_over_atomic": round(td / ta, 2), "det_index_build_us": round(build, 1),
                     "det_reduction_us": round(red, 1)})
        print(json.dumps(rows[-1]), flush=True)
    res = {"gpu": gpu, "torch": torch.__version__, "reps": args.reps,
           "method": "median of CUDA-event timings, atomic and det alternating, L2 overwritten before each call; "
                     "index build / reduction from torch.profiler kernel times of 5 det calls",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("gpu:", gpu)


if __name__ == "__main__":
    main()
