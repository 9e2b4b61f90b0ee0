#!/usr/bin/env python
"""Benchmark of the MoCoPCI neighbourhood hot path on B200 (contract: task brief / DESIGN.md section 7).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras]
                    [--dump-outputs DIR]

Headline metric (BASELINE.json): KNN queries/s, k=16, 16384 queries x 16384 refs per frame pair.
A *step* is one pass of ``knn_point(16, frame t, frame t+1)`` over the rank's batch of synthetic
LiDAR frame pairs -- 64 per GPU (the batch of BASELINE config 5); ranks own disjoint pairs and
there is no data-path collective => weak scaling.

  value       whole-job queries/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e         same metric through the host-buffer C-ABI call (pinned host clouds in, int64 indices
              out; H2D + D2H inside the timed region)
  roofline    the dominant kernel alone (knn_scan_tc_kernel): SURVEY 8d's 8 FLOP per pair / its
              CUDA-event time on the launching stream, against the FP32 FMA peak measured in the same
              run by the library's FFMA probe (north_star reports KNN against peak FP32)
  cpu_baseline  the reference's own CPU torch path (models/pointconv_util.py square_distance + topk,
              imported unmodified from baseline/_ref) on a bounded sample
  full_model  BASELINE's second metric: frame pairs/s of the unmodified reference MoCoPCI forward
              (models/m_models/mocopci.py) on the B200 kernels through mocopci_b200.install()
  eval64      BASELINE config 5: 64 frame pairs strong-scaled over the ranks -- inference + Chamfer
              + EMD per interpolated frame, one NCCL all-reduce of the metric sums at the end
  kernels     (extras, N=1) the other rows of SURVEY section 8d with their own rooflines

``--impl reference`` times only the CPU path (rank 0; other ranks exit 0).

``--dump-outputs DIR`` writes what the timed KNN call returned in its last timed step, so that two
builds can be compared output for output (the inputs depend on the rank only): a fixed, seeded
sample of DUMP_ROWS (frame pair, query) rows of the int64 indices, as float32, to
DIR/knn_idx.npy (DIR/knn_idx_rank<r>.npy when several ranks run), and the rows' positions as
DIR/knn_rows.npy (pair index, query index).
"""
import argparse
import ctypes
import glob
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "knn_queries_per_sec_k16_n16384"
UNIT = "queries/s"
NPTS = 16384
K = 16
PAIRS_PER_GPU = 64  # BASELINE config 5's batch; one knn_point call per step
EVAL_PAIRS = 64
FLOP_PER_PAIR = 8.0  # SURVEY 8d: 3 sub, 3 mul, 2 add (equivalently the expanded form)
T_INTERP = [0.4167, 0.5, 0.5833]  # train.py:49-55 with the defaults
DUMP_ROWS = 65536  # of the 64 x 16384 query rows a step returns: 4 MiB of indices as float32


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def committed_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/
    r*_traffic.json, written by tools/ncu_summary.py --traffic from an `ncu --set full` report of
    this command); None if no capture of the current kernel is committed."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not files:
        return None, None
    try:
        with open(files[-1]) as f:
            d = json.load(f)
        return d, os.path.relpath(files[-1], ROOT)
    except Exception:
        return None, None


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Summary of the samples that arrived in [t0, t1] (the timed region); if the region was
        shorter than two sampling periods, the samples of the surrounding load are used instead."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [l for t, l in self.lines if t0 is not None and t0 <= t <= t1 + 0.03]
        window = "timed region"
        if len(inside) < 2:
            inside = [l for _, l in self.lines[1:]]
            window = "warm-up + timed region (timed region shorter than two sampling periods)"
        for line in inside:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ---------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline
# ---------------------------------------------------------------------------------------------
def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm may use every core of the box."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(max(n, 1))
    return torch.get_num_threads()


def reference_cpu_knn():
    """``knn_point`` of the reference's own models/pointconv_util.py, imported UNMODIFIED from the
    checkout (baseline/_ref on the GPU box) with its CUDA / pytorch3d imports stubbed (neither is
    used by square_distance + topk). Falls back to the torch restatement oracle/torch_port.py only
    if no checkout travelled. Returns (callable, kind, description)."""
    from baseline import fetch_ref
    root = fetch_ref.root()
    where = None if root is None else (os.path.relpath(root, ROOT) if root.startswith(ROOT) else root)
    what = f"models/pointconv_util.py:67-88,129-140 imported unmodified from {where}"
    already = sys.modules.get("models.pointconv_util")
    if already is not None:  # the full-model leg imported it under install(): take the ORIGINAL function
        fn = already.knn_point
        return getattr(fn, "__b200pci_original__", fn), "reference", what
    if root is not None:
        import importlib
        import types
        before = set(sys.modules)
        saved = {n: sys.modules.get(n) for n in ("pointnet2_cuda", "pytorch3d", "pytorch3d.ops", "pytorch3d.loss")}
        for name in saved:
            sys.modules[name] = types.ModuleType(name)
        sys.modules["pytorch3d.ops"].knn_points = None
        sys.modules["pytorch3d.loss"].chamfer_distance = None
        sys.path.insert(0, root)
        try:
            pcu = importlib.import_module("models.pointconv_util")
            fn = pcu.knn_point
            return getattr(fn, "__b200pci_original__", fn), "reference", what
        except Exception as e:  # noqa: BLE001
            print(f"bench.py: reference import failed ({e!r}); using the torch port", file=sys.stderr)
        finally:
            sys.path.remove(root)
            for name in set(sys.modules) - before:
                sys.modules.pop(name, None)
            for name, mod in saved.items():
                if mod is None:
                    sys.modules.pop(name, None)
                else:
                    sys.modules[name] = mod
    from oracle import torch_port
    return torch_port.knn_point, "port", "oracle/torch_port.py restatement of models/pointconv_util.py:67-88,129-140"


def cpu_knn_baseline(reps, warm=1):
    """The reference's CPU torch path on ONE frame pair per repetition (bounded sample)."""
    from mocopci_b200 import synth
    fn, kind, what = reference_cpu_knn()
    a, b = synth.frame_pair(0, NPTS)
    a, b = a[None], b[None]
    times = []
    for i in range(warm + reps):
        t0 = time.perf_counter()
        idx = fn(K, a, b)
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    assert tuple(idx.shape) == (1, NPTS, K)
    return times, kind, what


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = use_all_host_threads()
    warm = min(args.warmup, 2)
    times, kind, what = cpu_knn_baseline(args.steps, warm=warm)
    total = sum(times)
    value = NPTS * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": warm, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "knn_point k=16, 16384 queries x 16384 refs per frame pair "
                               "(reference CPU torch path: square_distance + topk)",
                   "points": NPTS, "k": K, "pairs_per_step": 1},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"1 frame pair per step ({NPTS} queries x {NPTS} refs), "
                                   f"{len(times)} steps; torch {torch.__version__}; {what}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def ev_pair():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def time_steps(fn, steps, warmup, flush=None):
    """CUDA-event time of each step (ms); L2 flushed (untimed) before every step."""
    for _ in range(warmup):
        if flush is not None:
            flush()
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        if flush is not None:
            flush()
        a, b = ev_pair()
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def fp32_peak(_lib):
    """FFMA probe of the library: best of 10, scalar and packed; TFLOP/s."""
    sink = torch.zeros(4, device="cuda")
    fl = ctypes.c_double()
    best = 0.0
    for packed in (0, 1):
        def run():
            _lib.check(_lib.lib.b200pci_probe_fp32(packed, 4096, sink.data_ptr(), ctypes.byref(fl),
                                                   _lib.stream_ptr()))
        ts = time_steps(run, 10, 3)
        best = max(best, fl.value / (min(ts) * 1e-3) / 1e12)
    return best


def count_launches(fn):
    """Kernel launches of one call, by name, from CUPTI (torch.profiler sees every kernel of the
    process, ours included). Returns [(name, count)] in first-launch order."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():
        if "cuda" in str(getattr(e, "device_type", "")).lower() and not e.name.startswith(("Memcpy", "Memset")):
            names.append(e.name.split("<")[0].split("(")[0].replace("void ", "").replace("b200pci::", ""))
    out = []
    for n in names:
        for i, (m, c) in enumerate(out):
            if m == n:
                out[i] = (m, c + 1)
                break
        else:
            out.append((n, 1))
    return out


def graph_median(fn, steps=10, warm=3, fl=None):
    """Median CUDA-event time of a CUDA-graph replay of ``fn`` (so that the Python/ctypes launch
    overhead of tens of us does not hide short kernels; same kernels, same stream either way)."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        run = g.replay
    except Exception:  # noqa: BLE001
        run = fn
    return statistics.median(time_steps(run, steps, warm, fl))


def extras(_lib, peaks, fp32_tf, a, b, flush):
    """Other rows of SURVEY 8d on this rank's first 8 frame pairs: time + roofline each."""
    from mocopci_b200 import chamfer, emd_cuda, ops as p2u, pointconv_util as pcu
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    a, b = a[:8].contiguous(), b[:8].contiguous()
    B = a.shape[0]
    out = {}
    med = graph_median

    def fp(name, ms, flops, **kw):
        out[name] = dict(ms=ms, tflops=flops / (ms * 1e-3) / 1e12, bound="fp32",
                         frac=flops / (ms * 1e-3) / 1e12 / fp32_tf, **kw)

    def bw(name, ms, nbytes, **kw):
        out[name] = dict(ms=ms, gbs=nbytes / (ms * 1e-3) / 1e9, bound="hbm",
                         frac=nbytes / (ms * 1e-3) / 1e9 / hbm, **kw)

    pairs = float(B) * NPTS * NPTS
    fp("knn_k16_B8", med(lambda: pcu.knn_point(16, a, b), fl=flush), 8 * pairs)
    fp("knn_k32_B8", med(lambda: pcu.knn_point(32, a, b), fl=flush), 8 * pairs)
    fp("knn_k16_B1", med(lambda: pcu.knn_point(16, a[:1], b[:1])), 8.0 * NPTS * NPTS)
    fp("knn_k32_B1_self", med(lambda: pcu.knn_point(32, a[:1], a[:1])), 8.0 * NPTS * NPTS,
       note="the model's finest level (8 calls per forward)")
    fp("knn_k3_16384x2048_B1", med(lambda: pcu.knn_point(3, a[:1, :2048], b[:1])), 8.0 * NPTS * 2048,
       note="UpsampleFlow at l0 (15 calls per forward)")
    fp("chamfer_B8", med(lambda: chamfer.chamfer_distance(a, b)), 16 * pairs)
    t = med(lambda: p2u.furthest_point_sample(a, 4096), steps=3, warm=1)
    fp("fps_16384_to_4096", t, 8.0 * B * NPTS * 4095, us_per_iteration=t * 1e3 / 4095)
    fidx = p2u.furthest_point_sample(a, 4096)
    centres = pcu.index_points_gather(a, fidx)
    fp("ball_query_r0.5_ns32", med(lambda: p2u.ball_query(0.5, 32, a, centres)),
       8.0 * B * 4096 * NPTS, note="upper-bound work (early exit not subtracted)")
    idx = p2u.ball_query(0.5, 32, a, centres)
    feats = torch.randn(B, 128, NPTS, device="cuda", generator=torch.Generator("cuda").manual_seed(99))
    t = med(lambda: p2u.grouping_operation(feats, idx), fl=flush)
    bw("group_points_C128", t, 4.0 * B * (128 * 4096 * 32 + 4096 * 32 + 128 * NPTS))
    xyz_t = a.transpose(1, 2).contiguous()
    t = med(lambda: p2u.grouping_operation(xyz_t, idx), fl=flush)
    bw("group_points_C3", t, 4.0 * B * (3 * 4096 * 32 + 4096 * 32 + 3 * NPTS))
    t = med(lambda: p2u.query_and_group(0.5, 32, a, centres, feats), fl=flush)
    out["query_and_group_C128"] = dict(ms=t, note="ball_query + group xyz (minus centre) + group features + concat")
    # K3: index_points_group on the KNN result, [B,N,C] layout, C = 64 (fused row gather)
    kidx = pcu.knn_point(16, a, b)
    fbnc = torch.randn(B, NPTS, 64, device="cuda")
    t = med(lambda: pcu.index_points_group(fbnc, kidx), fl=flush)
    bw("index_points_group_C64_k16", t, 4.0 * B * (NPTS * 16 * 64 + NPTS * 64) + 8.0 * B * NPTS * 16)
    # feature propagation pyramid 64 -> 256 -> 1024 -> 4096 -> 16384 (config 3)
    nn_ms, nn_fl, it_ms, it_by = 0.0, 0.0, 0.0, 0.0
    levels = {}
    for n, m in ((256, 64), (1024, 256), (4096, 1024), (16384, 4096)):
        unknown, known = a[:, :n].contiguous(), a[:, :m].contiguous()
        t_nn = med(lambda: p2u.three_nn_weights(unknown, known))
        nn_ms += t_nn
        nn_fl += 8.0 * B * n * m
        w, i3, _ = p2u.three_nn_weights(unknown, known)
        f = torch.randn(B, 128, m, device="cuda")
        t_it = med(lambda: p2u.three_interpolate(f, i3, w), fl=flush)
        it_ms += t_it
        by = 4.0 * B * (128 * n + 128 * m + 6 * n)
        it_by += by
        levels[f"{m}->{n}"] = dict(three_nn_weights_ms=t_nn, three_interpolate_ms=t_it,
                                   three_interpolate_gbs=by / (t_it * 1e-3) / 1e9)
    fp("three_nn_weights_pyramid", nn_ms, nn_fl, note="three_nn + fused inverse-distance weights (T3)")
    bw("three_interpolate_pyramid_C128", it_ms, it_by, levels=levels)
    bw("three_interpolate_4096_to_16384_C128", levels["4096->16384"]["three_interpolate_ms"],
       4.0 * B * (128 * 16384 + 128 * 4096 + 6 * 16384))
    # f2 / f1: the model's feature-space KNN (l1: 2048 points, 64 channels, permuted view) and the fused
    # group() of PointConv(32) at level 0 (16384 x 32 neighbours x (3 + 32) channels)
    feat = torch.randn(1, 64, 2048, device="cuda").permute(0, 2, 1)
    t = med(lambda: pcu.knn_point_cosine(16, feat, feat))
    out["knn_point_cosine_2048_C64_k16"] = dict(ms=t, tensor_tflops=3 * 2.0 * 2048 * 2048 * 64 / (t * 1e-3) / 1e12,
                                                note="normalise+split pass and tcgen05 3xTF32 contraction + top-k; "
                                                     "39 calls per forward at 256..2048 points: latency bound")
    f32 = torch.randn(1, 32, NPTS, device="cuda").permute(0, 2, 1)
    gidx = pcu.knn_point(32, a[:1], a[:1])
    t = med(lambda: pcu._group_concat(a[:1], a[:1], f32, gidx), fl=flush)
    bw("group_concat_16384_k32_C32", t, 4.0 * (NPTS * 32 * 35 + NPTS * 32 * 3 + NPTS * 35) + 8.0 * NPTS * 32)
    # EMD at the BASELINE size: one 16384 x 16384 pair, forward-only (never stores match) and compat
    x1, x2 = a[:1].contiguous(), b[:1].contiguous()
    t = med(lambda: emd_cuda.emd_cost(x1, x2), steps=3, warm=1)
    ex2 = 30.0 * NPTS * NPTS  # 10 levels x 3 sweeps x n x m exponentials
    out["emd_cost_16384"] = dict(ms=t, gexp_per_s=ex2 / (t * 1e-3) / 1e9, bound="mufu",
                                 frac=ex2 / (t * 1e-3) / (148 * 16 * 1.965e9),
                                 note="forward-only approxmatch + matchcost, no match matrix; MUFU bound: "
                                      "30 x 16384^2 ex2 against 148 SMs x 16/clk x 1.965 GHz")
    t = med(lambda: emd_cuda.matchcost_forward(x1, x2, emd_cuda.approxmatch_forward(x1, x2)), steps=3, warm=1)
    out["emd_match_16384"] = dict(ms=t, note="approxmatch_forward + matchcost_forward (1.07 GB match matrix, "
                                             "read-modify-written by all 10 levels)")
    return out


def full_model_leg(steps, dist, world):
    """BASELINE's second metric: the UNMODIFIED reference model (imported from the checkout) on the
    B200 kernels through mocopci_b200.install(); one frame pair (B=1, 16384 points) per forward."""
    from baseline import fetch_ref
    root = fetch_ref.root()
    if root is None:
        return None, {"unavailable": "no reference checkout (baseline/_ref) next to bench.py"}
    import importlib
    import mocopci_b200
    from mocopci_b200 import synth
    mocopci_b200.install(reference_root=root)
    mm = importlib.import_module("models.m_models.mocopci")
    torch.manual_seed(0)
    net = mm.MoCoPCI().cuda().eval()
    rank = int(os.environ.get("RANK", "0"))
    a, b = synth.frame_pairs(1000 + rank, 1, NPTS)
    x1, x2 = a.permute(0, 2, 1).contiguous().cuda(), b.permute(0, 2, 1).contiguous().cuda()
    with torch.no_grad():
        for _ in range(2):
            net(x1, x2, None, T_INTERP, False)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        ts = []
        for _ in range(steps):
            e0, e1 = ev_pair()
            e0.record()
            out = net(x1, x2, None, T_INTERP, False)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
    tot = torch.tensor([sum(ts)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    info = {"frame_pairs_per_s": world * steps / (float(tot) * 1e-3), "unit": "frame pairs/s",
            "ms_per_forward": statistics.median(ts), "forwards_per_rank": steps, "batch": 1,
            "points": NPTS, "interpolated_frames": len(out),
            "model": "models/m_models/mocopci.py MoCoPCI (random init, seed 0, eval()), unmodified, "
                     f"imported from {os.path.relpath(root, ROOT) if root.startswith(ROOT) else root} "
                     "via mocopci_b200.install()"}
    return net, info


def eval64_leg(net, dist, rank, world):
    """BASELINE config 5: 64 frame pairs, contiguous shards over the ranks (strong scaling). Per
    pair: one forward (3 interpolated frames), then Chamfer + EMD of every interpolated frame
    against its target -- the loop of test.py:72-123 -- accumulated per frame and reduced with ONE
    all_reduce over NCCL at the end. Synthetic targets: the second input frame."""
    from mocopci_b200 import chamfer, ops, sharding, synth
    mine = sharding.shard_pairs(EVAL_PAIRS, rank, world)
    acc = sharding.MetricAccumulator(3, device="cuda")
    # the frames as a DataLoader with workers hands them over: ready in pinned host memory; the
    # host-to-device copy of every pair is inside the timed region
    frames = [tuple(t.pin_memory() for t in synth.frame_pairs(2000 + p, 1, NPTS)) for p in mine]
    # The forward is host-bound (the reference's Python launches ~6900 small kernels), the metrics
    # are device-bound (EMD: 30 grid-wide sweeps per frame): the metrics of pair i run on a second
    # stream while the host is already launching the forward of pair i+1.
    main = torch.cuda.current_stream()
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = ev_pair()
    e0.record()
    with torch.no_grad():
        for a_h, b_h in frames:
            a, b = a_h.cuda(non_blocking=True), b_h.cuda(non_blocking=True)
            if net is not None:
                preds = net(a.permute(0, 2, 1).contiguous(), b.permute(0, 2, 1).contiguous(), None, T_INTERP, False)
            else:
                preds = [a + (b - a).mean(1, keepdim=True) * t for t in T_INTERP]
            preds = [pred.contiguous() for pred in preds]
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for j, pred in enumerate(preds):
                    pred.record_stream(side)
                    cd = chamfer.chamfer_distance(pred, b)[0]                       # test.py:89
                    emd = ops.earth_mover_distance(pred, b, transpose=False).mean() / NPTS  # test.py:90
                    acc.add_tensors(j, cd, emd)
                b.record_stream(side)
    main.wait_stream(side)
    e1.record()
    totals = acc.reduce(dist)
    torch.cuda.synchronize()
    wall = torch.tensor([e0.elapsed_time(e1) * 1e-3, time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    return {"pairs": EVAL_PAIRS, "pairs_per_rank": len(mine), "scaling": "strong",
            "pairs_per_s": EVAL_PAIRS / float(wall[1]), "seconds": float(wall[1]),
            "device_seconds_max_rank": float(wall[0]),
            "with_model_inference": net is not None,
            "pipeline": "frames pre-loaded in pinned host memory (H2D copy timed); metrics of pair i on a second "
                        "stream beside the host-bound forward of pair i+1",
            "cd_mean_per_frame": totals["cd_mean"], "emd_mean_per_frame": totals["emd_mean"],
            "count_per_frame": totals["count"],
            "reduce": "one all_reduce(SUM) of a 9-element FP64 vector over NCCL" if dist is not None else "single rank"}


def dump_outputs(out_dir, idx, name):
    """A seeded sample of DUMP_ROWS rows of ``idx`` [pairs, queries, k] (the same rows every run)."""
    import numpy as np
    pairs, queries, _ = idx.shape
    rows = torch.randperm(pairs * queries, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort()[0]
    sample = idx.reshape(pairs * queries, -1)[rows.cuda()].float().cpu().numpy()  # indices < 2^24: exact
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), sample)
    if int(os.environ.get("RANK", "0")) == 0:  # the same rows on every rank
        np.save(os.path.join(out_dir, "knn_rows.npy"),
                np.stack([(rows // queries).numpy(), (rows % queries).numpy()], 1).astype(np.float64))


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (mocopci_b200 has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    from mocopci_b200 import _lib, host_api, pointconv_util as pcu, synth
    # host staging buffers next to this rank's GPU (matters for the host-buffer path at 8 ranks)
    numa_cpus = host_api.bind_to_gpu_numa_node(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks, peak_src = load_peaks()

    # this rank's frame pairs: refs = frame t, queries = frame t+1
    a_h, b_h = synth.frame_pairs(rank * PAIRS_PER_GPU, PAIRS_PER_GPU, NPTS)
    a_pin, b_pin = a_h.pin_memory(), b_h.pin_memory()
    a, b = a_pin.cuda(non_blocking=True), b_pin.cuda(non_blocking=True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    flush_rd = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")  # 256 MiB, only ever read
    flush_sink = torch.zeros(1, dtype=torch.float32, device="cuda")

    def flush():
        # write a buffer larger than L2 (evicts every input), then READ a second one so that the
        # cache is left full of CLEAN lines: after the write alone, the first ~126 MB a timed kernel
        # stores would each pay for the write-back of a dirty flush line (a 70 MB kernel measured
        # at half its bandwidth that way)
        flush_buf.zero_()
        torch.sum(flush_rd, dim=0, keepdim=True, out=flush_sink)

    def step():
        return pcu.knn_point(K, a, b)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # parity of the benchmarked workload, asserted once before timing: the first frame pair of
    # this rank against the C oracle (OpenMP, seconds) -- every index
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import cpu as orc  # checker only
        want = orc.knn_form(5, K, a_h[:1].numpy(), b_h[:1].numpy())[0]  # form 5: the reference as CUDA torch runs it
        got = step()[:1].cpu().numpy()
        assert (got == want).all(), "bench.py: KNN indices of the benchmarked pair differ from the oracle"
        parity = "pair 0 (16384 x 16384, k=16): all 262144 indices equal to oracle/oracle.c"
        del want, got

    fp32_tf = fp32_peak(_lib) if rank == 0 else 0.0
    launches = count_launches(step) if rank == 0 else []

    # ---- device-resident timing (value) + selection-kernel timing (roofline) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_warm = time.time()
    last = None
    while True:  # W warm-up steps, and at least 0.3 s of load so that nvidia-smi is sampling
        for _ in range(max(args.warmup, 3)):
            flush()
            # kept like the timed loop keeps it, so that the allocator already holds the two
            # output blocks the timed steps alternate between
            last = step()
        torch.cuda.synchronize()
        if time.time() - t_warm > 0.3:
            break
    barrier()
    t_region0 = time.time()
    _lib.check(_lib.lib.b200pci_debug_set(3, 1))
    evs = []
    for _ in range(args.steps):
        flush()
        e0, e1 = ev_pair()
        e0.record()
        last = step()
        e1.record()
        evs.append((e0, e1))
    barrier()
    t_region1 = time.time()
    step_ms = [x.elapsed_time(y) for x, y in evs]
    kern_ms = _lib.lib.b200pci_debug_get(3)
    kern_n = int(_lib.lib.b200pci_debug_get(4))
    _lib.check(_lib.lib.b200pci_debug_set(3, 0))
    clocks = sampler.stop(t_region0, t_region1) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, "knn_idx" if world == 1 else f"knn_idx_rank{rank}")
    del last
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)

    # ---- end to end through the host-buffer C-ABI call ----
    idx_host = torch.empty((PAIRS_PER_GPU, NPTS, K), dtype=torch.int64, pin_memory=True)
    for _ in range(3):
        host_api.knn_point_host(K, a_pin, b_pin, out=idx_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_api.knn_point_host(K, a_pin, b_pin, out=idx_host)  # synchronises its stream
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s)

    # the same call with int32 indices in the host buffer (what the pointnet2 ops consume; the
    # reference's knn_point returns int64, so the headline e2e above keeps int64): half the D2H bytes
    idx_host32 = torch.empty((PAIRS_PER_GPU, NPTS, K), dtype=torch.int32, pin_memory=True)
    e2e32_steps = max(3, min(args.steps, 10))
    host_api.knn_point_host(K, a_pin, b_pin, out=idx_host32)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e32_steps):
        host_api.knn_point_host(K, a_pin, b_pin, out=idx_host32)
    torch.cuda.synchronize()
    e2e32_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e32_s, op=dist.ReduceOp.MAX)
    e2e32_s = float(e2e32_s)

    # final metric reduction over NVLink: index checksum (the host path must agree with the device path)
    ref_idx = step()
    assert torch.equal(idx_host32.cuda().long(), ref_idx), "int32 host-buffer path disagrees with device path"
    checksum = ref_idx.sum().double().reshape(1)
    assert torch.equal(idx_host.cuda(), ref_idx), "host-buffer path disagrees with device path"
    del ref_idx
    if dist is not None:
        dist.all_reduce(checksum, op=dist.ReduceOp.SUM)

    # ---- BASELINE's second metric and config 5 ----
    net, full_model = (None, None)
    eval64 = None
    if not args.no_model:
        try:
            net, full_model = full_model_leg(args.model_steps, dist, world)
        except Exception as e:  # noqa: BLE001
            if world > 1:
                raise
            full_model = {"unavailable": f"{type(e).__name__}: {e}"}
    if not args.no_eval:
        eval64 = eval64_leg(net, dist, rank, world)

    queries_per_step = world * PAIRS_PER_GPU * NPTS
    line = None
    if rank == 0:
        flops_per_launch = FLOP_PER_PAIR * PAIRS_PER_GPU * NPTS * NPTS
        kern_avg_ms = kern_ms / max(kern_n, 1)
        achieved = flops_per_launch / (kern_avg_ms * 1e-3) / 1e12
        traffic, traffic_src = committed_traffic()
        n_launch = sum(c for _, c in launches)
        line = {
            "metric": METRIC, "value": queries_per_step * args.steps / (total_ms * 1e-3),
            "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "knn_point k=16 over a batch of 64 synthetic LiDAR frame pairs per GPU "
                                   "(queries: frame t+1, refs: frame t), 16384 points per frame",
                       "pairs_per_gpu": PAIRS_PER_GPU, "global_pairs": world * PAIRS_PER_GPU,
                       "points": NPTS, "k": K, "parallelism": f"frame pairs sharded over {world} GPU(s), "
                       "no data-path collective",
                       "l2": "before every timed step a 256 MiB buffer is written and a second 256 MiB buffer read "
                             "(L2 flushed and left clean; inputs are 25 MiB)",
                       "host_numa_binding": bool(numa_cpus)},
            "e2e": {"value": queries_per_step * args.steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": int(2 * PAIRS_PER_GPU * NPTS * 3 * 4),
                    "d2h_bytes_per_step": int(PAIRS_PER_GPU * NPTS * K * 8),
                    "api": "mocopci_b200.host_api.knn_point_host -> b200pci_knn_host (C ABI), "
                           "pinned host buffers, per GPU",
                    "int32_index_output": {"value": queries_per_step * e2e32_steps / e2e32_s, "unit": UNIT,
                                           "d2h_bytes_per_step": int(PAIRS_PER_GPU * NPTS * K * 4),
                                           "steps": e2e32_steps,
                                           "note": "same call, idx_is_int64 = 0; not the headline (the "
                                                   "reference's knn_point returns int64)"}},
            "gpu_launches": n_launch * args.steps,
            "launches_per_step": [f"{n} x{c}" if c > 1 else n for n, c in launches],
            "launches_source": "CUPTI kernel records of one step (torch.profiler), measured in this run",
            "roofline": {"bound": "fp32", "kernel": "knn_scan_tc_kernel", "achieved": achieved,
                         "peak": fp32_tf, "unit": "TFLOP/s", "frac": achieved / fp32_tf,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "traffic_source": (f"{traffic_src}: dram__bytes_read.sum + dram__bytes_write.sum of one "
                                            "`ncu --set full` capture" if traffic else None),
                         "traffic_config": (traffic or {}).get("config"),
                         "tensor_tflops": 4.0 * achieved,  # the filter's TF32 MMAs: 2 x 16 MAC per pair
                         "note": "filter arithmetic on tcgen05 (TF32 x TF32 -> FP32 in TMEM), exact "
                                 "re-evaluation of flagged groups on the FP32 pipe",
                         "whole_step_tflops": flops_per_launch / (total_ms / args.steps * 1e-3) / 1e12
                         if world == 1 else None,
                         "whole_step_frac": flops_per_launch / (total_ms / args.steps * 1e-3) / 1e12 / fp32_tf
                         if world == 1 else None,
                         "peak_source": "FFMA/FFMA2 probe (b200pci_probe_fp32) measured in this run, "
                                        "best of 10; MEASURED_PEAKS.json has no FP32 figure",
                         "algorithmic": f"8 FLOP x {PAIRS_PER_GPU} pairs x 16384 x 16384 per launch",
                         "kernel_ms": kern_avg_ms, "kernel_share_of_step": kern_ms / sum(step_ms)},
            "clocks": clocks, "checksum": float(checksum), "parity": parity,
            "peaks": {"hbm_gbs": peaks.get("hbm_gbs"), "source": peak_src, "fp32_tflops": fp32_tf},
            "full_model": full_model, "eval64": eval64,
        }
        if world == 1:  # the CPU baseline is reported at N=1 only
            reps = 5
            threads = use_all_host_threads()
            times, kind, what = cpu_knn_baseline(reps)
            line["cpu_baseline"] = {
                "value": NPTS / min(times), "unit": UNIT, "cores": threads, "kind": kind,
                "sample": f"1 frame pair ({NPTS} queries x {NPTS} refs), best of {reps} after 1 "
                          f"warm-up; median {NPTS / statistics.median(times):.0f} q/s; torch "
                          f"{torch.__version__}; {what}"}
        if not args.no_extras and world == 1:
            line["kernels"] = extras(_lib, peaks, fp32_tf, a, b, flush)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-model", action="store_true", help="skip the full-model leg")
    ap.add_argument("--no-eval", action="store_true", help="skip the config-5 eval leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the pre-timing oracle check")
    ap.add_argument("--model-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's KNN indices to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
