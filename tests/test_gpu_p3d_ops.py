"""pytorch3d's ball_query and sample_farthest_points on the B200 kernels (mocopci_b200.p3d_ops):
idx and dists bit for bit against the sequential restatement of tests/p3d_oracle.c, at the
benchmark's config-2 shape (8 frames of 16384 points, 4096 FPS centres, r = 0.5) and on ragged,
strided and tie-stress inputs; the ball-query distance gradient bit for bit against
orc_knn_backward under torch.use_deterministic_algorithms and within the FP32 summation bound
otherwise; routing and the absence of device-to-host copies in torch.profiler; CUDA-graph replay
with device-side lengths."""
import contextlib

import numpy as np
import pytest
import torch

from tests import knn_grad_oracle, p3d_oracle

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

U = 2.0 ** -24  # unit roundoff of FP32
FPS_KERNEL = "fps_p3d_cluster_kernel"
BQ_KERNEL = "ball_query_p3d_kernel"


@contextlib.contextmanager
def deterministic_algorithms(enabled):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(enabled)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


def bits(a):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def assert_bits(got, want, msg=""):
    g, w = bits(got), bits(want)
    assert g.shape == w.shape, (msg, g.shape, w.shape)
    bad = int((g != w).sum())
    assert bad == 0, f"{msg}: {bad} of {g.size} entries differ"


def kernel_name(raw):
    name = raw[5:] if raw.startswith("void ") else raw
    name = name.replace("(anonymous namespace)::", "").replace("b200pci::", "")
    depth = 0
    for i, ch in enumerate(name):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            return name[:i]
    return name


@pytest.fixture(scope="module")
def ops():
    from mocopci_b200 import p3d_ops
    return p3d_ops


@pytest.fixture(scope="module")
def frames():
    """bench.py's config 2: the 8 frames a of the first pairs and their 4096 pointnet2 FPS centres."""
    from mocopci_b200 import ops as p2u, pointconv_util as pcu, synth
    a, _ = synth.frame_pairs(0, 8)
    ad = a.cuda()
    centres = pcu.index_points_gather(ad, p2u.furthest_point_sample(ad, 4096))
    return ad, centres


def nn_want(p2, idx):
    """p2[b, idx] with zeros for -1, on the CPU."""
    p2, idx = p2.detach().cpu(), idx.cpu()
    B, P1, K = idx.shape
    g = torch.gather(p2, 1, idx.clamp_min(0).reshape(B, -1, 1).expand(-1, -1, 3)).reshape(B, P1, K, 3)
    return torch.where((idx >= 0)[..., None], g, torch.zeros(()))


def check_bq(ops, p1, p2, K, radius, l1=None, l2=None, msg=""):
    res = ops.ball_query(p1, p2, lengths1=l1, lengths2=l2, K=K, radius=radius)
    wi, wd = p3d_oracle.ball_query(p1.cpu().numpy(), p2.cpu().numpy(), K, radius,
                                   None if l1 is None else l1.cpu().numpy(), None if l2 is None else l2.cpu().numpy())
    np.testing.assert_array_equal(res.idx.cpu().numpy(), wi, err_msg=f"{msg}: idx")
    assert_bits(res.dists, wd, f"{msg}: dists")
    assert torch.equal(res.knn.cpu(), nn_want(p2, res.idx)), f"{msg}: knn"
    return res


# ------------------------------------------------------------------------------------------
# ball_query
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [32, 500])
def test_ball_query_config2_vs_oracle(ops, frames, K):
    a, centres = frames
    res = check_bq(ops, centres, a, K, 0.5, msg=f"config 2, K={K}")
    assert int((res.idx >= 0).sum(-1).min()) >= 1  # every centre finds itself


def test_ball_query_ragged_views_and_ties(ops):
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(3, 4, 6000)
    p1, p2 = b[:, :900].cuda(), a.cuda()
    l1 = torch.tensor([900, 0, 1, 517], device="cuda")
    l2 = torch.tensor([6000, 3000, 0, 1], device="cuda")
    check_bq(ops, p1, p2, 64, 1.5, l1, l2, "ragged")
    check_bq(ops, p1, p2, 64, 1.5, l1, None, "ragged p1 only")
    out_of_range = torch.tensor([-5, 7000, 6000, 2], device="cuda")  # clamped to [0, P]
    check_bq(ops, p1, p2, 16, 1.5, out_of_range.clamp(max=900), out_of_range, "clamped")
    # K > P2, every ref inside the ball
    small = p2[:, :20].contiguous()
    res = check_bq(ops, p1, small, 50, 1e4, l1, None, "K > P2")
    assert bool((res.idx[0, :, 20:] == -1).all()) and bool((res.idx[0, :, :20] >= 0).all())
    # strided [B, 3, N] views, as the model holds its clouds
    p1t, p2t = p1.transpose(1, 2).contiguous().transpose(1, 2), p2.transpose(1, 2).contiguous().transpose(1, 2)
    assert p1t.stride(2) != 1
    check_bq(ops, p1t, p2t, 64, 1.5, l1, l2, "views")
    # tie stress: integer grid, duplicated points; radius^2 = 4 is itself a distance (strict <)
    t1, t2 = synth.tie_stress_cloud(11, 3, 2000, grid=6).cuda(), synth.tie_stress_cloud(12, 3, 7000, grid=6).cuda()
    for radius in (2.0, 3.5):
        check_bq(ops, t1, t2, 500, radius, torch.tensor([2000, 1500, 1], device="cuda"),
                 torch.tensor([7000, 6999, 1], device="cuda"), f"tie stress r={radius}")


def test_ball_query_return_nn_false(ops, frames):
    a, centres = frames
    res = ops.ball_query(centres[:2], a[:2], K=16, radius=0.5, return_nn=False)
    assert res.knn is None
    want = ops.ball_query(centres[:2], a[:2], K=16, radius=0.5)
    assert torch.equal(res.idx, want.idx) and torch.equal(res.dists, want.dists)


def fp64_grad_p2(q, r, idx, gd):
    """FP64 grad_p2 of sum(gd * d2) and, per ref, the number of live slots and the sum of |d|."""
    q, r = q.astype(np.float64), r.astype(np.float64)
    B, S, K = idx.shape
    N = r.shape[1]
    live = idx >= 0
    j = np.where(live, idx, 0)
    bi = np.arange(B)[:, None, None]
    d = (2.0 * gd.astype(np.float64))[..., None] * (q[:, :, None, :] - r[bi, j])
    d = np.where(live[..., None], d, 0.0)
    flat = (bi * N + j).reshape(-1)
    gr, mag, cnt = np.zeros((B * N, 3)), np.zeros((B * N, 3)), np.zeros(B * N)
    np.add.at(gr, flat, -d.reshape(-1, 3))
    np.add.at(mag, flat, np.abs(d).reshape(-1, 3))
    np.add.at(cnt, flat, live.reshape(-1))
    return gr.reshape(B, N, 3), cnt.reshape(B, N, 1), mag.reshape(B, N, 3)


@pytest.mark.parametrize("case", ["config2_K500", "ragged_views"])
def test_ball_query_dists_backward(ops, frames, case):
    if case == "config2_K500":
        a, centres = frames
        p1, p2, K, radius, l1, l2 = centres, a, 500, 0.5, None, None
    else:
        from mocopci_b200 import synth
        a, b = synth.frame_pairs(5, 3, 5000)
        p1 = b[:, :800].cuda().transpose(1, 2).contiguous().transpose(1, 2)
        p2 = a.cuda()
        K, radius = 40, 1.0
        l1, l2 = torch.tensor([800, 0, 300], device="cuda"), torch.tensor([5000, 2000, 1], device="cuda")
    y = p2.detach().clone().requires_grad_(True)
    if case == "ragged_views":  # x is [B, 3, N]; the op sees the permuted view
        x = p1.detach().transpose(1, 2).contiguous().requires_grad_(True)
        xv = x.transpose(1, 2)
    else:
        x = xv = p1.detach().clone().requires_grad_(True)
    with deterministic_algorithms(True):
        res = ops.ball_query(xv, y, l1, l2, K=K, radius=radius, return_nn=False)
        g = torch.randn(res.dists.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(K))
        gx, gy = torch.autograd.grad(res.dists, (x, y), g)
        gx2, gy2 = torch.autograd.grad(ops.ball_query(xv, y, l1, l2, K=K, radius=radius, return_nn=False).dists,
                                       (x, y), g)
    gxv = gx.transpose(1, 2) if case == "ragged_views" else gx
    qh, rh = p1.detach().cpu().numpy(), p2.detach().cpu().numpy()
    ih, gh = res.idx.cpu().numpy(), g.cpu().numpy()
    wq, wr = knn_grad_oracle.knn_backward(qh, rh, ih, gh)
    assert_bits(gxv, wq, f"{case}: det grad_p1")
    assert_bits(gy, wr, f"{case}: det grad_p2")
    assert_bits(gx2, gx, f"{case}: det run to run")
    assert_bits(gy2, gy, f"{case}: det run to run")
    with deterministic_algorithms(False):
        res = ops.ball_query(xv, y, l1, l2, K=K, radius=radius, return_nn=False)
        ax, ay = torch.autograd.grad(res.dists, (x, y), g)
    axv = ax.transpose(1, 2) if case == "ragged_views" else ax
    assert_bits(axv, wq, f"{case}: atomic grad_p1")
    gr64, cnt, mag = fp64_grad_p2(qh, rh, ih, gh)
    err = np.abs(ay.cpu().numpy().astype(np.float64) - gr64)
    tol = (cnt + 2) * U * mag
    assert (err <= tol).all(), f"{case}: atomic grad_p2 off FP64 by {float((err - tol).max())} over the bound"


def test_ball_query_nn_backward(ops):
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(6, 2, 3000)
    x, y = b[:, :500].cuda().requires_grad_(True), a.cuda().requires_grad_(True)
    l2 = torch.tensor([3000, 100], device="cuda")
    res = ops.ball_query(x, y, None, l2, K=24, radius=1.0)
    w = torch.randn(res.knn.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    gd = torch.randn(res.dists.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    gx, gy = torch.autograd.grad((res.knn * w).sum() + (res.dists * gd).sum(), (x, y))
    # FP64 restatement: dists term as above plus w scattered into the rows idx points at
    idx = res.idx.cpu().numpy()
    gr64, cnt, mag = fp64_grad_p2(x.detach().cpu().numpy(), y.detach().cpu().numpy(), idx, gd.cpu().numpy())
    live = idx >= 0
    flat = (np.arange(2)[:, None, None] * 3000 + np.where(live, idx, 0)).reshape(-1)
    wn = np.where(live[..., None], w.cpu().numpy().astype(np.float64), 0.0).reshape(-1, 3)
    gw = np.zeros((2 * 3000, 3))
    np.add.at(gw, flat, wn)
    aw = np.zeros((2 * 3000, 3))
    np.add.at(aw, flat, np.abs(wn))
    cw = np.zeros((2 * 3000, 1))
    np.add.at(cw, flat, live.reshape(-1, 1).astype(np.float64))
    want = gr64 + gw.reshape(2, 3000, 3)
    tol = (cnt + cw.reshape(2, 3000, 1) + 3) * U * (mag + aw.reshape(2, 3000, 3))
    err = np.abs(gy.cpu().numpy().astype(np.float64) - want)
    assert (err <= tol).all(), float((err - tol).max())
    assert bool((gy[1, 100:] == 0).all())  # refs beyond lengths2 receive nothing


# ------------------------------------------------------------------------------------------
# sample_farthest_points
# ------------------------------------------------------------------------------------------
def check_fps(ops, pts, K, lengths=None, msg="", out=None):
    sel, idx = out if out is not None else ops.sample_farthest_points(pts, lengths=lengths, K=K)
    Kh = K.cpu().numpy() if isinstance(K, torch.Tensor) else K
    want = p3d_oracle.fps(pts.cpu().numpy(), Kh, None if lengths is None else lengths.cpu().numpy())
    np.testing.assert_array_equal(idx.cpu().numpy(), want, err_msg=msg)
    assert torch.equal(sel.cpu(), nn_want(pts, idx[:, :, None])[:, :, 0]), f"{msg}: selected_points"
    return sel, idx


def test_fps_config2_vs_oracle(ops, frames):
    a, _ = frames
    check_fps(ops, a, 4096, msg="8 x 16384 -> 4096")


def test_fps_ragged_tensor_k_and_ties(ops):
    from mocopci_b200 import synth
    pts = synth.frame_pairs(2, 4, 5000)[0].cuda()
    lengths = torch.tensor([5000, 0, 1, 2345], device="cuda")
    check_fps(ops, pts, 300, lengths, "ragged")
    check_fps(ops, pts, torch.tensor([300, 7, 5, 1]), lengths, "(B,) K on the CPU")
    check_fps(ops, pts, torch.tensor([10, 20, 30, 3000], device="cuda"), lengths, "(B,) K on the GPU")
    check_fps(ops, pts.transpose(1, 2).contiguous().transpose(1, 2), 200, lengths, "views")
    check_fps(ops, pts[:, :50], 80, None, "K > P")
    # ties: the furthest distance is shared by many points; lowest index first
    tie = synth.tie_stress_cloud(17, 3, 16384, grid=3).cuda()
    check_fps(ops, tie, 1024, torch.tensor([16384, 9000, 343], device="cuda"), "tie stress")
    # beyond the shared-memory mirror (more than 200 KB per cloud)
    big = synth.uniform_cloud(9, 2, 40000).cuda()
    check_fps(ops, big, 256, torch.tensor([40000, 39999], device="cuda"), "40000 points")


def test_fps_random_start_point(ops):
    from mocopci_b200 import synth
    pts = synth.frame_pairs(1, 3, 3000)[0].cuda()
    lengths = torch.tensor([3000, 10, 2000], device="cuda")
    torch.manual_seed(123)
    _, idx = ops.sample_farthest_points(pts, lengths, K=64, random_start_point=True)
    torch.manual_seed(123)
    start = [int(torch.randint(high=n, size=(1,)).item()) for n in (3000, 10, 2000)]
    want = p3d_oracle.fps(pts.cpu().numpy(), 64, lengths.cpu().numpy(), start)
    np.testing.assert_array_equal(idx.cpu().numpy(), want)
    assert idx[:, 0].tolist() == start


def test_fps_selected_points_backward(ops):
    from mocopci_b200 import synth
    pts = synth.frame_pairs(4, 2, 2000)[0].cuda().requires_grad_(True)
    lengths = torch.tensor([2000, 30], device="cuda")
    sel, idx = ops.sample_farthest_points(pts, lengths, K=50)
    assert idx.grad_fn is None or not idx.requires_grad
    w = torch.randn(sel.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    (g,) = torch.autograd.grad((sel * w).sum(), pts)
    want = torch.zeros(2, 2000, 3)
    ih, wh = idx.cpu(), w.cpu()
    for b in range(2):
        for t in range(50):
            if ih[b, t] >= 0:
                want[b, ih[b, t]] += wh[b, t]  # FPS picks are distinct here: one term per row
    assert torch.equal(g.cpu(), want)


# ------------------------------------------------------------------------------------------
# routing, host synchronisation, CUDA graphs
# ------------------------------------------------------------------------------------------
_PROFILE_SCRIPT = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
from mocopci_b200 import ops as p2u, p3d_ops as ops, pointconv_util as pcu, synth
a = synth.frame_pairs(0, 8)[0].cuda()
centres = pcu.index_points_gather(a, p2u.furthest_point_sample(a, 4096))
l2 = torch.tensor([16384, 9000] * 4, device="cuda")
x = centres.detach().clone().requires_grad_(True)
calls = {
    "ball_query": lambda: ops.ball_query(centres, a, None, l2, K=32, radius=0.5),
    "fps": lambda: ops.sample_farthest_points(a, l2, K=512),
    "fps_config2": lambda: ops.sample_farthest_points(a, K=4096),
    "grad": lambda: torch.autograd.grad(ops.ball_query(x, a, K=32, radius=0.5).dists.sum(), x),
}
out = {}
for name, fn in calls.items():
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out[name] = [e.name for e in prof.events() if "cuda" in str(getattr(e, "device_type", "")).lower()]
print(json.dumps(out))
"""


def test_profiler_kernels_and_no_device_to_host_copy():
    """The new kernels run, and neither op copies anything to the host. Profiled in a fresh process:
    after the profiler sessions of other test files in the same pytest process, the kernel records
    of these calls have come back empty."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _PROFILE_SCRIPT, root], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    raw = json.loads(res.stdout.strip().splitlines()[-1])
    names = {k: [kernel_name(n) for n in v] for k, v in raw.items()}
    to_host = ("DtoH", "Device -> Pageable", "Device -> Pinned")
    assert BQ_KERNEL in names["ball_query"], names["ball_query"]
    assert [n for n in names["fps"] if n.startswith(FPS_KERNEL)], names["fps"]
    assert FPS_KERNEL + "<4, true>" in names["fps_config2"], names["fps_config2"]
    for k in ("ball_query", "fps", "fps_config2"):
        assert not [n for n in names[k] if any(t in n for t in to_host)], (k, names[k])
    # with grad: forward and backward run the library's kernels
    assert BQ_KERNEL in names["grad"] and "knn_backward_kernel<long long>" in names["grad"], names["grad"]


def test_cuda_graph_replay_with_device_lengths(ops, frames):
    a, centres = frames
    p1, p2 = centres[:4].clone(), a[:4].clone()
    l1 = torch.tensor([4096, 4096, 100, 0], device="cuda")
    l2 = torch.tensor([16384, 5000, 16384, 16384], device="cuda")
    lf = torch.tensor([16384, 3000, 1, 0], device="cuda")
    eager = lambda: (ops.ball_query(p1, p2, l1, l2, K=32, radius=0.5), ops.sample_farthest_points(p2, lf, K=256))  # noqa: E731
    want = eager()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager()  # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = eager()
    g.replay()
    torch.cuda.synchronize()
    for got, ref in ((out[0].idx, want[0].idx), (out[0].dists, want[0].dists), (out[0].knn, want[0].knn),
                     (out[1][0], want[1][0]), (out[1][1], want[1][1])):
        assert torch.equal(got, ref)
    # new lengths in the captured buffers: the replay follows them
    l1.copy_(torch.tensor([10, 4096, 4096, 1], device="cuda"))
    l2.copy_(torch.tensor([16384, 16384, 2, 7000], device="cuda"))
    lf.copy_(torch.tensor([5, 16384, 9000, 200], device="cuda"))
    g.replay()
    torch.cuda.synchronize()
    want2 = eager()
    assert not torch.equal(want2[0].idx, want[0].idx) and not torch.equal(want2[1][1], want[1][1])
    for got, ref in ((out[0].idx, want2[0].idx), (out[0].dists, want2[0].dists), (out[0].knn, want2[0].knn),
                     (out[1][0], want2[1][0]), (out[1][1], want2[1][1])):
        assert torch.equal(got, ref)
    wi, _ = p3d_oracle.ball_query(p1.cpu().numpy(), p2.cpu().numpy(), 32, 0.5, l1.cpu().numpy(), l2.cpu().numpy())
    np.testing.assert_array_equal(out[0].idx.cpu().numpy(), wi)
    np.testing.assert_array_equal(out[1][1].cpu().numpy(), p3d_oracle.fps(p2.cpu().numpy(), 256, lf.cpu().numpy()))
