"""The deterministic gradients (b200pci_*_grad_det, b200pci_chamfer_backward_det) under
torch.use_deterministic_algorithms(True): bit for bit equal to sequential C loops (the oracle's
orc_*_grad in oracle/oracle.c; tests/grad_oracle.c for the row gathers and Chamfer), through the
C ABI and through the public autograd entry points; the same bits on two runs; routed to the new
kernels only when the flag is set; and a small differentiable pipeline built from the public API
gives the same loss and leaf gradients twice."""
import contextlib
import ctypes
import types

import numpy as np
import pytest
import torch

from tests import grad_oracle

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

NPTS = 16384
OLD = {"group_grad_kernel", "three_interpolate_grad_kernel", "rows_gather_grad_kernel", "chamfer_backward_kernel"}
CSR = {"scatter_hist_kernel", "scatter_scan_kernel", "scatter_fill_kernel", "scatter_sort_small_kernel",
       "scatter_sort_long_kernel"}


@contextlib.contextmanager
def deterministic_algorithms(enabled, warn_only=False):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(enabled, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


@pytest.fixture
def det():
    """torch.use_deterministic_algorithms(True) for one test, the previous setting restored after."""
    with deterministic_algorithms(True):
        yield


def bits(a):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def assert_bits(got, want, msg=""):
    g, w = bits(got), bits(want)
    assert g.shape == w.shape, (g.shape, w.shape)
    bad = int((g != w).sum())
    assert bad == 0, f"{msg}: {bad} of {g.size} entries differ"


def kernel_name(raw):
    """'void b200pci::fps_cluster_kernel<4, true, 8, 512>(int, ...)' -> 'fps_cluster_kernel<4, true, 8, 512>'."""
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


def launches(fn):
    """Run ``fn`` once under torch.profiler (CUPTI sees every kernel of the process, the library's
    included) -> (what fn returned, names of the library's kernels it launched, template arguments
    kept; torch's own kernels, e.g. the fill of an output, are left out)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [kernel_name(e.name) for e in prof.events()
             if "cuda" in str(getattr(e, "device_type", "")).lower()]
    return out, [n for n in names if not n.startswith(("at::", "Memcpy", "Memset"))]


def base(names):
    return {n.split("<")[0] for n in names}


def randn(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)).cuda()


def twice(fn):
    """fn() run twice: the second result must carry the same bits -> the first."""
    a = fn()
    b = fn()
    for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32)), "run-to-run difference"
    return a


# ------------------------------------------------------------------------------------------
# the C entry points
# ------------------------------------------------------------------------------------------
def L():
    from mocopci_b200 import _lib
    return _lib


def group_grad_det(grad_out, idx, N, init=None):
    """b200pci_group_points_grad_det (idx [B,P,S]) or b200pci_gather_points_grad_det (idx [B,P])."""
    lib = L()
    B, C = grad_out.shape[:2]
    gp = torch.zeros((B, C, N), device="cuda") if init is None else init.clone()
    T = idx[0].numel()
    ws = lib.workspace(lib.lib.b200pci_scatter_workspace_bytes(B, N, T), gp.device)
    if idx.dim() == 3:
        rc = lib.lib.b200pci_group_points_grad_det(B, C, N, idx.shape[1], idx.shape[2], grad_out.data_ptr(),
                                                   idx.data_ptr(), gp.data_ptr(), ws.data_ptr(), ws.numel(),
                                                   lib.stream_ptr())
    else:
        rc = lib.lib.b200pci_gather_points_grad_det(B, C, N, idx.shape[1], grad_out.data_ptr(), idx.data_ptr(),
                                                    gp.data_ptr(), ws.data_ptr(), ws.numel(), lib.stream_ptr())
    lib.check(rc, "group_grad_det")
    return gp


def interp_grad_det(grad_out, idx, weight, m):
    lib = L()
    B, C, n = grad_out.shape
    gp = torch.zeros((B, C, m), device="cuda")
    ws = lib.workspace(lib.lib.b200pci_scatter_workspace_bytes(B, m, 3 * n), gp.device)
    lib.check(lib.lib.b200pci_three_interpolate_grad_det(
        B, C, n, m, grad_out.data_ptr(), idx.data_ptr(), weight.data_ptr(), gp.data_ptr(), ws.data_ptr(),
        ws.numel(), lib.stream_ptr()), "three_interpolate_grad_det")
    return gp


def rows_grad_det(grad_out, idx, N):
    lib = L()
    B, C = grad_out.shape[0], grad_out.shape[-1]
    T = idx[0].numel()
    gp = torch.zeros((B, N, C), device="cuda")
    ws = lib.workspace(lib.lib.b200pci_scatter_workspace_bytes(B, N, T), gp.device)
    lib.check(lib.lib.b200pci_index_points_rows_grad_det(
        B, N, T, C, grad_out.data_ptr(), idx.data_ptr(), 1 if idx.dtype == torch.int64 else 0, gp.data_ptr(),
        ws.data_ptr(), ws.numel(), lib.stream_ptr()), "index_points_rows_grad_det")
    return gp


def chamfer_backward_det(x, y, ix, iy, g=1.0):
    lib = L()
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    gx, gy = torch.empty((B, N, 3), device="cuda"), torch.empty((B, M, 3), device="cuda")
    gl = torch.tensor([g], dtype=torch.float32, device="cuda")
    ws = lib.workspace(lib.lib.b200pci_chamfer_backward_det_workspace_bytes(B, N, M), x.device)
    lib.check(lib.lib.b200pci_chamfer_backward_det(
        B, N, M, x.data_ptr(), y.data_ptr(), ix.data_ptr(), iy.data_ptr(), gl.data_ptr(), gx.data_ptr(),
        gy.data_ptr(), ws.data_ptr(), ws.numel(), lib.stream_ptr()), "chamfer_backward_det")
    return gx, gy


def chamfer_indices(x, y):
    """The NN indices b200pci_chamfer_forward computes (idx_x [B,N], idx_y [B,M], int32)."""
    lib = L()
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    dx, dy = torch.empty((B, N), device="cuda"), torch.empty((B, M), device="cuda")
    ix = torch.empty((B, N), dtype=torch.int32, device="cuda")
    iy = torch.empty((B, M), dtype=torch.int32, device="cuda")
    loss = torch.empty((1,), device="cuda")
    ws = lib.workspace(lib.lib.b200pci_chamfer_workspace_bytes(B, N, M), x.device)
    xs, ys = x.stride(), y.stride()
    lib.check(lib.lib.b200pci_chamfer_forward(
        B, N, M, x.data_ptr(), xs[0], xs[1], xs[2], y.data_ptr(), ys[0], ys[1], ys[2], dx.data_ptr(),
        ix.data_ptr(), dy.data_ptr(), iy.data_ptr(), loss.data_ptr(), ws.data_ptr(), ws.numel(),
        lib.stream_ptr()), "chamfer_forward")
    return ix, iy


def orc_group_grad_into(orc, grad_out, idx, init):
    """orc_group_grad accumulating into a given (pre-filled) buffer."""
    g = np.ascontiguousarray(grad_out.cpu().numpy(), dtype=np.float32)
    i = np.ascontiguousarray(idx.cpu().numpy(), dtype=np.int32)
    out = np.ascontiguousarray(init.cpu().numpy(), dtype=np.float32).copy()
    B, C, N = out.shape
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    orc.lib().orc_group_grad(B, C, N, i.shape[1], i.shape[2], p(g), p(i), p(out))
    return out


# ------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pairs8():
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(0, 8)
    return types.SimpleNamespace(a=a, b=b, ad=a.cuda(), bd=b.cuda())


@pytest.fixture(scope="module")
def config2(pairs8):
    """bench.py's config 2 at B = 8: 4096 FPS centres, ball query r = 0.5, ns = 32."""
    from mocopci_b200 import ops as p2u, pointconv_util as pcu
    fidx = p2u.furthest_point_sample(pairs8.ad, 4096)
    centres = pcu.index_points_gather(pairs8.ad, fidx)
    idx = p2u.ball_query(0.5, 32, pairs8.ad, centres)
    return types.SimpleNamespace(fidx=fidx, idx=idx)


PYRAMID = [(256, 64), (1024, 256), (4096, 1024), (16384, 4096)]  # (unknown n, known m), config 3


# ------------------------------------------------------------------------------------------
# gather / group
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [128, 3])
def test_group_grad_config2_vs_oracle(orc, det, config2, C):
    from mocopci_b200 import ops as p2u
    idx = config2.idx
    gout = randn((8, C, 4096, 32), 100 + C)
    want = orc.group_grad(gout.cpu().numpy(), idx.cpu().numpy(), NPTS)
    assert_bits(twice(lambda: group_grad_det(gout, idx, NPTS)), want, "C ABI")
    feats = randn((8, C, NPTS), C).requires_grad_(True)

    def autograd():
        feats.grad = None
        p2u.grouping_operation(feats, idx).backward(gout)
        return feats.grad.clone()
    assert_bits(twice(autograd), want, "grouping_operation backward")


def test_gather_grad_config2_vs_oracle(orc, det, config2):
    from mocopci_b200 import ops as p2u
    gout = randn((8, 128, 4096), 7)
    want = orc.gather_grad(gout.cpu().numpy(), config2.fidx.cpu().numpy(), NPTS)
    assert_bits(twice(lambda: group_grad_det(gout, config2.fidx, NPTS)), want, "C ABI")
    feats = randn((8, 128, NPTS), 8).requires_grad_(True)

    def autograd():
        feats.grad = None
        p2u.gather_operation(feats, config2.fidx).backward(gout)
        return feats.grad.clone()
    assert_bits(twice(autograd), want, "gather_operation backward")


def test_group_grad_accumulates_into_prefilled_output(orc, det, config2):
    gout = randn((8, 16, 4096, 32), 11)
    init = randn((8, 16, NPTS), 12)
    want = orc_group_grad_into(orc, gout, config2.idx, init)
    assert_bits(twice(lambda: group_grad_det(gout, config2.idx, NPTS, init)), want)


def test_group_grad_odd_sizes_and_single_destination(orc, det):
    """T not a multiple of 4 (37 x 5), N = 1 (one bucket holds every position)."""
    g = torch.Generator().manual_seed(21)
    idx = torch.randint(0, 100, (3, 37, 5), generator=g, dtype=torch.int32).cuda()
    gout = randn((3, 11, 37, 5), 22)
    want = orc.group_grad(gout.cpu().numpy(), idx.cpu().numpy(), 100)
    assert_bits(twice(lambda: group_grad_det(gout, idx, 100)), want, "T = 185")
    idx1 = torch.zeros((2, 1000, 3), dtype=torch.int32, device="cuda")
    gout1 = randn((2, 5, 1000, 3), 23)
    want1 = orc.group_grad(gout1.cpu().numpy(), idx1.cpu().numpy(), 1)
    assert_bits(twice(lambda: group_grad_det(gout1, idx1, 1)), want1, "N = 1")


def test_group_grad_all_one_index(orc, det):
    """Every position points at the same destination: one bucket of all T = 131072 entries (the
    bucket is rebuilt in order by a scan of idx) at config 2's shape."""
    idx = torch.full((8, 4096, 32), 4321, dtype=torch.int32, device="cuda")
    gout = randn((8, 16, 4096, 32), 31)
    want = orc.group_grad(gout.cpu().numpy(), idx.cpu().numpy(), NPTS)
    assert_bits(twice(lambda: group_grad_det(gout, idx, NPTS)), want)


# ------------------------------------------------------------------------------------------
# three_interpolate
# ------------------------------------------------------------------------------------------
def test_three_interpolate_grad_pyramid_vs_oracle(orc, det, pairs8):
    from mocopci_b200 import ops as p2u
    for n, m in PYRAMID:
        w, idx, _ = p2u.three_nn_weights(pairs8.ad[:, :n].contiguous(), pairs8.ad[:, :m].contiguous())
        gout = randn((8, 128, n), n)
        want = orc.three_interpolate_grad(gout.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy(), m)
        assert_bits(twice(lambda: interp_grad_det(gout, idx, w, m)), want, f"{m}->{n} C ABI")
        f = randn((8, 128, m), m).requires_grad_(True)

        def autograd():
            f.grad = None
            p2u.three_interpolate(f, idx, w).backward(gout)
            return f.grad.clone()
        assert_bits(twice(autograd), want, f"{m}->{n} three_interpolate backward")


def test_three_interpolate_grad_fewer_than_three_known(orc, det):
    """m = 2: three_nn pads the third slot with index 0, so index 0 appears twice in a row."""
    from mocopci_b200 import ops as p2u, synth
    unknown, known = synth.uniform_cloud(5, 2, 300).cuda(), synth.uniform_cloud(6, 2, 2).cuda()
    w, idx, _ = p2u.three_nn_weights(unknown, known)
    assert bool((idx[..., 2] == 0).all())
    gout = randn((2, 9, 300), 41)
    want = orc.three_interpolate_grad(gout.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy(), 2)
    assert_bits(twice(lambda: interp_grad_det(gout, idx, w, 2)), want)


# ------------------------------------------------------------------------------------------
# [B,N,C] rows
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.int64, torch.int32])
def test_rows_grad_knn_shape_vs_oracle(orc, det, pairs8, dtype):
    """index_points_group_C64_k16: [8,16384,64] features gathered with knn_point(16, a, b)."""
    from mocopci_b200 import pointconv_util as pcu
    kidx = pcu.knn_point(16, pairs8.ad, pairs8.bd).to(dtype)
    gout = randn((8, NPTS, 16, 64), 51)
    want = grad_oracle.index_rows_grad(gout.cpu().numpy(), kidx.cpu().numpy(), NPTS)
    assert_bits(twice(lambda: rows_grad_det(gout, kidx, NPTS)), want, "C ABI")
    f = randn((8, NPTS, 64), 52).requires_grad_(True)

    def autograd():
        f.grad = None
        pcu.index_points_group(f, kidx).backward(gout)
        return f.grad.clone()
    assert_bits(twice(autograd), want, "index_points_group backward")


def test_rows_grad_group_query_autograd(orc, det):
    """group_query with autograd: the support cloud and its features get their gradients through
    the row-gather backward."""
    from mocopci_b200 import pointconv_util as pcu, synth
    s_xyz = synth.uniform_cloud(61, 2, 2048).cuda().requires_grad_(True)
    s_pts = randn((2, 2048, 32), 62).requires_grad_(True)
    q = synth.uniform_cloud(63, 2, 512).cuda()
    r = randn((2, 512, 16, 35), 64)

    def autograd():
        s_xyz.grad = s_pts.grad = None
        new_points, _ = pcu.group_query(16, s_xyz, q, s_pts)
        (new_points * r).sum().backward()
        return s_xyz.grad.clone(), s_pts.grad.clone()
    gx, gp = twice(autograd)
    idx = pcu.knn_point(16, s_xyz.detach(), q).cpu().numpy()
    rn = r.cpu().numpy()
    assert_bits(gx, grad_oracle.index_rows_grad(rn[..., :3], idx, 2048), "xyz")
    assert_bits(gp, grad_oracle.index_rows_grad(rn[..., 3:], idx, 2048), "features")


# ------------------------------------------------------------------------------------------
# Chamfer
# ------------------------------------------------------------------------------------------
def chamfer_inputs(case):
    from mocopci_b200 import synth
    if case == "lidar_B8":        # bench.py chamfer_B8
        return synth.frame_pairs(0, 8)
    if case == "lidar_B2_bcn_views":
        return synth.frame_pairs(1, 2)
    if case == "lidar_N_ne_M":
        a, b = synth.frame_pairs(2, 2)
        return a, b[:, :5000].contiguous()
    if case == "tie_stress":      # integer grid, half the points duplicated
        return synth.tie_stress_cloud(11, 2, 9000, grid=6), synth.tie_stress_cloud(12, 2, 7000, grid=6)
    raise ValueError(case)


@pytest.mark.parametrize("case", ["lidar_B8", "lidar_N_ne_M", "lidar_B2_bcn_views", "tie_stress"])
def test_chamfer_backward_vs_oracle(orc, det, case):
    from mocopci_b200 import chamfer
    x, y = chamfer_inputs(case)
    B = x.shape[0]
    xd, yd = x.cuda(), y.cuda()
    ix, iy = chamfer_indices(xd, yd)
    wx, wy = grad_oracle.chamfer_backward(x.numpy(), y.numpy(), ix.cpu().numpy(), iy.cpu().numpy(), 1.0)
    gx, gy = twice(lambda: chamfer_backward_det(xd, yd, ix, iy))
    assert_bits(gx, wx, "C ABI grad_x")
    assert_bits(gy, wy, "C ABI grad_y")
    if case == "lidar_B2_bcn_views":  # chamfer_loss(pc1, pc2) permutes [B,3,N] tensors
        x_leaf = x.permute(0, 2, 1).contiguous().cuda().requires_grad_(True)
        y_leaf = y.permute(0, 2, 1).contiguous().cuda().requires_grad_(True)
        views = lambda: (x_leaf.permute(0, 2, 1), y_leaf.permute(0, 2, 1))  # noqa: E731
    else:
        x_leaf, y_leaf = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
        views = lambda: (x_leaf, y_leaf)  # noqa: E731

    def autograd():
        x_leaf.grad = y_leaf.grad = None
        chamfer.chamfer_distance(*views())[0].backward()
        return x_leaf.grad.clone(), y_leaf.grad.clone()
    ax, ay = twice(autograd)
    if case == "lidar_B2_bcn_views":
        ax, ay = ax.permute(0, 2, 1), ay.permute(0, 2, 1)
    assert_bits(ax, wx, "chamfer_distance backward, x")
    assert_bits(ay, wy, "chamfer_distance backward, y")
    # and within the existing 1e-4 of FP64 autograd through the same indices
    xt, yt = x.double().requires_grad_(True), y.double().requires_grad_(True)
    bi = torch.arange(B)[:, None]
    ixt, iyt = ix.cpu().long(), iy.cpu().long()
    ref = ((xt - yt[bi, ixt]) ** 2).sum(-1).mean(-1) + ((yt - xt[bi, iyt]) ** 2).sum(-1).mean(-1)
    ref.mean().backward()
    np.testing.assert_allclose(ax.cpu().numpy(), xt.grad.float().numpy(), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(ay.cpu().numpy(), yt.grad.float().numpy(), rtol=1e-4, atol=1e-7)


# ------------------------------------------------------------------------------------------
# EMD's backward has no atomics: reproducible as it is
# ------------------------------------------------------------------------------------------
def test_emd_matchcost_backward_is_reproducible(det):
    from mocopci_b200 import emd_cuda, synth
    x1, x2 = synth.uniform_cloud(71, 2, 1024).cuda(), synth.uniform_cloud(72, 2, 1500).cuda()
    match = emd_cuda.approxmatch_forward(x1, x2)
    gc = torch.ones(2, device="cuda")
    twice(lambda: tuple(emd_cuda.matchcost_backward(gc, x1, x2, match)))


# ------------------------------------------------------------------------------------------
# routing
# ------------------------------------------------------------------------------------------
def backward_of(op):
    """-> a function running the backward of one public op on small inputs."""
    from mocopci_b200 import chamfer, ops as p2u, pointconv_util as pcu, synth
    if op == "group":
        f = randn((2, 8, 500), 81).requires_grad_(True)
        idx = torch.randint(0, 500, (2, 64, 8), generator=torch.Generator().manual_seed(82), dtype=torch.int32).cuda()
        out = p2u.grouping_operation(f, idx)
    elif op == "three_interpolate":
        f = randn((2, 8, 100), 83).requires_grad_(True)
        w, idx, _ = p2u.three_nn_weights(synth.uniform_cloud(84, 2, 400).cuda(), synth.uniform_cloud(85, 2, 100).cuda())
        out = p2u.three_interpolate(f, idx, w)
    elif op == "rows":
        f = randn((2, 500, 16), 86).requires_grad_(True)
        idx = torch.randint(0, 500, (2, 64, 8), generator=torch.Generator().manual_seed(87)).cuda()
        out = pcu.index_points_group(f, idx)
    else:
        x = synth.uniform_cloud(88, 2, 300).cuda().requires_grad_(True)
        out = chamfer.chamfer_distance(x, synth.uniform_cloud(89, 2, 200).cuda())[0]
    g = torch.ones_like(out)
    return lambda: out.backward(g)


NEW_KERNEL = {"group": "group_grad_det_kernel", "three_interpolate": "three_interpolate_grad_det_kernel",
              "rows": "rows_grad_det_kernel", "chamfer": "chamfer_grad_det_kernel"}
OLD_KERNEL = {"group": "group_grad_kernel", "three_interpolate": "three_interpolate_grad_kernel",
              "rows": "rows_gather_grad_kernel", "chamfer": "chamfer_backward_kernel"}


@pytest.mark.parametrize("op", ["group", "three_interpolate", "rows", "chamfer"])
@pytest.mark.parametrize("mode", ["deterministic", "warn_only", "off"])
def test_backward_routing(op, mode):
    with deterministic_algorithms(mode != "off", warn_only=mode == "warn_only"):
        _, names = launches(backward_of(op))
    if mode == "off":
        assert base(names) == {OLD_KERNEL[op]}, names
    else:
        assert not base(names) & OLD, names
        assert base(names) == CSR | {NEW_KERNEL[op]}, names


# ------------------------------------------------------------------------------------------
# end to end
# ------------------------------------------------------------------------------------------
def pipeline():
    """FPS -> query_and_group (features and cloud require grad) -> per-channel scaling and a mean
    pool -> three_interpolate back up -> Chamfer against a target, plus a feature term. Public API
    only, no matmul. -> (loss, gradients of every leaf)."""
    from mocopci_b200 import chamfer, ops as p2u, synth
    xyz = synth.uniform_cloud(91, 2, 4096).cuda().requires_grad_(True)
    target = synth.uniform_cloud(92, 2, 3000).cuda()
    feats = randn((2, 16, 4096), 93).requires_grad_(True)
    scale = randn((19,), 94).requires_grad_(True)
    fidx = p2u.furthest_point_sample(xyz.detach(), 512)
    centres = p2u.gather_operation(xyz.transpose(1, 2), fidx).transpose(1, 2)  # [2,512,3], differentiable
    grouped = p2u.query_and_group(0.3, 16, xyz, centres, feats)                # [2,19,512,16]
    pooled = (grouped * scale.view(1, -1, 1, 1)).mean(-1)                       # [2,19,512]
    w, idx, _ = p2u.three_nn_weights(xyz.detach(), centres.detach().contiguous())
    up = p2u.three_interpolate(pooled, idx, w)                                  # [2,19,4096]
    pred = xyz + 0.01 * up[:, :3].transpose(1, 2)
    loss = chamfer.chamfer_distance(pred, target)[0] + up[:, 3:].pow(2).mean()
    loss.backward()
    return loss.detach(), xyz.grad, feats.grad, scale.grad


def test_end_to_end_pipeline_is_bitwise_reproducible(det):
    first, second = pipeline(), pipeline()
    for name, a, b in zip(("loss", "xyz", "feats", "scale"), first, second):
        assert a is not None and bool(torch.isfinite(a).all()), name
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{name} differs between runs"
    assert float(first[2].abs().sum()) > 0 and float(first[1].abs().sum()) > 0
