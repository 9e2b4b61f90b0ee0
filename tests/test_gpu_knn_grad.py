"""The K-NN distance backward (b200pci_knn_backward, b200pci_knn_backward_det) and what is built on
it: the differentiable knn_points(...).dists, knn_points(return_nn=True) through the row gather, and
chamfer_distance's reduction options.

Through the C ABI, _det is bit for bit the sequential loop of tests/knn_grad_oracle.c (orc_knn_backward)
and so is the atomic entry point's grad_q; the atomic grad_r is within the worst-case bound of
recursive FP32 summation of FP64. Through the public API the gradients match FP64 autograd of the
torch restatement, are reproducible under torch.use_deterministic_algorithms, and the routing to
the kernels is visible in torch.profiler."""
import contextlib
from collections import Counter

import numpy as np
import pytest
import torch

from tests import grad_oracle, knn_grad_oracle

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

DIRECT_XYZ = 2
NPTS = 16384
CSR = {"scatter_hist_kernel", "scatter_scan_kernel", "scatter_fill_kernel", "scatter_sort_small_kernel",
       "scatter_sort_long_kernel"}
U = 2.0 ** -24  # unit roundoff of FP32


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
    assert g.shape == w.shape, (g.shape, w.shape)
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


def launches(fn):
    """Run ``fn`` under torch.profiler -> (its result, the library's kernel names in launch order;
    torch's own kernels and copies / fills left out)."""
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


# ------------------------------------------------------------------------------------------
# the C entry points
# ------------------------------------------------------------------------------------------
def knn(q, r, K, int64=True):
    from mocopci_b200 import pointconv_util as pcu
    return pcu._knn(K, r, q, DIRECT_XYZ, True, int64)


def knn_backward(q, r, idx, gd, det):
    """b200pci_knn_backward(_det) on (possibly strided) q [B,S,3], r [B,N,3]."""
    from mocopci_b200 import _lib
    B, S, K = idx.shape
    N = r.shape[1]
    gq = torch.full((B, S, 3), float("nan"), device="cuda")  # overwritten
    gr = torch.full((B, N, 3), float("nan"), device="cuda")
    qs, rs = q.stride(), r.stride()
    args = (B, S, N, K, q.data_ptr(), qs[0], qs[1], qs[2], r.data_ptr(), rs[0], rs[1], rs[2], idx.data_ptr(),
            1 if idx.dtype == torch.int64 else 0, gd.data_ptr(), gq.data_ptr(), gr.data_ptr())
    if det:
        ws = _lib.workspace(_lib.lib.b200pci_scatter_workspace_bytes(B, N, S * K), q.device)
        _lib.check(_lib.lib.b200pci_knn_backward_det(*args, ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
                   "knn_backward_det")
    else:
        _lib.check(_lib.lib.b200pci_knn_backward(*args, _lib.stream_ptr()), "knn_backward")
    return gq, gr


def fp64_grad_r(q, r, idx, gd):
    """FP64 grad_r and, per ref, the number of live slots and the sum of |d| over them."""
    q, r = q.astype(np.float64), r.astype(np.float64)
    B, S, K = idx.shape
    N = r.shape[1]
    live = (idx >= 0) & (idx < N) & (np.arange(K) < N)[None, None, :]
    j = np.where(live, idx, 0)
    bi = np.arange(B)[:, None, None]
    d = (2.0 * gd.astype(np.float64))[..., None] * (q[:, :, None, :] - r[bi, j])
    d = np.where(live[..., None], d, 0.0)
    flat = (bi * N + j).reshape(-1)
    gr = np.zeros((B * N, 3))
    mag = np.zeros((B * N, 3))
    cnt = np.zeros(B * N)
    np.add.at(gr, flat, -d.reshape(-1, 3))
    np.add.at(mag, flat, np.abs(d).reshape(-1, 3))
    np.add.at(cnt, flat, live.reshape(-1))
    return gr.reshape(B, N, 3), cnt.reshape(B, N, 1), mag.reshape(B, N, 3)


def check_c_abi(q, r, idx, gd, msg, q_host=None, r_host=None):
    """_det == oracle bit for bit (twice), the atomic grad_q too; the atomic grad_r within
    (n + 2) u sum|d| of FP64, n the number of terms of that ref."""
    qh = (q if q_host is None else q_host).detach().cpu().numpy()
    rh = (r if r_host is None else r_host).detach().cpu().numpy()
    ih, gh = idx.cpu().numpy(), gd.cpu().numpy()
    wq, wr = knn_grad_oracle.knn_backward(qh, rh, ih, gh)
    dq, dr = knn_backward(q, r, idx, gd, True)
    assert_bits(dq, wq, f"{msg}: det grad_q")
    assert_bits(dr, wr, f"{msg}: det grad_r")
    dq2, dr2 = knn_backward(q, r, idx, gd, True)
    assert_bits(dq2, dq, f"{msg}: det run to run")
    assert_bits(dr2, dr, f"{msg}: det run to run")
    aq, ar = knn_backward(q, r, idx, gd, False)
    assert_bits(aq, wq, f"{msg}: atomic grad_q")
    gr64, cnt, mag = fp64_grad_r(qh, rh, ih, gh)
    err = np.abs(ar.cpu().numpy().astype(np.float64) - gr64)
    tol = (cnt + 2) * U * mag
    assert (err <= tol).all(), f"{msg}: atomic grad_r off FP64 by {float((err - tol).max())} over the bound"
    return wq, wr


def lidar(B, seed=0):
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(seed, B)
    return a.cuda(), b.cuda()


@pytest.mark.parametrize("K", [1, 16, 64])
@pytest.mark.parametrize("dtype", [torch.int64, torch.int32])
def test_c_abi_vs_oracle(K, dtype):
    a, b = lidar(2, 1)
    q, r = a[:, :4096].contiguous(), b[:, :6000].contiguous()
    idx, _ = knn(q, r, K, dtype == torch.int64)
    gd = randn(idx.shape, K)
    check_c_abi(q, r, idx, gd, f"K={K} {dtype}")


def test_c_abi_k_greater_than_n_padding():
    """DIRECT_XYZ with K > N pads slots k >= N with (inf, 0): they contribute nothing, not even to ref 0."""
    from mocopci_b200 import synth
    q, r = synth.uniform_cloud(5, 3, 700).cuda(), synth.uniform_cloud(6, 3, 10).cuda()
    idx, dist = knn(q, r, 16)
    assert bool(torch.isinf(dist[..., 10:]).all()) and bool((idx[..., 10:] == 0).all())
    gd = randn(idx.shape, 7)  # non-zero on the padded slots too
    wq, wr = check_c_abi(q, r, idx, gd, "K > N")
    live_only = idx[..., :10].contiguous()
    lq, lr = knn_grad_oracle.knn_backward(q.cpu().numpy(), r.cpu().numpy(), live_only.cpu().numpy(),
                                          gd[..., :10].contiguous().cpu().numpy())
    assert_bits(wq, lq, "padding changes grad_q")
    assert_bits(wr, lr, "padding changes grad_r")


def test_c_abi_permuted_views():
    """[B,3,N] tensors passed as permuted views, as the model holds its clouds."""
    a, b = lidar(2, 3)
    q_bcn = a[:, :5000].permute(0, 2, 1).contiguous()
    r_bcn = b[:, :7000].permute(0, 2, 1).contiguous()
    q, r = q_bcn.permute(0, 2, 1), r_bcn.permute(0, 2, 1)
    assert q.stride(2) != 1 and r.stride(2) != 1
    idx, _ = knn(q, r, 16)
    check_c_abi(q, r, idx, randn(idx.shape, 8), "views", q.contiguous(), r.contiguous())


def test_c_abi_long_bucket():
    """Integer grid: ref 0 is the nearest neighbour of more than 4096 queries, so its bucket is
    rebuilt in order by the long-bucket pass of the CSR."""
    g = torch.Generator().manual_seed(9)
    grid = torch.stack(torch.meshgrid(*(torch.arange(4.0) * 10,) * 3, indexing="ij"), -1).reshape(1, 64, 3)
    r = grid.repeat(2, 1, 1).cuda()
    near = torch.randint(-3, 4, (2, 6000, 3), generator=g).float()          # around ref 0 = (0,0,0)
    far = torch.randint(0, 31, (2, 3000, 3), generator=g).float()
    q = torch.cat([near, far], 1).cuda()
    idx, _ = knn(q, r, 4)
    counts = torch.bincount(idx[0].reshape(-1), minlength=64)
    assert int(counts.max()) > 4096
    check_c_abi(q, r, idx, randn(idx.shape, 10), "long bucket")


def test_c_abi_b8_16384_k16():
    a, b = lidar(8)
    idx, _ = knn(a, b, 16)
    check_c_abi(a, b, idx, randn(idx.shape, 11), "8 x 16384^2, K=16")


# ------------------------------------------------------------------------------------------
# knn_points through autograd
# ------------------------------------------------------------------------------------------
def fp64_restatement(p1, p2, idx, w):
    """FP64 autograd of sum(w * ((p1[:, :, None] - p2[idx]) ** 2).sum(-1)) on the same idx."""
    x = p1.detach().double().cpu().requires_grad_(True)
    y = p2.detach().double().cpu().requires_grad_(True)
    bi = torch.arange(x.shape[0])[:, None, None]
    d = ((x[:, :, None] - y[bi, idx.cpu()]) ** 2).sum(-1)
    (d * w.double().cpu()).sum().backward()
    return x.grad, y.grad


def summation_bounds(p1, p2, idx, w):
    """Worst-case error of the FP32 sums against FP64, per element: (n + 2) u sum|d| for grad_p1
    (n = K terms) and grad_p2 (n = the ref's terms)."""
    q, r = p1.detach().cpu().double().numpy(), p2.detach().cpu().double().numpy()
    ih, wh = idx.cpu().numpy(), w.cpu().double().numpy()
    bi = np.arange(q.shape[0])[:, None, None]
    magq = np.abs(2.0 * wh[..., None] * (q[:, :, None, :] - r[bi, ih])).sum(2)
    _, cnt, magr = fp64_grad_r(q, r, ih, wh)
    return torch.from_numpy((ih.shape[2] + 2) * U * magq), torch.from_numpy((cnt + 2) * U * magr)


def close(got, want, tol, msg):
    err = (got.detach().cpu().double() - want).abs()
    assert bool((err <= tol + 1e-30).all()), f"{msg}: {float((err - tol).max())} over the bound"


@pytest.mark.parametrize("case", ["pair", "self", "views"])
@pytest.mark.parametrize("det", [False, True])
def test_knn_points_dists_backward_vs_fp64(case, det):
    from mocopci_b200 import chamfer
    a, b = lidar(2, 4)
    if case == "views":
        p1l = a[:, :3000].permute(0, 2, 1).contiguous().requires_grad_(True)
        p2l = b[:, :5000].permute(0, 2, 1).contiguous().requires_grad_(True)
        p1, p2 = p1l.permute(0, 2, 1), p2l.permute(0, 2, 1)
    elif case == "self":
        p1l = p2l = a[:, :5000].contiguous().requires_grad_(True)
        p1 = p2 = p1l
    else:
        p1l, p2l = a[:, :3000].contiguous().requires_grad_(True), b[:, :5000].contiguous().requires_grad_(True)
        p1, p2 = p1l, p2l
    w = randn((2, p1.shape[1], 16), 12)
    with deterministic_algorithms(det):
        out = chamfer.knn_points(p1, p2, K=16)
        assert out.dists.grad_fn is not None and out.idx.grad_fn is None
        (out.dists * w).sum().backward()
    want1, want2 = fp64_restatement(p1, p2, out.idx, w)
    tol1, tol2 = summation_bounds(p1, p2, out.idx, w)
    if case == "self":  # the two gradients are added once more in FP32
        close(p1l.grad, want1 + want2, tol1 + tol2 + 2 * U * (want1 + want2).abs(), "self-KNN")
        return
    g1, g2 = p1l.grad, p2l.grad
    if case == "views":
        g1, g2 = g1.permute(0, 2, 1), g2.permute(0, 2, 1)
    close(g1, want1, tol1, "grad p1")
    close(g2, want2, tol2, "grad p2")


def test_knn_points_deterministic_bits_and_oracle():
    """Two runs under the flag give the same bits, and those are orc_knn_backward's."""
    from mocopci_b200 import chamfer
    a, b = lidar(2, 5)
    p1, p2 = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    w = randn((2, NPTS, 16), 13)

    def run():
        p1.grad = p2.grad = None
        out = chamfer.knn_points(p1, p2, K=16)
        (out.dists * w).sum().backward()
        return out.idx, p1.grad.clone(), p2.grad.clone()
    with deterministic_algorithms(True):
        idx, g1, g2 = run()
        _, h1, h2 = run()
    assert_bits(h1, g1, "p1 run to run")
    assert_bits(h2, g2, "p2 run to run")
    wq, wr = knn_grad_oracle.knn_backward(a.cpu().numpy(), b.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy())
    assert_bits(g1, wq, "p1 vs oracle")
    assert_bits(g2, wr, "p2 vs oracle")


@pytest.mark.parametrize("det", [False, True])
def test_knn_points_backward_routing(det):
    from mocopci_b200 import chamfer
    a, b = lidar(1, 6)
    p1, p2 = a[:, :2000].clone().requires_grad_(True), b[:, :3000].clone().requires_grad_(True)
    with deterministic_algorithms(det):
        d = chamfer.knn_points(p1, p2, K=8).dists
        _, names = launches(lambda: d.backward(torch.ones_like(d)))
    if det:
        assert base(names) == CSR | {"knn_grad_q_det_kernel", "knn_grad_r_det_kernel"}, names
    else:
        assert base(names) == {"knn_backward_kernel"}, names


def test_knn_points_without_grad_is_unchanged():
    """No input requires grad (or grad is disabled): no autograd node, and the same launches as the
    plain search the function made before it was differentiable. Compared as a multiset: the search
    runs its per-query redo on a side stream beside the top-k kernel, so the two kernels start in
    either order."""
    from mocopci_b200 import chamfer, pointconv_util as pcu
    a, b = lidar(1, 7)
    _, want = launches(lambda: pcu._knn(16, b, a, DIRECT_XYZ, True))
    want = Counter(want)
    out, names = launches(lambda: chamfer.knn_points(a, b, K=16))
    assert out.dists.grad_fn is None and Counter(names) == want, (names, want)
    ref_idx, ref_d = pcu._knn(16, b, a, DIRECT_XYZ, True)
    assert torch.equal(out.idx, ref_idx) and torch.equal(bits_t(out.dists), bits_t(ref_d))
    ar = a.clone().requires_grad_(True)
    with torch.no_grad():
        out, names = launches(lambda: chamfer.knn_points(ar, b, K=16))
    assert out.dists.grad_fn is None and Counter(names) == want, (names, want)


def bits_t(t):
    return t.contiguous().view(torch.int32)


def test_knn_points_return_nn():
    """knn = p2[idx] bit for bit; its backward runs the row-gather grad kernels and allocates nothing
    of P1 x P2 size (3.2 GB per cloud at 16384^2 for a gather from an expanded p2)."""
    from mocopci_b200 import chamfer
    a, b = lidar(1, 8)
    p1, p2 = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    out = chamfer.knn_points(p1, p2, K=16, return_nn=True)
    bi = torch.arange(1, device="cuda")[:, None, None]
    assert torch.equal(bits_t(out.knn), bits_t(b[bi, out.idx]))
    g = randn(out.knn.shape, 14)
    for det, kernel in ((False, "rows_gather_grad_kernel"), (True, "rows_grad_det_kernel")):
        p2.grad = None
        with deterministic_algorithms(det):
            _, names = launches(lambda: out.knn.backward(g, retain_graph=True))
        assert kernel in base(names), names
        want = grad_oracle.index_rows_grad(g.cpu().numpy(), out.idx.cpu().numpy(), NPTS)
        if det:
            assert_bits(p2.grad, want, "return_nn backward")
        else:
            np.testing.assert_allclose(p2.grad.cpu().numpy(), want, rtol=1e-4, atol=1e-4)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - before
    assert peak < 256 << 20, f"peak {peak / 2**20:.0f} MiB"
    # small clouds: equal to pytorch3d's expanded gather too
    x, y = a[:, :300].contiguous(), b[:, :200].contiguous()
    o = chamfer.knn_points(x, y, K=5, return_nn=True)
    ref = torch.gather(y.unsqueeze(1).expand(1, 300, 200, 3), 2, o.idx.unsqueeze(-1).expand(1, 300, 5, 3))
    assert torch.equal(bits_t(o.knn), bits_t(ref))


# ------------------------------------------------------------------------------------------
# chamfer_distance
# ------------------------------------------------------------------------------------------
POINT = ["mean", "sum", "max", None]
BATCH = ["mean", "sum", None]
COMBOS = [(p, bt) for p in POINT for bt in BATCH if p is not None or bt is None]


def fp64_chamfer(x, y, dx, dy, ix, iy, weights, batch_reduction, point_reduction, single):
    """The contract of chamfer_distance's docstring in FP64: per-point terms from the oracle's nearest
    neighbours (their values checked against its FP32 minima), differentiable in x and y."""
    B = x.shape[0]
    bi = torch.arange(B)[:, None]
    tx = ((x - y[bi, torch.as_tensor(ix).long()]) ** 2).sum(-1)
    ty = ((y - x[bi, torch.as_tensor(iy).long()]) ** 2).sum(-1)
    np.testing.assert_allclose(tx.detach().numpy(), dx, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(ty.detach().numpy(), dy, rtol=1e-5, atol=1e-7)

    def reduce(t, P):
        if weights is not None:
            t = t * weights.view(B, 1)
        if point_reduction == "max":
            t = t.max(1).values
        elif point_reduction is not None:
            t = t.sum(1)
            if point_reduction == "mean":
                t = t / P
        if point_reduction is not None and batch_reduction is not None:
            t = t.sum()
            if batch_reduction == "mean":
                t = t / (weights.sum() if weights is not None else B)
        return t
    cx = reduce(tx, x.shape[1])
    if single:
        return cx
    cy = reduce(ty, y.shape[1])
    if point_reduction == "max":
        return torch.maximum(cx, cy)
    if point_reduction is not None:
        return cx + cy
    return cx, cy


@pytest.mark.parametrize("single", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("point_reduction,batch_reduction", COMBOS)
def test_chamfer_distance_options_vs_fp64(orc, point_reduction, batch_reduction, weighted, single):
    from mocopci_b200 import chamfer, synth
    B = 3
    x = synth.uniform_cloud(21, B, 400)
    y = synth.uniform_cloud(22, B, 250)
    wts = torch.tensor([0.5, 2.0, 1.25]) if weighted else None
    _, dx, dy, ix, iy = orc.chamfer(x.numpy(), y.numpy())
    xd, yd = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
    loss, normals = chamfer.chamfer_distance(xd, yd, weights=None if wts is None else wts.cuda(),
                                             batch_reduction=batch_reduction, point_reduction=point_reduction,
                                             single_directional=single)
    x64, y64 = x.double().requires_grad_(True), y.double().requires_grad_(True)
    want = fp64_chamfer(x64, y64, dx, dy, ix, iy, None if wts is None else wts.double(), batch_reduction,
                        point_reduction, single)
    if point_reduction is None and not single:
        assert normals == (None, None) and isinstance(loss, tuple)
        got_t, want_t = loss, want
    else:
        assert normals is None and isinstance(loss, torch.Tensor)
        got_t, want_t = (loss,), (want,)
    for g_, w_ in zip(got_t, want_t):
        assert g_.shape == w_.shape, (g_.shape, w_.shape)
        # FP32 sums of up to 400 positive terms: n u is 2.4e-5
        np.testing.assert_allclose(g_.detach().cpu().double().numpy(), w_.detach().numpy(), rtol=3e-5, atol=0)
    seed = torch.Generator().manual_seed(23)
    cots = [torch.rand(w_.shape, generator=seed, dtype=torch.float64) + 0.5 for w_ in want_t]
    torch.autograd.backward(list(got_t), [c.float().cuda() for c in cots])
    torch.autograd.backward(list(want_t), cots)
    for got, want_g in ((xd.grad, x64.grad), (yd.grad, y64.grad)):
        np.testing.assert_allclose(got.cpu().double().numpy(), want_g.numpy(), rtol=1e-4,
                                   atol=1e-5 * float(want_g.abs().max()))


@pytest.mark.parametrize("point_reduction,batch_reduction", COMBOS)
def test_chamfer_distance_all_zero_weights(point_reduction, batch_reduction):
    from mocopci_b200 import chamfer, synth
    x = synth.uniform_cloud(31, 2, 100).cuda().requires_grad_(True)
    y = synth.uniform_cloud(32, 2, 80).cuda().requires_grad_(True)
    loss, _ = chamfer.chamfer_distance(x, y, weights=torch.zeros(2, device="cuda"),
                                       batch_reduction=batch_reduction, point_reduction=point_reduction)
    want_shape = {None: (2, 100)}.get(point_reduction, () if batch_reduction is not None else (2,))
    parts = loss if isinstance(loss, tuple) else (loss,)
    assert parts[0].shape == want_shape
    for p in parts:
        assert bool((p == 0).all()) and p.requires_grad
    torch.autograd.backward(list(parts), [torch.ones_like(p) for p in parts])
    for t in (x, y):
        assert t.grad is not None and bool((t.grad == 0).all())


def test_chamfer_distance_defaults_unchanged():
    """Default arguments launch the fused Chamfer kernels (forward and backward) and give the loss
    b200pci_chamfer_forward computes, bit for bit; no K-NN backward is involved."""
    from mocopci_b200 import _lib, chamfer
    a, b = lidar(2, 9)
    x, y = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    (loss, normals), names = launches(lambda: chamfer.chamfer_distance(x, y))
    assert normals is None
    assert {"chamfer_reduce_kernel", "chamfer_final_kernel"} <= base(names), names
    _, bnames = launches(lambda: loss.backward())
    assert base(bnames) == {"chamfer_backward_kernel"}, bnames
    L = _lib.lib
    B, N, M = 2, NPTS, NPTS
    dxo, dyo = torch.empty((B, N), device="cuda"), torch.empty((B, M), device="cuda")
    ixo = torch.empty((B, N), dtype=torch.int32, device="cuda")
    iyo = torch.empty((B, M), dtype=torch.int32, device="cuda")
    lo = torch.empty((1,), device="cuda")
    ws = _lib.workspace(L.b200pci_chamfer_workspace_bytes(B, N, M), a.device)
    _lib.check(L.b200pci_chamfer_forward(B, N, M, a.data_ptr(), N * 3, 3, 1, b.data_ptr(), M * 3, 3, 1,
                                         dxo.data_ptr(), ixo.data_ptr(), dyo.data_ptr(), iyo.data_ptr(),
                                         lo.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "chamfer")
    assert_bits(loss.reshape(1), lo, "default loss")
    # abs_cosine has no effect without normals: still the fused path
    _, names2 = launches(lambda: chamfer.chamfer_distance(a, b, abs_cosine=False))
    assert "knn_backward_kernel" not in base(names2) and "chamfer_final_kernel" in base(names2)
