"""CPU tests of the K-NN distance backward (b200pci_knn_backward, b200pci_knn_backward_det): argument
errors, missing scratch and empty problems are decided on the host, without a device; the sequential
restatement the GPU tests compare with (tests/knn_grad_oracle.c, orc_knn_backward) agrees with FP64
autograd; and chamfer_distance rejects the arguments it does not implement before touching a GPU."""
import numpy as np
import pytest
import torch

from tests import knn_grad_oracle


@pytest.fixture(scope="module")
def lib():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import _lib
    return _lib


def call(L, name, B, S, N, K, q=None, r=None, idx=None, gd=None, gq=None, gr=None, ws=None, wsb=0):
    """One call of b200pci_knn_backward(_det) with [B,S,3] / [B,N,3] contiguous strides."""
    args = (B, S, N, K, q, S * 3, 3, 1, r, N * 3, 3, 1, idx, 1, gd, gq, gr)
    if name == "det":
        return L.b200pci_knn_backward_det(*args, ws, wsb, None)
    return L.b200pci_knn_backward(*args, None)


@pytest.mark.parametrize("name", ["atomic", "det"])
def test_knn_backward_argument_handling_without_gpu(lib, name):
    L = lib.lib
    P = 16  # a dummy non-null "device" pointer: every call below must return before touching it
    full = dict(q=P, r=P, idx=P, gd=P, gq=P, gr=P, ws=P, wsb=1 << 40)
    # empty problems: nothing to write
    assert call(L, name, 0, 10, 10, 4) == 0
    assert call(L, name, 3, 0, 0, 4) == 0
    # negative sizes
    for sizes in ((-1, 10, 10, 4), (1, -10, 10, 4), (1, 10, -10, 4), (1, 10, 10, -4)):
        assert call(L, name, *sizes, **full) == -1, sizes
        assert b"negative size" in L.b200pci_last_error()
    # null pointers
    for miss in ("q", "r", "idx", "gd", "gq", "gr"):
        assert call(L, name, 2, 10, 10, 4, **dict(full, **{miss: None})) == -1, miss
        assert b"null pointer" in L.b200pci_last_error()
    # the grid limit on B and 2^31 or more slots per cloud
    assert call(L, name, 70000, 10, 10, 4, **full) == -1
    assert b"batch" in L.b200pci_last_error()
    assert call(L, name, 1, 1 << 26, 10, 32, **full) == -1
    assert b"2^31" in L.b200pci_last_error()


def test_knn_backward_det_scratch_without_gpu(lib):
    L = lib.lib
    P = 16
    need = L.b200pci_scatter_workspace_bytes(2, 10, 7 * 4)
    base = dict(q=P, r=P, idx=P, gd=P, gq=P, gr=P)
    assert call(L, "det", 2, 7, 10, 4, **base, ws=None, wsb=need) == -3
    assert call(L, "det", 2, 7, 10, 4, **base, ws=P, wsb=need - 1) == -3
    assert b"workspace" in L.b200pci_last_error()
    assert call(L, "det", 2, 7, 10, 4, **base, ws=P, wsb=0) == -3
    with pytest.raises(RuntimeError, match="workspace"):
        lib.check(call(L, "det", 2, 7, 10, 4, **base), "knn_backward_det")


def fp64_knn_grad(q, r, idx, gd):
    """FP64 autograd of sum(gd * |q_i - r_idx|^2) over the live slots (k < N, 0 <= idx < N)."""
    B, S, K = idx.shape
    N = r.shape[1]
    qt = torch.tensor(q, dtype=torch.float64, requires_grad=True)
    rt = torch.tensor(r, dtype=torch.float64, requires_grad=True)
    it = torch.as_tensor(idx).long()
    live = (it >= 0) & (it < N) & (torch.arange(K) < N)[None, None, :]
    bi = torch.arange(B)[:, None, None]
    d = ((qt[:, :, None] - rt[bi, it.clamp(0, max(N - 1, 0))]) ** 2).sum(-1)
    (d * torch.as_tensor(gd, dtype=torch.float64) * live).sum().backward()
    return qt.grad.numpy(), rt.grad.numpy()


@pytest.mark.parametrize("K", [1, 5, 16])
def test_oracle_knn_backward_matches_fp64_autograd(K):
    rng = np.random.default_rng(K)
    q = rng.random((2, 200, 3), dtype=np.float32)
    r = rng.random((2, 90, 3), dtype=np.float32)
    idx = rng.integers(0, 90, (2, 200, K))
    gd = rng.standard_normal((2, 200, K), dtype=np.float32)
    gq, gr = knn_grad_oracle.knn_backward(q, r, idx, gd)
    wq, wr = fp64_knn_grad(q, r, idx, gd)
    np.testing.assert_allclose(gq, wq, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(gr, wr, rtol=1e-5, atol=1e-5)


def test_oracle_knn_backward_skips_padding_and_out_of_range():
    """K > N: slots k >= N are the (inf, 0) padding and add nothing; nor do indices outside [0, N)."""
    rng = np.random.default_rng(3)
    q = rng.random((1, 30, 3), dtype=np.float32)
    r = rng.random((1, 4, 3), dtype=np.float32)
    idx = rng.integers(-2, 6, (1, 30, 7))
    gd = rng.standard_normal((1, 30, 7), dtype=np.float32)
    gq, gr = knn_grad_oracle.knn_backward(q, r, idx, gd)
    wq, wr = fp64_knn_grad(q, r, idx, gd)
    np.testing.assert_allclose(gq, wq, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(gr, wr, rtol=1e-5, atol=1e-5)
    # the order of the contract: grad_q over k ascending, grad_r over the flat slot ascending
    wq32 = np.zeros_like(gq)
    wr32 = np.zeros_like(gr)
    for i in range(30):
        for k in range(4):
            j = idx[0, i, k]
            if 0 <= j < 4:
                d = np.float32(2 * gd[0, i, k]) * (q[0, i] - r[0, j])
                wq32[0, i] += d
                wr32[0, j] -= d
    np.testing.assert_array_equal(gq.view(np.int32), wq32.view(np.int32))
    np.testing.assert_array_equal(gr.view(np.int32), wr32.view(np.int32))


# ------------------------------------------------------------------------------------------
# chamfer_distance's argument checks run before any kernel (CPU tensors are never reached)
# ------------------------------------------------------------------------------------------
def cpu_clouds():
    g = torch.Generator().manual_seed(0)
    return torch.rand((2, 10, 3), generator=g), torch.rand((2, 7, 3), generator=g)


@pytest.mark.parametrize("kw", [
    dict(batch_reduction="median"), dict(point_reduction="min"), dict(point_reduction="none"),
    dict(point_reduction=None), dict(point_reduction=None, batch_reduction="sum"),
    dict(weights=torch.ones(3)), dict(weights=torch.ones(2, 1)), dict(weights=torch.tensor([1.0, -0.5])),
])
def test_chamfer_distance_value_errors(lib, kw):
    from mocopci_b200 import chamfer
    x, y = cpu_clouds()
    with pytest.raises(ValueError):
        chamfer.chamfer_distance(x, y, **kw)


@pytest.mark.parametrize("kw", [
    dict(x_lengths=torch.tensor([10, 9])), dict(y_lengths=torch.tensor([7, 7])),
    dict(x_normals=torch.zeros(2, 10, 3)), dict(y_normals=torch.zeros(2, 7, 3)), dict(norm=1),
    dict(norm=1, point_reduction="sum"), dict(unknown_option=True),
])
def test_chamfer_distance_not_implemented(lib, kw):
    from mocopci_b200 import chamfer
    x, y = cpu_clouds()
    with pytest.raises(NotImplementedError):
        chamfer.chamfer_distance(x, y, **kw)


def test_knn_points_not_implemented(lib):
    from mocopci_b200 import chamfer
    x, y = cpu_clouds()
    with pytest.raises(NotImplementedError):
        chamfer.knn_points(x, y, lengths1=torch.tensor([10, 10]))
    with pytest.raises(NotImplementedError):
        chamfer.knn_points(x, y, norm=1)
