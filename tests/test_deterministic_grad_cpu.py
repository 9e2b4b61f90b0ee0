"""CPU tests of the deterministic-gradient entry points (b200pci_*_grad_det, b200pci_chamfer_backward_det):
scratch sizes, argument errors and empty problems are decided on the host, without a device; and
the two sequential restatements the GPU tests compare with (tests/grad_oracle.c) agree with FP64
references."""
import numpy as np
import pytest
import torch

from tests import grad_oracle


@pytest.fixture(scope="module")
def lib():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import _lib
    return _lib


def test_scatter_workspace_sizes(lib):
    L = lib.lib
    ws = L.b200pci_scatter_workspace_bytes
    # offsets [B,N+1], cursors [B,N], source list [B,T] (int32) and the long-bucket list [B,N] (int64)
    assert ws(8, 16384, 4096 * 32) >= 8 * (16384 * 4 + 16385 * 4 + 4096 * 32 * 4 + 16384 * 8)
    assert ws(1, 1, 1) > 0
    assert ws(-1, 10, 10) == 0 and ws(1, -1, 10) == 0 and ws(1, 10, -1) == 0
    cw = L.b200pci_chamfer_backward_det_workspace_bytes
    assert cw(2, 100, 300) == ws(2, 100, 300) + ws(2, 300, 100)
    assert cw(-1, 1, 1) == 0


def test_det_entry_points_argument_handling_without_gpu(lib):
    L = lib.lib
    P = 16  # a dummy non-null "device" pointer: every call below must fail before touching it
    # empty problems: nothing to do
    assert L.b200pci_gather_points_grad_det(0, 3, 10, 4, None, None, None, None, 0, None) == 0
    assert L.b200pci_group_points_grad_det(1, 3, 10, 4, 0, None, None, None, None, 0, None) == 0
    assert L.b200pci_three_interpolate_grad_det(1, 0, 10, 5, None, None, None, None, None, 0, None) == 0
    assert L.b200pci_index_points_rows_grad_det(1, 10, 0, 4, None, None, 1, None, None, 0, None) == 0
    assert L.b200pci_chamfer_backward_det(0, 10, 10, None, None, None, None, None, None, None, None, 0, None) == 0
    # negative sizes
    assert L.b200pci_gather_points_grad_det(1, -3, 10, 4, None, None, None, None, 0, None) == -1
    assert b"negative size" in L.b200pci_last_error()
    assert L.b200pci_group_points_grad_det(1, 3, 10, -4, 2, None, None, None, None, 0, None) == -1
    assert L.b200pci_three_interpolate_grad_det(1, 3, -10, 5, None, None, None, None, None, 0, None) == -1
    assert L.b200pci_index_points_rows_grad_det(1, 10, -5, 4, None, None, 1, None, None, 0, None) == -1
    assert L.b200pci_chamfer_backward_det(1, -10, 10, None, None, None, None, None, None, None, None, 0, None) == -1
    # null pointers
    assert L.b200pci_gather_points_grad_det(1, 3, 10, 4, None, None, None, None, 0, None) == -1
    assert b"null pointer" in L.b200pci_last_error()
    assert L.b200pci_group_points_grad_det(1, 3, 10, 4, 2, P, None, P, P, 1 << 20, None) == -1
    assert L.b200pci_three_interpolate_grad_det(1, 3, 10, 5, P, P, None, P, P, 1 << 20, None) == -1
    assert L.b200pci_index_points_rows_grad_det(1, 10, 5, 4, P, None, 1, P, P, 1 << 20, None) == -1
    assert L.b200pci_chamfer_backward_det(1, 10, 10, P, P, P, None, P, P, P, P, 1 << 20, None) == -1
    assert b"null pointer" in L.b200pci_last_error()
    # 2^31 or more source positions per cloud
    assert L.b200pci_group_points_grad_det(1, 3, 10, 1 << 16, 1 << 15, P, P, P, P, 1 << 40, None) == -1
    assert b"2^31" in L.b200pci_last_error()
    assert L.b200pci_three_interpolate_grad_det(1, 3, 1 << 30, 5, P, P, P, P, P, 1 << 40, None) == -1
    assert L.b200pci_index_points_rows_grad_det(1, 10, 1 << 31, 4, P, P, 1, P, P, 1 << 40, None) == -1
    # the grid limits of the atomic twins
    assert L.b200pci_gather_points_grad_det(70000, 3, 10, 4, P, P, P, P, 1 << 40, None) == -1
    assert L.b200pci_index_points_rows_grad_det(70000, 10, 5, 4, P, P, 1, P, P, 1 << 40, None) == -1
    # missing or short scratch -> EWORKSPACE
    need = L.b200pci_scatter_workspace_bytes(2, 10, 4 * 3)
    assert L.b200pci_group_points_grad_det(2, 3, 10, 4, 3, P, P, P, None, need, None) == -3
    assert L.b200pci_group_points_grad_det(2, 3, 10, 4, 3, P, P, P, P, need - 1, None) == -3
    assert b"workspace" in L.b200pci_last_error()
    assert L.b200pci_gather_points_grad_det(2, 3, 10, 4, P, P, P, P, 0, None) == -3
    assert L.b200pci_three_interpolate_grad_det(2, 3, 4, 10, P, P, P, P, P,
                                                L.b200pci_scatter_workspace_bytes(2, 10, 12) - 1, None) == -3
    assert L.b200pci_index_points_rows_grad_det(2, 10, 5, 4, P, P, 0, P, None, 0, None) == -3
    cneed = L.b200pci_chamfer_backward_det_workspace_bytes(2, 10, 7)
    assert L.b200pci_chamfer_backward_det(2, 10, 7, P, P, P, P, P, P, P, P, cneed - 1, None) == -3
    with pytest.raises(RuntimeError, match="workspace"):
        lib.check(L.b200pci_chamfer_backward_det(2, 10, 7, P, P, P, P, P, P, P, None, 0, None),
                  "chamfer_backward_det")


def test_ops_keep_their_signatures_under_the_deterministic_flag(lib):
    """The routing is inside the wrappers: the reference's names and arguments are unchanged."""
    import inspect
    from mocopci_b200 import pointnet2_cuda
    assert list(inspect.signature(pointnet2_cuda.group_points_grad_wrapper).parameters) == [
        "b", "c", "n", "npoints", "nsample", "grad_out_tensor", "idx_tensor", "grad_points_tensor"]
    assert list(inspect.signature(pointnet2_cuda.three_interpolate_grad_wrapper).parameters) == [
        "b", "c", "n", "m", "grad_out_tensor", "idx_tensor", "weight_tensor", "grad_points_tensor"]


def test_oracle_chamfer_backward_matches_fp64_autograd(orc):
    rng = np.random.default_rng(5)
    x = rng.random((2, 300, 3), dtype=np.float32)
    y = rng.random((2, 170, 3), dtype=np.float32)
    _, _, _, ix, iy = orc.chamfer(x, y)
    gx, gy = grad_oracle.chamfer_backward(x, y, ix, iy, 1.0)
    xt = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    yt = torch.tensor(y, dtype=torch.float64, requires_grad=True)
    bi = torch.arange(2)[:, None]
    ref = (((xt - yt[bi, torch.as_tensor(ix).long()]) ** 2).sum(-1).mean(-1)
           + ((yt - xt[bi, torch.as_tensor(iy).long()]) ** 2).sum(-1).mean(-1))
    ref.mean().backward()
    np.testing.assert_allclose(gx, xt.grad.numpy(), rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(gy, yt.grad.numpy(), rtol=1e-5, atol=1e-9)


def test_oracle_index_rows_grad_is_a_sequential_scatter(orc):
    rng = np.random.default_rng(6)
    g = rng.standard_normal((2, 40, 7), dtype=np.float32)
    idx = rng.integers(-2, 12, (2, 40))  # out-of-range entries are skipped
    got = grad_oracle.index_rows_grad(g, idx, 10)
    want = np.zeros((2, 10, 7), np.float32)
    for b in range(2):
        for t in range(40):
            if 0 <= idx[b, t] < 10:
                want[b, idx[b, t]] += g[b, t]
    np.testing.assert_array_equal(got.view(np.int32), want.view(np.int32))
