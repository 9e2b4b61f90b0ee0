"""CPU checks of the float64 EMD restatement (tests/emd_reference.py) before the GPU tests trust it:
it agrees with the C oracle (oracle/oracle.c, the reference's FP32 algorithm with libm expf), keeps
the mass invariants of the algorithm, and reproduces the reference's known answer. Also the C ABI's
batch limit of the EMD cost and gradient entry points, checked without a device."""
import numpy as np
import pytest
import torch

from tests import emd_reference as R


def clouds(B, n, m, scale=0.5, offset=0.0, seed=0):
    """Seeded (B, n, 3) / (B, m, 3) float32 clouds, uniform in [-scale, scale]^3 + offset."""
    from mocopci_b200 import synth
    x1 = synth.uniform_cloud(seed + n, B, n) * scale + offset
    x2 = synth.uniform_cloud(seed + m + 3, B, m) * scale + offset
    return x1, x2


# Entries of match against another arithmetic's: 3e-3 absolute everywhere, 1e-2 relative on entries
# above 0.1. Smaller entries are ill-conditioned: on the 4096-point LiDAR pair the C oracle (FP32,
# libm expf) is 8.5% from FP64 on some entry above 1e-3, and FP64 itself moves by up to 18% there
# when every exp is perturbed by 2e-7 relative. Above 0.1, FP32 results were measured within 3.4e-3.
MATCH_ATOL, MATCH_RTOL, MATCH_RTOL_ABOVE = 3e-3, 1e-2, 0.1


def check_match(got, want):
    """-> (largest absolute gap, largest relative gap on entries of ``want`` above 0.1)."""
    got = torch.as_tensor(got).double()
    want = torch.as_tensor(want).double().to(got.device)
    err = (got - want).abs()
    big = want > MATCH_RTOL_ABOVE
    worst_abs = float(err.max()) if err.numel() else 0.0
    worst_rel = float((err[big] / want[big]).max()) if big.any() else 0.0
    assert worst_abs <= MATCH_ATOL and worst_rel <= MATCH_RTOL, (worst_abs, worst_rel)
    return worst_abs, worst_rel


def check_mass(match, n, m, line_rtol, saturated_rtol, total_rtol):
    """Invariants of ApproxMatch's output (B, m, n), whatever its arithmetic: match >= 0 and finite;
    a point of xyz1 gives at most multiL, one of xyz2 receives at most multiR; the total is
    min(n multiL, m multiR); the side with less mass is used up (its last level has exp = 1).
    Returns the largest deviations seen, relative to the bound each is checked against."""
    match = torch.as_tensor(match).double()
    multiL, multiR = R.multipliers(n, m)
    assert torch.isfinite(match).all() and (match >= 0).all()
    rows, cols = match.sum(1), match.sum(2)          # per xyz1 point (B, n), per xyz2 point (B, m)
    assert (rows <= multiL * (1 + line_rtol)).all(), float(rows.max())
    assert (cols <= multiR * (1 + line_rtol)).all(), float(cols.max())
    total = min(n * multiL, m * multiR)
    tot_dev = float(((match.sum((1, 2)) - total).abs() / total).max())
    assert tot_dev <= total_rtol, tot_dev
    sat_dev = 0.0
    if n * multiL <= m * multiR:
        sat_dev = max(sat_dev, float(((rows - multiL).abs() / multiL).max()))
    if m * multiR <= n * multiL:
        sat_dev = max(sat_dev, float(((cols - multiR).abs() / multiR).max()))
    assert sat_dev <= saturated_rtol, sat_dev
    return {"total": tot_dev, "saturated": sat_dev}


# (B, n, m, scale, offset): tile-free shapes the oracle runs in seconds; multipliers 1 and 3 on either
# side, single-point clouds, and a small cloud 1000 m from the origin
SHAPES = [(2, 128, 128, 0.5, 0.0), (1, 300, 1000, 0.5, 0.0), (1, 1000, 300, 0.5, 0.0),
          (1, 1000, 1000, 5.0, 0.0), (3, 65, 17, 0.5, 0.0), (1, 33, 1, 0.5, 0.0), (1, 1, 33, 0.5, 0.0),
          (1, 640, 640, 0.05, 1000.0)]


@pytest.mark.parametrize("B,n,m,scale,offset", SHAPES)
def test_reference_vs_oracle(orc, B, n, m, scale, offset):
    """FP64 restatement against the FP32 oracle: cost to 1e-5 relative (the FP32 algorithm was
    measured within 1.8e-6 of FP64 up to 4100 points), match by check_match, both the streaming
    cost and the closed form on the stored match."""
    x1, x2 = clouds(B, n, m, scale, offset)
    om = orc.emd_approxmatch(x1.numpy(), x2.numpy())
    oc = orc.emd_matchcost(x1.numpy(), x2.numpy(), om).astype(np.float64)
    match = R.approxmatch64(x1, x2)
    c_stream, c_closed = R.cost64(x1, x2).numpy(), R.matchcost64(x1, x2, match).numpy()
    np.testing.assert_allclose(c_stream, c_closed, rtol=1e-12)
    np.testing.assert_allclose(c_stream, oc, rtol=1e-5)
    check_match(om, match)
    # the oracle's matchcost on its own match is the closed form to FP32 summation error
    np.testing.assert_allclose(R.matchcost64(x1, x2, torch.from_numpy(om)).numpy(), oc, rtol=1e-5)
    check_mass(match, n, m, 1e-9, 1e-7, 1e-9)
    check_mass(om, n, m, 1e-5, 1e-4, 1e-5)      # the bounds the GPU tests use for FP32 results


def test_reference_block_size_does_not_matter():
    """cost64 and approxmatch64 give the same answer whatever the row block (a block edge that
    dropped or repeated a row would show)."""
    x1, x2 = clouds(2, 150, 70)
    np.testing.assert_allclose(R.cost64(x1, x2, block=16).numpy(), R.cost64(x1, x2, block=1000).numpy(),
                               rtol=1e-13)
    np.testing.assert_allclose(R.approxmatch64(x1, x2, block=7).numpy(),
                               R.approxmatch64(x1, x2, block=4096).numpy(), rtol=1e-12, atol=1e-15)


def test_reference_grad_closed_form():
    """matchcost_grad64 is the autograd gradient of grad_cost . matchcost64 with match held fixed."""
    x1, x2 = clouds(2, 40, 90)
    match = R.approxmatch64(x1, x2)
    g = torch.tensor([0.7, -1.9], dtype=torch.float64)
    p1, p2 = x1.double().requires_grad_(True), x2.double().requires_grad_(True)
    cost = (((p2[:, :, None, :] - p1[:, None, :, :]) ** 2).sum(-1) * match).sum((1, 2))
    np.testing.assert_allclose(cost.detach().numpy(), R.matchcost64(x1, x2, match).numpy(), rtol=1e-13)
    (cost * g).sum().backward()
    g1, g2 = R.matchcost_grad64(g, x1, x2, match)
    np.testing.assert_allclose(g1.numpy(), p1.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(g2.numpy(), p2.grad.numpy(), rtol=1e-10, atol=1e-12)


def test_reference_known_answer():
    """models/EMD/test_emd_loss.py:7-43: each point matched to the other cloud's far point, cost 0.71
    per pair, weighted loss 2.0116667 and its gradients."""
    p1 = torch.tensor([[[1.7, -0.1, 0.1], [0.1, 1.2, 0.3]]]).repeat(3, 1, 1)
    p2 = torch.tensor([[[0.3, 1.8, 0.2], [1.2, -0.2, 0.3]]]).repeat(3, 1, 1)
    match = R.approxmatch64(p1, p2)
    np.testing.assert_allclose(match.numpy(), np.array([[[0, 1], [1, 0]]] * 3), atol=1e-9)
    cost = R.cost64(p1, p2)
    np.testing.assert_allclose(cost.numpy(), 0.71, rtol=1e-6)
    w = torch.tensor([0.5, 2.0, 1 / 3], dtype=torch.float64)
    assert abs(float((cost * w).sum()) - 2.0116667) <= 1e-6 * 2.0116667
    g1, g2 = R.matchcost_grad64(w, p1, p2, match)
    np.testing.assert_allclose(g1[0].numpy(), [[0.5, 0.1, -0.2], [-0.2, -0.6, 0.1]], atol=1e-6)
    np.testing.assert_allclose(g2[0].numpy(), [[0.2, 0.6, -0.1], [-0.5, -0.1, 0.2]], atol=1e-6)
    np.testing.assert_allclose(g1[1].numpy(), 4 * g1[0].numpy(), rtol=1e-12)


def test_reference_empty_clouds():
    for n, m in ((0, 5), (5, 0), (0, 0)):
        x1, x2 = torch.zeros(2, n, 3), torch.zeros(2, m, 3)
        assert R.approxmatch64(x1, x2).shape == (2, m, n)
        assert R.cost64(x1, x2).tolist() == [0.0, 0.0]


@pytest.fixture(scope="module")
def lib():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import _lib
    return _lib


def test_emd_cost_and_grad_reject_batches_over_grid_limit(lib):
    """One grid row per pair: B > 65535 is EINVAL before anything reaches a device. Host buffers of
    the right sizes stand in for the device pointers; they are never read."""
    L, B = lib.lib, 70000
    buf = np.zeros(B * 3 * 4, np.float32)
    ws = np.zeros(L.b200pci_emd_workspace_bytes(B, 1, 1), np.uint8)
    p, w = buf.ctypes.data, ws.ctypes.data
    assert L.b200pci_emd_matchcost(B, 1, 1, p, p, p, p, w, ws.size, None) == -1
    assert b"batch too large" in L.b200pci_last_error()
    assert L.b200pci_emd_matchcost_grad(B, 1, 1, p, p, p, p, p, p, None) == -1
    assert b"batch too large" in L.b200pci_last_error()
    assert L.b200pci_emd_approxmatch(B, 1, 1, p, p, p, w, ws.size, None) == -1
    assert L.b200pci_emd_cost(B, 1, 1, p, p, p, w, ws.size, None) == -1
    assert L.b200pci_emd_matchcost(0, 1, 1, p, p, p, p, w, ws.size, None) == 0    # empty batch
    assert L.b200pci_emd_matchcost_grad(0, 1, 1, p, p, p, p, p, p, None) == 0
    # an empty cloud needs no gradient buffer of its own, the other one's still has to exist
    assert L.b200pci_emd_matchcost_grad(1, 0, 5, p, p, p, p, p, None, None) == -1
    assert b"null pointer" in L.b200pci_last_error()
