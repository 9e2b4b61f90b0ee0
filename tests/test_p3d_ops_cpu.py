"""CPU tests of pytorch3d's ball_query and sample_farthest_points (mocopci_b200.p3d_ops, the C entry
points b200pci_ball_query_p3d / b200pci_fps_p3d): argument errors are raised on the host before any
device is touched; the sequential restatement the GPU tests compare with (tests/p3d_oracle.c) agrees
with a float64 numpy restatement of the contract on small ragged batches; the pytorch3d shim exposes
both names."""
import numpy as np
import pytest
import torch

from tests import p3d_oracle


@pytest.fixture(scope="module")
def p3d():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import p3d_ops
    return p3d_ops


# ------------------------------------------------------------------------------------------
# argument errors (CPU tensors: every shape / value error comes before the device check)
# ------------------------------------------------------------------------------------------
def test_ball_query_argument_errors(p3d):
    p1, p2 = torch.zeros(2, 5, 3), torch.zeros(2, 7, 3)
    bad = [
        (dict(p1=torch.zeros(2, 5)), "p1 must be a"),
        (dict(p1=torch.zeros(2, 5, 2)), "p1 must be a"),
        (dict(p2=torch.zeros(2, 7, 4)), "p2 must be a"),
        (dict(p2=torch.zeros(3, 7, 3)), "batch size"),
        (dict(p1=torch.zeros(2, 5, 3, dtype=torch.float64)), "float32"),
        (dict(K=0), "K must be"),
        (dict(K=-3), "K must be"),
        (dict(K=2.0), "K must be"),
        (dict(radius=-0.1), "radius"),
        (dict(radius=float("nan")), "radius"),
    ]
    for over, msg in bad:
        args = dict(p1=p1, p2=p2, K=4, radius=0.5)
        args.update(over)
        with pytest.raises(ValueError, match=msg):
            p3d.ball_query(args.pop("p1"), args.pop("p2"), **args)
    with pytest.raises(RuntimeError, match="CUDA"):
        p3d.ball_query(p1, p2, K=4)


def test_ball_query_lengths_errors_before_device(p3d, monkeypatch):
    """lengths are checked after the CUDA check; make the CPU clouds pass it to reach them."""
    from mocopci_b200 import _lib
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: None)
    p1, p2 = torch.zeros(2, 5, 3), torch.zeros(2, 7, 3)
    for name in ("lengths1", "lengths2"):
        for val, msg in ((torch.zeros(3, dtype=torch.int64), r"\(2,\) tensor"),
                         (torch.zeros(2, 1, dtype=torch.int64), r"\(2,\) tensor"),
                         (torch.zeros(2, dtype=torch.int32), "int64"),
                         (torch.zeros(2), "int64"),
                         ([5, 5], r"\(2,\) tensor")):
            with pytest.raises(ValueError, match=msg):
                p3d.ball_query(p1, p2, **{name: val})


def test_sample_farthest_points_argument_errors(p3d, monkeypatch):
    pts = torch.zeros(2, 9, 3)
    for kw, msg in ((dict(points=torch.zeros(2, 9)), "points must be"),
                    (dict(points=torch.zeros(2, 9, 2)), "points must be"),
                    (dict(points=torch.zeros(2, 9, 3, dtype=torch.float16)), "float32"),
                    (dict(K=0), "K must be >= 1"),
                    (dict(K=torch.tensor([3, 0])), "every K must be >= 1"),
                    (dict(K=torch.tensor([3, 2, 1])), r"\(2,\) tensor"),
                    (dict(K=torch.tensor([3.0, 2.0])), "integer tensor"),
                    (dict(K="5"), "K must be an int"),
                    (dict(points=torch.zeros(1, 131073, 3)), "131072")):
        args = dict(points=pts, K=4)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            p3d.sample_farthest_points(args.pop("points"), **args)
    with pytest.raises(RuntimeError, match="CUDA"):
        p3d.sample_farthest_points(pts, K=4)
    from mocopci_b200 import _lib
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: None)
    for val, msg in ((torch.zeros(3, dtype=torch.int64), r"\(2,\) tensor"),
                     (torch.zeros(2, dtype=torch.int32), "int64")):
        with pytest.raises(ValueError, match=msg):
            p3d.sample_farthest_points(pts, lengths=val, K=4)


def test_c_entry_points_argument_handling_without_gpu(p3d):
    L = p3d._L
    P = 16  # dummy non-null "device" pointer: every call below returns before using it

    def bq(B, P1, P2, K, radius, p1=P, p2=P, idx=P, dists=P):
        return L.b200pci_ball_query_p3d(B, P1, P2, K, radius, p1, 0, 0, 0, p2, 0, 0, 0, None, None, idx, dists,
                                        None, None)

    assert bq(0, 5, 5, 4, 0.5) == 0 and bq(2, 0, 5, 4, 0.5) == 0
    for args, msg in (((-1, 5, 5, 4, 0.5), b"negative size"), ((1, 5, -5, 4, 0.5), b"negative size"),
                      ((1, 5, 5, 0, 0.5), b"K must be"), ((1, 5, 5, 4, -1.0), b"radius"),
                      ((1, 5, 5, 4, float("nan")), b"radius"), ((70000, 5, 5, 4, 0.5), b"batch")):
        assert bq(*args) == -1, args
        assert msg in L.b200pci_last_error()
    for miss in ("p1", "p2", "idx", "dists"):
        assert bq(1, 5, 5, 4, 0.5, **{miss: None}) == -1
        assert b"null pointer" in L.b200pci_last_error()

    def fps(B, Pn, M, points=P, idx=P):
        return L.b200pci_fps_p3d(B, Pn, M, points, 0, 0, 0, None, None, None, idx, None, None)

    assert fps(0, 5, 4) == 0 and fps(2, 5, 0) == 0
    for args, msg in (((-1, 5, 4), b"negative size"), ((1, -5, 4), b"negative size"),
                      ((1, 131073, 4), b"131072")):
        assert fps(*args) == -1, args
        assert msg in L.b200pci_last_error()
    assert fps(1, 5, 4, points=None) == -1 and b"null pointer" in L.b200pci_last_error()
    assert fps(1, 5, 4, idx=None) == -1 and b"null pointer" in L.b200pci_last_error()


def test_shim_exposes_ball_query_and_sample_farthest_points(p3d):
    from mocopci_b200 import chamfer, shim
    mods = shim._pytorch3d_shim()
    ops = mods["pytorch3d.ops"]
    assert ops.ball_query is p3d.ball_query
    assert ops.sample_farthest_points is p3d.sample_farthest_points
    # what was registered before stays as it was
    assert ops.knn_points is chamfer.knn_points and ops.knn_gather is chamfer.knn_gather
    assert mods["pytorch3d.loss"].chamfer_distance is chamfer.chamfer_distance


# ------------------------------------------------------------------------------------------
# the oracle against a float64 restatement of the contract
# ------------------------------------------------------------------------------------------
def np_ball_query(p1, p2, K, radius, l1, l2):
    p1, p2 = p1.astype(np.float64), p2.astype(np.float64)
    B, P1, _ = p1.shape
    r2 = float(np.float32(radius) * np.float32(radius))
    idx = np.full((B, P1, K), -1, np.int64)
    dists = np.zeros((B, P1, K), np.float64)
    for b in range(B):
        n1, n2 = min(max(l1[b], 0), P1), min(max(l2[b], 0), p2.shape[1])
        for i in range(n1):
            d2 = ((p1[b, i] - p2[b, :n2]) ** 2).sum(-1)
            hits = np.nonzero(d2 < r2)[0][:K]
            idx[b, i, :len(hits)] = hits
            dists[b, i, :len(hits)] = d2[hits]
    return idx, dists


def np_fps(pts, Ks, lengths, start):
    pts = pts.astype(np.float64)
    B, P, _ = pts.shape
    M = int(max(Ks))
    idx = np.full((B, M), -1, np.int64)
    for b in range(B):
        n = min(max(lengths[b], 0), P)
        m = min(Ks[b], n)
        if m == 0:
            continue
        last = start[b]
        idx[b, 0] = last
        mind = np.full(n, np.inf)
        for t in range(1, m):
            mind = np.minimum(mind, ((pts[b, :n] - pts[b, last]) ** 2).sum(-1))
            last = int(np.argmax(mind))  # first maximum: the lowest index wins a tie
            idx[b, t] = last
    return idx


def grid_cloud(rng, B, P, g=4):
    """Integer coordinates: every FP32 distance is exact, so FP32 and FP64 must agree bit for bit,
    ties included (many equal distances)."""
    return rng.integers(-g, g + 1, size=(B, P, 3)).astype(np.float32)


@pytest.mark.parametrize("K", [1, 5, 40])
def test_oracle_ball_query_vs_fp64(K):
    rng = np.random.default_rng(K)
    B, P1, P2 = 4, 23, 37
    l1, l2 = np.array([23, 0, 1, 17]), np.array([37, 5, 0, 30])
    p1, p2 = grid_cloud(rng, B, P1), grid_cloud(rng, B, P2)
    for radius in (0.0, 1.0, 2.5, 3.0, 100.0):  # 1.0 and 3.0: radius^2 is itself a distance (strict <)
        idx, dists = p3d_oracle.ball_query(p1, p2, K, radius, l1, l2)
        wi, wd = np_ball_query(p1, p2, K, radius, l1, l2)
        np.testing.assert_array_equal(idx, wi, err_msg=f"radius {radius}")
        np.testing.assert_array_equal(dists.astype(np.float64), wd, err_msg=f"radius {radius}")
    # random floats: FP32 and FP64 agree away from the boundary
    p1, p2 = rng.standard_normal((B, P1, 3)).astype(np.float32), rng.standard_normal((B, P2, 3)).astype(np.float32)
    idx, dists = p3d_oracle.ball_query(p1, p2, K, 1.1, l1, l2)
    wi, wd = np_ball_query(p1, p2, K, 1.1, l1, l2)
    np.testing.assert_array_equal(idx, wi)
    np.testing.assert_allclose(dists, wd, rtol=1e-6, atol=1e-6)
    # no lengths == full lengths
    full = p3d_oracle.ball_query(p1, p2, K, 1.1)
    want = p3d_oracle.ball_query(p1, p2, K, 1.1, [P1] * B, [P2] * B)
    np.testing.assert_array_equal(full[0], want[0])


def test_oracle_fps_vs_fp64():
    rng = np.random.default_rng(7)
    B, P = 5, 60
    lengths = np.array([60, 0, 1, 2, 41])
    for Ks in ([8] * B, [8, 3, 5, 1, 60], [60] * B):
        for start in ([0] * B, [5, 0, 0, 1, 40]):
            pts = grid_cloud(rng, B, P, g=2)  # 125 sites for 60 points: duplicates and ties everywhere
            got = p3d_oracle.fps(pts, Ks, lengths, start)
            np.testing.assert_array_equal(got, np_fps(pts, Ks, lengths, start), err_msg=f"K {Ks} start {start}")
    pts = rng.standard_normal((B, P, 3)).astype(np.float32)
    np.testing.assert_array_equal(p3d_oracle.fps(pts, 20, lengths), np_fps(pts, [20] * B, lengths, [0] * B))
    # beyond the cloud: -1
    got = p3d_oracle.fps(pts, 70, lengths)
    assert (got[:, 60:] == -1).all() and (got[1] == -1).all() and (got[2, 1:] == -1).all()
