"""GPU parity tests (run on the B200 box): every CUDA entry point, called through the
reference-facing Python layer (which goes through the C ABI), against
  * the CPU oracle (oracle/oracle.c) on seeded inputs,
  * the committed golden fixtures generated from the reference's own torch code, and
  * the reference's own CUDA kernels compiled unmodified into oracle/_ref (bitwise).
Bar: bit-exact for indices / gathers / distances in the reference arithmetic; 1e-5 relative for
Chamfer / EMD values (tolerance written at each assert). The reference's torch distance helpers
are restated in oracle/torch_port.py and run on the same CUDA tensors. Where a test compared with
the reference's compiled kernels, which need a MoCoPCI checkout, it compares with a stored snapshot
of kernel outputs instead (tests/kernel_snapshot.py), next to the oracle where the oracle covers
the operator.
"""
import glob
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import torch_port
from tests import kernel_snapshot as snapshot

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _OwnP2U:
    """mocopci_b200.ops behind the attribute names the tests use for the reference's module."""

    def __init__(self, ops_mod):
        for n in ("furthest_point_sample", "gather_operation", "three_nn", "three_interpolate",
                  "grouping_operation", "ball_query"):
            setattr(self, n, getattr(ops_mod, n))
        self._ops = ops_mod

    def QueryAndGroup(self, radius, nsample, use_xyz=True):
        return lambda xyz, new_xyz, features=None: self._ops.query_and_group(
            radius, nsample, xyz, new_xyz, features, use_xyz)


class _OwnEmd:
    def __init__(self, ops_mod):
        self.earth_mover_distance = ops_mod.earth_mover_distance
        self.EMD = ops_mod.emd_metric


@pytest.fixture(scope="module", params=["reference_wrappers", "own_api"])
def ops(request):
    """The operators under test, reached the way a user reaches them:
    * reference_wrappers: the REFERENCE's own pointnet2/pointnet2_utils.py, models/EMD/emd.py and
      models/utils.py (imported unmodified from a checkout when one is available, else their calls
      restated in tests/refwrappers.py) on top of mocopci_b200.install();
    * own_api: mocopci_b200.ops."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import mocopci_b200
    from mocopci_b200 import chamfer, emd_cuda, ops as own, pointconv_util, pointnet2_cuda, synth

    class O:
        pass
    o = O()
    o.api = request.param
    o.chamfer, o.emd_cuda, o.pcu, o.p2c, o.synth, o.own = (chamfer, emd_cuda, pointconv_util,
                                                           pointnet2_cuda, synth, own)
    if request.param == "reference_wrappers":
        import importlib
        from baseline import fetch_ref
        root = fetch_ref.root()
        mocopci_b200.install(reference_root=root)
        if root is not None:
            o.p2u = importlib.import_module("pointnet2.pointnet2_utils")
            emd_mod = importlib.import_module("models.EMD.emd")
            utils = importlib.import_module("models.utils")
            o.emd = types.SimpleNamespace(earth_mover_distance=emd_mod.earth_mover_distance, EMD=utils.EMD)
        else:
            from tests import refwrappers
            o.p2u = refwrappers
            o.emd = types.SimpleNamespace(earth_mover_distance=refwrappers.earth_mover_distance,
                                          EMD=refwrappers.EMD)
        assert o.p2u.pointnet2 is pointnet2_cuda          # the reference's wrappers run on our module
    else:
        o.p2u, o.emd = _OwnP2U(own), _OwnEmd(own)
    return o


def dev(a):
    return torch.as_tensor(a).cuda()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def installed_knn_point():
    """``knn_point`` as mocopci_b200.install() binds it in the reference's modules; the inputs of the
    tests that use it are all covered by the kernel, so the reference's own function is never run.
    install() only re-binds functions of imported reference modules, so without a checkout the
    binding is made directly with the helper it uses (shim._replacement)."""
    from mocopci_b200 import shim

    def reference_knn_point(*args):
        raise AssertionError("the installed knn_point fell back to the reference's torch code")
    return shim._replacement("knn_point", reference_knn_point)


# ------------------------------------------------------------------------------------------
# KNN (K1 + K2)
# ------------------------------------------------------------------------------------------
def check_knn_against_oracle(ops, orc, xyz, new_xyz, k):
    """Both evaluation orders of the reference's square_distance: "cpu" (CPU torch = BASELINE's CPU
    path, oracle form 0) and "cuda" (CUDA torch, the default; oracle form 5)."""
    for arith, form in (("cpu", 0), ("cuda", 5)):
        idx, dist = ops.pcu.knn_point_with_dist(k, dev(xyz), dev(new_xyz), arith=arith)
        torch.cuda.synchronize()
        oi, od = orc.knn_form(form, k, xyz, new_xyz)
        assert idx.dtype == torch.int64 and tuple(idx.shape) == oi.shape
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)          # bit-exact indices, ties -> lowest
        np.testing.assert_array_equal(bits(dist.cpu().numpy()), bits(od))  # bit-exact distances


@pytest.mark.parametrize("B,S,N,k", [(1, 1, 16, 16), (2, 257, 1000, 16), (1, 130, 513, 32),
                                      (3, 64, 2048, 3), (1, 1000, 700, 1), (2, 300, 4100, 8),
                                      (1, 77, 600, 5), (1, 50, 1500, 64),
                                      # k <= 4 at N >= 2048: two-pass path with the guaranteed bound
                                      (1, 700, 5000, 1), (2, 300, 3000, 4), (1, 1030, 9000, 3),
                                      (1, 100, 20000, 2)])
def test_knn_uniform_vs_oracle(ops, orc, B, S, N, k):
    xyz = ops.synth.uniform_cloud(100 + N, B, N).numpy()
    new = ops.synth.uniform_cloud(200 + S, B, S).numpy()
    check_knn_against_oracle(ops, orc, xyz, new, k)


@pytest.mark.parametrize("B,S,N,k", [(1, 700, 5000, 1), (2, 300, 3000, 4), (1, 1030, 9000, 3),
                                      (1, 100, 20000, 2)])
def test_knn_small_k_two_pass_forced(ops, orc, B, S, N, k):
    """k <= 4 takes the two-pass path (guaranteed sample bound) only from 2^25 pairs; test hook 7
    lowers that threshold so the oracle can check it on small inputs, EXPANDED (knn_point) and
    DIRECT (three_nn)."""
    from mocopci_b200 import _lib
    xyz = ops.synth.uniform_cloud(300 + N, B, N, -30.0, 30.0).numpy()
    new = ops.synth.uniform_cloud(400 + S, B, S, -30.0, 30.0).numpy()
    try:
        _lib.check(_lib.lib.b200pci_debug_set(7, 1))
        check_knn_against_oracle(ops, orc, xyz, new, k)
        u, kn = dev(new), dev(xyz)
        dist, idx = ops.p2u.three_nn(u, kn)
    finally:
        _lib.check(_lib.lib.b200pci_debug_set(7, 0))
    od2, oi = orc.three_nn(new, xyz)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(dist.cpu().numpy()), bits(np.sqrt(od2)))


def test_knn_tie_stress_vs_oracle(ops, orc):
    t = ops.synth.tie_stress_cloud(5, 2, 1200).numpy()
    for k in (3, 16, 32):
        check_knn_against_oracle(ops, orc, t, t, k)


def test_knn_lidar_split_path_vs_oracle(ops, orc):
    # B=1 with few queries -> the ref-split + merge path
    a, b = ops.synth.frame_pair(3, 8192)
    check_knn_against_oracle(ops, orc, a[None].numpy(), b[None, :700].numpy(), 16)


@pytest.mark.parametrize("k", [8, 16, 32, 64])
def test_knn_estimated_bound_path_vs_oracle(ops, orc, k):
    # N >= 8192 and k >= 8: threshold pre-pass + estimated admission bound + exact redo
    a, b = ops.synth.frame_pairs(5, 2)
    check_knn_against_oracle(ops, orc, a.numpy(), b[:, :1100].numpy(), k)


def test_knn_estimated_bound_tie_stress(ops, orc):
    t = ops.synth.tie_stress_cloud(21, 1, 9000, grid=9).numpy()
    check_knn_against_oracle(ops, orc, t, t[:, :900], 16)


@pytest.mark.parametrize("scale", [0.02, 0.3, 50.0])
def test_knn_forced_redo_and_overflow(ops, orc, scale):
    """Test hook: shrink (or blow up) the estimated bound so that most queries take the exact
    redo kernel (or overflow their pending lists); results must not change."""
    from mocopci_b200 import _lib
    a, b = ops.synth.frame_pairs(7, 1)
    try:
        _lib.check(_lib.lib.b200pci_debug_set(1, scale))
        check_knn_against_oracle(ops, orc, a.numpy(), b[:, :777].numpy(), 16)
        check_knn_against_oracle(ops, orc, a.numpy(), b[:, :300].numpy(), 32)
    finally:
        _lib.check(_lib.lib.b200pci_debug_set(1, 1.0))


def test_knn_degenerate_cloud_mass_redo(ops, orc):
    """A cloud of identical points: every ref is at the same distance, the estimated bound admits
    none of them (strict test), so EVERY query is flagged -> the tile-wise redo kernel (more than
    2048 flagged queries). Lowest indices win the ties."""
    xyz = np.tile(np.array([[1.5, -2.0, 0.25]], dtype=np.float32), (1, 9000, 1))
    new = ops.synth.uniform_cloud(5, 1, 3000, -5.0, 5.0).numpy()
    check_knn_against_oracle(ops, orc, xyz, new, 16)
    # half degenerate: 6000 copies of one point + 6000 spread points
    rest = ops.synth.uniform_cloud(6, 1, 6000, -5.0, 5.0).numpy()
    xyz2 = np.concatenate([xyz[:, :6000], rest], axis=1)
    check_knn_against_oracle(ops, orc, xyz2, new, 32)


@pytest.mark.parametrize("B,S,N,k,lo,hi", [(1, 700, 9000, 16, -1.0, 1.0), (2, 1100, 8192, 32, -50.0, 50.0),
                                            (1, 513, 16500, 8, -80.0, 80.0), (3, 129, 10000, 16, 900.0, 1000.0)])
def test_knn_two_pass_vs_oracle(ops, orc, B, S, N, k, lo, hi):
    """The two-pass path: the tensor-core filter (tcgen05 TF32, split operands) is a conservative
    pre-filter in front of the exact evaluation, so the result must reproduce the oracle bit for
    bit -- also far from the origin, where the relative slack of the filter is largest in absolute
    terms."""
    xyz = ops.synth.uniform_cloud(700 + N, B, N, lo, hi).numpy()
    new = ops.synth.uniform_cloud(800 + S, B, S, lo, hi).numpy()
    check_knn_against_oracle(ops, orc, xyz, new, k)


@pytest.mark.parametrize("k", [1, 3, 16, 32])
def test_knn_two_pass_clusters_vs_oracle(ops, orc, k):
    """The two-pass path on two far-apart Gaussian clusters (about +40 m and -55 m) with 1000 exact
    duplicates, queried by a permuted subset of the cloud: candidates crowd into few ref tiles and
    tie exactly. Oracle bit for bit in all three arithmetics; hook 7 sends k <= 4 to the two-pass
    path as well."""
    from mocopci_b200 import _lib, pointconv_util as pcu
    g = torch.Generator().manual_seed(k)
    clusters = torch.cat([torch.randn(2, 9000, 3, generator=g) * 0.5 + 40.0,
                          torch.randn(2, 7384, 3, generator=g) * 2.0 - 55.0], 1)
    clusters[:, 100:1100] = clusters[:, 3000:4000]                     # 1000 exact duplicates
    new = clusters[:, torch.randperm(16384, generator=g)][:, :5000].contiguous()
    for mode, form in ((pcu.DIST_EXPANDED_CUDA, 5), (pcu.DIST_DIRECT, 1), (pcu.DIST_DIRECT_XYZ, 2)):
        try:
            _lib.check(_lib.lib.b200pci_debug_set(7, 1))
            idx, dist = pcu._knn(k, clusters.cuda(), new.cuda(), mode, True)
        finally:
            _lib.check(_lib.lib.b200pci_debug_set(7, 0))
        oi, od = orc.knn_form(form, k, clusters.numpy(), new.numpy())
        np.testing.assert_array_equal(idx.cpu().numpy(), oi, err_msg=f"mode {mode}")
        np.testing.assert_array_equal(bits(dist.cpu().numpy()), bits(od), err_msg=f"mode {mode}")


@pytest.mark.parametrize("grid", [6, 20])
def test_knn_two_pass_tie_stress_vs_oracle(ops, orc, grid):
    """Exact ties on the two-pass path (integer-grid coordinates, half the points duplicated, N large
    enough for the tensor-core scan): the filter flags every tied ref, the keys pick the lowest index.
    grid = 6 puts ~4 points on every site (lists overflow -> exact redo), grid = 20 mostly pairs."""
    xyz = ops.synth.tie_stress_cloud(31 + grid, 2, 9000, grid).numpy()
    new = ops.synth.tie_stress_cloud(41 + grid, 2, 700, grid).numpy()
    for k in (8, 16, 32):
        check_knn_against_oracle(ops, orc, xyz, new, k)
    check_knn_against_oracle(ops, orc, xyz, xyz[:, :1500], 16)  # queries that coincide with refs


@pytest.mark.parametrize("k", [3, 16, 32])
def test_knn_topk_lane_balancing_does_not_change_results(ops, k):
    """knn_topk_kernel hands the 128 queries of a CTA to its threads in order of their candidate-list
    length (hook 20 = 1, default) instead of thread t = query t: a permutation of who does what, so
    indices and distance bits must be identical -- checked where the launch is large enough not to
    take the split kernel (12 clouds), with ragged S and with ties."""
    from mocopci_b200 import _lib, pointconv_util as pcu
    a, b = ops.synth.frame_pairs(90 + k, 12, 8192)
    ties = ops.synth.tie_stress_cloud(7, 12, 8192, grid=20)
    for xyz, new in ((a.cuda(), b[:, :8000].contiguous().cuda()), (ties.cuda(), ties.cuda())):
        try:
            _lib.check(_lib.lib.b200pci_debug_set(7, 1))      # k <= 4: two-pass path from small sizes on
            _lib.check(_lib.lib.b200pci_debug_set(20, 0))
            i0, d0 = pcu._knn(k, xyz, new, pcu.DIST_EXPANDED_CUDA, True)
            _lib.check(_lib.lib.b200pci_debug_set(20, 1))
            i1, d1 = pcu._knn(k, xyz, new, pcu.DIST_EXPANDED_CUDA, True)
        finally:
            _lib.check(_lib.lib.b200pci_debug_set(20, 1))
            _lib.check(_lib.lib.b200pci_debug_set(7, 0))
        assert torch.equal(i1, i0) and torch.equal(d1.view(torch.int32), d0.view(torch.int32))


@pytest.mark.parametrize("k", [8, 16, 32])
def test_knn_split_topk_kernel_equals_thread_per_query_kernel(ops, k):
    """Small launches of the two-pass path (one or two frame pairs) run knn_topk_split_kernel -- one
    thread per (query, group of ref splits), partial lists folded through shared memory -- instead
    of one thread per query (hook 18 = 0). Same candidate lists, so indices, distance bits and the
    rows left to the exact redo must be identical: LiDAR frames, a cloud against itself, duplicated
    points on an integer grid (ties across splits), S not a multiple of 128, int32 output."""
    from mocopci_b200 import _lib, pointconv_util as pcu
    a, b = ops.synth.frame_pairs(80 + k, 2)
    ties = ops.synth.tie_stress_cloud(5, 1, 12000, grid=24)
    cases = [("pair", a[:1].cuda(), b[:1].cuda()), ("self", a[:1].cuda(), a[:1].cuda()),
             ("two pairs, ragged S", a.cuda(), b[:, :9001].contiguous().cuda()),
             ("ties", ties.cuda(), ties[:, :8200].contiguous().cuda())]
    for name, xyz, new in cases:
        for mode in (pcu.DIST_EXPANDED_CUDA, pcu.DIST_DIRECT):
            try:
                _lib.check(_lib.lib.b200pci_debug_set(18, 0))
                i0, d0 = pcu._knn(k, xyz, new, mode, True)
                _lib.check(_lib.lib.b200pci_debug_set(18, 1))
                i1, d1 = pcu._knn(k, xyz, new, mode, True)
                j1, _ = pcu._knn(k, xyz, new, mode, False, int64=False)
            finally:
                _lib.check(_lib.lib.b200pci_debug_set(18, 1))
            assert torch.equal(i1, i0), f"{name} mode {mode}: {int((i1 != i0).sum())} indices differ"
            assert torch.equal(d1.view(torch.int32), d0.view(torch.int32)), f"{name} mode {mode}"
            assert torch.equal(j1.long(), i0)


def test_knn_exact_mode_equals_estimated(ops):
    from mocopci_b200 import _lib
    a, b = ops.synth.frame_pairs(9, 2)
    a, b = a.cuda(), b.cuda()
    i1, d1 = ops.pcu.knn_point_with_dist(16, a, b)
    try:
        _lib.check(_lib.lib.b200pci_debug_set(2, 1))
        i2, d2 = ops.pcu.knn_point_with_dist(16, a, b)
    finally:
        _lib.check(_lib.lib.b200pci_debug_set(2, 0))
    assert torch.equal(i1, i2) and torch.equal(d1.view(torch.int32), d2.view(torch.int32))


@pytest.mark.parametrize("B,S,N,k", [(1, 37, 8193, 16), (2, 129, 12345, 32), (1, 64, 70001, 16),
                                      (1, 5, 16384, 8), (3, 700, 9000, 24)])
def test_knn_odd_sizes_estimated_path(ops, orc, B, S, N, k):
    xyz = ops.synth.uniform_cloud(N, B, N, -40.0, 40.0).numpy()
    new = ops.synth.uniform_cloud(S + 1, B, S, -40.0, 40.0).numpy()
    check_knn_against_oracle(ops, orc, xyz, new, k)


def test_knn_points_direct_estimated_path(ops, orc):
    p1 = ops.synth.uniform_cloud(31, 2, 500).numpy()
    p2 = ops.synth.uniform_cloud(32, 2, 9001).numpy()
    r = ops.chamfer.knn_points(dev(p1), dev(p2), K=16)
    oi, od = orc.knn_form(2, 16, p2, p1)
    np.testing.assert_array_equal(r.idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(r.dists.cpu().numpy()), bits(od))


def test_knn_permuted_views(ops, orc):
    # the model passes permuted views of [B,3,N] (mocopci.py:1327); strides must be honoured
    xyz = ops.synth.uniform_cloud(1, 2, 900)
    new = ops.synth.uniform_cloud(2, 2, 333)
    xv = dev(xyz).permute(0, 2, 1).contiguous().permute(0, 2, 1)
    nv = dev(new).permute(0, 2, 1).contiguous().permute(0, 2, 1)
    assert not xv.is_contiguous()
    idx = ops.pcu.knn_point(16, xv, nv, arith="cpu")
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.knn_expanded(16, xyz.numpy(), new.numpy()))
    # CUDA torch reduces a permuted view's |p|^2 sequentially like the CPU: "cuda" == form 0 here
    idx = ops.pcu.knn_point(16, xv, nv)
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.knn_expanded(16, xyz.numpy(), new.numpy()))


@pytest.mark.parametrize("path", sorted(p for p in glob.glob(os.path.join(GOLDEN, "knn_*.npz"))
                                        if "sqdiff" not in p))
def test_knn_golden_reference(ops, path):
    """Against the reference's own torch output (tests/golden/make_golden.py): SURVEY 8c protocol."""
    g = np.load(path)
    xyz, new, k = g["xyz"], g["new_xyz"], int(g["k"])
    idx, dist = ops.pcu.knn_point_with_dist(k, dev(xyz), dev(new), arith="cpu")   # fixtures: CPU torch
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    ref_vals = g["ref_vals"]  # sorted k+1 smallest reference distances
    # (i) our selected distances are bitwise the reference's k smallest
    np.testing.assert_array_equal(bits(dist), bits(ref_vals[..., :k]))
    # (ii) same index set wherever the reference has no tie at the k-th distance
    ref_idx = np.sort(g["ref_idx"].astype(np.int64), -1)
    ours = np.sort(idx, -1)
    no_tie = ref_vals[..., k - 1] != ref_vals[..., k] if ref_vals.shape[-1] > k else \
        np.ones(ref_idx.shape[:-1], bool)
    assert (ours[no_tie] == ref_idx[no_tie]).all()
    # (iii) reference matrix rows: our distances are entries of the reference's D
    D = g["ref_D_rows"]
    got = np.take_along_axis(D, idx[:, : D.shape[1]], axis=-1)
    np.testing.assert_array_equal(bits(got), bits(dist[:, : D.shape[1]]))


@pytest.mark.parametrize("name", ["sqdiff_k16", "sqdiff_tie_k16"])
def test_knn_sqdiff_golden_reference(ops, name):
    """f3: models/pointT_layer2.py:20,62-63 (square_distance(xyz, xyz).argsort()[:, :, :k]) as run by
    the imported reference (tests/golden/make_golden.py): ascending distances bitwise equal, same
    index set wherever the reference has no tie at the k-th distance (argsort is not stable)."""
    g = np.load(os.path.join(GOLDEN, f"knn_{name}.npz"))
    xyz, k = dev(g["xyz"]), int(g["k"])
    idx = ops.pcu.knn_point_sqdiff(k, xyz, xyz, arith="cpu")          # the fixture is CPU torch's output
    assert idx.dtype == torch.int64
    idx = idx.cpu().numpy()
    x = g["xyz"]
    sel = np.take_along_axis(x[:, None].repeat(x.shape[1], 1), idx[..., None].repeat(3, -1), axis=2)
    diff = x[:, :, None, :] - sel
    d = (diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]) + diff[..., 2] * diff[..., 2]
    ref_vals = g["ref_vals"]
    np.testing.assert_array_equal(bits(d), bits(ref_vals[..., :k]))   # in order: ascending
    no_tie = ref_vals[..., k - 1] != ref_vals[..., k]
    assert (np.sort(idx, -1)[no_tie] == np.sort(g["ref_idx"].astype(np.int64), -1)[no_tie]).all()


@pytest.mark.parametrize("layout", ["contiguous", "permuted", "mixed"])
@pytest.mark.parametrize("B,S,N,k", [(1, 16384, 16384, 16), (1, 16384, 16384, 32), (2, 4096, 16384, 3),
                                      (1, 2048, 2048, 16), (3, 700, 1000, 8)])
def test_knn_bitwise_vs_reference_on_the_same_gpu(ops, B, S, N, k, layout):
    """The reference's square_distance + topk (models/pointconv_util.py:67-88,129-140, restated op
    for op in oracle/torch_port.py) executed by CUDA torch on this GPU: our default ("cuda")
    arithmetic reproduces its matrix entries BITWISE at the selected indices and selects the same
    k-distance multiset for every query; index sets equal wherever it has no tie. The
    reference_wrappers variant calls knn_point as install() binds it in the reference's modules,
    which returns the indices only."""
    a, b = ops.synth.frame_pairs(50 + k, B, max(S, N))
    xyz, new = a[:, :N].contiguous().cuda(), b[:, :S].contiguous().cuda()
    # the model mostly passes permuted views of [B,3,N] tensors (mocopci.py:1327); CUDA torch's
    # reduction order depends on that layout, and so must ours
    if layout in ("permuted", "mixed"):
        new = new.permute(0, 2, 1).contiguous().permute(0, 2, 1)
    if layout == "permuted":
        xyz = xyz.permute(0, 2, 1).contiguous().permute(0, 2, 1)
    D = torch_port.square_distance(new, xyz)
    if ops.api != "own_api":
        idx = installed_knn_point()(k, xyz, new)
        dist = torch.gather(D, 2, idx)
    else:
        idx, dist = ops.pcu.knn_point_with_dist(k, xyz, new)
        assert torch.equal(torch.gather(D, 2, idx).view(torch.int32), dist.view(torch.int32))
    vals = torch.topk(D, k + 1, dim=-1, largest=False, sorted=True)[0]
    assert torch.equal(vals[..., :k].view(torch.int32), dist.view(torch.int32))
    ref_idx = torch_port.knn_point(k, xyz, new)
    no_tie = vals[..., k - 1] != vals[..., k]
    assert bool((idx.sort(-1)[0] == ref_idx.sort(-1)[0]).all(-1)[no_tie].all())


@pytest.mark.parametrize("permuted", [False, True])
def test_knn_sqdiff_bitwise_vs_reference_on_the_same_gpu(ops, permuted):
    """f3 on the GPU: models/pointT_layer2.py:20,62-63 (restated in oracle/torch_port.py) executed by
    CUDA torch (its 3-element sum adds (dx^2 + dz^2) + dy^2, unlike the CPU): same ascending
    distances bit for bit."""
    xyz = ops.synth.lidar_frame(99, 2048)[None].cuda()
    if permuted:
        xyz = xyz.permute(0, 2, 1).contiguous().permute(0, 2, 1)
    D = torch_port.square_distance_sqdiff(xyz, xyz)
    ref_sorted = D.sort(-1)[0][:, :, :17]
    idx = ops.pcu.knn_point_sqdiff(16, xyz, xyz)
    assert torch.equal(torch.gather(D, 2, idx).view(torch.int32), ref_sorted[..., :16].view(torch.int32))
    no_tie = ref_sorted[..., 15] != ref_sorted[..., 16]
    ref_idx = D.argsort()[:, :, :16]
    assert bool((idx.sort(-1)[0] == ref_idx.sort(-1)[0]).all(-1)[no_tie].all())


@pytest.mark.parametrize("form", [1, 2, 3, 4])
@pytest.mark.parametrize("B,S,N,k", [(2, 300, 1000, 16), (1, 2048, 2048, 16), (1, 100, 9000, 3),
                                      (2, 600, 16384, 1), (1, 257, 700, 32)])
def test_knn_direct_forms_vs_oracle(ops, orc, form, B, S, N, k):
    """The direct-difference arithmetics (pointnet2 / pytorch3d / pointT_layer2 in CPU and CUDA torch's
    sum order) on every code path: indices and distance bits against the C oracle."""
    from mocopci_b200 import pointconv_util as pcu
    xyz = ops.synth.uniform_cloud(N + form, B, N, -20.0, 20.0).numpy()
    new = ops.synth.uniform_cloud(S + 7, B, S, -20.0, 20.0).numpy()
    idx, dist = pcu._knn(k, dev(xyz), dev(new), form, True)
    oi, od = orc.knn_form(form, k, xyz, new)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(dist.cpu().numpy()), bits(od))


@pytest.mark.parametrize("k", [16, 32])
def test_knn_full_benchmark_pair_vs_oracle(ops, orc, k):
    """One full 16384 x 16384 frame pair of the BENCHMARKED workload (bench.py: synth.frame_pairs(0, .))
    against the OpenMP C oracle: every index and every distance bit. The reference_wrappers variant
    calls knn_point as install() binds it in the reference's modules: every index, in the
    reference's CUDA torch arithmetic (oracle form 5)."""
    a, b = ops.synth.frame_pairs(0, 1)
    if ops.api != "own_api":
        idx = installed_knn_point()(k, dev(a), dev(b))
        np.testing.assert_array_equal(idx.cpu().numpy(), orc.knn_form(5, k, a.numpy(), b.numpy())[0])
        return
    check_knn_against_oracle(ops, orc, a.numpy(), b.numpy(), k)


def test_knn_host_api_odd_batches(ops, orc):
    """b200pci_knn_host (bench.py's e2e entry): odd batches make the two chunks differ in size, and
    the smaller chunk can need MORE scratch (make_plan is not monotonic in B)."""
    from mocopci_b200 import _lib, host_api
    for B, S, N, k in ((3, 640, 6400, 16), (5, 300, 3584, 3), (1, 100, 9000, 16), (7, 64, 7424, 32)):
        xyz = ops.synth.uniform_cloud(B * 7 + N, B, N, -10.0, 10.0)
        new = ops.synth.uniform_cloud(B * 5 + S, B, S, -10.0, 10.0)
        out = host_api.knn_point_host(k, xyz, new)
        assert out.dtype == torch.int64 and not out.is_cuda
        np.testing.assert_array_equal(out.numpy(), orc.knn_form(5, k, xyz.numpy(), new.numpy())[0])
        np.testing.assert_array_equal(host_api.knn_point_host(k, xyz, new, arith="cpu").numpy(),
                                      orc.knn_expanded(k, xyz.numpy(), new.numpy()))
        out32 = torch.empty((B, S, k), dtype=torch.int32, pin_memory=True)
        host_api.knn_point_host(k, xyz.pin_memory(), new.pin_memory(), out=out32)
        np.testing.assert_array_equal(out32.numpy(), out.numpy())
        for chunks in (1, 4, 8):
            try:
                _lib.check(_lib.lib.b200pci_debug_set(14, chunks))
                np.testing.assert_array_equal(host_api.knn_point_host(k, xyz, new).numpy(), out.numpy())
            finally:
                _lib.check(_lib.lib.b200pci_debug_set(14, 0))
    _lib.check(_lib.lib.b200pci_host_release())


def test_knn_host_api_tapered_schedule_matches_device_path(ops):
    """b200pci_knn_host with a batch large enough for the tapered chunk schedule (B >= 24: a small
    first chunk, then geometrically shrinking ones, knn.cu host_schedule): every row must equal the device-resident call on the same
    clouds -- which the tests above pin to the oracle -- on the two-pass path (5120-point clouds)
    and on the one-launch path, for repeated calls (buffer reuse) and both index widths."""
    from mocopci_b200 import _lib, host_api, pointconv_util as pcu
    for B, S, N, k in ((26, 5120, 5120, 16), (49, 700, 1500, 8), (33, 4608, 6144, 32)):
        xyz = ops.synth.uniform_cloud(B + N, B, N, -20.0, 20.0)
        new = ops.synth.uniform_cloud(B + S + 1, B, S, -20.0, 20.0)
        want = pcu.knn_point(k, xyz.cuda(), new.cuda()).cpu()
        for _ in range(2):
            got = host_api.knn_point_host(k, xyz, new)
            assert torch.equal(got, want)
        out32 = torch.empty((B, S, k), dtype=torch.int32, pin_memory=True)
        host_api.knn_point_host(k, xyz.pin_memory(), new.pin_memory(), out=out32)
        assert torch.equal(out32.long(), want)
    _lib.check(_lib.lib.b200pci_host_release())


# ------------------------------------------------------------------------------------------
# feature-space cosine KNN (f2)
# ------------------------------------------------------------------------------------------
COS_ATOL = 4e-6   # the reference's bmm and our tensor-core contraction sum C products in their own
COS_GAP = 8e-6    # order (and the tensor core truncates when aligning addends: measured 1.8e-6 at C = 256);
                  # neighbour sets must agree wherever the reference's gap is clear


def check_cosine(idx, dist, ref_D, k):
    """ref_D: the reference's cosine_distance matrix [B,S,N] (torch). (i) our k distances equal the
    reference's k smallest to COS_ATOL, and are what the reference has at our indices; (ii) same
    index set wherever the reference's k-th and (k+1)-th distances are more than COS_GAP apart."""
    kk = min(k + 1, ref_D.shape[-1])
    ref_vals, ref_idx = torch.topk(ref_D, kk, dim=-1, largest=False, sorted=True)
    assert float((dist - ref_vals[..., :k]).abs().max()) <= COS_ATOL
    assert float((torch.gather(ref_D, 2, idx) - dist).abs().max()) <= COS_ATOL
    assert bool((dist[..., 1:] >= dist[..., :-1]).all())
    if kk > k:
        clear = (ref_vals[..., k] - ref_vals[..., k - 1]) > COS_GAP
        same = (idx.sort(-1)[0] == ref_idx[..., :k].sort(-1)[0]).all(-1)
        assert bool(same[clear].all()), f"{int((~same & clear).sum())} index sets differ with a clear gap"
        return float(clear.float().mean())
    return 1.0


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "cos_*.npz"))))
def test_knn_point_cosine_golden_reference(ops, path):
    """Against the imported reference's own output on the CPU (tests/golden/make_golden.py), inputs as
    the permuted [B,C,N] views the model passes."""
    g = np.load(path)
    xyz, new, k = dev(g["xyz_t"]).permute(0, 2, 1), dev(g["new_t"]).permute(0, 2, 1), int(g["k"])
    assert ops.pcu.cosine_supported(k, xyz, new)
    idx, dist = ops.pcu.knn_point_cosine_with_dist(k, xyz, new)
    ref_vals = torch.as_tensor(g["ref_vals"]).cuda()
    assert float((dist - ref_vals[..., :k]).abs().max()) <= COS_ATOL
    clear = (ref_vals[..., k] - ref_vals[..., k - 1]) > COS_GAP
    ref_idx = torch.as_tensor(g["ref_idx"].astype(np.int64)).cuda()
    same = (idx.sort(-1)[0] == ref_idx.sort(-1)[0]).all(-1)
    assert bool(same[clear].all())


@pytest.mark.parametrize("B,S,N,C,k,permuted", [(1, 2048, 2048, 64, 16, True), (1, 512, 512, 128, 16, True),
                                                 (1, 256, 256, 256, 16, True), (2, 300, 1000, 64, 16, False),
                                                 (1, 129, 4096, 32, 32, False), (3, 77, 257, 16, 5, True),
                                                 (1, 1, 16, 512, 16, False), (2, 1000, 130, 48, 32, True)])
def test_knn_point_cosine_vs_reference_function(ops, orc, B, S, N, C, k, permuted):
    """Against the reference's cosine_distance + topk (models/pointconv_util.py:111-127,142-153,
    restated in oracle/torch_port.py) executed by CUDA torch on the same GPU, every row, and
    against the oracle; with a checkout, the installed helper too."""
    g = torch.Generator().manual_seed(B * 1000 + S + N + C)
    xyz = torch.randn(B, C, N, generator=g) if permuted else torch.randn(B, N, C, generator=g)
    new = torch.randn(B, C, S, generator=g) if permuted else torch.randn(B, S, C, generator=g)
    xd = xyz.cuda().permute(0, 2, 1) if permuted else xyz.cuda()
    nd = new.cuda().permute(0, 2, 1) if permuted else new.cuda()
    idx, dist = ops.pcu.knn_point_cosine_with_dist(k, xd, nd)
    assert idx.dtype == torch.int64 and tuple(idx.shape) == (B, S, k)
    frac = check_cosine(idx, dist, torch_port.cosine_distance(nd, xd), k)
    assert frac > 0.8
    oi, od = orc.knn_cosine(k, xd.contiguous().cpu().numpy(), nd.contiguous().cpu().numpy())
    np.testing.assert_allclose(dist.cpu().numpy(), od, rtol=0, atol=COS_ATOL)
    from baseline import fetch_ref
    if fetch_ref.root() is not None:
        # the installed replacement routes through the same kernel and returns the same indices
        import importlib
        import mocopci_b200
        mocopci_b200.install(reference_root=fetch_ref.root())
        ref = importlib.import_module("models.pointconv_util")
        assert hasattr(ref.knn_point_cosine, "__b200pci_original__")
        assert torch.equal(ref.knn_point_cosine(k, xd, nd), idx)


def test_knn_point_cosine_duplicates_and_unsupported(ops):
    """Duplicated feature rows (duplicated points) are exact ties: the lowest index wins. Shapes the
    kernel does not cover raise; with a checkout, they fall back to the reference's own torch code
    through the installed helper."""
    g = torch.Generator().manual_seed(5)
    base = torch.randn(1, 300, 64, generator=g)
    xyz = torch.cat([base, base], 1).cuda()          # ref j and j + 300 are identical
    idx, dist = ops.pcu.knn_point_cosine_with_dist(4, xyz, base.cuda())
    assert bool((idx[0, :, 0] == torch.arange(300, device="cuda")).all())       # itself, the lower copy
    assert bool((idx[0, :, 1] == torch.arange(300, device="cuda") + 300).all()) # then the duplicate
    assert float(dist[0, :, :2].abs().max()) <= COS_ATOL
    odd = torch.randn(1, 100, 50, generator=g).cuda()                            # C % 16 != 0
    assert not ops.pcu.cosine_supported(8, odd, odd)
    with pytest.raises(RuntimeError):
        ops.pcu.knn_point_cosine(8, odd, odd)
    from baseline import fetch_ref
    if fetch_ref.root() is not None:
        import importlib
        import mocopci_b200
        mocopci_b200.install(reference_root=fetch_ref.root())
        ref = importlib.import_module("models.pointconv_util")
        out = ref.knn_point_cosine(8, odd, odd)                                  # the reference's own code
        assert tuple(out.shape) == (1, 100, 8)


def test_knn_k_gt_n_raises(ops):
    xyz = dev(ops.synth.uniform_cloud(1, 1, 8))
    with pytest.raises(RuntimeError):
        ops.pcu.knn_point(16, xyz, xyz)


def test_knn_full_size_properties(ops):
    """BASELINE size (16384 x 16384, k=16): size-independent properties."""
    a, b = ops.synth.frame_pairs(0, 2)
    a, b = a.cuda(), b.cuda()
    idx, dist = ops.pcu.knn_point_with_dist(16, a, b)
    assert int(idx.min()) >= 0 and int(idx.max()) < 16384
    assert bool((dist[..., 1:] >= dist[..., :-1]).all())           # sorted
    assert bool((idx.sort(-1)[0][..., 1:] != idx.sort(-1)[0][..., :-1]).all())  # distinct
    # idempotence / self-consistency: self-KNN returns each point among its own neighbours
    sidx, sd = ops.pcu.knn_point_with_dist(16, a, a)
    me = torch.arange(16384, device="cuda").view(1, -1, 1)
    assert bool((sidx == me).any(-1).all())
    # k=16 result is a prefix of k=32
    idx32 = ops.pcu.knn_point(32, a, b)
    assert bool((idx32[..., :16] == idx).all())
    # distances recomputed with torch's expanded form on the selected pairs match to 1e-4 abs
    sel = torch.gather(a.unsqueeze(1).expand(-1, 16384, -1, -1), 2,
                       idx.unsqueeze(-1).expand(-1, -1, -1, 3))
    d_direct = ((sel - b.unsqueeze(2)) ** 2).sum(-1)
    assert float((d_direct - dist).abs().max()) < 5e-2  # expanded form cancellation at 80 m range


# ------------------------------------------------------------------------------------------
# pytorch3d.ops.knn_points shim (direct form)
# ------------------------------------------------------------------------------------------
def test_knn_points_direct(ops, orc):
    p1 = ops.synth.uniform_cloud(3, 2, 400).numpy()
    p2 = ops.synth.uniform_cloud(4, 2, 777).numpy()
    r = ops.chamfer.knn_points(dev(p1), dev(p2), K=16, return_nn=True)
    oi, od = orc.knn_form(2, 16, p2, p1)
    np.testing.assert_array_equal(r.idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(r.dists.cpu().numpy()), bits(od))
    nn = np.take_along_axis(p2[:, None].repeat(400, 1), oi[..., None].repeat(3, -1), axis=2)
    np.testing.assert_array_equal(r.knn.cpu().numpy(), nn)


# ------------------------------------------------------------------------------------------
# three_nn / three_interpolate (T1, T2)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n,m", [(2, 256, 64), (1, 1024, 256), (2, 1000, 333), (1, 40, 2), (1, 33, 1),
                                   (1, 3000, 2500), (2, 5000, 4096)])
def test_three_nn(ops, orc, B, n, m, request):
    u = ops.synth.uniform_cloud(n, B, n).numpy()
    kn = ops.synth.uniform_cloud(m + 7, B, m).numpy()
    dist, idx = ops.p2u.three_nn(dev(u), dev(kn))
    od2, oi = orc.three_nn(u, kn)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(dist.cpu().numpy()), bits(np.sqrt(od2)))


def test_three_nn_vs_reference_kernel(ops, orc):
    """The pybind-style entry point on a LiDAR frame: the oracle's squared distances and indices bit
    for bit, and the kernel snapshot."""
    a, _ = ops.synth.frame_pair(1, 4096)
    known = a[:1024][None].cuda().contiguous()
    unknown = a[None].cuda().contiguous()
    d2 = torch.empty((1, 4096, 3), device="cuda")
    idx = torch.empty((1, 4096, 3), dtype=torch.int32, device="cuda")
    ops.p2c.three_nn_wrapper(1, 4096, 1024, unknown, known, d2, idx)
    od2, oi = orc.three_nn(unknown.cpu().numpy(), known.cpu().numpy())
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(d2.cpu().numpy()), bits(od2))
    snapshot.check("three_nn/idx", idx)
    snapshot.check("three_nn/d2", d2)


@pytest.mark.parametrize("B,n,m", [(2, 256, 64), (1, 4096, 1024), (1, 16384, 4096), (1, 50, 3)])
def test_three_nn_weights_fused(ops, orc, B, n, m):
    """T3: three_nn + the caller-side inverse-distance weights (pointnet2_modules.py:139-144) in one
    call, BITWISE against the reference's composition -- its own three_nn wrapper followed by the
    same torch expressions on the GPU -- and against the oracle."""
    a = ops.synth.uniform_cloud(n + m, B, n, -3.0, 3.0)
    unknown, known = a.cuda(), a[:, :m].contiguous().cuda()
    weight, idx, dist = ops.own.three_nn_weights(unknown, known)
    rdist, ridx = ops.p2u.three_nn(unknown, known)               # sqrt(dist2), pointnet2_utils.py:97
    dist_recip = 1.0 / (rdist + 1e-8)                            # pointnet2_modules.py:140
    norm = torch.sum(dist_recip, dim=2, keepdim=True)            # :141
    rweight = dist_recip / norm                                  # :142
    assert torch.equal(idx, ridx)
    assert torch.equal(dist.view(torch.int32), rdist.view(torch.int32))
    assert torch.equal(weight.view(torch.int32), rweight.view(torch.int32))
    od2, oi = orc.three_nn(a.numpy(), a[:, :m].numpy())
    odist, ow = orc.three_nn_weights(od2)
    np.testing.assert_array_equal(bits(weight.cpu().numpy()), bits(ow))


@pytest.mark.parametrize("B,C,m,n", [(2, 128, 64, 256), (1, 5, 33, 1000), (2, 19, 1024, 4096),
                                     (1, 128, 4096, 16384), (2, 64, 1000, 5000)])
def test_three_interpolate_fwd_bwd(ops, orc, B, C, m, n):
    g = torch.Generator().manual_seed(C)
    feat = torch.randn(B, C, m, generator=g)
    idx = torch.randint(0, m, (B, n, 3), generator=g, dtype=torch.int32)
    w = torch.rand(B, n, 3, generator=g)
    w = w / w.sum(-1, keepdim=True)
    fd = feat.cuda().requires_grad_(True)
    out = ops.p2u.three_interpolate(fd, idx.cuda(), w.cuda())
    ref = orc.three_interpolate(feat.numpy(), idx.numpy(), w.numpy())
    np.testing.assert_array_equal(bits(out.detach().cpu().numpy()), bits(ref))      # bitwise
    snapshot.check(f"three_interpolate/{B}-{C}-{m}-{n}", out)
    go = torch.randn(B, C, n, generator=g)
    out.backward(go.cuda())
    gref = orc.three_interpolate_grad(go.numpy(), idx.numpy(), w.numpy(), m)
    # atomicAdd order differs run to run (also in the reference): 1e-5 relative + 1e-5 absolute
    np.testing.assert_allclose(fd.grad.cpu().numpy(), gref, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------
# gather / group (F2, G1, K3, K4)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,C,N,M", [(2, 3, 1000, 256), (1, 64, 4096, 1023), (3, 17, 50, 7)])
def test_gather_fwd_bwd(ops, orc, B, C, N, M):
    g = torch.Generator().manual_seed(N)
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, M), generator=g, dtype=torch.int32)
    fd = feat.cuda().requires_grad_(True)
    out = ops.p2u.gather_operation(fd, idx.cuda())
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.gather(feat.numpy(), idx.numpy()))
    snapshot.check(f"gather/{B}-{C}-{N}-{M}", out)
    go = torch.randn(B, C, M, generator=g)
    out.backward(go.cuda())
    np.testing.assert_allclose(fd.grad.cpu().numpy(), orc.gather_grad(go.numpy(), idx.numpy(), N),
                               rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("B,C,N,np_,ns", [(2, 3, 1000, 128, 32), (1, 35, 2048, 300, 16),
                                           (2, 7, 64, 33, 3), (1, 128, 4096, 1024, 32)])
def test_group_fwd_bwd(ops, orc, B, C, N, np_, ns):
    g = torch.Generator().manual_seed(np_)
    feat = torch.randn(B, C, N, generator=g)
    idx = torch.randint(0, N, (B, np_, ns), generator=g, dtype=torch.int32)
    fd = feat.cuda().requires_grad_(True)
    out = ops.p2u.grouping_operation(fd, idx.cuda())
    np.testing.assert_array_equal(out.detach().cpu().numpy(), orc.group(feat.numpy(), idx.numpy()))
    snapshot.check(f"group/{B}-{C}-{N}-{np_}-{ns}", out)
    go = torch.randn(B, C, np_, ns, generator=g)
    out.backward(go.cuda())
    np.testing.assert_allclose(fd.grad.cpu().numpy(), orc.group_grad(go.numpy(), idx.numpy(), N),
                               rtol=1e-4, atol=1e-4)


def test_index_points_helpers(ops, orc):
    pts = ops.synth.uniform_cloud(9, 2, 500)
    feats = torch.randn(2, 500, 35, generator=torch.Generator().manual_seed(1))
    idx = ops.pcu.knn_point(16, pts.cuda(), pts.cuda())
    grouped = ops.pcu.index_points_group(feats.cuda(), idx)
    assert tuple(grouped.shape) == (2, 500, 16, 35)
    exp = torch.gather(feats.unsqueeze(1).expand(-1, 500, -1, -1), 2,
                       idx.cpu().unsqueeze(-1).expand(-1, -1, -1, 35))
    assert torch.equal(grouped.cpu(), exp)
    fidx = ops.p2u.furthest_point_sample(pts.cuda(), 64)
    gathered = ops.pcu.index_points_gather(pts.cuda(), fidx)
    exp = torch.gather(pts, 1, fidx.cpu().long().unsqueeze(-1).expand(-1, -1, 3))
    assert torch.equal(gathered.cpu(), exp) and gathered.is_contiguous()


@pytest.mark.parametrize("B,N,S,K,C,permuted", [(2, 500, 300, 16, 35, False), (1, 2048, 777, 32, 64, False),
                                                 (2, 333, 100, 3, 3, False), (1, 1000, 500, 16, 128, True),
                                                 (2, 64, 10, 8, 5, True)])
def test_index_points_group_fused_fwd_bwd(ops, B, N, S, K, C, permuted):
    """K3: the fused [B,N,C] row gather against the reference's own composition
    (models/pointconv_util.py:181-192 restated with torch ops), strided (permuted) inputs,
    int64 indices, and its gradient against autograd through torch.gather."""
    g = torch.Generator().manual_seed(S + C)
    base = torch.randn(B, C, N, generator=g) if permuted else torch.randn(B, N, C, generator=g)
    idx = torch.randint(0, N, (B, S, K), generator=g, dtype=torch.int64)
    pd = base.cuda().requires_grad_(True)
    view = pd.permute(0, 2, 1) if permuted else pd
    out = ops.pcu.index_points_group(view, idx.cuda())
    assert tuple(out.shape) == (B, S, K, C) and out.is_contiguous()
    pr = base.clone().requires_grad_(True)
    vr = pr.permute(0, 2, 1) if permuted else pr
    exp = torch.gather(vr.unsqueeze(1).expand(-1, S, -1, -1), 2, idx.unsqueeze(-1).expand(-1, -1, -1, C))
    assert torch.equal(out.detach().cpu(), exp.detach())
    go = torch.randn(B, S, K, C, generator=g)
    out.backward(go.cuda())
    exp.backward(go)
    np.testing.assert_allclose(pd.grad.cpu().numpy(), pr.grad.numpy(), rtol=1e-4, atol=1e-4)
    # int32 indices (what the pointnet2 ops produce) give the same rows
    out32 = ops.pcu.index_points_group(view.detach(), idx.int().cuda())
    assert torch.equal(out32, out.detach())


@pytest.mark.parametrize("B,N,S,K,D,permuted", [(2, 500, 500, 16, 32, False), (1, 4096, 1024, 32, 64, True),
                                                 (2, 300, 77, 8, 0, False), (1, 2048, 2048, 32, 35, True),
                                                 (1, 64, 64, 64, 5, False), (1, 100, 33, 5, 6, False),
                                                 (1, 256, 64, 4, 700, False), (1, 128, 16, 4, 3000, False),
                                                 (1, 512, 512, 16, 128, True)])
def test_group_query_fused(ops, orc, B, N, S, K, D, permuted):
    """f1: group / group_query (models/pointconv_util.py:194-241) as ONE gather-subtract-concatenate
    kernel after the neighbour search, bitwise against the composition the reference writes
    (gather xyz - centre | gather points) on the same indices; the autograd path gives the same values;
    and the neighbours are those of the reference's knn_point in its CUDA torch arithmetic (the
    oracle's form 5); with a checkout, the reference's own group_query (imported, unpatched)
    agrees as neighbour SETS."""
    g = torch.Generator().manual_seed(N + S + D)
    s_xyz = (torch.rand(B, N, 3, generator=g) * 10).cuda()
    xyz = s_xyz if S == N else (torch.rand(B, S, 3, generator=g) * 10).cuda()
    pts = None
    if D:
        pts = torch.randn(B, D, N, generator=g).cuda().permute(0, 2, 1) if permuted else torch.randn(B, N, D, generator=g).cuda()
    new_points, rel = ops.pcu.group_query(K, s_xyz, xyz, pts)
    idx = ops.pcu.knn_point(K, s_xyz, xyz)
    exp_rel = torch.gather(s_xyz.unsqueeze(1).expand(-1, S, -1, -1), 2, idx.unsqueeze(-1).expand(-1, -1, -1, 3)) - xyz.unsqueeze(2)
    assert torch.equal(rel, exp_rel) and rel.is_contiguous()
    if D:
        exp_pts = torch.gather(pts.unsqueeze(1).expand(-1, S, -1, -1), 2, idx.unsqueeze(-1).expand(-1, -1, -1, D))
        assert torch.equal(new_points, torch.cat([exp_rel, exp_pts], -1)) and new_points.is_contiguous()
    else:
        assert new_points is rel
    # autograd path: same values, and gradients flow to the features
    if D:
        pg = pts.detach().clone().requires_grad_(True)
        np2, rel2 = ops.pcu.group_query(K, s_xyz, xyz, pg)
        assert torch.equal(np2.detach(), new_points) and torch.equal(rel2, rel)
        np2.sum().backward()
        assert pg.grad is not None and float(pg.grad.abs().sum()) > 0
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.knn_form(5, K, s_xyz.cpu().numpy(), xyz.cpu().numpy())[0])
    from baseline import fetch_ref
    if fetch_ref.root() is None:
        return
    # the reference's own function (torch KNN, unsorted neighbours): same sets per query
    import importlib
    import mocopci_b200
    from mocopci_b200 import shim
    mocopci_b200.install(reference_root=fetch_ref.root())
    ref = importlib.import_module("models.pointconv_util")
    orig = getattr(ref.group_query, shim._MARK)
    saved = {n: getattr(ref, n) for n in ("knn_point", "index_points_group")}
    try:   # run the reference's group_query on the reference's own helpers
        for n in saved:
            setattr(ref, n, getattr(saved[n], shim._MARK, saved[n]))
        r_np, r_rel = orig(K, s_xyz, xyz, pts)
    finally:
        for n, f in saved.items():
            setattr(ref, n, f)
    differ = (r_rel.sort(dim=2)[0] != rel.sort(dim=2)[0]).any(-1).any(-1)
    assert int(differ.sum()) <= max(1, B * S // 200)          # only rows with a tie at the k-th distance
    if D:
        d2 = (r_np.sort(dim=2)[0] != new_points.sort(dim=2)[0]).any(-1).any(-1)
        assert int(d2.sum()) <= max(1, B * S // 200)
    assert hasattr(ref.group, shim._MARK) and hasattr(ref.group_query, shim._MARK)
    a1, a2 = ref.group(min(K, N), s_xyz, pts)
    b1, b2 = ops.pcu.group(min(K, N), s_xyz, pts)
    assert torch.equal(a1, b1) and torch.equal(a2, b2)


# ------------------------------------------------------------------------------------------
# FPS (F1)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,M", [(2, 1000, 100), (1, 2048, 512), (3, 257, 64), (1, 16, 16),
                                    (2, 4096, 300), (1, 5000, 64), (1, 1, 4), (1, 3, 5)])
def test_fps_vs_oracle(ops, orc, B, N, M):
    xyz = ops.synth.uniform_cloud(N + M, B, N)
    idx = ops.p2u.furthest_point_sample(xyz.cuda(), M)
    oi, _ = orc.fps(xyz.numpy(), M)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)


def test_fps_ties_vs_reference_kernel(ops, orc):
    # integer grid with duplicates: many exactly equal distances -> exercises the tie order
    for N, M in ((1200, 200), (512, 128), (3000, 256)):
        xyz = ops.synth.tie_stress_cloud(N, 2, N, grid=3).cuda()
        idx = ops.p2u.furthest_point_sample(xyz, M)
        snapshot.check(f"fps_ties/{N}-{M}", idx)
        np.testing.assert_array_equal(idx.cpu().numpy(), orc.fps(xyz.cpu().numpy(), M)[0])


def test_fps_single_cta_and_cluster_kernels_agree(ops, orc):
    from mocopci_b200 import _lib
    for N, M in ((4096, 300), (5000, 64), (16384, 200), (20000, 50)):
        xyz = ops.synth.tie_stress_cloud(N + 1, 2, N, grid=5).cuda()
        a = ops.p2u.furthest_point_sample(xyz, M)          # cluster kernel (N >= 4096)
        try:
            _lib.check(_lib.lib.b200pci_debug_set(5, 1))
            b = ops.p2u.furthest_point_sample(xyz, M)      # single-CTA kernel
        finally:
            _lib.check(_lib.lib.b200pci_debug_set(5, 0))
        assert torch.equal(a, b), f"N={N}"
        if N <= 5000:
            np.testing.assert_array_equal(a.cpu().numpy(), orc.fps(xyz.cpu().numpy(), M)[0])


def test_fps_full_size_vs_reference_kernel(ops, orc):
    """16384 -> 4096 on two LiDAR frames: the oracle's indices, and indices and the distance buffer
    bit for bit against the kernel snapshot."""
    a, _ = ops.synth.frame_pairs(0, 2)
    oi = orc.fps(a.numpy(), 4096)[0]
    a = a.cuda()
    temp = torch.full((2, 16384), 1e10, device="cuda")
    idx = torch.empty((2, 4096), dtype=torch.int32, device="cuda")
    ops.p2c.furthest_point_sampling_wrapper(2, 16384, 4096, a, temp, idx)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    snapshot.check("fps_full/idx", idx)
    snapshot.check("fps_full/temp", temp)


# ------------------------------------------------------------------------------------------
# ball_query (Q1, G2)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,M,r,ns", [(2, 1000, 128, 0.3, 32), (1, 2048, 500, 0.05, 16),
                                         (2, 600, 77, 5.0, 8), (1, 513, 300, 0.2, 64)])
def test_ball_query_vs_oracle(ops, orc, B, N, M, r, ns):
    xyz = ops.synth.uniform_cloud(N, B, N)
    new = xyz[:, :M].contiguous()
    idx = ops.p2u.ball_query(r, ns, xyz.cuda(), new.cuda())
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.ball_query(r, ns, xyz.numpy(), new.numpy()))


def test_ball_query_dense_and_forced_redo(ops, orc):
    """Dense cloud with a radius that catches hundreds of refs per query (long pending lists,
    early stop at nsample) and the exact redo kernel forced for every query (test hook 6)."""
    from mocopci_b200 import _lib
    xyz = ops.synth.uniform_cloud(77, 2, 6000, -1.0, 1.0)
    new = xyz[:, :333].contiguous()
    want = orc.ball_query(0.6, 16, xyz.numpy(), new.numpy())
    np.testing.assert_array_equal(ops.p2u.ball_query(0.6, 16, xyz.cuda(), new.cuda()).cpu().numpy(), want)
    try:
        _lib.check(_lib.lib.b200pci_debug_set(6, 1))
        got = ops.p2u.ball_query(0.6, 16, xyz.cuda(), new.cuda())
        far = ops.p2u.ball_query(0.01, 16, xyz.cuda(), (new + 100.0).cuda())
    finally:
        _lib.check(_lib.lib.b200pci_debug_set(6, 0))
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    assert int(far.abs().sum()) == 0


@pytest.mark.parametrize("r,ns,shift", [(3.0, 128, 0.0), (1.5, 128, 0.0), (0.4, 96, 500.0), (6.0, 200, 0.0)])
def test_ball_query_large_nsample_split_overflow(ops, orc, r, ns, shift):
    """nsample > the 96-entry pending lists with the refs split over several CTAs (16384 refs, few
    queries): a split whose list overflowed must send the query to the exact redo instead of
    letting later splits fill the slots with higher indices. `shift` moves the cloud far from the
    origin, where the filter's relative slack flags many false-positive steps."""
    a, _ = ops.synth.frame_pairs(6, 1, 16384)
    a = (a + shift).contiguous()
    new = a[:, ::40].contiguous()                      # 410 queries: B*M small -> nsplit > 1
    got = ops.p2u.ball_query(r, ns, a.cuda(), new.cuda())
    np.testing.assert_array_equal(got.cpu().numpy(), orc.ball_query(r, ns, a.numpy(), new.numpy()))
    snapshot.check(f"ball_query_split/{r}-{ns}-{shift}", got)


def test_ball_query_lidar_vs_reference_kernel(ops, orc):
    a, _ = ops.synth.frame_pairs(2, 2, 8192)
    a = a.cuda()
    centres = ops.pcu.index_points_gather(a, ops.p2u.furthest_point_sample(a, 1024))
    idx = ops.p2u.ball_query(0.5, 32, a, centres)
    np.testing.assert_array_equal(idx.cpu().numpy(), orc.ball_query(0.5, 32, a.cpu().numpy(), centres.cpu().numpy()))
    snapshot.check("ball_query_lidar", idx)
    # no-hit rows stay all zero (pointnet2_utils.py:218)
    far = centres + 1000.0
    assert int(ops.p2u.ball_query(0.5, 32, a, far).abs().sum()) == 0


def test_query_and_group(ops, orc):
    a, _ = ops.synth.frame_pairs(4, 1, 4096)
    a = a.cuda()
    feats = torch.randn(1, 16, 4096, generator=torch.Generator().manual_seed(4)).cuda()
    centres = ops.pcu.index_points_gather(a, ops.p2u.furthest_point_sample(a, 256))
    out = ops.p2u.QueryAndGroup(2.0, 16)(a, centres, feats)
    assert tuple(out.shape) == (1, 19, 256, 16)
    # pointnet2_utils.py:250-264 on the oracle: ball_query, group of the cloud minus the centres |
    # group of the features
    a_np, c_np = a.cpu().numpy(), centres.cpu().numpy()
    oidx = orc.ball_query(2.0, 16, a_np, c_np)
    gx = orc.group(np.ascontiguousarray(a_np.transpose(0, 2, 1)), oidx) - c_np.transpose(0, 2, 1)[..., None]
    want = np.concatenate([gx, orc.group(feats.cpu().numpy(), oidx)], 1)
    np.testing.assert_array_equal(bits(out.cpu().numpy()), bits(want))
    snapshot.check("query_and_group", out)


@pytest.mark.parametrize("B,N,M,ns,C,use_xyz", [(2, 4096, 512, 32, 64, True), (1, 1000, 77, 5, 3, True),
                                                   (3, 300, 33, 7, 0, True), (2, 2048, 256, 16, 20, False),
                                                   (1, 16384, 4096, 32, 128, True)])
def test_query_group_fused_equals_reference_composition(ops, B, N, M, ns, C, use_xyz):
    """b200pci_query_group (own API: ops.query_and_group without autograd) writes the concatenated
    QueryAndGroup tensor in two launches; it must equal, bit for bit, the composition of
    pointnet2_utils.py:250-264 -- grouping_operation on the transposed cloud, minus the centres,
    grouping_operation on the features, torch.cat -- on the same ball_query indices, for group
    counts that are not multiples of four (scalar tail), without features and without xyz; and the
    autograd route (inputs that require grad) gives the same values. The reference_wrappers variant
    takes the composition from the reference's QueryAndGroup module itself."""
    from mocopci_b200 import ops as own
    g = torch.Generator().manual_seed(N + M + C)
    xyz = (torch.rand(B, N, 3, generator=g) * 8).cuda()
    centres = xyz[:, torch.randperm(N, generator=g)[:M]].contiguous()
    feats = torch.randn(B, C, N, generator=g).cuda() if C else None
    got = own.query_and_group(1.0, ns, xyz, centres, feats, use_xyz)
    idx = own.ball_query(1.0, ns, xyz, centres)
    rel = own.grouping_operation(xyz.transpose(1, 2).contiguous(), idx) - centres.transpose(1, 2).unsqueeze(-1)
    want = rel if feats is None else (torch.cat([rel, own.grouping_operation(feats, idx)], 1) if use_xyz
                                      else own.grouping_operation(feats, idx))
    if ops.api != "own_api":
        ref = ops.p2u.QueryAndGroup(1.0, ns, use_xyz=use_xyz)(xyz, centres, feats)
        assert torch.equal(ref, want)
        want = ref
    assert got.is_contiguous() and got.shape == want.shape and torch.equal(got, want)
    if feats is not None:
        fg = feats.clone().requires_grad_(True)
        via_autograd = own.query_and_group(1.0, ns, xyz, centres, fg, use_xyz)
        assert torch.equal(via_autograd.detach(), want)
        via_autograd.sum().backward()
        assert fg.grad is not None and float(fg.grad.abs().sum()) > 0


# ------------------------------------------------------------------------------------------
# Chamfer (C1)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,M", [(2, 500, 700), (1, 2048, 2048), (3, 64, 33), (1, 3000, 2500)])
def test_chamfer_vs_oracle(ops, orc, B, N, M):
    x = ops.synth.uniform_cloud(N, B, N)
    y = ops.synth.uniform_cloud(M + 1, B, M)
    xd, yd = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
    loss, _ = ops.chamfer.chamfer_distance(xd, yd)
    ol, dx, dy, ix, iy = orc.chamfer(x.numpy(), y.numpy())
    assert abs(float(loss) - ol) <= 1e-5 * abs(ol)  # 1e-5 relative (north_star)
    loss.backward()
    # analytic gradient from the oracle's NN indices
    xt, yt = x.double().requires_grad_(True), y.double().requires_grad_(True)
    ixt, iyt = torch.as_tensor(ix).long(), torch.as_tensor(iy).long()
    l = 0
    for b in range(B):
        l = l + ((xt[b] - yt[b][ixt[b]]) ** 2).sum(-1).mean() + ((yt[b] - xt[b][iyt[b]]) ** 2).sum(-1).mean()
    (l / B).backward()
    np.testing.assert_allclose(xd.grad.cpu().numpy(), xt.grad.float().numpy(), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(yd.grad.cpu().numpy(), yt.grad.float().numpy(), rtol=1e-4, atol=1e-7)


def test_chamfer_loss_layout_and_full_size(ops):
    a, b = ops.synth.frame_pairs(0, 1)
    pc1, pc2 = a.cuda().permute(0, 2, 1), b.cuda().permute(0, 2, 1)   # [B,3,N] views
    l12 = ops.chamfer.chamfer_loss(pc1, pc2)
    l21 = ops.chamfer.chamfer_loss(pc2, pc1)
    assert abs(float(l12) - float(l21)) <= 1e-6 * abs(float(l12))       # symmetry
    assert float(ops.chamfer.chamfer_loss(pc1, pc1)) == 0.0             # identity
    # against a chunked torch evaluation of the same definition, 1e-5 relative
    d = torch.cdist(b.cuda()[0].double(), a.cuda()[0].double()) ** 2
    ref = d.min(1)[0].mean() + d.min(0)[0].mean()
    assert abs(float(l12) - float(ref)) <= 1e-5 * float(ref)


# ------------------------------------------------------------------------------------------
# EMD (E1-E4)
# ------------------------------------------------------------------------------------------
def test_emd_known_answer(ops):
    """The reference's only results-pinning vector: models/EMD/test_emd_loss.py:7-43."""
    p1 = torch.tensor([[[1.7, -0.1, 0.1], [0.1, 1.2, 0.3]]]).repeat(3, 1, 1).cuda().requires_grad_(True)
    p2 = torch.tensor([[[0.3, 1.8, 0.2], [1.2, -0.2, 0.3]]]).repeat(3, 1, 1).cuda().requires_grad_(True)
    d = ops.emd.earth_mover_distance(p1, p2, transpose=False)
    loss = d[0] / 2 + d[1] * 2 + d[2] / 3
    loss.backward()
    q1, q2 = p1.detach().clone().requires_grad_(True), p2.detach().clone().requires_grad_(True)
    gt = (((q1[0, 0] - q2[0, 1]) ** 2).sum() + ((q1[0, 1] - q2[0, 0]) ** 2).sum()) / 2 + \
         (((q1[1, 0] - q2[1, 1]) ** 2).sum() + ((q1[1, 1] - q2[1, 0]) ** 2).sum()) * 2 + \
         (((q1[2, 0] - q2[2, 1]) ** 2).sum() + ((q1[2, 1] - q2[2, 0]) ** 2).sum()) / 3
    gt.backward()
    assert abs(float(loss) - float(gt)) <= 1e-5 * float(gt)     # 2.0116667
    assert abs(float(d[0]) - 0.71) < 1e-5
    np.testing.assert_allclose(p1.grad.cpu().numpy(), q1.grad.cpu().numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(p2.grad.cpu().numpy(), q2.grad.cpu().numpy(), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("B,n,m", [(2, 256, 256), (1, 1000, 500), (2, 300, 1200), (1, 2048, 2048)])
def test_emd_vs_reference_kernel(ops, orc, B, n, m):
    """approxmatch / matchcost / matchcost_backward against the kernel snapshot (match and grad1 bit
    for bit), and the cost against the oracle (libm expf there, ex2.approx here: 1e-3 relative)."""
    x1 = (ops.synth.uniform_cloud(n, B, n) * 0.5).cuda()
    x2 = (ops.synth.uniform_cloud(m + 3, B, m) * 0.5).cuda()
    key = f"emd/{B}-{n}-{m}"
    match = ops.emd_cuda.approxmatch_forward(x1, x2)
    snapshot.check(key + "/match", match)                                   # bitwise
    cost = ops.emd_cuda.matchcost_forward(x1, x2, match)
    snapshot.check(key + "/cost", cost, rtol=1e-5)                          # 1e-5 relative
    x1n, x2n = x1.cpu().numpy(), x2.cpu().numpy()
    np.testing.assert_allclose(cost.cpu().numpy(), orc.emd_matchcost(x1n, x2n, orc.emd_approxmatch(x1n, x2n)),
                               rtol=1e-3)
    gc = (torch.rand(B, generator=torch.Generator().manual_seed(n + m)) + 0.5).cuda()
    g1, g2 = ops.emd_cuda.matchcost_backward(gc, x1, x2, match)
    snapshot.check(key + "/grad1", g1)
    snapshot.check(key + "/grad2", g2, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("B,n,m", [(2, 256, 256), (1, 1000, 500), (2, 300, 1200), (1, 4096, 4096)])
def test_emd_cost_fused_vs_reference_kernel(ops, B, n, m):
    """Forward-only emd_cost (no match matrix) against approxmatch + matchcost, in the kernel
    snapshot and run now: 1e-5 relative (north_star's tolerance for EMD values)."""
    x1 = (ops.synth.uniform_cloud(n + 1, B, n) * 0.5).cuda()
    x2 = (ops.synth.uniform_cloud(m + 4, B, m) * 0.5).cuda()
    cost = ops.emd_cuda.emd_cost(x1, x2)
    snapshot.check(f"emd_cost/{B}-{n}-{m}", cost, rtol=1e-5)
    mine = ops.emd_cuda.matchcost_forward(x1, x2, ops.emd_cuda.approxmatch_forward(x1, x2))
    np.testing.assert_allclose(cost.cpu().numpy(), mine.cpu().numpy(), rtol=1e-5)


def test_emd_metric_vs_reference_kernel(ops, orc):
    """E4: EMD(pc1, pc2) = mean(cost) / M (models/utils.py:223-235) on a LiDAR frame pair, through the
    API under test, against the same formula on the kernel snapshot's cost (1e-5 relative) and on
    the oracle's (1e-3 relative: libm expf there, ex2.approx here)."""
    a, b = ops.synth.frame_pair(0, 4096)
    pc1, pc2 = a.cuda().T[None].contiguous(), b.cuda().T[None].contiguous()
    v = ops.emd.EMD(pc1, pc2)
    ref = snapshot.get("emd_metric")[0]
    assert abs(float(v) - float(ref)) <= 1e-5 * abs(float(ref))
    x1, x2 = a[None].numpy(), b[None].numpy()
    oref = float(orc.emd_matchcost(x1, x2, orc.emd_approxmatch(x1, x2)).mean()) / 4096
    assert abs(float(v) - oref) <= 1e-3 * abs(oref)


def test_emd_vs_oracle_small(ops, orc):
    x1 = ops.synth.uniform_cloud(1, 2, 128)
    x2 = ops.synth.uniform_cloud(2, 2, 128)
    match = ops.emd_cuda.approxmatch_forward(x1.cuda(), x2.cuda())
    om = orc.emd_approxmatch(x1.numpy(), x2.numpy())
    # the oracle uses libm expf, the GPU ex2.approx: tolerance, not bitwise
    np.testing.assert_allclose(match.cpu().numpy(), om, rtol=2e-2, atol=1e-5)
    cost = ops.emd_cuda.matchcost_forward(x1.cuda(), x2.cuda(), match)
    np.testing.assert_allclose(cost.cpu().numpy(), orc.emd_matchcost(x1.numpy(), x2.numpy(), om),
                               rtol=1e-4)


def test_emd_metric(ops):
    a, b = ops.synth.frame_pair(0, 2048)
    v = ops.emd.EMD(a.cuda().T[None], b.cuda().T[None])
    assert v.dim() == 0 and float(v) > 0
    assert float(ops.emd.EMD(a.cuda().T[None], a.cuda().T[None])) < 1e-6


# ------------------------------------------------------------------------------------------
# data path (f4)
# ------------------------------------------------------------------------------------------
def test_nldrive_dataset_device_staging_equals_reference_rows(ops, ref_root, tmp_path):
    """mocopci_b200.data.NLDriveDataset with device="cuda" (host gather into one pinned block + one
    H2D copy) and with gather_on_device=True (raw frame + indices shipped, rows gathered by
    b200pci_index_points_rows): the same rows as the reference's CPU tensors under the same seed."""
    if ops.api != "own_api":
        pytest.skip("own API only")
    import importlib
    from mocopci_b200 import data as ours
    from tests.test_host_cpu import _write_nldrive_fixture
    sys.path.insert(0, ref_root)
    try:
        ref = importlib.import_module("data.no_norm_datasets")
    finally:
        sys.path.remove(ref_root)
    root = str(tmp_path)
    lst = _write_nldrive_fixture(root, [20000, 900, 16384, 30000, 700, 16385, 2048, 64, 40000], seed=3)
    a = ref.NLDriveDataset(root, lst, num_points=16384, interval=4, num_frames=4)
    for kw in ({"device": "cuda"}, {"device": "cuda", "gather_on_device": True}):
        b = ours.NLDriveDataset(root, lst, num_points=16384, interval=4, num_frames=4, **kw)
        for index in (0, 1):
            np.random.seed(7 + index)
            ia, ga = a[index]
            np.random.seed(7 + index)
            ib, gb = b[index]
            for x, y in zip(ia + ga, ib + gb):
                assert y.is_cuda and y.dtype == torch.float32 and tuple(y.shape) == (16384, 3)
                assert torch.equal(x, y.cpu())
