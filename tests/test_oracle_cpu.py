"""CPU tests (no GPU): the oracle against the reference's golden vectors / known answers."""
import glob
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


@pytest.mark.parametrize("path", sorted(p for p in glob.glob(os.path.join(GOLDEN, "knn_*.npz"))
                                        if "sqdiff" not in p))
def test_oracle_knn_vs_reference_golden(orc, path):
    """oracle/oracle.c vs the reference's own torch output (tests/golden/make_golden.py)."""
    g = np.load(path)
    xyz, new, k = g["xyz"], g["new_xyz"], int(g["k"])
    # K1: distance matrix rows are bitwise the reference's square_distance
    D = orc.square_distance(new, xyz)
    rows = g["ref_D_rows"].shape[1]
    np.testing.assert_array_equal(bits(D[:, :rows]), bits(g["ref_D_rows"]))
    # K2: the k smallest distances are bitwise the reference's topk values ...
    idx, dist = orc.knn_expanded(k, xyz, new, return_dist=True)
    ref_vals = g["ref_vals"]
    np.testing.assert_array_equal(bits(dist), bits(ref_vals[..., :k]))
    # ... and the index sets agree wherever the reference has no tie at the k-th distance
    no_tie = ref_vals[..., k - 1] != ref_vals[..., k]
    ours, ref = np.sort(idx, -1), np.sort(g["ref_idx"].astype(np.int64), -1)
    assert (ours[no_tie] == ref[no_tie]).all()
    # ties: lowest index wins => our tied picks are the smallest indices at that distance
    tie_rows = np.argwhere(~no_tie)
    for b, q in tie_rows[:50]:
        kth = dist[b, q, k - 1]
        cand = np.flatnonzero(D[b, q] == kth) if q < rows else None
        if cand is not None:
            need = int((dist[b, q] == kth).sum())
            assert set(idx[b, q][dist[b, q] == kth]) == set(cand[:need])


@pytest.mark.parametrize("name", ["sqdiff_k16", "sqdiff_tie_k16"])
def test_oracle_sqdiff_vs_reference_golden(orc, name):
    """Form 3 (models/pointT_layer2.py:20,62-63) against the imported reference's argsort output."""
    g = np.load(os.path.join(GOLDEN, f"knn_{name}.npz"))
    xyz, k = g["xyz"], int(g["k"])
    idx, dist = orc.knn_form(3, k, xyz, xyz)
    ref_vals = g["ref_vals"]
    np.testing.assert_array_equal(bits(dist), bits(ref_vals[..., :k]))
    no_tie = ref_vals[..., k - 1] != ref_vals[..., k]
    assert (np.sort(idx, -1)[no_tie] == np.sort(g["ref_idx"].astype(np.int64), -1)[no_tie]).all()


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "cos_*.npz"))))
def test_oracle_cosine_vs_reference_golden(orc, path):
    """f2: orc_knn_cosine against the imported reference's knn_point_cosine (make_golden.py). The
    reference's sgemm sums in an unspecified order => tolerance 2e-6 absolute on the distances (a few
    ulp of 1), equal index sets wherever the reference's k-th and (k+1)-th distances are > 4e-6 apart."""
    g = np.load(path)
    xyz = np.ascontiguousarray(g["xyz_t"].transpose(0, 2, 1))
    new = np.ascontiguousarray(g["new_t"].transpose(0, 2, 1))
    k = int(g["k"])
    idx, dist = orc.knn_cosine(k, xyz, new)
    ref_vals = g["ref_vals"]
    np.testing.assert_allclose(dist, ref_vals[..., :k], rtol=0, atol=2e-6)
    clear = (ref_vals[..., k] - ref_vals[..., k - 1]) > 4e-6
    assert clear.mean() > 0.9
    assert (np.sort(idx, -1)[clear] == np.sort(g["ref_idx"].astype(np.int64), -1)[clear]).all()


def test_oracle_direct_forms_differ_only_in_rounding(orc):
    """Forms 1-3 are the same real-number distance with different rounding sequences: the values
    agree to a few ulp, the explicit formulas are reproduced bit for bit."""
    rng = np.random.default_rng(0)
    r = (rng.standard_normal((1, 500, 3)) * 20).astype(np.float32)
    q = (rng.standard_normal((1, 64, 3)) * 20).astype(np.float32)
    d = q[:, :, None, :] - r[:, None, :, :]
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    f64 = lambda a: a.astype(np.float64)  # noqa: E731
    fma = lambda a, b, c: (f64(a) * f64(b) + f64(c)).astype(np.float32)  # noqa: E731  (exact product, one rounding)
    want = {1: fma(dz, dz, fma(dx, dx, dy * dy)), 2: fma(dz, dz, fma(dy, dy, dx * dx)),
            3: (dx * dx + dy * dy) + dz * dz, 4: (dx * dx + dz * dz) + dy * dy}
    for form, full in want.items():
        idx, dist = orc.knn_form(form, 8, r, q)
        got = np.take_along_axis(full, idx, axis=-1)
        np.testing.assert_array_equal(bits(got), bits(dist))
        assert (np.diff(dist, axis=-1) >= 0).all()


def test_oracle_expanded_cuda_order(orc):
    """Form 5 = form 0 with |p|^2 summed as CUDA torch does, (x^2 + z^2) + y^2 (tools/gpu_probe.py: the
    bmm, the scaling and the in-place adds give the same bits on CPU and CUDA; the GPU tests check the
    kernel against the reference's own matrix on the device bit for bit)."""
    rng = np.random.default_rng(3)
    r = (rng.standard_normal((1, 400, 3)) * 30).astype(np.float32)
    q = (rng.standard_normal((1, 50, 3)) * 30).astype(np.float32)
    f64 = lambda a: a.astype(np.float64)  # noqa: E731
    fma = lambda a, b, c: (f64(a) * f64(b) + f64(c)).astype(np.float32)  # noqa: E731
    dot = fma(q[:, :, None, 2], r[:, None, :, 2], fma(q[:, :, None, 1], r[:, None, :, 1], q[:, :, None, 0] * r[:, None, :, 0]))
    nq = (q[..., 0] ** 2 + q[..., 2] ** 2) + q[..., 1] ** 2
    nr = (r[..., 0] ** 2 + r[..., 2] ** 2) + r[..., 1] ** 2
    D = ((np.float32(-2) * dot) + nq[:, :, None]) + nr[:, None, :]
    idx, dist = orc.knn_form(5, 8, r, q)
    np.testing.assert_array_equal(bits(np.take_along_axis(D, idx, -1)), bits(dist))
    np.testing.assert_array_equal(bits(np.sort(D, -1)[..., :8]), bits(dist))
    i0, d0 = orc.knn_form(0, 8, r, q)
    assert (np.abs(d0 - dist) <= 1e-3).all() and (bits(d0) != bits(dist)).any()


def test_oracle_three_nn_weights_ieee(orc):
    """T3 restatement (pointnet2_modules.py:139-144 over pointnet2_utils.py:97) against numpy's
    correctly rounded float32 sqrt / divide (what CUDA torch computes; CPU torch's vectorised
    sqrt is NOT correctly rounded -- 22 of 3072 values differ by one ulp on this container)."""
    rng = np.random.default_rng(1)
    d2 = np.abs(rng.standard_normal((4, 100, 3))).astype(np.float32) * 10
    d2[0, 0] = 0.0
    dist, w = orc.three_nn_weights(d2)
    s = np.sqrt(d2)
    r = np.float32(1.0) / (s + np.float32(1e-8))
    norm = (r[..., 0] + r[..., 2]) + r[..., 1]      # CUDA torch's order (tools/gpu_probe.py)
    np.testing.assert_array_equal(bits(dist), bits(s))
    np.testing.assert_array_equal(bits(w), bits(r / norm[..., None]))


def test_golden_report_says_oracle_is_pinned():
    rep = json.load(open(os.path.join(GOLDEN, "golden_report.json")))
    full = rep["full_16384x16384_k16"]
    assert full["oracle_distance_bit_mismatches"] == 0
    assert full["queries_with_different_kth_distance_multiset"] == 0
    for big in ("big_k16", "big_k32"):      # reach knn_scan_tc_kernel on the GPU (N >= 8192)
        assert rep[big]["oracle_queries_with_different_kth_distance_multiset"] == 0
    assert rep["sqdiff_k16"]["oracle_distance_bit_mismatches"] == 0
    for name, v in rep.items():
        if isinstance(v, dict) and "permuted_view_bit_mismatches" in v:
            assert v["oracle_distance_bit_mismatches"] == 0 and v["permuted_view_bit_mismatches"] == 0


def test_oracle_emd_known_answer(orc):
    """models/EMD/test_emd_loss.py:7-23: cost 0.71 per pair, weighted loss 2.0116667, grads."""
    p1 = np.array([[[1.7, -0.1, 0.1], [0.1, 1.2, 0.3]]], np.float32).repeat(3, 0)
    p2 = np.array([[[0.3, 1.8, 0.2], [1.2, -0.2, 0.3]]], np.float32).repeat(3, 0)
    match = orc.emd_approxmatch(p1, p2)
    assert abs(match[0, 0, 1] - 1.0) < 1e-6 and abs(match[0, 1, 0] - 1.0) < 1e-6
    assert match[0, 0, 0] < 1e-8 and match[0, 1, 1] < 1e-8
    cost = orc.emd_matchcost(p1, p2, match)
    np.testing.assert_allclose(cost, 0.71, rtol=1e-6)
    loss = cost[0] / 2 + cost[1] * 2 + cost[2] / 3
    gt = (0.5 ** 2 + 0.1 ** 2 + 0.2 ** 2 + 0.2 ** 2 + 0.6 ** 2 + 0.1 ** 2) * (0.5 + 2 + 1 / 3)
    assert abs(loss - gt) <= 1e-5 * gt
    g1, g2 = orc.emd_matchcost_grad(np.array([0.5, 2.0, 1 / 3], np.float32), p1, p2, match)
    np.testing.assert_allclose(g1[0], [[0.5, 0.1, -0.2], [-0.2, -0.6, 0.1]], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(g2[0], [[0.2, 0.6, -0.1], [-0.5, -0.1, 0.2]], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(g1[1], 4 * g1[0], rtol=1e-5)


def _fps_bruteforce(xyz, m):
    """Independent python model of sampling_gpu.cu:93-209 (per-thread strided scan + tree)."""
    n = xyz.shape[0]
    bs = 1
    while bs * 2 <= min(n, 1024):
        bs *= 2
    temp = np.full(n, 1e10, np.float32)
    out = [0]
    old = 0
    for _ in range(1, m):
        d = xyz - xyz[old]
        dx, dy, dz = d[:, 0], d[:, 1], d[:, 2]
        dist = (dz.astype(np.float64) * dz + (dx.astype(np.float64) * dx + (dy * dy).astype(np.float64)).astype(np.float32)).astype(np.float32)
        temp = np.minimum(dist, temp)
        best = np.full(bs, -1.0, np.float32)
        besti = np.zeros(bs, np.int64)
        for tid in range(bs):
            ks = np.arange(tid, n, bs)
            if len(ks):
                j = int(np.argmax(temp[ks]))  # first maximum == lowest k
                if temp[ks][j] > best[tid]:
                    best[tid], besti[tid] = temp[ks][j], ks[j]
        s = bs // 2
        while s >= 1:
            for tid in range(s):
                if best[tid + s] > best[tid]:
                    best[tid], besti[tid] = best[tid + s], besti[tid + s]
            s //= 2
        old = int(besti[0])
        out.append(old)
    return np.array(out, np.int32)


def test_oracle_fps_tie_order():
    from mocopci_b200 import synth
    from oracle import cpu as orc
    for n, m in ((40, 12), (100, 30), (257, 20)):
        xyz = synth.tie_stress_cloud(n, 1, n, grid=2).numpy()
        idx, _ = orc.fps(xyz, m)
        np.testing.assert_array_equal(idx[0], _fps_bruteforce(xyz[0], m))


def test_oracle_ball_query_and_three_nn_semantics(orc):
    xyz = np.array([[[0, 0, 0], [0.1, 0, 0], [5, 5, 5], [0.2, 0, 0], [0.05, 0, 0]]], np.float32)
    new = np.array([[[0, 0, 0], [9, 9, 9]]], np.float32)
    idx = orc.ball_query(0.15, 4, xyz, new)
    # first nsample hits in index order, padded with the first hit; no hit => zeros
    np.testing.assert_array_equal(idx[0, 0], [0, 1, 4, 0])
    np.testing.assert_array_equal(idx[0, 1], [0, 0, 0, 0])
    d2, i3 = orc.three_nn(new, xyz[:, :2])  # m = 2 < 3
    assert i3[0, 0, 2] == 0 and np.isinf(d2[0, 0, 2])
    np.testing.assert_array_equal(i3[0, 0, :2], [0, 1])
    # duplicates: the lowest index wins
    dup = np.zeros((1, 6, 3), np.float32)
    d2, i3 = orc.three_nn(new[:, :1], dup)
    np.testing.assert_array_equal(i3[0, 0], [0, 1, 2])


def test_oracle_chamfer_definition(orc):
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 50, 3)).astype(np.float32)
    y = rng.standard_normal((2, 70, 3)).astype(np.float32)
    loss, dx, dy, ix, iy = orc.chamfer(x, y)
    d = ((x[:, :, None].astype(np.float64) - y[:, None].astype(np.float64)) ** 2).sum(-1)
    ref = (d.min(2).mean(1) + d.min(1).mean(1)).mean()
    assert abs(loss - ref) <= 1e-6 * ref
    np.testing.assert_array_equal(ix, d.argmin(2))
    np.testing.assert_array_equal(iy, d.argmin(1))


def test_oracle_gather_group_interpolate(orc):
    rng = np.random.default_rng(1)
    f = rng.standard_normal((2, 5, 40)).astype(np.float32)
    idx = rng.integers(0, 40, (2, 7, 3)).astype(np.int32)
    g = orc.group(f, idx)
    for b in range(2):
        np.testing.assert_array_equal(g[b], f[b][:, idx[b]])
    np.testing.assert_array_equal(orc.gather(f, idx[:, :, 0]), g[..., 0])
    w = rng.random((2, 7, 3)).astype(np.float32)
    out = orc.three_interpolate(f, idx, w)
    np.testing.assert_allclose(out, (g * w[:, None]).sum(-1), rtol=1e-6, atol=1e-6)
    go = rng.standard_normal((2, 5, 7, 3)).astype(np.float32)
    gg = orc.group_grad(go, idx, 40)
    ref = np.zeros((2, 5, 40), np.float32)
    for b in range(2):
        for p in range(7):
            for s in range(3):
                ref[b, :, idx[b, p, s]] += go[b, :, p, s]
    np.testing.assert_allclose(gg, ref, rtol=1e-5, atol=1e-6)
