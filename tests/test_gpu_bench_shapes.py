"""Every call bench.py times, at the shape and on the inputs it times it with, against the C oracle
(oracle/oracle.c) or an exact torch composition on the GPU: bit for bit unless a tolerance is
written at the assert.

Several kernel configurations are chosen from the batch size or the point count (FPS cluster shape
and points per thread, one-launch vs two-pass neighbour search, split vs thread-per-query top-k,
gather variants). The smaller shapes of test_gpu_parity.py do not reach the ones the benchmark and
the model run, so each test here also records the kernels its call launched (torch.profiler) and
asserts the configuration the dispatch is meant to pick: a later dispatch change then fails here
instead of quietly moving the test to another path.

bench.py row                           test
headline (knn_point k=16, 64 pairs)    test_knn_headline_batch_vs_oracle
knn_k16_B8, knn_k32_B8                 test_knn_benchmark_batch_vs_oracle
knn_k16_B1                             test_knn_benchmark_single_pair_vs_oracle
knn_k32_B1_self                        test_knn_self_finest_level_vs_oracle
knn_k3_16384x2048_B1                   test_knn_k3_upsample_shape_vs_oracle
chamfer_B8                             test_chamfer_per_point_vs_oracle[lidar_B8]
fps_16384_to_4096                      test_fps_benchmark_call_vs_oracle (and test_fps_*)
ball_query_r0.5_ns32                   test_ball_query_benchmark_call_vs_oracle
group_points_C128, group_points_C3     test_group_points_benchmark_calls
query_and_group_C128                   test_query_and_group_benchmark_call
index_points_group_C64_k16             test_index_points_group_benchmark_call
three_nn_weights_pyramid               test_three_nn_weights_pyramid_vs_oracle
three_interpolate_pyramid_C128,        test_three_interpolate_pyramid_vs_oracle
  three_interpolate_4096_to_16384_C128
knn_point_cosine_2048_C64_k16          test_knn_point_cosine_benchmark_call_vs_oracle
group_concat_16384_k32_C32             test_group_concat_benchmark_call
emd_cost_16384, emd_match_16384        test_emd_16384
"""
import types

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

NPTS = 16384  # points per benchmark frame


def bits(a):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


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


# ------------------------------------------------------------------------------------------
# inputs as bench.py builds them
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pairs8():
    """bench.py's extras() inputs: the first 8 of the rank's frame pairs (refs a = frame t,
    queries b = frame t+1), on the CPU and on the GPU."""
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(0, 8)
    return types.SimpleNamespace(a=a, b=b, ad=a.cuda(), bd=b.cuda())


@pytest.fixture(scope="module")
def knn8_oracle(orc, pairs8):
    """Oracle form 5 (the reference's square_distance as CUDA torch sums it), k = 32, all 8 pairs.
    Neighbours are sorted by (distance, index), so the k = 16 answer is the first 16 columns."""
    return orc.knn_form(5, 32, pairs8.a.numpy(), pairs8.b.numpy())


def assert_two_pass_knn(names, k, split_topk=False):
    """The two-pass neighbour search: tensor-core scan in the expanded arithmetic, then the top-k
    kernel -- one thread per query, or one thread per (query, group of ref splits)."""
    assert "knn_scan_tc_kernel<0>" in names, names
    want = f"knn_topk_split_kernel<{k}>" if split_topk else f"knn_topk_kernel<{k}>"
    other = f"knn_topk_kernel<{k}>" if split_topk else f"knn_topk_split_kernel<{k}>"
    assert want in names and other not in names, names
    assert not base(names) & {"knn_mid_kernel", "knn_kernel"}, names


# ------------------------------------------------------------------------------------------
# KNN at the benchmark's batch sizes
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [16, 32])
def test_knn_benchmark_batch_vs_oracle(pairs8, knn8_oracle, k):
    """knn_k16_B8 / knn_k32_B8: knn_point(k, a, b) on the 8 benchmark pairs, every pair, every
    index; the distances of the same call with distances requested, bit for bit."""
    from mocopci_b200 import pointconv_util as pcu
    idx, names = launches(lambda: pcu.knn_point(k, pairs8.ad, pairs8.bd))
    oi, od = knn8_oracle
    got = idx.cpu().numpy()
    for p in range(8):
        np.testing.assert_array_equal(got[p], oi[p, :, :k], err_msg=f"pair {p}")
    idx2, dist = pcu.knn_point_with_dist(k, pairs8.ad, pairs8.bd)
    assert torch.equal(idx2, idx)
    np.testing.assert_array_equal(bits(dist), bits(od[..., :k]))
    assert_two_pass_knn(names, k)


def test_knn_benchmark_single_pair_vs_oracle(pairs8, knn8_oracle):
    """knn_k16_B1: one frame pair (a[:1], b[:1])."""
    from mocopci_b200 import pointconv_util as pcu
    idx, names = launches(lambda: pcu.knn_point(16, pairs8.ad[:1], pairs8.bd[:1]))
    np.testing.assert_array_equal(idx.cpu().numpy(), knn8_oracle[0][:1, :, :16])
    assert_two_pass_knn(names, 16, split_topk=True)


def test_knn_headline_batch_vs_oracle(orc):
    """The headline step: knn_point(16, a, b) over the 64 frame pairs of one GPU. The oracle checks
    four pairs spread over the batch (first, last and two between)."""
    from mocopci_b200 import pointconv_util as pcu, synth
    a, b = synth.frame_pairs(0, 64)
    idx, names = launches(lambda: pcu.knn_point(16, a.cuda(), b.cuda()))
    assert tuple(idx.shape) == (64, NPTS, 16)
    sel = [0, 21, 42, 63]
    oi, _ = orc.knn_form(5, 16, a[sel].numpy(), b[sel].numpy())
    got = idx[sel].cpu().numpy()
    for j, p in enumerate(sel):
        np.testing.assert_array_equal(got[j], oi[j], err_msg=f"pair {p}")
    assert_two_pass_knn(names, 16)


def test_knn_self_finest_level_vs_oracle(orc, pairs8):
    """knn_k32_B1_self: a cloud against itself, k = 32 (the model's finest level)."""
    from mocopci_b200 import pointconv_util as pcu
    a1 = pairs8.ad[:1]
    idx, names = launches(lambda: pcu.knn_point(32, a1, a1))
    oi, _ = orc.knn_form(5, 32, pairs8.a[:1].numpy(), pairs8.a[:1].numpy())
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    assert_two_pass_knn(names, 32, split_topk=True)


def test_knn_k3_upsample_shape_vs_oracle(orc, pairs8):
    """knn_k3_16384x2048_B1: 16384 queries against the first 2048 points of a frame (a strided view).
    B * S * N = 2^25 is exactly the pair count from which k <= 4 takes the two-pass path, so this
    call reaches it without any test hook."""
    from mocopci_b200 import pointconv_util as pcu
    refs = pairs8.ad[:1, :2048]
    assert 1 * NPTS * 2048 == 1 << 25
    (idx, dist), names = launches(lambda: pcu.knn_point_with_dist(3, refs, pairs8.bd[:1]))
    oi, od = orc.knn_form(5, 3, pairs8.a[:1, :2048].numpy(), pairs8.b[:1].numpy())
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(dist), bits(od))
    # (the threshold pre-pass on the FP32 pipe: 2048 refs give too small a sample for the tensor cores)
    assert "knn_tau_kernel<4>" in names, names
    assert_two_pass_knn(names, 3)


COS_ATOL = 4e-6   # as test_gpu_parity.py: the oracle sums the dot products in FP64, the tensor
COS_GAP = 8e-6    # cores in their own order; neighbour sets must agree wherever the gap is clear


def test_knn_point_cosine_benchmark_call_vs_oracle(orc):
    """knn_point_cosine_2048_C64_k16: 2048 feature vectors of 64 channels as the permuted [B,C,N]
    view the model passes, against themselves."""
    from mocopci_b200 import pointconv_util as pcu
    g = torch.Generator().manual_seed(64)
    feat = torch.randn(1, 64, 2048, generator=g).cuda().permute(0, 2, 1)
    (idx, dist), names = launches(lambda: pcu.knn_point_cosine_with_dist(16, feat, feat))
    f = feat.contiguous().cpu().numpy()
    oi, od = orc.knn_cosine(17, f, f)
    assert float(np.abs(dist.cpu().numpy() - od[..., :16]).max()) <= COS_ATOL
    assert bool((dist[..., 1:] >= dist[..., :-1]).all())
    clear = (od[..., 16] - od[..., 15]) > COS_GAP
    same = (np.sort(idx.cpu().numpy(), -1) == np.sort(oi[..., :16], -1)).all(-1)
    assert bool(same[clear].all()) and clear.mean() > 0.8, f"{int((~same & clear).sum())} sets differ"
    assert sorted(names) == ["cos_knn_kernel<16>", "cos_pack_kernel"], names


# ------------------------------------------------------------------------------------------
# Chamfer: per-point minima and indices, loss, backward
# ------------------------------------------------------------------------------------------
def chamfer_forward(x, y):
    """b200pci_chamfer_forward called as chamfer.py calls it, keeping what it writes per point:
    -> (loss, dist_x [B,N], idx_x [B,N], dist_y [B,M], idx_y [B,M])."""
    from mocopci_b200 import _lib
    L = _lib.lib
    B, N, _ = x.shape
    M = y.shape[1]
    f32, i32 = dict(dtype=torch.float32, device=x.device), dict(dtype=torch.int32, device=x.device)
    dist_x, idx_x = torch.empty((B, N), **f32), torch.empty((B, N), **i32)
    dist_y, idx_y = torch.empty((B, M), **f32), torch.empty((B, M), **i32)
    loss = torch.empty((1,), **f32)
    ws = _lib.workspace(L.b200pci_chamfer_workspace_bytes(B, N, M), x.device)
    xs, ys = x.stride(), y.stride()
    _lib.check(L.b200pci_chamfer_forward(
        B, N, M, x.data_ptr(), xs[0], xs[1], xs[2], y.data_ptr(), ys[0], ys[1], ys[2],
        dist_x.data_ptr(), idx_x.data_ptr(), dist_y.data_ptr(), idx_y.data_ptr(), loss.data_ptr(),
        ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "chamfer_forward")
    return loss[0], dist_x, idx_x, dist_y, idx_y


def chamfer_inputs(case):
    """-> (x [B,N,3], y [B,M,3]) on the CPU, contiguous."""
    from mocopci_b200 import synth
    if case == "uniform_B2":      # the one-launch kernel (small clouds)
        return synth.uniform_cloud(500, 2, 500), synth.uniform_cloud(701, 2, 700)
    if case == "lidar_B1":        # one pair: the smallest two-pass launch at the benchmark size
        return synth.frame_pairs(0, 1)
    if case == "lidar_B8":        # bench.py chamfer_B8
        return synth.frame_pairs(0, 8)
    if case == "lidar_B2_bcn_views":
        return synth.frame_pairs(1, 2)
    if case == "lidar_N_ne_M":
        a, b = synth.frame_pairs(2, 2)
        return a, b[:, :5000].contiguous()
    if case == "tie_stress":      # integer grid, half the points duplicated
        return synth.tie_stress_cloud(11, 2, 9000, grid=6), synth.tie_stress_cloud(12, 2, 7000, grid=6)
    if case == "lidar_shift_900":
        a, b = synth.frame_pairs(3, 1)
        return a + 900.0, b + 900.0
    raise ValueError(case)


CHAMFER_CASES = ["uniform_B2", "lidar_B1", "lidar_B8", "lidar_B2_bcn_views", "lidar_N_ne_M",
                 "tie_stress", "lidar_shift_900"]


@pytest.mark.parametrize("case", CHAMFER_CASES)
def test_chamfer_per_point_vs_oracle(orc, case):
    """Both K = 1 searches of Chamfer run in pytorch3d's arithmetic, fma(dz,dz,fma(dy,dy,dx*dx)),
    like knn_points: the per-point squared minima and nearest-neighbour indices equal the oracle's
    (orc_chamfer) bit for bit, lowest index first among equal distances, and equal
    knn_points(K=1) of the same clouds. The loss is the float32 rounding of the oracle's FP64 sum
    (within 1 ulp: both sum in FP64, in different orders). chamfer_distance -- the call bench.py
    and the model make, here with [B,3,N] views where chamfer_loss passes them -- gives the same
    loss, and its backward matches FP64 autograd through the oracle's indices."""
    from mocopci_b200 import chamfer
    x, y = chamfer_inputs(case)
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    if case == "lidar_B2_bcn_views":  # chamfer_loss(pc1, pc2) permutes [B,3,N] tensors
        x_leaf = x.permute(0, 2, 1).contiguous().cuda().requires_grad_(True)
        y_leaf = y.permute(0, 2, 1).contiguous().cuda().requires_grad_(True)
        xv, yv = x_leaf.permute(0, 2, 1), y_leaf.permute(0, 2, 1)
        assert xv.stride(2) == N
    else:
        x_leaf, y_leaf = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
        xv, yv = x_leaf, y_leaf
    with torch.no_grad():
        (loss, dx, ix, dy, iy), names = launches(lambda: chamfer_forward(xv, yv))
    ol, odx, ody, oix, oiy = orc.chamfer(x.numpy(), y.numpy())
    bad = {"dist_x": int((bits(dx) != bits(odx)).sum()), "idx_x": int((ix.cpu().numpy() != oix).sum()),
           "dist_y": int((bits(dy) != bits(ody)).sum()), "idx_y": int((iy.cpu().numpy() != oiy).sum())}
    assert not any(bad.values()), f"{case}: entries differing from the oracle {bad} of {B * N} / {B * M}"
    want = np.float32(ol)
    assert abs(int(bits(loss.reshape(1))[0]) - int(want.view(np.int32))) <= 1, (float(loss), ol)

    # knn_points (the other pytorch3d stand-in) finds the same neighbours with the same bits
    for p, q, d, i in ((xv, yv, dx, ix), (yv, xv, dy, iy)):
        r = chamfer.knn_points(p.detach(), q.detach(), K=1)
        assert torch.equal(r.idx[..., 0], i.long())
        assert torch.equal(r.dists[..., 0].view(torch.int32), d.view(torch.int32))

    # the public entry point: same loss bits; backward against FP64 autograd on the oracle's indices
    loss2, _ = chamfer.chamfer_distance(xv, yv)
    assert torch.equal(loss2.reshape(1).view(torch.int32), loss.reshape(1).view(torch.int32))
    if case == "lidar_B2_bcn_views":
        loss3 = chamfer.chamfer_loss(x_leaf.detach(), y_leaf.detach())
        assert torch.equal(loss3.reshape(1).view(torch.int32), loss.reshape(1).view(torch.int32))
    loss2.backward()
    xt, yt = x.double().requires_grad_(True), y.double().requires_grad_(True)
    bi = torch.arange(B)[:, None]
    ixt, iyt = torch.as_tensor(oix).long(), torch.as_tensor(oiy).long()
    ref = ((xt - yt[bi, ixt]) ** 2).sum(-1).mean(-1) + ((yt - xt[bi, iyt]) ** 2).sum(-1).mean(-1)
    ref.mean().backward()
    gx, gy = x_leaf.grad, y_leaf.grad
    if case == "lidar_B2_bcn_views":
        gx, gy = gx.permute(0, 2, 1), gy.permute(0, 2, 1)
    # the backward scatters with atomics (order varies run to run): 1e-4 relative
    np.testing.assert_allclose(gx.cpu().numpy(), xt.grad.float().numpy(), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(gy.cpu().numpy(), yt.grad.float().numpy(), rtol=1e-4, atol=1e-7)

    assert names.count("chamfer_reduce_kernel") == 1 and names.count("chamfer_final_kernel") == 1, names
    if case == "uniform_B2":  # the one-launch kernel, both directions
        assert names.count("knn_mid_kernel<1, 16>") == 2 and "knn_scan_tc_kernel" not in base(names), names
    else:  # two-pass search in the direct-difference arithmetic, both directions
        assert names.count("knn_scan_tc_kernel<1>") == 2, names
        assert names.count("knn_topk_kernel<1>") == 2, names


# ------------------------------------------------------------------------------------------
# FPS
# ------------------------------------------------------------------------------------------
def check_fps(orc, xyz, m, kernel):
    """furthest_point_sampling_wrapper (the reference's pybind signature; temp initialised to 1e10
    as pointnet2_utils.py does): the sampled indices and the final min-distance buffer against the
    oracle, bit for bit, and the one kernel launched."""
    from mocopci_b200 import pointnet2_cuda
    B, n, _ = xyz.shape
    xd = xyz.cuda()
    temp = torch.full((B, n), 1e10, device="cuda")
    idx = torch.empty((B, m), dtype=torch.int32, device="cuda")
    _, names = launches(lambda: pointnet2_cuda.furthest_point_sampling_wrapper(B, n, m, xd, temp, idx))
    oi, ot = orc.fps(xyz.numpy(), m)
    got = idx.cpu().numpy()
    for b in range(B):
        np.testing.assert_array_equal(got[b], oi[b], err_msg=f"cloud {b}")
    np.testing.assert_array_equal(bits(temp), bits(ot))
    assert names == [kernel], names


def fps_clouds(B, n):
    from mocopci_b200 import synth
    return synth.frame_pairs(0, B, n)[0]


def fps_m(n):
    """Samples per case: the oracle costs B x n x m (about a second per case on 8 cores)."""
    return 1024 if n <= 20000 else (512 if n <= 70000 else 256)


# (n, points per thread, cloud mirrored in shared memory) of the 8 x 512 cluster (5 clouds and more)
FPS_8X512 = [(4096, 2, True), (4097, 2, True), (16384, 4, True), (17066, 8, True), (17067, 8, False),
             (65536, 16, False), (131072, 32, False)]


@pytest.mark.parametrize("n,pt,mirror", FPS_8X512)
@pytest.mark.parametrize("B", [5, 8])
def test_fps_cluster_8x512_vs_oracle(orc, B, n, pt, mirror):
    """Every points-per-thread tier of the 8-CTA x 512-thread cluster, the mirror boundary
    (3 n floats <= 200 KiB: 17066 is the last point count mirrored) and ragged last chunks (4097,
    17066, 17067)."""
    check_fps(orc, fps_clouds(B, n), fps_m(n),
              f"fps_cluster_kernel<{pt}, {'true' if mirror else 'false'}, 8, 512>")


def test_fps_cluster_16x256_largest_cloud(orc):
    """Up to 4 clouds: the 16-CTA x 256-thread cluster, here at its largest cloud (32 points per
    thread, no mirror)."""
    check_fps(orc, fps_clouds(2, 131072), 256, "fps_cluster_kernel<32, false, 16, 256>")


def test_fps_single_cta_beyond_cluster_range(orc):
    """n > 131072: one CTA per cloud with the points left in global memory."""
    check_fps(orc, fps_clouds(1, 140000), 256, "fps_kernel<0, false>")


def test_fps_more_samples_than_points(orc):
    """m > n on a cluster path: after every point has been taken, all distances are 0 and the tie
    order alone decides."""
    check_fps(orc, fps_clouds(5, 4096), 5000, "fps_cluster_kernel<2, true, 8, 512>")


def test_fps_one_sample(orc):
    """m = 1: index 0 and the distance buffer left as given."""
    check_fps(orc, fps_clouds(8, NPTS), 1, "fps_cluster_kernel<4, true, 8, 512>")


def test_fps_cluster_tie_stress(orc):
    """Integer-grid cloud (grid 3: 343 sites for 16384 points): the furthest distance is tied
    between hundreds of points at every step."""
    from mocopci_b200 import synth
    check_fps(orc, synth.tie_stress_cloud(17, 6, NPTS, grid=3), 1024, "fps_cluster_kernel<4, true, 8, 512>")


# ------------------------------------------------------------------------------------------
# config 2 at B = 8: fps -> centres -> ball_query -> group / query_and_group
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def config2(pairs8):
    from mocopci_b200 import ops as p2u, pointconv_util as pcu
    a = pairs8.ad
    fidx, fps_names = launches(lambda: p2u.furthest_point_sample(a, 4096))
    centres = pcu.index_points_gather(a, fidx)
    idx, bq_names = launches(lambda: p2u.ball_query(0.5, 32, a, centres))
    feats = torch.randn(8, 128, NPTS, device="cuda", generator=torch.Generator("cuda").manual_seed(99))
    return types.SimpleNamespace(a=a, fidx=fidx, fps_names=fps_names, centres=centres, idx=idx,
                                 bq_names=bq_names, feats=feats)


def group_ref(features, idx):
    """grouping_operation as an exact torch.gather: out[b,c,p,s] = features[b,c,idx[b,p,s]]."""
    B, C, _ = features.shape
    _, P, S = idx.shape
    return torch.gather(features, 2, idx.long().reshape(B, 1, P * S).expand(B, C, P * S)).reshape(B, C, P, S)


def test_fps_benchmark_call_vs_oracle(orc, pairs8, config2):
    """fps_16384_to_4096: furthest_point_sample(a, 4096) on the 8 benchmark frames."""
    np.testing.assert_array_equal(config2.fidx.cpu().numpy(), orc.fps(pairs8.a.numpy(), 4096)[0])
    assert config2.fps_names == ["fps_cluster_kernel<4, true, 8, 512>"], config2.fps_names


def test_ball_query_benchmark_call_vs_oracle(orc, pairs8, config2):
    """ball_query_r0.5_ns32 on the 4096 FPS centres of each of the 8 frames; the centres are the
    exact rows index_points_gather picked."""
    a = pairs8.a
    want_c = torch.gather(a, 1, config2.fidx.cpu().long().unsqueeze(-1).expand(-1, -1, 3))
    assert torch.equal(config2.centres.cpu(), want_c)
    want = orc.ball_query(0.5, 32, a.numpy(), want_c.numpy())
    np.testing.assert_array_equal(config2.idx.cpu().numpy(), want)
    assert sorted(config2.bq_names) == ["ball_fallback_kernel", "ball_select_kernel", "knn_scan_kernel",
                                        "nbr_pack_refs_kernel"], config2.bq_names


@pytest.mark.parametrize("C", [128, 3])
def test_group_points_benchmark_calls(config2, C):
    """group_points_C128 (seeded features) and group_points_C3 (the transposed cloud) on the
    ball_query result: equal to torch.gather."""
    from mocopci_b200 import ops as p2u
    feats = config2.feats if C == 128 else config2.a.transpose(1, 2).contiguous()
    out, names = launches(lambda: p2u.grouping_operation(feats, config2.idx))
    assert tuple(out.shape) == (8, C, 4096, 32)
    assert torch.equal(out, group_ref(feats, config2.idx))
    assert names == ["group_kernel<true>"], names


def test_query_and_group_benchmark_call(config2):
    """query_and_group_C128: ball_query + [grouped cloud minus centre | grouped features] in one
    tensor, equal to that composition written with torch.gather on the same indices."""
    from mocopci_b200 import ops as p2u
    out, names = launches(lambda: p2u.query_and_group(0.5, 32, config2.a, config2.centres, config2.feats))
    rel = group_ref(config2.a.transpose(1, 2).contiguous(), config2.idx) - config2.centres.transpose(1, 2).unsqueeze(-1)
    want = torch.cat([rel, group_ref(config2.feats, config2.idx)], 1)
    assert out.shape == want.shape and torch.equal(out, want)
    assert sorted(names) == ["ball_fallback_kernel", "ball_select_kernel", "group_kernel<true>",
                             "group_xyz_rel_kernel<true>", "knn_scan_kernel", "nbr_pack_refs_kernel"], names


PYRAMID = [(256, 64), (1024, 256), (4096, 1024), (16384, 4096)]  # (unknown n, known m)
INTERPOLATE_KERNEL = {256: "three_interpolate_kernel", 1024: "three_interpolate_quad_kernel",
                      4096: "three_interpolate_quad_kernel", 16384: "three_interpolate_quad_kernel"}


def test_three_nn_weights_pyramid_vs_oracle(orc, pairs8):
    """three_nn_weights_pyramid: every level of the feature-propagation pyramid at B = 8 (prefixes
    of the benchmark frames): indices, distances and weights against orc.three_nn +
    orc.three_nn_weights, bit for bit."""
    from mocopci_b200 import ops as p2u
    for n, m in PYRAMID:
        unknown, known = pairs8.ad[:, :n].contiguous(), pairs8.ad[:, :m].contiguous()
        (w, idx, dist), names = launches(lambda: p2u.three_nn_weights(unknown, known))
        od2, oi = orc.three_nn(pairs8.a[:, :n].numpy(), pairs8.a[:, :m].numpy())
        odist, ow = orc.three_nn_weights(od2)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi, err_msg=f"{m}->{n}")
        np.testing.assert_array_equal(bits(dist), bits(odist), err_msg=f"{m}->{n}")
        np.testing.assert_array_equal(bits(w), bits(ow), err_msg=f"{m}->{n}")
        assert names.count("three_nn_finish_kernel") == 1, (n, m, names)
        if n == NPTS:  # two-pass search in the direct-difference arithmetic
            assert "knn_scan_tc_kernel<1>" in names and "knn_topk_kernel<3>" in names, names
        else:          # the one-launch kernel
            assert sorted(names) == ["knn_mid_kernel<1, 16>", "three_nn_finish_kernel"], (n, m, names)


def test_three_interpolate_pyramid_vs_oracle(orc, pairs8):
    """three_interpolate_pyramid_C128 and three_interpolate_4096_to_16384_C128: C = 128 features
    interpolated with the weights of each pyramid level, against orc.three_interpolate bit for bit."""
    from mocopci_b200 import ops as p2u
    g = torch.Generator("cuda").manual_seed(3)
    for n, m in PYRAMID:
        w, idx, _ = p2u.three_nn_weights(pairs8.ad[:, :n].contiguous(), pairs8.ad[:, :m].contiguous())
        f = torch.randn(8, 128, m, device="cuda", generator=g)
        out, names = launches(lambda: p2u.three_interpolate(f, idx, w))
        want = orc.three_interpolate(f.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy())
        np.testing.assert_array_equal(bits(out), bits(want), err_msg=f"{m}->{n}")
        assert names == [INTERPOLATE_KERNEL[n]], (n, m, names)


# ------------------------------------------------------------------------------------------
# row gathers
# ------------------------------------------------------------------------------------------
def test_index_points_group_benchmark_call(pairs8, knn8_oracle):
    """index_points_group_C64_k16: [B,N,C] features, C = 64, gathered with the k = 16 neighbours of
    the 8 benchmark pairs (int64), against torch's advanced indexing."""
    from mocopci_b200 import pointconv_util as pcu
    kidx = torch.as_tensor(knn8_oracle[0][..., :16]).cuda()
    assert torch.equal(kidx, pcu.knn_point(16, pairs8.ad, pairs8.bd))
    fbnc = torch.randn(8, NPTS, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(64))
    out, names = launches(lambda: pcu.index_points_group(fbnc, kidx))
    assert tuple(out.shape) == (8, NPTS, 16, 64) and out.is_contiguous()
    assert torch.equal(out, fbnc[torch.arange(8, device="cuda")[:, None, None], kidx])
    assert names == ["rows_gather_kernel<true, true>"], names


def test_group_concat_benchmark_call(orc, pairs8):
    """group_concat_16384_k32_C32: _group_concat(a[:1], a[:1], f32, gidx) with the k = 32 self
    neighbours and 32 feature channels as a permuted [B,C,N] view: [xyz[idx] - centre | feats[idx]]
    and xyz[idx] - centre, equal to the torch composition."""
    from mocopci_b200 import pointconv_util as pcu
    a1 = pairs8.ad[:1]
    f32 = torch.randn(1, 32, NPTS, device="cuda", generator=torch.Generator("cuda").manual_seed(32)).permute(0, 2, 1)
    gidx = pcu.knn_point(32, a1, a1)
    np.testing.assert_array_equal(gidx.cpu().numpy(), orc.knn_form(5, 32, pairs8.a[:1].numpy(), pairs8.a[:1].numpy())[0])
    (out, norm), names = launches(lambda: pcu._group_concat(a1, a1, f32, gidx))
    z = torch.zeros_like(gidx)
    rel = a1[z, gidx] - a1.unsqueeze(2)
    assert torch.equal(norm, rel)
    assert tuple(out.shape) == (1, NPTS, 32, 35) and torch.equal(out, torch.cat([rel, f32[z, gidx]], -1))
    assert names == ["group_concat_warp_kernel<true, 8>"], names


# ------------------------------------------------------------------------------------------
# EMD at 16384 x 16384
# ------------------------------------------------------------------------------------------
def test_emd_16384(pairs8):
    """emd_cost_16384 and emd_match_16384 on benchmark pair 0. The forward-only emd_cost (never
    stores the match matrix, approximate ex2) equals matchcost_forward(approxmatch_forward(...)) to
    1e-5 relative, and that matchcost equals a chunked FP64 evaluation of its formula
    (orc_emd_matchcost: sum over k, l of |p2_l - p1_k|^2 match[l, k]) on the same match matrix to
    1e-5 relative. The oracle's own approxmatch is not run at this size (minutes on a CPU)."""
    from mocopci_b200 import emd_cuda
    x1, x2 = pairs8.ad[:1].contiguous(), pairs8.bd[:1].contiguous()
    cost, cost_names = launches(lambda: emd_cuda.emd_cost(x1, x2))
    match, match_names = launches(lambda: emd_cuda.approxmatch_forward(x1, x2))
    mc = emd_cuda.matchcost_forward(x1, x2, match)
    c, m_ = float(cost[0]), float(mc[0])
    assert abs(c - m_) <= 1e-5 * abs(m_), (c, m_)
    p1, p2 = x1[0].double(), x2[0].double()
    ref = 0.0
    for l0 in range(0, NPTS, 1024):
        d = ((p2[l0:l0 + 1024, None, :] - p1[None, :, :]) ** 2).sum(-1)
        ref += float((d * match[0, l0:l0 + 1024].double()).sum())
    assert abs(m_ - ref) <= 1e-5 * ref, (m_, ref)
    assert "emd_cost_rows_kernel" not in base(cost_names), cost_names
    assert {"emd_init_kernel", "emd_rows1_kernel", "emd_rows2_kernel", "emd_cost_reduce_kernel"} <= base(cost_names)
    assert "emd_rows1_kernel<1, 1>" in match_names and "emd_rows1_kernel<3, 1>" in match_names, match_names
