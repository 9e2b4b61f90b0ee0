"""Model-level parity (M1 / BASELINE config 4): the UNMODIFIED reference model
(models/m_models/mocopci.py:1062-1097, imported from the checkout) on the B200 kernels.

1. shadow run: the reference's own stack (its CUDA kernels from oracle/_ref + its pure-torch
   helpers) drives one full forward at 16384 points, and every hot-path call it makes is replayed
   through the B200 kernel and compared with SURVEY 8c's protocol (tests/refstack.py);
2. end to end: the same network (same seed) through ``mocopci_b200.install()`` -- the product's
   own patching, nothing from tests/ in the loop -- against the reference stack's output.
"""
import importlib
import json
import os
import sys
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NPTS = 16384
T_INTERP = [0.4167, 0.5, 0.5833]   # train.py:49-55 / test.py:38-44 with the defaults


def _frames(npts, batch=1):
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(40, batch, npts)          # [B, N, 3] each
    return a.permute(0, 2, 1).contiguous().cuda(), b.permute(0, 2, 1).contiguous().cuda()


def _forget():
    from tests import cpu_natives
    from mocopci_b200 import shim
    shim.uninstall()
    cpu_natives.forget_reference_modules()
    for name in list(sys.modules):
        if name.startswith(("pytorch3d", "timm")) and getattr(sys.modules[name], "__file__", None) is None:
            del sys.modules[name]


def _build(seed=0):
    mm = importlib.import_module("models.m_models.mocopci")
    torch.manual_seed(seed)
    net = mm.MoCoPCI().cuda().eval()      # test.py never calls .eval(); dropout must be off here
    return net


def _time_forward(net, x1, x2, reps=3):
    import time
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        net(x1, x2, None, T_INTERP, False)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


def _load_reference_stack(ref_root):
    """Reference Python + reference kernels; refstack wrappers switch between ref / shadow."""
    from mocopci_b200 import emd_cuda, shim
    from tests import refstack
    _forget()
    sys.modules["pointnet2_cuda"] = refstack.dispatch_pointnet2_module()
    sys.modules["emd_cuda"] = emd_cuda
    p3d, loss, ops = (types.ModuleType(n) for n in ("pytorch3d", "pytorch3d.loss", "pytorch3d.ops"))
    ops.knn_points, ops.knn_gather, loss.chamfer_distance = refstack.torch_knn_points, None, None
    p3d.ops, p3d.loss = ops, loss
    sys.modules.update({"pytorch3d": p3d, "pytorch3d.loss": loss, "pytorch3d.ops": ops})
    sys.modules.update(shim._timm_shim())
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    pcu = importlib.import_module("models.pointconv_util")
    mm = importlib.import_module("models.m_models.mocopci")
    pt = importlib.import_module("models.pointT_layer2")
    assert not hasattr(pcu.knn_point, shim._MARK)          # really the reference's own helpers
    refstack.install_shadow_helpers([pcu, mm])
    refstack.install_shadow_transformer(pt)
    return refstack


@pytest.fixture(scope="module")
def reference_outputs(ref_root):
    """One shadow-mode forward and one plain reference-stack forward (same weights, same input)."""
    from tests import refgpu
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if not refgpu.available():   # a checkout is there: its kernels must be too, or the test would vanish
        pytest.fail("oracle/_ref/libref_*.so missing next to a MoCoPCI checkout: build them with "
                    "make -C oracle ref REF=<checkout>")
    rs = _load_reference_stack(ref_root)
    x1, x2 = _frames(NPTS)
    net = _build()
    rs.STATS.clear()
    del rs.FAILURES[:]
    rs.STACK["mode"] = "shadow"
    with torch.no_grad():
        out_shadow = net(x1, x2, None, T_INTERP, False)
    torch.cuda.synchronize()
    stats, failures = dict(rs.STATS), list(rs.FAILURES)
    rs.STACK["mode"] = "ref"
    with torch.no_grad():
        out_ref = net(x1, x2, None, T_INTERP, False)
        torch.cuda.synchronize()
        ref_ms = _time_forward(net, x1, x2)      # the reference stack on the same GPU, for the record
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "model_shadow_stats.json"), "w") as f:
        json.dump({"npts": NPTS, "calls": stats, "failures": failures,
                   "reference_stack_forward_ms": ref_ms}, f, indent=1)
    return {"shadow": [o.clone() for o in out_shadow], "ref": [o.clone() for o in out_ref],
            "stats": stats, "failures": failures, "ref_ms": ref_ms}


def test_model_shadow_every_hot_path_call(reference_outputs):
    r = reference_outputs
    assert not r["failures"], "\n".join(r["failures"][:20])
    s = r["stats"]
    # the forward really went through every replaced entry point, and every call was compared
    for name in ("furthest_point_sampling_wrapper", "gather_points_wrapper", "group_points_wrapper",
                 "knn_point", "knn_point_cosine", "index_points_group", "index_points_gather",
                 "group", "group_query", "knn_points", "transformer_knn"):
        assert s.get(name, 0) > 0, f"{name} never called"
        assert s.get(name + ":checked", 0) > 0, f"{name} never compared ({s})"
    assert s["knn_point:checked"] >= 90           # 93 Euclidean knn_point calls per forward (+ 24 knn_points)
    # shadow mode returns the reference results, so the two reference forwards are identical
    for a, b in zip(r["shadow"], r["ref"]):
        assert torch.equal(a, b)


def test_model_forward_through_install_matches_reference_stack(reference_outputs, ref_root):
    """The product path: fresh import of the reference modules under mocopci_b200.install()."""
    import mocopci_b200
    from mocopci_b200 import pointnet2_cuda, shim
    _forget()
    done = mocopci_b200.install(reference_root=ref_root)
    assert done == {}                                  # nothing imported yet: the hook patches later
    mm = importlib.import_module("models.m_models.mocopci")
    pcu = importlib.import_module("models.pointconv_util")
    p2u = importlib.import_module("models.pointnet2.pointnet2_utils")
    assert p2u.pointnet2 is pointnet2_cuda
    for mod in (mm, pcu):
        for name in ("knn_point", "knn_point_cosine", "index_points_group", "index_points_gather"):
            assert hasattr(getattr(mod, name), shim._MARK), f"{mod.__name__}.{name} not re-pointed"
    assert hasattr(mm.index_points, shim._MARK)
    x1, x2 = _frames(NPTS)
    net = _build()
    with torch.no_grad():
        out = net(x1, x2, None, T_INTERP, False)
    torch.cuda.synchronize()
    assert len(out) == 3
    report = []
    for j, (o, r) in enumerate(zip(out, reference_outputs["ref"])):
        assert o.shape == r.shape and torch.isfinite(o).all()
        diff = (o - r).abs()
        scale = float(r.abs().max())
        # Two separately executed networks: KNN neighbour ORDER differs (torch.topk is unsorted, ours
        # is sorted), so sums over neighbours are associated differently and the ~1e-6 differences
        # pass through FPS / KNN decisions on network-predicted points. The per-call parity is the
        # shadow test above; here the bar is: the bulk of the cloud agrees to 1e-3 of the scene
        # scale and the clouds are the same cloud (Chamfer distance between them ~ 0).
        from mocopci_b200 import chamfer
        cd = float(chamfer.chamfer_distance(o.contiguous(), r.contiguous())[0])
        med, p99, mx = (float(diff.median()), float(diff.flatten().kthvalue(int(0.99 * diff.numel()))[0]),
                        float(diff.max()))
        report.append({"frame": j, "median_abs": med, "p99_abs": p99, "max_abs": mx, "scale": scale,
                       "chamfer_between_outputs": cd})
        assert med <= 1e-3 * scale, report
        assert cd <= 1e-4 * scale * scale, report
    with torch.no_grad():
        ours_ms = _time_forward(net, x1, x2)
    with open(os.path.join(ROOT, "gpurun_out", "model_end_to_end_diff.json"), "w") as f:
        json.dump({"frames": report, "forward_ms": {"install_b200": ours_ms,
                                                    "reference_stack_same_gpu": reference_outputs["ref_ms"]},
                   "note": "reference stack = the reference's CUDA kernels (oracle/_ref) + its torch KNN "
                           "helpers; B = 1, 16384 points, wall clock with synchronisation, median of 3"},
                  f, indent=1)


def test_model_train_mode_and_eval_metrics_through_install(ref_root):
    """train=True path (mocopci.py:1077-1094: FPS down-sampling of the ground truth) plus the eval
    metrics of test.py:89-90 through the reference's own models/utils.py on the drop-in modules."""
    import mocopci_b200
    _forget()
    mocopci_b200.install(reference_root=ref_root)
    utils = importlib.import_module("models.utils")
    x1, x2 = _frames(4096)
    net = _build()
    gt = [x1.clone(), x2.clone(), x1.clone()]
    with torch.no_grad():
        f_lst, b_lst, gt_frame, out = net(x1, x2, gt, T_INTERP, True)
        assert len(gt_frame) == 3 and [g.shape[-1] for g in gt_frame[0]] == [4096, 1024, 256, 128]
        pred = out[1].permute(0, 2, 1).contiguous()      # [B,3,N] like test.py:88-90 expects
        cd = utils.chamfer_loss(pred, x1)
        emd = utils.EMD(pred, x1)
    assert cd.dim() == 0 and float(cd) > 0 and torch.isfinite(cd)
    assert emd.dim() == 0 and float(emd) > 0 and torch.isfinite(emd)


def test_time_embedding_single_readback_matches_the_reference_loop_on_cuda(ref_root):
    """models/m_models/mocopci.py:172-180 with the CUDA timestamps the model passes
    (mocopci.py:199): the reference converts one 0-d CUDA tensor per table element; the patched
    method reads `t` back once. Same table, bit for bit (the product is the float32 kernel's)."""
    import mocopci_b200
    from mocopci_b200 import shim
    _forget()
    mocopci_b200.install(reference_root=ref_root)
    mm = importlib.import_module("models.m_models.mocopci")
    classes = [c for c in vars(mm).values()
               if isinstance(c, type) and hasattr(vars(c).get("time_embedding"), shim._MARK)]
    assert classes
    for cls in classes:
        original = getattr(vars(cls)["time_embedding"], shim._MARK)
        for stamps in (T_INTERP, [0.0, 1.0, 0.25, 0.3333, 0.9999]):
            t = torch.tensor(stamps, dtype=torch.float32).cuda()
            for dim in (64, 128):
                assert torch.equal(cls.time_embedding(None, t, dim), original(None, t, dim))
