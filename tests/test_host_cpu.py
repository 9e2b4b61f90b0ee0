"""CPU tests (no GPU): the C ABI loads and exports everything include/b200pci.h declares, the
host-side mirror keeps the reference's names, argument errors surface as RuntimeError, the
synthetic generator is deterministic, and the sharded harness logic works under gloo (world 2)."""
import ctypes
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import _lib
    return _lib


def test_abi_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "b200pci.h")).read()
    declared = set(re.findall(r"\b(b200pci_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 24
    for name in declared:
        assert hasattr(lib.lib, name), f"{name} declared in b200pci.h but not exported"
    assert declared == set(lib.PROTOTYPES), "ctypes prototypes out of sync with the header"
    assert lib.lib.b200pci_version() == 100


def test_abi_argument_errors_without_gpu(lib):
    L = lib.lib
    # sizes / workspace queries never touch the device
    assert L.b200pci_knn_workspace_bytes(8, 16384, 16384, 16) >= 8 * 4 * 16384 * 4
    assert L.b200pci_emd_workspace_bytes(1, 100, 200) >= (100 + 200) * 2 * 4
    assert L.b200pci_three_nn_workspace_bytes(2, 10, 5) > 0
    # invalid arguments return EINVAL with a message instead of exiting the process
    rc = L.b200pci_knn(1, 4, 8, 16, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None)
    assert rc == -1 and b"out of range" in L.b200pci_last_error()
    rc = L.b200pci_knn(1, 4, 8, 99, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None)
    assert rc == -1
    with pytest.raises(RuntimeError, match="out of range"):
        lib.check(L.b200pci_knn(1, 4, 8, 16, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None,
                                0, None), "knn")
    assert L.b200pci_furthest_point_sampling(1, 0, 4, None, None, None, None) == -1
    assert L.b200pci_furthest_point_sampling(0, 10, 4, None, None, None, None) == 0  # empty batch
    assert L.b200pci_group_points(0, 3, 10, 4, 4, None, None, None, None) == 0
    assert L.b200pci_debug_set(99, 0.0) == -1
    for key in (8, 9, 17):  # keys of removed KNN paths: a stale caller fails instead of running the default
        assert L.b200pci_debug_set(key, 0.0) == -1 and L.b200pci_debug_set(key, 1.0) == -1


def test_new_entry_points_argument_handling_without_gpu(lib):
    """Shape rules of the round-2 entry points are decided on the host: unsupported cosine shapes report
    0 workspace bytes (the caller keeps the reference path), empty problems return 0 without touching
    the device, bad arguments give EINVAL with a message."""
    L = lib.lib
    ws = L.b200pci_knn_cosine_workspace_bytes
    assert ws(1, 2048, 2048, 64, 16) > 0 and ws(2, 300, 4096, 512, 32) > 0
    assert ws(1, 100, 100, 50, 8) == 0        # C % 16 != 0
    assert ws(1, 100, 100, 64, 33) == 0       # k > 32
    assert ws(1, 100, 5000, 64, 16) == 0      # N > 4096
    assert ws(1, 100, 8, 64, 16) == 0         # k > N
    assert L.b200pci_knn_cosine(1, 0, 100, 64, 16, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None) == 0
    rc = L.b200pci_knn_cosine(1, 10, 100, 50, 8, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None)
    assert rc == -1 and b"unsupported shape" in L.b200pci_last_error()
    assert L.b200pci_group_concat(0, 10, 10, 4, 3, None, 0, 0, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, None) == 0
    assert L.b200pci_group_concat(1, 10, 10, 0, 3, None, 0, 0, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, None) == 0
    assert L.b200pci_group_concat(1, 10, 10, 4, 3, None, 0, 0, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, None) == -1
    assert L.b200pci_emd_cost(0, 10, 10, None, None, None, None, 0, None) == 0
    assert L.b200pci_emd_cost(1, 10, 10, None, None, None, None, 0, None) == -1       # null cost
    assert L.b200pci_three_nn_weights(0, 10, 5, None, None, 1e-8, None, None, None, None, 0, None) == 0
    assert L.b200pci_three_nn_weights(1, 10, 5, None, None, 1e-8, None, None, None, None, 0, None) == -1
    assert L.b200pci_knn(1, 4, 8, 2, 9, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None) == -1   # bad mode
    assert b"dist_mode" in L.b200pci_last_error()
    assert L.b200pci_knn(1, 4, 64, 40, 3, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None) == -1  # SQDIFF: k <= 32
    assert L.b200pci_query_group(0, 10, 4, 4, 3, None, None, None, None, None, 1, None) == 0          # empty batch
    assert L.b200pci_query_group(1, 10, 4, 0, 3, None, None, None, None, None, 1, None) == 0          # nsample 0
    assert L.b200pci_query_group(1, 10, 4, 4, 0, None, None, None, None, None, 0, None) == -1         # nothing to group
    assert L.b200pci_query_group(1, 10, 4, 4, 3, None, None, None, None, None, 1, None) == -1         # null pointers
    assert b"null pointer" in L.b200pci_last_error()
    assert L.b200pci_host_release() in (0, -2)   # nothing to free; -2 only if no CUDA runtime/device


def test_ops_refuse_cpu_tensors(lib):
    from mocopci_b200 import ops, pointconv_util
    x = torch.rand(1, 32, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        pointconv_util.knn_point(4, x, x)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.furthest_point_sample(x, 8)


def test_api_keeps_reference_names(lib):
    from mocopci_b200 import chamfer, emd_cuda, ops, pointconv_util, pointnet2_cuda
    for n in ("furthest_point_sampling_wrapper", "gather_points_wrapper", "gather_points_grad_wrapper",
              "ball_query_wrapper", "group_points_wrapper", "group_points_grad_wrapper",
              "three_nn_wrapper", "three_interpolate_wrapper", "three_interpolate_grad_wrapper"):
        assert callable(getattr(pointnet2_cuda, n))  # pointnet2_api.cpp:10-24
    for n in ("approxmatch_forward", "matchcost_forward", "matchcost_backward"):
        assert callable(getattr(emd_cuda, n))  # emd.cpp:23-27
    for n in ("furthest_point_sample", "gather_operation", "three_nn", "three_interpolate",
              "grouping_operation", "ball_query", "query_and_group", "earth_mover_distance"):
        assert callable(getattr(ops, n))
    for n in ("knn_point", "knn_point_cosine", "index_points_gather", "index_points_group"):
        assert callable(getattr(pointconv_util, n))
    assert callable(chamfer.chamfer_distance) and callable(chamfer.knn_points) and callable(chamfer.knn_gather)


@pytest.fixture()
def clean_modules():
    """install() mutates sys.modules / sys.meta_path / sys.path: restore them afterwards."""
    from mocopci_b200 import shim
    from tests import cpu_natives
    saved_modules, saved_path = dict(sys.modules), list(sys.path)
    cpu_natives.forget_reference_modules()
    yield
    shim.uninstall()
    for k in list(sys.modules):
        if k not in saved_modules:
            del sys.modules[k]
    sys.modules.update(saved_modules)
    sys.path[:] = saved_path


def test_install_registers_dropin_modules(lib, clean_modules):
    import mocopci_b200
    fake = types.ModuleType("models.pointconv_util")
    fake.knn_point = lambda *a: "original"
    fake.alias = fake.knn_point
    sys.modules["models.pointconv_util"] = fake
    original = fake.knn_point
    patched = mocopci_b200.install()
    import emd_cuda
    import pointnet2_cuda
    assert pointnet2_cuda.__name__ == "mocopci_b200.pointnet2_cuda"
    assert emd_cuda.__name__ == "mocopci_b200.emd_cuda"
    from pytorch3d.loss import chamfer_distance
    from pytorch3d.ops import knn_gather, knn_points
    assert callable(chamfer_distance) and callable(knn_points) and callable(knn_gather)
    from timm.models.layers import DropPath, to_2tuple, trunc_normal_  # noqa: F401
    assert patched == {"models.pointconv_util": ["knn_point"]}
    from mocopci_b200 import shim
    assert getattr(fake.knn_point, shim._MARK) is original and fake.alias is fake.knn_point
    # inputs the kernels do not cover run the reference's own code (CPU tensors, C != 3)
    x = torch.rand(1, 8, 3)
    assert fake.knn_point(4, x, x) == "original"
    assert mocopci_b200.install() == {}            # idempotent
    shim.uninstall()
    assert fake.knn_point is original


def test_install_against_the_real_reference_modules(lib, ref_root, clean_modules):
    """install() BEFORE the reference is imported (the documented flow): the post-import hook must
    re-point every copy of the helpers in the real models.pointconv_util / models.m_models.mocopci
    (module globals, aliases included) and the pointT_layer2 neighbour search; the reference's own
    pointnet2_utils / EMD wrappers must bind our pybind look-alikes."""
    import importlib
    import mocopci_b200
    from mocopci_b200 import emd_cuda, pointnet2_cuda, shim
    assert mocopci_b200.install(reference_root=ref_root) == {}
    mm = importlib.import_module("models.m_models.mocopci")
    pcu = importlib.import_module("models.pointconv_util")
    pt = importlib.import_module("models.pointT_layer2")
    for mod in (mm, pcu):
        for name in shim._HELPERS:
            assert hasattr(getattr(mod, name), shim._MARK), f"{mod.__name__}.{name}"
    assert hasattr(mm.index_points, shim._MARK)                     # mocopci.py:12 alias
    assert hasattr(pt.square_distance, shim._MARK)
    assert importlib.import_module("pointnet2.pointnet2_utils").pointnet2 is pointnet2_cuda
    assert importlib.import_module("models.pointnet2.pointnet2_utils").pointnet2 is pointnet2_cuda
    assert importlib.import_module("models.EMD.emd").emd_cuda is emd_cuda
    assert importlib.import_module("models.utils").emd_cuda is emd_cuda
    # patching after the import works too, and uninstall restores the reference's own functions
    shim.uninstall()
    assert not hasattr(pcu.knn_point, shim._MARK) and not hasattr(pt.square_distance, shim._MARK)
    again = mocopci_b200.install()
    assert "models.pointconv_util" in again and "models.m_models.mocopci" in again
    # CPU inputs fall through to the reference's own torch code
    x = torch.rand(1, 40, 3)
    idx = pcu.knn_point(4, x, x)
    assert idx.shape == (1, 40, 4) and bool((idx[..., :1] >= 0).all())
    d = pt.square_distance(x, x)
    assert torch.is_tensor(d) and d.shape == (1, 40, 40)


def test_time_embedding_host_evaluation_is_bit_identical(lib, ref_root, clean_modules):
    """shim._patch_time_embedding: the reference's element-by-element sinusoid table
    (models/m_models/mocopci.py:172-180; one tensor -> Python scalar conversion per element) against
    the single read-back evaluation, on the reference's own timestamps and a few awkward ones."""
    import importlib
    import mocopci_b200
    from mocopci_b200 import shim
    mocopci_b200.install(reference_root=ref_root)
    mm = importlib.import_module("models.m_models.mocopci")
    sm = importlib.import_module("models.sim_models.simplified_trans")
    classes = [c for mod in (mm, sm) for c in vars(mod).values()
               if isinstance(c, type) and hasattr(vars(c).get("time_embedding"), shim._MARK)]
    assert len(classes) >= 2
    for cls in classes:
        original = getattr(vars(cls)["time_embedding"], shim._MARK)
        for stamps in ([0.4167, 0.5, 0.5833], [0.0, 1.0], [0.1, 1e-3, 0.999999, 3.25, 117.0]):
            t = torch.tensor(stamps, dtype=torch.float32)
            for dim in (64, 128, 7):
                want = original(None, t, dim)
                got = cls.time_embedding(None, t, dim)
                assert got.dtype == want.dtype and got.shape == want.shape
                assert torch.equal(got, want), (cls.__name__, stamps, dim)
        # anything but a 1-D float32 tensor runs the reference's own loop
        t64 = torch.tensor([0.5], dtype=torch.float64)
        assert torch.equal(cls.time_embedding(None, t64, 8), original(None, t64, 8))
    shim.uninstall()
    assert all(not hasattr(vars(c)["time_embedding"], shim._MARK) for c in classes)


def test_unmodified_reference_model_runs_through_install_on_cpu(lib, ref_root, clean_modules, orc):
    """Host logic of the drop-in, no GPU: the unmodified MoCoPCI model, imported AFTER install(),
    runs one forward at 2048 points with oracle-backed natives (tests/cpu_natives.py) -- every
    patched helper is reached and falls through to the reference's own code for CPU tensors."""
    import importlib
    import mocopci_b200
    from mocopci_b200 import shim, synth
    from tests import cpu_natives as cn
    mocopci_b200.install(reference_root=ref_root)
    sys.modules["pointnet2_cuda"] = cn.make_pointnet2_cuda()
    sys.modules["emd_cuda"] = cn.make_emd_cuda()
    sys.modules.update(cn.make_pytorch3d())
    calls = {}
    with cn.cuda_on_cpu():
        mm = importlib.import_module("models.m_models.mocopci")
        pcu = importlib.import_module("models.pointconv_util")
        for mod in (mm, pcu):
            for name in ("knn_point", "index_points_group", "index_points_gather"):
                fn = getattr(mod, name)
                assert hasattr(fn, shim._MARK)

                def counted(*a, _fn=fn, _key=f"{mod.__name__}.{name}"):
                    calls[_key] = calls.get(_key, 0) + 1
                    return _fn(*a)
                setattr(mod, name, counted)
        torch.manual_seed(0)
        net = mm.MoCoPCI().eval()
        x = [synth.lidar_frame(100 + i, 2048).t()[None].contiguous() for i in range(2)]
        with torch.no_grad():
            out = net(x[0], x[1], None, [0.4167, 0.5, 0.5833], False)
    assert len(out) == 3 and all(o.shape == (1, 2048, 3) and torch.isfinite(o).all() for o in out)
    assert calls.get("models.m_models.mocopci.knn_point", 0) >= 10
    assert calls.get("models.pointconv_util.knn_point", 0) >= 10
    assert calls.get("models.pointconv_util.index_points_group", 0) >= 10


def _write_nldrive_fixture(root, sizes, seed=0):
    """A one-scene NL-Drive look-alike: raw float32 [n,3] .bin frames and a scene list with two
    7-frame samples (4 inputs + 3 targets at interval 4, data/no_norm_datasets.py:59-63)."""
    rng = np.random.default_rng(seed)
    os.makedirs(os.path.join(root, "scene0"), exist_ok=True)
    names = []
    for i, n in enumerate(sizes):
        name = os.path.join("scene0", f"{i:04d}.bin")
        (rng.standard_normal((n, 3)) * 20).astype(np.float32).tofile(os.path.join(root, name))
        names.append(name)
    lst = os.path.join(root, "list.txt")
    with open(lst, "w") as f:
        f.write(" ".join(names[:7]) + "\n")
        f.write(" ".join(names[2:9]) + "\n")
    return lst


def test_nldrive_dataset_matches_the_reference_class(lib, ref_root, clean_modules, tmp_path):
    """SURVEY 8f-4: mocopci_b200.data.NLDriveDataset against the reference's own class
    (data/no_norm_datasets.py, imported unmodified) on raw frames larger AND smaller than num_points
    (sampling without replacement / in-order + padding with replacement): same tensors, bit for bit,
    and the global numpy generator is left in the same state."""
    import importlib
    from mocopci_b200 import data as ours
    sys.path.insert(0, ref_root)
    ref = importlib.import_module("data.no_norm_datasets")
    root = str(tmp_path)
    lst = _write_nldrive_fixture(root, [5000, 900, 1024, 3000, 700, 1025, 2048, 64, 4096])
    for num_points in (1024, 2048):
        a = ref.NLDriveDataset(root, lst, num_points=num_points, interval=4, num_frames=4)
        b = ours.NLDriveDataset(root, lst, num_points=num_points, interval=4, num_frames=4)
        assert len(a) == len(b) == 2
        for index in (0, 1, 0):
            np.random.seed(100 + index)
            ia, ga = a[index]
            state_a = np.random.get_state()[1].copy()
            np.random.seed(100 + index)
            ib, gb = b[index]
            state_b = np.random.get_state()[1].copy()
            assert len(ia) == len(ib) == 4 and len(ga) == len(gb) == 3
            for x, y in zip(ia + ga, ib + gb):
                assert x.dtype == y.dtype == torch.float32 and x.shape == y.shape == (num_points, 3)
                assert torch.equal(x, y)
            assert np.array_equal(state_a, state_b)
    with pytest.raises(ValueError, match="gather_on_device"):
        ours.NLDriveDataset(root, lst, gather_on_device=True)


def test_synthetic_frames_are_deterministic():
    from mocopci_b200 import synth
    a1, b1 = synth.frame_pair(3, 4096)
    a2, b2 = synth.frame_pair(3, 4096)
    assert torch.equal(a1, a2) and torch.equal(b1, b2)
    assert a1.shape == (4096, 3) and a1.dtype == torch.float32
    assert float(a1.norm(dim=1).max()) < 90 and float((a1 - b1).norm(dim=1).median()) < 2.5
    t = synth.tie_stress_cloud(1, 1, 100)
    assert len(np.unique(t[0].numpy(), axis=0)) <= 51


def test_sharded_eval_logic_gloo_world2():
    """The multi-GPU path of bench.py / eval harness on CPU: 2 ranks over gloo own disjoint frame
    pairs and reduce their metrics with one all_reduce."""
    env = dict(os.environ, REPO=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                          "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port",
                          "29617", os.path.join(ROOT, "tests", "_gloo_worker.py")],
                         env=env, capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "OK" in out.stdout


def test_bench_reference_arm_smoke():
    """`bench.py --impl reference` needs no GPU and prints one JSON line with the contract keys."""
    import json
    env = dict(os.environ, OMP_NUM_THREADS="8")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                         timeout=300, env=env)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "queries/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0
