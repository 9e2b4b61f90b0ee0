"""Generate the committed KNN golden fixtures from the REFERENCE'S OWN CODE.

Run in the authoring container only (needs /root/reference):

    python tests/golden/make_golden.py

It imports ``/root/reference/models/pointconv_util.py`` unmodified (its native/third-party
imports ``pointnet2_cuda`` and ``pytorch3d`` are stubbed in ``sys.modules`` -- they are not used by
``square_distance`` / ``knn_point``, pointconv_util.py:67-88,129-140), runs the reference on seeded
inputs on the CPU and stores inputs + outputs as small ``.npz`` files next to this script.
It also cross-checks the C oracle (oracle/oracle.c) against the reference at the full
BASELINE.json size (16384 x 16384) and writes the mismatch counts to ``golden_report.json``.

Nothing here runs on the GPU box; the tests only read the ``.npz`` / ``.json`` files.
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from mocopci_b200 import synth  # noqa: E402
from oracle import cpu as orc  # noqa: E402


def import_reference():
    for name in ("pointnet2_cuda", "pytorch3d", "pytorch3d.ops", "pytorch3d.loss"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["pytorch3d.ops"].knn_points = None
    sys.modules["pytorch3d.loss"].chamfer_distance = None
    sys.path.insert(0, "/root/reference")
    import importlib
    return importlib.import_module("models.pointconv_util")


def run_case(ref, name, xyz, new_xyz, k, report):
    """xyz: refs [B,N,3]; new_xyz: queries [B,S,3] (torch float32, CPU)."""
    D = ref.square_distance(new_xyz, xyz)
    idx = ref.knn_point(k, xyz, new_xyz)
    kk = min(k + 1, xyz.shape[1])
    vals = torch.topk(D, kk, dim=-1, largest=False, sorted=True)[0]
    # layout check: the model mostly passes permuted views of [B,3,N] (mocopci.py:1327)
    xyz_v = xyz.permute(0, 2, 1).contiguous().permute(0, 2, 1)
    new_v = new_xyz.permute(0, 2, 1).contiguous().permute(0, 2, 1)
    D_v = ref.square_distance(new_v, xyz_v)
    layout_mismatch = int((D_v.view(torch.int32) != D.view(torch.int32)).sum())
    # oracle cross-check
    D_o = orc.square_distance(new_xyz.numpy(), xyz.numpy())
    d_mismatch = int((D_o.view(np.int32) != D.numpy().view(np.int32)).sum())
    report[name] = {"shape": [int(x) for x in (xyz.shape[0], new_xyz.shape[1], xyz.shape[1])],
                    "k": k, "oracle_distance_bit_mismatches": d_mismatch,
                    "permuted_view_bit_mismatches": layout_mismatch}
    np.savez_compressed(
        os.path.join(HERE, f"knn_{name}.npz"),
        xyz=xyz.numpy(), new_xyz=new_xyz.numpy(), k=np.int32(k),
        ref_idx=idx.numpy().astype(np.int32), ref_vals=vals.numpy(),
        ref_D_rows=D[:, :8].numpy())
    print(name, report[name])


def run_big_case(ref, name, xyz, new_xyz, k, report):
    """Fixtures that reach the tensor-core scan (N >= 8192 refs): indices, the k+1 smallest values
    and 6 full rows of the reference's matrix are stored, not the matrix (files stay under 1 MB)."""
    D = ref.square_distance(new_xyz, xyz)
    idx = ref.knn_point(k, xyz, new_xyz)
    vals = torch.topk(D, k + 1, dim=-1, largest=False, sorted=True)[0]
    idx_o, dist_o = orc.knn_expanded(k, xyz.numpy(), new_xyz.numpy(), return_dist=True)
    d_ref = np.sort(np.take_along_axis(D.numpy(), idx.numpy(), axis=-1), axis=-1)
    report[name] = {"shape": [int(x) for x in (xyz.shape[0], new_xyz.shape[1], xyz.shape[1])], "k": k,
                    "oracle_queries_with_different_kth_distance_multiset":
                        int((d_ref.view(np.int32) != dist_o.view(np.int32)).any(axis=-1).sum()),
                    "oracle_queries_with_different_index_set":
                        int((np.sort(idx.numpy(), -1) != np.sort(idx_o, -1)).any(axis=-1).sum())}
    np.savez_compressed(
        os.path.join(HERE, f"knn_{name}.npz"),
        xyz=xyz.numpy(), new_xyz=new_xyz.numpy(), k=np.int32(k),
        ref_idx=idx.numpy().astype(np.int32), ref_vals=vals.numpy(), ref_D_rows=D[:, :6].numpy())
    print(name, report[name])


def run_sqdiff_case(name, xyz, k, report):
    """models/pointT_layer2.py:20,62-63: square_distance(xyz, xyz).argsort()[:, :, :k] (pure torch)."""
    import importlib
    pt = importlib.import_module("models.pointT_layer2")
    D = pt.square_distance(xyz, xyz)
    idx = D.argsort()[:, :, :k]
    vals = torch.sort(D, dim=-1)[0][:, :, :k + 1]
    idx_o, dist_o = orc.knn_form(3, k, xyz.numpy(), xyz.numpy())
    d_ref = np.take_along_axis(D.numpy(), idx.numpy(), axis=-1)
    report[name] = {"shape": [int(x) for x in xyz.shape], "k": k,
                    "reference": "models/pointT_layer2.py square_distance :6-20, argsort :62-63",
                    "oracle_distance_bit_mismatches":
                        int((d_ref.view(np.int32) != dist_o.view(np.int32)).sum()),
                    "oracle_queries_with_different_index_set":
                        int((np.sort(idx.numpy(), -1) != np.sort(idx_o, -1)).any(axis=-1).sum())}
    np.savez_compressed(os.path.join(HERE, f"knn_{name}.npz"), xyz=xyz.numpy(), k=np.int32(k),
                        ref_idx=idx.numpy().astype(np.int32), ref_vals=vals.numpy())
    print(name, report[name])


def run_cosine_case(ref, name, S, N, C, k, report, correlated=False):
    """models/pointconv_util.py:111-127,142-153 (pure torch): knn_point_cosine on random features,
    stored as PERMUTED [B,C,N] tensors like the model passes them. The reference's sgemm sums in an
    unspecified order, so the oracle comparison uses a tolerance (recorded here)."""
    g = torch.Generator().manual_seed(1000 + S + N + C)
    xyz_t = torch.randn(1, C, N, generator=g)
    new_t = torch.randn(1, C, S, generator=g)
    if correlated:  # neighbours that really are close: queries = noisy copies of refs
        new_t = xyz_t[:, :, torch.randint(0, N, (S,), generator=g)] + 0.05 * torch.randn(1, C, S, generator=g)
    xyz, new = xyz_t.permute(0, 2, 1), new_t.permute(0, 2, 1)
    D = ref.cosine_distance(new, xyz)
    idx = ref.knn_point_cosine(k, xyz, new)
    vals = torch.topk(D, k + 1, dim=-1, largest=False, sorted=True)[0]
    oi, od = orc.knn_cosine(k, xyz.contiguous().numpy(), new.contiguous().numpy())
    err = float(np.abs(od - vals.numpy()[..., :k]).max())
    gap = (vals[..., k] - vals[..., k - 1]).numpy()
    clear = gap > 4e-6
    same = (np.sort(oi, -1) == np.sort(idx.numpy(), -1)).all(-1)
    report[name] = {"shape": [1, S, N, C], "k": k, "oracle_max_abs_distance_error": err,
                    "queries_with_clear_gap": int(clear.sum()),
                    "oracle_index_set_mismatches_among_clear": int((~same & clear).sum())}
    np.savez_compressed(os.path.join(HERE, f"cos_{name}.npz"), xyz_t=xyz_t.numpy(), new_t=new_t.numpy(),
                        k=np.int32(k), ref_idx=idx.numpy().astype(np.int32), ref_vals=vals.numpy())
    print(name, report[name])


def main():
    torch.manual_seed(0)
    ref = import_reference()
    report = {"torch": torch.__version__, "threads": torch.get_num_threads(),
              "reference": "models/pointconv_util.py square_distance :67-88, knn_point :129-140"}

    a = synth.lidar_frame(1234, 2048)
    b = synth.next_frame(a, 1235)
    run_case(ref, "lidar_k16", a[None], b[None, :512], 16, report)
    run_case(ref, "lidar_self_k32", a[None, :1024], a[None, :1024], 32, report)
    u = synth.uniform_cloud(7, 2, 1000)
    q = synth.uniform_cloud(8, 2, 257)
    run_case(ref, "uniform_k32", u, q, 32, report)
    run_case(ref, "uniform_k3", u[:, :300], q[:, :128], 3, report)
    t = synth.tie_stress_cloud(11, 1, 512)
    run_case(ref, "tie_k16", t, t, 16, report)
    run_case(ref, "tie_k3", t, t[:, :200], 3, report)
    big = synth.uniform_cloud(3, 1, 256, -80.0, 80.0)
    run_case(ref, "wide_k16", big, big, 16, report)

    # reach knn_scan_tc_kernel (N >= 8192): a quarter of the queries of a full frame pair, k = 16,
    # and half a frame pair at k = 32
    fa, fb = synth.frame_pair(0)
    run_big_case(ref, "big_k16", fa[None], fb[None, :4096], 16, report)
    run_big_case(ref, "big_k32", fa[None, :8192], fb[None, 4096:6144], 32, report)
    run_sqdiff_case("sqdiff_k16", synth.lidar_frame(4321, 2048)[None], 16, report)
    run_sqdiff_case("sqdiff_tie_k16", synth.tie_stress_cloud(13, 1, 512), 16, report)

    run_cosine_case(ref, "c64_k16", 700, 1024, 64, 16, report)
    run_cosine_case(ref, "c128_k16", 512, 512, 128, 16, report, correlated=True)
    run_cosine_case(ref, "c256_k16", 256, 256, 256, 16, report)
    run_cosine_case(ref, "c32_k32", 300, 640, 32, 32, report, correlated=True)

    # Full-size cross-check (not stored): BASELINE.json config 0, one 2x16384 frame pair.
    fa, fb = synth.frame_pair(0)
    D = ref.square_distance(fb[None], fa[None])
    idx_ref = ref.knn_point(16, fa[None], fb[None])
    D_o = orc.square_distance(fb[None].numpy(), fa[None].numpy())
    mism = int((D_o.view(np.int32) != D.numpy().view(np.int32)).sum())
    idx_o, dist_o = orc.knn_expanded(16, fa[None].numpy(), fb[None].numpy(), return_dist=True)
    # set parity: compare sorted distance multisets at the returned indices
    d_ref = np.sort(np.take_along_axis(D.numpy(), idx_ref.numpy(), axis=-1), axis=-1)
    set_mism = int((d_ref.view(np.int32) != dist_o.view(np.int32)).any(axis=-1).sum())
    idx_mism = int((np.sort(idx_ref.numpy(), -1) != np.sort(idx_o, -1)).any(axis=-1).sum())
    report["full_16384x16384_k16"] = {
        "oracle_distance_bit_mismatches": mism,
        "queries_with_different_kth_distance_multiset": set_mism,
        "queries_with_different_index_set": idx_mism,
        "note": "index-set differences are only allowed where the reference has a tie at the "
                "k-th distance (torch.topk's tie choice is unspecified, SURVEY section 8c)"}
    print("full", report["full_16384x16384_k16"])
    with open(os.path.join(HERE, "golden_report.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
