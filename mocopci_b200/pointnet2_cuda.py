"""Drop-in for the reference's pybind module ``pointnet2_cuda``.

Same function names, positional arguments and in-place output convention as
pointnet2/src/pointnet2_api.cpp:10-24 (the caller allocates every output, the kernels write in
place on the current CUDA stream, the return value is ignored), so both
``pointnet2/pointnet2_utils.py`` and ``models/pointnet2/pointnet2_utils.py`` of the reference run
unchanged on top of it once ``mocopci_b200.install()`` has registered this module as
``sys.modules["pointnet2_cuda"]``. Failures raise ``RuntimeError`` instead of ``exit(-1)``.

Under ``torch.use_deterministic_algorithms(True)`` (``warn_only`` included) the three gradient
wrappers run the fixed-order ``*_grad_det`` kernels instead of the atomic ones: the gradients are
then the same bits on every run (include/b200pci.h, "deterministic gradients").
"""
import torch

from . import _lib

_L = _lib.lib


def _f32(t, name):
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous float32 tensor")
    _lib.require_cuda(t)
    return t.data_ptr()


def _i32(t, name):
    if t.dtype != torch.int32 or not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous int32 tensor")
    _lib.require_cuda(t)
    return t.data_ptr()


def furthest_point_sampling_wrapper(b, n, m, points_tensor, temp_tensor, idx_tensor):
    """sampling.cpp:38-49."""
    with _lib.on_device(points_tensor):
        _lib.check(_L.b200pci_furthest_point_sampling(
            b, n, m, _f32(points_tensor, "points"), _f32(temp_tensor, "temp"),
            _i32(idx_tensor, "idx"), _lib.stream_ptr()), "furthest_point_sampling")
    return 1


def gather_points_wrapper(b, c, n, npoints, points_tensor, idx_tensor, out_tensor):
    """sampling.cpp:11-22."""
    with _lib.on_device(points_tensor):
        _lib.check(_L.b200pci_gather_points(
            b, c, n, npoints, _f32(points_tensor, "points"), _i32(idx_tensor, "idx"),
            _f32(out_tensor, "out"), _lib.stream_ptr()), "gather_points")
    return 1


def gather_points_grad_wrapper(b, c, n, npoints, grad_out_tensor, idx_tensor, grad_points_tensor):
    """sampling.cpp:25-35."""
    with _lib.on_device(grad_out_tensor):
        if torch.are_deterministic_algorithms_enabled():
            ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(b, n, npoints), grad_out_tensor.device)
            _lib.check(_L.b200pci_gather_points_grad_det(
                b, c, n, npoints, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
                _f32(grad_points_tensor, "grad_points"), ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
                "gather_points_grad_det")
            return 1
        _lib.check(_L.b200pci_gather_points_grad(
            b, c, n, npoints, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
            _f32(grad_points_tensor, "grad_points"), _lib.stream_ptr()), "gather_points_grad")
    return 1


def ball_query_wrapper(b, n, m, radius, nsample, new_xyz_tensor, xyz_tensor, idx_tensor):
    """ball_query.cpp:16-28."""
    with _lib.on_device(xyz_tensor):
        nbytes = _L.b200pci_ball_query_workspace_bytes(b, n, m, nsample)
        ws = _lib.workspace(nbytes, xyz_tensor.device)
        _lib.check(_L.b200pci_ball_query(
            b, n, m, float(radius), nsample, _f32(new_xyz_tensor, "new_xyz"),
            _f32(xyz_tensor, "xyz"), _i32(idx_tensor, "idx"), ws.data_ptr(), ws.numel(),
            _lib.stream_ptr()), "ball_query")
    return 1


def group_points_wrapper(b, c, n, npoints, nsample, points_tensor, idx_tensor, out_tensor):
    """group_points.cpp:27-38."""
    with _lib.on_device(points_tensor):
        _lib.check(_L.b200pci_group_points(
            b, c, n, npoints, nsample, _f32(points_tensor, "points"), _i32(idx_tensor, "idx"),
            _f32(out_tensor, "out"), _lib.stream_ptr()), "group_points")
    return 1


def group_points_grad_wrapper(b, c, n, npoints, nsample, grad_out_tensor, idx_tensor,
                              grad_points_tensor):
    """group_points.cpp:11-24."""
    with _lib.on_device(grad_out_tensor):
        if torch.are_deterministic_algorithms_enabled():
            ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(b, n, npoints * nsample), grad_out_tensor.device)
            _lib.check(_L.b200pci_group_points_grad_det(
                b, c, n, npoints, nsample, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
                _f32(grad_points_tensor, "grad_points"), ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
                "group_points_grad_det")
            return 1
        _lib.check(_L.b200pci_group_points_grad(
            b, c, n, npoints, nsample, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
            _f32(grad_points_tensor, "grad_points"), _lib.stream_ptr()), "group_points_grad")
    return 1


def three_nn_wrapper(b, n, m, unknown_tensor, known_tensor, dist2_tensor, idx_tensor):
    """interpolate.cpp:14-25."""
    with _lib.on_device(unknown_tensor):
        nbytes = _L.b200pci_three_nn_workspace_bytes(b, n, m)
        ws = _lib.workspace(nbytes, unknown_tensor.device)
        _lib.check(_L.b200pci_three_nn(
            b, n, m, _f32(unknown_tensor, "unknown"), _f32(known_tensor, "known"),
            _f32(dist2_tensor, "dist2"), _i32(idx_tensor, "idx"), ws.data_ptr(), ws.numel(),
            _lib.stream_ptr()), "three_nn")


def three_interpolate_wrapper(b, c, m, n, points_tensor, idx_tensor, weight_tensor, out_tensor):
    """interpolate.cpp:28-41."""
    with _lib.on_device(points_tensor):
        _lib.check(_L.b200pci_three_interpolate(
            b, c, m, n, _f32(points_tensor, "points"), _i32(idx_tensor, "idx"),
            _f32(weight_tensor, "weight"), _f32(out_tensor, "out"), _lib.stream_ptr()),
            "three_interpolate")


def three_interpolate_grad_wrapper(b, c, n, m, grad_out_tensor, idx_tensor, weight_tensor,
                                   grad_points_tensor):
    """interpolate.cpp:44-57."""
    with _lib.on_device(grad_out_tensor):
        if torch.are_deterministic_algorithms_enabled():
            ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(b, m, 3 * n), grad_out_tensor.device)
            _lib.check(_L.b200pci_three_interpolate_grad_det(
                b, c, n, m, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
                _f32(weight_tensor, "weight"), _f32(grad_points_tensor, "grad_points"), ws.data_ptr(),
                ws.numel(), _lib.stream_ptr()), "three_interpolate_grad_det")
            return
        _lib.check(_L.b200pci_three_interpolate_grad(
            b, c, n, m, _f32(grad_out_tensor, "grad_out"), _i32(idx_tensor, "idx"),
            _f32(weight_tensor, "weight"), _f32(grad_points_tensor, "grad_points"),
            _lib.stream_ptr()), "three_interpolate_grad")
