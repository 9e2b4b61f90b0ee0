"""``pytorch3d.ops.ball_query`` and ``pytorch3d.ops.sample_farthest_points`` on the B200 kernels.

pytorch3d 0.7.5 is neither vendored nor installed here, so, as for ``knn_points`` (chamfer.py),
PARITY WITH PYTORCH3D ITSELF IS UNPINNED: the docstrings below state the contract, which is this
library's own (include/b200pci.h, P1 / P2), and the tests pin it. Both take ragged batches: the
per-cloud ``lengths`` stay on the device and the kernels read them there, so neither call
synchronises with the host (except ``sample_farthest_points`` with ``random_start_point=True`` or
a CUDA tensor ``K``, see there). Points are 3-D float32 CUDA tensors; there is no CPU fallback.

Gradients: ``ball_query``'s ``dists`` backpropagates into p1 and p2 through b200pci_knn_backward
(b200pci_knn_backward_det under torch.use_deterministic_algorithms), whose rules already fit:
``-1`` slots contribute nothing. ``nn`` and ``sample_farthest_points``' ``selected_points`` are rows
of the input written by the kernels; their gradient is scattered back by the fixed-order row-gather
backward (b200pci_index_points_rows_grad_det), which, unlike the atomic one, skips ``-1`` slots.
``idx`` carries no gradient. An autograd node exists only when an input requires grad.
"""
import torch
from torch.autograd import Function

from . import _lib
from .chamfer import _KNN
from .pointconv_util import _needs_grad

_L = _lib.lib


def _check_cloud(name, t, batch=None):
    if not isinstance(t, torch.Tensor) or t.dim() != 3 or t.shape[2] != 3:
        raise ValueError(f"{name} must be a (B, P, 3) tensor, got "
                         f"{tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__}")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {t.dtype}")
    if batch is not None and t.shape[0] != batch:
        raise ValueError(f"{name} has batch size {t.shape[0]}, expected {batch}")


def _check_lengths(name, lengths, B, like):
    """lengths: None or an int64 (B,) tensor on the clouds' device."""
    if lengths is None:
        return None
    if not isinstance(lengths, torch.Tensor) or lengths.dim() != 1 or lengths.shape[0] != B:
        raise ValueError(f"{name} must be a ({B},) tensor")
    if lengths.dtype != torch.int64:
        raise ValueError(f"{name} must be int64, got {lengths.dtype}")
    if like.is_cuda and lengths.device != like.device:
        raise ValueError(f"{name} must be on {like.device}, got {lengths.device}")
    return lengths.contiguous()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _rows_grad(grad_rows, idx, N, into):
    """into[b, idx[b,t], :] += grad_rows[b, t, :] in the fixed order of the _det kernel; -1 slots skipped."""
    B = idx.shape[0]
    T = idx[0].numel() if B > 0 else 0
    g = grad_rows.contiguous()
    ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(B, N, T), g.device)
    _lib.check(_L.b200pci_index_points_rows_grad_det(B, N, T, 3, g.data_ptr(), idx.data_ptr(), 1, into.data_ptr(),
                                                     ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
               "index_points_rows_grad_det")


# ---- ball_query --------------------------------------------------------------------------------
def _ball_query(p1, p2, lengths1, lengths2, K, radius, want_nn):
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    dev = p1.device
    with _lib.on_device(p1):
        idx = torch.empty((B, P1, K), dtype=torch.int64, device=dev)
        dists = torch.empty((B, P1, K), dtype=torch.float32, device=dev)
        nn = torch.empty((B, P1, K, 3), dtype=torch.float32, device=dev) if want_nn else None
        s1, s2 = p1.stride(), p2.stride()
        _lib.check(_L.b200pci_ball_query_p3d(
            B, P1, P2, K, radius, p1.data_ptr(), s1[0], s1[1], s1[2], p2.data_ptr(), s2[0], s2[1], s2[2],
            _ptr(lengths1), _ptr(lengths2), idx.data_ptr(), dists.data_ptr(), _ptr(nn), _lib.stream_ptr()),
            "ball_query_p3d")
    return dists, idx, nn


class _BallQuery(Function):
    """ball_query with a backward for dists (b200pci_knn_backward, _det under deterministic
    algorithms) and for nn (the fixed-order row-gather backward into p2)."""

    @staticmethod
    def forward(ctx, p1, p2, lengths1, lengths2, K, radius, want_nn):
        dists, idx, nn = _ball_query(p1, p2, lengths1, lengths2, K, radius, want_nn)
        ctx.save_for_backward(p1, p2, idx)
        ctx.mark_non_differentiable(idx)
        return (dists, idx, nn) if want_nn else (dists, idx)

    @staticmethod
    def backward(ctx, grad_dists, _grad_idx, grad_nn=None):
        p1, p2, idx = ctx.saved_tensors
        B, P1, K = idx.shape
        P2 = p2.shape[1]
        dev = p1.device
        with _lib.on_device(p1):
            gq = torch.empty((B, P1, 3), dtype=torch.float32, device=dev)
            gr = torch.empty((B, P2, 3), dtype=torch.float32, device=dev)
            g = grad_dists.contiguous()
            s1, s2 = p1.stride(), p2.stride()
            args = (B, P1, P2, K, p1.data_ptr(), s1[0], s1[1], s1[2], p2.data_ptr(), s2[0], s2[1], s2[2],
                    idx.data_ptr(), 1, g.data_ptr(), gq.data_ptr(), gr.data_ptr())
            if torch.are_deterministic_algorithms_enabled():  # fixed summation order (b200pci.h, _det)
                ws = _lib.workspace(_L.b200pci_scatter_workspace_bytes(B, P2, P1 * K), dev)
                _lib.check(_L.b200pci_knn_backward_det(*args, ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
                           "knn_backward_det")
            else:
                _lib.check(_L.b200pci_knn_backward(*args, _lib.stream_ptr()), "knn_backward")
            if grad_nn is not None:
                _rows_grad(grad_nn.reshape(B, P1 * K, 3), idx, P2, gr)
        return (gq if ctx.needs_input_grad[0] else None, gr if ctx.needs_input_grad[1] else None,
                None, None, None, None, None)


def ball_query(p1, p2, lengths1=None, lengths2=None, K=500, radius=0.2, return_nn=True):
    """``pytorch3d.ops.ball_query``: for each point of p1 (B, P1, 3) the first K points of p2
    (B, P2, 3), in index order, inside the ball of ``radius`` -> KNN(dists, idx, knn).

    For query i < lengths1[b], idx[b,i,:] (int64) holds the first K indices j < lengths2[b], in
    ascending j, with d2 < radius * radius (strict; radius squared in FP32), where
    d2 = fma(dz,dz,fma(dy,dy,dx*dx)), d = p1[b,i] - p2[b,j] (pytorch3d's CUDA arithmetic); dists
    holds those d2. Slots past the hits, and every slot of a query i >= lengths1[b], are idx = -1
    and dists = 0. knn (return_nn) is p2[b, idx] (B, P1, K, 3), zeros where idx = -1, else None.

    p1 / p2: float32 CUDA tensors, strided views accepted. lengths1 / lengths2: None (every cloud
    full) or int64 (B,) tensors on the same device, clamped to [0, P] by the kernel, never read on
    the host: the call takes no host synchronisation and is CUDA-graph capturable.
    ValueError: shapes, batch sizes, lengths of the wrong shape / dtype / device, K < 1, radius < 0
    or NaN. RuntimeError: CPU tensors."""
    _check_cloud("p1", p1)
    _check_cloud("p2", p2, p1.shape[0])
    B = p1.shape[0]
    if isinstance(K, bool) or not isinstance(K, int) or K < 1:
        raise ValueError(f"K must be an int >= 1, got {K!r}")
    radius = float(radius)
    if not radius >= 0.0:
        raise ValueError(f"radius must be >= 0, got {radius}")
    _lib.require_cuda(p1, p2)
    if p2.device != p1.device:
        raise ValueError(f"p1 and p2 are on different devices ({p1.device}, {p2.device})")
    lengths1 = _check_lengths("lengths1", lengths1, B, p1)
    lengths2 = _check_lengths("lengths2", lengths2, B, p1)
    if _needs_grad(p1, p2):
        out = _BallQuery.apply(p1, p2, lengths1, lengths2, K, radius, bool(return_nn))
        dists, idx, nn = out if return_nn else (out[0], out[1], None)
    else:
        dists, idx, nn = _ball_query(p1, p2, lengths1, lengths2, K, radius, bool(return_nn))
    return _KNN(dists=dists, idx=idx, knn=nn)


# ---- sample_farthest_points --------------------------------------------------------------------
def _fps(points, lengths, Kt, start, M):
    B, P, _ = points.shape
    dev = points.device
    with _lib.on_device(points):
        idx = torch.empty((B, M), dtype=torch.int64, device=dev)
        sel = torch.empty((B, M, 3), dtype=torch.float32, device=dev)
        s = points.stride()
        _lib.check(_L.b200pci_fps_p3d(B, P, M, points.data_ptr(), s[0], s[1], s[2], _ptr(lengths), _ptr(Kt),
                                      _ptr(start), idx.data_ptr(), sel.data_ptr(), _lib.stream_ptr()),
                   "fps_p3d")
    return sel, idx


class _Fps(Function):
    """sample_farthest_points with a backward for the selected rows (fixed-order row scatter)."""

    @staticmethod
    def forward(ctx, points, lengths, Kt, start, M):
        sel, idx = _fps(points, lengths, Kt, start, M)
        ctx.save_for_backward(idx)
        ctx.npoints = points.shape[1]
        ctx.mark_non_differentiable(idx)
        return sel, idx

    @staticmethod
    def backward(ctx, grad_sel, _grad_idx):
        (idx,) = ctx.saved_tensors
        B = idx.shape[0]
        with _lib.on_device(grad_sel):
            gp = torch.zeros((B, ctx.npoints, 3), dtype=torch.float32, device=grad_sel.device)
            _rows_grad(grad_sel, idx, ctx.npoints, gp)
        return gp, None, None, None, None


def sample_farthest_points(points, lengths=None, K=50, random_start_point=False):
    """``pytorch3d.ops.sample_farthest_points``: iterative farthest point sampling of points
    (B, P, 3) -> (selected_points (B, max K, 3), idx int64 (B, max K)).

    Per cloud, n = lengths[b] points and min(K_b, n) picks. The first pick is index 0, or with
    random_start_point ``torch.randint(high=n, size=(1,))`` drawn per cloud from torch's global
    generator (no draw for an empty cloud). Each later pick is the argmax over j < n of the running
    minimum, over the earlier picks, of d2 = fma(dz,dz,fma(dy,dy,dx*dx)); among equal values the
    LOWEST index wins (ops.furthest_point_sample keeps the pointnet2 kernel's order instead). Picks
    past min(K_b, n) are -1 and their rows of selected_points zeros. selected_points carries a
    gradient into points; idx none.

    K: an int >= 1, or a (B,) integer tensor with every entry >= 1. lengths: None or an int64 (B,)
    tensor on the points' device, clamped to [0, P] by the kernel. The call itself takes no host
    synchronisation, with two exceptions: random_start_point reads lengths on the host (pytorch3d's
    host loop), and a CUDA tensor K is read on the host for the output width (a CPU K is copied to
    the device instead). At most 131072 points per cloud.
    ValueError: shapes, lengths / K of the wrong shape or dtype, K < 1. RuntimeError: CPU points."""
    _check_cloud("points", points)
    B, P, _ = points.shape
    if isinstance(K, torch.Tensor):
        if K.dim() != 1 or K.shape[0] != B:
            raise ValueError(f"K must be an int or a ({B},) tensor")
        if K.dtype.is_floating_point or K.dtype.is_complex or K.dtype == torch.bool:
            raise ValueError(f"K must be an integer tensor, got {K.dtype}")
        if B > 0:
            kmin, kmax = (int(v) for v in torch.stack([K.min(), K.max()]).tolist())
        else:
            kmin = kmax = 1
        if kmin < 1:
            raise ValueError(f"every K must be >= 1, got {kmin}")
        M = kmax if B > 0 else 0
    elif isinstance(K, bool) or not isinstance(K, int):
        raise ValueError(f"K must be an int or a ({B},) tensor, got {type(K).__name__}")
    else:
        if K < 1:
            raise ValueError(f"K must be >= 1, got {K}")
        M = K
    if P > 131072:
        raise ValueError(f"sample_farthest_points: at most 131072 points per cloud, got {P}")
    _lib.require_cuda(points)
    lengths = _check_lengths("lengths", lengths, B, points)
    dev = points.device
    Kt = K.to(device=dev, dtype=torch.int64).contiguous() if isinstance(K, torch.Tensor) else None
    start = None
    if random_start_point:
        ns = lengths.tolist() if lengths is not None else [P] * B
        start = torch.tensor([int(torch.randint(high=min(n, P), size=(1,)).item()) if min(n, P) > 0 else 0
                              for n in ns], dtype=torch.int64).to(dev)
    if _needs_grad(points):
        return _Fps.apply(points, lengths, Kt, start, M)
    return _fps(points, lengths, Kt, start, M)
