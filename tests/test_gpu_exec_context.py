"""The kernels as bench.py and the eval loop run them, not only as one eager call on torch's default
stream: CUDA-graph capture and replay, a second stream, concurrent host threads, a second device.

A mistake in any of these (a launch on the wrong stream, a missing join of the library's side
stream, a counter that relies on zeroed scratch, per-thread state created on the wrong device or
during a capture) leaves every eager default-stream result unchanged. So every test here compares
with an eager call on the default stream with the same inputs, bit for bit (the forward kernels and
the `_det` backwards are run-to-run deterministic). What the C oracle covers (the KNN forms, FPS,
ball query, three_nn, Chamfer per point, the `_det` gradients) is also checked against it once, so
that stale output is never compared with stale output.

- Graphs: every call bench.py's extras() times is captured as graph_median captures it (the capture
  must succeed: graph_median would silently time the eager call instead), replayed, then replayed
  again on the next frame pairs copied into its static inputs. The second replay runs on the first
  one's leftover workspace. Also: the two-pass KNN's redo path with its side stream inside a graph,
  a capture that is a fresh host thread's first library call, forward + `_det` backward in a graph.
- A second stream: a stream held back (torch.cuda._sleep) copies the real inputs over buffers that
  hold another valid input set, runs the op and consumes its outputs before any synchronisation.
  A launch on the wrong stream reads the stale set; a missing join lets the consumer read rows the
  side stream has not written yet. Then the eval leg's pattern: KNN on the main stream, Chamfer +
  EMD on a second one, interleaved.
- Host threads, each with its own stream, and the host-buffer entry point from two threads.
- A second device (skipped unless two are visible).

The exact-redo path of the two-pass KNN only runs for queries its estimated bound flags; the tests
that need it force it with test hook 1 (b200pci_debug_set(1, scale < 1)) at a scale that flags
between 32 and 2048 queries, so that the per-query redo on the library's side stream has work to
do. The hooks are process-global: they are set before any thread starts and restored in `finally`.
"""
import contextlib
import threading

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

NPTS = 16384
SLEEP = 100_000_000   # torch.cuda._sleep cycles: ~50 ms at B200 clocks, far longer than any call here
REDO_SPARSE_MAX = 2048  # knn.cu: flagged queries up to which the per-query redo (side stream) runs


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def same(a, b):
    """Bitwise equality of tensors (float32 compared as int32: -0.0 != 0.0, NaN == NaN) or of
    tuples / lists of them."""
    if isinstance(a, (tuple, list)):
        return isinstance(b, (tuple, list)) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if a is None or b is None:
        return a is b
    if a.shape != b.shape or a.dtype != b.dtype or a.device != b.device:
        return False
    a, b = a.detach().contiguous(), b.detach().contiguous()
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


def assert_same(got, want, what):
    assert same(got, want), f"{what}: differs from the eager default-stream result"


def clone(out):
    if isinstance(out, (tuple, list)):
        return type(out)(clone(o) for o in out)
    return None if out is None else out.detach().clone()


def to(out, dev):
    if isinstance(out, (tuple, list)):
        return type(out)(to(o, dev) for o in out)
    return None if out is None else out.to(dev)


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


def L():
    from mocopci_b200 import _lib
    return _lib.lib


@contextlib.contextmanager
def redo_forced(scale):
    """Test hook 1: the estimated KNN admission bound times ``scale`` (process-global)."""
    from mocopci_b200 import _lib
    _lib.check(L().b200pci_debug_set(1, float(scale)), "debug_set")
    try:
        yield
    finally:
        _lib.check(L().b200pci_debug_set(1, 1.0), "debug_set")


@contextlib.contextmanager
def deterministic():
    """torch.use_deterministic_algorithms(True): the library's backwards take their `_det` path."""
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def knn_abi(k, refs, queries, ws, idx, dist, mode=5):
    """b200pci_knn on the current stream with caller-owned outputs and workspace (kept alive by the
    caller until it has synchronised: nothing the call reads can be recycled while it runs)."""
    from mocopci_b200 import _lib
    B, N, _ = refs.shape
    S = queries.shape[1]
    qs, rs = queries.stride(), refs.stride()
    _lib.check(L().b200pci_knn(B, S, N, k, mode, queries.data_ptr(), qs[0], qs[1], qs[2],
                               refs.data_ptr(), rs[0], rs[1], rs[2], idx.data_ptr(), 1,
                               dist.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "knn")


def knn_buffers(k, refs, queries):
    from mocopci_b200 import _lib
    B, N, _ = refs.shape
    S = queries.shape[1]
    dev = refs.device
    return (_lib.workspace(L().b200pci_knn_workspace_bytes(B, S, N, k), dev),
            torch.empty((B, S, k), dtype=torch.int64, device=dev),
            torch.empty((B, S, k), dtype=torch.float32, device=dev))


def chamfer_forward(x, y):
    """b200pci_chamfer_forward called as chamfer.py calls it, keeping what it writes per point:
    -> (loss, dist_x [B,N], idx_x [B,N], dist_y [B,M], idx_y [B,M])."""
    from mocopci_b200 import _lib
    B, N, _ = x.shape
    M = y.shape[1]
    f32, i32 = dict(dtype=torch.float32, device=x.device), dict(dtype=torch.int32, device=x.device)
    dist_x, idx_x = torch.empty((B, N), **f32), torch.empty((B, N), **i32)
    dist_y, idx_y = torch.empty((B, M), **f32), torch.empty((B, M), **i32)
    loss = torch.empty((1,), **f32)
    ws = _lib.workspace(L().b200pci_chamfer_workspace_bytes(B, N, M), x.device)
    xs, ys = x.stride(), y.stride()
    _lib.check(L().b200pci_chamfer_forward(
        B, N, M, x.data_ptr(), xs[0], xs[1], xs[2], y.data_ptr(), ys[0], ys[1], ys[2],
        dist_x.data_ptr(), idx_x.data_ptr(), dist_y.data_ptr(), idx_y.data_ptr(), loss.data_ptr(),
        ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "chamfer_forward")
    return loss, dist_x, idx_x, dist_y, idx_y


def bits(a):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


# ------------------------------------------------------------------------------------------
# inputs as bench.py builds them, and a second valid set of the same shapes
# ------------------------------------------------------------------------------------------
class Frames:
    """Input set 0 = bench.py's extras() inputs (frame pairs 0..7), set 1 = the next eight pairs.
    Everything derived from a set (FPS centres, ball-query / KNN indices, seeded features) is
    computed eagerly on the default stream and cached."""

    def __init__(self):
        from mocopci_b200 import synth
        self.cpu = [synth.frame_pairs(0, 8), synth.frame_pairs(8, 8)]
        self.gpu = [(a.cuda(), b.cuda()) for a, b in self.cpu]
        self._cache = {}

    def get(self, key, s):
        if (key, s) not in self._cache:
            self._cache[(key, s)] = getattr(self, "_" + key)(s)
        return self._cache[(key, s)]

    def _centres(self, s):
        from mocopci_b200 import ops as p2u, pointconv_util as pcu
        a = self.gpu[s][0]
        return pcu.index_points_gather(a, p2u.furthest_point_sample(a, 4096))

    def _ball(self, s):
        from mocopci_b200 import ops as p2u
        return p2u.ball_query(0.5, 32, self.gpu[s][0], self.get("centres", s))

    def _feats(self, s):
        return torch.randn(8, 128, NPTS, device="cuda", generator=torch.Generator("cuda").manual_seed(99 + s))

    def _kidx(self, s):
        from mocopci_b200 import pointconv_util as pcu
        return pcu.knn_point(16, *self.gpu[s])

    def _fbnc(self, s):
        return torch.randn(8, NPTS, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(64 + s))

    def _gidx(self, s):
        from mocopci_b200 import pointconv_util as pcu
        a1 = self.gpu[s][0][:1]
        return pcu.knn_point(32, a1, a1)

    def _f32(self, s):
        return torch.randn(1, 32, NPTS, device="cuda", generator=torch.Generator("cuda").manual_seed(32 + s))

    def _cos(self, s):
        return torch.randn(1, 64, 2048, device="cuda", generator=torch.Generator("cuda").manual_seed(2048 + s))


@pytest.fixture(scope="module")
def frames():
    return Frames()


def flagged_queries():
    """Queries the calling thread's last two-pass KNN call flagged for the exact redo."""
    return L().b200pci_debug_get(6)


@pytest.fixture(scope="module")
def redo_scale(frames):
    """A scale of the estimated bound at which knn_point(16) on one benchmark pair flags between 1
    and REDO_SPARSE_MAX queries: the per-query redo kernel then does real work on the side stream
    (more flags send the whole redo to the tile-wise kernel on the caller's stream)."""
    a, b = (t[:1] for t in frames.gpu[0])
    bufs = knn_buffers(16, a, b)
    counts = {}
    for scale in (0.3, 0.5, 0.65, 0.8, 0.9, 0.95, 0.98):
        with redo_forced(scale):
            knn_abi(16, a, b, *bufs)
            n = flagged_queries()
        counts[scale] = n
        if 32 <= n <= REDO_SPARSE_MAX:
            return scale
    pytest.fail(f"no scale flags 32..{REDO_SPARSE_MAX} queries: {counts}")


# ------------------------------------------------------------------------------------------
# 1. graph capture and replay of every bench.py row
# ------------------------------------------------------------------------------------------
PYRAMID = [(256, 64), (1024, 256), (4096, 1024), (16384, 4096)]  # (unknown n, known m)


def _pyr(frames, s, n, m):
    a = frames.gpu[s][0]
    return a[:, :n].contiguous(), a[:, :m].contiguous()


def _nn3(frames, s, n, m):
    from mocopci_b200 import ops as p2u
    w, i3, _ = p2u.three_nn_weights(*_pyr(frames, s, n, m))
    f = torch.randn(8, 128, m, device="cuda", generator=torch.Generator("cuda").manual_seed(1000 * s + m))
    return f, i3, w


def _rows():
    """bench.py extras() row -> (inputs(frames, set) -> tuple of tensors, call(*inputs), oracle check
    (orc, frames, set, output) or None). The call is bench.py's lambda on those inputs."""
    from mocopci_b200 import chamfer, emd_cuda, ops as p2u, pointconv_util as pcu
    ab = lambda f, s: f.gpu[s]  # noqa: E731

    def knn_b1_oracle(orc, f, s, out):
        a, b = f.cpu[s]
        oi, _ = orc.knn_form(5, 16, a[:1].numpy(), b[:1, :1024].numpy())
        np.testing.assert_array_equal(out[:, :1024].cpu().numpy(), oi)

    def fps_oracle(orc, f, s, out):
        np.testing.assert_array_equal(out[:1].cpu().numpy(), orc.fps(f.cpu[s][0][:1].numpy(), 4096)[0])

    def ball_oracle(orc, f, s, out):
        want = orc.ball_query(0.5, 32, f.cpu[s][0][:1].numpy(), f.get("centres", s)[:1].cpu().numpy())
        np.testing.assert_array_equal(out[:1].cpu().numpy(), want)

    def nn3_oracle(orc, f, s, out):
        a = f.cpu[s][0][:1]
        od2, oi = orc.three_nn(a.numpy(), a[:, :4096].contiguous().numpy())
        odist, ow = orc.three_nn_weights(od2)
        w, idx, dist = out
        np.testing.assert_array_equal(idx[:1].cpu().numpy(), oi)
        np.testing.assert_array_equal(bits(dist[:1]), bits(odist))
        np.testing.assert_array_equal(bits(w[:1]), bits(ow))

    rows = {
        "knn_k16_B8": (ab, lambda a, b: pcu.knn_point(16, a, b), None),
        "knn_k32_B8": (ab, lambda a, b: pcu.knn_point(32, a, b), None),
        "knn_k16_B1": (ab, lambda a, b: pcu.knn_point(16, a[:1], b[:1]), knn_b1_oracle),
        "knn_k32_B1_self": (ab, lambda a, b: pcu.knn_point(32, a[:1], a[:1]), None),
        "knn_k3_16384x2048_B1": (ab, lambda a, b: pcu.knn_point(3, a[:1, :2048], b[:1]), None),
        "chamfer_B8": (ab, lambda a, b: chamfer.chamfer_distance(a, b)[0], None),
        "fps_16384_to_4096": (lambda f, s: f.gpu[s][:1], lambda a: p2u.furthest_point_sample(a, 4096), fps_oracle),
        "ball_query_r0.5_ns32": (lambda f, s: (f.gpu[s][0], f.get("centres", s)),
                                 lambda a, c: p2u.ball_query(0.5, 32, a, c), ball_oracle),
        "group_points_C128": (lambda f, s: (f.get("feats", s), f.get("ball", s)),
                              lambda x, i: p2u.grouping_operation(x, i), None),
        "group_points_C3": (lambda f, s: (f.gpu[s][0].transpose(1, 2).contiguous(), f.get("ball", s)),
                            lambda x, i: p2u.grouping_operation(x, i), None),
        "query_and_group_C128": (lambda f, s: (f.gpu[s][0], f.get("centres", s), f.get("feats", s)),
                                 lambda a, c, x: p2u.query_and_group(0.5, 32, a, c, x), None),
        "index_points_group_C64_k16": (lambda f, s: (f.get("fbnc", s), f.get("kidx", s)),
                                       lambda x, i: pcu.index_points_group(x, i), None),
        "knn_point_cosine_2048_C64_k16": (lambda f, s: (f.get("cos", s),),
                                          lambda x: pcu.knn_point_cosine(16, x.permute(0, 2, 1), x.permute(0, 2, 1)),
                                          None),
        "group_concat_16384_k32_C32": (lambda f, s: (f.gpu[s][0], f.get("f32", s), f.get("gidx", s)),
                                       lambda a, x, i: pcu._group_concat(a[:1], a[:1], x.permute(0, 2, 1), i), None),
        "emd_cost_16384": (lambda f, s: (f.gpu[s][0][:1].contiguous(), f.gpu[s][1][:1].contiguous()),
                           lambda x1, x2: emd_cuda.emd_cost(x1, x2), None),
        "emd_match_16384": (lambda f, s: (f.gpu[s][0][:1].contiguous(), f.gpu[s][1][:1].contiguous()),
                            lambda x1, x2: emd_cuda.matchcost_forward(x1, x2, emd_cuda.approxmatch_forward(x1, x2)),
                            None),
    }
    for n, m in PYRAMID:
        rows[f"three_nn_weights_{m}->{n}"] = (
            lambda f, s, n=n, m=m: _pyr(f, s, n, m), lambda u, k: p2u.three_nn_weights(u, k),
            nn3_oracle if n == NPTS else None)
        rows[f"three_interpolate_{m}->{n}_C128"] = (
            lambda f, s, n=n, m=m: _nn3(f, s, n, m), lambda x, i, w: p2u.three_interpolate(x, i, w), None)
    return rows


ROW_NAMES = ["knn_k16_B8", "knn_k32_B8", "knn_k16_B1", "knn_k32_B1_self", "knn_k3_16384x2048_B1", "chamfer_B8",
             "fps_16384_to_4096", "ball_query_r0.5_ns32", "group_points_C128", "group_points_C3",
             "query_and_group_C128", "index_points_group_C64_k16"] + \
            [f"three_nn_weights_{m}->{n}" for n, m in PYRAMID] + \
            [f"three_interpolate_{m}->{n}_C128" for n, m in PYRAMID] + \
            ["knn_point_cosine_2048_C64_k16", "group_concat_16384_k32_C32", "emd_cost_16384", "emd_match_16384"]


def capture(fn):
    """graph_median's capture: two eager calls, synchronise, capture one call in torch.cuda.graph.
    -> (graph, the call's outputs as the graph writes them). A capture error propagates."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def replay(g, out):
    g.replay()
    torch.cuda.synchronize()
    return clone(out)


def check_graph(fn, ins0, ins1, what):
    """Capture ``fn`` on static copies of ``ins0``; replay; copy ``ins1`` into the static inputs and
    replay again. Each replay equals the eager call on its inputs; the two replays differ.
    -> (first replay, second replay)."""
    static = [t.clone() for t in ins0]
    g, out = capture(lambda: fn(*static))
    first = replay(g, out)
    assert_same(first, fn(*ins0), f"{what}: first replay")
    for t, new in zip(static, ins1):
        t.copy_(new)
    second = replay(g, out)
    assert_same(second, fn(*ins1), f"{what}: replay on new inputs")
    assert not same(second, first), f"{what}: the replay on new inputs returned the first replay's output"
    del g
    return first, second


@pytest.mark.parametrize("row", ROW_NAMES)
def test_graph_replay_of_bench_row(orc, frames, row):
    """Each row of bench.py's extras() captures (graph_median would otherwise time the eager call
    without saying so), its replay equals the eager call, and a replay on the next frame pairs --
    on the scratch the first replay left behind, and with the host-side decisions taken at capture
    -- equals the eager call on those."""
    inputs, fn, oracle = _rows()[row]
    _, second = check_graph(fn, inputs(frames, 0), inputs(frames, 1), row)
    if oracle is not None:
        oracle(orc, frames, 1, second)


def test_graph_redo_path_and_side_stream(orc, frames, redo_scale):
    """A 16384^2 KNN with the exact redo forced, captured: the graph holds the per-query redo on the
    library's side stream (forked and joined inside the capture) and the tile-wise redo, and its
    replays equal the eager call -- which equals the oracle and the un-forced search."""
    from mocopci_b200 import pointconv_util as pcu
    fn = lambda a, b: pcu.knn_point_with_dist(16, a[:1], b[:1])  # noqa: E731
    (a0, b0), (a1, b1) = frames.gpu
    with redo_forced(redo_scale):
        static = [a0.clone(), b0.clone()]
        g, out = capture(lambda: fn(*static))
        first, names = launches(lambda: replay(g, out))
        assert {"knn_fallback_kernel", "knn_redo_kernel"} <= base(names), names
        assert_same(first, fn(a0, b0), "first replay")
        static[0].copy_(a1)
        static[1].copy_(b1)
        second = replay(g, out)
        assert_same(second, fn(a1, b1), "replay on new inputs")
        assert not same(second, first)
    assert_same(second, fn(a1, b1), "replay vs the un-forced search")
    a, b = frames.cpu[1]
    oi, od = orc.knn_form(5, 16, a[:1].numpy(), b[:1].numpy())
    np.testing.assert_array_equal(second[0].cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(second[1]), bits(od))


def test_graph_first_library_call_of_a_thread(frames, redo_scale):
    """A new host thread whose FIRST library call is inside a capture: its thread-local side stream
    and events are created during the capture. The replays equal the eager call on the main thread,
    and the thread's redo counters are its own (b200pci_debug_get(6) is per thread)."""
    from mocopci_b200 import pointconv_util as pcu
    (a0, b0), (a1, b1) = frames.gpu
    fn = lambda a, b: pcu.knn_point(16, a[:1], b[:1])  # noqa: E731
    static = [a0.clone(), b0.clone()]
    res = {}

    def worker():
        try:
            res["flagged_before"] = flagged_queries()
            torch.cuda.set_device(0)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = fn(*static)
            res["first"] = replay(g, out)
            static[0].copy_(a1)
            static[1].copy_(b1)
            torch.cuda.synchronize()
            res["second"] = replay(g, out)
        except Exception as e:  # noqa: BLE001  (re-raised on the main thread)
            res["error"] = e

    with redo_forced(redo_scale):
        want0 = fn(a0, b0)
        bufs = knn_buffers(16, a1[:1], b1[:1])  # the counters debug_get reads live in this scratch
        knn_abi(16, a1[:1], b1[:1], *bufs)
        want1 = bufs[1]
        main_flagged = flagged_queries()
        t = threading.Thread(target=worker)
        t.start()
        t.join()
        if "error" in res:
            raise res["error"]
        assert flagged_queries() == main_flagged  # the main thread's last call, not the worker's
    assert res["flagged_before"] == -1.0  # nothing recorded for a thread that has made no call
    assert 32 <= main_flagged <= REDO_SPARSE_MAX
    assert_same(res["first"], want0, "first replay")
    assert_same(res["second"], want1, "replay on new inputs")


def _knn_dists_loss(x, y, w):
    from mocopci_b200 import chamfer
    return (chamfer.knn_points(x, y, K=16).dists * w).sum()


def _chamfer_loss(x, y, w):
    from mocopci_b200 import chamfer
    return chamfer.chamfer_distance(x, y)[0]


@pytest.mark.parametrize("loss_fn", [_knn_dists_loss, _chamfer_loss], ids=["knn_points_dists", "chamfer"])
def test_graph_forward_backward_det(frames, loss_fn):
    """Forward + backward captured under torch.use_deterministic_algorithms: the `_det` gradients
    of the replays equal the eager `_det` gradients, and the sequential C loops of
    tests/knn_grad_oracle.c / tests/grad_oracle.c."""
    from mocopci_b200 import chamfer
    from tests import grad_oracle, knn_grad_oracle
    (a0, b0), (a1, b1) = frames.gpu
    w = torch.rand(1, NPTS, 16, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    x = a0[:1].clone().requires_grad_(True)
    y = b0[:1].clone().requires_grad_(True)

    def step():
        return torch.autograd.grad(loss_fn(x, y, w), (x, y))

    def eager(a, b):
        xe, ye = a[:1].clone().requires_grad_(True), b[:1].clone().requires_grad_(True)
        return torch.autograd.grad(loss_fn(xe, ye, w), (xe, ye))

    with deterministic():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # warm-up of autograd off the default stream (torch's recipe)
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            grads = step()
        first = replay(g, grads)
        assert_same(first, eager(a0, b0), "first replay")
        with torch.no_grad():
            x.copy_(a1[:1])
            y.copy_(b1[:1])
        second = replay(g, grads)
        assert_same(second, eager(a1, b1), "replay on new inputs")
        assert not same(second, first)
    xs, ys = a1[:1].cpu().numpy(), b1[:1].cpu().numpy()
    if loss_fn is _knn_dists_loss:
        idx = chamfer.knn_points(a1[:1], b1[:1], K=16).idx
        want = knn_grad_oracle.knn_backward(xs, ys, idx.cpu().numpy(), w.cpu().numpy())
    else:
        ix = chamfer.knn_points(a1[:1], b1[:1], K=1).idx[..., 0]
        iy = chamfer.knn_points(b1[:1], a1[:1], K=1).idx[..., 0]
        want = grad_oracle.chamfer_backward(xs, ys, ix.cpu().numpy(), iy.cpu().numpy())
    for got, ref in zip(second, want):
        np.testing.assert_array_equal(bits(got), bits(ref))


# ------------------------------------------------------------------------------------------
# 2. a second stream
# ------------------------------------------------------------------------------------------
def late_on_stream(op, stale, fresh, before=None):
    """On a new stream s: hold s back, copy ``fresh`` over buffers holding ``stale`` (another valid
    input set), run ``op`` on the buffers and clone its outputs, all on s, with no synchronisation
    in between. ``before(s)`` (optional) enqueues other work first. -> the clones, after a
    device synchronisation. ``op`` runs once eagerly first: the first launch of a kernel loads
    its module (CUDA's lazy loading), which synchronises the device and would hide a launch on
    the wrong stream."""
    op(*stale)
    bufs = [t.clone() for t in stale]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    keep = before(s) if before is not None else None
    with torch.cuda.stream(s):
        torch.cuda._sleep(SLEEP)
        for b, f in zip(bufs, fresh):
            b.copy_(f)
        got = clone(op(*bufs))
    torch.cuda.synchronize()
    del keep
    return got


def test_late_inputs_two_pass_knn_with_busy_side_stream(orc, frames, redo_scale):
    """Two-pass KNN (redo forced) on a held-back stream. Before it, a second stream held back twice
    as long makes a redo-forced call of its own: the library's side stream (one per thread and
    device) runs that call's redo first, so this call's redo rows come late, and only the join
    makes the consumer on s wait for them. Outputs and scratch are owned here and stay alive until
    the device is synchronised."""
    (a0, b0), (a1, b1) = frames.gpu
    fresh = [a1[:1].contiguous(), b1[:1].contiguous()]
    stale = [a0[:1].contiguous(), b0[:1].contiguous()]
    blocker_in = [a0[1:2].contiguous(), b0[1:2].contiguous()]
    bufs = knn_buffers(16, *stale)

    def blocker(s):
        out = knn_buffers(16, *blocker_in)
        s2 = torch.cuda.Stream()
        with torch.cuda.stream(s2):
            torch.cuda._sleep(2 * SLEEP)
            knn_abi(16, *blocker_in, *out)
        return out

    def op(a, b):
        knn_abi(16, a, b, *bufs)
        return bufs[1], bufs[2]

    with redo_forced(redo_scale):
        got = late_on_stream(op, stale, fresh, before=blocker)
        assert 32 <= flagged_queries() <= REDO_SPARSE_MAX
        want = knn_buffers(16, *fresh)
        knn_abi(16, *fresh, *want)
    assert_same(got, want[1:], "two-pass KNN on a late stream")
    a, b = frames.cpu[1]
    oi, od = orc.knn_form(5, 16, a[:1].numpy(), b[:1].numpy())
    np.testing.assert_array_equal(got[0].cpu().numpy(), oi)
    np.testing.assert_array_equal(bits(got[1]), bits(od))


def test_late_inputs_chamfer_forward_and_det_backward(orc, frames, redo_scale):
    """Chamfer at 16384^2 (two-pass K = 1 searches, redo forced) and its `_det` backward on a
    held-back stream: per-point minima and indices equal the oracle's, loss and gradients the eager
    default-stream call's."""
    from mocopci_b200 import chamfer
    (a0, b0), (a1, b1) = frames.gpu
    fresh = [a1[:1].contiguous(), b1[:1].contiguous()]
    stale = [a0[:1].contiguous(), b0[:1].contiguous()]

    def op(x, y):
        per_point = chamfer_forward(x, y)[1:]
        xl, yl = x.detach().requires_grad_(True), y.detach().requires_grad_(True)
        loss = chamfer.chamfer_distance(xl, yl)[0]
        return (loss,) + tuple(torch.autograd.grad(loss, (xl, yl))) + per_point

    with redo_forced(redo_scale), deterministic():
        got = late_on_stream(op, stale, fresh)
        want = op(*fresh)
    assert_same(got, want, "Chamfer on a late stream")
    _, odx, ody, oix, oiy = orc.chamfer(frames.cpu[1][0][:1].numpy(), frames.cpu[1][1][:1].numpy())
    dx, ix, dy, iy = got[3:]
    np.testing.assert_array_equal(bits(dx), bits(odx))
    np.testing.assert_array_equal(bits(dy), bits(ody))
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)


def test_late_inputs_sampling_grouping_and_det_scatter(frames):
    """FPS (cluster kernel), ball query, query_and_group and the `_det` backward of
    grouping_operation on a held-back stream, equal to the eager default-stream calls."""
    from mocopci_b200 import ops as p2u, pointconv_util as pcu

    def op(a, feats):
        fidx = p2u.furthest_point_sample(a, 1024)
        centres = pcu.index_points_gather(a, fidx)
        idx = p2u.ball_query(0.5, 32, a, centres)
        qg = p2u.query_and_group(0.5, 32, a, centres, feats)
        fl = feats.detach().requires_grad_(True)
        grad = torch.autograd.grad((p2u.grouping_operation(fl, idx) * qg[:, 3:]).sum(), fl)[0]
        return fidx, idx, qg, grad

    f0 = frames.get("feats", 0)[:, :16].contiguous()
    f1 = frames.get("feats", 1)[:, :16].contiguous()
    stale, fresh = [frames.gpu[0][0], f0], [frames.gpu[1][0], f1]
    with deterministic():
        got = late_on_stream(op, stale, fresh)
        want = op(*fresh)
    for name, g, w in zip(("fps", "ball_query", "query_and_group", "group grad (_det)"), got, want):
        assert_same(g, w, f"{name} on a late stream")


def test_late_inputs_cosine_knn(orc, frames):
    """The cosine KNN (pack kernel with its in-stream tickets + tensor-core top-k) on a held-back
    stream: equal to the eager call; distances within the tensor cores' tolerance of the oracle."""
    from mocopci_b200 import pointconv_util as pcu

    def op(x):
        v = x.permute(0, 2, 1)
        return pcu.knn_point_cosine_with_dist(16, v, v)

    got = late_on_stream(op, [frames.get("cos", 0)], [frames.get("cos", 1)])
    assert_same(got, op(frames.get("cos", 1)), "cosine KNN on a late stream")
    f = frames.get("cos", 1).permute(0, 2, 1).contiguous().cpu().numpy()
    _, od = orc.knn_cosine(16, f, f)
    assert float(np.abs(got[1].cpu().numpy() - od).max()) <= 4e-6


def test_late_inputs_emd(frames):
    """emd_cost and approxmatch + matchcost (4096-point pair) on a held-back stream."""
    from mocopci_b200 import emd_cuda

    def op(x1, x2):
        match = emd_cuda.approxmatch_forward(x1, x2)
        return emd_cuda.emd_cost(x1, x2), match, emd_cuda.matchcost_forward(x1, x2, match)

    pair = lambda s: [frames.gpu[s][0][:1, :4096].contiguous(), frames.gpu[s][1][:1, :4096].contiguous()]  # noqa: E731
    got = late_on_stream(op, pair(0), pair(1))
    assert_same(got, op(*pair(1)), "EMD on a late stream")


def test_eval_leg_pattern(frames, redo_scale):
    """bench.py's eval leg: per round, the two-pass KNN rows on the main stream, then Chamfer + EMD
    of the round's prediction on a second stream (wait_stream / record_stream as bench.py does),
    while the next round's KNN is already launched on the main stream. Both streams fork the
    library's one side stream of this thread. Every output equals its serial eager result."""
    from mocopci_b200 import chamfer, ops, pointconv_util as pcu
    rounds = [(frames.gpu[s][0][p:p + 1].contiguous(), frames.gpu[s][1][p:p + 1].contiguous())
              for s in (0, 1) for p in (0, 5)]

    def forward(a, b):
        pred = (a + (b - a).mean(1, keepdim=True) * 0.5).contiguous()
        return pcu.knn_point_with_dist(16, a, b), pcu.knn_point(32, a, a), pred

    def metrics(pred, b):
        return chamfer.chamfer_distance(pred, b)[0], ops.earth_mover_distance(pred, b, transpose=False)

    with redo_forced(redo_scale), torch.no_grad():
        want = []
        for a, b in rounds:
            fw = forward(a, b)
            want.append((fw[0], fw[1], metrics(fw[2], b)))
        torch.cuda.synchronize()
        main = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        got = []
        for a, b in rounds:
            (idx16, d16), idx32, pred = forward(a, b)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                pred.record_stream(side)
                m = metrics(pred, b)
                b.record_stream(side)
            got.append(((idx16, d16), idx32, m))
        main.wait_stream(side)
        torch.cuda.synchronize()
    for r, (g, w) in enumerate(zip(got, want)):
        assert_same(g[0], w[0], f"round {r}: knn k=16")
        assert_same(g[1], w[1], f"round {r}: knn k=32 self")
        assert_same(g[2], w[2], f"round {r}: Chamfer + EMD on the second stream")


# ------------------------------------------------------------------------------------------
# 3. concurrent host threads
# ------------------------------------------------------------------------------------------
def _thread_work(a, b, feat):
    """One round of a worker: two-pass KNN, Chamfer, cosine KNN, a `_det` backward."""
    from mocopci_b200 import chamfer, pointconv_util as pcu
    knn = pcu.knn_point_with_dist(16, a, b)
    cd = chamfer.chamfer_distance(a, b)[0]
    v = feat.permute(0, 2, 1)
    cos = pcu.knn_point_cosine_with_dist(16, v, v)
    x = a.detach().requires_grad_(True)
    grad = torch.autograd.grad(chamfer.knn_points(x, b, K=16).dists.sum(), x)[0]
    return knn, cd, cos, grad


def run_threads(worker, n):
    errors, threads = [], []

    def wrap(t):
        try:
            worker(t)
        except Exception as e:  # noqa: BLE001  (re-raised below)
            errors.append(e)

    for t in range(n):
        threads.append(threading.Thread(target=wrap, args=(t,)))
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    if errors:
        raise errors[0]


def test_concurrent_host_threads(frames, redo_scale):
    """Three Python threads, each on its own stream, run three rounds of two-pass KNN (redo forced
    before they start), Chamfer, cosine KNN and a `_det` backward on their own inputs at once. Each
    result equals the serial one: the library's state (error string, side stream and events) is
    per thread."""
    nthreads, nrounds = 3, 3
    pair = lambda t, r: (3 * t + r) % 8  # noqa: E731
    inputs = [[(frames.gpu[t % 2][0][pair(t, r):pair(t, r) + 1].contiguous(),
                frames.gpu[t % 2][1][pair(t, r):pair(t, r) + 1].contiguous(),
                frames.get("cos", t % 2).roll(r, 2).contiguous()) for r in range(nrounds)]
              for t in range(nthreads)]
    got = [[] for _ in range(nthreads)]

    def worker(t):
        torch.cuda.set_device(0)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            for a, b, f in inputs[t]:
                got[t].append(clone(_thread_work(a, b, f)))
        s.synchronize()

    with redo_forced(redo_scale), deterministic():
        run_threads(worker, nthreads)
        want = [[_thread_work(*inp) for inp in per] for per in inputs]
    for t in range(nthreads):
        for r in range(nrounds):
            for name, g, w in zip(("knn", "chamfer", "cosine", "knn grad (_det)"), got[t][r], want[t][r]):
                assert_same(g, w, f"thread {t} round {r}: {name}")


def test_host_api_from_two_threads(frames):
    """knn_point_host (b200pci_knn_host: a per-thread, per-device copy pipeline and device buffer)
    from two threads at once equals the device path; b200pci_host_release() in one thread, while
    the other is inside a call, leaves the other thread's calls intact."""
    from mocopci_b200 import _lib, host_api, pointconv_util as pcu
    data = [(frames.cpu[t][0][:2].contiguous(), frames.cpu[t][1][:2].contiguous()) for t in (0, 1)]
    want = [pcu.knn_point(16, a.cuda(), b.cuda()).cpu() for a, b in data]
    barrier = threading.Barrier(2)
    got = [[], []]

    def worker(t):
        torch.cuda.set_device(0)
        a, b = data[t]
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for r in range(4):
                    barrier.wait()
                    if t == 0 and r == 2:  # while thread 1 makes its third call
                        _lib.check(_lib.lib.b200pci_host_release(), "host_release")
                    got[t].append(host_api.knn_point_host(16, a, b).clone())
        except Exception:
            barrier.abort()  # release the other thread
            raise

    run_threads(worker, 2)
    for t in (0, 1):
        assert len(got[t]) == 4
        for r, g in enumerate(got[t]):
            assert torch.equal(g, want[t]), f"thread {t} call {r}"


# ------------------------------------------------------------------------------------------
# 4. a second device
# ------------------------------------------------------------------------------------------
two_gpus = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs")


def _entry_points(a, b, feats, cosf):
    """Each Python entry point once, on tensors of one device (whatever device is current)."""
    from mocopci_b200 import chamfer, emd_cuda, ops as p2u, pointconv_util as pcu
    out = {"knn": pcu.knn_point_with_dist(16, a, b), "knn_k3": pcu.knn_point(3, a[:, :2048], b)}
    v = cosf.permute(0, 2, 1)
    out["cosine"] = pcu.knn_point_cosine_with_dist(16, v, v)
    fidx = p2u.furthest_point_sample(a, 1024)
    centres = pcu.index_points_gather(a, fidx)
    idx = p2u.ball_query(0.5, 32, a, centres)
    out.update(fps=fidx, ball=idx, group=p2u.grouping_operation(feats, idx),
               qag=p2u.query_and_group(0.5, 32, a, centres, feats))
    w, i3, d3 = p2u.three_nn_weights(a, a[:, :4096].contiguous())
    out.update(nn3=(w, i3, d3), interp=p2u.three_interpolate(feats[:, :, :4096].contiguous(), i3, w))
    kidx = out["knn"][0]
    out["rows"] = pcu.index_points_group(feats.transpose(1, 2), kidx)
    out["concat"] = pcu._group_concat(a, b, feats.transpose(1, 2), kidx)
    out["emd"] = emd_cuda.emd_cost(a[:, :2048].contiguous(), b[:, :2048].contiguous())
    x, y = a.detach().requires_grad_(True), b.detach().requires_grad_(True)
    loss = chamfer.chamfer_distance(x, y)[0]
    out["chamfer"] = (loss,) + tuple(torch.autograd.grad(loss, (x, y)))
    x = a.detach().requires_grad_(True)
    out["knn_grad"] = torch.autograd.grad(chamfer.knn_points(x, b, K=16).dists.sum(), x)[0]
    f = feats.detach().requires_grad_(True)
    out["group_grad"] = torch.autograd.grad(p2u.grouping_operation(f, idx).sum(), f)[0]
    return out


@two_gpus
class TestSecondDevice:
    def test_entry_points_on_cuda1_with_cuda0_current(self, frames, redo_scale):
        """With cuda:0 current, every entry point on cuda:1 tensors (the device guard, the per-device
        side stream and workspace) gives the cuda:0 result bit for bit."""
        a, b = frames.cpu[0][0][:1], frames.cpu[0][1][:1]
        feats, cosf = frames.get("feats", 0)[:1, :16].cpu(), frames.get("cos", 0).cpu()
        with redo_forced(redo_scale), deterministic(), torch.cuda.device(0):
            want = {k: to(v, "cpu") for k, v in _entry_points(*(t.to("cuda:0") for t in (a, b, feats, cosf))).items()}
            assert torch.cuda.current_device() == 0
            got = _entry_points(*(t.to("cuda:1") for t in (a, b, feats, cosf)))
            assert torch.cuda.current_device() == 0
            torch.cuda.synchronize(1)
        for name in want:
            assert all(t is None or t.device == torch.device("cuda", 1)
                       for t in (got[name] if isinstance(got[name], tuple) else (got[name],))), name
            assert same(to(got[name], "cpu"), want[name]), f"{name}: cuda:1 differs from cuda:0"

    def test_alternating_devices_in_one_thread(self, frames, redo_scale):
        """Two-pass KNN (redo forced) on cuda:1, then cuda:0, then cuda:1 from one thread, and the
        host-buffer path on each device: the per-device side streams and host contexts."""
        from mocopci_b200 import host_api, pointconv_util as pcu
        a, b = frames.cpu[1][0][:1], frames.cpu[1][1][:1]
        with redo_forced(redo_scale):
            want = to(pcu.knn_point_with_dist(16, a.cuda(0), b.cuda(0)), "cpu")
            for dev in (1, 0, 1):
                got = pcu.knn_point_with_dist(16, a.cuda(dev), b.cuda(dev))
                assert same(to(got, "cpu"), want), f"cuda:{dev}"
            for dev in (1, 0, 1):
                assert torch.equal(host_api.knn_point_host(16, a, b, device=f"cuda:{dev}"), want[0]), f"host, cuda:{dev}"

    def test_graph_on_cuda1(self, frames, redo_scale):
        """A capture on cuda:1 of the redo-forced two-pass KNN: replays equal the eager call."""
        from mocopci_b200 import pointconv_util as pcu
        fn = lambda a, b: pcu.knn_point_with_dist(16, a, b)  # noqa: E731
        ins = [[t[:1].to("cuda:1") for t in frames.cpu[s]] for s in (0, 1)]
        with redo_forced(redo_scale), torch.cuda.device(1):
            check_graph(fn, ins[0], ins[1], "cuda:1 graph")
