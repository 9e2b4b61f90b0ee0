"""EMD's kernels against float64 restatements of the same algorithm (tests/emd_reference.py, itself
checked against the C oracle by test_emd_reference_cpu.py), at the shapes where they can go wrong:
several 2048-point tiles per sweep, partial CTAs, the 16-value prefetch tail of sweep 3, multipliers
that truncate (300 x 1000 gives 3), single-point clouds, batch offsets, the lanes-per-row variants
of the forward-only emd_cost, empty clouds, and the benchmark's 16384 x 16384 pair.

Tolerances, each derived where it is used:
* match: 3e-3 absolute, and 1e-2 relative on entries above 0.1, against FP64 (check_match says why
  smaller entries get no relative bound). That alone can miss an error of size 1/n, so it always
  goes with the cost and mass checks, which are tight.
* cost: 1e-5 relative against FP64, the benchmark's 16384 x 16384 pair included (see
  test_emd_benchmark_pair_vs_fp64).
* grad1: bit for bit with the oracle's sequential loop on the same match.
* grad2: the rounding bound of its summation order (see grad_bound).
Run with -s to see the observed worst case next to each bound (lines starting "EMD").
"""
import math
import types

import numpy as np
import pytest
import torch

from tests import emd_reference as R
from tests.test_emd_reference_cpu import MATCH_ATOL, MATCH_RTOL, MATCH_RTOL_ABOVE, check_mass, check_match

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")]

U = 2.0 ** -24           # unit roundoff of float32
EMD_LANES_KEY = 19       # b200pci_debug_set key: lanes per row of emd_cost's sweeps (default 16)


def report(what, observed, bound):
    print(f"EMD {what}: observed {observed:.3g}, bound {bound:.3g}")


def bits(a):
    return np.ascontiguousarray(a.detach().cpu().numpy(), dtype=np.float32).view(np.int32)


def assert_bits(got, want, msg=""):
    g, w = bits(got), bits(torch.as_tensor(want))
    assert g.shape == w.shape, (msg, g.shape, w.shape)
    bad = int((g != w).sum())
    assert bad == 0, f"{msg}: {bad} of {g.size} entries differ"


def rel_gap(got, want):
    got, want = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    return float(((got - want).abs() / want.abs()).max())


@pytest.fixture(scope="module")
def emd():
    from mocopci_b200 import emd_cuda
    return emd_cuda


@pytest.fixture(scope="module")
def lanes():
    """Sets emd_cost's lanes per row for a block; always back to the default 16 afterwards."""
    from mocopci_b200 import _lib

    class Lanes:
        def __init__(self, rs):
            self.rs = rs

        def __enter__(self):
            assert _lib.lib.b200pci_debug_set(EMD_LANES_KEY, float(self.rs)) == 0

        def __exit__(self, *exc):
            _lib.lib.b200pci_debug_set(EMD_LANES_KEY, 16.0)
            return False
    return Lanes


@pytest.fixture(scope="module", params=["own_api", "reference_wrappers"])
def api(request):
    """earth_mover_distance as a user reaches it: mocopci_b200.ops, or the reference's
    models/EMD/emd.py (imported from a checkout when there is one, else restated in
    tests/refwrappers.py) on top of mocopci_b200.install()."""
    import mocopci_b200
    from mocopci_b200 import ops
    if request.param == "own_api":
        return types.SimpleNamespace(name=request.param, earth_mover_distance=ops.earth_mover_distance)
    import importlib
    from baseline import fetch_ref
    root = fetch_ref.root()
    mocopci_b200.install(reference_root=root)
    if root is not None:
        mod = importlib.import_module("models.EMD.emd")
    else:
        from tests import refwrappers as mod
    return types.SimpleNamespace(name=request.param, earth_mover_distance=mod.earth_mover_distance)


def make_case(case):
    """-> (xyz1, xyz2) float32 (B, n, 3) / (B, m, 3) on the GPU."""
    from mocopci_b200 import synth
    if case == "lidar":
        a, b = synth.frame_pair(0, 4096)
        return a[None].cuda(), b[None].cuda()
    B, n, m, scale, offset = case
    x1 = synth.uniform_cloud(n, B, n) * scale + offset
    x2 = synth.uniform_cloud(m + 3, B, m) * scale + offset
    return x1.cuda(), x2.cuda()


SHAPES = [(2, 256, 256), (1, 300, 1000), (1, 1000, 300), (3, 65, 17), (1, 33, 1), (1, 1, 33),
          (1, 2100, 4100), (1, 4100, 2100)]
CASES = ([(B, n, m, s, 0.0) for s in (0.5, 5.0) for (B, n, m) in SHAPES]
         + [(1, 640, 640, 0.05, 1000.0), "lidar"])
ORACLE_MAX = 2100 * 2100   # the C oracle's approxmatch runs where n * m is at most this


def case_id(c):
    return c if isinstance(c, str) else "B{}-{}x{}-s{}{}".format(*c[:4], "-off1000" if c[4] else "")


def grad_bound(chain, abs_sum, g):
    """A gradient coordinate is g * (sum of terms 2 match (a - b)). Each term: a rounded
    subtraction (2 match is exact); the terms are added by `chain` rounded operations in the worst
    lane (the first a rounded product); one more rounding multiplies by g. First order:
    |error| <= (chain + 2) u |g| sum |terms|."""
    return (chain + 2) * U * abs_sum * g.abs().double().reshape(-1, 1, 1)


def abs_terms(a, b, match_t):
    """sum_j |2 match_t[i, j] (a[i] - b[j])| per coordinate: (B, len(a), 3), float64."""
    a, b, mt = a.double(), b.double(), match_t.double().abs()
    return torch.stack([2 * (mt * (a[..., c, None] - b[..., None, :, c]).abs()).sum(-1) for c in range(3)], -1)


def check_grads(g1, g2, gc, x1, x2, match, what):
    """Against matchcost_grad64: grad1 is a sequential chain over m, grad2 a 32-lane strided sum over
    n plus a 5-step shuffle tree. Returns the largest observed fraction of each bound."""
    n, m = x1.shape[1], x2.shape[1]
    r1, r2 = R.matchcost_grad64(gc, x1, x2, match)
    b1 = grad_bound(m, abs_terms(x1, x2, match.transpose(1, 2)), gc) + 1e-35
    b2 = grad_bound(math.ceil(n / 32) + 5, abs_terms(x2, x1, match), gc) + 1e-35
    e1, e2 = (g1.double() - r1).abs(), (g2.double() - r2).abs()
    assert (e1 <= b1).all(), f"{what} grad1: {int((e1 > b1).sum())} coordinates outside the bound"
    assert (e2 <= b2).all(), f"{what} grad2: {int((e2 > b2).sum())} coordinates outside the bound"
    return float((e1 / b1).max()) if e1.numel() else 0.0, float((e2 / b2).max()) if e2.numel() else 0.0


# ------------------------------------------------------------------------------------------
# approxmatch, matchcost, matchcost_backward and emd_cost at each shape
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_emd_kernels_vs_fp64(emd, orc, lanes, case):
    x1, x2 = make_case(case)
    B, n, m = x1.shape[0], x1.shape[1], x2.shape[1]
    tag = case_id(case)

    # approxmatch: entries against FP64, then the tight mass invariants
    match = emd.approxmatch_forward(x1, x2)
    worst_abs, worst_rel = check_match(match, R.approxmatch64(x1, x2))
    report(f"{tag} match vs FP64, absolute", worst_abs, MATCH_ATOL)
    report(f"{tag} match vs FP64, relative above {MATCH_RTOL_ABOVE}", worst_rel, MATCH_RTOL)
    mass = check_mass(match, n, m, 1e-5, 1e-4, 1e-5)
    report(f"{tag} total mass", mass["total"], 1e-5)
    report(f"{tag} saturated side", mass["saturated"], 1e-4)
    if n * m <= ORACLE_MAX:
        om = torch.from_numpy(orc.emd_approxmatch(x1.cpu().numpy(), x2.cpu().numpy()))
        report(f"{tag} match vs oracle, absolute / relative", max(check_match(match, om)), MATCH_ATOL)

    # matchcost on the GPU's own match against the closed form; the algorithm's cost against FP64
    mc = emd.matchcost_forward(x1, x2, match)
    c_closed = R.matchcost64(x1, x2, match)
    c64 = R.cost64(x1, x2)
    report(f"{tag} matchcost vs FP64 on its match", rel_gap(mc, c_closed), 1e-5)
    report(f"{tag} matchcost(approxmatch) vs cost64", rel_gap(mc, c64), 1e-5)
    assert rel_gap(mc, c_closed) <= 1e-5 and rel_gap(mc, c64) <= 1e-5

    # gradients on the GPU's match: grad1 bit for bit with the oracle, grad2 within its bound
    gc = (torch.rand(B, generator=torch.Generator().manual_seed(n + 7 * m)) * 2 - 0.7).cuda()
    g1, g2 = emd.matchcost_backward(gc, x1, x2, match)
    o1, _ = orc.emd_matchcost_grad(gc.cpu().numpy(), x1.cpu().numpy(), x2.cpu().numpy(), match.cpu().numpy())
    assert_bits(g1, o1, f"{tag} grad1 vs oracle")
    f1, f2 = check_grads(g1, g2, gc, x1, x2, match, tag)
    report(f"{tag} grad1 vs FP64, fraction of its bound", f1, 1.0)
    report(f"{tag} grad2 vs FP64, fraction of its bound", f2, 1.0)

    # emd_cost in each lanes-per-row variant
    for rs in (4, 8, 16, 32):
        with lanes(rs):
            ec = emd.emd_cost(x1, x2)
        report(f"{tag} emd_cost RS={rs} vs cost64", rel_gap(ec, c64), 1e-5)
        assert rel_gap(ec, c64) <= 1e-5, rs
        assert rel_gap(ec, mc) <= 1e-5, rs


# ------------------------------------------------------------------------------------------
# batch independence and determinism
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [(3, 2100, 300, 0.5, 0.0), (3, 65, 17, 5.0, 0.0), (3, 700, 2100, 0.5, 0.0)],
                         ids=case_id)
def test_emd_batch_independence_and_determinism(emd, case):
    """A pair's results do not depend on the other pairs of the batch or on the run: no kernel of
    EMD uses atomics, so the B = 3 call equals three B = 1 calls, and a second run the first, bit
    for bit."""
    x1, x2 = make_case(case)
    gc = torch.tensor([0.5, -2.0, 1 / 3], device="cuda")

    def run(a, b, g):
        match = emd.approxmatch_forward(a, b)
        return [match, emd.matchcost_forward(a, b, match), emd.emd_cost(a, b),
                *emd.matchcost_backward(g, a, b, match)]
    names = ["match", "matchcost", "emd_cost", "grad1", "grad2"]
    full = run(x1, x2, gc)
    for got, want, name in zip(run(x1, x2, gc), full, names):
        assert_bits(got, want, f"second run, {name}")
    for b in range(3):
        one = run(x1[b:b + 1].contiguous(), x2[b:b + 1].contiguous(), gc[b:b + 1].contiguous())
        for got, want, name in zip(one, full, names):
            assert_bits(got[0], want[b], f"pair {b} alone, {name}")


# ------------------------------------------------------------------------------------------
# autograd through both APIs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [(3, 300, 1000, 0.5, 0.0), (2, 2100, 700, 5.0, 0.0)], ids=case_id)
def test_emd_autograd_vs_fp64(emd, api, case):
    """earth_mover_distance on (B, 3, n) inputs (transpose=True) and (B, n, 3) inputs; the loss is a
    non-uniform weighted sum of the per-pair costs, as in models/EMD/test_emd_loss.py. Gradients
    against matchcost_grad64 on approxmatch_forward's match, within each kernel's rounding bound.
    With one input requiring grad the other gets None and the value stays the same."""
    x1, x2 = make_case(case)
    B = x1.shape[0]
    w = torch.tensor([0.5, 2.0, 1 / 3][:B], device="cuda")
    match = emd.approxmatch_forward(x1, x2)
    want = emd.matchcost_forward(x1, x2, match)

    for transpose in (True, False):
        if transpose:
            l1 = x1.transpose(1, 2).contiguous().requires_grad_(True)
            l2 = x2.transpose(1, 2).contiguous().requires_grad_(True)
        else:
            l1, l2 = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
        cost = api.earth_mover_distance(l1, l2, transpose=transpose)
        assert_bits(cost, want, f"{api.name} transpose={transpose} cost")
        (cost * w).sum().backward()
        g1, g2 = (l1.grad.transpose(1, 2), l2.grad.transpose(1, 2)) if transpose else (l1.grad, l2.grad)
        f1, f2 = check_grads(g1, g2, w, x1, x2, match, f"{api.name} transpose={transpose}")
        report(f"{api.name} {case_id(case)} transpose={transpose} autograd grad1 / grad2 bound", max(f1, f2), 1.0)

        for only in (0, 1):
            a = l1.detach().clone().requires_grad_(only == 0)
            b = l2.detach().clone().requires_grad_(only == 1)
            c = api.earth_mover_distance(a, b, transpose=transpose)
            assert_bits(c, want, f"{api.name} only input {only} requires grad")
            (c * w).sum().backward()
            assert (a.grad is None) == (only == 1) and (b.grad is None) == (only == 0)
            got = a.grad if only == 0 else b.grad
            assert_bits(got, (l1.grad, l2.grad)[only], f"{api.name} gradient with one input requiring grad")


# ------------------------------------------------------------------------------------------
# the benchmark pair
# ------------------------------------------------------------------------------------------
def test_emd_benchmark_pair_vs_fp64(emd):
    """bench.py's eval metric, emd_cost at 16384 x 16384 on benchmark pair 0, and
    matchcost(approxmatch), against cost64 evaluated in float64 on the GPU: 1e-5 relative, as at
    the smaller shapes. The C oracle's cost of this pair is 2.9e-5 from cost64, but 2.8e-5 of that
    is its FP32 reduction of the cost (512 partial sums of 32 x 16384 terms); the FP64 closed form
    on the oracle's match is 7.9e-7 from cost64. The kernels reduce their per-row FP32 sums in
    FP64."""
    from mocopci_b200 import synth
    a, b = synth.frame_pairs(0, 1)
    x1, x2 = a.cuda(), b.cuda()
    cost = emd.emd_cost(x1, x2)
    match = emd.approxmatch_forward(x1, x2)
    mc = emd.matchcost_forward(x1, x2, match)
    c_closed = R.matchcost64(x1, x2, match)
    del match
    c64 = R.cost64(x1, x2)
    report("16384^2 emd_cost vs cost64", rel_gap(cost, c64), 1e-5)
    report("16384^2 matchcost(approxmatch) vs cost64", rel_gap(mc, c64), 1e-5)
    report("16384^2 emd_cost vs matchcost", rel_gap(cost, mc), 1e-5)
    report("16384^2 matchcost vs FP64 on its match", rel_gap(mc, c_closed), 1e-5)
    assert rel_gap(cost, c64) <= 1e-5 and rel_gap(mc, c64) <= 1e-5
    assert rel_gap(cost, mc) <= 1e-5 and rel_gap(mc, c_closed) <= 1e-5


# ------------------------------------------------------------------------------------------
# empty and degenerate inputs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n,m", [(2, 0, 5), (2, 5, 0), (0, 5, 7), (2, 0, 0)])
def test_emd_empty(emd, B, n, m):
    x1, x2 = torch.rand(B, n, 3, device="cuda"), torch.rand(B, m, 3, device="cuda")
    match = emd.approxmatch_forward(x1, x2)
    assert tuple(match.shape) == (B, m, n)
    for cost in (emd.matchcost_forward(x1, x2, match), emd.emd_cost(x1, x2)):
        assert tuple(cost.shape) == (B,) and bool((cost == 0).all())
    g1, g2 = emd.matchcost_backward(torch.ones(B, device="cuda"), x1, x2, match)
    assert tuple(g1.shape) == (B, n, 3) and tuple(g2.shape) == (B, m, 3)
    assert bool((g1 == 0).all()) and bool((g2 == 0).all())
    from mocopci_b200 import ops
    l1, l2 = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    c = ops.earth_mover_distance(l1, l2, transpose=False)
    c.sum().backward()
    assert bool((c == 0).all()) and bool((l1.grad == 0).all()) and bool((l2.grad == 0).all())


@pytest.mark.parametrize("case", [(1, 1000, 1000, 0.5, 0.0), (2, 2100, 2100, 5.0, 0.0), "lidar"], ids=case_id)
def test_emd_self_and_permutations(emd, case):
    """A cloud against itself, or a permutation of itself, costs nothing (below 1e-6 per point); and
    permuting either cloud's points leaves the cost of a pair unchanged to 1e-5 relative."""
    x1, x2 = make_case(case)
    n = x1.shape[1]
    g = torch.Generator().manual_seed(n)
    p1, p2 = torch.randperm(n, generator=g).cuda(), torch.randperm(x2.shape[1], generator=g).cuda()

    def both(a, b):
        a, b = a.contiguous(), b.contiguous()
        return emd.emd_cost(a, b), emd.matchcost_forward(a, b, emd.approxmatch_forward(a, b))
    for c in (*both(x1, x1), *both(x1, x1[:, p1])):
        assert float(c.max()) / n < 1e-6, float(c.max())
    base = both(x1, x2)
    for perm in (both(x1[:, p1], x2), both(x1, x2[:, p2])):
        for got, want in zip(perm, base):
            report(f"{case_id(case)} permuted cloud", rel_gap(got, want), 1e-5)
            assert rel_gap(got, want) <= 1e-5


# ------------------------------------------------------------------------------------------
# argument checks (all rejected on the host, before any launch)
# ------------------------------------------------------------------------------------------
def test_emd_match_and_grad_cost_are_validated(emd):
    x1, x2 = torch.rand(2, 30, 3, device="cuda"), torch.rand(2, 20, 3, device="cuda")
    match = emd.approxmatch_forward(x1, x2)
    gc = torch.ones(2, device="cuda")
    bad_matches = [torch.zeros(2, 30, 20, device="cuda"),                  # (B, n, m)
                   torch.zeros(2, 20, 29, device="cuda"),
                   torch.zeros(1, 20, 30, device="cuda"),
                   match.double(),
                   torch.zeros(2, 30, 20, device="cuda").transpose(1, 2),  # right shape, not contiguous
                   match.cpu()]
    for bad in bad_matches:
        with pytest.raises(RuntimeError, match="match must be"):
            emd.matchcost_backward(gc, x1, x2, bad)
        with pytest.raises(RuntimeError, match="match must be"):
            emd.matchcost_forward(x1, x2, bad)
    for bad in (torch.ones(1, device="cuda"), torch.ones(3, device="cuda"), torch.ones(2)):
        with pytest.raises(RuntimeError, match="grad_cost"):
            emd.matchcost_backward(bad, x1, x2, match)
    with pytest.raises(RuntimeError, match="CUDA"):
        emd.matchcost_backward(gc, x1, x2.cpu(), match)
    g1, g2 =emd.matchcost_backward(gc.view(2, 1), x1, x2, match)   # any shape with B elements
    assert_bits(g1, emd.matchcost_backward(gc, x1, x2, match)[0], "grad_cost of shape (B, 1)")
