"""Every compiled segment-reduce kernel, run once and compared bit for bit with an exact fp64 reference.

One case per instantiation (two for the sum kernels: sum and mean), built by tests/helpers/kernel_matrix.py: inputs on
a dyadic grid make every partial sum exact, so the result cannot depend on the summation order and must equal the
fp64 reference rounded once.  Each call runs under torch.profiler, and the test asserts that the instantiation it was
written for is among the kernels that ran, with its fixup kernel.  The output starts as NaN, so a row the kernels never
write shows up.
"""
import pytest
import torch

from tests.helpers import kernel_matrix as km

pytestmark = pytest.mark.gpu

try:
    _INV = km.inventory()
    _CASES = [c for t in sorted(_INV[0]) for c in km.cases_for(t)]
    _INV_ERROR = None
except Exception as e:     # reported by the tests below, not as a collection error of the whole suite
    _INV, _CASES, _INV_ERROR = (frozenset(), frozenset()), [], "%s: %s" % (type(e).__name__, e)

_RESULTS = {}   # case id -> (launched reduce tuples, launched fixup tuples, mismatch report)


def _run(case):
    if case.id not in _RESULTS:
        inp = km.make_inputs(case)
        ref = km.reference(case, inp)
        got, names = km.run_case(case, inp)
        parsed = [km.parse_kernel(n) for n in names]
        red = {p[1] for p in parsed if p and p[0] == "reduce"}
        fix = {p[1] for p in parsed if p and p[0] == "fixup"}
        _RESULTS[case.id] = (red, fix, km.mismatch_report(got, ref, inp))
    return _RESULTS[case.id]


def test_inventory_is_readable():
    assert _INV_ERROR is None, _INV_ERROR
    assert _CASES


@pytest.mark.parametrize("case", _CASES, ids=[c.id for c in _CASES])
def test_kernel_bit_exact(case):
    red, fix, report = _run(case)
    assert case.target in red, "ran %s instead of %s" % (sorted(red), case.target)
    assert (case.target[0], case.target[4]) in fix, "fixup kernel did not run: %s" % sorted(fix)
    assert not report, report


def test_every_compiled_kernel_launched_and_bit_exact():
    """The union of the instantiations the cases launched is the inventory, less the ones no call can reach."""
    assert _INV_ERROR is None, _INV_ERROR
    launched, inexact = set(), []
    for c in _CASES:
        red, _, report = _run(c)
        launched |= red
        if report:
            inexact.append(c.id)
    want = set(_INV[0]) - set(km.UNREACHABLE)
    never = sorted(want - launched)
    print("kernel matrix: %d of %d reachable instantiations launched, %d cases, %d not bit-exact "
          "(%d compiled, %d unreachable)" % (len(want & launched), len(want), len(_CASES), len(inexact),
                                             len(_INV[0]), len(km.UNREACHABLE)))
    assert not never, "never launched: " + ", ".join(km.tuple_id(t) for t in never)
    assert not (launched & set(km.UNREACHABLE)), "an 'unreachable' kernel ran"
    assert not inexact, "not bit-exact: " + ", ".join(inexact)


# ---- NaN and +-inf through every accumulation path -----------------------------------------------------------------
def _nonfinite_case(reduce, ring):
    t = ("float", 4, 32, 1, {"sum": 0, "max": 2, "min": 3}[reduce], 0 if reduce == "sum" else 2, 0)
    pf = {0: 0, 3: 3, 35: km.LEAN | 3}[ring]
    return km.Case(t[:6] + (pf,), reduce, 1, 128, "none", False, False, ring, 64, "plan", seed=11 + ring)


@pytest.mark.parametrize("reduce,ring", [("max", 0), ("min", 0), ("sum", 0), ("sum", 3), ("sum", 35)])
def test_nan_and_inf_propagate(reduce, ring):
    """NaN and +-inf in a hub row, a row cut by tile boundaries, a row cut by chunk boundaries and a row of the last
    chunk (the lean ring's remainder loop), on the register path, the first-generation ring and the lean ring."""
    case = _nonfinite_case(reduce, ring)
    inp = km.make_inputs(case)
    src = inp.src.clone()                 # src row = edge id: each value below reaches exactly one edge
    nan, inf = float("nan"), float("inf")
    for name, hits in {"hub": [(0.3, 3, nan), (0.6, 4, inf)],
                       "medium": [(0.5, 5, -inf), (0.7, 9, inf)],
                       "chunky": [(0.2, 6, inf), (0.8, 6, -inf)],
                       "last": [(0.0, 7, nan), (0.0, 8, -inf)]}.items():
        edges = torch.nonzero(inp.dst == inp.rows[name]).flatten()
        for frac, col, v in hits:
            src[int(edges[int(frac * (edges.numel() - 1))]), col] = v
    inp.src = src
    ref = km.reference(case, inp)
    assert bool(torch.isnan(ref).any()) and bool(torch.isinf(ref).any())
    got, names = km.run_case(case, inp)
    assert ("reduce", case.target) in [km.parse_kernel(n) for n in names]
    report = km.mismatch_report(got, ref, inp)
    assert not report, report


# ---- the unsorted fp32 sum: vector / scalar atomics (scatter_add_kernel, abi.cu) -------------------------------------
@pytest.mark.parametrize("W", [128, 7, 130])
@pytest.mark.parametrize("gather", [False, True])
def test_unsorted_fp32_sum_exact(W, gather):
    """On the grid the atomics' order does not matter either: bit-exact, with rows that receive nothing."""
    from geot_b200 import abi
    g = torch.Generator().manual_seed(W + gather)
    E, N, S = 30011, 900, 700
    dst = torch.randint(0, S - 3, (E,), generator=g)
    dst[dst == 5] = 6                     # row 5 and the last three rows receive nothing
    si = torch.randint(0, N, (E,), generator=g) if gather else None
    src = km._grid((N if gather else E, W), g, 16, 4, torch.float32)
    case = km.Case(("float", 1, 1, 1, 0, 0, 0), "sum", 1, W, "none", gather, False, 0, 64, "planless", 0)
    inp = km.Inputs(src, si, dst, None, S, {})
    ref = km.reference(case, inp)
    abi.lib().geot_b200_set_unsorted_mode(0)
    dev = lambda x: None if x is None else x.to("cuda")
    with km.env(GEOT_B200_UNSORTED_SORT=0):
        out, names = km.launched_kernels(lambda: abi.segment_reduce(dev(src), dev(si), dev(dst), None, "sum", S=S,
                                                                    sorted=False))
    kern = "scatter_add_kernel<float4>" if W % 4 == 0 else "scatter_add_kernel<float>"
    assert any(kern in n for n in names), names
    report = km.mismatch_report(out.cpu(), ref, inp)
    assert not report, report
