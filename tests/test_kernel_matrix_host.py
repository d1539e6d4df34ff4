"""Host checks of the kernel matrix (tests/helpers/kernel_matrix.py) -- no GPU needed.

The compiled segment-reduce kernels are listed from the library binary; every one must have a case that the restated
dispatch rules send to it (or a written reason why no call can reach it), the case graphs must have the row classes
where these kernels go wrong, and the exact reference must hold its precondition and agree with the C oracle.
"""
import collections

import pytest
import torch

import oracle
from tests.helpers import kernel_matrix as km

RTOL = {torch.float32: 1e-5, torch.float64: 1e-12, torch.bfloat16: 1e-2, torch.float16: 1e-2}


@pytest.fixture(scope="module")
def inv():
    return km.inventory()


@pytest.fixture(scope="module")
def cases(inv):
    return [c for t in sorted(inv[0]) for c in km.cases_for(t)]


def test_inventory_lists_reduce_and_fixup_kernels(inv):
    red, fix = inv
    assert len(red) > 0 and len(fix) > 0
    for t in red:
        assert (t[0], t[4]) in fix, "no segment_fixup_kernel<%s, %d> for %s" % (t[0], t[4], t)
    assert {(t[0], t[4]) for t in red} == set(fix)
    assert {t[0] for t in red} == set(km.DTYPES)
    assert {t[6] for t in red} >= {0, 2, 3, 35, 39, 99, 103, 163, 227}


def test_parse_kernel_normalises_profiler_and_cuobjdump_names():
    assert km.parse_kernel("void geot::segment_reduce_kernel<float, 4, 32, 1, 0, 1, 35>(geot::Params)") == \
        ("reduce", ("float", 4, 32, 1, 0, 1, 35))
    assert km.parse_kernel("void geot::segment_reduce_kernel<__nv_bfloat16, (int)8, (int)32, (int)2, (int)0, (int)2, "
                           "(int)227>(geot::Params)") == ("reduce", ("__nv_bfloat16", 8, 32, 2, 0, 2, 227))
    assert km.parse_kernel("void geot::segment_fixup_kernel<__half, 3>(geot::Params)") == ("fixup", ("__half", 3))
    assert km.parse_kernel("void (anonymous namespace)::zero_empty_rows_kernel(long const*)") is None


def test_every_compiled_kernel_has_a_case(inv):
    """An instantiation without a case means the kernel family grew without a test."""
    missing, wrong = [], []
    for t in sorted(inv[0]):
        try:
            cs = km.cases_for(t)
        except LookupError:
            cs = None
        if not cs:
            if t not in km.UNREACHABLE:
                missing.append(km.tuple_id(t))
            continue
        for c in cs:
            if km.dispatch(c) != t:
                wrong.append("%s -> %s" % (c.id, km.tuple_id(km.dispatch(c))))
    assert not missing, "no case reaches: " + ", ".join(missing)
    assert not wrong, "cases dispatched elsewhere: " + "; ".join(wrong)
    assert set(km.UNREACHABLE) <= set(inv[0]), "stale UNREACHABLE entries"
    for t, why in km.UNREACHABLE.items():
        assert why
        # no row width at all gives this shape with two or more heads
        assert not any(list(km._widths(t, h, m)) for h in range(2, 17) for m in (False, True))


def test_sum_kernels_run_sum_and_mean(cases):
    got = collections.defaultdict(set)
    for c in cases:
        got[c.target].add(c.reduce)
    for t, r in got.items():
        assert r == ({"sum", "mean"} if t[4] == 0 else {km.RED_NAMES[t[4]]}), t


def test_cases_cover_weight_layouts_options_and_shapes(cases):
    # weight modes: none through index_scatter and gather, [E], [E,H] and [H,E] with H >= 2, H = 16/sizeof(T) in [E,H]
    # on the per-head lean ring (its 16-byte weight load), H > 8 on the fallback ring
    wm0 = [c for c in cases if c.target[5] == 0 and c.target[4] == 0]
    assert any(c.gather for c in wm0) and any(not c.gather for c in wm0)
    assert any(c.weight == "edge" for c in cases)
    for lay in ("eh", "he"):
        assert any(c.weight == lay and c.H >= 2 and c.target[4] == 0 for c in cases)
        assert any(c.weight == lay and c.H >= 2 and c.target[4] != 0 for c in cases)
    for dt in ("float", "__nv_bfloat16", "__half"):
        assert any(c.target[0] == dt and c.target[6] & km.HEADW and c.weight == "eh" and c.H == 16 // km.esize(dt)
                   for c in cases), dt
    assert any(c.H > km.HEAD_MAX and c.ring & km.LEAN for c in cases)
    # the segment_reduce_ex forms: reached by every one of the four options between them
    ext = {c.mode for c in cases if c.target[6] & km.EXT}
    assert {"planless", "accumulate", "edge_perm", "mean_rowptr"} <= ext
    # VECW 1 both through a row width that is not a whole number of vectors and through a misaligned src
    v1 = [c for c in cases if c.target[1] == 1]
    assert any(c.misaligned for c in v1) and any(not c.misaligned for c in v1)
    # more than one column tile for every row shape that can have them
    shapes = collections.defaultdict(list)
    for c in cases:
        shapes[c.target[:4]].append(km.choose_config(c.W, c.F, c.target[0], not c.misaligned)[3])
    for s, tiles in shapes.items():
        dt, vecw, lpr, vpl = s
        if vpl == 4 or (vpl == 2 and vecw == 8):
            assert max(tiles) > 1, s
    # the fixup's long-chain forms: float4 (fp32 accumulator, W % 4 == 0, also W > 1024), scalar, fp64
    acc32 = [c for c in cases if c.target[0] != "double"]
    assert any(c.W % 4 == 0 and c.W > 1024 for c in acc32)
    assert any(c.W % 4 != 0 for c in acc32)
    assert any(c.target[0] == "double" for c in cases)


@pytest.mark.parametrize("lpr", [1, 2, 4, 8, 16, 32])
def test_case_graph_row_classes(lpr):
    chunk = 2 * lpr
    g = km.make_graph(lpr, chunk, torch.Generator().manual_seed(lpr))
    dst, S, rows = g.dst, g.S, g.rows
    E = dst.numel()
    tile = (km.K_THREADS // lpr) * chunk
    deg = torch.bincount(dst, minlength=S)
    assert bool((dst[1:] >= dst[:-1]).all())
    assert S > int(dst[-1]) + 1 and int(deg[-4:].sum()) == 0          # empty rows at the end ...
    assert int(deg[0]) == 0                                            # ... at the start ...
    inner = deg[int(dst[0]):int(dst[-1])]
    assert bool((inner == 0).any())                                    # ... and in the middle
    for d in range(1, 8):
        assert bool((deg == d).any()), d

    def tiles_cut(r):
        first = int(torch.nonzero(dst == r)[0])
        last = int(torch.nonzero(dst == r)[-1])
        return last // tile - first // tile, last // chunk - first // chunk
    assert tiles_cut(rows["hub"])[0] > km.K_LONG                       # the long-chain fixup
    assert 1 <= tiles_cut(rows["medium"])[0] <= km.K_LONG              # the short-chain fixup
    assert tiles_cut(rows["chunky"])[1] >= 2 and tiles_cut(rows["chunky"])[0] == 0
    if lpr > 1:                                                         # a last chunk of one whole batch and a part
        assert lpr < E % chunk < 2 * lpr and E % lpr != 0
    assert int(dst[-1]) == rows["last"]
    assert int(deg.max()) * 2 < km.EXACT_BOUND


def _sample(cases, n):
    step = max(1, len(cases) // n)
    return cases[::step]


def test_reference_precondition_and_rounding(cases):
    """For a spread of cases: every row's sum |p| is below 2^18 (the reference asserts it), the inputs are on the grid
    in the case's dtype, and the reference is a single rounding of the fp64 result."""
    for c in _sample(cases, 60):
        inp = km.make_inputs(c)
        assert torch.equal(inp.src.double() * 16, (inp.src.double() * 16).round())
        if inp.weight is not None:
            assert torch.equal(inp.weight.double() * 4, (inp.weight.double() * 4).round())
        ref = km.reference(c, inp)
        assert ref.dtype == c.dtype and tuple(ref.shape) == (inp.S, c.W)
        cnt = torch.bincount(inp.dst, minlength=inp.S)
        if inp.prior is None:
            assert bool((ref[cnt == 0] == 0).all()), c.id
        else:
            assert torch.equal(ref[cnt == 0], inp.prior[cnt == 0]), c.id


def test_reference_rounds_like_the_kernels():
    """mean: fp32(s) / fp32(n) as IEEE division, then the output type; accumulate: RN(prior + RN(s)) per pass."""
    c = km.Case(("__nv_bfloat16", 8, 32, 1, 0, 0, 0), "mean", 1, 8, "none", False, False, 0, 64, "plan", 0)
    inp = km.Inputs(torch.tensor([[1.0] * 8, [1.0] * 8, [0.0625] * 8]).bfloat16(), None, torch.tensor([0, 0, 0]),
                    None, 2, {})
    ref = km.reference(c, inp)
    assert torch.equal(ref[0], (torch.tensor(2.0625, dtype=torch.float32) / 3).bfloat16().expand(8))
    assert torch.equal(ref[1], torch.zeros(8, dtype=torch.bfloat16))
    c2 = km.Case(("__nv_bfloat16", 8, 32, 1, 0, 0, 0), "sum", 1, 8, "none", False, False, 0, 64, "accumulate", 0)
    inp2 = km.Inputs(torch.tensor([[2.0 ** -6] * 8]).bfloat16(), None, torch.tensor([0]), None, 2, {},
                     prior=torch.tensor([[4.0] * 8, [3.0] * 8]).bfloat16())
    ref2 = km.reference(c2, inp2)       # 4 + 2^-6 is a tie in bf16: rounds to even, 4
    assert torch.equal(ref2[0], torch.full((8,), 4.0).bfloat16()) and torch.equal(ref2[1], inp2.prior[1])


def test_prod_factors_stay_in_range(cases):
    for c in [c for c in cases if c.reduce == "prod"][::7]:
        ref = km.reference(c, km.make_inputs(c)).double()
        nz = ref[ref != 0].abs()
        assert bool(torch.isfinite(ref).all())
        assert float(nz.max()) <= 2.0 ** 8 and float(nz.min()) >= 2.0 ** -8, c.id


@pytest.mark.parametrize("dt", list(km.DTYPES))
def test_reference_agrees_with_the_oracle(dt, inv):
    """The exact reference is pinned to oracle.segment_reduce(acc64=True) within the oracle's tolerance, once per dtype
    and reduce op."""
    picked = {}
    for t in sorted(inv[0]):
        if t[0] != dt:
            continue
        for c in km.cases_for(t):
            if c.mode in ("plan", "planless") and c.W <= 300:
                picked.setdefault((c.reduce, c.weight), c)
    assert {r for r, _ in picked} == ({"sum", "mean", "max", "min", "prod"})
    for c in picked.values():
        inp = km.make_inputs(c)
        ref = km.reference(c, inp)
        w = inp.weight
        orc = oracle.segment_reduce(inp.src, inp.src_index, inp.dst, w, c.reduce, S=inp.S, H=c.H,
                                    weight_transposed=(c.weight == "he"), acc64=True)
        orc = orc.reshape(inp.S, c.W)
        if c.reduce in ("max", "min", "prod"):
            assert torch.equal(ref, orc), c.id
        else:
            g, e = ref.double(), orc.double()
            assert bool(((g - e).abs() <= RTOL[c.dtype] * e.abs() + 1e-30).all()), c.id
