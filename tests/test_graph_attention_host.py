"""Host-side checks of the fused graph attention -- no GPU needed, no compute calls: the C entries reject bad arguments
with their status codes before any CUDA call; the workspace formulas; the operators have their schemas, fakes and
autograd kernel, and no CPU path."""
import ctypes

import pytest
import torch

import geot_b200  # noqa: F401  (registers the operators, their fakes and the autograd)
from geot_b200 import abi


def _plan(E=10, sorted_=1, max_row=3):
    p = abi.GeotPlan()
    p.E, p.S, p.num_segments, p.max_degree, p.is_sorted, p.has_gaps, p.max_row = E, max_row + 1, 4, 3, sorted_, 0, max_row
    p.rowptr = 256
    return p


null = ctypes.c_void_p(0)
one = ctypes.c_void_p(256)       # never dereferenced: the calls must fail on validation
scale = ctypes.c_double(0.25)


def _common_checks(call, need, n_ptrs):
    for k in range(n_ptrs):          # every operand missing in turn
        ptrs = [one] * n_ptrs
        ptrs[k] = null
        assert call(ptrs=tuple(ptrs)) == 1, k
    assert call(s=None) == 1                                  # the scale is an operand too
    assert call(plan=None) == 1
    assert call(ws=null) == 1
    for kw in (dict(H=0), dict(H=-2), dict(F=0), dict(F=-1), dict(E=-1), dict(dtype=4), dict(dtype=-1), dict(N=-1),
               dict(H=1 << 40, F=1 << 40), dict(E=1 << 40, H=1 << 20, F=1 << 20)):
        assert call(**kw) == 1, kw
    assert call(E=0, plan=_plan(0)) == 5                      # empty
    assert call(plan=_plan(sorted_=0)) == 1                   # unsorted index
    assert call(plan=_plan(E=11)) == 1                        # a plan of another index
    assert call(N=3) == 1                                     # an index value (3) >= N_dst
    p = _plan()
    p.rowptr = None
    assert call(plan=p) == 1                                  # a plan without row pointers
    assert call(ws=ctypes.c_void_p(264)) == 3                 # misaligned workspace
    assert call(ws_bytes=need(10, 4, 8, abi.F32) - 1) == 3    # too small
    for dt in (abi.F32, abi.F64, abi.BF16, abi.F16):
        assert call(dtype=dt, ws_bytes=need(10, 4, 8, dt) - 1) == 3
    # one head wider than a launch (256 columns; 128 for fp64): unsupported, whatever the workspace
    assert call(H=1, F=257, ws_bytes=1 << 30) == 2
    assert call(H=1, F=129, dtype=abi.F64, ws_bytes=1 << 30) == 2


def test_forward_argument_validation_happens_before_any_device_work():
    L = abi.lib()
    f = L.geot_b200_graph_attention
    need = L.geot_b200_graph_attention_workspace_bytes
    ok = dict(E=10, H=4, F=8, dtype=abi.F32, plan=_plan(), N=4, ws=one, ws_bytes=need(10, 4, 8, abi.F32))

    def call(ptrs=(one,) * 7, s=ctypes.byref(scale), **kw):
        a = dict(ok, **kw)
        plan = ctypes.byref(a["plan"]) if a["plan"] is not None else None
        q, k, v, si, di, out, lse = ptrs
        return f(q, k, v, si, di, plan, a["N"], out, lse, a["E"], a["H"], a["F"], a["dtype"], s, a["ws"], a["ws_bytes"],
                 null)

    _common_checks(call, need, 7)


def test_grad_argument_validation_happens_before_any_device_work():
    L = abi.lib()
    f = L.geot_b200_graph_attention_grad
    need = L.geot_b200_graph_attention_grad_workspace_bytes
    ok = dict(E=10, H=4, F=8, dtype=abi.F32, plan=_plan(), N=4, ws=one, ws_bytes=need(10, 4, 8, abi.F32))

    def call(ptrs=(one,) * 11, s=ctypes.byref(scale), **kw):
        a = dict(ok, **kw)
        plan = ctypes.byref(a["plan"]) if a["plan"] is not None else None
        q, k, v, out, lse, g, si, di, gq, p, ds = ptrs
        return f(q, k, v, out, lse, g, si, di, plan, a["N"], gq, p, ds, a["E"], a["H"], a["F"], a["dtype"], s, a["ws"],
                 a["ws_bytes"], null)

    _common_checks(call, need, 11)


def _layout(E, H, F, acc, backward, es):
    """The workspace formula: chunks of 256 edges per warp (halved down to 32 while fewer than 8 * 148 tiles of 8
    chunks); two [tiles, piece] accumulator arrays (tile carries in and out) with piece = wc + 2 * (wc // F) (acc, m, s)
    forward and wc backward, wc = min(H * F, slab); one flag byte per tile; backward: the all-ones [H * F] factor of the
    dtype.  256-byte aligned pieces."""
    a = lambda x: (x + 255) // 256 * 256
    chunk = 256
    while chunk > 32 and -(-E // (8 * chunk)) < 8 * 148:
        chunk //= 2
    tiles = -(-E // (8 * chunk))
    wc = min(H * F, 128 if acc == 8 else 256)
    piece = wc if backward else wc + 2 * (wc // F)
    return 2 * a(tiles * piece * acc) + a(tiles) + (a(H * F * es) if backward else 0)


def test_workspace_bytes():
    L = abi.lib()
    for backward, ws in ((False, L.geot_b200_graph_attention_workspace_bytes),
                         (True, L.geot_b200_graph_attention_grad_workspace_bytes)):
        assert ws(0, 4, 8, abi.F32) == 256 and ws(10, 0, 8, abi.F32) == 256 and ws(10, 4, 0, abi.F32) == 256
        assert ws(10, 4, 8, 7) == 256
        for E in (1, 77, 10_000, 1_166_243, 114_615_892):
            for H, F in ((1, 5), (4, 32), (8, 32), (3, 200), (16, 1)):
                for dt, acc, es in ((abi.F32, 4, 4), (abi.F64, 8, 8), (abi.BF16, 4, 2), (abi.F16, 4, 2)):
                    assert ws(E, H, F, dt) == _layout(E, H, F, acc, backward, es), (backward, E, H, F, dt)
    # Reddit shape, 4 x 32 fp32: a few MB, against 1.8 GB for one [E, H] fp32 tensor
    assert L.geot_b200_graph_attention_workspace_bytes(114_615_892, 4, 32, abi.F32) < 100e6


def test_schemas():
    s = lambda op: str(op.default._schema)
    assert s(torch.ops.geot.graph_attention) == ("geot::graph_attention(Tensor q, Tensor k, Tensor v, Tensor src_index, "
                                                 "Tensor dst_index, float scale) -> (Tensor, Tensor)")
    assert s(torch.ops.geot.graph_attention_backward) == (
        "geot::graph_attention_backward(Tensor grad, Tensor q, Tensor k, Tensor v, Tensor out, Tensor lse, "
        "Tensor src_index, Tensor dst_index, float scale) -> (Tensor, Tensor, Tensor)")


def test_cuda_only_and_autograd_registered():
    for op in ("geot::graph_attention", "geot::graph_attention_backward"):
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op, "CUDA")
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(op, "CPU")      # no fallback
    assert torch._C._dispatch_has_kernel_for_dispatch_key("geot::graph_attention", "Autograd")
    x = torch.rand(5, 2, 4)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.graph_attention(x, x, x, torch.tensor([0, 1, 2]), torch.tensor([0, 0, 1]))


def test_fakes_trace():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        si = torch.empty(7, dtype=torch.long)
        for dt, acc in ((torch.float32, torch.float32), (torch.bfloat16, torch.float32), (torch.float64, torch.float64)):
            q, k = torch.empty(5, 3, 4, dtype=dt), torch.empty(6, 3, 4, dtype=dt)
            out, lse = torch.ops.geot.graph_attention(q, k, k, si, si, 0.5)
            assert out.shape == q.shape and out.dtype == dt and lse.shape == (5, 3) and lse.dtype == acc
            gq, p, ds = torch.ops.geot.graph_attention_backward(out, q, k, k, out, lse, si, si, 0.5)
            assert gq.shape == q.shape and p.shape == (7, 3) and ds.shape == (7, 3) and p.dtype == dt


def test_public_surface():
    import inspect
    from geot_b200 import gnn
    assert geot_b200.graph_attention is geot_b200.attention.graph_attention
    sig = inspect.signature(geot_b200.graph_attention)
    assert list(sig.parameters) == ["q", "k", "v", "src_index", "dst_index", "scale"]
    assert sig.parameters["scale"].default is None
    assert list(inspect.signature(gnn.TransformerConv).parameters) == [
        "in_channels", "out_channels", "heads", "concat", "bias", "root_weight"]
    conv = gnn.TransformerConv(8, 5, heads=3)
    for lin in (conv.lin_query, conv.lin_key, conv.lin_value, conv.lin_skip):
        assert lin.weight.shape == (15, 8) and lin.bias.shape == (15,)
    assert gnn.TransformerConv(8, 5, heads=3, concat=False).lin_skip.weight.shape == (5, 8)
    assert gnn.TransformerConv(8, 5, heads=3, root_weight=False).lin_skip is None
    nb = gnn.TransformerConv(8, 5, heads=3, bias=False)
    assert all(l.bias is None for l in (nb.lin_query, nb.lin_key, nb.lin_value, nb.lin_skip))
