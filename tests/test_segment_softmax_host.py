"""Host-side checks of the segment softmax -- no GPU needed, no compute calls: the C entries reject bad arguments with
their status codes before any CUDA call, the operators have their schemas, fakes and autograd kernel."""
import ctypes

import pytest
import torch

import geot_b200  # noqa: F401  (registers the operators, their fakes and the autograd)
from geot_b200 import abi


def _plan(E=10, sorted_=1):
    p = abi.GeotPlan()
    p.E, p.S, p.num_segments, p.max_degree, p.is_sorted, p.has_gaps, p.max_row = E, 4, 4, 3, sorted_, 0, 3
    return p


@pytest.mark.parametrize("entry", ["forward", "backward"])
def test_argument_validation_happens_before_any_device_work(entry):
    L = abi.lib()
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)  # never dereferenced: the calls must fail on validation
    ok = dict(E=10, H=4, dtype=abi.F32, plan=_plan(), ws=one, ws_bytes=1 << 20)
    n_ptrs = 3 if entry == "forward" else 4
    f = L.geot_b200_segment_softmax if entry == "forward" else L.geot_b200_segment_softmax_backward

    def call(ptrs=(one,) * n_ptrs, **kw):
        a = dict(ok, **kw)
        plan = ctypes.byref(a["plan"]) if a["plan"] is not None else None
        return f(*ptrs, a["E"], a["H"], a["dtype"], plan, a["ws"], a["ws_bytes"], null)

    for k in range(n_ptrs):            # every operand missing in turn
        ptrs = [one] * n_ptrs
        ptrs[k] = null
        assert call(ptrs=tuple(ptrs)) == 1
    assert call(plan=None) == 1
    assert call(ws=null) == 1
    assert call(H=0) == 1
    assert call(H=-3) == 1
    assert call(E=-1) == 1
    assert call(dtype=4) == 1
    assert call(dtype=-1) == 1
    assert call(E=0, plan=_plan(0)) == 5                        # empty
    assert call(plan=_plan(sorted_=0)) == 1                     # unsorted index
    assert call(plan=_plan(E=11)) == 1                          # a plan of another index
    assert call(ws=ctypes.c_void_p(264)) == 3                   # misaligned workspace
    need = L.geot_b200_segment_softmax_workspace_bytes(10, 4, abi.F32)
    assert call(ws_bytes=need - 1) == 3                         # too small
    for dt in (abi.F32, abi.F64, abi.BF16, abi.F16):
        assert call(dtype=dt, ws_bytes=L.geot_b200_segment_softmax_workspace_bytes(10, 4, dt) - 1) == 3


def test_workspace_bytes():
    L = abi.lib()
    ws = L.geot_b200_segment_softmax_workspace_bytes
    assert ws(0, 4, abi.F32) == 256 and ws(10, 0, abi.F32) == 256 and ws(10, 4, 7) == 256
    assert ws(1_000_000, 8, abi.F64) > ws(1_000_000, 8, abi.F32) > ws(1_000_000, 1, abi.F32)
    assert ws(1_000_000, 8, abi.BF16) == ws(1_000_000, 8, abi.F32)        # fp32 carries
    assert all(ws(E, H, abi.F32) % 256 == 0 for E in (1, 77, 10_000) for H in (1, 3, 300))


def test_schemas():
    s = lambda op: str(op.default._schema)
    assert s(torch.ops.geot.segment_softmax) == "geot::segment_softmax(Tensor src, Tensor index) -> Tensor"
    assert s(torch.ops.geot.segment_softmax_backward) == \
        "geot::segment_softmax_backward(Tensor out, Tensor grad_out, Tensor index) -> Tensor"


def test_cuda_only_and_autograd_registered():
    for op in ("geot::segment_softmax", "geot::segment_softmax_backward"):
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op, "CUDA")
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(op, "CPU")      # no fallback
    assert torch._C._dispatch_has_kernel_for_dispatch_key("geot::segment_softmax", "Autograd")
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.segment_softmax(torch.rand(4, 2), torch.tensor([0, 0, 1, 2]))


def test_fakes_trace():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        idx = torch.empty(7, dtype=torch.long)
        for shape in ((7,), (7, 3)):
            x = torch.empty(*shape)
            out = torch.ops.geot.segment_softmax(x, idx)
            assert out.shape == shape and out.dtype == x.dtype
            g = torch.ops.geot.segment_softmax_backward(out, out, idx)
            assert g.shape == shape
        xb = torch.empty(7, 4, dtype=torch.bfloat16)
        assert torch.ops.geot.segment_softmax(xb, idx).dtype == torch.bfloat16


def test_public_surface():
    import inspect
    from geot_b200 import gnn
    assert geot_b200.segment_softmax is geot_b200.softmax.segment_softmax
    assert list(inspect.signature(geot_b200.segment_softmax).parameters) == ["src", "index"]
    assert list(inspect.signature(gnn.GATConv).parameters) == [
        "in_channels", "out_channels", "heads", "concat", "negative_slope", "bias"]
    conv = gnn.GATConv(8, 5, heads=3)
    assert conv.lin.weight.shape == (15, 8) and conv.att_src.shape == (1, 3, 5) and conv.bias.shape == (15,)
    assert gnn.GATConv(8, 5, heads=3, concat=False).bias.shape == (5,)
    assert gnn.GATConv(8, 5, heads=3, bias=False).bias is None
