"""Host-side checks of the GATv2 score -- no GPU needed, no compute calls: the C entries reject bad arguments with their
status codes before any CUDA call; the workspace formula; the operators have their schemas, fakes and autograd kernel,
and no CPU path."""
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
slope = ctypes.c_double(0.2)


def test_score_argument_validation_happens_before_any_device_work():
    f = abi.lib().geot_b200_gatv2_score
    ok = dict(E=10, H=4, F=8, dtype=abi.F32)

    def call(ptrs=(one,) * 6, s=ctypes.byref(slope), **kw):
        a = dict(ok, **kw)
        return f(*ptrs, a["E"], a["H"], a["F"], a["dtype"], s, null)

    for k in range(6):               # every operand missing in turn
        ptrs = [one] * 6
        ptrs[k] = null
        assert call(ptrs=tuple(ptrs)) == 1
    assert call(s=None) == 1                                  # the slope is an operand too
    for kw in (dict(H=0), dict(H=-2), dict(F=0), dict(F=-1), dict(E=-1), dict(dtype=4), dict(dtype=-1),
               dict(H=1 << 40, F=1 << 40), dict(E=1 << 40, H=1 << 20, F=1 << 20)):
        assert call(**kw) == 1, kw
    assert call(E=0) == 5                                     # empty


def test_grad_argument_validation_happens_before_any_device_work():
    L = abi.lib()
    f = L.geot_b200_gatv2_grad
    need = L.geot_b200_gatv2_grad_workspace_bytes(10, 4, 8, abi.F32)
    ok = dict(E=10, H=4, F=8, dtype=abi.F32, plan=_plan(), S_out=4, ws=one, ws_bytes=need, grad_att=one)

    def call(ptrs=(one,) * 6, s=ctypes.byref(slope), out=one, **kw):
        a = dict(ok, **kw)
        plan = ctypes.byref(a["plan"]) if a["plan"] is not None else None
        return f(*ptrs, plan, a["S_out"], out, a["grad_att"], a["E"], a["H"], a["F"], a["dtype"], s, a["ws"],
                 a["ws_bytes"], null)

    for k in range(6):               # x_row, x_gat, att, grad_score, row_index, gat_index missing in turn
        ptrs = [one] * 6
        ptrs[k] = null
        assert call(ptrs=tuple(ptrs)) == 1
    assert call(out=null) == 1
    assert call(s=None) == 1
    assert call(plan=None) == 1
    assert call(ws=null) == 1
    for kw in (dict(H=0), dict(F=0), dict(E=-1), dict(dtype=4), dict(dtype=-1), dict(S_out=-1),
               dict(H=1 << 40, F=1 << 40)):
        assert call(**kw) == 1, kw
    assert call(E=0, plan=_plan(0)) == 5                      # empty
    assert call(plan=_plan(sorted_=0)) == 1                   # unsorted index
    assert call(plan=_plan(E=11)) == 1                        # a plan of another index
    assert call(S_out=3) == 1                                 # the plan's largest index (3) needs 4 output rows
    p = _plan()
    p.rowptr = None
    assert call(plan=p) == 1                                  # a plan without row pointers
    assert call(ws=ctypes.c_void_p(264)) == 3                 # misaligned workspace
    assert call(ws_bytes=need - 1) == 3                       # too small
    assert call(grad_att=null, ws_bytes=need - 1) == 3        # grad_att may be null: the workspace check comes next
    for dt in (abi.F32, abi.F64, abi.BF16, abi.F16):
        assert call(dtype=dt, ws_bytes=L.geot_b200_gatv2_grad_workspace_bytes(10, 4, 8, dt) - 1) == 3


def _layout(E, W, acc):
    """The workspace formula: chunks of 256 edges per warp (halved down to 32 while fewer than 8 * 148 tiles of 8
    chunks), three [tiles, min(W, slab)] accumulator arrays (tile carries in and out, grad_att partials), the
    [256, min(W, slab)] second-level grad_att partials and one flag byte per tile; 256-byte aligned pieces."""
    a = lambda x: (x + 255) // 256 * 256
    chunk = 256
    while chunk > 32 and -(-E // (8 * chunk)) < 8 * 148:
        chunk //= 2
    tiles = -(-E // (8 * chunk))
    wc = min(W, 128 if acc == 8 else 256)
    return 3 * a(tiles * wc * acc) + a(256 * wc * acc) + a(tiles)


def test_workspace_bytes():
    ws = abi.lib().geot_b200_gatv2_grad_workspace_bytes
    assert ws(0, 4, 8, abi.F32) == 256 and ws(10, 0, 8, abi.F32) == 256 and ws(10, 4, 0, abi.F32) == 256
    assert ws(10, 4, 8, 7) == 256
    for E in (1, 77, 10_000, 1_166_243, 114_615_892):
        for H, F in ((1, 5), (4, 32), (8, 32), (3, 200)):
            for dt, acc in ((abi.F32, 4), (abi.F64, 8), (abi.BF16, 4), (abi.F16, 4)):
                assert ws(E, H, F, dt) == _layout(E, H * F, acc), (E, H, F, dt)
    # Reddit shape, 4 x 32 fp32: tens of MB, against 58.7 GB for one [E, H * F] tensor
    assert ws(114_615_892, 4, 32, abi.F32) < 100e6


def test_schemas():
    s = lambda op: str(op.default._schema)
    assert s(torch.ops.geot.gatv2_score) == ("geot::gatv2_score(Tensor x_l, Tensor x_r, Tensor att, Tensor src_index, "
                                             "Tensor dst_index, float negative_slope) -> Tensor")
    assert s(torch.ops.geot.gatv2_score_backward) == (
        "geot::gatv2_score_backward(Tensor grad, Tensor x_l, Tensor x_r, Tensor att, Tensor src_index, Tensor dst_index, "
        "Tensor t_perm, Tensor t_dst_index, Tensor t_src_index, float negative_slope, bool need_x_l, bool need_x_r, "
        "bool need_att) -> (Tensor, Tensor, Tensor)")


def test_cuda_only_and_autograd_registered():
    for op in ("geot::gatv2_score", "geot::gatv2_score_backward"):
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op, "CUDA")
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(op, "CPU")      # no fallback
    assert torch._C._dispatch_has_kernel_for_dispatch_key("geot::gatv2_score", "Autograd")
    x = torch.rand(5, 2, 4)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.gatv2_score(x, x, torch.rand(2, 4), torch.tensor([0, 1, 2]), torch.tensor([0, 0, 1]))


def test_fakes_trace():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        si = torch.empty(7, dtype=torch.long)
        for dt in (torch.float32, torch.bfloat16):
            x_l, x_r, att = torch.empty(5, 3, 4, dtype=dt), torch.empty(6, 3, 4, dtype=dt), torch.empty(3, 4, dtype=dt)
            s = torch.ops.geot.gatv2_score(x_l, x_r, att, si, si, 0.2)
            assert s.shape == (7, 3) and s.dtype == dt
            gl, gr, ga = torch.ops.geot.gatv2_score_backward(s, x_l, x_r, att, si, si, si, si, si, 0.2, True, True, True)
            assert gl.shape == x_l.shape and gr.shape == x_r.shape and ga.shape == att.shape and gl.dtype == dt
            gl, gr, ga = torch.ops.geot.gatv2_score_backward(s, x_l, x_r, att, si, si, si, si, si, 0.2, False, True, False)
            assert gl.numel() == 0 and gr.shape == x_r.shape and ga.numel() == 0


def test_public_surface():
    import inspect
    from geot_b200 import gnn
    assert geot_b200.gatv2_score is geot_b200.gatv2.gatv2_score
    assert list(inspect.signature(geot_b200.gatv2_score).parameters) == [
        "x_l", "x_r", "att", "src_index", "dst_index", "negative_slope"]
    assert inspect.signature(geot_b200.gatv2_score).parameters["negative_slope"].default == 0.2
    assert list(inspect.signature(gnn.GATv2Conv).parameters) == [
        "in_channels", "out_channels", "heads", "concat", "negative_slope", "bias"]
    conv = gnn.GATv2Conv(8, 5, heads=3)
    assert conv.lin_l.weight.shape == (15, 8) and conv.lin_r.weight.shape == (15, 8)
    assert conv.att.shape == (1, 3, 5) and conv.bias.shape == (15,) and conv.lin_l.bias.shape == (15,)
    assert torch.equal(conv.lin_l.bias, torch.zeros(15)) and torch.equal(conv.bias, torch.zeros(15))
    assert gnn.GATv2Conv(8, 5, heads=3, concat=False).bias.shape == (5,)
    nb = gnn.GATv2Conv(8, 5, heads=3, bias=False)
    assert nb.bias is None and nb.lin_l.bias is None and nb.lin_r.bias is None
