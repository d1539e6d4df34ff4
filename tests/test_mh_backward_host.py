"""Host-side checks of the mh_spmm backward -- no GPU needed, no compute calls: geot_b200_sddmm_mh rejects bad
arguments before any CUDA call, geot::mh_spmm has an Autograd kernel, and geot::sddmm_mh_impl has a schema and a
fake."""
import ctypes

import torch

import geot_b200  # noqa: F401  (registers the operators, their fakes and the autograd)
from geot_b200 import abi


def test_sddmm_mh_argument_validation_happens_before_any_device_work():
    f = abi.lib().geot_b200_sddmm_mh
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)  # never dereferenced: the calls must fail on validation
    ok = dict(E=10, H=4, F=8, dtype=abi.F32, layout=abi.W_EDGE_HEAD)

    def call(ptrs=(one,) * 5, **kw):
        a = dict(ok, **kw)
        return f(*ptrs, a["E"], a["H"], a["F"], a["dtype"], a["layout"], null)

    assert call(E=-1) == 1
    assert call(H=0) == 1
    assert call(H=-2) == 1
    assert call(F=0) == 1
    assert call(F=-8) == 1
    assert call(dtype=9) == 1
    assert call(dtype=-1) == 1
    for layout in (abi.W_NONE, abi.W_EDGE, 7):
        assert call(layout=layout) == 1
    for k in range(5):      # each of mat1, row_index, mat2, col_index, out missing
        ptrs = [one] * 5
        ptrs[k] = null
        assert call(ptrs=tuple(ptrs)) == 1
    assert call(E=0) == 0
    assert call(ptrs=(null,) * 5, E=0, layout=abi.W_HEAD_EDGE) == 0      # empty buffers may be null


def test_mh_spmm_has_an_autograd_kernel():
    assert torch._C._dispatch_has_kernel_for_dispatch_key("geot::mh_spmm", "Autograd")
    s = str(torch.ops.geot.mh_spmm.default._schema)
    assert s == "geot::mh_spmm(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src, str reduce) -> Tensor"


def test_sddmm_mh_impl_has_a_schema_and_a_fake():
    s = str(torch.ops.geot.sddmm_mh_impl.default._schema)
    assert s == "geot::sddmm_mh_impl(Tensor src_index, Tensor dst_index, Tensor mat_1, Tensor mat_2, bool head_major) -> Tensor"
    assert torch._C._dispatch_has_kernel_for_dispatch_key("geot::sddmm_mh_impl", "CUDA")
    assert not torch._C._dispatch_has_kernel_for_dispatch_key("geot::sddmm_mh_impl", "CPU")   # no fallback
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        idx = torch.empty(7, dtype=torch.long)
        x = torch.empty(5, 3, 16)
        assert torch.ops.geot.sddmm_mh_impl(idx, idx, x, x, False).shape == (7, 3)
        assert torch.ops.geot.sddmm_mh_impl(idx, idx, x, x, True).shape == (3, 7)
