"""GPU checks of the mh_spmm backward: the multi-head SDDMM kernel (geot_b200_sddmm_mh / geot::sddmm_mh_impl) against
the C oracle, its H = 1 case against sddmm_coo, and the gradients of geot::mh_spmm against a torch restatement
(index_select * mul * index_add) in fp64, gradcheck, opcheck and a short training loop."""
import pytest
import torch

from tests.helpers import mh_oracle

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import geot_b200
    from geot_b200 import abi, transpose

DEV = "cuda"


def _graph(E, N, seed, sort=True, S=None):
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(N if S is None else S, generator=g) ** 3
    di = torch.multinomial(w / w.sum(), E, replacement=True, generator=g)
    si = torch.randint(0, N, (E,), generator=g)
    if sort:
        perm = torch.sort(di * N + si).indices
        si, di = si[perm], di[perm]
    return si.contiguous(), di.contiguous(), g


def _check(got, exp, tol):
    got, exp = got.detach().cpu().double(), exp.detach().cpu().double()
    if isinstance(tol, torch.Tensor):
        tol = tol.detach().cpu().double()
    assert got.shape == exp.shape, (got.shape, exp.shape)
    bad = (got - exp).abs() > tol
    assert not bad.any(), "%d bad, max err %.3e" % (int(bad.sum()), float((got - exp).abs().max()))


# ---- the kernel against the oracle ----------------------------------------------------------------------------------
SHAPES = [(4, 32, torch.float32), (8, 32, torch.bfloat16), (3, 5, torch.float32), (2, 130, torch.float32),
          (8, 8, torch.float16), (1, 64, torch.float32),
          (16, 16, torch.float32),      # above the 8-head fast path of the forward
          (4, 300, torch.float32),      # a wide row
          (4, 16, torch.float64), (3, 7, torch.float64)]


@pytest.mark.parametrize("H,F,dtype", SHAPES, ids=lambda v: str(v).replace("torch.", ""))
def test_sddmm_mh_vs_oracle(H, F, dtype):
    E, N = 5000, 300
    si, di, g = _graph(E, N, seed=H * 1000 + F)
    if dtype == torch.float32:          # mixed signs: tolerance from the conditioning of each dot product
        x1 = torch.rand(N, H, F, generator=g) - 0.25
        x2 = torch.rand(N, H, F, generator=g) - 0.25
    else:                               # 16-bit and fp64: positive data, relative tolerance
        x1 = (torch.rand(N, H, F, generator=g) + 0.1).to(dtype)
        x2 = (torch.rand(N, H, F, generator=g) + 0.1).to(dtype)
    for row, col in ((di, si), (si, di)):                               # sorted and unsorted row index
        exp = mh_oracle.sddmm_mh(col, row, x1, x2)
        if dtype == torch.float32:
            tol = 1e-5 * (x1[row].abs() * x2[col].abs()).sum(-1).double() + 1e-30
        else:
            tol = (1e-12 if dtype == torch.float64 else 1e-2) * exp.double().abs()
        for head_major in (False, True):
            got = torch.ops.geot.sddmm_mh_impl(col.to(DEV), row.to(DEV), x1.to(DEV), x2.to(DEV), head_major)
            assert got.dtype == dtype
            _check(got, exp.t() if head_major else exp, tol.t() if head_major else tol)
            got_abi = abi.sddmm_mh(x1.to(DEV), row.to(DEV), x2.to(DEV), col.to(DEV), head_major)
            assert torch.equal(got_abi, got)


def test_sddmm_mh_edge_cases():
    H, F = 4, 32
    x = torch.rand(7, H, F, device=DEV)
    one = torch.ops.geot.sddmm_mh_impl(torch.tensor([3], device=DEV), torch.tensor([5], device=DEV), x, x, False)
    _check(one, (x[5] * x[3]).sum(-1).view(1, H), 1e-6 * F)
    for head_major in (False, True):
        empty = torch.ops.geot.sddmm_mh_impl(torch.zeros(0, dtype=torch.long, device=DEV),
                                             torch.zeros(0, dtype=torch.long, device=DEV), x, x, head_major)
        assert empty.shape == ((H, 0) if head_major else (0, H))
    # one row spanning many chunks, with a ragged tail
    E = 70001
    di = torch.full((E,), 2, device=DEV)
    si = torch.randint(0, 7, (E,), device=DEV)
    exp = (x[di] * x[si]).sum(-1)
    _check(torch.ops.geot.sddmm_mh_impl(si, di, x, x, False), exp, 1e-5 * exp.abs())
    _check(torch.ops.geot.sddmm_mh_impl(si, di, x, x, True), exp.t(), 1e-5 * exp.t().abs())
    with pytest.raises(RuntimeError, match="same H and F"):
        torch.ops.geot.sddmm_mh_impl(si, di, x, torch.rand(7, H, 16, device=DEV), False)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16, torch.float16])
def test_sddmm_mh_single_head_is_sddmm_coo(dtype):
    for F in (5, 8, 64, 128, 136, 264, 1024):
        si, di, g = _graph(4000, 200, seed=F)
        x1 = torch.rand(200, F, generator=g).to(dtype).to(DEV)
        x2 = torch.rand(200, F, generator=g).to(dtype).to(DEV)
        si, di = si.to(DEV), di.to(DEV)
        ref = geot_b200.sddmm_coo_impl(si, di, x1, x2)
        for head_major in (False, True):
            got = torch.ops.geot.sddmm_mh_impl(si, di, x1.unsqueeze(1), x2.unsqueeze(1), head_major)
            assert torch.equal(got.reshape(-1), ref), (dtype, F)


# ---- gradients ------------------------------------------------------------------------------------------------------
def _restated(si, di, w_eh, x, reduce, S):
    out = torch.zeros((S,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    out = out.index_add(0, di, w_eh.unsqueeze(-1) * x.index_select(0, si))
    if reduce == "mean":
        deg = torch.bincount(di, minlength=S).clamp_min(1).to(x.dtype)
        out = out / deg.view(-1, 1, 1)
    return out


def _gap_graph(E=3000, N_used=60, N=65, S=80, seed=7):
    """dst rows with no edges (and none after the last one), src rows N_used .. N-1 that no edge reads"""
    si, di, g = _graph(E, N_used, seed=seed, S=S)
    di = torch.where(di % 5 == 1, di - 1, di)             # every fifth row empty
    di[-1] = S - 1
    perm = torch.sort(di * N + si).indices
    return si[perm].contiguous(), di[perm].contiguous(), N, S, g


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("reduce", ["sum", "mean"])
@pytest.mark.parametrize("layout", ["EH", "HE", "transposed"])
def test_gradients_vs_torch_restatement(dtype, reduce, layout):
    H, F = 4, 32
    si, di, N, S, g = _gap_graph()
    E = si.numel()
    w0 = torch.rand(E, H, generator=g).to(dtype)
    x0 = torch.rand(N, H, F, generator=g).to(dtype)
    gout = torch.rand(S, H, F, generator=g).to(dtype)
    rtol = 1e-4 if dtype == torch.float32 else 3e-2
    si_d, di_d = si.to(DEV), di.to(DEV)
    for wants in ((True, True), (True, False), (False, True)):
        w = (w0.t().contiguous() if layout == "HE" else w0).to(DEV).requires_grad_(wants[0])
        x = x0.to(DEV).requires_grad_(wants[1])
        if layout == "transposed":
            out = geot_b200.mh_spmm_transposed(si_d, di_d, w, x, reduce)
        else:
            out = geot_b200.mh_spmm(si_d, di_d, w, x, reduce)
        out.backward(gout.to(DEV))
        wr = w0.double().requires_grad_(wants[0])
        xr = x0.double().requires_grad_(wants[1])
        _restated(si, di, wr, xr, reduce, S).backward(gout.double())
        if wants[0]:
            exp = wr.grad.t() if layout == "HE" else wr.grad
            assert w.grad.shape == exp.shape and w.grad.dtype == dtype
            _check(w.grad, exp, rtol * exp.abs() + 1e-12)
        else:
            assert w.grad is None
        if wants[1]:
            assert x.grad.shape == x0.shape and x.grad.dtype == dtype
            _check(x.grad, xr.grad, rtol * xr.grad.abs() + 1e-12)
            assert x.grad[60:].abs().sum().item() == 0          # rows no edge reads
        else:
            assert x.grad is None


@pytest.mark.parametrize("head_major", [False, True])
def test_gradcheck_fp64(head_major):
    H, F = 3, 8
    si, di, g = _graph(40, 9, seed=11)
    di[-1] = 9
    si, di = si.to(DEV), di.to(DEV)
    w = torch.rand(40, H, generator=g, dtype=torch.float64)
    w = (w.t().contiguous() if head_major else w).to(DEV).requires_grad_(True)
    x = torch.rand(11, H, F, generator=g, dtype=torch.float64).to(DEV).requires_grad_(True)
    for reduce in ("sum", "mean"):
        assert torch.autograd.gradcheck(lambda w, x: geot_b200.mh_spmm(si, di, w, x, reduce), (w, x))


def test_backward_hits_the_transpose_cache():
    H, F = 4, 32
    si, di, N, S, g = _gap_graph(seed=3)
    si, di = si.to(DEV), di.to(DEV)
    w0 = torch.rand(si.numel(), H, generator=g).to(DEV)
    x0 = torch.rand(N, H, F, generator=g).to(DEV)
    transpose.clear_transpose_cache()
    grads = []
    for _ in range(2):
        x = x0.clone().requires_grad_(True)
        geot_b200.mh_spmm(si, di, w0, x).sum().backward()
        grads.append(x.grad)
    assert len(transpose._CACHE) == 1                          # the second backward found the first one's entry
    assert torch.equal(grads[0], grads[1])
    entry = next(iter(transpose._CACHE.values()))
    si2 = si.clone()
    si2[0] = (si2[0] + 1) % N                                  # another graph must not hit it
    x = x0.clone().requires_grad_(True)
    geot_b200.mh_spmm(si2, di, w0, x).sum().backward()
    assert len(transpose._CACHE) == 2
    assert transpose.transposed_edges(si, di) is entry
    xr = x0.double().requires_grad_(True)
    _restated(si2, di, w0.double(), xr, "sum", S).sum().backward()
    _check(x.grad, xr.grad, 1e-4 * xr.grad.abs() + 1e-12)


def test_gradients_arrive():
    si, di, g = _graph(2000, 50, seed=5)
    si, di = si.to(DEV), di.to(DEV)
    w = torch.rand(2000, 8, generator=g).to(DEV).requires_grad_(True)
    x = torch.rand(50, 8, 32, generator=g).to(DEV).requires_grad_(True)
    geot_b200.mh_spmm(si, di, w, x).square().sum().backward()
    assert w.grad is not None and x.grad is not None
    assert w.grad.abs().sum().item() > 0 and x.grad.abs().sum().item() > 0


def test_forward_unchanged_and_no_backward_for_max():
    si, di, g = _graph(3000, 80, seed=9)
    si, di = si.to(DEV), di.to(DEV)
    w0 = torch.rand(3000, 4, generator=g).to(DEV)
    x0 = torch.rand(80, 4, 32, generator=g).to(DEV)
    for reduce in ("sum", "mean", "max", "min", "prod"):
        ref = geot_b200.mh_spmm(si, di, w0, x0, reduce)
        w, x = w0.clone().requires_grad_(True), x0.clone().requires_grad_(True)
        out = geot_b200.mh_spmm(si, di, w, x, reduce)
        assert out.requires_grad
        assert torch.equal(out.detach(), ref), reduce
    with pytest.raises(NotImplementedError, match="max"):
        out = geot_b200.mh_spmm(si, di, w, x, "max")
        out.sum().backward()


def test_opcheck():
    si, di, g = _graph(500, 30, seed=13)
    di[-1] = 29
    si, di = si.to(DEV), di.to(DEV)
    x = torch.rand(30, 4, 16, generator=g).to(DEV)
    for w in (torch.rand(500, 4, generator=g), torch.rand(4, 500, generator=g)):
        torch.library.opcheck(torch.ops.geot.mh_spmm.default,
                              (si, di, w.to(DEV).requires_grad_(True), x.clone().requires_grad_(True), "sum"),
                              test_utils=("test_schema", "test_autograd_registration"))
    for head_major in (False, True):
        torch.library.opcheck(torch.ops.geot.sddmm_mh_impl.default, (si, di, x, x, head_major),
                              test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))


# ---- a short training loop ------------------------------------------------------------------------------------------
def _segment_softmax(logits, di, S):
    """softmax of [E, H] logits over the edges of each dst row"""
    idx = di.view(-1, 1).expand_as(logits)
    m = torch.full((S, logits.shape[1]), float("-inf"), device=logits.device).scatter_reduce(0, idx, logits, "amax")
    ex = (logits - m[di]).exp()
    den = torch.zeros(S, logits.shape[1], device=logits.device).index_add(0, di, ex)
    return ex / den[di]


def test_two_layer_attention_training_matches_restatement():
    H, F, N, E = 4, 16, 200, 3000
    si, di, g = _graph(E, N, seed=17)
    di[-1] = N - 1
    si, di = si.to(DEV), di.to(DEV)
    x0 = torch.randn(N, H * F, generator=g).to(DEV)
    target = torch.randn(N, H * F, generator=g).to(DEV)
    init = [t.to(DEV) for t in (torch.randn(H * F, H * F, generator=g) * 0.1, torch.randn(H, F, generator=g) * 0.1,
                                torch.randn(H, F, generator=g) * 0.1) * 2]

    def run(aggregate):
        params = [p.clone().requires_grad_(True) for p in init]
        opt = torch.optim.SGD(params, lr=0.5)
        losses = []
        for _ in range(5):
            x = x0
            for layer in range(2):
                W, a_src, a_dst = params[3 * layer:3 * layer + 3]
                h = (x @ W).view(N, H, F)
                logits = torch.nn.functional.leaky_relu((h * a_src).sum(-1)[si] + (h * a_dst).sum(-1)[di], 0.2)
                alpha = _segment_softmax(logits, di, N)
                x = aggregate(alpha, h).reshape(N, H * F)
                if layer == 0:
                    x = torch.nn.functional.elu(x)
            loss = (x - target).square().mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(loss.detach())
        return losses, [p.detach() for p in params]

    got_l, got_p = run(lambda alpha, h: geot_b200.mh_spmm(si, di, alpha, h))
    exp_l, exp_p = run(lambda alpha, h: _restated(si, di, alpha, h, "sum", N))
    for a, b in zip(got_l, exp_l):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-7), (got_l, exp_l)
    for a, b in zip(got_p, exp_p):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6)
