"""GPU checks of geot::segment_softmax and its backward (geot_b200_segment_softmax{,_backward}): exact on constant
logits, against an fp64 restatement within bounds derived from the kernels' accumulation order, special values as
torch.softmax, gradcheck / opcheck, determinism and input handling; and gnn.GATConv against an fp64 restatement of
PyG's GATConv math, forward, gradients and a short training loop."""
import pytest
import torch

from tests.helpers import softmax_oracle as so

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import geot_b200
    from geot_b200 import abi
    from geot_b200.gnn import GATConv, add_self_loops

DEV = "cuda"
DTYPES = [torch.float32, torch.float64, torch.bfloat16, torch.float16]
ids = lambda v: str(v).replace("torch.", "")


def _check(got, exp, tol):
    got, exp = got.detach().cpu().double(), exp.detach().cpu().double()
    if isinstance(tol, torch.Tensor):
        tol = tol.detach().cpu().double()
    assert got.shape == exp.shape, (got.shape, exp.shape)
    bad = ~((got - exp).abs() <= tol)
    assert not bad.any(), "%d bad of %d, max err %.3e" % (int(bad.sum()), bad.numel(), float((got - exp).abs().max()))


def _src(E, H, g, scale, dtype):
    x = (torch.rand(E, H, generator=g, dtype=torch.float64) * 2 - 1) * scale
    x = x.to(dtype)
    return x.view(E) if H == 1 else x


# ---- exact: constant logits in every row give 1 / deg, the accumulator's division ------------------------------------
@pytest.fixture(scope="module")
def exact_graph():
    return so.exact_graph()


@pytest.mark.parametrize("H", [1, 2, 3, 4, 8, 16])
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_constant_logits_are_exact(exact_graph, dtype, H):
    index, _ = exact_graph
    E = index.numel()
    g = torch.Generator().manual_seed(H)
    rows = int(index[-1]) + 1
    level = torch.randint(-8, 9, (rows, H), generator=g).to(dtype)          # exactly representable in every dtype
    src = level[index].contiguous()
    deg = so.degrees(index)
    acc = torch.float64 if dtype == torch.float64 else torch.float32
    exp = (1.0 / deg.to(acc)).view(E, 1).expand(E, H).to(dtype)
    src = src.view(E) if H == 1 else src
    exp = exp.reshape(src.shape)
    got = geot_b200.segment_softmax(src.to(DEV), index.to(DEV))
    assert got.dtype == dtype and got.shape == src.shape
    assert torch.equal(got.cpu(), exp)
    assert torch.equal(got.cpu()[deg == 1], torch.ones_like(exp[deg == 1]))   # a degree-1 row gives exactly 1


# ---- against fp64 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", [10.0, 1000.0])
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_forward_vs_fp64(dtype, scale):
    index, g = so.random_graph(30_000, 900, seed=int(scale), hub=9_001)
    E = index.numel()
    deg = so.degrees(index)
    for H in (1, 3, 8, 16):
        src = _src(E, H, g, scale, dtype)
        exp = so.softmax(src, index)
        got = geot_b200.segment_softmax(src.to(DEV), index.to(DEV))
        _check(got, exp, so.forward_tolerance(exp, deg, H, dtype, src, index))


def test_special_values_follow_torch_softmax():
    """NaN, +inf and all -inf rows: the NaN positions of a per-row torch.softmax, exactly; the finite values close."""
    index, g = so.random_graph(20_000, 400, seed=5, hub=5_000)
    E, H = index.numel(), 4
    x = (torch.rand(E, H, generator=g) * 20 - 10)
    rowptr = torch.cat([torch.zeros(1, dtype=torch.long), torch.bincount(index).cumsum(0)])
    rows = torch.nonzero(rowptr[1:] > rowptr[:-1]).view(-1)
    hub_row = int(torch.argmax(rowptr[1:] - rowptr[:-1]))
    picks = torch.cat([rows[torch.randperm(rows.numel(), generator=g)[:60]], torch.tensor([hub_row])])
    for k, r in enumerate(picks.tolist()):
        a, b = int(rowptr[r]), int(rowptr[r + 1])
        h = k % H
        kind = k % 5
        e = a + int(torch.randint(0, b - a, (1,), generator=g))
        if kind == 0:
            x[e, h] = float("nan")
        elif kind == 1:
            x[e, h] = float("inf")
        elif kind == 2:
            x[a:b, h] = float("-inf")
        elif kind == 3:
            x[e, h] = float("-inf")                              # one -inf among finite logits: 0 there
        else:
            x[a:b, h] = -1000.0
            x[e, h] = 1000.0
    got = geot_b200.segment_softmax(x.to(DEV), index.to(DEV)).cpu()
    exp = torch.empty_like(x)
    for r in rows.tolist():
        a, b = int(rowptr[r]), int(rowptr[r + 1])
        exp[a:b] = torch.softmax(x[a:b], 0)
    assert torch.equal(torch.isnan(got), torch.isnan(exp))
    fin = ~torch.isnan(exp)
    deg = so.degrees(index)
    clean = torch.where(torch.isnan(exp), 0.0, x)
    ref = so.softmax(clean, index)
    tol = so.forward_tolerance(ref, deg, H, torch.float32, clean, index)
    _check(got[fin], exp[fin], tol[fin] + 2.0 ** -24 * ref[fin].abs())       # (+ torch.softmax's own rounding)


# ---- backward -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_backward_vs_fp64(dtype):
    index, g = so.random_graph(30_000, 900, seed=3, hub=9_001)
    E = index.numel()
    deg = so.degrees(index)
    for H in (1, 4, 16):
        src = _src(E, H, g, 10.0, dtype).to(DEV).requires_grad_(True)
        gout = _src(E, H, g, 1.0, dtype)
        out = geot_b200.segment_softmax(src, index.to(DEV))
        out.backward(gout.to(DEV))
        exp, mag, diff = so.softmax_backward(out, gout, index)
        assert src.grad.dtype == dtype and src.grad.shape == src.shape
        _check(src.grad, exp, so.backward_tolerance(exp, out, mag, diff, deg, H, dtype))
        direct = torch.ops.geot.segment_softmax_backward(out.detach(), gout.to(DEV), index.to(DEV))
        assert torch.equal(direct, src.grad)


def test_gradcheck_fp64():
    index = torch.tensor([0, 0, 0, 1, 3, 3, 4, 4, 4, 4, 4, 6], device=DEV)
    g = torch.Generator().manual_seed(1)
    for H in (1, 3):
        x = torch.randn(index.numel(), H, generator=g, dtype=torch.float64).to(DEV).requires_grad_(True)
        src = x.view(-1) if H == 1 else x
        assert torch.autograd.gradcheck(lambda s: geot_b200.segment_softmax(s, index), (src,))


def test_opcheck():
    index, g = so.random_graph(500, 40, seed=2)
    index = index.to(DEV)
    for shape in ((500,), (500, 4)):
        x = torch.randn(*shape, generator=g).to(DEV)
        torch.library.opcheck(torch.ops.geot.segment_softmax.default, (x.requires_grad_(True), index),
                              test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))
        out = geot_b200.segment_softmax(x.detach(), index)
        torch.library.opcheck(torch.ops.geot.segment_softmax_backward.default, (out, torch.randn_like(out), index),
                              test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))


# ---- input handling -----------------------------------------------------------------------------------------------
def test_two_calls_are_bit_identical_and_abi_agrees():
    index, g = so.random_graph(200_000, 3_000, seed=4, hub=70_001)
    index = index.to(DEV)
    for H in (1, 8):
        x = _src(index.numel(), H, g, 10.0, torch.float32).to(DEV)
        a = geot_b200.segment_softmax(x, index)
        b = geot_b200.segment_softmax(x, index)
        assert torch.equal(a, b)
        assert torch.equal(abi.segment_softmax(x, index), a)
        gout = torch.randn_like(x)
        d1 = torch.ops.geot.segment_softmax_backward(a, gout, index)
        d2 = torch.ops.geot.segment_softmax_backward(a, gout, index)
        assert torch.equal(d1, d2)
        assert torch.equal(abi.segment_softmax_backward(a, gout, index), d1)


def test_unsorted_index_is_rejected():
    index = torch.tensor([0, 2, 1, 3], device=DEV)
    x = torch.rand(4, 2, device=DEV)
    with pytest.raises(RuntimeError, match="sorted"):
        geot_b200.segment_softmax(x, index)
    with pytest.raises(RuntimeError, match="sorted"):
        torch.ops.geot.segment_softmax_backward(x, x, index)
    plan = abi.DevicePlan(index)
    with pytest.raises(abi.AbiError, match="invalid argument"):
        abi.segment_softmax(x, index, plan)


def test_bad_operands_are_rejected():
    index = torch.tensor([0, 0, 1], device=DEV)
    with pytest.raises(RuntimeError, match="one row per index entry"):
        geot_b200.segment_softmax(torch.rand(4, 2, device=DEV), index)
    with pytest.raises(RuntimeError, match="unsupported dtype"):
        geot_b200.segment_softmax(torch.ones(3, 2, dtype=torch.int32, device=DEV), index)
    with pytest.raises(RuntimeError, match=r"\[E\] or \[E, H\]"):
        geot_b200.segment_softmax(torch.rand(3, 2, 2, device=DEV), index)
    with pytest.raises(RuntimeError, match="CUDA"):
        torch.ops.geot.segment_softmax(torch.rand(3, 2), index)
    with pytest.raises(RuntimeError, match="same shape"):
        torch.ops.geot.segment_softmax_backward(torch.rand(3, 2, device=DEV), torch.rand(3, 1, device=DEV), index)
    assert geot_b200.segment_softmax(torch.rand(0, 4, device=DEV), index[:0]).shape == (0, 4)


def test_int32_index_matches_int64():
    index, g = so.random_graph(50_000, 800, seed=6, hub=10_000)
    x = _src(index.numel(), 4, g, 10.0, torch.float32).to(DEV)
    a = geot_b200.segment_softmax(x, index.to(DEV))
    b = geot_b200.segment_softmax(x, index.to(DEV).int())
    assert torch.equal(a, b)
    xg = x.clone().requires_grad_(True)
    geot_b200.segment_softmax(xg, index.to(DEV).int()).square().sum().backward()
    xr = x.clone().requires_grad_(True)
    geot_b200.segment_softmax(xr, index.to(DEV)).square().sum().backward()
    assert torch.equal(xg.grad, xr.grad)


# ---- GATConv ------------------------------------------------------------------------------------------------------
def _gat_restated(conv, x, si, di):
    """PyG GATConv math without dropout, in fp64 on plain torch ops."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    h = (x.double() @ conv.lin.weight.double().t()).view(N, H, F)
    a_s = (h * conv.att_src.double()).sum(-1)
    a_d = (h * conv.att_dst.double()).sum(-1)
    logits = torch.nn.functional.leaky_relu(a_s[si] + a_d[di], conv.negative_slope)
    m = torch.full((N, H), float("-inf"), dtype=torch.float64, device=x.device).scatter_reduce(
        0, di.view(-1, 1).expand_as(logits), logits, "amax")
    ex = (logits - m[di]).exp()
    den = torch.zeros(N, H, dtype=torch.float64, device=x.device).index_add(0, di, ex)
    alpha = ex / den[di]
    out = torch.zeros(N, H, F, dtype=torch.float64, device=x.device).index_add(0, di, alpha.unsqueeze(-1) * h[si])
    out = out.reshape(N, H * F) if conv.concat else out.mean(1)
    return out + conv.bias.double() if conv.bias is not None else out


def _gat_graph(N=300, E=4000, seed=8):
    g = torch.Generator().manual_seed(seed)
    si = torch.randint(0, N, (E,), generator=g)
    di = (torch.rand(E, generator=g) ** 2 * (N - 10)).long()     # skewed; the last rows only get their self loop
    si, di, _ = add_self_loops(si.to(DEV), di.to(DEV), N)
    return si, di, g


@pytest.mark.parametrize("concat", [True, False])
def test_gatconv_forward_matches_restatement(concat):
    si, di, g = _gat_graph()
    torch.manual_seed(0)
    conv = GATConv(24, 16, heads=4, concat=concat).to(DEV)
    with torch.no_grad():
        conv.bias.normal_()
    x = torch.randn(300, 24, generator=g).to(DEV)
    got = conv(x, si, di)
    exp = _gat_restated(conv, x, si, di)
    assert got.shape == ((300, 64) if concat else (300, 16))
    _check(got, exp, 2e-5 * exp.abs() + 2e-5)


def test_gatconv_gradients_reach_every_parameter():
    si, di, g = _gat_graph(seed=9)
    torch.manual_seed(1)
    conv = GATConv(24, 16, heads=4).to(DEV)
    x = torch.randn(300, 24, generator=g).to(DEV).requires_grad_(True)
    target = torch.randn(300, 64, generator=g).to(DEV)
    (conv(x, si, di) - target).square().mean().backward()
    params = dict(conv.named_parameters())
    ref = GATConv(24, 16, heads=4).to(DEV).double()
    ref.load_state_dict(conv.state_dict())
    xr = x.detach().double().requires_grad_(True)
    (_gat_restated(ref, xr, si, di) - target.double()).square().mean().backward()
    for name, p in params.items():
        assert p.grad is not None and p.grad.abs().sum().item() > 0, name
        r = dict(ref.named_parameters())[name].grad
        _check(p.grad, r, 1e-4 * r.abs().max() + 1e-7)
    _check(x.grad, xr.grad, 1e-4 * xr.grad.abs().max() + 1e-7)


def test_two_layer_gat_training_matches_restatement():
    N = 300
    si, di, g = _gat_graph(N=N, seed=10)
    x0 = torch.randn(N, 32, generator=g).to(DEV)
    target = torch.randn(N, 8, generator=g).to(DEV)
    torch.manual_seed(2)
    init = [GATConv(32, 16, heads=4).to(DEV), GATConv(64, 8, heads=2, concat=False).to(DEV)]
    for conv in init:
        with torch.no_grad():
            conv.bias.normal_(0, 0.1)

    def run(forward, dtype):
        layers = [GATConv(32, 16, heads=4), GATConv(64, 8, heads=2, concat=False)]
        for layer, src in zip(layers, init):
            layer.to(DEV).to(dtype).load_state_dict(src.state_dict())
        params = [p for layer in layers for p in layer.parameters()]
        opt = torch.optim.SGD(params, lr=0.1)
        losses = []
        for _ in range(5):
            h = torch.nn.functional.elu(forward(layers[0], x0.to(dtype)))
            out = forward(layers[1], h)
            loss = (out - target.to(dtype)).square().mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(loss.detach().double())
        return losses, [p.detach().double() for p in params]

    got_l, got_p = run(lambda conv, x: conv(x, si, di), torch.float32)
    exp_l, exp_p = run(lambda conv, x: _gat_restated(conv, x, si, di), torch.float64)
    for a, b in zip(got_l, exp_l):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-7), (got_l, exp_l)      # fp32 kernels against fp64
    for a, b in zip(got_p, exp_p):
        assert torch.allclose(a, b, rtol=1e-3, atol=1e-5)


# ---- full size ----------------------------------------------------------------------------------------------------
def test_reddit_shape_full_size():
    """Reddit shape, 4 heads, fp32: the constant-logit exact check on every row (the hub included), and sampled rows
    (the hub included) against fp64."""
    import workloads
    G = workloads.power_law_graph("reddit")
    di = G.dst_index
    E, H = di.numel(), 4
    deg = torch.bincount(di)
    rows = deg.numel()
    level = torch.randint(-8, 9, (rows, H), device=DEV, dtype=torch.int32).float()
    got = geot_b200.segment_softmax(level[di], di)
    exp = (1.0 / deg[di].float()).view(E, 1).expand(E, H)
    assert torch.equal(got, exp)
    del got, exp, level
    gen = torch.Generator(device=DEV).manual_seed(0)
    x = torch.rand(E, H, generator=gen, device=DEV) * 20 - 10
    got = geot_b200.segment_softmax(x, di)
    rowptr = torch.cat([torch.zeros(1, dtype=torch.long, device=DEV), deg.cumsum(0)])
    hub = int(torch.argmax(deg))
    sample = torch.cat([torch.randperm(rows, generator=gen, device=DEV)[:200], torch.tensor([hub], device=DEV)])
    for r in sample.tolist():
        a, b = int(rowptr[r]), int(rowptr[r + 1])
        if a == b:
            continue
        exp = torch.softmax(x[a:b].double(), 0)
        d = torch.full((b - a,), b - a, dtype=torch.long)
        idx = torch.zeros(b - a, dtype=torch.long)
        _check(got[a:b], exp, so.forward_tolerance(exp.cpu(), d, H, torch.float32, x[a:b], idx))
