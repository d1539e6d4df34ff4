"""GPU checks of geot::gatv2_score and its backward (geot_b200_gatv2_score / geot_b200_gatv2_grad): exact on a dyadic
grid for every dtype and path, against an fp64 restatement within bounds derived from the accumulation order,
gradcheck / opcheck, determinism and input handling; gnn.GATv2Conv against an fp64 restatement of PyG's GATv2Conv math;
and one layer at the full Reddit shape."""
import math

import pytest
import torch

from tests.helpers import softmax_oracle as so
from tests.helpers.kernel_matrix import launched_kernels

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import geot_b200
    from geot_b200.gnn import GATv2Conv, add_self_loops

DEV = "cuda"
DTYPES = [torch.float32, torch.float64, torch.bfloat16, torch.float16]
ids = lambda v: str(v).replace("torch.", "")
TNAME = {torch.float32: "float", torch.float64: "double", torch.bfloat16: "__nv_bfloat16", torch.float16: "__half"}


def leaky(u, slope):
    return torch.where(u > 0, u, u * slope)


def restated_score(x_l, x_r, att, si, di, slope):
    """The score in torch ops (materialises [E, H, F])."""
    return (att.view(1, *att.shape[-2:]) * leaky(x_l[si] + x_r[di], slope)).sum(-1)


def reference(x_l, x_r, att, si, di, g, slope):
    """fp64 score and gradients (torch autograd of the restatement, on the GPU)."""
    xl = x_l.double().detach().requires_grad_(True)
    xr = x_r.double().detach().requires_grad_(True)
    a = att.double().detach().requires_grad_(True)
    s = restated_score(xl, xr, a, si, di, slope)
    gl, gr, ga = torch.autograd.grad(s, (xl, xr, a), g.double())
    return s.detach(), gl, gr, ga


def run(x_l, x_r, att, si, di, g, slope):
    xl, xr, a = (t.detach().clone().requires_grad_(True) for t in (x_l, x_r, att))
    s = geot_b200.gatv2_score(xl, xr, a, si, di, slope)
    s.backward(g)
    return s.detach(), xl.grad, xr.grad, a.grad


def grid(shape, gen, k, scale, dtype):
    return (torch.randint(-k, k + 1, shape, generator=gen, device=DEV).double() * scale).to(dtype)


# ---- exact: every partial sum is exact in the accumulator -----------------------------------------------------------
@pytest.fixture(scope="module")
def exact_graph():
    index, N = so.exact_graph()
    g = torch.Generator().manual_seed(1)
    src = torch.randint(0, N, (index.numel(),), generator=g)
    return src.to(DEV), index.to(DEV), N


def widths(dtype):
    """(F, vector path): whole 16-byte vectors per head; a width that is not one; a row of several column slabs."""
    full = 128 // torch.finfo(dtype).bits
    return [(2 * full, True), (5, False), (136, True)]


@pytest.mark.parametrize("H", [1, 2, 3, 8])
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_exact_on_a_dyadic_grid(exact_graph, dtype, H):
    """x = k/4 (|k| <= 4), att = j/4 (|j| <= 4), g = m/4 (|m| <= 4), slope 1/4: every product and partial sum of the
    score, of both node gradients (the hub has 80001 edges) and of grad_att is exact in fp32, so the kernels must
    equal the fp64 result rounded once.  Runs the vector, element-wise and wide / multi-slab paths."""
    si, di, N = exact_graph
    E = di.numel()
    gen = torch.Generator(device=DEV).manual_seed(7 * H)
    for F, vector in widths(dtype):
        if H * F > 600:
            continue
        x_l = grid((N, H, F), gen, 4, 0.25, dtype)
        x_r = grid((N, H, F), gen, 4, 0.25, dtype)
        att = grid((H, F), gen, 4, 0.25, dtype)
        g = grid((E, H), gen, 4, 0.25, dtype)
        (s, gl, gr, ga), names = launched_kernels(lambda: run(x_l, x_r, att, si, di, g, 0.25))
        es, egl, egr, ega = reference(x_l, x_r, att, si, di, g, 0.25)
        assert torch.equal(s, es.to(dtype)), (F, "score")
        assert torch.equal(gr, egr.to(dtype)), (F, "grad_x_r")
        assert torch.equal(gl, egl.to(dtype)), (F, "grad_x_l")
        assert torch.equal(ga, ega.to(dtype)), (F, "grad_att")
        # which kernels ran
        t = TNAME[dtype]
        full = 16 // s.element_size()
        grad_k = [n for n in names if "gatv2_grad_kernel<" in n]
        assert grad_k and all(("<%s, %d," % (t, full if vector else 1)) in n for n in grad_k), (F, grad_k)
        assert any("gatv2_fixup_kernel" in n for n in names) and any("gatv2_att_kernel" in n for n in names)
        score_k = [n for n in names if "sddmm_coo" in n and "Gatv2ScoreParams" in n]
        assert len(score_k) == 1, names
        hv = F // full
        lanes = vector and (H == 1 or (hv & (hv - 1)) == 0)
        if lanes:
            assert ("geot::sddmm_coo_kernel<%s, %d," % (t, full)) in score_k[0], score_k
        elif H == 1:
            assert ("geot::sddmm_coo_kernel<%s, 1," % t) in score_k[0], score_k
        else:
            assert "sddmm_coo_wide_kernel" in score_k[0], score_k


# ---- against fp64 at slope 0.2 ---------------------------------------------------------------------------------------
def unit(dtype):
    return 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24


def out_ulp(dtype):
    return {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}.get(dtype, 0.0)


@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_random_inputs_vs_fp64(dtype):
    """Error bounds from the accumulation order.  Score: a lane adds its columns of a head in sequence, a butterfly of
    at most 5 levels adds the lanes, so at most F + 5 additions; each term att * leaky(fl(a + b)) carries 2 u.  Node
    gradients: the edges of a row are added in sequence inside a chunk, the pieces of the row in chunk then tile order:
    at most 2 deg + 2 additions, then the product with att (1 u) and the rounding to the dtype.  grad_att: C <= 256
    edges of a chunk, 8 warps, at most ceil(tiles / 256 / 8) + 8 per slice and 32 + 8 over the slices."""
    index, gen = so.random_graph(40_000, 1_500, seed=3, hub=9_001)
    di = index.to(DEV)
    E, N = di.numel(), 1_500
    si = torch.randint(0, N, (E,), generator=gen).to(DEV)
    deg = torch.bincount(di, minlength=N).double()
    for H, F in ((1, 32), (4, 16), (3, 7)):
        x_l = (torch.randn(N, H, F, device=DEV, dtype=torch.float64)).to(dtype)
        x_r = (torch.randn(N, H, F, device=DEV, dtype=torch.float64)).to(dtype)
        att = (torch.randn(H, F, device=DEV, dtype=torch.float64)).to(dtype)
        g = (torch.randn(E, H, device=DEV, dtype=torch.float64)).to(dtype)
        s, gl, gr, ga = run(x_l, x_r, att, si, di, g, 0.2)
        es, egl, egr, ega = reference(x_l, x_r, att, si, di, g, 0.2)
        u, q = unit(dtype), out_ulp(dtype)
        xa = (x_l.double()[si].abs() + x_r.double()[di].abs())
        mag = (att.double().abs().view(1, H, F) * xa).sum(-1)
        # (16-bit outputs: the rounding to the dtype on top, relative to the accumulator's value)
        assert ((s.double() - es).abs() <= (1 + q) * (F + 8) * u * mag + q * es.abs() + torch.finfo(dtype).tiny).all()
        # node gradients: |g| summed over the row, times |att|
        for got, exp, row, other in ((gr, egr, di, N), (gl, egl, si, N)):
            m = torch.zeros(other, H, dtype=torch.float64, device=DEV).index_add_(0, row, g.double().abs())
            d = torch.bincount(row, minlength=other).double().view(-1, 1, 1)
            tol = ((1 + q) * (2 * d + 6) * u * m.unsqueeze(-1) * att.double().abs() + q * exp.abs() + torch.finfo(dtype).tiny)
            assert ((got.double() - exp).abs() <= tol).all()
        tiles = math.ceil(E / (8 * 32))
        depth = 256 + 8 + math.ceil(tiles / 256 / 8) + 8 + 32 + 8
        term = (g.double().abs().unsqueeze(-1) * xa).sum(0)
        assert ((ga.double() - ega).abs() <= (1 + q) * (depth + 4) * u * term + q * ega.abs() + torch.finfo(dtype).tiny).all()


# ---- autograd, operator checks, determinism, input handling ----------------------------------------------------------
def small_graph(E=3000, N=200, seed=0):
    g = torch.Generator().manual_seed(seed)
    di = torch.randint(0, N - 3, (E,), generator=g).sort().values
    si = torch.randint(0, N, (E,), generator=g)
    return si.to(DEV), di.to(DEV), N


def test_gradcheck_fp64():
    si, di, N = small_graph(300, 40)
    x_l = torch.randn(N, 2, 3, device=DEV, dtype=torch.float64, requires_grad=True)
    x_r = torch.randn(N, 2, 3, device=DEV, dtype=torch.float64, requires_grad=True)
    att = torch.randn(2, 3, device=DEV, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda a, b, c: geot_b200.gatv2_score(a, b, c, si, di, 0.2), (x_l, x_r, att))


def test_opcheck():
    si, di, N = small_graph()
    x_l = torch.randn(N, 4, 8, device=DEV, requires_grad=True)
    x_r = torch.randn(N, 4, 8, device=DEV, requires_grad=True)
    att = torch.randn(4, 8, device=DEV, requires_grad=True)
    torch.library.opcheck(torch.ops.geot.gatv2_score.default, (x_l, x_r, att, si, di, 0.2),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=ids)
def test_repeats_are_bit_identical_and_int32_matches(dtype):
    si, di, N = small_graph(50_000, 3_000, seed=4)
    x_l = torch.randn(N, 8, 32, device=DEV).to(dtype)
    x_r = torch.randn(N, 8, 32, device=DEV).to(dtype)
    att = torch.randn(8, 32, device=DEV).to(dtype)
    g = torch.randn(di.numel(), 8, device=DEV).to(dtype)
    a = run(x_l, x_r, att, si, di, g, 0.2)
    b = run(x_l, x_r, att, si, di, g, 0.2)
    c = run(x_l, x_r, att, si.int(), di.int(), g, 0.2)
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z)


def test_unsorted_index_refused_and_rows_beyond_the_last_index_are_zero():
    si, di, N = small_graph()
    x = torch.randn(N, 2, 8, device=DEV)
    att = torch.randn(2, 8, device=DEV)
    with pytest.raises(RuntimeError, match="sorted"):
        geot_b200.gatv2_score(x, x, att, si, di.flip(0))
    x_l, x_r = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    geot_b200.gatv2_score(x_l, x_r, att, si, di).sum().backward()
    last_dst, last_src = int(di[-1]), int(si.max())
    assert x_r.grad.shape == x.shape and torch.equal(x_r.grad[last_dst + 1:], torch.zeros_like(x_r.grad[last_dst + 1:]))
    assert torch.equal(x_l.grad[last_src + 1:], torch.zeros_like(x_l.grad[last_src + 1:]))
    empty = geot_b200.gatv2_score(x, x, att, si[:0], di[:0])
    assert empty.shape == (0, 2)


# ---- GATv2Conv ----------------------------------------------------------------------------------------------------
def restated_conv(conv, x, si, di):
    """fp64 restatement of the same layer in torch ops."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    W = lambda t: None if t is None else t.double()
    xl = torch.nn.functional.linear(x, W(conv.lin_l.weight), W(conv.lin_l.bias)).view(N, H, F)
    xr = torch.nn.functional.linear(x, W(conv.lin_r.weight), W(conv.lin_r.bias)).view(N, H, F)
    s = restated_score(xl, xr, conv.att.double(), si, di, conv.negative_slope)
    m = torch.full((N, H), -math.inf, dtype=torch.float64, device=DEV).scatter_reduce(0, di.view(-1, 1).expand(-1, H), s, "amax")
    e = (s - m[di]).exp()
    den = torch.zeros(N, H, dtype=torch.float64, device=DEV).index_add(0, di, e)
    alpha = e / den[di]
    out = torch.zeros(N, H, F, dtype=torch.float64, device=DEV).index_add(0, di, alpha.unsqueeze(-1) * xl[si])
    out = out.reshape(N, H * F) if conv.concat else out.mean(1)
    return out + conv.bias.double() if conv.bias is not None else out


@pytest.mark.parametrize("concat", [True, False])
def test_gatv2conv_forward_and_gradients_vs_fp64(concat):
    torch.manual_seed(0)
    si, di, N = small_graph(4000, 300, seed=2)
    si, di, _ = add_self_loops(si, di, N)
    conv = GATv2Conv(16, 8, heads=4, concat=concat).to(DEV)
    with torch.no_grad():
        conv.bias.uniform_(-0.1, 0.1)
    x = torch.randn(N, 16, device=DEV)
    out = conv(x, si, di)
    ref = restated_conv(conv, x.double(), si, di)
    assert torch.allclose(out.double(), ref, rtol=1e-4, atol=1e-5)
    gout = torch.randn_like(out)
    out.backward(gout)
    params = [conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight, conv.lin_r.bias, conv.att, conv.bias]
    got = [p.grad.clone() for p in params]
    conv.zero_grad()
    ref_grads = torch.autograd.grad(restated_conv(conv, x.double(), si, di), params, gout.double())
    for a, b in zip(got, ref_grads):
        assert torch.allclose(a.double(), b.double(), rtol=1e-3, atol=1e-5), float((a.double() - b.double()).abs().max())


def test_two_layer_training_loop_matches_restatement():
    torch.manual_seed(1)
    si, di, N = small_graph(6000, 400, seed=5)
    si, di, _ = add_self_loops(si, di, N)
    x = torch.randn(N, 12, device=DEV)
    y = torch.randint(0, 5, (N,), device=DEV)
    convs = [GATv2Conv(12, 8, heads=2).to(DEV), GATv2Conv(16, 5, heads=1).to(DEV)]
    ref = [GATv2Conv(12, 8, heads=2).to(DEV).double(), GATv2Conv(16, 5, heads=1).to(DEV).double()]
    for c, r in zip(convs, ref):
        r.load_state_dict({k: v.double() for k, v in c.state_dict().items()})
    opt = torch.optim.SGD([p for c in convs for p in c.parameters()], lr=0.1)
    opt_r = torch.optim.SGD([p for c in ref for p in c.parameters()], lr=0.1)
    for step in range(5):
        h = torch.relu(convs[0](x, si, di))
        loss = torch.nn.functional.cross_entropy(convs[1](h, si, di), y)
        hr = torch.relu(restated_conv(ref[0], x.double(), si, di))
        loss_r = torch.nn.functional.cross_entropy(restated_conv(ref[1], hr, si, di), y)
        assert abs(float(loss) - float(loss_r)) <= 1e-4 * max(1.0, abs(float(loss_r))), (step, float(loss), float(loss_r))
        opt.zero_grad(); loss.backward(); opt.step()
        opt_r.zero_grad(); loss_r.backward(); opt_r.step()


# ---- the Reddit shape at full size -----------------------------------------------------------------------------------
def test_reddit_shape_full_size():
    """One GATv2Conv layer (602 -> 4 x 32, fp32), forward and backward, on the Reddit-shape graph: one [E, H*F] fp32
    tensor would be E * 128 * 4 bytes; the peak stays far below it.  Sampled rows of grad_x_r and grad_x_l (the hub
    included) against an fp64 restatement of those rows only."""
    import workloads
    G = workloads.power_law_graph("reddit")
    si, di = G.src_index, G.dst_index
    E = di.numel()
    N = int(max(int(si.max()), int(di.max()))) + 1
    H, F = 4, 32
    gen = torch.Generator(device=DEV).manual_seed(0)
    x_l = torch.randn(N, H, F, device=DEV, generator=gen).requires_grad_(True)
    x_r = torch.randn(N, H, F, device=DEV, generator=gen).requires_grad_(True)
    att = torch.randn(H, F, device=DEV, generator=gen).requires_grad_(True)
    g = torch.randn(E, H, device=DEV, generator=gen)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s = geot_b200.gatv2_score(x_l, x_r, att, si, di, 0.2)
    s.backward(g)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    one = E * H * F * 4
    print("reddit gatv2 score fwd+bwd: E=%d peak above inputs %.2f GB, one [E, H*F] fp32 tensor %.1f GB"
          % (E, peak / 1e9, one / 1e9))
    assert peak < one / 3
    deg_d = torch.bincount(di, minlength=N)
    hub = int(torch.argmax(deg_d))
    rows = torch.cat([torch.randperm(N, generator=gen, device=DEV)[:64], torch.tensor([hub], device=DEV)])
    for which, row_idx, gat_idx, x_row, x_gat, got in (("x_r", di, si, x_r, x_l, x_r.grad), ("x_l", si, di, x_l, x_r, x_l.grad)):
        for r in rows.tolist():
            e = (row_idx == r).nonzero().view(-1)
            u = x_row.detach()[r].double().unsqueeze(0) + x_gat.detach()[gat_idx[e]].double()
            gg = g[e].double().unsqueeze(-1)
            exp = att.detach().double() * (gg * torch.where(u > 0, 1.0, 0.2)).sum(0)
            mag = att.detach().double().abs() * gg.abs().sum(0)
            tol = (2 * e.numel() + 6) * 2.0 ** -24 * mag + 1e-30
            assert ((got[r].double() - exp).abs() <= tol).all(), (which, r, e.numel())
