"""GPU checks of geot::graph_attention and its backward (geot_b200_graph_attention / geot_b200_graph_attention_grad):
exact on equal-score rows for every dtype and path, against an fp64 restatement within bounds derived from the
accumulation order, gradcheck / opcheck, determinism and input handling; gnn.TransformerConv against an fp64
restatement of PyG's TransformerConv math; and one layer at the full Reddit shape."""
import math

import pytest
import torch

from tests.helpers import attention_oracle as ao
from tests.helpers import softmax_oracle as so
from tests.helpers.kernel_matrix import launched_kernels

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import geot_b200
    from geot_b200.gnn import TransformerConv

DEV = "cuda"
DTYPES = [torch.float32, torch.float64, torch.bfloat16, torch.float16]
ids = lambda v: str(v).replace("torch.", "")
TNAME = {torch.float32: "float", torch.float64: "double", torch.bfloat16: "__nv_bfloat16", torch.float16: "__half"}


def run(q, k, v, si, di, g, scale=None):
    qq, kk, vv = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
    out = geot_b200.graph_attention(qq, kk, vv, si, di, scale)
    out.backward(g)
    return out.detach(), qq.grad, kk.grad, vv.grad


def grid(shape, gen, k, scale, dtype):
    return (torch.randint(-k, k + 1, shape, generator=gen, device=DEV).double() * scale).to(dtype)


# ---- exact: every score of a row is equal ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def exact_graph():
    index, N = so.exact_graph()
    g = torch.Generator().manual_seed(1)
    src = torch.randint(0, N, (index.numel(),), generator=g)
    return src.to(DEV), index.to(DEV), N


def widths(dtype):
    """(F, vector path, vectors per head and lane): whole 16-byte vectors per head; widths that are not (element-wise:
    one lane group of up to 32 lanes, and 33 / 70 (75 for fp64, where 70 is whole vectors) columns over 32 lanes, two and
    three -- run as four -- elements a lane); 64 columns a head, which at H = 8 runs as several launches over disjoint
    heads."""
    full = 128 // torch.finfo(dtype).bits
    wide = 75 if dtype == torch.float64 else 70
    return [(2 * full, True, 1), (5, False, 1), (33, False, 2), (wide, False, 4), (64, True, 1)]


@pytest.mark.parametrize("big", [False, True], ids=["small_scores", "scores_1000"])
@pytest.mark.parametrize("H", [1, 2, 3, 8])
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_exact_on_equal_scores(exact_graph, dtype, H, big):
    """k is one row repeated, so every score of a row is the same value: every exp(x - M) is exp(0) = 1, every rescale
    factor is exactly 1, s is the degree and acc the row sum of v.  With v = j/4 (|j| <= 4) that sum is exact in the
    accumulator (the hub has 80001 edges), so out must equal (fp64 row sum -> accumulator) / deg, rounded once.  With
    scores around +-1000 an implementation that did not subtract the max would overflow exp."""
    si, di, N = exact_graph
    gen = torch.Generator(device=DEV).manual_seed(11 * H + big)
    acc = torch.float64 if dtype == torch.float64 else torch.float32
    deg = torch.bincount(di, minlength=N)
    for F, vector, vph in widths(dtype):
        kr = grid((1, H, F), gen, 4, 0.25, dtype)
        kr[..., 0] = 1.0
        k = kr.expand(N, H, F).contiguous()
        q = grid((N, H, F), gen, 4, 0.25, dtype)
        if big:     # scores of about +-1000: x = <q, k> / sqrt(F) with q[..., 0] = +-1000 sqrt(F) and k[..., 0] = 1
            sign = torch.where(torch.rand(N, H, generator=gen, device=DEV) < 0.5, 1.0, -1.0)
            q[..., 0] = (sign * 1000.0 * math.sqrt(F)).to(dtype)
        v = grid((N, H, F), gen, 4, 0.25, dtype)
        with torch.no_grad():
            (out, lse), names = launched_kernels(lambda: torch.ops.geot.graph_attention(q, k, v, si, di, 1 / math.sqrt(F)))
        vsum = torch.zeros(N, H, F, dtype=torch.float64, device=DEV).index_add(0, di, v.double()[si])
        d = deg.to(acc).view(N, 1, 1)
        exp = torch.where(d > 0, vsum.to(acc) / d.clamp_min(1), 0.0).to(dtype)
        assert torch.equal(out, exp), (F, float((out.double() - exp.double()).abs().max()))
        assert torch.isfinite(lse[deg > 0]).all() and (lse[deg == 0] == float("-inf")).all()
        if big:
            assert lse[deg > 0].abs().max() > 500
        t = TNAME[dtype]
        full = 16 // out.element_size()
        fwd = [n for n in names if "attention_fwd_kernel<" in n]
        assert fwd and all(("<%s, %d," % (t, full if vector else 1)) in n for n in fwd), (F, fwd)
        assert all((", %d>" % vph) in n for n in fwd), (F, vph, fwd)
        assert any("attention_fixup_kernel" in n for n in names)
        assert not [n for n in names if "sddmm" in n or "softmax" in n or "segment_reduce" in n], names


def test_multi_launch_shape_runs_several_launches(exact_graph):
    """8 heads of 64 fp32 columns: 4 heads (256 columns) a launch, so two forward launches and two backward launches."""
    si, di, N = exact_graph
    q, k, v = (torch.randn(N, 8, 64, device=DEV) * 0.3 for _ in range(3))
    g = torch.randn(N, 8, 64, device=DEV)
    res, names = launched_kernels(lambda: run(q, k, v, si, di, g))
    assert len([n for n in names if "attention_fwd_kernel<float, 4," in n]) == 2, names
    assert len([n for n in names if "attention_grad_kernel<float, 4," in n]) == 2, names
    assert any("gatv2_fixup_kernel<float>" in n for n in names)
    out_tol, (tq, tk, tv) = ao.bounds(q, k, v, si, di, 1 / 8, g, res[0])
    eo, _, (eq, ek, ev) = ao.reference(q, k, v, si, di, 1 / 8, g)
    assert ((res[0].double() - eo).abs() <= out_tol).all()
    for got, exp, tol in zip(res[1:], (eq, ek, ev), (tq, tk, tv)):
        assert ((got.double() - exp).abs() <= tol).all()


# ---- random inputs against fp64 --------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=ids)
def test_random_inputs_vs_fp64(dtype):
    """Forward and all three gradients within the bounds of attention_oracle.bounds (derived there from the kernels'
    accumulation order), on a skewed graph with a hub row cut by many tiles."""
    index, gen = so.random_graph(40_000, 1_500, seed=3, hub=9_001)
    di = index.to(DEV)
    E, N = di.numel(), 1_500
    si = torch.randint(0, N, (E,), generator=gen).to(DEV)
    wide = 75 if dtype == torch.float64 else 70
    for H, F in ((1, 32), (4, 16), (3, 7), (2, 136), (2, 33), (2, wide)):
        if dtype == torch.float64 and F > 128:
            continue
        q, k, v = ((torch.randn(N, H, F, device=DEV, dtype=torch.float64) * 0.5).to(dtype) for _ in range(3))
        g = torch.randn(N, H, F, device=DEV, dtype=torch.float64).to(dtype)
        scale = 1 / math.sqrt(F)
        out, gq, gk, gv = run(q, k, v, si, di, g)
        out_tol, (tq, tk, tv) = ao.bounds(q, k, v, si, di, scale, g, out)
        eo, _, (eq, ek, ev) = ao.reference(q, k, v, si, di, scale, g)
        assert ((out.double() - eo).abs() <= out_tol).all(), (H, F, "out")
        for name, got, exp, tol in (("grad_q", gq, eq, tq), ("grad_k", gk, ek, tk), ("grad_v", gv, ev, tv)):
            assert ((got.double() - exp).abs() <= tol).all(), (H, F, name, float(((got.double() - exp).abs() / tol).max()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16], ids=ids)
def test_one_column_heads_fill_the_shared_memory(dtype):
    """F = 1: one launch holds 256 heads (128 for fp64), whose forward pieces take 48 KB of dynamic shared memory -- more
    than a kernel gets without the opt-in once its static shared memory is added.  Forward and gradients against fp64."""
    index, gen = so.random_graph(20_000, 600, seed=6, hub=3_001)
    di = index.to(DEV)
    E, N = di.numel(), 600
    si = torch.randint(0, N, (E,), generator=gen).to(DEV)
    H = 128 if dtype == torch.float64 else 256
    q, k, v = ((torch.randn(N, H, 1, device=DEV, dtype=torch.float64) * 0.5).to(dtype) for _ in range(3))
    g = torch.randn(N, H, 1, device=DEV, dtype=torch.float64).to(dtype)
    res, names = launched_kernels(lambda: run(q, k, v, si, di, g))
    assert len([n for n in names if "attention_fwd_kernel<" in n]) == 1, names
    out_tol, (tq, tk, tv) = ao.bounds(q, k, v, si, di, 1.0, g, res[0])
    eo, _, (eq, ek, ev) = ao.reference(q, k, v, si, di, 1.0, g)
    assert ((res[0].double() - eo).abs() <= out_tol).all()
    for got, exp, tol in zip(res[1:], (eq, ek, ev), (tq, tk, tv)):
        assert ((got.double() - exp).abs() <= tol).all()


# ---- autograd, operator checks, determinism, input handling ----------------------------------------------------------
def small_graph(E=3000, N=200, seed=0):
    g = torch.Generator().manual_seed(seed)
    di = torch.randint(0, N - 3, (E,), generator=g).sort().values
    si = torch.randint(0, N, (E,), generator=g)
    return si.to(DEV), di.to(DEV), N


def test_gradcheck_fp64():
    si, di, N = small_graph(300, 40)
    q, k, v = (torch.randn(N, 2, 3, device=DEV, dtype=torch.float64, requires_grad=True) for _ in range(3))
    assert torch.autograd.gradcheck(lambda a, b, c: geot_b200.graph_attention(a, b, c, si, di), (q, k, v))


def test_opcheck():
    si, di, N = small_graph()
    q, k, v = (torch.randn(N, 4, 8, device=DEV, requires_grad=True) for _ in range(3))
    torch.library.opcheck(torch.ops.geot.graph_attention.default, (q, k, v, si, di, 0.35),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    out, lse = torch.ops.geot.graph_attention(q, k, v, si, di, 0.35)
    g = torch.randn_like(out)
    torch.library.opcheck(torch.ops.geot.graph_attention_backward.default,
                          (g, q.detach(), k.detach(), v.detach(), out.detach(), lse, si, di, 0.35),
                          test_utils=("test_schema", "test_faketensor"))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=ids)
def test_repeats_are_bit_identical_and_int32_matches(dtype):
    si, di, N = small_graph(50_000, 3_000, seed=4)
    q, k, v = (torch.randn(N, 8, 32, device=DEV).to(dtype) for _ in range(3))
    g = torch.randn(N, 8, 32, device=DEV).to(dtype)
    a = run(q, k, v, si, di, g)
    b = run(q, k, v, si, di, g)
    c = run(q, k, v, si.int(), di.int(), g)
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z)


def test_unsorted_index_refused_and_rows_without_edges_are_zero():
    si, di, N = small_graph()
    x = torch.randn(N, 2, 8, device=DEV)
    with pytest.raises(RuntimeError, match="sorted"):
        geot_b200.graph_attention(x, x, x, si, di.flip(0))
    with pytest.raises(RuntimeError, match="rows"):
        geot_b200.graph_attention(x[: int(di[-1])], x, x, si, di)
    q = x.clone().requires_grad_(True)
    out = geot_b200.graph_attention(q, x, x, si, di)
    out.sum().backward()
    last = int(di[-1])
    assert out.shape == x.shape and torch.equal(out[last + 1:], torch.zeros_like(out[last + 1:]))
    assert torch.equal(q.grad[last + 1:], torch.zeros_like(q.grad[last + 1:]))
    empty = geot_b200.graph_attention(x, x, x, si[:0], di[:0])
    assert torch.equal(empty, torch.zeros_like(x))


def test_nan_in_q_makes_its_row_nan():
    si, di, N = small_graph()
    q, k, v = (torch.randn(N, 2, 8, device=DEV) for _ in range(3))
    r = int(di[len(di) // 2])
    q[r, 1, 3] = float("nan")
    out = geot_b200.graph_attention(q, k, v, si, di)
    assert torch.isnan(out[r, 1]).all() and not torch.isnan(out[r, 0]).any()
    others = torch.ones(N, dtype=torch.bool, device=DEV)
    others[r] = False
    assert not torch.isnan(out[others]).any()


# ---- TransformerConv -------------------------------------------------------------------------------------------------
def restated_conv(conv, x, si, di):
    """fp64 restatement of PyG's TransformerConv math (no beta, edge features or dropout) in torch ops."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    W = lambda t: None if t is None else t.double()
    lin = lambda m: torch.nn.functional.linear(x, W(m.weight), W(m.bias))
    q, k, v = lin(conv.lin_query).view(N, H, F), lin(conv.lin_key).view(N, H, F), lin(conv.lin_value).view(N, H, F)
    s = (q[di] * k[si]).sum(-1) / math.sqrt(F)
    m = torch.full((N, H), -math.inf, dtype=torch.float64, device=DEV).scatter_reduce(0, di.view(-1, 1).expand(-1, H), s, "amax")
    e = (s - m[di]).exp()
    den = torch.zeros(N, H, dtype=torch.float64, device=DEV).index_add(0, di, e)
    out = torch.zeros(N, H, F, dtype=torch.float64, device=DEV).index_add(0, di, (e / den[di]).unsqueeze(-1) * v[si])
    out = out.reshape(N, H * F) if conv.concat else out.mean(1)
    return out + lin(conv.lin_skip) if conv.lin_skip is not None else out


@pytest.mark.parametrize("root_weight", [True, False])
@pytest.mark.parametrize("concat", [True, False])
def test_transformerconv_forward_and_gradients_vs_fp64(concat, root_weight):
    torch.manual_seed(0)
    si, di, N = small_graph(4000, 300, seed=2)
    conv = TransformerConv(16, 8, heads=4, concat=concat, root_weight=root_weight).to(DEV)
    x = torch.randn(N, 16, device=DEV)
    out = conv(x, si, di)
    ref = restated_conv(conv, x.double(), si, di)
    assert torch.allclose(out.double(), ref, rtol=1e-4, atol=1e-5)
    gout = torch.randn_like(out)
    out.backward(gout)
    params = list(conv.parameters())
    got = [p.grad.clone() for p in params]
    conv.zero_grad()
    ref_grads = torch.autograd.grad(restated_conv(conv, x.double(), si, di), params, gout.double())
    for a, b in zip(got, ref_grads):
        assert torch.allclose(a.double(), b.double(), rtol=1e-3, atol=1e-5), float((a.double() - b.double()).abs().max())


def test_two_layer_training_loop_matches_restatement():
    torch.manual_seed(1)
    si, di, N = small_graph(6000, 400, seed=5)
    x = torch.randn(N, 12, device=DEV)
    y = torch.randint(0, 5, (N,), device=DEV)
    convs = [TransformerConv(12, 8, heads=2).to(DEV), TransformerConv(16, 5, heads=1).to(DEV)]
    ref = [TransformerConv(12, 8, heads=2).to(DEV).double(), TransformerConv(16, 5, heads=1).to(DEV).double()]
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
    """One attention layer (4 x 32, fp32) forward and backward on the Reddit-shape graph.  The forward's peak allocation
    stays below its outputs + workspace + one [E, H] tensor: no score or alpha is materialised.  Sampled rows of out
    (the hub included) against fp64 within attention_oracle.bounds."""
    import workloads
    G = workloads.power_law_graph("reddit")
    si, di = G.src_index, G.dst_index
    E = di.numel()
    N = int(max(int(si.max()), int(di.max()))) + 1
    H, F = 4, 32
    gen = torch.Generator(device=DEV).manual_seed(0)
    q, k, v = (torch.randn(N, H, F, device=DEV, generator=gen).requires_grad_(True) for _ in range(3))
    g = torch.randn(N, H, F, device=DEV, generator=gen)
    with torch.no_grad():
        torch.ops.geot.graph_attention(q, k, v, si, di, 1 / math.sqrt(F))      # the plan is cached from here on
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = geot_b200.graph_attention(q, k, v, si, di)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    from geot_b200 import abi
    ws = abi.lib().geot_b200_graph_attention_workspace_bytes(E, H, F, abi.F32)
    allowed = N * H * F * 4 + N * H * 4 + ws + E * H * 4
    print("reddit graph_attention fwd: E=%d peak %.3f GB (outputs + workspace %.3f GB, one [E, H] fp32 %.2f GB)"
          % (E, peak / 1e9, (N * H * F * 4 + N * H * 4 + ws) / 1e9, E * H * 4 / 1e9))
    assert peak < allowed
    out.backward(g)
    torch.cuda.synchronize()
    assert all(torch.isfinite(t.grad).all() for t in (q, k, v))
    deg = torch.bincount(di, minlength=N)
    hub = int(torch.argmax(deg))
    rows = torch.cat([torch.randperm(N, generator=gen, device=DEV)[:64], torch.tensor([hub], device=DEV)]).unique()
    sel = torch.isin(di, rows)
    ssi, sdi = si[sel], di[sel]
    tol = ao.bounds(q.detach(), k.detach(), v.detach(), ssi, sdi, 1 / math.sqrt(F))
    exp, _ = ao.reference(q.detach(), k.detach(), v.detach(), ssi, sdi, 1 / math.sqrt(F))
    assert ((out.detach()[rows].double() - exp[rows]).abs() <= tol[rows]).all()
