"""fp64 restatement of the fused graph attention (geot_b200/csrc/kernels/attention.cuh) and its gradients, and the error
bounds that follow from the kernels' accumulation order.  Everything runs on the device of the inputs, in fp64."""
import torch


def unit(dtype):
    """Unit roundoff of the accumulator: fp32 for fp32 / bf16 / fp16, fp64 for fp64."""
    return 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24


def out_ulp(dtype):
    """Relative rounding of a store to a 16-bit dtype (0 for fp32 / fp64: the accumulator's own type)."""
    return {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}.get(dtype, 0.0)


def reference(q, k, v, si, di, scale, g=None):
    """fp64 (out, lse) and, with g = d loss / d out, the gradients (grad_q, grad_k, grad_v), by torch autograd of the
    restatement: index_select, a per-row softmax, index_add."""
    N, H, F = q.shape
    qd, kd, vd = (t.detach().double().requires_grad_(g is not None) for t in (q, k, v))
    s = (qd[di] * kd[si]).sum(-1) * scale
    m = torch.full((N, H), float("-inf"), dtype=torch.float64, device=q.device).scatter_reduce(
        0, di.view(-1, 1).expand(-1, H), s, "amax")
    e = (s - m[di]).exp()
    den = torch.zeros(N, H, dtype=torch.float64, device=q.device).index_add(0, di, e)
    out = torch.zeros(N, H, F, dtype=torch.float64, device=q.device).index_add(0, di, (e / den[di]).unsqueeze(-1) * vd[si])
    lse = m + den.log()
    if g is None:
        return out.detach(), lse.detach()
    grads = torch.autograd.grad(out, (qd, kd, vd), g.double())
    return out.detach(), lse.detach(), grads


def bounds(q, k, v, si, di, scale, g=None, out_kernel=None):
    """Bounds on |kernel - fp64| for out and, with g, for (grad_q, grad_k, grad_v).  With u the accumulator's unit
    roundoff and deg the degree of a row:

    * score x = scale <q, k>: a lane adds its columns in sequence, a butterfly of at most 5 levels adds the lanes, then
      the product with scale: |dx| <= (F + 8) u scale sum_f |q k|.
    * Every weight exp(x - M) of a row reaches the final max through at most depth = 2 deg + 10 rescales (the edges of a
      chunk in sequence, then the chunk pieces and the tile chain), each exp(m - M) with 2 u and its product 1 u, and the
      exp argument x - M is rounded (|x - M| u): its relative error is at most
      eta = 2 max_row |dx| + u max_row |x - M| + 3 depth u.  acc and s share the factors of a common max; what differs
      from edge to edge is at most eta, so out = acc / s is off by 2 eta sum alpha |v|, plus depth u sum alpha |v| for the
      additions and 2 u |out| for the division; 16-bit outputs add one rounding.
    * Backward: lse = m + log s carries eta + u |lse| + u; p = exp(x - lse) carries
      eps_p = |dx| + d_lse + u |x - lse| + 2 u.  dp = <g, v[src]> and D = <g, out> carry (F + 8) u sum |g v| and
      (F + 8) u sum |g out| + sum |g| |d_out|, where d_out is the stored out's error (the kernel's out, when given).
      ds = scale p (dp - D) then carries scale p (|dp - D| (eps_p + 3 u) + d_dp + d_D), and p and ds are rounded to the
      dtype before the src-side passes.  grad_q = sum ds k, grad_k = sum ds q[dst], grad_v = sum p g[dst] add those
      per-edge errors times the other factor, and (2 deg + 10) u times the sum of |terms| for their own additions."""
    dt = q.dtype
    u, qo = unit(dt), out_ulp(dt)
    N, H, F = q.shape
    Nk = k.shape[0]
    dev = q.device
    qd, kd, vd = q.double(), k.double(), v.double()
    out, lse = reference(q, k, v, si, di, scale)
    x = (qd[di] * kd[si]).sum(-1) * scale
    dx = (F + 8) * u * scale * (qd[di] * kd[si]).abs().sum(-1)
    deg = torch.bincount(di, minlength=N).double()
    depth = (2 * deg + 10).view(N, 1)
    rowmax = lambda t: torch.zeros(N, H, dtype=torch.float64, device=dev).scatter_reduce(
        0, di.view(-1, 1).expand(-1, H), t, "amax", include_self=True)
    M = torch.full((N, H), float("-inf"), dtype=torch.float64, device=dev).scatter_reduce(
        0, di.view(-1, 1).expand(-1, H), x, "amax")
    eta = 2 * rowmax(dx) + u * rowmax((x - M[di]).abs()) + 3 * depth * u
    alpha = (x - lse[di]).exp()
    mag = torch.zeros(N, H, F, dtype=torch.float64, device=dev).index_add(0, di, alpha.unsqueeze(-1) * vd[si].abs())
    tiny = torch.finfo(dt).tiny
    out_tol = (2 * eta + depth * u).unsqueeze(-1) * mag + 2 * u * out.abs()
    out_tol = out_tol + qo * (out.abs() + out_tol) + tiny
    if g is None:
        return out_tol
    gd = g.double()
    o_used = out_kernel.double() if out_kernel is not None else out
    d_out = (o_used - out).abs() + out_tol
    d_lse = eta + u * lse.abs() + u
    eps_p = dx + d_lse[di] + u * (x - lse[di]).abs() + 2 * u
    dp = (gd[di] * vd[si]).sum(-1)
    D = (gd * out).sum(-1)
    d_dp = (F + 8) * u * (gd[di] * vd[si]).abs().sum(-1)
    d_D = ((F + 8) * u * (gd * out).abs().sum(-1) + (gd.abs() * d_out).sum(-1))[di]
    p = alpha
    ds = scale * p * (dp - D[di])
    d_ds = scale * p * ((dp - D[di]).abs() * (eps_p + 3 * u) + d_dp + d_D) + qo * ds.abs()
    d_p = p * eps_p + qo * p
    degk = torch.bincount(si, minlength=Nk).double().view(Nk, 1, 1)
    sum_dst = lambda t: torch.zeros(N, H, F, dtype=torch.float64, device=dev).index_add(0, di, t)
    sum_src = lambda t: torch.zeros(Nk, H, F, dtype=torch.float64, device=dev).index_add(0, si, t)
    t_q = sum_dst(d_ds.unsqueeze(-1) * kd[si].abs()) + depth.unsqueeze(-1) * u * sum_dst((ds.unsqueeze(-1) * kd[si]).abs())
    t_k = sum_src(d_ds.unsqueeze(-1) * qd[di].abs()) + (2 * degk + 10) * u * sum_src((ds.unsqueeze(-1) * qd[di]).abs())
    t_v = sum_src(d_p.unsqueeze(-1) * gd[di].abs()) + (2 * degk + 10) * u * sum_src((p.unsqueeze(-1) * gd[di]).abs())
    _, _, (eq, ek, ev) = reference(q, k, v, si, di, scale, g)
    fin = lambda t, e: t + qo * (e.abs() + t) + tiny
    return out_tol, (fin(t_q, eq), fin(t_k, ek), fin(t_v, ev))
