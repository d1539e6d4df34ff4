"""``geot.mh_spmm`` / ``mh_spmm_transposed`` (reference: ``geot/mh_spmm.py:4-12``).

``geot::mh_spmm`` is a C++ operator; its backward is registered on the operator itself, so ``mh_spmm``,
``mh_spmm_transposed`` (through the differentiable transpose of the weights) and FX-rewritten graphs
(``match_replace.py``) all get gradients.  For ``reduce="sum"``:

* src: the forward kernel on the transposed (src-sorted) edge list, cached per graph
  (``transpose.py``), with the weights carried into that edge order by ``geot_b200_permute_edges``;
* weight: the multi-head SDDMM ``dweight[e, h] = <grad[dst[e], h, :], src[src[e], h, :]>`` in the
  original edge order, returned in the caller's weight layout.

``mean`` scales the gradient rows by ``1 / deg(row)`` and then does the same.  ``max`` / ``min`` / ``prod``
have no backward: it needs the arg-indices of the forward, which the kernels do not produce.
"""
import torch


def mh_spmm(src_index: torch.Tensor, dst_index: torch.Tensor, weight: torch.Tensor, src: torch.Tensor,
            reduce: str = "sum") -> torch.Tensor:
    """``out[dst[e], h, :] (reduce)= weight[e, h] * src[src[e], h, :]``; src ``[N, H, F]``.

    ``weight`` is ``[E, H]`` or ``[H, E]``; the layout is read from the shape, ``[E, H]`` first
    (``csrc/cuda/wrapper/mh_spmm_base.h:38-49``).  fp32 / fp64 / bf16 / fp16 (fp32 accumulation).
    Differentiable in ``weight`` and ``src`` for ``sum`` and ``mean``.
    """
    return torch.ops.geot.mh_spmm(src_index, dst_index, weight, src, reduce)


def mh_spmm_transposed(src_index: torch.Tensor, dst_index: torch.Tensor, weight: torch.Tensor,
                       src: torch.Tensor, reduce: str = "sum") -> torch.Tensor:
    """Takes ``weight [E, H]`` and runs the ``[H, E]`` layout, like the reference
    (``geot/mh_spmm.py:8-12``)."""
    weight = weight.transpose(0, 1).contiguous()
    return torch.ops.geot.mh_spmm(src_index, dst_index, weight, src, reduce)


def src_side_spmm(src_index: torch.Tensor, dst_index: torch.Tensor, weight: torch.Tensor, x: torch.Tensor,
                  n_rows: int, head_major: bool = False) -> torch.Tensor:
    """``out[j, h, :] = sum_{e : src_index[e] = j} weight[e, h] * x[dst_index[e], h, :]``, ``[n_rows, H, F]``: the
    forward kernel on the cached transposed (src-sorted) edge list, with the weights (``[E, H]``, or ``[H, E]`` with
    ``head_major``) carried into that edge order by ``geot_b200_permute_edges``.  Rows past the largest src index are
    zero.  The src-side gradients of ``mh_spmm`` and of ``graph_attention``."""
    from . import abi
    from .transpose import transposed_edges
    t = transposed_edges(src_index, dst_index)
    w = weight.contiguous()
    with torch.cuda.device(w.device):
        if head_major:
            w_perm = torch.empty_like(w)
            for h in range(w.shape[0]):
                abi.permute_edges(w[h], t.perm, out=w_perm[h])
        else:
            w_perm = abi.permute_edges(w, t.perm)
    g = torch.ops.geot.mh_spmm(t.src_index, t.dst_index, w_perm, x, "sum")
    if g.shape[0] < n_rows:      # trailing src rows that no edge reads
        g = torch.cat([g, g.new_zeros((n_rows - g.shape[0],) + tuple(g.shape[1:]))], 0)
    return g


def _setup_context(ctx, inputs, output):
    src_index, dst_index, weight, src, reduce = inputs
    ctx.save_for_backward(src_index, dst_index, weight, src)
    ctx.reduce = reduce


def _backward(ctx, grad):
    src_index, dst_index, weight, src = ctx.saved_tensors
    if ctx.reduce not in ("sum", "mean"):
        raise NotImplementedError("geot.mh_spmm: no backward for reduce=%r (sum and mean only: the others need the "
                                  "arg-indices of the forward)" % ctx.reduce)
    E, H = src_index.numel(), src.shape[1]
    head_major = not (weight.shape[0] == E and weight.shape[1] == H)      # the forward's rule, [E, H] first
    grad = grad.contiguous()
    if ctx.reduce == "mean":
        deg = torch.ops.geot.format_preprocess(dst_index)[0].diff()        # cached plan; rows with no edges get 0
        acc = torch.float64 if grad.dtype == torch.float64 else torch.float32
        scale = torch.where(deg > 0, 1.0 / deg.clamp_min(1).to(acc), 0.0)
        grad = (grad * scale.view(-1, 1, 1)).to(grad.dtype)
    weight_grad = src_grad = None
    if ctx.needs_input_grad[3]:
        src_grad = src_side_spmm(src_index, dst_index, weight, grad, src.shape[0], head_major)
    if ctx.needs_input_grad[2]:
        # dst-sorted edge order: the kernel keeps the grad row in registers across a segment
        weight_grad = torch.ops.geot.sddmm_mh_impl(src_index, dst_index, grad, src, head_major)
    return None, None, weight_grad, src_grad, None


torch.library.register_autograd("geot::mh_spmm", _backward, setup_context=_setup_context)
