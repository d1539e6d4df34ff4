"""``gatv2_score``: the GATv2 attention score of every edge (PyG ``GATv2Conv``), fused, with a deterministic backward.

    score[e, h] = sum_f att[h, f] * leaky_relu(x_l[src[e], h, f] + x_r[dst[e], h, f])

Written in torch ops the score materialises several ``[E, H * F]`` tensors (the two gathers, their sum, the leaky_relu,
the product with ``att``) and autograd keeps some of them; its backward scatters into ``x_l`` and ``x_r`` with atomics.
``geot::gatv2_score`` is one SDDMM-style kernel with no ``[E, H * F]`` intermediate, and its backward
``geot::gatv2_score_backward`` is two edge-balanced segment passes without atomics (``include/geot_b200.h``): the dst pass
over the dst-sorted edges gives ``grad_x_r`` and ``grad_att``, the src pass over the cached transposed edge list
(``transpose.py``) gives ``grad_x_l``.  The forward saves its inputs only.
"""
import torch

from .index_scatter import _as_int64


def gatv2_score(x_l: torch.Tensor, x_r: torch.Tensor, att: torch.Tensor, src_index: torch.Tensor,
                dst_index: torch.Tensor, negative_slope: float = 0.2) -> torch.Tensor:
    """``[E, H]`` scores ``sum_f att[h, f] * leaky_relu(x_l[src_index[e], h, f] + x_r[dst_index[e], h, f])``.

    ``x_l`` is ``[N_l, H, F]``, ``x_r`` ``[N_r, H, F]``, ``att`` ``[H, F]`` (or ``[1, H, F]``), all of one dtype: fp32 /
    fp64 / bf16 / fp16, with fp32 accumulation for the 16-bit types.  ``src_index`` / ``dst_index`` are ``[E]`` int64 or
    int32; ``dst_index`` is non-decreasing.  Differentiable in ``x_l``, ``x_r`` and ``att``; the gradients are
    bit-reproducible."""
    if src_index.dtype == torch.int32:
        src_index = _as_int64(src_index)
    if dst_index.dtype == torch.int32:
        dst_index = _as_int64(dst_index)       # the widened copies are cached, so the plan cache keeps hitting
    if att.dim() == 3:
        att = att.reshape(att.shape[1], att.shape[2])
    return torch.ops.geot.gatv2_score(x_l, x_r, att, src_index, dst_index, float(negative_slope))


def _setup_context(ctx, inputs, output):
    x_l, x_r, att, src_index, dst_index, negative_slope = inputs
    ctx.save_for_backward(x_l, x_r, att, src_index, dst_index)
    ctx.negative_slope = negative_slope


def _backward(ctx, grad):
    from .transpose import transposed_edges
    x_l, x_r, att, src_index, dst_index = ctx.saved_tensors
    need_l, need_r, need_att = ctx.needs_input_grad[:3]
    if need_l:
        t = transposed_edges(src_index, dst_index)
        perm, t_dst, t_src = t.perm, t.dst_index, t.src_index
    else:
        perm = t_dst = t_src = src_index
    gl, gr, ga = torch.ops.geot.gatv2_score_backward(grad.contiguous(), x_l, x_r, att, src_index, dst_index, perm, t_dst,
                                                     t_src, ctx.negative_slope, need_l, need_r, need_att)
    return (gl if need_l else None), (gr if need_r else None), (ga if need_att else None), None, None, None


torch.library.register_autograd("geot::gatv2_score", _backward, setup_context=_setup_context)
