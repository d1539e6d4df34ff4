"""``graph_attention``: fused dot-product graph attention (the attention of PyG ``TransformerConv``), with a deterministic
backward that recomputes the attention weights.

    score[e, h] = scale * <q[dst[e], h, :], k[src[e], h, :]>
    out[i, h, :] = sum_{e : dst[e] = i} softmax_row(score)[e, h] * v[src[e], h, :]

Composed from ``sddmm_mh_impl``, ``segment_softmax`` and ``mh_spmm`` this is three kernels that write and re-read two
``[E, H]`` tensors.  ``geot::graph_attention`` is one edge-balanced pass with FlashAttention's online softmax: it stores
only ``out`` and the per-row log-sum-exp ``lse [N_dst, H]``, no ``[E, H]`` tensor.  The backward,
``geot::graph_attention_backward``, recomputes ``p = exp(score - lse)`` in one dst-sorted pass that gives ``grad_q`` and
the ``[E, H]`` weights ``p`` and ``scale * ds``; ``grad_v`` and ``grad_k`` are ``mh_spmm`` on the cached transposed edge
list with those weights (``mh_spmm.src_side_spmm``).  No atomics: the forward and every gradient are bit-reproducible.
"""
import math
from typing import Optional

import torch

from .index_scatter import _as_int64
from .mh_spmm import src_side_spmm


def graph_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, src_index: torch.Tensor,
                    dst_index: torch.Tensor, scale: Optional[float] = None) -> torch.Tensor:
    """``[N_dst, H, F]`` output ``out[i, h] = sum_{e : dst[e] = i} alpha[e, h] * v[src[e], h]`` with
    ``alpha = softmax over the row i of scale * <q[dst[e], h], k[src[e], h]>``.

    ``q`` is ``[N_dst, H, F]``, ``k`` and ``v`` ``[N_src, H, F]``, all of one dtype: fp32 / fp64 / bf16 / fp16, with fp32
    accumulation for the 16-bit types.  ``scale=None`` is ``1 / sqrt(F)``.  ``src_index`` / ``dst_index`` are ``[E]``
    int64 or int32; ``dst_index`` is non-decreasing with values below ``N_dst``.  Rows without edges are zero.
    Differentiable in ``q``, ``k`` and ``v``; the gradients are bit-reproducible."""
    if src_index.dtype == torch.int32:
        src_index = _as_int64(src_index)
    if dst_index.dtype == torch.int32:
        dst_index = _as_int64(dst_index)       # the widened copies are cached, so the plan cache keeps hitting
    if scale is None:
        scale = 1.0 / math.sqrt(q.shape[-1])
    return torch.ops.geot.graph_attention(q, k, v, src_index, dst_index, float(scale))[0]


def _setup_context(ctx, inputs, output):
    q, k, v, src_index, dst_index, scale = inputs
    out, lse = output
    ctx.save_for_backward(q, k, v, out, lse, src_index, dst_index)
    ctx.scale = scale
    ctx.mark_non_differentiable(lse)


def _backward(ctx, grad, grad_lse):
    q, k, v, out, lse, src_index, dst_index = ctx.saved_tensors
    need_q, need_k, need_v = ctx.needs_input_grad[:3]
    gq, p, ds = torch.ops.geot.graph_attention_backward(grad.contiguous(), q, k, v, out, lse, src_index, dst_index,
                                                        ctx.scale)
    gk = gv = None
    if dst_index.numel() == 0:
        gk = torch.zeros_like(k) if need_k else None
        gv = torch.zeros_like(v) if need_v else None
    else:
        if need_k:      # grad_k[j] = sum_{e : src = j} scale ds[e] q[dst[e]]
            gk = src_side_spmm(src_index, dst_index, ds, q.contiguous(), k.shape[0])
        if need_v:      # grad_v[j] = sum_{e : src = j} p[e] g[dst[e]]
            gv = src_side_spmm(src_index, dst_index, p, grad.contiguous(), v.shape[0])
    return (gq if need_q else None), gk, gv, None, None, None


torch.library.register_autograd("geot::graph_attention", _backward, setup_context=_setup_context)
