"""``segment_softmax``: the softmax of edge logits over the edges of each dst row -- the attention weights of a GAT
layer -- on a dst-sorted edge list.

``geot::segment_softmax`` is a C++ operator (one edge-balanced pass, no atomics, bit-reproducible; see
``include/geot_b200.h``); its backward ``grad_src = out * (grad_out - sum_row(out * grad_out))`` is the operator
``geot::segment_softmax_backward``, registered as the autograd of the forward.  It needs the forward's output only, so
that is what the forward saves.
"""
import torch

from .index_scatter import _as_int64


def segment_softmax(src: torch.Tensor, index: torch.Tensor) -> torch.Tensor:
    """``out[e, h] = exp(src[e, h]) / sum_{e' : index[e'] = index[e]} exp(src[e', h])`` (computed with the row maximum
    subtracted).  ``src`` is ``[E]`` or ``[E, H]``, fp32 / fp64 / bf16 / fp16 (fp32 accumulation for the 16-bit types);
    ``index`` is ``[E]`` int64 or int32 and non-decreasing.  Differentiable in ``src``."""
    if index.dtype == torch.int32:
        index = _as_int64(index)       # the widened copy is cached, so the plan cache keeps hitting
    return torch.ops.geot.segment_softmax(src, index)


def _setup_context(ctx, inputs, output):
    ctx.save_for_backward(output, inputs[1])


def _backward(ctx, grad):
    out, index = ctx.saved_tensors
    return torch.ops.geot.segment_softmax_backward(out, grad.contiguous(), index), None


torch.library.register_autograd("geot::segment_softmax", _backward, setup_context=_setup_context)
