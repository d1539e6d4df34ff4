"""Fake (meta) implementations of the C++-registered ``geot::*`` operators so that ``torch.export`` /
``torch.compile`` can trace through them.  The reference registers fakes only for its Python custom ops
(``geot/gather_scatter.py:12-18``, ``geot/gather_weight_scatter.py:21-28``, ``geot/csr_gws.py:30-37``);
``geot::mh_spmm`` and ``geot::index_scatter`` have none there (SURVEY 8f N4).  The number of output rows is
data dependent (``index[-1] + 1``), hence a fresh dynamic size.
"""
import torch


def _rows():
    return torch.library.get_ctx().new_dynamic_size()


@torch.library.register_fake("geot::index_scatter")
def _(dim, index, src, reduce, sorted):
    shape = list(src.shape)
    shape[dim] = _rows()
    return src.new_empty(shape)


@torch.library.register_fake("geot::gather_scatter_impl")
def _(src_index, dst_index, src):
    return src.new_empty([_rows(), src.shape[1]])


@torch.library.register_fake("geot::gather_scatter_reduce")
def _(src_index, dst_index, src, reduce):
    return src.new_empty([_rows(), src.shape[1]])


@torch.library.register_fake("geot::gather_weight_scatter_impl")
def _(src_index, dst_index, weight, src):
    return src.new_empty([_rows(), src.shape[1]])


@torch.library.register_fake("geot::gather_weight_scatter_reduce")
def _(src_index, dst_index, weight, src, reduce):
    return src.new_empty([_rows(), src.shape[1]])


@torch.library.register_fake("geot::mh_spmm")
def _(src_index, dst_index, weight, src, reduce):
    return src.new_empty([_rows(), src.shape[1], src.shape[2]])


@torch.library.register_fake("geot::sddmm_coo_impl")
def _(src_index, dst_index, mat_1, mat_2):
    return mat_1.new_empty([src_index.shape[0]])


@torch.library.register_fake("geot::sddmm_mh_impl")
def _(src_index, dst_index, mat_1, mat_2, head_major):
    E, H = src_index.shape[0], mat_1.shape[1]
    return mat_1.new_empty([H, E] if head_major else [E, H])


@torch.library.register_fake("geot::segment_softmax")
def _(src, index):
    return torch.empty_like(src, memory_format=torch.contiguous_format)


@torch.library.register_fake("geot::segment_softmax_backward")
def _(out, grad_out, index):
    return torch.empty_like(out, memory_format=torch.contiguous_format)


@torch.library.register_fake("geot::gatv2_score")
def _(x_l, x_r, att, src_index, dst_index, negative_slope):
    return x_l.new_empty([dst_index.shape[0], x_l.shape[1]])


@torch.library.register_fake("geot::gatv2_score_backward")
def _(grad, x_l, x_r, att, src_index, dst_index, t_perm, t_dst_index, t_src_index, negative_slope, need_x_l, need_x_r,
      need_att):
    def like(t, need):
        return t.new_empty(t.shape) if need else t.new_empty([0])
    return like(x_l, need_x_l), like(x_r, need_x_r), like(att, need_att)


@torch.library.register_fake("geot::graph_attention")
def _(q, k, v, src_index, dst_index, scale):
    acc = torch.float64 if q.dtype == torch.float64 else torch.float32
    return q.new_empty(q.shape), q.new_empty([q.shape[0], q.shape[1]], dtype=acc)


@torch.library.register_fake("geot::graph_attention_backward")
def _(grad, q, k, v, out, lse, src_index, dst_index, scale):
    E, H = dst_index.shape[0], q.shape[1]
    return q.new_empty(q.shape), q.new_empty([E, H]), q.new_empty([E, H])


@torch.library.register_fake("geot::csr_gws_impl")
def _(indptr, indices, weight, src):
    return src.new_empty([indptr.shape[0], src.shape[1]])


@torch.library.register_fake("geot::coo_to_csr_impl")
def _(coo_row):
    return coo_row.new_empty([_rows()], dtype=torch.int32)
