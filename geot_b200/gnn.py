"""PyG-free forward of the reference's GCN / GraphSAGE models on the geot operators (SURVEY 8f N1).

The reference's models are ``torch_geometric`` ``BasicGNN`` clones whose ``message_and_aggregate`` calls
geot (``/root/reference/models/gcn.py:26-60``, ``models/graphsage.py:26-64``, ``models/conv/spmm.py:5-14``).
PyG / torch_sparse are not part of this build, so the same math is restated on plain index tensors:

* GCN layer (``models/conv/gcnconv.py:212-259``): ``out = A_hat @ (x W) + b`` with
  ``A_hat[i,j] = d_i^-1/2 w_ij d_j^-1/2`` (``gcn_norm``, ``gcnconv.py:41-57``; ``d`` = weighted in-degree of the
  dst-sorted adjacency, optional self loops) -- one ``gather_weight_scatter`` per layer.  The reference
  recomputes ``gcn_norm`` on every forward unless ``cached``; here the normalised weights and the
  ``format_preprocess`` plan are computed once per graph.
* GraphSAGE layer (``models/conv/sageconv.py:122-154``, ``aggr="sum"`` as ``models/graphsage.py:48`` sets it):
  ``out = lin_l(sum_j x_j) + lin_r(x)`` -- one ``gather_scatter`` per layer.
* GAT layer (PyG ``GATConv`` without dropout): the attention softmax is ``segment_softmax``, the weighted
  aggregation ``mh_spmm`` -- both deterministic kernels of this library, both differentiable.
* GATv2 layer (PyG ``GATv2Conv``, ``share_weights=False``, without dropout and edge features): the attention score is
  the fused ``gatv2_score``, then ``segment_softmax`` and ``mh_spmm``.
* Transformer layer (PyG ``TransformerConv`` without ``beta``, edge features and dropout): the fused
  ``graph_attention`` (dot-product scores, softmax and aggregation in one pass), then the skip connection.
* Stack (``models/basicgnn.py:216-264``): ``conv -> ReLU`` for every layer but the last; dropout p = 0.

The dense ``lin`` layers are cuBLAS GEMMs through ``torch.nn.Linear`` (library code, not part of the hot
path).  ``forward_sharded`` runs the same stack with the node rows sharded over the GPUs of one box
(``geot_b200.dist``): the GEMM is row-local with replicated weights, the aggregation exchanges the src
rows once per layer (one all-gather, or the overlapped two-bucket exchange of ``dist.BucketedGather``).
"""
from typing import List, Optional

import torch
from torch import nn

from .gather_scatter import gather_scatter
from .gather_weight_scatter import gather_weight_scatter
from .mh_spmm import mh_spmm
from .softmax import segment_softmax
from .gatv2 import gatv2_score
from .attention import graph_attention


def add_self_loops(src_index: torch.Tensor, dst_index: torch.Tensor, num_nodes: int,
                   edge_weight: Optional[torch.Tensor] = None, fill_value: float = 1.0):
    """Sets the diagonal to ``fill_value`` (``torch_sparse.fill_diag`` semantics: existing self loops are
    replaced) and returns the edge list re-sorted by (dst, src)."""
    keep = src_index != dst_index
    loop = torch.arange(num_nodes, device=dst_index.device, dtype=dst_index.dtype)
    s = torch.cat([src_index[keep], loop])
    d = torch.cat([dst_index[keep], loop])
    w = None
    if edge_weight is not None:
        w = torch.cat([edge_weight[keep], edge_weight.new_full((num_nodes,), fill_value)])
    key, perm = torch.sort(d * num_nodes + s)
    return s[perm].contiguous(), d[perm].contiguous(), (w[perm].contiguous() if w is not None else None)


def gcn_norm(src_index: torch.Tensor, dst_index: torch.Tensor, num_nodes: int,
             edge_weight: Optional[torch.Tensor] = None, dtype=torch.float32) -> torch.Tensor:
    """Symmetric normalisation ``d_dst^-1/2 * w * d_src^-1/2`` of a dst-sorted edge list
    (``models/conv/gcnconv.py:41-57``: ``deg = sum(adj_t, dim=1)``, infinities -> 0)."""
    w = edge_weight if edge_weight is not None else torch.ones(dst_index.numel(), dtype=dtype, device=dst_index.device)
    deg = torch.zeros(num_nodes, dtype=w.dtype, device=w.device).index_add_(0, dst_index, w)
    dis = deg.pow(-0.5)
    dis.masked_fill_(dis == float("inf"), 0.0)
    return dis.index_select(0, dst_index) * w * dis.index_select(0, src_index)


def _pad_rows(out: torch.Tensor, n: int) -> torch.Tensor:
    """geot ops return ``dst_index[-1] + 1`` rows; trailing isolated nodes get zero rows."""
    if out.shape[0] >= n:
        return out
    return torch.cat([out, out.new_zeros([n - out.shape[0]] + list(out.shape[1:]))], 0)


class GCNConv(nn.Module):
    """``GCNConv_GS`` (``models/conv/gcnconv.py``): ``lin`` without bias, aggregation, then ``+ bias``."""

    def __init__(self, in_channels: int, out_channels: int, bias: bool = True):
        super().__init__()
        self.lin = nn.Linear(in_channels, out_channels, bias=False)
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None

    def forward(self, x, src_index, dst_index, norm_weight):
        h = self.lin(x)
        out = _pad_rows(gather_weight_scatter(src_index, dst_index, norm_weight, h), x.shape[0])
        return out + self.bias if self.bias is not None else out


class SAGEConv(nn.Module):
    """``SAGEConv_GS`` with ``aggr="sum"``, ``root_weight=True`` (``models/conv/sageconv.py:122-154``)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.lin_l = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, src_index, dst_index, reduce: str = "sum"):
        agg = _pad_rows(gather_scatter(src_index, dst_index, x, reduce), x.shape[0])
        return self.lin_l(agg) + self.lin_r(x)


class GATConv(nn.Module):
    """PyG's ``GATConv`` math without dropout, on a dst-sorted edge list (the caller adds self loops with
    ``add_self_loops``): ``h = lin(x)`` as ``[N, H, F]``; per edge and head
    ``alpha = softmax_row(leaky_relu(<h[src], att_src> + <h[dst], att_dst>))`` (``segment_softmax``); the aggregation
    ``out[dst] = sum alpha * h[src]`` is ``mh_spmm``; the heads are concatenated (``concat``) or averaged, then ``bias``
    is added.  Differentiable end to end."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, bias: bool = True):
        super().__init__()
        self.heads, self.out_channels, self.concat, self.negative_slope = heads, out_channels, concat, negative_slope
        self.lin = nn.Linear(in_channels, heads * out_channels, bias=False)
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        self.bias = nn.Parameter(torch.zeros(heads * out_channels if concat else out_channels)) if bias else None
        nn.init.xavier_uniform_(self.lin.weight)
        nn.init.xavier_uniform_(self.att_src)
        nn.init.xavier_uniform_(self.att_dst)

    def forward(self, x, src_index, dst_index):
        N, H, F = x.shape[0], self.heads, self.out_channels
        h = self.lin(x).view(N, H, F)
        a_src = (h * self.att_src).sum(-1)
        a_dst = (h * self.att_dst).sum(-1)
        logits = torch.nn.functional.leaky_relu(a_src.index_select(0, src_index) + a_dst.index_select(0, dst_index),
                                                self.negative_slope)
        alpha = segment_softmax(logits, dst_index)
        out = _pad_rows(mh_spmm(src_index, dst_index, alpha, h), N)
        out = out.reshape(N, H * F) if self.concat else out.mean(1)
        return out + self.bias if self.bias is not None else out


class GATv2Conv(nn.Module):
    """PyG's ``GATv2Conv`` math on a dst-sorted edge list (the caller adds self loops with ``add_self_loops``):
    ``x_l = lin_l(x)`` and ``x_r = lin_r(x)`` as ``[N, H, F]``; per edge and head
    ``score = sum_f att[h, f] * leaky_relu(x_l[src, h, f] + x_r[dst, h, f])`` (the fused ``gatv2_score``),
    ``alpha = softmax_row(score)`` (``segment_softmax``); the aggregation ``out[dst] = sum alpha * x_l[src]`` is
    ``mh_spmm``; the heads are concatenated (``concat``) or averaged, then ``bias`` is added.  ``lin_l``, ``lin_r`` and
    ``att`` get PyG's glorot initialisation, ``lin_l`` / ``lin_r`` carry a bias when ``bias`` is set, and the output bias
    starts at zero, as in PyG.  Left out of PyG's options: ``share_weights`` (always separate ``lin_l`` / ``lin_r``),
    ``edge_dim``, attention ``dropout``, ``add_self_loops`` (done by the caller) and ``residual``.  Differentiable end to
    end; no ``[E, H * F]`` tensor is materialised."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, bias: bool = True):
        super().__init__()
        self.heads, self.out_channels, self.concat, self.negative_slope = heads, out_channels, concat, negative_slope
        self.lin_l = nn.Linear(in_channels, heads * out_channels, bias=bias)
        self.lin_r = nn.Linear(in_channels, heads * out_channels, bias=bias)
        self.att = nn.Parameter(torch.empty(1, heads, out_channels))
        self.bias = nn.Parameter(torch.zeros(heads * out_channels if concat else out_channels)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        # PyG: Linear(weight_initializer="glorot") with zero biases, glorot(att), zeros(bias)
        for lin in (self.lin_l, self.lin_r):
            nn.init.xavier_uniform_(lin.weight)
            if lin.bias is not None:
                nn.init.zeros_(lin.bias)
        nn.init.xavier_uniform_(self.att)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x, src_index, dst_index):
        N, H, F = x.shape[0], self.heads, self.out_channels
        x_l = self.lin_l(x).view(N, H, F)
        x_r = self.lin_r(x).view(N, H, F)
        score = gatv2_score(x_l, x_r, self.att, src_index, dst_index, self.negative_slope)
        alpha = segment_softmax(score, dst_index)
        out = _pad_rows(mh_spmm(src_index, dst_index, alpha, x_l), N)
        out = out.reshape(N, H * F) if self.concat else out.mean(1)
        return out + self.bias if self.bias is not None else out


class TransformerConv(nn.Module):
    """PyG's ``TransformerConv`` math on a dst-sorted edge list (no self loops are added, as in PyG):
    ``q = lin_query(x)``, ``k = lin_key(x)``, ``v = lin_value(x)`` as ``[N, H, F]``; per edge and head
    ``alpha = softmax_row(<q[dst], k[src]> / sqrt(F))`` and ``out[dst] = sum alpha * v[src]`` (the fused
    ``graph_attention``, which materialises no ``[E, H]`` tensor); the heads are concatenated (``concat``) or averaged,
    then ``lin_skip(x)`` is added when ``root_weight`` is set.  ``lin_query``, ``lin_key`` and ``lin_value`` map to
    ``H * F`` and ``lin_skip`` to ``H * F`` (``concat``) or ``F``, all with a bias when ``bias`` is set and torch's default
    initialisation, as PyG's ``Linear``.  Left out of PyG's options: ``beta`` (the gated skip), ``edge_dim`` (edge
    features) and attention ``dropout``; one node set (no bipartite input).  Differentiable end to end."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True, bias: bool = True,
                 root_weight: bool = True):
        super().__init__()
        self.heads, self.out_channels, self.concat, self.root_weight = heads, out_channels, concat, root_weight
        self.lin_query = nn.Linear(in_channels, heads * out_channels, bias=bias)
        self.lin_key = nn.Linear(in_channels, heads * out_channels, bias=bias)
        self.lin_value = nn.Linear(in_channels, heads * out_channels, bias=bias)
        self.lin_skip = (nn.Linear(in_channels, heads * out_channels if concat else out_channels, bias=bias)
                         if root_weight else None)

    def forward(self, x, src_index, dst_index):
        N, H, F = x.shape[0], self.heads, self.out_channels
        q = self.lin_query(x).view(N, H, F)
        k = self.lin_key(x).view(N, H, F)
        v = self.lin_value(x).view(N, H, F)
        out = graph_attention(q, k, v, src_index, dst_index)
        out = out.reshape(N, H * F) if self.concat else out.mean(1)
        return out + self.lin_skip(x) if self.lin_skip is not None else out


class _Stack(nn.Module):
    def __init__(self, conv, in_channels, hidden_channels, num_layers, out_channels=None):
        super().__init__()
        out_channels = hidden_channels if out_channels is None else out_channels
        dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.convs = nn.ModuleList([conv(dims[i], dims[i + 1]) for i in range(num_layers)])

    def _run(self, x, *graph):
        for i, conv in enumerate(self.convs):
            x = conv(x, *graph)
            if i + 1 < len(self.convs):
                x = torch.relu(x)
        return x


class GCN(_Stack):
    """``GCN_GS`` (``models/gcn.py:26-33``): ``num_layers`` GCN layers, ReLU between them."""

    def __init__(self, in_channels, hidden_channels, num_layers, out_channels=None):
        super().__init__(GCNConv, in_channels, hidden_channels, num_layers, out_channels)

    def forward(self, x, src_index, dst_index, norm_weight):
        return self._run(x, src_index, dst_index, norm_weight)


class GraphSAGE(_Stack):
    """``GraphSAGE_GS`` (``models/graphsage.py:26-33``) with sum aggregation."""

    def __init__(self, in_channels, hidden_channels, num_layers, out_channels=None):
        super().__init__(SAGEConv, in_channels, hidden_channels, num_layers, out_channels)

    def forward(self, x, src_index, dst_index):
        return self._run(x, src_index, dst_index)


def forward_sharded(model: _Stack, x_local: torch.Tensor, shard, group=None, gather=None) -> torch.Tensor:
    """The same stack on a dst-row shard (``geot_b200.dist.GraphShard``): ``x_local`` are this rank's node
    rows; returns this rank's rows of the output.  Per layer: row-local GEMM(s) with replicated weights,
    the exchange of the src rows, aggregation into the local dst rows.  ``shard.weight`` carries the
    (globally normalised) GCN weights for a GCN stack and is ``None`` for GraphSAGE.

    ``gather``: a ``geot_b200.dist.BucketedGather`` built once for ``shard`` -- the exchange is then overlapped
    with the reduction (all-gather or needed-rows push transport, whichever the object was built with) and its
    per-graph state (buckets, plans, request lists) is shared by all layers.  ``None``: one all-gather per layer.
    Forward only (the overlapped exchange is not differentiable)."""
    from . import dist as gdist

    def aggregate(h):
        if gather is None:
            return gdist.sharded_gather_scatter(shard, h, "sum", group)
        return gather.aggregate(h.detach(), shard.weight, "sum")

    x = x_local
    for i, conv in enumerate(model.convs):
        if isinstance(conv, GCNConv):
            h = conv.lin(x)
            out = aggregate(h)
            if conv.bias is not None:
                out = out + conv.bias
        else:
            agg = aggregate(x)
            out = conv.lin_l(agg) + conv.lin_r(x)
        x = torch.relu(out) if i + 1 < len(model.convs) else out
    return x
