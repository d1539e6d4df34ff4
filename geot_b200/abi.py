"""ctypes binding of the C ABI (``include/geot_b200.h``) -- the call a non-torch host makes.

Used by the parity tests and by ``bench.py`` so that what is tested and timed is the exported
``extern "C"`` surface itself; torch tensors only provide device memory and streams here.
"""
import ctypes
import os

import torch

from . import LIB_PATH

F32, F64, BF16, F16 = 0, 1, 2, 3
SUM, MEAN, MAX, MIN, PROD = 0, 1, 2, 3, 4
W_NONE, W_EDGE, W_EDGE_HEAD, W_HEAD_EDGE = 0, 1, 2, 3
REDUCE = {"sum": SUM, "mean": MEAN, "max": MAX, "amax": MAX, "min": MIN, "amin": MIN, "prod": PROD}
DTYPE = {torch.float32: F32, torch.float64: F64, torch.bfloat16: BF16, torch.float16: F16}

# every symbol include/geot_b200.h declares
SYMBOLS = [
    "geot_b200_version", "geot_b200_arch", "geot_b200_status_string", "geot_b200_last_cuda_error",
    "geot_b200_index_last", "geot_b200_plan_bytes", "geot_b200_format_preprocess", "geot_b200_plan_shards",
    "geot_b200_workspace_bytes", "geot_b200_segment_reduce", "geot_b200_index_scatter",
    "geot_b200_gather_scatter", "geot_b200_gather_weight_scatter", "geot_b200_mh_spmm",
    "geot_b200_sddmm_coo", "geot_b200_sddmm_mh", "geot_b200_csr_to_coo", "geot_b200_permute_edges",
    "geot_b200_segment_reduce_host", "geot_b200_host_arena_release", "geot_b200_profile_enable", "geot_b200_profile_read",
    "geot_b200_push_rows", "geot_b200_push_rows_ex", "geot_b200_set_unsorted_mode",
    "geot_b200_host_last_transfer", "geot_b200_host_row_pointers", "geot_b200_segment_reduce_ex",
    "geot_b200_host_graph_create", "geot_b200_host_graph_reduce", "geot_b200_host_graph_last_transfer",
    "geot_b200_host_graph_destroy", "geot_b200_src_blocks_suggest", "geot_b200_src_blocks_bytes",
    "geot_b200_src_blocks_scratch_bytes", "geot_b200_src_blocks_build", "geot_b200_src_blocks_workspace_bytes",
    "geot_b200_segment_softmax_workspace_bytes", "geot_b200_segment_softmax", "geot_b200_segment_softmax_backward",
    "geot_b200_gatv2_score", "geot_b200_gatv2_grad_workspace_bytes", "geot_b200_gatv2_grad",
    "geot_b200_graph_attention_workspace_bytes", "geot_b200_graph_attention",
    "geot_b200_graph_attention_grad_workspace_bytes", "geot_b200_graph_attention_grad",
]


class GeotPlan(ctypes.Structure):
    _fields_ = [("E", ctypes.c_int64), ("S", ctypes.c_int64), ("num_segments", ctypes.c_int64),
                ("max_degree", ctypes.c_int64), ("is_sorted", ctypes.c_int32), ("has_gaps", ctypes.c_int32),
                ("rowptr", ctypes.c_void_p), ("max_row", ctypes.c_int64)]


MAX_SRC_BLOCKS = 16


class SrcBlocksC(ctypes.Structure):
    """geot_src_blocks_t."""
    _fields_ = [("E", ctypes.c_int64), ("n_blocks", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("bounds", ctypes.c_int64 * (MAX_SRC_BLOCKS + 1)), ("dst_index", ctypes.c_void_p),
                ("src_index", ctypes.c_void_p), ("edge_perm", ctypes.c_void_p)]


class ReduceOpts(ctypes.Structure):
    """geot_reduce_opts_t (geot_b200_segment_reduce_ex)."""
    _fields_ = [("struct_size", ctypes.c_size_t), ("accumulate", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("edge_perm", ctypes.c_void_p), ("mean_rowptr", ctypes.c_void_p), ("src_blocks", ctypes.POINTER(SrcBlocksC))]


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        path = os.environ.get("GEOT_B200_LIB") or LIB_PATH   # tuning builds (Makefile VARIANT=...)
        if not os.path.exists(path):
            raise ImportError("geot_b200: %s not built; there is no fallback" % path)
        L = ctypes.CDLL(path)
        L.geot_b200_status_string.restype = ctypes.c_char_p
        L.geot_b200_last_cuda_error.restype = ctypes.c_char_p
        L.geot_b200_plan_bytes.restype = ctypes.c_size_t
        L.geot_b200_plan_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64]
        L.geot_b200_workspace_bytes.restype = ctypes.c_size_t
        L.geot_b200_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int]
        vp, i64, ci, sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_size_t
        L.geot_b200_index_last.argtypes = [vp, i64, ctypes.POINTER(ctypes.c_int64), vp]
        L.geot_b200_format_preprocess.argtypes = [vp, i64, i64, vp, sz, ctypes.POINTER(GeotPlan), vp]
        L.geot_b200_plan_shards.argtypes = [ctypes.POINTER(GeotPlan), ci, ctypes.POINTER(ctypes.c_int64),
                                            ctypes.POINTER(ctypes.c_int64), vp]
        L.geot_b200_segment_reduce.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, i64, ci, ci, ci, ci,
                                               ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_segment_reduce_ex.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, i64, ci, ci, ci, ci,
                                                  ctypes.POINTER(GeotPlan), vp, sz, vp, ctypes.POINTER(ReduceOpts)]
        L.geot_b200_host_graph_create.argtypes = [vp, vp, i64, i64, i64, ctypes.POINTER(vp)]
        L.geot_b200_host_graph_reduce.argtypes = [vp, vp, vp, vp, i64, i64, ci, ci, ci]
        ull = ctypes.POINTER(ctypes.c_ulonglong)
        L.geot_b200_host_graph_last_transfer.argtypes = [vp, ull, ull, ull]
        L.geot_b200_host_graph_destroy.argtypes = [vp]
        L.geot_b200_src_blocks_suggest.argtypes = [i64, i64, i64, i64]
        L.geot_b200_src_blocks_bytes.restype = sz
        L.geot_b200_src_blocks_bytes.argtypes = [i64]
        L.geot_b200_src_blocks_scratch_bytes.restype = sz
        L.geot_b200_src_blocks_scratch_bytes.argtypes = [i64]
        L.geot_b200_src_blocks_build.argtypes = [vp, vp, i64, i64, ci, vp, sz, vp, sz, ctypes.POINTER(SrcBlocksC), vp]
        L.geot_b200_src_blocks_workspace_bytes.restype = sz
        L.geot_b200_src_blocks_workspace_bytes.argtypes = [ctypes.POINTER(SrcBlocksC), i64, ci]
        L.geot_b200_index_scatter.argtypes = [vp, vp, vp, i64, i64, i64, ci, ci, ci, ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_gather_scatter.argtypes = [vp, vp, vp, vp, i64, i64, i64, ci, ci, ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_gather_weight_scatter.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, ci, ci,
                                                      ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_mh_spmm.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, i64, ci, ci, ci,
                                        ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_sddmm_coo.argtypes = [vp, vp, vp, vp, vp, i64, i64, ci, vp]
        L.geot_b200_sddmm_mh.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, ci, ci, vp]
        L.geot_b200_segment_softmax_workspace_bytes.restype = sz
        L.geot_b200_segment_softmax_workspace_bytes.argtypes = [i64, i64, ci]
        L.geot_b200_segment_softmax.argtypes = [vp, vp, vp, i64, i64, ci, ctypes.POINTER(GeotPlan), vp, sz, vp]
        L.geot_b200_segment_softmax_backward.argtypes = [vp, vp, vp, vp, i64, i64, ci, ctypes.POINTER(GeotPlan), vp, sz,
                                                         vp]
        L.geot_b200_gatv2_score.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, i64, ci, ctypes.POINTER(ctypes.c_double), vp]
        L.geot_b200_gatv2_grad_workspace_bytes.restype = sz
        L.geot_b200_gatv2_grad_workspace_bytes.argtypes = [i64, i64, i64, ci]
        L.geot_b200_gatv2_grad.argtypes = [vp, vp, vp, vp, vp, vp, ctypes.POINTER(GeotPlan), i64, vp, vp, i64, i64, i64,
                                           ci, ctypes.POINTER(ctypes.c_double), vp, sz, vp]
        dp = ctypes.POINTER(ctypes.c_double)
        L.geot_b200_graph_attention_workspace_bytes.restype = sz
        L.geot_b200_graph_attention_workspace_bytes.argtypes = [i64, i64, i64, ci]
        L.geot_b200_graph_attention.argtypes = [vp, vp, vp, vp, vp, ctypes.POINTER(GeotPlan), i64, vp, vp, i64, i64, i64,
                                                ci, dp, vp, sz, vp]
        L.geot_b200_graph_attention_grad_workspace_bytes.restype = sz
        L.geot_b200_graph_attention_grad_workspace_bytes.argtypes = [i64, i64, i64, ci]
        L.geot_b200_graph_attention_grad.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, ctypes.POINTER(GeotPlan), i64, vp, vp,
                                                     vp, i64, i64, i64, ci, dp, vp, sz, vp]
        L.geot_b200_csr_to_coo.argtypes = [vp, ci, i64, i64, vp, vp]
        L.geot_b200_permute_edges.argtypes = [vp, vp, vp, i64, i64, vp]
        L.geot_b200_segment_reduce_host.argtypes = [vp, i64, vp, vp, vp, vp, i64, i64, i64, i64, ci, ci, ci]
        L.geot_b200_push_rows.argtypes = [vp, vp, vp, vp, vp, i64, i64, ci, vp]
        L.geot_b200_push_rows_ex.argtypes = [vp, vp, vp, vp, vp, i64, i64, ci, ci, vp]
        L.geot_b200_host_last_transfer.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.POINTER(ctypes.c_ulonglong)]
        L.geot_b200_host_row_pointers.argtypes = [vp, i64, i64, i64, vp, ci]
        L.geot_b200_set_unsorted_mode.argtypes = [ci]
        _lib = L
    return _lib


def profile_enable(n: int) -> None:
    check(lib().geot_b200_profile_enable(n), "profile_enable")


def profile_read(capacity: int = 4096):
    """Durations (ms) of the most recent main-kernel launches recorded since profile_enable."""
    buf = (ctypes.c_float * capacity)()
    cnt = ctypes.c_int(0)
    check(lib().geot_b200_profile_read(buf, capacity, ctypes.byref(cnt)), "profile_read")
    return [buf[i] for i in range(cnt.value)]


class AbiError(RuntimeError):
    pass


def check(status: int, what: str = "") -> None:
    if status != 0:
        L = lib()
        msg = L.geot_b200_status_string(status).decode()
        if status == 4:
            msg += ": " + L.geot_b200_last_cuda_error().decode()
        raise AbiError("geot_b200 %s failed: %s (status %d)" % (what, msg, status))


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class DevicePlan:
    """format_preprocess through the C ABI; owns its device buffer."""

    def __init__(self, dst_index: torch.Tensor, S: int = None):
        L = lib()
        E = dst_index.numel()
        if S is None:
            last = ctypes.c_int64(-1)
            check(L.geot_b200_index_last(_ptr(dst_index), E, ctypes.byref(last), _stream()), "index_last")
            S = last.value + 1
        nbytes = L.geot_b200_plan_bytes(E, S)
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=dst_index.device)
        self.c = GeotPlan()
        check(L.geot_b200_format_preprocess(_ptr(dst_index), E, S, _ptr(self.buf), nbytes,
                                            ctypes.byref(self.c), _stream()), "format_preprocess")
        self.S = S
        self.rowptr = self.buf[: (S + 1) * 8].view(torch.int64)

    def shards(self, parts: int):
        rb = (ctypes.c_int64 * (parts + 1))()
        eb = (ctypes.c_int64 * (parts + 1))()
        check(lib().geot_b200_plan_shards(ctypes.byref(self.c), parts, rb, eb, _stream()), "plan_shards")
        return list(rb), list(eb)


class Workspace:
    def __init__(self, E, W, dtype, device, sorted=True, src_blocks=None):
        n = lib().geot_b200_workspace_bytes(E, W, DTYPE[dtype], 1 if sorted else 0)
        if src_blocks is not None:      # every block partitions on its own
            n = max(n, lib().geot_b200_src_blocks_workspace_bytes(ctypes.byref(src_blocks.c), W, DTYPE[dtype]))
        self.buf = torch.empty(n, dtype=torch.uint8, device=device)
        self.nbytes = n


def src_blocks_suggest(E: int, S: int, N_src: int, row_bytes: int) -> int:
    """Number of src-row blocks worth using for this shape (1: do not block) -- geot_b200_src_blocks_suggest."""
    return int(lib().geot_b200_src_blocks_suggest(E, S, N_src, row_bytes))


class SrcBlocks:
    """The edge list regrouped by src-row block for the L2 (geot_b200_src_blocks_build); owns its device buffer."""

    def __init__(self, src_index: torch.Tensor, dst_index: torch.Tensor, N_src: int, n_blocks: int):
        L = lib()
        E = dst_index.numel()
        nbytes, sbytes = L.geot_b200_src_blocks_bytes(E), L.geot_b200_src_blocks_scratch_bytes(E)
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=dst_index.device)
        scratch = torch.empty(sbytes, dtype=torch.uint8, device=dst_index.device)
        self.c = SrcBlocksC()
        check(L.geot_b200_src_blocks_build(_ptr(src_index), _ptr(dst_index), E, N_src, n_blocks, _ptr(self.buf), nbytes,
                                           _ptr(scratch), sbytes, ctypes.byref(self.c), _stream()), "src_blocks_build")
        self.n_blocks = n_blocks
        self.bounds = [int(self.c.bounds[i]) for i in range(n_blocks + 1)]
        a = (E * 8 + 255) // 256 * 256
        self.dst_index = self.buf[:E * 8].view(torch.int64)
        self.src_index = self.buf[a:a + E * 8].view(torch.int64)
        self.edge_perm = self.buf[2 * a:2 * a + E * 4].view(torch.int32)


def segment_reduce(src, src_index, dst_index, weight, reduce="sum", *, S=None, H=1, weight_layout=None,
                   sorted=True, plan: DevicePlan = None, out=None, workspace: Workspace = None,
                   accumulate=False, edge_perm=None, mean_rowptr=None, src_blocks: "SrcBlocks" = None):
    """Device-pointer call of geot_b200_segment_reduce (geot_b200_segment_reduce_ex when one of ``accumulate`` /
    ``edge_perm`` [E] int32 / ``mean_rowptr`` [S+1] int64 / ``src_blocks`` is given).  Returns dst [S, W]."""
    E = dst_index.numel()
    W = src.numel() // src.shape[0]
    F = W // H
    if S is None:
        S = plan.S if plan is not None else int(dst_index.max()) + 1
    if weight_layout is None:
        weight_layout = W_NONE if weight is None else (W_EDGE if weight.dim() == 1 else W_EDGE_HEAD)
    if out is None:
        out = torch.empty([S] + list(src.shape[1:]), dtype=src.dtype, device=src.device)
    if workspace is None:
        workspace = Workspace(E, W, src.dtype, src.device, sorted, src_blocks)
    args = (_ptr(src), _ptr(src_index), _ptr(dst_index), _ptr(weight), _ptr(out), E, S, H, F, DTYPE[src.dtype],
            REDUCE[reduce], weight_layout, 1 if sorted else 0, ctypes.byref(plan.c) if plan is not None else None,
            _ptr(workspace.buf), workspace.nbytes, _stream())
    if accumulate or edge_perm is not None or mean_rowptr is not None or src_blocks is not None:
        assert edge_perm is None or (edge_perm.dtype == torch.int32 and edge_perm.numel() == E)
        assert mean_rowptr is None or (mean_rowptr.dtype == torch.int64 and mean_rowptr.numel() == S + 1)
        opts = ReduceOpts(ctypes.sizeof(ReduceOpts), 1 if accumulate else 0, 0,
                          edge_perm.data_ptr() if edge_perm is not None else None,
                          mean_rowptr.data_ptr() if mean_rowptr is not None else None,
                          ctypes.pointer(src_blocks.c) if src_blocks is not None else None)
        st = lib().geot_b200_segment_reduce_ex(*args, ctypes.byref(opts))
    else:
        st = lib().geot_b200_segment_reduce(*args)
    check(st, "segment_reduce")
    return out


def sddmm_coo(mat1, row_index, mat2, col_index):
    """out[e] = <mat1[row_index[e]], mat2[col_index[e]]> through geot_b200_sddmm_coo."""
    E = row_index.numel()
    out = torch.empty(E, dtype=mat1.dtype, device=mat1.device)
    check(lib().geot_b200_sddmm_coo(_ptr(mat1), _ptr(row_index), _ptr(mat2), _ptr(col_index), _ptr(out), E,
                                    mat1.shape[1], DTYPE[mat1.dtype], _stream()), "sddmm_coo")
    return out


def sddmm_mh(mat1, row_index, mat2, col_index, head_major=False):
    """out[e, h] = <mat1[row_index[e], h], mat2[col_index[e], h]> ([E, H], or [H, E] with head_major) through
    geot_b200_sddmm_mh; mat1 / mat2 [N, H, F]."""
    E, H, F = row_index.numel(), mat1.shape[1], mat1.shape[2]
    out = torch.empty([H, E] if head_major else [E, H], dtype=mat1.dtype, device=mat1.device)
    check(lib().geot_b200_sddmm_mh(_ptr(mat1), _ptr(row_index), _ptr(mat2), _ptr(col_index), _ptr(out), E, H, F,
                                   DTYPE[mat1.dtype], W_HEAD_EDGE if head_major else W_EDGE_HEAD, _stream()), "sddmm_mh")
    return out


def _softmax_workspace(E, H, dtype, device):
    n = lib().geot_b200_segment_softmax_workspace_bytes(E, H, DTYPE[dtype])
    return torch.empty(n, dtype=torch.uint8, device=device), n


def segment_softmax(src, dst_index, plan: DevicePlan = None):
    """Softmax of src [E] / [E, H] over the edges of each dst row (dst_index sorted) through geot_b200_segment_softmax."""
    E, H = dst_index.numel(), src[0].numel() if src.numel() else 1
    plan = plan if plan is not None else DevicePlan(dst_index)
    out = torch.empty_like(src)
    ws, n = _softmax_workspace(E, H, src.dtype, src.device)
    check(lib().geot_b200_segment_softmax(_ptr(src), _ptr(dst_index), _ptr(out), E, H, DTYPE[src.dtype],
                                          ctypes.byref(plan.c), _ptr(ws), n, _stream()), "segment_softmax")
    return out


def segment_softmax_backward(out, grad_out, dst_index, plan: DevicePlan = None):
    """grad_src = out * (grad_out - sum over the row of out * grad_out) through geot_b200_segment_softmax_backward."""
    E, H = dst_index.numel(), out[0].numel() if out.numel() else 1
    plan = plan if plan is not None else DevicePlan(dst_index)
    grad_src = torch.empty_like(out)
    ws, n = _softmax_workspace(E, H, out.dtype, out.device)
    check(lib().geot_b200_segment_softmax_backward(_ptr(out), _ptr(grad_out), _ptr(dst_index), _ptr(grad_src), E, H,
                                                   DTYPE[out.dtype], ctypes.byref(plan.c), _ptr(ws), n, _stream()),
          "segment_softmax_backward")
    return grad_src


def gatv2_score(x_l, x_r, att, src_index, dst_index, negative_slope=0.2):
    """[E, H] GATv2 scores sum_f att[h, f] * leaky_relu(x_l[src[e], h, f] + x_r[dst[e], h, f]) through
    geot_b200_gatv2_score; x_l / x_r [N, H, F], att [H, F]."""
    E, H, F = dst_index.numel(), x_l.shape[1], x_l.shape[2]
    out = torch.empty(E, H, dtype=x_l.dtype, device=x_l.device)
    check(lib().geot_b200_gatv2_score(_ptr(x_l), _ptr(x_r), _ptr(att), _ptr(src_index), _ptr(dst_index), _ptr(out), E, H,
                                      F, DTYPE[x_l.dtype], ctypes.byref(ctypes.c_double(negative_slope)), _stream()),
          "gatv2_score")
    return out


def gatv2_grad(x_row, x_gat, att, grad_score, row_index, gat_index, S_out, negative_slope=0.2, want_att=True,
               plan: DevicePlan = None):
    """One backward pass of the GATv2 score through geot_b200_gatv2_grad: (grad_row [S_out, H, F], grad_att [H, F] or
    None); row_index sorted."""
    E, H, F = row_index.numel(), x_row.shape[1], x_row.shape[2]
    plan = plan if plan is not None else DevicePlan(row_index)
    grad_row = torch.empty(S_out, H, F, dtype=x_row.dtype, device=x_row.device)
    grad_att = torch.empty(H, F, dtype=x_row.dtype, device=x_row.device) if want_att else None
    n = lib().geot_b200_gatv2_grad_workspace_bytes(E, H, F, DTYPE[x_row.dtype])
    ws = torch.empty(n, dtype=torch.uint8, device=x_row.device)
    check(lib().geot_b200_gatv2_grad(_ptr(x_row), _ptr(x_gat), _ptr(att), _ptr(grad_score), _ptr(row_index),
                                     _ptr(gat_index), ctypes.byref(plan.c), S_out, _ptr(grad_row),
                                     _ptr(grad_att) if want_att else None, E, H, F, DTYPE[x_row.dtype],
                                     ctypes.byref(ctypes.c_double(negative_slope)),
                                     _ptr(ws), n, _stream()), "gatv2_grad")
    return grad_row, grad_att


def graph_attention(q, k, v, src_index, dst_index, scale, N_dst=None, plan: DevicePlan = None):
    """(out [N_dst, H, F], lse [N_dst, H]) of the fused dot-product attention through geot_b200_graph_attention; q
    [N_dst, H, F], k / v [N_src, H, F], dst_index sorted."""
    E, H, F = dst_index.numel(), q.shape[1], q.shape[2]
    N_dst = q.shape[0] if N_dst is None else N_dst
    plan = plan if plan is not None else DevicePlan(dst_index)
    out = torch.empty(N_dst, H, F, dtype=q.dtype, device=q.device)
    acc = torch.float64 if q.dtype == torch.float64 else torch.float32
    lse = torch.empty(N_dst, H, dtype=acc, device=q.device)
    n = lib().geot_b200_graph_attention_workspace_bytes(E, H, F, DTYPE[q.dtype])
    ws = torch.empty(n, dtype=torch.uint8, device=q.device)
    check(lib().geot_b200_graph_attention(_ptr(q), _ptr(k), _ptr(v), _ptr(src_index), _ptr(dst_index), ctypes.byref(plan.c),
                                          N_dst, _ptr(out), _ptr(lse), E, H, F, DTYPE[q.dtype],
                                          ctypes.byref(ctypes.c_double(scale)), _ptr(ws), n, _stream()), "graph_attention")
    return out, lse


def graph_attention_grad(q, k, v, out, lse, grad_out, src_index, dst_index, scale, plan: DevicePlan = None):
    """(grad_q, p [E, H], scale * ds [E, H]) of the dst pass of the backward through geot_b200_graph_attention_grad."""
    E, H, F = dst_index.numel(), q.shape[1], q.shape[2]
    plan = plan if plan is not None else DevicePlan(dst_index)
    grad_q = torch.empty_like(q)
    p = torch.empty(E, H, dtype=q.dtype, device=q.device)
    ds = torch.empty(E, H, dtype=q.dtype, device=q.device)
    n = lib().geot_b200_graph_attention_grad_workspace_bytes(E, H, F, DTYPE[q.dtype])
    ws = torch.empty(n, dtype=torch.uint8, device=q.device)
    check(lib().geot_b200_graph_attention_grad(_ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(lse), _ptr(grad_out),
                                               _ptr(src_index), _ptr(dst_index), ctypes.byref(plan.c), q.shape[0],
                                               _ptr(grad_q), _ptr(p), _ptr(ds), E, H, F, DTYPE[q.dtype],
                                               ctypes.byref(ctypes.c_double(scale)), _ptr(ws), n, _stream()),
          "graph_attention_grad")
    return grad_q, p, ds


def csr_to_coo(rowptr, E):
    """Sorted COO row index [E] (int64) of a CSR row pointer (int32 or int64) through geot_b200_csr_to_coo."""
    out = torch.empty(E, dtype=torch.int64, device=rowptr.device)
    bits = 64 if rowptr.dtype == torch.int64 else 32
    check(lib().geot_b200_csr_to_coo(_ptr(rowptr), bits, rowptr.numel() - 1, E, _ptr(out), _stream()), "csr_to_coo")
    return out


def permute_edges(x, perm, out=None):
    """out[e] = x[perm[e]] for a per-edge operand ([E] or [E, H]) or a row matrix through geot_b200_permute_edges."""
    E = perm.numel()
    if out is None:
        out = x.new_empty([E] + list(x.shape[1:]))
    check(lib().geot_b200_permute_edges(_ptr(x), _ptr(perm), _ptr(out), E, x[0].numel() * x.element_size() if E else 2,
                                        _stream()), "permute_edges")
    return out


def push_rows(x, rows, dest_peer, dest_row, peer_bases_dev: int, aligned16: bool = True, max_ctas: int = 0):
    """peer_bases[dest_peer[e]][dest_row[e]] = x[rows[e]] through geot_b200_push_rows_ex.  ``peer_bases_dev``: device
    address of the array of per-GPU base pointers (``_SymmetricMemory.buffer_ptrs_dev``, or the ``data_ptr()`` of an
    int64 device tensor holding the addresses).  ``max_ctas`` > 0: a small grid for a push that overlaps a reduction."""
    n = rows.numel()
    row_bytes = x[0].numel() * x.element_size() if x.shape[0] else 4
    check(lib().geot_b200_push_rows_ex(_ptr(x), _ptr(rows), _ptr(dest_peer), _ptr(dest_row), ctypes.c_void_p(peer_bases_dev),
                                       n, row_bytes, 1 if aligned16 else 0, max_ctas, _stream()), "push_rows")


def host_last_transfer():
    """(h2d_bytes, d2h_bytes) the last segment_reduce_host call moved over the link."""
    a, b = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    check(lib().geot_b200_host_last_transfer(ctypes.byref(a), ctypes.byref(b)), "host_last_transfer")
    return a.value, b.value


def host_row_pointers(index: torch.Tensor, row0: int, rows: int, threads: int = 0) -> torch.Tensor:
    """CSR row pointer [rows + 1] of a sorted CPU index slice through geot_b200_host_row_pointers (pure host code)."""
    assert not index.is_cuda and index.dtype == torch.int64 and index.is_contiguous()
    out = torch.empty(rows + 1, dtype=torch.int64)
    check(lib().geot_b200_host_row_pointers(_ptr(index), index.numel(), row0, rows, _ptr(out), threads), "host_row_pointers")
    return out


def segment_reduce_host(src, src_index, dst_index, weight, reduce="sum", *, S, H=1, weight_layout=None, out=None):
    """Host-buffer call (geot_b200_segment_reduce_host): CPU tensors in, CPU tensor out."""
    E = dst_index.numel()
    W = src.numel() // src.shape[0]
    F = W // H
    if weight_layout is None:
        weight_layout = W_NONE if weight is None else (W_EDGE if weight.dim() == 1 else W_EDGE_HEAD)
    if out is None:
        out = torch.empty([S] + list(src.shape[1:]), dtype=src.dtype)
    st = lib().geot_b200_segment_reduce_host(_ptr(src), src.shape[0], _ptr(src_index), _ptr(dst_index), _ptr(weight),
                                            _ptr(out), E, S, H, F, DTYPE[src.dtype], REDUCE[reduce], weight_layout)
    check(st, "segment_reduce_host")
    return out


class HostGraph:
    """Resident host graph (geot_b200_host_graph_*): the index arrays are uploaded once; every ``reduce`` call ships
    only src (+ weights) and brings dst back.  CPU tensors in, CPU tensor out."""

    def __init__(self, src_index, dst_index, S: int, N_src: int):
        assert not dst_index.is_cuda and dst_index.dtype == torch.int64 and dst_index.is_contiguous()
        assert src_index is None or (not src_index.is_cuda and src_index.dtype == torch.int64 and src_index.is_contiguous())
        self.h = ctypes.c_void_p(0)
        self.E, self.S, self.N_src = dst_index.numel(), S, N_src
        check(lib().geot_b200_host_graph_create(_ptr(src_index), _ptr(dst_index), self.E, S, N_src, ctypes.byref(self.h)),
              "host_graph_create")

    def reduce(self, src, weight=None, reduce="sum", *, H=1, weight_layout=None, out=None):
        assert not src.is_cuda and src.is_contiguous()
        W = src.numel() // src.shape[0]
        if weight_layout is None:
            weight_layout = W_NONE if weight is None else (W_EDGE if weight.dim() == 1 else W_EDGE_HEAD)
        if out is None:
            out = torch.empty([self.S] + list(src.shape[1:]), dtype=src.dtype)
        check(lib().geot_b200_host_graph_reduce(self.h, _ptr(src), _ptr(weight), _ptr(out), H, W // H, DTYPE[src.dtype],
                                                REDUCE[reduce], weight_layout), "host_graph_reduce")
        return out

    def last_transfer(self):
        """(h2d bytes, d2h bytes) of the last reduce, and the bytes made resident at creation."""
        a, b, c = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        check(lib().geot_b200_host_graph_last_transfer(self.h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)),
              "host_graph_last_transfer")
        return a.value, b.value, c.value

    def close(self):
        if self.h:
            lib().geot_b200_host_graph_destroy(self.h)
            self.h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
