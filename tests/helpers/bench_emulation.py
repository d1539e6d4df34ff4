"""CPU emulation harness for bench.py's control flow (test infrastructure).

bench.py needs a GPU: it has no CPU path.  To test ITS host logic here (sharding, exchange forms, the timed region,
the end-to-end legs, the JSON contract) the CUDA runtime calls and the C-ABI calls it makes are replaced by stand-ins
-- the oracle plays the kernels, gloo plays NCCL -- and ``bench.run_own`` runs unchanged on top.  The numbers it
prints are meaningless; the keys, shapes and collective sequence are what is checked."""
import contextlib
import io
import json
import os
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def install(rank=0, world=1):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    import oracle

    class FakeEvent:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, *a):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    torch.cuda.is_available = lambda: True
    torch.cuda.set_device = lambda d: None
    torch.cuda.synchronize = lambda *a: None
    torch.cuda.empty_cache = lambda: None
    torch.cuda.Event = FakeEvent
    torch.cuda.current_stream = lambda *a: types.SimpleNamespace(synchronize=lambda: None, cuda_stream=0)
    torch.Tensor.pin_memory = lambda self: self
    orig_device = torch.device
    torch.device = lambda *a, **k: orig_device("cpu") if (a and a[0] == "cuda") else orig_device(*a, **k)
    init = dist.init_process_group
    dist.init_process_group = lambda backend, device_id=None: init("gloo", rank=rank, world_size=world)

    from geot_b200 import abi

    class DevicePlan:
        def __init__(self, di, S=None):
            self.S = S if S is not None else int(di[-1]) + 1
            deg = torch.bincount(di, minlength=self.S)
            self.rowptr = torch.cat([deg.new_zeros(1), deg.cumsum(0)])

    class Workspace:
        def __init__(self, *a, **k):
            self.nbytes = 0

    def segment_reduce(src, si, di, w, reduce="sum", *, S=None, H=1, weight_layout=None, sorted=True, plan=None, out=None,
                       workspace=None, accumulate=False, edge_perm=None, mean_rowptr=None, src_blocks=None):
        if w is not None and edge_perm is not None:
            w = w[edge_perm.long()]
        red = "sum" if mean_rowptr is not None else reduce
        r = oracle.segment_reduce(src.float(), si, di, None if w is None else w.float(), red, S=S, H=H)
        if mean_rowptr is not None and reduce == "mean":
            deg = (mean_rowptr[1:] - mean_rowptr[:-1]).clamp_min(1).float()
            r = r / deg.view([-1] + [1] * (r.dim() - 1))
        r = r.to(src.dtype)
        if out is not None:
            if accumulate:
                out += r
            else:
                out.copy_(r)
            return out
        return r

    def permute(x, perm, out=None):
        r = x[perm]
        if out is not None:
            out.copy_(r)
            return out
        return r

    class HostGraph:
        def __init__(self, si, di, S, N_src):
            self.si, self.di, self.S = si, di, S

        def reduce(self, src, weight=None, reduce="sum", *, H=1, weight_layout=None, out=None):
            return segment_reduce(src, self.si, self.di, weight, reduce, S=self.S, H=H, out=out)

        def last_transfer(self):
            return (700, 10, 5000)

        def close(self):
            pass

    calls = {"n": 0}
    abi.DevicePlan, abi.Workspace, abi.segment_reduce, abi.HostGraph = DevicePlan, Workspace, segment_reduce, HostGraph
    abi.segment_reduce_host = (lambda src, si, di, w, reduce="sum", *, S, H=1, weight_layout=None, out=None:
                               segment_reduce(src, si, di, w, reduce, S=S, H=H, out=out))
    abi.permute_edges = permute
    abi.src_blocks_suggest = lambda *a: 1
    abi.profile_enable = lambda n: calls.__setitem__("n", n)
    abi.profile_read = lambda cap=4096: [0.05] * min(cap, max(calls["n"], 1))
    abi.host_last_transfer = lambda: (1000, 10)
    abi.lib = lambda: types.SimpleNamespace(geot_b200_workspace_bytes=lambda *a: 256, geot_b200_host_arena_release=lambda: 0)


def run_own(workload, world=1, steps=2, warmup=3, dump_outputs=None):
    """bench.run_own under the emulation; returns rank 0's JSON line (None on the other ranks)."""
    import bench
    args = types.SimpleNamespace(gpus=world, steps=steps, warmup=warmup, impl="own", workload=workload,
                                 dump_outputs=dump_outputs)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.run_own(args)
    out = buf.getvalue().strip()
    return json.loads(out.splitlines()[-1]) if out else None


def worker(rank, world, port, exchange, workload, q, dump_outputs=None):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), GEOT_B200_EXCHANGE=exchange)
    install(rank, world)
    line = run_own(workload, world, dump_outputs=dump_outputs)
    if rank == 0:
        q.put(line)
