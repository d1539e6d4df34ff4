#!/usr/bin/env python
"""bench.py -- headline benchmark of the segment-reduction hot path (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl own|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload (BASELINE.json
configs[1], the configuration the metric is quoted on): gather_weight_scatter, GCN aggregation on a
synthetic Reddit-shape graph (232,965 nodes, 114,615,892 (dst,src)-sorted edges, F = 128, fp32).

  value      effective GB/s = algorithmic ("logical") bytes per step / time, inputs resident in HBM,
             called through the C ABI (libgeot_b200.so) with a cached format_preprocess plan.
  e2e        the same metric with HOST operands through the C ABI's resident host graph
             (geot_b200_host_graph_reduce: the static index arrays were uploaded once at create; every
             step copies src + weights host->device from pinned memory and the result device->host,
             inside the timed region).  The stateless host entry (geot_b200_segment_reduce_host, which
             also ships the index arrays every call) is timed beside it.
  roofline   the dominant kernel (segment_reduce_kernel) timed with CUDA events recorded by the library
             around that kernel alone, against the measured HBM copy bandwidth (MEASURED_PEAKS.json);
             three fractions: on logical bytes, on the DRAM bytes ncu counted, on compulsory bytes.
  cpu_baseline  the CPU restatement of the reference (oracle/, OpenMP over all host cores; torch's
             index_select*mul+index_add_ beside it) on a bounded sample of the same workload.
  parity     the timed configuration's own output checked in the same run: counting property (src = 1
             => in-degree, exact) and sampled rows (hubs included) against the CPU oracle.
  secondary  the other BASELINE.json configurations (N = 1: index_scatter on the Reddit shape and on
             config #1 with the reference's CPU path timed beside it, products gather_scatter, arxiv
             mh_spmm; N > 1: products gather_scatter F = 64 / 256, exchange-inclusive and pre-replicated).

--impl reference times the reference's CPU side of the path on the host cores (GeoT ships a CPU kernel
for index_scatter only -- numerically wrong, SURVEY 8a A5 -- and none for gather_weight_scatter, so the
arm is the oracle port / torch restatement; where oracle/_ref was built its csrc/cpu kernel is timed too
and labelled).  N > 1: one process per GPU under torchrun; the dst rows are sharded with balanced edge
counts, each rank reduces its own slice, the src rows travel each step inside the timed region
(GEOT_B200_EXCHANGE = push [default: the rows the peers' edges reference are stored into their symmetric
memory by one kernel, overlapped with the src-local edge bucket; src-remote bucket accumulated afterwards]
| bucket [the same two buckets around one NCCL all-gather] | allgather [one all-gather, then one
reduction] | replicated; strong scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm uses every host core (rank 0 alone runs it)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import torch  # noqa: E402

WORKLOADS = {
    # name: (graph, op, F, H, dtype)
    "reddit_gws": ("reddit", "gather_weight_scatter", 128, 1, torch.float32),
    "reddit_index_scatter": ("reddit", "index_scatter", 128, 1, torch.float32),
    "products_gs64": ("products", "gather_scatter", 64, 1, torch.float32),
    "products_gs256": ("products", "gather_scatter", 256, 1, torch.float32),
    # the products shape with a quarter of the dst rows isolated: shows what zero-filling rows without edges costs (it
    # happens inside the main kernel; the reference clears all of dst first, csrc/gather_scatter.cpp:27-30)
    "products_gs64_gaps": ("products+isolated", "gather_scatter", 64, 1, torch.float32),
    "arxiv_mh_spmm": ("arxiv", "mh_spmm", 32, 8, torch.bfloat16),
    "proteins_gws256": ("proteins", "gather_weight_scatter", 256, 1, torch.float32),
    "config1_index_scatter": ("config1", "index_scatter", 64, 1, torch.float32),
}
DTYPE_NAME = {torch.float32: "f32", torch.float64: "f64", torch.bfloat16: "bf16", torch.float16: "f16"}
EXCHANGES = {
    "bucket": "one ragged NCCL all-gather on a side stream, overlapped with the reduction of the src-local edge bucket; "
              "the src-remote bucket is accumulated into the same output afterwards (2 reductions, no combine pass)",
    "push": "ONE kernel stores the rows the peers' edges reference straight into their symmetric-memory buffers over "
            "NVLink (no NCCL on the data path), overlapped with the src-local edge bucket; src-remote bucket afterwards",
    "allgather": "one NCCL all-gather, then one reduction",
    "replicated": "NONE inside the step (src pre-replicated: kernel scaling only, SURVEY 8e)",
    "none": "no exchange (edge-aligned operands)",
}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6564.0, "measured on an NVIDIA B200 at 1000 W power limit: 4 GiB device copy, read + write bytes"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # clocks under load: the upper half of the samples (idle samples before/after the region excluded)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_workload(name, device, scale=1.0):
    import workloads as wl
    gname, op, F, H, dtype = WORKLOADS[name]
    s = torch.tensor([], dtype=dtype).element_size()
    if gname == "config1":
        E, S = 1_000_000, 50_000
        dst = wl.random_segments(E, S, device)
        g = wl.Graph("config1", S, None, dst, 0, 0.0)
    elif gname.endswith("+isolated"):
        g = wl.power_law_graph(gname.split("+")[0], device, scale, isolated=0.25)
    else:
        g = wl.power_law_graph(gname, device, scale)
    E, N = g.num_edges, g.num_nodes
    w = None
    if op == "index_scatter":
        x = torch.empty(E, F, device=device, dtype=dtype)
        gen = torch.Generator(device=device).manual_seed(1)
        for i in range(0, E, 1 << 24):
            x[i:i + (1 << 24)].uniform_(0, 1, generator=gen) if dtype == torch.float32 else x[i:i + (1 << 24)].copy_(
                torch.rand(min(1 << 24, E - i), F, device=device, generator=gen))
        si = None
    elif op == "mh_spmm":
        x = wl.features(N, (H, F), dtype, device)
        w = wl.edge_weights(E, H, dtype, device)
        si = g.src_index
    else:
        x = wl.features(N, F, dtype, device)
        if op == "gather_weight_scatter":
            w = wl.edge_weights(E, None, dtype, device)
        si = g.src_index
    S = int(g.dst_index[-1]) + 1
    return dict(name=name, graph=g, op=op, F=F, H=H, dtype=dtype, esize=s, x=x, w=w, si=si, di=g.dst_index, E=E, N=N, S=S,
                bytes_logical=wl.bytes_logical(op, E, S, N, F, H, s), bytes_compulsory=wl.bytes_compulsory(op, E, S, N, F, H, s))


# ---- CPU arm -----------------------------------------------------------------------------------------

def cpu_sample(wk, frac_edges=1.0 / 16, max_edges=8_000_000):
    """Bounded CPU-side sample of the workload: a prefix of the sorted edge list (whole segments)."""
    E = wk["E"]
    n = int(min(E, max(min(E, 1_000_000), min(max_edges, E * frac_edges))))
    di = wk["di"][:n].cpu()
    S = int(di[-1]) + 1
    si = wk["si"][:n].cpu() if wk["si"] is not None else None
    w = wk["w"][:n].cpu() if wk["w"] is not None else None
    x = wk["x"].cpu() if wk["si"] is not None else wk["x"][:n].cpu()
    import workloads as wl
    nbytes = wl.bytes_logical(wk["op"], n, S, x.shape[0], wk["F"], wk["H"], wk["esize"])
    return dict(n=n, S=S, di=di, si=si, w=w, x=x, bytes=nbytes, fraction=n / E)


def time_cpu(fn, warmup, steps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts), min(ts)


def cpu_arm(wk, warmup, steps):
    """Times the CPU restatements on a bounded sample with every host core.  Returns the cpu_baseline object, the
    per-step seconds of the fastest one and the sample fraction."""
    import oracle
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)                    # (torchrun workers start with OMP_NUM_THREADS=1)
    cores = oracle.set_threads(ncpu)
    sm = cpu_sample(wk)
    H = wk["H"]
    res = {}
    if wk["dtype"] == torch.float32:
        fn = lambda: oracle.segment_reduce(sm["x"], sm["si"], sm["di"], sm["w"], "sum", S=sm["S"], H=H, threads=True)
    else:   # the threaded C variant is fp32-only; low precision goes through the upcasting wrapper
        x32, w32 = sm["x"].float(), (sm["w"].float() if sm["w"] is not None else None)
        fn = lambda: oracle.segment_reduce(x32, sm["si"], sm["di"], w32, "sum", S=sm["S"], H=H, threads=True)
    res["oracle_port_openmp"] = time_cpu(fn, warmup, steps)

    def torch_fn():
        x = sm["x"].float()
        g = x if sm["si"] is None else x.index_select(0, sm["si"])
        if sm["w"] is not None:
            ww = sm["w"].float()
            g = g * (ww.unsqueeze(-1) if ww.dim() < g.dim() else ww)
        return torch.zeros([sm["S"]] + list(x.shape[1:])).index_add_(0, sm["di"], g)
    res["torch_restatement"] = time_cpu(torch_fn, warmup, steps)
    kind = "port"
    if wk["op"] == "index_scatter" and wk["dtype"] == torch.float32 and oracle.load_ref_extension():
        # the reference's own CPU kernel (csrc/cpu/index_scatter_cpu.cpp:136-155), unmodified, compiled by oracle/Makefile.ref
        ref = lambda: torch.ops.geot_ref.index_scatter(0, sm["di"], sm["x"], "sum", True)
        res["reference_csrc_cpu_NUMERICALLY_WRONG_A5"] = time_cpu(ref, warmup, steps)
    best = min((k for k in res if "WRONG" not in k), key=lambda k: res[k][0])
    gbs = {k: sm["bytes"] / v[0] / 1e9 for k, v in res.items()}
    sample = ("first %d of %d edges (%d dst rows; fraction %.4f) of the workload, sum; GB/s on the sample's logical bytes; avg of "
              "%d runs: " % (sm["n"], wk["E"], sm["S"], sm["fraction"], steps)
              + ", ".join("%s %.2f GB/s" % (k, v) for k, v in gbs.items())
              + "; os.cpu_count=%s omp_threads=%d torch_threads=%d" % (os.cpu_count(), cores, torch.get_num_threads()))
    obj = {"value": round(gbs[best], 3), "unit": "GB/s", "cores": cores, "kind": kind, "sample": sample,
           "sample_fraction": round(sm["fraction"], 6), "edges_per_s": sm["n"] / res[best][0], "which": best,
           "all_gbs": {k: round(v, 3) for k, v in gbs.items()}}
    return obj, res[best][0], sm["fraction"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.manual_seed(0)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    scale = 1.0 if dev == "cuda" else 1.0 / 16
    wk = build_workload(args.workload, dev, scale)
    steps, warmup = args.steps, args.warmup
    obj, sec, frac = cpu_arm(wk, warmup, steps)
    assert obj["cores"] > 1 or (os.cpu_count() or 1) == 1, "the CPU arm must use every host core"
    cfg = config_of(wk, args.gpus)
    cfg["sample_fraction"] = round(frac, 6)
    cfg["sample"] = "each step = the first %.4f of the workload's sorted edge list (whole segments)" % frac
    line = {
        "impl": "reference", "metric": metric_name(wk), "value": obj["value"], "unit": "GB/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE_NAME[wk["dtype"]],
        "data": "synthetic", "config": cfg,
        "cpu_baseline": obj,
        "e2e": {"value": obj["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "edges_per_s": obj["edges_per_s"], "gpu_launches": 0,
    }
    print(json.dumps(line))


def metric_name(wk):
    return "%s effective GB/s (logical bytes / time)" % wk["op"]


def config_of(wk, n_gpus, exchange="none"):
    g = wk["graph"]
    return {"workload": "%s: %s on synthetic %s-shape graph, %d nodes, %d (dst,src)-sorted edges, F=%d%s, %s" % (
                wk["name"], wk["op"], g.name, wk["N"], wk["E"], wk["F"], (" x H=%d" % wk["H"]) if wk["H"] > 1 else "",
                DTYPE_NAME[wk["dtype"]]),
            "edges": wk["E"], "nodes": wk["N"], "dst_rows": wk["S"], "F": wk["F"], "H": wk["H"],
            "max_degree": g.max_degree, "degree_cv": round(g.degree_cv, 3),
            "bytes_logical_per_step": wk["bytes_logical"], "bytes_compulsory_per_step": wk["bytes_compulsory"],
            "l2": "per-step input streams (%.2f GB) exceed the 126 MB L2; no explicit flush" % (
                (wk["bytes_compulsory"]) / 1e9),
            "parallelism": "1 GPU" if n_gpus == 1 else "dst rows sharded over %d GPUs (edge-balanced); src rows per step: %s" % (
                n_gpus, EXCHANGES[exchange])}


# ---- the GPU arm -------------------------------------------------------------------------------------

class Runner:
    """One workload set up for timing on this rank: the shard (N > 1), the exchange form, preallocated output and
    scratch, and `step()` = one pass of the hot path through the C ABI."""

    def __init__(self, wk, world, rank, dev, exchange):
        from geot_b200 import abi
        from geot_b200 import dist as gdist
        self.wk, self.world, self.rank, self.dev = wk, world, rank, dev
        self.abi, self.gdist = abi, gdist
        op, H = wk["op"], wk["H"]
        self.gather = op != "index_scatter"
        w = wk["w"]
        self.layout = abi.W_NONE if w is None else (abi.W_EDGE if w.dim() == 1 else abi.W_EDGE_HEAD)
        self.exchange = exchange if (world > 1 and self.gather) else "none"
        self.shard, self.bg, self.imbalance, self.exchanged = None, None, 1.0, None
        tail = list(wk["x"].shape[1:])
        if world > 1:
            sh = self.shard = gdist.shard_graph(wk["si"], wk["di"], w, rank, world)
            self.imbalance = sh.imbalance
            rb = sh.row_bounds
            e0, e1 = sh.edge_bounds[rank], sh.edge_bounds[rank + 1]
            self.di, self.si, self.w, self.S = sh.dst_index, sh.src_index, sh.weight, sh.num_local_rows
            self.row0 = rb[rank]
            self.x_edges = wk["x"][e0:e1].contiguous() if not self.gather else None
            self.x_local = wk["x"][rb[rank]:rb[rank + 1]].contiguous() if self.gather else None
            self.x_full = None
            if self.exchange in ("allgather", "replicated"):
                self.x_full = torch.empty([wk["N"]] + tail, dtype=wk["dtype"], device=dev)
            if self.exchange == "replicated":
                gdist.all_gather_rows(self.x_local, rb, out=self.x_full)
            if self.exchange in ("bucket", "push"):
                # passes: 0 = the library's choice (two overlapped passes when the local bucket's rows are long, else one)
                # phases: 0 = the library's choice (push at >= 6 GPUs: the exchange in two rounds, each followed by its edges)
                self.bg = gdist.BucketedGather(sh, transport="push" if self.exchange == "push" else "allgather",
                                               passes=int(os.environ.get("GEOT_B200_EXCHANGE_PASSES", "0")),
                                               phases=int(os.environ.get("GEOT_B200_EXCHANGE_PHASES", "0")),
                                               phase_steps=([int(v) for v in os.environ["GEOT_B200_EXCHANGE_STEPS"].split(",")]
                                                            if os.environ.get("GEOT_B200_EXCHANGE_STEPS") else None))
                self.exchanged = self.bg.exchanged_rows()
        else:
            self.di, self.si, self.w, self.S, self.row0 = wk["di"], wk["si"], w, wk["S"], 0
        self.E = self.di.numel()
        self.W = wk["F"] * H
        self.out = torch.empty([self.S] + tail, dtype=wk["dtype"], device=dev)
        self.plan = self.ws = self.blocks = None
        if self.bg is None and self.E > 0:
            self.plan = abi.DevicePlan(self.di, self.S)
            # src-row blocking for the L2 (built once per graph, like the plan): the library's own suggestion unless
            # GEOT_B200_SRC_BLOCKS forces a count (1 = off)
            nb = int(os.environ.get("GEOT_B200_SRC_BLOCKS", "0"))
            if self.gather and H == 1 and self.exchange in ("none", "replicated"):
                if nb <= 0:
                    nb = abi.src_blocks_suggest(self.E, self.S, wk["N"], self.W * wk["esize"]) if wk["esize"] >= 4 else 1
                if nb > 1:
                    self.blocks = abi.SrcBlocks(self.si, self.di, wk["N"], nb)
            self.ws = abi.Workspace(self.E, self.W, wk["dtype"], dev, src_blocks=self.blocks)
        self.n_blocks = self.blocks.n_blocks if self.blocks is not None else 1
        self.passes = self.bg.passes if self.bg is not None else 1
        self.phases = self.bg.phases if self.bg is not None else 1
        self.per_head_perm = 1 if (self.bg is not None and w is not None and w.dim() == 2 and self.passes == 2) else 0

    @property
    def calls_per_step(self):
        """Main-kernel launches of one step (known after the first step: a bucket may be src-blocked inside)."""
        return self.bg.main_launches() if self.bg is not None else self.n_blocks

    @property
    def launches_per_step(self):
        """This library's kernels per step: main + fixup per reduction pass (+ one push kernel per exchange round, + the
        per-head weight permutation)."""
        return 2 * self.calls_per_step + (self.phases if self.exchange == "push" else 0) + self.per_head_perm

    def reduce(self, x, w, out, reduce="sum"):
        """The op on this rank's operands: x = full src (N = 1) / this rank's src rows (N > 1 gather) / edge rows."""
        wk, abi = self.wk, self.abi
        if self.E == 0:
            return out.zero_()
        if self.bg is not None:
            return self.bg(x, w, reduce, out=out)
        if self.exchange == "allgather":
            x = self.gdist.all_gather_rows(x, self.shard.row_bounds, out=self.x_full)
        elif self.exchange == "replicated":
            # the timed step reads the pre-replicated matrix; any other operand (the parity check's) is gathered afresh
            x = self.x_full if x is self.x_local else self.gdist.all_gather_rows(x, self.shard.row_bounds)
        return abi.segment_reduce(x, self.si, self.di, w, reduce, S=self.S, H=wk["H"], weight_layout=self.layout if w is not None else abi.W_NONE,
                                  plan=self.plan, out=out, workspace=self.ws,
                                  src_blocks=self.blocks if reduce in ("sum", "mean") else None)

    def src_operand(self):
        if self.world == 1:
            return self.wk["x"]
        return self.x_local if self.gather else self.x_edges

    def step(self):
        self.reduce(self.src_operand(), self.w, self.out)


def barrier(world):
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def time_runner(r, steps, warmup, sampler=None, keep_output=False):
    """W warm-up steps, then exactly K steps between barrier + synchronize, CUDA events on the launching stream, max
    over ranks.  The main kernel's own duration comes from a SECOND loop of K steps with the library's profiling hook
    on (an event pair around every main-kernel launch): the timed loop itself carries no instrumentation -- an event
    record between the main kernel and its programmatically dependent fixup launch would serialise the two and cost
    the small shapes several microseconds per step.  `keep_output`: r.timed_output = a copy of what the last timed step
    wrote, taken before the second loop.  Returns (ms per step, main-kernel ms per step)."""
    import torch.distributed as dist
    abi = r.abi
    for _ in range(max(warmup, 3)):
        r.step()
    abi.profile_enable(0)
    # launch-bound shapes (a step of tens of microseconds: config #1, arxiv mh_spmm) are replayed from a CUDA graph of the
    # very same C-ABI call, so that the number is the GPU's and not the Python interpreter's
    run, r.launch = r.step, "eager"
    if r.world == 1 and r.wk["bytes_logical"] < 4e9 and os.environ.get("GEOT_B200_BENCH_GRAPH", "1") == "1":
        try:
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                r.step()
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
            run, r.launch = graph.replay, "cuda_graph_replay"
        except Exception as ex:          # the eager call is the same work; say which one was timed
            print("bench: CUDA graph capture failed, timing eager calls: %r" % (ex,), file=sys.stderr)
            torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    barrier(r.world)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        run()
    ev[1].record()
    barrier(r.world)
    total_ms = ev[0].elapsed_time(ev[1])
    if keep_output:
        r.timed_output = r.out.clone()
    abi.profile_enable(steps * r.calls_per_step)
    for _ in range(steps):
        r.step()
    barrier(r.world)
    kernel_ms = abi.profile_read(steps * r.calls_per_step)
    abi.profile_enable(0)
    kmean = (sum(kernel_ms) / steps) if kernel_ms else 0.0
    if r.world > 1:
        t = torch.tensor([total_ms, kmean], device=r.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, kmean = t.tolist()
    return total_ms / steps, kmean


DUMP_BYTES = 32 << 20       # --dump-outputs writes the whole output up to this size, a sample of its rows beyond


def dump_outputs(out, directory):
    """Writes the output of the timed step to DIR/output.npy (float64 for fp64 outputs, float32 otherwise) so that two
    builds can be compared output for output.  An output larger than DUMP_BYTES is written as a fixed, seeded sample of
    its rows, in ascending order; their indices go to DIR/output_rows.npy (float64)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    host = torch.float64 if out.dtype == torch.float64 else torch.float32
    S = out.shape[0]
    row_bytes = max(1, out.numel() // max(S, 1)) * torch.tensor([], dtype=host).element_size()
    k = min(S, max(1, DUMP_BYTES // row_bytes))
    rows_path = os.path.join(directory, "output_rows.npy")
    if k < S:
        rows = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:k].sort().values
        np.save(rows_path, rows.double().numpy())
        out = out.index_select(0, rows.to(out.device))
    elif os.path.exists(rows_path):
        os.remove(rows_path)
    np.save(os.path.join(directory, "output.npy"), out.to(host).cpu().numpy())


def parity_check(r, rows_k=40):
    """The timed configuration checked in the same run (the oracle is the checker only): (1) counting -- src = 1,
    weight = 1 => every output element equals its row's in-degree (exact in fp32; bf16 within 1e-2); (2) the timed
    step's own output on sampled rows (the 3 largest hubs, first, last, random ones) against the CPU oracle recomputed
    from the rows' edge slices (fp64 accumulation; 1e-5 relative for fp32, 1e-2 for bf16).  All-reduced over ranks."""
    import oracle
    import torch.distributed as dist
    wk = r.wk
    dtype = wk["dtype"]
    tol = 1e-5 if dtype in (torch.float32, torch.float64) else 1e-2
    res = {"counting_ok": True, "rows_ok": True, "rows_checked": 0, "max_rel_err": 0.0}
    if r.E > 0 and r.S > 0:
        deg = torch.bincount(r.di, minlength=r.S)
        src = r.src_operand()
        ones = torch.ones_like(src)
        w1 = torch.ones_like(r.w) if r.w is not None else None
        out = torch.full_like(r.out, 3.0)
        r.reduce(ones, w1, out)
        exp = deg.to(torch.float32).view([-1] + [1] * (out.dim() - 1)).expand_as(out)
        if dtype == torch.float32:
            res["counting_ok"] = bool(torch.equal(out, exp))
        else:
            res["counting_ok"] = bool(((out.float() - exp).abs() <= 1e-2 * exp).all())
        del ones, w1, out, exp
        # sampled rows of the timed step's output
        r.step()
        torch.cuda.synchronize()
        rowptr = torch.cat([deg.new_zeros(1), deg.cumsum(0)]).cpu()
        g = torch.Generator().manual_seed(1234 + r.rank)
        rows = torch.unique(torch.cat([torch.randint(0, r.S, (rows_k,), generator=g), torch.topk(deg.cpu(), min(3, r.S)).indices,
                                       torch.tensor([0, r.S - 1])]))
        x_all = wk["x"]                                   # full src (gather ops) / all edge rows (index_scatter)
        e_base = r.shard.edge_bounds[r.rank] if r.shard is not None else 0
        worst = 0.0
        for row in rows.tolist():
            b, e = int(rowptr[row]), int(rowptr[row + 1])
            got = r.out[row].cpu()
            if b == e:
                ok = float(got.abs().sum()) == 0.0
            else:
                w = r.w[b:e].cpu() if r.w is not None else None
                if r.gather:
                    uniq, inv = torch.unique(r.si[b:e], return_inverse=True)
                    xs, si = x_all[uniq].cpu(), inv.cpu()
                else:
                    xs, si = x_all[e_base + b:e_base + e].cpu(), None
                expv = oracle.segment_reduce(xs, si, torch.zeros(e - b, dtype=torch.int64), w, "sum", S=1, H=wk["H"],
                                             acc64=(dtype == torch.float32))[0]
                err = float(((got.double() - expv.double()).abs() / expv.double().abs().clamp_min(1e-30)).max())
                worst = max(worst, err)
                ok = err <= tol
            res["rows_ok"] = res["rows_ok"] and ok
            res["rows_checked"] += 1
        res["max_rel_err"] = worst
    if r.world > 1:
        t = torch.tensor([0.0 if res["counting_ok"] else 1.0, 0.0 if res["rows_ok"] else 1.0, res["max_rel_err"]],
                         device=r.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n = torch.tensor([float(res["rows_checked"])], device=r.dev, dtype=torch.float64)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
        res = {"counting_ok": t[0].item() == 0, "rows_ok": t[1].item() == 0, "rows_checked": int(n.item()), "max_rel_err": t[2].item()}
    res["ok"] = bool(res["counting_ok"] and res["rows_ok"])
    res["tolerance"] = tol
    res["max_rel_err"] = float("%.3g" % res["max_rel_err"])
    res["what"] = ("counting (src=1, weight=1 => in-degree) + the timed output's sampled rows (3 hubs, first, last, random) "
                   "vs the CPU oracle, every rank, all-reduced")
    return res


def fractions(wk, r, kmean, peak, traffic=None):
    """The main kernel's three roofline readings (per launch on this rank; N > 1: the slowest rank's time)."""
    import workloads as wl
    k_log = wl.bytes_logical(wk["op"], r.E, r.S, wk["N"], wk["F"], wk["H"], wk["esize"])
    k_comp = wl.bytes_compulsory(wk["op"], r.E, r.S, wk["N"], wk["F"], wk["H"], wk["esize"])
    if kmean <= 0:
        return k_log, k_comp, 0.0, {}
    achieved = k_log / (kmean * 1e-3) / 1e9
    f = {"frac_logical": round(achieved / peak, 4), "frac_compulsory": round(k_comp / (kmean * 1e-3) / 1e9 / peak, 4),
         "frac_dram": round(traffic / (kmean * 1e-3) / 1e9 / peak, 4) if traffic else None}
    return k_log, k_comp, achieved, f


def ncu_traffic(name):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tp)).get(name, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def summarize(wk, r, ms, kmean, peak, parity, world):
    """Compact record of one timed workload (the `secondary` entries)."""
    traffic = ncu_traffic(wk["name"]) if world == 1 else None
    _, k_comp, achieved, f = fractions(wk, r, kmean, peak, traffic)
    d = {"metric": metric_name(wk), "workload": config_of(wk, world, r.exchange)["workload"],
         "value": round(wk["bytes_logical"] / (ms * 1e-3) / 1e9, 2), "unit": "GB/s", "ms_per_step": round(ms, 4),
         "edges_per_s": wk["E"] / (ms * 1e-3), "kernel_ms": round(kmean, 4), "kernel_achieved_gbs": round(achieved, 1),
         "frac_of_measured_hbm": round(wk["bytes_logical"] / (ms * 1e-3) / 1e9 / peak, 4),
         "bytes_logical_per_step": wk["bytes_logical"], "bytes_compulsory_per_step": wk["bytes_compulsory"],
         "traffic": traffic, "exchange": r.exchange, "exchange_passes": r.passes, "exchange_rounds": r.phases,
         "main_kernel_launches_per_step": r.calls_per_step, "src_blocks": r.n_blocks, "launch": getattr(r, "launch", "eager"),
         "parity": parity}
    d.update(f)
    return d


def run_secondary(name, world, rank, dev, exchanges, steps, warmup, peak, with_cpu=False):
    """Builds workload `name` once and times it with every exchange form in `exchanges`; {form: record}."""
    wk = build_workload(name, dev)
    res = {}
    for exchange in exchanges:
        r = Runner(wk, world, rank, dev, exchange)
        ms, kmean = time_runner(r, steps, warmup)
        par = parity_check(r)
        d = summarize(wk, r, ms, kmean, peak, par, world)
        if r.exchanged is not None:
            d["src_rows_received_per_step_rank0"], d["src_rows_full_exchange_rank0"] = r.exchanged
        d["shard_imbalance"] = round(r.imbalance, 4)
        if with_cpu and rank == 0:
            d["cpu_baseline"], _, _ = cpu_arm(wk, warmup, steps)
        res[exchange] = d
        del r
        torch.cuda.empty_cache()
    del wk
    torch.cuda.empty_cache()
    return res


def e2e_multi(r, wk, world, rank, dev, n_e2e):
    """e2e at N > 1: every rank's operands start in pinned HOST memory; per step the rank copies ITS OWN src rows (1/N
    of the matrix) and its edge weights host->device, the src rows are exchanged GPU-to-GPU over NVLink exactly as in
    the device-resident step, and the rank's dst rows go device->host.  The shard's index arrays are resident (a GNN's
    graph is static).  Time = max over ranks between two barriers; bytes = sum over ranks."""
    import torch.distributed as dist
    ok, moved, e2e_step = 1, [0, 0], None
    big = (not r.gather) and (r.E * r.W * wk["esize"]) > 8e9          # edge-aligned src too large to pin
    try:
        if r.E > 0 and not big:
            src_dev = r.src_operand()
            h_x = src_dev.cpu().pin_memory()
            h_w = r.w.cpu().pin_memory() if r.w is not None else None
            h_out = torch.empty(r.out.shape, dtype=r.out.dtype).pin_memory()
            d_x, d_w = torch.empty_like(src_dev), (torch.empty_like(r.w) if r.w is not None else None)
            moved = [h_x.numel() * h_x.element_size() + (h_w.numel() * h_w.element_size() if h_w is not None else 0),
                     h_out.numel() * h_out.element_size()]

            def e2e_step():
                d_x.copy_(h_x, non_blocking=True)
                if d_w is not None:
                    d_w.copy_(h_w, non_blocking=True)
                r.reduce(d_x, d_w, r.out)
                h_out.copy_(r.out, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        elif big:
            ok = 0
    except Exception as ex:      # local failure only: the ranks agree on `ok` before any collective of this leg
        ok = 0
        print("rank %d: e2e leg failed: %r" % (rank, ex), file=sys.stderr)
    flag = torch.tensor([float(1 - ok)], device=dev, dtype=torch.float64)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    if flag.item() != 0:
        return None

    def one():
        if e2e_step is not None:
            e2e_step()
        elif r.bg is not None or r.exchange == "allgather":     # an empty shard still takes part in the exchange
            r.reduce(r.src_operand(), r.w, r.out)
    one()
    barrier(world)
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        one()
    barrier(world)
    el = (time.perf_counter() - t0) / n_e2e
    t = torch.tensor([el], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    b = torch.tensor([float(moved[0]), float(moved[1])], device=dev, dtype=torch.float64)
    dist.all_reduce(b, op=dist.ReduceOp.SUM)
    e2e_s = t[0].item()
    return {"value": round(wk["bytes_logical"] / e2e_s / 1e9, 2), "unit": "GB/s",
            "h2d_bytes_per_step": int(b[0].item()), "d2h_bytes_per_step": int(b[1].item()),
            "ms_per_step": round(e2e_s * 1e3, 3), "steps": n_e2e, "edges_per_s": wk["E"] / e2e_s,
            "api": "every rank: pinned host src rows of its own shard + edge weights -> device, geot_b200.dist exchange + "
                   "C-ABI reduction as in the device-resident step, dst rows -> pinned host; index arrays resident; timed "
                   "between two barriers, max over ranks; bytes summed over ranks"}


def e2e_single(r, wk, n_e2e):
    """e2e at N == 1: host buffers through the C ABI's resident host graph; the stateless host entry beside it."""
    abi = r.abi
    E, S, N, H = wk["E"], wk["S"], wk["N"], wk["H"]
    hx = wk["x"].cpu().pin_memory()
    hdi = r.di.cpu().pin_memory()
    hsi = r.si.cpu().pin_memory() if r.si is not None else None
    hw = r.w.cpu().pin_memory() if r.w is not None else None
    hout = torch.empty(r.out.shape, dtype=r.out.dtype).pin_memory()
    r.step()
    torch.cuda.synchronize()
    dev_out = r.out.cpu()
    layout = r.layout
    t0 = time.perf_counter()
    hg = abi.HostGraph(hsi, hdi, S, N if hsi is not None else 0)
    create_s = time.perf_counter() - t0
    call = lambda: hg.reduce(hx, hw, "sum", H=H, weight_layout=layout, out=hout)
    call()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        call()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / n_e2e
    h2d, d2h, resident = hg.last_transfer()
    tol = 1e-5 if wk["dtype"] == torch.float32 else 1e-2
    match = bool(((hout.double() - dev_out.double()).abs() <= 4 * tol * dev_out.double().abs().clamp_min(1e-30)).all())
    hg.close()
    st_call = lambda: abi.segment_reduce_host(hx, hsi, hdi, hw, "sum", S=S, H=H, weight_layout=layout, out=hout)
    st_call()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        st_call()
    torch.cuda.synchronize()
    st_s = (time.perf_counter() - t0) / n_e2e
    st_h2d, st_d2h = abi.host_last_transfer()
    abi.lib().geot_b200_host_arena_release()
    return {"value": round(wk["bytes_logical"] / e2e_s / 1e9, 2), "unit": "GB/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_s * 1e3, 3), "steps": n_e2e, "edges_per_s": E / e2e_s,
            "matches_device_result": match,
            "resident": {"index_bytes_uploaded_once": resident, "create_ms": round(create_s * 1e3, 1)},
            "api": "geot_b200_host_graph_reduce (C ABI; index arrays uploaded once by geot_b200_host_graph_create, outside the "
                   "timed region; per step pinned host src + weights H2D, kernels, dst D2H; host wall clock)",
            "stateless": {"api": "geot_b200_segment_reduce_host (every operand incl. the index arrays from the host each call)",
                          "ms_per_step": round(st_s * 1e3, 3), "value": round(wk["bytes_logical"] / st_s / 1e9, 2),
                          "h2d_bytes_per_step": st_h2d, "d2h_bytes_per_step": st_d2h}}


def run_own(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import geot_b200  # noqa: F401

    peak, peak_src = measured_peak_gbs()
    exchange = os.environ.get("GEOT_B200_EXCHANGE", "push")
    if exchange not in ("bucket", "push", "allgather", "replicated"):
        raise SystemExit("GEOT_B200_EXCHANGE must be bucket, push, allgather or replicated")
    wk = build_workload(args.workload, dev)
    r = Runner(wk, world, rank, dev, exchange)
    sampler = ClockSampler(local) if rank == 0 else None
    ms_per_step, kmean = time_runner(r, args.steps, args.warmup, sampler, keep_output=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # N > 1: each rank holds the output rows of its shard; rank 0 writes them assembled
        out = r.timed_output if world == 1 else r.gdist.all_gather_rows(r.timed_output, r.shard.row_bounds)
        if rank == 0:
            dump_outputs(out, args.dump_outputs)
        del r.timed_output, out
    value = wk["bytes_logical"] / (ms_per_step * 1e-3) / 1e9
    parity = parity_check(r)

    traffic = ncu_traffic(wk["name"]) if world == 1 else None
    _, k_comp, achieved, fr = fractions(wk, r, kmean, peak, traffic)
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic, "kernel": "geot::segment_reduce_kernel", "kernel_ms": round(kmean, 4),
                "kernel_share_of_step": round(kmean / ms_per_step, 4), "peak_source": peak_src,
                "frac_of_nominal_8000": round(achieved / 8000.0, 4),
                "note": "achieved = logical bytes per launch (rank 0's shard at N > 1) / CUDA-event duration of the main kernel "
                        "alone (events recorded by the library around it, in a second loop of the same K steps run right after the timed loop, "
                        "so that the timed steps carry no instrumentation; N > 1: all reduction launches of a step, slowest rank).  "
                        "For gathers the logical bytes include L2-served re-reads of src rows (SURVEY 8d), so `frac` = "
                        "frac_logical can exceed 1 and is NOT an HBM fraction: frac_dram (ncu dram bytes / kernel time) is what "
                        "the DRAM interface carried, frac_compulsory what it had to carry at least (%d bytes per launch)" % k_comp}
    roofline.update(fr)
    cfg = config_of(wk, world, r.exchange)
    cfg["src_blocks"] = ("%d (the edge list regrouped once per graph by src-row block for the L2; one pass per block, later passes "
                         "accumulate)" % r.n_blocks) if r.n_blocks > 1 else "1 (one pass)"
    if r.bg is not None:
        cfg["exchange_passes"] = ("%d (%s)" % (r.passes, "src-local bucket overlapped with the exchange, src-remote bucket accumulated"
                                                 if r.passes == 2 else "exchange, then one reduction over own + received rows"))
        cfg["exchange_rounds"] = r.phases
        cfg["main_kernel_launches_per_step"] = r.calls_per_step
    cfg["launch"] = getattr(r, "launch", "eager")
    meta = dict(metric=metric_name(wk), dtype=DTYPE_NAME[wk["dtype"]], config=cfg, E=wk["E"],
                launches=r.launches_per_step, exchange=r.exchange, imbalance=r.imbalance, exchanged=r.exchanged)

    n_e2e = args.steps
    cpu_obj = None
    if world > 1:
        e2e = e2e_multi(r, wk, world, rank, dev, n_e2e)
        if e2e is None:
            e2e = {"value": round(value, 2), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "note": "N > 1: the host-buffer leg was skipped (edge-aligned src too large to pin) or failed on some rank "
                           "(stderr); this repeats the device-resident value"}
    else:
        e2e = e2e_single(r, wk, n_e2e)
        cpu_obj, _, _ = cpu_arm(wk, args.warmup, args.steps)
    del r, wk
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations (every rank takes part at N > 1) ---------------------------------------
    secondary = {}
    if args.workload == "reddit_gws" and os.environ.get("GEOT_B200_BENCH_SECONDARY", "1") == "1":
        if world > 1:
            other = "push" if exchange != "push" else "bucket"
            for name in ("products_gs64", "products_gs256"):
                got = run_secondary(name, world, rank, dev, [exchange, other, "replicated"], args.steps, args.warmup, peak)
                secondary[name] = {
                    "inclusive": got[exchange], "inclusive_alt": got[other], "replicated": got["replicated"],
                    "note": "strong scaling of BASELINE configs[2]; `inclusive` moves the src rows inside the step with the "
                            "default exchange, `inclusive_alt` with the other overlapped transport, `replicated` is the "
                            "kernel-scaling number (src pre-replicated, SURVEY 8e)"}
        else:
            for name, cpu in (("reddit_index_scatter", False), ("config1_index_scatter", True), ("products_gs64", False),
                              ("products_gs64_gaps", False), ("products_gs256", False), ("arxiv_mh_spmm", False)):
                try:
                    secondary[name] = run_secondary(name, 1, 0, dev, ["none"], args.steps, args.warmup, peak, with_cpu=cpu)["none"]
                except Exception as ex:       # a secondary line must not cost the headline
                    secondary[name] = {"error": repr(ex)}
                    torch.cuda.empty_cache()
            if "error" not in secondary.get("products_gs64_gaps", {"error": 1}):
                secondary["products_gs64_gaps"]["note"] = (
                    "products shape with 25 % of the dst rows isolated: exactly the rows without edges are zeroed, by a small "
                    "kernel that reads them off the cached plan's row pointer (no memset of dst; the parity check covers the "
                    "empty rows); compare with products_gs64")

    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    line = {
        "metric": meta["metric"], "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": meta["dtype"], "data": "synthetic", "config": meta["config"],
        "edges_per_s": meta["E"] / (ms_per_step * 1e-3), "frac_of_measured_hbm": round(value / peak, 4),
        "frac_of_nominal_8000": round(value / 8000.0, 4),
        "roofline": roofline, "cpu_baseline": cpu_obj, "e2e": e2e, "parity": parity,
        "gpu_launches": meta["launches"] * args.steps, "clocks": clocks, "exchange": meta["exchange"],
        "shard_imbalance": round(meta["imbalance"], 4), "secondary": secondary,
    }
    if meta["exchanged"] is not None:
        line["config"]["src_rows_received_per_step_rank0"] = meta["exchanged"][0]
        line["config"]["src_rows_full_exchange_rank0"] = meta["exchanged"][1]
    print(json.dumps(line))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every timed loop: each workload on the GPU, the "
                    "host-buffer (e2e) legs and the CPU baselines")
    ap.add_argument("--warmup", type=int, default=5, help="untimed steps before each timed loop (at least 3 on the GPU)")
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="reddit_gws", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step to DIR/output.npy (see dump_outputs); with N > 1 "
                         "GPUs rank 0 writes the output assembled from every rank's rows")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs applies to --impl own")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
