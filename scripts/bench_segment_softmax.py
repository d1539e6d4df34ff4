"""Timings of the segment softmax (geot::segment_softmax) and its backward against the torch restatement a user would
otherwise write (scatter_reduce amax, gather, exp, index_add, gather, divide; backward: index_add of out * grad, gather,
multiply), and at arxiv one GATConv forward + backward step against the same layer restated on torch ops.  Shapes:
the arxiv graph of BASELINE config #4 at 8 heads in bf16 and fp32, and the Reddit graph at 4 heads in fp32 (index and
logits far beyond the L2).  CUDA events, best / median of --steps after --warmup; one JSON line per shape, with the
card's name and power limit read in the same run.  Bench support, not product.

    python scripts/bench_segment_softmax.py > bench_segment_softmax.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import geot_b200  # noqa: E402
import workloads as wl  # noqa: E402
from geot_b200.gnn import GATConv  # noqa: E402


def timed(fn, warmup, steps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return {"best": round(ts[0], 4), "median": round(ts[len(ts) // 2], 4)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def torch_softmax(logits, di, S):
    idx = di.view(-1, 1).expand_as(logits)
    m = torch.full((S, logits.shape[1]), float("-inf"), dtype=logits.dtype, device=logits.device)
    m = m.scatter_reduce(0, idx, logits, "amax")
    ex = (logits - m[di]).exp()
    den = torch.zeros(S, logits.shape[1], dtype=logits.dtype, device=logits.device).index_add(0, di, ex)
    return ex / den[di]


def torch_softmax_backward(out, grad, di, S):
    dot = torch.zeros(S, out.shape[1], dtype=out.dtype, device=out.device).index_add(0, di, out * grad)
    return out * (grad - dot[di])


def torch_gat(conv, x, si, di):
    """GATConv restated on torch ops: the softmax above and an index_add aggregation."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    h = conv.lin(x).view(N, H, F)
    logits = torch.nn.functional.leaky_relu((h * conv.att_src).sum(-1)[si] + (h * conv.att_dst).sum(-1)[di],
                                            conv.negative_slope)
    alpha = torch_softmax(logits, di, N)
    out = torch.zeros(N, H, F, dtype=x.dtype, device=x.device).index_add(0, di, alpha.unsqueeze(-1) * h[si])
    return out.reshape(N, H * F) + conv.bias


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    assert a.steps >= 10, "best / median of at least 10 steps"
    dev = "cuda"
    gpu = card()
    for gname, H, dtype in (("arxiv", 8, torch.bfloat16), ("arxiv", 8, torch.float32), ("reddit", 4, torch.float32)):
        g = wl.power_law_graph(gname, dev)
        N, E, si, di = g.num_nodes, g.num_edges, g.src_index, g.dst_index
        S = int(di[-1]) + 1
        gen = torch.Generator(device=dev).manual_seed(0)
        logits = (torch.rand(E, H, generator=gen, device=dev) * 20 - 10).to(dtype)
        grad = torch.randn(E, H, generator=gen, device=dev).to(dtype)
        s = logits.element_size()
        rec = {"graph": gname, "N": N, "E": E, "H": H, "dtype": str(dtype).replace("torch.", ""), "gpu": gpu,
               "steps": a.steps, "warmup": a.warmup}
        T = lambda fn: timed(fn, a.warmup, a.steps)  # noqa: E731
        out = geot_b200.segment_softmax(logits, di)     # builds and caches the plan outside the timed region
        rec["forward_ms"] = T(lambda: torch.ops.geot.segment_softmax(logits, di))
        rec["forward_GBps_logical"] = round(E * (8 + 2 * H * s) / rec["forward_ms"]["best"] / 1e6, 1)
        rec["backward_ms"] = T(lambda: torch.ops.geot.segment_softmax_backward(out, grad, di))
        rec["backward_GBps_logical"] = round(E * (8 + 3 * H * s) / rec["backward_ms"]["best"] / 1e6, 1)
        rec["torch_forward_ms"] = T(lambda: torch_softmax(logits, di, S))
        rec["torch_backward_ms"] = T(lambda: torch_softmax_backward(out, grad, di, S))
        rec["forward_speedup_vs_torch"] = round(rec["torch_forward_ms"]["best"] / rec["forward_ms"]["best"], 2)
        rec["backward_speedup_vs_torch"] = round(rec["torch_backward_ms"]["best"] / rec["backward_ms"]["best"], 2)
        ref = torch_softmax(logits.double(), di, S)
        rec["forward_max_abs_diff_vs_fp64"] = float((out.double() - ref).abs().max())
        del ref
        if gname == "arxiv":
            F_in, F = 128, 32
            torch.manual_seed(0)
            conv = GATConv(F_in, F, heads=H).to(dev).to(dtype)
            x = wl.features(N, F_in, dtype, dev).requires_grad_(True)
            gout = wl.features(N, H * F, dtype, dev, seed=5)

            def step(fwd):
                def run():
                    conv.zero_grad(set_to_none=True)
                    x.grad = None
                    fwd(conv, x, si, di).backward(gout)
                return run
            rec["gat_fwd_bwd_ms"] = T(step(lambda c, x, si, di: c(x, si, di)))
            rec["torch_gat_fwd_bwd_ms"] = T(step(torch_gat))
            rec["gat_speedup_vs_torch"] = round(rec["torch_gat_fwd_bwd_ms"]["best"] / rec["gat_fwd_bwd_ms"]["best"], 2)
            del conv, x, gout
        print(json.dumps(rec), flush=True)
        del g, si, di, logits, grad, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
