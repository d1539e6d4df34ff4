"""Timings of the fused dot-product graph attention (geot::graph_attention) against the composed forward
(sddmm_mh_impl -> segment_softmax -> mh_spmm), of its backward (the dst pass alone, and the whole autograd backward with
the two transposed mh_spmm passes), and of one TransformerConv forward + backward step against the same layer restated
on torch ops (gathers, scatter_reduce / exp / index_add softmax, index_add aggregation).  Shapes: the arxiv graph of
BASELINE config #4 at 8 x 32 in bf16 and fp32 (input width 128), and the Reddit graph at 4 x 32 in fp32 (input width
602), where the torch restatement is not run (its [E, H * F] tensors are 58.7 GB each).  CUDA events, best / median of
--steps after --warmup; one JSON line per shape, with the card's name and power limit read in the same run.  Bench
support, not product.

    python scripts/bench_graph_attention.py > bench_graph_attention.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import geot_b200  # noqa: E402
import workloads as wl  # noqa: E402
from geot_b200 import abi  # noqa: E402
from geot_b200.gnn import TransformerConv  # noqa: E402


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


def torch_transformer(conv, x, si, di):
    """TransformerConv restated on torch ops."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    q, k, v = conv.lin_query(x).view(N, H, F), conv.lin_key(x).view(N, H, F), conv.lin_value(x).view(N, H, F)
    score = (q[di] * k[si]).sum(-1) / math.sqrt(F)
    idx = di.view(-1, 1).expand_as(score)
    m = torch.full((N, H), float("-inf"), dtype=x.dtype, device=x.device).scatter_reduce(0, idx, score.detach(), "amax")
    ex = (score - m[di]).exp()
    den = torch.zeros(N, H, dtype=x.dtype, device=x.device).index_add(0, di, ex)
    out = torch.zeros(N, H, F, dtype=x.dtype, device=x.device).index_add(0, di, (ex / den[di]).unsqueeze(-1) * v[si])
    return out.reshape(N, H * F) + conv.lin_skip(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    assert a.steps >= 10, "best / median of at least 10 steps"
    dev = "cuda"
    gpu = card()
    for gname, H, F, F_in, dtype in (("arxiv", 8, 32, 128, torch.bfloat16), ("arxiv", 8, 32, 128, torch.float32),
                                     ("reddit", 4, 32, 602, torch.float32)):
        g = wl.power_law_graph(gname, dev)
        N, E, si, di = g.num_nodes, g.num_edges, g.src_index, g.dst_index
        W = H * F
        scale = 1 / math.sqrt(F)
        gen = torch.Generator(device=dev).manual_seed(0)
        q, k, v = (torch.randn(N, H, F, generator=gen, device=dev).to(dtype) for _ in range(3))
        gout = torch.randn(N, H, F, generator=gen, device=dev).to(dtype)
        s = q.element_size()
        acc = 8 if dtype == torch.float64 else 4
        rec = {"graph": gname, "N": N, "E": E, "H": H, "F": F, "dtype": str(dtype).replace("torch.", ""), "gpu": gpu,
               "steps": a.steps, "warmup": a.warmup}
        T = lambda fn: timed(fn, a.warmup, a.steps)  # noqa: E731
        out, lse = torch.ops.geot.graph_attention(q, k, v, si, di, scale)     # plan of dst_index, outside the timing
        rec["fused_fwd_ms"] = T(lambda: torch.ops.geot.graph_attention(q, k, v, si, di, scale))
        # logical bytes: k and v rows per edge, 16 index bytes per edge; per dst row the q row, the out row and lse
        rec["fused_fwd_logical_bytes"] = E * (2 * W * s + 16) + N * (2 * W * s + H * acc)
        rec["fused_fwd_GBps_logical"] = round(rec["fused_fwd_logical_bytes"] / rec["fused_fwd_ms"]["best"] / 1e6, 1)

        def composed():
            sc = torch.ops.geot.sddmm_mh_impl(si, di, q, k, False) * scale
            alpha = torch.ops.geot.segment_softmax(sc, di)
            return torch.ops.geot.mh_spmm(si, di, alpha, v, "sum")
        ref = composed()
        rec["fused_vs_composed_max_abs_diff"] = float((ref.float() - out[: ref.shape[0]].float()).abs().max())
        rec["composed_fwd_ms"] = T(composed)
        rec["sddmm_mh_ms"] = T(lambda: torch.ops.geot.sddmm_mh_impl(si, di, q, k, False))
        sc = torch.ops.geot.sddmm_mh_impl(si, di, q, k, False)
        rec["segment_softmax_ms"] = T(lambda: torch.ops.geot.segment_softmax(sc, di))
        alpha = torch.ops.geot.segment_softmax(sc, di)
        rec["mh_spmm_ms"] = T(lambda: torch.ops.geot.mh_spmm(si, di, alpha, v, "sum"))
        rec["fused_speedup_vs_composed"] = round(rec["composed_fwd_ms"]["best"] / rec["fused_fwd_ms"]["best"], 2)
        del sc, alpha, ref
        pd = abi.DevicePlan(di)
        rec["grad_dst_pass_ms"] = T(lambda: abi.graph_attention_grad(q, k, v, out, lse, gout, si, di, scale, pd))
        # logical bytes: k and v rows per edge, 16 index bytes, p and ds out; per dst row q, g, out in and grad_q out
        rec["grad_dst_pass_GBps_logical"] = round((E * (2 * W * s + 16 + 2 * H * s) + N * (4 * W * s + H * acc))
                                                  / rec["grad_dst_pass_ms"]["best"] / 1e6, 1)
        qq, kk, vv = (t.clone().requires_grad_(True) for t in (q, k, v))

        def fwd_bwd():
            qq.grad = kk.grad = vv.grad = None
            geot_b200.graph_attention(qq, kk, vv, si, di).backward(gout)
        rec["op_fwd_bwd_ms"] = T(fwd_bwd)
        del qq, kk, vv, pd
        torch.manual_seed(0)
        conv = TransformerConv(F_in, F, heads=H).to(dev).to(dtype)
        x = wl.features(N, F_in, dtype, dev).requires_grad_(True)
        go = wl.features(N, H * F, dtype, dev, seed=5)

        def step(fwd):
            def run():
                conv.zero_grad(set_to_none=True)
                x.grad = None
                fwd(conv, x, si, di).backward(go)
            return run
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        rec["transformerconv_fwd_bwd_ms"] = T(step(lambda c, x, si, di: c(x, si, di)))
        rec["transformerconv_peak_bytes"] = torch.cuda.max_memory_allocated()
        if gname == "arxiv":
            torch.cuda.reset_peak_memory_stats()
            rec["torch_transformerconv_fwd_bwd_ms"] = T(step(torch_transformer))
            rec["torch_transformerconv_peak_bytes"] = torch.cuda.max_memory_allocated()
            rec["transformerconv_speedup_vs_torch"] = round(rec["torch_transformerconv_fwd_bwd_ms"]["best"]
                                                            / rec["transformerconv_fwd_bwd_ms"]["best"], 2)
        print(json.dumps(rec), flush=True)
        del conv, x, go, g, si, di, q, k, v, gout, out, lse
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
