"""Timings of the fused GATv2 attention score (geot::gatv2_score) and its two backward passes, and one GATv2Conv
forward + backward step against the same layer restated on torch ops (gathers, leaky_relu, a product with att, the
softmax of scatter_reduce / exp / index_add, an index_add aggregation).  Shapes: the arxiv graph of BASELINE config #4
at 8 x 32 in bf16 and fp32 (input width 128), and the Reddit graph at 4 x 32 in fp32 (input width 602) with the fused
layer only: there the restatement's [E, H * F] tensors are recorded as computed bytes instead of being allocated.
The multi-head SDDMM (geot::sddmm_mh_impl, the weight gradient of mh_spmm) on the same shape is timed beside the score:
it moves the same bytes.  CUDA events, best / median of --steps after --warmup; one JSON line per shape, with the
card's name and power limit read in the same run.  Bench support, not product.

    python scripts/bench_gatv2.py > bench_gatv2.jsonl
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
from geot_b200 import abi  # noqa: E402
from geot_b200.gnn import GATv2Conv  # noqa: E402
from geot_b200.transpose import transposed_edges  # noqa: E402


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


def torch_gatv2(conv, x, si, di):
    """GATv2Conv restated on torch ops."""
    N, H, F = x.shape[0], conv.heads, conv.out_channels
    xl = conv.lin_l(x).view(N, H, F)
    xr = conv.lin_r(x).view(N, H, F)
    score = (conv.att * torch.nn.functional.leaky_relu(xl[si] + xr[di], conv.negative_slope)).sum(-1)
    idx = di.view(-1, 1).expand_as(score)
    m = torch.full((N, H), float("-inf"), dtype=x.dtype, device=x.device).scatter_reduce(0, idx, score.detach(), "amax")
    ex = (score - m[di]).exp()
    den = torch.zeros(N, H, dtype=x.dtype, device=x.device).index_add(0, di, ex)
    alpha = ex / den[di]
    out = torch.zeros(N, H, F, dtype=x.dtype, device=x.device).index_add(0, di, alpha.unsqueeze(-1) * xl[si])
    return out.reshape(N, H * F) + conv.bias


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
        gen = torch.Generator(device=dev).manual_seed(0)
        x_l = torch.randn(N, H, F, generator=gen, device=dev).to(dtype)
        x_r = torch.randn(N, H, F, generator=gen, device=dev).to(dtype)
        att = torch.randn(H, F, generator=gen, device=dev).to(dtype)
        grad = torch.randn(E, H, generator=gen, device=dev).to(dtype)
        s = x_l.element_size()
        rows_d, rows_s = int(di[-1]) + 1, int(si.max()) + 1
        rec = {"graph": gname, "N": N, "E": E, "H": H, "F": F, "dtype": str(dtype).replace("torch.", ""), "gpu": gpu,
               "steps": a.steps, "warmup": a.warmup}
        T = lambda fn: timed(fn, a.warmup, a.steps)  # noqa: E731
        geot_b200.gatv2_score(x_l, x_r, att, si, di)           # plan of dst_index, outside the timed region
        t = transposed_edges(si, di)
        pd, ps = abi.DevicePlan(di), abi.DevicePlan(t.dst_index)
        g_t = abi.permute_edges(grad, t.perm)
        rec["score_ms"] = T(lambda: torch.ops.geot.gatv2_score(x_l, x_r, att, si, di, 0.2))
        # logical bytes: two rows per edge (the x_r row is re-used while dst repeats: counted anyway), 16 index bytes,
        # the H outputs
        rec["score_GBps_logical"] = round(E * (2 * W * s + 16 + H * s) / rec["score_ms"]["best"] / 1e6, 1)
        rec["sddmm_mh_same_shape_ms"] = T(lambda: torch.ops.geot.sddmm_mh_impl(si, di, x_r, x_l, False))
        rec["grad_dst_pass_ms"] = T(lambda: abi.gatv2_grad(x_r, x_l, att, grad, di, si, N, 0.2, True, pd))
        rec["grad_dst_pass_GBps_logical"] = round((E * (W * s + 16 + H * s) + rows_d * W * s)
                                                  / rec["grad_dst_pass_ms"]["best"] / 1e6, 1)
        rec["grad_src_pass_ms"] = T(lambda: abi.gatv2_grad(x_l, x_r, att, g_t, t.dst_index, t.src_index, N, 0.2, False,
                                                           ps))
        rec["grad_src_pass_GBps_logical"] = round((E * (W * s + 16 + H * s) + rows_s * W * s)
                                                  / rec["grad_src_pass_ms"]["best"] / 1e6, 1)
        rec["torch_restatement_one_EHF_tensor_bytes"] = E * W * s
        del g_t
        torch.manual_seed(0)
        conv = GATv2Conv(F_in, F, heads=H).to(dev).to(dtype)
        x = wl.features(N, F_in, dtype, dev).requires_grad_(True)
        gout = wl.features(N, H * F, dtype, dev, seed=5)

        def step(fwd):
            def run():
                conv.zero_grad(set_to_none=True)
                x.grad = None
                fwd(conv, x, si, di).backward(gout)
            return run
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        rec["gatv2conv_fwd_bwd_ms"] = T(step(lambda c, x, si, di: c(x, si, di)))
        rec["gatv2conv_peak_bytes"] = torch.cuda.max_memory_allocated()
        if gname == "arxiv":
            torch.cuda.reset_peak_memory_stats()
            rec["torch_gatv2conv_fwd_bwd_ms"] = T(step(torch_gatv2))
            rec["torch_gatv2conv_peak_bytes"] = torch.cuda.max_memory_allocated()
            rec["gatv2conv_speedup_vs_torch"] = round(rec["torch_gatv2conv_fwd_bwd_ms"]["best"]
                                                      / rec["gatv2conv_fwd_bwd_ms"]["best"], 2)
        print(json.dumps(rec), flush=True)
        del conv, x, gout, g, si, di, x_l, x_r, att, grad, t
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
