"""Timings of the mh_spmm backward: the multi-head SDDMM weight gradient (geot::sddmm_mh_impl) against the composed
alternative (sddmm_coo on the [N*H, F] views with expanded indices), the src-gradient path, and the whole forward +
backward step.  Shapes: the arxiv graph of BASELINE config #4 at 8 heads x 32 in bf16 and fp32, and the Reddit graph at
4 x 32 fp32, a large attention layer whose index streams exceed the L2.  CUDA events, best / median of --steps after
--warmup; one JSON line per shape, with the card's name and power limit read in the same run.  Bench support, not
product.

    python scripts/bench_mh_backward.py > bench_mh_backward.jsonl
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    assert a.steps >= 10, "best / median of at least 10 steps"
    dev = "cuda"
    gpu = card()
    for gname, H, F, dtype in (("arxiv", 8, 32, torch.bfloat16), ("arxiv", 8, 32, torch.float32),
                               ("reddit", 4, 32, torch.float32)):
        g = wl.power_law_graph(gname, dev)
        N, E, si, di = g.num_nodes, g.num_edges, g.src_index, g.dst_index
        S = int(di[-1]) + 1
        x = wl.features(N, H * F, dtype, dev).view(N, H, F)
        grad = wl.features(S, H * F, dtype, dev, seed=5).view(S, H, F)
        w = wl.edge_weights(E, H, dtype, dev)
        s = x.element_size()
        rec = {"graph": gname, "N": N, "E": E, "H": H, "F": F, "dtype": str(dtype).replace("torch.", ""), "gpu": gpu,
               "steps": a.steps, "warmup": a.warmup}
        T = lambda fn: timed(fn, a.warmup, a.steps)  # noqa: E731
        rec["forward_ms"] = T(lambda: geot_b200.mh_spmm(si, di, w, x))
        # weight gradient: logical bytes = E * (2 rows + 16 B indices + H outputs)
        rec["wgrad_ms"] = T(lambda: torch.ops.geot.sddmm_mh_impl(si, di, grad, x, False))
        rec["wgrad_GBps_logical"] = round(E * (2 * H * F * s + 16 + H * s) / rec["wgrad_ms"]["best"] / 1e6, 1)
        # the composed alternative; its E*H expanded index pairs are built here, outside the timed region
        heads = torch.arange(H, device=dev)
        row_x = (di.view(-1, 1) * H + heads).reshape(-1)
        col_x = (si.view(-1, 1) * H + heads).reshape(-1)
        g2, x2 = grad.view(-1, F), x.view(-1, F)
        rec["wgrad_composed_ms"] = T(lambda: geot_b200.sddmm_coo_impl(col_x, row_x, g2, x2))
        rec["wgrad_speedup_vs_composed"] = round(rec["wgrad_composed_ms"]["best"] / rec["wgrad_ms"]["best"], 2)
        mine = torch.ops.geot.sddmm_mh_impl(si, di, grad, x, False).reshape(-1).double()
        theirs = geot_b200.sddmm_coo_impl(col_x, row_x, g2, x2).double()
        rec["wgrad_max_rel_diff_vs_composed"] = float(((mine - theirs).abs() / theirs.abs().clamp_min(1e-30)).max())
        del mine, theirs
        del row_x, col_x
        t = transposed_edges(si, di)

        def src_grad():
            w_perm = abi.permute_edges(w, t.perm)
            return torch.ops.geot.mh_spmm(t.src_index, t.dst_index, w_perm, grad, "sum")
        rec["src_grad_ms"] = T(src_grad)
        wr, xr = w.clone().requires_grad_(True), x.clone().requires_grad_(True)

        def step():
            wr.grad = xr.grad = None
            geot_b200.mh_spmm(si, di, wr, xr).backward(grad)
        rec["fwd_bwd_ms"] = T(step)
        if gname == "arxiv":     # at Reddit the restatement's E*W intermediates are ~59 GB each
            def torch_step():
                wr.grad = xr.grad = None
                out = torch.zeros(S, H, F, dtype=dtype, device=dev).index_add(0, di, wr.unsqueeze(-1) * xr.index_select(0, si))
                out.backward(grad)
            rec["torch_fwd_bwd_ms"] = T(torch_step)
            rec["speedup_vs_torch"] = round(rec["torch_fwd_bwd_ms"]["best"] / rec["fwd_bwd_ms"]["best"], 2)
        print(json.dumps(rec), flush=True)
        del g, si, di, x, grad, w, wr, xr, t
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
