"""bench.py's host logic on CPU: the JSON contract at N = 1 and the sharded flow at N = 2 (gloo), with the CUDA
runtime and C-ABI calls replaced by stand-ins (tests/helpers/bench_emulation.py: the oracle plays the kernels).
Numbers are meaningless here; keys, shapes and the collective sequence of every rank are what is checked."""
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONTRACT = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "parity", "secondary"]


def test_single_gpu_line_contract():
    # a fresh interpreter: the emulation monkeypatches torch.cuda and must not leak into the other tests
    code = ("import sys, json; sys.path.insert(0, %r); sys.path.insert(0, %r); from helpers import bench_emulation as be; "
            "be.install(); print(json.dumps(be.run_own('config1_index_scatter')))" % (ROOT, os.path.join(ROOT, "tests")))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert [k for k in CONTRACT if k not in line] == []
    assert line["n_gpus"] == 1 and line["higher_is_better"] is True and line["vs_baseline"] is None and line["dtype"] == "f32"
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "frac_logical", "frac_dram", "frac_compulsory"} <= set(line["roofline"])
    assert line["parity"]["ok"] is True and line["parity"]["rows_checked"] > 3
    assert line["e2e"]["matches_device_result"] is True and "stateless" in line["e2e"] and "resident" in line["e2e"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert "workload" in line["config"] and line["gpu_launches"] > 0


def _timed_output(workload):
    """What the timed step computes on `workload`'s seeded inputs under the emulation (the oracle plays the kernels)."""
    import bench
    import oracle
    wk = bench.build_workload(workload, "cpu")
    return wk, oracle.segment_reduce(wk["x"], wk["si"], wk["di"], wk["w"], "sum", S=wk["S"], H=wk["H"])


def test_dump_outputs(tmp_path):
    """--dump-outputs: the timed step's output as float32 .npy, whole or as a seeded sample of rows, the same from run to
    run."""
    import numpy as np
    whole, sampled = str(tmp_path / "whole"), str(tmp_path / "sampled")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); from helpers import bench_emulation as be; "
            "be.install(); import bench; be.run_own('config1_index_scatter', dump_outputs=%r); "
            "bench.DUMP_BYTES = 1 << 20; be.run_own('config1_index_scatter', dump_outputs=%r)"
            % (ROOT, os.path.join(ROOT, "tests"), whole, sampled))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(whole)) == ["output.npy"] and sorted(os.listdir(sampled)) == ["output.npy", "output_rows.npy"]
    full = np.load(os.path.join(whole, "output.npy"))
    assert full.dtype == np.float32 and full.shape == (50_000, 64)        # config #1: S = 50,000 segments, F = 64
    part, rows = np.load(os.path.join(sampled, "output.npy")), np.load(os.path.join(sampled, "output_rows.npy"))
    assert part.dtype == np.float32 and rows.dtype == np.float64 and part.nbytes <= 1 << 20
    assert part.shape == (rows.size, 64) and bool((np.diff(rows) > 0).all())
    assert np.array_equal(part, full[rows.astype(np.int64)])
    assert np.array_equal(full, _timed_output("config1_index_scatter")[1].numpy())


@pytest.mark.parametrize("exchange", ["bucket", "allgather", "replicated"])
def test_two_rank_flow_gloo(exchange, tmp_path):
    import numpy as np
    from helpers import bench_emulation as be
    dump = str(tmp_path / "dump")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=be.worker, args=(r, 2, port, exchange, "arxiv_mh_spmm", q, dump)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
    codes = [p.exitcode for p in procs]
    for p in procs:
        if p.is_alive():
            p.kill()
    assert codes == [0, 0], codes
    line = q.get(timeout=5)
    assert [k for k in CONTRACT if k not in line] == []
    assert line["n_gpus"] == 2 and line["exchange"] == exchange and line["scaling"] == "strong"
    # the N > 1 end-to-end leg ran on both ranks: bytes are summed over ranks (src rows + weights in, dst rows out)
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0 and "ms_per_step" in line["e2e"]
    assert line["parity"]["ok"] is True and line["parity"]["rows_checked"] > 6        # both ranks' rows
    if exchange == "bucket":
        got, full = line["config"]["src_rows_received_per_step_rank0"], line["config"]["src_rows_full_exchange_rank0"]
        assert 0 < got == full
    # --dump-outputs at N > 1: rank 0 writes the output assembled from both ranks' rows
    part, rows = np.load(os.path.join(dump, "output.npy")), np.load(os.path.join(dump, "output_rows.npy")).astype(np.int64)
    wk, exp = _timed_output("arxiv_mh_spmm")
    assert part.dtype == np.float32 and part.shape == (rows.size, wk["H"], wk["F"]) and int(rows[-1]) < wk["S"]
    exp = exp[torch.from_numpy(rows)].double()
    assert bool(((torch.from_numpy(part).double() - exp).abs() <= 1e-2 * exp.abs().clamp_min(1e-3)).all())
