"""HBM copy bandwidth of GPU 0: a 4 GiB device-to-device copy, read + write bytes over CUDA-event time.

bench.py takes its roofline fractions against this figure when no MEASURED_PEAKS.json is present; the recorded run is
profiles/hbm_copy_b200.txt.

    python scripts/hbm_copy.py
"""
import statistics
import subprocess

import torch


def main(nbytes=4 << 30, copies=20, reps=7):
    assert torch.cuda.is_available(), "needs a GPU"
    a = torch.ones(nbytes // 4, device="cuda")
    b = torch.empty_like(a)
    for _ in range(5):
        b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gbs = []
    for _ in range(reps):
        e0.record()
        for _ in range(copies):
            b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        gbs.append(2 * nbytes * copies / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print("GPU (name, power limit, max SM clock): %s" % card)
    print("copy of %d bytes x %d per repetition, read + write GB/s of %d repetitions: %s"
          % (nbytes, copies, reps, ", ".join("%.1f" % g for g in sorted(gbs))))
    print("median: %.1f GB/s" % statistics.median(gbs))


if __name__ == "__main__":
    main()
