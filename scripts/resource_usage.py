"""Static resource check of every compiled kernel (no GPU needed): registers / stack (spill) bytes per kernel from
`cuobjdump -res-usage` of the objects under build/geot_b200, written as a markdown table.
Usage: python scripts/resource_usage.py > profiles/<tag>_resource_usage.md"""
import glob, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
rows = []
for obj in sorted(glob.glob(os.path.join(ROOT, "build/geot_b200/*.o"))):
    try:
        txt = subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True).stdout
    except FileNotFoundError:
        sys.exit("cuobjdump not found")
    name = None
    for line in txt.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", line)
        if m and name:
            dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
            dem = re.sub(r"\(geot::.*\)$|\(.*Params\)$", "", dem).replace("geot::", "").replace("void ", "")
            rows.append((os.path.basename(obj), dem, int(m.group(1)), int(m.group(2))))
            name = None
print("# Static resource usage of every compiled kernel (`cuobjdump -res-usage`, sm_100a)\n")
print("Template arguments of `segment_reduce_kernel`: `<T, VECW, LPR, VPL, RED, WM, PF>` (RED 0 sum, 2 max, 3 min, 4 prod; "
      "WM 0 none, 1 per edge, 2 generic; PF 0 registers, 2/3 cp.async ring, 35/39 lean ring depth 3/7).\n")
print("%d kernels in %d objects; %d use stack (spill) memory.\n" % (len(rows), len({r[0] for r in rows}), sum(1 for r in rows if r[3])))
print("## Kernels with stack usage\n\n| object | kernel | registers | stack bytes |\n|---|---|---:|---:|")
for r in rows:
    if r[3]:
        print("| %s | `%s` | %d | %d |" % r)
print("\n## Default-dispatch kernels of the BASELINE workloads\n\n| kernel | registers | stack bytes |\n|---|---:|---:|")
want = ["segment_reduce_kernel<float, 4, 32, 1, 0, 1, 35>", "segment_reduce_kernel<float, 4, 32, 1, 0, 0, 39>",
        "segment_reduce_kernel<float, 4, 16, 1, 0, 0, 35>", "segment_reduce_kernel<float, 4, 32, 2, 0, 0, 35>",
        "segment_reduce_kernel<float, 4, 32, 2, 0, 1, 35>", "segment_reduce_kernel<float, 4, 16, 1, 0, 0, 39>",
        "segment_reduce_kernel<__nv_bfloat16, 8, 32, 1, 0, 2, 3>", "segment_fixup_kernel<float, 0>",
        "sddmm_coo_kernel<float, 4, 32, 1, 2, 32, 0, geot::SddmmParams>", "sddmm_coo_kernel<float, 4, 32, 2, 2, 8, 0, geot::SddmmParams>"]
for w in want:
    for r in rows:
        if r[1].startswith(w):
            print("| `%s` | %d | %d |" % (r[1], r[2], r[3]))
            break
    else:
        print("| `%s` | not built | |" % w)
print("\n## All kernels: registers (max per object)\n\n| object | kernels | max registers | with stack |\n|---|---:|---:|---:|")
for o in sorted({r[0] for r in rows}):
    rr = [r for r in rows if r[0] == o]
    print("| %s | %d | %d | %d |" % (o, len(rr), max(r[2] for r in rr), sum(1 for r in rr if r[3])))
