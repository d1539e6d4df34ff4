"""SASS evidence for the shipped kernels (no GPU needed): per default kernel of the library the counts of the memory
instructions that characterise its data path -- LDGSTS (cp.async), LDG / LDS / STG widths, REDG / ATOMG (atomics), UBLKCP
/ UTMALDG (TMA) -- from `cuobjdump -sass` of the built objects.
    python scripts/sass_summary.py > profiles/<tag>_sass_default_kernels.md
Bench support, not product."""
import collections, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WANT = [  # (object, demangled-name filter, what it is)
    ("inst_f32_0.o", "segment_reduce_kernel<float, 4, 32, 1, 0, 1, 35>", "gather_weight_scatter F=128 fp32 (Reddit gws, one pass): plain lean ring, depth 3"),
    ("inst_f32_0.o", "segment_reduce_kernel<float, 4, 32, 1, 0, 1, 99>", "the same with the segment_reduce_ex options (src-blocked / bucketed passes)"),
    ("inst_f32_0.o", "segment_reduce_kernel<float, 4, 32, 1, 0, 0, 39>", "index_scatter F=128 fp32 (Reddit index_scatter): lean ring, depth 7"),
    ("inst_f32_0.o", "segment_reduce_kernel<float, 4, 16, 1, 0, 0, 35>", "gather_scatter F=64 fp32 (products gs64)"),
    ("inst_f32_0.o", "segment_reduce_kernel<float, 4, 32, 2, 0, 0, 35>", "gather_scatter F=256 fp32 (products gs256)"),
    ("inst_bf16_0.o", "segment_reduce_kernel<__nv_bfloat16, 8, 32, 1, 0, 2, 163>", "mh_spmm 8x32 bf16 (arxiv): lean ring with per-head weights"),
    ("inst_f32_0.o", "segment_fixup_kernel<float, 0>", "fixup pass (programmatic dependent launch)"),
    ("sddmm.o", "sddmm_coo_kernel<float, 4, 32, 1, 2, 32, 0, geot::SddmmParams>", "SDDMM F=128 fp32 (backward of gather_weight_scatter)"),
    ("sddmm.o", "sddmm_coo_kernel<float, 4, 32, 2, 2, 8, 0, geot::SddmmParams>", "SDDMM 8 heads x 32 fp32 (weight gradient of mh_spmm, arxiv)"),
    ("exchange.o", "push_rows_kernel<uint4>", "push transport: rows into the peers' symmetric memory"),
    ("abi.o", "scatter_add_kernel<float4>", "index_scatter(sorted=False) fp32 sum: vector atomics"),
]
PAT = re.compile(r"^\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)")
KEEP = ("LDGSTS", "LDG", "LDS", "STG", "STS", "REDG", "RED", "ATOMG", "ATOM", "UBLKCP", "UTMALDG", "SHFL", "LDGDEPBAR", "DEPBAR", "ACQBULK", "SYNCS")


def kernels(obj):
    txt = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    out, name = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            name = re.sub(r"\((anonymous namespace)\)::", "", name).replace("geot::", "").replace("void ", "")
            out[name] = collections.Counter()
            continue
        m = PAT.match(line)
        if m and name:
            op = m.group(1)
            out[name]["_all"] += 1
            base = op.split(".")[0]
            if base in KEEP:
                out[name][op] += 1
    return out


print("# SASS of the shipped kernels (`cuobjdump -sass`, sm_100a): memory-path instruction counts\n")
print("Static counts per kernel (unrolled code: one count per emitted instruction, not per execution).  `LDGSTS` = cp.async "
      "(global -> shared, L1 bypass: `.BYPASS`), `REDG` = reduction atomics, `UBLKCP` / `UTMALDG` = TMA bulk / tensor copies.  "
      "The gather kernels move their rows with `LDGSTS.E.BYPASS.128` on purpose: the two TMA-filled rings were built, "
      "measured slower and removed (`r01_ring_sweep_run3_tma.txt`, `r02e_sass_gather4_ring.txt`).  No kernel on the sorted "
      "path holds an atomic.\n")
cache = {}
for obj, flt, what in WANT:
    path = os.path.join(ROOT, "build/geot_b200", obj)
    if path not in cache:
        cache[path] = kernels(path)
    hit = [(n, c) for n, c in cache[path].items() if n.startswith(flt)]
    if not hit:
        print("## `%s` -- NOT FOUND in %s\n" % (flt, obj))
        continue
    n, c = hit[0]
    print("## `%s`\n\n%s; %d SASS instructions.\n\n| instruction | count |\n|---|---:|" % (n.split("(")[0], what, c["_all"]))
    for op, k in sorted(c.items(), key=lambda x: (-x[1], x[0])):
        if op != "_all":
            print("| `%s` | %d |" % (op, k))
    print()
