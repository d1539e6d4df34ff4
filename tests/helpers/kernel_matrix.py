"""Every compiled segment-reduce kernel, the inputs that reach it, and an exact reference.

* Inventory: the ``segment_reduce_kernel<T, VECW, LPR, VPL, RED, WM, PF>`` and ``segment_fixup_kernel<T, RED>``
  instantiations in the library binary, read with ``cuobjdump -res-usage`` and ``c++filt`` (as
  ``scripts/resource_usage.py`` does).  ``parse_kernel`` also normalises the kernel names a profiler reports, so a test
  can prove which instantiation a call ran.
* Case builder: ``cases_for(tuple)`` derives a call that reaches that instantiation -- dtype, row width, heads,
  weight layout, ring variant (``GEOT_B200_RING``), chunk (``GEOT_B200_CHUNK``) and the ``segment_reduce_ex``
  options -- from the dispatch rules restated in ``choose_config`` / ``dispatch`` below.
* Exact reference: inputs live on a dyadic grid (src ``k/16``, ``|k| <= 16``; weights ``j/4``, ``|j| <= 8``), so every
  product is a multiple of 2^-6 of magnitude <= 2 and every partial sum of a row whose ``sum |p|`` stays below 2^18 is
  exact in an fp32 accumulator.  The sum is then independent of the summation order, and the kernel result must equal
  the fp64 sum rounded once to the output dtype, bit for bit.  ``reference`` asserts that precondition per row.
"""
from __future__ import annotations

import contextlib
import dataclasses
import functools
import os
import re
import shutil
import subprocess
import zlib

import torch

# template argument T -> torch dtype
DTYPES = {"float": torch.float32, "double": torch.float64, "__nv_bfloat16": torch.bfloat16, "__half": torch.float16}
RED_NAMES = {0: "sum", 2: "max", 3: "min", 4: "prod"}
# PF bits (segment_reduce.cuh: kDepthMask, kLeanFlag, kExtFlag, kHeadFlag) and other kernel constants
DEPTH, LEAN, EXT, HEADW = 15, 32, 64, 128
K_THREADS, HEAD_MAX, K_LONG = 256, 8, 32
EXACT_BOUND = 2.0 ** 18      # sum |p| of a row below this: every partial sum is exact in fp32

# Compiled, but no call can reach them: a sum with per-head weights (WM 2) needs H >= 2 heads, so a row of at least two
# elements -- two vectors when each head is a whole number of vectors, two elements otherwise -- and LPR 1 means the
# row is a single vector (choose_config, abi.cu:41-45; shape.wm, abi.cu:566).
UNREACHABLE = {
    (dt, vecw, 1, 1, 0, 2, 0): "sum with per-head weights needs H >= 2 heads, i.e. more than one vector per row; "
                               "LPR 1 is chosen only for a single-vector row"
    for dt in DTYPES for vecw in (1, 16 // torch.empty((), dtype=DTYPES[dt]).element_size())
}


def esize(dt: str) -> int:
    return torch.empty((), dtype=DTYPES[dt]).element_size()


def tuple_id(t) -> str:
    return "-".join(str(x) for x in t).replace("__nv_", "").replace("__", "")


# ---- inventory ----------------------------------------------------------------------------------------------------
def _tool(name: str) -> str:
    p = shutil.which(name)
    if p:
        return p
    for root in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if root and os.path.exists(os.path.join(root, "bin", name)):
            return os.path.join(root, "bin", name)
    raise RuntimeError("%s not found (PATH, $CUDA_HOME/bin, /usr/local/cuda/bin)" % name)


_KERNEL = re.compile(r"\b(segment_reduce_kernel|segment_fixup_kernel)<([^<>]*)>")


def parse_kernel(name: str):
    """('reduce', (T, VECW, LPR, VPL, RED, WM, PF)) or ('fixup', (T, RED)) for a demangled kernel name, else None."""
    m = _KERNEL.search(name)
    if not m:
        return None
    args = [re.sub(r"^\((?:unsigned )?\w+\)", "", a.strip()).replace("geot::", "") for a in m.group(2).split(",")]
    if args[0] not in DTYPES:
        return None
    nums = tuple(int(a.rstrip("uUlL")) for a in args[1:])
    kind = "reduce" if m.group(1) == "segment_reduce_kernel" else "fixup"
    if (kind, len(nums)) not in (("reduce", 6), ("fixup", 1)):
        return None
    return kind, (args[0],) + nums


def kernel_names(path: str):
    """Demangled names of every kernel in a CUDA binary (cuobjdump -res-usage, c++filt)."""
    out = subprocess.run([_tool("cuobjdump"), "-res-usage", path], capture_output=True, text=True, check=True).stdout
    mangled = re.findall(r"Function (\S+):", out)
    dem = subprocess.run([_tool("c++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                         check=True).stdout.splitlines()
    assert len(dem) == len(mangled)
    return dem


@functools.lru_cache(maxsize=None)
def inventory(path: str = None):
    """(reduce-kernel tuples, fixup-kernel tuples) compiled into the library (default: geot_b200.LIB_PATH)."""
    if path is None:
        import geot_b200
        path = geot_b200.LIB_PATH
    red, fix = set(), set()
    for n in kernel_names(path):
        k = parse_kernel(n)
        if k:
            (red if k[0] == "reduce" else fix).add(k[1])
    return frozenset(red), frozenset(fix)


# ---- dispatch, restated -------------------------------------------------------------------------------------------
def _pow2ceil(x: int) -> int:
    p = 1
    while p < x:
        p <<= 1
    return p


def choose_config(W: int, F: int, dt: str, vector_ok: bool):
    """(VECW, LPR, VPL, column tiles) -- the row-shape part of choose_config (abi.cu:37-56)."""
    full = 16 // esize(dt)
    vecw = full if (vector_ok and F % full == 0) else 1
    nvec = -(-W // vecw)
    if nvec <= 32:
        lpr, vpl = _pow2ceil(nvec), 1
    else:
        lpr, vpl = 32, (2 if (nvec <= 64 or vecw == 8) else 4)
    return vecw, lpr, vpl, -(-nvec // (lpr * vpl))


def _sub_batch(lpr: int, vpl: int, lean: bool) -> int:
    """ShapeOf<..>::U of a ring instantiation (segment_reduce.cuh:196-200, GEOT_RING_U = 0)."""
    if lean:
        u0 = 1 if vpl >= 4 else (2 if vpl == 2 else (4 if lpr >= 16 else (2 if lpr >= 8 else 1)))
    else:
        u0 = 2 if vpl >= 4 else 4
    return min(lpr, u0)


def _lean_depth(want: int, sb: int) -> int:
    """inst.cu:49-53."""
    d = want if want < sb else sb - 1
    while d > 0 and sb % (d + 1) != 0:
        d -= 1
    return d


def dispatch(case) -> tuple:
    """The instantiation launch_wm (inst.cu:55-107) picks for a case; ``max_blocks >= 1`` is taken as true (a kernel
    for which it is false is never launched, and the GPU coverage test would report it)."""
    dt, red = case.target[0], case.target[4]
    vecw, lpr, vpl, _ = choose_config(case.W, case.F, dt, not case.misaligned)
    # abi.cu:566; max / min / prod are built for the generic weight mode only (inst.cu:110-117)
    wm = 2 if red != 0 else (0 if case.weight == "none" else (1 if case.H == 1 else 2))
    pf, acc32 = case.ring, dt != "double"
    if red == 0 and vecw * esize(dt) == 16 and lpr >= 8:
        if pf & LEAN:
            sb = lpr // _sub_batch(lpr, vpl, True)
            if wm != 2 and acc32 and case.chunk % lpr == 0:
                da, db = _lean_depth(3, sb), _lean_depth(7, sb)
                ext = case.mode in ("planless", "accumulate", "edge_perm", "mean_rowptr", "mean_accumulate")
                d = db if (pf & DEPTH) > da and db != da else da
                return (dt, vecw, lpr, vpl, red, wm, LEAN | (EXT if ext else 0) | d)
            if wm == 2 and acc32 and case.chunk % lpr == 0 and case.H <= HEAD_MAX and case.mode != "edge_perm":
                ext = case.mode in ("planless", "accumulate", "mean_rowptr", "mean_accumulate")
                return (dt, vecw, lpr, vpl, red, wm, LEAN | HEADW | (EXT if ext else 0) | _lean_depth(3, sb))
            pf = 3 if vpl == 1 else 2
        pfmax = lpr // _sub_batch(lpr, vpl, False)
        if pf in (2, 3):
            return (dt, vecw, lpr, vpl, red, wm, min(pf, pfmax))
    return (dt, vecw, lpr, vpl, red, wm, 0)


# ---- cases --------------------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class Case:
    target: tuple       # (T, VECW, LPR, VPL, RED, WM, PF)
    reduce: str         # sum / mean / max / min / prod
    H: int
    F: int
    weight: str         # none / edge ([E]) / eh ([E, H]) / he ([H, E])
    gather: bool        # src_index given (else src row = edge id)
    misaligned: bool    # src starts one element past a 16-byte boundary
    ring: int           # GEOT_B200_RING
    chunk: int          # GEOT_B200_CHUNK
    mode: str           # plan / planless / accumulate / edge_perm / mean_rowptr / mean_accumulate
    seed: int

    @property
    def W(self):
        return self.H * self.F

    @property
    def dtype(self):
        return DTYPES[self.target[0]]

    @property
    def id(self):
        return "%s-%s-%s-W%d-H%d-%s" % (tuple_id(self.target), self.reduce, self.mode, self.W, self.H, self.weight)


def _widths(t, H: int, misaligned: bool, fmax: int = 1200):
    """(F, column tiles) with choose_config(H*F, F) == the target's (VECW, LPR, VPL)."""
    dt, vecw, lpr, vpl = t[:4]
    for F in range(1, fmax // H + 2):
        c = choose_config(H * F, F, dt, not misaligned)
        if c[:3] == (vecw, lpr, vpl):
            yield F, c[3]


def _pick_width(t, H, misaligned, k):
    """A row width for the target shape: more than one column tile where the shape has them (every third such case
    wider than 1024 elements: the fixup's float4 loop then runs more than once), else full or half-idle lanes."""
    c = list(_widths(t, H, misaligned))
    if not c:
        return None
    multi = [x for x in c if x[1] > 1]
    if multi:
        wide = [x for x in multi if H * x[0] > 1024 and H * x[0] < 1100]
        pool = wide if (k % 3 == 0 and wide) else [x for x in multi if x[1] == 2]
        return pool[(k // 3) % len(pool)][0]
    return (c[-1] if k % 2 == 0 else c[0])[0]


def _heads(t, k):
    """Candidate head counts for a target with weight mode 2 on the sum kernels."""
    dt, pf = t[0], t[6]
    full = 16 // esize(dt)
    if pf & HEADW:
        hs = [full, 2, 4, 8, 3, 5] if k % 2 == 0 else [2, 8, full, 3, 4]
        return [h for h in hs if 2 <= h <= HEAD_MAX]
    return [2, 4, 8, 3, 6, 16] if k % 2 == 0 else [8, 2, 5, 4, 16]


def cases_for(t):
    """Calls that reach instantiation ``t``: one per reduce op it serves (sum and mean for RED 0).  [] for an
    instantiation in UNREACHABLE."""
    if t in UNREACHABLE:
        return []
    dt, vecw, lpr, vpl, red, wm, pf = t
    full = 16 // esize(dt)
    k0 = zlib.crc32(repr(t).encode())
    chunk = 2 * lpr                      # a tile is 512 edges; a chunk holds two lane batches
    out = []
    for variant, reduce in enumerate(["sum", "mean"] if red == 0 else [RED_NAMES[red]]):
        k = k0 + 7 * variant
        ring = 0 if pf == 0 else (pf if pf in (1, 2, 3) else LEAN | (pf & DEPTH))
        misaligned = vecw == 1 and k % 3 == 0
        # weight layout and heads
        if red == 0:
            weight = {0: "none", 1: "edge"}.get(wm, "eh" if k % 2 == 0 else "he")
        else:
            weight = ["none", "edge", "eh", "he"][k % 4]
        head_opts = [1]
        if weight in ("eh", "he"):
            head_opts = _heads(t, k)
            if red == 0 and pf in (2, 3) and (pf == 3) == (vpl == 1) and k % 2 == 0:
                # the per-head lean ring's fallback (inst.cu:86): more heads than it serves, ring forced to lean
                head_opts, ring = [16, 12, 9], LEAN | 3
            elif red != 0:
                head_opts = head_opts + [1]
        H = F = None
        for h in head_opts:
            for mis in ([misaligned, not misaligned] if vecw == 1 else [False]):
                F = _pick_width(t, h, mis, k)
                if F is not None:
                    H, misaligned = h, mis
                    break
            if H is not None:
                break
        if H is None:
            raise LookupError("no row width reaches %s" % (t,))
        if H == 1 and weight in ("eh", "he"):
            weight = "edge"
        # options
        if pf & LEAN and not pf & EXT:
            modes = ["plan"]
        elif pf & EXT:
            modes = (["planless", "accumulate"] + (["edge_perm"] if wm == 1 else [])) if reduce == "sum" else \
                ["mean_rowptr", "mean_accumulate", "planless"]
        elif red == 0:
            modes = (["plan", "planless", "accumulate"] + (["edge_perm"] if wm == 1 else [])) if reduce == "sum" else \
                ["plan", "planless", "mean_rowptr", "mean_accumulate"]
        else:
            modes = ["plan", "planless"]
        mode = modes[(k // 5) % len(modes)]
        gather = True if (weight != "none" or reduce == "prod") else (k % 2 == 1)
        out.append(Case(t, reduce, H, F, weight, gather, misaligned, ring, chunk, mode, seed=k % 100003))
    return out


# ---- inputs -------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Graph:
    dst: torch.Tensor      # sorted dst_index [E]
    S: int                 # rows of the output (> dst[-1] + 1)
    rows: dict             # named rows: hub (> 32 tiles), medium (2-3 tiles), chunky (several chunks), last


def make_graph(lpr: int, chunk: int, g: torch.Generator) -> Graph:
    """Sorted dst index with empty runs at the start, in the middle and at the end, rows of degree 1-7, rows cut by
    chunk and tile boundaries, a hub cut by more than 32 tiles (the fixup's long-chain form) and a medium row cut by
    a few (its short-chain form); E leaves a ragged last chunk: one whole lane batch and a part of another."""
    tile = (K_THREADS // lpr) * chunk
    rnd = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    degs, rows = [0, 0, 0], {}

    def short(n, gap_every=0):
        for i in range(n):
            degs.append(rnd(1, 7))
            if gap_every and i % gap_every == gap_every - 1:
                degs.extend([0] * rnd(1, 3))

    short(40, gap_every=13)
    rows["medium"] = len(degs)
    degs.append(2 * tile + tile // 2 + 3)
    short(30, gap_every=11)
    rows["chunky"] = len(degs)
    degs.append(3 * chunk + 1)
    degs.append(chunk + chunk // 2 + 1)
    short(20)
    rows["hub"] = len(degs)
    degs.append(36 * tile + tile // 2 + 5)
    short(25, gap_every=9)
    rem = lpr + max(1, lpr // 2 - 1)         # edges in the last chunk: in (LPR, 2 LPR), not a multiple of LPR
    while sum(degs) % chunk != rem % chunk:
        need = (rem - sum(degs)) % chunk
        degs.append(min(need, rnd(1, 3)))
    rows["last"] = len(degs) - 1
    S = len(degs) + 4                         # and four empty rows at the end
    deg = torch.tensor(degs, dtype=torch.int64)
    dst = torch.repeat_interleave(torch.arange(len(degs)), deg)
    return Graph(dst, S, rows)


@dataclasses.dataclass
class Inputs:
    src: torch.Tensor            # [N, W]
    src_index: torch.Tensor      # [E] or None
    dst: torch.Tensor
    weight: torch.Tensor         # None / [E] / [E, H] / [H, E] (caller order)
    S: int
    rows: dict
    edge_perm: torch.Tensor = None    # int32 [E]: weight of edge e is weight[edge_perm[e]]
    mean_rowptr: torch.Tensor = None  # int64 [S+1]: the degrees mean divides by
    prior: torch.Tensor = None        # [S, W]: dst before an accumulating call


def _grid(shape, g, k, scale, dtype):
    """Integers in [-k, k] times 2^-scale."""
    return (torch.randint(-k, k + 1, shape, generator=g).double() * 2.0 ** -scale).to(dtype)


def make_inputs(case: Case) -> Inputs:
    g = torch.Generator().manual_seed(case.seed)
    lpr = case.target[2]
    gr = make_graph(lpr, case.chunk, g)
    dst, E, W, H, dt = gr.dst, gr.dst.numel(), case.W, case.H, case.dtype
    if case.reduce == "prod":
        # factors +-1, and +-2 / +-1/2 on at most two edges of a row (for src and weight each): |log2| of a row's
        # product stays <= 4, inside every dtype's range
        u = torch.rand(E, generator=g, dtype=torch.float64)
        order = torch.argsort(dst.double() + 0.5 * u)
        start = torch.zeros(gr.S + 1, dtype=torch.int64)
        start[1:] = torch.cumsum(torch.bincount(dst, minlength=gr.S), 0)
        rank = torch.empty(E, dtype=torch.int64)
        rank[order] = torch.arange(E) - start[dst[order]]
        nonunit = rank < 2

        def factors(shape):
            sign = torch.randint(0, 2, shape, generator=g).double() * 2 - 1
            mag = 2.0 ** torch.randint(-1, 2, shape, generator=g).double()
            nu = nonunit.view([E] + [1] * (len(shape) - 1)) if shape[0] == E else nonunit.view(1, E)
            return sign * torch.where(nu, mag, torch.ones_like(mag))
        per_edge = factors((E, W))
        src_index = torch.randperm(E, generator=g) if case.gather else None
        src = torch.empty(E, W, dtype=torch.float64)
        src[src_index if src_index is not None else torch.arange(E)] = per_edge
        src = src.to(dt)
        wshape = {"none": None, "edge": (E,), "eh": (E, H), "he": (H, E)}[case.weight]
        weight = factors(wshape).to(dt) if wshape else None
    else:
        N = 1500 if case.gather else E
        src_index = torch.randint(0, N, (E,), generator=g) if case.gather else None
        src = _grid((N, W), g, 16, 4, dt)
        wshape = {"none": None, "edge": (E,), "eh": (E, H), "he": (H, E)}[case.weight]
        weight = _grid(wshape, g, 8, 2, dt) if wshape else None
    inp = Inputs(src, src_index, dst, weight, gr.S, gr.rows)
    if case.mode == "edge_perm":
        inp.edge_perm = torch.randperm(E, generator=g).to(torch.int32)
    if case.mode in ("mean_rowptr", "mean_accumulate"):
        # degrees of a "complete" edge list that this call holds a part of: its own degree plus 0-3 more
        deg = torch.bincount(dst, minlength=gr.S) + torch.randint(0, 4, (gr.S,), generator=g)
        inp.mean_rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(deg, 0)])
    if case.mode in ("accumulate", "mean_accumulate"):
        inp.prior = _grid((gr.S, W), g, 16, 4, dt)
    return inp


# ---- exact reference ----------------------------------------------------------------------------------------------
def effective_weight(case: Case, inp: Inputs):
    """[E, H] fp64 weight of each edge in edge order (or None)."""
    if inp.weight is None:
        return None
    w = inp.weight.double()
    if case.weight == "edge":
        if inp.edge_perm is not None:
            w = w[inp.edge_perm.long()]
        return w.view(-1, 1)
    return w if case.weight == "eh" else w.t()


def contributions(case: Case, inp: Inputs) -> torch.Tensor:
    """p[e] = weight[e, h] * src[src_index[e]] (fp64, exact on the grid), [E, W]."""
    x = inp.src.double()
    x = x[inp.src_index] if inp.src_index is not None else x
    w = effective_weight(case, inp)
    if w is None:
        return x
    E = x.shape[0]
    return (x.view(E, case.H, case.F) * w.view(E, -1, 1)).reshape(E, case.W)


def _to_out(x64: torch.Tensor, dtype) -> torch.Tensor:
    """One rounding: fp64 -> dtype (via fp32 for 16-bit types, exact there by the precondition)."""
    if dtype == torch.float64:
        return x64.clone()
    return x64.float().to(dtype)


def reference(case: Case, inp: Inputs, p: torch.Tensor = None) -> torch.Tensor:
    """What the kernel must return, bit for bit: [S, W] in the case's dtype."""
    dt, S = case.dtype, inp.S
    p = contributions(case, inp) if p is None else p
    cnt = torch.bincount(inp.dst, minlength=S)
    has = (cnt > 0).view(S, 1)
    if case.reduce in ("max", "min", "prod"):
        name = {"max": "amax", "min": "amin", "prod": "prod"}[case.reduce]
        idx = inp.dst.view(-1, 1).expand_as(p)
        r = torch.zeros(S, case.W, dtype=torch.float64).scatter_reduce_(0, idx, p, name, include_self=False)
        return r.to(dt)
    finite = torch.where(torch.isfinite(p), p.abs(), torch.zeros_like(p))
    bound = torch.zeros(S, case.W, dtype=torch.float64).index_add_(0, inp.dst, finite)
    if inp.prior is not None:
        bound += inp.prior.double().abs()
    assert float(bound.max()) < EXACT_BOUND, "inputs off the exact grid: a row's sum |p| reaches 2^18"
    s = torch.zeros(S, case.W, dtype=torch.float64).index_add_(0, inp.dst, p)
    acc = torch.float64 if dt == torch.float64 else torch.float32
    v = s.to(acc)                                  # exact
    if case.reduce == "mean":
        n = cnt if inp.mean_rowptr is None else inp.mean_rowptr[1:] - inp.mean_rowptr[:-1]
        v = v / n.clamp_min(1).to(acc).view(S, 1)  # IEEE division in the accumulator type
    if inp.prior is not None:
        v = torch.where(has, inp.prior.to(acc) + v, inp.prior.to(acc))
    else:
        v = torch.where(has, v, torch.zeros_like(v))
    return v.to(dt)


# ---- running a case on the device ---------------------------------------------------------------------------------
@contextlib.contextmanager
def env(**kv):
    """Sets environment variables (read by the library on every call) for the duration of a block."""
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            os.environ[k] = str(v)
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def launched_kernels(fn):
    """Runs ``fn()`` under torch.profiler (CUDA activity) and returns (its result, the names of the kernels it ran)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, [e.name for e in prof.events()]


def run_case(case: Case, inp: Inputs, device="cuda"):
    """Calls geot_b200_segment_reduce(_ex) for the case; returns (dst on the CPU, names of the kernels launched)."""
    from geot_b200 import abi
    t = lambda x: None if x is None else x.to(device)
    N = inp.src.shape[0]
    if case.misaligned:
        buf = torch.zeros(N * case.W + 1, dtype=case.dtype, device=device)
        src = buf[1:].view(N, case.W)
        src.copy_(inp.src)
    else:
        src = t(inp.src)
    dst = t(inp.dst)
    layout = {"none": abi.W_NONE, "edge": abi.W_EDGE, "eh": abi.W_EDGE_HEAD, "he": abi.W_HEAD_EDGE}[case.weight]
    if inp.prior is not None:
        out = t(inp.prior).clone()
    else:
        out = torch.full((inp.S, case.W), float("nan"), dtype=case.dtype, device=device)
    with env(GEOT_B200_RING=case.ring, GEOT_B200_CHUNK=case.chunk):
        plan = abi.DevicePlan(dst, inp.S) if case.mode != "planless" else None
        ws = abi.Workspace(dst.numel(), case.W, case.dtype, device)
        torch.cuda.synchronize()
        _, names = launched_kernels(lambda: abi.segment_reduce(
            src, t(inp.src_index), dst, t(inp.weight), case.reduce, S=inp.S, H=case.H, weight_layout=layout,
            plan=plan, out=out, workspace=ws, accumulate=case.mode in ("accumulate", "mean_accumulate"),
            edge_perm=t(inp.edge_perm), mean_rowptr=t(inp.mean_rowptr)))
    return out.cpu(), names


def row_class(inp: Inputs, r: int) -> str:
    for k, v in inp.rows.items():
        if v == r:
            return k
    cnt = int((inp.dst == r).sum())
    return "empty" if cnt == 0 else "degree %d" % cnt


def mismatch_report(got: torch.Tensor, exp: torch.Tensor, inp: Inputs) -> str:
    """'' when got equals exp (NaN where exp is NaN, equal values elsewhere), else which rows differ and how."""
    nan_ok = torch.equal(torch.isnan(got), torch.isnan(exp))
    g0 = torch.where(torch.isnan(got), torch.zeros_like(got), got)
    e0 = torch.where(torch.isnan(exp), torch.zeros_like(exp), exp)
    if nan_ok and torch.equal(g0, e0):
        return ""
    bad = (torch.isnan(got) != torch.isnan(exp)) | (g0 != e0)
    rows = torch.nonzero(bad.any(1)).flatten().tolist()
    parts = []
    for r in rows[:6]:
        c = torch.nonzero(bad[r]).flatten().tolist()
        parts.append("row %d (%s): %d cols, col %d got %r want %r" % (
            r, row_class(inp, r), len(c), c[0], float(got[r, c[0]]), float(exp[r, c[0]])))
    return "%d of %d rows differ; %s" % (len(rows), got.shape[0], "; ".join(parts))
