"""Host-side checks of the drop-in boundary -- no GPU needed, no compute calls.

The C-ABI library must load, export every symbol include/geot_b200.h declares, answer its host-only
queries, reject bad arguments before touching the device, and the torch bindings must register the
reference's operator schemas with no CPU implementation behind them (no fallback).
"""
import ctypes
import os
import re

import pytest
import torch

import geot_b200
from geot_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "geot_b200.h")).read()
    return sorted(set(re.findall(r"GEOT_API[^;]*?\b(geot_b200_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    declared = _declared_symbols()
    assert len(declared) >= 15
    assert sorted(abi.SYMBOLS) == declared
    L = ctypes.CDLL(geot_b200.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name


def test_version_arch_status_strings():
    L = abi.lib()
    assert L.geot_b200_version() == 200
    assert L.geot_b200_arch() == 100
    assert L.geot_b200_status_string(0) == b"ok"
    assert b"invalid" in L.geot_b200_status_string(1)
    assert torch.ops.geot.abi_version() == 200


def test_library_is_sm100a_only():
    """The shipped SASS is sm_100a and nothing else (no multi-arch fat binary, no PTX-JIT fallback)."""
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", geot_b200.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_host_queries():
    L = abi.lib()
    assert L.geot_b200_plan_bytes(1000, 10) >= 11 * 8
    assert L.geot_b200_plan_bytes(1000, 10) % 256 == 0
    small = L.geot_b200_workspace_bytes(1000, 32, abi.F32, 1)
    big = L.geot_b200_workspace_bytes(10_000_000, 128, abi.F32, 1)
    assert 0 < small < big
    assert small % 256 == 0
    # the unsorted path needs the sort buffers on top
    assert L.geot_b200_workspace_bytes(1_000_000, 32, abi.F32, 0) > L.geot_b200_workspace_bytes(1_000_000, 32, abi.F32, 1) + 4 * 8 * 1_000_000 - 4096


def test_argument_validation_happens_before_any_device_work():
    L = abi.lib()
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)  # never dereferenced: the calls must fail on validation
    f = L.geot_b200_segment_reduce
    assert f(null, null, one, null, one, 10, 4, 1, 8, abi.F32, abi.SUM, abi.W_NONE, 1, None, one, 1 << 20, null) == 1
    assert f(one, null, one, null, one, 0, 4, 1, 8, abi.F32, abi.SUM, abi.W_NONE, 1, None, one, 1 << 20, null) == 5   # empty
    assert f(one, null, one, null, one, 10, 4, 1, 8, 9, abi.SUM, abi.W_NONE, 1, None, one, 1 << 20, null) == 1        # dtype
    assert f(one, null, one, null, one, 10, 4, 1, 8, abi.F32, 7, abi.W_NONE, 1, None, one, 1 << 20, null) == 1        # reduce
    assert f(one, null, one, null, one, 10, 4, 1, 8, abi.F32, abi.SUM, abi.W_EDGE, 1, None, one, 1 << 20, null) == 1  # weight missing
    assert f(one, null, one, null, one, 10, 4, 1, 8, abi.F32, abi.SUM, abi.W_NONE, 1, None, ctypes.c_void_p(264), 1 << 20, null) == 3  # misaligned ws
    assert L.geot_b200_gather_scatter(one, null, one, one, 10, 4, 8, abi.F32, abi.SUM, None, one, 1 << 20, null) == 1  # src_index missing
    assert L.geot_b200_mh_spmm(one, one, one, one, one, 10, 4, 2, 8, abi.F32, abi.SUM, abi.W_EDGE, None, one, 1 << 20, null) == 1
    # host-buffer entries: the row ranges of the slices come from dst_index read at 0, at every cut and at E-1, so an
    # index that leaves [0, S) or decreases there is refused before any CUDA call
    E = 8192
    di = torch.arange(E) // 4
    S = int(di[-1]) + 1
    neg = di.clone()
    neg[0] = -1
    rotated = di.roll(E // 2)
    host = L.geot_b200_segment_reduce_host
    for idx, rows in ((di, S - 1), (neg, S), (rotated, S)):
        assert host(one, S, one, idx.data_ptr(), null, one, E, rows, 1, 8, abi.F32, abi.SUM, abi.W_NONE) == 1
    big = (torch.arange(200_000) // 4).roll(100_000)
    h = ctypes.c_void_p(0)
    assert L.geot_b200_host_graph_create(one, big.data_ptr(), big.numel(), 50_000, 50_000, ctypes.byref(h)) == 1
    assert not h.value
    with pytest.raises(abi.AbiError, match="invalid argument"):
        abi.check(1, "x")


def test_operator_schemas_match_the_reference():
    """csrc/index_scatter.cpp:43-47, gather_scatter.cpp:16-17, gather_weight_scatter.cpp:12-14, mh_spmm.cpp:23."""
    s = lambda op: str(op.default._schema)
    assert s(torch.ops.geot.index_scatter) == "geot::index_scatter(int dim, Tensor index, Tensor src, str reduce, bool sorted) -> Tensor"
    assert s(torch.ops.geot.gather_scatter_impl) == "geot::gather_scatter_impl(Tensor src_index, Tensor dst_index, Tensor src) -> Tensor"
    assert s(torch.ops.geot.gather_weight_scatter_impl) == "geot::gather_weight_scatter_impl(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src) -> Tensor"
    assert s(torch.ops.geot.mh_spmm) == "geot::mh_spmm(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src, str reduce) -> Tensor"
    assert s(torch.ops.geot.gather_scatter) == "geot::gather_scatter(Tensor src_index, Tensor dst_index, Tensor src) -> Tensor"
    assert s(torch.ops.geot.gather_weight_scatter) == "geot::gather_weight_scatter(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src) -> Tensor"


def test_python_surface_matches_the_reference_package():
    for name in ["index_scatter", "gather_scatter", "gather_weight_scatter", "mh_spmm", "mh_spmm_transposed"]:
        assert callable(getattr(geot_b200, name))
    import inspect
    assert list(inspect.signature(geot_b200.index_scatter).parameters) == ["dim", "src", "index", "reduce", "sorted"]
    assert list(inspect.signature(geot_b200.mh_spmm).parameters) == ["src_index", "dst_index", "weight", "src", "reduce"]


def test_no_cpu_fallback():
    idx = torch.tensor([0, 0, 1, 2])
    x = torch.rand(4, 4)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.index_scatter(0, x, idx)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.gather_scatter(idx, idx, x)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.gather_weight_scatter(idx, idx, torch.rand(4), x)
    with pytest.raises((NotImplementedError, RuntimeError)):
        geot_b200.mh_spmm(idx, idx, torch.rand(4, 2), torch.rand(4, 2, 4))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "geot_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "geot_oracle" not in text, f


@pytest.mark.parametrize("threads", [1, 3, 16])
def test_host_row_pointers_match_the_oracle(threads):
    """The host-side segment-pointer pass of the compact transport (pure CPU code of the library): bit-exact against
    the oracle's rowptr (= coo_to_csr) on whole indices and on slices, with gaps, hubs and single-edge rows."""
    import oracle
    from geot_b200 import abi
    g = torch.Generator().manual_seed(threads)
    for (E, N, skew) in [(1, 1, 1), (50, 400, 1), (20000, 300, 3), (200000, 50000, 2), (300000, 7, 1)]:
        w = torch.rand(N, generator=g) ** skew
        di = torch.multinomial(w / w.sum(), E, replacement=True, generator=g).sort().values.contiguous()
        S = int(di[-1]) + 1
        exp = oracle.rowptr(di, S)
        assert torch.equal(abi.host_row_pointers(di, 0, S, threads), exp)
        assert torch.equal(abi.host_row_pointers(di, 0, S + 9, threads)[S:], torch.full((10,), E))     # trailing empty rows
        # a slice cut at a segment boundary, rows relative to its first row (what the host entry sends per slice)
        e0 = int(exp[S // 2])
        r0 = S // 2
        sl = di[e0:].contiguous()
        got = abi.host_row_pointers(sl, r0, S - r0, threads)
        assert torch.equal(got, exp[r0:] - e0)


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """include/geot_b200.h compiles as C99 (no C++, no torch types) and a C host links against the library: the
    example a cgo / JNI maintainer would start from (examples/abi_host_example.c).  The pure-host helper runs here;
    the device call reports the missing GPU through the status code instead of crashing (no CPU path)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "abi_host_example")
    libdir = os.path.join(root, "geot_b200", "lib")
    cmd = ["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I" + os.path.join(root, "include"),
           os.path.join(root, "examples", "abi_host_example.c"), "-L" + libdir, "-lgeot_b200", "-Wl,-rpath," + libdir, "-o", exe]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert "rowptr: 0 2 3 3 6" in run.stdout, run.stdout + run.stderr
    if torch.cuda.is_available():
        assert "dst[3] = 20 200" in run.stdout and "dst[2] = 0 0" in run.stdout and run.returncode == 0
    else:
        assert run.returncode == 0 and "CUDA error" in run.stdout, run.stdout + run.stderr


def test_library_has_no_torch_dependency_and_exports_only_the_abi():
    """The boundary is a plain C-ABI library: it links the CUDA runtime and the C/C++ runtimes, nothing of torch / ATen /
    Python, and its dynamic symbol table defines only geot_b200_* functions (everything else is hidden)."""
    import subprocess
    lib = geot_b200.LIB_PATH
    needed = subprocess.run(["readelf", "-d", lib], capture_output=True, text=True).stdout
    libs = re.findall(r"Shared library: \[([^\]]+)\]", needed)
    assert libs, needed
    assert not [l for l in libs if re.search(r"torch|c10|python|aten|nccl", l, re.I)], libs
    assert any(l.startswith("libcudart") for l in libs), libs
    syms = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True).stdout
    defined = [ln.split()[-1] for ln in syms.splitlines() if len(ln.split()) >= 3 and ln.split()[-2] in ("T", "t")]
    foreign = [s for s in defined if not s.startswith("geot_b200_") and s not in ("_init", "_fini")]
    assert foreign == [], foreign[:10]
    assert sorted(set(defined) - {"_init", "_fini"}) == sorted(abi.SYMBOLS)


def test_ctypes_binding_matches_the_header_arity_and_types():
    """geot_b200/abi.py declares argtypes by hand: every function's arity and the pointer / integer class of every
    argument must agree with include/geot_b200.h (a wrong argtypes entry corrupts arguments silently)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "geot_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    L = abi.lib()
    checked = 0
    for m in re.finditer(r"GEOT_API\s+([\w\s\*]+?)\s*\b(geot_b200_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        params = [] if args in ("", "void") else [a.strip() for a in args.split(",")]
        fn = getattr(L, name)
        if fn.argtypes is None:
            assert not params or name in ("geot_b200_profile_enable", "geot_b200_profile_read", "geot_b200_status_string"), name
            continue
        assert len(fn.argtypes) == len(params), (name, len(fn.argtypes), params)
        for at, p in zip(fn.argtypes, params):
            is_ptr = "*" in p or "cudaStream_t" in p
            if is_ptr:
                assert at is ctypes.c_void_p or hasattr(at, "contents") or issubclass(at, ctypes._Pointer), (name, p, at)
            elif "int64_t" in p:
                assert at is ctypes.c_int64, (name, p, at)
            elif "size_t" in p:
                assert at is ctypes.c_size_t, (name, p, at)
            else:
                assert at is ctypes.c_int, (name, p, at)
        checked += 1
    assert checked >= 18, checked


def test_reference_side_binding_compiles(tmp_path):
    """INTEGRATION.md section 2 as a real translation unit (examples/reference_binding_gws.cpp): the body GeoT's
    csrc/gather_weight_scatter.cpp gets after the swap compiles against the torch headers and include/geot_b200.h."""
    import subprocess
    from torch.utils.cpp_extension import include_paths
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = (["g++", "-std=c++17", "-O0", "-fPIC", "-c", os.path.join(root, "examples", "reference_binding_gws.cpp"),
            "-I" + os.path.join(root, "include"), "-I/usr/local/cuda/include", "-o", str(tmp_path / "binding.o")]
           + ["-I" + p for p in include_paths()])
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]


def test_reference_import_name_resolves():
    """`import geot` (the reference's package name, /root/reference/geot/__init__.py:4-9) is served by geot_b200."""
    import geot
    import geot_b200
    for name in ("index_scatter", "gather_scatter", "gather_weight_scatter", "mh_spmm", "mh_spmm_transposed", "csr_gws", "coo_to_csr"):
        assert getattr(geot, name) is getattr(geot_b200, name), name
    from geot.match_replace import pattern_transform
    assert pattern_transform is geot_b200.pattern_transform
    # the reference's other import paths (test/compile/*.py: `import geot.match_replace as replace`, `import geot.csr_gws`)
    import geot.match_replace as replace
    import geot.csr_gws            # noqa: F401  (a module in sys.modules; the attribute stays the operator, as in the reference)
    from geot.gather_weight_scatter import gather_weight_scatter
    assert replace.pattern_transform is geot_b200.pattern_transform and callable(geot.csr_gws)
    assert gather_weight_scatter is geot_b200.gather_weight_scatter


def test_mean_division_identity():
    """The kernels divide by the segment length with one multiply and two FMAs (segment_reduce.cuh div_by_count:
    q = v * RN(1/n); q' = fma(fma(-q, n, v), RN(1/n), q)) instead of a division per element.  Restated in numpy
    (fp32 FMA emulated through fp64: products of two fp32 values are exact there) it must equal IEEE fp32 division for
    integer n, including the n = 2^k - 1 significands where the plain reciprocal multiply is off by one ulp."""
    import numpy as np
    rng = np.random.default_rng(0)

    def fma32(a, b, c):
        return np.float32(np.float64(a) * np.float64(b) + np.float64(c))
    ns = np.concatenate([np.arange(1, 5000), 2 ** np.arange(1, 24) - 1, rng.integers(1, 300000, 20000)]).astype(np.float32)
    plain_bad = 0
    for trial in range(6):
        if trial == 0:
            a = ns.copy()                                        # mean of ones
        elif trial == 1:
            a = (ns * np.float32(3.0)).astype(np.float32)
        else:
            a = (rng.random(ns.size).astype(np.float32) * ns * np.float32(1.7)).astype(np.float32)
        inv = (np.float32(1.0) / ns).astype(np.float32)
        q = (a * inv).astype(np.float32)
        got = fma32(fma32(-q, ns, a), inv, q)
        assert np.array_equal(got, (a / ns).astype(np.float32)), trial
        plain_bad += int((q != (a / ns).astype(np.float32)).sum())
    assert plain_bad > 0          # (the correction step is needed: the plain product is not always the quotient)


def test_src_blocks_suggestion_rule():
    """geot_b200_src_blocks_suggest (pure host arithmetic): high-reuse graphs whose src matrix exceeds what the L2 keeps
    are blocked, resident or low-reuse ones are not (profiles/r02a_blocks.txt, r02a_l2probe.txt)."""
    from geot_b200 import abi
    assert abi.src_blocks_suggest(114_615_892, 232_965, 232_965, 512) == 2        # Reddit shape, F = 128 fp32: 119 MB
    assert abi.src_blocks_suggest(39_561_252, 132_534, 132_534, 1024) == 2        # proteins shape, F = 256: 136 MB
    assert abi.src_blocks_suggest(114_615_892, 232_965, 232_965, 256) == 1        # 60 MB: already resident
    assert abi.src_blocks_suggest(61_859_140, 2_449_029, 2_449_029, 256) == 1     # products: degree 25, no reuse to save
    assert abi.src_blocks_suggest(1_166_243, 169_343, 169_343, 512) == 1          # arxiv
    # dst-row shards keep the rule's verdict: a Reddit-shape shard of 8 still blocks, the hub shard of the products shape
    # (40 edges per row against a 627 MB matrix: 9 passes of 4.5 edges per row, measured 3.2x slower) does not
    assert abi.src_blocks_suggest(14_327_639, 28_837, 232_965, 512) == 2
    assert abi.src_blocks_suggest(8_203_841, 201_546, 2_449_029, 256) == 1
    assert abi.src_blocks_suggest(400_000_000, 232_965, 2_000_000, 512) == 1      # 15 blocks: outside the measured regime
    assert abi.src_blocks_suggest(0, 1, 1, 4) == 1
