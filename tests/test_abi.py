"""The C-ABI library loads without a GPU, exports every symbol the two headers
declare, and refuses to compute without a device (no CPU fallback)."""
import ctypes
import os
import re

import pytest

import gaast_b200 as g
from gaast_b200 import _lib as L
from gaast_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set(re.findall(r"\b(gaast_[a-z0-9_]+)\s*\(", text))
    # function-pointer typedefs are not exports
    names -= set(re.findall(r"\(\*\s*(gaast_[a-z0-9_]+)\s*\)", text))
    return names


def test_every_declared_symbol_is_exported_and_bound():
    declared = _declared("gaast_b200.h") | _declared("gaast_b200_host.h")
    assert len(declared) > 60
    lib = ctypes.CDLL(L.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in include/ but not exported"
        assert name in L.PROTOTYPES, f"{name} has no ctypes prototype in gaast_b200/_lib.py"
    for name in L.PROTOTYPES:
        assert name in declared, f"{name} is bound but not declared in include/"


def test_struct_layouts_match_header():
    assert ctypes.sizeof(L.Term) == 16 and ctypes.sizeof(L.Op) == 32 and ctypes.sizeof(L.InputDesc) == 16
    assert L.lib.gaast_version().startswith(b"gaast_b200")


def test_offline_plan_and_kernel_source():
    """A plan can be created, costed and turned into CUDA source with no device."""
    w = W.WORKLOADS["cfg1"]
    plan = g.Plan(None, W.specialize(w))
    assert plan.cost() == (176, 48)  # SURVEY.md 8d: 176 B and 24 terms per element
    src = plan.kernel_source()
    assert "gaast_eval" in src and "d_fma" in src
    assert plan.root_grades() == [2]
    with pytest.raises(g.GaastError) as ei:
        plan.eval([])
    assert ei.value.status in (L.ERR_NO_DEVICE, L.ERR_SHAPE)


@pytest.mark.parametrize("name,cost", [("cfg2", (80, 320)), ("cfg2_full", (168, 672)), ("cfg3", (1536, 8192)),
                                       ("cfg4", (2200, 3210)), ("cfg5", (1152, 3216))])
def test_algorithmic_cost_of_the_workloads(name, cost):
    w = W.WORKLOADS[name]
    assert g.Plan(None, W.specialize(w)).cost(w.broadcast_mask()) == cost


@pytest.fixture
def scratch_cache(tmp_path, monkeypatch):
    """A private kernel-cache directory: GAAST_KERNEL_CACHE is honoured only together with
    GAAST_TEST_HOOKS=1, and the library reads its environment once -- gaast_reload_env() re-reads it."""
    monkeypatch.setenv("GAAST_TEST_HOOKS", "1")
    monkeypatch.setenv("GAAST_KERNEL_CACHE", str(tmp_path))
    L.lib.gaast_reload_env()
    yield tmp_path
    monkeypatch.delenv("GAAST_TEST_HOOKS")
    monkeypatch.delenv("GAAST_KERNEL_CACHE")
    L.lib.gaast_reload_env()


def test_generated_kernels_compile_for_sm100a(scratch_cache):
    """NVRTC cross-compiles the specialised kernel without a GPU (fresh cache dir); the second
    request is served from the cache after its manifest has been verified."""
    w = W.WORKLOADS["cfg2"]
    plan = g.Plan(None, W.specialize(w))
    info = plan.precompile(w.broadcast_mask())
    assert "origin=nvrtc" in info
    assert any(f.endswith(".cubin") for f in os.listdir(scratch_cache))
    assert any(f.endswith(".manifest") for f in os.listdir(scratch_cache))
    info2 = plan.precompile(w.broadcast_mask())
    assert "origin=override" in info2 and "unverified" not in info2  # a redirected cache says so in the origin


def test_kernel_source_is_the_precompiled_kernel(scratch_cache):
    """gaast_plan_kernel_source returns the text of the kernel gaast_plan_precompile compiles (the one gaast_eval
    launches for an aligned batch), for every call of every workload whose kernel the build precompiles.  It runs in a
    fresh process, as the build does: once torch is imported, NVRTC is torch's, whose ptxas may report spills, and a
    kernel that spills is rebuilt with more rows parked in shared memory."""
    import subprocess
    import sys
    check = """if True:
        import os
        import gaast_b200 as g
        from gaast_b200 import workloads as W
        for w in W.WORKLOADS.values():
            plan = g.Plan(None, W.specialize(w))
            for arith, with_sum, store_out, dtype in W.precompile_variants(w):
                kw = dict(broadcast_slots=w.broadcast_mask(), arith=arith, with_sum=with_sum, store_out=store_out, dtype=dtype)
                key = [t for t in plan.precompile(**kw).split() if t.startswith("key=")][0][4:]
                src = open(os.path.join(os.environ["GAAST_KERNEL_CACHE"], key + ".cu")).read()
                assert src == plan.kernel_source(**kw), (w.name, kw)
            plan.free()
    """
    r = subprocess.run([sys.executable, "-c", check], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def test_kernel_cache_override_needs_the_test_hook(tmp_path, monkeypatch):
    """GAAST_KERNEL_CACHE alone does not redirect the cache: the in-tree one keeps serving."""
    monkeypatch.setenv("GAAST_KERNEL_CACHE", str(tmp_path))
    L.lib.gaast_reload_env()
    try:
        w = W.WORKLOADS["cfg1"]
        info = g.Plan(None, W.specialize(w)).precompile(w.broadcast_mask())
        assert os.listdir(tmp_path) == []
        assert "origin=cache" in info or "origin=nvrtc" in info
    finally:
        monkeypatch.delenv("GAAST_KERNEL_CACHE")
        L.lib.gaast_reload_env()


def test_cached_cubins_are_verified_against_their_manifest(tmp_path):
    """A cached cubin is loaded only when the manifest next to it names the source just generated and the
    bytes on disk (sha256 of both, architecture, compile options).  One flipped byte, or a missing manifest,
    makes the entry a cache miss: it is recompiled and rewritten, never loaded."""
    import hashlib
    import shutil
    cache = os.path.join(os.path.dirname(os.path.abspath(g.__file__)), "kernel_cache")
    w = W.WORKLOADS["cfg1"]
    plan = g.Plan(None, W.specialize(w))
    info = plan.precompile(w.broadcast_mask())
    key = [t for t in info.split() if t.startswith("key=")][0][4:]
    cubin, manifest = os.path.join(cache, key + ".cubin"), os.path.join(cache, key + ".manifest")
    text = open(manifest).read()
    fields = dict(l.split(" ", 1) for l in text.strip().split("\n")[1:])
    assert fields["cubin_sha256"] == hashlib.sha256(open(cubin, "rb").read()).hexdigest()
    assert fields["source_sha256"] == hashlib.sha256(open(os.path.join(cache, key + ".cu"), "rb").read()).hexdigest()
    assert fields["arch"] == "sm_100a"
    assert "origin=cache" in plan.precompile(w.broadcast_mask())
    keep = tmp_path / "cubin.bak"
    shutil.copy(cubin, keep)
    try:
        with open(cubin, "r+b") as f:  # flip one byte of the cached cubin
            f.seek(100)
            b = f.read(1)
            f.seek(100)
            f.write(bytes([b[0] ^ 0xFF]))
        assert "origin=nvrtc" in plan.precompile(w.broadcast_mask())  # rejected, recompiled, rewritten
        again = dict(l.split(" ", 1) for l in open(manifest).read().strip().split("\n")[1:])
        assert again["cubin_sha256"] == hashlib.sha256(open(cubin, "rb").read()).hexdigest()
        assert again["source_sha256"] == fields["source_sha256"]
        assert "origin=cache" in plan.precompile(w.broadcast_mask())
        os.remove(manifest)  # a cubin without a manifest is not trusted either
        assert "origin=nvrtc" in plan.precompile(w.broadcast_mask())
        assert os.path.exists(manifest)
    finally:
        if not os.path.exists(manifest):  # leave a loadable entry behind whatever happened
            shutil.copy(keep, cubin)
            open(manifest, "w").write(text)


def test_no_device_means_no_compute():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(g.GaastError) as ei:
        g.Ctx(0)
    assert ei.value.status == L.ERR_NO_DEVICE


def test_host_memory_entries_validate_their_arguments():
    """gaast_host_alloc / _register check their arguments before any CUDA call: status codes without a device."""
    import ctypes as C
    out = L.vp()
    assert L.lib.gaast_host_alloc(64, 7, C.byref(out)) == L.ERR_INVALID and not out.value
    assert L.lib.gaast_host_alloc(0, L.HOST_DEFAULT, C.byref(out)) == L.ERR_INVALID
    assert L.lib.gaast_host_alloc(64, L.HOST_DEFAULT, None) == L.ERR_INVALID
    assert L.lib.gaast_host_register(None, 64) == L.ERR_INVALID
    assert L.lib.gaast_host_unregister(None) == L.ERR_INVALID
    assert L.lib.gaast_host_free(None) == L.OK
    import torch
    if not torch.cuda.is_available():
        # without a device the allocation itself is an error, never a crash
        assert L.lib.gaast_host_alloc(64, L.HOST_DEFAULT, C.byref(out)) != L.OK and not out.value


def test_huge_plans_are_left_to_the_table_engine():
    """G(8,0) A*B has 65 536 terms: the code generator refuses, AUTO falls back to the table engine."""
    from gaast_b200.expr import Input, mv
    full = tuple(range(9))
    ast = (mv(Input(0, full)) * mv(Input(1, full))).specialize([1.0] * 8)
    plan = g.Plan(None, ast)
    assert plan.cost() == (8 * 3 * 256, 2 * 65536)
    with pytest.raises(g.GaastError) as ei:
        plan.kernel_source()
    assert ei.value.status == L.ERR_JIT and "table engine" in str(ei.value)


def test_offline_precompile_of_a_dense_warp_plan():
    """A full product in G(7): too wide for the specialised engine, so the build-time precompile step
    analyses it for the dense-warp engine (term table complete, +-1, factorisation verified) and compiles
    that kernel with NVRTC -- all without a device.  A degenerate metric does not qualify."""
    from gaast_b200.device import Plan
    from gaast_b200.expr import Input, mv as pmv
    full = tuple(range(8))
    a, b = pmv(Input(0, full)), pmv(Input(1, full))
    plan = Plan(None, (a * b).specialize([1.0, 1.0, 1.0, 1.0, -1.0, -1.0, 1.0]))
    info = plan.precompile(0, L.ARITH_FMA, False, True)
    # a geometric product under a +-1 metric: the matrix-representation kernel of that engine (G(5,2) = M8(C))
    assert "gaast_dense_matrix" in info and "dense-matrix(n=7 M16 x1 cols=8)" in info and "fma/elem=2048" in info
    plan.set_tuning(0, 1048576)  # ... and the term-by-term kernel on request
    info = plan.precompile(0, L.ARITH_FMA, False, True)
    assert "gaast_dense_warp" in info and "dense-warp(n=7)" in info
    bad = Plan(None, (a * b).specialize([1.0] * 6 + [0.0]))
    with pytest.raises(L.GaastError) as ei:
        bad.precompile(0, L.ARITH_FMA, False, True)
    assert ei.value.status == L.ERR_JIT


def test_offline_analysis_of_dense_warp_chains_and_grade_restricted_plans():
    """The dense-warp analysis without a device: product chains, grade-restricted buffers (sigma / lambda
    recovered by GF(2) propagation), outer products; and plans it must leave alone."""
    from gaast_b200.device import Plan
    from gaast_b200.expr import Input, mv as pmv
    n = 8
    metric = [1.0] * 6 + [-1.0] * 2
    full, even = tuple(range(n + 1)), tuple(range(0, n + 1, 2))
    a, b, r = pmv(Input(0, full)), pmv(Input(1, full)), pmv(Input(2, even))
    # chains of geometric products get the matrix-representation kernel (G(6,2) = M8(H): 2^(8+5) multiplications), a
    # chain with an outer product keeps the term-by-term kernel
    for expr, products, kernel in ((a * b, 1, "gaast_dense_matrix"), (r * a * r.rev(), 2, "gaast_dense_matrix"),
                                   ((a ^ b) * r, 2, "gaast_dense_warp"), (-(a * b), 1, "gaast_dense_matrix")):
        info = Plan(None, expr.specialize(metric)).precompile(0, L.ARITH_FMA, False, True)
        assert kernel in info and f"x{products} product(s)" in info, info
        assert ("fma/elem=8192" in info) == (kernel == "gaast_dense_matrix"), info
    info = Plan(None, (a * b + a).specialize(metric)).precompile(0, L.ARITH_FMA, False, True)
    assert "gaast_dense_matrix" in info  # an input added into the product's buffer joins the product's store
    for expr in ((a * b).norm_sq().sqrt() * a, (a * b) * 2.5):  # a scalar op; a literal operand
        with pytest.raises(L.GaastError):
            Plan(None, expr.specialize(metric)).precompile(0, L.ARITH_FMA, False, True)
