"""f32 batches evaluated in binary64 (GAAST_ARITH_F64) on a machine without a GPU: the generated kernels and the table
engine run by the CPU stand-in of tests/kernel_emu (through tests/wide_emu.py), against the oracle evaluated on the widened inputs.

The bars (include/gaast_b200.h, DESIGN.md 3.4): STRICT | F64 is bit-identical to float32(the reference's operation
sequence in binary64 on the widened inputs); FMA | F64 is within 0.5 ulp(binary32) of the f64 oracle plus the f64 bar
(1e-12 of max(|ref|, sum |terms|)) -- one rounding per stored result; batch sums add the unrounded binary64 results and
are held to 1e-12 against the exact sum of the f64 oracle."""
import math
import os
import re

import numpy as np
import pytest

import gaast_b200 as g
from gaast_b200 import _lib as L
from gaast_b200 import workloads as W
from gaast_b200.expr import Input, mv as pmv
from tests.helpers import assert_bit_exact, oracle_abs_scale, oracle_eval, run_plan_numpy
from tests.wide_emu import prefetch_wide, run_wide_kernel, run_wide_table_engine

pytestmark = pytest.mark.timeout(900)

STRICT64 = L.ARITH_STRICT | L.ARITH_F64
FMA64 = L.ARITH_FMA | L.ARITH_F64
NAMES = ["cfg1", "cfg2", "cfg2_full", "cfg3", "cfg4", "cfg5"]
# the algebraic lowerings that must still fire when f32 batches are evaluated in binary64
LOWERING = {"cfg2": "linear-map", "cfg2_full": "linear-map", "cfg3": "dense-matrep", "cfg5": "reflection"}


def f32_inputs(w, batch):
    host = [{k: v.astype(np.float32) for k, v in d.items()} for d in W.host_inputs(w, batch)]
    return host, [{k: v.astype(np.float64) for k, v in d.items()} for d in host]


def strict_want(ast, host64, batch):
    """float32(the plan's operation sequence in binary64 on the widened inputs)."""
    with np.errstate(all="ignore"):
        want = run_plan_numpy(ast.plan_dict(), host64, batch, dtype=np.float64)
    return {k: v.astype(np.float32) for k, v in want.items()}


def assert_within_one_rounding(got, want, scale, what):
    """|dev - oracle64| <= 0.5 ulp32 + 1e-12 max(|oracle64|, sum |terms|), component by component."""
    assert sorted(got) == sorted(want), what
    for k in want:
        gv = np.asarray(got[k])
        assert gv.dtype == np.float32, f"{what}: grade {k} stored as {gv.dtype}"
        g64, w = gv.astype(np.float64), want[k]
        ulp = np.spacing(np.maximum(np.abs(w), np.abs(g64)).astype(np.float32)).astype(np.float64)
        tol = 0.5 * ulp + 1e-12 * np.maximum(np.abs(w), np.abs(scale[k])) + 1e-300
        err = np.abs(g64 - w)
        bad = err > tol
        assert not bad.any(), f"{what}: grade {k}: {int(bad.sum())} components off, worst {err.max():.3e} ({(err / tol).max():.2f} x bar)"


@pytest.fixture(scope="module")
def workload_kernels():
    cases = []
    for name in NAMES:
        w = W.WORKLOADS[name]
        for arith in (STRICT64, FMA64):
            cases.append((W.specialize(w), [bc for _, bc in w.inputs], arith, np.float32))
    prefetch_wide(cases)


@pytest.mark.parametrize("name", NAMES)
def test_wide_kernels(name, workload_kernels):
    w = W.WORKLOADS[name]
    batch = 262  # not a multiple of 4: the aligned kernel is launched over the padding (containment is checked)
    host, host64 = f32_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    ast = W.specialize(w)
    out, _, info = run_wide_kernel(ast, host, bcs, batch, arith=STRICT64, dtype=np.float32)
    assert "arith=f64" in info["source"].split("\n")[0]
    assert_bit_exact(out, strict_want(ast, host64, batch), f"{name} strict|f64 [{info['notes']}]")
    out, _, info = run_wide_kernel(ast, host, bcs, batch, arith=FMA64, dtype=np.float32)
    if name in LOWERING:
        assert LOWERING[name] in info["notes"], info["notes"]
    want = oracle_eval(w.build, w.metric, host64, bcs, batch)
    scale = oracle_abs_scale(w.build, w.metric, host64, bcs, batch)
    assert_within_one_rounding(out, want, scale, f"{name} fma|f64 [{info['notes']}]")


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("store_out", [True, False])
def test_wide_batch_sums(name, store_out):
    """The batch-sum adds the unrounded binary64 results: 1e-12 of the scale against the exact sum of the f64 oracle
    (the sum of the stored binary32 values would be ~1e-8 off)."""
    w = W.WORKLOADS[name]
    batch = 256
    host, host64 = f32_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    ast = W.specialize(w)
    out, sums, info = run_wide_kernel(ast, host, bcs, batch, arith=FMA64, with_sum=True, store_out=store_out,
                                           grid=2, dtype=np.float32)
    want = oracle_eval(w.build, w.metric, host64, bcs, batch)
    scale = oracle_abs_scale(w.build, w.metric, host64, bcs, batch)
    if store_out:
        assert_within_one_rounding(out, want, scale, f"{name} sum kernel's stores")
    for k in want:
        exact = np.array([math.fsum(row) for row in want[k]])
        tol = 1e-12 * np.maximum(np.abs(want[k]).sum(axis=1), scale[k].sum(axis=1)) + 1e-300
        err = np.abs(sums[k] - exact)
        assert (err <= tol).all(), f"{name} [{info['notes']}]: batch-sum of grade {k} off by {(err / tol).max():.1f} x the bar"


def test_wide_sparse_inputs_and_projection():
    """cfg5 with a sparse bivector input and a projected result, and the projected plan alone: strict bit-exact."""
    w = W.WORKLOADS["cfg5"]
    ast = W.specialize(w)
    batch = 262
    host, host64 = f32_inputs(w, batch)
    keep_in = list(range(0, 66, 3))
    for h in (host, host64):
        h[1][2][[i for i in range(66) if i not in keep_in]] = 0.0
    comps = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}
    want = strict_want(ast, host64, batch)
    sel = {2: want[2][comps[2]]}
    sparse_host = [host[0], {2: host[1][2][keep_in]}]
    out, _, info = run_wide_kernel(ast, sparse_host, [False, False], batch, arith=STRICT64, dtype=np.float32,
                                        present={(1, 2): keep_in}, components=comps)
    assert_bit_exact(out, sel, f"sparse inputs + projection [{info['notes']}]")
    out, _, info = run_wide_kernel(ast, sparse_host, [False, False], batch, arith=STRICT64, dtype=np.float32,
                                        present={(1, 2): keep_in})
    assert_bit_exact(out, want, f"sparse inputs [{info['notes']}]")
    out, _, info = run_wide_kernel(ast, host, [False, False], batch, arith=STRICT64, dtype=np.float32, components=comps)
    assert "projection(" in info["notes"]
    assert_bit_exact(out, sel, f"projected [{info['notes']}]")


def _literal_case():
    """Coefficients that binary32 cannot hold: a non-unit metric and a literal factor.  The f32 variant rounds them; the
    binary64 arithmetic must not."""
    metric = [1.0, 0.7, -1.3]
    a, b = pmv(Input(0, (1,))), pmv(Input(1, (1,)))
    return ((a * b) * 0.1).specialize(metric), 2


def test_wide_coefficients_stay_binary64():
    ast, slots = _literal_case()
    batch = 262
    rng = np.random.default_rng(5)
    host = [{1: rng.uniform(-1, 1, (3, batch)).astype(np.float32)} for _ in range(slots)]
    host64 = [{k: v.astype(np.float64) for k, v in d.items()} for d in host]
    want = strict_want(ast, host64, batch)
    out, _, info = run_wide_kernel(ast, host, [False] * slots, batch, arith=STRICT64, dtype=np.float32)
    assert_bit_exact(out, want, f"literals strict|f64 [{info['notes']}]")
    out, _ = run_wide_table_engine(ast, host, [False] * slots, batch, strict=True)
    assert_bit_exact(out, want, "literals on the table engine")


def _random_seeds():
    from tests.test_random_exprs import GPU_SEEDS
    return GPU_SEEDS[:6]


@pytest.mark.parametrize("seed", _random_seeds())
def test_wide_random_expressions(seed):
    from tests.test_random_exprs import BATCH, evaluate_case
    n, metric, slots, inputs, _, ast, _, _ = evaluate_case(seed)
    in32 = [{k: v.astype(np.float32) for k, v in d.items()} for d in inputs]
    in64 = [{k: v.astype(np.float64) for k, v in d.items()} for d in in32]
    with np.errstate(all="ignore"):
        want = strict_want(ast, in64, BATCH)
        out, _, info = run_wide_kernel(ast, in32, [bc for _, bc in slots], BATCH, arith=STRICT64, dtype=np.float32)
    assert_bit_exact(out, want, f"seed {seed} strict|f64 [{info['notes']}]")


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg4", "cfg5"])
def test_wide_table_engine(name):
    """The table engine with binary32 batches and a binary64 workspace: strict bit-exact, including its batch-sum."""
    w = W.WORKLOADS[name]
    batch = 70
    host, host64 = f32_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    ast = W.specialize(w)
    want = strict_want(ast, host64, batch)
    out, sums = run_wide_table_engine(ast, host, bcs, batch, strict=True, with_sum=True)
    assert_bit_exact(out, want, f"{name} table strict|f64")
    want64 = oracle_eval(w.build, w.metric, host64, bcs, batch)
    scale = oracle_abs_scale(w.build, w.metric, host64, bcs, batch)
    for k in want64:
        exact = np.array([math.fsum(row) for row in want64[k]])
        tol = 1e-12 * np.maximum(np.abs(want64[k]).sum(axis=1), scale[k].sum(axis=1)) + 1e-300
        assert (np.abs(sums[k] - exact) <= tol).all(), f"{name}: table batch-sum of grade {k} off"


# ---- source, keys and errors ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_wide_sources(name):
    w = W.WORKLOADS[name]
    plan = g.Plan(None, W.specialize(w))
    b = w.broadcast_mask()
    for arith in (L.ARITH_FMA, L.ARITH_STRICT):
        # on f64 batches the flag changes nothing: the same text, hence the same cache key
        assert plan.kernel_source(b, arith | L.ARITH_F64) == plan.kernel_source(b, arith)
        assert plan.kernel_source(b, arith | L.ARITH_F64, True, False) == plan.kernel_source(b, arith, True, False)
        wide = plan.kernel_source(b, arith | L.ARITH_F64, dtype=L.F32)
        f32 = plan.kernel_source(b, arith, dtype=L.F32)
        assert wide != f32
        assert "dtype=f32 arith=f64" in wide.split("\n")[0] and "arith=f64" not in f32.split("\n")[0]
        assert "f32-storage-f64-arith" in wide.split("\n")[1]
        assert "__double2float_rn" in wide and "const float* __restrict__" in wide
    plan.free()


def test_unknown_arith_bits_are_invalid():
    w = W.WORKLOADS["cfg1"]
    plan = g.Plan(None, W.specialize(w))
    for arith in (4, 8, 6, -1):
        with pytest.raises(L.GaastError) as e:
            plan.precompile(w.broadcast_mask(), arith, dtype=L.F32)
        assert e.value.status == L.ERR_INVALID
        assert L.lib.gaast_plan_kernel_source(plan._h, w.broadcast_mask(), arith, 4, None, 0) == 0
        assert "unknown arith" in L.last_error()
    plan.free()


def test_precompiled_variants_include_the_wide_mode():
    for w in W.WORKLOADS.values():
        v = W.precompile_variants(w)
        assert (FMA64, False, True, L.F32) in v
        assert ((FMA64, True, True, L.F32) in v) == bool(w.sum_root)


def test_rust_constant_matches_the_header():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    h = open(os.path.join(root, "include", "gaast_b200.h")).read()
    rs = open(os.path.join(root, "rust", "gaast-b200-sys", "src", "lib.rs")).read()
    assert int(re.search(r"#define GAAST_ARITH_F64 (\d+)", h).group(1)) == L.ARITH_F64 == 2
    assert int(re.search(r"pub const GAAST_ARITH_F64: c_int = (\d+);", rs).group(1)) == L.ARITH_F64
