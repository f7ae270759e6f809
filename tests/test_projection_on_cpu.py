"""Projected plans (gaast_plan_create_projected) on a machine without a GPU: the kernel text of an offline plan, and the
generated kernels executed by the CPU stand-in of tests/kernel_emu against the oracle's selected rows.

A projected plan keeps only chosen root components; the others are zero and are neither computed nor stored.  In
strict arithmetic every stored component is bit-identical to the oracle (each output keeps the reference's term order),
FMA arithmetic stays within 1e-12, and the batch-sum has one column per stored component."""
import ctypes as C
from math import comb

import numpy as np
import pytest

import gaast_b200 as g
from gaast_b200 import _lib as L
from gaast_b200 import workloads as W
from tests.helpers import REL_TOL_F32, assert_bit_exact, assert_close, oracle_abs_scale, oracle_eval, run_plan_numpy
from tests.kernel_emu import run_generated_kernel

pytestmark = pytest.mark.timeout(600)

NAMES = ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"]


def seeded_projection(name, plan, seed=0):
    """About a third of each root grade's components, drawn from a seeded generator (at least one per grade).  cfg3
    (every grade of G(6)) also keeps grade 3 whole and empties grade 6."""
    rng = np.random.default_rng(1000 + seed)
    comps = {}
    for k in plan.root_grades():
        c = comb(plan.n, k)
        comps[k] = sorted(int(i) for i in rng.choice(c, max(1, c // 3), replace=False))
    if name == "cfg3":
        del comps[3]  # (not listed: kept whole)
        comps[6] = []
    return comps


def select(res, comps):
    return {k: (v[comps[k]] if k in comps else v) for k, v in res.items()}


def bmask_of(w):
    return sum(1 << s for s, (_, bc) in enumerate(w.inputs) if bc)


# ---- 1. the identity projection is gaast_plan_create's plan ------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_identity_projection_same_source(name):
    w = W.WORKLOADS[name]
    ast = W.specialize(w)
    plain = g.Plan(None, ast)
    ident = g.Plan(None, ast, components={k: range(comb(plain.n, k)) for k in plain.root_grades()})
    for dtype in (L.F64, L.F32):
        for with_sum in (False, True):
            kw = dict(broadcast_slots=bmask_of(w), with_sum=with_sum, dtype=dtype)
            assert ident.kernel_source(**kw) == plain.kernel_source(**kw), (name, dtype, with_sum)
    assert ident.cost(bmask_of(w)) == plain.cost(bmask_of(w))


# ---- 2. generated projected kernels against the oracle -----------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_projected_kernels_match_oracle(name):
    w = W.WORKLOADS[name]
    ast = W.specialize(w)
    comps = seeded_projection(name, g.Plan(None, ast))
    batch = 301
    host = W.host_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    want = select(oracle_eval(w.build, w.metric, host, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host, bcs, batch), comps)
    out, _, info = run_generated_kernel(ast, host, bcs, batch, arith=L.ARITH_STRICT, components=comps)
    assert "projection(" in info["notes"], info["notes"]
    assert_bit_exact(out, want, f"{name} projected strict [{info['notes']}]")
    out, _, info = run_generated_kernel(ast, host, bcs, batch, arith=L.ARITH_FMA, components=comps)
    assert_close(out, want, scale, what=f"{name} projected fma [{info['notes']}]")


@pytest.mark.parametrize("name", NAMES)
def test_projected_kernels_f32(name):
    w = W.WORKLOADS[name]
    ast = W.specialize(w)
    comps = seeded_projection(name, g.Plan(None, ast), seed=1)
    batch = 262
    host = [{k: v.astype(np.float32) for k, v in d.items()} for d in W.host_inputs(w, batch)]
    host64 = [{k: v.astype(np.float64) for k, v in d.items()} for d in host]
    bcs = [bc for _, bc in w.inputs]
    with np.errstate(all="ignore"):
        want32 = select(run_plan_numpy(ast.plan_dict(), host, batch, dtype=np.float32), comps)
    out, _, info = run_generated_kernel(ast, host, bcs, batch, arith=L.ARITH_STRICT, dtype=np.float32, components=comps)
    assert_bit_exact(out, want32, f"{name} projected f32 strict [{info['notes']}]")
    out, _, info = run_generated_kernel(ast, host, bcs, batch, arith=L.ARITH_FMA, dtype=np.float32, components=comps)
    want = select(oracle_eval(w.build, w.metric, host64, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host64, bcs, batch), comps)
    assert_close({k: v.astype(np.float64) for k, v in out.items()}, want, scale, rel=REL_TOL_F32,
                 what=f"{name} projected f32 fma [{info['notes']}]")


SUM_CASES = [("cfg1", 0), ("cfg2", 0), ("cfg3", 0), ("cfg4", 0), ("cfg5", 0), ("cfg5", 262144),
             ("cfg5", 65536 | 262144)]


@pytest.mark.parametrize("name,variant", SUM_CASES, ids=[f"{n}-v{v}" for n, v in SUM_CASES])
@pytest.mark.parametrize("store_out", [True, False])
def test_projected_batch_sum(name, variant, store_out):
    """One sum column per stored component, in stored-row order; sums in shared memory (variant 0) and in tensor
    memory (262144; with 65536 the kernel without the reflection lowering)."""
    w = W.WORKLOADS[name]
    ast = W.specialize(w)
    comps = seeded_projection(name, g.Plan(None, ast), seed=2)
    batch = 600
    host = W.host_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    want = select(oracle_eval(w.build, w.metric, host, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host, bcs, batch), comps)
    out, sums, info = run_generated_kernel(ast, host, bcs, batch, arith=L.ARITH_FMA, with_sum=True, store_out=store_out,
                                           tuning=(0, variant), grid=2, components=comps)
    if variant & 262144:
        assert "sum-in-tmem" in info["notes"], info["notes"]
    if store_out:
        assert_close(out, want, scale, what=f"{name} projected + sum [{info['notes']}]")
    for k in want:
        assert sums[k].shape == (want[k].shape[0],)
        ref = want[k].sum(axis=1)
        tol = 1e-12 * np.maximum(np.abs(want[k]).sum(axis=1), scale[k].sum(axis=1)) + 1e-300
        assert (np.abs(sums[k] - ref) <= tol).all(), f"{name}: projected batch-sum of grade {k} off [{info['notes']}]"


def test_projected_plan_with_sparse_inputs():
    """cfg5 with a sparse bivector input and a projected result: strict bit-exact against the oracle."""
    w = W.WORKLOADS["cfg5"]
    ast = W.specialize(w)
    batch = 257
    host = W.host_inputs(w, batch)
    keep_in = list(range(0, 66, 3))
    host[1][2][[i for i in range(66) if i not in keep_in]] = 0.0
    want = oracle_eval(w.build, w.metric, host, [False, False], batch)
    comps = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}
    sparse_host = [host[0], {2: host[1][2][keep_in]}]
    out, _, info = run_generated_kernel(ast, sparse_host, [False, False], batch, arith=L.ARITH_STRICT,
                                        present={(1, 2): keep_in}, components=comps)
    assert_bit_exact(out, select(want, comps), f"sparse inputs + projection [{info['notes']}]")


def test_projection_lowers_fma_count():
    """Pruned liveness executes fewer FMAs: cfg5 with 9 of its 66 components; cfg3's matrix-representation product is
    kept (its outputs computed whole, only the selected ones stored) when that is cheaper than the pruned terms."""
    def fma(src):
        return src.count("d_fma(") + src.count("d_mul(")
    w = W.WORKLOADS["cfg5"]
    ast = W.specialize(w)
    plain = g.Plan(None, ast).kernel_source()
    proj = g.Plan(None, ast, components={2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}).kernel_source()
    assert "projection(9/66,pruned)" in proj.split("\n")[1]
    assert fma(proj) < fma(plain)
    ast3 = W.specialize(W.WORKLOADS["cfg3"])
    many = g.Plan(None, ast3, components={6: []}).kernel_source()  # 63 of 64
    assert "projection(63/64,whole)" in many.split("\n")[1] and "dense-matrep" in many.split("\n")[1]
    few = g.Plan(None, ast3, components={0: [0], 1: [], 2: [], 3: [], 4: [], 5: [], 6: []}).kernel_source()
    assert "projection(1/64,pruned)" in few.split("\n")[1] and "dense-matrep" not in few.split("\n")[1]


# ---- 3. errors on an offline plan ------------------------------------------------------------------------------------
def _create(ast, maps):
    out = L.vp()
    ptrs = None if maps is None else (C.POINTER(L.u64) * max(1, len(maps)))(
        *[C.cast(m, C.POINTER(L.u64)) if m is not None else None for m in maps])
    return L.lib.gaast_plan_create_projected(None, ast.lower(), ptrs, C.byref(out)), out


def test_projection_errors():
    ast = W.specialize(W.WORKLOADS["cfg5"])
    empty = (L.u64 * 2)(0, 0)
    st, out = _create(ast, [empty])
    assert st == L.ERR_SHAPE and not out.value
    st, out = _create(ast, None)
    assert st == L.ERR_INVALID and not out.value
    # bits past C(12, 2) = 66 are ignored: component 1 plus every bit of the second word above bit 1
    bits = (L.u64 * 2)(1 << 1, ~0x3 & (2 ** 64 - 1))
    st, out = _create(ast, [bits])
    assert st == L.OK
    p1 = g.Plan(None, ast, components={2: [1]})
    buf = C.create_string_buffer(1 << 22)
    L.lib.gaast_plan_kernel_source(out, 0, L.ARITH_FMA, 0, buf, len(buf))
    assert buf.value.decode() == p1.kernel_source()
    L.lib.gaast_plan_destroy(out)
    # every bit set (past C(n,k) too): the identity projection
    st, out = _create(ast, [(L.u64 * 2)(2 ** 64 - 1, 2 ** 64 - 1)])
    assert st == L.OK
    L.lib.gaast_plan_kernel_source(out, 0, L.ARITH_FMA, 0, buf, len(buf))
    assert buf.value.decode() == g.Plan(None, ast).kernel_source()
    L.lib.gaast_plan_destroy(out)
