"""Projected plans (gaast_plan_create_projected) on the device: a plan that keeps only chosen root components and writes
them to a sparse output batch.  Held to the oracle's selected rows (strict arithmetic bit for bit on the specialised and
on the table engine, FMA within 1e-12), to the unprojected plan's rows, and to math.fsum for the batch sums."""
import ctypes as C
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from tests.helpers import (REL_TOL_F32, assert_bit_exact, assert_close, oracle_abs_scale, oracle_eval,  # noqa: E402
                           run_plan_numpy)
from tests.test_gpu_batch_sum import REL_SUM, SumBuffer, fsum_cols  # noqa: E402

NAMES = ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"]
CFG5_9 = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}


@pytest.fixture(scope="module")
def ctx():
    return g.Ctx(0)


def seeded_projection(name, n, grades, seed=0):
    """About a third of each root grade (at least one component); cfg3 keeps grade 3 whole and empties grade 6."""
    rng = np.random.default_rng(2000 + seed)
    comps = {k: sorted(int(i) for i in rng.choice(comb(n, k), max(1, comb(n, k) // 3), replace=False)) for k in grades}
    if name == "cfg3":
        del comps[3]
        comps[6] = []
    return comps


def select(res, comps):
    return {k: (v[comps[k]] if k in comps else v) for k, v in res.items()}


def upload(ctx, w, host, dtype=L.F64):
    return [g.DeviceBatch.from_host(ctx, w.n, d, broadcast=bc, dtype=dtype) for d, (_, bc) in zip(host, w.inputs)]


def setup(ctx, name, batch, seed=0, dtype=L.F64):
    w = W.WORKLOADS[name]
    ast = W.specialize(w)
    plain = g.Plan(ctx, ast)
    comps = seeded_projection(name, w.n, plain.root_grades(), seed)
    proj = g.Plan(ctx, ast, components=comps)
    host = W.host_inputs(w, batch)
    if dtype == L.F32:
        host = [{k: v.astype(np.float32) for k, v in d.items()} for d in host]
    return w, ast, plain, proj, comps, host, upload(ctx, w, host, dtype)


def fma_of(kernel):
    return int([t for t in kernel.split() if t.startswith("fma/elem=")][0][9:])


# ---- 1. cfg1-cfg5 against the oracle's selected rows ---------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("batch", [1000, 1001])
def test_projected_against_oracle(ctx, name, batch):
    w, ast, plain, proj, comps, host, dev = setup(ctx, name, batch)
    bcs = [bc for _, bc in w.inputs]
    want = select(oracle_eval(w.build, w.metric, host, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host, bcs, batch), comps)
    for engine in (L.ENGINE_AUTO, L.ENGINE_SPECIALIZED):
        out = proj.eval(dev, engine=engine, arith=L.ARITH_FMA)
        ctx.sync()
        assert_close(out.to_host(), want, scale, what=f"{name} projected fma [{proj.last_kernel()}]")
    full = plain.eval(dev, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_STRICT).to_host()
    for engine, tag in ((L.ENGINE_SPECIALIZED, "engine=specialized"), (L.ENGINE_TABLE, "engine=table")):
        out = proj.eval(dev, engine=engine, arith=L.ARITH_STRICT)
        ctx.sync()
        assert tag in proj.last_kernel(), proj.last_kernel()
        got = out.to_host()
        assert_bit_exact(got, want, f"{name} projected strict {tag}")
        assert_bit_exact(got, select(full, comps), f"{name} projected strict {tag} vs the unprojected plan")
        for k in got:
            assert out.stored_rows(k) == (len(comps[k]) if k in comps else comb(w.n, k))


@pytest.mark.parametrize("name", NAMES)
def test_projected_f32(ctx, name):
    batch = 1002
    w, ast, plain, proj, comps, host, dev = setup(ctx, name, batch, seed=1, dtype=L.F32)
    bcs = [bc for _, bc in w.inputs]
    with np.errstate(all="ignore"):
        want32 = select(run_plan_numpy(ast.plan_dict(), host, batch, dtype=np.float32), comps)
    out = proj.eval(dev, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_STRICT)
    ctx.sync()
    assert_bit_exact(out.to_host(), want32, f"{name} projected f32 strict")
    host64 = [{k: v.astype(np.float64) for k, v in d.items()} for d in host]
    want = select(oracle_eval(w.build, w.metric, host64, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host64, bcs, batch), comps)
    out = proj.eval(dev, arith=L.ARITH_FMA)
    ctx.sync()
    assert_close({k: v.astype(np.float64) for k, v in out.to_host().items()}, want, scale, rel=REL_TOL_F32,
                 what=f"{name} projected f32 fma")


def test_wrapped_sparse_output_takes_the_unaligned_kernel(ctx):
    """A caller-owned sparse output (gaast_batch_wrap_sparse) with an odd length: one element per thread."""
    import torch
    batch = 999
    w, ast, plain, proj, comps, host, dev = setup(ctx, "cfg5", batch)
    want = select(oracle_eval(w.build, w.metric, host, [False, False], batch), comps)
    t = torch.full((len(comps[2]), batch), float("nan"), dtype=torch.float64, device="cuda:0")
    bits = (L.u64 * 2)()
    for i in comps[2]:
        bits[i // 64] |= 1 << (i % 64)
    pres = (C.POINTER(L.u64) * 1)(C.cast(bits, C.POINTER(L.u64)))
    ptrs = (L.vp * 1)(t.data_ptr())
    h = L.vp()
    L.check(L.lib.gaast_batch_wrap_sparse(ctx._h, w.n, 1 << 2, batch, batch, 0, L.F64, pres, ptrs, C.byref(h)))
    out = g.DeviceBatch(h, ctx, w.n, keep=(t, bits))
    torch.cuda.synchronize()
    proj.eval(dev, out=out, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_STRICT)
    ctx.sync()
    assert "elems/thread=1" in proj.last_kernel(), proj.last_kernel()
    assert_bit_exact({2: t.cpu().numpy()}, want, "wrapped sparse output")


# ---- 2. the policy the generator takes, and the FMAs it executes -------------------------------------------------
def test_fma_count_and_policy(ctx):
    batch = 4096
    # cfg5, 9 of 66: pruned liveness, strictly fewer FMAs
    w, ast, plain, _, _, host, dev = setup(ctx, "cfg5", batch)
    proj = g.Plan(ctx, ast, components=CFG5_9)
    plain.eval(dev, engine=L.ENGINE_SPECIALIZED)
    proj.eval(dev, engine=L.ENGINE_SPECIALIZED)
    ctx.sync()
    assert fma_of(proj.last_kernel()) < fma_of(plain.last_kernel()), (proj.last_kernel(), plain.last_kernel())
    src = proj.kernel_source()
    assert "projection(9/66,pruned)" in src.split("\n")[1]
    # cfg3: the matrix-representation product stays when most components are kept, the pruned terms when few are
    w3, ast3, plain3, _, _, host3, dev3 = setup(ctx, "cfg3", batch)
    plain3.eval(dev3, engine=L.ENGINE_SPECIALIZED)
    ctx.sync()
    base = fma_of(plain3.last_kernel())
    for comps, policy in (({6: []}, "whole"), ({0: [0], 1: [], 2: [], 3: [1], 4: [], 5: [], 6: []}, "pruned")):
        p = g.Plan(ctx, ast3, components=comps)
        notes = p.kernel_source().split("\n")[1]
        assert f",{policy})" in notes, notes
        assert ("dense-matrep" in notes) == (policy == "whole"), notes
        p.eval(dev3, engine=L.ENGINE_SPECIALIZED)
        ctx.sync()
        assert fma_of(p.last_kernel()) <= base, (p.last_kernel(), base)
        bcs = [False, False]
        want = select(oracle_eval(w3.build, w3.metric, host3, bcs, batch), comps)
        scale = select(oracle_abs_scale(w3.build, w3.metric, host3, bcs, batch), comps)
        assert_close(p.eval(dev3).to_host(), want, scale, what=f"cfg3 {policy}")


# ---- 3. batch sums --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,variant,path", [("cfg5", 0, "smem"), ("cfg5", 262144, "tmem"), ("cfg3", 0, "tmem"),
                                               ("cfg1", 0, "smem"), ("cfg2", 0, "smem"), ("cfg4", 0, None)])
def test_projected_batch_sum(ctx, name, variant, path):
    batch = 20_000
    w, ast, plain, proj, comps, host, dev = setup(ctx, name, batch, seed=2)
    proj.set_tuning(0, variant)
    bcs = [bc for _, bc in w.inputs]
    want = select(oracle_eval(w.build, w.metric, host, bcs, batch), comps)
    scale = select(oracle_abs_scale(w.build, w.metric, host, bcs, batch), comps)
    grades = sorted(want)
    cols = sum(want[k].shape[0] for k in grades)
    wcat = np.concatenate([want[k] for k in grades])
    scat = np.concatenate([scale[k] for k in grades])
    bound = REL_SUM * np.maximum(np.abs(wcat), scat).sum(axis=1)
    for store in (True, False):
        buf = SumBuffer(cols)
        out = proj.alloc_output(batch) if store else None
        proj.eval_sum(dev, buf.ptr, out=out, engine=L.ENGINE_SPECIALIZED)
        got = buf.read(ctx)  # (the guards right after the stored-count vector are checked here)
        assert (np.abs(got - fsum_cols(wcat)) <= bound).all(), f"{name} projected sum [{proj.last_kernel()}]"
        notes = proj.kernel_source(with_sum=True, store_out=store, broadcast_slots=sum(
            1 << s for s, (_, bc) in enumerate(w.inputs) if bc)).split("\n")[1]
        if path == "tmem":
            assert "sum-in-tmem" in notes, notes
        elif path == "smem":
            assert "sum-in-tmem" not in notes, notes
        if store:
            assert_close(out.to_host(), want, scale, what=f"{name} projected + sum")
    # the table engine sums the same columns
    buf = SumBuffer(cols)
    proj.eval_sum(dev, buf.ptr, out=None, engine=L.ENGINE_TABLE)
    assert (np.abs(buf.read(ctx) - fsum_cols(wcat)) <= bound).all(), f"{name} projected sum, table engine"
    # an empty batch zeroes exactly the stored count
    empty = upload(ctx, w, [{k: v[:, :0] if not bc else v for k, v in d.items()} for d, (_, bc) in zip(host, w.inputs)])
    buf = SumBuffer(cols)
    proj.eval_sum(empty, buf.ptr, out=None)
    assert (buf.read(ctx) == 0.0).all()


# ---- 4. the output contract -----------------------------------------------------------------------------------------
def test_output_contract(ctx):
    batch = 512
    w, ast, plain, proj, comps, host, dev = setup(ctx, "cfg5", batch)
    sparse_out = proj.alloc_output(batch)
    with pytest.raises(g.GaastError) as ei:
        plain.eval(dev, out=sparse_out)
    assert ei.value.status == L.ERR_SHAPE
    with pytest.raises(g.GaastError) as ei:
        proj.eval(dev, out=plain.alloc_output(batch))
    assert ei.value.status == L.ERR_SHAPE
    other = g.DeviceBatch.alloc_sparse(ctx, w.n, {2: comps[2][1:]}, batch)
    with pytest.raises(g.GaastError) as ei:
        proj.eval(dev, out=other)
    assert ei.value.status == L.ERR_SHAPE
    with pytest.raises(g.GaastError) as ei:
        proj.eval(dev, out=sparse_out, engine=L.ENGINE_DENSE_WARP)
    assert ei.value.status == L.ERR_UNSUPPORTED
    hin = [np.ascontiguousarray(host[0][1]), np.ascontiguousarray(host[1][2])]
    hout = np.zeros((len(comps[2]), batch))
    with pytest.raises(g.GaastError) as ei:
        proj.eval_host(hin, [(1,), (2,)], [False, False], batch, hout)
    assert ei.value.status == L.ERR_UNSUPPORTED
    # the identity projection is the plain plan: dense out, bit-identical results
    ident = g.Plan(ctx, ast, components={2: range(66)})
    a = ident.eval(dev, out=plain.alloc_output(batch), arith=L.ARITH_FMA)
    b = plain.eval(dev, arith=L.ARITH_FMA)
    ctx.sync()
    assert_bit_exact(a.to_host(), b.to_host(), "identity projection")
    # cost: stored components only, the reference's flops
    assert proj.cost()[0] == 8 * (12 + 66 + len(comps[2])) and proj.cost()[1] == plain.cost()[1]


# ---- 5. chaining and records ----------------------------------------------------------------------------------
def test_chain_and_records(ctx):
    batch = 777
    w, ast, plain, proj, comps, host, dev = setup(ctx, "cfg5", batch)
    proj = g.Plan(ctx, ast, components=CFG5_9)
    first = proj.eval(dev, arith=L.ARITH_STRICT)
    ctx.sync()
    dense_first = plain.eval(dev, arith=L.ARITH_STRICT).to_host()
    zeroed = np.zeros_like(dense_first[2])
    zeroed[CFG5_9[2]] = dense_first[2][CFG5_9[2]]
    # records: unselected components are +0
    rec = first.to_records()
    assert np.array_equal(rec.T.view(np.uint64), zeroed.view(np.uint64))
    # the sparse result as the X of a second sandwich, against the dense chain with the zeros written out
    second = plain.eval([dev[0], first], arith=L.ARITH_STRICT)
    ctx.sync()
    Xd = g.DeviceBatch.from_host(ctx, w.n, {2: zeroed})
    ref = plain.eval([dev[0], Xd], arith=L.ARITH_STRICT)
    ctx.sync()
    assert_bit_exact(second.to_host(), ref.to_host(), "projected result chained as a sparse input")


# ---- 6. full size and capture -----------------------------------------------------------------------------------
def test_full_size_cfg5_on_device():
    """cfg5 at 32 M elements, 9 of 66 components, strict: the stored rows equal the unprojected plan's, on the device."""
    import torch
    ctx = g.Ctx.on_torch_stream(0)
    try:
        w = W.WORKLOADS["cfg5"]
        length = 32 * 1024 * 1024
        tin = W.torch_inputs(w, length, "cuda:0")
        torch.cuda.synchronize()
        dev = [g.DeviceBatch.wrap_torch(ctx, w.n, t, broadcast=bc) for t, (_, bc) in zip(tin, w.inputs)]
        plain, proj = g.Plan(ctx, W.specialize(w)), g.Plan(ctx, W.specialize(w), components=CFG5_9)
        full = torch.empty((66, length), dtype=torch.float64, device="cuda:0")
        part = torch.empty((9, length), dtype=torch.float64, device="cuda:0")
        outf = g.DeviceBatch.wrap_torch(ctx, w.n, {2: full})
        h = L.vp()
        bits = (L.u64 * 2)()
        for i in CFG5_9[2]:
            bits[i // 64] |= 1 << (i % 64)
        pres = (C.POINTER(L.u64) * 1)(C.cast(bits, C.POINTER(L.u64)))
        L.check(L.lib.gaast_batch_wrap_sparse(ctx._h, w.n, 1 << 2, length, length, 0, L.F64, pres,
                                              (L.vp * 1)(part.data_ptr()), C.byref(h)))
        outp = g.DeviceBatch(h, ctx, w.n, keep=(part, bits))
        plain.eval(dev, out=outf, arith=L.ARITH_STRICT)
        proj.eval(dev, out=outp, arith=L.ARITH_STRICT)
        ctx.sync()
        torch.cuda.synchronize()
        sel = full[CFG5_9[2]]
        assert torch.equal(sel.view(torch.int64), part.view(torch.int64))
        # a CUDA-graph capture of the projected eval, replayed bit-identically
        part2 = part.clone()
        part.fill_(float("nan"))
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ctx.torch_stream):
            proj.eval(dev, out=outp, arith=L.ARITH_STRICT)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(part.view(torch.int64), part2.view(torch.int64))
        del graph
    finally:
        torch.cuda.set_stream(torch.cuda.default_stream(0))
