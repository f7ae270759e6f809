"""f32 batches evaluated in binary64 (GAAST_ARITH_F64, include/gaast_b200.h) on the device.

Bars: STRICT | F64 bit-identical to float32(the plan's operation sequence in binary64 on the widened inputs), on both
engines (so the two engines agree bit for bit); FMA | F64 within 0.5 ulp(binary32) + 1e-12 of max(|ref|, sum |terms|)
of the f64 oracle; batch sums within 1e-12 of the exact sum of the f64 oracle (they add the unrounded results)."""
import math
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from gaast_b200.expr import Input, mv as pmv  # noqa: E402
from tests.guarded_layout import GuardedBatch, check, check_owned, poison_owned  # noqa: E402
from tests.helpers import assert_bit_exact, oracle_abs_scale, oracle_eval  # noqa: E402
from tests.test_f32_wide_on_cpu import (FMA64, LOWERING, NAMES, STRICT64, assert_within_one_rounding,  # noqa: E402
                                        f32_inputs, strict_want)

ENGINES = [("table", L.ENGINE_TABLE), ("specialized", L.ENGINE_SPECIALIZED)]


@pytest.fixture(scope="module")
def ctx():
    c = g.Ctx(0)
    yield c
    c.close()


def upload(ctx, w, host):
    return [g.DeviceBatch.from_host(ctx, w.n, host[s], broadcast=bc, dtype=L.F32) for s, (_, bc) in enumerate(w.inputs)]


@pytest.mark.parametrize("name", NAMES)
def test_workloads_on_both_engines(ctx, name):
    w = W.WORKLOADS[name]
    batch = 4096 + 6
    host, host64 = f32_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    ast = W.specialize(w)
    want32 = strict_want(ast, host64, batch)
    want = oracle_eval(w.build, w.metric, host64, bcs, batch)
    scale = oracle_abs_scale(w.build, w.metric, host64, bcs, batch)
    plan = g.Plan(ctx, ast)
    dev = upload(ctx, w, host)
    strict = {}
    for ename, engine in ENGINES:
        out = plan.eval(dev, engine=engine, arith=STRICT64)
        ctx.sync()
        assert out.dtype == L.F32 and f"engine={ename}" in plan.last_kernel()
        strict[ename] = out.to_host()
        assert_bit_exact(strict[ename], want32, f"{name} {ename} strict|f64 [{plan.last_kernel()}]")
        out = plan.eval(dev, engine=engine, arith=FMA64)
        ctx.sync()
        assert f"engine={ename}" in plan.last_kernel()
        assert_within_one_rounding(out.to_host(), want, scale, f"{name} {ename} fma|f64 [{plan.last_kernel()}]")
    for k in strict["table"]:
        assert np.array_equal(strict["table"][k].view(np.uint32), strict["specialized"][k].view(np.uint32))
    notes = plan.kernel_source(w.broadcast_mask(), FMA64, dtype=L.F32).split("\n")[1]
    if name in LOWERING:
        assert LOWERING[name] in notes, notes
    plan.free()


LAYOUTS = {"odd-length-owned": None, "odd-stride": (1, 0), "misaligned": (0, 1), "odd-stride-misaligned": (3, 1)}


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg5"])
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_guarded_layouts(ctx, name, layout):
    """Caller-owned inputs and outputs with gaps after each row and misaligned base pointers, and an odd length into a
    library-owned output: values (strict, bit-exact) and write containment.  cfg2 reads its rotor as a broadcast
    operand."""
    import torch
    w = W.WORKLOADS[name]
    length = 1001
    host, host64 = f32_inputs(w, length)
    ast = W.specialize(w)
    want32 = strict_want(ast, host64, length)
    plan = g.Plan(ctx, ast)
    lay = LAYOUTS[layout]
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
        if lay is None:
            dev = upload(ctx, w, host)
            out = poison_owned(plan.alloc_output(length, L.F32))
            guarded_in, gout = [], None
        else:
            dev, guarded_in = [], []
            for s, (grades, bc) in enumerate(w.inputs):
                gb = GuardedBatch.dense(w.n, grades, 1 if bc else length, gap=lay[0], offset=lay[1], dtype=np.float32,
                                        role="in", device="cuda:0")
                gb.fill(host[s])
                guarded_in.append(gb)
                dev.append(gb.wrap(ctx, w.n, broadcast=bc))
            gout = GuardedBatch({k: comb(w.n, k) for k in plan.root_grades()}, length, gap=lay[0], offset=lay[1],
                                dtype=np.float32, role="out", device="cuda:0")
            out = gout.wrap(ctx, w.n)
        torch.cuda.synchronize()
        before = [(b, b.bits()) for b in guarded_in]
        plan.eval(dev, out=out, engine=engine, arith=STRICT64)
        ctx.sync()
        what = f"{name} {layout} [{plan.last_kernel()}]"
        check([gout] if gout else [], before, what)
        got = gout.values() if gout else out.to_host()
        if gout is None:
            check_owned(got, np.float32, what)
        assert_bit_exact(got, want32, what)
    plan.free()


class SumBuffer:
    def __init__(self, cols):
        import torch
        self.t = torch.full((max(1, cols),), float("nan"), dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()

    def read(self, ctx):
        ctx.sync()
        return self.t.cpu().numpy()


@pytest.mark.parametrize("name", ["cfg1", "cfg5"])
@pytest.mark.parametrize("length", [1, 129, 1001, 200_000 + 3])
@pytest.mark.parametrize("stored", [True, False], ids=["stored", "sums-only"])
def test_batch_sums(ctx, name, length, stored):
    """The sums add the unrounded binary64 results: 1e-12 against the exact sum of the f64 oracle, stored output or
    out=None; 200 003 elements span many tiles and blocks."""
    w = W.WORKLOADS[name]
    host, host64 = f32_inputs(w, length)
    bcs = [bc for _, bc in w.inputs]
    want = oracle_eval(w.build, w.metric, host64, bcs, length)
    scale = oracle_abs_scale(w.build, w.metric, host64, bcs, length)
    plan = g.Plan(ctx, W.specialize(w))
    dev = upload(ctx, w, host)
    cols = sum(comb(w.n, k) for k in plan.root_grades())
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
        out = plan.alloc_output(length, L.F32) if stored else None
        buf = SumBuffer(cols)
        plan.eval_sum(dev, buf.t.data_ptr(), out=out, engine=engine, arith=FMA64)
        sums = buf.read(ctx)
        what = f"{name} n={length} [{plan.last_kernel()}]"
        c = 0
        for k in plan.root_grades():
            exact = np.array([math.fsum(row) for row in want[k]])
            tol = 1e-12 * np.maximum(np.abs(want[k]).sum(axis=1), scale[k].sum(axis=1)) + 1e-300
            err = np.abs(sums[c:c + comb(w.n, k)] - exact)
            assert (err <= tol).all(), f"{what}: grade {k} off by {(err / tol).max():.1f} x the bar"
            c += comb(w.n, k)
        if stored:
            assert_within_one_rounding(out.to_host(), want, scale, what)
    plan.free()


def test_sparse_inputs_projection_and_exp_log(ctx):
    w = W.WORKLOADS["cfg5"]
    ast = W.specialize(w)
    length = 1001
    host, host64 = f32_inputs(w, length)
    keep = list(range(0, 66, 3))
    for h in (host, host64):
        h[1][2][[i for i in range(66) if i not in keep]] = 0.0
    want32 = strict_want(ast, host64, length)
    dev = [g.DeviceBatch.from_host(ctx, w.n, host[0], dtype=L.F32),
           g.DeviceBatch.from_host_sparse(ctx, w.n, {2: (keep, host[1][2][keep])}, dtype=L.F32)]
    plan = g.Plan(ctx, ast)
    got = plan.eval(dev, arith=STRICT64).to_host()
    ctx.sync()
    assert_bit_exact(got, want32, f"sparse [{plan.last_kernel()}]")
    comps = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}
    proj = g.Plan(ctx, ast, components=comps)
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
        dense_in = upload(ctx, w, host)
        out = proj.eval(dense_in, out=proj.alloc_output(length, L.F32), engine=engine, arith=STRICT64)
        ctx.sync()
        assert_bit_exact(out.to_host(), {2: want32[2][comps[2]]}, f"projected [{proj.last_kernel()}]")
    # exp / log: a rotor from a bivector, R X ~R
    from tests.test_explog import _oracle
    n = 3
    rng = np.random.default_rng(4)
    hb = [{2: rng.uniform(-2, 2, (3, length)).astype(np.float32)}, {1: rng.uniform(-1, 1, (3, length)).astype(np.float32)}]
    build = lambda b, x: ((b * -0.5).exp() * x * (b * -0.5).exp().rev()).g(1)  # noqa: E731
    want = _oracle(build, [1.0] * n, [{k: v.astype(np.float64) for k, v in d.items()} for d in hb], length)
    ep = g.Plan(ctx, build(pmv(Input(0, (2,))), pmv(Input(1, (1,)))).specialize([1.0] * n))
    edev = [g.DeviceBatch.from_host(ctx, n, d, dtype=L.F32) for d in hb]
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
        for arith in (STRICT64, FMA64):
            got = ep.eval(edev, engine=engine, arith=arith).to_host()
            ctx.sync()
            for k in want:
                ulp = np.spacing(np.abs(want[k]).astype(np.float32)).astype(np.float64)
                tol = 1e-12 * np.maximum(np.abs(want[k]), 1.0) + 0.5 * ulp
                err = np.abs(got[k].astype(np.float64) - want[k])
                assert (err <= tol).all(), (engine, arith, k, err.max())


def test_eval_host_f32_matches_the_device(ctx):
    w = W.WORKLOADS["cfg2"]
    batch = 300_000 + 6
    host, _ = f32_inputs(w, batch)
    bcs = [bc for _, bc in w.inputs]
    plan = g.Plan(ctx, W.specialize(w))
    want = plan.eval(upload(ctx, w, host), engine=L.ENGINE_SPECIALIZED, arith=FMA64).to_host()
    ctx.sync()
    flat_in = [np.ascontiguousarray(np.concatenate([d[k] for k in gr], axis=0)) for (gr, _), d in zip(w.inputs, host)]
    rows = sum(comb(w.n, k) for k in plan.root_grades())
    out = np.zeros((rows, batch), dtype=np.float32)
    plan.eval_host(flat_in, [gr for gr, _ in w.inputs], bcs, batch, out, engine=L.ENGINE_SPECIALIZED, arith=FMA64)
    r = 0
    for k in plan.root_grades():
        assert np.array_equal(out[r:r + comb(w.n, k)].view(np.uint32), want[k].view(np.uint32)), k
        r += comb(w.n, k)


def test_errors_and_the_f64_identity(ctx):
    w = W.WORKLOADS["cfg1"]
    batch = 1000
    host, host64 = f32_inputs(w, batch)
    plan = g.Plan(ctx, W.specialize(w))
    dev32 = upload(ctx, w, host)
    with pytest.raises(L.GaastError) as e:
        plan.eval(dev32, engine=L.ENGINE_DENSE_WARP, arith=FMA64)
    assert e.value.status == L.ERR_UNSUPPORTED
    dev64 = [g.DeviceBatch.from_host(ctx, w.n, host64[s], broadcast=bc) for s, (_, bc) in enumerate(w.inputs)]
    with pytest.raises(L.GaastError) as e:
        plan.eval([dev64[0]] + dev32[1:], out=plan.alloc_output(batch, L.F32), arith=FMA64)
    assert e.value.status == L.ERR_SHAPE
    for arith in (4, 6, 8):
        with pytest.raises(L.GaastError) as e:
            plan.eval(dev32, arith=arith)
        assert e.value.status == L.ERR_INVALID
    for arith in (L.ARITH_FMA, L.ARITH_STRICT):
        for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
            a = plan.eval(dev64, engine=engine, arith=arith).to_host()
            ka = plan.last_kernel().split(" grid=")[0] + plan.last_kernel().split("key=")[-1]
            b = plan.eval(dev64, engine=engine, arith=arith | L.ARITH_F64).to_host()
            kb = plan.last_kernel().split(" grid=")[0] + plan.last_kernel().split("key=")[-1]
            ctx.sync()
            assert ka == kb
            for k in a:
                assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64))
    plan.free()


def test_graph_replay_and_launch_count():
    import torch
    w = W.WORKLOADS["cfg5"]
    length = 300_000 + 6
    ctx = g.Ctx.on_torch_stream(0)
    try:
        host, _ = f32_inputs(w, length)
        plan = g.Plan(ctx, W.specialize(w))
        dev = upload(ctx, w, host)
        cols = sum(comb(w.n, k) for k in plan.root_grades())
        out = plan.alloc_output(length, L.F32)
        direct = SumBuffer(cols)
        plan.eval_sum(dev, direct.t.data_ptr(), out=out, engine=L.ENGINE_SPECIALIZED, arith=FMA64)
        want_sum, want_out = direct.read(ctx), out.to_host()
        ctx.sync()
        counts = []
        for _ in range(2):
            n0 = ctx.launch_count
            plan.eval_sum(dev, direct.t.data_ptr(), out=out, engine=L.ENGINE_SPECIALIZED, arith=FMA64)
            ctx.sync()
            counts.append(ctx.launch_count - n0)
        # a later call only launches: the uniform prologue, the kernel and the partial-sum reduction
        assert counts[0] == counts[1] and 2 <= counts[0] <= 4, (counts, plan.last_kernel())
        buf = SumBuffer(cols)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ctx.torch_stream):
            plan.eval_sum(dev, buf.t.data_ptr(), out=out, engine=L.ENGINE_SPECIALIZED, arith=FMA64)
        for _ in range(2):
            buf.t.fill_(float("nan"))
            graph.replay()
            torch.cuda.synchronize()
            assert np.array_equal(buf.read(ctx).view(np.uint64), want_sum.view(np.uint64))
            got = out.to_host()
            ctx.sync()
            for k in got:
                assert np.array_equal(got[k].view(np.uint32), want_out[k].view(np.uint32))
        del graph
    finally:
        torch.cuda.set_stream(torch.cuda.default_stream(0))
        ctx.sync()


def test_cfg5_at_32m_elements(ctx):
    """cfg5 at 32 M elements (f32 batches made on the device), against the oracle on 4 096 seeded sample columns."""
    import torch
    w = W.WORKLOADS["cfg5"]
    length = 32 << 20
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(32)
    tensors = []
    for grades, bc in w.inputs:
        tensors.append({k: torch.empty((comb(w.n, k), 1 if bc else length), dtype=torch.float32, device="cuda:0")
                        .uniform_(-1.0, 1.0, generator=gen) for k in grades})
    tctx = g.Ctx.on_torch_stream(0)
    try:
        plan = g.Plan(tctx, W.specialize(w))
        dev = [g.DeviceBatch.wrap_torch(tctx, w.n, t, broadcast=bc) for t, (_, bc) in zip(tensors, w.inputs)]
        out_t = {k: torch.empty((comb(w.n, k), length), dtype=torch.float32, device="cuda:0") for k in plan.root_grades()}
        plan.eval(dev, out=g.DeviceBatch.wrap_torch(tctx, w.n, out_t), engine=L.ENGINE_SPECIALIZED, arith=FMA64)
        tctx.sync()
        assert "engine=specialized" in plan.last_kernel()
        cols = np.sort(np.random.default_rng(7).choice(length, 4096, replace=False))
        idx = torch.from_numpy(cols).to("cuda:0")
        host64 = [{k: (v[:, :1] if bc else v[:, idx]).double().cpu().numpy() for k, v in t.items()}
                  for t, (_, bc) in zip(tensors, w.inputs)]
        bcs = [bc for _, bc in w.inputs]
        want = oracle_eval(w.build, w.metric, host64, bcs, len(cols))
        scale = oracle_abs_scale(w.build, w.metric, host64, bcs, len(cols))
        got = {k: v[:, idx].cpu().numpy() for k, v in out_t.items()}
        assert_within_one_rounding(got, want, scale, f"cfg5 32M [{plan.last_kernel()}]")
    finally:
        torch.cuda.set_stream(torch.cuda.default_stream(0))
        tctx.sync()
