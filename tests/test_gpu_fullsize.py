"""Parity at the FULL BASELINE.json batch sizes, through size-independent properties
(the oracle cannot evaluate 16-64 M elements in seconds), plus an oracle check of
a strided sample of the very same device inputs.

 * exact homogeneity: scaling an operand by 2 scales the result by 2 or 4, bit for bit
   (powers of two commute with every rounding);
 * invariants of the algebra: a unit rotor / an invertible vector sandwich preserves
   the scalar product X.X (within 1e-12 of the sum of magnitudes);
 * a 4096-element strided sample downloaded and compared with the oracle."""
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from tests.helpers import assert_close, oracle_abs_scale, oracle_eval  # noqa: E402

SAMPLE = 4096


def _setup(name):
    import torch
    w = W.WORKLOADS[name]
    ctx = g.Ctx.on_torch_stream(0)
    tin = W.torch_inputs(w, w.batch, torch.device("cuda", 0))
    ins = [g.DeviceBatch.wrap_torch(ctx, w.n, t, broadcast=bc) for t, (_, bc) in zip(tin, w.inputs)]
    plan = g.Plan(ctx, W.specialize(w))
    return torch, w, ctx, tin, ins, plan


def _out_tensors(torch, w, plan, n):
    return {k: torch.empty((comb(w.n, k), n), dtype=torch.float64, device="cuda:0") for k in plan.root_grades()}


def _sample_check(torch, w, tin, out_t, n):
    idx = torch.arange(0, n, max(1, n // SAMPLE), device="cuda:0")[:SAMPLE]
    host = []
    for t, (_, bc) in zip(tin, w.inputs):
        host.append({k: (v if bc else v[:, idx]).cpu().numpy() for k, v in t.items()})
    bcs = [bc for _, bc in w.inputs]
    m = len(idx)
    want = oracle_eval(w.build, w.metric, host, bcs, m)
    scale = oracle_abs_scale(w.build, w.metric, host, bcs, m)
    got = {k: v[:, idx].cpu().numpy() for k, v in out_t.items()}
    assert_close(got, want, scale, what=f"{w.name} full-size strided sample")


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_full_batch_sample_matches_oracle_and_is_homogeneous(name):
    torch, w, ctx, tin, ins, plan = _setup(name)
    n = w.batch
    out_t = _out_tensors(torch, w, plan, n)
    out = g.DeviceBatch.wrap_torch(ctx, w.n, out_t)
    plan.eval(ins, out=out)
    torch.cuda.synchronize()
    _sample_check(torch, w, tin, out_t, n)
    # homogeneity in the LAST input slot: x -> 2x.  Degree of the result in that slot:
    degree = {"cfg1": None, "cfg2": 1, "cfg3": 1, "cfg4": 2, "cfg5": 1}[name]
    if degree is None:
        return
    ref = {k: v.clone() for k, v in out_t.items()}
    for v in tin[-1].values():
        v.mul_(2.0)
    plan.eval(ins, out=out)
    torch.cuda.synchronize()
    for k in ref:
        assert torch.equal(out_t[k], ref[k] * float(2 ** degree)), f"{name}: result is not exactly homogeneous of degree {degree}"
    del ref, out_t, tin
    torch.cuda.empty_cache()


def test_cfg2_unit_rotor_sandwich_preserves_the_conformal_norm():
    torch, w, ctx, tin, ins, plan = _setup("cfg2")
    n = w.batch
    out_t = _out_tensors(torch, w, plan, n)
    plan.eval(ins, out=g.DeviceBatch.wrap_torch(ctx, w.n, out_t))
    torch.cuda.synchronize()
    met = torch.tensor(w.metric, dtype=torch.float64, device="cuda:0").reshape(-1, 1)
    x, y = tin[1][1], out_t[1]
    # R is a product of 4 unit vectors with squares +-1: (R ~R)^2 == 1, so y.y == x.x
    qx, qy = (met * x * x).sum(0), (met * y * y).sum(0)
    mag = (x * x).sum(0) + (y * y).sum(0)
    assert bool(((qx - qy).abs() <= 1e-11 * mag).all())


def test_cfg5_vector_sandwich_preserves_the_bivector_norm_and_batch_sum():
    torch, w, ctx, tin, ins, plan = _setup("cfg5")
    n = w.batch
    out_t = _out_tensors(torch, w, plan, n)
    sums = torch.zeros(66, dtype=torch.float64, device="cuda:0")
    plan.eval_sum(ins, sums.data_ptr(), out=g.DeviceBatch.wrap_torch(ctx, w.n, out_t))
    torch.cuda.synchronize()
    # metric of the bivector basis e_i e_j: (e_i e_j)^2 = -m_i m_j  => X.X = -sum m_i m_j X_ij^2
    m = w.metric
    coef = torch.tensor([-(m[i] * m[j]) for j in range(12) for i in range(j)], dtype=torch.float64, device="cuda:0")
    # component order inside grade 2: ascending bitmask (e1e2, e1e3, e2e3, e1e4, ...): pairs (i<j) sorted by (j, i)
    x, y = tin[1][2], out_t[2]
    qx, qy = (coef[:, None] * x * x).sum(0), (coef[:, None] * y * y).sum(0)
    mag = (x * x).sum(0) + (y * y).sum(0)
    # conditioning: V.V >= 0.1 by construction; the inverse amplifies rounding by <= 12/0.1
    assert bool(((qx - qy).abs() <= 1e-9 * mag).all())
    # fused batch-sum (per-thread column sums in shared memory: the reflection lowering parks no rows, so the
    # accumulators stay out of tensor memory) against a plain torch reduction of the stored result
    ref = out_t[2].sum(dim=1)
    scale = out_t[2].abs().sum(dim=1)
    assert bool(((sums - ref).abs() <= 1e-12 * scale).all())
    _sample_check(torch, w, tin, out_t, n)


def test_more_than_2_pow_31_elements_in_one_batch():
    """Maximum sizes: a batch longer than 2^31 elements (every row is 17 GB, the second row of a grade starts beyond
    2^34 bytes) through the specialised engine (strict and FMA), the table engine, and the batch-sum: element indices,
    row offsets and grid sizes must all be 64-bit clean.  G(2,0), v (vector) * s (scalar): the reference computes
    0.0 + (v_i * s) * 1.0 per component, which torch reproduces bit for bit on the device; the last elements of the
    batch -- where a 32-bit index would have wrapped -- are also compared with the oracle."""
    import torch
    from gaast_b200.expr import Input, mv as pmv
    n_elem = (1 << 31) + 4096 + 3
    free, _ = torch.cuda.mem_get_info(0)
    need = 5 * n_elem * 8 + (8 << 30)
    if free < need:
        torch.cuda.empty_cache()
        free, _ = torch.cuda.mem_get_info(0)
    assert free >= need, f"needs {need >> 30} GiB of free device memory, {free >> 30} GiB available"
    ctx = g.Ctx.on_torch_stream(0)
    gen = torch.Generator(device="cuda:0").manual_seed(31)
    v = torch.rand((2, n_elem), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1
    s = torch.rand((1, n_elem), dtype=torch.float64, device="cuda:0", generator=gen) * 2 - 1
    out_t = torch.empty((2, n_elem), dtype=torch.float64, device="cuda:0")
    metric = [1.0, 1.0]
    build = lambda a, b: a * b  # noqa: E731
    plan = g.Plan(ctx, build(pmv(Input(0, (1,))), pmv(Input(1, (0,)))).specialize(metric))
    ins = [g.DeviceBatch.wrap_torch(ctx, 2, {1: v}), g.DeviceBatch.wrap_torch(ctx, 2, {0: s})]
    out = g.DeviceBatch.wrap_torch(ctx, 2, {1: out_t})
    tail = slice(n_elem - 1000, n_elem)
    host = [{1: v[:, tail].cpu().numpy()}, {0: s[:, tail].cpu().numpy()}]
    want_tail = oracle_eval(build, metric, host, [False, False], 1000)[1]

    def check(what):
        torch.cuda.synchronize()
        step = 1 << 28
        for lo in range(0, n_elem, step):
            hi = min(n_elem, lo + step)
            assert torch.equal(out_t[:, lo:hi], v[:, lo:hi] * s[:, lo:hi] + 0.0), f"{what}: elements {lo}..{hi}"
        assert np.array_equal(out_t[:, tail].cpu().numpy(), want_tail), f"{what}: the last 1000 elements against the oracle"
        out_t.zero_()

    for engine, arith, what in ((L.ENGINE_SPECIALIZED, L.ARITH_STRICT, "specialised strict"),
                                (L.ENGINE_SPECIALIZED, L.ARITH_FMA, "specialised fma"),
                                (L.ENGINE_TABLE, L.ARITH_STRICT, "table strict")):
        plan.eval(ins, out=out, engine=engine, arith=arith)
        check(what)
    sums = torch.zeros(2, dtype=torch.float64, device="cuda:0")
    plan.eval_sum(ins, sums.data_ptr(), out=out)
    torch.cuda.synchronize()
    ref = torch.zeros(2, dtype=torch.float64, device="cuda:0")
    mag = torch.zeros(2, dtype=torch.float64, device="cuda:0")
    for lo in range(0, n_elem, 1 << 28):
        hi = min(n_elem, lo + (1 << 28))
        ref += out_t[:, lo:hi].sum(dim=1)
        mag += out_t[:, lo:hi].abs().sum(dim=1)
    assert torch.all((sums - ref).abs() <= 1e-12 * mag), (sums, ref, mag)
    check("specialised fma + batch-sum")
