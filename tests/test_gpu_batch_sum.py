"""Batch sums (gaast_eval_sum) on the device, on every path the library can take to produce them, against an
exactly rounded reference.

gaast has no batches, so the sum has no reference definition.  Its reference here is `math.fsum` per root column
(columns in the library's order: root grades ascending, blades ascending inside a grade) of the oracle's
per-element results.  Two bars per column:

1. against the oracle:  |dev - fsum(oracle)| <= 1e-12 * sum_e max(|oracle_e|, scale_e), scale = sum of |terms|
   (tests/helpers.oracle_abs_scale) -- the per-element FMA error plus the reduction error.  f32 batches are held to
   the f32 per-element bar of the suite instead (REL_TOL_F32 = 1e-5, tests/test_gpu_f32.py);
2. the reduction alone, whenever the per-element result was stored:  |dev - fsum(stored)| <= 1e-13 * sum_e |stored_e|.
   One dropped, doubled or misplaced element moves a sum by about 1/N of that scale, orders of magnitude more than the
   bar.  f32 results are widened to f64 first: the sums accumulate in f64.  A sums-only run (out=None) is held to the
   same bar against the values the stored run wrote.

The code generator has several ways to sum (per-thread column sums in shared memory with one or two elements per
thread; accumulators in tensor memory with or without a per-tile stash; a guarded persistent loop), the table engine
has its own, and the per-block partials are added in one or two levels.  Every case asserts which of them it ran
(kernel source notes, `Plan.last_kernel()`), so that a change of heuristics fails here instead of silently testing
something else."""
import math
import re
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from gaast_b200.expr import Input, mv as pmv  # noqa: E402
from tests.helpers import REL_TOL_F32, oracle_abs_scale, oracle_eval  # noqa: E402

REL_SUM = 1e-12     # bar 1 (f64)
REL_REDUCE = 1e-13  # bar 2
GUARD = 3           # doubles before and after the sum vector; 3 * 8 bytes also leaves the sum pointer 8- but not 16-byte aligned
SENTINEL = 1234.5


class Case:
    def __init__(self, name, metric, slots, build, workload=None):
        self.name, self.metric, self.slots, self.build, self.workload = name, metric, slots, build, workload

    @property
    def n(self):
        return len(self.metric)

    @property
    def bcs(self):
        return [bc for _, bc in self.slots]

    def bmask(self):
        return sum(1 << s for s, bc in enumerate(self.bcs) if bc)

    def specialize(self):
        return self.build(*[pmv(Input(s, gr)) for s, (gr, _) in enumerate(self.slots)]).specialize(self.metric)

    def host(self, length, seed=0):
        if self.workload:  # the benchmark's inputs (a unit rotor for cfg2, |V.V| >= 0.1 for cfg5)
            return W.host_inputs(W.WORKLOADS[self.workload], length, None if seed == 0 else seed)
        rng = np.random.default_rng(0xB5A0 + seed + sum(map(ord, self.name)))
        return [{k: rng.uniform(-1, 1, (comb(self.n, k), 1 if bc else length)) for k in gr} for gr, bc in self.slots]

    def torch_inputs(self, length, torch):
        if self.workload:
            return W.torch_inputs(W.WORKLOADS[self.workload], length, "cuda:0")
        gen = torch.Generator(device="cuda:0").manual_seed(0xB5A1)
        return [{k: torch.empty((comb(self.n, k), length), dtype=torch.float64, device="cuda:0").uniform_(-1, 1, generator=gen)
                 for k in gr} for gr, _ in self.slots]


def _workload(name):
    w = W.WORKLOADS[name]
    return Case(name, w.metric, w.inputs, w.build, workload=name)


FULL6, FULL8 = tuple(range(7)), tuple(range(9))
G84 = [1.0] * 8 + [-1.0] * 4
CASES = {c.name: c for c in [
    _workload("cfg1"), _workload("cfg2"), _workload("cfg2_full"), _workload("cfg3"), _workload("cfg4"), _workload("cfg5"),
    Case("G6_AB_g2", [1.0] * 6, [(FULL6, False)] * 2, lambda a, b: (a * b).g(2)),
    # U independent of V: no reflection lowering, the product is expanded and rows are parked in shared memory
    Case("G84_VXU_g2", G84, [((1,), False), ((2,), False), ((1,), False)], lambda v, x, u: (v * x * u).g(2)),
    Case("G8_AB", [1.0] * 8, [(FULL8, False)] * 2, lambda a, b: a * b),
]}

# The path the code generator takes for each plan with a batch-sum, f64, default tuning: (notes of the kernel source
# that must appear, elements per thread).  No "sum-in-tmem" note = per-thread column sums in shared memory.
PATHS = {
    "cfg1": ("", 2),
    "cfg2": ("linear-map(5 outputs)", 2),
    "cfg2_full": ("linear-map(16 outputs)", 2),
    "cfg3": ("sum-in-tmem(256cols,stash=64)", 1),
    "cfg4": ("", 1),
    "cfg5": ("reflection(1 sandwich)", 1),
    "G6_AB_g2": ("parked=31 sum-in-tmem(64cols,stash=15)", 1),
    "G84_VXU_g2": ("parked=44 sum-in-tmem(256cols,stash=62)", 1),  # 62 columns stashed, 4 added one by one
}
# cfg5 under the tuning variants of the CPU emulation's batch-sum cases (tests/test_kernels_on_cpu.py::SUM_CASES)
VARIANTS = {
    262144: ("reflection(1 sandwich)", "sum-in-tmem(256cols,stash=62)"),  # tensor memory without parked rows
    65536: ("parked=32", "sum-in-tmem(256cols,stash=62)"),                # no reflection: parked rows, stash
    65536 | 128: ("parked=32", "sum-in-tmem(256cols,stash=0)"),           # ... every column added one by one
    65536 | 32: ("parked=32", ""),                                        # ... column sums in shared memory
}


# ---- helpers ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = g.Ctx(0)
    yield c
    c.close()


def columns(d):
    """{grade: [C(n,k), N]} -> [cols, N] in the library's column order, f64."""
    return np.concatenate([np.asarray(d[k], dtype=np.float64) for k in sorted(d)], axis=0)


def fsum_cols(a):
    return np.array([math.fsum(row.tolist()) for row in a])


class SumBuffer:
    """The caller's sum vector: `cols` doubles prefilled with NaN (a sum that is accumulated into instead of
    overwritten stays NaN), GUARD sentinel doubles on each side, and a pointer that is 8- but not 16-byte aligned."""

    def __init__(self, cols):
        import torch
        self.torch, self.cols = torch, cols
        self.t = torch.empty(cols + 2 * GUARD, dtype=torch.float64, device="cuda:0")
        self.ptr = self.t.data_ptr() + GUARD * 8
        assert self.ptr % 16 == 8
        self.refill()

    def refill(self):
        self.t.fill_(SENTINEL)
        self.t[GUARD:GUARD + self.cols] = float("nan")
        self.torch.cuda.synchronize()  # (torch's stream is not the library's)

    def read(self, ctx):
        ctx.sync()
        h = self.t.cpu().numpy()
        assert (h[:GUARD] == SENTINEL).all() and (h[GUARD + self.cols:] == SENTINEL).all(), \
            f"the batch-sum wrote outside its {self.cols} doubles: {h[:GUARD]} / {h[GUARD + self.cols:]}"
        return h[GUARD:GUARD + self.cols].copy()


def eval_sum(ctx, plan, dev, cols, out=None, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_FMA, buf=None):
    buf = buf or SumBuffer(cols)
    plan.eval_sum(dev, buf.ptr, out=out, engine=engine, arith=arith)
    return buf.read(ctx)


def assert_oracle_bar(got, want, scale, rel=REL_SUM, what=""):
    ref = fsum_cols(want)
    bound = rel * np.maximum(np.abs(want), scale).sum(axis=1)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {len(got)} column sums off the oracle; worst column "
                           f"{int(np.argmax(err / np.maximum(bound, 1e-300)))}: err {err.max():.3e}, bound {bound[np.argmax(err)]:.3e}")


def assert_reduction_bar(got, stored, what=""):
    ref = fsum_cols(stored)
    bound = REL_REDUCE * np.abs(stored).sum(axis=1)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {len(got)} column sums off the exact sum of the stored "
                           f"results; worst err {err.max():.3e} (bound {bound[np.argmax(err)]:.3e})")


def kernel_path(plan, case, dtype=L.F64, store=True, present=None):
    """(notes, elements per thread) of the kernel the code generator makes for an aligned batch."""
    src = plan.kernel_source(case.bmask(), with_sum=True, store_out=store, dtype=dtype, present=present)
    notes = src.split("\n")[1]
    ept = int(re.search(r"#define GAAST_EPT (\d)", src).group(1))
    return notes, ept


def assert_path(notes, ept, expect_notes, expect_ept, what=""):
    for tok in expect_notes.split():
        assert tok in notes, f"{what}: expected '{tok}' in the kernel notes: {notes}"
    if "sum-in-tmem" not in expect_notes:
        assert "sum-in-tmem" not in notes, f"{what}: expected column sums in shared memory: {notes}"
    assert ept == expect_ept, f"{what}: {ept} elements per thread, expected {expect_ept}"


def launched(plan):
    """(engine, grid, block, elements per thread) of the last launch (printed: pytest -s lists the kernels run)."""
    k = plan.last_kernel()
    print("  launched:", k)
    m = re.search(r"engine=specialized .*grid=(\d+) block=(\d+) elems/thread=(\d+)", k)
    if m:
        return "specialized", int(m.group(1)), int(m.group(2)), int(m.group(3))
    m = re.search(r"engine=table grid=(\d+) block=(\d+)", k)
    assert m, k
    return "table", int(m.group(1)), int(m.group(2)), 1


def upload(ctx, case, host, dtype=L.F64):
    return [g.DeviceBatch.from_host(ctx, case.n, h, broadcast=bc, dtype=dtype) for h, bc in zip(host, case.bcs)]


def reference(case, host, length):
    as64 = [{k: np.asarray(v, dtype=np.float64) for k, v in d.items()} for d in host]
    return (columns(oracle_eval(case.build, case.metric, as64, case.bcs, length)),
            columns(oracle_abs_scale(case.build, case.metric, as64, case.bcs, length)))


def run_stored_and_sums_only(ctx, case, plan, length, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_FMA, dtype=L.F64,
                             host=None, dev=None, what=""):
    """eval_sum with the result stored and without (out=None), both held to both bars; returns the launches."""
    if host is None:
        host = case.host(length)
        if dtype == L.F32:
            host = [{k: v.astype(np.float32) for k, v in d.items()} for d in host]
    dev = dev or upload(ctx, case, host, dtype)
    want, scale = reference(case, host, length)
    cols = want.shape[0]
    rel = REL_TOL_F32 if dtype == L.F32 else REL_SUM
    out = plan.alloc_output(length, dtype)
    got = eval_sum(ctx, plan, dev, cols, out=out, engine=engine, arith=arith)
    stored_launch = launched(plan)
    stored = columns(out.to_host())
    assert stored.shape == want.shape
    assert_oracle_bar(got, want, scale, rel, f"{what} stored")
    assert_reduction_bar(got, stored, f"{what} stored")
    got2 = eval_sum(ctx, plan, dev, cols, out=None, engine=engine, arith=arith)
    nostore_launch = launched(plan)
    assert_oracle_bar(got2, want, scale, rel, f"{what} out=None")
    assert_reduction_bar(got2, stored, f"{what} out=None")
    return stored_launch, nostore_launch


# ---- the path matrix -------------------------------------------------------------------------------------------
MATRIX = [(name, L.F64, 0) for name in PATHS] + [("cfg3", L.F32, 0), ("cfg5", L.F32, 0)] + \
         [("cfg5", L.F64, v) for v in VARIANTS]


@pytest.mark.parametrize("name,dtype,variant", MATRIX,
                         ids=[f"{n}-{'f32' if d else 'f64'}" + (f"-v{v}" if v else "") for n, d, v in MATRIX])
def test_path_matrix(ctx, name, dtype, variant):
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    if variant:
        plan.set_tuning(0, variant)
        expect = " ".join(VARIANTS[variant])
        expect_ept = 1
    else:
        expect, expect_ept = PATHS[name]
    for store in (True, False):
        notes, ept = kernel_path(plan, case, dtype, store)
        assert_path(notes, ept, expect, expect_ept, f"{name} store={store}")
    length = 4096 + 130  # ragged against one tile (128 elements) and one two-element tile (256)
    for la in run_stored_and_sums_only(ctx, case, plan, length, dtype=dtype, what=f"{name} v{variant}"):
        assert la[0] == "specialized" and la[3] == ept, plan.last_kernel()


# ---- lengths at the edges ----------------------------------------------------------------------------------------
LENGTHS = [1, 127, 128, 129, 255, 257, 1001]


@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("name", sorted(PATHS))
def test_lengths_at_the_edges(ctx, name, length):
    """An odd length cannot use 128-bit accesses: the two-element kernels run their one-element variant (a batch-sum
    never runs over the padding of the rows).  The tensor-memory kernels' idle lanes shadow element n-1 and must add
    nothing."""
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    _, ept = PATHS[name]
    for la in run_stored_and_sums_only(ctx, case, plan, length, what=f"{name} n={length}"):
        assert la[0] == "specialized", plan.last_kernel()
        assert la[3] == (1 if length % 2 else ept), plan.last_kernel()


# ---- the table engine ------------------------------------------------------------------------------------------
TABLE = [(name, arith, dtype) for name in sorted(PATHS) for arith in (L.ARITH_FMA, L.ARITH_STRICT) for dtype in (L.F64, L.F32)]


@pytest.mark.parametrize("name,arith,dtype", TABLE,
                         ids=[f"{n}-{'strict' if a else 'fma'}-{'f32' if d else 'f64'}" for n, a, d in TABLE])
def test_table_engine(ctx, name, arith, dtype):
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    for la in run_stored_and_sums_only(ctx, case, plan, 1000 + 37, engine=L.ENGINE_TABLE, arith=arith, dtype=dtype,
                                       what=f"{name} table"):
        assert la[0] == "table", plan.last_kernel()


def test_plan_only_the_table_engine_can_sum(ctx):
    """G(8,0) full A*B (65 536 terms, 256 columns): too large to specialise; the dense engine has no batch-sum.
    AUTO sums it on the table engine (workspace in global memory); the dense engine refuses."""
    case = CASES["G8_AB"]
    plan = g.Plan(ctx, case.specialize())
    for la in run_stored_and_sums_only(ctx, case, plan, 300, engine=L.ENGINE_AUTO, what="G8 A*B auto"):
        assert la[0] == "table" and "ws=global" in plan.last_kernel(), plan.last_kernel()
    dev = upload(ctx, case, case.host(300))
    for out in (plan.alloc_output(300), None):
        with pytest.raises(g.GaastError) as ei:
            eval_sum(ctx, plan, dev, 256, out=out, engine=L.ENGINE_DENSE_WARP)
        assert ei.value.status == L.ERR_UNSUPPORTED


# ---- sparse inputs ---------------------------------------------------------------------------------------------
def _sparse(rng, n, k, length, keep):
    c = comb(n, k)
    idx = sorted(rng.choice(c, size=min(keep, c), replace=False).tolist())
    compact = rng.uniform(-1, 1, (len(idx), length))
    dense = np.zeros((c, length))
    dense[idx] = compact
    return idx, compact, dense


@pytest.mark.parametrize("name", ["cfg5", "G6_AB"])
def test_sparse_inputs(ctx, name):
    """Sparse per-grade storage with a batch-sum, against the oracle on the dense inputs: cfg5 with 9 of X's 66
    components (column sums in shared memory); G(6) A*B with some grades of both operands sparse (tensor memory)."""
    rng = np.random.default_rng(23)
    length = 2048 + 6
    if name == "cfg5":
        case = CASES["cfg5"]
        host = case.host(length)
        idx, compact, dense = _sparse(rng, 12, 2, length, 9)
        host[1] = {2: dense}
        stored = [host[0], {2: (idx, compact)}]
        expect = ("reflection(1 sandwich)", 1)
    else:
        case = Case("G6_AB", [1.0] * 6, [(FULL6, False)] * 2, lambda a, b: a * b)
        host, stored = [], []
        for s in range(2):
            h, st = {}, {}
            for k in FULL6:
                if (k + s) % 2:
                    idx, compact, dense = _sparse(rng, 6, k, length, max(1, comb(6, k) // 2))
                    h[k], st[k] = dense, (idx, compact)
                else:
                    h[k] = st[k] = rng.uniform(-1, 1, (comb(6, k), length))
            host.append(h)
            stored.append(st)
        expect = ("sum-in-tmem(256cols,stash=64)", 1)
    plan = g.Plan(ctx, case.specialize())
    present = {(s, k): v[0] for s, st in enumerate(stored) for k, v in st.items() if isinstance(v, tuple)}
    notes, ept = kernel_path(plan, case, present=present)
    assert_path(notes, ept, *expect, what=f"{name} sparse")
    dev = [g.DeviceBatch.from_host_sparse(ctx, case.n, st) for st in stored]
    for la in run_stored_and_sums_only(ctx, case, plan, length, engine=L.ENGINE_AUTO, host=host, dev=dev,
                                       what=f"{name} sparse"):
        assert la[0] == "specialized", plan.last_kernel()


# ---- contract of the sum vector ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg1", "cfg3", "cfg5", "G84_VXU_g2"])
def test_empty_batch_writes_zeros(ctx, name):
    """No elements: every engine, stored or not, overwrites the NaN-filled sum vector with zeros (and nothing beyond)."""
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    dev = [g.DeviceBatch.from_host(ctx, case.n, h, broadcast=True) if bc else g.DeviceBatch.alloc(ctx, case.n, gr, 0)
           for h, (gr, bc) in zip(case.host(1), case.slots)]
    cols = sum(comb(case.n, k) for k in plan.root_grades())
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE, L.ENGINE_AUTO):
        for out in (plan.alloc_output(0), None):
            got = eval_sum(ctx, plan, dev, cols, out=out, engine=engine)
            assert (got == 0.0).all(), f"{name}: engine {engine}: {got}"


@pytest.mark.parametrize("name", ["cfg1", "G6_AB_g2"])
def test_sum_vector_is_overwritten_not_accumulated(ctx, name):
    """A second call into the same, not refilled, vector gives the same bits: it is overwritten, not added to."""
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    length = 4096 + 2
    dev = upload(ctx, case, case.host(length))
    cols = sum(comb(case.n, k) for k in plan.root_grades())
    for engine in (L.ENGINE_SPECIALIZED, L.ENGINE_TABLE):
        buf = SumBuffer(cols)
        first = eval_sum(ctx, plan, dev, cols, engine=engine, buf=buf)
        again = eval_sum(ctx, plan, dev, cols, engine=engine, buf=buf)
        assert np.isfinite(first).all() and np.array_equal(again.view(np.uint64), first.view(np.uint64)), engine


# ---- large batches: capped persistent grid, two-level reduction, exact-zero construction ---------------------------
# (odd in slot: negating these slots of an element negates its result exactly -- every rounding is sign-symmetric)
ODD_SLOTS = {"cfg1": (0, 1), "cfg5": (1,), "G6_AB_g2": (0,)}
BLOCKS = 24_000  # tiles: blocks of the uncapped grid; the persistent grid is then larger than 2048 blocks whatever the
                 # number of resident blocks per SM (it is resident x max(4, tiles / (8 x resident)) blocks)


def _large_exact_zero(case, plan, torch, ctx):
    """Inputs whose second half negates the first in the odd slots: the exact sum of every column is 0.  Length:
    BLOCKS tiles and a ragged, even tail (a pair (i, i + N/2) per element)."""
    _, ept = PATHS[case.name]
    length = BLOCKS * 128 * ept + 74
    tin = case.torch_inputs(length, torch)
    h = length // 2
    for s, d in enumerate(tin):
        for t in d.values():
            t[:, h:] = -t[:, :h] if s in ODD_SLOTS[case.name] else t[:, :h]
    torch.cuda.synchronize()
    ins = [g.DeviceBatch.wrap_torch(ctx, case.n, t) for t in tin]
    out_t = {k: torch.empty((comb(case.n, k), length), dtype=torch.float64, device="cuda:0") for k in plan.root_grades()}
    return length, ept, tin, ins, out_t


def _assert_capped_two_level(plan, length, ept, launches, small_launches, what):
    engine, grid, block, got_ept = launched(plan)
    assert engine == "specialized" and got_ept == ept, plan.last_kernel()
    assert grid > 2048, f"{what}: grid {grid}: not the two-level reduction"
    tile = block * ept
    assert grid * tile * 2 <= length and length % tile, f"{what}: grid {grid} does not loop over several tiles, ragged"
    assert launches == small_launches + 1, f"{what}: {launches} launches, one level took {small_launches}"


def _check_exact_zero(torch, got, out_t, what):
    scale = torch.cat([t.abs().sum(dim=1) for _, t in sorted(out_t.items())]).cpu().numpy()
    assert (np.abs(got) <= REL_REDUCE * scale).all(), f"{what}: exact sum 0, got {np.abs(got).max():.3e} at scale {scale.min():.3e}"


@pytest.mark.parametrize("name", ["cfg1", "cfg5"])
def test_two_level_reduction_exact_zero(ctx, name):
    """A persistent grid of more than 2048 blocks, each looping over several tiles, the last one ragged; the
    partials are added in two levels.  With an exact column sum of zero a dropped or repeated tile anywhere shows."""
    import torch
    case = CASES[name]
    plan = g.Plan(ctx, case.specialize())
    cols = sum(comb(case.n, k) for k in plan.root_grades())
    small = upload(ctx, case, case.host(4096))
    c0 = ctx.launch_count
    eval_sum(ctx, plan, small, cols)
    small_launches = ctx.launch_count - c0
    length, ept, tin, ins, out_t = _large_exact_zero(case, plan, torch, ctx)
    out = g.DeviceBatch.wrap_torch(ctx, case.n, out_t)
    c0 = ctx.launch_count
    got = eval_sum(ctx, plan, ins, cols, out=out)
    _assert_capped_two_level(plan, length, ept, ctx.launch_count - c0, small_launches, name)
    _check_exact_zero(torch, got, out_t, f"{name} stored")
    if name == "cfg1":  # (3 columns: cheap enough to sum exactly on the host)
        stored = torch.cat([t for _, t in sorted(out_t.items())]).cpu().numpy()
        assert (fsum_cols(stored) == 0.0).all()
        assert_reduction_bar(got, stored, f"{name} two-level")
    again = eval_sum(ctx, plan, ins, cols, out=None)
    _check_exact_zero(torch, again, out_t, f"{name} out=None")
    again2 = eval_sum(ctx, plan, ins, cols, out=None)
    assert np.array_equal(again.view(np.uint64), again2.view(np.uint64)), "two-level sums differ between equal launches"
    # the table engine's blocks loop over the batch too (its grid stops at 8 blocks per SM)
    tab = eval_sum(ctx, plan, ins, cols, out=out, engine=L.ENGINE_TABLE)
    engine, grid, _, _ = launched(plan)
    assert engine == "table" and grid * 32 * 2 <= length, plan.last_kernel()
    _check_exact_zero(torch, tab, out_t, f"{name} table engine")
    del tin, ins, out, out_t
    torch.cuda.empty_cache()


def test_state_across_calls_tensor_memory_two_level(ctx):
    """One plan (tensor-memory accumulators with the per-tile stash), calls of changing size and kind: large (two
    levels) -> small -> large -> large without output -> large.  Each is checked; equal launches give equal bits.
    Stale partial rows of the large grid, or a stale stash, would show in the small call or the repeated ones."""
    import torch
    case = CASES["G6_AB_g2"]
    plan = g.Plan(ctx, case.specialize())
    cols = 15
    small_len = 1001 + 2
    small_host = case.host(small_len, seed=5)
    small_dev = upload(ctx, case, small_host)
    want, scale = reference(case, small_host, small_len)
    c0 = ctx.launch_count
    small_out = plan.alloc_output(small_len)
    first_small = eval_sum(ctx, plan, small_dev, cols, out=small_out)
    small_launches = ctx.launch_count - c0
    assert_oracle_bar(first_small, want, scale, what="small, first")

    length, ept, tin, ins, out_t = _large_exact_zero(case, plan, torch, ctx)
    out = g.DeviceBatch.wrap_torch(ctx, case.n, out_t)
    c0 = ctx.launch_count
    big = eval_sum(ctx, plan, ins, cols, out=out)
    _assert_capped_two_level(plan, length, ept, ctx.launch_count - c0, small_launches, "G6_AB_g2")
    assert "sum-in-tmem(64cols,stash=15)" in kernel_path(plan, case)[0]
    stored = out_t[2].cpu().numpy()
    assert (fsum_cols(stored) == 0.0).all()
    assert_reduction_bar(big, stored, "large")
    _check_exact_zero(torch, big, out_t, "large")

    small = eval_sum(ctx, plan, small_dev, cols, out=small_out)
    assert_oracle_bar(small, want, scale, what="small after large")
    assert_reduction_bar(small, columns(small_out.to_host()), "small after large")
    assert np.array_equal(small.view(np.uint64), first_small.view(np.uint64)), "small sum changed after a large call"
    big2 = eval_sum(ctx, plan, ins, cols, out=out)
    assert np.array_equal(big2.view(np.uint64), big.view(np.uint64)), "large sum changed after a small call"
    big_none = eval_sum(ctx, plan, ins, cols, out=None)
    assert_reduction_bar(big_none, stored, "large, out=None")
    big3 = eval_sum(ctx, plan, ins, cols, out=out)
    assert np.array_equal(big3.view(np.uint64), big.view(np.uint64)), "large sum changed after a sums-only call"
    del tin, ins, out, out_t
    torch.cuda.empty_cache()


# ---- determinism and CUDA graphs ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg5", "G6_AB_g2"])
def test_graph_replay_gives_the_same_bits(name):
    """eval_sum captured in a CUDA graph and replayed gives the bits of the direct call (equal launch shape); so do two
    direct calls (tensor-memory and shared-memory paths)."""
    import torch
    case = CASES[name]
    ctx = g.Ctx.on_torch_stream(0)
    try:
        plan = g.Plan(ctx, case.specialize())
        length = 300_000 + 6
        dev = upload(ctx, case, case.host(length))
        cols = sum(comb(case.n, k) for k in plan.root_grades())
        out = plan.alloc_output(length)
        direct = eval_sum(ctx, plan, dev, cols, out=out)
        direct2 = eval_sum(ctx, plan, dev, cols, out=out)
        assert np.array_equal(direct.view(np.uint64), direct2.view(np.uint64))
        buf = SumBuffer(cols)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ctx.torch_stream):
            plan.eval_sum(dev, buf.ptr, out=out, engine=L.ENGINE_SPECIALIZED)
        for _ in range(2):
            buf.refill()
            graph.replay()
            torch.cuda.synchronize()
            got = buf.read(ctx)
            assert np.array_equal(got.view(np.uint64), direct.view(np.uint64)), "graph replay differs from the direct call"
        del graph
    finally:
        torch.cuda.set_stream(torch.cuda.default_stream(0))
        ctx.sync()
