"""Where every eval path writes: results against the oracle, and nothing stored outside `[0, len)` of a caller's rows.

Each case runs on poisoned, guarded layouts (tests/guarded_layout.py): caller-owned batches live in flat buffers with
guard scalars on both sides, a gap after every row and a chosen pointer alignment, all of it filled with a quiet-NaN
sentinel first; library-owned outputs are poisoned in `[0, len)`.  After the call the output guards and gaps must
still hold the sentinel, no result may still hold it (a store that never happened), and every input buffer must be
bit-identical to its state before the call.

Each case also asserts the path it ran from `Plan.last_kernel()`: the engine, and for the specialised engine the
launch that gaast_eval chose (csrc/device/runtime.cu, launch_length), restated by `predicted_launch`.  Per plan and
arithmetic two reference kernel keys are recorded: an owned batch of even length takes the aligned kernel, an odd
wrapped batch the unaligned one (one element per thread).  A case's `key=` must be the key of its predicted class; a
batch widened over an owned output's padding counts as aligned.

Values: strict arithmetic bit for bit against the oracle (f32: the reference's operation sequence in binary32,
run_plan_numpy), FMA arithmetic within REL_TOL (REL_TOL_F32) of max(|oracle|, sum of |terms|)."""
import re
from functools import lru_cache
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200.expr import Input, mv as pmv  # noqa: E402
from tests.guarded_layout import (GuardedBatch, check, check_owned, poison_owned, predicted_launch,  # noqa: E402
                                  streams_of)
from tests.helpers import (REL_TOL, REL_TOL_F32, AbsPlanAst, assert_bit_exact, assert_close,  # noqa: E402
                           oracle_abs_scale, oracle_eval, run_plan_numpy)
from tests.test_gpu_batch_sum import CASES, Case  # noqa: E402
from tests.test_gpu_projection import seeded_projection  # noqa: E402

OWNED = "owned"
STRICT, FMA = L.ARITH_STRICT, L.ARITH_FMA
SPEC, TABLE, DENSE = L.ENGINE_SPECIALIZED, L.ENGINE_TABLE, L.ENGINE_DENSE_WARP
PIPELINED = 65536 | 8        # cfg5 without the reflection lowering (parked rows) + persistent TMA pipeline (bit 3)
DENSE_TMEM = 131072 | 8192   # cfg3 without the matrix representation, operand in tensor memory (bits 17 + 13)
TMEM_PARTIAL = 262144        # cfg5: column sums in tensor memory, 62 of 66 columns stashed
NO_MATRIX = 1048576          # the dense engine's term-by-term kernel (bit 20)


class Lay:
    """A guarded caller-owned layout: gap scalars after each row, base offset in scalars (alignment mod 16 bytes)."""

    def __init__(self, gap=0, offset=0):
        self.gap, self.offset = gap, offset


@pytest.fixture(scope="module")
def ctx():
    c = g.Ctx(0)
    yield c
    c.close()


def np_dtype(dtype):
    return np.float32 if dtype == L.F32 else np.float64


def host_of(case: Case, length: int, dtype):
    host = case.host(length)
    return [{k: v.astype(np_dtype(dtype)) for k, v in d.items()} for d in host]


@lru_cache(maxsize=None)
def _reference(name, length, dtype, arith, comps):
    case = CASES[name] if name in CASES else EXTRA[name]
    host = host_of(case, length, dtype)
    as64 = [{k: v.astype(np.float64) for k, v in d.items()} for d in host]
    sel = (lambda r: {k: (v[list(dict(comps)[k])] if k in dict(comps) else v) for k, v in r.items()}) if comps else (lambda r: r)
    if arith == STRICT and dtype == L.F32:
        with np.errstate(all="ignore"):
            return sel(run_plan_numpy(case.specialize().plan_dict(), host, length, dtype=np.float32)), None
    want = sel(oracle_eval(case.build, case.metric, as64, case.bcs, length))
    if arith == STRICT:
        return want, None
    return want, sel(oracle_abs_scale(case.build, case.metric, as64, case.bcs, length))


def assert_values(case, length, dtype, arith, got, comps=None, what=""):
    ck = tuple(sorted((k, tuple(v)) for k, v in comps.items())) if comps else None
    want, scale = _reference(case.name, length, dtype, arith, ck)
    if arith == STRICT:
        assert_bit_exact(got, want, what)
    else:
        assert_close({k: v.astype(np.float64) for k, v in got.items()}, want, scale,
                     rel=REL_TOL_F32 if dtype == L.F32 else REL_TOL, what=what)


def make_plan(ctx, case, tuning=None, components=None):
    plan = g.Plan(ctx, case.specialize(), components=components)
    if tuning:
        plan.set_tuning(0, tuning)
    return plan


def run(ctx, case, plan, length, ins, out, engine=SPEC, arith=FMA, dtype=L.F64, with_sum=False, components=None,
        what=""):
    """One guarded call: ins[slot] = OWNED | Lay, out = OWNED | Lay | None (sums only).  Checks the write extent and
    the values; returns (last_kernel, predicted launch class)."""
    import torch
    host = host_of(case, length, dtype)
    n = case.n
    dev, guarded_in = [], []
    for s, ((grades, bc), lay) in enumerate(zip(case.slots, ins)):
        if lay == OWNED:
            dev.append(g.DeviceBatch.from_host(ctx, n, host[s], broadcast=bc, dtype=dtype))
            continue
        gb = GuardedBatch.dense(n, grades, 1 if bc else length, gap=lay.gap, offset=lay.offset, dtype=np_dtype(dtype),
                                role="in", device="cuda:0")
        gb.fill(host[s])
        guarded_in.append(gb)
        dev.append(gb.wrap(ctx, n, broadcast=bc))
    gout = None
    if out == OWNED:
        ob = poison_owned(plan.alloc_output(length, dtype))
    elif out is None:
        ob = None
    else:
        rows = {k: (len(components[k]) if components and k in components else comb(n, k)) for k in plan.root_grades()}
        gout = GuardedBatch(rows, length, gap=out.gap, offset=out.offset, dtype=np_dtype(dtype), role="out", device="cuda:0")
        ob = gout.wrap_sparse(ctx, n, {k: (components or {}).get(k) for k in rows}) if components else gout.wrap(ctx, n)
    torch.cuda.synchronize()  # (torch's stream is not the library's)
    before = [(b, b.bits()) for b in guarded_in]
    per_element = [d for d, (_, bc) in zip(dev, case.slots) if not bc] + ([ob] if ob is not None else [])
    predicted = predicted_launch(np.dtype(np_dtype(dtype)).itemsize, length, streams_of(per_element), out == OWNED,
                                 with_sum)[0]
    if with_sum:
        sums = torch.full((sum(ob.stored_rows(k) for k in ob.grade_set()) if ob is not None else 1,), float("nan"),
                          dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        plan.eval_sum(dev, sums.data_ptr(), out=ob, engine=engine, arith=arith)
    else:
        plan.eval(dev, out=ob, engine=engine, arith=arith)
    ctx.sync()
    kern = plan.last_kernel()
    what = f"{what} [{kern}]"
    check([gout] if gout else [], before, what)
    if ob is not None and length:
        got = gout.values() if gout else ob.to_host()
        if out == OWNED:
            check_owned(got, np_dtype(dtype), what)
        assert_values(case, length, dtype, arith, got, components, what)
    return kern, predicted


def key_of(kern):
    m = re.search(r"key=(\S+)", kern)
    assert m, kern
    return m.group(1)


_KEYS = {}


def reference_keys(ctx, case, arith, dtype, tuning=None, with_sum=False, components=None):
    """{"aligned": key, "unaligned": key} of the specialised kernels of a plan: an owned batch of even length, and an
    odd batch in caller-owned memory without room to widen.  The two are one kernel when the aligned one already runs
    one element per thread without TMA (then the unaligned form prints the same text)."""
    k = (case.name, arith, dtype, tuning, with_sum, repr(components))
    if k not in _KEYS:
        plan = make_plan(ctx, case, tuning, components)
        slots = len(case.slots)
        kern, cls = run(ctx, case, plan, 256, [OWNED] * slots, OWNED, arith=arith, dtype=dtype, with_sum=with_sum,
                        components=components, what="aligned reference")
        assert cls == "aligned" and "engine=specialized" in kern, kern
        aligned, aligned_kern = key_of(kern), kern
        kern, cls = run(ctx, case, plan, 255, [Lay()] * slots, Lay(), arith=arith, dtype=dtype, with_sum=with_sum,
                        components=components, what="unaligned reference")
        assert cls == "unaligned" and "engine=specialized" in kern and "elems/thread=1 " in kern, kern
        src = plan.kernel_source(case.bmask(), arith=arith, with_sum=with_sum, dtype=dtype)
        one_by_one = "elems/thread=1 " in aligned_kern and "tma-" not in src.split("\n")[1]
        assert (key_of(kern) == aligned) == one_by_one, (aligned_kern, kern)
        _KEYS[k] = {"aligned": aligned, "padded": aligned, "unaligned": key_of(kern)}
    return _KEYS[k]


def assert_specialized(ctx, case, kern, cls, expect, arith, dtype, tuning=None, with_sum=False, components=None):
    assert cls == expect, f"layout predicted {cls}, the case expects {expect}"
    assert "engine=specialized" in kern, kern
    assert key_of(kern) == reference_keys(ctx, case, arith, dtype, tuning, with_sum, components)[cls], (cls, kern)
    if cls == "unaligned":
        assert "elems/thread=1 " in kern, kern


def batch_slot(case):
    return next(s for s, (_, bc) in enumerate(case.slots) if not bc)


# ---- 1. the alignment classes of launch_length ----------------------------------------------------------------------
def _layouts(case, dtype):
    """(id, length, ins, out, expected class) per layout; f32 offsets of 4 and 12 bytes, f64 of 8."""
    q = 4 if dtype == L.F32 else 2
    slots = len(case.slots)
    s0 = batch_slot(case)
    even, odd = 1000, 1001
    one_off = lambda lay: [lay if s == s0 else OWNED for s in range(slots)]  # noqa: E731
    out = [
        ("aligned-even-wrapped", even, [Lay(gap=q)] * slots, Lay(gap=q), "aligned"),
        ("padded-owned-inputs", odd, [OWNED] * slots, OWNED, "padded"),
        ("padded-wrapped-inputs-gap", odd, [Lay(gap=q - 1)] * slots, OWNED, "padded"),
        ("unaligned-odd-wrapped-output", odd, [OWNED] * slots, Lay(), "unaligned"),
        ("unaligned-odd-wrapped-inputs", odd, [Lay()] * slots, OWNED, "unaligned"),
        ("unaligned-input-off16", even, one_off(Lay(gap=q, offset=1)), OWNED, "unaligned"),
        ("unaligned-output-only-off16", even, [OWNED] * slots, Lay(gap=q, offset=q - 1), "unaligned"),
        ("unaligned-odd-stride", even, [Lay(gap=1)] * slots, OWNED, "unaligned"),
    ]
    if any(bc for _, bc in case.slots):  # a misaligned broadcast operand is one element: no reason to leave the fast kernel
        out.append(("aligned-broadcast-off16", even, [Lay(offset=1) if bc else OWNED for _, bc in case.slots], OWNED,
                    "aligned"))
    return out


ALIGN = [(name, dtype, arith, lid) for name in ("cfg1", "cfg2", "cfg3", "cfg5") for dtype in (L.F64, L.F32)
         for arith in (STRICT, FMA) for lid, *_ in _layouts(CASES[name], dtype)]


@pytest.mark.parametrize("name,dtype,arith,layout", ALIGN, ids=[
    f"{n}-specialized-{'f32' if d else 'f64'}-{'strict' if a else 'fma'}-{lid}" for n, d, a, lid in ALIGN])
def test_alignment_classes(ctx, name, dtype, arith, layout):
    case = CASES[name]
    _, length, ins, out, expect = next(x for x in _layouts(case, dtype) if x[0] == layout)
    plan = make_plan(ctx, case)
    kern, cls = run(ctx, case, plan, length, ins, out, arith=arith, dtype=dtype, what=f"{name} {layout}")
    assert_specialized(ctx, case, kern, cls, expect, arith, dtype)


F32_TAILS = [(length, off) for length in (1001, 1002, 1003) for off in (1, 2, 3)]


@pytest.mark.parametrize("length,offset", F32_TAILS, ids=[f"cfg1-specialized-f32-strict-unaligned-len{n % 4}mod4-off{4 * o}B"
                                                         for n, o in F32_TAILS])
def test_f32_lengths_and_offsets(ctx, length, offset):
    """f32: 16 bytes are 4 elements.  A wrapped output 4, 8 or 12 bytes off a 16-byte boundary takes the unaligned
    kernel whatever the length; an owned output widens every length that is not a multiple of 4."""
    case = CASES["cfg1"]
    plan = make_plan(ctx, case)
    kern, cls = run(ctx, case, plan, length, [OWNED] * 3, Lay(offset=offset), arith=STRICT, dtype=L.F32,
                    what=f"f32 n={length} off={offset}")
    assert_specialized(ctx, case, kern, cls, "unaligned", STRICT, L.F32)
    if offset == 1:
        kern, cls = run(ctx, case, plan, length, [OWNED] * 3, OWNED, arith=STRICT, dtype=L.F32, what=f"f32 n={length} owned")
        assert_specialized(ctx, case, kern, cls, "padded", STRICT, L.F32)


# ---- 2. tails of the kernel shapes whose idle lanes shadow the last element (guard_stores) ----------------------------
EXTRA = {}
TAIL_SHAPES = {  # id -> (case, tuning, with_sum, the kernel notes of the aligned variant)
    "cfg5-v65544-persistent-pipelined": ("cfg5", PIPELINED, False, ("parked=32", "tma-pipelined")),
    "G6_AB_g2-tmem-sum-full-stash": ("G6_AB_g2", None, True, ("sum-in-tmem(64cols,stash=15)",)),
    "cfg3-v139264-operand-in-tmem": ("cfg3", DENSE_TMEM, False, ("dense-rolled", "tma-staged")),
}
TAIL_LENGTHS = [1, 3, 127, 130, 257, 4099]  # (q - 1 = 1 for f64); 130: a last TMA tile of 2 elements


def _assert_notes(ctx, case, tuning, with_sum, notes):
    plan = make_plan(ctx, case, tuning)
    src = plan.kernel_source(case.bmask(), with_sum=with_sum).split("\n")[1]
    for t in notes:
        assert t in src, (t, src)


TAILS = [(shape, length, out) for shape in TAIL_SHAPES for length in TAIL_LENGTHS for out in ("owned", "wrapped")]


@pytest.mark.parametrize("shape,length,out", TAILS, ids=[f"{s}-len{n}-{o}-out" for s, n, o in TAILS])
def test_tails_of_guarded_store_shapes(ctx, shape, length, out):
    name, tuning, with_sum, notes = TAIL_SHAPES[shape]
    case = CASES[name]
    _assert_notes(ctx, case, tuning, with_sum, notes)
    plan = make_plan(ctx, case, tuning)
    slots = len(case.slots)
    o = OWNED if out == "owned" else Lay(gap=0 if length % 2 else 2)
    kern, cls = run(ctx, case, plan, length, [OWNED] * slots, o, arith=FMA, with_sum=with_sum, what=f"{shape} n={length}")
    expect = ("aligned" if length % 2 == 0 else "unaligned" if (with_sum or out == "wrapped") else "padded")
    assert_specialized(ctx, case, kern, cls, expect, FMA, L.F64, tuning, with_sum)


LARGE = {"cfg5-v65544-persistent-pipelined": 1_000_000, "G6_AB_g2-tmem-sum-full-stash": 2_000_002,
         "cfg3-v139264-operand-in-tmem": 100_002}


@pytest.mark.parametrize("shape", sorted(LARGE), ids=[f"{s}-aligned-len{LARGE[s]}" for s in sorted(LARGE)])
def test_large_guarded_store_shapes(ctx, shape):
    """Lengths at which every persistent block loops over several tiles.  Every element is compared on the device
    against the strict table engine with the sum-of-|terms| scale (tests/helpers.AbsPlanAst); the last 1 000 elements
    and a strided sample of 1 000 against the oracle."""
    import torch
    name, tuning, with_sum, notes = TAIL_SHAPES[shape]
    case, length = CASES[name], LARGE[shape]
    plan = make_plan(ctx, case, tuning)
    tin = case.torch_inputs(length, torch)
    ins = [g.DeviceBatch.wrap_torch(ctx, case.n, t, broadcast=bc) for t, bc in zip(tin, case.bcs)]
    gout = GuardedBatch({k: comb(case.n, k) for k in plan.root_grades()}, length, role="out", device="cuda:0")
    ob = gout.wrap(ctx, case.n)
    torch.cuda.synchronize()
    cols = sum(comb(case.n, k) for k in plan.root_grades())
    if with_sum:
        sums = torch.full((cols,), float("nan"), dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        plan.eval_sum(ins, sums.data_ptr(), out=ob, engine=SPEC, arith=FMA)
    else:
        plan.eval(ins, out=ob, engine=SPEC, arith=FMA)
    ctx.sync()
    kern = plan.last_kernel()
    cls = predicted_launch(8, length, streams_of(ins + [ob]), False, with_sum)[0]
    assert_specialized(ctx, case, kern, cls, "aligned", FMA, L.F64, tuning, with_sum)
    grid, block = (int(x) for x in re.search(r"grid=(\d+) block=(\d+)", kern).groups())
    if "pipelined" in shape or with_sum:
        assert length > 2 * grid * block, f"each persistent block should loop over several tiles: {kern}"
    check([gout], what=f"{shape} n={length} [{kern}]")
    # every element: against the strict table engine, compared on the device
    strict = {k: torch.empty((comb(case.n, k), length), dtype=torch.float64, device="cuda:0") for k in plan.root_grades()}
    scale = {k: torch.empty_like(v) for k, v in strict.items()}
    torch.cuda.synchronize()
    plain = make_plan(ctx, case)
    plain.eval(ins, out=g.DeviceBatch.wrap_torch(ctx, case.n, strict), engine=TABLE, arith=STRICT)
    ctx.sync()
    idx = np.unique(np.r_[np.arange(length - 1000, length), np.linspace(0, length - 1, 1000).astype(np.int64)])
    host_sample = [{k: v[:, idx].cpu().numpy() for k, v in t.items()} for t in tin]
    for t in tin:
        for v in t.values():
            v.abs_()
    torch.cuda.synchronize()
    g.Plan(ctx, AbsPlanAst(case.specialize())).eval(ins, out=g.DeviceBatch.wrap_torch(ctx, case.n, scale), engine=TABLE,
                                                    arith=STRICT)
    ctx.sync()
    got = {k: b.view for k, b in gout.grades.items()}
    for k in plan.root_grades():
        err = (got[k] - strict[k]).abs()
        bad = ~(err <= REL_TOL * torch.maximum(strict[k].abs(), scale[k]))
        assert not bool(bad.any()), f"{shape}: grade {k}: {int(bad.sum())} elements off the strict table engine"
    want = oracle_eval(case.build, case.metric, host_sample, case.bcs, len(idx))
    wscale = oracle_abs_scale(case.build, case.metric, host_sample, case.bcs, len(idx))
    assert_close({k: v[:, idx].cpu().numpy() for k, v in got.items()}, want, wscale, what=f"{shape} sample vs oracle")


# ---- 3. batch sums with a stored output --------------------------------------------------------------------------
SUMS = {"cfg1-smem-column-sums": ("cfg1", None, ""), "G6_AB_g2-tmem-full-stash": ("G6_AB_g2", None, "stash=15"),
        "cfg5-v262144-tmem-partial-stash": ("cfg5", TMEM_PARTIAL, "stash=62")}
SUM_CASES = [(s, n, o) for s in SUMS for n in (1000, 1001) for o in ("wrapped", "owned")]


@pytest.mark.parametrize("shape,length,out", SUM_CASES, ids=[f"{s}-len{n}-{o}-out" for s, n, o in SUM_CASES])
def test_batch_sum_stored_output(ctx, shape, length, out):
    name, tuning, note = SUMS[shape]
    case = CASES[name]
    plan = make_plan(ctx, case, tuning)
    src = plan.kernel_source(case.bmask(), with_sum=True).split("\n")[1]
    assert (note in src) if note else ("sum-in-tmem" not in src), src
    o = OWNED if out == "owned" else Lay(gap=3 if length % 2 else 2, offset=0 if length % 2 else 1)
    kern, cls = run(ctx, case, plan, length, [OWNED] * len(case.slots), o, arith=FMA, with_sum=True,
                    what=f"{shape} n={length}")
    expect = "aligned" if length % 2 == 0 and out == "owned" else "unaligned"
    assert_specialized(ctx, case, kern, cls, expect, FMA, L.F64, tuning, True)


# ---- 4. the table engine -------------------------------------------------------------------------------------------
G9 = Case("G9_AB", [1.0] * 9, [(tuple(range(10)), False)] * 2, lambda a, b: a * b)
EXTRA[G9.name] = G9
TABLE_CASES = [("cfg1", "shared", d, a) for d in (L.F64, L.F32) for a in (STRICT, FMA)] + \
              [("cfg2", "shared", L.F64, STRICT), ("G9_AB", "global", L.F64, STRICT), ("G9_AB", "global", L.F64, FMA),
               ("G9_AB", "shared", L.F32, FMA)]  # (in f32 G(9)'s workspace fits in shared memory)


@pytest.mark.parametrize("name,ws,dtype,arith", TABLE_CASES, ids=[
    f"{n}-table-ws={w}-{'f32' if d else 'f64'}-{'strict' if a else 'fma'}" for n, w, d, a in TABLE_CASES])
def test_table_engine(ctx, name, ws, dtype, arith):
    case = CASES.get(name) or EXTRA[name]
    plan = make_plan(ctx, case)
    length = 40 if ws == "global" else 1001
    lay = Lay(gap=1, offset=1)
    ins = [Lay(offset=1) if bc else lay for _, bc in case.slots]
    kern, _ = run(ctx, case, plan, length, ins, Lay(gap=2, offset=1), engine=TABLE, arith=arith, dtype=dtype,
                  what=f"{name} table")
    assert "engine=table" in kern and f"ws={ws}" in kern, kern


# ---- 5. the dense engine -------------------------------------------------------------------------------------------
F8, F7 = tuple(range(9)), tuple(range(8))
for c in [Case("G8_AB", [1.0] * 8, [(F8, False)] * 2, lambda a, b: a * b),
          Case("G8_RXR", [1.0] * 8, [(F8, True), (F8, False)], lambda r, x: r * x * r.rev()),
          Case("G7_AB", [1.0] * 7, [(F7, False)] * 2, lambda a, b: a * b),
          Case("G8_outer", [1.0] * 8, [(F8, False)] * 2, lambda a, b: a ^ b)]:
    EXTRA[c.name] = c
DENSE_CASES = [("G8_AB", 0, "kernel=matrix products=1"), ("G8_RXR", 0, "kernel=matrix products=2"),
               ("G8_AB", NO_MATRIX, "gaast_dense_warp"), ("G7_AB", NO_MATRIX, "gaast_dense_warp"),
               ("G8_outer", 0, "gaast_dense_warp")]
DENSE_LENGTHS = [77, 130]


@pytest.mark.parametrize("length", DENSE_LENGTHS)
@pytest.mark.parametrize("name,tuning,expect", DENSE_CASES, ids=[f"{n}-dense-v{t}-{e.split()[0]}" for n, t, e in DENSE_CASES])
def test_dense_engine(ctx, name, tuning, expect, length):
    """Lengths that are not a multiple of the tile, inputs and outputs in caller-owned rows 8- but not 16-byte
    aligned, with a gap."""
    case = EXTRA[name]
    plan = make_plan(ctx, case, tuning)
    ins = [Lay(offset=1) if bc else Lay(gap=1, offset=1) for _, bc in case.slots]
    kern, _ = run(ctx, case, plan, length, ins, Lay(gap=3, offset=1), engine=DENSE, arith=FMA, what=f"{name} dense")
    assert "engine=dense_warp" in kern and all(t in kern for t in expect.split()), kern
    if tuning == NO_MATRIX:
        assert "kernel=matrix" not in kern, kern
    tile = int(re.search(r"tile=(\d+)", kern).group(1))
    assert length % tile, f"the length should leave a partial tile: {kern}"


# ---- 6. projected plans: sparse outputs in caller-owned rows ---------------------------------------------------------
CFG5_9 = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}
CFG3_WHOLE = seeded_projection("cfg3", 6, range(7))  # about a third of each grade; grade 3 whole, grade 6 emptied
PROJ = [("cfg5", "pruned", 1000, Lay(gap=2, offset=0), "aligned"), ("cfg5", "pruned", 1001, Lay(gap=3, offset=1), "unaligned"),
        ("cfg3", "whole", 1000, Lay(gap=2, offset=0), "aligned"), ("cfg3", "whole", 1001, Lay(gap=1, offset=1), "unaligned")]


@pytest.mark.parametrize("name,kind,length,lay,expect", PROJ, ids=[f"{p[0]}-projection-{p[1]}-specialized-{p[4]}-len{p[2]}"
                                                                   for p in PROJ])
def test_projected_sparse_output(ctx, name, kind, length, lay, expect):
    """The kernel stores only the selected rows, into a wrapped sparse output with a gap after every row."""
    case = CASES[name]
    comps = CFG5_9 if name == "cfg5" else CFG3_WHOLE
    plan = make_plan(ctx, case, components=comps)
    assert f",{kind})" in plan.kernel_source(case.bmask()).split("\n")[1]
    kern, cls = run(ctx, case, plan, length, [OWNED] * len(case.slots), lay, arith=STRICT, components=comps,
                    what=f"{name} projected")
    assert_specialized(ctx, case, kern, cls, expect, STRICT, L.F64, components=comps)


# ---- 7. sparse inputs whose root components have no term ------------------------------------------------------------
@pytest.mark.parametrize("length,lay,expect", [(1000, Lay(gap=2), "aligned"), (1001, Lay(gap=0, offset=1), "unaligned")],
                         ids=["G3-e1-times-e1-specialized-aligned", "G3-e1-times-e1-specialized-unaligned"])
def test_structurally_zero_root_components(ctx, length, lay, expect):
    """A and B store only e1 in G(3): A*B has terms for the scalar only, yet every component of the root grades (0
    and 2) must be written, as the reference's +-0."""
    import torch
    n, metric = 3, [1.0] * 3
    build = lambda a, b: a * b  # noqa: E731
    rng = np.random.default_rng(9)
    vals = [rng.uniform(-1, 1, (1, length)) for _ in range(2)]
    host = [{1: np.concatenate([v, np.zeros((2, length))])} for v in vals]
    plan = g.Plan(ctx, build(pmv(Input(0, (1,))), pmv(Input(1, (1,)))).specialize(metric))
    dev = [g.DeviceBatch.from_host_sparse(ctx, n, {1: ([0], v)}) for v in vals]
    gout = GuardedBatch({k: comb(n, k) for k in plan.root_grades()}, length, gap=lay.gap, offset=lay.offset, role="out",
                        device="cuda:0")
    torch.cuda.synchronize()
    ob = gout.wrap(ctx, n)
    plan.eval(dev, out=ob, engine=L.ENGINE_AUTO, arith=STRICT)
    ctx.sync()
    kern = plan.last_kernel()
    assert plan.root_grades() == [0, 2] and "engine=specialized" in kern, kern
    assert predicted_launch(8, length, streams_of(dev + [ob]), False)[0] == expect
    assert ("elems/thread=1 " in kern) == (expect == "unaligned"), kern
    check([gout], what=f"sparse e1*e1 [{kern}]")
    assert_bit_exact(gout.values(), oracle_eval(build, metric, host, [False, False], length), "sparse e1*e1")


# ---- 8. every input broadcast, the empty batch, AUTO's first tiny call -------------------------------------------------
BCAST = Case("cfg1_all_broadcast", [1.0] * 3, [(tuple(range(4)), True)] * 3, lambda a, b, c: (a + b * c).g(2))
EXTRA[BCAST.name] = BCAST


@pytest.mark.parametrize("out,expect", [("owned", "padded"), ("wrapped", "unaligned")],
                         ids=["all-broadcast-specialized-padded-owned-out", "all-broadcast-specialized-unaligned-wrapped-out"])
def test_every_input_broadcast(ctx, out, expect):
    """One element (n = 1) from broadcast operands only: an owned output is widened to two, a wrapped one is not."""
    plan = make_plan(ctx, BCAST)
    ins = [Lay(gap=1, offset=1)] * 3
    kern, cls = run(ctx, BCAST, plan, 1, ins, OWNED if out == "owned" else Lay(gap=0, offset=1), arith=STRICT,
                    what="all broadcast")
    assert cls == expect and "engine=specialized" in kern, (cls, kern)
    assert ("elems/thread=1 " in kern) == (expect == "unaligned"), kern


def test_empty_batch_writes_nothing(ctx):
    case = CASES["cfg1"]
    plan = make_plan(ctx, case)
    for engine in (L.ENGINE_AUTO, SPEC, TABLE):
        run(ctx, case, plan, 0, [Lay(gap=2, offset=1)] * 3, Lay(gap=2, offset=1), engine=engine, what="empty batch")


def test_auto_first_tiny_call_then_specialized(ctx):
    """AUTO: a plan's first call on a handful of elements goes to the table engine (no kernel is worth compiling for
    it); a later large call on the same plan to the specialised engine.  A freshly poisoned output each time."""
    case = CASES["cfg1"]
    plan = make_plan(ctx, case)
    kern, _ = run(ctx, case, plan, 10, [OWNED] * 3, Lay(gap=1, offset=1), engine=L.ENGINE_AUTO, arith=STRICT, what="tiny")
    assert "engine=table" in kern, kern
    kern, cls = run(ctx, case, plan, 200_000, [OWNED] * 3, Lay(gap=2), engine=L.ENGINE_AUTO, arith=STRICT, what="large")
    assert_specialized(ctx, case, kern, cls, "aligned", STRICT, L.F64)
