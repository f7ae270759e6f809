"""Per-segment sums of a batch's stored rows (gaast_batch_segment_sum) on the device.

Reference: `math.fsum` per (segment, stored row) of the downloaded rows.  Bar: |dev - fsum| <= 1e-13 * sum |x| over
the segment, the reduction bar of tests/test_gpu_batch_sum.py; f32 batches too (their sums accumulate in f64)."""
import math
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from tests.helpers import oracle_abs_scale, oracle_eval  # noqa: E402

torch = pytest.importorskip("torch")

REL_REDUCE = 1e-13
REL_SUM = 1e-12
CHUNK = 4096  # the library's chunk size (segments.cu)
CFG5_ROOT = (12, [2])  # G(8,4) grade 2: 66 rows


@pytest.fixture(scope="module")
def ctx():
    return g.Ctx(0)


def offs(offsets):
    """Offsets on the device, ready for the ctx's own stream."""
    t = torch.tensor(offsets, dtype=torch.int64, device="cuda:0")
    torch.cuda.synchronize()
    return t


def stored(b):
    """The stored rows [S, len] as float64, grades ascending."""
    return np.concatenate([b.download(k).astype(np.float64) for k in b.grade_set()], axis=0)


def reference(x, offsets):
    n = len(offsets) - 1
    want, scale = np.zeros((n, x.shape[0])), np.zeros((n, x.shape[0]))
    for j in range(n):
        a, e = int(offsets[j]), int(offsets[j + 1])
        for r in range(x.shape[0]):
            seg = x[r, a:e].tolist()
            want[j, r] = math.fsum(seg)
            scale[j, r] = math.fsum(abs(v) for v in seg)
    return want, scale


def check(b, offsets, x=None):
    x = stored(b) if x is None else x
    off = offs(offsets)
    got = b.segment_sum(off)
    b.ctx.sync()
    got = got.cpu().numpy()
    want, scale = reference(x, offsets)
    err = np.abs(got - want)
    assert (err <= REL_REDUCE * scale).all(), (np.argwhere(err > REL_REDUCE * scale)[:5], err.max())
    empty = np.diff(np.asarray(offsets)) == 0
    assert (got[empty] == 0).all() and not np.signbit(got[empty]).any()
    return got


def random_batch(ctx, n, grades, length, dtype=L.F64, seed=0):
    rng = np.random.default_rng(seed)
    return g.DeviceBatch.from_host(ctx, n, {k: rng.standard_normal((comb(n, k), length)) for k in grades}, dtype=dtype)


def layouts(length, rng):
    lens = rng.integers(0, 41, size=length)
    rand = np.concatenate([[0], np.cumsum(lens)])
    rand = list(rand[rand <= length])
    edges = sorted({0, length, *[c for k in range(CHUNK, length, CHUNK) for c in (k - 1, k, k + 1) if 0 < c < length]})
    return {
        "ones": list(range(length + 1)),
        "random_0_40": rand,
        "whole": [0, length],
        "chunk_edges": edges,
        "many_chunks": [0, 5, length - 3, length],
        "inner_range": [9, 9, 4000, 4100, length - 11],
        "empty_pile": [0, 10] + [70] * 70 + [71, length],
    }


# ---- layouts x batches ---------------------------------------------------------------------------------------------
BATCHES = {
    "G3_full": (3, [0, 1, 2, 3], L.F64),
    "cfg5_root": (*CFG5_ROOT, L.F64),
    "G10_g2": (10, [2], L.F64),
    "G3_full_f32": (3, [0, 1, 2, 3], L.F32),
    "cfg5_root_f32": (*CFG5_ROOT, L.F32),
}


@pytest.mark.parametrize("name", list(BATCHES))
def test_layouts(ctx, name):
    n, grades, dtype = BATCHES[name]
    length = 9 * CHUNK + 77
    b = random_batch(ctx, n, grades, length, dtype, seed=len(name))
    x = stored(b)
    rng = np.random.default_rng(1)
    for offsets in layouts(length, rng).values():
        check(b, offsets, x)


def test_sparse_input_batch(ctx):
    rng = np.random.default_rng(2)
    length = 3 * CHUNK + 5
    b = g.DeviceBatch.from_host_sparse(ctx, 6, {1: ([0, 3, 5], rng.standard_normal((3, length))),
                                                2: rng.standard_normal((15, length))})
    assert sum(b.stored_rows(k) for k in b.grade_set()) == 18
    for offsets in layouts(length, rng).values():
        check(b, offsets)


def test_projected_plan_output(ctx):
    w = W.WORKLOADS["cfg5"]
    comps = {2: [0, 5, 11, 17, 30, 41, 52, 60, 65]}
    plan = g.Plan(ctx, W.specialize(w), components=comps)
    length = 2 * CHUNK + 300
    host = W.host_inputs(w, length)
    dev = [g.DeviceBatch.from_host(ctx, w.n, d, broadcast=bc) for d, (_, bc) in zip(host, w.inputs)]
    out = plan.eval(dev)
    got = check(out, [0, 1, 2, 50, CHUNK + 1, length])
    assert got.shape == (5, 9)


def test_wrapped_torch_batch_with_padding_stride(ctx):
    length, stride = 2 * CHUNK + 9, 2 * CHUNK + 100
    base = torch.randn((3, stride), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    b = g.DeviceBatch.wrap_torch(ctx, 3, {1: base[:, :length]})
    assert b.stride == stride and b.length == length
    check(b, [0, 7, CHUNK, CHUNK + 40, length])
    check(b, [0, length])


# ---- scale -----------------------------------------------------------------------------------------------------------
def test_2_25_columns_with_spanning_segments(ctx):
    length = (1 << 25) + 7
    rng = np.random.default_rng(4)
    b = random_batch(ctx, 3, [1], length, seed=4)
    cuts = sorted(set(rng.integers(1, length, 40).tolist()) | {CHUNK * 100, CHUNK * 100 + 1})
    check(b, [0, *cuts, length])
    check(b, [0, length])


def test_row_beyond_2_31_columns(ctx):
    """One f32 row of more than 2^31 columns holding col % 7: every sum is an exact integer, so any order gives it, and
    a column index cut to 32 bits reads the wrong values."""
    length = (1 << 31) + (1 << 20) + 3
    row = (torch.arange(length, dtype=torch.int64, device="cuda:0") % 7).to(torch.float32).reshape(1, length)
    torch.cuda.synchronize()
    b = g.DeviceBatch.wrap_torch(ctx, 0, {0: row})
    offsets = [0, 5, (1 << 31) - 9, (1 << 31) + 100, (1 << 31) + 100, length]

    def exact(a, e):  # sum of c % 7 over [a, e)
        f = lambda m: (m // 7) * 21 + sum(range(m % 7))  # noqa: E731
        return float(f(e) - f(a))

    got = b.segment_sum(offs(offsets))
    ctx.sync()
    got = got.cpu().numpy()[:, 0]
    assert got.tolist() == [exact(offsets[j], offsets[j + 1]) for j in range(len(offsets) - 1)]
    del b, row
    torch.cuda.empty_cache()


# ---- contract ----------------------------------------------------------------------------------------------------------
def test_overwrite_guards_and_empty(ctx):
    length = 2 * CHUNK + 3
    b = random_batch(ctx, 3, [1], length, seed=5)
    offsets = [0, 0, 10, CHUNK + 1, CHUNK + 1, length, length]
    n = len(offsets) - 1
    buf = torch.full((n * 3 + 6,), float("nan"), dtype=torch.float64, device="cuda:0")
    buf[:3] = 1234.5
    buf[-3:] = 1234.5
    off = offs(offsets)
    inner = buf[3:-3].view(n, 3)
    torch.cuda.synchronize()
    b.segment_sum(off, out=inner)
    ctx.sync()
    host = buf.cpu().numpy()
    assert (host[:3] == 1234.5).all() and (host[-3:] == 1234.5).all()
    got = host[3:-3].reshape(n, 3)
    assert not np.isnan(got).any()
    want, scale = reference(stored(b), offsets)
    assert (np.abs(got - want) <= REL_REDUCE * scale).all()
    assert not np.signbit(got[[0, 3, 5]]).any() and (got[[0, 3, 5]] == 0).all()


def test_no_segments_launches_nothing(ctx):
    b = random_batch(ctx, 3, [1], 100, seed=6)
    off = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    before = ctx.launch_count
    out = b.segment_sum(off)
    assert out.shape == (0, 3) and ctx.launch_count == before


def test_launch_count(ctx):
    b = random_batch(ctx, 3, [1], 5000, seed=7)
    off = offs([0, 100, 5000])
    b.segment_sum(off)
    for _ in range(3):
        before = ctx.launch_count
        b.segment_sum(off)
        assert ctx.launch_count - before == 2


def test_invalid_offsets_give_nan(ctx):
    length = 3 * CHUNK + 1
    b = random_batch(ctx, 3, [1], length, seed=8)
    good = [0, 10, CHUNK + 3, length]
    for bad in ([0, 100, 50, length], [-1, 10, length], [0, 10, length + 1], [0, 2 * CHUNK, CHUNK, 0]):
        got = b.segment_sum(offs(bad))
        ctx.sync()
        assert torch.isnan(got).all(), bad
        check(b, good)


def _call(b, ptr_off, n_seg, ptr_sums):
    return L.lib.gaast_batch_segment_sum(b._h if b is not None else None, L.vp(ptr_off), n_seg, L.vp(ptr_sums))


def test_error_statuses(ctx):
    b = random_batch(ctx, 3, [1], 100, seed=9)
    off = offs([0, 50, 100])
    sums = torch.empty((2, 3), dtype=torch.float64, device="cuda:0")
    raw = torch.empty(64, dtype=torch.uint8, device="cuda:0")
    host_off = np.array([0, 50, 100], dtype=np.int64)
    host_sums = np.zeros(6)
    before = ctx.launch_count
    assert _call(None, off.data_ptr(), 2, sums.data_ptr()) == L.ERR_INVALID
    assert _call(b, 0, 2, sums.data_ptr()) == L.ERR_INVALID
    assert _call(b, off.data_ptr(), 2, 0) == L.ERR_INVALID
    assert _call(b, off.data_ptr() + 4, 2, sums.data_ptr()) == L.ERR_INVALID
    assert _call(b, off.data_ptr(), 2, raw.data_ptr() + 4) == L.ERR_INVALID
    assert _call(b, host_off.ctypes.data, 2, sums.data_ptr()) == L.ERR_INVALID
    assert _call(b, off.data_ptr(), 2, host_sums.ctypes.data) == L.ERR_INVALID
    one = g.DeviceBatch.from_host(ctx, 3, {1: np.ones(3)}, broadcast=True)
    assert _call(one, off.data_ptr(), 2, sums.data_ptr()) == L.ERR_SHAPE
    assert ctx.launch_count == before
    assert _call(b, 0, 0, 0) == L.OK and ctx.launch_count == before


# ---- determinism -------------------------------------------------------------------------------------------------------
def test_repeat_graph_and_second_ctx_are_bit_identical():
    length = 40 * CHUNK + 123
    rng = np.random.default_rng(10)
    host = {2: rng.standard_normal((66, length))}
    cuts = sorted(set(rng.integers(0, length, 300).tolist()))
    offsets = [0, *cuts, length]
    ctx = g.Ctx.on_torch_stream(0)
    try:
        b = g.DeviceBatch.from_host(ctx, 12, host)
        off = offs(offsets)
        first = b.segment_sum(off).clone()
        again = b.segment_sum(off)
        torch.cuda.synchronize()
        assert torch.equal(first.view(torch.int64), again.view(torch.int64))
        out = torch.full_like(first, float("nan"))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ctx.torch_stream):
            b.segment_sum(off, out=out)
        for _ in range(2):
            out.fill_(float("nan"))
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(out.view(torch.int64), first.view(torch.int64))
        del graph
    finally:
        torch.cuda.set_stream(torch.cuda.default_stream(0))
        ctx.sync()
    ctx2 = g.Ctx(0)
    b2 = g.DeviceBatch.from_host(ctx2, 12, host)
    other = b2.segment_sum(off)
    ctx2.sync()
    assert torch.equal(other.view(torch.int64), first.view(torch.int64))


# ---- end to end --------------------------------------------------------------------------------------------------------
def test_cfg5_plan_then_segments_against_the_oracle(ctx):
    w = W.WORKLOADS["cfg5"]
    plan = g.Plan(ctx, W.specialize(w))
    length = 6000
    host = W.host_inputs(w, length)
    bcs = [bc for _, bc in w.inputs]
    dev = [g.DeviceBatch.from_host(ctx, w.n, d, broadcast=bc) for d, bc in zip(host, bcs)]
    out = plan.eval(dev)
    offsets = [0, 1, 17, 4096, 4097, 5000, length]
    got = out.segment_sum(offs(offsets))
    ctx.sync()
    got = got.cpu().numpy()
    want = oracle_eval(w.build, w.metric, host, bcs, length)[2]
    scale = oracle_abs_scale(w.build, w.metric, host, bcs, length)[2]
    for j in range(len(offsets) - 1):
        a, e = offsets[j], offsets[j + 1]
        for r in range(66):
            ref = math.fsum(want[r, a:e].tolist())
            bar = REL_SUM * math.fsum(np.maximum(np.abs(want[r, a:e]), scale[r, a:e]).tolist())
            assert abs(got[j, r] - ref) <= bar, (j, r, got[j, r], ref)
    # one segment over the whole batch agrees with gaast_eval_sum at the same bar (not bit for bit: another order)
    whole = out.segment_sum(offs([0, length]))
    dsum = torch.full((66,), float("nan"), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    plan.eval_sum(dev, dsum.data_ptr(), out=plan.alloc_output(length))
    ctx.sync()
    bar = REL_SUM * np.array([math.fsum(np.maximum(np.abs(want[r]), scale[r]).tolist()) for r in range(66)])
    assert (np.abs(whole.cpu().numpy()[0] - dsum.cpu().numpy()) <= bar).all()
