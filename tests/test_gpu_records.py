"""Element-major records (gaast_batch_pack_records / _unpack_records / _upload_records / _download_records): one
multivector per record, its components in slot order, moved into and out of the batch's per-grade rows bit for bit.

The batch side is read back with the per-grade gaast_batch_download and compared with numpy's transpose of the same
records; scalars are compared as integers, and the inputs are random bit patterns plus -0.0, subnormals, +-inf and
NaNs with distinct payloads.  Round trips run every length up to 2^27 scalars per side (wider algebras stop at the
lengths below that; G(16) runs a handful of elements)."""
from math import comb

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from gaast_b200.expr import grade_mask  # noqa: E402
from tests.helpers import assert_bit_exact, assert_close, oracle_abs_scale, oracle_eval  # noqa: E402

torch = pytest.importorskip("torch")

FULL = {n: tuple(range(n + 1)) for n in (3, 5, 6, 10, 12, 16)}
ALGEBRAS = [(3, (2,)), (3, FULL[3]), (5, (1,)), (12, (2,)), (6, FULL[6]), (10, FULL[10]), (12, FULL[12]),
            (16, FULL[16])]
LENGTHS = [1, 31, 32, 33, 127, 1000, 2**20 + 3]
MAX_SCALARS = 2**27


@pytest.fixture(scope="module")
def ctx():
    return g.Ctx.on_torch_stream(0)


def _width(n, grades):
    return sum(comb(n, k) for k in grades)


def _types(dtype):
    return (np.float32, np.uint32, torch.int32) if dtype == L.F32 else (np.float64, np.uint64, torch.int64)


def _bits(rng, shape, dtype):
    """Random bit patterns (every class of float, NaN payloads included) with the special values planted."""
    fl, ui, _ = _types(dtype)
    a = rng.integers(0, np.iinfo(ui).max, size=shape, dtype=ui, endpoint=True)
    flat = a.reshape(-1)
    sign = ui(1) << ui(8 * np.dtype(ui).itemsize - 1)
    exp_all = ui(0x7F800000) if ui is np.uint32 else ui(0x7FF0000000000000)
    specials = [sign, ui(1), sign | ui(1), ui(3), exp_all, sign | exp_all, exp_all | ui(1), exp_all | ui(0x12345),
                sign | exp_all | ui(0x2A), exp_all | ui(0x777)]
    for i, v in enumerate(specials[:flat.size]):
        flat[(i * 7919) % flat.size] = v
    return a


def _dev(host_bits, offset_scalars=0):
    """A device copy of `host_bits` starting `offset_scalars` past a 256-byte boundary: (allocation, the copy as a
    uint8 view of it, its address).  Callers keep the first two alive until the stream has used the address."""
    es = host_bits.dtype.itemsize
    raw = torch.empty(host_bits.size * es + 512, dtype=torch.uint8, device="cuda")
    base = (raw.data_ptr() + 255) // 256 * 256 - raw.data_ptr() + offset_scalars * es
    view = raw[base:base + host_bits.size * es]
    view.copy_(torch.from_numpy(host_bits.reshape(-1).view(np.uint8)).cuda())
    return raw, view, view.data_ptr()


def _host(view, shape, ui):
    return view.cpu().numpy().view(ui).reshape(shape)


def _slots(n, record_grades):
    """Record column of each grade's first component."""
    out, off = {}, 0
    for k in record_grades:
        out[k] = off
        off += comb(n, k)
    return out


def _batch_bits(b, n, grades, ui):
    return {k: b.download(k).view(ui) for k in grades}


def _check_batch(b, n, grades, record_grades, recs, ui, what):
    off = _slots(n, record_grades)
    for k, got in _batch_bits(b, n, grades, ui).items():
        want = recs[:, off[k]:off[k] + comb(n, k)].T
        assert np.array_equal(got, want), f"{what}: grade {k} differs from the records' transpose"


# ---------------------------------------------------------------------------------------------------- 1. round trip
@pytest.mark.parametrize("dtype", [L.F64, L.F32], ids=["f64", "f32"])
@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("n,grades", ALGEBRAS, ids=[f"G{n}{''.join(map(str, gr))}" for n, gr in ALGEBRAS])
def test_round_trip_bit_for_bit(ctx, n, grades, length, dtype):
    K = _width(n, grades)
    if length * K > MAX_SCALARS or (n == 16 and length > 33):
        pytest.skip("above this test's size cap")
    fl, ui, _ = _types(dtype)
    rng = np.random.default_rng(length * 131 + n * 7 + K + dtype)
    mask = grade_mask(grades)
    recs = _bits(rng, (length, K), dtype)
    b = g.DeviceBatch.alloc(ctx, n, grades, length, dtype=dtype)
    raw, view, ptr = _dev(recs, 0)
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(ptr), mask))
    ctx.sync()
    _check_batch(b, n, grades, grades, recs, ui, "pack")
    out_raw, out_view, out_ptr = _dev(np.zeros_like(recs), 1)  # one scalar past a 256-byte boundary
    L.check(L.lib.gaast_batch_unpack_records(b._h, 0, length, L.vp(out_ptr), mask))
    ctx.sync()
    assert np.array_equal(_host(out_view, recs.shape, ui), recs), "unpack"
    # sub-ranges, from and to pointers one scalar past a 256-byte boundary
    for first in sorted({f for f in (1, 7, length - 5) if 0 < f < length}):
        count = length - first
        sub = _bits(rng, (count, K), dtype)
        sraw, _, sptr = _dev(sub, 1)
        L.check(L.lib.gaast_batch_pack_records(b._h, first, count, L.vp(sptr), mask))
        recs[first:] = sub
        uraw, uview, uptr = _dev(np.zeros_like(sub), 1)
        L.check(L.lib.gaast_batch_unpack_records(b._h, first, count, L.vp(uptr), mask))
        ctx.sync()
        _check_batch(b, n, grades, grades, recs, ui, f"pack first={first}")
        assert np.array_equal(_host(uview, sub.shape, ui), sub), f"unpack first={first}"


# ---------------------------------------------------------------------------------------------------- 2. batch kinds
@pytest.mark.parametrize("dtype", [L.F64, L.F32], ids=["f64", "f32"])
def test_wrapped_batch_with_separate_grade_tensors(ctx, dtype):
    n, grades, length, stride = 5, (1, 3), 1000, 1029
    fl, ui, _ = _types(dtype)
    tdt = torch.float32 if dtype == L.F32 else torch.float64
    tensors = {k: torch.empty((comb(n, k), stride), dtype=tdt, device="cuda")[:, :length] for k in grades}
    b = g.DeviceBatch.wrap_torch(ctx, n, tensors)
    assert b.stride == stride
    K, mask = _width(n, grades), grade_mask(grades)
    recs = _bits(np.random.default_rng(5), (length, K), dtype)
    _, view, ptr = _dev(recs, 1)
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(ptr), mask))
    ctx.sync()
    off = _slots(n, grades)
    for k in grades:
        got = tensors[k].cpu().numpy().view(ui)
        assert np.array_equal(got, recs[:, off[k]:off[k] + comb(n, k)].T), k
    _, uview, uptr = _dev(np.zeros_like(recs), 0)
    L.check(L.lib.gaast_batch_unpack_records(b._h, 0, length, L.vp(uptr), mask))
    ctx.sync()
    assert np.array_equal(_host(uview, recs.shape, ui), recs)


def test_sparse_batch_drops_absent_components_and_unpacks_them_as_zero(ctx):
    n, length = 12, 1001
    rng = np.random.default_rng(9)
    idx = sorted(rng.choice(66, size=9, replace=False).tolist())
    b = g.DeviceBatch.from_host_sparse(ctx, n, {1: np.zeros((12, length)), 2: (idx, np.zeros((9, length)))})
    K, mask = 12 + 66, grade_mask((1, 2))
    recs = _bits(rng, (length, K), L.F64)
    _, _, ptr = _dev(recs, 1)
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(ptr), mask))
    ctx.sync()
    assert np.array_equal(b.download(1).view(np.uint64), recs[:, :12].T)
    assert np.array_equal(b.download(2).view(np.uint64), recs[:, 12 + np.array(idx)].T)
    nan = np.full_like(recs, 0x7FF8DEAD00000000)
    _, uview, uptr = _dev(nan, 0)
    L.check(L.lib.gaast_batch_unpack_records(b._h, 0, length, L.vp(uptr), mask))
    ctx.sync()
    want = np.zeros_like(recs)
    want[:, :12] = recs[:, :12]
    want[:, 12 + np.array(idx)] = recs[:, 12 + np.array(idx)]
    assert np.array_equal(_host(uview, recs.shape, np.uint64), want)  # absent components: +0 bits


def test_broadcast_batch_takes_exactly_one_record(ctx):
    n, grades = 5, (0, 2, 4)
    K, mask = _width(n, grades), grade_mask(grades)
    b = g.DeviceBatch.alloc(ctx, n, grades, 1, broadcast=True)
    recs = _bits(np.random.default_rng(3), (1, K), L.F64)
    _, view, ptr = _dev(recs, 1)
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, 1, L.vp(ptr), mask))
    ctx.sync()
    _check_batch(b, n, grades, grades, recs, np.uint64, "broadcast")
    for first, count in ((0, 0), (0, 2), (1, 1), (1, 0)):
        assert L.lib.gaast_batch_pack_records(b._h, first, count, L.vp(ptr), mask) == L.ERR_SHAPE, (first, count)
        assert L.lib.gaast_batch_unpack_records(b._h, first, count, L.vp(ptr), mask) == L.ERR_SHAPE, (first, count)


# ------------------------------------------------------------------------------------------------ 3. superset records
@pytest.mark.parametrize("n", [3, 5, 10])  # G(10) full records move in chunks: partial and empty ones here
@pytest.mark.parametrize("grades", [(1,), (2,), (0, 2)])
def test_superset_records(ctx, n, grades):
    length = 1000
    full = FULL[n] if n in FULL else tuple(range(n + 1))
    K, fmask = _width(n, full), grade_mask(full)
    recs = _bits(np.random.default_rng(n * 10 + len(grades)), (length, K), L.F64)
    b = g.DeviceBatch.alloc(ctx, n, grades, length)
    _, _, ptr = _dev(recs, 1)
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(ptr), fmask))
    ctx.sync()
    _check_batch(b, n, grades, full, recs, np.uint64, "superset pack")
    _, uview, uptr = _dev(np.full_like(recs, 0x7FF8000000000001), 0)
    L.check(L.lib.gaast_batch_unpack_records(b._h, 0, length, L.vp(uptr), fmask))
    ctx.sync()
    got = _host(uview, recs.shape, np.uint64)
    off = _slots(n, full)
    want = np.zeros_like(recs)
    for k in grades:
        want[:, off[k]:off[k] + comb(n, k)] = recs[:, off[k]:off[k] + comb(n, k)]
    assert np.array_equal(got, want), "every scalar of the range is written: the batch's value or +0"


# --------------------------------------------------------------------------------------------- 4. ranges and guards
@pytest.mark.parametrize("dtype", [L.F64, L.F32], ids=["f64", "f32"])
def test_ranges_leave_everything_else_untouched(ctx, dtype):
    n, grades, length = 12, (2,), 1000
    fl, ui, _ = _types(dtype)
    K, mask = 66, grade_mask(grades)
    sentinel = _bits(np.random.default_rng(1), (66, length), dtype)
    b = g.DeviceBatch.from_host(ctx, n, {2: sentinel.view(fl)}, dtype=dtype)
    first, count = 37, 501
    sub = _bits(np.random.default_rng(2), (count, K), dtype)
    _, _, ptr = _dev(sub, 1)
    L.check(L.lib.gaast_batch_pack_records(b._h, first, count, L.vp(ptr), mask))
    ctx.sync()
    want = sentinel.copy()
    want[:, first:first + count] = sub.T
    assert np.array_equal(b.download(2).view(ui), want)
    # unpack into the middle of a guarded buffer: the guards stay
    guard = 67
    buf = _bits(np.random.default_rng(4), (count * K + 2 * guard,), dtype)
    _, view, bptr = _dev(buf, 1)
    L.check(L.lib.gaast_batch_unpack_records(b._h, first, count, L.vp(bptr + guard * buf.dtype.itemsize), mask))
    ctx.sync()
    got = _host(view, buf.shape, ui)
    assert np.array_equal(got[:guard], buf[:guard]) and np.array_equal(got[-guard:], buf[-guard:])
    assert np.array_equal(got[guard:-guard].reshape(count, K), sub)


def test_launch_counts(ctx):
    b = g.DeviceBatch.alloc(ctx, 3, FULL[3], 100)
    recs = torch.zeros((100, 8), dtype=torch.float64, device="cuda")
    mask = grade_mask(FULL[3])
    n0 = ctx.launch_count
    assert L.lib.gaast_batch_pack_records(b._h, 5, 0, None, mask) == L.OK
    assert L.lib.gaast_batch_unpack_records(b._h, 100, 0, None, mask) == L.OK
    assert L.lib.gaast_batch_upload_records(b._h, 0, 0, None, mask) == L.OK
    assert L.lib.gaast_batch_download_records(b._h, 0, 0, None, mask) == L.OK
    assert ctx.launch_count == n0
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, 100, L.vp(recs.data_ptr()), mask))
    assert ctx.launch_count == n0 + 1
    L.check(L.lib.gaast_batch_unpack_records(b._h, 0, 100, L.vp(recs.data_ptr()), mask))
    assert ctx.launch_count == n0 + 2
    ctx.sync()


# -------------------------------------------------------------------------------------------------------- 5. errors
def test_errors(ctx):
    b = g.DeviceBatch.alloc(ctx, 3, (0, 2), 100)
    recs = torch.zeros((100, 8), dtype=torch.float64, device="cuda")
    p = L.vp(recs.data_ptr())
    for fn in (L.lib.gaast_batch_pack_records, L.lib.gaast_batch_unpack_records):
        assert fn(b._h, 0, 100, p, grade_mask((2,))) == L.ERR_SHAPE  # lacks grade 0
        assert fn(b._h, 0, 100, p, grade_mask((0, 1))) == L.ERR_SHAPE
        assert fn(b._h, 0, 100, p, 0xF0) == L.ERR_SHAPE  # grades above n
        assert fn(b._h, 1, 100, p, grade_mask(FULL[3])) == L.ERR_SHAPE
        assert fn(b._h, 101, 0, p, grade_mask(FULL[3])) == L.ERR_SHAPE
        assert fn(b._h, 0, 1, None, grade_mask(FULL[3])) == L.ERR_INVALID
        assert fn(None, 0, 1, p, grade_mask(FULL[3])) == L.ERR_INVALID
    for fn in (L.lib.gaast_batch_upload_records, L.lib.gaast_batch_download_records):
        assert fn(b._h, 0, 1, None, grade_mask(FULL[3])) == L.ERR_INVALID
        assert fn(b._h, 99, 2, None, grade_mask(FULL[3])) == L.ERR_SHAPE
        assert fn(None, 0, 1, None, grade_mask(FULL[3])) == L.ERR_INVALID
    # a batch of no grade takes no record of no component (records of zero scalars)
    empty = g.DeviceBatch.alloc(ctx, 3, (), 100)
    host = np.zeros(8)
    for fn in (L.lib.gaast_batch_pack_records, L.lib.gaast_batch_unpack_records):
        assert fn(empty._h, 0, 100, p, 0) == L.ERR_SHAPE
    for fn in (L.lib.gaast_batch_upload_records, L.lib.gaast_batch_download_records):
        assert fn(empty._h, 0, 100, L.vp(host.ctypes.data), 0) == L.ERR_SHAPE
    ctx.sync()


# ------------------------------------------------------------------------------------------------- 6. host variants
@pytest.mark.parametrize("chunk_mib", [None, 1])
@pytest.mark.parametrize("dtype", [L.F64, L.F32], ids=["f64", "f32"])
def test_host_variants_match_the_device_path(ctx, monkeypatch, chunk_mib, dtype):
    if chunk_mib:
        monkeypatch.setenv("GAAST_HOST_CHUNK_MIB", str(chunk_mib))
        L.lib.gaast_reload_env()
    try:
        n, grades, length = 12, (1, 2), 100_003  # 1 MiB chunks: 1344 records (f64) each, a ragged last one
        fl, ui, _ = _types(dtype)
        K, mask = 78, grade_mask(grades)
        recs = _bits(np.random.default_rng(11), (length, K), dtype)
        dev = g.DeviceBatch.alloc(ctx, n, grades, length, dtype=dtype)
        _, _, ptr = _dev(recs, 1)
        L.check(L.lib.gaast_batch_pack_records(dev._h, 0, length, L.vp(ptr), mask))
        want = _batch_bits(dev, n, grades, ui)
        pageable = g.DeviceBatch.from_records(ctx, n, grades, recs.view(fl), dtype=dtype)
        pinned_arr = g.HostArray(length, K, dtype=fl)
        pinned_arr.array[:] = recs.view(fl)
        pinned = g.DeviceBatch.alloc(ctx, n, grades, length, dtype=dtype)
        pinned.pack_records(pinned_arr.array)
        for what, b in (("pageable", pageable), ("pinned", pinned)):
            got = _batch_bits(b, n, grades, ui)
            for k in grades:
                assert np.array_equal(got[k], want[k]), (what, k)
        assert np.array_equal(pageable.to_records().view(ui), recs)
        out = g.HostArray(length, K, dtype=fl)
        L.check(L.lib.gaast_batch_download_records(pinned._h, 0, length, L.vp(out.array.ctypes.data), mask))
        ctx.sync()
        assert np.array_equal(out.array.view(ui), recs)
        pinned_arr.free()
        out.free()
    finally:
        if chunk_mib:
            monkeypatch.delenv("GAAST_HOST_CHUNK_MIB")
            L.lib.gaast_reload_env()


# -------------------------------------------------------------------------------------------------- 7. end to end
def _records_of(n, data, grades):
    return np.ascontiguousarray(np.concatenate([np.atleast_2d(np.asarray(data[k]).reshape(comb(n, k), -1))
                                                for k in grades], axis=0).T)


def _grades_of_records(n, recs, grades):
    off = _slots(n, grades)
    return {k: np.ascontiguousarray(recs[:, off[k]:off[k] + comb(n, k)].T) for k in grades}


@pytest.mark.parametrize("arith", [L.ARITH_STRICT, L.ARITH_FMA], ids=["strict", "fma"])
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_end_to_end_records_in_and_out(ctx, name, arith):
    w = W.WORKLOADS[name]
    length = 4099
    host = W.host_inputs(w, length)
    bcs = [bc for _, bc in w.inputs]
    plan = g.Plan(ctx, W.specialize(w))
    root = plan.root_grades()
    ref_in = [g.DeviceBatch.from_host(ctx, w.n, host[s], broadcast=bc) for s, bc in enumerate(bcs)]
    ref = plan.eval(ref_in, arith=arith).to_host()
    want = oracle_eval(w.build, w.metric, host, bcs, length)
    if arith == L.ARITH_STRICT:
        assert_bit_exact(ref, want, f"{name} per-grade path")
    else:
        assert_close(ref, want, oracle_abs_scale(w.build, w.metric, host, bcs, length), what=f"{name} per-grade path")
    recs = [_records_of(w.n, host[s], grades) for s, (grades, _) in enumerate(w.inputs)]
    via_host = [g.DeviceBatch.from_records(ctx, w.n, grades, recs[s], broadcast=bc)
                for s, (grades, bc) in enumerate(w.inputs)]
    via_dev = [g.DeviceBatch.from_records(ctx, w.n, grades, torch.from_numpy(recs[s]).cuda(), broadcast=bc)
               for s, (grades, bc) in enumerate(w.inputs)]
    ref_bits = _records_of(w.n, ref, root).view(np.uint64)
    out_h = plan.eval(via_host, arith=arith).to_records()
    assert np.array_equal(out_h.view(np.uint64), ref_bits), f"{name}: host records path"
    out_dev = torch.empty((length, _width(w.n, root)), dtype=torch.float64, device="cuda")
    plan.eval(via_dev, arith=arith).to_records(out=out_dev)
    ctx.sync()
    assert np.array_equal(out_dev.cpu().numpy().view(np.uint64), ref_bits), f"{name}: device records path"


# ------------------------------------------------------------------------------------------------- 8. graph capture
def test_graph_capture_of_pack_eval_unpack(ctx):
    w = W.WORKLOADS["cfg1"]
    length = 4099
    plan = g.Plan(ctx, W.specialize(w))
    K = 8
    rec_in = [torch.empty((length, K), dtype=torch.float64, device="cuda") for _ in range(3)]
    rec_out = torch.empty((length, 3), dtype=torch.float64, device="cuda")
    ins = [g.DeviceBatch.alloc(ctx, 3, FULL[3], length) for _ in range(3)]
    out = plan.alloc_output(length)

    def step():
        for b, r in zip(ins, rec_in):
            b.pack_records(r)
        plan.eval(ins, out=out)
        out.to_records(out=rec_out)

    rng = np.random.default_rng(21)
    for r in rec_in:
        r.copy_(torch.from_numpy(rng.uniform(-1, 1, (length, K))))
    step()  # warm-up: row maps, kernel
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=ctx.torch_stream):
        step()
    for trial in range(2):
        for r in rec_in:
            r.copy_(torch.from_numpy(rng.uniform(-1, 1, (length, K))))
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        replayed = rec_out.clone()
        rec_out.fill_(float("nan"))
        step()
        torch.cuda.synchronize()
        assert torch.equal(replayed.view(torch.int64), rec_out.view(torch.int64)), trial


# ------------------------------------------------------------------------------------------------- 9. large indices
def test_large_indices_f32(ctx):
    """f32 G(8,4) bivector records with len x 66 > 2^32 scalars (about 18 GB per side)."""
    n, K, length = 12, 66, 2**26 + 12345
    assert length * K > 2**32
    recs = torch.randint(-2**31, 2**31 - 1, (length, K), dtype=torch.int32, device="cuda")
    batch = torch.empty((K, length), dtype=torch.float32, device="cuda")
    b = g.DeviceBatch.wrap_torch(ctx, n, {2: batch})
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(recs.data_ptr()), grade_mask((2,))))
    ctx.sync()
    gen = torch.Generator(device="cuda").manual_seed(1234)
    e = torch.randint(0, length, (1 << 20,), device="cuda", generator=gen)
    c = torch.randint(0, K, (1 << 20,), device="cuda", generator=gen)
    e = torch.cat([e, torch.full((K,), length - 1, device="cuda"), torch.full((K,), length - 2, device="cuda")])
    c = torch.cat([c, torch.arange(K, device="cuda"), torch.arange(K, device="cuda")])
    got = batch.view(torch.int32)[c, e]
    assert torch.equal(got, recs[e, c])
    del recs, batch, got
    b.free()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("dtype", [L.F64, L.F32], ids=["f64", "f32"])
def test_wide_records_at_full_length(ctx, dtype):
    """G(10) full records (1024 components, moved in chunks) at 2^20 + 3 elements: 8.6 GB per side in f64, compared
    on the device."""
    n, K, length = 10, 1024, 2**20 + 3
    _, _, ti = _types(dtype)
    fdt = torch.float32 if dtype == L.F32 else torch.float64
    mask = grade_mask(FULL[10])
    gen = torch.Generator(device="cuda").manual_seed(77)
    recs = torch.randint(-2**31, 2**31 - 1, (length, K * (2 if ti == torch.int64 else 1)), dtype=torch.int32,
                         device="cuda", generator=gen).view(ti)
    rows = torch.empty((K, length), dtype=fdt, device="cuda")
    off = _slots(n, FULL[10])
    b = g.DeviceBatch.wrap_torch(ctx, n, {k: rows[off[k]:off[k] + comb(n, k)] for k in FULL[10]})
    L.check(L.lib.gaast_batch_pack_records(b._h, 0, length, L.vp(recs.data_ptr()), mask))
    ctx.sync()
    assert torch.equal(rows.view(ti), recs.t())
    out = torch.full_like(recs, -1)
    first = 7
    L.check(L.lib.gaast_batch_unpack_records(b._h, first, length - first, L.vp(out[first:].data_ptr()), mask))
    ctx.sync()
    assert torch.equal(out[first:], recs[first:]) and bool((out[:first] == -1).all())
    del recs, rows, out
    b.free()
    torch.cuda.empty_cache()
