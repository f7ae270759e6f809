"""The write-extent checker of tests/guarded_layout.py, held to planted violations on numpy buffers: a write into a
gap, a write into a guard, a missing store and a changed input must each be reported with their grade, row and
column, and a clean call must pass.  (tests/test_gpu_write_extent.py relies on the checker on the device.)"""
import numpy as np
import pytest

from tests.guarded_layout import GUARD, GuardedBatch, check, poison, predicted_launch, sentinel, violations


def _call(dtype, gap=3, offset=1, length=7):
    """A 'call' that does everything right: inputs filled, every output scalar of [0, len) written."""
    rng = np.random.default_rng(5)
    a = GuardedBatch({0: 1, 1: 3}, length, gap=gap, offset=offset, dtype=dtype, role="in")
    a.fill({0: rng.uniform(-1, 1, (1, length)), 1: rng.uniform(-1, 1, (3, length))})
    out = GuardedBatch({2: 3}, length, gap=gap, offset=offset, dtype=dtype, role="out")
    before = a.bits()
    out.grades[2].view[...] = 0.5  # the kernel's stores
    return a, before, out


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_layout_and_a_clean_call(dtype):
    a, before, out = _call(dtype)
    assert violations([out], [(a, before)]) == []
    b = out.grades[2]
    esize = np.dtype(dtype).itemsize
    assert b.stride == 10 and b.start == GUARD + 1 and (b.start * esize) % 16 == esize % 16
    flat = b.bits()
    assert (flat[:b.start] == sentinel(dtype, "out")).all() and (flat[b.start + 3 * 10:] == sentinel(dtype, "out")).all()
    assert (flat[b.start + 7:b.start + 10] == sentinel(dtype, "out")).all()  # the gap of row 0
    assert sentinel(dtype, "in") != sentinel(dtype, "out")
    assert np.isnan(poison(np.empty(3, dtype=dtype), "in")).all()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_write_into_a_gap_is_caught(dtype):
    a, before, out = _call(dtype)
    out.grades[2].flat[out.grades[2].start + 1 * 10 + 7] = 1.0  # row 1, first column past the length
    found = violations([out], [(a, before)])
    assert len(found) == 1 and "output grade 2 row 1 column 7 (gap)" in found[0] and "outside" in found[0], found


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_write_into_a_guard_is_caught(dtype):
    a, before, out = _call(dtype)
    b = out.grades[2]
    b.flat[b.start + 3 * 10 + 2] = 0.0  # the trailing guard, third scalar
    b.flat[b.start - 1] = -0.0  # the last scalar of the leading guard
    found = violations([out], [(a, before)])
    assert len(found) == 2, found
    assert "output grade 2 row -1 column -1 (leading guard)" in found[0], found
    assert "output grade 2 row 3 column 2 (trailing guard)" in found[1], found


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_missing_store_is_caught(dtype):
    a, before, out = _call(dtype)
    b = out.grades[2]
    poison(b.view[2:3, 6:7], "out")  # the last element of the last row was never stored
    found = violations([out], [(a, before)])
    assert len(found) == 1 and "output grade 2 row 2 column 6:" in found[0] and "never written" in found[0], found
    with pytest.raises(AssertionError, match="grade 2 row 2 column 6"):
        check([out], [(a, before)], "planted")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_input_sentinel_in_a_result_is_caught(dtype):
    a, before, out = _call(dtype)
    poison(out.grades[2].view[0:1, 0:1], "in")  # a value read from an input's padding
    found = violations([out], [(a, before)])
    assert len(found) == 1 and "output grade 2 row 0 column 0:" in found[0] and "input sentinel" in found[0], found


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_changed_input_is_caught(dtype):
    a, before, out = _call(dtype)
    a.grades[1].view[1, 4] = 2.0  # inside the rows
    a.grades[0].flat[a.grades[0].start + 8] = 2.0  # in the gap of the one-row grade
    found = violations([out], [(a, before)])
    assert len(found) == 2, found
    assert "input grade 0 row 0 column 8 (gap): changed" in found[0], found
    assert "input grade 1 row 1 column 4: changed" in found[1], found


def test_predicted_launch():
    """launch_length's decision, restated: 128-bit rows, whole strides, and the widened odd batch."""
    al = [(4096, 1024), (8192, 1024)]
    assert predicted_launch(8, 1000, al, owned_output=True) == ("aligned", 1000)
    assert predicted_launch(8, 1001, al, owned_output=True) == ("padded", 1002)
    assert predicted_launch(8, 1001, al, owned_output=True, with_sum=True) == ("unaligned", 1001)
    assert predicted_launch(8, 1001, al, owned_output=False) == ("unaligned", 1001)
    assert predicted_launch(8, 1001, [(4096, 1001)], owned_output=True) == ("unaligned", 1001)  # no room to widen
    assert predicted_launch(8, 1000, [(4096 + 8, 1024)], owned_output=True) == ("unaligned", 1000)  # 8 bytes off
    assert predicted_launch(8, 1000, [(4096, 1001)], owned_output=True) == ("unaligned", 1000)  # odd stride
    assert predicted_launch(4, 1001, [(4096, 1004)], owned_output=True) == ("padded", 1004)
    assert predicted_launch(4, 1002, [(4096, 1004)], owned_output=True) == ("padded", 1004)
    assert predicted_launch(4, 1000, [(4096 + 4, 1004)], owned_output=True) == ("unaligned", 1000)
    assert predicted_launch(4, 1000, [(4096, 1002)], owned_output=True) == ("unaligned", 1000)
    assert predicted_launch(8, 1, [], owned_output=True) == ("padded", 2)  # every input broadcast, owned output
