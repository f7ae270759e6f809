"""gaast_batch_segment_sum's kernels (csrc/device/segments.cu) on the CPU, with 64-column chunks: bit for bit the
documented order of the additions, on every segment layout; NaN everywhere for invalid offsets, and a correct next
call on the same batch."""
import numpy as np
import pytest

from tests.kernel_emu import segments as SE

E = 64


def _layouts(length, rng):
    lens = rng.integers(0, 41, size=length)
    rand = np.concatenate([[0], np.cumsum(lens)])
    rand = rand[rand <= length]
    edges = sorted({0, length, *[c for k in range(E, length, E) for c in (k - 1, k, k + 1) if 0 < c < length]})
    return {
        "ones": list(range(length + 1)),
        "random_0_40": list(rand),
        "whole": [0, length],
        "chunk_edges": edges,
        "many_chunks": [0, 3, length - 2, length],
        "inner_range": [7, 7, 100, 101, 101, length - 9],
        "empty_pile": [0, 10] + [70] * 70 + [71, length],  # more than 32 boundaries in one window of 32 columns
    }


def _check(batch, rows, offsets):
    got = batch.segment_sum(offsets)
    want = SE.replay(rows, offsets, E)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.int64), want.view(np.int64)), np.nanmax(np.abs(got - want))
    empty = np.diff(np.asarray(offsets)) == 0
    assert not np.signbit(got[empty]).any()  # empty segments: +0.0
    return got


@pytest.mark.parametrize("S,dtype", [(1, np.float64), (8, np.float64), (20, np.float64), (3, np.float32)])
def test_layouts_match_the_documented_order(S, dtype):
    rng = np.random.default_rng(S)
    length = 40 * E + 5  # a ragged last chunk; 41 chunks: a segment over all of them takes two groups of 32 pieces
    rows = rng.standard_normal((S, length)).astype(dtype)
    batch = SE.SegmentBatch(rows, E)
    for name, offsets in _layouts(length, rng).items():
        _check(batch, rows, offsets)


def test_short_batches():
    rng = np.random.default_rng(7)
    for length in (0, 1, 31, 32, 33, E, E + 1):
        rows = rng.standard_normal((2, length))
        batch = SE.SegmentBatch(rows, E)
        _check(batch, rows, [0, length])
        _check(batch, rows, list(range(length + 1)))
        _check(batch, rows, [0, 0, length, length])


def test_invalid_offsets_give_nan_and_the_next_call_is_right():
    rng = np.random.default_rng(3)
    length = 5 * E + 3
    rows = rng.standard_normal((3, length))
    batch = SE.SegmentBatch(rows, E)
    valid = [0, 10, 70, 200, length]
    for bad in ([0, 100, 50, length], [-1, 10, length], [0, 10, length + 1], [0, 300, 200, 100, 0]):
        got = batch.segment_sum(bad)
        assert np.isnan(got).all(), bad
        _check(batch, rows, valid)  # (the flag was cleared)


def test_sums_are_overwritten_and_guards_stay():
    rng = np.random.default_rng(5)
    length = 3 * E
    rows = rng.standard_normal((4, length))
    batch = SE.SegmentBatch(rows, E)
    offsets = [0, 0, 5, 130, 130, length]
    buf = np.full((len(offsets) - 1 + 2, 4), np.nan)
    buf[0] = buf[-1] = 1234.5
    inner = buf[1:-1]
    got = batch.segment_sum(offsets, inner)
    assert not np.isnan(got).any()
    assert (buf[0] == 1234.5).all() and (buf[-1] == 1234.5).all()
    want = SE.replay(rows, offsets, E)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
