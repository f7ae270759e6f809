"""TEST INFRASTRUCTURE: poisoned, guarded batch layouts and the check of what a call wrote.

A parity test that reads back `[0, len)` of an output cannot see a store that landed past the end of a row (on a
wrapped batch whose stride equals its length that is column 0 of the next row, which another block writes too) or a
store that never happened (allocators hand back the block a previous, correct result was just freed from).  Here
every grade of a batch lives in one flat buffer of its own:

    [base offset] [GUARD guard scalars] [rows x stride] [GUARD guard scalars],   stride = len + gap

and every scalar of it starts out as a sentinel: a quiet NaN whose payload says whether the buffer is an input or an
output.  After the call, `check` holds the output buffers to "the sentinel everywhere outside `[r*stride, r*stride +
len)` of every row r, and no sentinel inside", and every input buffer to its own bits before the call.  The base
offset sets the alignment of the data pointer modulo 16 bytes (the caching allocators return 512-byte aligned blocks,
and GUARD scalars are a whole number of 16 bytes).

The buffers are numpy arrays, or CUDA tensors when `device` is given: tests/test_write_extent_on_cpu.py holds the
checker itself to planted violations on numpy buffers.

`predicted_launch` restates the specialised engine's launch decision (launch_length, csrc/device/runtime.cu), so that
a test can say which kernel a layout must take and assert it from `Plan.last_kernel()`."""
from __future__ import annotations

import ctypes as C
from math import comb
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

GUARD = 16  # guard scalars on each side of the rows: 128 bytes of f64, 64 of f32
# quiet NaNs with payloads that no arithmetic produces (the device returns its canonical NaN for a NaN result)
SENTINEL = {(np.dtype(np.float64), "in"): 0x7FF8_0000_6A5E_1A1A, (np.dtype(np.float64), "out"): 0x7FF8_0000_6A5E_0E0E,
            (np.dtype(np.float32), "in"): 0x7FC0_1A1A, (np.dtype(np.float32), "out"): 0x7FC0_0E0E}
BITS = {np.dtype(np.float64): np.uint64, np.dtype(np.float32): np.uint32}


def sentinel(dtype, role: str) -> int:
    return SENTINEL[(np.dtype(dtype), role)]


def poison(arr: np.ndarray, role: str) -> np.ndarray:
    """Fills a numpy float array with the sentinel of `role`, bit for bit; returns it."""
    arr.view(BITS[arr.dtype])[...] = sentinel(arr.dtype, role)
    return arr


class GradeBuffer:
    """One grade's flat buffer and the [rows, len] view of its data."""

    def __init__(self, grade: int, rows: int, length: int, stride: int, offset: int, dtype, role: str, device=None):
        self.grade, self.rows, self.length, self.stride, self.role = grade, rows, length, stride, role
        self.dtype = np.dtype(dtype)
        self.start = offset + GUARD  # the scalar index of row 0, column 0
        size = self.start + rows * stride + GUARD
        bits = sentinel(self.dtype, role)
        if device is None:
            self.flat = poison(np.empty(size, dtype=self.dtype), role)
            self.view = np.lib.stride_tricks.as_strided(self.flat[self.start:], (rows, length),
                                                        (stride * self.dtype.itemsize, self.dtype.itemsize))
        else:
            import torch
            ibits = torch.int64 if self.dtype == np.float64 else torch.int32
            fdt = torch.float64 if self.dtype == np.float64 else torch.float32
            self.flat = torch.full((size,), bits, dtype=ibits, device=device).view(fdt)
            self.view = self.flat.as_strided((rows, length), (stride, 1), self.start)

    @property
    def ptr(self) -> int:
        """Address of row 0."""
        if isinstance(self.flat, np.ndarray):
            return self.flat.ctypes.data + self.start * self.dtype.itemsize
        return self.flat.data_ptr() + self.start * self.dtype.itemsize

    def bits(self) -> np.ndarray:
        """A host copy of the whole flat buffer as unsigned integers."""
        flat = self.flat if isinstance(self.flat, np.ndarray) else self.flat.cpu().numpy()
        return flat.view(BITS[self.dtype]).copy()

    def values(self) -> np.ndarray:
        """A host copy of the [rows, len] data."""
        b = self.bits()[self.start:self.start + self.rows * self.stride].view(self.dtype)
        return b.reshape(self.rows, self.stride)[:, :self.length].copy() if self.rows else np.zeros((0, self.length), self.dtype)

    def where(self, i: int) -> str:
        """Names flat index i: its grade, row and column (the guards as row -1 / row `rows`)."""
        rel = i - self.start
        if rel < 0:
            return f"grade {self.grade} row -1 column {rel} (leading guard)"
        if rel >= self.rows * self.stride:
            return f"grade {self.grade} row {self.rows} column {rel - self.rows * self.stride} (trailing guard)"
        r, c = divmod(rel, self.stride)
        return f"grade {self.grade} row {r} column {c}" + (" (gap)" if c >= self.length else "")

    def in_range(self) -> np.ndarray:
        """Mask of the flat scalars inside [r*stride, r*stride + len) of some row r."""
        m = np.zeros(self.start + self.rows * self.stride + GUARD, dtype=bool)
        rows = m[self.start:self.start + self.rows * self.stride].reshape(max(self.rows, 0), self.stride)
        rows[:, :self.length] = True
        return m


class GuardedBatch:
    """A batch of one grade set in guarded, poisoned buffers: {grade: GradeBuffer}.  rows[k] = the stored rows of
    grade k (C(n,k) for a dense grade)."""

    def __init__(self, rows: Dict[int, int], length: int, gap: int = 0, offset: int = 0, dtype=np.float64,
                 role: str = "in", device=None):
        assert gap >= 0 and 0 <= offset * np.dtype(dtype).itemsize < 16
        self.length, self.stride, self.role, self.dtype = length, length + gap, role, np.dtype(dtype)
        self.grades = {k: GradeBuffer(k, r, length, length + gap, offset, dtype, role, device) for k, r in sorted(rows.items())}

    @staticmethod
    def dense(n: int, grades: Iterable[int], length: int, **kw) -> "GuardedBatch":
        return GuardedBatch({k: comb(n, k) for k in grades}, length, **kw)

    def views(self) -> Dict[int, object]:
        return {k: b.view for k, b in self.grades.items()}

    def fill(self, data: Dict[int, np.ndarray]):
        """Writes data[k] ([rows, len]) into the rows; guards and gaps keep the sentinel."""
        for k, b in self.grades.items():
            src = np.asarray(data[k], dtype=self.dtype).reshape(b.rows, b.length)
            if isinstance(b.view, np.ndarray):
                b.view[...] = src
            else:
                import torch
                b.view.copy_(torch.from_numpy(np.ascontiguousarray(src)))

    def values(self) -> Dict[int, np.ndarray]:
        return {k: b.values() for k, b in self.grades.items()}

    def bits(self) -> Dict[int, np.ndarray]:
        return {k: b.bits() for k, b in self.grades.items()}

    def wrap(self, ctx, n: int, broadcast: bool = False):
        """The caller-owned DeviceBatch over these buffers (DeviceBatch.wrap_torch)."""
        import gaast_b200 as g
        if self.length == 0:  # (torch gives an empty view no address: wrap the buffers' row-0 addresses directly)
            assert not broadcast
            return self.wrap_sparse(ctx, n, {})
        return g.DeviceBatch.wrap_torch(ctx, n, self.views(), broadcast=broadcast)

    def wrap_sparse(self, ctx, n: int, components: Dict[int, Optional[Sequence[int]]]):
        """The caller-owned sparse DeviceBatch over these buffers (gaast_batch_wrap_sparse): components[k] = the
        stored component indices of grade k, or None for a dense grade."""
        import gaast_b200 as g
        from gaast_b200 import _lib as L
        grades = sorted(self.grades)
        bitmaps = []
        for k in grades:
            if components.get(k) is None:
                bitmaps.append(None)
                continue
            bits = (L.u64 * ((comb(n, k) + 63) // 64))()
            for i in components[k]:
                bits[int(i) // 64] |= 1 << (int(i) % 64)
            bitmaps.append(bits)
        pres = (C.POINTER(L.u64) * len(grades))(*[C.cast(b, C.POINTER(L.u64)) if b is not None else None for b in bitmaps])
        ptrs = (L.vp * len(grades))(*[self.grades[k].ptr for k in grades])
        h = L.vp()
        L.check(L.lib.gaast_batch_wrap_sparse(ctx._h, n, sum(1 << k for k in grades), self.length, self.stride, 0,
                                              L.F32 if self.dtype == np.float32 else L.F64, pres, ptrs, C.byref(h)))
        return g.DeviceBatch(h, ctx, n, keep=(self, bitmaps))


def violations(outputs: Sequence[GuardedBatch] = (), inputs: Sequence[Tuple[GuardedBatch, Dict[int, np.ndarray]]] = (),
               limit: int = 8) -> List[str]:
    """What a call did wrong to its guarded batches: outputs[i] must hold the output sentinel everywhere outside the
    rows' [0, len) and no sentinel inside; inputs[i] = (batch, its bits() before the call) must be bit-identical."""
    found: List[str] = []
    for batch in outputs:
        for k, b in batch.grades.items():
            bits = b.bits()
            inside = b.in_range()
            out_s, in_s = sentinel(b.dtype, "out"), sentinel(b.dtype, "in")
            for i in np.flatnonzero(~inside & (bits != out_s))[:limit]:
                found.append(f"output {b.where(int(i))}: written outside the batch (0x{int(bits[i]):x})")
            for i in np.flatnonzero(inside & (bits == out_s))[:limit]:
                found.append(f"output {b.where(int(i))}: never written (still the output sentinel)")
            for i in np.flatnonzero(inside & (bits == in_s))[:limit]:
                found.append(f"output {b.where(int(i))}: holds the input sentinel (a read outside an input)")
    for batch, before in inputs:
        for k, b in batch.grades.items():
            bits = b.bits()
            for i in np.flatnonzero(bits != before[k])[:limit]:
                found.append(f"input {b.where(int(i))}: changed (0x{int(before[k][i]):x} -> 0x{int(bits[i]):x})")
    return found


def check(outputs: Sequence[GuardedBatch] = (), inputs: Sequence[Tuple[GuardedBatch, Dict[int, np.ndarray]]] = (),
          what: str = ""):
    found = violations(outputs, inputs)
    assert not found, f"{what}: {len(found)} write-extent violation(s):\n  " + "\n  ".join(found)


def check_owned(values: Dict[int, np.ndarray], dtype, what: str = ""):
    """A library-owned output poisoned in [0, len) before the call (`poison_owned`): no element may still hold a
    sentinel.  (Its row padding belongs to the library and is not checked.)"""
    bt = BITS[np.dtype(dtype)]
    for k, v in values.items():
        bits = np.ascontiguousarray(v).view(bt)
        for role in ("out", "in"):
            hit = np.argwhere(bits == sentinel(dtype, role))
            assert not len(hit), (f"{what}: owned output grade {k} row {hit[0][0]} column {hit[0][1]} holds the {role}put "
                                  f"sentinel ({len(hit)} elements)")


def poison_owned(batch):
    """Writes the output sentinel over [0, len) of every stored row of a library-owned DeviceBatch."""
    from gaast_b200 import _lib as L
    dt = np.float32 if batch.dtype == L.F32 else np.float64
    for k in batch.grade_set():
        if batch.stored_rows(k):
            batch.upload(k, poison(np.empty((batch.stored_rows(k), batch.length), dtype=dt), "out"))
    return batch


def predicted_launch(esize: int, length: int, streams: Sequence[Tuple[int, int]], owned_output: bool,
                     with_sum: bool = False) -> Tuple[str, int]:
    """The specialised engine's launch for a call: ("aligned" | "padded" | "unaligned", launch length).
    streams = (row-0 address, row stride in scalars) of every per-element (not broadcast) row array the call reads or
    writes.  128-bit accesses need every such row 16-byte aligned, a stride of whole 16 bytes and at least the launch
    length; an odd length is widened over a library-owned output's padding when no batch-sum would see it."""
    quantum = 16 // esize

    def rows_fit(n):
        return all(ptr % 16 == 0 and stride % quantum == 0 and stride >= n for ptr, stride in streams)

    if length % quantum == 0:
        return ("aligned" if rows_fit(length) else "unaligned"), length
    padded = -(-length // quantum) * quantum
    if not with_sum and owned_output and rows_fit(padded):
        return "padded", padded
    return "unaligned", length


def streams_of(batches) -> List[Tuple[int, int]]:
    """(row-0 address, stride) of every stored grade of `batches`: the per-element DeviceBatches of a call (leave out
    its broadcast operands and a null output)."""
    out = []
    for b in batches:
        for k in b.grade_set():
            if b.stored_rows(k):
                out.append((b.grade_ptr(k), b.stride))
    return out
