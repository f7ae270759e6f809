"""Device side of the host mirror: Ctx, DeviceBatch, Plan.

`DeviceBatch` is the device-resident counterpart of the reference's
`GradedData` / `GradedDataMut` (src/graded.rs:43-79): one f64 array per grade,
C(n,k) rows x batch columns, batch innermost.  `Plan.eval` replaces
`SpecializedAst::eval` (src/eval.rs:12-19) for whole batches.

Everything here calls the C ABI of include/gaast_b200.h.  PyTorch is used only
as plumbing (device memory for wrapped tensors, the current stream).
"""
from __future__ import annotations

import ctypes as C
from math import comb
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

from . import _lib as L
from .expr import SpecializedAst, grade_mask, grades_of


class Ctx:
    """One device + one stream (gaast_ctx)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        out = L.vp()
        L.check(L.lib.gaast_ctx_create(int(device), L.vp(stream) if stream else None, C.byref(out)))
        self._h = out
        self.device = int(device)

    @staticmethod
    def on_torch_stream(device: int = 0) -> "Ctx":
        """A ctx launching on a torch stream that is made current, so that
        torch.cuda.Event timing and torch tensors are stream-ordered with it."""
        return _torch_stream_ctx(device)

    def sync(self):
        L.check(L.lib.gaast_ctx_sync(self._h))

    @property
    def stream(self) -> int:
        return L.lib.gaast_ctx_stream(self._h) or 0

    @property
    def launch_count(self) -> int:
        return L.lib.gaast_ctx_launch_count(self._h)

    def fp64_peak(self, seconds: float = 0.02) -> float:
        """Live FP64 FMA-pipe throughput of this device in TFLOP/s (gaast_diag_fp64_peak)."""
        out = C.c_double(0.0)
        L.check(L.lib.gaast_diag_fp64_peak(self._h, float(seconds), C.byref(out)))
        return out.value

    def close(self):
        h, self._h = self._h, None
        if h:
            L.lib.gaast_ctx_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _torch_stream_ctx(device: int) -> Ctx:
    # torch's default stream is the legacy NULL stream (handle 0), for which
    # the library would create a private stream: use a real torch stream.
    import torch
    torch.cuda.set_device(device)
    s = torch.cuda.Stream(device)
    torch.cuda.set_stream(s)
    ctx = Ctx(device, s.cuda_stream)
    ctx.torch_stream = s  # keep alive
    return ctx


def _np_dtype(dtype: int):
    return np.float32 if dtype == L.F32 else np.float64


class DeviceBatch:
    """gaast_batch: per grade k a [C(n,k)][stride] device array, f64 (the reference's type) or,
    with dtype=L.F32, binary32 (the reduced-precision variant)."""

    def __init__(self, handle, ctx: Ctx, n: int, keep=()):
        self._h = handle
        self.ctx = ctx
        self.n = n
        self._keep = keep

    @staticmethod
    def alloc(ctx: Ctx, n: int, grades: Iterable[int], length: int, broadcast: bool = False,
              dtype: int = L.F64) -> "DeviceBatch":
        out = L.vp()
        L.check(L.lib.gaast_batch_alloc_typed(ctx._h, n, grade_mask(grades), int(length), int(broadcast), int(dtype),
                                              C.byref(out)))
        return DeviceBatch(out, ctx, n)

    @staticmethod
    def wrap_torch(ctx: Ctx, n: int, tensors: Dict[int, "object"], broadcast: bool = False) -> "DeviceBatch":
        """Wrap caller-owned CUDA float64 (or, all of them, float32) tensors {grade: [C(n,k), len]} (row-major).  The
        batch's row stride is that of its multi-row tensors (a one-row grade has none of its own)."""
        grades = sorted(tensors)
        length = None
        ptrs = []
        kinds = {str(t.dtype) for t in tensors.values()}
        assert kinds <= {"torch.float64"} or kinds <= {"torch.float32"}, "one scalar type per batch"
        dtype = L.F32 if kinds == {"torch.float32"} else L.F64
        multi = [tensors[k] for k in grades if tensors[k].shape[0] > 1]
        stride = multi[0].stride(0) if multi else (tensors[grades[0]].shape[1] if grades else 0)
        for k in grades:
            t = tensors[k]
            assert t.is_cuda and t.dim() == 2 and t.shape[0] == comb(n, k)
            assert t.stride(1) == 1 or t.shape[1] == 1
            if length is None:
                length = t.shape[1]
            assert t.shape[1] == length
            if t.shape[0] > 1:
                assert t.stride(0) == stride, "all grades must share one row stride"
            ptrs.append(t.data_ptr())
        arr = (L.vp * len(ptrs))(*ptrs)
        out = L.vp()
        L.check(L.lib.gaast_batch_wrap_typed(ctx._h, n, grade_mask(grades), int(length), int(stride), int(broadcast),
                                             dtype, arr, C.byref(out)))
        return DeviceBatch(out, ctx, n, keep=tuple(tensors.values()))

    @staticmethod
    def from_host(ctx: Ctx, n: int, data: Dict[int, np.ndarray], broadcast: bool = False,
                  dtype: int = L.F64) -> "DeviceBatch":
        """Upload {grade: [C(n,k), len]} as `dtype` (a 1-D array is one broadcast element)."""
        grades = sorted(data)
        arrs = {k: np.ascontiguousarray(np.asarray(data[k], dtype=_np_dtype(dtype))) for k in grades}
        for k in grades:
            if arrs[k].ndim == 1:
                arrs[k] = arrs[k].reshape(-1, 1)
        length = arrs[grades[0]].shape[1] if grades else 0
        b = DeviceBatch.alloc(ctx, n, grades, length, broadcast, dtype)
        for k in grades:
            b.upload(k, arrs[k])
        ctx.sync()
        return b

    @staticmethod
    def alloc_sparse(ctx: Ctx, n: int, components: Dict[int, Optional[Iterable[int]]], length: int,
                     broadcast: bool = False, dtype: int = L.F64) -> "DeviceBatch":
        """An uninitialised batch in sparse per-grade storage (gaast_batch_alloc_sparse): components[grade] = the
        stored component indices, or None for a dense grade."""
        grades = sorted(components)
        bitmaps = [_bitmap(n, k, components[k]) for k in grades]
        ptrs = (C.POINTER(L.u64) * max(1, len(grades)))(*[C.cast(b, C.POINTER(L.u64)) if b is not None else None for b in bitmaps])
        out = L.vp()
        L.check(L.lib.gaast_batch_alloc_sparse(ctx._h, n, grade_mask(grades), int(length), int(broadcast), int(dtype), ptrs,
                                               C.byref(out)))
        return DeviceBatch(out, ctx, n)

    @staticmethod
    def from_host_sparse(ctx: Ctx, n: int, data: Dict[int, "tuple"], broadcast: bool = False,
                         dtype: int = L.F64) -> "DeviceBatch":
        """Sparse per-grade storage (gaast_batch_alloc_sparse): data[grade] = (stored component indices, array
        [len(indices), batch]), or a plain [C(n,k), batch] array for a dense grade.  Components that are not
        stored are zero for every element; the kernel generated for this pattern never loads or multiplies them."""
        grades = sorted(data)
        length = None
        bitmaps, arrays = [], {}
        for k in grades:
            item = data[k]
            if isinstance(item, tuple):
                idx, arr = item
                arr = np.ascontiguousarray(np.asarray(arr, dtype=_np_dtype(dtype)))
                idx = [int(i) for i in idx]
                assert list(idx) == sorted(set(idx)) and arr.shape[0] == len(idx) and all(0 <= i < comb(n, k) for i in idx)
                words = (comb(n, k) + 63) // 64
                bits = (L.u64 * words)()
                for i in idx:
                    bits[i // 64] |= 1 << (i % 64)
                bitmaps.append(bits)
            else:
                arr = np.ascontiguousarray(np.asarray(item, dtype=_np_dtype(dtype)))
                bitmaps.append(None)
            arrays[k] = arr
            length = arr.shape[1] if length is None else length
            assert arr.shape[1] == length
        ptrs = (C.POINTER(L.u64) * max(1, len(grades)))(*[C.cast(b, C.POINTER(L.u64)) if b is not None else None for b in bitmaps])
        out = L.vp()
        L.check(L.lib.gaast_batch_alloc_sparse(ctx._h, n, grade_mask(grades), int(length or 0), int(broadcast), int(dtype), ptrs,
                                               C.byref(out)))
        b = DeviceBatch(out, ctx, n, keep=tuple(bitmaps))
        for k in grades:
            if arrays[k].shape[0]:
                b.upload(k, arrays[k])
        ctx.sync()
        return b

    @staticmethod
    def from_records(ctx: Ctx, n: int, grades: Iterable[int], records, record_grades: Optional[Iterable[int]] = None,
                     broadcast: bool = False, dtype: int = L.F64) -> "DeviceBatch":
        """A batch of `grades` from element-major records (len, K_rec): one multivector per row, the components of
        `record_grades` (default: `grades`) in slot order.  A numpy array goes through the host path, a contiguous
        CUDA torch tensor through the device path; either must already have the batch's scalar type."""
        grades = list(grades)
        b = DeviceBatch.alloc(ctx, n, grades, int(records.shape[0]), broadcast, dtype)
        b.pack_records(records, 0, grades if record_grades is None else record_grades)
        return b

    def _record_mask(self, records, record_grades) -> int:
        mask = grade_mask(self.grade_set() if record_grades is None else record_grades)
        width = sum(comb(self.n, k) for k in grades_of(mask))
        assert records.ndim == 2 and records.shape[1] == width, f"records must be (count, {width})"
        assert str(records.dtype).endswith("float32" if self.dtype == L.F32 else "float64"), "records have another dtype"
        return mask

    def pack_records(self, records, first: int = 0, record_grades: Optional[Iterable[int]] = None):
        """Batch columns [first, first + len(records)) from records (gaast_batch_upload_records for a numpy array,
        which returns when the copy is done; gaast_batch_pack_records, stream-ordered, for a CUDA tensor)."""
        mask = self._record_mask(records, record_grades)
        if isinstance(records, np.ndarray):
            records = np.ascontiguousarray(records)
            L.check(L.lib.gaast_batch_upload_records(self._h, int(first), records.shape[0], records.ctypes.data_as(L.vp), mask))
            self.ctx.sync()  # `records` may be a temporary
        else:
            assert records.is_cuda and records.is_contiguous(), "device records must be a contiguous CUDA tensor"
            L.check(L.lib.gaast_batch_pack_records(self._h, int(first), int(records.shape[0]), L.vp(records.data_ptr()), mask))

    def to_records(self, record_grades: Optional[Iterable[int]] = None, out=None):
        """The whole batch as records (length, K_rec) of `record_grades` (default: the batch's grades); components
        the batch does not store are +0.  Returns a numpy array, or fills the contiguous CUDA tensor `out`
        (stream-ordered) and returns it."""
        if out is None:
            width = sum(comb(self.n, k) for k in (self.grade_set() if record_grades is None else record_grades))
            arr = np.empty((self.length, width), dtype=_np_dtype(self.dtype))
            mask = self._record_mask(arr, record_grades)
            L.check(L.lib.gaast_batch_download_records(self._h, 0, self.length, arr.ctypes.data_as(L.vp), mask))
            self.ctx.sync()
            return arr
        mask = self._record_mask(out, record_grades)
        assert out.is_cuda and out.is_contiguous() and out.shape[0] == self.length
        L.check(L.lib.gaast_batch_unpack_records(self._h, 0, self.length, L.vp(out.data_ptr()), mask))
        return out

    def segment_sum(self, offsets, out=None):
        """Per-segment sums of the stored rows (gaast_batch_segment_sum): segment j is columns [offsets[j], offsets[j+1]).
        `offsets` is a CUDA int64 tensor of n_segments + 1 values on the batch's device.  Returns, or fills, a CUDA
        float64 tensor [n_segments, S] (S = the stored rows, grades ascending); stream-ordered on the ctx stream.
        Offsets that are not non-decreasing within [0, length] give NaN everywhere."""
        import torch
        assert offsets.is_cuda and offsets.dtype == torch.int64 and offsets.dim() == 1 and offsets.is_contiguous(), \
            "offsets must be a contiguous 1-D CUDA int64 tensor"
        n_seg = max(0, offsets.shape[0] - 1)
        S = sum(self.stored_rows(k) for k in self.grade_set())
        if out is None:
            out = torch.empty((n_seg, S), dtype=torch.float64, device=offsets.device)
        assert out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (n_seg, S)
        L.check(L.lib.gaast_batch_segment_sum(self._h, L.vp(offsets.data_ptr()), n_seg, L.vp(out.data_ptr())))
        return out

    def stored_rows(self, k: int) -> int:
        return L.lib.gaast_batch_stored_rows(self._h, k)

    @property
    def length(self) -> int:
        return L.lib.gaast_batch_len(self._h)

    @property
    def stride(self) -> int:
        return L.lib.gaast_batch_stride(self._h)

    @property
    def dtype(self) -> int:
        return L.lib.gaast_batch_dtype(self._h)

    def grade_set(self) -> List[int]:  # Graded::grade_set, graded.rs:20-30
        return grades_of(L.lib.gaast_batch_grade_mask(self._h))

    def grade_ptr(self, k: int) -> int:  # GradedData::grade_slice, graded.rs:46
        return L.lib.gaast_batch_grade_ptr(self._h, k) or 0

    def upload(self, k: int, host: np.ndarray):
        f32 = self.dtype == L.F32
        host = np.ascontiguousarray(host, dtype=_np_dtype(self.dtype))
        assert host.ndim == 2 and host.shape[0] == self.stored_rows(k)
        fn = L.lib.gaast_batch_upload_f32 if f32 else L.lib.gaast_batch_upload
        L.check(fn(self._h, k, host.ctypes.data_as(L.vp), host.shape[1]))
        self.ctx.sync()  # `host` may be a temporary

    def download(self, k: int) -> np.ndarray:
        f32 = self.dtype == L.F32
        out = np.empty((self.stored_rows(k), self.length), dtype=_np_dtype(self.dtype))
        fn = L.lib.gaast_batch_download_f32 if f32 else L.lib.gaast_batch_download
        L.check(fn(self._h, k, out.ctypes.data_as(L.vp), out.shape[1]))
        self.ctx.sync()
        return out

    def to_host(self) -> Dict[int, np.ndarray]:
        return {k: self.download(k) for k in self.grade_set()}

    def zero(self):  # GradedDataMut::init_null_mv, graded.rs:55
        L.check(L.lib.gaast_batch_zero(self._h))

    def free(self):
        h, self._h = self._h, None
        if h:
            L.lib.gaast_batch_free(h)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Plan:
    """gaast_plan: a lowered SpecializedAst, reusable with new inputs.

    `components` = {root grade: [component indices]} makes a projected plan (gaast_plan_create_projected): only those
    components of the listed grades are stored, a grade that is not listed is kept whole, and the result is a sparse
    output batch (`alloc_output` allocates the matching one)."""

    def __init__(self, ctx: Optional[Ctx], ast: SpecializedAst, components: Optional[Dict[int, Iterable[int]]] = None):
        self.ctx = ctx
        self.ast = ast  # owns the plan description
        out = L.vp()
        self.components = None
        if components is None:
            L.check(L.lib.gaast_plan_create(ctx._h if ctx else None, ast.lower(), C.byref(out)))
        else:
            desc = ast.lower()
            n, grades = desc.contents.n, grades_of(desc.contents.buffer_masks[0])
            assert set(components) <= set(grades), "components of a grade the root does not have"
            self.components = {k: (sorted(int(i) for i in components[k]) if k in components else None) for k in grades}
            bitmaps = [_bitmap(n, k, self.components[k]) for k in grades]
            ptrs = (C.POINTER(L.u64) * max(1, len(grades)))(*[C.cast(b, C.POINTER(L.u64)) if b is not None else None
                                                               for b in bitmaps])
            L.check(L.lib.gaast_plan_create_projected(ctx._h if ctx else None, desc, ptrs, C.byref(out)))
        self._h = out
        self.n = L.lib.gaast_plan_dim(out)

    def root_grades(self) -> List[int]:
        return grades_of(L.lib.gaast_plan_root_mask(self._h))

    def num_slots(self) -> int:
        return L.lib.gaast_plan_num_slots(self._h)

    def slot_grades(self, slot: int) -> List[int]:
        return grades_of(L.lib.gaast_plan_slot_mask(self._h, slot))

    def cost(self, broadcast_slots: int = 0):
        b, f = L.u64(), L.u64()
        L.check(L.lib.gaast_plan_cost(self._h, broadcast_slots, C.byref(b), C.byref(f)))
        return b.value, f.value

    def set_tuning(self, elems_per_thread: int = 0, variant: int = 0):
        L.check(L.lib.gaast_plan_set_tuning(self._h, elems_per_thread, variant))

    def kernel_source(self, broadcast_slots: int = 0, arith: int = L.ARITH_FMA, with_sum: bool = False,
                      store_out: bool = True, dtype: int = L.F64, present: Optional[Dict] = None) -> str:
        """`present` = {(slot, grade): stored component indices} for inputs in sparse per-grade storage."""
        flags = int(bool(with_sum)) | (0 if store_out else 2) | (4 if dtype == L.F32 else 0)  # GAAST_SRC_*
        if present:
            keys = [(s, k) for s in range(self.num_slots()) for k in self.slot_grades(s)]
            maps = []
            for s, k in keys:
                if (s, k) not in present:
                    maps.append(None)
                    continue
                bits = (L.u64 * ((comb(self.n, k) + 63) // 64))()
                for i in present[(s, k)]:
                    bits[int(i) // 64] |= 1 << (int(i) % 64)
                maps.append(bits)
            ptrs = (C.POINTER(L.u64) * max(1, len(keys)))(*[C.cast(b, C.POINTER(L.u64)) if b is not None else None for b in maps])
            call = lambda buf, cap: L.lib.gaast_plan_kernel_source_sparse(self._h, broadcast_slots, arith, flags, ptrs,  # noqa: E731
                                                                          len(keys), buf, cap)
        else:
            call = lambda buf, cap: L.lib.gaast_plan_kernel_source(self._h, broadcast_slots, arith, flags, buf, cap)  # noqa: E731
        n = call(None, 0)
        if n == 0:
            raise L.GaastError(L.ERR_JIT, L.last_error())
        buf = C.create_string_buffer(n + 1)
        call(buf, n + 1)
        return buf.value.decode()

    def precompile(self, broadcast_slots: int = 0, arith: int = L.ARITH_FMA, with_sum: bool = False,
                   store_out: bool = True, dtype: int = L.F64) -> str:
        L.check(L.lib.gaast_plan_precompile_typed(self._h, broadcast_slots, arith, int(with_sum), int(store_out),
                                                  int(dtype)))
        return self.last_kernel()

    def last_kernel(self) -> str:
        return (L.lib.gaast_plan_last_kernel(self._h) or b"").decode()

    def alloc_output(self, length: int, dtype: int = L.F64) -> DeviceBatch:
        """The output batch `eval` writes: dense, or for a projected plan sparse in the plan's components."""
        if self.components is not None:
            return DeviceBatch.alloc_sparse(self.ctx, self.n, self.components, length, dtype=dtype)
        return DeviceBatch.alloc(self.ctx, self.n, self.root_grades(), length, dtype=dtype)

    def eval(self, inputs: Sequence[DeviceBatch], out: Optional[DeviceBatch] = None, engine: int = L.ENGINE_AUTO,
             arith: int = L.ARITH_FMA) -> DeviceBatch:
        """out[i] = expr(inputs[0][i], inputs[1][i], ...); stream-ordered."""
        if self.ctx is None:
            raise L.GaastError(L.ERR_NO_DEVICE, "offline plan (created without a ctx): there is no CPU evaluation path")
        if out is None:
            length = next((b.length for b in inputs if not _is_broadcast(b)), 1)
            out = self.alloc_output(length, inputs[0].dtype if inputs else L.F64)
        arr = (L.vp * max(1, len(inputs)))(*[b._h for b in inputs])
        L.check(L.lib.gaast_eval(self._h, arr, len(inputs), out._h, engine, arith))
        return out

    def eval_sum(self, inputs: Sequence[DeviceBatch], dev_sum_ptr: int, out: Optional[DeviceBatch] = None,
                 engine: int = L.ENGINE_AUTO, arith: int = L.ARITH_FMA):
        """Writes sum_i out[i] to `dev_sum_ptr` (device memory): one double per root component, or for a projected
        plan one per stored component (grades ascending, stored components ascending).  `out` may be None."""
        arr = (L.vp * max(1, len(inputs)))(*[b._h for b in inputs])
        L.check(L.lib.gaast_eval_sum(self._h, arr, len(inputs), out._h if out else None, L.vp(dev_sum_ptr), engine,
                                     arith))

    def eval_host(self, host_in: Sequence[np.ndarray], in_grades: Sequence[Iterable[int]],
                  in_broadcast: Sequence[bool], length: int, host_out: np.ndarray, host_stride: Optional[int] = None,
                  engine: int = L.ENGINE_AUTO, arith: int = L.ARITH_FMA):
        """Host arrays in / out (see gaast_eval_host).  Arrays are [rows][host_stride] float64, or all
        float32 (gaast_eval_host_f32)."""
        n_in = len(host_in)
        ptrs = (L.vp * max(1, n_in))(*[_host_ptr(a) for a in host_in])
        masks = (L.u32 * max(1, n_in))(*[grade_mask(g) for g in in_grades])
        bc = (C.c_int * max(1, n_in))(*[int(bool(x)) for x in in_broadcast])
        stride = int(host_stride if host_stride is not None else length)
        f32 = str(getattr(host_out, "dtype", "")).endswith("float32")  # numpy or torch, all arrays of one type
        fn = L.lib.gaast_eval_host_f32 if f32 else L.lib.gaast_eval_host
        L.check(fn(self._h, ptrs, masks, bc, n_in, int(length), stride, L.vp(_host_ptr(host_out)), engine, arith))

    def free(self):
        h, self._h = self._h, None
        if h:
            L.lib.gaast_plan_destroy(h)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Comm:
    """gaast_comm: the all-reduce of batch-sum vectors across the GPUs of one node, behind the C ABI: the library's
    own kernel over NVLink peer memory (`transport == "peer"`), NCCL as the fallback.  `Comm(ctxs)` = one process
    driving several devices; `Comm.join(ctx, n, rank, id)` = one process per device, `Comm.unique_id()` drawn on
    rank 0 and shipped by the caller."""

    def __init__(self, ctxs: Sequence[Ctx], _handle=None):
        self.ctxs = list(ctxs)
        if _handle is None:
            arr = (L.vp * len(self.ctxs))(*[c._h for c in self.ctxs])
            out = L.vp()
            L.check(L.lib.gaast_comm_create(arr, len(self.ctxs), C.byref(out)))
            _handle = out
        self._h = _handle

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        L.check(L.lib.gaast_comm_unique_id(buf))
        return buf.raw

    @staticmethod
    def join(ctx: Ctx, n_ranks: int, rank: int, uid: bytes) -> "Comm":
        out = L.vp()
        L.check(L.lib.gaast_comm_create_rank(ctx._h, int(n_ranks), int(rank), uid, C.byref(out)))
        return Comm([ctx], _handle=out)

    @property
    def size(self) -> int:
        return L.lib.gaast_comm_size(self._h)

    @property
    def transport(self) -> str:
        """"peer" or "nccl" (gaast_comm_transport)."""
        return (L.lib.gaast_comm_transport(self._h) or b"").decode()

    def set_transport(self, transport: int):
        """L.COMM_AUTO / COMM_NCCL / COMM_PEER; every rank must make the same call."""
        L.check(L.lib.gaast_comm_set_transport(self._h, int(transport)))

    def allreduce_sum(self, dev_ptrs: Sequence[int], count: int):
        """In place on every local device: dev_ptrs[i] -> `count` doubles on self.ctxs[i]'s device."""
        assert len(dev_ptrs) == len(self.ctxs)
        arr = (L.vp * len(dev_ptrs))(*[L.vp(p) for p in dev_ptrs])
        L.check(L.lib.gaast_comm_allreduce_sum(self._h, arr, int(count)))

    def close(self):
        h, self._h = self._h, None
        if h:
            L.lib.gaast_comm_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostArray:
    """A page-locked [rows][cols] host array for the host-array entry points (gaast_host_alloc): `.array` is a numpy
    view of it.  `write_combined=True` is for arrays the host only fills (inputs of gaast_eval_host)."""

    def __init__(self, rows: int, cols: int, dtype=np.float64, write_combined: bool = False):
        self.dtype = np.dtype(dtype)
        self.nbytes = int(rows) * int(cols) * self.dtype.itemsize
        out = L.vp()
        L.check(L.lib.gaast_host_alloc(self.nbytes, L.HOST_WRITE_COMBINED if write_combined else L.HOST_DEFAULT, C.byref(out)))
        self._p = out
        buf = (C.c_char * self.nbytes).from_address(out.value)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(int(rows), int(cols))

    def free(self):
        p, self._p = self._p, None
        if p:
            self.array = None
            L.lib.gaast_host_free(p)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pin_host(a: np.ndarray):
    """Pins an existing numpy array in place (gaast_host_register); returns a callable that unpins it."""
    L.check(L.lib.gaast_host_register(L.vp(a.ctypes.data), a.nbytes))
    return lambda: L.check(L.lib.gaast_host_unregister(L.vp(a.ctypes.data)))


def _bitmap(n: int, k: int, idx: Optional[Iterable[int]]):
    """gaast_batch_alloc_sparse's presence bitmap of grade k (None = the whole grade)."""
    if idx is None:
        return None
    bits = (L.u64 * ((comb(n, k) + 63) // 64))()
    for i in idx:
        assert 0 <= int(i) < comb(n, k), f"component {i} outside grade {k}"
        bits[int(i) // 64] |= 1 << (int(i) % 64)
    return bits


def _is_broadcast(b: DeviceBatch) -> bool:
    return False if b.length != 1 else True


def _host_ptr(a) -> int:
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return int(a)
