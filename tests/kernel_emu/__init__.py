"""TEST INFRASTRUCTURE: run a GENERATED kernel on the CPU.

`gaast_plan_kernel_source` returns the CUDA source the specialised engine compiles with NVRTC for a plan (an offline
plan needs no GPU).  `run_generated_kernel` compiles exactly that text with g++ -- behind `cuda_on_cpu.h`, a host
stand-in for threads, barriers, shared memory, mbarrier/TMA and tensor memory; only the prelude's inline-PTX helper
definitions are cut out, the shim supplies them -- and executes the grid thread by thread on numpy arrays laid out like
device batches.  What comes out is what the code generator printed, evaluated with IEEE arithmetic: the CPU suite can
hold the generator (term order, sign folding, the lowerings, strict arithmetic) to the oracle without a GPU.
It says nothing about NVRTC, ptxas or the hardware; tests/test_gpu_*.py do that on the device.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import re
import subprocess
import tempfile
import threading
from math import comb
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

import gaast_b200 as g
from gaast_b200 import _lib as L
from tests.guarded_layout import BITS, poison, sentinel

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_STREAMS = 96


class EmuLaunch(C.Structure):
    _fields_ = [("sptr", C.c_void_p * MAX_STREAMS), ("srow", C.c_longlong * MAX_STREAMS),
                ("bcast", C.c_ulonglong * 2), ("n", C.c_longlong), ("consts", C.c_void_p), ("uniform", C.c_void_p),
                ("partials", C.c_void_p), ("n_sum_cols", C.c_int), ("total_cols", C.c_int), ("root_col", C.c_int),
                ("store_out", C.c_int), ("grid", C.c_int), ("threaded", C.c_int), ("which", C.c_int)]


def _strip_strings(line: str) -> str:
    """The line without the contents of its string literals (braces inside PTX text do not nest C++ scopes)."""
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', line)


def host_source(cuda_src: str) -> str:
    """The generated source with the inline-PTX helper definitions of the prelude removed (cuda_on_cpu.h has host
    versions under the same names) and shared-memory declarations turned into host ones.  Everything else -- the
    kernels themselves in particular -- is kept character for character."""
    lines = cuda_src.split("\n")
    out: List[str] = []
    i = 0
    while i < len(lines):
        ln = lines[i]
        starts_def = ln.startswith("__device__ __forceinline__") or ln.startswith("template <")
        if starts_def:
            depth, seen, j = 0, False, i
            while j < len(lines):
                s = _strip_strings(lines[j])
                depth += s.count("{") - s.count("}")
                seen = seen or "{" in s
                if seen and depth == 0:
                    break
                j += 1
            block = lines[i:j + 1]
            text = "\n".join(block)
            if "__global__" not in text and re.search(r'asm volatile\(\s*"[^"]', text):  # a PTX helper: the shim has it
                i = j + 1
                continue
            out.extend(block)
            i = j + 1
            continue
        if ln.startswith("#define GAAST_TM_ACC("):  # the tcgen05.ld/st accumulate macro (PTX inside) ...
            while lines[i].rstrip().endswith("\\"):
                i += 1
            i += 1
            continue
        if ln.startswith("GAAST_TM_ACC("):  # ... and its three instantiations
            depth = 0
            while True:
                s = _strip_strings(lines[i])
                depth += s.count("(") - s.count(")")
                i += 1
                if depth == 0:
                    break
            continue
        out.append(ln)
        i += 1
    src = "\n".join(out)
    src = src.replace("extern __shared__", "extern")
    src = re.sub(r"\b__shared__\b", "static", src)
    return src


# -O0: straight-line kernels of thousands of statements compile in about a second (the batches are tiny, run time does
# not matter); -ffp-contract=off: the compiler never fuses a*b+c on its own (strict arithmetic is two roundings; an FMA
# is spelled fma() in the source and is correctly rounded whether it becomes an instruction or a libm call)
FLAGS = ["-std=c++17", "-O0", "-ffp-contract=off", "-mfma", "-fPIC", "-pthread", "-w"]
# GAAST_EMU_ASAN=1 (with LD_PRELOAD=libasan.so libstdc++.so.6): the kernels run under AddressSanitizer on batches whose
# rows are padded exactly as the library pads them (128 bytes) -- an access outside a batch or outside shared memory
# aborts the run
ASAN = os.environ.get("GAAST_EMU_ASAN") == "1"
if ASAN:
    FLAGS += ["-fsanitize=address", "-fno-omit-frame-pointer", "-g"]
_cache: Dict[str, C.CDLL] = {}
_tmp = None
_locks: Dict[str, threading.Lock] = {}
_locks_guard = threading.Lock()


def _build_lock(key: str) -> threading.Lock:
    with _locks_guard:
        return _locks.setdefault(key, threading.Lock())


def _ensure_tmp():
    global _tmp
    if _tmp is None:
        # one precompiled header of the shim per session: the standard headers cost more than most kernels
        _tmp = tempfile.TemporaryDirectory(prefix="gaast_kernel_emu_")
        for name in ("cuda_on_cpu.h", "driver.inc"):
            with open(os.path.join(HERE, name)) as f, open(os.path.join(_tmp.name, name), "w") as o:
                o.write(f.read())
        r = subprocess.run(["g++", *FLAGS, "-x", "c++-header", os.path.join(_tmp.name, "cuda_on_cpu.h"), "-o",
                            os.path.join(_tmp.name, "cuda_on_cpu.h.gch")], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ rejected cuda_on_cpu.h:\n" + r.stderr[-3000:])


def _compile(cuda_src: str, f32: bool = False) -> C.CDLL:
    global _tmp
    body = host_source(cuda_src)
    key = hashlib.sha256((body + str(f32)).encode()).hexdigest()[:24]  # (of the text that is compiled: dlopen caches by path)
    if key in _cache:
        return _cache[key]
    _ensure_tmp()
    has_uniform = 'void __launch_bounds__(32) gaast_uniform(' in cuda_src
    text = ('#include "cuda_on_cpu.h"\n' + ("#define EMU_HAS_UNIFORM 1\n" if has_uniform else "") + body +
            '\n#include "driver.inc"\n')
    so = os.path.join(_tmp.name, key + ".so")
    with _build_lock(key):  # (two threads asking for the same text: one build, the other finds the library)
        if key in _cache:
            return _cache[key]
        if not os.path.exists(so):
            cpp = os.path.join(_tmp.name, key + ".cpp")
            with open(cpp, "w") as f:
                f.write(text)
            # (the f32 variant defines GAAST_EMU_F32: the precompiled header does not apply, g++ reads the header itself)
            part = so + f".{threading.get_ident()}.part"
            cmd = ["g++", *FLAGS, *(["-DGAAST_EMU_F32"] if f32 else []), "-shared", "-I", _tmp.name, cpp, "-o", part]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("g++ rejected the generated kernel:\n" + r.stderr[-3000:])
            os.replace(part, so)
        lib = C.CDLL(so)
        lib.emu_launch.argtypes = [C.POINTER(EmuLaunch)]
        lib.emu_launch.restype = C.c_int
        _cache[key] = lib
        return lib


def prefetch(ast, broadcast, variants, tuning=None):
    """Compile the kernels of several (arith, with_sum, store_out, dtype) variants of one plan side by side (g++ is the
    cost of a test here, and the box has more than one core); run_generated_kernel then finds them in the cache."""
    from concurrent.futures import ThreadPoolExecutor
    plan = g.Plan(None, ast)
    if tuning is not None:
        plan.set_tuning(*tuning)
    bmask = sum(1 << s for s in range(plan.num_slots()) if broadcast[s])
    jobs = []
    for arith, with_sum, store_out, dtype in variants:
        f32 = dtype == np.float32
        jobs.append((plan.kernel_source(broadcast_slots=bmask, arith=arith, with_sum=with_sum, store_out=store_out,
                                        dtype=L.F32 if f32 else L.F64), f32))
    _ensure_tmp()  # (the precompiled header first)
    jobs = list(dict.fromkeys(jobs))  # (two variants may print the same text: one build each)
    with ThreadPoolExecutor(max_workers=4) as ex:
        list(ex.map(lambda j: _compile(*j), jobs))


def prefetch_many(cases, workers: int = 6):
    """cases: iterable of (ast, broadcast flags, arith, dtype[, with_sum[, tuning]]).  Compiles their kernels side by
    side; a plan the generator refuses is left for the test to report."""
    from concurrent.futures import ThreadPoolExecutor
    jobs = []
    for case in cases:
        ast, broadcast, arith, dtype = case[:4]
        with_sum = case[4] if len(case) > 4 else False
        plan = g.Plan(None, ast)
        if len(case) > 5 and case[5] is not None:
            plan.set_tuning(*case[5])
        bmask = sum(1 << s for s in range(plan.num_slots()) if broadcast[s])
        f32 = dtype == np.float32
        try:
            jobs.append((plan.kernel_source(broadcast_slots=bmask, arith=arith, with_sum=with_sum,
                                            dtype=L.F32 if f32 else L.F64), f32))
        except L.GaastError:
            pass
    _ensure_tmp()
    jobs = list(dict.fromkeys(jobs))  # (two tuning variants may print the same text: one build each)
    with ThreadPoolExecutor(max_workers=workers) as ex:
        list(ex.map(lambda j: _compile(*j), jobs))


def needs_threads(cuda_src: str) -> bool:
    body = cuda_src[cuda_src.index('extern "C" __global__'):]
    return bool(re.search(r"__syncthreads|mbar_wait|__shfl_xor_sync", body))


FAULTS = {1: "a barrier / shuffle in sequential mode", 2: "a bulk copy that is not a multiple of 16 bytes",
          3: "an mbarrier phase that never completes", 4: "a tensor-memory allocation the hardware would refuse",
          5: "a tensor-memory access outside the warp's lanes / the 512 columns"}


def run_generated_kernel(ast, inputs: Sequence[Dict[int, np.ndarray]], broadcast: Sequence[bool], batch: int,
                         arith: int = L.ARITH_FMA, with_sum: bool = False, tuning: Optional[Tuple[int, int]] = None,
                         grid: Optional[int] = None, store_out: bool = True, dtype=np.float64,
                         present: Optional[Dict] = None, components: Optional[Dict[int, Sequence[int]]] = None):
    """Evaluate the specialised engine's kernel for `ast` (a gaast_b200.expr.SpecializedAst) on host arrays.
    inputs[slot] = {grade: (C(n,k), batch) array, or (C(n,k), 1) for a broadcast slot}.
    present = {(slot, grade): stored component indices} for inputs in sparse per-grade storage: that grade's array
    then holds the stored rows only, in component order.
    components = {root grade: stored component indices} makes the plan a projected one (gaast_plan_create_projected; a
    grade that is not listed is kept whole): out[k] and sums[k] then hold the stored components of grade k only, in
    component order.
    Returns (out: {grade: (C, batch)}, sums or None, info) where info = {"notes", "threads", "ept", "grid", "source"}."""
    plan = g.Plan(None, ast, components=components)
    if tuning is not None:
        plan.set_tuning(*tuning)
    n = plan.n
    root_rows = {k: len(set(components[k])) if components and k in components else comb(n, k) for k in plan.root_grades()}
    slots = plan.num_slots()
    bmask = sum(1 << s for s in range(slots) if broadcast[s])
    f32 = dtype == np.float32
    src = plan.kernel_source(broadcast_slots=bmask, arith=arith, with_sum=with_sum, store_out=store_out,
                             dtype=L.F32 if f32 else L.F64, present=present)
    lib = _compile(src, f32)
    threads, ept = lib.emu_threads(), lib.emu_elems_per_thread()
    per_block = threads * ept
    padded = (batch + per_block - 1) // per_block * per_block  # (generous: a whole block's worth)
    if ASAN:
        padded = (batch + 15) // 16 * 16  # rows on 128-byte boundaries: gaast_batch_alloc's layout, nothing more
    launch = EmuLaunch()
    keep = []
    si = 0
    for s in range(slots):
        for k in plan.slot_grades(s):
            rows = len(present[(s, k)]) if present and (s, k) in present else comb(n, k)
            src_arr = np.asarray(inputs[s][k], dtype=dtype)
            # the padding holds the input sentinel: it is never part of a result
            if broadcast[s]:
                arr = poison(np.empty((rows, 4), dtype=dtype), "in")
                arr[:, 0] = src_arr.reshape(rows, -1)[:, 0]
                launch.bcast[si >> 6] |= 1 << (si & 63)
            else:
                assert src_arr.shape == (rows, batch), (src_arr.shape, rows, batch)
                arr = poison(np.empty((rows, padded), dtype=dtype), "in")
                arr[:, :batch] = src_arr
            keep.append(arr)
            launch.sptr[si] = arr.ctypes.data
            launch.srow[si] = arr.shape[1]
            si += 1
    outs = {}
    for k in plan.root_grades():
        arr = poison(np.empty((max(1, root_rows[k]), padded), dtype=dtype), "out")[:root_rows[k]]  # (an emptied grade: no rows)
        outs[k] = arr
        launch.sptr[si] = arr.ctypes.data
        launch.srow[si] = padded
        si += 1
    assert si <= MAX_STREAMS
    desc = ast.lower().contents
    consts = np.array([desc.const_values[i] for i in range(desc.n_const_values)] + [0.0], dtype=np.float64)
    uniform = np.full(1 << 16, np.nan)
    root_cols = sum(root_rows.values())
    threaded = needs_threads(src)
    if grid is None:
        grid = max(1, (batch + per_block - 1) // per_block)
    partials = np.full((grid + 1, max(1, root_cols)), np.nan)
    # gaast_eval's contract for the kernel `kernel_source` returns (the ALIGNED variant, csrc/device/runtime.cu): rows on
    # 16-byte boundaries and an even element count -- an odd batch into a library-owned output is launched over its
    # padding column too; with a batch-sum the runtime switches to the one-element-per-thread variant instead
    quantum = 4 if f32 else 2  # elements per 16 bytes
    launch_n = (batch + quantum - 1) // quantum * quantum
    if with_sum:
        assert batch % max(quantum, ept) == 0, "emulated batch-sum: use an aligned batch (the padding must not reach the sums)"
    launch.n = launch_n
    launch.consts = consts.ctypes.data
    launch.uniform = uniform.ctypes.data
    launch.partials = partials.ctypes.data
    launch.n_sum_cols = root_cols
    launch.store_out = int(store_out)
    launch.grid = grid
    launch.threaded = int(threaded)
    if "gaast_uniform(" in src:
        launch.which = 1
        rc = lib.emu_launch(C.byref(launch))
        assert rc == 0, f"uniform prologue: {FAULTS.get(rc, rc)}"
    launch.which = 0
    rc = lib.emu_launch(C.byref(launch))
    assert rc == 0, f"generated kernel: {FAULTS.get(rc, rc)}"
    # write containment: the aligned kernel may store into the padding columns it was launched over, and nowhere else
    for k, v in outs.items():
        stray = np.argwhere(v[:, launch_n:].view(BITS[v.dtype]) != sentinel(v.dtype, "out"))
        assert not len(stray), (f"generated kernel: {len(stray)} store(s) beyond the launch length {launch_n}; first: grade "
                                f"{k} row {stray[0][0]} column {launch_n + stray[0][1]}")
    out = {k: v[:, :batch].copy() for k, v in outs.items()}
    sums = None
    if with_sum:
        sums, c = {}, 0
        tot = partials[:grid].sum(axis=0)
        for k in plan.root_grades():
            sums[k] = tot[c:c + root_rows[k]]
            c += root_rows[k]
    info = {"notes": src.split("\n")[1], "threads": threads, "ept": ept, "grid": grid, "threaded": threaded,
            "source": src}
    return out, sums, info
