"""TEST INFRASTRUCTURE: the CPU runs of tests/kernel_emu for f32 batches evaluated in binary64 (GAAST_ARITH_F64).

tests/kernel_emu runs the f32 variant with binary32 everywhere: its generated kernels are compiled with the binary32
staging helpers (GAAST_EMU_F32), and its table-engine library instantiates `table_engine_kernel<float, ...>`.  In this
mode a generated kernel parks binary64 values (the f64 staging helpers) and rounds its stores with
`__double2float_rn`, and the table engine reads binary32 batches into a binary64 workspace
(`table_engine_kernel<double, ..., float>`).  The wrappers below run the same harness with exactly those differences:
  * run_wide_kernel / prefetch_wide: kernel_emu's own runs, with a kernel of this mode (its header says `arith=f64`)
    compiled without GAAST_EMU_F32 and with a host `__double2float_rn` (the host's conversion rounds to nearest even);
  * run_wide_table_engine: kernel_emu.table_engine's run on a library whose driver instantiates the binary32-batch
    cases as `table_engine_kernel<double, ..., float>` (the driver's text, with that one substitution)."""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import subprocess
import tempfile
import threading

import numpy as np

from tests import kernel_emu as KE
from tests.kernel_emu import table_engine as TE

_D2F = "static inline float __double2float_rn(double a) { return float(a); }\n"
_lock = threading.Lock()


def _is_wide(cuda_src: str) -> bool:
    return " arith=f64" in cuda_src.split("\n", 1)[0]


@contextlib.contextmanager
def _wide_kernels():
    plain = KE._compile

    def compile_(cuda_src, f32=False):
        return plain(_D2F + cuda_src, False) if _is_wide(cuda_src) else plain(cuda_src, f32)

    with _lock:
        KE._compile = compile_
        try:
            yield
        finally:
            KE._compile = plain


def run_wide_kernel(*args, **kw):
    """kernel_emu.run_generated_kernel for a kernel of this mode (arith carries GAAST_ARITH_F64, dtype=np.float32)."""
    with _wide_kernels():
        return KE.run_generated_kernel(*args, **kw)


def prefetch_wide(cases, workers: int = 6):
    with _wide_kernels():
        KE.prefetch_many(cases, workers)


_table_lib = None
_table_tmp = None


def _wide_table_library() -> C.CDLL:
    global _table_lib, _table_tmp
    if _table_lib is not None:
        return _table_lib
    _table_tmp = tempfile.TemporaryDirectory(prefix="gaast_table_wide_emu_")
    driver = open(os.path.join(KE.HERE, "table_driver.inc")).read()
    kernel, esize = "table_engine_kernel<T, S, U, G>", "const size_t esize = L->f32 ? 4 : 8;"
    assert kernel in driver and esize in driver, "tests/kernel_emu/table_driver.inc instantiates the kernel differently now"
    # a binary32 batch (T = float in the driver's cases) is evaluated with a binary64 workspace
    driver = driver.replace(kernel, "table_engine_kernel<double, S, U, G, T>").replace(esize, "const size_t esize = 8;")
    with open(os.path.join(_table_tmp.name, "table_driver_wide.inc"), "w") as f:
        f.write(driver)
    cpp = os.path.join(_table_tmp.name, "table_engine_wide_emu.cpp")
    with open(cpp, "w") as f:
        f.write('#include "cuda_on_cpu.h"\n#include <cstdio>\n#include "device_plan.hpp"\nusing std::min;\n'
                "namespace gaast {\n" + TE.kernel_text() + "\n}  // namespace gaast\n" + '#include "table_driver_wide.inc"\n')
    so = os.path.join(_table_tmp.name, "table_engine_wide_emu.so")
    cmd = ["g++", *[x for x in KE.FLAGS if x != "-O0"], "-O1", "-shared", "-I", _table_tmp.name, "-I", KE.HERE, "-I", TE.CSRC,
           "-I", os.path.join(TE.ROOT, "include"), cpp, os.path.join(TE.CSRC, "device_plan.cpp"),
           os.path.join(TE.CSRC, "common.cpp"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ rejected the table engine:\n" + r.stderr[-4000:])
    lib = C.CDLL(so)
    lib.emu_table_launch.argtypes = [C.POINTER(TE.TableLaunchEmu)]
    lib.emu_table_launch.restype = C.c_int
    _table_lib = lib
    return lib


def run_wide_table_engine(ast, inputs, broadcast, batch, **kw):
    """kernel_emu.table_engine.run_table_engine on binary32 batches evaluated in binary64."""
    lib = _wide_table_library()
    with _lock:
        plain = TE._library
        TE._library = lambda: lib
        try:
            return TE.run_table_engine(ast, inputs, broadcast, batch, dtype=np.float32, **kw)
        finally:
            TE._library = plain
