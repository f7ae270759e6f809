"""TEST INFRASTRUCTURE: the generated kernel of a PROJECTED plan (gaast_plan_create_projected) run on the CPU.

The same run as tests/kernel_emu.run_generated_kernel -- the CUDA text the code generator prints, compiled with g++
behind cuda_on_cpu.h and executed thread by thread on numpy arrays laid out like device batches -- for a plan that
stores only chosen root components: the output arrays hold the stored rows of each root grade and the batch-sum
vector one column per stored component."""
from __future__ import annotations

import ctypes as C
from math import comb
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

import gaast_b200 as g
from gaast_b200 import _lib as L
from tests.kernel_emu import ASAN, FAULTS, MAX_STREAMS, EmuLaunch, _compile, needs_threads


def run_projected_kernel(ast, inputs: Sequence[Dict[int, np.ndarray]], broadcast: Sequence[bool], batch: int,
                         components: Dict[int, Sequence[int]], arith: int = L.ARITH_FMA, with_sum: bool = False,
                         tuning: Optional[Tuple[int, int]] = None, grid: Optional[int] = None, store_out: bool = True,
                         dtype=np.float64, present: Optional[Dict] = None):
    """Evaluate the specialised engine's kernel for `ast` (a gaast_b200.expr.SpecializedAst) on host arrays.
    inputs[slot] = {grade: (C(n,k), batch) array, or (C(n,k), 1) for a broadcast slot}.
    present = {(slot, grade): stored component indices} for inputs in sparse per-grade storage: that grade's array
    then holds the stored rows only, in component order.
    components = {root grade: stored component indices} (a grade that is not listed is kept whole): the plan is
    gaast_plan_create_projected's, and out[k] / sums[k] hold the stored components of grade k only, in component order.
    Returns (out: {grade: (C, batch)}, sums or None, info) where info = {"notes", "threads", "ept", "grid", "source"}."""
    plan = g.Plan(None, ast, components=components)
    if tuning is not None:
        plan.set_tuning(*tuning)
    n = plan.n
    root_rows = {k: comb(n, k) if k not in components else len(set(components[k]))
                 for k in plan.root_grades()}
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
            if broadcast[s]:
                arr = np.zeros((rows, 4), dtype=dtype)
                arr[:, 0] = src_arr.reshape(rows, -1)[:, 0]
                launch.bcast[si >> 6] |= 1 << (si & 63)
            else:
                assert src_arr.shape == (rows, batch), (src_arr.shape, rows, batch)
                arr = np.full((rows, padded), np.nan, dtype=dtype)  # the padding is never part of a result
                arr[:, :batch] = src_arr
            keep.append(arr)
            launch.sptr[si] = arr.ctypes.data
            launch.srow[si] = arr.shape[1]
            si += 1
    outs = {}
    for k in plan.root_grades():
        arr = np.full((max(1, root_rows[k]), padded), np.nan, dtype=dtype)[:root_rows[k]]  # (an emptied grade: no rows)
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
