#!/usr/bin/env python
"""bench.py -- multivector products/s of the B200 batch evaluator (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one evaluation of the workload's expression over one full batch of
synthetic random multivectors resident in HBM (one kernel launch).  The line says only
what THIS run measured:

* headline (`value`, `roofline`): the workload of `--workload` (default cfg2 = BASELINE
  configs[1]), weak scaling under torchrun (every rank a full BASELINE batch, no
  collective in the step).  Exactly K steps are timed, after W warm-up steps (at least 3);
  `ms_per_step` is (max over ranks of the CUDA-event time of the K steps) / K.  A short window
  (the default K = 20 of cfg2 lasts ~16 ms) runs at burst clocks; the power-capped steady state
  needs K steps to last >= 0.5 s (cfg2: K ~ 650).
  `--dump-outputs DIR` writes what the last timed step computed (see dump_outputs).
* `e2e`: the same metric through gaast_eval_host (pinned HOST arrays in and out, H2D +
  kernels + D2H in the timed region), run on EVERY rank at the same time between two
  barriers; value = elements of all ranks / the slowest rank's time.
* `cfg5_sharded`: BASELINE configs[4] as it is defined -- ONE 32 M batch sharded over the
  N ranks (strong scaling), gaast_eval_sum + gaast_comm_allreduce_sum (NCCL, 66 doubles)
  inside the timed step, with the single-GPU time of the same batch measured on rank 0 of
  the same box in the same run, the step time without the all-reduce, and a check of the
  all-reduced vector against torch.distributed.
* `other_workloads` (N = 1): the other BASELINE configs, device-resident and (cfg3, cfg5)
  end to end on a bounded sub-batch, plus one full G(8,0) product on the dense-warp engine.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "multivector_products_per_sec"
UNIT = "products/s"
FP64_SUSTAINED_SECONDS = 0.5  # length of the sustained live FP64-peak probe (gaast_diag_fp64_peak)
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much

# stdout carries exactly ONE line, the JSON record.  Libraries print there too (NCCL announces its
# version on stdout when the process group starts): file descriptor 1 is pointed at stderr for the
# whole run and the record is written to the original stdout at the end.
_REAL_STDOUT = None


def _claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# FP64 FMA-pipe peak.  MEASURED_PEAKS.json carries no f64 figure, so the denominator is this repo's own
# microbenchmark (profiles/fp64_peak.cu -> profiles/r1_fp64_peak.txt, 36.84 TFLOP/s; 148 SMs x 64 DFMA/clk x
# 1.965 GHz = 37.2 nominal); `roofline.fp64_peak_source` says so in the line.
FP64_PEAK_TFLOPS = float(os.environ.get("GAAST_FP64_PEAK_TFLOPS", "0") or 0) or 36.84
FP64_PEAK_SOURCE = "profiles/r1_fp64_peak.txt (this repo's DFMA microbenchmark; MEASURED_PEAKS.json has no f64 figure)"


def _ncu_traffic(kernel_desc: str, elements: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of
    the cubin that ran -- profiles/ncu_traffic.json is keyed by the cubin key `gaast_plan_last_kernel` reports.
    A capture taken at another batch length is scaled by the element ratio (and says so); a kernel whose key
    has no capture reports null and the reason."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception as ex:
        return None, f"profiles/ncu_traffic.json unreadable: {ex}"
    key = None
    for tok in kernel_desc.split():
        if tok.startswith("key="):
            key = tok[4:]
    if not key:
        return None, "the kernel that ran has no cubin key (library kernel)"
    ent = table.get(key)
    if not ent:
        return None, f"no ncu capture committed for cubin {key}"
    scale = elements / float(ent["elements"])
    note = ent["source"] + (f" (captured at {ent['elements']} elements, scaled x{scale:g})" if scale != 1.0 else "")
    if "dram_pct_of_peak" in ent:
        # the second denominator: what ncu itself calls DRAM throughput in that capture (% of the device's DRAM peak;
        # MEASURED_PEAKS' copy bandwidth is ~80 % of it)
        note += f"; gpu__dram_throughput {ent['dram_pct_of_peak']:.1f} % of peak in that capture ({ent.get('ncu_ms', '?')} ms under ncu)"
    return int(ent["dram_bytes"] * scale), note


def _executed_fma(kernel_desc: str):
    """FMAs per element the generated kernel executes (the code generator counts them and reports
    `fma/elem=` in gaast_plan_last_kernel); None for library kernels."""
    for tok in kernel_desc.split():
        if tok.startswith("fma/elem="):
            try:
                return int(tok[9:])
            except ValueError:
                return None
    return None


class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.gpu = gpu_index
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, power, reasons = [], [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "samples_under_load": len(busy), "reasons": sorted(reasons),
                "covers": "the headline workload's warm-up and timed steps (sampled every 50 ms)"}


def _dist():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------ CPU baseline ----
def _oracle_ast(w, count):
    from gaast_b200 import workloads as W
    from tests.helpers import oracle_expr
    from oracle import gaast_oracle as go
    host = W.host_inputs(w, count)
    expr = oracle_expr(w.build, host, [bc for _, bc in w.inputs])
    return expr.specialize(go.Algebra(w.metric))


def cpu_port_rate(w, target_seconds: float, threads: int, storage: int):
    """Elements/s of the oracle's C++ port of eval.rs (oracle/eval_port.cpp) on a bounded sample."""
    from oracle import port
    probe = 2000 * max(1, threads)
    ast = _oracle_ast(w, probe)
    port.eval_port(ast, min(64, probe), storage, 1)  # warm (builds the .so on first use)
    t0 = time.perf_counter()
    port.eval_port(ast, probe, storage, threads)
    dt = time.perf_counter() - t0
    rate = probe / dt
    count = int(max(probe, min(rate * target_seconds, 4_000_000)))
    if count > probe:
        ast = _oracle_ast(w, count)
        t0 = time.perf_counter()
        port.eval_port(ast, count, storage, threads)
        dt = time.perf_counter() - t0
        rate = count / dt
    return rate, count, dt


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (the oracle's C++ restatement of
    eval.rs -- there is no rustc in this image, so not the Rust binary) on all host threads.
    The timed arm uses the reference's own storage model (GradeMapMV: a hash map of vectors, fresh
    cache per element); the same port with dense arrays and reused buffers is timed once beside it
    (`cpu_baseline.dense_storage_value`) so that both ratios are on record."""
    rank, world, _ = _dist()
    if rank != 0:
        return
    from gaast_b200 import workloads as W
    w = W.WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    per_step = max(2.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    from oracle import port
    rate, count, _ = cpu_port_rate(w, per_step, threads, storage=1)
    ast = _oracle_ast(w, count)
    for _ in range(args.warmup):
        port.eval_port(ast, count, 1, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        port.eval_port(ast, count, 1, threads)
    dt = time.perf_counter() - t0
    value = count * args.steps / dt * w.products
    dense_rate, dense_count, dense_dt = cpu_port_rate(w, 4.0, threads, storage=0)
    sample = (f"{count} elements per step of {w.name} (full batch {w.batch}); GradeMapMV-like hash-map storage, "
              f"fresh cache per element, {threads} threads over batch ranges")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{w.name}: {w.title}", "batch_per_gpu": w.batch, "sample_elements": count},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "dense_storage_value": dense_rate * w.products,
                         "dense_storage_sample": f"{dense_count} elements, {dense_dt:.1f} s, the same port with dense per-grade "
                                                 f"arrays and buffers reused across elements, {threads} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


# ------------------------------------------------------------------------ GPU arm ----
def _root_cols(plan, w):
    from math import comb
    return sum(comb(w.n, k) for k in plan.root_grades())


class Resident:
    """One workload resident in HBM on this rank: plan, input/output sets, the step closure."""

    def __init__(self, ctx, w, torch, batch=None, engine=None, tuning=None, f32=False, with_sum=None, seed_shift=0,
                 torch_out=False, arith=None):
        import gaast_b200 as g
        from gaast_b200 import _lib as L
        from gaast_b200 import workloads as W
        self.ctx, self.w, self.torch = ctx, w, torch
        self.dev = torch.device("cuda", ctx.device)
        self.n = n = batch or w.batch
        self.f32 = f32
        self.plan = g.Plan(ctx, W.specialize(w))
        if tuning:
            self.plan.set_tuning(*tuning)
        self.bytes_per_elem, self.flops_per_elem = self.plan.cost(w.broadcast_mask())
        if f32:
            self.bytes_per_elem //= 2
        # L2 hygiene: a step must not find its inputs in the 126 MB L2.  Large workloads are larger
        # than L2 by themselves; small ones (cfg1: 185 MB) rotate over several input/output sets.
        self.n_sets = max(1, min(8, -(-(1 << 30) // max(1, n * self.bytes_per_elem))))
        if os.environ.get("GAAST_BENCH_NO_ROTATE"):
            self.n_sets = 1  # diagnostic only: lets a small batch stay L2-resident
        self.sets = []
        for k in range(self.n_sets):
            t = W.torch_inputs(w, n, self.dev, seed=(None if k == 0 and not seed_shift else W.seed_of(w) + 1000 * k + seed_shift))
            if f32:
                t = [{kk: v.float() for kk, v in x.items()} for x in t]
            i = [g.DeviceBatch.wrap_torch(ctx, w.n, x, broadcast=bc) for x, (_, bc) in zip(t, w.inputs)]
            if torch_out:  # the output as torch tensors, so that torch can check sums on the device
                from math import comb
                ot = {k2: torch.empty((comb(w.n, k2), n), dtype=torch.float32 if f32 else torch.float64, device=self.dev)
                      for k2 in self.plan.root_grades()}
                o = g.DeviceBatch.wrap_torch(ctx, w.n, ot)
                o.tensors = ot
            else:
                o = self.plan.alloc_output(n, L.F32 if f32 else L.F64)
            self.sets.append((t, i, o))
        self.use_sum = w.sum_root if with_sum is None else with_sum
        self.sums = torch.zeros(_root_cols(self.plan, w), dtype=torch.float64, device=self.dev)
        self.engine = L.ENGINE_AUTO if engine is None else engine
        self.arith = L.ARITH_FMA if arith is None else arith
        self.counter = 0
        self.last_set = None  # index into self.sets of the most recent step (or graph capture of one)
        self.comm = None

    def step(self):
        self.last_set = self.counter % self.n_sets
        _, s_in, s_out = self.sets[self.last_set]
        self.counter += 1
        if self.use_sum:
            self.plan.eval_sum(s_in, self.sums.data_ptr(), out=s_out, engine=self.engine, arith=self.arith)
            if self.comm is not None:
                # the only collective of the path: the root vector (66 doubles for cfg5), through the library's own
                # communicator (gaast_comm_allreduce_sum: NCCL behind the C ABI), ordered on the ctx stream
                self.comm.allreduce_sum([self.sums.data_ptr()], self.sums.numel())
        else:
            self.plan.eval(s_in, out=s_out, engine=self.engine, arith=self.arith)

    def kernel(self):
        return self.plan.last_kernel()


def timed(res, steps, warmup, torch, dist, world, allow_graph=True):
    """Warm up, then time exactly `steps` steps, bracketed by CUDA events on the ctx stream, with a
    barrier + synchronize on both sides; returns the MAX over ranks of that time, per step, and
    `last_set`, the input/output set of the last timed step."""
    ctx = res.ctx
    dev = res.dev
    for _ in range(max(3, warmup)):
        res.step()
    torch.cuda.synchronize()
    # Launch-bound steps (cfg1: 185 MB, ~30 us per kernel) are captured once into a CUDA graph and
    # replayed: the evaluation is stream-ordered and allocates nothing after its first call, so the
    # C ABI is capturable as it is.  Everything else is launched directly.
    expect_us = res.n * res.bytes_per_elem / 6.5e6
    use_graph = (allow_graph and world == 1 and not res.use_sum and expect_us < 200.0
                 and not os.environ.get("GAAST_BENCH_NO_GRAPH"))
    graph = None
    if use_graph:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ctx.torch_stream):
            for _ in range(steps):
                res.step()
        graph.replay()  # untimed: the first launch of a graph also uploads it to the device
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = ctx.launch_count
    # ~1 ms of device spin ahead of the window: the host enqueues the first steps meanwhile, so that the window holds
    # the steps' device time and not the idle device waiting for the first launch after the synchronize
    torch.cuda._sleep(2_000_000)
    e0.record()
    if graph is not None:
        graph.replay()
    else:
        for _ in range(steps):
            res.step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    last_set = res.last_set  # (a graph replays the steps of its capture: the last captured step's set)
    launches = ctx.launch_count - launches0  # this library's kernels only (NCCL's all-reduce kernel is not counted)
    if graph is not None:
        launches = steps * max(1, launches_per_step(res))
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # the slowest rank
    ms = float(ms.item())
    return {"ms_per_step": ms / steps, "timed_region_s": ms / 1e3, "launches": launches, "cuda_graph": graph is not None,
            "last_set": last_set}


def launches_per_step(res):
    """Kernels one step launches (counted on an extra, untimed step; used for graph replays, whose launches
    the library's counter does not see)."""
    c0 = res.ctx.launch_count
    res.step()
    res.torch.cuda.synchronize()
    return res.ctx.launch_count - c0


def dump_columns(length, bytes_per_column, budget):
    """Batch columns that --dump-outputs writes: None (all of them) when they fit in `budget` bytes, else a fixed,
    seeded, sorted sample, the same for every run with the same batch length."""
    import numpy as np
    keep = max(1, budget // max(1, bytes_per_column))
    if length <= keep:
        return None
    return np.sort(np.random.default_rng(0x6AA57D00).choice(length, size=keep, replace=False))


class _GradeView:
    """Grade k of a library-allocated batch ([rows][stride] in device memory) as a CUDA array interface, so that
    torch.as_tensor sees it without a copy."""

    def __init__(self, batch, k):
        from gaast_b200 import _lib as L
        size = 4 if batch.dtype == L.F32 else 8
        self.__cuda_array_interface__ = {"shape": (batch.stored_rows(k), batch.length), "strides": (batch.stride * size, size),
                                         "typestr": f"<f{size}", "data": (batch.grade_ptr(k), False), "version": 2}


def dump_outputs(path, res, last_set):
    """What the caller of the timed path received from its last step, as <path>/<name>.npy in the run's float type:
    `out_g<k>` per root grade ([C(n,k), columns]) and, for a batch-sum plan, `sum` (the root vector).  When the
    per-element outputs exceed DUMP_BYTES in all, the same seeded sample of columns (dump_columns) is taken of each
    grade."""
    import numpy as np
    torch = res.torch
    out = res.sets[last_set][2]
    grades = res.plan.root_grades()
    arrays = {f"out_g{k}": (out.tensors[k] if hasattr(out, "tensors") else torch.as_tensor(_GradeView(out, k), device=res.dev))
              for k in grades}
    whole = {"sum": res.sums} if res.use_sum else {}
    per_column = sum(a.shape[0] * a.element_size() for a in arrays.values())
    budget = DUMP_BYTES - sum(a.numel() * a.element_size() for a in whole.values()) - 1024 * (len(arrays) + len(whole))
    cols = dump_columns(res.n, per_column, budget)
    if cols is not None:
        idx = torch.from_numpy(cols).to(res.dev)
        arrays = {name: a.index_select(1, idx) for name, a in arrays.items()}
    torch.cuda.synchronize()
    os.makedirs(path, exist_ok=True)
    for name, a in {**arrays, **whole}.items():
        np.save(os.path.join(path, name + ".npy"), a.contiguous().cpu().numpy())


def measure_e2e(res, steps, torch, dist, world, elements=None, host_mem="torch"):
    """Same metric through gaast_eval_host: pinned host arrays in and out, H2D + kernel + D2H in the timed
    region.  Under torchrun EVERY rank runs its own pipeline at the same time (barrier before and after);
    returns the slowest rank's time."""
    from math import comb
    w, plan = res.w, res.plan
    n = min(res.n, elements or res.n)
    tin = res.sets[0][0]
    host_in, grades, bcs, keep = [], [], [], []
    h2d = 0
    dt = next(iter(tin[0].values())).dtype  # float64, or float32 for the f32 variant
    es = 4 if dt == torch.float32 else 8
    for t, (gr, bc) in zip(tin, w.inputs):
        rows = sum(comb(w.n, k) for k in gr)
        if host_mem != "torch" and not bc:
            # the library's own page-locked allocation (gaast_host_alloc), write-combined for "gaast-wc": inputs are only
            # ever written by the host
            import numpy as np
            import gaast_b200 as g
            ha = g.HostArray(rows, n, dtype=np.float32 if dt == torch.float32 else np.float64, write_combined=host_mem == "gaast-wc")
            keep.append(ha)
            h = torch.from_numpy(ha.array)
        else:
            h = torch.empty((rows, 1 if bc else n), dtype=dt, pin_memory=True)
        r = 0
        for k in gr:
            c = comb(w.n, k)
            h[r:r + c].copy_(t[k] if bc else t[k][:, :n])
            r += c
        host_in.append(h)
        grades.append(gr)
        bcs.append(bc)
        h2d += rows * es * (1 if bc else n)
    out_rows = _root_cols(plan, w)
    host_out = torch.empty((out_rows, n), dtype=dt, pin_memory=True)
    torch.cuda.synchronize()
    plan.eval_host(host_in, grades, bcs, n, host_out)  # warm-up: allocates the device buffer sets
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        plan.eval_host(host_in, grades, bcs, n, host_out)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = max(e0.elapsed_time(e1), wall * 1e3)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=res.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    # sanity: the result equals the resident path's (same inputs, same kernel)
    res.counter = 0
    res.step()
    torch.cuda.synchronize()
    k0 = plan.root_grades()[0]
    o = res.sets[0][2]
    ref = (o.tensors[k0][:, :1000].cpu().numpy() if hasattr(o, "tensors") else o.download(k0)[:, :1000])
    got = host_out[:ref.shape[0], :1000].numpy()
    ok = bool((ref == got).all())
    return {"ms_per_step": ms / steps, "h2d": h2d, "d2h": out_rows * es * n, "matches_resident": ok, "elements": n}


FP64_LIVE_SUSTAINED = [None]  # set by run_gpu once measured; other_workloads report their fraction of it too


def _workload_record(res, t, peak_gbs, w):
    s = t["ms_per_step"] / 1e3
    n = res.n
    kernel = res.kernel()
    traffic, traffic_src = _ncu_traffic(kernel, n) if not res.f32 else (None, "no capture of the f32 kernels")
    rec = {"elements_per_s": n / s, "products_per_s": n / s * w.products, "ms_per_step": t["ms_per_step"],
           "timed_region_s": t["timed_region_s"],
           "hbm_gbs": n * res.bytes_per_elem / s / 1e9, "hbm_frac": n * res.bytes_per_elem / s / 1e9 / peak_gbs,
           "fp64_tflops": n * res.flops_per_elem / s / 1e12,
           "fp64_frac": n * res.flops_per_elem / s / 1e12 / FP64_PEAK_TFLOPS,
           "bound": w.bound, "ncu_traffic_bytes": traffic, "ncu_traffic_source": traffic_src,
           "batch": n, "kernel": kernel, "io_sets_rotated": res.n_sets, "cuda_graph": t["cuda_graph"]}
    fma = _executed_fma(kernel)
    if fma is not None:
        rec["fma_per_element_executed"] = fma
        rec["fp64_tflops_executed"] = n * 2.0 * fma / s / 1e12
    if FP64_LIVE_SUSTAINED[0]:
        rec["fp64_frac_of_live_sustained_peak"] = rec["fp64_tflops"] / FP64_LIVE_SUSTAINED[0]
    return rec


def run_cfg5_sharded(ctx, torch, dist, rank, world, steps, warmup, peak_gbs):
    """BASELINE configs[4]: ONE 32 M batch of G(8,4) (V*X*V.vinv()).g(2), sharded over the ranks, with the
    batch-sum: gaast_eval_sum on every shard + gaast_comm_allreduce_sum of the 66-double root vector inside
    the timed step.  Strong scaling; the single-GPU time of the same 32 M batch is measured on rank 0 first."""
    import gaast_b200 as g
    from gaast_b200 import workloads as W
    from gaast_b200.dist import shard_range
    w = W.WORKLOADS["cfg5"]
    total = w.batch
    rec = {"workload": f"{w.name}: {w.title}", "batch_total": total, "n_gpus": world, "scaling": "strong",
           "collective": "gaast_comm_allreduce_sum (66 f64, sum) on the ctx stream, inside every timed step"}
    one_ms = None
    if world > 1:
        # (1) the same 32 M batch on ONE GPU of this box (rank 0; the other ranks wait at the barrier inside timed())
        if rank == 0:
            r1 = Resident(ctx, w, torch, batch=total)
            t1 = timed(r1, steps, warmup, torch, dist, 1, allow_graph=False)
            one_ms = t1["ms_per_step"]
            rec["one_gpu"] = {"ms_per_step": one_ms, "elements_per_s": total / one_ms * 1e3,
                              "products_per_s": total / one_ms * 1e3 * w.products,
                              "hbm_frac": total * r1.bytes_per_elem / one_ms / 1e6 / peak_gbs, "kernel": r1.kernel(),
                              "note": "gaast_eval_sum over the whole batch on rank 0's GPU while the other ranks idle"}
            del r1
            torch.cuda.empty_cache()
        dist.barrier()
    b0, b1 = shard_range(total, rank, world)
    res = Resident(ctx, w, torch, batch=b1 - b0, seed_shift=7919 * rank, torch_out=True)
    if world > 1:
        uid = [g.Comm.unique_id() if rank == 0 else None]  # torch.distributed only ships the 128-byte id
        dist.broadcast_object_list(uid, src=0)
        res.comm = g.Comm.join(ctx, world, rank, uid[0])
        rec["collective_transport"] = res.comm.transport  # "peer": the library's one-shot kernel over NVLink peer memory
        rec["collective"] += {"peer": "; transport: this library's peer-memory kernel (one launch, NVLink stores + flags, rank-ordered sum)",
                              "nccl": "; transport: ncclAllReduce"}.get(res.comm.transport, "")
    t = timed(res, steps, warmup, torch, dist, world, allow_graph=False)
    s = t["ms_per_step"] / 1e3
    rec.update({"ms_per_step": t["ms_per_step"], "timed_region_s": t["timed_region_s"], "shard_elements": res.n,
                "elements_per_s": total / s, "products_per_s": total / s * w.products,
                "hbm_gbs_per_gpu": res.n * res.bytes_per_elem / s / 1e9,
                "hbm_frac_per_gpu": res.n * res.bytes_per_elem / s / 1e9 / peak_gbs,
                "kernel": res.kernel(), "gpu_launches": t["launches"]})
    # (2) the check: the all-reduced vector of the last step against torch.distributed's all-reduce of torch sums
    res.counter = 0
    res.step()
    torch.cuda.synchronize()
    got = res.sums.clone()
    o = res.sets[0][2]
    want = torch.cat([o.tensors[k].sum(dim=1) for k in sorted(o.tensors)])
    mag = torch.cat([o.tensors[k].abs().sum(dim=1) for k in sorted(o.tensors)])
    if world > 1:
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        dist.all_reduce(mag, op=dist.ReduceOp.SUM)
    err = float(((got - want).abs() / mag.clamp_min(1e-300)).max().item())
    rec["sum_check"] = bool(err <= 1e-12)
    rec["sum_check_detail"] = {"max_abs_err_over_sum_abs": err, "tolerance": 1e-12,
                               "against": "torch.distributed.all_reduce(SUM) of per-rank torch.sum over the output arrays"}
    # (3) the same step without the collective: what the all-reduce costs
    if world > 1:
        comm, res.comm = res.comm, None
        t0 = timed(res, steps, warmup, torch, dist, world, allow_graph=False)
        res.comm = comm
        rec["ms_per_step_without_allreduce"] = t0["ms_per_step"]
        rec["allreduce_cost_ms"] = t["ms_per_step"] - t0["ms_per_step"]
        if comm.transport == "peer":
            # (4) the same step with NCCL carrying the 66 doubles instead of the library's peer-memory kernel
            from gaast_b200 import _lib as L
            comm.set_transport(L.COMM_NCCL)
            tn = timed(res, steps, warmup, torch, dist, world, allow_graph=False)
            comm.set_transport(L.COMM_AUTO)
            rec["ms_per_step_with_nccl_allreduce"] = tn["ms_per_step"]
            rec["nccl_allreduce_cost_ms"] = tn["ms_per_step"] - t0["ms_per_step"]
        one = torch.tensor([one_ms or 0.0], dtype=torch.float64, device=res.dev)
        dist.all_reduce(one, op=dist.ReduceOp.MAX)
        one_ms = float(one.item())
        rec["speedup_vs_one_gpu_same_box"] = one_ms / t["ms_per_step"]
        rec["scaling_efficiency"] = one_ms / t["ms_per_step"] / world
        comm.close()
    return rec


def run_gpu(args):
    import torch
    import torch.distributed as dist
    rank, world, local = _dist()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import gaast_b200 as g
    from gaast_b200 import _lib as L
    from gaast_b200 import workloads as W
    ctx = g.Ctx.on_torch_stream(local)
    w = W.WORKLOADS[args.workload]
    peak_gbs, peak_src = _peaks()
    f32 = args.dtype == "f32"

    batch = args.batch
    if args.strong and world > 1:
        from gaast_b200.dist import shard_range
        b0, b1 = shard_range(batch or w.batch, rank, world)
        batch = b1 - b0  # the BASELINE batch split into contiguous, 16-byte aligned slices
    # live FP64 FMA-pipe peak of THIS box (gaast_diag_fp64_peak: independent DFMA chains): a 20 ms burst on the idle
    # GPU, and -- measured after the headline, below -- 0.5 s sustained, the like-for-like denominator of a kernel
    # timed over >= 0.5 s, i.e. with --steps large enough (an FP64-heavy B200 is power-capped well below 1965 MHz by
    # then); the burst figure is the one to set beside a short timed window
    fp64_live = None
    if rank == 0 and not f32:
        try:
            fp64_live = {"burst_tflops": ctx.fp64_peak(0.02)}
        except Exception as ex:
            fp64_live = {"error": f"{type(ex).__name__}: {ex}"}
    sampler = ClockSampler(local) if rank == 0 else None
    res = Resident(ctx, w, torch, batch=batch, engine={'auto': 0, 'table': 1, 'specialized': 2}[args.engine],
                   tuning=(args.ept, args.variant) if (args.ept or args.variant) else None,
                   with_sum=False if args.no_sum else None, f32=f32, arith={"fma": 0, "strict": 1}[args.arith])
    if res.use_sum and world > 1:
        uid = [g.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        res.comm = g.Comm.join(ctx, world, rank, uid[0])
    t = timed(res, args.steps, args.warmup, torch, dist, world)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, t["last_set"])

    n = res.n
    sec = t["ms_per_step"] / 1e3
    elems_per_s = n * world / sec
    value = elems_per_s * w.products
    gbs = n * res.bytes_per_elem / sec / 1e9
    tflops = n * res.flops_per_elem / sec / 1e12
    kernel = res.kernel()
    traffic, traffic_src = (None, "no capture of the f32 kernels") if f32 else _ncu_traffic(kernel, n)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": t["ms_per_step"], "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": f"{w.name}: {w.title}" + (" [f32 variant: not the reference's precision]" if f32 else ""),
                   "batch_per_gpu": n, "elements_per_s": elems_per_s,
                   "products_per_element": w.products, "parallelism": f"batch-sharded x{world}, no data-path collective"
                   + (" (+66-double NCCL all-reduce for the batch-sum, gaast_comm_allreduce_sum)" if res.comm is not None else ""),
                   "l2": f"inputs+outputs {n * res.bytes_per_elem / 1e9:.2f} GB per step (126 MB L2), "
                         f"{res.n_sets} input/output set(s) used in rotation",
                   "timing": f"{args.steps} timed steps ({t['timed_region_s']:.4f} s of device time), "
                             f"max over ranks of their CUDA-event time"
                             + ("; a window under 0.5 s runs at burst clocks" if t["timed_region_s"] < 0.5 else ""),
                   "io_sets_rotated": res.n_sets,
                   "kernel": kernel, "cuda_graph": t["cuda_graph"]},
        "gpu_launches": t["launches"],
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": n * res.bytes_per_elem,
                     "fp64_tflops_algorithmic": tflops, "fp64_peak_tflops": FP64_PEAK_TFLOPS,
                     "fp64_peak_source": FP64_PEAK_SOURCE, "fp64_frac_algorithmic": tflops / FP64_PEAK_TFLOPS},
    }
    fma = _executed_fma(kernel)
    if fma is not None:
        # a lowered plan executes fewer FMAs than the reference's term count (cfg2: the 160 terms of R X ~R become a
        # 25-FMA linear map): the algorithmic figure counts the reference's terms, this one the kernel's own
        line["roofline"]["fma_per_element_executed"] = fma
        line["roofline"]["fp64_tflops_executed"] = n * 2.0 * fma / sec / 1e12
        line["roofline"]["fp64_frac_executed"] = n * 2.0 * fma / sec / 1e12 / FP64_PEAK_TFLOPS
    if clocks is not None:
        line["clocks"] = clocks
    if fp64_live is not None and "error" not in fp64_live:
        try:
            if world > 1:
                pass  # (rank 0 only measures while the other ranks wait at the next barrier)
            fp64_live["sustained_tflops"] = ctx.fp64_peak(FP64_SUSTAINED_SECONDS)
            fp64_live["how"] = ("gaast_diag_fp64_peak on this GPU in this run: 20 ms burst before the timed region, "
                                f"{FP64_SUSTAINED_SECONDS} s sustained after it")
        except Exception as ex:
            fp64_live["error"] = f"{type(ex).__name__}: {ex}"
    if fp64_live is not None:
        line["roofline"]["fp64_peak_live"] = fp64_live
        FP64_LIVE_SUSTAINED[0] = fp64_live.get("sustained_tflops")

    if f32:  # no CPU leg for the f32 variant (the reference is f64-only); its FMA-pipe peak is not the f64 one
        args.no_cpu = True
        args.all = False
        for key in [k for k in line["roofline"] if k.startswith(("fp64_", "fma_"))]:
            line["roofline"].pop(key)
        line["roofline"]["fp32_tflops"] = tflops
    if not args.no_e2e:
        try:
            e = measure_e2e(res, max(2, min(args.steps, 3)), torch, dist, world, host_mem=args.e2e_host)
            line["e2e"] = {"value": e["elements"] * world / (e["ms_per_step"] / 1e3) * w.products, "unit": UNIT,
                           "h2d_bytes_per_step": e["h2d"], "d2h_bytes_per_step": e["d2h"],
                           "ms_per_step": e["ms_per_step"], "matches_resident": e["matches_resident"],
                           "host_memory": {"torch": "torch pin_memory (cudaHostAlloc)", "gaast": "gaast_host_alloc",
                                           "gaast-wc": "gaast_host_alloc, inputs write-combined"}[args.e2e_host],
                           # PCIe is the bound of this leg: tools/pcie_peak.py measured 55.6 (H2D alone), 55.0 (D2H alone)
                           # and 47.1 GB/s each way at the same time on this pool (profiles/r1_pcie_peak.txt)
                           "gbs_each_way_per_gpu": max(e["h2d"], e["d2h"]) / (e["ms_per_step"] * 1e6),
                           "note": ("gaast_eval_host_f32" if f32 else "gaast_eval_host")
                           + ": pinned host arrays, chunked H2D/kernel/D2H pipeline"
                           + (f"; all {world} ranks at the same time between two barriers, slowest rank's time" if world > 1 else "")}
        except Exception as ex:  # keep the headline line even if the host leg fails
            line["e2e"] = {"error": f"{type(ex).__name__}: {ex}"}
    del res
    torch.cuda.empty_cache()

    if not args.no_sharded and not f32:
        try:
            rec = run_cfg5_sharded(ctx, torch, dist, rank, world, args.steps, args.warmup, peak_gbs)
            line["cfg5_sharded"] = rec
        except Exception as ex:
            line["cfg5_sharded"] = {"error": f"{type(ex).__name__}: {ex}"}
        torch.cuda.empty_cache()

    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            r1, c1, d1 = cpu_port_rate(w, 8.0, 1, storage=1)
            r0, c0, d0 = cpu_port_rate(w, 4.0, 1, storage=0)
            line["cpu_baseline"] = {
                "value": r1 * w.products, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"first {c1} elements of the same synthetic workload, {d1:.1f} s, oracle/eval_port.cpp "
                          f"(C++ restatement of eval.rs with GradeMapMV-like hash-map storage; not the Rust binary)",
                "dense_storage_value": r0 * w.products,
                "host_cpus": os.cpu_count(),
            }
        except Exception as ex:
            line["cpu_baseline"] = {"error": f"{type(ex).__name__}: {ex}"}

    if rank == 0 and world == 1 and args.all:
        others = {}
        for name in ("cfg1", "cfg3", "cfg4", "cfg5"):
            if name == w.name:
                continue
            try:
                torch.cuda.empty_cache()
                ow = W.WORKLOADS[name]
                r = Resident(ctx, ow, torch)
                tt = timed(r, args.steps, args.warmup, torch, dist, 1)
                others[name] = _workload_record(r, tt, peak_gbs, ow)
                if name in ("cfg3", "cfg5") and not args.no_e2e:
                    # end to end on a bounded sub-batch (the full batches are 26-37 GB of pinned host memory; the
                    # leg is PCIe-bound, so its rate does not depend on the batch length)
                    e = measure_e2e(r, 2, torch, dist, 1, elements=4 << 20)
                    others[name]["e2e"] = {"value": e["elements"] / (e["ms_per_step"] / 1e3) * ow.products, "unit": UNIT,
                                           "elements": e["elements"], "h2d_bytes_per_step": e["h2d"],
                                           "d2h_bytes_per_step": e["d2h"], "ms_per_step": e["ms_per_step"],
                                           "matches_resident": e["matches_resident"]}
                del r
            except Exception as ex:
                others[name] = {"error": f"{type(ex).__name__}: {ex}"}
        # the same two workloads with their algebraic lowering switched off (code generator variant bits 17 / 16): the
        # reference's own term count executed FMA by FMA -- what the lowered kernels above are to be compared with
        for name, base, variant, what in (("cfg3_unlowered", "cfg3", 131072, "rolled 4 096-FMA dense product (no matrix representation)"),
                                          ("cfg5_unlowered", "cfg5", 65536, "1 608-FMA sandwich through the 232-component intermediate (no reflection lowering)")):
            try:
                torch.cuda.empty_cache()
                ow = W.WORKLOADS[base]
                r = Resident(ctx, ow, torch, tuning=(0, variant))
                tt = timed(r, args.steps, args.warmup, torch, dist, 1)
                others[name] = _workload_record(r, tt, peak_gbs, ow)
                others[name]["what"] = what
                del r
            except Exception as ex:
                others[name] = {"error": f"{type(ex).__name__}: {ex}"}
        # GAAST_ARITH_STRICT on the specialised engine: the reference's own term list in the reference's order, (l * r) * coeff
        # then +, no contraction and no lowering -- results BIT-IDENTICAL to eval.rs (tests/test_gpu_parity.py holds both engines
        # to that).  The default arithmetic (FMA, within 1e-12) is what every other entry runs; this is what exactness costs.
        from gaast_b200 import _lib as L
        strict = {}
        for name in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
            try:
                torch.cuda.empty_cache()
                ow = W.WORKLOADS[name]
                r = Resident(ctx, ow, torch, engine=L.ENGINE_SPECIALIZED, arith=L.ARITH_STRICT, with_sum=False)
                tt = timed(r, args.steps, args.warmup, torch, dist, 1)
                rec = _workload_record(r, tt, peak_gbs, ow)
                strict[name] = {k: rec[k] for k in ("elements_per_s", "products_per_s", "ms_per_step", "hbm_frac", "batch", "kernel")}
                del r
            except Exception as ex:
                strict[name] = {"error": f"{type(ex).__name__}: {ex}"}
        strict["what"] = ("the five BASELINE workloads in GAAST_ARITH_STRICT on the specialised engine (no batch-sum): bit-identical to "
                          "the reference's (l*r)*coeff-then-add sequence; 3 FP64 instructions per term instead of one FMA, no lowering")
        others["strict_arithmetic"] = strict
        try:
            torch.cuda.empty_cache()
            others["dense_warp_g8"] = run_dense_warp(ctx, torch, dist, args.steps, args.warmup, peak_gbs)
            others["dense_warp_g8_termwise"] = run_dense_warp(ctx, torch, dist, args.steps, args.warmup, peak_gbs,
                                                              variant=1048576)
            others["dense_g10"] = run_dense_warp(ctx, torch, dist, args.steps, args.warmup, peak_gbs, n=10, batch=64 * 1024)
        except Exception as ex:
            others["dense_warp_g8"] = {"error": f"{type(ex).__name__}: {ex}"}
        line["other_workloads"] = others

    if rank == 0:
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_dense_warp(ctx, torch, dist, steps, warmup, peak_gbs, n=8, batch=256 * 1024, variant=0):
    """One FULL geometric product A*B of 2^n-component multivectors in G(n,0) on the dense engine: no BASELINE config
    exercises that engine, these entries are its driver-visible numbers.  Default: the matrix-representation kernel
    (csrc/device/dense_matrix.cu: the product as real matrix products on the FP64 tensor cores, 2^(n+MX) multiplications
    instead of the 4^n terms `fp64_tflops` counts -- the figure to read is hbm_frac, the kernel moves 3 x 2^n doubles per
    product).  variant 1048576: the term-by-term kernel of the same engine (one warp per multivector, 4^n DFMAs)."""
    from gaast_b200 import workloads as W
    w = W.Workload(f"dense_g{n}", f"G({n},0) A*B, full {1 << n}-component multivectors (dense engine)", [1.0] * n,
                   [(tuple(range(n + 1)), False)] * 2, lambda A, B: A * B, batch, 1, bound="fp64" if variant else "hbm")
    r = Resident(ctx, w, torch, tuning=(0, variant) if variant else None)
    tt = timed(r, steps, warmup, torch, dist, 1, allow_graph=False)
    rec = _workload_record(r, tt, peak_gbs, w)
    rec["what"] = ("term-by-term dense-warp kernel (4^n DFMAs per product)" if variant else
                   "matrix-representation kernel: fp64_tflops counts the reference's 4^n terms (it may exceed the FP64 peak); "
                   "fp64_tflops_executed counts the DMMA multiplications only, not the transforms' additions")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg2", help="cfg1..cfg5 (default cfg2 = BASELINE configs[1])")
    ap.add_argument("--batch", type=int, default=None, help="override the batch length (default: the BASELINE size)")
    ap.add_argument("--impl", default="gaast_b200", choices=["gaast_b200", "reference"])
    ap.add_argument("--engine", default="auto", choices=["auto", "table", "specialized"])
    ap.add_argument("--arith", default="fma", choices=["fma", "strict"],
                    help="fma: one FMA per term, lowerings on (within 1e-12); strict: the reference's own operation sequence, bit-identical")
    ap.add_argument("--ept", type=int, default=0, help="tuning: elements per thread of the specialised kernel")
    ap.add_argument("--variant", type=int, default=0, help="tuning: code generator policy bits")
    ap.add_argument("--no-sum", action="store_true", help="skip the batch-sum node of cfg5")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"],
                    help="f64 = the reference's precision (default, the BASELINE metric); f32 = the reduced-precision variant")
    ap.add_argument("--strong", action="store_true", help="headline workload: shard ONE BASELINE batch over the ranks")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-host", default="torch", choices=["torch", "gaast", "gaast-wc"],
                    help="page-locked host arrays of the e2e leg: torch's, or the library's own (write-combined inputs)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the cfg5_sharded section")
    ap.add_argument("--all", action="store_true", default=True, help="also time the other BASELINE workloads (N=1)")
    ap.add_argument("--only", dest="all", action="store_false",
                    help="the headline workload only (no other_workloads, no cfg5_sharded)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload computed to DIR/<name>.npy (at most "
                         "64 MB: a fixed, seeded sample of the batch columns when the outputs are larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gaast_b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl gaast_b200)")
    if not args.all:
        args.no_sharded = True
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
