"""f32 batches evaluated in binary64 (GAAST_ARITH_F64) against the f64 and f32 variants: time, bandwidth and error of
the specialised kernels of cfg1-cfg5 at their BASELINE batch lengths, one JSON line per (workload, variant).

    python tools/f32_wide_bw.py > profiles/f32_wide_bw.jsonl

Variants: "f64" (f64 batches, FMA arithmetic), "f32" (f32 batches, binary32 FMA arithmetic) and "f32_wide" (f32
batches, GAAST_ARITH_FMA | GAAST_ARITH_F64).  Inputs are drawn on the device (uniform in [-1, 1], seeded; the f32
batches hold the f64 values rounded to binary32).  Each variant is warmed up, then the three are timed in turn with
CUDA events, `--rounds` times over `--reps` calls each, alternating within one process; ms is the median round.
GB/s counts the algorithmic bytes (gaast_plan_cost: the inputs read and the results written, at the batch's element
size); copy_frac = that rate over a torch device-to-device copy timed in the same process.  fma/elem and the key come
from last_kernel.  Error: the largest |result - oracle| over 2 048 seeded sample columns, in ulps of binary32 at the
oracle's value (the f64 oracle on the widened f32 inputs).  The card's name and power limit (nvidia-smi, read only)
are on every line."""
import argparse
import json
import os
import subprocess
import sys
from math import comb

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from tests.helpers import oracle_eval  # noqa: E402

VARIANTS = [("f64", L.F64, L.ARITH_FMA), ("f32", L.F32, L.ARITH_FMA), ("f32_wide", L.F32, L.ARITH_FMA | L.ARITH_F64)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:
        return f"unknown ({e})", "unknown"


def time_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    args = ap.parse_args()
    gpu, power = gpu_info()
    ctx = g.Ctx.on_torch_stream(0)
    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    copy_gbps = 2 * src.numel() / time_ms(lambda: dst.copy_(src), 10) / 1e6
    del src, dst
    for name in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
        if args.only and name not in args.only.split(","):
            continue
        w = W.WORKLOADS[name]
        n, batch = w.n, w.batch
        gen = torch.Generator(device="cuda")
        gen.manual_seed(2024)
        t64 = [{k: torch.empty((comb(n, k), 1 if bc else batch), dtype=torch.float64, device="cuda")
                .uniform_(-1.0, 1.0, generator=gen) for k in grades} for grades, bc in w.inputs]
        t32 = [{k: v.float() for k, v in d.items()} for d in t64]
        t64 = [{k: v.double() for k, v in d.items()} for d in t32]  # the same values in both types
        plan = g.Plan(ctx, W.specialize(w))
        bslots = w.broadcast_mask()
        bytes64, _ = plan.cost(bslots)
        calls, outs = {}, {}
        for label, dtype, arith in VARIANTS:
            ts = t64 if dtype == L.F64 else t32
            dev = [g.DeviceBatch.wrap_torch(ctx, n, t, broadcast=bc) for t, (_, bc) in zip(ts, w.inputs)]
            out = plan.alloc_output(batch, dtype)
            calls[label] = (lambda dev=dev, out=out, arith=arith:
                            plan.eval(dev, out=out, engine=L.ENGINE_SPECIALIZED, arith=arith))
            outs[label] = out
        kernels = {}
        for label, _, _ in VARIANTS:  # warm-up: every kernel loaded, every first-call allocation made
            calls[label]()
            calls[label]()
            torch.cuda.synchronize()
            kernels[label] = plan.last_kernel()
        times = {label: [] for label, _, _ in VARIANTS}
        for _ in range(args.rounds):
            for label, _, _ in VARIANTS:
                times[label].append(time_ms(calls[label], args.reps))
        cols = np.sort(np.random.default_rng(7).choice(batch, 2048, replace=False))
        idx = torch.from_numpy(cols).to("cuda")
        host = [{k: (v[:, :1] if bc else v[:, idx]).cpu().numpy() for k, v in d.items()} for d, (_, bc) in zip(t64, w.inputs)]
        want = oracle_eval(w.build, w.metric, host, [bc for _, bc in w.inputs], len(cols))
        for label, dtype, arith in VARIANTS:
            calls[label]()
            ctx.sync()
            got = outs[label].to_host()
            ctx.sync()
            ulps = 0.0
            for k in want:
                ref = want[k]
                ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
                ulps = max(ulps, float((np.abs(got[k][:, cols].astype(np.float64) - ref) / ulp).max()))
            ms = float(np.median(times[label]))
            es = 4 if dtype == L.F32 else 8
            nbytes = bytes64 // 8 * es * batch
            kern = kernels[label]
            line = dict(workload=name, variant=label, elements=batch, ms=round(ms, 4),
                        ms_rounds=[round(t, 4) for t in times[label]], gbps=round(nbytes / ms / 1e6, 1),
                        copy_gbps=round(copy_gbps, 1), copy_frac=round(nbytes / ms / 1e6 / copy_gbps, 3),
                        fma_per_elem=int(kern.split("fma/elem=")[1].split()[0]), key=kern.split("key=")[1].split()[0],
                        max_err_f32_ulps=round(ulps, 3), sample_columns=len(cols), gpu=gpu, power_limit=power,
                        reps=args.reps, rounds=args.rounds)
            print(json.dumps(line), flush=True)
        plan.free()
        del t64, t32, outs, calls
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
