"""Time of projected plans (gaast_plan_create_projected) against their unprojected plans on the device, one JSON line
per pair.

    python tools/projection_bw.py > profiles/projection_bw.jsonl

Pairs: cfg5 at 32 M elements, unprojected against a seeded 9-of-66 projection of its bivector result; cfg2 at 64 M
elements, grade 1 with all 5 components against 3 of them.  The two plans of a pair run alternately in one process,
each timed with CUDA events over `--reps` calls after a warm-up; every working set is well above the 126 MB L2.  GB/s
counts the algorithmic bytes of gaast_plan_cost (inputs read + stored root components written).  Beside them: fma/elem
of the kernel that ran, and the card's name and power limit (nvidia-smi, read only) in the same run."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200 import workloads as W  # noqa: E402
from tools.records_bw import gpu_info  # noqa: E402

M = 1 << 20
# name, elements, {root grade: selected components}
PAIRS = [
    ("cfg5", 32 * M, {2: sorted(np.random.default_rng(9).choice(66, 9, replace=False).tolist())}),
    ("cfg2", 64 * M, {1: [0, 2, 4]}),
]


def fma_of(kernel):
    return int([t for t in kernel.split() if t.startswith("fma/elem=")][0][9:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two plans")
    args = ap.parse_args()
    name_gpu, power = gpu_info()
    ctx = g.Ctx.on_torch_stream(0)
    for name, count, comps in PAIRS:
        w = W.WORKLOADS[name]
        tin = W.torch_inputs(w, count, "cuda:0")
        torch.cuda.synchronize()
        dev = [g.DeviceBatch.wrap_torch(ctx, w.n, t, broadcast=bc) for t, (_, bc) in zip(tin, w.inputs)]
        bmask = sum(1 << s for s, (_, bc) in enumerate(w.inputs) if bc)
        plans = {"unprojected": g.Plan(ctx, W.specialize(w)), "projected": g.Plan(ctx, W.specialize(w), components=comps)}
        outs = {k: p.alloc_output(count) for k, p in plans.items()}
        ms = {k: [] for k in plans}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k, p in plans.items():  # warm-up: kernels loaded, scratch allocated
            p.eval(dev, out=outs[k])
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for k, p in plans.items():
                p.eval(dev, out=outs[k])
                e0.record()
                for _ in range(args.reps):
                    p.eval(dev, out=outs[k])
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1) / args.reps)
        line = dict(workload=name, elements=count, selected={str(k): v for k, v in comps.items()}, reps=args.reps,
                    rounds=args.rounds)
        for k, p in plans.items():
            bpe, fpe = p.cost(bmask)
            best = min(ms[k])
            line[k] = dict(ms=round(best, 4), ms_all=[round(x, 4) for x in ms[k]], bytes_per_elem=bpe, flops_per_elem=fpe,
                           gbps=round(bpe * count / best / 1e6, 1), fma_per_elem=fma_of(p.last_kernel()),
                           kernel=p.last_kernel().split(" key=")[0])
        u, pr = line["unprojected"], line["projected"]
        line.update(time_ratio=round(pr["ms"] / u["ms"], 3), bytes_ratio=round(pr["bytes_per_elem"] / u["bytes_per_elem"], 3),
                    gbps_ratio=round(pr["gbps"] / u["gbps"], 3), gpu=name_gpu, power_limit=power)
        print(json.dumps(line), flush=True)
        del dev, tin, outs, plans
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
