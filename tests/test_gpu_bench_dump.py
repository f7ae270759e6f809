"""bench.py --dump-outputs: the arrays the last timed step computed, checked against the oracle on the inputs of the
input/output set that step used -- the whole output of a small batch (directly launched and CUDA-graph steps, f64 and
f32), a seeded column sample of one larger than the 64 MB limit, and the batch-sum vector of a plan with a batch-sum
node -- and the launches of the timed region against exactly --steps steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS, WARMUP = 3, 1


def _launches_per_step(w, inputs, f32):
    """Kernels one evaluation of `w` launches, counted by the library, on the bench's own kind of step."""
    import torch
    import gaast_b200 as g
    from gaast_b200 import _lib as L
    from gaast_b200 import workloads as W
    ctx = g.Ctx.on_torch_stream(0)
    plan = g.Plan(ctx, W.specialize(w))
    dev = [g.DeviceBatch.wrap_torch(ctx, w.n, x, broadcast=bc) for x, (_, bc) in zip(inputs, w.inputs)]
    out = plan.alloc_output(next(iter(inputs[-1].values())).shape[1], L.F32 if f32 else L.F64)
    sums = torch.zeros(4096, dtype=torch.float64, device="cuda:0")

    def step():
        if w.sum_root:
            plan.eval_sum(dev, sums.data_ptr(), out=out)
        else:
            plan.eval(dev, out=out)

    step()
    torch.cuda.synchronize()
    c0 = ctx.launch_count
    step()
    ctx.sync()
    return ctx.launch_count - c0


@pytest.mark.parametrize("name,batch,dtype,graph", [("cfg1", 4096, "f64", True), ("cfg1", 4096, "f32", True),
                                                    ("cfg2", 2 << 20, "f64", False), ("cfg5", 4096, "f64", False)])
def test_dump_outputs_match_the_oracle(name, batch, dtype, graph, tmp_path):
    import torch
    import bench
    from gaast_b200 import workloads as W
    from tests.helpers import REL_TOL, REL_TOL_F32, assert_close, oracle_abs_scale, oracle_eval
    w = W.WORKLOADS[name]
    f32 = dtype == "f32"
    out_dir = tmp_path / "dump"
    env = dict(os.environ)
    if not graph:
        env["GAAST_BENCH_NO_GRAPH"] = "1"  # launches counted by the library, not derived from one extra step
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", name, "--batch", str(batch), "--only",
                        "--no-e2e", "--no-cpu", "--dtype", dtype, "--steps", str(STEPS), "--warmup", str(WARMUP),
                        "--dump-outputs", str(out_dir)], env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().split("\n")[-1])
    assert line["config"]["cuda_graph"] == (graph and not w.sum_root)
    files = sorted(os.listdir(out_dir))
    assert sum(os.path.getsize(out_dir / f) for f in files) <= bench.DUMP_BYTES
    got = {int(f[5:-4]): np.load(out_dir / f) for f in files if f.startswith("out_g")}

    # the sets rotate step by step from set 0; the warm-up runs max(3, W) steps before the K timed ones
    n_sets = line["config"]["io_sets_rotated"]
    assert n_sets > 1
    k = (max(3, WARMUP) + STEPS - 1) % n_sets
    dev = torch.device("cuda", 0)
    inputs = W.torch_inputs(w, batch, dev, seed=W.seed_of(w) + 1000 * k)
    if f32:
        inputs = [{g: v.float() for g, v in x.items()} for x in inputs]
    assert line["gpu_launches"] == STEPS * _launches_per_step(w, inputs, f32)
    host = [{g: v.double().cpu().numpy() for g, v in d.items()} for d in inputs]
    bcs = [bc for _, bc in w.inputs]
    rows = sum(a.shape[0] for a in got.values())
    size = 4 if f32 else 8
    cols = bench.dump_columns(batch, rows * size, bench.DUMP_BYTES - 1024 * len(files) - (rows * 8 if w.sum_root else 0))
    assert (cols is not None) == (name == "cfg2")  # 2 M five-component f64 outputs are 84 MB: sampled
    if cols is not None:
        host = [d if bc else {g: v[:, cols] for g, v in d.items()} for d, bc in zip(host, bcs)]
    n = batch if cols is None else len(cols)
    want = oracle_eval(w.build, w.metric, host, bcs, n)
    assert {g: v.dtype for g, v in got.items()} == {g: np.dtype(np.float32 if f32 else np.float64) for g in want}
    assert_close({g: v.astype(np.float64) for g, v in got.items()}, want, oracle_abs_scale(w.build, w.metric, host, bcs, n),
                 rel=REL_TOL_F32 if f32 else REL_TOL, what=f"{name} {dtype} dump vs oracle (set {k})")
    assert ("sum.npy" in files) == w.sum_root
    if w.sum_root:
        s = np.load(out_dir / "sum.npy")
        ref = np.concatenate([got[g].sum(axis=1) for g in sorted(got)])
        mag = np.concatenate([np.abs(got[g]).sum(axis=1) for g in sorted(got)])
        assert s.shape == ref.shape and np.all(np.abs(s - ref) <= 1e-12 * mag)
