"""Bandwidth of the per-segment sums (gaast_batch_segment_sum) on the device, one JSON line per case.

    python tools/segment_sum_bw.py > profiles/segment_sum_bw.jsonl

Shapes: cfg5's root (G(8,4) grade 2, 66 rows) at 32 M columns and G(3) full (8 rows) at 64 M columns, f64 and f32,
each with segments of 1, 16, 1024 and 2^20 columns and as one segment.  Every case is timed with CUDA events over at
least --seconds of calls after a warm-up; every working set is well above the 126 MB L2.  Per line:
  bytes       the stored rows read, the sums written (8 bytes each) and the offsets read;
  gbps        bytes / time, and copy_frac: that over the rate of a torch device-to-device copy of the rows (bytes read
              plus written), timed in the same run;
  torch_ms    torch.segment_reduce(rows, "sum", lengths=..., axis=1) on the same rows (f32 rows are summed in f32),
              and for one segment also rows.sum(dim=1);
  gpu, power_limit   the card's name and power limit (nvidia-smi, read only), on every line."""
import argparse
import json
import os
import subprocess
import sys
from math import comb

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402

M = 1 << 20
SHAPES = [  # name, n, grades, columns, dtype
    ("cfg5_root", 12, [2], 32 * M, L.F64),
    ("G3_full", 3, [0, 1, 2, 3], 64 * M, L.F64),
    ("cfg5_root_f32", 12, [2], 32 * M, L.F32),
    ("G3_full_f32", 3, [0, 1, 2, 3], 64 * M, L.F32),
]
SEGMENT_LENGTHS = [1, 16, 1024, 1 << 20, None]  # None: one segment over the whole batch


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def time_ms(fn, seconds):
    """Mean time of one call in ms, over at least `seconds` of calls after a warm-up."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(3, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=0.5)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    gpu, power = gpu_info()
    ctx = g.Ctx.on_torch_stream(0)
    want = args.shapes.split(",")
    for name, n, grades, length, dtype in SHAPES:
        if name not in want:
            continue
        tdt = torch.float32 if dtype == L.F32 else torch.float64
        S = sum(comb(n, k) for k in grades)
        rows = torch.randn((S, length), dtype=tdt, device="cuda:0")
        tensors, r0 = {}, 0
        for k in grades:
            c = comb(n, k)
            tensors[k] = rows[r0:r0 + c]
            r0 += c
        torch.cuda.synchronize()
        b = g.DeviceBatch.wrap_torch(ctx, n, tensors)
        row_bytes = S * length * rows.element_size()
        dst = torch.empty_like(rows)
        copy_ms = time_ms(lambda: dst.copy_(rows), args.seconds)
        copy_gbps = 2 * row_bytes / copy_ms / 1e6
        del dst
        for seg in SEGMENT_LENGTHS:
            seg_len = length if seg is None else seg
            n_seg = (length + seg_len - 1) // seg_len
            offsets = torch.clamp(torch.arange(n_seg + 1, dtype=torch.int64, device="cuda:0") * seg_len, max=length)
            out = torch.empty((n_seg, S), dtype=torch.float64, device="cuda:0")
            torch.cuda.synchronize()
            ms = time_ms(lambda: b.segment_sum(offsets, out=out), args.seconds)
            nbytes = row_bytes + n_seg * S * 8 + (n_seg + 1) * 8
            line = dict(shape=name, rows=S, columns=length, dtype="f32" if dtype == L.F32 else "f64",
                        segment_length=seg_len, segments=n_seg, bytes=nbytes, ms=round(ms, 4),
                        gbps=round(nbytes / ms / 1e6, 1), copy_gbps=round(copy_gbps, 1),
                        copy_frac=round(nbytes / ms / 1e6 / copy_gbps, 3))
            del out
            lengths = (offsets[1:] - offsets[:-1]).unsqueeze(0).expand(S, -1).contiguous()  # (axis 1: one row per row)
            try:
                line["torch_segment_reduce_ms"] = round(time_ms(
                    lambda: torch.segment_reduce(rows, "sum", lengths=lengths, axis=1), args.seconds), 4)
            except Exception as e:  # (an unsupported size is part of the comparison)
                line["torch_segment_reduce_ms"] = f"failed: {type(e).__name__}: {str(e)[:120]}"
            torch.cuda.empty_cache()
            if seg is None:
                line["torch_sum_ms"] = round(time_ms(lambda: rows.sum(dim=1), args.seconds), 4)
            line.update(gpu=gpu, power_limit=power)
            print(json.dumps(line), flush=True)
            torch.cuda.empty_cache()
        del b, rows, tensors
        torch.cuda.empty_cache()
    ctx.sync()


if __name__ == "__main__":
    main()
