"""Bandwidth of the record transposes (gaast_records_pack / gaast_records_unpack) on the device, one JSON line per shape.

    python tools/records_bw.py > profiles/records_bw.jsonl

Each shape is timed with CUDA events over `--reps` calls after a warm-up; every working set is well above the 126 MB
L2.  GB/s counts bytes read plus bytes written.  Beside it:
  copy_frac   the rate over that of a torch device-to-device copy of the same bytes, timed in the same process;
  torch_ms    what a caller does without this library's transpose: `records.t().contiguous()` (pack; the rows of
              each grade are then slices of the result) or `rows.t().contiguous()` (unpack; records wider than the
              stored rows: zero them, then scatter the rows' transpose into their columns);
  host_*      for the host path (page-locked records): gaast_batch_upload_records against the per-grade
              gaast_batch_upload of the same bytes already in SoA form, and against numpy's transpose + that upload.
The card's name and power limit (nvidia-smi, read only) are on every line."""
import argparse
import json
import os
import subprocess
import sys
import time
from math import comb

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gaast_b200 as g  # noqa: E402
from gaast_b200 import _lib as L  # noqa: E402
from gaast_b200.expr import grade_mask  # noqa: E402

M = 1 << 20
# name, n, batch grades, record grades, elements, dtype, stored components of grade 2 (sparse) or None, host-path elements
SHAPES = [
    ("cfg2_X", 5, (1,), (1,), 64 * M, L.F64, None, 16 * M),
    ("cfg5_X", 12, (2,), (2,), 32 * M, L.F64, None, 2 * M),
    ("cfg3_A", 6, tuple(range(7)), tuple(range(7)), 16 * M, L.F64, None, 0),
    ("G10_full", 10, tuple(range(11)), tuple(range(11)), 1 * M, L.F64, None, 0),
    ("G12_full", 12, tuple(range(13)), tuple(range(13)), 256 * 1024, L.F64, None, 0),
    ("cfg2_X_f32", 5, (1,), (1,), 64 * M, L.F32, None, 16 * M),
    ("cfg5_X_f32", 12, (2,), (2,), 32 * M, L.F32, None, 2 * M),
    ("G3_full_into_g2", 3, (2,), tuple(range(4)), 64 * M, L.F64, None, 0),
    ("cfg5_X_sparse_9of66", 12, (2,), (2,), 32 * M, L.F64, 9, 0),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # the numbers are still worth printing
        return f"unknown ({e})", "unknown"


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_ms(fn, reps):
    fn()
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--only", default="", help="comma-separated shape names")
    args = ap.parse_args()
    name_gpu, power = gpu_info()
    ctx = g.Ctx.on_torch_stream(0)
    for name, n, grades, rgrades, count, dtype, sparse_keep, host_count in SHAPES:
        if args.only and name not in args.only.split(","):
            continue
        es = 4 if dtype == L.F32 else 8
        tdt = torch.int32 if dtype == L.F32 else torch.int64
        K = sum(comb(n, k) for k in rgrades)
        mask = grade_mask(rgrades)
        if sparse_keep:
            idx = list(range(0, comb(n, 2), comb(n, 2) // sparse_keep))[:sparse_keep]
            bits = (L.u64 * 2)()
            for i in idx:
                bits[i // 64] |= 1 << (i % 64)
            ptrs = (L.C.POINTER(L.u64) * 1)(L.C.cast(bits, L.C.POINTER(L.u64)))
            out = L.vp()
            L.check(L.lib.gaast_batch_alloc_sparse(ctx._h, n, grade_mask(grades), count, 0, dtype, ptrs, L.C.byref(out)))
            b = g.DeviceBatch(out, ctx, n, keep=(bits,))
        else:
            b = g.DeviceBatch.alloc(ctx, n, grades, count, dtype=dtype)
        stored = sum(b.stored_rows(k) for k in grades)
        recs = torch.randint(-2**31, 2**31 - 1, (count, K * es // 4), dtype=torch.int32, device="cuda").view(tdt)
        out_recs = torch.empty_like(recs)
        pack = lambda: L.check(L.lib.gaast_batch_pack_records(b._h, 0, count, L.vp(recs.data_ptr()), mask))  # noqa: E731
        unpack = lambda: L.check(L.lib.gaast_batch_unpack_records(b._h, 0, count, L.vp(out_recs.data_ptr()), mask))  # noqa: E731
        pack_ms, unpack_ms = time_ms(pack, args.reps), time_ms(unpack, args.reps)
        pack_bytes = (count * K + count * stored) * es
        unpack_bytes = (count * stored + count * K) * es
        # a torch copy of the same bytes: half read, half written
        src = torch.empty(pack_bytes // 2, dtype=torch.uint8, device="cuda")
        dst = torch.empty_like(src)
        copy_ms = time_ms(lambda: dst.copy_(src), args.reps)
        copy_gbps = 2 * src.numel() / copy_ms / 1e6
        del src, dst
        rows = torch.empty((stored, count), dtype=tdt, device="cuda")
        torch_pack_ms = time_ms(lambda: recs.t().contiguous(), args.reps)
        if stored == K:
            torch_unpack_ms = time_ms(lambda: rows.t().contiguous(), args.reps)
        else:  # the records' other components are +0: zero them, then scatter the stored rows
            cols, off = [], 0
            for k in rgrades:
                if k in grades:
                    cols += [off + c for c in (idx if sparse_keep else range(comb(n, k)))]
                off += comb(n, k)
            cols = torch.tensor(cols, device="cuda")
            full = torch.empty((count, K), dtype=tdt, device="cuda")

            def torch_unpack():
                full.zero_()
                full[:, cols] = rows.t()
            torch_unpack_ms = time_ms(torch_unpack, args.reps)
            del full
        del rows
        line = dict(shape=name, n=n, batch_grades=list(grades), record_grades=list(rgrades), elements=count,
                    dtype="f32" if dtype == L.F32 else "f64", K_rec=K, stored_rows=stored,
                    pack_ms=round(pack_ms, 4), pack_gbps=round(pack_bytes / pack_ms / 1e6, 1),
                    unpack_ms=round(unpack_ms, 4), unpack_gbps=round(unpack_bytes / unpack_ms / 1e6, 1),
                    copy_gbps=round(copy_gbps, 1),
                    pack_copy_frac=round(pack_bytes / pack_ms / 1e6 / copy_gbps, 3),
                    unpack_copy_frac=round(unpack_bytes / unpack_ms / 1e6 / copy_gbps, 3),
                    torch_pack_ms=round(torch_pack_ms, 4), torch_unpack_ms=round(torch_unpack_ms, 4),
                    pack_vs_torch=round(torch_pack_ms / pack_ms, 2), unpack_vs_torch=round(torch_unpack_ms / unpack_ms, 2))
        del recs, out_recs
        b.free()
        torch.cuda.empty_cache()
        if host_count:
            fl = np.float32 if dtype == L.F32 else np.float64
            hb = g.DeviceBatch.alloc(ctx, n, grades, host_count, dtype=dtype)
            hrec = g.HostArray(host_count, K, dtype=fl)
            hrec.array[:] = np.random.default_rng(0).uniform(-1, 1, (host_count, K))
            soa = g.HostArray(K, host_count, dtype=fl)
            up = L.lib.gaast_batch_upload_f32 if dtype == L.F32 else L.lib.gaast_batch_upload
            off = 0
            soa_ptrs = []
            for k in grades:
                soa_ptrs.append((k, soa.array[off:off + comb(n, k)].ctypes.data))
                off += comb(n, k)

            def upload_records():
                L.check(L.lib.gaast_batch_upload_records(hb._h, 0, host_count, L.vp(hrec.array.ctypes.data), mask))
                ctx.sync()

            def upload_soa():
                for k, p in soa_ptrs:
                    L.check(up(hb._h, k, L.vp(p), host_count))
                ctx.sync()

            def transpose_and_upload():
                soa.array[:] = hrec.array.T
                upload_soa()

            rec_ms = host_ms(upload_records, 3)
            soa_ms = host_ms(upload_soa, 3)
            tr_ms = host_ms(transpose_and_upload, 2)
            line.update(host_elements=host_count, host_records_ms=round(rec_ms, 2), host_soa_upload_ms=round(soa_ms, 2),
                        host_numpy_transpose_upload_ms=round(tr_ms, 2), host_records_vs_soa=round(soa_ms / rec_ms, 3),
                        host_gbps=round(host_count * K * es / rec_ms / 1e6, 1))
            hrec.free()
            soa.free()
            hb.free()
        line.update(gpu=name_gpu, power_limit=power, reps=args.reps)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
