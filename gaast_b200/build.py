"""In-tree build of libgaast_b200.so (nvcc, sm_100a only).

    python -m gaast_b200.build [--force] [--no-precompile]

The shared library carries the C ABI of include/gaast_b200.h (device side) and
include/gaast_b200_host.h (host mirror of gaast's phases 1-3).  After linking,
the specialised kernels of the shipped workloads are generated and compiled
into gaast_b200/kernel_cache/ (NVRTC, no device needed), so that nothing
compiles at run time on the GPU box for them.
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libgaast_b200.so")
NVCC = os.environ.get("NVCC", shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")

SOURCES = [
    "common.cpp",
    "device_plan.cpp",
    "host/host_expr.cpp",
    "host/host_lower.cpp",
    "host/host_capi.cpp",
    "device/codegen.cpp",
    "device/jit.cpp",
    "device/comm.cu",
    "device/table_engine.cu",
    "device/dense_warp.cu",
    "device/dense_matrix.cu",
    "device/records.cu",
    "device/segments.cu",
    "device/runtime.cu",
    "device/host_pipeline.cu",
    "device/diag.cu",
]
HEADERS = ["common.hpp", "device_plan.hpp", "runtime.hpp", "eval_args.h", "host/host.hpp", "device/dense_warp_kernel.h", "device/dense_matrix_kernel.h",
           "../../include/gaast_b200.h", "../../include/gaast_b200_host.h"]

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC,-Wall,-Wextra",
          "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def _write_args_text():
    """eval_args.h pasted as a raw string literal for the code generator."""
    src = os.path.join(CSRC, "eval_args.h")
    dst = os.path.join(CSRC, "eval_args_text.inc")
    text = 'R"GAASTARGS(' + open(src).read() + ')GAASTARGS"\n'
    if not os.path.exists(dst) or open(dst).read() != text:
        with open(dst, "w") as f:
            f.write(text)
    # the dense-warp device code, pasted into the per-plan source NVRTC compiles
    src = os.path.join(CSRC, "device", "dense_warp_kernel.h")
    dst = os.path.join(CSRC, "device", "dense_warp_kernel_text.inc")
    text = 'R"GAASTDW(' + open(src).read() + ')GAASTDW"\n'
    if not os.path.exists(dst) or open(dst).read() != text:
        with open(dst, "w") as f:
            f.write(text)
    # ... and the matrix-representation kernel of the same engine (one NVRTC build per tile shape)
    src = os.path.join(CSRC, "device", "dense_matrix_kernel.h")
    dst = os.path.join(CSRC, "device", "dense_matrix_kernel_text.inc")
    text = 'R"GAASTDM(' + open(src).read() + ')GAASTDM"\n'
    if not os.path.exists(dst) or open(dst).read() != text:
        with open(dst, "w") as f:
            f.write(text)


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force: bool = False, verbose: bool = False) -> str:
    _write_args_text()
    os.makedirs(OBJ, exist_ok=True)
    hdr_time = _newest([os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(CSRC, "eval_args_text.inc")])
    jobs = []
    objs = []
    for rel in SOURCES:
        src = os.path.join(CSRC, rel)
        obj = os.path.join(OBJ, rel.replace("/", "_") + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time):
            cmd = [NVCC, *ARCH, *COMMON, "-c", src, "-o", obj]
            if rel.endswith(".cu"):
                cmd[1:1] = ["-Xptxas", "-v"] if verbose else []
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for cmd, r in ex.map(run, jobs):
                if verbose and (r.stdout or r.stderr):
                    print(r.stdout, r.stderr, file=sys.stderr)
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if jobs or not os.path.exists(LIB):
        cmd = [NVCC, *ARCH, "-shared", "-o", LIB, *objs, "-Xcompiler", "-fPIC", "-ldl", "-lpthread",
               "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return LIB


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--no-precompile", action="store_true")
    args = ap.parse_args(argv)
    lib = build(args.force, args.verbose)
    print("built", lib)
    if not args.no_precompile:
        from . import workloads
        n = workloads.precompile_all(verbose=True)
        print(f"kernel cache: {n} specialised kernels ready in {os.path.join(HERE, 'kernel_cache')}")


if __name__ == "__main__":
    main()
