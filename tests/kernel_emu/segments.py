"""TEST INFRASTRUCTURE: the per-segment sum kernels (csrc/device/segments.cu) on the CPU.

The device code of segments.cu -- from its chunk-size constant to the end of the span kernel, character for
character -- is compiled with g++ behind cuda_on_cpu.h and a small chunk size (GAAST_SEGMENT_CHUNK), so that every
segment layout the device meets at millions of columns (pieces at chunk edges, segments over many chunks, many
boundaries in one window of 32 columns) occurs at a few thousand.  `replay` is the documented order of the
additions in numpy: the kernels must match it bit for bit."""
from __future__ import annotations

import ctypes as C
import os
import re
import subprocess
import tempfile
from typing import Dict, Sequence

import numpy as np

from . import FLAGS, HERE

ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "gaast_b200", "csrc")

# what the kernels use beyond cuda_on_cpu.h: shuffles from any lane, warp votes, one atomic
PRELUDE = r"""
#include <algorithm>
#include <climits>
using std::min;
static uint64_t emu_seg_x[kEmuMaxThreads];
template <class T>
static inline T __shfl_sync(unsigned, T v, int src) {
    const int t = int(threadIdx.x), w = t >> 5;
    uint64_t bits = 0;
    std::memcpy(&bits, &v, sizeof(T));
    emu_seg_x[t] = bits;
    pthread_barrier_wait(&emu_warp_bar[w]);
    const uint64_t r = emu_seg_x[(w << 5) | (src & 31)];
    pthread_barrier_wait(&emu_warp_bar[w]);
    T out;
    std::memcpy(&out, &r, sizeof(T));
    return out;
}
static inline unsigned __ballot_sync(unsigned, bool p) {
    const int t = int(threadIdx.x), w = t >> 5;
    emu_seg_x[t] = p ? 1u : 0u;
    pthread_barrier_wait(&emu_warp_bar[w]);
    unsigned m = 0;
    for (int l = 0; l < 32; ++l) m |= unsigned(emu_seg_x[(w << 5) | l]) << l;
    pthread_barrier_wait(&emu_warp_bar[w]);
    return m;
}
static inline bool __any_sync(unsigned m, bool p) { return __ballot_sync(m, p) != 0u; }
static inline bool __all_sync(unsigned m, bool p) { return __ballot_sync(m, p) == 0xffffffffu; }
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) {
    return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST);
}
"""

_libs: Dict[int, C.CDLL] = {}
_tmp = None


def kernel_text() -> str:
    src = open(os.path.join(CSRC, "device", "segments.cu")).read()
    begin = src.index("#ifndef GAAST_SEGMENT_CHUNK")
    end = src.index("// ---- end of device code ----")
    text = src[begin:end]
    assert "asm" not in text, "segments.cu has inline PTX the host stand-in does not know"
    hpp = open(os.path.join(CSRC, "runtime.hpp")).read()
    row = re.search(r"struct RecordRow \{.*?\};", hpp, flags=re.S).group(0)
    return row + "\n" + text


def library(chunk: int) -> C.CDLL:
    global _tmp
    if chunk in _libs:
        return _libs[chunk]
    if _tmp is None:
        _tmp = tempfile.TemporaryDirectory(prefix="gaast_segments_emu_")
    cpp = os.path.join(_tmp.name, f"segments_{chunk}.cpp")
    with open(cpp, "w") as f:
        f.write('#include "cuda_on_cpu.h"\n' + PRELUDE + f"#define GAAST_SEGMENT_CHUNK {chunk}\n" + "namespace gaast {\n" +
                kernel_text() + "\n}  // namespace gaast\n" + '#include "segments_driver.inc"\n')
    so = os.path.join(_tmp.name, f"segments_{chunk}.so")
    cmd = ["g++", *[x for x in FLAGS if x != "-O0"], "-O1", "-shared", "-I", HERE, cpp, "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ rejected segments.cu:\n" + r.stderr[-4000:])
    lib = C.CDLL(so)
    lib.emu_segment_sum.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p,
                                    C.c_void_p]
    lib.emu_segment_sum.restype = C.c_int
    lib.emu_segment_chunk.restype = C.c_longlong
    assert lib.emu_segment_chunk() == chunk
    _libs[chunk] = lib
    return lib


class SegmentBatch:
    """Stored rows [S][length] laid out as gaast_batch_alloc lays them out (rows padded to 128 bytes, NaN in the
    padding), and the scratch a batch keeps between calls."""

    def __init__(self, rows: np.ndarray, chunk: int):
        self.S, self.length = rows.shape
        self.dtype = rows.dtype
        quantum = 128 // rows.dtype.itemsize
        stride = max(quantum, (self.length + quantum - 1) // quantum * quantum)
        self.buf = np.full((self.S, stride), np.nan, dtype=rows.dtype)
        self.buf[:, :self.length] = rows
        self.chunk = chunk
        nc = max(1, (self.length + chunk - 1) // chunk)
        self.scratch = np.zeros(32 + nc * 8 + 2 * nc * self.S * 8, dtype=np.uint8)  # segment_scratch_bytes

    def segment_sum(self, offsets: Sequence[int], sums: np.ndarray = None) -> np.ndarray:
        lib = library(self.chunk)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        if sums is None:
            sums = np.full((max(1, n), self.S), np.nan)
        ptrs = (C.c_ulonglong * self.S)(*[self.buf[r].ctypes.data for r in range(self.S)])
        rc = lib.emu_segment_sum(ptrs, self.S, int(self.dtype == np.float32), self.length, offsets.ctypes.data, n,
                                 sums.ctypes.data, self.scratch.ctypes.data)
        assert rc == 0, f"segment kernels: emulation fault {rc}"
        return sums[:n]


def _lane_tree(v):
    v = list(v)
    d = 1
    while d < 32:
        for i in range(0, 32, 2 * d):
            v[i] = v[i] + v[i + d]
        d *= 2
    return v[0]


def _pairwise(p):
    if len(p) == 1:
        return p[0]
    h = 1
    while h * 2 < len(p):
        h *= 2
    return _pairwise(p[:h]) + _pairwise(p[h:])


def replay(rows: np.ndarray, offsets: Sequence[int], chunk: int) -> np.ndarray:
    """The documented order of the additions (DESIGN.md 3.7) for valid offsets, in float64."""
    S, length = rows.shape
    x = rows.astype(np.float64)
    n = len(offsets) - 1
    out = np.zeros((n, S))
    for j in range(n):
        lo, hi = int(offsets[j]), int(offsets[j + 1])
        if hi <= lo:
            continue
        pieces = []
        c = lo
        while c < hi:
            e = min(hi, (c // chunk + 1) * chunk)
            pieces.append((c, e))
            c = e
        for r in range(S):
            sums = []
            for a, b in pieces:
                lanes = [0.0] * 32
                for col in range(a, b):
                    lanes[col % 32] = lanes[col % 32] + float(x[r, col])
                sums.append(_lane_tree(lanes))
            out[j, r] = _pairwise(sums)
    return out
