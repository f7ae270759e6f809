"""The five BASELINE.json workloads (and a few small extras) as expressions over
input slots.  Shared by bench.py, the tests and the build-time kernel cache.

Each workload's `build` takes one expression per input slot and combines them
with the reference's operators only, so the SAME function builds the product
expression (gaast_b200.expr) and, in the tests, the oracle's expression.
"""
from __future__ import annotations

from dataclasses import dataclass
from math import comb
from typing import Callable, Dict, List, Sequence, Tuple

import numpy as np

M = 1 << 20


@dataclass
class Workload:
    name: str
    title: str
    metric: List[float]                       # diagonal metric, e_i . e_i
    inputs: List[Tuple[Tuple[int, ...], bool]]  # per slot: (grades, broadcast)
    build: Callable                           # (*leaf_exprs) -> Expr
    batch: int                                # BASELINE batch length
    products: int                             # product nodes per expression (products/s = elements/s x this)
    bound: str = "hbm"                        # roofline that bounds it (SURVEY.md 8d)
    sum_root: bool = False                    # batch-sum node at the root (cfg5)

    @property
    def n(self) -> int:
        return len(self.metric)

    def rows(self, slot: int) -> int:
        return sum(comb(self.n, k) for k in self.inputs[slot][0])

    def broadcast_mask(self) -> int:
        m = 0
        for s, (_, bc) in enumerate(self.inputs):
            if bc:
                m |= 1 << s
        return m


def _cfg1(A, B, C):  # README expression D = <A + B*C>_2
    return (A + B * C).g(2)


def _cfg2(R, X):  # conformal rotor sandwich, grade-1 part
    return (R * X * R.rev()).g(1)


def _cfg2_full(R, X):
    return R * X * R.rev()


def _cfg3(A, B):  # full geometric product
    return A * B


def _cfg4(a, b, C):
    # Cached, reused sub-expression P = a ^ b; a grade-restricted outer and a
    # grade-restricted inner product, recombined: E = (P ^ C) (P . C).
    # (SURVEY.md proposed (P ^ C) + (P & C); the reference PANICS on that one:
    # Addition hands the full wanted set {0,4} to both children and the outer
    # product's maximal grade set {4} fails `includes`, specialize.rs:113-117.)
    P = a ^ b
    return (P.clone() ^ C) * (P & C)


def _cfg5(V, X):  # versor inverse + sandwich, grade-2 part
    return (V * X * V.vinv()).g(2)


def _full(n):
    return tuple(range(n + 1))


WORKLOADS: Dict[str, Workload] = {w.name: w for w in [
    Workload("cfg1", "G(3,0) <A + B*C>_2, A,B,C full multivectors", [1.0] * 3,
             [(_full(3), False)] * 3, _cfg1, 1 * M, 1),
    Workload("cfg2", "G(4,1) (R*X*~R).g(1), R one fixed rotor (broadcast), X grade-1 points", [1.0] * 4 + [-1.0],
             [((0, 2, 4), True), ((1,), False)], _cfg2, 64 * M, 2),
    Workload("cfg2_full", "G(4,1) R*X*~R without projection (root grades 1,3,5)", [1.0] * 4 + [-1.0],
             [((0, 2, 4), True), ((1,), False)], _cfg2_full, 64 * M, 2),
    Workload("cfg3", "G(6,0) A*B, full 64-component multivectors", [1.0] * 6,
             [(_full(6), False)] * 2, _cfg3, 16 * M, 1, bound="fp64"),
    Workload("cfg4", "G(10,0) P=a^b; (P^C)*(P&C), a,b vectors, C bivector", [1.0] * 10,
             [((1,), False), ((1,), False), ((2,), False)], _cfg4, 8 * M, 3),
    Workload("cfg5", "G(8,4) (V*X*V.vinv()).g(2), V vector, X bivector, + batch-sum", [1.0] * 8 + [-1.0] * 4,
             [((1,), False), ((2,), False)], _cfg5, 32 * M, 4, sum_root=True),
]}


def product_expr(w: Workload):
    """The workload as a gaast_b200.expr expression over Input slots."""
    from .expr import Input, mv
    leaves = [mv(Input(s, grades)) for s, (grades, _) in enumerate(w.inputs)]
    return w.build(*leaves)


def specialize(w: Workload):
    return product_expr(w).specialize(w.metric)


# ---- synthetic inputs (SURVEY.md 8d) ----------------------------------------------
def seed_of(w: Workload) -> int:
    if w.name in WORKLOADS:
        return 0x6AA57000 + sorted(WORKLOADS).index(w.name)
    return 0x6AA57100 + sum(ord(c) for c in w.name)  # ad-hoc workloads (bench.py's dense-warp entry)


def _vec_sq(metric, v):
    return sum(m * x * x for m, x in zip(metric, v))


def _gp_blades(metric, a: Dict[int, float], b: Dict[int, float]) -> Dict[int, float]:
    """Geometric product of two sparse multivectors keyed by blade bitmask
    (host-side helper to synthesise a rotor; not the evaluator)."""
    out: Dict[int, float] = {}
    for ba, va in a.items():
        for bb, vb in b.items():
            s, t = 0, ba >> 1
            while t:
                s += bin(t & bb).count("1")
                t >>= 1
            c = -1.0 if s & 1 else 1.0
            common, i = ba & bb, 0
            while common:
                if common & 1:
                    c *= metric[i]
                common >>= 1
                i += 1
            out[ba ^ bb] = out.get(ba ^ bb, 0.0) + va * vb * c
    return out


def _blades_to_grades(n: int, mvb: Dict[int, float], grades: Sequence[int]) -> Dict[int, np.ndarray]:
    of_grade: Dict[int, List[int]] = {k: [] for k in range(n + 1)}
    for b in range(1 << n):
        of_grade[bin(b).count("1")].append(b)
    return {k: np.array([mvb.get(b, 0.0) for b in of_grade[k]], dtype=np.float64) for k in grades}


def host_inputs(w: Workload, length: int, seed: int = None) -> List[Dict[int, np.ndarray]]:
    """Per slot {grade: [C(n,k), length]} (broadcast slots: [C(n,k), 1]), uniform(-1,1)."""
    rng = np.random.default_rng(seed_of(w) if seed is None else seed)
    n = w.n
    out: List[Dict[int, np.ndarray]] = []
    for s, (grades, bc) in enumerate(w.inputs):
        if w.name.startswith("cfg2") and s == 0:
            # a fixed unit rotor: product of 4 random unit non-null vectors
            R = {0: 1.0}
            for _ in range(4):
                while True:
                    v = rng.uniform(-1, 1, n)
                    q = _vec_sq(w.metric, v)
                    if abs(q) > 0.2:
                        break
                v = v / np.sqrt(abs(q))
                R = _gp_blades(w.metric, R, {1 << i: float(v[i]) for i in range(n)})
            g = _blades_to_grades(n, R, grades)
            out.append({k: g[k].reshape(-1, 1) for k in grades})
            continue
        cols = 1 if bc else length
        d = {k: rng.uniform(-1, 1, (comb(n, k), cols)) for k in grades}
        if w.name == "cfg5" and s == 0:
            # mixed signature: keep |V.V| >= 0.1 so that vinv is well conditioned
            v = d[1]
            met = np.array(w.metric).reshape(-1, 1)
            while True:
                q = (met * v * v).sum(0)
                bad = np.abs(q) < 0.1
                if not bad.any():
                    break
                v[:, bad] = rng.uniform(-1, 1, (n, int(bad.sum())))
        out.append(d)
    return out


def torch_inputs(w: Workload, length: int, device, seed: int = None):
    """Synthetic inputs generated on the device: per slot {grade: tensor [C(n,k), length]}."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed_of(w) if seed is None else seed)
    host = host_inputs(w, 4, seed)  # broadcast operands (and their constraints) come from the host recipe
    out = []
    for s, (grades, bc) in enumerate(w.inputs):
        if bc:
            out.append({k: torch.from_numpy(host[s][k][:, :1].copy()).to(device) for k in grades})
            continue
        d = {}
        for k in grades:
            t = torch.empty((comb(w.n, k), length), dtype=torch.float64, device=device)
            t.uniform_(-1.0, 1.0, generator=g)
            d[k] = t
        if w.name == "cfg5" and s == 0:
            met = torch.tensor(w.metric, dtype=torch.float64, device=device).reshape(-1, 1)
            v = d[1]
            for _ in range(64):
                q = (met * v * v).sum(0)
                bad = q.abs() < 0.1
                nbad = int(bad.sum())
                if nbad == 0:
                    break
                v[:, bad] = torch.empty((w.n, nbad), dtype=torch.float64, device=device).uniform_(-1.0, 1.0, generator=g)
        out.append(d)
    return out


# ---- build-time kernel cache --------------------------------------------------------
def precompile_variants(w: Workload):
    """The (arith, with_sum, store_out, dtype) calls of `w` whose kernels the build compiles ahead of time."""
    from . import _lib as L
    variants = [(L.ARITH_FMA, False, True, L.F64), (L.ARITH_STRICT, False, True, L.F64)]
    if w.sum_root:
        variants += [(L.ARITH_FMA, True, True, L.F64), (L.ARITH_FMA, True, False, L.F64)]
    # the f32 variant of the same plans (bench.py --dtype f32, tests/test_gpu_f32.py)
    variants += [(L.ARITH_FMA, False, True, L.F32), (L.ARITH_STRICT, False, True, L.F32)]
    if w.sum_root:
        variants += [(L.ARITH_FMA, True, True, L.F32)]
    # f32 batches evaluated in binary64 (tests/test_gpu_f32_wide.py, tools/f32_wide_bw.py)
    variants += [(L.ARITH_FMA | L.ARITH_F64, False, True, L.F32)]
    if w.sum_root:
        variants += [(L.ARITH_FMA | L.ARITH_F64, True, True, L.F32)]
    return variants


def precompile_all(verbose: bool = False, fresh: bool = True) -> int:
    """Generate + compile the specialised kernels of every workload (no device needed)."""
    import os
    import shutil
    from . import _lib as L
    from .device import Plan
    if fresh and not (os.environ.get("GAAST_TEST_HOOKS") and os.environ.get("GAAST_KERNEL_CACHE")):
        # entries are keyed by a hash of their source: drop the ones older generators left behind
        shutil.rmtree(os.path.join(os.path.dirname(os.path.abspath(__file__)), "kernel_cache"), ignore_errors=True)
    count = 0
    for w in WORKLOADS.values():
        plan = Plan(None, specialize(w))
        for arith, with_sum, store, dtype in precompile_variants(w):
            info = plan.precompile(w.broadcast_mask(), arith, with_sum, store, dtype)
            count += 1
            if verbose:
                mode = ('strict' if arith & L.ARITH_STRICT else 'fma') + ('|f64' if arith & L.ARITH_F64 else '')
                print(f"  {w.name:10s} {'f32' if dtype else 'f64'} arith={mode:6s} sum={int(with_sum)} "
                      f"store={int(store)}: {info}")
        plan.free()
    # bench.py also times cfg3 / cfg5 with their algebraic lowering switched off (variant bits 17 / 16)
    for name, variant, with_sum in (("cfg3", 131072, False), ("cfg5", 65536, True)):
        w = WORKLOADS[name]
        plan = Plan(None, specialize(w))
        plan.set_tuning(0, variant)
        info = plan.precompile(w.broadcast_mask(), L.ARITH_FMA, with_sum, True, L.F64)
        count += 1
        if verbose:
            print(f"  {name:10s} f64 arith=fma    sum={int(with_sum)} store=1 variant={variant}: {info}")
        plan.free()
    # the dense engine's kernels for full products (bench.py's dense entries, tests/test_gpu_dense_matrix.py): one
    # matrix-representation kernel per SHAPE of the representation (csrc/device/dense_matrix.cu), shared by every
    # signature of that shape, plus the term-by-term kernel of the benchmarked G(8,0) product
    from .expr import Input, mv as pmv
    dense = [([1.0] * 7, None, 0), ([1.0] * 6 + [-1.0], None, 0), ([1.0] * 4 + [-1.0] * 3, None, 0), ([1.0] * 8, None, 0),
             ([1.0] * 8, None, 1048576), ([1.0] * 9, None, 0), ([1.0] * 10, None, 0), ([1.0] * 11, None, 0),
             ([1.0] * 8 + [-1.0] * 4, tuple(range(0, 13, 2)), 0)]
    for metric, grades, variant in dense:
        n = len(metric)
        gr = tuple(range(n + 1)) if grades is None else grades
        plan = Plan(None, (pmv(Input(0, gr)) * pmv(Input(1, gr))).specialize(metric))
        if variant:
            plan.set_tuning(0, variant)
        info = plan.precompile(0, L.ARITH_FMA, False, True, L.F64)
        count += 1
        if verbose:
            print(f"  dense G({sum(m > 0 for m in metric)},{sum(m < 0 for m in metric)}) variant={variant}: {info}")
        plan.free()
    return count
