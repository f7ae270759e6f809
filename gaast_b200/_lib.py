"""ctypes binding of libgaast_b200.so (include/gaast_b200.h, gaast_b200_host.h).

The library is built in-tree by `python -m gaast_b200.build` (or
`__graft_entry__.build()`); importing this module fails loudly if it is
missing -- there is no Python or CPU fallback for the device path."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgaast_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m gaast_b200.build` "
        "(nvcc, sm_100a).  gaast_b200 has no fallback path.")

lib = C.CDLL(LIB_PATH)

u16, u32, u64, i64 = C.c_uint16, C.c_uint32, C.c_uint64, C.c_int64
vp = C.c_void_p

(OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_PANIC, ERR_NO_DEVICE, ERR_CUDA, ERR_OOM, ERR_JIT,
 ERR_SHAPE) = range(9)
STATUS_NAMES = ["OK", "INVALID", "UNSUPPORTED", "PANIC", "NO_DEVICE", "CUDA", "OOM", "JIT", "SHAPE"]

ENGINE_AUTO, ENGINE_TABLE, ENGINE_SPECIALIZED, ENGINE_DENSE_WARP = 0, 1, 2, 3
HOST_DEFAULT, HOST_WRITE_COMBINED = 0, 1
COMM_AUTO, COMM_NCCL, COMM_PEER = 0, 1, 2
ARITH_FMA, ARITH_STRICT = 0, 1
F64, F32 = 0, 1  # gaast_dtype

OP_ADD_INPUT, OP_MUL_TERMS, OP_NEG_GRADES, OP_SCALAR_INV, OP_SCALAR_SQRT, OP_EXP, OP_LOG = range(7)
INPUT_BATCH, INPUT_CONST = 0, 1
PROD_GEOMETRIC, PROD_OUTER, PROD_INNER, PROD_LCONTRACT, PROD_RCONTRACT = range(5)


class Term(C.Structure):
    _fields_ = [("out", u16), ("a", u16), ("b", u16), ("flags", u16), ("coeff", C.c_double)]


class Op(C.Structure):
    _fields_ = [("kind", u32), ("dst", u32), ("a", u32), ("b", u32), ("mask", u32),
                ("term_begin", u32), ("term_count", u32), ("reserved", u32)]


class InputDesc(C.Structure):
    _fields_ = [("kind", u32), ("grade_mask", u32), ("slot", u32), ("const_offset", u32)]


class PlanDesc(C.Structure):
    _fields_ = [("n", u32), ("n_buffers", u32), ("buffer_masks", C.POINTER(u32)),
                ("n_inputs", u32), ("inputs", C.POINTER(InputDesc)),
                ("n_const_values", u32), ("const_values", C.POINTER(C.c_double)),
                ("n_ops", u32), ("ops", C.POINTER(Op)),
                ("n_terms", u32), ("terms", C.POINTER(Term)),
                ("n_slots", u32), ("reserved", u32)]


class NodeInfo(C.Structure):
    _fields_ = [("kind", u32), ("child0", u32), ("child1", u32), ("scalar_op", u32),
                ("minimal_grade_set", u64), ("maximal_grade_set", u64), ("num_uses", u32),
                ("input_index", u32), ("n_terms", u32), ("reserved", u32)]


class CompMul(C.Structure):
    _fields_ = [("left_grade", u32), ("left_index", u32), ("right_grade", u32), ("right_index", u32),
                ("result_grade", u32), ("result_index", u32), ("coeff", C.c_double)]


GRADE_SELECTOR = C.CFUNCTYPE(u64, i64, i64, vp)
GRADE_FILTER = C.CFUNCTYPE(u64, u64, vp)


class GaastError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"[{STATUS_NAMES[status] if 0 <= status < len(STATUS_NAMES) else status}] {message}")
        self.status = status


def _proto(name, restype, *argtypes):
    f = getattr(lib, name)
    f.restype = restype
    f.argtypes = list(argtypes)
    return f


# Every symbol the two headers declare, with its prototype.  tests/test_abi.py
# checks this table against include/*.h.
PROTOTYPES = {
    # gaast_b200.h
    "gaast_last_error": (C.c_char_p,),
    "gaast_reload_env": (None,),
    "gaast_version": (C.c_char_p,),
    "gaast_ctx_create": (C.c_int, C.c_int, vp, C.POINTER(vp)),
    "gaast_ctx_destroy": (C.c_int, vp),
    "gaast_ctx_sync": (C.c_int, vp),
    "gaast_host_alloc": (C.c_int, C.c_size_t, C.c_int, C.POINTER(vp)),
    "gaast_host_free": (C.c_int, vp),
    "gaast_host_register": (C.c_int, vp, C.c_size_t),
    "gaast_host_unregister": (C.c_int, vp),
    "gaast_ctx_stream": (vp, vp),
    "gaast_ctx_launch_count": (u64, vp),
    "gaast_plan_create": (C.c_int, vp, C.POINTER(PlanDesc), C.POINTER(vp)),
    "gaast_plan_create_projected": (C.c_int, vp, C.POINTER(PlanDesc), C.POINTER(C.POINTER(u64)), C.POINTER(vp)),
    "gaast_plan_destroy": (C.c_int, vp),
    "gaast_plan_cost": (C.c_int, vp, u64, C.POINTER(u64), C.POINTER(u64)),
    "gaast_plan_root_mask": (u32, vp),
    "gaast_plan_dim": (u32, vp),
    "gaast_plan_num_slots": (u32, vp),
    "gaast_plan_slot_mask": (u32, vp, u32),
    "gaast_plan_kernel_source": (C.c_size_t, vp, u64, C.c_int, C.c_int, C.c_char_p, C.c_size_t),
    "gaast_plan_kernel_source_sparse": (C.c_size_t, vp, u64, C.c_int, C.c_int, C.POINTER(C.POINTER(u64)), u32, C.c_char_p,
                                        C.c_size_t),
    "gaast_plan_precompile": (C.c_int, vp, u64, C.c_int, C.c_int, C.c_int),
    "gaast_plan_precompile_typed": (C.c_int, vp, u64, C.c_int, C.c_int, C.c_int, C.c_int),
    "gaast_plan_set_tuning": (C.c_int, vp, C.c_int, C.c_int),
    "gaast_plan_last_kernel": (C.c_char_p, vp),
    "gaast_diag_fp64_peak": (C.c_int, vp, C.c_double, C.POINTER(C.c_double)),
    "gaast_diag_matrix_rep": (C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                              C.POINTER(C.c_double), C.POINTER(C.c_double)),
    "gaast_batch_alloc": (C.c_int, vp, u32, u32, u64, C.c_int, C.POINTER(vp)),
    "gaast_batch_wrap": (C.c_int, vp, u32, u32, u64, u64, C.c_int, C.POINTER(vp), C.POINTER(vp)),
    "gaast_batch_alloc_typed": (C.c_int, vp, u32, u32, u64, C.c_int, C.c_int, C.POINTER(vp)),
    "gaast_batch_wrap_typed": (C.c_int, vp, u32, u32, u64, u64, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp)),
    "gaast_batch_alloc_sparse": (C.c_int, vp, u32, u32, u64, C.c_int, C.c_int, C.POINTER(C.POINTER(u64)), C.POINTER(vp)),
    "gaast_batch_wrap_sparse": (C.c_int, vp, u32, u32, u64, u64, C.c_int, C.c_int, C.POINTER(C.POINTER(u64)),
                                C.POINTER(vp), C.POINTER(vp)),
    "gaast_batch_stored_rows": (u32, vp, u32),
    "gaast_batch_dtype": (C.c_int, vp),
    "gaast_batch_free": (C.c_int, vp),
    "gaast_batch_len": (u64, vp),
    "gaast_batch_stride": (u64, vp),
    "gaast_batch_grade_mask": (u32, vp),
    "gaast_batch_grade_ptr": (vp, vp, u32),
    "gaast_batch_upload": (C.c_int, vp, u32, vp, u64),
    "gaast_batch_download": (C.c_int, vp, u32, vp, u64),
    "gaast_batch_upload_f32": (C.c_int, vp, u32, vp, u64),
    "gaast_batch_download_f32": (C.c_int, vp, u32, vp, u64),
    "gaast_batch_zero": (C.c_int, vp),
    "gaast_batch_pack_records": (C.c_int, vp, u64, u64, vp, u32),
    "gaast_batch_unpack_records": (C.c_int, vp, u64, u64, vp, u32),
    "gaast_batch_upload_records": (C.c_int, vp, u64, u64, vp, u32),
    "gaast_batch_download_records": (C.c_int, vp, u64, u64, vp, u32),
    "gaast_eval": (C.c_int, vp, C.POINTER(vp), u32, vp, C.c_int, C.c_int),
    "gaast_eval_sum": (C.c_int, vp, C.POINTER(vp), u32, vp, vp, C.c_int, C.c_int),
    "gaast_eval_host": (C.c_int, vp, C.POINTER(vp), C.POINTER(u32), C.POINTER(C.c_int), u32, u64, u64, vp,
                        C.c_int, C.c_int),
    "gaast_eval_host_f32": (C.c_int, vp, C.POINTER(vp), C.POINTER(u32), C.POINTER(C.c_int), u32, u64, u64, vp,
                            C.c_int, C.c_int),
    "gaast_comm_create": (C.c_int, C.POINTER(vp), u32, C.POINTER(vp)),
    "gaast_comm_unique_id": (C.c_int, C.c_char_p),
    "gaast_comm_create_rank": (C.c_int, vp, u32, u32, C.c_char_p, C.POINTER(vp)),
    "gaast_comm_size": (u32, vp),
    "gaast_comm_transport": (C.c_char_p, vp),
    "gaast_comm_set_transport": (C.c_int, vp, C.c_int),
    "gaast_comm_allreduce_sum": (C.c_int, vp, C.POINTER(vp), C.c_size_t),
    "gaast_comm_destroy": (C.c_int, vp),
    # gaast_b200_host.h
    "gaast_expr_input": (vp, u32, u32),
    "gaast_expr_const": (vp, u32, u32, C.POINTER(C.c_double), C.c_size_t),
    "gaast_expr_scalar": (vp, C.c_double),
    "gaast_expr_basis_vector": (vp, u32, u32),
    "gaast_expr_clone": (vp, vp),
    "gaast_expr_free": (None, vp),
    "gaast_expr_add": (vp, vp, vp),
    "gaast_expr_sub": (vp, vp, vp),
    "gaast_expr_neg": (vp, vp),
    "gaast_expr_product": (vp, vp, vp, C.c_int),
    "gaast_expr_product_custom": (vp, vp, vp, GRADE_SELECTOR, vp),
    "gaast_expr_div_scalar": (vp, vp, C.c_double),
    "gaast_expr_rev": (vp, vp),
    "gaast_expr_ginvol": (vp, vp),
    "gaast_expr_conj": (vp, vp),
    "gaast_expr_exp": (vp, vp),
    "gaast_expr_log": (vp, vp),
    "gaast_expr_pow": (vp, vp, vp),
    "gaast_expr_sqrt": (vp, vp),
    "gaast_expr_g": (vp, vp, i64),
    "gaast_expr_gselect_mask": (vp, vp, u64),
    "gaast_expr_gselect": (vp, vp, GRADE_FILTER, vp),
    "gaast_expr_scal": (vp, vp, vp),
    "gaast_expr_norm_sq": (vp, vp),
    "gaast_expr_sinv": (vp, vp),
    "gaast_expr_vinv": (vp, vp),
    "gaast_specialize": (C.c_int, vp, u32, C.POINTER(C.c_double), C.POINTER(vp)),
    "gaast_spec_free": (None, vp),
    "gaast_spec_num_nodes": (u32, vp),
    "gaast_spec_root": (u32, vp),
    "gaast_spec_dim": (u32, vp),
    "gaast_spec_node": (C.c_int, vp, u32, C.POINTER(NodeInfo)),
    "gaast_spec_node_terms": (C.c_int, vp, u32, C.POINTER(CompMul), C.c_size_t),
    "gaast_spec_lower": (C.c_int, vp, C.POINTER(C.POINTER(PlanDesc))),
}

for _name, (_res, *_args) in PROTOTYPES.items():
    _proto(_name, _res, *_args)


def last_error() -> str:
    return (lib.gaast_last_error() or b"").decode()


def check(status: int):
    if status != OK:
        raise GaastError(status, last_error())


def check_ptr(p):
    if not p:
        raise GaastError(ERR_INVALID, last_error())
    return p
