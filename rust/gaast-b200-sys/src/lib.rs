//! Raw bindings to `include/gaast_b200.h` -- the C ABI of the B200 batch evaluator that replaces
//! `SpecializedAst::eval` (gaast `src/eval.rs:12-115`) for device-resident batches.
//!
//! UNCOMPILED: no Rust toolchain exists in the image this repository is built in.  The block below
//! is kept in step with the header by `tests/test_rust_binding.py` (every exported symbol, its arity
//! and its scalar types; the size of every `#[repr(C)]` struct).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const GAAST_MAX_DIM: u32 = 16;
pub const GAAST_COMM_ID_BYTES: usize = 128;

/// gaast_status
pub const GAAST_OK: c_int = 0;
pub const GAAST_ERR_INVALID: c_int = 1;
pub const GAAST_ERR_UNSUPPORTED: c_int = 2; // Exponential / Logarithm: todo!() in eval.rs:112-113
pub const GAAST_ERR_PANIC: c_int = 3; // the reference would panic on this AST
pub const GAAST_ERR_NO_DEVICE: c_int = 4;
pub const GAAST_ERR_CUDA: c_int = 5;
pub const GAAST_ERR_OOM: c_int = 6;
pub const GAAST_ERR_JIT: c_int = 7;
pub const GAAST_ERR_SHAPE: c_int = 8;

/// gaast_op_kind
pub const GAAST_OP_ADD_INPUT: u32 = 0; // eval.rs:45-50
pub const GAAST_OP_MUL_TERMS: u32 = 1; // eval.rs:61-86
pub const GAAST_OP_NEG_GRADES: u32 = 2; // eval.rs:55-60, 87-102
pub const GAAST_OP_SCALAR_INV: u32 = 3; // eval.rs:103-110
pub const GAAST_OP_SCALAR_SQRT: u32 = 4;
// exp / log of a k-vector with a scalar square: this library's definition (eval.rs:112-113 is todo!() in gaast; the
// emitter of rust/patches/0002 keeps returning LowerError::Unsupported for those nodes until gaast defines them)
pub const GAAST_OP_EXP: u32 = 5;
pub const GAAST_OP_LOG: u32 = 6;

/// gaast_input_kind
pub const GAAST_INPUT_BATCH: u32 = 0;
pub const GAAST_INPUT_CONST: u32 = 1;

/// gaast_engine / gaast_arith / gaast_dtype
pub const GAAST_ENGINE_AUTO: c_int = 0;
pub const GAAST_ENGINE_TABLE: c_int = 1;
pub const GAAST_ENGINE_SPECIALIZED: c_int = 2;
pub const GAAST_ENGINE_DENSE_WARP: c_int = 3;
pub const GAAST_ARITH_FMA: c_int = 0;
pub const GAAST_ARITH_STRICT: c_int = 1;
// OR-ed into `arith`: f32 batches evaluated in binary64, each stored result rounded once
pub const GAAST_ARITH_F64: c_int = 2;
pub const GAAST_F64: c_int = 0;
pub const GAAST_F32: c_int = 1;
pub const GAAST_HOST_DEFAULT: c_int = 0;
pub const GAAST_HOST_WRITE_COMBINED: c_int = 1;
pub const GAAST_COMM_AUTO: c_int = 0;
pub const GAAST_COMM_NCCL: c_int = 1;
pub const GAAST_COMM_PEER: c_int = 2;
// flags of gaast_plan_kernel_source's `with_sum` argument
pub const GAAST_SRC_WITH_SUM: c_int = 1;
pub const GAAST_SRC_NO_STORE: c_int = 2;
pub const GAAST_SRC_F32: c_int = 4;

/// `IndividualCompMul` (ast/base_types.rs:46-55) with (grade, index) resolved to buffer slots.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct gaast_term {
    pub out: u16,
    pub a: u16,
    pub b: u16,
    pub flags: u16,
    pub coeff: f64,
} // 16 bytes

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct gaast_op {
    pub kind: u32,
    pub dst: u32,
    pub a: u32,
    pub b: u32,
    pub mask: u32,
    pub term_begin: u32,
    pub term_count: u32,
    pub reserved: u32,
} // 32 bytes

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct gaast_input_desc {
    pub kind: u32,
    pub grade_mask: u32,
    pub slot: u32,
    pub const_offset: u32,
} // 16 bytes

#[repr(C)]
pub struct gaast_plan_desc {
    pub n: u32,
    pub n_buffers: u32,
    pub buffer_masks: *const u32,
    pub n_inputs: u32,
    pub inputs: *const gaast_input_desc,
    pub n_const_values: u32,
    pub const_values: *const f64,
    pub n_ops: u32,
    pub ops: *const gaast_op,
    pub n_terms: u32,
    pub terms: *const gaast_term,
    pub n_slots: u32,
    pub reserved: u32,
} // 88 bytes

/// Opaque handles.
pub enum gaast_ctx {}
pub enum gaast_plan {}
pub enum gaast_batch {}
pub enum gaast_comm {}

/// `int64_t` of the header (the CSR offsets of gaast_batch_segment_sum).
pub type int64_t = i64;

#[link(name = "gaast_b200")]
extern "C" {
    pub fn gaast_last_error() -> *const c_char;
    pub fn gaast_reload_env();
    pub fn gaast_version() -> *const c_char;

    pub fn gaast_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut gaast_ctx) -> c_int;
    pub fn gaast_ctx_destroy(ctx: *mut gaast_ctx) -> c_int;
    pub fn gaast_ctx_sync(ctx: *mut gaast_ctx) -> c_int;
    pub fn gaast_host_alloc(bytes: usize, flags: c_int, out: *mut *mut c_void) -> c_int;
    pub fn gaast_host_free(p: *mut c_void) -> c_int;
    pub fn gaast_host_register(p: *mut c_void, bytes: usize) -> c_int;
    pub fn gaast_host_unregister(p: *mut c_void) -> c_int;
    pub fn gaast_ctx_stream(ctx: *mut gaast_ctx) -> *mut c_void;
    pub fn gaast_ctx_launch_count(ctx: *mut gaast_ctx) -> u64;

    pub fn gaast_plan_create(ctx: *mut gaast_ctx, desc: *const gaast_plan_desc, out: *mut *mut gaast_plan) -> c_int;
    pub fn gaast_plan_create_projected(ctx: *mut gaast_ctx, desc: *const gaast_plan_desc, root_present: *const *const u64, out: *mut *mut gaast_plan) -> c_int;
    pub fn gaast_plan_destroy(plan: *mut gaast_plan) -> c_int;
    pub fn gaast_plan_cost(plan: *const gaast_plan, broadcast_slots: u64, bytes_per_elem: *mut u64, flops_per_elem: *mut u64) -> c_int;
    pub fn gaast_plan_root_mask(plan: *const gaast_plan) -> u32;
    pub fn gaast_plan_dim(plan: *const gaast_plan) -> u32;
    pub fn gaast_plan_num_slots(plan: *const gaast_plan) -> u32;
    pub fn gaast_plan_slot_mask(plan: *const gaast_plan, slot: u32) -> u32;
    pub fn gaast_plan_kernel_source(plan: *mut gaast_plan, broadcast_slots: u64, arith: c_int, with_sum: c_int, buf: *mut c_char, cap: usize) -> usize;
    pub fn gaast_plan_kernel_source_sparse(plan: *mut gaast_plan, broadcast_slots: u64, arith: c_int, with_sum: c_int, present: *const *const u64, n_present: u32, buf: *mut c_char, cap: usize) -> usize;
    pub fn gaast_plan_precompile(plan: *mut gaast_plan, broadcast_slots: u64, arith: c_int, with_sum: c_int, store_out: c_int) -> c_int;
    pub fn gaast_plan_precompile_typed(plan: *mut gaast_plan, broadcast_slots: u64, arith: c_int, with_sum: c_int, store_out: c_int, dtype: c_int) -> c_int;
    pub fn gaast_plan_set_tuning(plan: *mut gaast_plan, elems_per_thread: c_int, variant: c_int) -> c_int;

    pub fn gaast_batch_alloc(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, broadcast: c_int, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_wrap(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, stride: u64, broadcast: c_int, grade_ptrs: *const *mut c_void, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_alloc_typed(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, broadcast: c_int, dtype: c_int, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_wrap_typed(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, stride: u64, broadcast: c_int, dtype: c_int, grade_ptrs: *const *mut c_void, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_alloc_sparse(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, broadcast: c_int, dtype: c_int, present: *const *const u64, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_wrap_sparse(ctx: *mut gaast_ctx, n: u32, grade_mask: u32, len: u64, stride: u64, broadcast: c_int, dtype: c_int, present: *const *const u64, grade_ptrs: *const *mut c_void, out: *mut *mut gaast_batch) -> c_int;
    pub fn gaast_batch_stored_rows(b: *const gaast_batch, grade: u32) -> u32;
    pub fn gaast_batch_dtype(b: *const gaast_batch) -> c_int;
    pub fn gaast_batch_free(b: *mut gaast_batch) -> c_int;
    pub fn gaast_batch_len(b: *const gaast_batch) -> u64;
    pub fn gaast_batch_stride(b: *const gaast_batch) -> u64;
    pub fn gaast_batch_grade_mask(b: *const gaast_batch) -> u32;
    pub fn gaast_batch_grade_ptr(b: *const gaast_batch, grade: u32) -> *mut c_void;
    pub fn gaast_batch_upload(b: *mut gaast_batch, grade: u32, host: *const f64, host_stride: u64) -> c_int;
    pub fn gaast_batch_download(b: *const gaast_batch, grade: u32, host: *mut f64, host_stride: u64) -> c_int;
    pub fn gaast_batch_upload_f32(b: *mut gaast_batch, grade: u32, host: *const f32, host_stride: u64) -> c_int;
    pub fn gaast_batch_download_f32(b: *const gaast_batch, grade: u32, host: *mut f32, host_stride: u64) -> c_int;
    pub fn gaast_batch_zero(b: *mut gaast_batch) -> c_int;
    pub fn gaast_batch_pack_records(b: *mut gaast_batch, first: u64, count: u64, records: *const c_void, record_mask: u32) -> c_int;
    pub fn gaast_batch_unpack_records(b: *const gaast_batch, first: u64, count: u64, records: *mut c_void, record_mask: u32) -> c_int;
    pub fn gaast_batch_upload_records(b: *mut gaast_batch, first: u64, count: u64, host_records: *const c_void, record_mask: u32) -> c_int;
    pub fn gaast_batch_download_records(b: *const gaast_batch, first: u64, count: u64, host_records: *mut c_void, record_mask: u32) -> c_int;
    pub fn gaast_batch_segment_sum(b: *const gaast_batch, dev_offsets: *const int64_t, n_segments: u64, dev_sums: *mut f64) -> c_int;

    pub fn gaast_eval(plan: *mut gaast_plan, inputs: *const *mut gaast_batch, n_inputs: u32, out: *mut gaast_batch, engine: c_int, arith: c_int) -> c_int;
    pub fn gaast_eval_sum(plan: *mut gaast_plan, inputs: *const *mut gaast_batch, n_inputs: u32, out: *mut gaast_batch, dev_sum: *mut f64, engine: c_int, arith: c_int) -> c_int;
    pub fn gaast_eval_host(plan: *mut gaast_plan, host_in: *const *const f64, in_masks: *const u32, in_broadcast: *const c_int, n_inputs: u32, len: u64, host_stride: u64, host_out: *mut f64, engine: c_int, arith: c_int) -> c_int;
    pub fn gaast_eval_host_f32(plan: *mut gaast_plan, host_in: *const *const f32, in_masks: *const u32, in_broadcast: *const c_int, n_inputs: u32, len: u64, host_stride: u64, host_out: *mut f32, engine: c_int, arith: c_int) -> c_int;

    pub fn gaast_comm_create(ctxs: *const *mut gaast_ctx, n: u32, out: *mut *mut gaast_comm) -> c_int;
    pub fn gaast_comm_unique_id(id: *mut u8) -> c_int;
    pub fn gaast_comm_create_rank(ctx: *mut gaast_ctx, n_ranks: u32, rank: u32, id: *const u8, out: *mut *mut gaast_comm) -> c_int;
    pub fn gaast_comm_size(comm: *const gaast_comm) -> u32;
    pub fn gaast_comm_transport(comm: *const gaast_comm) -> *const c_char;
    pub fn gaast_comm_set_transport(comm: *mut gaast_comm, transport: c_int) -> c_int;
    pub fn gaast_comm_allreduce_sum(comm: *mut gaast_comm, dev_sums: *const *mut f64, count: usize) -> c_int;
    pub fn gaast_comm_destroy(comm: *mut gaast_comm) -> c_int;

    pub fn gaast_diag_fp64_peak(ctx: *mut gaast_ctx, seconds: f64, tflops: *mut f64) -> c_int;
    pub fn gaast_diag_matrix_rep(n: u32, neg_mask: u32, shape: *mut i32, a: *const f64, b: *const f64, c: *mut f64) -> c_int;
    pub fn gaast_plan_last_kernel(plan: *const gaast_plan) -> *const c_char;
}
