/* gaast_b200.h -- C ABI of the B200-native batched evaluator for gaast's phase 4.
 *
 * This is the drop-in boundary: what a `gaast-b200-sys` Rust FFI crate binds
 * (INTEGRATION.md shows the `extern "C"` block).  It replaces, for BATCHES of
 * multivectors resident on the device, the reference's
 *
 *     SpecializedAst<T>::eval::<R>() -> R                 src/eval.rs:12-19
 *       store_in_cache / add_to_res                        src/eval.rs:21-115
 *       the term loop  res += l * r * coeff                src/eval.rs:77-83
 *     GradedData::grade_slice / GradedDataMut::*           src/graded.rs:43-79
 *
 * Everything here is plain C: opaque handles, pointers and sizes.  No call
 * unwinds; every call returns a gaast_status and records a message readable
 * with gaast_last_error().  There is NO CPU fallback: without a CUDA device
 * gaast_ctx_create() fails with GAAST_ERR_NO_DEVICE.
 *
 * Threading: handles are thread-compatible, not thread-safe (no internal locking
 * on the hot path): use one ctx per host thread / device.  A plan belongs to the
 * ctx it was created on and is NOT shareable between threads or streams: besides
 * its immutable description it owns per-call device scratch (batch-sum partials,
 * hoisted shared-operand values, workspaces) and its compiled kernels, all ordered
 * on the ctx stream.  Create one plan per ctx from the same description -- that is
 * cheap, the cubins come from the cache.  A plan's description is immutable after
 * creation and it may be evaluated any number of times with new inputs: the
 * "precompiled AST reused with new inputs" the reference's README:80-83 asks for.
 *
 * Allocation: gaast_eval / gaast_eval_sum allocate device scratch (and load their
 * kernel) only on the FIRST call of a plan with a given kernel variant -- engine,
 * arithmetic, dtype, broadcast pattern, alignment class -- sized for the largest
 * launch of that variant; the dense-warp engine also when the batch grows.  Every
 * later call only enqueues kernels on the ctx stream and can be captured in a CUDA
 * graph.  No environment variable is read on that path (see gaast_reload_env).
 */
#ifndef GAAST_B200_H
#define GAAST_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GAAST_MAX_DIM 16u /* vector-space dimension n; 2^n <= 65536 blade slots */

typedef enum gaast_status {
    GAAST_OK = 0,
    GAAST_ERR_INVALID = 1,     /* malformed argument / plan */
    GAAST_ERR_UNSUPPORTED = 2, /* Exponential / Logarithm: todo!() in eval.rs:112-113 */
    GAAST_ERR_PANIC = 3,       /* the reference would panic on this AST (unwrap/assert) */
    GAAST_ERR_NO_DEVICE = 4,   /* no CUDA device: the product path refuses to run */
    GAAST_ERR_CUDA = 5,
    GAAST_ERR_OOM = 6,
    GAAST_ERR_JIT = 7,         /* NVRTC unavailable or compilation failed */
    GAAST_ERR_SHAPE = 8        /* batch does not match what the plan expects */
} gaast_status;

/* ------------------------------------------------------------------ plan --
 * The flat, grade-blocked lowering of a SpecializedAst that gaast's
 * specialize.rs emits on the host (in this repo: gaast_b200_host.h does it).
 *
 * Buffers  = the reference's cache entries: the root and every product operand
 *            (eval.rs:21-33, 67-68), each with its minimal grade set.  A buffer
 *            stores, for the grades of its mask in ascending order, C(n,k)
 *            components each; a component's position in that concatenation is
 *            its SLOT.  Buffer 0 is the root.
 * Ops      = the reference's execution trace of add_to_res, in order.  Running
 *            them in order on zero-initialised buffers reproduces eval.rs
 *            exactly, including its in-place quirks (SURVEY.md Q1).
 * Terms    = IndividualCompMul (ast/base_types.rs:46-55) with (grade, index)
 *            already resolved to slots, in the reference's emission order
 *            (specialize.rs:162-183).
 */
typedef struct gaast_term {
    uint16_t out;   /* slot in the op's dst buffer   */
    uint16_t a;     /* slot in the op's left buffer  */
    uint16_t b;     /* slot in the op's right buffer */
    uint16_t flags; /* reserved, 0 */
    double coeff;   /* signed metric coefficient (algebra.rs:73-83) */
} gaast_term;       /* 16 bytes */

typedef enum gaast_op_kind {
    GAAST_OP_ADD_INPUT = 0,  /* dst += input[a] on grades `mask`      eval.rs:45-50 */
    GAAST_OP_MUL_TERMS = 1,  /* dst += sum terms(left=a, right=b)     eval.rs:61-86 */
    GAAST_OP_NEG_GRADES = 2, /* dst = -dst on grades `mask`           eval.rs:55-60,87-102 */
    GAAST_OP_SCALAR_INV = 3, /* dst[grade 0] = 1/dst[grade 0]         eval.rs:103-110 */
    GAAST_OP_SCALAR_SQRT = 4,/* dst[grade 0] = sqrt(dst[grade 0])     eval.rs:103-110 */
    /* The two ops below have NO reference evaluation: eval.rs:112-113 is `todo!()` for Exponential / Logarithm
     * (README.md:79 "versor exponentiation & logarithm" is on gaast's roadmap).  They implement this library's
     * own definition, consistent with the grade rules the reference already has (grade_set.rs:181-197: exp of
     * a single-graded k-vector holds grades {0, k}; log of <A>_0 + <A>_k holds grade k), for a k-vector B whose
     * square is a scalar (every blade: any vector, any bivector in dimension <= 3, the bivector of a simple
     * rotor ...), with q = <B B>_0 = sum_i (e_i)^2 B_i^2 over B's components:
     *     exp(B)     = c(q) + s(q) B     q < 0: cos x, sin x / x   q > 0: cosh x, sinh x / x   (x = sqrt|q|)   q = 0: 1, 1
     *     log(a + B) = t(a, q) B         q < 0: atan2(x, a) / x    q > 0: atanh(x / a) / x                     q = 0: 1 / a
     * (the scalar part ln|a + B| is not part of the reference's grade rule for log: 0 for a unit rotor).
     * `a` = source buffer (evaluated like a product operand, eval.rs:67-68), `mask` = the single grade k,
     * terms [term_begin, term_begin + term_count) = one per component of grade k in slot order with
     * a == b == that component's slot in the source buffer and coeff == the square of its basis blade. */
    GAAST_OP_EXP = 5,        /* dst += exp(B),      B = grade k of buffer a (the scalar part only if dst holds grade 0) */
    GAAST_OP_LOG = 6         /* dst += log(a0 + B), a0 = grade 0, B = grade k of buffer a */
} gaast_op_kind;

typedef struct gaast_op {
    uint32_t kind;       /* gaast_op_kind */
    uint32_t dst;        /* destination buffer */
    uint32_t a;          /* ADD_INPUT: input index; MUL_TERMS: left buffer */
    uint32_t b;          /* MUL_TERMS: right buffer */
    uint32_t mask;       /* ADD_INPUT / NEG_GRADES: grade mask */
    uint32_t term_begin; /* MUL_TERMS: range in `terms` */
    uint32_t term_count;
    uint32_t reserved;
} gaast_op;              /* 32 bytes */

typedef enum gaast_input_kind {
    GAAST_INPUT_BATCH = 0, /* bound at eval time: inputs[slot] */
    GAAST_INPUT_CONST = 1  /* literal carried by the plan (basis vectors, scalars) */
} gaast_input_kind;

typedef struct gaast_input_desc {
    uint32_t kind;         /* gaast_input_kind */
    uint32_t grade_mask;   /* grades the GradedObj holds (its Graded::grade_set) */
    uint32_t slot;         /* BATCH: index into the `inputs` array given to eval */
    uint32_t const_offset; /* CONST: first value in `const_values` (grades ascending) */
} gaast_input_desc;

typedef struct gaast_plan_desc {
    uint32_t n;                       /* vector-space dimension */
    uint32_t n_buffers;
    const uint32_t* buffer_masks;     /* [n_buffers] minimal grade sets; [0] = root */
    uint32_t n_inputs;
    const gaast_input_desc* inputs;   /* [n_inputs] */
    uint32_t n_const_values;
    const double* const_values;
    uint32_t n_ops;
    const gaast_op* ops;              /* [n_ops] in reference execution order */
    uint32_t n_terms;
    const gaast_term* terms;          /* [n_terms] */
    uint32_t n_slots;                 /* number of distinct BATCH slots eval expects */
    uint32_t reserved;
} gaast_plan_desc;

/* ------------------------------------------------------------- handles ---- */
typedef struct gaast_ctx gaast_ctx;     /* one device + one stream */
typedef struct gaast_plan gaast_plan;   /* validated plan + its device tables + compiled kernels */
typedef struct gaast_batch gaast_batch; /* device-resident SoA batch: one f64 (or f32) array per grade */

/* Evaluation engines (all run on the GPU; there is no host engine). */
typedef enum gaast_engine {
    GAAST_ENGINE_AUTO = 0,        /* specialised when the plan can be specialised (NVRTC or the kernel cache),
                                     the dense engine for large dense product chains in G(7..12), else table */
    GAAST_ENGINE_TABLE = 1,       /* generic table-driven kernels compiled into this library */
    GAAST_ENGINE_SPECIALIZED = 2, /* straight-line sm_100a kernel generated from the plan */
    GAAST_ENGINE_DENSE_WARP = 3   /* chains of dense products of multivectors in G(n), +-1 metric, FMA arithmetic
                                     (GAAST_ERR_UNSUPPORTED for any other plan).  Chains of GEOMETRIC products,
                                     n = 7..12: the real matrix representation of the algebra on the FP64 tensor
                                     cores, 2^(n+MX) multiplications instead of 4^n (gaast_diag_matrix_rep; its
                                     rounding error is bounded norm-wise, not per component: tuning variant bit 20
                                     selects the term-by-term kernel instead).  Outer products, contractions and
                                     mixed chains, n = 7..10: one warp per multivector, one DFMA per term.  AUTO
                                     picks the engine when such a plan is too large to specialise. */
} gaast_engine;

typedef enum gaast_arith {
    GAAST_ARITH_FMA = 0,   /* one DFMA per term (default; within 1e-12 of eval.rs) */
    GAAST_ARITH_STRICT = 1 /* (l*r)*coeff then add, reference order: bit-identical to eval.rs */
} gaast_arith;

/* Scalar type of a batch.  f64 is the reference's type (eval.rs works on f64 only) and the
 * type every parity claim is made in.  f32 is this library's reduced-precision variant
 * (SURVEY.md 8f rank 4): the same plans evaluated in IEEE binary32 -- half the HBM bytes.
 * All batches of one gaast_eval call must share one dtype; plan literals and term
 * coefficients are rounded to binary32; batch sums still accumulate in f64. */
typedef enum gaast_dtype {
    GAAST_F64 = 0,
    GAAST_F32 = 1
} gaast_dtype;

/* Last error message of the calling thread (never NULL). */
const char* gaast_last_error(void);
/* The library reads its tuning / diagnostic environment variables (GAAST_HOST_CHUNK_MIB, GAAST_GRID_MULT,
 * GAAST_NO_KERNEL_CACHE, GAAST_NVRTC, GAAST_NCCL, ... and, only together with GAAST_TEST_HOOKS=1,
 * GAAST_KERNEL_CACHE) ONCE, at the first gaast_ctx_create / first use -- never on the evaluation path.
 * This re-reads them: for tests and timing experiments, not thread-safe against running evaluations. */
void gaast_reload_env(void);
/* Library version string, and the CUDA arch the embedded kernels were built for. */
const char* gaast_version(void);

/* ctx: `stream` is a cudaStream_t (or NULL for a private non-blocking stream). */
gaast_status gaast_ctx_create(int device, void* stream, gaast_ctx** out);
gaast_status gaast_ctx_destroy(gaast_ctx* ctx);
gaast_status gaast_ctx_sync(gaast_ctx* ctx);
void* gaast_ctx_stream(gaast_ctx* ctx);
/* Counts kernel launches issued by this library on `ctx` since creation. */
uint64_t gaast_ctx_launch_count(gaast_ctx* ctx);

/* plan: validates `desc` (copying everything it needs) and uploads its tables.
 * ctx may be NULL for an offline plan (kernel_source / precompile only). */
gaast_status gaast_plan_create(gaast_ctx* ctx, const gaast_plan_desc* desc, gaast_plan** out);
/* A projected plan: the same expression, keeping only chosen root components (a component-level counterpart of
 * the grade projection .g(k)); the others are zero, and the result is a SPARSE output batch (gaast_batch_alloc_sparse
 * with the same bitmaps).  root_present[i] describes the i-th grade of the root mask, ascending: a bitmap of C(n,k)
 * bits in gaast_batch_alloc_sparse's convention (bit c of word c / 64 = component c is stored), or NULL for the
 * whole grade.  Normalised as a batch's bitmaps are: bits past C(n,k) are ignored, a grade with every bit set is
 * dense, a grade with none stores nothing.  Selecting every component gives a plan indistinguishable from
 * gaast_plan_create's.  A projection that stores no component at all is GAAST_ERR_SHAPE, a NULL root_present
 * GAAST_ERR_INVALID; every other check is gaast_plan_create's.  ctx == NULL gives an offline plan (kernel_source /
 * precompile then return and compile the projected kernels).
 *   - gaast_eval / gaast_eval_sum accept only an output batch that matches: the same dimension, exactly the root grade
 *     set, not broadcast, and per grade the same stored components (dense where the whole grade is selected).  Any
 *     other output batch is GAAST_ERR_SHAPE, a dense one too when some grade is only partly selected.
 *   - The kernels never compute a term that feeds only dropped components.  In GAAST_ARITH_STRICT each stored
 *     component is bit-identical to the same component of the unprojected plan, on the specialised and the table
 *     engine (every output keeps the reference's term order).
 *   - gaast_eval_sum writes one double per STORED root component, in the output batch's stored-row order (grades
 *     ascending, stored components ascending), with `out` present or NULL; an empty batch zeroes that many doubles.
 *   - GAAST_ENGINE_DENSE_WARP is GAAST_ERR_UNSUPPORTED (AUTO never picks it for a projected plan), and so are
 *     gaast_eval_host / _f32: their pipeline allocates dense output batches. */
gaast_status gaast_plan_create_projected(gaast_ctx* ctx, const gaast_plan_desc* desc, const uint64_t* const* root_present,
                                         gaast_plan** out);
gaast_status gaast_plan_destroy(gaast_plan* plan);
/* Algorithmic bytes and flops per batch element (SURVEY.md 8d), for f64 batches (f32: half the bytes): 8 x (f64 read
 * from non-broadcast inputs in the grades the plan reads + f64 written in the
 * root grades -- for a projected plan the stored root components only) and 2 x terms (the reference's terms: it has
 * no projection, so a projected plan reports the flops of the whole expression).  `broadcast_slots` bit s = slot s
 * is broadcast. */
gaast_status gaast_plan_cost(const gaast_plan* plan, uint64_t broadcast_slots, uint64_t* bytes_per_elem,
                             uint64_t* flops_per_elem);
uint32_t gaast_plan_root_mask(const gaast_plan* plan);
uint32_t gaast_plan_dim(const gaast_plan* plan);
uint32_t gaast_plan_num_slots(const gaast_plan* plan);
/* Grades of batch slot `slot` that the plan actually reads. */
uint32_t gaast_plan_slot_mask(const gaast_plan* plan, uint32_t slot);
/* CUDA source of the specialised kernel for this plan (for inspection / offline
 * nvcc -Xptxas -v / the CPU run of the generated text in tests/kernel_emu); returns the length, copies at most `cap`
 * bytes (NUL-terminated).  `with_sum` is a set of GAAST_SRC_* flags: 0 / 1 keep their meaning (plain kernel / fused
 * batch-sum); GAAST_SRC_NO_STORE = the kernel gaast_eval_sum launches with out == NULL (sums only),
 * GAAST_SRC_F32 = the kernel of the f32 variant. */
#define GAAST_SRC_WITH_SUM 1
#define GAAST_SRC_NO_STORE 2
#define GAAST_SRC_F32 4
size_t gaast_plan_kernel_source(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, char* buf,
                                size_t cap);
/* The same for inputs in sparse per-grade storage (gaast_batch_alloc_sparse): present[i] is the presence bitmap of the
 * i-th (slot, grade) array the plan reads -- slots in order, within a slot the grades of gaast_plan_slot_mask in
 * ascending order -- or NULL where that array is dense; n_present = the number of such arrays. */
size_t gaast_plan_kernel_source_sparse(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum,
                                       const uint64_t* const* present, uint32_t n_present, char* buf, size_t cap);
/* Generates and compiles the specialised kernel into the in-tree cubin cache
 * without a device (the plan may have been created with ctx == NULL).  Used
 * by the build step so that the shipped workloads never compile at run time. */
gaast_status gaast_plan_precompile(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, int store_out);
/* The same for the kernels of a given gaast_dtype (gaast_plan_precompile = GAAST_F64). */
gaast_status gaast_plan_precompile_typed(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, int store_out,
                                         int dtype);
/* Tuning knobs of the specialised engine: elements per thread (0 = choose,
 * 1, or 2 = 128-bit accesses) and emission-policy bits (0 = choose).  The bits that switch an algebraic
 * lowering OFF (each replaces sums over an output's own terms by a re-associated form, FMA arithmetic only):
 * 2048 shared-operand linear map, 65536 reflection form of a vector sandwich, 131072 matrix form of a full G(6)
 * product, 1048576 matrix-representation kernel of the dense engine. */
gaast_status gaast_plan_set_tuning(gaast_plan* plan, int elems_per_thread, int variant);

/* batch: the device-resident counterpart of GradedData (graded.rs:43-47): for
 * every grade k of `grade_mask` one f64 array of C(n,k) rows x `len` columns,
 * batch-innermost (element i of component c at rows[c * stride + i]).
 * len == 1 with broadcast != 0 makes a shared operand (batch stride 0). */
gaast_status gaast_batch_alloc(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                               gaast_batch** out);
/* Wrap caller-owned device arrays (e.g. another library's allocation): one
 * pointer per grade of the mask, ascending, each [C(n,k)][stride] f64. */
gaast_status gaast_batch_wrap(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                              int broadcast, void* const* grade_ptrs, gaast_batch** out);
/* The same two constructors with an explicit scalar type (gaast_dtype); the arrays are then
 * [C(n,k)][stride] of that type. */
gaast_status gaast_batch_alloc_typed(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                                     int dtype, gaast_batch** out);
gaast_status gaast_batch_wrap_typed(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                                    int broadcast, int dtype, void* const* grade_ptrs, gaast_batch** out);
/* Sparse per-grade storage (the reference's README.md:102-104 caveat: "one array per grade imposes a dense
 * storage whatever the grade; a sparse storage for some grades would be necessary for higher-dimension
 * spaces").  A sparse batch stores, for grade k, only SOME of the C(n,k) components; the others are zero for
 * every element.  present[i] (i-th grade of the mask, ascending) is a bitmap of C(n,k) bits -- bit c of word
 * c / 64 set = component c is stored -- or NULL for a dense grade; the grade's array is then
 * [stored rows][stride], rows in ascending component order (uploads / downloads / wrapped pointers use that
 * compact shape; gaast_batch_stored_rows gives its height).  Input batches only: a kernel is specialised for the
 * sparsity pattern it is given -- loads of absent components and every term that reads them disappear -- so
 * sparse batches need the specialised engine (GAAST_ENGINE_AUTO or _SPECIALIZED; GAAST_ERR_UNSUPPORTED on the
 * table and dense-warp engines), in either arithmetic. */
gaast_status gaast_batch_alloc_sparse(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                                      int dtype, const uint64_t* const* present, gaast_batch** out);
gaast_status gaast_batch_wrap_sparse(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                                     int broadcast, int dtype, const uint64_t* const* present, void* const* grade_ptrs,
                                     gaast_batch** out);
uint32_t gaast_batch_stored_rows(const gaast_batch* b, uint32_t grade);
int gaast_batch_dtype(const gaast_batch* b);
gaast_status gaast_batch_free(gaast_batch* b);
uint64_t gaast_batch_len(const gaast_batch* b);
uint64_t gaast_batch_stride(const gaast_batch* b);
uint32_t gaast_batch_grade_mask(const gaast_batch* b);
/* Device pointer of grade k's [C(n,k)][stride] array (GradedData::grade_slice). */
void* gaast_batch_grade_ptr(const gaast_batch* b, uint32_t grade);
/* Stream-ordered copies of one grade: host array is [C(n,k)][host_stride]. */
gaast_status gaast_batch_upload(gaast_batch* b, uint32_t grade, const double* host, uint64_t host_stride);
gaast_status gaast_batch_download(const gaast_batch* b, uint32_t grade, double* host, uint64_t host_stride);
/* The same copies for f32 batches (GAAST_ERR_SHAPE on a dtype mismatch, both ways). */
gaast_status gaast_batch_upload_f32(gaast_batch* b, uint32_t grade, const float* host, uint64_t host_stride);
gaast_status gaast_batch_download_f32(const gaast_batch* b, uint32_t grade, float* host, uint64_t host_stride);
/* GradedDataMut::init_null_mv: zero every grade. */
gaast_status gaast_batch_zero(gaast_batch* b);

/* Element-major records: one multivector stored contiguously, as a GradedData or a Vec<[f64; K]> holds it.  A record
 * of `record_mask` is the components of its grades, grades ascending and components in the algebra's order within a
 * grade (the batch's slot order for that mask), K = sum over its grades of C(n,k) scalars of the batch's dtype.
 * Records are packed without gaps: record j (batch column first + j) starts at scalar j * K.  The record scalar type
 * is the batch's, so the pointers are untyped; scalars are copied bit for bit (-0.0, subnormals, NaN payloads).
 * GAAST_ERR_SHAPE when record_mask is empty or lacks a grade of the batch, when first + count > len, or when a
 * broadcast batch is given anything but first = 0, count = 1; GAAST_ERR_INVALID for a null batch, or a null pointer with count > 0.
 * count == 0 returns GAAST_OK and launches nothing.  The first call for a given record_mask builds the batch's
 * row map for it (a device table freed by gaast_batch_free); every later call only enqueues its kernel(s) on the
 * ctx stream and can be captured in a CUDA graph. */
/* Device records -> batch columns [first, first + count).  `records` is device memory of the batch's device (or
 * managed memory) holding `count` records of record_mask, which must include every grade of the batch; another
 * pointer is GAAST_ERR_INVALID, checked before any launch.  Components the batch does not store (other grades, absent
 * components of a sparse grade) are ignored.  One kernel launch on the ctx stream. */
gaast_status gaast_batch_pack_records(gaast_batch* b, uint64_t first, uint64_t count, const void* records,
                                      uint32_t record_mask);
/* Batch columns [first, first + count) -> `count` device records of record_mask.  EVERY component of every record is
 * written: the batch's value where it stores one, +0 elsewhere (the element as a multivector of record_mask). */
gaast_status gaast_batch_unpack_records(const gaast_batch* b, uint64_t first, uint64_t count, void* records,
                                        uint32_t record_mask);
/* The same from / to host memory (pageable or page-locked), through a device staging buffer owned by the ctx, in
 * chunks of GAAST_HOST_CHUNK_MIB: per chunk a copy and a kernel launch.  Stream-ordered like gaast_batch_upload /
 * _download: synchronise the ctx before reading downloaded records or reusing uploaded ones in page-locked memory. */
gaast_status gaast_batch_upload_records(gaast_batch* b, uint64_t first, uint64_t count, const void* host_records,
                                        uint32_t record_mask);
gaast_status gaast_batch_download_records(const gaast_batch* b, uint64_t first, uint64_t count, void* host_records,
                                          uint32_t record_mask);

/* eval: out[i] = expr(inputs[0][i], inputs[1][i], ...) for i in [0, len).
 * `inputs` has plan.n_slots entries; `out` must carry exactly the plan's root
 * grade set (SURVEY.md Q3).  Stream-ordered, asynchronous. */
gaast_status gaast_eval(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out,
                        int engine, int arith);

/* Batch-sum node (no reference definition: gaast has no batches): evaluates the
 * plan and reduces the root over the batch on the device, writing
 * sum_i out[i] as [root comps] f64 to `dev_sum` (device memory; a projected plan: [stored root comps]).  The
 * reduction is fused in the kernel epilogue; per-CTA partials are then added
 * in a fixed order, so the result is deterministic for a given launch shape.
 * `out` may be NULL to skip materialising the per-element result. */
gaast_status gaast_eval_sum(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out,
                            double* dev_sum, int engine, int arith);

/* Page-locked host memory for the host-array entry points (gaast_eval_host, gaast_batch_upload /
 * _download).  The reference keeps its multivectors in ordinary Rust allocations (`GradeMapMV`: a
 * HashMap<Grade, Vec<f64>>, src/graded.rs:174); a caller that wants the copies of gaast_eval_host to overlap either
 * allocates its arrays here or pins the ones it has (gaast_host_register takes any allocation, e.g.
 * the buffer of a Vec<f64>; it must be unregistered before it is freed).  Memory is pinned for every
 * device of the process.  GAAST_HOST_WRITE_COMBINED asks for write-combined pages: for arrays the host
 * only WRITES (inputs) -- reading them back from the CPU is very slow. */
#define GAAST_HOST_DEFAULT 0
#define GAAST_HOST_WRITE_COMBINED 1
gaast_status gaast_host_alloc(size_t bytes, int flags, void** out);
gaast_status gaast_host_free(void* p);
gaast_status gaast_host_register(void* p, size_t bytes);
gaast_status gaast_host_unregister(void* p);

/* End-to-end convenience used for the `e2e` measurement: host arrays in, host
 * arrays out, chunked so that H2D, kernels and D2H overlap.  host_in[s] points
 * to [comps of slot s][host_stride] (grades of in_masks[s] ascending), or, for a
 * broadcast slot, to [comps of slot s] contiguous values; host_out is
 * [root comps][host_stride].  Pinned (page-locked) host memory is needed for the
 * copies to overlap; pageable arrays give the same result, but the driver then
 * stages every copy and the three streams serialise.  Synchronous: returns when
 * host_out is complete.  On an error all copies already issued are drained before
 * the call returns, so the caller may release its arrays. */
gaast_status gaast_eval_host(gaast_plan* plan, const double* const* host_in, const uint32_t* in_masks,
                             const int* in_broadcast, uint32_t n_inputs, uint64_t len, uint64_t host_stride,
                             double* host_out, int engine, int arith);

/* The same pipeline for binary32 host arrays (the f32 variant; half the PCIe traffic). */
gaast_status gaast_eval_host_f32(gaast_plan* plan, const float* const* host_in, const uint32_t* in_masks,
                                 const int* in_broadcast, uint32_t n_inputs, uint64_t len, uint64_t host_stride,
                                 float* host_out, int engine, int arith);

/* ------------------------------------------------------------------ comm --
 * Multi-GPU (SURVEY.md 8e): batch elements are independent, so a batch is sharded into
 * contiguous slices, one per device, and every device evaluates its slice with its own ctx /
 * plan / batches -- no communication.  The ONE collective of the path is the all-reduce of the
 * batch-sum vector gaast_eval_sum leaves on each device (66 doubles for the G(8,4) workload):
 * a kernel of this library over NVLink / NVSwitch peer memory (gaast_comm_transport below), NCCL
 * for the set-up and as the fallback.  NCCL is loaded with dlopen("libnccl.so.2"):
 * GAAST_ERR_UNSUPPORTED if it is not installed.  gaast has no counterpart (it is single-threaded and batch-less). */
typedef struct gaast_comm gaast_comm;
#define GAAST_COMM_ID_BYTES 128u
/* One process driving n devices of one node: ctxs[i] is rank i (ncclCommInitAll). */
gaast_status gaast_comm_create(gaast_ctx* const* ctxs, uint32_t n, gaast_comm** out);
/* One process per device: rank 0 draws an id (GAAST_COMM_ID_BYTES bytes), the caller ships it to
 * the other processes by its own means, every process then joins with its ctx and rank. */
gaast_status gaast_comm_unique_id(unsigned char* id);
gaast_status gaast_comm_create_rank(gaast_ctx* ctx, uint32_t n_ranks, uint32_t rank, const unsigned char* id,
                                    gaast_comm** out);
uint32_t gaast_comm_size(const gaast_comm* comm);
/* How gaast_comm_allreduce_sum moves its vector.  "peer": this library's own one-shot all-reduce over NVLink /
 * NVSwitch peer memory -- one kernel launch per device; every rank stores its vector into every peer's mailbox
 * (cudaDeviceEnablePeerAccess within a process, CUDA IPC between processes), raises a flag, waits for the others'
 * flags and adds the contributions in rank order, so the total is bit-identical on every rank; vectors of up to 512
 * doubles.  "nccl": ncclAllReduce.  A communicator uses "peer" whenever every rank could map every other (the ranks
 * agree on this at creation; GAAST_COMM=nccl in the environment opts out) and falls back to NCCL otherwise, or for
 * longer vectors.  gaast_comm_set_transport overrides per communicator -- every rank must make the same call;
 * GAAST_COMM_PEER returns GAAST_ERR_UNSUPPORTED when peer memory is not available. */
#define GAAST_COMM_AUTO 0
#define GAAST_COMM_NCCL 1
#define GAAST_COMM_PEER 2
const char* gaast_comm_transport(const gaast_comm* comm);
gaast_status gaast_comm_set_transport(gaast_comm* comm, int transport);
/* In place: dev_sums[i] addresses `count` doubles on the i-th LOCAL device of the communicator (all
 * of them after gaast_comm_create, exactly one after gaast_comm_create_rank); afterwards every
 * device holds the element-wise total over all ranks.  Ordered on each ctx's stream, asynchronous; with
 * the peer transport a launch carries no host-side state (the epoch lives in device memory) and may be
 * captured in a CUDA graph.  Every rank must issue the same sequence of all-reduces. */
gaast_status gaast_comm_allreduce_sum(gaast_comm* comm, double* const* dev_sums, size_t count);
gaast_status gaast_comm_destroy(gaast_comm* comm);

/* Diagnostic: the FP64 FMA-pipe throughput of ctx's device in TFLOP/s, measured by running independent
 * DFMA chains (64 DFMA / clk / SM is the pipe's limit) for about `seconds` of device time on the ctx
 * stream.  The roofline denominator of the compute-bound workloads, taken on the same box under the same
 * conditions as the kernel: a short call (0.02) gives the burst figure, a long one (0.5) the sustained,
 * power-capped one.  Synchronous. */
gaast_status gaast_diag_fp64_peak(gaast_ctx* ctx, double seconds, double* tflops);

/* Diagnostic, no device needed: the real matrix representation the dense engine's matrix kernel uses for the
 * geometric product of G(n) with a +-1 metric (bit i of neg_mask set: e_i^2 = -1; csrc/device/dense_matrix.cu).
 * shape[0..3] receive MX, DB, DL, has_lx: 2^DB products of 2^MX x 2^MX by 2^MX x 2^DL matrices per element, i.e.
 * 2^(n + MX) multiplications instead of 4^n.  When a, b, c are non-null, c = a b is computed ON THE HOST through
 * that representation (2^n doubles each, indexed by blade bitmask) -- the mirror of the kernel the tests compare
 * with the reference's term tables.  GAAST_ERR_UNSUPPORTED when the algebra has no representation the kernel
 * can use (n < 7, n > 12, degenerate metric). */
gaast_status gaast_diag_matrix_rep(uint32_t n, uint32_t neg_mask, int32_t* shape, const double* a, const double* b, double* c);

/* Name and launch shape of the kernel the last gaast_eval on this plan used. */
const char* gaast_plan_last_kernel(const gaast_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* GAAST_B200_H */
