// Internal structures of the device runtime (ctx / batch / plan handles) and
// the interfaces between its translation units.
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "device_plan.hpp"
#include "eval_args.h"

namespace gaast {

// A kernel specialised for one plan (codegen.cpp), compiled by NVRTC or loaded
// from the in-tree cubin cache (jit.cpp).
struct JitKernel {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t kernel = nullptr;      // per-element kernel
    cudaKernel_t uniform_kernel = nullptr;  // optional: hoisted broadcast-only prologue (1 thread)
    std::string name;
    std::string key;        // cache key (hash of the source + flags)
    std::string origin;     // "cache" | "nvrtc"
    int threads = 0;        // block size
    int elems_per_thread = 1;
    int min_blocks = 1;
    int n_uniform = 0;      // doubles the uniform prologue writes
    size_t smem_bytes = 0;  // dynamic shared memory (batch-sum accumulators, parked rows)
    bool pipelined = false; // persistent grid: blocks stride over the tiles
    bool one_tile_blocks = false;
    int regs = 0;
    size_t local_bytes = 0; // spills
    int blocks_per_sm = 1;
    int fma_per_elem = 0;   // FMAs (or mul + add pairs) one element executes in this kernel
    ~JitKernel();
};

struct CodegenOptions {
    uint64_t broadcast_slots = 0;
    int arith = GAAST_ARITH_FMA;
    bool with_sum = false;
    bool store_out = true;
    int elems_per_thread = 0;  // 0 = choose
    int variant = 0;           // GAAST_CODEGEN_* bit flags (tuning knobs; 0 = defaults)
    bool pipelined = true;     // parked rows arrive by TMA in a persistent, double-buffered block (needs 16-byte aligned rows)
    bool tma_stage = false;    // one-tile blocks: parked rows copied to shared memory by TMA bulk copies (aligned rows)
    int extra_parked = 0;      // more input rows parked in shared memory (raised while ptxas reports spills)
    bool f32 = false;          // binary32 batches and arithmetic (the f32 variant); batch sums stay in double
    bool wide = false;         // with f32: binary64 arithmetic on the binary32 batches (GAAST_ARITH_F64), one rounding per store
    // Sparse per-grade storage of the bound inputs: per stream (device_plan.hpp) a bitmap of the components its grade
    // array stores (empty = dense).  Components that are not stored are zero for every element: their loads become
    // the constant 0 and every term that reads them is dropped (exactly, in strict arithmetic too: x + 0 * y == x
    // for finite y); stored rows are addressed by their rank.
    std::vector<std::vector<uint64_t>> sparse;
    uint64_t sparse_hash = 0;
    // What tells two specialised kernels of one plan apart (the bitmaps by their hash): the plan's map key.
    auto key() const {
        return std::make_tuple(broadcast_slots, arith, with_sum, store_out, elems_per_thread, variant, pipelined, tma_stage,
                               f32, wide, sparse_hash);
    }
};

struct CodegenResult {
    std::string source;
    std::string kernel_name;
    std::string uniform_kernel_name;  // empty when nothing was hoisted
    int threads = 128;
    int elems_per_thread = 1;
    int min_blocks = 1;
    int n_uniform = 0;
    int n_sum_cols = 0;
    size_t smem_bytes = 0;
    bool pipelined = false;
    bool one_tile_blocks = false;  // the kernel handles exactly one tile per block: the grid must cover the batch
    int parked = 0, parkable = 0;  // input rows parked in shared memory / rows that could be
    int fma_per_elem = 0;          // product terms the per-element kernel executes (after lowering / dead-code removal)
    std::string notes;  // human-readable summary of the decisions taken
};

// codegen.cpp: CUDA source of the specialised kernel for a plan.
CodegenResult generate_kernel(const DevicePlanHost& h, const CodegenOptions& opt);

// jit.cpp: source -> cubin (NVRTC, found with dlopen) with an on-disk cache.
bool jit_available(std::string* why);
// Compiles (or finds in the cache) without touching a device.  Returns the cubin.
std::vector<char> jit_cubin(const CodegenResult& cg, std::string* key, std::string* origin, std::string* log);
// Generates and compiles the kernel for `opt`, parking more input rows in shared
// memory while ptxas reports register spills.  `cg` receives the final source.
std::vector<char> build_specialized(const DevicePlanHost& h, CodegenOptions opt, CodegenResult* cg, std::string* key,
                                    std::string* origin);
size_t spill_bytes_from_log(const std::string& ptxas_log, const std::string& kernel);
// Loads a cubin on the current device.
std::shared_ptr<JitKernel> jit_load(const CodegenResult& cg, const std::vector<char>& cubin);
std::string jit_cache_dir();

// table_engine.cu
struct TableLaunch {
    int threads = 0;
    int grid = 0;
    size_t smem = 0;
    bool global_ws = false;
    size_t ws_doubles_per_block = 0;  // global workspace: columns x 32 lanes
};
// f32: binary32 batches; wide: evaluated in binary64 (the workspace is then sized in doubles)
TableLaunch table_engine_shape(const gaast_ctx& ctx, const DevicePlanHost& h, long long n, bool with_sum, bool f32, bool wide);
cudaError_t table_engine_launch(const EvalArgs& args, const TableLaunch& shape, bool strict, bool with_sum, bool f32,
                                bool wide, cudaStream_t stream);
// (the partials buffer must have room for kReduceStage1Rows more rows of n_cols doubles: the two-level reduction's scratch)
constexpr int kReduceStage1Rows = 296;
cudaError_t reduce_partials_launch(const double* partials, int n_blocks, int n_cols, double* out,
                                   cudaStream_t stream);
const char* table_engine_arch();

// dense_warp.cu: chains of dense products of full-grade buffers in G(n), n = 7..10, one warp per multivector
struct DenseWarpProduct {                 // tables of one product op
    std::vector<uint32_t> lambda_words;   // [32]: bit blo of word alo = lambda(alo, blo) is -1
    std::vector<uint32_t> present_words;  // [32]: bit blo of word alo = the product keeps the pair (alo, blo)
    std::vector<uint32_t> toggle;         // [J][J], J = 2^n / 32: sign-bit masks that step sigma(ahi - 1, g) to sigma(ahi, g)
    std::vector<uint8_t> sigma;           // [J][J]: 0 = +1, 1 = -1, 2 = the product drops the pair of high parts
    bool complete = true;                 // every pair kept (geometric product): the generic kernel can run it
};
struct DenseWarpOperand {   // where a full-grade buffer lives when a product reads or writes it
    int slot = -1;          // >= 0: a batch input (read only)
    int scratch = -1;       // >= 0: a scratch buffer of the plan (an earlier product)
    bool root = false;      // the root's grade arrays (written by the last product)
    uint32_t neg_mask = 0;  // grades whose sign flips on the way (Negation / Reverse / GradeInvolution)
    uint32_t grade_mask = 0;  // grades that hold data (operand) / that are stored (result)
};
struct DenseWarpStep {
    DenseWarpProduct prod;
    bool geometric = false;   // keeps every pair its buffers' grades allow, signs of a +-1 metric: the matrix kernel applies
    uint32_t neg_mask = 0;    // that metric (bit i: e_i^2 = -1)
    DenseWarpOperand L, R, O;
    bool accumulate = false;  // O already holds an earlier product of the same sum: add to it
    DenseWarpOperand C;       // optional addend (slot >= 0): a batch input summed into the same buffer
};
// dense_matrix.cu: the real matrix representation of G(p,q) the matrix kernel of the dense engine multiplies in
struct MatrixRep {
    uint32_t n = 0, neg_mask = 0;  // bit i of neg_mask: e_i^2 = -1
    int mx = 0, db = 0, dl = 0;    // 2^db products of 2^mx x 2^mx by 2^mx x 2^dl matrices per element
    std::vector<uint32_t> entry;   // [2^n], index x * 2^(db+dl) + t: blade bitmask | sign << 31
    std::vector<uint8_t> lx;       // [2^mx]: sign mask of the left matrix, M(a)[i][l] *= (-1)^popc(lx[i ^ l] & l)
    bool has_lx = false;
};
struct DenseMatLaunch {
    int T = 0, RC = 1, threads = 0, grid = 0, blocks_per_sm = 1;
    bool pipe = true, csep = true;
    size_t smem = 0;
};
struct DenseWarpHost {
    uint32_t n = 0;
    std::shared_ptr<MatrixRep> mat;       // set when every product is a geometric product under one +-1 metric
    std::vector<uint16_t> blade_of_slot;  // [2^n]
    std::vector<int> gstart;              // first slot of grade k
    std::vector<DenseWarpStep> steps;     // one per product, in the plan's order
    int n_scratch = 0;
    bool complete = true;                 // every product keeps every pair
};
struct DenseWarpBuffers {  // per-grade arrays of one operand / result at launch time
    double* ptr[GAAST_MAX_DIM + 2] = {};
    long long row[GAAST_MAX_DIM + 2] = {};
    bool shared = false;  // a broadcast input: one element for the whole batch
};
struct DenseWarpLaunch {
    int T = 0, LD = 0, threads = 0, grid = 0;
    size_t smem = 0;
};
bool dense_warp_analyse(const DevicePlanHost& h, DenseWarpHost* out);
DenseWarpLaunch dense_warp_shape(const gaast_ctx& ctx, uint32_t n, long long batch);
cudaError_t dense_warp_launch(const DenseWarpHost& prog, const DenseWarpStep& step, const DenseWarpBuffers& L,
                              const DenseWarpBuffers& R, const DenseWarpBuffers& O, const DenseWarpBuffers& C, long long batch,
                              const uint16_t* d_blade_of_slot, const DenseWarpLaunch& shape, cudaKernel_t jit_kernel,
                              cudaStream_t stream);
CodegenResult dense_warp_codegen(uint32_t n, const DenseWarpProduct& prod, const DenseWarpLaunch& shape);
bool matrix_rep_plan(uint32_t n, uint32_t neg_mask, MatrixRep* out);
void matrix_rep_apply(const MatrixRep& rep, const double* a, const double* b, double* c);
std::vector<uint32_t> matrix_rep_device_table(const MatrixRep& rep);
DenseMatLaunch dense_matrix_shape(const gaast_ctx& ctx, const MatrixRep& rep, long long batch);
CodegenResult dense_matrix_codegen(const MatrixRep& rep, const DenseMatLaunch& shape);
cudaError_t dense_matrix_launch(const DenseWarpHost& prog, const DenseWarpStep& step, const DenseWarpBuffers& L,
                                const DenseWarpBuffers& R, const DenseWarpBuffers& O, const DenseWarpBuffers& C, long long batch,
                                const uint32_t* d_src, const uint8_t* d_lx, unsigned long long* d_rows, const DenseMatLaunch& shape,
                                cudaKernel_t kernel, cudaStream_t stream);

// host_pipeline.cu
struct HostPipe;
void host_pipe_destroy(HostPipe* p);

// records.cu: element-major records <-> the batch's rows.  A batch keeps one RecordMap per record mask it has
// been packed from or unpacked to: built on the first call for that mask, so that later calls only launch.
struct RecordRow {
    unsigned long long ptr;  // device address of the stored row (batch column 0)
    uint32_t comp;           // its component in the record
    uint32_t pad;
};
struct RecordMap {
    void* d_table = nullptr;  // RecordRow[n_rows], then uint32_t chunk_row[n_chunks + 1]
    size_t n_rows = 0;
    int K = 0, Kc = 0, E = 0, pitch = 0, n_chunks = 0, max_grid = 1;
    size_t smem = 0;
    int tile_scalars = 0, rows_bytes = 0, unpack_max_grid = 1;  // shared memory: the chunk's rows, then the tile (two: unpack)
    size_t unpack_smem = 0;
};
void records_shape(RecordMap& m, int K, size_t es, int sm_count);
cudaError_t records_launch(const RecordMap& m, bool unpack, size_t es, void* records, long long first, long long count,
                           cudaStream_t stream);

// segments.cu: per-segment sums of a batch's stored rows (gaast_batch_segment_sum).  The scratch -- a flag, the chunks'
// spanning segments and their head / tail partials -- is sized from the batch's length and stored rows and owned by the
// batch; it must start zeroed.  Two kernel launches.
size_t segment_scratch_bytes(long long len, int S);
cudaError_t segment_sum_launch(const RecordRow* rows, int S, size_t es, long long len, const long long* offsets,
                               long long n, double* sums, void* scratch, cudaStream_t stream);
long long segment_chunk();  // columns per chunk: fixes the order of the additions

}  // namespace gaast

struct gaast_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t h2d = nullptr, d2h = nullptr;  // lazily created for gaast_eval_host
    void* staging = nullptr;  // gaast_batch_upload_records / _download_records: one chunk of records
    size_t staging_bytes = 0;
    uint64_t launches = 0;
    int sm_count = 0;
    int smem_optin = 0;
    int cc_major = 0, cc_minor = 0;
};

struct gaast_batch {
    gaast_ctx* ctx = nullptr;
    uint32_t n = 0, mask = 0;
    uint64_t len = 0, stride = 0;
    bool broadcast = false, owned = false;
    int dtype = GAAST_F64;  // the pointers below address f32 arrays when dtype == GAAST_F32
    size_t esize() const { return dtype == GAAST_F32 ? 4 : 8; }
    double* base = nullptr;
    double* grade_ptr[GAAST_MAX_DIM + 1] = {};
    uint32_t rows = 0;  // rows stored, over all grades
    // sparse per-grade storage: present[k] = bitmap of the C(n,k) components grade k stores (empty = all of them);
    // stored rows are compacted in ascending component order
    std::vector<uint64_t> present[GAAST_MAX_DIM + 1];
    uint32_t stored[GAAST_MAX_DIM + 1] = {};  // rows stored per grade
    bool sparse = false;
    mutable std::map<uint32_t, gaast::RecordMap> records;  // by record mask (gaast_batch_pack_records / _unpack_records)
    mutable void* segment_scratch = nullptr;  // gaast_batch_segment_sum: allocated on its first call
};

struct gaast_plan {
    gaast_ctx* ctx = nullptr;  // null: offline plan (source generation / precompilation only)
    gaast::DevicePlanHost h;
    gaast::MicroOp* d_micro = nullptr;
    gaast::TermChunk* d_chunks = nullptr;
    double* d_consts = nullptr;
    double* d_partials = nullptr;
    size_t partials_cap = 0;
    double* d_ws = nullptr;  // table engine: global workspace when shared memory is too small
    size_t ws_cap = 0;
    double* d_uniform = nullptr;
    size_t uniform_cap = 0;
    std::string last_kernel;
    // specialised kernels, keyed by the options they were generated with
    using JitKey = decltype(gaast::CodegenOptions().key());
    std::map<JitKey, std::shared_ptr<gaast::JitKernel>> jit;
    // why a variant could not be built (its entry in `jit` is null): per variant, never sticky for the plan
    std::map<JitKey, std::string> jit_errors;
    int variant = 0;
    int force_ept = 0;
    gaast::HostPipe* pipe = nullptr;  // device buffer sets of gaast_eval_host
    // dense-warp engine: analysed on first use (0 = not yet, 1 = eligible, -1 = not a full product)
    int dense_warp_state = 0;
    gaast::DenseWarpHost dense_warp;
    uint16_t* d_dw_blades = nullptr;
    std::map<std::pair<int, int>, std::shared_ptr<gaast::JitKernel>> dw_jit;  // (step, block size): kernel with sigma folded in
    std::vector<double*> d_dw_scratch;  // intermediate products: [2^n][stride] each
    size_t dw_scratch_stride = 0;
    bool dw_jit_failed = false;  // NVRTC unavailable: keep using the generic kernel
    // ... its matrix-representation kernel (dense_matrix.cu): tables of the algebra, one kernel per tile shape
    uint32_t* d_dm_src = nullptr;
    uint8_t* d_dm_lx = nullptr;
    unsigned long long* d_dm_rows = nullptr;  // per-launch row address tables: 3 x 2^n
    std::map<int, std::shared_ptr<gaast::JitKernel>> dm_jit;  // by elements per tile
    bool dm_jit_failed = false;
};
