// Table engine: the generic, plan-interpreting evaluator (sm_100a).
//
// One thread evaluates one batch element.  The element's buffers -- the
// reference's cache entries (eval.rs:21-33) -- live in a per-block workspace
// [total_cols][threads] in shared memory (column-major over threads, so every
// access is bank-conflict free), or in global memory when the plan is too wide.
// The block walks the plan's micro-ops in reference execution order.  For a
// product (eval.rs:77-83) the term table is streamed chunk by chunk into shared
// memory by the TMA unit (cp.async.bulk + mbarrier, double buffered) while the
// threads consume the previous chunk; terms are pre-sorted by output slot, so
// each run accumulates one output in a register, in the reference's term order.
//
// This engine is the always-available path: any valid plan runs here.  The
// specialised engine (codegen.cpp) is the fast path.
#include <cstdint>

#include "../runtime.hpp"

namespace gaast {

namespace {

constexpr int kStageBytes = int(sizeof(TermChunk));
constexpr int kBarOffset = 2 * kStageBytes;
constexpr int kWsOffset = ((kBarOffset + 16) + 127) / 128 * 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on `bar`.
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "GAAST_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra GAAST_DONE;\n"
        "bra GAAST_WAIT;\n"
        "GAAST_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

template <bool kStrict>
__device__ __forceinline__ double term_acc(double acc, double l, double r, double c) {
    if (kStrict) return __dadd_rn(acc, __dmul_rn(__dmul_rn(l, r), c));  // eval.rs:82, no contraction
    return fma(l * c, r, acc);
}
// the f32 variant: the same operation sequence in binary32 (coefficients rounded to binary32)
template <bool kStrict>
__device__ __forceinline__ float term_acc(float acc, float l, float r, float c) {
    if (kStrict) return __fadd_rn(acc, __fmul_rn(__fmul_rn(l, r), c));
    return fmaf(l * c, r, acc);
}
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double inv_rn(double a) { return __ddiv_rn(1.0, a); }
__device__ __forceinline__ float inv_rn(float a) { return __fdiv_rn(1.0f, a); }
__device__ __forceinline__ double sqrt_rn(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ float sqrt_rn(float a) { return __fsqrt_rn(a); }

// exp / log of a k-vector with a scalar square (GAAST_OP_EXP / GAAST_OP_LOG: this library's definition, the reference
// has todo!() there).  q = <B B>_0.  Near q = 0 both branches share one series: sin x / x = sinh x / x = 1 + q / 6,
// cos x = cosh x = 1 + q / 2, atan(x / a) / x = atanh(x / a) / x = (1 + q / (3 a^2)) / a  (q = -+ x^2).
template <class T>
__device__ __forceinline__ void exp_factors(T q, T* c, T* s) {
    const double qq = double(q);
    if (fabs(qq) < 1e-8) { *c = T(1.0 + 0.5 * qq); *s = T(1.0 + qq / 6.0); return; }
    const double x = sqrt(fabs(qq));
    if (qq < 0) { *c = T(cos(x)); *s = T(sin(x) / x); }
    else { *c = T(cosh(x)); *s = T(sinh(x) / x); }
}
template <class T>
__device__ __forceinline__ T log_factor(T a0, T q) {
    const double a = double(a0), qq = double(q);
    if (fabs(qq) < 1e-8 * a * a && a > 0) return T((1.0 + qq / (3.0 * a * a)) / a);
    const double x = sqrt(fabs(qq));
    return T(qq < 0 ? atan2(x, a) / x : atanh(x / a) / x);
}

// Thread layout: lane = batch element (32 per block and tile), warp = work group.  The
// element's workspace is shared by the block's warps: inside a micro-op they split the rows
// (loads, sign flips, stores) or the output runs of a term chunk (products), so a block
// keeps 8 warps busy on 32 elements' worth of shared memory -- 4-8x the warps a
// thread-per-element layout could hold.  Two runs never write the same output inside a
// chunk, chunks are separated by a barrier, and a run accumulates its terms in table order:
// every component still sums in the reference's order.
// kGlobalWs is a template parameter so that, in the common case, the compiler knows the
// workspace is shared memory and emits LDS/STS instead of generic loads and stores.
constexpr int kLanes = 32;
// T = scalar type of the arithmetic and of the workspace (double, or float for the f32 variant), St = scalar type of the
// batches (float for f32 batches, also when they are evaluated in double: loads widen, stores round once);
// the batch-sum columns are double in every case, add the unrounded T results and follow the T workspace.
template <class T, bool kStrict, bool kSum, bool kGlobalWs, class St = T>
__global__ void __launch_bounds__(256) table_engine_kernel(const __grid_constant__ EvalArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    TermChunk* stage = reinterpret_cast<TermChunk*>(smem_raw);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + kBarOffset);
    const int tid = threadIdx.x, lane = tid & 31, grp = tid >> 5, G = blockDim.x >> 5;
    const int cols = a.total_cols + (kSum ? a.n_sum_cols : 0);  // (the global workspace is sized in doubles)
    T* ws = kGlobalWs ? reinterpret_cast<T*>(a.ws_global + size_t(blockIdx.x) * cols * kLanes)
                      : reinterpret_cast<T*>(smem_raw + kWsOffset);
    T* w = ws + lane;  // column c of this lane's element: w[c * kLanes]
    // sum columns: doubles behind the T columns (8-byte aligned: total_cols * 32 lanes * sizeof(T))
    double* sum_ws = reinterpret_cast<double*>(ws + size_t(a.total_cols) * kLanes);
    double* sw = sum_ws + lane;

    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (kSum)
        for (int c = grp; c < a.n_sum_cols; c += G) sw[size_t(c) * kLanes] = 0.0;
    __syncthreads();

    const long long tile_step = (long long)gridDim.x * kLanes;
    const long long first = (long long)blockIdx.x * kLanes;
    long long n_tiles = first < a.n ? (a.n - first + tile_step - 1) / tile_step : 0;
    const long long total_chunks = n_tiles * a.n_chunks;  // chunk loads this block will consume
    long long q = 0;                                       // running chunk sequence number

    auto issue = [&](long long seq) {  // thread 0 only
        const int s = int(seq & 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&mbar[s], kStageBytes);
        tma_bulk_g2s(&stage[s], a.chunks + (seq % a.n_chunks), kStageBytes, &mbar[s]);
    };
    if (tid == 0 && total_chunks > 0) issue(0);

    for (long long base = first; base < a.n; base += tile_step) {
        const long long e = base + lane;
        const bool active = e < a.n;
        for (int c = grp; c < a.total_cols; c += G) w[size_t(c) * kLanes] = T(0);  // init_null_mv, eval.rs:27-30
        __syncthreads();

        for (int m = 0; m < a.n_micro; ++m) {
            const MicroOp op = a.micro[m];
            switch (op.kind) {
                case MK_LOAD_ADD: {  // eval.rs:45-50
                    const bool bc = (a.bcast[op.a >> 6] >> (op.a & 63)) & 1;
                    const St* src = reinterpret_cast<const St*>(a.sptr[op.a]) + (long long)op.b * a.srow[op.a] + (bc ? 0 : e);
                    const long long rs = a.srow[op.a];
                    for (uint32_t r = grp; r < op.count; r += G) {
                        T* d = &w[size_t(op.dst_col + r) * kLanes];
                        const T v = active ? T(__ldg(src + r * rs)) : T(0);
                        *d = kStrict ? add_rn(*d, v) : (*d + v);
                    }
                    break;
                }
                case MK_CONST_ADD:
                    for (uint32_t r = grp; r < op.count; r += G) {
                        T* d = &w[size_t(op.dst_col + r) * kLanes];
                        *d = *d + T(a.consts[op.a + r]);
                    }
                    break;
                case MK_MUL: {  // eval.rs:61-86
                    const T* wl = w + size_t(op.a) * kLanes;
                    const T* wr = w + size_t(op.b) * kLanes;
                    T* wd = w + size_t(op.dst_col) * kLanes;
                    for (uint32_t ci = 0; ci < op.count; ++ci) {
                        if (tid == 0 && q + 1 < total_chunks) issue(q + 1);
                        mbar_wait(&mbar[q & 1], unsigned(q >> 1) & 1);
                        const TermChunk& ch = stage[q & 1];
                        const uint32_t n_runs = ch.n_runs;
                        for (uint32_t r = grp; r < n_runs; r += G) {  // this warp's output runs
                            uint32_t s = ch.run_start[r];
                            const uint32_t end = ch.run_start[r + 1];
                            T* o = wd + size_t(ch.terms[s].out) * kLanes;
                            T acc = *o;
                            // four terms per trip: their 4 table reads and 8 operand reads are
                            // independent, only the accumulator chains (reference order kept)
                            for (; s + 4 <= end; s += 4) {
                                const gaast_term t0 = ch.terms[s], t1 = ch.terms[s + 1], t2 = ch.terms[s + 2],
                                                 t3 = ch.terms[s + 3];
                                const T l0 = wl[size_t(t0.a) * kLanes], r0 = wr[size_t(t0.b) * kLanes];
                                const T l1 = wl[size_t(t1.a) * kLanes], r1 = wr[size_t(t1.b) * kLanes];
                                const T l2 = wl[size_t(t2.a) * kLanes], r2 = wr[size_t(t2.b) * kLanes];
                                const T l3 = wl[size_t(t3.a) * kLanes], r3 = wr[size_t(t3.b) * kLanes];
                                acc = term_acc<kStrict>(acc, l0, r0, T(t0.coeff));
                                acc = term_acc<kStrict>(acc, l1, r1, T(t1.coeff));
                                acc = term_acc<kStrict>(acc, l2, r2, T(t2.coeff));
                                acc = term_acc<kStrict>(acc, l3, r3, T(t3.coeff));
                            }
                            for (; s < end; ++s) {
                                const gaast_term t = ch.terms[s];
                                acc = term_acc<kStrict>(acc, wl[size_t(t.a) * kLanes], wr[size_t(t.b) * kLanes], T(t.coeff));
                            }
                            *o = acc;
                        }
                        __syncthreads();  // stage q&1 may be refilled; the next chunk may continue an output
                        ++q;
                    }
                    break;
                }
                case MK_NEG:  // graded.rs:61-65
                    for (uint32_t r = grp; r < op.count; r += G) {
                        T* d = &w[size_t(op.dst_col + r) * kLanes];
                        *d = -*d;
                    }
                    break;
                case MK_INV:  // eval.rs:107
                    if (grp == 0) {
                        T* d = &w[size_t(op.dst_col) * kLanes];
                        *d = inv_rn(*d);
                    }
                    break;
                case MK_SQRT:  // eval.rs:108
                    if (grp == 0) {
                        T* d = &w[size_t(op.dst_col) * kLanes];
                        *d = sqrt_rn(*d);
                    }
                    break;
                case MK_EXP:    // dst += exp(B): grade 0 += c(q), grade k += s(q) B
                case MK_LOG:    // dst += log(a0 + B): grade k += t(a0, q) B
                    if (grp == 0) {  // (rare ops on C(n,k) components: one warp, in component order)
                        const T* src = w + size_t(op.a) * kLanes;
                        T q = T(0);
                        for (uint32_t r = 0; r < op.count; ++r) q = term_acc<kStrict>(q, src[size_t(r) * kLanes], src[size_t(r) * kLanes], T(a.consts[op.chunk0 + r]));
                        T f;
                        if (op.kind == MK_EXP) {
                            T c;
                            exp_factors(q, &c, &f);
                            if (op.b != 0xFFFFFFFFu) {
                                T* d0 = &w[size_t(op.b) * kLanes];
                                *d0 = kStrict ? add_rn(*d0, c) : (*d0 + c);
                            }
                        } else {
                            f = log_factor(w[size_t(op.b) * kLanes], q);
                        }
                        for (uint32_t r = 0; r < op.count; ++r) {
                            T* d = &w[size_t(op.dst_col + r) * kLanes];
                            *d = term_acc<kStrict>(*d, f, src[size_t(r) * kLanes], T(1));
                        }
                    }
                    break;
                case MK_STORE: {
                    St* dst = reinterpret_cast<St*>(a.sptr[op.a]) + (long long)op.b * a.srow[op.a] + e;
                    const long long rs = a.srow[op.a];
                    for (uint32_t r = grp; r < op.count; r += G) {
                        const T v = w[size_t(op.dst_col + r) * kLanes];
                        if (active && a.store_out) dst[r * rs] = St(v);  // (double -> float: round to nearest even)
                        if (kSum && active) {
                            double* sc = &sw[size_t(op.pad0 + r) * kLanes];  // (pad0: the run's first batch-sum column)
                            *sc = *sc + double(v);
                        }
                    }
                    break;
                }
            }
            if (op.kind != MK_MUL) __syncthreads();  // the next micro-op may read what other warps wrote
        }
    }

    if (kSum) {
        // Fixed-order block reduction of the per-lane column sums.
        __syncthreads();
        for (int c = tid; c < a.n_sum_cols; c += blockDim.x) {
            const double* col = sum_ws + size_t(c) * kLanes;
            double s = 0.0;
            for (int t = 0; t < kLanes; ++t) s += col[t];
            a.partials[size_t(blockIdx.x) * a.n_sum_cols + c] = s;
        }
    }
}

// out[c] = sum over blocks of partials[b][c], in block order (deterministic).
__global__ void reduce_partials_kernel(const double* __restrict__ partials, int n_blocks, int n_cols,
                                       double* __restrict__ out) {
    // one block per column; thread t adds blocks t, t+256, ... in order, then a fixed tree:
    // the result depends on the launch shape only, never on timing
    __shared__ double tree[256];
    const int c = blockIdx.x;
    double s = 0.0;
    for (int b = threadIdx.x; b < n_blocks; b += 256) s += partials[size_t(b) * n_cols + c];
    tree[threadIdx.x] = s;
    __syncthreads();
    for (int half = 128; half > 0; half >>= 1) {
        if (threadIdx.x < half) tree[threadIdx.x] += tree[threadIdx.x + half];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[c] = tree[0];
}

// First level for many partial rows (the batch-sum kernels run up to 64 blocks per resident slot: ~19 000 rows of
// 66 doubles on a B200): block j owns a contiguous range of rows and streams it as one flat array -- thread t reads
// elements t, t + T, t + 2T, ... with T the largest multiple of n_cols <= 256, so that a thread always meets the SAME
// column and a warp reads 256 contiguous bytes (the one-block-per-column kernel above reads 8 bytes per 528-byte
// stride: 60 us for 19 000 rows, a seventh of the sharded cfg5 step at 8 GPUs).  Row ranges, thread assignment and the
// fixed-order combination of the T / n_cols lanes of a column depend on the launch shape only: deterministic.
__global__ void reduce_partials_stage1(const double* __restrict__ partials, int n_blocks, int n_cols, int rows_per_block,
                                       double* __restrict__ out) {
    __shared__ double lanes[256];
    const int T = (256 / n_cols) * n_cols;
    const int r0 = blockIdx.x * rows_per_block;
    const int r1 = min(n_blocks, r0 + rows_per_block);
    double s = 0.0;
    if (int(threadIdx.x) < T && r0 < r1) {
        const double* base = partials + size_t(r0) * n_cols;
        const size_t count = size_t(r1 - r0) * n_cols;
        for (size_t i = threadIdx.x; i < count; i += T) s += base[i];
    }
    lanes[threadIdx.x] = s;
    __syncthreads();
    if (int(threadIdx.x) < n_cols) {
        double v = 0.0;
        for (int t = threadIdx.x; t < T; t += n_cols) v += lanes[t];
        out[size_t(blockIdx.x) * n_cols + threadIdx.x] = v;
    }
}

// T = Scalars<arithmetic type, batch type> (below)
template <class T, bool kStrict, bool kSum, bool kGlobalWs>
cudaError_t launch_g(const EvalArgs& args, const TableLaunch& shape, cudaStream_t stream) {
    auto k = table_engine_kernel<typename T::compute, kStrict, kSum, kGlobalWs, typename T::storage>;
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(shape.smem));
    if (err != cudaSuccess) return err;
    k<<<shape.grid, shape.threads, shape.smem, stream>>>(args);
    return cudaGetLastError();
}
template <class T, class St>
struct Scalars {
    using compute = T;
    using storage = St;
};
template <class T, class St, bool kStrict, bool kSum>
cudaError_t launch_t(const EvalArgs& args, const TableLaunch& shape, cudaStream_t stream) {
    return shape.global_ws ? launch_g<Scalars<T, St>, kStrict, kSum, true>(args, shape, stream)
                           : launch_g<Scalars<T, St>, kStrict, kSum, false>(args, shape, stream);
}
template <class T, class St>
cudaError_t launch_s(const EvalArgs& args, const TableLaunch& shape, bool strict, bool with_sum, cudaStream_t stream) {
    if (strict) return with_sum ? launch_t<T, St, true, true>(args, shape, stream) : launch_t<T, St, true, false>(args, shape, stream);
    return with_sum ? launch_t<T, St, false, true>(args, shape, stream) : launch_t<T, St, false, false>(args, shape, stream);
}

}  // namespace

TableLaunch table_engine_shape(const gaast_ctx& ctx, const DevicePlanHost& h, long long n, bool with_sum, bool f32, bool wide) {
    TableLaunch s;
    const size_t cols = h.total_cols + (with_sum ? h.stored_cols : 0);
    // one tile = 32 elements; the workspace holds the arithmetic's type, the sum columns are doubles in every variant
    const size_t ws_bytes = (h.total_cols * (f32 && !wide ? sizeof(float) : sizeof(double)) + (with_sum ? h.stored_cols * sizeof(double) : 0)) * kLanes;
    s.threads = 256;                                         // 8 warps share the tile's work
    s.global_ws = kWsOffset + ws_bytes > size_t(ctx.smem_optin);
    s.smem = s.global_ws ? kWsOffset : kWsOffset + ws_bytes;
    s.ws_doubles_per_block = cols * kLanes;
    const long long tiles = (n + kLanes - 1) / kLanes;
    int per_sm = int(size_t(ctx.smem_optin) / (s.smem + 1024));
    per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);  // 2048 threads per SM
    const long long g = (long long)ctx.sm_count * per_sm;
    s.grid = int(tiles < g ? (tiles > 0 ? tiles : 1) : g);
    return s;
}

cudaError_t table_engine_launch(const EvalArgs& args, const TableLaunch& shape, bool strict, bool with_sum, bool f32,
                                bool wide, cudaStream_t stream) {
    if (f32 && wide) return launch_s<double, float>(args, shape, strict, with_sum, stream);
    return f32 ? launch_s<float, float>(args, shape, strict, with_sum, stream)
               : launch_s<double, double>(args, shape, strict, with_sum, stream);
}

cudaError_t reduce_partials_launch(const double* partials, int n_blocks, int n_cols, double* out,
                                   cudaStream_t stream) {
    if (n_cols <= 0) return cudaSuccess;
    if (n_blocks > 2048 && n_cols <= 256) {
        // two levels; the caller's buffer has room for kReduceStage1Rows more rows behind the partials
        const int g1 = kReduceStage1Rows;
        const int rows_per_block = (n_blocks + g1 - 1) / g1;
        double* tmp = const_cast<double*>(partials) + size_t(n_blocks) * n_cols;
        reduce_partials_stage1<<<g1, 256, 0, stream>>>(partials, n_blocks, n_cols, rows_per_block, tmp);
        reduce_partials_kernel<<<n_cols, 256, 0, stream>>>(tmp, g1, n_cols, out);
        return cudaGetLastError();
    }
    reduce_partials_kernel<<<n_cols, 256, 0, stream>>>(partials, n_blocks, n_cols, out);
    return cudaGetLastError();
}

const char* table_engine_arch() { return "sm_100a"; }

}  // namespace gaast
