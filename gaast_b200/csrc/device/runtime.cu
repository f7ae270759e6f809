// C ABI of the device side (include/gaast_b200.h): ctx, batch, plan, eval.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../runtime.hpp"

using gaast::Error;

namespace {

void cuda_check(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return;
    gaast_status st = GAAST_ERR_CUDA;
    if (e == cudaErrorMemoryAllocation) st = GAAST_ERR_OOM;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) st = GAAST_ERR_NO_DEVICE;
    throw Error(st, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}

template <class F>
gaast_status guard(F&& f) {
    try {
        f();
        return GAAST_OK;
    } catch (const Error& e) {
        gaast::set_last_error(e.what());
        return e.status;
    } catch (const std::bad_alloc&) {
        gaast::set_last_error("out of host memory");
        return GAAST_ERR_OOM;
    } catch (const std::exception& e) {
        gaast::set_last_error(e.what());
        return GAAST_ERR_INVALID;
    }
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cuda_check(cudaSetDevice(dev), "cudaSetDevice");
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

template <class T>
void upload(T*& dst, const std::vector<T>& src, cudaStream_t s) {
    dst = nullptr;
    if (src.empty()) return;
    cuda_check(cudaMalloc(&dst, src.size() * sizeof(T)), "cudaMalloc(plan table)");
    cuda_check(cudaMemcpyAsync(dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, s), "upload plan table");
}

void ensure(double*& p, size_t& cap, size_t want) {
    if (want <= cap) return;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cuda_check(cudaMalloc(&p, want * sizeof(double)), "cudaMalloc(scratch)");
    cap = want;
}

// Fills the stream table of EvalArgs and validates the bound batches.
void bind_streams(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out, bool need_out,
                  gaast::EvalArgs& a, uint64_t* broadcast_slots, long long* n_out, int* dtype_out,
                  std::vector<std::vector<uint64_t>>* sparse_out = nullptr, uint64_t* sparse_hash = nullptr) {
    const gaast::DevicePlanHost& h = plan->h;
    if (n_inputs != h.n_slots) throw Error(GAAST_ERR_SHAPE, "eval: the plan expects " + std::to_string(h.n_slots) + " input batches");
    if (h.n_slots && !inputs) throw Error(GAAST_ERR_INVALID, "eval: null inputs array");
    long long n = -1;
    int dtype = -1;  // one scalar type per call
    auto same_dtype = [&](const gaast_batch* b) {
        if (dtype < 0) dtype = b->dtype;
        if (b->dtype != dtype) throw Error(GAAST_ERR_SHAPE, "eval: f64 and f32 batches cannot be mixed in one call");
    };
    if (out) {
        same_dtype(out);
        if (out->n != h.n) throw Error(GAAST_ERR_SHAPE, "eval: output batch has another dimension");
        if (out->mask != h.buffer_masks[0])
            throw Error(GAAST_ERR_SHAPE, "eval: output batch must carry exactly the root grade set");
        if (out->broadcast) throw Error(GAAST_ERR_SHAPE, "eval: output batch cannot be a broadcast operand");
        if (!h.projected) {
            if (out->sparse)
                throw Error(GAAST_ERR_SHAPE, "eval: the output batch must be dense (sparse storage is for inputs and for "
                                             "the results of projected plans)");
        } else {
            for (uint32_t i = h.n_in_streams; i < h.streams.size(); ++i)
                if (out->present[h.streams[i].grade] != h.root_present[i - h.n_in_streams])
                    throw Error(GAAST_ERR_SHAPE, "eval: the output batch must store exactly the components the projected "
                                                 "plan keeps (grade " + std::to_string(h.streams[i].grade) + " differs)");
        }
        n = (long long)out->len;
    } else if (need_out) {
        throw Error(GAAST_ERR_INVALID, "eval: null output batch");
    }
    *broadcast_slots = 0;
    for (uint32_t s = 0; s < h.n_slots; ++s) {
        const gaast_batch* b = inputs[s];
        if (!b) throw Error(GAAST_ERR_INVALID, "eval: null input batch");
        same_dtype(b);
        if (b->n != h.n) throw Error(GAAST_ERR_SHAPE, "eval: input batch has another dimension");
        if (h.slot_masks[s] & ~b->mask)
            throw Error(GAAST_ERR_SHAPE, "eval: input batch " + std::to_string(s) + " lacks a grade the plan reads");
        if (b->broadcast) {
            *broadcast_slots |= uint64_t(1) << s;
        } else {
            if (n < 0) n = (long long)b->len;
            if ((long long)b->len != n) throw Error(GAAST_ERR_SHAPE, "eval: batch lengths differ");
        }
    }
    if (n < 0) n = 1;  // everything is broadcast: one element
    *n_out = n;
    *dtype_out = dtype < 0 ? GAAST_F64 : dtype;
    const size_t esize = dtype == GAAST_F32 ? 4 : 8;
    std::memset(&a, 0, sizeof a);
    for (size_t i = 0; i < h.streams.size(); ++i) {
        const gaast::Stream& st = h.streams[i];
        if (st.slot == 0xFFFFFFFFu) {
            a.sptr[i] = out ? out->grade_ptr[st.grade] : nullptr;
            a.srow[i] = out ? (long long)out->stride : 0;
        } else {
            const gaast_batch* b = inputs[st.slot];
            a.sptr[i] = b->grade_ptr[st.grade];
            a.srow[i] = (long long)b->stride;
            if (b->broadcast) a.bcast[i >> 6] |= 1ull << (i & 63);
            if (sparse_out && !b->present[st.grade].empty()) {
                if (sparse_out->empty()) sparse_out->resize(h.streams.size());
                (*sparse_out)[i] = b->present[st.grade];
                uint64_t hsh = 0x9E3779B97F4A7C15ull * (i + 1);
                for (uint64_t w : b->present[st.grade]) hsh = (hsh ^ w) * 0xD6E8FEB86659FD93ull + 0x632BE59BD9B4E019ull;
                *sparse_hash ^= hsh;
            }
        }
    }
    // results are stored component by component while later components still read the inputs:
    // an output array overlapping an input array would be read after it was overwritten
    for (size_t o = h.n_in_streams; o < h.streams.size() && out; ++o) {
        const char* ob = reinterpret_cast<const char*>(a.sptr[o]);
        const char* oe = ob + size_t(h.stored_rows(o)) * size_t(a.srow[o]) * esize;
        for (size_t i = 0; i < h.n_in_streams; ++i) {
            const char* ib = reinterpret_cast<const char*>(a.sptr[i]);
            const gaast_batch* ibatch = inputs[h.streams[i].slot];
            const char* ie = ib + size_t(ibatch->stored[h.streams[i].grade]) * size_t(a.srow[i]) * esize;
            if (ob < ie && ib < oe) throw Error(GAAST_ERR_INVALID, "eval: the output batch overlaps an input batch");
        }
    }
    a.n = n;
    a.consts = plan->d_consts;
    a.total_cols = int(h.total_cols);
    a.root_col = int(h.buf_col[0]);
    a.store_out = out ? 1 : 0;
}

// The specialised kernel gaast_eval launches for a call; kernel_source and precompile name it through this function too.
// A batch it cannot address with 128-bit accesses gets one element per thread and no TMA (bulk copies need 16-byte
// aligned row segments).
gaast::CodegenOptions specialized_options(const gaast_plan* plan, uint64_t broadcast_slots, int arith, bool with_sum,
                                          bool store_out, bool f32, const std::vector<std::vector<uint64_t>>& sparse,
                                          uint64_t sparse_hash, bool aligned) {
    gaast::CodegenOptions opt;
    opt.broadcast_slots = broadcast_slots;
    opt.arith = arith;
    opt.with_sum = with_sum;
    opt.store_out = store_out;
    opt.f32 = f32;
    opt.sparse = sparse;
    opt.sparse_hash = sparse_hash;
    opt.variant = plan->variant;
    opt.elems_per_thread = aligned ? plan->force_ept : 1;
    // TMA-pipelined staging is opt-in (variant bit 3): measured slower than plain blocks on cfg3 / cfg5
    opt.pipelined = aligned && (plan->variant & 8);
    opt.tma_stage = aligned && !opt.pipelined && !with_sum && !(plan->variant & 1024);
    return opt;
}

// A chain of geometric products runs on the dense engine's matrix-representation kernel unless variant bit 20 asks
// for the term-by-term kernels.
bool wants_matrix_kernel(const gaast_plan* plan, const gaast::DenseWarpHost& prog) { return prog.mat && !(plan->variant & 1048576); }

// Generates and compiles (or finds in the cache) one kernel of the dense engine for a device of `dev`'s shape and a
// batch of `batch` elements: the term-by-term kernel of product `step` with its signs folded at compile time, or for
// step < 0 the matrix-representation kernel of the chain (dense_matrix.cu).  `*cg` receives its source.
std::vector<char> build_dense(const gaast::DenseWarpHost& prog, const gaast_ctx& dev, long long batch, int step,
                              gaast::CodegenResult* cg, std::string* key, std::string* origin, std::string* log) {
    *cg = step >= 0 ? gaast::dense_warp_codegen(prog.n, prog.steps[size_t(step)].prod, gaast::dense_warp_shape(dev, prog.n, batch))
                    : gaast::dense_matrix_codegen(*prog.mat, gaast::dense_matrix_shape(dev, *prog.mat, batch));
    return gaast::jit_cubin(*cg, key, origin, log);
}

}  // namespace

gaast::JitKernel::~JitKernel() {
    if (lib) cudaLibraryUnload(lib);
}

extern "C" {

const char* gaast_version(void) { return "gaast_b200 0.1 (sm_100a)"; }

gaast_status gaast_ctx_create(int device, void* stream, gaast_ctx** out) {
    return guard([&] {
        if (!out) throw Error(GAAST_ERR_INVALID, "null output pointer");
        *out = nullptr;
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            throw Error(GAAST_ERR_NO_DEVICE, std::string("no CUDA device: gaast_b200 has no CPU path (") +
                                                 (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") + ")");
        if (device < 0 || device >= count) throw Error(GAAST_ERR_NO_DEVICE, "device ordinal out of range");
        (void)gaast::tuning();  // the environment is read here, once, never on the evaluation path
        DeviceGuard dg(device);  // the caller's current device is restored on return
        auto ctx = std::make_unique<gaast_ctx>();
        ctx->device = device;
        cudaDeviceProp prop;
        cuda_check(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
        ctx->sm_count = prop.multiProcessorCount;
        ctx->smem_optin = int(prop.sharedMemPerBlockOptin);
        ctx->cc_major = prop.major;
        ctx->cc_minor = prop.minor;
        if (prop.major != 10)
            throw Error(GAAST_ERR_NO_DEVICE, "device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                                                 ": this library carries sm_100a code only");
        if (stream) {
            ctx->stream = static_cast<cudaStream_t>(stream);
        } else {
            cuda_check(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking), "cudaStreamCreate");
            ctx->own_stream = true;
        }
        *out = ctx.release();
    });
}

gaast_status gaast_ctx_destroy(gaast_ctx* ctx) {
    return guard([&] {
        if (!ctx) return;
        if (ctx->staging) {
            DeviceGuard dg(ctx->device);
            cudaStreamSynchronize(ctx->stream);
            cudaFree(ctx->staging);
        }
        if (ctx->h2d) cudaStreamDestroy(ctx->h2d);
        if (ctx->d2h) cudaStreamDestroy(ctx->d2h);
        if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
    });
}

// Page-locked host memory for the host-array entry points (portable: pinned for every device of the process)
gaast_status gaast_host_alloc(size_t bytes, int flags, void** out) {
    return guard([&] {
        if (!out) throw Error(GAAST_ERR_INVALID, "host_alloc: null out");
        *out = nullptr;
        if (flags != GAAST_HOST_DEFAULT && flags != GAAST_HOST_WRITE_COMBINED) throw Error(GAAST_ERR_INVALID, "host_alloc: unknown flags");
        if (!bytes) throw Error(GAAST_ERR_INVALID, "host_alloc: zero bytes");
        const unsigned f = cudaHostAllocPortable | (flags == GAAST_HOST_WRITE_COMBINED ? cudaHostAllocWriteCombined : 0u);
        cuda_check(cudaHostAlloc(out, bytes, f), "cudaHostAlloc");
    });
}

gaast_status gaast_host_free(void* p) {
    return guard([&] {
        if (p) cuda_check(cudaFreeHost(p), "cudaFreeHost");
    });
}

gaast_status gaast_host_register(void* p, size_t bytes) {
    return guard([&] {
        if (!p || !bytes) throw Error(GAAST_ERR_INVALID, "host_register: null or empty range");
        cuda_check(cudaHostRegister(p, bytes, cudaHostRegisterPortable), "cudaHostRegister");
    });
}

gaast_status gaast_host_unregister(void* p) {
    return guard([&] {
        if (!p) throw Error(GAAST_ERR_INVALID, "host_unregister: null pointer");
        cuda_check(cudaHostUnregister(p), "cudaHostUnregister");
    });
}

gaast_status gaast_ctx_sync(gaast_ctx* ctx) {
    return guard([&] {
        if (!ctx) throw Error(GAAST_ERR_INVALID, "null ctx");
        cuda_check(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
    });
}

void* gaast_ctx_stream(gaast_ctx* ctx) { return ctx ? ctx->stream : nullptr; }
uint64_t gaast_ctx_launch_count(gaast_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------- plan ----
static gaast_status plan_create(gaast_ctx* ctx, const gaast_plan_desc* desc, const uint64_t* const* root_present,
                                gaast_plan** out) {
    return guard([&] {
        if (!out) throw Error(GAAST_ERR_INVALID, "null output pointer");
        *out = nullptr;
        if (!desc) throw Error(GAAST_ERR_INVALID, "null plan description");
        auto plan = std::make_unique<gaast_plan>();
        plan->ctx = ctx;
        plan->h.build(*desc, root_present);
        if (ctx) {
            DeviceGuard dg(ctx->device);
            upload(plan->d_micro, plan->h.micro, ctx->stream);
            upload(plan->d_chunks, plan->h.chunks, ctx->stream);
            upload(plan->d_consts, plan->h.const_values, ctx->stream);
            cuda_check(cudaStreamSynchronize(ctx->stream), "plan upload");
        }
        *out = plan.release();
    });
}

gaast_status gaast_plan_create(gaast_ctx* ctx, const gaast_plan_desc* desc, gaast_plan** out) {
    return plan_create(ctx, desc, nullptr, out);
}

gaast_status gaast_plan_create_projected(gaast_ctx* ctx, const gaast_plan_desc* desc, const uint64_t* const* root_present,
                                         gaast_plan** out) {
    if (out) *out = nullptr;
    if (!root_present) {
        gaast::set_last_error("plan_create_projected: null root bitmap array");
        return GAAST_ERR_INVALID;
    }
    return plan_create(ctx, desc, root_present, out);
}

gaast_status gaast_plan_destroy(gaast_plan* plan) {
    return guard([&] {
        if (!plan) return;
        if (plan->ctx) {
            DeviceGuard dg(plan->ctx->device);
            // kernels of this plan may still be in flight (an asynchronous eval on a temporary plan): nothing is
            // unloaded or freed before the stream has drained
            cudaStreamSynchronize(plan->ctx->stream);
            if (plan->ctx->h2d) cudaStreamSynchronize(plan->ctx->h2d);
            if (plan->ctx->d2h) cudaStreamSynchronize(plan->ctx->d2h);
            plan->jit.clear();
            if (plan->pipe) gaast::host_pipe_destroy(plan->pipe);
            cudaFree(plan->d_micro);
            cudaFree(plan->d_chunks);
            cudaFree(plan->d_consts);
            cudaFree(plan->d_partials);
            cudaFree(plan->d_ws);
            cudaFree(plan->d_uniform);
            cudaFree(plan->d_dw_blades);
            cudaFree(plan->d_dm_src);
            cudaFree(plan->d_dm_lx);
            cudaFree(plan->d_dm_rows);
            plan->dm_jit.clear();
            plan->dw_jit.clear();
            for (double* p : plan->d_dw_scratch) cudaFree(p);
        }
        delete plan;
    });
}

gaast_status gaast_plan_cost(const gaast_plan* plan, uint64_t broadcast_slots, uint64_t* bytes_per_elem,
                             uint64_t* flops_per_elem) {
    return guard([&] {
        if (!plan) throw Error(GAAST_ERR_INVALID, "null plan");
        const auto& h = plan->h;
        uint64_t doubles = 0;
        for (size_t i = 0; i < h.streams.size(); ++i) {
            const auto& st = h.streams[i];
            if (st.slot != 0xFFFFFFFFu && (broadcast_slots >> st.slot & 1)) continue;
            doubles += h.stored_rows(i);  // (a projected root: its stored components only)
        }
        if (bytes_per_elem) *bytes_per_elem = 8 * doubles;
        if (flops_per_elem) *flops_per_elem = 2 * h.total_terms;
    });
}

uint32_t gaast_plan_root_mask(const gaast_plan* plan) { return plan ? plan->h.buffer_masks[0] : 0; }
uint32_t gaast_plan_dim(const gaast_plan* plan) { return plan ? plan->h.n : 0; }
uint32_t gaast_plan_slot_mask(const gaast_plan* plan, uint32_t slot) {
    return (plan && slot < plan->h.n_slots) ? plan->h.slot_masks[slot] : 0;
}
uint32_t gaast_plan_num_slots(const gaast_plan* plan) { return plan ? plan->h.n_slots : 0; }
const char* gaast_plan_last_kernel(const gaast_plan* plan) { return plan ? plan->last_kernel.c_str() : ""; }

gaast_status gaast_plan_set_tuning(gaast_plan* plan, int elems_per_thread, int variant) {
    return guard([&] {
        if (!plan) throw Error(GAAST_ERR_INVALID, "null plan");
        plan->force_ept = elems_per_thread;
        plan->variant = variant;
    });
}

static size_t kernel_source_impl(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum,
                                 const uint64_t* const* present, uint32_t n_present, char* buf, size_t cap) {
    size_t len = 0;
    gaast_status st = guard([&] {
        if (!plan) throw Error(GAAST_ERR_INVALID, "null plan");
        const bool sum = (with_sum & GAAST_SRC_WITH_SUM) != 0, store = !(with_sum & GAAST_SRC_NO_STORE);
        if (!store && !sum) throw Error(GAAST_ERR_INVALID, "kernel_source: a kernel that neither stores nor sums");
        std::vector<std::vector<uint64_t>> sparse;
        if (present) {
            const gaast::DevicePlanHost& h = plan->h;
            if (n_present != h.n_in_streams) throw Error(GAAST_ERR_SHAPE, "kernel_source_sparse: one bitmap pointer per (slot, grade) the plan reads");
            sparse.resize(h.streams.size());
            for (uint32_t i = 0; i < n_present; ++i) {
                if (!present[i]) continue;
                const size_t words = (size_t(h.streams[i].rows) + 63) / 64;
                sparse[i].assign(present[i], present[i] + words);
            }
        }
        // the kernel gaast_eval launches for an aligned batch
        gaast::CodegenResult cg = gaast::generate_kernel(
            plan->h, specialized_options(plan, broadcast_slots, arith, sum, store, (with_sum & GAAST_SRC_F32) != 0, sparse, 0, true));
        len = cg.source.size();
        if (buf && cap) {
            const size_t ncopy = std::min(cap - 1, len);
            std::memcpy(buf, cg.source.data(), ncopy);
            buf[ncopy] = 0;
        }
    });
    return st == GAAST_OK ? len : 0;
}

size_t gaast_plan_kernel_source(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, char* buf,
                                size_t cap) {
    return kernel_source_impl(plan, broadcast_slots, arith, with_sum, nullptr, 0, buf, cap);
}

size_t gaast_plan_kernel_source_sparse(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum,
                                       const uint64_t* const* present, uint32_t n_present, char* buf, size_t cap) {
    return kernel_source_impl(plan, broadcast_slots, arith, with_sum, present, n_present, buf, cap);
}

gaast_status gaast_plan_precompile(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, int store_out) {
    return gaast_plan_precompile_typed(plan, broadcast_slots, arith, with_sum, store_out, GAAST_F64);
}

gaast_status gaast_plan_precompile_typed(gaast_plan* plan, uint64_t broadcast_slots, int arith, int with_sum, int store_out,
                                         int dtype) {
    return guard([&] {
        if (!plan) throw Error(GAAST_ERR_INVALID, "null plan");
        const bool f32 = dtype == GAAST_F32;
        auto options = [&](bool aligned) {
            return specialized_options(plan, broadcast_slots, arith, with_sum != 0, store_out != 0, f32, {}, 0, aligned);
        };
        gaast::CodegenResult cg;
        std::string key, origin;
        try {
            gaast::build_specialized(plan->h, options(true), &cg, &key, &origin);
            // ... and the variant gaast_eval takes for a batch it cannot address with 128-bit accesses / TMA row copies (an
            // odd length or a misaligned pointer in caller-owned memory).  With both in the cache no shape of a shipped
            // workload compiles at run time.
            try {
                gaast::CodegenResult unaligned;
                gaast::build_specialized(plan->h, options(false), &unaligned, nullptr, nullptr);
            } catch (const Error&) {
                // (a plan whose unaligned form does not fit is evaluated by the table engine for such batches)
            }
        } catch (const Error&) {
            // too large / too wide to specialise: a full high-dimensional product gets its dense-warp kernel instead
            gaast::DenseWarpHost dw;
            if (f32 || with_sum || arith != GAAST_ARITH_FMA || plan->h.projected || !gaast::dense_warp_analyse(plan->h, &dw)) throw;
            gaast_ctx b200;  // offline: the launch shape of a B200 (227 KB of shared memory per block, 148 SMs)
            b200.sm_count = 148;
            b200.smem_optin = 232448;
            for (size_t i = 0; i < dw.steps.size(); ++i)  // one kernel per product (equal tables share a cubin)
                build_dense(dw, b200, 1 << 20, int(i), &cg, &key, &origin, nullptr);
            cg.notes += " x" + std::to_string(dw.steps.size()) + " product(s)";
            if (wants_matrix_kernel(plan, dw)) {
                const std::string dw_notes = cg.notes;
                std::string log;
                build_dense(dw, b200, 1 << 20, -1, &cg, &key, &origin, &log);
                cg.notes = dw_notes + " " + cg.notes;
                const size_t used = log.find("Used ", log.find("Function properties for " + cg.kernel_name));
                if (used != std::string::npos)
                    cg.notes += " regs=" + std::to_string(std::atoi(log.c_str() + used + 5)) +
                                " spill=" + std::to_string(gaast::spill_bytes_from_log(log, cg.kernel_name)) + "B";
            }
        }
        plan->last_kernel = cg.kernel_name + " key=" + key + " origin=" + origin + " fma/elem=" + std::to_string(cg.fma_per_elem) +
                            " " + cg.notes;
    });
}

// --------------------------------------------------------------- batch ----
static gaast_status batch_make(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                               int broadcast, int dtype, void* const* grade_ptrs, gaast_batch** out,
                               const uint64_t* const* present = nullptr) {
    return guard([&] {
        if (!out) throw Error(GAAST_ERR_INVALID, "null output pointer");
        *out = nullptr;
        if (!ctx) throw Error(GAAST_ERR_INVALID, "null ctx");
        if (n > GAAST_MAX_DIM) throw Error(GAAST_ERR_INVALID, "dimension above GAAST_MAX_DIM");
        if (grade_mask & ~((2u << n) - 1)) throw Error(GAAST_ERR_INVALID, "grade mask has grades above n");
        if (broadcast && len != 1) throw Error(GAAST_ERR_INVALID, "a broadcast batch holds exactly one element");
        if (dtype != GAAST_F64 && dtype != GAAST_F32) throw Error(GAAST_ERR_INVALID, "unknown dtype");
        auto b = std::make_unique<gaast_batch>();
        b->dtype = dtype;
        const size_t es = b->esize();
        const uint64_t row_quantum = 128 / es;  // rows start on 128-byte boundaries
        b->ctx = ctx;
        b->n = n;
        b->mask = grade_mask;
        b->len = len;
        b->broadcast = broadcast != 0;
        b->rows = 0;
        {
            uint32_t gi = 0;
            for (uint32_t k = 0; k <= n; ++k) {
                if (!(grade_mask >> k & 1)) continue;
                const uint32_t full = uint32_t(gaast::binomial(n, k));
                b->stored[k] = full;
                if (present && present[gi]) {
                    const size_t words = (full + 63) / 64;
                    b->present[k].assign(present[gi], present[gi] + words);
                    if (full % 64) b->present[k].back() &= (~0ull) >> (64 - full % 64);
                    uint32_t cnt = 0;
                    for (uint64_t w : b->present[k]) cnt += uint32_t(__builtin_popcountll(w));
                    if (cnt == full) b->present[k].clear();  // every component stored: a dense grade
                    else { b->stored[k] = cnt; b->sparse = true; }
                }
                b->rows += b->stored[k];
                ++gi;
            }
        }
        DeviceGuard dg(ctx->device);
        if (grade_ptrs) {
            if (stride < len) throw Error(GAAST_ERR_INVALID, "stride smaller than the batch length");
            b->stride = stride;
            uint32_t i = 0;
            for (uint32_t k = 0; k <= n; ++k)
                if (grade_mask >> k & 1) {
                    if (!grade_ptrs[i] && len && b->stored[k]) throw Error(GAAST_ERR_INVALID, "null grade pointer");
                    b->grade_ptr[k] = static_cast<double*>(grade_ptrs[i++]);
                }
        } else {
            b->stride = (len + row_quantum - 1) / row_quantum * row_quantum;
            if (b->stride == 0) b->stride = row_quantum;
            const size_t total = size_t(b->rows) * b->stride;
            if (total) {
                cuda_check(cudaMalloc(&b->base, total * es), "cudaMalloc(batch)");
                b->owned = true;
            }
            size_t row = 0;
            for (uint32_t k = 0; k <= n; ++k)
                if (grade_mask >> k & 1) {
                    b->grade_ptr[k] = reinterpret_cast<double*>(reinterpret_cast<char*>(b->base) + row * b->stride * es);
                    row += b->stored[k];
                }
        }
        *out = b.release();
    });
}

gaast_status gaast_batch_alloc(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                               gaast_batch** out) {
    return batch_make(ctx, n, grade_mask, len, 0, broadcast, GAAST_F64, nullptr, out);
}

gaast_status gaast_batch_alloc_typed(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                                     int dtype, gaast_batch** out) {
    return batch_make(ctx, n, grade_mask, len, 0, broadcast, dtype, nullptr, out);
}

gaast_status gaast_batch_wrap(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                              int broadcast, void* const* grade_ptrs, gaast_batch** out) {
    if (!grade_ptrs) {
        gaast::set_last_error("null grade pointer array");
        return GAAST_ERR_INVALID;
    }
    return batch_make(ctx, n, grade_mask, len, stride, broadcast, GAAST_F64, grade_ptrs, out);
}

gaast_status gaast_batch_wrap_typed(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                                    int broadcast, int dtype, void* const* grade_ptrs, gaast_batch** out) {
    if (!grade_ptrs) {
        gaast::set_last_error("null grade pointer array");
        return GAAST_ERR_INVALID;
    }
    return batch_make(ctx, n, grade_mask, len, stride, broadcast, dtype, grade_ptrs, out);
}

gaast_status gaast_batch_alloc_sparse(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, int broadcast,
                                      int dtype, const uint64_t* const* present, gaast_batch** out) {
    if (!present) {
        gaast::set_last_error("null presence-bitmap array");
        return GAAST_ERR_INVALID;
    }
    return batch_make(ctx, n, grade_mask, len, 0, broadcast, dtype, nullptr, out, present);
}

gaast_status gaast_batch_wrap_sparse(gaast_ctx* ctx, uint32_t n, uint32_t grade_mask, uint64_t len, uint64_t stride,
                                     int broadcast, int dtype, const uint64_t* const* present, void* const* grade_ptrs,
                                     gaast_batch** out) {
    if (!present || !grade_ptrs) {
        gaast::set_last_error("null presence-bitmap or grade pointer array");
        return GAAST_ERR_INVALID;
    }
    return batch_make(ctx, n, grade_mask, len, stride, broadcast, dtype, grade_ptrs, out, present);
}

uint32_t gaast_batch_stored_rows(const gaast_batch* b, uint32_t grade) {
    if (!b || grade > b->n || !(b->mask >> grade & 1)) return 0;
    return b->stored[grade];
}

int gaast_batch_dtype(const gaast_batch* b) { return b ? b->dtype : GAAST_F64; }

gaast_status gaast_batch_free(gaast_batch* b) {
    return guard([&] {
        if (!b) return;
        if ((b->owned && b->base) || !b->records.empty()) {
            DeviceGuard dg(b->ctx->device);
            if (b->owned && b->base) cudaFree(b->base);
            for (auto& kv : b->records) cudaFree(kv.second.d_table);
        }
        delete b;
    });
}

uint64_t gaast_batch_len(const gaast_batch* b) { return b ? b->len : 0; }
uint64_t gaast_batch_stride(const gaast_batch* b) { return b ? b->stride : 0; }
uint32_t gaast_batch_grade_mask(const gaast_batch* b) { return b ? b->mask : 0; }
void* gaast_batch_grade_ptr(const gaast_batch* b, uint32_t grade) {
    if (!b || grade > b->n || !(b->mask >> grade & 1)) return nullptr;
    return b->grade_ptr[grade];
}

static void batch_copy(const gaast_batch* b, uint32_t grade, void* host, uint64_t host_stride, bool to_device, int dtype) {
    if (!b) throw Error(GAAST_ERR_INVALID, "null batch");
    if (b->dtype != dtype) throw Error(GAAST_ERR_SHAPE, "the batch holds another scalar type than the host array");
    const size_t es = b->esize();
    if (grade > b->n || !(b->mask >> grade & 1)) throw Error(GAAST_ERR_SHAPE, "the batch does not hold this grade");
    if (!host) throw Error(GAAST_ERR_INVALID, "null host pointer");
    if (host_stride < b->len) throw Error(GAAST_ERR_INVALID, "host stride smaller than the batch length");
    const size_t rows = b->stored[grade];  // (a sparse grade: the stored rows, compact)
    if (!rows || !b->len) return;
    DeviceGuard dg(b->ctx->device);
    double* dev = b->grade_ptr[grade];
    if (to_device)
        cuda_check(cudaMemcpy2DAsync(dev, b->stride * es, host, host_stride * es, b->len * es, rows, cudaMemcpyHostToDevice,
                                     b->ctx->stream),
                   "batch upload");
    else
        cuda_check(cudaMemcpy2DAsync(host, host_stride * es, dev, b->stride * es, b->len * es, rows, cudaMemcpyDeviceToHost,
                                     b->ctx->stream),
                   "batch download");
}

gaast_status gaast_batch_upload(gaast_batch* b, uint32_t grade, const double* host, uint64_t host_stride) {
    return guard([&] { batch_copy(b, grade, const_cast<double*>(host), host_stride, true, GAAST_F64); });
}
gaast_status gaast_batch_upload_f32(gaast_batch* b, uint32_t grade, const float* host, uint64_t host_stride) {
    return guard([&] { batch_copy(b, grade, const_cast<float*>(host), host_stride, true, GAAST_F32); });
}
gaast_status gaast_batch_download_f32(const gaast_batch* b, uint32_t grade, float* host, uint64_t host_stride) {
    return guard([&] { batch_copy(b, grade, host, host_stride, false, GAAST_F32); });
}
gaast_status gaast_batch_download(const gaast_batch* b, uint32_t grade, double* host, uint64_t host_stride) {
    return guard([&] { batch_copy(b, grade, host, host_stride, false, GAAST_F64); });
}
gaast_status gaast_batch_zero(gaast_batch* b) {
    return guard([&] {
        if (!b) throw Error(GAAST_ERR_INVALID, "null batch");
        DeviceGuard dg(b->ctx->device);
        for (uint32_t k = 0; k <= b->n; ++k)
            if (b->mask >> k & 1)
                cuda_check(cudaMemsetAsync(b->grade_ptr[k], 0, size_t(b->stored[k]) * b->stride * b->esize(), b->ctx->stream),
                           "batch zero");
    });
}

// ------------------------------------------------------------- records ----
// Checks a records call and returns the batch's row map for `record_mask`, building it on the first call (null when
// count == 0: nothing to do).
static const gaast::RecordMap* records_prepare(const gaast_batch* b, uint64_t first, uint64_t count, uint32_t record_mask,
                                               const char* what) {
    if (!b) throw Error(GAAST_ERR_INVALID, std::string(what) + ": null batch");
    if (!record_mask) throw Error(GAAST_ERR_SHAPE, std::string(what) + ": empty record mask (records of no component)");
    if (record_mask & ~((2u << b->n) - 1)) throw Error(GAAST_ERR_SHAPE, std::string(what) + ": record mask has grades above n");
    if (b->mask & ~record_mask) throw Error(GAAST_ERR_SHAPE, std::string(what) + ": the record mask lacks a grade of the batch");
    if (b->broadcast && (first != 0 || count != 1))
        throw Error(GAAST_ERR_SHAPE, std::string(what) + ": a broadcast batch holds one element: first = 0, count = 1");
    if (first > b->len || count > b->len - first)
        throw Error(GAAST_ERR_SHAPE, std::string(what) + ": first + count exceeds the batch length");
    if (!count) return nullptr;
    auto it = b->records.find(record_mask);
    if (it != b->records.end()) return &it->second;
    // stored rows in record-component order: grades ascending, within a grade the stored components ascending
    std::vector<gaast::RecordRow> rows;
    const size_t es = b->esize();
    uint32_t off = 0;
    for (uint32_t k = 0; k <= b->n; ++k) {
        if (!(record_mask >> k & 1)) continue;
        const uint32_t full = uint32_t(gaast::binomial(b->n, k));
        if (b->mask >> k & 1) {
            const std::vector<uint64_t>& present = b->present[k];
            uint32_t rank = 0;
            for (uint32_t c = 0; c < full; ++c) {
                if (!present.empty() && !(present[c / 64] >> (c % 64) & 1)) continue;
                const char* row = reinterpret_cast<const char*>(b->grade_ptr[k]) + size_t(rank++) * b->stride * es;
                rows.push_back({reinterpret_cast<unsigned long long>(row), off + c, 0});
            }
        }
        off += full;
    }
    gaast::RecordMap m;
    gaast::records_shape(m, int(off), es, b->ctx->sm_count);
    m.n_rows = rows.size();
    std::vector<uint32_t> chunk_row(size_t(m.n_chunks) + 1);
    for (int q = 0; q <= m.n_chunks; ++q)
        chunk_row[size_t(q)] = uint32_t(std::lower_bound(rows.begin(), rows.end(), uint32_t(q) * uint32_t(m.Kc),
                                                         [](const gaast::RecordRow& r, uint32_t c) { return r.comp < c; }) -
                                        rows.begin());
    const size_t row_bytes = rows.size() * sizeof(gaast::RecordRow), bytes = row_bytes + chunk_row.size() * sizeof(uint32_t);
    cuda_check(cudaMalloc(&m.d_table, bytes), "cudaMalloc(record row map)");
    cudaError_t e = cudaMemcpyAsync(m.d_table, rows.data(), row_bytes, cudaMemcpyHostToDevice, b->ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(static_cast<char*>(m.d_table) + row_bytes, chunk_row.data(), chunk_row.size() * sizeof(uint32_t),
                            cudaMemcpyHostToDevice, b->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->ctx->stream);  // (the host vectors go out of scope)
    if (e != cudaSuccess) {
        cudaFree(m.d_table);
        cuda_check(e, "upload record row map");
    }
    return &b->records.emplace(record_mask, m).first->second;
}

// Device entry points: `records` must be device memory the kernel can address, aligned to the scalar type.
static void records_device(const gaast_batch* b, uint64_t first, uint64_t count, void* records, uint32_t record_mask,
                           bool unpack) {
    const char* what = unpack ? "unpack_records" : "pack_records";
    if (!b) throw Error(GAAST_ERR_INVALID, std::string(what) + ": null batch");
    DeviceGuard dg(b->ctx->device);
    const gaast::RecordMap* m = records_prepare(b, first, count, record_mask, what);
    if (!m) return;
    if (!records) throw Error(GAAST_ERR_INVALID, std::string(what) + ": null records pointer");
    if (reinterpret_cast<uintptr_t>(records) % b->esize())
        throw Error(GAAST_ERR_INVALID, std::string(what) + ": records pointer not aligned to the scalar type");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, records) != cudaSuccess) {
        cudaGetLastError();
        throw Error(GAAST_ERR_INVALID, std::string(what) + ": records pointer is not known to CUDA");
    }
    const bool ok = attr.type == cudaMemoryTypeManaged || (attr.type == cudaMemoryTypeDevice && attr.device == b->ctx->device);
    if (!ok)
        throw Error(GAAST_ERR_INVALID, std::string(what) + ": records pointer is not device memory of the batch's device "
                                                           "(host records go through gaast_batch_upload_records / _download_records)");
    cuda_check(gaast::records_launch(*m, unpack, b->esize(), records, (long long)first, (long long)count, b->ctx->stream),
               unpack ? "launch gaast_records_unpack" : "launch gaast_records_pack");
    b->ctx->launches++;
}

// Host entry points: chunks of GAAST_HOST_CHUNK_MIB through the ctx's staging buffer, all on the ctx stream (stream
// order makes the reuse of the one buffer safe): copy, then pack -- or unpack, then copy.
static void records_host(const gaast_batch* b, uint64_t first, uint64_t count, void* host, uint32_t record_mask, bool download) {
    const char* what = download ? "download_records" : "upload_records";
    if (!b) throw Error(GAAST_ERR_INVALID, std::string(what) + ": null batch");
    gaast_ctx* ctx = b->ctx;
    DeviceGuard dg(ctx->device);
    const gaast::RecordMap* m = records_prepare(b, first, count, record_mask, what);
    if (!m) return;
    if (!host) throw Error(GAAST_ERR_INVALID, std::string(what) + ": null host pointer");
    const size_t rec_bytes = size_t(m->K) * b->esize();
    const size_t want = std::max(size_t(gaast::tuning().host_chunk_mib) << 20, rec_bytes);
    if (ctx->staging_bytes != want) {
        if (ctx->staging) {
            cuda_check(cudaStreamSynchronize(ctx->stream), "staging buffer");
            cudaFree(ctx->staging);
            ctx->staging = nullptr;
            ctx->staging_bytes = 0;
        }
        cuda_check(cudaMalloc(&ctx->staging, want), "cudaMalloc(record staging buffer)");
        ctx->staging_bytes = want;
    }
    const uint64_t chunk = ctx->staging_bytes / rec_bytes;
    char* h = static_cast<char*>(host);
    for (uint64_t off = 0; off < count; off += chunk) {
        const uint64_t n = std::min(chunk, count - off);
        char* hp = h + off * rec_bytes;
        if (!download)
            cuda_check(cudaMemcpyAsync(ctx->staging, hp, n * rec_bytes, cudaMemcpyHostToDevice, ctx->stream), "records H2D");
        cuda_check(gaast::records_launch(*m, download, b->esize(), ctx->staging, (long long)(first + off), (long long)n, ctx->stream),
                   download ? "launch gaast_records_unpack" : "launch gaast_records_pack");
        ctx->launches++;
        if (download)
            cuda_check(cudaMemcpyAsync(hp, ctx->staging, n * rec_bytes, cudaMemcpyDeviceToHost, ctx->stream), "records D2H");
    }
}

gaast_status gaast_batch_pack_records(gaast_batch* b, uint64_t first, uint64_t count, const void* records, uint32_t record_mask) {
    return guard([&] { records_device(b, first, count, const_cast<void*>(records), record_mask, false); });
}
gaast_status gaast_batch_unpack_records(const gaast_batch* b, uint64_t first, uint64_t count, void* records,
                                        uint32_t record_mask) {
    return guard([&] { records_device(b, first, count, records, record_mask, true); });
}
gaast_status gaast_batch_upload_records(gaast_batch* b, uint64_t first, uint64_t count, const void* host_records,
                                        uint32_t record_mask) {
    return guard([&] { records_host(b, first, count, const_cast<void*>(host_records), record_mask, false); });
}
gaast_status gaast_batch_download_records(const gaast_batch* b, uint64_t first, uint64_t count, void* host_records,
                                          uint32_t record_mask) {
    return guard([&] { records_host(b, first, count, host_records, record_mask, true); });
}

// ---------------------------------------------------------------- eval ----
static std::shared_ptr<gaast::JitKernel> get_specialized(gaast_plan* plan, const gaast::CodegenOptions& opt) {
    const gaast_plan::JitKey key = opt.key();
    auto it = plan->jit.find(key);
    if (it != plan->jit.end()) {
        // a negative entry: THIS variant failed to build before (other variants of the plan are unaffected)
        if (!it->second) throw Error(GAAST_ERR_JIT, plan->jit_errors[key]);
        return it->second;
    }
    try {
        gaast::CodegenResult cg;
        std::string ckey, origin;
        std::vector<char> cubin = gaast::build_specialized(plan->h, opt, &cg, &ckey, &origin);
        auto k = gaast::jit_load(cg, cubin);
        k->key = ckey;
        k->origin = origin;
        k->fma_per_elem = cg.fma_per_elem;
        plan->jit.emplace(key, k);
        return k;
    } catch (const Error& e) {
        plan->jit.emplace(key, nullptr);
        plan->jit_errors[key] = e.what();
        throw;
    }
}

// build_dense's kernel for n elements on the plan's device, loaded once per launch shape (the matrix kernel is shared by
// every signature of its shape).  Null when it is not wanted or cannot be built (never tried again for the plan): for a
// product, the dense-warp engine then runs the generic kernel compiled into the library.
static std::shared_ptr<gaast::JitKernel> dense_kernel(gaast_plan* plan, long long n, int step) {
    const gaast::DenseWarpHost& prog = plan->dense_warp;
    std::shared_ptr<gaast::JitKernel>* slot;
    if (step >= 0) {
        if (plan->dw_jit_failed || gaast::tuning().dense_warp_generic) return nullptr;
        slot = &plan->dw_jit[std::make_pair(step, gaast::dense_warp_shape(*plan->ctx, prog.n, n).threads)];
    } else {
        if (!wants_matrix_kernel(plan, prog) || plan->dm_jit_failed) return nullptr;
        const gaast::DenseMatLaunch s = gaast::dense_matrix_shape(*plan->ctx, *prog.mat, n);
        slot = &plan->dm_jit[s.RC * 4194304 + s.threads * 8192 + s.T * 64 + s.blocks_per_sm * 4 + int(s.pipe) * 2 + int(s.csep)];
    }
    if (*slot) return *slot;
    try {
        gaast::CodegenResult cg;
        std::string key, origin;
        const std::vector<char> cubin = build_dense(prog, *plan->ctx, n, step, &cg, &key, &origin, nullptr);
        auto k = gaast::jit_load(cg, cubin);
        k->key = key;
        k->origin = origin;
        k->fma_per_elem = cg.fma_per_elem;
        return *slot = k;
    } catch (const Error&) {
        (step >= 0 ? plan->dw_jit_failed : plan->dm_jit_failed) = true;
        return nullptr;
    }
}

// One gaast_eval call, validated and bound to its batches (bind_streams).
struct EvalCall {
    gaast_plan* plan;
    gaast_batch* out;  // null: sums only
    int arith;
    bool with_sum, f32 = false;
    gaast::EvalArgs a{};
    uint64_t bslots = 0;  // broadcast input slots
    long long n = 0;
    std::vector<std::vector<uint64_t>> sparse{};  // the inputs' stored components, and a hash of them
    uint64_t sparse_hash = 0;
};

// Whether the dense-warp engine can evaluate the call: a chain of dense products, f64, FMA arithmetic, per-element
// operands.  The first call analyses the plan and uploads its tables.
static bool dense_warp_ready(EvalCall& c) {
    gaast_plan* plan = c.plan;
    const gaast::DevicePlanHost& h = plan->h;
    if (c.with_sum || c.f32 || c.arith != GAAST_ARITH_FMA || !c.out) return false;
    if (plan->dense_warp_state == 0) {
        plan->dense_warp_state = gaast::dense_warp_analyse(h, &plan->dense_warp) ? 1 : -1;
        if (plan->dense_warp_state == 1) {
            upload(plan->d_dw_blades, plan->dense_warp.blade_of_slot, plan->ctx->stream);
            if (plan->dense_warp.mat) {
                upload(plan->d_dm_src, gaast::matrix_rep_device_table(*plan->dense_warp.mat), plan->ctx->stream);
                upload(plan->d_dm_lx, plan->dense_warp.mat->lx, plan->ctx->stream);
                cuda_check(cudaMalloc(&plan->d_dm_rows, ((size_t(3) << h.n) + (size_t(3) << plan->dense_warp.mat->mx)) *
                                                            sizeof(unsigned long long)),  // row addresses + flag words
                           "cudaMalloc(dense-matrix row tables)");
            }
        }
    }
    if (plan->dense_warp_state != 1) return false;
    if (h.n > 10 && !dense_kernel(plan, c.n, -1)) return false;  // no term-by-term kernel above n = 10: the matrix kernel or nothing
    // products that drop pairs (outer products, contractions) need their per-plan kernel
    for (size_t i = 0; i < plan->dense_warp.steps.size() && !plan->dense_warp.complete; ++i)
        if (!plan->dense_warp.steps[i].prod.complete && !dense_kernel(plan, c.n, int(i))) return false;
    return true;
}

// The launch length of the specialised kernel and whether it can address the batch with 128-bit accesses: every
// per-element row 16-byte aligned and as long as the launch, every stride a whole number of 16 bytes.  An odd-length
// batch (the ragged tail of a chunked run) still takes the aligned kernel when the library owns the output batch: rows
// are padded to 128 bytes, so the launch simply covers the padding column(s) too.  Inputs are only read there;
// caller-owned (wrapped) outputs are never written beyond their length, and a batch-sum must not see the padding.
struct LaunchLength { bool aligned; long long n; };
static LaunchLength launch_length(const EvalCall& c) {
    const gaast::DevicePlanHost& h = c.plan->h;
    const long long quantum = c.f32 ? 4 : 2;  // elements per 16 bytes
    auto rows_fit = [&](long long len) {
        for (size_t i = 0; i < h.streams.size(); ++i) {
            if ((c.a.bcast[i >> 6] >> (i & 63) & 1) || !c.a.sptr[i]) continue;  // (broadcast operands: one element)
            if (c.a.srow[i] < len || (c.a.srow[i] % quantum) || (reinterpret_cast<uintptr_t>(c.a.sptr[i]) & 15)) return false;
        }
        return true;
    };
    if (c.n % quantum == 0) return {rows_fit(c.n), c.n};
    const long long padded = (c.n + quantum - 1) / quantum * quantum;
    if (!c.with_sum && (!c.out || c.out->owned) && rows_fit(padded)) return {true, padded};
    return {false, c.n};
}

enum class Engine { dense_warp, specialized, table };

// Which engine evaluates the call; `*jk` receives the specialised kernel.  AUTO takes the specialised kernel, else a
// dense enough product's dense-warp engine, else the table engine.
static Engine choose_engine(EvalCall& c, int engine, std::shared_ptr<gaast::JitKernel>* jk) {
    const gaast::DevicePlanHost& h = c.plan->h;
    if (engine == GAAST_ENGINE_DENSE_WARP) {
        if (h.projected)
            throw Error(GAAST_ERR_UNSUPPORTED, "dense-warp engine: a projected plan is evaluated by the specialised or the "
                                               "table engine");
        if (!dense_warp_ready(c))
            throw Error(GAAST_ERR_UNSUPPORTED,
                        "dense-warp engine: the plan is not a chain of dense products (geometric, outer, contraction) of "
                        "full-grade per-element f64 operands in G(n), 7 <= n <= 10, with a +-1 metric, evaluated in FMA "
                        "arithmetic without batch-sum");
        return Engine::dense_warp;
    }
    if (engine == GAAST_ENGINE_TABLE) return Engine::table;
    if (engine != GAAST_ENGINE_AUTO && engine != GAAST_ENGINE_SPECIALIZED) throw Error(GAAST_ERR_INVALID, "unknown engine");
    // AUTO: a handful of elements of a plan never specialised before is not worth generating and
    // compiling a kernel for (0.3-3 s): the table engine evaluates it at once.
    const bool any_sparse = !c.sparse.empty();
    if (engine == GAAST_ENGINE_AUTO && c.plan->jit.empty() && !any_sparse &&
        double(c.n) * double(h.total_terms > 0 ? h.total_terms : 1) < 2e6)
        return Engine::table;
    // (a batch widened over the output's padding stays widened for the engine that takes over below)
    const LaunchLength len = launch_length(c);
    c.n = c.a.n = len.n;
    try {
        *jk = get_specialized(c.plan, specialized_options(c.plan, c.bslots, c.arith, c.with_sum, c.out != nullptr, c.f32,
                                                          c.sparse, c.sparse_hash, len.aligned));
        return Engine::specialized;
    } catch (const Error&) {
        // AUTO: this variant cannot be specialised (too large, or no NVRTC and no cached cubin): another engine
        // evaluates it.  The failure is remembered per variant (get_specialized), so an odd-length call that needs
        // another kernel does not take the fast path away from aligned calls.
        if (engine == GAAST_ENGINE_SPECIALIZED || any_sparse) throw;  // (no other engine reads a sparse batch)
    }
    // too large / too wide to specialise: a full high-dimensional product still has a fast engine
    // (the engine always runs COMPLETE 4^n products.  Measured per kept pair: 12-15 TFLOP/s against 1.2-2.1 on
    // the table engine at n = 7, 8 -- worth it while the plan keeps at least 1/8 of the pairs; at n = 9, 10 the
    // table engine's workspace is in global memory (0.09 TFLOP/s): 1/64.  exp/rotor_square.py, exp/big_products.py)
    const double min_density = h.n <= 8 ? 1.0 / 8.0 : 1.0 / 64.0;
    if (!h.projected && dense_warp_ready(c) &&
        double(h.total_terms) >= min_density * double(c.plan->dense_warp.steps.size()) * std::pow(4.0, double(h.n)))
        return Engine::dense_warp;
    return Engine::table;
}

// Points a batch-sum kernel at the plan's partials, sized for the largest grid its engine can launch for the plan so
// that only the first call allocates.
static void bind_partials(EvalCall& c, size_t max_grid) {
    if (!c.with_sum) return;
    ensure(c.plan->d_partials, c.plan->partials_cap, (max_grid + gaast::kReduceStage1Rows) * size_t(c.a.n_sum_cols));
    c.a.partials = c.plan->d_partials;
}

// Each launcher enqueues its engine's kernels, describes them in last_kernel and returns the grid it launched.
static int launch_dense_warp(EvalCall& c) {
    gaast_plan* plan = c.plan;
    gaast_ctx* ctx = plan->ctx;
    const gaast::DevicePlanHost& h = plan->h;
    const gaast::DenseWarpHost& prog = plan->dense_warp;
    const long long n = c.n;
    // scratch buffers for the intermediate products: [2^n][stride], rows on 128-byte boundaries
    const size_t stride = (size_t(n) + 15) / 16 * 16;
    if (plan->d_dw_scratch.size() < size_t(prog.n_scratch) || plan->dw_scratch_stride < stride) {
        for (double* p : plan->d_dw_scratch) cudaFree(p);
        plan->d_dw_scratch.assign(size_t(prog.n_scratch), nullptr);
        plan->dw_scratch_stride = 0;
        for (double*& p : plan->d_dw_scratch)
            cuda_check(cudaMalloc(&p, (size_t(1) << h.n) * stride * sizeof(double)), "cudaMalloc(dense-warp scratch)");
        plan->dw_scratch_stride = stride;
    }
    auto buffers_of = [&](const gaast::DenseWarpOperand& o) {
        gaast::DenseWarpBuffers b;
        size_t root_stream = h.n_in_streams;  // the root's grade arrays follow the inputs, grades ascending
        for (uint32_t k = 0; k <= h.n; ++k) {
            if (!(o.grade_mask >> k & 1)) continue;  // no data / not stored: the kernel never touches it
            if (o.slot >= 0) {
                const int si = h.stream_of(uint32_t(o.slot), k);
                if (si < 0) throw Error(GAAST_ERR_INVALID, "dense-warp engine: the plan has no stream for a grade it reads");
                b.ptr[k] = c.a.sptr[si];
                b.row[k] = c.a.srow[si];
                b.shared = (c.bslots >> o.slot) & 1;  // a fixed operand (the rotor of R X ~R): stride 0
            } else if (o.root) {
                b.ptr[k] = c.a.sptr[root_stream];
                b.row[k] = c.a.srow[root_stream];
                ++root_stream;
            } else {
                b.ptr[k] = plan->d_dw_scratch[size_t(o.scratch)] + size_t(prog.gstart[k]) * plan->dw_scratch_stride;
                b.row[k] = (long long)plan->dw_scratch_stride;
            }
        }
        return b;
    };
    if (std::shared_ptr<gaast::JitKernel> dmk = dense_kernel(plan, n, -1)) {
        const gaast::DenseMatLaunch mshape = gaast::dense_matrix_shape(*ctx, *prog.mat, n);
        for (const gaast::DenseWarpStep& step : prog.steps) {
            cuda_check(gaast::dense_matrix_launch(prog, step, buffers_of(step.L), buffers_of(step.R), buffers_of(step.O),
                                                  step.C.slot >= 0 ? buffers_of(step.C) : gaast::DenseWarpBuffers(), n,
                                                  plan->d_dm_src, plan->d_dm_lx, plan->d_dm_rows, mshape,
                                                  dmk->kernel, ctx->stream),
                       "launch dense-matrix kernel");
            ctx->launches += 2;  // the row-address prologue and the product
        }
        char desc[400];
        std::snprintf(desc, sizeof desc,
                      "gaast_dense_matrix engine=dense_warp kernel=matrix origin=%s products=%zu grid=%d block=%d smem=%zu "
                      "tile=%d elements regs=%d spill=%zuB blocks/SM=%d fma/elem=%d key=%s M%d x%d cols=%d",
                      dmk->origin.c_str(), prog.steps.size(), mshape.grid, mshape.threads, mshape.smem, mshape.T, dmk->regs,
                      dmk->local_bytes, mshape.blocks_per_sm, dmk->fma_per_elem, dmk->key.c_str(), 1 << prog.mat->mx,
                      1 << prog.mat->db, 1 << prog.mat->dl);
        plan->last_kernel = desc;
        return mshape.grid;
    }
    const gaast::DenseWarpLaunch shape = gaast::dense_warp_shape(*ctx, h.n, n);
    std::shared_ptr<gaast::JitKernel> dwk;
    for (size_t i = 0; i < prog.steps.size(); ++i) {
        const gaast::DenseWarpStep& step = prog.steps[i];
        dwk = dense_kernel(plan, n, int(i));
        cuda_check(gaast::dense_warp_launch(prog, step, buffers_of(step.L), buffers_of(step.R), buffers_of(step.O),
                                            step.C.slot >= 0 ? buffers_of(step.C) : gaast::DenseWarpBuffers(), n,
                                            plan->d_dw_blades, shape, dwk ? dwk->kernel : nullptr, ctx->stream),
                   "launch dense-warp engine");
        ctx->launches++;
    }
    char desc[320];
    std::snprintf(desc, sizeof desc,
                  "%s engine=dense_warp origin=%s products=%zu grid=%d block=%d smem=%zu tile=%d elements regs=%d",
                  dwk ? "gaast_dense_warp" : "dense_warp_kernel", dwk ? dwk->origin.c_str() : "library",
                  prog.steps.size(), shape.grid, shape.threads, shape.smem, shape.T, dwk ? dwk->regs : 0);
    plan->last_kernel = desc;
    return shape.grid;
}

static int launch_specialized(EvalCall& c, const gaast::JitKernel& jk) {
    gaast_ctx* ctx = c.plan->ctx;
    const long long per_block = (long long)jk.threads * jk.elems_per_thread;
    const long long blocks = (c.n + per_block - 1) / per_block;
    if (blocks > 0x7fffffffLL) throw Error(GAAST_ERR_SHAPE, "batch too long for one launch");
    int grid = int(blocks);
    size_t max_grid = size_t(grid);
    if ((c.with_sum || jk.pipelined || gaast::tuning().force_persistent) && !jk.one_tile_blocks) {
        // persistent grid: the batch-sum epilogue keeps per-block partials, and the TMA-pipelined
        // kernels loop over their tiles; blocks stride over the batch
        // sum-only kernels: many short-lived blocks overlap better than one long-lived block per resident slot, but
        // every block pays its epilogue (column sums -> partials), so a block should still see ~8 tiles.  Measured
        // on cfg5 + sum (ms per step at 4 / 8 / 16 / 32 / 64 blocks per slot): 32 M elements 6.42 / 6.20 / - / 5.97 /
        // 5.92; 8 M (the 4-GPU shard) 1.577 / 1.535 / 1.505 / 1.501 / 1.558; 4 M (the 8-GPU shard) 0.787 / 0.770 /
        // 0.770 / 0.793 / 0.857.
        const long long resident = (long long)ctx->sm_count * jk.blocks_per_sm;
        long long mult = jk.pipelined ? 1 : std::min(64LL, std::max(4LL, blocks / (8 * resident)));
        if (gaast::tuning().grid_mult > 0) mult = gaast::tuning().grid_mult;
        const long long cap = resident * mult;
        if (grid > cap) grid = int(cap);
        max_grid = size_t(resident * std::max(64LL, mult));  // (>= the capped grid of every call of this variant)
    }
    bind_partials(c, max_grid);
    if (jk.n_uniform > 0) {
        ensure(c.plan->d_uniform, c.plan->uniform_cap, size_t(jk.n_uniform));
        c.a.uniform = c.plan->d_uniform;
        void* params[] = {&c.a};
        cuda_check(cudaLaunchKernel(reinterpret_cast<const void*>(jk.uniform_kernel), dim3(1), dim3(32), params, 0,
                                    ctx->stream),
                   "launch uniform prologue");
        ctx->launches++;
    }
    c.a.lookahead = ctx->sm_count * jk.blocks_per_sm;  // resident blocks: the look-ahead distance of the L2 prefetch variant
    if (gaast::tuning().lookahead >= 0) c.a.lookahead = gaast::tuning().lookahead;
    void* params[] = {&c.a};
    cuda_check(cudaLaunchKernel(reinterpret_cast<const void*>(jk.kernel), dim3(grid), dim3(jk.threads), params, jk.smem_bytes,
                                ctx->stream),
               "launch specialised kernel");
    ctx->launches++;
    char desc[512];
    std::snprintf(desc, sizeof desc,
                  "%s engine=specialized origin=%s grid=%d block=%d elems/thread=%d regs=%d spill=%zuB fma/elem=%d key=%s",
                  jk.name.c_str(), jk.origin.c_str(), grid, jk.threads, jk.elems_per_thread, jk.regs, jk.local_bytes,
                  jk.fma_per_elem, jk.key.c_str());
    c.plan->last_kernel = desc;
    return grid;
}

static int launch_table(EvalCall& c) {
    gaast_plan* plan = c.plan;
    gaast_ctx* ctx = plan->ctx;
    const gaast::TableLaunch shape = gaast::table_engine_shape(*ctx, plan->h, c.n, c.with_sum, c.f32);
    // scratch is sized for the largest grid the engine ever launches (8 blocks per SM)
    const size_t max_grid = std::max(size_t(shape.grid), size_t(ctx->sm_count) * 8);
    if (shape.global_ws) {
        ensure(plan->d_ws, plan->ws_cap, max_grid * shape.ws_doubles_per_block);
        c.a.ws_global = plan->d_ws;
    }
    bind_partials(c, max_grid);
    c.a.micro = plan->d_micro;
    c.a.chunks = plan->d_chunks;
    c.a.n_micro = int(plan->h.micro.size());
    c.a.n_chunks = int(plan->h.chunks.size());
    cuda_check(gaast::table_engine_launch(c.a, shape, c.arith == GAAST_ARITH_STRICT, c.with_sum, c.f32, ctx->stream),
               "launch table engine");
    ctx->launches++;
    char desc[256];
    std::snprintf(desc, sizeof desc, "table_engine_kernel engine=table grid=%d block=%d smem=%zu ws=%s", shape.grid,
                  shape.threads, shape.smem, shape.global_ws ? "global" : "shared");
    plan->last_kernel = desc;
    return shape.grid;
}

static void eval_impl(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out, double* dev_sum,
                      bool with_sum, int engine, int arith) {
    if (!plan) throw Error(GAAST_ERR_INVALID, "null plan");
    gaast_ctx* ctx = plan->ctx;
    if (!ctx) throw Error(GAAST_ERR_NO_DEVICE, "this plan was created without a ctx (offline): it cannot be evaluated");
    if (arith != GAAST_ARITH_FMA && arith != GAAST_ARITH_STRICT) throw Error(GAAST_ERR_INVALID, "unknown arith mode");
    if (with_sum && !dev_sum) throw Error(GAAST_ERR_INVALID, "eval_sum: null sum pointer");
    DeviceGuard dg(ctx->device);
    EvalCall c{plan, out, arith, with_sum};
    int dtype = GAAST_F64;
    bind_streams(plan, inputs, n_inputs, out, !with_sum, c.a, &c.bslots, &c.n, &dtype, &c.sparse, &c.sparse_hash);
    c.f32 = dtype == GAAST_F32;
    if (!c.sparse.empty() && (engine == GAAST_ENGINE_TABLE || engine == GAAST_ENGINE_DENSE_WARP))
        throw Error(GAAST_ERR_UNSUPPORTED, "sparse batches are evaluated by the specialised engine only (the kernel is "
                                           "generated for the sparsity pattern): use GAAST_ENGINE_AUTO or GAAST_ENGINE_SPECIALIZED");
    const int sum_cols = int(plan->h.stored_cols);  // one column per stored root component
    c.a.n_sum_cols = with_sum ? sum_cols : 0;
    if (c.n == 0) {
        if (with_sum) cuda_check(cudaMemsetAsync(dev_sum, 0, sum_cols * sizeof(double), ctx->stream), "zero sum");
        return;
    }
    std::shared_ptr<gaast::JitKernel> jk;
    const Engine e = choose_engine(c, engine, &jk);
    const int grid = e == Engine::dense_warp ? launch_dense_warp(c) : e == Engine::specialized ? launch_specialized(c, *jk)
                                                                                                : launch_table(c);
    if (with_sum) {
        cuda_check(gaast::reduce_partials_launch(plan->d_partials, grid, sum_cols, dev_sum, ctx->stream),
                   "launch partial-sum reduction");
        ctx->launches += (grid > 2048 && sum_cols <= 256) ? 2 : 1;  // (many partial rows: two-level reduction)
    }
}

gaast_status gaast_eval(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out, int engine,
                        int arith) {
    return guard([&] { eval_impl(plan, inputs, n_inputs, out, nullptr, false, engine, arith); });
}

gaast_status gaast_eval_sum(gaast_plan* plan, gaast_batch* const* inputs, uint32_t n_inputs, gaast_batch* out,
                            double* dev_sum, int engine, int arith) {
    return guard([&] { eval_impl(plan, inputs, n_inputs, out, dev_sum, true, engine, arith); });
}

}  // extern "C"
