// gaast_eval_host: host arrays in, host arrays out.  The batch is cut into
// chunks that flow through three device buffer sets, so that the H2D copy of
// chunk i+1, the kernel of chunk i and the D2H copy of chunk i-1 overlap
// (PCIe is full duplex; three streams, events between them).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "../runtime.hpp"

using gaast::Error;

namespace gaast {

struct HostPipe {
    static constexpr int kSets = 3;
    gaast_ctx* ctx = nullptr;
    uint64_t chunk = 0;
    int dtype = GAAST_F64;
    std::vector<uint32_t> masks;
    std::vector<int> bcast;
    std::vector<gaast_batch*> in[kSets];
    gaast_batch* out[kSets] = {};
    cudaEvent_t h2d_done[kSets] = {}, comp_done[kSets] = {}, d2h_done[kSets] = {};
    ~HostPipe() {
        for (int s = 0; s < kSets; ++s) {
            for (gaast_batch* b : in[s])
                if (b) gaast_batch_free(b);
            if (out[s]) gaast_batch_free(out[s]);
            if (h2d_done[s]) cudaEventDestroy(h2d_done[s]);
            if (comp_done[s]) cudaEventDestroy(comp_done[s]);
            if (d2h_done[s]) cudaEventDestroy(d2h_done[s]);
        }
    }
};

void host_pipe_destroy(HostPipe* p) { delete p; }

}  // namespace gaast

namespace {

void ck(cudaError_t e, const char* what) {
    if (e != cudaSuccess) throw Error(GAAST_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
void ckg(gaast_status s) {
    if (s != GAAST_OK) throw Error(s, gaast::last_error());
}

uint32_t rows_of(uint32_t n, uint32_t mask) {
    uint32_t r = 0;
    for (uint32_t k = 0; k <= n; ++k)
        if (mask >> k & 1) r += uint32_t(gaast::binomial(n, k));
    return r;
}

}  // namespace

namespace {
// Restores the caller's current device when the call returns, on every path.
struct ScopedDevice {
    int prev = -1;
    void enter(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) ck(cudaSetDevice(dev), "cudaSetDevice");
    }
    ~ScopedDevice() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};
}  // namespace

static gaast_status eval_host_impl(gaast_plan* plan, const void* const* host_in_v, const uint32_t* in_masks,
                                   const int* in_broadcast, uint32_t n_inputs, uint64_t len, uint64_t host_stride,
                                   void* host_out_v, int dtype, int engine, int arith) {
    ScopedDevice dev_guard;
    gaast::HostPipe* live_pipe = nullptr;  // set once copies may be in flight: the error path drains them
    uint64_t live_chunk = 0;
    // On an error in the middle of the pipeline earlier H2D / D2H copies still touch the caller's host arrays:
    // drain the three streams before returning, and give the buffer sets their full length back.
    auto drain = [&] {
        if (!live_pipe || !plan || !plan->ctx) return;
        gaast_ctx* c = plan->ctx;
        if (c->h2d) cudaStreamSynchronize(c->h2d);
        cudaStreamSynchronize(c->stream);
        if (c->d2h) cudaStreamSynchronize(c->d2h);
        for (int set = 0; set < gaast::HostPipe::kSets; ++set) {
            for (size_t s = 0; s < live_pipe->in[set].size(); ++s)
                if (live_pipe->in[set][s]) live_pipe->in[set][s]->len = live_pipe->bcast[s] ? 1 : live_chunk;
            if (live_pipe->out[set]) live_pipe->out[set]->len = live_chunk;
        }
        cudaGetLastError();
    };
    try {
        if (dtype != GAAST_F64 && dtype != GAAST_F32) throw Error(GAAST_ERR_INVALID, "eval_host: unknown dtype");
        const size_t es = dtype == GAAST_F32 ? 4 : 8;
        const char* const* host_in = reinterpret_cast<const char* const*>(host_in_v);
        char* host_out = static_cast<char*>(host_out_v);
        if (!plan || !plan->ctx) throw Error(GAAST_ERR_INVALID, "eval_host: null or offline plan");
        gaast_ctx* ctx = plan->ctx;
        const auto& h = plan->h;
        if (h.projected)
            throw Error(GAAST_ERR_UNSUPPORTED, "eval_host: a projected plan (gaast_plan_create_projected) writes a sparse "
                                               "output batch: evaluate it with gaast_eval on device batches");
        if (n_inputs != h.n_slots) throw Error(GAAST_ERR_SHAPE, "eval_host: wrong number of inputs");
        if ((n_inputs && (!host_in || !in_masks || !in_broadcast)) || !host_out)
            throw Error(GAAST_ERR_INVALID, "eval_host: null argument");
        if (host_stride < len) throw Error(GAAST_ERR_INVALID, "eval_host: host stride smaller than the batch length");
        dev_guard.enter(ctx->device);
        if (!ctx->h2d) ck(cudaStreamCreateWithFlags(&ctx->h2d, cudaStreamNonBlocking), "stream");
        if (!ctx->d2h) ck(cudaStreamCreateWithFlags(&ctx->d2h, cudaStreamNonBlocking), "stream");

        // chunk: about 32 MiB of the widest side per chunk, a multiple of 4096 elements
        uint32_t in_rows = 0;
        for (uint32_t s = 0; s < n_inputs; ++s)
            if (!in_broadcast[s]) in_rows += rows_of(h.n, in_masks[s]);
        const uint32_t out_rows = h.buf_cols[0];
        const uint32_t wide = std::max<uint32_t>(1, std::max(in_rows, out_rows));
        const uint64_t chunk_mib = uint64_t(gaast::tuning().host_chunk_mib);
        uint64_t chunk = (chunk_mib << 20) / (uint64_t(es) * wide);
        chunk = std::max<uint64_t>(4096, chunk / 4096 * 4096);
        chunk = std::min<uint64_t>(chunk, (len + 4095) / 4096 * 4096);
        if (chunk == 0) chunk = 4096;

        gaast::HostPipe* p = plan->pipe;
        bool rebuild = !p || p->chunk != chunk || p->masks.size() != n_inputs || p->dtype != dtype;
        if (p && !rebuild)
            for (uint32_t s = 0; s < n_inputs; ++s)
                if (p->masks[s] != in_masks[s] || p->bcast[s] != (in_broadcast[s] != 0)) rebuild = true;
        if (rebuild) {
            if (p) gaast::host_pipe_destroy(p);
            plan->pipe = nullptr;
            auto np = std::make_unique<gaast::HostPipe>();
            np->ctx = ctx;
            np->chunk = chunk;
            np->dtype = dtype;
            np->masks.assign(in_masks, in_masks + n_inputs);
            np->bcast.resize(n_inputs);
            for (uint32_t s = 0; s < n_inputs; ++s) np->bcast[s] = in_broadcast[s] != 0;
            for (int set = 0; set < gaast::HostPipe::kSets; ++set) {
                np->in[set].assign(n_inputs, nullptr);
                for (uint32_t s = 0; s < n_inputs; ++s)
                    ckg(gaast_batch_alloc_typed(ctx, h.n, in_masks[s], np->bcast[s] ? 1 : chunk, np->bcast[s], dtype,
                                                &np->in[set][s]));
                ckg(gaast_batch_alloc_typed(ctx, h.n, h.buffer_masks[0], chunk, 0, dtype, &np->out[set]));
                ck(cudaEventCreateWithFlags(&np->h2d_done[set], cudaEventDisableTiming), "event");
                ck(cudaEventCreateWithFlags(&np->comp_done[set], cudaEventDisableTiming), "event");
                ck(cudaEventCreateWithFlags(&np->d2h_done[set], cudaEventDisableTiming), "event");
            }
            plan->pipe = p = np.release();
        }

        auto copy_rows = [&](double* dev, uint64_t dev_stride, const char* host, uint64_t hstride, uint64_t width,
                             uint32_t rows, bool to_dev, cudaStream_t st) {
            if (!rows || !width) return;
            if (to_dev)
                ck(cudaMemcpy2DAsync(dev, dev_stride * es, host, hstride * es, width * es, rows, cudaMemcpyHostToDevice, st),
                   "H2D");
            else
                ck(cudaMemcpy2DAsync(const_cast<char*>(host), hstride * es, dev, dev_stride * es, width * es, rows,
                                     cudaMemcpyDeviceToHost, st),
                   "D2H");
        };

        // the caller's stream must have finished producing before we read; it also owns ordering afterwards
        ck(cudaStreamSynchronize(ctx->stream), "sync");
        live_pipe = p;
        live_chunk = chunk;
        uint64_t it = 0;
        for (uint64_t off = 0; off < len; off += chunk, ++it) {
            const int set = int(it % gaast::HostPipe::kSets);
            const uint64_t w = std::min<uint64_t>(chunk, len - off);
            // H2D (waits until the kernel that last read this set has finished)
            if (it >= gaast::HostPipe::kSets) ck(cudaStreamWaitEvent(ctx->h2d, p->comp_done[set], 0), "wait");
            for (uint32_t s = 0; s < n_inputs; ++s) {
                gaast_batch* b = p->in[set][s];
                const uint32_t rows = rows_of(h.n, in_masks[s]);
                if (p->bcast[s]) {
                    // a shared operand: the host array is [rows] contiguous, one value per component
                    copy_rows(b->base, b->stride, host_in[s], 1, 1, rows, true, ctx->h2d);
                } else {
                    copy_rows(b->base, b->stride, host_in[s] + off * es, host_stride, w, rows, true, ctx->h2d);
                }
                b->len = p->bcast[s] ? 1 : w;
            }
            ck(cudaEventRecord(p->h2d_done[set], ctx->h2d), "record");
            // kernel (waits for its inputs, and for the D2H that last read this set's output)
            ck(cudaStreamWaitEvent(ctx->stream, p->h2d_done[set], 0), "wait");
            if (it >= gaast::HostPipe::kSets) ck(cudaStreamWaitEvent(ctx->stream, p->d2h_done[set], 0), "wait");
            p->out[set]->len = w;
            ckg(gaast_eval(plan, p->in[set].data(), n_inputs, p->out[set], engine, arith));
            ck(cudaEventRecord(p->comp_done[set], ctx->stream), "record");
            // D2H
            ck(cudaStreamWaitEvent(ctx->d2h, p->comp_done[set], 0), "wait");
            copy_rows(p->out[set]->base, p->out[set]->stride, host_out + off * es, host_stride, w, out_rows, false, ctx->d2h);
            ck(cudaEventRecord(p->d2h_done[set], ctx->d2h), "record");
        }
        ck(cudaStreamSynchronize(ctx->d2h), "sync");
        ck(cudaStreamSynchronize(ctx->stream), "sync");
        for (int set = 0; set < gaast::HostPipe::kSets; ++set) {
            for (uint32_t s = 0; s < n_inputs; ++s) p->in[set][s]->len = p->bcast[s] ? 1 : chunk;
            p->out[set]->len = chunk;
        }
        return GAAST_OK;
    } catch (const Error& e) {
        drain();
        gaast::set_last_error(e.what());
        return e.status;
    } catch (const std::exception& e) {
        drain();
        gaast::set_last_error(e.what());
        return GAAST_ERR_INVALID;
    }
}

extern "C" gaast_status gaast_eval_host(gaast_plan* plan, const double* const* host_in, const uint32_t* in_masks,
                                        const int* in_broadcast, uint32_t n_inputs, uint64_t len, uint64_t host_stride,
                                        double* host_out, int engine, int arith) {
    return eval_host_impl(plan, reinterpret_cast<const void* const*>(host_in), in_masks, in_broadcast, n_inputs, len,
                          host_stride, host_out, GAAST_F64, engine, arith);
}

extern "C" gaast_status gaast_eval_host_f32(gaast_plan* plan, const float* const* host_in, const uint32_t* in_masks,
                                            const int* in_broadcast, uint32_t n_inputs, uint64_t len, uint64_t host_stride,
                                            float* host_out, int engine, int arith) {
    return eval_host_impl(plan, reinterpret_cast<const void* const*>(host_in), in_masks, in_broadcast, n_inputs, len,
                          host_stride, host_out, GAAST_F32, engine, arith);
}
