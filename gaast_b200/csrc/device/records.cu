// Element-major records <-> the batch's per-grade rows (gaast_batch_pack_records / _unpack_records).
//
// A record is one multivector stored contiguously: K scalars, the components of the record mask's grades in
// slot order.  Records [count][K] and the batch's rows [row][stride] are the two sides of a transpose.  A block
// takes one tile -- E consecutive elements x a chunk of Kc record components -- through shared memory:
//   record side: the tile's records are contiguous when the chunk is the whole record (one flat span), else one
//                span of Kc scalars per record; 16-byte accesses on the aligned body of a span, scalar ones at
//                its ragged ends (the records pointer is only scalar-aligned);
//   batch side:  one warp moves 32 consecutive elements of one stored row.
// The tile pitch is odd (in scalars), so that a warp reading or writing one component of 32 consecutive elements
// touches 32 different banks, f64 and f32 alike.  Scalars are moved as 32- or 64-bit integers: bits, not values.
// Stored rows are in record-component order (grades ascending on both sides, components ascending within a
// grade), so the rows of a component chunk are one contiguous range of the row table.
#include <cuda_pipeline.h>

#include <algorithm>

#include "../runtime.hpp"

namespace gaast {
namespace {
constexpr int kThreads = 256;

}  // namespace

struct RecordArgs {
    const RecordRow* rows;  // [stored rows]: row address (column 0) and record component
    const uint32_t* chunk_row;     // [n_chunks + 1]: the rows of component chunk q are [chunk_row[q], chunk_row[q + 1])
    void* rec;                     // record 0 = batch column `first`
    long long first, count;
    long long n_tiles;
    int K, Kc, E, pitch, n_chunks;
    int tile_scalars;  // unpack: scalars per tile buffer (E * pitch, rounded up to 16 bytes)
    int rows_bytes;    // shared memory ahead of the tile(s): the rows of one chunk
};

namespace {

// Moves the flat span g[0, N) of records to / from the tile: scalar i of the span is tile[(i / L) * pitch + i % L].
// Called by `nth` threads (thread `tid` of them) together.
template <class T, bool kToTile, int kSpanUnroll>  // (16-byte record accesses in flight per thread)
__device__ __forceinline__ void span_copy(T* g, int N, T* tile, int L, int pitch, int tid, int nth) {
    constexpr int V = 16 / sizeof(T);
    auto at = [&](int i) -> T& {
        const int r = i / L;
        return tile[r * pitch + (i - r * L)];
    };
    const int head = min(N, int((16 - (reinterpret_cast<uintptr_t>(g) & 15)) & 15) / int(sizeof(T)));
    const int nv = (N - head) / V;
    const int body_end = head + nv * V;
    for (int i = tid; i < head; i += nth) {
        if (kToTile) at(i) = g[i];
        else g[i] = at(i);
    }
    for (int i = body_end + tid; i < N; i += nth) {
        if (kToTile) at(i) = g[i];
        else g[i] = at(i);
    }
    uint4* gv = reinterpret_cast<uint4*>(g + head);
    for (int v0 = tid; v0 < nv; v0 += kSpanUnroll * nth) {
        uint4 x[kSpanUnroll];
        if (kToTile) {
#pragma unroll
            for (int u = 0; u < kSpanUnroll; ++u)
                if (v0 + u * nth < nv) x[u] = gv[v0 + u * nth];
        }
#pragma unroll
        for (int u = 0; u < kSpanUnroll; ++u) {
            const int v = v0 + u * nth;
            if (v >= nv) break;
            T* s = reinterpret_cast<T*>(&x[u]);
            const int i = head + v * V;
            int r = i / L, c = i - r * L;
#pragma unroll
            for (int j = 0; j < V; ++j) {
                T& t = tile[r * pitch + c];
                if (kToTile) t = s[j];
                else s[j] = t;
                if (++c == L) {
                    c = 0;
                    ++r;
                }
            }
            if (!kToTile) gv[v] = x[u];
        }
    }
}

// Records -> tile, or tile -> records, for the tile of elements [e0, e0 + ne) x components [c0, c0 + nc).
template <class T, bool kToTile>
__device__ __forceinline__ void record_side(const RecordArgs& a, T* tile, long long e0, int ne, int c0, int nc) {
    T* rec = static_cast<T*>(a.rec);
    if (nc == a.K) {  // whole records: one contiguous span
        span_copy<T, kToTile, 6>(rec + e0 * a.K, ne * a.K, tile, a.K, a.pitch, threadIdx.x, kThreads);
    } else {          // a chunk of each record: one span per record, one warp per span
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        for (int e = warp; e < ne; e += kThreads / 32)
            span_copy<T, kToTile, 2>(rec + (e0 + e) * a.K + c0, nc, tile + e * a.pitch, nc, a.pitch, lane, 32);
    }
}

// The rows of component chunk q into shared memory (the row loops read them once per pair; from global memory each
// read would wait on a load the streaming traffic has evicted from L1).  With one chunk a block loads them once.
__device__ __forceinline__ void load_rows(const RecordArgs& a, RecordRow* srows, int q) {
    const int r0 = int(a.chunk_row[q]), nrows = int(a.chunk_row[q + 1]) - r0;
    for (int i = threadIdx.x; i < nrows; i += kThreads) srows[i] = a.rows[r0 + i];
}

}  // namespace

template <class T>
__global__ void __launch_bounds__(kThreads, 4) gaast_records_pack(const __grid_constant__ RecordArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RecordRow* const srows = reinterpret_cast<RecordRow*>(smem_raw);
    T* tile = reinterpret_cast<T*>(smem_raw + a.rows_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (a.n_chunks == 1) load_rows(a, srows, 0);
    for (long long t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
        const int q = int(t % a.n_chunks);
        const long long e0 = t / a.n_chunks * a.E;
        const int ne = int(min((long long)a.E, a.count - e0));
        const int c0 = q * a.Kc, nc = min(a.Kc, a.K - c0);
        if (a.n_chunks > 1) load_rows(a, srows, q);
        record_side<T, true>(a, tile, e0, ne, c0, nc);
        __syncthreads();
        const int nrows = int(a.chunk_row[q + 1] - a.chunk_row[q]);
        const int groups = (ne + 31) >> 5;
        for (int p = warp; p < nrows * groups; p += kThreads / 32) {
            const int r = p / groups, e = (p - r * groups) * 32 + lane;
            const RecordRow row = srows[r];
            if (e < ne) reinterpret_cast<T*>(row.ptr)[a.first + e0 + e] = tile[e * a.pitch + (int(row.comp) - c0)];
        }
        __syncthreads();
    }
}

// Issues the batch-row loads of one unpack tile straight into shared memory (cp.async: no register staging, so the
// whole tile is in flight at once), after a +0 fill when the chunk has components the batch does not store.
template <class T>
__device__ __forceinline__ void unpack_issue(const RecordArgs& a, RecordRow* srows, T* tile, long long t) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = int(t % a.n_chunks);
    const long long e0 = t / a.n_chunks * a.E;
    const int ne = int(min((long long)a.E, a.count - e0));
    const int c0 = q * a.Kc, nc = min(a.Kc, a.K - c0);
    const int nrows = int(a.chunk_row[q + 1] - a.chunk_row[q]);
    if (nrows < nc) {  // components the batch does not store: +0 in the record
        for (int i = threadIdx.x; i < ne * a.pitch; i += kThreads) tile[i] = T(0);
    }
    if (a.n_chunks > 1) {
        __syncthreads();  // every thread has issued the previous tile's copies from the row table
        load_rows(a, srows, q);
    }
    if (nrows < nc || a.n_chunks > 1) __syncthreads();
    const int groups = (ne + 31) >> 5;
    const int pairs = nrows * groups;
    for (int p = warp; p < pairs; p += kThreads / 32) {
        const int r = p / groups, e = (p - r * groups) * 32 + lane;
        const RecordRow row = srows[r];
        if (e < ne)
            __pipeline_memcpy_async(&tile[e * a.pitch + (int(row.comp) - c0)],
                                    reinterpret_cast<const T*>(row.ptr) + a.first + e0 + e, sizeof(T));
    }
    __pipeline_commit();
}

// Two tiles per block: the row loads of the next tile are in flight while the current one is written out as records.
template <class T>
__global__ void __launch_bounds__(kThreads, 4) gaast_records_unpack(const __grid_constant__ RecordArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RecordRow* const srows = reinterpret_cast<RecordRow*>(smem_raw);
    T* const buf0 = reinterpret_cast<T*>(smem_raw + a.rows_bytes);
    T* const buf1 = buf0 + a.tile_scalars;
    long long t = blockIdx.x;
    if (a.n_chunks == 1) {
        load_rows(a, srows, 0);
        __syncthreads();
    }
    if (t < a.n_tiles) unpack_issue<T>(a, srows, buf0, t);
    for (int cur = 0; t < a.n_tiles; t += gridDim.x, cur ^= 1) {
        if (t + gridDim.x < a.n_tiles) {
            unpack_issue<T>(a, srows, cur ? buf0 : buf1, t + gridDim.x);
            __pipeline_wait_prior(1);  // every group but the one just issued: the current tile has landed
        } else {
            __pipeline_wait_prior(0);
        }
        __syncthreads();
        const int q = int(t % a.n_chunks);
        const long long e0 = t / a.n_chunks * a.E;
        const int ne = int(min((long long)a.E, a.count - e0));
        const int c0 = q * a.Kc, nc = min(a.Kc, a.K - c0);
        record_side<T, false>(a, cur ? buf1 : buf0, e0, ne, c0, nc);
        __syncthreads();  // (the buffer is refilled by the next iteration's issue)
    }
}

namespace {
template <class T>
const void* kernel_of(bool unpack) {
    return unpack ? reinterpret_cast<const void*>(&gaast_records_unpack<T>) : reinterpret_cast<const void*>(&gaast_records_pack<T>);
}
}  // namespace

// Tile shape for records of K scalars of `es` bytes: about 32 KB of shared memory, at most 48 KB (unpack keeps two),
// behind the chunk's row table.
// Records of up to 48 KB / 32 / es components are moved whole (E elements at a time, E a multiple of 32 close to
// 32 KB / (pitch * es), at most 1024); wider ones in chunks of 1 KB of each record, 32 elements at a time.
void records_shape(RecordMap& m, int K, size_t es, int sm_count) {
    const int limit = 48 * 1024;
    m.K = K;
    m.Kc = (32 * size_t(K + 1) * es <= size_t(limit)) ? K : int(1024 / es);
    m.pitch = m.Kc | 1;
    const size_t row_bytes = size_t(m.pitch) * es;
    int E = int((32 * 1024 / row_bytes + 16) / 32 * 32);
    E = std::max(32, std::min({E, 1024, int(limit / row_bytes) / 32 * 32}));
    m.E = E;
    m.n_chunks = (K + m.Kc - 1) / m.Kc;
    m.rows_bytes = int(size_t(m.Kc) * sizeof(RecordRow));
    m.tile_scalars = int((size_t(E) * row_bytes + 15) / 16 * 16 / es);
    m.smem = size_t(m.rows_bytes) + size_t(m.tile_scalars) * es;             // up to 54 KB, an opt-in
    m.unpack_smem = size_t(m.rows_bytes) + 2 * size_t(m.tile_scalars) * es;  // double-buffered: up to 102 KB
    auto grid_of = [&](const void* k, size_t smem) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
        cudaGetLastError();
        return std::max(1, per_sm * sm_count);
    };
    const void* unpack = es == 4 ? kernel_of<uint32_t>(true) : kernel_of<unsigned long long>(true);
    const void* pack = es == 4 ? kernel_of<uint32_t>(false) : kernel_of<unsigned long long>(false);
    // the largest any shape asks for (two 48 KB tiles behind 383 rows), so that no map lowers another's limit
    const int opt_in = 2 * limit + 8 * 1024;
    cudaFuncSetAttribute(unpack, cudaFuncAttributeMaxDynamicSharedMemorySize, opt_in);
    cudaFuncSetAttribute(pack, cudaFuncAttributeMaxDynamicSharedMemorySize, opt_in);
    cudaGetLastError();
    m.max_grid = grid_of(pack, m.smem);
    m.unpack_max_grid = grid_of(unpack, m.unpack_smem);
}

cudaError_t records_launch(const RecordMap& m, bool unpack, size_t es, void* records, long long first, long long count,
                           cudaStream_t stream) {
    RecordArgs a;
    a.rows = reinterpret_cast<const RecordRow*>(m.d_table);
    a.chunk_row = reinterpret_cast<const uint32_t*>(static_cast<const char*>(m.d_table) + m.n_rows * sizeof(RecordRow));
    a.rec = records;
    a.first = first;
    a.count = count;
    a.n_tiles = (count + m.E - 1) / m.E * m.n_chunks;
    a.K = m.K;
    a.Kc = m.Kc;
    a.E = m.E;
    a.pitch = m.pitch;
    a.n_chunks = m.n_chunks;
    a.tile_scalars = m.tile_scalars;
    a.rows_bytes = m.rows_bytes;
    const int grid = int(std::min<long long>(a.n_tiles, unpack ? m.unpack_max_grid : m.max_grid));
    void* params[] = {&a};
    const void* k = es == 4 ? kernel_of<uint32_t>(unpack) : kernel_of<unsigned long long>(unpack);
    return cudaLaunchKernel(k, dim3(grid), dim3(kThreads), params, unpack ? m.unpack_smem : m.smem, stream);
}

}  // namespace gaast
