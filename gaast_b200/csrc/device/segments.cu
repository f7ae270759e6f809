// Per-segment sums of a batch's stored rows (gaast_batch_segment_sum).
//
// Segment j is batch columns [O[j], O[j + 1]) of the CSR offsets O[0..n].  The batch is cut into chunks of kSegChunk
// consecutive columns, independent of the segments, and the chunk size alone fixes the order of the additions:
//   piece     the part of a segment inside one chunk.  Lane l (0..31) of a warp sums the piece's columns c with
//             c % 32 == l, in ascending order, starting from +0.0; the 32 lane partials (+0.0 for a lane without a
//             column) are added in the aligned binary tree over lane positions: (0,1) (2,3) ..., then pairs of pairs.
//   segment   inside one chunk: its piece.  Across chunks: its pieces p_0 .. p_{m-1} in chunk order, added in the
//             pairwise tree P(p_0..p_{m-1}) = P(p_0..p_{h-1}) + P(p_h..p_{m-1}), h the largest power of two below m.
//   empty     +0.0.
// No partial sum is ever -0.0 (each starts from +0.0), so an absent lane or leaf can be read as +0.0: the masked
// trees below and the zero-padded ones give the same bits.
//
// gaast_segment_pieces (one block per chunk and group of rows, one warp per one or two rows) walks its chunk in windows
// of 32 aligned columns.  Each lane finds the segment of its column from a cursor and one load of the next 32
// offsets; a piece that starts and ends in the chunk is written to the sums, the piece of a segment that started in an
// earlier chunk goes to the chunk's `head` partial, the piece of one that continues past the chunk to its `tail`
// partial.  The block also writes +0 for the empty segments it owns (those whose first column lies in the chunk) and
// checks the offsets of those segments.  gaast_segment_spans then adds the pieces of every segment that spans chunks
// (one warp per segment and row), or writes NaN everywhere when some chunk found the offsets invalid, and resets that
// flag for the next call.  Two launches per call, whatever the offsets.
#include <algorithm>
#include <climits>

#include "../runtime.hpp"

namespace gaast {

// ---- device code: tests/kernel_emu/segments.py compiles the text from here to the launch helpers on the host ----
#ifndef GAAST_SEGMENT_CHUNK
#define GAAST_SEGMENT_CHUNK 4096
#endif
constexpr long long kSegChunk = GAAST_SEGMENT_CHUNK;  // columns per chunk: a multiple of 32
constexpr int kSegThreads = 256;
constexpr unsigned kSegFull = 0xffffffffu;

struct SegmentArgs {
    const RecordRow* rows;     // [S]: the stored rows, in the order of the sums
    const long long* offsets;  // [n + 1]
    long long n, len, n_chunks;
    int S;
    double* sums;     // [n][S]
    double* head;     // [S][n_chunks]: piece of the segment that started in an earlier chunk
    double* tail;     // [S][n_chunks]: piece of the segment that continues into the next chunk
    long long* span;  // [n_chunks]: the segment that starts in this chunk and spans chunks, or -1
    unsigned long long* state;  // [0]: offsets found invalid, [1]: blocks of gaast_segment_spans done
};

// #{m in [0, m_end) : O[m] <= key} for non-decreasing O, by one warp: a 32-ary search, a probe per lane and step.  For
// any O the result is in [0, m_end] and never decreases when `key` grows, so the chunks' ranges of owned segments
// partition [0, n) whatever the offsets are.
__device__ __forceinline__ long long seg_count_le(const long long* O, long long m_end, long long key, int lane) {
    long long lo = 0, hi = m_end;  // the count lies in [lo, hi]
    while (lo < hi) {
        const long long step = (hi - lo + 31) / 32;
        const bool probe = lo + (long long)lane * step < hi;
        const long long q = min(lo + (long long)(lane + 1) * step, hi) - 1;  // the last element of the lane's block
        const unsigned fail = __ballot_sync(kSegFull, probe && O[q] > key);
        if (!fail) {
            lo = hi;
        } else {
            const int t = __ffs(int(fail)) - 1;  // the first block whose last element exceeds key
            hi = min(lo + (long long)(t + 1) * step, hi) - 1;
            lo += (long long)t * step;
        }
    }
    return lo;
}

// The aligned binary tree over lane positions, over the lanes whose bit s of `same` says that the partner half of step
// s holds lanes of their own segment: every lane ends with the sum over its segment's lanes.
__device__ __forceinline__ double seg_tree(double v, unsigned same, int lane) {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const int d = 1 << s;
        const int src = (lane & d) ? ((lane & ~d) | (d - 1)) : ((lane | d) & ~(d - 1));  // the partner half's nearest lane
        const double u = __shfl_sync(kSegFull, v, src);
        if (same >> s & 1) v = (lane & d) ? u + v : v + u;
    }
    return v;
}

// The same tree over all 32 lanes.
__device__ __forceinline__ double seg_tree_all(double v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) v = v + __shfl_xor_sync(kSegFull, v, d);
    return v;
}

// Segment of each lane's column `col` in the window starting at `ws`: the largest j with O[j] <= col (-1 before O[0],
// n from O[n] on), from J = that of column ws - 1.  *nb receives O[key + 1], the column where the lane's segment ends;
// *quiet is set when no segment starts in the window.
__device__ __forceinline__ long long seg_keys(const long long* O, long long n, long long J, long long ws, long long col,
                                              int lane, long long* nb, bool* quiet) {
    const long long next = J + 1 <= n ? O[J + 1] : LLONG_MAX;  // (the same address for every lane)
    *quiet = next > ws + 31;
    if (*quiet) {  // the common case of long segments
        *nb = next;
        return J;
    }
    long long key = J, base = J;
    bool done = false;
    for (;;) {  // 32 offsets at a time: as many rounds as the window has boundaries / 32, plus one
        const long long idx = base + 1 + lane;
        const long long b = idx <= n ? O[idx] : LLONG_MAX;
        // cnt = #{m : b_m <= col} by a binary search over the lanes (b is sorted when the offsets are)
        int lo = 0;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1)
            if (__shfl_sync(kSegFull, b, lo + s - 1) <= col) lo += s;
        const long long at = __shfl_sync(kSegFull, b, lo);
        const int cnt = lo + (at <= col ? 1 : 0);
        const long long end = __shfl_sync(kSegFull, b, min(cnt, 31));
        if (!done) {
            key = min(base + cnt, n);
            *nb = cnt < 32 ? end : LLONG_MAX;
            done = cnt < 32;
        }
        if (__all_sync(kSegFull, done)) break;
        base += 32;
    }
    return key;
}

// Where the piece of segment `key` (ending at column `end`) goes for row r: the chunk's head or tail partial, or the sum.
__device__ __forceinline__ double* seg_dest(const SegmentArgs& a, long long key, long long end, int r, long long head,
                                             long long c, long long c0) {
    if (key == head) return a.head + (long long)r * a.n_chunks + c;
    if (end > c0 + kSegChunk) return a.tail + (long long)r * a.n_chunks + c;
    return a.sums + key * a.S + r;
}

template <class T, int R, int U>  // R rows per warp, U windows loaded per step (R * U = 4 loads in flight per lane)
__global__ void __launch_bounds__(kSegThreads, 3) gaast_segment_pieces(const __grid_constant__ SegmentArgs a) {
    const int lane = int(threadIdx.x & 31), warp = int(threadIdx.x >> 5);
    const long long* O = a.offsets;
    const long long n = a.n, c = blockIdx.x, c0 = c * kSegChunk, cend = min(c0 + kSegChunk, a.len);
    const long long NC = a.n_chunks;
    // the segments the chunk owns: those whose first column lies in it (the first and the last chunk: all before / after)
    const long long own0 = c == 0 ? 0 : seg_count_le(O, n, c0 - 1, lane);
    const long long own1 = c == NC - 1 ? n : seg_count_le(O, n, c0 + kSegChunk - 1, lane);
    const int row0 = int(blockIdx.y) * 8 * R + warp * R;
    const int nr = min(R, a.S - row0);
    if (blockIdx.y == 0 && warp == 0) {  // check the owned offsets; note the segment that spans chunks from here
        bool bad = (c == 0 && O[0] < 0) || (c == NC - 1 && O[n] > a.len);
        for (long long j = own0 + lane; j < own1; j += 32) bad |= O[j + 1] < O[j];
        if (__any_sync(kSegFull, bad) && lane == 0) a.state[0] = 1ull;
        if (lane == 0) a.span[c] = (c + 1 < NC && own1 > own0 && O[own1] > c0 + kSegChunk) ? own1 - 1 : -1;
    }
    if (nr <= 0) return;
    for (long long j = own0 + lane; j < own1; j += 32)  // empty owned segments: +0
        if (O[j + 1] <= O[j])
            for (int k = 0; k < nr; ++k) a.sums[j * a.S + row0 + k] = 0.0;
    const T* p[R];
#pragma unroll
    for (int k = 0; k < R; ++k) p[k] = reinterpret_cast<const T*>(a.rows[row0 + min(k, nr - 1)].ptr);
    const long long head = own0 - 1;  // the segment holding column c0 - 1 (if any): its piece here is the head piece
    long long J = head;               // cursor: the segment of the column before the window
    long long prevkey = LLONG_MIN;    // the lane's segment one window back (none before the chunk's first window)
    double acc[R];
#pragma unroll
    for (int k = 0; k < R; ++k) acc[k] = 0.0;
    const long long nwin = cend > c0 ? (cend - c0 + 31) / 32 : 0;
        for (long long w0 = 0; w0 < nwin; w0 += U) {
        double x[U][R];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long col = c0 + (w0 + u) * 32 + lane;
#pragma unroll
            for (int k = 0; k < R; ++k) x[u][k] = (k < nr && col < a.len) ? double(__ldg(p[k] + col)) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long w = w0 + u;
            if (w >= nwin) break;
            const long long ws = c0 + w * 32, col = ws + lane;
            long long nb;
            bool quiet;
            long long key = seg_keys(O, n, J, ws, col, lane, &nb, &quiet);
            if (quiet && nb > ws + 32 && ws + 32 < cend) {  // nothing starts or ends in the window: add and go on
#pragma unroll
                for (int k = 0; k < R; ++k) acc[k] = (key == prevkey ? acc[k] : 0.0) + x[u][k];
                prevkey = key;
                continue;
            }
            if (col >= a.len) key = -1;
            const bool valid = key >= 0 && key < n;
            const bool ends = valid && (nb <= col + 1 || col + 1 == cend);  // the lane holds its piece's last column
            const long long p0 = __shfl_sync(kSegFull, key, 0);
            const long long end0 = __shfl_sync(kSegFull, nb, 0);
            // the first lane's segment was already under way in the previous window: lanes past its end carry its
            // partials from there
            const bool carried = w > 0 && p0 == J && p0 >= 0 && p0 < n;
            unsigned same = 0;
#pragma unroll
            for (int s = 0; s < 5; ++s) {
                const int d = 1 << s;
                const int src = (lane & d) ? ((lane & ~d) | (d - 1)) : ((lane | d) & ~(d - 1));
                if (__shfl_sync(kSegFull, key, src) == key) same |= 1u << s;
            }
            const bool mine = ends && !(carried && key == p0);  // a piece this lane writes from the segmented tree
            const bool need_x = __any_sync(kSegFull, mine);
            const bool need_y = carried && __any_sync(kSegFull, ends && key == p0);
#pragma unroll
            for (int k = 0; k < R; ++k) {
                if (k >= nr) break;
                double carry = 0.0;
                if (key == prevkey) {
                    acc[k] = acc[k] + x[u][k];
                } else {
                    carry = acc[k];
                    acc[k] = 0.0 + x[u][k];
                }
                if (need_x) {
                    const double v = seg_tree(acc[k], same, lane);
                    if (mine) *seg_dest(a, key, nb, row0 + k, head, c, c0) = v;
                }
                if (need_y) {
                    const double v = seg_tree_all(key == p0 ? acc[k] : (prevkey == p0 ? carry : 0.0));
                    if (lane == 0) *seg_dest(a, p0, end0, row0 + k, head, c, c0) = v;
                }
            }
            prevkey = key;
            J = __shfl_sync(kSegFull, key, 31);
        }
    }
}

// Adds the pieces of the segments that span chunks (block x = the chunk they start in, one warp per row), or writes NaN
// over every sum when a chunk found the offsets invalid.  The last block to finish clears the flag for the next call.
__global__ void __launch_bounds__(kSegThreads) gaast_segment_spans(const __grid_constant__ SegmentArgs a) {
    const int lane = int(threadIdx.x & 31), warp = int(threadIdx.x >> 5);
    const long long c = blockIdx.x, NC = a.n_chunks, n = a.n;
    const long long* O = a.offsets;
    const int r = int(blockIdx.y) * 8 + warp;
    const bool bad = *reinterpret_cast<volatile unsigned long long*>(a.state) != 0ull;
    if (r < a.S) {
        if (bad) {
            const long long c0 = c * kSegChunk;
            const long long own0 = c == 0 ? 0 : seg_count_le(O, n, c0 - 1, lane);
            const long long own1 = c == NC - 1 ? n : seg_count_le(O, n, c0 + kSegChunk - 1, lane);
            for (long long j = own0 + lane; j < own1; j += 32) a.sums[j * a.S + r] = __longlong_as_double(0x7ff8000000000000LL);
        } else if (a.span[c] >= 0) {
            const long long j = a.span[c];
            const long long ce = min(NC - 1, (min(O[j + 1], a.len) - 1) / kSegChunk);
            const long long m = ce - c + 1;  // pieces: tail[c], head[c + 1 .. ce]
            const double* hrow = a.head + (long long)r * NC;
            const double t0 = a.tail[(long long)r * NC + c];
            auto leaf = [&](long long i) { return i == 0 ? t0 : (i < m ? hrow[c + i] : 0.0); };
            // groups of 32 pieces, each by the tree over lanes; the group sums by a binary counter whose pending
            // subtree of 2^L groups lives in lane L
            double st = 0.0;
            const long long G = (m + 31) / 32;
            for (long long g0 = 0; g0 < G; g0 += 4) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = leaf((g0 + u) * 32 + lane);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const long long g = g0 + u;
                    if (g >= G) break;
                    double s = seg_tree_all(v[u]);
                    int L = 0;
                    for (; (g >> L) & 1; ++L) s = __shfl_sync(kSegFull, st, L) + s;
                    if (lane == L) st = s;
                }
            }
            double total = 0.0;
            bool first = true;
            for (int L = 0; L < 64 && (G >> L) != 0; ++L) {  // the complete subtrees, smallest first
                if (!((G >> L) & 1)) continue;
                const double s = __shfl_sync(kSegFull, st, L);
                total = first ? s : s + total;
                first = false;
            }
            if (lane == 0) a.sums[j * a.S + r] = total;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long done = atomicAdd(a.state + 1, 1ull);
        if (done == (unsigned long long)gridDim.x * gridDim.y - 1) {  // every block has read the flag
            a.state[0] = 0ull;
            a.state[1] = 0ull;
        }
    }
}
// ---- end of device code ----

namespace {
template <class T>
const void* pieces_kernel(int R) {
    if (R == 2) return reinterpret_cast<const void*>(&gaast_segment_pieces<T, 2, 2>);
    return reinterpret_cast<const void*>(&gaast_segment_pieces<T, 1, 4>);
}
}  // namespace

size_t segment_scratch_bytes(long long len, int S) {
    const long long NC = std::max(1LL, (len + kSegChunk - 1) / kSegChunk);
    return 32 + size_t(NC) * sizeof(long long) + 2 * size_t(NC) * size_t(S) * sizeof(double);
}

cudaError_t segment_sum_launch(const RecordRow* rows, int S, size_t es, long long len, const long long* offsets,
                               long long n, double* sums, void* scratch, cudaStream_t stream) {
    SegmentArgs a;
    a.rows = rows;
    a.offsets = offsets;
    a.n = n;
    a.len = len;
    a.n_chunks = std::max(1LL, (len + kSegChunk - 1) / kSegChunk);
    a.S = S;
    a.sums = sums;
    char* p = static_cast<char*>(scratch);
    a.state = reinterpret_cast<unsigned long long*>(p);  // (zeroed when the scratch is allocated; the span kernel leaves it so)
    p += 32;
    a.span = reinterpret_cast<long long*>(p);
    p += size_t(a.n_chunks) * sizeof(long long);
    a.head = reinterpret_cast<double*>(p);
    a.tail = a.head + size_t(a.n_chunks) * size_t(S);
    const int R = S >= 16 ? 2 : 1;
    void* params[] = {&a};
    const dim3 grid1(unsigned(a.n_chunks), unsigned((S + 8 * R - 1) / (8 * R)));
    cudaError_t e = cudaLaunchKernel(es == 4 ? pieces_kernel<float>(R) : pieces_kernel<double>(R), grid1, dim3(kSegThreads),
                                     params, 0, stream);
    if (e != cudaSuccess) return e;
    const dim3 grid2(unsigned(a.n_chunks), unsigned((S + 7) / 8));
    return cudaLaunchKernel(reinterpret_cast<const void*>(&gaast_segment_spans), grid2, dim3(kSegThreads), params, 0, stream);
}

long long segment_chunk() { return kSegChunk; }

}  // namespace gaast
