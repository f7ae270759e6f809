// Device-side view of a plan: validated copy of the flat description plus the
// derived layouts every engine needs (buffer columns, input/output streams,
// micro-ops, output-sorted term chunks).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "common.hpp"
#include "eval_args.h"

namespace gaast {

constexpr int kMaxStreams = GAAST_MAX_STREAMS;  // (input, grade) and (root, grade) arrays a kernel can address
constexpr int kChunkTerms = 512;    // terms per TMA-staged chunk of the table engine
constexpr int kChunkRunSlots = 520; // u16 run starts per chunk (kChunkTerms + 1, padded to 16 B)

// One (batch input, grade) or (root, grade) device array.
struct Stream {
    uint32_t slot;    // BATCH slot, or UINT32_MAX for the root output
    uint32_t grade;
    uint32_t rows;    // C(n, grade)
};

// What the table engine executes; one per contiguous run of rows.
enum MicroKind : uint32_t { MK_LOAD_ADD = 0, MK_CONST_ADD, MK_MUL, MK_NEG, MK_INV, MK_SQRT, MK_STORE, MK_EXP, MK_LOG };
// MK_EXP / MK_LOG: dst_col = first column of grade k in the destination, a = first column of grade k in the source,
// b = column of grade 0 (EXP: in the destination, LOG: in the source), count = C(n,k), chunk0 = offset of the
// components' blade squares in the plan's constants.
struct MicroOp {
    uint32_t kind;
    uint32_t dst_col;  // first workspace column written (MK_STORE: read)
    uint32_t a;        // LOAD_ADD/STORE: stream id; CONST_ADD: const offset; MUL: left column base
    uint32_t b;        // LOAD_ADD/STORE: first row in the stream; MUL: right column base
    uint32_t count;    // rows / columns; MUL: number of chunks
    uint32_t chunk0;   // MUL: first chunk record
    uint32_t pad0;     // STORE: first batch-sum column of the run
    uint32_t pad1;
};

// A fixed-size record the table engine pulls into shared memory with one
// cp.async.bulk (TMA) copy.  Terms are stably sorted by output slot, so a run
// [run_start[r], run_start[r+1]) accumulates one output in reference order.
struct alignas(16) TermChunk {
    uint32_t n_terms;
    uint32_t n_runs;
    uint32_t pad[2];
    uint16_t run_start[kChunkRunSlots];
    gaast_term terms[kChunkTerms];
};
static_assert(sizeof(TermChunk) % 16 == 0, "TMA bulk copies need 16-byte multiples");

struct DevicePlanHost {
    // validated copies
    uint32_t n = 0, n_slots = 0;
    std::vector<uint32_t> buffer_masks;
    std::vector<gaast_input_desc> inputs;
    std::vector<double> const_values;
    std::vector<gaast_op> ops;
    std::vector<gaast_term> terms;
    // derived
    std::vector<uint32_t> gdim;        // C(n,k)
    std::vector<uint32_t> buf_col;     // first workspace column of each buffer
    std::vector<uint32_t> buf_cols;    // columns in each buffer
    uint32_t total_cols = 0;
    std::vector<Stream> streams;       // inputs first, then root grades
    uint32_t n_in_streams = 0;
    std::vector<uint32_t> slot_masks;  // per BATCH slot: union of grades the plan reads
    std::vector<uint32_t> slot_decl;   // per BATCH slot: grade set declared by the GradedObj
    std::vector<MicroOp> micro;
    std::vector<TermChunk> chunks;
    uint64_t total_terms = 0;
    // Projection of the root (gaast_plan_create_projected): the root components the plan stores.  `projected` is set
    // only when some grade is partly selected; a grade with every component selected is dense (empty bitmap).
    bool projected = false;
    std::vector<std::vector<uint64_t>> root_present;  // per root grade, ascending: bitmap of stored components (empty = all)
    std::vector<int32_t> root_row;      // per root column: its row in its grade's array (rank among the stored), -1 = not stored
    std::vector<int32_t> root_sum_col;  // per root column: its batch-sum column (rank among all stored components), -1
    uint32_t stored_cols = 0;           // stored root components: the width of the batch-sum vector

    uint32_t col_of(uint32_t buf, uint32_t grade) const;  // first column of `grade` inside `buf`
    int stream_of(uint32_t slot, uint32_t grade) const;
    uint32_t stored_rows(size_t stream) const;  // rows of a stream's array: C(n,k), or the projected count for the root
    // Throws gaast::Error on malformed descriptions.  `root_present` (one bitmap pointer per root grade, null = the
    // whole grade) projects the root onto the components it selects.
    void build(const gaast_plan_desc& d, const uint64_t* const* root_present = nullptr);
};

}  // namespace gaast
