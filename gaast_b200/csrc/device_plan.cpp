// Validation of a flat plan description and derivation of everything the
// engines need from it.  Nothing here trusts the caller: this is the FFI
// boundary a foreign host (gaast's Rust) talks to.
#include "device_plan.hpp"

#include <algorithm>
#include <cstring>

namespace gaast {

static uint32_t cols_of(const std::vector<uint32_t>& gdim, uint32_t mask) {
    uint32_t c = 0;
    for (size_t k = 0; k < gdim.size(); ++k)
        if (mask >> k & 1) c += gdim[k];
    return c;
}

uint32_t DevicePlanHost::col_of(uint32_t buf, uint32_t grade) const {
    uint32_t c = buf_col[buf];
    for (uint32_t k = 0; k < grade; ++k)
        if (buffer_masks[buf] >> k & 1) c += gdim[k];
    return c;
}

int DevicePlanHost::stream_of(uint32_t slot, uint32_t grade) const {
    for (size_t i = 0; i < streams.size(); ++i)
        if (streams[i].slot == slot && streams[i].grade == grade) return int(i);
    return -1;
}

uint32_t DevicePlanHost::stored_rows(size_t stream) const {
    const Stream& st = streams[stream];
    if (st.slot != 0xFFFFFFFFu || root_present[stream - n_in_streams].empty()) return st.rows;
    uint32_t c = 0;
    for (uint64_t w : root_present[stream - n_in_streams]) c += uint32_t(__builtin_popcountll(w));
    return c;
}

void DevicePlanHost::build(const gaast_plan_desc& d, const uint64_t* const* present) {
    auto bad = [](const std::string& m) { throw Error(GAAST_ERR_INVALID, "plan: " + m); };
    if (d.n > GAAST_MAX_DIM) bad("dimension above GAAST_MAX_DIM");
    if (d.n_buffers == 0 || !d.buffer_masks) bad("no buffers (buffer 0 must be the root)");
    if ((d.n_inputs && !d.inputs) || (d.n_ops && !d.ops) || (d.n_terms && !d.terms) ||
        (d.n_const_values && !d.const_values))
        bad("null array with non-zero count");
    n = d.n;
    n_slots = d.n_slots;
    if (n_slots > 64) bad("more than 64 batch slots");
    const uint32_t full = (2u << n) - 1;
    gdim.resize(n + 1);
    for (uint32_t k = 0; k <= n; ++k) gdim[k] = uint32_t(binomial(n, k));
    buffer_masks.assign(d.buffer_masks, d.buffer_masks + d.n_buffers);
    inputs.assign(d.inputs, d.inputs + d.n_inputs);
    const_values.assign(d.const_values, d.const_values + d.n_const_values);
    ops.assign(d.ops, d.ops + d.n_ops);
    terms.assign(d.terms, d.terms + d.n_terms);

    buf_col.resize(d.n_buffers);
    buf_cols.resize(d.n_buffers);
    total_cols = 0;
    for (uint32_t b = 0; b < d.n_buffers; ++b) {
        if (buffer_masks[b] & ~full) bad("buffer grade mask has grades above n");
        buf_col[b] = total_cols;
        buf_cols[b] = cols_of(gdim, buffer_masks[b]);
        total_cols += buf_cols[b];
    }
    if (total_cols == 0) total_cols = 1;  // keep shared-memory sizing well defined

    slot_masks.assign(n_slots, 0);
    slot_decl.assign(n_slots, 0);
    std::vector<char> slot_seen(n_slots, 0);
    for (auto& in : inputs) {
        if (in.grade_mask & ~full) {
            // A GradedObj may declare grades above n (e.g. a literal built for a
            // larger space); the reference clips them at reification (expr.rs:17).
            in.grade_mask &= full;
        }
        if (in.kind == GAAST_INPUT_BATCH) {
            if (in.slot >= n_slots) bad("input slot out of range");
            if (slot_seen[in.slot] && slot_decl[in.slot] != in.grade_mask)
                bad("one batch slot is declared with two different grade sets");
            slot_seen[in.slot] = 1;
            slot_decl[in.slot] = in.grade_mask;
        } else if (in.kind == GAAST_INPUT_CONST) {
            if (uint64_t(in.const_offset) + cols_of(gdim, in.grade_mask) > const_values.size())
                bad("constant input overruns const_values");
        } else {
            bad("unknown input kind");
        }
    }

    // ---- ops -> micro-ops -------------------------------------------------------
    total_terms = 0;
    for (const gaast_op& op : ops) {
        if (op.dst >= d.n_buffers) bad("op destination buffer out of range");
        switch (op.kind) {
            case GAAST_OP_ADD_INPUT: {
                if (op.a >= inputs.size()) bad("ADD_INPUT: input index out of range");
                const gaast_input_desc& in = inputs[op.a];
                if (op.mask & ~in.grade_mask) bad("ADD_INPUT: grade not held by the input");
                if (op.mask & ~buffer_masks[op.dst]) bad("ADD_INPUT: grade not held by the destination");
                if (in.kind == GAAST_INPUT_BATCH) slot_masks[in.slot] |= op.mask;
                break;
            }
            case GAAST_OP_MUL_TERMS: {
                if (op.a >= d.n_buffers || op.b >= d.n_buffers) bad("MUL_TERMS: operand buffer out of range");
                if (uint64_t(op.term_begin) + op.term_count > terms.size()) bad("MUL_TERMS: term range out of bounds");
                if (op.a == op.dst || op.b == op.dst) bad("MUL_TERMS: destination aliases an operand");
                for (uint32_t t = op.term_begin; t < op.term_begin + op.term_count; ++t) {
                    const gaast_term& tm = terms[t];
                    if (tm.out >= buf_cols[op.dst] || tm.a >= buf_cols[op.a] || tm.b >= buf_cols[op.b])
                        bad("MUL_TERMS: component slot out of range");
                }
                total_terms += op.term_count;
                break;
            }
            case GAAST_OP_NEG_GRADES:
                if (op.mask & ~buffer_masks[op.dst]) bad("NEG_GRADES: grade not held by the destination");
                break;
            case GAAST_OP_SCALAR_INV:
            case GAAST_OP_SCALAR_SQRT:
                if (!(buffer_masks[op.dst] & 1)) bad("scalar op on a buffer without grade 0");
                break;
            case GAAST_OP_EXP:
            case GAAST_OP_LOG: {
                if (op.a >= d.n_buffers || op.a == op.dst) bad("EXP / LOG: source buffer out of range or aliasing the destination");
                if (!op.mask || (op.mask & (op.mask - 1)) || (op.mask & ~full)) bad("EXP / LOG: `mask` must name one grade");
                const uint32_t k = uint32_t(__builtin_ctz(op.mask));
                if (k == 0) bad("EXP / LOG: the k-vector part cannot be grade 0");
                if (!(buffer_masks[op.a] >> k & 1) || !(buffer_masks[op.dst] >> k & 1))
                    bad("EXP / LOG: grade k must be held by the source and by the destination");
                if (op.kind == GAAST_OP_LOG && !(buffer_masks[op.a] & 1)) bad("LOG: the source lacks grade 0");
                if (uint64_t(op.term_begin) + op.term_count > terms.size() || op.term_count != gdim[k])
                    bad("EXP / LOG: needs one term (blade square) per component of grade k");
                const uint32_t first = col_of(op.a, k) - buf_col[op.a];
                for (uint32_t i = 0; i < op.term_count; ++i) {
                    const gaast_term& tm = terms[op.term_begin + i];
                    if (tm.a != first + i || tm.b != first + i) bad("EXP / LOG: term i must address component i of grade k");
                }
                total_terms += 2 * uint64_t(op.term_count);  // the square and the scaling, per component
                break;
            }
            default: bad("unknown op kind");
        }
    }

    // streams: every (slot, grade) the plan reads, then the root's grades
    streams.clear();
    for (uint32_t s = 0; s < n_slots; ++s)
        for (uint32_t k = 0; k <= n; ++k)
            if (slot_masks[s] >> k & 1) streams.push_back(Stream{s, k, gdim[k]});
    n_in_streams = uint32_t(streams.size());
    for (uint32_t k = 0; k <= n; ++k)
        if (buffer_masks[0] >> k & 1) streams.push_back(Stream{0xFFFFFFFFu, k, gdim[k]});
    if (streams.size() > size_t(kMaxStreams)) bad("too many (input, grade) arrays for one kernel");

    // projection: normalised as gaast_batch_alloc_sparse normalises a batch's bitmaps (bits past C(n,k) ignored, a
    // grade with every bit set is dense), so that a batch allocated from the same bitmaps matches the plan
    projected = false;
    root_present.assign(streams.size() - n_in_streams, {});
    root_row.assign(buf_cols[0], -1);
    root_sum_col.assign(buf_cols[0], -1);
    stored_cols = 0;
    for (size_t i = n_in_streams, col = 0; i < streams.size(); ++i) {
        const uint32_t full = streams[i].rows;
        std::vector<uint64_t>& bits = root_present[i - n_in_streams];
        if (present && present[i - n_in_streams]) {
            bits.assign(present[i - n_in_streams], present[i - n_in_streams] + (full + 63) / 64);
            if (full % 64) bits.back() &= (~0ull) >> (64 - full % 64);
            uint32_t cnt = 0;
            for (uint64_t w : bits) cnt += uint32_t(__builtin_popcountll(w));
            if (cnt == full) bits.clear();
            else projected = true;
        }
        for (uint32_t c = 0, row = 0; c < full; ++c, ++col)
            if (bits.empty() || (bits[c / 64] >> (c % 64) & 1)) {
                root_row[col] = int32_t(row++);
                root_sum_col[col] = int32_t(stored_cols++);
            }
    }
    if (present && stored_cols == 0) throw Error(GAAST_ERR_SHAPE, "plan: the projection stores no root component");

    micro.clear();
    chunks.clear();
    auto push = [&](uint32_t kind, uint32_t dst, uint32_t a, uint32_t b, uint32_t count, uint32_t chunk0 = 0) {
        micro.push_back(MicroOp{kind, dst, a, b, count, chunk0, 0, 0});
    };
    for (const gaast_op& op : ops) {
        switch (op.kind) {
            case GAAST_OP_ADD_INPUT: {
                const gaast_input_desc& in = inputs[op.a];
                uint32_t coff = in.const_offset;
                for (uint32_t k = 0; k <= n; ++k) {
                    if (!(in.grade_mask >> k & 1)) continue;
                    if (op.mask >> k & 1) {
                        if (in.kind == GAAST_INPUT_BATCH)
                            push(MK_LOAD_ADD, col_of(op.dst, k), uint32_t(stream_of(in.slot, k)), 0, gdim[k]);
                        else
                            push(MK_CONST_ADD, col_of(op.dst, k), coff, 0, gdim[k]);
                    }
                    coff += gdim[k];
                }
                break;
            }
            case GAAST_OP_MUL_TERMS: {
                // stable sort by output slot keeps, per output, the reference's term order
                std::vector<gaast_term> t(terms.begin() + op.term_begin, terms.begin() + op.term_begin + op.term_count);
                std::stable_sort(t.begin(), t.end(), [](const gaast_term& x, const gaast_term& y) { return x.out < y.out; });
                const uint32_t chunk0 = uint32_t(chunks.size());
                for (size_t pos = 0; pos < t.size();) {
                    TermChunk c;
                    std::memset(&c, 0, sizeof c);
                    const size_t cnt = std::min<size_t>(kChunkTerms, t.size() - pos);
                    c.n_terms = uint32_t(cnt);
                    uint32_t runs = 0;
                    for (size_t i = 0; i < cnt; ++i) {
                        c.terms[i] = t[pos + i];
                        if (i == 0 || t[pos + i].out != t[pos + i - 1].out) c.run_start[runs++] = uint16_t(i);
                    }
                    c.run_start[runs] = uint16_t(cnt);
                    c.n_runs = runs;
                    chunks.push_back(c);
                    pos += cnt;
                }
                push(MK_MUL, buf_col[op.dst], buf_col[op.a], buf_col[op.b], uint32_t(chunks.size()) - chunk0, chunk0);
                break;
            }
            case GAAST_OP_NEG_GRADES:
                for (uint32_t k = 0; k <= n; ++k)
                    if (op.mask >> k & 1) push(MK_NEG, col_of(op.dst, k), 0, 0, gdim[k]);
                break;
            case GAAST_OP_SCALAR_INV: push(MK_INV, col_of(op.dst, 0), 0, 0, 1); break;
            case GAAST_OP_SCALAR_SQRT: push(MK_SQRT, col_of(op.dst, 0), 0, 0, 1); break;
            case GAAST_OP_EXP:
            case GAAST_OP_LOG: {
                const uint32_t k = uint32_t(__builtin_ctz(op.mask));
                const uint32_t coff = uint32_t(const_values.size());  // the blade squares join the plan's constants
                for (uint32_t i = 0; i < op.term_count; ++i) const_values.push_back(terms[op.term_begin + i].coeff);
                push(op.kind == GAAST_OP_EXP ? MK_EXP : MK_LOG, col_of(op.dst, k), col_of(op.a, k),
                     op.kind == GAAST_OP_LOG ? col_of(op.a, 0) : (buffer_masks[op.dst] & 1) ? col_of(op.dst, 0) : 0xFFFFFFFFu,
                     gdim[k], coff);  // (EXP into an accumulator without grade 0 -- a projection pruned it: no scalar part)
                break;
            }
        }
    }
    // one store per run of consecutive stored components: workspace column, stream, first stored row, count, and
    // (pad0) the run's first batch-sum column
    for (uint32_t i = n_in_streams; i < streams.size(); ++i) {
        const uint32_t c0 = col_of(0, streams[i].grade) - buf_col[0];
        for (uint32_t c = c0; c < c0 + streams[i].rows;) {
            if (root_row[c] < 0) { ++c; continue; }
            uint32_t e = c;
            while (e < c0 + streams[i].rows && root_row[e] >= 0) ++e;
            push(MK_STORE, buf_col[0] + c, i, uint32_t(root_row[c]), e - c);
            micro.back().pad0 = uint32_t(root_sum_col[c]);
            c = e;
        }
    }
}

}  // namespace gaast
