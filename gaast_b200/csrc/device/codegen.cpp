// Specialised engine, step 1: plan -> straight-line CUDA source.
//
// The plan's ops are executed SYMBOLICALLY, one value node per buffer
// component, in the reference's execution order (eval.rs:35-115).  What comes
// out is a DAG whose leaves are input loads / literals and whose inner nodes
// are the reference's arithmetic: `acc + l*r*coeff` links (eval.rs:82), input
// additions (graded.rs:74), 1/x and sqrt (eval.rs:107-108).  Sign flips
// (Negation / Reverse / GradeInvolution, graded.rs:61-65) are folded into the
// references between nodes: negation is exact in IEEE arithmetic, so this
// changes no result bit.  Dead components are dropped.  The DAG is then printed
// as one kernel in which every index is a literal and every value a register:
//
//  * one thread evaluates one batch element (two with 128-bit accesses when the
//    live state is small); all sums / reverses / involutions / projections are
//    fused, intermediates never touch HBM;
//  * values that depend only on broadcast operands and literals are hoisted into
//    a one-thread prologue kernel (they are the same for every element);
//  * per product, the emission order is chosen from the register budget:
//      TABLE   reference order (left operand reused, one accumulator per output),
//      GATHER  one output chain at a time, operands produced on demand
//              (keeps a wide product's outputs out of the register file),
//      BLOCKED dense products: XOR-coset tiles of the Cayley table so that a
//              tile touches 2^h left, 2^h right and 2^h output components.
//    TABLE and GATHER keep the reference's per-component summation order.
//
// GAAST_ARITH_STRICT prints `(l*r)*coeff` then `+` with round-to-nearest
// intrinsics and never simplifies: bit-identical to eval.rs.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <map>
#include <set>
#include <sstream>

#include "../runtime.hpp"

namespace gaast {

namespace {

const char kEvalArgsText[] =
#include "../eval_args_text.inc"
    ;

enum NodeKind : uint8_t { N_ZERO, N_CONST, N_LOAD, N_ACC, N_ADD, N_INV, N_SQRT, N_EXPC, N_EXPS, N_LOGF };
// N_EXPC / N_EXPS: the two factors of exp(B) as functions of q = <B B>_0 (a);  N_LOGF: the factor of log(a0 + B) as a
// function of a0 (a) and q (b).  GAAST_OP_EXP / GAAST_OP_LOG: this library's definition (eval.rs:112-113 is todo!()).
inline bool is_unary(NodeKind k) { return k == N_INV || k == N_SQRT || k == N_EXPC || k == N_EXPS; }
inline bool is_binary(NodeKind k) { return k == N_ADD || k == N_LOGF; }

struct Ref {
    int id = 0;
    bool neg = false;
};

struct Node {
    NodeKind k = N_ZERO;
    Ref a, b, c;        // ACC: prev, left, right.  ADD: a + b.  INV/SQRT: a
    double cval = 0.0;  // CONST value / ACC coefficient
    int stream = -1;    // LOAD
    uint32_t row = 0;   // LOAD
    int op = -1;        // ACC: index of the MUL_TERMS op it belongs to
    uint32_t out_slot = 0, l_slot = 0, r_slot = 0;  // ACC: the term's slots in its op's buffers
    bool uniform = false;
    bool reload = false;  // LOAD: parked in the thread's shared-memory column, re-read at every use
    int smem_row = -1;    // reload: its row in the per-block staging area
    bool pinned = false;  // LOAD: must stay in a register (statically indexed operand of a rolled product)
    bool live = false;
    int export_idx = -1;  // uniform boundary node: index in EvalArgs::uniform
};

enum Policy { P_TABLE, P_GATHER, P_BLOCKED, P_DENSE };

std::string lit(double v) {
    char buf[64];
    std::snprintf(buf, sizeof buf, "%.17g", v);
    std::string s = buf;
    if (s.find_first_of(".eEn") == std::string::npos) s += ".0";
    return s;
}

struct Gen {
    const DevicePlanHost& h;
    const CodegenOptions& opt;
    const bool strict;
    std::vector<Node> nodes;
    std::vector<std::vector<Ref>> buf;            // [buffer][slot]
    std::map<std::pair<int, uint32_t>, int> loads;  // (stream, row) -> node
    std::vector<std::vector<int>> op_accs;        // per plan op: its ACC nodes in table order
    std::vector<Policy> op_policy;
    std::vector<std::vector<uint32_t>> slot_blade;  // per buffer: blade bitmask of every slot
    int ept = 1;

    // Scalar type of the generated arithmetic: "double", or "float" for the f32 variant.  Every
    // emitted declaration goes through it, so the f64 text is unchanged by the f32 support.
    const bool f32;
    const std::string S;
    const size_t esize;

    Gen(const DevicePlanHost& hh, const CodegenOptions& o)
        : h(hh), opt(o), strict(o.arith == GAAST_ARITH_STRICT), f32(o.f32), S(o.f32 ? "float" : "double"), esize(o.f32 ? 4 : 8) {}

    // A projected plan stores root column `col` only when root_row[col] >= 0.  With `prune`, root liveness starts from
    // those columns alone (set after the lowering passes, which match patterns on the whole root buffer).
    bool prune = false;
    bool stored(size_t col) const { return h.root_row[col] >= 0; }

    int add(const Node& n) {
        nodes.push_back(n);
        return int(nodes.size()) - 1;
    }
    bool is_zero(Ref r) const { return nodes[r.id].k == N_ZERO; }

    bool slot_broadcast(uint32_t slot) const { return (opt.broadcast_slots >> slot) & 1; }

    Ref load(int stream, uint32_t row) {
        // sparse per-grade storage: a component the bound batch does not store is the constant zero (and every term
        // that reads it is dropped below); a stored one is addressed by its rank among the stored rows
        if (size_t(stream) < opt.sparse.size() && !opt.sparse[size_t(stream)].empty()) {
            const auto& bits = opt.sparse[size_t(stream)];
            if (!(bits[row / 64] >> (row % 64) & 1)) return Ref{0, false};
            uint32_t rank = 0;
            for (uint32_t w = 0; w < row / 64; ++w) rank += uint32_t(__builtin_popcountll(bits[w]));
            rank += uint32_t(__builtin_popcountll(bits[row / 64] & ((1ull << (row % 64)) - 1)));
            row = rank;
        }
        auto key = std::make_pair(stream, row);
        auto it = loads.find(key);
        if (it != loads.end()) return Ref{it->second, false};
        Node n;
        n.k = N_LOAD;
        n.stream = stream;
        n.row = row;
        n.uniform = slot_broadcast(h.streams[stream].slot);
        const int id = add(n);
        loads.emplace(key, id);
        return Ref{id, false};
    }
    Ref constant(double v) {
        Node n;
        n.k = N_CONST;
        n.cval = v;
        n.uniform = true;
        return Ref{add(n), false};
    }
    Ref make_add(Ref a, Ref b) {
        if (!strict) {
            if (is_zero(a)) return b;
            if (is_zero(b)) return a;
        }
        Node n;
        n.k = N_ADD;
        n.a = a;
        n.b = b;
        n.uniform = nodes[a.id].uniform && nodes[b.id].uniform;
        return Ref{add(n), false};
    }
    Ref make_acc(Ref prev, Ref l, Ref r, double coeff, int op) {
        if (!strict && (is_zero(l) || is_zero(r) || coeff == 0.0)) return prev;
        Node n;
        n.k = N_ACC;
        n.a = prev;
        n.b = l;
        n.c = r;
        n.cval = coeff;
        n.op = op;
        n.uniform = nodes[prev.id].uniform && nodes[l.id].uniform && nodes[r.id].uniform;
        const int id = add(n);
        op_accs[op].push_back(id);
        return Ref{id, false};
    }
    Ref make_unary(NodeKind k, Ref a) {
        Node n;
        n.k = k;
        n.a = a;
        n.uniform = nodes[a.id].uniform;
        return Ref{add(n), false};
    }

    // ---- symbolic execution of the plan (eval.rs:35-115) -------------------------
    void build() {
        Node z;
        z.k = N_ZERO;
        z.uniform = true;
        add(z);  // node 0 == +0.0, the init_null_mv content (eval.rs:27-30)
        buf.resize(h.buffer_masks.size());
        for (size_t b = 0; b < buf.size(); ++b) buf[b].assign(h.buf_cols[b], Ref{0, false});
        op_accs.resize(h.ops.size());
        for (size_t oi = 0; oi < h.ops.size(); ++oi) {
            const gaast_op& op = h.ops[oi];
            switch (op.kind) {
                case GAAST_OP_ADD_INPUT: {
                    const gaast_input_desc& in = h.inputs[op.a];
                    uint32_t coff = in.const_offset;
                    for (uint32_t k = 0; k <= h.n; ++k) {
                        if (!(in.grade_mask >> k & 1)) continue;
                        if (op.mask >> k & 1) {
                            const uint32_t col0 = h.col_of(op.dst, k) - h.buf_col[op.dst];
                            for (uint32_t r = 0; r < h.gdim[k]; ++r) {
                                Ref src = in.kind == GAAST_INPUT_BATCH ? load(h.stream_of(in.slot, k), r)
                                                                       : constant(h.const_values[coff + r]);
                                Ref& d = buf[op.dst][col0 + r];
                                d = make_add(d, src);
                            }
                        }
                        coff += h.gdim[k];
                    }
                    break;
                }
                case GAAST_OP_MUL_TERMS:
                    for (uint32_t t = op.term_begin; t < op.term_begin + op.term_count; ++t) {
                        const gaast_term& tm = h.terms[t];
                        Ref& d = buf[op.dst][tm.out];
                        const size_t before = nodes.size();
                        d = make_acc(d, buf[op.a][tm.a], buf[op.b][tm.b], tm.coeff, int(oi));
                        if (nodes.size() != before) {
                            nodes.back().out_slot = tm.out;
                            nodes.back().l_slot = tm.a;
                            nodes.back().r_slot = tm.b;
                        }
                    }
                    break;
                case GAAST_OP_NEG_GRADES:
                    for (uint32_t k = 0; k <= h.n; ++k)
                        if (op.mask >> k & 1) {
                            const uint32_t col0 = h.col_of(op.dst, k) - h.buf_col[op.dst];
                            for (uint32_t r = 0; r < h.gdim[k]; ++r) buf[op.dst][col0 + r].neg ^= true;
                        }
                    break;
                case GAAST_OP_SCALAR_INV:
                case GAAST_OP_SCALAR_SQRT: {
                    const uint32_t col0 = h.col_of(op.dst, 0) - h.buf_col[op.dst];
                    Ref& d = buf[op.dst][col0];
                    d = make_unary(op.kind == GAAST_OP_SCALAR_INV ? N_INV : N_SQRT, d);
                    break;
                }
                case GAAST_OP_EXP:
                case GAAST_OP_LOG: {
                    const uint32_t k = uint32_t(__builtin_ctz(op.mask));
                    const uint32_t src0 = h.col_of(op.a, k) - h.buf_col[op.a], dst0 = h.col_of(op.dst, k) - h.buf_col[op.dst];
                    Ref q{0, false};  // <B B>_0, in component order
                    for (uint32_t i = 0; i < op.term_count; ++i)
                        q = make_acc(q, buf[op.a][src0 + i], buf[op.a][src0 + i], h.terms[op.term_begin + i].coeff, int(oi));
                    if (strict && is_zero(q)) q = make_add(q, Ref{0, false});
                    Ref f;
                    if (op.kind == GAAST_OP_EXP) {
                        if (h.buffer_masks[op.dst] & 1) {
                            Ref& d0 = buf[op.dst][h.col_of(op.dst, 0) - h.buf_col[op.dst]];
                            d0 = make_add(d0, make_unary(N_EXPC, q));
                        }
                        f = make_unary(N_EXPS, q);
                    } else {
                        Node nf;
                        nf.k = N_LOGF;
                        nf.a = buf[op.a][h.col_of(op.a, 0) - h.buf_col[op.a]];
                        nf.b = q;
                        nf.uniform = nodes[nf.a.id].uniform && nodes[q.id].uniform;
                        f = Ref{add(nf), false};
                    }
                    const Ref one = constant(1.0);
                    (void)one;
                    for (uint32_t i = 0; i < op.term_count; ++i) {
                        Ref& d = buf[op.dst][dst0 + i];
                        const size_t before = nodes.size();
                        d = make_acc(d, f, buf[op.a][src0 + i], 1.0, int(oi));
                        if (nodes.size() != before) {
                            nodes.back().out_slot = dst0 + i;
                            nodes.back().l_slot = 0;
                            nodes.back().r_slot = src0 + i;
                        }
                    }
                    break;
                }
            }
        }
    }

    // ---- shared-operand lowering: the expression as a linear map of its batch inputs ----------
    // When every operand a batch value meets is shared by the whole batch (a fixed rotor in
    // R X ~R, a fixed B in B C, literals), each root component is  sum_j M_j x_j + m  with
    // coefficients M_j, m that depend on the shared operands only.  The coefficients are built
    // as uniform nodes -- the one-thread prologue kernel evaluates them once per launch -- and
    // the per-element kernel shrinks to one FMA per (root component, batch component) pair:
    // cfg2 goes from 160 to 25 FMAs per element.  Summation order differs from the reference
    // (results stay within the 1e-12 bar); never applied in strict arithmetic.
    static constexpr int kConstKey = -1;
    using LinMap = std::map<int, Ref>;  // batch load node (or kConstKey) -> uniform coefficient

    Ref flip(Ref r, bool neg) const { return Ref{r.id, bool(r.neg ^ neg)}; }
    bool uniform_only(const LinMap& m) const { return m.empty() || (m.size() == 1 && m.begin()->first == kConstKey); }

    // keys-only analysis: false = not linear in the batch inputs
    bool lin_keys(int id, std::vector<char>& state, std::vector<std::set<int>>& keys) {
        if (state[id]) return state[id] == 1;
        const Node& n = nodes[id];
        std::set<int> k;
        bool ok = true;
        auto uni = [](const std::set<int>& s) { return s.empty() || (s.size() == 1 && *s.begin() == kConstKey); };
        switch (n.k) {
            case N_ZERO: break;
            case N_CONST: k.insert(kConstKey); break;
            case N_LOAD: k.insert(n.uniform ? kConstKey : id); break;
            case N_ADD:
                ok = lin_keys(n.a.id, state, keys) && lin_keys(n.b.id, state, keys);
                if (ok) { k = keys[n.a.id]; k.insert(keys[n.b.id].begin(), keys[n.b.id].end()); }
                break;
            case N_ACC:
                ok = lin_keys(n.a.id, state, keys) && lin_keys(n.b.id, state, keys) && lin_keys(n.c.id, state, keys);
                if (ok) {
                    const bool lu = uni(keys[n.b.id]), ru = uni(keys[n.c.id]);
                    if (!lu && !ru) { ok = false; break; }
                    k = keys[n.a.id];
                    if (!keys[n.b.id].empty() && !keys[n.c.id].empty()) {
                        const std::set<int>& other = lu ? keys[n.c.id] : keys[n.b.id];
                        k.insert(other.begin(), other.end());
                    }
                }
                break;
            case N_INV:
            case N_SQRT:
            case N_EXPC:
            case N_EXPS:
                ok = lin_keys(n.a.id, state, keys) && uni(keys[n.a.id]);
                if (ok) k.insert(kConstKey);
                break;
            case N_LOGF:
                ok = lin_keys(n.a.id, state, keys) && uni(keys[n.a.id]) && lin_keys(n.b.id, state, keys) && uni(keys[n.b.id]);
                if (ok) k.insert(kConstKey);
                break;
        }
        state[id] = ok ? 1 : 2;
        keys[id] = std::move(k);
        return ok;
    }

    Ref umul(Ref u, Ref v, double c, int op) {  // uniform * uniform * c
        if (is_zero(u) || is_zero(v) || c == 0.0) return Ref{0, false};
        if (nodes[u.id].k == N_CONST && nodes[u.id].cval == 1.0 && std::fabs(c) == 1.0) return flip(v, u.neg ^ (c < 0));
        if (nodes[v.id].k == N_CONST && nodes[v.id].cval == 1.0 && std::fabs(c) == 1.0) return flip(u, v.neg ^ (c < 0));
        return make_acc(Ref{0, false}, u, v, c, op);
    }

    const LinMap& lin_build(int id, std::map<int, LinMap>& memo, Ref one, int op) {
        auto it = memo.find(id);
        if (it != memo.end()) return it->second;
        const Node n = nodes[id];  // copy: `nodes` grows below
        LinMap m;
        auto accumulate = [&](LinMap& dst, int key, Ref coef) {
            if (is_zero(coef)) return;
            auto f = dst.find(key);
            if (f == dst.end()) dst.emplace(key, coef);
            else f->second = make_add(f->second, coef);
        };
        switch (n.k) {
            case N_ZERO: break;
            case N_CONST: m.emplace(kConstKey, Ref{id, false}); break;
            case N_LOAD:
                if (n.uniform) m.emplace(kConstKey, Ref{id, false});
                else m.emplace(id, one);
                break;
            case N_ADD:
                for (const auto& kv : LinMap(lin_build(n.a.id, memo, one, op))) accumulate(m, kv.first, flip(kv.second, n.a.neg));
                for (const auto& kv : LinMap(lin_build(n.b.id, memo, one, op))) accumulate(m, kv.first, flip(kv.second, n.b.neg));
                break;
            case N_ACC: {
                for (const auto& kv : LinMap(lin_build(n.a.id, memo, one, op))) accumulate(m, kv.first, flip(kv.second, n.a.neg));
                const LinMap L = lin_build(n.b.id, memo, one, op), R = lin_build(n.c.id, memo, one, op);
                if (L.empty() || R.empty()) break;
                const bool left_uniform = uniform_only(L);
                const LinMap& U = left_uniform ? L : R;
                const LinMap& V = left_uniform ? R : L;
                const Ref u = flip(U.begin()->second, left_uniform ? n.b.neg : n.c.neg);
                const bool vneg = left_uniform ? n.c.neg : n.b.neg;
                for (const auto& kv : V) accumulate(m, kv.first, umul(u, flip(kv.second, vneg), n.cval, op));
                break;
            }
            case N_INV:
            case N_SQRT:
            case N_EXPC:
            case N_EXPS:
            case N_LOGF: m.emplace(kConstKey, Ref{id, false}); break;  // uniform argument(s) (checked by lin_keys)
        }
        return memo.emplace(id, std::move(m)).first->second;
    }

    // ---- factoring a common scalar out of a product -------------------------------------------
    // In  T * (Y s)  where the right operand is a buffer of single-term products with ONE common
    // factor s (the versor inverse V^-1 = ~V * (1 / |V|^2) of cfg5), every term carries s:
    // sum_t T_t (Y_w s) c  ==  s * sum_t T_t Y_w c.  The scaled buffer then never exists -- its
    // registers are freed (12 doubles in cfg5, i.e. 12 fewer parked rows) -- at the price of one
    // multiplication per output.  Exact in real arithmetic, a different rounding sequence:
    // FMA arithmetic only.  Returns the number of products rewritten.
    size_t factor_common_scalars(int pseudo_op) {
        if (strict) return 0;
        std::vector<int> refs(nodes.size(), 0);
        auto count_refs = [&]() {
            std::fill(refs.begin(), refs.end(), 0);
            refs.resize(nodes.size(), 0);
            for (const Node& n : nodes) {
                if (n.k == N_ACC) { ++refs[n.a.id]; ++refs[n.b.id]; ++refs[n.c.id]; }
                else if (is_binary(n.k)) { ++refs[n.a.id]; ++refs[n.b.id]; }
                else if (is_unary(n.k)) ++refs[n.a.id];
            }
            for (Ref r : buf[0]) ++refs[r.id];  // only the root buffer is read after the symbolic run
        };
        size_t rewritten = 0;
        for (size_t oi = 0; oi < h.ops.size(); ++oi) {
            if (h.ops[oi].kind != GAAST_OP_MUL_TERMS || op_accs[oi].size() < 8) continue;
            // candidate common factor: an operand shared by every right operand's defining product
            std::set<int> common;
            bool ok = true, first = true;
            std::map<int, int> uses_of_right;  // right operand node -> how many of this op's terms read it
            std::set<uint32_t> started;
            for (int id : op_accs[oi]) {
                const Node& nd = nodes[id];
                const Node& r = nodes[nd.c.id];
                if (r.k != N_ACC || !is_zero(r.a) || r.uniform) { ok = false; break; }
                std::set<int> here{r.b.id, r.c.id};
                if (first) common = here;
                else {
                    std::set<int> both;
                    for (int x : common) if (here.count(x)) both.insert(x);
                    common = both;
                }
                first = false;
                if (common.empty()) { ok = false; break; }
                ++uses_of_right[nd.c.id];
                if (!started.count(nd.out_slot)) {
                    if (!is_zero(nd.a)) { ok = false; break; }  // accumulators must start from zero
                    started.insert(nd.out_slot);
                }
            }
            if (!ok || common.size() != 1 || uses_of_right.size() < 2) continue;
            const int s = *common.begin();
            count_refs();
            for (const auto& kv : uses_of_right)
                if (refs[kv.first] != kv.second) ok = false;  // the scaled buffer must have no other reader
            if (!ok) continue;
            // rewrite the terms: right operand Y instead of (Y s), coefficient absorbs the inner one
            std::map<uint32_t, int> last;  // out slot -> last link
            for (int id : op_accs[oi]) {
                Node& nd = nodes[id];
                const Node r = nodes[nd.c.id];
                const bool y_is_left = r.c.id == s;
                const Ref y = y_is_left ? r.b : r.c;
                const Ref sr = y_is_left ? r.c : r.b;
                const bool neg = nd.c.neg ^ y.neg ^ sr.neg;
                nd.cval = nd.cval * r.cval * (neg ? -1.0 : 1.0);
                nd.c = Ref{y.id, false};
                nd.uniform = nodes[nd.a.id].uniform && nodes[nd.b.id].uniform && nodes[y.id].uniform;
                last[nd.out_slot] = id;
            }
            // one multiplication by s per output, and every reader of the output sees the product
            std::map<int, int> replace;
            for (const auto& kv : last) {
                const Ref scaled = make_acc(Ref{0, false}, Ref{kv.second, false}, Ref{s, false}, 1.0, pseudo_op);
                replace[kv.second] = scaled.id;
            }
            auto fix = [&](Ref& r, int self) {
                auto it = replace.find(r.id);
                if (it != replace.end() && it->second != self) r.id = it->second;
            };
            for (size_t id = 0; id < nodes.size(); ++id) {
                Node& n = nodes[id];
                if (n.k == N_ACC && n.op == int(oi)) { fix(n.b, int(id)); fix(n.c, int(id)); continue; }  // own chain links stay
                if (n.k == N_ACC || is_binary(n.k) || is_unary(n.k)) {
                    fix(n.a, int(id));
                    if (n.k == N_ACC || is_binary(n.k)) fix(n.b, int(id));
                    if (n.k == N_ACC) fix(n.c, int(id));
                }
            }
            for (auto& b : buf)
                for (Ref& r : b) fix(r, -1);
            ++rewritten;
        }
        return rewritten;
    }

    // Returns the number of root components rewritten (0 = lowering not applicable / not worthwhile).
    size_t lower_linear(int pseudo_op) {
        if (strict) return 0;
        std::vector<char> state(nodes.size(), 0);
        std::vector<std::set<int>> keys(nodes.size());
        size_t entries = 0, batch_keys = 0;
        for (Ref r : buf[0]) {
            if (!lin_keys(r.id, state, keys)) return 0;
            entries += keys[r.id].size();
            for (int k : keys[r.id]) batch_keys += k != kConstKey;
        }
        size_t terms = 0;
        for (const Node& n : nodes) terms += n.live && n.k == N_ACC && !n.uniform;
        if (batch_keys == 0 || entries > 4096 || terms < 2 * entries) return 0;
        const Ref one = constant(1.0);
        std::map<int, LinMap> memo;
        size_t rewritten = 0;
        for (Ref& r : buf[0]) {
            const LinMap m = lin_build(r.id, memo, one, pseudo_op);
            Ref acc{0, false};
            auto c = m.find(kConstKey);
            if (c != m.end()) acc = c->second;
            for (const auto& kv : m) {
                if (kv.first == kConstKey) continue;
                acc = make_acc(acc, kv.second, Ref{kv.first, false}, 1.0, pseudo_op);
            }
            r = flip(acc, r.neg);
            ++rewritten;
        }
        return rewritten;
    }

    // ---- reflection lowering: a vector sandwich  (v X) w  with  w = s v ------------------------
    // For a vector v and ANY multivector X:  v X = X^ v + 2 (v _| X)   (X^ = grade involution, _| = left
    // contraction; from e_i e_j = -e_j e_i + 2 g_ij, valid for every diagonal metric).  With w parallel to v
    // the product v w is a scalar c = sum_i m_i v_i w_i, so
    //        (v X) w  =  c X^  +  2 (v _| X) w.
    // The reference evaluates the left side literally (eval.rs:61-86 twice): for cfg5's versor sandwich
    // V X V^-1 with a grade-1 versor that is 792 + 792 terms through a 232-component intermediate; the right
    // side needs the 12-component contraction (132 terms), its product with w restricted to the root's
    // grades (132 terms), c (12) and one FMA per root component -- the kernel becomes a pure HBM stream.
    // Everything is checked on the plan before rewriting: both products are complete geometric products on
    // the grades they keep, v and w are grade-1 buffers, every w_i is the SAME scalar node times v_i, the
    // intermediate has no other reader, and the metric is recovered (and cross-checked) from the first
    // product's own coefficients.  A different rounding sequence (still within the 1e-12 bar, checked against
    // the oracle and the strict engine): FMA arithmetic only.  variant bit 16 switches the pass off.
    size_t lower_reflections(int pseudo_op) {
        if (strict) return 0;
        if (slot_blade.empty()) compute_blades();
        size_t rewritten = 0;
        const size_t n_ops = h.ops.size();
        auto grade_of = [](uint32_t blade) { return uint32_t(__builtin_popcount(blade)); };
        for (size_t oR = 0; oR < n_ops; ++oR) {
            const gaast_op& R = h.ops[oR];
            if (R.kind != GAAST_OP_MUL_TERMS) continue;
            const uint32_t D = R.dst, T = R.a, Wb = R.b;
            if (T == 0 || T == D || Wb == T || h.buffer_masks[Wb] != 2u) continue;
            // the one op that writes T: a product V * X with a grade-1 left operand, before R
            int oK = -1;
            bool ok = true;
            for (size_t i = 0; i < n_ops && ok; ++i) {
                const gaast_op& o = h.ops[i];
                if (o.dst == T) {
                    if (oK >= 0 || o.kind != GAAST_OP_MUL_TERMS || i > oR) ok = false;
                    oK = int(i);
                }
                if (o.kind == GAAST_OP_MUL_TERMS && i != oR && (o.a == T || o.b == T)) ok = false;  // T has another reader
            }
            if (!ok || oK < 0) continue;
            const gaast_op& K = h.ops[size_t(oK)];
            const uint32_t Vb = K.a, Xb = K.b;
            if (h.buffer_masks[Vb] != 2u || Vb == T || Xb == T || Xb == D || Vb == D) continue;
            for (size_t i = size_t(oK) + 1; i < n_ops && ok; ++i)  // operands must keep the value the products saw
                if (h.ops[i].dst == Vb || h.ops[i].dst == Xb || (i > oR && h.ops[i].dst == Wb)) ok = false;
            for (size_t i = size_t(oK) + 1; i < oR && ok; ++i)
                if (h.ops[i].dst == T) ok = false;
            if (!ok) continue;
            const uint32_t n = h.n;
            const auto& bV = slot_blade[Vb];
            const auto& bX = slot_blade[Xb];
            const auto& bT = slot_blade[T];
            const auto& bD = slot_blade[D];
            const auto& bW = slot_blade[Wb];
            if (bV.size() != n || bW.size() != n) continue;
            // w_i = (one common scalar node) * v_i, with one common sign and coefficient
            int s_id = -1;
            bool sign0 = false;
            double coef0 = 0.0;
            for (uint32_t i = 0; i < n && ok; ++i) {
                const Ref wr = buf[Wb][i], vr = buf[Vb][i];
                const Node& w = nodes[wr.id];
                if (w.k != N_ACC || !is_zero(w.a) || w.uniform) { ok = false; break; }
                const bool v_left = w.b.id == vr.id, v_right = w.c.id == vr.id;
                if (!v_left && !v_right) { ok = false; break; }
                const Ref other = v_left ? w.c : w.b;
                if (other.id == vr.id) { ok = false; break; }
                const bool sign = wr.neg ^ w.b.neg ^ w.c.neg ^ vr.neg ^ (w.cval < 0);
                if (i == 0) { s_id = other.id; sign0 = sign; coef0 = std::fabs(w.cval); }
                else if (other.id != s_id || sign != sign0 || std::fabs(w.cval) != coef0) ok = false;
            }
            if (!ok || s_id < 0) continue;
            // both products complete on the grades they keep (a geometric product, not an outer / inner one)
            auto complete = [&](const gaast_op& op, const std::vector<uint32_t>& bl, const std::vector<uint32_t>& br,
                                const std::vector<uint32_t>& bo, uint32_t out_mask) {
                size_t expect = 0;
                for (uint32_t a : bl)
                    for (uint32_t b : br) expect += (out_mask >> grade_of(a ^ b)) & 1;
                if (expect != op.term_count) return false;
                for (uint32_t t = op.term_begin; t < op.term_begin + op.term_count; ++t) {
                    const gaast_term& tm = h.terms[t];
                    if (tm.a >= bl.size() || tm.b >= br.size() || tm.out >= bo.size()) return false;
                    if ((bl[tm.a] ^ br[tm.b]) != bo[tm.out]) return false;
                }
                return true;
            };
            if (!complete(K, bV, bX, bT, h.buffer_masks[T]) || !complete(R, bT, bW, bD, h.buffer_masks[D])) continue;
            // metric from the first product's coefficients:  e_i B = (-1)^(bits of B below i) m_i (B \ i)  for i in B
            std::vector<double> metric(n, 0.0);
            std::vector<char> have(n, 0);
            for (uint32_t t = K.term_begin; t < K.term_begin + K.term_count && ok; ++t) {
                const gaast_term& tm = h.terms[t];
                const uint32_t a = bV[tm.a], b = bX[tm.b];
                const uint32_t i = uint32_t(__builtin_ctz(a));
                if (!(b & a)) continue;
                const double m = tm.coeff * ((__builtin_popcount(b & (a - 1)) & 1) ? -1.0 : 1.0);
                if (m == 0.0) ok = false;
                if (have[i] && metric[i] != m) ok = false;
                metric[i] = m;
                have[i] = 1;
            }
            for (uint32_t i = 0; i < n; ++i) ok = ok && have[bV[i] ? uint32_t(__builtin_ctz(bV[i])) : 0];
            if (!ok) continue;
            // R's chain per output: what it was started from (the buffer's content before R) and its last link --
            // the value every later reader of the buffer sees (sign flips live in the references to it)
            std::vector<Ref> prior(bD.size(), Ref{0, false});
            std::vector<char> touched(bD.size(), 0);
            for (int id : op_accs[oR]) {
                const Node& nd = nodes[id];
                if (!touched[nd.out_slot]) { prior[nd.out_slot] = nd.a; touched[nd.out_slot] = 1; }
            }
            std::vector<int> last(bD.size(), -1);
            for (int id : op_accs[oR]) last[nodes[id].out_slot] = id;
            if (op_accs[oR].empty()) continue;  // nothing of this product survives (an empty root)
            // ---- build the right-hand side ----
            const size_t first_new = nodes.size();
            Ref c{0, false};  // v . w
            for (uint32_t i = 0; i < n; ++i) {
                const uint32_t e = uint32_t(__builtin_ctz(bV[i]));
                uint32_t wi = 0;
                while (wi < n && bW[wi] != bV[i]) ++wi;
                c = make_acc(c, buf[Vb][i], buf[Wb][wi], metric[e], pseudo_op);
            }
            std::vector<Ref> U(bT.size(), Ref{0, false});  // v _| X: the terms of V * X that lower the grade
            for (uint32_t t = K.term_begin; t < K.term_begin + K.term_count; ++t) {
                const gaast_term& tm = h.terms[t];
                if (grade_of(bT[tm.out]) + 1 != grade_of(bX[tm.b])) continue;
                U[tm.out] = make_acc(U[tm.out], buf[Vb][tm.a], buf[Xb][tm.b], tm.coeff, pseudo_op);
            }
            std::map<uint32_t, uint32_t> x_slot_of_blade;
            for (uint32_t sx = 0; sx < bX.size(); ++sx) x_slot_of_blade[bX[sx]] = sx;
            std::vector<Ref> res(bD.size());
            for (size_t o = 0; o < bD.size(); ++o) {
                if (!touched[o]) continue;
                Ref acc = prior[o];
                auto xs = x_slot_of_blade.find(bD[o]);
                if (xs != x_slot_of_blade.end()) {
                    const Ref x = buf[Xb][xs->second];
                    acc = make_acc(acc, flip(x, grade_of(bD[o]) & 1), c, 1.0, pseudo_op);  // c X^
                }
                res[o] = acc;
            }
            // 2 (v _| X) w: the factor 2 goes into the contraction once per component (exact), so that every term
            // below keeps a +-1 coefficient and stays ONE FMA
            const Ref two = constant(2.0);
            std::vector<char> doubled(U.size(), 0);
            for (uint32_t t = R.term_begin; t < R.term_begin + R.term_count; ++t) {
                const gaast_term& tm = h.terms[t];
                if (!touched[tm.out] || is_zero(U[tm.a])) continue;
                if (!doubled[tm.a]) {
                    U[tm.a] = make_acc(Ref{0, false}, U[tm.a], two, 1.0, pseudo_op);
                    doubled[tm.a] = 1;
                }
                res[tm.out] = make_acc(res[tm.out], U[tm.a], buf[Wb][tm.b], tm.coeff, pseudo_op);
            }
            // every reader of the old chain ends (later ops on the same buffer, the root) now reads the new values
            std::map<int, Ref> replace;
            for (size_t o = 0; o < bD.size(); ++o)
                if (touched[o]) replace[last[o]] = res[o];
            // (the nodes created above, from first_new on, never refer to the old chain ends)
            auto fix = [&](Ref& r) {
                auto it = replace.find(r.id);
                if (it != replace.end()) r = Ref{it->second.id, bool(r.neg ^ it->second.neg)};
            };
            for (size_t id = 0; id < first_new && id < nodes.size(); ++id) {
                Node& nd = nodes[id];
                if (nd.k == N_ACC && nd.op == int(oR)) continue;  // the old chain itself (now dead)
                if (nd.k == N_ACC || is_binary(nd.k) || is_unary(nd.k)) {
                    fix(nd.a);
                    if (nd.k == N_ACC || is_binary(nd.k)) fix(nd.b);
                    if (nd.k == N_ACC) fix(nd.c);
                }
            }
            for (auto& bb : buf)
                for (Ref& r : bb) fix(r);
            ++rewritten;
        }
        return rewritten;
    }

    void mark_live() {
        std::vector<int> stack;
        for (size_t col = 0; col < buf[0].size(); ++col)
            if (!prune || stored(col)) stack.push_back(buf[0][col].id);
        while (!stack.empty()) {
            const int id = stack.back();
            stack.pop_back();
            Node& n = nodes[id];
            if (n.live) continue;
            n.live = true;
            if (n.k == N_ACC) {
                stack.push_back(n.a.id);
                stack.push_back(n.b.id);
                stack.push_back(n.c.id);
            } else if (is_binary(n.k)) {
                stack.push_back(n.a.id);
                stack.push_back(n.b.id);
            } else if (is_unary(n.k)) {
                stack.push_back(n.a.id);
            }
        }
    }

    static bool is_leaf(const Node& n) { return n.k == N_ZERO || n.k == N_CONST || n.k == N_LOAD; }

    // Uniform inner nodes consumed by per-element nodes (or stored) are exported
    // by the prologue kernel.
    int n_export = 0;
    void mark_exports() {
        auto want = [&](Ref r) {
            Node& n = nodes[r.id];
            if (n.uniform && !is_leaf(n) && n.export_idx < 0) n.export_idx = n_export++;
        };
        for (Node& n : nodes) {
            if (!n.live || n.uniform) continue;
            if (n.k == N_ACC) {
                want(n.a);
                want(n.b);
                want(n.c);
            } else if (is_binary(n.k)) {
                want(n.a);
                want(n.b);
            } else if (is_unary(n.k)) {
                want(n.a);
            }
        }
        for (size_t col = 0; col < buf[0].size(); ++col)
            if (stored(col)) want(buf[0][col]);
    }

    void compute_blades() {
        // slot -> blade: grades ascending, inside a grade the masks of that
        // popcount in ascending numeric order (algebra.rs:221-246)
        std::vector<std::vector<uint32_t>> of_grade(h.n + 1);
        for (uint32_t b = 0; b < (1u << h.n); ++b) of_grade[__builtin_popcount(b)].push_back(b);
        if (!slot_blade.empty()) return;
        slot_blade.resize(h.buffer_masks.size());
        for (size_t b = 0; b < h.buffer_masks.size(); ++b)
            for (uint32_t k = 0; k <= h.n; ++k)
                if (h.buffer_masks[b] >> k & 1)
                    slot_blade[b].insert(slot_blade[b].end(), of_grade[k].begin(), of_grade[k].end());
    }

    // ---- emission ------------------------------------------------------------------
    std::ostringstream body;
    std::vector<char> emitted;
    bool in_prologue = false;
    bool in_loop = false;  // emitting the per-element body (not the hoisted shared values)
    int indent = 2;

    std::string var(int id) const { return "v" + std::to_string(id); }
    void line(const std::string& s) { body << std::string(size_t(indent) * 2, ' ') << s << "\n"; }

    // Operand text for a consumer of type `wide` (per-element) or scalar.
    std::string opnd(Ref r, bool wide, bool flip = false, const std::string& name = std::string()) const {
        const Node& n = nodes[r.id];
        const bool neg = r.neg ^ flip;
        std::string s;
        if (n.k == N_ZERO)
            s = "0.0";
        else if (n.k == N_CONST)
            s = lit(n.cval);
        else
            s = name.empty() ? var(r.id) : name;
        const bool scalar = n.uniform;
        if (neg) s = (n.k == N_ZERO || n.k == N_CONST) ? "(-" + s + ")" : (scalar ? "(-" + s + ")" : "d_neg(" + s + ")");
        if (wide && scalar) s = "U(" + s + ")";
        return s;
    }

    void emit_node_line(int id) {
        const Node& n = nodes[id];
        const bool wide = !n.uniform;
        const std::string ty = wide ? "const D " : "const " + S + " ";
        const std::string v = var(id);
        if (!in_prologue && n.uniform && n.export_idx >= 0) {
            // inside the element loop the table pointer is opaque (`uni`), so that the compiler
            // does not hoist a wide table into registers
            line("const " + S + " " + v + " = __ldg(" + (in_loop ? "uni" : f32 ? "reinterpret_cast<const float*>(a.uniform)" : "a.uniform") +
                 " + " + std::to_string(n.export_idx) + ");");
            return;
        }
        switch (n.k) {
            case N_ZERO:
            case N_CONST: return;
            case N_LOAD: {
                const std::string s = std::to_string(n.stream);
                if (n.uniform)
                    line("const " + S + " " + v + " = __ldg(s" + s + " + " + std::to_string(n.row) + " * r" + s + ");");
                else
                    line("const D " + v + " = d_load(s" + s + " + " + std::to_string(n.row) + " * r" + s + " + e);");
                return;
            }
            case N_ADD:
                line(ty + v + " = " + (strict ? "d_adds(" : "d_add(") + opnd(n.a, wide) + ", " + opnd(n.b, wide) + ");");
                return;
            case N_INV: line(ty + v + " = d_inv(" + opnd(n.a, wide) + ");"); return;
            case N_SQRT: line(ty + v + " = d_sqrt(" + opnd(n.a, wide) + ");"); return;
            case N_EXPC: line(ty + v + " = d_expc(" + opnd(n.a, wide) + ");"); return;
            case N_EXPS: line(ty + v + " = d_exps(" + opnd(n.a, wide) + ");"); return;
            case N_LOGF: line(ty + v + " = d_logf(" + opnd(n.a, wide) + ", " + opnd(n.b, wide) + ");"); return;
            case N_ACC: {
                const std::string ln = use_name(n.b), rn = use_name(n.c);
                line(ty + v + " = " +
                     acc_rhs(n, wide, opnd(n.b, wide, acc_flip(n), ln), opnd(n.c, wide, false, rn), opnd(n.a, wide),
                             is_zero(n.a)) + ";");
                return;
            }
        }
    }

    // A RELOAD input row is not kept in a register.  It is parked once per
    // element in the thread's private column of a shared-memory staging area
    // ([row][thread], bank-conflict free, no barrier needed: a thread only reads
    // what it wrote) and every use re-reads it with a volatile LDS into a
    // temporary that dies at once.  (Re-reading global memory through L1 does not
    // work: ptxas merges identical ld.global.nc and keeps the value live.)
    int reload_counter = 0;
    std::string load_addr(const Node& n) const {
        const std::string s = std::to_string(n.stream);
        return "s" + s + " + " + std::to_string(n.row) + " * r" + s + " + e";
    }
    std::string smem_read(const Node& n) const {
        return "xs_ld<" + std::to_string(size_t(n.smem_row) * esize) + " * GAAST_THREADS>(xb)";
    }
    std::string use_name(Ref r) {
        const Node& n = nodes[r.id];
        if (n.k != N_LOAD || n.uniform || !n.reload || in_prologue) return std::string();
        const std::string nm = "x" + std::to_string(r.id) + "_" + std::to_string(reload_counter++);
        line("const D " + nm + " = " + smem_read(n) + ";");
        return nm;
    }
    // All parked rows are fetched at the top of the element body (one burst of
    // independent loads), then stored to shared memory.
    bool pipelined = false;  // parked rows arrive by TMA (persistent block, double buffered), not by LDG + STS
    // Block-uniform tile loop: lanes past the end of the batch shadow the last element.  Their
    // stores are NOT guarded: they write the bits the element's own lane writes, to the same
    // address, and a guard costs a branch per store (measured on cfg5 + sum: 8.07 -> 7.75 ms).
    // Only additive side effects (batch sums) look at `active`.
    bool guard_stores = false;
    bool sum_in_smem = false;   // batch-sum kept as per-thread column sums in shared memory
    bool sum_in_tmem = false;   // ... or in tensor memory (tcgen05.ld / tcgen05.st), the default when it fits
    void emit_staging() {
        if (pipelined) return;
        std::vector<int> ids;
        for (size_t id = 0; id < nodes.size(); ++id)
            if (nodes[id].live && nodes[id].k == N_LOAD && nodes[id].reload && !nodes[id].uniform) ids.push_back(int(id));
        for (size_t i = 0; i < ids.size(); i += 16) {
            const size_t end = std::min(ids.size(), i + 16);
            for (size_t j = i; j < end; ++j)
                line("const D g" + std::to_string(ids[j]) + " = d_load(" + load_addr(nodes[ids[j]]) + ");");
            for (size_t j = i; j < end; ++j)
                line("xs_st<" + std::to_string(size_t(nodes[ids[j]].smem_row) * esize) + " * GAAST_THREADS>(xb, g" +
                     std::to_string(ids[j]) + ");");
        }
    }

    // `acc + l*r*coeff` (eval.rs:82) as an expression over already formatted operands.
    bool acc_flip(const Node& n) const { return !strict && std::fabs(n.cval) == 1.0 && n.cval < 0; }
    std::string acc_rhs(const Node& n, bool wide, const std::string& L, const std::string& R, const std::string& P,
                        bool p_zero) const {
        const double c = n.cval;
        const bool unit = std::fabs(c) == 1.0;
        if (strict) {
            // (l * r) * coeff, then +; multiplying by +-1 is exact
            std::string prod = "d_muls(" + L + ", " + R + ")";
            if (unit) {
                if (c < 0) prod = wide ? "d_neg(" + prod + ")" : "(-" + prod + ")";
            } else {
                prod = "d_muls(" + prod + ", " + (wide ? "U(" + lit(c) + ")" : lit(c)) + ")";
            }
            return "d_adds(" + P + ", " + prod + ")";
        }
        if (unit) return p_zero ? "d_mul(" + L + ", " + R + ")" : "d_fma(" + L + ", " + R + ", " + P + ")";
        const std::string cl = wide ? "U(" + lit(c) + ")" : lit(c);
        const std::string prod = "d_mul(" + L + ", " + R + ")";
        return p_zero ? "d_mul(" + prod + ", " + cl + ")" : "d_fma(" + prod + ", " + cl + ", " + P + ")";
    }

    void emit(int id) {
        if (emitted[id]) return;
        Node& n = nodes[id];
        if (is_leaf(n) || (!in_prologue && n.uniform && n.export_idx >= 0)) {
            emitted[id] = 1;
            if (!(n.k == N_LOAD && n.reload && !n.uniform && !in_prologue)) emit_node_line(id);
            return;
        }
        if (n.k == N_ACC) {
            const Policy pol = (in_prologue || n.uniform) ? P_GATHER : op_policy[n.op];
            if (pol == P_TABLE) {
                if (size_t(n.op) < table_in_progress.size() && table_in_progress[n.op]) {
                    // a term of the op that is being emitted, wanted by an EARLIER term of the same op (two rewriting
                    // passes on one plan leave their new terms in creation order, not in dependency order): emit
                    // this one now -- the values are SSA names, any topological order is the same kernel
                    emit(n.a.id);
                    emit(n.b.id);
                    emit(n.c.id);
                    if (emitted[id]) return;
                    emitted[id] = 1;
                    emit_node_line(id);
                    store_if_root(id);
                    return;
                }
                emit_op_table(n.op);
                return;
            }
            if (pol == P_BLOCKED) {
                emit_op_blocked(n.op);
                return;
            }
            if (pol == P_DENSE) {
                emit_op_dense(n.op);
                return;
            }
            // GATHER: walk the chain back to its first un-emitted link, then forward
            std::vector<int> chain;
            int cur = id;
            while (!emitted[cur] && nodes[cur].k == N_ACC && nodes[cur].op == n.op) {
                chain.push_back(cur);
                cur = nodes[cur].a.id;
            }
            emit(cur);
            for (auto it = chain.rbegin(); it != chain.rend(); ++it) {
                emit(nodes[*it].b.id);
                emit(nodes[*it].c.id);
                emitted[*it] = 1;
                emit_node_line(*it);
            }
            return;
        }
        if (is_binary(n.k)) {
            emit(n.a.id);
            emit(n.b.id);
        } else {
            emit(n.a.id);
        }
        emitted[id] = 1;
        emit_node_line(id);
    }

    std::vector<char> table_in_progress;  // per op: emit_op_table is walking its terms
    void emit_op_table(int op) {
        if (table_in_progress.size() < op_accs.size()) table_in_progress.resize(op_accs.size(), 0);
        table_in_progress[op] = 1;
        for (size_t i = 0; i < op_accs[op].size(); ++i) {
            const int id = op_accs[op][i];
            if (!nodes[id].live || emitted[id]) continue;
            if (nodes[id].uniform && !in_prologue) continue;
            emit(nodes[id].a.id);
            emit(nodes[id].b.id);
            emit(nodes[id].c.id);
            if (emitted[id]) continue;  // (reached through one of its own operands' readers)
            emitted[id] = 1;
            emit_node_line(id);
            store_if_root(id);
        }
        table_in_progress[op] = 0;
    }

    // Root components are stored (and batch-summed) as soon as their value
    // exists, so that finished outputs do not occupy registers.
    struct RootSlot {
        size_t stream;
        uint32_t row, col;  // row: among the grade's stored rows; col: root column
        bool neg;
        uint32_t sum_col;   // batch-sum column (rank among the stored root components)
    };
    std::multimap<int, RootSlot> root_of;  // node id -> root slots holding it
    std::vector<char> root_done;
    void emit_root(const RootSlot& rs, int id) {
        if (in_prologue || root_done[rs.col]) return;
        root_done[rs.col] = 1;
        const std::string val = opnd(Ref{id, rs.neg}, true);
        const std::string guard = guard_stores ? "if (active) " : "";
        if (opt.store_out)
            line("d_store(s" + std::to_string(rs.stream) + " + " + std::to_string(rs.row) + " * r" +
                 std::to_string(rs.stream) + " + e, " + val + ");");
        if (sum_in_smem)
            line(guard + "sums[" + std::to_string(rs.sum_col) + " * GAAST_THREADS + tid] += d_hsum(" + val + ");");
        if (sum_in_tmem) {
            // Accumulators are numbered in emission order (column pair 2k for the k-th finished
            // component).  The first `sum_stash` components only park their value in a second
            // range of tensor-memory columns (one STTM, nothing to wait for); the running sums
            // absorb the whole stash at the end of the tile, 16 components per
            // tcgen05.ld/st.  Components beyond the stash capacity are added one by one.
            const size_t k = sum_order.size();
            sum_order.push_back(rs.sum_col);
            if (k < sum_stash)
                line("tm_put(tb + " + std::to_string(2 * h.stored_cols + 2 * k) + "u, d_hsum(" + val + "));");
            else  // warp-collective: idle lanes add zero
                line("tm_add(tb + " + std::to_string(2 * k) + "u, active ? d_hsum(" + val + ") : 0.0);");
        }
    }
    size_t sum_stash = 0;             // components whose per-tile value is parked in tensor memory
    std::vector<uint32_t> sum_order;  // batch-sum columns in the order their sums are updated
    void store_if_root(int id) {
        if (in_prologue) return;
        auto range = root_of.equal_range(id);
        for (auto it = range.first; it != range.second; ++it) emit_root(it->second, id);
    }

    // Dense products: tiles of the Cayley table indexed by the high blade bits
    // of (output, left).  A tile's outputs form one XOR coset, so it touches at
    // most 2^h outputs, 2^h left and 2^h right components.  The coset's
    // accumulators stay in registers across the tiles of its row; input rows are
    // re-loaded per tile (L1 hits after their first touch) into tile-local
    // variables, so their registers die with the tile.  Changes the summation
    // order inside a component: never used for GAAST_ARITH_STRICT.
    int tile_counter = 0;
    void emit_op_blocked(int op) {
        const gaast_op& pop = h.ops[op];
        const int hb = blocked_low_bits;
        std::map<uint32_t, std::map<uint32_t, std::vector<int>>> tiles;  // out_high -> left_high -> ACC nodes
        std::map<uint32_t, int> first_link, last_link;                    // out slot -> node
        for (int id : op_accs[op]) {
            const Node& n = nodes[id];
            if (!n.live) continue;
            tiles[slot_blade[pop.dst][n.out_slot] >> hb][slot_blade[pop.a][n.l_slot] >> hb].push_back(id);
            if (!first_link.count(n.out_slot)) first_link[n.out_slot] = id;
            last_link[n.out_slot] = id;
        }
        for (auto& row : tiles) {
            // accumulators of this output coset, initialised with the pre-op value
            std::set<uint32_t> outs;
            for (auto& t : row.second)
                for (int id : t.second) outs.insert(nodes[id].out_slot);
            std::map<uint32_t, bool> started;
            for (uint32_t o : outs) {
                const Ref pre = nodes[first_link[o]].a;
                emit(pre.id);
                const std::string q = "q" + std::to_string(last_link[o]);
                if (is_zero(pre)) {
                    line("D " + q + ";");
                    started[o] = false;
                } else {
                    line("D " + q + " = " + opnd(pre, true) + ";");
                    started[o] = true;
                }
            }
            for (auto& t : row.second) {
                // operands that live in registers are declared at function scope, before the tile's braces
                for (int id : t.second)
                    for (Ref r : {nodes[id].b, nodes[id].c})
                        if (!(nodes[r.id].k == N_LOAD && !nodes[r.id].uniform && nodes[r.id].reload)) emit(r.id);
                line("{");
                ++indent;
                std::map<int, std::string> local;
                auto name_of = [&](Ref r) -> std::string {
                    const Node& n = nodes[r.id];
                    if (n.k == N_LOAD && !n.uniform && n.reload) {
                        auto it = local.find(r.id);
                        if (it != local.end()) return it->second;
                        const std::string s = std::to_string(n.stream);
                        const std::string nm = "t" + std::to_string(r.id) + "_" + std::to_string(tile_counter);
                        line("const D " + nm + " = " + smem_read(n) + ";");
                        (void)s;
                        local.emplace(r.id, nm);
                        return nm;
                    }
                    emit(r.id);
                    return std::string();
                };
                std::vector<std::pair<std::string, std::string>> names;
                for (int id : t.second) names.push_back({name_of(nodes[id].b), name_of(nodes[id].c)});
                size_t i = 0;
                for (int id : t.second) {
                    const Node& n = nodes[id];
                    const std::string q = "q" + std::to_string(last_link[n.out_slot]);
                    const std::string L = opnd(n.b, true, acc_flip(n), names[i].first);
                    const std::string R = opnd(n.c, true, false, names[i].second);
                    line(q + " = " + acc_rhs(n, true, L, R, q, !started[n.out_slot]) + ";");
                    started[n.out_slot] = true;
                    ++i;
                }
                --indent;
                line("}");
                ++tile_counter;
            }
            for (uint32_t o : outs) {
                const int fin = last_link[o];
                line("const D " + var(fin) + " = q" + std::to_string(fin) + ";");
                store_if_root(fin);
            }
        }
        for (int id : op_accs[op]) emitted[id] = 1;
    }
    int blocked_low_bits = 4;

    // ---- DENSE: a full geometric product written straight to the root, as a ROLLED loop ----
    // G(n) = G(hi) (x) G(lo) with lo = the 4 lowest basis vectors.  For blades a = (ah, al),
    // b = (bh, bl) the coefficient factorises:  c(a,b) = sigma(ah,bh) * (-1)^(|ah||bl|) * lambda(al,bl)
    // (pairs (i in a, j in b, i > j): hi-hi, hi-lo = all of them, lo-hi = none, lo-lo).
    // So all tiles of the Cayley table are the SAME 256-FMA lo-product up to a per-tile factor
    // and a grade involution of the right operand's lo part.  The kernel loops over the output
    // coset oh (not unrolled: the right operand's rows, the tile factor and the output rows are
    // looked up), with the 2^hi left cosets unrolled (left operand in registers).  Code size
    // drops from 2^(2n) to 2^hi * 256 FMAs (cfg3: 64 KB -> 16 KB, inside the instruction cache:
    // the straight-line version lost 1.25 of 5.3 stall cycles per instruction to `no_instruction`).
    struct Dense {
        int op = -1, n = 0, H = 1;
        std::vector<Ref> left;          // [blade]
        std::vector<int> right;         // [blade] parked load nodes
        std::vector<int> out_col;       // [blade] root column
        std::vector<char> out_neg;      // [blade]
        std::vector<double> sigma;      // [ah * H + bh]
        std::vector<double> lambda;     // [al * 16 + bl]
        bool unit_sigma = true;
        // matrix-representation product (n = 6, +-1 metric): see plan_matrep
        struct MatRep {
            struct Tri { int out, a, b, sign; };
            bool ok = false;
            int tau_blade[64], tau_sign[64];  // tensor basis element tau = k0 + 4 k1 + 16 k2  ==  sign * e_blade
            bool fast[3] = {false, false, false};  // the factor is M_2(R) and is multiplied in its matrix-unit basis
            int F[3][4][4];                   // fast factor: matrix entry e = 2 row + col from basis coefficient k; else identity
            std::vector<Tri> tri[3];          // the factor's multiplication table: 8 entries (2 x 2 matmul) or 16
            int group = 1;                    // a full-table factor: its output index labels the four accumulator groups
            int n_fma = 0, n_add = 0;         // operations per element
            int perm[6];
        } mr;
        std::vector<char> right_neg;          // [blade] the right operand enters negated (A * B.ginvol()); matrix path only
    } dense;
    std::ostringstream file_scope, kernel_setup;
    bool dense_tmem = false;  // DENSE: left operand parked in tensor memory (3 blocks per SM instead of 2)
    bool dense_by_blade = false;  // DENSE: shared-memory row of a right-operand component = its blade index
    size_t setup_doubles = 0;  // shared memory reserved ahead of the sums / staging areas

    bool plan_dense(int op, const std::vector<int>& refcount) {
        const gaast_op& pop = h.ops[op];
        const int n = int(h.n), hb = blocked_low_bits;
        if (n <= hb || n > 6 || pop.dst != 0) return false;
        const size_t B = size_t(1) << n;
        Dense d;
        d.op = op;
        d.n = n;
        d.H = 1 << (n - hb);
        d.left.assign(B, Ref{-1, false});
        d.right.assign(B, -1);
        d.right_neg.assign(B, 0);
        d.out_col.assign(B, -1);
        d.out_neg.assign(B, 0);
        d.sigma.assign(size_t(d.H) * d.H, 0.0);
        d.lambda.assign(256, 0.0);
        std::vector<double> coeff(B * B, 0.0);
        std::vector<char> seen(B * B, 0);
        std::vector<int> last(B, -1);
        size_t count = 0;
        for (int id : op_accs[op]) {
            const Node& nd = nodes[id];
            if (!nd.live || nd.uniform) return false;
            const uint32_t a = slot_blade[pop.a][nd.l_slot], b = slot_blade[pop.b][nd.r_slot];
            const uint32_t o = slot_blade[pop.dst][nd.out_slot];
            if ((a ^ b) != o || seen[a * B + b]) return false;
            seen[a * B + b] = 1;
            coeff[a * B + b] = nd.cval;
            ++count;
            if (d.left[a].id >= 0 && (d.left[a].id != nd.b.id || d.left[a].neg != nd.b.neg)) return false;
            d.left[a] = nd.b;
            const Node& r = nodes[nd.c.id];
            if (r.k != N_LOAD || r.uniform) return false;
            if (d.right[b] >= 0 && (d.right[b] != nd.c.id || bool(d.right_neg[b]) != nd.c.neg)) return false;
            d.right[b] = nd.c.id;
            d.right_neg[b] = nd.c.neg;
            if (last[o] < 0 && !is_zero(nd.a)) return false;  // accumulators must start from zero
            last[o] = id;
        }
        if (count != B * B) return false;
        // every output must be a root component, used by nothing else
        for (size_t o = 0; o < B; ++o) {
            if (last[o] < 0 || refcount[last[o]] != 0) return false;
            for (size_t col = 0; col < buf[0].size(); ++col)
                if (buf[0][col].id == last[o]) {
                    if (d.out_col[o] >= 0 || buf[0][col].neg) return false;
                    d.out_col[o] = int(col);
                }
            if (d.out_col[o] < 0) return false;
        }
        // factorisation, verified term by term
        const uint32_t lo = (1u << hb) - 1;
        for (int ah = 0; ah < d.H; ++ah)
            for (int bh = 0; bh < d.H; ++bh) {
                d.sigma[ah * d.H + bh] = coeff[(size_t(ah) << hb) * B + (size_t(bh) << hb)];
                if (std::fabs(d.sigma[ah * d.H + bh]) != 1.0) d.unit_sigma = false;
            }
        for (uint32_t al = 0; al <= lo; ++al)
            for (uint32_t bl = 0; bl <= lo; ++bl) d.lambda[al * 16 + bl] = coeff[size_t(al) * B + bl];
        for (size_t a = 0; a < B; ++a)
            for (size_t b = 0; b < B; ++b) {
                const int ah = int(a >> hb), bh = int(b >> hb);
                const uint32_t al = uint32_t(a) & lo, bl = uint32_t(b) & lo;
                const double chi = (__builtin_popcount(ah) * __builtin_popcount(bl)) & 1 ? -1.0 : 1.0;
                if (coeff[a * B + b] != d.sigma[ah * d.H + bh] * chi * d.lambda[al * 16 + bl]) return false;
            }
        // (a negated right operand is folded into the signs: undo it in the table the schemes are derived from)
        bool any_right_neg = false;
        for (size_t b = 0; b < B; ++b) any_right_neg |= bool(d.right_neg[b]);
        if (d.unit_sigma) plan_matrep(d, coeff);
        if (any_right_neg && !d.mr.ok) return false;  // only the matrix path takes per-blade signs
        // a projected root: the rolled product stores whole cosets, and its 4^n FMAs are never fewer than the terms
        // of the selected components -- only the matrix path (fewer FMAs than the full table) is kept
        if (h.projected && !d.mr.ok) return false;
        dense = d;
        return true;
    }

    // ---- the full geometric product of G(6) through its matrix representation ------------------
    // G(p,q), p + q = 6, is a tensor product of three 4-dimensional algebras that commute with each other:
    // with Omega_j = g_1 ... g_2j (the generators taken in some order g), factor j is generated by
    // x_j = Omega_j g_(2j+1) and y_j = Omega_j g_(2j+2), which anticommute and square to +-1.  A factor with a
    // generator of square +1 is the algebra of real 2 x 2 matrices, M_2(R): in the basis of matrix units its
    // product costs 8 multiplications instead of 16; a factor with x^2 = y^2 = -1 is the quaternions.  Every
    // basis element of the tensor product is +- one blade (a signed permutation of the 64 components), the
    // change to matrix units is one add / subtract per component and factor, and the 4 096-term product
    // becomes, with two factors in matrix form,  2 x 128 (operand transforms) + 8 x 16 x 8 = 1 024 FMAs + 128 + 64
    // (result transform, scaling) = 1 472 FP64 operations: G(6,0) = M_2(R) (x) H (x) M_2(R) = M_4(H).  The generator
    // order is searched for the most M_2(R) factors; one factor is always multiplied out in full (its output index
    // labels the accumulator groups), so at most two are taken in matrix form (G(0,6) = H (x) M_2(R) (x) H has one:
    // 2 048 FMAs).  The tables are derived from the plan's own coefficient table and the scheme is checked
    // numerically against that table before it is used (variant bit 17 switches it off: the 4 096-FMA rolled product).
    // A different summation order and a few roundings per component more than the reference: FMA arithmetic only.
    using MatRep = Dense::MatRep;
    static void matrep_apply(const MatRep& m, const double* A, const double* Bv, double* C) {
        auto along = [&](double* v, int j, bool transpose) {  // apply F[j] (or its transpose) along axis j
            const int stride = j == 0 ? 1 : j == 1 ? 4 : 16;
            double out[64];
            for (int base = 0; base < 64; ++base) {
                if ((base / stride) % 4) continue;
                for (int e = 0; e < 4; ++e) {
                    double acc = 0;
                    for (int k = 0; k < 4; ++k) acc += (transpose ? m.F[j][k][e] : m.F[j][e][k]) * v[base + k * stride];
                    out[base + e * stride] = acc;
                }
            }
            for (int i = 0; i < 64; ++i) v[i] = out[i];
        };
        double a2[64], b2[64], c2[64] = {};
        for (int tau = 0; tau < 64; ++tau) {
            a2[tau] = m.tau_sign[tau] * A[m.tau_blade[tau]];
            b2[tau] = m.tau_sign[tau] * Bv[m.tau_blade[tau]];
        }
        for (int j = 0; j < 3; ++j) { along(a2, j, false); along(b2, j, false); }
        for (const auto& t0 : m.tri[0])
            for (const auto& t1 : m.tri[1])
                for (const auto& t2 : m.tri[2])
                    c2[t0.out + 4 * t1.out + 16 * t2.out] +=
                        t0.sign * t1.sign * t2.sign * a2[t0.a + 4 * t1.a + 16 * t2.a] * b2[t0.b + 4 * t1.b + 16 * t2.b];
        double scale = 1.0;
        for (int j = 0; j < 3; ++j) {
            along(c2, j, true);
            if (m.fast[j]) scale *= 0.5;
        }
        for (int tau = 0; tau < 64; ++tau) C[m.tau_blade[tau]] = scale * m.tau_sign[tau] * c2[tau];
    }

    bool plan_matrep(Dense& d, const std::vector<double>& coeff) const {
        if (d.n != 6 || (opt.variant & 131072)) return false;
        const int B = 64;
        for (double c : coeff)
            if (std::fabs(c) != 1.0) return false;
        struct SB { int blade; int sign; };
        auto mul = [&](SB a, SB b) { return SB{a.blade ^ b.blade, a.sign * b.sign * (coeff[size_t(a.blade) * B + b.blade] < 0 ? -1 : 1)}; };
        int perm[6] = {0, 1, 2, 3, 4, 5};
        MatRep best;
        int best_fast = 0;
        do {
            MatRep m;
            SB basis[3][4];
            SB omega{0, 1};
            int alpha[3], beta[3];
            for (int j = 0; j < 3; ++j) {
                const SB g1{1 << perm[2 * j], 1}, g2{1 << perm[2 * j + 1], 1};
                const SB x = mul(omega, g1), y = mul(omega, g2);
                basis[j][0] = SB{0, 1};
                basis[j][1] = x;
                basis[j][2] = y;
                basis[j][3] = mul(x, y);
                alpha[j] = mul(x, x).sign;
                beta[j] = mul(y, y).sign;
                omega = mul(mul(omega, g1), g2);
            }
            int n_fast = 0;
            for (int j = 0; j < 3; ++j) {
                m.fast[j] = alpha[j] > 0 || beta[j] > 0;
                n_fast += m.fast[j];
            }
            if (n_fast == 3) { m.fast[1] = false; n_fast = 2; }  // one factor stays in full form: the accumulator groups
            if (n_fast <= best_fast) continue;
            m.group = !m.fast[1] ? 1 : !m.fast[0] ? 0 : 2;
            // tensor basis -> signed blade (must be a bijection)
            bool seen[64] = {};
            bool ok = true;
            for (int k2 = 0; k2 < 4 && ok; ++k2)
                for (int k1 = 0; k1 < 4 && ok; ++k1)
                    for (int k0 = 0; k0 < 4; ++k0) {
                        const SB t = mul(mul(basis[0][k0], basis[1][k1]), basis[2][k2]);
                        if (seen[t.blade]) { ok = false; break; }
                        seen[t.blade] = true;
                        m.tau_blade[k0 + 4 * k1 + 16 * k2] = t.blade;
                        m.tau_sign[k0 + 4 * k1 + 16 * k2] = t.sign;
                    }
            if (!ok) continue;
            for (int j = 0; j < 3 && ok; ++j) {
                for (int e = 0; e < 4; ++e)
                    for (int k = 0; k < 4; ++k) m.F[j][e][k] = e == k;
                if (m.fast[j]) {
                    // 2 x 2 real representation: a generator of square +1 is diag(1, -1), the other one off-diagonal
                    int X[4], Y[4];  // row-major
                    if (alpha[j] > 0) {
                        X[0] = 1; X[1] = 0; X[2] = 0; X[3] = -1;
                        Y[0] = 0; Y[1] = 1; Y[2] = beta[j]; Y[3] = 0;
                    } else {
                        Y[0] = 1; Y[1] = 0; Y[2] = 0; Y[3] = -1;
                        X[0] = 0; X[1] = 1; X[2] = alpha[j]; X[3] = 0;
                    }
                    const int XY[4] = {X[0] * Y[0] + X[1] * Y[2], X[0] * Y[1] + X[1] * Y[3], X[2] * Y[0] + X[3] * Y[2], X[2] * Y[1] + X[3] * Y[3]};
                    const int I2[4] = {1, 0, 0, 1};
                    for (int e = 0; e < 4; ++e) {
                        m.F[j][e][0] = I2[e];
                        m.F[j][e][1] = X[e];
                        m.F[j][e][2] = Y[e];
                        m.F[j][e][3] = XY[e];
                    }
                    for (int i = 0; i < 2; ++i)  // C(i,l) += A(i,jj) B(jj,l)
                        for (int jj = 0; jj < 2; ++jj)
                            for (int l = 0; l < 2; ++l) m.tri[j].push_back({2 * i + l, 2 * i + jj, 2 * jj + l, 1});
                } else {
                    for (int pp = 0; pp < 4 && ok; ++pp)
                        for (int q = 0; q < 4; ++q) {
                            const SB r = mul(basis[j][pp], basis[j][q]);
                            int k = -1;
                            for (int c = 0; c < 4; ++c)
                                if (basis[j][c].blade == r.blade) k = c;
                            if (k < 0) { ok = false; break; }
                            m.tri[j].push_back({k, pp, q, r.sign * basis[j][k].sign});
                        }
                }
            }
            if (!ok) continue;
            // numerical check of the whole scheme against the plan's own table
            double A[64], Bv[64], want[64] = {}, got[64];
            uint64_t seed = 0x9E3779B97F4A7C15ull;
            auto rnd = [&]() {
                seed ^= seed << 13; seed ^= seed >> 7; seed ^= seed << 17;
                return double(int64_t(seed >> 11) % 2001 - 1000) / 1000.0;
            };
            for (int i = 0; i < 64; ++i) { A[i] = rnd(); Bv[i] = rnd(); }
            for (int a = 0; a < 64; ++a)
                for (int b = 0; b < 64; ++b) want[a ^ b] += coeff[size_t(a) * B + b] * A[a] * Bv[b];
            matrep_apply(m, A, Bv, got);
            for (int i = 0; i < 64; ++i)
                if (std::fabs(got[i] - want[i]) > 1e-9) ok = false;
            if (tuning().codegen_debug)
                std::fprintf(stderr, "[gaast codegen] matrep: order %d%d%d%d%d%d fast=%d%d%d check %s (got[0]=%g want[0]=%g)\n", perm[0], perm[1],
                             perm[2], perm[3], perm[4], perm[5], int(m.fast[0]), int(m.fast[1]), int(m.fast[2]), ok ? "ok" : "FAILED", got[0], want[0]);
            if (!ok) continue;
            for (int i = 0; i < 6; ++i) m.perm[i] = perm[i];
            m.n_fma = int(m.tri[0].size() * m.tri[1].size() * m.tri[2].size());
            m.n_add = 64 * n_fast * 3 + 64;  // two operand transforms and the result's, one scaling per component
            m.ok = true;
            best = m;
            best_fast = n_fast;
            if (best_fast == 2) break;
        } while (std::next_permutation(perm, perm + 6));
        if (!best.ok) return false;
        d.mr = best;
        return true;
    }

    // A value of the matrix path under construction: an expression text and a pending sign (signs are free: they
    // end up as operand modifiers of the add or FMA that consumes the value).
    struct SV {
        std::string text;
        int sign = 1;
    };
    std::string sv_text(const SV& v, int extra = 1) const { return v.sign * extra < 0 ? "d_neg(" + v.text + ")" : v.text; }
    // sum_k coef[k] * in[k] over the nonzero coefficients (one or two of them): an alias, or one add
    SV sv_combine(const std::string& name, const int coef[4], const SV in[4]) {
        int idx[4], c = 0;
        for (int k = 0; k < 4; ++k)
            if (coef[k]) idx[c++] = k;
        if (c == 1) return SV{in[idx[0]].text, in[idx[0]].sign * coef[idx[0]]};
        line("const " + S + " " + name + " = d_add(" + sv_text(in[idx[0]], coef[idx[0]]) + ", " + sv_text(in[idx[1]], coef[idx[1]]) + ");");
        return SV{name, 1};
    }

    void emit_op_dense_matrep(int op) {
        const Dense& d = dense;
        const MatRep& m = d.mr;
        std::vector<std::pair<size_t, uint32_t>> col_at;  // root column -> (stream, stored row)
        for (size_t si = h.n_in_streams; si < h.streams.size(); ++si)
            for (uint32_t r = 0; r < h.streams[si].rows; ++r) col_at.push_back({si, uint32_t(h.root_row[col_at.size()])});
        const int g = m.group, ja = g == 0 ? 1 : 0, jb = g == 2 ? 1 : 2;  // the group factor and the two others (ja < jb)
        const int st[3] = {1, 4, 16};
        auto T = [&](int kg, int ka, int kb) { return kg * st[g] + ka * st[ja] + kb * st[jb]; };
        auto smem_off = [&](int tau) { return std::to_string(size_t(nodes[d.right[m.tau_blade[tau]]].smem_row) * esize) + " * GAAST_THREADS"; };
        auto tag = [](int a, int b) { return std::to_string(a) + "_" + std::to_string(b); };
        // transforms a 4 x 4 block (ka, kb) along both axes; `out[ea][eb]`
        auto transform = [&](const std::string& prefix, SV in[4][4], SV out[4][4], bool transpose) {
            SV mid[4][4];
            for (int kb = 0; kb < 4; ++kb)
                for (int ea = 0; ea < 4; ++ea) {
                    int coef[4];
                    SV col[4];
                    for (int ka = 0; ka < 4; ++ka) { coef[ka] = transpose ? m.F[ja][ka][ea] : m.F[ja][ea][ka]; col[ka] = in[ka][kb]; }
                    mid[ea][kb] = sv_combine(prefix + "u" + tag(ea, kb), coef, col);
                }
            for (int ea = 0; ea < 4; ++ea)
                for (int eb = 0; eb < 4; ++eb) {
                    int coef[4];
                    SV row[4];
                    for (int kb = 0; kb < 4; ++kb) { coef[kb] = transpose ? m.F[jb][kb][eb] : m.F[jb][eb][kb]; row[kb] = mid[ea][kb]; }
                    out[ea][eb] = sv_combine(prefix + "w" + tag(ea, eb), coef, row);
                }
        };
        // ---- right operand: signed permutation + the fast transforms, in place in shared memory, one group index at a time ----
        auto right_operand = [&]() {
        for (int kg = 0; kg < 4; ++kg) {
            line("{");
            ++indent;
            SV in[4][4], out[4][4];
            for (int kb = 0; kb < 4; ++kb)
                for (int ka = 0; ka < 4; ++ka) {
                    const int tau = T(kg, ka, kb);
                    line("const " + S + " r" + tag(ka, kb) + " = xs_ld<" + smem_off(tau) + ">(xb);");
                    in[ka][kb] = SV{"r" + tag(ka, kb), m.tau_sign[tau] * (d.right_neg[size_t(m.tau_blade[tau])] ? -1 : 1)};
                }
            transform("", in, out, false);
            for (int ea = 0; ea < 4; ++ea)
                for (int eb = 0; eb < 4; ++eb) line("xs_st<" + smem_off(T(kg, ea, eb)) + ">(xb, " + sv_text(out[ea][eb]) + ");");
            --indent;
            line("}");
        }
        };
        if (!dense_tmem) right_operand();  // (tensor-memory variant: the left operand first, its 128 registers die early)
        // ---- left operand: the same transforms in registers ----
        // (variant bit 13: the transformed operand is then parked in the thread's tensor-memory lane, 16 components
        // per tcgen05.st / tcgen05.ld, and the kernel needs ~110 registers instead of 250: 3 blocks per SM)
        for (int a = 0; a < 64; ++a) emit(d.left[a].id);
        SV am[4][4][4];  // [kg][ea][eb]
        for (int kg = 0; kg < 4; ++kg) {
            if (dense_tmem) { line("{"); ++indent; }
            SV in[4][4];
            for (int kb = 0; kb < 4; ++kb)
                for (int ka = 0; ka < 4; ++ka) {
                    const int tau = T(kg, ka, kb);
                    const Ref x = d.left[size_t(m.tau_blade[tau])];
                    in[ka][kb] = SV{opnd(Ref{x.id, false}, true), m.tau_sign[tau] * (x.neg ? -1 : 1)};
                }
            transform("a" + std::to_string(kg), in, am[kg], false);
            if (dense_tmem) {
                std::string args;
                for (int ea = 0; ea < 4; ++ea)
                    for (int eb = 0; eb < 4; ++eb) args += ", " + sv_text(am[kg][ea][eb]);
                line("tm_put16(tb + " + std::to_string(32 * kg) + "u" + args + ");");
                --indent;
                line("}");
            }
        }
        if (dense_tmem) {
            line("tm_wait_st();");
            right_operand();
        }
        // ---- the product: per output index of the group factor, 16 accumulators over the two other factors ----
        int bcount = 0;
        for (int og = 0; og < 4; ++og) {
            line("{");
            ++indent;
            bool started[4][4] = {};
            for (int c = 0; c < 16; ++c) line(S + " c" + tag(c / 4, c % 4) + ";");
            for (const auto& tg : m.tri[g]) {
                if (tg.out != og) continue;
                SV aslice[4][4];
                if (dense_tmem) {
                    line("{");
                    ++indent;
                    std::string names;
                    for (int c = 0; c < 16; ++c) names += std::string(c ? ", " : "") + "a" + std::to_string(c);
                    line("double " + names + ";");
                    line("tm_get16(tb + " + std::to_string(32 * tg.a) + "u, " + names + ");");
                    for (int ea = 0; ea < 4; ++ea)
                        for (int eb = 0; eb < 4; ++eb) aslice[ea][eb] = SV{"a" + std::to_string(4 * ea + eb), 1};
                } else {
                    for (int ea = 0; ea < 4; ++ea)
                        for (int eb = 0; eb < 4; ++eb) aslice[ea][eb] = am[tg.a][ea][eb];
                }
                for (int ba = 0; ba < 4; ++ba)
                    for (int bb = 0; bb < 4; ++bb) {
                        // right-operand-major: the FMAs that share one value fresh from shared memory are consecutive
                        const std::string b = "b" + std::to_string(bcount++);
                        line("const " + S + " " + b + " = xs_ld<" + smem_off(T(tg.b, ba, bb)) + ">(xb);");
                        for (const auto& ta : m.tri[ja]) {
                            if (ta.b != ba) continue;
                            for (const auto& tb : m.tri[jb]) {
                                if (tb.b != bb) continue;
                                const std::string c = "c" + tag(ta.out, tb.out);
                                const std::string A = sv_text(aslice[ta.a][tb.a], tg.sign * ta.sign * tb.sign);
                                if (!started[ta.out][tb.out]) line(c + " = d_mul(" + A + ", " + b + ");");
                                else line(c + " = d_fma(" + A + ", " + b + ", " + c + ");");
                                started[ta.out][tb.out] = true;
                            }
                        }
                    }
                if (dense_tmem) { --indent; line("}"); }
            }
            // back to the tensor basis (the transposed transforms, 1/2 per matrix-form factor), sign, store
            SV cin[4][4], cout[4][4];
            for (int ea = 0; ea < 4; ++ea)
                for (int eb = 0; eb < 4; ++eb) cin[ea][eb] = SV{"c" + tag(ea, eb), 1};
            transform("o", cin, cout, true);
            double scale = 1.0;
            for (int j = 0; j < 3; ++j)
                if (m.fast[j]) scale *= 0.5;
            for (int ka = 0; ka < 4; ++ka)
                for (int kb = 0; kb < 4; ++kb) {
                    const int tau = T(og, ka, kb);
                    const size_t oc = size_t(d.out_col[size_t(m.tau_blade[tau])]);
                    if (!stored(oc)) continue;  // (projected away: computed, never stored)
                    const auto at = col_at[oc];
                    const double f = scale * m.tau_sign[tau] * cout[ka][kb].sign;
                    const std::string v = f == 1.0 ? cout[ka][kb].text : "d_mul(U(" + lit(f) + "), " + cout[ka][kb].text + ")";
                    if (opt.store_out)
                        line(std::string(guard_stores ? "if (active) " : "") + "d_store(s" + std::to_string(at.first) + " + " +
                             std::to_string(at.second) + " * r" + std::to_string(at.first) + " + e, " + v + ");");
                }
            --indent;
            line("}");
        }
        for (int id : op_accs[op]) emitted[id] = 1;
        for (int o = 0; o < 64; ++o) root_done[d.out_col[o]] = 1;
    }

    void emit_op_dense(int op) {
        const Dense& d = dense;
        if (d.mr.ok) {
            emit_op_dense_matrep(op);
            return;
        }
        const int hb = blocked_low_bits, B = 1 << d.n;
        // root column -> (stream, row)
        std::vector<std::pair<size_t, uint32_t>> col_at;
        for (size_t si = h.n_in_streams; si < h.streams.size(); ++si)
            for (uint32_t r = 0; r < h.streams[si].rows; ++r) col_at.push_back({si, r});
        const size_t root0 = h.n_in_streams;
        // ---- lookup tables (constant memory) ----
        file_scope << "__constant__ unsigned kDenseB[" << B << "] = {";
        for (int b = 0; b < B; ++b)
            file_scope << (b ? ", " : "") << size_t(nodes[d.right[b]].smem_row) * esize << " * GAAST_THREADS";
        file_scope << "};\n__constant__ unsigned short kDenseOutStream[" << B << "] = {";
        for (int o = 0; o < B; ++o) file_scope << (o ? ", " : "") << col_at[d.out_col[o]].first;
        file_scope << "};\n__constant__ unsigned short kDenseOutRow[" << B << "] = {";
        for (int o = 0; o < B; ++o) file_scope << (o ? ", " : "") << col_at[d.out_col[o]].second;
        file_scope << "};\n";
        if (d.unit_sigma) {
            file_scope << "__constant__ unsigned kDenseSigma[" << d.H * d.H << "] = {";  // [ah][oh] sign-bit masks
            for (int ah = 0; ah < d.H; ++ah)
                for (int oh = 0; oh < d.H; ++oh)
                    file_scope << ((ah || oh) ? ", " : "") << (d.sigma[ah * d.H + (oh ^ ah)] < 0 ? "0x80000000u" : "0u");
        } else {
            file_scope << "__constant__ " << S << " kDenseSigma[" << d.H * d.H << "] = {";
            for (int ah = 0; ah < d.H; ++ah)
                for (int oh = 0; oh < d.H; ++oh) file_scope << ((ah || oh) ? ", " : "") << lit(d.sigma[ah * d.H + (oh ^ ah)]);
        }
        file_scope << "};\n";
        // ---- per-block table of output offsets (the root's grade arrays are separate allocations) ----
        kernel_setup << "  long long* const dense_out = reinterpret_cast<long long*>(sums);\n";
        if (f32)  // EvalArgs carries the array addresses as double*: measure the distance in floats
            kernel_setup << "  if (tid < " << B << ")\n    dense_out[tid] = (long long)(reinterpret_cast<const float*>(a.sptr[kDenseOutStream[tid]]) - "
                         << "reinterpret_cast<const float*>(a.sptr[" << root0
                         << "])) + (long long)kDenseOutRow[tid] * a.srow[kDenseOutStream[tid]];\n  __syncthreads();\n";
        else
        kernel_setup << "  if (tid < " << B << ")\n    dense_out[tid] = (long long)(a.sptr[kDenseOutStream[tid]] - a.sptr[" << root0
                     << "]) + (long long)kDenseOutRow[tid] * a.srow[kDenseOutStream[tid]];\n  __syncthreads();\n";
        if (dense_tmem) {
            // ---- left operand: TENSOR MEMORY.  With the left operand in registers (128 of them)
            // only 2 blocks fit an SM and 8 warps cannot keep the FP64 pipe busy (63 %).  Parked in
            // the thread's TMEM lane (2 columns per component, blade b at column 2b) the kernel
            // needs ~130 registers: 3 blocks, 12 warps.  Both loops are rolled; a tile's 16 left
            // components arrive with ONE tcgen05.ld (32x32b.x32).
            for (int ah = 0; ah < d.H; ++ah) {
                for (int al = 0; al < 16; ++al) emit(d.left[(ah << hb) + al].id);
                std::string args;
                for (int al = 0; al < 16; ++al) args += ", " + opnd(d.left[(ah << hb) + al], true);
                line("tm_put16(tb + " + std::to_string(32 * ah) + "u" + args + ");");
            }
            line("tm_wait_st();");
            line("#pragma unroll 1");
            line("for (int oh = 0; oh < " + std::to_string(d.H) + "; ++oh) {");
            ++indent;
            for (int ol = 0; ol < 16; ++ol) line("double q" + std::to_string(ol) + " = 0.0;");
            line("#pragma unroll 1");
            line("for (int ah = 0; ah < " + std::to_string(d.H) + "; ++ah) {");
            ++indent;
            line("double a0, a1, a2, a3, a4, a5, a6, a7, a8, a9, a10, a11, a12, a13, a14, a15;");
            line("tm_get16(tb + 32u * ah, a0, a1, a2, a3, a4, a5, a6, a7, a8, a9, a10, a11, a12, a13, a14, a15);");
            line("const unsigned* const rows = kDenseB + ((oh ^ ah) << " + std::to_string(hb) + ");");
            line((d.unit_sigma ? std::string("const unsigned sg = ") : std::string("const double sg = ")) +
                 "kDenseSigma[ah * " + std::to_string(d.H) + " + oh];");
            // (-1)^(|ah||bl|): a grade involution of the right operand's lo part when |ah| is odd
            line("const unsigned inv = (__popc(ah) & 1) ? 0x80000000u : 0u;");
            for (int bl = 0; bl < 16; ++bl) {
                const std::string raw = "xs_ldd(xb + rows[" + std::to_string(bl) + "])";
                const bool oddbl = __builtin_popcount(bl) & 1;
                if (d.unit_sigma)
                    line("const double b" + std::to_string(bl) + " = flip_sign(" + raw + ", sg" + (oddbl ? " ^ inv" : "") + ");");
                else
                    line("const double b" + std::to_string(bl) + " = " + (oddbl ? "flip_sign(" + raw + ", inv)" : raw) + " * sg;");
            }
            for (int bl = 0; bl < 16; ++bl)  // right-operand-major: see the register path below
                for (int al = 0; al < 16; ++al) {
                    const double cc = d.lambda[al * 16 + bl];
                    if (cc == 0.0) continue;
                    const std::string q = "q" + std::to_string(al ^ bl);
                    const std::string A = std::string(cc < 0 ? "-" : "") + "a" + std::to_string(al);
                    const std::string Bv = "b" + std::to_string(bl);
                    if (std::fabs(cc) == 1.0)
                        line(q + " = fma(" + A + ", " + Bv + ", " + q + ");");
                    else
                        line(q + " = fma(" + A + " * " + Bv + ", " + lit(std::fabs(cc)) + ", " + q + ");");
                }
            --indent;
            line("}");
        } else {
        // ---- left operand: registers ----
        for (int a = 0; a < B; ++a) emit(d.left[a].id);
        line("#pragma unroll 1");
        line("for (int oh = 0; oh < " + std::to_string(d.H) + "; ++oh) {");
        ++indent;
        for (int ol = 0; ol < 16; ++ol) line(S + " q" + std::to_string(ol) + " = 0.0;");
        for (int ah = 0; ah < d.H; ++ah) {
            line("{");
            ++indent;
            if (dense_by_blade)
                line("const unsigned xr = xb + (unsigned)((oh ^ " + std::to_string(ah) + ") << " + std::to_string(hb) + ") * (unsigned)(" +
                     std::to_string(esize) + " * GAAST_THREADS);");
            else
            line("const unsigned* const rows = kDenseB + ((oh ^ " + std::to_string(ah) + ") << " + std::to_string(hb) + ");");
            line((d.unit_sigma ? std::string("const unsigned sg = ") : "const " + S + " sg = ") + "kDenseSigma[" +
                 std::to_string(ah * d.H) + " + oh];");
            const bool odd = __builtin_popcount(ah) & 1;
            for (int bl = 0; bl < 16; ++bl) {
                const std::string raw = dense_by_blade ? "xs_ld<" + std::to_string(size_t(bl) * esize) + " * GAAST_THREADS>(xr)"
                                                       : "xs_ldd(xb + rows[" + std::to_string(bl) + "])";
                if (d.unit_sigma)
                    line("const " + S + " b" + std::to_string(bl) + " = flip_sign(" + raw + ", sg);");
                else
                    line("const " + S + " b" + std::to_string(bl) + " = " + raw + " * sg;");
            }
            // Right-operand-major order: the 16 FMAs that share one right value b (fresh from shared memory)
            // are consecutive, so that ptxas keeps them together as each LDS lands and serves b from the
            // operand reuse cache.  A DFMA whose three register pairs all come from the register file
            // occupies the FP64 pipe for ~3.1 cycles instead of 2 (profiles/fp64_reuse.cu: 25.5 TFLOP/s
            // without reuse, 31.6 with); in left-operand-major source order ptxas interleaved the tile as the
            // loads arrived and kept .reuse on 30 % of the DFMAs (23.2 TFLOP/s), in this order on 78 % (26.5).
            for (int bl = 0; bl < 16; ++bl)
                for (int al = 0; al < 16; ++al) {
                    double cc = d.lambda[al * 16 + bl];
                    if (odd && (__builtin_popcount(bl) & 1)) cc = -cc;
                    if (cc == 0.0) continue;
                    const std::string q = "q" + std::to_string(al ^ bl);
                    const std::string A = opnd(d.left[(ah << hb) + al], true, cc < 0);
                    const std::string Bv = "b" + std::to_string(bl);
                    if (std::fabs(cc) == 1.0)
                        line(q + " = d_fma(" + A + ", " + Bv + ", " + q + ");");
                    else
                        line(q + " = d_fma(d_mul(" + A + ", " + Bv + "), " + lit(std::fabs(cc)) + ", " + q + ");");
                }
            --indent;
            line("}");
        }
        }
        // ---- store the finished coset ----
        if (opt.store_out) {
            // (with the operand in tensor memory whole warps run: a lane past the end of the batch shadows the last
            // element and must not store -- unguarded, its result from a stale staging row overwrote that element)
            if (guard_stores) line("if (active) {");
            line(S + "* const ro = s" + std::to_string(root0) + " + e;");
            for (int ol = 0; ol < 16; ++ol)
                line("ro[dense_out[(oh << " + std::to_string(hb) + ") + " +
                     std::to_string(ol) + "]] = q" + std::to_string(ol) + ";");
            if (guard_stores) line("}");
        }
        --indent;
        line("}");
        for (int id : op_accs[op]) emitted[id] = 1;
        for (int o = 0; o < B; ++o) root_done[d.out_col[o]] = 1;
    }

};

const char kPreludeExpLog[] = R"GAAST(
// exp / log factors of a k-vector with a scalar square q = <B B>_0 (GAAST_OP_EXP / GAAST_OP_LOG; the same functions as
// in table_engine.cu).  Near q = 0 both branches share one series.
__device__ __forceinline__ double s_expc(double q) {
  if (fabs(q) < 1e-8) return 1.0 + 0.5 * q;
  const double x = sqrt(fabs(q));
  return q < 0 ? cos(x) : cosh(x);
}
__device__ __forceinline__ double s_exps(double q) {
  if (fabs(q) < 1e-8) return 1.0 + q / 6.0;
  const double x = sqrt(fabs(q));
  return q < 0 ? sin(x) / x : sinh(x) / x;
}
__device__ __forceinline__ double s_logf(double a, double q) {
  if (fabs(q) < 1e-8 * a * a && a > 0) return (1.0 + q / (3.0 * a * a)) / a;
  const double x = sqrt(fabs(q));
  return q < 0 ? atan2(x, a) / x : atanh(x / a) / x;
}
)GAAST";

const char kPrelude[] = R"GAAST(
#if GAAST_EPT == 2
typedef double2 D;
__device__ __forceinline__ D U(double x) { return make_double2(x, x); }
__device__ __forceinline__ D d_load(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ void d_store(double* p, D v) { *reinterpret_cast<double2*>(p) = v; }
__device__ __forceinline__ D d_neg(D a) { return make_double2(-a.x, -a.y); }
__device__ __forceinline__ D d_fma(D a, D b, D c) { return make_double2(fma(a.x, b.x, c.x), fma(a.y, b.y, c.y)); }
__device__ __forceinline__ D d_mul(D a, D b) { return make_double2(a.x * b.x, a.y * b.y); }
__device__ __forceinline__ D d_add(D a, D b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ D d_muls(D a, D b) { return make_double2(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)); }
__device__ __forceinline__ D d_adds(D a, D b) { return make_double2(__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y)); }
__device__ __forceinline__ D d_inv(D a) { return make_double2(__ddiv_rn(1.0, a.x), __ddiv_rn(1.0, a.y)); }
__device__ __forceinline__ D d_sqrt(D a) { return make_double2(__dsqrt_rn(a.x), __dsqrt_rn(a.y)); }
__device__ __forceinline__ D d_expc(D a) { return make_double2(s_expc(a.x), s_expc(a.y)); }
__device__ __forceinline__ D d_exps(D a) { return make_double2(s_exps(a.x), s_exps(a.y)); }
__device__ __forceinline__ D d_logf(D a, D q) { return make_double2(s_logf(a.x, q.x), s_logf(a.y, q.y)); }
__device__ __forceinline__ double d_hsum(D a) { return a.x + a.y; }
#else
typedef double D;
__device__ __forceinline__ D U(double x) { return x; }
__device__ __forceinline__ D d_load(const double* p) { return __ldg(p); }
template <int OFF>
__device__ __forceinline__ void xs_st(unsigned base, double v) {
  // no "memory" clobber: volatile asm statements keep their order among themselves, which is all
  // the staging area needs, and ordinary loads / stores may be scheduled across them
  asm volatile("st.shared.f64 [%0+%1], %2;" ::"r"(base), "n"(OFF), "d"(v));
}
template <int OFF>
__device__ __forceinline__ double xs_ld(unsigned base) {
  double v;
  asm volatile("ld.volatile.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(base), "n"(OFF));
  return v;
}
__device__ __forceinline__ double xs_ldd(unsigned addr) {
  double v;
  asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ double flip_sign(double v, unsigned mask) {
  return __hiloint2double(__double2hiint(v) ^ (int)mask, __double2loint(v));
}
)GAAST";

// type-independent part of the prelude (tensor memory, TMA, mbarrier), shared by both scalar types
const char kPreludeShared[] = R"GAAST(// Tensor memory (TMEM) as per-thread scratch: one lane per thread, 32-bit columns
__device__ __forceinline__ void tm_alloc(unsigned* slot, unsigned cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   (unsigned)__cvta_generic_to_shared(slot)), "r"(cols) : "memory");
}
__device__ __forceinline__ void tm_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;"); }
__device__ __forceinline__ void tm_dealloc(unsigned taddr, unsigned cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tm_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tm_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_put(unsigned taddr, double v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__double2loint(v)),
               "r"(__double2hiint(v)));
}
__device__ __forceinline__ double tm_get(unsigned taddr) {
  unsigned lo, hi;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  return __hiloint2double((int)hi, (int)lo);
}
__device__ __forceinline__ void tm_add(unsigned taddr, double v) { tm_put(taddr, tm_get(taddr) + v); }
// Running sums absorb parked per-tile values: acc[i] += stash[i] for N consecutive components
// (2 columns each).  FULL = every lane of the tile holds a real element; otherwise idle lanes add zero.
#define GAAST_TM_ACC(NAME, N, SHAPE, OUTS_A, OUTS_S, INS)                                                         \
  template <bool FULL>                                                                                            \
  __device__ __forceinline__ void NAME(unsigned acc, unsigned stash, bool active) {                               \
    unsigned a[2 * N], s[2 * N];                                                                                   \
    asm volatile("tcgen05.ld.sync.aligned.32x32b." SHAPE ".b32 {" OUTS_S "}, [%" #INS "];" : GAAST_TM_OUT##N(a) : "r"(acc));   \
    asm volatile("tcgen05.ld.sync.aligned.32x32b." SHAPE ".b32 {" OUTS_S "}, [%" #INS "];" : GAAST_TM_OUT##N(s) : "r"(stash)); \
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");                                                   \
    _Pragma("unroll") for (int i = 0; i < N; ++i) {                                                                \
      const double sv = __hiloint2double((int)s[2 * i + 1], (int)s[2 * i]);                                        \
      const double r = __hiloint2double((int)a[2 * i + 1], (int)a[2 * i]) + (FULL || active ? sv : 0.0);           \
      a[2 * i] = (unsigned)__double2loint(r);                                                                      \
      a[2 * i + 1] = (unsigned)__double2hiint(r);                                                                  \
    }                                                                                                              \
    asm volatile("tcgen05.st.sync.aligned.32x32b." SHAPE ".b32 [%0], {" OUTS_A "};" ::"r"(acc), GAAST_TM_IN##N(a)); \
  }
#define GAAST_TM_OUT1(r) "=r"(r[0]), "=r"(r[1])
#define GAAST_TM_OUT4(r) "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
#define GAAST_TM_OUT16(r)                                                                                          \
  "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),      \
      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),       \
      "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),      \
      "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
#define GAAST_TM_IN1(r) "r"(r[0]), "r"(r[1])
#define GAAST_TM_IN4(r) "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
#define GAAST_TM_IN16(r)                                                                                           \
  "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),    \
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),  \
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),  \
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
GAAST_TM_ACC(tm_acc1, 1, "x2", "%1, %2", "%0, %1", 2)
GAAST_TM_ACC(tm_acc4, 4, "x8", "%1, %2, %3, %4, %5, %6, %7, %8", "%0, %1, %2, %3, %4, %5, %6, %7", 8)
GAAST_TM_ACC(tm_acc16, 16, "x32",
             "%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, "
             "%25, %26, %27, %28, %29, %30, %31, %32",
             "%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
             "%24, %25, %26, %27, %28, %29, %30, %31",
             32)
#define GAAST_LOHI(v) "r"(__double2loint(v)), "r"(__double2hiint(v))
__device__ __forceinline__ void tm_put16(unsigned taddr, double v0, double v1, double v2, double v3, double v4, double v5,
                                         double v6, double v7, double v8, double v9, double v10, double v11, double v12,
                                         double v13, double v14, double v15) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      GAAST_LOHI(v0), GAAST_LOHI(v1), GAAST_LOHI(v2), GAAST_LOHI(v3), GAAST_LOHI(v4), GAAST_LOHI(v5), GAAST_LOHI(v6),
      GAAST_LOHI(v7), GAAST_LOHI(v8), GAAST_LOHI(v9), GAAST_LOHI(v10), GAAST_LOHI(v11), GAAST_LOHI(v12), GAAST_LOHI(v13),
      GAAST_LOHI(v14), GAAST_LOHI(v15));
}
__device__ __forceinline__ void tm_get16(unsigned taddr, double& v0, double& v1, double& v2, double& v3, double& v4,
                                         double& v5, double& v6, double& v7, double& v8, double& v9, double& v10,
                                         double& v11, double& v12, double& v13, double& v14, double& v15) {
  unsigned r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  v0 = __hiloint2double(r[1], r[0]);    v1 = __hiloint2double(r[3], r[2]);    v2 = __hiloint2double(r[5], r[4]);
  v3 = __hiloint2double(r[7], r[6]);    v4 = __hiloint2double(r[9], r[8]);    v5 = __hiloint2double(r[11], r[10]);
  v6 = __hiloint2double(r[13], r[12]);  v7 = __hiloint2double(r[15], r[14]);  v8 = __hiloint2double(r[17], r[16]);
  v9 = __hiloint2double(r[19], r[18]);  v10 = __hiloint2double(r[21], r[20]); v11 = __hiloint2double(r[23], r[22]);
  v12 = __hiloint2double(r[25], r[24]); v13 = __hiloint2double(r[27], r[26]); v14 = __hiloint2double(r[29], r[28]);
  v15 = __hiloint2double(r[31], r[30]);
}
// TMA (bulk async copy) + mbarrier plumbing of the pipelined kernels
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_row(double* dst, const double* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void l2_prefetch_row(const double* src, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "GAAST_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra GAAST_DONE;\n"
      "bra GAAST_WAIT;\n"
      "GAAST_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
)GAAST";

const char kPreludeTail[] = R"GAAST(__device__ __forceinline__ void d_store(double* p, D v) { *p = v; }
__device__ __forceinline__ double d_hsum(D a) { return a; }
#endif
__device__ __forceinline__ double d_neg(double a) { return -a; }
__device__ __forceinline__ double d_fma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ double d_mul(double a, double b) { return a * b; }
__device__ __forceinline__ double d_add(double a, double b) { return a + b; }
__device__ __forceinline__ double d_muls(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double d_adds(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double d_inv(double a) { return __ddiv_rn(1.0, a); }
__device__ __forceinline__ double d_sqrt(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ double d_expc(double a) { return s_expc(a); }
__device__ __forceinline__ double d_exps(double a) { return s_exps(a); }
__device__ __forceinline__ double d_logf(double a, double q) { return s_logf(a, q); }
)GAAST";


// The f32 variant: same generated structure, binary32 arithmetic (FFMA), 4-byte rows.  Batch sums
// still accumulate in double.  Two elements per thread = one 64-bit access.
const char kPreludeF32Head[] = R"GAAST(
typedef float S;
#if GAAST_EPT == 2
typedef float2 D;
__device__ __forceinline__ D U(float x) { return make_float2(x, x); }
__device__ __forceinline__ D d_load(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ void d_store(float* p, D v) { *reinterpret_cast<float2*>(p) = v; }
__device__ __forceinline__ D d_neg(D a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ D d_fma(D a, D b, D c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
__device__ __forceinline__ D d_mul(D a, D b) { return make_float2(a.x * b.x, a.y * b.y); }
__device__ __forceinline__ D d_add(D a, D b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ D d_muls(D a, D b) { return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
__device__ __forceinline__ D d_adds(D a, D b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
__device__ __forceinline__ D d_inv(D a) { return make_float2(__fdiv_rn(1.0f, a.x), __fdiv_rn(1.0f, a.y)); }
__device__ __forceinline__ D d_sqrt(D a) { return make_float2(__fsqrt_rn(a.x), __fsqrt_rn(a.y)); }
__device__ __forceinline__ D d_expc(D a) { return make_float2((float)s_expc(a.x), (float)s_expc(a.y)); }
__device__ __forceinline__ D d_exps(D a) { return make_float2((float)s_exps(a.x), (float)s_exps(a.y)); }
__device__ __forceinline__ D d_logf(D a, D q) { return make_float2((float)s_logf(a.x, q.x), (float)s_logf(a.y, q.y)); }
__device__ __forceinline__ double d_hsum(D a) { return (double)a.x + (double)a.y; }
#else
typedef float D;
__device__ __forceinline__ D U(float x) { return x; }
__device__ __forceinline__ D d_load(const float* p) { return __ldg(p); }
template <int OFF>
__device__ __forceinline__ void xs_st(unsigned base, float v) {
  asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(base), "n"(OFF), "f"(v));
}
template <int OFF>
__device__ __forceinline__ float xs_ld(unsigned base) {
  float v;
  asm volatile("ld.volatile.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(base), "n"(OFF));
  return v;
}
__device__ __forceinline__ float xs_ldd(unsigned addr) {
  float v;
  asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float flip_sign(float v, unsigned mask) { return __uint_as_float(__float_as_uint(v) ^ mask); }
)GAAST";

const char kPreludeF32Tail[] = R"GAAST(__device__ __forceinline__ void tma_row(float* dst, const float* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void l2_prefetch_row(const float* src, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void d_store(float* p, D v) { *p = v; }
__device__ __forceinline__ double d_hsum(D a) { return (double)a; }
#endif
__device__ __forceinline__ float d_neg(float a) { return -a; }
__device__ __forceinline__ float d_fma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ float d_mul(float a, float b) { return a * b; }
__device__ __forceinline__ float d_add(float a, float b) { return a + b; }
__device__ __forceinline__ float d_muls(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float d_adds(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float d_inv(float a) { return __fdiv_rn(1.0f, a); }
__device__ __forceinline__ float d_sqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ float d_expc(float a) { return (float)s_expc(a); }
__device__ __forceinline__ float d_exps(float a) { return (float)s_exps(a); }
__device__ __forceinline__ float d_logf(float a, float q) { return (float)s_logf(a, q); }
)GAAST";

}  // namespace

static CodegenResult generate(const DevicePlanHost& h, const CodegenOptions& opt, bool prune) {
    Gen g(h, opt);
    g.build();
    g.mark_live();
    std::ostringstream notes;
    const int pseudo_op = int(h.ops.size());  // the linear-map lowering's FMAs belong to an extra "op"
    g.op_accs.resize(h.ops.size() + 1);
    size_t reflected = 0;
    if (!(opt.variant & 65536)) {
        reflected = g.lower_reflections(pseudo_op);
        if (reflected) {
            for (Node& n : g.nodes) n.live = false;
            g.mark_live();
            notes << "reflection(" << reflected << " sandwich" << (reflected > 1 ? "es) " : ") ");
        }
    }
    // Opt-in (variant bit 12): measured on cfg5 it frees 12 register rows but does not pay --
    // 7.20 ms vs 7.15 ms at 36 parked rows, and with fewer parked rows (20-28, still no spills)
    // ptxas has no slack left to overlap loads and FMAs: 9.1-9.4 ms.
    // Both passes rewrite the same sandwich (the factoring pulls 1/(v.v) out of the last product, the reflection pass
    // replaces that product): a plan the reflection pass took is left alone -- factoring first handed it terms it then
    // matched against their old operands (wrong results, found by tests/test_kernels_on_cpu.py).
    if ((opt.variant & 4096) && !reflected) {
        const size_t factored = g.factor_common_scalars(pseudo_op);
        if (factored) {
            for (Node& n : g.nodes) n.live = false;
            g.mark_live();
            notes << "scalar-factored(" << factored << " products) ";
        }
    }
    if (!(opt.variant & 2048)) {
        const size_t lowered = g.lower_linear(pseudo_op);
        if (lowered) {
            for (Node& n : g.nodes) n.live = false;
            g.mark_live();
            notes << "linear-map(" << lowered << " outputs) ";
        }
    }
    {
        // Straight-line code costs ~16 bytes and a few compiler milliseconds per term: beyond
        // ~24k live terms (a 1.5 MB kernel) the table engine is the better engine.
        size_t live_terms = 0;
        for (const Node& n : g.nodes) live_terms += n.live && n.k == N_ACC;
        if (live_terms > 24576 && !(opt.variant & 64))
            throw Error(GAAST_ERR_JIT, "plan too large for the specialised engine (" + std::to_string(live_terms) +
                                           " live terms): use the table engine");
    }
    if (prune) {
        g.prune = true;
        for (Node& n : g.nodes) n.live = false;
        g.mark_live();
    }
    if (h.projected) notes << "projection(" << h.stored_cols << "/" << h.buf_cols[0] << (prune ? ",pruned" : ",whole") << ") ";
    g.mark_exports();
    g.compute_blades();

    // ---- size of the live state, per product -------------------------------------
    size_t live_loads = 0;
    for (const Node& n : g.nodes)
        if (n.live && n.k == N_LOAD && !n.uniform) ++live_loads;
    const size_t root_cols = h.stored_cols;  // batch-sum columns
    // (an f32 value takes one register instead of two: the budgets below nearly double)
    const size_t kAccBudget = opt.f32 ? 128 : 72;  // values a thread can keep as accumulators next to its operands
    g.op_policy.assign(h.ops.size() + 1, P_TABLE);
    size_t widest = 0;
    int res_parked = 0, res_parkable = 0;
    size_t live_estimate = 0;  // doubles a thread keeps live (widest in-register product + resident rows)
    const size_t kDenseBudget = opt.f32 ? 160 : 110;  // values: outputs + operands of a product that may all be live
    const size_t kLiveBudget = opt.f32 ? 224 : 124;   // values a thread can hold in 255 registers next to addresses
    std::vector<int> uses(g.nodes.size(), 0);  // how many live product terms read each node
    std::set<int> blocked_loads;
    size_t widest_table = 0;
    for (size_t oi = 0; oi < h.ops.size(); ++oi) {
        if (h.ops[oi].kind != GAAST_OP_MUL_TERMS) continue;
        std::set<uint32_t> outs;
        std::set<int> ls, rs;
        size_t live_terms = 0, load_opnds = 0;
        for (int id : g.op_accs[oi]) {
            const Node& n = g.nodes[id];
            if (!n.live || n.uniform) continue;
            ++live_terms;
            outs.insert(n.out_slot);
            ls.insert(n.b.id);
            rs.insert(n.c.id);
            ++uses[n.b.id];
            ++uses[n.c.id];
        }
        for (int id : ls) load_opnds += g.nodes[id].k == N_LOAD && !g.nodes[id].uniform;
        for (int id : rs) load_opnds += g.nodes[id].k == N_LOAD && !g.nodes[id].uniform;
        const bool dense = !g.strict && outs.size() + ls.size() + rs.size() > kDenseBudget &&
                           live_terms * 4 >= ls.size() * rs.size() && load_opnds * 4 >= (ls.size() + rs.size()) * 3;
        Policy pol = outs.size() > kAccBudget ? P_GATHER : P_TABLE;
        // Strict arithmetic cannot block a dense product (the reference's term order is per output), and one accumulator per
        // output NEXT TO both operands in registers does not fit: 64 + 64 + 64 values for G(6) A*B spilled 888 bytes per thread.
        // One output chain at a time instead (cfg3 strict: 30.0 -> 20.2 ms, profiles/r2_strict_policies.txt).
        if (g.strict) {
            // (strict operands are 0.0 + row, the reference's add_grades_from onto a zeroed buffer: count those as rows)
            auto rowish = [&](int id) {
                const Node& n = g.nodes[id];
                if (n.uniform) return false;
                if (n.k == N_LOAD) return true;
                return n.k == N_ADD && g.nodes[n.a.id].k == N_ZERO && g.nodes[n.b.id].k == N_LOAD;
            };
            size_t row_opnds = 0;
            for (int id : ls) row_opnds += rowish(id);
            for (int id : rs) row_opnds += rowish(id);
            if (outs.size() + row_opnds > kLiveBudget + (opt.f32 ? 64 : 32)) pol = P_GATHER;
        }
        if (dense && outs.size() <= 144) pol = P_BLOCKED;  // (up to 2 x the f64 accumulator budget)
        if (opt.variant & 1) pol = P_TABLE;
        if (opt.variant & 2) pol = P_GATHER;
        if (pol == P_BLOCKED && !opt.with_sum && !opt.pipelined && !(opt.variant & 512) && g.dense.op < 0) {
            std::vector<int> refcount(g.nodes.size(), 0);
            for (const Node& n : g.nodes) {
                if (!n.live) continue;
                if (n.k == N_ACC) { ++refcount[n.a.id]; ++refcount[n.b.id]; ++refcount[n.c.id]; }
                else if (is_binary(n.k)) { ++refcount[n.a.id]; ++refcount[n.b.id]; }
                else if (is_unary(n.k)) ++refcount[n.a.id];
            }
            if (g.plan_dense(int(oi), refcount)) pol = P_DENSE;
        }
        g.op_policy[oi] = pol;
        if (pol == P_DENSE) {  // right operand parked (rows looked up per tile), left operand in registers
            for (int id : rs) blocked_loads.insert(id);
            for (int id : ls) g.nodes[id].pinned = true;
        }
        if (pol == P_BLOCKED) {
            // right operands are re-fetched per tile; left ones too unless variant bit 2 keeps them in registers
            for (int id : rs)
                if (g.nodes[id].k == N_LOAD) blocked_loads.insert(id);
            // (measured on cfg3: left operand in registers 19.6 TFLOP/s, both parked 13.4)
            if ((opt.variant & 4) || ls.size() > kAccBudget)
                for (int id : ls)
                    if (g.nodes[id].k == N_LOAD) blocked_loads.insert(id);
        }
        if (pol == P_TABLE) widest_table = std::max(widest_table, outs.size());
        widest = std::max(widest, outs.size());
        notes << "op" << oi << ":"
              << (pol == P_TABLE ? "table" : pol == P_GATHER ? "gather" : pol == P_DENSE ? (g.dense.mr.ok ? "dense-matrep" : "dense-rolled") : "blocked")
              << "(outs=" << outs.size() << ",terms=" << live_terms << ") ";
    }
    for (int id : g.op_accs[pseudo_op]) {
        const Node& n = g.nodes[id];
        if (!n.live || n.uniform) continue;
        ++uses[n.b.id];
        ++uses[n.c.id];
    }
    for (int id : blocked_loads) g.nodes[id].reload = true;
    // Register pressure of everything else: the widest in-register product plus the
    // input rows that stay live.  Rows with the fewest uses are re-fetched first.
    {
        std::vector<std::pair<int, int>> cand;  // (uses, node)
        size_t kept = 0;
        for (size_t id = 0; id < g.nodes.size(); ++id) {
            const Node& n = g.nodes[id];
            if (!n.live || n.k != N_LOAD || n.uniform || n.reload) continue;
            ++kept;
            if (uses[id] > 1 && !n.pinned) cand.push_back({uses[id], int(id)});
        }
        size_t pressure = widest_table + kept + 12;
        live_estimate = pressure;
        size_t want = pressure > kLiveBudget ? pressure - kLiveBudget : 0;
        if (opt.variant >> 24) want = size_t(opt.variant >> 24) - 1;  // tuning override: variant |= (count + 1) << 24
        want += size_t(opt.extra_parked);  // raised by the compile-and-check loop while ptxas reports spills
        std::sort(cand.begin(), cand.end());
        size_t n_reload = 0;
        for (auto& c : cand) {
            if (n_reload >= want) break;
            g.nodes[c.second].reload = true;
            ++n_reload;
        }
        if (n_reload) notes << "parked=" << n_reload << " ";
        res_parked = int(n_reload);
        res_parkable = int(cand.size());
    }
    int n_smem_rows = 0;
    for (Node& n : g.nodes)
        if (n.live && n.k == N_LOAD && n.reload && !n.uniform) n.smem_row = n_smem_rows++;
    // Rolled dense product: the right operand's rows are laid out by blade (row = blade index), so that
    // a tile's 16 values sit at compile-time offsets from ONE base address (coset * 16 rows) instead
    // of being looked up row by row in a constant table (GAAST_DENSE_TABLE_ROWS=1 keeps the table: A/B runs).
    g.dense_by_blade = false;
    if (g.dense.op >= 0) {
        bool only_right = true;
        std::set<int> right(g.dense.right.begin(), g.dense.right.end());
        for (size_t id = 0; id < g.nodes.size(); ++id) {
            const Node& n = g.nodes[id];
            if (n.live && n.k == N_LOAD && n.reload && !n.uniform && !right.count(int(id))) only_right = false;
        }
        if (only_right && int(right.size()) == n_smem_rows && !tuning().dense_table_rows) {
            for (size_t b = 0; b < g.dense.right.size(); ++b) g.nodes[g.dense.right[b]].smem_row = int(b);
            g.dense_by_blade = true;
        }
    }
    int ept = opt.elems_per_thread;
    if (ept != 1 && ept != 2) ept = (live_loads + root_cols + widest <= (opt.f32 ? 96u : 48u)) ? 2 : 1;
    if (n_smem_rows) ept = 1;  // the staging area holds one double per row and thread
    g.ept = ept;
    const int threads = (opt.variant & 16384) ? 64 : 128;  // (tuning knob: 64-thread blocks = twice as many, half as large tiles per SM)

    CodegenResult res;
    res.kernel_name = "gaast_eval";
    res.threads = threads;
    res.elems_per_thread = ept;
    res.n_uniform = g.n_export;
    res.n_sum_cols = opt.with_sum ? int(root_cols) : 0;
    constexpr size_t kSmemLimit = 227 * 1024;
    // Batch-sum with the per-element result also stored: the block sums its own freshly
    // written output tile back from L2 (row segments are contiguous), instead of keeping
    // per-thread column sums in shared memory (measured: MIO-bound, profiles/r1_cfg5_sum_v2_ncu.txt).
    // Batch-sum accumulators in tensor memory (2 columns per component and lane; allocations are
    // powers of two >= 32 columns, and two resident blocks must share the SM's 512 columns).
    // Room for a stash of per-tile values next to the accumulators is taken when it is free
    // (an allocation is a power of two anyway) or cheap (at most 256 of the SM's 512 columns).
    uint32_t tmem_cols = 32;
    while (tmem_cols < 2 * root_cols) tmem_cols *= 2;
    while (tmem_cols < 4 * root_cols && tmem_cols < 256) tmem_cols *= 2;
    // Tensor memory pays when shared memory (MIO) is the busy resource, i.e. when input rows are parked there
    // (round-1 cfg5: per-thread column sums in shared memory 10.0 ms, TMEM stash 8.35 ms).  A kernel without parked rows
    // -- cfg5 after the reflection lowering -- has the LSU idle and keeps its column sums in shared memory: 5.92 ms
    // against 5.98 ms with the stash (and 5.75 ms without any sum), at 64 blocks per resident slot.
    const bool tmem_sum = opt.with_sum && ept == 1 && !opt.pipelined && !(opt.variant & 32) && tmem_cols <= 256 &&
                          (n_smem_rows > 0 || (opt.variant & 262144));
    const size_t sum_doubles = g.dense.op >= 0 ? (size_t(1) << h.n)  // table of output offsets (dense excludes the sum)
                               : !opt.with_sum ? 0
                               : tmem_sum      ? ((threads / 32) * root_cols + 2 + 15) / 16 * 16
                                               : root_cols * size_t(threads);
    const size_t pipe_bytes = sum_doubles * 8 + size_t(2 * n_smem_rows) * threads * 8 + 16;
    // (TMA staging and the persistent pipeline are f64-only: the f32 variant parks rows with LDG + STS)
    const bool pipelined = opt.pipelined && n_smem_rows > 0 && ept == 1 && pipe_bytes <= kSmemLimit / 2 && !opt.f32;
    if (sum_doubles * 8 + size_t(n_smem_rows) * threads * g.esize > kSmemLimit)
        throw Error(GAAST_ERR_JIT, "plan too wide for the specialised engine (shared-memory staging exceeds 227 KB)");
    // TMA staging pays off when most rows are parked (dense products: cfg3 21.2 -> 22.8 TFLOP/s);
    // with a few dozen parked rows next to register rows, LDG + STS is as fast (cfg5: 0.83 vs 0.80)
    bool has_dense = false;
    for (Policy p : g.op_policy) has_dense |= p == P_DENSE || p == P_BLOCKED;
    const bool tma_stage = opt.tma_stage && has_dense && n_smem_rows > 0 && ept == 1 && !pipelined && !opt.with_sum;
    const bool par_issue = (opt.variant & 256) && !opt.f32;     // opt-in experiments (f64 only), see DESIGN.md
    const bool look_ahead = (opt.variant & 32768) && !opt.f32;
    g.dense_tmem = tma_stage && g.dense.op >= 0 && (opt.variant & 8192) && !opt.f32;
    g.pipelined = pipelined;
    g.guard_stores = pipelined || tmem_sum || g.dense_tmem;
    g.sum_in_smem = opt.with_sum && !tmem_sum;
    g.sum_in_tmem = tmem_sum;
    g.sum_stash = tmem_sum && !(opt.variant & 128) ? std::min<size_t>(root_cols, (tmem_cols - 2 * root_cols) / 2) : 0;
    res.pipelined = pipelined;
    res.smem_bytes = pipelined ? pipe_bytes : sum_doubles * 8 + size_t(n_smem_rows) * threads * g.esize + (tma_stage ? 16 : 0);
    res.one_tile_blocks = tma_stage;
    if (tma_stage) notes << "tma-staged ";
    if (tmem_sum) notes << "sum-in-tmem(" << tmem_cols << "cols,stash=" << g.sum_stash << ") ";
    if (pipelined) notes << "tma-pipelined ";
    res.parked = res_parked;
    res.parkable = res_parkable;
    for (const Node& n : g.nodes) res.fma_per_elem += n.live && n.k == N_ACC && !n.uniform;
    if (g.dense.op >= 0 && g.dense.mr.ok) {
        // the matrix-representation product executes 1 024 (2 048) FMAs + 448 (256) additions / scalings for the op's 4 096 terms:
        // reported as flop / 2, so that 2 x fma/elem stays the executed flop count
        res.fma_per_elem += (2 * g.dense.mr.n_fma + g.dense.mr.n_add) / 2 - 4096;
    }

    std::ostringstream src;
    src << "// generated by gaast_b200 codegen: n=" << h.n << " terms=" << h.total_terms << " arith="
        << (g.strict ? "strict" : "fma") << " sum=" << int(opt.with_sum) << " store=" << int(opt.store_out)
        << " bcast=0x" << std::hex << opt.broadcast_slots << std::dec << (opt.f32 ? " dtype=f32" : "") << "\n// " << notes.str() << "\n";
    // Small kernels are pure streaming: ask for several resident blocks so that ptxas does not
    // trade occupancy for hoisting (cfg2_full: 254 registers without this, 2 blocks per SM).
    const size_t live_regs = live_estimate * size_t(ept);
    // (ptxas treats the hint as a register budget to spend: only give it when it is a tight one)
    // (rolled dense product in f32: 64 left components + a 16 x 16 tile = ~110 registers, 4 blocks per SM)
    const int min_blocks = g.dense_tmem ? 3
                           : g.dense.op >= 0 ? (opt.f32 ? 4 : (opt.variant & 524288) ? 3 : 1)  // (bit 19: experiment, 168 registers)
                           : live_regs <= (opt.f32 ? 80u : 40u) ? 8 : live_regs <= (opt.f32 ? 128u : 64u) ? 4 : 1;
    res.min_blocks = min_blocks;
    src << "#define GAAST_EPT " << ept << "\n#define GAAST_THREADS " << threads << "\n#define GAAST_MIN_BLOCKS "
        << min_blocks << "\n";
    src << kEvalArgsText << "\nusing gaast::EvalArgs;\n" << kPreludeExpLog << (opt.f32 ? kPreludeF32Head : kPrelude) << kPreludeShared << (opt.f32 ? kPreludeF32Tail : kPreludeTail) << "\n";

    std::ostringstream loop_strides;
    auto stream_decls = [&](std::ostringstream& o, bool prologue) {
        std::set<int> used;
        for (const Node& n : g.nodes)
            if (n.live && n.k == N_LOAD && (!prologue || n.uniform)) used.insert(n.stream);
        if (!prologue && opt.store_out)
            for (size_t i = h.n_in_streams; i < h.streams.size(); ++i) used.insert(int(i));
        for (int s : used) {
            const bool out = size_t(s) >= h.n_in_streams;
            if (opt.f32)
                o << "  " << (out ? "float* __restrict__ s" : "const float* __restrict__ s") << s << " = reinterpret_cast<"
                  << (out ? "float*" : "const float*") << ">(a.sptr[" << s << "]); const long long R" << s << " = a.srow[" << s
                  << "]; const long long r" << s << " = R" << s << ";\n";
            else
            o << "  " << (out ? "double* __restrict__ s" : "const double* __restrict__ s") << s << " = a.sptr[" << s
              << "]; const long long R" << s << " = a.srow[" << s << "]; const long long r" << s << " = R" << s << ";\n";
            // Inside the element loop the stride is made opaque: otherwise the compiler hoists
            // every `row * stride` out of the loop and keeps dozens of 64-bit offsets live.
            if (!prologue)
                loop_strides << "    long long r" << s << " = R" << s << "; asm volatile(\"\" : \"+l\"(r" << s << "));\n";
        }
    };

    // ---- prologue: values shared by the whole batch --------------------------------
    if (g.n_export > 0) {
        res.uniform_kernel_name = "gaast_uniform";
        g.emitted.assign(g.nodes.size(), 0);
        g.in_prologue = true;
        g.indent = 1;
        g.body.str("");
        std::vector<std::pair<int, int>> exports;  // (index, node)
        for (size_t id = 0; id < g.nodes.size(); ++id)
            if (g.nodes[id].live && g.nodes[id].export_idx >= 0) exports.push_back({g.nodes[id].export_idx, int(id)});
        std::sort(exports.begin(), exports.end());
        for (auto& ex : exports) g.emit(ex.second);
        src << "extern \"C\" __global__ void __launch_bounds__(32) gaast_uniform(const __grid_constant__ EvalArgs a) {\n";
        src << "  if (threadIdx.x != 0 || blockIdx.x != 0) return;\n";
        stream_decls(src, true);
        if (opt.f32) src << "  float* __restrict__ uo = reinterpret_cast<float*>(const_cast<double*>(a.uniform));\n";
        else src << "  double* __restrict__ uo = const_cast<double*>(a.uniform);\n";
        src << g.body.str();
        for (auto& ex : exports) src << "  uo[" << ex.first << "] = " << g.var(ex.second) << ";\n";
        src << "}\n\n";
    }

    // ---- per-element kernel -----------------------------------------------------------
    g.emitted.assign(g.nodes.size(), 0);
    g.in_prologue = false;
    g.indent = 2;
    g.body.str("");
    // leaves shared by the whole batch are read once, outside the element loop
    std::ostringstream uni;
    {
        g.indent = 1;
        std::vector<char> used(g.nodes.size(), 0);
        for (const Node& n : g.nodes) {
            if (!n.live || n.uniform) continue;
            used[n.a.id] = used[n.b.id] = used[n.c.id] = 1;
        }
        for (size_t col = 0; col < g.buf[0].size(); ++col)
            if (g.stored(col)) used[g.buf[0][col].id] = 1;
        // a handful of shared values live in registers for the whole kernel; a large table of
        // them (a wide linear map) is read at its point of use instead (uniform, L1-resident)
        size_t n_shared = 0;
        for (size_t id = 0; id < g.nodes.size(); ++id) {
            const Node& n = g.nodes[id];
            n_shared += n.live && n.uniform && used[id] && (n.k == N_LOAD || n.export_idx >= 0);
        }
        for (size_t id = 0; id < g.nodes.size() && n_shared <= 32; ++id) {
            const Node& n = g.nodes[id];
            if (!n.live || !n.uniform || !used[id]) continue;
            if (n.k == N_LOAD || n.export_idx >= 0) g.emit(int(id));
        }
        uni << g.body.str();
        g.body.str("");
        g.indent = 2;
        g.in_loop = true;
        if (g.n_export > 0 && opt.f32)
            loop_strides << "    const float* uni = reinterpret_cast<const float*>(a.uniform); asm volatile(\"\" : \"+l\"(uni));\n";
        else if (g.n_export > 0) loop_strides << "    const double* uni = a.uniform; asm volatile(\"\" : \"+l\"(uni));\n";
    }
    // root components, in slot order
    {
        std::vector<Gen::RootSlot> slots;  // the stored ones (a projected plan: the selected components)
        uint32_t col = 0;
        for (size_t si = h.n_in_streams; si < h.streams.size(); ++si)
            for (uint32_t r = 0; r < h.streams[si].rows; ++r, ++col)
                if (g.stored(col))
                    slots.push_back(Gen::RootSlot{si, uint32_t(h.root_row[col]), col, g.buf[0][col].neg, uint32_t(h.root_sum_col[col])});
        g.root_done.assign(h.buf_cols[0], 0);
        g.root_of.clear();
        // one-tile blocks with TMA staging: the parked rows are already on their way to shared
        // memory (bulk copies issued by thread 0 at kernel start); otherwise LDG + STS here
        if (!tma_stage) g.emit_staging();
        // Rows that stay in registers and are read by several terms are fetched in one
        // burst at the top of the body: loads issued lazily in the middle of a
        // register-bound body expose one full memory latency each.
        if (!(opt.variant & 16))
            for (size_t id = 0; id < g.nodes.size(); ++id) {
                const Node& n = g.nodes[id];
                if (n.live && n.k == N_LOAD && !n.uniform && !n.reload && uses[id] >= 2) g.emit(int(id));
            }
        if (tma_stage) g.line("mbar_wait(stage_bar, 0u);  // parked rows have landed");
        for (const auto& rs : slots) g.root_of.emplace(g.buf[0][rs.col].id, rs);
        for (const auto& rs : slots) {
            const int id = g.buf[0][rs.col].id;
            g.emit(id);            // products store their outputs as soon as they are complete ...
            g.emit_root(rs, id);   // ... everything else (leaves, sums, unary results) is stored here
        }
    }
    if (tma_stage && par_issue) {  // parked row -> (stream, row), for the lanes that issue the copies
        std::vector<const Node*> parked(size_t(n_smem_rows), nullptr);
        for (const Node& n : g.nodes)
            if (n.live && n.k == N_LOAD && !n.uniform && n.reload) parked[size_t(n.smem_row)] = &n;
        g.file_scope << "__constant__ unsigned short kStageStream[" << n_smem_rows << "] = {";
        for (int r = 0; r < n_smem_rows; ++r) g.file_scope << (r ? ", " : "") << parked[size_t(r)]->stream;
        g.file_scope << "};\n__constant__ unsigned short kStageRow[" << n_smem_rows << "] = {";
        for (int r = 0; r < n_smem_rows; ++r) g.file_scope << (r ? ", " : "") << parked[size_t(r)]->row;
        g.file_scope << "};\n";
        if (look_ahead) {
            std::ostringstream ls, lr;
            bool first = true;
            for (const Node& n : g.nodes)
                if (n.live && n.k == N_LOAD && !n.uniform) {
                    ls << (first ? "" : ", ") << n.stream;
                    lr << (first ? "" : ", ") << n.row;
                    first = false;
                }
            g.file_scope << "__constant__ unsigned short kLoadStream[] = {" << ls.str() << "};\n__constant__ unsigned short kLoadRow[] = {"
                         << lr.str() << "};\n";
        }
    }
    src << g.file_scope.str();
    if (tmem_sum) {  // accumulator k (emission order) -> root column
        src << "__device__ const short gaast_sum_col[" << root_cols << "] = {";
        for (size_t k = 0; k < g.sum_order.size(); ++k) src << (k ? ", " : "") << g.sum_order[k];
        src << "};\n";
    }
    src << "extern \"C\" __global__ void " << (min_blocks > 1 ? "__launch_bounds__(GAAST_THREADS, GAAST_MIN_BLOCKS)" : "__launch_bounds__(GAAST_THREADS)")
        << " gaast_eval(const __grid_constant__ EvalArgs a) {\n";
    src << "  const int tid = threadIdx.x;\n";
    stream_decls(src, false);
    if (opt.with_sum || n_smem_rows) src << "  extern __shared__ double sums[];\n";
    src << g.kernel_setup.str();
    if (g.sum_in_smem) src << "  for (int c = 0; c < " << root_cols << "; ++c) sums[c * GAAST_THREADS + tid] = 0.0;\n";
    if (tmem_sum) {
        // Batch-sum accumulators live in TENSOR MEMORY: each thread owns one TMEM lane, 2 columns
        // per root component.  Registers are full and shared memory (MIO) is the saturated
        // resource of these kernels (profiles/r1_cfg5_sum_v2_ncu.txt); TMEM has its own datapath.
        src << "  const int lane = tid & 31, warp = tid >> 5;\n";
        src << "  unsigned* const tslot = reinterpret_cast<unsigned*>(sums + " << (threads / 32) * root_cols << ");\n";
        src << "  if (warp == 0) { tm_alloc(tslot, " << tmem_cols << "u); tm_relinquish(); }\n";
        src << "  tm_fence_before_sync();\n  __syncthreads();\n  tm_fence_after_sync();\n";
        src << "  const unsigned tmem_base = *tslot;\n";
        src << "  const unsigned tb = tmem_base + ((unsigned)(warp * 32) << 16);\n";
        src << "  for (int c = 0; c < " << root_cols << "; ++c) tm_put(tb + 2u * c, 0.0);\n";
        src << "  tm_wait_st();\n";
    }
    src << uni.str();
    if (pipelined) {
        // Persistent block, two staging buffers.  The TMA unit copies the parked rows
        // of tile t+2 into the buffer tile t has just released (one bulk copy per row:
        // a row's 128-element segment is contiguous in the batch-innermost layout),
        // completion is signalled on an mbarrier; the rows a thread keeps in registers
        // are pulled into L2 two tiles ahead with bulk prefetches.
        const int P = n_smem_rows;
        std::vector<const Node*> parked(size_t(P), nullptr), in_regs;
        for (const Node& n : g.nodes) {
            if (!n.live || n.k != N_LOAD || n.uniform) continue;
            if (n.reload) parked[size_t(n.smem_row)] = &n;
            else in_regs.push_back(&n);
        }
        src << "  double* const stage0 = sums + " << sum_doubles << ";\n";
        src << "  unsigned long long* const mbar = reinterpret_cast<unsigned long long*>(stage0 + 2 * " << P
            << " * GAAST_THREADS);\n";
        src << "  const long long n_tiles = (a.n + GAAST_THREADS - 1) / GAAST_THREADS;\n";
        src << "  if (tid == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); fence_mbar_init(); }\n";
        src << "  __syncthreads();\n";
        src << "  auto issue = [&](long long tile, int s) {\n";
        src << "    const long long e0 = tile * GAAST_THREADS;\n";
        src << "    const long long left = a.n - e0;\n";
        src << "    const unsigned bytes = (unsigned)((left < GAAST_THREADS ? left : GAAST_THREADS) * 8);\n";
        src << "    double* const dst = stage0 + s * " << P << " * GAAST_THREADS;\n";
        src << "    fence_proxy_async();\n";
        src << "    mbar_expect_tx(&mbar[s], bytes * " << P << "u);\n";
        for (int r = 0; r < P; ++r)
            src << "    tma_row(dst + " << r << " * GAAST_THREADS, s" << parked[size_t(r)]->stream << " + "
                << parked[size_t(r)]->row << " * r" << parked[size_t(r)]->stream << " + e0, bytes, &mbar[s]);\n";
        for (const Node* n : in_regs)
            src << "    l2_prefetch_row(s" << n->stream << " + " << n->row << " * r" << n->stream << " + e0, bytes);\n";
        src << "  };\n";
        src << "  if (tid == 0) {\n";
        src << "    if ((long long)blockIdx.x < n_tiles) issue(blockIdx.x, 0);\n";
        src << "    if ((long long)blockIdx.x + gridDim.x < n_tiles) issue((long long)blockIdx.x + gridDim.x, 1);\n";
        src << "  }\n";
        src << "  int it = 0;\n";
        src << "  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {\n";
        src << loop_strides.str();
        src << "    const int s = it & 1;\n";
        src << "    const long long e_raw = tile * GAAST_THREADS + tid;\n";
        src << "    const bool active = e_raw < a.n;\n";
        src << "    const long long e = active ? e_raw : a.n - 1;  // idle lanes of the last tile shadow a valid element\n";
        src << "    const unsigned xb = (unsigned)__cvta_generic_to_shared(stage0 + s * " << P
            << " * GAAST_THREADS + (int)(e - tile * GAAST_THREADS));\n";
        src << "    mbar_wait(&mbar[s], (unsigned)(it >> 1) & 1u);\n";
        src << g.body.str();
        src << "    __syncthreads();  // every thread is done with buffer s: refill it for tile + 2 * gridDim\n";
        src << "    if (tid == 0) {\n";
        src << "      const long long nt = tile + 2LL * gridDim.x;\n";
        src << "      if (nt < n_tiles) issue(nt, s);\n";
        src << "    }\n";
        src << "  }\n";
    } else if (tmem_sum) {
        if (n_smem_rows)
            {
                if (opt.f32) src << "  const unsigned xb = (unsigned)__cvta_generic_to_shared(reinterpret_cast<float*>(sums + " << sum_doubles << ") + tid);\n";
                else src << "  const unsigned xb = (unsigned)__cvta_generic_to_shared(sums + " << sum_doubles << " + tid);\n";
            }
        src << "  const long long n_tiles = (a.n + GAAST_THREADS - 1) / GAAST_THREADS;\n";
        src << "  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {\n";
        src << loop_strides.str();
        src << "    const long long e0 = tile * GAAST_THREADS;\n";
        src << "    const bool active = e0 + tid < a.n;\n";
        src << "    const long long e = active ? e0 + tid : a.n - 1;  // idle lanes of the last tile shadow a valid element\n";
        if (!g.sum_stash) src << "    tm_wait_st();  // the previous tile's sum updates have landed in tensor memory\n";
        src << g.body.str();
        if (g.sum_stash) {
            // end of the tile: the running sums absorb the stash (registers are free here)
            src << "    tm_wait_st();  // stash and earlier sum updates have landed in tensor memory\n";
            for (int full = 1; full >= 0; --full) {
                src << (full ? "    if (e0 + GAAST_THREADS <= a.n) {\n" : "    } else {\n");
                size_t k = 0;
                auto batch = [&](size_t n, const char* fn) {
                    for (; k + n <= g.sum_stash; k += n)
                        src << "      " << fn << "<" << (full ? "true" : "false") << ">(tb + " << 2 * k << "u, tb + "
                            << 2 * root_cols + 2 * k << "u, active);\n";
                };
                batch(16, "tm_acc16");
                batch(4, "tm_acc4");
                batch(1, "tm_acc1");
            }
            src << "    }\n";
        }
        src << "  }\n";
    } else if (tma_stage) {
        // One tile per block.  Thread 0 hands the tile's parked rows to the TMA unit (one bulk
        // copy per row segment, completion on an mbarrier) before anything else; every thread
        // then issues the loads of its register rows and only waits for the TMA data afterwards.
        const int P = n_smem_rows;
        std::vector<const Node*> parked(size_t(P), nullptr);
        for (const Node& n : g.nodes)
            if (n.live && n.k == N_LOAD && !n.uniform && n.reload) parked[size_t(n.smem_row)] = &n;
        if (opt.f32) src << "  float* const stage0 = reinterpret_cast<float*>(sums + " << sum_doubles << ");\n";
        else src << "  double* const stage0 = sums + " << sum_doubles << ";\n";
        src << "  unsigned long long* const stage_bar = reinterpret_cast<unsigned long long*>(stage0 + " << P
            << " * GAAST_THREADS);\n";
        src << "  const long long e0 = (long long)blockIdx.x * GAAST_THREADS;\n";
        src << "  if (tid == 0) { mbar_init(stage_bar, 1); fence_mbar_init(); }\n";
        src << "  __syncthreads();\n";
        if (par_issue) {
            // (opt-in) the 32 lanes of warp 0 issue the row copies side by side -- lane l takes rows
            // l, l + 32, ... -- instead of thread 0 issuing all of them one after the other
            src << "  if (tid < 32 && e0 < a.n) {\n";
            src << "    const long long left = a.n - e0;\n";
            src << "    const unsigned bytes = (unsigned)((left < GAAST_THREADS ? left : GAAST_THREADS) * " << g.esize << ");\n";
            src << "    fence_proxy_async();\n";
            src << "    if (tid == 0) mbar_expect_tx(stage_bar, bytes * " << P << "u);\n";
            src << "    for (int r = tid; r < " << P << "; r += 32)\n";
            src << "      tma_row(stage0 + r * GAAST_THREADS, a.sptr[kStageStream[r]] + (long long)kStageRow[r] * "
                   "a.srow[kStageStream[r]] + e0, bytes, stage_bar);\n";
            src << "  }\n";
        } else {
        src << "  if (tid == 0 && e0 < a.n) {\n";
        src << "    const long long left = a.n - e0;\n";
        src << "    const unsigned bytes = (unsigned)((left < GAAST_THREADS ? left : GAAST_THREADS) * " << g.esize << ");\n";
        src << "    fence_proxy_async();\n";
        src << "    mbar_expect_tx(stage_bar, bytes * " << P << "u);\n";
        for (int r = 0; r < P; ++r)
            src << "    tma_row(stage0 + " << r << " * GAAST_THREADS, s" << parked[size_t(r)]->stream << " + "
                << parked[size_t(r)]->row << " * r" << parked[size_t(r)]->stream << " + e0, bytes, stage_bar);\n";
        src << "  }\n";
        }
        if (look_ahead) {
            // L2 look-ahead (opt-in): one lane of the second warp asks the L2 for the input rows of the
            // tile that will run `a.lookahead` blocks later -- the block that takes this one's place on the
            // SM -- so that its loads find their data on chip instead of paying an HBM round trip.
            if (par_issue) {
                size_t n_loads = 0;
                for (const Node& n : g.nodes) n_loads += n.live && n.k == N_LOAD && !n.uniform;
                src << "  if (tid >= 32 && tid < 64 && a.lookahead > 0) {\n";
                src << "    const long long pe0 = e0 + (long long)a.lookahead * GAAST_THREADS;\n";
                src << "    if (pe0 < a.n) {\n";
                src << "      const long long left = a.n - pe0;\n";
                src << "      const unsigned bytes = (unsigned)((left < GAAST_THREADS ? left : GAAST_THREADS) * " << g.esize << ");\n";
                src << "      for (int r = tid - 32; r < " << n_loads << "; r += 32)\n";
                src << "        l2_prefetch_row(a.sptr[kLoadStream[r]] + (long long)kLoadRow[r] * a.srow[kLoadStream[r]] + pe0, bytes);\n";
                src << "    }\n  }\n";
            } else {
            src << "  if (tid == 32 && a.lookahead > 0) {\n";
            src << "    const long long pe0 = e0 + (long long)a.lookahead * GAAST_THREADS;\n";
            src << "    if (pe0 < a.n) {\n";
            src << "      const long long left = a.n - pe0;\n";
            src << "      const unsigned bytes = (unsigned)((left < GAAST_THREADS ? left : GAAST_THREADS) * " << g.esize << ");\n";
            for (const Node& n : g.nodes)
                if (n.live && n.k == N_LOAD && !n.uniform)
                    src << "      l2_prefetch_row(s" << n.stream << " + " << n.row << " * r" << n.stream << " + pe0, bytes);\n";
            src << "    }\n  }\n";
            }
        }
        src << "  const unsigned xb = (unsigned)__cvta_generic_to_shared(stage0 + tid);\n";
        if (g.dense_tmem) {
            // whole warps run the tcgen05 instructions: lanes past the end of the batch shadow the
            // last element and do not store
            src << "  const int warp = tid >> 5;\n";
            src << "  unsigned* const tslot = reinterpret_cast<unsigned*>(stage_bar + 1);\n";
            src << "  if (warp == 0) { tm_alloc(tslot, 128u); tm_relinquish(); }\n";
            src << "  tm_fence_before_sync();\n  __syncthreads();\n  tm_fence_after_sync();\n";
            src << "  const unsigned tmem_base = *tslot;\n";
            src << "  const unsigned tb = tmem_base + ((unsigned)(warp * 32) << 16);\n";
            src << "  const bool active = e0 + tid < a.n;\n";
            src << "  const long long e = active ? e0 + tid : a.n - 1;\n";
            src << "  {\n";
            src << loop_strides.str();
            src << g.body.str();
            src << "  }\n";
            src << "  tm_fence_before_sync();\n  __syncthreads();\n";
            src << "  if (warp == 0) tm_dealloc(tmem_base, 128u);\n";
        } else {
            src << "  const long long e = e0 + tid;\n";
            src << "  if (e < a.n) {\n";
            src << loop_strides.str();
            src << g.body.str();
            src << "  }\n";
        }
    } else {
        if (n_smem_rows)
            {
                if (opt.f32) src << "  const unsigned xb = (unsigned)__cvta_generic_to_shared(reinterpret_cast<float*>(sums + " << sum_doubles << ") + tid);\n";
                else src << "  const unsigned xb = (unsigned)__cvta_generic_to_shared(sums + " << sum_doubles << " + tid);\n";
            }
        src << "  for (long long e = ((long long)blockIdx.x * GAAST_THREADS + tid) * GAAST_EPT; e < a.n;\n"
               "       e += (long long)gridDim.x * GAAST_THREADS * GAAST_EPT) {\n";
        src << loop_strides.str();
        src << g.body.str();
        src << "  }\n";
    }
    if (tmem_sum) {
        // per-lane sums -> warp (shuffle tree) -> block (fixed warp order) -> partials
        src << "  tm_wait_st();\n";
        src << "  for (int c = 0; c < " << root_cols << "; ++c) {\n";
        src << "    double v = tm_get(tb + 2u * c);\n";
        src << "    #pragma unroll\n";
        src << "    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);\n";
        src << "    if (lane == 0) sums[warp * " << root_cols << " + gaast_sum_col[c]] = v;\n";
        src << "  }\n";
        src << "  tm_fence_before_sync();\n";
        src << "  __syncthreads();\n";
        src << "  for (int c = tid; c < " << root_cols << "; c += GAAST_THREADS) {\n";
        src << "    double v = 0.0;\n";
        src << "    for (int w = 0; w < GAAST_THREADS / 32; ++w) v += sums[w * " << root_cols << " + c];\n";
        src << "    a.partials[(long long)blockIdx.x * " << root_cols << " + c] = v;\n";
        src << "  }\n";
        src << "  if (warp == 0) tm_dealloc(tmem_base, " << tmem_cols << "u);\n";
    } else if (opt.with_sum) {
        src << "  __syncthreads();\n";
        src << "  for (int c = tid; c < " << root_cols << "; c += GAAST_THREADS) {\n";
        src << "    double s = 0.0;\n";
        src << "    for (int t = 0; t < GAAST_THREADS; ++t) s += sums[c * GAAST_THREADS + t];\n";
        src << "    a.partials[(long long)blockIdx.x * " << root_cols << " + c] = s;\n";
        src << "  }\n";
    }
    src << "}\n";
    res.source = src.str();
    res.notes = notes.str();
    return res;
}

CodegenResult generate_kernel(const DevicePlanHost& h, const CodegenOptions& opt) {
    if (!h.projected) return generate(h, opt, false);
    // A projected plan: root liveness from the selected components drops every term that feeds only the others.  A
    // matrix-representation product needs all of its outputs, so it only survives in the kernel that keeps the whole
    // root live (and stores the selected components): that kernel is taken when it executes fewer FMAs.
    CodegenResult pruned = generate(h, opt, true);
    try {
        CodegenResult whole = generate(h, opt, false);
        if (whole.fma_per_elem < pruned.fma_per_elem) return whole;
    } catch (const Error&) {
    }
    return pruned;
}

}  // namespace gaast
