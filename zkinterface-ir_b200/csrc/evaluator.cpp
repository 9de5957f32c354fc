// zkb_evaluator — mirror of `Evaluator<B>` (rust/src/consumers/evaluator.rs:158-753) and of
// `Source` (rust/src/consumers/source.rs:45-193) over the recording GPU backend.
//
// The control flow of ingest_gate / ingest_subcircuit / compute_weight / exp is reproduced
// callback for callback (so the recorded program is op-for-op what the reference would ask of a
// ZKBackend), but nothing is evaluated here: assertions are resolved by the device and the
// reference's violation strings are rebuilt in get_violations from the first failing assertion.
#include <dirent.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <functional>
#include <atomic>
#include <chrono>
#include <deque>
#include <thread>
#include <unordered_map>

#include "context.h"
#include "file_bytes.h"
#include "ir.h"

using namespace zkb;

namespace {

struct Fatal {  // conditions on which the reference panics
    std::string msg;
};
struct EvalErr {  // Err(Box<dyn Error>) of the reference
    std::string msg;
};

struct FunctionDecl {  // evaluator.rs:130-136
    std::shared_ptr<std::vector<ir::Gate>> body;
    std::shared_ptr<std::vector<std::vector<uint8_t>>> consts;  // the message's constant table the body indexes
    uint64_t instance_nbr, witness_nbr, output_count, input_count;
    // A body made of plain gates only (no Free, Instance, Witness, no nested structure) that is well formed for a fresh
    // scope — every wire read was written before or is an input, nothing is written twice, every output is written —
    // behaves identically on every invocation: it is run over a flat array of local wires instead of a Scope
    // (n_local > 0).  Anything else goes through ingest_subcircuit, which reports errors where the reference does.
    uint32_t n_local = 0;
    // index of the body's Template in the Program (loop-structured recording, program.h), -1: not compiled yet, -2: the
    // body does not qualify
    mutable int tmpl = -1;
};

uint32_t simple_body_locals(const std::vector<ir::Gate>& body, uint64_t n_out, uint64_t n_in) {
    constexpr uint64_t kMaxLocal = 1u << 16;
    if (n_out + n_in >= kMaxLocal) return 0;
    uint64_t top = n_out + n_in;
    for (const auto& g : body) {
        switch (g.type) {
            case ir::G_CONSTANT: case ir::G_ASSERT_ZERO: case ir::G_COPY: case ir::G_ADD: case ir::G_MUL: case ir::G_ADD_CONSTANT:
            case ir::G_MUL_CONSTANT: case ir::G_AND: case ir::G_XOR: case ir::G_NOT: break;
            default: return 0;
        }
        if (g.w0 >= kMaxLocal || g.w1 >= kMaxLocal || g.w2 >= kMaxLocal) return 0;
        top = std::max(top, std::max(g.w0, std::max(g.w1, g.w2)) + 1);
    }
    std::vector<uint8_t> defined(top, 0);
    for (uint64_t w = n_out; w < n_out + n_in; w++) defined[w] = 1;
    for (const auto& g : body) {
        const bool two = g.type == ir::G_ADD || g.type == ir::G_MUL || g.type == ir::G_AND || g.type == ir::G_XOR;
        if (g.type == ir::G_ASSERT_ZERO) {
            if (!defined[g.w0]) return 0;
            continue;
        }
        if (g.type != ir::G_CONSTANT && !defined[g.w1]) return 0;
        if (two && !defined[g.w2]) return 0;
        if (defined[g.w0]) return 0;
        defined[g.w0] = 1;
    }
    for (uint64_t w = 0; w < n_out; w++)
        if (!defined[w]) return 0;
    return (uint32_t)std::max<uint64_t>(top, 1);
}

using Queue = std::deque<uint32_t>;  // positions in the instance / witness value streams
constexpr uint32_t kNoWitnessValue = 0xFFFFFFFFu;  // flatten mode: a Witness gate recorded without a value
using Iters = std::vector<std::pair<std::string, uint64_t>>;

std::string u64s(uint64_t v) { return std::to_string((unsigned long long)v); }

}  // namespace

static unsigned parse_threads();

struct zkb_evaluator {
    zkb_ctx* c;
    std::string err;

    // Evaluator state, evaluator.rs:158-170
    Scope values;
    std::vector<uint8_t> modulus_le;
    Queue instance_queue, witness_queue;
    std::vector<std::vector<uint8_t>> instance_values, witness_values;  // the streams themselves
    bool is_boolean = false;
    std::unordered_map<std::string, FunctionDecl> known_functions;
    bool verified_at_least_one_gate = false;
    bool has_error = false;
    std::string found_error;
    bool fatal = false;

    bool evaluated = false;
    std::vector<std::string> violations;
    std::vector<uint8_t> flat_out[3];  // flatten output (instance, witness, relation), owned here
    std::vector<Scope*> scope_pool;

    // ---- value sets (batch mode, zkb.h section 4) -------------------------------------------------------------------
    // Set j's statement is: the common instance values, set j's; the common witness values, set j's; the relation.  The
    // relation is recorded once, against the longest streams: stream positions past the common values stand for the sets'
    // values.  Values of all sets are kept packed, trimmed of trailing zero bytes, one arena per stream.
    struct Arena {
        std::vector<uint8_t> bytes;
        std::vector<uint64_t> end{0};  // value k is bytes[end[k], end[k + 1])
        size_t widest = 0;
        uint64_t size() const { return end.size() - 1; }
        void push(const std::vector<uint8_t>& v) {
            size_t n = v.size();
            while (n > 0 && v[n - 1] == 0) n--;
            bytes.insert(bytes.end(), v.data(), v.data() + n);
            end.push_back(bytes.size());
            widest = std::max(widest, n);
        }
    };
    struct ValueSet {
        uint64_t inst0, n_inst, wit0, n_wit;  // ranges in the arenas
    };
    Arena set_inst, set_wit;
    std::vector<ValueSet> sets;
    uint64_t max_set_inst = 0, max_set_wit = 0;
    bool relation_seen = false;
    uint32_t n_common_inst = 0, n_common_wit = 0;  // stream positions of the common values, fixed at the first relation
    // the first recording error or panic in batch mode (it ends the recording, as in a single statement): value handles
    // recorded before it, its text, and whether it is a panic
    uint32_t global_cut = UINT32_MAX;
    std::string global_cut_msg;
    bool global_cut_fatal = false;
    std::vector<zkb_ctx*> devices;  // zkb_evaluator_use_devices: the batch is split over these contexts
    bool batch_evaluated = false, batch_sharded = false;
    std::vector<int> set_status;
    std::vector<std::vector<std::string>> set_violations;
    std::vector<uint32_t> set_cut;  // value handles recorded before each set's cut (UINT32_MAX: none)

    bool batch() const { return !sets.empty(); }

    explicit zkb_evaluator(zkb_ctx* ctx) : c(ctx) {}
    ~zkb_evaluator() {
        for (auto s : scope_pool) delete s;
    }

    Program& prog() { return c->prog; }

    static constexpr uint64_t kMaxDepth = 512;  // nested ingest_subcircuit calls (Call / AnonCall / For / Switch bodies)
    uint64_t depth = 0;

    // work accounting against zkb_set_limits (not in the reference, which would run until memory is exhausted)
    uint64_t steps = 0;
    void step(uint64_t n = 1) {
        steps += n;
        if (steps > c->max_steps || steps < n) throw EvalErr{"zkb: resource limit exceeded (max_steps)"};
    }

    Scope* new_scope() {
        if (scope_pool.empty()) {
            Scope* s = new Scope();
            s->track = true;
            return s;
        }
        Scope* s = scope_pool.back();
        scope_pool.pop_back();
        return s;
    }
    void release_scope(Scope* s) {
        s->clear();
        scope_pool.push_back(s);
    }

    // ---- scope helpers, evaluator.rs:775-797 -------------------------------------------------
    static uint32_t get(const Scope& sc, uint64_t id) {
        uint32_t v = sc.get(id);
        if (v == Scope::kNone) throw EvalErr{"No value given for wire_" + u64s(id)};
        return v;
    }
    static void set(Scope& sc, uint64_t id, uint32_t v) {
        if (!sc.set(id, v)) throw EvalErr{"Wire_" + u64s(id) + " already has a value in this scope."};
    }
    static void remove(Scope& sc, uint64_t id) {
        if (!sc.remove(id)) throw EvalErr{"No value given for wire_" + u64s(id)};
    }

    // ---- structs/wire.rs:179-203 ---------------------------------------------------------------
    void expand_wirelist(const ir::WireList& wl, std::vector<uint64_t>& out) {
        out.clear();
        for (const auto& e : wl) {
            if (!e.is_range) {
                out.push_back(e.first);
            } else {
                if (e.last <= e.first)
                    throw EvalErr{"In WireRange, last WireId (" + u64s(e.last) + ") must be strictly greater than first WireId (" +
                                  u64s(e.first) + ")."};
                if (e.last - e.first > (1ull << 32)) throw EvalErr{"zkb: wire range too large"};
                step(e.last - e.first);
                for (uint64_t w = e.first; w <= e.last; w++) out.push_back(w);
            }
        }
    }

    // ---- structs/iterators.rs:349-403 ----------------------------------------------------------
    // affine form of an expression, or false (a DivConst, or a product of two iterator-dependent sides, inside)
    static bool affine_of(const ir::IterExpr& e, ir::AffineIterExpr& out) {
        auto add_term = [](ir::AffineIterExpr& f, const std::string& name, uint64_t coef) {
            for (auto& t : f.terms)
                if (t.first == name) {
                    t.second += coef;
                    return;
                }
            f.terms.push_back({name, coef});
        };
        switch (e.type) {
            case 1: out.c0 = e.value; return true;
            case 2: out.terms.push_back({e.name, 1}); return true;
            case 3: case 4: case 5: {
                ir::AffineIterExpr a, b;
                if (!affine_of(*e.l, a) || !affine_of(*e.r, b)) return false;
                if (e.type == 5) {
                    if (!a.terms.empty() && !b.terms.empty()) return false;
                    const ir::AffineIterExpr& k = a.terms.empty() ? a : b;   // the constant side
                    const ir::AffineIterExpr& x = a.terms.empty() ? b : a;
                    out.c0 = k.c0 * x.c0;
                    for (const auto& t : x.terms) out.terms.push_back({t.first, t.second * k.c0});
                    return true;
                }
                out = a;
                if (e.type == 3) out.c0 += b.c0;
                else out.c0 -= b.c0;
                for (const auto& t : b.terms) add_term(out, t.first, e.type == 3 ? t.second : (uint64_t)0 - t.second);
                return true;
            }
            default: return false;
        }
    }
    static uint64_t lookup_iter(const std::string& name, const Iters& known) {
        for (size_t i = known.size(); i-- > 0;)
            if (known[i].first == name) return known[i].second;
        // evaluate_iterexpr_list unwraps the Err: a panic in the reference (iterators.rs:400)
        throw Fatal{"Unknown iterator name " + name};
    }
    static uint64_t eval_iterexpr(const ir::IterExpr& e, const Iters& known) {
        if (!e.affine_tried) {
            e.affine_tried = true;
            if (e.type >= 3) {  // constants and names are already one step
                auto f = std::make_shared<ir::AffineIterExpr>();
                if (affine_of(e, *f)) e.affine = f;
            }
        }
        if (e.affine) {
            uint64_t v = e.affine->c0;
            for (const auto& t : e.affine->terms) v += t.second * lookup_iter(t.first, known);
            return v;
        }
        switch (e.type) {
            case 1: return e.value;
            case 2: return lookup_iter(e.name, known);
            case 3: return eval_iterexpr(*e.l, known) + eval_iterexpr(*e.r, known);  // release build: wrapping
            case 4: return eval_iterexpr(*e.l, known) - eval_iterexpr(*e.r, known);
            case 5: return eval_iterexpr(*e.l, known) * eval_iterexpr(*e.r, known);
            case 6:
                if (e.value == 0) throw Fatal{"attempt to divide by zero"};
                return eval_iterexpr(*e.l, known) / e.value;
        }
        throw Fatal{"Unknown Iterator Expression type"};
    }
    void eval_iterexpr_list(const ir::IterExprList& l, const Iters& known, std::vector<uint64_t>& out) {
        out.clear();
        for (const auto& el : l) {
            uint64_t a = eval_iterexpr(el.first, known);
            if (!el.is_range) {
                out.push_back(a);
            } else {
                uint64_t b = eval_iterexpr(el.last, known);
                if (b >= a && b - a > (1ull << 32)) throw EvalErr{"zkb: iterator range too large"};
                if (b < a) continue;
                step(b - a);
                const size_t o = out.size();
                out.resize(o + (size_t)(b - a) + 1);
                uint64_t* dst = out.data() + o;
                for (uint64_t k = 0; k <= b - a; k++) dst[k] = a + k;
            }
        }
    }
    static void iters_set(Iters& k, const std::string& name, uint64_t v) {  // HashMap::insert
        for (auto& kv : k)
            if (kv.first == name) {
                kv.second = v;
                return;
            }
        k.push_back({name, v});
    }
    static void iters_remove(Iters& k, const std::string& name) {
        for (size_t i = 0; i < k.size(); i++)
            if (k[i].first == name) {
                k.erase(k.begin() + i);
                return;
            }
    }

    // ---- evaluator.rs:78-126 -------------------------------------------------------------------
    uint32_t as_mul(uint32_t a, uint32_t b) { return is_boolean ? prog().and_(a, b) : prog().multiply(a, b); }
    uint32_t as_add(uint32_t a, uint32_t b) { return is_boolean ? prog().xor_(a, b) : prog().add(a, b); }
    uint32_t as_negate(uint32_t w) {
        if (is_boolean) return prog().copy(w);
        std::vector<uint8_t> m1 = prog().minus_one_le();
        return prog().mul_constant(w, m1.data(), m1.size());
    }
    uint32_t as_add_one(uint32_t w) {
        if (is_boolean) return prog().not_(w);
        uint8_t one = 1;
        return prog().add_constant(w, &one, 1);
    }
    // evaluator.rs:801-820: recursive square-and-multiply, MSB -> LSB; the recursion bottoms out in
    // copy(base) at exponent 1 and then, per lower bit, squares and (bit set) multiplies by base.
    uint32_t exp(uint32_t base, const BigU& exponent) {
        size_t nb = exponent.bits();
        uint32_t acc = prog().copy(base);
        for (size_t i = nb - 1; i-- > 0;) {
            acc = as_mul(acc, acc);
            if (exponent.bit(i)) acc = as_mul(acc, base);
        }
        return acc;
    }
    // evaluator.rs:823-839
    uint32_t compute_weight(const std::vector<uint8_t>& case_val, uint32_t condition) {
        uint32_t case_wire = prog().constant(case_val.data(), case_val.size());
        BigU exponent = BigU::from_bytes_le(modulus_le.data(), modulus_le.size());
        exponent.sub(BigU(1));
        uint32_t minus_cond = as_negate(condition);
        uint32_t base = as_add(case_wire, minus_cond);
        uint32_t base_to_exp = exp(base, exponent);
        uint32_t right = as_negate(base_to_exp);
        return as_add_one(right);
    }

    void check_arity(const std::string& name, const FunctionDecl& f, size_t n_out, size_t n_in) {  // :449-454
        if (n_out != f.output_count)
            throw EvalErr{"Wrong number of output variables in call to function " + name + " (Expected " + u64s(f.output_count) +
                          " / Got " + u64s(n_out) + ")."};
        if (n_in != f.input_count)
            throw EvalErr{"Wrong number of input variables in call to function " + name + " (Expected " + u64s(f.input_count) +
                          " / Got " + u64s(n_in) + ")."};
    }

    // ingest_subcircuit for a FunctionDecl with n_local > 0: same callbacks in the same order (a copy per input, the
    // gates, a copy per output: evaluator.rs:698-746 with the simple arms of :344-418 inlined), local wires in an array
    std::vector<uint32_t> locals;
    void ingest_simple_function(const FunctionDecl& f, const std::vector<uint64_t>& outs, const std::vector<uint64_t>& ins, Scope& scope,
                                const uint32_t* weight) {
        Program& p = prog();
        if (locals.size() < f.n_local) locals.resize(f.n_local);
        uint32_t* L = locals.data();
        const size_t n_out = outs.size();
        for (size_t idx = 0; idx < ins.size(); idx++) L[n_out + idx] = p.copy(get(scope, ins[idx]));
        const auto& consts = *f.consts;
        for (const ir::Gate& g : *f.body) {
            if (p.n_total_values() >= c->max_values) throw EvalErr{"zkb: resource limit exceeded (max_values)"};
            step();
            switch (g.type) {
                case ir::G_CONSTANT: {
                    const auto& v = consts[g.const_idx];
                    L[g.w0] = p.constant(v.data(), v.size());
                } break;
                case ir::G_ASSERT_ZERO: {
                    uint32_t z = weight ? as_mul(*weight, L[g.w0]) : p.copy(L[g.w0]);
                    p.assert_zero(z, g.w0);
                    p.ir_gates++;
                } break;
                case ir::G_COPY: L[g.w0] = p.copy(L[g.w1]); break;
                case ir::G_ADD: L[g.w0] = p.add(L[g.w1], L[g.w2]); p.ir_gates++; break;
                case ir::G_MUL: L[g.w0] = p.multiply(L[g.w1], L[g.w2]); p.ir_gates++; break;
                case ir::G_AND: L[g.w0] = p.and_(L[g.w1], L[g.w2]); p.ir_gates++; break;
                case ir::G_XOR: L[g.w0] = p.xor_(L[g.w1], L[g.w2]); p.ir_gates++; break;
                case ir::G_ADD_CONSTANT: {
                    const auto& v = consts[g.const_idx];
                    L[g.w0] = p.add_constant(L[g.w1], v.data(), v.size());
                    p.ir_gates++;
                } break;
                case ir::G_MUL_CONSTANT: {
                    const auto& v = consts[g.const_idx];
                    L[g.w0] = p.mul_constant(L[g.w1], v.data(), v.size());
                    p.ir_gates++;
                } break;
                default: L[g.w0] = p.not_(L[g.w1]); p.ir_gates++; break;  // G_NOT
            }
        }
        for (size_t idx = 0; idx < n_out; idx++) set(scope, outs[idx], p.copy(L[idx]));
    }
    // ---- loop-structured recording: a For loop over a plain function becomes ONE call group (program.h) -----------------
    // Over p = 2 the body qualifies when every gate is a value-defining simple gate the device interpreter runs on reduced values:
    // no AssertZero, no Copy (an output that aliases a raw
    // input would carry its unreduced integer on), and no Not directly on a call input (Not tests the RAW integer of an
    // input value, evaluator.rs:932-938; And / Xor / Add / Mul only see the low bit mod 2).  Prime fields: arith_template_of.
    int template_of(const FunctionDecl& f) {
        if (f.tmpl != -1) return f.tmpl;
        f.tmpl = -2;
        Program& p = prog();
        if (!p.binary) return f.tmpl = arith_template_of(f);
        if (!f.n_local || f.n_local > kMaxTemplateRegs || f.body->size() > kMaxTemplateOps || f.input_count > kMaxGroupInputs ||
            f.output_count == 0)
            return f.tmpl;
        Template t;
        t.n_out = (uint32_t)f.output_count;
        t.n_in = (uint32_t)f.input_count;
        t.n_regs = f.n_local;
        auto is_input = [&](uint64_t w) { return w >= f.output_count && w < f.output_count + f.input_count; };
        for (const ir::Gate& g : *f.body) {
            TmplOp o{};
            o.dst = (uint8_t)g.w0;
            o.a = (uint8_t)g.w1;
            o.b = (uint32_t)g.w2;
            switch (g.type) {
                case ir::G_CONSTANT: {
                    const auto& v = (*f.consts)[g.const_idx];
                    o.kind = V_CONST;
                    o.a = 0;
                    o.b = p.intern_const(v.data(), v.size());
                    if (p.const_unreduced[o.b]) return f.tmpl;  // a constant >= p stays a raw integer (trap 1)
                    t.cb[CB_CONSTANT]++;
                } break;
                case ir::G_ADD: o.kind = V_ADD; t.cb[CB_ADD]++; t.n_two++; break;
                case ir::G_MUL: o.kind = V_MUL; t.cb[CB_MUL]++; t.n_two++; break;
                case ir::G_AND: o.kind = V_AND; t.cb[CB_AND]++; t.n_two++; break;
                case ir::G_XOR: o.kind = V_XOR; t.cb[CB_XOR]++; t.n_two++; break;
                case ir::G_ADD_CONSTANT: case ir::G_MUL_CONSTANT: {
                    const auto& v = (*f.consts)[g.const_idx];
                    o.kind = g.type == ir::G_ADD_CONSTANT ? V_ADDC : V_MULC;
                    o.b = p.intern_const(v.data(), v.size());
                    t.cb[g.type == ir::G_ADD_CONSTANT ? CB_ADDC : CB_MULC]++;
                    t.n_one++;
                } break;
                case ir::G_NOT:
                    if (is_input(g.w1)) return f.tmpl;
                    o.kind = V_NOT;
                    o.b = 0;
                    t.cb[CB_NOT]++;
                    t.n_one++;
                    break;
                default: return f.tmpl;  // AssertZero, Copy
            }
            if (g.type != ir::G_CONSTANT) t.ir_gates++;
            t.ops.push_back(o);
        }
        t.cb[CB_COPY] = f.input_count + f.output_count;
        p.templates.push_back(std::move(t));
        f.tmpl = (int)p.templates.size() - 1;
        return f.tmpl;
    }

    // Prime fields: Constant (< p), Add, Mul, AddConstant, MulConstant, and AssertZero on a register the body computed.  And /
    // Xor / Not / Copy act on raw integers (evaluator.rs:924-938; a copy of an input would carry its unreduced integer on) and
    // an AssertZero on an input tests the raw integer (trap 1): such bodies run gate by gate.  Registers are renamed by
    // liveness in one linear scan (outputs pinned to 0 .. n_out-1, inputs start at n_out), so the device register file holds
    // the values live at once rather than every wire of the body.
    int arith_template_of(const FunctionDecl& f) {
        Program& p = prog();
        const uint64_t n_out = f.output_count, n_in = f.input_count;
        if (!f.n_local || f.body->size() > kMaxTemplateOps || n_in > kMaxGroupInputs || n_out == 0 || n_out + n_in > kMaxTemplateRegs)
            return -2;
        auto is_input = [&](uint64_t w) { return w >= n_out && w < n_out + n_in; };
        std::vector<int32_t> last(f.n_local, -1);  // index of the last gate reading each wire
        for (size_t i = 0; i < f.body->size(); i++) {
            const ir::Gate& g = (*f.body)[i];
            switch (g.type) {
                case ir::G_CONSTANT: break;
                case ir::G_ASSERT_ZERO:
                    if (is_input(g.w0)) return -2;
                    last[g.w0] = (int32_t)i;
                    break;
                case ir::G_ADD: case ir::G_MUL: last[g.w1] = last[g.w2] = (int32_t)i; break;
                case ir::G_ADD_CONSTANT: case ir::G_MUL_CONSTANT: last[g.w1] = (int32_t)i; break;
                default: return -2;  // And, Xor, Not, Copy
            }
        }
        Template t;
        t.n_out = (uint32_t)n_out;
        t.n_in = (uint32_t)n_in;
        std::vector<int32_t> reg(f.n_local, -1);
        for (uint64_t w = n_out; w < n_out + n_in; w++) reg[w] = (int32_t)w;
        std::vector<uint32_t> free_regs;  // kept in descending order: back() is the lowest free register
        uint32_t n_regs = (uint32_t)(n_out + n_in);
        auto release = [&](uint64_t w, size_t i) {
            if (w >= n_out && last[w] <= (int32_t)i && reg[w] >= 0) {
                free_regs.insert(std::upper_bound(free_regs.begin(), free_regs.end(), (uint32_t)reg[w], std::greater<uint32_t>()),
                                 (uint32_t)reg[w]);
                reg[w] = -1;
            }
        };
        for (size_t i = 0; i < f.body->size(); i++) {
            const ir::Gate& g = (*f.body)[i];
            TmplOp o{};
            switch (g.type) {
                case ir::G_CONSTANT: {
                    const auto& v = (*f.consts)[g.const_idx];
                    o.kind = V_CONST;
                    o.b = p.intern_const(v.data(), v.size());
                    if (p.const_unreduced[o.b]) return -2;  // a constant >= p stays a raw integer (trap 1)
                    t.cb[CB_CONSTANT]++;
                } break;
                case ir::G_ADD: case ir::G_MUL:
                    o.kind = g.type == ir::G_ADD ? V_ADD : V_MUL;
                    o.a = (uint8_t)reg[g.w1];
                    o.b = (uint32_t)reg[g.w2];
                    t.cb[g.type == ir::G_ADD ? CB_ADD : CB_MUL]++;
                    t.n_two++;
                    break;
                case ir::G_ADD_CONSTANT: case ir::G_MUL_CONSTANT: {  // reduced result: a constant >= p is fine here
                    const auto& v = (*f.consts)[g.const_idx];
                    o.kind = g.type == ir::G_ADD_CONSTANT ? V_ADDC : V_MULC;
                    o.a = (uint8_t)reg[g.w1];
                    o.b = p.intern_const(v.data(), v.size());
                    t.cb[g.type == ir::G_ADD_CONSTANT ? CB_ADDC : CB_MULC]++;
                    t.n_one++;
                } break;
                default:  // G_ASSERT_ZERO (the unrolled loop asserts a copy of the wire: one Copy callback each)
                    o.kind = T_ASSERT;
                    o.a = (uint8_t)reg[g.w0];
                    o.b = (uint32_t)t.assert_wire.size();
                    t.assert_wire.push_back(g.w0);
                    t.cb[CB_ASSERT_ZERO]++;
                    t.cb[CB_COPY]++;
                    break;
            }
            if (g.type != ir::G_CONSTANT) t.ir_gates++;
            if (g.type == ir::G_ASSERT_ZERO) {
                release(g.w0, i);
            } else {
                if (g.type != ir::G_CONSTANT) release(g.w1, i);
                if (g.type == ir::G_ADD || g.type == ir::G_MUL) release(g.w2, i);
                uint32_t r;
                if (g.w0 < n_out) {
                    r = (uint32_t)g.w0;
                } else if (!free_regs.empty()) {
                    r = free_regs.back();
                    free_regs.pop_back();
                } else {
                    r = n_regs++;
                }
                if (n_regs > kMaxTemplateRegs) return -2;
                reg[g.w0] = (int32_t)r;
                o.dst = (uint8_t)r;
                release(g.w0, i);  // a value nothing reads: its register is free again at once
            }
            t.ops.push_back(o);
        }
        t.n_regs = n_regs;
        t.cb[CB_COPY] += n_in + n_out;
        p.templates.push_back(std::move(t));
        return (int)p.templates.size() - 1;
    }

    struct AffineWire {
        uint64_t w0, stride;
    };
    // wires of an iterator-expression list at loop value i0, with their step per loop iteration; false: not affine
    bool affine_wires(const ir::IterExprList& l, Iters& iters, const std::string& var, uint64_t i0, std::vector<AffineWire>& out) {
        out.clear();
        iters_set(iters, var, i0);
        // value v0 at loop index i0 and step st per iteration (wrapping arithmetic, as the reference's release build); false
        // when the expression is not linear in the loop variable (a product of two dependent sides, a DivConst of one)
        std::function<bool(const ir::IterExpr&, uint64_t&, uint64_t&)> form = [&](const ir::IterExpr& e, uint64_t& v0, uint64_t& st) {
            switch (e.type) {
                case 1: v0 = e.value; st = 0; return true;
                case 2: v0 = lookup_iter(e.name, iters); st = e.name == var ? 1 : 0; return true;
                case 3: case 4: case 5: {
                    uint64_t a0, sa, b0, sb;
                    if (!form(*e.l, a0, sa) || !form(*e.r, b0, sb)) return false;
                    if (e.type == 3) { v0 = a0 + b0; st = sa + sb; }
                    else if (e.type == 4) { v0 = a0 - b0; st = sa - sb; }
                    else {
                        if (sa != 0 && sb != 0) return false;
                        v0 = a0 * b0;
                        st = sa * b0 + sb * a0;
                    }
                    return true;
                }
                case 6: {
                    uint64_t a0, sa;
                    if (e.value == 0 || !form(*e.l, a0, sa) || sa != 0) return false;
                    v0 = a0 / e.value;
                    st = 0;
                    return true;
                }
            }
            return false;
        };
        for (const auto& el : l) {
            uint64_t a, sa;
            if (!form(el.first, a, sa)) return false;
            if (!el.is_range) {
                out.push_back({a, sa});
                continue;
            }
            uint64_t b, sb;
            if (!form(el.last, b, sb) || sa != sb) return false;
            if (b < a) continue;
            if (b - a > 4096) return false;
            for (uint64_t w = a;; w++) {
                out.push_back({w, sa});
                if (w == b) break;
            }
        }
        return true;
    }

    // true: the whole loop has been recorded as one call group, with the state the gate-by-gate loop would leave (bindings,
    // callback counts, work accounting).  false: nothing was changed; the caller runs the loop gate by gate, which also
    // reports every error where the reference does.
    bool try_call_group(const ir::Complex& cx, const FunctionDecl& f, Scope& scope, Iters& iters, const uint32_t* weight) {
        Program& p = prog();
        if (getenv("ZKB_NO_CALL_GROUPS") != nullptr || weight || p.keep_copies || p.expand_on || !p.field_set) return false;
        if (cx.last < cx.first || cx.last - cx.first < 3 || cx.last - cx.first >= (1ull << 28)) return false;
        if (!p.binary && cx.last - cx.first + 1 < kArithGroupMinCalls) return false;
        const int ti = template_of(f);
        if (ti < 0) return false;
        const uint64_t n = cx.last - cx.first + 1;
        std::vector<AffineWire> wo, wi;
        Iters saved = iters;
        bool ok = false;
        try {
            ok = affine_wires(cx.it_outputs, iters, cx.name, cx.first, wo) && affine_wires(cx.it_inputs, iters, cx.name, cx.first, wi);
        } catch (const Fatal&) {
        } catch (const EvalErr&) {
        }
        iters = saved;
        const Template& t = p.templates[ti];
        if (!ok || wo.size() != t.n_out || wi.size() != t.n_in) return false;
        // outputs: every call writes its own block of unbound wires
        const uint64_t S = wo[0].stride;
        uint64_t lo = wo[0].w0, hi = wo[0].w0;
        for (const auto& a : wo) {
            if (a.stride != S) return false;
            lo = std::min(lo, a.w0);
            hi = std::max(hi, a.w0);
        }
        if (S == 0 || S >= (1ull << 32) || hi - lo >= S || hi >= (1ull << 40)) return false;
        for (size_t a = 0; a < wo.size(); a++)
            for (size_t b = a + 1; b < wo.size(); b++)
                if (wo[a].w0 == wo[b].w0) return false;
        const uint64_t n_new = n * t.n_out;
        const uint64_t out_last = hi + S * (n - 1);
        const bool plain_scope = scope.sparse.empty();  // every binding is in the dense table: it can be walked directly
        {
            const uint32_t* d = scope.dense.data();
            const uint64_t dn = scope.dense.size();
            if (plain_scope && out_last < dn) {  // branch-free walks: the loops pipeline
                uint32_t all = Scope::kNone;
                for (const auto& a : wo)
                    for (uint64_t c = 0, w = a.w0; c < n; c++, w += S) all &= d[w];
                if (all != Scope::kNone) return false;
            } else {
                for (const auto& a : wo)
                    for (uint64_t c = 0, w = a.w0; c < n; c++, w += S)
                        if (plain_scope ? (w < dn && d[w] != Scope::kNone) : scope.get(w) != Scope::kNone) return false;
            }
        }
        // inputs: bound before the loop, level-0 values (inputs or outputs of earlier groups), handles in arithmetic progression
        CallGroup cg;
        cg.tmpl = (uint32_t)ti;
        cg.n_calls = (uint32_t)n;
        cg.n_out = t.n_out;
        cg.depth = 0;
        for (const auto& a : wi) {
            if (a.w0 >= (1ull << 40) || (a.stride >= (1ull << 32) && a.stride != 0)) return false;
            const uint32_t h0 = scope.get(a.w0);
            if (h0 == Scope::kNone) return false;
            uint32_t st = 0, h_last = h0;
            if (a.stride != 0) {
                const uint32_t h1 = scope.get(a.w0 + a.stride);
                if (h1 == Scope::kNone || h1 <= h0) return false;
                st = h1 - h0;
                if ((uint64_t)h0 + (uint64_t)st * (n - 1) >= 0xFFFFFFFFull) return false;
                h_last = h0 + st * (uint32_t)(n - 1);
                if (is_callout(h0) != is_callout(h_last)) return false;
                const uint32_t* d = scope.dense.data();
                const uint64_t dn = scope.dense.size();
                uint32_t expect = h0;
                if (plain_scope && a.w0 + a.stride * (n - 1) < dn) {
                    uint32_t diff = 0;
                    for (uint64_t c = 0, w = a.w0; c < n; c++, w += a.stride, expect += st) diff |= d[w] ^ expect;
                    if (diff) return false;
                } else {
                    for (uint64_t c = 0, w = a.w0; c < n; c++, w += a.stride, expect += st) {
                        const uint32_t h = plain_scope ? (w < dn ? d[w] : Scope::kNone) : scope.get(w);
                        if (h != expect) return false;
                    }
                }
            }
            if (is_callout(h0)) {  // outputs of the groups first .. last touched
                const CallGroup* g0 = &p.group_of_callout(callout_index(h0));
                const CallGroup* g1 = &p.group_of_callout(callout_index(h_last));
                for (const CallGroup* g = g0; g <= g1; g++) cg.depth = std::max(cg.depth, g->depth + 1);
            } else {
                const uint8_t* kind = p.kind.data();
                uint8_t worst = kind[h0];
                if (st != 0)
                    for (uint64_t c = 0, h = h0; c < n; c++, h += st) worst = std::max(worst, kind[h]);
                if (worst > V_WITNESS) return false;
            }
            cg.in_base.push_back(h0);
            cg.in_stride.push_back(st);
        }
        if (p.n_total_values() + n_new >= c->max_values || (uint64_t)p.n_callouts + n_new >= kMaxCallouts) return false;  // the gate-by-gate loop reports the limit
        const uint64_t n_group_asserts = n * t.assert_wire.size();
        if ((uint64_t)p.asserts.size() + n_group_asserts >= kNoSeq) return false;
        step(n * (1 + f.body->size()));
        // ---- commit: the outputs are implicit values (program.h), only the scope learns about them
        c->max_values = std::min<uint64_t>(c->max_values, kCalloutBit - 256);  // explicit handles stay below the callout space
        cg.first_callout = p.n_callouts;
        const uint32_t h_first = kCalloutBit | cg.first_callout;
        if (plain_scope && scope.ensure_dense(out_last, n_new)) {
            uint32_t* d = scope.dense.data();
            for (uint32_t k = 0; k < t.n_out; k++) {
                uint32_t h = h_first + k;
                for (uint64_t c = 0, w = wo[k].w0; c < n; c++, w += S, h += t.n_out) d[w] = h;
            }
            scope.bulk_inserted(n_new);
        } else {
            for (uint64_t c = 0; c < n; c++)
                for (uint32_t k = 0; k < t.n_out; k++) set(scope, wo[k].w0 + S * c, h_first + (uint32_t)(c * t.n_out + k));
        }
        p.n_callouts += (uint32_t)n_new;
        // the calls' assertions, in the unrolled loop's order: call c's k-th is seq0 + c * A + k
        cg.seq0 = (uint32_t)p.asserts.size();
        if (n_group_asserts) {
            std::vector<AssertRec> call(t.assert_wire.size());
            for (size_t k = 0; k < call.size(); k++) call[k] = AssertRec{kGroupAssertValue, p.n_values(), t.assert_wire[k]};
            p.asserts.reserve(p.asserts.size() + n_group_asserts);
            for (uint64_t c = 0; c < n; c++) p.asserts.insert(p.asserts.end(), call.begin(), call.end());
        }
        for (int k = 0; k < CB_KINDS; k++) p.cb_count[k] += n * t.cb[k];
        p.ir_gates += n * t.ir_gates;
        p.groups.push_back(std::move(cg));
        return true;
    }

    void call_function(const FunctionDecl& f, const std::vector<uint64_t>& outs, const std::vector<uint64_t>& ins, Scope& scope,
                       Iters& fresh, Queue& instances, Queue& witnesses, const uint32_t* weight) {
        if (f.n_local) ingest_simple_function(f, outs, ins, scope, weight);
        else ingest_subcircuit(*f.body, *f.consts, outs, ins, scope, fresh, instances, witnesses, weight);
    }

    // ---- evaluator.rs:698-746 --------------------------------------------------------------------
    void ingest_subcircuit(const std::vector<ir::Gate>& sub, const std::vector<std::vector<uint8_t>>& consts,
                           const std::vector<uint64_t>& outs, const std::vector<uint64_t>& ins, Scope& scope, Iters& iters,
                           Queue& instances, Queue& witnesses, const uint32_t* weight) {
        // Function bodies may call themselves (directly or through each other): the reference recurses until its stack
        // overflows.  The reader caps syntactic nesting at 512; the same bound on dynamic nesting turns that abort into
        // a latched evaluation error.
        if (depth >= kMaxDepth) throw EvalErr{"zkb: calls nested too deep (limit " + u64s(kMaxDepth) + ")"};
        Scope* ns = new_scope();
        depth++;
        try {
            // Long input / output lists (a loop body handed a whole block of wires) are moved table to table; whatever the
            // fast loops cannot take — an unbound input, an output that is already bound, ids outside the dense tables —
            // is left to the one-by-one code below, which reports it as the reference does.
            Program& p = prog();
            const size_t n_in = ins.size(), n_out = outs.size();
            size_t idx = 0;
            if (n_in >= 32 && !p.keep_copies && scope.sparse.empty() && ns->ensure_dense(n_out + n_in - 1, n_in)) {
                const uint32_t* src = scope.dense.data();
                const uint64_t sn = scope.dense.size();
                uint32_t* dst = ns->dense.data() + n_out;  // a fresh scope: nothing is bound
                for (; idx < n_in; idx++) {
                    const uint64_t id = ins[idx];
                    if (id >= sn || src[id] == Scope::kNone) break;
                    dst[idx] = src[id];
                }
                p.cb_count[CB_COPY] += idx;
                ns->bulk_inserted(idx);
            }
            for (; idx < n_in; idx++) set(*ns, idx + n_out, p.copy(get(scope, ins[idx])));
            for (const auto& g : sub) ingest_gate(g, consts, *ns, iters, instances, witnesses, weight);
            idx = 0;
            if (n_out >= 32 && !p.keep_copies && scope.sparse.empty() && ns->sparse.empty() && n_out <= ns->dense.size()) {
                uint64_t hi = 0;
                for (size_t k = 0; k < n_out; k++) hi = std::max(hi, outs[k]);
                if (scope.ensure_dense(hi, n_out)) {
                    const uint32_t* src = ns->dense.data();
                    uint32_t* dst = scope.dense.data();
                    for (; idx < n_out; idx++) {
                        const uint64_t id = outs[idx];
                        if (src[idx] == Scope::kNone || dst[id] != Scope::kNone) break;
                        dst[id] = src[idx];
                    }
                    p.cb_count[CB_COPY] += idx;
                    scope.bulk_inserted(idx);
                }
            }
            for (; idx < n_out; idx++) set(scope, outs[idx], p.copy(get(*ns, idx)));
        } catch (...) {
            depth--;
            release_scope(ns);
            throw;
        }
        depth--;
        release_scope(ns);
    }

    // ---- evaluator.rs:318-691 --------------------------------------------------------------------
    void ingest_gate(const ir::Gate& g, const std::vector<std::vector<uint8_t>>& consts, Scope& scope, Iters& iters,
                     Queue& instances, Queue& witnesses, const uint32_t* weight) {
        Program& p = prog();
        if (p.n_total_values() >= c->max_values) throw EvalErr{"zkb: resource limit exceeded (max_values)"};
        step();
        switch (g.type) {
            case ir::G_CONSTANT: {  // :345-348
                const auto& v = consts[g.const_idx];
                set(scope, g.w0, p.constant(v.data(), v.size()));
            } break;
            case ir::G_ASSERT_ZERO: {  // :350-364
                uint32_t w = get(scope, g.w0);
                uint32_t z = weight ? as_mul(*weight, w) : p.copy(w);
                p.assert_zero(z, g.w0);
                p.ir_gates++;
            } break;
            case ir::G_COPY:  // :366-370
                set(scope, g.w0, p.copy(get(scope, g.w1)));
                break;
            case ir::G_ADD: case ir::G_MUL: case ir::G_AND: case ir::G_XOR: {  // :372-384, 400-412
                uint32_t l = get(scope, g.w1);
                uint32_t r = get(scope, g.w2);
                uint32_t res = g.type == ir::G_ADD ? p.add(l, r) : g.type == ir::G_MUL ? p.multiply(l, r)
                               : g.type == ir::G_AND ? p.and_(l, r) : p.xor_(l, r);
                p.ir_gates++;
                set(scope, g.w0, res);
            } break;
            case ir::G_ADD_CONSTANT: case ir::G_MUL_CONSTANT: {  // :386-398
                uint32_t l = get(scope, g.w1);
                const auto& v = consts[g.const_idx];
                uint32_t res = g.type == ir::G_ADD_CONSTANT ? p.add_constant(l, v.data(), v.size()) : p.mul_constant(l, v.data(), v.size());
                p.ir_gates++;
                set(scope, g.w0, res);
            } break;
            case ir::G_NOT:  // :414-418
                p.ir_gates++;
                set(scope, g.w0, p.not_(get(scope, g.w1)));
                break;
            case ir::G_INSTANCE: {  // :420-427
                if (instances.empty()) throw EvalErr{"Not enough instance to consume"};
                uint32_t pos = instances.front();
                instances.pop_front();
                p.cb_count[CB_INSTANCE]++;
                if (pos + 1 > p.n_instance) p.n_instance = pos + 1;
                set(scope, g.w0, p.push_value(V_INSTANCE, 0, pos));
            } break;
            case ir::G_WITNESS: {  // :429-432 + PlaintextBackend::witness :944-946 (None => panic)
                if (witnesses.empty() && p.keep_copies) {
                    // the IRFlattener accepts witness(None): the gate is emitted, no value is pushed (flattening.rs:178-190,
                    // builder.rs:261-263) — flattening a relation as the verifier, without a witness file
                    p.cb_count[CB_WITNESS]++;
                    set(scope, g.w0, p.push_value(V_WITNESS, 0, kNoWitnessValue));
                    break;
                }
                if (witnesses.empty()) throw Fatal{"Missing witness value for PlaintextBackend"};
                uint32_t pos = witnesses.front();
                witnesses.pop_front();
                p.cb_count[CB_WITNESS]++;
                if (pos + 1 > p.n_witness) p.n_witness = pos + 1;
                set(scope, g.w0, p.push_value(V_WITNESS, 0, pos));
            } break;
            case ir::G_FREE: {  // :434-439
                uint64_t last = g.has_last ? g.w1 : g.w0;
                if (last > g.w0) step(last - g.w0);
                for (uint64_t w = g.w0; w <= last; w++) {
                    remove(scope, w);
                    if (w == UINT64_MAX) break;
                }
            } break;
            case ir::G_CALL: {  // :441-471
                auto it = known_functions.find(g.cx->name);
                if (it == known_functions.end()) throw EvalErr{"Unknown function"};
                const FunctionDecl& f = it->second;
                std::vector<uint64_t> eo, ei;
                expand_wirelist(g.cx->outputs, eo);
                expand_wirelist(g.cx->inputs, ei);
                check_arity(g.cx->name, f, eo.size(), ei.size());
                Iters fresh;  // named calls do NOT see the caller's iterators (:456)
                call_function(f, eo, ei, scope, fresh, instances, witnesses, weight);
            } break;
            case ir::G_ANON_CALL: {  // :473-491
                std::vector<uint64_t> eo, ei;
                expand_wirelist(g.cx->outputs, eo);
                expand_wirelist(g.cx->inputs, ei);
                ingest_subcircuit(g.cx->body, consts, eo, ei, scope, iters, instances, witnesses, weight);
            } break;
            case ir::G_FOR: {  // :495-559
                const ir::Complex& cx = *g.cx;
                std::vector<uint64_t> eo, ei;
                // the callee is resolved once per loop (definitions only happen at the head of a relation message, never
                // while its gates run); an unknown function is still reported by the first iteration that needs it
                const FunctionDecl* callee = nullptr;
                if (!cx.body_is_anon) {
                    auto it = known_functions.find(cx.fn_name);
                    if (it != known_functions.end()) callee = &it->second;
                }
                // the For gate lists its outputs: the scope's table is sized once for the loop (same memory bound as
                // one-by-one insertion) instead of doubling its way up while the iterations bind them
                {
                    uint64_t hi = 0, cnt = 0;
                    for (const auto& el : cx.outputs) {
                        const uint64_t top = el.is_range ? el.last : el.first;
                        if (top >= el.first && top - el.first < (1ull << 32)) {
                            hi = std::max(hi, top);
                            cnt += top - el.first + 1;
                        }
                    }
                    if (cnt >= 1024 && scope.sparse.empty()) scope.ensure_dense(hi, cnt);
                }
                if (callee && try_call_group(cx, *callee, scope, iters, weight)) {  // the whole loop as one call group
                    iters_remove(iters, cx.name);
                    break;
                }
                Iters fresh;
                for (uint64_t i = cx.first; i <= cx.last; i++) {
                    step();
                    iters_set(iters, cx.name, i);
                    if (!cx.body_is_anon) {
                        if (!callee) throw EvalErr{"Unknown function"};
                        const FunctionDecl& f = *callee;
                        eval_iterexpr_list(cx.it_outputs, iters, eo);
                        eval_iterexpr_list(cx.it_inputs, iters, ei);
                        check_arity(cx.fn_name, f, eo.size(), ei.size());
                        fresh.clear();
                        call_function(f, eo, ei, scope, fresh, instances, witnesses, weight);
                    } else {
                        eval_iterexpr_list(cx.it_outputs, iters, eo);
                        eval_iterexpr_list(cx.it_inputs, iters, ei);
                        ingest_subcircuit(cx.body, consts, eo, ei, scope, iters, instances, witnesses, weight);
                    }
                    if (i == UINT64_MAX) break;
                }
                iters_remove(iters, cx.name);
            } break;
            case ir::G_SWITCH: {  // :563-688
                const ir::Complex& cx = *g.cx;
                uint64_t max_i = 0, max_w = 0;
                for (const auto& br : cx.branches) {  // :565-581
                    uint64_t ic, wc;
                    if (!br.is_anon) {
                        auto it = known_functions.find(br.name);
                        if (it == known_functions.end()) throw EvalErr{"Unknown function"};
                        ic = it->second.instance_nbr;
                        wc = it->second.witness_nbr;
                    } else {
                        ic = br.instance_count;
                        wc = br.witness_count;
                    }
                    max_i = std::max(max_i, ic);
                    max_w = std::max(max_w, wc);
                }
                // :586-591: the first `max` queued values are handed (cloned) to every branch
                Queue new_instances, new_witnesses;
                for (uint64_t k = 0, n = std::min<uint64_t>(instances.size(), max_i); k < n; k++) {
                    new_instances.push_back(instances.front());
                    instances.pop_front();
                }
                for (uint64_t k = 0, n = std::min<uint64_t>(witnesses.size(), max_w); k < n; k++) {
                    new_witnesses.push_back(witnesses.front());
                    witnesses.pop_front();
                }
                std::vector<uint64_t> eo, ei;
                expand_wirelist(cx.outputs, eo);  // :597
                std::vector<Scope*> branch_scopes;
                std::vector<uint32_t> weights;
                auto cleanup = [&]() {
                    for (auto s : branch_scopes) release_scope(s);
                    branch_scopes.clear();
                };
                try {
                    size_t nb = std::min(cx.cases.size(), cx.branches.size());  // zip
                    for (size_t k = 0; k < nb; k++) {  // :600-670
                        const auto& br = cx.branches[k];
                        uint32_t bw = compute_weight(consts[cx.cases[k]], get(scope, g.w0));
                        uint32_t wbw = weight ? as_mul(*weight, bw) : bw;
                        Scope* bs = new_scope();
                        branch_scopes.push_back(bs);
                        Queue qi = new_instances, qw = new_witnesses;
                        if (!br.is_anon) {
                            auto it = known_functions.find(br.name);
                            if (it == known_functions.end()) throw EvalErr{"Unknown function: " + br.name};
                            const FunctionDecl& f = it->second;
                            expand_wirelist(br.inputs, ei);
                            check_arity(br.name, f, eo.size(), ei.size());
                            for (uint64_t w : ei) bs->set(w, p.copy(get(scope, w)));  // HashMap::insert (:626-629)
                            Iters fresh;
                            call_function(f, eo, ei, *bs, fresh, qi, qw, &wbw);
                        } else {
                            expand_wirelist(br.inputs, ei);
                            for (uint64_t w : ei) bs->set(w, p.copy(get(scope, w)));
                            ingest_subcircuit(br.subcircuit, consts, eo, ei, *bs, iters, qi, qw, &wbw);
                        }
                        weights.push_back(wbw);
                    }
                    for (uint64_t ow : eo) {  // :673-687
                        uint8_t zero = 0;
                        uint32_t acc = p.constant(&zero, 1);
                        for (size_t k = 0; k < branch_scopes.size(); k++) {
                            uint32_t ww = as_mul(get(*branch_scopes[k], ow), weights[k]);
                            acc = as_add(acc, ww);
                        }
                        set(scope, ow, acc);
                    }
                } catch (...) {
                    cleanup();
                    throw;
                }
                cleanup();
            } break;
            default:
                throw EvalErr{"No gate type"};
        }
    }

    // ---- evaluator.rs:232-303 ----------------------------------------------------------------------
    void ingest_values(const ir::Message& m) {
        modulus_le = m.header.field_characteristic;  // ingest_header: last header wins
        bool inst = m.type == ir::MSG_INSTANCE;
        auto& store = inst ? instance_values : witness_values;
        auto& q = inst ? instance_queue : witness_queue;
        for (const auto& v : m.values) {
            if (store.size() >= 0xFFFFFFF0u) throw EvalErr{"zkb: too many input values"};
            q.push_back((uint32_t)store.size());
            store.push_back(v);
        }
    }

    void ingest_relation(ir::Message& m) {
        modulus_le = m.header.field_characteristic;
        is_boolean = (m.gate_mask & ir::M_BOOL) == ir::M_BOOL;  // contains_feature(gate_mask, BOOL), :262
        std::string e;
        if (!prog().set_field(m.header.field_characteristic.data(), m.header.field_characteristic.size(), m.header.field_degree, e))
            throw EvalErr{e};
        c->is_boolean = is_boolean;
        if (!m.gates.empty()) verified_at_least_one_gate = true;
        auto consts = std::make_shared<std::vector<std::vector<uint8_t>>>(std::move(m.consts));
        for (auto& f : m.functions) {  // :273-284, later definitions overwrite
            FunctionDecl d;
            d.body = std::make_shared<std::vector<ir::Gate>>(std::move(f.body));
            d.consts = consts;
            d.instance_nbr = f.instance_count;
            d.witness_nbr = f.witness_count;
            d.output_count = f.output_count;
            d.input_count = f.input_count;
            d.n_local = getenv("ZKB_NO_SIMPLE_CALLS") ? 0 : simple_body_locals(*d.body, d.output_count, d.input_count);
            known_functions[f.name] = std::move(d);
        }
        Iters iters;
        const size_t n_gates = m.gates.size();
        for (size_t i = 0; i < n_gates; i++) {
            if (i + 8 < n_gates) {
                const ir::Gate& ahead = m.gates[i + 8];
                values.prefetch(ahead.w1);
                values.prefetch(ahead.w2);
            }
            ingest_gate(m.gates[i], *consts, values, iters, instance_queue, witness_queue, nullptr);
        }
    }


    // ---- flat relation messages, recorded in bulk straight from the FlatBuffers tables ----------------------------------
    // A builder-produced flat relation is a run of messages of 100 000 simple gates.  For a window of such messages the
    // serial gate loop (ingest_relation above, evaluator.rs:288-301) is replaced by three passes over the tables in place —
    // no owned Gate structs — each spread over the parse threads, one message per task:
    //   count   gate kinds per message (value handles, assertion and input-stream positions are prefix sums of these)
    //   define  every value-defining gate writes its SSA row (kind, operand WIRE ids) and binds its output wire in the
    //           scope table with a compare-and-swap: a wire that already has a value is a conflict
    //   resolve operand wire ids -> value handles; an operand must have been bound by an EARLIER gate (smaller handle)
    // Anything irregular — a structured gate, Copy, Free, a re-used or undefined wire, too few instance / witness values,
    // a resource limit, a malformed table — makes the window fall back, untouched, to the serial path, which reports the
    // error exactly where and how the reference does.  Regular windows give the state the serial path would give.
    struct FlatCount {
        uint64_t n_gates = 0, n_values = 0, n_asserts = 0, n_inst = 0, n_wit = 0, n_const_gates = 0, max_w0 = 0;
        uint64_t by_type[ir::G_WITNESS + 1] = {0};
        std::vector<std::pair<const uint8_t*, uint32_t>> consts;  // bytes of the constant-bearing gates, in order
        ir::FlatRelationHead head;
        bool ok = false;
    };
    struct FlatFill {
        zkb_evaluator* ev;
        uint32_t v, a, inst, wit, ci;  // running value handle / assertion index / stream cursors / constant-gate index
        const uint32_t* cidx;          // pool index of this message's k-th constant-bearing gate
        const uint32_t* inst_pos;
        const uint32_t* wit_pos;
        uint32_t v_lo, v_hi;           // undo pass: handles of the window being rolled back
        bool conflict = false;
    };
    static bool flat_count_fn(void* ctx, const ir::FlatGate& g) {
        FlatCount& k = *(FlatCount*)ctx;
        k.n_gates++;
        k.by_type[g.type]++;
        if (g.type == ir::G_ASSERT_ZERO) {
            k.n_asserts++;
            return true;
        }
        k.n_values++;
        if (g.w0 > k.max_w0) k.max_w0 = g.w0;
        if (g.type == ir::G_INSTANCE) k.n_inst++;
        else if (g.type == ir::G_WITNESS) k.n_wit++;
        if (g.cbytes) k.consts.emplace_back(g.cbytes, g.clen);
        return g.w0 < 0xFFFFFFFFull;  // operand wire ids are staged in the 32-bit operand columns
    }
    static bool flat_fill_fn(void* ctx, const ir::FlatGate& g) {
        FlatFill& f = *(FlatFill*)ctx;
        Program& p = f.ev->prog();
        if (g.type == ir::G_ASSERT_ZERO) {
            if (g.w0 >= 0xFFFFFFFFull) return !(f.conflict = true);
            p.asserts[f.a++] = AssertRec{(uint32_t)g.w0, f.v, g.w0};  // value: the wire for now (resolved below)
            return true;
        }
        uint8_t kind;
        uint32_t a = 0, b = 0;
        switch (g.type) {
            case ir::G_CONSTANT: kind = V_CONST; b = f.cidx[f.ci++]; break;
            case ir::G_ADD: kind = V_ADD; break;
            case ir::G_MUL: kind = V_MUL; break;
            case ir::G_AND: kind = V_AND; break;
            case ir::G_XOR: kind = V_XOR; break;
            case ir::G_NOT: kind = V_NOT; break;
            case ir::G_ADD_CONSTANT: kind = V_ADDC; b = f.cidx[f.ci++]; break;
            case ir::G_MUL_CONSTANT: kind = V_MULC; b = f.cidx[f.ci++]; break;
            case ir::G_INSTANCE: kind = V_INSTANCE; b = f.inst_pos[f.inst++]; break;
            default: kind = V_WITNESS; b = f.wit_pos[f.wit++]; break;
        }
        if (kind >= V_ADD) {
            if (g.w1 >= 0xFFFFFFFFull || g.w2 >= 0xFFFFFFFFull) return !(f.conflict = true);
            a = (uint32_t)g.w1;
            if (kind == V_ADD || kind == V_MUL || kind == V_AND || kind == V_XOR) b = (uint32_t)g.w2;
        }
        p.kind[f.v] = kind;
        p.opa[f.v] = a;
        p.opb[f.v] = b;
        uint32_t expect = Scope::kNone;
        if (!__atomic_compare_exchange_n(&f.ev->values.dense[g.w0], &expect, f.v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED))
            return !(f.conflict = true);  // "Wire_{id} already has a value in this scope."
        f.v++;
        return true;
    }
    static bool flat_undo_fn(void* ctx, const ir::FlatGate& g) {  // unbind the wires this window bound
        FlatFill& f = *(FlatFill*)ctx;
        if (g.type == ir::G_ASSERT_ZERO || g.w0 >= f.ev->values.dense.size()) return true;
        uint32_t& d = f.ev->values.dense[g.w0];
        if (d >= f.v_lo && d < f.v_hi) d = Scope::kNone;
        return true;
    }

    template <class F>
    static void parallel_for(size_t n, unsigned threads, F f) {
        std::atomic<size_t> next{0};
        auto work = [&]() {
            for (size_t i; (i = next.fetch_add(1)) < n;) f(i);
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < threads && t < n; t++) pool.emplace_back(work);
        work();
        for (auto& th : pool) th.join();
    }

    // Returns how many messages, from w0 on, have been recorded (a prefix of the window: the leading run of flat relation
    // messages).  0: nothing was changed; *serial_n then says how many leading messages the serial path should take before
    // the bulk path is tried again (the leading run of other messages, or the whole window after an irregularity).
    size_t ingest_flat_window(const uint8_t* buf, const std::vector<std::pair<size_t, size_t>>& msgs, size_t w0, size_t w1, unsigned threads,
                              size_t* serial_n) {
        Program& p = prog();
        *serial_n = w1 - w0;
        if (fatal || evaluated || batch_evaluated || has_error || p.keep_copies || p.expand_on || !values.sparse.empty() || getenv("ZKB_NO_FLAT_INGEST")) return 0;
        size_t nm = w1 - w0;
        static const bool timing = getenv("ZKB_TIMING") != nullptr;
        auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        double t_0 = now();
        auto lap = [&](const char* what) {
            if (!timing) return;
            double t = now();
            fprintf(stderr, "  flat window: %-8s %.4f s\n", what, t - t_0);
            t_0 = t;
        };
        std::vector<FlatCount> cnt(nm);
        parallel_for(nm, threads, [&](size_t i) {
            std::string e;
            cnt[i].ok = ir::walk_flat_relation(buf + msgs[w0 + i].first, msgs[w0 + i].second, cnt[i].head, flat_count_fn, &cnt[i], false, e) == ir::FLAT_OK;
        });
        lap("count");
        {
            size_t n_ok = 0;
            while (n_ok < nm && cnt[n_ok].ok) n_ok++;
            if (n_ok == 0) {  // the window starts with other messages (instance / witness values, structured relations)
                size_t n_bad = 0;
                while (n_bad < nm && !cnt[n_bad].ok) n_bad++;
                *serial_n = n_bad;
                return 0;
            }
            nm = n_ok;
            w1 = w0 + nm;
            cnt.resize(nm);
        }
        begin_relation();
        uint64_t tv = 0, ta = 0, ti = 0, tw = 0, tg = 0, max_w0 = 0;
        for (auto& k : cnt) {
            tv += k.n_values; ta += k.n_asserts; ti += k.n_inst; tw += k.n_wit; tg += k.n_gates;
            max_w0 = std::max(max_w0, k.max_w0);
        }
        const uint64_t v0 = p.n_values(), a0 = p.asserts.size();
        if (tv == 0 || v0 + tv >= c->max_values || steps + tg > c->max_steps || a0 + ta >= 0xFFFFFFF0ull) return 0;
        if (ti > instance_queue.size() || tw > witness_queue.size()) return 0;  // the serial path reports where the stream runs dry
        // the scope stays a dense table only while ids are within a small multiple of the values bound (context.h)
        if (max_w0 >= Scope::kDenseLimit || max_w0 > 4 * (values.n_sets + tv + 1024)) return 0;
        // header / field of every message, as ingest_relation does (:262-267); any change of field goes the serial way
        for (auto& k : cnt) {
            if (p.field_set && k.head.header.field_characteristic != p.modulus_le) return 0;
            std::string e;
            if (!p.set_field(k.head.header.field_characteristic.data(), k.head.header.field_characteristic.size(), k.head.header.field_degree, e))
                return 0;
        }
        // ---- point of no return for the cheap part: constants are interned (harmless if the window falls back later)
        std::vector<std::vector<uint32_t>> cidx(nm);
        for (size_t i = 0; i < nm; i++) {
            cidx[i].reserve(cnt[i].consts.size());
            for (auto& cb : cnt[i].consts) cidx[i].push_back(p.intern_const(cb.first, cb.second));
        }
        std::vector<uint32_t> inst_pos(instance_queue.begin(), instance_queue.begin() + ti), wit_pos(witness_queue.begin(), witness_queue.begin() + tw);
        // Room for the whole buffer at once, sized from its length (a flat gate takes >= 56 bytes of tables), with the fresh
        // pages touched by all threads: growing 9 bytes per value window by window would copy the columns again and again
        // and take every page fault on this thread.
        const uint64_t est = v0 + std::max<uint64_t>(tv, (msgs.back().first + msgs.back().second - msgs[w0].first) / 56);
        if (p.kind.capacity() < v0 + tv) {
            p.kind.reserve(est);
            p.opa.reserve(est);
            p.opb.reserve(est);
            const uint64_t a_est = a0 + std::max<uint64_t>(ta, (est - v0) * (ta + 1) / (tv + 1) * 5 / 4);
            p.asserts.reserve(a_est);
            struct Span { uint8_t* lo; uint8_t* hi; };
            const Span spans[4] = {{(uint8_t*)p.kind.data() + v0, (uint8_t*)p.kind.data() + p.kind.capacity()},
                                   {(uint8_t*)(p.opa.data() + v0), (uint8_t*)(p.opa.data() + p.opa.capacity())},
                                   {(uint8_t*)(p.opb.data() + v0), (uint8_t*)(p.opb.data() + p.opb.capacity())},
                                   {(uint8_t*)(p.asserts.data() + a0), (uint8_t*)(p.asserts.data() + p.asserts.capacity())}};
            constexpr size_t kChunk = 4u << 20;
            std::vector<std::pair<uint8_t*, uint8_t*>> chunks;
            for (const Span& sp : spans)
                for (uint8_t* q = sp.lo; q < sp.hi; q += kChunk) chunks.emplace_back(q, std::min(sp.hi, q + kChunk));
            parallel_for(chunks.size(), threads, [&](size_t i) {
                for (volatile uint8_t* q = chunks[i].first; q < chunks[i].second; q += 4096) *q = 0;  // capacity beyond size(): ours, unread
            });
        }
        p.kind.resize(v0 + tv);
        p.opa.resize(v0 + tv);
        p.opb.resize(v0 + tv);
        p.asserts.resize(a0 + ta);
        const size_t dense0 = values.dense.size();
        if (max_w0 >= values.dense.size()) {
            // wires of a flat relation are numbered as they are defined: the table the rest of the buffer needs, in one step
            uint64_t want = std::max<uint64_t>(max_w0 + 1, std::min<uint64_t>(values.n_sets + (est - v0), 4 * (values.n_sets + tv + 1024)));
            size_t n = values.dense.size() ? values.dense.size() : 16;
            while (n < want) n *= 2;
            const size_t old = values.dense.size();
            values.dense.reserve(n);
            constexpr size_t kChunk = 1u << 20;  // entries
            const size_t nch = (n - old + kChunk - 1) / kChunk;
            uint32_t* d = values.dense.data();
            parallel_for(nch, threads, [&](size_t i) {  // first touch + fill by all threads; resize() below then runs over resident pages
                const size_t lo = old + i * kChunk, hi = std::min(n, lo + kChunk);
                for (size_t k = lo; k < hi; k++) ((volatile uint32_t*)d)[k] = Scope::kNone;
            });
            values.dense.resize(n, Scope::kNone);
        }
        std::vector<FlatFill> fill(nm);
        {
            uint64_t v = v0, a = a0, ii = 0, ww = 0;
            for (size_t i = 0; i < nm; i++) {
                fill[i] = FlatFill{this, (uint32_t)v, (uint32_t)a, 0, 0, 0, cidx[i].data(), inst_pos.data() + ii, wit_pos.data() + ww,
                                   (uint32_t)v0, (uint32_t)(v0 + tv), false};
                v += cnt[i].n_values; a += cnt[i].n_asserts; ii += cnt[i].n_inst; ww += cnt[i].n_wit;
            }
        }
        lap("prepare");
        std::atomic<bool> bad{false};
        parallel_for(nm, threads, [&](size_t i) {
            std::string e;
            ir::FlatRelationHead h;
            int rc = ir::walk_flat_relation(buf + msgs[w0 + i].first, msgs[w0 + i].second, h, flat_fill_fn, &fill[i], true, e);
            if (rc != ir::FLAT_OK || fill[i].conflict) bad = true;
        });
        lap("define");
        // resolve: operand wires -> handles of values bound EARLIER in program order
        if (!bad) {
            const uint32_t* dense = values.dense.data();
            const size_t dn = values.dense.size();
            const size_t chunks = (tv + 65535) / 65536, achunks = (ta + 65535) / 65536;
            parallel_for(chunks + achunks, threads, [&](size_t ch) {
                if (ch < chunks) {
                    const uint64_t lo = v0 + ch * 65536, hi = std::min<uint64_t>(v0 + tv, lo + 65536);
                    for (uint64_t v = lo; v < hi; v++) {
                        const uint8_t k = p.kind[v];
                        if (k < V_ADD) continue;
                        const uint32_t wa = p.opa[v];
                        const uint32_t ra = wa < dn ? dense[wa] : Scope::kNone;
                        if (ra >= v) { bad = true; return; }  // undefined (kNone) or bound later: "No value given for wire_{id}"
                        p.opa[v] = ra;
                        if (k == V_ADD || k == V_MUL || k == V_AND || k == V_XOR) {
                            const uint32_t wb = p.opb[v];
                            const uint32_t rb = wb < dn ? dense[wb] : Scope::kNone;
                            if (rb >= v) { bad = true; return; }
                            p.opb[v] = rb;
                        }
                    }
                } else {
                    const uint64_t lo = a0 + (ch - chunks) * 65536, hi = std::min<uint64_t>(a0 + ta, lo + 65536);
                    for (uint64_t a = lo; a < hi; a++) {
                        AssertRec& r = p.asserts[a];
                        const uint32_t rv = r.value < dn ? dense[r.value] : Scope::kNone;
                        if (rv >= r.pos) { bad = true; return; }
                        r.value = rv;
                    }
                }
            });
        }
        lap("resolve");
        if (bad) {  // undo: the window is replayed gate by gate by the serial path
            parallel_for(nm, threads, [&](size_t i) {
                std::string e;
                ir::FlatRelationHead h;
                ir::walk_flat_relation(buf + msgs[w0 + i].first, msgs[w0 + i].second, h, flat_undo_fn, &fill[i], false, e);
            });
            (void)dense0;  // a grown table stays grown: kNone entries are indistinguishable from absent ones
            p.kind.resize(v0);
            p.opa.resize(v0);
            p.opb.resize(v0);
            p.asserts.resize(a0);
            return 0;
        }
        // commit the bookkeeping the serial loop does gate by gate
        for (auto& k : cnt) {
            modulus_le = k.head.header.field_characteristic;
            is_boolean = (k.head.gate_mask & ir::M_BOOL) == ir::M_BOOL;
            if (k.n_gates) verified_at_least_one_gate = true;
            p.cb_count[CB_CONSTANT] += k.by_type[ir::G_CONSTANT];
            p.cb_count[CB_ADD] += k.by_type[ir::G_ADD];
            p.cb_count[CB_MUL] += k.by_type[ir::G_MUL];
            p.cb_count[CB_ADDC] += k.by_type[ir::G_ADD_CONSTANT];
            p.cb_count[CB_MULC] += k.by_type[ir::G_MUL_CONSTANT];
            p.cb_count[CB_AND] += k.by_type[ir::G_AND];
            p.cb_count[CB_XOR] += k.by_type[ir::G_XOR];
            p.cb_count[CB_NOT] += k.by_type[ir::G_NOT];
            p.cb_count[CB_INSTANCE] += k.by_type[ir::G_INSTANCE];
            p.cb_count[CB_WITNESS] += k.by_type[ir::G_WITNESS];
            p.cb_count[CB_COPY] += k.by_type[ir::G_ASSERT_ZERO];  // an unweighted assertion tests a copy (:355)
            p.cb_count[CB_ASSERT_ZERO] += k.by_type[ir::G_ASSERT_ZERO];
            p.ir_gates += k.n_gates - k.by_type[ir::G_CONSTANT] - k.by_type[ir::G_INSTANCE] - k.by_type[ir::G_WITNESS];
        }
        c->is_boolean = is_boolean;
        steps += tg;
        values.n_sets += tv;
        values.live += tv;
        for (uint64_t k = 0; k < ti; k++) p.n_instance = std::max(p.n_instance, inst_pos[k] + 1);
        for (uint64_t k = 0; k < tw; k++) p.n_witness = std::max(p.n_witness, wit_pos[k] + 1);
        instance_queue.erase(instance_queue.begin(), instance_queue.begin() + ti);
        witness_queue.erase(witness_queue.begin(), witness_queue.begin() + tw);
        return nm;
    }

    // The first relation message fixes the streams: in batch mode, positions n_common .. n_common + (longest set) - 1 follow
    // the common values in both queues.
    void begin_relation() {
        if (relation_seen) return;
        relation_seen = true;
        if (!batch()) return;
        n_common_inst = (uint32_t)instance_values.size();
        n_common_wit = (uint32_t)witness_values.size();
        for (uint64_t k = 0; k < max_set_inst; k++) instance_queue.push_back(n_common_inst + (uint32_t)k);
        for (uint64_t k = 0; k < max_set_wit; k++) witness_queue.push_back(n_common_wit + (uint32_t)k);
    }

    // Evaluator::ingest_message, :213-230: errors latch, later messages are skipped
    int ingest_parsed(ir::Message& m) {
        if (fatal) return fail(ZKB_E_FATAL, err);
        if (evaluated || batch_evaluated) return fail(ZKB_E_ARG, "evaluator already finished (get_violations was called)");
        if (batch() && relation_seen && m.type != ir::MSG_RELATION)
            return fail(ZKB_E_ARG, "with value sets, common instance / witness values must come before the first relation message");
        if (m.type == ir::MSG_RELATION) begin_relation();
        if (has_error) return ZKB_OK;
        try {
            if (m.type == ir::MSG_RELATION) ingest_relation(m);
            else ingest_values(m);
        } catch (const EvalErr& e) {
            has_error = true;
            found_error = e.msg;
            ctx_latch(c, e.msg);
            if (batch()) {
                global_cut = prog().n_values();
                global_cut_msg = e.msg;
            }
        } catch (const Fatal& f) {
            if (batch()) {  // not an error of the call: a cut point of every set that gets this far (decided per set)
                has_error = true;
                global_cut = prog().n_values();
                global_cut_msg = f.msg;
                global_cut_fatal = true;
                return ZKB_OK;
            }
            if (assertion_fails_before(f)) return ZKB_OK;
            fatal = true;
            return fail(ZKB_E_FATAL, f.msg);
        } catch (const Program::ProgramPanic& f) {  // ExpandDefinable's panics (exp_definable.rs:62-64, ...)
            fatal = true;
            return fail(ZKB_E_FATAL, f.msg);
        }
        return ZKB_OK;
    }

    int ingest_bytes(const uint8_t* buf, size_t len) {
        ir::Message m;
        std::string e;
        if (!ir::read_message(buf, len, m, e)) {
            // Evaluator::from_messages unwraps parse errors (:193): the reference aborts
            fatal = true;
            return fail(ZKB_E_FORMAT, e);
        }
        return ingest_parsed(m);
    }

    int fail(int code, const std::string& m) {
        err = m;
        return code;
    }

    // The deferred evaluation shared by one statement and by value sets: levelize + upload the recorded program (once),
    // pack the streams (common values, then each set's; one set of the common values alone without sets) and run them as
    // one batch, split over the communicator of zkb_evaluator_use_devices when there are at least as many sets as contexts.
    // t_begin >= 0: ZKB_TIMING report of the phases.
    int run_recorded(std::vector<zkb_verdict>& v, double t_begin) {
        Program& p = prog();
        auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        if (!c->finalized) {
            c->live_values.clear();
            values.for_each([&](uint64_t, uint32_t h) {
                if (!is_callout(h)) c->live_values.push_back(h);  // group outputs (implicit values) are always kept
            });
            int rc = ctx_finalize(c, 0);
            if (rc != ZKB_OK) return fail(rc, c->err);
        }
        if (t_begin >= 0) fprintf(stderr, "finish: live wires + levelize + program upload %.3f s\n", now() - t_begin);
        const size_t S = std::max<size_t>(sets.size(), 1);
        // one stride for every set: the widest value over all of them (raw values >= p keep their bytes, trap 1)
        size_t stride = (size_t)p.nlimb * 4;
        for (const auto* vals : {&instance_values, &witness_values})
            for (const auto& x : *vals) {
                size_t n = x.size();
                while (n > 0 && x[n - 1] == 0) n--;
                stride = std::max(stride, n);
            }
        stride = std::max(stride, std::max(set_inst.widest, set_wit.widest));
        stride = (stride + 3) / 4 * 4;
        // [set][position][stride]; one shared vector (set stride 0) when no set brings values of that stream
        auto pack = [&](const std::vector<std::vector<uint8_t>>& common, const Arena& a, uint32_t need, uint64_t ValueSet::*first,
                        uint64_t ValueSet::*count, uint64_t& set_stride) {
            const bool per_set = a.size() > 0;
            const size_t per = (size_t)std::max<uint32_t>(need, 1) * stride;
            set_stride = per_set ? per : 0;
            std::vector<uint8_t> out(per_set ? per * S : per, 0);
            parallel_for(per_set ? S : 1, parse_threads(), [&](size_t j) {
                uint8_t* o = out.data() + j * set_stride;
                uint32_t k = 0;
                for (; k < need && k < common.size(); k++) {
                    size_t n = common[k].size();
                    while (n > 0 && common[k][n - 1] == 0) n--;
                    memcpy(o + (size_t)k * stride, common[k].data(), n);
                }
                if (!per_set) return;
                const uint64_t v0 = sets[j].*first, nv = sets[j].*count;
                for (uint64_t i = 0; i < nv && k < need; i++, k++)
                    memcpy(o + (size_t)k * stride, a.bytes.data() + a.end[v0 + i], a.end[v0 + i + 1] - a.end[v0 + i]);
            });
            return out;
        };
        uint64_t iss = 0, wss = 0;
        const std::vector<uint8_t> ib = pack(instance_values, set_inst, p.n_instance, &ValueSet::inst0, &ValueSet::n_inst, iss);
        const std::vector<uint8_t> wb = pack(witness_values, set_wit, p.n_witness, &ValueSet::wit0, &ValueSet::n_wit, wss);
        v.assign(S, zkb_verdict{});
        const double t_eval = now();
        batch_sharded = batch() && devices.size() > 1 && S >= devices.size();
        int rc = batch_sharded ? zkb_evaluate_sharded(devices.data(), (int)devices.size(), ib.data(), iss, wb.data(), wss, (uint32_t)stride, (uint32_t)S, v.data())
                               : zkb_evaluate(c, ib.data(), iss, wb.data(), wss, (uint32_t)stride, (uint32_t)S, v.data());
        if (rc != ZKB_OK) return fail(rc, c->err);
        if (t_begin >= 0) fprintf(stderr, "finish: zkb_evaluate (allocations, input upload, kernels, verdict) %.3f s\n", now() - t_eval);
        return ZKB_OK;
    }

    // The deferred evaluation: levelize + upload the recorded program (once), run it for the queued instance / witness
    // values (a batch of one), and rebuild the reference's text for the first failing assertion (:357-362).
    int evaluate_recorded(bool& have_error, std::string& first_error) {
        have_error = false;
        Program& p = prog();
        const bool timing = getenv("ZKB_TIMING") != nullptr;
        auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t_begin = now();
        if (!p.field_set || p.n_values() == 0) return ZKB_OK;
        std::vector<zkb_verdict> vs;
        int rc = run_recorded(vs, timing ? t_begin : -1.0);
        if (rc != ZKB_OK) return rc;
        const zkb_verdict& v = vs[0];
        if (v.first_fail_seq != UINT64_MAX) {
            uint64_t w = p.asserts[v.first_fail_seq].src_wire;
            first_error = "Wire_" + u64s(w) + " (may be weighted) should be 0, while it is not";  // :357-362
            have_error = true;
        }
        return ZKB_OK;
    }

    // A condition on which the reference panics was met while recording.  The reference evaluates as it goes: had an
    // assertion recorded BEFORE this point failed, its error would have latched (:213-221) and the panic would never have
    // been reached.  So the recorded prefix is evaluated now; true = an assertion fails, the statement is decided.
    bool assertion_fails_before(const Fatal&) {
        Program& p = prog();
        if (!c->has_gpu || p.keep_copies || !p.field_set || p.asserts.empty() || c->finalized) return false;
        bool have = false;
        std::string msg;
        if (evaluate_recorded(have, msg) != ZKB_OK || !have) return false;
        has_error = true;
        found_error = msg;
        ctx_latch(c, msg);
        return true;
    }

    // ---- get_violations, :199-208, with the deferred evaluation in the middle -------------------------
    int finish() {
        if (evaluated) return ZKB_OK;
        if (fatal) return fail(ZKB_E_FATAL, err);
        violations.clear();
        if (!verified_at_least_one_gate) violations.push_back("Did not receive any gate to verify.");
        std::string first_error;
        bool have_error = false;
        int rc = evaluate_recorded(have_error, first_error);
        if (rc != ZKB_OK) return rc;
        if (!have_error && has_error) {
            first_error = found_error;
            have_error = true;
        }
        if (have_error) violations.push_back(first_error);
        evaluated = true;
        return ZKB_OK;
    }

    // ---- value sets ------------------------------------------------------------------------------------------------------
    // One set from a concatenation of size-prefixed Instance / Witness messages (`where` names the source in errors).  The
    // set is committed by add_value_set_end once all of its buffers have been read.
    int add_value_set_bytes(const uint8_t* buf, size_t len, const std::string& where) {
        std::vector<std::pair<size_t, size_t>> msgs;
        ir::split_messages(buf, len, msgs);
        for (size_t i = 0; i < msgs.size(); i++) {
            ir::Message m;
            std::string e;
            if (!ir::read_message(buf + msgs[i].first, msgs[i].second, m, e)) return fail(ZKB_E_FORMAT, where + ": " + e);
            if (m.type == ir::MSG_RELATION)
                return fail(ZKB_E_ARG, where + ": a value set holds Instance and Witness messages only (message " + u64s(i) + " is a Relation)");
            Arena& a = m.type == ir::MSG_INSTANCE ? set_inst : set_wit;
            for (const auto& v : m.values) a.push(v);
        }
        return ZKB_OK;
    }
    int add_value_set_begin() {
        if (fatal) return fail(ZKB_E_FATAL, err);
        if (prog().keep_copies) return fail(ZKB_E_ARG, "value sets need an evaluating backend (not flatten / expand-definable)");
        if (relation_seen) return fail(ZKB_E_ARG, "every value set must be added before the first relation message");
        if (batch_evaluated || evaluated) return fail(ZKB_E_ARG, "evaluator already finished");
        sets.push_back(ValueSet{set_inst.size(), 0, set_wit.size(), 0});
        return ZKB_OK;
    }
    int add_value_set_end(int rc) {
        ValueSet& s = sets.back();
        if (rc == ZKB_OK) {
            s.n_inst = set_inst.size() - s.inst0;
            s.n_wit = set_wit.size() - s.wit0;
            if (instance_values.size() + s.n_inst >= 0xFFFFFFF0u || witness_values.size() + s.n_wit >= 0xFFFFFFF0u)
                rc = fail(ZKB_E_ARG, "zkb: too many input values");
        }
        if (rc != ZKB_OK) {  // the set is not added
            set_inst.bytes.resize(set_inst.end[s.inst0]);
            set_inst.end.resize(s.inst0 + 1);
            set_wit.bytes.resize(set_wit.end[s.wit0]);
            set_wit.end.resize(s.wit0 + 1);
            sets.pop_back();
            return rc;
        }
        max_set_inst = std::max(max_set_inst, s.n_inst);
        max_set_wit = std::max(max_set_wit, s.n_wit);
        return ZKB_OK;
    }

    // Handle of the first value that consumed each stream position, then the minimum over every later position: entry L is
    // where a stream of L values is first found empty (a Switch hands its branches copies of a prefix of the queue, so a
    // position can be skipped; any later one consumed first marks the same point).
    std::vector<uint32_t> first_use_after(uint8_t kind, uint64_t n_pos) {
        const Program& p = prog();
        std::vector<uint32_t> f(n_pos + 1, UINT32_MAX);
        for (uint32_t v = 0, n = p.n_values(); v < n; v++)
            if (p.kind[v] == kind && p.opb[v] < n_pos && f[p.opb[v]] == UINT32_MAX) f[p.opb[v]] = v;
        for (uint64_t k = n_pos; k-- > 0;) f[k] = std::min(f[k], f[k + 1]);
        return f;
    }
    // assertions recorded before value handle h was pushed (an assertion's pos is the number of values recorded before it)
    uint64_t seq_before(uint32_t h) {
        const auto& a = prog().asserts;
        return (uint64_t)(std::upper_bound(a.begin(), a.end(), h, [](uint32_t x, const AssertRec& r) { return x < r.pos; }) - a.begin());
    }

    // Cut of each set: the earliest of its instance stream found empty, its witness stream found empty, the global cut.
    // 0 none, 1 instance, 2 witness, 3 global; the handle in set_cut.
    std::vector<uint8_t> compute_cuts() {
        const uint64_t ni = n_common_inst + max_set_inst, nw = n_common_wit + max_set_wit;
        const std::vector<uint32_t> fi = first_use_after(V_INSTANCE, ni), fw = first_use_after(V_WITNESS, nw);
        std::vector<uint8_t> what(sets.size(), 0);
        set_cut.assign(sets.size(), UINT32_MAX);
        for (size_t j = 0; j < sets.size(); j++) {
            const uint32_t ci = relation_seen ? fi[n_common_inst + sets[j].n_inst] : UINT32_MAX;
            const uint32_t cw = relation_seen ? fw[n_common_wit + sets[j].n_wit] : UINT32_MAX;
            uint32_t cut = global_cut;
            uint8_t w = global_cut != UINT32_MAX ? 3 : 0;
            if (cw < cut) cut = cw, w = 2;
            if (ci < cut) cut = ci, w = 1;
            set_cut[j] = cut;
            what[j] = w;
        }
        return what;
    }

    // Evaluates every set in one batch (once) and decides each one as finish() decides a single statement: the first failing
    // assertion if it comes before the set's cut, else the cut's error (status OK) or panic (ZKB_E_FATAL).
    int evaluate_batch() {
        if (batch_evaluated) return ZKB_OK;
        if (fatal) return fail(ZKB_E_FATAL, err);
        Program& p = prog();
        const size_t S = sets.size();
        const std::vector<uint8_t> what = compute_cuts();
        std::vector<uint64_t> first_fail(S, UINT64_MAX);
        if (p.field_set && p.n_values() > 0) {
            std::vector<zkb_verdict> v;
            int rc = run_recorded(v, -1.0);
            if (rc != ZKB_OK) return rc;
            for (size_t j = 0; j < S; j++) first_fail[j] = v[j].first_fail_seq;
        }
        set_status.assign(S, ZKB_OK);
        set_violations.assign(S, {});
        for (size_t j = 0; j < S; j++) {
            auto& out = set_violations[j];
            if (!verified_at_least_one_gate) out.push_back("Did not receive any gate to verify.");
            const uint64_t cut_seq = what[j] ? seq_before(set_cut[j]) : UINT64_MAX;
            if (first_fail[j] != UINT64_MAX && first_fail[j] < cut_seq) {
                out.push_back("Wire_" + u64s(p.asserts[first_fail[j]].src_wire) + " (may be weighted) should be 0, while it is not");
            } else if (what[j] == 1) {
                out.push_back("Not enough instance to consume");
            } else if (what[j] == 2 || (what[j] == 3 && global_cut_fatal)) {
                set_status[j] = ZKB_E_FATAL;
                out.assign(1, what[j] == 2 ? std::string("Missing witness value for PlaintextBackend") : global_cut_msg);
            } else if (what[j] == 3) {
                out.push_back(global_cut_msg);
            }
        }
        batch_evaluated = true;
        return ZKB_OK;
    }

    // the context that evaluated set j, and j's index in its block of the batch
    zkb_ctx* owner_of(size_t j, uint32_t& idx) {
        if (!batch_sharded) {
            idx = (uint32_t)j;
            return c;
        }
        const uint64_t S = sets.size(), n = devices.size();
        for (uint64_t r = 0; r < n; r++) {
            const uint64_t lo = S * r / n, hi = S * (r + 1) / n;
            if (j >= lo && j < hi) {
                idx = (uint32_t)(j - lo);
                return devices[r];
            }
        }
        idx = 0;
        return c;
    }
};

static bool has_sieve_ext(const std::string& p);

// --------------------------------------------------------------------------------------------------
// flatten: the statement `zki_sieve flatten` writes (cli.rs:442-472) — what the reference's IRFlattener backend
// (consumers/flattening.rs:42-191) emits through a GateBuilder when it sits behind the Evaluator: one SIMPLE gate per
// ZKBackend callback (copies included, no Free), output wire ids allocated 0, 1, 2, ... (builder.rs:229-233, 251-256),
// the consumed instance / witness values re-emitted in consumption order, messages cut every 100 000 gates / values
// (builder.rs:45-49, 79-100).  In flatten mode Program records copies as values, so a value handle IS that wire id.
// --------------------------------------------------------------------------------------------------
namespace {

std::vector<uint8_t> minimal_le(const uint8_t* p, size_t n) {  // BigUint::to_bytes_le: no trailing zeros, zero is [0]
    while (n > 0 && p[n - 1] == 0) n--;
    if (n == 0) return std::vector<uint8_t>{0};
    return std::vector<uint8_t>(p, p + n);
}

std::vector<uint8_t> const_bytes(const Program& p, uint32_t idx) {
    if (p.const_unreduced[idx]) return minimal_le(p.const_raw[idx].data(), p.const_raw[idx].size());
    const int N = std::max(p.nlimb, 1);
    std::vector<uint8_t> b((size_t)N * 4);
    for (int k = 0; k < N; k++) {
        uint32_t w = p.const_limbs[(size_t)idx * N + k];
        memcpy(&b[(size_t)k * 4], &w, 4);
    }
    return minimal_le(b.data(), b.size());
}

constexpr size_t kMaxLen = 100 * 1000;  // MessageBuilder::max_len

}  // namespace

static int flatten_statement(zkb_evaluator* ev, std::vector<uint8_t>& inst_out, std::vector<uint8_t>& wit_out,
                             std::vector<uint8_t>& rel_out) {
    Program& p = ev->prog();
    if (!p.keep_copies) return ev->fail(ZKB_E_ARG, "zkb_evaluator_set_flatten(ev, 1) must be called before ingesting");
    if (ev->fatal) return ev->fail(ZKB_E_FATAL, ev->err);
    inst_out.clear();
    wit_out.clear();
    rel_out.clear();
    if (!p.field_set) return ZKB_OK;  // no relation reached the backend: the builder was never created
    ir::Header h;
    h.version = "1.0.0";  // IR_VERSION, structs/mod.rs:36
    h.field_characteristic = p.modulus_le;
    h.field_degree = 1;
    ir::Message inst, wit, rel;
    inst.type = ir::MSG_INSTANCE;
    wit.type = ir::MSG_WITNESS;
    rel.type = ir::MSG_RELATION;
    inst.header = wit.header = rel.header = h;
    rel.gate_mask = ev->c->is_boolean ? ir::M_BOOL : ir::M_ARITH;
    rel.feat_mask = ir::M_SIMPLE;
    auto append = [](std::vector<uint8_t>& out, const ir::Message& m) {
        std::vector<uint8_t> b = ir::write_message(m);
        out.insert(out.end(), b.begin(), b.end());
    };
    auto push_gate = [&](const ir::Gate& g) {
        rel.gates.push_back(g);
        if (rel.gates.size() >= kMaxLen) {
            append(rel_out, rel);
            rel.gates.clear();
            rel.consts.clear();
        }
    };
    auto add_const = [&](std::vector<uint8_t>&& b) {
        rel.consts.push_back(std::move(b));
        return (uint32_t)rel.consts.size() - 1;
    };
    const uint32_t n = p.n_values();
    size_t ai = 0;
    for (uint32_t v = 0; v <= n; v++) {
        for (; ai < p.asserts.size() && p.asserts[ai].pos == v; ai++) {
            ir::Gate g;
            g.type = ir::G_ASSERT_ZERO;
            g.w0 = p.asserts[ai].value;
            push_gate(g);
        }
        if (v == n) break;
        ir::Gate g;
        g.w0 = v;
        const uint32_t a = p.opa[v], b = p.opb[v];
        switch (p.kind[v]) {
            case V_CONST: g.type = ir::G_CONSTANT; g.const_idx = add_const(const_bytes(p, b)); break;
            case V_INSTANCE: {
                g.type = ir::G_INSTANCE;
                const auto& val = ev->instance_values[b];
                inst.values.push_back(minimal_le(val.data(), val.size()));
                if (inst.values.size() == kMaxLen) {
                    append(inst_out, inst);
                    inst.values.clear();
                }
            } break;
            case V_WITNESS: {
                g.type = ir::G_WITNESS;
                if (b == kNoWitnessValue) break;  // witness(None): gate only
                const auto& val = ev->witness_values[b];
                wit.values.push_back(minimal_le(val.data(), val.size()));
                if (wit.values.size() == kMaxLen) {
                    append(wit_out, wit);
                    wit.values.clear();
                }
            } break;
            case V_ADD: g.type = ir::G_ADD; g.w1 = a; g.w2 = b; break;
            case V_MUL: g.type = ir::G_MUL; g.w1 = a; g.w2 = b; break;
            case V_AND: g.type = ir::G_AND; g.w1 = a; g.w2 = b; break;
            case V_XOR: g.type = ir::G_XOR; g.w1 = a; g.w2 = b; break;
            case V_ADDC: g.type = ir::G_ADD_CONSTANT; g.w1 = a; g.const_idx = add_const(const_bytes(p, b)); break;
            case V_MULC: g.type = ir::G_MUL_CONSTANT; g.w1 = a; g.const_idx = add_const(const_bytes(p, b)); break;
            case V_NOT: g.type = ir::G_NOT; g.w1 = a; break;
            case V_COPY: g.type = ir::G_COPY; g.w1 = a; break;
            default: return ev->fail(ZKB_E_ARG, "corrupt program");
        }
        push_gate(g);
    }
    // MessageBuilder::finish, builder.rs:124-135
    if (!inst.values.empty()) append(inst_out, inst);
    if (!wit.values.empty()) append(wit_out, wit);
    if (!rel.gates.empty()) append(rel_out, rel);
    return ZKB_OK;
}

// reader -> owned structs -> writer, for round-trip tests of the two halves (any message kind, any gate)
extern "C" int zkb_debug_rewrite_message(zkb_ctx* c, const uint8_t* buf, size_t len, const uint8_t** out, size_t* out_len) {
    static thread_local std::vector<uint8_t> scratch;
    ir::Message m;
    std::string e;
    if (!ir::read_message(buf, len, m, e)) return c->fail(ZKB_E_FORMAT, e);
    scratch = ir::write_message(m);
    *out = scratch.data();
    *out_len = scratch.size();
    return ZKB_OK;
}

// zkb_gate[] -> a SIMPLE relation as size-prefixed messages of at most 100 000 gates (what a GateBuilder over a
// MemorySink produces for the same gate list, builder.rs:93-98); workload generator for large `.sieve` inputs
extern "C" int zkb_debug_write_flat_relation(zkb_ctx* c, const uint8_t* modulus_le, size_t modulus_len, int is_boolean,
                                             const zkb_gate* gates, uint64_t n_gates, const uint8_t* const_pool_le, size_t const_stride,
                                             uint64_t n_consts, const uint8_t** out, size_t* out_len) {
    static thread_local std::vector<uint8_t> scratch;
    scratch.clear();
    ir::Message rel;
    rel.type = ir::MSG_RELATION;
    rel.header.version = "1.0.0";
    rel.header.field_characteristic.assign(modulus_le, modulus_le + modulus_len);
    rel.header.field_degree = 1;
    rel.gate_mask = is_boolean ? ir::M_BOOL : ir::M_ARITH;
    rel.feat_mask = ir::M_SIMPLE;
    auto flush = [&]() {
        std::vector<uint8_t> b = ir::write_message(rel);
        scratch.insert(scratch.end(), b.begin(), b.end());
        rel.gates.clear();
        rel.consts.clear();
    };
    for (uint64_t i = 0; i < n_gates; i++) {
        const zkb_gate& g = gates[i];
        ir::Gate o;
        o.type = g.op;
        switch (g.op) {
            case ZKB_G_CONSTANT: case ZKB_G_ADD_CONSTANT: case ZKB_G_MUL_CONSTANT: {
                if (g.b >= n_consts) return c->fail(ZKB_E_ARG, "constant index out of range");
                const uint8_t* v = const_pool_le + (size_t)g.b * const_stride;
                size_t n = const_stride;
                while (n > 1 && v[n - 1] == 0) n--;
                rel.consts.emplace_back(v, v + n);
                o.const_idx = (uint32_t)rel.consts.size() - 1;
                o.w0 = g.out;
                o.w1 = g.a;
            } break;
            case ZKB_G_ASSERT_ZERO: o.w0 = g.a; break;
            case ZKB_G_COPY: case ZKB_G_NOT: o.w0 = g.out; o.w1 = g.a; break;
            case ZKB_G_ADD: case ZKB_G_MUL: case ZKB_G_AND: case ZKB_G_XOR: o.w0 = g.out; o.w1 = g.a; o.w2 = g.b; break;
            case ZKB_G_INSTANCE: case ZKB_G_WITNESS: o.w0 = g.out; break;
            case ZKB_G_FREE: o.w0 = g.a; o.w1 = g.b; o.has_last = g.b != g.a; break;
            default: return c->fail(ZKB_E_ARG, "unknown gate opcode");
        }
        rel.gates.push_back(o);
        if (rel.gates.size() >= kMaxLen) flush();
    }
    if (!rel.gates.empty() || n_gates == 0) flush();
    *out = scratch.data();
    *out_len = scratch.size();
    return ZKB_OK;
}

extern "C" int zkb_evaluator_set_flatten(zkb_evaluator* ev, int on) {
    if (ev->batch()) return ev->fail(ZKB_E_ARG, "value sets need an evaluating backend (not flatten / expand-definable)");
    if (ev->prog().n_values() > 0) return ev->fail(ZKB_E_ARG, "flatten mode must be chosen before anything is recorded");
    ev->prog().keep_copies = on != 0;
    return ZKB_OK;
}

// `zki_sieve expand-definable --gate-set <s>` (cli.rs:513-553): ExpandDefinable wraps the flattener
extern "C" int zkb_evaluator_set_expand_definable(zkb_evaluator* ev, const char* gate_set) {
    if (ev->batch()) return ev->fail(ZKB_E_ARG, "value sets need an evaluating backend (not flatten / expand-definable)");
    if (ev->prog().n_values() > 0) return ev->fail(ZKB_E_ARG, "expand-definable must be chosen before anything is recorded");
    uint16_t mask = 0;
    std::string e;
    if (!ir::parse_gate_set(gate_set ? gate_set : "", mask, e)) return ev->fail(ZKB_E_SEMANTIC, e);  // relation.rs:144-167
    ev->prog().keep_copies = true;
    ev->prog().expand_on = true;
    ev->prog().expand_mask = mask;
    return ZKB_OK;
}

extern "C" int zkb_evaluator_flatten(zkb_evaluator* ev, const uint8_t** instance, size_t* instance_len, const uint8_t** witness,
                                     size_t* witness_len, const uint8_t** relation, size_t* relation_len) {
    int rc = flatten_statement(ev, ev->flat_out[0], ev->flat_out[1], ev->flat_out[2]);
    if (rc != ZKB_OK) return rc;
    const uint8_t** ptr[3] = {instance, witness, relation};
    size_t* len[3] = {instance_len, witness_len, relation_len};
    for (int i = 0; i < 3; i++) {
        if (ptr[i]) *ptr[i] = ev->flat_out[i].data();
        if (len[i]) *len[i] = ev->flat_out[i].size();
    }
    return ZKB_OK;
}

// FilesSink::new_clean + the three conventional file names (producers/sink.rs:67-104, 139-153)
extern "C" int zkb_evaluator_flatten_to_dir(zkb_evaluator* ev, const char* out_dir) {
    std::string dir = out_dir;
    if (has_sieve_ext(dir)) return ev->fail(ZKB_E_ARG, "IR flattening requires a directory as output value");  // cli.rs:459-460
    int rc = flatten_statement(ev, ev->flat_out[0], ev->flat_out[1], ev->flat_out[2]);
    if (rc != ZKB_OK) return rc;
    std::string acc;
    for (size_t i = 0; i <= dir.size(); i++) {  // create_dir_all
        if (i == dir.size() || dir[i] == '/') {
            if (!acc.empty()) mkdir(acc.c_str(), 0777);
        }
        if (i < dir.size()) acc.push_back(dir[i]);
    }
    if (DIR* d = opendir(dir.c_str())) {  // clean_workspace: remove existing *.sieve
        while (dirent* e = readdir(d)) {
            std::string full = dir + "/" + e->d_name;
            if (has_sieve_ext(full)) remove(full.c_str());
        }
        closedir(d);
    } else {
        return ev->fail(ZKB_E_ARG, "cannot create directory " + dir);
    }
    const char* names[3] = {"000_instance.sieve", "001_witness.sieve", "002_relation.sieve"};
    for (int i = 0; i < 3; i++) {
        std::string path = dir + "/" + names[i];
        FILE* fp = fopen(path.c_str(), "wb");
        if (!fp) return ev->fail(ZKB_E_ARG, "cannot write " + path);
        size_t n = ev->flat_out[i].size();
        if (n && fwrite(ev->flat_out[i].data(), 1, n, fp) != n) {
            fclose(fp);
            return ev->fail(ZKB_E_ARG, "short write to " + path);
        }
        fclose(fp);
    }
    return ZKB_OK;
}

// --------------------------------------------------------------------------------------------------
// Source: file discovery and ordering, rust/src/consumers/source.rs:64-89, 165-193
// --------------------------------------------------------------------------------------------------
static bool has_sieve_ext(const std::string& p) {
    size_t slash = p.find_last_of('/');
    std::string name = slash == std::string::npos ? p : p.substr(slash + 1);
    size_t dot = name.find_last_of('.');
    return dot != std::string::npos && dot > 0 && name.substr(dot + 1) == "sieve";
}

namespace zkb {
int list_workspace_files(const char* const* paths, size_t n, std::vector<std::string>& out, std::string& err) {
    for (size_t i = 0; i < n; i++) {
        std::string p = paths[i];
        if (has_sieve_ext(p)) {
            out.push_back(p);
        } else if (p == "-") {
            if (n > 1) {  // source.rs:170-173
                err = "Cannot combine files and stdin";
                return ZKB_E_ARG;
            }
            out.push_back(p);  // BufferSource::Stdin, source.rs:69-71
        } else {
            DIR* d = opendir(p.c_str());
            if (!d) {
                err = "cannot read directory " + p;
                return ZKB_E_ARG;
            }
            while (dirent* e = readdir(d)) {
                std::string name = e->d_name;
                std::string full = p + (p.size() && p.back() == '/' ? "" : "/") + name;
                if (has_sieve_ext(full)) out.push_back(full);
            }
            closedir(d);
        }
    }
    // from_filenames: lexical sort, then a STABLE sort on instance < witness < relation < other
    std::sort(out.begin(), out.end());
    auto key = [](const std::string& p) {
        size_t slash = p.find_last_of('/');
        std::string name = slash == std::string::npos ? p : p.substr(slash + 1);
        if (name.find("instance") != std::string::npos) return 0;
        if (name.find("witness") != std::string::npos) return 1;
        if (name.find("relation") != std::string::npos) return 3;
        return 4;
    };
    std::stable_sort(out.begin(), out.end(), [&](const std::string& a, const std::string& b) { return key(a) < key(b); });
    return ZKB_OK;
}

}  // namespace zkb

extern "C" zkb_evaluator* zkb_evaluator_create(zkb_ctx* backend) { return new zkb_evaluator(backend); }
extern "C" void zkb_evaluator_destroy(zkb_evaluator* ev) { delete ev; }
extern "C" const char* zkb_evaluator_last_error(zkb_evaluator* ev) { return ev->err.c_str(); }

extern "C" int zkb_evaluator_ingest_message(zkb_evaluator* ev, const uint8_t* buf, size_t len) { return ev->ingest_bytes(buf, len); }

// FlatBuffers -> owned structs is the expensive half of ingestion (about 80 % for flat relations) and messages
// are independent of each other there, so a large buffer (a builder-produced relation arrives as one message per
// 100 000 gates) is parsed by a small thread pool, one window of messages at a time; flattening / recording then
// consumes the parsed messages strictly in order, so errors surface exactly where the serial loop would meet them
// (a malformed message is fatal when it is reached: Evaluator::from_messages unwraps it, evaluator.rs:193).
static unsigned parse_threads() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("ZKB_PARSE_THREADS");
        unsigned hw = std::thread::hardware_concurrency();
        v = e ? atoi(e) : (int)std::min(16u, hw ? hw : 1u);
        if (v < 1) v = 1;
    }
    return (unsigned)v;
}

extern "C" int zkb_evaluator_ingest_buffer(zkb_evaluator* ev, const uint8_t* buf, size_t len) {
    NvtxRange r_ing("zkb:host_parse_flatten");
    std::vector<std::pair<size_t, size_t>> msgs;
    ir::split_messages(buf, len, msgs);
    const unsigned T = parse_threads();
    static const size_t min_bytes = getenv("ZKB_PARALLEL_INGEST_MIN_BYTES") ? (size_t)atoll(getenv("ZKB_PARALLEL_INGEST_MIN_BYTES")) : ((size_t)1 << 20);
    if (T < 2 || msgs.size() < 2 || len < min_bytes) {
        for (auto& m : msgs) {
            int rc = ev->ingest_bytes(buf + m.first, m.second);
            if (rc != ZKB_OK) return rc;
        }
        return ZKB_OK;
    }
    const size_t window = (size_t)T * 4;
    double t_parse = 0, t_ing = 0;
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_flat = 0;
    size_t n_flat = 0;
    for (size_t w0 = 0, next_w0 = 0; w0 < msgs.size(); w0 = next_w0) {
        double ta = now();
        size_t w1 = std::min(msgs.size(), w0 + window);
        size_t serial_n = 0;
        const size_t done = ev->ingest_flat_window(buf, msgs, w0, w1, T, &serial_n);  // flat relation messages: from the tables in place
        if (done) {
            t_flat += now() - ta;
            n_flat += done;
            next_w0 = w0 + done;
            continue;
        }
        w1 = w0 + serial_n;
        next_w0 = w1;
        std::vector<ir::Message> parsed(w1 - w0);
        std::vector<std::string> errs(w1 - w0);
        std::vector<char> ok(w1 - w0, 0);
        std::atomic<size_t> next{w0};
        auto work = [&]() {
            for (size_t i; (i = next.fetch_add(1)) < w1;)
                ok[i - w0] = ir::read_message(buf + msgs[i].first, msgs[i].second, parsed[i - w0], errs[i - w0]) ? 1 : 0;
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < T && t < w1 - w0; t++) pool.emplace_back(work);
        work();
        for (auto& th : pool) th.join();
        double tb = now();
        t_parse += tb - ta;
        for (size_t i = w0; i < w1; i++) {
            if (!ok[i - w0]) {
                ev->fatal = true;
                return ev->fail(ZKB_E_FORMAT, errs[i - w0]);
            }
            int rc = ev->ingest_parsed(parsed[i - w0]);
            if (rc != ZKB_OK) return rc;
            parsed[i - w0] = ir::Message();  // release the owned structs as soon as they are recorded
        }
        t_ing += now() - tb;
    }
    if (getenv("ZKB_TIMING")) fprintf(stderr, "flat windows %.3f s (%zu of %zu messages), parse %.3f s ingest %.3f s\n", t_flat, n_flat, msgs.size(), t_parse, t_ing);
    return ZKB_OK;
}

extern "C" int zkb_evaluator_ingest_paths(zkb_evaluator* ev, const char* const* paths, size_t n_paths) {
    std::vector<std::string> files;
    std::string e;
    int rc = zkb::list_workspace_files(paths, n_paths, files, e);
    if (rc != ZKB_OK) return ev->fail(rc, e);
    for (const auto& f : files) {
        zkb::FileBytes data;
        if (!data.open(f)) {
            fprintf(stderr, "Warning: failed to open file %s\n", f.c_str());  // source.rs:132
            continue;
        }
        rc = zkb_evaluator_ingest_buffer(ev, data.data, data.size);
        if (rc != ZKB_OK) return rc;
    }
    return ZKB_OK;
}

extern "C" int zkb_evaluator_get_violations(zkb_evaluator* ev, size_t* n) {
    if (ev->batch()) return ev->fail(ZKB_E_ARG, "the evaluator holds value sets: use zkb_evaluator_batch_result");
    int rc = ev->finish();
    if (rc != ZKB_OK) return rc;
    *n = ev->violations.size();
    return ZKB_OK;
}

extern "C" const char* zkb_evaluator_violation(zkb_evaluator* ev, size_t i) {
    return i < ev->violations.size() ? ev->violations[i].c_str() : nullptr;
}

extern "C" int zkb_evaluator_get_wire(zkb_evaluator* ev, uint64_t wire_id, uint8_t* out, size_t cap, size_t* len) {
    if (ev->batch()) return ev->fail(ZKB_E_ARG, "the evaluator holds value sets: use zkb_evaluator_get_wire_of");
    int rc = ev->finish();
    if (rc != ZKB_OK) return rc;
    uint32_t v = ev->values.get(wire_id);
    if (v == Scope::kNone) return ev->fail(ZKB_E_SEMANTIC, "No value given for wire_" + u64s(wire_id));  // :750-752, 787-791
    zkb_wire w = v;
    memset(out, 0, cap);
    rc = zkb_read_values(ev->c, 0, &w, 1, out, cap);
    if (rc != ZKB_OK) return ev->fail(rc, ev->c->err);
    size_t n = cap;
    while (n > 1 && out[n - 1] == 0) n--;
    if (len) *len = n;
    return ZKB_OK;
}

extern "C" int zkb_evaluator_lookup(zkb_evaluator* ev, uint64_t wire_id, zkb_wire* out) {
    uint32_t v = ev->values.get(wire_id);
    if (v == Scope::kNone) return ev->fail(ZKB_E_SEMANTIC, "No value given for wire_" + u64s(wire_id));
    *out = v;
    return ZKB_OK;
}

// ---- value sets (batch mode) ------------------------------------------------------------------------------------------
extern "C" int zkb_evaluator_add_value_set_buffer(zkb_evaluator* ev, const uint8_t* buf, size_t len) {
    int rc = ev->add_value_set_begin();
    if (rc != ZKB_OK) return rc;
    return ev->add_value_set_end(ev->add_value_set_bytes(buf, len, "value set " + u64s(ev->sets.size() - 1)));
}

extern "C" int zkb_evaluator_add_value_set_paths(zkb_evaluator* ev, const char* const* paths, size_t n_paths) {
    std::vector<std::string> files;
    std::string e;
    int rc = zkb::list_workspace_files(paths, n_paths, files, e);
    if (rc != ZKB_OK) return ev->fail(rc, e);
    if ((rc = ev->add_value_set_begin()) != ZKB_OK) return rc;
    for (const auto& f : files) {
        zkb::FileBytes data;
        if (!data.open(f)) {
            rc = ev->fail(ZKB_E_ARG, "cannot read " + f);
            break;
        }
        if ((rc = ev->add_value_set_bytes(data.data, data.size, f)) != ZKB_OK) break;
    }
    return ev->add_value_set_end(rc);
}

extern "C" size_t zkb_evaluator_value_sets(zkb_evaluator* ev) { return ev->sets.size(); }

extern "C" int zkb_evaluator_use_devices(zkb_evaluator* ev, zkb_ctx** ctxs, int n) {
    if (!ctxs || n < 1 || ctxs[0] != ev->c) return ev->fail(ZKB_E_ARG, "zkb_evaluator_use_devices: ctxs[0] must be the evaluator's backend");
    if (ev->batch_evaluated) return ev->fail(ZKB_E_ARG, "the batch has already been evaluated");
    for (int i = 0; i < n; i++) {
        int rank = -1, size = 0;
        if (!ctxs[i] || zkb_comm_info(ctxs[i], &rank, &size, nullptr, nullptr) != ZKB_OK || rank != i || size != n)
            return ev->fail(ZKB_E_ARG, "zkb_evaluator_use_devices: pass the contexts of one communicator in the order given to zkb_comm_init");
    }
    ev->devices.assign(ctxs, ctxs + n);
    return ZKB_OK;
}

static int batch_ready(zkb_evaluator* ev, uint64_t set) {
    if (!ev->batch()) return ev->fail(ZKB_E_ARG, "no value set has been added");
    if (set >= ev->sets.size()) return ev->fail(ZKB_E_ARG, "value set index " + u64s(set) + " out of range (" + u64s(ev->sets.size()) + " sets)");
    return ev->evaluate_batch();
}

extern "C" int zkb_evaluator_batch_result(zkb_evaluator* ev, uint64_t set, int* status, size_t* n_violations) {
    int rc = batch_ready(ev, set);
    if (rc != ZKB_OK) return rc;
    if (status) *status = ev->set_status[set];
    if (n_violations) *n_violations = ev->set_violations[set].size();
    return ZKB_OK;
}

extern "C" const char* zkb_evaluator_batch_violation(zkb_evaluator* ev, uint64_t set, size_t i) {
    if (!ev->batch_evaluated || set >= ev->set_violations.size() || i >= ev->set_violations[set].size()) return nullptr;
    return ev->set_violations[set][i].c_str();
}

extern "C" int zkb_evaluator_get_wire_of(zkb_evaluator* ev, uint64_t set, uint64_t wire_id, uint8_t* out, size_t cap, size_t* len) {
    int rc = batch_ready(ev, set);
    if (rc != ZKB_OK) return rc;
    if (ev->set_status[set] != ZKB_OK) return ev->fail(ev->set_status[set], ev->set_violations[set][0]);
    // The top scope is the one the whole recording left.  A set whose streams run out earlier stops at its cut, where its
    // own statement's scope can differ (wires freed or bound after the cut): its wires are not answered from this scope.
    if (ev->set_cut[set] != UINT32_MAX)
        return ev->fail(ZKB_E_ARG, "value set " + u64s(set) + " stops recording before the relation ends: wire values are read for sets recorded in full");
    uint32_t v = ev->values.get(wire_id);
    if (v == Scope::kNone) return ev->fail(ZKB_E_SEMANTIC, "No value given for wire_" + u64s(wire_id));
    uint32_t idx = 0;
    zkb_ctx* owner = ev->owner_of(set, idx);
    zkb_wire w = v;
    memset(out, 0, cap);
    rc = zkb_read_values(owner, idx, &w, 1, out, cap);
    if (rc != ZKB_OK) return ev->fail(rc, owner->err);
    size_t n = cap;
    while (n > 1 && out[n - 1] == 0) n--;
    if (len) *len = n;
    return ZKB_OK;
}

// stream cut of a value set, from the recording alone (no device): *what 0 none, 1 its instance stream runs out, 2 its witness
// stream runs out, 3 the recording's own error or panic; *seq the assertions recorded before that point
extern "C" int zkb_debug_value_set_cut(zkb_evaluator* ev, uint64_t set, uint64_t* seq, int* what) {
    if (set >= ev->sets.size()) return ev->fail(ZKB_E_ARG, "value set index " + u64s(set) + " out of range (" + u64s(ev->sets.size()) + " sets)");
    const std::vector<uint8_t> w = ev->compute_cuts();
    *what = w[set];
    *seq = w[set] ? ev->seq_before(ev->set_cut[set]) : UINT64_MAX;
    return ZKB_OK;
}
