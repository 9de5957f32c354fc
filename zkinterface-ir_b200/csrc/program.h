// Host-side recorded program and its levelized device plan.
//
// `Program` is the recording half of the deferred backend: every ZKBackend
// callback of the reference (rust/src/consumers/evaluator.rs:17-76) appends one
// SSA value instead of computing it — the same idea as the reference's own
// `IRFlattener` (rust/src/consumers/flattening.rs:83-190).  `copy` is an alias
// (no value is created: the copy of a wire has, by definition, the same value).
//
// `Plan` is the host-preparation pass of BASELINE.json:north_star: ASAP
// levelization of the SSA list into wavefronts, per-level sorting by opcode,
// slot assignment in level order (so every level writes one contiguous slot
// range), and fusion of AssertZero into the producing gate.
#pragma once
#include <stdint.h>

#include <string>
#include <unordered_map>
#include <vector>

#include "bigu.h"
#include "field.cuh"

namespace zkb {

// SSA value kinds (what produced the value)
enum ValKind : uint8_t {
    V_CONST = 0,   // b = const-pool index
    V_INSTANCE,    // b = index in the instance stream
    V_WITNESS,     // b = index in the witness stream
    V_ADD,
    V_MUL,
    V_ADDC,  // b = const-pool index
    V_MULC,  // b = const-pool index
    V_AND,
    V_XOR,
    V_NOT,
    V_COPY,  // only recorded in flatten mode (Program::keep_copies); otherwise a copy is an alias
    V_CALLOUT,  // output of a call group (below); never stored in Program::kind — such values have implicit handles
    V_KINDS
};

// ---- loop-structured recording (SURVEY.md section 8a rows 8 / 12, config C5) ---------------------------------------------
// A For loop whose body is a call of a plain named function, with iterator expressions affine in the loop variable and
// inputs that exist before the loop, is n_calls runs of one small straight-line program over affinely moving operands.
// Instead of n_calls x |body| SSA values and as many 16-byte device descriptors, the Program keeps the body ONCE (a
// Template: register-to-register ops, registers = outputs, inputs, locals as in the function's own wire numbering) and one
// CallGroup per loop execution; only the calls' OUTPUTS become SSA values, because only they can be named by later gates —
// the locals of a call die with its scope (evaluator.rs:698-746).  Those outputs are IMPLICIT values: handle =
// kCalloutBit | index, indices handed out consecutively (call c, output k of a group: first_callout + c * n_out + k), no
// entry in kind / opa / opb, wavefront 0, slot = Plan::callout_slot0 + index, always stored and readable — so neither the
// recorder nor the levelizer does any per-output work (C5: 2^24 outputs of 2^23 calls).  The device expands a group
// inside one kernel, every call's locals living in registers (kernels.cu: k_bool_groups).
constexpr uint32_t kCalloutBit = 0x80000000u;
constexpr uint32_t kMaxCallouts = 0x7FFFFF00u;
inline bool is_callout(uint32_t h) { return (h & kCalloutBit) != 0; }  // (Scope::kNone has the bit too: test it first)
inline uint32_t callout_index(uint32_t h) { return h & ~kCalloutBit; }
// Over a prime field a loop qualifies only with at least kArithGroupMinCalls calls: below that the gate-by-gate recording
// is small and one launch per depth costs more than it saves.  Its body may hold AssertZero (TmplOp kind T_ASSERT); a call's
// k-th assertion has the sequence number seq0 + call * n_asserts + k, which is the unrolled loop's program order.
constexpr uint64_t kArithGroupMinCalls = 1024;
constexpr uint8_t T_ASSERT = 0xF0;  // template-only op kind: AssertZero on register a, b = its ordinal k inside the body
// AssertRec::value of an assertion inside a call group: the asserted value is a call-local wire that has no handle
constexpr uint32_t kGroupAssertValue = 0xFFFFFFFFu;
struct TmplOp {       // 8 bytes
    uint8_t kind;     // ValKind: V_CONST (b = const-pool index), V_ADD, V_MUL, V_ADDC / V_MULC (b = const-pool index), V_AND, V_XOR, V_NOT;
                      // T_ASSERT (prime fields)
    uint8_t dst;      // register written
    uint8_t a;        // register read
    uint8_t pad;
    uint32_t b;       // register read (two-input ops) or const-pool index
};
struct Template {
    uint32_t n_out = 0, n_in = 0, n_regs = 0;
    std::vector<TmplOp> ops;
    uint64_t cb[12] = {0};   // callbacks one call makes, by CbKind (copies of the inputs and outputs included)
    uint64_t ir_gates = 0;
    uint64_t n_two = 0, n_one = 0;  // two-input / one-input value gates (algorithmic bytes, SURVEY.md section 8d)
    std::vector<uint64_t> assert_wire;  // per AssertZero of the body, in order: its local wire id (what a violation names)
};
struct CallGroup {
    uint32_t tmpl = 0;
    uint32_t n_calls = 0;
    uint32_t first_callout = 0;  // index of output 0 of call 0; call c, output k is first_callout + c * n_out + k
    uint32_t depth = 0;        // 0: reads input values only; d: reads outputs of groups of depth < d as well
    std::vector<uint32_t> in_base, in_stride;  // per input position: handle of call c's input = base + stride * c
    uint32_t n_out = 0;
    uint32_t seq0 = 0;  // assertion sequence number of call 0's first AssertZero (templates with assertions)
};

// callback counters (one per ZKBackend method that the Evaluator drives)
enum CbKind { CB_CONSTANT = 0, CB_INSTANCE, CB_WITNESS, CB_ADD, CB_MUL, CB_ADDC, CB_MULC, CB_AND, CB_XOR,
              CB_NOT, CB_COPY, CB_ASSERT_ZERO, CB_KINDS };

// device opcodes (GateOp.meta & 0xff)
enum DevOp : uint32_t { D_ADD = 0, D_MUL, D_ADDC, D_MULC, D_AND, D_XOR, D_NOT, D_ASSERT, D_OPS };
constexpr uint32_t F_ASSERT = 1u << 8;    // result must be zero; assert seq in Plan::op_assert_seq
constexpr uint32_t F_NOSTORE = 1u << 9;   // value is consumed by nothing but the fused assert
constexpr uint32_t F_RAW = 1u << 10;      // operand a is an input value: consult its "raw value >= p" flag (trap 1)
constexpr uint32_t F_RAWB = 1u << 11;     // operand b (of And / Xor) is an input value: likewise
// stored, but no gate reads it (a live wire nothing consumes, an observable assertion sum): only a read-back needs the
// store, so a tile that is overwritten by the next one may skip it (TileGeom::skip_mask)
constexpr uint32_t F_SINK = 1u << 12;
constexpr uint32_t kNoSeq = 0xFFFFFFFFu;
constexpr uint32_t kNoSlot = 0xFFFFFFFFu;

struct GateOp {  // 16 bytes, one per device gate
    uint32_t a;     // operand slot
    uint32_t b;     // operand slot, or const-pool index for ADDC/MULC
    uint32_t out;   // destination slot
    uint32_t meta;  // DevOp | flags
};

struct AssertRec {
    uint32_t value;     // asserted SSA value
    uint32_t pos;       // number of SSA values recorded before it (program position)
    uint64_t src_wire;  // local-scope wire id of the AssertZero gate (evaluator.rs:357-362)
};

// Device form of a call group: thread <-> (call, witness word).  An operand's slot is base + stride * call, or — when the
// slots the plan gave the input values are not an arithmetic progression — table[base + call] (stride == kTableStride).
constexpr uint32_t kMaxGroupInputs = 8;
constexpr uint32_t kMaxTemplateRegs = 48;
constexpr uint32_t kMaxTemplateOps = 128;
constexpr uint32_t kTableStride = 0xFFFFFFFFu;
struct GroupDesc {  // 16-byte aligned
    uint32_t tmpl_off;   // first op of the template in the op array
    uint32_t n_ops;
    uint32_t n_out, n_in;
    uint32_t n_calls;
    uint32_t out_slot;   // slot of output 0 of call 0; outputs are consecutive slots
    uint32_t first_call; // calls of the groups before this one in the same launch (prefix sum: thread -> group search)
    uint32_t pad;        // prime fields: CallGroup::seq0 (0 for p = 2)
    uint32_t in_base[kMaxGroupInputs];
    uint32_t in_stride[kMaxGroupInputs];
};
// A template op as the device interpreter wants it (32 bytes, two 16-byte loads, no decoding and no branch): byte offsets of
// the registers in the CTA's shared-memory register file (register r of thread t at (r * kGroupThreads + t) * 4), and the
// op as four masks of one bitwise form,  r = (a & b & m_and) ^ ((a ^ b) & m_xor) ^ (a & m_a) ^ m_c :
//   Xor / Add: m_xor = ~0;  And / Mul: m_and = ~0;  Not: m_a = m_c = ~0;  AddConstant c: m_a = ~0, m_c = -c;
//   MulConstant c: m_a = -c;  Constant c: m_c = -c   (c = the constant mod 2; one-input ops read a twice)
constexpr uint32_t kGroupThreads = 256;
// fwd: bit 0 / bit 1 = operand a / b is the result of the previous op, which the interpreter still holds in registers (5 of the
// 16 operand reads of C5's body): no shared-memory load for it
//
// Over a prime field (kernels.cu: k_arith_groups) the same 32 bytes carry register NUMBERS (the kernel picks the CTA size,
// hence the layout of the register file, at launch) and the op itself:
//   dst_off, a_off, b_off = registers, fwd as above, m_and = AG_* kind, m_xor = const-pool index (AG_CONST / AG_ADDC /
//   AG_MULC), m_a = the assertion's ordinal k in the body (AG_ASSERT), m_c = assertions per call (AG_ASSERT)
struct GroupOp {
    uint32_t dst_off, a_off, b_off, fwd;
    uint32_t m_and, m_xor, m_a, m_c;
};
enum ArithGroupKind : uint32_t { AG_ADD = 0, AG_MUL, AG_ADDC, AG_MULC, AG_CONST, AG_ASSERT };
constexpr uint32_t kGroupHintShift = 7;  // Plan::group_hints: one entry per 128 calls of a launch

struct InputLoad {  // level-0 values: filled by the input kernel on every pass
    uint32_t slot;
    uint32_t kind;   // V_CONST / V_INSTANCE / V_WITNESS
    uint32_t index;  // const-pool index or stream index
    uint32_t pad;
};

class Program {
public:
    // ---- field -----------------------------------------------------------
    bool field_set = false;
    std::vector<uint8_t> modulus_le;  // as given (trailing zeros kept)
    BigU modulus;
    bool binary = false;  // p == 2: bit-sliced device path
    int nlimb = 0;
    FieldParams fp{};

    // PlaintextBackend::set_field, evaluator.rs:866-875 (+ device limits)
    bool set_field(const uint8_t* mod_le, size_t len, uint32_t degree, std::string& err);

    // ---- recording -------------------------------------------------------
    std::vector<uint8_t> kind;
    std::vector<uint32_t> opa, opb;
    std::vector<AssertRec> asserts;
    uint64_t cb_count[CB_KINDS] = {0};
    uint64_t ir_gates = 0;  // Add/Mul/AddC/MulC/And/Xor/Not/AssertZero IR gates ingested (metric numerator)
    uint32_t n_instance = 0, n_witness = 0;

    // const pool: canonical residues (< p), nlimb limbs each; unreduced inputs remembered raw
    std::vector<uint32_t> const_limbs;
    std::vector<uint8_t> const_unreduced;                 // 1 if the raw constant was >= p
    std::vector<std::vector<uint8_t>> const_raw;          // raw bytes (only kept when unreduced)
    std::unordered_map<std::string, uint32_t> const_index;
    uint32_t n_consts() const { return (uint32_t)const_unreduced.size(); }
    uint32_t intern_const(const uint8_t* le, size_t n);

    std::vector<Template> templates;
    std::vector<CallGroup> groups;  // ascending first_callout
    uint32_t n_callouts = 0;
    uint64_t n_total_values() const { return (uint64_t)kind.size() + n_callouts; }
    bool valid_handle(uint64_t h) const { return h < kind.size() || (h >= kCalloutBit && h - kCalloutBit < n_callouts); }
    // the group whose outputs include callout index i
    const CallGroup& group_of_callout(uint32_t i) const {
        size_t lo = 0, hi = groups.size();
        while (hi - lo > 1) {
            const size_t mid = (lo + hi) / 2;
            if (groups[mid].first_callout <= i) lo = mid;
            else hi = mid;
        }
        return groups[lo];
    }

    uint32_t n_values() const { return (uint32_t)kind.size(); }
    uint32_t push_value(uint8_t k, uint32_t a, uint32_t b) {
        kind.push_back(k);
        opa.push_back(a);
        opb.push_back(b);
        return (uint32_t)kind.size() - 1;
    }
    // ZKBackend-shaped recording methods
    uint32_t constant(const uint8_t* le, size_t n) { cb_count[CB_CONSTANT]++; return push_value(V_CONST, 0, intern_const(le, n)); }
    uint32_t instance() { cb_count[CB_INSTANCE]++; return push_value(V_INSTANCE, 0, n_instance++); }
    uint32_t witness() { cb_count[CB_WITNESS]++; return push_value(V_WITNESS, 0, n_witness++); }
    // flatten mode (the reference's IRFlattener, flattening.rs:83-88): a copy is a gate with its own output wire, so
    // value handles coincide with the wire ids GateBuilder would allocate.  Such a program is written out, not run.
    bool keep_copies = false;
    uint32_t copy(uint32_t a) {
        cb_count[CB_COPY]++;
        return keep_copies ? push_value(V_COPY, a, 0) : a;
    }
    // `ExpandDefinable` (rust/src/consumers/exp_definable.rs:24-139) in front of the flattener: with expand_on, gates
    // outside `expand_mask` (gate-set bits of relation.rs:15-25) are rewritten — AddConstant / MulConstant into
    // Constant + Add / Mul, And <-> Mul, Xor <-> Add, Not into AddConstant(1) — and the conditions on which the
    // reference panics throw ProgramPanic with its text.
    struct ProgramPanic {
        std::string msg;
    };
    bool expand_on = false;
    uint16_t expand_mask = 0;
    bool allowed(uint16_t bit) const { return !expand_on || (expand_mask & bit) == bit; }
    uint32_t add(uint32_t a, uint32_t b) {
        if (!allowed(0x0001)) {
            if (!allowed(0x0100)) throw ProgramPanic{"Cannot replace ADD by XOR if XOR is not supported."};
            return raw(CB_XOR, V_XOR, a, b);
        }
        return raw(CB_ADD, V_ADD, a, b);
    }
    uint32_t multiply(uint32_t a, uint32_t b) {
        if (!allowed(0x0004)) {
            if (!allowed(0x0200)) throw ProgramPanic{"Cannot replace MUL by AND if AND is not supported."};
            return raw(CB_AND, V_AND, a, b);
        }
        return raw(CB_MUL, V_MUL, a, b);
    }
    uint32_t add_constant(uint32_t a, const uint8_t* le, size_t n) {
        if (!allowed(0x0002)) return add(a, constant(le, n));
        cb_count[CB_ADDC]++;
        return push_value(V_ADDC, a, intern_const(le, n));
    }
    uint32_t mul_constant(uint32_t a, const uint8_t* le, size_t n) {
        if (!allowed(0x0008)) return multiply(a, constant(le, n));
        cb_count[CB_MULC]++;
        return push_value(V_MULC, a, intern_const(le, n));
    }
    uint32_t and_(uint32_t a, uint32_t b) {
        if (!allowed(0x0200)) {
            if (!allowed(0x0004)) throw ProgramPanic{"Cannot replace AND by MUL if MUL is not supported."};
            return multiply(a, b);
        }
        return raw(CB_AND, V_AND, a, b);
    }
    uint32_t xor_(uint32_t a, uint32_t b) {
        if (!allowed(0x0100)) {
            if (!allowed(0x0001)) throw ProgramPanic{"Cannot replace XOR by ADD if ADD is not supported."};
            return add(a, b);
        }
        return raw(CB_XOR, V_XOR, a, b);
    }
    uint32_t not_(uint32_t a) {
        if (!allowed(0x0400)) {
            if (!allowed(0x0001)) throw ProgramPanic{"Cannot replace NOT by ADD if ADD is not supported."};
            const uint8_t one = 1;
            return add_constant(a, &one, 1);
        }
        cb_count[CB_NOT]++;
        return push_value(V_NOT, a, 0);
    }
    uint32_t raw(int cb, uint8_t kind, uint32_t a, uint32_t b) {
        cb_count[cb]++;
        return push_value(kind, a, b);
    }
    void assert_zero(uint32_t v, uint64_t src_wire) {
        cb_count[CB_ASSERT_ZERO]++;
        asserts.push_back(AssertRec{v, n_values(), src_wire});
    }
    // constants the Evaluator needs: p-1 and 1 as little-endian bytes
    std::vector<uint8_t> minus_one_le() const;
};

// threads of the host passes that are split over chunks (ZKB_PLAN_THREADS, default min(8, cores))
unsigned plan_threads();

struct Plan {
    uint32_t n_slots = 0;
    uint32_t n_levels = 0;
    std::vector<uint32_t> slot_of_value;  // SSA value -> slot (kNoSlot if never stored)
    std::vector<uint8_t> readable;        // value can be read back after the run (its slot is not re-used)
    bool slot_reuse = true;               // liveness-based slot re-use (off: one slot per stored value)
    uint64_t n_reused_slots = 0;
    uint64_t n_raw_ops = 0;               // ops that need the raw-input flags (assert / not directly on an input)
    uint64_t n_sink_ops = 0;              // ops flagged F_SINK
    // level-major, opcode-sorted inside a level; inside an opcode group of the hot range (Add, Mul, AddC, MulC) the gates
    // are ordered by their shared operand (Plan::build), so the readers of one wire run back to back
    std::vector<GateOp> ops;
    std::vector<uint32_t> op_assert_seq;  // parallel to ops
    std::vector<uint64_t> level_off;      // n_levels + 1 offsets into ops
    std::vector<uint64_t> level_rare;     // per level: where the rare opcodes (>= D_AND) start
    std::vector<InputLoad> loads;
    // raw-semantics bookkeeping (SURVEY.md §8a trap 1): asserts applied directly to an input value
    std::vector<uint32_t> input_assert_seq;    // assert seq ...
    std::vector<uint32_t> input_assert_value;  // ... on this level-0 SSA value
    // call groups, in launch order: depth_off[d] .. depth_off[d + 1] are the groups of depth d (one launch each, between the
    // input kernel and the first wavefront)
    std::vector<GroupDesc> group_descs;
    std::vector<GroupOp> group_ops;
    std::vector<uint32_t> group_hints;  // per launch, per 2^kGroupHintShift calls: the group (relative to the launch) holding the first of them
    std::vector<uint32_t> hint_off;     // per depth: where its hints start
    std::vector<uint32_t> group_tables;
    std::vector<uint32_t> depth_off;
    uint32_t group_regs = 0;  // registers of the widest template
    uint32_t callout_slot0 = 0, n_callouts = 0;  // group outputs: slot of implicit value i = callout_slot0 + i
    uint32_t slot_of(uint32_t h) const { return is_callout(h) ? callout_slot0 + callout_index(h) : slot_of_value[h]; }
    bool is_readable(uint32_t h) const { return is_callout(h) || readable[h]; }
    std::vector<uint32_t> callout_assert_seq, callout_assert_value;  // AssertZero directly on a group output: tested in wavefront 1
    // accounting for bench.py (algorithmic bytes per witness, SURVEY.md §8d)
    uint64_t n_dev_ops[D_OPS] = {0};
    uint64_t algo_bytes_per_witness = 0;
    uint32_t max_level_ops = 0;

    // keep_all: every value stays readable (zkb_read_values); otherwise values consumed by
    // nothing but their own assert are not stored.
    void build(const Program& prog, bool keep_all, const std::vector<uint32_t>* live_values);
};

}  // namespace zkb
