// zkb_ctx: recording backend + batched GPU evaluation (sections 1-3 of include/zkb.h).
//
// Reference seam: `trait ZKBackend` + `PlaintextBackend` (rust/src/consumers/evaluator.rs:17-76,
// 848-947) and the simple arms of `Evaluator::ingest_gate` (:344-439).  The backend is deferred:
// callbacks record SSA values (program.h; long regular runs of zkb_push_gates in bulk on several threads); zkb_finalize
// levelizes; zkb_run streams tiles of witnesses through one kernel launch per wavefront — or, for launch-bound programs,
// through one launch for all wavefronts (cluster / grid barrier, or the barrier-free dataflow launch).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>

#include "context.h"

using namespace zkb;

#define CUDA_TRY(c, expr)                                                                              \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess)                                                                        \
            return (c)->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #expr); \
    } while (0)

namespace zkb {

bool ctx_record_ok(zkb_ctx* c) { return !c->has_pending; }

void ctx_latch(zkb_ctx* c, const std::string& msg) {
    if (!c->has_pending) {
        c->has_pending = true;
        c->pending_error = msg;
    }
}

static int ensure_fail_vectors(zkb_ctx* c, uint32_t n);

template <class T>
static int upload_vec(zkb_ctx* c, T*& dptr, const std::vector<T>& v) {
    if (dptr) {
        cudaFree(dptr);
        dptr = nullptr;
    }
    if (v.empty()) return ZKB_OK;
    CUDA_TRY(c, cudaMalloc((void**)&dptr, v.size() * sizeof(T)));
    CUDA_TRY(c, cudaMemcpyAsync(dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    return ZKB_OK;
}

int ctx_result_buffer(zkb_ctx* c, size_t n_words) {
    if (n_words <= c->h_res_cap) return ZKB_OK;
    if (c->h_res) cudaFreeHost(c->h_res);
    c->h_res = nullptr;
    c->h_res_cap = 0;
    size_t cap = std::max<size_t>(n_words, 1024);
    CUDA_TRY(c, cudaHostAlloc((void**)&c->h_res, cap * 4, cudaHostAllocDefault));
    c->h_res_cap = cap;
    return ZKB_OK;
}

int ctx_upload_groups(zkb_ctx* c) {
    int rc;
    if ((rc = upload_vec(c, c->d_group_descs, c->plan.group_descs)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_group_ops, c->plan.group_ops)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_group_tables, c->plan.group_tables)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_group_hints, c->plan.group_hints)) != ZKB_OK) return rc;
    group_jit_start(c);  // the templates as straight-line code, compiled in the background (group_jit.cpp)
    return ZKB_OK;
}

int ctx_finalize(zkb_ctx* c, int keep_values) {
    if (!c->prog.field_set) return c->fail(ZKB_E_ARG, "zkb_finalize: set_field was never called");
    if (c->prog.keep_copies) return c->fail(ZKB_E_ARG, "this context records in flatten mode: the program can be written out, not evaluated");
    const bool keep_all = keep_values == 1;
    // observable values: whatever is still bound in the flat scope, plus the Evaluator's live wires
    std::vector<uint32_t> live;
    if (keep_values != 2) {
        live = c->live_values;
        c->flat_scope.for_each([&](uint64_t, uint32_t v) { live.push_back(v); });
    }
    if (const char* e = getenv("ZKB_SLOT_REUSE")) c->plan.slot_reuse = atoi(e) != 0;
    // small programs over 1- / 2-limb fields keep one slot per value: a single witness then runs as a barrier-free dataflow
    // launch (k_levels_flow), which needs every slot written once; the wire store of such a program is small either way
    // (ZKB_FLOW_WIDE=1: the same for wider fields, for the flag-word variant that measured slower than the barriers)
    else if (!c->prog.binary && (c->prog.nlimb <= 2 || getenv("ZKB_FLOW_WIDE")) && c->prog.n_values() <= (1u << 22)) c->plan.slot_reuse = false;
    {
        NvtxRange r("zkb:levelize");
        c->plan.build(c->prog, keep_all, &live);
    }
    capture_reset(c, false);  // the device ops are about to be replaced
    c->keep_all = keep_all;
    c->finalized = true;
    c->resident_tile = -1;
    c->inputs_uploaded = false;
    if (!c->has_gpu) {  // host-only context: plan can be inspected, not run (ZKB_GROUP_JIT=2: and its group kernel generated + compiled)
        group_jit_start(c);
        return ZKB_OK;
    }
    NvtxRange r_up("zkb:program_upload");
    int rc;
    if ((rc = upload_vec(c, c->d_ops, c->plan.ops)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_aseq, c->plan.op_assert_seq)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_loads, c->plan.loads)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_consts, c->prog.const_limbs)) != ZKB_OK) return rc;
    if ((rc = upload_vec(c, c->d_level_off, c->plan.level_off)) != ZKB_OK) return rc;
    if ((rc = ctx_upload_groups(c)) != ZKB_OK) return rc;
    if (c->plan.n_raw_ops > 0 && (rc = upload_vec(c, c->d_const_flags, c->prog.const_unreduced)) != ZKB_OK) return rc;
    // raw bytes of the constants >= p, for the bitwise gates that take them unreduced (evaluator.rs:924-930)
    c->const_raw_stride = 0;
    if (c->plan.n_raw_ops > 0 && !c->prog.binary) {
        size_t widest = 0;
        for (const auto& r : c->prog.const_raw) widest = std::max(widest, r.size());
        if (widest) {
            c->const_raw_stride = (uint32_t)((widest + 3) / 4 * 4);
            std::vector<uint8_t> raw((size_t)c->prog.n_consts() * c->const_raw_stride, 0);
            for (size_t i = 0; i < c->prog.const_raw.size(); i++)
                memcpy(&raw[i * c->const_raw_stride], c->prog.const_raw[i].data(), c->prog.const_raw[i].size());
            if ((rc = upload_vec(c, c->d_const_raw, raw)) != ZKB_OK) return rc;
            CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // `raw` is pageable and about to go out of scope
        }
    }
    if (!c->prog.binary) launch_to_mont(c->prog.nlimb, c->d_consts, c->prog.n_consts(), c->prog.fp, c->stream);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ZKB_OK;
}

}  // namespace zkb

// ------------------------------------------------------------------------------------------
// 1. lifecycle
// ------------------------------------------------------------------------------------------
extern "C" zkb_ctx* zkb_create(int device) {
    zkb_ctx* c = new zkb_ctx();
    c->device = device;
    if (device < 0) return c;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        c->err = std::string("zkb_create: no usable CUDA device: ") + cudaGetErrorString(e);
        return c;
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        c->err = std::string("zkb_create: ") + cudaGetErrorString(e);
        return c;
    }
    c->sm_count = prop.multiProcessorCount;
    c->coop_supported = prop.cooperativeLaunch != 0;
    if (const char* g = getenv("ZKB_L2_FETCH_GRANULARITY")) {  // experiment knob (32 / 64 / 128): DRAM bytes fetched per L2 miss
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g));
        size_t got = 0;
        cudaDeviceGetLimit(&got, cudaLimitMaxL2FetchGranularity);
        if (getenv("ZKB_DEBUG")) fprintf(stderr, "zkb: L2 fetch granularity %zu B\n", got);
    }
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        c->err = std::string("zkb_create: ") + cudaGetErrorString(e);
        return c;
    }
    for (int i = 0; i < 4; i++) cudaEventCreate(&c->ev[i]);
    cudaMalloc((void**)&c->d_unreduced, sizeof(uint32_t));
    cudaMalloc((void**)&c->d_barrier, sizeof(uint32_t));  // arrival counter of the grid barrier (kernels.cu: grid_barrier)
    cudaMemset(c->d_barrier, 0, sizeof(uint32_t));
    ctx_result_buffer(c, 8192);  // pinned verdict buffer up front: cudaHostAlloc costs a millisecond, not for the first run to pay
    c->has_gpu = true;
    return c;
}

extern "C" void zkb_destroy(zkb_ctx* c) {
    if (!c) return;
    if (c->has_gpu) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        cudaFree(c->d_ops);
        cudaFree(c->d_aseq);
        cudaFree(c->d_loads);
        cudaFree(c->d_consts);
        cudaFree(c->d_level_off);
        cudaFree(c->d_group_descs);
        cudaFree(c->d_group_ops);
        cudaFree(c->d_group_tables);
        cudaFree(c->d_group_hints);
        if (c->h_res) cudaFreeHost(c->h_res);
        cudaFree(c->d_const_flags);
        cudaFree(c->d_const_raw);
        cudaFree(c->d_rawflag);
        cudaFree(c->d_store);
        cudaFree(c->d_inst);
        cudaFree(c->d_wit);
        cudaFree(c->d_first_fail);
        cudaFree(c->d_scratch_fail);
        cudaFree(c->d_unreduced);
        cudaFree(c->d_barrier);
        cudaFree(c->d_flow_flags);
        cudaFree(c->d_tab_slot);
        cudaFree(c->d_tab_opb);
        cudaFree(c->d_tab_readable);
        cudaFree(c->d_tab_kind);
        cudaFree(c->d_cap_desc);
        cudaFree(c->d_cap_raw);
        cudaFree(c->d_cap_unsunk);
        cudaFree(c->d_cap_out);
        r1cs_free(c);
        comm_free(c);
        group_jit_free(c);
        for (int i = 0; i < 4; i++)
            if (c->ev[i]) cudaEventDestroy(c->ev[i]);
        for (auto e : c->tile_ev) cudaEventDestroy(e);
        cudaStreamDestroy(c->stream);
    }
    delete c;
}

extern "C" const char* zkb_last_error(zkb_ctx* c) { return c ? c->err.c_str() : "null context"; }
extern "C" const char* zkb_pending_error(zkb_ctx* c) { return (c && c->has_pending) ? c->pending_error.c_str() : nullptr; }

// ------------------------------------------------------------------------------------------
// 2. ZKBackend seam
// ------------------------------------------------------------------------------------------
extern "C" int zkb_set_field(zkb_ctx* c, const uint8_t* modulus_le, size_t len, uint32_t degree, int is_boolean) {
    std::string err;
    if (!c->prog.set_field(modulus_le, len, degree, err)) {
        bool ref_err = err.rfind("zkb:", 0) != 0;
        return c->fail(ref_err ? ZKB_E_SEMANTIC : ZKB_E_UNSUPPORTED, err);
    }
    c->is_boolean = is_boolean != 0;
    return ZKB_OK;
}

static int write_le(zkb_ctx* c, const std::vector<uint8_t>& v, uint8_t* out, size_t cap, size_t* len) {
    if (cap < v.size()) return c->fail(ZKB_E_ARG, "output buffer too small");
    memcpy(out, v.data(), v.size());
    if (len) *len = v.size();
    return ZKB_OK;
}

extern "C" int zkb_one(zkb_ctx* c, uint8_t* out, size_t cap, size_t* len) { return write_le(c, {1}, out, cap, len); }
extern "C" int zkb_zero(zkb_ctx* c, uint8_t* out, size_t cap, size_t* len) { return write_le(c, {0}, out, cap, len); }
extern "C" int zkb_minus_one(zkb_ctx* c, uint8_t* out, size_t cap, size_t* len) {
    // PlaintextBackend::minus_one, evaluator.rs:881-886
    if (!c->prog.field_set) return c->fail(ZKB_E_SEMANTIC, "Modulus is not initiated, used `set_field()` before calling.");
    return write_le(c, c->prog.minus_one_le(), out, cap, len);
}

#define REC_PROLOGUE(c)                                                                         \
    if ((c)->is_replica) return (c)->fail(ZKB_E_ARG, "this context holds a replica of another rank's program: nothing can be recorded here"); \
    if (!(c)->prog.field_set) return (c)->fail(ZKB_E_ARG, "set_field must be called before recording"); \
    if ((c)->finalized) return (c)->fail(ZKB_E_ARG, "program already finalized");               \
    if ((c)->prog.n_total_values() >= (c)->max_values) return (c)->fail(ZKB_E_UNSUPPORTED, "zkb: resource limit exceeded (max_values)")
#define CHECK_WIRE(c, w) \
    if (!(c)->prog.valid_handle(w)) return (c)->fail(ZKB_E_ARG, "unknown wire handle")

extern "C" int zkb_copy(zkb_ctx* c, zkb_wire a, zkb_wire* out) {
    REC_PROLOGUE(c);
    CHECK_WIRE(c, a);
    *out = c->prog.copy((uint32_t)a);
    return ZKB_OK;
}
extern "C" int zkb_constant(zkb_ctx* c, const uint8_t* v, size_t len, zkb_wire* out) {
    REC_PROLOGUE(c);
    *out = c->prog.constant(v, len);
    return ZKB_OK;
}
extern "C" int zkb_assert_zero(zkb_ctx* c, zkb_wire a, uint64_t src_wire_id) {
    REC_PROLOGUE(c);
    CHECK_WIRE(c, a);
    c->prog.assert_zero((uint32_t)a, src_wire_id);
    return ZKB_OK;
}
#define BINOP(NAME, METHOD)                                                        \
    extern "C" int NAME(zkb_ctx* c, zkb_wire a, zkb_wire b, zkb_wire* out) {       \
        REC_PROLOGUE(c);                                                           \
        CHECK_WIRE(c, a);                                                          \
        CHECK_WIRE(c, b);                                                          \
        *out = c->prog.METHOD((uint32_t)a, (uint32_t)b);                           \
        return ZKB_OK;                                                             \
    }
BINOP(zkb_add, add)
BINOP(zkb_multiply, multiply)
BINOP(zkb_and, and_)
BINOP(zkb_xor, xor_)
extern "C" int zkb_add_constant(zkb_ctx* c, zkb_wire a, const uint8_t* v, size_t len, zkb_wire* out) {
    REC_PROLOGUE(c);
    CHECK_WIRE(c, a);
    *out = c->prog.add_constant((uint32_t)a, v, len);
    return ZKB_OK;
}
extern "C" int zkb_mul_constant(zkb_ctx* c, zkb_wire a, const uint8_t* v, size_t len, zkb_wire* out) {
    REC_PROLOGUE(c);
    CHECK_WIRE(c, a);
    *out = c->prog.mul_constant((uint32_t)a, v, len);
    return ZKB_OK;
}
extern "C" int zkb_not(zkb_ctx* c, zkb_wire a, zkb_wire* out) {
    REC_PROLOGUE(c);
    CHECK_WIRE(c, a);
    *out = c->prog.not_((uint32_t)a);
    return ZKB_OK;
}
extern "C" int zkb_instance(zkb_ctx* c, zkb_wire* out) {
    REC_PROLOGUE(c);
    *out = c->prog.instance();
    return ZKB_OK;
}
extern "C" int zkb_witness(zkb_ctx* c, zkb_wire* out) {
    REC_PROLOGUE(c);
    *out = c->prog.witness();
    return ZKB_OK;
}

// ------------------------------------------------------------------------------------------
// 3. bulk flat gates — the simple arms of Evaluator::ingest_gate (evaluator.rs:344-439)
// ------------------------------------------------------------------------------------------
// Bulk form of the gate loop below for long regular runs (what a builder-produced relation is: C3 = 2^24 gates in one call),
// the same three passes as the Evaluator's bulk ingest of flat FlatBuffers messages (evaluator.cpp: ingest_flat_window), over
// chunks of the gate array on the plan threads:
//   count    values / assertions / stream positions per chunk -> prefix sums give every chunk its handle range
//   define   kind + operand WIRES written at the final position, the output wire bound with a compare-and-swap
//   resolve  operand wires -> handles of values bound EARLIER in program order
// Anything irregular — Copy, Free, a wire defined twice or used before its definition, an index out of range, flatten /
// expand-definable mode, ids the dense scope table may not hold — undoes everything and returns false: the gate loop then
// runs from the start and reports the error where the reference does.  true: recorded, state as the gate loop leaves it.
static bool push_gates_bulk(zkb_ctx* c, const zkb_gate* gates, uint64_t n_gates, const std::vector<uint32_t>& cidx) {
    Program& p = c->prog;
    Scope& sc = c->flat_scope;
    const unsigned T = plan_threads();
    if (n_gates < (1u << 16) || T < 2 || p.keep_copies || p.expand_on || !sc.sparse.empty() || getenv("ZKB_NO_BULK_PUSH")) return false;
    constexpr uint64_t kChunk = 1u << 16;
    const uint64_t n_chunks = (n_gates + kChunk - 1) / kChunk;
    struct Count {
        uint64_t values = 0, asserts = 0, inst = 0, wit = 0, by_op[16] = {0};
        uint32_t max_out = 0;
        bool ok = true;
    };
    std::vector<Count> cnt(n_chunks);
    auto parallel = [&](uint64_t n, auto fn) {
        std::atomic<uint64_t> next{0};
        auto work = [&]() {
            for (uint64_t i; (i = next.fetch_add(1)) < n;) fn(i);
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < T && t < n; t++) pool.emplace_back(work);
        work();
        for (auto& th : pool) th.join();
    };
    const uint64_t n_consts = cidx.size();
    parallel(n_chunks, [&](uint64_t ch) {
        Count& k = cnt[ch];
        const uint64_t lo = ch * kChunk, hi = std::min(n_gates, lo + kChunk);
        for (uint64_t i = lo; i < hi; i++) {
            const zkb_gate& g = gates[i];
            switch (g.op) {
                case ZKB_G_ASSERT_ZERO: k.asserts++; break;
                case ZKB_G_CONSTANT: case ZKB_G_ADD_CONSTANT: case ZKB_G_MUL_CONSTANT:
                    if (g.b >= n_consts) k.ok = false;
                    // fall through
                case ZKB_G_ADD: case ZKB_G_MUL: case ZKB_G_AND: case ZKB_G_XOR: case ZKB_G_NOT:
                    k.values++;
                    k.max_out = std::max(k.max_out, g.out);
                    break;
                case ZKB_G_INSTANCE: k.values++; k.inst++; k.max_out = std::max(k.max_out, g.out); break;
                case ZKB_G_WITNESS: k.values++; k.wit++; k.max_out = std::max(k.max_out, g.out); break;
                default: k.ok = false; break;  // Copy, Free, unknown opcodes
            }
            k.by_op[g.op & 15]++;
        }
    });
    uint64_t tv = 0, ta = 0, ti = 0, tw = 0;
    uint32_t max_out = 0;
    for (const Count& k : cnt) {
        if (!k.ok) return false;
        tv += k.values; ta += k.asserts; ti += k.inst; tw += k.wit;
        max_out = std::max(max_out, k.max_out);
    }
    const uint64_t v0 = p.n_values(), a0 = p.asserts.size();
    if (tv == 0 || p.n_total_values() + tv >= c->max_values || v0 + tv >= kCalloutBit || a0 + ta >= 0xFFFFFFF0ull) return false;
    if ((uint64_t)p.n_instance + ti >= 0xFFFFFFFFull || (uint64_t)p.n_witness + tw >= 0xFFFFFFFFull) return false;
    if (!sc.ensure_dense(max_out, tv)) return false;
    p.kind.resize(v0 + tv);
    p.opa.resize(v0 + tv);
    p.opb.resize(v0 + tv);
    p.asserts.resize(a0 + ta);
    struct Base { uint64_t v, a, inst, wit; };
    std::vector<Base> base(n_chunks);
    {
        uint64_t v = v0, a = a0, ii = p.n_instance, ww = p.n_witness;
        for (uint64_t ch = 0; ch < n_chunks; ch++) {
            base[ch] = Base{v, a, ii, ww};
            v += cnt[ch].values; a += cnt[ch].asserts; ii += cnt[ch].inst; ww += cnt[ch].wit;
        }
    }
    std::atomic<bool> bad{false};
    uint32_t* dense = sc.dense.data();
    const size_t dn = sc.dense.size();
    parallel(n_chunks, [&](uint64_t ch) {
        uint64_t v = base[ch].v, a = base[ch].a, ii = base[ch].inst, ww = base[ch].wit;
        const uint64_t lo = ch * kChunk, hi = std::min(n_gates, lo + kChunk);
        for (uint64_t i = lo; i < hi; i++) {
            const zkb_gate& g = gates[i];
            if (g.op == ZKB_G_ASSERT_ZERO) {
                p.asserts[a++] = AssertRec{g.a, (uint32_t)v, g.a};  // value: the wire for now (resolved below)
                continue;
            }
            uint8_t kind;
            uint32_t oa = 0, ob = 0;
            switch (g.op) {
                case ZKB_G_CONSTANT: kind = V_CONST; ob = cidx[g.b]; break;
                case ZKB_G_ADD: kind = V_ADD; oa = g.a; ob = g.b; break;
                case ZKB_G_MUL: kind = V_MUL; oa = g.a; ob = g.b; break;
                case ZKB_G_AND: kind = V_AND; oa = g.a; ob = g.b; break;
                case ZKB_G_XOR: kind = V_XOR; oa = g.a; ob = g.b; break;
                case ZKB_G_NOT: kind = V_NOT; oa = g.a; break;
                case ZKB_G_ADD_CONSTANT: kind = V_ADDC; oa = g.a; ob = cidx[g.b]; break;
                case ZKB_G_MUL_CONSTANT: kind = V_MULC; oa = g.a; ob = cidx[g.b]; break;
                case ZKB_G_INSTANCE: kind = V_INSTANCE; ob = (uint32_t)ii++; break;
                default: kind = V_WITNESS; ob = (uint32_t)ww++; break;
            }
            p.kind[v] = kind;
            p.opa[v] = oa;
            p.opb[v] = ob;
            uint32_t expect = Scope::kNone;
            if (!__atomic_compare_exchange_n(&dense[g.out], &expect, (uint32_t)v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
                bad = true;  // "Wire_{id} already has a value in this scope."
                return;
            }
            v++;
        }
    });
    if (!bad) {
        const uint64_t vchunks = (tv + kChunk - 1) / kChunk, achunks = (ta + kChunk - 1) / kChunk;
        parallel(vchunks + achunks, [&](uint64_t ch) {
            if (ch < vchunks) {
                const uint64_t lo = v0 + ch * kChunk, hi = std::min(v0 + tv, lo + kChunk);
                for (uint64_t v = lo; v < hi; v++) {
                    const uint8_t k = p.kind[v];
                    if (k < V_ADD) continue;
                    const uint32_t wa = p.opa[v];
                    const uint32_t ra = wa < dn ? dense[wa] : Scope::kNone;
                    if (ra >= v) { bad = true; return; }  // undefined, bound later, or an implicit value: the gate loop decides
                    p.opa[v] = ra;
                    if (k == V_ADD || k == V_MUL || k == V_AND || k == V_XOR) {
                        const uint32_t wb = p.opb[v];
                        const uint32_t rb = wb < dn ? dense[wb] : Scope::kNone;
                        if (rb >= v) { bad = true; return; }
                        p.opb[v] = rb;
                    }
                }
            } else {
                const uint64_t lo = a0 + (ch - vchunks) * kChunk, hi = std::min(a0 + ta, lo + kChunk);
                for (uint64_t a = lo; a < hi; a++) {
                    AssertRec& r = p.asserts[a];
                    const uint32_t rv = r.value < dn ? dense[r.value] : Scope::kNone;
                    if (rv >= r.pos) { bad = true; return; }
                    r.value = rv;
                }
            }
        });
    }
    if (bad) {  // undo: unbind what this call bound, drop its values
        parallel(n_chunks, [&](uint64_t ch) {
            const uint64_t lo = ch * kChunk, hi = std::min(n_gates, lo + kChunk);
            for (uint64_t i = lo; i < hi; i++) {
                const zkb_gate& g = gates[i];
                if (g.op == ZKB_G_ASSERT_ZERO || g.out >= dn) continue;
                const uint32_t d = __atomic_load_n(&dense[g.out], __ATOMIC_RELAXED);
                if (d != Scope::kNone && d >= v0 && d < v0 + tv) __atomic_store_n(&dense[g.out], Scope::kNone, __ATOMIC_RELAXED);
            }
        });
        p.kind.resize(v0);
        p.opa.resize(v0);
        p.opb.resize(v0);
        p.asserts.resize(a0);
        return false;
    }
    uint64_t by_op[16] = {0};
    for (const Count& k : cnt)
        for (int o = 0; o < 16; o++) by_op[o] += k.by_op[o];
    p.cb_count[CB_CONSTANT] += by_op[ZKB_G_CONSTANT];
    p.cb_count[CB_ADD] += by_op[ZKB_G_ADD];
    p.cb_count[CB_MUL] += by_op[ZKB_G_MUL];
    p.cb_count[CB_ADDC] += by_op[ZKB_G_ADD_CONSTANT];
    p.cb_count[CB_MULC] += by_op[ZKB_G_MUL_CONSTANT];
    p.cb_count[CB_AND] += by_op[ZKB_G_AND];
    p.cb_count[CB_XOR] += by_op[ZKB_G_XOR];
    p.cb_count[CB_NOT] += by_op[ZKB_G_NOT];
    p.cb_count[CB_INSTANCE] += by_op[ZKB_G_INSTANCE];
    p.cb_count[CB_WITNESS] += by_op[ZKB_G_WITNESS];
    p.cb_count[CB_COPY] += by_op[ZKB_G_ASSERT_ZERO];  // an unweighted assertion tests a copy (evaluator.rs:355)
    p.cb_count[CB_ASSERT_ZERO] += by_op[ZKB_G_ASSERT_ZERO];
    p.ir_gates += n_gates - by_op[ZKB_G_CONSTANT] - by_op[ZKB_G_INSTANCE] - by_op[ZKB_G_WITNESS];
    p.n_instance += (uint32_t)ti;
    p.n_witness += (uint32_t)tw;
    sc.bulk_inserted(tv);
    return true;
}

extern "C" int zkb_push_gates(zkb_ctx* c, const zkb_gate* gates, uint64_t n_gates, const uint8_t* pool, size_t cstride,
                              uint64_t n_consts) {
    REC_PROLOGUE(c);
    if (c->has_pending) return c->fail(ZKB_E_SEMANTIC, c->pending_error);  // evaluator.rs:214-216: latched
    NvtxRange r_rec("zkb:record_gates");
    Program& p = c->prog;
    Scope& sc = c->flat_scope;
    char buf[96];
    auto no_value = [&](uint64_t id) {
        snprintf(buf, sizeof buf, "No value given for wire_%llu", (unsigned long long)id);  // evaluator.rs:787-797
        ctx_latch(c, buf);
        return c->fail(ZKB_E_SEMANTIC, buf);
    };
    auto already = [&](uint64_t id) {
        snprintf(buf, sizeof buf, "Wire_%llu already has a value in this scope.", (unsigned long long)id);  // :775-785
        ctx_latch(c, buf);
        return c->fail(ZKB_E_SEMANTIC, buf);
    };
    // constants of this call are interned once
    std::vector<uint32_t> cidx(n_consts);
    for (uint64_t i = 0; i < n_consts; i++) cidx[i] = p.intern_const(pool + i * cstride, cstride);
    if (push_gates_bulk(c, gates, n_gates, cidx)) return ZKB_OK;
    p.kind.reserve(p.kind.size() + n_gates);
    p.opa.reserve(p.opa.size() + n_gates);
    p.opb.reserve(p.opb.size() + n_gates);
    for (uint64_t i = 0; i < n_gates; i++) {
        const zkb_gate& g = gates[i];
        if (p.n_total_values() >= c->max_values) return c->fail(ZKB_E_UNSUPPORTED, "zkb: resource limit exceeded (max_values)");
        uint32_t va = 0, vb = 0, res = 0;
        switch (g.op) {
            case ZKB_G_CONSTANT:
                if (g.b >= n_consts) return c->fail(ZKB_E_ARG, "constant index out of range");
                p.cb_count[CB_CONSTANT]++;
                res = p.push_value(V_CONST, 0, cidx[g.b]);
                if (!sc.set(g.out, res)) return already(g.out);
                break;
            case ZKB_G_ASSERT_ZERO:
                if ((va = sc.get(g.a)) == Scope::kNone) return no_value(g.a);
                p.copy(va);  // evaluator.rs:355: unweighted asserts test a copy
                p.assert_zero(va, g.a);
                p.ir_gates++;
                break;
            case ZKB_G_COPY:
                if ((va = sc.get(g.a)) == Scope::kNone) return no_value(g.a);
                if (!sc.set(g.out, p.copy(va))) return already(g.out);
                break;
            case ZKB_G_ADD:
            case ZKB_G_MUL:
            case ZKB_G_AND:
            case ZKB_G_XOR:
                if ((va = sc.get(g.a)) == Scope::kNone) return no_value(g.a);
                if ((vb = sc.get(g.b)) == Scope::kNone) return no_value(g.b);
                res = g.op == ZKB_G_ADD ? p.add(va, vb) : g.op == ZKB_G_MUL ? p.multiply(va, vb)
                      : g.op == ZKB_G_AND ? p.and_(va, vb) : p.xor_(va, vb);
                p.ir_gates++;
                if (!sc.set(g.out, res)) return already(g.out);
                break;
            case ZKB_G_ADD_CONSTANT:
            case ZKB_G_MUL_CONSTANT:
                if ((va = sc.get(g.a)) == Scope::kNone) return no_value(g.a);
                if (g.b >= n_consts) return c->fail(ZKB_E_ARG, "constant index out of range");
                p.cb_count[g.op == ZKB_G_ADD_CONSTANT ? CB_ADDC : CB_MULC]++;
                res = p.push_value(g.op == ZKB_G_ADD_CONSTANT ? V_ADDC : V_MULC, va, cidx[g.b]);
                p.ir_gates++;
                if (!sc.set(g.out, res)) return already(g.out);
                break;
            case ZKB_G_NOT:
                if ((va = sc.get(g.a)) == Scope::kNone) return no_value(g.a);
                res = p.not_(va);
                p.ir_gates++;
                if (!sc.set(g.out, res)) return already(g.out);
                break;
            case ZKB_G_INSTANCE:
                if (!sc.set(g.out, p.instance())) return already(g.out);
                break;
            case ZKB_G_WITNESS:
                if (!sc.set(g.out, p.witness())) return already(g.out);
                break;
            case ZKB_G_FREE:
                for (uint64_t w = g.a; w <= (uint64_t)g.b; w++)
                    if (!sc.remove(w)) return no_value(w);
                break;
            default:
                return c->fail(ZKB_E_ARG, "unknown gate opcode");
        }
    }
    return ZKB_OK;
}

extern "C" int zkb_scope_lookup(zkb_ctx* c, uint64_t wire, zkb_wire* out) {
    uint32_t v = c->flat_scope.get(wire);
    if (v == Scope::kNone) {
        char buf[64];
        snprintf(buf, sizeof buf, "No value given for wire_%llu", (unsigned long long)wire);
        return c->fail(ZKB_E_SEMANTIC, buf);
    }
    *out = v;
    return ZKB_OK;
}

extern "C" int zkb_finalize(zkb_ctx* c, int keep_values) {
    if (c->finalized) return c->fail(ZKB_E_ARG, "program already finalized");
    if (keep_values < 0 || keep_values > 2) return c->fail(ZKB_E_ARG, "keep_values must be 0, 1 or 2");
    return ctx_finalize(c, keep_values);
}

// ------------------------------------------------------------------------------------------
// evaluation
// ------------------------------------------------------------------------------------------
static size_t elem_bytes(const zkb_ctx* c) { return (size_t)c->prog.nlimb * 4; }

// bytes of wire store for a tile of 2^log2_wt witnesses
static size_t store_bytes_for(const zkb_ctx* c, uint32_t log2_wt) {
    if (c->prog.binary) return (size_t)std::max<uint32_t>(c->plan.n_slots, 1) * ((size_t)1 << log2_wt) / 8;
    return (size_t)std::max<uint32_t>(c->plan.n_slots, 1) * elem_bytes(c) * ((size_t)1 << log2_wt);
}

static int choose_tile(zkb_ctx* c, uint32_t n_batch) {
    uint32_t want = 0;
    while (((uint64_t)1 << want) < n_batch) want++;
    uint32_t min_l2 = c->prog.binary ? 5 : 0;
    if (want < min_l2) want = min_l2;
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(c, cudaMemGetInfo(&free_b, &total_b));
    size_t budget = free_b + c->store_bytes;  // our own store will be released/reused
    budget = budget > ((size_t)768 << 20) ? budget - ((size_t)768 << 20) : budget / 2;
    if (const char* s = getenv("ZKB_MAX_STORE_MB")) budget = std::min(budget, (size_t)atoll(s) << 20);
    uint32_t l2 = want;
    while (l2 > min_l2 && store_bytes_for(c, l2) > budget) l2--;
    if (const char* s = getenv("ZKB_TILE_LOG2")) {
        uint32_t f = (uint32_t)atoi(s);
        if (f >= min_l2 && f < l2) l2 = f;
    }
    if (store_bytes_for(c, l2) > budget)
        return c->fail(ZKB_E_CUDA, "wire store does not fit in device memory even for the smallest tile");
    size_t need = store_bytes_for(c, l2);
    if (need > c->store_bytes || c->store_bytes > need * 4) {
        if (c->d_store) cudaFree(c->d_store);
        c->d_store = nullptr;
        c->store_bytes = 0;
        CUDA_TRY(c, cudaMalloc((void**)&c->d_store, need));
        c->store_bytes = need;
    }
    c->log2_wt = l2;
    c->resident_tile = -1;
    // per (input, lane) "raw integer >= p" flags, only when some gate tests an input value directly (trap 1)
    size_t flag_bytes = c->plan.n_raw_ops > 0 ? (c->plan.loads.size() << l2) : 0;
    if (flag_bytes > c->rawflag_bytes) {
        if (c->d_rawflag) cudaFree(c->d_rawflag);
        c->d_rawflag = nullptr;
        c->rawflag_bytes = 0;
        CUDA_TRY(c, cudaMalloc((void**)&c->d_rawflag, flag_bytes));
        c->rawflag_bytes = flag_bytes;
    }
    return ZKB_OK;
}

static int ensure_bytes(zkb_ctx* c, uint8_t*& d, size_t& cap, size_t need) {
    if (need <= cap && d) return ZKB_OK;
    if (d) cudaFree(d);
    d = nullptr;
    cap = 0;
    if (need == 0) need = 16;
    CUDA_TRY(c, cudaMalloc((void**)&d, need));
    cap = need;
    return ZKB_OK;
}

extern "C" int zkb_upload_inputs(zkb_ctx* c, const uint8_t* inst, uint64_t inst_set_stride, const uint8_t* wit,
                                 uint64_t wit_set_stride, uint32_t value_stride, uint32_t n_batch) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called before evaluation");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (n_batch == 0) return c->fail(ZKB_E_ARG, "n_batch must be > 0");
    const Program& p = c->prog;
    if (value_stride == 0 && (p.n_instance || p.n_witness)) return c->fail(ZKB_E_ARG, "value_stride must be > 0");
    // the reference consumes values from queues: too few instances is an Err string (evaluator.rs:420-427),
    // a missing witness value is a panic (evaluator.rs:944-946).  Callers state the counts via the strides.
    if (p.n_instance && !inst) return c->fail(ZKB_E_SEMANTIC, "Not enough instance to consume");
    if (p.n_witness && !wit) return c->fail(ZKB_E_FATAL, "Missing witness value for PlaintextBackend");
    if (inst_set_stride != 0 && inst_set_stride < (uint64_t)p.n_instance * value_stride)
        return c->fail(ZKB_E_SEMANTIC, "Not enough instance to consume");
    if (wit_set_stride != 0 && wit_set_stride < (uint64_t)p.n_witness * value_stride)
        return c->fail(ZKB_E_FATAL, "Missing witness value for PlaintextBackend");
    CUDA_TRY(c, cudaSetDevice(c->device));
    NvtxRange r_h2d("zkb:h2d_inputs");
    int rc = choose_tile(c, n_batch);
    if (rc != ZKB_OK) return rc;
    CUDA_TRY(c, cudaEventRecord(c->ev[0], c->stream));
    size_t ib = p.n_instance ? (inst_set_stride ? (size_t)inst_set_stride * n_batch : (size_t)p.n_instance * value_stride) : 0;
    size_t wb = p.n_witness ? (wit_set_stride ? (size_t)wit_set_stride * n_batch : (size_t)p.n_witness * value_stride) : 0;
    if ((rc = ensure_bytes(c, c->d_inst, c->inst_bytes, ib)) != ZKB_OK) return rc;
    if ((rc = ensure_bytes(c, c->d_wit, c->wit_bytes, wb)) != ZKB_OK) return rc;
    if (ib) CUDA_TRY(c, cudaMemcpyAsync(c->d_inst, inst, ib, cudaMemcpyHostToDevice, c->stream));
    if (wb) CUDA_TRY(c, cudaMemcpyAsync(c->d_wit, wit, wb, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaEventRecord(c->ev[1], c->stream));
    c->in.inst = c->d_inst;
    c->in.wit = c->d_wit;
    c->in.inst_set_stride = inst_set_stride;
    c->in.wit_set_stride = wit_set_stride;
    c->in.stride = value_stride;
    c->n_batch = n_batch;
    if ((rc = ensure_fail_vectors(c, n_batch)) != ZKB_OK) return rc;
    c->inputs_uploaded = true;
    c->resident_tile = -1;
    c->cap_valid = false;
    return ZKB_OK;
}

// run one tile of witnesses through every wavefront.  full = false: the next tile overwrites this one's wire store before
// anything can read it back, so the level kernels skip the results no gate reads (F_SINK) and the tile is not left resident
// (zkb_read_values re-runs it in full).  ZKB_SINK_STORES=1 stores them on every tile.
static void run_tile(zkb_ctx* c, uint32_t tile, bool full, uint32_t* d_fail, uint64_t* launches, uint64_t* level_launches) {
    const Plan& pl = c->plan;
    const Program& p = c->prog;
    TileGeom g;
    g.log2_wt = c->log2_wt;
    g.batch0 = tile << c->log2_wt;
    uint32_t wt = 1u << c->log2_wt;
    g.n_valid = std::min<uint32_t>(wt, c->n_batch - g.batch0);
    const char* ss = getenv("ZKB_SINK_STORES");
    g.skip_mask = full || (ss && atoi(ss) != 0) ? 0u : F_SINK;
    const int64_t resident = full ? (int64_t)tile : -1;
    uint8_t* rawflag = pl.n_raw_ops > 0 ? c->d_rawflag : nullptr;
    RawCtx rawctx;
    rawctx.rawflag = rawflag;
    rawctx.loads = c->d_loads;
    rawctx.const_raw = c->const_raw_stride ? c->d_const_raw : nullptr;
    rawctx.const_raw_stride = c->const_raw_stride;
    rawctx.pad = 0;
    rawctx.in = c->in;
    if (p.binary)
        launch_bool_load_inputs(c->d_loads, (uint32_t)pl.loads.size(), c->d_store, c->d_consts, c->in, g, c->d_unreduced, rawflag,
                                c->d_const_flags, c->sm_count, c->stream);
    else
        launch_load_inputs(p.nlimb, c->d_loads, (uint32_t)pl.loads.size(), c->d_store, c->d_consts, c->in, g, c->d_unreduced, rawflag,
                           c->d_const_flags, p.fp, c->sm_count, c->stream);
    (*launches)++;
    const bool timed = level_launches != nullptr && d_fail != c->d_scratch_fail;
    if (timed) {
        while (c->tile_ev.size() < 2 * (size_t)(tile + 1)) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            c->tile_ev.push_back(e);
        }
        cudaEventRecord(c->tile_ev[2 * tile], c->stream);
    }
    // call groups: one launch per dependency depth, before the first wavefront (their outputs are level-0 values)
    for (size_t d = 0; d + 1 < pl.depth_off.size(); d++) {
        const uint32_t lo = pl.depth_off[d], hi = pl.depth_off[d + 1];
        if (hi == lo) continue;
        const uint64_t calls = (uint64_t)pl.group_descs[hi - 1].first_call + pl.group_descs[hi - 1].n_calls;
        if (!p.binary)
            launch_arith_groups(p.nlimb, c->d_group_descs + lo, hi - lo, calls, c->d_group_ops, c->d_group_tables, c->d_group_hints + pl.hint_off[d],
                                c->d_store, c->d_consts, d_fail, g, p.fp, pl.group_regs, c->sm_count, c->stream);
        else if (!group_jit_launch(c, c->d_group_descs + lo, hi - lo, calls, c->d_group_hints + pl.hint_off[d], g.log2_wt - 5, (void*)c->stream))
            launch_bool_groups(c->d_group_descs + lo, hi - lo, calls, c->d_group_ops, c->d_group_tables, c->d_group_hints + pl.hint_off[d],
                               c->d_store, g, pl.group_regs, c->sm_count, c->stream, pl.group_ops.data(), (uint32_t)pl.group_ops.size());
        (*launches)++;
        if (level_launches) (*level_launches)++;
    }
    // launch-bound programs (levels far too small to fill the chip): all wavefronts in one cooperative launch
    bool coop = !p.binary && pl.n_levels > 1 && ((uint64_t)pl.max_level_ops << c->log2_wt) <= (uint64_t)c->sm_count * 8192;
    if (const char* e = getenv("ZKB_COOP")) coop = coop && atoi(e) != 0;
    // one witness, no slot written twice: every wavefront in one dataflow launch, no barrier.  Wide elements (flag words) are
    // opt-in (ZKB_FLOW_WIDE=1): two fences per hop made it 1.3-2.1 x SLOWER than the barrier kernels on every shape tried
    // (profiles/r02n_ab_flow_wide.log) — kept as the measured negative of DESIGN.md section 10
    if (!p.binary && p.nlimb >= 4 && c->log2_wt == 0 && pl.n_levels > 1 && pl.n_reused_slots == 0 && c->coop_supported &&
        getenv("ZKB_FLOW_WIDE")) {
        const char* e = getenv("ZKB_FLOW");
        const char* em = getenv("ZKB_FLOW_MIN");
        if ((!e || atoi(e) != 0) && pl.max_level_ops >= (uint32_t)(em ? atoi(em) : 256)) {
            cudaError_t err = cudaSuccess;
            if (c->flow_flags_cap < pl.n_slots) {
                if (c->d_flow_flags) cudaFree(c->d_flow_flags);
                c->d_flow_flags = nullptr;
                c->flow_flags_cap = 0;
                err = cudaMalloc((void**)&c->d_flow_flags, (size_t)pl.n_slots * 4);
                if (err == cudaSuccess) err = cudaMemsetAsync(c->d_flow_flags, 0, (size_t)pl.n_slots * 4, c->stream);
                if (err == cudaSuccess) c->flow_flags_cap = pl.n_slots;
                c->flow_epoch = 0;
            }
            if (err == cudaSuccess && ++c->flow_epoch == 0) {  // the run counter wrapped: start over with clean flags
                err = cudaMemsetAsync(c->d_flow_flags, 0, c->flow_flags_cap * 4, c->stream);
                c->flow_epoch = 1;
            }
            if (err == cudaSuccess)
                err = launch_levels_flow_wide(p.nlimb, c->d_ops, c->d_aseq, c->d_level_off, pl.n_levels, c->d_store, c->d_consts, d_fail, rawctx, g,
                                              p.fp, c->sm_count, pl.max_level_ops, (uint32_t)pl.loads.size() + pl.n_callouts, c->d_flow_flags,
                                              c->flow_epoch, c->stream);
            if (err == cudaSuccess) {
                (*launches)++;
                if (level_launches) (*level_launches)++;
                if (timed) cudaEventRecord(c->tile_ev[2 * tile + 1], c->stream);
                c->resident_tile = resident;
                return;
            }
            if (getenv("ZKB_DEBUG")) fprintf(stderr, "zkb: dataflow launch failed: %s\n", cudaGetErrorString(err));
            cudaGetLastError();
        }
    }
    // 1- / 2-limb fields: the value is its own flag (k_levels_flow)
    if (!p.binary && p.nlimb <= 2 && c->log2_wt == 0 && pl.n_levels > 1 && pl.n_reused_slots == 0 && c->coop_supported) {
        const char* e = getenv("ZKB_FLOW");
        const char* em = getenv("ZKB_FLOW_MIN");
        // a program whose wavefronts fit a few warps stays on the cluster-barrier kernel: producer and consumer lanes of ONE warp
        // exchanging values through L2 measured 10 us per wavefront (C1), the cluster barrier 0.23 us (profiles/r02l_ab_flow*.log)
        if ((!e || atoi(e) != 0) && pl.max_level_ops >= (uint32_t)(em ? atoi(em) : 256)) {
            cudaError_t err = launch_levels_flow(p.nlimb, c->d_ops, c->d_aseq, c->d_level_off, pl.n_levels, c->d_store, c->d_consts, d_fail, rawctx,
                                                 g, p.fp, c->sm_count, pl.max_level_ops, (uint32_t)pl.loads.size() + pl.n_callouts, pl.n_slots,
                                                 c->stream);
            if (err == cudaSuccess) {
                *launches += 2;  // marker fill + the launch
                if (level_launches) (*level_launches)++;
                if (timed) cudaEventRecord(c->tile_ev[2 * tile + 1], c->stream);
                c->resident_tile = resident;
                return;
            }
            if (getenv("ZKB_DEBUG")) fprintf(stderr, "zkb: dataflow launch failed: %s\n", cudaGetErrorString(err));
            cudaGetLastError();
        }
    }
    uint32_t first_level = 0;  // levels [0, first_level) have been run by the all-levels launches below
    if (coop && c->coop_supported) {
        // Runs of at least three consecutive wavefronts that each fit one thread-block cluster (8 x 512 threads, two
        // items per thread) go to the cluster-barrier kernel, the wavefronts between them to the grid-barrier kernel:
        // a random circuit is narrow at both ends and wide in the middle.
        const uint64_t kClusterItems = 8 * 512 * 2;
        auto items = [&](uint32_t l) { return (pl.level_off[l + 1] - pl.level_off[l]) << c->log2_wt; };
        std::vector<uint8_t> narrow(pl.n_levels);
        for (uint32_t l = 0; l < pl.n_levels; l++) narrow[l] = items(l) <= kClusterItems;
        for (uint32_t l = 0; l < pl.n_levels;) {  // short narrow runs are not worth a launch of their own
            uint32_t e = l;
            while (e < pl.n_levels && narrow[e] == narrow[l]) e++;
            if (narrow[l] && e - l < 3 && !(l == 0 && e == pl.n_levels))
                for (uint32_t k = l; k < e; k++) narrow[k] = 0;
            l = e;
        }
        bool ok = true;
        for (uint32_t l = 0; l < pl.n_levels && ok;) {
            uint32_t e = l;
            uint64_t widest = 0;
            while (e < pl.n_levels && narrow[e] == narrow[l]) widest = std::max(widest, items(e++));
            cudaError_t err = launch_levels_coop(p.nlimb, c->d_ops, c->d_aseq, c->d_level_off + l, e - l, c->d_store, c->d_consts, d_fail,
                                                 rawctx, g, p.fp, c->sm_count, narrow[l] ? widest : std::max(widest, kClusterItems + 1),
                                                 c->d_barrier, &c->barrier_epoch, c->stream);
            if (err != cudaSuccess) {
                if (getenv("ZKB_DEBUG")) fprintf(stderr, "zkb: cooperative launch failed: %s\n", cudaGetErrorString(err));
                cudaGetLastError();          // not launchable cooperatively: one launch per level from here on
                c->coop_supported = false;
                ok = false;
                break;
            }
            (*launches)++;
            if (level_launches) (*level_launches)++;
            first_level = e;
            l = e;
        }
        if (first_level == pl.n_levels) {
            if (timed) cudaEventRecord(c->tile_ev[2 * tile + 1], c->stream);
            c->resident_tile = resident;
            return;
        }
    }
    for (uint32_t l = first_level; l < pl.n_levels; l++) {
        uint64_t lo = pl.level_off[l], mid = pl.level_rare[l], hi = pl.level_off[l + 1];
        if (p.binary) {
            // a run of wavefronts of at most 1024 items each (gate x vector of words): one CTA, one launch for the run
            const uint32_t log2_vecs = c->log2_wt - 5 - (c->log2_wt >= 7 ? 2 : 0);
            auto small = [&](uint32_t k) { return ((pl.level_off[k + 1] - pl.level_off[k]) << log2_vecs) <= 1024; };
            uint32_t e = l;
            while (e < pl.n_levels && small(e)) e++;
            if (e - l >= 2 && !getenv("ZKB_NO_BOOL_CTA_RUNS")) {
                launch_bool_levels_cta(c->d_ops, c->d_aseq, c->d_level_off + l, e - l, c->d_store, c->d_consts, d_fail, rawflag, g, c->stream);
                (*launches)++;
                if (level_launches) (*level_launches)++;
                l = e - 1;
                continue;
            }
            if (hi > lo) {
                launch_bool_level(c->d_ops + lo, c->d_aseq + lo, hi - lo, c->d_store, c->d_consts, d_fail, rawflag, g, c->sm_count, c->stream);
                (*launches)++;
                (*level_launches)++;
            }
            continue;
        }
        if (mid > lo) {
            launch_level(p.nlimb, c->d_ops + lo, c->d_aseq + lo, mid - lo, c->d_store, c->d_consts, d_fail, rawctx, g, p.fp, c->sm_count, false,
                         c->stream);
            (*launches)++;
            (*level_launches)++;
        }
        if (hi > mid) {
            launch_level(p.nlimb, c->d_ops + mid, c->d_aseq + mid, hi - mid, c->d_store, c->d_consts, d_fail, rawctx, g, p.fp, c->sm_count, true,
                         c->stream);
            (*launches)++;
            (*level_launches)++;
        }
    }
    if (timed) cudaEventRecord(c->tile_ev[2 * tile + 1], c->stream);
    c->resident_tile = resident;
}

// SURVEY.md §8a trap 1: values >= p stay RAW in the reference.  The device works on residues, which is exact for add / mul
// (the reference reduces their results).  The raw-sensitive consumers of an input value are resolved ON THE DEVICE:
// k_load_inputs writes a per-(input, witness) "raw integer >= p" flag; the assert / not gates that read an input directly
// (F_RAW) treat a flagged operand as the non-zero integer it is, and an and / xor gate with a flagged operand re-reads its
// raw bytes (still resident in d_inst / d_wit / the raw constant table) and works on the unreduced integer (bitwise_raw).
namespace zkb {

static int ensure_fail_vectors(zkb_ctx* c, uint32_t n) {
    if (n <= c->first_fail_cap) return ZKB_OK;
    if (c->d_first_fail) cudaFree(c->d_first_fail);
    if (c->d_scratch_fail) cudaFree(c->d_scratch_fail);
    c->d_first_fail = c->d_scratch_fail = nullptr;
    c->first_fail_cap = 0;
    CUDA_TRY(c, cudaMalloc((void**)&c->d_first_fail, (size_t)n * 4));
    CUDA_TRY(c, cudaMalloc((void**)&c->d_scratch_fail, (size_t)n * 4));
    c->first_fail_cap = n;
    return ZKB_OK;
}

// One pass over the resident inputs.  `first` / `n_total`: this context's witnesses are [first, first + n_batch) of a batch
// of n_total sharded over the contexts of a communicator (comm.cu); the verdict vector is then MIN-reduced over the ranks
// (the path's only collective, SURVEY.md section 8e) and `out` holds all n_total verdicts on every rank.  A plain run is
// first = 0, n_total = n_batch, collective = false.
int ctx_run(zkb_ctx* c, zkb_verdict* out, uint32_t first, uint32_t n_total, bool collective) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called before evaluation");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (!c->inputs_uploaded) return c->fail(ZKB_E_ARG, "zkb_upload_inputs must be called before zkb_run");
    if ((uint64_t)first + c->n_batch > n_total) return c->fail(ZKB_E_ARG, "this rank's witnesses do not fit in the batch");
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = ensure_fail_vectors(c, n_total);
    if (rc != ZKB_OK) return rc;
    const uint32_t wt = 1u << c->log2_wt;
    const uint32_t n_tiles = (c->n_batch + wt - 1) / wt;
    c->cap_valid = false;
    uint32_t cap_E = 0;
    if (c->cap_n) {  // every captured value takes E bytes: the widest of an element, an input value and a listed raw constant
        const size_t eb = c->prog.binary ? 4 : elem_bytes(c);
        cap_E = (uint32_t)((std::max<size_t>({eb, c->in.stride, c->cap_raw_stride}) + 3) / 4 * 4);
        const size_t need = (size_t)c->n_batch * c->cap_n * cap_E;
        if (need > c->cap_out_bytes) {
            cudaFree(c->d_cap_out);
            c->d_cap_out = nullptr;
            c->cap_out_bytes = 0;
            if (cudaMalloc((void**)&c->d_cap_out, need) != cudaSuccess) {
                cudaGetLastError();  // not sticky: the context stays usable
                char buf[160];
                snprintf(buf, sizeof buf, "capture buffer of %zu bytes (%u witnesses x %llu values x %u) does not fit in device memory",
                         need, c->n_batch, (unsigned long long)c->cap_n, cap_E);
                return c->fail(ZKB_E_CUDA, buf);
            }
            c->cap_out_bytes = need;
        }
    }
    uint64_t launches = 0, level_launches = 0;
    CUDA_TRY(c, cudaEventRecord(c->ev[2], c->stream));
    launch_fill_u32(c->d_first_fail, 0xFFFFFFFFu, n_total, c->sm_count, c->stream);
    CUDA_TRY(c, cudaMemsetAsync(c->d_unreduced, 0, 4, c->stream));
    launches++;
    {
        NvtxRange r_lv("zkb:levels");
        for (uint32_t t = 0; t < n_tiles; t++) {
            run_tile(c, t, t == n_tiles - 1, c->d_first_fail + first, &launches, &level_launches);
            if (!c->cap_n) continue;
            // after the tile's last wavefront, before the next tile overwrites the store; outside the tile's level events
            TileGeom g{c->log2_wt, std::min<uint32_t>(1u << c->log2_wt, c->n_batch - (t << c->log2_wt)), t << c->log2_wt, 0};
            CUDA_TRY(c, launch_capture(c->prog.binary ? 0 : c->prog.nlimb, c->d_cap_desc, (uint32_t)c->cap_n, c->d_store, c->in, c->d_cap_raw,
                                       c->cap_raw_stride, g, cap_E, c->d_cap_out, c->prog.fp, c->stream));
            launches++;
        }
    }
    if (collective) {
        NvtxRange r_ar("zkb:verdict_allreduce");
        if ((rc = comm_allreduce_min_u32(c, c->d_first_fail, n_total)) != ZKB_OK) return rc;
    }
    NvtxRange r_d2h("zkb:verdict_d2h");
    if ((rc = ctx_result_buffer(c, (size_t)n_total + 1)) != ZKB_OK) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(c->h_res, c->d_first_fail, (size_t)n_total * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->h_res + n_total, c->d_unreduced, 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaEventRecord(c->ev[3], c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
    c->timing.total_ms = ms;
    c->timing.h2d_ms = 0;
    float lv = 0;
    for (uint32_t t = 0; t < n_tiles; t++) {
        float x = 0;
        cudaEventElapsedTime(&x, c->tile_ev[2 * t], c->tile_ev[2 * t + 1]);
        lv += x;
    }
    c->timing.levels_ms = lv;       // level kernels only, summed over tiles
    c->timing.load_ms = ms - lv;    // input conversion, verdict fill / all-reduce / copy, gaps
    c->timing.level_launches = level_launches;
    c->timing.kernel_launches = launches;
    c->n_unreduced_inputs = c->h_res[n_total];
    c->cap_E = cap_E;
    c->cap_valid = c->cap_n > 0;
    if (out)
        for (uint32_t j = 0; j < n_total; j++) {
            uint32_t f = c->h_res[j];
            memset(&out[j], 0, sizeof(zkb_verdict));
            out[j].ok = (f == 0xFFFFFFFFu) && !c->has_pending;
            out[j].first_fail_seq = f == 0xFFFFFFFFu ? UINT64_MAX : f;
        }
    return ZKB_OK;
}

void ctx_finish_e2e_timing(zkb_ctx* c) {
    float h2d = 0, total = 0;
    cudaEventElapsedTime(&h2d, c->ev[0], c->ev[1]);
    cudaEventElapsedTime(&total, c->ev[0], c->ev[3]);
    c->timing.h2d_ms = h2d;
    c->timing.total_ms = total;
}

}  // namespace zkb

extern "C" int zkb_run(zkb_ctx* c, zkb_verdict* out) { return ctx_run(c, out, 0, c->n_batch, false); }

extern "C" int zkb_evaluate(zkb_ctx* c, const uint8_t* inst, uint64_t inst_set_stride, const uint8_t* wit, uint64_t wit_set_stride,
                            uint32_t value_stride, uint32_t n_batch, zkb_verdict* out) {
    int rc = zkb_upload_inputs(c, inst, inst_set_stride, wit, wit_set_stride, value_stride, n_batch);
    if (rc != ZKB_OK) return rc;
    rc = zkb_run(c, out);
    if (rc != ZKB_OK) return rc;
    ctx_finish_e2e_timing(c);
    return ZKB_OK;
}

extern "C" int zkb_assert_info(zkb_ctx* c, uint64_t seq, uint64_t* src_wire_id) {
    if (seq >= c->prog.asserts.size()) return c->fail(ZKB_E_ARG, "assert index out of range");
    *src_wire_id = c->prog.asserts[seq].src_wire;
    return ZKB_OK;
}

// replica contexts keep the value tables on the device (comm.cu): fetch the entries of the requested handles
__global__ void k_gather_value_tables(const uint64_t* __restrict__ handles, uint32_t n, uint64_t n_values, const uint32_t* __restrict__ t_slot,
                                      const uint32_t* __restrict__ t_opb, const uint8_t* __restrict__ t_read, const uint8_t* __restrict__ t_kind,
                                      uint32_t callout_slot0, uint32_t n_callouts,
                                      uint32_t* __restrict__ out) {  // out: 4 x uint32 per handle {slot, opb, readable, kind}
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t v = handles[i];
    if (v >= kCalloutBit && v - kCalloutBit < n_callouts) {  // output of a call group: implicit value (program.h)
        out[4 * i] = callout_slot0 + (uint32_t)(v - kCalloutBit);
        out[4 * i + 1] = 0;
        out[4 * i + 2] = 1;
        out[4 * i + 3] = V_CALLOUT;
        return;
    }
    if (v >= n_values) {
        out[4 * i + 3] = 0xFFFFFFFFu;  // unknown handle
        return;
    }
    out[4 * i] = t_slot[v];
    out[4 * i + 1] = t_opb[v];
    out[4 * i + 2] = t_read[v];
    out[4 * i + 3] = t_kind[v];
}

// Per requested value: its slot, kind and operand b (constant-pool index / stream position of an input), from the host
// tables or, on a replica, from the device tables (k_gather_value_tables).  Fails on an unknown handle or a value that
// was not kept on the device.
static int resolve_values(zkb_ctx* c, const zkb_wire* values, uint64_t n, std::vector<uint32_t>& slots, std::vector<uint32_t>& kinds,
                          std::vector<uint32_t>& opbs) {
    const Program& p = c->prog;
    slots.resize(n);
    kinds.resize(n);
    opbs.resize(n);
    if (c->is_replica) {
        uint64_t* d_h = nullptr;
        uint32_t* d_t = nullptr;
        std::vector<uint32_t> t(4 * std::max<size_t>(n, 1));
        CUDA_TRY(c, cudaMalloc((void**)&d_h, std::max<size_t>(n, 1) * 8));
        CUDA_TRY(c, cudaMalloc((void**)&d_t, t.size() * 4));
        CUDA_TRY(c, cudaMemcpyAsync(d_h, values, n * 8, cudaMemcpyHostToDevice, c->stream));
        if (n) k_gather_value_tables<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(d_h, (uint32_t)n, c->replica_n_values, c->d_tab_slot, c->d_tab_opb,
                                                                                       c->d_tab_readable, c->d_tab_kind, c->plan.callout_slot0,
                                                                                       c->plan.n_callouts, d_t);
        CUDA_TRY(c, cudaMemcpyAsync(t.data(), d_t, n * 16, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        cudaFree(d_h);
        cudaFree(d_t);
        for (uint64_t i = 0; i < n; i++) {
            if (t[4 * i + 3] == 0xFFFFFFFFu) return c->fail(ZKB_E_ARG, "unknown wire handle");
            slots[i] = t[4 * i + 2] ? t[4 * i] : kNoSlot;
            opbs[i] = t[4 * i + 1];
            kinds[i] = t[4 * i + 3];
        }
    } else {
        for (uint64_t i = 0; i < n; i++) {
            if (!p.valid_handle(values[i])) return c->fail(ZKB_E_ARG, "unknown wire handle");
            const uint32_t h = (uint32_t)values[i];
            slots[i] = c->plan.is_readable(h) ? c->plan.slot_of(h) : kNoSlot;
            kinds[i] = is_callout(h) ? (uint32_t)V_CALLOUT : p.kind[h];
            opbs[i] = is_callout(h) ? 0 : p.opb[h];
        }
    }
    for (uint64_t i = 0; i < n; i++)
        if (slots[i] == kNoSlot)
            return c->fail(ZKB_E_ARG, "value was not kept on device (finalize with keep_all_values = 1 to read every value)");
    return ZKB_OK;
}

extern "C" int zkb_read_values(zkb_ctx* c, uint32_t batch_idx, const zkb_wire* values, uint64_t n, uint8_t* out, size_t stride) {
    if (!c->finalized || !c->inputs_uploaded) return c->fail(ZKB_E_ARG, "nothing has been evaluated yet");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (batch_idx >= c->n_batch) return c->fail(ZKB_E_ARG, "batch index out of range");
    const Program& p = c->prog;
    const size_t eb = p.binary ? 4 : elem_bytes(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    uint32_t tile = batch_idx >> c->log2_wt;
    if (c->resident_tile != (int64_t)tile) {
        uint64_t a = 0, b = 0;
        launch_fill_u32(c->d_scratch_fail, 0xFFFFFFFFu, c->n_batch, c->sm_count, c->stream);
        run_tile(c, tile, true, c->d_scratch_fail, &a, &b);
    }
    std::vector<uint32_t> slots, kinds, opbs;
    int rc = resolve_values(c, values, n, slots, kinds, opbs);
    if (rc != ZKB_OK) return rc;
    uint32_t *d_slots = nullptr, *d_out = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&d_slots, std::max<size_t>(n, 1) * 4));
    CUDA_TRY(c, cudaMalloc((void**)&d_out, std::max<size_t>(n, 1) * eb));
    CUDA_TRY(c, cudaMemcpyAsync(d_slots, slots.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
    uint32_t lane = batch_idx & ((1u << c->log2_wt) - 1);
    if (p.binary) launch_bool_read_values(d_slots, (uint32_t)n, c->d_store, lane, c->log2_wt, d_out, c->stream);
    else launch_read_values(p.nlimb, d_slots, (uint32_t)n, c->d_store, lane, c->log2_wt, d_out, p.fp, c->stream);
    std::vector<uint8_t> host(std::max<size_t>(n, 1) * eb);
    CUDA_TRY(c, cudaMemcpyAsync(host.data(), d_out, n * eb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    cudaFree(d_slots);
    cudaFree(d_out);
    // raw inputs for the trap-1 case: an input value is reported as the reference holds it (unreduced)
    std::vector<uint8_t> raw_in;
    for (uint64_t i = 0; i < n; i++) {
        uint8_t* dst = out + i * stride;
        memset(dst, 0, stride);
        const uint8_t* src = host.data() + i * eb;
        size_t nb = eb;
        std::vector<uint8_t> tmp;
        if (kinds[i] == V_CONST && p.const_unreduced[opbs[i]]) {
            src = p.const_raw[opbs[i]].data();
            nb = p.const_raw[opbs[i]].size();
        } else if (kinds[i] == V_INSTANCE || kinds[i] == V_WITNESS) {
            bool is_inst = kinds[i] == V_INSTANCE;
            size_t off = (size_t)batch_idx * (is_inst ? c->in.inst_set_stride : c->in.wit_set_stride) + (size_t)opbs[i] * c->in.stride;
            tmp.resize(c->in.stride);
            CUDA_TRY(c, cudaMemcpy(tmp.data(), (is_inst ? c->d_inst : c->d_wit) + off, c->in.stride, cudaMemcpyDeviceToHost));
            raw_in.swap(tmp);
            src = raw_in.data();
            nb = raw_in.size();
        }
        while (nb > 0 && src[nb - 1] == 0) nb--;
        if (nb > stride) return c->fail(ZKB_E_ARG, "output stride too small for the value");
        memcpy(dst, src, nb);
    }
    return ZKB_OK;
}

namespace zkb {

void capture_mark_sinks(zkb_ctx* c, bool set) {
    if (c->cap_n_unsunk) launch_set_sink(c->d_ops, c->d_cap_unsunk, c->cap_n_unsunk, set, c->stream);
}

void capture_reset(zkb_ctx* c, bool restore_sinks) {
    if (c->has_gpu) {
        if (restore_sinks && c->cap_n_unsunk) {
            capture_mark_sinks(c, true);
            cudaStreamSynchronize(c->stream);  // the op list is freed below
        }
        cudaFree(c->d_cap_desc);
        cudaFree(c->d_cap_raw);
        cudaFree(c->d_cap_unsunk);
    }
    c->d_cap_desc = nullptr;
    c->d_cap_raw = nullptr;
    c->d_cap_unsunk = nullptr;
    c->cap_n_unsunk = 0;
    c->cap_raw_stride = 0;
    c->cap_n = 0;
    c->cap_valid = false;
}

}  // namespace zkb

extern "C" int zkb_capture_values(zkb_ctx* c, const zkb_wire* values, uint64_t n) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called first");
    if (n >= 0xFFFFFFFFull) return c->fail(ZKB_E_ARG, "too many values to capture");
    if (c->has_gpu) CUDA_TRY(c, cudaSetDevice(c->device));
    std::vector<uint32_t> slots, kinds, opbs;
    int rc = resolve_values(c, values, n, slots, kinds, opbs);
    if (rc != ZKB_OK) return rc;  // the previous list stays
    const Program& p = c->prog;
    auto raw_const = [&](uint64_t i) { return kinds[i] == V_CONST && p.const_unreduced[opbs[i]]; };
    size_t widest = 0;
    for (uint64_t i = 0; i < n; i++)
        if (raw_const(i)) widest = std::max(widest, p.const_raw[opbs[i]].size());
    const uint32_t raw_stride = (uint32_t)((widest + 3) / 4 * 4);
    std::vector<CaptureDesc> desc(n);
    std::vector<uint8_t> raw;
    std::vector<uint32_t> slot_bits(c->plan.n_slots / 32 + 1, 0);  // slots whose producer must store on every tile
    for (uint64_t i = 0; i < n; i++) {
        if (kinds[i] == V_INSTANCE || kinds[i] == V_WITNESS) {
            desc[i] = CaptureDesc{slots[i], kinds[i] == V_INSTANCE ? (uint32_t)CAP_INSTANCE : (uint32_t)CAP_WITNESS, opbs[i], 0};
        } else if (raw_const(i)) {
            desc[i] = CaptureDesc{slots[i], CAP_RAW_CONST, (uint32_t)(raw.size() / raw_stride), 0};
            const auto& r = p.const_raw[opbs[i]];
            raw.insert(raw.end(), r.begin(), r.end());
            raw.resize(raw.size() + raw_stride - r.size(), 0);
        } else {
            desc[i] = CaptureDesc{slots[i], CAP_STORE, 0, 0};
            slot_bits[slots[i] >> 5] |= 1u << (slots[i] & 31);
        }
    }
    capture_reset(c, true);
    if (!c->has_gpu || n == 0) {  // a host-only context only validates the list
        c->cap_n = n;
        return ZKB_OK;
    }
    // descriptors, raw rows and the sink search; the bitmap and the found-op count live in one scratch allocation
    uint32_t* d_scratch = nullptr;
    const size_t scratch_words = slot_bits.size() + 1;
    cudaError_t e = cudaMalloc((void**)&c->d_cap_desc, n * sizeof(CaptureDesc));
    if (e == cudaSuccess && !raw.empty()) e = cudaMalloc((void**)&c->d_cap_raw, raw.size());
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_cap_unsunk, n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_scratch, scratch_words * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_cap_desc, desc.data(), n * sizeof(CaptureDesc), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && !raw.empty()) e = cudaMemcpyAsync(c->d_cap_raw, raw.data(), raw.size(), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_scratch, slot_bits.data(), slot_bits.size() * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_scratch + slot_bits.size(), 0, 4, c->stream);
    uint32_t n_found = 0;
    if (e == cudaSuccess) {
        const uint64_t n_ops = c->is_replica ? c->replica_n_ops : c->plan.ops.size();
        launch_unsink(c->d_ops, n_ops, d_scratch, c->d_cap_unsunk, (uint32_t)n, d_scratch + slot_bits.size(), c->sm_count, c->stream);
        e = cudaMemcpyAsync(&n_found, d_scratch + slot_bits.size(), 4, cudaMemcpyDeviceToHost, c->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);  // (also: the pageable sources above are copied)
    cudaFree(d_scratch);
    // a written value has one producer and a captured slot is not re-used, so at most n ops are found
    c->cap_n_unsunk = std::min<uint32_t>(n_found, (uint32_t)n);
    c->cap_raw_stride = raw_stride;
    c->cap_n = n;
    if (e != cudaSuccess) {
        cudaGetLastError();
        capture_reset(c, true);
        return c->fail(ZKB_E_CUDA, std::string("zkb_capture_values: ") + cudaGetErrorString(e));
    }
    return ZKB_OK;
}

extern "C" int zkb_read_captured(zkb_ctx* c, uint32_t first, uint32_t n_witnesses, uint8_t* out, size_t stride) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called first");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (!c->cap_valid) return c->fail(ZKB_E_ARG, "nothing has been captured yet (zkb_capture_values, then a run)");
    if ((uint64_t)first + n_witnesses > c->n_batch) return c->fail(ZKB_E_ARG, "batch index out of range");
    CUDA_TRY(c, cudaSetDevice(c->device));
    const size_t E = c->cap_E, n = c->cap_n;
    const uint8_t* src = c->d_cap_out + (size_t)first * n * E;
    if (stride == E) {  // the device layout: one copy
        CUDA_TRY(c, cudaMemcpyAsync(out, src, (size_t)n_witnesses * n * E, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        return ZKB_OK;
    }
    // other strides: through a host buffer, a block of witnesses at a time
    const size_t per_w = n * E;
    const uint32_t chunk = (uint32_t)std::max<size_t>(1, ((size_t)64 << 20) / std::max<size_t>(per_w, 1));
    std::vector<uint8_t> host(std::min<size_t>(chunk, n_witnesses) * per_w);
    for (uint32_t w0 = 0; w0 < n_witnesses; w0 += chunk) {
        const uint32_t nw = std::min(chunk, n_witnesses - w0);
        CUDA_TRY(c, cudaMemcpyAsync(host.data(), src + (size_t)w0 * per_w, nw * per_w, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        for (size_t k = 0; k < (size_t)nw * n; k++) {
            const uint8_t* v = host.data() + k * E;
            uint8_t* dst = out + ((size_t)w0 * n + k) * stride;
            if (stride > E) {
                memcpy(dst, v, E);
                memset(dst + E, 0, stride - E);
            } else {
                for (size_t b = stride; b < E; b++)
                    if (v[b]) return c->fail(ZKB_E_ARG, "output stride too small for the value");
                memcpy(dst, v, stride);
            }
        }
    }
    return ZKB_OK;
}

extern "C" int zkb_set_limits(zkb_ctx* c, uint64_t max_values, uint64_t max_steps) {
    if (max_values > 0xFFFFFF00ull) return c->fail(ZKB_E_ARG, "max_values above the 32-bit handle space");
    if (max_values) c->max_values = max_values;
    if (max_steps) c->max_steps = max_steps;
    return ZKB_OK;
}

// FNV-1a over the whole device plan (ops, assertion table, input loads, slot map, level offsets): two plans of the
// same program must be identical whatever the number of host threads that built them
extern "C" int zkb_debug_plan_hash(zkb_ctx* c, uint64_t* out) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called first");
    if (c->is_replica) return c->fail(ZKB_E_ARG, "replica context: the host copy of the plan lives on the root rank");
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](const void* p, size_t n) {
        const uint8_t* b = (const uint8_t*)p;
        for (size_t i = 0; i < n; i++) {
            h ^= b[i];
            h *= 1099511628211ull;
        }
    };
    const Plan& pl = c->plan;
    mix(pl.ops.data(), pl.ops.size() * sizeof(GateOp));
    mix(pl.op_assert_seq.data(), pl.op_assert_seq.size() * 4);
    mix(pl.loads.data(), pl.loads.size() * sizeof(InputLoad));
    mix(pl.slot_of_value.data(), pl.slot_of_value.size() * 4);
    mix(pl.readable.data(), pl.readable.size());
    mix(pl.level_off.data(), pl.level_off.size() * 8);
    mix(pl.level_rare.data(), pl.level_rare.size() * 8);
    mix(pl.group_descs.data(), pl.group_descs.size() * sizeof(GroupDesc));
    mix(pl.group_ops.data(), pl.group_ops.size() * sizeof(GroupOp));
    mix(pl.group_hints.data(), pl.group_hints.size() * 4);
    mix(pl.group_tables.data(), pl.group_tables.size() * 4);
    mix(&pl.callout_slot0, 4);
    mix(&pl.n_callouts, 4);
    mix(&pl.n_slots, 4);
    mix(&pl.n_reused_slots, 8);
    mix(pl.n_dev_ops, sizeof(pl.n_dev_ops));
    *out = h;
    return ZKB_OK;
}

extern "C" int zkb_get_stats(zkb_ctx* c, zkb_stats* s) {
    memset(s, 0, sizeof(*s));
    const Program& p = c->prog;
    s->n_values = c->is_replica ? c->replica_n_values + c->plan.n_callouts : p.n_total_values();
    s->n_asserts = p.asserts.size();
    s->n_instance = p.n_instance;
    s->n_witness = p.n_witness;
    s->n_consts = p.n_consts();
    s->ir_gates = p.ir_gates;
    for (int i = 0; i < CB_KINDS; i++) s->callbacks[i] = p.cb_count[i];
    s->nlimb = (uint32_t)p.nlimb;
    s->binary = p.binary;
    if (c->finalized) {
        s->n_slots = c->plan.n_slots;
        s->n_levels = c->plan.n_levels;
        s->n_device_ops = c->is_replica ? c->replica_n_ops : c->plan.ops.size();
        s->algo_bytes_per_witness = c->plan.algo_bytes_per_witness;
        s->n_sink_ops = c->plan.n_sink_ops;
    }
    s->n_call_groups = c->plan.group_descs.empty() ? p.groups.size() : c->plan.group_descs.size();
    for (const auto& g : p.groups) s->n_group_calls += g.n_calls;
    if (p.groups.empty())
        for (const auto& g : c->plan.group_descs) s->n_group_calls += g.n_calls;  // replica: only the plan came over
    if (c->finalized) {
        for (size_t d = 0; d + 1 < c->plan.depth_off.size(); d++) s->n_group_launches += c->plan.depth_off[d + 1] > c->plan.depth_off[d];
        s->n_group_table_slots = c->plan.group_tables.size();
    }
    s->group_jit_state = (int64_t)group_jit_state(c);
    if (c->inputs_uploaded) {
        s->tile_witnesses = 1u << c->log2_wt;
        s->n_tiles = (c->n_batch + s->tile_witnesses - 1) / s->tile_witnesses;
    }
    return ZKB_OK;
}

extern "C" int zkb_get_timing(zkb_ctx* c, zkb_timing* t) {
    *t = c->timing;
    return ZKB_OK;
}

extern "C" int zkb_get_program(zkb_ctx* c, uint64_t first, uint64_t n, uint8_t* kinds, uint32_t* a, uint32_t* b) {
    const Program& p = c->prog;
    if (c->is_replica) return c->fail(ZKB_E_ARG, "replica context: the recorded program lives on the root rank");
    if (first + n > p.n_values()) return c->fail(ZKB_E_ARG, "program range out of bounds");  // explicit values only
    for (uint64_t i = 0; i < n; i++) {
        kinds[i] = p.kind[first + i];
        a[i] = p.opa[first + i];
        b[i] = p.opb[first + i];
    }
    return ZKB_OK;
}

extern "C" int zkb_get_const(zkb_ctx* c, uint64_t idx, uint8_t* out, size_t cap, size_t* len) {
    const Program& p = c->prog;
    if (idx >= p.n_consts()) return c->fail(ZKB_E_ARG, "constant index out of range");
    size_t nb = (size_t)p.nlimb * 4;
    if (cap < nb) return c->fail(ZKB_E_ARG, "output buffer too small");
    memcpy(out, &p.const_limbs[idx * (size_t)p.nlimb], nb);
    if (len) *len = nb;
    return ZKB_OK;
}

extern "C" int zkb_assert_value(zkb_ctx* c, uint64_t seq, zkb_wire* value) {
    if (seq >= c->prog.asserts.size()) return c->fail(ZKB_E_ARG, "assert index out of range");
    if (c->prog.asserts[seq].value == kGroupAssertValue) return c->fail(ZKB_E_ARG, "assertion inside a call group: its value is a call-local wire");
    *value = c->prog.asserts[seq].value;
    return ZKB_OK;
}

extern "C" int zkb_debug_plan_ops(zkb_ctx* c, uint64_t first, uint64_t n, uint32_t* ops4, uint32_t* values) {
    if (!c->finalized) return c->fail(ZKB_E_ARG, "zkb_finalize must be called first");
    if (c->is_replica) return c->fail(ZKB_E_ARG, "replica context: the host copy of the plan lives on the root rank");
    const Plan& pl = c->plan;
    if (first > pl.ops.size() || n > pl.ops.size() - first) return c->fail(ZKB_E_ARG, "op range out of bounds");
    if (values && pl.n_reused_slots != 0) return c->fail(ZKB_E_ARG, "op values need a plan without slot re-use");
    std::vector<uint32_t> value_of_slot;
    if (values) {
        value_of_slot.assign(pl.n_slots, kNoSlot);
        for (uint32_t v = 0; v < (uint32_t)pl.slot_of_value.size(); v++)
            if (pl.slot_of_value[v] != kNoSlot) value_of_slot[pl.slot_of_value[v]] = v;
    }
    for (uint64_t i = 0; i < n; i++) {
        const GateOp& g = pl.ops[first + i];
        ops4[4 * i] = g.a;
        ops4[4 * i + 1] = g.b;
        ops4[4 * i + 2] = g.out;
        ops4[4 * i + 3] = g.meta;
        if (values) values[i] = g.out < pl.n_slots ? value_of_slot[g.out] : kNoSlot;
    }
    return ZKB_OK;
}

extern "C" int zkb_level_info(zkb_ctx* c, uint64_t level, uint64_t out[5]) {
    if (!c->finalized || level >= c->plan.n_levels) return c->fail(ZKB_E_ARG, "level out of range");
    if (c->is_replica) return c->fail(ZKB_E_ARG, "replica context: the host copy of the plan lives on the root rank");
    const Plan& pl = c->plan;
    const uint64_t E = c->prog.binary ? 1 : (uint64_t)c->prog.nlimb * 4;
    uint64_t lo = pl.level_off[level], hi = pl.level_off[level + 1];
    out[0] = hi - lo;
    out[1] = pl.level_rare[level] - lo;
    out[2] = out[3] = out[4] = 0;
    for (uint64_t i = lo; i < hi; i++) {
        uint32_t m = pl.ops[i].meta, opc = m & 0xff;
        if (m & F_ASSERT) out[2]++;
        if (m & F_NOSTORE) out[3]++;
        if (opc == D_ASSERT) out[4] += E;
        else out[4] += ((opc == D_ADD || opc == D_MUL || opc == D_AND || opc == D_XOR) ? 3 * E : 2 * E) + ((m & F_ASSERT) ? E : 0);
    }
    return ZKB_OK;
}

// the run-time specialisation of the call-group kernel (group_jit.cpp): block until its compilation has ended
extern "C" int zkb_debug_group_jit_wait(zkb_ctx* c, int* state, double* compile_seconds) {
    const int st = group_jit_wait(c);
    if (state) *state = st;
    if (compile_seconds) *compile_seconds = group_jit_compile_seconds(c);
    if (st == -1) c->err = std::string("group kernel specialisation failed: ") + group_jit_log(c);
    return ZKB_OK;
}
extern "C" const char* zkb_debug_group_jit_source(zkb_ctx* c) { return group_jit_source(c); }
