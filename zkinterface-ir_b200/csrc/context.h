// Internal: the context behind zkb_ctx (one host thread + one device).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/zkb.h"
#include "kernels.cuh"
#include "program.h"

namespace zkb {

// wire id -> SSA value map of one scope (HashMap<WireId, B::Wire>, evaluator.rs:158-160).  Ids that stay within a small
// multiple of the number of insertions made so far (sequentially numbered wires: every builder-produced relation) live in
// a dense vector; anything else goes to a hash map, so memory is proportional to the work done in the scope, never to the
// largest wire id a (possibly hostile) gate names.
class Scope {
public:
    static constexpr uint32_t kNone = 0xFFFFFFFFu;
    static constexpr uint64_t kDenseLimit = 1ull << 32;
    std::vector<uint32_t> dense;
    std::unordered_map<uint64_t, uint32_t> sparse;
    uint64_t live = 0;
    uint64_t n_sets = 0;              // insertions since the last clear(): bounds the dense part
    bool track = false;               // pooled scopes remember the dense ids they touched, so clear() is O(touched)
    std::vector<uint32_t> touched;
    bool touched_all = false;         // bulk insertions are not listed: clear() wipes the whole table

    // operand ids of a gate a few iterations ahead: random circuits read the map all over, so the loads are started early
    void prefetch(uint64_t id) const {
        if (id < dense.size()) __builtin_prefetch(&dense[id]);
    }
    uint32_t get(uint64_t id) const {
        if (id < dense.size() && dense[id] != kNone) return dense[id];
        if (sparse.empty()) return kNone;
        auto it = sparse.find(id);
        return it == sparse.end() ? kNone : it->second;
    }
    // returns false if the id already had a value (the new value is stored anyway, like HashMap::insert)
    bool set(uint64_t id, uint32_t v) {
        if (id < dense.size() && dense[id] != kNone) {
            dense[id] = v;
            return false;
        }
        if (!sparse.empty()) {
            auto it = sparse.find(id);
            if (it != sparse.end()) {
                it->second = v;
                return false;
            }
        }
        n_sets++;
        live++;
        if (id >= dense.size() && id < kDenseLimit && id <= 4 * (n_sets + 1024)) {
            size_t n = dense.size() ? dense.size() : 16;
            while (n <= id) n *= 2;
            dense.resize(n, kNone);
        }
        if (id < dense.size()) {
            dense[id] = v;
            if (track) touched.push_back((uint32_t)id);
        } else {
            sparse.emplace(id, v);
        }
        return true;
    }
    // bulk insertion (call groups, sub-scope plumbing): after ensure_dense(hi, n) the caller writes up to n UNBOUND ids
    // <= hi straight into `dense` and reports how many with bulk_inserted().  The same memory bound as set().
    bool ensure_dense(uint64_t hi, uint64_t n_new) {
        if (hi < dense.size()) return true;
        if (hi >= kDenseLimit || hi > 4 * (n_sets + n_new + 1024)) return false;
        // sized for the request (a loop that announces 2^24 outputs gets 2^24 entries, not the next power of two), but never
        // growing by less than half, so repeated requests stay amortized
        size_t n = std::max<size_t>({(size_t)hi + 1, dense.size() + dense.size() / 2, (size_t)16});
        dense.resize(n, kNone);
        return true;
    }
    void bulk_inserted(uint64_t n) {
        n_sets += n;
        live += n;
        touched_all = true;
    }
    bool remove(uint64_t id) {
        if (id < dense.size() && dense[id] != kNone) {
            dense[id] = kNone;
            live--;
            return true;
        }
        if (!sparse.empty() && sparse.erase(id)) {
            live--;
            return true;
        }
        return false;
    }
    void clear() {
        if (dense.size() > (1u << 20)) {  // a pooled scope does not keep a large table alive
            std::vector<uint32_t>().swap(dense);
        } else if (track && !touched_all && touched.size() < dense.size() / 8) {
            for (uint32_t id : touched) dense[id] = kNone;
        } else {
            std::fill(dense.begin(), dense.end(), kNone);
        }
        touched.clear();
        touched_all = false;
        sparse.clear();
        live = 0;
        n_sets = 0;
    }
    template <class F>
    void for_each(F f) const {
        for (size_t i = 0; i < dense.size(); i++)
            if (dense[i] != kNone) f((uint64_t)i, dense[i]);
        for (auto& kv : sparse) f(kv.first, kv.second);
    }
};

struct R1csDev;    // r1cs.cu
struct CommState;  // comm.cu
struct GroupJit;   // group_jit.cpp

// NVTX range over a phase of the path (host flatten / levelize / H2D / levels / D2H): shows up on the Nsight Systems and
// ncu timelines; costs a predicted-not-taken branch when no tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

}  // namespace zkb

struct zkb_ctx {
    int device = -1;
    bool has_gpu = false;
    int sm_count = 148;
    std::string err;

    zkb::Program prog;
    zkb::Plan plan;
    bool is_boolean = false;
    bool finalized = false;
    bool keep_all = false;
    zkb::Scope flat_scope;           // zkb_push_gates
    std::vector<uint32_t> live_values;  // observable values supplied by the Evaluator at finalize
    bool has_pending = false;
    std::string pending_error;       // first recording error (latched)
    // resource limits of the host pass (zkb_set_limits): a malformed or hostile statement (a For over 2^60
    // iterations, a 2^32-wire range) must end in an error, not in an exhausted host
    uint64_t max_values = 0xFFFFFF00ull;  // SSA values (handles are 32-bit)
    uint64_t max_steps = 1ull << 40;      // gates ingested + loop iterations + wires expanded

    // device state
    cudaStream_t stream = nullptr;
    zkb::GateOp* d_ops = nullptr;
    uint32_t* d_aseq = nullptr;
    zkb::InputLoad* d_loads = nullptr;
    uint32_t* d_consts = nullptr;
    uint64_t* d_level_off = nullptr;
    zkb::GroupDesc* d_group_descs = nullptr;  // call groups (program.h), launch order
    zkb::GroupOp* d_group_ops = nullptr;
    uint32_t* d_group_tables = nullptr;
    uint32_t* d_group_hints = nullptr;
    uint8_t* d_const_flags = nullptr;   // per constant: raw value >= p
    uint8_t* d_const_raw = nullptr;     // raw bytes of the constants (const_raw_stride each), when a bitwise gate may need them
    uint32_t const_raw_stride = 0;
    uint32_t n_unreduced_inputs = 0;    // instance / witness values >= p seen by the last run
    uint8_t* d_rawflag = nullptr;       // per (input load, lane): raw value >= p (only when plan.n_raw_ops > 0)
    size_t rawflag_bytes = 0;
    bool coop_supported = false;
    uint32_t* d_store = nullptr;
    size_t store_bytes = 0;
    uint32_t log2_wt = 0;
    uint8_t* d_inst = nullptr;
    uint8_t* d_wit = nullptr;
    size_t inst_bytes = 0, wit_bytes = 0;
    zkb::InputDesc in{};
    uint32_t n_batch = 0;
    uint32_t* d_first_fail = nullptr;
    uint32_t* d_scratch_fail = nullptr;
    size_t first_fail_cap = 0;
    uint32_t* d_unreduced = nullptr;
    uint32_t* d_flow_flags = nullptr;  // dataflow launch over wide elements: per slot, the number of the run that wrote it
    size_t flow_flags_cap = 0;
    uint32_t flow_epoch = 0;
    uint32_t* d_barrier = nullptr;   // monotonic arrival counter of the grid barrier
    uint32_t barrier_epoch = 0;      // its value once every launch issued so far has finished
    int64_t resident_tile = -1;
    bool inputs_uploaded = false;
    uint32_t* h_res = nullptr;       // pinned: the verdict vector + the unreduced-input count of a run land here (a copy to
    size_t h_res_cap = 0;            // pageable memory is staged and synchronous: tens of microseconds per small copy)
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> tile_ev;
    zkb_timing timing{};

    // capture list (zkb_capture_values): written out for every witness after each tile of a run (k_capture)
    uint64_t cap_n = 0;                      // values in the list (a host-only context validates and counts them)
    zkb::CaptureDesc* d_cap_desc = nullptr;
    uint8_t* d_cap_raw = nullptr;            // raw bytes of the listed constants >= p, cap_raw_stride each
    uint32_t cap_raw_stride = 0;
    uint32_t* d_cap_unsunk = nullptr;        // device ops whose F_SINK the list cleared (restored when the list goes)
    uint32_t cap_n_unsunk = 0;
    uint8_t* d_cap_out = nullptr;            // n_batch x cap_n x cap_E bytes, witness-major
    size_t cap_out_bytes = 0;
    uint32_t cap_E = 0;
    bool cap_valid = false;                  // d_cap_out holds a run over the current list and inputs

    zkb::R1csDev* r1cs = nullptr;
    zkb::GroupJit* gjit = nullptr;   // run-time specialisation of the call-group kernel (group_jit.cpp), if any

    // multi-GPU (include/zkb.h section 7): this context's rank in a communicator, and whether its program is a replica
    // received from the root rank (device plan + the host tables evaluation and read-back need; nothing was recorded here)
    zkb::CommState* comm = nullptr;
    bool is_replica = false;
    uint64_t replica_n_ops = 0, replica_n_values = 0;
    uint32_t *d_tab_slot = nullptr, *d_tab_opb = nullptr;      // replica: value -> slot / operand b, on the device
    uint8_t *d_tab_readable = nullptr, *d_tab_kind = nullptr;  // replica: value -> readable / kind

    int fail(int code, const std::string& msg) {
        err = msg;
        return code;
    }
};

namespace zkb {
// shared helpers implemented in backend.cu
int ctx_upload_groups(zkb_ctx* c);  // plan.group_* -> device
// group_jit.cpp
void group_jit_start(zkb_ctx* c);
void group_jit_free(zkb_ctx* c);
int group_jit_wait(zkb_ctx* c);
int group_jit_state(zkb_ctx* c);
const char* group_jit_log(zkb_ctx* c);
const char* group_jit_source(zkb_ctx* c);
double group_jit_compile_seconds(zkb_ctx* c);
bool group_jit_launch(zkb_ctx* c, const zkb::GroupDesc* d_descs, uint32_t n_groups, uint64_t total_calls, const uint32_t* d_hints,
                      uint32_t log2_words, void* stream);
int ctx_result_buffer(zkb_ctx* c, size_t n_words);  // c->h_res holds at least n_words
int ctx_finalize(zkb_ctx* c, int keep_values);  // 0 live wires, 1 all values, 2 verdicts only
bool ctx_record_ok(zkb_ctx* c);  // false when a recording error is latched
void ctx_latch(zkb_ctx* c, const std::string& msg);
void r1cs_free(zkb_ctx* c);
int ctx_run(zkb_ctx* c, zkb_verdict* out, uint32_t first, uint32_t n_total, bool collective);
void ctx_finish_e2e_timing(zkb_ctx* c);
// the capture list's cleared F_SINK flags: back on (set = true) or off again, in the device ops
void capture_mark_sinks(zkb_ctx* c, bool set);
// forget the capture list; restore_sinks = false when the device ops it changed are being replaced
void capture_reset(zkb_ctx* c, bool restore_sinks);
// comm.cu
int comm_allreduce_min_u32(zkb_ctx* c, uint32_t* d_buf, size_t n);  // in place, on c->stream
void comm_free(zkb_ctx* c);
}  // namespace zkb
