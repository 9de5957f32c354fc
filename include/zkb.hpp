// zkb.hpp — header-only C++ mirror of the reference's consumer API over the C ABI of zkb.h.
//
// The reference is Rust; where a C++ host wants the same shapes, these classes carry the reference's names and
// call order (file:line into /root/reference/rust/src):
//   zkb::Source      consumers/source.rs:45-118     from_directory / from_dirs_and_files / from_buffers
//   zkb::GpuBackend  consumers/evaluator.rs:17-76   one method per `trait ZKBackend` method (deferred, batched)
//   zkb::Evaluator   consumers/evaluator.rs:158-753 from_messages / ingest_message / get_violations / get
//   zkb::Validator   consumers/validator.rs:68-152  new_as_prover / new_as_verifier / ingest_message / get_violations
//   zkb::Stats       consumers/stats.rs:43-112      from_messages / ingest_message, to_json_pretty (serde_json)
// Errors: the reference's `Result<T, Box<dyn Error>>` becomes zkb::Error (code = zkb_status, what() = the text).
#ifndef ZKB_HPP
#define ZKB_HPP

#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "zkb.h"

namespace zkb {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

using Value = std::vector<uint8_t>;  // structs/value.rs:11: little-endian bytes

// consumers/source.rs:45-118
class Source {
public:
    static Source from_directory(const std::string& path) { return from_dirs_and_files({path}); }
    static Source from_dirs_and_files(std::vector<std::string> paths) {
        Source s;
        s.paths_ = std::move(paths);
        return s;
    }
    static Source from_buffers(std::vector<std::vector<uint8_t>> buffers) {
        Source s;
        s.buffers_ = std::move(buffers);
        s.in_memory_ = true;
        return s;
    }
    bool in_memory() const { return in_memory_; }
    const std::vector<std::string>& paths() const { return paths_; }
    const std::vector<std::vector<uint8_t>>& buffers() const { return buffers_; }

private:
    std::vector<std::string> paths_;
    std::vector<std::vector<uint8_t>> buffers_;
    bool in_memory_ = false;
};

namespace detail {
template <class H, class IngestBuffer, class IngestPaths, class Check>
void ingest_source(H* h, const Source& src, IngestBuffer ingest_buffer, IngestPaths ingest_paths, Check check) {
    if (src.in_memory()) {
        for (const auto& b : src.buffers()) check(ingest_buffer(h, b.data(), b.size()));
    } else {
        std::vector<const char*> ptrs;
        for (const auto& p : src.paths()) ptrs.push_back(p.c_str());
        check(ingest_paths(h, ptrs.data(), ptrs.size()));
    }
}
}  // namespace detail

// `impl ZKBackend`: Wire = SSA handle, FieldElement = little-endian bytes.  device < 0: host-only (record / flatten).
class GpuBackend {
public:
    using Wire = zkb_wire;
    using FieldElement = Value;

    explicit GpuBackend(int device = 0) : ctx_(zkb_create(device)) {
        if (device >= 0 && zkb_last_error(ctx_)[0]) {
            std::string m = zkb_last_error(ctx_);
            zkb_destroy(ctx_);
            throw Error(ZKB_E_CUDA, m);
        }
    }
    ~GpuBackend() { zkb_destroy(ctx_); }
    GpuBackend(const GpuBackend&) = delete;
    GpuBackend& operator=(const GpuBackend&) = delete;

    static FieldElement from_bytes_le(const uint8_t* val, size_t len) { return FieldElement(val, val + len); }
    void set_field(const Value& modulus, uint32_t degree = 1, bool is_boolean = false) {
        check(zkb_set_field(ctx_, modulus.data(), modulus.size(), degree, is_boolean));
    }
    FieldElement one() { return element(zkb_one); }
    FieldElement minus_one() { return element(zkb_minus_one); }
    FieldElement zero() { return element(zkb_zero); }
    Wire copy(Wire a) { Wire o; check(zkb_copy(ctx_, a, &o)); return o; }
    Wire constant(const FieldElement& v) { Wire o; check(zkb_constant(ctx_, v.data(), v.size(), &o)); return o; }
    void assert_zero(Wire a, uint64_t src_wire_id = 0) { check(zkb_assert_zero(ctx_, a, src_wire_id)); }
    Wire add(Wire a, Wire b) { Wire o; check(zkb_add(ctx_, a, b, &o)); return o; }
    Wire multiply(Wire a, Wire b) { Wire o; check(zkb_multiply(ctx_, a, b, &o)); return o; }
    Wire add_constant(Wire a, const FieldElement& v) { Wire o; check(zkb_add_constant(ctx_, a, v.data(), v.size(), &o)); return o; }
    Wire mul_constant(Wire a, const FieldElement& v) { Wire o; check(zkb_mul_constant(ctx_, a, v.data(), v.size(), &o)); return o; }
    Wire and_(Wire a, Wire b) { Wire o; check(zkb_and(ctx_, a, b, &o)); return o; }
    Wire xor_(Wire a, Wire b) { Wire o; check(zkb_xor(ctx_, a, b, &o)); return o; }
    Wire not_(Wire a) { Wire o; check(zkb_not(ctx_, a, &o)); return o; }
    Wire instance() { Wire o; check(zkb_instance(ctx_, &o)); return o; }
    Wire witness() { Wire o; check(zkb_witness(ctx_, &o)); return o; }

    // batched evaluation (zkb.h section 3)
    void set_limits(uint64_t max_values, uint64_t max_steps) { check(zkb_set_limits(ctx_, max_values, max_steps)); }
    void finalize(int keep_values = 0) { check(zkb_finalize(ctx_, keep_values)); }
    std::vector<zkb_verdict> evaluate(const uint8_t* instances, uint64_t instance_set_stride, const uint8_t* witnesses,
                                      uint64_t witness_set_stride, uint32_t value_stride, uint32_t n_batch) {
        std::vector<zkb_verdict> out(n_batch);
        check(zkb_evaluate(ctx_, instances, instance_set_stride, witnesses, witness_set_stride, value_stride, n_batch, out.data()));
        return out;
    }
    // values of every witness of each following run (zkb_capture_values); empty clears the list
    void capture(const std::vector<Wire>& values) { check(zkb_capture_values(ctx_, values.data(), values.size())); }
    // witnesses [first, first + n_witnesses) of the last run, value-minor: n_witnesses x n_values x stride bytes
    std::vector<uint8_t> read_captured(uint32_t first, uint32_t n_witnesses, uint64_t n_values, size_t stride = 32) {
        std::vector<uint8_t> out((size_t)n_witnesses * n_values * stride);
        check(zkb_read_captured(ctx_, first, n_witnesses, out.data(), stride));
        return out;
    }
    std::vector<uint8_t> read_values(uint32_t batch_idx, const std::vector<Wire>& values, size_t stride = 32) {
        std::vector<uint8_t> out(values.size() * stride);
        check(zkb_read_values(ctx_, batch_idx, values.data(), values.size(), out.data(), stride));
        return out;
    }
    zkb_stats stats() { zkb_stats s; check(zkb_get_stats(ctx_, &s)); return s; }
    const char* pending_error() { return zkb_pending_error(ctx_); }
    zkb_ctx* raw() { return ctx_; }

private:
    void check(int rc) {
        if (rc != ZKB_OK) throw Error(rc, zkb_last_error(ctx_));
    }
    template <class F>
    FieldElement element(F f) {
        uint8_t buf[64];
        size_t n = 0;
        check(f(ctx_, buf, sizeof buf, &n));
        return FieldElement(buf, buf + n);
    }
    zkb_ctx* ctx_;
};

// `Evaluator<B>` over `.sieve` bytes
class Evaluator {
public:
    explicit Evaluator(GpuBackend& backend) : backend_(backend), ev_(zkb_evaluator_create(backend.raw())) {}
    ~Evaluator() { zkb_evaluator_destroy(ev_); }
    Evaluator(const Evaluator&) = delete;
    Evaluator& operator=(const Evaluator&) = delete;

    // Evaluator::from_messages(source.iter_messages(), &mut backend): construct, then ingest the source
    void from_messages(const Source& src) {
        detail::ingest_source(ev_, src, zkb_evaluator_ingest_buffer, zkb_evaluator_ingest_paths, [&](int rc) { check(rc); });
    }
    void ingest_message(const uint8_t* buf, size_t len) { check(zkb_evaluator_ingest_message(ev_, buf, len)); }
    std::vector<std::string> get_violations() {
        size_t n = 0;
        check(zkb_evaluator_get_violations(ev_, &n));
        std::vector<std::string> v;
        for (size_t i = 0; i < n; i++) v.emplace_back(zkb_evaluator_violation(ev_, i));
        return v;
    }
    Value get(uint64_t wire_id) {  // Evaluator::get, evaluator.rs:750-752
        uint8_t buf[64];
        size_t n = 0;
        check(zkb_evaluator_get_wire(ev_, wire_id, buf, sizeof buf, &n));
        return Value(buf, buf + n);
    }
    // flatten / expand-definable (consumers/flattening.rs, exp_definable.rs): choose before ingesting
    void set_flatten(bool on = true) { check(zkb_evaluator_set_flatten(ev_, on)); }
    void set_expand_definable(const std::string& gate_set) { check(zkb_evaluator_set_expand_definable(ev_, gate_set.c_str())); }
    void flatten_to_dir(const std::string& out_dir) { check(zkb_evaluator_flatten_to_dir(ev_, out_dir.c_str())); }
    struct Flattened {
        std::vector<uint8_t> instance, witness, relation;
    };
    Flattened flatten() {
        const uint8_t* p[3];
        size_t n[3];
        check(zkb_evaluator_flatten(ev_, &p[0], &n[0], &p[1], &n[1], &p[2], &n[2]));
        return Flattened{{p[0], p[0] + n[0]}, {p[1], p[1] + n[1]}, {p[2], p[2] + n[2]}};
    }
    GpuBackend& backend() { return backend_; }

    // value sets (zkb.h section 4): one relation, one statement per set; every set before the first relation message
    void add_value_set(const Source& src) {
        if (src.in_memory()) {
            std::vector<uint8_t> all;
            for (const auto& b : src.buffers()) all.insert(all.end(), b.begin(), b.end());
            check(zkb_evaluator_add_value_set_buffer(ev_, all.data(), all.size()));
        } else {
            std::vector<const char*> ptrs;
            for (const auto& p : src.paths()) ptrs.push_back(p.c_str());
            check(zkb_evaluator_add_value_set_paths(ev_, ptrs.data(), ptrs.size()));
        }
    }
    // the contexts of one communicator (zkb_comm_init order), ctxs[0] = backend().raw()
    void use_devices(std::vector<zkb_ctx*> ctxs) { check(zkb_evaluator_use_devices(ev_, ctxs.data(), (int)ctxs.size())); }
    struct SetResult {
        int status;                           // ZKB_OK, or ZKB_E_FATAL: the statement panics, violations[0] is the panic text
        std::vector<std::string> violations;  // what get_violations returns for the set's statement
    };
    std::vector<SetResult> get_batch_violations() {
        std::vector<SetResult> out;
        const size_t n_sets = zkb_evaluator_value_sets(ev_);
        if (n_sets == 0) check(zkb_evaluator_batch_result(ev_, 0, nullptr, nullptr));
        for (size_t j = 0; j < n_sets; j++) {
            SetResult r;
            size_t n = 0;
            check(zkb_evaluator_batch_result(ev_, j, &r.status, &n));
            for (size_t i = 0; i < n; i++) r.violations.emplace_back(zkb_evaluator_batch_violation(ev_, j, i));
            out.push_back(std::move(r));
        }
        return out;
    }
    Value get(uint64_t set, uint64_t wire_id) {  // Evaluator::get for one set
        uint8_t buf[64];
        size_t n = 0;
        check(zkb_evaluator_get_wire_of(ev_, set, wire_id, buf, sizeof buf, &n));
        return Value(buf, buf + n);
    }

private:
    void check(int rc) {
        if (rc != ZKB_OK) throw Error(rc, zkb_evaluator_last_error(ev_));
    }
    GpuBackend& backend_;
    zkb_evaluator* ev_;
};

class Validator {
public:
    static Validator new_as_prover() { return Validator(true); }
    static Validator new_as_verifier() { return Validator(false); }
    explicit Validator(bool as_prover) : v_(zkb_validator_create(as_prover)) {}
    Validator(Validator&& o) noexcept : v_(o.v_) { o.v_ = nullptr; }
    ~Validator() {
        if (v_) zkb_validator_destroy(v_);
    }
    void ingest_message(const uint8_t* buf, size_t len) { check(zkb_validator_ingest_message(v_, buf, len)); }
    void ingest_source(const Source& src) {
        detail::ingest_source(v_, src, zkb_validator_ingest_buffer, zkb_validator_ingest_paths, [&](int rc) { check(rc); });
    }
    size_t how_many_violations() { return zkb_validator_how_many_violations(v_); }
    std::vector<std::string> get_violations() {
        size_t n = 0;
        check(zkb_validator_get_violations(v_, &n));
        std::vector<std::string> out;
        for (size_t i = 0; i < n; i++) out.emplace_back(zkb_validator_violation(v_, i));
        return out;
    }

private:
    void check(int rc) {
        if (rc != ZKB_OK) throw Error(rc, zkb_validator_last_error(v_));
    }
    zkb_validator* v_;
};

class Stats {
public:
    Stats() : m_(zkb_metrics_create()) {}
    ~Stats() { zkb_metrics_destroy(m_); }
    Stats(const Stats&) = delete;
    Stats& operator=(const Stats&) = delete;
    void ingest_message(const uint8_t* buf, size_t len) { check(zkb_metrics_ingest_message(m_, buf, len)); }
    void from_messages(const Source& src) {
        detail::ingest_source(m_, src, zkb_metrics_ingest_buffer, zkb_metrics_ingest_paths, [&](int rc) { check(rc); });
    }
    std::string to_json_pretty() { return zkb_metrics_json(m_); }

private:
    void check(int rc) {
        if (rc != ZKB_OK) throw Error(rc, zkb_metrics_last_error(m_));
    }
    zkb_metrics* m_;
};

}  // namespace zkb
#endif  // ZKB_HPP
