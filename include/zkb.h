/* zkb.h — C ABI of the B200 satisfiability evaluator for the zkInterface SIEVE IR.
 *
 * This is the drop-in boundary for ONE path of the reference (dryajov/zkinterface-ir,
 * `zki_sieve` 3.0.0): what `zki_sieve evaluate` does through
 * `Evaluator<PlaintextBackend>` (rust/src/consumers/evaluator.rs), i.e. gate-by-gate
 * evaluation of a relation against instance/witness values, for a whole BATCH of
 * witnesses at once on the GPU.  Plain pointers and sizes only; every entry point
 * cites the reference interface it replaces.  A Rust `impl ZKBackend for GpuBackend`
 * binds section 2 one-to-one (see INTEGRATION.md); section 4 mirrors `Evaluator` +
 * `Source` for callers that start from `.sieve` bytes.
 *
 * Conventions
 *   - every function returns ZKB_OK (0) or a negative zkb_status; the message is
 *     available from zkb_last_error(ctx) until the next call on that ctx.
 *     (reference: `Result<T> = Result<T, Box<dyn Error>>`, rust/src/lib.rs:47)
 *   - an UNSATISFIED statement is not an error: it is reported in zkb_verdict.
 *   - field elements cross the boundary as little-endian byte strings
 *     (`Value`, rust/src/structs/value.rs:11); trailing zeros optional.
 *   - the caller owns all buffers it passes; the library copies what it keeps.
 *   - one ctx = one host thread + one device.  Not thread-safe; contexts are independent.
 *   - there is NO CPU fallback: evaluation entry points fail with ZKB_E_CUDA when the
 *     context has no CUDA device.
 */
#ifndef ZKB_H
#define ZKB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    ZKB_OK = 0,
    ZKB_E_ARG = -1,          /* bad argument / call order */
    ZKB_E_FORMAT = -2,       /* malformed .sieve message (reference: Err("Missing ...")) */
    ZKB_E_SEMANTIC = -3,     /* evaluation error the reference reports as a violation string */
    ZKB_E_CUDA = -4,         /* CUDA runtime failure or no device */
    ZKB_E_FATAL = -5,        /* condition on which the reference PANICS (same text) */
    ZKB_E_UNSUPPORTED = -6   /* outside the device path (field wider than 256 bits, even modulus != 2, ...) */
} zkb_status;

typedef struct zkb_ctx zkb_ctx;

/* ZKBackend::Wire of the GPU backend: an SSA value handle (evaluator.rs:18). */
typedef uint64_t zkb_wire;

/* ------------------------------------------------------------------ 1. lifecycle */
/* device >= 0: CUDA device ordinal.  device < 0: host-only context (record / plan /
 * inspect; every evaluation call fails with ZKB_E_CUDA). */
zkb_ctx* zkb_create(int device);
void zkb_destroy(zkb_ctx* ctx);
const char* zkb_last_error(zkb_ctx* ctx);
/* Resource limits of the host pass (0 keeps the current value).  The reference unrolls whatever the statement
 * says until the host runs out of memory; here a For over 2^60 iterations or a 2^32-wire range in a malformed /
 * hostile message ends in "zkb: resource limit exceeded (...)" (a latched evaluation error).
 *   max_values : SSA values recorded (default and maximum 2^32 - 256, handles are 32-bit)
 *   max_steps  : gates ingested + loop iterations + wires expanded by the Evaluator mirror (default 2^40) */
int zkb_set_limits(zkb_ctx* ctx, uint64_t max_values, uint64_t max_steps);

/* ------------------------------------------------------------------ 2. ZKBackend seam
 * One function per method of `trait ZKBackend` (evaluator.rs:17-76).  The backend is
 * DEFERRED: each call records one SSA op and returns its handle; nothing is computed
 * until zkb_evaluate.  `assert_zero` therefore always returns ZKB_OK — the verdict
 * (which assertion failed first, per witness) comes back from zkb_evaluate. */

/* ZKBackend::set_field (evaluator.rs:28; PlaintextBackend :866-875: "Modulus cannot be
 * zero." / "Field should be of degree 1"). */
int zkb_set_field(zkb_ctx* ctx, const uint8_t* modulus_le, size_t len, uint32_t degree, int is_boolean);
/* ZKBackend::one / minus_one / zero (evaluator.rs:31-35): little-endian bytes into out[cap]. */
int zkb_one(zkb_ctx* ctx, uint8_t* out_le, size_t cap, size_t* len);
int zkb_minus_one(zkb_ctx* ctx, uint8_t* out_le, size_t cap, size_t* len);
int zkb_zero(zkb_ctx* ctx, uint8_t* out_le, size_t cap, size_t* len);
/* ZKBackend::copy (evaluator.rs:38) — an alias: returns the same handle. */
int zkb_copy(zkb_ctx* ctx, zkb_wire a, zkb_wire* out);
/* ZKBackend::constant (evaluator.rs:41). */
int zkb_constant(zkb_ctx* ctx, const uint8_t* val_le, size_t len, zkb_wire* out);
/* ZKBackend::assert_zero (evaluator.rs:46).  src_wire_id: the IR wire id the Evaluator
 * would print in "Wire_{id} (may be weighted) should be 0, while it is not" (:357-362). */
int zkb_assert_zero(zkb_ctx* ctx, zkb_wire a, uint64_t src_wire_id);
/* ZKBackend::add / multiply / add_constant / mul_constant (evaluator.rs:49-55). */
int zkb_add(zkb_ctx* ctx, zkb_wire a, zkb_wire b, zkb_wire* out);
int zkb_multiply(zkb_ctx* ctx, zkb_wire a, zkb_wire b, zkb_wire* out);
int zkb_add_constant(zkb_ctx* ctx, zkb_wire a, const uint8_t* val_le, size_t len, zkb_wire* out);
int zkb_mul_constant(zkb_ctx* ctx, zkb_wire a, const uint8_t* val_le, size_t len, zkb_wire* out);
/* ZKBackend::and / xor / not (evaluator.rs:58-62). */
int zkb_and(zkb_ctx* ctx, zkb_wire a, zkb_wire b, zkb_wire* out);
int zkb_xor(zkb_ctx* ctx, zkb_wire a, zkb_wire b, zkb_wire* out);
int zkb_not(zkb_ctx* ctx, zkb_wire a, zkb_wire* out);
/* ZKBackend::instance / witness (evaluator.rs:66-75).  The VALUE is not passed here: the
 * call reserves the next position of the instance / witness stream, and the values of all
 * witnesses of a batch are supplied to zkb_evaluate (consumption is data-independent, so
 * one recorded program serves every witness). */
int zkb_instance(zkb_ctx* ctx, zkb_wire* out);
int zkb_witness(zkb_ctx* ctx, zkb_wire* out);

/* ------------------------------------------------------------------ 3. bulk gates, evaluation */

/* Flat gates = the simple arms of Evaluator::ingest_gate (evaluator.rs:344-439), as an
 * array.  Wire ids are IR wire ids of ONE scope (re-usable after FREE); errors and their
 * texts follow evaluator.rs:775-797 ("Wire_{id} already has a value in this scope." /
 * "No value given for wire_{id}"). */
typedef enum {
    ZKB_G_CONSTANT = 1, /* out, b = index into the constant pool      gates.rs:20 */
    ZKB_G_ASSERT_ZERO,  /* a                                            gates.rs:22 */
    ZKB_G_COPY,         /* out, a */
    ZKB_G_ADD,          /* out, a, b */
    ZKB_G_MUL,          /* out, a, b */
    ZKB_G_ADD_CONSTANT, /* out, a, b = constant-pool index */
    ZKB_G_MUL_CONSTANT, /* out, a, b = constant-pool index */
    ZKB_G_AND,          /* out, a, b */
    ZKB_G_XOR,          /* out, a, b */
    ZKB_G_NOT,          /* out, a */
    ZKB_G_INSTANCE,     /* out */
    ZKB_G_WITNESS,      /* out */
    ZKB_G_FREE          /* a = first, b = last (inclusive; b < a frees nothing) */
} zkb_gate_op;          /* same numbering as DirectiveSet 1..13, sieve_ir_generated.rs:422-442 */

typedef struct {
    uint8_t op; /* zkb_gate_op */
    uint8_t pad[3];
    uint32_t out;
    uint32_t a;
    uint32_t b;
} zkb_gate;

/* const_pool_le: n_consts values of const_stride bytes each (little-endian). */
int zkb_push_gates(zkb_ctx* ctx, const zkb_gate* gates, uint64_t n_gates, const uint8_t* const_pool_le,
                   size_t const_stride, uint64_t n_consts);

/* Host preparation: levelize the recorded SSA list into wavefronts, assign wire-store slots
 * (liveness-based re-use), fuse assertions, upload the device program.  keep_values:
 *   0  values bound to wires that are still live in the top scope stay readable (zkb_read_values,
 *      Evaluator::get) — the state the reference's Evaluator holds when it finishes;
 *   1  every recorded value stays readable (wire-by-wire parity checks; no slot re-use);
 *   2  verdicts only: nothing is kept, slots are re-used as soon as their last reader ran. */
int zkb_finalize(zkb_ctx* ctx, int keep_values);

typedef struct {
    uint8_t ok; /* 1: every assertion holds for this witness (the statement is TRUE) */
    uint8_t pad[7];
    uint64_t first_fail_seq; /* index (program order) of the first failing assert_zero; UINT64_MAX if none */
} zkb_verdict;

/* Evaluate the program for n_batch independent (instance, witness) pairs.
 *   instances_le : n_instance values of value_stride bytes per pair; pair j at
 *                  instances_le + j*instance_set_stride (instance_set_stride 0: one shared vector)
 *   witnesses_le : likewise for the short witness.
 * Timed end-to-end by bench.py: H2D of inputs, all kernels, D2H of the verdicts.
 * Replaces the per-gate loop Evaluator::ingest_relation -> ingest_gate -> PlaintextBackend
 * (evaluator.rs:288-301, 318-439, 908-938). */
int zkb_evaluate(zkb_ctx* ctx, const uint8_t* instances_le, uint64_t instance_set_stride, const uint8_t* witnesses_le,
                 uint64_t witness_set_stride, uint32_t value_stride, uint32_t n_batch, zkb_verdict* out);
/* The same in two steps, so a caller can keep inputs resident in HBM and re-run. */
int zkb_upload_inputs(zkb_ctx* ctx, const uint8_t* instances_le, uint64_t instance_set_stride, const uint8_t* witnesses_le,
                      uint64_t witness_set_stride, uint32_t value_stride, uint32_t n_batch);
int zkb_run(zkb_ctx* ctx, zkb_verdict* out);

/* IR wire id recorded with assertion `seq` (for the reference's violation text). */
int zkb_assert_info(zkb_ctx* ctx, uint64_t seq, uint64_t* src_wire_id);
/* Error found while RECORDING (e.g. "No value given for wire_7"); the reference reports it as
 * the violation unless an assertion failed earlier in program order.  NULL if none. */
const char* zkb_pending_error(zkb_ctx* ctx);

/* Canonical residues (little-endian, `stride` bytes each, zero padded) of recorded values for
 * witness batch_idx of the last evaluation — what Evaluator::get (evaluator.rs:750-752) returns
 * for wires bound to those values.  Requires zkb_finalize(ctx, 1). */
int zkb_read_values(zkb_ctx* ctx, uint32_t batch_idx, const zkb_wire* values, uint64_t n, uint8_t* out_le, size_t stride);
/* Values to capture on every following run (zkb_evaluate / zkb_run / zkb_comm_* / *_sharded), for every witness of the
 * batch: the device writes them out tile by tile while the batch is evaluated, so no tile is run again to read them.
 * After zkb_finalize; n = 0 clears the list.  Same readability rule and errors as zkb_read_values.  A new zkb_finalize
 * (or a program broadcast to this rank) clears the list.  A captured value that no gate reads is stored on every tile. */
int zkb_capture_values(zkb_ctx* ctx, const zkb_wire* values, uint64_t n);
/* What the last run captured for this context's witnesses [first, first + n_witnesses):
 * out_le[(j - first) * n * stride + i * stride] = value i of witness j, in the bytes zkb_read_values(ctx, j, ...) returns
 * (canonical residue; the raw bytes of an instance / witness value or of a constant >= p; 0/1 over p = 2).  Needs a run
 * since the last zkb_capture_values, zkb_finalize or input upload.  On a rank of a communicator, j indexes the rank's own
 * block of the batch. */
int zkb_read_captured(zkb_ctx* ctx, uint32_t first, uint32_t n_witnesses, uint8_t* out_le, size_t stride);
/* value currently bound to IR wire id `wire` in the flat scope of zkb_push_gates */
int zkb_scope_lookup(zkb_ctx* ctx, uint64_t wire, zkb_wire* out);

typedef struct {
    uint64_t n_values;      /* SSA values recorded */
    uint64_t n_asserts;
    uint64_t n_instance;    /* values consumed from the instance stream per pair */
    uint64_t n_witness;
    uint64_t n_consts;
    uint64_t ir_gates;      /* Add/Mul/AddConstant/MulConstant/And/Xor/Not/AssertZero gates ingested */
    uint64_t callbacks[12]; /* constant, instance, witness, add, mul, addc, mulc, and, xor, not, copy, assert_zero */
    uint64_t n_slots;       /* wire-store slots (after finalize) */
    uint64_t n_levels;
    uint64_t n_device_ops;
    uint64_t algo_bytes_per_witness; /* SURVEY.md section 8d algorithmic bytes */
    uint32_t nlimb;         /* 32-bit limbs per element (0 before set_field) */
    uint32_t binary;        /* p == 2 */
    uint32_t tile_witnesses;/* witnesses resident per pass (after upload) */
    uint32_t n_tiles;
    uint64_t n_call_groups; /* For loops over a plain function or an anonymous body of plain gates kept as ONE
                             * loop-structured descriptor each (evaluator.rs:495-559 + :441-471; over a prime field: loops of
                             * >= 1024 calls whose body holds Constant / Add / Mul / AddConstant / MulConstant and AssertZero
                             * on computed wires, carried loops included): the device expands them, only the calls' outputs
                             * are SSA values (kind 11 in zkb_get_program) */
    uint64_t n_group_calls; /* function calls those groups stand for */
    uint64_t n_group_launches;     /* after finalize: kernel launches that expand them (one per dependency depth) */
    uint64_t n_group_table_slots;  /* after finalize: operand slots listed explicitly (inputs whose slots are not an
                                    * arithmetic progression over the calls) */
    int64_t group_jit_state;       /* the groups' run-time specialised kernel: -2 none, -1 unavailable (the interpreter kernel
                                    * runs; always so over a prime field), 0 compiling in the background, 2 compiled, 3 loaded
                                    * and in use */
    uint64_t n_sink_ops;           /* after finalize: stored results that no gate reads (only a read-back needs them; tiles
                                    * other than the last one run skip their stores) */
    uint64_t n_carried_groups;     /* of n_call_groups, the carried loops (prime fields): call c reads output k of call c - d,
                                    * 1 <= d <= 4 (over fields of at most 64 bits: loops of >= 2^20 calls), and calls c < d read seeds that are
                                    * instance / witness / constant values or
                                    * outputs of earlier groups.  Each runs as a chain, one thread per witness walking the calls
                                    * in order; they count in n_group_calls and n_group_launches too */
} zkb_stats;
int zkb_get_stats(zkb_ctx* ctx, zkb_stats* out);

/* Inspection of the recorded SSA program (host preparation parity checks): values
 * [first, first+n) -> kind (0 const, 1 instance, 2 witness, 3 add, 4 mul, 5 addc, 6 mulc, 7 and,
 * 8 xor, 9 not, 11 output of a call group: a = group, b = call * n_outputs + position), operand a (value handle), operand b (value handle, or constant-pool index for
 * const/addc/mulc, or stream position for instance/witness). */
int zkb_get_program(zkb_ctx* ctx, uint64_t first, uint64_t n, uint8_t* kinds, uint32_t* a, uint32_t* b);
/* canonical residue of constant-pool entry idx (little-endian) */
int zkb_get_const(zkb_ctx* ctx, uint64_t idx, uint8_t* out_le, size_t cap, size_t* len);
/* wavefront `level` of the device plan: out[0] gates, out[1] of which Add/Mul/AddC/MulC, out[2] with a fused
 * assertion, out[3] not stored, out[4] algorithmic bytes per witness (3E per two-operand gate, 2E per
 * one-operand gate, E per assertion; SURVEY.md section 8d) */
int zkb_level_info(zkb_ctx* ctx, uint64_t level, uint64_t out[5]);
/* asserted value handle of assertion seq; ZKB_E_ARG for an assertion inside a call group (its value is a call-local wire
 * without a handle; zkb_assert_info still gives its local wire id) */
int zkb_assert_value(zkb_ctx* ctx, uint64_t seq, zkb_wire* value);

typedef struct {
    float h2d_ms;       /* input upload */
    float load_ms;      /* input-conversion kernels */
    float levels_ms;    /* all level kernels (CUDA events on the library's stream) */
    float total_ms;     /* first byte uploaded .. verdicts on host */
    uint64_t level_launches;
    uint64_t kernel_launches;
} zkb_timing;
int zkb_get_timing(zkb_ctx* ctx, zkb_timing* out);

/* ------------------------------------------------------------------ 4. Evaluator / Source
 * Mirror of `Evaluator<B>` (evaluator.rs:158-753) driven from `.sieve` bytes, with `Source`
 * (rust/src/consumers/source.rs:59-118) file discovery and ordering.  The evaluator records
 * into `backend`; get_violations triggers the GPU evaluation and reproduces the reference's
 * violation strings (evaluator.rs:199-208, 357-362). */
typedef struct zkb_evaluator zkb_evaluator;
zkb_evaluator* zkb_evaluator_create(zkb_ctx* backend);
void zkb_evaluator_destroy(zkb_evaluator* ev);
/* Evaluator::ingest_message on ONE size-prefixed FlatBuffers message (Message::try_from). */
int zkb_evaluator_ingest_message(zkb_evaluator* ev, const uint8_t* buf, size_t len);
/* Source::from_buffers + iter_messages: a concatenation of size-prefixed messages. */
int zkb_evaluator_ingest_buffer(zkb_evaluator* ev, const uint8_t* buf, size_t len);
/* Source::from_dirs_and_files + Evaluator::from_messages: files / directories of *.sieve,
 * ordered instance < witness < relation (source.rs:69-89). */
int zkb_evaluator_ingest_paths(zkb_evaluator* ev, const char* const* paths, size_t n_paths);
/* Evaluator::get_violations: evaluates (once) and returns the number of violation strings. */
int zkb_evaluator_get_violations(zkb_evaluator* ev, size_t* n_violations);
const char* zkb_evaluator_violation(zkb_evaluator* ev, size_t i);
/* Evaluator::get(id): canonical little-endian residue of a live top-scope wire. */
int zkb_evaluator_get_wire(zkb_evaluator* ev, uint64_t wire_id, uint8_t* out_le, size_t cap, size_t* len);
/* value handle (for zkb_read_values on any witness of a batch) bound to a live top-scope wire */
int zkb_evaluator_lookup(zkb_evaluator* ev, uint64_t wire_id, zkb_wire* out);
const char* zkb_evaluator_last_error(zkb_evaluator* ev);

/* Value sets: one relation checked against many instance / witness sets in one device batch.  A value set is a group of
 * Instance / Witness messages; values ingested with the calls above are COMMON to every set.  Set j's statement is: the
 * common instance messages, then set j's; the common witness messages, then set j's; the relation message(s).  Its result
 * is what zkb_evaluator_get_violations returns for that statement on its own (evaluator.rs:199-208).
 * Batch mode begins with the first set; every set must be added before the first relation message, and so must the common
 * values.  The relation is recorded once, against the longest streams; while recording, a panic no longer fails the ingest
 * call: like a recording error, it ends the recording and is decided per set.  Refused with ZKB_E_ARG: a set after a
 * relation message, a Relation message inside a set, a set on a flatten / expand-definable evaluator, get_violations /
 * get_wire once a set is added, a set index out of range.  A host-only backend records; its batch results are ZKB_E_CUDA. */
/* One set from a concatenation of size-prefixed Instance / Witness messages. */
int zkb_evaluator_add_value_set_buffer(zkb_evaluator* ev, const uint8_t* buf, size_t len);
/* One set from files / directories of *.sieve, in Source order (source.rs:69-89); errors name the file. */
int zkb_evaluator_add_value_set_paths(zkb_evaluator* ev, const char* const* paths, size_t n_paths);
/* number of value sets added */
size_t zkb_evaluator_value_sets(zkb_evaluator* ev);
/* Split the batch over the contexts of one communicator (zkb_comm_init, same order; ctxs[0] is the evaluator's backend)
 * with zkb_evaluate_sharded.  With fewer sets than contexts the batch runs on ctxs[0] alone. */
int zkb_evaluator_use_devices(zkb_evaluator* ev, zkb_ctx** ctxs, int n);
/* Result of set `set`; the first call evaluates the whole batch (once).  *status ZKB_OK: the set's violation strings
 * follow (none: the statement is TRUE); ZKB_E_FATAL: the reference panics on this statement, the one string is the
 * panic text.  The call itself fails only for the whole batch (argument, CUDA). */
int zkb_evaluator_batch_result(zkb_evaluator* ev, uint64_t set, int* status, size_t* n_violations);
const char* zkb_evaluator_batch_violation(zkb_evaluator* ev, uint64_t set, size_t i);
/* Evaluator::get(id) for one set: read back on the context that evaluated it, from the top scope the whole recording left.
 * ZKB_E_FATAL for a set whose statement panics.  ZKB_E_ARG for a set whose recording stops early (a stream of its own runs
 * out, or the relation's own error is reached: its violations end with that error), since its statement's scope at that
 * point can differ from the final one. */
int zkb_evaluator_get_wire_of(zkb_evaluator* ev, uint64_t set, uint64_t wire_id, uint8_t* out_le, size_t cap, size_t* len);

/* `zki_sieve flatten` (cli.rs:442-472): the Evaluator driving the reference's IRFlattener backend
 * (consumers/flattening.rs:42-191) instead of an evaluating one.  Call set_flatten(ev, 1) BEFORE ingesting; the
 * statement is then recorded gate for gate as the IRFlattener's GateBuilder would emit it (one SIMPLE gate per
 * ZKBackend callback incl. copies, wire ids 0, 1, 2, ..., messages of at most 100 000 gates / values) and can be
 * written out, not evaluated (host only, no device needed).
 *   zkb_evaluator_flatten        : MemorySink — three buffers of size-prefixed messages, owned by ev
 *   zkb_evaluator_flatten_to_dir : FilesSink::new_clean — 000_instance / 001_witness / 002_relation .sieve */
int zkb_evaluator_set_flatten(zkb_evaluator* ev, int on);
/* `zki_sieve expand-definable --gate-set <s>` (cli.rs:513-553): flatten mode with `ExpandDefinable`
 * (consumers/exp_definable.rs:24-139) in front of the flattener — gates outside the given gate set ("arithmetic",
 * "boolean" or a comma-separated list of @add,@addc,@mul,@mulc,@xor,@and,@not; relation.rs:144-167) are rewritten
 * (AddConstant/MulConstant -> Constant + Add/Mul, And <-> Mul, Xor <-> Add, Not -> AddConstant(1)); an impossible
 * rewrite is ZKB_E_FATAL with the reference's panic text. */
int zkb_evaluator_set_expand_definable(zkb_evaluator* ev, const char* gate_set);
int zkb_evaluator_flatten(zkb_evaluator* ev, const uint8_t** instance, size_t* instance_len, const uint8_t** witness,
                          size_t* witness_len, const uint8_t** relation, size_t* relation_len);
int zkb_evaluator_flatten_to_dir(zkb_evaluator* ev, const char* out_dir);

/* ------------------------------------------------------------------ 4b. Validator
 * Mirror of `Validator` (rust/src/consumers/validator.rs:68-829): the semantic / syntactic checks of
 * `zki_sieve validate` and `valid-eval-metrics` (cli.rs:302-313, 333-363), with the reference's violation texts.
 * Host only.  as_prover 1: Validator::new_as_prover, 0: new_as_verifier (:108-117). */
typedef struct zkb_validator zkb_validator;
zkb_validator* zkb_validator_create(int as_prover);
void zkb_validator_destroy(zkb_validator* v);
/* Validator::ingest_message on one size-prefixed message / a concatenation of messages / Source paths */
int zkb_validator_ingest_message(zkb_validator* v, const uint8_t* buf, size_t len);
int zkb_validator_ingest_buffer(zkb_validator* v, const uint8_t* buf, size_t len);
int zkb_validator_ingest_paths(zkb_validator* v, const char* const* paths, size_t n_paths);
/* Validator::get_violations (:136-144): runs the end-of-statement checks once, returns the number of violations */
int zkb_validator_get_violations(zkb_validator* v, size_t* n_violations);
const char* zkb_validator_violation(zkb_validator* v, size_t i);
/* Validator::how_many_violations (:150-152): violations so far, without the end-of-statement checks */
size_t zkb_validator_how_many_violations(zkb_validator* v);
/* wires still live (the reference prints "WARNING: few variables were not freed." when non-zero, :139-141) */
uint64_t zkb_validator_live_wires(zkb_validator* v);
/* loop / expansion budget (gates + loop iterations + wires expanded); default 2^40, 0 keeps the current value */
int zkb_validator_set_limits(zkb_validator* v, uint64_t max_steps);
const char* zkb_validator_last_error(zkb_validator* v);

/* ------------------------------------------------------------------ 4c. Stats
 * Mirror of `Stats` (rust/src/consumers/stats.rs:11-287): what the `metrics` / `valid-eval-metrics` verbs print
 * (cli.rs:322-363).  zkb_metrics_json: the JSON `serde_json::to_writer_pretty(&stats)` writes (fields in declaration
 * order; `functions` is a HashMap in the reference, so its key order is unspecified there, sorted here).  Host only. */
typedef struct zkb_metrics zkb_metrics;
zkb_metrics* zkb_metrics_create(void);
void zkb_metrics_destroy(zkb_metrics* m);
int zkb_metrics_ingest_message(zkb_metrics* m, const uint8_t* buf, size_t len);
int zkb_metrics_ingest_buffer(zkb_metrics* m, const uint8_t* buf, size_t len);
int zkb_metrics_ingest_paths(zkb_metrics* m, const char* const* paths, size_t n_paths);
const char* zkb_metrics_json(zkb_metrics* m);
const char* zkb_metrics_last_error(zkb_metrics* m);

/* ------------------------------------------------------------------ 5. R1CS (Az o Bz = Cz)
 * The satisfiability check that `zkif-to-ir` + `evaluate` performs gate by gate on an R1CS
 * (rust/src/producers/from_r1cs.rs:110-125), done as three CSR sparse mod-p mat-vecs and a
 * fused Hadamard check.  Row r holds  (A_r . z)(B_r . z) - (C_r . z) == 0 (mod p). */
typedef struct {
    uint64_t n_rows;
    const uint64_t* row_ptr;  /* n_rows + 1 */
    const uint32_t* col;      /* variable ids, nnz */
    const uint32_t* coef_idx; /* index into the coefficient table, nnz */
} zkb_csr;
int zkb_r1cs_load(zkb_ctx* ctx, const zkb_csr* A, const zkb_csr* B, const zkb_csr* C, const uint8_t* coef_table_le,
                  size_t coef_stride, uint64_t n_coefs, uint64_t n_vars);
/* z_le: n_batch assignment vectors of n_vars values (z[0] must be 1), value_stride bytes each.
 * verdict.first_fail_seq = first violated row. */
int zkb_r1cs_check(zkb_ctx* ctx, const uint8_t* z_le, uint64_t z_set_stride, uint32_t value_stride, uint32_t n_batch,
                   zkb_verdict* out);
int zkb_r1cs_upload(zkb_ctx* ctx, const uint8_t* z_le, uint64_t z_set_stride, uint32_t value_stride, uint32_t n_batch);
int zkb_r1cs_run(zkb_ctx* ctx, zkb_verdict* out);

/* ------------------------------------------------------------------ 6. debug / measurement
 * Not part of the drop-in surface.  field_ops: r[i] = a[i] op b[i] on the device for n elements of nlimb 32-bit
 * limbs (op 0: modular add; 1: Montgomery product as the kernels compute it; 2: portable CIOS product).
 * field_throughput: register-resident dependent chains of `iters` operations per thread -> operations/s. */
int zkb_debug_field_ops(zkb_ctx* ctx, int op, const uint32_t* a, const uint32_t* b, uint32_t* r, uint64_t n);
int zkb_debug_field_throughput(zkb_ctx* ctx, int op, uint32_t iters, double* ops_per_second);
/* Call groups are expanded by an interpreter kernel at first; meanwhile their templates are compiled (NVRTC, background thread)
 * into a kernel that keeps a call's registers in registers, used from the next evaluation after it is ready.  This call
 * blocks until the compilation has ended (state as in zkb_stats.group_jit_state); _source returns the generated CUDA. */
int zkb_debug_group_jit_wait(zkb_ctx* ctx, int* state, double* compile_seconds);
const char* zkb_debug_group_jit_source(zkb_ctx* ctx);
/* random 32-byte gathers (8 in flight per thread, L2-only loads) from a table of table_bytes: bytes gathered per second —
 * the ceiling of the one-assignment R1CS check, whose traffic is z[col] look-ups in a vector larger than L2 */
int zkb_debug_gather_throughput(zkb_ctx* ctx, uint64_t table_bytes, uint32_t iters, double* bytes_per_second);
/* microseconds per barrier of a kernel that only synchronises: kind 0 cooperative_groups' grid.sync(), 1 the counter barrier
 * the all-levels kernel uses, 2 the hardware barrier of one 8-CTA cluster; blocks CTAs of 256 threads (0: one per SM).
 * n_levels x this is the latency floor of a single-witness statement evaluated in one launch. */
int zkb_debug_barrier_cost(zkb_ctx* ctx, int kind, uint32_t blocks, uint32_t n_barriers, double* us_per_barrier);
/* Device layout of kind 0 (tiles of fewer than 32 assignments: ones and general terms in separate classes) or 1 (wider
 * tiles: one class per matrix, ones tagged inside it), host-only contexts: counts = {slices, term groups, rows}; slices: 4 x uint32 per slice
 * {first group, A ones | A general << 16, B ones | B general << 16, C ones | C general << 16} (group counts per term
 * class); terms: 32 x {col, coefficient tag} per group (tag 0xFFFFFFFF: padding, 0xFFFFFFFE: coefficient one, else the
 * table index; zero coefficients are dropped); row_ids: sorted position -> row.  NULL pointers are skipped. */
/* hash of the finalized device plan (ops, assertion table, input loads, slot map): the levelizer's threaded passes must
 * give the plan its sequential form gives (ZKB_PLAN_THREADS) */
int zkb_debug_plan_hash(zkb_ctx* ctx, uint64_t* out);
/* device ops [first, first + n) of the finalized plan: ops4 = 4 x uint32 per op {a, b, out, meta}; values (NULL: skipped) = the
 * SSA value each op computes (0xFFFFFFFF: not stored).  values needs a plan without slot re-use (zkb_finalize(ctx, 1)). */
int zkb_debug_plan_ops(zkb_ctx* ctx, uint64_t first, uint64_t n, uint32_t* ops4, uint32_t* values);
/* FlatBuffers reader -> owned structs -> writer on one size-prefixed message (round-trip tests); *out is valid until
 * the next call on this thread. */
int zkb_debug_rewrite_message(zkb_ctx* ctx, const uint8_t* buf, size_t len, const uint8_t** out, size_t* out_len);
/* zkb_gate[] -> a SIMPLE relation as size-prefixed messages of at most 100 000 gates (GateBuilder + MemorySink,
 * builder.rs:93-98): generator of large `.sieve` inputs for the reader / Evaluator path. */
int zkb_debug_write_flat_relation(zkb_ctx* ctx, const uint8_t* modulus_le, size_t modulus_len, int is_boolean,
                                  const zkb_gate* gates, uint64_t n_gates, const uint8_t* const_pool_le, size_t const_stride,
                                  uint64_t n_consts, const uint8_t** out, size_t* out_len);
int zkb_debug_r1cs_layout(zkb_ctx* ctx, int kind, uint64_t counts[3], uint32_t* slices, uint32_t* terms, uint32_t* row_ids);
/* Cut point of value set `set`, from the recording alone (host-only contexts too): *what 0 none, 1 its instance stream is
 * found empty, 2 its witness stream is found empty, 3 the recording's own error / panic; *seq = assertions recorded before
 * that point (UINT64_MAX: none).  A failing assertion with a smaller seq is the set's violation; else the cut decides. */
int zkb_debug_value_set_cut(zkb_evaluator* ev, uint64_t set, uint64_t* seq, int* what);

/* ------------------------------------------------------------------ 7. multi-GPU (witness-batch sharding)
 * The reference is single-threaded (evaluator.rs:191-230 checks one witness at a time); the path shards over independent
 * witnesses (SURVEY.md section 8e): ONE levelized program, replicated on every device; rank r evaluates a contiguous block
 * of the batch; the only exchange is one MIN all-reduce (NCCL over NVLink) of the per-witness first-failing-assertion
 * vector, i.e. an AND of the verdict bits.  A rank is a context.  The relation is recorded and finalized on ONE rank (the
 * root); zkb_comm_broadcast_program ships its device plan to the others with ncclBroadcast — they never see the relation.
 *
 *   one process, N devices   ctxs[i] = zkb_create(dev_i);  zkb_comm_init(ctxs, N);  record + zkb_finalize on ctxs[0];
 *                            zkb_evaluate_sharded(ctxs, N, ...)           (one host thread per device inside the call)
 *   one process per device   rank 0: zkb_comm_unique_id(&id), hand it to the peers (the launcher's job: MPI, a file, torchrun's
 *                            store); every rank: zkb_comm_init_rank(ctx, &id, N, rank); rank 0 records + finalizes;
 *                            every rank: zkb_comm_broadcast_program(ctx, 0), then zkb_comm_evaluate / zkb_comm_run per batch.
 *
 * The zkb_comm_* calls marked COLLECTIVE must be made by every rank of the communicator; an argument error is reported
 * before anything is exchanged, a CUDA / NCCL failure on one rank inside a collective leaves the others waiting (as with
 * NCCL itself).  NCCL is bound at run time from libnccl.so.2; contexts of ONE process that share a device (a test set-up:
 * NCCL refuses duplicate GPUs) exchange through peer copies on their own streams instead. */
typedef struct {
    uint8_t bytes[128]; /* ncclUniqueId */
} zkb_comm_id;
int zkb_comm_unique_id(zkb_comm_id* out);
int zkb_comm_init_rank(zkb_ctx* ctx, const zkb_comm_id* id, int n_ranks, int rank); /* COLLECTIVE */
/* SURVEY.md section 8b: the contexts of one process form a communicator, rank i = ctxs[i]. */
int zkb_comm_init(zkb_ctx** ctxs, int n);
/* transport: 0 single rank, 1 NCCL, 2 in-process peer copies; nccl_version as ncclGetVersion reports it (0 if unused) */
int zkb_comm_info(zkb_ctx* ctx, int* rank, int* n_ranks, int* transport, int* nccl_version);
/* COLLECTIVE.  The root's finalized program -> every other rank (which must not hold a program of its own).  The peers can
 * then evaluate, read values back (zkb_read_values) and answer zkb_assert_info / zkb_get_stats; they cannot record. */
int zkb_comm_broadcast_program(zkb_ctx* ctx, int root);
/* COLLECTIVE.  This rank evaluates witnesses [first, first + n_local) of a batch of n_total (host buffers as in zkb_evaluate,
 * holding this rank's n_local pairs); out[n_total] receives the verdicts of the WHOLE batch on every rank. */
int zkb_comm_evaluate(zkb_ctx* ctx, const uint8_t* instances_le, uint64_t instance_set_stride, const uint8_t* witnesses_le,
                      uint64_t witness_set_stride, uint32_t value_stride, uint32_t n_local, uint32_t first, uint32_t n_total,
                      zkb_verdict* out);
/* COLLECTIVE.  The same over the inputs already resident on this rank (zkb_upload_inputs / a previous zkb_comm_evaluate). */
int zkb_comm_run(zkb_ctx* ctx, uint32_t first, uint32_t n_total, zkb_verdict* out);
/* One process, N devices: zkb_evaluate over a batch split into N contiguous blocks, witness j on rank j*N/n_batch.
 * The program finalized on ctxs[0] is broadcast on first use.  Buffers hold the whole batch; out[n_batch]. */
int zkb_evaluate_sharded(zkb_ctx** ctxs, int n, const uint8_t* instances_le, uint64_t instance_set_stride,
                         const uint8_t* witnesses_le, uint64_t witness_set_stride, uint32_t value_stride, uint32_t n_batch,
                         zkb_verdict* out);
int zkb_run_sharded(zkb_ctx** ctxs, int n, uint32_t n_batch, zkb_verdict* out);

#ifdef __cplusplus
}
#endif
#endif /* ZKB_H */
