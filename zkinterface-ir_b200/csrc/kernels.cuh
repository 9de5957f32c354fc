// Launch wrappers of the sm_100a kernels (kernels.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "field.cuh"
#include "program.h"

namespace zkb {

// Wire store layout (limb-chunk-major, witness-minor):
//   an element of N 32-bit limbs is split in NC = max(1, N/4) chunks of CW = min(N, 4) limbs;
//   chunk c of slot s for witness lane j lives at  ((s*NC + c) * Wt + j) * CW  (uint32 units),
//   so a warp reading one chunk of one slot for 32 consecutive witnesses issues one fully
//   coalesced 16-byte-per-lane (512 B) request when N >= 4.
struct TileGeom {
    uint32_t log2_wt;   // witnesses per tile (power of two)
    uint32_t n_valid;   // lanes of this tile that hold real witnesses
    uint32_t batch0;    // global index of lane 0
    uint32_t skip_mask; // op flags whose results the level kernels do not store (besides F_NOSTORE): F_SINK on a tile that
                        // the next one overwrites before anything reads it back, else 0
};

struct InputDesc {
    const uint8_t* inst;      // instance values, raw little-endian, `stride` bytes each
    const uint8_t* wit;       // witness values
    uint64_t inst_set_stride; // bytes between consecutive witnesses' instance vectors (0: shared)
    uint64_t wit_set_stride;  // bytes between consecutive witnesses' witness vectors
    uint32_t stride;          // bytes per value
    uint32_t pad;
};

// What the gates that must see an input's RAW integer need (SURVEY.md section 8a trap 1: constant / instance / witness
// values >= p stay unreduced in the reference; assert_zero and not test the raw integer, and / xor operate on it).
struct RawCtx {
    const uint8_t* rawflag;     // per (input load, lane): raw value >= p; nullptr when no gate of the program needs it
    const InputLoad* loads;     // input slot -> (kind, stream index): input slots are the load indices
    const uint8_t* const_raw;   // raw little-endian bytes of the constants, const_raw_stride each (nullptr: none is >= p)
    uint32_t const_raw_stride;
    uint32_t pad;
    InputDesc in;
};

// arithmetic fields (odd p, Montgomery form)
void launch_to_mont(int nlimb, uint32_t* consts, uint32_t n, const FieldParams& fp, cudaStream_t s);
void launch_load_inputs(int nlimb, const InputLoad* loads, uint32_t n_loads, uint32_t* store, const uint32_t* consts_mont,
                        InputDesc in, TileGeom g, uint32_t* unreduced_count, uint8_t* rawflag, const uint8_t* const_flags,
                        const FieldParams& fp, int sm_count, cudaStream_t s);
void launch_level(int nlimb, const GateOp* ops, const uint32_t* aseq, uint64_t n_ops, uint32_t* store,
                  const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g, const FieldParams& fp,
                  int sm_count, bool rare, cudaStream_t s);
// every wavefront in one cooperative launch (grid barrier between levels); for launch-bound programs
cudaError_t launch_levels_coop(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                               uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                               const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t* barrier_ctr,
                               uint32_t* barrier_epoch, cudaStream_t s);
// every wavefront in one cooperative launch with no barrier: dataflow on "not computed yet" marker words (one witness, 1- / 2-limb
// fields, plans without slot re-use; kernels.cu: k_levels_flow).  fill_from .. n_slots: the computed slots.
cudaError_t launch_levels_flow(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                               uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                               const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t fill_from, uint32_t n_slots,
                               cudaStream_t s);
// the same for 4- / 8-limb fields: a flag word per slot holds the number (epoch) of the run that produced the value
cudaError_t launch_levels_flow_wide(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                                    uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                                    const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t n_ready, uint32_t* flags,
                                    uint32_t epoch, cudaStream_t s);
// microseconds per barrier of a kernel that does nothing else (kind 0: cooperative_groups grid.sync, 1: the counter barrier of
// k_levels_coop, 2: the hardware barrier of one 8-CTA cluster)
cudaError_t measure_barrier_cost(int kind, unsigned blocks, unsigned n_barriers, uint32_t* barrier_ctr, uint32_t* barrier_epoch,
                                 cudaStream_t s, cudaEvent_t ev0, cudaEvent_t ev1, float* us_per_barrier);
// call groups of one depth over a prime field (k_arith_groups): n_regs = the widest template's register count; first_fail gets
// the calls' failing assertions
void launch_arith_groups(int nlimb, const GroupDesc* descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* gops, const uint32_t* tables,
                         const uint32_t* hints, uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g,
                         const FieldParams& fp, uint32_t n_regs, int sm_count, cudaStream_t s);
uint32_t arith_group_threads(int nlimb, uint32_t n_regs);  // its CTA size
// carried loops of one depth (k_arith_chain, Plan::chain_descs): carry = their Plan::chain_carry rows, n_regs = Plan::chain_regs
// (rings and staging registers included)
void launch_arith_chain(int nlimb, const GroupDesc* descs, const uint32_t* carry, uint32_t n_chains, const GroupOp* gops, const uint32_t* tables,
                        uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g, const FieldParams& fp, uint32_t n_regs,
                        int sm_count, cudaStream_t s);
void launch_read_values(int nlimb, const uint32_t* slots, uint32_t n, const uint32_t* store, uint32_t lane, uint32_t log2_wt,
                        uint32_t* out, const FieldParams& fp, cudaStream_t s);

// p = 2: bit-sliced, one uint32 word = 32 witnesses
void launch_bool_load_inputs(const InputLoad* loads, uint32_t n_loads, uint32_t* store, const uint32_t* const_bits, InputDesc in,
                             TileGeom g, uint32_t* unreduced_count, uint8_t* rawflag, const uint8_t* const_flags, int sm_count,
                             cudaStream_t s);
void launch_bool_level(const GateOp* ops, const uint32_t* aseq, uint64_t n_ops, uint32_t* store, const uint32_t* const_bits,
                       uint32_t* first_fail, const uint8_t* rawflag, TileGeom g, int sm_count, cudaStream_t s);
// a run of wavefronts that each fit one CTA, in one launch (level_off: offsets into ops, relative to `ops`' own origin)
void launch_bool_levels_cta(const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels, uint32_t* store,
                            const uint32_t* const_bits, uint32_t* first_fail, const uint8_t* rawflag, TileGeom g, cudaStream_t s);
// call groups of one depth (program.h): n_regs = the widest template's register count
void launch_bool_groups(const GroupDesc* descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* gops, const uint32_t* tables,
                        const uint32_t* hints, uint32_t* store, TileGeom g, uint32_t n_regs, int sm_count, cudaStream_t s,
                        const GroupOp* host_ops, uint32_t n_host_ops);  // host copy of all templates' ops: sent as a kernel parameter when small
void launch_bool_read_values(const uint32_t* slots, uint32_t n, const uint32_t* store, uint32_t lane, uint32_t log2_wt,
                             uint32_t* out, cudaStream_t s);

// capture list (zkb_capture_values): what one captured value is read from
enum CaptureKind : uint32_t {
    CAP_STORE = 0,  // the wire store at `slot` (canonical residue; 0/1 over p = 2)
    CAP_INSTANCE,   // raw bytes of instance value `opb` (d_inst)
    CAP_WITNESS,    // raw bytes of witness value `opb` (d_wit)
    CAP_RAW_CONST,  // row `opb` of the capture list's table of constants >= p
};
struct CaptureDesc {
    uint32_t slot, kind, opb, pad;
};
// one tile's captured values -> out, witness-major: value i of tile lane j at out + ((g.batch0 + j) * n + i) * E bytes
// (E a multiple of 4, the value zero padded to E).  nlimb = 0: p = 2 (k_bool_capture), else k_capture<nlimb>.
cudaError_t launch_capture(int nlimb, const CaptureDesc* descs, uint32_t n, const uint32_t* store, InputDesc in, const uint8_t* raw_consts,
                           uint32_t raw_stride, TileGeom g, uint32_t E, uint8_t* out, const FieldParams& fp, cudaStream_t s);
// ops whose result lands in a slot marked in slot_bits and that carry F_SINK: clear the flag and list the op (up to cap of
// them; *n_found counts all).  launch_set_sink: F_SINK on (set) or off the listed ops.
void launch_unsink(GateOp* ops, uint64_t n_ops, const uint32_t* slot_bits, uint32_t* found, uint32_t cap, uint32_t* n_found, int sm_count,
                   cudaStream_t s);
void launch_set_sink(GateOp* ops, const uint32_t* idx, uint32_t n, bool set, cudaStream_t s);

void launch_fill_u32(uint32_t* p, uint32_t v, uint64_t n, int sm_count, cudaStream_t s);

}  // namespace zkb
